#!/usr/bin/env python
"""Benchmark of the hot path (BASELINE.json): Connector env-steps/s with the random agent at
10x10 / 5 agents, 65 536 envs per GPU (configs[1]), plus solved ParallelRandomWalk boards/s
as secondary lines.

    python bench.py --gpus N --steps K --warmup W            # our CUDA path
    python bench.py --steps K --dump-outputs DIR             # ... and the outputs of its last timed step as DIR/*.npy
    python bench.py --impl reference --gpus N --steps K ...  # the CPU arm (oracle, all host threads)

A "step" is one VmapAutoResetWrapper(Connector).step over the whole batch with actions from the
random policy: random-action sampling + Connector.step + observation + auto-reset (regeneration
of finished envs with ParallelRandomWalkGenerator), i.e. one iteration of the reference's
`agent=random` benchmark loop (benchmark_on_random_agent.py:59-102).  Prints ONE JSON line.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

# torchrun exports OMP_NUM_THREADS=1 to its workers.  libgomp reads it when it is first loaded, and a
# later num_threads(n) clause then runs the CPU arm 8x SLOWER than a single thread (measured), so the
# value is replaced by the core count before anything that links OpenMP is imported.
if os.environ.get("OMP_NUM_THREADS") == "1" and "RANK" in os.environ:
    try:
        os.environ["OMP_NUM_THREADS"] = str(max(1, len(os.sched_getaffinity(0))))
    except AttributeError:
        os.environ["OMP_NUM_THREADS"] = str(os.cpu_count() or 1)

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

G, N = 10, 5
ENVS_PER_GPU = 65536
TIME_LIMIT = 50
CELLS = G * G
STATE_BYTES = 4 * CELLS + 4 + 28 * N + 8            # 552 (SURVEY 8)
TS_BYTES = 4 * N * CELLS + 5 * N + 4 + 8 * N + 1 + 12  # obs + mask + step_count + reward/discount + step_type + extras = 2082
STEP_BYTES = STATE_BYTES + 4 * N + STATE_BYTES + TS_BYTES  # 3206 B per env-step (SURVEY 8d)
PRW_BOARD_BYTES = {(10, 5): 488, (20, 10): 1768, (32, 16): 4360}
SE_MEAN_SWEEPS_14_7 = 9.86  # extend_wires_jax sweeps per 14x14/7 board, mean over split(PRNGKey(0), 262144) (oracle; tools/se_stats.py)
METRIC = "connector_env_steps_per_sec"
UNIT = "env-steps/s"


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20", "-i", str(self.index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.f.close()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        with open(self.path) as f:
            for line in f:
                p = [x.strip() for x in line.split(",")]
                if len(p) < 9:
                    continue
                try:
                    sm.append(float(p[1]))
                    mx.append(float(p[2]))
                except ValueError:
                    continue
                for nm, v in zip(names, p[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
        os.unlink(self.path)
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


# issue roofline of the generator kernels: one warp-instruction per clock per SM sub-partition
SMSP_PER_SM = 4


def _issue_peak(sm_count: int, sm_mhz: float) -> float:
    return sm_count * SMSP_PER_SM * sm_mhz * 1e6  # warp-instructions / s


def _profile_number(key: str):
    """A per-launch / per-board figure from the committed ncu captures (profiles/traffic.json), or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f).get(key)
    except Exception:
        return None


class Dist:
    """The multi-GPU plumbing of the bench: barrier, max over ranks (NCCL); no-ops at N = 1."""

    def __init__(self, world, dev):
        self.world, self.dev = world, dev

    def sync(self):
        import torch
        import torch.distributed as dist

        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def max(self, x: float) -> float:
        import torch
        import torch.distributed as dist

        if self.world == 1:
            return float(x)
        t = torch.tensor([x], dtype=torch.float64, device=self.dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())


def timed_samples(dd: Dist, enqueue, steps: int, min_ms: float = 60.0, samples: int = 5, probe_blocks: int = 2):
    """Device time of `steps`-step blocks.  One SAMPLE = R blocks of exactly `steps` steps enqueued back to back
    between two CUDA events (R chosen so that a sample lasts >= min_ms; a single 20-step block is 0.6 ms, far
    too short to time alone, and events between the blocks would serialise launches that are chained head to
    tail); bracketed by barrier + synchronize, max over ranks.  Returns (R, [ms per block for each sample])."""
    import torch

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    dd.sync()
    e0.record()
    for _ in range(probe_blocks):
        enqueue(steps)
    e1.record()
    dd.sync()
    est = dd.max(e0.elapsed_time(e1) / probe_blocks)
    R = int(min(2000, max(1, -(-min_ms // max(est, 1e-3)))))
    out = []
    for _ in range(samples):
        dd.sync()
        e0.record()
        for _ in range(R):
            enqueue(steps)
        e1.record()
        dd.sync()
        out.append(dd.max(e0.elapsed_time(e1)) / R)
    return R, out


def timed_window(dd: Dist, enqueue, steps: int, spin_cycles: int = 2_000_000) -> float:
    """Device time in ms of exactly `steps` steps enqueued back to back between two CUDA events, max over ranks.
    A spin kernel of about 1 ms ahead of the first event keeps the stream busy while the host enqueues the first
    launches, so the window times the steps and not the host's launch latency."""
    import torch

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    dd.sync()
    torch.cuda._sleep(spin_cycles)
    e0.record()
    enqueue(steps)
    e1.record()
    dd.sync()
    return dd.max(e0.elapsed_time(e1))


DUMP_ENVS = 16384  # envs sampled for --dump-outputs: 45 MB at 10x10/5, under a budget of 64 MB


def _dump_outputs(path, state, ts, act, t, B):
    """The last timed step as a caller of rbg_connector_rollout_random receives it: TimeStep `t` of the stacked outputs, the
    actions taken in that step and the State after it, for a fixed seeded sample of envs (all of them when B <= DUMP_ENVS).
    Keys (uint32) as float64, everything else as float32: codes, counts and coordinates are small integers, exact in both."""
    import numpy as np
    import torch

    idx = np.arange(B) if B <= DUMP_ENVS else np.sort(np.random.default_rng(0).choice(B, DUMP_ENVS, replace=False))
    sel = torch.from_numpy(idx).to(state.grid.device)
    o, a = ts.observation, state.agents
    arrays = {
        "env_index": (torch.from_numpy(idx), np.float64),
        "observation_grid": (o.grid[t], np.float32), "observation_action_mask": (o.action_mask[t], np.float32), "observation_step_count": (o.step_count[t], np.float32),
        "reward": (ts.reward[t], np.float32), "discount": (ts.discount[t], np.float32), "step_type": (ts.step_type[t], np.float32),
        "num_connections": (ts.extras["num_connections"][t], np.float32), "ratio_connections": (ts.extras["ratio_connections"][t], np.float32),
        "total_path_length": (ts.extras["total_path_length"][t], np.float32), "action": (act[t], np.float32),
        "state_grid": (state.grid, np.float32), "state_step_count": (state.step_count, np.float32), "state_key": (state.key.view(torch.int32), np.float64),
        "agent_id": (a.id, np.float32), "agent_start": (a.start, np.float32), "agent_target": (a.target, np.float32), "agent_position": (a.position, np.float32),
    }
    os.makedirs(path, exist_ok=True)
    total = 0
    for name, (x, dtype) in arrays.items():
        x = x if name == "env_index" else x.index_select(0, sel)
        v = x.cpu().numpy()
        if name == "state_key":
            v = v.view(np.uint32)
        v = v.astype(dtype)
        total += v.nbytes
        np.save(os.path.join(path, f"{name}.npy"), v)
    assert total <= 64 << 20, total


def _stats(xs):
    return {"median": round(statistics.median(xs), 6), "min": round(min(xs), 6), "max": round(max(xs), 6)}


# ------------------------------------------------------------------ our arm
def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    import __graft_entry__ as ge

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if rank == 0:
        ge.build_library()
    if world > 1:
        dist.barrier()
    import routing_board_generation_b200 as rbg
    from routing_board_generation_b200 import engine, sharding

    lib = rbg._lib.load()
    dev = torch.device("cuda", local)
    dd = Dist(world, dev)
    B = args.envs
    total = B * world  # weak scaling: 65 536 envs per GPU
    keys = sharding.shard_keys(rbg.PRNGKey(0), total, rank, world)
    env = rbg.VmapAutoResetWrapper(rbg.Connector(generator=rbg.ParallelRandomWalkGenerator(G, N), time_limit=TIME_LIMIT))
    state, ts = env.reset(keys)

    # The timed loop drives the engine the way the reference's training / benchmark loop does: a
    # scan of `n_steps` = 20 env steps per call (configs/env/connector.yaml:27), here one
    # rbg_connector_rollout_random call per chunk writing stacked [20, B, ...] TimeSteps.
    chunk = args.chunk
    ts = engine.alloc_timestep(B, G, N, chunk)
    act = torch.empty((chunk, B, N), dtype=torch.int32, device=dev)

    last = {}

    def run_steps(k):
        while k > 0:
            n = min(k, chunk)
            engine.connector_rollout_random(state, n, TIME_LIMIT, -0.03, 0.1, autoreset_kind="parallel_random_walk", out=ts, actions=act, owner=env)
            last["t"] = n - 1  # the slot of the stacked outputs that holds the latest step
            k -= n

    # Burn-in to the stationary regime: right after reset() every env is at step 0, so the
    # first episodes end in lock-step (all survivors hit time_limit together); a few episode
    # lengths later terminations are spread evenly (about 4 % of the envs per step).
    run_steps(args.burnin)
    run_steps(max(args.warmup, 3))
    dd.sync()

    # ---- timed region: exactly K steps, device-timed, max over ranks
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    rbg.launch_count(reset=True)
    ms_window = timed_window(dd, run_steps, args.steps)
    launches = rbg.launch_count()
    value = total * args.steps / (ms_window / 1e3)
    if args.dump_outputs and rank == 0:
        _dump_outputs(args.dump_outputs, state, ts, act, last["t"], B)

    # ---- the dominant kernel alone: event pairs recorded inside the library around every launch
    # (which also switches the head-to-tail chaining of consecutive launches off), over a second pass
    rbg._lib.kernel_timing(True)
    for k in ("env", "prw", "rollout"):
        rbg._lib.kernel_time(k)
    n_pass = max(args.steps, 10 * chunk)
    run_steps(n_pass)
    torch.cuda.synchronize()
    n_env, ms_env = rbg._lib.kernel_time("env")
    n_prw, ms_prw = rbg._lib.kernel_time("prw")
    n_ro, ms_ro = rbg._lib.kernel_time("rollout")
    rbg._lib.kernel_timing(False)
    clocks = sampler.stop() if rank == 0 else None  # sampled over the timed region and the kernel-timing pass
    peak, peak_src = _peaks()
    steps_per_launch = n_pass / max(n_ro, 1)
    # State read once + written once per launch; per step only the emitted TimeStep and the actions
    alg = B * (2 * STATE_BYTES + steps_per_launch * (TS_BYTES + 4 * N))
    # The timed region holds nothing but launches of this one kernel (one per 20-step chunk, each INCLUDING the
    # regeneration of finished envs), chained head to tail, so its average launch duration over the region is the
    # region's device time / launches.  The same launch timed ALONE (event pair around it, not chained: its ragged tail
    # and the generator warps' drain are exposed) is reported next to it.
    launches_timed = -(-args.steps // chunk)
    k_ms = ms_window / launches_timed
    achieved = alg * (args.steps / launches_timed / steps_per_launch) / (k_ms / 1e3) / 1e9
    alone_ms = ms_ro / max(n_ro, 1)
    alone = alg / (alone_ms / 1e3) / 1e9
    step_alg = B * (TS_BYTES + 4 * N + 2 * STATE_BYTES / steps_per_launch)  # algorithmic bytes of one whole step
    step_gbs = step_alg / (ms_window / args.steps / 1e3) / 1e9
    roofline = {"kernel": "rollout_persist_kernel", "bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 4),
                "traffic": _profile_number("rollout_persist_kernel"), "algorithmic_bytes_per_launch": int(alg), "steps_per_launch": steps_per_launch,
                "avg_launch_ms": round(k_ms, 5), "peak_source": peak_src, "kernel_share_of_step": round(ms_ro / max(ms_ro + ms_prw + ms_env, 1e-9), 4),
                "other_kernels_in_the_step": {"prw_kernel_launches": n_prw, "env_kernel_launches": n_env},
                "note": "one launch = 20 steps over the whole batch INCLUDING the regeneration of finished envs (generator warps inside the rollout CTAs); avg_launch_ms = device time of the timed region / launches in it (consecutive launches are chained head to tail by programmatic dependent launch)",
                "launch_timed_alone": {"avg_launch_ms": round(alone_ms, 5), "achieved": round(alone, 1), "frac": round(alone / peak, 4),
                                       "note": "the same launch bracketed by its own event pair in a separate pass: not chained, so the ragged end of a persistent grid and the generator warps' drain are exposed"},
                "whole_step": {"achieved": round(step_gbs, 1), "frac": round(step_gbs / peak, 4),
                               "note": "algorithmic bytes of a step / the timed region's ms_per_step; the step is that one kernel, so this equals `frac` up to the State's share"}}

    # ---- e2e: the env-step call with HOST buffers through the C-ABI (rbg_connector_step_host_io):
    # actions H2D from pinned memory, step, whole TimeStep D2H, every step.
    e2e = None
    cpu_baseline = None
    # the legs below are additions to the headline numbers above: an error in one of them (it would hit every rank alike) is
    # reported in its place instead of costing the run its line
    if not args.skip_e2e:
        try:
            e2e = _e2e_host(args, rbg, lib, state, B, world, rank, dev)
        except Exception as e:  # noqa: BLE001
            e2e = {"value": None, "unit": UNIT, "error": repr(e)}
    del ts, act
    torch.cuda.empty_cache()
    sm_mhz = (clocks or {}).get("sm_max_mhz") or 1965.0
    secondary = []
    if not args.skip_secondary:
        try:
            secondary = _secondary(args, rbg, dd, peak, rank, world, sm_mhz)
        except Exception as e:  # noqa: BLE001
            secondary = [{"error": repr(e)}]
    if rank == 0 and world == 1 and not args.skip_cpu:
        try:
            cpu_baseline = _cpu_baseline(budget_s=args.cpu_seconds, burnin=args.burnin, envs=B)
            if not args.skip_secondary:
                _cpu_secondary(secondary, budget_s=max(2.0, args.cpu_seconds / 3))
        except Exception as e:  # noqa: BLE001
            cpu_baseline = cpu_baseline or {"value": None, "error": repr(e)}

    if rank == 0:
        line = {
            "metric": METRIC, "value": round(value, 1), "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": round(ms_window / args.steps, 5), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32",
            "data": "synthetic (keys = split(PRNGKey(0), B), random-policy actions)",
            "config": {"workload": "connector_step_random_agent_autoreset_prw", "grid": G, "agents": N, "envs_per_gpu": B, "envs_total": total, "time_limit": TIME_LIMIT,
                       "generator": "ParallelRandomWalkGenerator", "parallelism": f"env-sharded x{world}", "burnin_steps": args.burnin,
                       "api": f"rbg_connector_rollout_random, {chunk} steps per call (the reference's n_steps scan), State in place, stacked TimeSteps and actions written every step",
                       "l2": f"no flush: every step writes {(TS_BYTES + 4 * N) * B / 1e6:.0f} MB per GPU into a fresh slice of the stacked [{chunk}, B, ...] outputs ({(TS_BYTES + 4 * N) * B * chunk / 1e9:.1f} GB per call), far beyond the 126 MB L2"},
            "timing": {"what": f"exactly {args.steps} steps ({launches_timed} rollout calls) enqueued back to back between two CUDA events (barrier + synchronize on both sides, max over ranks); "
                               "the window includes the ramp of its first launch and the drain of its last, which a short window does not amortise",
                       "window_ms": round(ms_window, 4)},
            "roofline": roofline, "cpu_baseline": cpu_baseline, "e2e": e2e, "gpu_launches": launches, "clocks": clocks, "secondary": secondary,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def _e2e_host(args, rbg, lib, state, B, world, rank, dev):
    """The env step as a host-side consumer sees it (rbg_connector_step_host_io): every step the
    actions are copied H2D from pinned memory and the whole TimeStep (observation, mask, reward,
    discount, step_type, extras) is copied back D2H; the State is the env's own device-resident
    state, exactly as in the reference's loop."""
    import numpy as np
    import torch
    import torch.distributed as dist

    L = rbg._lib

    def pinned(shape, dtype):
        return torch.empty(shape, dtype=dtype).pin_memory()

    hts = dict(obs=pinned((B, N, G, G), torch.int32), mask=pinned((B, N, 5), torch.uint8), sc=pinned((B,), torch.int32), reward=pinned((B, N), torch.float32), discount=pinned((B, N), torch.float32),
               step_type=pinned((B,), torch.int8), nc=pinned((B,), torch.int32), rc=pinned((B,), torch.float32), tpl=pinned((B,), torch.int32))
    act = pinned((B, N), torch.int32)
    rng = np.random.default_rng(rank)
    act.copy_(torch.from_numpy(rng.integers(0, 5, size=(B, N)).astype(np.int32)))
    a = state.agents
    s = L.rbg_state(state.grid.data_ptr(), state.step_count.data_ptr(), a.id.data_ptr(), a.start.data_ptr(), a.target.data_ptr(), a.position.data_ptr(), state.key.data_ptr())
    t = L.rbg_timestep(*(hts[k].data_ptr() for k in ("obs", "mask", "sc", "reward", "discount", "step_type", "nc", "rc", "tpl")))
    params = L.rbg_env_params(TIME_LIMIT, -0.03, 0.1, 0)
    h2d = act.numel() * 4
    d2h = sum(v.numel() * v.element_size() for v in hts.values())

    def step():
        L.check(lib.rbg_connector_step_host_io(C.byref(s), act.data_ptr(), B, G, N, C.byref(params), C.byref(t), -1))

    for _ in range(24):  # the library tries four host-thread counts on its first sixteen calls of a batch shape and keeps the fastest
        step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    k = max(3, min(args.steps, 30))
    # five groups of exactly k synchronous steps; every group's time is the max over ranks, the median group is reported
    # (the hosts of this pool are shared VMs: a group can lose a third of its rate to a neighbour)
    groups = []
    for _ in range(5):
        if world > 1:
            dist.barrier()
        L.host_transfer_stats(reset=True)
        t0 = time.perf_counter()
        for _ in range(k):
            step()  # synchronous: returns after the TimeStep has landed in the host buffers
        gdt = time.perf_counter() - t0
        h2d_moved, d2h_moved, host_threads = L.host_transfer_stats()
        tt = torch.tensor([gdt], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        groups.append(float(tt.item()))
    dt = statistics.median(groups)
    # context: what the bus gives a plain pinned D2H copy of the int32 observation buffer alone
    dobs = torch.empty((B, N, G, G), dtype=torch.int32, device=dev)
    hts["obs"].copy_(dobs, non_blocking=True)
    torch.cuda.synchronize()
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c0.record()
    for _ in range(5):
        hts["obs"].copy_(dobs, non_blocking=True)
    c1.record()
    torch.cuda.synchronize()
    bus = dobs.numel() * 4 * 5 / (c0.elapsed_time(c1) / 1e3) / 1e9
    delivered = d2h * k / dt / 1e9
    moved = d2h_moved / dt / 1e9
    packed = host_threads > 0
    # context: the host half of the packed transport alone (byte codes already in pinned host memory -> the int32 observation
    # buffer, same thread count, every rank at once): what this host's memory system allows the call to deliver
    ceiling = None
    if packed:
        src8 = torch.empty((B, N, G, G), dtype=torch.uint8).pin_memory()
        src8.random_(0, 16)
        n_obs = src8.numel()
        widen = lib.rbg_host_widen4 if d2h_moved // k < n_obs else lib.rbg_host_widen  # the transport the step used
        for _ in range(2):
            L.check(widen(src8.data_ptr(), hts["obs"].data_ptr(), n_obs))
        if world > 1:
            dist.barrier()
        w0 = time.perf_counter()
        for _ in range(5):
            L.check(widen(src8.data_ptr(), hts["obs"].data_ptr(), n_obs))
        wt = torch.tensor([(time.perf_counter() - w0) / 5], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(wt, op=dist.ReduceOp.MAX)
        wdt = float(wt.item())
        ceiling = {"env_steps_per_s": round(B * world / wdt, 1), "int32_gbs_per_rank": round(n_obs * 4 / wdt / 1e9, 1), "frac": round((B * world * k / dt) / (B * world / wdt), 4),
                   "note": "rbg_host_widen / rbg_host_widen4 of one step's observation alone on every rank at once (codes resident in pinned host memory, no GPU work, no bus): the rate at which this host's cores and memory system can write the API's int32 observation; `frac` = e2e value / this"}
        del src8
    return {"value": round(B * world * k / dt, 1), "unit": UNIT, "h2d_bytes_per_step": int(h2d_moved // k), "d2h_bytes_per_step": int(d2h_moved // k), "steps": k,
            "api": "rbg_connector_step_host_io (pinned host actions in, full TimeStep out to host memory, State device-resident, auto-reset on)",
            "transport": ((f"observation codes (<= 3 N = {3 * N}) cross the bus as {'nibbles, two cells per byte,' if d2h_moved // k < B * N * G * G else 'uint8'} and are widened to the API's int32 "
                           f"by {host_threads} host threads inside the call (slices pipelined)")
                          if packed else "int32 observation over the bus (RBG_HOST_IO_WIDE=1)"),
            "host_threads": host_threads, "timestep_bytes_delivered_per_step": int(d2h),
            "timer": "host wall clock around synchronous calls, max over ranks; median of five groups of `steps` steps",
            "group_values": [round(B * world * k / g, 1) for g in groups],
            "bytes_counted": "by the library where it enqueues the copies (rbg_host_transfer_stats)",
            "d2h_gbs": round(moved, 1), "delivered_gbs": round(delivered, 1), "pinned_d2h_copy_gbs": round(bus, 1),
            "delivered_vs_plain_int32_copy": round(delivered / bus, 3), "host_widen_ceiling": ceiling}


def _secondary(args, rbg, dd, peak, rank, world, sm_mhz):
    """The other BASELINE configs, on every rank (weak scaling like the headline: per-GPU sizes fixed, keys =
    this rank's slice of split(PRNGKey(0), total)), device-timed, max over ranks; rank 0 keeps the lines.
      configs[0]/[2]  ParallelRandomWalkBoard.generate_board: 10x10/5 and 20x20/10 x 131 072 boards per GPU (= 1 M boards at N = 8), 32x32/16
      configs[3]      SeedExtension 14x14/7 x 65 536 boards + rbg_validate on every board
      configs[4]      fused generate + reset + rollout 32x32/16, 8 192 envs per GPU, 20 steps per call
      and the headline workload through the per-step API."""
    import torch

    from routing_board_generation_b200 import sharding

    out = []
    sm_count = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    issue_peak = _issue_peak(sm_count, sm_mhz)

    def timed(fn, reps, min_ms=40.0):
        for _ in range(2):
            fn()
        _, ms = timed_samples(dd, lambda _k: fn(), 1, min_ms=min_ms, samples=3, probe_blocks=max(1, reps // 4))
        return statistics.median(ms), ms

    def issue(line, key, units_per_s):
        """fraction of the issue roofline: warp-instructions per unit (committed ncu capture) x units/s / (SMs x 4 x f)"""
        wi = _profile_number(key)
        if wi:
            line["roofline"] = {"bound": "issue", "unit": "warp-inst/s", "warp_inst_per_unit": wi, "achieved": round(wi * units_per_s / world, 1), "peak": round(issue_peak, 1),
                                "frac": round(wi * units_per_s / world / issue_peak, 4), "peak_source": f"{sm_count} SMs x 4 SMSP x {sm_mhz:.0f} MHz x 1 warp-inst/clk", "warp_inst_source": f"profiles/traffic.json[{key}]"}

    for (g, n, b) in ((10, 5, 65536), (20, 10, 131072), (32, 16, 32768)):
        keys = sharding.shard_keys(rbg.PRNGKey(0), b * world, rank, world)
        board = rbg.ParallelRandomWalkBoard(g, g, n)
        ms, all_ms = timed(lambda: board.generate_board(keys), 10)
        bytes_ = PRW_BOARD_BYTES[(g, n)] * b
        line = {"metric": "prw_solved_boards_per_sec", "workload": f"ParallelRandomWalkBoard.generate_board {g}x{g}/{n}, {b} boards per GPU ({b * world} total)", "grid": g, "agents": n, "value": round(b * world / (ms / 1e3), 1), "unit": "boards/s",
                "n_gpus": world, "ms_per_batch": round(ms, 4), "ms_samples": [round(x, 4) for x in all_ms], "output_gbs_per_gpu": round(bytes_ / (ms / 1e3) / 1e9, 2), "hbm_frac": round(bytes_ / (ms / 1e3) / 1e9 / peak, 5),
                "bound": "integer issue (threefry2x32), see DESIGN.md"}
        issue(line, f"prw_kernel_{g}x{g}_{n}_warp_inst_per_board", b * world / (ms / 1e3))
        out.append(line)
        if (g, n) == (10, 5):
            # the consumer of solved boards in the reference's benchmark: EvaluateEmptyBoard statistics per board
            solved = board.generate_board(keys)[2]
            ms2, all2 = timed(lambda: rbg.engine.board_statistics(solved), 10)
            sb = (8 * g * g + 8) * b  # int32 board in, int32 scored board out, two int32 per board
            out.append({"metric": "board_statistics_boards_per_sec", "workload": f"EvaluateEmptyBoard statistics (scored board, count_detours, heatmap_score_diversity) {g}x{g}/{n}, {b} boards per GPU",
                        "value": round(b * world / (ms2 / 1e3), 1), "unit": "boards/s", "n_gpus": world, "ms_per_batch": round(ms2, 4), "ms_samples": [round(x, 4) for x in all2],
                        "output_gbs_per_gpu": round(sb / (ms2 / 1e3) / 1e9, 1), "hbm_frac": round(sb / (ms2 / 1e3) / 1e9 / peak, 4), "bound": "issue (G^3 / 32 row-column scans per lane for count_detours)"})
            del solved
        del keys
    # the headline workload through the per-step API (one rbg_connector_step_random call per env step:
    # env_warp_kernel + reset kernel + side-stream cache refill), for callers that cannot use the fused rollout
    g, n, b = G, N, 65536
    env = rbg.VmapAutoResetWrapper(rbg.Connector(generator=rbg.ParallelRandomWalkGenerator(g, n), time_limit=TIME_LIMIT))
    box = {"st": env.reset(sharding.shard_keys(rbg.PRNGKey(0), b * world, rank, world))[0]}
    ts1 = rbg.engine.alloc_timestep(b, g, n)

    def one_step():
        box["st"], _, _ = rbg.engine.connector_step(box["st"], None, TIME_LIMIT, -0.03, 0.1, autoreset_kind="parallel_random_walk", inplace=True, random_policy=True, out=ts1, owner=env)

    for _ in range(args.burnin):
        one_step()
    _, ms_l = timed_samples(dd, lambda k: [one_step() for _ in range(k)], 20, min_ms=40.0, samples=3)
    ms = statistics.median(ms_l) / 20
    out.append({"metric": "connector_env_steps_per_sec", "workload": f"per-step API (one Python call = one rbg_connector_step_random per env step) {g}x{g}/{n}, {b} envs per GPU", "value": round(b * world / (ms / 1e3), 1), "unit": "env-steps/s",
                "n_gpus": world, "ms_per_step": round(ms, 5), "ms_per_step_samples": [round(x / 20, 5) for x in ms_l], "output_gbs_per_gpu": round(STEP_BYTES * b / (ms / 1e3) / 1e9, 1), "hbm_frac": round(STEP_BYTES * b / (ms / 1e3) / 1e9 / peak, 4)})
    del ts1, box, env
    # fused generate + reset + rollout at the A2C rollout shape (BASELINE configs[4]): 32x32 / 16 agents, 20 steps
    g, n, b, T = 32, 16, 8192, 20
    env = rbg.VmapAutoResetWrapper(rbg.Connector(generator=rbg.ParallelRandomWalkGenerator(g, n), time_limit=TIME_LIMIT))
    st, _ = env.reset(sharding.shard_keys(rbg.PRNGKey(0), b * world, rank, world))
    ts_big = rbg.engine.alloc_timestep(b, g, n, T)
    for _ in range(6):  # past the first episodes
        env.rollout_random(st, T, out=ts_big)
    ms, all_ms = timed(lambda: env.rollout_random(st, T, out=ts_big), 5, min_ms=30.0)
    step_bytes = 4 * n * g * g + 5 * n + 4 + 8 * n + 1 + 12 + 4 * n  # what a fused step must emit (SURVEY 8d: 65 825 B)
    out.append({"metric": "connector_env_steps_per_sec", "workload": f"fused generate+reset+rollout {g}x{g}/{n}, {b} envs per GPU, {T} steps per call", "value": round(b * world * T / (ms / 1e3), 1), "unit": "env-steps/s",
                "n_gpus": world, "ms_per_step": round(ms / T, 4), "ms_per_call_samples": [round(x, 4) for x in all_ms], "output_gbs_per_gpu": round(step_bytes * b * T / (ms / 1e3) / 1e9, 1),
                "hbm_frac": round(step_bytes * b * T / (ms / 1e3) / 1e9 / peak, 4), "bound": "hbm"})
    del ts_big, st, env
    torch.cuda.empty_cache()
    # SeedExtension 14x14/7 (BASELINE configs[3]): generation + on-device validity of every board, at the batch round 1
    # used (one wave of the extend kernel: bound by the slowest board's 45 sweeps) and at dataset-generation scale (the
    # reference builds its offline dataset of number_of_boards = 100 000 boards, agent_training/configs/env/connector.yaml:15)
    g, n = 14, 7
    board = rbg.SeedExtensionBoard(g, g, n)
    # floor of the pipeline: the key chain alone (key, random_key = split(key) per cell and sweep, SE_LOOK = 8 cells past the
    # sweep) at the ALU-pipe rate of the chain microbenchmark (tools/micro/tf_chain_bench.cu: 196 cycles per chain step and
    # warp with the SM sub-partition's ALU pipe saturated), 32 boards per warp, mean sweeps per board from the oracle
    chain_floor = sm_count * 4 * sm_mhz * 1e6 / (SE_MEAN_SWEEPS_14_7 * (g * g + 8) * 196.0 / 32.0)
    for b in (65536, 262144):
        keys = sharding.shard_keys(rbg.PRNGKey(0), b * world, rank, world)
        res = {}

        def se():
            res["solved"] = board.return_solved_board(keys)
            res["flags"] = rbg.engine.validate(res["solved"], n)

        ms, all_ms = timed(se, 5, min_ms=30.0)
        rate = b * world / (ms / 1e3)
        line = {"metric": "seedext_solved_boards_per_sec", "workload": f"SeedExtensionBoard.return_solved_board {g}x{g}/{n}, {b} boards per GPU + rbg_validate", "boards_per_gpu": b, "value": round(rate, 1), "unit": "boards/s",
                "n_gpus": world, "ms_per_batch": round(ms, 4), "ms_samples": [round(x, 4) for x in all_ms], "invalid_boards": int((res["flags"] != 0).sum()),
                "bound": "sequential threefry chain per board (G*G*sweeps dependent split() steps) on the ALU pipe, see DESIGN.md K3",
                "chain_floor": {"boards_per_s_per_gpu": round(chain_floor, 1), "frac": round(rate / world / chain_floor, 4),
                                "note": "what the GPU would do if the pipeline were nothing but the key chain at the measured ALU-pipe rate: 196 cycles per chain step and warp, 32 boards per warp, 9.86 sweeps per board"}}
        issue(line, f"seedext_pipeline_14x14_7_b{b}_warp_inst_per_board", rate)
        out.append(line)
        del keys, res
    # SequentialRandomWalkBoard.generate (SURVEY 8 f4; the reference quotes 685 us for ONE 10x10/5 board and its vmap fails)
    g, n, b = 10, 5, 65536
    keys = sharding.shard_keys(rbg.PRNGKey(0), b * world, rank, world)
    sboard = rbg.SequentialRandomWalkBoard(g, g, n)
    ms, all_ms = timed(lambda: sboard.generate(keys), 5, min_ms=30.0)
    line = {"metric": "seqrw_boards_per_sec", "workload": f"SequentialRandomWalkBoard.generate {g}x{g}/{n}, {b} boards per GPU", "grid": g, "agents": n, "value": round(b * world / (ms / 1e3), 1), "unit": "boards/s",
            "n_gpus": world, "ms_per_batch": round(ms, 4), "ms_samples": [round(x, 4) for x in all_ms], "bound": "integer issue (threefry2x32), see DESIGN.md K5"}
    issue(line, f"seqrw_kernel_{g}x{g}_{n}_warp_inst_per_board", b * world / (ms / 1e3))
    out.append(line)
    del keys
    return out if rank == 0 else []


# ------------------------------------------------------------------ CPU arm
def _cpu_workload(orc, B, nthreads, burnin=0):
    """reset B envs with the oracle, run `burnin` untimed steps (the same stationary regime as the GPU arm:
    episode ends desynchronised, about 4 % of the envs reset per step) and return a stepping closure
    (random policy + auto-reset step)."""
    kref = orc.split(orc.PRNGKey(0), B)
    st, _ = orc.connector_reset_batch("parallel_random_walk", kref, G, N, nthreads=nthreads)
    box = {"st": st, "ts": None}

    def step():
        act = orc.random_actions_batch(box["st"], nthreads=nthreads)
        # state updated in place, timestep buffers reused: no allocation inside the timed loop
        box["st"], box["ts"] = orc.connector_step_batch(box["st"], act, time_limit=TIME_LIMIT, autoreset_kind="parallel_random_walk", nthreads=nthreads, inplace=True, out=box["ts"])
        return box["ts"]

    for _ in range(burnin):
        step()
    return step


def _host_threads() -> int:
    """Every core this process may run on.  Not omp_get_max_threads(): torchrun exports OMP_NUM_THREADS=1
    to its workers, which would quietly turn the CPU arm into a single-thread run at --gpus > 1."""
    try:
        n = max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        n = max(1, os.cpu_count() or 1)
    return n


def _cpu_baseline(budget_s: float = 12.0, burnin: int = 160, envs: int = ENVS_PER_GPU):
    """The oracle port on every host core: the SAME batch and the same burn-in as the GPU arm and the
    reference arm, for a bounded number of steps."""
    cores = _host_threads()
    from oracle import oracle as orc

    orc.build()
    step = _cpu_workload(orc, envs, cores, burnin=burnin)
    n, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < budget_s or n < 5:
        step()
        n += 1
    dt = time.perf_counter() - t0
    return {"value": round(envs * n / dt, 1), "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{n} auto-reset random-agent steps over {envs} envs 10x10/5 after {burnin} burn-in steps (the GPU arm's batch and regime), OpenMP over envs, {dt:.1f} s"}


def _cpu_secondary(secondary, budget_s: float = 4.0):
    """boards/s of the CPU port for the generator lines (all host cores, bounded samples), and the reference's own
    NumPy BFSBoard generator (BASELINE's secondary baseline, README.md:88-93) where /root/reference is mounted
    (the build container; it does not exist on the GPU box)."""
    cores = _host_threads()
    from oracle import oracle as orc

    def rate(fn, n0):
        n, t0, done = n0, time.perf_counter(), 0
        while True:
            fn(n)
            done += n
            dt = time.perf_counter() - t0
            if dt > budget_s:
                return done / dt, done, dt
            n = min(n * 2, 1 << 16)

    se_cpu = None
    for line in secondary:
        if line.get("metric") == "prw_solved_boards_per_sec":
            g, n = line["grid"], line["agents"]
            v, done, dt = rate(lambda k: orc.prw_generate_batch(orc.split(orc.PRNGKey(1), k), g, n, nthreads=cores), 512)
            line["cpu_baseline"] = {"value": round(v, 1), "unit": "boards/s", "cores": cores, "kind": "port", "sample": f"{done} boards {g}x{g}/{n} in {dt:.1f} s, OpenMP over boards"}
        elif line.get("metric") == "seqrw_boards_per_sec":
            g, n = line["grid"], line["agents"]
            v, done, dt = rate(lambda k: orc.seqrw_generate_batch(orc.split(orc.PRNGKey(1), k), g, n, nthreads=cores), 512)
            line["cpu_baseline"] = {"value": round(v, 1), "unit": "boards/s", "cores": cores, "kind": "port", "sample": f"{done} boards {g}x{g}/{n} in {dt:.1f} s, OpenMP over boards"}
        elif line.get("metric") == "seedext_solved_boards_per_sec":
            if se_cpu is None:
                v, done, dt = rate(lambda k: orc.seedext_solved_batch(orc.split(orc.PRNGKey(1), k), 14, 7, nthreads=cores), 256)
                se_cpu = {"value": round(v, 1), "unit": "boards/s", "cores": cores, "kind": "port", "sample": f"{done} boards 14x14/7 in {dt:.1f} s, OpenMP over boards"}
            line["cpu_baseline"] = se_cpu
    bfs = {"metric": "numpy_bfs_board_boards_per_sec", "workload": "reference NumPy BFSBoard(10, 10, 5).return_solved_board() in a Python loop, single process (README.md:88-93)", "unit": "boards/s"}
    if os.path.isdir("/root/reference/routing_board_generation"):
        try:
            r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "time_bfs_board_numpy.py"), "150"], capture_output=True, text=True, timeout=120)
            d = json.loads(r.stdout.strip().splitlines()[-1])
            bfs.update(value=d["boards_per_sec"], cores=1, kind="reference", sample=f"{d['boards']} boards in {d['seconds']} s, measured in this run")
        except Exception as e:  # noqa: BLE001
            bfs.update(value=None, note=f"failed here: {e!r}")
    else:
        bfs.update(value=None, kind="reference", note="the reference is not mounted on this box; build-container figure: 456 boards/s on one core (profiles/r01_cpu_baselines.md, tools/time_bfs_board_numpy.py)")
    secondary.append(bfs)


def run_reference(args):
    """The reference's CPU implementation of the path.  The reference is pure Python on JAX and
    neither jax nor jumanji exist in this image (DESIGN.md), so this arm times the C oracle port
    with every host thread, on the GPU arm's batch and after the same burn-in."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = _host_threads()
    from oracle import oracle as orc

    orc.build()
    B = args.envs
    step = _cpu_workload(orc, B, cores, burnin=args.burnin)
    for _ in range(max(args.warmup, 1)):
        step()
    # blocks of exactly K steps until the sample is long enough to time (one block of 20 steps is 0.3 s here)
    blocks = []
    t_all = time.perf_counter()
    while len(blocks) < 3 or (time.perf_counter() - t_all < args.cpu_seconds and len(blocks) < 50):
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step()
        blocks.append(time.perf_counter() - t0)
    dt = statistics.median(blocks)
    value = B * args.steps / dt
    world = int(os.environ.get("WORLD_SIZE", "1"))
    line = {
        "impl": "reference", "metric": METRIC, "value": round(value, 1), "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 1), "ms_per_step": round(dt / args.steps * 1e3, 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32", "data": "synthetic (keys = split(PRNGKey(0), B), random-policy actions)",
        "config": {"workload": "connector_step_random_agent_autoreset_prw", "grid": G, "agents": N, "envs_per_gpu": B, "envs_total": B, "time_limit": TIME_LIMIT, "generator": "ParallelRandomWalkGenerator",
                   "parallelism": f"OpenMP x{cores} host threads", "burnin_steps": args.burnin},
        "timing": {"what": f"{len(blocks)} blocks of exactly {args.steps} steps, host wall clock, median", "ms_per_block": _stats([b * 1e3 for b in blocks])},
        "cpu_baseline": {"value": round(value, 1), "unit": UNIT, "cores": cores, "kind": "port", "sample": f"{len(blocks)} x {args.steps} steps over {B} envs after {args.burnin} burn-in steps (rank 0 only; the CPU arm does not scale with --gpus)"},
        "e2e": {"value": round(value, 1), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=500, help="timed steps: exactly this many, in one window")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs", type=int, default=ENVS_PER_GPU, help="envs per GPU")
    ap.add_argument("--burnin", type=int, default=160, help="untimed steps after reset() so that episode ends are desynchronised")
    ap.add_argument("--chunk", type=int, default=20, help="env steps per rollout call (the reference's n_steps)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-secondary", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs (rank 0's envs, a fixed sample of at most "
                    f"{DUMP_ENVS}) to DIR/<name>.npy, to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()

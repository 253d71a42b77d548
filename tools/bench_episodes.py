"""Random-agent evaluation throughput: the episode kernel against today's Connector.step loop.

For each workload (ParallelRandomWalk boards, time_limit 50) it first checks that both arms give the same per-episode
metrics, then times them with CUDA events, alternating the arms in the same run, each window >= --min-ms:
  (a) RandomAgentEvaluator.episode_metrics (State-only reset + episode_warp_kernel), and the episode kernel alone
      on a ready State (engine.connector_episodes_random);
  (b) Connector.reset, then `time_limit` plain Connector.step calls driven by make_random_policy_connector(),
      accumulating the same metrics in torch from each env's first LAST step (after a fresh reset every env has had
      LAST by then, so the loop needs no host synchronisation).
Rates: episodes/s = B / time, env-steps/s = sum(episode_length) / time (the same numerator for every arm).
Prints one JSON line per workload (and writes them to --out when given) with the card name, power limit and max SM
clock read in the same run.

    python tools/bench_episodes.py [--shapes 10x10/5x65536,32x32/16x8192] [--rounds 7] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRICS = ("episode_return", "episode_length", "num_connections", "ratio_connections", "total_path_length")


def gpu_info(index: int) -> dict:
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(index)], capture_output=True, text=True, check=True).stdout
    name, plim, smax = (x.strip() for x in out.strip().split(","))
    return {"gpu": name, "power_limit_w": float(plim), "sm_clock_max_mhz": float(smax)}


def step_loop(rbg, env, policy, keys, time_limit):
    """Arm (b): reset, then `time_limit` Connector.step calls; each env's metrics come from its first LAST step."""
    import torch

    st, _ = env.reset(keys)
    B, N = st.agents.id.shape
    dev = st.grid.device
    ret = torch.zeros((B, N), dtype=torch.float32, device=dev)
    length = torch.zeros(B, dtype=torch.int32, device=dev)
    ncon = torch.zeros(B, dtype=torch.int32, device=dev)
    ratio = torch.zeros(B, dtype=torch.float32, device=dev)
    tpl = torch.zeros(B, dtype=torch.int32, device=dev)
    done = torch.zeros(B, dtype=torch.bool, device=dev)
    for _ in range(time_limit):
        st, ts = env.step(st, policy(st))
        alive = ~done
        ret = torch.where(alive[:, None], ret + ts.reward, ret)
        length += alive.int()
        last = alive & (ts.step_type == 2)
        ncon = torch.where(last, ts.extras["num_connections"], ncon)
        ratio = torch.where(last, ts.extras["ratio_connections"], ratio)
        tpl = torch.where(last, ts.extras["total_path_length"], tpl)
        done |= last
    return dict(episode_return=ret, episode_length=length, num_connections=ncon, ratio_connections=ratio, total_path_length=tpl), done


def window_ms(fn, reps: int) -> float:
    import torch

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / reps


def calibrate(fn, min_ms: float) -> int:
    """Calls per window so that a window lasts >= min_ms (after two warm-up calls)."""
    fn()
    fn()
    reps = 1
    while True:
        t = window_ms(fn, reps) * reps
        if t >= min_ms:
            return reps
        reps = max(reps + 1, int(reps * min_ms * 1.2 / max(t, 1e-3)))


def run_shape(rbg, G: int, N: int, B: int, time_limit: int, rounds: int, min_ms: float, seed: int) -> dict:
    import torch

    gen = rbg.ParallelRandomWalkGenerator(G, N)
    env = rbg.Connector(generator=gen, time_limit=time_limit)
    policy = rbg.make_random_policy_connector()
    ev = rbg.RandomAgentEvaluator(env, B)
    keys = rbg.split(rbg.PRNGKey(seed), B)
    st = gen(keys)

    # ---- the arms must agree before they are timed
    a = ev.episode_metrics(keys)
    b, done = step_loop(rbg, env, policy, keys, time_limit)
    assert bool(done.all()), "an env had no LAST step within time_limit steps of its reset"
    for k in METRICS:
        x, y = a[k], b[k]
        if x.dtype == torch.float32:
            x, y = x.view(torch.int32), y.view(torch.int32)
        assert torch.equal(x, y), f"{k}: the episode kernel and the Connector.step loop disagree"
    env_steps = int(a["episode_length"].to(torch.int64).sum())

    arms = {
        "evaluator": lambda: ev.episode_metrics(keys),
        "kernel": lambda: rbg.engine.connector_episodes_random(st, time_limit=time_limit),
        "step_loop": lambda: step_loop(rbg, env, policy, keys, time_limit),
    }
    reps = {k: calibrate(f, min_ms) for k, f in arms.items()}
    ms = {k: [] for k in arms}
    for _ in range(rounds):  # alternate the arms so that drift and neighbours hit them alike
        for k, f in arms.items():
            ms[k].append(window_ms(f, reps[k]))
    res = {"workload": f"PRW {G}x{G}/{N}", "B": B, "time_limit": time_limit, "env_steps": env_steps, "mean_episode_length": env_steps / B, "rounds": rounds,
           "min_window_ms": min_ms}
    for k in arms:
        med = statistics.median(ms[k])
        res[k] = {"ms_median": med, "ms_min": min(ms[k]), "ms_max": max(ms[k]), "calls_per_window": reps[k],
                  "episodes_per_s": B / (med * 1e-3), "env_steps_per_s": env_steps / (med * 1e-3)}
    res["speedup_evaluator_vs_step_loop"] = res["step_loop"]["ms_median"] / res["evaluator"]["ms_median"]
    res["speedup_kernel_vs_step_loop"] = res["step_loop"]["ms_median"] / res["kernel"]["ms_median"]
    return res


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--shapes", default="10x10/5x65536,32x32/16x8192", help="GxG/NxB,...")
    ap.add_argument("--time-limit", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--min-ms", type=float, default=60.0)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--out", default=None, help="also write the JSON lines here")
    args = ap.parse_args()

    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench_episodes.py needs a CUDA device")
    import __graft_entry__ as ge

    ge.build_library()
    import routing_board_generation_b200 as rbg

    info = gpu_info(torch.cuda.current_device())
    lines = []
    for spec in args.shapes.split(","):
        gg, rest = spec.split("/")
        G = int(gg.split("x")[0])
        N, B = (int(x) for x in rest.split("x"))
        res = run_shape(rbg, G, N, B, args.time_limit, args.rounds, args.min_ms, args.seed)
        res.update(info)
        lines.append(json.dumps(res))
        print(lines[-1], flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()

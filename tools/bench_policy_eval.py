"""Policy evaluation throughput: PolicyEvaluator (one eval-step launch per policy call) against a Connector.step loop,
with --live-only its two modes against each other, and with --cuda-graph its default mode against its CUDA-graph mode.

The policy is "keyed", a pure torch function of the action mask and the action key (agent a takes the
((key0 ^ a * 0x9E3779B9) mod n)-th of its n legal actions), so that every arm computes the same episodes, or "mlp", a
seeded two-layer float32 MLP (G*G -> 128 -> 5) over each agent's observation.grid with an argmax over the legal
actions: a policy whose cost grows with the rows it is given.  For each workload (ParallelRandomWalk boards,
time_limit 50) it first checks that the arms give the same per-episode metrics (for "mlp" it reports whether they do:
a matrix product may round a row differently at another batch size), then times them with CUDA events, alternating
the arms in the same run, each window >= --min-ms:
  (a) PolicyEvaluator.episode_metrics: Connector.reset, then policy -> eval step until no env is live, one host wait
      per step on a count read one step late;
  (b) Connector.reset, then `time_limit` plain Connector.step calls driven by the same policy and action keys, with
      the metrics accumulated in torch from each env's first LAST step (as tools/bench_episodes.py step_loop);
  (c) eval_step_kernel alone: its device time summed over the steps of (a), from the library's kernel timing
      (rbg_kernel_time(RBG_K_EVAL_STEP)), which brackets each launch with an event pair.
With --live-only, (b) is replaced by
  (d) PolicyEvaluator(live_only=True).episode_metrics: the policy sees only the live envs, one host wait per step to
      read their number;
  (e) the live step kernel alone (eval_step_kernel<LIST>), timed as (c) over the steps of (d).
With --cuda-graph, (b) is replaced by
  (f) PolicyEvaluator(cuda_graph=True).episode_metrics: the eager reset copied into static buffers, then one launch of
      the captured loop (split, policy, eval step, loop condition) that runs on the device until no env is live; the
      capture happens in the agreement check, before any timed window.  Its loop iterations are reported.
Policy rows per evaluation (the rows the policy was handed, summed over its calls) are counted for (a) and (d).
Rates: episodes/s = B / time, env-steps/s = sum(episode_length) / time (the same numerator for every arm).
Kernel bandwidth: the bytes one live env-step moves (computed from the shape below) times sum(episode_length), over the
kernel time of (c); a dead env costs its live byte.  DESIGN K2's count for a full Connector.step (3 206 B at 10x10/5,
74 937 B at 32x32/16) is given beside it.  The HBM fraction is against 7.7 TB/s (the HGX B200 data sheet, one GPU).
Prints one JSON line per workload (and writes them to --out when given) with the card name, power limit and max SM
clock read in the same run.

    python tools/bench_policy_eval.py [--shapes 10x10/5x65536,32x32/16x8192] [--policy keyed|mlp] [--live-only | --cuda-graph] [--rounds 7] [--out FILE]
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
HBM_BYTES_PER_S = 7.7e12
K2_BYTES = {(10, 5): 3206, (32, 16): 74937}  # DESIGN K2: one Connector.step, State + TimeStep


def gpu_info(index: int) -> dict:
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(index)], capture_output=True, text=True, check=True).stdout
    name, plim, smax = (x.strip() for x in out.strip().split(","))
    return {"gpu": name, "power_limit_w": float(plim), "sm_clock_max_mhz": float(smax)}


def eval_step_bytes(G: int, N: int) -> int:
    """HBM bytes of one live env-step of eval_step_kernel.  Read: live byte, grid, position + target, action,
    step_count, the record's return and length.  Written: observation, action mask, reward, discount, step_type,
    obs step_count, extras, State step_count and position, the two grid cells of a moved agent (counted for every agent),
    the record's return and length.  The terminal step's extras and live byte (17 B once per episode) are left out."""
    cells = G * G
    read = 1 + 4 * cells + 16 * N + 4 * N + 4 + 4 * N + 4
    write = 4 * N * cells + 5 * N + 4 * N + 4 * N + 1 + 4 + 12 + 4 + 8 * N + 8 * N + 4 * N + 4
    return read + write


def keyed_policy(obs, key):
    import torch

    mask = obs.action_mask
    n = mask.sum(-1)
    a = (torch.arange(mask.shape[1], dtype=torch.int64, device=mask.device) * 0x9E3779B9) & 0xFFFFFFFF
    k0 = key.view(torch.int32)[:, 0].to(torch.int64) & 0xFFFFFFFF
    k = (k0[:, None] ^ a[None, :]) % n
    c = mask.to(torch.int64)  # running count of legal actions (torch.cumsum over 5 entries is a slow scan on the GPU)
    for i in range(1, c.shape[-1]):
        c[..., i] += c[..., i - 1]
    return (mask & (c == (k + 1)[..., None])).to(torch.int8).argmax(-1).to(torch.int32)


class MlpPolicy:
    """A seeded two-layer MLP over each agent's observation.grid (float32), argmax of its logits over the legal actions."""

    def __init__(self, G: int, hidden: int = 128, seed: int = 0):
        import torch

        g = torch.Generator().manual_seed(seed)
        self.w1 = (torch.randn(G * G, hidden, generator=g) / G).cuda()
        self.b1 = (torch.randn(hidden, generator=g) * 0.1).cuda()
        self.w2 = (torch.randn(hidden, 5, generator=g) / hidden ** 0.5).cuda()

    def __call__(self, obs, key):
        import torch

        L, N = obs.grid.shape[:2]
        h = torch.relu(obs.grid.reshape(L * N, -1).to(torch.float32) @ self.w1 + self.b1)
        logits = (h @ self.w2).reshape(L, N, 5).masked_fill(~obs.action_mask, float("-inf"))
        return logits.argmax(-1).to(torch.int32)


class RowCounter:
    """Counts the rows a policy is handed (a host-side shape: no device sync)."""

    def __init__(self, policy):
        self.policy, self.rows, self.calls = policy, 0, 0

    def __call__(self, obs, key):
        self.rows += obs.grid.shape[0]
        self.calls += 1
        return self.policy(obs, key)


def step_loop(rbg, env, policy, keys, time_limit):
    """Arm (b): reset, then `time_limit` Connector.step calls; each env's metrics come from its first LAST step."""
    import torch

    st, ts = env.reset(keys)
    B, N = st.agents.id.shape
    dev = st.grid.device
    ret = torch.zeros((B, N), dtype=torch.float32, device=dev)
    length = torch.zeros(B, dtype=torch.int32, device=dev)
    ncon = torch.zeros(B, dtype=torch.int32, device=dev)
    ratio = torch.zeros(B, dtype=torch.float32, device=dev)
    tpl = torch.zeros(B, dtype=torch.int32, device=dev)
    done = torch.zeros(B, dtype=torch.bool, device=dev)
    chain = rbg.engine.split_each(keys)[:, 1]
    for _ in range(time_limit):
        s = rbg.engine.split_each(chain)
        chain = s[:, 0]
        st, ts = env.step(st, policy(ts.observation, s[:, 1].contiguous()))
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


def kernel_window(rbg, ev, keys, reps: int):
    """(eval_step_kernel ms per evaluation, launches per evaluation) over `reps` evaluations with kernel timing on."""
    rbg._lib.kernel_timing(True)
    try:
        rbg._lib.kernel_time("eval_step")  # drop what was recorded before
        for _ in range(reps):
            ev.episode_metrics(keys)
        n, ms = rbg._lib.kernel_time("eval_step")
    finally:
        rbg._lib.kernel_timing(False)
    return ms / reps, n / reps


def _same(a: dict, b: dict) -> bool:
    import torch

    return all(torch.equal(x.view(torch.int32) if x.dtype == torch.float32 else x, y.view(torch.int32) if y.dtype == torch.float32 else y)
               for x, y in ((a[k], b[k]) for k in METRICS))


def run_shape(rbg, G: int, N: int, B: int, time_limit: int, rounds: int, min_ms: float, seed: int, policy_name: str, live_only: bool,
              cuda_graph: bool = False) -> dict:
    import torch

    policy = keyed_policy if policy_name == "keyed" else MlpPolicy(G, seed=seed)
    env = rbg.Connector(generator=rbg.ParallelRandomWalkGenerator(G, N), time_limit=time_limit)
    ev = rbg.PolicyEvaluator(env, policy, B)
    ev_live = rbg.PolicyEvaluator(env, policy, B, live_only=True)
    ev_graph = rbg.PolicyEvaluator(env, policy, B, cuda_graph=True) if cuda_graph else None
    keys = rbg.split(rbg.PRNGKey(seed), B)

    # ---- the arms must agree before they are timed (a keyed policy: bit for bit)
    count = RowCounter(policy)
    a = rbg.PolicyEvaluator(env, count, B).episode_metrics(keys)
    rows = {"evaluator": count.rows}
    env_steps = int(a["episode_length"].to(torch.int64).sum())
    max_length = int(a["episode_length"].max())
    res = {"workload": f"PRW {G}x{G}/{N}", "policy": policy_name, "B": B, "time_limit": time_limit, "env_steps": env_steps, "mean_episode_length": env_steps / B,
           "max_episode_length": max_length}
    if live_only:
        count = RowCounter(policy)
        b = rbg.PolicyEvaluator(env, count, B, live_only=True).episode_metrics(keys)
        rows["evaluator_live"] = count.rows
        res["env_steps_live"] = int(b["episode_length"].to(torch.int64).sum())
        res["modes_agree_bit_for_bit"] = _same(a, b)
        if policy_name == "keyed":
            assert res["modes_agree_bit_for_bit"], "PolicyEvaluator's two modes disagree"
            assert rows["evaluator_live"] == env_steps, "the live mode handed the policy a row that is not a live env-step"
    elif cuda_graph:
        b = ev_graph.episode_metrics(keys)  # (captures the loop)
        res["loop_iterations"] = ev_graph.loop_steps
        res["modes_agree_bit_for_bit"] = _same(a, b)
        if policy_name == "keyed":
            assert res["modes_agree_bit_for_bit"], "PolicyEvaluator's default and CUDA-graph modes disagree"
            assert res["loop_iterations"] == max_length, "the device-side loop did not stop after the longest episode"
    else:
        b, done = step_loop(rbg, env, policy, keys, time_limit)
        assert bool(done.all()), "an env had no LAST step within time_limit steps of its reset"
        res["modes_agree_bit_for_bit"] = _same(a, b)
        if policy_name == "keyed":
            assert res["modes_agree_bit_for_bit"], "PolicyEvaluator and the Connector.step loop disagree"
    res["policy_rows_per_evaluation"] = rows

    # ---- library launches: the evaluator's, less those of its reset, per step
    torch.cuda.synchronize()
    rbg.launch_count(reset=True)
    env.reset(keys)
    reset_launches = rbg.launch_count(reset=True)
    ev.episode_metrics(keys)
    eval_launches = rbg.launch_count(reset=True)
    _, steps = kernel_window(rbg, ev, keys, 1)
    steps_live = kernel_window(rbg, ev_live, keys, 1)[1] if live_only else None

    arms = {"evaluator": lambda: ev.episode_metrics(keys)}
    if live_only:
        arms["evaluator_live"] = lambda: ev_live.episode_metrics(keys)
    elif cuda_graph:
        arms["evaluator_graph"] = lambda: ev_graph.episode_metrics(keys)
    else:
        arms["step_loop"] = lambda: step_loop(rbg, env, policy, keys, time_limit)
    kernels = {"kernel": ev, "kernel_live": ev_live} if live_only else {"kernel": ev}
    reps = {k: calibrate(f, min_ms) for k, f in arms.items()}
    ms = {k: [] for k in list(arms) + list(kernels)}
    for _ in range(rounds):  # alternate the arms so that drift and neighbours hit them alike
        for k, f in arms.items():
            ms[k].append(window_ms(f, reps[k]))
        for k, e in kernels.items():
            ms[k].append(kernel_window(rbg, e, keys, reps["evaluator"])[0])
    nbytes = eval_step_bytes(G, N)
    res.update({"eval_steps_per_evaluation": steps, "library_launches_per_step": (eval_launches - reset_launches) / steps,
                "reset_launches": reset_launches, "rounds": rounds, "min_window_ms": min_ms})
    if live_only:
        res["live_steps_per_evaluation"] = steps_live
    for k in ms:
        med = statistics.median(ms[k])
        res[k] = {"ms_median": med, "ms_min": min(ms[k]), "ms_max": max(ms[k]), "episodes_per_s": B / (med * 1e-3), "env_steps_per_s": env_steps / (med * 1e-3)}
        if k in reps:
            res[k]["calls_per_window"] = reps[k]
    kms = res["kernel"]["ms_median"]
    res["kernel"].update({"us_per_step": kms * 1e3 / steps, "bytes_per_live_env_step": nbytes, "bytes_per_evaluation": nbytes * env_steps,
                          "achieved_bytes_per_s": nbytes * env_steps / (kms * 1e-3), "hbm_fraction": nbytes * env_steps / (kms * 1e-3) / HBM_BYTES_PER_S})
    if (G, N) in K2_BYTES:
        kb = K2_BYTES[(G, N)]
        res["kernel"].update({"k2_bytes_per_env_step": kb, "hbm_fraction_at_k2_bytes": kb * env_steps / (kms * 1e-3) / HBM_BYTES_PER_S})
    if live_only:
        res["kernel_live"]["us_per_step"] = res["kernel_live"]["ms_median"] * 1e3 / steps_live
        res["speedup_live_vs_default"] = res["evaluator"]["ms_median"] / res["evaluator_live"]["ms_median"]
    elif cuda_graph:
        res["speedup_graph_vs_default"] = res["evaluator"]["ms_median"] / res["evaluator_graph"]["ms_median"]
    else:
        res["speedup_evaluator_vs_step_loop"] = res["step_loop"]["ms_median"] / res["evaluator"]["ms_median"]
    return res


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--shapes", default="10x10/5x65536,32x32/16x8192", help="GxG/NxB,...")
    ap.add_argument("--time-limit", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--min-ms", type=float, default=60.0)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--policy", choices=("keyed", "mlp"), default="keyed")
    ap.add_argument("--live-only", action="store_true", help="time PolicyEvaluator(live_only=True) against the default mode instead of the step loop")
    ap.add_argument("--cuda-graph", action="store_true", help="time PolicyEvaluator(cuda_graph=True) against the default mode instead of the step loop")
    ap.add_argument("--out", default=None, help="also write the JSON lines here")
    args = ap.parse_args()
    if args.live_only and args.cuda_graph:
        raise SystemExit("--live-only and --cuda-graph are two different comparisons: pick one")

    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench_policy_eval.py needs a CUDA device")
    import __graft_entry__ as ge

    ge.build_library()
    import routing_board_generation_b200 as rbg

    info = gpu_info(torch.cuda.current_device())
    lines = []
    for spec in args.shapes.split(","):
        gg, rest = spec.split("/")
        G = int(gg.split("x")[0])
        N, B = (int(x) for x in rest.split("x"))
        res = run_shape(rbg, G, N, B, args.time_limit, args.rounds, args.min_ms, args.seed, args.policy, args.live_only, args.cuda_graph)
        res.update(info)
        lines.append(json.dumps(res))
        print(lines[-1], flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()

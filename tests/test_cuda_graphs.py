"""CUDA graphs: the device-side evaluation loop (rbg_eval_loop_*, engine.EvalLoop, PolicyEvaluator(cuda_graph=True)),
Connector steps captured into torch CUDA graphs and replayed, and the calls the library refuses while a stream is
capturing.  Results are compared bit for bit (integers exactly, float32 by their bits) with the same work done
eagerly.  The argument checks run without a device; everything else needs one (`-m gpu`)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from test_policy_eval import GENS, METRICS, POLICIES, _keys, _np, _state_np, _ts_np, keyed_torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge

    ge.build_library()
    import routing_board_generation_b200 as pkg

    return pkg._lib.load()


# ------------------------------------------------------------------ no device
def test_eval_loop_kernel_id_and_symbols_match_header():
    import routing_board_generation_b200 as pkg

    with open(os.path.join(ROOT, "include", "rbg_b200.h")) as f:
        src = re.sub(r"/\*.*?\*/", "", f.read(), flags=re.S)
    L = pkg._lib
    assert L.KERNELS["eval_loop"] == int(re.search(r"#define RBG_K_EVAL_LOOP (\d+)", src).group(1))
    for name in ("rbg_eval_loop_create", "rbg_eval_loop_condition", "rbg_eval_loop_finalize", "rbg_eval_loop_launch", "rbg_eval_loop_destroy"):
        params = re.search(rf"int {name}\((.*?)\);", src, flags=re.S).group(1).split(",")
        assert len(L.SYMBOLS[name][1]) == len(params), name


def test_eval_loop_argument_errors(lib):
    """NULL or bad arguments return -1 with a message before any CUDA call (no device needed)."""
    h, c = C.c_void_p(), C.c_uint64()
    assert lib.rbg_eval_loop_create(None, C.byref(c)) == -1 and b"NULL" in lib.rbg_last_error()
    assert lib.rbg_eval_loop_create(C.byref(h), None) == -1 and b"NULL" in lib.rbg_last_error()
    buf = (C.c_int32 * 2)()
    p = C.cast(buf, C.c_void_p)
    assert lib.rbg_eval_loop_condition(1, None, p, 5, None) == -1 and b"NULL" in lib.rbg_last_error()
    assert lib.rbg_eval_loop_condition(1, p, None, 5, None) == -1 and b"NULL" in lib.rbg_last_error()
    assert lib.rbg_eval_loop_condition(1, p, p, 0, None) == -1 and b"max_steps" in lib.rbg_last_error()
    assert lib.rbg_eval_loop_finalize(None, p) == -1 and b"NULL" in lib.rbg_last_error()
    assert lib.rbg_eval_loop_finalize(p, None) == -1 and b"NULL" in lib.rbg_last_error()
    assert lib.rbg_eval_loop_launch(None, None) == -1 and b"NULL" in lib.rbg_last_error()
    assert lib.rbg_eval_loop_destroy(None) == -1 and b"NULL" in lib.rbg_last_error()


def test_cuda_graph_with_live_only_raises():
    import routing_board_generation_b200 as rbg

    env = rbg.Connector(generator=rbg.ParallelRandomWalkGenerator(10, 5))
    with pytest.raises(ValueError, match="static batch shape"):
        rbg.PolicyEvaluator(env, keyed_torch, 64, live_only=True, cuda_graph=True)


# ----------------------------------------------------- the evaluator, graph mode
def _graph_vs_eager(rbg, env, policy, keys, where):
    """PolicyEvaluator(cuda_graph=True) against the default mode on the same keys: every metric bit for bit, and the
    loop's iterations = the longest episode (the eager loop's live steps)."""
    pt = POLICIES[policy][1] if isinstance(policy, str) else policy
    ref = rbg.PolicyEvaluator(env, pt, keys.shape[0]).episode_metrics(keys)
    ev = rbg.PolicyEvaluator(env, pt, keys.shape[0], cuda_graph=True)
    got = ev.episode_metrics(keys)
    for k in METRICS:
        a, b = _np(got[k]), _np(ref[k])
        assert a.shape == b.shape and np.array_equal(a.view(np.uint32) if a.dtype == np.float32 else a, b.view(np.uint32) if b.dtype == np.float32 else b), f"{k} {where}"
    assert ev.loop_steps == int(ref["episode_length"].max()), where
    ev.close()
    return ref


@pytest.mark.gpu
@pytest.mark.parametrize("policy", ["keyed", "greedy"])
@pytest.mark.parametrize("kind", ["parallel_random_walk", "uniform"])
@pytest.mark.parametrize("G,N", [(10, 5), (7, 3), (40, 1)])  # 7 x 7: cells % 4 != 0; 40 x 40 / 1: > 48 KB of shared memory
@pytest.mark.parametrize("time_limit", [1, 2, 50])
def test_graph_evaluator_matches_eager(rbg, orc, policy, kind, G, N, time_limit):
    B = 1024 if G < 32 else 512
    keys, _ = _keys(rbg, orc, G * 100 + N + time_limit, B)
    env = rbg.Connector(generator=getattr(rbg, GENS[kind])(G, N), time_limit=time_limit)
    ref = _graph_vs_eager(rbg, env, policy, keys, f"({policy} {kind} {G}x{G}/{N} time_limit {time_limit})")
    assert int(ref["episode_length"].max()) <= time_limit


@pytest.mark.gpu
@pytest.mark.parametrize("policy", ["keyed", "greedy"])
@pytest.mark.parametrize("kind", ["seed_extension", "sequential_random_walk"])
def test_graph_evaluator_other_generators(rbg, orc, policy, kind):
    keys, _ = _keys(rbg, orc, 77, 1500)
    _graph_vs_eager(rbg, rbg.Connector(generator=getattr(rbg, GENS[kind])(10, 5), time_limit=50), policy, keys, kind)


@pytest.mark.gpu
def test_graph_evaluator_dataset_and_user_generator(rbg, orc):
    import torch

    gen = rbg.BoardDatasetGeneratorJAX(10, 5, board_name="offline_parallel_rw", number_of_boards=37)
    keys, _ = _keys(rbg, orc, 78, 1200)
    _graph_vs_eager(rbg, rbg.Connector(generator=gen, time_limit=30), "keyed", keys, "dataset generator")

    G, N = 6, 2

    class RowsGenerator(rbg.Generator):
        def __call__(self, key):
            k = rbg.engine.as_keys(key)[0].view(torch.int32).to(torch.int64) & 0xFFFFFFFF
            Bk = k.shape[0]
            c0, c1 = (k[:, 0] % G).int(), (k[:, 1] % G).int()
            start = torch.stack([torch.stack([torch.zeros_like(c0), c0], -1), torch.stack([torch.full_like(c1, 2), c1], -1)], 1)
            target = torch.stack([torch.stack([torch.ones_like(c0) * (G - 1), c1], -1), torch.stack([torch.full_like(c1, 4), c0], -1)], 1)
            grid = torch.zeros((Bk, G, G), dtype=torch.int32, device=k.device)
            b = torch.arange(Bk, device=k.device)
            for i in range(N):
                grid[b, start[:, i, 0].long(), start[:, i, 1].long()] = 2 + 3 * i
                grid[b, target[:, i, 0].long(), target[:, i, 1].long()] = 3 + 3 * i
            newkey = rbg.engine.split_each(rbg.engine.as_keys(key)[0], 2)[:, 0].contiguous()
            return rbg.State(key=newkey, grid=grid, step_count=torch.zeros(Bk, dtype=torch.int32, device=k.device),
                             agents=rbg.Agent(id=torch.arange(N, dtype=torch.int32, device=k.device).expand(Bk, N).contiguous(), start=start.int().contiguous(),
                                              target=target.int().contiguous(), position=start.int().contiguous()))

    keys, _ = _keys(rbg, orc, 79, 500)
    _graph_vs_eager(rbg, rbg.VmapAutoResetWrapper(rbg.Connector(generator=RowsGenerator(G, N), time_limit=12)), "keyed", keys, "user generator")


@pytest.mark.gpu
@pytest.mark.parametrize("wrapped", [False, True])
def test_graph_evaluator_multi_to_single(rbg, orc, wrapped):
    keys, _ = _keys(rbg, orc, 31, 2048)
    env = rbg.Connector(generator=rbg.ParallelRandomWalkGenerator(10, 5), time_limit=50)
    _graph_vs_eager(rbg, rbg.VmapAutoResetWrapper(rbg.MultiToSingleWrapper(env)) if wrapped else env, "keyed", keys, f"MultiToSingleWrapper {wrapped}")


@pytest.mark.gpu
@pytest.mark.parametrize("G,N,B", [(10, 5, 65536), (32, 16, 8192)])
def test_graph_evaluator_full_size(rbg, orc, G, N, B):
    keys, _ = _keys(rbg, orc, 2, B)
    env = rbg.Connector(generator=rbg.ParallelRandomWalkGenerator(G, N), time_limit=50)
    _graph_vs_eager(rbg, env, "keyed", keys, f"({G}x{G}/{N} x {B})")


@pytest.mark.gpu
def test_graph_evaluator_reuse_and_rebuild(rbg, orc):
    """Two run_evaluation calls replay one graph; a new batch size captures a new one; both agree with the default mode."""
    import torch

    env = rbg.MultiToSingleWrapper(rbg.Connector(generator=rbg.UniformRandomGenerator(10, 5), time_limit=50))
    eager = rbg.PolicyEvaluator(env, POLICIES["greedy"][1], 3000)
    ev = rbg.PolicyEvaluator(env, POLICIES["greedy"][1], 3000, cuda_graph=True)
    for seed in (4, 5):
        got, ref = ev.run_evaluation(rbg.PRNGKey(seed)), eager.run_evaluation(rbg.PRNGKey(seed))
        for k in METRICS:
            assert torch.equal(got[k], ref[k]), (seed, k)
    first = ev._captured
    assert first.B == 3000
    keys = rbg.split(rbg.PRNGKey(6), 700)
    got, ref = ev.episode_metrics(keys), eager.episode_metrics(keys)
    assert ev._captured is not first and ev._captured.B == 700
    for k in METRICS:
        assert torch.equal(got[k], ref[k]), k
    ev.close()
    assert ev._captured is None


# ------------------------------------------------------------ captured steps
def _leaves(ts, act=None):
    d = _ts_np(ts)
    if act is not None:
        d["action"] = _np(act)
    return d


@pytest.mark.gpu
@pytest.mark.parametrize("random_policy", [False, True])
@pytest.mark.parametrize("k", [1, 2, 3])
@pytest.mark.parametrize("time_limit", [1, 2, 3])
@pytest.mark.parametrize("kind", ["parallel_random_walk", "uniform", "seed_extension", "sequential_random_walk", "dataset"])
def test_captured_autoreset_steps_match_eager(rbg, orc, kind, time_limit, k, random_policy):
    """After one eager step, k auto-reset steps (VmapAutoResetWrapper.step(inplace=True) on random_actions, or
    step_random) are captured into one graph and replayed 3 times, each replay followed by an eager step; every TimeStep
    (and sampled action) and the final State equal the same sequence run eagerly on a second env of the same
    generator.  time_limit 1 to 3: envs finish in consecutive steps, so the next-episode cache misses and the
    synchronous reset path runs inside the graph."""
    import torch

    G, N, B, R = 10, 5, 512, 3
    if kind == "dataset":
        gen = rbg.BoardDatasetGeneratorJAX(G, N, board_name="offline_parallel_rw", number_of_boards=37)
    else:
        gen = getattr(rbg, GENS[kind])(G, N)
    env_g = rbg.VmapAutoResetWrapper(rbg.Connector(generator=gen, time_limit=time_limit))
    env_e = rbg.VmapAutoResetWrapper(rbg.Connector(generator=gen, time_limit=time_limit))
    keys, _ = _keys(rbg, orc, 1000 + time_limit * 10 + k, B)
    st_g, _ = env_g.reset(keys)
    st_e, _ = env_e.reset(keys)

    def step(env, st):
        if random_policy:
            _, ts, act = env.step_random(st, inplace=True)
            return ts, act
        act = rbg.engine.random_actions(st)
        _, ts = env.step(st, act, inplace=True)
        return ts, act

    got, ref = [], []
    got.append(_leaves(*step(env_g, st_g)))
    ref.append(_leaves(*step(env_e, st_e)))
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        outs = [step(env_g, st_g) for _ in range(k)]
    for _ in range(R):
        graph.replay()
        got += [_leaves(*o) for o in outs]
        ref += [_leaves(*step(env_e, st_e)) for _ in range(k)]
        got.append(_leaves(*step(env_g, st_g)))
        ref.append(_leaves(*step(env_e, st_e)))
    assert len(got) == len(ref) == 1 + R * (k + 1)
    for i, (a, b) in enumerate(zip(got, ref)):
        for name in b:
            assert np.array_equal(a[name], b[name]), f"step {i}: {name}"
    sg, se = _state_np(st_g), _state_np(st_e)
    for name in se:
        assert np.array_equal(sg[name], se[name]), f"final state.{name}"


@pytest.mark.gpu
def test_captured_reset_and_eval_step(rbg, orc):
    """Connector.reset (a kernel generator) and one evaluation step captured together; a replay on new keys equals the
    eager calls."""
    import torch

    G, N, B = 10, 5, 700
    env = rbg.Connector(generator=rbg.ParallelRandomWalkGenerator(G, N), time_limit=50)
    keys = rbg.split(rbg.PRNGKey(1), B)
    act = torch.zeros((B, N), dtype=torch.int32, device="cuda")

    def run():
        st, ts = rbg.engine.connector_reset("parallel_random_walk", keys, G, N)
        m = {k: torch.zeros((B, N) if k == "episode_return" else (B,), dtype=torch.float32 if k in ("episode_return", "ratio_connections") else torch.int32, device="cuda")
             for k in METRICS}
        live = torch.ones(B, dtype=torch.uint8, device="cuda")
        count = torch.full((1,), B, dtype=torch.int32, device="cuda")
        act.copy_(rbg.engine.random_actions(st))
        rbg.engine.connector_eval_step(st, act, live, count, m, ts)
        return st, ts, m

    run()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        st_g, ts_g, m_g = run()
    keys.copy_(rbg.split(rbg.PRNGKey(2), B))
    graph.replay()
    st_e, ts_e, m_e = run()
    for a, b in ((_state_np(st_g), _state_np(st_e)), (_ts_np(ts_g), _ts_np(ts_e)), ({k: _np(v) for k, v in m_g.items()}, {k: _np(v) for k, v in m_e.items()})):
        for name in b:
            assert np.array_equal(a[name], b[name]), name


# ------------------------------------------------------------------ refusals
def _oracle_step_ok(rbg, orc, env, st, kind, time_limit):
    """An eager auto-reset step of `st` equals the oracle's."""
    s0 = _state_np(st)
    act = orc.random_actions_batch(s0)
    rs, rts = orc.connector_step_batch(s0, act, time_limit=time_limit, autoreset_kind=kind)
    st2, ts2 = env.step(st, rbg.engine.as_tensor(act))
    got_s, got_t = _state_np(st2), _ts_np(ts2)
    for name in rs:
        assert np.array_equal(got_s[name], rs[name]), f"state.{name}"
    for name in ("obs", "action_mask", "reward", "discount", "step_type"):
        assert np.array_equal(got_t[name], rts[name]), f"timestep.{name}"


@pytest.mark.gpu
def test_refusals_inside_a_capture(rbg, orc):
    import torch

    G, N, B, TL = 10, 5, 256, 3
    kind = "parallel_random_walk"
    keys, _ = _keys(rbg, orc, 5, B)
    conn = rbg.Connector(generator=rbg.ParallelRandomWalkGenerator(G, N), time_limit=TL)
    env = rbg.VmapAutoResetWrapper(conn)

    def refused(fn, exc, match):
        graph = torch.cuda.CUDAGraph()
        with pytest.raises(exc, match=match):
            with torch.cuda.graph(graph):
                fn()
        del graph
        torch.cuda.synchronize()

    # the first use of an auto-reset workspace (Python refuses before allocating it)
    st, _ = env.reset(keys)
    refused(lambda: env.step_random(st, inplace=True), RuntimeError, "step once outside the capture")
    _oracle_step_ok(rbg, orc, env, st, kind, TL)
    # a workspace that the library has forgotten: its re-adoption
    st, _ = env.reset(keys)
    ws = rbg.engine._workspace(B, G, N, conn)
    rbg._lib.check(rbg._lib.load().rbg_workspace_release(ws.data_ptr()))
    refused(lambda: env.step_random(st, inplace=True), rbg.RbgError, "step once outside the capture")
    _oracle_step_ok(rbg, orc, env, st, kind, TL)
    # any launch while kernel timing is on
    rbg._lib.kernel_timing(True)
    try:
        refused(lambda: env.step_random(st, inplace=True), rbg.RbgError, "kernel timing")
        refused(lambda: rbg.engine.split_each(keys), rbg.RbgError, "kernel timing")
    finally:
        rbg._lib.kernel_timing(False)
        for name in rbg._lib.KERNELS:
            rbg._lib.kernel_time(name)
    _oracle_step_ok(rbg, orc, env, st, kind, TL)
    # the fused rollout
    refused(lambda: env.rollout_random(st, 4), rbg.RbgError, "rollout_random")
    _oracle_step_ok(rbg, orc, env, st, kind, TL)

    # auto-reset with a user Generator selects the finished envs on the host
    class Wrapped(rbg.Generator):
        def __call__(self, key):
            return rbg.engine.generator_state("uniform", rbg.engine.as_keys(key)[0], G, N)

    uenv = rbg.VmapAutoResetWrapper(rbg.Connector(generator=Wrapped(G, N), time_limit=TL))
    ust, _ = uenv.reset(keys)
    refused(lambda: uenv.step_random(ust, inplace=True), RuntimeError, "user Generator")
    _oracle_step_ok(rbg, orc, env, st, kind, TL)

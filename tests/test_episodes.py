"""Random-agent episodes on the device (rbg_connector_episodes_random, engine.connector_episodes_random,
RandomAgentEvaluator) against the CPU oracle stepped until each env's first LAST step, and against the existing GPU
Connector.step path.  Integers exactly, float32 returns and ratios by their bits.  Every test but the header check
needs a CUDA device (`-m gpu`)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
METRICS = ("episode_return", "episode_length", "num_connections", "ratio_connections", "total_path_length")
STATE_FIELDS = ("grid", "step_count", "agent_id", "start", "target", "position", "key")
GENS = {"parallel_random_walk": "ParallelRandomWalkGenerator", "uniform": "UniformRandomGenerator", "seed_extension": "SeedExtensionGenerator",
        "sequential_random_walk": "SequentialRandomWalkGenerator"}


def test_episode_metrics_struct_matches_header():
    """ctypes' rbg_episode_metrics has the header's fields, in its order, all pointers."""
    import routing_board_generation_b200 as pkg

    with open(os.path.join(ROOT, "include", "rbg_b200.h")) as f:
        src = re.sub(r"/\*.*?\*/", "", f.read(), flags=re.S)
    body = re.search(r"typedef struct rbg_episode_metrics \{(.*?)\} rbg_episode_metrics;", src, flags=re.S).group(1)
    fields = re.findall(r"^\s*\w+\s*\*\s*(\w+)\s*;", body, flags=re.M)
    assert fields == list(METRICS)
    L = pkg._lib
    assert [f[0] for f in L.rbg_episode_metrics._fields_] == fields
    assert C.sizeof(L.rbg_episode_metrics) == len(fields) * C.sizeof(C.c_void_p)
    assert L.KERNELS["episodes"] == int(re.search(r"#define RBG_K_EPISODES (\d+)", src).group(1))


# ------------------------------------------------------------------ helpers
def _np(t):
    import torch

    if t.dtype == torch.uint32:
        return t.view(torch.int32).cpu().numpy().view(np.uint32)
    return t.cpu().numpy()


def _state_np(st):
    a = st.agents
    return dict(grid=_np(st.grid), step_count=_np(st.step_count), agent_id=_np(a.id), start=_np(a.start), target=_np(a.target), position=_np(a.position), key=_np(st.key))


def _keys(rbg, orc, seed, B):
    k = rbg.split(rbg.PRNGKey(seed), B)
    ref = orc.split(orc.PRNGKey(seed), B)
    assert np.array_equal(_np(k), ref)
    return k, ref


def oracle_episodes(orc, st, time_limit, timestep_reward=-0.03, connected_reward=0.1):
    """The oracle's plain Connector.step (autoreset_kind=-1) under its random policy, each env stepped until its first
    LAST step; returns in float32, added in step order.  -> (metrics, State after each env's terminal step)."""
    st = {k: v.copy() for k, v in st.items()}
    B, N = st["target"].shape[:2]
    m = dict(episode_return=np.zeros((B, N), np.float32), episode_length=np.zeros(B, np.int32), num_connections=np.zeros(B, np.int32),
             ratio_connections=np.zeros(B, np.float32), total_path_length=np.zeros(B, np.int32))
    alive = np.arange(B)
    while alive.size:
        sub = {k: v[alive] for k, v in st.items()}
        nsub, ts = orc.connector_step_batch(sub, orc.random_actions_batch(sub), time_limit=time_limit, timestep_reward=timestep_reward,
                                            connected_reward=connected_reward, autoreset_kind=-1)
        m["episode_return"][alive] = m["episode_return"][alive] + ts["reward"]
        m["episode_length"][alive] += 1
        for k in st:
            st[k][alive] = nsub[k]
        last = ts["step_type"] == 2
        for k in ("num_connections", "ratio_connections", "total_path_length"):
            m[k][alive[last]] = ts[k][last]
        alive = alive[~last]
    return m, st


def _assert_metrics(got, ref, where=""):
    for k in METRICS:
        g, r = _np(got[k]), ref[k]
        if r.dtype == np.float32:
            g, r = g.view(np.uint32), r.view(np.uint32)
        assert g.shape == r.shape and np.array_equal(g, r), f"{k} differs {where}"


def _assert_state(st, ref, where=""):
    got = _state_np(st)
    for k in STATE_FIELDS:
        assert np.array_equal(got[k], ref[k]), f"final_state.{k} differs {where}"


def _check_against_oracle(rbg, orc, st, time_limit, where=""):
    ref, rfin = oracle_episodes(orc, _state_np(st), time_limit)
    got = rbg.engine.connector_episodes_random(st, time_limit=time_limit, final_state=True)
    _assert_metrics(got, ref, where)
    _assert_state(got["final_state"], rfin, where)
    return ref


def _generator_state(rbg, orc, kind, G, N, B, seed):
    keys, kref = _keys(rbg, orc, seed, B)
    st = getattr(rbg, GENS[kind])(G, N)(keys)
    assert np.array_equal(_np(st.grid), orc.state_batch(kind, kref, G, N)["grid"])
    return st


# ------------------------------------------------------------ oracle parity
SHAPES = [(5, 3), (10, 5), (7, 6), (32, 16), (40, 32), (2, 1)]  # G x G / N; 7 x 7 and 5 x 5: cells % 4 != 0
# few agents on a big board: a CTA's grids need more than 48 KB of shared memory (40 x 40 / 1: 200 KB)
BIG_SMEM_SHAPES = [(40, 1), (28, 2), (40, 4), (20, 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["parallel_random_walk", "uniform"])
@pytest.mark.parametrize("G,N", SHAPES)
@pytest.mark.parametrize("time_limit", [1, 7, 50])
def test_episodes_match_oracle(rbg, orc, kind, G, N, time_limit):
    B = 2048 if G < 32 else 512
    st = _generator_state(rbg, orc, kind, G, N, B, seed=G * 100 + N + time_limit)
    ref = _check_against_oracle(rbg, orc, st, time_limit, f"({kind} {G}x{G}/{N} time_limit {time_limit})")
    assert int(ref["episode_length"].max()) <= time_limit


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["parallel_random_walk", "uniform"])
@pytest.mark.parametrize("G,N", BIG_SMEM_SHAPES)
def test_episodes_big_shared_memory_shapes(rbg, orc, kind, G, N):
    st = _generator_state(rbg, orc, kind, G, N, 3000, seed=G + N)
    _check_against_oracle(rbg, orc, st, 50, f"({kind} {G}x{G}/{N})")


@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, 31, 33, 2048])
@pytest.mark.parametrize("G,N", [(10, 5), (7, 6), (40, 32)])
def test_episodes_batch_sizes(rbg, orc, B, G, N):
    """Ragged warps and groups: a batch that does not fill a warp, one env more than a warp of 1-lane groups, ..."""
    st = _generator_state(rbg, orc, "parallel_random_walk", G, N, B, seed=B + G)
    _check_against_oracle(rbg, orc, st, 50, f"(B={B} {G}x{G}/{N})")


@pytest.mark.gpu
@pytest.mark.parametrize("kind,G,N", [("seed_extension", 10, 5), ("sequential_random_walk", 10, 5), ("seed_extension", 7, 3), ("sequential_random_walk", 16, 8)])
def test_other_generators_through_the_evaluator(rbg, orc, kind, G, N):
    B = 1500
    keys, kref = _keys(rbg, orc, 77, B)
    env = rbg.Connector(generator=getattr(rbg, GENS[kind])(G, N), time_limit=50)
    got = rbg.RandomAgentEvaluator(env, B).episode_metrics(keys)
    ref, _ = oracle_episodes(orc, orc.state_batch(kind, kref, G, N), 50)
    _assert_metrics(got, ref, kind)


@pytest.mark.gpu
def test_dataset_generator_through_the_evaluator(rbg, orc):
    G, N, B = 10, 5, 1200
    gen = rbg.BoardDatasetGeneratorJAX(G, N, board_name="offline_parallel_rw", number_of_boards=37)
    keys, kref = _keys(rbg, orc, 78, B)
    got = rbg.RandomAgentEvaluator(rbg.Connector(generator=gen, time_limit=30), B).episode_metrics(keys)
    ref, _ = oracle_episodes(orc, orc.dataset_state_batch(kref, G, N, _np(gen.heads), _np(gen.targets)), 30)
    _assert_metrics(got, ref, "dataset generator")


@pytest.mark.gpu
def test_user_generator_through_the_evaluator(rbg, orc):
    """Any `Generator` subclass: its own __call__ builds the reset State (here: two wires on fixed rows)."""
    import torch

    G, N, B = 6, 2, 500

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

    gen = RowsGenerator(G, N)
    keys, _ = _keys(rbg, orc, 79, B)
    got = rbg.RandomAgentEvaluator(rbg.VmapAutoResetWrapper(rbg.Connector(generator=gen, time_limit=12)), B).episode_metrics(keys)
    ref, _ = oracle_episodes(orc, _state_np(gen(keys)), 12)
    _assert_metrics(got, ref, "user generator")


@pytest.mark.gpu
@pytest.mark.parametrize("G,N,steps,time_limit", [(10, 5, 4, 50), (10, 5, 9, 7), (7, 6, 3, 5), (32, 16, 6, 20)])
def test_mid_episode_starts(rbg, orc, G, N, steps, time_limit):
    """States after a few random-policy Connector.step calls: PATH cells on the grid, connected agents, and (past the
    time limit) step_count >= time_limit, whose episode is one step long."""
    B = 1024
    st = _generator_state(rbg, orc, "parallel_random_walk", G, N, B, seed=5 + steps)
    env, policy = rbg.Connector(generator=rbg.ParallelRandomWalkGenerator(G, N), time_limit=time_limit), rbg.make_random_policy_connector()
    for _ in range(steps):
        st, _ = env.step(st, policy(st))
    ref = _check_against_oracle(rbg, orc, st, time_limit, f"after {steps} steps")
    past = _np(st.step_count) >= time_limit
    assert np.all(ref["episode_length"][past] == 1)
    if steps > time_limit:
        assert past.any()


@pytest.mark.gpu
@pytest.mark.parametrize("G,N,B", [(10, 5, 65536), (32, 16, 8192)])
def test_full_size_matches_oracle(rbg, orc, G, N, B):
    st = _generator_state(rbg, orc, "parallel_random_walk", G, N, B, seed=2)
    _check_against_oracle(rbg, orc, st, 50, f"({G}x{G}/{N} x {B})")


@pytest.mark.gpu
def test_agrees_with_connector_step_loop(rbg, orc):
    """The metrics equal those taken from each env's first LAST in a plain Connector.step loop on the GPU."""
    import torch

    G, N, B, TL = 10, 5, 4096, 50
    keys, _ = _keys(rbg, orc, 9, B)
    env, policy = rbg.Connector(generator=rbg.ParallelRandomWalkGenerator(G, N), time_limit=TL), rbg.make_random_policy_connector()
    st, _ = env.reset(keys)
    got = rbg.engine.connector_episodes_random(st, time_limit=TL)
    dev = st.grid.device
    ret = torch.zeros((B, N), dtype=torch.float32, device=dev)
    length = torch.zeros(B, dtype=torch.int32, device=dev)
    extras = {k: torch.zeros(B, dtype=d, device=dev) for k, d in (("num_connections", torch.int32), ("ratio_connections", torch.float32), ("total_path_length", torch.int32))}
    done = torch.zeros(B, dtype=torch.bool, device=dev)
    while not bool(done.all()):
        st, ts = env.step(st, policy(st))
        alive = ~done
        ret = torch.where(alive[:, None], ret + ts.reward, ret)
        length += alive.int()
        last = alive & (ts.step_type == 2)
        for k in extras:
            extras[k] = torch.where(last, ts.extras[k], extras[k])
        done |= last
    ref = dict(episode_return=_np(ret), episode_length=_np(length), **{k: _np(v) for k, v in extras.items()})
    _assert_metrics(got, ref, "against the Connector.step loop")


@pytest.mark.gpu
def test_start_is_read_only_and_empty_batch(rbg, orc):
    import torch

    st = _generator_state(rbg, orc, "uniform", 10, 5, 3000, seed=11)
    before = _state_np(st)
    rbg.engine.connector_episodes_random(st, time_limit=50, final_state=True)
    torch.cuda.synchronize()
    for k in STATE_FIELDS:
        assert np.array_equal(_state_np(st)[k], before[k]), f"start.{k} was written"
    lib = rbg._lib.load()
    params = rbg._lib.rbg_env_params(50, -0.03, 0.1, -1)
    assert lib.rbg_connector_episodes_random(None, 0, 10, 5, C.byref(params), None, None, None) == 0


@pytest.mark.gpu
def test_argument_errors(rbg, orc):
    import torch

    lib = rbg._lib.load()
    B, G, N = 8, 10, 5
    st = _generator_state(rbg, orc, "parallel_random_walk", G, N, B, seed=1)
    s = rbg.engine._state_struct(st)
    dev = st.grid.device
    bufs = [torch.empty((B, N), dtype=torch.float32, device=dev)] + [torch.empty(B, dtype=d, device=dev) for d in (torch.int32, torch.int32, torch.float32, torch.int32)]
    m = rbg._lib.rbg_episode_metrics(*(b.data_ptr() for b in bufs))
    ok = rbg._lib.rbg_env_params(50, -0.03, 0.1, -1)
    call = lambda s_=C.byref(s), Bx=B, Gx=G, Nx=N, p=C.byref(ok), m_=C.byref(m), f=None: lib.rbg_connector_episodes_random(s_, Bx, Gx, Nx, p, m_, f, None)

    assert call() == 0
    assert call(s_=None) == -1 and b"NULL" in lib.rbg_last_error()
    assert call(p=None) == -1 and b"params" in lib.rbg_last_error()
    assert call(m_=None) == -1 and b"NULL" in lib.rbg_last_error()
    for i in range(5):
        bad = rbg._lib.rbg_episode_metrics(*(0 if j == i else b.data_ptr() for j, b in enumerate(bufs)))
        assert call(m_=C.byref(bad)) == -1 and b"NULL" in lib.rbg_last_error()
    fin = rbg.engine._state_struct(rbg.engine.alloc_state(B, G, N))
    fin.key = None
    assert call(f=C.byref(fin)) == -1 and b"final_state" in lib.rbg_last_error()
    assert call(Gx=41) == -1 and b"grid size" in lib.rbg_last_error()
    assert call(Gx=1) == -1 and b"grid size" in lib.rbg_last_error()
    assert call(Nx=0) == -1 and b"num_agents" in lib.rbg_last_error()
    assert call(Nx=33) == -1 and b"num_agents" in lib.rbg_last_error()
    assert call(Bx=-1) == -1
    for kind in (0, 1, 3):
        ar = rbg._lib.rbg_env_params(50, -0.03, 0.1, kind)
        assert call(p=C.byref(ar)) == -1 and b"autoreset_kind" in lib.rbg_last_error()
    torch.cuda.synchronize()


# ---------------------------------------------------------------- evaluator
@pytest.mark.gpu
def test_evaluator_multi_to_single_sums_agents(rbg, orc):
    G, N, B = 10, 5, 2048
    keys, kref = _keys(rbg, orc, 31, B)
    env = rbg.Connector(generator=rbg.ParallelRandomWalkGenerator(G, N), time_limit=50)
    single = rbg.RandomAgentEvaluator(rbg.VmapAutoResetWrapper(rbg.MultiToSingleWrapper(env)), B).episode_metrics(keys)
    multi = rbg.RandomAgentEvaluator(env, B).episode_metrics(keys)
    ref, _ = oracle_episodes(orc, orc.state_batch("parallel_random_walk", kref, G, N), 50)
    _assert_metrics(multi, ref)
    assert tuple(single["episode_return"].shape) == (B,)
    np.testing.assert_allclose(_np(single["episode_return"]), ref["episode_return"].astype(np.float64).sum(-1), rtol=1e-5, atol=1e-5)
    for k in METRICS[1:]:
        assert np.array_equal(_np(single[k]), ref[k])


@pytest.mark.gpu
def test_evaluator_run_evaluation_is_the_mean(rbg):
    import torch

    B = 3000
    ev = rbg.RandomAgentEvaluator(rbg.MultiToSingleWrapper(rbg.Connector(generator=rbg.UniformRandomGenerator(10, 5), time_limit=50)), B)
    key = rbg.PRNGKey(4)
    means = ev.run_evaluation(key)
    per = ev.episode_metrics(rbg.split(key, B))
    assert sorted(means) == sorted(METRICS)
    for k in METRICS:
        assert means[k].dim() == 0
        assert torch.equal(means[k], per[k].to(torch.float32).mean(dim=0)), k
    assert 1.0 <= float(means["episode_length"]) <= 50.0


@pytest.mark.gpu
def test_evaluator_single_key_is_unbatched(rbg, orc):
    G, N = 10, 5
    env = rbg.Connector(generator=rbg.ParallelRandomWalkGenerator(G, N), time_limit=50)
    ev = rbg.RandomAgentEvaluator(env, 1)
    key = rbg.PRNGKey(6)
    one = ev.episode_metrics(key)
    assert tuple(one["episode_return"].shape) == (N,)
    for k in METRICS[1:]:
        assert one[k].dim() == 0
    ref, _ = oracle_episodes(orc, orc.state_batch("parallel_random_walk", orc.PRNGKey(6)[None], G, N), 50)
    _assert_metrics({k: v[None] for k, v in one.items()}, ref, "single key")


@pytest.mark.gpu
def test_evaluator_applies_a_linear_reward_aggregator(rbg, orc):
    """MultiToSingleWrapper(reward_aggregator=torch.mean): the mean of the per-agent returns; a non-linear aggregator is refused."""
    import torch

    G, N, B = 10, 5, 1024
    keys, _ = _keys(rbg, orc, 32, B)
    env = rbg.Connector(generator=rbg.ParallelRandomWalkGenerator(G, N), time_limit=50)
    per_agent = rbg.RandomAgentEvaluator(env, B).episode_metrics(keys)["episode_return"]
    mean = rbg.RandomAgentEvaluator(rbg.MultiToSingleWrapper(env, reward_aggregator=torch.mean), B).episode_metrics(keys)["episode_return"]
    assert torch.equal(mean, per_agent.mean(dim=-1))
    with pytest.raises(ValueError):
        rbg.RandomAgentEvaluator(rbg.MultiToSingleWrapper(env, reward_aggregator=torch.amax), B)

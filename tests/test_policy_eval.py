"""Policy evaluation on the device (rbg_connector_eval_step, engine.connector_eval_step, PolicyEvaluator) against the
plain Connector.step of the GPU library and of the CPU oracle, with the same policy driving both sides.  Integers
exactly, float32 by their bits.  Every test but the header check needs a CUDA device (`-m gpu`).

The test policies are pure integer functions of the action mask and the action key, written once in numpy (for the
oracle loop) and once in torch (for the evaluator):
  keyed:  agent a takes the ((key0 ^ a * 0x9E3779B9) mod n)-th of its n legal actions, in action order;
  greedy: the first legal move, else NOOP;
  noop:   NOOP."""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
METRICS = ("episode_return", "episode_length", "num_connections", "ratio_connections", "total_path_length")
STATE_FIELDS = ("grid", "step_count", "agent_id", "start", "target", "position", "key")
TS_FIELDS = ("obs", "action_mask", "obs_step_count", "reward", "discount", "step_type", "num_connections", "ratio_connections", "total_path_length")
GENS = {"parallel_random_walk": "ParallelRandomWalkGenerator", "uniform": "UniformRandomGenerator", "seed_extension": "SeedExtensionGenerator",
        "sequential_random_walk": "SequentialRandomWalkGenerator"}
SHAPES = [(5, 3), (10, 5), (7, 6), (32, 16), (40, 32), (2, 1)]  # G x G / N; 7 x 7 and 5 x 5: cells % 4 != 0
# few agents on a big board: a CTA's grids need more than 48 KB of shared memory (40 x 40 / 1: 200 KB)
BIG_SMEM_SHAPES = [(40, 1), (28, 2), (40, 4), (20, 1)]
GOLDEN = 0x9E3779B9


def test_eval_step_kernel_id_and_symbol_match_header():
    """RBG_K_EVAL_STEP is _lib.KERNELS["eval_step"], RBG_K_COUNT counts every kernel id, and the ctypes signature of
    rbg_connector_eval_step has the header's number of parameters."""
    import routing_board_generation_b200 as pkg

    with open(os.path.join(ROOT, "include", "rbg_b200.h")) as f:
        src = re.sub(r"/\*.*?\*/", "", f.read(), flags=re.S)
    L = pkg._lib
    assert L.KERNELS["eval_step"] == int(re.search(r"#define RBG_K_EVAL_STEP (\d+)", src).group(1))
    assert int(re.search(r"#define RBG_K_COUNT (\d+)", src).group(1)) == len(L.KERNELS) == max(L.KERNELS.values()) + 1
    params = re.search(r"int rbg_connector_eval_step\((.*?)\);", src, flags=re.S).group(1).split(",")
    assert len(L.SYMBOLS["rbg_connector_eval_step"][1]) == len(params) == 11


# ------------------------------------------------------------------ policies
def keyed_np(mask, ak):
    mask = mask.astype(bool)
    n = mask.sum(-1).astype(np.uint64)
    a = (np.arange(mask.shape[1], dtype=np.uint64) * GOLDEN) & 0xFFFFFFFF
    k = ((ak[:, 0].astype(np.uint64)[:, None] ^ a[None, :]) % n).astype(np.int64)
    return np.argmax(mask & (np.cumsum(mask, -1) == (k + 1)[..., None]), -1).astype(np.int32)


def greedy_np(mask, ak):
    m = mask.astype(bool)[..., 1:]
    return np.where(m.any(-1), m.argmax(-1) + 1, 0).astype(np.int32)


def noop_np(mask, ak):
    return np.zeros(mask.shape[:2], np.int32)


def keyed_torch(obs, key):
    import torch

    mask = obs.action_mask
    n = mask.sum(-1)
    a = (torch.arange(mask.shape[1], dtype=torch.int64, device=mask.device) * GOLDEN) & 0xFFFFFFFF
    k0 = key.view(torch.int32)[:, 0].to(torch.int64) & 0xFFFFFFFF
    k = (k0[:, None] ^ a[None, :]) % n
    c = mask.to(torch.int64)  # running count of legal actions (torch.cumsum over 5 entries is a slow scan on the GPU)
    for i in range(1, c.shape[-1]):
        c[..., i] += c[..., i - 1]
    return (mask & (c == (k + 1)[..., None])).to(torch.int8).argmax(-1).to(torch.int32)


def greedy_torch(obs, key):
    import torch

    m = obs.action_mask[..., 1:]
    return torch.where(m.any(-1), m.to(torch.int8).argmax(-1) + 1, 0).to(torch.int32)


def noop_torch(obs, key):
    import torch

    return torch.zeros(obs.action_mask.shape[:2], dtype=torch.int32, device=obs.action_mask.device)


POLICIES = {"keyed": (keyed_np, keyed_torch), "greedy": (greedy_np, greedy_torch), "noop": (noop_np, noop_torch)}


def test_policies_agree_between_numpy_and_torch():
    """The two spellings of each test policy give the same actions (on the CPU)."""
    import torch

    from routing_board_generation_b200.types import Observation

    rng = np.random.default_rng(0)
    mask = rng.random((257, 7, 5)) < 0.5
    mask[..., 0] = True
    mask[:5, :, 1:] = False
    ak = rng.integers(0, 2**32, size=(257, 2), dtype=np.uint64).astype(np.uint32)
    obs = Observation(grid=None, action_mask=torch.from_numpy(mask), step_count=None)
    key = torch.from_numpy(ak.view(np.int32)).view(torch.uint32)
    for name, (pn, pt) in POLICIES.items():
        ref = pn(mask, ak)
        assert np.all(mask[np.arange(257)[:, None], np.arange(7)[None, :], ref]), name
        assert np.array_equal(pt(obs, key).numpy(), ref), name


# ------------------------------------------------------------------ helpers
def _np(t):
    import torch

    if t.dtype == torch.uint32:
        return t.view(torch.int32).cpu().numpy().view(np.uint32)
    if t.dtype == torch.bool:
        return t.cpu().numpy().astype(np.uint8)
    return t.cpu().numpy()


def _state_np(st):
    a = st.agents
    return dict(grid=_np(st.grid), step_count=_np(st.step_count), agent_id=_np(a.id), start=_np(a.start), target=_np(a.target), position=_np(a.position), key=_np(st.key))


def _ts_np(ts):
    o, x = ts.observation, ts.extras
    return dict(obs=_np(o.grid), action_mask=_np(o.action_mask), obs_step_count=_np(o.step_count), reward=_np(ts.reward), discount=_np(ts.discount),
                step_type=_np(ts.step_type), **{k: _np(x[k]) for k in ("num_connections", "ratio_connections", "total_path_length")})


def _state_gpu(rbg, s):
    import torch

    t = lambda a: rbg.engine.as_tensor(a)
    return rbg.State(key=rbg.engine.as_tensor(s["key"], torch.uint32), grid=t(s["grid"]), step_count=t(s["step_count"]),
                     agents=rbg.Agent(id=t(s["agent_id"]), start=t(s["start"]), target=t(s["target"]), position=t(s["position"])))


def _bits(a):
    return a.view(np.uint32) if a.dtype == np.float32 else a


def _eq(got, ref, what):
    assert got.shape == ref.shape and np.array_equal(_bits(got), _bits(ref)), f"{what} differs"


def _keys(rbg, orc, seed, B):
    k = rbg.split(rbg.PRNGKey(seed), B)
    ref = orc.split(orc.PRNGKey(seed), B)
    assert np.array_equal(_np(k), ref)
    return k, ref


def _assert_metrics(got, ref, where=""):
    for k in METRICS:
        _eq(_np(got[k]), ref[k], f"{k} {where}")


def oracle_policy_episodes(rbg, orc, st, keys, policy_np, time_limit):
    """The oracle's plain Connector.step (autoreset_kind=-1) under `policy_np` on the oracle's own observation, each env
    stepped until its first LAST step, with PolicyEvaluator's action keys (from engine.split_each, pinned against the
    oracle elsewhere); returns in float32, added in step order."""
    st = {k: v.copy() for k, v in st.items()}
    B, N = st["target"].shape[:2]
    mask = orc.connector_observe_batch(st)["action_mask"]
    m = dict(episode_return=np.zeros((B, N), np.float32), episode_length=np.zeros(B, np.int32), num_connections=np.zeros(B, np.int32),
             ratio_connections=np.zeros(B, np.float32), total_path_length=np.zeros(B, np.int32))
    chain = rbg.engine.split_each(keys)[:, 1]
    alive = np.arange(B)
    while alive.size:
        s = rbg.engine.split_each(chain)
        chain, ak = s[:, 0], _np(s[:, 1].contiguous())
        sub = {k: v[alive] for k, v in st.items()}
        nsub, ts = orc.connector_step_batch(sub, policy_np(mask[alive], ak[alive]), time_limit=time_limit, autoreset_kind=-1)
        m["episode_return"][alive] = m["episode_return"][alive] + ts["reward"]
        m["episode_length"][alive] += 1
        for k in st:
            st[k][alive] = nsub[k]
        mask[alive] = ts["action_mask"]
        last = ts["step_type"] == 2
        for k in ("num_connections", "ratio_connections", "total_path_length"):
            m[k][alive[last]] = ts[k][last]
        alive = alive[~last]
    return m


def _check_evaluator(rbg, orc, env, st_np, keys, policy, time_limit, where):
    pn, pt = POLICIES[policy]
    got = rbg.PolicyEvaluator(env, pt, keys.shape[0]).episode_metrics(keys)
    ref = oracle_policy_episodes(rbg, orc, st_np, keys, pn, time_limit)
    _assert_metrics(got, ref, where)
    assert int(ref["episode_length"].max()) <= time_limit
    return ref


# ------------------------------------------------------- the kernel, one step
@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, 31, 33, 2048])
@pytest.mark.parametrize("G,N", SHAPES + BIG_SMEM_SHAPES)
@pytest.mark.parametrize("steps,time_limit", [(3, 50), (5, 6)])
def test_eval_step_matches_connector_step(rbg, orc, G, N, B, steps, time_limit):
    """Mid-episode States, a random live mask, TimeStep / record prefilled with sentinels: live rows equal the plain
    Connector.step (the GPU library's; for the shapes whose Connector.step needs more than 48 KB of shared memory per
    CTA, the oracle's), dead rows are untouched, and live / live_count / the record are updated as documented."""
    import torch

    seed = G * 1000 + N * 10 + B + steps
    rng = np.random.default_rng(seed)
    _, kref = _keys(rbg, orc, seed, B)
    s0 = orc.state_batch("parallel_random_walk", kref, G, N)
    for _ in range(steps):  # PATH cells, connected agents, and with time_limit 6 a step that ends every episode
        s0, _ = orc.connector_step_batch(s0, orc.random_actions_batch(s0), time_limit=time_limit, autoreset_kind=-1)
    act = rng.integers(0, 5, size=(B, N)).astype(np.int32)
    live0 = (rng.random(B) < 0.7).astype(np.uint8)
    if (G, N) in BIG_SMEM_SHAPES:
        rs, rts = orc.connector_step_batch(s0, act, time_limit=time_limit, autoreset_kind=-1)
    else:
        rs, rts = rbg.engine.connector_step(_state_gpu(rbg, s0), rbg.engine.as_tensor(act), time_limit=time_limit, autoreset_kind=-1)
        rs, rts = _state_np(rs), _ts_np(rts)

    dev = torch.device("cuda")
    st = _state_gpu(rbg, s0)
    ts = rbg.engine.alloc_timestep(B, G, N)
    for t, v in ((ts.observation.grid, -7), (ts.observation.action_mask, True), (ts.observation.step_count, -3), (ts.reward, 1234.5), (ts.discount, -2.0),
                 (ts.step_type, 9), (ts.extras["num_connections"], -11), (ts.extras["ratio_connections"], 7.25), (ts.extras["total_path_length"], -13)):
        t.fill_(v)
    ts0 = _ts_np(ts)
    acc0 = dict(episode_return=rng.integers(-40, 40, size=(B, N)).astype(np.float32) * np.float32(0.37), episode_length=rng.integers(0, 9, B).astype(np.int32),
                num_connections=np.full(B, -5, np.int32), ratio_connections=np.full(B, -0.5, np.float32), total_path_length=np.full(B, -6, np.int32))
    acc = {k: rbg.engine.as_tensor(v) for k, v in acc0.items()}
    live = rbg.engine.as_tensor(live0)
    count0 = int(live0.sum()) + 17
    live_count = torch.full((1,), count0, dtype=torch.int32, device=dev)
    rbg.engine.connector_eval_step(st, rbg.engine.as_tensor(act), live, live_count, acc, ts, time_limit=time_limit)

    on = live0 != 0
    got_s, got_ts = _state_np(st), _ts_np(ts)
    for k in STATE_FIELDS:
        _eq(got_s[k][on], rs[k][on], f"state.{k} (live)")
        _eq(got_s[k][~on], s0[k][~on], f"state.{k} (dead)")
    for k in TS_FIELDS:
        _eq(got_ts[k][on], rts[k][on], f"timestep.{k} (live)")
        _eq(got_ts[k][~on], ts0[k][~on], f"timestep.{k} (dead)")
    last = on & (rts["step_type"] == 2)
    exp = {k: v.copy() for k, v in acc0.items()}
    exp["episode_return"][on] = acc0["episode_return"][on] + rts["reward"][on]  # float32 + float32, round to nearest
    exp["episode_length"][on] += 1
    for k in ("num_connections", "ratio_connections", "total_path_length"):
        exp[k][last] = rts[k][last]
    _assert_metrics(acc, exp, "(record)")
    assert np.array_equal(_np(live), np.where(last, 0, live0).astype(np.uint8))
    assert int(live_count.item()) == count0 - int(last.sum())
    if time_limit == 6:
        assert last.sum() == on.sum()


@pytest.mark.gpu
def test_eval_step_on_a_dead_batch_writes_nothing(rbg, orc):
    import torch

    G, N, B = 10, 5, 300
    _, kref = _keys(rbg, orc, 3, B)
    s0 = orc.state_batch("uniform", kref, G, N)
    st = _state_gpu(rbg, s0)
    ts = rbg.engine.alloc_timestep(B, G, N)
    ts.observation.grid.fill_(-1)
    ts0 = _ts_np(ts)
    acc = {k: torch.zeros((B, N) if k == "episode_return" else (B,), dtype=torch.float32 if k in ("episode_return", "ratio_connections") else torch.int32, device="cuda")
           for k in METRICS}
    live = torch.zeros(B, dtype=torch.uint8, device="cuda")
    live_count = torch.zeros(1, dtype=torch.int32, device="cuda")
    rbg.engine.connector_eval_step(st, torch.ones((B, N), dtype=torch.int32, device="cuda"), live, live_count, acc, ts)
    for k in STATE_FIELDS:
        _eq(_state_np(st)[k], s0[k], f"state.{k}")
    for k in TS_FIELDS:
        _eq(_ts_np(ts)[k], ts0[k], f"timestep.{k}")
    assert all(int(v.abs().sum()) == 0 for v in acc.values()) and int(live_count.item()) == 0


# ------------------------------------------------ the evaluator, whole episodes
@pytest.mark.gpu
@pytest.mark.parametrize("policy", list(POLICIES))
@pytest.mark.parametrize("kind", ["parallel_random_walk", "uniform"])
@pytest.mark.parametrize("G,N", SHAPES)
@pytest.mark.parametrize("time_limit", [1, 7, 50])
def test_evaluator_matches_oracle(rbg, orc, policy, kind, G, N, time_limit):
    B = 2048 if G < 32 else 512
    keys, kref = _keys(rbg, orc, G * 100 + N + time_limit, B)
    env = rbg.Connector(generator=getattr(rbg, GENS[kind])(G, N), time_limit=time_limit)
    _check_evaluator(rbg, orc, env, orc.state_batch(kind, kref, G, N), keys, policy, time_limit, f"({policy} {kind} {G}x{G}/{N} time_limit {time_limit})")


@pytest.mark.gpu
@pytest.mark.parametrize("policy", ["keyed", "greedy"])
@pytest.mark.parametrize("kind,G,N", [("seed_extension", 10, 5), ("sequential_random_walk", 10, 5), ("seed_extension", 7, 3), ("sequential_random_walk", 16, 8)])
def test_evaluator_other_generators(rbg, orc, policy, kind, G, N):
    B = 1500
    keys, kref = _keys(rbg, orc, 77, B)
    env = rbg.Connector(generator=getattr(rbg, GENS[kind])(G, N), time_limit=50)
    _check_evaluator(rbg, orc, env, orc.state_batch(kind, kref, G, N), keys, policy, 50, kind)


@pytest.mark.gpu
def test_evaluator_dataset_generator(rbg, orc):
    G, N, B = 10, 5, 1200
    gen = rbg.BoardDatasetGeneratorJAX(G, N, board_name="offline_parallel_rw", number_of_boards=37)
    keys, kref = _keys(rbg, orc, 78, B)
    st = orc.dataset_state_batch(kref, G, N, _np(gen.heads), _np(gen.targets))
    _check_evaluator(rbg, orc, rbg.Connector(generator=gen, time_limit=30), st, keys, "keyed", 30, "dataset generator")


@pytest.mark.gpu
def test_evaluator_user_generator(rbg, orc):
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
    env = rbg.VmapAutoResetWrapper(rbg.Connector(generator=gen, time_limit=12))
    _check_evaluator(rbg, orc, env, _state_np(gen(keys)), keys, "keyed", 12, "user generator")


@pytest.mark.gpu
@pytest.mark.parametrize("G,N,B", [(10, 5, 65536), (32, 16, 8192)])
def test_evaluator_full_size_matches_oracle(rbg, orc, G, N, B):
    keys, kref = _keys(rbg, orc, 2, B)
    env = rbg.Connector(generator=rbg.ParallelRandomWalkGenerator(G, N), time_limit=50)
    _check_evaluator(rbg, orc, env, orc.state_batch("parallel_random_walk", kref, G, N), keys, "keyed", 50, f"({G}x{G}/{N} x {B})")


@pytest.mark.gpu
@pytest.mark.parametrize("policy", list(POLICIES))
def test_evaluator_agrees_with_connector_step_loop(rbg, orc, policy):
    """The metrics equal those taken from each env's first LAST in a plain Connector.step loop on the GPU, driven by the
    same policy on the same observations and action keys."""
    import torch

    G, N, B, TL = 10, 5, 4096, 50
    keys, _ = _keys(rbg, orc, 9, B)
    pt = POLICIES[policy][1]
    env = rbg.Connector(generator=rbg.ParallelRandomWalkGenerator(G, N), time_limit=TL)
    got = rbg.PolicyEvaluator(env, pt, B).episode_metrics(keys)
    st, ts = env.reset(keys)
    dev = st.grid.device
    ret = torch.zeros((B, N), dtype=torch.float32, device=dev)
    length = torch.zeros(B, dtype=torch.int32, device=dev)
    extras = {k: torch.zeros(B, dtype=d, device=dev) for k, d in (("num_connections", torch.int32), ("ratio_connections", torch.float32), ("total_path_length", torch.int32))}
    done = torch.zeros(B, dtype=torch.bool, device=dev)
    chain = rbg.engine.split_each(keys)[:, 1]
    while not bool(done.all()):
        s = rbg.engine.split_each(chain)
        chain = s[:, 0]
        st, ts = env.step(st, pt(ts.observation, s[:, 1].contiguous()))
        alive = ~done
        ret = torch.where(alive[:, None], ret + ts.reward, ret)
        length += alive.int()
        last = alive & (ts.step_type == 2)
        for k in extras:
            extras[k] = torch.where(last, ts.extras[k], extras[k])
        done |= last
    ref = dict(episode_return=_np(ret), episode_length=_np(length), **{k: _np(v) for k, v in extras.items()})
    _assert_metrics(got, ref, "against the Connector.step loop")


# ---------------------------------------------------------- evaluator surface
@pytest.mark.gpu
def test_evaluator_multi_to_single_sum_and_mean(rbg, orc):
    """MultiToSingleWrapper: torch.sum (the default) and torch.mean of the per-agent returns; a non-linear aggregator is
    refused; the other metrics are per env as without the wrapper."""
    import torch

    G, N, B = 10, 5, 2048
    keys, _ = _keys(rbg, orc, 31, B)
    env = rbg.Connector(generator=rbg.ParallelRandomWalkGenerator(G, N), time_limit=50)
    multi = rbg.PolicyEvaluator(env, keyed_torch, B).episode_metrics(keys)
    total = rbg.PolicyEvaluator(rbg.VmapAutoResetWrapper(rbg.MultiToSingleWrapper(env)), keyed_torch, B).episode_metrics(keys)
    mean = rbg.PolicyEvaluator(rbg.MultiToSingleWrapper(env, reward_aggregator=torch.mean), keyed_torch, B).episode_metrics(keys)
    assert tuple(total["episode_return"].shape) == (B,)
    assert torch.equal(total["episode_return"], multi["episode_return"].sum(dim=-1))
    assert torch.equal(mean["episode_return"], multi["episode_return"].mean(dim=-1))
    for k in METRICS[1:]:
        assert torch.equal(total[k], multi[k]) and torch.equal(mean[k], multi[k]), k
    with pytest.raises(ValueError):
        rbg.PolicyEvaluator(rbg.MultiToSingleWrapper(env, reward_aggregator=torch.amax), keyed_torch, B)


@pytest.mark.gpu
def test_evaluator_run_evaluation_is_the_mean(rbg):
    import torch

    B = 3000
    ev = rbg.PolicyEvaluator(rbg.MultiToSingleWrapper(rbg.Connector(generator=rbg.UniformRandomGenerator(10, 5), time_limit=50)), greedy_torch, B)
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
    import torch

    G, N = 10, 5
    env = rbg.Connector(generator=rbg.ParallelRandomWalkGenerator(G, N), time_limit=50)
    ev = rbg.PolicyEvaluator(env, keyed_torch, 1)
    key = rbg.PRNGKey(6)
    one = ev.episode_metrics(key)
    assert tuple(one["episode_return"].shape) == (N,)
    for k in METRICS[1:]:
        assert one[k].dim() == 0
    batched = ev.episode_metrics(key[None])
    for k in METRICS:
        assert torch.equal(one[k], batched[k][0]), k


@pytest.mark.gpu
def test_argument_errors(rbg, orc):
    import torch

    lib = rbg._lib.load()
    B, G, N = 8, 10, 5
    _, kref = _keys(rbg, orc, 1, B)
    st = _state_gpu(rbg, orc.state_batch("parallel_random_walk", kref, G, N))
    ts = rbg.engine.alloc_timestep(B, G, N)
    dev = st.grid.device
    s, t = rbg.engine._state_struct(st), rbg.engine._timestep_struct(ts)
    act = torch.zeros((B, N), dtype=torch.int32, device=dev)
    live = torch.ones(B, dtype=torch.uint8, device=dev)
    count = torch.full((1,), B, dtype=torch.int32, device=dev)
    bufs = [torch.zeros((B, N), dtype=torch.float32, device=dev)] + [torch.zeros(B, dtype=d, device=dev) for d in (torch.int32, torch.int32, torch.float32, torch.int32)]
    m = rbg._lib.rbg_episode_metrics(*(b.data_ptr() for b in bufs))
    ok = rbg._lib.rbg_env_params(50, -0.03, 0.1, -1)

    def call(s_=C.byref(s), a=act.data_ptr(), lv=live.data_ptr(), lc=count.data_ptr(), Bx=B, Gx=G, Nx=N, p=C.byref(ok), t_=C.byref(t), m_=C.byref(m)):
        return lib.rbg_connector_eval_step(s_, a, lv, lc, Bx, Gx, Nx, p, t_, m_, None)

    assert call() == 0
    assert lib.rbg_connector_eval_step(None, None, None, None, 0, G, N, None, None, None, None) == 0  # an empty batch
    assert call(s_=None) == -1 and b"state" in lib.rbg_last_error()
    assert call(a=None) == -1 and b"action" in lib.rbg_last_error()
    assert call(lv=None) == -1 and b"live" in lib.rbg_last_error()
    assert call(lc=None) == -1 and b"live_count" in lib.rbg_last_error()
    assert call(p=None) == -1 and b"params" in lib.rbg_last_error()
    assert call(t_=None) == -1 and b"timestep" in lib.rbg_last_error()
    assert call(m_=None) == -1 and b"acc" in lib.rbg_last_error()
    for i in range(5):
        bad = rbg._lib.rbg_episode_metrics(*(0 if j == i else b.data_ptr() for j, b in enumerate(bufs)))
        assert call(m_=C.byref(bad)) == -1 and b"NULL" in lib.rbg_last_error()
    bad_ts = rbg.engine._timestep_struct(ts)
    bad_ts.reward = None
    assert call(t_=C.byref(bad_ts)) == -1 and b"NULL" in lib.rbg_last_error()
    assert call(Gx=41) == -1 and b"grid size" in lib.rbg_last_error()
    assert call(Gx=1) == -1 and b"grid size" in lib.rbg_last_error()
    assert call(Nx=0) == -1 and b"num_agents" in lib.rbg_last_error()
    assert call(Nx=33) == -1 and b"num_agents" in lib.rbg_last_error()
    assert call(Bx=-1) == -1
    for kind in (0, 1, 2, 3, 4):
        ar = rbg._lib.rbg_env_params(50, -0.03, 0.1, kind)
        assert call(p=C.byref(ar)) == -1 and b"autoreset_kind" in lib.rbg_last_error()
    with pytest.raises(ValueError):
        rbg.engine.connector_eval_step(st, act, live.to(torch.int32), count, dict(zip(METRICS, bufs)), ts)
    torch.cuda.synchronize()

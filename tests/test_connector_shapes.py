"""Every Connector entry point against the oracle at every lane layout of the warp kernels and at both board parities.

The warp kernels give each env Np lanes (the next power of two >= N), so one warp holds K = 32 / Np envs, and a board
whose cell count is not a multiple of 4 (odd G) takes the scalar instantiations.  A CTA of four warps keeps K grids per
warp in shared memory, which passes the default 48 KB for few agents on a big board.  Each row of SHAPES is one lane
layout at one parity or one side of that limit.  The batch of 2 * 4 * K + K // 2 + 1 envs fills two CTAs and leaves a
third whose last warp is ragged.  Integers are compared exactly and float32 values by their bits, at every step.
"""
import ctypes as C

import numpy as np
import pytest

from test_episodes import oracle_episodes
from test_gpu_parity import _assert_state, _assert_timestep, _keys, _np
from test_policy_eval import POLICIES, oracle_policy_episodes

pytestmark = pytest.mark.gpu

SHAPES = [
    # Np 1: 32 envs per warp
    (2, 1),     # the smallest board
    (5, 1),     # odd G
    (19, 1),    # the last N = 1 board whose step fits 48 KB of shared memory
    (20, 1),    # the first one above 48 KB
    (33, 1),    # odd G above 48 KB
    (36, 1),    # the fused rollout does not fit 200 KB: step-wise
    (40, 1),    # the largest board: 200 KB for the step
    # Np 2: 16 envs per warp
    (7, 2),     # odd G
    (27, 2),    # odd G, the last N = 2 board within 48 KB
    (28, 2),    # the first N = 2 board above 48 KB
    (39, 2),    # odd G above 48 KB
    (40, 2),
    # Np 4: 8 envs per warp
    (5, 3),     # odd G
    (39, 4),    # odd G, 128 bytes under 48 KB
    (40, 3),    # above 48 KB, one idle lane per env
    (40, 4),    # above 48 KB
    # Np 8: 4 envs per warp
    (9, 7),     # odd G
    (16, 8),
    # Np 16: 2 envs per warp
    (11, 9),    # odd G
    (17, 16),   # odd G, every lane busy
    (40, 16),
    # Np 32: one env per warp
    (6, 17),
    (8, 32),    # dense: 2N = G * G, every cell a head or a target
    (13, 25),   # odd G
    (40, 32),   # the largest shape
]
# one row per Np class also runs as a single env
SINGLE = [(40, 1), (39, 2), (40, 3), (9, 7), (11, 9), (13, 25)]


def _batch(N):
    Np = 1
    while Np < N:
        Np *= 2
    K = 32 // Np
    return 2 * 4 * K + K // 2 + 1


CASES = [(G, N, _batch(N)) for G, N in SHAPES] + [(G, N, 1) for G, N in SINGLE]
GENS = {"parallel_random_walk": "ParallelRandomWalkGenerator", "uniform": "UniformRandomGenerator", "seed_extension": "SeedExtensionGenerator",
        "sequential_random_walk": "SequentialRandomWalkGenerator"}


def _env(rbg, kind, G, N, time_limit, reward=None):
    if kind == "dataset":
        gen = rbg.BoardDatasetGeneratorJAX(G, N, board_name="offline_parallel_rw", number_of_boards=7)
    else:
        gen = getattr(rbg, GENS[kind])(G, N)
    reward_fn = rbg.DenseRewardFn(*reward) if reward else None
    return rbg.Connector(generator=gen, reward_fn=reward_fn, time_limit=time_limit)


def _reset(rbg, orc, env, kind, G, N, B, seed):
    """env.reset on split(PRNGKey(seed), B) against the oracle -> (State, oracle State, oracle dataset or None)."""
    keys, kref = _keys(rbg, orc, seed, B)
    st, ts = env.reset(keys)
    if kind == "dataset":
        ds = (_np(env._generator.heads), _np(env._generator.targets))
        rst = orc.dataset_state_batch(kref, G, N, *ds)
        rts = orc.connector_observe_batch(rst)
    else:
        ds = None
        rst, rts = orc.connector_reset_batch(kind, kref, G, N)
    _assert_state(st, rst, "after reset")
    _assert_timestep(ts, rts, "after reset")
    return st, rst, ds


def _actions(rbg, orc, rng, st, rst, t):
    """Three kinds in turn: the library's random policy (legal moves: long walks, connections), unconstrained codes in
    [-1, 7) (illegal moves, collisions, out-of-range codes) and all NOOP."""
    B, N = rst["target"].shape[:2]
    if t % 3 == 0:
        act = orc.random_actions_batch(rst)
        assert np.array_equal(_np(rbg.make_random_policy_connector()(st)), act), f"random policy differs at step {t}"
        return act
    if t % 3 == 1:
        return rng.integers(-1, 7, size=(B, N)).astype(np.int32)
    return np.zeros((B, N), np.int32)


def _same(got, ref):
    bits = lambda a: a.view(np.uint32) if a.dtype == np.float32 else a
    return got.shape == ref.shape and np.array_equal(bits(got), bits(ref))


def _rewards(ts, rts, reward):
    """Both reward values occur in the oracle's rewards, so the ones the kernel used are checked."""
    tr, cr = np.float32(reward[0]), np.float32(reward[1])
    r = rts["reward"]
    return bool((r == tr).any()), bool((r == cr).any() or (r == cr + tr).any())


# ------------------------------------------------------------------ reset and plain steps
@pytest.mark.parametrize("kind", ["parallel_random_walk", "uniform"])
@pytest.mark.parametrize("time_limit", [2, 5])
@pytest.mark.parametrize("G,N,B", CASES)
def test_reset_and_steps(rbg, orc, kind, time_limit, G, N, B):
    """Connector.reset, then 2 * time_limit + 2 plain Connector.steps (past the LAST step), in place every other step."""
    env = _env(rbg, kind, G, N, time_limit)
    st, rst, _ = _reset(rbg, orc, env, kind, G, N, B, seed=G * 1000 + N * 10 + time_limit)
    rng = np.random.default_rng(G * 100 + N)
    n_last = 0
    for t in range(2 * time_limit + 2):
        act = _actions(rbg, orc, rng, st, rst, t)
        a = rbg.engine.as_tensor(act)
        if t % 2:
            st, ts = rbg.engine.connector_step(st, a, **env._env_args(), inplace=True)
        else:
            st, ts = env.step(st, a)
        rst, rts = orc.connector_step_batch(rst, act, time_limit=time_limit)
        _assert_state(st, rst, f"at step {t}")
        _assert_timestep(ts, rts, f"at step {t}")
        n_last += int((rts["step_type"] == 2).sum())
    assert n_last >= B


# ------------------------------------------------------------------ auto-reset steps
SEQRW_ROWS = [(5, 1), (20, 1), (40, 1), (28, 2), (39, 2), (40, 4), (9, 7), (17, 16), (13, 25), (40, 32)]
AUTORESET = ([("parallel_random_walk", *c) for c in CASES] + [("uniform", *c) for c in CASES] + [("dataset", *c) for c in CASES]
             + [("seed_extension", G, N, B) for G, N, B in CASES if N <= (G // 2) ** 2]
             + [("sequential_random_walk", G, N, B) for G, N, B in CASES if (G, N) in SEQRW_ROWS])


@pytest.mark.parametrize("kind,G,N,B", AUTORESET)
def test_autoreset_steps(rbg, orc, kind, G, N, B):
    """VmapAutoResetWrapper.step and step_random in turn with time_limit 2: every env resets every other step, so the
    next-episode cache is drained and both the cached and the synchronous reset paths run."""
    time_limit = 2
    env = rbg.VmapAutoResetWrapper(_env(rbg, kind, G, N, time_limit))
    st, rst, ds = _reset(rbg, orc, env, kind, G, N, B, seed=G * 1000 + N * 10 + 7)
    rng = np.random.default_rng(G * 100 + N + 1)
    for t in range(8):
        if t % 2:
            act = orc.random_actions_batch(rst)
            st, ts, got = env.step_random(st, inplace=t % 4 == 1)
            assert np.array_equal(_np(got), act), f"random actions differ at step {t}"
        else:
            act = _actions(rbg, orc, rng, st, rst, t // 2)
            st, ts = env.step(st, rbg.engine.as_tensor(act), inplace=t % 4 == 2)
        rst, rts = orc.connector_step_batch(rst, act, time_limit=time_limit, autoreset_kind=kind, dataset=ds)
        _assert_state(st, rst, f"at step {t}")
        _assert_timestep(ts, rts, f"at step {t}")


# ------------------------------------------------------------------ fused rollout
def _check_rollout(rbg, orc, env, st, rst, kind, T, time_limit, ds, reward=(-0.03, 0.1), where=""):
    st, ts, act = env.rollout_random(st, T)
    for t in range(T):
        a = orc.random_actions_batch(rst)
        assert np.array_equal(_np(act[t]), a), f"actions differ at step {t} {where}"
        rst, rts = orc.connector_step_batch(rst, a, time_limit=time_limit, timestep_reward=reward[0], connected_reward=reward[1], autoreset_kind=kind, dataset=ds)
        _assert_timestep(ts[t], rts, f"at step {t} {where}")
    _assert_state(st, rst, f"after the rollout {where}")
    return st, rst


@pytest.mark.parametrize("kind", ["parallel_random_walk", "uniform", "dataset"])
@pytest.mark.parametrize("G,N,B", CASES)
def test_rollout(rbg, orc, kind, G, N, B):
    """rollout_random over 23 steps (across the 20-step launch chunk), a second rollout from its State, then one
    step_random on the same workspace, against oracle steps under the oracle's random actions."""
    time_limit = 5
    env = rbg.VmapAutoResetWrapper(_env(rbg, kind, G, N, time_limit))
    st, rst, ds = _reset(rbg, orc, env, kind, G, N, B, seed=G * 1000 + N * 10 + 9)
    st, rst = _check_rollout(rbg, orc, env, st, rst, kind, 23, time_limit, ds, where="(first)")
    st, rst = _check_rollout(rbg, orc, env, st, rst, kind, 7, time_limit, ds, where="(second)")
    a = orc.random_actions_batch(rst)
    st, ts, got = env.step_random(st)
    assert np.array_equal(_np(got), a)
    rst, rts = orc.connector_step_batch(rst, a, time_limit=time_limit, autoreset_kind=kind, dataset=ds)
    _assert_state(st, rst, "after the step that follows the rollouts")
    _assert_timestep(ts, rts, "at the step that follows the rollouts")


# ------------------------------------------------------------------ non-default rewards
# -0.7 + 2.3 rounds in float32; with -1e-3 and 1e4 the float32 sum of a return in step order differs from any other
# order or precision
REWARDS = [(-0.7, 2.3), (-1e-3, 1e4)]
REWARD_ROWS = [(5, 1), (40, 4), (13, 25)]


@pytest.mark.parametrize("reward", REWARDS)
@pytest.mark.parametrize("G,N", REWARD_ROWS)
def test_rewards_step_and_autoreset(rbg, orc, reward, G, N):
    """Connector.step and VmapAutoResetWrapper.step_random with a DenseRewardFn of its own."""
    B, tl = _batch(N), 6
    kw = dict(timestep_reward=reward[0], connected_reward=reward[1])
    env = _env(rbg, "uniform", G, N, tl, reward)
    st, rst, _ = _reset(rbg, orc, env, "uniform", G, N, B, seed=G + N)
    seen = [False, False]
    for t in range(tl + 2):
        act = orc.random_actions_batch(rst)
        st, ts = env.step(st, rbg.engine.as_tensor(act))
        rst, rts = orc.connector_step_batch(rst, act, time_limit=tl, **kw)
        _assert_state(st, rst, f"at step {t}")
        _assert_timestep(ts, rts, f"at step {t}")
        seen = [s or r for s, r in zip(seen, _rewards(ts, rts, reward))]
    wrapped = rbg.VmapAutoResetWrapper(env)
    for t in range(tl + 2):
        act = orc.random_actions_batch(rst)
        st, ts, got = wrapped.step_random(st)
        assert np.array_equal(_np(got), act)
        rst, rts = orc.connector_step_batch(rst, act, time_limit=tl, autoreset_kind="uniform", **kw)
        _assert_state(st, rst, f"at auto-reset step {t}")
        _assert_timestep(ts, rts, f"at auto-reset step {t}")
        seen = [s or r for s, r in zip(seen, _rewards(ts, rts, reward))]
    assert seen[0] and seen[1], "a timestep and a connected reward must both occur"


@pytest.mark.parametrize("kind", ["parallel_random_walk", "dataset"])
@pytest.mark.parametrize("reward", REWARDS)
@pytest.mark.parametrize("G,N", REWARD_ROWS)
def test_rewards_rollout(rbg, orc, kind, reward, G, N):
    """rollout_random (the persistent kernel for ParallelRandomWalk, rollout_warp_kernel for the dataset)."""
    tl = 4
    env = rbg.VmapAutoResetWrapper(_env(rbg, kind, G, N, tl, reward))
    st, rst, ds = _reset(rbg, orc, env, kind, G, N, _batch(N), seed=G + N + 1)
    _check_rollout(rbg, orc, env, st, rst, kind, 23, tl, ds, reward)


@pytest.mark.parametrize("reward", REWARDS)
@pytest.mark.parametrize("G,N", REWARD_ROWS)
def test_rewards_evaluators(rbg, orc, reward, G, N):
    """RandomAgentEvaluator and PolicyEvaluator: per-agent returns in float32, added in step order."""
    B, tl = _batch(N), 20
    env = _env(rbg, "uniform", G, N, tl, reward)
    keys, kref = _keys(rbg, orc, G * 7 + N, B)
    s0 = orc.state_batch("uniform", kref, G, N)
    got = rbg.RandomAgentEvaluator(env, B).episode_metrics(keys)
    ref, _ = oracle_episodes(orc, s0, tl, timestep_reward=reward[0], connected_reward=reward[1])
    for k, v in ref.items():
        assert _same(_np(got[k]), v), f"RandomAgentEvaluator {k} differs"
    pn, pt = POLICIES["greedy"]
    got = rbg.PolicyEvaluator(env, pt, B).episode_metrics(keys)
    ref = oracle_policy_episodes(rbg, orc, s0, keys, pn, tl, timestep_reward=reward[0], connected_reward=reward[1])
    for k, v in ref.items():
        assert _same(_np(got[k]), v), f"PolicyEvaluator {k} differs"


@pytest.mark.parametrize("reward", REWARDS)
@pytest.mark.parametrize("G,N", REWARD_ROWS)
def test_rewards_step_host_io(rbg, orc, reward, G, N):
    """rbg_connector_step_host_io: host actions in, host TimeStep out, auto-reset with ParallelRandomWalk."""
    L, lib = rbg._lib, rbg._lib.load()
    B, tl = _batch(N), 3
    env = rbg.VmapAutoResetWrapper(_env(rbg, "parallel_random_walk", G, N, tl, reward))
    st, rst, _ = _reset(rbg, orc, env, "parallel_random_walk", G, N, B, seed=G + N + 2)
    h = dict(obs=np.empty((B, N, G, G), np.int32), mask=np.empty((B, N, 5), np.uint8), sc=np.empty(B, np.int32), reward=np.empty((B, N), np.float32),
             discount=np.empty((B, N), np.float32), step_type=np.empty(B, np.int8), nc=np.empty(B, np.int32), rc=np.empty(B, np.float32), tpl=np.empty(B, np.int32))
    a = st.agents
    s = L.rbg_state(st.grid.data_ptr(), st.step_count.data_ptr(), a.id.data_ptr(), a.start.data_ptr(), a.target.data_ptr(), a.position.data_ptr(), st.key.data_ptr())
    t = L.rbg_timestep(*(h[k].ctypes.data for k in ("obs", "mask", "sc", "reward", "discount", "step_type", "nc", "rc", "tpl")))
    params = L.rbg_env_params(tl, reward[0], reward[1], 0)
    for step in range(8):
        act = orc.random_actions_batch(rst)
        L.check(lib.rbg_connector_step_host_io(C.byref(s), act.ctypes.data, B, G, N, C.byref(params), C.byref(t), -1))
        rst, rts = orc.connector_step_batch(rst, act, time_limit=tl, timestep_reward=reward[0], connected_reward=reward[1], autoreset_kind="parallel_random_walk")
        got = dict(obs=h["obs"], action_mask=h["mask"], obs_step_count=h["sc"], reward=h["reward"], discount=h["discount"], step_type=h["step_type"],
                   num_connections=h["nc"], ratio_connections=h["rc"], total_path_length=h["tpl"])
        for k, v in got.items():
            assert _same(v, rts[k]), f"{k} differs at step {step}"
        _assert_state(st, rst, f"at step {step}")

"""Dataset board picks against jax 0.4.8's randint, at spans on both sides of 2**16.

`BoardDatasetGeneratorJAX.__call__` picks a stored board with `which = randint(key, (), 0, K)`.  The library makes that
draw in three kernels (dataset_state_kernel for the reset and the evaluators' reset, env_warp_kernel for the per-step
auto-reset, rollout_warp_kernel for the fused dataset rollout) and the oracle makes it in `randint_from_bits`.

jax 0.4.8 `_randint` (jax/_src/random.py), for an int32 result (nbits = 32, unsigned_dtype = uint32):

    k1, k2 = _split(key)
    higher_bits, lower_bits = rbits(k1), rbits(k2)
    span = lax.convert_element_type(maxval - minval, unsigned_dtype)
    span = lax.select(maxval <= minval, lax.full_like(span, 1), span)
    multiplier = lax.rem(lax._const(span, 2 ** (nbits // 2)), span)
    multiplier = lax.rem(lax.mul(multiplier, multiplier), span)
    random_offset = lax.add(lax.mul(lax.rem(higher_bits, span), multiplier), lax.rem(lower_bits, span))
    random_offset = lax.rem(random_offset, span)
    return lax.add(minval, lax.convert_element_type(random_offset, dtype))

Every operation works on uint32 values, and XLA's unsigned multiply wraps modulo 2**32.  For a span above 2**16 the
multiplier is 2**16, whose square 2**32 wraps to 0: the draw is `lower_bits % span` and the first draw plays no part.
A square taken in 64 bits gives 2**32 mod span instead, which differs from 0 at every span above 2**16 that is not a
power of two (the reference's offline training stores 100 000 boards).  The lines above were read from the jax 0.4.8
source.  jax itself cannot run in this test suite, so the behaviour at large spans rests on that reading and on XLA's
wrap-around rule, not on a run of jax.

`jax_randint` restates those lines on NumPy uint32 arrays.  Only threefry (`orc.split`, `orc.random_bits`, pinned by the
reference goldens) comes from the oracle.  The CPU tests hold the oracle's randint and the jax shim's randint to it.
The GPU tests hold every dataset entry point to it, and every State / TimeStep leaf to the oracle, at dataset sizes
around 2**16; at non-power-of-two sizes above 2**16 a guard checks that a 64-bit square would have picked other boards.
"""
import importlib.util
import os
import sys

import numpy as np
import pytest

from oracle import oracle as orc
from test_episodes import _assert_metrics, oracle_episodes
from test_gpu_parity import _assert_state, _assert_timestep, _keys, _np
from test_policy_eval import POLICIES, oracle_policy_episodes

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
U32 = np.uint32


def _words(key, size):
    """random_bits(k1, 32, (size,)), random_bits(k2, 32, (size,)) with k1, k2 = split(key)."""
    k1, k2 = orc.split(key)
    return orc.random_bits(k1, size), orc.random_bits(k2, size)


def jax_randint(key, lo, hi, n=None):
    """jax 0.4.8 `randint(key, shape, lo, hi)` with int32 lo, hi: shape () when n is None, else (n,)."""
    size = 1 if n is None else n
    higher_bits, lower_bits = _words(key, size)
    span = np.full(size, (hi - lo) & 0xFFFFFFFF, U32)
    if hi <= lo:
        span[:] = 1
    multiplier = U32(2**16) % span
    multiplier = (multiplier * multiplier) % span  # uint32 * uint32 wraps, as XLA's does
    random_offset = ((higher_bits % span) * multiplier + lower_bits % span) % span
    out = (U32(lo & 0xFFFFFFFF) + random_offset).view(np.int32)  # int32 minval + offset, modulo 2**32
    return int(out[0]) if n is None else out


def randint_64bit_square(key, K):
    """The draw with the multiplier squared in 64 bits, as the library made it before: the sensitivity guard's
    counterfactual."""
    hb, lb = (int(w[0]) for w in _words(key, 1))
    m = (65536 % K) ** 2 % K
    return ((hb % K) * m + lb % K) % 2**32 % K


def _shim_random():
    """tests/tools/jax_shim's jax.random, loaded under a private name so that no `jax` module is installed."""
    name, path = "_jax_shim_for_picks", os.path.join(ROOT, "tests", "tools", "jax_shim", "jax")
    if name not in sys.modules:
        spec = importlib.util.spec_from_file_location(name, os.path.join(path, "__init__.py"), submodule_search_locations=[path])
        mod = importlib.util.module_from_spec(spec)
        sys.modules[name] = mod
        spec.loader.exec_module(mod)
    return sys.modules[name].random


# ------------------------------------------------------------------ CPU: randint
EMPTY = [(0, 0), (5, 5), (7, 3), (-4, -4), (3, -7)]                    # hi <= lo: span 1, the value is lo
POW2 = [(0, 2**k) for k in range(1, 31)]
OTHER = [(0, s) for s in (3, 7, 1000, 65535, 65536, 65537, 65538, 99999, 100000, 131071, 1048583, 2**31 - 1)]
NEGATIVE = [(-1, 1), (-5, 100), (-100000, -34463), (-70000, 30000), (-2**30, 2**30 - 1)]  # spans 2, 105, 65 537, 100 000, 2**31 - 1
SPANS = [pytest.param(lo, hi, n, id=f"{lo}:{hi}") for cls, n in ((EMPTY, 400), (POW2, 100), (OTHER, 250), (NEGATIVE, 400)) for lo, hi in cls]


def _test_keys(lo, hi, n):
    return orc.split(orc.PRNGKey((hi - lo) & 0x7FFFFFFF), n)


def test_jax_randint_known_answers(goldens):
    """SURVEY B0: randint(PRNGKey(0), (), 0, hi) = 0, 2, 2 for hi = 2, 4, 10."""
    assert [jax_randint(orc.PRNGKey(0), 0, hi) for hi in (2, 4, 10)] == goldens["rng"]["randint_key0_hi_2_4_10"]


@pytest.mark.parametrize("lo,hi,n", SPANS)
def test_oracle_randint(lo, hi, n):
    """orc.randint, scalar and with n draws (odd n pads the threefry counters), equals jax_randint."""
    keys = _test_keys(lo, hi, n)
    got = np.array([orc.randint(k, lo, hi) for k in keys])
    ref = np.array([jax_randint(k, lo, hi) for k in keys])
    assert np.array_equal(got, ref), f"{int((got != ref).sum())} of {n} scalar draws differ"
    for k in keys[:20]:
        for m in (1, 6, 7):
            assert np.array_equal(orc.randint(k, lo, hi, m), jax_randint(k, lo, hi, m)), f"n={m}"


@pytest.mark.parametrize("lo,hi,n", SPANS)
def test_shim_randint(lo, hi, n):
    """The jax shim's jax.random.randint, which made the Connector fixtures, equals jax_randint."""
    jr = _shim_random()
    keys = _test_keys(lo, hi, n)
    got = np.array([int(jr.randint(k, (), lo, hi)) for k in keys])
    ref = np.array([jax_randint(k, lo, hi) for k in keys])
    assert np.array_equal(got, ref), f"{int((got != ref).sum())} of {n} scalar draws differ"
    for k in keys[:20]:
        for m in (6, 7):
            assert np.array_equal(np.asarray(jr.randint(k, (m,), lo, hi)), jax_randint(k, lo, hi, m)), f"n={m}"


def test_spans_above_2_16_take_the_low_draw():
    """For every span above 2**16 the value is lo + lower_bits % span, whatever the first draw."""
    rng = np.random.default_rng(7)
    spans = np.concatenate([rng.integers(2**16 + 1, 2**31, 300), [2**16 + 1, 2**31 - 1]])
    keys = orc.split(orc.PRNGKey(11), spans.size)
    jr = _shim_random()
    for span, k in zip(spans.tolist(), keys):
        lo = -(span // 3)
        want = lo + int(_words(k, 1)[1][0]) % span
        assert jax_randint(k, lo, lo + span) == want, span
        assert orc.randint(k, lo, lo + span) == want, span
        assert int(jr.randint(k, (), lo, lo + span)) == want, span


# ------------------------------------------------------------------ GPU: every dataset entry point
gpu = pytest.mark.gpu
KS = [1, 2, 3, 65535, 65536, 65537, 100000, 131072, 1048583]
DATASETS = [("offline_parallel_rw", K) for K in KS] + [("offline_seed_extension", 100000)]  # the reference's default board
_CACHE = {}  # the 10x10/5 datasets, shared by the tests of this file


@pytest.fixture(scope="module", autouse=True)
def _free_datasets():
    yield
    _CACHE.clear()


def _split0(keys):
    """split(key)[0] of every row."""
    return np.stack([orc.split(k)[0] for k in keys])


def _dataset(rbg, board_name, G, N, K, cache=True):
    """BoardDatasetGeneratorJAX and its host copy (heads, targets); a sample of the stored boards is checked against
    the oracle's boards of split(PRNGKey(0), K)."""
    if (board_name, G, N, K) in _CACHE:
        return _CACHE[board_name, G, N, K]
    gen = rbg.BoardDatasetGeneratorJAX(G, N, board_name=board_name, number_of_boards=K)
    ds = (_np(gen.heads), _np(gen.targets))
    assert ds[0].shape == ds[1].shape == (K, 2, N)
    rng = np.random.default_rng(K)
    for i in sorted({0, K // 2, K - 1, *rng.integers(0, K, 8).tolist()}):
        k = orc.split_slice(orc.PRNGKey(0), K, i, 1)[0]
        if board_name == "offline_seed_extension":
            h, t = orc.seedext_starts_ends(k, G, N, randomness=1.0, two_sided=False)
        else:
            h, t, _, _ = orc.prw_generate(k, G, N)
        assert np.array_equal(ds[0][i], h) and np.array_equal(ds[1][i], t), f"stored board {i}"
    if cache:
        _CACHE[board_name, G, N, K] = gen, ds
    return gen, ds


def _check_picks(rk, start, target, ds, K, where=""):
    """The envs whose randint keys are rk[M,2] took boards jax_randint(rk, 0, K) of the dataset (start / target
    int32[M,N,2]).  Above 2**16 a non-power-of-two K is only tested if a 64-bit square would have picked other boards
    for nearly every env; and where a quarter of the boards or more lie at or above index 2**16, some picks do."""
    heads, targets = ds
    which = np.array([jax_randint(k, 0, K) for k in rk])
    assert np.array_equal(start, heads[which].transpose(0, 2, 1)), f"start differs from the jax pick {where}"
    assert np.array_equal(target, targets[which].transpose(0, 2, 1)), f"target differs from the jax pick {where}"
    if K > 65536 and K & (K - 1):
        old = np.array([randint_64bit_square(k, K) for k in rk])
        other = (heads[old] != heads[which]).any(axis=(1, 2)) | (targets[old] != targets[which]).any(axis=(1, 2))
        assert other.mean() >= 0.99, f"only {other.mean():.3f} of the picks are sensitive to the multiplier {where}"
    if K - 65536 >= K // 4:
        assert (which >= 65536).any(), f"no pick at or above 2**16 {where}"


@gpu
@pytest.mark.parametrize("board_name,K", DATASETS)
def test_generator_call(rbg, board_name, K):
    """gen(keys) (engine.dataset_state, dataset_state_kernel) at B = 1, 7 and 4 099, and on one unbatched key."""
    G, N = 10, 5
    gen, ds = _dataset(rbg, board_name, G, N, K)
    rks, starts, tgts = [], [], []
    for B in (1, 7, 4099):
        keys, kref = _keys(rbg, orc, K % 9973 + B, B)
        st = gen(keys)
        _assert_state(st, orc.dataset_state_batch(kref, G, N, *ds), f"(B={B})")
        rks.append(_split0(kref))
        starts.append(_np(st.agents.start))
        tgts.append(_np(st.agents.target))
    one = gen(rbg.PRNGKey(K))
    assert one.grid.shape == (G, G)
    k1 = orc.PRNGKey(K)[None]
    _assert_state(one.map(lambda t: t[None]), orc.dataset_state_batch(k1, G, N, *ds), "(one key)")
    _check_picks(np.concatenate(rks + [_split0(k1)]), np.concatenate(starts + [_np(one.agents.start)[None]]),
                 np.concatenate(tgts + [_np(one.agents.target)[None]]), ds, K)


@gpu
@pytest.mark.parametrize("board_name,K", DATASETS)
def test_connector_reset(rbg, board_name, K):
    """Connector.reset (rbg_connector_reset_dataset): State and restart TimeStep."""
    G, N, B = 10, 5, 1000
    gen, ds = _dataset(rbg, board_name, G, N, K)
    keys, kref = _keys(rbg, orc, K % 9973 + 1, B)
    st, ts = rbg.Connector(generator=gen, time_limit=1).reset(keys)
    rst = orc.dataset_state_batch(kref, G, N, *ds)
    _assert_state(st, rst)
    _assert_timestep(ts, orc.connector_observe_batch(rst))
    _check_picks(_split0(kref), _np(st.agents.start), _np(st.agents.target), ds, K)


@gpu
@pytest.mark.parametrize("board_name,K", DATASETS)
def test_autoreset_steps(rbg, board_name, K):
    """VmapAutoResetWrapper.step and step_random (env_warp_kernel) with time_limit 1: every env ends its episode and
    picks a board at every step, with key split(state.key)[0]."""
    G, N, B = 10, 5, 600
    gen, ds = _dataset(rbg, board_name, G, N, K)
    env = rbg.VmapAutoResetWrapper(rbg.Connector(generator=gen, time_limit=1))
    keys, kref = _keys(rbg, orc, K % 9973 + 2, B)
    st, _ = env.reset(keys)
    rst = orc.dataset_state_batch(kref, G, N, *ds)
    rng = np.random.default_rng(K)
    rks, starts, tgts = [], [], []
    for t in range(4):
        rks.append(_split0(_split0(rst["key"])))
        if t % 2:
            act = orc.random_actions_batch(rst)
            st, ts, got = env.step_random(st, inplace=t == 3)
            assert np.array_equal(_np(got), act), f"random actions differ at step {t}"
        else:
            act = rng.integers(0, 5, size=(B, N)).astype(np.int32)
            st, ts = env.step(st, rbg.engine.as_tensor(act), inplace=t == 2)
        rst, rts = orc.connector_step_batch(rst, act, time_limit=1, autoreset_kind="dataset", dataset=ds)
        assert (rts["step_type"] == 2).all()
        _assert_state(st, rst, f"at step {t}")
        _assert_timestep(ts, rts, f"at step {t}")
        starts.append(_np(st.agents.start))
        tgts.append(_np(st.agents.target))
    _check_picks(np.concatenate(rks), np.concatenate(starts), np.concatenate(tgts), ds, K)


ROLLOUT = ([("offline_parallel_rw", 10, 5, K) for K in KS]      # rollout_warp_kernel, observation staged in shared memory
           + [("offline_parallel_rw", 7, 3, K) for K in KS]  # cells % 4 != 0: the scalar rollout_warp_kernel<0>
           + [("offline_parallel_rw", 36, 1, K) for K in KS]     # more than 200 KB of shared memory: the step-wise fallback
           + [("offline_seed_extension", 10, 5, 100000)])


@gpu
@pytest.mark.parametrize("board_name,G,N,K", ROLLOUT)
def test_rollout(rbg, board_name, G, N, K):
    """rollout_random over 23 steps, across the 20-step launch chunk, with time_limit 1: every env picks a board at
    every step.  Every TimeStep leaf and the final State against the oracle, whose picks are checked at every step."""
    B, T = 160, 23
    gen, ds = _dataset(rbg, board_name, G, N, K, cache=(G, N) == (10, 5))
    env = rbg.VmapAutoResetWrapper(rbg.Connector(generator=gen, time_limit=1))
    keys, kref = _keys(rbg, orc, K % 9973 + G, B)
    st, _ = env.reset(keys)
    rst = orc.dataset_state_batch(kref, G, N, *ds)
    st, ts, act = env.rollout_random(st, T)
    rks, starts, tgts = [], [], []
    for t in range(T):
        rks.append(_split0(_split0(rst["key"])))
        a = orc.random_actions_batch(rst)
        assert np.array_equal(_np(act[t]), a), f"actions differ at step {t}"
        rst, rts = orc.connector_step_batch(rst, a, time_limit=1, autoreset_kind="dataset", dataset=ds)
        _assert_timestep(ts[t], rts, f"at step {t}")
        starts.append(rst["start"])
        tgts.append(rst["target"])
    _assert_state(st, rst, "after the rollout")
    _check_picks(np.concatenate(rks), np.concatenate(starts), np.concatenate(tgts), ds, K, "(oracle)")
    _check_picks(rks[-1], _np(st.agents.start), _np(st.agents.target), ds, K, "(after the rollout)")


@gpu
@pytest.mark.parametrize("board_name,K", DATASETS)
def test_evaluators(rbg, board_name, K):
    """RandomAgentEvaluator (engine.dataset_state) and PolicyEvaluator (Connector.reset): the boards the evaluator's
    reset takes, and the episode metrics against the oracle's episodes from the oracle's reset."""
    G, N, B, tl = 10, 5, 500, 5
    gen, ds = _dataset(rbg, board_name, G, N, K)
    env = rbg.Connector(generator=gen, time_limit=tl)
    keys, kref = _keys(rbg, orc, K % 9973 + 3, B)
    rst = orc.dataset_state_batch(kref, G, N, *ds)
    ev = rbg.RandomAgentEvaluator(env, B)
    s0 = ev._reset_state(keys)
    _assert_state(s0, rst, "(RandomAgentEvaluator reset)")
    _check_picks(_split0(kref), _np(s0.agents.start), _np(s0.agents.target), ds, K)
    ref, _ = oracle_episodes(orc, rst, tl)
    _assert_metrics(ev.episode_metrics(keys), ref, "RandomAgentEvaluator")
    pn, pt = POLICIES["keyed"]
    ref = oracle_policy_episodes(rbg, orc, rst, keys, pn, tl)
    _assert_metrics(rbg.PolicyEvaluator(env, pt, B).episode_metrics(keys), ref, "PolicyEvaluator")

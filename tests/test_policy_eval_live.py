"""Policy evaluation on the live envs only (rbg_connector_eval_step_live, engine.connector_eval_step_live,
PolicyEvaluator(live_only=True)) against the CPU oracle's plain Connector.step and against the default mode of
PolicyEvaluator.  Integers exactly, float32 by their bits.  Every test but the header check needs a CUDA device
(`-m gpu`).  The test policies and helpers are those of test_policy_eval.py."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from test_policy_eval import (BIG_SMEM_SHAPES, GENS, METRICS, POLICIES, SHAPES, STATE_FIELDS, _assert_metrics, _eq, _keys, _np, _state_gpu, _state_np,
                              greedy_torch, keyed_torch, oracle_policy_episodes)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_live_step_symbol_matches_header():
    """rbg_connector_eval_step_live has the header's number of parameters in the ctypes table."""
    import routing_board_generation_b200 as pkg

    with open(os.path.join(ROOT, "include", "rbg_b200.h")) as f:
        src = re.sub(r"/\*.*?\*/", "", f.read(), flags=re.S)
    params = re.search(r"int rbg_connector_eval_step_live\((.*?)\);", src, flags=re.S).group(1).split(",")
    assert len(pkg._lib.SYMBOLS["rbg_connector_eval_step_live"][1]) == len(params) == 13


def _obs_np(obs):
    return dict(obs=_np(obs.grid), action_mask=_np(obs.action_mask), obs_step_count=_np(obs.step_count))


# ------------------------------------------------------- the kernel, step by step
def _fits(G, N, B):  # the observation of the whole batch in at most 1 GB (int32), on the device and for the oracle
    return B * N * G * G <= 2**28


LIST_CASES = [(G, N, L) for G, N in SHAPES + BIG_SMEM_SHAPES for L in (1, 31, 33, 2048, 65536) if _fits(G, N, L + L // 4 + 3)]


@pytest.mark.gpu
@pytest.mark.parametrize("G,N,L", LIST_CASES)
@pytest.mark.parametrize("time_limit", [50, 3])
def test_live_step_matches_oracle(rbg, orc, G, N, L, time_limit):
    """From reset States, steps over arbitrary lists: the first an unsorted subset of the envs, then the survivors of
    the step before, shuffled or as compacted, with random (also illegal) actions.  At every step the listed envs' State
    and record equal the oracle's Connector.step of those envs, order_out / count_out list the survivors in list order,
    observation row r is survivor r's, and rows past the count, unlisted envs and the action buffer are untouched."""
    import torch

    B = L + L // 4 + 3
    seed = G * 1000 + N * 10 + L + time_limit
    rng = np.random.default_rng(seed)
    _, kref = _keys(rbg, orc, seed, B)
    s_ref = orc.state_batch("parallel_random_walk", kref, G, N)
    dev = torch.device("cuda")
    st = _state_gpu(rbg, s_ref)
    obs = rbg.engine.alloc_timestep(B, G, N).observation
    acc_ref = dict(episode_return=rng.integers(-40, 40, size=(B, N)).astype(np.float32) * np.float32(0.37), episode_length=rng.integers(0, 9, B).astype(np.int32),
                   num_connections=np.full(B, -5, np.int32), ratio_connections=np.full(B, -0.5, np.float32), total_path_length=np.full(B, -6, np.int32))
    acc = {k: rbg.engine.as_tensor(v) for k, v in acc_ref.items()}
    lst = rng.permutation(B)[:L].astype(np.int32)  # unsorted, and B - L envs never listed
    order_in = torch.full((B,), -9, dtype=torch.int32, device=dev)
    order_out = torch.full((B,), -9, dtype=torch.int32, device=dev)
    count = torch.full((1,), -1, dtype=torch.int32, device=dev)
    for step in range(4):
        Ls = lst.size
        if Ls == 0:
            break
        order_in[:Ls] = rbg.engine.as_tensor(lst)
        order_out.fill_(-9)
        for t, v in ((obs.grid, -7), (obs.action_mask, True), (obs.step_count, -3)):
            t.fill_(v)
        act = rng.integers(0, 5, size=(Ls, N)).astype(np.int32)
        action = torch.full((B, N), 77, dtype=torch.int32, device=dev)  # rows >= Ls are not the step's
        action[:Ls] = rbg.engine.as_tensor(act)
        act_before = _np(action)
        rs, rts = orc.connector_step_batch({k: v[lst] for k, v in s_ref.items()}, act, time_limit=time_limit, autoreset_kind=-1)
        rbg.engine.connector_eval_step_live(st, action[:Ls], order_in, Ls, order_out, count, acc, obs, time_limit=time_limit)

        for k in s_ref:
            s_ref[k][lst] = rs[k]
        last = rts["step_type"] == 2
        acc_ref["episode_return"][lst] = acc_ref["episode_return"][lst] + rts["reward"]
        acc_ref["episode_length"][lst] += 1
        for k in ("num_connections", "ratio_connections", "total_path_length"):
            acc_ref[k][lst[last]] = rts[k][last]
        where = f"(step {step}, L {Ls})"
        got_s = _state_np(st)
        for k in STATE_FIELDS:
            _eq(got_s[k], s_ref[k], f"state.{k} {where}")
        _assert_metrics(acc, acc_ref, where)
        surv = lst[~last]
        n = surv.size
        assert int(count.item()) == n, where
        got_order = _np(order_out)
        assert np.array_equal(got_order[:n], surv) and np.all(got_order[n:] == -9), f"order_out {where}"
        got_obs = _obs_np(obs)
        for k in ("obs", "action_mask", "obs_step_count"):
            _eq(got_obs[k][:n], rts[k][~last], f"observation.{k} {where}")
        assert np.all(got_obs["obs"][n:] == -7) and np.all(got_obs["action_mask"][n:] == 1) and np.all(got_obs["obs_step_count"][n:] == -3), f"rows past the count {where}"
        assert np.array_equal(_np(action), act_before), f"action {where}"
        lst = rng.permutation(surv).astype(np.int32) if step % 2 == 0 else surv
    if time_limit == 3:
        assert lst.size == 0  # every listed env ended at its third step


# ------------------------------------------------ the evaluator, both modes
def _check_live(rbg, orc, env, st_np, keys, policy, time_limit, where):
    """live_only=True equals the oracle's episodes and the default mode, bit for bit."""
    pn, pt = POLICIES[policy]
    got = rbg.PolicyEvaluator(env, pt, keys.shape[0], live_only=True).episode_metrics(keys)
    ref = oracle_policy_episodes(rbg, orc, st_np, keys, pn, time_limit)
    _assert_metrics(got, ref, f"{where} against the oracle")
    masked = rbg.PolicyEvaluator(env, pt, keys.shape[0]).episode_metrics(keys)
    _assert_metrics(got, {k: _np(v) for k, v in masked.items()}, f"{where} against the default mode")


@pytest.mark.gpu
@pytest.mark.parametrize("policy", list(POLICIES))
@pytest.mark.parametrize("kind", ["parallel_random_walk", "uniform"])
@pytest.mark.parametrize("G,N", SHAPES + BIG_SMEM_SHAPES)
@pytest.mark.parametrize("time_limit", [1, 7, 50])
def test_live_evaluator_matches_oracle_and_default(rbg, orc, policy, kind, G, N, time_limit):
    B = 2048 if G < 32 else 512
    keys, kref = _keys(rbg, orc, G * 100 + N + time_limit + 5, B)
    env = rbg.Connector(generator=getattr(rbg, GENS[kind])(G, N), time_limit=time_limit)
    _check_live(rbg, orc, env, orc.state_batch(kind, kref, G, N), keys, policy, time_limit, f"({policy} {kind} {G}x{G}/{N} time_limit {time_limit})")


@pytest.mark.gpu
@pytest.mark.parametrize("kind,G,N", [("seed_extension", 10, 5), ("sequential_random_walk", 16, 8)])
def test_live_evaluator_other_generators(rbg, orc, kind, G, N):
    keys, kref = _keys(rbg, orc, 80, 1500)
    env = rbg.Connector(generator=getattr(rbg, GENS[kind])(G, N), time_limit=50)
    _check_live(rbg, orc, env, orc.state_batch(kind, kref, G, N), keys, "keyed", 50, kind)


@pytest.mark.gpu
def test_live_evaluator_dataset_generator(rbg, orc):
    G, N, B = 10, 5, 1200
    gen = rbg.BoardDatasetGeneratorJAX(G, N, board_name="offline_parallel_rw", number_of_boards=37)
    keys, kref = _keys(rbg, orc, 81, B)
    st = orc.dataset_state_batch(kref, G, N, _np(gen.heads), _np(gen.targets))
    _check_live(rbg, orc, rbg.Connector(generator=gen, time_limit=30), st, keys, "greedy", 30, "dataset generator")


@pytest.mark.gpu
def test_live_evaluator_user_generator(rbg, orc):
    """A `Generator` subclass whose __call__ builds the reset State: two wires at key-dependent columns."""
    import torch

    G, N, B = 6, 2, 500

    class ColumnsGenerator(rbg.Generator):
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

    gen = ColumnsGenerator(G, N)
    keys, _ = _keys(rbg, orc, 82, B)
    _check_live(rbg, orc, rbg.Connector(generator=gen, time_limit=12), _state_np(gen(keys)), keys, "keyed", 12, "user generator")


@pytest.mark.gpu
@pytest.mark.parametrize("G,N,B", [(10, 5, 65536), (32, 16, 8192)])
def test_live_evaluator_full_size(rbg, orc, G, N, B):
    keys, kref = _keys(rbg, orc, 3, B)
    env = rbg.Connector(generator=rbg.ParallelRandomWalkGenerator(G, N), time_limit=50)
    _check_live(rbg, orc, env, orc.state_batch("parallel_random_walk", kref, G, N), keys, "keyed", 50, f"({G}x{G}/{N} x {B})")


# ---------------------------------------------------------- what the policy sees
@pytest.mark.gpu
@pytest.mark.parametrize("G,N,B,time_limit", [(10, 5, 3000, 50), (7, 6, 777, 9)])
def test_live_policy_sees_the_live_envs_in_env_order(rbg, orc, G, N, B, time_limit):
    """At every call the rows are exactly the envs still in their first episode, in ascending env order: each row (its
    observation and its action key, which is unique to the env and step) equals that env's row in the default mode at
    the same step; the batch sizes add up to the env-steps."""
    import torch

    keys, _ = _keys(rbg, orc, 83, B)
    env = rbg.Connector(generator=rbg.ParallelRandomWalkGenerator(G, N), time_limit=time_limit)

    def recorder(calls):
        def policy(obs, key):
            calls.append((obs.grid.clone(), obs.action_mask.clone(), obs.step_count.clone(), key.clone()))
            return keyed_torch(obs, key)
        return policy

    full, live = [], []
    ref = rbg.PolicyEvaluator(env, recorder(full), B).episode_metrics(keys)
    got = rbg.PolicyEvaluator(env, recorder(live), B, live_only=True).episode_metrics(keys)
    _assert_metrics(got, {k: _np(v) for k, v in ref.items()}, "(recording policy)")
    length = ref["episode_length"]
    assert len(live) == int(length.max())
    assert sum(c[0].shape[0] for c in live) == int(length.to(torch.int64).sum())
    for t, (grid, mask, sc, key) in enumerate(live):
        envs = torch.nonzero(length > t).flatten()  # live at call t, ascending
        g_all, m_all, s_all, k_all = full[t]
        assert grid.shape[0] == envs.numel() and key.shape == (envs.numel(), 2), f"call {t}"
        assert torch.equal(key.view(torch.int32), k_all.view(torch.int32)[envs]), f"action keys at call {t}"
        assert torch.equal(grid, g_all[envs]) and torch.equal(mask, m_all[envs]) and torch.equal(sc, s_all[envs]), f"observation at call {t}"


# ------------------------------------------------------------------ edge cases
@pytest.mark.gpu
def test_live_one_env_and_an_all_first_step_batch(rbg, orc):
    """B = 1; and with time_limit 1 every env ends at its first step, so the policy is called once."""
    G, N = 10, 5
    keys, kref = _keys(rbg, orc, 84, 1)
    env = rbg.Connector(generator=rbg.ParallelRandomWalkGenerator(G, N), time_limit=50)
    _check_live(rbg, orc, env, orc.state_batch("parallel_random_walk", kref, G, N), keys, "keyed", 50, "B = 1")

    calls = []

    def policy(obs, key):
        calls.append(obs.grid.shape[0])
        return greedy_torch(obs, key)

    B = 5000
    keys, kref = _keys(rbg, orc, 85, B)
    env1 = rbg.Connector(generator=rbg.UniformRandomGenerator(G, N), time_limit=1)
    got = rbg.PolicyEvaluator(env1, policy, B, live_only=True).episode_metrics(keys)
    assert calls == [B]
    assert bool((got["episode_length"] == 1).all())
    _assert_metrics(got, oracle_policy_episodes(rbg, orc, orc.state_batch("uniform", kref, G, N), keys, POLICIES["greedy"][0], 1), "time_limit 1")


@pytest.mark.gpu
def test_live_multi_to_single_sum_and_mean(rbg, orc):
    import torch

    G, N, B = 10, 5, 2048
    keys, _ = _keys(rbg, orc, 86, B)
    env = rbg.Connector(generator=rbg.ParallelRandomWalkGenerator(G, N), time_limit=50)
    multi = rbg.PolicyEvaluator(env, keyed_torch, B, live_only=True).episode_metrics(keys)
    total = rbg.PolicyEvaluator(rbg.MultiToSingleWrapper(env), keyed_torch, B, live_only=True).episode_metrics(keys)
    mean = rbg.PolicyEvaluator(rbg.MultiToSingleWrapper(env, reward_aggregator=torch.mean), keyed_torch, B, live_only=True).episode_metrics(keys)
    masked = rbg.PolicyEvaluator(rbg.MultiToSingleWrapper(env), keyed_torch, B).episode_metrics(keys)
    assert torch.equal(total["episode_return"], multi["episode_return"].sum(dim=-1))
    assert torch.equal(mean["episode_return"], multi["episode_return"].mean(dim=-1))
    for k in METRICS:
        assert torch.equal(total[k], masked[k]), k
    for k in METRICS[1:]:
        assert torch.equal(total[k], multi[k]) and torch.equal(mean[k], multi[k]), k


@pytest.mark.gpu
def test_live_single_key_and_run_evaluation(rbg):
    import torch

    G, N = 10, 5
    env = rbg.Connector(generator=rbg.ParallelRandomWalkGenerator(G, N), time_limit=50)
    ev = rbg.PolicyEvaluator(env, keyed_torch, 1, live_only=True)
    key = rbg.PRNGKey(6)
    one = ev.episode_metrics(key)
    assert tuple(one["episode_return"].shape) == (N,)
    batched = ev.episode_metrics(key[None])
    for k in METRICS:
        assert torch.equal(one[k], batched[k][0]), k

    B = 3000
    ev = rbg.PolicyEvaluator(rbg.MultiToSingleWrapper(rbg.Connector(generator=rbg.UniformRandomGenerator(G, N), time_limit=50)), greedy_torch, B, live_only=True)
    key = rbg.PRNGKey(4)
    means = ev.run_evaluation(key)
    per = ev.episode_metrics(rbg.split(key, B))
    default = rbg.PolicyEvaluator(ev.eval_env, greedy_torch, B).run_evaluation(key)
    assert sorted(means) == sorted(METRICS)
    for k in METRICS:
        assert torch.equal(means[k], per[k].to(torch.float32).mean(dim=0)), k
        assert torch.equal(means[k], default[k]), k


# ---------------------------------------------------------------- argument errors
@pytest.mark.gpu
def test_live_argument_errors(rbg, orc):
    """Each documented error, with no kernel launched and no buffer written."""
    import torch

    lib = rbg._lib.load()
    B, G, N = 8, 10, 5
    _, kref = _keys(rbg, orc, 1, B)
    s_np = orc.state_batch("parallel_random_walk", kref, G, N)
    st = _state_gpu(rbg, s_np)
    ts = rbg.engine.alloc_timestep(B, G, N)
    dev = st.grid.device
    s = rbg.engine._state_struct(st)
    o = ts.observation
    t = rbg._lib.rbg_timestep(o.grid.data_ptr(), o.action_mask.data_ptr(), o.step_count.data_ptr(), None, None, None, None, None, None)
    act = torch.zeros((B, N), dtype=torch.int32, device=dev)
    orders = torch.arange(2 * B, dtype=torch.int32, device=dev) % B
    oin, oout = orders[:B], orders[B:]
    count = torch.full((1,), -1, dtype=torch.int32, device=dev)
    bufs = [torch.zeros((B, N), dtype=torch.float32, device=dev)] + [torch.zeros(B, dtype=d, device=dev) for d in (torch.int32, torch.int32, torch.float32, torch.int32)]
    m = rbg._lib.rbg_episode_metrics(*(b.data_ptr() for b in bufs))
    ok = rbg._lib.rbg_env_params(50, -0.03, 0.1, -1)

    def call(s_=C.byref(s), a=act.data_ptr(), oi=oin.data_ptr(), L=B, oo=oout.data_ptr(), c=count.data_ptr(), Bx=B, Gx=G, Nx=N, p=C.byref(ok), t_=C.byref(t),
             m_=C.byref(m)):
        return lib.rbg_connector_eval_step_live(s_, a, oi, L, oo, c, Bx, Gx, Nx, p, t_, m_, None)

    torch.cuda.synchronize()
    launches = rbg.launch_count(reset=True)
    assert lib.rbg_connector_eval_step_live(None, None, None, 0, None, None, B, G, N, None, None, None, None) == 0  # an empty list
    errors = [
        (dict(L=-1), b"list length"), (dict(L=B + 1), b"list length"), (dict(Bx=-1, L=0), b"B="),
        (dict(s_=None), b"state"), (dict(a=None), b"action"), (dict(oi=None), b"order_in"), (dict(oo=None), b"order_out"), (dict(c=None), b"count_out"),
        (dict(oo=oin.data_ptr()), b"overlap"), (dict(oo=oin.data_ptr() + 4 * (B - 1)), b"overlap"), (dict(oi=oout.data_ptr() + 4), b"overlap"),
        (dict(p=None), b"params"), (dict(t_=None), b"timestep"), (dict(m_=None), b"acc"), (dict(Gx=41), b"grid size"), (dict(Nx=0), b"num_agents"),
    ]
    for kind in (0, 1, 2, 3, 4):
        errors.append((dict(p=C.byref(rbg._lib.rbg_env_params(50, -0.03, 0.1, kind))), b"autoreset_kind"))
    for field in ("obs_grid", "action_mask", "obs_step_count"):
        bad = rbg._lib.rbg_timestep(o.grid.data_ptr(), o.action_mask.data_ptr(), o.step_count.data_ptr(), None, None, None, None, None, None)
        setattr(bad, field, None)
        errors.append((dict(t_=C.byref(bad)), b"NULL observation"))
    for i in range(5):
        errors.append((dict(m_=C.byref(rbg._lib.rbg_episode_metrics(*(0 if j == i else b.data_ptr() for j, b in enumerate(bufs))))), b"NULL"))
    unaligned = rbg._lib.rbg_timestep(o.grid.data_ptr() + 4, o.action_mask.data_ptr(), o.step_count.data_ptr(), None, None, None, None, None, None)
    for kw, msg in errors:
        assert call(**kw) == -1, kw
        assert msg in lib.rbg_last_error(), (kw, lib.rbg_last_error())
    assert call(t_=C.byref(unaligned)) == -2 and b"aligned" in lib.rbg_last_error()
    assert rbg.launch_count(reset=True) == 0
    for k in STATE_FIELDS:
        _eq(_state_np(st)[k], s_np[k], f"state.{k}")
    assert all(int(b.abs().sum()) == 0 for b in bufs) and int(count.item()) == -1
    assert np.array_equal(_np(orders), np.arange(2 * B) % B)

    with pytest.raises(ValueError):  # the engine: int64 order buffers, a short list buffer
        rbg.engine.connector_eval_step_live(st, act, oin.to(torch.int64), B, oout, count, dict(zip(METRICS, bufs)), o)
    with pytest.raises(ValueError):
        rbg.engine.connector_eval_step_live(st, act, oin[:3], B, oout, count, dict(zip(METRICS, bufs)), o)
    assert call() == 0
    torch.cuda.synchronize()
    _, rts = orc.connector_step_batch(s_np, np.zeros((B, N), np.int32), time_limit=50, autoreset_kind=-1)
    assert int(count.item()) == int((rts["step_type"] != 2).sum())
    assert rbg.launch_count(reset=True) == 1

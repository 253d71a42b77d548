"""The host-buffer variants of the C-ABI against the oracle: rbg_connector_reset_host, rbg_connector_step_host,
rbg_connector_step_host_io and rbg_prw_generate_host.

These calls are more than a copy around the device calls.  Each one carves its device buffers out of one scratch per
device, cuts the batch into slices of a multiple of 64 envs (reset / generate: 4 slices from 4 096 envs on, step: 8,
step_host_io: 8, and 16 from 32 768 on) and runs the slices on the library's three streams, every slice copying in,
computing and copying out on its own stream, one cudaMemcpyAsync per leaf.  The step keeps one auto-reset workspace
per slice in that scratch from one call to the next, and a SeedExtension or SequentialRandomWalk reset runs the
generator pipelines of three slices at once.

Every host output buffer is filled with a sentinel before each call, so that a leaf that is not copied, or is copied
to the wrong place, cannot pass on an earlier call's values.  Every GPU matrix runs twice against the same oracle
results: with NumPy (pageable) buffers, whose copies the driver stages synchronously, and with pinned buffers from
rbg_host_alloc, whose copies really are asynchronous.  Integers are compared exactly, float32 values by their bits,
all 7 State and 9 TimeStep leaves at every call.  The argument checks return before any CUDA call and run without a
GPU.
"""
import ctypes as C

import numpy as np
import pytest

from test_connector_shapes import _rewards
from test_gpu_parity import PRW_CONFIGS, _np

SENTINEL = 0x7F
KINDS = {"parallel_random_walk": 0, "uniform": 1, "seed_extension": 2, "dataset": 3, "sequential_random_walk": 4}
STATE_LEAVES = ("grid", "step_count", "agent_id", "start", "target", "position", "key")  # rbg_state field order
TS_LEAVES = ("obs", "action_mask", "obs_step_count", "reward", "discount", "step_type", "num_connections", "ratio_connections",
             "total_path_length")  # rbg_timestep field order
MEMORIES = ("pageable", "pinned")


def _state_layout(G, N):
    return dict(grid=((G, G), np.int32), step_count=((), np.int32), agent_id=((N,), np.int32), start=((N, 2), np.int32),
                target=((N, 2), np.int32), position=((N, 2), np.int32), key=((2,), np.uint32))


def _ts_layout(G, N):
    return dict(obs=((N, G, G), np.int32), action_mask=((N, 5), np.uint8), obs_step_count=((), np.int32), reward=((N,), np.float32),
                discount=((N,), np.float32), step_type=((), np.int8), num_connections=((), np.int32), ratio_connections=((), np.float32),
                total_path_length=((), np.int32))


class HostBuffers:
    """Arrays in pageable (NumPy) or pinned (rbg_host_alloc) host memory; close() frees the pinned ones."""

    def __init__(self, lib, memory):
        self.lib, self.pinned, self._ptrs = lib, memory == "pinned", []

    def array(self, shape, dtype):
        if not self.pinned:
            return np.empty(shape, dtype)
        count = int(np.prod(shape))
        nbytes = max(count * np.dtype(dtype).itemsize, 1)
        p = self.lib.rbg_host_alloc(nbytes)
        assert p, self.lib.rbg_last_error()
        self._ptrs.append(p)
        return np.frombuffer((C.c_uint8 * nbytes).from_address(p), dtype=dtype, count=count).reshape(shape)

    def state(self, B, G, N):
        return {k: self.array((B, *s), d) for k, (s, d) in _state_layout(G, N).items()}

    def timestep(self, B, G, N):
        return {k: self.array((B, *s), d) for k, (s, d) in _ts_layout(G, N).items()}

    def close(self):
        for p in self._ptrs:
            self.lib.rbg_host_free(p)
        self._ptrs = []


@pytest.fixture
def host_mem(rbg):
    """host_mem(memory) -> HostBuffers; pinned buffers are freed when the test ends."""
    lib, made = rbg._lib.load(), []

    def make(memory):
        made.append(HostBuffers(lib, memory))
        return made[-1]

    yield make
    for hb in made:
        hb.close()


def _c_state(L, d):
    return L.rbg_state(*(d[k].ctypes.data for k in STATE_LEAVES))


def _c_ts(L, d):
    return L.rbg_timestep(*(d[k].ctypes.data for k in TS_LEAVES))


def _fill(bufs):
    for a in bufs.values():
        a.view(np.uint8).fill(SENTINEL)


def _untouched(bufs):
    return all((a.view(np.uint8) == SENTINEL).all() for a in bufs.values())


def _check(got, ref, leaves, prefix, where):
    """Every leaf bit for bit; a mismatch names the leaf, how many envs differ and the first of them."""
    for k in leaves:
        g, r = got[k], ref[k]
        assert g.shape == r.shape, f"{prefix}{k} has shape {g.shape}, the oracle {r.shape} {where}"
        if r.dtype == np.float32:
            g, r = g.view(np.uint32), r.view(np.uint32)
        bad = np.flatnonzero((g != r).reshape(len(g), -1).any(axis=1))
        assert bad.size == 0, f"{prefix}{k} differs {where}: {bad.size} of {len(g)} envs, the first at env {bad[0]}"


def _dataset(rbg, G, N, K):
    """BoardDatasetGeneratorJAX's K boards: the generator (its pins live on the device) and the pins on the host."""
    gen = rbg.BoardDatasetGeneratorJAX(G, N, board_name="offline_parallel_rw", number_of_boards=K)
    return gen, (_np(gen.heads), _np(gen.targets))


def _params(L, time_limit, kind, gen=None, reward=(-0.03, 0.1)):
    code = -1 if kind is None else KINDS[kind]
    if kind == "dataset":
        return L.rbg_env_params(time_limit, reward[0], reward[1], code, gen.heads.data_ptr(), gen.targets.data_ptr(), gen.heads.shape[0])
    return L.rbg_env_params(time_limit, reward[0], reward[1], code)


def _start_state(orc, kind, G, N, B, seed, ds):
    """The oracle's State after a reset with `kind`'s generator (ParallelRandomWalk for the plain step)."""
    kref = orc.split(orc.PRNGKey(seed), B)
    if kind == "dataset":
        return orc.dataset_state_batch(kref, G, N, *ds)
    return orc.state_batch(kind or "parallel_random_walk", kref, G, N)


def _trajectory(orc, rst, calls, time_limit, kind, ds, seed, reward=(-0.03, 0.1)):
    """[(action, State, TimeStep)] of `calls` oracle steps: the random policy, and every third step unconstrained codes
    in [-1, 7) (illegal moves, collisions, out-of-range codes)."""
    rng = np.random.default_rng(seed)
    B, N = rst["target"].shape[:2]
    out = []
    for t in range(calls):
        act = rng.integers(-1, 7, size=(B, N)).astype(np.int32) if t % 3 == 2 else orc.random_actions_batch(rst)
        rst, rts = orc.connector_step_batch(rst, act, time_limit=time_limit, timestep_reward=reward[0], connected_reward=reward[1],
                                            autoreset_kind=-1 if kind is None else kind, dataset=ds)
        out.append((act, rst, rts))
    return out


# ------------------------------------------------------------------ 1. rbg_connector_reset_host
RESET_KINDS = ("parallel_random_walk", "uniform", "seed_extension", "sequential_random_walk")
RESET_CASES = ([(kind, 10, 5, B) for kind in RESET_KINDS for B in (1, 65, 4095, 4096, 4097)]  # 1 slice, 4 even, 4 with a ragged last
               + [(kind, G, N, 4097) for kind in RESET_KINDS[:2] for G, N in ((5, 3), (20, 10), (40, 32), (20, 1))]  # 20x20/1: > 48 KB
               + [("seed_extension", 14, 7, 9000), ("sequential_random_walk", 3, 2, 4097), ("sequential_random_walk", 17, 9, 4097)])


@pytest.mark.gpu
@pytest.mark.parametrize("kind,G,N,B", RESET_CASES)
def test_reset_host(rbg, orc, host_mem, kind, G, N, B):
    """Connector(generator).reset from host keys into host State / TimeStep buffers."""
    L, lib = rbg._lib, rbg._lib.load()
    kref = orc.split(orc.PRNGKey(G * 1000 + N * 10 + B), B)
    rst, rts = orc.connector_reset_batch(kind, kref, G, N)
    for memory in MEMORIES:
        hb = host_mem(memory)
        keys = hb.array((B, 2), np.uint32)
        keys[:] = kref
        st, ts = hb.state(B, G, N), hb.timestep(B, G, N)
        _fill(st)
        _fill(ts)
        rc = lib.rbg_connector_reset_host(KINDS[kind], keys.ctypes.data, B, G, N, C.byref(_c_state(L, st)), C.byref(_c_ts(L, ts)), -1)
        assert rc == 0, lib.rbg_last_error()
        where = f"after reset_host ({kind}, {memory})"
        _check(st, rst, STATE_LEAVES, "state.", where)
        _check(ts, rts, TS_LEAVES, "timestep.", where)


@pytest.mark.gpu
def test_host_call_that_fails_part_way(rbg, orc, host_mem):
    """A SeedExtension reset or auto-reset that the generator refuses (10 agents, 9 seed cells on a 6x6 lattice) fails
    after the call has enqueued copies: it returns the generator's error, leaves every output buffer as it was, and the
    next call is right."""
    L, lib = rbg._lib, rbg._lib.load()
    G, N, B = 6, 10, 4097
    hb = host_mem("pinned")
    keys = hb.array((B, 2), np.uint32)
    keys[:] = orc.split(orc.PRNGKey(3), B)
    st, ts = hb.state(B, G, N), hb.timestep(B, G, N)
    _fill(st)
    _fill(ts)
    assert lib.rbg_connector_reset_host(KINDS["seed_extension"], keys.ctypes.data, B, G, N, C.byref(_c_state(L, st)), C.byref(_c_ts(L, ts)), -1) == -1
    assert b"lattice" in lib.rbg_last_error()
    assert _untouched(st) and _untouched(ts), "reset_host wrote its outputs although it failed"
    s0 = orc.state_batch("parallel_random_walk", keys, G, N)
    inp = hb.state(B, G, N)
    for k in STATE_LEAVES:
        inp[k][:] = s0[k]
    act = hb.array((B, N), np.int32)
    act[:] = orc.random_actions_batch(s0)
    params = _params(L, 1, "seed_extension")
    assert lib.rbg_connector_step_host(C.byref(_c_state(L, inp)), C.byref(_c_state(L, st)), act.ctypes.data, B, G, N, C.byref(params),
                                       C.byref(_c_ts(L, ts)), -1) == -1
    assert b"lattice" in lib.rbg_last_error()
    assert _untouched(st) and _untouched(ts), "step_host wrote its outputs although it failed"
    rc = lib.rbg_connector_reset_host(KINDS["parallel_random_walk"], keys.ctypes.data, B, G, N, C.byref(_c_state(L, st)), C.byref(_c_ts(L, ts)), -1)
    assert rc == 0, lib.rbg_last_error()
    rst, rts = orc.connector_reset_batch("parallel_random_walk", keys, G, N)
    _check(st, rst, STATE_LEAVES, "state.", "after the failed calls")
    _check(ts, rts, TS_LEAVES, "timestep.", "after the failed calls")


# ------------------------------------------------------------------ 2. rbg_connector_step_host
STEP_KINDS = [(None, 0), ("parallel_random_walk", 0), ("uniform", 0), ("seed_extension", 0), ("sequential_random_walk", 0), ("dataset", 7),
              ("dataset", 100000)]  # (auto-reset kind or None for the plain step, dataset boards)
STEP_CASES = ([(kind, K, tl, B) for kind, K in STEP_KINDS for tl in (1, 3) for B in (65, 4096, 4097)]  # 1 slice, 8 even, 8 with a ragged last
              + [("parallel_random_walk", 0, 1, 33000)])
CALLS = 6


def _step_host_run(rbg, lib, hb, s0, traj, B, G, N, params, where):
    """Steps `traj` with rbg_connector_step_host from State s0: out != in on even calls, in place on odd ones."""
    L = rbg._lib
    cur, other = hb.state(B, G, N), hb.state(B, G, N)
    for k in STATE_LEAVES:
        cur[k][:] = s0[k]
    ts, act = hb.timestep(B, G, N), hb.array((B, N), np.int32)
    for t, (a, rst, rts) in enumerate(traj):
        act[:] = a
        out = cur if t % 2 else other
        if out is not cur:
            _fill(out)
        _fill(ts)
        rc = lib.rbg_connector_step_host(C.byref(_c_state(L, cur)), C.byref(_c_state(L, out)), act.ctypes.data, B, G, N, C.byref(params),
                                         C.byref(_c_ts(L, ts)), -1)
        assert rc == 0, lib.rbg_last_error()
        w = f"at call {t} ({'in place' if out is cur else 'in != out'}) {where}"
        _check(out, rst, STATE_LEAVES, "state.", w)
        _check(ts, rts, TS_LEAVES, "timestep.", w)
        if out is not cur:
            cur, other = out, cur


@pytest.mark.gpu
@pytest.mark.parametrize("kind,K,time_limit,B", STEP_CASES)
def test_step_host(rbg, orc, host_mem, kind, K, time_limit, B):
    """Connector.step, or VmapAutoResetWrapper.step with each generator kind, on host State / action / TimeStep buffers:
    six consecutive calls (the per-slice workspaces carry over), with time limit 1 every env resets at every call."""
    L, lib = rbg._lib, rbg._lib.load()
    G, N = 10, 5
    gen, ds = _dataset(rbg, G, N, K) if kind == "dataset" else (None, None)
    s0 = _start_state(orc, kind, G, N, B, seed=B + time_limit, ds=ds)
    traj = _trajectory(orc, s0, CALLS, time_limit, kind, ds, seed=B)
    params = _params(L, time_limit, kind, gen)
    for memory in MEMORIES:
        _step_host_run(rbg, lib, host_mem(memory), s0, traj, B, G, N, params, f"({kind}, K={K}, {memory})")


@pytest.mark.gpu
def test_step_host_reward(rbg, orc, host_mem):
    """A DenseRewardFn of its own: both reward values occur, and the kernel used them."""
    L, lib = rbg._lib, rbg._lib.load()
    G, N, B, tl, reward = 10, 5, 4097, 3, (-0.7, 2.3)
    s0 = _start_state(orc, "uniform", G, N, B, seed=5, ds=None)
    traj = _trajectory(orc, s0, CALLS, tl, "uniform", None, seed=5, reward=reward)
    seen = np.array([_rewards(None, rts, reward) for _, _, rts in traj]).any(axis=0)
    assert seen.all(), "a timestep and a connected reward must both occur"
    params = _params(L, tl, "uniform", reward=reward)
    for memory in MEMORIES:
        _step_host_run(rbg, lib, host_mem(memory), s0, traj, B, G, N, params, f"(reward {reward}, {memory})")


@pytest.mark.gpu
def test_step_host_alternating_batches(rbg, orc, host_mem):
    """Two env batches of one shape stepped call by call (A, B, A, B ...): the signature does not change, so every call
    finds the other batch's per-slice next-episode caches, whose entries must only serve an env whose key they carry."""
    L, lib = rbg._lib, rbg._lib.load()
    G, N, B, tl = 10, 5, 4097, 2
    params = _params(L, tl, "parallel_random_walk")
    runs = []
    for i in range(2):
        s0 = _start_state(orc, "parallel_random_walk", G, N, B, seed=70 + i, ds=None)
        runs.append((s0, _trajectory(orc, s0, CALLS, tl, "parallel_random_walk", None, seed=70 + i)))
    for memory in MEMORIES:
        hb = host_mem(memory)
        bufs = []
        for s0, _ in runs:
            st = hb.state(B, G, N)
            for k in STATE_LEAVES:
                st[k][:] = s0[k]
            bufs.append((st, hb.timestep(B, G, N)))
        act = hb.array((B, N), np.int32)
        for t in range(CALLS):
            for i, ((st, ts), (_, traj)) in enumerate(zip(bufs, runs)):
                a, rst, rts = traj[t]
                act[:] = a
                _fill(ts)
                rc = lib.rbg_connector_step_host(C.byref(_c_state(L, st)), C.byref(_c_state(L, st)), act.ctypes.data, B, G, N, C.byref(params),
                                                 C.byref(_c_ts(L, ts)), -1)
                assert rc == 0, lib.rbg_last_error()
                where = f"at call {t} of batch {'AB'[i]} ({memory})"
                _check(st, rst, STATE_LEAVES, "state.", where)
                _check(ts, rts, TS_LEAVES, "timestep.", where)


# ------------------------------------------------------------------ 3. rbg_connector_step_host_io
IO_KINDS = [(None, 0), ("uniform", 0), ("seed_extension", 0), ("sequential_random_walk", 0), ("dataset", 100000)]
IO_SHAPES = [(10, 5), (14, 7)]  # observation codes <= 15 cross the bus as nibbles, larger ones as bytes
IO_CASES = ([(kind, K, tl, G, N, 4097) for kind, K in IO_KINDS for tl in (1, 3) for G, N in IO_SHAPES]  # 8 slices
            + [("seed_extension", 0, 1, 10, 5, 33001)])  # 16 slices


def _device_state(s0):
    """The State in device tensors (State.key as int32 bits), made on the default stream."""
    import torch

    return {k: torch.from_numpy(np.ascontiguousarray(v).view(np.int32) if v.dtype == np.uint32 else np.ascontiguousarray(v)).cuda()
            for k, v in s0.items()}


def _host_state(dst):
    return {k: _np(v).view(np.uint32) if k == "key" else _np(v) for k, v in dst.items()}


@pytest.mark.gpu
@pytest.mark.parametrize("kind,K,time_limit,G,N,B", IO_CASES)
def test_step_host_io(rbg, orc, host_mem, kind, K, time_limit, G, N, B):
    """Env-pool step: device State in place, host actions in, host TimeStep out, with every auto-reset kind; the byte
    counters say what crossed the bus."""
    L, lib = rbg._lib, rbg._lib.load()
    gen, ds = _dataset(rbg, G, N, K) if kind == "dataset" else (None, None)
    s0 = _start_state(orc, kind, G, N, B, seed=G + B + time_limit, ds=ds)
    traj = _trajectory(orc, s0, CALLS, time_limit, kind, ds, seed=G + B)
    params = _params(L, time_limit, kind, gen)
    obs_moved = B * N * G * G // (2 if 3 * N <= 15 and (N * G * G) % 2 == 0 else 1)
    for memory in MEMORIES:
        hb = host_mem(memory)
        dst = _device_state(s0)
        s = L.rbg_state(*(dst[k].data_ptr() for k in STATE_LEAVES))
        ts, act = hb.timestep(B, G, N), hb.array((B, N), np.int32)
        L.host_transfer_stats(reset=True)
        for t, (a, rst, rts) in enumerate(traj):
            act[:] = a
            _fill(ts)
            rc = lib.rbg_connector_step_host_io(C.byref(s), act.ctypes.data, B, G, N, C.byref(params), C.byref(_c_ts(L, ts)), -1)
            assert rc == 0, lib.rbg_last_error()
            where = f"at call {t} ({kind}, K={K}, {memory})"
            _check(_host_state(dst), rst, STATE_LEAVES, "state.", where)
            _check(ts, rts, TS_LEAVES, "timestep.", where)
        h2d, d2h, _ = L.host_transfer_stats()
        assert h2d == CALLS * B * N * 4 and d2h == CALLS * (obs_moved + B * (N * 5 + 4 + N * 8 + 1 + 12)), (h2d, d2h)


# ------------------------------------------------------------------ 4. call order across the shared scratch
def calls_in_turn(rbg, orc, memory):
    """All four host calls in turn on one device scratch: reset_host, step_host x3, step_host_io x2, prw_generate_host at
    a batch whose buffers outgrow the scratch (it is reallocated), step_host x2, reset_host with SeedExtension and
    step_host x2 with its auto-reset; every call against the oracle."""
    L, lib = rbg._lib, rbg._lib.load()
    G, N, B, tl = 10, 5, 4097, 2
    hb = HostBuffers(lib, memory)
    st, ts, act = hb.state(B, G, N), hb.timestep(B, G, N), hb.array((B, N), np.int32)
    keys = hb.array((B, 2), np.uint32)

    def reset(kind, seed):
        keys[:] = orc.split(orc.PRNGKey(seed), B)
        _fill(st)
        _fill(ts)
        rc = lib.rbg_connector_reset_host(KINDS[kind], keys.ctypes.data, B, G, N, C.byref(_c_state(L, st)), C.byref(_c_ts(L, ts)), -1)
        assert rc == 0, lib.rbg_last_error()
        rst, rts = orc.connector_reset_batch(kind, keys, G, N)
        _check(st, rst, STATE_LEAVES, "state.", f"after reset_host ({kind}, {memory})")
        _check(ts, rts, TS_LEAVES, "timestep.", f"after reset_host ({kind}, {memory})")
        return rst

    def step_host(rst, kind, calls, seed, tag):
        params = _params(L, tl, kind)
        for t, (a, rst, rts) in enumerate(_trajectory(orc, rst, calls, tl, kind, None, seed)):
            act[:] = a
            _fill(ts)
            rc = lib.rbg_connector_step_host(C.byref(_c_state(L, st)), C.byref(_c_state(L, st)), act.ctypes.data, B, G, N, C.byref(params),
                                             C.byref(_c_ts(L, ts)), -1)
            assert rc == 0, lib.rbg_last_error()
            _check(st, rst, STATE_LEAVES, "state.", f"at step_host call {t} {tag} ({memory})")
            _check(ts, rts, TS_LEAVES, "timestep.", f"at step_host call {t} {tag} ({memory})")
        return rst

    try:
        rst = reset("parallel_random_walk", 81)
        rst = step_host(rst, "parallel_random_walk", 3, 82, "after reset_host")
        dst = _device_state(rst)
        s = L.rbg_state(*(dst[k].data_ptr() for k in STATE_LEAVES))
        params = _params(L, tl, "parallel_random_walk")
        for t, (a, rst, rts) in enumerate(_trajectory(orc, rst, 2, tl, "parallel_random_walk", None, 83)):
            act[:] = a
            _fill(ts)
            rc = lib.rbg_connector_step_host_io(C.byref(s), act.ctypes.data, B, G, N, C.byref(params), C.byref(_c_ts(L, ts)), -1)
            assert rc == 0, lib.rbg_last_error()
            _check(_host_state(dst), rst, STATE_LEAVES, "state.", f"at step_host_io call {t} ({memory})")
            _check(ts, rts, TS_LEAVES, "timestep.", f"at step_host_io call {t} ({memory})")
        for k, v in _host_state(dst).items():
            st[k][:] = v
        # 65 536 boards take about 32 MB of device buffers, about three times what the calls above took
        B2 = 65536
        k2 = hb.array((B2, 2), np.uint32)
        k2[:] = orc.split(orc.PRNGKey(84), B2)
        gen = dict(heads=hb.array((B2, 2, N), np.int32), targets=hb.array((B2, 2, N), np.int32), solved=hb.array((B2, G, G), np.int32))
        _fill(gen)
        rc = lib.rbg_prw_generate_host(k2.ctypes.data, B2, G, N, gen["heads"].ctypes.data, gen["targets"].ctypes.data, gen["solved"].ctypes.data, -1)
        assert rc == 0, lib.rbg_last_error()
        rh, rt, rs, _ = orc.prw_generate_batch(k2, G, N)
        _check(gen, dict(heads=rh, targets=rt, solved=rs), ("heads", "targets", "solved"), "", f"after prw_generate_host ({memory})")
        step_host(rst, "parallel_random_walk", 2, 85, "after prw_generate_host")
        rst = reset("seed_extension", 86)
        step_host(rst, "seed_extension", 2, 87, "after the SeedExtension reset_host")
    finally:
        hb.close()


@pytest.mark.gpu
@pytest.mark.parametrize("memory", MEMORIES)
def test_host_calls_in_turn(rbg, memory):
    """calls_in_turn in a process of its own: the library's scratch only grows, so it starts empty there and the
    generate call really reallocates it."""
    import os
    import subprocess
    import sys

    here = os.path.dirname(os.path.abspath(__file__))
    code = (f"import sys; sys.path[:0] = [{os.path.dirname(here)!r}, {here!r}]\n"
            "import routing_board_generation_b200 as rbg, test_host_variants as t\n"
            "from oracle import oracle as orc\n"
            f"orc.build(); t.calls_in_turn(rbg, orc, {memory!r}); print('ok')\n")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and r.stdout.strip().endswith("ok"), (r.stdout[-800:], r.stderr[-2000:])


# ------------------------------------------------------------------ 5. rbg_prw_generate_host
@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, 4096, 4097])
@pytest.mark.parametrize("G,N", PRW_CONFIGS)
def test_prw_generate_host(rbg, orc, host_mem, G, N, B):
    """ParallelRandomWalkBoard.generate_board from host keys into host heads / targets / solved."""
    lib = rbg._lib.load()
    kref = orc.split(orc.PRNGKey(G * 100 + N + B), B)
    rh, rt, rs, _ = orc.prw_generate_batch(kref, G, N)
    ref = dict(heads=rh, targets=rt, solved=rs)
    for memory in MEMORIES:
        hb = host_mem(memory)
        keys = hb.array((B, 2), np.uint32)
        keys[:] = kref
        out = dict(heads=hb.array((B, 2, N), np.int32), targets=hb.array((B, 2, N), np.int32), solved=hb.array((B, G, G), np.int32))
        _fill(out)
        rc = lib.rbg_prw_generate_host(keys.ctypes.data, B, G, N, out["heads"].ctypes.data, out["targets"].ctypes.data, out["solved"].ctypes.data, -1)
        assert rc == 0, lib.rbg_last_error()
        _check(out, ref, ("heads", "targets", "solved"), "", f"after prw_generate_host ({memory})")


# ------------------------------------------------------------------ 6. argument contract (no GPU needed)
@pytest.fixture(scope="module")
def cabi():
    import __graft_entry__ as ge

    ge.build_library()
    import routing_board_generation_b200 as pkg

    return pkg._lib, pkg._lib.load()


def _arg_buffers(B, G, N):
    st = {k: np.zeros((B, *s), d) for k, (s, d) in _state_layout(G, N).items()}
    ts = {k: np.zeros((B, *s), d) for k, (s, d) in _ts_layout(G, N).items()}
    _fill(st)
    _fill(ts)
    return st, ts, np.zeros((B, 2), np.uint32), np.zeros((B, N), np.int32)


def test_host_variants_empty_batch(cabi):
    """B = 0 with every pointer NULL is an empty call that succeeds."""
    L, lib = cabi
    assert lib.rbg_prw_generate_host(None, 0, 10, 5, None, None, None, -1) == 0
    assert lib.rbg_connector_reset_host(0, None, 0, 10, 5, None, None, -1) == 0
    assert lib.rbg_connector_step_host(None, None, None, 0, 10, 5, None, None, -1) == 0
    assert lib.rbg_connector_step_host_io(None, None, 0, 10, 5, None, None, -1) == 0


def test_host_variants_null_arguments(cabi):
    """A NULL keys / State / TimeStep / params / action (or a State field) is RBG_EINVAL with a message."""
    L, lib = cabi
    B, G, N = 8, 10, 5
    st, ts, keys, act = _arg_buffers(B, G, N)
    s, t, p = C.byref(_c_state(L, st)), C.byref(_c_ts(L, ts)), C.byref(L.rbg_env_params(3, -0.03, 0.1, 0))
    k, a = keys.ctypes.data, act.ctypes.data
    h = np.zeros((B, 2, N), np.int32)
    for args in ((None, h.ctypes.data, h.ctypes.data, st["grid"].ctypes.data), (k, None, h.ctypes.data, st["grid"].ctypes.data),
                 (k, h.ctypes.data, None, st["grid"].ctypes.data), (k, h.ctypes.data, h.ctypes.data, None)):
        assert lib.rbg_prw_generate_host(args[0], B, G, N, *args[1:], -1) == -1 and b"NULL" in lib.rbg_last_error()
    for args in ((None, s, t), (k, None, t), (k, s, None)):
        assert lib.rbg_connector_reset_host(0, args[0], B, G, N, *args[1:], -1) == -1 and b"NULL" in lib.rbg_last_error()
    for args in ((None, s, a, p, t), (s, None, a, p, t), (s, s, None, p, t), (s, s, a, None, t), (s, s, a, p, None)):
        assert lib.rbg_connector_step_host(*args[:3], B, G, N, args[3], args[4], -1) == -1 and b"NULL" in lib.rbg_last_error()
    for args in ((None, a, p, t), (s, None, p, t), (s, a, None, t), (s, a, p, None)):
        assert lib.rbg_connector_step_host_io(args[0], args[1], B, G, N, *args[2:], -1) == -1 and b"NULL" in lib.rbg_last_error()
    holed = _c_state(L, st)
    holed.key = None
    assert lib.rbg_connector_step_host_io(C.byref(holed), a, B, G, N, p, t, -1) == -1 and b"NULL field" in lib.rbg_last_error()
    assert _untouched(st) and _untouched(ts)


@pytest.mark.parametrize("B,G,N,what", [(-1, 10, 5, b"B="), (2**30, 10, 5, b"too large"), (8, 1, 1, b"grid size"), (8, 41, 5, b"grid size"),
                                        (8, 10, 0, b"num_agents"), (8, 10, 33, b"num_agents"), (8, 2, 5, b"cells")])
def test_host_variants_reject_dimensions(cabi, B, G, N, what):
    """Out-of-range B, G and N (and more agents than cells) are RBG_EINVAL before any pointer is looked at."""
    L, lib = cabi
    p = C.byref(L.rbg_env_params(3, -0.03, 0.1, 0))
    for rc in (lib.rbg_prw_generate_host(None, B, G, N, None, None, None, -1), lib.rbg_connector_reset_host(0, None, B, G, N, None, None, -1),
               lib.rbg_connector_step_host(None, None, None, B, G, N, p, None, -1), lib.rbg_connector_step_host_io(None, None, B, G, N, p, None, -1)):
        assert rc == -1 and what in lib.rbg_last_error()


def test_uniform_reset_host_needs_two_cells_per_agent(cabi):
    """5 agents fit a 3x3 board for a random walk, not for the uniform generator's 2N distinct cells."""
    L, lib = cabi
    assert lib.rbg_connector_reset_host(KINDS["uniform"], None, 8, 3, 5, None, None, -1) == -1 and b"need 10 cells" in lib.rbg_last_error()


def test_host_variants_reject_kinds(cabi):
    """A reset kind the call cannot run (the dataset kind has no way to pass its boards here), an auto-reset kind above
    RBG_GEN_SEQRW and a dataset auto-reset without boards are RBG_EINVAL with a message, and no output is written."""
    L, lib = cabi
    B, G, N = 8, 10, 5
    st, ts, keys, act = _arg_buffers(B, G, N)
    s, t = C.byref(_c_state(L, st)), C.byref(_c_ts(L, ts))
    assert lib.rbg_connector_reset_host(KINDS["dataset"], keys.ctypes.data, B, G, N, s, t, -1) == -1
    assert b"RBG_GEN_DATASET" in lib.rbg_last_error()
    for kind in (-1, 5):
        assert lib.rbg_connector_reset_host(kind, keys.ctypes.data, B, G, N, s, t, -1) == -1
        assert f"unknown generator kind {kind}".encode() in lib.rbg_last_error()
    for params, what in ((L.rbg_env_params(3, -0.03, 0.1, 5), b"unknown autoreset generator kind 5"),
                         (L.rbg_env_params(3, -0.03, 0.1, 3), b"dataset_heads"),
                         (L.rbg_env_params(3, -0.03, 0.1, 3, act.ctypes.data, act.ctypes.data, 0), b"dataset_K=0")):
        assert lib.rbg_connector_step_host(s, s, act.ctypes.data, B, G, N, C.byref(params), t, -1) == -1 and what in lib.rbg_last_error()
        assert lib.rbg_connector_step_host_io(s, act.ctypes.data, B, G, N, C.byref(params), t, -1) == -1 and what in lib.rbg_last_error()
    assert _untouched(st) and _untouched(ts)

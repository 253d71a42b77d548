"""Batched functional layer over the C-ABI: torch CUDA tensors in / out.

Every function takes a leading batch axis B (the reference's vmap axis) and
launches on torch's current CUDA stream.  Arrays from other frameworks come in
through DLPack (`as_tensor`), results can go back out the same way
(`tensor.__dlpack__()` / `jax.dlpack.from_dlpack`).
"""
from __future__ import annotations

import ctypes as C
import itertools
import weakref
from typing import Dict, Optional, Tuple

import numpy as np
import torch

from . import _lib
from ._lib import GEN_DATASET, GEN_PRW, GEN_SEEDEXT, GEN_SEQRW, GEN_UNIFORM, rbg_env_params, rbg_state, rbg_timestep
from .types import Agent, Observation, State, TimeStep

GENERATOR_KINDS = {"parallel_random_walk": GEN_PRW, "uniform": GEN_UNIFORM, "seed_extension": GEN_SEEDEXT, "dataset": GEN_DATASET, "sequential_random_walk": GEN_SEQRW}


_cuda_checked = False


def _device() -> torch.device:
    global _cuda_checked
    if not _cuda_checked:  # checked once: the per-step API is called tens of thousands of times per second
        if not torch.cuda.is_available():
            raise RuntimeError("routing-board-generation_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        _cuda_checked = True
    return torch.device("cuda", torch.cuda.current_device())


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def _stream() -> int:
    if _raw_stream is not None:
        return _raw_stream(torch.cuda.current_device())
    return torch.cuda.current_stream().cuda_stream


def as_tensor(x, dtype: Optional[torch.dtype] = None) -> torch.Tensor:
    """torch tensor / DLPack producer (JAX, CuPy, ...) / NumPy / list -> contiguous CUDA tensor."""
    dev = _device()
    if isinstance(x, torch.Tensor):
        t = x
    elif hasattr(x, "__dlpack__"):
        t = torch.from_dlpack(x)
    else:
        a = np.asarray(x)
        if a.dtype == np.uint32:  # keep the bits, torch's uint32 host support is thin
            t = torch.from_numpy(a.view(np.int32).copy()).view(torch.uint32)
        else:
            t = torch.from_numpy(np.ascontiguousarray(a))
    if t.device != dev:
        t = t.to(dev, non_blocking=True)
    if dtype is not None and t.dtype != dtype:
        if dtype == torch.uint32 and t.dtype == torch.int32:
            t = t.view(torch.uint32)
        elif dtype == torch.int32 and t.dtype == torch.uint32:
            t = t.view(torch.int32)
        else:
            t = t.to(dtype)
    return t.contiguous()


def as_keys(key) -> Tuple[torch.Tensor, bool]:
    """Raw threefry keys uint32[2] or uint32[B,2] -> (uint32[B,2] on device, was_batched)."""
    t = as_tensor(key)
    if t.dtype == torch.int32:
        t = t.view(torch.uint32)
    elif t.dtype != torch.uint32:  # wider ints: keep the low 32 bits
        t = t.to(torch.int64).to(torch.int32).view(torch.uint32)
    if t.shape[-1] != 2 or t.dim() not in (1, 2):
        raise ValueError(f"PRNG key must have shape (2,) or (B, 2), got {tuple(t.shape)}")
    return t.reshape(-1, 2).contiguous(), t.dim() == 2


def PRNGKey(seed: int) -> torch.Tensor:
    """jax.random.PRNGKey(seed) for the threefry2x32 impl: (seed >> 32, seed & 0xffffffff)."""
    a = np.array([(int(seed) >> 32) & 0xFFFFFFFF, int(seed) & 0xFFFFFFFF], dtype=np.uint32)
    return as_tensor(a, torch.uint32)


def key_to_host(key) -> np.ndarray:
    t = key if isinstance(key, torch.Tensor) else as_tensor(key)
    return t.view(torch.int32).cpu().numpy().view(np.uint32)


def split(key, num: int = 2, offset: int = 0, count: Optional[int] = None) -> torch.Tensor:
    """Rows [offset, offset+count) of jax.random.split(key, num) as uint32[count,2] on the device."""
    k = key_to_host(key).reshape(-1)
    if k.shape != (2,):
        raise ValueError("split() takes a single key of shape (2,)")
    count = num - offset if count is None else count
    out = torch.empty((count, 2), dtype=torch.uint32, device=_device())
    karr = (C.c_uint32 * 2)(int(k[0]), int(k[1]))
    _lib.check(_lib.load().rbg_split_keys(karr, num, offset, count, out.data_ptr(), _stream()))
    return out


def split_each(keys: torch.Tensor, num: int = 2) -> torch.Tensor:
    """jax.vmap(lambda k: jax.random.split(k, num))(keys): uint32[B,2] -> uint32[B,num,2]."""
    keys, _ = as_keys(keys)
    out = torch.empty((keys.shape[0], num, 2), dtype=torch.uint32, device=_device())
    _lib.check(_lib.load().rbg_split_each(keys.data_ptr(), keys.shape[0], num, out.data_ptr(), _stream()))
    return out


def _env_params(time_limit, timestep_reward, connected_reward, autoreset_kind, dataset=None):
    """rbg_env_params; `dataset` = (heads int32[K,2,N], targets int32[K,2,N]) device tensors for kind "dataset".
    Returns (params, keepalive)."""
    if isinstance(autoreset_kind, str):
        autoreset_kind = GENERATOR_KINDS[autoreset_kind]
    p = rbg_env_params(int(time_limit), float(timestep_reward), float(connected_reward), int(autoreset_kind), None, None, 0)
    keep = None
    if autoreset_kind == GEN_DATASET:
        if dataset is None:
            raise ValueError("auto-reset with the dataset generator needs dataset=(heads, targets)")
        heads, targets = (as_tensor(t, torch.int32) for t in dataset)
        if heads.dim() != 3 or heads.shape[1] != 2 or heads.shape != targets.shape:
            raise ValueError(f"dataset heads / targets must be int32[K,2,N], got {tuple(heads.shape)} / {tuple(targets.shape)}")
        p.dataset_heads, p.dataset_targets, p.dataset_K = heads.data_ptr(), targets.data_ptr(), heads.shape[0]
        keep = (heads, targets)
    return p, keep


# ------------------------------------------------------------------ structs
def _state_struct(st: State) -> rbg_state:
    a = st.agents
    return rbg_state(st.grid.data_ptr(), st.step_count.data_ptr(), a.id.data_ptr(), a.start.data_ptr(), a.target.data_ptr(), a.position.data_ptr(), st.key.data_ptr())


def alloc_state(B: int, G: int, N: int) -> State:
    dev = _device()
    i32 = dict(dtype=torch.int32, device=dev)
    return State(
        key=torch.empty((B, 2), dtype=torch.uint32, device=dev),
        grid=torch.empty((B, G, G), **i32),
        step_count=torch.empty((B,), **i32),
        agents=Agent(id=torch.empty((B, N), **i32), start=torch.empty((B, N, 2), **i32), target=torch.empty((B, N, 2), **i32), position=torch.empty((B, N, 2), **i32)),
    )


def alloc_timestep(B: int, G: int, N: int, T: Optional[int] = None) -> TimeStep:
    """TimeStep buffers for a batch of B envs; with T, stacked [T, B, ...] (a rollout)."""
    dev = _device()
    lead = (B,) if T is None else (T, B)
    return TimeStep(
        step_type=torch.empty(lead, dtype=torch.int8, device=dev),
        reward=torch.empty(lead + (N,), dtype=torch.float32, device=dev),
        discount=torch.empty(lead + (N,), dtype=torch.float32, device=dev),
        observation=Observation(
            grid=torch.empty(lead + (N, G, G), dtype=torch.int32, device=dev),
            action_mask=torch.empty(lead + (N, 5), dtype=torch.bool, device=dev),
            step_count=torch.empty(lead, dtype=torch.int32, device=dev),
        ),
        extras={
            "num_connections": torch.empty(lead, dtype=torch.int32, device=dev),
            "ratio_connections": torch.empty(lead, dtype=torch.float32, device=dev),
            "total_path_length": torch.empty(lead, dtype=torch.int32, device=dev),
        },
    )


def _timestep_struct(ts: TimeStep) -> rbg_timestep:
    o, x = ts.observation, ts.extras
    return rbg_timestep(o.grid.data_ptr(), o.action_mask.data_ptr(), o.step_count.data_ptr(), ts.reward.data_ptr(), ts.discount.data_ptr(), ts.step_type.data_ptr(), x["num_connections"].data_ptr(), x["ratio_connections"].data_ptr(), x["total_path_length"].data_ptr())


def _dims(st: State) -> Tuple[int, int, int]:
    B, G, _ = st.grid.shape
    return B, G, st.agents.id.shape[1]


def _contig_state(st: State) -> State:
    a = st.agents
    if (st.grid.is_contiguous() and st.step_count.is_contiguous() and st.key.is_contiguous() and a.id.is_contiguous() and a.start.is_contiguous()
            and a.target.is_contiguous() and a.position.is_contiguous()):
        return st
    return st.map(lambda t: t if t.is_contiguous() else t.contiguous())


# --------------------------------------------------------------- generators
def prw_generate(keys: torch.Tensor, G: int, N: int, with_stats: bool = False):
    """ParallelRandomWalkBoard.generate_board over keys[B,2] -> heads[B,2,N], targets[B,2,N], solved[B,G,G]."""
    B = keys.shape[0]
    dev = _device()
    heads = torch.empty((B, 2, N), dtype=torch.int32, device=dev)
    targets = torch.empty((B, 2, N), dtype=torch.int32, device=dev)
    solved = torch.empty((B, G, G), dtype=torch.int32, device=dev)
    stats = torch.empty((B, 2), dtype=torch.int32, device=dev) if with_stats else None
    _lib.check(_lib.load().rbg_prw_generate(keys.data_ptr(), B, G, N, heads.data_ptr(), targets.data_ptr(), solved.data_ptr(), stats.data_ptr() if with_stats else None, _stream()))
    return (heads, targets, solved, stats) if with_stats else (heads, targets, solved)


def generator_state(kind, keys: torch.Tensor, G: int, N: int, out: Optional[State] = None) -> State:
    kind = GENERATOR_KINDS[kind] if isinstance(kind, str) else kind
    B = keys.shape[0]
    st = alloc_state(B, G, N) if out is None else out
    s = _state_struct(st)
    _lib.check(_lib.load().rbg_generator_state(kind, keys.data_ptr(), B, G, N, C.byref(s), _stream()))
    return st


def dataset_state(keys: torch.Tensor, G: int, N: int, heads: torch.Tensor, targets: torch.Tensor) -> State:
    """BoardDatasetGeneratorJAX.__call__ over keys[B,2]: pick one of the K stored boards per key."""
    B = keys.shape[0]
    st = alloc_state(B, G, N)
    s = _state_struct(st)
    _lib.check(_lib.load().rbg_dataset_state(keys.data_ptr(), B, G, N, heads.data_ptr(), targets.data_ptr(), heads.shape[0], C.byref(s), _stream()))
    return st


def seedext_solved(keys: torch.Tensor, G: int, N: int, randomness: float = 0.0, two_sided: bool = True, iterations: int = 1, extension_steps: float = 1e23) -> torch.Tensor:
    B = keys.shape[0]
    solved = torch.empty((B, G, G), dtype=torch.int32, device=_device())
    steps = -1 if extension_steps >= 2**62 else int(extension_steps)
    _lib.check(_lib.load().rbg_seedext_solved(keys.data_ptr(), B, G, N, float(randomness), int(bool(two_sided)), int(iterations), steps, solved.data_ptr(), _stream()))
    return solved


def seedext_starts_ends(keys: torch.Tensor, G: int, N: int, randomness: float = 0.0, two_sided: bool = True, iterations: int = 1, extension_steps: float = 1e23):
    B = keys.shape[0]
    dev = _device()
    starts = torch.empty((B, 2, N), dtype=torch.int32, device=dev)
    ends = torch.empty((B, 2, N), dtype=torch.int32, device=dev)
    steps = -1 if extension_steps >= 2**62 else int(extension_steps)
    _lib.check(_lib.load().rbg_seedext_starts_ends(keys.data_ptr(), B, G, N, float(randomness), int(bool(two_sided)), int(iterations), steps, starts.data_ptr(), ends.data_ptr(), _stream()))
    return starts, ends


def seqrw_generate(keys: torch.Tensor, G: int, N: int, as_float32: bool = True, with_stats: bool = False):
    """SequentialRandomWalkBoard.generate over keys[B,2] -> board[B,G,G] (float32 codes like the reference, or int32);
    with_stats adds int32[B,2] = (attempt that succeeded, 0 = none: zero board; steps of that attempt)."""
    B = keys.shape[0]
    dev = _device()
    board = torch.empty((B, G, G), dtype=torch.float32 if as_float32 else torch.int32, device=dev)
    stats = torch.empty((B, 2), dtype=torch.int32, device=dev) if with_stats else None
    _lib.check(_lib.load().rbg_seqrw_generate(keys.data_ptr(), B, G, N, board.data_ptr(), int(bool(as_float32)), stats.data_ptr() if with_stats else None, _stream()))
    return (board, stats) if with_stats else board


def seqrw_starts_ends(keys: torch.Tensor, G: int, N: int):
    B = keys.shape[0]
    dev = _device()
    starts = torch.empty((B, 2, N), dtype=torch.int32, device=dev)
    ends = torch.empty((B, 2, N), dtype=torch.int32, device=dev)
    _lib.check(_lib.load().rbg_seqrw_starts_ends(keys.data_ptr(), B, G, N, starts.data_ptr(), ends.data_ptr(), _stream()))
    return starts, ends


def validate(boards: torch.Tensor, N: int) -> torch.Tensor:
    boards = as_tensor(boards, torch.int32)
    if boards.dim() == 2:
        boards = boards[None]
    B, G, _ = boards.shape
    flags = torch.empty((B,), dtype=torch.int32, device=_device())
    _lib.check(_lib.load().rbg_validate(boards.data_ptr(), B, G, N, flags.data_ptr(), _stream()))
    return flags


def board_statistics(boards: torch.Tensor, count_current_wire: bool = False, with_scores: bool = True):
    """EvaluateEmptyBoard over boards[B,G,G] (or [G,G]): (scored[B,G,G] or None, count_detours[B], heatmap_score_diversity[B])."""
    boards = as_tensor(boards, torch.int32)
    single = boards.dim() == 2
    if single:
        boards = boards[None]
    B, G, _ = boards.shape
    dev = _device()
    scored = torch.empty((B, G, G), dtype=torch.int32, device=dev) if with_scores else None
    det = torch.empty((B,), dtype=torch.int32, device=dev)
    div = torch.empty((B,), dtype=torch.int32, device=dev)
    _lib.check(_lib.load().rbg_board_statistics(boards.data_ptr(), B, G, int(bool(count_current_wire)), scored.data_ptr() if with_scores else None, det.data_ptr(), div.data_ptr(), _stream()))
    if single:
        return (scored[0] if with_scores else None), det[0], div[0]
    return scored, det, div


# ---------------------------------------------------------------- connector
def connector_observe(st: State, out: Optional[TimeStep] = None) -> TimeStep:
    st = _contig_state(st)
    B, G, N = _dims(st)
    ts = alloc_timestep(B, G, N) if out is None else out
    s, t = _state_struct(st), _timestep_struct(ts)
    _lib.check(_lib.load().rbg_connector_observe(C.byref(s), B, G, N, C.byref(t), _stream()))
    return ts


def connector_reset(kind, keys: torch.Tensor, G: int, N: int, dataset=None) -> Tuple[State, TimeStep]:
    kind = GENERATOR_KINDS[kind] if isinstance(kind, str) else kind
    B = keys.shape[0]
    st, ts = alloc_state(B, G, N), alloc_timestep(B, G, N)
    s, t = _state_struct(st), _timestep_struct(ts)
    if kind == GEN_DATASET:
        heads, targets = (as_tensor(x, torch.int32) for x in dataset)
        _lib.check(_lib.load().rbg_connector_reset_dataset(keys.data_ptr(), B, G, N, heads.data_ptr(), targets.data_ptr(), heads.shape[0], C.byref(s), C.byref(t), _stream()))
    else:
        _lib.check(_lib.load().rbg_connector_reset(kind, keys.data_ptr(), B, G, N, C.byref(s), C.byref(t), _stream()))
    return st, ts


_workspaces: Dict[Tuple, torch.Tensor] = {}
_ws_tokens = itertools.count(1)


def _workspace(B: int, G: int, N: int, owner=None) -> torch.Tensor:
    """Auto-reset scratch (reset lists + the next-episode cache) of one env batch.  Keyed by the
    owning wrapper when there is one, so two batches of the same shape do not evict each other's
    cache entries; kept alive for the process (kernels queued on the stream may still be filling it
    when the caller drops its last State)."""
    dev = _device()
    token = None
    if owner is not None:  # id(owner) can be reused by a later env: give every owner its own token
        token = getattr(owner, "_rbg_ws_token", None)
        if token is None:
            token = next(_ws_tokens)
            try:
                owner._rbg_ws_token = token
            except AttributeError:
                token = ("id", id(owner))
    k = (dev.index, B, G, N, token)
    if k not in _workspaces:
        nbytes = int(_lib.load().rbg_step_workspace_bytes(B, G, N))
        _workspaces[k] = torch.empty((nbytes + 15) // 16 * 16, dtype=torch.uint8, device=dev)
        if owner is not None and not isinstance(token, tuple):
            weakref.finalize(owner, _drop_workspace, k).atexit = False  # nothing to release once the process is exiting
    return _workspaces[k]


def _drop_workspace(k) -> None:
    """The owning env is gone: let the library forget the workspace (waits for the work queued on it) and free it."""
    ws = _workspaces.pop(k, None)
    if ws is not None:
        try:
            _lib.load().rbg_workspace_release(ws.data_ptr())
        except Exception:
            pass


def connector_step(st: State, action, time_limit: int = 50, timestep_reward: float = -0.03, connected_reward: float = 0.1, autoreset_kind=-1, inplace: bool = False, random_policy: bool = False, out: Optional[TimeStep] = None, owner=None, dataset=None):
    """Connector.step (autoreset_kind < 0) or VmapAutoResetWrapper(Connector).step over a batch.

    random_policy=True ignores `action`, samples the uniform-over-legal-actions policy in the
    same launch and returns the sampled actions as a third value.
    """
    if isinstance(autoreset_kind, str):
        autoreset_kind = GENERATOR_KINDS[autoreset_kind]
    st = _contig_state(st)
    B, G, N = _dims(st)
    new = st if inplace else alloc_state(B, G, N)
    ts = alloc_timestep(B, G, N) if out is None else out
    params, _keep = _env_params(time_limit, timestep_reward, connected_reward, autoreset_kind, dataset)
    ws = _workspace(B, G, N, owner) if 0 <= autoreset_kind != GEN_DATASET else None
    s_in, s_out, t = _state_struct(st), _state_struct(new), _timestep_struct(ts)
    lib = _lib.load()
    if random_policy:
        act = torch.empty((B, N), dtype=torch.int32, device=_device())
        _lib.check(lib.rbg_connector_step_random(C.byref(s_in), C.byref(s_out), act.data_ptr(), B, G, N, C.byref(params), C.byref(t), ws.data_ptr() if ws is not None else None, _stream()))
        return new, ts, act
    act = as_tensor(action, torch.int32).reshape(B, N)
    _lib.check(lib.rbg_connector_step(C.byref(s_in), C.byref(s_out), act.data_ptr(), B, G, N, C.byref(params), C.byref(t), ws.data_ptr() if ws is not None else None, _stream()))
    return new, ts


def connector_rollout_random(st: State, n_steps: int, time_limit: int = 50, timestep_reward: float = -0.03, connected_reward: float = 0.1, autoreset_kind="parallel_random_walk", out: Optional[TimeStep] = None, actions: Optional[torch.Tensor] = None, owner=None, dataset=None):
    """n_steps auto-reset random-policy steps in ONE library call (the reference's `n_steps` scan).
    `st` is updated in place; returns (st, TimeStep stacked [n_steps, B, ...], actions[n_steps, B, N])."""
    if isinstance(autoreset_kind, str):
        autoreset_kind = GENERATOR_KINDS[autoreset_kind]
    B, G, N = _dims(st)
    for t in (st.grid, st.step_count, st.key, st.agents.id, st.agents.start, st.agents.target, st.agents.position):
        if not t.is_contiguous():
            raise ValueError("rollout updates the State in place: its leaves must be contiguous")
    ts = alloc_timestep(B, G, N, n_steps) if out is None else out
    act = torch.empty((n_steps, B, N), dtype=torch.int32, device=_device()) if actions is None else actions
    params, _keep = _env_params(time_limit, timestep_reward, connected_reward, autoreset_kind, dataset)
    ws = _workspace(B, G, N, owner) if autoreset_kind != GEN_DATASET else None
    s, t = _state_struct(st), _timestep_struct(ts)
    _lib.check(_lib.load().rbg_connector_rollout_random(C.byref(s), act.data_ptr(), n_steps, B, G, N, C.byref(params), C.byref(t), ws.data_ptr() if ws is not None else None, _stream()))
    return st, ts, act


def random_actions(st: State) -> torch.Tensor:
    st = _contig_state(st)
    B, G, N = _dims(st)
    act = torch.empty((B, N), dtype=torch.int32, device=_device())
    s = _state_struct(st)
    _lib.check(_lib.load().rbg_random_actions(C.byref(s), B, G, N, act.data_ptr(), _stream()))
    return act

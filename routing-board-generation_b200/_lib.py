"""ctypes binding of librbg_b200.so (the C-ABI in include/rbg_b200.h).

There is no CPU path: if the shared library is missing or no CUDA device is
usable, calls raise -- they never fall back to the oracle or to eager torch.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("RBG_B200_LIB") or os.path.join(_HERE, "lib", "librbg_b200.so")  # override: A/B builds of the same CUDA library

GEN_PRW, GEN_UNIFORM, GEN_SEEDEXT, GEN_DATASET, GEN_SEQRW = 0, 1, 2, 3, 4
MAX_G, MAX_N = 40, 32


class RbgError(RuntimeError):
    """A C-ABI call returned a negative RBG_E* code."""

    def __init__(self, code: int, message: str):
        super().__init__(f"librbg_b200 error {code}: {message}")
        self.code = code


class rbg_state(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("grid", "step_count", "agent_id", "start", "target", "position", "key")]


class rbg_timestep(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("obs_grid", "action_mask", "obs_step_count", "reward", "discount", "step_type", "num_connections", "ratio_connections", "total_path_length")]


class rbg_env_params(C.Structure):
    _fields_ = [("time_limit", C.c_int32), ("timestep_reward", C.c_float), ("connected_reward", C.c_float), ("autoreset_kind", C.c_int32),
                ("dataset_heads", C.c_void_p), ("dataset_targets", C.c_void_p), ("dataset_K", C.c_int64)]


class rbg_episode_metrics(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("episode_return", "episode_length", "num_connections", "ratio_connections", "total_path_length")]


# every symbol include/rbg_b200.h declares: (restype, argtypes)
_vp, _i64, _int, _f = C.c_void_p, C.c_int64, C.c_int, C.c_float
_SP, _TP, _EP, _MP = C.POINTER(rbg_state), C.POINTER(rbg_timestep), C.POINTER(rbg_env_params), C.POINTER(rbg_episode_metrics)
SYMBOLS = {
    "rbg_version": (_int, []),
    "rbg_last_error": (C.c_char_p, []),
    "rbg_device_info": (_int, [C.POINTER(_int), C.POINTER(_int)]),
    "rbg_split_keys": (_int, [C.POINTER(C.c_uint32), _i64, _i64, _i64, _vp, _vp]),
    "rbg_prw_generate": (_int, [_vp, _i64, _int, _int, _vp, _vp, _vp, _vp, _vp]),
    "rbg_generator_state": (_int, [_int, _vp, _i64, _int, _int, _SP, _vp]),
    "rbg_dataset_state": (_int, [_vp, _i64, _int, _int, _vp, _vp, _i64, _SP, _vp]),
    "rbg_connector_reset_dataset": (_int, [_vp, _i64, _int, _int, _vp, _vp, _i64, _SP, _TP, _vp]),
    "rbg_split_each": (_int, [_vp, _i64, _int, _vp, _vp]),
    "rbg_seedext_solved": (_int, [_vp, _i64, _int, _int, _f, _int, _int, _i64, _vp, _vp]),
    "rbg_seedext_starts_ends": (_int, [_vp, _i64, _int, _int, _f, _int, _int, _i64, _vp, _vp, _vp]),
    "rbg_seqrw_generate": (_int, [_vp, _i64, _int, _int, _vp, _int, _vp, _vp]),
    "rbg_seqrw_starts_ends": (_int, [_vp, _i64, _int, _int, _vp, _vp, _vp]),
    "rbg_connector_observe": (_int, [_SP, _i64, _int, _int, _TP, _vp]),
    "rbg_connector_reset": (_int, [_int, _vp, _i64, _int, _int, _SP, _TP, _vp]),
    "rbg_step_workspace_bytes": (_i64, [_i64, _int, _int]),
    "rbg_workspace_release": (_int, [_vp]),
    "rbg_connector_step": (_int, [_SP, _SP, _vp, _i64, _int, _int, _EP, _TP, _vp, _vp]),
    "rbg_random_actions": (_int, [_SP, _i64, _int, _int, _vp, _vp]),
    "rbg_connector_step_random": (_int, [_SP, _SP, _vp, _i64, _int, _int, _EP, _TP, _vp, _vp]),
    "rbg_connector_rollout_random": (_int, [_SP, _vp, _i64, _i64, _int, _int, _EP, _TP, _vp, _vp]),
    "rbg_connector_episodes_random": (_int, [_SP, _i64, _int, _int, _EP, _MP, _SP, _vp]),
    "rbg_connector_eval_step": (_int, [_SP, _vp, _vp, _vp, _i64, _int, _int, _EP, _TP, _MP, _vp]),
    "rbg_validate": (_int, [_vp, _i64, _int, _int, _vp, _vp]),
    "rbg_board_statistics": (_int, [_vp, _i64, _int, _int, _vp, _vp, _vp, _vp]),
    "rbg_prw_generate_host": (_int, [_vp, _i64, _int, _int, _vp, _vp, _vp, _int]),
    "rbg_connector_reset_host": (_int, [_int, _vp, _i64, _int, _int, _SP, _TP, _int]),
    "rbg_connector_step_host": (_int, [_SP, _SP, _vp, _i64, _int, _int, _EP, _TP, _int]),
    "rbg_connector_step_host_io": (_int, [_SP, _vp, _i64, _int, _int, _EP, _TP, _int]),
    "rbg_host_widen": (_int, [_vp, _vp, _i64]),
    "rbg_host_widen4": (_int, [_vp, _vp, _i64]),
    "rbg_host_transfer_stats": (_int, [C.POINTER(_i64), C.POINTER(_i64), C.POINTER(_int), _int]),
    "rbg_host_alloc": (_vp, [_i64]),
    "rbg_host_free": (None, [_vp]),
    "rbg_launch_count": (_i64, [_int]),
    "rbg_kernel_timing": (_int, [_int]),
    "rbg_kernel_time": (_int, [_int, C.POINTER(_i64), C.POINTER(C.c_double)]),
}

_lib = None


def load() -> C.CDLL:
    """Load the in-tree shared library; fail loudly when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise ImportError(
                f"{SO_PATH} is missing: build it with `python routing-board-generation_b200/build.py` "
                "(or __graft_entry__.build()). There is no CPU fallback."
            )
        lib = C.CDLL(SO_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(lib, name)  # AttributeError if the .so lacks a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc: int) -> None:
    if rc != 0:
        raise RbgError(rc, load().rbg_last_error().decode("utf-8", "replace"))


def launch_count(reset: bool = False) -> int:
    return int(load().rbg_launch_count(1 if reset else 0))


KERNELS = {"prw": 0, "env": 1, "random_actions": 2, "split": 3, "validate": 4, "seedext": 5, "rollout": 6, "seqrw": 7, "episodes": 8, "eval_step": 9}


def kernel_timing(enable: bool) -> None:
    check(load().rbg_kernel_timing(1 if enable else 0))


def kernel_time(kernel) -> tuple:
    """(launches, total device ms) of one kernel since the last call; synchronises on its events."""
    kid = KERNELS[kernel] if isinstance(kernel, str) else int(kernel)
    n, ms = _i64(0), C.c_double(0.0)
    check(load().rbg_kernel_time(kid, C.byref(n), C.byref(ms)))
    return int(n.value), float(ms.value)


def host_transfer_stats(reset: bool = False) -> tuple:
    """(H2D bytes, D2H bytes, host widening threads) of the _host_io calls since the last reset."""
    a, b, t = _i64(0), _i64(0), _int(0)
    check(load().rbg_host_transfer_stats(C.byref(a), C.byref(b), C.byref(t), 1 if reset else 0))
    return int(a.value), int(b.value), int(t.value)

"""ctypes binding of include/manytor_b200.h.

The library is the product: if it is missing, or there is no sm_100 device, the
calls below raise -- there is no CPU fallback anywhere in this package.
"""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

MT_MAX_JOINTS = 8
MT_MAX_OBJ = 32
MT_STATS_WORDS = 8
MT_ABI_VERSION = 3
MT_OBS_F32 = 0
MT_OBS_F16 = 1
MT_STEP_INDEX_MAX = 1 << 62

STATS_FIELDS = ("env_steps", "episodes", "terminated", "reward_sum", "length_sum", "catches",
                "ground_steps", "live_reward_sum")


class MtConfig(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32),
        ("device", C.c_int32),
        ("n_envs", C.c_int64),
        ("env_id_base", C.c_int64),
        ("n_joints", C.c_int32),
        ("n_obj", C.c_int32),
        ("dh", (C.c_float * 4) * MT_MAX_JOINTS),
        ("obs_frame", C.c_int32),
        ("ground_frame_a", C.c_int32),
        ("ground_frame_b", C.c_int32),
        ("catch_frame", C.c_int32),
        ("radius", C.c_float),
        ("catch_tol", C.c_float),
        ("substeps", C.c_int32),
        ("horizon", C.c_int32),
        ("terminate_on_ground", C.c_int32),
        ("auto_reset", C.c_int32),
        ("obs_after_reset", C.c_int32),
        ("fk_mode", C.c_int32),
        ("action_low", C.c_int32),
        ("action_high", C.c_int32),
        ("seed", C.c_uint64),
        ("obs_dtype", C.c_int32),
    ]


class MtStats(C.Structure):
    _fields_ = [(name, C.c_int64) for name in STATS_FIELDS]


class MantorLibraryError(RuntimeError):
    pass


# every symbol include/manytor_b200.h declares: (restype, argtypes)
_P = C.c_void_p
SIGNATURES = {
    "mt_abi_version": (C.c_int, []),
    "mt_last_error": (C.c_char_p, []),
    "mt_config_init": (C.c_int, [C.POINTER(MtConfig)]),
    "mt_create": (C.c_int, [C.POINTER(MtConfig), C.POINTER(_P)]),
    "mt_destroy": (C.c_int, [_P]),
    "mt_get_config": (C.c_int, [_P, C.POINTER(MtConfig)]),
    "mt_set_seed": (C.c_int, [_P, C.c_uint64]),
    "mt_get_step_index": (C.c_int, [_P, C.POINTER(C.c_uint64)]),
    "mt_set_step_index": (C.c_int, [_P, C.c_uint64]),
    "mt_reset": (C.c_int, [_P, _P, _P]),
    "mt_observe": (C.c_int, [_P, _P, _P]),
    "mt_step": (C.c_int, [_P, _P, _P, _P, _P, _P, _P]),
    "mt_step_final": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "mt_sample_actions": (C.c_int, [_P, _P, _P]),
    "mt_rollout_random": (C.c_int, [_P, C.c_int32, _P, _P, _P, _P]),
    "mt_rollout": (C.c_int, [_P, C.c_int32, _P, _P, _P, _P, _P, _P]),
    "mt_rollout_final": (C.c_int, [_P, C.c_int32, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "mt_rollout_branches": (C.c_int, [_P, C.c_int32, C.c_int64, _P, _P, C.c_float, _P, _P, _P, _P, _P]),
    "mt_rollout_branches_random": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int64, _P, _P, _P, C.c_float, _P, _P, _P,
                                             _P, _P]),
    "mt_branch_actions": (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.c_int64, _P, _P, _P]),
    "mt_step_host": (C.c_int, [_P, _P, _P, _P, _P]),
    "mt_host_step_mode": (C.c_int, [_P]),
    "mt_host_alloc": (C.c_int, [C.POINTER(_P), C.c_uint64]),
    "mt_host_free": (C.c_int, [_P]),
    "mt_set_points": (C.c_int, [_P, _P, _P, _P]),
    "mt_get_points": (C.c_int, [_P, _P, C.c_int32, _P]),
    "mt_set_state": (C.c_int, [_P, _P, _P, _P, _P, _P, _P]),
    "mt_get_state": (C.c_int, [_P, _P, _P, _P, _P, _P]),
    "mt_get_reset_counts": (C.c_int, [_P, _P, _P]),
    "mt_set_reset_counts": (C.c_int, [_P, _P, _P, _P]),
    "mt_set_objective_stream": (C.c_int, [_P, _P, C.c_int32]),
    "mt_fetch_env": (C.c_int, [_P, C.c_int64, _P, _P, _P, _P, _P]),
    "mt_stats_device": (C.c_int, [_P, _P, _P]),
    "mt_stats_host": (C.c_int, [_P, C.POINTER(MtStats)]),
    "mt_stats_clear": (C.c_int, [_P, _P]),
    "mt_stats_allreduce": (C.c_int, [C.POINTER(_P), C.c_int32, C.POINTER(MtStats)]),
    "mt_stats_allreduce_comm": (C.c_int, [_P, _P, _P, _P]),
    "mt_stats_peer_buffer_bytes": (C.c_int64, [C.c_int32]),
    "mt_stats_allreduce_peers": (C.c_int, [_P, _P, C.c_int32, C.c_int32, _P, _P]),
    "mt_fk": (C.c_int, [C.POINTER(MtConfig), C.c_int32, _P, _P, C.c_int64, _P]),
    "mt_dh": (C.c_int, [_P, _P, C.c_int64, _P]),
    "mt_joints": (C.c_int, [_P, _P, _P, C.c_int64, _P]),
    "mt_r_theta": (C.c_int, [_P, _P, _P, C.c_int64, _P]),
    "mt_launch_count": (C.c_int64, [_P]),
    "mt_bytes_per_env_step": (C.c_int64, [_P, C.c_int32, C.c_int32]),
    "mt_set_timing": (C.c_int, [_P, C.c_int32]),
    "mt_last_kernel_ms": (C.c_int, [_P, C.POINTER(C.c_float)]),
}

_lib = None
_by_path = {}


def library_path() -> str:
    return _build.LIB_PATH


def load(path: str = None) -> C.CDLL:
    """dlopen the in-tree library and bind every declared symbol (fails loudly).
    `path` loads another build of the same ABI (A/B timing of kernel variants, tools/ab.py)."""
    global _lib
    if path is None and _lib is not None:
        return _lib
    if path is not None and path in _by_path:
        return _by_path[path]
    explicit = path is not None
    path = path or library_path()
    if not os.path.exists(path):
        raise MantorLibraryError(
            f"{path} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
            "(manytor_b200 has no CPU fallback)")
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the .so does not export it
        fn.restype = res
        fn.argtypes = args
    if lib.mt_abi_version() != MT_ABI_VERSION:
        raise MantorLibraryError(f"ABI mismatch: library {lib.mt_abi_version()} != binding {MT_ABI_VERSION}")
    if explicit:
        _by_path[path] = lib
    else:
        _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        msg = load().mt_last_error()
        raise MantorLibraryError(f"manytor_b200 error {rc}: {msg.decode(errors='replace') if msg else ''}")


def default_config() -> MtConfig:
    cfg = MtConfig()
    check(load().mt_config_init(C.byref(cfg)))
    return cfg

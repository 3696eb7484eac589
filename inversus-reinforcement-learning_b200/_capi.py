"""ctypes binding of include/inversus_b200.h (the C ABI). No torch types cross this boundary.

The library is loaded from the in-tree build only (libinversus_b200.so next to this file). If it
is missing the import of the product fails loudly: there is no CPU or PyTorch fallback.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import _build

OK = 0
ERR_INVALID_ARG, ERR_CUDA, ERR_INVALID_ACTION, ERR_BULLET_OVERFLOW, ERR_NOT_RESET, ERR_NO_DEVICE = -1, -2, -3, -4, -5, -6
MODE = {"dummy": 0, "selfplay": 1}
DIFFICULTY = {"easy": 0, "hard": 1}
OBS_DTYPE = {"f32": 0, "float32": 0, "bf16": 1, "bfloat16": 1, "u8": 2, "uint8": 2, "none": 3}
FLAG_AUTO_RESET, FLAG_P2_VIEW, FLAG_REWARD_F64 = 1, 2, 4
(BUF_OBS_P1, BUF_EXTRA_P1, BUF_OBS_P2, BUF_EXTRA_P2, BUF_REWARD, BUF_DONE, BUF_INFO,
 BUF_EPISODE_STEPS, BUF_EPISODE_RETURN, BUF_PACKED_STATE, BUF_DEBUG_RESULT, BUF_REWARD_F64) = range(12)
(PHASE_TRY_MOVE, PHASE_SPAWN_BULLET, PHASE_WIDE_SHOT, PHASE_RELOAD, PHASE_UPDATE_BULLETS,
 PHASE_STEP_PLAYERS, PHASE_ENGINE_RESET, PHASE_DUMMY_POLICY) = range(8)


class Config(C.Structure):
    _fields_ = [("n_envs", C.c_int64), ("env_id_base", C.c_int64), ("seed", C.c_uint64),
                ("mode", C.c_int32), ("difficulty", C.c_int32), ("max_episode_steps", C.c_int32),
                ("device", C.c_int32), ("obs_dtype", C.c_int32), ("flags", C.c_uint32)]


class EnvState(C.Structure):
    _fields_ = [("tiles", C.c_uint32 * 5), ("p1", C.c_int32 * 5), ("p2", C.c_int32 * 5),
                ("n_bullets", C.c_int32), ("bullets", (C.c_int8 * 4) * 16),
                ("step_count", C.c_int32), ("episode", C.c_uint32), ("episode_return", C.c_double)]


# numpy mirror of inv_env_state (same memory layout)
STATE_DTYPE = np.dtype([
    ("tiles", np.uint32, (5,)), ("p1", np.int32, (5,)), ("p2", np.int32, (5,)),
    ("n_bullets", np.int32), ("bullets", np.int8, (16, 4)), ("step_count", np.int32),
    ("episode", np.uint32), ("episode_return", np.float64)], align=True)
assert STATE_DTYPE.itemsize == C.sizeof(EnvState), (STATE_DTYPE.itemsize, C.sizeof(EnvState))

# numpy mirror of inv_episode_event (one finished episode, inv_step_host_events)
EVENT_DTYPE = np.dtype([("env", np.int64), ("episode_return", np.float64), ("episode_steps", np.int32),
                        ("info", np.uint32)], align=True)
assert EVENT_DTYPE.itemsize == 24

# every symbol include/inversus_b200.h declares: (restype, argtypes)
_P = C.POINTER
SYMBOLS = {
    "inv_abi_version": (C.c_int, []),
    "inv_last_error": (C.c_char_p, []),
    "inv_device_count": (C.c_int, []),
    "inv_create": (C.c_int, [_P(Config), _P(C.c_void_p)]),
    "inv_destroy": (C.c_int, [C.c_void_p]),
    "inv_get_config": (C.c_int, [C.c_void_p, _P(Config)]),
    "inv_reset": (C.c_int, [C.c_void_p, C.c_void_p]),
    "inv_reset_envs": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "inv_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "inv_step_host": (C.c_int, [C.c_void_p] + [C.c_void_p] * 11),
    "inv_step_host_events": (C.c_int, [C.c_void_p] * 7 + [C.c_int64, _P(C.c_int64)]),
    "inv_reset_host": (C.c_int, [C.c_void_p] + [C.c_void_p] * 4),
    "inv_set_host_path": (C.c_int, [C.c_void_p, C.c_int, C.c_double]),
    "inv_get_host_path": (C.c_int, [C.c_void_p, _P(C.c_int), _P(C.c_double), _P(C.c_double), _P(C.c_double)]),
    "inv_host_expand_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int]),
    "inv_host_stage_action_ids": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64]),
    "inv_host_alloc": (C.c_int, [_P(C.c_void_p), C.c_int64]),
    "inv_host_free": (C.c_int, [C.c_void_p]),
    "inv_get_buffer": (C.c_int, [C.c_void_p, C.c_int, _P(C.c_void_p), _P(C.c_int64)]),
    "inv_set_draw_table": (C.c_int, [C.c_void_p, C.c_void_p]),
    "inv_export_state": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64]),
    "inv_import_state": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64]),
    "inv_load_packed_state": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "inv_obs_from_packed": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int, C.c_int,
                                      C.c_void_p, C.c_void_p, C.c_void_p]),
    "inv_debug_phase": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "inv_poll_status": (C.c_int, [C.c_void_p, C.c_void_p, _P(C.c_uint32)]),
    "inv_launch_count": (C.c_int64, [C.c_void_p]),
    "inv_ln_relu_partials": (C.c_int, [C.c_int32]),
    "inv_ln_relu_fwd": (C.c_int, [C.c_void_p] * 5 + [C.c_int64, C.c_int32, C.c_int32, C.c_float] + [C.c_void_p] * 4),
    "inv_ln_relu_bwd": (C.c_int, [C.c_void_p] * 8 + [C.c_int64, C.c_int32, C.c_int32] + [C.c_void_p] * 6),
    "inv_transpose_cast": (C.c_int, [C.c_void_p, C.c_int32, C.c_int64, C.c_void_p, C.c_int32, C.c_int64, C.c_int64,
                                     C.c_int32, C.c_int32, C.c_void_p]),
    "inv_encode_partials_floats": (C.c_int, []),
    "inv_encode_fwd": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int] + [C.c_void_p] * 4 + [C.c_float] + [C.c_void_p] * 5),
    "inv_encode_bwd": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int] + [C.c_void_p] * 13),
    "inv_conv3x3_wgrad_scratch_floats": (C.c_int64, [C.c_int32, C.c_int32]),
    "inv_conv3x3_wgrad": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "inv_gae": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_double, C.c_int32,
                          C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "inv_select_actions": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int64, C.c_uint64, C.c_int,
                                     C.c_int, C.c_void_p, C.c_void_p]),
    "inv_episode_tally": (C.c_int, [C.c_void_p] * 5 + [C.c_int64, C.c_int64, C.c_int64, C.c_int32] + [C.c_void_p] * 4),
    "inv_scripted_actions": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_uint64, C.c_int, C.c_int,
                                       C.c_void_p, C.c_void_p]),
}

_lib = None


class InversusError(RuntimeError):
    pass


def library_path() -> str:
    # INVERSUS_B200_LIB selects another build of the SAME library (kernel-shape experiments under profiles/)
    return os.environ.get("INVERSUS_B200_LIB") or _build.LIB_PATH


def load() -> C.CDLL:
    """Load libinversus_b200.so (must have been built: `python -c 'import __graft_entry__ as g; g.build()'`)."""
    global _lib
    if _lib is None:
        path = library_path()
        if not os.path.exists(path):
            raise InversusError(
                f"{path} is missing. Build it with __graft_entry__.build() (nvcc, sm_100a). "
                "This simulator has no CPU or PyTorch fallback.")
        lib = C.CDLL(path)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(lib, name)  # AttributeError if the ABI and the header drifted apart
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def last_error() -> str:
    return (load().inv_last_error() or b"").decode("utf-8", "replace")


def check(rc: int) -> None:
    """Map a status code to the exception type the reference raises for the same condition."""
    if rc == OK:
        return
    msg = last_error()
    if rc == ERR_INVALID_ACTION:
        raise ValueError(msg or "Invalid action_id: must be 0-12")  # env_wrappers.py:66
    if rc == ERR_INVALID_ARG:
        raise ValueError(msg)                                       # env_wrappers.py:309,316
    raise InversusError(f"inversus_b200 error {rc}: {msg}")

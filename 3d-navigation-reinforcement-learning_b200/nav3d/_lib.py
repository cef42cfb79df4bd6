"""ctypes binding of ``libnav3d_b200.so`` (C ABI in ``include/nav3d.h``).

There is no fallback: if the shared library is missing this module raises, and if no CUDA device is usable every
engine call fails with the library's own error message."""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

PKG_ROOT = Path(__file__).resolve().parent.parent          # 3d-navigation-reinforcement-learning_b200/
REPO_ROOT = PKG_ROOT.parent
LIB_PATH = PKG_ROOT / "lib" / "libnav3d_b200.so"

ABI_VERSION = 2
OBS_DIM = 80
STATE_INTS = 16
ENV_CUBIC, ENV_SIMPLE = 0, 1
OK = 0
ENV_STATE_LOADED, ENV_STATE_BAD_ENV, ENV_STATE_INVALID = 0, 1, 2     # nav3d_load_envs status codes

STATUS_NAMES = {0: "NAV3D_OK", -1: "NAV3D_ERR_INVALID", -2: "NAV3D_ERR_UNSUPPORTED", -3: "NAV3D_ERR_CUDA",
                -4: "NAV3D_ERR_NOMEM", -5: "NAV3D_ERR_ROOM"}


class Nav3dError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"{STATUS_NAMES.get(code, code)}: {message}")
        self.code = code


class Config(C.Structure):
    _fields_ = [("abi_version", C.c_int32), ("device", C.c_int32), ("n_envs", C.c_int32), ("env_kind", C.c_int32),
                ("local_map_length", C.c_int32), ("auto_reset", C.c_int32), ("lanes_per_env", C.c_int32),
                ("env_id0", C.c_uint32), ("seed", C.c_uint64), ("crash_penalty", C.c_double),
                ("cell_size", C.c_double)]


class RoomDesc(C.Structure):
    _fields_ = [("width", C.c_int32), ("depth", C.c_int32), ("height", C.c_int32), ("wall_code", C.c_int32),
                ("grid", C.c_void_p), ("has_start", C.c_int32), ("start_x", C.c_int32), ("start_y", C.c_int32),
                ("start_z", C.c_int32)]


class RewardParams(C.Structure):
    """``nav3d_reward_params``: the literals of ``compute_reward`` (reference ``envs/CubicEnv.py:169-224``)."""
    _fields_ = [(n, C.c_double) for n in ("step_cost", "revisit_unit", "revisit_cap", "crash_penalty", "near_wall_bonus",
                                          "repeat_bonus", "reverse_penalty", "explore_bonus", "finish_bonus",
                                          "truncation_penalty")]


# every symbol include/nav3d.h declares: (restype, argtypes)
_P = C.c_void_p
SYMBOLS = {
    "nav3d_last_error": (C.c_char_p, []),
    "nav3d_abi_version": (C.c_int, []),
    "nav3d_create": (C.c_int, [C.POINTER(Config), C.POINTER(_P)]),
    "nav3d_destroy": (None, [_P]),
    "nav3d_reward_params_default": (None, [C.POINTER(RewardParams)]),
    "nav3d_set_reward_params": (C.c_int, [_P, C.POINTER(RewardParams)]),
    "nav3d_load_rooms": (C.c_int, [_P, C.c_int32, C.POINTER(RoomDesc)]),
    "nav3d_room_info": (C.c_int, [_P, C.c_int32, C.POINTER(C.c_int32)]),
    "nav3d_room_free_cell": (C.c_int, [_P, C.c_int32, C.c_int32, C.POINTER(C.c_int32)]),
    "nav3d_obs_dim": (C.c_int, [_P]),
    "nav3d_num_envs": (C.c_int, [_P]),
    "nav3d_lanes_per_env": (C.c_int, [_P]),
    "nav3d_reset": (C.c_int, [_P, _P, C.c_int32, _P, _P, _P]),
    "nav3d_step": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "nav3d_step_host": (C.c_int, [_P, _P, _P, _P, _P, _P]),
    "nav3d_rollout_random": (C.c_int, [_P, C.c_int32, C.c_uint32, _P, _P, _P, _P, _P, _P]),
    "nav3d_rollout_actions": (C.c_int, [_P, C.c_int32] + [_P] * 10),
    "nav3d_get_state": (C.c_int, [_P, _P, _P]),
    "nav3d_get_grid": (C.c_int, [_P, C.c_int32, _P, _P]),
    "nav3d_snapshot_bytes": (C.c_size_t, [_P]),
    "nav3d_snapshot": (C.c_int, [_P, _P, C.c_size_t]),
    "nav3d_restore": (C.c_int, [_P, _P, C.c_size_t]),
    "nav3d_env_state_bytes": (C.c_size_t, [_P]),
    "nav3d_save_envs": (C.c_int, [_P, _P, C.c_int32, _P, _P, _P]),
    "nav3d_load_envs": (C.c_int, [_P, _P, C.c_int32, _P, _P, _P, _P]),
    "nav3d_sample_actions": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_uint64, C.c_uint32, C.c_uint32, _P, C.c_int32, _P, _P, _P, _P]),
    "nav3d_gae": (C.c_int, [_P, _P, _P, _P, _P, C.c_float, C.c_float, C.c_int32, C.c_int32, _P, _P, _P]),
    "nav3d_lstm_prepare": (C.c_int, [_P]),
    "nav3d_lstm_forward": (C.c_int, [_P] * 8 + [C.c_int32] * 5 + [_P] * 5),
    "nav3d_lstm_backward": (C.c_int, [_P] * 8 + [C.c_int32] * 5 + [_P] * 5),
    "nav3d_launch_count": (C.c_uint64, [_P]),
    "nav3d_device_bytes": (C.c_size_t, [_P]),
}

_lib = None


def load():
    """Load the CUDA library (once).  Raises if it has not been built: run ``python -c 'import __graft_entry__ as g; g.build()'``."""
    global _lib
    if _lib is not None:
        return _lib
    try:
        import torch  # noqa: F401  (first, so that the process uses the cuBLAS torch ships; ours binds to the same SONAME)
    except Exception:  # noqa: BLE001
        pass
    path = Path(os.environ.get("NAV3D_LIB", LIB_PATH))
    if not path.exists():
        raise ImportError(f"{path} is missing: build it with __graft_entry__.build() (nvcc, sm_100a). "
                          "nav3d has no CPU fallback.")
    lib = C.CDLL(str(path))
    for name, (restype, argtypes) in SYMBOLS.items():
        fn = getattr(lib, name)
        fn.restype = restype
        fn.argtypes = argtypes
    if lib.nav3d_abi_version() != ABI_VERSION:
        raise ImportError(f"{path}: ABI version {lib.nav3d_abi_version()} != {ABI_VERSION}")
    _lib = lib
    return lib


def check(code: int):
    if code != OK:
        raise Nav3dError(code, load().nav3d_last_error().decode("utf-8", "replace"))

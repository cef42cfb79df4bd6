"""ctypes front end of tests/emu/libnav3d_emu.so (the device logic of csrc/nav3d_core.cuh compiled for the host, one
lane per env).  A debugging aid for the GPU-less build container; tests only."""
import ctypes as C
import subprocess
from pathlib import Path

import numpy as np

import os

from __graft_entry__ import find_nvcc

HERE = Path(__file__).resolve().parent / "emu"
ASAN = os.environ.get("NAV3D_EMU_ASAN") == "1"          # tools/emu_asan.sh: the same source under AddressSanitizer + UBSan
LIB = HERE / ("libnav3d_emu_asan.so" if ASAN else "libnav3d_emu.so")
CORE = HERE.parent.parent / "3d-navigation-reinforcement-learning_b200" / "csrc" / "nav3d_core.cuh"
_lib = None


def build():
    src = HERE / "nav3d_emu.cu"
    if True:
        if not LIB.exists() or LIB.stat().st_mtime < max(src.stat().st_mtime, CORE.stat().st_mtime):
            extra = (["-g", "-DNAV3D_EMU_ASAN", "-Xcompiler", "-fsanitize=address", "-Xcompiler", "-fsanitize=undefined", "-Xcompiler",
                      "-fno-omit-frame-pointer", "-Xcompiler", "-fno-sanitize-recover=undefined"] if ASAN else [])
            subprocess.check_call([find_nvcc(), "-O2", "-std=c++17", "-Wno-deprecated-gpu-targets", "-shared", "-Xcompiler",
                                   "-fPIC", *extra, "-o", str(LIB), str(src)], stdout=subprocess.DEVNULL)


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(str(LIB))
        P, I = C.c_void_p, C.c_int
        L.emu_create.restype = P
        L.emu_create.argtypes = [I, I, C.c_double, C.c_uint64, C.c_uint32, I, I, P, P, P, I, I, C.c_double, I, I, P]
        L.emu_reward_params_reject.restype = C.c_char_p
        L.emu_reward_params_reject.argtypes = [P]
        L.emu_py_round2.restype = C.c_double
        L.emu_py_round2.argtypes = [C.c_double]
        L.emu_destroy.argtypes = [P]
        L.emu_room_n_free.restype = I
        L.emu_room_n_free.argtypes = [P, I]
        L.emu_reset.argtypes = [P, P, I, P, P]
        L.emu_step.argtypes = [P] * 9
        L.emu_get_state.argtypes = [P, P]
        L.emu_get_grid.argtypes = [P, I, P]
        _lib = L
    return _lib


def _p(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


class EmuEngine:
    def __init__(self, n, rooms, L=4, crash_penalty=-2.0, seed=0, env_id0=0, auto_reset=True, simple=False, cell_size=0.25,
                 lanes=1, descending=False, reward=None):
        """``reward``: the ten ``nav3d_reward_params`` values in field order (``oracle.c_oracle.reward_values``) or None for
        the reference's literals with ``crash_penalty``."""
        self.n = n
        self.obs_dim = 6 * L + 7 if simple else 80
        self.rooms = rooms
        dims = np.array([r.grid.shape for r in rooms], dtype=np.int32)
        offs = np.zeros(len(rooms), dtype=np.uint32)
        o = 0
        for i, r in enumerate(rooms):
            offs[i] = o
            o += r.grid.size
        dense = np.concatenate([np.ascontiguousarray(r.grid, dtype=np.int8).ravel() for r in rooms])
        rw = None if reward is None else np.ascontiguousarray(reward, dtype=np.float64)
        assert rw is None or rw.shape == (10,)
        self.h = lib().emu_create(n, L, crash_penalty, seed, env_id0, int(auto_reset), len(rooms), _p(dims), _p(dense),
                                  _p(offs), int(rooms[0].wall_code), int(simple), cell_size, int(lanes), int(descending),
                                  _p(rw))
        self.obs = np.zeros((n, self.obs_dim), np.float32)
        self.reward = np.zeros(n, np.float32)
        self.reward64 = np.zeros(n, np.float64)
        self.term = np.zeros(n, np.uint8)
        self.trunc = np.zeros(n, np.uint8)
        self.tobs = np.zeros((n, self.obs_dim), np.float32)
        self.eps = np.zeros((n, 8), np.int32)

    def n_free(self, r):
        return lib().emu_room_n_free(self.h, r)

    def reset(self, picks=None, env_ids=None):
        if picks is not None:
            picks = np.ascontiguousarray(picks, dtype=np.int32)
        if env_ids is not None:
            env_ids = np.ascontiguousarray(env_ids, dtype=np.int32)
        n = self.n if env_ids is None else len(env_ids)
        lib().emu_reset(self.h, _p(env_ids), n, _p(picks), _p(self.obs))
        return self.obs

    def step(self, actions):
        a = np.ascontiguousarray(actions, dtype=np.int64)
        lib().emu_step(self.h, _p(a), _p(self.obs), _p(self.reward), _p(self.reward64), _p(self.term), _p(self.trunc),
                       _p(self.tobs), _p(self.eps))

    def state(self):
        out = np.zeros((self.n, 16), np.int32)
        lib().emu_get_state(self.h, _p(out))
        return out

    def grid(self, env):
        st = self.state()[env]
        w, d, h = self.rooms[st[13]].grid.shape
        out = np.zeros((w, d, h), np.int16)
        lib().emu_get_grid(self.h, env, _p(out))
        return out

    def __del__(self):
        try:
            lib().emu_destroy(self.h)
        except Exception:  # noqa: BLE001
            pass

"""ctypes front end of tests/emu/libnav3d_emu_blobs.so: the env-state blob calls in the host emulation (tests/emu/
nav3d_emu_blobs.cu), on top of tests/emu_harness.EmuEngine.  A debugging aid for the GPU-less build container; tests only."""
import ctypes as C
import subprocess

import numpy as np

from __graft_entry__ import find_nvcc
from emu_harness import ASAN, CORE, HERE, EmuEngine

LIB = HERE / ("libnav3d_emu_blobs_asan.so" if ASAN else "libnav3d_emu_blobs.so")
_lib = None


def build():
    srcs = [HERE / "nav3d_emu_blobs.cu", HERE / "nav3d_emu.cu", CORE]
    if not LIB.exists() or LIB.stat().st_mtime < max(s.stat().st_mtime for s in srcs):
        extra = (["-g", "-DNAV3D_EMU_ASAN", "-Xcompiler", "-fsanitize=address", "-Xcompiler", "-fsanitize=undefined", "-Xcompiler",
                  "-fno-omit-frame-pointer", "-Xcompiler", "-fno-sanitize-recover=undefined"] if ASAN else [])
        subprocess.check_call([find_nvcc(), "-O2", "-std=c++17", "-Wno-deprecated-gpu-targets", "-shared", "-Xcompiler",
                               "-fPIC", *extra, "-o", str(LIB), str(srcs[0])], stdout=subprocess.DEVNULL)


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(str(LIB))
        P, I, U64 = C.c_void_p, C.c_int, C.c_uint64
        L.emu_signature.restype = U64
        L.emu_signature.argtypes = [P, I, P, P, P, I]
        L.emu_env_state_bytes.restype = C.c_long
        L.emu_env_state_bytes.argtypes = [P]
        L.emu_save_envs.argtypes = [P, U64, P, I, P, P]
        L.emu_load_envs.argtypes = [P, U64, P, I, P, P, P]
        _lib = L
    return _lib


def _p(a):
    return C.c_void_p(a.ctypes.data)


class EmuBlobs(EmuEngine):
    """EmuEngine plus save / load / take, the adapter tests/env_state_checks.py drives."""

    def __init__(self, n, rooms, **kwargs):
        super().__init__(n, rooms, **kwargs)
        dims = np.array([r.grid.shape for r in rooms], dtype=np.int32)
        offs = np.cumsum([0] + [r.grid.size for r in rooms[:-1]]).astype(np.uint32)
        dense = np.concatenate([np.ascontiguousarray(r.grid, dtype=np.int8).ravel() for r in rooms])
        self.sig = lib().emu_signature(self.h, len(rooms), _p(dims), _p(dense), _p(offs), int(rooms[0].wall_code))

    def save(self, ids):
        ids = np.ascontiguousarray(ids, np.int32)
        out = np.zeros((len(ids), lib().emu_env_state_bytes(self.h)), np.uint8)
        lib().emu_save_envs(self.h, self.sig, _p(ids), len(ids), _p(self.obs), _p(out))
        return out

    def load(self, ids, blobs):
        ids = np.ascontiguousarray(ids, np.int32)
        blobs = np.ascontiguousarray(blobs)
        status = np.full(len(ids), 255, np.uint8)
        lib().emu_load_envs(self.h, self.sig, _p(ids), len(ids), _p(blobs), _p(self.obs), _p(status))
        return status

    @staticmethod
    def take(blobs, idx):
        return blobs[idx]

"""ctypes front end of tests/emu/libnav3d_emu_weights.so: nav3d_set_room_weights in the host emulation (tests/emu/
nav3d_emu_weights.cu), on top of tests/emu_rollout.EmuRollout.  A debugging aid for the GPU-less build container; tests only."""
import ctypes as C
import subprocess

import numpy as np

from __graft_entry__ import find_nvcc
from emu_harness import ASAN, CORE, HERE
from emu_rollout import EmuRollout

LIB = HERE / ("libnav3d_emu_weights_asan.so" if ASAN else "libnav3d_emu_weights.so")
_lib = None


def build():
    srcs = [HERE / "nav3d_emu_weights.cu", HERE / "nav3d_emu.cu", CORE]
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
        L.emu_set_room_weights.restype = C.c_int
        L.emu_set_room_weights.argtypes = [C.c_void_p, C.c_void_p]
        L.emu_get_room_cdf.argtypes = [C.c_void_p, C.c_void_p]
        L.emu_free_room_cdf.argtypes = [C.c_void_p]
        _lib = L
    return _lib


def _p(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


class EmuWeights(EmuRollout):
    """EmuRollout plus the room-draw table of nav3d_set_room_weights."""

    def set_room_weights(self, weights=None) -> int:
        """Returns the status (0 installed, 1 rejected)."""
        w = None if weights is None else np.ascontiguousarray(weights, dtype=np.float32)
        assert w is None or w.shape == (len(self.rooms),)
        return lib().emu_set_room_weights(self.h, _p(w))

    def room_cdf(self) -> np.ndarray:
        out = np.zeros(len(self.rooms), np.uint64)
        lib().emu_get_room_cdf(self.h, _p(out))
        return out

    def __del__(self):
        try:
            lib().emu_free_room_cdf(self.h)
        except Exception:  # noqa: BLE001
            pass
        super().__del__()

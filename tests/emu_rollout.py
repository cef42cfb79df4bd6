"""ctypes front end of tests/emu/libnav3d_emu_rollout.so: nav3d_rollout_actions in the host emulation (tests/emu/
nav3d_emu_rollout.cu), on top of tests/emu_harness.EmuEngine.  A debugging aid for the GPU-less build container; tests only."""
import ctypes as C
import subprocess

import numpy as np

from __graft_entry__ import find_nvcc
from emu_harness import ASAN, CORE, HERE, EmuEngine

LIB = HERE / ("libnav3d_emu_rollout_asan.so" if ASAN else "libnav3d_emu_rollout.so")
_lib = None


def build():
    srcs = [HERE / "nav3d_emu_rollout.cu", HERE / "nav3d_emu.cu", CORE]
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
        L.emu_rollout_actions.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 9
        _lib = L
    return _lib


def _p(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


class EmuRollout(EmuEngine):
    """EmuEngine plus the fused rollout with caller-supplied actions."""

    def rollout(self, actions, obs=None, obs_last=None, reward=None, reward64=None, term=None, trunc=None, tobs=None,
                eps=None):
        """``actions`` u8 [T, n]; every output is a caller-owned numpy array (or None) laid out as nav3d_rollout_actions
        takes it.  ``obs_last`` defaults to this engine's own observation array when ``obs`` is None."""
        a = np.ascontiguousarray(actions, dtype=np.uint8)
        assert a.ndim == 2 and a.shape[1] == self.n
        if obs is None and obs_last is None:
            obs_last = self.obs
        lib().emu_rollout_actions(self.h, a.shape[0], _p(a), _p(obs), _p(obs_last), _p(reward), _p(reward64), _p(term),
                                  _p(trunc), _p(tobs), _p(eps))
        if obs is not None and a.shape[0]:
            self.obs[:] = obs[-1]

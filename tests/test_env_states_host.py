"""Env-state blobs (nav3d_save_envs / nav3d_load_envs) without a GPU: the C entry points exist and check their arguments
before touching a device, and the per-env copy functions of csrc/nav3d_core.cuh — the ones the kernels run — pass the
round-trip, clone and live-part scenarios in the host emulation (tests/emu/nav3d_emu_blobs.cu).  tools/emu_asan.sh runs this file under
AddressSanitizer too, with every env fenced to the part of its block its room owns."""
import ctypes as C

import numpy as np
import pytest

from __graft_entry__ import find_nvcc
from conftest import ROOMS
from nav3d.rooms import load_room_dir, load_room_file

NEW_SYMBOLS = ("nav3d_env_state_bytes", "nav3d_save_envs", "nav3d_load_envs")


def test_new_symbols_are_declared_bound_and_exported():
    import __graft_entry__ as g
    g.build_lib()
    from nav3d import _lib
    from test_capi_symbols import header_symbols
    lib = _lib.load()
    for name in NEW_SYMBOLS:
        assert name in header_symbols() and name in _lib.SYMBOLS and hasattr(lib, name)
    assert lib.nav3d_abi_version() == 2


def test_c_calls_reject_bad_arguments_without_a_device():
    from nav3d import _lib
    lib = _lib.load()
    host = np.zeros(4096, np.uint8)          # a real address: never dereferenced, every call fails before that
    p = C.c_void_p(host.ctypes.data + (-host.ctypes.data) % 16)
    odd = C.c_void_p(p.value + 4)

    def err():
        return lib.nav3d_last_error().decode()
    assert lib.nav3d_env_state_bytes(None) == 0
    assert lib.nav3d_save_envs(None, None, -1, p, p, None) == -1 and "n must be" in err()
    assert lib.nav3d_save_envs(None, None, 4, None, p, None) == -1 and "obs and blobs" in err()
    assert lib.nav3d_save_envs(None, None, 4, p, None, None) == -1 and "obs and blobs" in err()
    assert lib.nav3d_save_envs(None, None, 4, p, odd, None) == -1 and "aligned" in err()
    assert lib.nav3d_save_envs(None, None, 4, p, p, None) == -1 and "engine is NULL" in err()
    assert lib.nav3d_load_envs(None, None, -1, p, p, None, None) == -1 and "n must be" in err()
    assert lib.nav3d_load_envs(None, None, 4, None, p, None, None) == -1 and "obs and blobs" in err()
    assert lib.nav3d_load_envs(None, None, 4, p, None, None, None) == -1 and "obs and blobs" in err()
    assert lib.nav3d_load_envs(None, None, 4, odd, p, None, None) == -1 and "aligned" in err()
    assert lib.nav3d_load_envs(None, None, 4, p, p, p, None) == -1 and "engine is NULL" in err()


needs_nvcc = pytest.mark.skipif(find_nvcc() is None, reason="nvcc needed to build the host emulation")


def emu_blob_engine(*args, **kwargs):
    from emu_blobs import EmuBlobs
    return EmuBlobs(*args, **kwargs)


@needs_nvcc
def test_emu_round_trip_p3_training():
    from env_state_checks import round_trip
    rooms = load_room_dir(ROOMS / "P3_training", sort=True)
    e = emu_blob_engine(96, rooms, L=10, seed=3)
    assert round_trip(e, 7) > 0            # some loaded envs auto-reset inside the replayed window


@needs_nvcc
def test_emu_clone_matches_oracle(oracle):
    from env_state_checks import clone
    rooms = load_room_dir(ROOMS / "P3_training", sort=True)
    n, L, seed = 64, 10, 5
    e = emu_blob_engine(n, rooms, L=L, seed=seed)
    orooms = [oracle.OracleRoom(r.grid, -2) for r in rooms]
    ov = oracle.OracleVec(n, orooms, L, -2.0, seed, 0, True)
    nf = [r.n_free for r in orooms]
    clone(e, 11, nf, [r.free_cells() for r in rooms], lambda env, ep: oracle.pick(seed, env, ep, nf), oracle_vec=ov)


@needs_nvcc
def test_emu_live_part_across_room_sizes():
    from edge_rooms import degenerate_rooms
    from env_state_checks import live_part
    rooms = [load_room_file(ROOMS / "P3_training" / "maze_7x7_seed22.txt"), degenerate_rooms()[3],
             load_room_file(ROOMS / "P3_training" / "kitchen2.txt"), load_room_file(ROOMS / "P2_training" / "tightcorridor.txt")]
    sizes = [r.grid.size for r in rooms]
    assert sizes[2] == max(sizes) and sizes[1] == min(sizes)
    picks = np.array([[r, 0] for r in range(4)] * 2, np.int32)
    e = emu_blob_engine(8, rooms, L=10, seed=1, auto_reset=False)
    live_part(e, picks)


@needs_nvcc
def test_emu_simple_round_trip_and_clone(oracle):
    from env_state_checks import clone, round_trip
    rooms = [load_room_file(ROOMS / "P3_training" / n, simple=True) for n in ("maze_3d_tunnels.txt", "kitchen2.txt",
                                                                                 "maze_7x7_seed22.txt")]
    e = emu_blob_engine(48, rooms, L=4, seed=2, simple=True)
    round_trip(e, 3)
    nf = [len(r.free_cells()) for r in rooms]
    e = emu_blob_engine(32, rooms, L=4, seed=4, simple=True)
    clone(e, 9, nf, [r.free_cells() for r in rooms], lambda env, ep: oracle.pick3(4, env, ep, nf), simple=True)

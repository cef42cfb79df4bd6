"""nav3d_rollout_actions without a GPU: the C entry point exists and checks its arguments before touching the engine, and
the fused rollout's T-step loop — the record held outside the engine (step_lane / step_commit with REG_STATE), the per-step
outputs of rollout_step_io, auto-resets inside the loop — run in the host emulation (tests/emu/nav3d_emu_rollout.cu) is
bit-equal to T emulated nav3d_step calls and to the C oracle.  tools/emu_asan.sh runs this file under AddressSanitizer too."""
import ctypes as C

import numpy as np
import pytest

from __graft_entry__ import find_nvcc
from conftest import ROOMS
from lockstep import compare_grids, compare_step
from nav3d.rooms import load_room_dir, load_room_file


def test_symbol_is_declared_bound_and_exported():
    import __graft_entry__ as g
    g.build_lib()
    from nav3d import _lib
    from test_capi_symbols import header_symbols
    lib = _lib.load()
    assert "nav3d_rollout_actions" in header_symbols() and "nav3d_rollout_actions" in _lib.SYMBOLS
    assert hasattr(lib, "nav3d_rollout_actions") and lib.nav3d_abi_version() == 2


def test_c_call_rejects_bad_arguments_in_order_without_a_device():
    from nav3d import _lib
    lib = _lib.load()
    host = np.zeros(4096, np.uint8)          # a real address: never dereferenced, every call fails before that
    p = C.c_void_p(host.ctypes.data + (-host.ctypes.data) % 16)
    odd = C.c_void_p(p.value + 4)

    def call(T, actions, obs, obs_last, terminal_obs=None):
        rc = lib.nav3d_rollout_actions(None, T, actions, obs, obs_last, None, None, None, None, terminal_obs, None, None)
        return rc, lib.nav3d_last_error().decode()

    rc, msg = call(-1, None, None, None)
    assert rc == -1 and "T must be" in msg
    rc, msg = call(4, None, None, None)
    assert rc == -1 and "actions is required" in msg
    rc, msg = call(4, p, None, None)
    assert rc == -1 and "one of obs / obs_last" in msg
    for args in ((odd, None), (None, odd), (p, None, odd)):
        rc, msg = call(4, p, *args)
        assert rc == -1 and "aligned" in msg
    for args in ((p, None), (None, p), (p, p, p)):
        rc, msg = call(4, p, *args)
        assert rc == -1 and "engine is NULL" in msg
    rc, msg = call(0, p, p, None)
    assert rc == -1 and "engine is NULL" in msg


needs_nvcc = pytest.mark.skipif(find_nvcc() is None, reason="nvcc needed to build the host emulation")
SENTINEL = 0x7F


def run_against_steps(oracle, rooms, n, L, T, seed, lanes=1, auto_reset=True, pre_steps=20, a_hi=6, outputs="all",
                      descending=False, picks=None):
    """Engines A (rollout) and B (T emulated nav3d_step calls) and the oracle from the same state after `pre_steps` steps:
    every output row, the rows left untouched, the final records and knowledge grids.  Returns the number of episode ends
    inside the rollout per env."""
    from emu_harness import EmuEngine
    from emu_rollout import EmuRollout
    kw = dict(L=L, crash_penalty=-2.0, seed=seed, env_id0=0, auto_reset=auto_reset, lanes=lanes, descending=descending)
    A, B = EmuRollout(n, rooms, **kw), EmuEngine(n, rooms, **kw)
    ov = oracle.OracleVec(n, [oracle.OracleRoom(r.grid, -2) for r in rooms], L, -2.0, seed, 0, auto_reset)
    A.reset(picks), B.reset(picks), ov.reset(picks)
    rng = np.random.default_rng(seed + 100)
    for _ in range(pre_steps):
        a = rng.integers(0, 6, size=n)
        A.step(a), B.step(a), ov.step(a)
    acts = rng.integers(0, a_hi, size=(T, n)).astype(np.uint8)
    full = outputs == "all"
    o = {k: None for k in ("obs", "reward", "reward64", "term", "trunc", "tobs", "eps")}
    if full or "obs" in outputs:
        o["obs"] = np.full((T, n, 80), np.nan, np.float32)
    if full or "reward" in outputs:
        o["reward"] = np.zeros((T, n), np.float32)
    if full or "reward64" in outputs:
        o["reward64"] = np.zeros((T, n), np.float64)
    if full or "flags" in outputs:
        o["term"], o["trunc"] = np.full((T, n), 9, np.uint8), np.full((T, n), 9, np.uint8)
    if full or "tobs" in outputs:
        o["tobs"] = np.full((T, n, 80 * 4), SENTINEL, np.uint8).view(np.float32)
    if full or "eps" in outputs:
        o["eps"] = np.full((T, n, 32), SENTINEL, np.uint8).view(np.int32)
    A.rollout(acts, **o)
    ends = np.zeros(n, np.int64)
    for t in range(T):
        a = np.minimum(acts[t], 5).astype(np.int64)
        B.step(a)
        ov.step(a)
        done = (B.term | B.trunc) != 0
        ends += done
        tag = f"t={t}"
        if o["obs"] is not None:
            assert np.array_equal(o["obs"][t].view(np.uint32), B.obs.view(np.uint32)), f"{tag}: obs"
        if o["reward"] is not None:
            assert np.array_equal(o["reward"][t], B.reward), f"{tag}: reward"
        if o["reward64"] is not None:
            assert np.array_equal(o["reward64"][t], B.reward64), f"{tag}: reward64"
        if o["term"] is not None:
            assert np.array_equal(o["term"][t], B.term) and np.array_equal(o["trunc"][t], B.trunc), f"{tag}: flags"
        if o["tobs"] is not None:
            reset = done if auto_reset else np.zeros(n, bool)
            rows = o["tobs"][t].view(np.uint8).reshape(n, -1)
            assert np.array_equal(o["tobs"][t][reset].view(np.uint32), B.tobs[reset].view(np.uint32)), f"{tag}: terminal obs"
            assert (rows[~reset] == SENTINEL).all(), f"{tag}: a terminal_obs row of an env that did not reset was written"
        if o["eps"] is not None:
            rows = o["eps"][t].view(np.uint8).reshape(n, -1)
            assert np.array_equal(o["eps"][t][done], B.eps[done]), f"{tag}: episodes"
            assert (rows[~done] == SENTINEL).all(), f"{tag}: an episodes row of an env that did not finish was written"
        if full:
            compare_step(f"emu rollout {tag}", t, ov, o["obs"][t], o["reward"][t], o["reward64"][t], o["term"][t],
                         o["trunc"][t], o["tobs"][t] if auto_reset else None, o["eps"][t], None)
    assert np.array_equal(A.obs.view(np.uint32), B.obs.view(np.uint32)), "the last observation"
    assert np.array_equal(A.state(), B.state()), "final records"
    assert np.array_equal(A.state()[:, :15].astype(np.int64), ov.state()), "final records vs oracle"
    for i in range(n):
        assert np.array_equal(A.grid(i), B.grid(i)), f"knowledge grid of env {i}"
    compare_grids("emu rollout", ov, A.grid, range(n))
    return ends


# G > 1: the emulation runs the lanes of a group in descending order.  In ascending order lane 0 stores a cell's
# overflow byte (counts >= 29) before a sibling has read it, which real lanes of one warp step never see; the emulated
# nav3d_step has the same artefact, so the oracle can only be held to the descending order.
@needs_nvcc
@pytest.mark.parametrize("lanes", [1, 2, 4, 8, 16, 32])
def test_emu_p1_training_every_lane_width(oracle, lanes):
    rooms = load_room_dir(ROOMS / "P1_training", sort=True)
    run_against_steps(oracle, rooms, n=24, L=10, T=60, seed=lanes, lanes=lanes, a_hi=256, descending=lanes > 1)


@needs_nvcc
@pytest.mark.parametrize("lanes", [1, 2, 4, 8, 16, 32])
def test_emu_edge_rooms_every_lane_width(oracle, lanes):
    from edge_rooms import degenerate_rooms, max_size_rooms
    rooms = max_size_rooms() + degenerate_rooms()
    picks = np.array([[i % len(rooms), 0] for i in range(12)], np.int32)
    ends = run_against_steps(oracle, rooms, n=12, L=15, T=80, seed=30 + lanes, lanes=lanes, a_hi=9, descending=lanes > 1,
                             picks=picks, pre_steps=0)
    assert ends[2] > 0 and ends[8] > 0     # the single-cell room ends an episode on every step


@needs_nvcc
def test_emu_several_resets_per_env_inside_one_rollout(oracle):
    rooms = [load_room_file(ROOMS / "P2_training" / "tightcorridor.txt"),
             load_room_file(ROOMS / "P3_training" / "maze_3d_tunnels.txt")]
    assert sorted(len(r.free_cells()) for r in rooms) == [149, 302]
    ends = run_against_steps(oracle, rooms, n=16, L=10, T=700, seed=5, a_hi=256)
    assert ends.min() >= 2                 # truncation at 149 / 302 steps: every env restarts at least twice


@needs_nvcc
def test_emu_auto_reset_off_runs_past_done(oracle):
    rooms = [load_room_file(ROOMS / "P3_training" / "maze_3d_tunnels.txt")]
    ends = run_against_steps(oracle, rooms, n=8, L=10, T=250, seed=6, auto_reset=False, pre_steps=0)
    assert ends.min() > 1                  # every env keeps stepping (and reporting truncated) past step 149


@needs_nvcc
@pytest.mark.parametrize("outputs", [("reward",), ("flags", "eps"), ("reward64", "tobs"), ("obs", "eps")])
def test_emu_obs_last_and_null_outputs(oracle, outputs):
    """Subsets of the outputs; without "obs" only the last step's rows are formed, into the engine's own array."""
    rooms = load_room_dir(ROOMS / "P3_training", sort=True)[:5] + [load_room_file(ROOMS / "P2_training" / "tightcorridor.txt")]
    run_against_steps(oracle, rooms, n=20, L=10, T=330, seed=7, a_hi=256, outputs=outputs)


@needs_nvcc
def test_emu_zero_steps_change_nothing(oracle):
    from emu_rollout import EmuRollout
    rooms = load_room_dir(ROOMS / "P1_training", sort=True)
    e = EmuRollout(8, rooms, L=10, seed=1)
    e.reset()
    st, obs = e.state(), e.obs.copy()
    e.rollout(np.zeros((0, 8), np.uint8))
    assert np.array_equal(e.state(), st) and np.array_equal(e.obs.view(np.uint32), obs.view(np.uint32))

"""Host-side check of the packed-representation logic (csrc/nav3d_core.cuh compiled for the CPU, one lane per env)
against the oracle.  This is a debugging aid for the GPU-less container; the parity tests proper are -m gpu."""
import numpy as np
import pytest

from __graft_entry__ import find_nvcc
from conftest import ROOMS
from lockstep import compare_grids, compare_step
from nav3d.rooms import load_room_dir, load_room_file

pytestmark = pytest.mark.skipif(find_nvcc() is None, reason="nvcc needed to build the host emulation")


def run_lockstep(oracle, rooms, n, L, steps, seed, auto_reset=True, crash=-2.0, check_state_every=1, lanes=1,
                 descending=False):
    from emu_harness import EmuEngine
    orooms = [oracle.OracleRoom(r.grid, -2) for r in rooms]
    ov = oracle.OracleVec(n, orooms, L, crash, seed, 0, auto_reset)
    em = EmuEngine(n, rooms, L, crash, seed, 0, auto_reset, lanes=lanes, descending=descending)
    for i, r in enumerate(orooms):
        assert em.n_free(i) == r.n_free
    o0 = ov.reset()
    e0 = em.reset()
    assert np.array_equal(e0.view(np.uint32), o0.view(np.uint32))
    assert np.array_equal(em.state()[:, :15].astype(np.int64), ov.state())
    rng = np.random.default_rng(seed + 1)
    n_done = 0
    for t in range(steps):
        a = rng.integers(0, 6, size=n)
        ov.step(a)
        em.step(a)
        st = em.state() if t % check_state_every == 0 else None
        compare_step("emu", t, ov, em.obs, em.reward, em.reward64, em.term, em.trunc, em.tobs, em.eps, st, crash)
        n_done += int((ov.terminated | ov.truncated).sum())
    compare_grids("emu", ov, em.grid, range(0, n, max(1, n // 8)))
    return n_done


def test_emu_p1_training_autoreset(oracle):
    rooms = load_room_dir(ROOMS / "P1_training", sort=True)
    n_done = run_lockstep(oracle, rooms, n=48, L=10, steps=2200, seed=3)
    assert n_done > 0          # the 12x12x12 room truncates at 1000 steps


def test_emu_heterogeneous_rooms(oracle):
    rooms = load_room_dir(ROOMS / "P3_training", sort=True) + [load_room_file(ROOMS / "P2_training" / "tightcorridor.txt")]
    n_done = run_lockstep(oracle, rooms, n=72, L=10, steps=700, seed=11, check_state_every=7)
    assert n_done > 0          # maze_3d_tunnels (149 free) and tightcorridor (302) truncate early


@pytest.mark.parametrize("lanes", [2, 4, 8, 16, 32])
@pytest.mark.parametrize("descending", [False, True])
def test_emu_lane_groups(oracle, lanes, descending):
    """The G lanes of a group run one after the other, in either order: no lane may depend on what a sibling wrote in the
    same step (readers of a word another lane marks re-derive the marks themselves)."""
    rooms = load_room_dir(ROOMS / "P1_training", sort=True)[:3] + [load_room_file(ROOMS / "P3_training" / "maze_7x7_seed22.txt"),
                                                                    load_room_file(ROOMS / "P3_training" / "kitchen2.txt")]
    n_done = run_lockstep(oracle, rooms, n=24, L=10, steps=1100, seed=lanes, lanes=lanes, descending=descending,
                          check_state_every=3)
    assert n_done > 0
    from edge_rooms import degenerate_rooms, max_size_rooms
    run_lockstep(oracle, max_size_rooms() + degenerate_rooms(), n=16, L=15, steps=300, seed=9, lanes=lanes, descending=descending)


@pytest.mark.parametrize("L", [1, 4, 15, 40])
def test_emu_ray_lengths(oracle, L):
    rooms = [load_room_file(ROOMS / "P3_training" / "maze_7x7_seed22.txt"), load_room_file(ROOMS / "P3_training" / "kitchen2.txt"),
             load_room_file(ROOMS / "P2_training" / "small_bedroom.txt")]
    run_lockstep(oracle, rooms, n=24, L=L, steps=400, seed=L, crash=-0.5)


def test_emu_engine_limits_and_degenerate_rooms(oracle):
    from edge_rooms import degenerate_rooms, max_size_rooms, thin_open_rooms
    assert run_lockstep(oracle, max_size_rooms(), n=12, L=15, steps=600, seed=2, check_state_every=5) >= 0
    assert run_lockstep(oracle, degenerate_rooms(), n=16, L=10, steps=300, seed=4) > 0
    assert run_lockstep(oracle, thin_open_rooms(), n=12, L=4, steps=200, seed=6) > 0
    # counters beyond the u8 range: no auto-reset in the two-cell room, 400 steps (the oracle's int64 grid is compared
    # after clamping to 255; observations clip at 20 and rewards at 25, so every output stays identical)
    run_lockstep(oracle, degenerate_rooms()[3:], n=4, L=10, steps=400, seed=8, auto_reset=False)


def test_emu_no_autoreset_runs_past_done(oracle):
    rooms = [load_room_file(ROOMS / "P3_training" / "maze_3d_tunnels.txt")]
    run_lockstep(oracle, rooms, n=8, L=10, steps=400, seed=5, auto_reset=False)


def test_emu_replays_reference_golden_traces(cubic_traces):
    from emu_harness import EmuEngine
    from lockstep import replay_golden_trace
    n_term = 0
    for c in cubic_traces:
        room = load_room_file(ROOMS / c["room"])
        replay_golden_trace(c, room, lambda rooms, L, crash, ar: EmuEngine(1, rooms, L, crash, 0, 0, ar))
        n_term += int(c["state"][:, 7].max())
    assert n_term >= 2      # the coverage-policy traces reach the 84 % termination branch


def test_emu_simple_env_replays_reference_golden_traces(simple_traces):
    from emu_harness import EmuEngine
    from lockstep import replay_simple_golden_trace
    n_term = 0
    for c in simple_traces:
        room = load_room_file(ROOMS / c["room"], simple=True)
        replay_simple_golden_trace(c, room, lambda rooms, L: EmuEngine(1, rooms, L, -2.0, 0, 0, False, simple=True))
        n_term += int(c["state"][:, 7].max())
    assert n_term >= 1

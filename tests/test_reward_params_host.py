"""Non-default reward parameters and simpleEnv cell sizes without a GPU: the engine's rejection rules, its simpleEnv
distance rounding against CPython's round, and the host emulation of the step kernels (csrc/nav3d_core.cuh) in lock-step
with the parametrized oracle.  tools/emu_asan.sh runs this file under AddressSanitizer + UBSan."""
import numpy as np
import pytest

from __graft_entry__ import find_nvcc
from conftest import ROOMS
from lockstep import compare_grids, compare_step
from nav3d.rooms import load_room_dir, load_room_file
from reward_sets import ACCEPTED, INT32_MAX, REJECTED, SETS, rejects

needs_nvcc = pytest.mark.skipif(find_nvcc() is None, reason="nvcc needed to build the host emulation")
CELL_SIZES = [0.005 * k for k in range(1, 201)]


def test_oracle_round2_is_python_round(oracle):
    """simpleEnv's distances are round(count * cell_size, 2) (simpleEnv.py:337).  At 0.175 and count 1 the product is
    0.17499999999999998890 in binary, which CPython rounds to 0.17; rint(x * 100) / 100 gave 0.18."""
    bad = [(cs, c) for cs in CELL_SIZES for c in range(256) if oracle.py_round2(c * cs) != round(c * cs, 2)]
    assert not bad, f"{len(bad)} (cell_size, count) pairs differ from CPython, e.g. {bad[:5]}"
    assert oracle.py_round2(1 * 0.175) == 0.17


@needs_nvcc
def test_engine_round2_is_python_round():
    """The engine builds its distance table with the same function (nav3d_core.cuh py_round2); at 0.25 it gives what
    rint(x * 100) / 100 gave before, so existing simpleEnv outputs do not change."""
    from emu_harness import lib
    r2 = lib().emu_py_round2
    bad = [(cs, c) for cs in CELL_SIZES for c in range(256) if r2(c * cs) != round(c * cs, 2)]
    assert not bad, f"{len(bad)} (cell_size, count) pairs differ from CPython, e.g. {bad[:5]}"
    assert all(r2(c * 0.25) == np.rint(c * 0.25 * 100.0) / 100.0 for c in range(256))


@needs_nvcc
def test_rejection_rules_match_the_documented_ones():
    """emu_reward_params_reject is the engine's check (reward_params_reject); the restatement in reward_sets follows
    include/nav3d.h.  Both must agree on every listed set and on random sets around the two boundaries."""
    from emu_harness import lib
    from oracle.c_oracle import reward_values
    rng = np.random.default_rng(0)
    cases = [p for _, p in SETS]
    for _ in range(3000):
        p = {}
        if rng.random() < 0.5:
            cap = float(rng.choice([0.0, 0.5, 1.0, -0.3, 12.5]))
            p["revisit_cap"] = cap
            p["revisit_unit"] = float(rng.choice([0.0, -0.01, cap / 255.0, rng.uniform(-0.01, 0.1)]))
        for f in ("explore_bonus", "step_cost", "reverse_penalty", "near_wall_bonus"):
            if rng.random() < 0.3:
                p[f] = float(rng.choice([-1, 1]) * rng.uniform(0, 400))
        cases.append(p)
    for p in cases:
        why = lib().emu_reward_params_reject(reward_values(p).ctypes.data)
        kind = rejects(p)
        assert (why is None) == (kind is None), f"{p}: engine says {why!r}, the documented rule {kind!r}"
        if kind is not None:
            assert {"saturation": b"saturate at 255", "overflow": b"int32"}[kind] in why, (p, why)
    assert {k for k, _ in REJECTED} == {"revisit_unit_neg", "saturation_out", "saturation_unit_0.001", "overflow_out",
                                       "overflow_explore_1e6"}


def _lockstep(oracle, rooms, n, L, steps, seed, reward, auto_reset=True, lanes=1):
    from emu_harness import EmuEngine
    from oracle.c_oracle import reward_values
    orooms = [oracle.OracleRoom(r.grid, -2) for r in rooms]
    crash = reward_values(reward)[3]
    ov = oracle.OracleVec(n, orooms, L, crash, seed, 0, auto_reset, reward=reward)
    em = EmuEngine(n, rooms, L, crash, seed, 0, auto_reset, lanes=lanes, reward=reward_values(reward))
    ov.reset()
    em.reset()
    rng = np.random.default_rng(seed + 1)
    n_done = 0
    for t in range(steps):
        a = rng.integers(0, 6, size=n)
        ov.step(a)
        em.step(a)
        compare_step("emu", t, ov, em.obs, em.reward, em.reward64, em.term, em.trunc, em.tobs, em.eps, em.state())
        n_done += int((ov.terminated | ov.truncated).sum())
    compare_grids("emu", ov, em.grid, range(0, n, max(1, n // 4)))
    return n_done


@needs_nvcc
@pytest.mark.parametrize("name,reward", ACCEPTED, ids=[k for k, _ in ACCEPTED])
def test_emu_reward_params_lockstep(oracle, name, reward):
    """Every accepted set: rewards bit for bit, episode records and state[15] exactly as the documented rule gives them,
    in rooms where episodes end (truncation and the 84 % finish) and with auto-reset on and off."""
    rooms = [load_room_file(ROOMS / "P3_training" / "maze_3d_tunnels.txt"),
             load_room_file(ROOMS / "P2_training" / "tightcorridor.txt")]
    assert _lockstep(oracle, rooms, n=12, L=10, steps=330, seed=7, reward=reward, lanes=4 if "x2" in name else 1) > 0
    from edge_rooms import degenerate_rooms
    _lockstep(oracle, degenerate_rooms(), n=8, L=10, steps=120, seed=3, reward=reward, auto_reset=False)


@needs_nvcc
def test_emu_return_saturates_past_done():
    """A plain-gym env (auto_reset = 0) stepped on past done earns the finish bonus on every step; 2.5e5 steps take the
    return past 2^31 centi, where it must stay at the int32 maximum (it wrapped to negative values before)."""
    from edge_rooms import degenerate_rooms
    from emu_rollout import EmuRollout
    rooms = degenerate_rooms()[3:4]            # two free cells, one above the other: up and down visit both
    em = EmuRollout(2, rooms, L=4, auto_reset=False)
    em.reset()
    T = 250_000
    em.rollout(np.tile(np.array([[4], [5]], np.uint8), (T // 2, 2)))
    st = em.state()
    assert (st[:, 10] == 1).all(), "the env must be done"
    assert (st[:, 15] == INT32_MAX).all(), f"return so far {st[:, 15]}"

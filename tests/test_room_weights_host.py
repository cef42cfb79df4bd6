"""Weighted room draw (include/nav3d.h nav3d_set_room_weights) without a GPU.

The reference table builder (tests/room_weights_ref.py, the header's rule in Python integers) is checked in exact
arithmetic (``fractions``): the uniform table, exact zeros, exact uniformity for equal weights, the stated error bound,
rejection.  The host emulation runs the builder arithmetic and the binary-search draw of csrc/nav3d_core.cuh
(tests/emu/nav3d_emu_weights.cu), and must equal the reference table bit for bit and step lock-step with the C oracle's
envs resetting through the same table, through auto-resets and the fused rollout.
tools/emu_asan.sh runs this file under AddressSanitizer + UBSan too."""
from fractions import Fraction

import numpy as np
import pytest

from __graft_entry__ import find_nvcc
from conftest import ROOMS
from lockstep import compare_grids, compare_step
from nav3d.rooms import load_room_dir, load_room_file
import room_weights_ref as rw

TWO32 = 1 << 32
needs_nvcc = pytest.mark.skipif(find_nvcc() is None, reason="nvcc needed to build the host emulation")


def uniform_ref(n):
    return np.array([((j + 1) * TWO32 + n - 1) // n for j in range(n)], dtype=np.uint64)


def probs(cdf):
    c = [0] + [int(x) for x in cdf]
    return [Fraction(c[j + 1] - c[j], TWO32) for j in range(len(cdf))]


def bound(n, p):
    """include/nav3d.h: |P_j - w_j / W| <= (2 + (n - 1) w_j / W) 2^-32 + 2^-52."""
    return (2 + (n - 1) * p) * Fraction(1, TWO32) + Fraction(1, 1 << 52)


def random_vectors(rng, count=200):
    out = []
    for i in range(count):
        n = int(rng.integers(1, 48))
        kind = i % 6
        if kind == 0:
            w = rng.random(n)
        elif kind == 1:
            w = rng.random(n) * (rng.random(n) < 0.5)               # zeros
        elif kind == 2:
            w = np.exp(rng.normal(0, 20, n).clip(-80, 80))                       # magnitudes far apart: q_j rounds to 0 for some rooms
        elif kind == 3:
            w = np.zeros(n); w[rng.integers(0, n)] = rng.random() + 1e-3   # a single nonzero room
        elif kind == 4:
            w = rng.random(n); w[0] = 0.0; w[-1] = 0.0 if n > 1 else 1.0    # first and last room at zero
        else:
            w = rng.integers(0, 4, n).astype(np.float64)           # small integers with ties
        w = w.astype(np.float32)
        if not (w > 0).any():
            w[-1] = 1.0
        out.append(w)
    return out


def test_uniform_table_and_its_search(oracle):
    rng = np.random.default_rng(0)
    sizes = list(range(1, 2049)) + sorted(int(x) for x in rng.integers(2049, 65536, 64)) + [65535]
    for n in sizes:
        want = uniform_ref(n)
        st, cdf = rw.cdf_build(None, n)
        assert st == 0 and np.array_equal(cdf, want), n
        st, cdf = rw.cdf_build(np.full(n, 0.37, np.float32))
        assert st == 0 and np.array_equal(cdf, want), f"equal weights at n={n}"
        # the search over the uniform table is (u * n) >> 32: edge words around every threshold and random words
        edges = np.concatenate([want[:-1], want[:-1] - 1, [0, 1, TWO32 - 1, TWO32 >> 1]]).astype(np.uint64)
        u = np.concatenate([edges[edges < TWO32], rng.integers(0, TWO32, 64, dtype=np.uint64)])
        room = np.searchsorted(want[:-1], u, side="right")
        assert np.array_equal(room, (u * np.uint64(n)) >> np.uint64(32)), n
        for x in u[:: max(1, len(u) // 8)]:
            assert rw.cdf_draw(want, int(x)) == (int(x) * n) >> 32 == rw.cdf_draw(None, int(x), n)


def test_weighted_tables_exact_properties(oracle):
    for w in random_vectors(np.random.default_rng(1)):
        n = len(w)
        st, cdf = rw.cdf_build(w)
        assert st == 0
        assert int(cdf[-1]) == TWO32 and (np.diff(cdf.astype(np.int64)) >= 0).all()
        P = probs(cdf)
        W = sum(Fraction(float(x)) for x in w)
        for j in range(n):
            p = Fraction(float(w[j])) / W
            if w[j] == 0:
                assert P[j] == 0, (w, j)
            assert abs(P[j] - p) <= bound(n, p), (w, j, float(P[j] - p))
            q = int((float(w[j]) / float(w.max())) * 4294967296.0)
            if w[j] > 0 and q == 0:
                assert P[j] == 0, "a positive weight that q_j rounds to 0 is never drawn"


def test_positive_weight_below_resolution_has_probability_zero(oracle):
    w = np.array([1.0, 1e-10, 0.5], np.float32)
    st, cdf = rw.cdf_build(w)
    assert st == 0 and probs(cdf)[1] == 0 and probs(cdf)[0] > 0


def test_bound_is_reached_within_the_stated_form(oracle):
    """Many rooms just under one q unit each: the large room carries almost all of their lost mass, which is what the
    (n - 1) w_j / W term of the bound covers."""
    n = 1000
    w = np.full(n, np.float32(0.99 / TWO32), np.float32); w[0] = 1.0
    st, cdf = rw.cdf_build(w)
    P = probs(cdf)
    W = sum(Fraction(float(x)) for x in w)
    p0 = Fraction(float(w[0])) / W
    assert P[0] == 1 and abs(P[0] - p0) > 100 * Fraction(1, TWO32) and abs(P[0] - p0) <= bound(n, p0)


@pytest.mark.parametrize("bad", ["nan", "inf", "-inf", "negative", "zeros", "negative_zeros"])
def test_rejected_vectors(oracle, bad):
    w = np.array([1.0, 2.0, 0.5, 3.0], np.float32)
    if bad == "nan":
        w[2] = np.nan
    elif bad == "inf":
        w[1] = np.inf
    elif bad == "-inf":
        w[3] = -np.inf
    elif bad == "negative":
        w[0] = -1e-30
    elif bad == "zeros":
        w[:] = 0
    else:
        w[:] = -0.0
    st, cdf = rw.cdf_build(w)
    assert st == 1 and cdf is None


def test_negative_zero_counts_as_zero(oracle):
    w = np.array([-0.0, 1.0, 2.0], np.float32)
    st, cdf = rw.cdf_build(w)
    assert st == 0 and probs(cdf)[0] == 0 and np.array_equal(cdf, rw.cdf_build(np.abs(w))[1])


# ---- host emulation ----------------------------------------------------------------------------------------------------

def lockstep_rooms(simple=False):
    """Rooms where episodes end within a few hundred random steps, plus shells of tests/edge_rooms.py."""
    rooms = [load_room_file(ROOMS / "P3_training" / "maze_3d_tunnels.txt", simple=simple),
             load_room_file(ROOMS / "P2_training" / "tightcorridor.txt", simple=simple)]
    if simple:
        return rooms + [load_room_file(ROOMS / "P3_training" / "kitchen2.txt", simple=True)]
    from edge_rooms import degenerate_rooms
    return rooms + load_room_dir(ROOMS / "P1_training", sort=True)[:2] + degenerate_rooms()


WEIGHTS = {"cubic": np.array([5.0, 0.0, 1.0, 0.25, 3.0, 0.0, 2.0, 1.5], np.float32),
           "simple": np.array([0.0, 3.0, 1.0], np.float32)}


@needs_nvcc
def test_emulated_builder_equals_oracle(oracle):
    from emu_weights import EmuWeights
    rooms = lockstep_rooms()
    em = EmuWeights(4, rooms, L=10)
    assert np.array_equal(em.room_cdf(), uniform_ref(len(rooms)))
    for w in random_vectors(np.random.default_rng(2), 60):
        full = np.zeros(len(rooms), np.float32)
        full[: min(len(w), len(rooms))] = w[: len(rooms)]
        if not (full > 0).any():
            full[0] = 1.0
        st, want = rw.cdf_build(full)
        assert em.set_room_weights(full) == st == 0
        assert np.array_equal(em.room_cdf(), want), full
    before = em.room_cdf()
    for bad in (np.nan, np.inf, -1.0):
        w = np.ones(len(rooms), np.float32); w[3] = bad
        assert em.set_room_weights(w) == 1 and np.array_equal(em.room_cdf(), before)
    assert em.set_room_weights(np.zeros(len(rooms), np.float32)) == 1 and np.array_equal(em.room_cdf(), before)
    assert em.set_room_weights(None) == 0 and np.array_equal(em.room_cdf(), uniform_ref(len(rooms)))


@needs_nvcc
def test_emulated_builder_at_65535_rooms(oracle):
    """The builder's arithmetic at the engine's largest room count (the emulation is given copies of one tiny room)."""
    from emu_weights import EmuWeights
    from edge_rooms import degenerate_rooms
    tiny = degenerate_rooms()[0]
    n = 65535
    em = EmuWeights(1, [tiny] * n, L=4)
    assert np.array_equal(em.room_cdf(), uniform_ref(n))
    w = np.random.default_rng(3).random(n).astype(np.float32) * (np.arange(n) % 7 != 0)
    st, want = rw.cdf_build(w)
    assert em.set_room_weights(w) == st == 0 and np.array_equal(em.room_cdf(), want)


def weighted_pair(oracle, rooms, n, seed, lanes=1, auto_reset=True, weights=None):
    from emu_weights import EmuWeights
    em = EmuWeights(n, rooms, L=10, seed=seed, auto_reset=auto_reset, lanes=lanes)
    w = WEIGHTS["cubic"] if weights is None else weights
    st, cdf = rw.cdf_build(w)
    assert st == 0 and em.set_room_weights(w) == 0
    ov = rw.WeightedOracleVec(n, [oracle.OracleRoom(r.grid, -2) for r in rooms], 10, -2.0, seed, 0, auto_reset, cdf)
    return em, ov


@needs_nvcc
@pytest.mark.parametrize("lanes", [1, 4])
@pytest.mark.parametrize("auto_reset", [True, False])
def test_emulated_steps_follow_the_weighted_table(oracle, lanes, auto_reset):
    rooms = lockstep_rooms()
    n = 48
    em, ov = weighted_pair(oracle, rooms, n, seed=11 + lanes, lanes=lanes, auto_reset=auto_reset)
    assert np.array_equal(em.reset().view(np.uint32), ov.reset().view(np.uint32))
    rng = np.random.default_rng(lanes)
    n_done, seen = 0, set()
    for t in range(330):
        a = rng.integers(0, 6, size=n)
        ov.step(a), em.step(a)
        st = em.state()
        compare_step(f"weighted emu lanes={lanes}", t, ov, em.obs, em.reward, em.reward64, em.term, em.trunc, em.tobs,
                     em.eps, st)
        n_done += int((ov.terminated | ov.truncated).sum())
        seen |= set(st[:, 13].tolist())
    assert n_done > 0
    assert not seen & {1, 5}, f"rooms of weight 0 were drawn: {sorted(seen)}"
    compare_grids("weighted emu", ov, em.grid, range(0, n, 7))


@needs_nvcc
def test_emulated_rollout_actions_follow_the_weighted_table(oracle):
    """The fused rollout's in-loop auto-resets (tests/emu/nav3d_emu_rollout.cu) draw from the table, every output checked."""
    from emu_weights import EmuWeights
    rooms = lockstep_rooms()
    n, T = 40, 330
    em = EmuWeights(n, rooms, L=10, seed=5)
    st, cdf = rw.cdf_build(WEIGHTS["cubic"])
    assert em.set_room_weights(WEIGHTS["cubic"]) == 0
    ov = rw.WeightedOracleVec(n, [oracle.OracleRoom(r.grid, -2) for r in rooms], 10, -2.0, 5, 0, True, cdf)
    assert np.array_equal(em.reset().view(np.uint32), ov.reset().view(np.uint32))
    acts = np.random.default_rng(6).integers(0, 6, size=(T, n)).astype(np.uint8)
    o = dict(obs=np.zeros((T, n, 80), np.float32), reward=np.zeros((T, n), np.float32),
             reward64=np.zeros((T, n), np.float64), term=np.zeros((T, n), np.uint8), trunc=np.zeros((T, n), np.uint8),
             tobs=np.zeros((T, n, 80), np.float32), eps=np.zeros((T, n, 8), np.int32))
    em.rollout(acts, **o)
    n_done = 0
    for t in range(T):
        ov.step(acts[t])
        compare_step("weighted emu rollout", t, ov, o["obs"][t], o["reward"][t], o["reward64"][t], o["term"][t],
                     o["trunc"][t], o["tobs"][t], o["eps"][t], None)
        n_done += int((ov.terminated | ov.truncated).sum())
    assert n_done > 0
    assert np.array_equal(em.state()[:, :15].astype(np.int64), ov.state())


@needs_nvcc
def test_emulated_simple_env_follows_the_weighted_table(oracle):
    from emu_weights import EmuWeights
    rooms = lockstep_rooms(simple=True)
    n, L, seed = 48, 10, 7
    st, cdf = rw.cdf_build(WEIGHTS["simple"])
    ov = rw.WeightedSimpleVec(n, [oracle.OracleRoom(r.grid, 2) for r in rooms], L, 0.25, seed, 0, True, cdf=cdf)
    em = EmuWeights(n, rooms, L=L, seed=seed, simple=True)
    assert em.set_room_weights(WEIGHTS["simple"]) == 0
    assert np.array_equal(em.reset().view(np.uint32), ov.reset().view(np.uint32))
    rng = np.random.default_rng(seed)
    n_done = 0
    for t in range(330):
        a = rng.integers(0, 6, size=n)
        ov.step(a), em.step(a)
        assert np.array_equal(em.obs.view(np.uint32), ov.obs.view(np.uint32)), t
        assert np.array_equal(em.reward64, ov.reward), t
        assert np.array_equal(em.term, ov.terminated) and np.array_equal(em.trunc, ov.truncated), t
        assert np.array_equal(em.state()[:, 13], np.array(ov.room_idx)), t
        n_done += int((ov.terminated | ov.truncated).sum())
    assert n_done > 0 and 0 not in set(ov.room_idx)


def test_reference_picks_are_the_oracle_picks(oracle):
    """Without a table, and with the uniform one, the reference's Philox picks are the C oracle's own (orc_pick / orc_pick3):
    the restatement keys the reset stream exactly as the oracle and the engine do."""
    nf = [7, 1, 130, 52, 9]
    _, uni = rw.cdf_build(None, len(nf))
    for seed in (0, 1, 0x123456789ABCDEF):
        for env in (0, 5, 0xFFFFFFFF):
            for ep in (0, 1, 77):
                assert rw.pick(seed, env, ep, nf) == rw.pick(seed, env, ep, nf, uni) == oracle.pick(seed, env, ep, nf)
                assert rw.pick3(seed, env, ep, nf) == rw.pick3(seed, env, ep, nf, uni) == oracle.pick3(seed, env, ep, nf)


@needs_nvcc
def test_emulation_without_a_table_draws_uniformly(oracle):
    """An emulated engine that is never given a table (the draw's host-only fallback) resets exactly as one holding the
    uniform table."""
    from emu_weights import EmuWeights
    rooms = lockstep_rooms()
    a, b = EmuWeights(64, rooms, L=10, seed=3), EmuWeights(64, rooms, L=10, seed=3)
    assert b.set_room_weights(None) == 0
    assert np.array_equal(a.reset().view(np.uint32), b.reset().view(np.uint32))
    rng = np.random.default_rng(3)
    for _ in range(330):
        x = rng.integers(0, 6, size=64)
        a.step(x), b.step(x)
    assert np.array_equal(a.state(), b.state())

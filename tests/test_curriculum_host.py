"""CPU checks of the room curriculum: the room_stats reference against a plain loop, the learning-progress rule (nav3d/
curriculum.py lp_rule) against its float64 NumPy restatement, RoomCurriculum state round trips, and a gloo world-size-2
run in which both ranks install identical weights computed from the summed windows."""
import ctypes
import os
import socket
import sys
from pathlib import Path

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import room_stats_ref as ref

ROOT = Path(__file__).resolve().parent.parent
HERE = Path(__file__).resolve().parent


class FakeEngine:
    """The part of nav3d.Engine a RoomCurriculum uses, on the CPU: room_stats through the reference, and a record of the
    weight vectors it is given."""

    def __init__(self, room_free):
        self.device = torch.device("cpu")
        self.room_free = list(room_free)
        self.installed = []

    def room_stats(self, terminated, truncated, episodes, out=None):
        s, _ = ref.room_stats_ref(terminated.numpy(), truncated.numpy(), episodes.numpy(), len(self.room_free))
        out += torch.from_numpy(s)
        return out

    def set_room_weights(self, weights, *, check=True):
        self.installed.append(weights.clone())


def test_room_stat_struct_is_64_bytes():
    from nav3d._lib import RoomStat
    from nav3d.engine import ROOM_STAT_FIELDS
    assert ctypes.sizeof(RoomStat) == 64 and RoomStat.return_centi_sum.offset == 48
    assert tuple(f for f, _ in RoomStat._fields_) == ROOM_STAT_FIELDS == ref.FIELDS


def test_reference_equals_plain_loop():
    rng = np.random.default_rng(0)
    for R, T, N, d in ((1, 3, 17, 0.5), (5, 4, 33, 0.2), (3, 2, 40, 1.0), (7, 1, 50, 0.0)):
        te, tr, ep = ref.random_rows(rng, T, N, R, d)
        # a few flagged rows the call must reject: rooms out of range, NaN / inf / huge returns
        flat = ep.reshape(-1, 8)
        done = np.nonzero((te | tr).reshape(-1))[0]
        if len(done) >= 4:
            flat[done[0], 5] = R
            flat[done[1], 5] = -1
            flat[done[2], 0] = np.array([np.nan], np.float32).view(np.int32)[0]
            flat[done[3], 0] = np.array([1e18], np.float32).view(np.int32)[0]
        a, bad_a = ref.room_stats_ref(te, tr, ep, R)
        b, bad_b = ref.room_stats_loop(te, tr, ep, R)
        assert np.array_equal(a, b) and bad_a == bad_b == (len(done) >= 4)
    # half-way cents round to even
    te = np.ones(4, np.uint8)
    ep = np.zeros((4, 8), np.int32)
    ep[:, 0] = np.array([0.125, 0.375, -0.125, 2.5], np.float32).view(np.int32)   # 12.5, 37.5, -12.5, 250 cents
    s, _ = ref.room_stats_ref(te, np.zeros(4, np.uint8), ep, 1)
    assert s[0, 6] == 12 + 38 - 12 + 250


def rule(window, tf, fast, slow, seen, **kw):
    from nav3d.curriculum import lp_rule
    t = lambda x, dt: torch.as_tensor(np.asarray(x), dtype=dt)   # noqa: E731
    out = lp_rule(t(window, torch.int64), t(tf, torch.float64), t(fast, torch.float64), t(slow, torch.float64),
                  t(seen, torch.bool), kw.get("alpha_fast", 0.1), kw.get("alpha_slow", 0.02), kw.get("uniform_mix", 0.2))
    return [o.numpy() for o in out]


def window_of(n, visited):
    w = np.zeros((len(n), 8), np.int64)
    w[:, 0], w[:, 5] = n, visited
    return w


def test_rule_matches_reference():
    rng = np.random.default_rng(1)
    R = 9
    tf = rng.integers(1, 500, R).astype(np.float64)
    fast, slow, seen = np.zeros(R), np.zeros(R), np.zeros(R, bool)
    for it in range(30):
        n = rng.integers(0, 5, R) * (rng.random(R) < 0.7)
        w = window_of(n, (n * tf * rng.random(R)).astype(np.int64))
        got = rule(w, tf, fast, slow, seen)
        want = ref.lp_rule_ref(w, tf, fast, slow, seen)
        for g, x in zip(got, want):
            assert np.allclose(g, x, rtol=1e-12, atol=0), it
        assert np.array_equal(got[2], want[2])
        fast, slow, seen = want[0], want[1], want[2]
        assert abs(got[4].sum() - 1.0) < 1e-12


def test_rule_no_data_is_uniform_and_first_observation_initialises_both_averages():
    R = 4
    tf = np.array([10.0, 20.0, 30.0, 40.0])
    z = np.zeros(R)
    fast, slow, seen, lp, p = rule(window_of([0] * R, [0] * R), tf, z, z, np.zeros(R, bool))
    assert not seen.any() and np.array_equal(p, np.full(R, 0.25)) and np.array_equal(lp, np.ones(R))
    fast, slow, seen, lp, p = rule(window_of([2, 0, 1, 0], [10, 0, 15, 0]), tf, z, z, np.zeros(R, bool))
    assert np.array_equal(seen, [True, False, True, False])
    assert fast[0] == slow[0] == 0.5 and fast[2] == slow[2] == 0.5
    # observed rooms have no progress yet and the unobserved ones stand in with 1: they share the (1 - eps) part
    assert np.array_equal(lp, [0.0, 1.0, 0.0, 1.0])
    assert np.allclose(p, [0.05, 0.45, 0.05, 0.45], rtol=1e-15)


def test_constant_score_room_gets_the_uniform_floor():
    """Room 0 always scores 1 (the one-cell room); room 1 improves; room 2 is never observed."""
    R, eps = 3, 0.2
    tf = np.array([1.0, 50.0, 20.0])
    fast, slow, seen = np.zeros(R), np.zeros(R), np.zeros(R, bool)
    for it in range(6):
        fast, slow, seen, lp, p = rule(window_of([8, 2, 0], [8, 2 * (10 + 5 * it), 0]), tf, fast, slow, seen,
                                       uniform_mix=eps)
        assert lp[0] == 0.0
        if it == 0:                                            # no progress yet: the unobserved room stands in with 1
            assert np.array_equal(lp, [0.0, 0.0, 1.0])
            assert np.allclose(p, [eps / R, eps / R, eps / R + 1 - eps], rtol=1e-15)
        else:
            assert lp[1] > 0 and lp[2] == lp[1]                # the unobserved room stands in with the best LP
            assert abs(p[0] - eps / R) <= 1e-15
            assert abs(p[1] - p[2]) <= 1e-15 and abs(p.sum() - 1.0) <= 1e-15


def test_state_dict_round_trip():
    from nav3d.curriculum import RoomCurriculum
    rng = np.random.default_rng(2)
    eng = FakeEngine([1, 36, 70])
    cur = RoomCurriculum(eng, alpha_fast=0.3, alpha_slow=0.05, uniform_mix=0.1)
    for _ in range(3):
        te, tr, ep = ref.random_rows(rng, 4, 16, 3, 0.4, max_len=30)
        ep[..., 3] = np.minimum(np.abs(ep[..., 3]), 1)
        cur.observe(torch.from_numpy(te), torch.from_numpy(tr), torch.from_numpy(ep))
        cur.update()
    te, tr, ep = ref.random_rows(rng, 2, 16, 3, 0.4)
    cur.observe(torch.from_numpy(te), torch.from_numpy(tr), torch.from_numpy(ep))     # a window in progress
    sd = cur.state_dict()
    eng2 = FakeEngine([1, 36, 70])
    other = RoomCurriculum(eng2)
    other.load_state_dict(sd)
    for k, v in other.state_dict().items():
        assert (torch.equal(v, sd[k]) if isinstance(v, torch.Tensor) else v == sd[k]), k
    assert torch.equal(eng2.installed[-1], eng.installed[-1])
    cur.update(); other.update()
    assert torch.equal(cur.probabilities(), other.probabilities())


def _worker(rank, world, port, out):
    for p in (str(ROOT), str(HERE)):
        if p not in sys.path:
            sys.path.insert(0, p)
    import _nav3d_path  # noqa: F401
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.set_num_threads(1)
    from nav3d.curriculum import RoomCurriculum
    eng = FakeEngine([1, 36, 70, 12])
    cur = RoomCurriculum(eng)
    rng = np.random.default_rng(10 + rank)                # different episodes per rank
    windows = []
    for _ in range(3):
        te, tr, ep = ref.random_rows(rng, 3, 32, 4, 0.3, max_len=10)
        cur.observe(torch.from_numpy(te), torch.from_numpy(tr), torch.from_numpy(ep))
        windows.append(cur.window.clone())
        cur.update()
    parts = [[torch.zeros_like(w) for _ in range(world)] for w in windows]
    for w, pl in zip(windows, parts):
        dist.all_gather(pl, w)
    if rank == 0:
        np.savez(out, w0=np.stack([torch.stack(p).numpy() for p in parts]),
                 a=torch.stack(eng.installed).numpy())
    else:
        np.savez(out + ".1.npz", a=torch.stack(eng.installed).numpy())
    dist.barrier()
    dist.destroy_process_group()


def test_gloo_ranks_install_identical_weights(tmp_path):
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    out = str(tmp_path / "cur.npz")
    mp.spawn(_worker, args=(2, port, out), nprocs=2, join=True)
    z0, z1 = np.load(out), np.load(out + ".1.npz")
    assert np.array_equal(z0["a"], z1["a"])
    # one process applying the rule to the summed windows installs the same weights
    tf = np.array([1.0, 36.0, 70.0, 12.0])
    fast, slow, seen = np.zeros(4), np.zeros(4), np.zeros(4, bool)
    for k, per_rank in enumerate(z0["w0"]):
        fast, slow, seen, _, p = ref.lp_rule_ref(per_rank.sum(axis=0), tf, fast, slow, seen)
        assert np.allclose(z0["a"][k].astype(np.float64), p.astype(np.float32).astype(np.float64), rtol=1e-6, atol=0)

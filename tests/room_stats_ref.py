"""Reference for per-room episode statistics (include/nav3d.h nav3d_room_stats) in exact NumPy integers, and a float64
NumPy restatement of the learning-progress room curriculum (nav3d/curriculum.py lp_rule).  Test infrastructure only."""
import numpy as np

FIELDS = ("episodes", "terminated", "time_limit", "length_sum", "bumps_sum", "visited_sum", "return_centi_sum", "reserved")
TWO63 = 9223372036854775808.0


def room_stats_ref(terminated, truncated, episodes, n_rooms):
    """(int64 [n_rooms, 8], bad): the sums nav3d_room_stats adds for flags u8 [..., N] and episodes int32 [..., N, 8].
    Row counted iff terminated | truncated; a flagged row with room outside 0..n_rooms-1, or a return that is not finite
    or has |100 * return| >= 2^63, is dropped and makes bad True.  Sums wrap mod 2^64 (int64 arithmetic)."""
    te = np.asarray(terminated, np.uint8).reshape(-1)
    tr = np.asarray(truncated, np.uint8).reshape(-1)
    ep = np.ascontiguousarray(episodes, np.int32).reshape(-1, 8)
    rows = np.nonzero((te | tr) != 0)[0]
    e = ep[rows]
    room = e[:, 5].astype(np.int64)
    ret100 = 100.0 * e[:, 0].view(np.float32).astype(np.float64)
    with np.errstate(invalid="ignore"):
        ok = (room >= 0) & (room < n_rooms) & (np.abs(ret100) < TWO63)
    bad = bool((~ok).any())
    rows, e, room, ret100 = rows[ok], e[ok], room[ok], ret100[ok]
    is_term = te[rows] != 0
    cols = [np.ones(len(rows), np.int64), is_term.astype(np.int64), (~is_term).astype(np.int64),
            e[:, 1].astype(np.int64), e[:, 2].astype(np.int64), e[:, 3].astype(np.int64), np.rint(ret100).astype(np.int64)]
    out = np.zeros((n_rooms, 8), np.int64)
    if len(rows):
        order = np.argsort(room, kind="stable")
        r_sorted = room[order]
        starts = np.r_[0, np.nonzero(np.diff(r_sorted))[0] + 1]
        with np.errstate(over="ignore"):
            for k, c in enumerate(cols):
                out[r_sorted[starts], k] = np.add.reduceat(c[order], starts)
    return out, bad


def room_stats_loop(terminated, truncated, episodes, n_rooms):
    """The same definition as a plain Python loop over rows (Python integers, wrapped to int64 at the end)."""
    te = np.asarray(terminated, np.uint8).reshape(-1)
    tr = np.asarray(truncated, np.uint8).reshape(-1)
    ep = np.ascontiguousarray(episodes, np.int32).reshape(-1, 8)
    acc = [[0] * 8 for _ in range(n_rooms)]
    bad = False
    for i in range(len(te)):
        if not (te[i] or tr[i]):
            continue
        room = int(ep[i, 5])
        r = float(ep[i, 0:1].view(np.float32)[0])
        if not (0 <= room < n_rooms) or not np.isfinite(r) or abs(100.0 * r) >= TWO63:
            bad = True
            continue
        a = acc[room]
        a[0] += 1
        a[1] += int(te[i] != 0)
        a[2] += int(te[i] == 0)
        a[3] += int(ep[i, 1]); a[4] += int(ep[i, 2]); a[5] += int(ep[i, 3])
        a[6] += int(round(100.0 * r))               # Python's round is half to even, 100 * r is exact in f64
    wrap = lambda v: ((v + (1 << 63)) % (1 << 64)) - (1 << 63)   # noqa: E731
    return np.array([[wrap(v) for v in a] for a in acc], np.int64).reshape(n_rooms, 8), bad


def lp_rule_ref(window, total_free, fast, slow, seen, alpha_fast=0.1, alpha_slow=0.02, uniform_mix=0.2):
    """The curriculum rule in float64 NumPy, element by element: returns new (fast, slow, seen, lp, p)."""
    window = np.asarray(window, np.int64)
    R = window.shape[0]
    fast, slow, seen = np.array(fast, np.float64), np.array(slow, np.float64), np.array(seen, bool)
    for j in range(R):
        n = int(window[j, 0])
        if n == 0:
            continue
        m = float(window[j, 5]) / (float(n) * float(total_free[j]))
        if not seen[j]:
            fast[j] = slow[j] = m
            seen[j] = True
        else:
            fast[j] = fast[j] + alpha_fast * (m - fast[j])
            slow[j] = slow[j] + alpha_slow * (m - slow[j])
    lp = np.where(seen, np.abs(fast - slow), 0.0)
    best = lp[seen].max() if seen.any() else 0.0
    lp = np.where(seen, lp, best if best > 0 else 1.0)
    total = lp.sum()
    p = uniform_mix / R + (1.0 - uniform_mix) * lp / total if total > 0 else np.full(R, 1.0 / R)
    return fast, slow, seen, lp, p


def random_rows(rng, T, N, n_rooms, density, max_len=4096):
    """Flags u8 [T, N] and episodes int32 [T, N, 8] with `density` of the rows done (a third terminated only, a third
    truncated only, a third both); every other row holds garbage (random words, rooms out of range included)."""
    M = T * N
    eps = rng.integers(-2 ** 31, 2 ** 31, size=(M, 8), dtype=np.int32)
    done = rng.random(M) < density
    kind = rng.integers(0, 3, M)
    te = (done & (kind != 1)).astype(np.uint8) * rng.integers(1, 256, M).astype(np.uint8)
    tr = (done & (kind != 0)).astype(np.uint8) * rng.integers(1, 256, M).astype(np.uint8)
    te[done & (kind != 1) & (te == 0)] = 1
    tr[done & (kind != 0) & (tr == 0)] = 1
    d = np.nonzero(done)[0]
    ret = (rng.standard_normal(len(d)) * 300.0).astype(np.float32)
    eps[d, 0] = ret.view(np.int32)
    eps[d, 1] = rng.integers(1, max_len, len(d))
    eps[d, 2] = rng.integers(0, max_len, len(d))
    eps[d, 3] = rng.integers(1, max_len, len(d))
    eps[d, 5] = rng.integers(0, n_rooms, len(d))
    return te.reshape(T, N), tr.reshape(T, N), eps.reshape(T, N, 8)

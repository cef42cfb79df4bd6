"""Scenarios of the env-state blob tests (nav3d_save_envs / nav3d_load_envs), shared by the host emulation
(tests/test_env_states_host.py) and the GPU (tests/test_gpu_env_states.py).

An engine adapter provides reset(picks=None), step(actions), state() -> int [n, 16], grid(env), save(ids) -> blobs,
load(ids, blobs) -> u8 status [n], take(blobs, idx) -> blobs[idx], and after every call the numpy attributes obs, reward,
reward64, term, trunc, tobs, eps (the rows the last step / reset / load wrote).  Every comparison is bit-exact."""
import numpy as np

from lockstep import compare_step


def outputs(e, ids, st=None):
    """The outputs of the listed envs after a step, with the rows that only a finished episode writes masked elsewhere."""
    st = e.state() if st is None else st
    done = ((e.term[ids] | e.trunc[ids]) != 0)[:, None]
    return {"obs": e.obs[ids].view(np.uint32).copy(), "reward64": e.reward64[ids].copy(),
            "reward": e.reward[ids].view(np.uint32).copy(), "term": e.term[ids].copy(), "trunc": e.trunc[ids].copy(),
            "tobs": np.where(done, e.tobs[ids].view(np.uint32), 0), "eps": np.where(done, e.eps[ids], 0),
            "state": st[ids].copy()}


def assert_same(tag, want, got):
    for k in want:
        if not np.array_equal(want[k], got[k]):
            rows = np.nonzero((want[k] != got[k]).reshape(len(want[k]), -1).any(axis=1))[0]
            raise AssertionError(f"{tag}: {k} differs in rows {rows[:8].tolist()}")


def round_trip(e, n_actions_seed, pre=130, post=130, frac=3):
    """Pre-roll, save a random 1/frac of the envs, record `post` steps, load the blobs back, replay the same actions: the
    loaded envs must repeat every output, their auto-resets included.  Returns the number of episode ends replayed."""
    rng = np.random.default_rng(n_actions_seed)
    n = e.n
    e.reset()
    for _ in range(pre):
        e.step(rng.integers(0, 6, size=n))
    ids = np.sort(rng.choice(n, n // frac, replace=False)).astype(np.int32)
    obs_at_save = e.obs[ids].view(np.uint32).copy()
    blobs = e.save(ids)
    acts = rng.integers(0, 6, size=(post, n))
    rec, n_end = [], 0
    for t in range(post):
        e.step(acts[t])
        rec.append(outputs(e, ids))
        n_end += int((e.term[ids] | e.trunc[ids]).sum())
    grids = [e.grid(int(i)) for i in ids]
    status = e.load(ids, blobs)
    assert (status == 0).all(), f"load status {np.unique(status)}"
    assert np.array_equal(e.obs[ids].view(np.uint32), obs_at_save), "loaded obs rows differ from the rows at save time"
    for t in range(post):
        e.step(acts[t])
        assert_same(f"round trip t={t}", rec[t], outputs(e, ids))
    for i, g in zip(ids, grids):
        assert np.array_equal(e.grid(int(i)), g), f"round trip: knowledge grid of env {i}"
    return n_end


def clone(e, seed, room_free, starts, pick, oracle_vec=None, pre=60, max_post=600, grid_every=40, simple=False):
    """Save env `a`, load that one blob into every other env, step all envs with the same action: every clone equals `a`
    until the common first auto-reset; then each clone's (room, start) is the Philox pick of its OWN global id at the
    blob's episode counter.  `pick(env, episode) -> (room, k[, kg])`; `starts[r]`: the room's free cells, or its fixed
    start.  `oracle_vec`: a CubicEnv oracle of the same n envs, stepped with the same actions: every env is compared with it
    before the save, env a alone after it (the oracle knows nothing of the clones)."""
    rng = np.random.default_rng(seed)
    n = e.n
    e.reset()
    acts_pre = rng.integers(0, 6, size=(pre, n))
    if oracle_vec is not None:
        oracle_vec.reset()
    for t in range(pre):
        e.step(acts_pre[t])
        if oracle_vec is not None:
            _oracle_step(oracle_vec, e, t, acts_pre[t], slice(0, n))
    st = e.state()
    # the env that will end its episode first (truncation at n_free steps), so that the reset comes within max_post
    left = np.array([room_free[st[i, 13]] - st[i, 6] for i in range(n)])
    a = int(np.argmin(left))
    assert left[a] < max_post
    blob = e.save(np.array([a], np.int32))
    dst = np.array([i for i in range(n) if i != a], np.int32)
    status = e.load(dst, e.take(blob, np.zeros(len(dst), np.int64)))
    assert (status == 0).all()
    st = e.state()
    assert (st[dst] == st[a]).all(), "clone records"
    assert (e.obs[dst].view(np.uint32) == e.obs[a].view(np.uint32)).all(), "clone observation rows"
    ga = e.grid(a)
    for i in dst:
        assert np.array_equal(e.grid(int(i)), ga), f"clone {i}: knowledge grid"
    episode = int(st[a, 14])
    every = np.arange(n)
    for t in range(max_post):
        act = int(rng.integers(0, 6))
        e.step(np.full(n, act))
        if oracle_vec is not None:
            _oracle_step(oracle_vec, e, pre + t, np.full(n, act), slice(a, a + 1))
        st = e.state()
        out = outputs(e, every, st)
        want = {k: np.repeat(v[a:a + 1], len(dst), axis=0) for k, v in out.items()}
        got = {k: v[dst] for k, v in out.items()}
        if e.term[a] | e.trunc[a]:
            # the step that ends the episode: identical up to the reset, whose picks are keyed by the destination
            for k in ("state", "obs"):
                want.pop(k), got.pop(k)
            assert_same(f"clone end t={t}", want, got)
            for i in every:
                p = pick(int(i), episode)
                r = p[0]
                assert st[i, 13] == r, f"clone {i}: room {st[i, 13]} after the reset, want {r}"
                assert st[i, 14] == episode + 1
                assert tuple(st[i, :3]) == tuple(starts[r][p[1]]), f"clone {i}: start {st[i, :3]} want {starts[r][p[1]]}"
                if simple:
                    assert tuple(st[i, 7:10]) == tuple(starts[r][p[2]]), f"clone {i}: goal"
            return t + 1
        assert_same(f"clone t={t}", want, got)
        if t % grid_every == 0:
            ga = e.grid(a)
            for i in dst[:: max(1, len(dst) // 8)]:
                assert np.array_equal(e.grid(int(i)), ga), f"clone {i} t={t}: knowledge grid"
    raise AssertionError("env a did not reach its auto-reset")


class _Rows:
    """The rows `r` of an oracle vector, with the attribute names lockstep.compare_step reads."""

    def __init__(self, ov, r):
        for k in ("obs", "reward", "terminated", "truncated", "terminal_obs", "ep_ret", "ep_len", "ep_bumps", "ep_visited"):
            setattr(self, k, getattr(ov, k)[r])
        self._state = ov.state()[r]

    def state(self):
        return self._state


def _oracle_step(ov, e, t, actions, r):
    ov.step(actions)
    compare_step("oracle", t, _Rows(ov, r), e.obs[r], e.reward[r], e.reward64[r], e.term[r], e.trunc[r], e.tobs[r], e.eps[r],
                 e.state()[r])


def live_part(e, picks, saturate_env=0):
    """Envs in rooms of different sizes (auto_reset off; `picks` puts env i and its twin i + n/2 in the same room): drive
    env `saturate_env` to a counter of 255 (bumping into the ceiling) and two cells to >= 29 (ping-pong), then load blob
    j -> env i across room sizes and check each loaded env against the twin of its source, step by step."""
    n = e.n
    h = n // 2
    e.reset(picks=picks)
    rng = np.random.default_rng(5)
    for t in range(900):
        a = rng.integers(0, 6, size=n)
        if t < 300:
            a[:] = 4                    # up until the ceiling, then bump in place: the counter saturates at 255
        elif t < 420:
            a[:] = 2                    # turn around and move: two cells counted up past 29 (overflow bytes)
        a[h:] = a[:h]
        e.step(a)
    g = e.grid(saturate_env)
    assert g.max() == 255, "no saturated counter"
    assert ((g >= 29) & (g < 255)).any(), "no counter in the overflow range"
    blobs = e.save(np.arange(h, dtype=np.int32))
    # env i <- blob of env perm[i]: a cycle over all the first half, so each env gets a room of another size
    perm = np.roll(np.arange(h), 1)
    want_grid = {i: e.grid(int(perm[i])) for i in range(h)}
    status = e.load(np.arange(h, dtype=np.int32), e.take(blobs, perm))
    assert (status == 0).all()
    st = e.state()
    twin = perm + h                     # the untouched twin of each env's source
    assert (st[:h] == st[twin]).all()
    assert (e.obs[:h].view(np.uint32) == e.obs[twin].view(np.uint32)).all()
    for i in range(h):
        assert np.array_equal(e.grid(i), want_grid[i]), f"env {i} <- blob {perm[i]}: knowledge grid"
    for t in range(300):
        a = rng.integers(0, 6, size=n)
        a[:h] = a[twin]
        e.step(a)
        out = outputs(e, np.arange(n))
        assert_same(f"live part t={t}", {k: v[twin] for k, v in out.items()}, {k: v[:h] for k, v in out.items()})
    for i in range(h):
        assert np.array_equal(e.grid(i), e.grid(int(twin[i]))), f"env {i}: knowledge grid after 300 steps"

"""Reference for the weighted room draw (include/nav3d.h nav3d_set_room_weights), restated from the header in Python
integers and IEEE f64 (Python's float division is correctly rounded, as the engine's): the table builder, the draw, the
Philox reset picks that go through it, and vec layers that auto-reset through a table on top of the C oracle's env dynamics
(oracle/c_oracle.py), which draws uniformly on its own.  Test infrastructure only."""
import numpy as np

from oracle import c_oracle

TWO32 = 1 << 32
STREAM_RESET = 0x52455345


def cdf_build(weights, n=None):
    """(status, uint64 cdf [n]): the uniform table for weights None (then n is needed), else the header's rule
    q_j = floor(fl64(w_j / w_max) * 2^32), C_j = q_0 + ... + q_j, cdf[j] = ceil(2^32 C_j / C_{n-1}).  Status 1 (cdf None)
    for a NaN, infinite or negative weight or an all-zero vector."""
    if weights is None:
        return 0, np.array([((j + 1) * TWO32 + n - 1) // n for j in range(n)], dtype=np.uint64)
    w = [float(x) for x in np.ascontiguousarray(weights, dtype=np.float32).ravel()]
    if any(not np.isfinite(x) or x < 0 for x in w) or not any(x > 0 for x in w):
        return 1, None
    w_max = max(w)
    q = [int((x / w_max) * 4294967296.0) for x in w]
    total, c, out = sum(q), 0, []
    for qj in q:
        c += qj
        out.append(-(-(c << 32) // total))
    return 0, np.array(out, dtype=np.uint64)


def cdf_draw(cdf, u, n=None):
    """room = #{ j < n-1 : cdf[j] <= u }, the definition itself (cdf None: (u * n) >> 32)."""
    if cdf is None:
        return (int(u) * int(n)) >> 32
    c = np.asarray(cdf, dtype=np.uint64)
    return int(np.count_nonzero(c[:-1] <= np.uint64(u)))


def _reset_words(seed, env_id, episode):
    return c_oracle.philox4x32_10([int(env_id) & 0xFFFFFFFF, int(episode) & 0xFFFFFFFF, 0, STREAM_RESET],
                                  [int(seed) & 0xFFFFFFFF, (int(seed) >> 32) & 0xFFFFFFFF])


def pick(seed, env_id, episode, n_free, cdf=None):
    """(room, k) of a CubicEnv Philox reset: word 0 through the table, word 1 into the chosen room's free cells."""
    o = _reset_words(seed, env_id, episode)
    r = cdf_draw(cdf, o[0], len(n_free))
    return r, (int(o[1]) * int(n_free[r])) >> 32


def pick3(seed, env_id, episode, n_free, cdf=None):
    """(room, k, kg) of a simpleEnv Philox reset: word 2 picks the goal in the same room."""
    o = _reset_words(seed, env_id, episode)
    r = cdf_draw(cdf, o[0], len(n_free))
    return r, (int(o[1]) * int(n_free[r])) >> 32, (int(o[2]) * int(n_free[r])) >> 32


class WeightedOracleVec:
    """N CubicEnv oracles with the SB3 auto-reset whose Philox resets draw the room through `cdf` (None = uniform): one
    single-env c_oracle.OracleVec per env, reset with explicit picks (pick above), so the oracle's dynamics, episode
    records and state columns are used unchanged.  The attributes are those of c_oracle.OracleVec."""

    def __init__(self, n, orooms, L=10, crash_penalty=-2.0, seed=0, env_id0=0, auto_reset=True, cdf=None):
        self.n, self.seed, self.auto_reset, self.cdf = n, seed, auto_reset, cdf
        self.ids = [env_id0 + i for i in range(n)]
        self.n_free = [r.n_free for r in orooms]
        self.envs = [c_oracle.OracleVec(1, orooms, L, crash_penalty, seed, env_id0 + i, False) for i in range(n)]
        self.obs = np.zeros((n, 80), np.float32)
        self.terminal_obs = np.zeros((n, 80), np.float32)
        self.reward = np.zeros(n, np.float64)
        self.terminated = np.zeros(n, np.uint8)
        self.truncated = np.zeros(n, np.uint8)
        self.ep_ret = np.zeros(n, np.float64)
        self.ep_len = np.zeros(n, np.int64)
        self.ep_bumps = np.zeros(n, np.int64)
        self.ep_visited = np.zeros(n, np.int64)
        self.ep_ret32 = np.zeros(n, np.float32)

    def set_room_cdf(self, cdf=None):
        self.cdf = cdf

    def set_ids(self, ids):
        """Local env i plays global env ids[i] (to check a sample of a larger engine)."""
        self.ids = [int(i) for i in ids]

    def _reset_one(self, i):
        v = self.envs[i]
        episode = c_oracle.lib().orc_vec_episode(v.h, 0)
        v.reset(np.array([pick(self.seed, self.ids[i], episode, self.n_free, self.cdf)], dtype=np.int32))
        self.obs[i] = v.obs[0]

    def reset(self):
        for i in range(self.n):
            self._reset_one(i)
        return self.obs

    def step(self, actions):
        for i, v in enumerate(self.envs):
            v.step(np.array([actions[i]], dtype=np.int64))
            self.obs[i], self.reward[i] = v.obs[0], v.reward[0]
            self.terminated[i], self.truncated[i] = v.terminated[0], v.truncated[0]
            if v.terminated[0] or v.truncated[0]:
                self.ep_ret[i], self.ep_len[i], self.ep_bumps[i] = v.ep_ret[0], v.ep_len[0], v.ep_bumps[0]
                self.ep_visited[i], self.ep_ret32[i] = v.ep_visited[0], v.ep_ret32[0]
                if self.auto_reset:
                    self.terminal_obs[i] = v.obs[0]
                    self._reset_one(i)
        return self.obs, self.reward, self.terminated, self.truncated

    def state(self):
        return np.concatenate([v.state() for v in self.envs])

    def ret_centi(self):
        return np.concatenate([v.ret_centi() for v in self.envs])

    def grid(self, i):
        return self.envs[i].grid(0)


class WeightedSimpleVec(c_oracle.OracleSimpleVec):
    """c_oracle.OracleSimpleVec whose Philox resets draw the room through `cdf` (None = uniform)."""

    def __init__(self, *args, cdf=None, **kwargs):
        super().__init__(*args, **kwargs)
        self.cdf = cdf

    def _reset_one(self, i):
        r, k, kg = pick3(self.seed, self.env_id0 + i, self.episode[i], self.n_free, self.cdf)
        self.episode[i] += 1
        self.room_idx[i] = r
        room = self.rooms[r]
        self.envs[i].reset(room, room.free_cell(k), room.free_cell(kg))
        self.obs[i] = self.envs[i].get_obs()

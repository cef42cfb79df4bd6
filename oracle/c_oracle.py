"""ctypes front end of the CPU oracle (``nav3d_oracle.c``).  TEST INFRASTRUCTURE ONLY.

Imported only by tests/, ``__graft_entry__.smoke()`` and ``bench.py``'s cpu_baseline / ``--impl reference`` legs.
The product package never imports this module."""
from __future__ import annotations

import ctypes as C
import subprocess
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
LIB = HERE / "libnav3d_oracle.so"
_lib = None


def build(force: bool = False):
    src = HERE / "nav3d_oracle.c"
    if force or not LIB.exists() or LIB.stat().st_mtime < src.stat().st_mtime:
        subprocess.check_call(["make", "-C", str(HERE), "-B", "libnav3d_oracle.so"], stdout=subprocess.DEVNULL)
    return LIB


def lib():
    global _lib
    if _lib is not None:
        return _lib
    build()
    L = C.CDLL(str(LIB))
    P, I, D = C.c_void_p, C.c_int, C.c_double
    sig = {
        "orc_room_create": (P, [I, I, I, P, I]), "orc_room_destroy": (None, [P]), "orc_room_n_free": (I, [P]),
        "orc_room_free_cell": (None, [P, I, P]),
        "orc_cubic_create": (P, [I, D]), "orc_cubic_destroy": (None, [P]),
        "orc_cubic_reset": (None, [P, P, I, I, I, P]), "orc_cubic_step": (None, [P, I, P, P, P, P]),
        "orc_cubic_state": (None, [P, P]), "orc_cubic_grid": (P, [P]),
        "orc_simple_create": (P, [I, D]), "orc_simple_destroy": (None, [P]),
        "orc_simple_reset": (None, [P, P, I, I, I, I, I, I]), "orc_simple_obs": (None, [P, P]),
        "orc_simple_step": (None, [P, I, P, P, P, P]), "orc_simple_state": (None, [P, P]),
        "orc_simple_grid": (P, [P]),
        "orc_philox4x32_10": (None, [P, P, P]),
        "orc_pick": (None, [C.c_uint64, C.c_uint32, C.c_uint32, I, P, P, P]),
        "orc_action": (I, [C.c_uint64, C.c_uint32, C.c_uint32]),
        "orc_pick3": (None, [C.c_uint64, C.c_uint32, C.c_uint32, I, P, P, P, P]),
        "orc_vec_create": (P, [I, I, P, I, D, C.c_uint64, C.c_uint32, I]), "orc_vec_destroy": (None, [P]),
        "orc_vec_env": (P, [P, I]), "orc_vec_room_idx": (I, [P, I]), "orc_vec_episode": (C.c_uint32, [P, I]),
        "orc_vec_reset": (None, [P, P, P]), "orc_vec_set_ids": (None, [P, P]), "orc_vec_state": (None, [P, P]),
        "orc_vec_step": (None, [P, P, P, P, P, P, P, P, P, P, P]),
        "orc_vec_rollout_random": (C.c_long, [P, I, C.c_uint32, P, P]),
        "orc_vec_rollout_random_obs": (C.c_long, [P, I, C.c_uint32, P]),
        "orc_cubic_set_reward": (None, [P, P]), "orc_cubic_ret_centi": (C.c_long, [P]),
        "orc_cubic_episode_return": (C.c_float, [P]), "orc_py_round2": (D, [D]),
        "orc_vec_set_reward": (None, [P, P]), "orc_vec_ret_centi": (None, [P, P]), "orc_vec_ep_return32": (None, [P, P]),
        "orc_set_threads": (None, [I]), "orc_get_threads": (I, []), "orc_hw_threads": (I, []),
    }
    for name, (res, args) in sig.items():
        f = getattr(L, name)
        f.restype, f.argtypes = res, args
    _lib = L
    return L


def _p(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


REWARD_FIELDS = ("step_cost", "revisit_unit", "revisit_cap", "crash_penalty", "near_wall_bonus", "repeat_bonus",
                 "reverse_penalty", "explore_bonus", "finish_bonus", "truncation_penalty")
REWARD_DEFAULTS = dict(zip(REWARD_FIELDS, (-0.05, 0.02, 0.5, -2.0, 0.15, 0.05, 0.5, 1.0, 100.0, -5.0)))


def reward_values(reward=None, crash_penalty: float = -2.0) -> np.ndarray:
    """The ten reward parameters (include/nav3d.h ``nav3d_reward_params``, field order) as float64: the reference's
    literals with ``crash_penalty``, overridden by the entries of the dict ``reward``."""
    d = dict(REWARD_DEFAULTS, crash_penalty=crash_penalty)
    for k, v in (reward or {}).items():
        if k not in d:
            raise KeyError(f"unknown reward parameter {k!r}")
        d[k] = float(v)
    return np.array([d[k] for k in REWARD_FIELDS], dtype=np.float64)


def py_round2(x: float) -> float:
    """The oracle's restatement of CPython's ``round(x, 2)`` (simpleEnv distances)."""
    return lib().orc_py_round2(float(x))


class OracleRoom:
    def __init__(self, grid: np.ndarray, wall_code: int = -2):
        g = np.ascontiguousarray(grid, dtype=np.int8)
        self.grid = g
        self.dims = g.shape
        self.wall_code = wall_code
        self.h = lib().orc_room_create(g.shape[0], g.shape[1], g.shape[2], _p(g), wall_code)
        self.n_free = lib().orc_room_n_free(self.h)

    def free_cell(self, k: int):
        out = np.zeros(3, dtype=np.int32)
        lib().orc_room_free_cell(self.h, int(k), _p(out))
        return tuple(int(v) for v in out)

    def __del__(self):
        try:
            lib().orc_room_destroy(self.h)
        except Exception:  # noqa: BLE001
            pass


CUBIC_STATE = ("x", "y", "z", "facing", "visited_count", "bump_count", "step_count", "near_wall", "was_near_wall",
               "last_bump", "done", "cells_insight_down", "last_action")


class OracleCubic:
    """One CubicEnv ``GridAgent`` (reference ``envs/CubicEnv.py``) with injected (room, start) picks.  ``reward``: a dict
    of ``nav3d_reward_params`` fields that replace the reference's literals (``reward_values``)."""

    def __init__(self, L: int = 4, crash_penalty: float = -2.0, reward=None):
        self.L = L
        self.h = lib().orc_cubic_create(L, crash_penalty)
        self.room = None
        if reward is not None:
            self.set_reward(reward, crash_penalty)

    def set_reward(self, reward=None, crash_penalty: float = -2.0):
        self._rw = reward_values(reward, crash_penalty)
        lib().orc_cubic_set_reward(self.h, _p(self._rw))

    def ret_centi(self) -> int:
        """The running episode return in 1/100 units (nav3d_get_state column 15)."""
        return int(lib().orc_cubic_ret_centi(self.h))

    def episode_return(self) -> float:
        """nav3d_episode.episode_return for the episode so far (f32)."""
        return float(lib().orc_cubic_episode_return(self.h))

    def reset(self, room: OracleRoom, start) -> np.ndarray:
        self.room = room
        obs = np.zeros(80, dtype=np.float32)
        lib().orc_cubic_reset(self.h, room.h, int(start[0]), int(start[1]), int(start[2]), _p(obs))
        return obs

    def step(self, action: int):
        obs = np.zeros(80, dtype=np.float32)
        r = C.c_double()
        te, tr = C.c_int(), C.c_int()
        lib().orc_cubic_step(self.h, int(action), _p(obs), C.byref(r), C.byref(te), C.byref(tr))
        return obs, r.value, bool(te.value), bool(tr.value)

    def state(self) -> np.ndarray:
        out = np.zeros(13, dtype=np.int64)
        lib().orc_cubic_state(self.h, _p(out))
        return out

    def grid(self) -> np.ndarray:
        w, d, h = self.room.dims
        ptr = lib().orc_cubic_grid(self.h)
        return np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_long)), shape=(w, d, h)).copy()

    def __del__(self):
        try:
            lib().orc_cubic_destroy(self.h)
        except Exception:  # noqa: BLE001
            pass


class OracleSimple:
    """One simpleEnv ``GridAgent`` (reference ``envs/simpleEnv.py``) with injected (room, start, goal) picks."""

    def __init__(self, L: int = 4, cell_size: float = 0.25):
        self.L = L
        self.h = lib().orc_simple_create(L, cell_size)
        self.room = None

    @property
    def obs_dim(self):
        return 6 * self.L + 7

    def reset(self, room: OracleRoom, start, goal) -> None:
        self.room = room
        lib().orc_simple_reset(self.h, room.h, *[int(v) for v in start], *[int(v) for v in goal])

    def get_obs(self) -> np.ndarray:
        obs = np.zeros(self.obs_dim, dtype=np.float32)
        lib().orc_simple_obs(self.h, _p(obs))
        return obs

    def step(self, action: int):
        obs = np.zeros(self.obs_dim, dtype=np.float32)
        r = C.c_double()
        te, tr = C.c_int(), C.c_int()
        lib().orc_simple_step(self.h, int(action), _p(obs), C.byref(r), C.byref(te), C.byref(tr))
        return obs, r.value, bool(te.value), bool(tr.value)

    def state(self) -> np.ndarray:
        out = np.zeros(8, dtype=np.int64)
        lib().orc_simple_state(self.h, _p(out))
        return out

    def grid(self) -> np.ndarray:
        w, d, h = self.room.dims
        ptr = lib().orc_simple_grid(self.h)
        return np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_long)), shape=(w, d, h)).copy()

    def __del__(self):
        try:
            lib().orc_simple_destroy(self.h)
        except Exception:  # noqa: BLE001
            pass


def philox4x32_10(ctr, key) -> np.ndarray:
    c = np.asarray(ctr, dtype=np.uint32)
    k = np.asarray(key, dtype=np.uint32)
    o = np.zeros(4, dtype=np.uint32)
    lib().orc_philox4x32_10(_p(c), _p(k), _p(o))
    return o


def pick(seed: int, env_id: int, episode: int, n_free) -> tuple:
    nf = np.ascontiguousarray(n_free, dtype=np.int32)
    r, k = C.c_int(), C.c_int()
    lib().orc_pick(seed, env_id, episode, len(nf), _p(nf), C.byref(r), C.byref(k))
    return r.value, k.value


def pick3(seed: int, env_id: int, episode: int, n_free) -> tuple:
    nf = np.ascontiguousarray(n_free, dtype=np.int32)
    r, k, kg = C.c_int(), C.c_int(), C.c_int()
    lib().orc_pick3(seed, env_id, episode, len(nf), _p(nf), C.byref(r), C.byref(k), C.byref(kg))
    return r.value, k.value, kg.value


class OracleSimpleVec:
    """N simpleEnv oracles + auto-reset with Philox (room, start, goal) picks (mirrors the engine's NAV3D_ENV_SIMPLE mode:
    reset = the reference's reset() followed by one get_obs())."""

    def __init__(self, n, rooms, L=4, cell_size=0.25, seed=0, env_id0=0, auto_reset=True):
        self.n, self.rooms, self.L, self.seed, self.env_id0, self.auto_reset = n, list(rooms), L, seed, env_id0, auto_reset
        self.envs = [OracleSimple(L, cell_size) for _ in range(n)]
        self.episode = [0] * n
        self.room_idx = [0] * n
        self.n_free = [r.n_free for r in self.rooms]
        d = 6 * L + 7
        self.obs = np.zeros((n, d), np.float32)
        self.terminal_obs = np.zeros((n, d), np.float32)
        self.reward = np.zeros(n, np.float64)
        self.terminated = np.zeros(n, np.uint8)
        self.truncated = np.zeros(n, np.uint8)

    def _reset_one(self, i):
        r, k, kg = pick3(self.seed, self.env_id0 + i, self.episode[i], self.n_free)
        self.episode[i] += 1
        self.room_idx[i] = r
        room = self.rooms[r]
        self.envs[i].reset(room, room.free_cell(k), room.free_cell(kg))
        self.obs[i] = self.envs[i].get_obs()

    def reset(self):
        for i in range(self.n):
            self._reset_one(i)
        return self.obs

    def step(self, actions):
        for i in range(self.n):
            o, r, te, tr = self.envs[i].step(int(actions[i]))
            self.obs[i], self.reward[i], self.terminated[i], self.truncated[i] = o, r, te, tr
            if (te or tr) and self.auto_reset:
                self.terminal_obs[i] = o
                self._reset_one(i)

    def state(self):
        """int64 [n, 10]: x y z facing visited bump step done room episode"""
        out = np.zeros((self.n, 10), np.int64)
        for i, e in enumerate(self.envs):
            s = e.state()
            out[i] = [s[0], s[1], s[2], s[3], s[4], s[5], s[6], s[7], self.room_idx[i], self.episode[i]]
        return out


def action(seed: int, env_id: int, t: int) -> int:
    return lib().orc_action(seed, env_id, t)


class OracleVec:
    """N CubicEnv oracles + the SB3-VecEnv auto-reset contract + Philox picks (mirrors ``nav3d.BatchedCubicEnv``)."""

    def __init__(self, n: int, rooms, L: int = 4, crash_penalty: float = -2.0, seed: int = 0, env_id0: int = 0,
                 auto_reset: bool = True, reward=None):
        self.n = n
        self.rooms = list(rooms)
        self.crash_penalty = crash_penalty
        arr = (C.c_void_p * len(self.rooms))(*[r.h for r in self.rooms])
        self.h = lib().orc_vec_create(n, len(self.rooms), arr, L, crash_penalty, seed, env_id0, int(auto_reset))
        if reward is not None:
            self.set_reward(reward)
        self.obs = np.zeros((n, 80), dtype=np.float32)
        self.reward = np.zeros(n, dtype=np.float64)
        self.terminated = np.zeros(n, dtype=np.uint8)
        self.truncated = np.zeros(n, dtype=np.uint8)
        self.terminal_obs = np.zeros((n, 80), dtype=np.float32)
        self.ep_ret = np.zeros(n, dtype=np.float64)
        self.ep_len = np.zeros(n, dtype=np.int64)
        self.ep_bumps = np.zeros(n, dtype=np.int64)
        self.ep_visited = np.zeros(n, dtype=np.int64)
        self.ep_ret32 = np.zeros(n, dtype=np.float32)

    def set_reward(self, reward=None):
        """Replace the reward literals of every env from the next step on (a dict of ``nav3d_reward_params`` fields;
        unnamed fields take the reference's values and the vec's crash penalty)."""
        self._rw = reward_values(reward, self.crash_penalty)
        lib().orc_vec_set_reward(self.h, _p(self._rw))

    def ret_centi(self) -> np.ndarray:
        """int64 [n]: each env's running episode return in 1/100 units (nav3d_get_state column 15)."""
        out = np.zeros(self.n, dtype=np.int64)
        lib().orc_vec_ret_centi(self.h, _p(out))
        return out

    def reset(self, picks=None) -> np.ndarray:
        if picks is not None:
            picks = np.ascontiguousarray(picks, dtype=np.int32)
        lib().orc_vec_reset(self.h, _p(picks), _p(self.obs))
        return self.obs

    def step(self, actions):
        a = np.ascontiguousarray(actions, dtype=np.int64)
        lib().orc_vec_step(self.h, _p(a), _p(self.obs), _p(self.reward), _p(self.terminated), _p(self.truncated),
                           _p(self.terminal_obs), _p(self.ep_ret), _p(self.ep_len), _p(self.ep_bumps),
                           _p(self.ep_visited))
        lib().orc_vec_ep_return32(self.h, _p(self.ep_ret32))
        return self.obs, self.reward, self.terminated, self.truncated

    def rollout_random(self, T: int, t0: int = 0):
        rs, dc = C.c_double(), C.c_long()
        n = lib().orc_vec_rollout_random(self.h, T, t0, C.byref(rs), C.byref(dc))
        return n, rs.value, dc.value

    def rollout_random_obs(self, T: int, t0: int = 0) -> np.ndarray:
        """T random-action steps like ``rollout_random``; ``self.obs`` holds the observation after the last one."""
        lib().orc_vec_rollout_random_obs(self.h, T, t0, _p(self.obs))
        return self.obs

    def state(self) -> np.ndarray:
        """int64 [n, 15]: CUBIC_STATE columns + room index + episode number."""
        out = np.zeros((self.n, 15), dtype=np.int64)
        lib().orc_vec_state(self.h, _p(out))
        return out

    def set_ids(self, ids):
        """Local env i plays global env ``ids[i]`` (to check a sample of a larger sharded job)."""
        ids = np.ascontiguousarray(ids, dtype=np.uint32)
        assert ids.shape == (self.n,)
        lib().orc_vec_set_ids(self.h, _p(ids))

    def grid(self, i: int) -> np.ndarray:
        room = self.rooms[lib().orc_vec_room_idx(self.h, i)]
        w, d, h = room.dims
        ptr = lib().orc_cubic_grid(lib().orc_vec_env(self.h, i))
        return np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_long)), shape=(w, d, h)).copy()

    def __del__(self):
        try:
            lib().orc_vec_destroy(self.h)
        except Exception:  # noqa: BLE001
            pass


def set_threads(n: int):
    lib().orc_set_threads(int(n))


def hw_threads() -> int:
    return lib().orc_hw_threads()

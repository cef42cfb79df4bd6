"""``Engine``: one GPU's shard of batched environments — a thin, typed wrapper over the C ABI (``include/nav3d.h``).

PyTorch is used only for device memory and streams (tensors in, tensors out); all computation happens in the
library's CUDA kernels."""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import numpy as np
import torch

from . import _lib
from ._lib import Config, Nav3dError, RoomDesc, check
from .rooms import Room

EPISODE_DTYPE = np.dtype([("episode_return", np.float32), ("length", np.int32), ("bumps", np.int32),
                          ("visited", np.int32), ("total_free", np.int32), ("room", np.int32),
                          ("terminated", np.int32), ("truncated", np.int32)])

STATE_FIELDS = ("x", "y", "z", "facing", "visited_count", "bump_count", "step_count", "near_wall", "was_near_wall",
                "last_bump", "done", "cells_insight_down", "last_action", "room", "episode", "return_centi")


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


class Engine:
    def __init__(self, n_envs: int, rooms: Sequence[Room], *, local_map_length: int = 4, crash_penalty: float = -2.0,
                 auto_reset: bool = True, seed: int = 0, env_id0: int = 0, device: int = 0, lanes_per_env: int = 0,
                 env_kind: int = _lib.ENV_CUBIC, cell_size: float = 0.25):
        self._lib = _lib.load()
        self._h = C.c_void_p()
        if not torch.cuda.is_available():
            raise RuntimeError("nav3d needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        self.device = torch.device("cuda", int(device))
        cfg = Config(abi_version=_lib.ABI_VERSION, device=int(device), n_envs=int(n_envs), env_kind=int(env_kind),
                     local_map_length=int(local_map_length), auto_reset=int(bool(auto_reset)),
                     lanes_per_env=int(lanes_per_env), env_id0=int(env_id0) & 0xFFFFFFFF,
                     seed=int(seed) & 0xFFFFFFFFFFFFFFFF, crash_penalty=float(crash_penalty),
                     cell_size=float(cell_size))
        torch.cuda.init()
        with torch.cuda.device(self.device):
            torch.zeros(1, device=self.device)          # make sure the primary context exists
            check(self._lib.nav3d_create(C.byref(cfg), C.byref(self._h)))
        self.n_envs = int(n_envs)
        self.local_map_length = int(local_map_length)
        self.crash_penalty = float(crash_penalty)
        self.auto_reset = bool(auto_reset)
        self.seed = int(seed)
        self.env_id0 = int(env_id0)
        self.env_kind = int(env_kind)
        self.obs_dim = int(self._lib.nav3d_obs_dim(self._h))
        self.pick_cols = 3 if self.env_kind == _lib.ENV_SIMPLE else 2      # simpleEnv also draws a goal cell
        self.rooms: list = []
        self._step_args: dict = {}
        self.load_rooms(rooms)

    # ---- rooms -------------------------------------------------------------------------------------------------
    def load_rooms(self, rooms: Sequence[Room]):
        rooms = list(rooms)
        if not rooms:
            raise ValueError("at least one room is required")
        descs = (RoomDesc * len(rooms))()
        keep = []
        for i, r in enumerate(rooms):
            g = np.ascontiguousarray(r.grid, dtype=np.int8)
            keep.append(g)
            w, d, h = g.shape
            st = getattr(r, "start", None)
            descs[i] = RoomDesc(width=w, depth=d, height=h, wall_code=int(r.wall_code), grid=g.ctypes.data,
                                has_start=int(st is not None), start_x=int(st[0]) if st else 0,
                                start_y=int(st[1]) if st else 0, start_z=int(st[2]) if st else 0)
        check(self._lib.nav3d_load_rooms(self._h, len(rooms), descs))
        self.rooms = rooms
        info = (C.c_int32 * 6)()
        self.room_dims, self.room_free, self.room_walls = [], [], []
        for i in range(len(rooms)):
            check(self._lib.nav3d_room_info(self._h, i, info))
            self.room_dims.append((info[0], info[1], info[2]))
            self.room_free.append(int(info[3]))
            self.room_walls.append(int(info[4]))

    def set_reward_params(self, **kwargs):
        """Override literals of ``compute_reward`` (reference ``envs/CubicEnv.py:169-224``); names are the fields of
        ``nav3d_reward_params``.  Unnamed ones keep their current reference default."""
        p = _lib.RewardParams()
        self._lib.nav3d_reward_params_default(C.byref(p))
        p.crash_penalty = self.crash_penalty
        for k, v in kwargs.items():
            if not hasattr(p, k):
                raise TypeError(f"unknown reward parameter {k!r}")
            setattr(p, k, float(v))
        check(self._lib.nav3d_set_reward_params(self._h, C.byref(p)))
        self.crash_penalty = float(p.crash_penalty)

    def free_cell(self, room: int, k: int):
        xyz = (C.c_int32 * 3)()
        check(self._lib.nav3d_room_free_cell(self._h, int(room), int(k), xyz))
        return int(xyz[0]), int(xyz[1]), int(xyz[2])

    # ---- reset / step ------------------------------------------------------------------------------------------
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def new_obs(self) -> torch.Tensor:
        return torch.empty((self.n_envs, self.obs_dim), dtype=torch.float32, device=self.device)

    def reset(self, obs: Optional[torch.Tensor] = None, env_ids: Optional[torch.Tensor] = None,
              picks: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Reset all envs (``env_ids=None``) or the listed ones.  ``picks``: int32 [n,2] (room, k-th free cell) — [n,3] with
        the goal's free-cell index for simpleEnv — or None for Philox picks.  Returns the [n_envs, obs_dim] observation tensor (only the reset rows are rewritten)."""
        if obs is None:
            obs = self.new_obs()
        self._check(obs, torch.float32, (self.n_envs, self.obs_dim), "obs")
        if env_ids is not None:
            env_ids = env_ids.to(device=self.device, dtype=torch.int32).contiguous()
            n = env_ids.numel()
        else:
            n = self.n_envs
        if picks is not None:
            picks = picks.to(device=self.device, dtype=torch.int32).contiguous()
            if tuple(picks.shape) != (n, self.pick_cols):
                raise ValueError(f"picks must have shape ({n}, {self.pick_cols})")
        with torch.cuda.device(self.device):
            check(self._lib.nav3d_reset(self._h, _ptr(env_ids), n, _ptr(picks), _ptr(obs), self._stream()))
        return obs

    def step(self, actions: torch.Tensor, obs: torch.Tensor, reward: torch.Tensor, terminated: torch.Tensor,
             truncated: torch.Tensor, *, reward64: Optional[torch.Tensor] = None,
             terminal_obs: Optional[torch.Tensor] = None, episodes: Optional[torch.Tensor] = None):
        """One ``step`` of every env, asynchronous on the current CUDA stream; all tensors live on the engine's device.

        Argument validation is memoised on (address, shape, dtype, contiguity) of every buffer, so a rollout loop that cycles
        through the same buffers pays for the checks once (the call is then ~2x cheaper on the host, which is what bounds
        small batches).  The library makes the engine's device current itself and restores the caller's."""
        tensors = (actions, obs, reward, reward64, terminated, truncated, terminal_obs, episodes)
        key = tuple(None if t is None else (t.data_ptr(), t.shape, t.dtype, t.is_contiguous()) for t in tensors)
        args = self._step_args.get(key)
        if args is None:
            N = self.n_envs
            self._check(actions, torch.int64, (N,), "actions")
            self._check(obs, torch.float32, (N, self.obs_dim), "obs")
            self._check(reward, torch.float32, (N,), "reward")
            self._check(terminated, torch.uint8, (N,), "terminated")
            self._check(truncated, torch.uint8, (N,), "truncated")
            if reward64 is not None:
                self._check(reward64, torch.float64, (N,), "reward64")
            if terminal_obs is not None:
                self._check(terminal_obs, torch.float32, (N, self.obs_dim), "terminal_obs")
            if episodes is not None:
                self._check(episodes, torch.int32, (N, 8), "episodes")
            args = tuple(_ptr(t) for t in tensors)
            if len(self._step_args) >= 16384:        # (a rollout with one action row per step cycles through thousands of keys)
                self._step_args.clear()
            self._step_args[key] = args
        check(self._lib.nav3d_step(self._h, *args, self._stream()))

    def step_host(self, actions: torch.Tensor, obs: torch.Tensor, reward: torch.Tensor, terminated: torch.Tensor,
                  truncated: torch.Tensor):
        """The same step through HOST (ideally pinned) buffers; copies in, steps, copies out, waits."""
        for t, name in ((actions, "actions"), (obs, "obs"), (reward, "reward"), (terminated, "terminated"),
                        (truncated, "truncated")):
            if t.is_cuda or not t.is_contiguous():
                raise ValueError(f"{name} must be a contiguous CPU tensor")
        check(self._lib.nav3d_step_host(self._h, _ptr(actions), _ptr(obs), _ptr(reward), _ptr(terminated),
                                        _ptr(truncated)))

    def rollout_random(self, T: int, t0: int = 0, *, obs: Optional[torch.Tensor] = None,
                       obs_last: Optional[torch.Tensor] = None, reward: Optional[torch.Tensor] = None,
                       done: Optional[torch.Tensor] = None, actions_out: Optional[torch.Tensor] = None):
        N = self.n_envs
        if obs is not None:
            self._check(obs, torch.float32, (T, N, self.obs_dim), "obs")
        if obs_last is not None:
            self._check(obs_last, torch.float32, (N, self.obs_dim), "obs_last")
        if reward is not None:
            self._check(reward, torch.float32, (T, N), "reward")
        if done is not None:
            self._check(done, torch.uint8, (T, N), "done")
        if actions_out is not None:
            self._check(actions_out, torch.uint8, (T, N), "actions_out")
        with torch.cuda.device(self.device):
            check(self._lib.nav3d_rollout_random(self._h, int(T), int(t0) & 0xFFFFFFFF, _ptr(obs), _ptr(obs_last),
                                                 _ptr(reward), _ptr(done), _ptr(actions_out), self._stream()))

    def rollout_actions(self, actions: torch.Tensor, *, obs: Optional[torch.Tensor] = None,
                        obs_last: Optional[torch.Tensor] = None, reward: Optional[torch.Tensor] = None,
                        reward64: Optional[torch.Tensor] = None, terminated: Optional[torch.Tensor] = None,
                        truncated: Optional[torch.Tensor] = None, terminal_obs: Optional[torch.Tensor] = None,
                        episodes: Optional[torch.Tensor] = None):
        """T steps of every env with the rows of ``actions`` [T, n_envs] in one fused launch (``nav3d_rollout_actions``):
        every output and the final engine state equal those of T ``step`` calls with the same rows.

        ``actions``: uint8 on the engine's device is passed as it is (``rollout_random``'s ``actions_out`` replays as it
        is); any other integer dtype is clamped to 0..5 and cast, which is what ``step`` does to int64.  The outputs are
        ``step``'s with a leading T axis, all optional; ``obs_last`` [n_envs, obs_dim] receives the last step's rows when
        ``obs`` is None, and one of the two is required.  Rows of ``terminal_obs`` and ``episodes`` are written only where
        an episode ended.  Asynchronous on the current stream; with uint8 actions it allocates nothing and can be captured
        in a CUDA graph."""
        if (not isinstance(actions, torch.Tensor) or actions.dim() != 2 or actions.dtype.is_floating_point
                or actions.dtype.is_complex or actions.dtype == torch.bool):
            raise ValueError(f"actions must be a 2-D integer tensor [T, {self.n_envs}], got "
                             f"{getattr(actions, 'dtype', type(actions))} {tuple(getattr(actions, 'shape', ()))}")
        T, N = int(actions.shape[0]), self.n_envs
        if actions.dtype != torch.uint8:
            actions = actions.to(self.device).clamp(0, 5).to(torch.uint8).contiguous()
        self._check(actions, torch.uint8, (T, N), "actions")
        for t, dtype, shape, name in ((obs, torch.float32, (T, N, self.obs_dim), "obs"),
                                      (obs_last, torch.float32, (N, self.obs_dim), "obs_last"),
                                      (reward, torch.float32, (T, N), "reward"),
                                      (reward64, torch.float64, (T, N), "reward64"),
                                      (terminated, torch.uint8, (T, N), "terminated"),
                                      (truncated, torch.uint8, (T, N), "truncated"),
                                      (terminal_obs, torch.float32, (T, N, self.obs_dim), "terminal_obs"),
                                      (episodes, torch.int32, (T, N, 8), "episodes")):
            if t is not None:
                self._check(t, dtype, shape, name)
        if obs is None and obs_last is None:
            raise ValueError("one of obs / obs_last is required")
        if T == 0:                     # (the buffers of an empty rollout have no storage to pass)
            return
        with torch.cuda.device(self.device):
            check(self._lib.nav3d_rollout_actions(self._h, T, _ptr(actions), _ptr(obs), _ptr(obs_last), _ptr(reward),
                                                  _ptr(reward64), _ptr(terminated), _ptr(truncated), _ptr(terminal_obs),
                                                  _ptr(episodes), self._stream()))

    # ---- state -------------------------------------------------------------------------------------------------
    def get_state(self) -> torch.Tensor:
        """int32 [n_envs, 16]; columns are ``STATE_FIELDS``."""
        out = torch.empty((self.n_envs, _lib.STATE_INTS), dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            check(self._lib.nav3d_get_state(self._h, _ptr(out), self._stream()))
        return out

    def get_grid(self, env: int) -> np.ndarray:
        """The reference's ``internal_grid`` of one env, int16 [W, D, H] (visit counters saturate at 255)."""
        st = self.get_state()[env].cpu().numpy()
        w, d, h = self.room_dims[int(st[13])]
        out = torch.empty((w, d, h), dtype=torch.int16, device=self.device)
        with torch.cuda.device(self.device):
            check(self._lib.nav3d_get_grid(self._h, int(env), _ptr(out), self._stream()))
        return out.cpu().numpy()

    def snapshot(self) -> np.ndarray:
        n = self._lib.nav3d_snapshot_bytes(self._h)
        buf = np.empty(n, dtype=np.uint8)
        check(self._lib.nav3d_snapshot(self._h, C.c_void_p(buf.ctypes.data), n))
        return buf

    def restore(self, buf: np.ndarray):
        buf = np.ascontiguousarray(buf, dtype=np.uint8)
        check(self._lib.nav3d_restore(self._h, C.c_void_p(buf.ctypes.data), buf.size))

    # ---- env-state blobs ---------------------------------------------------------------------------------------------
    @property
    def env_state_bytes(self) -> int:
        """Bytes of one env-state blob (``nav3d_env_state_bytes``)."""
        return int(self._lib.nav3d_env_state_bytes(self._h))

    def _env_ids(self, env_ids) -> torch.Tensor:
        """A list, range, numpy array, CPU or device tensor of env ids -> contiguous int32 [n] on the engine's device.  Ids
        that do not fit int32 become -1 (out of range) instead of wrapping onto a valid env."""
        t = env_ids if isinstance(env_ids, torch.Tensor) else torch.as_tensor(np.asarray(env_ids, dtype=np.int64))
        if t.dim() != 1 or t.dtype.is_floating_point or t.dtype.is_complex or t.dtype == torch.bool:
            raise ValueError(f"env_ids must be a 1-D integer sequence or tensor, got {t.dtype} {tuple(t.shape)}")
        if t.dtype != torch.int32:
            t = torch.where((t < 0) | (t >= self.n_envs), torch.full_like(t, -1), t)
        return t.to(device=self.device, dtype=torch.int32).contiguous()

    def save_envs(self, env_ids, obs: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """The complete state of the listed envs as uint8 [n, env_state_bytes] blobs on the engine's device.

        ``obs`` is the observation array the last step / reset / load wrote: a blob carries its env's current row, which
        cannot be recomputed from the env's record.  Asynchronous on the current stream; with a device tensor of ids and an
        ``out`` buffer it can be captured in a CUDA graph.  An out-of-range id yields a blob every load rejects."""
        ids = self._env_ids(env_ids)
        n, B = ids.numel(), self.env_state_bytes
        self._check(obs, torch.float32, (self.n_envs, self.obs_dim), "obs")
        if out is None:
            out = torch.empty((n, B), dtype=torch.uint8, device=self.device)
        self._check(out, torch.uint8, (n, B), "out")
        with torch.cuda.device(self.device):
            check(self._lib.nav3d_save_envs(self._h, _ptr(ids), n, _ptr(obs), _ptr(out), self._stream()))
        return out

    def load_envs(self, env_ids, states: torch.Tensor, obs: torch.Tensor, *, check: bool = True) -> torch.Tensor:
        """Overwrite the listed envs with ``states[i]`` (blobs from ``save_envs`` of this or an equally configured engine)
        and write their observation rows into ``obs``, which is returned.  Cloning env ``a`` into envs ``dst``::

            engine.load_envs(dst, engine.save_envs([a], obs)[[0] * len(dst)], obs)

        ``check=True``: the ids must be in range and distinct (a ``Nav3dError`` otherwise, before anything is written), and
        the per-blob status is read back after the launch (one synchronisation; device-tensor ids cost one more); a blob this
        engine cannot load leaves its env untouched and raises a ``Nav3dError`` naming every bad entry.
        ``check=False``: nothing synchronises (for use inside a captured CUDA graph); the ids must be distinct, and rejected
        blobs leave their envs untouched silently."""
        ids = self._env_ids(env_ids)
        n, B = ids.numel(), self.env_state_bytes
        self._check(states, torch.uint8, (n, B), "states")
        self._check(obs, torch.float32, (self.n_envs, self.obs_dim), "obs")
        status = None
        if check:
            h = ids.cpu().numpy()
            bad = np.nonzero((h < 0) | (h >= self.n_envs))[0]
            if len(bad):
                raise Nav3dError(-1, f"load_envs: env ids out of range 0..{self.n_envs - 1} at entries "
                                     f"{bad[:16].tolist()} (ids {h[bad[:16]].tolist()})")
            uniq, counts = np.unique(h, return_counts=True)
            if (counts > 1).any():
                raise Nav3dError(-1, f"load_envs: env ids must be distinct; repeated: {uniq[counts > 1][:16].tolist()}")
            status = torch.empty(n, dtype=torch.uint8, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self._lib.nav3d_load_envs(self._h, _ptr(ids), n, _ptr(states), _ptr(obs), _ptr(status),
                                                 self._stream()))
        if check and n:
            st = status.cpu().numpy()
            bad = np.nonzero(st != _lib.ENV_STATE_LOADED)[0]
            if len(bad):
                raise Nav3dError(-1, f"load_envs: {len(bad)} of {n} blobs were not loaded (their envs are unchanged): "
                                     + ", ".join(f"entry {i} -> env {int(h[i])}: "
                                                 + ("env id out of range" if st[i] == _lib.ENV_STATE_BAD_ENV else
                                                    "not a valid blob for this engine") for i in bad[:16]))
        return obs

    @property
    def launch_count(self) -> int:
        return int(self._lib.nav3d_launch_count(self._h))

    @property
    def device_bytes(self) -> int:
        return int(self._lib.nav3d_device_bytes(self._h))

    @property
    def lanes_per_env(self) -> int:
        return int(self._lib.nav3d_lanes_per_env(self._h))

    # ---- plumbing ----------------------------------------------------------------------------------------------
    def _check(self, t: torch.Tensor, dtype, shape, name: str):
        if not isinstance(t, torch.Tensor) or t.dtype != dtype or tuple(t.shape) != tuple(shape):
            raise ValueError(f"{name} must be a {dtype} tensor of shape {tuple(shape)}, got "
                             f"{getattr(t, 'dtype', type(t))} {tuple(getattr(t, 'shape', ()))}")
        if t.device != self.device:
            raise ValueError(f"{name} must live on {self.device}, got {t.device}")
        if not t.is_contiguous():
            raise ValueError(f"{name} must be contiguous")

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.nav3d_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):  # noqa: D401
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass

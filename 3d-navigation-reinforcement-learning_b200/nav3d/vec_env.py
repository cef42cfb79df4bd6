"""``BatchedCubicEnv`` — the GPU-resident replacement for ``SubprocVecEnv([make_env_fn(...)] * n)``
(reference ``train/Grid_Train.py:118-126``, ``:170-173``, ``:191-192``; ``train/Train_Further.py:133-141``).

It follows stable-baselines3's ``VecEnv`` contract (third-party, un-vendored by the reference):
``reset() -> obs``, ``step_async(actions)`` / ``step_wait() -> (obs, rewards, dones, infos)``, auto-reset on done with the
pre-reset observation kept as ``terminal_observation`` and ``TimeLimit.truncated = truncated and not terminated``;
``Monitor``'s per-episode ``{"r", "l"}`` record is produced on the device.

The native fast path returns torch CUDA tensors (no host round-trip); ``infos`` is a ``StepInfo`` holding tensors.
``StepInfo.to_dicts()`` renders the SB3 list-of-dicts form (one device->host copy) for code that wants it."""
from __future__ import annotations

import time
from dataclasses import dataclass
from typing import List, Optional, Sequence

import numpy as np
import torch

from .engine import Engine
from .rooms import Room, default_box_room, load_room_dir
from .spaces import cubic_spaces


@dataclass
class StepInfo:
    terminated: torch.Tensor            # uint8 [N]
    truncated: torch.Tensor             # uint8 [N]
    terminal_observation: torch.Tensor  # f32 [N, 80]; rows valid where done
    episodes: torch.Tensor              # int32 [N, 8] view of nav3d_episode; rows valid where done

    def __getitem__(self, t) -> "StepInfo":
        """Step t of the per-step tensors ``BatchedCubicEnv.step_sequence`` returns (they carry a leading T axis)."""
        return StepInfo(self.terminated[t], self.truncated[t], self.terminal_observation[t], self.episodes[t])

    def to_dicts(self, t_start: Optional[float] = None) -> List[dict]:
        term = self.terminated.cpu().numpy().astype(bool)
        trunc = self.truncated.cpu().numpy().astype(bool)
        done = term | trunc
        infos: List[dict] = [{} for _ in range(term.shape[0])]
        if done.any():
            idx = np.nonzero(done)[0]
            tobs = self.terminal_observation[torch.as_tensor(idx, device=self.terminal_observation.device)].cpu().numpy()
            eps = self.episodes.cpu().numpy()
            ret = eps[:, 0].view(np.float32)
            now = time.time()
            for j, i in enumerate(idx):
                infos[i]["terminal_observation"] = tobs[j]
                infos[i]["TimeLimit.truncated"] = bool(trunc[i] and not term[i])
                infos[i]["episode"] = {"r": round(float(ret[i]), 6), "l": int(eps[i, 1]),
                                       "t": round(now - t_start, 6) if t_start else 0.0}
                infos[i]["bumps"] = int(eps[i, 2])
                infos[i]["visited"] = int(eps[i, 3])
                infos[i]["total_free"] = int(eps[i, 4])
        return infos


class BatchedCubicEnv:
    """N CubicEnv ``GridAgent`` instances stepped by one CUDA kernel launch.

    Parameters mirror ``GridAgent.__init__`` (``envs/CubicEnv.py:17-29``) where they affect dynamics.  ``rooms`` (a list
    of ``Room``) overrides ``room_path``; with neither, the reference's default 20x20x12 hollow box is used."""

    def __init__(self, room_path=None, num_envs: int = 8, local_map_length: int = 4, crash_penalty: float = -2.0,
                 *, rooms: Optional[Sequence[Room]] = None, seed: int = 0, device: int = 0, auto_reset: bool = True,
                 env_id0: int = 0, lanes_per_env: int = 0, sort_rooms: bool = False,
                 width: int = 20, depth: int = 20, height: int = 12):
        if rooms is None:
            rooms = load_room_dir(room_path, sort=sort_rooms) if room_path is not None else [default_box_room(width, depth, height)]
        self.engine = Engine(num_envs, rooms, local_map_length=local_map_length, crash_penalty=crash_penalty,
                             auto_reset=auto_reset, seed=seed, env_id0=env_id0, device=device,
                             lanes_per_env=lanes_per_env)
        self.num_envs = int(num_envs)
        self.device = self.engine.device
        self.action_space, self.observation_space = cubic_spaces()
        self.local_map_length = int(local_map_length)
        self.crash_penalty = float(crash_penalty)
        self.render_mode = None
        N, dev = self.num_envs, self.device
        self._obs = torch.zeros((N, 80), dtype=torch.float32, device=dev)
        self._reward = torch.zeros(N, dtype=torch.float32, device=dev)
        self._term = torch.zeros(N, dtype=torch.uint8, device=dev)
        self._trunc = torch.zeros(N, dtype=torch.uint8, device=dev)
        self._tobs = torch.zeros((N, 80), dtype=torch.float32, device=dev)
        self._eps = torch.zeros((N, 8), dtype=torch.int32, device=dev)
        self._pending: Optional[torch.Tensor] = None
        self._t_start = time.time()

    # ---- VecEnv API --------------------------------------------------------------------------------------------
    def reset(self, picks: Optional[torch.Tensor] = None) -> torch.Tensor:
        self.engine.reset(self._obs, picks=picks)
        return self._obs

    def step_async(self, actions) -> None:
        a = torch.as_tensor(actions)
        self._pending = a.to(device=self.device, dtype=torch.int64, non_blocking=True).contiguous()

    def step_wait(self, out_obs: Optional[torch.Tensor] = None):
        if self._pending is None:
            raise RuntimeError("step_wait() called without step_async()")
        obs = self._obs if out_obs is None else out_obs
        self.engine.step(self._pending, obs, self._reward, self._term, self._trunc,
                         terminal_obs=self._tobs, episodes=self._eps)
        self._pending = None
        dones = (self._term | self._trunc).bool()
        return obs, self._reward, dones, StepInfo(self._term, self._trunc, self._tobs, self._eps)

    def step(self, actions, out_obs: Optional[torch.Tensor] = None):
        self.step_async(actions)
        return self.step_wait(out_obs)

    def seed(self, seed: Optional[int] = None):
        return [None] * self.num_envs

    def step_sequence(self, actions):
        """T calls of ``step()`` with the rows of ``actions`` [T, num_envs] in one fused launch (``Engine.rollout_actions``).

        Returns ``obs`` [T, N, 80], ``rewards`` [T, N], ``dones`` [T, N] (bool) and a ``StepInfo`` whose tensors carry the
        same leading T axis; ``info[t]`` is step t's (``sb3_infos(info[t])`` renders it).  Rows of terminal_observation and
        episodes are valid where ``dones``.  The env's own observation buffer is left equal to ``obs[-1]``, so ``step()``,
        ``save_envs()`` and ``step_sequence()`` continue from there."""
        a = torch.as_tensor(actions)
        if a.dim() != 2 or a.shape[1] != self.num_envs:
            raise ValueError(f"actions must have shape (T, {self.num_envs}), got {tuple(a.shape)}")
        a = a.to(self.device)
        T, N, dev = int(a.shape[0]), self.num_envs, self.device
        obs = torch.empty((T, N, 80), dtype=torch.float32, device=dev)
        rewards = torch.empty((T, N), dtype=torch.float32, device=dev)
        term = torch.empty((T, N), dtype=torch.uint8, device=dev)
        trunc = torch.empty((T, N), dtype=torch.uint8, device=dev)
        tobs = torch.zeros((T, N, 80), dtype=torch.float32, device=dev)
        eps = torch.zeros((T, N, 8), dtype=torch.int32, device=dev)
        self.engine.rollout_actions(a, obs=obs, reward=rewards, terminated=term, truncated=trunc, terminal_obs=tobs,
                                    episodes=eps)
        if T:
            self._obs.copy_(obs[-1])
        return obs, rewards, (term | trunc).bool(), StepInfo(term, trunc, tobs, eps)

    def close(self) -> None:
        self.engine.close()

    def get_attr(self, attr_name: str, indices=None):
        cols = {"x": 0, "y": 1, "z": 2, "facing": 3, "visited_count": 4, "bump_count": 5, "step_count": 6,
                "near_wall": 7, "was_near_wall": 8, "last_bump": 9, "done": 10, "cells_insight_down": 11,
                "last_action": 12}
        idx = list(range(self.num_envs)) if indices is None else list(np.atleast_1d(indices))
        if attr_name in cols:
            st = self.engine.get_state()[:, cols[attr_name]].cpu().numpy()
            return [int(st[i]) for i in idx]
        if attr_name in ("total_free_cells", "max_steps"):
            rooms = self.engine.get_state()[:, 13].cpu().numpy()
            return [self.engine.room_free[int(rooms[i])] for i in idx]
        if attr_name in ("local_map_length", "crash_penalty", "render_mode", "action_space", "observation_space"):
            return [getattr(self, attr_name)] * len(idx)
        raise AttributeError(attr_name)

    def set_attr(self, attr_name, value, indices=None):
        raise NotImplementedError("per-env attributes live on the GPU; rebuild the env to change them")

    def env_method(self, method_name, *args, indices=None, **kwargs):
        if method_name == "get_position":
            st = self.engine.get_state()[:, :3].cpu().numpy()
            idx = list(range(self.num_envs)) if indices is None else list(np.atleast_1d(indices))
            return [tuple(int(v) for v in st[i]) for i in idx]
        raise NotImplementedError(method_name)

    def env_is_wrapped(self, wrapper_class, indices=None):
        n = self.num_envs if indices is None else len(np.atleast_1d(indices))
        return [False] * n

    # ---- extras ------------------------------------------------------------------------------------------------
    def state(self) -> torch.Tensor:
        return self.engine.get_state()

    def save_envs(self, indices, obs: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Complete state of the listed envs as uint8 [n, engine.env_state_bytes] device blobs (``Engine.save_envs``).
        ``obs`` is the current observation array: this env's own buffer by default; pass the tensor the last
        ``step_wait(out_obs=...)`` wrote when it was elsewhere."""
        return self.engine.save_envs(indices, self._obs if obs is None else obs)

    def load_envs(self, indices, states: torch.Tensor, obs: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Overwrite the listed envs with blobs from ``save_envs`` and write their observation rows into ``obs`` (this env's
        own buffer by default), which is returned.  Raises ``Nav3dError`` for bad ids or blobs (``Engine.load_envs``)."""
        return self.engine.load_envs(indices, states, self._obs if obs is None else obs)

    def sb3_infos(self, info: StepInfo) -> List[dict]:
        return info.to_dicts(self._t_start)


class NumpyVecEnv:
    """The numpy face of a batched env, for host-side trainers written against stable-baselines3's ``VecEnv``
    (``reset() -> np.ndarray``, ``step_async`` / ``step_wait() -> (obs, rewards, dones, infos)`` with SB3's list-of-dicts
    ``infos``: ``terminal_observation``, ``TimeLimit.truncated`` and Monitor's ``episode`` record).  It wraps
    ``BatchedCubicEnv`` (or anything with its interface) and costs one device->host copy per step — the contract of the
    reference's ``SubprocVecEnv`` (``train/Grid_Train.py:170-173``), not the fast path."""

    def __init__(self, env):
        self.env = env
        self.num_envs = env.num_envs
        self.action_space, self.observation_space = env.action_space, env.observation_space
        self.render_mode = None
        self._t_start = time.time()
        self._actions = None

    def reset(self):
        return self.env.reset().detach().cpu().numpy().copy()

    def step_async(self, actions) -> None:
        self._actions = np.asarray(actions, dtype=np.int64)

    def step_wait(self):
        if self._actions is None:
            raise RuntimeError("step_wait() called without step_async()")
        obs, rewards, dones, info = self.env.step(torch.as_tensor(self._actions))
        self._actions = None
        return (obs.detach().cpu().numpy().copy(), rewards.detach().cpu().numpy().astype(np.float32),
                dones.detach().cpu().numpy().astype(bool), StepInfo.to_dicts(info, self._t_start))

    def step(self, actions):
        self.step_async(actions)
        return self.step_wait()

    def close(self) -> None:
        self.env.close()

    def seed(self, seed=None):
        return [None] * self.num_envs

    def get_attr(self, attr_name, indices=None):
        return self.env.get_attr(attr_name, indices)

    def env_method(self, method_name, *args, indices=None, **kwargs):
        return self.env.env_method(method_name, *args, indices=indices, **kwargs)

    def env_is_wrapped(self, wrapper_class, indices=None):
        n = self.num_envs if indices is None else len(np.atleast_1d(indices))
        return [False] * n


class BatchedSimpleEnv:
    """N ``envs/simpleEnv.py::GridAgent`` instances on the GPU (the reference's older env variant; no driver imports it).

    ``reset()`` is the reference's ``reset()`` followed by one ``get_obs()`` (the reference's own ``reset`` returns
    ``None``, ``simpleEnv.py:79-107``).  Observations are ``6*L+7`` floats (``:233-265``)."""

    def __init__(self, room_path=None, num_envs: int = 8, local_map_length: int = 4, *, rooms=None, seed: int = 0,
                 device: int = 0, auto_reset: bool = True, env_id0: int = 0, lanes_per_env: int = 0,
                 cell_size: float = 0.25, sort_rooms: bool = False, width: int = 20, depth: int = 20, height: int = 12):
        from . import _lib
        from .spaces import simple_spaces
        if rooms is None:
            rooms = (load_room_dir(room_path, simple=True, sort=sort_rooms) if room_path is not None
                     else [default_box_room(width, depth, height, simple=True)])
        self.engine = Engine(num_envs, rooms, local_map_length=local_map_length, auto_reset=auto_reset, seed=seed,
                             env_id0=env_id0, device=device, lanes_per_env=lanes_per_env, env_kind=_lib.ENV_SIMPLE,
                             cell_size=cell_size)
        self.num_envs, self.device = int(num_envs), self.engine.device
        self.action_space, self.observation_space = simple_spaces(local_map_length)
        N, dev, d = self.num_envs, self.device, self.engine.obs_dim
        self._obs = torch.zeros((N, d), dtype=torch.float32, device=dev)
        self._reward = torch.zeros(N, dtype=torch.float32, device=dev)
        self._term = torch.zeros(N, dtype=torch.uint8, device=dev)
        self._trunc = torch.zeros(N, dtype=torch.uint8, device=dev)
        self._tobs = torch.zeros((N, d), dtype=torch.float32, device=dev)
        self._eps = torch.zeros((N, 8), dtype=torch.int32, device=dev)
        self._pending = None

    def reset(self, picks=None):
        self.engine.reset(self._obs, picks=picks)
        return self._obs

    def step_async(self, actions):
        self._pending = torch.as_tensor(actions).to(device=self.device, dtype=torch.int64).contiguous()

    def step_wait(self):
        self.engine.step(self._pending, self._obs, self._reward, self._term, self._trunc, terminal_obs=self._tobs,
                         episodes=self._eps)
        self._pending = None
        return self._obs, self._reward, (self._term | self._trunc).bool(), StepInfo(self._term, self._trunc, self._tobs, self._eps)

    def step(self, actions):
        self.step_async(actions)
        return self.step_wait()

    def save_envs(self, indices, obs: Optional[torch.Tensor] = None) -> torch.Tensor:
        """As ``BatchedCubicEnv.save_envs``."""
        return self.engine.save_envs(indices, self._obs if obs is None else obs)

    def load_envs(self, indices, states: torch.Tensor, obs: Optional[torch.Tensor] = None) -> torch.Tensor:
        """As ``BatchedCubicEnv.load_envs``."""
        return self.engine.load_envs(indices, states, self._obs if obs is None else obs)

    def close(self):
        self.engine.close()

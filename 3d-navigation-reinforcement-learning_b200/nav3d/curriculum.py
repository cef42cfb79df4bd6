"""``RoomCurriculum``: a learning-progress curriculum over an env's rooms, kept on the device.

Each rollout, ``observe`` adds the finished episodes of every env step to a per-room window (``Engine.room_stats``, one
kernel launch, no synchronisation, capturable in a CUDA graph).  ``update`` turns the window into room weights and installs
them with ``set_room_weights(check=False)``, so the next resets draw rooms from them.  The rule (``lp_rule``):

* the score of room j is its mean explored fraction over the window, ``m_j = visited_sum_j / (n_j * total_free_j)``: it
  rises with learning long before an episode reaches the 84 % that terminates it;
* a fast and a slow exponential moving average follow the score, ``f_j += alpha_fast (m_j - f_j)``,
  ``s_j += alpha_slow (m_j - s_j)``, both set to ``m_j`` at a room's first observation; rooms without a finished episode in
  the window keep their state;
* learning progress ``LP_j = |f_j - s_j|`` (Matiisen et al. 2017, teacher-student curriculum learning; Kanitscheider et al.
  2021); a room never observed gets the largest LP of the observed rooms when that is positive, else 1;
* ``p_j = uniform_mix / R + (1 - uniform_mix) LP_j / sum(LP)`` when ``sum(LP) > 0``, else ``1 / R``.

A room whose score has stopped changing (solved, or one the policy cannot solve yet: its episodes still end by truncation)
gets exactly ``uniform_mix / R`` of the draw while another room is still progressing.

Data parallel: with ``torch.distributed`` initialised and world > 1, ``update`` sums the int64 windows of all ranks with one
all-reduce before applying the rule, so every rank installs bit-identical weights and engines draw the same rooms for the
same global env ids (DESIGN.md section 7)."""
from __future__ import annotations

from typing import Dict, Tuple

import torch

from .engine import ROOM_STAT_FIELDS

EPISODES, VISITED = ROOM_STAT_FIELDS.index("episodes"), ROOM_STAT_FIELDS.index("visited_sum")


def lp_rule(window: torch.Tensor, total_free: torch.Tensor, fast: torch.Tensor, slow: torch.Tensor, seen: torch.Tensor,
            alpha_fast: float, alpha_slow: float, uniform_mix: float
            ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    """One application of the rule, in float64 on the tensors' device, without a host synchronisation.

    ``window``: int64 [R, 8] stats (``ROOM_STAT_FIELDS``); ``total_free``: float64 [R]; ``fast``, ``slow``: float64 [R];
    ``seen``: bool [R].  Returns the new ``(fast, slow, seen, lp, p)``; ``lp`` is NaN-free and holds the value used for
    every room (the stand-in for rooms never observed)."""
    n = window[:, EPISODES].to(torch.float64)
    obs = n > 0
    m = window[:, VISITED].to(torch.float64) / (torch.where(obs, n, torch.ones_like(n)) * total_free)
    first = obs & ~seen
    fast = torch.where(first, m, torch.where(obs, fast + alpha_fast * (m - fast), fast))
    slow = torch.where(first, m, torch.where(obs, slow + alpha_slow * (m - slow), slow))
    seen = seen | obs
    lp = torch.where(seen, (fast - slow).abs(), torch.zeros_like(fast))
    best = lp.max()
    lp = torch.where(seen, lp, torch.where(best > 0, best, torch.ones_like(best)))
    R = lp.numel()
    total = lp.sum()
    p = torch.where(total > 0, uniform_mix / R + (1.0 - uniform_mix) * lp / torch.where(total > 0, total, torch.ones_like(total)),
                    torch.full_like(lp, 1.0 / R))
    return fast, slow, seen, lp, p


class RoomCurriculum:
    """Learning-progress room weights for one env (``BatchedCubicEnv``, ``BatchedSimpleEnv`` or an ``Engine``).

    Parameters:
      alpha_fast  -- step of the fast moving average of each room's score (default 0.1)
      alpha_slow  -- step of the slow moving average (default 0.02)
      uniform_mix -- share of the draw spread uniformly over all rooms, epsilon (default 0.2): every room keeps at least
                     ``uniform_mix / R`` of the draw

    ``RecurrentPPO(..., curriculum=cur)`` calls ``observe`` after every env step and ``update`` after every rollout."""

    def __init__(self, env, *, alpha_fast: float = 0.1, alpha_slow: float = 0.02, uniform_mix: float = 0.2):
        if not (0.0 < alpha_fast <= 1.0 and 0.0 < alpha_slow <= 1.0):
            raise ValueError("alpha_fast and alpha_slow must lie in (0, 1]")
        if not 0.0 <= uniform_mix <= 1.0:
            raise ValueError("uniform_mix must lie in [0, 1]")
        self.env = env
        self.engine = getattr(env, "engine", env)
        self.alpha_fast, self.alpha_slow, self.uniform_mix = float(alpha_fast), float(alpha_slow), float(uniform_mix)
        dev = self.engine.device
        R = len(self.engine.room_free)
        self.n_rooms = R
        self.total_free = torch.tensor([float(f) for f in self.engine.room_free], dtype=torch.float64, device=dev)
        self.window = torch.zeros((R, len(ROOM_STAT_FIELDS)), dtype=torch.int64, device=dev)
        self.fast = torch.zeros(R, dtype=torch.float64, device=dev)
        self.slow = torch.zeros(R, dtype=torch.float64, device=dev)
        self.seen = torch.zeros(R, dtype=torch.bool, device=dev)
        self.lp = torch.ones(R, dtype=torch.float64, device=dev)
        self.p = torch.full((R,), 1.0 / R, dtype=torch.float64, device=dev)
        self.weights = self.p.to(torch.float32)            # the vector last passed to set_room_weights
        self.summary = torch.tensor([float(R), 1.0 / R, 1.0 / R], dtype=torch.float64, device=dev)
        self.updates = 0
        self._dist = None
        try:
            import torch.distributed as dist
            if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
                self._dist = dist
        except Exception:  # noqa: BLE001
            self._dist = None

    def observe(self, terminated: torch.Tensor, truncated: torch.Tensor, episodes: torch.Tensor) -> None:
        """Add the finished episodes of one step ([N] flags, [N, 8] episodes) or of T steps ([T, N], [T, N, 8]) to the
        window: one ``room_stats`` launch on the current stream, nothing synchronised."""
        self.engine.room_stats(terminated, truncated, episodes, out=self.window)

    @torch.no_grad()
    def update(self) -> torch.Tensor:
        """Apply the rule to the window (summed over ranks), install the weights, zero the window.  Sync-free apart from
        the all-reduce; returns ``probabilities()``."""
        if self._dist is not None:
            self._dist.all_reduce(self.window)
        self.fast, self.slow, self.seen, self.lp, self.p = lp_rule(
            self.window, self.total_free, self.fast, self.slow, self.seen, self.alpha_fast, self.alpha_slow, self.uniform_mix)
        self.weights = self.p.to(torch.float32)
        self.engine.set_room_weights(self.weights, check=False)
        self.window.zero_()
        self._summarise()
        self.updates += 1
        return self.p

    def _summarise(self) -> None:
        """``summary`` = (effective number of rooms exp(H(p)), min p, max p), on the device."""
        h = -(self.p * torch.log(torch.where(self.p > 0, self.p, torch.ones_like(self.p)))).sum()
        self.summary = torch.stack([h.exp(), self.p.min(), self.p.max()])

    def probabilities(self) -> torch.Tensor:
        """float64 [R]: p of the last update (uniform before the first).  The engine draws from float32(p) through its
        table: ``env.room_probabilities()`` gives the exact probabilities installed."""
        return self.p

    def state_dict(self) -> Dict[str, object]:
        return dict(alpha_fast=self.alpha_fast, alpha_slow=self.alpha_slow, uniform_mix=self.uniform_mix,
                    updates=self.updates, window=self.window.cpu(), fast=self.fast.cpu(), slow=self.slow.cpu(),
                    seen=self.seen.cpu(), lp=self.lp.cpu(), p=self.p.cpu())

    def load_state_dict(self, sd: Dict[str, object]) -> None:
        """Restore a ``state_dict`` taken over the same rooms, and install its weights when it had made an update."""
        if tuple(sd["window"].shape) != tuple(self.window.shape):
            raise ValueError(f"curriculum state is for {sd['window'].shape[0]} rooms, this env has {self.n_rooms}")
        self.alpha_fast, self.alpha_slow = float(sd["alpha_fast"]), float(sd["alpha_slow"])
        self.uniform_mix, self.updates = float(sd["uniform_mix"]), int(sd["updates"])
        for k in ("window", "fast", "slow", "seen", "lp", "p"):
            getattr(self, k).copy_(sd[k])
        self.weights = self.p.to(torch.float32)
        if self.updates:
            self.engine.set_room_weights(self.weights, check=False)
        self._summarise()

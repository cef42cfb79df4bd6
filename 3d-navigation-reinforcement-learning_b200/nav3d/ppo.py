"""``RecurrentPPO`` — GPU-resident LSTM-PPO over ``BatchedCubicEnv`` (SURVEY §8f row 1).

Replaces, for the reference's training scripts, ``sb3_contrib.RecurrentPPO("MlpLstmPolicy", env, **ppo_hp)`` as built at
``train/Grid_Train.py:198-205`` with the hyper-parameters of ``:82-88`` (lr 3e-4, n_steps 2048, batch_size 64, gamma 0.99,
gae_lambda 0.95, ent_coef 0.01, vf_coef 0.5, clip_range 0.2, n_epochs 10) and driven by ``model.learn(total_timesteps,
reset_num_timesteps=False, callback=...)`` / ``model.save`` / ``RecurrentPPO.load`` (``:228-233``,
``train/Train_Further.py:146``, ``train/evaluate_grid.py:165``, ``:186-191`` ``model.predict``).  sb3-contrib is
third-party and un-vendored; what is restated here is its published algorithm:

* rollout: per step, policy forward with LSTM states zeroed at episode starts, categorical sample, env step; when an
  episode ends by time limit only (``truncated and not terminated``) the reward gets ``gamma * V(terminal_observation)``
  with the critic state after that step; buffers are time-major and live in HBM — the env kernel writes each step's
  observation straight into ``obs[t+1]`` of the rollout tensor (no host round trip anywhere in the loop);
* GAE(lambda) backward scan (``nav3d_gae``), returns = advantages + values;
* update: ``n_epochs`` passes over shuffled minibatches of fixed-length sequence chunks (truncated BPTT from the LSTM state
  recorded at the chunk's first step, SB3's behaviour for ``batch_size < n_steps``), clipped surrogate + ``vf_coef`` * MSE
  value loss + ``ent_coef`` * entropy bonus, per-minibatch advantage normalisation, Adam(eps 1e-5), grad-norm clip 0.5;
* data parallel: every rank owns an env shard and its own rollout; gradients are averaged with ONE NCCL all-reduce per
  minibatch over a flat gradient buffer (SURVEY §8e) — the only collective of the whole training loop.

What differs from SB3 on purpose: minibatches are built from whole sequence chunks of many envs (so a minibatch is a few
large GEMM calls), sampling uses the engine's Philox streams (results independent of the shard count), episode statistics
are reduced on the device, a rollout is replayed as CUDA graphs from the second one on, and minibatches small enough to be
launch-bound are replayed as one CUDA graph each (DESIGN.md §6b)."""
from __future__ import annotations

import io
import json
import math
import time
import zipfile
from pathlib import Path
from typing import Callable, Dict, List, Optional, Sequence

import numpy as np
import torch
import torch.nn.functional as F

from .policy import LSTMState, RecurrentActorCritic

FORMAT_VERSION = 1


def _append_zip_suffix(path) -> Path:
    p = Path(path)
    return p if p.suffix else p.with_suffix(".zip")           # SB3's save/load add ".zip" only when there is no suffix


class RecurrentPPO:
    def __init__(self, env, *, policy_kwargs: Optional[dict] = None, learning_rate: float = 3e-4, n_steps: int = 128,
                 batch_size: int = 128, n_epochs: int = 10, gamma: float = 0.99, gae_lambda: float = 0.95,
                 clip_range: float = 0.2, ent_coef: float = 0.0, vf_coef: float = 0.5, max_grad_norm: float = 0.5,
                 normalize_advantage: bool = True, seq_len: Optional[int] = None, seed: Optional[int] = 0,
                 verbose: int = 0, ops=None, device=None, policy: str = "MlpLstmPolicy", allow_tf32: bool = True,
                 cuda_graph: bool = True, graph_chunk: int = 128, graph_update_max: int = 8192, curriculum=None):
        if policy != "MlpLstmPolicy":
            raise ValueError("only MlpLstmPolicy is implemented (the one the reference trains)")
        self.policy_kwargs = dict(policy_kwargs or {})
        self.learning_rate, self.n_steps, self.batch_size, self.n_epochs = float(learning_rate), int(n_steps), int(batch_size), int(n_epochs)
        self.gamma, self.gae_lambda, self.clip_range = float(gamma), float(gae_lambda), float(clip_range)
        self.ent_coef, self.vf_coef, self.max_grad_norm = float(ent_coef), float(vf_coef), float(max_grad_norm)
        self.normalize_advantage = bool(normalize_advantage)
        self.seed, self.verbose = seed, int(verbose)
        self.cuda_graph, self.graph_chunk, self.graph_update_max = bool(cuda_graph), int(graph_chunk), int(graph_update_max)
        self.num_timesteps = 0
        self.n_updates = 0
        # nav3d.curriculum.RoomCurriculum or None: observes every env step, updates the room weights after every rollout
        self.curriculum = curriculum
        self._curriculum_log: Dict[str, float] = {}
        self._iteration = 0
        self.seq_len = int(seq_len) if seq_len else math.gcd(self.n_steps, self.batch_size)
        if self.n_steps % self.seq_len or self.batch_size % self.seq_len:
            raise ValueError(f"seq_len {self.seq_len} must divide n_steps {self.n_steps} and batch_size {self.batch_size}")
        self.env = None
        self.device = torch.device(device) if device is not None else (env.device if env is not None else torch.device("cpu"))
        if seed is not None:
            torch.manual_seed(int(seed))
        if allow_tf32 and self.device.type == "cuda":
            torch.backends.cuda.matmul.allow_tf32 = True
            torch.backends.cudnn.allow_tf32 = True
        self.policy = RecurrentActorCritic(**self.policy_kwargs).to(self.device)
        self._dist = None
        self.world, self.rank = 1, 0
        try:
            import torch.distributed as dist
            if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
                self._dist, self.world, self.rank = dist, dist.get_world_size(), dist.get_rank()
        except Exception:  # noqa: BLE001
            self._dist = None
        self._flatten_grads()
        if self._dist is not None:                                   # identical replicas: rank 0's initialisation wins
            for p in self.policy.parameters():
                self._dist.broadcast(p.data, src=0)
        # capturable: the step counter lives on the device, so an optimizer step can be part of a CUDA graph
        self.optimizer = torch.optim.Adam(self.policy.parameters(), lr=self.learning_rate, eps=1e-5,
                                          capturable=self.device.type == "cuda")
        self._ops = ops
        self._gen = torch.Generator(device=self.device)
        self._gen.manual_seed(int(seed or 0) + 7919)
        self.logger: List[Dict[str, float]] = []
        self._ep_return_mean = float("nan")
        self._ep_len_mean = float("nan")
        if env is not None:
            self.set_env(env)

    # ---- plumbing ----------------------------------------------------------------------------------------------
    def _flatten_grads(self):
        """All gradients live in one flat buffer: zeroing is one memset and the data-parallel average is one all-reduce."""
        params = [p for p in self.policy.parameters() if p.requires_grad]
        n = sum(p.numel() for p in params)
        self._flat_grad = torch.zeros(n, dtype=torch.float32, device=self.device)
        o = 0
        for p in params:
            p.grad = self._flat_grad[o:o + p.numel()].view_as(p)
            o += p.numel()
        self._params = params

    def set_env(self, env):
        """``model.set_env(train_env)`` (train/Grid_Train.py:208): new rollout storage, fresh episode starts."""
        self.env = env
        N, T, S = env.num_envs, self.n_steps, self.seq_len
        dev = self.device
        Fd = self.policy.obs_dim
        self.num_envs = N
        if self._ops is None:
            from .train_ops import DeviceOps
            eng = getattr(env, "engine", None)
            self._ops = DeviceOps(seed=(self.seed or 0) ^ 0x5DEECE66D, env_id0=getattr(eng, "env_id0", 0))
        self._obs = torch.zeros((T + 1, N, Fd), dtype=torch.float32, device=dev)
        self._actions = torch.zeros((T, N), dtype=torch.int64, device=dev)
        self._rewards = torch.zeros((T, N), dtype=torch.float32, device=dev)
        self._values = torch.zeros((T, N), dtype=torch.float32, device=dev)
        self._logp = torch.zeros((T, N), dtype=torch.float32, device=dev)
        self._starts = torch.zeros((T, N), dtype=torch.uint8, device=dev)
        self._adv = torch.zeros((T, N), dtype=torch.float32, device=dev)
        self._ret = torch.zeros((T, N), dtype=torch.float32, device=dev)
        L, H = self.policy.n_lstm_layers, self.policy.lstm_hidden_size
        self._chunk_states = torch.zeros((T // S, 4, L, N, H), dtype=torch.float32, device=dev)
        self._state: LSTMState = self.policy.initial_state(N, dev)
        self._last_starts = torch.ones(N, dtype=torch.uint8, device=dev)
        self._obs[0].copy_(env.reset())
        self._carry_obs = False           # True once obs[T] of a finished rollout has to become obs[0] of the next
        self._graph = None                # CUDA graph of one whole rollout (captured at the second rollout)
        self._upd = self._upd_graph = None   # CUDA graph of one minibatch update (small minibatches only)
        self._upd_warm = 0
        # Philox policy-stream position: a device counter (so a captured rollout draws fresh numbers on replay)
        self._step_base = torch.zeros(1, dtype=torch.int32, device=dev) if dev.type == "cuda" else None

    # ---- rollout -----------------------------------------------------------------------------------------------
    def _rollout_step(self, t: int, state: LSTMState, starts: torch.Tensor, ep: torch.Tensor, sync_free: bool):
        """One env step of the rollout: policy forward, sample, env step (the kernel writes obs[t+1]), time-limit
        bootstrap, episode statistics.  ``sync_free``: no device->host read (what a CUDA-graph capture needs) — the
        bootstrap value is then computed for every env and masked instead of only when a time limit was hit."""
        env, pol, S = self.env, self.policy, self.seq_len
        if t % S == 0:
            cs = self._chunk_states[t // S]
            for j in range(4):
                cs[j].copy_(state[j])
        self._starts[t].copy_(starts)
        logits, values, state = pol.forward_step(self._obs[t], state, starts)
        self._ops.sample_actions(logits, t, False, actions=self._actions[t], log_prob=self._logp[t],
                                 step_offset=self._step_base)
        self._values[t].copy_(values)
        _, reward, dones, info = env.step(self._actions[t], out_obs=self._obs[t + 1])
        if self.curriculum is not None:
            self.curriculum.observe(info.terminated, info.truncated, info.episodes)
        self._rewards[t].copy_(reward)
        time_limit = (info.truncated != 0) & (info.terminated == 0)
        if sync_free or bool(time_limit.any()):
            # bootstrap through the time limit: V(terminal_observation) with the critic state after this step
            tv = pol.values_step(info.terminal_observation, state, torch.zeros_like(starts))
            self._rewards[t].add_(self.gamma * tv * time_limit.to(tv.dtype))
        dm = dones.to(torch.float32)
        ep[0] += dm.sum()
        ep[1] += (info.episodes[:, 0].view(torch.float32) * dm).sum()
        ep[2] += (info.episodes[:, 1].to(torch.float32) * dm).sum()
        return state, dones.to(torch.uint8)

    def _finish_rollout(self, state: LSTMState, starts: torch.Tensor):
        last_values = self.policy.values_step(self._obs[self.n_steps], state, starts)
        self._ops.gae(self._rewards, self._values, self._starts, last_values.contiguous(), starts.contiguous(),
                      self.gamma, self.gae_lambda, self._adv, self._ret)
        if self._step_base is not None:
            self._step_base.add_(self.n_steps)

    @torch.no_grad()
    def collect_rollouts(self, callback=None) -> bool:
        """Fill the rollout buffers with ``n_steps`` env steps of every env and compute advantages/returns.

        On a CUDA device, from the second rollout on, the whole rollout — n_steps x (policy forward, sampling kernel, env
        step kernel, bootstrap, statistics) + GAE — is ONE CUDA graph replay (SURVEY §8f row 3: env and policy inference
        fused into one launch from the host's point of view).  The first rollout runs eagerly and doubles as the warm-up
        that graph capture needs (long rollouts are captured as several graphs of ``graph_chunk`` steps replayed back to
        back).  Callbacks are then stepped after the replay; the policy does not change inside a
        rollout, so an evaluation triggered by them sees the same policy as it would have mid-rollout."""
        T = self.n_steps
        use_graph = self.cuda_graph and self.device.type == "cuda" and self._carry_obs
        if use_graph and self._graph is None:
            try:
                self._capture_rollout_graph()
            except Exception as ex:  # noqa: BLE001
                self.cuda_graph = False
                use_graph = False
                if self.verbose:
                    print(f"CUDA-graph capture of the rollout failed ({ex!r}); continuing with eager launches")
        if use_graph:
            for graph in self._graph:
                graph.replay()
            for _ in range(T):
                self.num_timesteps += self.num_envs * self.world
                if callback is not None and callback.on_step(self) is False:
                    return False
            ep = self._g_ep
        else:
            ep = torch.zeros(3, dtype=torch.float32, device=self.device)
            state, starts = self._state, self._last_starts
            if self._carry_obs:
                self._obs[0].copy_(self._obs[T])
            self._carry_obs = True
            for t in range(T):
                state, starts = self._rollout_step(t, state, starts, ep, sync_free=False)
                self.num_timesteps += self.num_envs * self.world
                if callback is not None and callback.on_step(self) is False:
                    return False
            self._finish_rollout(state, starts)
            for j in range(4):
                self._state[j].copy_(state[j])
            self._last_starts.copy_(starts)
        if self.curriculum is not None:
            # eager, outside any captured graph (its all-reduce); the next replay draws resets from the new table
            self.curriculum.update()
            n, r, l, rooms, p_min, p_max = torch.cat([ep.double(), self.curriculum.summary]).cpu().tolist()
            self._curriculum_log = dict(curriculum_rooms=rooms, curriculum_p_min=p_min, curriculum_p_max=p_max)
        else:
            n, r, l = ep.cpu().tolist()
        if n > 0:
            self._ep_return_mean, self._ep_len_mean = r / n, l / n
        self._episodes_this_rollout = int(n)
        return True

    def _capture_rollout_graph(self):
        """Capture the rollout as ceil(n_steps / graph_chunk) CUDA graphs that share one memory pool and are replayed back
        to back (one graph of a 2 048-step rollout — ≈ 120 k nodes — takes minutes to instantiate; 128-step graphs are
        linear in the step count).  State and episode starts flow from chunk to chunk through the static tensors."""
        T, C = self.n_steps, max(1, min(self.n_steps, self.graph_chunk))
        n_chunks = (T + C - 1) // C
        self._g_ep = torch.zeros(3, dtype=torch.float32, device=self.device)
        graphs, pool = [], None
        if getattr(self, "_roll_stream", None) is None:
            self._roll_stream = torch.cuda.Stream(device=self.device)
        if self.policy.fused_lstm:
            from .train_ops import lstm_prepare_stream
            lstm_prepare_stream(self._roll_stream)       # the fused LSTM's cuBLAS handle must exist before the capture
        torch.cuda.synchronize(self.device)
        for k in range(n_chunks):
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, pool=pool, stream=self._roll_stream):
                if k == 0:
                    self._g_ep.zero_()
                    self._obs[0].copy_(self._obs[T])
                state, starts = self._state, self._last_starts
                for t in range(k * C, min(T, (k + 1) * C)):
                    state, starts = self._rollout_step(t, state, starts, self._g_ep, sync_free=True)
                if k == n_chunks - 1:
                    self._finish_rollout(state, starts)
                for j in range(4):
                    self._state[j].copy_(state[j])
                self._last_starts.copy_(starts)
            pool = graph.pool()
            graphs.append(graph)
        self._graph = graphs

    # ---- update ------------------------------------------------------------------------------------------------
    def _chunk_view(self, x: torch.Tensor) -> torch.Tensor:
        """[T, N, ...] -> [S, (T/S)*N, ...]: sequence chunk k of env n becomes column k*N + n."""
        T, N = x.shape[0], x.shape[1]
        S = self.seq_len
        K = T // S
        rest = x.shape[2:]
        return x.reshape(K, S, N, *rest).transpose(0, 1).reshape(S, K * N, *rest)

    def _minibatch(self, data: dict, idx: torch.Tensor, cuts, acc: torch.Tensor) -> None:
        """One PPO minibatch update on the sequences ``idx`` (columns of the chunk-view tensors in ``data``): forward over
        the sequences, clipped surrogate + value + entropy loss, backward into the flat gradient buffer, (all-reduce,)
        norm clip, Adam step; running sums of the statistics go to ``acc``.  Sync-free, so it can be captured."""
        pol = self.policy
        mb_obs = data["obs"].index_select(1, idx)
        mb_state = tuple(data["state0"][j].index_select(1, idx).contiguous() for j in range(4))
        mb_starts = data["starts"].index_select(1, idx)
        logits, values, _ = pol.forward_sequence(mb_obs, mb_state, mb_starts, cuts)
        logp_all = F.log_softmax(logits, dim=-1)
        mb_actions = data["actions"].index_select(1, idx)
        logp = logp_all.gather(-1, mb_actions.unsqueeze(-1)).squeeze(-1)
        entropy = -(logp_all.exp() * logp_all).sum(-1)
        adv = data["adv"].index_select(1, idx)
        if self.normalize_advantage and adv.numel() > 1:
            adv = (adv - adv.mean()) / (adv.std() + 1e-8)
        old_logp = data["old_logp"].index_select(1, idx)
        ratio = torch.exp(logp - old_logp)
        pl1 = adv * ratio
        pl2 = adv * torch.clamp(ratio, 1.0 - self.clip_range, 1.0 + self.clip_range)
        policy_loss = -torch.min(pl1, pl2).mean()
        value_loss = F.mse_loss(data["ret"].index_select(1, idx), values)
        entropy_loss = -entropy.mean()
        loss = policy_loss + self.ent_coef * entropy_loss + self.vf_coef * value_loss
        self._flat_grad.zero_()
        loss.backward()
        if self._dist is not None:
            self._dist.all_reduce(self._flat_grad)
            self._flat_grad.div_(self.world)
        gnorm = self._flat_grad.norm()
        self._flat_grad.mul_(torch.clamp(self.max_grad_norm / (gnorm + 1e-6), max=1.0))
        self.optimizer.step()
        with torch.no_grad():
            log_ratio = logp - old_logp
            acc += torch.stack([policy_loss, value_loss, entropy_loss, ((ratio - 1.0) - log_ratio).mean(),
                                ((ratio - 1.0).abs() > self.clip_range).float().mean(), loss]).detach()

    def _update_graph_wanted(self, n_seq: int, b_seq: int) -> bool:
        """Small minibatches are bound by ≈ 700 kernel launches each (the reference's 64-transition minibatches take
        4.9 ms eagerly for well under 1 ms of device work): replay them as one CUDA graph.  Large minibatches are device-
        bound and keep the eager path, where the critic branch overlaps the actor's on a second stream."""
        return (self.cuda_graph and self.device.type == "cuda" and self._dist is None and n_seq % b_seq == 0
                and b_seq * self.seq_len <= self.graph_update_max and self.policy.n_lstm_layers == 1
                and self.policy.fused_lstm)

    def train(self) -> Dict[str, float]:
        pol, S, T, N = self.policy, self.seq_len, self.n_steps, self.num_envs
        K = T // S
        n_seq = K * N
        b_seq = max(1, min(n_seq, self.batch_size // S))
        fresh = dict(obs=self._chunk_view(self._obs[:T]), actions=self._chunk_view(self._actions),
                     old_logp=self._chunk_view(self._logp), adv=self._chunk_view(self._adv), ret=self._chunk_view(self._ret),
                     starts=self._chunk_view(self._starts),
                     state0=self._chunk_states.permute(1, 2, 0, 3, 4).reshape(4, pol.n_lstm_layers, n_seq, pol.lstm_hidden_size))
        use_graph = self._update_graph_wanted(n_seq, b_seq)
        if use_graph:
            # the graph reads its operands from fixed addresses: keep the chunk views in persistent buffers
            if self._upd is None:
                self._upd = {k: torch.empty_like(v) for k, v in fresh.items()}
                self._upd_idx = torch.zeros(b_seq, dtype=torch.int64, device=self.device)
                self._upd_acc = torch.zeros(6, dtype=torch.float32, device=self.device)
                self._upd_stream = torch.cuda.Stream(device=self.device)
                if pol.fused_lstm:
                    from .train_ops import lstm_prepare_stream
                    lstm_prepare_stream(self._upd_stream)
            for k, v in fresh.items():
                self._upd[k].copy_(v)
            # cuts=None = mask the LSTM state at EVERY timestep.  The fused LSTM (the default: capturable, the episode-start
            # mask is an operand) ignores cuts; if torch's LSTM runs instead (fused_lstm off, several layers) no fixed cut
            # list would be right for all the minibatches one captured graph replays.
            data, acc, cuts = self._upd, self._upd_acc, None
            acc.zero_()
            # everything of a captured minibatch lives on ONE stream (also the warm-up runs, so that autograd's gradient
            # accumulators are bound to the capture stream and not to the policy's side stream)
            two_streams, pol.two_streams = pol.two_streams, False
        else:
            data = fresh
            acc = torch.zeros(6, dtype=torch.float32, device=self.device)
            # timesteps (relative to a chunk) at which any sequence has an episode start: the only places where the LSTM
            # state must be masked when cuDNN runs the stretches in between.  One small device->host read per rollout.
            cut_flags = data["starts"].any(dim=1).cpu().numpy()
            cuts = [0] + [int(t) for t in np.nonzero(cut_flags)[0] if t > 0]
        stats = dict(policy_loss=0.0, value_loss=0.0, entropy_loss=0.0, approx_kl=0.0, clip_fraction=0.0, loss=0.0)
        n_mb = 0
        for _ in range(self.n_epochs):
            perm = torch.randperm(n_seq, device=self.device, generator=self._gen)
            for i0 in range(0, n_seq, b_seq):
                idx = perm[i0:i0 + b_seq]
                if not use_graph:
                    self._minibatch(data, idx, cuts, acc)
                else:
                    cur = torch.cuda.current_stream(self.device)
                    self._upd_idx.copy_(idx)
                    self._upd_stream.wait_stream(cur)
                    if self._upd_graph is None and self._upd_warm < 2:
                        with torch.cuda.stream(self._upd_stream):          # eager warm-up on the capture stream
                            self._minibatch(data, self._upd_idx, cuts, acc)
                        self._upd_warm += 1
                    else:
                        if self._upd_graph is None:
                            graph = torch.cuda.CUDAGraph()
                            with torch.cuda.graph(graph, stream=self._upd_stream, capture_error_mode="thread_local"):
                                self._minibatch(data, self._upd_idx, cuts, acc)
                            self._upd_graph = graph
                        with torch.cuda.stream(self._upd_stream):
                            self._upd_graph.replay()
                    cur.wait_stream(self._upd_stream)
                n_mb += 1
            self.n_updates += 1
        if use_graph:
            pol.two_streams = two_streams
        vals = (acc / max(1, n_mb)).cpu().tolist()
        for k, v in zip(("policy_loss", "value_loss", "entropy_loss", "approx_kl", "clip_fraction", "loss"), vals):
            stats[k] = float(v)
        y, yp = self._ret.flatten(), self._values.flatten()
        var_y = y.var()
        stats["explained_variance"] = float("nan") if float(var_y) == 0 else float(1 - (y - yp).var() / var_y)
        stats["minibatches"] = n_mb
        stats["rollout_reward_mean"] = float(self._rewards.mean())
        return stats

    # ---- learn -------------------------------------------------------------------------------------------------
    def learn(self, total_timesteps: int, reset_num_timesteps: bool = True, callback=None, log_interval: int = 1):
        """``model.learn(total_timesteps=seg_steps, reset_num_timesteps=False, callback=eval_callback)``
        (train/Grid_Train.py:228).  Timesteps count env steps summed over all envs and all ranks."""
        if self.env is None:
            raise RuntimeError("no environment: pass env= or call set_env()")
        if reset_num_timesteps:
            self.num_timesteps = 0
            target = int(total_timesteps)
        else:
            target = self.num_timesteps + int(total_timesteps)
        if callback is not None and hasattr(callback, "init_callback"):
            callback.init_callback(self)
        t_start, steps_start = time.time(), self.num_timesteps
        while self.num_timesteps < target:
            if not self.collect_rollouts(callback):
                break
            stats = self.train()
            self._iteration += 1
            dt = max(time.time() - t_start, 1e-9)
            rec = dict(iteration=self._iteration, total_timesteps=self.num_timesteps,
                       fps=(self.num_timesteps - steps_start) / dt, ep_rew_mean=self._ep_return_mean,
                       ep_len_mean=self._ep_len_mean, episodes=self._episodes_this_rollout, n_updates=self.n_updates,
                       **stats, **self._curriculum_log)
            self.logger.append(rec)
            if self.verbose and self.rank == 0 and self._iteration % max(1, log_interval) == 0:
                print("| iter {iteration:5d} | steps {total_timesteps:11d} | fps {fps:11.0f} | ep_rew_mean {ep_rew_mean:9.2f} | "
                      "ep_len_mean {ep_len_mean:8.1f} | loss {loss:8.4f} | pi {policy_loss:8.4f} | vf {value_loss:9.4f} | "
                      "ent {entropy_loss:7.4f} | kl {approx_kl:7.4f} | clip {clip_fraction:5.3f} |".format(**rec), flush=True)
        return self

    # ---- inference ---------------------------------------------------------------------------------------------
    @torch.no_grad()
    def predict(self, observation, state=None, episode_start=None, deterministic: bool = False):
        """``model.predict(obs, state=state, episode_start=[...], deterministic=True)`` (train/evaluate_grid.py:186-191).
        Accepts numpy or torch observations of shape [80] or [B, 80]; returns (actions, state) of the same kind."""
        is_np = not isinstance(observation, torch.Tensor)
        obs = torch.as_tensor(np.asarray(observation) if is_np else observation, dtype=torch.float32, device=self.device)
        single = obs.dim() == 1
        if single:
            obs = obs.unsqueeze(0)
        B = obs.shape[0]
        if state is None:
            state = self.policy.initial_state(B, self.device)
        if episode_start is None:
            starts = torch.zeros(B, dtype=torch.uint8, device=self.device)
        else:
            starts = torch.as_tensor(np.asarray(episode_start, dtype=np.uint8) if not isinstance(episode_start, torch.Tensor)
                                     else episode_start, device=self.device).to(torch.uint8).reshape(B)
        logits, _, state = self.policy.forward_step(obs, state, starts)
        if deterministic:
            actions = logits.argmax(dim=-1)
        else:
            actions = torch.multinomial(torch.softmax(logits, dim=-1), 1, generator=self._gen).squeeze(-1)
        if is_np:
            a = actions.cpu().numpy()
            return (a[0] if single else a), state
        return (actions[0] if single else actions), state

    # ---- checkpoints -------------------------------------------------------------------------------------------
    def _data(self) -> dict:
        return dict(format_version=FORMAT_VERSION, policy_class="MlpLstmPolicy", policy_kwargs=self.policy.kwargs(),
                    learning_rate=self.learning_rate, n_steps=self.n_steps, batch_size=self.batch_size,
                    n_epochs=self.n_epochs, gamma=self.gamma, gae_lambda=self.gae_lambda, clip_range=self.clip_range,
                    ent_coef=self.ent_coef, vf_coef=self.vf_coef, max_grad_norm=self.max_grad_norm,
                    normalize_advantage=self.normalize_advantage, seq_len=self.seq_len, seed=self.seed,
                    num_timesteps=self.num_timesteps, n_updates=self.n_updates, iteration=self._iteration)

    def save(self, path) -> Path:
        """``model.save(save_path)`` (train/Grid_Train.py:232-233): a ``.zip`` holding ``data`` (JSON hyper-parameters and
        counters), ``policy.pth`` and ``policy.optimizer.pth`` (torch state dicts; parameter names follow sb3-contrib), and
        ``curriculum.pth`` (``RoomCurriculum.state_dict``) when a curriculum is set."""
        p = _append_zip_suffix(path)
        p.parent.mkdir(parents=True, exist_ok=True)
        if self.rank != 0:
            return p
        with zipfile.ZipFile(p, "w", compression=zipfile.ZIP_STORED) as z:
            z.writestr("data", json.dumps(self._data(), indent=1))
            members = [("policy.pth", self.policy.state_dict()), ("policy.optimizer.pth", self.optimizer.state_dict())]
            if self.curriculum is not None:
                members.append(("curriculum.pth", self.curriculum.state_dict()))
            for name, sd in members:
                buf = io.BytesIO()
                torch.save(sd, buf)
                z.writestr(name, buf.getvalue())
            z.writestr("_nav3d_version", "nav3d-b200 RecurrentPPO checkpoint, format %d" % FORMAT_VERSION)
        return p

    @classmethod
    def load(cls, path, env=None, device=None, verbose: int = 0, ops=None, curriculum=None, **overrides) -> "RecurrentPPO":
        """``RecurrentPPO.load(model_path, env=train_env, verbose=1)`` (train/Train_Further.py:146).  ``curriculum``: a
        ``RoomCurriculum`` the model uses from now on; it takes the checkpoint's curriculum state when there is one."""
        p = Path(path)
        if not p.exists():
            p = _append_zip_suffix(path)
        with zipfile.ZipFile(p, "r") as z:
            data = json.loads(z.read("data").decode())
            policy_sd = torch.load(io.BytesIO(z.read("policy.pth")), map_location="cpu", weights_only=True)
            opt_sd = torch.load(io.BytesIO(z.read("policy.optimizer.pth")), map_location="cpu", weights_only=True)
            cur_sd = (torch.load(io.BytesIO(z.read("curriculum.pth")), map_location="cpu", weights_only=True)
                      if curriculum is not None and "curriculum.pth" in z.namelist() else None)
        if data.get("format_version") != FORMAT_VERSION:
            raise ValueError(f"{p}: unsupported checkpoint format {data.get('format_version')}")
        kw = {k: data[k] for k in ("learning_rate", "n_steps", "batch_size", "n_epochs", "gamma", "gae_lambda", "clip_range",
                                  "ent_coef", "vf_coef", "max_grad_norm", "normalize_advantage", "seq_len", "seed")}
        kw.update(overrides)
        model = cls(env, policy_kwargs=data["policy_kwargs"], verbose=verbose, ops=ops, device=device, curriculum=curriculum,
                    **kw)
        if cur_sd is not None:
            curriculum.load_state_dict(cur_sd)
        model.policy.load_state_dict(policy_sd)
        model._flatten_grads()                                # load_state_dict keeps the parameters; re-pin the gradients
        model.optimizer.load_state_dict(opt_sd)
        model.num_timesteps, model.n_updates, model._iteration = data["num_timesteps"], data["n_updates"], data["iteration"]
        return model

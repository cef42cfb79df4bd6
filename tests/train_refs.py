"""Plain-PyTorch fp32 restatements of the rollout-loop kernels (``csrc/nav3d_train.cu``), float64 references of the
sampling, GAE and fused-LSTM kernels with error bounds, and an oracle-backed stand-in for ``nav3d.BatchedCubicEnv``.
TEST INFRASTRUCTURE ONLY: the GPU tests check the CUDA kernels against these, and the CPU tests run the trainer's host
logic on them (the product has no CPU path)."""
from types import SimpleNamespace

import numpy as np
import torch

EPS32 = 2.0 ** -23                      # float32 machine epsilon (twice the unit roundoff)
POLICY_STREAM = 0x504F4C49              # "POLI", include/nav3d.h nav3d_sample_actions
# (env, step, word 0) of the policy stream with seed 1234: word 0 >= 0xFFFFFF80, where float(word) / 2^32 rounds to 1.0,
# and word 0 < 256, where u = (word >> 8) / 2^24 is 0.  The sampling edge tests run these counters.
U_ONE_COUNTERS = [(1734339, 8, 0xFFFFFFFC), (2932430, 5, 0xFFFFFF9E), (2717627, 7, 0xFFFFFFDD), (3343352, 7, 0xFFFFFFDD),
                  (2594146, 12, 0xFFFFFFA4)]
U_ZERO_COUNTERS = [(29672, 3, 0x3C), (1635937, 9, 0xA8)]
_M32 = np.uint64(0xFFFFFFFF)


def philox4x32_10_np(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 over arrays of counters (broadcast against each other), in uint64 arithmetic: the vectorized twin
    of ``oracle.c_oracle.philox4x32_10``.  Returns the four output words as uint32 arrays."""
    c = [np.asarray(v, dtype=np.uint64) & _M32 for v in np.broadcast_arrays(c0, c1, c2, c3)]
    k0, k1 = int(k0) & 0xFFFFFFFF, int(k1) & 0xFFFFFFFF
    for _ in range(10):
        p0 = c[0] * np.uint64(0xD2511F53)
        p1 = c[2] * np.uint64(0xCD9E8D57)
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ np.uint64(k0), p1 & _M32, (p0 >> np.uint64(32)) ^ c[3] ^ np.uint64(k1), p0 & _M32]
        k0, k1 = (k0 + 0x9E3779B9) & 0xFFFFFFFF, (k1 + 0xBB67AE85) & 0xFFFFFFFF
    return tuple(v.astype(np.uint32) for v in c)


def policy_word0(seed, env_ids, step):
    """Word 0 of the policy stream at counter (env_id, step, 0, "POLI") with the key of ``seed`` (all mod 2^32)."""
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    ids = np.asarray(env_ids, dtype=np.uint64) & _M32
    return philox4x32_10_np(ids, int(step) & 0xFFFFFFFF, 0, POLICY_STREAM, seed & 0xFFFFFFFF, seed >> 32)[0]


def sample_reference64(logits, seed, env_id0, step, step_offset=0):
    """The draw include/nav3d.h documents for nav3d_sample_actions, in float64.

    u = (word0 >> 8) / 2^24 with word0 from counter (env_id0 + i, step + step_offset, 0, "POLI"); action = first k with
    cdf[k] > u, cdf the float64 cumulative softmax.  Returns a SimpleNamespace of float64 numpy arrays (rows of ``logits``):
      action, log_prob (of that action), log_softmax [N, A], entropy (0 * log 0 counted as 0), u, cdf [N, A], p [N, A],
      margin = min |u - cdf[k]| over the decision boundaries k, near = u lies within cdf_bound of a decision boundary (a
      row the fp32 kernel may draw differently), greedy / greedy_log_prob (first maximum), and the per-row fp32 bounds:
      cdf_bound[k]  how far the kernel's fp32 walk may move boundary k, in units of u (see ``_cdf_bound``);
      lp_bound[k]   how far the kernel's fp32 log_softmax may be from log_prob64[k];
      ent_bound     how far the kernel's fp32 entropy may be from entropy64."""
    l = np.asarray(torch.as_tensor(logits).detach().cpu(), dtype=np.float64)
    N, A = l.shape
    ids = (int(env_id0) + np.arange(N, dtype=np.uint64)) & _M32
    w0 = policy_word0(seed, ids, (int(step) + int(step_offset)) & 0xFFFFFFFF)
    u = (w0 >> np.uint32(8)).astype(np.float64) * 2.0 ** -24
    mx = l.max(axis=1, keepdims=True)
    d = mx - l                                                   # >= 0, +inf for masked entries
    e = np.exp(-d)
    s = e.sum(axis=1, keepdims=True)
    cdf = np.cumsum(e, axis=1) / s
    action = np.argmax(cdf > u[:, None], axis=1)
    lse = np.log(s)
    lp = -d - lse
    p = e / s
    with np.errstate(invalid="ignore"):
        plp = np.where(p > 0, p * lp, 0.0)
    entropy = -plp.sum(axis=1)
    # decision boundaries: the top of every interval with nonzero weight, except where the rest of the row's mass is
    # below 2^-30 (there both the float64 walk and the kernel's stop for any u <= 1 - 2^-24)
    live = p > 0
    decisive = live & (cdf < 1.0 - 2.0 ** -30)
    cdf_bound = _cdf_bound(e, s, d)
    margin = np.where(decisive, np.abs(u[:, None] - cdf), np.inf).min(axis=1)
    near = (decisive & (np.abs(u[:, None] - cdf) <= cdf_bound)).any(axis=1)
    # log_prob = fl(fl(row[a] - mx) - logf(sum)): two subtractions, logf (1 ulp) of a sum whose relative error is at most
    # the walk's total (cdf_bound's last column), each charged a full eps32
    lse_err = cdf_bound[:, -1:] + EPS32 * (np.abs(lse) + 1.0)
    with np.errstate(invalid="ignore"):
        lp_bound = EPS32 * (d + np.abs(lp)) + lse_err
    # entropy = -sum_k expf(lp_k) * lp_k: each term carries lp_k's error, expf's 2 ulp and the product's rounding, the
    # running sum one rounding per term
    with np.errstate(invalid="ignore"):
        term = np.where(live, p * ((np.abs(lp) + 1.0) * (lp_bound + 2 * EPS32)), 0.0)
    ent_bound = term.sum(axis=1) + A * EPS32 * (entropy + EPS32)
    rows = np.arange(N)
    greedy = np.argmax(l == mx, axis=1)
    return SimpleNamespace(action=action, log_prob=lp[rows, action], log_softmax=lp, entropy=entropy, u=u, margin=margin,
                           near=near, cdf=cdf, p=p,
                           cdf_bound=cdf_bound, lp_bound=lp_bound, ent_bound=ent_bound, greedy=greedy,
                           greedy_log_prob=lp[rows, greedy], word0=w0)


def _cdf_bound(e, s, d):
    """Per boundary k, a bound (in units of u) on how far the kernel's fp32 decision `u * sum < acc_k` can sit from the
    float64 `u < cdf[k]`.  Charged: each weight expf(fl(row[k] - mx)) is off by the subtraction's rounding (d_k e^-d_k
    eps32 <= eps32) plus expf's 2 ulp (2 eps32 e_k); each running-sum addition rounds once (eps32 * acc_j); the target
    u * sum rounds once and uses the computed sum, which carries the whole walk's error.  eps32 (not the unit roundoff
    eps32 / 2) throughout, so the bound has a factor of 2 in hand."""
    with np.errstate(invalid="ignore"):
        eta = np.where(e > 0, e * (2 + d) * EPS32, 0.0)
    acc = np.cumsum(e, axis=1)
    err_acc = EPS32 * np.cumsum(acc, axis=1) + np.cumsum(eta, axis=1)
    return (err_acc + err_acc[:, -1:] + EPS32 * s) / s


def gae_reference64(rewards, values, starts, last_values, last_dones, gamma, lam, c=2.0):
    """GAE in float64 (numpy, time-major [T][N]) with gamma and lambda rounded to float32 as the kernel receives them,
    plus per-element error bounds for an fp32 evaluation of the same recursion:
        B_t = c eps32 (|r_t| + gamma |V_{t+1}| nnt + |V_t| + |A_t| + gamma lambda nnt |A_{t+1}|) + gamma lambda nnt B_{t+1}
    with nnt = 1 - start_{t+1} (1 - last_dones at t = T-1) and B_T = 0: every product and sum of a step rounds once,
    charged a full eps32 each (c = 2 covers the two roundings in delta and the two in the update), and the previous
    step's error is carried by the same factor as A.  Returns (adv, ret, adv_bound, ret_bound), ret_bound = B + eps32 |ret|."""
    f = lambda t: np.asarray(torch.as_tensor(t).detach().cpu(), dtype=np.float64)
    r, v, st, lv, ld = f(rewards), f(values), f(starts), f(last_values), f(last_dones)
    g, gl = float(np.float32(gamma)), float(np.float32(lam))
    gl = g * gl
    T = r.shape[0]
    adv, bnd = np.zeros_like(r), np.zeros_like(r)
    a_next, b_next, v_next, nnt = np.zeros_like(lv), np.zeros_like(lv), lv, 1.0 - ld
    for t in reversed(range(T)):
        a = r[t] + g * v_next * nnt - v[t] + gl * nnt * a_next
        b = c * EPS32 * (np.abs(r[t]) + g * np.abs(v_next) * nnt + np.abs(v[t]) + np.abs(a) + gl * nnt * np.abs(a_next)) \
            + gl * nnt * b_next
        adv[t], bnd[t] = a, b
        a_next, b_next, v_next, nnt = a, b, v[t], 1.0 - st[t]
    ret = adv + v
    return adv, ret, bnd, bnd + EPS32 * np.abs(ret)


def lstm_reference64(x, w_ih, w_hh, b_ih, b_hh, h0, c0, starts):
    """The fused LSTM's masked recurrence written out step by step in plain torch, in the dtype and on the device of its
    inputs (float64 for the reference; autograd gives the four parameter gradients):
        h, c <- h * keep_t, c * keep_t   (keep_t = 1 - starts[t])
        i, f, g, o = sigma, sigma, tanh, sigma (x_t W_ih^T + b_ih + h W_hh^T + b_hh)
        c <- f c + i g ;  h <- o tanh(c)
    Returns (h_all [S, B, H], h_last, c_last)."""
    h, c = h0, c0
    ys = []
    for t in range(x.shape[0]):
        keep = (1 - starts[t].to(x.dtype)).unsqueeze(-1)
        h, c = h * keep, c * keep
        gi, gf, gg, go = (x[t] @ w_ih.T + b_ih + h @ w_hh.T + b_hh).chunk(4, dim=-1)
        c = torch.sigmoid(gf) * c + torch.sigmoid(gi) * torch.tanh(gg)
        h = torch.sigmoid(go) * torch.tanh(c)
        ys.append(h)
    return torch.stack(ys), h, c


def lstm_with_cuts(lstm, x, h0, c0, starts):
    """torch.nn.LSTM (cuDNN on the GPU) over the sequence cut at every step where some env starts an episode, the state
    of those envs zeroed at the cut: the trainer's cuDNN path."""
    S, B = starts.shape
    cuts = [0] + [t for t in range(1, S) if bool(starts[t].any())] + [S]
    h, c = h0.unsqueeze(0), c0.unsqueeze(0)
    outs = []
    for a, b in zip(cuts[:-1], cuts[1:]):
        keep = (1 - starts[a].to(x.dtype)).view(1, B, 1)
        y, (h, c) = lstm(x[a:b], (h * keep, c * keep))
        outs.append(y)
    return torch.cat(outs), h[0], c[0]


def gae_reference(rewards, values, starts, last_values, last_dones, gamma, lam):
    """SB3's compute_returns_and_advantage, time-major, fp32."""
    T = rewards.shape[0]
    adv = torch.zeros_like(rewards)
    gae = torch.zeros_like(last_values)
    for t in reversed(range(T)):
        if t == T - 1:
            nnt, nv = 1.0 - last_dones.float(), last_values
        else:
            nnt, nv = 1.0 - starts[t + 1].float(), values[t + 1]
        delta = rewards[t] + gamma * nv * nnt - values[t]
        gae = delta + gamma * lam * nnt * gae
        adv[t] = gae
    return adv, adv + values


class TorchOps:
    """Same interface as nav3d.train_ops.DeviceOps, in torch, on any device."""

    def __init__(self, seed=0):
        self.gen = torch.Generator().manual_seed(seed)

    def sample_actions(self, logits, step, greedy=False, actions=None, log_prob=None, entropy=None, step_offset=None):
        lp = torch.log_softmax(logits, dim=-1)
        a = lp.argmax(-1) if greedy else torch.multinomial(lp.exp().cpu(), 1, generator=self.gen).squeeze(-1).to(logits.device)
        l = lp.gather(-1, a.unsqueeze(-1)).squeeze(-1)
        if actions is not None:
            actions.copy_(a)
        if log_prob is not None:
            log_prob.copy_(l)
        if entropy is not None:
            entropy.copy_(-(lp.exp() * lp).sum(-1))
        return (actions if actions is not None else a), (log_prob if log_prob is not None else l)

    def gae(self, rewards, values, episode_starts, last_values, last_dones, gamma, gae_lambda, advantages, returns):
        a, r = gae_reference(rewards, values, episode_starts, last_values, last_dones, gamma, gae_lambda)
        advantages.copy_(a)
        returns.copy_(r)


class OracleBatchedEnv:
    """``nav3d.BatchedCubicEnv``'s interface on the CPU oracle (``oracle.c_oracle.OracleVec``), torch CPU tensors."""

    def __init__(self, rooms, num_envs, local_map_length=10, seed=0, crash_penalty=-2.0):
        from oracle import c_oracle
        self.ov = c_oracle.OracleVec(num_envs, [c_oracle.OracleRoom(r.grid, -2) for r in rooms], local_map_length,
                                     crash_penalty, seed, 0, True)
        self.num_envs = num_envs
        self.device = torch.device("cpu")
        self.engine = SimpleNamespace(env_id0=0)
        self._obs = torch.zeros((num_envs, 80), dtype=torch.float32)
        self._eps = torch.zeros((num_envs, 8), dtype=torch.int32)

    def reset(self, picks=None):
        self._obs.copy_(torch.from_numpy(self.ov.reset(picks)))
        return self._obs

    def step(self, actions, out_obs=None):
        ov = self.ov
        ov.step(torch.as_tensor(actions).cpu().numpy())
        obs = self._obs if out_obs is None else out_obs
        obs.copy_(torch.from_numpy(ov.obs))
        term, trunc = torch.from_numpy(ov.terminated.copy()), torch.from_numpy(ov.truncated.copy())
        done = (ov.terminated | ov.truncated).astype(bool)
        eps = self._eps.numpy()
        eps[done, 0] = ov.ep_ret[done].astype(np.float32).view(np.int32)
        eps[done, 1], eps[done, 2], eps[done, 3] = ov.ep_len[done], ov.ep_bumps[done], ov.ep_visited[done]
        eps[done, 6], eps[done, 7] = ov.terminated[done], ov.truncated[done]
        info = SimpleNamespace(terminated=term, truncated=trunc, terminal_observation=torch.from_numpy(ov.terminal_obs.copy()),
                               episodes=self._eps)
        return obs, torch.from_numpy(ov.reward.astype(np.float32)), torch.from_numpy(done), info

    def close(self):
        pass

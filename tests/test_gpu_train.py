"""-m gpu: the rollout-loop kernels (csrc/nav3d_train.cu, through the C ABI) and the fused LSTM (csrc/nav3d_lstm.cu)
against float64 references with fp32 error bounds (tests/train_refs.py), and the LSTM-PPO trainer end to end on the
GPU-resident env."""
import math

import numpy as np
import pytest
import torch

from conftest import ROOMS
from train_refs import (EPS32, U_ONE_COUNTERS, U_ZERO_COUNTERS, gae_reference64, lstm_reference64, lstm_with_cuts,
                        sample_reference64)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops():
    from nav3d.train_ops import DeviceOps
    return DeviceOps(seed=1234, env_id0=0)


def _check_gae(ops, r, v, s, lv, ld, gamma, lam):
    """The kernel against gae_reference64: every advantage within B_t, every return within B_t + eps32 |ret_t|."""
    adv, ret = torch.empty_like(r), torch.empty_like(r)
    ops.gae(r, v, s, lv, ld, gamma, lam, adv, ret)
    want_a, want_r, bound_a, bound_r = gae_reference64(r, v, s, lv, ld, gamma, lam)
    err_a = np.abs(adv.cpu().double().numpy() - want_a)
    err_r = np.abs(ret.cpu().double().numpy() - want_r)
    assert np.all(np.isfinite(err_a)) and np.all(np.isfinite(err_r))
    assert np.all(err_a <= bound_a), (err_a.max(), float((err_a / np.maximum(bound_a, 1e-300)).max()))
    assert np.all(err_r <= bound_r), (err_r.max(), float((err_r / np.maximum(bound_r, 1e-300)).max()))
    return adv, ret


def _gae_inputs(T, N, seed, p_start=0.05, p_done=0.3):
    g = torch.Generator(device="cuda").manual_seed(seed)
    dev = "cuda"
    r = torch.randn((T, N), generator=g, device=dev)
    v = torch.randn((T, N), generator=g, device=dev)
    s = (torch.rand((T, N), generator=g, device=dev) < p_start).to(torch.uint8)
    lv = torch.randn(N, generator=g, device=dev)
    ld = (torch.rand(N, generator=g, device=dev) < p_done).to(torch.uint8)
    return r, v, s, lv, ld


@pytest.mark.parametrize("T,N", [(1, 1), (7, 33), (64, 5000), (2048, 8), (1, 257), (64, 1), (64, 255), (64, 257),
                                 (64, 2 ** 20 + 3)])
def test_gae_kernel_matches_torch_reference(ops, T, N):
    """nav3d_gae at ragged N and the trainer's shape (T = 64, 2^20 envs) against float64 GAE with the bound B_t of
    gae_reference64 (fp32 rounding of every operation, carried back through the recursion)."""
    _check_gae(ops, *_gae_inputs(T, N, T * 1000 + N), 0.99, 0.95)


@pytest.mark.parametrize("case", ["gamma_lambda_1_long", "gamma_0", "all_starts", "no_starts", "last_dones_none",
                                  "large_cancelling_rewards"])
def test_gae_kernel_regimes(ops, case):
    """gamma = lambda = 1 over 4096 steps (no discount: the error grows fastest), gamma = 0 (A = r - V), every step an
    episode start with every last_done set, none of either, and rewards of about 1e4 against values that cancel them
    (advantages far smaller than their inputs)."""
    T, N, gamma, lam, p_start, p_done = 64, 300, 0.99, 0.95, 0.05, 0.3
    if case == "gamma_lambda_1_long":
        T, N, gamma, lam, p_start, p_done = 4096, 64, 1.0, 1.0, 0.0, 0.0
    elif case == "gamma_0":
        gamma = 0.0
    elif case == "all_starts":
        p_start, p_done = 1.0, 1.0
    elif case == "no_starts":
        p_start, p_done = 0.0, 0.0
    elif case == "last_dones_none":
        p_done = 0.0
    r, v, s, lv, ld = _gae_inputs(T, N, 99, p_start, p_done)
    if case == "large_cancelling_rewards":
        # V_t = r_t + gamma V_{t+1} (1 - start_{t+1}) + small: the exact discounted return plus noise
        r = 1e4 * r
        nxt, nnt = lv.double() * 1e4, 1.0 - ld.double()
        vv = torch.empty((T, N), dtype=torch.float64, device="cuda")
        for t in reversed(range(T)):
            vv[t] = r[t].double() + float(np.float32(gamma)) * nxt * nnt + v[t].double()
            nxt, nnt = vv[t], 1.0 - s[t].double()
        v, lv = vv.float(), (lv * 1e4).contiguous()
    adv, ret = _check_gae(ops, r, v, s, lv, ld, gamma, lam)
    if case == "large_cancelling_rewards":
        assert adv.abs().max().item() < 1e-2 * r.abs().max().item()
    if case == "gamma_lambda_1_long":
        # no discount, no starts: A_0 = sum of all rewards + last value - V_0
        want = r.double().sum(0) + lv.double() - v[0].double()
        assert torch.allclose(adv[0].double(), want, rtol=0, atol=1e-4 * (r.abs().sum(0).max().item() + 1))
    # starts[0] only feeds the step before t = 0, which does not exist: flipping it changes nothing, bit for bit
    s2 = s.clone()
    s2[0] ^= 1
    adv2, ret2 = torch.empty_like(r), torch.empty_like(r)
    ops.gae(r, v, s2, lv, ld, gamma, lam, adv2, ret2)
    assert torch.equal(adv, adv2) and torch.equal(ret, ret2)


def test_sample_actions_logprob_entropy_greedy(ops):
    g = torch.Generator(device="cuda").manual_seed(0)
    logits = 3.0 * torch.randn((4099, 6), generator=g, device="cuda")
    ent = torch.empty(4099, device="cuda")
    a, lp = ops.sample_actions(logits, step=3, entropy=ent)
    ref = torch.log_softmax(logits, dim=-1)
    assert a.dtype == torch.int64 and int(a.min()) >= 0 and int(a.max()) <= 5
    assert torch.allclose(lp, ref.gather(-1, a.unsqueeze(-1)).squeeze(-1), atol=2e-6, rtol=1e-5)
    assert torch.allclose(ent, -(ref.exp() * ref).sum(-1), atol=2e-6, rtol=1e-5)
    ga, glp = ops.sample_actions(logits, step=3, greedy=True)
    assert torch.equal(ga, logits.argmax(-1))
    assert torch.allclose(glp, ref.max(-1).values, atol=2e-6, rtol=1e-5)
    # deterministic in (seed, env id, step); a different step gives a different draw
    a2, _ = ops.sample_actions(logits, step=3)
    a3, _ = ops.sample_actions(logits, step=4)
    assert torch.equal(a, a2) and not torch.equal(a, a3)


def test_sample_actions_distribution_and_shard_independence():
    from nav3d.train_ops import DeviceOps
    N = 600_000
    probs = torch.tensor([0.05, 0.4, 0.1, 0.25, 0.15, 0.05])
    logits = probs.log().repeat(N, 1).cuda().contiguous()
    full = DeviceOps(seed=77, env_id0=0)
    a, _ = full.sample_actions(logits, step=11)
    counts = torch.bincount(a, minlength=6).cpu().double()
    expected = probs.double() * N
    chi2 = float(((counts - expected) ** 2 / expected).sum())
    assert chi2 < 25.7, (chi2, counts)                     # 5 dof, p = 1e-4
    # two shards keyed by global env id reproduce the single-shard draw
    half = N // 2
    lo, _ = DeviceOps(seed=77, env_id0=0).sample_actions(logits[:half], step=11)
    hi, _ = DeviceOps(seed=77, env_id0=half).sample_actions(logits[half:], step=11)
    assert torch.equal(torch.cat([lo, hi]), a)
    # successive steps are independent: lag-1 agreement is what independence predicts
    b, _ = full.sample_actions(logits, step=12)
    agree = float((a == b).double().mean())
    assert abs(agree - float((probs ** 2).sum())) < 0.005


def _sampling_logits(N, A, scale, seed):
    """scale * N(0, 1) logits, with every 16th row of each kind below: the first half masked (-inf), the last half
    masked, all but one masked, one logit 200 above the rest (their fp32 weights underflow to 0), all equal."""
    rng = np.random.default_rng(seed)
    lg = (scale * rng.standard_normal((N, A))).astype(np.float32)
    kind = np.arange(N) % 16
    j = rng.integers(0, A, size=N)
    if A > 1:
        lg[kind == 1, :A // 2] = -np.inf
        lg[kind == 2, A - A // 2:] = -np.inf
        r = np.nonzero(kind == 3)[0]
        keep = lg[r, j[r]].copy()
        lg[r] = -np.inf
        lg[r, j[r]] = keep
        r = np.nonzero(kind == 4)[0]
        top = lg[r, j[r]].copy()
        lg[r] = top[:, None] - 200.0 - np.abs(rng.standard_normal((len(r), A))).astype(np.float32)
        lg[r, j[r]] = top
    lg[kind == 5] = lg[kind == 5, :1]
    return lg


def _check_draws(logits, seed, env_id0, step, step_offset=0, cap=0.0, label=""):
    """nav3d_sample_actions against sample_reference64, row by row.

    * Every row: the drawn action has nonzero fp32 weight (never a -inf logit, never one more than 105 below the row's
      maximum, whose expf is 0), and u lies in its interval [cdf[a-1], cdf[a]) widened by the fp32 bound of each end
      (_cdf_bound: the weights' and the running sum's rounding, A + 4 roundings of order eps32 * sum).
    * Rows whose u is farther than that bound from every decision boundary: the action equals the float64 draw.  The
      others ("near" rows) are counted and printed; at most cap * N of them, rounded up, are allowed.
    * log_prob within lp_bound of the float64 log-softmax of the drawn action (two fp32 subtractions and logf of the
      walk's sum), entropy within ent_bound of the float64 entropy (each of the A terms carries its log-prob's error,
      expf's 2 ulp and a product's rounding; the running sum one rounding per term); both finite on every row."""
    from nav3d.train_ops import DeviceOps
    N, A = logits.shape
    lg = torch.from_numpy(logits).cuda()
    ent = torch.empty(N, device="cuda")
    off = torch.tensor([step_offset], dtype=torch.int32, device="cuda") if step_offset else None
    a, lp = DeviceOps(seed=seed, env_id0=env_id0).sample_actions(lg, step=step, entropy=ent, step_offset=off)
    a, lp, ent = a.cpu().numpy(), lp.cpu().double().numpy(), ent.cpu().double().numpy()
    ref = sample_reference64(logits, seed, env_id0, step, step_offset)
    rows = np.arange(N)
    assert a.min() >= 0 and a.max() < A
    d = logits.max(axis=1).astype(np.float64) - logits[rows, a].astype(np.float64)
    assert np.all(d < 105.0), np.nonzero(d >= 105.0)[0][:10]
    lo = np.where(a > 0, ref.cdf[rows, np.maximum(a - 1, 0)] - ref.cdf_bound[rows, np.maximum(a - 1, 0)], -1.0)
    hi = ref.cdf[rows, a] + ref.cdf_bound[rows, a]
    bad = np.nonzero(~((lo <= ref.u) & (ref.u < hi)))[0]
    assert len(bad) == 0, (label, bad[:10], a[bad[:10]], ref.action[bad[:10]], ref.u[bad[:10]])
    differ = a != ref.action
    assert not np.any(differ & ~ref.near), (label, np.nonzero(differ & ~ref.near)[0][:10])
    n_near = int(ref.near.sum())
    print(f"sample_actions {label}: {n_near} of {N} rows within the fp32 bound of a CDF boundary "
          f"({int(differ.sum())} drawn differently from float64)")
    assert n_near <= math.ceil(cap * N), (label, n_near)
    assert np.all(np.isfinite(lp)) and np.all(np.isfinite(ent))
    assert np.all(np.abs(lp - ref.log_softmax[rows, a]) <= ref.lp_bound[rows, a]), label
    assert np.all(np.abs(ent - ref.entropy) <= ref.ent_bound), (label, float(np.abs(ent - ref.entropy).max()))
    return a, ref


def _near_cap(A):
    """The share of rows allowed to fall within the fp32 bound of a boundary.  Up to 33 actions: 1e-4 (one row of
    4099).  Beyond, rows inside the bound are inherent to fp32, not a weakness of the kernel: a row has up to A
    boundaries and each boundary's bound grows like A eps32, so the share grows like A^2 eps32 (on these inputs, which
    alone decide it: 0.8 % of rows at A = 255 and 12.5 % at A = 1024 with near-uniform logits).  There the cap is
    2 A^2 eps32, and every row is still held to the interval check."""
    return 1e-4 if A <= 33 else 2 * A * A * EPS32


@pytest.mark.parametrize("A", [1, 2, 3, 6, 7, 32, 33, 255, 1024])
@pytest.mark.parametrize("scale", [0.01, 3.0, 40.0])
def test_sample_actions_match_float64_draw(A, scale):
    """Exact draws at a ragged N = 4099 for every action count the ABI allows up to 1024, near-uniform to near-greedy
    rows, masked entries, underflowing weights and ties (see _sampling_logits, _check_draws)."""
    lg = _sampling_logits(4099, A, scale, A * 1000 + int(scale * 100))
    _check_draws(lg, 1234, 0, 3 + A, cap=_near_cap(A), label=f"A={A} scale={scale}")


def test_sample_actions_match_float64_draw_at_trainer_scale():
    """A = 6 at the trainer's 2^20 envs (+3, ragged), at a nonzero env_id0 and through the device step offset."""
    lg = _sampling_logits(2 ** 20 + 3, 6, 3.0, 6)
    _check_draws(lg, 77, 12345, 40, step_offset=7, cap=1e-4, label="A=6 N=2^20+3")


@pytest.mark.parametrize("env,step", [(e, s) for e, s, _ in U_ONE_COUNTERS])
@pytest.mark.parametrize("row,want", [([0.0, -math.inf], 0), ([0.0, -200.0], 0),
                                      ([0.3, -1.2, 0.8, 0.1, -0.5, -math.inf], 4),
                                      ([0.3, -1.2, 0.8, 0.1, -0.5, 0.4], 5)])
def test_sample_actions_u_near_one(env, step, row, want):
    """Counters whose Philox word 0 is at least 0xFFFFFF80: u = (word >> 8) / 2^24 = 1 - 2^-24, so the draw is the last
    action with nonzero weight.  (u = word / 2^32 rounded to 1.0 in fp32 there, and the CDF walk fell through to the
    last action whatever its weight: action 1 of [0, -inf] with log_prob -inf.)"""
    from nav3d.train_ops import DeviceOps
    lg = torch.tensor([row], dtype=torch.float32, device="cuda")
    a, lp = DeviceOps(seed=1234, env_id0=env).sample_actions(lg, step=step)
    ref = sample_reference64(lg, 1234, env, step)
    assert ref.action[0] == want
    assert int(a[0]) == want and math.isfinite(float(lp[0])), (int(a[0]), float(lp[0]))
    assert abs(float(lp[0]) - ref.log_prob[0]) <= ref.lp_bound[0, want]


@pytest.mark.parametrize("env,step", [(e, s) for e, s, _ in U_ZERO_COUNTERS])
@pytest.mark.parametrize("row,want", [([-math.inf, 0.0], 1), ([-math.inf, -math.inf, 0.5, 1.0, -0.3, 0.2], 2)])
def test_sample_actions_u_zero(env, step, row, want):
    """Counters whose word 0 is below 256 (u = 0): the first action with nonzero weight, past leading masked ones."""
    from nav3d.train_ops import DeviceOps
    lg = torch.tensor([row], dtype=torch.float32, device="cuda")
    a, lp = DeviceOps(seed=1234, env_id0=env).sample_actions(lg, step=step)
    assert int(a[0]) == want == sample_reference64(lg, 1234, env, step).action[0] and math.isfinite(float(lp[0]))


def test_sample_actions_counter_wraps():
    """step + *step_offset and env_id0 + i are taken mod 2^32."""
    from nav3d.train_ops import DeviceOps
    lg = _sampling_logits(300, 6, 1.0, 5)
    ops = DeviceOps(seed=9, env_id0=2 ** 32 - 100)
    off = torch.tensor([5], dtype=torch.int32, device="cuda")
    x = torch.from_numpy(lg).cuda()
    a1, _ = ops.sample_actions(x, step=2 ** 32 - 3, step_offset=off)
    a2, _ = ops.sample_actions(x, step=2)
    assert torch.equal(a1, a2)
    _check_draws(lg, 9, 2 ** 32 - 100, 2 ** 32 - 3, step_offset=5, cap=1e-4, label="wrapped counters")


def test_sample_actions_entropy_with_masked_logits():
    """-inf logits add 0 to the entropy (0 log 0 = 0, as torch.distributions.Categorical counts it), not NaN."""
    from nav3d.train_ops import DeviceOps
    rows = [[0.0, -math.inf, 1.0, -math.inf], [-math.inf, 2.0, 2.0, 2.0], [-math.inf, -math.inf, -math.inf, 0.5]]
    lg = torch.tensor(rows, dtype=torch.float32, device="cuda")
    ent = torch.empty(3, device="cuda")
    _, lp = DeviceOps(seed=3).sample_actions(lg, step=0, entropy=ent)
    ref = sample_reference64(lg, 3, 0, 0)
    got = ent.cpu().double().numpy()
    assert np.all(np.isfinite(got)), got
    assert np.all(np.abs(got - ref.entropy) <= ref.ent_bound), (got, ref.entropy)
    want = torch.distributions.Categorical(logits=lg.double()).entropy().cpu().numpy()
    assert np.allclose(got, want, rtol=1e-6, atol=1e-6)


def test_sample_actions_greedy_ties_and_masks():
    """greedy: the first maximum wins on ties, masked entries included, and log_prob is the float64 max log-softmax."""
    from nav3d.train_ops import DeviceOps
    rng = np.random.default_rng(11)
    lg = (np.round(rng.standard_normal((4099, 7)) * 2) / 2).astype(np.float32)     # coarse values: many ties
    lg[rng.random((4099, 7)) < 0.3] = -np.inf
    lg[np.arange(4099), rng.integers(0, 7, 4099)] = 0.5                               # at least one finite entry
    x = torch.from_numpy(lg).cuda()
    ent = torch.empty(4099, device="cuda")
    a, lp = DeviceOps(seed=1).sample_actions(x, step=0, greedy=True, entropy=ent)
    ref = sample_reference64(lg, 1, 0, 0)
    rows = np.arange(4099)
    a = a.cpu().numpy()
    assert np.array_equal(a, ref.greedy) and np.array_equal(a, np.argmax(lg, axis=1))
    assert int((lg == lg.max(axis=1, keepdims=True)).sum(axis=1).max()) > 1          # ties were present
    assert np.all(np.abs(lp.cpu().double().numpy() - ref.greedy_log_prob) <= ref.lp_bound[rows, a])
    assert np.all(np.abs(ent.cpu().double().numpy() - ref.entropy) <= ref.ent_bound)


def test_train_ops_reject_cpu_tensors(ops):
    with pytest.raises(RuntimeError):
        ops.sample_actions(torch.zeros((4, 6)), step=0)


def test_ppo_learns_on_gpu_env(tmp_path):
    """A short run on an 8x8x6 hollow box (144 free cells, so 144-step episodes): bookkeeping, finite statistics, the
    evaluation callback, a checkpoint round trip — and the policy learns (episode return rises from about -1 for the
    untrained policy to above +20 within 0.8 M steps; measured curve in DESIGN.md)."""
    from nav3d import BatchedCubicEnv
    from nav3d.evaluation import EvalCallback, evaluate_policy
    from nav3d.ppo import RecurrentPPO
    from nav3d.rooms import rooms_from_grids
    g = np.zeros((8, 8, 6), dtype=np.int8)
    g[0], g[-1], g[:, 0], g[:, -1], g[:, :, 0], g[:, :, -1] = -2, -2, -2, -2, -2, -2
    rooms = rooms_from_grids([g])
    env = BatchedCubicEnv(rooms=rooms, num_envs=256, local_map_length=10, seed=3)
    eval_env = BatchedCubicEnv(rooms=rooms, num_envs=8, local_map_length=10, seed=4)
    model = RecurrentPPO(env, policy_kwargs=dict(net_arch=dict(pi=[256, 256, 128], vf=[256, 256, 128]), lstm_hidden_size=256,
                                                 n_lstm_layers=1),
                         learning_rate=3e-4, n_steps=64, batch_size=64 * 64, n_epochs=4, gamma=0.99, gae_lambda=0.95,
                         ent_coef=0.01, vf_coef=0.5, clip_range=0.2, seed=0)
    iters = 48
    cb = EvalCallback(eval_env, best_model_save_path=tmp_path, log_path=tmp_path, eval_freq=64 * 16, n_eval_episodes=8, verbose=0)
    launches0 = env.engine.launch_count
    model.learn(total_timesteps=iters * 64 * 256, callback=cb)
    assert model.num_timesteps == iters * 64 * 256 and len(model.logger) == iters
    assert env.engine.launch_count - launches0 >= 2 * 64           # host-side launches: the eager rollout + the capture; later rollouts are graph replays
    for rec in model.logger:
        assert all(math.isfinite(rec[k]) for k in ("loss", "policy_loss", "value_loss", "entropy_loss", "approx_kl"))
    curve = [r["ep_rew_mean"] for r in model.logger if math.isfinite(r["ep_rew_mean"])]
    assert curve[-1] > curve[0] + 10.0, (curve[0], curve[-1])
    assert len(cb.evaluations_timesteps) == 3 and (tmp_path / "best_model.zip").exists()
    path = model.save(tmp_path / "ckpt")
    again = RecurrentPPO.load(path, env=env)
    obs = torch.rand((16, 80), device=env.device)
    a1, _ = model.predict(obs, deterministic=True)
    a2, _ = again.predict(obs, deterministic=True)
    assert torch.equal(a1, a2)
    st = evaluate_policy(again, eval_env, n_eval_episodes=8, return_episode_stats=True)
    assert len(st["r"]) == 8 and (st["total_free"] == 144).all()


def _lstm_errors(got, ref):
    return [(got_t.detach().double() - ref_t.detach().double()).abs().max().item() for got_t, ref_t in zip(got, ref)]


def _check_fused_lstm(S, B, F, H, starts_of, gain=1.0, seed=0):
    """nav3d_lstm_forward / nav3d_lstm_backward against lstm_reference64 (float64) on y, h_last, c_last and the
    gradients of (y * wgt).sum() with respect to W_ih, W_hh, b_ih and b_hh (the kernel's db serves both biases).  wgt has
    whole zero timesteps, the last one included, so some dh_all slices are zero.

    The tolerance is a yardstick, not a constant: the error torch's own fp32 computation of the same function makes
    against float64 on the same inputs.  Without TF32 that is torch.nn.LSTM (cuDNN) run with cuts at the resets; with TF32
    it is lstm_reference64 run in fp32 with TF32 matmuls.  Each of the kernel's errors must be at most 4x the yardstick's
    plus a floor of 16 eps32 max|ref| (for quantities torch happens to get almost exactly right)."""
    from nav3d.train_ops import fused_lstm
    old = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    g = torch.Generator(device="cuda").manual_seed(seed * 1000 + S * 7 + B)
    k = gain / math.sqrt(H)
    p32 = [((torch.rand(shape, generator=g, device="cuda") * 2 - 1) * k).contiguous()
           for shape in ((4 * H, F), (4 * H, H), (4 * H,), (4 * H,))]
    x = torch.randn((S, B, F), generator=g, device="cuda")
    h0 = torch.randn((B, H), generator=g, device="cuda") * 0.5
    c0 = torch.randn((B, H), generator=g, device="cuda") * 0.5
    starts = starts_of(g, S, B)
    wgt = torch.randn((S, B, H), generator=g, device="cuda")
    if S > 1:
        wgt[1::3] = 0
        wgt[-1] = 0
    names = ("y", "h_last", "c_last", "dW_ih", "dW_hh", "db_ih", "db_hh")

    def run(fn, params, dtype, w=wgt):
        leaves = [p.detach().to(dtype).requires_grad_(True) for p in params]
        y, h, c = fn(leaves)
        (y * w.to(dtype)).sum().backward()
        return [y, h, c] + [p.grad for p in leaves]

    ref = run(lambda P: lstm_reference64(x.double(), *P, h0.double(), c0.double(), starts), p32, torch.float64)
    scale = [r.abs().max().item() for r in ref]
    try:
        torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
        lstm = torch.nn.LSTM(F, H).cuda()

        def cudnn(P):
            for dst, src in zip((lstm.weight_ih_l0, lstm.weight_hh_l0, lstm.bias_ih_l0, lstm.bias_hh_l0), P):
                dst.data.copy_(src.detach())
            y, h, c = lstm_with_cuts(lstm, x, h0, c0, starts)
            return y, h, c

        yard = run(cudnn, p32, torch.float32)
        yard = yard[:3] + [p.grad for p in lstm.parameters()]
        fused = run(lambda P: fused_lstm(x, *P, h0, c0, starts, tf32=False), p32, torch.float32)
        torch.backends.cuda.matmul.allow_tf32 = True
        # torch computes a product with one row as a matrix-vector product, which never uses TF32 (the kernel's cuBLAS
        # GEMMs do at any B).  The TF32 yardstick therefore runs the batch twice side by side, the copy with zero loss
        # weight: its products stay on the TF32 matrix path, and rows do not mix, so its outputs are those of the batch.
        two = lambda t, dim: torch.cat([t, t], dim=dim)

        def tf32_yardstick(P):
            y, h, c = lstm_reference64(two(x, 1), *P, two(h0, 0), two(c0, 0), two(starts, 1))
            return y, h[:B], c[:B]

        yard_tf = run(tf32_yardstick, p32, torch.float32, w=torch.cat([wgt, torch.zeros_like(wgt)], dim=1))
        yard_tf[0] = yard_tf[0][:, :B]
        fused_tf = run(lambda P: fused_lstm(x, *P, h0, c0, starts, tf32=True), p32, torch.float32)
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old
    for mode, got, yardstick in (("fp32", fused, yard), ("tf32", fused_tf, yard_tf)):
        e_got, e_yard = _lstm_errors(got, ref), _lstm_errors(yardstick, ref)
        floor = [16 * EPS32 * sc for sc in scale]
        # a quantity can be exactly 0 on every side (dW_hh when every h_in is 0)
        ratios = {n: eg / max(ey, fl) if max(ey, fl) > 0 else (0.0 if eg == 0 else math.inf)
                  for n, eg, ey, fl in zip(names, e_got, e_yard, floor)}
        print(f"fused_lstm {mode} S={S} B={B} F={F} H={H}: kernel / yardstick error " +
              " ".join(f"{n}={r:.2f}" for n, r in ratios.items()))
        for n, eg, ey, fl in zip(names, e_got, e_yard, floor):
            assert math.isfinite(eg) and eg <= 4 * ey + fl, (mode, n, eg, ey, fl)


@pytest.mark.parametrize("S,B,F,H,p_start", [(1, 3, 5, 8, 0.5), (9, 6, 7, 10, 0.3), (17, 33, 80, 64, 0.15), (128, 512, 80, 256, 0.01), (64, 700, 80, 256, 0.0),
                                             (1, 1, 1, 1, 0.0), (1, 1, 1, 1, 1.0), (2, 1, 3, 1, 0.5), (5, 7, 3, 257, 0.3),
                                             (1, 591, 8, 16, 0.0), (2, 296, 8, 16, 0.1), (593, 1, 4, 8, 0.05),
                                             (512, 64, 16, 64, 0.0), (9, 6, 7, 10, 1.0)])
def test_fused_lstm_matches_torch_lstm(S, B, F, H, p_start):
    """The fused LSTM, fp32 and TF32, forward and all four parameter gradients, against float64 (_check_fused_lstm).
    Shapes: H = 1 and S = 1; B*H not a multiple of 256 with 4H over five 256-column tiles (H = 257); S*B = 591, 592 and
    593 around column_sum_kernel's split into min(S*B, 592) row slabs; 512 steps with no reset (error carried through c);
    a reset at every step (p_start = 1); the trainer's (128, 512, 80, 256) and (64, 700, 80, 256)."""
    _check_fused_lstm(S, B, F, H, lambda g, S, B: (torch.rand((S, B), generator=g, device="cuda") < p_start).to(torch.uint8))


@pytest.mark.parametrize("case", ["starts_only_at_t0", "saturated_gates"])
def test_fused_lstm_special_inputs(case):
    """Episode starts for every env at t = 0 and nowhere else; gates driven into saturation by weights x 20."""
    if case == "starts_only_at_t0":
        def starts_of(g, S, B):
            s = torch.zeros((S, B), dtype=torch.uint8, device="cuda")
            s[0] = 1
            return s
        _check_fused_lstm(33, 40, 12, 48, starts_of)
    else:
        _check_fused_lstm(33, 40, 12, 48, lambda g, S, B: (torch.rand((S, B), generator=g, device="cuda") < 0.1).to(torch.uint8),
                          gain=20.0)


def test_policy_fused_and_cudnn_paths_agree():
    """RecurrentActorCritic.forward_sequence through the fused LSTM (default on CUDA) and through cuDNN with cuts, and with
    the critic branch on its own stream or not: same logits/values and the same gradients (TF32 off)."""
    from nav3d.policy import RecurrentActorCritic
    old = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    try:
        torch.manual_seed(0)
        pol = RecurrentActorCritic(net_arch=dict(pi=[256, 256, 128], vf=[256, 256, 128]), lstm_hidden_size=256).cuda()
        S, B = 32, 96
        obs = torch.rand((S, B, 80), device="cuda")
        starts = (torch.rand((S, B), device="cuda") < 0.05).to(torch.uint8)
        state = tuple(0.3 * torch.randn((1, B, 256), device="cuda") for _ in range(4))
        cuts = [0] + [t for t in range(1, S) if bool(starts[t].any())]
        results = []
        for fused, two in ((False, False), (True, False), (True, True), (False, True)):
            pol.fused_lstm, pol.two_streams = fused, two
            pol.zero_grad()
            logits, values, st = pol.forward_sequence(obs, state, starts, cuts)
            (logits.square().mean() + values.square().mean()).backward()
            torch.cuda.synchronize()
            results.append((logits.detach(), values.detach(), [s.detach() for s in st], [p.grad.clone() for p in pol.parameters()]))
        base = results[0]
        for r in results[1:]:
            assert torch.allclose(r[0], base[0], atol=1e-5) and torch.allclose(r[1], base[1], atol=1e-5)
            assert all(torch.allclose(a, b, atol=5e-5) for a, b in zip(r[2], base[2]))
            for a, b in zip(r[3], base[3]):
                assert (a - b).abs().max().item() <= 1e-4 * (b.abs().max().item() + 1e-6)
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old


def test_cuda_graph_rollout_equals_eager_rollout():
    """From the second rollout on, collect_rollouts replays ONE CUDA graph of the whole rollout; it must fill the buffers
    exactly like the eager loop (same Philox draws through the device-side step counter, same env steps, same GAE)."""
    from nav3d import BatchedCubicEnv
    from nav3d.ppo import RecurrentPPO
    from nav3d.rooms import load_room_file
    # 149- and 302-step episodes: resets and time limits fall inside every rollout after the first
    rooms = [load_room_file(ROOMS / "P3_training" / "maze_3d_tunnels.txt"), load_room_file(ROOMS / "P2_training" / "tightcorridor.txt")]
    models = []
    for graph in (False, True):
        env = BatchedCubicEnv(rooms=rooms, num_envs=192, local_map_length=10, seed=5)
        m = RecurrentPPO(env, policy_kwargs=dict(net_arch=dict(pi=[64, 64], vf=[64, 64]), lstm_hidden_size=64), n_steps=96,
                         batch_size=96 * 64, n_epochs=1, seed=3, cuda_graph=graph, graph_chunk=40)   # 3 graphs: 40 + 40 + 16 steps
        models.append(m)
    calls = [0, 0]

    class Count:
        def __init__(self, i): self.i = i
        def on_step(self, model):
            calls[self.i] += 1
            return True
    for r in range(4):
        for i, m in enumerate(models):
            assert m.collect_rollouts(Count(i))
        a, b = models
        assert (b._graph is not None) == (r >= 1) and a._graph is None and (r < 1 or len(b._graph) == 3)
        assert torch.equal(a._actions, b._actions) and torch.equal(a._obs, b._obs) and torch.equal(a._starts, b._starts)
        assert torch.allclose(a._rewards, b._rewards, atol=1e-5) and torch.allclose(a._values, b._values, atol=1e-5)
        assert torch.allclose(a._adv, b._adv, atol=1e-4) and torch.allclose(a._logp, b._logp, atol=1e-5)
        assert torch.allclose(a._chunk_states, b._chunk_states, atol=1e-5)
        assert a.num_timesteps == b.num_timesteps == (r + 1) * 96 * 192 and calls[0] == calls[1] == (r + 1) * 96
        assert a._episodes_this_rollout == b._episodes_this_rollout
        assert (math.isnan(a._ep_return_mean) and math.isnan(b._ep_return_mean)) or abs(a._ep_return_mean - b._ep_return_mean) < 1e-3
    assert int(a._starts.sum()) > 0 and a._episodes_this_rollout > 0
    # training between graph replays keeps working (the graph reads the parameters in place)
    b.train()
    assert b.collect_rollouts()


def test_cuda_graph_update_equals_eager_update():
    """Small minibatches (launch-bound) are replayed as ONE CUDA graph per minibatch (forward, backward, clip, Adam); after
    the same rollouts and the same shuffles the parameters must agree with the eager update."""
    from nav3d import BatchedCubicEnv
    from nav3d.ppo import RecurrentPPO
    from nav3d.rooms import load_room_file
    old = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    rooms = [load_room_file(ROOMS / "P3_training" / "maze_3d_tunnels.txt")]
    try:
        models = []
        for graph in (False, True):
            env = BatchedCubicEnv(rooms=rooms, num_envs=8, local_map_length=10, seed=5)
            m = RecurrentPPO(env, policy_kwargs=dict(net_arch=dict(pi=[64, 64], vf=[64, 64]), lstm_hidden_size=64), n_steps=64,
                             batch_size=32, n_epochs=2, ent_coef=0.01, seed=3, cuda_graph=graph, allow_tf32=False)
            models.append(m)
        torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
        a, b = models
        # two iterations: the first holds the eager warm-up minibatches, the capture and replays, the second replays only.
        # (Adam turns rounding-level gradient differences into lr-sized steps, so longer runs drift apart legitimately.)
        for it in range(2):
            for m in models:
                m.collect_rollouts()
            assert torch.equal(a._actions, b._actions), it            # same policy so far -> same rollout
            sa, sb = a.train(), b.train()
            assert sa["minibatches"] == sb["minibatches"] == 2 * (64 * 8 // 32)
            pa = torch.cat([p.detach().flatten() for p in a.policy.parameters()])
            pb = torch.cat([p.detach().flatten() for p in b.policy.parameters()])
            rel = float((pa - pb).norm() / pa.norm())
            assert rel < 5e-4, (it, rel)
            for k in ("policy_loss", "value_loss", "entropy_loss", "approx_kl"):
                assert abs(sa[k] - sb[k]) <= 1e-3 * (1.0 + abs(sa[k])), (k, sa[k], sb[k])
        assert b._upd_graph is not None and a._upd_graph is None
        # the optimizer state of a graph-trained model survives a checkpoint round trip
        import tempfile
        with tempfile.TemporaryDirectory() as d:
            path = b.save(d + "/m")
            c = RecurrentPPO.load(path, env=BatchedCubicEnv(rooms=rooms, num_envs=8, local_map_length=10, seed=5))
            c.collect_rollouts(); c.train()
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old


def test_cuda_graph_update_masks_episode_starts_inside_a_chunk():
    """ADVICE r1 (high): episodes that end in the middle of a sequence chunk.  A 5x6x5 room has 36 free cells, so every
    episode is truncated after 36 steps and each 64-step chunk holds one or two resets; the replayed (graph) update
    must zero the LSTM state there exactly like the eager update: same losses, same parameters."""
    import numpy as np
    from edge_rooms import rooms_from_grids
    from nav3d import BatchedCubicEnv
    from nav3d.ppo import RecurrentPPO
    g = np.zeros((5, 6, 5), dtype=np.int8)
    g[0], g[-1], g[:, 0], g[:, -1], g[:, :, 0], g[:, :, -1] = -2, -2, -2, -2, -2, -2
    rooms = rooms_from_grids([g])
    old = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    try:
        torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
        models = []
        for graph in (False, True):
            env = BatchedCubicEnv(rooms=rooms, num_envs=8, local_map_length=10, seed=5)
            models.append(RecurrentPPO(env, policy_kwargs=dict(net_arch=dict(pi=[64, 64], vf=[64, 64]), lstm_hidden_size=64),
                                       n_steps=64, batch_size=64, n_epochs=2, ent_coef=0.01, seed=3, cuda_graph=graph,
                                       allow_tf32=False))
        a, b = models
        for it in range(2):
            for m in models:
                m.collect_rollouts()
            assert torch.equal(a._actions, b._actions), it
            starts = a._starts.view(64, 8)
            assert int(starts[1:].sum()) >= 8                      # resets strictly inside the chunks
            sa, sb = a.train(), b.train()
            pa = torch.cat([p.detach().flatten() for p in a.policy.parameters()])
            pb = torch.cat([p.detach().flatten() for p in b.policy.parameters()])
            rel = float((pa - pb).norm() / pa.norm())
            assert rel < 5e-4, (it, rel)
            for k in ("policy_loss", "value_loss", "entropy_loss", "approx_kl"):
                assert abs(sa[k] - sb[k]) <= 1e-3 * (1.0 + abs(sa[k])), (k, sa[k], sb[k])
        assert b._upd_graph is not None and a._upd_graph is None
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old

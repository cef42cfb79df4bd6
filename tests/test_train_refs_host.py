"""CPU checks of the float64 references in tests/train_refs.py that the GPU tests hold the trainer's kernels to: the numpy
Philox port against the C oracle and the Random123 known answers, the pinned policy-stream counters the sampling edge
tests rely on, the LSTM restatement against torch.nn.LSTM, and the GAE reference and its error bound."""
import numpy as np
import pytest
import torch

from train_refs import (EPS32, POLICY_STREAM, U_ONE_COUNTERS, U_ZERO_COUNTERS, gae_reference, gae_reference64,
                        lstm_reference64, lstm_with_cuts, philox4x32_10_np, policy_word0, sample_reference64)


def test_philox_port_known_answers():
    """Random123's kat_vectors for philox4x32_10."""
    kat = [((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
           ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
           ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
            (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1))]
    for ctr, key, want in kat:
        assert tuple(int(w) for w in philox4x32_10_np(*ctr, *key)) == want


def test_philox_port_matches_oracle(oracle):
    rng = np.random.default_rng(5)
    ctr = rng.integers(0, 2 ** 32, size=(64, 4), dtype=np.uint64)
    key = rng.integers(0, 2 ** 32, size=(64, 2), dtype=np.uint64)
    for c, k in zip(ctr, key):
        got = np.array([int(w) for w in philox4x32_10_np(*c, *k)], dtype=np.uint32)
        assert np.array_equal(got, oracle.philox4x32_10(c.astype(np.uint32), k.astype(np.uint32))), (c, k)
    # vectorized over counters = element by element
    ids = rng.integers(0, 2 ** 32, size=100, dtype=np.uint64)
    words = philox4x32_10_np(ids, 77, 0, POLICY_STREAM, 1234, 9)
    for i in (0, 17, 99):
        assert [int(w[i]) for w in words] == list(oracle.philox4x32_10([int(ids[i]), 77, 0, POLICY_STREAM], [1234, 9]))


@pytest.mark.parametrize("env,step,word", U_ONE_COUNTERS + U_ZERO_COUNTERS)
def test_pinned_policy_counters(oracle, env, step, word):
    assert int(policy_word0(1234, [env], step)[0]) == word
    assert int(oracle.philox4x32_10([env, step, 0, POLICY_STREAM], [1234, 0])[0]) == word
    ref = sample_reference64(np.array([[0.0, -np.inf, 0.0]], dtype=np.float32), 1234, env, step)
    assert ref.u[0] == (word >> 8) * 2.0 ** -24
    assert ref.action[0] == (2 if word >= 0xFFFFFF80 else 0)


def test_sample_reference_counter_wraps():
    """env_id0 + i and step + step_offset are taken mod 2^32."""
    lg = np.zeros((300, 4), dtype=np.float32)
    a = sample_reference64(lg, 7, 2 ** 32 - 100, 2 ** 32 - 3, 5)
    b = sample_reference64(lg, 7, 2 ** 32 - 100, 2)
    assert np.array_equal(a.u, b.u)
    ids = (2 ** 32 - 100 + np.arange(300)) % 2 ** 32
    assert np.array_equal(a.word0, policy_word0(7, ids, 2))


def test_sample_reference_masks_and_entropy():
    lg = np.array([[-np.inf, 1.0, 2.0, -np.inf], [0.0, -200.0, -np.inf, -np.inf], [3.0, 3.0, 3.0, 3.0]], dtype=np.float32)
    r = sample_reference64(lg, 1, 0, 0)
    assert np.all(np.isfinite(r.entropy)) and np.all(np.isfinite(r.log_prob))
    p = np.exp(np.array([1.0, 2.0]) - np.logaddexp(1.0, 2.0))
    assert r.entropy[0] == pytest.approx(-(p * np.log(p)).sum(), rel=1e-14)
    assert r.entropy[2] == pytest.approx(np.log(4.0), rel=1e-14)
    assert r.action[0] in (1, 2) and r.action[1] == 0
    assert r.greedy.tolist() == [2, 0, 0]
    # the fp32 bounds: of the order of eps32, larger for wide rows
    assert np.all(r.cdf_bound[:, -1] < 16 * EPS32)
    wide = sample_reference64(np.zeros((1, 1024), dtype=np.float32), 1, 0, 0)
    assert wide.cdf_bound[0, -1] > 512 * EPS32


def test_lstm_reference_matches_torch_lstm_float64():
    """The restatement against torch.nn.LSTM in float64 on the CPU, run in pieces cut at the resets."""
    torch.manual_seed(0)
    S, B, F, H = 11, 5, 3, 7
    lstm = torch.nn.LSTM(F, H).double()
    x = torch.randn(S, B, F, dtype=torch.float64)
    h0, c0 = torch.randn(B, H, dtype=torch.float64), torch.randn(B, H, dtype=torch.float64)
    starts = (torch.rand(S, B) < 0.3).to(torch.uint8)
    starts[0, 0], starts[4] = 1, 1
    wgt = torch.randn(S, B, H, dtype=torch.float64)
    y, h, c = lstm_with_cuts(lstm, x, h0, c0, starts)
    (y * wgt).sum().backward()
    want = [p.grad.clone() for p in lstm.parameters()]
    params = [p.detach().clone().requires_grad_(True) for p in lstm.parameters()]
    y2, h2, c2 = lstm_reference64(x, *params, h0, c0, starts)
    (y2 * wgt).sum().backward()
    for a, b in ((y2, y), (h2, h), (c2, c)):
        assert (a - b).abs().max().item() < 1e-12
    for p, g in zip(params, want):
        assert (p.grad - g).abs().max().item() < 1e-12


@pytest.mark.parametrize("T,N,gamma,lam,p_start", [(1, 7, 0.99, 0.95, 0.1), (64, 257, 0.99, 0.95, 0.05),
                                                   (512, 16, 1.0, 1.0, 0.0), (33, 9, 0.0, 0.95, 0.5)])
def test_gae_reference64_and_its_bound(T, N, gamma, lam, p_start):
    """The float64 GAE agrees with the fp32 restatement, and the fp32 restatement's error lies inside the bound."""
    g = torch.Generator().manual_seed(T + N)
    r, v = torch.randn((T, N), generator=g), torch.randn((T, N), generator=g)
    s = (torch.rand((T, N), generator=g) < p_start).to(torch.uint8)
    lv = torch.randn(N, generator=g)
    ld = (torch.rand(N, generator=g) < 0.3).to(torch.uint8)
    gamma32, lam32 = float(np.float32(gamma)), float(np.float32(lam))
    a32, r32 = gae_reference(r, v, s, lv, ld, gamma32, lam32)
    adv, ret, ab, rb = gae_reference64(r, v, s, lv, ld, gamma, lam)
    assert np.all(np.abs(a32.double().numpy() - adv) <= ab)
    assert np.all(np.abs(r32.double().numpy() - ret) <= rb)
    # one step written out by hand
    t, n = T - 1, N - 1
    nnt = 1.0 - float(ld[n])
    want = float(r[t, n]) + gamma32 * float(lv[n]) * nnt - float(v[t, n])
    if T > 1:
        nnt = 1.0 - float(s[t, n])
        want_prev = float(r[t - 1, n]) + gamma32 * float(v[t, n]) * nnt - float(v[t - 1, n]) + gamma32 * lam32 * nnt * want
        assert adv[t - 1, n] == pytest.approx(want_prev, rel=1e-14, abs=1e-14)
    assert adv[t, n] == pytest.approx(want, rel=1e-14, abs=1e-14) and ret[t, n] == pytest.approx(want + float(v[t, n]), rel=1e-14)
    # the bound is tight enough to mean something: within 1e4 eps32 of the advantages' scale at these lengths
    assert ab.max() < 1e4 * EPS32 * (np.abs(adv).max() + 1.0)

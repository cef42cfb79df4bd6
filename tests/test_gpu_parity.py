"""Parity tests proper: the CUDA path (through the C ABI) against the CPU oracle and the reference's golden traces.
Integer state, flags, observations (f32), rewards (f64 and f32) and the per-episode return (the documented 1/100-unit
rule, restated by the oracle) are compared BIT-EXACTLY; the return is also held to the documented bound against the f64
sum of the rewards (tests/lockstep.py)."""
import numpy as np
import pytest

from conftest import ROOMS
from lockstep import compare_grids, compare_step, replay_golden_trace
from nav3d.rooms import load_room_dir, load_room_file

pytestmark = pytest.mark.gpu


def lockstep(oracle, rooms, n, L, steps, seed, lanes, auto_reset=True, crash=-2.0, state_every=10, env_id0=0):
    import torch
    from gpu_harness import GpuEngine
    orooms = [oracle.OracleRoom(r.grid, -2) for r in rooms]
    ov = oracle.OracleVec(n, orooms, L, crash, seed, env_id0, auto_reset)
    oracle.set_threads(oracle.hw_threads())
    g = GpuEngine(n, rooms, L, crash, seed, env_id0, auto_reset, lanes)
    for i, r in enumerate(orooms):
        assert g.n_free(i) == r.n_free
    o0 = ov.reset()
    g0 = g.reset()
    assert np.array_equal(g0.view(np.uint32), o0.view(np.uint32)), "reset observations"
    assert np.array_equal(g.state()[:, :15].astype(np.int64), ov.state()), "reset state"
    rng = np.random.default_rng(seed + 1)
    n_done = 0
    for t in range(steps):
        a = rng.integers(0, 6, size=n)
        ov.step(a)
        g.step(a)
        st = g.state() if (t % state_every == 0 or t == steps - 1) else None
        compare_step(f"gpu lanes={lanes}", t, ov, g.obs, g.reward, g.reward64, g.term, g.trunc, g.tobs, g.eps, st, crash)
        n_done += int((ov.terminated | ov.truncated).sum())
    compare_grids(f"gpu lanes={lanes}", ov, g.grid, range(0, n, max(1, n // 16)))
    torch.cuda.synchronize()
    return n_done


@pytest.mark.parametrize("lanes", [1, 2, 4, 8, 16, 32])
def test_small_lockstep_all_lane_widths(oracle, lanes):
    rooms = load_room_dir(ROOMS / "P1_training", sort=True)
    n_done = lockstep(oracle, rooms, n=200, L=10, steps=1100, seed=3, lanes=lanes, state_every=25)
    assert n_done > 0


def test_config2_4096_envs_p1_training(oracle):
    """BASELINE.json configs[1]: 4096 envs over all P1_training rooms, L=10, random actions, auto-reset."""
    rooms = load_room_dir(ROOMS / "P1_training", sort=True)
    n_done = lockstep(oracle, rooms, n=4096, L=10, steps=1050, seed=42, lanes=0, state_every=50)
    assert n_done >= 500       # every env in the 12x12x12 room truncates at step 1000


def test_config3_heterogeneous_p2_p3(oracle):
    """BASELINE.json configs[2] (sampled): P2_training + P3_training rooms, per-env room index, incl. kitchen2 / open mazes."""
    rooms = load_room_dir(ROOMS / "P2_training", sort=True) + load_room_dir(ROOMS / "P3_training", sort=True)
    names = [r.name for r in rooms]
    assert "kitchen2.txt" in names and "maze_7x7_seed22.txt" in names and len(rooms) == 42
    n_done = lockstep(oracle, rooms, n=4096, L=10, steps=400, seed=7, lanes=0, state_every=40)
    assert n_done > 0


@pytest.mark.parametrize("L,lanes", [(1, 8), (4, 32), (15, 4), (40, 4), (31, 2), (32, 1)])
def test_ray_lengths_and_crash_penalty(oracle, L, lanes):
    rooms = [load_room_file(ROOMS / "P3_training" / "maze_7x7_seed22.txt"), load_room_file(ROOMS / "P3_training" / "kitchen2.txt"),
             load_room_file(ROOMS / "P2_training" / "small_bedroom.txt"), load_room_file(ROOMS / "P3_training" / "maze_3d_tunnels.txt")]
    lockstep(oracle, rooms, n=256, L=L, steps=400, seed=L, lanes=lanes, crash=-0.5)


def test_no_autoreset_steps_past_done(oracle):
    rooms = [load_room_file(ROOMS / "P3_training" / "maze_3d_tunnels.txt")]
    lockstep(oracle, rooms, n=64, L=10, steps=400, seed=5, lanes=8, auto_reset=False)


@pytest.mark.parametrize("lanes", [8, 32])
def test_reference_golden_traces(cubic_traces, lanes):
    """Every trace captured from the unmodified reference (tests/golden/cubic_traces.npz), incl. the termination branch."""
    from gpu_harness import GpuEngine
    sel = cubic_traces if lanes == 8 else cubic_traces[:4] + cubic_traces[-3:]
    for c in sel:
        room = load_room_file(ROOMS / c["room"])
        replay_golden_trace(c, room, lambda rooms, L, crash, ar: GpuEngine(1, rooms, L, crash, 0, 0, ar, lanes))


def test_sharding_independence(oracle):
    """Results do not depend on how envs are split over engines (one engine per GPU in production)."""
    import torch
    from gpu_harness import GpuEngine
    rooms = load_room_dir(ROOMS / "P1_training", sort=True)
    n, steps = 512, 300
    whole = GpuEngine(n, rooms, 10, seed=9)
    halves = [GpuEngine(n // 2, rooms, 10, seed=9, env_id0=0), GpuEngine(n // 2, rooms, 10, seed=9, env_id0=n // 2)]
    o = whole.reset()
    oh = np.concatenate([h.reset() for h in halves])
    assert np.array_equal(o.view(np.uint32), oh.view(np.uint32))
    rng = np.random.default_rng(0)
    for t in range(steps):
        a = rng.integers(0, 6, size=n)
        whole.step(a)
        for i, h in enumerate(halves):
            h.step(a[i * n // 2:(i + 1) * n // 2])
        assert np.array_equal(whole.obs.view(np.uint32), np.concatenate([h.obs for h in halves]).view(np.uint32))
        assert np.array_equal(whole.reward64, np.concatenate([h.reward64 for h in halves]))
    assert np.array_equal(whole.state()[:, :14], np.concatenate([h.state() for h in halves])[:, :14])


@pytest.mark.parametrize("n,T", [(1024, 1100), (1013, 550)])
def test_fused_random_rollout_matches_oracle(oracle, n, T):
    """nav3d_rollout_random with every observation, reward, done flag and action written: each of the T steps equals the
    oracle's, auto-resets included (1013 envs: the last warp of the thread-per-env kernel is ragged)."""
    import torch
    from nav3d import Engine
    rooms = load_room_dir(ROOMS / "P1_training", sort=True)
    seed = 17
    orooms = [oracle.OracleRoom(r.grid, -2) for r in rooms]
    ov = oracle.OracleVec(n, orooms, 10, -2.0, seed, 100, True)
    oracle.set_threads(oracle.hw_threads())
    ov.reset()
    eng = Engine(n, rooms, local_map_length=10, seed=seed, env_id0=100)
    eng.reset()
    chunk = 275
    for t0 in range(0, T, chunk):
        obs = torch.zeros((chunk, n, 80), dtype=torch.float32, device=eng.device)
        rew = torch.zeros((chunk, n), dtype=torch.float32, device=eng.device)
        done = torch.zeros((chunk, n), dtype=torch.uint8, device=eng.device)
        acts = torch.zeros((chunk, n), dtype=torch.uint8, device=eng.device)
        eng.rollout_random(chunk, t0, obs=obs, reward=rew, done=done, actions_out=acts)
        obs, rew, done, acts = obs.cpu().numpy(), rew.cpu().numpy(), done.cpu().numpy(), acts.cpu().numpy()
        for t in range(chunk):
            a = np.array([oracle.action(seed, 100 + i, t0 + t) for i in range(n)]) if t < 2 else acts[t].astype(np.int64)
            assert np.array_equal(a, acts[t])
            ov.step(a)
            assert np.array_equal(obs[t].view(np.uint32), ov.obs.view(np.uint32)), f"rollout obs t={t0 + t}"
            assert np.array_equal(rew[t], ov.reward.astype(np.float32)), f"rollout reward t={t0 + t}"
            assert np.array_equal(done[t], ov.terminated | ov.truncated), f"rollout done t={t0 + t}"
    assert np.array_equal(eng.get_state().cpu().numpy()[:, :15].astype(np.int64), ov.state())
    # the action stream itself: compare every action of a few steps with the oracle's Philox restatement
    for t in (0, 1, 500):
        ref = np.array([oracle.action(seed, 100 + i, t) for i in range(0, n, 37)])
        assert ref.min() >= 0 and ref.max() <= 5


def test_step_host_matches_device_path(oracle):
    import torch
    from nav3d import Engine
    rooms = load_room_dir(ROOMS / "P1_training", sort=True)
    n = 333
    a_eng = Engine(n, rooms, local_map_length=10, seed=4)
    b_eng = Engine(n, rooms, local_map_length=10, seed=4)
    dev = a_eng.device
    obs_d = a_eng.reset()
    b_eng.reset()
    rew_d = torch.zeros(n, device=dev); te_d = torch.zeros(n, dtype=torch.uint8, device=dev); tr_d = torch.zeros(n, dtype=torch.uint8, device=dev)
    obs_h = torch.zeros((n, 80)).pin_memory(); rew_h = torch.zeros(n).pin_memory()
    te_h = torch.zeros(n, dtype=torch.uint8).pin_memory(); tr_h = torch.zeros(n, dtype=torch.uint8).pin_memory()
    g = torch.Generator().manual_seed(0)
    for t in range(1100):
        a = torch.randint(0, 6, (n,), generator=g, dtype=torch.int64)
        a_eng.step(a.to(dev), obs_d, rew_d, te_d, tr_d)
        b_eng.step_host(a.pin_memory(), obs_h, rew_h, te_h, tr_h)
        assert torch.equal(obs_d.cpu(), obs_h) and torch.equal(rew_d.cpu(), rew_h)
        assert torch.equal(te_d.cpu(), te_h) and torch.equal(tr_d.cpu(), tr_h)


def test_full_size_sample_against_oracle(oracle):
    """BASELINE.json configs[3] size: 2^20 envs on one GPU, fused random rollout; a strided sample of 512 envs is
    replayed by the oracle (same global env ids, same Philox streams) and compared bit-exactly, and size-independent
    invariants are checked on all envs."""
    import torch
    from nav3d import Engine
    rooms = load_room_dir(ROOMS / "P1_training", sort=True)
    n, T, seed = 1 << 20, 48, 23
    eng = Engine(n, rooms, local_map_length=10, seed=seed)
    obs = eng.reset()
    ids = np.arange(0, n, n // 512, dtype=np.uint32)
    orooms = [oracle.OracleRoom(r.grid, -2) for r in rooms]
    ov = oracle.OracleVec(len(ids), orooms, 10, -2.0, seed, 0, True)
    ov.set_ids(ids)
    o0 = ov.reset()
    tid = torch.as_tensor(ids.astype(np.int64), device=eng.device)
    assert np.array_equal(obs[tid].cpu().numpy().view(np.uint32), o0.view(np.uint32))
    rew = torch.zeros((T, n), dtype=torch.float32, device=eng.device)
    done = torch.zeros((T, n), dtype=torch.uint8, device=eng.device)
    eng.rollout_random(T, 0, obs_last=obs, reward=rew, done=done)
    rsum = np.zeros(len(ids))
    for t in range(T):
        a = np.array([oracle.action(seed, int(i), t) for i in ids])
        ov.step(a)
        assert np.array_equal(rew[t][tid].cpu().numpy(), ov.reward.astype(np.float32)), f"t={t}"
    assert np.array_equal(obs[tid].cpu().numpy().view(np.uint32), ov.obs.view(np.uint32))
    st = eng.get_state()
    assert np.array_equal(st[tid].cpu().numpy()[:, :15].astype(np.int64), ov.state())
    # invariants over all 2^20 envs
    assert bool(((obs >= 0) & (obs <= 1)).all())
    assert bool((obs[:, 64:68].sum(dim=1) == 1).all()) and bool((obs[:, 73:] == 0).all())
    free = torch.as_tensor(eng.room_free, device=eng.device)[st[:, 13].long()]
    assert bool((st[:, 4] <= free).all()) and bool((st[:, 6] == T).all()) and bool((st[:, 4] >= 1).all())
    assert torch.allclose(obs[:, 72], st[:, 4].float() / free.float(), rtol=0, atol=1e-7)


def test_fused_full_observation_rollout_full_size(oracle):
    """What bench.py reports as extra.fused_rollout_full: nav3d_rollout_random at 2^20 envs, T = 32, ALL observations
    written ([32, 2^20, 80] f32).  Two launches back to back; a strided sample of 512 envs is replayed by the oracle and
    every one of the 64 steps compared (observation bits, f32 reward, done), then the final state."""
    import torch
    from nav3d import Engine
    rooms = load_room_dir(ROOMS / "P1_training", sort=True)
    n, T, seed = 1 << 20, 32, 77
    eng = Engine(n, rooms, local_map_length=10, seed=seed)
    eng.reset()
    ids = np.arange(11, n, n // 512, dtype=np.uint32)
    orooms = [oracle.OracleRoom(r.grid, -2) for r in rooms]
    ov = oracle.OracleVec(len(ids), orooms, 10, -2.0, seed, 0, True)
    ov.set_ids(ids)
    ov.reset()
    tid = torch.as_tensor(ids.astype(np.int64), device=eng.device)
    obs = torch.zeros((T, n, 80), dtype=torch.float32, device=eng.device)
    rew = torch.zeros((T, n), dtype=torch.float32, device=eng.device)
    done = torch.zeros((T, n), dtype=torch.uint8, device=eng.device)
    for launch in range(2):
        eng.rollout_random(T, launch * T, obs=obs, reward=rew, done=done)
        o, r, d = obs[:, tid].cpu().numpy(), rew[:, tid].cpu().numpy(), done[:, tid].cpu().numpy()
        for t in range(T):
            ov.step(np.array([oracle.action(seed, int(i), launch * T + t) for i in ids]))
            assert np.array_equal(o[t].view(np.uint32), ov.obs.view(np.uint32)), f"obs launch {launch} t={t}"
            assert np.array_equal(r[t], ov.reward.astype(np.float32)) and np.array_equal(d[t], ov.terminated | ov.truncated)
        assert bool(((obs >= 0) & (obs <= 1)).all()) and bool((obs[:, :, 73:] == 0).all())
    assert np.array_equal(eng.get_state()[tid].cpu().numpy()[:, :15].astype(np.int64), ov.state())


def test_config3_full_size_sample_against_oracle(oracle):
    """BASELINE.json configs[2] at its full size: 65 536 envs over the 42 P2+P3 training rooms (heterogeneous sizes, per-env
    room index), stepped one launch per step with host-chosen random actions; a strided sample of 512 envs is replayed by
    the oracle under the same global env ids and compared bit-exactly every step; invariants over all envs."""
    import torch
    from nav3d import Engine
    rooms = load_room_dir(ROOMS / "P2_training", sort=True) + load_room_dir(ROOMS / "P3_training", sort=True)
    n, T, seed = 65536, 320, 31
    eng = Engine(n, rooms, local_map_length=10, seed=seed)
    dev = eng.device
    obs = eng.reset()
    ids = np.arange(0, n, n // 512, dtype=np.uint32)
    orooms = [oracle.OracleRoom(r.grid, -2) for r in rooms]
    ov = oracle.OracleVec(len(ids), orooms, 10, -2.0, seed, 0, True)
    ov.set_ids(ids)
    tid = torch.as_tensor(ids.astype(np.int64), device=dev)
    assert np.array_equal(obs[tid].cpu().numpy().view(np.uint32), ov.reset().view(np.uint32))
    rew = torch.zeros(n, device=dev); rew64 = torch.zeros(n, dtype=torch.float64, device=dev)
    te = torch.zeros(n, dtype=torch.uint8, device=dev); tr = torch.zeros(n, dtype=torch.uint8, device=dev)
    rng = np.random.default_rng(seed)
    n_done = 0
    for t in range(T):
        a = rng.integers(0, 6, size=n)
        eng.step(torch.as_tensor(a, device=dev), obs, rew, te, tr, reward64=rew64)
        ov.step(a[ids])
        assert np.array_equal(obs[tid].cpu().numpy().view(np.uint32), ov.obs.view(np.uint32)), f"obs t={t}"
        assert np.array_equal(rew64[tid].cpu().numpy(), ov.reward), f"reward t={t}"
        assert np.array_equal(te[tid].cpu().numpy(), ov.terminated) and np.array_equal(tr[tid].cpu().numpy(), ov.truncated)
        n_done += int((ov.terminated | ov.truncated).sum())
    assert n_done > 0                                       # maze_3d_tunnels (149 steps) and tightcorridor (302) end inside
    st = eng.get_state()
    assert np.array_equal(st[tid].cpu().numpy()[:, :15].astype(np.int64), ov.state())
    rooms_used = torch.unique(st[:, 13]).numel()
    assert rooms_used == 42
    free = torch.as_tensor(eng.room_free, device=dev)[st[:, 13].long()]
    assert bool(((obs >= 0) & (obs <= 1)).all()) and bool((obs[:, 64:68].sum(dim=1) == 1).all()) and bool((obs[:, 73:] == 0).all())
    assert bool((st[:, 4] <= free).all()) and bool((st[:, 4] >= 1).all()) and bool((st[:, 6] <= T).all())
    assert torch.allclose(obs[:, 72], st[:, 4].float() / free.float(), rtol=0, atol=1e-7)


@pytest.mark.parametrize("lanes", [1, 4])
def test_kernel_variants(oracle, lanes):
    """Both step kernels — one thread per env (step_tpe_kernel) and G lanes per env (step_call_kernel<G>) — must give the
    same bits, auto-reset (an out-of-line device call at the end of the step) included."""
    rooms = [load_room_file(ROOMS / "P3_training" / "maze_3d_tunnels.txt"), load_room_file(ROOMS / "P2_training" / "tightcorridor.txt"),
             load_room_file(ROOMS / "P1_training" / "Empty_room_3mx3mx3m_0.25m_cellsize.txt")]
    n_done = lockstep(oracle, rooms, n=1500, L=10, steps=650, seed=21, lanes=lanes, state_every=50)
    assert n_done > 1500


def test_benched_path_full_size_with_truncation_wave(oracle):
    """The exact thing bench.py times: nav3d_step (default lanes, programmatic dependent launch on) at 2^20 envs on
    P1_training, 1 100 steps, so that the synchronous truncation wave of the 12x12x12 room at step 1 000 and the auto-resets
    run at full size.  512 strided envs are replayed by the oracle EVERY step (observation, f64 reward, flags), invariants
    are checked over all envs at intervals and at the end."""
    import torch
    from nav3d import Engine
    rooms = load_room_dir(ROOMS / "P1_training", sort=True)
    n, T, seed = 1 << 20, 1100, 2024
    eng = Engine(n, rooms, local_map_length=10, seed=seed)
    dev = eng.device
    obs = eng.reset()
    ids = np.arange(7, n, n // 512, dtype=np.uint32)
    orooms = [oracle.OracleRoom(r.grid, -2) for r in rooms]
    ov = oracle.OracleVec(len(ids), orooms, 10, -2.0, seed, 0, True)
    ov.set_ids(ids)
    tid = torch.as_tensor(ids.astype(np.int64), device=dev)
    assert np.array_equal(obs[tid].cpu().numpy().view(np.uint32), ov.reset().view(np.uint32))
    rew = torch.zeros(n, device=dev); rew64 = torch.zeros(n, dtype=torch.float64, device=dev)
    te = torch.zeros(n, dtype=torch.uint8, device=dev); tr = torch.zeros(n, dtype=torch.uint8, device=dev)
    tobs = torch.zeros((n, 80), device=dev)
    g = torch.Generator(device=dev).manual_seed(5)
    free_t = torch.as_tensor(eng.room_free, device=dev)
    n_done = n_done_all = 0
    for t in range(T):
        a = torch.randint(0, 6, (n,), generator=g, device=dev, dtype=torch.int64)
        eng.step(a, obs, rew, te, tr, reward64=rew64, terminal_obs=tobs)
        ov.step(a[tid].cpu().numpy())
        assert np.array_equal(obs[tid].cpu().numpy().view(np.uint32), ov.obs.view(np.uint32)), f"obs t={t}"
        assert np.array_equal(rew64[tid].cpu().numpy(), ov.reward), f"reward t={t}"
        assert np.array_equal(te[tid].cpu().numpy(), ov.terminated) and np.array_equal(tr[tid].cpu().numpy(), ov.truncated), f"flags t={t}"
        d = (ov.terminated | ov.truncated).astype(bool)
        if d.any():
            assert np.array_equal(tobs[tid].cpu().numpy()[d].view(np.uint32), ov.terminal_obs[d].view(np.uint32)), f"terminal obs t={t}"
        n_done += int(d.sum())
        if t in (998, 999, 1000) or t % 275 == 0 or t == T - 1:
            st = eng.get_state()
            free = free_t[st[:, 13].long()]
            n_done_all += int((te | tr).sum())
            assert bool(((obs >= 0) & (obs <= 1)).all()) and bool((obs[:, 64:68].sum(dim=1) == 1).all()) and bool((obs[:, 73:] == 0).all())
            assert bool((st[:, 4] <= free).all()) and bool((st[:, 4] >= 1).all()) and bool((st[:, 6] < free).all())
            assert torch.allclose(obs[:, 72], st[:, 4].float() / free.float(), rtol=0, atol=1e-7)
    assert n_done > 50 and n_done_all > 100000          # a fifth of the envs play the 1 000-step room: they all end at step 1 000
    st = eng.get_state()
    assert np.array_equal(st[tid].cpu().numpy()[:, :15].astype(np.int64), ov.state())
    for j in (0, 100, 511):
        assert np.array_equal(eng.get_grid(int(ids[j])), np.minimum(ov.grid(j), 255).astype(np.int16))


@pytest.mark.parametrize("lanes", [1, 4, 32])
def test_engine_limits_and_degenerate_rooms(oracle, lanes):
    """64x64x16 rooms (bit 63 / bit 15 of the packed words, open boundary faces), single-cell / corridor / slab rooms,
    wall-less rooms, and visit counters past the u8 range."""
    from edge_rooms import degenerate_rooms, max_size_rooms, thin_open_rooms
    lockstep(oracle, max_size_rooms(), n=300, L=15, steps=500, seed=2, lanes=lanes, state_every=25)
    assert lockstep(oracle, degenerate_rooms(), n=400, L=10, steps=300, seed=4, lanes=lanes) > 0
    assert lockstep(oracle, thin_open_rooms(), n=300, L=4, steps=200, seed=6, lanes=lanes) > 0
    lockstep(oracle, degenerate_rooms()[3:], n=64, L=10, steps=400, seed=8, lanes=lanes, auto_reset=False)


@pytest.mark.parametrize("lanes", [1, 4, 16])
def test_partial_reset_of_listed_envs(oracle, lanes):
    """nav3d_reset with env_ids + injected picks (the manual gym-style reset of SOME envs, auto_reset off): the listed envs
    restart exactly like the reference's reset with those (room, start) draws, every other env is untouched, and all keep
    stepping in lock-step with one scalar oracle per env."""
    from gpu_harness import GpuEngine
    rooms = [load_room_file(ROOMS / "P3_training" / "maze_7x7_seed22.txt"), load_room_file(ROOMS / "P2_training" / "tightcorridor.txt"),
             load_room_file(ROOMS / "P3_training" / "kitchen2.txt")]
    orooms = [oracle.OracleRoom(r.grid, -2) for r in rooms]
    n, L = 48, 10
    rng = np.random.default_rng(9)
    g = GpuEngine(n, rooms, L, -2.0, 1, 0, False, lanes)
    envs = [oracle.OracleCubic(L, -2.0) for _ in range(n)]

    def draw(k):
        r = rng.integers(0, len(rooms), size=k)
        return np.stack([r, np.array([rng.integers(0, orooms[i].n_free) for i in r])], axis=1).astype(np.int32)

    picks = draw(n)
    obs = g.reset(picks=picks)
    for i in range(n):
        o = envs[i].reset(orooms[picks[i, 0]], orooms[picks[i, 0]].free_cell(picks[i, 1]))
        assert np.array_equal(obs[i].view(np.uint32), o.view(np.uint32))

    def lockstep_steps(k):
        for _ in range(k):
            a = rng.integers(0, 6, size=n)
            g.step(a)
            for i in range(n):
                o, r, te, tr = envs[i].step(int(a[i]))
                assert np.array_equal(g.obs[i].view(np.uint32), o.view(np.uint32)) and g.reward64[i] == r
                assert bool(g.term[i]) == te and bool(g.trunc[i]) == tr
    lockstep_steps(40)
    before_state, before_obs = g.state().copy(), g.obs.copy()
    ids = np.array([40, 3, 17, 41], dtype=np.int32)                 # unordered on purpose
    p2 = draw(len(ids))
    obs = g.reset(picks=p2, env_ids=ids)
    others = np.setdiff1d(np.arange(n), ids)
    assert np.array_equal(obs[others].view(np.uint32), before_obs[others].view(np.uint32))
    st = g.state()
    assert np.array_equal(st[others], before_state[others])
    for j, i in enumerate(ids):
        o = envs[i].reset(orooms[p2[j, 0]], orooms[p2[j, 0]].free_cell(p2[j, 1]))
        assert np.array_equal(obs[i].view(np.uint32), o.view(np.uint32))
        assert st[i, 6] == 0 and st[i, 4] == 1 and st[i, 13] == p2[j, 0] and st[i, 14] == before_state[i, 14] + 1
    lockstep_steps(60)
    for i in (3, 17, 0, 47):
        assert np.array_equal(g.grid(i), np.minimum(envs[i].grid(), 255).astype(np.int16))


def test_snapshot_restore_replays_identically(oracle):
    """nav3d_snapshot / nav3d_restore: the complete mutable state (records + knowledge) round-trips through host memory."""
    import torch
    from gpu_harness import GpuEngine
    rooms = load_room_dir(ROOMS / "P3_training", sort=True)
    n = 700
    g = GpuEngine(n, rooms, 10, -2.0, 13, 0, True, 4)
    g.reset()
    rng = np.random.default_rng(1)
    acts = rng.integers(0, 6, size=(260, n))
    for t in range(130):
        g.step(acts[t], pull=False)
    snap = g.eng.snapshot()
    assert snap.nbytes > n * 32
    first = []
    for t in range(130, 260):
        g.step(acts[t])
        first.append((g.obs.copy(), g.reward64.copy(), g.term.copy(), g.trunc.copy(), g.eps.copy()))
    st1, grid1 = g.state().copy(), g.grid(5).copy()
    g.eng.restore(snap)
    for t in range(130, 260):
        g.step(acts[t])
        o, r, te, tr, ep = first[t - 130]
        assert np.array_equal(g.obs.view(np.uint32), o.view(np.uint32)) and np.array_equal(g.reward64, r)
        assert np.array_equal(g.term, te) and np.array_equal(g.trunc, tr)
    assert np.array_equal(g.state(), st1) and np.array_equal(g.grid(5), grid1)
    with pytest.raises(Exception):
        g.eng.restore(snap[:-1])
    torch.cuda.synchronize()


def test_scalar_facade_matches_reference_traces(cubic_traces, capsys):
    """envs.CubicEnv.GridAgent (the drop-in for the reference's own scripts) with reset(seed=s): the room and start come
    from CPython's `random` exactly like the reference, so the golden traces (seeded resets) replay bit-for-bit."""
    from pathlib import Path

    from envs.CubicEnv import GridAgent
    from envs.Venv import GridAgent as VenvAgent
    assert VenvAgent is GridAgent
    for c in cubic_traces[:2] + cubic_traces[-2:]:
        p = ROOMS / c["room"]
        env = GridAgent(room_path=str(p.parent), local_map_length=c["L"], crash_penalty=c["crash_penalty"])
        env.rooms = [Path(p)]
        obs, info = env.reset(seed=c["seed"])
        assert info == {} and obs.dtype == np.float32 and obs.shape == (80,)
        assert (env.x, env.y, env.z) == tuple(c["start"]) and env.total_free_cells == c["total_free"]
        assert np.array_equal(obs.view(np.uint32), c["obs"][0].view(np.uint32))
        n = min(c["n"], 250) if c["policy"] == "random" else c["n"]
        for t in range(n):
            o, r, term, trunc, _ = env.step(int(c["actions"][t]))
            assert isinstance(r, float) and r == c["reward"][t]
            assert [env.x, env.y, env.z, env.facing, env.visited_count, env.bump_count, env.step_count, int(term), int(trunc)] == list(c["state"][t])
            assert np.array_equal(o.view(np.uint32), c["obs"][t + 1].view(np.uint32))
        assert env.get_position() == (env.x, env.y, env.z) and env.done == bool(c["state"][n - 1][7])
        if n == c["n"]:
            assert np.array_equal(env.internal_grid, np.minimum(c["final_ig"], 255))
        env.close()
    capsys.readouterr()


def test_scalar_facade_render_text_matches_reference(capsys):
    """a11: render() in text mode (CubicEnv.py:475-499) prints exactly what the unmodified reference printed
    (tests/golden/render_text.json, written by tests/golden/make_render_golden.py); close() releases the engine."""
    import json
    from pathlib import Path

    from envs.CubicEnv import GridAgent
    g = json.loads((Path(__file__).parent / "golden" / "render_text.json").read_text())
    p = ROOMS / g["room"]
    env = GridAgent(room_path=str(p.parent), local_map_length=g["L"], render_mode="human")
    env.rooms = [Path(p)]
    env.reset(seed=g["seed"])
    capsys.readouterr()
    env.render()
    assert capsys.readouterr().out == g["frames"]["0"]
    actions = np.random.default_rng(g["action_seed"]).integers(0, 6, size=120)
    for t, a in enumerate(actions, 1):
        env.step(int(a))
        if str(t) in g["frames"]:
            capsys.readouterr()
            env.render()
            assert capsys.readouterr().out == g["frames"][str(t)], f"frame after step {t}"
    env.render_mode = None
    env.render()                                   # any other mode: no output (:480-481)
    assert capsys.readouterr().out == ""
    env.close()
    env.close()                                    # idempotent


def test_batched_vec_env_contract(oracle):
    """nav3d.BatchedCubicEnv: SB3 VecEnv-shaped API (reset/step_async/step_wait, dones, terminal_observation, episode)."""
    import torch
    from nav3d import BatchedCubicEnv
    rooms = [load_room_file(ROOMS / "P3_training" / "maze_3d_tunnels.txt")]
    venv = BatchedCubicEnv(rooms=rooms, num_envs=64, local_map_length=10, seed=3)
    assert venv.num_envs == 64 and venv.action_space.n == 6 and venv.observation_space.shape == (80,)
    obs = venv.reset()
    assert obs.shape == (64, 80) and obs.is_cuda
    g = torch.Generator().manual_seed(0)
    seen_done = 0
    for t in range(200):
        a = torch.randint(0, 6, (64,), generator=g)
        venv.step_async(a)
        obs, rew, dones, info = venv.step_wait()
        assert rew.dtype == torch.float32 and dones.dtype == torch.bool
        if bool(dones.any()):
            infos = venv.sb3_infos(info)
            for i in torch.nonzero(dones).flatten().tolist():
                assert infos[i]["terminal_observation"].shape == (80,) and infos[i]["episode"]["l"] == 149
                assert infos[i]["TimeLimit.truncated"] is True
                seen_done += 1
            st = venv.state().cpu().numpy()
            assert (st[dones.cpu().numpy(), 6] == 0).all()          # auto-reset: step_count is back to 0
    assert seen_done == 64
    assert venv.get_attr("total_free_cells") == [149] * 64 and len(venv.env_method("get_position")) == 64
    venv.close()


def test_numpy_vec_env_adapter_on_gpu():
    """nav3d.NumpyVecEnv over BatchedCubicEnv: the SubprocVecEnv-shaped numpy interface of a host-side trainer."""
    from nav3d import BatchedCubicEnv, NumpyVecEnv
    rooms = [load_room_file(ROOMS / "P3_training" / "maze_3d_tunnels.txt")]
    venv = NumpyVecEnv(BatchedCubicEnv(rooms=rooms, num_envs=16, local_map_length=10, seed=2))
    obs = venv.reset()
    assert obs.shape == (16, 80) and obs.dtype == np.float32
    rng = np.random.default_rng(1)
    ends = 0
    for t in range(160):
        obs, rew, dones, infos = venv.step(rng.integers(0, 6, size=16))
        for i in np.nonzero(dones)[0]:
            ends += 1
            assert infos[i]["TimeLimit.truncated"] in (True, False) and infos[i]["episode"]["l"] == 149
            assert infos[i]["terminal_observation"].shape == (80,) and infos[i]["total_free"] == 149
    assert ends == 16 and venv.get_attr("total_free_cells") == [149] * 16
    assert len(venv.env_method("get_position")) == 16
    venv.close()

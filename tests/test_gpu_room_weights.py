"""Weighted room draw on the GPU (include/nav3d.h nav3d_set_room_weights / nav3d_get_room_cdf).

The device table must equal the reference table bit for bit; with uniform weights every output equals an engine that was never
given weights; with a weighted table every path that draws a room from the Philox stream (nav3d_reset, the auto-resets of
nav3d_step and nav3d_step_host, both fused rollouts, simpleEnv) runs lock-step with the oracle drawing from the same
table (tests/room_weights_ref.py).  Graph replays read the current table; rejected vectors leave it as it was."""
import numpy as np
import pytest
import torch

from conftest import ROOMS
from lockstep import compare_grids, compare_step
from nav3d.rooms import load_room_dir, load_room_file
import room_weights_ref as rw

pytestmark = pytest.mark.gpu
TWO32 = 1 << 32


def lockstep_rooms(simple=False):
    """Rooms where episodes end within a few hundred random steps, plus the shells of tests/edge_rooms.py."""
    rooms = [load_room_file(ROOMS / "P3_training" / "maze_3d_tunnels.txt", simple=simple),
             load_room_file(ROOMS / "P2_training" / "tightcorridor.txt", simple=simple)]
    if simple:
        return rooms + [load_room_file(ROOMS / "P3_training" / "kitchen2.txt", simple=True)]
    from edge_rooms import degenerate_rooms
    return rooms + load_room_dir(ROOMS / "P1_training", sort=True)[:2] + degenerate_rooms()


W8 = np.array([5.0, 0.0, 1.0, 0.25, 3.0, 0.0, 2.0, 1.5], np.float32)      # rooms 1 and 5 never drawn
W8_B = np.array([0.0, 4.0, 0.0, 1.0, 0.5, 2.0, 0.0, 0.0], np.float32)


def tiny_rooms(n):
    from edge_rooms import degenerate_rooms
    return [degenerate_rooms()[0]] * n


def engine(rooms, n, seed=0, lanes=0, auto_reset=True, env_id0=0, **kw):
    from nav3d import Engine
    return Engine(n, rooms, local_map_length=10, seed=seed, lanes_per_env=lanes, auto_reset=auto_reset, env_id0=env_id0,
                  **kw)


def make_pair(oracle, rooms, n, w, seed, lanes=0, auto_reset=True, env_id0=0):
    from gpu_harness import GpuEngine
    ov = rw.WeightedOracleVec(n, [oracle.OracleRoom(r.grid, -2) for r in rooms], 10, -2.0, seed, env_id0, auto_reset)
    g = GpuEngine(n, rooms, 10, -2.0, seed, env_id0, auto_reset, lanes)
    if w is not None:
        st, cdf = rw.cdf_build(w)
        assert st == 0
        g.eng.set_room_weights(w)
        assert np.array_equal(g.eng.room_cdf().cpu().numpy().astype(np.uint64), cdf)
        ov.set_room_cdf(cdf)
    assert np.array_equal(g.reset().view(np.uint32), ov.reset().view(np.uint32))
    return ov, g


def run_steps(tag, ov, g, actions):
    n_done = 0
    for t, a in enumerate(actions):
        ov.step(a)
        g.step(a)
        compare_step(tag, t, ov, g.obs, g.reward, g.reward64, g.term, g.trunc, g.tobs, g.eps, g.state())
        n_done += int((ov.terminated | ov.truncated).sum())
    return n_done


# ---- the table ---------------------------------------------------------------------------------------------------------

def weight_vectors(n, rng):
    out = [rng.random(n), rng.random(n) * (rng.random(n) < 0.5), np.exp(rng.normal(0, 20, n).clip(-80, 80)), np.zeros(n),
           rng.random(n), rng.random(n), rng.integers(0, 4, n).astype(np.float64)]
    out[3][rng.integers(0, n)] = 0.7                       # a single nonzero room
    out[4][0] = 0.0                                        # first room at zero
    out[5][-1] = 0.0 if n > 1 else 1.0                     # last room at zero
    res = []
    for w in out:
        w = w.astype(np.float32)
        if not (w > 0).any():
            w[0] = 1.0
        res.append(w)
    return res


@pytest.mark.parametrize("n_rooms", [1, 2, 25, 65535])
def test_device_table_equals_oracle(oracle, n_rooms):
    rooms = tiny_rooms(n_rooms) if n_rooms != 25 else load_room_dir(ROOMS / "P2_training", sort=True)
    assert len(rooms) == n_rooms
    eng = engine(rooms, 8)
    _, uni = rw.cdf_build(None, n_rooms)
    assert np.array_equal(eng.room_cdf().cpu().numpy().astype(np.uint64), uni)
    for w in weight_vectors(n_rooms, np.random.default_rng(n_rooms)):
        st, want = rw.cdf_build(w)
        assert st == 0
        eng.set_room_weights(w)
        got = eng.room_cdf().cpu().numpy().astype(np.uint64)
        assert np.array_equal(got, want), f"n={n_rooms}: first difference at {np.nonzero(got != want)[0][:4]}"
        p = eng.room_probabilities().cpu().numpy()
        assert np.array_equal(p, np.diff(want.astype(np.float64), prepend=0.0) / 2.0 ** 32)
        assert (p[w == 0] == 0).all()
    eng.set_room_weights(None)
    assert np.array_equal(eng.room_cdf().cpu().numpy().astype(np.uint64), uni)


def test_positive_weight_below_resolution_reads_as_zero():
    eng = engine(tiny_rooms(3), 4)
    eng.set_room_weights([1.0, 1e-10, 0.5])
    p = eng.room_probabilities().cpu().numpy()
    assert p[1] == 0.0 and p[0] > 0 and p[2] > 0 and p.sum() == 1.0


def test_set_room_weights_is_one_launch():
    eng = engine(tiny_rooms(25), 16)
    for w in (np.ones(25), None, np.arange(25, dtype=np.float32), [np.nan] * 25):
        before = eng.launch_count
        eng.set_room_weights(w, check=False)
        assert eng.launch_count == before + 1


@pytest.mark.parametrize("bad", ["nan", "inf", "negative", "zeros"])
def test_rejected_vectors_leave_the_table(oracle, bad):
    from nav3d import Nav3dError
    rooms = lockstep_rooms()
    ov, g = make_pair(oracle, rooms, 64, W8, seed=4)
    before = g.eng.room_cdf().clone()
    w = W8.copy()
    if bad == "nan":
        w[2] = np.nan
    elif bad == "inf":
        w[0] = np.inf
    elif bad == "negative":
        w[4] = -0.5
    else:
        w[:] = 0
    with pytest.raises(Nav3dError) as ei:
        g.eng.set_room_weights(w)
    assert {"nan": "NaN", "inf": "infinite", "negative": "negative", "zeros": "all weights are 0"}[bad] in str(ei.value)
    status = torch.full((1,), 7, dtype=torch.uint8, device=g.eng.device)
    from nav3d import _lib
    from nav3d.engine import _ptr
    wt = torch.as_tensor(w).to(g.eng.device)
    _lib.check(g.eng._lib.nav3d_set_room_weights(g.eng._h, _ptr(wt), _ptr(status), g.eng._stream()))
    assert int(status.item()) == 1
    assert torch.equal(g.eng.room_cdf(), before)
    assert run_steps(f"after rejected {bad}", ov, g, np.random.default_rng(4).integers(0, 6, size=(330, 64))) > 0
    with pytest.raises(ValueError):
        g.eng.set_room_weights(np.ones(len(rooms) + 1))
    with pytest.raises(ValueError):
        g.eng.set_room_weights(np.ones((2, len(rooms))))


def test_load_rooms_restores_the_uniform_table(oracle):
    rooms = lockstep_rooms()
    eng = engine(rooms, 8)
    eng.set_room_weights(W8)
    eng.load_rooms(rooms)
    _, uni = rw.cdf_build(None, len(rooms))
    assert np.array_equal(eng.room_cdf().cpu().numpy().astype(np.uint64), uni)


# ---- uniform weights change nothing --------------------------------------------------------------------------------------

def _outputs(eng, T, seed, n, simple=False):
    """Everything an engine produces through reset, steps with truncation waves, step_host and both rollouts."""
    dev, d = eng.device, eng.obs_dim
    out = {}
    obs = eng.reset()
    out["reset"] = obs.clone()
    rng = np.random.default_rng(seed)
    rew, r64 = torch.zeros(n, device=dev), torch.zeros(n, dtype=torch.float64, device=dev)
    te, tr = torch.zeros(n, dtype=torch.uint8, device=dev), torch.zeros(n, dtype=torch.uint8, device=dev)
    tobs, eps = torch.zeros((n, d), device=dev), torch.zeros((n, 8), dtype=torch.int32, device=dev)
    steps = []
    for t in range(T):
        a = torch.as_tensor(rng.integers(0, 6, size=n)).to(dev)
        eng.step(a, obs, rew, te, tr, reward64=r64, terminal_obs=tobs, episodes=eps)
        steps.append(torch.cat([obs.flatten().view(torch.int32), rew.view(torch.int32), r64.view(torch.int32),
                                te.int(), tr.int(), tobs.flatten().view(torch.int32), eps.flatten()]))
    out["steps"] = torch.stack(steps)
    pin = [torch.zeros(n, dtype=torch.int64).pin_memory(), torch.zeros((n, d)).pin_memory(), torch.zeros(n).pin_memory(),
           torch.zeros(n, dtype=torch.uint8).pin_memory(), torch.zeros(n, dtype=torch.uint8).pin_memory()]
    hs = []
    for t in range(40):
        pin[0][:] = torch.as_tensor(rng.integers(0, 6, size=n))
        eng.step_host(*pin)
        hs.append(torch.cat([pin[1].flatten().view(torch.int32), pin[2].view(torch.int32), pin[3].int(), pin[4].int()]))
    out["step_host"] = torch.stack(hs)
    if not simple:
        o = torch.empty((64, n, 80), device=dev)
        r = torch.empty((64, n), device=dev)
        dn = torch.empty((64, n), dtype=torch.uint8, device=dev)
        ac = torch.empty((64, n), dtype=torch.uint8, device=dev)
        eng.rollout_random(64, 0, obs=o, reward=r, done=dn, actions_out=ac)
        out["rollout_random"] = [o.clone(), r.clone(), dn.clone(), ac.clone()]
        acts = torch.as_tensor(rng.integers(0, 6, size=(64, n)).astype(np.uint8)).to(dev)
        buf = dict(obs=torch.zeros((64, n, 80), device=dev), reward64=torch.zeros((64, n), dtype=torch.float64, device=dev),
                   terminated=torch.zeros((64, n), dtype=torch.uint8, device=dev),
                   truncated=torch.zeros((64, n), dtype=torch.uint8, device=dev),
                   terminal_obs=torch.zeros((64, n, 80), device=dev),
                   episodes=torch.zeros((64, n, 8), dtype=torch.int32, device=dev))
        eng.rollout_actions(acts, **buf)
        out["rollout_actions"] = list(buf.values())
    out["state"] = eng.get_state()
    return out


def _same(a, b, tag):
    for k in a:
        xs, ys = (a[k], b[k]) if isinstance(a[k], list) else ([a[k]], [b[k]])
        for x, y in zip(xs, ys):
            assert torch.equal(x.view(torch.uint8) if x.is_floating_point() else x,
                               y.view(torch.uint8) if y.is_floating_point() else y), f"{tag}: {k} differs"


@pytest.mark.parametrize("lanes", [1, 4])
@pytest.mark.parametrize("value", [1.0, 3.5e-30, 7e30])
def test_uniform_weights_change_nothing(lanes, value):
    rooms = lockstep_rooms()
    n = 2048 + 45
    ref = _outputs(engine(rooms, n, seed=3, lanes=lanes), 330, 1, n)
    eng = engine(rooms, n, seed=3, lanes=lanes)
    eng.set_room_weights(np.full(len(rooms), value, np.float32))
    _same(ref, _outputs(eng, 330, 1, n), f"lanes={lanes} w={value}")


def test_uniform_weights_change_nothing_simple():
    from nav3d import _lib
    rooms = lockstep_rooms(simple=True)
    n = 1024 + 3
    ref = _outputs(engine(rooms, n, seed=2, env_kind=_lib.ENV_SIMPLE), 330, 2, n, simple=True)
    eng = engine(rooms, n, seed=2, env_kind=_lib.ENV_SIMPLE)
    eng.set_room_weights([2.0] * len(rooms))
    _same(ref, _outputs(eng, 330, 2, n, simple=True), "simple")


# ---- weighted lock-step ------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("lanes,auto_reset", [(1, True), (4, True), (32, True), (1, False), (4, False)])
def test_step_lockstep_weighted(oracle, lanes, auto_reset):
    ov, g = make_pair(oracle, lockstep_rooms(), 64, W8, seed=lanes, lanes=lanes, auto_reset=auto_reset)
    acts = np.random.default_rng(lanes + 50).integers(0, 6, size=(330, 64))
    n_done = run_steps(f"weighted lanes={lanes}", ov, g, acts)
    assert n_done > 0
    compare_grids("weighted", ov, g.grid, range(0, 64, 9))


def test_partial_reset_weighted(oracle):
    """nav3d_reset with env_ids and Philox picks: each listed env draws (room, k) from the table at its episode counter."""
    rooms = lockstep_rooms()
    n, seed = 256, 8
    _, cdf = rw.cdf_build(W8)
    g = engine(rooms, n, seed=seed, auto_reset=False)
    g.set_room_weights(W8)
    obs = g.reset()
    ids = np.arange(3, n, 5, dtype=np.int32)
    for _ in range(3):
        before = g.get_state().cpu().numpy()
        g.reset(obs, env_ids=torch.as_tensor(ids))
        st = g.get_state().cpu().numpy()
        nf = [g.room_free[r] for r in range(len(rooms))]
        for i in ids:
            room, k = rw.pick(seed, int(i), int(before[i, 14]), nf, cdf)
            start = rooms[room].start if getattr(rooms[room], "start", None) else tuple(rooms[room].free_cells()[k])
            assert st[i, 13] == room and tuple(st[i, :3]) == tuple(start) and st[i, 14] == before[i, 14] + 1, i
            orc = oracle.OracleCubic(10)
            want = orc.reset(oracle.OracleRoom(rooms[room].grid, -2), start)
            assert np.array_equal(obs[i].cpu().numpy().view(np.uint32), want.view(np.uint32)), i
        others = np.setdiff1d(np.arange(n), ids)
        assert np.array_equal(st[others], before[others])
    assert not set(st[ids, 13].tolist()) & {1, 5}


@pytest.mark.parametrize("lanes", [1, 4])
def test_rollout_random_weighted(oracle, lanes):
    n, T = 64, 300
    ov, g = make_pair(oracle, lockstep_rooms(), n, W8, seed=5, lanes=lanes)
    dev = g.eng.device
    obs = torch.empty((T, n, 80), device=dev)
    rew = torch.empty((T, n), device=dev)
    done = torch.empty((T, n), dtype=torch.uint8, device=dev)
    acts = torch.empty((T, n), dtype=torch.uint8, device=dev)
    g.eng.rollout_random(T, 0, obs=obs, reward=rew, done=done, actions_out=acts)
    o = [x.cpu().numpy() for x in (obs, rew, done, acts)]
    n_done = 0
    for t in range(T):
        ov.step(o[3][t].astype(np.int64))
        assert np.array_equal(o[1][t], ov.reward.astype(np.float32)), t
        assert np.array_equal(o[2][t], ov.terminated | ov.truncated), t
        assert np.array_equal(o[0][t].view(np.uint32), ov.obs.view(np.uint32)), t
        n_done += int(o[2][t].sum())
    assert n_done > 0
    st = g.state()
    assert np.array_equal(st[:, :15].astype(np.int64), ov.state()) and np.array_equal(st[:, 15], ov.ret_centi())


@pytest.mark.parametrize("lanes", [1, 8])
def test_rollout_actions_weighted(oracle, lanes):
    n, T = 64, 330
    ov, g = make_pair(oracle, lockstep_rooms(), n, W8, seed=9, lanes=lanes)
    dev = g.eng.device
    acts = np.random.default_rng(3).integers(0, 6, size=(T, n)).astype(np.uint8)
    buf = dict(obs=torch.empty((T, n, 80), device=dev), reward=torch.empty((T, n), device=dev),
               reward64=torch.empty((T, n), dtype=torch.float64, device=dev),
               terminated=torch.empty((T, n), dtype=torch.uint8, device=dev),
               truncated=torch.empty((T, n), dtype=torch.uint8, device=dev),
               terminal_obs=torch.zeros((T, n, 80), device=dev), episodes=torch.zeros((T, n, 8), dtype=torch.int32, device=dev))
    g.eng.rollout_actions(torch.as_tensor(acts).to(dev), **buf)
    o = {k: v.cpu().numpy() for k, v in buf.items()}
    for t in range(T):
        ov.step(acts[t])
        compare_step(f"weighted rollout_actions lanes={lanes}", t, ov, o["obs"][t], o["reward"][t], o["reward64"][t],
                     o["terminated"][t], o["truncated"][t], o["terminal_obs"][t], o["episodes"][t], None)
    st = g.state()
    assert np.array_equal(st[:, :15].astype(np.int64), ov.state())
    rooms_done = o["episodes"][..., 5][(o["terminated"] | o["truncated"]).astype(bool)]
    assert len(rooms_done) and not set(rooms_done.tolist()) & {1, 5}


def test_step_host_weighted(oracle):
    """nav3d_step_host at 65 536 + 45 envs (four chunks): a strided sample against the oracle."""
    rooms = lockstep_rooms()
    n, seed = 65536 + 45, 12
    _, cdf = rw.cdf_build(W8)
    eng = engine(rooms, n, seed=seed)
    eng.set_room_weights(W8)
    eng.reset()
    sample = np.arange(0, n, 997)
    ov = rw.WeightedOracleVec(len(sample), [oracle.OracleRoom(r.grid, -2) for r in rooms], 10, -2.0, seed, 0, True)
    ov.set_ids(sample)
    ov.set_room_cdf(cdf)
    ov.reset()
    pin = [torch.zeros(n, dtype=torch.int64).pin_memory(), torch.zeros((n, 80)).pin_memory(), torch.zeros(n).pin_memory(),
           torch.zeros(n, dtype=torch.uint8).pin_memory(), torch.zeros(n, dtype=torch.uint8).pin_memory()]
    rng = np.random.default_rng(seed)
    n_done = 0
    for t in range(330):
        a = rng.integers(0, 6, size=n)
        pin[0][:] = torch.as_tensor(a)
        eng.step_host(*pin)
        ov.step(a[sample])
        assert np.array_equal(pin[1].numpy()[sample].view(np.uint32), ov.obs.view(np.uint32)), t
        assert np.array_equal(pin[2].numpy()[sample], ov.reward.astype(np.float32)), t
        n_done += int(ov.terminated.sum() + ov.truncated.sum())
    assert n_done > 0
    assert np.array_equal(eng.get_state().cpu().numpy()[sample, :15].astype(np.int64), ov.state())


def test_simple_env_weighted(oracle):
    from nav3d import Engine, _lib
    rooms = lockstep_rooms(simple=True)
    w = np.array([0.0, 3.0, 1.0], np.float32)
    _, cdf = rw.cdf_build(w)
    n, L, seed = 64, 10, 21
    ov = rw.WeightedSimpleVec(n, [oracle.OracleRoom(r.grid, 2) for r in rooms], L, 0.25, seed, 0, True, cdf=cdf)
    eng = Engine(n, rooms, local_map_length=L, seed=seed, env_kind=_lib.ENV_SIMPLE)
    eng.set_room_weights(w)
    dev, d = eng.device, eng.obs_dim
    obs = eng.reset()
    assert np.array_equal(obs.cpu().numpy().view(np.uint32), ov.reset().view(np.uint32))
    rew, r64 = torch.zeros(n, device=dev), torch.zeros(n, dtype=torch.float64, device=dev)
    te, tr = torch.zeros(n, dtype=torch.uint8, device=dev), torch.zeros(n, dtype=torch.uint8, device=dev)
    tobs = torch.zeros((n, d), device=dev)
    rng = np.random.default_rng(seed)
    n_done = 0
    for t in range(330):
        a = rng.integers(0, 6, size=n)
        ov.step(a)
        eng.step(torch.as_tensor(a).to(dev), obs, rew, te, tr, reward64=r64, terminal_obs=tobs)
        assert np.array_equal(obs.cpu().numpy().view(np.uint32), ov.obs.view(np.uint32)), t
        assert np.array_equal(r64.cpu().numpy(), ov.reward), t
        assert np.array_equal(te.cpu().numpy(), ov.terminated) and np.array_equal(tr.cpu().numpy(), ov.truncated), t
        st = eng.get_state().cpu().numpy()
        assert np.array_equal(st[:, 13], np.array(ov.room_idx)) and np.array_equal(st[:, 14], np.array(ov.episode)), t
        n_done += int((ov.terminated | ov.truncated).sum())
    assert n_done > 0 and 0 not in set(ov.room_idx)


def test_million_envs_one_generation(oracle):
    """2^20 envs: the first reset's rooms against the oracle's draw for every env; zero-weight rooms never drawn over
    several reset generations (each nav3d_reset is a new episode number)."""
    rooms = lockstep_rooms()
    n, seed = 1 << 20, 17
    _, cdf = rw.cdf_build(W8)
    eng = engine(rooms, n, seed=seed, auto_reset=False)
    eng.set_room_weights(W8)
    obs = eng.reset()
    st = eng.get_state().cpu().numpy()
    nf = [eng.room_free[r] for r in range(len(rooms))]
    sample = np.arange(0, n, 61)
    want = np.array([rw.pick(seed, int(i), 0, nf, cdf)[0] for i in sample])
    assert np.array_equal(st[sample, 13], want)
    counts = np.bincount(st[:, 13], minlength=len(rooms))
    for _ in range(4):
        eng.reset(obs)
        counts += np.bincount(eng.get_state()[:, 13].cpu().numpy(), minlength=len(rooms))
    assert counts[1] == 0 and counts[5] == 0
    p = W8 / W8.sum()
    for j in np.nonzero(p)[0]:
        assert abs(counts[j] / (5 * n) - p[j]) < 6 * np.sqrt(p[j] * (1 - p[j]) / (5 * n)), (j, counts)


# ---- graphs, sharding, blobs ---------------------------------------------------------------------------------------------

def test_graph_replays_read_the_current_table(oracle):
    """The table lives at a fixed device address: weights set eagerly between replays of a captured step graph change the
    rooms the replays draw; and set_room_weights itself captured with a device weight tensor installs its current
    contents at each replay."""
    rooms = lockstep_rooms()
    n, T = 256, 40
    ov, g = make_pair(oracle, rooms, n, W8, seed=6)
    dev = g.eng.device
    acts = np.random.default_rng(6).integers(0, 6, size=(3 * T + 1, n))
    a_dev = torch.as_tensor(acts[-1]).to(dev)
    g.step(acts[-1])                                       # one eager step first (module loading), the oracle alongside
    ov.step(acts[-1])
    torch.cuda.synchronize()
    ov2, g2 = ov, g
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        g2.eng.step(a_dev, g2.d_obs, g2.d_reward, g2.d_term, g2.d_trunc, reward64=g2.d_reward64, terminal_obs=g2.d_tobs,
                    episodes=g2.d_eps)
    for phase, w in enumerate((W8, W8_B, None)):
        if phase:
            g2.eng.set_room_weights(w)
            ov2.set_room_cdf(rw.cdf_build(w, len(rooms))[1])
        for t in range(phase * T, (phase + 1) * T):
            a_dev.copy_(torch.as_tensor(acts[t]))
            graph.replay()
            g2._pull()
            ov2.step(acts[t])
            compare_step(f"graph phase {phase}", t, ov2, g2.obs, g2.reward, g2.reward64, g2.term, g2.trunc, g2.tobs,
                         g2.eps, g2.state())
    # capture set_room_weights itself
    wt = torch.as_tensor(W8).to(dev)
    g2.eng.set_room_weights(wt, check=False)
    torch.cuda.synchronize()
    gw = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gw):
        g2.eng.set_room_weights(wt, check=False)
    wt.copy_(torch.as_tensor(W8_B))
    gw.replay()
    torch.cuda.synchronize()
    assert np.array_equal(g2.eng.room_cdf().cpu().numpy().astype(np.uint64), rw.cdf_build(W8_B)[1])


def test_sharded_engines_draw_the_same_rooms():
    rooms = lockstep_rooms()
    n, seed = 4096, 23
    full = engine(rooms, n, seed=seed)
    halves = [engine(rooms, n // 2, seed=seed, env_id0=h * (n // 2)) for h in (0, 1)]
    for e in [full] + halves:
        e.set_room_weights(W8)
    engines = [full] + halves
    outs = [e.reset() for e in engines]
    assert torch.equal(outs[0], torch.cat(outs[1:]))
    rng = np.random.default_rng(seed)
    for t in range(330):
        a = torch.as_tensor(rng.integers(0, 6, size=n)).to(full.device)
        for e, o, aa in zip(engines, outs, (a, a[: n // 2].contiguous(), a[n // 2:].contiguous())):
            m = e.n_envs
            e.step(aa, o, torch.zeros(m, device=e.device), torch.zeros(m, dtype=torch.uint8, device=e.device),
                   torch.zeros(m, dtype=torch.uint8, device=e.device))
    st = [e.get_state() for e in engines]
    assert torch.equal(st[0], torch.cat(st[1:]))
    assert torch.equal(outs[0], torch.cat(outs[1:]))


def test_blob_continues_until_its_next_reset_then_follows_the_destination_table(oracle):
    rooms = lockstep_rooms()
    n, seed = 48, 10
    ov, src = make_pair(oracle, rooms, n, W8, seed=seed)
    acts = np.random.default_rng(10).integers(0, 6, size=(400, n))
    run_steps("source", ov, src, acts[:70])
    from gpu_harness import GpuEngine
    dst = GpuEngine(n, rooms, 10, -2.0, seed, 0, True, 0)
    dst.eng.set_room_weights(W8_B)
    dst.reset()
    ids = torch.arange(n, dtype=torch.int32, device=dst.eng.device)
    dst.eng.load_envs(ids, src.eng.save_envs(ids, src.d_obs), dst.d_obs)
    assert np.array_equal(dst.state(), src.state())
    ov.set_room_cdf(rw.cdf_build(W8_B)[1])
    assert run_steps("destination", ov, dst, acts[70:]) > 0

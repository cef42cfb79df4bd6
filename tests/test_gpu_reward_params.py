"""Non-default reward parameters and simpleEnv cell sizes on the GPU, against the parametrized oracle.

Every accepted parameter set (tests/reward_sets.py) runs lock-step through nav3d_step at every lane width, both fused
rollouts at one thread per env and in lane groups, and nav3d_step_host across its four-chunk pipeline.  Rewards (f64 and
f32), flags, observations, terminal observations and the integer state are compared bit for bit; the episode record's
return and state column 15 are compared exactly with the oracle's restatement of the documented 1/100-unit rule, and the
return is held to the documented bound against the f64 sum of the rewards (tests/lockstep.py)."""
import numpy as np
import pytest
import torch

from conftest import ROOMS
from lockstep import compare_grids, compare_step
from nav3d.rooms import load_room_dir, load_room_file
from oracle.c_oracle import reward_values
from reward_sets import ACCEPTED, INT32_MAX, REJECTED, full

pytestmark = pytest.mark.gpu
SET_IDS = [k for k, _ in ACCEPTED]
NAMED = dict(ACCEPTED)


def lockstep_rooms():
    """Rooms where episodes end within a few hundred steps (maze_3d_tunnels truncates at 149, tightcorridor at 302),
    a P1 room and the degenerate shells of tests/edge_rooms.py (two cells, 1-wide corridors)."""
    from edge_rooms import degenerate_rooms
    return ([load_room_file(ROOMS / "P3_training" / "maze_3d_tunnels.txt"),
             load_room_file(ROOMS / "P2_training" / "tightcorridor.txt")]
            + load_room_dir(ROOMS / "P1_training", sort=True)[:2] + degenerate_rooms())


def make_pair(oracle, rooms, n, reward, seed, auto_reset=True, lanes=0, L=10, env_id0=0):
    from gpu_harness import GpuEngine
    crash = float(reward_values(reward)[3])
    ov = oracle.OracleVec(n, [oracle.OracleRoom(r.grid, -2) for r in rooms], L, crash, seed, env_id0, auto_reset,
                          reward=reward)
    g = GpuEngine(n, rooms, L, crash, seed, env_id0, auto_reset, lanes)
    g.eng.set_reward_params(**reward)
    assert g.eng.reward_params == full(dict(reward, crash_penalty=crash))
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


@pytest.mark.parametrize("lanes", [1, 2, 4, 8, 16, 32])
@pytest.mark.parametrize("name,reward", ACCEPTED, ids=SET_IDS)
def test_step_lockstep(oracle, name, reward, lanes):
    auto_reset = lanes != 2                     # lanes = 2 runs plain-gym envs on past done
    ov, g = make_pair(oracle, lockstep_rooms(), 64, reward, seed=lanes, auto_reset=auto_reset, lanes=lanes)
    rng = np.random.default_rng(lanes + 100)
    n_done = run_steps(f"{name} lanes={lanes}", ov, g, rng.integers(0, 6, size=(330, 64)))
    assert n_done > 0
    compare_grids(name, ov, g.grid, range(0, 64, 9))


def _pull(d):
    return {k: (None if v is None else v.cpu().numpy()) for k, v in d.items()}


@pytest.mark.parametrize("lanes", [1, 4])
@pytest.mark.parametrize("name,reward", ACCEPTED, ids=SET_IDS)
def test_rollout_random_lockstep(oracle, name, reward, lanes):
    """nav3d_rollout_random's rewards, done flags and observations against the oracle replaying the actions it played."""
    n, T = 64, 200
    ov, g = make_pair(oracle, lockstep_rooms(), n, reward, seed=5, lanes=lanes)
    dev = g.eng.device
    obs = torch.empty((T, n, 80), device=dev)
    rew = torch.empty((T, n), device=dev)
    done = torch.empty((T, n), dtype=torch.uint8, device=dev)
    acts = torch.empty((T, n), dtype=torch.uint8, device=dev)
    g.eng.rollout_random(T, 0, obs=obs, reward=rew, done=done, actions_out=acts)
    o = _pull(dict(obs=obs, rew=rew, done=done, acts=acts))
    for t in range(T):
        ov.step(o["acts"][t].astype(np.int64))
        tag = f"{name} rollout_random lanes={lanes} t={t}"
        assert np.array_equal(o["rew"][t], ov.reward.astype(np.float32)), tag
        assert np.array_equal(o["done"][t], ov.terminated | ov.truncated), tag
        assert np.array_equal(o["obs"][t].view(np.uint32), ov.obs.view(np.uint32)), tag
    st = g.state()
    assert np.array_equal(st[:, :15].astype(np.int64), ov.state()) and np.array_equal(st[:, 15], ov.ret_centi()), name


@pytest.mark.parametrize("lanes", [1, 8])
@pytest.mark.parametrize("name,reward", ACCEPTED, ids=SET_IDS)
def test_rollout_actions_lockstep(oracle, name, reward, lanes):
    """nav3d_rollout_actions with every output, against the oracle step by step."""
    n, T = 64, 330
    auto_reset = lanes == 1
    ov, g = make_pair(oracle, lockstep_rooms(), n, reward, seed=9, auto_reset=auto_reset, lanes=lanes)
    dev = g.eng.device
    acts = np.random.default_rng(3).integers(0, 6, size=(T, n)).astype(np.uint8)
    buf = dict(obs=torch.empty((T, n, 80), device=dev), reward=torch.empty((T, n), device=dev),
               reward64=torch.empty((T, n), dtype=torch.float64, device=dev),
               terminated=torch.empty((T, n), dtype=torch.uint8, device=dev),
               truncated=torch.empty((T, n), dtype=torch.uint8, device=dev),
               terminal_obs=torch.zeros((T, n, 80), device=dev), episodes=torch.zeros((T, n, 8), dtype=torch.int32, device=dev))
    g.eng.rollout_actions(torch.as_tensor(acts).to(dev), **buf)
    o = _pull(buf)
    for t in range(T):
        ov.step(acts[t])
        compare_step(f"{name} rollout_actions lanes={lanes}", t, ov, o["obs"][t], o["reward"][t], o["reward64"][t],
                     o["terminated"][t], o["truncated"][t], o["terminal_obs"][t] if auto_reset else None,
                     o["episodes"][t], None)
    st = g.state()
    assert np.array_equal(st[:, :15].astype(np.int64), ov.state()) and np.array_equal(st[:, 15], ov.ret_centi()), name


@pytest.mark.parametrize("name", ["defaults", "non_centi"])
def test_step_host_four_chunks(oracle, name):
    """nav3d_step_host at 65 536 + 45 envs: four chunks on two streams whose boundaries fall mid-warp.  Bit for bit
    against nav3d_step on a second engine, and a strided sample (every chunk, auto-resets included) against the oracle."""
    from nav3d import Engine
    reward = NAMED[name]
    rooms = [load_room_file(ROOMS / "P3_training" / "maze_3d_tunnels.txt")] + load_room_dir(ROOMS / "P1_training", sort=True)[:1]
    n, seed, steps = 65536 + 45, 12, 170
    a_eng = Engine(n, rooms, local_map_length=10, seed=seed)
    b_eng = Engine(n, rooms, local_map_length=10, seed=seed)
    for e in (a_eng, b_eng):
        e.set_reward_params(**reward)
    dev = a_eng.device
    obs_d = a_eng.reset()
    b_eng.reset()
    ids = np.unique(np.concatenate([np.arange(0, n, 331), np.arange(n - 40, n), [16383, 16384, 32767, 32768, 49151, 49152]]))
    ov = oracle.OracleVec(len(ids), [oracle.OracleRoom(r.grid, -2) for r in rooms], 10, -2.0, seed, 0, True, reward=reward)
    ov.set_ids(ids)
    ov.reset()
    assert np.array_equal(obs_d.cpu().numpy()[ids].view(np.uint32), ov.obs.view(np.uint32))
    rew_d = torch.zeros(n, device=dev)
    te_d, tr_d = torch.zeros(n, dtype=torch.uint8, device=dev), torch.zeros(n, dtype=torch.uint8, device=dev)
    obs_h, rew_h = torch.zeros((n, 80)).pin_memory(), torch.zeros(n).pin_memory()
    te_h, tr_h = torch.zeros(n, dtype=torch.uint8).pin_memory(), torch.zeros(n, dtype=torch.uint8).pin_memory()
    gen = torch.Generator().manual_seed(0)
    n_done = 0
    for t in range(steps):
        a = torch.randint(0, 6, (n,), generator=gen, dtype=torch.int64)
        a_eng.step(a.to(dev), obs_d, rew_d, te_d, tr_d)
        b_eng.step_host(a.pin_memory(), obs_h, rew_h, te_h, tr_h)
        assert torch.equal(obs_d.cpu(), obs_h) and torch.equal(rew_d.cpu(), rew_h), f"{name} t={t}"
        assert torch.equal(te_d.cpu(), te_h) and torch.equal(tr_d.cpu(), tr_h), f"{name} t={t}"
        ov.step(a.numpy()[ids])
        assert np.array_equal(obs_h.numpy()[ids].view(np.uint32), ov.obs.view(np.uint32)), f"{name} t={t}: obs vs oracle"
        assert np.array_equal(rew_h.numpy()[ids], ov.reward.astype(np.float32)), f"{name} t={t}: reward vs oracle"
        assert np.array_equal(te_h.numpy()[ids], ov.terminated) and np.array_equal(tr_h.numpy()[ids], ov.truncated)
        n_done += int((ov.terminated | ov.truncated).sum())
        if t % 40 == 0 or t == steps - 1:
            sa, sb = a_eng.get_state().cpu().numpy(), b_eng.get_state().cpu().numpy()
            assert np.array_equal(sa, sb), f"{name} t={t}: state"
            assert np.array_equal(sb[ids, :15].astype(np.int64), ov.state()) and np.array_equal(sb[ids, 15], ov.ret_centi())
    assert n_done > 0


def test_rejected_sets_leave_the_engine_unchanged(oracle):
    """Every set the rules reject fails with NAV3D_ERR_UNSUPPORTED and the engine keeps stepping with its old values."""
    from nav3d import Nav3dError
    ov, g = make_pair(oracle, lockstep_rooms(), 32, {"step_cost": -0.1}, seed=2)
    for name, reward in REJECTED:
        with pytest.raises(Nav3dError) as ei:
            g.eng.set_reward_params(**reward)
        assert ei.value.code == -2, name
        assert g.eng.reward_params["step_cost"] == -0.1, name
    run_steps("after rejections", ov, g, np.random.default_rng(0).integers(0, 6, size=(60, 32)))


def test_saturated_visit_count(oracle):
    """Action 4 under the ceiling of a room with 302 free cells: the agent's cell passes 255 visits.  At the defaults the
    penalty is capped long before, so the engine's saturated count still gives the reference's rewards; a set for which
    the saturation would change the penalty (unit 0.001, cap 1: the 256th visit costs 0.256) is refused."""
    from nav3d import Nav3dError
    rooms = [load_room_file(ROOMS / "P2_training" / "tightcorridor.txt")]
    n, T = 32, 300
    ov, g = make_pair(oracle, rooms, n, {}, seed=4)
    acts = np.full((T, n), 4, np.uint8)
    dev = g.eng.device
    r64 = torch.empty((T, n), dtype=torch.float64, device=dev)
    g.eng.rollout_actions(torch.as_tensor(acts).to(dev), obs_last=g.d_obs, reward64=r64)
    r64 = r64.cpu().numpy()
    for t in range(T):
        ov.step(acts[t])
        assert np.array_equal(r64[t], ov.reward), f"t={t}"
    assert max(int(ov.grid(i).max()) for i in range(n)) > 256
    st = g.state()
    assert np.array_equal(st[:, :15].astype(np.int64), ov.state()) and np.array_equal(st[:, 15], ov.ret_centi())
    with pytest.raises(Nav3dError) as ei:
        g.eng.set_reward_params(revisit_unit=0.001, revisit_cap=1.0)
    assert ei.value.code == -2 and "saturate" in str(ei.value)


def test_return_saturates_on_a_never_reset_env():
    """auto_reset = 0 at the defaults: after done every step earns the finish bonus (+94.45 net), so 2.5e5 steps take the
    return past 2^31 centi.  It must stay at the int32 maximum, not wrap."""
    from edge_rooms import degenerate_rooms
    from nav3d import Engine
    n, T = 32, 250_000
    eng = Engine(n, degenerate_rooms()[3:4], local_map_length=10, auto_reset=False, seed=1)
    eng.reset()
    acts = torch.tensor([[4], [5]], dtype=torch.uint8).repeat(T // 2, n).to(eng.device)
    eng.rollout_actions(acts, obs_last=eng.new_obs())
    st = eng.get_state().cpu().numpy()
    assert (st[:, 10] == 1).all()
    assert (st[:, 15] == INT32_MAX).all(), st[:, 15]


def test_mid_run_change_takes_effect_at_the_next_step(oracle):
    ov, g = make_pair(oracle, lockstep_rooms(), 48, {}, seed=6)
    acts = np.random.default_rng(6).integers(0, 6, size=(300, 48))
    run_steps("defaults", ov, g, acts[:97])
    new = NAMED["non_centi"]
    g.eng.set_reward_params(**new)
    ov.set_reward(new)
    assert run_steps("non_centi after the change", ov, g, acts[97:]) > 0


def test_unnamed_fields_keep_their_values(oracle):
    """A second set_reward_params call changes only the fields it names."""
    ov, g = make_pair(oracle, lockstep_rooms(), 32, {"step_cost": -0.1}, seed=8)
    g.eng.set_reward_params(explore_bonus=2.0)
    assert g.eng.reward_params == full({"step_cost": -0.1, "explore_bonus": 2.0})
    ov.set_reward({"step_cost": -0.1, "explore_bonus": 2.0})
    run_steps("two calls", ov, g, np.random.default_rng(8).integers(0, 6, size=(200, 32)))


def test_blob_continues_with_the_destination_parameters(oracle):
    """Blobs hold no reward parameters: saved under one set, loaded into an engine with another, an env continues with the
    destination's values, its return so far carried over."""
    from gpu_harness import GpuEngine
    a_set, b_set = {"explore_bonus": 3.0, "step_cost": -0.01}, NAMED["non_centi"]
    rooms = lockstep_rooms()
    ov, src = make_pair(oracle, rooms, 48, a_set, seed=10)
    acts = np.random.default_rng(10).integers(0, 6, size=(260, 48))
    run_steps("source", ov, src, acts[:70])
    dst = GpuEngine(48, rooms, 10, -2.0, 10, 0, True, 0)
    dst.eng.set_reward_params(**b_set)
    dst.reset()
    ids = torch.arange(48, dtype=torch.int32, device=dst.eng.device)
    dst.eng.load_envs(ids, src.eng.save_envs(ids, src.d_obs), dst.d_obs)
    assert np.array_equal(dst.state(), src.state())
    ov.set_reward(b_set)
    assert run_steps("destination", ov, dst, acts[70:]) > 0


def test_graph_replays_the_parameters_it_captured(oracle):
    """Parameters are launch arguments: a graph captured before set_reward_params replays the old values."""
    from gpu_harness import GpuEngine
    rooms = lockstep_rooms()
    n, T = 256, 64
    a = GpuEngine(n, rooms, 10, -2.0, 3, 0, True, 0)
    b = GpuEngine(n, rooms, 10, -2.0, 3, 0, True, 0)
    a.reset(); b.reset()
    dev = a.eng.device
    acts = torch.randint(0, 6, (T, n), generator=torch.Generator().manual_seed(3), dtype=torch.uint8).to(dev)
    ra, rb = torch.empty((T, n), dtype=torch.float64, device=dev), torch.empty((T, n), dtype=torch.float64, device=dev)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        a.eng.rollout_actions(acts, obs_last=a.d_obs, reward64=ra)
    a.eng.set_reward_params(**NAMED["non_centi"])
    graph.replay()
    b.eng.rollout_actions(acts, obs_last=b.d_obs, reward64=rb)
    torch.cuda.synchronize()
    assert torch.equal(ra, rb), "the replay must use the captured (default) parameters"
    assert np.array_equal(a.state(), b.state())
    a.eng.rollout_actions(acts, obs_last=a.d_obs, reward64=ra)
    b.eng.rollout_actions(acts, obs_last=b.d_obs, reward64=rb)
    assert not torch.equal(ra, rb), "an ordinary launch uses the new parameters"


def test_simple_env_rejects_reward_params():
    from nav3d import Engine, Nav3dError, _lib
    rooms = [load_room_file(ROOMS / "P3_training" / "maze_3d_tunnels.txt", simple=True)]
    eng = Engine(4, rooms, local_map_length=4, env_kind=_lib.ENV_SIMPLE)
    with pytest.raises(Nav3dError) as ei:
        eng.set_reward_params(step_cost=-0.1)
    assert ei.value.code == -2


@pytest.mark.parametrize("cell_size,L", [(0.175, 10), (0.075, 10), (0.3, 10), (0.25, 16)])
def test_simple_cell_sizes(oracle, cell_size, L):
    """simpleEnv against the oracle at cell sizes whose distances round differently under rint(x * 100) / 100 (0.175,
    0.075) and at L = 16, where 6L + 7 = 103 makes the engine pick 2 lanes per env."""
    from nav3d import Engine, _lib
    rooms = [load_room_file(ROOMS / "P3_training" / n, simple=True) for n in ("maze_3d_tunnels.txt", "kitchen2.txt")] + \
            [load_room_file(ROOMS / "P2_training" / "tightcorridor.txt", simple=True)]
    n, steps, seed = 64, 330, 21
    ov = oracle.OracleSimpleVec(n, [oracle.OracleRoom(r.grid, 2) for r in rooms], L, cell_size, seed, 0, True)
    eng = Engine(n, rooms, local_map_length=L, seed=seed, env_kind=_lib.ENV_SIMPLE, cell_size=cell_size)
    assert eng.lanes_per_env == (2 if L == 16 else 1)
    dev, d = eng.device, eng.obs_dim
    obs = eng.reset()
    assert np.array_equal(obs.cpu().numpy().view(np.uint32), ov.reset().view(np.uint32))
    rew, r64 = torch.zeros(n, device=dev), torch.zeros(n, dtype=torch.float64, device=dev)
    te, tr = torch.zeros(n, dtype=torch.uint8, device=dev), torch.zeros(n, dtype=torch.uint8, device=dev)
    tobs = torch.zeros((n, d), device=dev)
    rng = np.random.default_rng(seed)
    n_done = 0
    for t in range(steps):
        a = rng.integers(0, 6, size=n)
        ov.step(a)
        eng.step(torch.as_tensor(a).to(dev), obs, rew, te, tr, reward64=r64, terminal_obs=tobs)
        assert np.array_equal(obs.cpu().numpy().view(np.uint32), ov.obs.view(np.uint32)), t
        assert np.array_equal(r64.cpu().numpy(), ov.reward), t
        assert np.array_equal(te.cpu().numpy(), ov.terminated) and np.array_equal(tr.cpu().numpy(), ov.truncated), t
        done = (ov.terminated | ov.truncated).astype(bool)
        assert np.array_equal(tobs.cpu().numpy()[done].view(np.uint32), ov.terminal_obs[done].view(np.uint32)), t
        n_done += int(done.sum())
    assert n_done > 0

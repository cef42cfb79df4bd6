"""Engine.rollout_actions (nav3d_rollout_actions) on the GPU: one call equals T nav3d_step calls with the same action rows,
bit for bit — every output row, the rows left untouched, the final records and env-state blobs of every env."""
import ctypes as C

import numpy as np
import pytest

from conftest import ROOMS
from nav3d.rooms import load_room_dir, load_room_file

pytestmark = pytest.mark.gpu
SENTINEL = 0x7F


def p1_rooms():
    return load_room_dir(ROOMS / "P1_training", sort=True)


def short_episode_rooms():
    """P2/P3 rooms with tightcorridor (302 free cells) and maze_3d_tunnels (149): several auto-resets per env per launch."""
    return (load_room_dir(ROOMS / "P3_training", sort=True)[:6] + load_room_dir(ROOMS / "P2_training", sort=True)[:4]
            + [load_room_file(ROOMS / "P2_training" / "tightcorridor.txt"),
               load_room_file(ROOMS / "P3_training" / "maze_3d_tunnels.txt")])


def engine(n, rooms, L=10, seed=0, lanes=0, auto_reset=True, **kw):
    from nav3d import Engine
    return Engine(n, rooms, local_map_length=L, seed=seed, lanes_per_env=lanes, auto_reset=auto_reset, **kw)


class Stepper:
    """An engine with nav3d_step's own output buffers."""

    def __init__(self, eng):
        import torch
        self.eng, n, dev = eng, eng.n_envs, eng.device
        self.obs = eng.reset()
        self.rew = torch.zeros(n, device=dev)
        self.rew64 = torch.zeros(n, dtype=torch.float64, device=dev)
        self.te = torch.zeros(n, dtype=torch.uint8, device=dev)
        self.tr = torch.zeros(n, dtype=torch.uint8, device=dev)
        self.tobs = torch.zeros((n, 80), device=dev)
        self.eps = torch.zeros((n, 8), dtype=torch.int32, device=dev)

    def step(self, a):
        self.eng.step(a.long(), self.obs, self.rew, self.te, self.tr, reward64=self.rew64, terminal_obs=self.tobs,
                      episodes=self.eps)

    def blobs(self, obs):
        import torch
        out = torch.zeros((self.eng.n_envs, self.eng.env_state_bytes), dtype=torch.uint8, device=self.eng.device)
        return self.eng.save_envs(torch.arange(self.eng.n_envs, dtype=torch.int32, device=self.eng.device), obs, out=out)


def rollout_buffers(T, n, dev, outputs="all"):
    import torch
    full = outputs == "all"
    want = lambda k: full or k in outputs   # noqa: E731
    b = dict(obs=None, obs_last=None, reward=None, reward64=None, terminated=None, truncated=None, terminal_obs=None,
             episodes=None)
    if want("obs"):
        b["obs"] = torch.full((T, n, 80), float("nan"), device=dev)
    else:
        b["obs_last"] = torch.full((n, 80), float("nan"), device=dev)
    if want("reward"):
        b["reward"] = torch.zeros((T, n), device=dev)
    if want("reward64"):
        b["reward64"] = torch.zeros((T, n), dtype=torch.float64, device=dev)
    if want("flags"):
        b["terminated"] = torch.full((T, n), 9, dtype=torch.uint8, device=dev)
        b["truncated"] = torch.full((T, n), 9, dtype=torch.uint8, device=dev)
    if want("tobs"):
        b["terminal_obs"] = torch.full((T, n, 320), SENTINEL, dtype=torch.uint8, device=dev).view(torch.float32)
    if want("eps"):
        b["episodes"] = torch.full((T, n, 32), SENTINEL, dtype=torch.uint8, device=dev).view(torch.int32)
    return b


def check_equivalence(rooms, n, T, L=10, seed=0, lanes=0, auto_reset=True, pre_steps=30, a_hi=256, outputs="all"):
    """Engine A runs rollout_actions, engine B (same config) T nav3d_step calls with the same rows.  Returns the number of
    episode ends inside the rollout per env."""
    import torch
    A, B = Stepper(engine(n, rooms, L, seed, lanes, auto_reset)), Stepper(engine(n, rooms, L, seed, lanes, auto_reset))
    dev = A.eng.device
    g = torch.Generator(device="cpu").manual_seed(seed)
    for _ in range(pre_steps):
        a = torch.randint(0, 6, (n,), generator=g).to(dev)
        A.step(a)
        B.step(a)
    acts = torch.randint(0, a_hi, (T, n), generator=g, dtype=torch.uint8).to(dev)
    buf = rollout_buffers(T, n, dev, outputs)
    launches = A.eng.launch_count
    A.eng.rollout_actions(acts, **buf)
    assert A.eng.launch_count == launches + 1
    ends = torch.zeros(n, dtype=torch.int64, device=dev)
    u32 = lambda x: x.view(torch.int32)   # noqa: E731  (bit-exact float comparison)
    for t in range(T):
        B.step(acts[t])
        done = (B.te | B.tr) != 0
        ends += done
        reset = done & auto_reset
        tag = f"t={t}"
        if buf["obs"] is not None:
            assert torch.equal(u32(buf["obs"][t]), u32(B.obs)), f"{tag}: obs"
        if buf["reward"] is not None:
            assert torch.equal(u32(buf["reward"][t]), u32(B.rew)), f"{tag}: reward"
        if buf["reward64"] is not None:
            assert torch.equal(buf["reward64"][t].view(torch.int64), B.rew64.view(torch.int64)), f"{tag}: reward64"
        if buf["terminated"] is not None:
            assert torch.equal(buf["terminated"][t], B.te) and torch.equal(buf["truncated"][t], B.tr), f"{tag}: flags"
        if buf["terminal_obs"] is not None:
            rows = buf["terminal_obs"][t].view(torch.uint8)
            assert torch.equal(u32(buf["terminal_obs"][t][reset]), u32(B.tobs[reset])), f"{tag}: terminal_obs"
            assert bool((rows[~reset] == SENTINEL).all()), f"{tag}: terminal_obs row of an env that did not reset written"
        if buf["episodes"] is not None:
            rows = buf["episodes"][t].view(torch.uint8)
            assert torch.equal(buf["episodes"][t][done], B.eps[done]), f"{tag}: episodes"
            assert bool((rows[~done] == SENTINEL).all()), f"{tag}: episodes row of an env that did not finish written"
    last = buf["obs"][-1] if buf["obs"] is not None else buf["obs_last"]
    assert torch.equal(u32(last), u32(B.obs)), "last observation"
    assert torch.equal(A.eng.get_state(), B.eng.get_state()), "final records"
    assert torch.equal(A.blobs(last.contiguous()), B.blobs(B.obs)), "env-state blobs of every env"
    for i in (0, n // 2, n - 1):
        assert np.array_equal(A.eng.get_grid(i), B.eng.get_grid(i)), f"knowledge grid of env {i}"
    return ends.cpu().numpy()


@pytest.mark.parametrize("lanes", [1, 2, 4, 8, 16, 32])
def test_equals_steps_every_lane_width_p1_ragged(lanes):
    check_equivalence(p1_rooms(), n=1013, T=24, seed=lanes, lanes=lanes)


@pytest.mark.parametrize("lanes", [0, 4])
def test_equals_steps_with_several_resets_per_launch(lanes):
    """Two large P3 rooms next to maze_3d_tunnels and tightcorridor, which truncate after 149 and 302 steps: a quarter of
    the resets land in the maze, so within 460 steps many envs end two or three episodes.  (The C oracle, replaying the
    same seed and actions, counts 194 envs with two or more ends and at most three.)"""
    rooms = (load_room_dir(ROOMS / "P3_training", sort=True)[:2]
             + [load_room_file(ROOMS / "P2_training" / "tightcorridor.txt"),
                load_room_file(ROOMS / "P3_training" / "maze_3d_tunnels.txt")])
    ends = check_equivalence(rooms, n=1013, T=460, seed=11, lanes=lanes, pre_steps=0)
    assert (ends >= 2).sum() >= 100 and ends.max() >= 3


@pytest.mark.parametrize("lanes", [0, 8])
def test_equals_steps_without_auto_reset(lanes):
    rooms = [load_room_file(ROOMS / "P3_training" / "maze_3d_tunnels.txt"), load_room_file(ROOMS / "P2_training" / "tightcorridor.txt")]
    ends = check_equivalence(rooms, n=300, T=360, seed=3, lanes=lanes, auto_reset=False, pre_steps=0)
    assert ends.max() > 1                    # envs keep stepping past done


@pytest.mark.parametrize("outputs", [("reward",), ("flags", "eps"), ("reward64", "tobs"), ("obs",), ("obs", "eps")])
@pytest.mark.parametrize("lanes", [0, 4])
def test_obs_last_and_null_outputs(outputs, lanes):
    check_equivalence(short_episode_rooms(), n=517, T=330, seed=7, lanes=lanes, outputs=outputs, pre_steps=0)


def replay_random(eng, obs, T, t0):
    """rollout_random from the current state, then the same state replayed through rollout_actions(actions_out)."""
    import torch
    n, dev = eng.n_envs, eng.device
    ids = torch.arange(n, dtype=torch.int32, device=dev)
    blobs = eng.save_envs(ids, obs)
    o1 = torch.empty((T, n, 80), device=dev)
    r1 = torch.empty((T, n), device=dev)
    d1 = torch.empty((T, n), dtype=torch.uint8, device=dev)
    acts = torch.empty((T, n), dtype=torch.uint8, device=dev)
    eng.rollout_random(T, t0, obs=o1, reward=r1, done=d1, actions_out=acts)
    after = eng.get_state()
    eng.load_envs(ids, blobs, obs, check=False)
    o2 = torch.empty_like(o1)
    r2 = torch.empty_like(r1)
    te = torch.empty_like(d1)
    tr = torch.empty_like(d1)
    eng.rollout_actions(acts, obs=o2, reward=r2, terminated=te, truncated=tr)
    assert torch.equal(o1.view(torch.int32), o2.view(torch.int32)), "obs"
    assert torch.equal(r1.view(torch.int32), r2.view(torch.int32)), "reward"
    assert torch.equal(d1, te | tr), "done"
    assert torch.equal(after, eng.get_state()), "final records"
    obs.copy_(o2[-1])
    return int(d1.sum())


@pytest.mark.parametrize("lanes", [0, 4])
def test_replays_a_random_rollout(lanes):
    eng = engine(1013, short_episode_rooms(), seed=4, lanes=lanes)
    obs = eng.reset()
    assert replay_random(eng, obs, 350, 0) > 0


def test_replays_a_random_rollout_at_full_size():
    """2^20 envs of P1_training, T = 32, every observation written, two launches in a row."""
    eng = engine(1 << 20, p1_rooms(), seed=1)
    obs = eng.reset()
    replay_random(eng, obs, 32, 0)
    replay_random(eng, obs, 32, 32)


def test_branching_from_one_saved_env():
    """One env of a running engine cloned into k envs of a planning engine with the same signature, k different
    sequences: each branch equals a stepwise replay of its sequence."""
    import torch
    rooms = short_episode_rooms()
    src = Stepper(engine(64, rooms, seed=2))
    g = torch.Generator(device="cpu").manual_seed(0)
    for _ in range(60):
        src.step(torch.randint(0, 6, (64,), generator=g).to(src.eng.device))
    blob = src.eng.save_envs([5], src.obs)
    k, T = 16, 200
    plan, ref = engine(k, rooms, seed=9, lanes=4), Stepper(engine(k, rooms, seed=9))
    dev = plan.device
    pobs = plan.new_obs()
    plan.load_envs(range(k), blob[[0] * k], pobs)
    ref.eng.load_envs(range(k), blob[[0] * k], ref.obs)
    seqs = torch.randint(0, 6, (T, k), generator=g, dtype=torch.uint8).to(dev)
    o = torch.empty((T, k, 80), device=dev)
    r = torch.empty((T, k), dtype=torch.float64, device=dev)
    te = torch.empty((T, k), dtype=torch.uint8, device=dev)
    tr = torch.empty((T, k), dtype=torch.uint8, device=dev)
    plan.rollout_actions(seqs, obs=o, reward64=r, terminated=te, truncated=tr)
    for t in range(T):
        ref.step(seqs[t])
        assert torch.equal(o[t].view(torch.int32), ref.obs.view(torch.int32)), f"t={t}: obs"
        assert torch.equal(r[t], ref.rew64) and torch.equal(te[t], ref.te) and torch.equal(tr[t], ref.tr), f"t={t}"
    assert torch.equal(plan.get_state(), ref.eng.get_state())
    assert len({tuple(x) for x in plan.get_state()[:, :3].cpu().numpy().tolist()}) > 1     # the branches diverged


def test_cuda_graph_capture_equals_eager():
    import torch
    eng = engine(2048, short_episode_rooms(), seed=6)
    obs = eng.reset()
    dev, n, T = eng.device, 2048, 64
    g = torch.Generator(device="cpu").manual_seed(1)
    ids = torch.arange(n, dtype=torch.int32, device=dev)
    blobs = eng.save_envs(ids, obs)
    acts = torch.randint(0, 6, (T, n), generator=g, dtype=torch.uint8).to(dev)
    buf = rollout_buffers(T, n, dev)

    def snap():
        torch.cuda.synchronize()
        return [x.clone() for x in buf.values() if x is not None] + [eng.get_state()]
    eng.rollout_actions(acts, **buf)
    want = snap()
    eng.load_envs(ids, blobs, obs, check=False)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        eng.rollout_actions(acts, **buf)
    for rep in range(2):
        eng.load_envs(ids, blobs, obs, check=False)
        for x in buf.values():
            if x is not None:
                x.view(torch.uint8).fill_(SENTINEL)
        graph.replay()
        got = snap()
        for k, (w, v) in enumerate(zip(want, got)):
            assert torch.equal(w.view(torch.uint8), v.view(torch.uint8)), f"replay {rep}: output {k} differs from eager"


def test_errors_and_launch_count():
    import torch
    from nav3d import Nav3dError, _lib
    eng = engine(64, p1_rooms())
    acts = torch.zeros((4, 64), dtype=torch.uint8, device=eng.device)
    with pytest.raises(Nav3dError, match="reset") as ei:
        eng.rollout_actions(acts, obs_last=eng.new_obs())
    assert ei.value.code == -1
    simple = engine(64, load_room_dir(ROOMS / "P3_training", sort=True, simple=True)[:3], L=4, env_kind=_lib.ENV_SIMPLE)
    simple.reset()
    with pytest.raises(Nav3dError) as ei:
        simple.rollout_actions(acts, obs_last=torch.zeros((64, simple.obs_dim), device=eng.device))
    assert ei.value.code == -2
    obs = eng.reset()
    st, before = eng.get_state(), eng.launch_count
    rc = eng._lib.nav3d_rollout_actions(eng._h, 0, C.c_void_p(acts.data_ptr()), None, C.c_void_p(obs.data_ptr()),
                                        None, None, None, None, None, None, None)
    assert rc == 0 and eng.launch_count == before and torch.equal(eng.get_state(), st)
    eng.rollout_actions(acts[:0], obs_last=obs)
    assert eng.launch_count == before + 1 and torch.equal(eng.get_state(), st)      # (+1: the get_state above)
    eng.rollout_actions(acts.long() + 3, obs_last=obs)          # int64 rows: clamped to 0..5 on the device
    assert eng.launch_count == before + 3                       # get_state + one rollout (the clamp is torch's)
    with pytest.raises(ValueError):
        eng.rollout_actions(acts)                               # neither obs nor obs_last
    with pytest.raises(ValueError):
        eng.rollout_actions(acts[:, :32].contiguous(), obs_last=obs)
    with pytest.raises(ValueError):
        eng.rollout_actions(acts, obs=torch.zeros((3, 64, 80), device=eng.device))


def test_vec_env_step_sequence_equals_steps():
    import torch
    from nav3d import BatchedCubicEnv
    kw = dict(rooms=short_episode_rooms(), num_envs=300, local_map_length=10, seed=5)
    a_env, b_env = BatchedCubicEnv(**kw), BatchedCubicEnv(**kw)
    a_env.reset()
    b_env.reset()
    acts = torch.randint(0, 6, (320, 300), generator=torch.Generator().manual_seed(3))
    obs, rew, dones, info = a_env.step_sequence(acts)
    assert obs.shape == (320, 300, 80) and dones.dtype == torch.bool and info.episodes.shape == (320, 300, 8)
    for t in range(320):
        o, r, d, i = b_env.step(acts[t])
        assert torch.equal(obs[t].view(torch.int32), o.view(torch.int32)) and torch.equal(rew[t], r) and torch.equal(dones[t], d)
        assert torch.equal(info[t].terminated, i.terminated) and torch.equal(info[t].truncated, i.truncated)
        assert torch.equal(info[t].terminal_observation[d], i.terminal_observation[d])
        assert torch.equal(info[t].episodes[d], i.episodes[d])
    assert int(dones.sum()) > 0
    assert [x["episode"]["l"] for x in a_env.sb3_infos(info[319]) if "episode" in x] == \
        [x["episode"]["l"] for x in b_env.sb3_infos(i) if "episode" in x]
    assert torch.equal(a_env._obs, obs[-1])
    more = torch.randint(0, 6, (300,), generator=torch.Generator().manual_seed(4))
    assert torch.equal(a_env.step(more)[0], b_env.step(more)[0])      # step() continues from where step_sequence left off

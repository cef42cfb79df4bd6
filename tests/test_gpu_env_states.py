"""Env-state blobs on the GPU: Engine.save_envs / Engine.load_envs (nav3d_save_envs / nav3d_load_envs) through the C ABI.
Every comparison is bit-exact: integer state, knowledge grids, observation rows (as u32), f64 and f32 rewards, flags."""
import ctypes as C

import numpy as np
import pytest

from conftest import ROOMS
from nav3d.rooms import load_room_dir, load_room_file

pytestmark = pytest.mark.gpu


class GpuBlobs:
    """nav3d.Engine with numpy views of its outputs, as tests/env_state_checks.py drives it."""

    def __init__(self, n, rooms, L=10, seed=0, env_id0=0, auto_reset=True, lanes=0, simple=False):
        import torch
        from nav3d import Engine, _lib
        self.n = n
        self.eng = Engine(n, rooms, local_map_length=L, auto_reset=auto_reset, seed=seed, env_id0=env_id0,
                          lanes_per_env=lanes, env_kind=_lib.ENV_SIMPLE if simple else _lib.ENV_CUBIC)
        dev, d = self.eng.device, self.eng.obs_dim
        self.d_obs = torch.full((n, d), float("nan"), dtype=torch.float32, device=dev)
        self.d_reward = torch.zeros(n, dtype=torch.float32, device=dev)
        self.d_reward64 = torch.zeros(n, dtype=torch.float64, device=dev)
        self.d_term = torch.zeros(n, dtype=torch.uint8, device=dev)
        self.d_trunc = torch.zeros(n, dtype=torch.uint8, device=dev)
        self.d_tobs = torch.zeros((n, d), dtype=torch.float32, device=dev)
        self.d_eps = torch.zeros((n, 8), dtype=torch.int32, device=dev)
        self._pull()

    def _pull(self):
        self.obs = self.d_obs.cpu().numpy()
        self.reward = self.d_reward.cpu().numpy()
        self.reward64 = self.d_reward64.cpu().numpy()
        self.term = self.d_term.cpu().numpy()
        self.trunc = self.d_trunc.cpu().numpy()
        self.tobs = self.d_tobs.cpu().numpy()
        self.eps = self.d_eps.cpu().numpy()

    def reset(self, picks=None):
        import torch
        self.eng.reset(self.d_obs, picks=None if picks is None else torch.as_tensor(np.asarray(picks, np.int32)))
        self._pull()

    def step(self, actions):
        import torch
        a = torch.as_tensor(np.asarray(actions, dtype=np.int64)).to(self.eng.device)
        self.eng.step(a, self.d_obs, self.d_reward, self.d_term, self.d_trunc, reward64=self.d_reward64,
                      terminal_obs=self.d_tobs, episodes=self.d_eps)
        self._pull()

    def state(self):
        return self.eng.get_state().cpu().numpy()

    def grid(self, env):
        return self.eng.get_grid(env)

    def save(self, ids):
        return self.eng.save_envs(ids, self.d_obs)

    def load(self, ids, blobs):
        self.eng.load_envs(ids, blobs, self.d_obs)          # check=True: raises unless every blob loaded
        self._pull()
        return np.zeros(len(ids), np.uint8)

    @staticmethod
    def take(blobs, idx):
        import torch
        return blobs[torch.as_tensor(np.asarray(idx, np.int64), device=blobs.device)]

    def raw_load(self, ids, blobs):
        """nav3d_load_envs with a status array, no Python-side checks."""
        import torch
        from nav3d.engine import _ptr
        ids = torch.as_tensor(np.asarray(ids, np.int32), device=self.eng.device)
        status = torch.full((len(ids),), 255, dtype=torch.uint8, device=self.eng.device)
        rc = self.eng._lib.nav3d_load_envs(self.eng._h, _ptr(ids), len(ids), _ptr(blobs), _ptr(self.d_obs), _ptr(status),
                                           C.c_void_p(torch.cuda.current_stream().cuda_stream))
        assert rc == 0
        self._pull()
        return status.cpu().numpy()


def p3_rooms(simple=False):
    return load_room_dir(ROOMS / "P3_training", sort=True, simple=simple)


def starts_of(rooms):
    """Per room: the start cell of every free-cell index k (the room's fixed start if it has a usable one)."""
    out = []
    for r in rooms:
        fc = r.free_cells()
        st = getattr(r, "start", None)
        if st is not None and all(0 <= st[i] < r.grid.shape[i] for i in range(3)) and r.grid[tuple(st)] != r.wall_code:
            fc = np.repeat(np.asarray([st]), len(fc), axis=0)
        out.append(fc)
    return out


@pytest.mark.parametrize("lanes", [0, 4])
def test_round_trip_replays_bit_for_bit(lanes):
    """512 envs of P3_training (kitchen2 and the open-shell mazes), a random third saved after 130 steps, 130 steps
    recorded, loaded back, replayed: the loaded envs repeat every output, their auto-resets included."""
    from env_state_checks import round_trip
    e = GpuBlobs(512, p3_rooms(), L=10, seed=3, lanes=lanes)
    assert round_trip(e, 7) > 0


def test_clone_broadcast_matches_oracle(oracle):
    from env_state_checks import clone
    rooms = p3_rooms()
    n, L, seed = 64, 10, 5
    e = GpuBlobs(n, rooms, L=L, seed=seed)
    orooms = [oracle.OracleRoom(r.grid, -2) for r in rooms]
    ov = oracle.OracleVec(n, orooms, L, -2.0, seed, 0, True)
    nf = [r.n_free for r in orooms]
    assert nf == e.eng.room_free
    clone(e, 11, nf, starts_of(rooms), lambda env, ep: oracle.pick(seed, env, ep, nf), oracle_vec=ov)


def test_across_engines_and_lane_widths():
    """Saved on a lanes=1 engine (seed 1), loaded into a lanes=4 engine with another seed, n_envs and env_id0."""
    from env_state_checks import outputs
    rooms = p3_rooms()
    src = GpuBlobs(96, rooms, L=10, seed=1, lanes=1)
    dst = GpuBlobs(50, rooms, L=10, seed=2, env_id0=1000, lanes=4)
    assert src.eng.env_state_bytes == dst.eng.env_state_bytes
    rng = np.random.default_rng(0)
    src.reset()
    dst.reset()
    for _ in range(100):
        src.step(rng.integers(0, 6, size=96))
        dst.step(rng.integers(0, 6, size=50))
    s_ids = np.arange(0, 64, 2, dtype=np.int32)
    d_ids = np.arange(10, 42, dtype=np.int32)
    dst.load(d_ids, src.save(s_ids))
    assert np.array_equal(dst.state()[d_ids], src.state()[s_ids])
    assert np.array_equal(dst.obs[d_ids].view(np.uint32), src.obs[s_ids].view(np.uint32))
    for i, j in zip(s_ids, d_ids):
        assert np.array_equal(dst.grid(int(j)), src.grid(int(i))), f"grid of src {i} / dst {j}"
    alive = np.ones(len(s_ids), bool)
    for t in range(200):
        a = rng.integers(0, 6, size=96)
        b = rng.integers(0, 6, size=50)
        b[d_ids] = a[s_ids]
        src.step(a)
        dst.step(b)
        o_s, o_d = outputs(src, s_ids), outputs(dst, d_ids)
        ended = (src.term[s_ids] | src.trunc[s_ids]) != 0
        for k in o_s:
            if k in ("state", "obs"):            # the reset after an episode end draws from the destination's stream
                sel = alive & ~ended
            else:
                sel = alive
            assert np.array_equal(o_s[k][sel], o_d[k][sel]), f"t={t}: {k} differs"
        alive &= ~ended
    assert alive.sum() < len(alive)              # some pairs reached their reset


@pytest.mark.parametrize("lanes", [0, 8])
def test_live_part_across_room_sizes(lanes):
    from edge_rooms import degenerate_rooms
    from env_state_checks import live_part
    rooms = [load_room_file(ROOMS / "P3_training" / "maze_7x7_seed22.txt"), degenerate_rooms()[3],
             load_room_file(ROOMS / "P3_training" / "kitchen2.txt"), load_room_file(ROOMS / "P2_training" / "tightcorridor.txt")]
    sizes = [r.grid.size for r in rooms]
    assert sizes[2] == max(sizes) and sizes[1] == min(sizes)
    e = GpuBlobs(8, rooms, L=10, seed=1, auto_reset=False, lanes=lanes)
    live_part(e, np.array([[r, 0] for r in range(4)] * 2, np.int32))


def test_simple_env_round_trip_and_clone(oracle):
    from env_state_checks import clone, round_trip
    rooms = [load_room_file(ROOMS / "P3_training" / n, simple=True) for n in ("maze_3d_tunnels.txt", "kitchen2.txt",
                                                                                 "maze_7x7_seed22.txt")]
    e = GpuBlobs(96, rooms, L=4, seed=2, simple=True)
    assert e.eng.obs_dim == 31
    round_trip(e, 3)
    nf = [len(r.free_cells()) for r in rooms]
    e = GpuBlobs(32, rooms, L=4, seed=4, simple=True)
    clone(e, 9, nf, [r.free_cells() for r in rooms], lambda env, ep: oracle.pick3(4, env, ep, nf), simple=True)


def test_rejection():
    import torch
    from nav3d import Engine, Nav3dError
    rooms = p3_rooms()[:6]
    e = GpuBlobs(16, rooms, L=10, seed=1)
    e.reset()
    rng = np.random.default_rng(1)
    for _ in range(20):
        e.step(rng.integers(0, 6, size=16))
    B = e.eng.env_state_bytes

    def foreign(g):
        g.reset()
        g.step(np.ones(g.n, np.int64))
        blob = g.save([0])
        buf = torch.zeros((1, B), dtype=torch.uint8, device=blob.device)
        m = min(B, blob.shape[1])
        buf[:, :m] = blob[:, :m]
        return buf
    cases = {
        "other L": foreign(GpuBlobs(4, rooms, L=4)),
        "other rooms": foreign(GpuBlobs(4, p3_rooms()[1:7], L=10)),
        "other kind": foreign(GpuBlobs(4, p3_rooms(simple=True)[:6], L=10, simple=True)),
        "zeroed": torch.zeros((1, B), dtype=torch.uint8, device=e.eng.device),
        "out-of-range id": e.save([16 + 5]),
    }
    for name, blob in cases.items():
        target = 3
        st0, g0, o0 = e.state()[target].copy(), e.grid(target), e.obs[target].copy()
        status = e.raw_load([target], blob)
        assert status.tolist() == [2], f"{name}: status {status}"
        assert np.array_equal(e.state()[target], st0) and np.array_equal(e.grid(target), g0), f"{name}: env changed"
        assert np.array_equal(e.obs[target].view(np.uint32), o0.view(np.uint32)), f"{name}: obs row changed"
        with pytest.raises(Nav3dError, match="not a valid blob"):
            e.eng.load_envs([target], blob, e.d_obs)
    good = e.save([0, 1])
    st0 = e.state()
    with pytest.raises(Nav3dError, match="out of range"):
        e.eng.load_envs([2, 16], good, e.d_obs)
    with pytest.raises(Nav3dError, match="distinct"):
        e.eng.load_envs([2, 2], good, e.d_obs)
    assert np.array_equal(e.state(), st0), "a rejected id list must change nothing"
    assert e.raw_load([2, 99], good).tolist() == [0, 1]
    with pytest.raises(ValueError):
        e.eng.load_envs([2, 3], good.float(), e.d_obs)
    with pytest.raises(ValueError):
        e.eng.load_envs([2, 3], good[:, :-16].contiguous(), e.d_obs)
    with pytest.raises(ValueError):
        e.eng.load_envs([2], good, e.d_obs)
    with pytest.raises(ValueError):
        e.eng.load_envs([2, 3], good, e.d_obs[:8])
    with pytest.raises(ValueError):
        e.eng.save_envs([2, 3], e.d_obs, out=torch.empty((2, B - 16), dtype=torch.uint8, device=e.eng.device))
    with pytest.raises(ValueError):
        e.eng.save_envs([2, 3], e.d_obs.double())
    fresh = Engine(4, rooms, local_map_length=10)
    with pytest.raises(Nav3dError, match="reset"):
        fresh.save_envs([0], fresh.new_obs())


def test_cuda_graph_load_then_steps():
    """load_envs(check=False) followed by 8 steps, captured once and replayed twice: each replay equals the eager run."""
    import torch
    from nav3d import Engine
    rooms = load_room_dir(ROOMS / "P1_training", sort=True)
    n, T = 256, 8
    eng = Engine(n, rooms, local_map_length=10, seed=9)
    dev = eng.device
    obs = eng.reset()
    rng = np.random.default_rng(2)
    rew = torch.zeros(n, device=dev)
    te = torch.zeros(n, dtype=torch.uint8, device=dev)
    tr = torch.zeros(n, dtype=torch.uint8, device=dev)
    for _ in range(40):
        eng.step(torch.as_tensor(rng.integers(0, 6, size=n), device=dev), obs, rew, te, tr)
    ids = torch.arange(0, n, 2, dtype=torch.int32, device=dev)
    blobs = eng.save_envs(ids, obs)
    acts = torch.as_tensor(rng.integers(0, 6, size=(T, n)), device=dev)
    o_t = torch.zeros((T, n, 80), device=dev)
    r_t = torch.zeros((T, n), dtype=torch.float64, device=dev)
    r32 = torch.zeros((T, n), device=dev)
    te_t = torch.zeros((T, n), dtype=torch.uint8, device=dev)
    tr_t = torch.zeros((T, n), dtype=torch.uint8, device=dev)
    tobs = torch.zeros((n, 80), device=dev)

    def body():
        eng.load_envs(ids, blobs, obs, check=False)
        for t in range(T):
            eng.step(acts[t], o_t[t], r32[t], te_t[t], tr_t[t], reward64=r_t[t], terminal_obs=tobs)

    def snap():
        torch.cuda.synchronize()
        i = ids.long()
        return [x[:, i].cpu().numpy().copy() for x in (o_t.view(torch.int32), r_t, r32.view(torch.int32), te_t, tr_t)] + \
            [eng.get_state()[i].cpu().numpy()]
    body()
    want = snap()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        body()
    for rep in range(2):
        for x in (o_t, r_t, r32, te_t, tr_t):
            x.zero_()
        g.replay()
        got = snap()
        for k, (w, v) in enumerate(zip(want, got)):
            assert np.array_equal(w, v), f"replay {rep}: output {k} differs from the eager run"

"""Per-room episode statistics on the GPU (include/nav3d.h nav3d_room_stats) and the learning-progress room curriculum of
RecurrentPPO (nav3d/curriculum.py).

The kernel must equal tests/room_stats_ref.py bit for bit on both sides of its shared-memory cut-over (256 rooms), at every
flag alignment, with garbage in every row that is not flagged done; on real engine output; inside a CUDA graph.  The trainer
must install exactly the table of the weights the float64 rule gives for the window it read."""
import ctypes
import functools

import numpy as np
import pytest
import torch

from conftest import ROOMS
import room_stats_ref as ref
import room_weights_ref as rw

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)


@functools.lru_cache(maxsize=4)
def engine_for(n_rooms, n_envs):
    from edge_rooms import degenerate_rooms
    from nav3d import Engine
    return Engine(n_envs, [degenerate_rooms()[0]] * n_rooms, local_map_length=4, seed=0)


def dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).to(DEV)


def check_equal(got, want, tag):
    got = got.cpu().numpy()
    if not np.array_equal(got, want):
        bad = np.nonzero((got != want).any(axis=1))[0]
        raise AssertionError(f"{tag}: rooms {bad[:8].tolist()} differ: got {got[bad[:2]].tolist()} want {want[bad[:2]].tolist()}")


GRID = [(R, T, N, d) for R in (1, 2, 5, 257, 4096, 65535) for T in (1, 7, 32) for N in (1, 31, 4099)
        for d in (0.0, 1e-3, 0.5, 1.0)]
BIG = [(R, T, (1 << 20) + 3, d) for R in (5, 257, 65535) for T in (1, 32) for d in (1e-3, 1.0)] + [(5, 32, (1 << 20) + 3, 0.0)]


@pytest.mark.parametrize("R,T,N,d", GRID + BIG)
def test_kernel_equals_reference(R, T, N, d):
    rng = np.random.default_rng(R * 1000003 + T * 101 + N + int(d * 1000))
    te, tr, ep = ref.random_rows(rng, T, N, R, d)
    want, bad = ref.room_stats_ref(te, tr, ep, R)
    assert not bad
    eng = engine_for(R, N)
    tt, rr, ee = dev(te), dev(tr), dev(ep)
    got = eng.room_stats(tt if T > 1 else tt[0], rr if T > 1 else rr[0], ee if T > 1 else ee[0], check=True)
    check_equal(got, want, f"R={R} T={T} N={N} d={d}")
    eng.room_stats(tt, rr, ee, out=got)                      # accumulates, never zeroes
    check_equal(got, 2 * want, "second call")


@pytest.mark.parametrize("R", [1, 5, 257, 65535])
@pytest.mark.parametrize("room", ["first", "last"])
def test_every_row_done_in_one_room(R, room):
    rng = np.random.default_rng(R)
    T, N = 32, 1 << 16
    te, tr, ep = ref.random_rows(rng, T, N, R, 1.0)
    ep[..., 5] = 0 if room == "first" else R - 1
    want, _ = ref.room_stats_ref(te, tr, ep, R)
    assert want[ep[0, 0, 5], 0] == T * N
    check_equal(engine_for(R, N).room_stats(dev(te), dev(tr), dev(ep), check=True), want, f"one room R={R}")


@pytest.mark.parametrize("R", [5, 4096])
def test_every_flag_and_episode_alignment(R):
    """Flag views at every byte offset mod 16 (terminated and truncated at equal and at different offsets), episode views
    at 16-byte and at 4-byte-only offsets."""
    rng = np.random.default_rng(7)
    T, N = 7, 4099
    M = T * N
    eng = engine_for(R, N)
    te, tr, ep = ref.random_rows(rng, T, N, R, 0.5)
    want, _ = ref.room_stats_ref(te, tr, ep, R)
    buf_t = torch.zeros(M + 64, dtype=torch.uint8, device=DEV)
    buf_r = torch.zeros(M + 64, dtype=torch.uint8, device=DEV)
    buf_e = torch.zeros(M * 8 + 8, dtype=torch.int32, device=DEV)
    for eoff in (0, 1, 2, 3):
        e_view = buf_e[eoff:eoff + M * 8].view(T, N, 8)
        e_view.copy_(dev(ep))
        for ot in range(16):
            for orr in sorted({ot, (ot + 5) % 16}):
                t_view = buf_t[ot:ot + M].view(T, N)
                r_view = buf_r[orr:orr + M].view(T, N)
                t_view.copy_(dev(te)); r_view.copy_(dev(tr))
                assert t_view.data_ptr() % 16 == (buf_t.data_ptr() + ot) % 16
                got = eng.room_stats(t_view, r_view, e_view, check=True)
                check_equal(got, want, f"offsets term {ot} trunc {orr} episodes {4 * eoff} bytes")


def test_bad_rows_are_not_counted_and_flag_status():
    from nav3d import Nav3dError
    R, T, N = 5, 3, 300
    rng = np.random.default_rng(3)
    te, tr, ep = ref.random_rows(rng, T, N, R, 0.3)
    flat = ep.reshape(-1, 8)
    done = np.nonzero((te | tr).reshape(-1))[0]
    good, _ = ref.room_stats_ref(te, tr, ep, R)
    eng = engine_for(R, N)
    for i, (col, val) in enumerate(((5, R), (5, -1), (5, 1 << 30), (0, np.float32(np.nan)), (0, np.float32(np.inf)),
                                    (0, np.float32(-np.inf)), (0, np.float32(1e17)))):
        e2 = ep.copy().reshape(-1, 8)
        row = done[i]
        e2[row, col] = np.array([val], np.float32).view(np.int32)[0] if col == 0 else val
        want, bad = ref.room_stats_ref(te, tr, e2.reshape(T, N, 8), R)
        assert bad
        removed = good - want
        assert removed[:, 0].sum() == 1                    # exactly the bad row is missing
        status = torch.full((1,), 7, dtype=torch.uint8, device=DEV)
        out = torch.zeros((R, 8), dtype=torch.int64, device=DEV)
        tt, rr, ee = dev(te), dev(tr), dev(e2)             # kept alive until the kernel has run
        eng._lib.nav3d_room_stats(eng._h, T, ctypes.c_void_p(tt.data_ptr()), ctypes.c_void_p(rr.data_ptr()),
                                  ctypes.c_void_p(ee.data_ptr()), ctypes.c_void_p(out.data_ptr()),
                                  ctypes.c_void_p(status.data_ptr()), None)
        torch.cuda.synchronize()
        assert int(status.item()) == 1
        check_equal(out, want, f"bad row {col}={val}")
        with pytest.raises(Nav3dError, match="not counted"):
            eng.room_stats(dev(te), dev(tr), dev(e2.reshape(T, N, 8)), check=True)
    # good rows only: status 0, also when garbage sits in the rows that are not flagged
    status = torch.full((1,), 7, dtype=torch.uint8, device=DEV)
    out = torch.zeros((R, 8), dtype=torch.int64, device=DEV)
    tt, rr, ee = dev(te), dev(tr), dev(ep)
    assert eng._lib.nav3d_room_stats(eng._h, T, ctypes.c_void_p(tt.data_ptr()), ctypes.c_void_p(rr.data_ptr()),
                                     ctypes.c_void_p(ee.data_ptr()), ctypes.c_void_p(out.data_ptr()),
                                     ctypes.c_void_p(status.data_ptr()), None) == 0
    torch.cuda.synchronize()
    assert int(status.item()) == 0
    check_equal(out, good, "good rows")


def test_invalid_arguments_and_empty_call():
    R, N = 5, 64
    eng = engine_for(R, N)
    lib, P = eng._lib, ctypes.c_void_p
    te = torch.zeros((2, N), dtype=torch.uint8, device=DEV)
    ep = torch.zeros((2, N, 8), dtype=torch.int32, device=DEV)
    out = torch.zeros((R, 8), dtype=torch.int64, device=DEV)
    ok = [P(te.data_ptr()), P(te.data_ptr()), P(ep.data_ptr()), P(out.data_ptr())]
    assert lib.nav3d_room_stats(eng._h, -1, *ok, None, None) == -1
    for k in range(4):
        args = list(ok)
        args[k] = None
        assert lib.nav3d_room_stats(eng._h, 2, *args, None, None) == -1
    assert lib.nav3d_room_stats(None, 2, *ok, None, None) == -1
    before = eng.launch_count
    assert lib.nav3d_room_stats(eng._h, 0, *ok, None, None) == 0
    eng.room_stats(te[:0], te[:0], ep[:0], out=out)
    assert eng.launch_count == before
    eng.room_stats(te, te, ep, out=out)
    assert eng.launch_count == before + 1
    with pytest.raises(ValueError):
        eng.room_stats(te, te, ep[..., :4].contiguous())
    with pytest.raises(ValueError):
        eng.room_stats(te, te, ep, out=torch.zeros((R + 1, 8), dtype=torch.int64, device=DEV))


def engine_rooms():
    from edge_rooms import degenerate_rooms
    from nav3d.rooms import load_room_dir
    return degenerate_rooms() + load_room_dir(ROOMS / "P1_training", sort=True)


def test_rollout_output_per_step_and_lanes():
    from nav3d import Engine
    rooms = engine_rooms()
    R, T, N = len(rooms), 64, 4096
    actions = torch.randint(0, 6, (T, N), dtype=torch.uint8, device=DEV, generator=torch.Generator(DEV).manual_seed(0))
    results = []
    for lanes in (1, 4):
        eng = Engine(N, rooms, local_map_length=10, seed=5, lanes_per_env=lanes)
        obs = eng.reset()
        te = torch.zeros((T, N), dtype=torch.uint8, device=DEV)
        tr = torch.zeros_like(te)
        ep = torch.full((T, N, 8), -7, dtype=torch.int32, device=DEV)      # stale rows hold garbage
        eng.rollout_actions(actions, obs_last=obs, terminated=te, truncated=tr, episodes=ep)
        got = eng.room_stats(te, tr, ep, check=True)
        want, bad = ref.room_stats_ref(te.cpu().numpy(), tr.cpu().numpy(), ep.cpu().numpy(), R)
        assert not bad and (want[:, 0] > 0).sum() >= 2
        check_equal(got, want, f"rollout lanes={lanes}")
        per_step = torch.zeros_like(got)
        for t in range(T):
            eng.room_stats(te[t], tr[t], ep[t], out=per_step)
        assert torch.equal(per_step, got)
        results.append(got)
    assert torch.equal(results[0], results[1])


def test_simple_env_is_accepted():
    from nav3d import BatchedSimpleEnv
    from nav3d.room_tools import generate_room
    from nav3d.rooms import rooms_from_grids
    grids = [np.where(generate_room("empty", s) != 0, 2, 0).astype(np.int8) for s in ((5, 5, 4), (4, 4, 4), (6, 4, 3))]
    env = BatchedSimpleEnv(rooms=rooms_from_grids(grids, wall_code=2), num_envs=512, local_map_length=4, seed=2)
    env.reset()
    R = len(env.engine.rooms)
    acc = torch.zeros((R, 8), dtype=torch.int64, device=DEV)
    want = np.zeros((R, 8), np.int64)
    g = torch.Generator(DEV).manual_seed(1)
    for _ in range(300):
        _, _, _, info = env.step(torch.randint(0, 6, (512,), device=DEV, generator=g))
        env.engine.room_stats(info.terminated, info.truncated, info.episodes, out=acc, check=True)
        want += ref.room_stats_ref(info.terminated.cpu().numpy(), info.truncated.cpu().numpy(),
                                   info.episodes.cpu().numpy(), R)[0]
    assert want[:, 0].sum() > 0
    check_equal(acc, want, "simpleEnv")


def test_graph_replay_accumulates():
    R, T, N = 257, 4, 8192
    eng = engine_for(R, N)
    te, tr, ep = ref.random_rows(np.random.default_rng(11), T, N, R, 0.5)
    want, _ = ref.room_stats_ref(te, tr, ep, R)
    tt, rr, ee = dev(te), dev(tr), dev(ep)
    out = torch.zeros((R, 8), dtype=torch.int64, device=DEV)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        eng.room_stats(tt, rr, ee, out=out)                 # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        eng.room_stats(tt, rr, ee, out=out)
    out.zero_()
    for k in range(1, 4):
        graph.replay()
        torch.cuda.synchronize()
        check_equal(out, k * want, f"replay {k}")


# ---- the trainer ---------------------------------------------------------------------------------------------------------

def curriculum_rooms():
    from edge_rooms import degenerate_rooms
    from nav3d.room_tools import generate_room
    from nav3d.rooms import rooms_from_grids
    return [degenerate_rooms()[0]] + rooms_from_grids([generate_room("empty", (6, 5, 5))])     # 1 and 36 free cells


def make_recording_curriculum(env):
    from nav3d.curriculum import RoomCurriculum

    class Recording(RoomCurriculum):
        def update(self):
            w = self.window.cpu().numpy().copy()
            before = (self.fast.cpu().numpy(), self.slow.cpu().numpy(), self.seen.cpu().numpy())
            p = super().update()
            self.log.append(dict(window=w, before=before, weights=self.weights.cpu().numpy(), p=p.cpu().numpy(),
                                 lp=self.lp.cpu().numpy(), cdf=self.engine.room_cdf().cpu().numpy().astype(np.uint64)))
            return p

    cur = Recording(env)
    cur.log = []
    return cur


def test_trainer_installs_the_rule_and_resumes(tmp_path):
    from nav3d import BatchedCubicEnv
    from nav3d.curriculum import RoomCurriculum
    from nav3d.ppo import RecurrentPPO
    env = BatchedCubicEnv(rooms=curriculum_rooms(), num_envs=256, local_map_length=4, seed=9)
    R = 2
    cur = make_recording_curriculum(env)
    model = RecurrentPPO(env, policy_kwargs=dict(net_arch=dict(pi=[32], vf=[32]), lstm_hidden_size=32), n_steps=64,
                         batch_size=64 * 64, n_epochs=1, seed=0, curriculum=cur)
    model.learn(total_timesteps=3 * 64 * 256)
    assert model._graph is not None, "rollouts 2 and 3 must replay the captured graph"
    assert len(cur.log) == 3
    tf = np.array([1.0, 36.0])
    eps = cur.uniform_mix
    for k, rec in enumerate(cur.log):
        w = rec["window"]
        assert w[0, 0] > 0 and w[1, 0] > 0, "episodes end in both rooms within every rollout"
        assert w[0, 5] == w[0, 0]                            # the one-cell room's score is always 1
        _, _, _, lp, p = ref.lp_rule_ref(w, tf, *rec["before"], cur.alpha_fast, cur.alpha_slow, eps)
        assert np.allclose(rec["p"], p, rtol=1e-12, atol=0)
        assert np.array_equal(rec["weights"], rec["p"].astype(np.float32))
        st, cdf = rw.cdf_build(rec["weights"])
        assert st == 0 and np.array_equal(rec["cdf"], cdf)
        P = np.diff(cdf.astype(np.float64), prepend=0.0) / 2.0 ** 32
        W = rec["weights"].astype(np.float64)
        share = W[0] / W.sum()
        assert abs(P[0] - share) <= (2 + (R - 1) * share) * 2.0 ** -32 + 2.0 ** -52
        target = eps / R if rec["lp"][1] > 0 else 1.0 / R
        assert abs(share - target) <= 1e-7 * target, (k, share, target)
        assert abs(model.logger[k]["curriculum_p_min"] - p.min()) < 1e-12
        assert abs(model.logger[k]["curriculum_p_max"] - p.max()) < 1e-12
    assert cur.log[0]["lp"][1] == 0 and any(r["lp"][1] > 0 for r in cur.log[1:])

    path = model.save(tmp_path / "m.zip")
    sd = cur.state_dict()
    env2 = BatchedCubicEnv(rooms=curriculum_rooms(), num_envs=256, local_map_length=4, seed=9)
    cur2 = RoomCurriculum(env2)
    RecurrentPPO.load(path, env=env2, curriculum=cur2)
    for k, v in cur2.state_dict().items():
        assert (torch.equal(v, sd[k]) if isinstance(v, torch.Tensor) else v == sd[k]), k
    assert torch.equal(env2.engine.room_cdf(), env.engine.room_cdf())
    m3 = RecurrentPPO.load(path, env=BatchedCubicEnv(rooms=curriculum_rooms(), num_envs=256, local_map_length=4, seed=9))
    assert m3.curriculum is None                            # without a curriculum the member is ignored

"""Lock-step differential check shared by the CPU (emulated) and GPU parity tests: an engine-like object is stepped
next to ``oracle.c_oracle.OracleVec`` on identical actions; every output is compared every step."""
import numpy as np


def episode_return_bound(length, ret):
    """include/nav3d.h's bound on |episode_return - sum of the episode's f64 rewards|: 0.005 per rounded term (at most
    five a step plus the finish and truncation terms), the f32 rounding of the result, and 1e-3 of f64 rounding."""
    return 0.005 * (5 * np.asarray(length, np.float64) + 2) + 2.0 ** -24 * np.abs(ret) + 1e-3


def compare_step(tag, t, ov, obs, reward, reward64, term, trunc, tobs, eps, state, crash_penalty=-2.0):
    done = (ov.terminated | ov.truncated).astype(bool)
    assert np.array_equal(term, ov.terminated), f"{tag} t={t}: terminated differs at {np.nonzero(term != ov.terminated)[0][:8]}"
    assert np.array_equal(trunc, ov.truncated), f"{tag} t={t}: truncated differs at {np.nonzero(trunc != ov.truncated)[0][:8]}"
    bad = np.nonzero((obs.view(np.uint32) != ov.obs.view(np.uint32)).any(axis=1))[0]
    if len(bad):
        i = bad[0]
        cols = np.nonzero(obs[i].view(np.uint32) != ov.obs[i].view(np.uint32))[0]
        raise AssertionError(f"{tag} t={t}: obs differs for {len(bad)} envs; env {i} cols {cols[:10]} "
                             f"got {obs[i][cols[:10]]} want {ov.obs[i][cols[:10]]}")
    if reward64 is not None:
        assert np.array_equal(reward64, ov.reward), f"{tag} t={t}: f64 reward differs at {np.nonzero(reward64 != ov.reward)[0][:8]}"
    assert np.array_equal(reward, ov.reward.astype(np.float32)), f"{tag} t={t}: f32 reward differs"
    if done.any():
        if tobs is not None:
            assert np.array_equal(tobs[done].view(np.uint32), ov.terminal_obs[done].view(np.uint32)), f"{tag} t={t}: terminal obs"
        if eps is not None:
            e = eps[done]
            assert np.array_equal(e[:, 1], ov.ep_len[done]), f"{tag} t={t}: episode length"
            assert np.array_equal(e[:, 2], ov.ep_bumps[done]), f"{tag} t={t}: episode bumps"
            assert np.array_equal(e[:, 3], ov.ep_visited[done]), f"{tag} t={t}: episode visited"
            ret = e[:, 0].copy().view(np.float32)
            want = ov.ep_ret32[done]
            assert np.array_equal(ret.view(np.uint32), want.view(np.uint32)), f"{tag} t={t}: episode return {ret} vs {want}"
            err = np.abs(ret.astype(np.float64) - ov.ep_ret[done])
            assert (err <= episode_return_bound(ov.ep_len[done], ov.ep_ret[done])).all(), \
                f"{tag} t={t}: episode return {ret} is {err.max()} from the f64 sum {ov.ep_ret[done]}"
            assert np.array_equal(e[:, 6], ov.terminated[done]) and np.array_equal(e[:, 7], ov.truncated[done])
    if state is not None:
        os_ = ov.state()
        # x y z facing visited bump step near was_near last_bump done down last_action room episode
        got = state[:, :15].astype(np.int64)
        bad = np.nonzero((got != os_).any(axis=1))[0]
        if len(bad):
            i = bad[0]
            raise AssertionError(f"{tag} t={t}: state differs for {len(bad)} envs; env {i} got {got[i]} want {os_[i]}")
        if state.shape[1] > 15:
            rc = ov.ret_centi()
            bad = np.nonzero(state[:, 15].astype(np.int64) != rc)[0]
            assert not len(bad), f"{tag} t={t}: return so far (state[15]) differs for {len(bad)} envs; env {bad[0]} " \
                                 f"got {state[bad[0], 15]} want {rc[bad[0]]}"


def compare_grids(tag, ov, grid_fn, envs):
    for i in envs:
        want = np.minimum(ov.grid(i), 255).astype(np.int16)
        got = grid_fn(i)
        assert got.shape == want.shape, f"{tag}: grid shape env {i}"
        assert np.array_equal(got, want), f"{tag}: knowledge grid of env {i} differs in {int((got != want).sum())} cells"


def replay_golden_trace(c, room, make_engine):
    """Replays one reference trace (tests/golden/cubic_traces.npz) through an engine with one env and an injected start
    pick.  `make_engine(rooms, L, crash_penalty, auto_reset)` returns an object with reset(picks)/step(actions)/state()/
    grid(env) and numpy attributes obs, reward, reward64, term, trunc."""
    fc = room.free_cells()
    k = int(np.nonzero((fc == np.asarray(c["start"])).all(axis=1))[0][0])
    eng = make_engine([room], c["L"], c["crash_penalty"], False)
    obs0 = np.array(eng.reset(picks=np.array([[0, k]], dtype=np.int32)))
    tag = f"{c['room']} L={c['L']} {c['policy']}"
    assert np.array_equal(obs0[0].view(np.uint32), c["obs"][0].view(np.uint32)), f"{tag}: reset obs"
    n = c["n"]
    for t in range(n):
        eng.step(np.array([c["actions"][t]], dtype=np.int64))
        s = eng.state()[0]
        got = [s[0], s[1], s[2], s[3], s[4], s[5], s[6], int(eng.term[0]), int(eng.trunc[0])]
        assert got == list(c["state"][t]), f"{tag} t={t}: state {got} want {list(c['state'][t])}"
        assert [s[7], s[8], s[9]] == list(c["flags"][t]), f"{tag} t={t}: flags"
        assert np.array_equal(eng.obs[0].view(np.uint32), c["obs"][t + 1].view(np.uint32)), f"{tag} t={t}: obs"
        assert eng.reward64[0] == c["reward"][t], f"{tag} t={t}: reward {eng.reward64[0]} want {c['reward'][t]}"
        assert eng.reward[0] == np.float32(c["reward"][t]), f"{tag} t={t}: f32 reward"
    assert np.array_equal(eng.grid(0), np.minimum(c["final_ig"], 255).astype(np.int16)), f"{tag}: final knowledge grid"


def replay_simple_golden_trace(c, room, make_engine):
    """Replays one simpleEnv reference trace (tests/golden/simple_traces.npz): reset with injected (room, start, goal),
    the reference's `reset(); get_obs()` then n steps.  `make_engine(rooms, L)` returns an engine-like object."""
    fc = room.free_cells()
    k = int(np.nonzero((fc == np.asarray(c["start"])).all(axis=1))[0][0])
    kg = int(np.nonzero((fc == np.asarray(c["goal"])).all(axis=1))[0][0])
    eng = make_engine([room], c["L"])
    obs0 = np.array(eng.reset(picks=np.array([[0, k, kg]], dtype=np.int32)))
    tag = f"simple {c['room']} L={c['L']}"
    assert np.array_equal(obs0[0].view(np.uint32), c["obs"][0].view(np.uint32)), f"{tag}: reset obs {obs0[0]} vs {c['obs'][0]}"
    for t in range(c["n"]):
        eng.step(np.array([c["actions"][t]], dtype=np.int64))
        s = eng.state()[0]
        got = [s[0], s[1], s[2], s[3], s[4], s[5], s[6], int(eng.term[0]), int(eng.trunc[0])]
        assert got == list(c["state"][t]), f"{tag} t={t}: state {got} want {list(c['state'][t])}"
        assert np.array_equal(eng.obs[0].view(np.uint32), c["obs"][t + 1].view(np.uint32)), \
            f"{tag} t={t}: obs {eng.obs[0]} want {c['obs'][t + 1]}"
        assert eng.reward64[0] == c["reward"][t], f"{tag} t={t}: reward {eng.reward64[0]} want {c['reward'][t]}"
    assert np.array_equal(eng.grid(0), c["final_ig"].astype(np.int16)), f"{tag}: final knowledge grid"

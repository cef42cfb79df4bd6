// nav3d_emu_rollout.cu — DEBUGGING AID, tests only.  nav3d_rollout_actions in the host emulation: each env runs its T steps
// back to back with its record held outside the engine (step_lane / step_commit with REG_STATE, as the fused rollout
// kernels run them), the per-step outputs addressed by rollout_step_io and the actions read by rollout_action of
// csrc/nav3d_core.cuh.  Built as its own library around nav3d_emu.cu (tests/emu_rollout.py), so it takes the handles
// emu_create returns.
#include "nav3d_emu.cu"

template <int G> static void rollout_env(Emu *e, const RolloutIO &ro, int T, int env) {
    const long long N = e->P.n_envs;
    EnvState st = e->states[env];                  // the kernels' register copy of the record
    for (int t = 0; t < T; t++) {
        const StepIO io = rollout_step_io(ro, t, T, N);
        const int action = rollout_action(ro, t, N, env);
        StepCtx c;
        uint32_t nbr = 0, bits = 0;
        for (int i = 0; i < G; i++) {
            const int lane = e->descending ? G - 1 - i : i;
            StepCtx ci;
            nbr |= step_lane<G, true>(e->P, io, env, lane, action, e->lut, env, &st, ci);
            c = ci;
        }
        step_commit<G, true>(e->P, io, env, 0, c, nbr, env, &st, &bits);
        if (c.will_reset) {
            reset_one_philox<G>(e, env, st.episode, io.obs ? io.obs + (size_t)env * kObsDim : nullptr);
            st = e->states[env];                   // the new episode's record
        }
    }
    e->states[env] = st;
}

extern "C" {

void emu_rollout_actions(void *h, int T, const uint8_t *actions, float *obs, float *obs_last, float *reward,
                         double *reward64, uint8_t *term, uint8_t *trunc, float *terminal_obs, void *episodes) {
    Emu *e = (Emu *)h;
    RolloutIO ro;
    ro.actions = actions; ro.obs = obs; ro.obs_last = obs_last; ro.reward = reward; ro.reward64 = reward64;
    ro.terminated = term; ro.truncated = trunc; ro.terminal_obs = terminal_obs; ro.episodes = episodes;
    for (int env = 0; env < e->P.n_envs; env++) { EMU_DISPATCH(e->G, rollout_env<G>(e, ro, T, env)) }
}
}

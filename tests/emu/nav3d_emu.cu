// nav3d_emu.cu — DEBUGGING AID, tests only.  Compiles the device logic of csrc/nav3d_core.cuh for the HOST so that the
// packed-representation logic can be checked against the oracle in the GPU-less build container.  The G lanes of an env's
// group run one after the other (ascending or descending lane order), the group's OR-reduction happens between the two
// halves of a step.  It is not linked into libnav3d_b200.so and nothing in the product imports it; it says little about
// the concurrency of the real kernels, which only the -m gpu tests exercise.
#include "../../3d-navigation-reinforcement-learning_b200/csrc/nav3d_core.cuh"

#include <cmath>
#include <cstdlib>
#include <cstring>
#include <vector>

using namespace nav3d;

struct Emu {
    EngineParams P{};
    std::vector<RoomDev> rooms;
    std::vector<uint16_t> occz;
    std::vector<unsigned long long> occ64;
    std::vector<uint32_t> free_cells;
    std::vector<EnvState> states;
    std::vector<uint8_t> know;
    float lut[nav3d::kLutSize];
    std::vector<float> dist_lut;
    bool simple = false;
    int G = 1;
    bool descending = false;
};

// Address-sanitizer build (tools/emu_asan.sh; compute-sanitizer is not available on the GPU pool): an env may only touch
// the part of its knowledge block that its CURRENT room owns — the K bricks of that room and the overflow bytes of its cells;
// everything else of the block (sized for the largest room of the set) is poisoned, so that an index computed from a wrong
// room, a negative coordinate or a missing border shows up as an ASan report instead of silently landing in padding.
#ifdef NAV3D_EMU_ASAN
#include <sanitizer/asan_interface.h>
static void fence_env(Emu *e, int env, uint32_t room) {
    uint8_t *blk = e->know.data() + (size_t)env * e->P.env_stride;
    const RoomDev &R = e->rooms[room];
    ASAN_POISON_MEMORY_REGION(blk, e->P.env_stride);
    ASAN_UNPOISON_MEMORY_REGION(blk, k_bytes(R));
    ASAN_UNPOISON_MEMORY_REGION(blk + e->P.ovf_off, (size_t)R.W * R.D * R.H);
}
#else
static void fence_env(Emu *, int, uint32_t) {}
#endif

template <int G> static void reset_one(Emu *e, int env, uint32_t room, uint32_t k, uint32_t ep_after, float *orow) {
    ResetCtx c;
    uint32_t nbr = 0;
    fence_env(e, env, room);
    for (int lane = 0; lane < G; lane++) reset_clear<G>(e->P, env, lane, room);
    for (int i = 0; i < G; i++) {
        const int lane = e->descending ? G - 1 - i : i;
        ResetCtx ci;
        nbr |= reset_lane<G>(e->P, env, lane, room, k, ep_after, e->lut, orow, ci);
        c = ci;
    }
    reset_commit(e->P, env, 0, c, nbr);
}
template <int G> static void reset_one_philox(Emu *e, int env, uint32_t episode, float *orow) {
    uint32_t room, k;
    reset_picks(e->P, env, episode, room, k);
    reset_one<G>(e, env, room, k, episode + 1u, orow);
}
template <int G> static void step_all(Emu *e, const StepIO &io, const long long *actions) {
    for (int env = 0; env < e->P.n_envs; env++) {
        StepCtx c;
        uint32_t nbr = 0;
        for (int i = 0; i < G; i++) {
            const int lane = e->descending ? G - 1 - i : i;
            StepCtx ci;
            nbr |= step_lane<G>(e->P, io, env, lane, (int)actions[env], e->lut, env, nullptr, ci);
            c = ci;
        }
        step_commit<G>(e->P, io, env, 0, c, nbr, env, nullptr, nullptr);
        if (c.will_reset) reset_one_philox<G>(e, env, e->states[env].episode, io.obs + (size_t)env * kObsDim);
    }
}
#define EMU_DISPATCH(G_, CALL)                                                                   \
    switch (G_) {                                                                                \
        case 1: { constexpr int G = 1; CALL; } break;   case 2: { constexpr int G = 2; CALL; } break;   \
        case 4: { constexpr int G = 4; CALL; } break;   case 8: { constexpr int G = 8; CALL; } break;   \
        case 16: { constexpr int G = 16; CALL; } break; default: { constexpr int G = 32; CALL; } break; \
    }

extern "C" {

void *emu_create(int n_envs, int L, double crash, unsigned long long seed, unsigned env_id0, int auto_reset, int n_rooms,
                 const int *dims, const int8_t *dense, const unsigned *dense_off, int wall_code, int simple, double cell_size,
                 int lanes, int descending, const double *reward /* the ten nav3d_reward_params fields, NULL = reference */) {
    Emu *e = new Emu();
    e->simple = simple != 0;
    e->G = lanes; e->descending = descending != 0;
    size_t max_k = 0, max_cells = 0;
    for (int r = 0; r < n_rooms; r++) {
        const int W = dims[3 * r], D = dims[3 * r + 1], H = dims[3 * r + 2];
        const int8_t *g = dense + dense_off[r];
        RoomDev R{};
        R.W = W; R.D = D; R.H = H;
        if (e->simple) { R.ntx = (W + 3) / 4; R.nty = (D + 3) / 4; R.nzb = 1; }
        else { R.ntx = (W + 3 + 3) / 4; R.nty = (D + 3 + 3) / 4; R.nzb = (H + 5) / 6; }
        R.occz_off = (uint32_t)e->occz.size();
        for (int x = 0; x < W; x++) for (int y = 0; y < D; y++) {
            uint16_t b = 0;
            for (int z = 0; z < H; z++) if (g[(x * D + y) * H + z] == wall_code) b |= 1u << z;
            e->occz.push_back(b);
        }
        R.occx_off = (uint32_t)e->occ64.size();
        for (int y = 0; y < D; y++) for (int z = 0; z < H; z++) {
            unsigned long long b = 0;
            for (int x = 0; x < W; x++) if (g[(x * D + y) * H + z] == wall_code) b |= 1ull << x;
            e->occ64.push_back(b);
        }
        R.occy_off = (uint32_t)e->occ64.size();
        for (int x = 0; x < W; x++) for (int z = 0; z < H; z++) {
            unsigned long long b = 0;
            for (int y = 0; y < D; y++) if (g[(x * D + y) * H + z] == wall_code) b |= 1ull << y;
            e->occ64.push_back(b);
        }
        R.free_off = (uint32_t)e->free_cells.size();
        uint32_t nf = 0;
        for (int x = 1; x < W - 1; x++) for (int y = 1; y < D - 1; y++) for (int z = 1; z < H - 1; z++)
            if (g[(x * D + y) * H + z] != wall_code) { e->free_cells.push_back(x | (y << 8) | (z << 16)); nf++; }
        R.n_free = nf;
        e->rooms.push_back(R);
        max_k = std::max(max_k, (size_t)(e->simple ? k2_bytes(R) : k_bytes(R)));
        max_cells = std::max(max_cells, (size_t)W * D * H);
    }
    size_t ovf_off = (max_k + 127) / 128 * 128, stride = ovf_off + (max_cells + 127) / 128 * 128;
    if (e->simple) { ovf_off = 0; stride = (max_k + 127) / 128 * 128; }
    for (int c = 0; c <= L; c++) e->dist_lut.push_back((float)py_round2((double)c * cell_size));
    e->states.assign((size_t)n_envs, EnvState{});
    e->know.assign(stride * (size_t)n_envs, 0xAB);     // poison: a reset must clear what it uses
#ifdef NAV3D_EMU_ASAN
    if (!e->simple) ASAN_POISON_MEMORY_REGION(e->know.data(), e->know.size());   // nothing is owned before the first reset
#endif
    for (int i = 0; i < kLutSize; i++) e->lut[i] = 0.f;
    for (int i = 0; i < 32; i++) {
        const int v = i == 0 ? -1 : (i == 1 ? -2 : std::min(i - 2, 20));
        e->lut[i] = (float)(v + 2) / 22.0f;
    }
    for (int i = 0; i < 6; i++) e->lut[nav3d::kLutFifth + i] = (float)i / 5.0f;
    for (int i = 0; i < 32; i++) e->lut[nav3d::kLutDown + i] = (float)i / (float)L;
    EngineParams &P = e->P;
    P.rooms = e->rooms.data(); P.occz = e->occz.data(); P.occ64 = e->occ64.data(); P.free_cells = e->free_cells.data();
    P.states = e->states.data(); P.know = e->know.data(); P.env_stride = stride; P.ovf_off = (uint32_t)ovf_off;
    P.n_envs = n_envs; P.n_rooms = n_rooms; P.L = L; P.env_id0 = env_id0; P.seed_lo = (uint32_t)seed;
    P.seed_hi = (uint32_t)(seed >> 32); P.auto_reset = auto_reset;
    P.rw = reward ? reward_params_from(reward) : reference_reward_params(crash);
    P.dist_lut = e->dist_lut.data(); P.obs_dim = e->simple ? 6 * L + 7 : kObsDim;
    return e;
}
// the engine's rule for nav3d_set_reward_params (NULL = accepted) and its simpleEnv distance rounding
const char *emu_reward_params_reject(const double *reward) { return reward_params_reject(reward_params_from(reward)); }
double emu_py_round2(double x) { return py_round2(x); }
void emu_destroy(void *h) {
#ifdef NAV3D_EMU_ASAN
    ASAN_UNPOISON_MEMORY_REGION(((Emu *)h)->know.data(), ((Emu *)h)->know.size());
#endif
    delete (Emu *)h;
}
// negative control of the sanitizer build: reads the byte at `offset` of an env's knowledge block (outside the fence -> report)
int emu_probe(void *h, int env, long offset) {
    Emu *e = (Emu *)h;
    const volatile uint8_t *p = e->know.data() + (size_t)env * e->P.env_stride + offset;
    return *p;
}
long emu_owned_k_bytes(void *h, int env) { Emu *e = (Emu *)h; return (long)k_bytes(e->rooms[e->states[env].room]); }
int emu_room_n_free(void *h, int r) { return (int)((Emu *)h)->rooms[r].n_free; }

void emu_reset(void *h, const int *env_ids, int n, const int *picks, float *obs) {
    Emu *e = (Emu *)h;
    for (int i = 0; i < n; i++) {
        const int env = env_ids ? env_ids[i] : i;
        const uint32_t ep = e->states[env].episode;
        float *orow = obs ? obs + (size_t)env * e->P.obs_dim : nullptr;
        if (e->simple) {
            if (picks) simple_reset_env<1>(e->P, env, 0, 0, (uint32_t)picks[3 * i], (uint32_t)picks[3 * i + 1], (uint32_t)picks[3 * i + 2], ep + 1, orow);
            else simple_reset_env_philox<1>(e->P, env, 0, 0, ep, orow);
            continue;
        }
        if (picks) { EMU_DISPATCH(e->G, reset_one<G>(e, env, (uint32_t)picks[2 * i], (uint32_t)picks[2 * i + 1], ep + 1, orow)) }
        else { EMU_DISPATCH(e->G, reset_one_philox<G>(e, env, ep, orow)) }
    }
}
void emu_step(void *h, const long long *actions, float *obs, float *reward, double *reward64, uint8_t *term,
              uint8_t *trunc, float *terminal_obs, void *episodes) {
    Emu *e = (Emu *)h;
    StepIO io;
    io.actions = actions; io.obs = obs; io.reward = reward; io.reward64 = reward64; io.terminated = term;
    io.truncated = trunc; io.terminal_obs = terminal_obs; io.episodes = episodes; io.env0 = 0; io.env_n = e->P.n_envs;
    if (e->simple) {
        for (int env = 0; env < e->P.n_envs; env++) simple_step_env<1>(e->P, io, env, 0, 0, (int)actions[env], env);
        return;
    }
    EMU_DISPATCH(e->G, step_all<G>(e, io, actions))
}
void emu_get_state(void *h, int *out) {
    Emu *e = (Emu *)h;
    for (int env = 0; env < e->P.n_envs; env++) {
        const EnvState s = e->states[env];
        int *o = out + (size_t)env * 16;
        o[0] = s.x; o[1] = s.y; o[2] = s.z; o[3] = s.facing; o[4] = s.visited_count; o[5] = s.bump_count;
        o[6] = s.step_count; o[7] = (s.flags & kNearWall) != 0; o[8] = (s.flags & kWasNearWall) != 0;
        o[9] = (s.flags & kLastBump) != 0; o[10] = (s.flags & kDone) != 0; o[11] = s.down; o[12] = s.last_action;
        o[13] = s.room; o[14] = s.episode; o[15] = s.ret_centi;
        if (e->simple) { o[7] = s.down; o[8] = s.blocked6; o[9] = s.own_count; o[11] = 0; }
    }
}
void emu_get_grid(void *h, int env, int16_t *out) {
    Emu *e = (Emu *)h;
    const EnvState s = e->states[env];
    const RoomDev R = e->rooms[s.room];
    const uint8_t *envk = e->know.data() + (size_t)env * e->P.env_stride;
    const uint32_t *K = (const uint32_t *)envk;
    if (e->simple) {
        for (int x = 0; x < R.W; x++) for (int y = 0; y < R.D; y++) for (int z = 0; z < R.H; z++)
            out[(x * R.D + y) * R.H + z] = (int16_t)(k2_code(K[s_index(R, x, y)], z) - 1);
        return;
    }
    for (int x = 0; x < R.W; x++) for (int y = 0; y < R.D; y++) for (int z = 0; z < R.H; z++) {
        const uint32_t code = (K[k_index(R, x, y, z / 6)] >> (5 * (z % 6))) & 31u;
        int16_t v = (int16_t)code - 2;
        if (code == kCodeUnknown) v = -1;
        else if (code == kCodeWall) v = -2;
        else if (code == kCodeOverflow) v = (int16_t)(kOverflowBase + envk[e->P.ovf_off + ovf_index(R, x, y, z)]);
        out[(x * R.D + y) * R.H + z] = v;
    }
}
}

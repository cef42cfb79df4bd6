// nav3d_core.cuh — per-environment logic of the batched CubicEnv step, written once and instantiated for a group of
// G cooperating lanes (G = 1 .. 32).  Everything here is device code for sm_100a; the functions are also marked
// __host__ so that tests/emu can run the SAME source on the CPU (lanes of a group one after the other) as a debugging
// aid (never shipped, never on the product path).
//
// Reference being replaced (semantics, not structure): envs/CubicEnv.py of Noimps/3D-Navigation-Reinforcement-Learning
//   step :110-132, do_action :134-166, compute_reward :169-224, _get_3d_local_map :229-251, get_obs :254-312,
//   _mark_visited :322-343, _sense_direction :345-397, reset :77-108, load_room's start pick :450-462.
//
// Data model (DESIGN.md §3).  The reference keeps one int64 per voxel per env (internal_grid: -2 known wall, -1 unknown,
// 0 seen, >=1 visit counter).  Here:
//   * the static room occupancy, shared by all envs, is bit-packed in three orientations so that each of the six
//     axis-aligned rays is ONE word + a bit scan (no per-cell march):
//        occz[x][y] : u16, bit z        occx[y][z] : u64, bit x        occy[x][z] : u64, bit y
//   * the per-env knowledge is ONE volume K of 5-bit codes:  0 unknown (-1) · 1 known wall (-2) · 2 + c visit count c
//     (c = 0 seen, 1 .. 28) · 31 count >= 29 (exact value = 29 + a byte of the overflow volume, which nothing else reads).
//     Six z-consecutive codes make one u32 (a "column word"); 4x4 columns x 6 levels = one 64-byte brick = one DRAM
//     atom; the z-bricks of a 4x4-column tile are adjacent.  The volume carries a border of 2 (low) / 1 (high) unknown
//     columns in x and y, so the 4x4x4 window never needs an in-bounds test in x or y.
//   * the env record caches the codes of the agent's six neighbours and the exact count of its own cell, so a step
//     knows where it moves, whether that is a first visit and what the new counter is BEFORE it loads anything; every
//     load of the step (window columns, ray marking) is therefore issued in one batch.
//   Observations clip counters at 20 and the reward at 25 (CubicEnv.py:273-274, :180); counters saturate at 255.
// Within a step every word of K has at most one writer, and whoever reads a word that is being marked in the same step
// re-derives the marks from the ray extents in registers, so the window gather never waits for the marking stores.
// Two mappings of envs to threads share this source:
//   * G = 1 with STAGED (the default kernels of nav3d_engine.cu): one thread owns an env; its observation row leaves in
//     compact form through a shared-memory staging tile that the warp expands and writes out, and its ray marking is
//     queued for the warp (MarkQueue) instead of being done in the thread;
//   * G = 2 .. 32 lanes per env (and G = 1 without STAGED, as the host emulation runs it): the lanes split the window
//     columns and the marking tiles, each lane streams its own float4s; the only cross-lane traffic is one OR-reduction of
//     the neighbour codes.
#pragma once
#include <stdint.h>
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cuda_runtime.h>

#define NAV3D_HD __host__ __device__ __forceinline__

namespace nav3d {

constexpr int kObsDim = 80;
// Shared look-up table of the step kernels: [0, 32) observation value of a 5-bit code = (clip(v, -2, 20) + 2) / 22
// (CubicEnv.py:273-275); [32, 38) k / 5 for last_action (:284); [64, 96) d / L for cells_insight_down when L <= 31
// (:287).  All entries are correctly rounded f32 quotients, i.e. the same bits as computing them in place.
constexpr int kLutSize = 96, kLutFifth = 32, kLutDown = 64;
constexpr uint32_t kStreamReset = 0x52455345u;   // include/nav3d.h "Random streams"
constexpr uint32_t kStreamAction = 0x41435449u;

// 5-bit knowledge codes
constexpr uint32_t kCodeUnknown = 0u, kCodeWall = 1u, kCodeSeen = 2u, kCodeOverflow = 31u;
constexpr int kOverflowBase = 29;                // code 31 <=> count >= 29
constexpr uint32_t kFieldLsb = 0x02108421u;      // bit 0 of each of the six 5-bit fields of a column word
constexpr int kPadLo = 2;                        // border columns of K below x = 0 / y = 0

// flag bits of EnvState::flags
constexpr uint32_t kNearWall = 1u, kWasNearWall = 2u, kLastBump = 4u, kDone = 8u;

struct alignas(32) RoomDev {       // one per room, read-only after nav3d_load_rooms
    uint16_t W, D, H, ntx;         // dims; ntx = tiles of 4 columns along x (CubicEnv: of the bordered volume)
    uint16_t nty, nzb;             // nty likewise along y; nzb = ceil(H/6) z-bricks
    uint32_t n_free;               // total_free_cells == max_steps (CubicEnv.py:450-459)
    uint32_t occz_off;             // u16 index into occz pool, [x][y]
    uint32_t occx_off;             // u64 index into occ64 pool, [y][z], bit x
    uint32_t occy_off;             // u64 index into occ64 pool, [x][z], bit y
    uint32_t free_off;             // u32 index into the free-cell pool (x | y<<8 | z<<16, reference scan order)
};
static_assert(sizeof(RoomDev) == 32, "RoomDev must be one 32-byte sector");

struct alignas(32) EnvState {      // one 32-byte sector per env: read once, written once per step
    uint8_t x, y, z, facing;
    uint8_t last_action, flags, down, blocked6;   // blocked6 bit d: a move in direction d bumps (simpleEnv: goal y)
    uint16_t step_count, visited_count;           // both saturate at 65535 (a room has at most 53 816 free cells)
    uint16_t bump_count, room;
    uint32_t nbr;                  // 5-bit codes of the six neighbour cells, direction d at bit 5d
    int32_t ret_centi;             // running episode return in 1/100 units, crash penalties excluded
    uint32_t episode;              // number of resets so far == index into the Philox reset stream
    uint8_t own_count;             // exact visit counter of the agent's cell, saturating at 255 (simpleEnv: goal z)
    uint8_t pad[3];
};
static_assert(sizeof(EnvState) == 32, "EnvState must be one 32-byte sector");

// Reward constants of compute_reward (CubicEnv.py:169-224); include/nav3d.h nav3d_reward_params mirrors this.  The c_*
// fields hold the fixed terms except the crash penalty in 1/100 units for the integer episode-return accumulator; the
// revisit term's cents are rounded from the f64 penalty of each step (step_commit).
struct RewardParams {
    double step_cost, revisit_unit, revisit_cap, crash_penalty, near_wall_bonus, repeat_bonus, reverse_penalty,
        explore_bonus, finish_bonus, truncation_penalty;
    int32_t c_step, c_near_wall, c_repeat, c_reverse, c_explore, c_finish, c_trunc;
};

// centi-units of one reward term, rounded half away from zero (exact for multiples of 0.01 up to |v| <= 1e6)
NAV3D_HD int32_t reward_centi(double v) {
#ifdef __CUDA_ARCH__
    const double s = __dmul_rn(v, 100.0);      // not fused with the add below: the host rounds v * 100 first, too
#else
    const double s = v * 100.0;
#endif
    return (int32_t)(s + (v < 0 ? -0.5 : 0.5));
}

// v = the ten fields of nav3d_reward_params in declaration order
inline RewardParams reward_params_from(const double v[10]) {
    RewardParams w;
    w.step_cost = v[0]; w.revisit_unit = v[1]; w.revisit_cap = v[2]; w.crash_penalty = v[3]; w.near_wall_bonus = v[4];
    w.repeat_bonus = v[5]; w.reverse_penalty = v[6]; w.explore_bonus = v[7]; w.finish_bonus = v[8];
    w.truncation_penalty = v[9];
    w.c_step = reward_centi(w.step_cost); w.c_near_wall = reward_centi(w.near_wall_bonus);
    w.c_repeat = reward_centi(w.repeat_bonus); w.c_reverse = reward_centi(w.reverse_penalty);
    w.c_explore = reward_centi(w.explore_bonus); w.c_finish = reward_centi(w.finish_bonus);
    w.c_trunc = reward_centi(w.truncation_penalty);
    return w;
}
// The reference's literals (CubicEnv.py:175, :179-180, :187, :193, :199, :203, :209, :215, :221).
inline RewardParams reference_reward_params(double crash_penalty) {
    const double v[10] = {-0.05, 0.02, 0.5, crash_penalty, 0.15, 0.05, 0.5, 1.0, 100.0, -5.0};
    return reward_params_from(v);
}

// Why a parameter set of finite values within [-1e6, 1e6] cannot be honoured, or nullptr (include/nav3d.h,
// nav3d_set_reward_params).
//  - The record keeps the agent cell's visit count saturated at 255, so min(count * unit, cap) must not change once the
//    count passes 255: unit == 0, or unit > 0 and 255 * unit >= cap.
//  - ret_centi is an int32: the largest |cents| one step can add, over 65 535 steps, plus one finish and one truncation
//    term, must fit.  Both the count (1..255) and the penalty are monotone, so the revisit extremes are at counts 1 and 255.
inline const char *reward_params_reject(const RewardParams &w) {
    if (!(w.revisit_unit == 0.0 || (w.revisit_unit > 0.0 && 255.0 * w.revisit_unit >= w.revisit_cap)))
        return "revisit_unit must be 0, or positive with 255 * revisit_unit >= revisit_cap: visit counts saturate at 255, "
               "so min(count * revisit_unit, revisit_cap) must not change past count 255";
    auto a = [](long long c) { return c < 0 ? -c : c; };
    const double p1 = w.revisit_unit < w.revisit_cap ? w.revisit_unit : w.revisit_cap;
    const double p255 = 255.0 * w.revisit_unit < w.revisit_cap ? 255.0 * w.revisit_unit : w.revisit_cap;
    const long long rev = std::max(a(reward_centi(p1)), a(reward_centi(p255)));
    const long long per_step = a(w.c_step) + rev + a(w.c_near_wall) + std::max(a(w.c_repeat), a(w.c_reverse)) + a(w.c_explore);
    if (65535LL * per_step + a(w.c_finish) + a(w.c_trunc) > 2147483647LL)
        return "the largest episode return these parameters allow (65 535 steps) does not fit the int32 accumulator of "
               "1/100 units";
    return nullptr;
}

// Python's round(x, 2): the exact binary value of x rounded to two decimals (ties to even), as glibc's printf does, then
// parsed back.  rint(x * 100) / 100 is not the same: 0.175 * 100 rounds onto the tie 17.5 and gives 0.18, while
// round(0.175, 2) is 0.17 (0.175 is slightly below 0.175 in binary).
inline double py_round2(double x) {
    char buf[64];
    std::snprintf(buf, sizeof buf, "%.2f", x);
    return std::strtod(buf, nullptr);
}

struct EngineParams {
    const RoomDev *rooms;
    const uint16_t *occz;
    const unsigned long long *occ64;
    const uint32_t *free_cells;
    const uint32_t *room_start;    // per room: x | y<<8 | z<<16 of the file's "Start position" or 0xffffffff (may be null)
    EnvState *states;
    uint8_t *know;                 // per-env knowledge storage: [K bricks | overflow bytes]
    unsigned long long env_stride; // bytes per env in `know`
    uint32_t ovf_off;              // byte offset of the overflow volume inside an env block
    int32_t n_envs, n_rooms, L;
    uint32_t env_id0, seed_lo, seed_hi;
    int32_t auto_reset;
    RewardParams rw;
    const float *dist_lut;         // simpleEnv: round(count * cell_size, 2) as f32, count = 0..L (simpleEnv.py:337)
    int32_t obs_dim;               // 80 (CubicEnv) or 6L+7 (simpleEnv)
    int32_t mark_cap;              // entries of a warp's marking list (32 x mark_tasks_per_lane of the loaded room set)
};

struct StepIO {                    // per-launch output pointers (any may be null except obs)
    const long long *actions;
    float *obs;
    float *reward;
    double *reward64;
    uint8_t *terminated, *truncated;
    float *terminal_obs;
    void *episodes;                // nav3d_episode*
    int env0, env_n;               // the launch covers envs [env0, env0 + env_n); outputs are indexed by the env itself
};

// ---------------------------------------------------------------------------------------------------------------
// small helpers
// ---------------------------------------------------------------------------------------------------------------
NAV3D_HD int ffs64(unsigned long long v) {
#ifdef __CUDA_ARCH__
    return __ffsll((long long)v);
#else
    return v ? __builtin_ctzll(v) + 1 : 0;
#endif
}
NAV3D_HD int clz64(unsigned long long v) {
#ifdef __CUDA_ARCH__
    return __clzll((long long)v);
#else
    return v ? __builtin_clzll(v) : 64;
#endif
}
NAV3D_HD int ffs32(uint32_t v) {
#ifdef __CUDA_ARCH__
    return __ffs((int)v);
#else
    return v ? __builtin_ctz(v) + 1 : 0;
#endif
}
NAV3D_HD int clz32(uint32_t v) {
#ifdef __CUDA_ARCH__
    return __clz((int)v);
#else
    return v ? __builtin_clz(v) : 32;
#endif
}
NAV3D_HD float fdiv_rn(float a, float b) {
#ifdef __CUDA_ARCH__
    return __fdiv_rn(a, b);
#else
    return a / b;
#endif
}
template <typename T> NAV3D_HD T ldg(const T *p) {
#ifdef __CUDA_ARCH__
    return __ldg(p);
#else
    return *p;
#endif
}
NAV3D_HD int imin(int a, int b) { return a < b ? a : b; }
// a + b clamped to the int32 range (the episode-return accumulator of an env stepped on past done, auto_reset = 0)
NAV3D_HD int add_saturate(int a, int b) {
    const long long s = (long long)a + b;
    return s > 2147483647LL ? 2147483647 : (s < -2147483647LL - 1 ? (int)(-2147483647LL - 1) : (int)s);
}
NAV3D_HD int imax(int a, int b) { return a > b ? a : b; }
// Streaming (evict-first) stores for data that is written once and not read again by this engine (observations, rewards,
// flags): keeps them from evicting the per-env knowledge lines that the NEXT step will touch again from L2.
NAV3D_HD void store_stream(float4 *p, float4 v) {
#ifdef __CUDA_ARCH__
    __stcs(p, v);
#else
    *p = v;
#endif
}
NAV3D_HD void store_stream(float *p, float v) {
#ifdef __CUDA_ARCH__
    __stcs(p, v);
#else
    *p = v;
#endif
}

// Observation rows.  Direct: a lane streams its float4 straight to the caller's row.  STAGED (thread-per-env kernels): a
// thread leaves its row in COMPACT form in its slot of a shared-memory staging tile — kStageStride u32 apart (odd: the 32
// rows fall into 32 different banks): words 0..15 the sixteen window columns as four 5-bit codes each, word 16 the packed
// scalars, word 17 the f32 bits of visited / total — and the WARP then expands the 32 rows through the code table and writes
// them out with fully coalesced 128-bit stores (flush_rows in nav3d_engine.cu): 16 full sectors per store instruction
// instead of 32 half sectors, and 100 bytes of shared memory per env instead of 336.
constexpr int kStageStride = 25;
constexpr int kStageScalars = 16, kStageExplored = 17;
NAV3D_HD uint32_t float_bits(float f) {
#ifdef __CUDA_ARCH__
    return __float_as_uint(f);
#else
    uint32_t u; __builtin_memcpy(&u, &f, 4); return u;
#endif
}

template <int G> NAV3D_HD unsigned group_mask(int lane_in_warp) {
    return (G >= 32 ? 0xffffffffu : ((1u << G) - 1u)) << (lane_in_warp & ~(G - 1) & 31);
}
template <int G> NAV3D_HD void group_sync(int lane_in_warp) {
#ifdef __CUDA_ARCH__
    if (G > 1) __syncwarp(group_mask<G>(lane_in_warp));
#else
    (void)lane_in_warp;
#endif
}
// OR over the G lanes of a group; every lane gets the result.  The host build (one lane at a time) reduces outside.
template <int G> NAV3D_HD uint32_t group_or(uint32_t v, int lane_in_warp) {
#ifdef __CUDA_ARCH__
    if (G > 1) {
        const unsigned m = group_mask<G>(lane_in_warp);
#pragma unroll
        for (int o = G / 2; o > 0; o >>= 1) v |= __shfl_xor_sync(m, v, o);
    }
#else
    (void)lane_in_warp;
#endif
    return v;
}

// Philox4x32-10 (Salmon et al., SC'11)
NAV3D_HD void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1,
                            uint32_t &o0, uint32_t &o1) {
#pragma unroll
    for (int r = 0; r < 10; r++) {
        unsigned long long p0 = (unsigned long long)0xD2511F53u * c0;
        unsigned long long p1 = (unsigned long long)0xCD9E8D57u * c2;
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
        uint32_t n1 = (uint32_t)p1;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        uint32_t n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    o0 = c0; o1 = c1;
}
NAV3D_HD void philox4x32_10_4(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t *o) {
#pragma unroll
    for (int r = 0; r < 10; r++) {
        unsigned long long p0 = (unsigned long long)0xD2511F53u * c0;
        unsigned long long p1 = (unsigned long long)0xCD9E8D57u * c2;
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
        uint32_t n1 = (uint32_t)p1;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        uint32_t n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    o[0] = c0; o[1] = c1; o[2] = c2; o[3] = c3;
}
NAV3D_HD uint32_t mulhi_range(uint32_t u, uint32_t n) { return (uint32_t)(((unsigned long long)u * n) >> 32); }

// ---------------------------------------------------------------------------------------------------------------
// knowledge-storage addressing (CubicEnv).  Bordered coordinates xp = x + kPadLo, yp = y + kPadLo.
// ---------------------------------------------------------------------------------------------------------------
NAV3D_HD int div6(int q) { return (q * 43) >> 8; }                    // exact for 0 <= q < 48
NAV3D_HD uint32_t k_xpart(const RoomDev &R, int xp) { return (uint32_t)((((xp >> 2) * R.nzb) << 4) + ((xp & 3) << 2)); }
NAV3D_HD uint32_t k_ypart(const RoomDev &R, int yp) { return (uint32_t)((((yp >> 2) * R.ntx * R.nzb) << 4) + (yp & 3)); }
// u32 index of the column word of cell column (x, y), z-brick zb
NAV3D_HD uint32_t k_index(const RoomDev &R, int x, int y, int zb) {
    return k_xpart(R, x + kPadLo) + k_ypart(R, y + kPadLo) + ((uint32_t)zb << 4);
}
NAV3D_HD uint32_t k_bytes(const RoomDev &R) { return (uint32_t)R.ntx * R.nty * R.nzb * 64u; }
NAV3D_HD uint32_t ovf_index(const RoomDev &R, int x, int y, int z) { return (uint32_t)((x * R.D + y) * R.H + z); }
NAV3D_HD uint32_t count_code(int c) { return (uint32_t)imin(c + 2, 31); }   // code of a seen free cell with counter c

// simpleEnv keeps its own column tiles (u32 per column, 4x4 columns per 64-byte tile), unbordered
NAV3D_HD uint32_t s_index(const RoomDev &R, int x, int y) {
    return (uint32_t)((((y >> 2) * R.ntx + (x >> 2)) << 4) + ((x & 3) << 2) + (y & 3));
}

// ---------------------------------------------------------------------------------------------------------------
// rays: _sense_direction (CubicEnv.py:345-397) for all six directions at once, from the packed occupancy
// ---------------------------------------------------------------------------------------------------------------
struct Rays {
    int x0, x1, y0, y1, z0, z1; // inclusive extents of the cells the +-x / +-y / +-z rays examine (wall ends included)
    uint32_t wall6;            // bit d: the ray in direction d ended on a wall (that cell becomes -2)
    int near_wall;             // a wall at distance 1 in any direction (:378-379)
    int down;                  // free cells seen below (:394-395)
    uint32_t blocked6;         // bit d set: a move in direction d bumps (wall or room edge at distance 1);
                               // d = 0 +x, 1 -x, 2 +y, 3 -y, 4 +z, 5 -z.  Cached in the record for the next step's move.
};

// cells p+1 .. p+n along increasing bit index of w.  SHORT (ray length <= 31): only the 32 cells next to p can matter, so
// the scan runs on one 32-bit word (a wall further away reads as "none", which is what f > n means anyway).
// ext = cells examined (up to and including the first wall), wall = 1 if the last of them is a wall.
template <bool SHORT>
NAV3D_HD void ray_up(unsigned long long w, int p, int n, int &ext, int &wall) {
    ext = 0; wall = 0;
    if (n <= 0) return;
    unsigned long long m = w >> (p + 1);                 // n > 0 implies p + 1 <= 63
    int f = SHORT ? ffs32((uint32_t)m) : ffs64(m);       // 1-based distance of the first wall, 0 = none
    if (f != 0 && f <= n) { ext = f; wall = 1; }
    else ext = n;
}
// cells p-1 .. p-n along decreasing bit index of w
template <bool SHORT>
NAV3D_HD void ray_down(unsigned long long w, int p, int n, int &ext, int &wall) {
    ext = 0; wall = 0;
    if (n <= 0) return;                                  // n > 0 implies 1 <= p <= 63
    unsigned long long m = w << (64 - p);                // bit 63 = cell p-1
    int f;
    if (SHORT) { const uint32_t hi = (uint32_t)(m >> 32); f = hi ? clz32(hi) + 1 : 0; }
    else f = m ? clz64(m) + 1 : 0;
    if (f != 0 && f <= n) { ext = f; wall = 1; }
    else ext = n;
}

template <bool SHORT>
NAV3D_HD Rays cast_rays_t(const EngineParams &P, const RoomDev &R, int x, int y, int z) {
    const int L = P.L, W = R.W, D = R.D, H = R.H;
    unsigned long long wx = ldg(P.occ64 + R.occx_off + (uint32_t)(y * H + z));
    unsigned long long wy = ldg(P.occ64 + R.occy_off + (uint32_t)(x * H + z));
    unsigned long long wz = ldg(P.occz + R.occz_off + (uint32_t)(x * D + y));
    Rays r;
    int ext, wall, n;
    uint32_t blk = 0, w6 = 0, near = 0;
#define NAV3D_RAY(d, CALL, ROOM_LEFT, DST, SIGN)                                                        \
    n = imin(L, (ROOM_LEFT)); CALL;                                                                     \
    DST = SIGN ext; w6 |= (uint32_t)wall << (d); near |= (uint32_t)(wall && ext == 1);                  \
    blk |= (uint32_t)((wall && ext == 1) || n <= 0) << (d);
    NAV3D_RAY(0, ray_up<SHORT>(wx, x, n, ext, wall), W - 1 - x, r.x1, x +)
    NAV3D_RAY(1, ray_down<SHORT>(wx, x, n, ext, wall), x, r.x0, x -)
    NAV3D_RAY(2, ray_up<SHORT>(wy, y, n, ext, wall), D - 1 - y, r.y1, y +)
    NAV3D_RAY(3, ray_down<SHORT>(wy, y, n, ext, wall), y, r.y0, y -)
    NAV3D_RAY(4, ray_up<SHORT>(wz, z, n, ext, wall), H - 1 - z, r.z1, z +)
    NAV3D_RAY(5, ray_down<SHORT>(wz, z, n, ext, wall), z, r.z0, z -)
#undef NAV3D_RAY
    r.down = ext - wall;                                  // the last ray cast is the one going down
    r.wall6 = w6;
    r.near_wall = (int)near;
    r.blocked6 = blk;
    return r;
}
NAV3D_HD Rays cast_rays(const EngineParams &P, const RoomDev &R, int x, int y, int z) {
    return P.L <= 31 ? cast_rays_t<true>(P, R, x, y, z) : cast_rays_t<false>(P, R, x, y, z);
}

// ---------------------------------------------------------------------------------------------------------------
// get_obs (CubicEnv.py:254-312): fold the rays into K, gather the 4x4x4 window, write the 80 floats
// ---------------------------------------------------------------------------------------------------------------
struct ObsScalars {
    int facing, last_action, was_near_wall, last_bump, down;
    uint32_t visited, total_free;
};

// Lane -> window columns.  Column j = 4*dxi + dyi of the 4x4 (x,y) window, dyi = (lane & 3) + b*G (b < NY),
// dxi = (lane >> 2) + a*XS (a < NX).  A lane with dxi >= 4 (G = 32) has no column.
template <int G> struct WinMap {
    static constexpr int NY = G >= 4 ? 1 : 4 / G;
    static constexpr int NX = G >= 16 ? 1 : (16 / G) / NY;
    static constexpr int XS = G >= 4 ? G / 4 : 1;
    static constexpr int NC = NX * NY;                   // columns per lane
};

// the codes of window cells z-2 .. z+1 of one column, 5 bits each from bit 0, out of the column's (at most) two words
NAV3D_HD uint32_t window_quad(uint32_t lo, uint32_t hi, int s) {
    const unsigned long long v = (unsigned long long)lo | ((unsigned long long)hi << 30);
    return (uint32_t)(s >= 0 ? (v >> (5 * s)) : (v << (-5 * s))) & 0xfffffu;
}

// Steps 3-6 of get_obs: the 9 scalars + zero padding = 4 more float4 (:279-307)
template <int G, bool STAGED = false>
NAV3D_HD void write_scalars(const EngineParams &P, int lane, const ObsScalars &sc, const float *lut,
                            float *__restrict__ obs_row) {
    if (STAGED) {          // compact: facing | last_action << 2 | was_near_wall << 5 | last_bump << 6 | down << 8
        uint32_t *row = reinterpret_cast<uint32_t *>(obs_row);
        row[kStageScalars] = (uint32_t)sc.facing | ((uint32_t)sc.last_action << 2) | ((uint32_t)sc.was_near_wall << 5) |
                             ((uint32_t)sc.last_bump << 6) | ((uint32_t)sc.down << 8);
        row[kStageExplored] = float_bits(fdiv_rn((float)sc.visited, (float)sc.total_free));
    } else for (int j = 16 + lane; j < 20; j += G) {
        float4 v;
        if (j == 16) {
            v.x = sc.facing == 0 ? 1.f : 0.f; v.y = sc.facing == 1 ? 1.f : 0.f;
            v.z = sc.facing == 2 ? 1.f : 0.f; v.w = sc.facing == 3 ? 1.f : 0.f;
        } else if (j == 17) {
            // float(k)/5, count/L and visited/total are f64 quotients rounded to f32 in the reference (:284-291); for
            // integers below 2^24 that equals the correctly rounded f32 quotient (53 >= 2*24+2, Figueroa 1995).
            // (the two small quotients come from the shared table: same correctly rounded bits, no division sequence)
            v.x = lut[kLutFifth + sc.last_action];
            v.y = (float)sc.was_near_wall;
            v.z = (float)sc.last_bump;
            v.w = P.L <= 31 ? lut[kLutDown + sc.down] : fdiv_rn((float)sc.down, (float)P.L);
        } else if (j == 18) {
            v.x = fdiv_rn((float)sc.visited, (float)sc.total_free);
            v.y = v.z = v.w = 0.f;
        } else {
            v.x = v.y = v.z = v.w = 0.f;
        }
        store_stream(reinterpret_cast<float4 *>(obs_row) + j, v);
    }
}

// Ray marking by the WARP (thread-per-env kernels).  With one thread per env a warp executes the union of its 32 envs'
// paths: marking in the thread costs every lane the longest run of the warp.  Instead a thread on a first visit only
// QUEUES its marking tiles — one u32 per tile: word index of the tile in the env's block (16 bits) | lane (5) << 16 | tile
// number along the run (5) << 21 | z field (3) << 26 | y run (words tile + j instead of tile + 4j) << 29 | a single wall-end
// word << 30 — in a shared-memory list of the warp, with the free range and the centre coordinate of its two runs in
// `desc`, and after the step all 32 lanes work the list off evenly (coop_marks in nav3d_engine.cu), each deriving the cell
// mask of its tile from the run's description.  No two tasks of a step touch the same word: their order does not matter.
struct MarkQueue {
    uint32_t *tasks;               // the warp's list (EngineParams::mark_cap entries)
    int *count;                    // its length
    uint32_t *desc;                // [2][32]: per lane the x run and the y run as first | last << 8 | centre << 16
    int lane;                      // this thread's lane (the flush finds the env's block and the runs through it)
};
// Worst case per lane: an x run and a y run of min(2L+1, room width / depth) cells = (len + 6) / 4 tiles each, + 4 wall ends.
NAV3D_HD int mark_tasks_per_lane(int L, int max_w, int max_d) {
    return (imin(2 * L + 1, max_w) + 6) / 4 + (imin(2 * L + 1, max_d) + 6) / 4 + 4;
}

// A code-0 field at bit `sh` of w becomes `code`; returns the new word.
NAV3D_HD uint32_t mark_field(uint32_t w, int sh, uint32_t code) { return ((w >> sh) & 31u) ? w : (w | (code << sh)); }

// The centre column: visit counter of the agent's cell (do_action :156-166 — the caller supplies the new value) and,
// when `mark`, the +-z rays (:264-266 for directions up/down).  cw[b] = word of z-brick b, updated in place.
NAV3D_HD void centre_update(uint32_t *cw, int nzb, int z, int c_new, bool mark, int mz0, int mz1, const Rays &r) {
    const int wup = (int)((r.wall6 >> 4) & 1u), wdn = (int)((r.wall6 >> 5) & 1u);
    const int f0 = imax(r.z0 + wdn, mz0), f1 = imin(r.z1 - wup, mz1);      // free cells of the z run still to be marked
    const bool end_up = mark && wup && r.z1 >= mz0 && r.z1 <= mz1, end_dn = mark && wdn && r.z0 >= mz0 && r.z0 <= mz1;
#pragma unroll
    for (int b = 0; b < 3; b++) {
        if (b >= nzb) break;
        uint32_t w = cw[b];
        const int zlo = 6 * b;
        if (z >= zlo && z < zlo + 6) {
            const int sh = 5 * (z - zlo);
            w = (w & ~(31u << sh)) | (count_code(c_new) << sh);
        }
        if (mark) {
            // zero fields of the free range become "seen" (2); a wall end becomes 1
            const int a = imax(f0, zlo) - zlo, e = imin(f1, zlo + 5) - zlo;
            if (a <= e) {
                uint32_t t = w | (w >> 1) | (w >> 2);
                t |= t >> 2;                                                 // bit 5f = OR of the five bits of field f
                const uint32_t range = kFieldLsb & ((2u << (5 * e)) - 1u) & ~((1u << (5 * a)) - 1u);
                w |= (~t & range) << 1;
            }
            if (end_up && r.z1 >= zlo && r.z1 < zlo + 6) w = mark_field(w, 5 * (r.z1 - zlo), kCodeWall);
            if (end_dn && r.z0 >= zlo && r.z0 < zlo + 6) w = mark_field(w, 5 * (r.z0 - zlo), kCodeWall);
        }
        cw[b] = w;
    }
}

// get_obs (CubicEnv.py:254-312) + the visit-counter update of the agent's cell, for one lane of the env's group.
//   c_new    new counter of the agent's cell (the code written into K and shown in the window)
//   fresh    this is the first time the agent stands here (or a reset): only then can the rays reveal anything — every
//            earlier stay already marked them, marks are never erased within an episode
//   persist  write the ray marks to memory (false when the env is about to be reset: only the observation needs them)
//   mdir     the move that brought the agent here (0 +x, 1 -x, 2 +y, 3 -y, 4 +z, 5 -z; -1 = none: a reset).  The cell it
//            left lies one step back on that axis and its rays along the axis already covered everything this cell's rays
//            cover except the single cell at distance exactly L ahead: that run shrinks to the one far cell.
// Returns this lane's share of the neighbour codes (OR over the group = EnvState::nbr).
template <int G, bool STAGED = false>
NAV3D_HD uint32_t observe(const EngineParams &P, const RoomDev &R, uint8_t *envk, int lane, int x, int y, int z,
                          const Rays &r, int c_new, bool fresh, bool persist, int mdir, const ObsScalars &sc,
                          const float *lut, float *__restrict__ obs_row, const MarkQueue *mq = nullptr) {
    using M = WinMap<G>;
    uint32_t *__restrict__ K = reinterpret_cast<uint32_t *>(envk);
    const int L = P.L, nzb = R.nzb;
    // window rows z-2 .. z+1 inside the column words
    const int q = z - 2;
    const int zb = q >= 0 ? div6(q) : 0, s = q - 6 * zb;            // s in [-2, 5]
    const bool need_hi = s > 2 && zb + 1 < nzb;
    const uint32_t zoff = (uint32_t)zb << 4;
    const int dy0 = lane & 3, dx0 = lane >> 2;
    const bool has_cols = dx0 < 4;

    // ---- 1. every load of the step.  Window columns first (bordered volume: no bounds tests).
    uint32_t lo[M::NC], hi[M::NC];
    if (has_cols) {
#pragma unroll
        for (int b = 0; b < M::NY; b++) {
            const uint32_t yp = k_ypart(R, y + dy0 + b * G) + zoff;
#pragma unroll
            for (int a = 0; a < M::NX; a++) {
                const uint32_t idx = yp + k_xpart(R, x + dx0 + a * M::XS);
                lo[b * M::NX + a] = K[idx];
                hi[b * M::NX + a] = need_hi ? K[idx + 16] : 0u;
            }
        }
    }
    // Ray marking (Step 1 of get_obs, :264-266), x and y runs without the centre column (its owner takes that).
    const bool mark = fresh && persist;
    int mx0 = r.x0, mx1 = r.x1, my0 = r.y0, my1 = r.y1, mz0 = r.z0, mz1 = r.z1;      // runs; empty when hi < lo
    if (mdir == 0) { mx0 = r.x1; mx1 = (r.x1 - x == L) ? r.x1 : r.x1 - 1; }
    else if (mdir == 1) { mx1 = r.x0; mx0 = (x - r.x0 == L) ? r.x0 : r.x0 + 1; }
    else if (mdir == 2) { my0 = r.y1; my1 = (r.y1 - y == L) ? r.y1 : r.y1 - 1; }
    else if (mdir == 3) { my1 = r.y0; my0 = (y - r.y0 == L) ? r.y0 : r.y0 + 1; }
    else if (mdir == 4) { mz0 = r.z1; mz1 = (r.z1 - z == L) ? r.z1 : r.z1 - 1; }
    else if (mdir == 5) { mz1 = r.z0; mz0 = (z - r.z0 == L) ? r.z0 : r.z0 + 1; }
    // Free cells of the x run (row y) and of the y run (column x) become "seen"; a run's wall end is a point mark.  The
    // centre column is skipped (its owner writes it).  Lane-strided, U cells per lane per chunk, loads before stores.
    const int zbz = div6(z), zsh = 5 * (z - 6 * zbz);
    const uint32_t zoffz = (uint32_t)zbz << 4;
    const uint32_t xpc = k_xpart(R, x + kPadLo), ypc = k_ypart(R, y + kPadLo);
    const bool hasx = mark && mx1 >= mx0, hasy = mark && my1 >= my0;
    const bool wxh = hasx && (r.wall6 & 1u) && mx1 == r.x1, wxl = hasx && (r.wall6 & 2u) && mx0 == r.x0;
    const bool wyh = hasy && (r.wall6 & 4u) && my1 == r.y1, wyl = hasy && (r.wall6 & 8u) && my0 == r.y0;
    const int fx0 = mx0 + (wxl ? 1 : 0), fx1 = hasx ? mx1 - (wxh ? 1 : 0) : fx0 - 1;
    const int fy0 = my0 + (wyl ? 1 : 0), fy1 = hasy ? my1 - (wyh ? 1 : 0) : fy0 - 1;
    const uint32_t xmul = (uint32_t)R.nzb << 4, ymul = (uint32_t)(R.ntx * R.nzb) << 4;
    const uint32_t xbase = ypc + zoffz, ybase = xpc + zoffz;
    // Tile by tile: the four cells of a run inside one 4x4-column tile are the words tile + 4j (x run) or tile + j (y run:
    // one 128-bit load), so a cell costs no address arithmetic.  Lane-strided over the tiles, UT tiles per lane per run
    // per round; a word that is not to be marked reads as all ones ("nothing to do").
    constexpr int UT = G >= 4 ? 1 : (G == 2 ? 2 : 3);
    const int xt0 = (fx0 + kPadLo) >> 2, xt1 = fx1 >= fx0 ? (fx1 + kPadLo) >> 2 : xt0 - 1;
    const int yt0 = (fy0 + kPadLo) >> 2, yt1 = fy1 >= fy0 ? (fy1 + kPadLo) >> 2 : yt0 - 1;
    // bit c + pad of a run mask: cell c of the run is to be marked (free range, centre column excluded); a tile's four
    // cells are then four consecutive bits (bordered coordinates < 64 + pad + 1 fit 64 + 3 bits: rooms are at most 64 wide,
    // so the mask is kept as 64 bits of cells 0 .. 63 - pad and the top cells are handled by the clamp below)
    auto run_mask = [&](int c_lo, int c_hi, int skip) {
        unsigned long long m = 0ull;
        if (c_hi >= c_lo) {
            const int n = c_hi - c_lo + 1;                           // 1 .. 64
            m = (n >= 64 ? ~0ull : ((1ull << n) - 1ull)) << c_lo;    // bit c: cell c (c_lo >= 0)
            m &= ~(1ull << skip);
        }
        return m;
    };
    const unsigned long long xrm = run_mask(fx0, fx1, x), yrm = run_mask(fy0, fy1, y);
    // the four cells 4T - pad .. 4T - pad + 3 of tile T
    auto tile_mask = [&](unsigned long long rm, int T) {
        const int c0 = 4 * T - kPadLo;                               // >= -pad
        return (uint32_t)(c0 >= 0 ? (rm >> c0) : (rm << (-c0))) & 0xfu;
    };
    uint32_t xw[UT][4], pw[4], ym[UT];
    uint4 yw[UT];
    auto tiles_load = [&](int tx, int ty) {
#pragma unroll
        for (int u = 0; u < UT; u++) {
            const int Tx = tx + lane + u * G, Ty = ty + lane + u * G;
            const uint32_t mxm = Tx <= xt1 ? tile_mask(xrm, Tx) : 0u, mym = Ty <= yt1 ? tile_mask(yrm, Ty) : 0u;
            const uint32_t bx = xbase + (uint32_t)Tx * xmul, by = ybase + (uint32_t)Ty * ymul;
#pragma unroll
            for (int j = 0; j < 4; j++) xw[u][j] = ((mxm >> j) & 1u) ? K[bx + 4 * j] : 0xffffffffu;
            // (nothing may consume the loaded words here: a use right behind its load would stall the issue of the next)
            ym[u] = mym;
            yw[u] = make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu);
            if (mym) yw[u] = *reinterpret_cast<const uint4 *>(K + by);
        }
    };
    auto tiles_store = [&](int tx, int ty) {
#pragma unroll
        for (int u = 0; u < UT; u++) {
            const uint32_t bx = xbase + (uint32_t)(tx + lane + u * G) * xmul, by = ybase + (uint32_t)(ty + lane + u * G) * ymul;
#pragma unroll
            for (int j = 0; j < 4; j++)
                if (((xw[u][j] >> zsh) & 31u) == 0u) K[bx + 4 * j] = xw[u][j] | (kCodeSeen << zsh);
            const uint32_t yv[4] = {yw[u].x, yw[u].y, yw[u].z, yw[u].w};
#pragma unroll
            for (int j = 0; j < 4; j++)
                if (((ym[u] >> j) & 1u) && ((yv[j] >> zsh) & 31u) == 0u) K[by + j] = yv[j] | (kCodeSeen << zsh);
        }
    };
    const bool pon[4] = {wxh, wxl, wyh, wyl};
    const uint32_t pidx[4] = {k_xpart(R, r.x1 + kPadLo) + xbase, k_xpart(R, r.x0 + kPadLo) + xbase,
                              k_ypart(R, r.y1 + kPadLo) + ybase, k_ypart(R, r.y0 + kPadLo) + ybase};
    constexpr bool queued = STAGED;                            // the warp marks (coop_marks): only queue the tiles here (mq != NULL)
    // (queued) reserve the list slots now; the slots are written further down, once the centre column's loads are issued as
    // well: the shared-memory atomic's latency would otherwise stall this warp's issue right here
    int q_at = 0, q_n = 0;
#ifdef __CUDA_ARCH__
    if (queued && mark) {
        q_n = (xt1 - xt0 + 1) + (yt1 - yt0 + 1) + (int)wxh + (int)wxl + (int)wyh + (int)wyl;
        if (q_n > 0) q_at = atomicAdd(mq->count, q_n);
    }
#endif
    if (!queued) tiles_load(xt0, yt0);
#pragma unroll
    for (int d = 0; d < 4; d++) pw[d] = (!queued && pon[d] && (d & (G - 1)) == lane) ? K[pidx[d]] : 0xffffffffu;
    // The owner of the centre column loads all of its words: counter update + the z rays.
    bool owner = false;
#pragma unroll
    for (int b = 0; b < M::NY; b++)
#pragma unroll
        for (int a = 0; a < M::NX; a++) owner = owner || (dx0 + a * M::XS == 2 && dy0 + b * G == 2);
    uint32_t cw[3] = {0u, 0u, 0u}, cw_old[3] = {0u, 0u, 0u};
    const uint32_t cbase = xpc + ypc;
    if (owner) {
#pragma unroll
        for (int b = 0; b < 3; b++) if (b < nzb) cw_old[b] = cw[b] = K[cbase + ((uint32_t)b << 4)];
    }
#ifdef __CUDA_ARCH__
    if (queued && q_n > 0) {
        int at = q_at;
        const uint32_t tag = ((uint32_t)mq->lane << 16) | ((uint32_t)(z - 6 * zbz) << 26);
        mq->desc[mq->lane] = (uint32_t)(fx0 & 255) | ((uint32_t)(fx1 & 255) << 8) | ((uint32_t)x << 16);
        mq->desc[32 + mq->lane] = (uint32_t)(fy0 & 255) | ((uint32_t)(fy1 & 255) << 8) | ((uint32_t)y << 16);
        for (int T = xt0; T <= xt1; T++) mq->tasks[at++] = (xbase + (uint32_t)T * xmul) | tag | ((uint32_t)T << 21);
        for (int T = yt0; T <= yt1; T++) mq->tasks[at++] = (ybase + (uint32_t)T * ymul) | tag | ((uint32_t)T << 21) | (1u << 29);
#pragma unroll
        for (int d = 0; d < 4; d++)
            if (pon[d]) mq->tasks[at++] = pidx[d] | tag | (1u << 30);
    }
#endif

    // ---- 2. stores to K
    if (owner) {
        centre_update(cw, nzb, z, c_new, fresh, mz0, mz1, r);
        // a first visit about to be discarded by a reset (persist == false) still shows its marks in the observation
#pragma unroll
        for (int b = 0; b < 3; b++) if (b < nzb && persist && cw[b] != cw_old[b]) K[cbase + ((uint32_t)b << 4)] = cw[b];
    }
    if (!queued) {
        tiles_store(xt0, yt0);
#pragma unroll
        for (int d = 0; d < 4; d++)
            if (((pw[d] >> zsh) & 31u) == 0u) K[pidx[d]] = pw[d] | (kCodeWall << zsh);
        // the rest of long runs, both runs per round so that their loads share one latency
        for (int k = G * UT; xt0 + k <= xt1 || yt0 + k <= yt1; k += G * UT) {
            tiles_load(xt0 + k, yt0 + k);
            tiles_store(xt0 + k, yt0 + k);
        }
    }

    // ---- 3. the window: clip to [-2, 20], (m + 2) / 22 (:273-275), one float4 per column; neighbour codes
    uint32_t nbr = 0;
    if (has_cols) {
#pragma unroll
        for (int b = 0; b < M::NY; b++) {
            const int dyi = dy0 + b * G, cy = y + dyi - 2;
#pragma unroll
            for (int a = 0; a < M::NX; a++) {
                const int dxi = dx0 + a * M::XS, cx = x + dxi - 2;
                const int c = b * M::NX + a;
                uint32_t quad;
                if (dxi == 2 && dyi == 2) {
                    // centre column: from the updated words (zb may be one past the last brick when need_hi is false)
                    const uint32_t wlo = zb == 0 ? cw[0] : (zb == 1 ? cw[1] : cw[2]);
                    const uint32_t whi = !need_hi ? 0u : (zb == 0 ? cw[1] : cw[2]);
                    quad = window_quad(wlo, whi, s);
                    nbr |= ((quad >> 15) & 31u) << 20;            // z+1 -> direction 4
                    nbr |= ((quad >> 5) & 31u) << 25;             // z-1 -> direction 5
                } else {
                    quad = window_quad(lo[c], hi[c], s);
                    if (fresh) {
                        // cells this step's rays see may not be in memory yet (another lane marks them): same rule here
                        if (dyi == 2 && cx >= r.x0 && cx <= r.x1 && ((quad >> 10) & 31u) == 0u)
                            quad |= (((cx == r.x1 && (r.wall6 & 1u)) || (cx == r.x0 && (r.wall6 & 2u))) ? kCodeWall : kCodeSeen) << 10;
                        if (dxi == 2 && cy >= r.y0 && cy <= r.y1 && ((quad >> 10) & 31u) == 0u)
                            quad |= (((cy == r.y1 && (r.wall6 & 4u)) || (cy == r.y0 && (r.wall6 & 8u))) ? kCodeWall : kCodeSeen) << 10;
                    }
                    const uint32_t mid = (quad >> 10) & 31u;
                    if (dyi == 2 && dxi == 3) nbr |= mid;          // +x -> direction 0
                    if (dyi == 2 && dxi == 1) nbr |= mid << 5;     // -x
                    if (dxi == 2 && dyi == 3) nbr |= mid << 10;    // +y
                    if (dxi == 2 && dyi == 1) nbr |= mid << 15;    // -y
                }
                if (obs_row != nullptr) {
                    if (STAGED) reinterpret_cast<uint32_t *>(obs_row)[dxi * 4 + dyi] = quad;
                    else {
                        float4 v;
                        v.x = lut[quad & 31u]; v.y = lut[(quad >> 5) & 31u];
                        v.z = lut[(quad >> 10) & 31u]; v.w = lut[quad >> 15];
                        store_stream(reinterpret_cast<float4 *>(obs_row) + (dxi * 4 + dyi), v);
                    }
                }
            }
        }
    }
    if (obs_row != nullptr) write_scalars<G, STAGED>(P, lane, sc, lut, obs_row);
    return nbr;
}

// ---------------------------------------------------------------------------------------------------------------
// reset (CubicEnv.py:77-108) of one env, room/start already chosen.  Two halves around the group's OR-reduction.
// ---------------------------------------------------------------------------------------------------------------
struct ResetCtx { int x, y, z; uint32_t room, episode_after; Rays r; };

// internal_grid = full(-1) (:84): nothing seen, nothing counted.  (The overflow bytes need no clearing: one is only read
// for a cell whose code says so, and it is written when the code first does.)  Lane's share; a group_sync follows.
template <int G>
NAV3D_HD void reset_clear(const EngineParams &P, int env, int lane, uint32_t room_idx) {
    const uint32_t n = k_bytes(P.rooms[room_idx]) >> 4;
    uint4 *k4 = reinterpret_cast<uint4 *>(P.know + (unsigned long long)env * P.env_stride);
    const uint4 zero = make_uint4(0u, 0u, 0u, 0u);
    for (uint32_t i = lane; i < n; i += G) k4[i] = zero;
}

template <int G, bool STAGED = false>
NAV3D_HD uint32_t reset_lane(const EngineParams &P, int env, int lane, uint32_t room_idx, uint32_t k,
                             uint32_t episode_after, const float *lut, float *obs_row, ResetCtx &c,
                             const MarkQueue *mq = nullptr) {
    const RoomDev R = P.rooms[room_idx];
    uint8_t *envk = P.know + (unsigned long long)env * P.env_stride;
    uint32_t cell = ldg(P.free_cells + R.free_off + k);               // possible_start_pose[k] (:450-462)
    if (P.room_start != nullptr) {                                    // ... unless the room file fixes the start (:461)
        const uint32_t fixed = ldg(P.room_start + room_idx);
        if (fixed != 0xffffffffu) cell = fixed;
    }
    c.x = cell & 0xff; c.y = (cell >> 8) & 0xff; c.z = (cell >> 16) & 0xff;
    c.room = room_idx; c.episode_after = episode_after;
    c.r = cast_rays(P, R, c.x, c.y, c.z);                             // get_obs() inside reset (:108)
    ObsScalars sc;
    sc.facing = 0; sc.last_action = 0; sc.was_near_wall = 0; sc.last_bump = 0; sc.down = c.r.down;
    sc.visited = 1; sc.total_free = R.n_free;
    // internal_grid[start] = 1 (:85), then the first sensing pass
    return observe<G, STAGED>(P, R, envk, lane, c.x, c.y, c.z, c.r, 1, true, true, -1, sc, lut, obs_row, mq);
}

NAV3D_HD void reset_commit(const EngineParams &P, int env, int lane, const ResetCtx &c, uint32_t nbr) {
    if (lane != 0) return;
    EnvState st;
    st.x = (uint8_t)c.x; st.y = (uint8_t)c.y; st.z = (uint8_t)c.z; st.facing = 0;
    st.last_action = 0; st.flags = (uint8_t)(c.r.near_wall ? kNearWall : 0u); st.down = (uint8_t)c.r.down;
    st.blocked6 = (uint8_t)c.r.blocked6;
    st.step_count = 0; st.visited_count = 1; st.bump_count = 0; st.room = (uint16_t)c.room;
    st.nbr = nbr; st.ret_centi = 0; st.episode = c.episode_after; st.own_count = 1;
    st.pad[0] = st.pad[1] = st.pad[2] = 0;
    P.states[env] = st;
}

template <int G>
NAV3D_HD void reset_env(const EngineParams &P, int env, int lane, int lane_in_warp, uint32_t room_idx, uint32_t k,
                        uint32_t episode_after, const float *lut, float *obs_row) {
    ResetCtx c;
    reset_clear<G>(P, env, lane, room_idx);
    group_sync<G>(lane_in_warp);
    const uint32_t part = reset_lane<G>(P, env, lane, room_idx, k, episode_after, lut, obs_row, c);
    reset_commit(P, env, lane, c, group_or<G>(part, lane_in_warp));
}

NAV3D_HD void reset_picks(const EngineParams &P, int env, uint32_t episode, uint32_t &room, uint32_t &k) {
    uint32_t u0, u1;
    philox4x32_10(P.env_id0 + (uint32_t)env, episode, 0u, kStreamReset, P.seed_lo, P.seed_hi, u0, u1);
    room = mulhi_range(u0, (uint32_t)P.n_rooms);                      // random.choice(self.rooms) (:407)
    k = mulhi_range(u1, ldg(&P.rooms[room].n_free));                  // random.choice(possible_start_pose) (:462)
}

template <int G>
NAV3D_HD void reset_env_philox(const EngineParams &P, int env, int lane, int lane_in_warp, uint32_t episode,
                               const float *lut, float *obs_row) {
    uint32_t room, k;
    reset_picks(P, env, episode, room, k);
    reset_env<G>(P, env, lane, lane_in_warp, room, k, episode + 1u, lut, obs_row);
}

// ---------------------------------------------------------------------------------------------------------------
// step (CubicEnv.py:110-132) of one env.  Two halves around the group's OR-reduction of the neighbour codes.
// ---------------------------------------------------------------------------------------------------------------
struct EpisodeRec { float episode_return; int32_t length, bumps, visited, total_free, room, terminated, truncated; };

struct StepCtx {                   // what the second half needs; identical in every lane of the group
    EnvState st;                   // the record the step started from
    int x, y, z, facing, a, c_new, down;
    uint32_t flags, step_count, visited, n_free, blocked6;
    uint32_t ovf_at;               // G > 1: offset in the env's block of the agent cell's overflow byte
    bool bumped, explored, done, truncated, will_reset, near_wall;
};

// REG_STATE (fused multi-step rollouts): the env's record lives in the caller's registers (`rs`, every lane holds a
// copy and every lane computes the new one) instead of making a round trip through global memory each step.
// STAGED (G == 1): the observation row is assembled in `stage_row` (shared memory) and `*dst_slot` receives the global row
// it belongs to (obs or terminal_obs; NULL = nobody reads it); the warp writes it out afterwards.
template <int G, bool REG_STATE = false, bool STAGED = false>
NAV3D_HD uint32_t step_lane(const EngineParams &P, const StepIO &io, int env, int lane, int action, const float *lut,
                            long long row /* row index for the output arrays */, const EnvState *rs, StepCtx &c,
                            float *stage_row = nullptr, float **dst_slot = nullptr, const MarkQueue *mq = nullptr) {
    const EnvState st = REG_STATE ? *rs : P.states[env];
    const RoomDev R = P.rooms[st.room];
    uint8_t *envk = P.know + (unsigned long long)env * P.env_stride;
    c.st = st;
    c.n_free = R.n_free;

    const int a = action < 0 ? 0 : (action > 5 ? 5 : action);
    uint32_t flags = st.flags;
    if (flags & kNearWall) flags = (flags | kWasNearWall) & ~kNearWall;          // :111-113
    const uint32_t step_count = st.step_count == 0xffffu ? 0xffffu : st.step_count + 1u;   // :115
    c.truncated = step_count >= R.n_free;                                        // :116, max_steps = total_free (:459)

    // do_action (:134-166).  Whether the move bumps and the counter of the target cell were worked out by the previous
    // step's observation (record fields blocked6 / nbr), so the new position, the new counter and with them every address
    // and every branch of this step are known as soon as the record arrives.
    int x = st.x, y = st.y, z = st.z, facing = st.facing;
    uint32_t dir;                                                                // index into blocked6 / nbr
    if (a < 4) {
        facing = (facing + a) & 3;                                               // table :135-140 == rotate by a; :148-151
        dir = (0x1302u >> (facing * 4)) & 3u;                                    // N -> +y (2), E -> +x (0), S -> -y (3), W -> -x (1)
    } else dir = (uint32_t)a;                                                    // 4 -> +z, 5 -> -z
    const bool moved = !((st.blocked6 >> dir) & 1u);                             // _mark_visited :328-332
    int c_old = st.own_count;
    if (moved) {
        x += (dir == 0) - (dir == 1);
        y += (dir == 2) - (dir == 3);
        z += (dir == 4) - (dir == 5);
        const uint32_t tcode = (st.nbr >> (5u * dir)) & 31u;                     // >= 2: a free cell the rays have seen
        c_old = (int)tcode - 2;
        if (tcode == kCodeOverflow) c_old = kOverflowBase + envk[P.ovf_off + ovf_index(R, x, y, z)];
    }
    // entering: 0 -> 1 (+visited, explored) or v -> v+1 (:335-341); then the unconditional += 1 at the final
    // position (:165-166).  A bump only gets the latter.
    c.bumped = !moved;
    c.explored = moved && c_old == 0;
    c.c_new = imin(255, c_old + (moved ? 2 : 1));
    c.visited = st.visited_count + (c.explored ? 1u : 0u);
    // termination test of compute_reward (:212-214): visited/total >= 0.84 in f64.  For total <= 65536 this is
    // exactly 25*visited >= 21*total (tests/test_host_logic.py::test_finish_threshold_integer_form).
    c.done = 25u * c.visited >= 21u * R.n_free;
    c.will_reset = P.auto_reset && (c.done || c.truncated);
    c.x = x; c.y = y; c.z = z; c.facing = facing; c.a = a; c.flags = flags; c.step_count = step_count;

    const Rays r = cast_rays(P, R, x, y, z);
    c.down = r.down; c.blocked6 = r.blocked6; c.near_wall = r.near_wall != 0;
    // The agent cell's exact count past 28.  With G > 1 the sibling lanes read the byte of the cell they move into
    // above, in the same step, so the store waits for step_commit, after the group's reduction.
    if (G == 1) {
        if (c.c_new >= kOverflowBase && !c.will_reset) envk[P.ovf_off + ovf_index(R, x, y, z)] = (uint8_t)(c.c_new - kOverflowBase);
    } else c.ovf_at = P.ovf_off + ovf_index(R, x, y, z);

    // get_obs (:122)
    float *orow = io.obs ? io.obs + row * kObsDim : nullptr;
    if (c.will_reset) orow = io.terminal_obs ? io.terminal_obs + row * kObsDim : nullptr;
    ObsScalars sc;
    sc.facing = facing; sc.last_action = st.last_action; sc.was_near_wall = (flags & kWasNearWall) != 0;
    sc.last_bump = (flags & kLastBump) != 0; sc.down = r.down; sc.visited = c.visited; sc.total_free = R.n_free;
    if (STAGED) { *dst_slot = orow; if (orow != nullptr) orow = stage_row; }
    if (c.will_reset && orow == nullptr) return 0u;        // nothing observes the last state of the episode
    return observe<G, STAGED>(P, R, envk, lane, x, y, z, r, c.c_new, c.explored, !c.will_reset, moved ? (int)dir : -2, sc,
                              lut, orow, mq);
}

template <int G, bool REG_STATE = false>
NAV3D_HD void step_commit(const EngineParams &P, const StepIO &io, int env, int lane, const StepCtx &c, uint32_t nbr,
                          long long row, EnvState *rs, uint32_t *done_bits) {
    if (!REG_STATE && lane != 0) return;
    const bool writer = lane == 0;
    const EnvState &st = c.st;
    const RewardParams &w = P.rw;
    uint32_t flags = c.flags;
    if (c.near_wall) flags |= kNearWall;
    // compute_reward (:169-224), same operations in the same order, f64
    double rew = w.step_cost;
    const double pen = (double)c.c_new * w.revisit_unit;
    const double revisit = (pen < w.revisit_cap) ? pen : w.revisit_cap;
    rew -= revisit;
    int cents = w.c_step - reward_centi(revisit);
    uint32_t bump_count = st.bump_count;
    if (c.bumped) {
        flags |= kLastBump;
        if (bump_count != 0xffffu) bump_count++;
        rew += w.crash_penalty;
    } else {
        flags &= ~kLastBump;
        if (flags & kWasNearWall) { flags &= ~kWasNearWall; rew += w.near_wall_bonus; cents += w.c_near_wall; }
        if (st.last_action != 2 && c.a == st.last_action && st.last_action < 4) { rew += w.repeat_bonus; cents += w.c_repeat; }
        if (st.last_action == 2 && c.a == 2) { rew -= w.reverse_penalty; cents -= w.c_reverse; }
    }
    if (c.explored) { rew += w.explore_bonus; cents += w.c_explore; }
    if (c.done) { flags |= kDone; rew += w.finish_bonus; cents += w.c_finish; }
    if (c.truncated) { rew += w.truncation_penalty; cents += w.c_trunc; }
    const int ret_centi = add_saturate(st.ret_centi, cents);

    if (G > 1 && writer && c.c_new >= kOverflowBase && !c.will_reset)
        P.know[(unsigned long long)env * P.env_stride + c.ovf_at] = (uint8_t)(c.c_new - kOverflowBase);
    if (writer) {
        if (!REG_STATE || io.reward) store_stream(io.reward + row, (float)rew);
        if (io.reward64) io.reward64[row] = rew;
        if (!REG_STATE || io.terminated) io.terminated[row] = c.done ? 1 : 0;
        if (!REG_STATE || io.truncated) io.truncated[row] = c.truncated ? 1 : 0;
    }
    if (REG_STATE && done_bits) *done_bits = (c.done ? 1u : 0u) | (c.truncated ? 2u : 0u);
    if (writer && (c.done || c.truncated) && io.episodes) {
        EpisodeRec ep;
        ep.episode_return = (float)((double)ret_centi / 100.0 + (double)bump_count * w.crash_penalty);
        ep.length = (int32_t)c.step_count; ep.bumps = (int32_t)bump_count; ep.visited = (int32_t)c.visited;
        ep.total_free = (int32_t)c.n_free; ep.room = st.room; ep.terminated = c.done; ep.truncated = c.truncated;
        reinterpret_cast<EpisodeRec *>(io.episodes)[row] = ep;
    }
    if (!c.will_reset) {
        EnvState ns;
        ns.x = (uint8_t)c.x; ns.y = (uint8_t)c.y; ns.z = (uint8_t)c.z; ns.facing = (uint8_t)c.facing;
        ns.last_action = (uint8_t)c.a; ns.flags = (uint8_t)flags; ns.down = (uint8_t)c.down; ns.blocked6 = (uint8_t)c.blocked6;
        ns.step_count = (uint16_t)c.step_count; ns.visited_count = (uint16_t)c.visited; ns.bump_count = (uint16_t)bump_count;
        ns.room = st.room; ns.nbr = nbr; ns.ret_centi = ret_centi; ns.episode = st.episode;
        ns.own_count = (uint8_t)c.c_new; ns.pad[0] = ns.pad[1] = ns.pad[2] = 0;
        if (REG_STATE) *rs = ns;
        else P.states[env] = ns;
    }
}

// Returns true when the env finished its episode and must be reset by the caller (auto_reset).
template <int G, bool REG_STATE = false, bool STAGED = false>
NAV3D_HD bool step_env(const EngineParams &P, const StepIO &io, int env, int lane, int lane_in_warp, int action,
                       const float *lut, long long row, EnvState *rs = nullptr, uint32_t *done_bits = nullptr,
                       float *stage_row = nullptr, float **dst_slot = nullptr, const MarkQueue *mq = nullptr) {
    StepCtx c;
    const uint32_t part = step_lane<G, REG_STATE, STAGED>(P, io, env, lane, action, lut, row, rs, c, stage_row, dst_slot, mq);
    step_commit<G, REG_STATE>(P, io, env, lane, c, group_or<G>(part, lane_in_warp), row, rs, done_bits);
    return c.will_reset;
}

// The [T][n_envs] arrays of one fused rollout (nav3d_rollout_actions; nav3d_rollout_random fills obs / obs_last / reward
// and its own done / actions_out / t0, and leaves the rest null).  Any output may be null; with obs == null only the last
// step's rows are formed, into obs_last [n_envs][80].
struct RolloutIO {
    const uint8_t *actions;        // caller-supplied actions; values > 5 act as 5 (step_lane clamps)
    float *obs, *obs_last, *reward;
    double *reward64;
    uint8_t *terminated, *truncated;
    float *terminal_obs;
    void *episodes;                // nav3d_episode*
    uint8_t *done, *actions_out;   // Philox actions: terminated | truncated, and the actions played
    uint32_t t0;                   // Philox actions: step index of the first step in the env's action stream
};

// The StepIO of step t of a fused rollout: rows stay indexed by env, the row offsets are 64-bit ([32][2^20][80] f32 is
// 10.7 GB).
NAV3D_HD StepIO rollout_step_io(const RolloutIO &ro, int t, int T, long long n_envs) {
    const long long r0 = (long long)t * n_envs;
    StepIO io;
    io.actions = nullptr;
    io.obs = ro.obs ? ro.obs + r0 * kObsDim : (t == T - 1 ? ro.obs_last : nullptr);
    io.reward = ro.reward ? ro.reward + r0 : nullptr;
    io.reward64 = ro.reward64 ? ro.reward64 + r0 : nullptr;
    io.terminated = ro.terminated ? ro.terminated + r0 : nullptr;
    io.truncated = ro.truncated ? ro.truncated + r0 : nullptr;
    io.terminal_obs = ro.terminal_obs ? ro.terminal_obs + r0 * kObsDim : nullptr;
    io.episodes = ro.episodes ? static_cast<EpisodeRec *>(ro.episodes) + r0 : nullptr;
    io.env0 = 0; io.env_n = (int)n_envs;
    return io;
}
NAV3D_HD int rollout_action(const RolloutIO &ro, int t, long long n_envs, long long env) {
    return ro.actions[(long long)t * n_envs + env];
}

// ===============================================================================================================
// simpleEnv (envs/simpleEnv.py): ternary knowledge grid, ray-cell observations, goal reward
//   step :109-150, do_action :152-186, compute_reward :189-217, get_obs :219-265, _mark_visited :273-298,
//   _sense_direction :301-337, reset :79-107, load_room's start/goal picks :404-426.
// Knowledge: 2 bits per cell — 00 unknown (-1), 01 seen free (0), 10 visited (1), 11 marked blocked (2) — stored per (x,y)
// column as one u32 (low half = bit-plane 0, high half = bit-plane 1, bit z), in 4x4-column tiles of 64 B.
// EnvState reuse: down = goal x, blocked6 = goal y, own_count = goal z.
// ===============================================================================================================
NAV3D_HD uint32_t k2_bytes(const RoomDev &R) { return (uint32_t)R.ntx * R.nty * 64u; }
NAV3D_HD int k2_code(uint32_t w, int z) { return (int)(((w >> z) & 1u) | (((w >> (16 + z)) & 1u) << 1)); }
NAV3D_HD float k2_value(int code) { return code == 0 ? -1.0f : (float)(code - 1); }

NAV3D_HD void simple_ray(unsigned long long w, int p, int n, bool up, int &ext, int &nfree) {
    int wall;
    if (up) ray_up<false>(w, p, n, ext, wall); else ray_down<false>(w, p, n, ext, wall);
    nfree = ext - wall;
}

// get_obs (simpleEnv.py:219-265) at (x,y,z): marks the knowledge and writes the 6L+7 floats.  `centre` is the centre
// column's word as every lane holds it (after the move's visit update); the updated word is stored by lane 0.
// The six rays are evaluated once per absolute axis direction a (0 +x, 1 -x, 2 +y, 3 -y, 4 +z, 5 -z) and kept packed in
// registers — free count in byte a of `nf6`, "a wall stopped it" / "a 2 is appended" in bit a of `wall6` / `blk6` — so that
// the per-cell loop below needs no indexed local array.
template <int G>
NAV3D_HD void simple_observe(const EngineParams &P, const RoomDev &R, uint32_t *K, int lane, int lane_in_warp, int x, int y,
                             int z, int facing, uint32_t centre_mem, uint32_t centre, int last_action, float *obs_row) {
    const int L = P.L, W = R.W, D = R.D, H = R.H;
    const unsigned long long wx = ldg(P.occ64 + R.occx_off + (uint32_t)(y * H + z));
    const unsigned long long wy = ldg(P.occ64 + R.occy_off + (uint32_t)(x * H + z));
    const unsigned long long wz = ldg(P.occz + R.occz_off + (uint32_t)(x * D + y));
    unsigned long long nf6 = 0;
    uint32_t wall6 = 0, blk6 = 0;
    {
        int ext, nfree, room_left;
#define NAV3D_SIMPLE_RAY(a, W_, P_, UP, LEFT)                                                               \
        room_left = (LEFT); simple_ray(W_, P_, imin(L, room_left), UP, ext, nfree);                         \
        nf6 |= (unsigned long long)nfree << (8 * (a));                                                      \
        wall6 |= (uint32_t)(ext > nfree) << (a);                     /* a wall stopped the ray (:321-324) */ \
        blk6 |= (uint32_t)((ext > nfree) || (nfree == room_left && nfree < L)) << (a);   /* ... or the room ended (:311-319) */
        NAV3D_SIMPLE_RAY(0, wx, x, true, W - 1 - x)
        NAV3D_SIMPLE_RAY(1, wx, x, false, x)
        NAV3D_SIMPLE_RAY(2, wy, y, true, D - 1 - y)
        NAV3D_SIMPLE_RAY(3, wy, y, false, y)
        NAV3D_SIMPLE_RAY(4, wz, z, true, H - 1 - z)
        NAV3D_SIMPLE_RAY(5, wz, z, false, z)
#undef NAV3D_SIMPLE_RAY
    }
    // vertical rays: all in the centre column; fold their marks into one word
    const int nup = (int)((nf6 >> 32) & 0xff), ndn = (int)((nf6 >> 40) & 0xff);
    uint32_t free_z = (((1u << nup) - 1u) << (z + 1)) | (((1u << ndn) - 1u) << (z - ndn));
    uint32_t block_z = 0;
    if (wall6 & 16u) block_z |= 1u << (z + nup + 1);
    else if ((blk6 & 16u) && nup >= 1) block_z |= 1u << (z + nup);                 // last in-bounds cell becomes 2 (:314-317)
    if (wall6 & 32u) block_z |= 1u << (z - ndn - 1);
    else if ((blk6 & 32u) && ndn >= 1) block_z |= 1u << (z - ndn);
    const uint32_t lo0 = centre & 0xffffu, hi0 = centre >> 16;
    const uint32_t lo1 = lo0 | (free_z & ~hi0 & ~lo0);                           // unknown -> seen (:327-328)
    const uint32_t centre_seen = lo1 | (hi0 << 16);                              // what the ray cells report
    const uint32_t centre_new = (lo1 | block_z) | ((hi0 | block_z) << 16);
    // ray order :243: forward, left, right, backward, up, down.  Headings N=+y, E=+x, S=-y, W=-x; heading -> axis
    // direction index is the same nibble table the move uses (N -> 2, E -> 0, S -> 3, W -> 1).
    // The four horizontal rays, CH ray cells per lane per round: every word of a round is loaded before any is used or
    // stored (a load -> test -> store chain per cell would serialise one memory latency per cell).
    constexpr int CH = 4;
    int adir[4], ddx[4], ddy[4];
#pragma unroll
    for (int d = 0; d < 4; d++) {
        const int h = (facing + ((0x2130 >> (4 * d)) & 3)) & 3;                  // fwd +0, left +3, right +1, back +2
        adir[d] = (0x1302 >> (4 * h)) & 3;
        ddx[d] = (h == 1) - (h == 3); ddy[d] = (h == 0) - (h == 2);
    }
    for (int s0 = 1; s0 <= L; s0 += CH * G) {
        uint32_t w[4][CH];
#pragma unroll
        for (int d = 0; d < 4; d++) {
            const int nfree = (int)((nf6 >> (8 * adir[d])) & 0xff);
            const bool wall = (wall6 >> adir[d]) & 1u, blocked = (blk6 >> adir[d]) & 1u;
#pragma unroll
            for (int u = 0; u < CH; u++) {
                const int sN = s0 + lane + u * G;
                const bool need = sN <= L && (sN <= nfree || (sN == nfree + 1 && blocked && wall));
                w[d][u] = need ? K[s_index(R, x + ddx[d] * sN, y + ddy[d] * sN)] : 0u;
            }
        }
#pragma unroll
        for (int d = 0; d < 4; d++) {
            const int nfree = (int)((nf6 >> (8 * adir[d])) & 0xff);
            const bool wall = (wall6 >> adir[d]) & 1u, blocked = (blk6 >> adir[d]) & 1u;
#pragma unroll
            for (int u = 0; u < CH; u++) {
                const int sN = s0 + lane + u * G;
                if (sN > L) continue;
                float v = -1.0f;                                              // padding (:334-335)
                const uint32_t old = w[d][u];
                uint32_t n = old;
                bool touch = false;
                if (sN <= nfree) {
                    int code = k2_code(old, z);
                    if (code == 0) { code = 1; n |= 1u << z; }                // -1 -> 0
                    v = k2_value(code);
                    if (sN == nfree && blocked && !wall) n |= (1u << z) | (1u << (16 + z));   // then becomes 2
                    touch = true;
                } else if (sN == nfree + 1 && blocked) {
                    v = 2.0f;
                    if (wall) { n = old | (1u << z) | (1u << (16 + z)); touch = true; }
                }
                if (touch && n != old) K[s_index(R, x + ddx[d] * sN, y + ddy[d] * sN)] = n;
                if (obs_row) obs_row[d * L + sN - 1] = v;
            }
        }
    }
    // the two vertical rays: all of their cells are in the centre column's word
#pragma unroll
    for (int d = 4; d < 6; d++) {
        const int dz = (d == 4) ? 1 : -1;
        const int nfree = (int)((nf6 >> (8 * d)) & 0xff);
        const bool blocked = (blk6 >> d) & 1u;
        for (int sN = 1 + lane; sN <= L; sN += G) {
            float v = -1.0f;
            if (sN <= nfree) v = k2_value(k2_code(centre_seen, z + dz * sN));
            else if (sN == nfree + 1 && blocked) v = 2.0f;
            if (obs_row) obs_row[d * L + sN - 1] = v;
        }
    }
    if (obs_row) {
        for (int i = lane; i < 7; i += G) {
            float v = (float)last_action;
            if (i < 6) {
                int a = i;
                if (i < 4) { const int h = (facing + ((0x2130 >> (4 * i)) & 3)) & 3; a = (0x1302 >> (4 * h)) & 3; }
                v = ldg(P.dist_lut + (int)((nf6 >> (8 * a)) & 0xff));
            }
            obs_row[6 * L + i] = v;
        }
    }
    if (lane == 0 && centre_new != centre_mem) K[s_index(R, x, y)] = centre_new;
    (void)lane_in_warp;
}

template <int G>
NAV3D_HD void simple_reset_env(const EngineParams &P, int env, int lane, int lane_in_warp, uint32_t room_idx, uint32_t k,
                               uint32_t kg, uint32_t episode_after, float *obs_row) {
    const RoomDev R = P.rooms[room_idx];
    uint32_t *K = reinterpret_cast<uint32_t *>(P.know + (unsigned long long)env * P.env_stride);
    {
        uint4 zero = make_uint4(0u, 0u, 0u, 0u);
        uint4 *k4 = reinterpret_cast<uint4 *>(K);
        const uint32_t n = k2_bytes(R) >> 4;
        for (uint32_t i = lane; i < n; i += G) k4[i] = zero;
    }
    group_sync<G>(lane_in_warp);
    const uint32_t cell = ldg(P.free_cells + R.free_off + k), goal = ldg(P.free_cells + R.free_off + kg);
    const int x = cell & 0xff, y = (cell >> 8) & 0xff, z = (cell >> 16) & 0xff;
    const uint32_t centre = 1u << (16 + z);                                       // internal_grid[start] = 1 (:85)
    simple_observe<G>(P, R, K, lane, lane_in_warp, x, y, z, 0, 0u, centre, 0, obs_row);
    if (lane == 0) {
        EnvState st;
        st.x = (uint8_t)x; st.y = (uint8_t)y; st.z = (uint8_t)z; st.facing = 0; st.last_action = 0; st.flags = 0;
        st.down = (uint8_t)(goal & 0xff); st.blocked6 = (uint8_t)((goal >> 8) & 0xff); st.own_count = (uint8_t)((goal >> 16) & 0xff);
        st.step_count = 0; st.visited_count = 1; st.bump_count = 0; st.ret_centi = 0; st.nbr = 0;
        st.episode = episode_after; st.room = (uint16_t)room_idx; st.pad[0] = st.pad[1] = st.pad[2] = 0;
        P.states[env] = st;
    }
}

template <int G>
NAV3D_HD void simple_reset_env_philox(const EngineParams &P, int env, int lane, int lane_in_warp, uint32_t episode,
                                      float *obs_row) {
    uint32_t u[4];
    philox4x32_10_4(P.env_id0 + (uint32_t)env, episode, 0u, kStreamReset, P.seed_lo, P.seed_hi, u);
    const uint32_t room = mulhi_range(u[0], (uint32_t)P.n_rooms);                 // random.choice(self.rooms) (:351)
    const uint32_t nf = ldg(&P.rooms[room].n_free);
    simple_reset_env<G>(P, env, lane, lane_in_warp, room, mulhi_range(u[1], nf), mulhi_range(u[2], nf), episode + 1u, obs_row);
}

// STAGED (G == 1, the thread-per-env kernel): the 6L+7 floats go to `stage_row` (shared memory), `*dst_slot` receives the
// global row they belong to (NULL = none), and the auto-reset is left to the caller (returns true when it is due), which
// runs it after the warp has written the staged rows out.
template <int G, bool STAGED = false>
NAV3D_HD bool simple_step_env(const EngineParams &P, const StepIO &io, int env, int lane, int lane_in_warp, int action,
                              long long row, float *stage_row = nullptr, float **dst_slot = nullptr) {
    const EnvState st = P.states[env];
    const RoomDev R = P.rooms[st.room];
    uint32_t *K = reinterpret_cast<uint32_t *>(P.know + (unsigned long long)env * P.env_stride);
    const int a = action < 0 ? 0 : (action > 5 ? 5 : action);
    const uint32_t step_count = st.step_count == 0xffffu ? 0xffffu : st.step_count + 1u;
    const bool truncated = step_count >= R.n_free;                                 // :110-111, max_steps = total_free (:404)
    int x = st.x, y = st.y, z = st.z, facing = st.facing;
    int tx = x, ty = y, tz = z;
    if (a < 4) {
        facing = (facing + a) & 3;
        tx += (facing == 1) - (facing == 3);
        ty += (facing == 0) - (facing == 2);
    } else tz += (a == 4) ? 1 : -1;
    bool moved = false;
    if (tx >= 0 && tx < R.W && ty >= 0 && ty < R.D && tz >= 0 && tz < R.H) {
        const uint32_t ow = ldg(P.occz + R.occz_off + (uint32_t)(tx * R.D + ty));
        moved = !((ow >> tz) & 1u);
    }
    if (moved) { x = tx; y = ty; z = tz; }
    const uint32_t centre_mem = K[s_index(R, x, y)];
    uint32_t centre = centre_mem;
    group_sync<G>(lane_in_warp);                 // every lane holds the old word before lane 0 rewrites it
    bool explored = false;
    if (moved) {                                 // _mark_visited :286-294: 0 or -1 become 1; 1 and 2 stay
        const int code = k2_code(centre, z);
        if (code <= 1) { explored = true; centre = (centre & ~(1u << z)) | (1u << (16 + z)); }
    }
    const uint32_t visited = st.visited_count + (explored ? 1u : 0u);
    const int gx = st.down, gy = st.blocked6, gz = st.own_count;
    bool done = (st.flags & kDone) != 0;
    int hits = 0;
    for (int i = 0; i < 5; i++) if (x == gx && y == gy && z - i == gz) hits++;     // :203-208
    done = done || hits > 0;
    const bool will_reset = P.auto_reset && (done || truncated);
    float *orow = io.obs + row * P.obs_dim;
    if (will_reset) orow = io.terminal_obs ? io.terminal_obs + row * P.obs_dim : nullptr;
    if (STAGED) { *dst_slot = orow; if (orow) orow = stage_row; }
    if (!will_reset || orow)
        simple_observe<G>(P, R, K, lane, lane_in_warp, x, y, z, facing, centre_mem, centre, a, orow);
    if (lane == 0) {
        double rew = -0.1;                                                         // compute_reward :191-215
        int cents = -10;
        uint32_t bump_count = st.bump_count;
        if (!moved) { if (bump_count != 0xffffu) bump_count++; rew += -10.0; cents -= 1000; }
        if (a != 2 && a < 4) { rew += 0.05; cents += 5; }                          // last_action was already set to a (:139)
        for (int i = 0; i < hits; i++) { rew += 100.0; cents += 10000; }
        if (explored) { rew += 1.0; cents += 100; }
        const int ret_centi = st.ret_centi + cents;
        store_stream(io.reward + row, (float)rew);
        if (io.reward64) io.reward64[row] = rew;
        io.terminated[row] = done ? 1 : 0;
        io.truncated[row] = truncated ? 1 : 0;
        if ((done || truncated) && io.episodes) {
            EpisodeRec ep;
            ep.episode_return = (float)((double)ret_centi / 100.0);
            ep.length = (int32_t)step_count; ep.bumps = (int32_t)bump_count; ep.visited = (int32_t)visited;
            ep.total_free = (int32_t)R.n_free; ep.room = st.room; ep.terminated = done; ep.truncated = truncated;
            reinterpret_cast<EpisodeRec *>(io.episodes)[row] = ep;
        }
        if (!will_reset) {
            EnvState ns = st;
            ns.x = (uint8_t)x; ns.y = (uint8_t)y; ns.z = (uint8_t)z; ns.facing = (uint8_t)facing; ns.last_action = (uint8_t)a;
            ns.flags = (uint8_t)(done ? kDone : 0u);
            ns.step_count = (uint16_t)step_count; ns.visited_count = (uint16_t)visited; ns.bump_count = (uint16_t)bump_count;
            ns.ret_centi = ret_centi;
            P.states[env] = ns;
        }
    }
    if (will_reset && !STAGED) {
        group_sync<G>(lane_in_warp);
        simple_reset_env_philox<G>(P, env, lane, lane_in_warp, st.episode, io.obs + row * P.obs_dim);
    }
    return will_reset;
}

// ---------------------------------------------------------------------------------------------------------------
// env-state blobs (nav3d_save_envs / nav3d_load_envs): the complete state of one env, self-describing, fixed size.
//   [0, 32)          BlobHeader
//   [32, 64)         EnvState, unchanged
//   [64, know_off)   the env's current observation row (obs_dim f32), padded to a multiple of 16 bytes (padding not written)
//   [know_off, +env_stride)  the knowledge block with the engine's own offsets: K at 0, overflow bytes at ovf_off.  Only the
//                    live part of the blob's room is written: k_bytes (simpleEnv k2_bytes) of K and W*D*H overflow bytes —
//                    the range a reset clears and a step can read.
// The per-env copy is split over `nl` lanes (lane = 0 .. nl-1); the device kernels run it with a warp per env, the host
// emulation with one lane.
// ---------------------------------------------------------------------------------------------------------------
constexpr uint32_t kBlobMagic = 0x4e334445u;     // "ED3N" little-endian
constexpr uint32_t kBlobVersion = 1u;
constexpr uint32_t kBlobObsOff = 64;
constexpr uint8_t kBlobLoaded = 0, kBlobBadEnv = 1, kBlobInvalid = 2;   // nav3d_load_envs status codes

struct alignas(16) BlobHeader {
    uint32_t magic, version;
    unsigned long long signature;  // engine signature (nav3d_load_rooms): env kind, L, env_stride and the room table
    uint32_t room;                 // == EnvState::room
    uint32_t k_live, ovf_live;     // bytes of K and of the overflow volume the blob holds
    uint32_t obs_dim;
};
static_assert(sizeof(BlobHeader) == 32, "blob header");

NAV3D_HD bool simple_kind(const EngineParams &P) { return P.obs_dim != kObsDim; }
NAV3D_HD unsigned long long blob_know_off(const EngineParams &P) {
    return kBlobObsOff + (((unsigned long long)P.obs_dim * 4u + 15u) & ~15ull);
}
NAV3D_HD unsigned long long blob_bytes(const EngineParams &P) { return blob_know_off(P) + P.env_stride; }
NAV3D_HD uint32_t blob_k_live(const EngineParams &P, const RoomDev &R) { return simple_kind(P) ? k2_bytes(R) : k_bytes(R); }
NAV3D_HD uint32_t blob_ovf_live(const EngineParams &P, const RoomDev &R) {
    return simple_kind(P) ? 0u : (uint32_t)R.W * R.D * R.H;
}

NAV3D_HD uint4 load_stream(const uint4 *p) {
#ifdef __CUDA_ARCH__
    return __ldcs(p);
#else
    return *p;
#endif
}
NAV3D_HD void store_stream(uint4 *p, uint4 v) {
#ifdef __CUDA_ARCH__
    __stcs(p, v);
#else
    *p = v;
#endif
}

// n bytes from src to dst, both 16-byte aligned: 16-byte copies (four in flight per lane), then the < 16 tail bytes.
// STREAM_LD / STREAM_ST: evict-first hint on the blob side.
template <bool STREAM_LD, bool STREAM_ST>
NAV3D_HD void copy_live(uint8_t *dst, const uint8_t *src, uint32_t n, int lane, int nl) {
    const uint4 *s4 = reinterpret_cast<const uint4 *>(src);
    uint4 *d4 = reinterpret_cast<uint4 *>(dst);
    const uint32_t n16 = n >> 4;
    uint32_t i = (uint32_t)lane;
    for (; i + 3u * nl < n16; i += 4u * nl) {
        uint4 v[4];
#pragma unroll
        for (int j = 0; j < 4; j++) v[j] = STREAM_LD ? load_stream(s4 + i + j * nl) : s4[i + j * nl];
#pragma unroll
        for (int j = 0; j < 4; j++) {
            if (STREAM_ST) store_stream(d4 + i + j * nl, v[j]);
            else d4[i + j * nl] = v[j];
        }
    }
    for (; i < n16; i += nl) {
        const uint4 v = STREAM_LD ? load_stream(s4 + i) : s4[i];
        if (STREAM_ST) store_stream(d4 + i, v);
        else d4[i] = v;
    }
    for (uint32_t b = (n16 << 4) + (uint32_t)lane; b < n; b += nl) dst[b] = src[b];
}

// One observation row (obs_dim f32; 16-byte aligned rows of CubicEnv move as float4, simpleEnv rows as f32)
template <bool STREAM_ST>
NAV3D_HD void copy_row(float *dst, const float *src, int obs_dim, int lane, int nl) {
    if ((obs_dim & 3) == 0 && ((reinterpret_cast<uintptr_t>(dst) | reinterpret_cast<uintptr_t>(src)) & 15u) == 0) {
        for (int i = lane; i < obs_dim / 4; i += nl) {
            const float4 v = reinterpret_cast<const float4 *>(src)[i];
            if (STREAM_ST) store_stream(reinterpret_cast<float4 *>(dst) + i, v);
            else reinterpret_cast<float4 *>(dst)[i] = v;
        }
    } else {
        for (int i = lane; i < obs_dim; i += nl) {
            if (STREAM_ST) store_stream(dst + i, src[i]);
            else dst[i] = src[i];
        }
    }
}

// save: env -> blob.  An env id outside 0..n_envs-1 gets a header with magic 0, which every load rejects.
NAV3D_HD void save_env_lane(const EngineParams &P, unsigned long long sig, int env, const float *obs, uint8_t *blob, int lane,
                            int nl) {
    BlobHeader *h = reinterpret_cast<BlobHeader *>(blob);
    if (env < 0 || env >= P.n_envs) {
        if (lane == 0) { BlobHeader z{}; *h = z; }
        return;
    }
    const EnvState st = P.states[env];
    const RoomDev R = P.rooms[st.room];
    const uint32_t k_live = blob_k_live(P, R), ovf_live = blob_ovf_live(P, R);
    if (lane == 0) {
        BlobHeader hd;
        hd.magic = kBlobMagic; hd.version = kBlobVersion; hd.signature = sig; hd.room = st.room;
        hd.k_live = k_live; hd.ovf_live = ovf_live; hd.obs_dim = (uint32_t)P.obs_dim;
        *h = hd;
        *reinterpret_cast<EnvState *>(blob + sizeof(BlobHeader)) = st;
    }
    copy_row<true>(reinterpret_cast<float *>(blob + kBlobObsOff), obs + (unsigned long long)env * P.obs_dim, P.obs_dim, lane, nl);
    const uint8_t *envk = P.know + (unsigned long long)env * P.env_stride;
    uint8_t *bk = blob + blob_know_off(P);
    copy_live<false, true>(bk, envk, k_live, lane, nl);
    if (ovf_live) copy_live<false, true>(bk + P.ovf_off, envk + P.ovf_off, ovf_live, lane, nl);
}

// load, part 1: may `blob` be loaded into `env` of this engine?  Reads the header and the record only.
NAV3D_HD uint8_t blob_status(const EngineParams &P, unsigned long long sig, int env, const uint8_t *blob) {
    if (env < 0 || env >= P.n_envs) return kBlobBadEnv;
    const BlobHeader h = *reinterpret_cast<const BlobHeader *>(blob);
    if (h.magic != kBlobMagic || h.version != kBlobVersion || h.signature != sig || h.room >= (uint32_t)P.n_rooms ||
        h.obs_dim != (uint32_t)P.obs_dim)
        return kBlobInvalid;
    const RoomDev R = P.rooms[h.room];
    const EnvState st = *reinterpret_cast<const EnvState *>(blob + sizeof(BlobHeader));
    if (h.k_live != blob_k_live(P, R) || h.ovf_live != blob_ovf_live(P, R) || st.room != h.room || st.x >= R.W ||
        st.y >= R.D || st.z >= R.H)
        return kBlobInvalid;
    return kBlobLoaded;
}

// load, part 2 (a blob that blob_status accepted): blob -> env, and the blob's observation row -> obs.
NAV3D_HD void load_env_lane(const EngineParams &P, int env, const uint8_t *blob, float *obs, int lane, int nl) {
    const BlobHeader h = *reinterpret_cast<const BlobHeader *>(blob);
    uint8_t *envk = P.know + (unsigned long long)env * P.env_stride;
    const uint8_t *bk = blob + blob_know_off(P);
    copy_live<true, false>(envk, bk, h.k_live, lane, nl);
    if (h.ovf_live) copy_live<true, false>(envk + P.ovf_off, bk + P.ovf_off, h.ovf_live, lane, nl);
    copy_row<true>(obs + (unsigned long long)env * P.obs_dim, reinterpret_cast<const float *>(blob + kBlobObsOff), P.obs_dim,
                   lane, nl);
    if (lane == 0) P.states[env] = *reinterpret_cast<const EnvState *>(blob + sizeof(BlobHeader));
}

// Engine signature (host side, nav3d_load_rooms): FNV-1a 64 over the env kind, L, env_stride and, per room, its dims, wall
// code, dense grid and the start cell it resets to (0xffffffff: random).  Lanes, seed, env_id0 and the reward parameters
// are deliberately not part of it: blobs move between engines that differ only in those.
inline unsigned long long sig_bytes(unsigned long long h, const void *p, size_t n) {
    const uint8_t *b = static_cast<const uint8_t *>(p);
    for (size_t i = 0; i < n; i++) { h ^= b[i]; h *= 0x100000001b3ull; }
    return h;
}
inline unsigned long long sig_engine(int kind, int L, unsigned long long env_stride) {
    const int32_t v[2] = {kind, L};
    return sig_bytes(sig_bytes(0xcbf29ce484222325ull, v, sizeof v), &env_stride, sizeof env_stride);
}
inline unsigned long long sig_room(unsigned long long h, int W, int D, int H, int wall_code, const int8_t *grid, uint32_t start) {
    const int32_t v[5] = {W, D, H, wall_code, (int32_t)start};
    return sig_bytes(sig_bytes(h, v, sizeof v), grid, (size_t)W * D * H);
}

}  // namespace nav3d

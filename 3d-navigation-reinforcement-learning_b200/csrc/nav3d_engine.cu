// nav3d_engine.cu — kernels and C ABI of libnav3d_b200.so (see include/nav3d.h).
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -shared -Xcompiler -fPIC (see __graft_entry__.build).
// CUDA runtime only: no torch types, no CPU fallback.
#include "nav3d_core.cuh"
#include "../../include/nav3d.h"

#include <nvtx3/nvToolsExt.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <cstring>
#include <string>
#include <vector>

using namespace nav3d;

static_assert(sizeof(EpisodeRec) == sizeof(nav3d_episode), "episode record layout");
static_assert(kObsDim == NAV3D_OBS_DIM, "obs dim");

namespace {

constexpr int kBlock = 128;   // threads per CTA for the per-env kernels

thread_local std::string g_err;
int fail(int code, const std::string &msg) { g_err = msg; return code; }

#define CUDA_TRY(expr)                                                                                      \
    do {                                                                                                    \
        cudaError_t _e = (expr);                                                                            \
        if (_e != cudaSuccess)                                                                              \
            return fail(NAV3D_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));                \
    } while (0)

__device__ __forceinline__ void fill_lut(float *lut, int L) {
    // nav3d_core.cuh kLut*: observation value of a knowledge code = (clip(v, -2, 20) + 2) / 22 (CubicEnv.py:273-275),
    // k / 5 (:284), d / L (:287); correctly rounded f32 quotients like NumPy's
    for (int t = threadIdx.x; t < kLutSize; t += blockDim.x) {
        if (t < 32) {
            const int v = t == 0 ? -1 : (t == 1 ? -2 : min(t - 2, 20));
            lut[t] = __fdiv_rn((float)(v + 2), 22.0f);
        } else if (t >= kLutFifth && t < kLutFifth + 6) lut[t] = __fdiv_rn((float)(t - kLutFifth), 5.0f);
        else if (t >= kLutDown && t < kLutSize) lut[t] = __fdiv_rn((float)(t - kLutDown), (float)L);
    }
    __syncthreads();
}

// NVTX ranges around the entry points (SURVEY §5): visible in nsys / ncu --nvtx timelines, no-ops otherwise.
struct NvtxRange {
    explicit NvtxRange(const char *name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
};

// ---------------------------------------------------------------------------------------------------------------
// load_room's grid -> packed room (CubicEnv.py:421-459).  One CTA per room.
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) pack_rooms_kernel(const int8_t *__restrict__ dense,
                                                         const uint32_t *__restrict__ dense_off,
                                                         const int32_t *__restrict__ wall_code, RoomDev *rooms,
                                                         uint16_t *occz, unsigned long long *occ64, uint32_t *free_cells,
                                                         uint32_t *n_wall) {
    __shared__ uint32_t cnt[NAV3D_MAX_WIDTH * NAV3D_MAX_DEPTH + 1];
    __shared__ uint32_t walls;
    const int r = blockIdx.x, tid = threadIdx.x, nt = blockDim.x;
    const RoomDev R = rooms[r];
    const int W = R.W, D = R.D, H = R.H;
    const int8_t *g = dense + dense_off[r];
    const int wc = wall_code[r];
    if (tid == 0) walls = 0;
    __syncthreads();
    // column words: occz[x][y], bit z
    const uint32_t zin = H >= 3 ? (((1u << (H - 1)) - 1u) & ~1u) : 0u;   // interior layers 1..H-2
    for (int c = tid; c < W * D; c += nt) {
        const int x = c / D, y = c - x * D;
        uint32_t bits = 0;
        for (int z = 0; z < H; z++) bits |= (g[(size_t)c * H + z] == wc ? 1u : 0u) << z;
        occz[R.occz_off + c] = (uint16_t)bits;
        const bool interior = x >= 1 && x <= W - 2 && y >= 1 && y <= D - 2;
        cnt[c] = interior ? __popc(~bits & zin) : 0u;
        atomicAdd(&walls, (uint32_t)__popc(bits));
    }
    // row words along x: occx[y][z], bit x
    for (int c = tid; c < D * H; c += nt) {
        const int y = c / H, z = c - y * H;
        unsigned long long bits = 0;
        for (int x = 0; x < W; x++) bits |= (unsigned long long)(g[((size_t)x * D + y) * H + z] == wc) << x;
        occ64[R.occx_off + c] = bits;
    }
    // row words along y: occy[x][z], bit y
    for (int c = tid; c < W * H; c += nt) {
        const int x = c / H, z = c - x * H;
        unsigned long long bits = 0;
        for (int y = 0; y < D; y++) bits |= (unsigned long long)(g[((size_t)x * D + y) * H + z] == wc) << y;
        occ64[R.occy_off + c] = bits;
    }
    __syncthreads();
    // exclusive scan of the per-column free counts in (x, y) order: possible_start_pose order (:450-457)
    if (tid == 0) {
        uint32_t run = 0;
        for (int c = 0; c < W * D; c++) { uint32_t v = cnt[c]; cnt[c] = run; run += v; }
        cnt[W * D] = run;
        rooms[r].n_free = run;
        n_wall[r] = walls;
    }
    __syncthreads();
    for (int c = tid; c < W * D; c += nt) {
        const int x = c / D, y = c - x * D;
        const bool interior = x >= 1 && x <= W - 2 && y >= 1 && y <= D - 2;
        if (!interior) continue;
        uint32_t freebits = ~(uint32_t)occz[R.occz_off + c] & zin;
        uint32_t o = R.free_off + cnt[c];
        while (freebits) {
            const int z = __ffs(freebits) - 1;
            freebits &= freebits - 1;
            free_cells[o++] = (uint32_t)x | ((uint32_t)y << 8) | ((uint32_t)z << 16);
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// per-env kernels: G lanes per env, kBlock / G envs per CTA
// ---------------------------------------------------------------------------------------------------------------
template <int G>
__global__ void __launch_bounds__(kBlock) reset_kernel(EngineParams P, const int32_t *__restrict__ env_ids, int n,
                                                       const int32_t *__restrict__ picks, float *obs) {
    __shared__ float lut[kLutSize];
    fill_lut(lut, P.L);
    const long long gid = (long long)blockIdx.x * kBlock + threadIdx.x;
    const long long idx = gid / G;
    const int lane = (int)(gid % G), liw = threadIdx.x & 31;
    if (idx >= n) return;
    const int env = env_ids ? env_ids[idx] : (int)idx;
    if (env < 0 || env >= P.n_envs) return;
    float *orow = obs ? obs + (long long)env * kObsDim : nullptr;
    const uint32_t episode = P.states[env].episode;
    group_sync<G>(liw);   // every lane has read the episode counter before lane 0 rewrites the state
    if (picks) {
        uint32_t room = (uint32_t)picks[2 * idx];
        room = room < (uint32_t)P.n_rooms ? room : (uint32_t)P.n_rooms - 1u;
        uint32_t nf = P.rooms[room].n_free, k = (uint32_t)picks[2 * idx + 1];
        k = k < nf ? k : nf - 1u;
        reset_env<G>(P, env, lane, liw, room, k, episode + 1u, lut, orow);
    } else {
        reset_env_philox<G>(P, env, lane, liw, episode, lut, orow);
    }
}

// Out-of-line reset for the single-launch step kernel: called at the very end of a step, when almost nothing is live, so
// the kernel's register count stays that of the step itself.
template <int G>
__device__ __noinline__ void reset_out_of_line(const EngineParams &P, int env, int lane, int liw, uint32_t episode,
                                               const float *lut, float *obs_row) {
    reset_env_philox<G>(P, env, lane, liw, episode, lut, obs_row);
}

template <int G, int MINB>
__global__ void __launch_bounds__(kBlock, MINB) step_call_kernel(const __grid_constant__ EngineParams P, StepIO io) {
    __shared__ float lut[kLutSize];
    // Programmatic dependent launch: when launched with the stream-serialisation attribute this grid may become resident
    // while the previous kernel of the stream is still draining; everything up to the wait (table fill, index math) overlaps
    // that tail, and the next kernel is allowed to do the same with ours.  Without the attribute both are no-ops.
    asm volatile("griddepcontrol.launch_dependents;");
    fill_lut(lut, P.L);
    asm volatile("griddepcontrol.wait;" ::: "memory");
    const long long gid = (long long)blockIdx.x * kBlock + threadIdx.x;
    if (gid / G >= io.env_n) return;
    const long long env = io.env0 + gid / G;
    const int lane = (int)(gid % G), liw = threadIdx.x & 31;
    const int action = (int)io.actions[env];
    if (step_env<G>(P, io, (int)env, lane, liw, action, lut, env)) {
        const uint32_t episode = P.states[env].episode;       // untouched by a step that ends its episode
        group_sync<G>(liw);                                    // all lanes are done reading the old knowledge
        reset_out_of_line<G>(P, (int)env, lane, liw, episode, lut, io.obs + env * kObsDim);
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Thread-per-env kernels (CubicEnv, lanes_per_env = 1): nothing of a step is computed twice, every load of a step is issued
// by the one thread that needs it, and the only cooperation is in data movement — the warp writes the 32 observation rows
// it assembled in shared memory with coalesced 128-bit stores, and clears the knowledge of the envs it resets together.
// ---------------------------------------------------------------------------------------------------------------
// The warp's 32 staged (compact) rows -> their global rows (dst[e] == NULL: env e has none): get_obs Steps 2-6
// (CubicEnv.py:270-307) — clip to [-2, 20] and (m + 2) / 22 through the code table, facing one-hot, the scalar quotients,
// zero padding.  Two passes so that every store instruction runs ONE code path: the 16 window float4 of two envs per
// instruction (lane l: column l % 16 of env 2i + l / 16: 2 x 256 contiguous bytes), then the 4 scalar float4 of eight envs
// per instruction (lane l: quad 16 + l % 4 of env 8i + l / 4: 8 x 64 contiguous bytes).
// CONTIG: the 32 rows are consecutive rows of one array starting at d0 (the usual case: no env of the warp finished, none is
// past the range) — no destination look-up, no test per store.
template <bool CONTIG>
__device__ __forceinline__ void flush_rows_t(const uint32_t *stage, float *const *dst, float *d0, int lane, const float *lut, int L) {
    const int j = lane & 15, eh = lane >> 4;
#pragma unroll 4
    for (int i = 0; i < 16; i++) {
        const int e = 2 * i + eh;
        float *d = CONTIG ? d0 + e * kObsDim : dst[e];
        if (!CONTIG && d == nullptr) continue;                     // (a row that was not staged holds stale words)
        const uint32_t q = stage[e * kStageStride + j];
        float4 v;
        v.x = lut[q & 31u]; v.y = lut[(q >> 5) & 31u]; v.z = lut[(q >> 10) & 31u]; v.w = lut[q >> 15];
        __stcs(reinterpret_cast<float4 *>(d) + j, v);
    }
    const int k = lane & 3, e4 = lane >> 2;
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const int e = 8 * i + e4;
        float *d = CONTIG ? d0 + e * kObsDim : dst[e];
        if (!CONTIG && d == nullptr) continue;
        const uint32_t sc = stage[e * kStageStride + kStageScalars], down = sc >> 8;
        const float ex = __uint_as_float(stage[e * kStageStride + kStageExplored]);
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (k == 0) {                                              // facing one-hot (:279-280)
            const uint32_t f = sc & 3u;
            v.x = f == 0 ? 1.f : 0.f; v.y = f == 1 ? 1.f : 0.f; v.z = f == 2 ? 1.f : 0.f; v.w = f == 3 ? 1.f : 0.f;
        } else if (k == 1) {                                       // last_action / 5, was_near_wall, last_bump, down / L (:284-287)
            v.x = lut[kLutFifth + ((sc >> 2) & 7u)];
            v.y = (float)((sc >> 5) & 1u);
            v.z = (float)((sc >> 6) & 1u);
            v.w = L <= 31 ? lut[kLutDown + down] : __fdiv_rn((float)down, (float)L);
        } else if (k == 2) v.x = ex;                               // visited / total (:291); quad 19 is padding
        __stcs(reinterpret_cast<float4 *>(d) + 16 + k, v);
    }
}
__device__ __forceinline__ void flush_rows(const float *stage_f, float *const *dst, int lane, const float *lut, int L) {
    const uint32_t *stage = reinterpret_cast<const uint32_t *>(stage_f);
    __syncwarp();
    float *d0 = dst[0];
    const bool contig = __all_sync(0xffffffffu, d0 != nullptr && dst[lane] == d0 + lane * kObsDim);
    if (contig) flush_rows_t<true>(stage, dst, d0, lane, lut, L);
    else flush_rows_t<false>(stage, dst, d0, lane, lut, L);
    __syncwarp();
}

// Per-warp shared-memory workspace of the thread-per-env kernels: the staged rows with their destinations, and the warp's
// list of marking tiles with the env each lane plays.
struct WarpWork {
    float stage[32 * kStageStride];
    float *dst[32];
    uint32_t *tasks;               // this warp's slice of the CTA's dynamic shared memory (P.mark_cap entries)
    uint32_t env_of_lane[32];
    uint32_t desc[64];             // MarkQueue::desc
    int n_tasks;
};
// dynamic shared memory of a thread-per-env CTA: one marking list per warp
__device__ __forceinline__ uint32_t *warp_tasks(const EngineParams &P) {
    extern __shared__ uint32_t dyn_tasks[];
    return dyn_tasks + (threadIdx.x >> 5) * P.mark_cap;
}

// Step 1 of get_obs (CubicEnv.py:264-266) for the x / y rays of every env of the warp that is on a first visit: the lanes
// share the queued tiles evenly.  A task is up to four words of one tile (x run: words tile + 4j, y run: tile + j, a wall
// end: one word); a word whose field at the agent's height is still 0 (unknown) becomes "seen" (2) or "known wall" (1).
// `between` (the row flush) runs while the first round's loads are in flight.
template <typename F>
__device__ __forceinline__ void coop_marks(const EngineParams &P, WarpWork *w, int lane, F &&between) {
    __syncwarp();                                                // every lane has queued its tiles
    const int total = w->n_tasks;
    constexpr int CH = 4;                                        // tasks per lane per round: all loads before the first use
    bool first = true;
    for (int i0 = 0; i0 < total || first; i0 += 32 * CH) {
        uint32_t v[CH][4], meta[CH];
        uint32_t *Kp[CH];
#pragma unroll
        for (int c = 0; c < CH; c++) {
            const int i = i0 + c * 32 + lane;
            const uint32_t t = i < total ? w->tasks[i] : 0u;      // (no task: empty mask below, z field 0)
            const uint32_t tl = (t >> 16) & 31u, yrun = (t >> 29) & 1u;
            meta[c] = t;
            Kp[c] = reinterpret_cast<uint32_t *>(P.know + (unsigned long long)w->env_of_lane[tl] * P.env_stride) + (t & 0xffffu);
            // the tile's cells 4T - pad + j that lie in the run's free range and are not its centre
            const uint32_t d = w->desc[yrun * 32u + tl];
            const int c0 = 4 * (int)((t >> 21) & 31u) - kPadLo;
            const int lo_ = min(max((int)(d & 255u) - c0, 0), 4), up = min(max(c0 + 3 - (int)((d >> 8) & 255u), 0), 4);
            uint32_t m = (0xfu << lo_) & (0xfu >> up) & 0xfu;
            const int sk = (int)((d >> 16) & 255u) - c0;
            if (sk >= 0 && sk <= 3) m &= ~(1u << sk);
            if (t & (1u << 30)) m = 1u;                            // a wall end: the one word the task names
            if (i >= total) m = 0u;
            const uint32_t stride = yrun ? 1u : 4u;
#pragma unroll
            for (int j = 0; j < 4; j++) v[c][j] = ((m >> j) & 1u) ? Kp[c][j * stride] : 0xffffffffu;
        }
        if (first) { between(); first = false; }
#pragma unroll
        for (int c = 0; c < CH; c++) {
            const uint32_t t = meta[c], zsh = 5u * ((t >> 26) & 7u), stride = (t & (1u << 29)) ? 1u : 4u;
            const uint32_t code = ((t & (1u << 30)) ? kCodeWall : kCodeSeen) << zsh;
#pragma unroll
            for (int j = 0; j < 4; j++)
                if (((v[c][j] >> zsh) & 31u) == 0u) Kp[c][j * stride] = v[c][j] | code;
        }
    }
    __syncwarp();                                                // the marks are visible to the warp's next loads
    if (lane == 0) w->n_tasks = 0;
    __syncwarp();
}

// Auto-reset of the warp's envs whose lanes say `mine` (CubicEnv.py:77-108 with Philox picks).  Out of line so that the
// step keeps its registers.  The new record goes to P.states.
template <bool STAGED>
__device__ __noinline__ void tpe_reset(const EngineParams &P, bool mine, uint32_t env, uint32_t episode, bool have_picks,
                                       uint32_t room, uint32_t k, const float *lut, float *obs, WarpWork *w, int lane) {
    const unsigned rmask = __ballot_sync(0xffffffffu, mine);
    if (mine && !have_picks) reset_picks(P, (int)env, episode, room, k);
    // internal_grid = full(-1) (:84): the whole warp sweeps each env's bricks
    for (unsigned m = rmask; m; m &= m - 1u) {
        const int src = __ffs((int)m) - 1;
        const uint32_t e = __shfl_sync(0xffffffffu, env, src), r = __shfl_sync(0xffffffffu, room, src);
        const uint32_t n = k_bytes(P.rooms[r]) >> 4;
        uint4 *k4 = reinterpret_cast<uint4 *>(P.know + (unsigned long long)e * P.env_stride);
        const uint4 zero = make_uint4(0u, 0u, 0u, 0u);
        for (uint32_t i = (uint32_t)lane; i < n; i += 32u) k4[i] = zero;
    }
    __syncwarp();
    if (STAGED) w->dst[lane] = nullptr;
    if (mine) {
        ResetCtx c;
        float *row = obs ? obs + (unsigned long long)env * kObsDim : nullptr;
        MarkQueue mq{w->tasks, &w->n_tasks, w->desc, lane};
        if (STAGED) { w->dst[lane] = row; if (row) row = w->stage + lane * kStageStride; }
        const uint32_t nbr = reset_lane<1, STAGED>(P, (int)env, 0, room, k, episode + 1u, lut, row, c, STAGED ? &mq : nullptr);
        reset_commit(P, (int)env, 0, c, nbr);
    }
    if (STAGED) coop_marks(P, w, lane, [&]() { flush_rows(w->stage, w->dst, lane, lut, P.L); });
}

template <int BLOCK, bool STAGED>
__device__ __forceinline__ void step_tpe_body(const EngineParams &P, const StepIO &io) {
    __shared__ float lut[kLutSize];
    __shared__ WarpWork work[STAGED ? BLOCK / 32 : 1];
    asm volatile("griddepcontrol.launch_dependents;");          // programmatic dependent launch, as in step_call_kernel
    fill_lut(lut, P.L);
    asm volatile("griddepcontrol.wait;" ::: "memory");
    const int lane = threadIdx.x & 31;
    WarpWork *w = work + (STAGED ? threadIdx.x >> 5 : 0);
    const long long gid = (long long)blockIdx.x * BLOCK + threadIdx.x;
    if (gid - lane >= io.env_n) return;                          // the whole warp is past the range
    const bool valid = gid < io.env_n;
    const long long env = io.env0 + gid;
    if (STAGED) {
        w->dst[lane] = nullptr; w->env_of_lane[lane] = (uint32_t)env;
        if (lane == 0) { w->n_tasks = 0; w->tasks = warp_tasks(P); }
        __syncwarp();
    }
    bool rst = false;
    if (valid) {
        MarkQueue mq{w->tasks, &w->n_tasks, w->desc, lane};
        rst = step_env<1, false, STAGED>(P, io, (int)env, 0, lane, (int)io.actions[env], lut, env, nullptr, nullptr,
                                         w->stage + lane * kStageStride, w->dst + lane, STAGED ? &mq : nullptr);
    }
    if (STAGED) coop_marks(P, w, lane, [&]() { flush_rows(w->stage, w->dst, lane, lut, P.L); });
    if (__any_sync(0xffffffffu, rst)) {
        const uint32_t episode = rst ? P.states[env].episode : 0u;   // untouched by a step that ends its episode
        tpe_reset<STAGED>(P, rst, (uint32_t)env, episode, false, 0u, 0u, lut, io.obs, w, lane);
    }
}
template <int BLOCK, int MINB, bool STAGED>
__global__ void __launch_bounds__(BLOCK, MINB) step_tpe_kernel(const __grid_constant__ EngineParams P, StepIO io) {
    step_tpe_body<BLOCK, STAGED>(P, io);
}
__global__ void __launch_bounds__(kBlock) reset_tpe_kernel(const __grid_constant__ EngineParams P,
                                                           const int32_t *__restrict__ env_ids, int n,
                                                           const int32_t *__restrict__ picks, float *obs) {
    __shared__ float lut[kLutSize];
    __shared__ WarpWork work[kBlock / 32];
    fill_lut(lut, P.L);
    const int lane = threadIdx.x & 31;
    WarpWork *w = work + (threadIdx.x >> 5);
    const long long idx = (long long)blockIdx.x * kBlock + threadIdx.x;
    if (idx - lane >= n) return;
    int env = idx < n ? (env_ids ? env_ids[idx] : (int)idx) : -1;
    const bool mine = env >= 0 && env < P.n_envs;
    uint32_t episode = 0, room = 0, k = 0;
    if (mine) {
        episode = P.states[env].episode;
        if (picks) {
            room = (uint32_t)picks[2 * idx];
            room = room < (uint32_t)P.n_rooms ? room : (uint32_t)P.n_rooms - 1u;
            const uint32_t nf = P.rooms[room].n_free;
            k = (uint32_t)picks[2 * idx + 1];
            k = k < nf ? k : nf - 1u;
        }
    }
    w->env_of_lane[lane] = mine ? (uint32_t)env : 0u;
    if (lane == 0) { w->n_tasks = 0; w->tasks = warp_tasks(P); }
    __syncwarp();
    tpe_reset<true>(P, mine, (uint32_t)env, episode, picks != nullptr, room, k, lut, obs, w, lane);
}

// T fused steps per env, thread per env.  The record stays in the thread's registers for the whole rollout and the
// knowledge lines it touches stay in L2, so DRAM sees the outputs the caller asked for plus one pass over the touched lines.
// CALLER_ACTIONS: the actions are the caller's u8 [T][N] rows (nav3d_rollout_actions) and every output of nav3d_step may
// be written; otherwise they come from the env's Philox action stream (BASELINE.md §4 config 4: nav3d_rollout_random,
// which also fills `done` and `actions_out`).  The Philox branches keep their own StepIO set-up: written through
// rollout_step_io, nav3d_rollout_random compiled to different (if equivalent) SASS.
template <int BLOCK, bool STAGED, bool CALLER_ACTIONS>
__device__ __forceinline__ void rollout_tpe_body(const EngineParams &P, int T, uint32_t t0, float *obs, float *obs_last,
                                                 float *reward, uint8_t *done, uint8_t *actions_out, const RolloutIO *ro) {
    __shared__ float lut[kLutSize];
    __shared__ WarpWork work[STAGED ? BLOCK / 32 : 1];
    fill_lut(lut, P.L);
    const int lane = threadIdx.x & 31;
    WarpWork *w = work + (STAGED ? threadIdx.x >> 5 : 0);
    const long long gid = (long long)blockIdx.x * BLOCK + threadIdx.x;
    const long long N = P.n_envs;
    if (gid - lane >= N) return;
    const bool valid = gid < N;
    const long long env = gid;
    if (STAGED) {
        w->env_of_lane[lane] = (uint32_t)env;
        if (lane == 0) { w->n_tasks = 0; w->tasks = warp_tasks(P); }
        __syncwarp();
    }
    const MarkQueue mq{w->tasks, &w->n_tasks, w->desc, lane};
    EnvState st;
    if (valid) st = P.states[env];
    for (int t = 0; t < T; t++) {
        StepIO io;
        if constexpr (CALLER_ACTIONS) {
            io = rollout_step_io(*ro, t, T, N);
        } else {
            io.actions = nullptr;
            // obs == NULL: only the last step's observation is written out
            io.obs = obs ? obs + (long long)t * N * kObsDim : (t == T - 1 ? obs_last : nullptr);
            io.reward = reward ? reward + (long long)t * N : nullptr;
            io.reward64 = nullptr; io.terminated = nullptr; io.truncated = nullptr;
            io.terminal_obs = nullptr; io.episodes = nullptr;
            io.env0 = 0; io.env_n = P.n_envs;
        }
        if (STAGED) w->dst[lane] = nullptr;
        bool rst = false;
        if (valid) {
            uint32_t u0, u1, bits = 0;
            int action;
            if constexpr (CALLER_ACTIONS) {
                action = rollout_action(*ro, t, N, env);
            } else {
                philox4x32_10(P.env_id0 + (uint32_t)env, t0 + (uint32_t)t, 0u, kStreamAction, P.seed_lo, P.seed_hi, u0, u1);
                action = (int)mulhi_range(u0, 6u);
            }
            rst = step_env<1, true, STAGED>(P, io, (int)env, 0, lane, action, lut, env, &st, &bits,
                                            w->stage + lane * kStageStride, w->dst + lane, STAGED ? &mq : nullptr);
            if constexpr (!CALLER_ACTIONS) {
                if (done) done[(long long)t * N + env] = bits ? 1 : 0;
                if (actions_out) actions_out[(long long)t * N + env] = (uint8_t)action;
            }
        }
        if (STAGED) coop_marks(P, w, lane, [&]() { flush_rows(w->stage, w->dst, lane, lut, P.L); });
        if (__any_sync(0xffffffffu, rst)) {
            tpe_reset<STAGED>(P, rst, (uint32_t)env, st.episode, false, 0u, 0u, lut, io.obs, w, lane);
            if (rst) st = P.states[env];           // the new episode's record (written by this very thread)
        }
    }
    if (valid) P.states[env] = st;
}
template <int BLOCK, int MINB, bool STAGED>
__global__ void __launch_bounds__(BLOCK, MINB) rollout_tpe_kernel(const __grid_constant__ EngineParams P, int T, uint32_t t0,
                                                                  float *obs, float *obs_last, float *reward, uint8_t *done,
                                                                  uint8_t *actions_out) {
    rollout_tpe_body<BLOCK, STAGED, false>(P, T, t0, obs, obs_last, reward, done, actions_out, nullptr);
}
template <int BLOCK, int MINB>
__global__ void __launch_bounds__(BLOCK, MINB) rollout_actions_tpe_kernel(const __grid_constant__ EngineParams P, int T,
                                                                          const __grid_constant__ RolloutIO ro) {
    rollout_tpe_body<BLOCK, true, true>(P, T, 0u, nullptr, nullptr, nullptr, nullptr, nullptr, &ro);
}
// T fused steps per env, G lanes per env, actions as in rollout_tpe_body (SURVEY §8f row 3).  An env's record and the
// knowledge lines it touches stay in L1/L2 for the whole rollout, so DRAM sees the outputs the caller asked for plus one
// pass over the touched lines.  When only the last observation is requested the intermediate observations are never
// formed.  The reset is an out-of-line call (as in step_call_kernel) so that the loop body keeps the step's 64 registers.
template <int G, bool CALLER_ACTIONS>
__device__ __forceinline__ void rollout_group_body(const EngineParams &P, int T, uint32_t t0, float *obs, float *obs_last,
                                                   float *reward, uint8_t *done, uint8_t *actions_out,
                                                   float *reward_scratch, const RolloutIO *ro) {
    __shared__ float lut[kLutSize];
    fill_lut(lut, P.L);
    const long long gid = (long long)blockIdx.x * kBlock + threadIdx.x;
    const long long env = gid / G;
    if (env >= P.n_envs) return;
    const int lane = (int)(gid % G), liw = threadIdx.x & 31;
    const long long N = P.n_envs;
    EnvState st = P.states[env];          // the record stays in registers for the whole rollout (every lane holds a copy)
    for (int t = 0; t < T; t++) {
        uint32_t u0, u1;
        int action;
        if constexpr (CALLER_ACTIONS) {
            action = rollout_action(*ro, t, N, env);
        } else {
            philox4x32_10(P.env_id0 + (uint32_t)env, t0 + (uint32_t)t, 0u, kStreamAction, P.seed_lo, P.seed_hi, u0, u1);
            action = (int)mulhi_range(u0, 6u);
        }
        StepIO io;
        if constexpr (CALLER_ACTIONS) {
            io = rollout_step_io(*ro, t, T, N);
        } else {
            io.actions = nullptr;
            // obs == NULL: only the last step's observation is kept; the earlier steps form none (and skip the window gather)
            io.obs = obs ? obs + (long long)t * N * kObsDim : (t == T - 1 ? obs_last : nullptr);
            io.reward = reward ? reward + (long long)t * N : reward_scratch;
            io.reward64 = nullptr;
            io.terminated = nullptr; io.truncated = nullptr;
            io.terminal_obs = nullptr; io.episodes = nullptr;
            io.env0 = 0; io.env_n = P.n_envs;
        }
        uint32_t bits = 0;
        if (step_env<G, true>(P, io, (int)env, lane, liw, action, lut, env, &st, &bits)) {
            group_sync<G>(liw);            // all lanes are done reading the old knowledge
            reset_out_of_line<G>(P, (int)env, lane, liw, st.episode, lut, io.obs ? io.obs + env * kObsDim : nullptr);
            group_sync<G>(liw);            // lane 0's record of the new episode is visible
            st = P.states[env];
        }
        if constexpr (!CALLER_ACTIONS) {
            if (lane == 0) {
                if (done) done[(long long)t * N + env] = bits ? 1 : 0;
                if (actions_out) actions_out[(long long)t * N + env] = (uint8_t)action;
            }
        }
        group_sync<G>(liw);   // lane 0's counter store and every lane's S stores are visible to the next step
    }
    if (lane == 0) P.states[env] = st;
}
template <int G, int MINB>
__global__ void __launch_bounds__(kBlock, MINB) rollout_kernel(const __grid_constant__ EngineParams P, int T, uint32_t t0,
                                                            float *obs, float *obs_last, float *reward, uint8_t *done,
                                                            uint8_t *actions_out, float *reward_scratch,
                                                            uint8_t *term_scratch, uint8_t *trunc_scratch) {
    rollout_group_body<G, false>(P, T, t0, obs, obs_last, reward, done, actions_out, reward_scratch, nullptr);
}
template <int G, int MINB>
__global__ void __launch_bounds__(kBlock, MINB) rollout_actions_kernel(const __grid_constant__ EngineParams P, int T,
                                                                    const __grid_constant__ RolloutIO ro) {
    rollout_group_body<G, true>(P, T, 0u, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, &ro);
}

template <int G>
__global__ void __launch_bounds__(kBlock) simple_reset_kernel(EngineParams P, const int32_t *__restrict__ env_ids, int n,
                                                              const int32_t *__restrict__ picks, float *obs) {
    const long long gid = (long long)blockIdx.x * kBlock + threadIdx.x;
    const long long idx = gid / G;
    const int lane = (int)(gid % G), liw = threadIdx.x & 31;
    if (idx >= n) return;
    const int env = env_ids ? env_ids[idx] : (int)idx;
    if (env < 0 || env >= P.n_envs) return;
    float *orow = obs ? obs + (long long)env * P.obs_dim : nullptr;
    const uint32_t episode = P.states[env].episode;
    group_sync<G>(liw);
    if (picks) {
        uint32_t room = (uint32_t)picks[3 * idx];
        room = room < (uint32_t)P.n_rooms ? room : (uint32_t)P.n_rooms - 1u;
        const uint32_t nf = P.rooms[room].n_free;
        uint32_t k = (uint32_t)picks[3 * idx + 1], kg = (uint32_t)picks[3 * idx + 2];
        k = k < nf ? k : nf - 1u; kg = kg < nf ? kg : nf - 1u;
        simple_reset_env<G>(P, env, lane, liw, room, k, kg, episode + 1u, orow);
    } else {
        simple_reset_env_philox<G>(P, env, lane, liw, episode, orow);
    }
}

// simpleEnv, one thread per env: the 6L+7 floats of a row (124 B at L = 4: never 16-byte aligned, so a lane writing its own
// row needs one 4-byte store per float) are assembled in shared memory and the warp writes its 32 rows — contiguous in the
// caller's [N, 6L+7] array — with coalesced 128-byte store instructions.  Dynamic shared memory: kBlock x stride floats.
__device__ __forceinline__ void flush_rows_n(const float *stage, int stride, float *const *dst, int obs_dim, int lane) {
    __syncwarp();
    float *d0 = dst[0];
    if (stride == obs_dim && __all_sync(0xffffffffu, d0 != nullptr && dst[lane] == d0 + lane * obs_dim)) {
        // the usual case: 32 consecutive rows of one array, staged back to back (6L+7 is odd: conflict-free as it is) —
        // one linear copy of 32 x (6L+7) floats, 128 bytes per store instruction
        const int n = 32 * obs_dim;
#pragma unroll 4
        for (int i = lane; i < n; i += 32) __stcs(d0 + i, stage[i]);
    } else {
        int e = 0, j = lane;
        while (j >= obs_dim) { j -= obs_dim; e++; }
        while (e < 32) {
            float *d = dst[e];
            if (d != nullptr) __stcs(d + j, stage[e * stride + j]);
            j += 32;
            while (j >= obs_dim) { j -= obs_dim; e++; }
        }
    }
    __syncwarp();
}

__global__ void __launch_bounds__(kBlock, 6) simple_step_tpe_kernel(const __grid_constant__ EngineParams P, StepIO io, int stride) {
    extern __shared__ float stage_dyn[];
    __shared__ float *dst_all[kBlock];
    asm volatile("griddepcontrol.launch_dependents;");
    const int lane = threadIdx.x & 31, wbase = threadIdx.x & ~31;
    float *stage = stage_dyn + wbase * stride;
    float **dst = dst_all + wbase;
    const long long gid = (long long)blockIdx.x * kBlock + threadIdx.x;
    asm volatile("griddepcontrol.wait;" ::: "memory");
    if (gid - lane >= io.env_n) return;
    const bool valid = gid < io.env_n;
    const long long env = io.env0 + gid;
    dst[lane] = nullptr;
    bool rst = false;
    if (valid)
        rst = simple_step_env<1, true>(P, io, (int)env, 0, lane, (int)io.actions[env], env, stage + lane * stride, dst + lane);
    flush_rows_n(stage, stride, dst, P.obs_dim, lane);
    if (__any_sync(0xffffffffu, rst)) {
        dst[lane] = nullptr;
        if (rst) {
            dst[lane] = io.obs + env * P.obs_dim;
            simple_reset_env_philox<1>(P, (int)env, 0, lane, P.states[env].episode, stage + lane * stride);
        }
        flush_rows_n(stage, stride, dst, P.obs_dim, lane);
    }
}

template <int G, int MINB>
__global__ void __launch_bounds__(kBlock, MINB) simple_step_kernel(EngineParams P, StepIO io) {
    asm volatile("griddepcontrol.launch_dependents;");
    const long long gid = (long long)blockIdx.x * kBlock + threadIdx.x;
    asm volatile("griddepcontrol.wait;" ::: "memory");      // programmatic dependent launch, as in step_call_kernel
    if (gid / G >= io.env_n) return;
    const long long env = io.env0 + gid / G;
    const int lane = (int)(gid % G), liw = threadIdx.x & 31;
    simple_step_env<G>(P, io, (int)env, lane, liw, (int)io.actions[env], env);
}

__global__ void simple_get_grid_kernel(EngineParams P, int env, int16_t *out) {
    const EnvState s = P.states[env];
    const RoomDev R = P.rooms[s.room];
    const int n = R.W * R.D * R.H;
    const uint32_t *K = reinterpret_cast<const uint32_t *>(P.know + (unsigned long long)env * P.env_stride);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int z = i % R.H, y = (i / R.H) % R.D, x = i / (R.H * R.D);
        out[i] = (int16_t)(k2_code(K[s_index(R, x, y)], z) - 1);
    }
}

__global__ void get_state_kernel(EngineParams P, int32_t *out) {
    const int env = blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= P.n_envs) return;
    const EnvState s = P.states[env];
    int32_t *o = out + (long long)env * NAV3D_STATE_INTS;
    o[0] = s.x; o[1] = s.y; o[2] = s.z; o[3] = s.facing;
    o[4] = (int32_t)s.visited_count; o[5] = (int32_t)s.bump_count; o[6] = (int32_t)s.step_count;
    o[7] = (s.flags & kNearWall) != 0; o[8] = (s.flags & kWasNearWall) != 0; o[9] = (s.flags & kLastBump) != 0;
    o[10] = (s.flags & kDone) != 0; o[11] = s.down; o[12] = s.last_action; o[13] = s.room;
    o[14] = (int32_t)s.episode; o[15] = s.ret_centi;
    if (P.obs_dim != kObsDim) { o[7] = s.down; o[8] = s.blocked6; o[9] = s.own_count; o[11] = 0; }   // simpleEnv: the goal cell
}

__global__ void get_grid_kernel(EngineParams P, int env, int16_t *out) {
    const EnvState s = P.states[env];
    const RoomDev R = P.rooms[s.room];
    const int n = R.W * R.D * R.H;
    const uint8_t *envk = P.know + (unsigned long long)env * P.env_stride;
    const uint32_t *K = reinterpret_cast<const uint32_t *>(envk);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int z = i % R.H, y = (i / R.H) % R.D, x = i / (R.H * R.D);
        const int zb = z / 6;
        const uint32_t code = (K[k_index(R, x, y, zb)] >> (5 * (z - 6 * zb))) & 31u;
        int16_t v = (int16_t)((int)code - 2);
        if (code == kCodeUnknown) v = -1;
        else if (code == kCodeWall) v = -2;
        else if (code == kCodeOverflow) v = (int16_t)(kOverflowBase + envk[P.ovf_off + ovf_index(R, x, y, z)]);
        out[i] = v;
    }
}

// Records of envs that were never reset: every move bumps, so stepping such an env by mistake stays inside its block.
__global__ void init_states_kernel(EnvState *states, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    EnvState s{};
    s.blocked6 = 0x3f;
    states[i] = s;
}

// Env-state blobs, a warp per listed env (nav3d_core.cuh save_env_lane / load_env_lane).  A pure copy of the live part of
// the env's block: HBM-bound.  Blob stores (save) and blob loads (load) carry the evict-first hint, so that a large save or
// load does not push the knowledge lines of a running rollout out of L2.
__global__ void __launch_bounds__(kBlock) save_envs_kernel(const __grid_constant__ EngineParams P, unsigned long long sig,
                                                           const int32_t *__restrict__ env_ids, int n,
                                                           const float *__restrict__ obs, uint8_t *blobs,
                                                           unsigned long long blob_bytes) {
    const long long i = ((long long)blockIdx.x * kBlock + threadIdx.x) >> 5;
    if (i >= n) return;
    const int env = env_ids ? env_ids[i] : (int)i;
    save_env_lane(P, sig, env, obs, blobs + (unsigned long long)i * blob_bytes, threadIdx.x & 31, 32);
}
__global__ void __launch_bounds__(kBlock) load_envs_kernel(const __grid_constant__ EngineParams P, unsigned long long sig,
                                                           const int32_t *__restrict__ env_ids, int n,
                                                           const uint8_t *blobs, unsigned long long blob_bytes, float *obs,
                                                           uint8_t *status) {
    const long long i = ((long long)blockIdx.x * kBlock + threadIdx.x) >> 5;
    if (i >= n) return;
    const int lane = threadIdx.x & 31;
    const int env = env_ids ? env_ids[i] : (int)i;
    const uint8_t *blob = blobs + (unsigned long long)i * blob_bytes;
    const uint8_t st = blob_status(P, sig, env, blob);      // the whole header is checked before anything is written
    if (status && lane == 0) status[i] = st;
    if (st == kBlobLoaded) load_env_lane(P, env, blob, obs, lane, 32);
}

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

}  // namespace

// ---------------------------------------------------------------------------------------------------------------
// engine
// ---------------------------------------------------------------------------------------------------------------
struct nav3d_engine {
    nav3d_config cfg{};
    int G = 8;
    EngineParams P{};
    std::vector<RoomDev> h_rooms;
    std::vector<uint32_t> h_free;
    std::vector<uint32_t> h_nwall;
    RoomDev *d_rooms = nullptr;
    uint16_t *d_occz = nullptr;
    unsigned long long *d_occ64 = nullptr;
    uint32_t *d_free = nullptr, *d_start = nullptr;
    EnvState *d_states = nullptr;
    uint8_t *d_know = nullptr;
    size_t know_bytes = 0, room_bytes = 0;
    // scratch for rollout / host path
    float *d_reward = nullptr, *d_obs = nullptr;
    uint8_t *d_term = nullptr, *d_trunc = nullptr;
    long long *d_actions = nullptr;
    int minb = 0;               // __launch_bounds__ min CTAs/SM variant of the step kernel (tuning knob)
    bool simple = false;        // NAV3D_ENV_SIMPLE
    int simple_stride = 0;      // simpleEnv, lanes_per_env == 1: floats per staged row (odd: conflict-free), 0 = not staged
    bool tpe_staged = true;     // thread-per-env kernels: rows staged in shared memory, marking by the warp (NAV3D_TPE_STAGED)
    int tpe_block = 64;         // their CTA size (NAV3D_TPE_BLOCK)
    bool reset_seen = false;    // a nav3d_reset (or nav3d_restore / nav3d_load_envs) call has been made since the rooms were loaded
    unsigned long long signature = 0;   // engine signature of env-state blobs (nav3d_core.cuh sig_engine / sig_room)
    bool pdl = true;            // programmatic dependent launch of the step kernel (NAV3D_PDL=0 switches it off)
    float *d_dist_lut = nullptr;
    cudaStream_t own_stream = nullptr;
    static constexpr int kHostChunks = 4;          // nav3d_step_host pipeline depth
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t chunk_done[kHostChunks] = {};
    uint64_t launches = 0;
};

namespace {

// Makes the engine's device current for the duration of one ABI call and puts the caller's device back afterwards: the
// caller (torch) tracks the current device itself and must not find it changed behind its back.
struct DeviceGuard {
    int prev = -1, want = -1;
    cudaError_t err = cudaSuccess;
    explicit DeviceGuard(int device) : want(device) {
        err = cudaGetDevice(&prev);
        if (err == cudaSuccess && prev != want) err = cudaSetDevice(want);
    }
    ~DeviceGuard() { if (prev >= 0 && prev != want) cudaSetDevice(prev); }
};
#define NAV3D_DEVICE(e)                                                                                            \
    DeviceGuard _dev_guard((e)->cfg.device);                                                                       \
    if (_dev_guard.err != cudaSuccess)                                                                             \
    return fail(NAV3D_ERR_CUDA, std::string("cudaSetDevice: ") + cudaGetErrorString(_dev_guard.err))

void free_rooms(nav3d_engine *e) {
    cudaFree(e->d_rooms); cudaFree(e->d_occz); cudaFree(e->d_occ64); cudaFree(e->d_free); cudaFree(e->d_know);
    cudaFree(e->d_start); e->d_start = nullptr;
    e->d_rooms = nullptr; e->d_occz = nullptr; e->d_occ64 = nullptr; e->d_free = nullptr; e->d_know = nullptr;
    e->know_bytes = 0; e->room_bytes = 0;
    e->h_rooms.clear(); e->h_free.clear(); e->h_nwall.clear();
}

template <typename F> int dispatch_lanes(int G, F &&f) {
    switch (G) {
        case 1: return f(std::integral_constant<int, 1>());
        case 2: return f(std::integral_constant<int, 2>());
        case 4: return f(std::integral_constant<int, 4>());
        case 8: return f(std::integral_constant<int, 8>());
        case 16: return f(std::integral_constant<int, 16>());
        case 32: return f(std::integral_constant<int, 32>());
    }
    return fail(NAV3D_ERR_INVALID, "lanes_per_env must be 1, 2, 4, 8, 16 or 32");
}

unsigned grid_for(long long n_groups, int G) {
    const long long threads = n_groups * G;
    return (unsigned)((threads + kBlock - 1) / kBlock);
}

int check_ready(const nav3d_engine *e) {
    if (!e) return fail(NAV3D_ERR_INVALID, "engine is NULL");
    if (e->h_rooms.empty()) return fail(NAV3D_ERR_INVALID, "no rooms loaded: call nav3d_load_rooms first");
    return NAV3D_OK;
}
// the reference raises AttributeError when step() precedes reset() (no self.x yet); here: an error code
int check_steppable(const nav3d_engine *e) {
    if (int rc = check_ready(e)) return rc;
    if (!e->reset_seen) return fail(NAV3D_ERR_INVALID, "envs were not reset since the rooms were loaded: call nav3d_reset first");
    return NAV3D_OK;
}

}  // namespace

namespace nav3d { int fail_with(int code, const std::string &msg) { return fail(code, msg); } }   // for nav3d_train.cu

extern "C" {

const char *nav3d_last_error(void) { return g_err.c_str(); }
int nav3d_abi_version(void) { return NAV3D_ABI_VERSION; }

int nav3d_create(const nav3d_config *cfg, nav3d_engine **out) {
    if (!cfg || !out) return fail(NAV3D_ERR_INVALID, "cfg/out is NULL");
    *out = nullptr;
    if (cfg->abi_version != NAV3D_ABI_VERSION) return fail(NAV3D_ERR_INVALID, "abi_version mismatch");
    if (cfg->n_envs <= 0) return fail(NAV3D_ERR_INVALID, "n_envs must be positive");
    if (cfg->env_kind != NAV3D_ENV_CUBIC && cfg->env_kind != NAV3D_ENV_SIMPLE)
        return fail(NAV3D_ERR_INVALID, "env_kind must be NAV3D_ENV_CUBIC or NAV3D_ENV_SIMPLE");
    if (cfg->local_map_length < 1 || cfg->local_map_length > 255)
        return fail(NAV3D_ERR_UNSUPPORTED, "local_map_length must be in 1..255");
    // Defaults from the sweeps in DESIGN.md §6: one thread per env — CubicEnv: the step_tpe / rollout_tpe kernels, 8 CTAs of
    // 64 threads per SM at 128 registers; simpleEnv: simple_step_tpe_kernel (rows of more than 95 floats: 2 lanes per env).
    const int simple_dim = 6 * cfg->local_map_length + 7;
    int G = cfg->lanes_per_env == 0 ? ((cfg->env_kind == NAV3D_ENV_SIMPLE && simple_dim > 95) ? 2 : 1) : cfg->lanes_per_env;
    if (!(G == 1 || G == 2 || G == 4 || G == 8 || G == 16 || G == 32))
        return fail(NAV3D_ERR_INVALID, "lanes_per_env must be 0, 1, 2, 4, 8, 16 or 32");
    int ndev = 0;
    CUDA_TRY(cudaGetDeviceCount(&ndev));
    if (cfg->device < 0 || cfg->device >= ndev) return fail(NAV3D_ERR_INVALID, "device ordinal out of range");
    CUDA_TRY(cudaSetDevice(cfg->device));
    nav3d_engine *e = new (std::nothrow) nav3d_engine();
    if (!e) return fail(NAV3D_ERR_NOMEM, "out of host memory");
    e->cfg = *cfg;
    e->G = G;
    e->minb = (cfg->env_kind == NAV3D_ENV_SIMPLE || G > 1) ? 8 : 3;
    if (const char *mb = getenv("NAV3D_MINB")) { if (atoi(mb) > 0) e->minb = atoi(mb); }   // tuning knob (tools/*sweep.sh)
    if (const char *pd = getenv("NAV3D_PDL")) e->pdl = atoi(pd) != 0;
    if (const char *v = getenv("NAV3D_TPE_STAGED")) e->tpe_staged = atoi(v) != 0;
    if (const char *v = getenv("NAV3D_TPE_BLOCK")) e->tpe_block = atoi(v) == 128 ? 128 : 64;
    const size_t N = (size_t)cfg->n_envs;
    cudaError_t err = cudaSuccess;
    if ((err = cudaMalloc(&e->d_states, N * sizeof(EnvState))) != cudaSuccess ||
        (err = cudaMalloc(&e->d_reward, N * sizeof(float))) != cudaSuccess ||
        (err = cudaMalloc(&e->d_term, N)) != cudaSuccess || (err = cudaMalloc(&e->d_trunc, N)) != cudaSuccess ||
        (err = cudaStreamCreateWithFlags(&e->own_stream, cudaStreamNonBlocking)) != cudaSuccess) {
        nav3d_destroy(e);
        return fail(NAV3D_ERR_CUDA, std::string("nav3d_create: ") + cudaGetErrorString(err));
    }
    EngineParams &P = e->P;
    P.states = e->d_states;
    P.n_envs = cfg->n_envs;
    P.L = cfg->local_map_length;
    P.env_id0 = cfg->env_id0;
    P.seed_lo = (uint32_t)cfg->seed;
    P.seed_hi = (uint32_t)(cfg->seed >> 32);
    P.auto_reset = cfg->auto_reset ? 1 : 0;
    P.rw = reference_reward_params(cfg->crash_penalty);
    e->simple = cfg->env_kind == NAV3D_ENV_SIMPLE;
    if (e->simple && G == 1 && simple_dim <= 95) {
        e->simple_stride = simple_dim;          // 6L+7 is odd: 32 rows at this stride fall into 32 different banks
        if (!e->tpe_staged) e->simple_stride = 0;
        else cudaFuncSetAttribute(simple_step_tpe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)(kBlock * e->simple_stride * sizeof(float)));
    }
    P.obs_dim = e->simple ? 6 * cfg->local_map_length + 7 : kObsDim;
    if (e->simple) {
        // distances of simpleEnv: round(count * cell_size, 2) (simpleEnv.py:337) then float32
        std::vector<float> lut((size_t)cfg->local_map_length + 1);
        for (int c = 0; c <= cfg->local_map_length; c++)
            lut[(size_t)c] = (float)(std::nearbyint((double)c * cfg->cell_size * 100.0) / 100.0);
        if ((err = cudaMalloc(&e->d_dist_lut, lut.size() * sizeof(float))) != cudaSuccess ||
            (err = cudaMemcpy(e->d_dist_lut, lut.data(), lut.size() * sizeof(float), cudaMemcpyHostToDevice)) != cudaSuccess) {
            nav3d_destroy(e);
            return fail(NAV3D_ERR_CUDA, std::string("nav3d_create: ") + cudaGetErrorString(err));
        }
        P.dist_lut = e->d_dist_lut;
    }
    *out = e;
    return NAV3D_OK;
}

void nav3d_destroy(nav3d_engine *e) {
    if (!e) return;
    DeviceGuard guard(e->cfg.device);
    free_rooms(e);
    cudaFree(e->d_states); cudaFree(e->d_reward); cudaFree(e->d_term); cudaFree(e->d_trunc);
    cudaFree(e->d_obs); cudaFree(e->d_actions); cudaFree(e->d_dist_lut);
    if (e->own_stream) cudaStreamDestroy(e->own_stream);
    if (e->copy_stream) {
        cudaStreamDestroy(e->copy_stream);
        for (auto &ev : e->chunk_done) if (ev) cudaEventDestroy(ev);
    }
    delete e;
}

int nav3d_load_rooms(nav3d_engine *e, int32_t n_rooms, const nav3d_room_desc *rooms) {
    if (!e || !rooms) return fail(NAV3D_ERR_INVALID, "engine/rooms is NULL");
    if (n_rooms <= 0 || n_rooms > 65535) return fail(NAV3D_ERR_UNSUPPORTED, "n_rooms must be in 1..65535");
    NAV3D_DEVICE(e);
    std::vector<RoomDev> hr((size_t)n_rooms);
    std::vector<uint32_t> dense_off((size_t)n_rooms);
    std::vector<int32_t> wall((size_t)n_rooms);
    size_t n_dense = 0, n_occz = 0, n_occ64 = 0, n_free_cap = 0, max_k = 0, max_cells = 0;
    int max_w = 1, max_d = 1;
    std::vector<uint32_t> start((size_t)n_rooms, 0xffffffffu);
    for (int i = 0; i < n_rooms; i++) {
        const nav3d_room_desc &d = rooms[i];
        if (!d.grid) return fail(NAV3D_ERR_INVALID, "room grid is NULL");
        if (d.width < 1 || d.depth < 1 || d.height < 1)
            return fail(NAV3D_ERR_ROOM, "room " + std::to_string(i) + ": non-positive dimension");
        if (d.width > NAV3D_MAX_WIDTH || d.depth > NAV3D_MAX_DEPTH || d.height > NAV3D_MAX_HEIGHT)
            return fail(NAV3D_ERR_UNSUPPORTED, "room " + std::to_string(i) + ": " + std::to_string(d.width) + "x" +
                                                   std::to_string(d.depth) + "x" + std::to_string(d.height) +
                                                   " exceeds the 64x64x16 limit of this build");
        RoomDev &R = hr[(size_t)i];
        R.W = (uint16_t)d.width; R.D = (uint16_t)d.depth; R.H = (uint16_t)d.height;
        if (e->simple) {       // one u32 per column, 4x4 columns per 64-byte tile
            R.ntx = (uint16_t)((d.width + 3) / 4); R.nty = (uint16_t)((d.depth + 3) / 4); R.nzb = 1;
        } else {               // bordered volume: 2 columns below, 1 above (the window reaches x-2 .. x+1); 6 levels per brick
            R.ntx = (uint16_t)((d.width + kPadLo + 1 + 3) / 4); R.nty = (uint16_t)((d.depth + kPadLo + 1 + 3) / 4);
            R.nzb = (uint16_t)((d.height + 5) / 6);
        }
        R.n_free = 0;
        R.occz_off = (uint32_t)n_occz;  n_occz += (size_t)d.width * d.depth;
        R.occx_off = (uint32_t)n_occ64; n_occ64 += (size_t)d.depth * d.height;
        R.occy_off = (uint32_t)n_occ64; n_occ64 += (size_t)d.width * d.height;
        R.free_off = (uint32_t)n_free_cap; n_free_cap += (size_t)d.width * d.depth * d.height;
        dense_off[(size_t)i] = (uint32_t)n_dense; n_dense += (size_t)d.width * d.depth * d.height;
        wall[(size_t)i] = d.wall_code;
        max_k = std::max(max_k, (size_t)(e->simple ? k2_bytes(R) : k_bytes(R)));
        max_cells = std::max(max_cells, (size_t)d.width * d.depth * d.height);
        max_w = std::max(max_w, (int)d.width); max_d = std::max(max_d, (int)d.depth);
        // "Start position=" of the room file (CubicEnv.py:415-416, :461-466): used instead of a random start when it is a
        // cell of the room and not a wall (the reference re-picks a random one otherwise)
        if (d.has_start && d.start_x >= 0 && d.start_x < d.width && d.start_y >= 0 && d.start_y < d.depth && d.start_z >= 0 &&
            d.start_z < d.height &&
            d.grid[((size_t)d.start_x * d.depth + d.start_y) * d.height + d.start_z] != d.wall_code)
            start[(size_t)i] = (uint32_t)d.start_x | ((uint32_t)d.start_y << 8) | ((uint32_t)d.start_z << 16);
    }
    std::vector<int8_t> dense(n_dense);
    for (int i = 0; i < n_rooms; i++)
        std::memcpy(dense.data() + dense_off[(size_t)i], rooms[i].grid,
                    (size_t)rooms[i].width * rooms[i].depth * rooms[i].height);

    free_rooms(e);
    int8_t *d_dense = nullptr; uint32_t *d_off = nullptr, *d_nwall = nullptr; int32_t *d_wall = nullptr;
    // per-env block: [K bricks of the largest room | overflow bytes (one per cell, touched only by counters >= 29)]
    e->P.mark_cap = 32 * mark_tasks_per_lane(e->cfg.local_map_length, max_w, max_d);
    if (!e->simple && max_k / 4 > 65536)          // a marking task names its tile by a 16-bit word index (MarkQueue)
        return fail(NAV3D_ERR_UNSUPPORTED, "room too large for the marking-task encoding (K volume above 65 536 words)");
    if (!e->simple) {
        // The default thread-per-env kernels: ask for no more shared memory than their 8 CTAs per SM need, so that the rest
        // of the 256 KB stays L1 (experiment knob NAV3D_CARVEOUT = percent of the maximum shared memory; 0 = driver's choice)
        const size_t per_cta = 7680 + 2 * e->P.mark_cap * sizeof(uint32_t) + 1024;
        int pct = (int)((8 * per_cta * 100 + 228 * 1024 - 1) / (228 * 1024));
        if (const char *v = getenv("NAV3D_CARVEOUT")) pct = atoi(v);
        if (pct > 0 && pct <= 100) {
            cudaFuncSetAttribute(step_tpe_kernel<64, 8, true>, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
            cudaFuncSetAttribute(rollout_tpe_kernel<64, 8, true>, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
            cudaFuncSetAttribute(rollout_actions_tpe_kernel<64, 8>, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
        }
    }
    size_t ovf_off = align_up(max_k, 128), stride = ovf_off + align_up(max_cells, 128);
    if (e->simple) { ovf_off = 0; stride = align_up(max_k, 128); }
    const size_t know_bytes = stride * (size_t)e->cfg.n_envs;
    auto cleanup_tmp = [&]() { cudaFree(d_dense); cudaFree(d_off); cudaFree(d_nwall); cudaFree(d_wall); };
#define LOAD_TRY(expr)                                                                                      \
    do {                                                                                                    \
        cudaError_t _e = (expr);                                                                            \
        if (_e != cudaSuccess) {                                                                            \
            cleanup_tmp(); free_rooms(e);                                                                   \
            return fail(_e == cudaErrorMemoryAllocation ? NAV3D_ERR_NOMEM : NAV3D_ERR_CUDA,                 \
                        std::string(#expr) + ": " + cudaGetErrorString(_e));                                \
        }                                                                                                   \
    } while (0)
    LOAD_TRY(cudaMalloc(&d_dense, n_dense));
    LOAD_TRY(cudaMalloc(&d_off, sizeof(uint32_t) * n_rooms));
    LOAD_TRY(cudaMalloc(&d_nwall, sizeof(uint32_t) * n_rooms));
    LOAD_TRY(cudaMalloc(&d_wall, sizeof(int32_t) * n_rooms));
    LOAD_TRY(cudaMalloc(&e->d_rooms, sizeof(RoomDev) * n_rooms));
    LOAD_TRY(cudaMalloc(&e->d_occz, sizeof(uint16_t) * n_occz));
    LOAD_TRY(cudaMalloc(&e->d_occ64, sizeof(unsigned long long) * n_occ64));
    LOAD_TRY(cudaMalloc(&e->d_free, sizeof(uint32_t) * n_free_cap));
    LOAD_TRY(cudaMalloc(&e->d_know, know_bytes));
    LOAD_TRY(cudaMalloc(&e->d_start, sizeof(uint32_t) * n_rooms));
    LOAD_TRY(cudaMemcpy(e->d_start, start.data(), sizeof(uint32_t) * n_rooms, cudaMemcpyHostToDevice));
    LOAD_TRY(cudaMemcpy(d_dense, dense.data(), n_dense, cudaMemcpyHostToDevice));
    LOAD_TRY(cudaMemcpy(d_off, dense_off.data(), sizeof(uint32_t) * n_rooms, cudaMemcpyHostToDevice));
    LOAD_TRY(cudaMemcpy(d_wall, wall.data(), sizeof(int32_t) * n_rooms, cudaMemcpyHostToDevice));
    LOAD_TRY(cudaMemcpy(e->d_rooms, hr.data(), sizeof(RoomDev) * n_rooms, cudaMemcpyHostToDevice));
    LOAD_TRY(cudaMemset(e->d_free, 0, sizeof(uint32_t) * n_free_cap));
    pack_rooms_kernel<<<n_rooms, 256>>>(d_dense, d_off, d_wall, e->d_rooms, e->d_occz, e->d_occ64, e->d_free, d_nwall);
    e->launches++;
    LOAD_TRY(cudaGetLastError());
    e->h_free.resize(n_free_cap);
    e->h_nwall.resize((size_t)n_rooms);
    LOAD_TRY(cudaMemcpy(hr.data(), e->d_rooms, sizeof(RoomDev) * n_rooms, cudaMemcpyDeviceToHost));
    LOAD_TRY(cudaMemcpy(e->h_free.data(), e->d_free, sizeof(uint32_t) * n_free_cap, cudaMemcpyDeviceToHost));
    LOAD_TRY(cudaMemcpy(e->h_nwall.data(), d_nwall, sizeof(uint32_t) * n_rooms, cudaMemcpyDeviceToHost));
    init_states_kernel<<<(e->cfg.n_envs + 255) / 256, 256>>>(e->d_states, e->cfg.n_envs);
    LOAD_TRY(cudaGetLastError());
    LOAD_TRY(cudaDeviceSynchronize());
#undef LOAD_TRY
    cleanup_tmp();
    for (int i = 0; i < n_rooms; i++)
        if (hr[(size_t)i].n_free == 0) {
            free_rooms(e);
            // the reference would fail in random.choice([]) (CubicEnv.py:462)
            return fail(NAV3D_ERR_ROOM, "room " + std::to_string(i) + " has no free interior cell");
        }
    e->h_rooms = hr;
    e->know_bytes = know_bytes;
    e->signature = sig_engine(e->cfg.env_kind, e->cfg.local_map_length, stride);
    for (int i = 0; i < n_rooms; i++)
        e->signature = sig_room(e->signature, rooms[i].width, rooms[i].depth, rooms[i].height, rooms[i].wall_code,
                                rooms[i].grid, start[(size_t)i]);
    e->room_bytes = sizeof(RoomDev) * n_rooms + 2 * n_occz + 8 * n_occ64 + 4 * n_free_cap;
    EngineParams &P = e->P;
    P.rooms = e->d_rooms; P.occz = e->d_occz; P.occ64 = e->d_occ64; P.free_cells = e->d_free;
    P.know = e->d_know; P.env_stride = stride; P.ovf_off = (uint32_t)ovf_off; P.n_rooms = n_rooms;
    P.room_start = e->d_start;
    e->reset_seen = false;
    return NAV3D_OK;
}

void nav3d_reward_params_default(nav3d_reward_params *out) {
    if (!out) return;
    const RewardParams w = reference_reward_params(-2.0);
    out->step_cost = w.step_cost; out->revisit_unit = w.revisit_unit; out->revisit_cap = w.revisit_cap;
    out->crash_penalty = w.crash_penalty; out->near_wall_bonus = w.near_wall_bonus; out->repeat_bonus = w.repeat_bonus;
    out->reverse_penalty = w.reverse_penalty; out->explore_bonus = w.explore_bonus; out->finish_bonus = w.finish_bonus;
    out->truncation_penalty = w.truncation_penalty;
}

int nav3d_set_reward_params(nav3d_engine *e, const nav3d_reward_params *p) {
    if (!e || !p) return fail(NAV3D_ERR_INVALID, "engine/params is NULL");
    if (e->simple) return fail(NAV3D_ERR_UNSUPPORTED, "reward parameters apply to NAV3D_ENV_CUBIC only");
    const double v[10] = {p->step_cost, p->revisit_unit, p->revisit_cap, p->crash_penalty, p->near_wall_bonus, p->repeat_bonus,
                          p->reverse_penalty, p->explore_bonus, p->finish_bonus, p->truncation_penalty};
    for (double x : v) if (!std::isfinite(x) || std::fabs(x) > 1e6) return fail(NAV3D_ERR_INVALID, "reward parameter out of range");
    RewardParams w = reference_reward_params(p->crash_penalty);
    w.step_cost = p->step_cost; w.revisit_unit = p->revisit_unit; w.revisit_cap = p->revisit_cap;
    w.near_wall_bonus = p->near_wall_bonus; w.repeat_bonus = p->repeat_bonus; w.reverse_penalty = p->reverse_penalty;
    w.explore_bonus = p->explore_bonus; w.finish_bonus = p->finish_bonus; w.truncation_penalty = p->truncation_penalty;
    w.c_step = reward_centi(w.step_cost); w.c_revisit_unit = reward_centi(w.revisit_unit);
    w.c_revisit_cap = reward_centi(w.revisit_cap); w.c_near_wall = reward_centi(w.near_wall_bonus);
    w.c_repeat = reward_centi(w.repeat_bonus); w.c_reverse = reward_centi(w.reverse_penalty);
    w.c_explore = reward_centi(w.explore_bonus); w.c_finish = reward_centi(w.finish_bonus);
    w.c_trunc = reward_centi(w.truncation_penalty);
    e->P.rw = w;
    return NAV3D_OK;
}

int nav3d_room_info(nav3d_engine *e, int32_t room, int32_t *out6) {
    if (int rc = check_ready(e)) return rc;
    if (!out6 || room < 0 || room >= (int)e->h_rooms.size()) return fail(NAV3D_ERR_INVALID, "bad room index");
    const RoomDev &R = e->h_rooms[(size_t)room];
    out6[0] = R.W; out6[1] = R.D; out6[2] = R.H; out6[3] = (int32_t)R.n_free; out6[4] = (int32_t)e->h_nwall[(size_t)room];
    out6[5] = 0;
    return NAV3D_OK;
}

int nav3d_room_free_cell(nav3d_engine *e, int32_t room, int32_t k, int32_t *xyz) {
    if (int rc = check_ready(e)) return rc;
    if (!xyz || room < 0 || room >= (int)e->h_rooms.size()) return fail(NAV3D_ERR_INVALID, "bad room index");
    const RoomDev &R = e->h_rooms[(size_t)room];
    if (k < 0 || (uint32_t)k >= R.n_free) return fail(NAV3D_ERR_INVALID, "free-cell index out of range");
    const uint32_t c = e->h_free[R.free_off + (uint32_t)k];
    xyz[0] = c & 0xff; xyz[1] = (c >> 8) & 0xff; xyz[2] = (c >> 16) & 0xff;
    return NAV3D_OK;
}

int nav3d_obs_dim(const nav3d_engine *e) { return e ? e->P.obs_dim : 0; }
int nav3d_num_envs(const nav3d_engine *e) { return e ? e->cfg.n_envs : 0; }
int nav3d_lanes_per_env(const nav3d_engine *e) { return e ? e->G : 0; }
uint64_t nav3d_launch_count(const nav3d_engine *e) { return e ? e->launches : 0; }
size_t nav3d_device_bytes(const nav3d_engine *e) {
    if (!e) return 0;
    return e->know_bytes + e->room_bytes + (size_t)e->cfg.n_envs * (sizeof(EnvState) + 6);
}

int nav3d_reset(nav3d_engine *e, const int32_t *env_ids, int32_t n, const int32_t *picks, float *obs, void *stream) {
    if (int rc = check_ready(e)) return rc;
    if (n < 0 || (!env_ids && n > e->cfg.n_envs)) return fail(NAV3D_ERR_INVALID, "n out of range");
    if (n == 0) return NAV3D_OK;
    if (obs && !e->simple && ((uintptr_t)obs & 15u)) return fail(NAV3D_ERR_INVALID, "obs must be 16-byte aligned");
    NAV3D_DEVICE(e);
    NvtxRange range("nav3d_reset");
    e->reset_seen = true;
    cudaStream_t s = (cudaStream_t)stream;
    int rc = NAV3D_OK;
    if (!e->simple && e->G == 1)
        reset_tpe_kernel<<<grid_for(n, 1), kBlock, (kBlock / 32) * e->P.mark_cap * sizeof(uint32_t), s>>>(e->P, env_ids, n, picks, obs);
    else rc = dispatch_lanes(e->G, [&](auto g) {
        constexpr int G = decltype(g)::value;
        if (e->simple) simple_reset_kernel<G><<<grid_for(n, G), kBlock, 0, s>>>(e->P, env_ids, n, picks, obs);
        else reset_kernel<G><<<grid_for(n, G), kBlock, 0, s>>>(e->P, env_ids, n, picks, obs);
        return NAV3D_OK;
    });
    if (rc) return rc;
    e->launches++;
    CUDA_TRY(cudaGetLastError());
    return NAV3D_OK;
}

}  // extern "C"

namespace {

// Launch the step of envs [env0, env0 + n) on `s` (the whole engine: env0 = 0, n = n_envs).
int launch_step(nav3d_engine *e, StepIO io, int env0, int n, cudaStream_t s) {
    io.env0 = env0; io.env_n = n;
    const int minb = e->minb;
    int rc = dispatch_lanes(e->G, [&](auto g) {
        constexpr int G = decltype(g)::value;
        const unsigned grid = grid_for(n, G);
        cudaLaunchConfig_t cfg{};
        cfg.gridDim = dim3(grid); cfg.blockDim = dim3(kBlock); cfg.dynamicSmemBytes = 0; cfg.stream = s;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = e->pdl ? 1 : 0;
        cfg.attrs = attr; cfg.numAttrs = 1;
        if (e->simple) {
            if (G == 1 && e->simple_stride > 0) {      // thread per env, staged rows (6L+7 <= 95 floats)
                cfg.dynamicSmemBytes = (size_t)kBlock * e->simple_stride * sizeof(float);
                cudaLaunchKernelEx(&cfg, simple_step_tpe_kernel, e->P, io, e->simple_stride);
                return NAV3D_OK;
            }
            if (minb == 6) cudaLaunchKernelEx(&cfg, simple_step_kernel<G, 6>, e->P, io);
            else cudaLaunchKernelEx(&cfg, simple_step_kernel<G, 8>, e->P, io);
            return NAV3D_OK;
        }
        if (G == 1) {                                  // thread per env: staged, coalesced observation stores
            const bool staged = e->tpe_staged;
            // Default: 64-thread CTAs, 8 per SM (128 registers, 16 warps per SM) — the sweep of DESIGN.md §6; NAV3D_TPE_BLOCK=128
            // selects the 128-thread kernels (NAV3D_MINB 3: 168 registers / 12 warps, 4: 128 / 16)
            const int tblock = e->tpe_block;
            cfg.dynamicSmemBytes = (size_t)(tblock / 32) * e->P.mark_cap * sizeof(uint32_t);   // one marking list per warp
            if (tblock == 64 && staged) {
                cfg.gridDim = dim3((unsigned)((n + 63) / 64)); cfg.blockDim = dim3(64);
                cudaLaunchKernelEx(&cfg, step_tpe_kernel<64, 8, true>, e->P, io);
                return NAV3D_OK;
            }
            switch (minb * 2 + (staged ? 1 : 0)) {
                case 8: cudaLaunchKernelEx(&cfg, step_tpe_kernel<128, 4, false>, e->P, io); break;
                case 9: cudaLaunchKernelEx(&cfg, step_tpe_kernel<128, 4, true>, e->P, io); break;
                case 6: cudaLaunchKernelEx(&cfg, step_tpe_kernel<128, 3, false>, e->P, io); break;
                default: cudaLaunchKernelEx(&cfg, step_tpe_kernel<128, 3, true>, e->P, io); break;
            }
            return NAV3D_OK;
        }
        if (minb == 6) cudaLaunchKernelEx(&cfg, step_call_kernel<G, 6>, e->P, io);
        else cudaLaunchKernelEx(&cfg, step_call_kernel<G, 8>, e->P, io);
        return NAV3D_OK;
    });
    if (rc) return rc;
    e->launches += 1;
    CUDA_TRY(cudaGetLastError());
    return NAV3D_OK;
}

}  // namespace

extern "C" {

int nav3d_step(nav3d_engine *e, const int64_t *actions, float *obs, float *reward, double *reward64,
               uint8_t *terminated, uint8_t *truncated, float *terminal_obs, nav3d_episode *episodes, void *stream) {
    if (int rc = check_steppable(e)) return rc;
    if (!actions || !obs || !reward || !terminated || !truncated)
        return fail(NAV3D_ERR_INVALID, "actions, obs, reward, terminated and truncated are required");
    if (!e->simple && (((uintptr_t)obs & 15u) || (terminal_obs && ((uintptr_t)terminal_obs & 15u))))
        return fail(NAV3D_ERR_INVALID, "obs / terminal_obs must be 16-byte aligned");
    NAV3D_DEVICE(e);
    NvtxRange range("nav3d_step");
    StepIO io;
    io.actions = reinterpret_cast<const long long *>(actions);
    io.obs = obs; io.reward = reward; io.reward64 = reward64; io.terminated = terminated; io.truncated = truncated;
    io.terminal_obs = terminal_obs; io.episodes = episodes;
    return launch_step(e, io, 0, e->cfg.n_envs, (cudaStream_t)stream);
}

// The host-buffer step is a copy pipeline: the envs are cut into chunks; chunk c's actions go up and its step runs on the
// compute stream while chunk c-1's observations, rewards and flags come down on the copy stream.  The device->host copy of
// the observations (320 B per env) is what bounds this path (PCIe), so everything else hides behind it.
int nav3d_step_host(nav3d_engine *e, const int64_t *actions, float *obs, float *reward, uint8_t *terminated,
                    uint8_t *truncated) {
    if (int rc = check_steppable(e)) return rc;
    if (!actions || !obs || !reward || !terminated || !truncated) return fail(NAV3D_ERR_INVALID, "NULL host buffer");
    NAV3D_DEVICE(e);
    NvtxRange range("nav3d_step_host");
    const size_t N = (size_t)e->cfg.n_envs;
    const size_t obs_dim = (size_t)e->P.obs_dim;
    if (!e->d_obs) CUDA_TRY(cudaMalloc(&e->d_obs, N * obs_dim * sizeof(float)));
    if (!e->d_actions) CUDA_TRY(cudaMalloc(&e->d_actions, N * sizeof(long long)));
    if (!e->copy_stream) {
        CUDA_TRY(cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking));
        for (auto &ev : e->chunk_done) CUDA_TRY(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    }
    cudaStream_t sc = e->own_stream, sd = e->copy_stream;
    const int chunks = N >= 65536 ? nav3d_engine::kHostChunks : 1;
    StepIO io;
    io.actions = e->d_actions; io.obs = e->d_obs; io.reward = e->d_reward; io.reward64 = nullptr;
    io.terminated = e->d_term; io.truncated = e->d_trunc; io.terminal_obs = nullptr; io.episodes = nullptr;
    for (int c = 0; c < chunks; c++) {
        const size_t b0 = N * c / chunks, b1 = N * (c + 1) / chunks, cnt = b1 - b0;
        CUDA_TRY(cudaMemcpyAsync(e->d_actions + b0, actions + b0, cnt * sizeof(long long), cudaMemcpyHostToDevice, sc));
        if (int rc = launch_step(e, io, (int)b0, (int)cnt, sc)) return rc;
        CUDA_TRY(cudaEventRecord(e->chunk_done[c], sc));
        CUDA_TRY(cudaStreamWaitEvent(sd, e->chunk_done[c], 0));
        CUDA_TRY(cudaMemcpyAsync(obs + b0 * obs_dim, e->d_obs + b0 * obs_dim, cnt * obs_dim * sizeof(float), cudaMemcpyDeviceToHost, sd));
        CUDA_TRY(cudaMemcpyAsync(reward + b0, e->d_reward + b0, cnt * sizeof(float), cudaMemcpyDeviceToHost, sd));
        CUDA_TRY(cudaMemcpyAsync(terminated + b0, e->d_term + b0, cnt, cudaMemcpyDeviceToHost, sd));
        CUDA_TRY(cudaMemcpyAsync(truncated + b0, e->d_trunc + b0, cnt, cudaMemcpyDeviceToHost, sd));
    }
    CUDA_TRY(cudaStreamSynchronize(sd));
    CUDA_TRY(cudaStreamSynchronize(sc));
    return NAV3D_OK;
}

int nav3d_rollout_random(nav3d_engine *e, int32_t T, uint32_t t0, float *obs, float *obs_last, float *reward,
                         uint8_t *done, uint8_t *actions_out, void *stream) {
    if (int rc = check_steppable(e)) return rc;
    if (T < 0) return fail(NAV3D_ERR_INVALID, "T must be >= 0");

    if (e->simple) return fail(NAV3D_ERR_UNSUPPORTED, "nav3d_rollout_random is implemented for NAV3D_ENV_CUBIC only");
    if (T == 0) return NAV3D_OK;
    if (!obs && !obs_last) return fail(NAV3D_ERR_INVALID, "one of obs / obs_last is required");
    if ((obs && ((uintptr_t)obs & 15u)) || (obs_last && ((uintptr_t)obs_last & 15u)))
        return fail(NAV3D_ERR_INVALID, "obs must be 16-byte aligned");
    NAV3D_DEVICE(e);
    NvtxRange range("nav3d_rollout_random");
    cudaStream_t s = (cudaStream_t)stream;
    int rc = dispatch_lanes(e->G, [&](auto g) {
        constexpr int G = decltype(g)::value;
        if (G == 1) {
            const int tblock = e->tpe_block;
            if (tblock == 64)
                rollout_tpe_kernel<64, 8, true><<<(unsigned)((e->cfg.n_envs + 63) / 64), 64, 2 * e->P.mark_cap * sizeof(uint32_t), s>>>(e->P, T, t0, obs, obs_last,
                                                                                                  reward, done, actions_out);
            else if (e->minb == 4)
                rollout_tpe_kernel<128, 4, true><<<grid_for(e->cfg.n_envs, 1), kBlock, 4 * e->P.mark_cap * sizeof(uint32_t), s>>>(e->P, T, t0, obs, obs_last, reward,
                                                                                            done, actions_out);
            else
                rollout_tpe_kernel<128, 3, true><<<grid_for(e->cfg.n_envs, 1), kBlock, 4 * e->P.mark_cap * sizeof(uint32_t), s>>>(e->P, T, t0, obs, obs_last, reward,
                                                                                            done, actions_out);
            return NAV3D_OK;
        }
        rollout_kernel<G, 6><<<grid_for(e->cfg.n_envs, G), kBlock, 0, s>>>(e->P, T, t0, obs, obs_last, reward, done, actions_out,
                                                                           e->d_reward, e->d_term, e->d_trunc);
        return NAV3D_OK;
    });
    if (rc) return rc;
    e->launches++;
    CUDA_TRY(cudaGetLastError());
    return NAV3D_OK;
}

int nav3d_rollout_actions(nav3d_engine *e, int32_t T, const uint8_t *actions, float *obs, float *obs_last, float *reward,
                          double *reward64, uint8_t *terminated, uint8_t *truncated, float *terminal_obs,
                          nav3d_episode *episodes, void *stream) {
    if (T < 0) return fail(NAV3D_ERR_INVALID, "T must be >= 0");
    if (!actions) return fail(NAV3D_ERR_INVALID, "actions is required");
    if (!obs && !obs_last) return fail(NAV3D_ERR_INVALID, "one of obs / obs_last is required");
    if (((uintptr_t)obs | (uintptr_t)obs_last | (uintptr_t)terminal_obs) & 15u)
        return fail(NAV3D_ERR_INVALID, "obs / obs_last / terminal_obs must be 16-byte aligned");
    if (int rc = check_steppable(e)) return rc;
    if (e->simple) return fail(NAV3D_ERR_UNSUPPORTED, "nav3d_rollout_actions is implemented for NAV3D_ENV_CUBIC only");
    if (T == 0) return NAV3D_OK;
    NAV3D_DEVICE(e);
    NvtxRange range("nav3d_rollout_actions");
    RolloutIO ro;
    ro.actions = actions; ro.obs = obs; ro.obs_last = obs_last; ro.reward = reward; ro.reward64 = reward64;
    ro.terminated = terminated; ro.truncated = truncated; ro.terminal_obs = terminal_obs; ro.episodes = episodes;
    cudaStream_t s = (cudaStream_t)stream;
    const int n = e->cfg.n_envs;
    int rc = dispatch_lanes(e->G, [&](auto g) {
        constexpr int G = decltype(g)::value;
        if constexpr (G == 1) {           // the launch configurations of nav3d_rollout_random
            const size_t smem = (size_t)(e->tpe_block / 32) * e->P.mark_cap * sizeof(uint32_t);
            if (e->tpe_block == 64) rollout_actions_tpe_kernel<64, 8><<<(unsigned)((n + 63) / 64), 64, smem, s>>>(e->P, T, ro);
            else if (e->minb == 4) rollout_actions_tpe_kernel<128, 4><<<grid_for(n, 1), kBlock, smem, s>>>(e->P, T, ro);
            else rollout_actions_tpe_kernel<128, 3><<<grid_for(n, 1), kBlock, smem, s>>>(e->P, T, ro);
        } else {
            rollout_actions_kernel<G, 6><<<grid_for(n, G), kBlock, 0, s>>>(e->P, T, ro);
        }
        return NAV3D_OK;
    });
    if (rc) return rc;
    e->launches++;
    CUDA_TRY(cudaGetLastError());
    return NAV3D_OK;
}

int nav3d_get_state(nav3d_engine *e, int32_t *state, void *stream) {
    if (int rc = check_ready(e)) return rc;
    if (!state) return fail(NAV3D_ERR_INVALID, "state is NULL");
    NAV3D_DEVICE(e);
    get_state_kernel<<<(e->cfg.n_envs + 255) / 256, 256, 0, (cudaStream_t)stream>>>(e->P, state);
    e->launches++;
    CUDA_TRY(cudaGetLastError());
    return NAV3D_OK;
}

int nav3d_get_grid(nav3d_engine *e, int32_t env, int16_t *grid, void *stream) {
    if (int rc = check_ready(e)) return rc;
    if (!grid || env < 0 || env >= e->cfg.n_envs) return fail(NAV3D_ERR_INVALID, "bad env index / NULL grid");
    NAV3D_DEVICE(e);
    if (e->simple) simple_get_grid_kernel<<<32, 256, 0, (cudaStream_t)stream>>>(e->P, env, grid);
    else get_grid_kernel<<<32, 256, 0, (cudaStream_t)stream>>>(e->P, env, grid);
    e->launches++;
    CUDA_TRY(cudaGetLastError());
    return NAV3D_OK;
}

size_t nav3d_snapshot_bytes(const nav3d_engine *e) {
    if (!e || e->h_rooms.empty()) return 0;
    return (size_t)e->cfg.n_envs * sizeof(EnvState) + e->know_bytes;
}

int nav3d_snapshot(nav3d_engine *e, void *host_buf, size_t bytes) {
    if (int rc = check_ready(e)) return rc;
    if (!host_buf || bytes != nav3d_snapshot_bytes(e)) return fail(NAV3D_ERR_INVALID, "snapshot buffer size mismatch");
    NAV3D_DEVICE(e);
    CUDA_TRY(cudaDeviceSynchronize());
    const size_t sb = (size_t)e->cfg.n_envs * sizeof(EnvState);
    CUDA_TRY(cudaMemcpy(host_buf, e->d_states, sb, cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaMemcpy((char *)host_buf + sb, e->d_know, e->know_bytes, cudaMemcpyDeviceToHost));
    return NAV3D_OK;
}

int nav3d_restore(nav3d_engine *e, const void *host_buf, size_t bytes) {
    if (int rc = check_ready(e)) return rc;
    if (!host_buf || bytes != nav3d_snapshot_bytes(e)) return fail(NAV3D_ERR_INVALID, "snapshot buffer size mismatch");
    NAV3D_DEVICE(e);
    CUDA_TRY(cudaDeviceSynchronize());
    const size_t sb = (size_t)e->cfg.n_envs * sizeof(EnvState);
    CUDA_TRY(cudaMemcpy(e->d_states, host_buf, sb, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(e->d_know, (const char *)host_buf + sb, e->know_bytes, cudaMemcpyHostToDevice));
    e->reset_seen = true;
    return NAV3D_OK;
}

size_t nav3d_env_state_bytes(const nav3d_engine *e) {
    if (!e || e->h_rooms.empty()) return 0;
    return (size_t)blob_bytes(e->P);
}

int nav3d_save_envs(nav3d_engine *e, const int32_t *env_ids, int32_t n, const float *obs, void *blobs, void *stream) {
    if (n < 0) return fail(NAV3D_ERR_INVALID, "n must be >= 0");
    if (!obs || !blobs) return fail(NAV3D_ERR_INVALID, "obs and blobs are required");
    if (((uintptr_t)blobs & 15u)) return fail(NAV3D_ERR_INVALID, "blobs must be 16-byte aligned");
    if (int rc = check_steppable(e)) return rc;
    if (!env_ids && n > e->cfg.n_envs) return fail(NAV3D_ERR_INVALID, "n out of range");
    if (!e->simple && ((uintptr_t)obs & 15u)) return fail(NAV3D_ERR_INVALID, "obs must be 16-byte aligned");
    if (n == 0) return NAV3D_OK;
    NAV3D_DEVICE(e);
    NvtxRange range("nav3d_save_envs");
    save_envs_kernel<<<grid_for(n, 32), kBlock, 0, (cudaStream_t)stream>>>(e->P, e->signature, env_ids, n, obs,
                                                                              static_cast<uint8_t *>(blobs), blob_bytes(e->P));
    e->launches++;
    CUDA_TRY(cudaGetLastError());
    return NAV3D_OK;
}

int nav3d_load_envs(nav3d_engine *e, const int32_t *env_ids, int32_t n, const void *blobs, float *obs, uint8_t *status,
                    void *stream) {
    if (n < 0) return fail(NAV3D_ERR_INVALID, "n must be >= 0");
    if (!obs || !blobs) return fail(NAV3D_ERR_INVALID, "obs and blobs are required");
    if (((uintptr_t)blobs & 15u)) return fail(NAV3D_ERR_INVALID, "blobs must be 16-byte aligned");
    if (int rc = check_ready(e)) return rc;
    if (!env_ids && n > e->cfg.n_envs) return fail(NAV3D_ERR_INVALID, "n out of range");
    if (!e->simple && ((uintptr_t)obs & 15u)) return fail(NAV3D_ERR_INVALID, "obs must be 16-byte aligned");
    if (n == 0) return NAV3D_OK;
    NAV3D_DEVICE(e);
    NvtxRange range("nav3d_load_envs");
    e->reset_seen = true;
    load_envs_kernel<<<grid_for(n, 32), kBlock, 0, (cudaStream_t)stream>>>(e->P, e->signature, env_ids, n,
                                                                              static_cast<const uint8_t *>(blobs),
                                                                              blob_bytes(e->P), obs, status);
    e->launches++;
    CUDA_TRY(cudaGetLastError());
    return NAV3D_OK;
}

}  // extern "C"

/*
 * nav3d.h — C ABI of libnav3d_b200.so: GPU-resident, batched voxel-navigation environments for NVIDIA B200 (sm_100a).
 *
 * The reference (Noimps/3D-Navigation-Reinforcement-Learning) has no native boundary: its environment is the Python
 * class envs/CubicEnv.py::GridAgent, driven one OS process per env through stable-baselines3's SubprocVecEnv
 * (train/Grid_Train.py:170-173, :191-192).  This header is the boundary a maintainer binds instead (ctypes stub in
 * INTEGRATION.md).  Each entry point names the reference code it replaces.
 *
 * Conventions
 *   - plain C types only; every pointer documented as DEVICE points into the memory of the engine's CUDA device
 *     (e.g. torch.Tensor.data_ptr()); HOST pointers are ordinary process memory.
 *   - `stream` is a CUDA stream handle (cudaStream_t / CUstream) passed as void*; NULL = the legacy default stream.
 *     Calls that take a stream are asynchronous on it and never synchronise the host.
 *   - return value: NAV3D_OK (0) or a negative nav3d_status; nav3d_last_error() gives the message of the calling
 *     thread's last failure.  Nothing throws across this boundary.
 *   - one engine per device (or several); calls on one engine must be serialised by the caller; engines are independent.
 *   - there is NO CPU fallback: without a usable CUDA device every call fails with NAV3D_ERR_CUDA.
 *
 * Limits (checked, NAV3D_ERR_UNSUPPORTED): room width, depth <= 64, height <= 16 (the reference's largest shipped room
 * is 48x32x12); local_map_length in 1..255; at most 65535 rooms per engine.
 *
 * Random streams (counter-based Philox4x32-10, Salmon et al. SC'11) — documented because the oracle restates them:
 *   key = (seed & 0xffffffff, seed >> 32);  counter = (global_env_id, index, 0, stream_tag)
 *   stream_tag 0x52455345: index = episode number of that env (0 for the first reset); output word 0 -> room index,
 *                          word 1 -> index k into the room's list of free interior cells (x-major, then y, then z —
 *                          the order envs/CubicEnv.py:450-457 builds possible_start_pose in)
 *   stream_tag 0x41435449: index = rollout step t; output word 0 -> action
 *   a 32-bit word u maps to [0, n) as (u * n) >> 32.
 *   global_env_id = config.env_id0 + local env index, so results do not depend on how envs are sharded over GPUs.
 */
#ifndef NAV3D_H
#define NAV3D_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NAV3D_ABI_VERSION 2
#define NAV3D_OBS_DIM 80          /* envs/CubicEnv.py:58-62 */
#define NAV3D_NUM_ACTIONS 6       /* envs/CubicEnv.py:56   */
#define NAV3D_STATE_INTS 16       /* ints per env written by nav3d_get_state */
#define NAV3D_MAX_WIDTH 64
#define NAV3D_MAX_DEPTH 64
#define NAV3D_MAX_HEIGHT 16

typedef enum {
    NAV3D_OK = 0,
    NAV3D_ERR_INVALID = -1,       /* bad argument (NULL, out of range, engine without rooms, ...) */
    NAV3D_ERR_UNSUPPORTED = -2,   /* outside the limits above */
    NAV3D_ERR_CUDA = -3,          /* CUDA runtime error; message carries cudaGetErrorString */
    NAV3D_ERR_NOMEM = -4,
    NAV3D_ERR_ROOM = -5           /* malformed room (no free interior cell, bad dims) */
} nav3d_status;

typedef enum {
    NAV3D_ENV_CUBIC = 0,          /* envs/CubicEnv.py::GridAgent  — 80 f32 observations, visit-count knowledge grid   */
    NAV3D_ENV_SIMPLE = 1          /* envs/simpleEnv.py::GridAgent — 6L+7 f32 observations, ternary knowledge grid     */
} nav3d_env_kind;

typedef struct nav3d_engine nav3d_engine;

/* Constructor arguments.  Mirrors the kwargs of GridAgent.__init__ (envs/CubicEnv.py:17-29) that affect dynamics. */
typedef struct {
    int32_t abi_version;          /* = NAV3D_ABI_VERSION */
    int32_t device;               /* CUDA device ordinal */
    int32_t n_envs;               /* environments held by this engine (this GPU's shard) */
    int32_t env_kind;             /* nav3d_env_kind */
    int32_t local_map_length;     /* ray length L (CubicEnv.py:25; 10 in train/Grid_Train.py:36) */
    int32_t auto_reset;           /* 1: finished envs reset inside nav3d_step (SB3 VecEnv contract), 0: plain gym */
    int32_t lanes_per_env;        /* threads per env: 1 (one thread owns an env; rows leave through a shared-memory
                                     staging tile, written by the warp), 2,4,8,16,32 (lanes cooperate on one env);
                                     0 = engine default = 1 (simpleEnv with 6L+7 > 95: 2) */
    uint32_t env_id0;             /* global id of local env 0 (sharding) */
    uint64_t seed;                /* Philox key */
    double crash_penalty;         /* CubicEnv.py:28, -2.0 */
    double cell_size;             /* CubicEnv.py:24 / simpleEnv.py:22, 0.25 (simpleEnv distances only) */
} nav3d_config;

/* One parsed room: what load_room leaves in self.grid (envs/CubicEnv.py:421-438), as int8, C order [x][y][z].
 * A cell equal to `wall_code` is a wall: -2 for CubicEnv (after the reference's 2 -> -2 rewrite, :434), 2 for simpleEnv. */
typedef struct {
    int32_t width, depth, height;
    int32_t wall_code;
    const int8_t *grid;           /* HOST, width*depth*height bytes */
    int32_t has_start;            /* 1: the room file has a "Start position=" line (envs/CubicEnv.py:415-416) */
    int32_t start_x, start_y, start_z;   /* used for every reset into this room unless it is a wall or outside the room,
                                          * in which case a random free cell is drawn as the reference does (:461-466) */
} nav3d_room_desc;

/* The literals of compute_reward (envs/CubicEnv.py:169-224) as a POD; nav3d_reward_params_default fills in the
 * reference's values, which is what an engine uses until nav3d_set_reward_params is called (CubicEnv only).
 *   reward = step_cost - min(visit_count * revisit_unit, revisit_cap)
 *            + (bumped ? crash_penalty : [was_near_wall] near_wall_bonus + [same horizontal action again] repeat_bonus
 *                                        - [backwards twice] reverse_penalty)
 *            + [first visit] explore_bonus + [>= 84 % explored] finish_bonus + [step limit] truncation_penalty
 *
 * Episode return.  Each step adds to an int32 in 1/100 units (nav3d_get_state column 15) every term but the crash
 * penalty, each rounded on its own: round(100 * v) half away from zero, for the revisit term of the f64 value
 * min(visit_count * revisit_unit, revisit_cap) of that step.  nav3d_episode.episode_return is then
 * (float)(centi / 100.0 + bump_count * crash_penalty).  It equals the f64 sum of the episode's rewards up to f64 and
 * f32 rounding when every parameter except crash_penalty is a multiple of 0.01 (true for the reference's); in general
 *     |episode_return - sum of rewards| <= 0.005 * (5 * length + 2) + 2^-24 * |episode_return| + 1e-3
 * (at most five rounded terms a step, plus the finish and truncation terms).  The accumulator saturates at the int32
 * limits instead of wrapping; only an env stepped on past done with auto_reset = 0 can reach them (about 2.3e5 steps
 * at the defaults), since every accepted parameter set keeps one episode within them.
 *
 * nav3d_set_reward_params checks, and fails with NAV3D_ERR_UNSUPPORTED (nav3d_last_error names the rule) for:
 *   - saturation: the visit count of the agent's cell saturates at 255, so the set must give the same
 *     min(count * revisit_unit, revisit_cap) for every count past 255: revisit_unit == 0, or revisit_unit > 0 and
 *     255.0 * revisit_unit >= revisit_cap (in f64);
 *   - overflow: 65535 * M + |c(finish_bonus)| + |c(truncation_penalty)| must fit an int32, where c(v) is a term in
 *     1/100 units as above and M, the largest |cents| of one step, is |c(step_cost)| + max(|c(min(revisit_unit,
 *     revisit_cap))|, |c(min(255 * revisit_unit, revisit_cap))|) + |c(near_wall_bonus)| + max(|c(repeat_bonus)|,
 *     |c(reverse_penalty)|) + |c(explore_bonus)|.
 * A value that is not finite or exceeds 1e6 in magnitude gives NAV3D_ERR_INVALID.  A rejected set leaves the engine's
 * parameters as they were. */
typedef struct {
    double step_cost;             /* -0.05  :175 */
    double revisit_unit;          /*  0.02  :179 */
    double revisit_cap;           /*  0.5   :180 */
    double crash_penalty;         /* -2.0   :28, :187 (same value as nav3d_config.crash_penalty) */
    double near_wall_bonus;       /*  0.15  :193 */
    double repeat_bonus;          /*  0.05  :199 */
    double reverse_penalty;       /*  0.5   :203 (subtracted) */
    double explore_bonus;         /*  1.0   :209 */
    double finish_bonus;          /* 100.0  :215 */
    double truncation_penalty;    /* -5.0   :221 */
} nav3d_reward_params;

/* Written by nav3d_step only for envs whose episode ended in that step (Monitor's info["episode"] plus the
 * attributes train/evaluate_grid.py:216-218 reads). 32 bytes. */
typedef struct {
    float episode_return;         /* sum of rewards of the finished episode */
    int32_t length;               /* step_count at the end */
    int32_t bumps;                /* bump_count */
    int32_t visited;              /* visited_count */
    int32_t total_free;           /* total_free_cells of the finished room */
    int32_t room;                 /* room index of the finished episode */
    int32_t terminated;           /* 1 if >= 84 % explored (CubicEnv) / goal reached (simpleEnv) */
    int32_t truncated;
} nav3d_episode;

const char *nav3d_last_error(void);
int nav3d_abi_version(void);

/* GridAgent.__init__ (envs/CubicEnv.py:17-74).  Allocates nothing per room yet. */
int nav3d_create(const nav3d_config *cfg, nav3d_engine **out);
void nav3d_destroy(nav3d_engine *e);

void nav3d_reward_params_default(nav3d_reward_params *out);
/* Takes effect from the next launch on; may be called at any time, mid-episode too (host-side copy, no device work).
 * The parameters are copied into each kernel's launch arguments, so a CUDA graph captured before this call keeps
 * replaying with the values it captured: capture the graph again after changing them.  Env-state blobs hold no reward
 * parameters: a loaded env continues with those of the engine it is loaded into.  CubicEnv only (NAV3D_ERR_UNSUPPORTED
 * for simpleEnv).  The accepted sets are described at nav3d_reward_params. */
int nav3d_set_reward_params(nav3d_engine *e, const nav3d_reward_params *params);

/* The room table: replaces the per-reset text parse + free-cell scan of load_room (envs/CubicEnv.py:402-459).
 * Dense grids are uploaded once; a CUDA kernel packs each room into bit-packed occupancy words (three orientations)
 * and builds the ordered free-cell list; per-env knowledge storage is sized for the largest room.
 * After this call the envs must be reset before they are stepped: nav3d_step / nav3d_step_host / nav3d_rollout_random
 * fail with NAV3D_ERR_INVALID until nav3d_reset has been called (the reference raises AttributeError for step-before-
 * reset); an env that a partial reset left out only bumps in place until it is reset. */
int nav3d_load_rooms(nav3d_engine *e, int32_t n_rooms, const nav3d_room_desc *rooms);
/* out6 = width, depth, height, total_free_cells (= max_steps, CubicEnv.py:459), n_wall_cells, reserved.  Synchronises. */
int nav3d_room_info(nav3d_engine *e, int32_t room, int32_t *out6);
/* HOST out: the k-th free interior cell of `room` as x,y,z (possible_start_pose[k], CubicEnv.py:450-457). Synchronises. */
int nav3d_room_free_cell(nav3d_engine *e, int32_t room, int32_t k, int32_t *xyz);
int nav3d_obs_dim(const nav3d_engine *e);
int nav3d_num_envs(const nav3d_engine *e);
int nav3d_lanes_per_env(const nav3d_engine *e);

/* GridAgent.reset (envs/CubicEnv.py:77-108) for a set of envs.
 *   env_ids : DEVICE int32[n] or NULL = envs 0..n-1 (then n must be <= n_envs); the listed ids must be distinct (two
 *             resets of one env in one call race on its record and knowledge)
 *   picks   : DEVICE int32[n][2] = (room index, k-th free cell) per listed env — the two random.choice draws of
 *             load_room (:407, :462) — for a NAV3D_ENV_SIMPLE engine int32[n][3]: the third column is the index of the goal in the
 *             same free-cell list (envs/simpleEnv.py:419-426) — or NULL = draw them from the env's Philox reset stream.
 *             A room with a usable "Start position" starts there whatever k says.
 *   obs     : DEVICE f32[n_envs][obs_dim]; rows of the listed envs are written; may be NULL */
int nav3d_reset(nav3d_engine *e, const int32_t *env_ids, int32_t n, const int32_t *picks, float *obs, void *stream);

/* GridAgent.step (envs/CubicEnv.py:110-132) for all envs of the engine, plus — when auto_reset — the
 * SubprocVecEnv worker's "if done: stash terminal_observation, reset" (SURVEY §8b B2).
 *   actions      : DEVICE int64[n_envs], values 0..5
 *   obs          : DEVICE f32[n_envs][obs_dim], 16-byte aligned (a [t,:,:] slice of a rollout buffer is fine)
 *   reward       : DEVICE f32[n_envs]  (the f64 reward of compute_reward rounded to f32, as SB3 stores it)
 *   reward64     : DEVICE f64[n_envs] or NULL
 *   terminated, truncated : DEVICE u8[n_envs]
 *   terminal_obs : DEVICE f32[n_envs][obs_dim] or NULL; written only for envs that were auto-reset
 *   episodes     : DEVICE nav3d_episode[n_envs] or NULL; written only for envs whose episode ended */
int nav3d_step(nav3d_engine *e, const int64_t *actions, float *obs, float *reward, double *reward64,
               uint8_t *terminated, uint8_t *truncated, float *terminal_obs, nav3d_episode *episodes, void *stream);

/* Same step through HOST buffers: the call a CPU-side trainer (SB3's VecEnv.step_wait, Grid_Train.py:228) makes.
 * Copies actions host->device, steps, copies obs/reward/terminated/truncated device->host and waits for them.  Large
 * batches run as a four-chunk pipeline on two internal streams (upload + step of a chunk overlap the download of the
 * previous one); pinned (page-locked) host buffers are needed for the copies to be asynchronous. */
int nav3d_step_host(nav3d_engine *e, const int64_t *actions, float *obs, float *reward, uint8_t *terminated,
                    uint8_t *truncated);

/* T fused steps with uniform random actions from the env's Philox action stream (indices t0 .. t0+T-1):
 * the "synthetic random-action rollout" of BASELINE.json.  One launch; each env's steps run back to back with its record
 * in registers, and every step does the full work of nav3d_step (marking, window gather, reward, auto-reset).
 *   obs    : DEVICE f32[T][n_envs][obs_dim] or NULL (then only the last observation is written, to obs_last)
 *   obs_last: DEVICE f32[n_envs][obs_dim] or NULL
 *   reward : DEVICE f32[T][n_envs] or NULL;  done : DEVICE u8[T][n_envs] or NULL (terminated | truncated)
 *   actions_out : DEVICE u8[T][n_envs] or NULL */
int nav3d_rollout_random(nav3d_engine *e, int32_t T, uint32_t t0, float *obs, float *obs_last, float *reward,
                         uint8_t *done, uint8_t *actions_out, void *stream);

/* T fused steps of every env with CALLER-SUPPLIED actions: the same work, outputs and auto-resets as T successive
 * nav3d_step calls with the rows of `actions`, in one launch (record in registers, knowledge lines on chip across steps).
 * Every byte it writes, and the engine state it leaves (nav3d_get_state, nav3d_get_grid, nav3d_save_envs blobs), equal
 * those of the T nav3d_step calls; rows those calls would leave untouched are left untouched.
 *   actions      : DEVICE u8[T][n_envs] (required); values > 5 act as 5, as nav3d_step clamps.  nav3d_rollout_random's
 *                  actions_out is in this format, so a random rollout can be replayed as it is.
 *   obs          : DEVICE f32[T][n_envs][80] or NULL;  obs_last : DEVICE f32[n_envs][80] or NULL (one of them required;
 *                  with obs == NULL only the last step's rows are formed, as in nav3d_rollout_random)
 *   reward       : DEVICE f32[T][n_envs] or NULL;   reward64 : DEVICE f64[T][n_envs] or NULL
 *   terminated, truncated : DEVICE u8[T][n_envs] or NULL
 *   terminal_obs : DEVICE f32[T][n_envs][80] or NULL; row [t][i] written only if env i auto-reset in step t
 *   episodes     : DEVICE nav3d_episode[T][n_envs] or NULL; row [t][i] written only if env i's episode ended in step t
 * obs / obs_last / terminal_obs 16-byte aligned.  CubicEnv only (NAV3D_ERR_UNSUPPORTED for simpleEnv, as
 * nav3d_rollout_random).  The arguments are checked in this order before the engine is: T >= 0, actions, obs / obs_last,
 * alignment.  T == 0 does nothing.  Asynchronous, no allocation, no synchronisation: capturable in a CUDA graph. */
int nav3d_rollout_actions(nav3d_engine *e, int32_t T, const uint8_t *actions, float *obs, float *obs_last,
                          float *reward, double *reward64, uint8_t *terminated, uint8_t *truncated,
                          float *terminal_obs, nav3d_episode *episodes, void *stream);

/* Integer state of every env (attributes read by the reference's callers: get_position CubicEnv.py:399-400,
 * visited_count/bump_count/done evaluate_grid.py:216-218, ...).  DEVICE int32[n_envs][NAV3D_STATE_INTS]:
 *  0 x  1 y  2 z  3 facing  4 visited_count  5 bump_count  6 step_count  7 near_wall  8 was_near_wall  9 last_bump
 * 10 done  11 cells_insight_down  12 last_action  13 room index  14 episode number  15 return so far, in 1/100 units,
 *    excluding crash penalties; CubicEnv: saturating at the int32 limits (see nav3d_reward_params) */
int nav3d_get_state(nav3d_engine *e, int32_t *state, void *stream);
/* self.internal_grid of one env (CubicEnv.py:84-85) rebuilt from the packed representation, DEVICE int16
 * [width][depth][height] of the env's current room (C order).   Visit counters saturate at 255. */
int nav3d_get_grid(nav3d_engine *e, int32_t env, int16_t *grid, void *stream);

/* Checkpoint / restore of the complete mutable engine state (scalars + knowledge grids), HOST buffers. */
size_t nav3d_snapshot_bytes(const nav3d_engine *e);
int nav3d_snapshot(nav3d_engine *e, void *host_buf, size_t bytes);
int nav3d_restore(nav3d_engine *e, const void *host_buf, size_t bytes);

/* ---- env-state blobs: save the complete state of listed envs on the device and load it back, into the same envs or into
 * others (ALE's cloneState / restoreState, per env).  Go-Explore-style archives, branching (one blob loaded into k envs),
 * evaluation from fixed mid-episode states.
 *
 * A blob is nav3d_env_state_bytes bytes, 16-byte aligned, in caller-owned DEVICE memory; blob i of a call is at
 * blobs + i * nav3d_env_state_bytes.  It holds a header (magic, format version, engine signature, room index, live byte
 * counts), the env's 32-byte record (position, counters, episode number, return so far, ...), its observation row and its
 * knowledge volume.  Only the live part of the knowledge is written — that of the env's current room — so a save of envs
 * in small rooms moves little even in an engine sized for a large one; bytes past the live parts are left as they were.
 * Blobs are plain bytes: they may be copied, duplicated, moved to another device or written to a file.
 *
 * The engine signature hashes the env kind, local_map_length, the per-env block size and the room table (each room's dims,
 * wall code, grid and start position).  A blob loads into any engine with the same signature: lanes_per_env, seed, env_id0,
 * n_envs, auto_reset and the reward parameters may differ.
 *
 * Observations: obs[68..70] of a CubicEnv row are the PREVIOUS step's last_action, was_near_wall and last_bump, which the
 * record no longer holds, so the row cannot be recomputed from it.  nav3d_save_envs therefore copies each listed env's row
 * out of `obs`, which must be the observation array the last nav3d_step / nav3d_reset / nav3d_load_envs wrote for that
 * env, and nav3d_load_envs writes the row back.
 *
 * Semantics: a loaded env continues exactly as the saved env would have, with one exception: randomness stays keyed by
 * the DESTINATION — its global id (env_id0 + index) and the engine seed — at the blob's episode counter.  Loading a blob
 * back into the env it came from replays that env bit for bit, its later auto-resets included; a blob loaded into another
 * env is identical until that env's next reset, which draws from the destination's Philox reset stream.
 *
 * Both calls are asynchronous on `stream`: no synchronisation, no allocation, no host copy, so they can be captured in a
 * CUDA graph.  Both take env_ids = DEVICE int32[n] or NULL = envs 0..n-1 (then n <= n_envs). */

/* Bytes of one env-state blob of this engine (fixed once rooms are loaded; 0 before). */
size_t nav3d_env_state_bytes(const nav3d_engine *e);
/* Copy the complete state of the listed envs into blobs[i] (DEVICE, n * nav3d_env_state_bytes).
 *   obs : DEVICE f32[n_envs][obs_dim]: the caller's CURRENT observation of every env (required; see above)
 * An env id outside 0..n_envs-1 gets a blob with an invalid magic, which every load rejects (status 2).  Env ids may
 * repeat.  Fails with NAV3D_ERR_INVALID until the envs have been reset (or restored / loaded). */
int nav3d_save_envs(nav3d_engine *e, const int32_t *env_ids, int32_t n, const float *obs, void *blobs, void *stream);
/* Overwrite the listed envs with blobs[i] and write their observation rows into obs (DEVICE f32[n_envs][obs_dim]).
 *   status : DEVICE u8[n] or NULL: 0 loaded, 1 env id out of range, 2 blob not valid for this engine (env untouched)
 * Every blob's header (magic, version, signature, room index < n_rooms, live sizes) is checked before anything of its env
 * is written.  The listed env ids must be distinct; blobs may repeat (loading one blob into many envs is the clone).
 * Counts as a reset for the step-before-reset check, as nav3d_restore does. */
int nav3d_load_envs(nav3d_engine *e, const int32_t *env_ids, int32_t n, const void *blobs, float *obs,
                    uint8_t *status, void *stream);

/* ---- rollout-loop kernels of the LSTM-PPO trainer (SURVEY §8f row 1).  Engine-free: they run on the CUDA device that is
 * current on the calling thread; all buffers are DEVICE pointers; asynchronous on `stream`.  They replace, in the
 * reference's third-party stack (sb3-contrib RecurrentPPO driven by train/Grid_Train.py:198-228), the per-step
 * `distribution.get_actions()/log_prob()` and `RecurrentRolloutBuffer.compute_returns_and_advantage`. ---- */

/* Categorical sampling from policy logits f32[n][n_actions] (row-major).  u = (word0 >> 8) / 2^24, where word0 is word 0
 * of Philox4x32-10 with counter = (env_id0 + i, step + *step_offset, 0, 0x504f4c49) (both sums mod 2^32) and the key of
 * `seed`, so u lies in [0, 1 - 2^-24]; action = first k with cumsum(softmax)[k] > u.  step_offset: DEVICE u32[1] or
 * NULL (= 0) — a counter in device memory, so that a CUDA graph that captured a whole rollout draws fresh numbers on
 * every replay.
 * A logits row may hold -inf entries (masked actions) if at least one entry is finite: masked actions are never drawn
 * and add 0 to the entropy.  A row containing +inf or NaN gives undefined output.
 * greedy != 0: argmax instead (SB3's deterministic=True, train/evaluate_grid.py:186-191).
 *   actions : int64[n] (directly usable by nav3d_step)   log_prob : f32[n] or NULL   entropy : f32[n] or NULL */
int nav3d_sample_actions(const float *logits, int32_t n, int32_t n_actions, uint64_t seed, uint32_t env_id0,
                         uint32_t step, const uint32_t *step_offset, int32_t greedy, int64_t *actions, float *log_prob,
                         float *entropy, void *stream);

/* GAE(lambda) over a time-major rollout: rewards, values f32[T][n]; episode_starts u8[T][n] (1 = step t is the first of
 * an episode); last_values f32[n] = V(s_T); last_dones u8[n] = the episode ended at step T-1.
 *   A_t = delta_t + gamma*lambda*(1-start_{t+1})*A_{t+1},  delta_t = r_t + gamma*V_{t+1}*(1-start_{t+1}) - V_t
 *   advantages, returns (= A + V) : f32[T][n] */
int nav3d_gae(const float *rewards, const float *values, const uint8_t *episode_starts, const float *last_values,
              const uint8_t *last_dones, float gamma, float gae_lambda, int32_t T, int32_t n, float *advantages,
              float *returns, void *stream);

/* One-layer LSTM over a sequence minibatch with episode-start resets (the PPO update's recurrent pass).  Replaces the
 * `nn.LSTM` calls of sb3-contrib's RecurrentActorCriticPolicy._process_sequence inside RecurrentPPO.train()
 * (train/Grid_Train.py:228), which cut the sequence at every reset.  torch weight layout: w_ih f32[4H][F], w_hh f32[4H][H],
 * b_ih, b_hh f32[4H], gate order i,f,g,o.  Row-major, time-major buffers; the recurrent GEMMs are cuBLAS calls
 * (tf32 != 0: TF32 tensor-op math), everything else one fused kernel per timestep.
 *   x f32[S][B][F]; h0, c0 f32[B][H]; starts u8[S][B] (1 = the state entering step t is zeroed)
 *   out: gates f32[S][B][4H] (activated i,f,g,o, kept for backward), h_in f32[S][B][H] (masked state entering each step),
 *        h_all, c_all f32[S][B][H] (h_all is the layer output; the final state is row S-1 of h_all / c_all) */
/* Creates the cuBLAS handle + workspace the two calls below use on `stream` (they do it lazily otherwise).  Call it BEFORE a
 * CUDA-graph capture on that stream begins: handle creation allocates, which a capture forbids; afterwards
 * nav3d_lstm_forward / nav3d_lstm_backward are capturable on it. */
int nav3d_lstm_prepare(void *stream);
int nav3d_lstm_forward(const float *x, const float *w_ih, const float *w_hh, const float *b_ih, const float *b_hh,
                       const float *h0, const float *c0, const uint8_t *starts, int32_t S, int32_t B, int32_t F, int32_t H,
                       int32_t tf32, float *gates, float *h_in, float *h_all, float *c_all, void *stream);
/* Backward of the above for a loss that depends on h_all only: dh_all f32[S][B][H] in; `gates` is overwritten with the
 * gradients w.r.t. the gate pre-activations; out dw_ih f32[4H][F], dw_hh f32[4H][H], db f32[4H] (gradient of b_ih and of
 * b_hh alike).  scratch: f32[2*B*H + S*B].  No gradient is produced for x, h0 or c0 (observations and carried states are
 * constants of the PPO update). */
int nav3d_lstm_backward(const float *x, const float *w_hh, const float *c0, const uint8_t *starts, const float *h_in,
                        const float *c_all, float *gates, const float *dh_all, int32_t S, int32_t B, int32_t F, int32_t H,
                        int32_t tf32, float *dw_ih, float *dw_hh, float *db, float *scratch, void *stream);

/* Number of CUDA kernels this library has launched since the engine was created (bench.py's gpu_launches). */
uint64_t nav3d_launch_count(const nav3d_engine *e);
/* Bytes of device memory the engine holds. */
size_t nav3d_device_bytes(const nav3d_engine *e);

#ifdef __cplusplus
}
#endif
#endif /* NAV3D_H */

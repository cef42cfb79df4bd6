// nav3d_train.cu — the small per-env kernels of the rollout loop that sit between the env step and the torch GEMMs of the
// LSTM-PPO trainer (SURVEY §8f row 1): categorical action sampling from the policy logits with the engine's counter-based
// Philox streams, and the generalised-advantage backward scan.  Both are per-env streaming passes (HBM-bound, no
// contraction): one thread per env, time-major [T][N] buffers so that every load and store of a warp is one coalesced run.
//
// What they replace in the reference's stack (third-party stable-baselines3 / sb3-contrib, un-vendored, un-pinned):
//   * RecurrentPPO.collect_rollouts: `distribution.get_actions()` + `distribution.log_prob(actions)` per step
//     (called from train/Grid_Train.py:228 `model.learn`)
//   * RecurrentRolloutBuffer.compute_returns_and_advantage (GAE(lambda), gamma = 0.99, gae_lambda = 0.95 at
//     train/Grid_Train.py:84-87)
#include "nav3d_core.cuh"
#include "../../include/nav3d.h"

#include <string>

using namespace nav3d;

namespace {

constexpr uint32_t kStreamPolicy = 0x504f4c49u;   // "POLI": counter = (global_env_id, step index, 0, tag)

// One thread per env.  Inverse-CDF sampling on softmax(logits) with u = (Philox word >> 8) / 2^24; the same pass gives
// log pi(a|s) and the entropy, so the rollout needs no second softmax.  A row may mask actions with -inf as long as one
// entry is finite: masked actions get weight 0, are never drawn and add 0 to the entropy.
template <bool GREEDY>
__global__ void __launch_bounds__(256) sample_actions_kernel(const float *__restrict__ logits, int N, int A,
                                                             uint32_t env_id0, uint32_t step,
                                                             const uint32_t *__restrict__ step_offset, uint32_t seed_lo,
                                                             uint32_t seed_hi, long long *__restrict__ actions,
                                                             float *__restrict__ log_prob, float *__restrict__ entropy) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const float *row = logits + (long long)n * A;
    float mx = row[0];
    int arg = 0;
    for (int k = 1; k < A; k++) {
        const float v = row[k];
        if (v > mx) { mx = v; arg = k; }          // first maximum, like torch.argmax
    }
    float sum = 0.f;
    for (int k = 0; k < A; k++) sum += expf(row[k] - mx);
    const float lse = logf(sum);
    int a = arg;
    if (!GREEDY) {
        uint32_t u0, u1;
        // step_offset lives in device memory so that a CUDA graph of a whole rollout can be replayed with fresh draws
        const uint32_t idx = step + (step_offset ? *step_offset : 0u);
        philox4x32_10(env_id0 + (uint32_t)n, idx, 0u, kStreamPolicy, seed_lo, seed_hi, u0, u1);
        // u = top 24 bits / 2^24 is exact in fp32 and at most 1 - 2^-24, so target < sum, which is the final acc: the walk
        // always stops inside the loop, on a term with nonzero weight.  ((float)u0 / 2^32 rounds to 1.0 for the top 128
        // words, and the walk then fell through to A - 1 whatever its weight.)
        const float u = (float)(u0 >> 8) * 0x1p-24f;
        const float target = u * sum;
        float acc = 0.f;
        a = A - 1;
        for (int k = 0; k < A; k++) {
            acc += expf(row[k] - mx);
            if (target < acc) { a = k; break; }
        }
    }
    actions[n] = a;
    if (log_prob) log_prob[n] = row[a] - mx - lse;
    if (entropy) {
        float h = 0.f;
        for (int k = 0; k < A; k++) {
            const float lp = row[k] - mx - lse;
            const float p = expf(lp);
            if (p > 0.f) h -= p * lp;                // p = 0 (a -inf logit) adds 0, not 0 * -inf = NaN
        }
        entropy[n] = h;
    }
}

// GAE(lambda) backward scan, one thread per env:
//   delta_t = r_t + gamma * V_{t+1} * (1 - start_{t+1}) - V_t ;  A_t = delta_t + gamma * lambda * (1 - start_{t+1}) * A_{t+1}
// with V_T = last_values, start_T = last_dones; returns = A + V.
__global__ void __launch_bounds__(256) gae_kernel(const float *__restrict__ rewards, const float *__restrict__ values,
                                                  const uint8_t *__restrict__ starts, const float *__restrict__ last_values,
                                                  const uint8_t *__restrict__ last_dones, float gamma, float lam, int T,
                                                  int N, float *__restrict__ adv, float *__restrict__ ret) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    float next_v = last_values[n];
    float next_nt = last_dones[n] ? 0.f : 1.f;
    float gae = 0.f;
#pragma unroll 4
    for (int t = T - 1; t >= 0; t--) {
        const long long i = (long long)t * N + n;
        const float r = rewards[i], v = values[i];
        const float st = starts[i] ? 0.f : 1.f;        // becomes next_nt of step t-1
        const float delta = r + gamma * next_v * next_nt - v;
        gae = delta + gamma * lam * next_nt * gae;
        adv[i] = gae;
        ret[i] = gae + v;
        next_v = v;
        next_nt = st;
    }
}

}  // namespace

namespace nav3d { int fail_with(int code, const std::string &msg); }   // nav3d_engine.cu: sets nav3d_last_error()
static int train_fail(int code, const std::string &msg) { return nav3d::fail_with(code, msg); }

extern "C" {

int nav3d_sample_actions(const float *logits, int32_t n, int32_t n_actions, uint64_t seed, uint32_t env_id0,
                         uint32_t step, const uint32_t *step_offset, int32_t greedy, int64_t *actions, float *log_prob,
                         float *entropy, void *stream) {
    if (!logits || !actions) return train_fail(NAV3D_ERR_INVALID, "logits and actions are required");
    if (n < 0 || n_actions < 1 || n_actions > 1024) return train_fail(NAV3D_ERR_INVALID, "bad n / n_actions");
    if (n == 0) return NAV3D_OK;
    cudaStream_t s = (cudaStream_t)stream;
    const unsigned grid = (unsigned)((n + 255) / 256);
    long long *a = reinterpret_cast<long long *>(actions);
    if (greedy)
        sample_actions_kernel<true><<<grid, 256, 0, s>>>(logits, n, n_actions, env_id0, step, step_offset, (uint32_t)seed,
                                                         (uint32_t)(seed >> 32), a, log_prob, entropy);
    else
        sample_actions_kernel<false><<<grid, 256, 0, s>>>(logits, n, n_actions, env_id0, step, step_offset, (uint32_t)seed,
                                                          (uint32_t)(seed >> 32), a, log_prob, entropy);
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return train_fail(NAV3D_ERR_CUDA, std::string("nav3d_sample_actions: ") + cudaGetErrorString(err));
    return NAV3D_OK;
}

int nav3d_gae(const float *rewards, const float *values, const uint8_t *episode_starts, const float *last_values,
              const uint8_t *last_dones, float gamma, float gae_lambda, int32_t T, int32_t n, float *advantages,
              float *returns, void *stream) {
    if (!rewards || !values || !episode_starts || !last_values || !last_dones || !advantages || !returns)
        return train_fail(NAV3D_ERR_INVALID, "nav3d_gae: NULL buffer");
    if (T < 0 || n < 0) return train_fail(NAV3D_ERR_INVALID, "nav3d_gae: negative size");
    if (T == 0 || n == 0) return NAV3D_OK;
    gae_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(rewards, values, episode_starts, last_values,
                                                                            last_dones, gamma, gae_lambda, T, n,
                                                                            advantages, returns);
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return train_fail(NAV3D_ERR_CUDA, std::string("nav3d_gae: ") + cudaGetErrorString(err));
    return NAV3D_OK;
}

}  // extern "C"

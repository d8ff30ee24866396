// replay.cu - device replay buffer for off-policy learners (SB3 ReplayBuffer / OffPolicyAlgorithm._store_transition
// semantics, restated in tests/test_gpu_replay.py; deviations in DESIGN.md 5).
//
// A ring of `rows` rows x N envs in HBM.  Observations are kept as planes, one (P, ld) block per row, laid out like
// the env's own S planes, so that storing a step is P coalesced plane copies: inserts (N transitions per step) are
// the bulk traffic, a gradient step samples a few thousand.  The sampler gathers one transition per thread and
// over-fetches (a 32-byte sector per 8-byte element).
//
// pos, full and the sample-call counter live in device memory (sdcgym_replay.counters) and are advanced by
// stream-ordered one-thread kernels, never by the host: a CUDA graph of collect + sample writes fresh rows and draws
// fresh indices on every replay.
//
// Built like vecnorm.cu, with FMA contraction allowed: the normalisation goes through normalize.cuh, whose roundings
// are all explicit, so the sampler's normalised values are bit-identical to sdcgym_vecnorm_apply / _reward.
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/sdcgym.h"
#include "normalize.cuh"
#include "replay_index.cuh"

namespace sdcgym {

constexpr int kReplayThreads = 256;
constexpr int kReplayMaxPlanes = 4 * SDCGYM_MAX_M;

// row `pos` of the observations: the planes the action is about to be taken on (before the step overwrites them)
__global__ void __launch_bounds__(kReplayThreads) replay_store_obs_kernel(const sdcgym_replay rb,
                                                                          const double* __restrict__ S, int64_t s_ld) {
    const int64_t pos = rb.counters[0];
    const int p = blockIdx.y;
    double* dst = rb.obs + (pos * rb.P + p) * rb.ld;
    const double* src = S + p * s_ld;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < rb.N; i += (int64_t)gridDim.x * blockDim.x)
        dst[i] = src[i];
}

// row `pos` of everything else, after the step.  blockIdx.y < P: next-observation plane y (the terminal plane for envs
// whose episode ended, the auto-reset state has already replaced S there); blockIdx.y == P: actions, reward, done.
__global__ void __launch_bounds__(kReplayThreads) replay_store_kernel(const sdcgym_replay rb, const double* __restrict__ S,
                                                                      const double* __restrict__ terminal, int64_t s_ld,
                                                                      const uint8_t* __restrict__ flags,
                                                                      const double* __restrict__ reward,
                                                                      const double* __restrict__ action,
                                                                      int64_t action_stride) {
    const int64_t pos = rb.counters[0];
    const int p = blockIdx.y;
    const int64_t i0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, step = (int64_t)gridDim.x * blockDim.x;
    if (p < rb.P) {
        double* dst = rb.next_obs + (pos * rb.P + p) * rb.ld;
        const double* s = S + p * s_ld;
        const double* t = terminal ? terminal + p * s_ld : nullptr;
        for (int64_t i = i0; i < rb.N; i += step) dst[i] = (t && (flags[i] & SDCGYM_FLAG_DONE)) ? t[i] : s[i];
        return;
    }
    // one env per thread: a warp's A loads / stores cover 32 * A contiguous doubles, merged in L1 / L2
    const int A = rb.A;
    double* da = rb.actions + pos * rb.N * A;
    for (int64_t i = i0; i < rb.N; i += step) {
        for (int k = 0; k < A; k++) da[i * A + k] = action[i * action_stride + k];
        rb.rewards[pos * rb.N + i] = reward[i];
        rb.dones[pos * rb.N + i] = flags[i] & SDCGYM_FLAG_DONE;
    }
}

__global__ void replay_advance_kernel(int64_t* counters, int64_t rows) {
    int64_t pos = counters[0] + 1;
    if (pos == rows) {
        pos = 0;
        counters[1] = 1;
    }
    counters[0] = pos;
}

__global__ void replay_count_call_kernel(int64_t* counters) { counters[2] += 1; }

// one sample per thread: indices from replay_index, gather, normalise (obs_mean == NULL: raw observations,
// ret_var == NULL: raw rewards).  Outputs: obs / next_obs planes [P][B], actions [B][A], rewards [B], dones [B].
__global__ void __launch_bounds__(kReplayThreads) replay_sample_kernel(
    const sdcgym_replay rb, int64_t B, const double* __restrict__ obs_mean, const double* __restrict__ obs_var,
    const double* __restrict__ ret_var, double eps, double clip_obs, double clip_reward, double* __restrict__ obs,
    double* __restrict__ next_obs, double* __restrict__ actions, double* __restrict__ rewards,
    double* __restrict__ dones) {
    __shared__ double s_mean[kReplayMaxPlanes], s_is[kReplayMaxPlanes];
    if (obs_mean && threadIdx.x < rb.P) {
        s_mean[threadIdx.x] = obs_mean[threadIdx.x];
        s_is[threadIdx.x] = norm_inv_std(obs_var[threadIdx.x], eps);
    }
    __syncthreads();
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= B) return;
    const int64_t* c = rb.counters;
    const uint32_t upper = (uint32_t)(c[1] ? rb.rows : c[0]);
    uint32_t row, env;
    replay_index(rb.seed, (uint32_t)c[2], (uint64_t)j, upper, (uint32_t)rb.N, &row, &env);
    const int64_t base = (int64_t)row * rb.P * rb.ld + env;
    for (int p = 0; p < rb.P; p++) {
        double x = rb.obs[base + p * rb.ld], y = rb.next_obs[base + p * rb.ld];
        if (obs_mean) {
            x = norm_obs(x, s_mean[p], s_is[p], clip_obs);
            y = norm_obs(y, s_mean[p], s_is[p], clip_obs);
        }
        obs[p * B + j] = x;
        next_obs[p * B + j] = y;
    }
    const int64_t t = (int64_t)row * rb.N + env;
    for (int k = 0; k < rb.A; k++) actions[j * rb.A + k] = rb.actions[t * rb.A + k];
    double r = rb.rewards[t];
    if (ret_var) r = norm_reward(r, ret_var[0], eps, clip_reward);
    rewards[j] = r;
    dones[j] = (double)rb.dones[t];
}

static int replay_check(const sdcgym_replay* rb) {
    if (!rb) return SDCGYM_ENULL;
    if (rb->P < 1 || rb->P > kReplayMaxPlanes || rb->A < 1 || rb->rows < 1 || rb->N < 1 || rb->ld < rb->N)
        return SDCGYM_EINVAL;
    if (rb->rows > (int64_t)UINT32_MAX || rb->N > (int64_t)UINT32_MAX) return SDCGYM_EINVAL;  // 32-bit index draws
    if (!rb->obs || !rb->next_obs || !rb->actions || !rb->rewards || !rb->dones || !rb->counters) return SDCGYM_ENULL;
    return 0;
}

static unsigned replay_grid(int64_t n) {
    int64_t g = (n + kReplayThreads - 1) / kReplayThreads;
    return (unsigned)(g < 148 * 8 ? g : 148 * 8);
}

}  // namespace sdcgym

using namespace sdcgym;

extern "C" int sdcgym_replay_store_obs(const sdcgym_replay* rb, const double* S, int64_t s_ld, void* stream) {
    if (int rc = replay_check(rb)) return rc;
    if (s_ld < rb->N) return SDCGYM_EINVAL;
    if (!S) return SDCGYM_ENULL;
    replay_store_obs_kernel<<<dim3(replay_grid(rb->N), rb->P), kReplayThreads, 0, (cudaStream_t)stream>>>(*rb, S, s_ld);
    return (int)cudaGetLastError();
}

extern "C" int sdcgym_replay_store(const sdcgym_replay* rb, const double* S, const double* terminal, int64_t s_ld,
                                   const uint8_t* flags, const double* reward, const double* action,
                                   int64_t action_stride, void* stream) {
    if (int rc = replay_check(rb)) return rc;
    if (s_ld < rb->N || action_stride < rb->A) return SDCGYM_EINVAL;
    if (!S || !flags || !reward || !action) return SDCGYM_ENULL;
    cudaStream_t s = (cudaStream_t)stream;
    replay_store_kernel<<<dim3(replay_grid(rb->N), rb->P + 1), kReplayThreads, 0, s>>>(
        *rb, S, terminal, s_ld, flags, reward, action, action_stride);
    replay_advance_kernel<<<1, 1, 0, s>>>(rb->counters, rb->rows);
    return (int)cudaGetLastError();
}

extern "C" int sdcgym_replay_sample(const sdcgym_replay* rb, int64_t B, const double* obs_mean, const double* obs_var,
                                    const double* ret_var, double eps, double clip_obs, double clip_reward, double* obs,
                                    double* next_obs, double* actions, double* rewards, double* dones, void* stream) {
    if (int rc = replay_check(rb)) return rc;
    if (B < 0 || (uint64_t)B > (uint64_t)INT32_MAX * kReplayThreads) return SDCGYM_EINVAL;
    if (B == 0) return 0;
    if (!obs || !next_obs || !actions || !rewards || !dones || (obs_mean && !obs_var)) return SDCGYM_ENULL;
    cudaStream_t s = (cudaStream_t)stream;
    replay_sample_kernel<<<(unsigned)((B + kReplayThreads - 1) / kReplayThreads), kReplayThreads, 0, s>>>(
        *rb, B, obs_mean, obs_var, ret_var, eps, clip_obs, clip_reward, obs, next_obs, actions, rewards, dones);
    replay_count_call_kernel<<<1, 1, 0, s>>>(rb->counters);
    return (int)cudaGetLastError();
}

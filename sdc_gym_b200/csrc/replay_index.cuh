// replay_index.cuh - which stored transition replay sample j of sample call c draws (csrc/replay.cu), host and
// device.  sdc_gym_b200/replay.py restates it in numpy; tests/host_shim/replay_shim.cpp compiles it for the host.
//
// SB3's ReplayBuffer.sample draws batch_inds ~ U{0 .. upper-1} (upper = rows when the ring is full, else pos) and
// env_inds ~ U{0 .. n_envs-1} with replacement from numpy's global generator.  Here they come from the Philox
// stream of csrc/philox.cuh with
//   key     = (seed_lo, seed_hi)
//   counter = (j_lo, j_hi, c, kReplayTag)
// so a sample depends on (seed, c, j) only: a captured CUDA graph that advances the device-side call counter draws
// fresh indices on every replay.  kReplayTag is non-zero, and the lambda stream's 4th counter word is always 0, so
// the two streams never share a counter.
#pragma once
#include "philox.cuh"

namespace sdcgym {

constexpr uint32_t kReplayTag = 0x5250u;  // "RP"

SDCGYM_HD uint32_t mulhi32(uint32_t a, uint32_t b) { return (uint32_t)(((uint64_t)a * b) >> 32); }

// Lemire's multiply-high map of a uniform 32-bit word onto {0 .. n-1}: every value is hit by floor(2^32 / n) or
// ceil(2^32 / n) words, so the bias of a drawn row (env) is below upper / 2^32 (n_envs / 2^32) relative to its 1 / n
// share: 2.5e-4 at 2^20 envs, far below what a minibatch of a few thousand samples can resolve.
SDCGYM_HD void replay_index(uint64_t seed, uint32_t call, uint64_t j, uint32_t upper, uint32_t n_envs, uint32_t* row,
                            uint32_t* env) {
    const philox4 x = philox4x32_10((uint32_t)j, (uint32_t)(j >> 32), call, kReplayTag, (uint32_t)seed,
                                    (uint32_t)(seed >> 32));
    *row = mulhi32(x.v[0], upper);
    *env = mulhi32(x.v[1], n_envs);
}

}  // namespace sdcgym

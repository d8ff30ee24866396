// vecnorm.cu - device-side VecNormalize (SB3 semantics restated: RunningMeanStd with Chan's merge, clip to
// +-clip) over the observation planes and the reward/return planes, plus the ResidualLoss sweep.
//
// Reference call sites: utils/utils.py:295-312 (VecNormalize(env, norm_obs, norm_reward, gamma)),
// dp_playground.py:235-258 (ResidualLoss.take_step).  SB3 itself is third-party and not installed: its
// documented semantics are restated ("parity unpinned", DESIGN.md 2).  Complex observations are normalised on
// their re / im planes separately (SB3 on complex128 is ill-defined, SURVEY 8b(v)).
//
// All reductions use a fixed block count and a fixed summation tree: deterministic run to run.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <atomic>
#include <math_constants.h>

#include "../../include/sdcgym.h"
#include "bulk_copy.cuh"
#include "normalize.cuh"
#include "specrad.cuh"

namespace sdcgym {

constexpr int kAccThreads = 256;

__device__ __forceinline__ double2 block_sum2(double a, double b) {
    __shared__ double sa[kAccThreads / 32], sb[kAccThreads / 32];
    for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_down_sync(0xffffffffu, a, o);
        b += __shfl_down_sync(0xffffffffu, b, o);
    }
    if ((threadIdx.x & 31) == 0) {
        sa[threadIdx.x >> 5] = a;
        sb[threadIdx.x >> 5] = b;
    }
    __syncthreads();
    a = (threadIdx.x < kAccThreads / 32) ? sa[threadIdx.x] : 0.0;
    b = (threadIdx.x < kAccThreads / 32) ? sb[threadIdx.x] : 0.0;
    if (threadIdx.x < 32)
        for (int o = 16; o > 0; o >>= 1) {
            a += __shfl_down_sync(0xffffffffu, a, o);
            b += __shfl_down_sync(0xffffffffu, b, o);
        }
    __syncthreads();
    return make_double2(a, b);
}

// The statistics arithmetic is spelled with explicit roundings so that every kernel that performs it (the
// three-kernel sequence and the fused single-launch update) produces the same bits whatever the compiler contracts.
__device__ __forceinline__ void acc_one(double x, double s, double& a, double& b) {
    const double d = __dsub_rn(x, s);
    a = __dadd_rn(a, d);
    b = __fma_rn(d, d, b);
}
__device__ __forceinline__ double advance_return(double ret, double gamma, double reward) {
    return __fma_rn(ret, gamma, reward);
}
// RunningMeanStd.update_from_moments with the batch given as shifted sums (shift = the running mean itself)
__device__ __forceinline__ void rms_merge_one(double n, double batch, double sa, double sb, double& mean, double& var) {
    const double d1 = __ddiv_rn(sa, batch);  // batch_mean - running mean
    const double d1sq = __dmul_rn(d1, d1);
    const double bvar = fmax(__dsub_rn(__ddiv_rn(sb, batch), d1sq), 0.0);  // population variance of the batch
    const double tot = __dadd_rn(n, batch);
    const double cross = __ddiv_rn(__dmul_rn(__dmul_rn(d1sq, n), batch), tot);
    const double m2 = __dadd_rn(__dadd_rn(__dmul_rn(var, n), __dmul_rn(bvar, batch)), cross);
    mean = __dadd_rn(mean, __ddiv_rn(__dmul_rn(d1, batch), tot));
    var = __ddiv_rn(m2, tot);
}

// RunningMeanStd.update_from_moments with the batch given as shifted sums (shift = the running mean itself)
__global__ void rms_merge_kernel(int P, double batch_count, const double* __restrict__ sums, double* __restrict__ mean,
                                 double* __restrict__ var, double* __restrict__ count) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    const double n = count[0];
    if (p < P && batch_count > 0) {
        double m = mean[p], v = var[p];
        rms_merge_one(n, batch_count, sums[p], sums[P + p], m, v);
        mean[p] = m;
        var[p] = v;
    }
    __syncthreads();
    if (blockIdx.x == 0 && threadIdx.x == 0 && batch_count > 0) count[1] = n + batch_count;  // committed by the host-side swap
}
__global__ void rms_commit_kernel(double* __restrict__ count) { count[0] = count[1]; }

// ---- single-rank fast path: accumulate + fold + merge in ONE launch ----------------------------------------------
// Same partial sums as acc_partial_kernel (stat_accumulate: same slices, same tree), then the block that finishes last
// folds the kStatBlocks partials of every plane in index order and applies the merge - bit-identical to the three-kernel
// sequence accumulate -> merge -> commit, without the three launches (a normalised sdc-v1 step of 2^20 envs is a
// 115 us kernel: five 2-7 us launches per statistic were a fifth of the step).
// RETURNS: the plane is the discounted return, advanced in the same pass: ret <- ret * gamma + reward.
//
// Several ranks (one process per GPU): the same launch also performs the all-reduce of the moment sums, over peer
// memory (NVLink / NVSwitch P2P stores into every rank's exchange region, include/sdcgym.h sdcgym_xchg) instead of an
// NCCL call between an accumulate and a merge kernel: the block that folds this rank's partial sums
//   1. stores its 2P + 1 numbers (shifted sums, shifted square sums, env count) into slot [parity][rank] of EVERY rank's
//      region, fences system-wide and raises flag [parity][rank] = seq there,
//   2. waits until the `world` flags of its own region show seq,
//   3. adds the slots in rank order (the same order on every rank: the normalisers stay bit-identical) and merges.
// Two parities: a rank can be at most one exchange ahead of a peer (it needs the peer's flag of the previous one).
struct XchgDev {
    int world, rank;
    unsigned long long seq;
    int stride;  // doubles per slot
    double* peer[SDCGYM_MAX_RANKS];  // exchange regions of all ranks (peer[rank] = the local one)
};
__device__ __forceinline__ double* xchg_slot(double* region, int world, int stride, int parity, int r) {
    return region + ((size_t)parity * world + r) * stride;
}
__device__ __forceinline__ unsigned long long* xchg_flags(double* region, int world, int stride, int parity) {
    return reinterpret_cast<unsigned long long*>(region + (size_t)2 * world * stride) + (size_t)parity * world;
}

// Wait for a peer's flag with a deadline (~20 s of SM clocks): a rank that never arrives (crashed process) must not
// leave this kernel spinning forever.  Returns false on timeout; the caller then poisons the statistics with NaN so the
// failure is visible in the very next normalised observation.
__device__ __forceinline__ bool xchg_wait(volatile unsigned long long* flag, unsigned long long seq) {
    const long long t0 = clock64();
    while (*flag != seq) {
        if (clock64() - t0 > 40000000000ll) return false;
    }
    return true;
}

// ---- the statistics pass -----------------------------------------------------------------------------------------
// One env per thread, planes in the inner loop: thread t of block b visits envs b*256 + t + k*(296*256) and, for each,
// kStatGroup planes at a time - the access pattern that streams the plane layout at the copy peak
// (tools/plane_stream_bench.cu: 21 planes in, 6.2-6.9 TB/s; the previous plane-per-block-row grid of 64 x P short-lived
// blocks reached 3.6).  296 blocks of 256 threads = exactly one resident wave (2 per SM) whatever the plane count; a
// block walks its envs once per plane group.  Plane index `nobs` (when `has_ret`) is the discounted return, advanced
// in the same pass: ret <- ret * gamma + reward.
// Fixed grid, fixed per-thread order, fixed block tree, partials folded in block order: deterministic, and the same
// bits from every kernel that calls stat_accumulate (the three-kernel sequence, the fused update, the in-kernel exchange).
#ifndef SDCGYM_STAT_UNROLL
#define SDCGYM_STAT_UNROLL 1
#endif
#ifndef SDCGYM_STAT_GROUP
#define SDCGYM_STAT_GROUP 7
#endif
constexpr int kStatBlocks = 296, kStatGroup = SDCGYM_STAT_GROUP, kStatUnroll = SDCGYM_STAT_UNROLL;

struct StatIn {
    int nobs, has_ret;        // observation planes X[nobs][ld]; optional return plane
    int64_t N, ld;
    const double* X;
    const double* shift_obs;  // [nobs] or nullptr (no shift)
    const double* reward;     // return plane: ret <- ret * gamma + reward
    double gamma;
    double* ret;
    const double* shift_ret;  // [1] or nullptr
};

// partial[(q * kStatBlocks + blockIdx.x) * 2 + {0, 1}] for every plane q: the block walks its envs once per group of
// kStatGroup planes (different planes each time: nothing is read twice)
__device__ __forceinline__ void stat_accumulate(const StatIn& in, double* __restrict__ partial) {
    const int planes = in.nobs + in.has_ret;
    constexpr int64_t stride = (int64_t)kStatBlocks * kAccThreads;
    // the shifts are read from shared memory where they are used: 2 x kStatGroup registers less per thread
    __shared__ double shift[4 * SDCGYM_MAX_M + 1];
    for (int q = threadIdx.x; q < planes; q += kAccThreads)
        shift[q] = (q < in.nobs) ? (in.shift_obs ? in.shift_obs[q] : 0.0) : (in.shift_ret ? in.shift_ret[0] : 0.0);
    __syncthreads();
    for (int q0 = 0; q0 < planes; q0 += kStatGroup) {
        double a[kStatGroup], b[kStatGroup];
#pragma unroll
        for (int j = 0; j < kStatGroup; j++) {
            a[j] = 0.0;
            b[j] = 0.0;
        }
        // kStatUnroll envs x kStatGroup planes of loads per round (predicated past the end), and the NEXT round's loads
        // are issued before this round's values are consumed (two register buffers): without that every round is an
        // exposed DRAM round trip (measured: time = bytes / 6 TB/s + rounds x ~1.3 us).  The return plane is advanced
        // and stored when its round is consumed (restrict pointers: the stores do not hold back the next loads).  The
        // accumulation itself stays in env order, so neither the unrolling nor the pipelining changes a single bit.
        const double* __restrict__ X = in.X;
        const double* __restrict__ reward = in.reward;
        double* __restrict__ ret = in.ret;
        const int jret = (in.has_ret && planes - 1 >= q0 && planes - 1 < q0 + kStatGroup) ? planes - 1 - q0 : -1;
        constexpr int64_t round = kStatUnroll * stride;
        auto load = [&](double (&v)[kStatUnroll][kStatGroup], double (&w)[kStatUnroll], int64_t i) {
#pragma unroll
            for (int k = 0; k < kStatUnroll; k++) {
                const int64_t e = i + k * stride;
#pragma unroll
                for (int j = 0; j < kStatGroup; j++) {
                    const int q = q0 + j;
                    v[k][j] = 0.0;
                    if (e < in.N) {
                        if (q < in.nobs) v[k][j] = X[(int64_t)q * in.ld + e];
                        else if (q < planes) v[k][j] = ret[e];
                    }
                }
                w[k] = (jret >= 0 && e < in.N) ? reward[e] : 0.0;
            }
        };
        auto consume = [&](const double (&v)[kStatUnroll][kStatGroup], const double (&w)[kStatUnroll], int64_t i) {
#pragma unroll
            for (int k = 0; k < kStatUnroll; k++) {
                const int64_t e = i + k * stride;
#pragma unroll
                for (int j = 0; j < kStatGroup; j++) {
                    if (q0 + j < planes && e < in.N) {
                        double x = v[k][j];
                        if (j == jret) {
                            x = advance_return(x, in.gamma, w[k]);
                            ret[e] = x;
                        }
                        acc_one(x, shift[q0 + j], a[j], b[j]);
                    }
                }
            }
        };
        double v0[kStatUnroll][kStatGroup], v1[kStatUnroll][kStatGroup], w0[kStatUnroll], w1[kStatUnroll];
        int64_t i = (int64_t)blockIdx.x * kAccThreads + threadIdx.x;
        load(v0, w0, i);
        while (i < in.N) {
            load(v1, w1, i + round);
            consume(v0, w0, i);
            i += round;
            if (i >= in.N) break;
            load(v0, w0, i + round);
            consume(v1, w1, i);
            i += round;
        }
#pragma unroll
        for (int j = 0; j < kStatGroup; j++) {
            const int q = q0 + j;
            if (q < planes) {  // (block-uniform)
                const double2 r = block_sum2(a[j], b[j]);
                if (threadIdx.x == 0) {
                    partial[((int64_t)q * kStatBlocks + blockIdx.x) * 2] = r.x;
                    partial[((int64_t)q * kStatBlocks + blockIdx.x) * 2 + 1] = r.y;
                }
            }
        }
    }
}
// ---- the same pass with the planes arriving by bulk asynchronous copies -------------------------------------------
// stat_accumulate issues its loads and then waits a DRAM round trip once per kStatUnroll envs: ~24 exposed round trips
// per block at 2^20 envs (57 us for 176 MB = 3.3 TB/s).  Here a block owns the same envs in the same order (tile k of
// block b = envs (b + 296 k) * 256 ...: thread t still sees b*256 + t + k*296*256), but the tiles of kStreamGroup
// planes x 256 envs (2 KB per plane) are fetched by cp.async.bulk into a ring of kStreamDepth shared-memory stages,
// completion on one mbarrier per stage; thread 0 re-arms a stage as soon as every thread has pulled its element out of
// it.  Same per-thread order, same block tree, same partial layout: bit-identical to stat_accumulate (tested), which
// still serves small batches, unaligned plane strides and the ragged last tile.
#ifndef SDCGYM_STAT_STREAM_GROUP
#define SDCGYM_STAT_STREAM_GROUP 11
#endif
#ifndef SDCGYM_STAT_STREAM_DEPTH
#define SDCGYM_STAT_STREAM_DEPTH 3
#endif
constexpr int kStreamGroup = SDCGYM_STAT_STREAM_GROUP, kStreamDepth = SDCGYM_STAT_STREAM_DEPTH;
constexpr int kStatTile = kAccThreads;                                  // envs per tile
constexpr int kStatStageBytes = (kStreamGroup + 1) * kStatTile * 8;     // (+1: the reward plane next to the return plane)
constexpr int kStatStreamSmem = kStreamDepth * kStatStageBytes;

__device__ __forceinline__ void stat_accumulate_stream(const StatIn& in, double* __restrict__ partial, unsigned char* ring,
                                                       unsigned long long* bars) {
    const int planes = in.nobs + in.has_ret;
    const int groups = (planes + kStreamGroup - 1) / kStreamGroup;
    const int64_t tiles = in.N / kStatTile;  // full tiles; the ragged rest is read directly by the block that owns it
    const int64_t mine = tiles > blockIdx.x ? (tiles - blockIdx.x + kStatBlocks - 1) / kStatBlocks : 0;
    const int64_t total = mine * groups;
    const int64_t tail_i = tiles * kStatTile + threadIdx.x;
    const bool own_tail = (tiles % kStatBlocks) == blockIdx.x && tail_i < in.N;
    if (threadIdx.x == 0) {
        for (int d = 0; d < kStreamDepth; d++) mbar_init(&bars[d], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    // warp 0: lane 0 arms stage n % depth, then lane j issues the copy of plane j of sequence element n = (group, k-th
    // own tile) - one thread issuing all the copies of a stage serialises them (measured: see profiles/README.md)
    auto issue = [&](int64_t n) {
        const int lane = threadIdx.x;
        const int g = (int)(n / mine);
        const int64_t e0 = (blockIdx.x + (n % mine) * kStatBlocks) * kStatTile;
        const int st = (int)(n % kStreamDepth), q0 = g * kStreamGroup;
        const int cnt = min(kStreamGroup, planes - q0);
        const bool with_ret = in.has_ret && q0 + cnt == planes;
        unsigned char* stage = ring + (size_t)st * kStatStageBytes;
        if (lane == 0) mbar_expect_tx(&bars[st], (unsigned)((cnt + (with_ret ? 1 : 0)) * kStatTile * 8));
        __syncwarp();
        if (lane < cnt) {
            const int q = q0 + lane;
            const double* src = (q < in.nobs) ? in.X + (int64_t)q * in.ld + e0 : in.ret + e0;
            bulk_g2s(stage + lane * kStatTile * 8, src, kStatTile * 8, &bars[st]);
        } else if (lane == kStreamGroup && with_ret) {
            bulk_g2s(stage + kStreamGroup * kStatTile * 8, in.reward + e0, kStatTile * 8, &bars[st]);
        }
    };
    static_assert(kStreamGroup < 32, "one lane of warp 0 per plane of a stage");
    if (threadIdx.x < 32)
        for (int64_t n = 0; n < kStreamDepth && n < total; n++) issue(n);
    int64_t n = 0;
    for (int g = 0; g < groups; g++) {
        const int q0 = g * kStreamGroup;
        double a[kStreamGroup], b[kStreamGroup], s[kStreamGroup];
#pragma unroll
        for (int j = 0; j < kStreamGroup; j++) {
            a[j] = 0.0;
            b[j] = 0.0;
            const int q = q0 + j;
            s[j] = 0.0;
            if (q < in.nobs) s[j] = in.shift_obs ? in.shift_obs[q] : 0.0;
            else if (q < planes) s[j] = in.shift_ret ? in.shift_ret[0] : 0.0;
        }
        const int jret = (in.has_ret && planes - 1 >= q0 && planes - 1 < q0 + kStreamGroup) ? planes - 1 - q0 : -1;
        for (int64_t k = 0; k < mine; k++, n++) {
            const int st = (int)(n % kStreamDepth);
            mbar_wait(&bars[st], (unsigned)((n / kStreamDepth) & 1));
            const double* stage = reinterpret_cast<const double*>(ring + (size_t)st * kStatStageBytes);
            double v[kStreamGroup + 1];
#pragma unroll
            for (int j = 0; j <= kStreamGroup; j++) v[j] = stage[j * kStatTile + threadIdx.x];
            __syncthreads();  // everybody has its element: the stage is free
            if (threadIdx.x < 32 && n + kStreamDepth < total) issue(n + kStreamDepth);
#pragma unroll
            for (int j = 0; j < kStreamGroup; j++) {
                if (q0 + j < planes) {
                    double x = v[j];
                    if (j == jret) {
                        x = advance_return(x, in.gamma, v[kStreamGroup]);
                        in.ret[(blockIdx.x + k * kStatBlocks) * kStatTile + threadIdx.x] = x;
                    }
                    acc_one(x, s[j], a[j], b[j]);
                }
            }
        }
        if (own_tail) {
#pragma unroll
            for (int j = 0; j < kStreamGroup; j++) {
                const int q = q0 + j;
                if (q < in.nobs) acc_one(in.X[(int64_t)q * in.ld + tail_i], s[j], a[j], b[j]);
                else if (q < planes) {
                    const double x = advance_return(in.ret[tail_i], in.gamma, in.reward[tail_i]);
                    in.ret[tail_i] = x;
                    acc_one(x, s[j], a[j], b[j]);
                }
            }
        }
#pragma unroll
        for (int j = 0; j < kStreamGroup; j++) {
            const int q = q0 + j;
            if (q < planes) {  // (block-uniform)
                const double2 r = block_sum2(a[j], b[j]);
                if (threadIdx.x == 0) {
                    partial[((int64_t)q * kStatBlocks + blockIdx.x) * 2] = r.x;
                    partial[((int64_t)q * kStatBlocks + blockIdx.x) * 2 + 1] = r.y;
                }
            }
        }
    }
}

// Fold the kStatBlocks partials of plane q: one warp per plane, lane l adds partials l, l + 32, ... in that order (all
// loads of a lane in flight together), then a fixed butterfly over the lanes.  (A single thread walking the 148
// partials is a chain of L2 round trips: 21 such threads were 40 us of a 55 us kernel.)  Every lane returns the sums.
__device__ __forceinline__ void stat_fold(const double* __restrict__ partial, int q, double& sa, double& sb) {
    const int lane = threadIdx.x & 31;
    constexpr int kPer = (kStatBlocks + 31) / 32;
    double va[kPer], vb[kPer];
#pragma unroll
    for (int r = 0; r < kPer; r++) {
        const int k = lane + 32 * r;
        va[r] = (k < kStatBlocks) ? __ldcg(&partial[((int64_t)q * kStatBlocks + k) * 2]) : 0.0;
        vb[r] = (k < kStatBlocks) ? __ldcg(&partial[((int64_t)q * kStatBlocks + k) * 2 + 1]) : 0.0;
    }
    sa = 0.0;
    sb = 0.0;
#pragma unroll
    for (int r = 0; r < kPer; r++) {
        sa += va[r];
        sb += vb[r];
    }
    for (int o = 16; o > 0; o >>= 1) {
        sa += __shfl_xor_sync(0xffffffffu, sa, o);
        sb += __shfl_xor_sync(0xffffffffu, sb, o);
    }
}

// the three-kernel sequence: partial sums, then the fold
template <bool STREAM>
__global__ void __launch_bounds__(kAccThreads, 2) acc_partial_kernel(const StatIn in, double* __restrict__ partial) {
    if constexpr (STREAM) {
        extern __shared__ __align__(128) unsigned char ring[];
        __shared__ __align__(8) unsigned long long bars[kStreamDepth];
        stat_accumulate_stream(in, partial, ring, bars);
    } else {
        stat_accumulate(in, partial);
    }
}
__global__ void __launch_bounds__(kAccThreads) acc_final_kernel(int P, const double* __restrict__ partial, double* __restrict__ out) {
    for (int p = threadIdx.x >> 5; p < P; p += kAccThreads / 32) {  // one warp per plane
        double a, b;
        stat_fold(partial, p, a, b);
        if ((threadIdx.x & 31) == 0) {
            out[p] = a;
            out[P + p] = b;
        }
    }
}

struct StatOut {
    double *omean, *ovar, *ocount, *osums;  // observation statistics (nobs planes), sums [2 nobs (+1)]
    double *rmean, *rvar, *rcount, *rsums;  // return statistics
};

// accumulate + fold + merge in ONE launch; DIST: with the all-reduce over peer memory in between (see above)
template <bool DIST, bool STREAM>
__global__ void __launch_bounds__(kAccThreads, 2) stat_update_kernel(const StatIn in, const StatOut out, double* __restrict__ partial,
                                                                  unsigned int* ticket, const XchgDev xc) {
    if constexpr (STREAM) {
        extern __shared__ __align__(128) unsigned char ring[];
        __shared__ __align__(8) unsigned long long bars[kStreamDepth];
        stat_accumulate_stream(in, partial, ring, bars);
    } else {
        stat_accumulate(in, partial);
    }
    __shared__ bool last;
    if (threadIdx.x == 0) {
        __threadfence();
        const unsigned int t = atomicAdd(ticket, 1u);
        last = (t == gridDim.x - 1);
    }
    __syncthreads();
    if (!last) return;
    __threadfence();
    const int nobs = in.nobs, PP = in.nobs + in.has_ret;
    const double on = nobs ? out.ocount[0] : 0.0, rn = in.has_ret ? out.rcount[0] : 0.0;
    double batch = (double)in.N;
    __shared__ double fa[4 * SDCGYM_MAX_M + 1], fb[4 * SDCGYM_MAX_M + 1];
    __shared__ int timed_out;
    if (threadIdx.x == 0) timed_out = 0;
    __syncthreads();
    for (int q = threadIdx.x >> 5; q < PP; q += kAccThreads / 32) {  // one warp per plane
        double sa, sb;
        stat_fold(partial, q, sa, sb);
        if ((threadIdx.x & 31) == 0) {
            fa[q] = sa;
            fb[q] = sb;
        }
    }
    __syncthreads();
    if (DIST) {
        const int parity = (int)(xc.seq & 1ull);
        for (int q = threadIdx.x; q < PP; q += kAccThreads)
            for (int rk = 0; rk < xc.world; rk++) {
                double* slot = xchg_slot(xc.peer[rk], xc.world, xc.stride, parity, xc.rank);
                slot[q] = fa[q];
                slot[PP + q] = fb[q];
            }
        if (threadIdx.x == 0)
            for (int rk = 0; rk < xc.world; rk++) xchg_slot(xc.peer[rk], xc.world, xc.stride, parity, xc.rank)[2 * PP] = batch;
        __threadfence_system();
        __syncthreads();
        if (threadIdx.x < xc.world) {
            volatile unsigned long long* remote = xchg_flags(xc.peer[threadIdx.x], xc.world, xc.stride, parity) + xc.rank;
            *remote = xc.seq;
            volatile unsigned long long* mine = xchg_flags(xc.peer[xc.rank], xc.world, xc.stride, parity) + threadIdx.x;
            if (!xchg_wait(mine, xc.seq)) timed_out = 1;
        }
        __threadfence_system();
        __syncthreads();
        double* region = xc.peer[xc.rank];
        batch = timed_out ? CUDART_NAN : 0.0;
        for (int rk = 0; rk < xc.world; rk++) batch += __ldcv(xchg_slot(region, xc.world, xc.stride, parity, rk) + 2 * PP);
        for (int q = threadIdx.x; q < PP; q += kAccThreads) {
            double sa = 0.0, sb = 0.0;
            for (int rk = 0; rk < xc.world; rk++) {
                const double* slot = xchg_slot(region, xc.world, xc.stride, parity, rk);
                sa += __ldcv(slot + q);
                sb += __ldcv(slot + PP + q);
            }
            fa[q] = sa;
            fb[q] = sb;
        }
        __syncthreads();
    }
    const bool merge = (batch > 0.0) || (batch != batch);  // (NaN batch: a peer timed out - poison the statistics)
    for (int q = threadIdx.x; q < PP; q += kAccThreads) {
        if (q < nobs) {
            out.osums[q] = fa[q];
            out.osums[nobs + q] = fb[q];
            double m = out.omean[q], v = out.ovar[q];
            if (merge) rms_merge_one(on, batch, fa[q], fb[q], m, v);
            out.omean[q] = m;
            out.ovar[q] = v;
        } else {
            out.rsums[0] = fa[q];
            out.rsums[1] = fb[q];
            double m = out.rmean[0], v = out.rvar[0];
            if (merge) rms_merge_one(rn, batch, fa[q], fb[q], m, v);
            out.rmean[0] = m;
            out.rvar[0] = v;
        }
    }
    if (threadIdx.x == 0) {
        if (nobs) {
            out.ocount[0] = on + batch;
            out.ocount[1] = on + batch;
        }
        if (in.has_ret) {
            out.rcount[0] = rn + batch;
            out.rcount[1] = rn + batch;
        }
        *ticket = 0u;  // self-cleaning: ready for the next launch on this stream
    }
}

__global__ void apply_kernel(int64_t N, int64_t ld, const double* __restrict__ X, const double* __restrict__ mean,
                             const double* __restrict__ var, double eps, double clip, double* __restrict__ Y) {
    const int p = blockIdx.y;
    const double m = mean[p], is = norm_inv_std(var[p], eps);
    // one 8-byte element per thread and iteration: measured 5.6 TB/s (86 % of the copy peak); a 128-bit variant
    // (two envs per access) measured 15 % slower
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (int64_t)gridDim.x * blockDim.x)
        Y[(int64_t)p * ld + i] = norm_obs(X[(int64_t)p * ld + i], m, is, clip);
}

__global__ void returns_kernel(int64_t N, const double* __restrict__ reward, double gamma, double* __restrict__ ret) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < N) ret[i] = advance_return(ret[i], gamma, reward[i]);
}
__global__ void reward_apply_kernel(int64_t N, const double* __restrict__ reward, const uint8_t* __restrict__ flags,
                                    const double* __restrict__ ret_var, double eps, double clip, int normalize,
                                    double* __restrict__ out, double* __restrict__ ret) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    double r = reward[i];
    if (normalize) r = norm_reward(r, ret_var[0], eps, clip);
    out[i] = r;
    if (ret && flags && (flags[i] & SDCGYM_FLAG_DONE)) ret[i] = 0.0;
}

// ---- ResidualLoss.take_step (dp_playground.py:247-258): u' = u + P^{-1} r_old, r' = u0 - C u', ||r'||inf -------
template <int M>
struct ResParams {
    double Q[M * M];
    double Qd[M * M];
    int64_t N;
    const double *lam, *qd, *Cs, *u0, *u, *r_old;
    double *u_out, *r_out, *norm_out;
    double* grad;  // optional [N][A][2]: d ||r'||inf / d theta_k as complex g (d = Re(sum g_k d theta_k))
    double dt;
    int32_t prec_type, qd_is_complex, n_act;
};

template <int M>
__global__ void __launch_bounds__(128) residual_step_kernel(const __grid_constant__ ResParams<M> p) {
    const int64_t i = (int64_t)blockIdx.x * 128 + threadIdx.x;
    if (i >= p.N) return;
    const C2 z{p.lam[2 * i] * p.dt, p.lam[2 * i + 1] * p.dt};
    C2 Qd[M * M];
    const int w = p.qd_is_complex ? 2 : 1;
    const double* row = p.qd ? p.qd + i * (int64_t)p.n_act * w : nullptr;
    int k = 0;
#pragma unroll
    for (int r = 0; r < M; r++)
#pragma unroll
        for (int c = 0; c < M; c++) {
            C2 d{0.0, 0.0};
            bool take = false;
            switch (p.prec_type) {
            case SDCGYM_PREC_DIAG: take = (c == r); break;
            case SDCGYM_PREC_LOWER_DIAG: take = (r == c + 1); break;
            case SDCGYM_PREC_LOWER_TRI: take = (c <= r); break;
            case SDCGYM_PREC_STRICTLY_LOWER_TRI: take = (c < r); break;
            default: break;
            }
            if (p.prec_type == SDCGYM_PREC_FIXED) d.r = (c <= r) ? p.Qd[r * M + c] : 0.0;
            else if (take) {
                d.r = row[k * w];
                if (p.qd_is_complex) d.i = row[k * w + 1];
                k++;
            }
            Qd[r * M + c] = d;
        }
    // delta = P^{-1} r_old by forward substitution, P = I - z Qd (lower triangular)
    C2 un[M], dl[M];
#pragma unroll
    for (int r = 0; r < M; r++) {
        C2 acc{p.r_old[(i * M + r) * 2], p.r_old[(i * M + r) * 2 + 1]};
#pragma unroll
        for (int c = 0; c < r; c++) acc = c_add(acc, c_mul(c_mul(z, Qd[r * M + c]), dl[c]));
        dl[r] = c_div(acc, c_sub(C2{1.0, 0.0}, c_mul(z, Qd[r * M + r])));
        un[r] = c_add(C2{p.u[(i * M + r) * 2], p.u[(i * M + r) * 2 + 1]}, dl[r]);
    }
    double nrm = 0.0;
    bool nan = false;
    int kmax = 0;
    C2 rk{0.0, 0.0};
#pragma unroll
    for (int r = 0; r < M; r++) {
        C2 acc{0.0, 0.0};
#pragma unroll
        for (int c = 0; c < M; c++) {
            C2 cij;
            if (p.Cs) cij = C2{p.Cs[((i * M + r) * M + c) * 2], p.Cs[((i * M + r) * M + c) * 2 + 1]};
            else cij = C2{(r == c ? 1.0 : 0.0) - z.r * p.Q[r * M + c], -z.i * p.Q[r * M + c]};
            acc = c_add(acc, c_mul(cij, un[c]));
        }
        C2 res = c_sub(C2{p.u0[(i * M + r) * 2], p.u0[(i * M + r) * 2 + 1]}, acc);
        p.u_out[(i * M + r) * 2] = un[r].r;
        p.u_out[(i * M + r) * 2 + 1] = un[r].i;
        p.r_out[(i * M + r) * 2] = res.r;
        p.r_out[(i * M + r) * 2 + 1] = res.i;
        double a = hypot(res.r, res.i);
        nan |= isnan(a);
        if (a > nrm) {
            nrm = a;
            kmax = r;
            rk = res;
        }
    }
    p.norm_out[i] = nan ? CUDART_NAN : nrm;
    if (p.grad) {
        // d r' = -z C P^{-1} dQd delta  =>  d ||r'||inf = Re( conj(r'_k)/|r'_k| * (-z) a_i delta_j dQd_ij ),
        // a = P^{-T} C_{k,:}^T (back substitution on the upper-triangular P^T), k = argmax |r'_m|
        C2 a[M];
#pragma unroll
        for (int m = M - 1; m >= 0; m--) {
            C2 ck{0.0, 0.0};
#pragma unroll
            for (int r = 0; r < M; r++)
                if (r == kmax) {
                    if (p.Cs) ck = C2{p.Cs[((i * M + r) * M + m) * 2], p.Cs[((i * M + r) * M + m) * 2 + 1]};
                    else ck = C2{(r == m ? 1.0 : 0.0) - z.r * p.Q[r * M + m], -z.i * p.Q[r * M + m]};
                }
            C2 acc = ck;
#pragma unroll
            for (int q = m + 1; q < M; q++) acc = c_add(acc, c_mul(c_mul(z, Qd[q * M + m]), a[q]));  // - P_qm a_q
            a[m] = c_div(acc, c_sub(C2{1.0, 0.0}, c_mul(z, Qd[m * M + m])));
        }
        C2 f{0.0, 0.0};
        if (nrm > 0.0 && !nan) f = c_mul(c_scale(c_conj(rk), 1.0 / nrm), C2{-z.r, -z.i});
        double* g = p.grad + i * (int64_t)p.n_act * 2;
        int kk = 0;
#pragma unroll
        for (int r = 0; r < M; r++)
#pragma unroll
            for (int c = 0; c < M; c++) {
                bool take = false;
                switch (p.prec_type) {
                case SDCGYM_PREC_DIAG: take = (c == r); break;
                case SDCGYM_PREC_LOWER_DIAG: take = (r == c + 1); break;
                case SDCGYM_PREC_LOWER_TRI: take = (c <= r); break;
                case SDCGYM_PREC_STRICTLY_LOWER_TRI: take = (c < r); break;
                default: break;
                }
                if (take) {
                    const C2 gv = c_mul(f, c_mul(a[r], dl[c]));
                    g[2 * kk] = gv.r;
                    g[2 * kk + 1] = gv.i;
                    kk++;
                }
            }
    }
}

template <int M>
static int launch_residual(const sdcgym_rho_desc* d, int64_t N, const double* lam, const double* qd, const double* Cs,
                           const double* u0, const double* u, const double* r_old, double* u_out, double* r_out,
                           double* norm_out, double* grad, cudaStream_t s) {
    ResParams<M> p;
    for (int k = 0; k < M * M; k++) {
        p.Q[k] = d->Q[k];
        p.Qd[k] = d->Qd_fixed[k];
    }
    p.N = N; p.lam = lam; p.qd = qd; p.Cs = Cs; p.u0 = u0; p.u = u; p.r_old = r_old;
    p.u_out = u_out; p.r_out = r_out; p.norm_out = norm_out; p.grad = grad;
    p.dt = d->dt; p.prec_type = d->prec_type; p.qd_is_complex = d->qd_is_complex;
    p.n_act = sdcgym_num_actions(M, d->prec_type);
    residual_step_kernel<M><<<(unsigned)((N + 127) / 128), 128, 0, s>>>(p);
    return (int)cudaGetLastError();
}

// ---- generalised advantage estimation over a device rollout (SB3 RolloutBuffer.compute_returns_and_advantage) ----
// one thread per env, reverse scan over the T stored steps; every access is coalesced along the env axis.
__global__ void __launch_bounds__(256) gae_kernel(int T, int64_t N, const double* __restrict__ rewards,
                                                  const double* __restrict__ values,
                                                  const uint8_t* __restrict__ episode_starts,
                                                  const double* __restrict__ last_values,
                                                  const uint8_t* __restrict__ last_dones, double gamma, double lam,
                                                  double* __restrict__ advantages, double* __restrict__ returns) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= N) return;
    double last_gae = 0.0;
    double next_value = last_values[i];
    double next_non_terminal = last_dones[i] ? 0.0 : 1.0;
    for (int t = T - 1; t >= 0; t--) {
        const int64_t k = (int64_t)t * N + i;
        const double v = values[k];
        const double delta = rewards[k] + gamma * next_value * next_non_terminal - v;
        last_gae = delta + gamma * lam * next_non_terminal * last_gae;
        advantages[k] = last_gae;
        returns[k] = last_gae + v;
        next_value = v;
        next_non_terminal = episode_starts[k] ? 0.0 : 1.0;
    }
}

}  // namespace sdcgym

using namespace sdcgym;

extern "C" int sdcgym_gae(int T, int64_t N, const double* rewards, const double* values, const uint8_t* episode_starts,
                          const double* last_values, const uint8_t* last_dones, double gamma, double gae_lambda,
                          double* advantages, double* returns, void* stream) {
    if (T < 0 || N < 0) return SDCGYM_EINVAL;
    if (T == 0 || N == 0) return 0;
    if (!rewards || !values || !episode_starts || !last_values || !last_dones || !advantages || !returns) return SDCGYM_ENULL;
    gae_kernel<<<(unsigned)((N + 255) / 256), 256, 0, (cudaStream_t)stream>>>(T, N, rewards, values, episode_starts,
                                                                            last_values, last_dones, gamma, gae_lambda,
                                                                            advantages, returns);
    return (int)cudaGetLastError();
}

static int fill_xchg(const sdcgym_xchg* x, int P, XchgDev& d) {
    if (!x) return SDCGYM_ENULL;
    if (x->world < 1 || x->world > SDCGYM_MAX_RANKS || x->rank < 0 || x->rank >= x->world) return SDCGYM_EINVAL;
    if (x->slot_doubles < 2 * P + 1 || x->seq == 0) return SDCGYM_EINVAL;
    d.world = x->world;
    d.rank = x->rank;
    d.seq = x->seq;
    d.stride = x->slot_doubles;
    for (int r = 0; r < x->world; r++) {
        if (!x->peers[r]) return SDCGYM_ENULL;
        d.peer[r] = static_cast<double*>(x->peers[r]);
    }
    return 0;
}

extern "C" size_t sdcgym_xchg_bytes(int world, int slot_doubles) {
    if (world < 1 || slot_doubles < 1) return 0;
    return ((size_t)2 * world * slot_doubles) * sizeof(double) + (size_t)2 * world * sizeof(unsigned long long);
}

extern "C" int sdcgym_vecnorm_scratch_doubles(int P) { return P * kStatBlocks * 2 + 2; }  // partials + the ticket word

// the bulk-copy variant needs full tiles for every block and 16-byte aligned plane rows
static bool stat_stream_ok(const StatIn& in) {
    const bool off = getenv("SDCGYM_NO_STAT_STREAM") != nullptr;  // A/B switch (read per call: the parity test toggles it)
    if (off || in.N < (int64_t)kStatBlocks * kStatTile) return false;
    auto al = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
    if (in.nobs && (!al(in.X) || (in.ld & 1))) return false;
    if (in.has_ret && (!al(in.ret) || !al(in.reward))) return false;
    return true;
}
// dynamic shared memory above 48 KB is an opt-in per kernel AND per device
template <class K>
static cudaError_t stat_smem_attr(K kernel) {
    static std::atomic<uint64_t> configured{0};
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    const uint64_t bit = (dev >= 0 && dev < 64) ? (uint64_t(1) << dev) : 0;
    if (!(configured.load(std::memory_order_relaxed) & bit)) {
        e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kStatStreamSmem);
        if (e != cudaSuccess) return e;
        configured.fetch_or(bit, std::memory_order_relaxed);
    }
    return cudaSuccess;
}

// one launch for any combination of observation planes and return plane, single rank or in-kernel exchange
static int launch_stat_update(int nobs, int64_t N, int64_t ld, const double* X, const double* reward, double gamma,
                              double* returns, bool has_ret, double* omean, double* ovar, double* ocount, double* osums,
                              double* rmean, double* rvar, double* rcount, double* rsums, double* scratch,
                              const sdcgym_xchg* xchg, void* stream) {
    const int PP = nobs + (has_ret ? 1 : 0);
    if (PP < 1 || nobs > 4 * SDCGYM_MAX_M || N < 0 || ld < N) return SDCGYM_EINVAL;
    if (!scratch) return SDCGYM_ENULL;
    if (nobs && ((N > 0 && !X) || !omean || !ovar || !ocount || !osums)) return SDCGYM_ENULL;
    if (has_ret && ((N > 0 && (!reward || !returns)) || !rmean || !rvar || !rcount || !rsums)) return SDCGYM_ENULL;
    if (!xchg && N == 0) return 0;  // (an empty shard still takes part in an exchange)
    StatIn in{nobs, has_ret ? 1 : 0, N, ld, X, omean, reward, gamma, returns, rmean};
    StatOut out{omean, ovar, ocount, osums, rmean, rvar, rcount, rsums};
    unsigned int* ticket = reinterpret_cast<unsigned int*>(scratch + (int64_t)PP * kStatBlocks * 2);
    const dim3 grid(kStatBlocks);
    const bool stream_ok = stat_stream_ok(in);
    cudaStream_t s = (cudaStream_t)stream;
    cudaError_t e = cudaSuccess;
    if (xchg) {
        XchgDev d{};
        int rc = fill_xchg(xchg, PP, d);
        if (rc) return rc;
        if (stream_ok) {
            if ((e = stat_smem_attr(stat_update_kernel<true, true>)) != cudaSuccess) return (int)e;
            stat_update_kernel<true, true><<<grid, kAccThreads, kStatStreamSmem, s>>>(in, out, scratch, ticket, d);
        } else {
            stat_update_kernel<true, false><<<grid, kAccThreads, 0, s>>>(in, out, scratch, ticket, d);
        }
    } else if (stream_ok) {
        if ((e = stat_smem_attr(stat_update_kernel<false, true>)) != cudaSuccess) return (int)e;
        stat_update_kernel<false, true><<<grid, kAccThreads, kStatStreamSmem, s>>>(in, out, scratch, ticket, XchgDev{});
    } else {
        stat_update_kernel<false, false><<<grid, kAccThreads, 0, s>>>(in, out, scratch, ticket, XchgDev{});
    }
    return (int)cudaGetLastError();
}

extern "C" int sdcgym_vecnorm_update(int P, int64_t N, int64_t ld, const double* X, double* mean, double* var,
                                     double* count2, double* scratch, double* sums, void* stream) {
    if (P < 1) return SDCGYM_EINVAL;
    return launch_stat_update(P, N, ld, X, nullptr, 0.0, nullptr, false, mean, var, count2, sums, nullptr, nullptr, nullptr,
                              nullptr, scratch, nullptr, stream);
}
extern "C" int sdcgym_vecnorm_update_returns(int64_t N, const double* reward, double gamma, double* returns, double* mean,
                                             double* var, double* count2, double* scratch, double* sums, void* stream) {
    return launch_stat_update(0, N, N, nullptr, reward, gamma, returns, true, nullptr, nullptr, nullptr, nullptr, mean, var,
                              count2, sums, scratch, nullptr, stream);
}
extern "C" int sdcgym_vecnorm_update_dist(int P, int64_t N, int64_t ld, const double* X, double* mean, double* var,
                                          double* count2, double* scratch, double* sums, const sdcgym_xchg* xchg,
                                          void* stream) {
    if (P < 1 || !xchg) return xchg ? SDCGYM_EINVAL : SDCGYM_ENULL;
    return launch_stat_update(P, N, ld, X, nullptr, 0.0, nullptr, false, mean, var, count2, sums, nullptr, nullptr, nullptr,
                              nullptr, scratch, xchg, stream);
}
extern "C" int sdcgym_vecnorm_update_returns_dist(int64_t N, const double* reward, double gamma, double* returns,
                                                  double* mean, double* var, double* count2, double* scratch,
                                                  double* sums, const sdcgym_xchg* xchg, void* stream) {
    if (!xchg) return SDCGYM_ENULL;
    return launch_stat_update(0, N, N, nullptr, reward, gamma, returns, true, nullptr, nullptr, nullptr, nullptr, mean, var,
                              count2, sums, scratch, xchg, stream);
}
extern "C" int sdcgym_vecnorm_update_both(int P, int64_t N, int64_t ld, const double* X, const double* reward, double gamma,
                                          double* returns, double* obs_mean, double* obs_var, double* obs_count2,
                                          double* ret_mean, double* ret_var, double* ret_count2, double* scratch,
                                          double* sums_obs, double* sums_ret, const sdcgym_xchg* xchg, void* stream) {
    if (P < 1) return SDCGYM_EINVAL;
    return launch_stat_update(P, N, ld, X, reward, gamma, returns, true, obs_mean, obs_var, obs_count2, sums_obs, ret_mean,
                              ret_var, ret_count2, sums_ret, scratch, xchg, stream);
}

extern "C" int sdcgym_vecnorm_accumulate(int P, int64_t N, int64_t ld, const double* X, const double* shift,
                                         double* scratch, double* sums, void* stream) {
    if (P < 1 || P > 4 * SDCGYM_MAX_M || N < 0 || ld < N) return SDCGYM_EINVAL;
    if (!X || !scratch || !sums) return SDCGYM_ENULL;
    cudaStream_t s = (cudaStream_t)stream;
    StatIn in{P, 0, N, ld, X, shift, nullptr, 0.0, nullptr, nullptr};
    if (stat_stream_ok(in)) {
        cudaError_t e = stat_smem_attr(acc_partial_kernel<true>);
        if (e != cudaSuccess) return (int)e;
        acc_partial_kernel<true><<<kStatBlocks, kAccThreads, kStatStreamSmem, s>>>(in, scratch);
    } else {
        acc_partial_kernel<false><<<kStatBlocks, kAccThreads, 0, s>>>(in, scratch);
    }
    acc_final_kernel<<<1, kAccThreads, 0, s>>>(P, scratch, sums);
    return (int)cudaGetLastError();
}

// ---- exchange regions: cudaMalloc'd (legacy CUDA IPC needs that), zeroed, shared between the ranks' processes by IPC
//      handle; opening a handle enables peer access to the owning device ----
extern "C" int sdcgym_ipc_alloc(size_t bytes, void** dev_ptr, unsigned char* handle64) {
    if (!dev_ptr || !handle64) return SDCGYM_ENULL;
    if (bytes == 0) return SDCGYM_EINVAL;
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e != cudaSuccess) return (int)e;
    e = cudaMemset(p, 0, bytes);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    cudaIpcMemHandle_t h;
    if (e == cudaSuccess) e = cudaIpcGetMemHandle(&h, p);
    if (e != cudaSuccess) {
        cudaFree(p);
        return (int)e;
    }
    memcpy(handle64, &h, 64);
    *dev_ptr = p;
    return 0;
}
extern "C" int sdcgym_ipc_open(const unsigned char* handle64, void** dev_ptr) {
    if (!handle64 || !dev_ptr) return SDCGYM_ENULL;
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, 64);
    return (int)cudaIpcOpenMemHandle(dev_ptr, h, cudaIpcMemLazyEnablePeerAccess);
}
extern "C" int sdcgym_ipc_close(void* dev_ptr) { return dev_ptr ? (int)cudaIpcCloseMemHandle(dev_ptr) : 0; }
extern "C" int sdcgym_ipc_free(void* dev_ptr) { return dev_ptr ? (int)cudaFree(dev_ptr) : 0; }

extern "C" int sdcgym_vecnorm_merge(int P, double batch_count, const double* sums, double* mean, double* var,
                                    double* count2, void* stream) {
    if (P < 1 || P > 1024) return SDCGYM_EINVAL;
    if (!sums || !mean || !var || !count2) return SDCGYM_ENULL;
    cudaStream_t s = (cudaStream_t)stream;
    rms_merge_kernel<<<1, 1024, 0, s>>>(P, batch_count, sums, mean, var, count2);
    if (batch_count > 0) rms_commit_kernel<<<1, 1, 0, s>>>(count2);
    return (int)cudaGetLastError();
}

extern "C" int sdcgym_vecnorm_apply(int P, int64_t N, int64_t ld, const double* X, const double* mean, const double* var,
                                    double eps, double clip, double* Y, void* stream) {
    if (P < 1 || N < 0 || ld < N) return SDCGYM_EINVAL;
    if (N == 0) return 0;
    if (!X || !Y || !mean || !var) return SDCGYM_ENULL;
    unsigned gx = (unsigned)((N + 255) / 256);
    if (gx > 148 * 8) gx = 148 * 8;
    apply_kernel<<<dim3(gx, P), 256, 0, (cudaStream_t)stream>>>(N, ld, X, mean, var, eps, clip, Y);
    return (int)cudaGetLastError();
}

extern "C" int sdcgym_vecnorm_returns(int64_t N, const double* reward, double gamma, double* returns, void* stream) {
    if (N < 0) return SDCGYM_EINVAL;
    if (N == 0) return 0;
    if (!reward || !returns) return SDCGYM_ENULL;
    returns_kernel<<<(unsigned)((N + 255) / 256), 256, 0, (cudaStream_t)stream>>>(N, reward, gamma, returns);
    return (int)cudaGetLastError();
}

extern "C" int sdcgym_vecnorm_reward(int64_t N, const double* reward, const uint8_t* flags, const double* ret_var,
                                     double eps, double clip, int normalize, double* out, double* returns, void* stream) {
    if (N < 0) return SDCGYM_EINVAL;
    if (N == 0) return 0;
    if (!reward || !out || (normalize && !ret_var)) return SDCGYM_ENULL;
    reward_apply_kernel<<<(unsigned)((N + 255) / 256), 256, 0, (cudaStream_t)stream>>>(N, reward, flags, ret_var, eps, clip,
                                                                                      normalize, out, returns);
    return (int)cudaGetLastError();
}

extern "C" int sdcgym_residual_step(const sdcgym_rho_desc* d, int64_t N, const double* lam, const double* qd,
                                    const double* Cs, const double* u0, const double* u, const double* r_old,
                                    double* u_out, double* r_out, double* norm_out, double* grad, void* stream) {
    if (!d) return SDCGYM_ENULL;
    if (!sdcgym_supported(d->M, d->prec_type)) return SDCGYM_EUNSUPPORTED;
    if (N < 0) return SDCGYM_EINVAL;
    if (N == 0) return 0;
    if (!lam || !u0 || !u || !r_old || !u_out || !r_out || !norm_out) return SDCGYM_ENULL;
    if (d->prec_type != SDCGYM_PREC_FIXED && !qd) return SDCGYM_ENULL;
    if (grad && d->prec_type == SDCGYM_PREC_FIXED) return SDCGYM_EUNSUPPORTED;
    cudaStream_t s = (cudaStream_t)stream;
    switch (d->M) {
#define C(m) case m: return launch_residual<m>(d, N, lam, qd, Cs, u0, u, r_old, u_out, r_out, norm_out, grad, s);
        C(2) C(3) C(4) C(5) C(6) C(7) C(8) C(9)
#undef C
    }
    return SDCGYM_EUNSUPPORTED;
}

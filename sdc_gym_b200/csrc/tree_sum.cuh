// tree_sum.cuh - deterministic device sums over samples of one value vector per sample (the reduced gradients of
// sdcgym_spectral_radius_grad_sum and sdcgym_residual_sweeps_sum).
//
// Every value is summed by a balanced binary tree whose shape depends on N alone: each 128-sample tile folds its
// samples (5 shuffle levels per warp, then (w0 + w1) + (w2 + w3)) into one partial per value, and
// rho_grad_sum_fold_kernel (specrad.cu) folds groups of kFold consecutive partials until one is left.  No atomics, no
// dependence on the SM count or on timing: the same inputs give the same bits.  Padding lanes add exact zeros.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace sdcgym {

constexpr int kFold = 256;

__device__ __forceinline__ double warp_tree_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    return v;  // lane 0
}

// Folds scratch = the tile partials [nv][T] into sums [nv], using the rest of scratch for the intermediate levels: a
// scratch of sdcgym_spectral_radius_grad_sum_scratch_doubles(M, prec_type, N) doubles holds every level for
// nv = 1 + 2 sdcgym_num_actions(M, prec_type) values.  Returns cudaGetLastError().
int grad_sum_fold(int64_t T, int nv, double* scratch, double* sums, cudaStream_t s);

}  // namespace sdcgym

// normalize.cuh - the VecNormalize arithmetic (SB3: clip((x - mean) / sqrt(var + eps), +-clip) for observations,
// clip(r / sqrt(ret_var + eps), +-clip) for rewards), shared by every kernel that applies it (csrc/vecnorm.cu's
// apply / reward kernels and csrc/replay.cu's sampler) so that they produce the same bits.
//
// Every rounding is explicit (__dsub_rn, __dmul_rn, correctly rounded division and square root): there is no
// multiply-add the compiler could contract, so the result is the same with -fmad=true and -fmad=false.
#pragma once

namespace sdcgym {

// 1 / sqrt(var + eps): computed once per plane by the observation kernels
__device__ __forceinline__ double norm_inv_std(double var, double eps) { return 1.0 / sqrt(var + eps); }

__device__ __forceinline__ double norm_obs(double x, double mean, double inv_std, double clip) {
    const double v = __dmul_rn(__dsub_rn(x, mean), inv_std);
    return fmin(fmax(v, -clip), clip);
}

__device__ __forceinline__ double norm_reward(double r, double ret_var, double eps, double clip) {
    return fmin(fmax(r / sqrt(ret_var + eps), -clip), clip);
}

}  // namespace sdcgym

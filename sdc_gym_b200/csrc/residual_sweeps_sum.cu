// residual_sweeps_sum.cu - sdcgym_residual_sweeps_sum: the K-sweep residual loss of ONE shared parameter row and its
// gradient, summed over a lambda batch or a lambda grid on the device (see residual_sweeps.cuh, tree_sum.cuh,
// include/sdcgym.h).  No per-sample gradient, u_K or r_K is stored.
#include "residual_sweeps.cuh"
#include "specrad_params.cuh"
#include "tree_sum.cuh"

namespace sdcgym {

template <int M>
struct SweepSumParams {
    SweepParams<M> s;  // s.lam NULL: grid mode; s.norm_out optional; u_out, r_out, grad unused
    int64_t grid_re, grid_im, grid_first;
    double re_lo, re_hi, im_lo, im_hi;
    int32_t reduction;
};

// partials [nv][T] (T = gridDim.x tiles, nv = 1 + 2 n_act values): f, then Re / Im of each parameter's weighted g
template <int M, int PT, bool QC>
__global__ void __launch_bounds__(128) residual_sweeps_sum_kernel(const __grid_constant__ SweepSumParams<M> p,
                                                                  double* __restrict__ partials) {
    __shared__ double part[4][1 + M * (M + 1)];
    const int64_t i = (int64_t)blockIdx.x * 128 + threadIdx.x;
    double f = 0.0;
    C2 gw[M * M];
    if (i < p.s.N) {
        double lr, li, nK;
        if (p.s.lam) {
            lr = p.s.lam[2 * i];
            li = p.s.lam[2 * i + 1];
        } else {
            grid_lambda(p, p.grid_first + i, lr, li);
        }
        f = residual_sweeps_reduced<M, PT, QC>(p.s, i, C2{lr * p.s.dt, li * p.s.dt}, p.reduction, nK, gw);
        if (p.s.norm_out) p.s.norm_out[i] = nK;
    } else {
#pragma unroll
        for (int q = 0; q < M * M; q++) gw[q] = C2{0.0, 0.0};
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    f = warp_tree_sum(f);
    if (lane == 0) part[warp][0] = f;
    int k = 0;
#pragma unroll
    for (int a = 0; a < M; a++)
#pragma unroll
        for (int c = 0; c <= a; c++)
            if (sweep_param<PT>(a, c)) {
                const double gr = warp_tree_sum(gw[a * M + c].r), gi = warp_tree_sum(gw[a * M + c].i);
                if (lane == 0) {
                    part[warp][1 + 2 * k] = gr;
                    part[warp][2 + 2 * k] = gi;
                }
                k++;
            }
    __syncthreads();
    if ((int)threadIdx.x < 1 + 2 * k) {
        const int j = threadIdx.x;
        partials[(int64_t)j * gridDim.x + blockIdx.x] = (part[0][j] + part[1][j]) + (part[2][j] + part[3][j]);
    }
}

template <int M, int PT, bool QC>
static int launch_sum(const SweepSumParams<M>& p, double* scratch, double* sums, cudaStream_t s) {
    const int64_t T = (p.s.N + 127) / 128;
    residual_sweeps_sum_kernel<M, PT, QC><<<(unsigned)T, 128, 0, s>>>(p, scratch);
    return grad_sum_fold(T, 1 + 2 * p.s.n_act, scratch, sums, s);
}

template <int M, int PT>
static int launch_sum_layout(const SweepSumParams<M>& p, bool qc, double* scratch, double* sums, cudaStream_t s) {
    return qc ? launch_sum<M, PT, true>(p, scratch, sums, s) : launch_sum<M, PT, false>(p, scratch, sums, s);
}

template <int M>
static int launch_residual_sweeps_sum(const sdcgym_rho_desc* d, int64_t N, int sweeps, int reduction,
                                      const double* lam, const double* qd, const double* u0, const double* u,
                                      const double* r, double* norm_out, double* scratch, double* sums,
                                      cudaStream_t s) {
    SweepSumParams<M> p;
    fill_sweep_params<M>(p.s, d, N, sweeps, lam, qd, u0, u, r, nullptr, nullptr, norm_out, nullptr);
    p.grid_re = d->grid_re;
    p.grid_im = d->grid_im;
    p.grid_first = d->grid_first;
    p.re_lo = d->re_lo;
    p.re_hi = d->re_hi;
    p.im_lo = d->im_lo;
    p.im_hi = d->im_hi;
    p.reduction = reduction;
    const bool qc = d->qd_is_complex != 0;
    switch (d->prec_type) {
    case SDCGYM_PREC_DIAG: return launch_sum_layout<M, SDCGYM_PREC_DIAG>(p, qc, scratch, sums, s);
    case SDCGYM_PREC_LOWER_DIAG: return launch_sum_layout<M, SDCGYM_PREC_LOWER_DIAG>(p, qc, scratch, sums, s);
    case SDCGYM_PREC_LOWER_TRI: return launch_sum_layout<M, SDCGYM_PREC_LOWER_TRI>(p, qc, scratch, sums, s);
    case SDCGYM_PREC_STRICTLY_LOWER_TRI:
        return launch_sum_layout<M, SDCGYM_PREC_STRICTLY_LOWER_TRI>(p, qc, scratch, sums, s);
    }
    return SDCGYM_EUNSUPPORTED;
}

}  // namespace sdcgym

using namespace sdcgym;

extern "C" int sdcgym_residual_sweeps_sum(const sdcgym_rho_desc* d, int64_t N, int sweeps, int reduction,
                                          const double* lam, const double* qd, const double* u0, const double* u,
                                          const double* r, double* norm_out, double* scratch, double* sums,
                                          void* stream) {
    if (!d || !qd || !scratch || !sums) return SDCGYM_ENULL;
    const int given = (u0 != nullptr) + (u != nullptr) + (r != nullptr);
    if (given != 0 && given != 3) return SDCGYM_ENULL;
    if (!sdcgym_supported(d->M, d->prec_type) || d->prec_type == SDCGYM_PREC_FIXED) return SDCGYM_EUNSUPPORTED;
    if (d->qd_broadcast != 1 || N < 0 || sweeps < 1 || sweeps > kMaxSweeps) return SDCGYM_EINVAL;
    if (reduction != SDCGYM_SWEEPS_MEAN && reduction != SDCGYM_SWEEPS_LOG_RATIO) return SDCGYM_EINVAL;
    if (!lam && given) return SDCGYM_EINVAL;
    if (N > 0 && !lam &&
        (d->grid_re <= 0 || d->grid_im <= 0 || d->grid_first < 0 || d->grid_first + N > d->grid_re * d->grid_im))
        return SDCGYM_EINVAL;
    cudaStream_t s = (cudaStream_t)stream;
    if (N == 0)
        return (int)cudaMemsetAsync(sums, 0, (1 + 2 * (size_t)sdcgym_num_actions(d->M, d->prec_type)) * sizeof(double), s);
    switch (d->M) {
#define C(m) case m: return launch_residual_sweeps_sum<m>(d, N, sweeps, reduction, lam, qd, u0, u, r, norm_out, scratch, sums, s);
        C(2) C(3) C(4) C(5) C(6) C(7) C(8) C(9)
#undef C
    }
    return SDCGYM_EUNSUPPORTED;
}

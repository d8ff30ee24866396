// specrad.cu - sdcgym_spectral_radius / _grad / _grad_sum: batched rho(K) kernel launchers (see specrad.cuh, include/sdcgym.h).
#include "specrad_params.cuh"
#include "tree_sum.cuh"

namespace sdcgym {

#ifndef SDCGYM_RHO_MINB
#define SDCGYM_RHO_MINB 4  // 128 registers, 16 warps/SM: +25 % over 2 blocks/SM (profiles/README.md)
#endif
template <int M>
__global__ void __launch_bounds__(128, (M <= 5) ? SDCGYM_RHO_MINB : 1) rho_kernel(const __grid_constant__ RhoParams<M> p) {
    rho_one<M>(p, (int64_t)blockIdx.x * 128 + threadIdx.x);
}

template <int M>
__global__ void __launch_bounds__(128, (M <= 5) ? 2 : 1) rho_grad_kernel(const __grid_constant__ RhoParams<M> p,
                                                                        double* __restrict__ grad) {
    rho_grad_one<M>(p, (int64_t)blockIdx.x * 128 + threadIdx.x, grad);
}

// ---- sum over samples of rho and d rho / d theta for ONE shared parameter row (tree_sum.cuh) ----------------------
// partials [nv][T] (T = gridDim.x tiles, nv = 1 + 2 n_act values): rho, then Re / Im of each parameter's g
template <int M>
__global__ void __launch_bounds__(128, (M <= 5) ? 2 : 1) rho_grad_sum_kernel(const __grid_constant__ RhoParams<M> p,
                                                                            double* __restrict__ partials) {
    __shared__ double part[4][1 + M * (M + 1)];
    const int64_t i = (int64_t)blockIdx.x * 128 + threadIdx.x;
    double rho;
    C2 G[M * M];
    if (rho_grad_eval<M>(p, i, rho, G)) {
        if (p.rho) p.rho[i] = rho;
    } else {
        rho = 0.0;
#pragma unroll
        for (int k = 0; k < M * M; k++) G[k] = C2{0.0, 0.0};
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    rho = warp_tree_sum(rho);
    if (lane == 0) part[warp][0] = rho;
    int k = 0;
#pragma unroll
    for (int r = 0; r < M; r++)
#pragma unroll
        for (int c = 0; c < M; c++) {
            if (is_qd_param(p.prec_type, r, c)) {  // uniform over the block
                const double gr = warp_tree_sum(G[r * M + c].r), gi = warp_tree_sum(G[r * M + c].i);
                if (lane == 0) {
                    part[warp][1 + 2 * k] = gr;
                    part[warp][2 + 2 * k] = gi;
                }
                k++;
            }
        }
    __syncthreads();
    const int nv = 1 + 2 * p.n_act;
    if ((int)threadIdx.x < nv) {
        const int j = threadIdx.x;
        partials[(int64_t)j * gridDim.x + blockIdx.x] = (part[0][j] + part[1][j]) + (part[2][j] + part[3][j]);
    }
}

// Population form: row y = blockIdx.y at p.qd + y * qd_rs writes the [nv][T] partials of rho_grad_sum_kernel for that
// row to segments [y * nv, y * nv + nv) of partials [gridDim.y * nv][T].  The body is rho_grad_sum_kernel's with the row
// offset; it is spelled out because moving that body into a shared device function changes the code nvcc generates
// for rho_grad_sum_kernel itself.
template <int M>
__global__ void __launch_bounds__(128, (M <= 5) ? 2 : 1) rho_grad_sum_population_kernel(
    const __grid_constant__ RhoParams<M> p, int64_t qd_rs, double* __restrict__ partials) {
    __shared__ double part[4][1 + M * (M + 1)];
    const int64_t i = (int64_t)blockIdx.x * 128 + threadIdx.x;
    double rho;
    C2 G[M * M];
    if (!rho_grad_eval<M, true>(p, i, rho, G, (int64_t)blockIdx.y * qd_rs)) {
        rho = 0.0;
#pragma unroll
        for (int k = 0; k < M * M; k++) G[k] = C2{0.0, 0.0};
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    rho = warp_tree_sum(rho);
    if (lane == 0) part[warp][0] = rho;
    int k = 0;
#pragma unroll
    for (int r = 0; r < M; r++)
#pragma unroll
        for (int c = 0; c < M; c++) {
            if (is_qd_param(p.prec_type, r, c)) {  // uniform over the block
                const double gr = warp_tree_sum(G[r * M + c].r), gi = warp_tree_sum(G[r * M + c].i);
                if (lane == 0) {
                    part[warp][1 + 2 * k] = gr;
                    part[warp][2 + 2 * k] = gi;
                }
                k++;
            }
        }
    __syncthreads();
    const int nv = 1 + 2 * p.n_act;
    if ((int)threadIdx.x < nv) {
        const int j = threadIdx.x;
        partials[((int64_t)blockIdx.y * nv + j) * gridDim.x + blockIdx.x] =
            (part[0][j] + part[1][j]) + (part[2][j] + part[3][j]);
    }
}

// in [nv][T] -> out [nv][ceil(T / kFold)]: block (b, j) folds in[j][b*kFold .. b*kFold + kFold) by a balanced tree
__global__ void __launch_bounds__(kFold) rho_grad_sum_fold_kernel(int64_t T, const double* __restrict__ in,
                                                                   double* __restrict__ out) {
    __shared__ double part[kFold / 32];
    const int64_t t = (int64_t)blockIdx.x * kFold + threadIdx.x;
    const int64_t j = blockIdx.y;
    double v = warp_tree_sum(t < T ? in[j * T + t] : 0.0);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) part[warp] = v;
    __syncthreads();
    if (warp == 0) {
        v = lane < kFold / 32 ? part[lane] : 0.0;
#pragma unroll
        for (int o = kFold / 64; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
        if (lane == 0) out[j * gridDim.x + blockIdx.x] = v;
    }
}

// Fold level sizes: T_0 = ceil(N / 128) tile partials, T_{l+1} = ceil(T_l / kFold); the fold that produces a single
// value writes the sums, every other level lives in the scratch buffer.
static int64_t grad_sum_scratch_values(int64_t N) {
    int64_t T = (N + 127) / 128, total = T;
    while (T > 1) {
        T = (T + kFold - 1) / kFold;
        if (T > 1) total += T;
    }
    return total;
}

template <int M>
static int launch_rho_grad_sum(const sdcgym_rho_desc* d, int64_t N, const double* lam, const double* qd, double* rho,
                               double* scratch, double* sums, cudaStream_t s) {
    RhoParams<M> p;
    fill_rho_params<M>(p, d, N, lam, qd, rho);
    const int64_t T = (N + 127) / 128;
    rho_grad_sum_kernel<M><<<(unsigned)T, 128, 0, s>>>(p, scratch);
    return grad_sum_fold(T, 1 + 2 * p.n_act, scratch, sums, s);
}

// P rows in launches of at most 65535 / nv rows (the fold's gridDim.y is rows * nv); each launch folds its rows' P * nv
// segments like the single-row call folds its nv, in its own share of the scratch (P times the single-row size)
template <int M>
static int launch_rho_grad_sum_population(const sdcgym_rho_desc* d, int64_t N, const double* lam, int64_t P,
                                          const double* qd, int64_t qd_rs, double* scratch, double* sums,
                                          cudaStream_t s) {
    RhoParams<M> p;
    fill_rho_params<M>(p, d, N, lam, qd, nullptr);
    const int nv = 1 + 2 * p.n_act;
    const int64_t T = (N + 127) / 128, per_row = nv * grad_sum_scratch_values(N), chunk = 65535 / nv;
    for (int64_t r0 = 0; r0 < P; r0 += chunk) {
        const int64_t rows = P - r0 < chunk ? P - r0 : chunk;
        p.qd = qd + r0 * qd_rs;
        double* part = scratch + r0 * per_row;
        rho_grad_sum_population_kernel<M><<<dim3((unsigned)T, (unsigned)rows), 128, 0, s>>>(p, qd_rs, part);
        const int e = grad_sum_fold(T, (int)(rows * nv), part, sums + r0 * nv, s);
        if (e) return e;
    }
    return 0;
}

int grad_sum_fold(int64_t T, int nv, double* scratch, double* sums, cudaStream_t s) {
    double* in = scratch;
    while (true) {
        const int64_t To = (T + kFold - 1) / kFold;
        double* out = (To == 1) ? sums : in + (int64_t)nv * T;
        rho_grad_sum_fold_kernel<<<dim3((unsigned)To, (unsigned)nv), kFold, 0, s>>>(T, in, out);
        if (To == 1) break;
        in = out;
        T = To;
    }
    return (int)cudaGetLastError();
}

template <int M>
static int launch_rho_grad(const sdcgym_rho_desc* d, int64_t N, const double* lam, const double* qd, double* rho,
                           double* grad, cudaStream_t s) {
    RhoParams<M> p;
    fill_rho_params<M>(p, d, N, lam, qd, rho);
    rho_grad_kernel<M><<<(unsigned)((N + 127) / 128), 128, 0, s>>>(p, grad);
    return (int)cudaGetLastError();
}

template <int M>
static int launch_rho(const sdcgym_rho_desc* d, int64_t N, const double* lam, const double* qd, double* rho,
                      cudaStream_t s) {
    RhoParams<M> p;
    fill_rho_params<M>(p, d, N, lam, qd, rho);
    rho_kernel<M><<<(unsigned)((N + 127) / 128), 128, 0, s>>>(p);
    return (int)cudaGetLastError();
}

}  // namespace sdcgym

using namespace sdcgym;

extern "C" int sdcgym_spectral_radius(const sdcgym_rho_desc* d, int64_t N, const double* lam, const double* qd,
                                      double* rho, void* stream) {
    if (!d) return SDCGYM_ENULL;
    if (!sdcgym_supported(d->M, d->prec_type)) return SDCGYM_EUNSUPPORTED;
    if (N < 0) return SDCGYM_EINVAL;
    if (N == 0) return 0;  // an empty shard (dist.shard_range allows them) is a no-op, whatever the other arguments
    if (!lam && (d->grid_re <= 0 || d->grid_im <= 0 || d->grid_first < 0 || d->grid_first + N > d->grid_re * d->grid_im))
        return SDCGYM_EINVAL;
    if (!rho) return SDCGYM_ENULL;
    if (d->prec_type != SDCGYM_PREC_FIXED && !qd) return SDCGYM_ENULL;
    if (d->prec_type == SDCGYM_PREC_FIXED) {
        for (int r = 0; r < d->M; r++)
            for (int c = r + 1; c < d->M; c++)
                if (d->Qd_fixed[r * d->M + c] != 0.0) return SDCGYM_EUNSUPPORTED;  // not lower triangular
    }
    cudaStream_t s = (cudaStream_t)stream;
    switch (d->M) {
#define C(m) case m: return launch_rho<m>(d, N, lam, qd, rho, s);
        C(2) C(3) C(4) C(5) C(6) C(7) C(8) C(9)
#undef C
    }
    return SDCGYM_EUNSUPPORTED;
}

extern "C" int sdcgym_spectral_radius_grad(const sdcgym_rho_desc* d, int64_t N, const double* lam, const double* qd,
                                           double* rho, double* grad, void* stream) {
    if (!d) return SDCGYM_ENULL;
    if (!sdcgym_supported(d->M, d->prec_type)) return SDCGYM_EUNSUPPORTED;
    if (d->prec_type == SDCGYM_PREC_FIXED) return SDCGYM_EUNSUPPORTED;  // nothing to differentiate
    if (N < 0 || d->qd_broadcast) return SDCGYM_EINVAL;
    if (N == 0) return 0;
    if (!lam || !qd || !rho || !grad) return SDCGYM_ENULL;
    cudaStream_t s = (cudaStream_t)stream;
    switch (d->M) {
#define C(m) case m: return launch_rho_grad<m>(d, N, lam, qd, rho, grad, s);
        C(2) C(3) C(4) C(5) C(6) C(7) C(8) C(9)
#undef C
    }
    return SDCGYM_EUNSUPPORTED;
}

extern "C" int64_t sdcgym_spectral_radius_grad_sum_scratch_doubles(int M, int prec_type, int64_t N) {
    if (!sdcgym_supported(M, prec_type) || prec_type == SDCGYM_PREC_FIXED) return SDCGYM_EUNSUPPORTED;
    if (N < 0) return SDCGYM_EINVAL;
    return (1 + 2 * (int64_t)sdcgym_num_actions(M, prec_type)) * grad_sum_scratch_values(N);
}

extern "C" int sdcgym_spectral_radius_grad_sum(const sdcgym_rho_desc* d, int64_t N, const double* lam,
                                               const double* qd, double* rho, double* scratch, double* sums,
                                               void* stream) {
    if (!d || !qd || !scratch || !sums) return SDCGYM_ENULL;
    if (!sdcgym_supported(d->M, d->prec_type) || d->prec_type == SDCGYM_PREC_FIXED) return SDCGYM_EUNSUPPORTED;
    if (!d->qd_broadcast || N < 0) return SDCGYM_EINVAL;
    if (N > 0 && !lam &&
        (d->grid_re <= 0 || d->grid_im <= 0 || d->grid_first < 0 || d->grid_first + N > d->grid_re * d->grid_im))
        return SDCGYM_EINVAL;
    cudaStream_t s = (cudaStream_t)stream;
    if (N == 0)
        return (int)cudaMemsetAsync(sums, 0, (1 + 2 * (size_t)sdcgym_num_actions(d->M, d->prec_type)) * sizeof(double), s);
    switch (d->M) {
#define C(m) case m: return launch_rho_grad_sum<m>(d, N, lam, qd, rho, scratch, sums, s);
        C(2) C(3) C(4) C(5) C(6) C(7) C(8) C(9)
#undef C
    }
    return SDCGYM_EUNSUPPORTED;
}

extern "C" int sdcgym_spectral_radius_grad_sum_population(const sdcgym_rho_desc* d, int64_t N, const double* lam,
                                                          int64_t P, const double* qd, int64_t qd_rs, double* scratch,
                                                          double* sums, void* stream) {
    if (!d || !qd || !scratch || !sums) return SDCGYM_ENULL;
    if (!sdcgym_supported(d->M, d->prec_type) || d->prec_type == SDCGYM_PREC_FIXED) return SDCGYM_EUNSUPPORTED;
    if (!d->qd_broadcast || P < 1 || N < 0) return SDCGYM_EINVAL;
    if (N > 0 && !lam &&
        (d->grid_re <= 0 || d->grid_im <= 0 || d->grid_first < 0 || d->grid_first + N > d->grid_re * d->grid_im))
        return SDCGYM_EINVAL;
    cudaStream_t s = (cudaStream_t)stream;
    if (N == 0)
        return (int)cudaMemsetAsync(
            sums, 0, (size_t)P * (1 + 2 * (size_t)sdcgym_num_actions(d->M, d->prec_type)) * sizeof(double), s);
    switch (d->M) {
#define C(m) case m: return launch_rho_grad_sum_population<m>(d, N, lam, P, qd, qd_rs, scratch, sums, s);
        C(2) C(3) C(4) C(5) C(6) C(7) C(8) C(9)
#undef C
    }
    return SDCGYM_EUNSUPPORTED;
}

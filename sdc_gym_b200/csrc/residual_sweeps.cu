// residual_sweeps.cu - sdcgym_residual_sweeps: ||r_K||_inf after K sweeps and its gradient (see residual_sweeps.cuh,
// include/sdcgym.h).
#include "residual_sweeps.cuh"

namespace sdcgym {

template <int M, int PT, bool QC, bool GRAD>
__global__ void __launch_bounds__(128) residual_sweeps_kernel(const __grid_constant__ SweepParams<M> p) {
    residual_sweeps_one<M, PT, QC, GRAD>(p, (int64_t)blockIdx.x * 128 + threadIdx.x);
}

template <int M, int PT, bool QC, bool GRAD>
static int launch_sweeps(const SweepParams<M>& p, cudaStream_t s) {
    residual_sweeps_kernel<M, PT, QC, GRAD><<<(unsigned)((p.N + 127) / 128), 128, 0, s>>>(p);
    return (int)cudaGetLastError();
}

template <int M, int PT>
static int launch_sweeps_layout(const SweepParams<M>& p, bool qc, bool grad, cudaStream_t s) {
    if (qc) return grad ? launch_sweeps<M, PT, true, true>(p, s) : launch_sweeps<M, PT, true, false>(p, s);
    return grad ? launch_sweeps<M, PT, false, true>(p, s) : launch_sweeps<M, PT, false, false>(p, s);
}

template <int M>
static int launch_residual_sweeps(const sdcgym_rho_desc* d, int64_t N, int sweeps, const double* lam, const double* qd,
                                  const double* u0, const double* u, const double* r, double* u_out, double* r_out,
                                  double* norm_out, double* grad, cudaStream_t s) {
    SweepParams<M> p;
    fill_sweep_params<M>(p, d, N, sweeps, lam, qd, u0, u, r, u_out, r_out, norm_out, grad);
    const bool qc = d->qd_is_complex != 0, g = grad != nullptr;
    switch (d->prec_type) {
    case SDCGYM_PREC_DIAG: return launch_sweeps_layout<M, SDCGYM_PREC_DIAG>(p, qc, g, s);
    case SDCGYM_PREC_LOWER_DIAG: return launch_sweeps_layout<M, SDCGYM_PREC_LOWER_DIAG>(p, qc, g, s);
    case SDCGYM_PREC_LOWER_TRI: return launch_sweeps_layout<M, SDCGYM_PREC_LOWER_TRI>(p, qc, g, s);
    case SDCGYM_PREC_STRICTLY_LOWER_TRI: return launch_sweeps_layout<M, SDCGYM_PREC_STRICTLY_LOWER_TRI>(p, qc, g, s);
    case SDCGYM_PREC_FIXED: return launch_sweeps<M, SDCGYM_PREC_FIXED, false, false>(p, s);
    }
    return SDCGYM_EUNSUPPORTED;
}

}  // namespace sdcgym

using namespace sdcgym;

extern "C" int sdcgym_residual_sweeps(const sdcgym_rho_desc* d, int64_t N, int sweeps, const double* lam,
                                      const double* qd, const double* u0, const double* u, const double* r,
                                      double* u_out, double* r_out, double* norm_out, double* grad, void* stream) {
    if (!d || !lam || !norm_out) return SDCGYM_ENULL;
    const int given = (u0 != nullptr) + (u != nullptr) + (r != nullptr);
    if (given != 0 && given != 3) return SDCGYM_ENULL;
    if (!sdcgym_supported(d->M, d->prec_type)) return SDCGYM_EUNSUPPORTED;
    if (N < 0 || sweeps < 1 || sweeps > kMaxSweeps) return SDCGYM_EINVAL;
    if (grad && d->prec_type == SDCGYM_PREC_FIXED) return SDCGYM_EUNSUPPORTED;
    if (d->prec_type != SDCGYM_PREC_FIXED && !qd) return SDCGYM_ENULL;
    if (N == 0) return 0;
    cudaStream_t s = (cudaStream_t)stream;
    switch (d->M) {
#define C(m) case m: return launch_residual_sweeps<m>(d, N, sweeps, lam, qd, u0, u, r, u_out, r_out, norm_out, grad, s);
        C(2) C(3) C(4) C(5) C(6) C(7) C(8) C(9)
#undef C
    }
    return SDCGYM_EUNSUPPORTED;
}

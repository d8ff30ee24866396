// tests/host_shim/sweeps_shim.cpp - TEST INFRASTRUCTURE ONLY.
//
// Host build of the K-sweep residual loss body (sdc_gym_b200/csrc/residual_sweeps.cuh, the header
// csrc/residual_sweeps.cu instantiates), run over host arrays one "thread" at a time, so that the CPU suite can check
// it against the mp reference.  Build: g++ -O1 -std=c++17 -fPIC -shared sweeps_shim.cpp
#include <cmath>
#include <cstdint>
using std::isnan;

#include "../../sdc_gym_b200/csrc/residual_sweeps.cuh"

using namespace sdcgym;

extern "C" int sdcgym_num_actions(int M, int prec_type) {
    switch (prec_type) {
    case SDCGYM_PREC_DIAG: return M;
    case SDCGYM_PREC_LOWER_DIAG: return M - 1;
    case SDCGYM_PREC_LOWER_TRI: return M * (M + 1) / 2;
    case SDCGYM_PREC_STRICTLY_LOWER_TRI: return M * (M - 1) / 2;
    default: return 0;
    }
}

template <int M, int PT, bool QC, bool GRAD>
static int run(const SweepParams<M>& p) {
    for (int64_t i = 0; i < p.N; i++) residual_sweeps_one<M, PT, QC, GRAD>(p, i);
    return 0;
}

template <int M, int PT>
static int run_layout(const SweepParams<M>& p, bool qc, bool grad) {
    if (qc) return grad ? run<M, PT, true, true>(p) : run<M, PT, true, false>(p);
    return grad ? run<M, PT, false, true>(p) : run<M, PT, false, false>(p);
}

template <int M>
static int sweeps_m(const sdcgym_rho_desc* d, int64_t N, int sweeps, const double* lam, const double* qd,
                    const double* u0, const double* u, const double* r, double* u_out, double* r_out, double* norm_out,
                    double* grad) {
    SweepParams<M> p;
    fill_sweep_params<M>(p, d, N, sweeps, lam, qd, u0, u, r, u_out, r_out, norm_out, grad);
    const bool qc = d->qd_is_complex != 0, g = grad != nullptr;
    switch (d->prec_type) {
    case SDCGYM_PREC_DIAG: return run_layout<M, SDCGYM_PREC_DIAG>(p, qc, g);
    case SDCGYM_PREC_LOWER_DIAG: return run_layout<M, SDCGYM_PREC_LOWER_DIAG>(p, qc, g);
    case SDCGYM_PREC_LOWER_TRI: return run_layout<M, SDCGYM_PREC_LOWER_TRI>(p, qc, g);
    case SDCGYM_PREC_STRICTLY_LOWER_TRI: return run_layout<M, SDCGYM_PREC_STRICTLY_LOWER_TRI>(p, qc, g);
    case SDCGYM_PREC_FIXED: return run<M, SDCGYM_PREC_FIXED, false, false>(p);
    }
    return -2;
}

extern "C" int shim_residual_sweeps(const sdcgym_rho_desc* d, int64_t N, int sweeps, const double* lam,
                                    const double* qd, const double* u0, const double* u, const double* r,
                                    double* u_out, double* r_out, double* norm_out, double* grad) {
    if (sweeps < 1 || sweeps > kMaxSweeps) return -1;
    switch (d->M) {
#define C(m) case m: return sweeps_m<m>(d, N, sweeps, lam, qd, u0, u, r, u_out, r_out, norm_out, grad);
        C(2) C(3) C(4) C(5) C(6) C(7) C(8) C(9)
#undef C
    }
    return -2;
}

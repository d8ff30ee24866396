// tests/host_shim/sweeps_sum_shim.cpp - TEST INFRASTRUCTURE ONLY.
//
// Host build of the per-sample contribution of sdcgym_residual_sweeps_sum (residual_sweeps_reduced in
// sdc_gym_b200/csrc/residual_sweeps.cuh, the body csrc/residual_sweeps_sum.cu sums), one "thread" at a time, so that
// the CPU suite can check each sample's value and weighted gradient against the mp reference.
// Build: g++ -O1 -std=c++17 -fPIC -shared sweeps_sum_shim.cpp
#include <cmath>
#include <cstdint>
using std::isnan;
using std::log;

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

// f[N], nK[N], gw[N][A][2]: the weighted gradient in the layout's parameter order
template <int M, int PT, bool QC>
static int run(const SweepParams<M>& p, int reduction, double* f, double* nK, double* gw) {
    for (int64_t i = 0; i < p.N; i++) {
        C2 g[M * M];
        f[i] = residual_sweeps_reduced<M, PT, QC>(p, i, C2{p.lam[2 * i] * p.dt, p.lam[2 * i + 1] * p.dt}, reduction,
                                                  nK[i], g);
        int k = 0;
        for (int a = 0; a < M; a++)
            for (int c = 0; c <= a; c++)
                if (sweep_param<PT>(a, c)) {
                    gw[(i * p.n_act + k) * 2] = g[a * M + c].r;
                    gw[(i * p.n_act + k) * 2 + 1] = g[a * M + c].i;
                    k++;
                }
    }
    return 0;
}

template <int M, int PT>
static int run_layout(const SweepParams<M>& p, bool qc, int reduction, double* f, double* nK, double* gw) {
    return qc ? run<M, PT, true>(p, reduction, f, nK, gw) : run<M, PT, false>(p, reduction, f, nK, gw);
}

template <int M>
static int reduced_m(const sdcgym_rho_desc* d, int64_t N, int sweeps, int reduction, const double* lam,
                     const double* qd, const double* u0, const double* u, const double* r, double* f, double* nK,
                     double* gw) {
    SweepParams<M> p;
    fill_sweep_params<M>(p, d, N, sweeps, lam, qd, u0, u, r, nullptr, nullptr, nullptr, nullptr);
    const bool qc = d->qd_is_complex != 0;
    switch (d->prec_type) {
    case SDCGYM_PREC_DIAG: return run_layout<M, SDCGYM_PREC_DIAG>(p, qc, reduction, f, nK, gw);
    case SDCGYM_PREC_LOWER_DIAG: return run_layout<M, SDCGYM_PREC_LOWER_DIAG>(p, qc, reduction, f, nK, gw);
    case SDCGYM_PREC_LOWER_TRI: return run_layout<M, SDCGYM_PREC_LOWER_TRI>(p, qc, reduction, f, nK, gw);
    case SDCGYM_PREC_STRICTLY_LOWER_TRI:
        return run_layout<M, SDCGYM_PREC_STRICTLY_LOWER_TRI>(p, qc, reduction, f, nK, gw);
    }
    return -2;
}

extern "C" int shim_residual_sweeps_reduced(const sdcgym_rho_desc* d, int64_t N, int sweeps, int reduction,
                                            const double* lam, const double* qd, const double* u0, const double* u,
                                            const double* r, double* f, double* nK, double* gw) {
    if (sweeps < 1 || sweeps > kMaxSweeps) return -1;
    switch (d->M) {
#define C(m) case m: return reduced_m<m>(d, N, sweeps, reduction, lam, qd, u0, u, r, f, nK, gw);
        C(2) C(3) C(4) C(5) C(6) C(7) C(8) C(9)
#undef C
    }
    return -2;
}

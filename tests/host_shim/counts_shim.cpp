// tests/host_shim/counts_shim.cpp - TEST INFRASTRUCTURE ONLY.
//
// Host build of sdcgym_full_solve_counts: full_solve_counts_kernel (sdc_gym_b200/csrc/step_kernels.cuh, step_one with
// ResetEval) with the threads of each 128-thread block run one after the other, the block's histogram counted in a
// local array and added to `hist` once per block, as on the device.  The last block runs the clamped threads
// (tid >= N) too.
// Build: g++ -O1 -std=c++17 -fPIC -shared -ffp-contract=off -mfma counts_shim.cpp
#include <cmath>
#include <cstdint>
#include <cstring>
#include <vector>
using std::isinf;
using std::isnan;

#include "../../sdc_gym_b200/csrc/step_params.cuh"

using namespace sdcgym;

template <int M>
static int counts_m(const sdcgym_env_desc* d, const sdcgym_lambda_grid* g, int64_t N, const double* lam,
                    const double* action, int64_t a_es, int64_t a_cs, int32_t* niter, double* res, uint8_t* flags,
                    double* lam_out, int64_t* hist) {
    sdcgym_state st{};
    st.N = st.ld = N;
    StepParams<M> p;
    fill_params<M>(p, d, &st);
    p.action = action;
    p.a_es = a_es;
    p.a_cs = a_cs;
    p.info_niter = niter;
    p.info_res = res;
    p.flags = flags;
    p.info_lam = lam_out;
    p.autoreset = 0;
    p.strategy = SDCGYM_REW_ITERATION_ONLY;
    ResetEval src{};
    src.lam = g ? nullptr : lam;
    if (g) {
        src.grid_re = g->n_re;
        src.grid_im = g->n_im;
        src.grid_first = g->first;
        src.re_lo = g->re_lo;
        src.re_hi = g->re_hi;
        src.im_lo = g->im_lo;
        src.im_hi = g->im_hi;
    }
    bool dense = d->prec_type != SDCGYM_PREC_DIAG;
    if (d->prec_type == SDCGYM_PREC_FIXED) {
        bool diagonal = true;
        for (int r = 0; r < M; r++)
            for (int c = 0; c < M; c++)
                if (r != c && d->Qd_fixed[r * M + c] != 0.0) diagonal = false;
        dense = !diagonal;
    }
    constexpr int HD = HoldPolicy<M>::diag, HS = HoldPolicy<M>::dense;
    const int nbins = d->max_iters + 3;
    if (hist) std::memset(hist, 0, sizeof(int64_t) * nbins);
    std::vector<int> block_hist(nbins);
    double side[4 * M * M];  // the shared-memory side store of one thread (stride 2)
    cplx pside[2 * 2 * M * M];
    for (int64_t b0 = 0; b0 < N; b0 += kBlock) {
        std::fill(block_hist.begin(), block_hist.end(), 0);
        src.hist = hist ? block_hist.data() : nullptr;
        for (int64_t tid = b0; tid < b0 + kBlock; tid++) {
            if (d->blas_variant == 0) {
                if (dense) step_one<M, 0, 0, true, HS, NoAfterLoads, 0, ResetEval>(p, tid, side, 2, pside, 2, nullptr, NoAfterLoads(), 0, src);
                else step_one<M, 0, 0, false, HD, NoAfterLoads, 0, ResetEval>(p, tid, side, 2, pside, 2, nullptr, NoAfterLoads(), 0, src);
            } else {
                if (dense) step_one<M, 0, 1, true, HS, NoAfterLoads, 0, ResetEval>(p, tid, side, 2, pside, 2, nullptr, NoAfterLoads(), 0, src);
                else step_one<M, 0, 1, false, HD, NoAfterLoads, 0, ResetEval>(p, tid, side, 2, pside, 2, nullptr, NoAfterLoads(), 0, src);
            }
        }
        if (hist)
            for (int k = 0; k < nbins; k++) hist[k] += block_hist[k];
    }
    return 0;
}

extern "C" int shim_full_solve_counts(const sdcgym_env_desc* d, const sdcgym_lambda_grid* g, int64_t N,
                                      const double* lam, const double* action, int64_t a_es, int64_t a_cs,
                                      int32_t* niter, double* res, uint8_t* flags, double* lam_out, int64_t* hist) {
    switch (d->M) {
#define C(m) case m: return counts_m<m>(d, g, N, lam, action, a_es, a_cs, niter, res, flags, lam_out, hist);
        C(2) C(3) C(4) C(5) C(6) C(7) C(8) C(9)
#undef C
    }
    return -2;
}

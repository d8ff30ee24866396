// tests/host_shim/shim.cpp - TEST INFRASTRUCTURE ONLY.
//
// Compiles the very templates the CUDA kernels instantiate (sdc_gym_b200/csrc/*.cuh: step_one, reset_one,
// rho_one, cinv_exact, ...) for the host with g++, and runs them over host arrays one "thread" at a time.
// This lets the CPU-only test suite (`-m "not gpu"`) catch logic errors in the kernel bodies before GPU time
// is spent.  It is never loaded by the sdc_gym_b200 package and is not a fallback: same C ABI structs,
// symbols prefixed `shim_`.
//
// Build: g++ -O1 -std=c++17 -fPIC -shared -ffp-contract=off -mfma -x c++ shim.cpp  (tests/host_shim/build.py)
#include <cstdint>
#include <cstring>
#include <cmath>
using std::isnan;
using std::isinf;

#include "../../sdc_gym_b200/csrc/step_params.cuh"
#include "../../sdc_gym_b200/csrc/specrad.cuh"

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

template <int M>
static int reset_m(const sdcgym_env_desc* d, const sdcgym_state* st, const double* lam_in, const uint8_t* mask,
                   double* old_states) {
    StepParams<M> p;
    fill_params<M>(p, d, st);
    p.lam_in = lam_in;
    p.mask = mask;
    p.old_states = old_states;
    for (int64_t i = 0; i < p.N; i++) {
        if (d->blas_variant == 0) reset_one<M, 0>(p, i);
        else reset_one<M, 1>(p, i);
    }
    return 0;
}

template <int M>
static int step_m(const sdcgym_env_desc* d, const sdcgym_state* st, const sdcgym_step_io* io) {
    StepParams<M> p;
    fill_params<M>(p, d, st);
    fill_step_io<M>(p, io);
    bool dense = d->prec_type != SDCGYM_PREC_DIAG;
    const bool full = d->env_kind == SDCGYM_ENV_FULL;
    if (d->prec_type == SDCGYM_PREC_FIXED) {
        bool diagonal = true;
        for (int r = 0; r < M; r++)
            for (int c = 0; c < M; c++)
                if (r != c && d->Qd_fixed[r * M + c] != 0.0) diagonal = false;
        dense = !diagonal;
    }
    constexpr int HD = HoldPolicy<M>::diag, HS = HoldPolicy<M>::dense;
    // emulate whole thread blocks so the i >= N clamping path is exercised too
    const int64_t nthreads = (p.N + kBlock - 1) / kBlock * kBlock;
    double side[4 * M * M];  // stands in for the shared-memory side store of HOLD >= 3 (stride 2 to catch stride bugs)
    constexpr int HV1 = HoldPolicy<M>::step;
    cplx pside[2 * 2 * M * M];  // complex side store of HOLD == 5 (stride 2)
    for (int64_t i = 0; i < nthreads; i++) {
        if (d->blas_variant == 0) {
            if (full) { if (dense) step_one<M, 0, 0, true, HS>(p, i, side, 2, pside, 2); else step_one<M, 0, 0, false, HD>(p, i, side, 2, pside, 2); }
            else      { if (dense) step_one<M, 1, 0, true, HS>(p, i, side, 2, pside, 2); else step_one<M, 1, 0, false, HV1>(p, i, side, 2, pside, 2); }
        } else {
            if (full) { if (dense) step_one<M, 0, 1, true, HS>(p, i, side, 2, pside, 2); else step_one<M, 0, 1, false, HD>(p, i, side, 2, pside, 2); }
            else      { if (dense) step_one<M, 1, 1, true, HS>(p, i, side, 2, pside, 2); else step_one<M, 1, 1, false, HV1>(p, i, side, 2, pside, 2); }
        }
    }
    return 0;
}


// phased dense full solve (step_one PHASE), the pass sequence of launch_phased_dense (csrc/step_inst.cu) with the
// "threads" of every pass run one after the other; needs sdcgym_state.phase_*
template <int M>
static int step_phased_m(const sdcgym_env_desc* d, const sdcgym_state* st, const sdcgym_step_io* io, const int* stops,
                         int nstops, int split) {
    if constexpr (M <= 7) {
        StepParams<M> p;
        fill_params<M>(p, d, st);
        fill_step_io<M>(p, io);
        if (!p.cont_list || !p.cont_count || !p.pinv_scratch || nstops < 1) return -3;
        constexpr int HS = HoldPolicy<M>::dense;
        double side[3 * 2 * M * M];  // stride 3
        cplx pside[3 * 2 * M * M];
        int32_t* const lists = p.cont_list;
        int32_t* const counts = p.cont_count;
        for (int k = 0; k < SDCGYM_PHASE_COUNTERS; k++) counts[k] = 0;
        const int64_t nthreads = (p.N + kBlock - 1) / kBlock * kBlock;
        p.it_stop = stops[0];
        p.min_lanes = 33;  // at the sweep count, whatever the occupancy (the host build has no warps)
        p.cont_count = counts;
        if (split) {  // inverse_kernel, then the first sweeps with the inverse reloaded
            for (int64_t i = 0; i < nthreads; i++) {
                if (d->blas_variant == 0) step_one<M, 0, 0, true, 0, NoAfterLoads, 3>(p, i);
                else step_one<M, 0, 1, true, 0, NoAfterLoads, 3>(p, i);
            }
            for (int64_t i = 0; i < nthreads; i++) {
                if (d->blas_variant == 0) step_one<M, 0, 0, true, HS, NoAfterLoads, 4>(p, i, side, 3, pside, 3);
                else step_one<M, 0, 1, true, HS, NoAfterLoads, 4>(p, i, side, 3, pside, 3);
            }
        } else {
            for (int64_t i = 0; i < nthreads; i++) {
                if (d->blas_variant == 0) step_one<M, 0, 0, true, HS, NoAfterLoads, 1>(p, i, side, 3, pside, 3);
                else step_one<M, 0, 1, true, HS, NoAfterLoads, 1>(p, i, side, 3, pside, 3);
            }
        }
        for (int j = 1; j <= nstops; j++) {
            if (stops[j - 1] >= p.max_iters) break;
            p.it_stop = (j < nstops) ? stops[j] : 0x7fffffff;
            p.min_lanes = (j < nstops) ? 33 : 0;
            p.cont_list = lists + (int64_t)(j & 1) * p.N;
            p.cont_count = counts + j;
            const int32_t* in = lists + (int64_t)((j - 1) & 1) * p.N;
            const int64_t n = counts[j - 1], nt = (n + kBlock - 1) / kBlock * kBlock;
            for (int64_t t = 0; t < nt; t++) {
                const int64_t idx = t < n ? (int64_t)in[t] : p.N;
                if (d->blas_variant == 0) step_one<M, 0, 0, true, HS, NoAfterLoads, 2>(p, idx, side, 3, pside, 3);
                else step_one<M, 0, 1, true, HS, NoAfterLoads, 2>(p, idx, side, 3, pside, 3);
            }
        }
        return 0;
    }
    return -2;
}
extern "C" int shim_step_phased(const sdcgym_env_desc* d, const sdcgym_state* st, const sdcgym_step_io* io,
                                const int* stops, int nstops, int split) {
    if (d->env_kind != SDCGYM_ENV_FULL) return -2;
    switch (d->M) {
    case 2: return step_phased_m<2>(d, st, io, stops, nstops, split);
    case 3: return step_phased_m<3>(d, st, io, stops, nstops, split);
    case 4: return step_phased_m<4>(d, st, io, stops, nstops, split);
    case 5: return step_phased_m<5>(d, st, io, stops, nstops, split);
    case 6: return step_phased_m<6>(d, st, io, stops, nstops, split);
    case 7: return step_phased_m<7>(d, st, io, stops, nstops, split);
    }
    return -2;
}

extern "C" int shim_reset(const sdcgym_env_desc* d, const sdcgym_state* st, const double* lam_in, const uint8_t* mask,
                          double* old_states) {
    switch (d->M) {
    case 2: return reset_m<2>(d, st, lam_in, mask, old_states);
    case 3: return reset_m<3>(d, st, lam_in, mask, old_states);
    case 4: return reset_m<4>(d, st, lam_in, mask, old_states);
    case 5: return reset_m<5>(d, st, lam_in, mask, old_states);
    case 6: return reset_m<6>(d, st, lam_in, mask, old_states);
    case 7: return reset_m<7>(d, st, lam_in, mask, old_states);
    case 8: return reset_m<8>(d, st, lam_in, mask, old_states);
    case 9: return reset_m<9>(d, st, lam_in, mask, old_states);
    }
    return -2;
}

extern "C" int shim_step(const sdcgym_env_desc* d, const sdcgym_state* st, const sdcgym_step_io* io) {
    switch (d->M) {
    case 2: return step_m<2>(d, st, io);
    case 3: return step_m<3>(d, st, io);
    case 4: return step_m<4>(d, st, io);
    case 5: return step_m<5>(d, st, io);
    case 6: return step_m<6>(d, st, io);
    case 7: return step_m<7>(d, st, io);
    case 8: return step_m<8>(d, st, io);
    case 9: return step_m<9>(d, st, io);
    }
    return -2;
}

// ---- the shared-memory formulation of the large dense kernels (HOLD 5), not selected by HoldPolicy but kept
//      parity-tested ----
template <int M>
static int step_m_hold5(const sdcgym_env_desc* d, const sdcgym_state* st, const sdcgym_step_io* io) {
    if constexpr (M > kRegInvMaxM) {
        StepParams<M> p;
        fill_params<M>(p, d, st);
        fill_step_io<M>(p, io);
        cplx pside[3 * 2 * M * M];  // stride 3
        for (int64_t i = 0; i < p.N; i++) {
            if (d->env_kind == SDCGYM_ENV_FULL) step_one<M, 0, 0, true, 5>(p, i, nullptr, 1, pside, 3);
            else step_one<M, 1, 0, true, 5>(p, i, nullptr, 1, pside, 3);
        }
        return 0;
    }
    return -2;
}
template <int M>
static int step_m_hold9(const sdcgym_env_desc* d, const sdcgym_state* st, const sdcgym_step_io* io) {
    StepParams<M> p;
    fill_params<M>(p, d, st);
    fill_step_io<M>(p, io);
    double side[3 * 2 * M * M];  // stride 3
    for (int64_t i = 0; i < p.N; i++) {
        if (d->env_kind == SDCGYM_ENV_FULL) step_one<M, 0, 0, true, 9>(p, i, side, 3);
        else step_one<M, 1, 0, true, 9>(p, i, side, 3);
    }
    return 0;
}
extern "C" int shim_step_hold9(const sdcgym_env_desc* d, const sdcgym_state* st, const sdcgym_step_io* io) {
    switch (d->M) {
    case 8: return step_m_hold9<8>(d, st, io);
    case 9: return step_m_hold9<9>(d, st, io);
    }
    return -2;
}

extern "C" int shim_step_hold5(const sdcgym_env_desc* d, const sdcgym_state* st, const sdcgym_step_io* io) {
    switch (d->M) {
    case 8: return step_m_hold5<8>(d, st, io);
    case 9: return step_m_hold5<9>(d, st, io);
    }
    return -2;
}

// ---- spectral radius ----
#include "../../sdc_gym_b200/csrc/specrad_params.cuh"

template <int M>
static int rho_m(const sdcgym_rho_desc* d, int64_t N, const double* lam, const double* qd, double* rho) {
    RhoParams<M> p;
    fill_rho_params<M>(p, d, N, lam, qd, rho);
    for (int64_t i = 0; i < N; i++) rho_one<M>(p, i);
    return 0;
}

extern "C" int shim_spectral_radius(const sdcgym_rho_desc* d, int64_t N, const double* lam, const double* qd, double* rho) {
    switch (d->M) {
    case 2: return rho_m<2>(d, N, lam, qd, rho);
    case 3: return rho_m<3>(d, N, lam, qd, rho);
    case 4: return rho_m<4>(d, N, lam, qd, rho);
    case 5: return rho_m<5>(d, N, lam, qd, rho);
    case 6: return rho_m<6>(d, N, lam, qd, rho);
    case 7: return rho_m<7>(d, N, lam, qd, rho);
    case 8: return rho_m<8>(d, N, lam, qd, rho);
    case 9: return rho_m<9>(d, N, lam, qd, rho);
    }
    return -2;
}

// ---- direct access to the exact inverse template (row-major complex in/out) ----
template <int M>
static void cinv_m(const double* P, double* out, int variant) {
    if (variant >= 2) {  // register-resident formulation (exact_inv_reg.cuh)
        double Ar[M * M], Ai[M * M], Br[M * M], Bi[M * M];
        for (int r = 0; r < M; r++)
            for (int c = 0; c < M; c++) {
                Ar[r + c * M] = P[(r * M + c) * 2];
                Ai[r + c * M] = P[(r * M + c) * 2 + 1];
            }
        if (variant == 2) cinv_exact_reg<M, 0>(Ar, Ai, Br, Bi);
        else cinv_exact_reg<M, 1>(Ar, Ai, Br, Bi);
        for (int r = 0; r < M; r++)
            for (int c = 0; c < M; c++) {
                out[(r * M + c) * 2] = Br[r + c * M];
                out[(r * M + c) * 2 + 1] = Bi[r + c * M];
            }
        return;
    }
    cplx A[M * M], B[M * M];
    for (int r = 0; r < M; r++)
        for (int c = 0; c < M; c++) A[r + c * M] = cplx{P[(r * M + c) * 2], P[(r * M + c) * 2 + 1]};
    if (variant == 0) cinv_exact<M, 0>(A, B);
    else cinv_exact<M, 1>(A, B);
    for (int r = 0; r < M; r++)
        for (int c = 0; c < M; c++) {
            out[(r * M + c) * 2] = B[r + c * M].re;
            out[(r * M + c) * 2 + 1] = B[r + c * M].im;
        }
}
extern "C" int shim_cinv(int M, const double* P, double* out, int variant) {
    switch (M) {
    case 2: cinv_m<2>(P, out, variant); return 0;
    case 3: cinv_m<3>(P, out, variant); return 0;
    case 4: cinv_m<4>(P, out, variant); return 0;
    case 5: cinv_m<5>(P, out, variant); return 0;
    case 6: cinv_m<6>(P, out, variant); return 0;
    case 7: cinv_m<7>(P, out, variant); return 0;
    case 8: cinv_m<8>(P, out, variant); return 0;
    case 9: cinv_m<9>(P, out, variant); return 0;
    }
    return -2;
}

template <int M>
static int rho_grad_m(const sdcgym_rho_desc* d, int64_t N, const double* lam, const double* qd, double* rho, double* grad) {
    RhoParams<M> p;
    fill_rho_params<M>(p, d, N, lam, qd, rho);
    for (int64_t i = 0; i < N; i++) rho_grad_one<M>(p, i, grad);
    return 0;
}
extern "C" int shim_spectral_radius_grad(const sdcgym_rho_desc* d, int64_t N, const double* lam, const double* qd,
                                         double* rho, double* grad) {
    switch (d->M) {
    case 2: return rho_grad_m<2>(d, N, lam, qd, rho, grad);
    case 3: return rho_grad_m<3>(d, N, lam, qd, rho, grad);
    case 4: return rho_grad_m<4>(d, N, lam, qd, rho, grad);
    case 5: return rho_grad_m<5>(d, N, lam, qd, rho, grad);
    case 6: return rho_grad_m<6>(d, N, lam, qd, rho, grad);
    case 7: return rho_grad_m<7>(d, N, lam, qd, rho, grad);
    case 8: return rho_grad_m<8>(d, N, lam, qd, rho, grad);
    case 9: return rho_grad_m<9>(d, N, lam, qd, rho, grad);
    }
    return -2;
}

// ---- certified substitution sweep mode (fast_kernels.cuh): certificate + fast step (+ per-sweep trace of r~ and the
//      margin for the bound-dominance property test) + the exact kernel over the fallback list ----
#include "../../sdc_gym_b200/csrc/fast_kernels.cuh"

template <int M>
static int step_certified_m(const sdcgym_env_desc* d, const sdcgym_state* st, const sdcgym_step_io* io, double* trace,
                            int run_fallback) {
    StepParams<M> p;
    fill_params<M>(p, d, st);
    fill_step_io<M>(p, io);
    FastWork fw{st->cert, st->fallback_list, st->fallback_count};
    fw.count[0] = 0;
    const int64_t nthreads = (p.N + kBlock - 1) / kBlock * kBlock;
    for (int64_t i = 0; i < p.N; i++) {
        if (d->blas_variant == 0) cert_one<M, 0>(p, fw, i);
        else cert_one<M, 1>(p, fw, i);
    }
    const size_t tstride = (size_t)d->max_iters * (2 * M + 2);
    for (int64_t i = 0; i < nthreads; i++) {
        double* t = (trace && i < p.N) ? trace + (size_t)i * tstride : nullptr;
        if (d->blas_variant == 0) fast_step_one<M, 0, true>(p, fw, i, t);
        else fast_step_one<M, 1, true>(p, fw, i, t);
    }
    if (run_fallback) {
        constexpr int HD = HoldPolicy<M>::diag;
        double side[4 * M * M];
        cplx pside[2 * 2 * M * M];
        const int count = fw.count[0];
        fw.count[1] += count;
        for (int t = 0; t < count; t++) {
            const int64_t idx = fw.list[t];
            if (d->blas_variant == 0) step_one<M, 0, 0, false, HD>(p, idx, side, 2, pside, 2);
            else step_one<M, 0, 1, false, HD>(p, idx, side, 2, pside, 2);
        }
    }
    return 0;
}

extern "C" int shim_step_certified(const sdcgym_env_desc* d, const sdcgym_state* st, const sdcgym_step_io* io,
                                   double* trace, int run_fallback) {
    switch (d->M) {
    case 2: return step_certified_m<2>(d, st, io, trace, run_fallback);
    case 3: return step_certified_m<3>(d, st, io, trace, run_fallback);
    case 4: return step_certified_m<4>(d, st, io, trace, run_fallback);
    case 5: return step_certified_m<5>(d, st, io, trace, run_fallback);
    case 6: return step_certified_m<6>(d, st, io, trace, run_fallback);
    case 7: return step_certified_m<7>(d, st, io, trace, run_fallback);
    case 8: return step_certified_m<8>(d, st, io, trace, run_fallback);
    case 9: return step_certified_m<9>(d, st, io, trace, run_fallback);
    }
    return -2;
}

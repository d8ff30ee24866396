// step_kernels.cuh - the SDC env kernels: reset, step (sdc-v0 full solve / sdc-v1 single sweep) with fused
// reward, convergence logic and DummyVecEnv-style auto-reset.  One env per thread; u, r, lambda*dt, the
// preconditioner inverse and (for small M) the whole system matrix C live in registers; the collocation
// matrix Q arrives as a __grid_constant__ kernel parameter, i.e. in the constant bank, so every Q entry is
// an immediate constant operand of the DMUL that uses it.  No shared memory, no memory traffic inside the
// sweep loop.
//
// Reference statements reproduced (sdc_gym/envs/sdc_env.py): reset :306-332, step (sdc-v0) :209-273,
// step (sdc-v1) :507-572, _scale_action :125-132, _get_prec :134-191, _compute_pinv :193-201, rewards
// :334-463.  Rounding sequence: SURVEY.md Appendix A / A.2 (exact_math.cuh).
#pragma once
#include "../../include/sdcgym.h"
#include "exact_math.cuh"
#include "fast_div.cuh"
#include "exact_inv_reg.cuh"
#include "philox.cuh"

namespace sdcgym {

constexpr int kBlock = 128;
constexpr int kRegInvMaxM = 7;  // largest M whose exact inverse runs on register-resident LU factors (exact_inv_reg.cuh)

template <int M>
struct StepParams {
    double Q[M * M];
    double Qd[M * M];  // fixed real Q_delta (SDCGYM_PREC_FIXED)
    int64_t N, ld;
    double* lam;
    double* S;
    double* resnorm;
    int32_t* niter;
    int32_t* episodes;
    uint32_t* rng_ctr;
    double* norm_init;  // optional plane: scaled norm of the episode's initial residual (sdcgym_state.norm_init)
    const double* action;
    int64_t a_es, a_cs;
    double* reward;
    uint8_t* flags;
    double* info_res;
    int32_t* info_niter;
    double* info_lam;
    double* term;
    double* old_states;
    const double* lam_in;  // reset only
    const uint8_t* mask;   // reset only
    double dt, restol, step_penalty, residual_weight, norm_factor;
    double re_lo, re_hi, im_lo, im_hi, ix0, ix1;
    uint64_t seed;
    int64_t env_offset;
    int32_t prec_type, is_complex, do_scale, max_iters, strategy, autoreset, curriculum;
    double log_restol_nf;  // math.log(restol * norm_factor) (sdc_env.py:346), evaluated once on the host
    // phased full solve (dense Q_delta, see step_one PHASE): sweep count at which a pass hands its unfinished envs over
    int32_t it_stop;
    int32_t min_lanes;     // ... and only while fewer than this many lanes of the warp are still iterating (33: always)
    int32_t* cont_list;    // [<= N] indices of the envs this pass suspended (next pass's work list)
    int32_t* cont_count;   // [1] length of cont_list (zeroed before the first pass)
    double* pinv_scratch;  // [2 M^2][ld] inverse of P of the suspended envs (plane 2k: Re, 2k+1: Im of entry k = row*M+col)
};

// Where a step reads its per-env inputs from.  Default (nullptr): the global planes of StepParams, element `i`.  The
// streaming sdc-v1 kernel (stream_kernels.cuh) stages a whole tile of envs in shared memory with bulk asynchronous
// copies and points these at the staged copy (plane stride `ld`, element `i` within the tile); outputs always go to
// the global planes.
struct StepInputs {
    const double* lam;        // [2][ld]
    const double* S;          // [4M][ld]
    const double* resnorm;    // [ld]
    const int32_t* niter;     // [ld]
    const int32_t* episodes;  // [ld]
    const uint32_t* rng_ctr;  // [ld]
    const double* norm_init;  // [ld] or nullptr
    const double* action;     // env-major rows, same strides as StepParams::a_es / a_cs; nullptr: no actions
    int64_t ld;
    int64_t i;
};

// ---- C = eye(M) - (lam*dt)*Q, one row (sdc_env.py:302-304; Appendix A step 2).  0 - x is written -x
//      (differs only in the sign of an exact zero). ----
template <int M>
SDCGYM_HD void c_row(const double (&Q)[M * M], double zr, double zi, int i, double (&cr)[M],
                                      double (&ci)[M]) {
#pragma unroll
    for (int j = 0; j < M; j++) {
        double q = Q[i * M + j];
        cr[j] = (i == j) ? dsub(1.0, dmul(zr, q)) : -dmul(zr, q);
        ci[j] = -dmul(zi, q);
    }
}

// ---- lambda draw (sdc_env.py:282-300): real part first, then imaginary part ----
template <int M>
SDCGYM_HD void draw_lambda(const StepParams<M>& p, int64_t i, uint32_t ctr, int32_t episodes,
                                            double& lr, double& li) {
    uint64_t g = (uint64_t)(p.env_offset + i);
    philox4 x = philox4x32_10((uint32_t)g, (uint32_t)(g >> 32), ctr, 0u, (uint32_t)p.seed, (uint32_t)(p.seed >> 32));
    double lo = p.re_lo;
    if (p.curriculum) {
        // np.interp(num_episodes, interval, reversed(lambda_real_interval))
        double x0 = p.ix0, x1 = p.ix1, e = (double)episodes;
        if (e <= x0) lo = p.re_hi;
        else if (e >= x1) lo = p.re_lo;
        else {
            double slope = ddiv(dsub(p.re_lo, p.re_hi), dsub(x1, x0));
            lo = dadd(dmul(slope, dsub(e, x0)), p.re_hi);
        }
    }
    lr = dadd(lo, dmul(dsub(p.re_hi, lo), u53(x.v[0], x.v[1])));
    li = dadd(p.im_lo, dmul(dsub(p.im_hi, p.im_lo), u53(x.v[2], x.v[3])));
}

// ---- initial state of an episode: u = 1, r = u0 - C @ u (sdc_env.py:306-314) ----
template <int M, int V>
SDCGYM_HD void initial_state(const double (&Q)[M * M], double zr, double zi, double (&ur)[M],
                                              double (&ui)[M], double (&rr)[M], double (&ri)[M]) {
#pragma unroll
    for (int m = 0; m < M; m++) {
        ur[m] = 1.0;
        ui[m] = 0.0;
    }
#pragma unroll
    for (int m = 0; m < M; m++) {
        double cr[M], ci[M], yr, yi;
        c_row<M>(Q, zr, zi, m, cr, ci);
        zgemv_rowdot<M, V>(cr, ci, ur, ui, yr, yi);
        rr[m] = dsub(1.0, yr);
        ri[m] = -yi;
    }
}

template <int M>
SDCGYM_HD void store_state(double* __restrict__ S, int64_t ld, int64_t i, const double (&ur)[M],
                                            const double (&ui)[M], const double (&rr)[M], const double (&ri)[M]) {
#pragma unroll
    for (int m = 0; m < M; m++) {
        S[(2 * m) * ld + i] = ur[m];
        S[(2 * m + 1) * ld + i] = ui[m];
        S[(2 * M + 2 * m) * ld + i] = rr[m];
        S[(2 * M + 2 * m + 1) * ld + i] = ri[m];
    }
}

// collect_states buffer (reference layout (2M, max_iters) complex128 per env): write column `col`
template <int M>
SDCGYM_HD void store_column(double* __restrict__ os, int64_t e, int max_iters, int col,
                                             const double (&ur)[M], const double (&ui)[M], const double (&rr)[M],
                                             const double (&ri)[M]) {
    double* base = os + (size_t)e * (2 * M) * max_iters * 2;
#pragma unroll
    for (int m = 0; m < M; m++) {
        double* pu = base + ((size_t)m * max_iters + col) * 2;
        double* pr = base + ((size_t)(M + m) * max_iters + col) * 2;
        pu[0] = ur[m];
        pu[1] = ui[m];
        pr[0] = rr[m];
        pr[1] = ri[m];
    }
}

template <int M>
SDCGYM_HD double scaled_inf_norm(const double (&vr)[M], const double (&vi)[M], double nf) {
    double tr[M], ti[M];
#pragma unroll
    for (int m = 0; m < M; m++) {
        tr[m] = dmul(vr[m], nf);  // numpy complex * real scalar
        ti[m] = dmul(vi[m], nf);
    }
    // same value as inf_norm (abs(v).max()): numpy's |.| is evaluated only for the node that provably attains the
    // maximum (one division + square root instead of M of them)
    return inf_norm_fast<M>(tr, ti);
}

// the norm_init plane (when present) is written by every reset: ||r0||inf scaled by norm_factor.  `plain` is ||r0||inf.
template <int M>
SDCGYM_HD void store_norm_init(const StepParams<M>& p, int64_t i, const double (&rr)[M], const double (&ri)[M], double plain) {
    if (p.norm_init) p.norm_init[i] = (p.norm_factor == 1.0) ? plain : scaled_inf_norm<M>(rr, ri, p.norm_factor);
}

// =====================================================================================================
// reset kernel
// =====================================================================================================
template <int M, int V>
SDCGYM_HD void reset_one(const StepParams<M>& p, int64_t i) {
    if (i >= p.N) return;
    if (p.mask && !p.mask[i]) return;
    int32_t ep = p.episodes[i] + 1;
    p.episodes[i] = ep;
    p.niter[i] = 0;
    double lr, li;
    if (p.lam_in) {
        lr = p.lam_in[i];
        li = p.lam_in[p.ld + i];
    } else {
        uint32_t ctr = p.rng_ctr[i];
        draw_lambda<M>(p, i, ctr, ep, lr, li);
        p.rng_ctr[i] = ctr + 1;
    }
    p.lam[i] = lr;
    p.lam[p.ld + i] = li;
    double zr = dmul(lr, p.dt), zi = dmul(li, p.dt);
    double ur[M], ui[M], rr[M], ri[M];
    initial_state<M, V>(p.Q, zr, zi, ur, ui, rr, ri);
    store_state<M>(p.S, p.ld, i, ur, ui, rr, ri);
    const double n0 = inf_norm_fast<M>(rr, ri);
    p.resnorm[i] = n0;
    store_norm_init<M>(p, i, rr, ri, n0);
    if (p.old_states) {
        store_column<M>(p.old_states, i, p.max_iters, 0, ur, ui, rr, ri);
        double* base = p.old_states + (size_t)i * (2 * M) * p.max_iters * 2;
        for (int row = 0; row < 2 * M; row++)
            for (int c = 1; c < p.max_iters; c++) {
                base[((size_t)row * p.max_iters + c) * 2] = 0.0;
                base[((size_t)row * p.max_iters + c) * 2 + 1] = 0.0;
            }
    }
}

// =====================================================================================================
// rewards (sdc_env.py:334-463), evaluated once per env after the sweeps
// =====================================================================================================
template <int M>
SDCGYM_HD_NOINLINE double reward_func(int strategy, double sp, double rw, double nf, double restol, int max_iters,
                                           double norm_old_scaled, double norm_init_scaled, const double (&rr)[M],
                                           const double (&ri)[M], double nr, bool converged, int steps,
                                           double log_restol_nf) {
    switch (strategy) {
    case SDCGYM_REW_ITERATION_ONLY:
        return dmul((double)(-steps), sp);
    case SDCGYM_REW_RESIDUAL_CHANGE: {
        double b = (nf == 1.0) ? nr : scaled_inf_norm<M>(rr, ri, nf);
        double rew = fabs(ddiv(dsub(log(norm_old_scaled), log(b)), dsub(log(norm_init_scaled), log_restol_nf)));
        rew = dmul(rew, rw);
        rew = dsub(rew, dmul((double)steps, sp));
        return rew;
    }
    case SDCGYM_REW_GAUSS_KERNEL: {
        double ginv = ddiv(1.0, restol);
        double x = dmul(nr, ginv);
        double gd = exp(ddiv(-dmul(x, x), 2.0));
        double extra = 1.0;
        if (converged) {
            double k = (double)(max_iters + 1 - steps);
            extra = dmul(dmul(k, k), 10.0);
        }
        return dmul(gd, extra);
    }
    case SDCGYM_REW_FAST_CONVERGENCE:
    case SDCGYM_REW_SMOOTH_FAST_CONVERGENCE:
    case SDCGYM_REW_SMOOTHER_FAST_CONVERGENCE: {
        double extra = 1.0;
        if (converged) {
            double k = (double)(max_iters + 1 - steps);
            extra = dmul(dmul(k, k), 10.0);
        }
        double rew = (nr == 0.0) ? 1000.0 : -log(nr);
        if (strategy == SDCGYM_REW_SMOOTH_FAST_CONVERGENCE && rew > 1.0) rew = dadd(1.0, log(rew));
        rew = dmul(rew, extra);
        if (strategy == SDCGYM_REW_SMOOTHER_FAST_CONVERGENCE && rew > 1.0) rew = dadd(1.0, log(rew));
        return rew;
    }
    default:
        return d_nan();
    }
}

// Integer-pipe classification thresholds for "is ||r||inf < t ?" / "is ||r||inf > t ?" decisions.
// With H = absmax_hi(r):  Lmax in [from_hi(H), from_hi(H+1)),  Lmax <= ||r||inf <= 1.4143 * Lmax.
struct HiBand {
    int lo;  // H <= lo  =>  ||r||inf <  t   for sure
    int hi;  // H >= hi  =>  ||r||inf >  t   for sure (and >= t)
};
SDCGYM_HD HiBand make_band(double t) {
    HiBand b;
    if (!(t >= 0.0) || isinf(t)) {  // NaN / negative / inf threshold: always take the exact path
        b.lo = -1;
        b.hi = 0x7fffffff;
    } else {
        b.lo = hi_word(ddiv(t, 1.4143)) - 2;
        b.hi = hi_word(t) + 1;
    }
    return b;
}

// =====================================================================================================
// step kernel.  KIND: SDCGYM_ENV_FULL / SDCGYM_ENV_STEP.  DENSE: Pinv is a full M x M matrix obtained by
// the exact np.linalg.inv emulation (any non-diagonal Q_delta), otherwise Pinv is diagonal (prec=None,
// diag actions).  HOLD: 2 = keep Re and Im of C in registers, 1 = only Re (Im re-derived from the constant bank),
// 0 = recompute z*q on use, 3 = Re in registers and Im in shared memory (`side`, element k of this thread at
// side[k * side_stride]; the LDS run on the memory pipe beside the saturated FP64 pipe), 4 = Re and Im in shared
// memory, 5 (dense kernels with M > kRegInvMaxM) = C *and* the M x M inverse in shared memory as complex pairs
// (`pside`: elements [0, M^2) hold the LU work matrix during the inverse and C afterwards, [M^2, 2 M^2) hold Pinv).
// =====================================================================================================
#ifdef __CUDA_ARCH__
#define SDCGYM_WARP_ANY(x) __any_sync(0xffffffffu, (x))
#else
#define SDCGYM_WARP_ANY(x) (x)
#endif

// one 128-bit shared-memory load of a (re, im) pair; volatile so that it stays a load inside the sweep loop
SDCGYM_HD cplx ld_pair(const cplx* p) {
#ifdef __CUDA_ARCH__
    cplx v;
    asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v.re), "=d"(v.im) : "r"((unsigned)__cvta_generic_to_shared(p)));
    return v;
#else
    return *p;
#endif
}

// ---- tensor memory (TMEM) as a per-thread scratch store (HOLD 10) ----
// TMEM is 128 lanes x 512 32-bit columns per SM, read and written with tcgen05.ld / tcgen05.st: warp w of a CTA reaches
// lanes 32 (w % 4) ... + 31, thread t of the warp its own lane.  A thread's (re, im) pair is four consecutive columns.
// All of these are .sync.aligned: the whole warp must execute them together.
#ifdef __CUDA_ARCH__
__device__ __forceinline__ void tmem_st_pair(uint32_t taddr, double re, double im) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "r"(__double2loint(re)),
                 "r"(__double2hiint(re)), "r"(__double2loint(im)), "r"(__double2hiint(im))
                 : "memory");
}
__device__ __forceinline__ void tmem_ld_pair(uint32_t taddr, int (&w)[4]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3])
                 : "r"(taddr)
                 : "memory");
}
template <int N>
__device__ __forceinline__ void tmem_ld_cols(uint32_t taddr, int* w) {  // N = 4, 8 or 16 consecutive columns
    static_assert(N == 4 || N == 8 || N == 16, "");
    if constexpr (N == 4) {
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
                     : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3])
                     : "r"(taddr)
                     : "memory");
    } else if constexpr (N == 8) {
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                     : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3]), "=r"(w[4]), "=r"(w[5]), "=r"(w[6]), "=r"(w[7])
                     : "r"(taddr)
                     : "memory");
    } else {
        asm volatile(
            "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
            : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3]), "=r"(w[4]), "=r"(w[5]), "=r"(w[6]), "=r"(w[7]), "=r"(w[8]),
              "=r"(w[9]), "=r"(w[10]), "=r"(w[11]), "=r"(w[12]), "=r"(w[13]), "=r"(w[14]), "=r"(w[15])
            : "r"(taddr)
            : "memory");
    }
}
// one row of C (M pairs = 4 M columns) in as few loads as the power-of-two shapes allow
template <int M>
__device__ __forceinline__ void tmem_ld_row(uint32_t taddr, int (&w)[4 * M]) {
    constexpr int n = 4 * M;
    int done = 0;
    if constexpr (n >= 16) {
        tmem_ld_cols<16>(taddr, w);
        done = 16;
    }
    if constexpr ((n & 15) >= 8) {
        tmem_ld_cols<8>(taddr + (n & ~15), w + (n & ~15));
        done += 8;
    }
    if constexpr ((n & 7) >= 4) tmem_ld_cols<4>(taddr + (n & ~7), w + (n & ~7));
    (void)done;
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
#endif

struct NoAfterLoads {
    SDCGYM_HD void operator()() const {}
};

// Where a full solve starts from and what it leaves behind.  EnvPlanes (default): the env's own state planes
// (StepParams::lam, S, resnorm, ...), read at the start and written back at the end, with the reward and the auto-reset.
struct EnvPlanes {
    static constexpr bool kEval = false;
    SDCGYM_HD void lambda(int64_t, double&, double&) const {}
    SDCGYM_HD void count(bool, int, bool, bool, int) const {}
    SDCGYM_HD const double* action(const double* a) const { return a; }  // base of the action rows: StepParams::action
};

// Evaluation of the sdc-v0 full solve from the reset state (sdcgym_full_solve_counts): lambda from an interleaved list
// or the node of a tensor grid, (u, r) and ||r0|| from the statements of reset_one, and no state planes at all - no
// reward, no terminal state, no auto-reset.  The results leave through StepParams::info_niter / info_res / flags /
// info_lam; `hist` (shared memory of the block, or nullptr) counts the outcome of every valid thread:
// [0, max_iters] niter of the converged nodes, max_iters + 1 err, max_iters + 2 out of sweeps.
struct ResetEval {
    static constexpr bool kEval = true;
    const double* lam;  // [N][2], or nullptr: node grid_first + i of the grid below
    int64_t grid_re, grid_im, grid_first;
    double re_lo, re_hi, im_lo, im_hi;
    int* hist;
    // grid_lambda (specrad_params.cuh) as the translation units built with contraction compile it: one FMA, spelled out
    // here because this unit is built with -fmad=false
    SDCGYM_HD void lambda(int64_t i, double& lr, double& li) const {
        if (lam) {
            lr = lam[2 * i];
            li = lam[2 * i + 1];
            return;
        }
        const int64_t g = grid_first + i, a = g / grid_im, b = g - a * grid_im;
        lr = (grid_re > 1) ? dfma(dsub(re_hi, re_lo), ddiv((double)a, (double)(grid_re - 1)), re_lo) : re_lo;
        li = (grid_im > 1) ? dfma(dsub(im_hi, im_lo), ddiv((double)b, (double)(grid_im - 1)), im_lo) : im_lo;
    }
    SDCGYM_HD void count(bool valid, int it, bool conv, bool err, int max_iters) const {
        if (!hist || !valid) return;
        const int bin = err ? max_iters + 1 : (conv ? it : max_iters + 2);
#ifdef __CUDA_ARCH__
        atomicAdd(hist + bin, 1);
#else
        hist[bin]++;
#endif
    }
    SDCGYM_HD const double* action(const double* a) const { return a; }
};

// ResetEval for a population of shared action rows (sdcgym_full_solve_counts_population): the block's row is
// blockIdx.y, at StepParams::action + blockIdx.y * a_rs, and every node reads it as one shared row (a_es = 0).  `row`
// is set per block by the kernel, so StepParams stays in the constant bank.
struct PopulationEval : ResetEval {
    int64_t a_rs;       // doubles between the starts of consecutive rows
    const double* row;  // this block's row
    SDCGYM_HD const double* action(const double*) const { return row; }
};

// `after_loads` runs once every input of the env sits in registers (non-dense kernels): the streaming kernel releases
// its shared-memory stage there and starts the next tile's copies.
//
// PHASE (sdc-v0 full solve, dense Q_delta): envs of a warp stop after very different sweep counts (lower_tri, M = 5:
// 39 % within 8 sweeps, 33 % run all 50; ncu: 18.6 of 32 lanes active, strictly_lower_tri 11.4), and a warp runs until
// its last env is done.  The phased launch regroups the stragglers: PHASE 1 = first pass over all envs (inverse +
// sweeps), PHASE 2 = a later pass over the compacted list of unfinished envs.  A warp hands over once all its running
// envs have done p.it_stop sweeps and fewer than p.min_lanes of its lanes are still iterating (warps that stay busy
// never hand over and cost nothing extra).  An env that is still running at the hand-over is SUSPENDED: its (u, r) go to the state planes, its sweep count to the niter plane (the
// resnorm plane keeps the norm the divergence test compares against), the inverse to p.pinv_scratch (first pass only)
// and its index to p.cont_list; a PHASE 2 pass picks it up with exactly those bits, so the sweep sequence of every
// env - and therefore every output - is the one of the single-launch kernel.  PHASE 0 = no phases (unchanged code).
// Src: EnvPlanes, or ResetEval (sdc-v0 full solve from the reset state, PHASE 0, no StepInputs).
template <int M, int KIND, int V, bool DENSE, int HOLD, class AfterLoads = NoAfterLoads, int PHASE = 0,
          class Src = EnvPlanes>
SDCGYM_HD void step_one(const StepParams<M>& p, const int64_t tid, double* side = nullptr, const int side_stride = 1,
                        cplx* pside = nullptr, const int pstride = 1, const StepInputs* in = nullptr,
                        AfterLoads after_loads = AfterLoads(), const uint32_t taddr = 0, const Src& src = Src()) {
    constexpr bool kEval = Src::kEval;
    static_assert(!kEval || (KIND == SDCGYM_ENV_FULL && PHASE == 0 && HOLD != 10), "evaluation: single-launch full solve");
    const bool valid = tid < p.N;
    const int64_t i = valid ? tid : p.N - 1;
    const int64_t ld = p.ld;
    // input side (see StepInputs): staged tile or the global planes
    const double* const in_lam = in ? in->lam : p.lam;
    const double* const in_S = in ? in->S : p.S;
    const int64_t ild = in ? in->ld : ld, ii = in ? in->i : i;

    // ---- phase 0: every global load of this env is issued here, in one basic block, so that a single DRAM round trip
    //      covers them all (placed at their uses they end up behind the branches of the division slow paths, one
    //      exposed latency each) ----
    double lr, li;
    if constexpr (kEval) {
        src.lambda(i, lr, li);
    } else {
        lr = in_lam[ii];
        li = in_lam[ild + ii];
    }
    double araw[DENSE ? 1 : M], aimg[DENSE ? 1 : M];
    if (!DENSE) {
#pragma unroll
        for (int k = 0; k < M; k++) {
            araw[k] = 0.0;
            aimg[k] = 0.0;
            if (p.prec_type != SDCGYM_PREC_FIXED) {
                if (in) {  // staged rows (shared memory: plain loads)
                    araw[k] = in->action[ii * p.a_es + k * p.a_cs];
                    if (p.is_complex) aimg[k] = in->action[ii * p.a_es + k * p.a_cs + 1];
                } else {
                    araw[k] = ld_ro(src.action(p.action) + i * p.a_es + k * p.a_cs);
                    if (p.is_complex) aimg[k] = ld_ro(src.action(p.action) + i * p.a_es + k * p.a_cs + 1);
                }
            }
        }
    }
#ifdef __CUDA_ARCH__
    if constexpr (DENSE) {
        // the Q_delta entries are read one by one while P is built (an action row is M(M+1)/2 doubles at most per
        // env, too many to hold next to the LU factors): without this the first pass over P is a chain of exposed
        // load latencies (ncu: 14 % of the samples of the M = 5 lower_tri kernel on the first load uses).  Pull the
        // row's cache lines into L1 now; the loads below then hit.
        if (src.action(p.action) && p.prec_type != SDCGYM_PREC_FIXED) {
            const double* row = src.action(p.action) + i * p.a_es;
            constexpr int kMaxLines = (M * (M + 1) * 8 + 127) / 128 + 1;  // complex lower_tri row, unaligned start
            const int64_t row_doubles = p.a_es < (int64_t)M * (M + 1) ? p.a_es : (int64_t)M * (M + 1);
#pragma unroll
            for (int l = 0; l < kMaxLines; l++)
                if ((int64_t)l * 16 < row_doubles) asm volatile("prefetch.global.L1 [%0];" ::"l"(row + l * 16));
        }
    }
#endif
    double ur[M], ui[M], rr[M], ri[M];
    auto load_state = [&]() {
#pragma unroll
        for (int m = 0; m < M; m++) {
            ur[m] = in_S[(2 * m) * ild + ii];
            ui[m] = in_S[(2 * m + 1) * ild + ii];
            rr[m] = in_S[(2 * M + 2 * m) * ild + ii];
            ri[m] = in_S[(2 * M + 2 * m + 1) * ild + ii];
        }
    };
    if (!DENSE && !kEval) load_state();  // the dense kernels need the registers for the inverse first
    // (evaluation: the reset state is derived from lambda once z is known, below)
    double nr_old = kEval ? 0.0 : (in ? in->resnorm[ii] : p.resnorm[i]);
    static_assert(PHASE == 0 || (DENSE && KIND == SDCGYM_ENV_FULL && HOLD != 5), "phased launches: dense full solves");
    int it = (KIND == SDCGYM_ENV_STEP || PHASE == 2) ? (in ? in->niter[ii] : p.niter[i]) : 0;
    // the auto-reset needs these at the very end
    int32_t ep_old = p.autoreset ? (in ? in->episodes[ii] : p.episodes[i]) : 0;
    uint32_t ctr_old = p.autoreset ? (in ? in->rng_ctr[ii] : p.rng_ctr[i]) : 0u;
    // cached ||initial residual|| of the episode (residual_change reward); NaN marks "not cached: re-derive"
    double ninit_cached = d_nan();
    // (sdc-v1 only: one more live value and one more store in the sdc-v0 kernel measured 2 % on the headline step, and a
    //  full solve amortises the re-derivation over ~43 sweeps)
    constexpr bool kUseNinit = (KIND == SDCGYM_ENV_STEP);
    if (kUseNinit && p.strategy == SDCGYM_REW_RESIDUAL_CHANGE && p.norm_init)
        ninit_cached = (in && in->norm_init) ? in->norm_init[ii] : p.norm_init[i];
#ifdef __CUDA_ARCH__
    // consume everything here: keeps the loads above this point.  (Not for the dense kernels: they load the Q_delta
    // entries next and a barrier here would only add a second exposed round trip - measured 20 % slower at M = 3.)
    if (!DENSE) {
        asm volatile("" : "+d"(lr), "+d"(li), "+d"(nr_old), "+r"(it), "+r"(ep_old), "+r"(ctr_old));
        // (ninit_cached needs no entry: the streaming kernel's release callback below starts with a block barrier,
        //  which the compiler does not move shared-memory loads across; listing it cost the sdc-v0 kernel 2 %)
#pragma unroll
        for (int k = 0; k < M; k++) asm volatile("" : "+d"(araw[k]), "+d"(aimg[k]));
        if constexpr (!kEval) {
#pragma unroll
            for (int m = 0; m < M; m++) asm volatile("" : "+d"(ur[m]), "+d"(ui[m]), "+d"(rr[m]), "+d"(ri[m]));
        }
    }
#endif
    if (!DENSE) after_loads();
    const double zr = dmul(lr, p.dt), zi = dmul(li, p.dt);

    // ---- preconditioner inverse ----
    constexpr bool PS = DENSE && (HOLD == 5);  // Pinv (and C) live in the complex side store
    static_assert(HOLD != 5 || (DENSE && M > kRegInvMaxM), "HOLD 5 is for the large dense kernels");
    constexpr int NP = DENSE ? (PS ? 1 : M * M) : M;
    double Pr[NP], Pi[NP];
    if (!DENSE) {
        double pre_r[DENSE ? 1 : M], pre_i[DENSE ? 1 : M];  // diagonal of P = I - z*Qd
#pragma unroll
        for (int k = 0; k < M; k++) {
            cplx zq;
            if (p.prec_type == SDCGYM_PREC_FIXED) {
                // fixed *diagonal* Q_delta (prec='min' / 'zeros'): the dense inverse of a diagonal matrix is the
                // diagonal of reciprocals (bit-identical, tests/test_blas_fingerprint.py), so these run here
                const double d = p.Qd[k * M + k];
                zq = cplx{dmul(zr, d), dmul(zi, d)};
            } else if (p.is_complex) {
                cplx d{araw[DENSE ? 0 : k], aimg[DENSE ? 0 : k]};
                zq = (p.do_scale & SDCGYM_ACTION_F32) ? cmul_np_f32(cplx{zr, zi}, d) : cmul_np(cplx{zr, zi}, d);
            } else {
                double a = araw[DENSE ? 0 : k];
                double d = a;
                if (p.do_scale & SDCGYM_ACTION_SCALE) d = (a <= -1.0) ? 0.0 : ((a >= 1.0) ? 1.0 : dmul(0.5, dadd(a, 1.0)));
                zq = (p.do_scale & SDCGYM_ACTION_F32) ? cmul_np_f32(cplx{zr, zi}, cplx{d, 0.0}) : cplx{dmul(zr, d), dmul(zi, d)};
            }
            pre_r[DENSE ? 0 : k] = dsub(1.0, zq.re);
            pre_i[DENSE ? 0 : k] = -zq.im;
        }
        if constexpr (!DENSE && KIND == SDCGYM_ENV_FULL) {
            // the M reciprocals together: their divisions interleave (fast_div.cuh); +1.7 % at M = 3, 7, neutral at 5
            crecip_batch<M, V == 0>(pre_r, pre_i, Pr, Pi);
        } else if constexpr (!DENSE) {
            // sdc-v1 is memory bound and register starved (80 registers): one reciprocal at a time
#pragma unroll
            for (int k = 0; k < M; k++) {
                const cplx inv = crecip<V == 0>(cplx{pre_r[k], pre_i[k]});
                Pr[k] = inv.re;
                Pi[k] = inv.im;
            }
        }
    } else {
        // P = eye(M) - (lam*dt)*Qd, column-major; Qd from the action layout (dp_playground.py:194-207) or fixed
        auto qd_entry = [&](int r, int c, int k) {
            cplx d{0.0, 0.0};
            if (p.prec_type == SDCGYM_PREC_FIXED) {
                d.re = p.Qd[r * M + c];
            } else if (k >= 0) {
                if (p.is_complex) {
                    d.re = ld_ro(src.action(p.action) + i * p.a_es + k * p.a_cs);
                    d.im = ld_ro(src.action(p.action) + i * p.a_es + k * p.a_cs + 1);
                } else {
                    const double a = ld_ro(src.action(p.action) + i * p.a_es + k * p.a_cs);
                    d.re = a;
                    if (p.do_scale & SDCGYM_ACTION_SCALE) d.re = (a <= -1.0) ? 0.0 : ((a >= 1.0) ? 1.0 : dmul(0.5, dadd(a, 1.0)));
                }
            }
            return d;
        };
        // index of entry (r, c) in the action vector for the run-time layout, -1 if the entry is structurally zero
        auto act_index = [&](int r, int c) {
            switch (p.prec_type) {
            case SDCGYM_PREC_LOWER_DIAG: return (r == c + 1) ? c : -1;
            case SDCGYM_PREC_LOWER_TRI: return (c <= r) ? r * (r + 1) / 2 + c : -1;
            case SDCGYM_PREC_STRICTLY_LOWER_TRI: return (c < r) ? r * (r - 1) / 2 + c : -1;
            case SDCGYM_PREC_DIAG: return (c == r) ? r : -1;
            default: return -1;
            }
        };
        const bool f32_qd = (p.do_scale & SDCGYM_ACTION_F32) && p.prec_type != SDCGYM_PREC_FIXED;
        auto zq_entry = [&](int r, int c) {
            const cplx d = qd_entry(r, c, act_index(r, c));
            return f32_qd ? cmul_np_f32(cplx{zr, zi}, d) : cmul_np(cplx{zr, zi}, d);
        };
        if constexpr (PHASE == 3) {
            // inverse only (split first pass): P -> exact inverse -> work planes, nothing else; no Pinv array, the
            // entries leave as they are produced
            static_assert(M <= kRegInvMaxM, "the split first pass is for the register-resident inverse");
            RegMatrix<M> A;
#pragma unroll
            for (int r = 0; r < M; r++)
#pragma unroll
                for (int c = 0; c < M; c++) {
                    const cplx zq = zq_entry(r, c);
                    A.R(r, c) = dsub((r == c) ? 1.0 : 0.0, zq.re);
                    A.I(r, c) = dsub(0.0, zq.im);
                }
            cinv_exact_reg_cols<M, V>(A, [&](int r, int c, double re, double im) {
                if (valid) {
                    p.pinv_scratch[(2 * (r * M + c)) * ld + i] = re;
                    p.pinv_scratch[(2 * (r * M + c) + 1) * ld + i] = im;
                }
            });
            return;
        } else if constexpr (PHASE == 2 || PHASE == 4) {
            // resumed env (2) / first sweeps after the inverse-only kernel (4): the inverse computed earlier (same bits)
#pragma unroll
            for (int k = 0; k < M * M; k++) {
                Pr[(DENSE && !PS) ? k : 0] = p.pinv_scratch[(2 * k) * ld + i];
                Pi[(DENSE && !PS) ? k : 0] = p.pinv_scratch[(2 * k + 1) * ld + i];
            }
        } else if constexpr (M <= kRegInvMaxM) {
            RegMatrix<M> A;
#pragma unroll
            for (int r = 0; r < M; r++)
#pragma unroll
                for (int c = 0; c < M; c++) {
                    const cplx zq = zq_entry(r, c);
                    A.R(r, c) = dsub((r == c) ? 1.0 : 0.0, zq.re);
                    A.I(r, c) = dsub(0.0, zq.im);
                }
            // the inverse arrives column by column: only the LU factors and one column are live in registers
            cinv_exact_reg_cols<M, V>(A, [&](int r, int c, double re, double im) {
                Pr[(DENSE && !PS) ? r * M + c : 0] = re;
                Pi[(DENSE && !PS) ? r * M + c : 0] = im;
            });
        } else if constexpr (HOLD == 8 || HOLD == 9) {
            // M = 8, 9: the LU work matrix does not fit the register file: it lives in the side store (shared memory,
            // same per-thread slots that hold C afterwards), the code stays fully unrolled over static indices
            StridedMatrix<M> A{side, side_stride};
#pragma unroll
            for (int r = 0; r < M; r++)
#pragma unroll
                for (int c = 0; c < M; c++) {
                    const cplx zq = zq_entry(r, c);
                    A.R(r, c) = dsub((r == c) ? 1.0 : 0.0, zq.re);
                    A.I(r, c) = dsub(0.0, zq.im);
                }
            cinv_exact_reg_cols<M, V>(A, [&](int r, int c, double re, double im) {
                Pr[(DENSE && !PS) ? r * M + c : 0] = re;
                Pi[(DENSE && !PS) ? r * M + c : 0] = im;
            });
        } else if constexpr (PS) {
            cplx* A = pside;                                // LU work matrix now, C later (same per-thread slots)
            cplx* B = pside + (size_t)M * M * pstride;      // the inverse stays here
#pragma unroll 1
            for (int r = 0; r < M; r++)
#pragma unroll 1
                for (int c = 0; c < M; c++) {
                    const cplx zq = zq_entry(r, c);
                    A[(r + c * M) * pstride] = cplx{dsub((r == c) ? 1.0 : 0.0, zq.re), dsub(0.0, zq.im)};
                }
            cinv_exact<M, V>(A, B, pstride);
        } else {
            cplx A[M * M], B[M * M];  // column-major work arrays (local memory)
#pragma unroll 1
            for (int r = 0; r < M; r++)
#pragma unroll 1
                for (int c = 0; c < M; c++) {
                    const cplx zq = zq_entry(r, c);
                    A[r + c * M] = cplx{dsub((r == c) ? 1.0 : 0.0, zq.re), dsub(0.0, zq.im)};
                }
            cinv_exact<M, V>(A, B);
#pragma unroll
            for (int r = 0; r < M; r++)
#pragma unroll
                for (int c = 0; c < M; c++) {
                    Pr[DENSE ? r * M + c : 0] = B[r + c * M].re;
                    Pi[DENSE ? r * M + c : 0] = B[r + c * M].im;
                }
        }
    }

    if constexpr (HOLD == 9) {
        // the LU work matrix is dead: its slots now hold Pinv (re at k, im at M^2 + k), read back in every sweep
#pragma unroll
        for (int k = 0; k < M * M; k++) {
            side[k * side_stride] = Pr[DENSE ? k : 0];
            side[(M * M + k) * side_stride] = Pi[DENSE ? k : 0];
        }
    }

    // ---- system matrix (optionally register resident) ----
    // experimental residency (tuning only): 6 = Re(C) in shared memory and Im(C) re-derived
    constexpr bool CS = (HOLD == 4 || HOLD == 8);  // C lives in the (double) side store
    constexpr int NCR = (HOLD >= 1 && HOLD <= 3) ? M * M : 1, NCI = (HOLD == 2) ? M * M : 1;
    double Cr[NCR], Ci[NCI];
    static_assert(HOLD != 10 || (!DENSE && KIND == SDCGYM_ENV_FULL && 4 * M * M <= 128), "HOLD 10: C in tensor memory");
#ifdef __CUDA_ARCH__
    if constexpr (HOLD == 10) __syncwarp();  // (the reciprocals above have divergent slow paths)
#endif
    if (HOLD >= 1 && HOLD != 9) {
#pragma unroll
        for (int r = 0; r < M; r++)
#pragma unroll
            for (int c = 0; c < M; c++) {
                double q = p.Q[r * M + c];
                const double crv = (r == c) ? dsub(1.0, dmul(zr, q)) : -dmul(zr, q);
                if (HOLD <= 3) Cr[(HOLD >= 1 && HOLD <= 3) ? r * M + c : 0] = crv;
                if (CS) side[(M * M + r * M + c) * side_stride] = crv;
                if (HOLD == 2) Ci[(HOLD == 2) ? r * M + c : 0] = -dmul(zi, q);
                if (HOLD == 3 || CS) side[(r * M + c) * side_stride] = -dmul(zi, q);
                if (HOLD == 5 || HOLD == 7) pside[(r * M + c) * pstride] = cplx{crv, -dmul(zi, q)};
#ifdef __CUDA_ARCH__
                if constexpr (HOLD == 10) tmem_st_pair(taddr + 4 * (r * M + c), crv, -dmul(zi, q));
#endif
                if (HOLD == 6) side[(r * M + c) * side_stride] = crv;
            }
    }
#ifdef __CUDA_ARCH__
    if constexpr (HOLD == 10) tmem_wait_st();
#endif


    if constexpr (kEval) {
        // reset_one's statements: u = 1, r = u0 - C u, ||r0||
        initial_state<M, V>(p.Q, zr, zi, ur, ui, rr, ri);
        nr_old = inf_norm_fast<M>(rr, ri);
    } else if (DENSE) {
        load_state();
    }

    // sdc-v1 needs the previous residual for the reward when norm_factor != 1
    double norm_old_scaled = nr_old;
    if (KIND == SDCGYM_ENV_STEP && p.strategy == SDCGYM_REW_RESIDUAL_CHANGE && p.norm_factor != 1.0)
        norm_old_scaled = scaled_inf_norm<M>(rr, ri, p.norm_factor);

    // one sweep: u += Pinv @ r ; r = u0 - C @ u      (sdc_env.py:229-231 / :516-519)
    // (`commit`: HOLD 10 runs the sweep with the whole warp - its tensor-memory loads are warp-collective - and keeps
    //  the new state only in the lanes that are still iterating)
    auto sweep = [&](const bool commit = true) {
        // when C is not register resident its entries are re-derived from z and the constant-bank Q on every
        // sweep; the empty asm keeps the compiler from hoisting those products back out of the loop (which
        // would turn them into spills).
        double zr_s = zr, zi_s = zi;
        // volatile: the side store is loop invariant, and a hoisted load is a register again
        const volatile double* vside = side;
        const volatile cplx* vp = pside;
        (void)vside;
        (void)vp;
#ifdef __CUDA_ARCH__
        if (HOLD < 2 || HOLD == 6 || HOLD == 9) asm volatile("" : "+d"(zr_s), "+d"(zi_s));  // (HOLD 3 never uses zi_s)
#endif
        double dr[M], di[M];
#pragma unroll
        for (int m = 0; m < M; m++) {
            if (!DENSE) {
                diag_rowdot<M, V>(m, Pr[m], Pi[m], rr[m], ri[m], dr[m], di[m]);
            } else {
                double ar[M], ai[M];
#pragma unroll
                for (int c = 0; c < M; c++) {
                    if (PS) {
                        ar[c] = vp[(M * M + m + c * M) * pstride].re;  // B is column-major
                        ai[c] = vp[(M * M + m + c * M) * pstride].im;
                    } else if (HOLD == 9) {
                        ar[c] = vside[(m * M + c) * side_stride];
                        ai[c] = vside[(M * M + m * M + c) * side_stride];
                    } else {
                        ar[c] = Pr[(DENSE && !PS) ? m * M + c : 0];
                        ai[c] = Pi[(DENSE && !PS) ? m * M + c : 0];
                    }
                }
                zgemv_rowdot<M, V>(ar, ai, rr, ri, dr[m], di[m]);
            }
        }
#pragma unroll
        for (int m = 0; m < M; m++) {
            // HOLD 10: lanes that are done keep u (and therefore get the very same r back from the row products below)
            if (HOLD != 10 || commit) {
                ur[m] = dadd(ur[m], dr[m]);
                ui[m] = dadd(ui[m], di[m]);
            }
        }
#pragma unroll
        for (int m = 0; m < M; m++) {
            double cr[M], ci[M], yr, yi;
#ifdef __CUDA_ARCH__
            if constexpr (HOLD == 10) {
                // row m of C from tensor memory: M warp-collective loads of one (re, im) pair per lane, one wait
                int w[4 * M];
                tmem_ld_row<M>(taddr + 4 * (m * M), w);
                tmem_wait_ld();
#pragma unroll
                for (int c = 0; c < M; c++) {
                    cr[c] = __hiloint2double(w[4 * c + 1], w[4 * c]);
                    ci[c] = __hiloint2double(w[4 * c + 3], w[4 * c + 2]);
                }
            }
#endif
#pragma unroll
            for (int c = 0; c < M; c++) {
                if (HOLD == 10) break;
                double q = p.Q[m * M + c];
                cplx t7{0.0, 0.0};
                if (HOLD == 7) t7 = ld_pair(&pside[(m * M + c) * pstride]);  // HOLD 7: C as (re, im) pairs, one LDS.128
                if (HOLD == 7) cr[c] = t7.re;
                else if (HOLD == 5) cr[c] = vp[(m * M + c) * pstride].re;
                else if (HOLD == 6) cr[c] = vside[(m * M + c) * side_stride];
                else if (CS) cr[c] = vside[(M * M + m * M + c) * side_stride];
                else if (HOLD >= 1 && HOLD != 9) cr[c] = Cr[(HOLD >= 1 && HOLD <= 3) ? m * M + c : 0];
                else cr[c] = (m == c) ? dsub(1.0, dmul(zr_s, q)) : -dmul(zr_s, q);
                if (HOLD == 7) ci[c] = t7.im;
                else if (HOLD == 5) ci[c] = vp[(m * M + c) * pstride].im;
                else if (HOLD == 6) ci[c] = -dmul(zi_s, q);
                else if (HOLD == 2) ci[c] = Ci[(HOLD == 2) ? m * M + c : 0];
                else if (HOLD == 3 || CS) ci[c] = vside[(m * M + c) * side_stride];
                else ci[c] = -dmul(zi_s, q);
            }
            zgemv_rowdot<M, V>(cr, ci, ur, ui, yr, yi);
            rr[m] = dsub(1.0, yr);
            ri[m] = -yi;
        }
    };

    const double thr = dmul(nr_old, 100.0);  // norm_res_old * 100
    bool conv = false, err = false;
    double nr = nr_old;

    if (KIND == SDCGYM_ENV_FULL) {
        // while not done and niter < max_iters  (sdc_env.py:224-247); per-lane early exit by warp vote
        const HiBand bc = make_band(p.restol), be = make_band(thr);
        const SqBand sc = make_sqband(p.restol), se = make_sqband(thr);
        bool act = p.max_iters > 0 && (PHASE == 0 || valid);
        while (SDCGYM_WARP_ANY(act)) {
            if constexpr (HOLD == 10) {
#ifdef __CUDA_ARCH__
                __syncwarp();
#endif
                sweep(act);  // warp-collective; commits where act
            }
            if (act) {
                it++;
                if constexpr (HOLD != 10) sweep();
                // decide `err` (nr is NaN/Inf or nr > thr) and `conv` (nr < restol) without forming nr:
                // stage 1 on the integer pipe, stage 2 on squared magnitudes, exact norm as a last resort.
                const int H = absmax_hi<M>(rr, ri);
                const bool amb_e = (H > be.lo) && (H < be.hi), amb_c = (H > bc.lo) && (H < bc.hi);
                if (H >= be.hi) {
                    err = true;  // NaN / Inf / > 100 x
                } else if (!(amb_e || amb_c)) {
                    conv = H <= bc.lo;
                } else {
                    const double s2 = sq_absmax<M>(rr, ri);
                    // 0 = surely below the threshold, 1 = surely above, 2 = undecided
                    const int ge = !amb_e ? 0 : (!se.ok ? 2 : (s2 < se.lo2 ? 0 : (s2 > se.hi2 ? 1 : 2)));
                    const int gc = !amb_c ? (H <= bc.lo ? 0 : 1) : (!sc.ok ? 2 : (s2 < sc.lo2 ? 0 : (s2 > sc.hi2 ? 1 : 2)));
                    if (ge == 2 || gc == 2) {
                        // copy first: passing rr/ri themselves would force a store of both arrays to local
                        // memory on every sweep, not just here
                        double tr[M], ti[M];
#pragma unroll
                        for (int m = 0; m < M; m++) {
                            tr[m] = rr[m];
                            ti[m] = ri[m];
                        }
                        const double nx = inf_norm_slow<M>(tr, ti);
                        err = isnan(nx) || isinf(nx) || nx > thr;
                        if (!err) conv = nx < p.restol;
                    } else {
                        err = ge == 1;
                        conv = !err && gc == 0;
                    }
                }
                if (p.old_states && valid && it < p.max_iters) store_column<M>(p.old_states, i, p.max_iters, it, ur, ui, rr, ri);
                act = !err && !conv && it < p.max_iters;
            }
            // hand-over: every env still iterating has done p.it_stop sweeps and the warp has thinned out to fewer
            // than p.min_lanes of them (min_lanes > 32: at it_stop whatever the occupancy) - the stragglers are regrouped
            if constexpr (PHASE != 0) {
#ifdef __CUDA_ARCH__
                const unsigned running = __ballot_sync(0xffffffffu, act);
                const unsigned young = __ballot_sync(0xffffffffu, act && it < p.it_stop);
                if (young == 0u && __popc(running) < p.min_lanes) break;
#else
                if (!(act && it < p.it_stop) && (act ? 1 : 0) < p.min_lanes) break;
#endif
            }
        }
        if constexpr (PHASE != 0) {
            // still running at the hand-over count: suspend (the warp is converged here: the loop exit is a warp vote)
            const bool susp = act;
#ifdef __CUDA_ARCH__
            const unsigned sm = __ballot_sync(0xffffffffu, susp);
            if (sm) {
                const int lane = (int)(threadIdx.x & 31u), leader = __ffs(sm) - 1;
                int base = 0;
                if (lane == leader) base = atomicAdd(p.cont_count, __popc(sm));
                base = __shfl_sync(0xffffffffu, base, leader);
                if (susp) p.cont_list[base + __popc(sm & ((1u << lane) - 1u))] = (int32_t)i;
            }
#else
            if (susp) p.cont_list[p.cont_count[0]++] = (int32_t)i;
#endif
            if (susp) {
                store_state<M>(p.S, ld, i, ur, ui, rr, ri);
                p.niter[i] = it;
                if constexpr (PHASE == 1) {
                    const volatile double* ps = side;
                    (void)ps;
#pragma unroll
                    for (int k = 0; k < M * M; k++) {
                        p.pinv_scratch[(2 * k) * ld + i] = (HOLD == 9) ? ps[k * side_stride] : Pr[(DENSE && !PS) ? k : 0];
                        p.pinv_scratch[(2 * k + 1) * ld + i] = (HOLD == 9) ? ps[(M * M + k) * side_stride] : Pi[(DENSE && !PS) ? k : 0];
                    }
                }
                return;
            }
        }
        if (p.max_iters > 0) nr = inf_norm_fast<M>(rr, ri);
    } else {
        sweep();
        nr = inf_norm_fast<M>(rr, ri);
        it++;
        err = isnan(nr) || isinf(nr);
        err = err || nr > thr;
        conv = nr < p.restol;
    }

    // ---- reward ----
    double rew = 0.0;
    if constexpr (kEval) {
        src.count(valid, it, conv, err, p.max_iters);
    } else if (err) {
        rew = dmul(-p.step_penalty, (double)(p.max_iters + 1));
    } else if (p.strategy == SDCGYM_REW_ITERATION_ONLY) {
        rew = dmul((double)(-it), p.step_penalty);
    } else {
        double norm_init_scaled = 0.0;
        if (p.strategy == SDCGYM_REW_RESIDUAL_CHANGE) {
            if (kUseNinit && p.norm_init) {
                norm_init_scaled = ninit_cached;  // written by the reset of this episode (same function, same bits)
            } else {
                // initial residual of the episode is a function of lambda only: recompute it
                double tu[M], tv[M], ir[M], ii2[M];
                initial_state<M, V>(p.Q, zr, zi, tu, tv, ir, ii2);
                norm_init_scaled = scaled_inf_norm<M>(ir, ii2, p.norm_factor);
            }
            if (KIND == SDCGYM_ENV_FULL) norm_old_scaled = norm_init_scaled;  // reward_func(initial_residual, ...)
        }
        rew = reward_func<M>(p.strategy, p.step_penalty, p.residual_weight, p.norm_factor, p.restol, p.max_iters,
                             norm_old_scaled, norm_init_scaled, rr, ri, nr, conv, it, p.log_restol_nf);
    }

    const bool done = (KIND == SDCGYM_ENV_FULL) ? true : (conv || it >= p.max_iters || err);
    if (!valid) return;

    if (p.reward) p.reward[i] = rew;
    if (p.flags)
        p.flags[i] = (uint8_t)((done ? SDCGYM_FLAG_DONE : 0) | (conv ? SDCGYM_FLAG_CONVERGED : 0) | (err ? SDCGYM_FLAG_ERR : 0));
    if (p.info_res) p.info_res[i] = nr;
    if (p.info_niter) p.info_niter[i] = it;
    if (p.info_lam) {
        p.info_lam[2 * i] = lr;  // interleaved complex128, directly viewable by the host layer
        p.info_lam[2 * i + 1] = li;
    }
    if constexpr (kEval) return;
    if (KIND == SDCGYM_ENV_STEP && p.old_states && it < p.max_iters)
        store_column<M>(p.old_states, i, p.max_iters, it, ur, ui, rr, ri);

    if (done && p.term) store_state<M>(p.term, ld, i, ur, ui, rr, ri);

    if (done && p.autoreset) {
        // DummyVecEnv: obs = env.reset() right after the terminal step
        int32_t ep = ep_old + 1;
        p.episodes[i] = ep;
        uint32_t ctr = ctr_old;
        double nlr, nli;
        draw_lambda<M>(p, i, ctr, ep, nlr, nli);
        p.rng_ctr[i] = ctr + 1;
        p.lam[i] = nlr;
        p.lam[ld + i] = nli;
        const double nzr = dmul(nlr, p.dt), nzi = dmul(nli, p.dt);
        initial_state<M, V>(p.Q, nzr, nzi, ur, ui, rr, ri);
        store_state<M>(p.S, ld, i, ur, ui, rr, ri);
        const double n0 = inf_norm_fast<M>(rr, ri);
        p.resnorm[i] = n0;
        if (kUseNinit) store_norm_init<M>(p, i, rr, ri, n0);
        p.niter[i] = 0;
    } else {
        store_state<M>(p.S, ld, i, ur, ui, rr, ri);
        p.resnorm[i] = nr;
        p.niter[i] = it;
    }
}

#ifdef __CUDACC__
template <int M, int V>
__global__ void __launch_bounds__(kBlock) reset_kernel(const __grid_constant__ StepParams<M> p) {
    reset_one<M, V>(p, (int64_t)blockIdx.x * kBlock + threadIdx.x);
}

template <int M, int KIND, int V, bool DENSE, int HOLD, int MINB = 1, int BLOCK = kBlock>
__global__ void __launch_bounds__(BLOCK, MINB) step_kernel(const __grid_constant__ StepParams<M> p) {
    if constexpr (HOLD == 5 || HOLD == 7) {
        extern __shared__ double2 pside_smem[];  // [2*M*M][BLOCK] complex: LU/C then Pinv of every thread
        step_one<M, KIND, V, DENSE, HOLD>(p, (int64_t)blockIdx.x * BLOCK + threadIdx.x, nullptr, 1,
                                          reinterpret_cast<cplx*>(pside_smem) + threadIdx.x, BLOCK);
    } else if constexpr (HOLD >= 3) {
        extern __shared__ double side_smem[];  // [M*M or 2*M*M][BLOCK]: Im(C) (and Re(C)) of every thread, conflict free
        step_one<M, KIND, V, DENSE, HOLD>(p, (int64_t)blockIdx.x * BLOCK + threadIdx.x, side_smem + threadIdx.x, BLOCK);
    } else {
        step_one<M, KIND, V, DENSE, HOLD>(p, (int64_t)blockIdx.x * BLOCK + threadIdx.x);
    }
}

// full solve, diagonal Q_delta, the system matrix C of every env in TENSOR MEMORY (HOLD 10).  The shipped kernel keeps C
// in shared memory and is co-limited by the FP64 pipe (77 %) and the shared-memory pipe (81 %: 25 LDS.128 per sweep
// and thread); tensor memory has its own path to the register file.  One CTA = 128 threads = the 128 TMEM lanes, a
// thread's C = 4 M^2 32-bit columns of its lane (M = 5: 100 of an allocation of 128; four CTAs fill the SM's 512).
template <int M, int V, int MINB>
__global__ void __launch_bounds__(128, MINB) step_tmem_kernel(const __grid_constant__ StepParams<M> p) {
    constexpr uint32_t kCols = (4 * M * M <= 32) ? 32u : ((4 * M * M <= 64) ? 64u : 128u);
    static_assert(4 * M * M <= 128, "C does not fit a quarter of the tensor memory");
    __shared__ uint32_t tbase;
    const uint32_t warp = threadIdx.x >> 5;
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                         (uint32_t)__cvta_generic_to_shared(&tbase)),
                     "r"(kCols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t taddr = tbase + ((warp * 32u) << 16);
    step_one<M, SDCGYM_ENV_FULL, V, false, 10>(p, (int64_t)blockIdx.x * 128 + threadIdx.x, nullptr, 1, nullptr, 1, nullptr,
                                               NoAfterLoads(), taddr);
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();  // (every thread comes back from step_one: its early exits are returns of the inlined body)
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tbase), "r"(kCols) : "memory");
}

// phased full solve of dense Q_delta (step_one PHASE): PHASE 1 = all envs, one per thread; PHASE 2 = the envs of
// `list[0 .. *count)` (a fixed grid strides over the list, whose length only the device knows; threads past the end
// run a clamped env that never sweeps and stores nothing)
// (PHASE 4 = the first sweeps of all envs after inverse_kernel has left every inverse in the work planes)
template <int M, int V, int HOLD, int MINB, int BLOCK, int PHASE>
__global__ void __launch_bounds__(BLOCK, MINB) step_phase_kernel(const __grid_constant__ StepParams<M> p,
                                                                 const int32_t* __restrict__ list,
                                                                 const int32_t* __restrict__ count) {
    static_assert(PHASE == 1 || PHASE == 2 || PHASE == 4, "");
    const int64_t n = (PHASE != 2) ? p.N : (int64_t)count[0];
    for (int64_t base = (int64_t)blockIdx.x * BLOCK; base < n; base += (int64_t)gridDim.x * BLOCK) {
        const int64_t t = base + threadIdx.x;
        const int64_t idx = (PHASE != 2) ? t : ((t < n) ? (int64_t)list[t] : p.N);
        if constexpr (HOLD == 7) {
            extern __shared__ double2 pside_smem[];
            step_one<M, SDCGYM_ENV_FULL, V, true, HOLD, NoAfterLoads, PHASE>(p, idx, nullptr, 1, reinterpret_cast<cplx*>(pside_smem) + threadIdx.x, BLOCK);
        } else if constexpr (HOLD >= 3) {
            extern __shared__ double side_smem[];
            step_one<M, SDCGYM_ENV_FULL, V, true, HOLD, NoAfterLoads, PHASE>(p, idx, side_smem + threadIdx.x, BLOCK);
        } else {
            step_one<M, SDCGYM_ENV_FULL, V, true, HOLD, NoAfterLoads, PHASE>(p, idx);
        }
    }
}

// split first pass, part one: the exact inverse of every env's P into the work planes.  Only the LU factors and one
// column are live (no Pinv array, no state, no C): fewer registers, more warps per SM and a third of the code of
// the full first pass - the inverse is bound by latency and instruction fetch, not by the FP64 pipe
template <int M, int V, int MINB>
__global__ void __launch_bounds__(kBlock, MINB) inverse_kernel(const __grid_constant__ StepParams<M> p) {
    step_one<M, SDCGYM_ENV_FULL, V, true, 0, NoAfterLoads, 3>(p, (int64_t)blockIdx.x * kBlock + threadIdx.x);
}

template <int M, int HOLD, int BLOCK = kBlock>
__host__ __device__ constexpr size_t step_kernel_smem_bytes() {
    return HOLD == 3 ? (size_t)M * M * BLOCK * sizeof(double)
                     : ((HOLD == 4 || HOLD == 7 || HOLD == 8 || HOLD == 9) ? (size_t)2 * M * M * BLOCK * sizeof(double)
                                  : (HOLD == 5 ? (size_t)4 * M * M * BLOCK * sizeof(double)
                                               : (HOLD == 6 ? (size_t)M * M * BLOCK * sizeof(double) : 0)));
}

// sdcgym_full_solve_counts: step_kernel's full solve from the reset state (step_one with ResetEval).  With `hist`
// (int64 [max_iters + 3]) the block counts its outcomes in shared memory behind the side store and adds each non-zero
// bin to `hist` once: integer sums, so the result does not depend on the order of the blocks.
template <int M, int V, bool DENSE, int HOLD, int MINB, int BLOCK>
__global__ void __launch_bounds__(BLOCK, MINB) full_solve_counts_kernel(const __grid_constant__ StepParams<M> p,
                                                                        const __grid_constant__ ResetEval src,
                                                                        unsigned long long* __restrict__ hist) {
    extern __shared__ double2 eval_smem[];  // [side store of HOLD][BLOCK], then the block's histogram (int)
    constexpr size_t kSide = step_kernel_smem_bytes<M, HOLD, BLOCK>() / sizeof(double2);
    const int nbins = p.max_iters + 3;
    ResetEval ev = src;
    ev.hist = hist ? reinterpret_cast<int*>(eval_smem + kSide) : nullptr;
    if (hist) {
        for (int k = threadIdx.x; k < nbins; k += BLOCK) ev.hist[k] = 0;
        __syncthreads();
    }
    const int64_t tid = (int64_t)blockIdx.x * BLOCK + threadIdx.x;
    if constexpr (HOLD == 5 || HOLD == 7) {
        step_one<M, SDCGYM_ENV_FULL, V, DENSE, HOLD, NoAfterLoads, 0, ResetEval>(
            p, tid, nullptr, 1, reinterpret_cast<cplx*>(eval_smem) + threadIdx.x, BLOCK, nullptr, NoAfterLoads(), 0, ev);
    } else if constexpr (HOLD >= 3) {
        step_one<M, SDCGYM_ENV_FULL, V, DENSE, HOLD, NoAfterLoads, 0, ResetEval>(
            p, tid, reinterpret_cast<double*>(eval_smem) + threadIdx.x, BLOCK, nullptr, 1, nullptr, NoAfterLoads(), 0, ev);
    } else {
        step_one<M, SDCGYM_ENV_FULL, V, DENSE, HOLD, NoAfterLoads, 0, ResetEval>(p, tid, nullptr, 1, nullptr, 1, nullptr,
                                                                                 NoAfterLoads(), 0, ev);
    }
    if (hist) {
        __syncthreads();  // (every thread comes back from step_one: its exits are returns of the inlined body)
        for (int k = threadIdx.x; k < nbins; k += BLOCK)
            if (ev.hist[k]) atomicAdd(hist + k, (unsigned long long)ev.hist[k]);
    }
}

// sdcgym_full_solve_counts_population: full_solve_counts_kernel for each row of a population, row blockIdx.y at
// p.action + blockIdx.y * src.a_rs (p.a_es = 0), its histogram (required) at hist + blockIdx.y * (max_iters + 3).
// Block (x, y) runs what block x of full_solve_counts_kernel runs for that one row.  The body is that kernel's, spelled
// out: moving it into a shared device function changes the code nvcc generates for full_solve_counts_kernel.
template <int M, int V, bool DENSE, int HOLD, int MINB, int BLOCK>
__global__ void __launch_bounds__(BLOCK, MINB) full_solve_counts_population_kernel(
    const __grid_constant__ StepParams<M> p, const __grid_constant__ PopulationEval src,
    unsigned long long* __restrict__ hist) {
    extern __shared__ double2 eval_smem[];  // [side store of HOLD][BLOCK], then the block's histogram (int)
    constexpr size_t kSide = step_kernel_smem_bytes<M, HOLD, BLOCK>() / sizeof(double2);
    const int nbins = p.max_iters + 3;
    PopulationEval ev = src;
    ev.row = p.action + (int64_t)blockIdx.y * src.a_rs;
    ev.hist = reinterpret_cast<int*>(eval_smem + kSide);
    hist += (int64_t)blockIdx.y * nbins;
    for (int k = threadIdx.x; k < nbins; k += BLOCK) ev.hist[k] = 0;
    __syncthreads();
    const int64_t tid = (int64_t)blockIdx.x * BLOCK + threadIdx.x;
    if constexpr (HOLD == 5 || HOLD == 7) {
        step_one<M, SDCGYM_ENV_FULL, V, DENSE, HOLD, NoAfterLoads, 0, PopulationEval>(
            p, tid, nullptr, 1, reinterpret_cast<cplx*>(eval_smem) + threadIdx.x, BLOCK, nullptr, NoAfterLoads(), 0, ev);
    } else if constexpr (HOLD >= 3) {
        step_one<M, SDCGYM_ENV_FULL, V, DENSE, HOLD, NoAfterLoads, 0, PopulationEval>(
            p, tid, reinterpret_cast<double*>(eval_smem) + threadIdx.x, BLOCK, nullptr, 1, nullptr, NoAfterLoads(), 0, ev);
    } else {
        step_one<M, SDCGYM_ENV_FULL, V, DENSE, HOLD, NoAfterLoads, 0, PopulationEval>(
            p, tid, nullptr, 1, nullptr, 1, nullptr, NoAfterLoads(), 0, ev);
    }
    __syncthreads();  // (every thread comes back from step_one: its exits are returns of the inlined body)
    for (int k = threadIdx.x; k < nbins; k += BLOCK)
        if (ev.hist[k]) atomicAdd(hist + k, (unsigned long long)ev.hist[k]);
}
#endif

}  // namespace sdcgym

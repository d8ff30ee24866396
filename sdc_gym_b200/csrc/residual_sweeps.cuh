// residual_sweeps.cuh - K sweeps of the SDC iteration and the exact gradient of ||r_K||_inf through all of them, one
// sample per thread (sdcgym_residual_sweeps, include/sdcgym.h).
//
// Forward, k = 0 .. K-1 (ResidualLoss.take_step, dp_playground.py:247-258, chained; SDC_Fix_Env's fixed sweep count):
//     delta_k = P^{-1} r_k          P = I - z Qd(theta), z = lam*dt, forward substitution (P is lower triangular)
//     u_{k+1} = u_k + delta_k
//     r_{k+1} = u0 - C u_{k+1}      C = I - z Q, evaluated as u0 - u + z (Q u)
// No early stop and no divergence test.  Output ||r_K||_inf (m = the first index attaining it), optionally u_K, r_K.
//
// Gradient (reverse sweep), with f = e_m conj(r_K,m) / |r_K,m| and d||r_K|| = Re sum_p g_p d theta_p:
//     v_K = -C^T f
//     for k = K-1 .. 0:   w_k = P^{-T} v_{k+1}  (back substitution on the upper-triangular P^T)
//                         G  += w_k delta_k^T   (only the entries of the layout, in get_qdmat order)
//                         v_k = v_{k+1} - C^T w_k
//     g = z G
// u0 and the incoming u enter as constants.  The forward pass keeps delta_0 .. delta_{K-1} in a per-thread array
// (K <= kMaxSweeps): kMaxSweeps * M * 16 bytes of local memory per thread (4000 B at M = 5, 7200 B at M = 9),
// which is allocated for the resident threads only, not per sample.  The value-only instantiation keeps none.
//
// Edge cases: ||r_K|| = 0 (e.g. lambda = 0) gives g = 0.  A norm that overflowed is +inf; a NaN in any component of
// r_K makes the norm NaN.  Both give g = 0, as does a NaN norm.  A finite norm whose gradient exceeds the float64
// range (a diverging iteration) gets non-finite entries in g.
#pragma once
#include "../../include/sdcgym.h"
#include "specrad.cuh"

namespace sdcgym {

constexpr int kMaxSweeps = 50;  // the envs' max_iters

template <int M>
struct SweepParams {
    double Q[M * M];
    double Qd[M * M];  // SDCGYM_PREC_FIXED only
    int64_t N;
    const double* lam;             // [N][2]
    const double* qd;              // [N][A](x2), or one row with qd_broadcast
    const double *u0, *u, *r;      // [N][M][2] each, or all NULL: the reset state u0 = u = 1, r = u0 - C 1
    double *u_out, *r_out;         // [N][M][2], optional
    double* norm_out;              // [N]
    double* grad;                  // [N][A][2], optional
    double dt;
    int32_t sweeps, qd_broadcast, n_act;
};

// is (r, c) a parameter of layout PT (compile-time twin of is_qd_param)
template <int PT>
SDCGYM_HD constexpr bool sweep_param(int r, int c) {
    return PT == SDCGYM_PREC_DIAG ? c == r
         : PT == SDCGYM_PREC_LOWER_DIAG ? r == c + 1
         : PT == SDCGYM_PREC_LOWER_TRI ? c <= r
         : PT == SDCGYM_PREC_STRICTLY_LOWER_TRI ? c < r
         : false;
}

// r = u0 - u + z (Q u)
template <int M>
SDCGYM_HD void sweep_residual(const double (&Q)[M * M], C2 z, const C2 (&u0)[M], const C2 (&u)[M], C2 (&r)[M]) {
#pragma unroll
    for (int a = 0; a < M; a++) {
        C2 qu{0.0, 0.0};
#pragma unroll
        for (int c = 0; c < M; c++) qu = C2{qu.r + Q[a * M + c] * u[c].r, qu.i + Q[a * M + c] * u[c].i};
        r[a] = c_add(c_sub(u0[a], u[a]), c_mul(z, qu));
    }
}

// The per-sample body is shared by the per-sample kernel (residual_sweeps_one) and the reduced kernel
// (residual_sweeps_reduced): residual_sweeps_body evaluates and hands its results to an output policy `Out`, which
// either stores them (SweepStore) or keeps what the reduction needs (SweepReduce).  The forward and reverse sweeps stay
// in one function body, and the per-sample path forms z from lam inside it (Out::kGivenZ false): factored into
// functions of their own, or with z passed in, nvcc generates different code for residual_sweeps_kernel.

// ||r||_inf = max_a hypot(r_a): nrm, m the first index attaining it, nan_seen if any component of r is NaN (the norm
// is then NaN)
template <int M>
SDCGYM_HD void sweep_norm(const C2 (&r)[M], double& nrm, int& m, bool& nan_seen) {
    nrm = 0.0;
    nan_seen = false;
    m = 0;
#pragma unroll
    for (int a = 0; a < M; a++) {
        const double v = hypot(r[a].r, r[a].i);
        nan_seen |= isnan(r[a].r) || isnan(r[a].i);
        if (v > nrm) {
            nrm = v;
            m = a;
        }
    }
}

// Out receives, in this order: start(r_0) the starting residual, norm(n_K) (NaN where r_K has a NaN), state(u_K, r_K),
// and with GRAD grad(k, q, g_k) for each parameter k, q = its dense index r * M + c (g = 0 where n_K is 0, +inf or
// NaN).
template <int M, int PT, bool QC, bool GRAD, class Out>
SDCGYM_HD void residual_sweeps_body(const SweepParams<M>& p, int64_t i, Out& out) {
    const C2 z = Out::kGivenZ ? out.z : C2{p.lam[2 * i] * p.dt, p.lam[2 * i + 1] * p.dt};
    // zQd = z * Qd on and below the diagonal, inv[r] = 1 / P_rr
    C2 zQd[M * M], inv[M];
    constexpr int w = QC ? 2 : 1;
    const double* row = (PT == SDCGYM_PREC_FIXED) ? nullptr : p.qd + (p.qd_broadcast ? 0 : i * (int64_t)p.n_act * w);
    int k = 0;
#pragma unroll
    for (int r = 0; r < M; r++)
#pragma unroll
        for (int c = 0; c <= r; c++) {
            C2 d{0.0, 0.0};
            if (PT == SDCGYM_PREC_FIXED) {
                d.r = p.Qd[r * M + c];
            } else if (sweep_param<PT>(r, c)) {
                d.r = row[k * w];
                if (QC) d.i = row[k * w + 1];
                k++;
            }
            zQd[r * M + c] = c_mul(z, d);
        }
#pragma unroll
    for (int r = 0; r < M; r++) inv[r] = c_div(C2{1.0, 0.0}, c_sub(C2{1.0, 0.0}, zQd[r * M + r]));

    C2 u0[M], u[M], r[M];
    if (p.u0) {
#pragma unroll
        for (int a = 0; a < M; a++) {
            u0[a] = C2{p.u0[(i * M + a) * 2], p.u0[(i * M + a) * 2 + 1]};
            u[a] = C2{p.u[(i * M + a) * 2], p.u[(i * M + a) * 2 + 1]};
            r[a] = C2{p.r[(i * M + a) * 2], p.r[(i * M + a) * 2 + 1]};
        }
    } else {
#pragma unroll
        for (int a = 0; a < M; a++) u0[a] = u[a] = C2{1.0, 0.0};
        sweep_residual<M>(p.Q, z, u0, u, r);
    }
    out.start(r);

    C2 hist[GRAD ? kMaxSweeps * M : 1];  // delta_k, k = 0 .. K-1
    for (int s = 0; s < p.sweeps; s++) {
        C2 dl[M];
#pragma unroll
        for (int a = 0; a < M; a++) {
            C2 acc = r[a];
#pragma unroll
            for (int c = 0; c < a; c++)
                if (PT == SDCGYM_PREC_FIXED || sweep_param<PT>(a, c)) acc = c_add(acc, c_mul(zQd[a * M + c], dl[c]));
            dl[a] = c_mul(acc, inv[a]);
            u[a] = c_add(u[a], dl[a]);
            if (GRAD) hist[s * M + a] = dl[a];
        }
        sweep_residual<M>(p.Q, z, u0, u, r);
    }

    double nrm;
    int m;
    bool nan_seen;
    sweep_norm<M>(r, nrm, m, nan_seen);
    out.norm(nan_seen ? nan("") : nrm);
    out.state(u, r);
    if constexpr (GRAD) {
        C2 G[M * M];
#pragma unroll
        for (int q = 0; q < M * M; q++) G[q] = C2{0.0, 0.0};
        const bool ok = nrm > 0.0 && nrm <= 1.7976931348623157e308 && !nan_seen;
        if (ok) {
            // f_m = conj(r_m) / |r_m|;  v = -C^T f = -f_m (e_m - z Q_{m,:}^T)
            C2 fm{0.0, 0.0};
#pragma unroll
            for (int a = 0; a < M; a++)
                if (a == m) fm = c_scale(c_conj(r[a]), 1.0 / nrm);
            const C2 zf = c_mul(z, fm);
            C2 v[M];
#pragma unroll
            for (int c = 0; c < M; c++) {
                double qmc = 0.0;
#pragma unroll
                for (int a = 0; a < M; a++)
                    if (a == m) qmc = p.Q[a * M + c];
                v[c] = c_scale(zf, qmc);
                if (c == m) v[c] = c_sub(v[c], fm);
            }
            for (int s = p.sweeps - 1; s >= 0; s--) {
                C2 wv[M];
#pragma unroll
                for (int a = M - 1; a >= 0; a--) {
                    C2 acc = v[a];
#pragma unroll
                    for (int q = a + 1; q < M; q++)
                        if (PT == SDCGYM_PREC_FIXED || sweep_param<PT>(q, a)) acc = c_add(acc, c_mul(zQd[q * M + a], wv[q]));
                    wv[a] = c_mul(acc, inv[a]);
                }
#pragma unroll
                for (int a = 0; a < M; a++)
#pragma unroll
                    for (int c = 0; c <= a; c++)
                        if (sweep_param<PT>(a, c)) G[a * M + c] = c_add(G[a * M + c], c_mul(wv[a], hist[s * M + c]));
                // v -= C^T w = w - z Q^T w
#pragma unroll
                for (int c = 0; c < M; c++) {
                    C2 qw{0.0, 0.0};
#pragma unroll
                    for (int a = 0; a < M; a++) qw = C2{qw.r + p.Q[a * M + c] * wv[a].r, qw.i + p.Q[a * M + c] * wv[a].i};
                    v[c] = c_add(c_sub(v[c], wv[c]), c_mul(z, qw));
                }
            }
        }
        int kk = 0;
#pragma unroll
        for (int a = 0; a < M; a++)
#pragma unroll
            for (int c = 0; c <= a; c++)
                if (sweep_param<PT>(a, c)) {
                    out.grad(kk, a * M + c, ok ? c_mul(z, G[a * M + c]) : C2{0.0, 0.0});
                    kk++;
                }
    }
}

// the per-sample outputs of sdcgym_residual_sweeps: norm_out[i], optionally u_out[i], r_out[i], and grad[i] = g
template <int M, int PT>
struct SweepStore {
    static constexpr bool kGivenZ = false;  // z = lam[i] dt
    static constexpr C2 z{0.0, 0.0};
    const SweepParams<M>& p;
    int64_t i;
    SDCGYM_HD void start(const C2 (&)[M]) {}
    SDCGYM_HD void norm(double v) { p.norm_out[i] = v; }
    SDCGYM_HD void state(const C2 (&u)[M], const C2 (&r)[M]) {
#pragma unroll
        for (int a = 0; a < M; a++) {
            if (p.u_out) {
                p.u_out[(i * M + a) * 2] = u[a].r;
                p.u_out[(i * M + a) * 2 + 1] = u[a].i;
            }
            if (p.r_out) {
                p.r_out[(i * M + a) * 2] = r[a].r;
                p.r_out[(i * M + a) * 2 + 1] = r[a].i;
            }
        }
    }
    SDCGYM_HD void grad(int k, int, C2 gv) {
        double* g = p.grad + i * (int64_t)p.n_act * 2;
        g[2 * k] = gv.r;
        g[2 * k + 1] = gv.i;
    }
};

// sample i: PT the layout (SDCGYM_PREC_FIXED: p.Qd), QC complex parameters, GRAD write the gradient
template <int M, int PT, bool QC, bool GRAD>
SDCGYM_HD void residual_sweeps_one(const SweepParams<M>& p, int64_t i) {
    if (i >= p.N) return;
    SweepStore<M, PT> out{p, i};
    residual_sweeps_body<M, PT, QC, GRAD>(p, i, out);
}

// Reductions of sdcgym_residual_sweeps_sum: per-sample value f and weight of g
//   SDCGYM_SWEEPS_MEAN       f = n_K                g
//   SDCGYM_SWEEPS_LOG_RATIO  f = log(n_K / n_0)     g / n_K
// with n_0 = ||r_0||_inf of the starting residual (same hypot / max / NaN rule as n_K) and g = 0 where n_K is 0, +inf
// or NaN.  log_ratio: a sample with n_0 = 0 (lambda = 0 from the reset state) contributes exact zeros to f and to the
// gradient; any other non-finite f (n_K = 0 gives -inf, NaN) is returned as it is.
template <int M>
struct SweepReduce {
    static constexpr bool kGivenZ = true;
    C2 z;  // lambda dt, from the list or the grid
    int reduction;
    double n0, nK, f;
    C2 (&gw)[M * M];  // the weighted g, dense (the caller zeroes it: entries outside the layout stay 0)
    SDCGYM_HD void start(const C2 (&r)[M]) {
        int m;
        bool nan_seen;
        sweep_norm<M>(r, n0, m, nan_seen);
        if (nan_seen) n0 = nan("");
    }
    SDCGYM_HD void norm(double v) {
        nK = v;
        f = reduction != SDCGYM_SWEEPS_LOG_RATIO ? nK : n0 == 0.0 ? 0.0 : log(nK / n0);
    }
    SDCGYM_HD void state(const C2 (&)[M], const C2 (&)[M]) {}
    SDCGYM_HD void grad(int, int q, C2 gv) {
        if (reduction != SDCGYM_SWEEPS_LOG_RATIO)
            gw[q] = gv;
        else if (n0 != 0.0 && nK > 0.0 && nK <= 1.7976931348623157e308)  // elsewhere g = 0, and 0 / n_K may be NaN
            gw[q] = c_scale(gv, 1.0 / nK);
    }
};

// Sample i of sdcgym_residual_sweeps_sum, lambda given as z = lambda dt: returns f, sets nK = n_K (NaN where r_K has a
// NaN) and gw = the weighted g
template <int M, int PT, bool QC>
SDCGYM_HD double residual_sweeps_reduced(const SweepParams<M>& p, int64_t i, C2 z, int reduction, double& nK,
                                         C2 (&gw)[M * M]) {
#pragma unroll
    for (int q = 0; q < M * M; q++) gw[q] = C2{0.0, 0.0};
    SweepReduce<M> out{z, reduction, 0.0, 0.0, 0.0, gw};
    residual_sweeps_body<M, PT, QC, true>(p, i, out);
    nK = out.nK;
    return out.f;
}

template <int M>
inline void fill_sweep_params(SweepParams<M>& p, const sdcgym_rho_desc* d, int64_t N, int sweeps, const double* lam,
                              const double* qd, const double* u0, const double* u, const double* r, double* u_out,
                              double* r_out, double* norm_out, double* grad) {
    for (int k = 0; k < M * M; k++) {
        p.Q[k] = d->Q[k];
        p.Qd[k] = d->Qd_fixed[k];
    }
    p.N = N;
    p.lam = lam;
    p.qd = qd;
    p.u0 = u0;
    p.u = u;
    p.r = r;
    p.u_out = u_out;
    p.r_out = r_out;
    p.norm_out = norm_out;
    p.grad = grad;
    p.dt = d->dt;
    p.sweeps = sweeps;
    p.qd_broadcast = d->qd_broadcast;
    p.n_act = sdcgym_num_actions(M, d->prec_type);
}

}  // namespace sdcgym

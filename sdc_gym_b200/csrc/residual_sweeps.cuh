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

// sample i: PT the layout (SDCGYM_PREC_FIXED: p.Qd), QC complex parameters, GRAD write the gradient
template <int M, int PT, bool QC, bool GRAD>
SDCGYM_HD void residual_sweeps_one(const SweepParams<M>& p, int64_t i) {
    if (i >= p.N) return;
    const C2 z{p.lam[2 * i] * p.dt, p.lam[2 * i + 1] * p.dt};
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

    double nrm = 0.0;
    bool nan_seen = false;
    int m = 0;
#pragma unroll
    for (int a = 0; a < M; a++) {
        const double v = hypot(r[a].r, r[a].i);
        nan_seen |= isnan(r[a].r) || isnan(r[a].i);
        if (v > nrm) {
            nrm = v;
            m = a;
        }
    }
    p.norm_out[i] = nan_seen ? nan("") : nrm;
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
        double* g = p.grad + i * (int64_t)p.n_act * 2;
        int kk = 0;
#pragma unroll
        for (int a = 0; a < M; a++)
#pragma unroll
            for (int c = 0; c <= a; c++)
                if (sweep_param<PT>(a, c)) {
                    const C2 gv = ok ? c_mul(z, G[a * M + c]) : C2{0.0, 0.0};
                    g[2 * kk] = gv.r;
                    g[2 * kk + 1] = gv.i;
                    kk++;
                }
    }
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

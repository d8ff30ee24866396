// specrad_params.cuh - parameter block and per-matrix body of the spectral-radius kernel.
#pragma once
#include "../../include/sdcgym.h"
#include "specrad.cuh"

extern "C" int sdcgym_num_actions(int M, int prec_type);

namespace sdcgym {

template <int M>
struct RhoParams {
    double Q[M * M];
    double Qd[M * M];
    int64_t N;
    const double* lam;  // [N][2] or NULL (grid mode)
    const double* qd;   // [N][A](x2) or one row (broadcast) or NULL
    double* rho;
    double dt;
    int64_t grid_re, grid_im, grid_first;
    double re_lo, re_hi, im_lo, im_hi;
    int32_t prec_type, qd_is_complex, qd_broadcast, n_act;
};

// Is the dense entry (r, c) of Q_delta a parameter of the action layout prec_type?  Parameters are numbered in
// row-major order of the entries for which this holds.
SDCGYM_HD bool is_qd_param(int prec_type, int r, int c) {
    switch (prec_type) {
    case SDCGYM_PREC_DIAG: return c == r;
    case SDCGYM_PREC_LOWER_DIAG: return r == c + 1;
    case SDCGYM_PREC_LOWER_TRI: return c <= r;
    case SDCGYM_PREC_STRICTLY_LOWER_TRI: return c < r;
    default: return false;
    }
}

// lambda = lr + i li at node g of the (p.grid_re x p.grid_im) tensor grid over [p.re_lo, p.re_hi] x [p.im_lo, p.im_hi]:
// row-major over (re, im), end points included (np.linspace semantics).  P: any parameter block with these fields
// (read through the reference: passing them by value changes the code nvcc generates for rho_kernel).
template <class P>
SDCGYM_HD void grid_lambda(const P& p, int64_t g, double& lr, double& li) {
    int64_t a = g / p.grid_im, b = g - a * p.grid_im;
    lr = (p.grid_re > 1) ? p.re_lo + (p.re_hi - p.re_lo) * ((double)a / (double)(p.grid_re - 1)) : p.re_lo;
    li = (p.grid_im > 1) ? p.im_lo + (p.im_hi - p.im_lo) * ((double)b / (double)(p.grid_im - 1)) : p.im_lo;
}

// ROW: the parameter row is p.qd + qd_off for every sample (a population row, sdcgym_spectral_radius_grad_sum_population)
template <int M, bool ROW = false>
SDCGYM_HD bool rho_inputs(const RhoParams<M>& p, int64_t i, double& lr, double& li, C2 (&Qd)[M * M],
                          int64_t qd_off = 0) {
    if (i >= p.N) return false;
    if (p.lam) {
        lr = p.lam[2 * i];
        li = p.lam[2 * i + 1];
    } else {
        grid_lambda(p, p.grid_first + i, lr, li);
    }
    const int w = p.qd_is_complex ? 2 : 1;
    const double* row = p.qd ? p.qd + (ROW ? qd_off : (p.qd_broadcast ? 0 : i * (int64_t)p.n_act * w)) : nullptr;
    int k = 0;
#pragma unroll
    for (int r = 0; r < M; r++)
#pragma unroll
        for (int c = 0; c < M; c++) {
            C2 d{0.0, 0.0};
            // is_qd_param spelled out: calling it here changes the code nvcc generates for rho_kernel<8>, <9>
            bool take = false;
            switch (p.prec_type) {
            case SDCGYM_PREC_DIAG: take = (c == r); break;
            case SDCGYM_PREC_LOWER_DIAG: take = (r == c + 1); break;
            case SDCGYM_PREC_LOWER_TRI: take = (c <= r); break;
            case SDCGYM_PREC_STRICTLY_LOWER_TRI: take = (c < r); break;
            default: break;
            }
            if (p.prec_type == SDCGYM_PREC_FIXED) {
                d.r = (c <= r) ? p.Qd[r * M + c] : 0.0;
            } else if (take) {
                d.r = row[k * w];
                if (p.qd_is_complex) d.i = row[k * w + 1];
                k++;
            }
            Qd[r * M + c] = d;
        }
    return true;
}

template <int M>
SDCGYM_HD void rho_one(const RhoParams<M>& p, int64_t i) {
    double lr, li;
    C2 Qd[M * M];
    if (!rho_inputs<M>(p, i, lr, li, Qd)) return;
    p.rho[i] = spectral_radius_one<M>(p.Q, lr * p.dt, li * p.dt, Qd);
}

// rho of sample i and G = d rho / d Qd (dense, spectral_radius_grad_one); false past the end of the batch.
template <int M, bool ROW = false>
SDCGYM_HD bool rho_grad_eval(const RhoParams<M>& p, int64_t i, double& rho, C2 (&G)[M * M], int64_t qd_off = 0) {
    double lr, li;
    C2 Qd[M * M];
    if (!rho_inputs<M, ROW>(p, i, lr, li, Qd, qd_off)) return false;
    rho = spectral_radius_grad_one<M>(p.Q, lr * p.dt, li * p.dt, Qd, G);
    return true;
}

// rho and d rho / d(parameter k) for the action layout of prec_type: grad[i][k] = g (complex, interleaved),
// d rho = Re(sum_k g_k d theta_k); for real parameters the derivative is Re(g_k).
template <int M>
SDCGYM_HD void rho_grad_one(const RhoParams<M>& p, int64_t i, double* __restrict__ grad) {
    double rho;
    C2 G[M * M];
    if (!rho_grad_eval<M>(p, i, rho, G)) return;
    p.rho[i] = rho;
    double* g = grad + i * (int64_t)p.n_act * 2;
    int k = 0;
#pragma unroll
    for (int r = 0; r < M; r++)
#pragma unroll
        for (int c = 0; c < M; c++) {
            if (is_qd_param(p.prec_type, r, c)) {
                g[2 * k] = G[r * M + c].r;
                g[2 * k + 1] = G[r * M + c].i;
                k++;
            }
        }
}

template <int M>
inline void fill_rho_params(RhoParams<M>& p, const sdcgym_rho_desc* d, int64_t N, const double* lam, const double* qd,
                            double* rho) {
    for (int k = 0; k < M * M; k++) {
        p.Q[k] = d->Q[k];
        p.Qd[k] = d->Qd_fixed[k];
    }
    p.N = N;
    p.lam = lam;
    p.qd = qd;
    p.rho = rho;
    p.dt = d->dt;
    p.grid_re = d->grid_re;
    p.grid_im = d->grid_im;
    p.grid_first = d->grid_first;
    p.re_lo = d->re_lo;
    p.re_hi = d->re_hi;
    p.im_lo = d->im_lo;
    p.im_hi = d->im_hi;
    p.prec_type = d->prec_type;
    p.qd_is_complex = d->qd_is_complex;
    p.qd_broadcast = d->qd_broadcast;
    p.n_act = sdcgym_num_actions(M, d->prec_type);
}

}  // namespace sdcgym

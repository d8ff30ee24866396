// specrad.cuh - batched spectral radius of the SDC iteration matrix, one matrix per thread.
//
//   rho( lam*dt * inv(I - lam*dt*Qd) @ (Q - Qd) )        dp_playground.py:216-228, sdc_env.py:421-425
//
// The reference evaluates this with LAPACK (inv + matmul + zgeev) per sample.  Here each thread
//   1. forms K = z * P^{-1} (Q - Qd) by forward substitution (all supported Q_delta are lower triangular:
//      diag / lower_diag / lower_tri / strictly_lower_tri layouts and the fixed LU^T, MIN, EE, zeros),
//   2. reduces K to upper Hessenberg form with Householder reflectors,
//   3. runs the explicitly shifted complex QR iteration (Wilkinson shift, Givens rotations, deflation from
//      the bottom) and keeps max |eigenvalue|.
// Everything is unrolled over compile-time indices with run-time predicates so the M x M matrix stays in
// registers (M <= 5) instead of local memory.  Power iteration is unusable here: |mu_2/mu_1| has median
// 0.95 on the lambda box (SURVEY.md 7, hard part 4).  Target accuracy: 1e-10 relative against LAPACK.
//
// Unlike the env kernels nothing here has to follow a particular rounding sequence, so this file is compiled
// with FMA contraction enabled.
#pragma once
#include "exact_math.cuh"

#ifndef SDCGYM_QR_HOOK
#define SDCGYM_QR_HOOK(hi)  // experiment hook (tools/qr_iteration_count.cpp): one QR step on the leading (hi+1) block
#endif

namespace sdcgym {

struct C2 {
    double r, i;
};
SDCGYM_HD C2 c_add(C2 a, C2 b) { return C2{a.r + b.r, a.i + b.i}; }
SDCGYM_HD C2 c_sub(C2 a, C2 b) { return C2{a.r - b.r, a.i - b.i}; }
SDCGYM_HD C2 c_mul(C2 a, C2 b) { return C2{a.r * b.r - a.i * b.i, a.r * b.i + a.i * b.r}; }
SDCGYM_HD C2 c_conj(C2 a) { return C2{a.r, -a.i}; }
SDCGYM_HD C2 c_scale(C2 a, double s) { return C2{a.r * s, a.i * s}; }
SDCGYM_HD double c_abs2(C2 a) { return a.r * a.r + a.i * a.i; }
SDCGYM_HD double c_abs1(C2 a) { return fabs(a.r) + fabs(a.i); }
SDCGYM_HD C2 c_div(C2 a, C2 b) {  // Smith's algorithm
    C2 q;
    if (fabs(b.r) >= fabs(b.i)) {
        double t = b.i / b.r, d = b.r + b.i * t;
        q.r = (a.r + a.i * t) / d;
        q.i = (a.i - a.r * t) / d;
    } else {
        double t = b.r / b.i, d = b.r * t + b.i;
        q.r = (a.r * t + a.i) / d;
        q.i = (a.i * t - a.r) / d;
    }
    return q;
}
SDCGYM_HD double rsqrt_pos(double x) {  // 1 / sqrt(x), x > 0
#ifdef __CUDA_ARCH__
    return rsqrt(x);
#else
    return 1.0 / sqrt(x);
#endif
}
SDCGYM_HD C2 c_sqrt(C2 a) {  // principal square root
    double mag = sqrt(c_abs2(a));
    if (mag == 0.0) return C2{0.0, 0.0};
    if (a.r >= 0.0) {
        double re = sqrt(0.5 * (mag + a.r));
        return C2{re, a.i / (2.0 * re)};
    }
    double im = sqrt(0.5 * (mag - a.r));
    return C2{fabs(a.i) / (2.0 * im), a.i >= 0.0 ? im : -im};
}

// eigenvalue modulus maximum of the M x M complex matrix H (row-major, destroyed)
template <int M>
SDCGYM_HD double max_abs_eig(C2 (&H)[M * M], C2* mu_out = nullptr) {
#define H_(i, j) H[(i) * M + (j)]
    // ---- Householder reduction to upper Hessenberg form ----
#pragma unroll
    for (int k = 0; k < M - 2; k++) {
        double nrm2 = 0.0;
#pragma unroll
        for (int i = k + 1; i < M; i++) nrm2 += c_abs2(H_(i, k));
        double tail2 = nrm2 - c_abs2(H_(k + 1, k));
        if (tail2 > 0.0 && nrm2 > 0.0) {
            double nrm = sqrt(nrm2);
            C2 x0 = H_(k + 1, k);
            double ax0 = sqrt(c_abs2(x0));
            C2 phase = (ax0 == 0.0) ? C2{1.0, 0.0} : C2{x0.r / ax0, x0.i / ax0};
            C2 alpha = c_scale(phase, -nrm);  // x -> alpha e1
            C2 v[M];
#pragma unroll
            for (int i = 0; i < M; i++) v[i] = (i > k) ? H_(i, k) : C2{0.0, 0.0};
            v[k + 1] = c_sub(v[k + 1], alpha);
            double vn2 = 0.0;
#pragma unroll
            for (int i = k + 1; i < M; i++) vn2 += c_abs2(v[i]);
            double beta = 2.0 / vn2;
            // H <- (I - beta v v^H) H
#pragma unroll
            for (int j = 0; j < M; j++) {
                C2 s{0.0, 0.0};
#pragma unroll
                for (int i = k + 1; i < M; i++) s = c_add(s, c_mul(c_conj(v[i]), H_(i, j)));
                s = c_scale(s, beta);
#pragma unroll
                for (int i = k + 1; i < M; i++) H_(i, j) = c_sub(H_(i, j), c_mul(v[i], s));
            }
            // H <- H (I - beta v v^H)
#pragma unroll
            for (int i = 0; i < M; i++) {
                C2 s{0.0, 0.0};
#pragma unroll
                for (int j = k + 1; j < M; j++) s = c_add(s, c_mul(H_(i, j), v[j]));
                s = c_scale(s, beta);
#pragma unroll
                for (int j = k + 1; j < M; j++) H_(i, j) = c_sub(H_(i, j), c_mul(s, c_conj(v[j])));
            }
#pragma unroll
            for (int i = k + 2; i < M; i++) H_(i, k) = C2{0.0, 0.0};
        }
    }

    // ---- is the matrix numerically singular?  A well-trained Q_delta makes Q - Qd (nearly) singular (MIN: one
    //      eigenvalue ~1e-10 next to a cluster of three around 0.2), and then ONE unshifted step deflates the null
    //      eigenvalue at once and the remaining, hard cluster is iterated on a smaller block: 13 instead of 21 QR steps
    //      on the MIN grid (profiles/README.md).  |det H| by Hyman's recurrence on the Hessenberg form (~2 % of the
    //      work) against the scale (||H||_F^2 / M)^(M/2); any other matrix takes the Wilkinson shift from the start. ----
    bool zero_first = false;
    if (M >= 3) {
        C2 xh[M];
        xh[M - 1] = C2{1.0, 0.0};
        bool ok = true;
        double prod2 = 1.0;
#pragma unroll
        for (int i = M - 1; i >= 1; i--) {
            C2 s{0.0, 0.0};
#pragma unroll
            for (int j = i; j < M; j++) s = c_add(s, c_mul(H_(i, j), xh[j]));
            const C2 sub = H_(i, i - 1);
            const double a2 = c_abs2(sub);
            ok = ok && (a2 > 1e-60) && (a2 < 1e60);
            prod2 *= a2;
            const double ia2 = ok ? -1.0 / a2 : 0.0;  // x_{i-1} = -s / sub = -s conj(sub) / |sub|^2
            xh[i - 1] = c_scale(c_mul(s, c_conj(sub)), ia2);
        }
        C2 top{0.0, 0.0};
        double fro2 = 0.0;
#pragma unroll
        for (int j = 0; j < M; j++) top = c_add(top, c_mul(H_(0, j), xh[j]));
#pragma unroll
        for (int k = 0; k < M * M; k++) fro2 += c_abs2(H[k]);
        double scale2 = 1.0;  // (fro2 / M)^M = scale^2
#pragma unroll
        for (int k = 0; k < M; k++) scale2 *= fro2 * (1.0 / M);
        const double det2 = c_abs2(top) * prod2;
        zero_first = ok && (det2 <= 1e-12 * scale2) && (scale2 > 0.0) && (scale2 < 1e300);
    }

    // ---- shifted QR on the Hessenberg matrix, deflating from the bottom ----
    const double eps = 2.220446049250313e-16;
    double rho = 0.0;
    C2 mu_max{0.0, 0.0};
    int hi = M - 1;
    int its = 0;
    bool failed = false;
    for (int guard = 0; guard < 40 * M && hi > 0; guard++) {
        // negligible sub-diagonal at the bottom of the active block?
        C2 sub{0.0, 0.0}, d0{0.0, 0.0}, d1{0.0, 0.0}, b01{0.0, 0.0};
#pragma unroll
        for (int k = 1; k < M; k++)
            if (k == hi) {
                sub = H_(k, k - 1);
                d0 = H_(k - 1, k - 1);
                d1 = H_(k, k);
                b01 = H_(k - 1, k);
            }
        double scale = c_abs1(d0) + c_abs1(d1);
        if (c_abs1(sub) <= eps * scale || c_abs1(sub) == 0.0) {
            double a = sqrt(c_abs2(d1));
            if (a > rho) mu_max = d1;
            rho = a > rho ? a : rho;
            hi--;
            its = 0;
            continue;
        }
        if (its >= 60) {
            failed = true;
            break;
        }
        // Wilkinson shift: eigenvalue of [[d0, b01], [sub, d1]] closer to d1
        C2 mu;
        if (zero_first) {
            mu = C2{0.0, 0.0};
            zero_first = false;
        } else if (its == 10 || its == 20) {
            mu = C2{d1.r + fabs(sub.r) + fabs(sub.i), d1.i};  // exceptional shift
        } else {
            C2 half = c_scale(c_sub(d0, d1), 0.5);
            C2 bc = c_mul(b01, sub);
            C2 disc = c_sqrt(c_add(c_mul(half, half), bc));
            C2 p = c_add(half, disc), q = c_sub(half, disc);
            C2 den = (c_abs2(p) >= c_abs2(q)) ? p : q;
            mu = (c_abs2(den) == 0.0) ? d1 : c_sub(d1, c_div(bc, den));
        }
        its++;
        SDCGYM_QR_HOOK(hi);
#pragma unroll
        for (int k = 0; k < M; k++)
            if (k <= hi) H_(k, k) = c_sub(H_(k, k), mu);
        // QR factorisation by Givens rotations G_k = [[c, s], [-conj(s), c]] with REAL c (zlartg convention:
        // c = |x| / r, s = (x / |x|) conj(y) / r): a real cosine makes every rotated element 6 instead of 10 FP64
        // instructions.  The rotations are kept for the RQ product.
        double gc[M];
        C2 gs[M];
#pragma unroll
        for (int k = 0; k < M - 1; k++) {
            gc[k] = 1.0;
            gs[k] = C2{0.0, 0.0};
            if (k < hi) {
                const C2 x = H_(k, k), y = H_(k + 1, k);
                const double ax2 = c_abs2(x), ay2 = c_abs2(y);
                if (ay2 > 0.0) {
                    if (ax2 > 0.0) {
                        const double ir = rsqrt_pos(ax2 + ay2), iax = rsqrt_pos(ax2);
                        gc[k] = ax2 * iax * ir;
                        gs[k] = c_scale(c_mul(c_scale(x, iax), c_conj(y)), ir);
                    } else {
                        gc[k] = 0.0;
                        gs[k] = c_scale(c_conj(y), rsqrt_pos(ay2));
                    }
                }
                const double c = gc[k];
                const C2 s = gs[k];
#pragma unroll
                for (int j = k; j < M; j++) {
                    if (j <= hi) {
                        const C2 a = H_(k, j), b = H_(k + 1, j);
                        H_(k, j) = C2{c * a.r + (s.r * b.r - s.i * b.i), c * a.i + (s.r * b.i + s.i * b.r)};
                        H_(k + 1, j) = C2{c * b.r - (s.r * a.r + s.i * a.i), c * b.i - (s.r * a.i - s.i * a.r)};
                    }
                }
            }
        }
        // RQ: H <- H G_k^H, G_k^H = [[c, -s], [conj(s), c]], applied to the columns
#pragma unroll
        for (int k = 0; k < M - 1; k++) {
            if (k < hi) {
                const double c = gc[k];
                const C2 s = gs[k];
#pragma unroll
                for (int i = 0; i <= k + 1; i++) {
                    const C2 a = H_(i, k), b = H_(i, k + 1);
                    H_(i, k) = C2{c * a.r + (b.r * s.r + b.i * s.i), c * a.i + (b.i * s.r - b.r * s.i)};
                    H_(i, k + 1) = C2{c * b.r - (a.r * s.r - a.i * s.i), c * b.i - (a.r * s.i + a.i * s.r)};
                }
            }
        }
#pragma unroll
        for (int k = 0; k < M; k++)
            if (k <= hi) H_(k, k) = c_add(H_(k, k), mu);
    }
    if (failed || hi > 0) return d_nan();
    double a = sqrt(c_abs2(H_(0, 0)));
    if (a > rho) mu_max = H_(0, 0);
    if (mu_out) *mu_out = mu_max;
    return a > rho ? a : rho;
#undef H_
}

// K = z * P^{-1} (Q - Qd) with P = I - z Qd lower triangular.  Qd: row-major dense complex (upper part ignored).
template <int M>
SDCGYM_HD double spectral_radius_one(const double* Q, double zr, double zi, const C2 (&Qd)[M * M]) {
    const C2 z{zr, zi};
    C2 X[M * M];
#pragma unroll
    for (int i = 0; i < M; i++) {
        C2 pii = c_sub(C2{1.0, 0.0}, c_mul(z, Qd[i * M + i]));
        C2 inv = c_div(C2{1.0, 0.0}, pii);
#pragma unroll
        for (int c = 0; c < M; c++) {
            C2 acc{0.0, 0.0};
#pragma unroll
            for (int j = 0; j < i; j++) acc = c_add(acc, c_mul(Qd[i * M + j], X[j * M + c]));
            C2 b = C2{Q[i * M + c], 0.0};
            if (c <= i) b = c_sub(b, Qd[i * M + c]);
            X[i * M + c] = c_mul(c_add(b, c_mul(z, acc)), inv);
        }
    }
#pragma unroll
    for (int k = 0; k < M * M; k++) X[k] = c_mul(z, X[k]);
    return max_abs_eig<M>(X);
}

// ---------------------------------------------------------------------------------------------------------
// Gradient of rho with respect to the Q_delta entries (SURVEY 8f item 2: what jax.value_and_grad(loss) needs,
// dp_playground.py:1073).  For a simple dominant eigenvalue mu with right / left eigenvectors x, y:
//     d mu = y^H dK x / (y^H x),        K = z P^{-1} (Q - Qd),  P = I - z Qd
//     dK   = z P^{-1} dQd (K - I)       =>  d mu / d Qd_ij = z conj(w_i) (mu - 1) x_j / (y^H x),   w = P^{-H} y
//     d rho = Re( conj(mu)/|mu| d mu )  =>  g_ij = conj(mu)/|mu| * d mu / d Qd_ij   (d rho = Re(sum g_ij dQd_ij))
// Eigenvectors come from three steps of inverse iteration on (B - mu' I) with a slightly perturbed shift, where
// B = D^{-1} K D is K balanced by powers of two (LAPACK zgebal without permutations).  P^{-1} grows geometrically
// along the rows for large |z Qd|, so the entries of x and y span many orders of magnitude; on K itself their small
// entries would carry errors of eps * max|x|, and the lower_diag / strictly_lower_tri gradients pair exactly those
// small entries with each other.  On B they come out to a few eps each, componentwise.  The LU with partial
// pivoting is unrolled with predicated row swaps so everything stays in registers for small M.
// ---------------------------------------------------------------------------------------------------------
template <int M>
SDCGYM_HD void balance(C2 (&B)[M * M], double (&dsc)[M]) {
#pragma unroll
    for (int i = 0; i < M; i++) dsc[i] = 1.0;
    bool changed = true;
    for (int sweep = 0; sweep < 16 && changed; sweep++) {
        changed = false;
#pragma unroll
        for (int i = 0; i < M; i++) {
            double c = 0.0, r = 0.0;
#pragma unroll
            for (int j = 0; j < M; j++)
                if (j != i) {
                    c += c_abs1(B[j * M + i]);
                    r += c_abs1(B[i * M + j]);
                }
            if (!(c > 0.0 && r > 0.0 && c < 1e300 && r < 1e300)) continue;
            const int e = (ilogb(r) - ilogb(c)) / 2;  // column i times 2^e, row i times 2^-e: c 2^e ~ r 2^-e
            const double f = ldexp(1.0, e), g = ldexp(1.0, -e);
            if (e == 0 || !(c * f + r * g < 0.95 * (c + r))) continue;
            changed = true;
            dsc[i] *= f;
#pragma unroll
            for (int j = 0; j < M; j++) {
                B[j * M + i] = c_scale(B[j * M + i], f);
                B[i * M + j] = c_scale(B[i * M + j], g);
            }
        }
    }
}
template <int M>
SDCGYM_HD void lu_factor(C2 (&A)[M * M], int (&piv)[M]) {
#pragma unroll
    for (int k = 0; k < M; k++) {
        int p = k;
        double best = c_abs1(A[k * M + k]);
#pragma unroll
        for (int i = k + 1; i < M; i++) {
            const double v = c_abs1(A[i * M + k]);
            if (v > best) {
                best = v;
                p = i;
            }
        }
        piv[k] = p;
        // swap the active columns only: the multipliers of earlier steps stay in the row order they were computed
        // in, which is the order lu_solve applies them in (interleaved with the swaps, LINPACK dgefa/dgesl)
#pragma unroll
        for (int q = k + 1; q < M; q++) {
            const bool sw = (p == q);
#pragma unroll
            for (int c = k; c < M; c++) {
                const C2 t = A[k * M + c];
                A[k * M + c] = sw ? A[q * M + c] : t;
                A[q * M + c] = sw ? t : A[q * M + c];
            }
        }
        C2 d = A[k * M + k];
        if (c_abs2(d) == 0.0) d = C2{1e-300, 0.0};  // exactly singular shift: any tiny pivot does for inverse iteration
        A[k * M + k] = d;
        const C2 inv = c_div(C2{1.0, 0.0}, d);
#pragma unroll
        for (int i = k + 1; i < M; i++) {
            const C2 l = c_mul(A[i * M + k], inv);
            A[i * M + k] = l;
#pragma unroll
            for (int c = k + 1; c < M; c++) A[i * M + c] = c_sub(A[i * M + c], c_mul(l, A[k * M + c]));
        }
    }
}
template <int M>
SDCGYM_HD void lu_solve(const C2 (&A)[M * M], const int (&piv)[M], C2 (&b)[M]) {
#pragma unroll
    for (int k = 0; k < M; k++) {
#pragma unroll
        for (int q = k + 1; q < M; q++) {
            const bool sw = (piv[k] == q);
            const C2 t = b[k];
            b[k] = sw ? b[q] : t;
            b[q] = sw ? t : b[q];
        }
#pragma unroll
        for (int i = k + 1; i < M; i++) b[i] = c_sub(b[i], c_mul(A[i * M + k], b[k]));
    }
#pragma unroll
    for (int k = M - 1; k >= 0; k--) {
#pragma unroll
        for (int c = k + 1; c < M; c++) b[k] = c_sub(b[k], c_mul(A[k * M + c], b[c]));
        b[k] = c_div(b[k], A[k * M + k]);
    }
}
template <int M>
SDCGYM_HD void normalize_vec(C2 (&v)[M]) {
    double m = 0.0;
#pragma unroll
    for (int i = 0; i < M; i++) m = fmax(m, c_abs1(v[i]));
    const double s = (m > 0.0 && m < 1e300) ? 1.0 / m : 1.0;
#pragma unroll
    for (int i = 0; i < M; i++) v[i] = c_scale(v[i], s);
}

// rho and its gradient: grad[(i*M + j)] = g_ij (complex), for the structurally non-zero (lower-triangular) entries.
template <int M>
SDCGYM_HD double spectral_radius_grad_one(const double* Q, double zr, double zi, const C2 (&Qd)[M * M], C2 (&G)[M * M]) {
    const C2 z{zr, zi};
    C2 K[M * M], H[M * M];
#pragma unroll
    for (int i = 0; i < M; i++) {
        const C2 inv = c_div(C2{1.0, 0.0}, c_sub(C2{1.0, 0.0}, c_mul(z, Qd[i * M + i])));
#pragma unroll
        for (int c = 0; c < M; c++) {
            C2 acc{0.0, 0.0};
#pragma unroll
            for (int j = 0; j < i; j++) acc = c_add(acc, c_mul(Qd[i * M + j], K[j * M + c]));
            C2 b = C2{Q[i * M + c], 0.0};
            if (c <= i) b = c_sub(b, Qd[i * M + c]);
            K[i * M + c] = c_mul(c_add(b, c_mul(z, acc)), inv);  // K holds X = P^{-1}(Q - Qd) for now
        }
    }
#pragma unroll
    for (int k = 0; k < M * M; k++) {
        K[k] = c_mul(z, K[k]);
        H[k] = K[k];
    }
    C2 mu;
    const double rho = max_abs_eig<M>(H, &mu);
#pragma unroll
    for (int k = 0; k < M * M; k++) G[k] = C2{0.0, 0.0};
    if (!(rho > 1e-300) || rho != rho) return rho;  // mu = 0 (lambda = 0) or failed iteration: zero gradient
    double dsc[M];
    balance<M>(K, dsc);  // K <- D^{-1} K D, the same eigenvalues
    // shifted matrices: A = K - mu' I (right vector), At = A^H (left vector)
    const C2 mus = c_mul(mu, C2{1.0 + 3e-11, 2e-11});
    C2 A[M * M], At[M * M];
#pragma unroll
    for (int i = 0; i < M; i++)
#pragma unroll
        for (int j = 0; j < M; j++) {
            C2 a = K[i * M + j];
            if (i == j) a = c_sub(a, mus);
            A[i * M + j] = a;
            At[j * M + i] = c_conj(a);
        }
    int piv[M], pivt[M];
    lu_factor<M>(A, piv);
    lu_factor<M>(At, pivt);
    C2 x[M], y[M];
#pragma unroll
    for (int i = 0; i < M; i++) {
        x[i] = C2{1.0, 0.1 * (i + 1)};
        y[i] = C2{1.0, -0.1 * (i + 1)};
    }
#pragma unroll
    for (int it = 0; it < 3; it++) {
        lu_solve<M>(A, piv, x);
        normalize_vec<M>(x);
        lu_solve<M>(At, pivt, y);
        normalize_vec<M>(y);
    }
    // back to the eigenvectors of K: x = D x_B, y = D^{-1} y_B (exact: D holds powers of two)
#pragma unroll
    for (int i = 0; i < M; i++) {
        x[i] = c_scale(x[i], dsc[i]);
        y[i] = c_scale(y[i], 1.0 / dsc[i]);
    }
    normalize_vec<M>(x);
    normalize_vec<M>(y);
    // w = P^{-H} y: P^H is upper triangular with entries conj(P_ji); back substitution
    C2 w[M];
#pragma unroll
    for (int i = M - 1; i >= 0; i--) {
        C2 acc = y[i];
#pragma unroll
        for (int j = i + 1; j < M; j++) {
            // (P^H)_{ij} = conj(P_{ji}) = conj(-z Qd_{ji})
            acc = c_add(acc, c_mul(c_conj(c_mul(z, Qd[j * M + i])), w[j]));
        }
        w[i] = c_div(acc, c_conj(c_sub(C2{1.0, 0.0}, c_mul(z, Qd[i * M + i]))));
    }
    C2 yhx{0.0, 0.0};
#pragma unroll
    for (int i = 0; i < M; i++) yhx = c_add(yhx, c_mul(c_conj(y[i]), x[i]));
    // common factor: conj(mu)/|mu| * z * (mu - 1) / (y^H x)
    C2 f = c_mul(c_scale(c_conj(mu), 1.0 / rho), c_mul(z, c_sub(mu, C2{1.0, 0.0})));
    f = c_div(f, yhx);
#pragma unroll
    for (int i = 0; i < M; i++)
#pragma unroll
        for (int j = 0; j <= i; j++) G[i * M + j] = c_mul(f, c_mul(c_conj(w[i]), x[j]));
    return rho;
}

}  // namespace sdcgym

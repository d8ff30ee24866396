"""TEST INFRASTRUCTURE ONLY: extended-precision (mpmath, 40 digits) reference of the loss gradients.

The inputs are the exact float64 values a kernel receives: ``Q`` (``collocation_matrix(M)``), the dense
``Qd = qdmat_from_output(theta)`` and ``z = fl(lam.real * dt) + i fl(lam.imag * dt)``.  Everything after that runs
in mpmath, so the results are the true values of the operation on those inputs to far below float64 rounding.

``SpecRadRef``: ``rho = |mu|``, ``mu`` the dominant eigenvalue of ``K = z P^{-1} (Q - Qd)``, ``P = I - z Qd``.
LAPACK's eigenpair only seeds a Newton iteration on the bordered eigen-system in mp; the gradient then follows
from the left/right eigenvector formula (``d rho = Re sum_k g_k d theta_k``, the kernel's convention).
``rho_directional`` is the independent check: a central difference in mp that never uses eigenvectors of the
formula, only Newton-refined eigenvalues of the perturbed matrices; ``formula_directional`` is the same derivative
from the formula, also in mp.

``ResidualRef``: ``u' = u + P^{-1} r``, ``r' = u0 - C u'`` (``C`` given, or ``I - z Q``), ``||r'||_inf`` and its
gradient, with the same kind of independent difference in ``residual_directional``.
"""
from __future__ import annotations

import mpmath as mp
import numpy as np
import scipy.linalg

DPS = 40
_CTX = mp.MPContext()
_CTX.dps = DPS


def param_index(M, prec_type):
    """(row, col) of parameter k of the action layout, in the kernels' order"""
    if prec_type == "diag":
        return [(r, r) for r in range(M)]
    if prec_type == "lower_diag":
        return [(r + 1, r) for r in range(M - 1)]
    if prec_type == "lower_tri":
        return [(r, c) for r in range(M) for c in range(r + 1)]
    if prec_type == "strictly_lower_tri":
        return [(r, c) for r in range(M) for c in range(r)]
    raise ValueError(prec_type)


def z_of(lam, dt):
    """z exactly as the kernels form it: each component of lambda times dt, rounded once"""
    lam = complex(lam)
    return complex(np.float64(lam.real) * np.float64(dt), np.float64(lam.imag) * np.float64(dt))


def _m(A):
    A = np.atleast_2d(np.asarray(A, dtype=np.complex128))
    return _CTX.matrix([[_CTX.mpc(complex(v)) for v in row] for row in A])


def _c(v):
    return complex(v)


def _qd_mp(M, prec_type, theta, dtheta=None, s=0):
    """dense Qd in mp, optionally moved by s * dtheta along the parameters"""
    Qd = _CTX.zeros(M, M)
    for k, (r, c) in enumerate(param_index(M, prec_type)):
        v = _CTX.mpc(complex(theta[k]))
        if dtheta is not None:
            v += s * _CTX.mpc(complex(dtheta[k]))
        Qd[r, c] = v
    return Qd


def _K(Q, z, Qd):
    M = Q.rows
    P = _CTX.eye(M) - z * Qd
    return z * (_CTX.inverse(P) * (Q - Qd)), P


def _newton(K, mu, x, tol):
    """refine an eigenpair (mu, x) of K: Newton on [K - mu I, -x; e_p^T, 0] with x_p fixed to 1"""
    M = K.rows
    p = max(range(M), key=lambda i: abs(x[i]))
    x = x / x[p]
    for _ in range(12):
        J = _CTX.zeros(M + 1, M + 1)
        rhs = _CTX.zeros(M + 1, 1)
        r = K * x - mu * x
        for i in range(M):
            for j in range(M):
                J[i, j] = K[i, j]
            J[i, i] -= mu
            J[i, M] = -x[i]
            rhs[i] = -r[i]
        J[M, p] = 1
        d = _CTX.lu_solve(J, rhs)
        for i in range(M):
            x[i] += d[i]
        mu += d[M]
        if abs(d[M]) <= tol * abs(mu) and max(abs(d[i]) for i in range(M)) <= tol:
            break
    return mu, x


def _dominant(K, real_matrix):
    """LAPACK's dominant eigenpair (and left vector) of float64(K), plus the modulus gap and separation to the other
    eigenvalues; for a real K the conjugate partner of a complex mu does not count (it gives the same real gradient)"""
    Kf = np.array(K.tolist(), dtype=np.complex128)
    w, vl, vr = scipy.linalg.eig(Kf, left=True, right=True)
    k = int(np.argmax(abs(w)))
    a0 = abs(w[k])
    rest = np.delete(w, k)
    if real_matrix and w[k].imag != 0 and len(rest):
        rest = np.delete(rest, np.argmin(abs(rest - np.conj(w[k]))))
    if len(rest) == 0 or a0 == 0:
        return w[k], vr[:, k], vl[:, k], 1.0, 1.0
    return w[k], vr[:, k], vl[:, k], float((a0 - np.max(abs(rest))) / a0), float(np.min(abs(rest - w[k])) / a0)


class SpecRadRef:
    """mp reference of rho and its gradient for one sample; attributes rho, mu, g (complex, parameter order),
    kappa (eigenvalue condition number ||x|| ||y|| / |y^H x|), modgap ((|mu_1| - |mu_2|) / |mu_1|),
    sep (min_j |mu_j - mu_1| / |mu_1|).  ``real_matrix``: K is real (real lambda
    and outputs), so conj(mu) is an eigenvalue too and is left out of modgap and sep."""

    def __init__(self, Q, lam, dt, theta, prec_type, real_matrix=False):
        Q = np.asarray(Q, dtype=np.float64)
        M = self.M = Q.shape[0]
        self.prec_type = prec_type
        self.theta = np.asarray(theta)
        self.z = _CTX.mpc(z_of(lam, dt))
        self.Qm = _m(Q)
        Qd = _qd_mp(M, prec_type, self.theta)
        K, P = _K(self.Qm, self.z, Qd)
        if self.z == 0:
            self.rho, self.mu, self.g = 0.0, 0.0, np.zeros(len(self.theta), np.complex128)
            self._g = [_CTX.mpc(0)] * len(self.theta)
            self.kappa, self.modgap, self.sep = 1.0, 1.0, 1.0
            return
        mu0, x0, y0, self.modgap, self.sep = _dominant(K, real_matrix)
        tol = _CTX.mpf(10) ** (-(DPS - 5))
        mu, x = _newton(K, _CTX.mpc(complex(mu0)), _m(x0).T, tol)
        _, y = _newton(K.H, _CTX.conj(mu), _m(y0).T, tol)
        self._mu_mp, self._x = mu, x
        w = _CTX.lu_solve(P.H, y)
        yhx = (y.H * x)[0]
        f = _CTX.conj(mu) / abs(mu) * self.z * (mu - 1) / yhx
        self._g = [f * _CTX.conj(w[r]) * x[c] for r, c in param_index(M, prec_type)]
        self.g = np.array([_c(v) for v in self._g])
        self.rho = float(abs(mu))
        self.mu = _c(mu)
        self.kappa = float(_CTX.norm(x) * _CTX.norm(y) / abs(yhx))

    def rho_directional(self, d, h=1e-15):
        """d rho along the parameter direction d by a central difference in mp (no eigenvector formula)"""
        h = _CTX.mpf(h)
        tol = _CTX.mpf(10) ** (-(DPS - 5))
        vals = []
        for s in (1, -1):
            Qd = _qd_mp(self.M, self.prec_type, self.theta, d, s * h)
            K, _ = _K(self.Qm, self.z, Qd)
            mu, _ = _newton(K, self._mu_mp, self._x.copy(), tol)
            vals.append(abs(mu))
        return (vals[0] - vals[1]) / (2 * h)

    def formula_directional(self, d):
        """Re sum_k g_k d_k in mp"""
        return _formula_directional(self._g, d)


def _formula_directional(g, d):
    return _CTX.re(_CTX.fsum(gk * _CTX.mpc(complex(dk)) for gk, dk in zip(g, d)))


def twin_grad(Q, lam, dt, theta, prec_type):
    """the same formula in plain float64 (numpy inverse, LAPACK zgeev left + right vectors): what an fp64 computation
    of the gradient achieves on these inputs.  Returns (rho, g)."""
    Q = np.asarray(Q, dtype=np.float64)
    M = Q.shape[0]
    z = z_of(lam, dt)
    Qd = np.zeros((M, M), np.complex128)
    for k, (r, c) in enumerate(param_index(M, prec_type)):
        Qd[r, c] = theta[k]
    P = np.eye(M) - z * Qd
    K = z * np.linalg.inv(P) @ (Q - Qd)
    w, vl, vr = scipy.linalg.eig(K, left=True, right=True)
    k = int(np.argmax(abs(w)))
    mu, x, y = w[k], vr[:, k], vl[:, k]
    if mu == 0:
        return 0.0, np.zeros(len(theta), np.complex128)
    wv = np.linalg.solve(P.conj().T, y)
    f = np.conj(mu) / abs(mu) * z * (mu - 1) / (np.conj(y) @ x)
    return float(abs(mu)), np.array([f * np.conj(wv[r]) * x[c] for r, c in param_index(M, prec_type)])


class ResidualRef:
    """mp reference of one ResidualLoss step for one sample: u_new, r_new, norm = ||r_new||_inf, g (d norm =
    Re sum_k g_k d theta_k), kmax and gap2 = (|r'|_(1) - |r'|_(2)) / |r'|_(1) (the max is not differentiable where
    it vanishes).  ``C`` None means C = I - z Q."""

    def __init__(self, Q, lam, dt, theta, prec_type, u0, u, r_old, C=None):
        Q = np.asarray(Q, dtype=np.float64)
        M = self.M = Q.shape[0]
        self.prec_type = prec_type
        self.theta = np.asarray(theta)
        self.z = _CTX.mpc(z_of(lam, dt))
        self.Cm = (_CTX.eye(M) - self.z * _m(Q)) if C is None else _m(C)
        self.u0, self.u, self.r_old = _m(u0).T, _m(u).T, _m(r_old).T
        Qd = _qd_mp(M, prec_type, self.theta)
        P = _CTX.eye(M) - self.z * Qd
        delta = _CTX.lu_solve(P, self.r_old)
        un = self.u + delta
        rn = self.u0 - self.Cm * un
        mags = [abs(rn[i]) for i in range(M)]
        order = sorted(range(M), key=lambda i: -mags[i])
        k = order[0]
        self.kmax = k
        self.norm = float(mags[k])
        self.gap2 = float((mags[k] - mags[order[1]]) / mags[k]) if mags[k] > 0 and M > 1 else 1.0
        self.u_new = np.array([_c(v) for v in un])
        self.r_new = np.array([_c(v) for v in rn])
        if mags[k] == 0:
            self.g = np.zeros(len(self.theta), np.complex128)
            self._g = [_CTX.mpc(0)] * len(self.theta)
            return
        a = _CTX.lu_solve(P.T, self.Cm[k, :].T)
        f = _CTX.conj(rn[k]) / mags[k] * (-self.z)
        self._g = [f * a[r] * delta[c] for r, c in param_index(M, prec_type)]
        self.g = np.array([_c(v) for v in self._g])

    def norm_at(self, d, s):
        Qd = _qd_mp(self.M, self.prec_type, self.theta, d, s)
        P = _CTX.eye(self.M) - self.z * Qd
        rn = self.u0 - self.Cm * (self.u + _CTX.lu_solve(P, self.r_old))
        return max(abs(rn[i]) for i in range(self.M))

    def residual_directional(self, d, h=1e-15):
        """d ||r'||_inf along d by a central difference in mp"""
        h = _CTX.mpf(h)
        return (self.norm_at(d, h) - self.norm_at(d, -h)) / (2 * h)

    def formula_directional(self, d):
        return _formula_directional(self._g, d)


def residual_twin(Q, lam, dt, theta, prec_type, u0, u, r_old, C=None):
    """float64 twin of ResidualRef: (u_new, r_new, norm, g)"""
    Q = np.asarray(Q, dtype=np.float64)
    M = Q.shape[0]
    z = z_of(lam, dt)
    Qd = np.zeros((M, M), np.complex128)
    for k, (r, c) in enumerate(param_index(M, prec_type)):
        Qd[r, c] = theta[k]
    P = np.eye(M) - z * Qd
    C = np.eye(M) - z * Q if C is None else np.asarray(C)
    delta = np.linalg.solve(P, r_old)
    un = u + delta
    rn = u0 - C @ un
    k = int(np.argmax(abs(rn)))
    nrm = abs(rn[k])
    if nrm == 0:
        return un, rn, 0.0, np.zeros(len(theta), np.complex128)
    a = np.linalg.solve(P.T, C[k, :])
    f = np.conj(rn[k]) / nrm * (-z)
    return un, rn, float(nrm), np.array([f * a[r] * delta[c] for r, c in param_index(M, prec_type)])

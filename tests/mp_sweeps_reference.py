"""TEST INFRASTRUCTURE ONLY: extended-precision (mpmath, 40 digits) reference of the K-sweep residual loss.

Same conventions as ``tests/mp_reference.py``, whose helpers it uses: the inputs are the exact float64 values a kernel
receives (``Q``, the layout's ``theta`` and ``z = fl(lam.real * dt) + i fl(lam.imag * dt)``), and everything after
that runs in mpmath.

``SweepsRef``: K sweeps of the ResidualLoss iteration and the gradient of ``||r_K||_inf`` through all of them (adjoint
sweep), with ``norm_directional``, an independent central difference in mp of the forward sweeps.  ``sweeps_twin``:
the same in plain float64, what a float64 computation achieves on the same inputs.
"""
from __future__ import annotations

import numpy as np

from tests.mp_reference import _CTX, _c, _formula_directional, _m, _qd_mp, param_index, z_of


def _lower_solve(P, b):
    """x = P^{-1} b for lower-triangular P, in mp"""
    M = P.rows
    x = _CTX.zeros(M, 1)
    for i in range(M):
        x[i] = (b[i] - _CTX.fsum(P[i, j] * x[j] for j in range(i))) / P[i, i]
    return x


def _upper_solve_t(P, b):
    """x = P^{-T} b for lower-triangular P (back substitution on P^T), in mp"""
    M = P.rows
    x = _CTX.zeros(M, 1)
    for i in reversed(range(M)):
        x[i] = (b[i] - _CTX.fsum(P[j, i] * x[j] for j in range(i + 1, M))) / P[i, i]
    return x


class SweepsRef:
    """mp reference of K sweeps of the ResidualLoss iteration for one sample (no early stop):
    delta_k = P^{-1} r_k, u_{k+1} = u_k + delta_k, r_{k+1} = u0 - C u_{k+1}, C = I - z Q.  ``u0``, ``u``, ``r``
    None: the envs' reset state u0 = u = 1, r = u0 - C 1 (exact in mp).  Attributes u_K, r_K, norm = ||r_K||_inf,
    kmax, gap2 (as ResidualRef) and g, d norm = Re sum_k g_k d theta_k, from the adjoint sweep
        v_K = -C^T f, f = e_m conj(r_m) / |r_m|;  for k = K-1 .. 0: w = P^{-T} v, G += z w delta_k^T, v -= C^T w.
    ``norm_directional`` is the independent check: a central difference in mp of the forward sweeps."""

    def __init__(self, Q, lam, dt, theta, prec_type, K, u0=None, u=None, r=None):
        Q = np.asarray(Q, dtype=np.float64)
        M = self.M = Q.shape[0]
        self.prec_type, self.K = prec_type, int(K)
        self.theta = np.asarray(theta)
        self.z = _CTX.mpc(z_of(lam, dt))
        self.Cm = _CTX.eye(M) - self.z * _m(Q)
        if u0 is None:
            self.u0 = _CTX.ones(M, 1)
            self.u = _CTX.ones(M, 1)
            self.r = self.u0 - self.Cm * self.u
        else:
            self.u0, self.u, self.r = _m(u0).T, _m(u).T, _m(r).T
        P = self._P(self.theta)
        un, rn, deltas = self._forward(P)
        mags = [abs(rn[i]) for i in range(M)]
        order = sorted(range(M), key=lambda i: -mags[i])
        k = order[0]
        self.kmax = k
        self.norm = float(mags[k])
        self.gap2 = float((mags[k] - mags[order[1]]) / mags[k]) if mags[k] > 0 and M > 1 else 1.0
        self.u_K = np.array([_c(v) for v in un])
        self.r_K = np.array([_c(v) for v in rn])
        idx = param_index(M, prec_type)
        if mags[k] == 0:
            self._g = [_CTX.mpc(0)] * len(idx)
        else:
            f = _CTX.zeros(M, 1)
            f[k] = _CTX.conj(rn[k]) / mags[k]
            v = -(self.Cm.T * f)
            G = [_CTX.mpc(0)] * len(idx)
            for dl in reversed(deltas):
                w = _upper_solve_t(P, v)
                G = [G[p] + self.z * w[a] * dl[c] for p, (a, c) in enumerate(idx)]
                v = v - self.Cm.T * w
            self._g = G
        self.g = np.array([_c(v) for v in self._g], np.complex128)

    def _P(self, theta, dtheta=None, s=0):
        Qd = _qd_mp(self.M, self.prec_type, theta, dtheta, s)
        return _CTX.eye(self.M) - self.z * Qd

    def _forward(self, P):
        u, r, deltas = self.u.copy(), self.r.copy(), []
        for _ in range(self.K):
            dl = _lower_solve(P, r)
            u = u + dl
            r = self.u0 - self.Cm * u
            deltas.append(dl)
        return u, r, deltas

    def norm_at(self, d, s):
        _, rn, _ = self._forward(self._P(self.theta, d, s))
        return max(abs(rn[i]) for i in range(self.M))

    def norm_directional(self, d, h=1e-15):
        """d ||r_K||_inf along d by a central difference in mp"""
        h = _CTX.mpf(h)
        return (self.norm_at(d, h) - self.norm_at(d, -h)) / (2 * h)

    def formula_directional(self, d):
        return _formula_directional(self._g, d)


def sweeps_twin(Q, lam, dt, theta, prec_type, K, u0=None, u=None, r=None):
    """float64 twin of SweepsRef (numpy solves): (u_K, r_K, norm, g)"""
    Q = np.asarray(Q, dtype=np.float64)
    M = Q.shape[0]
    z = z_of(lam, dt)
    Qd = np.zeros((M, M), np.complex128)
    idx = param_index(M, prec_type)
    for k, (a, c) in enumerate(idx):
        Qd[a, c] = theta[k]
    P = np.eye(M) - z * Qd
    C = np.eye(M) - z * Q
    if u0 is None:
        u0, u = np.ones(M, np.complex128), np.ones(M, np.complex128)
        r = u0 - C @ u
    u, r, deltas = np.array(u, np.complex128), np.array(r, np.complex128), []
    for _ in range(K):
        dl = np.linalg.solve(P, r)
        u = u + dl
        r = u0 - C @ u
        deltas.append(dl)
    m = int(np.argmax(abs(r)))
    nrm = abs(r[m])
    g = np.zeros(len(idx), np.complex128)
    if nrm == 0 or not np.isfinite(nrm):
        return u, r, float(nrm), g
    f = np.zeros(M, np.complex128)
    f[m] = np.conj(r[m]) / nrm
    v = -C.T @ f
    for dl in reversed(deltas):
        w = np.linalg.solve(P.T, v)
        g += np.array([z * w[a] * dl[c] for a, c in idx])
        v = v - C.T @ w
    return u, r, float(nrm), g

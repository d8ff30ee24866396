"""Loss gradients against a 40-digit reference (tests/mp_reference.py), on the CPU.

1. The reference checks itself: its eigenvector-formula gradient against an mp central difference that uses no
   eigenvectors, for M = 2..9 and every Q_delta layout, and the same for the ResidualLoss gradient.
2. The host build of ``spectral_radius_grad_one`` (csrc/specrad.cuh, the template the GPU kernel instantiates) for
   M = 2..9, per sample and per entry.

Error model, per sample (eps = 2^-52, kappa = ||x|| ||y|| / |y^H x| of the dominant eigenvalue):
    rho:  |rho - rho_mp| / rho_mp                      <= 128 eps kappa
    g:    max_k |g_k - g_mp,k| / max_k |g_mp,k|         <= 64 max(twin error, eps kappa)
The twin is the same formula in plain float64 (numpy inverse, LAPACK zgeev left and right vectors, which balances
first) on the same inputs: what float64 achieves on that sample.  Measured on this grid: the template is at most
5x the twin (median 0.3x) and rho at most 9.2 eps kappa.  Samples whose dominant eigenvalue is ill-conditioned
(kappa > 1e6) or not unique in modulus (modulus gap < 1e-6, the conjugate partner of a real K excepted) are
excluded, and their number is asserted to stay small.
"""
import ctypes

import numpy as np
import pytest

from sdc_gym_b200 import _lib
from sdc_gym_b200.collocation import collocation_matrix
from sdc_gym_b200.precond import fixed_preconditioner, num_actions
from tests import host_shim
from tests import mp_reference as R

EPS = np.finfo(np.float64).eps
LAYOUTS = ("diag", "lower_diag", "lower_tri", "strictly_lower_tri")
C_GRAD, C_RHO, KAPPA_MAX, GAP_MIN = 64.0, 128.0, 1e6, 1e-6


def host_grad(M, prec_type, lam, qd, dt):
    L = host_shim.shim()
    L.shim_spectral_radius_grad.argtypes = [ctypes.POINTER(_lib.RhoDesc), ctypes.c_int64] + [ctypes.c_void_p] * 4
    d = _lib.RhoDesc()
    d.M, d.prec_type, d.dt, d.qd_is_complex = M, _lib.PREC_TYPES[prec_type], dt, int(np.iscomplexobj(qd))
    for k, v in enumerate(collocation_matrix(M).reshape(-1)):
        d.Q[k] = v
    lam = np.ascontiguousarray(lam, np.complex128)
    qd = np.ascontiguousarray(qd)
    rho, g = np.zeros(len(lam)), np.zeros((len(lam), qd.shape[1]), np.complex128)
    assert L.shim_spectral_radius_grad(ctypes.byref(d), len(lam), lam.ctypes.data, qd.ctypes.data, rho.ctypes.data,
                                       g.ctypes.data) == 0
    return rho, g


def draw(rng, M, prec_type, n, *, cplx=True, real_lam=False):
    """lambda in [-100, 0] x i[-10, 0] (real: imaginary part 0); outputs in [0.02, 0.3] (0.08 strictly lower)
    + i[-0.05, 0.05]"""
    A = num_actions(M, prec_type)
    hi = 0.08 if prec_type == "strictly_lower_tri" else 0.3
    lam = rng.uniform(-100, 0, n) + (0j if real_lam else 1j * rng.uniform(-10, 0, n))
    qd = rng.uniform(0.02, hi, (n, A))
    if cplx:
        qd = qd + 1j * rng.uniform(-0.05, 0.05, (n, A))
    return np.asarray(lam, np.complex128), qd


def check_specrad(M, prec_type, lam, qd, dt, rho, g, *, real=False):
    """per-sample comparison of a kernel's (rho, g) with the mp reference under the error model of the module
    docstring; ``real``: real outputs, so only Re(g) is the derivative.  Returns (kernel errors, twin errors,
    number excluded)."""
    Q = collocation_matrix(M)
    ek, et, excluded = [], [], 0
    for i in range(len(lam)):
        ref = R.SpecRadRef(Q, lam[i], dt, qd[i], prec_type, real_matrix=real and lam[i].imag == 0)
        _, tw = R.twin_grad(Q, lam[i], dt, qd[i], prec_type)
        assert abs(rho[i] - ref.rho) <= C_RHO * EPS * ref.kappa * ref.rho, (M, prec_type, i, rho[i], ref.rho)
        if ref.kappa > KAPPA_MAX or ref.modgap < GAP_MIN:
            excluded += 1
            continue
        gk, gr, gt = (g[i].real, ref.g.real, tw.real) if real else (g[i], ref.g, tw)
        s = np.max(np.abs(gr))
        e_k, e_t = np.max(np.abs(gk - gr)) / s, np.max(np.abs(gt - gr)) / s
        assert e_k <= C_GRAD * max(e_t, EPS * ref.kappa), (M, prec_type, dt, i, e_k, e_t, ref.kappa)
        ek.append(e_k)
        et.append(e_t)
    return np.array(ek), np.array(et), excluded


@pytest.mark.parametrize("M", range(2, 10))
def test_reference_gradient_formula_against_mp_difference(M):
    """the reference's eigenvector formula (rho) and its residual-gradient formula agree with central differences in
    mp along random complex and real directions, to ~25 digits"""
    rng = np.random.default_rng(900 + M)
    Q = collocation_matrix(M)
    for prec_type in LAYOUTS:
        lam, qd = draw(rng, M, prec_type, 2)
        lam_r, qd_r = draw(rng, M, prec_type, 1, cplx=False, real_lam=True)
        cases = [(lam[0], qd[0], 1.0), (lam[1], qd[1], 0.1), (lam_r[0], qd_r[0], 1.0)]
        for lam_i, qd_i, dt in cases:
            real = not np.iscomplexobj(qd_i) and lam_i.imag == 0
            ref = R.SpecRadRef(Q, lam_i, dt, qd_i, prec_type, real_matrix=real)
            d = rng.normal(size=len(qd_i)) + (0 if real else 1j * rng.normal(size=len(qd_i)))
            an, fd = ref.formula_directional(d), ref.rho_directional(d)
            assert abs(fd - an) <= 1e-20 * np.sum(np.abs(ref.g) * np.abs(d)), (prec_type, fd, an)
        u0 = rng.uniform(0, 1, M) + 1j * rng.uniform(0, 1, M)
        u = rng.uniform(0, 1, M) + 1j * rng.uniform(0, 1, M)
        r_old = rng.normal(size=M) + 1j * rng.normal(size=M)
        C = np.eye(M) - lam[0] * Q + 1e-3 * (rng.normal(size=(M, M)) + 1j * rng.normal(size=(M, M)))
        for C_arg in (C, None):
            ref = R.ResidualRef(Q, lam[0], 0.5, qd[0], prec_type, u0, u, r_old, C_arg)
            assert ref.gap2 > 1e-6
            d = rng.normal(size=len(qd[0])) + 1j * rng.normal(size=len(qd[0]))
            an, fd = ref.formula_directional(d), ref.residual_directional(d)
            assert abs(fd - an) <= 1e-20 * np.sum(np.abs(ref.g) * np.abs(d)), (prec_type, fd, an)


@pytest.mark.parametrize("M", range(2, 10))
def test_host_gradient_template_against_mp_reference(M):
    """host build of spectral_radius_grad_one, per sample and per entry: complex outputs at dt = 1 and 0.1, real
    outputs, and real lambda with real outputs (a real K whose dominant eigenvalue is often a conjugate pair: both
    members give the same real gradient)"""
    rng = np.random.default_rng(M)
    n_total, n_excluded = 0, 0
    for prec_type in LAYOUTS:
        for n, dt, cplx, real_lam in ((8, 1.0, True, False), (4, 0.1, True, False), (4, 1.0, False, False),
                                      (4, 1.0, False, True)):
            lam, qd = draw(rng, M, prec_type, n, cplx=cplx, real_lam=real_lam)
            rho, g = host_grad(M, prec_type, lam, qd, dt)
            _, _, ex = check_specrad(M, prec_type, lam, qd, dt, rho, g, real=not cplx)
            n_total += n
            n_excluded += ex
    assert n_excluded <= 0.03 * n_total, (n_excluded, n_total)


def test_host_gradient_edges():
    """lambda = 0 gives rho = 0 and g = 0 exactly; Q_delta within 1e-4 of MIN (K numerically singular, the QR takes
    its unshifted first step) is as accurate as anywhere else where the dominant eigenvalue is well conditioned"""
    for M in (3, 5, 9):
        for prec_type in LAYOUTS:
            A = num_actions(M, prec_type)
            qd = np.full((3, A), 0.1 + 0.01j)
            rho, g = host_grad(M, prec_type, np.zeros(3), qd, 1.0)
            assert np.all(rho == 0.0) and np.all(g == 0.0)
    rng = np.random.default_rng(5)
    n_excluded = 0
    for M in (3, 4, 5, 7):
        base = np.diag(fixed_preconditioner("min", M))
        n = 8
        lam = rng.uniform(-100, 0, n) + 1j * rng.uniform(-10, 0, n)
        qd = base[None] + rng.uniform(-1e-4, 1e-4, (n, M))
        rho, g = host_grad(M, "diag", lam, qd, 1.0)
        n_excluded += check_specrad(M, "diag", lam, qd, 1.0, rho, g, real=True)[2]
    assert n_excluded == 0  # kappa reaches 1.5e4 here: MIN clusters eigenvalues around the dominant one

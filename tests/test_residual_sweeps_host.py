"""CPU: ``sdcgym_residual_sweeps`` - the ABI's refusals, and the host build of the per-sample body
(csrc/residual_sweeps.cuh, the template the GPU kernel instantiates) against the 40-digit reference
``tests/mp_sweeps_reference.SweepsRef`` of K sweeps and of their adjoint, per sample and per entry.

Error model, per sample (eps = 2^-52, s(P) = || |P^{-1}| |P| ||_inf the Skeel condition number of P = I - z Qd):
    u_K, g:      max error / max |reference|                          <= 64 max(twin error, K M eps s(P))
    r_K, norm:   max error / (max |u0| + || |C| |u_K| ||_inf)          <= 64 max(twin error, K M eps s(P))
The twin is the same iteration and adjoint in plain float64 (numpy solves) on the same inputs.  The gradient check
leaves out samples whose two largest |r_K,m| are within 1e-6 relative (the max has no derivative there) and samples
whose ||r_K|| has converged into the rounding noise of r_K (below 1e-9 of the scale above), where no float64
computation determines the derivative; both are counted.  Where the float64 twin overflows (a diverging iteration at
K = 50), the kernel's norm must be +inf or NaN with g = 0; where only the twin's gradient overflows, the reference
gradient must be beyond the float64 range.
"""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from sdc_gym_b200 import _lib
from sdc_gym_b200.collocation import collocation_matrix
from sdc_gym_b200.precond import num_actions
from tests import mp_reference as R
from tests import mp_sweeps_reference as S
from tests.test_loss_reference_host import C_GRAD, EPS, LAYOUTS, draw

HERE = os.path.dirname(os.path.abspath(__file__))
ENULL, EUNSUPPORTED, EINVAL = -3, -2, -1
P = ctypes.c_void_p(0x1000)  # a non-NULL pointer that no checked call reaches
NOISE = 1e-9


def _desc(M=5, prec_type="diag", dt=1.0, cplx=False, broadcast=0):
    d = _lib.RhoDesc()
    d.M, d.prec_type, d.dt = M, _lib.PREC_TYPES[prec_type], dt
    d.qd_is_complex, d.qd_broadcast = int(cplx), broadcast
    if 2 <= M <= 9:
        for k, v in enumerate(collocation_matrix(M).reshape(-1)):
            d.Q[k] = v
    return d


def _call(d, N=4, K=5, lam=P, qd=P, u0=None, u=None, r=None, u_out=None, r_out=None, norm=P, grad=None):
    L = _lib.load()
    return L.sdcgym_residual_sweeps(None if d is None else ctypes.byref(d), N, K, lam, qd, u0, u, r, u_out, r_out,
                                    norm, grad, None)


def test_refusals_and_empty_batch():
    assert _call(None) == ENULL
    assert _call(_desc(), lam=None) == ENULL
    assert _call(_desc(), norm=None) == ENULL
    assert _call(_desc(), qd=None) == ENULL
    for u0, u, r in ((P, None, None), (None, P, None), (None, None, P), (P, P, None), (None, P, P)):
        assert _call(_desc(), u0=u0, u=u, r=r) == ENULL
    assert _call(_desc(M=1)) == EUNSUPPORTED
    assert _call(_desc(M=10)) == EUNSUPPORTED
    bad = _desc()
    bad.prec_type = 9
    assert _call(bad) == EUNSUPPORTED
    assert _call(_desc(prec_type="fixed"), grad=P) == EUNSUPPORTED
    assert _call(_desc(), N=-1) == EINVAL
    for K in (0, -1, 51, 1000):
        assert _call(_desc(), K=K) == EINVAL
    # N = 0 launches nothing: the pointers are never dereferenced
    assert _call(_desc(), N=0) == 0
    assert _call(_desc(), N=0, u0=P, u=P, r=P, u_out=P, r_out=P, grad=P) == 0
    assert _call(_desc(prec_type="fixed"), N=0, qd=None) == 0


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("sweeps_shim") / "libsweeps_shim.so")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-o", so,
                           os.path.join(HERE, "host_shim", "sweeps_shim.cpp")])
    L = ctypes.CDLL(so)
    L.shim_residual_sweeps.argtypes = ([ctypes.POINTER(_lib.RhoDesc), ctypes.c_int64, ctypes.c_int]
                                       + [ctypes.c_void_p] * 9)
    L.shim_residual_sweeps.restype = ctypes.c_int
    return L


def host_sweeps(L, M, prec_type, lam, theta, dt, K, u0=None, u=None, r=None):
    """the host build on (lam [B], theta [B, A] or one row [A]); returns (u_K, r_K, norms, g) as numpy arrays"""
    theta = np.ascontiguousarray(theta)
    d = _desc(M, prec_type, dt, np.iscomplexobj(theta), int(theta.ndim == 1))
    lam = np.ascontiguousarray(lam, np.complex128)
    B, A = len(lam), num_actions(M, prec_type)
    ins = [None if x is None else np.ascontiguousarray(x, np.complex128) for x in (u0, u, r)]
    u_out, r_out = np.zeros((B, M), np.complex128), np.zeros((B, M), np.complex128)
    norms, g = np.zeros(B), np.zeros((B, A), np.complex128)
    ptr = lambda x: None if x is None else x.ctypes.data  # noqa: E731
    assert L.shim_residual_sweeps(ctypes.byref(d), B, K, lam.ctypes.data, theta.ctypes.data, *map(ptr, ins),
                                  u_out.ctypes.data, r_out.ctypes.data, norms.ctypes.data, g.ctypes.data) == 0
    return u_out, r_out, norms, g


def skeel(z, M, prec_type, theta):
    Qd = np.zeros((M, M), np.complex128)
    for k, (a, c) in enumerate(R.param_index(M, prec_type)):
        Qd[a, c] = theta[k]
    Pm = np.eye(M) - z * Qd
    return np.max(np.sum(np.abs(np.linalg.inv(Pm)) @ np.abs(Pm), axis=1))


def check_sweeps(M, prec_type, lam, theta, dt, K, outs, *, u0=None, u=None, r=None, real=False):
    """per-sample comparison of K sweeps (u_K, r_K, norms, g) with SweepsRef under the module's error model.  theta
    [B, A] (or one row [A]); u0/u/r [B, M] or None (reset state).  Returns (kernel errors, twin errors, left out)."""
    u_K, r_K, norms, g = outs
    Q = collocation_matrix(M)
    ek, et, left_out = [], [], 0
    for i in range(len(lam)):
        th = theta if np.ndim(theta) == 1 else theta[i]
        ins = (None, None, None) if u0 is None else (u0[i], u[i], r[i])
        ref = S.SweepsRef(Q, lam[i], dt, th, prec_type, K, *ins)
        tu, tr, tn, tg = S.sweeps_twin(Q, lam[i], dt, th, prec_type, K, *ins)
        z = R.z_of(lam[i], dt)
        floor = K * M * EPS * skeel(z, M, prec_type, th)
        Cm = np.eye(M) - z * Q
        su = np.max(np.abs(ref.u_K))
        u0i = np.ones(M) if u0 is None else u0[i]
        sr = np.max(np.abs(u0i)) + np.max(np.abs(Cm) @ np.abs(ref.u_K))
        if not np.isfinite(tn):  # float64 overflows on this sample: so must the kernel, with g = 0
            assert not np.isfinite(norms[i]) and np.all(g[i] == 0), (M, prec_type, K, i, norms[i])
            left_out += 1
            continue
        for got, want, twin, scale, what in ((u_K[i], ref.u_K, tu, su, "u_K"), (r_K[i], ref.r_K, tr, sr, "r_K"),
                                             (norms[i], ref.norm, tn, sr, "norm")):
            e_k, e_t = np.max(np.abs(got - want)) / scale, np.max(np.abs(twin - want)) / scale
            assert e_k <= C_GRAD * max(e_t, floor), (what, M, prec_type, K, i, e_k, e_t, floor)
        if ref.norm == 0:
            assert np.all(g[i] == 0)
            continue
        if ref.gap2 < 1e-6 or ref.norm < NOISE * sr:
            left_out += 1
            continue
        if not np.all(np.isfinite(tg)):  # the adjoint of a diverging iteration leaves the float64 range
            assert np.max(np.abs(ref.g)) > 1e300
            left_out += 1
            continue
        gk, gr, gt = (g[i].real, ref.g.real, tg.real) if real else (g[i], ref.g, tg)
        s = np.max(np.abs(gr))
        e_k, e_t = np.max(np.abs(gk - gr)) / s, np.max(np.abs(gt - gr)) / s
        assert e_k <= C_GRAD * max(e_t, floor), ("g", M, prec_type, K, dt, i, e_k, e_t, floor)
        ek.append(e_k)
        et.append(e_t)
    return np.array(ek), np.array(et), left_out


def random_state(rng, M, n):
    u0 = rng.uniform(0, 1, (n, M)) + 1j * rng.uniform(0, 1, (n, M))
    u = rng.uniform(0, 1, (n, M)) + 1j * rng.uniform(0, 1, (n, M))
    r = rng.normal(size=(n, M)) + 1j * rng.normal(size=(n, M))
    return u0, u, r


@pytest.mark.parametrize("M", [2, 5, 9])
def test_reference_adjoint_against_mp_difference(M):
    """SweepsRef's adjoint sweep agrees with a central difference of its forward sweeps in mp, to ~25 digits, from the
    reset state and from a given state, along complex and real directions"""
    rng = np.random.default_rng(1100 + M)
    Q = collocation_matrix(M)
    for prec_type in LAYOUTS:
        lam, theta = draw(rng, M, prec_type, 2)
        u0, u, r = random_state(rng, M, 1)
        for K, ins, dt in ((1, (None, None, None), 1.0), (7, (u0[0], u[0], r[0]), 0.5), (12, (None, None, None), 1.0)):
            ref = S.SweepsRef(Q, lam[K % 2], dt, theta[K % 2], prec_type, K, *ins)
            assert ref.gap2 > 1e-6
            for d in (rng.normal(size=theta.shape[1]) + 1j * rng.normal(size=theta.shape[1]),
                      rng.normal(size=theta.shape[1])):
                an, fd = ref.formula_directional(d), ref.norm_directional(d)
                assert abs(fd - an) <= 1e-20 * np.sum(np.abs(ref.g) * np.abs(d)), (prec_type, K, fd, an)
    # K = 1 is ResidualRef's one-step gradient
    lam, theta = draw(rng, M, "lower_tri", 1)
    u0, u, r = random_state(rng, M, 1)
    one = R.ResidualRef(Q, lam[0], 0.5, theta[0], "lower_tri", u0[0], u[0], r[0])
    ks = S.SweepsRef(Q, lam[0], 0.5, theta[0], "lower_tri", 1, u0[0], u[0], r[0])
    assert np.allclose(ks.g, one.g, rtol=1e-30, atol=1e-25 * np.max(np.abs(one.g)))


@pytest.mark.parametrize("M", range(2, 10))
def test_host_sweeps_against_mp_reference(shim, M):
    """host build, every layout, real and complex theta, dt = 1 and 0.5, K = 1, 2, 7, 50, from the reset state and
    from a given state, per sample and per entry"""
    rng = np.random.default_rng(1200 + M)
    n_checked, n_left = 0, 0
    for prec_type in LAYOUTS:
        for cplx in (True, False):
            for dt in (1.0, 0.5):
                for K in (1, 2, 7, 50):
                    lam, theta = draw(rng, M, prec_type, 2, cplx=cplx)
                    outs = host_sweeps(shim, M, prec_type, lam, theta, dt, K)
                    ek, _, lo = check_sweeps(M, prec_type, lam, theta, dt, K, outs, real=not cplx)
                    u0, u, r = random_state(rng, M, 2)
                    outs = host_sweeps(shim, M, prec_type, lam, theta, dt, K, u0, u, r)
                    ek2, _, lo2 = check_sweeps(M, prec_type, lam, theta, dt, K, outs, u0=u0, u=u, r=r,
                                               real=not cplx)
                    n_checked += len(ek) + len(ek2)
                    n_left += lo + lo2
    assert n_checked >= 0.6 * (n_checked + n_left), (n_checked, n_left)


def test_host_sweeps_edges(shim):
    """lambda = 0: r stays 0 from the reset state, norm 0 and g = 0; K = 1 equals the one-step reference; one shared row
    gives the bits of the expanded rows; a sample that overflows is +inf with g = 0 next to finite samples"""
    rng = np.random.default_rng(7)
    for M in (3, 5, 9):
        for prec_type in LAYOUTS:
            lam, theta = draw(rng, M, prec_type, 4)
            lam[1] = 0.0
            _, r_K, norms, g = host_sweeps(shim, M, prec_type, lam, theta, 1.0, 5)
            assert norms[1] == 0.0 and np.all(r_K[1] == 0) and np.all(g[1] == 0)
            row = theta[0]
            a = host_sweeps(shim, M, prec_type, lam, row, 1.0, 7)
            b = host_sweeps(shim, M, prec_type, lam, np.repeat(row[None], 4, axis=0), 1.0, 7)
            for x, y in zip(a, b):
                assert np.array_equal(x, y)
    M = 5
    lam = np.array([-50.0 + 0j, -1e10 + 0j, -30 - 3j, np.nan + 0j])
    theta = np.full((4, M), 0.2)
    theta[1] = 0.0  # u += r: the error grows by |z| rho(Q) per sweep and overflows
    _, _, norms, g = host_sweeps(shim, M, "diag", lam, theta, 1.0, 50)
    assert np.isfinite(norms[[0, 2]]).all() and np.any(g[0] != 0) and np.any(g[2] != 0)
    assert not np.isfinite(norms[1]) and np.all(g[1] == 0)
    assert np.isnan(norms[3]) and np.all(g[3] == 0)

"""CPU: ``sdcgym_residual_sweeps_sum`` - the ABI's refusals, and the host build of its per-sample contribution
(``residual_sweeps_reduced`` in csrc/residual_sweeps.cuh, the body the reduced GPU kernel sums) against the 40-digit
reference ``tests/mp_sweeps_reference.SweepsRef`` and an mp central difference of log(n_K / n_0).

Per sample, with n = ||r_K||_inf, n_0 = ||r_0||_inf and g the gradient of n:
    mean:       f = n,               weighted gradient g         (the bits of the per-sample body)
    log_ratio:  f = log(n / n_0),    weighted gradient g / n
Tolerances follow tests/test_residual_sweeps_host.py: C_GRAD times the larger of the float64 twin's error and the
floor K M eps s(P), here scaled by sr / n (an absolute error of the norm of sr * floor is a relative error of
sr * floor / n in log n and in g / n).  Samples that module leaves out are left out here too.
"""
import ctypes
import math
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
from tests.test_residual_sweeps_host import NOISE, _desc, host_sweeps, random_state, skeel
from tests.test_residual_sweeps_host import shim as sweeps_shim  # noqa: F401  (fixture)

HERE = os.path.dirname(os.path.abspath(__file__))
ENULL, EUNSUPPORTED, EINVAL = -3, -2, -1
P = ctypes.c_void_p(0x1000)  # a non-NULL pointer that no checked call reaches
MEAN, LOG_RATIO = 0, 1


def _call(d, N=4, K=5, reduction=MEAN, lam=P, qd=P, u0=None, u=None, r=None, norm=None, scratch=P, sums=P):
    L = _lib.load()
    return L.sdcgym_residual_sweeps_sum(None if d is None else ctypes.byref(d), N, K, reduction, lam, qd, u0, u, r,
                                        norm, scratch, sums, None)


def test_refusals():
    ok = _desc(broadcast=1)
    assert _call(None) == ENULL
    assert _call(ok, qd=None) == ENULL
    assert _call(ok, scratch=None) == ENULL
    assert _call(ok, sums=None) == ENULL
    for u0, u, r in ((P, None, None), (None, P, None), (None, None, P), (P, P, None), (None, P, P)):
        assert _call(ok, u0=u0, u=u, r=r) == ENULL
    assert _call(_desc(M=1, broadcast=1)) == EUNSUPPORTED
    assert _call(_desc(M=10, broadcast=1)) == EUNSUPPORTED
    bad = _desc(broadcast=1)
    bad.prec_type = 9
    assert _call(bad) == EUNSUPPORTED
    assert _call(_desc(prec_type="fixed", broadcast=1)) == EUNSUPPORTED
    assert _call(_desc(broadcast=0)) == EINVAL
    assert _call(_desc(broadcast=2)) == EINVAL
    assert _call(ok, N=-1) == EINVAL
    for K in (0, -1, 51, 1000):
        assert _call(ok, K=K) == EINVAL
    for red in (-1, 2, 7):
        assert _call(ok, reduction=red) == EINVAL
    # grid mode (lam NULL): the range [grid_first, grid_first + N) must lie inside the grid, and the state is the
    # reset state
    g = _desc(broadcast=1)
    g.grid_re, g.grid_im, g.grid_first = 4, 3, 0
    assert _call(g, N=13, lam=None) == EINVAL
    assert _call(g, N=12, lam=None, u0=P, u=P, r=P) == EINVAL
    g.grid_first = 10
    assert _call(g, N=3, lam=None) == EINVAL
    g.grid_first = -1
    assert _call(g, N=1, lam=None) == EINVAL
    g.grid_first, g.grid_im = 0, 0
    assert _call(g, N=1, lam=None) == EINVAL
    g.grid_im, g.grid_re = 3, 0
    assert _call(g, N=1, lam=None) == EINVAL


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("sweeps_sum_shim") / "libsweeps_sum_shim.so")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-o", so,
                           os.path.join(HERE, "host_shim", "sweeps_sum_shim.cpp")])
    L = ctypes.CDLL(so)
    L.shim_residual_sweeps_reduced.argtypes = ([ctypes.POINTER(_lib.RhoDesc), ctypes.c_int64, ctypes.c_int,
                                                ctypes.c_int] + [ctypes.c_void_p] * 8)
    L.shim_residual_sweeps_reduced.restype = ctypes.c_int
    return L


def host_reduced(L, M, prec_type, lam, row, dt, K, reduction, u0=None, u=None, r=None):
    """the host build of one shared row over lam [B]: (f [B], n_K [B], weighted g [B, A]) as numpy arrays"""
    row = np.ascontiguousarray(row)
    d = _desc(M, prec_type, dt, np.iscomplexobj(row), 1)
    lam = np.ascontiguousarray(lam, np.complex128)
    B, A = len(lam), num_actions(M, prec_type)
    ins = [None if x is None else np.ascontiguousarray(x, np.complex128) for x in (u0, u, r)]
    f, nK, gw = np.zeros(B), np.zeros(B), np.zeros((B, A), np.complex128)
    ptr = lambda x: None if x is None else x.ctypes.data  # noqa: E731
    assert L.shim_residual_sweeps_reduced(ctypes.byref(d), B, K, reduction, lam.ctypes.data, row.ctypes.data,
                                          *map(ptr, ins), f.ctypes.data, nK.ctypes.data, gw.ctypes.data) == 0
    return f, nK, gw


def _log_ratio_fd(ref, n0, d, h=1e-15):
    """d log(n_K / n_0) along d by a central difference in mp of the forward sweeps (n_0 does not depend on theta)"""
    ctx = R._CTX
    h = ctx.mpf(h)
    return (ctx.log(ref.norm_at(d, h) / n0) - ctx.log(ref.norm_at(d, -h) / n0)) / (2 * h)


@pytest.mark.parametrize("M", [2, 5, 9])
def test_log_ratio_contribution_against_mp_reference(shim, sweeps_shim, M):
    """every layout, real and complex rows, K = 1, 7, 50, from the reset state and from a given state: the mean
    contribution is the per-sample body's bits, the log_ratio contribution matches SweepsRef per sample and per entry,
    and its gradient matches an mp central difference of log(n_K / n_0)"""
    rng = np.random.default_rng(3100 + M)
    Q = collocation_matrix(M)
    ctx = R._CTX
    n_checked, n_left = 0, 0
    for prec_type in LAYOUTS:
        for cplx in (True, False):
            for K in (1, 7, 50):
                lam, theta = draw(rng, M, prec_type, 2, cplx=cplx)
                row = theta[0]
                for given in (False, True):
                    ins = random_state(rng, M, 2) if given else (None, None, None)
                    _, _, norms, g = host_sweeps(sweeps_shim, M, prec_type, lam, row, 1.0, K, *ins)
                    f, nK, gw = host_reduced(shim, M, prec_type, lam, row, 1.0, K, MEAN, *ins)
                    eq = lambda a, b: np.array_equal(a, b, equal_nan=True)  # noqa: E731
                    assert eq(nK, norms) and eq(f, norms) and eq(gw, g)
                    f, nK, gw = host_reduced(shim, M, prec_type, lam, row, 1.0, K, LOG_RATIO, *ins)
                    assert eq(nK, norms)
                    for i in range(len(lam)):
                        st = (None, None, None) if not given else (ins[0][i], ins[1][i], ins[2][i])
                        ref = S.SweepsRef(Q, lam[i], 1.0, row, prec_type, K, *st)
                        tu, tr, tn, tg = S.sweeps_twin(Q, lam[i], 1.0, row, prec_type, K, *st)
                        n0 = max(abs(ref.r[a]) for a in range(M))
                        z = R.z_of(lam[i], 1.0)
                        C = np.eye(M) - z * Q
                        r0_t = (np.ones(M) - C @ np.ones(M)) if not given else st[2]
                        n0_t = np.max(np.abs(r0_t))
                        u0i = np.ones(M) if not given else st[0]
                        sr = np.max(np.abs(u0i)) + np.max(np.abs(C) @ np.abs(ref.u_K))
                        floor = K * M * EPS * skeel(z, M, prec_type, row)
                        if (not np.isfinite(tn) or ref.norm == 0 or ref.gap2 < 1e-6 or ref.norm < NOISE * sr
                                or not np.all(np.isfinite(tg))):
                            n_left += 1
                            continue
                        rel = floor * (1 + sr / ref.norm)
                        f_ref = float(ctx.log(ctx.mpf(ref.norm) / n0))
                        f_t = math.log(tn / n0_t)
                        assert abs(f[i] - f_ref) <= C_GRAD * max(abs(f_t - f_ref), rel), (prec_type, K, i, f[i], f_ref)
                        w_ref = ref.g / ref.norm
                        s = np.max(np.abs(w_ref))
                        gk, gt = (gw[i], tg / tn) if cplx else (gw[i].real, (tg / tn).real)
                        wr = w_ref if cplx else w_ref.real
                        e_k, e_t = np.max(np.abs(gk - wr)) / s, np.max(np.abs(gt - wr)) / s
                        assert e_k <= C_GRAD * max(e_t, rel), (prec_type, K, i, e_k, e_t, rel)
                        # the weighted gradient is exactly g * (1 / n) of the per-sample body
                        assert np.array_equal(gw[i], g[i] * (1.0 / norms[i]))
                        if i == 0:  # the independent check: a central difference in mp
                            d = rng.normal(size=row.shape) + (1j * rng.normal(size=row.shape) if cplx else 0)
                            fd = float(_log_ratio_fd(ref, n0, d))
                            an = float(np.real(np.sum(gw[i] * d)))
                            scale = float(np.sum(np.abs(w_ref) * np.abs(d)))
                            assert abs(fd - an) <= C_GRAD * max(e_t, rel) * scale, (prec_type, K, fd, an)
                        n_checked += 1
    assert n_checked >= 0.6 * (n_checked + n_left), (n_checked, n_left)


def test_contribution_edges(shim):
    """lambda = 0 from the reset state (n_0 = 0): both reductions add exact zeros; a given state with r = 0 but u not
    the solution (n_0 = 0, n_K > 0): log_ratio adds zeros, mean adds n_K and its gradient; a NaN lambda gives NaN f"""
    M = 5
    rng = np.random.default_rng(11)
    for prec_type in LAYOUTS:
        lam, theta = draw(rng, M, prec_type, 3)
        lam[1] = 0.0
        lam[2] = complex(np.nan, 0.0)
        for red in (MEAN, LOG_RATIO):
            f, nK, gw = host_reduced(shim, M, prec_type, lam, theta[0], 1.0, 5, red)
            assert f[1] == 0.0 and nK[1] == 0.0 and np.all(gw[1] == 0)
            assert np.isfinite(f[0]) and np.any(gw[0] != 0)
            assert np.isnan(f[2]) and np.all(gw[2] == 0)
        u0, u, _ = random_state(rng, M, 3)
        r = np.zeros((3, M), np.complex128)
        lam[1:] = lam[0]
        f, nK, gw = host_reduced(shim, M, prec_type, lam, theta[0], 1.0, 3, LOG_RATIO, u0, u, r)
        assert np.all(f == 0.0) and np.all(gw == 0) and np.all(nK > 0)
        f, nK, gw = host_reduced(shim, M, prec_type, lam, theta[0], 1.0, 3, MEAN, u0, u, r)
        assert np.array_equal(f, nK) and np.all(f > 0) and np.all(np.any(gw != 0, axis=1))

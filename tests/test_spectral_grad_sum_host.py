"""CPU: argument checks of sdcgym_spectral_radius_grad_sum and its scratch-size query.  Every refusal returns before
any CUDA call, so these run without a GPU (the pointers are never dereferenced)."""
import ctypes

import pytest

from sdc_gym_b200 import _lib
from sdc_gym_b200.precond import num_actions

ENULL, EUNSUPPORTED, EINVAL = -3, -2, -1
P = ctypes.c_void_p(0x1000)  # a non-NULL pointer that no checked call reaches


def _desc(M=5, prec_type="diag", broadcast=1):
    d = _lib.RhoDesc()
    d.M, d.prec_type, d.qd_broadcast, d.dt = M, _lib.PREC_TYPES[prec_type], broadcast, 1.0
    return d


def _call(d, N=4, lam=P, qd=P, rho=None, scratch=P, sums=P):
    L = _lib.load()
    return L.sdcgym_spectral_radius_grad_sum(None if d is None else ctypes.byref(d), N, lam, qd, rho, scratch, sums,
                                             None)


def test_refusals():
    assert _call(None) == ENULL
    assert _call(_desc(), qd=None) == ENULL
    assert _call(_desc(), scratch=None) == ENULL
    assert _call(_desc(), sums=None) == ENULL
    assert _call(_desc(M=1)) == EUNSUPPORTED
    assert _call(_desc(M=10)) == EUNSUPPORTED
    bad = _desc()
    bad.prec_type = 9
    assert _call(bad) == EUNSUPPORTED
    assert _call(_desc(prec_type="fixed")) == EUNSUPPORTED
    assert _call(_desc(broadcast=0)) == EINVAL
    assert _call(_desc(), N=-1) == EINVAL
    # grid mode (lam NULL): the range [grid_first, grid_first + N) must lie inside the grid
    g = _desc()
    g.grid_re, g.grid_im, g.grid_first = 4, 3, 0
    assert _call(g, N=13, lam=None) == EINVAL
    g.grid_first = 10
    assert _call(g, N=3, lam=None) == EINVAL
    g.grid_first = -1
    assert _call(g, N=1, lam=None) == EINVAL
    g.grid_first, g.grid_im = 0, 0
    assert _call(g, N=1, lam=None) == EINVAL
    g.grid_im, g.grid_re = 3, 0
    assert _call(g, N=1, lam=None) == EINVAL


def test_scratch_size_is_monotone_and_zero_at_n_zero():
    L = _lib.load()
    f = L.sdcgym_spectral_radius_grad_sum_scratch_doubles
    assert f(5, _lib.PREC_TYPES["fixed"], 10) == EUNSUPPORTED
    assert f(10, 0, 10) == EUNSUPPORTED and f(5, 9, 10) == EUNSUPPORTED
    assert f(5, 0, -1) == EINVAL
    for M in (2, 5, 9):
        for pt in ("diag", "lower_diag", "lower_tri", "strictly_lower_tri"):
            code = _lib.PREC_TYPES[pt]
            nv = 1 + 2 * num_actions(M, pt)
            assert f(M, code, 0) == 0
            assert f(M, code, 1) == nv  # one tile partial, folded straight into the sums
            ns = [0, 1, 127, 128, 129, 128 * 256, 128 * 256 + 1, 1 << 20, 4096 * 4096, 1 << 40]
            sizes = [f(M, code, n) for n in ns]
            assert sizes == sorted(sizes), (M, pt, sizes)
            for n, s in zip(ns, sizes):
                tiles = -(-n // 128)
                assert s % nv == 0 and s >= nv * tiles  # room for every tile's partial
                assert s <= nv * (tiles + tiles // 255 + 64)  # plus the much smaller fold levels

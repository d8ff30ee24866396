"""CPU: the population entry points of ABI 14 (``sdcgym_full_solve_counts_population``,
``sdcgym_spectral_radius_grad_sum_population``) - every refusal returns before any CUDA call, so these run without a
device (the pointers are never dereferenced) - and the host-side rules of ``PopulationSummary``."""
import ctypes
import os
import re

import numpy as np

from sdc_gym_b200 import _lib
from sdc_gym_b200.iterations import CountSummary, PopulationSummary, count_stats
from tests import host_shim

ENULL, EUNSUPPORTED, EINVAL = -3, -2, -1
P = ctypes.c_void_p(0x1000)  # a non-NULL pointer that no checked call reaches
HERE = os.path.dirname(os.path.abspath(__file__))


def test_abi_version():
    L = _lib.load()
    assert _lib.ABI_VERSION == 14 and L.sdcgym_abi_version() == 14
    names = _lib.exported_symbols()
    assert "sdcgym_full_solve_counts_population" in names
    assert "sdcgym_spectral_radius_grad_sum_population" in names


# ---- counts ---------------------------------------------------------------------------------------------------------
def _edesc(M=5, prec=None, prec_type="diag", kind="sdc-v0"):
    return host_shim.make_desc(kind, M, prec=prec, prec_type=prec_type)


def _grid(n_re=4, n_im=3, first=0):
    g = _lib.LambdaGrid()
    g.n_re, g.n_im, g.first = n_re, n_im, first
    g.re_lo, g.re_hi, g.im_lo, g.im_hi = -100.0, 0.0, -10.0, 0.0
    return g


def _counts(d, grid=None, N=4, lam=P, npop=3, action=P, a_rs=5, a_cs=1, hist=P):
    L = _lib.load()
    return L.sdcgym_full_solve_counts_population(None if d is None else ctypes.byref(d),
                                                 None if grid is None else ctypes.byref(grid), N, lam, npop, action,
                                                 a_rs, a_cs, hist, None)


def test_counts_refusals():
    ok = _edesc()
    assert _counts(None) == ENULL
    assert _counts(ok, hist=None) == ENULL
    assert _counts(ok, action=None) == ENULL
    assert _counts(ok, lam=None) == ENULL  # list mode needs lambdas
    assert _counts(_edesc(kind="sdc-v1")) == EUNSUPPORTED
    for prec in ("LU", "min"):  # a fixed preconditioner has no rows
        assert _counts(_edesc(prec=prec)) == EUNSUPPORTED
    for M in (1, 10):
        bad = _edesc()
        bad.M = M
        assert _counts(bad) == EUNSUPPORTED
    bad = _edesc()
    bad.prec_type = 9
    assert _counts(bad) == EUNSUPPORTED
    bad = _edesc()
    bad.blas_variant = 2
    assert _counts(bad) == EUNSUPPORTED
    for npop in (0, -1):
        assert _counts(ok, npop=npop) == EINVAL
    assert _counts(ok, N=-1) == EINVAL
    for it in (-1, 16385):
        bad = _edesc()
        bad.max_iters = it
        assert _counts(bad) == EINVAL
    assert _counts(ok, grid=_grid(), N=13, lam=None) == EINVAL
    assert _counts(ok, grid=_grid(first=10), N=3, lam=None) == EINVAL
    assert _counts(ok, grid=_grid(first=-1), N=1, lam=None) == EINVAL
    assert _counts(ok, grid=_grid(n_im=0), N=1, lam=None) == EINVAL
    assert _counts(ok, grid=_grid(n_re=0), N=1, lam=None) == EINVAL


# ---- rho sums -------------------------------------------------------------------------------------------------------
def _rdesc(M=5, prec_type="diag", broadcast=1):
    d = _lib.RhoDesc()
    d.M, d.prec_type, d.qd_broadcast, d.dt = M, _lib.PREC_TYPES[prec_type], broadcast, 1.0
    return d


def _rho(d, N=4, lam=P, npop=3, qd=P, qd_rs=5, scratch=P, sums=P):
    L = _lib.load()
    return L.sdcgym_spectral_radius_grad_sum_population(None if d is None else ctypes.byref(d), N, lam, npop, qd, qd_rs,
                                                        scratch, sums, None)


def test_rho_refusals():
    assert _rho(None) == ENULL
    assert _rho(_rdesc(), qd=None) == ENULL
    assert _rho(_rdesc(), scratch=None) == ENULL
    assert _rho(_rdesc(), sums=None) == ENULL
    assert _rho(_rdesc(M=1)) == EUNSUPPORTED
    assert _rho(_rdesc(M=10)) == EUNSUPPORTED
    bad = _rdesc()
    bad.prec_type = 9
    assert _rho(bad) == EUNSUPPORTED
    assert _rho(_rdesc(prec_type="fixed")) == EUNSUPPORTED
    assert _rho(_rdesc(broadcast=0)) == EINVAL
    for npop in (0, -1):
        assert _rho(_rdesc(), npop=npop) == EINVAL
    assert _rho(_rdesc(), N=-1) == EINVAL
    g = _rdesc()
    g.grid_re, g.grid_im, g.grid_first = 4, 3, 0
    assert _rho(g, N=13, lam=None) == EINVAL
    g.grid_first = 10
    assert _rho(g, N=3, lam=None) == EINVAL
    g.grid_first = -1
    assert _rho(g, N=1, lam=None) == EINVAL
    g.grid_first, g.grid_im = 0, 0
    assert _rho(g, N=1, lam=None) == EINVAL


def test_scratch_is_documented_as_p_times_the_single_row_size():
    """there is no population scratch query: the header states P times the single-row size, which the Python layer
    allocates"""
    with open(os.path.join(HERE, "..", "include", "sdcgym.h")) as f:
        text = " ".join(re.sub(r"^\s*\* ", "", line) for line in f.read().splitlines())
    text = " ".join(text.split())
    i = text.index("int sdcgym_spectral_radius_grad_sum_population(")
    comment = text[text.rindex("/*", 0, i): i]
    assert re.search(r"P \* sdcgym_spectral_radius_grad_sum_scratch_doubles\(M, prec_type, N\) doubles", comment)
    assert "sdcgym_spectral_radius_grad_sum_population_scratch" not in text
    with open(os.path.join(HERE, "..", "sdc_gym_b200", "loss.py")) as f:
        assert "P * n_scratch" in f.read()


# ---- PopulationSummary on host histograms ---------------------------------------------------------------------------
class _HostHist:
    """stands in for the device tensor: ``.cpu().numpy()`` and indexing"""

    def __init__(self, a):
        self.a = np.asarray(a, np.int64)
        self.shape = self.a.shape

    def cpu(self):
        return self

    def numpy(self):
        return self.a

    def __getitem__(self, k):
        return _HostHist(self.a[k])


def test_population_summary_rows_are_count_summaries():
    rng = np.random.default_rng(0)
    nb = 53
    h = rng.integers(0, 5, (6, nb))
    h[1] = 0  # empty set: rate 0, mean 666
    h[2, :50] = 0  # nothing succeeds (only converged-at-50, err and exhausted)
    h[3] = 0
    h[3, 1] = 1  # the lambda = 0 node alone
    s = PopulationSummary(_HostHist(h), 50)
    assert len(s) == 6 and s.hist.shape == (6, nb)
    for p in range(6):
        one = CountSummary(_HostHist(h[p]), 50)
        r = s[p]
        for k in ("count", "n_err", "n_exhausted", "n_success", "success_rate", "mean_niter"):
            assert getattr(r, k) == getattr(one, k), (p, k)
            assert float(getattr(s, k)[p]) == float(getattr(one, k)), (p, k)
    assert s.success_rate[1] == 0.0 and s.mean_niter[1] == 666.0 and s[1].mean_niter == 666
    assert s.mean_niter[2] == 666.0 and s.count[2] == h[2].sum() and s[3].mean_niter == 1.0
    # the 50th-sweep rule: bin 50 is counted but is not a success
    hh = np.zeros(nb, np.int64)
    hh[50], hh[10] = 3, 1
    c = count_stats(hh, 50)
    assert c[0] == 4 and c[3] == 1 and c[4] == 0.25 and c[5] == 10.0

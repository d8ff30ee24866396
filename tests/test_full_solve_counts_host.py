"""CPU: ``sdcgym_full_solve_counts`` - the ABI's refusals with no device, and the host build of its per-node path
(full_solve_counts_kernel: step_one with ResetEval, tests/host_shim/counts_shim.cpp) against the golden ``sdc-v0``
cases, the env path of the same host build, and the correctly rounded grid nodes."""
import ctypes
import os
import subprocess
from fractions import Fraction

import numpy as np
import pytest

from sdc_gym_b200 import _lib
from sdc_gym_b200.precond import num_actions
from tests import host_shim
from tests.helpers import assert_same, case_arrays, case_ids, case_meta

HERE = os.path.dirname(os.path.abspath(__file__))
ENULL, EUNSUPPORTED, EINVAL = -3, -2, -1
P = ctypes.c_void_p(0x1000)  # a non-NULL pointer that no checked call reaches
MAX_ITERS = 50


def _desc(M=5, prec=None, prec_type="diag", kind="sdc-v0", **kw):
    return host_shim.make_desc(kind, M, prec=prec, prec_type=prec_type, **kw)


def _call(d, grid=None, N=4, lam=P, action=P, a_es=5, a_cs=1, hist=None):
    L = _lib.load()
    return L.sdcgym_full_solve_counts(None if d is None else ctypes.byref(d), None if grid is None else ctypes.byref(grid),
                                      N, lam, action, a_es, a_cs, None, None, None, None, hist, None)


def _grid(n_re=4, n_im=3, first=0, box=(-100.0, 0.0, -10.0, 0.0)):
    g = _lib.LambdaGrid()
    g.n_re, g.n_im, g.first = n_re, n_im, first
    g.re_lo, g.re_hi, g.im_lo, g.im_hi = box
    return g


def test_refusals():
    ok = _desc()
    assert _call(None) == ENULL
    assert _call(_desc(kind="sdc-v1")) == EUNSUPPORTED
    for M in (1, 10):
        bad = _desc()
        bad.M = M
        assert _call(bad) == EUNSUPPORTED
    bad = _desc()
    bad.prec_type = 9
    assert _call(bad) == EUNSUPPORTED
    bad = _desc()
    bad.blas_variant = 2
    assert _call(bad) == EUNSUPPORTED
    assert _call(ok, N=-1) == EINVAL
    for it in (-1, 16385):
        bad = _desc()
        bad.max_iters = it
        assert _call(bad) == EINVAL
    # actions: required for a learned layout, refused with a fixed prec
    assert _call(ok, action=None) == ENULL
    assert _call(_desc(prec="LU"), action=P) == EINVAL
    assert _call(_desc(prec="min"), action=P) == EINVAL
    # list mode needs lambdas
    assert _call(ok, lam=None) == ENULL
    # grid mode: one shared row, and the node range inside the grid
    assert _call(ok, grid=_grid(), N=12, lam=None, a_es=5) == EINVAL
    assert _call(ok, grid=_grid(), N=13, lam=None, a_es=0) == EINVAL
    assert _call(ok, grid=_grid(first=10), N=3, lam=None, a_es=0) == EINVAL
    assert _call(ok, grid=_grid(first=-1), N=1, lam=None, a_es=0) == EINVAL
    assert _call(ok, grid=_grid(n_im=0), N=1, lam=None, a_es=0) == EINVAL
    assert _call(ok, grid=_grid(n_re=0), N=1, lam=None, a_es=0) == EINVAL
    # N = 0 without a histogram launches nothing
    assert _call(ok, N=0, lam=None, action=None) == 0
    assert _call(ok, grid=_grid(), N=0, lam=None, action=None, a_es=0) == 0


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("counts_shim") / "libcounts_shim.so")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-mfma", "-o", so,
                           os.path.join(HERE, "host_shim", "counts_shim.cpp")])
    L = ctypes.CDLL(so)
    L.shim_full_solve_counts.argtypes = [ctypes.POINTER(_lib.EnvDesc), ctypes.POINTER(_lib.LambdaGrid), ctypes.c_int64,
                                         ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64] + \
        [ctypes.c_void_p] * 5
    L.shim_full_solve_counts.restype = ctypes.c_int
    return L


def host_counts(L, d, lam=None, actions=None, shared=False, grid=None, N=None):
    """(niter, residual, flags, lam_out, hist) of the host build; actions (N, A) rows or, with shared, one row (A,)"""
    if grid is None:
        lam = np.ascontiguousarray(lam, np.complex128)
        N = len(lam)
    a = es = cs = None
    if actions is not None:
        a = np.ascontiguousarray(actions)
        w = 2 if np.iscomplexobj(a) else 1
        es, cs = (0 if shared else a.shape[-1] * w), w
    niter, res = np.full(N, -1, np.int32), np.full(N, np.nan)
    flags, lam_out = np.full(N, 255, np.uint8), np.full((N, 2), np.nan)
    hist = np.full(d.max_iters + 3, -1, np.int64)
    rc = L.shim_full_solve_counts(ctypes.byref(d), None if grid is None else ctypes.byref(grid), N,
                                  None if grid is not None else lam.ctypes.data, None if a is None else a.ctypes.data,
                                  es or 0, cs or 0, niter.ctypes.data, res.ctypes.data, flags.ctypes.data,
                                  lam_out.ctypes.data, hist.ctypes.data)
    assert rc == 0
    return niter, res, flags, lam_out.view(np.complex128).reshape(N), hist


def _hist_of(niter, flags, max_iters=MAX_ITERS):
    conv, err = (flags & 2) != 0, (flags & 4) != 0
    h = np.bincount(niter[conv & ~err], minlength=max_iters + 3)[: max_iters + 3].astype(np.int64)
    h[max_iters + 1] = int(err.sum())
    h[max_iters + 2] = int((~conv & ~err).sum())
    return h


V0_CASES = [c for c in case_ids() if case_meta(c)["kind"] == "sdc-v0"]


@pytest.mark.parametrize("name", V0_CASES)
def test_golden_first_step(shim, name):
    """the step after the reset of every golden sdc-v0 case: niter and residual bit-equal to the reference, flags equal
    to the env path's (reset + step of the same host build), the histogram the bincount of the per-node outputs"""
    meta, g = case_meta(name), case_arrays(name)
    M, n = meta["M"], meta["n"]
    d = _desc(M, prec=meta["prec"], prec_type=meta["prec_type"] if meta["prec"] is None else "diag", dt=meta["dt"],
              restol=meta["restol"], cplx=meta["cplx"], do_scale=meta["do_scale"], use_doubles=meta["use_doubles"])
    A = 0 if meta["prec"] else num_actions(M, meta["prec_type"])
    act = g["actions"][:, 0, :A] if A else None
    niter, res, flags, lam_out, hist = host_counts(shim, d, g["lam"], act)
    assert np.array_equal(niter, g["niter"][:, 0]), name
    assert_same(res, g["residual"][:, 0], f"{name} residual")
    assert np.array_equal(lam_out, g["lam"])
    env = host_shim.ShimBatch(d, n)
    env.reset(g["lam"])
    out = env.step(act)
    assert np.array_equal(flags, env.flags[:n]) and np.array_equal(niter, out["niter"])
    assert np.array_equal(hist, _hist_of(niter, flags)) and hist.sum() == n  # the clamped threads are not counted
    if A:  # one row shared by every node (a_es = 0) is the per-node rows all equal to it
        row = act[0]
        s_niter, s_res, s_flags, _, s_hist = host_counts(shim, d, g["lam"], row, shared=True)
        e_niter, e_res, e_flags, _, e_hist = host_counts(shim, d, g["lam"], np.tile(row, (n, 1)))
        assert np.array_equal(s_niter, e_niter) and assert_same(s_res, e_res, name) is None
        assert np.array_equal(s_flags, e_flags) and np.array_equal(s_hist, e_hist)


def fma_node(lo, hi, a, n):
    """fma(hi - lo, a / (n - 1), lo), correctly rounded (the node of grid_lambda in the contracted builds)"""
    if n <= 1:
        return lo
    return float(Fraction(hi - lo) * Fraction(a / (n - 1)) + Fraction(lo))


def test_grid_nodes_are_the_fused_nodes(shim):
    """grid mode: lam_out is the correctly rounded fma node (the bits of SpectralRadiusLoss.grid), including nodes where
    the unfused form lo + (hi - lo) * (a / (n - 1)) rounds differently; every node's outputs equal list mode's on
    those lambdas; rows of the grid concatenate to it; the corner lambda = 0 converges as the env path says"""
    n_re, n_im, box = 37, 41, (-100.0, 0.0, -10.0, 0.0)
    d = _desc(5, prec="min")
    niter, res, flags, lam_out, hist = host_counts(shim, d, grid=_grid(n_re, n_im, 0, box), N=n_re * n_im)
    a, b = np.divmod(np.arange(n_re * n_im), n_im)
    ref = np.array([complex(fma_node(box[0], box[1], int(i), n_re), fma_node(box[2], box[3], int(j), n_im))
                    for i, j in zip(a, b)])
    assert np.array_equal(lam_out.view(np.float64), ref.view(np.float64))
    unfused = box[0] + (box[1] - box[0]) * (a / (n_re - 1))
    assert np.any(unfused != ref.real), "the grid has no node where the two forms differ"
    l_niter, l_res, l_flags, _, l_hist = host_counts(shim, d, lam_out)
    assert np.array_equal(niter, l_niter) and np.array_equal(flags, l_flags) and np.array_equal(hist, l_hist)
    assert_same(res, l_res, "grid vs list")
    # rows 10..20 of the grid: the same nodes and outputs
    r_niter, r_res, _, r_lam, _ = host_counts(shim, d, grid=_grid(n_re, n_im, 10 * n_im, box), N=10 * n_im)
    assert np.array_equal(r_lam, lam_out[10 * n_im: 20 * n_im]) and np.array_equal(r_niter, niter[10 * n_im: 20 * n_im])
    # the corner node lambda = 0: r0 = 0, converged (after the one sweep the env also takes)
    assert lam_out[-1] == 0 and (flags[-1] & 2) and not (flags[-1] & 4) and res[-1] == 0.0
    env = host_shim.ShimBatch(d, 1)
    env.reset([0.0])
    assert env.step(None)["niter"][0] == niter[-1]


def test_reset_norm_matters(shim):
    """the divergence test compares with ||r0|| of the reset state: a lambda whose residual first grows is an err node in
    the env path and here (with ||r0|| read as 0 every node would be err)"""
    d = _desc(5, prec="zeros")
    lam = np.array([-100.0 + 0j, -0.5 + 0j, -3.0 - 1.0j])
    niter, res, flags, _, hist = host_counts(shim, d, lam)
    env = host_shim.ShimBatch(d, 3)
    env.reset(lam)
    out = env.step(None)
    assert np.array_equal(niter, out["niter"]) and np.array_equal(flags, env.flags[:3])
    assert (flags[0] & 4) and not (flags[1] & 4) and (flags[1] & 2)
    assert hist[MAX_ITERS + 1] == 1 and hist.sum() == 3

"""GPU: the reduced K-sweep residual loss of ONE shared parameter row (``residual_sweeps_sum_kernel`` through
``sdcgym_residual_sweeps_sum``, ``ResidualLoss.sweeps_shared_value_and_grad`` / ``sweeps_grid_value_and_grad``) against
the per-sample kernel (``ResidualLoss.sweeps(..., with_grad=True)``) with its contributions summed exactly by
``math.fsum``."""
import ctypes
import math
import os
import socket

import numpy as np
import pytest
import torch

from sdc_gym_b200 import _lib
from sdc_gym_b200.loss import SWEEPS_REDUCTIONS, ResidualLoss
from tests.test_gpu_spectral_grad_sum import IM_BOX, LAYOUTS, RE_BOX, _lams, _row, assert_tree_sums, host_grid

pytestmark = pytest.mark.gpu

EPS = np.finfo(np.float64).eps


def fused(loss, N, K, reduction, lam=None, row=None, grid=None, state=None, stream=None):
    """sdcgym_residual_sweeps_sum straight through the C ABI with the per-sample norm requested: (sums (1 + 2A,),
    norms (N,)) as numpy.  ``grid=(n_re, n_im, first)`` selects grid mode over the default box; ``state`` = (u0, u, r)."""
    sr = loss._sr
    d = _lib.RhoDesc.from_buffer_copy(sr._desc)
    qd, is_c, _ = sr._outputs_tensor(row, 1)
    d.qd_is_complex, d.qd_broadcast = is_c, 1
    lam_r = None
    if grid is None:
        lam_r = torch.view_as_real(torch.as_tensor(np.asarray(lam, np.complex128), device=loss.device).contiguous())
        d.grid_re = d.grid_im = d.grid_first = 0
    else:
        d.grid_re, d.grid_im, d.grid_first = grid
        d.re_lo, d.re_hi, d.im_lo, d.im_hi = *RE_BOX, *IM_BOX
    st = [None] * 3 if state is None else [loss._c128(x, (N, loss.M)) for x in state]
    L = sr._L
    n_scratch = L.sdcgym_spectral_radius_grad_sum_scratch_doubles(loss.M, d.prec_type, N)
    scratch = torch.full((max(n_scratch, 1),), np.nan, dtype=torch.float64, device=loss.device)  # never NULL
    sums = torch.full((1 + 2 * sr.n_out,), np.nan, dtype=torch.float64, device=loss.device)
    norms = torch.full((N,), np.nan, dtype=torch.float64, device=loss.device)
    s = torch.cuda.current_stream() if stream is None else stream
    ptr = lambda t: None if t is None else t.data_ptr()  # noqa: E731
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        rc = L.sdcgym_residual_sweeps_sum(ctypes.byref(d), N, K, SWEEPS_REDUCTIONS[reduction], ptr(lam_r),
                                          qd.data_ptr(), *map(ptr, st), norms.data_ptr(), scratch.data_ptr(),
                                          sums.data_ptr(), ctypes.c_void_p(s.cuda_stream))
    _lib.check(rc, "sdcgym_residual_sweeps_sum")
    torch.cuda.synchronize()
    return sums.cpu().numpy(), norms.cpu().numpy()


def start_norms(loss, lam, state):
    """n_0 = ||r_0||_inf on the host: the given residuals, or the reset state's r_0 = z (Q 1) (as sweep_residual)"""
    if state is not None:
        return np.max(np.abs(np.asarray(state[2])), axis=1)
    q1 = np.zeros(loss.M)
    for c in range(loss.M):
        q1 = q1 + loss.Q[:, c]
    z = lam.real * loss.dt + 1j * (lam.imag * loss.dt)
    return np.max(np.abs(z[:, None] * q1[None, :]), axis=1)


def contributions(loss, lam, row, K, reduction, state=None):
    """per-sample (f, weighted g) from the per-sample kernel, and its norms, as numpy"""
    st = (None, None, None) if state is None else state
    _, _, n, g = loss.sweeps(lam, row, K, *st, with_grad=True)
    n, g = n.cpu().numpy(), g.cpu().numpy()
    if reduction == "mean":
        return n, g, n
    n0 = start_norms(loss, lam, state)
    with np.errstate(divide="ignore", invalid="ignore"):
        f = np.where(n0 == 0, 0.0, np.log(n / n0))
        ok = (n0 != 0) & (n > 0) & np.isfinite(n)
        w = np.where(ok[:, None], g * (1.0 / np.where(ok, n, 1.0))[:, None], 0.0)
    return f, w, n


def columns(f, g):
    g = np.asarray(g).reshape(len(f), -1)
    return [f] + [c for k in range(g.shape[1]) for c in (g[:, k].real, g[:, k].imag)]


def assert_sums(sums, f, g, B, reduction):
    """the tree bound; log_ratio adds one rounding per sample (the host's log, n_0) to the value column"""
    cols = columns(f, g)
    assert_tree_sums(sums[1:], cols[1:], B)
    depth = math.ceil(math.log2(B)) + 2
    exact = math.fsum(f.tolist())
    bound = depth * EPS * math.fsum(np.abs(f).tolist())
    if reduction == "log_ratio":
        bound += 4 * EPS * math.fsum(np.maximum(np.abs(f), 1.0).tolist())
    assert abs(sums[0] - exact) <= bound, (sums[0], exact, bound)


def _state(rng, M, B):
    u0 = rng.uniform(0, 1, (B, M)) + 1j * rng.uniform(0, 1, (B, M))
    u = rng.uniform(0, 1, (B, M)) + 1j * rng.uniform(0, 1, (B, M))
    r = rng.normal(size=(B, M)) + 1j * rng.normal(size=(B, M))
    return u0, u, r


# ---- 1. sums against the per-sample kernel ------------------------------------------------------------------------
@pytest.mark.parametrize("M", range(2, 10))
def test_sums_match_per_sample_kernel(M):
    rng = np.random.default_rng(500 + M)
    for pt in LAYOUTS:
        loss = ResidualLoss(M, 1.0, pt)
        for complex_row in (False, True):
            row = _row(rng, M, pt, complex_row)
            for K in (1, 5, 50):
                for B in (1, 127, 128, 129, 4099):
                    lam = _lams(rng, B)
                    for state in (None, _state(rng, M, B)):
                        for red in ("mean", "log_ratio"):
                            sums, norms = fused(loss, B, K, red, lam=lam, row=row, state=state)
                            f, w, n = contributions(loss, lam, row, K, red, state)
                            assert np.array_equal(norms, n, equal_nan=True), (M, pt, complex_row, K, B, red)
                            if not (np.isfinite(f).all() and np.isfinite(w).all()):  # a diverging sample reaches
                                assert not np.isfinite(sums).all()                    # the sums unchanged
                                continue
                            assert_sums(sums, f, w, B, red)


@pytest.mark.parametrize("M,pt", [(5, "diag"), (5, "lower_tri"), (9, "diag"), (9, "lower_tri")])
def test_sums_match_per_sample_kernel_2_20(M, pt):
    rng = np.random.default_rng(11 * M)
    B, K = 1 << 20, 5
    loss = ResidualLoss(M, 1.0, pt)
    row, lam = _row(rng, M, pt, True), _lams(rng, B)
    for red in ("mean", "log_ratio"):
        sums, norms = fused(loss, B, K, red, lam=lam, row=row)
        f, w, n = contributions(loss, lam, row, K, red)
        assert np.array_equal(norms, n)
        assert_sums(sums, f, w, B, red)


# ---- 2. grid mode -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("pt", ["diag", "lower_tri"])
@pytest.mark.parametrize("n_re,n_im", [(33, 17), (257, 129)])
def test_grid_mode_matches_host_lambdas(n_re, n_im, pt):
    M, K = 5, 5
    rng = np.random.default_rng(n_re + len(pt))
    loss = ResidualLoss(M, 1.0, pt)
    row = _row(rng, M, pt, True)
    N = n_re * n_im
    lam_h = host_grid(n_re, n_im)
    for red in ("mean", "log_ratio"):
        sums, norms = fused(loss, N, K, red, row=row, grid=(n_re, n_im, 0))
        f, w, n = contributions(loss, lam_h, row, K, red)
        assert norms[-1] == 0.0  # the corner lambda = 0 of the box
        for j, c in enumerate(columns(f, w)):
            assert abs(sums[j] - math.fsum(c.tolist())) <= 1e-12 * math.fsum(np.abs(c).tolist()), (red, j)
        # the corner node alone adds exact zeros
        corner, cn = fused(loss, 1, K, red, row=row, grid=(n_re, n_im, N - 1))
        assert np.array_equal(corner, np.zeros_like(corner)) and cn[0] == 0.0
        # a range of rows in the middle of the grid (grid_first > 0)
        _, norms2 = fused(loss, 5 * n_im, K, red, row=row, grid=(n_re, n_im, 3 * n_im))
        assert np.array_equal(norms2, norms[3 * n_im: 8 * n_im])


# ---- 3. determinism -----------------------------------------------------------------------------------------------
def test_same_bits_on_every_call_and_stream():
    M, pt = 6, "lower_tri"
    rng = np.random.default_rng(3)
    loss = ResidualLoss(M, 1.0, pt)
    row, lam = _row(rng, M, pt, True), _lams(rng, 300_001)
    side = torch.cuda.Stream()
    for red in ("mean", "log_ratio"):
        a, _ = fused(loss, lam.size, 7, red, lam=lam, row=row)
        b, _ = fused(loss, lam.size, 7, red, lam=lam, row=row)
        c, _ = fused(loss, lam.size, 7, red, lam=lam, row=row, stream=side)
        assert a.tobytes() == b.tobytes() == c.tobytes()
        g1 = fused(loss, 513 * 257, 7, red, row=row, grid=(513, 257, 0))[0]
        g2 = fused(loss, 513 * 257, 7, red, row=row, grid=(513, 257, 0), stream=side)[0]
        assert g1.tobytes() == g2.tobytes()
        v1, d1 = loss.sweeps_shared_value_and_grad(lam, row, 7, reduction=red)
        v2, d2 = loss.sweeps_shared_value_and_grad(lam, row, 7, reduction=red)
        assert float(v1) == float(v2) and torch.equal(d1, d2)


# ---- 4. shards ----------------------------------------------------------------------------------------------------
def test_row_shards_reproduce_the_full_grid():
    M, pt, n_re, n_im, K = 5, "lower_tri", 33, 17, 5
    rng = np.random.default_rng(4)
    loss = ResidualLoss(M, 1.0, pt)
    row = _row(rng, M, pt, True)
    N = n_re * n_im
    for red in ("mean", "log_ratio"):
        full_v, full_g = loss.sweeps_grid_value_and_grad(n_re, n_im, RE_BOX, IM_BOX, row, K, red)
        all_v, all_g = loss.sweeps_grid_value_and_grad(n_re, n_im, RE_BOX, IM_BOX, row, K, red, rows=(0, n_re))
        assert float(full_v) == float(all_v) and torch.equal(full_g, all_g)
        assert full_g.shape == (loss._sr.n_out,) and full_g.is_complex()
        v, g = 0.0, np.zeros(loss._sr.n_out, np.complex128)
        for lo, hi in ((0, 11), (11, 12), (12, 12), (12, 33)):
            sv, sg = loss.sweeps_grid_value_and_grad(n_re, n_im, RE_BOX, IM_BOX, row, K, red, rows=(lo, hi))
            assert sg.shape == (loss._sr.n_out,)
            if hi == lo:
                assert math.isnan(float(sv)) and not sg.abs().sum()
                continue
            v += float(sv) * (hi - lo) / n_re
            g += sg.cpu().numpy() * (hi - lo) / n_re
        f, w, _ = contributions(loss, host_grid(n_re, n_im), row, K, red)
        tol = (math.ceil(math.log2(N)) + 6) * EPS / N
        assert abs(v - float(full_v)) <= tol * float(np.abs(f).sum()) + 8 * EPS * max(1.0, abs(v))
        assert np.all(np.abs(g.real - full_g.real.cpu().numpy()) <= tol * np.abs(w.real).sum(0) + 1e-300)
        assert np.all(np.abs(g.imag - full_g.imag.cpu().numpy()) <= tol * np.abs(w.imag).sum(0) + 1e-300)
    with pytest.raises(ValueError):
        loss.sweeps_grid_value_and_grad(n_re, n_im, RE_BOX, IM_BOX, row, K, rows=(12, 34))
    with pytest.raises(ValueError):
        loss.sweeps_grid_value_and_grad(n_re, n_im, RE_BOX, IM_BOX, row, K, rows=(5, 4))


def _dist_worker(rank, ws, port, backend, tmp):
    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank if backend == "nccl" else 0)
    dist.init_process_group(backend, rank=rank, world_size=ws)
    try:
        loss = ResidualLoss(5, 1.0, "lower_tri")
        row = _row(np.random.default_rng(4), 5, "lower_tri", True)
        v, g = loss.sweeps_grid_value_and_grad(3, 65, RE_BOX, IM_BOX, row, 5, "log_ratio")  # 2 + 1 rows
        np.save(os.path.join(tmp, f"r{rank}.npy"), np.concatenate([[float(v)], g.cpu().numpy().view(np.float64)]))
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(600)
@pytest.mark.parametrize("backend", ["gloo", "nccl"])
def test_two_rank_grid_value_and_grad(tmp_path, backend):
    """rows=None over two ranks (gloo: both on one device; nccl: one device each) against the single-process call"""
    import torch.multiprocessing as mp

    if backend == "nccl" and torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_dist_worker, args=(2, port, backend, str(tmp_path)), nprocs=2, join=True)
    r0, r1 = np.load(tmp_path / "r0.npy"), np.load(tmp_path / "r1.npy")
    assert np.array_equal(r0, r1)
    loss = ResidualLoss(5, 1.0, "lower_tri")
    row = _row(np.random.default_rng(4), 5, "lower_tri", True)
    v, g = loss.sweeps_grid_value_and_grad(3, 65, RE_BOX, IM_BOX, row, 5, "log_ratio")
    ref = np.concatenate([[float(v)], g.cpu().numpy().view(np.float64)])
    assert np.allclose(r0, ref, rtol=1e-13, atol=1e-16)


# ---- 5. gradients -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("red", ["mean", "log_ratio"])
@pytest.mark.parametrize("pt", ["diag", "lower_tri"])
def test_grid_gradient_against_central_difference(pt, red):
    M, n_re, n_im, K = 5, 65, 33, 5
    rng = np.random.default_rng(5)
    loss = ResidualLoss(M, 1.0, pt)
    row = _row(rng, M, pt, True)
    _, g = loss.sweeps_grid_value_and_grad(n_re, n_im, RE_BOX, IM_BOX, row, K, red)  # JAX convention
    direction = rng.normal(size=row.shape) + 1j * rng.normal(size=row.shape)
    h = 1e-7
    fp = float(loss.sweeps_grid_value_and_grad(n_re, n_im, RE_BOX, IM_BOX, row + h * direction, K, red)[0])
    fm = float(loss.sweeps_grid_value_and_grad(n_re, n_im, RE_BOX, IM_BOX, row - h * direction, K, red)[0])
    an = float(np.real(np.sum(g.cpu().numpy() * direction)))
    assert abs((fp - fm) / (2 * h) - an) <= 2e-6 * abs(an), ((fp - fm) / (2 * h), an)


@pytest.mark.parametrize("given", [False, True])
@pytest.mark.parametrize("complex_row", [False, True])
@pytest.mark.parametrize("pt", ["diag", "lower_tri"])
def test_autograd_matches_per_sample_autograd(pt, complex_row, given):
    M, B, K = 5, 4096, 7
    rng = np.random.default_rng(6)
    loss = ResidualLoss(M, 1.0, pt)
    row, lam = _row(rng, M, pt, complex_row), torch.as_tensor(_lams(rng, B), device="cuda")
    st = tuple(torch.as_tensor(x, device="cuda") for x in _state(rng, M, B)) if given else (None, None, None)
    n0 = (st[2].abs().amax(1) if given else
          torch.as_tensor(start_norms(loss, lam.cpu().numpy(), None), device="cuda"))
    for red in ("mean", "log_ratio"):
        theta = torch.as_tensor(row, device="cuda").requires_grad_(True)
        v = loss.sweeps_shared_differentiable(lam, theta, K, *st, reduction=red)
        (2.0 * v).backward()
        ref = torch.as_tensor(row, device="cuda").requires_grad_(True)
        n = loss.sweeps_differentiable(lam, ref, K, *st)
        vr = n.mean() if red == "mean" else torch.log(n / n0).mean()
        (2.0 * vr).backward()
        assert theta.grad.shape == ref.grad.shape and theta.grad.dtype == ref.grad.dtype
        assert abs(float(v.detach()) - float(vr.detach())) <= 1e-12 * abs(float(vr.detach()))
        assert torch.allclose(theta.grad, ref.grad, rtol=1e-12, atol=1e-12 * float(ref.grad.abs().max()))
    theta = torch.as_tensor(row, device="cuda").requires_grad_(True)
    gv = loss.sweeps_grid_differentiable(65, 33, RE_BOX, IM_BOX, theta, K, "log_ratio")
    gv.backward()
    v_ref, g_ref = loss.sweeps_grid_value_and_grad(65, 33, RE_BOX, IM_BOX, row, K, "log_ratio", convention="torch")
    assert float(gv.detach()) == float(v_ref) and torch.equal(theta.grad, g_ref)


# ---- 6. memory ----------------------------------------------------------------------------------------------------
def test_grid_gradient_memory_stays_small():
    M, pt, n, K = 9, "lower_tri", 2048, 50
    loss = ResidualLoss(M, 1.0, pt)
    row = _row(np.random.default_rng(9), M, pt, True)
    for red in ("mean", "log_ratio"):
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        v, g = loss.sweeps_grid_value_and_grad(n, n, RE_BOX, IM_BOX, row, K, red)
        torch.cuda.synchronize()
        assert torch.cuda.max_memory_allocated() - base < 64 << 20
        assert g.shape == (loss._sr.n_out,) and torch.isfinite(g).all()
        # after 50 sweeps some nodes' r_K is exactly 0, and log(0 / n_0) = -inf reaches the log_ratio mean
        assert math.isfinite(float(v)) if red == "mean" else float(v) == -math.inf


# ---- 7. empty and invalid input -----------------------------------------------------------------------------------
def test_empty_batch_and_invalid_input():
    loss = ResidualLoss(5, 1.0, "diag")
    row = np.full(5, 0.3)
    for red in ("mean", "log_ratio"):
        v, g = loss.sweeps_shared_value_and_grad(np.zeros(0, np.complex128), row, 5, reduction=red)
        assert math.isnan(float(v)) and g.shape == (5,) and not g.abs().sum()
        v, g = loss.sweeps_grid_value_and_grad(8, 8, RE_BOX, IM_BOX, row, 5, red, rows=(3, 3))
        assert math.isnan(float(v)) and g.shape == (5,) and not g.abs().sum()
    sums, _ = fused(loss, 0, 5, "mean", lam=np.zeros(0, np.complex128), row=row)
    assert np.array_equal(sums, np.zeros(11))  # N = 0 writes zeros
    lam = _lams(np.random.default_rng(0), 4)
    with pytest.raises(ValueError):
        loss.sweeps_shared_value_and_grad(lam, row, 5, reduction="sum")
    with pytest.raises(ValueError):
        loss.sweeps_grid_value_and_grad(8, 8, RE_BOX, IM_BOX, row, 5, reduction="max")
    with pytest.raises(ValueError):
        loss.sweeps_grid_value_and_grad(8, 8, RE_BOX, IM_BOX, row, 5, rows=(0, 9))
    with pytest.raises(ValueError):
        loss.sweeps_shared_value_and_grad(lam, np.full((4, 5), 0.3), 5)
    with pytest.raises(ValueError):
        loss.sweeps_shared_value_and_grad(lam, row, 5, u0s=np.ones((4, 5)))
    with pytest.raises(ValueError):
        ResidualLoss(5, 1.0, prec="LU").sweeps_shared_value_and_grad(lam, None, 5)
    with pytest.raises(_lib.SdcGymError):
        loss.sweeps_shared_value_and_grad(lam, row, 51)


# ---- 8. example ---------------------------------------------------------------------------------------------------
def test_example_with_sweeps_and_grid_lowers_its_loss():
    import importlib.util

    path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "examples",
                        "train_diag_spectral_radius.py")
    spec = importlib.util.spec_from_file_location("train_diag_example", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    history, theta = mod.main(["--M", "5", "--sweeps", "5", "--grid", "64", "--steps", "60"])
    assert history[-1] < history[0] and np.isfinite(theta).all()

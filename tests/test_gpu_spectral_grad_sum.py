"""GPU: the reduced spectral-radius gradient of ONE shared parameter row (``rho_grad_sum_kernel`` through
``sdcgym_spectral_radius_grad_sum``, ``SpectralRadiusLoss.shared_value_and_grad`` / ``grid_value_and_grad``) against
the per-sample kernel (``radii_and_grads`` on the expanded row) summed exactly with ``math.fsum``."""
import ctypes
import math
import os
import socket

import numpy as np
import pytest
import torch

from sdc_gym_b200 import _lib
from sdc_gym_b200.loss import SpectralRadiusLoss
from sdc_gym_b200.precond import num_actions

pytestmark = pytest.mark.gpu

LAYOUTS = ("diag", "lower_diag", "lower_tri", "strictly_lower_tri")
RE_BOX, IM_BOX = (-100.0, 0.0), (-10.0, 0.0)
EPS = np.finfo(np.float64).eps


def _row(rng, M, pt, complex_row):
    A = num_actions(M, pt)
    hi = 0.08 if pt == "strictly_lower_tri" else 0.3
    r = rng.uniform(0.02, hi, A)
    return r + 1j * rng.uniform(-0.05, 0.05, A) if complex_row else r


def _lams(rng, B):
    return rng.uniform(*RE_BOX, B) + 1j * rng.uniform(*IM_BOX, B)


def fused(loss, N, lam=None, row=None, grid=None, stream=None):
    """sdcgym_spectral_radius_grad_sum straight through the C ABI with the per-sample rho requested:
    (sums (1 + 2A,), rho (N,)) as numpy.  ``grid=(n_re, n_im, first)`` selects grid mode over the default box."""
    d = _lib.RhoDesc.from_buffer_copy(loss._desc)
    qd, is_c, _ = loss._outputs_tensor(row, 1)
    d.qd_is_complex, d.qd_broadcast = is_c, 1
    lam_r = None
    if grid is None:
        lam_r = torch.view_as_real(torch.as_tensor(np.asarray(lam, np.complex128), device=loss.device).contiguous())
        d.grid_re = d.grid_im = d.grid_first = 0
    else:
        d.grid_re, d.grid_im, d.grid_first = grid
        d.re_lo, d.re_hi, d.im_lo, d.im_hi = *RE_BOX, *IM_BOX
    L = loss._L
    n_scratch = L.sdcgym_spectral_radius_grad_sum_scratch_doubles(loss.M, d.prec_type, N)
    scratch = torch.full((max(n_scratch, 1),), np.nan, dtype=torch.float64, device=loss.device)  # never NULL
    sums = torch.full((1 + 2 * loss.n_out,), np.nan, dtype=torch.float64, device=loss.device)
    rho = torch.full((N,), np.nan, dtype=torch.float64, device=loss.device)
    s = torch.cuda.current_stream() if stream is None else stream
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        rc = L.sdcgym_spectral_radius_grad_sum(ctypes.byref(d), N, None if lam_r is None else lam_r.data_ptr(),
                                               qd.data_ptr(), rho.data_ptr(), scratch.data_ptr(), sums.data_ptr(),
                                               ctypes.c_void_p(s.cuda_stream))
    _lib.check(rc, "sdcgym_spectral_radius_grad_sum")
    torch.cuda.synchronize()
    return sums.cpu().numpy(), rho.cpu().numpy()


def columns(rho, g):
    """rho and the interleaved Re / Im columns of g, in the order of the sums"""
    g = np.asarray(g).reshape(len(rho), -1)
    return [rho] + [c for k in range(g.shape[1]) for c in (g[:, k].real, g[:, k].imag)]


def assert_tree_sums(sums, cols, B, extra_levels=0):
    """each sum within (ceil(log2 B) + 2) eps sum|x_i| of the exact sum of its column"""
    depth = math.ceil(math.log2(B)) + 2 + extra_levels
    for j, c in enumerate(cols):
        exact = math.fsum(c.tolist())
        bound = depth * EPS * math.fsum(np.abs(c).tolist())
        assert abs(sums[j] - exact) <= bound, (j, B, sums[j], exact, bound)


def host_grid(n_re, n_im, lo=0, hi=None):
    """the grid's lambdas for rows lo..hi-1, formed on the host like rho_inputs (up to FMA contraction)"""
    hi = n_re if hi is None else hi
    a = np.arange(lo, hi, dtype=np.float64)[:, None]
    b = np.arange(n_im, dtype=np.float64)[None, :]
    re = RE_BOX[0] + (RE_BOX[1] - RE_BOX[0]) * (a / (n_re - 1))
    im = IM_BOX[0] + (IM_BOX[1] - IM_BOX[0]) * (b / (n_im - 1))
    return (re + 1j * im).reshape(-1)


# ---- 1. sums against the per-sample kernel ------------------------------------------------------------------------
SMALL_B = (1, 127, 128, 129, 4099)


@pytest.mark.parametrize("M", range(2, 10))
def test_sums_match_per_sample_kernel(M):
    rng = np.random.default_rng(100 + M)
    for dt in (1.0, 0.37):
        for pt in LAYOUTS:
            loss = SpectralRadiusLoss(M, dt, pt)
            for complex_row in (False, True):
                row = _row(rng, M, pt, complex_row)
                for B in SMALL_B:
                    lam = _lams(rng, B)
                    sums, rho = fused(loss, B, lam=lam, row=row)
                    rho_ref, g_ref = loss.radii_and_grads(lam, row)
                    rho_ref, g_ref = rho_ref.cpu().numpy(), g_ref.cpu().numpy()
                    assert np.array_equal(rho, rho_ref), (M, dt, pt, complex_row, B)
                    assert not np.isnan(rho_ref).any()
                    assert_tree_sums(sums, columns(rho_ref, g_ref), B)


# B = 2^20 for a subset: the exact reference sums of 2^20 x (1 + 2A) values dominate the run time
@pytest.mark.parametrize("M,pt,complex_row,dt", [(5, "diag", True, 1.0), (5, "lower_tri", True, 1.0),
                                                 (9, "diag", True, 1.0), (9, "lower_tri", True, 1.0),
                                                 (9, "strictly_lower_tri", False, 0.37),
                                                 (2, "lower_diag", True, 0.37)])
def test_sums_match_per_sample_kernel_2_20(M, pt, complex_row, dt):
    rng = np.random.default_rng(7 * M)
    B = 1 << 20
    loss = SpectralRadiusLoss(M, dt, pt)
    row, lam = _row(rng, M, pt, complex_row), _lams(rng, B)
    sums, rho = fused(loss, B, lam=lam, row=row)
    rho_ref, g_ref = loss.radii_and_grads(lam, row)
    rho_ref, g_ref = rho_ref.cpu().numpy(), g_ref.cpu().numpy()
    assert np.array_equal(rho, rho_ref) and not np.isnan(rho_ref).any()
    assert_tree_sums(sums, columns(rho_ref, g_ref), B)


# ---- 2. grid mode -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("pt", ["diag", "lower_tri"])
@pytest.mark.parametrize("n_re,n_im", [(33, 17), (257, 129)])
def test_grid_mode_matches_grid_and_host_lambdas(n_re, n_im, pt):
    M = 5
    rng = np.random.default_rng(n_re + len(pt))
    loss = SpectralRadiusLoss(M, 1.0, pt)
    row = _row(rng, M, pt, True)
    N = n_re * n_im
    sums, rho = fused(loss, N, row=row, grid=(n_re, n_im, 0))
    grid_rho = loss.grid(n_re, n_im, RE_BOX, IM_BOX, row).reshape(-1).cpu().numpy()
    assert np.array_equal(rho, grid_rho)
    assert rho[-1] == 0.0  # the corner lambda = 0 of the box
    assert_tree_sums(sums[:1], [grid_rho], N)
    rho_h, g_h = loss.radii_and_grads(host_grid(n_re, n_im), row)
    cols = columns(rho_h.cpu().numpy(), g_h.cpu().numpy())
    for j, c in enumerate(cols[1:], start=1):
        assert abs(sums[j] - math.fsum(c.tolist())) <= 1e-12 * math.fsum(np.abs(c).tolist()), j
    # a range of rows in the middle of the grid (grid_first > 0)
    sums2, rho2 = fused(loss, 5 * n_im, row=row, grid=(n_re, n_im, 3 * n_im))
    assert np.array_equal(rho2, grid_rho[3 * n_im: 8 * n_im])


# ---- 3. determinism -----------------------------------------------------------------------------------------------
def test_same_bits_on_every_call_and_stream():
    M, pt = 6, "lower_tri"
    rng = np.random.default_rng(3)
    loss = SpectralRadiusLoss(M, 1.0, pt)
    row, lam = _row(rng, M, pt, True), _lams(rng, 300_001)
    a, _ = fused(loss, lam.size, lam=lam, row=row)
    b, _ = fused(loss, lam.size, lam=lam, row=row)
    side = torch.cuda.Stream()
    c, _ = fused(loss, lam.size, lam=lam, row=row, stream=side)
    assert a.tobytes() == b.tobytes() == c.tobytes()
    g1 = fused(loss, 513 * 257, row=row, grid=(513, 257, 0))[0]
    g2 = fused(loss, 513 * 257, row=row, grid=(513, 257, 0), stream=side)[0]
    assert g1.tobytes() == g2.tobytes()
    v1, d1 = loss.shared_value_and_grad(lam, row)
    v2, d2 = loss.shared_value_and_grad(lam, row)
    assert float(v1) == float(v2) and torch.equal(d1, d2)


# ---- 4. shards ----------------------------------------------------------------------------------------------------
def test_row_shards_reproduce_the_full_grid():
    M, pt, n_re, n_im = 5, "lower_tri", 33, 17
    rng = np.random.default_rng(4)
    loss = SpectralRadiusLoss(M, 1.0, pt)
    row = _row(rng, M, pt, True)
    full_v, full_g = loss.grid_value_and_grad(n_re, n_im, RE_BOX, IM_BOX, row)
    all_v, all_g = loss.grid_value_and_grad(n_re, n_im, RE_BOX, IM_BOX, row, rows=(0, n_re))
    assert float(full_v) == float(all_v) and torch.equal(full_g, all_g)
    assert full_g.shape == (loss.n_out,) and full_g.is_complex()
    v, g = 0.0, np.zeros(loss.n_out, np.complex128)
    for lo, hi in ((0, 11), (11, 12), (12, 12), (12, 33)):
        sv, sg = loss.grid_value_and_grad(n_re, n_im, RE_BOX, IM_BOX, row, rows=(lo, hi))
        assert sg.shape == (loss.n_out,)
        if hi == lo:
            assert math.isnan(float(sv)) and not sg.abs().sum()
            continue
        v += float(sv) * (hi - lo) / n_re
        g += sg.cpu().numpy() * (hi - lo) / n_re
    # tolerance: the tree bound on the mean, from the per-sample values over the host grid
    rho_h, g_h = loss.radii_and_grads(host_grid(n_re, n_im), row)
    N = n_re * n_im
    tol = (math.ceil(math.log2(N)) + 6) * EPS / N
    assert abs(v - float(full_v)) <= tol * float(rho_h.abs().sum())
    gh = g_h.cpu().numpy()
    assert np.all(np.abs(g.real - full_g.real.cpu().numpy()) <= tol * np.abs(gh.real).sum(0) + 1e-300)
    assert np.all(np.abs(g.imag - full_g.imag.cpu().numpy()) <= tol * np.abs(gh.imag).sum(0) + 1e-300)
    with pytest.raises(ValueError):
        loss.grid_value_and_grad(n_re, n_im, RE_BOX, IM_BOX, row, rows=(12, 34))


def _dist_worker(rank, ws, port, backend, tmp):
    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank if backend == "nccl" else 0)
    dist.init_process_group(backend, rank=rank, world_size=ws)
    try:
        loss = SpectralRadiusLoss(5, 1.0, "lower_tri")
        row = _row(np.random.default_rng(4), 5, "lower_tri", True)
        v, g = loss.grid_value_and_grad(3, 65, RE_BOX, IM_BOX, row)  # 2 + 1 rows on two ranks
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
    loss = SpectralRadiusLoss(5, 1.0, "lower_tri")
    row = _row(np.random.default_rng(4), 5, "lower_tri", True)
    v, g = loss.grid_value_and_grad(3, 65, RE_BOX, IM_BOX, row)
    ref = np.concatenate([[float(v)], g.cpu().numpy().view(np.float64)])
    assert np.allclose(r0, ref, rtol=1e-13, atol=1e-16)


# ---- 5. derivative ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("pt", ["diag", "lower_tri"])
def test_grid_gradient_against_central_difference(pt):
    M, n_re, n_im = 5, 65, 33
    rng = np.random.default_rng(5)
    loss = SpectralRadiusLoss(M, 1.0, pt)
    row = _row(rng, M, pt, True)
    _, g = loss.grid_value_and_grad(n_re, n_im, RE_BOX, IM_BOX, row)  # JAX convention
    direction = rng.normal(size=row.shape)
    h = 1e-7
    fp = float(loss.grid_mean(n_re, n_im, RE_BOX, IM_BOX, row + h * direction))
    fm = float(loss.grid_mean(n_re, n_im, RE_BOX, IM_BOX, row - h * direction))
    an = float(np.real(np.sum(g.cpu().numpy() * direction)))
    assert abs((fp - fm) / (2 * h) - an) <= 2e-6 * abs(an), ((fp - fm) / (2 * h), an)


# ---- 6. autograd --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("complex_row", [False, True])
@pytest.mark.parametrize("pt", ["diag", "lower_tri"])
def test_autograd_on_one_row(pt, complex_row):
    M, B = 5, 4096
    rng = np.random.default_rng(6)
    loss = SpectralRadiusLoss(M, 1.0, pt)
    row, lam = _row(rng, M, pt, complex_row), _lams(rng, B)
    v_ref, g_ref = loss.shared_value_and_grad(lam, row, convention="torch")
    for shape in ((loss.n_out,), (1, loss.n_out)):
        theta = torch.as_tensor(row.reshape(shape), device="cuda").requires_grad_(True)
        v = loss.differentiable(torch.as_tensor(lam, device="cuda"), theta)
        (2.0 * v).backward()
        assert theta.grad.shape == shape and theta.grad.dtype == theta.dtype
        assert abs(float(v.detach()) - float(v_ref)) <= 1e-12 * abs(float(v_ref))
        assert torch.allclose(theta.grad.reshape(-1), 2.0 * g_ref, rtol=1e-12, atol=0)
    # the same value and gradient as the per-sample path on the expanded row
    v_exp, g_exp = loss.value_and_grad(lam, np.tile(row, (B, 1)), convention="torch")
    assert abs(float(v_exp) - float(v_ref)) <= 1e-13 * float(v_ref)
    assert torch.allclose(g_exp.sum(0), g_ref, rtol=1e-12, atol=1e-15)
    assert g_ref.is_complex() == complex_row
    gv_ref, gg_ref = loss.grid_value_and_grad(65, 33, RE_BOX, IM_BOX, row, convention="torch")
    theta = torch.as_tensor(row, device="cuda").requires_grad_(True)
    gv = loss.grid_differentiable(65, 33, RE_BOX, IM_BOX, theta)
    gv.backward()
    assert theta.grad.shape == (loss.n_out,)
    assert abs(float(gv.detach()) - float(gv_ref)) <= 1e-12 * abs(float(gv_ref))
    assert torch.allclose(theta.grad, gg_ref, rtol=1e-12, atol=0)


def test_empty_batch_and_bad_rows():
    loss = SpectralRadiusLoss(5, 1.0, "diag")
    v, g = loss.shared_value_and_grad(np.zeros(0, np.complex128), np.full(5, 0.3))
    assert math.isnan(float(v)) and g.shape == (5,) and not g.abs().sum()
    with pytest.raises(ValueError):
        loss.shared_value_and_grad(_lams(np.random.default_rng(0), 4), np.full((4, 5), 0.3))
    sums, _ = fused(loss, 0, lam=np.zeros(0, np.complex128), row=np.full(5, 0.3))
    assert np.array_equal(sums, np.zeros(11))  # N = 0 writes zeros


# ---- 7. memory ----------------------------------------------------------------------------------------------------
def test_grid_gradient_memory_stays_small():
    M, pt, n = 9, "lower_tri", 2048
    loss = SpectralRadiusLoss(M, 1.0, pt)
    row = _row(np.random.default_rng(9), M, pt, True)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    v, g = loss.grid_value_and_grad(n, n, RE_BOX, IM_BOX, row)
    torch.cuda.synchronize()
    assert torch.cuda.max_memory_allocated() - base < 64 << 20
    assert math.isfinite(float(v)) and g.shape == (loss.n_out,)

"""GPU: populations of shared Q_delta rows (``sdcgym_full_solve_counts_population``,
``sdcgym_spectral_radius_grad_sum_population``; ``IterationCounts.population_*``, ``SpectralRadiusLoss.population_*``)
against the single-row calls on each row, bit for bit."""
import os
import socket

import numpy as np
import pytest
import torch

from sdc_gym_b200 import PopulationSummary
from sdc_gym_b200.iterations import IterationCounts
from sdc_gym_b200.loss import SpectralRadiusLoss
from sdc_gym_b200.precond import num_actions

pytestmark = pytest.mark.gpu

RE_BOX, IM_BOX = (-100.0, 0.0), (-10.0, 0.0)
LAYOUTS = ("diag", "lower_diag", "lower_tri", "strictly_lower_tri")
STATS = ("count", "n_err", "n_exhausted", "n_success", "success_rate", "mean_niter")

# the layouts of test_gpu_full_solve_counts.CONFIGS that take rows
ROW_CONFIGS = [
    dict(prec_type="diag", cplx=False, do_scale=True, free_action_space=False),
    dict(prec_type="diag", cplx=False, do_scale=False, free_action_space=False),
    dict(prec_type="diag", cplx=True),
    dict(prec_type="diag", cplx=False),
    dict(prec_type="lower_diag", cplx=False, do_scale=False, free_action_space=False),
    dict(prec_type="lower_tri", cplx=True),
    dict(prec_type="strictly_lower_tri", cplx=False, do_scale=False, free_action_space=False),
    dict(prec_type="lower_tri", cplx=False, do_scale=True, free_action_space=False, use_doubles=False),
    dict(prec_type="diag", cplx=True, use_doubles=False),
]


def _lams(rng, n):
    """random lambdas of the box plus the special nodes of test_gpu_full_solve_counts: 0, far outside the box (err),
    -4 and -5 (exhausted)"""
    lam = rng.uniform(*RE_BOX, n) + 1j * rng.uniform(*IM_BOX, n)
    special = [0.0, -1e4, -3e3 + 50j, -4.0, -5.0, -700.0 - 300j, -0.3 - 0.1j, -1.0]
    lam[: min(n, len(special))] = special[: min(n, len(special))]
    return lam


def _population(rng, P, M, prec_type, cplx, do_scale, use_doubles=True):
    """P rows: MIN's diagonal (diag layouts), zeros, then random rows"""
    A = num_actions(M, prec_type)
    if cplx:
        rows = rng.uniform(0, 0.4, (P, A)) + 1j * rng.uniform(-0.05, 0.05, (P, A))
    else:
        rows = rng.uniform(-1, 1, (P, A)) if do_scale else rng.uniform(0, 0.5, (P, A))
    if P > 1:
        rows[1] = 0.0
    if prec_type == "diag":
        from sdc_gym_b200.collocation import collocation_matrix
        from sdc_gym_b200.precond import fixed_preconditioner

        mn = np.diag(fixed_preconditioner("min", M, collocation_matrix(M)))
        rows[0] = (2 * mn - 1) if do_scale else mn
    if not use_doubles:
        rows = rows.astype(np.complex64 if cplx else np.float32)
    return rows


def _split(cfg):
    cfg = dict(cfg)
    return cfg.pop("cplx"), cfg


def _assert_summary_rows(pop, singles, what):
    assert isinstance(pop, PopulationSummary) and len(pop) == len(singles)
    for p, one in enumerate(singles):
        assert np.array_equal(pop.hist[p], one.hist), (what, p)
        for k in STATS:
            assert getattr(pop[p], k) == getattr(one, k), (what, p, k)
            assert float(getattr(pop, k)[p]) == float(getattr(one, k)), (what, p, k)


# ---- 1. counts ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M", range(2, 10))
def test_counts_list_mode(M):
    rng = np.random.default_rng(10 * M)
    lam = _lams(rng, 300)
    for cfg in ROW_CONFIGS:
        cplx, kw = _split(cfg)
        ev = IterationCounts(M, 1.0, 1e-10, blas_variant=M % 2, **kw)
        for P in (1, 3, 7):
            rows = _population(rng, P, M, kw["prec_type"], cplx, kw.get("do_scale", False), kw.get("use_doubles", True))
            pop = ev.population_summary(lam, torch.as_tensor(rows))
            _assert_summary_rows(pop, [ev.summary(lam, torch.as_tensor(r)) for r in rows], f"M={M} {cfg} P={P}")


@pytest.mark.parametrize("M", range(2, 10))
def test_counts_grid_mode_and_shards(M):
    rng = np.random.default_rng(20 + M)
    n_re, n_im = 37, 53
    for cfg in ROW_CONFIGS:
        cplx, kw = _split(cfg)
        ev = IterationCounts(M, 1.0, 1e-10, blas_variant=0, **kw)
        rows = _population(rng, 7 if cfg is ROW_CONFIGS[0] else 3, M, kw["prec_type"], cplx,
                           kw.get("do_scale", False), kw.get("use_doubles", True))
        pop = ev.population_grid_summary(n_re, n_im, RE_BOX, IM_BOX, rows)
        _assert_summary_rows(pop, [ev.grid_summary(n_re, n_im, RE_BOX, IM_BOX, r) for r in rows], f"M={M} {cfg}")
        for lo, hi in ((0, 9), (9, 9), (9, 37)):
            part = ev.population_grid_summary(n_re, n_im, RE_BOX, IM_BOX, rows, rows=(lo, hi))
            _assert_summary_rows(part, [ev.grid_summary(n_re, n_im, RE_BOX, IM_BOX, r, rows=(lo, hi)) for r in rows],
                                 f"M={M} {cfg} rows {lo}..{hi}")


def test_counts_reach_every_outcome():
    """the lambdas above give converged, err and exhausted nodes for the zero row"""
    ev = IterationCounts(5, 1.0, 1e-10, "diag", blas_variant=0)
    s = ev.population_summary(_lams(np.random.default_rng(1), 300), np.zeros((2, 5)))
    assert (s.n_err > 0).all() and (s.n_exhausted > 0).all() and (s.n_success > 0).all()


# ---- 2. rho sums ----------------------------------------------------------------------------------------------------
def _rho_rows(rng, P, M, pt, cplx):
    A = num_actions(M, pt)
    hi = 0.08 if pt == "strictly_lower_tri" else 0.3
    r = rng.uniform(0.02, hi, (P, A))
    return r + 1j * rng.uniform(-0.05, 0.05, (P, A)) if cplx else r


def _assert_rho_rows(loss, means, grads, singles, what):
    for p, (m, g) in enumerate(singles):
        assert torch.equal(means[p], m), (what, p)
        assert torch.equal(grads[p], g), (what, p)


@pytest.mark.parametrize("M", range(2, 10))
@pytest.mark.parametrize("pt", LAYOUTS)
def test_rho_sums_list_mode(M, pt):
    rng = np.random.default_rng(M * 7 + len(pt))
    loss = SpectralRadiusLoss(M, 1.0, pt)
    for N in (77, 1000):
        lam = rng.uniform(*RE_BOX, N) + 1j * rng.uniform(*IM_BOX, N)
        for cplx in (False, True):
            for P in (1, 3, 7):
                rows = _rho_rows(rng, P, M, pt, cplx)
                means, grads = loss.population_value_and_grad(lam, rows)
                assert means.shape == (P,) and grads.shape == (P, loss.n_out)
                _assert_rho_rows(loss, means, grads, [loss.shared_value_and_grad(lam, r) for r in rows],
                                 f"M={M} {pt} N={N} cplx={cplx} P={P}")


@pytest.mark.parametrize("M", range(2, 10))
def test_rho_sums_grid_mode(M):
    """grid sizes below 128, not a multiple of 128, and above 128 * 256 nodes (two fold levels)"""
    rng = np.random.default_rng(300 + M)
    for pt in LAYOUTS:
        loss = SpectralRadiusLoss(M, 1.0, pt)
        for (n_re, n_im) in ((7, 11), (37, 53)) + (((190, 190),) if pt in ("diag", "lower_tri") else ()):
            for cplx in (False, True):
                P = 3 if n_re < 100 else 2
                rows = _rho_rows(rng, P, M, pt, cplx)
                means, grads = loss.population_grid_value_and_grad(n_re, n_im, RE_BOX, IM_BOX, rows)
                _assert_rho_rows(loss, means, grads,
                                 [loss.grid_value_and_grad(n_re, n_im, RE_BOX, IM_BOX, r) for r in rows],
                                 f"M={M} {pt} {n_re}x{n_im} cplx={cplx}")
        # shards
        rows = _rho_rows(rng, 3, M, pt, False)
        for lo, hi in ((0, 5), (5, 5), (5, 37)):
            means, grads = loss.population_grid_value_and_grad(37, 53, RE_BOX, IM_BOX, rows, rows=(lo, hi))
            singles = [loss.grid_value_and_grad(37, 53, RE_BOX, IM_BOX, r, rows=(lo, hi)) for r in rows]
            if lo == hi:
                assert torch.isnan(means).all() and not grads.any()
            else:
                _assert_rho_rows(loss, means, grads, singles, f"M={M} {pt} rows {lo}..{hi}")


def test_rho_sums_empty_batch():
    loss = SpectralRadiusLoss(5, 1.0, "diag")
    means, grads = loss.population_value_and_grad(np.zeros(0, np.complex128), np.full((3, 5), 0.2))
    assert means.shape == (3,) and torch.isnan(means).all() and grads.shape == (3, 5) and not grads.any()


# ---- 3. chunks of rows ----------------------------------------------------------------------------------------------
def test_chunking_beyond_the_grid_limit():
    """M = 9 lower_tri has nv = 91 sums per row: 800 rows take two fold launches (65535 / 91 = 720 rows each)"""
    rng = np.random.default_rng(9)
    loss = SpectralRadiusLoss(9, 1.0, "lower_tri")
    rows = _rho_rows(rng, 800, 9, "lower_tri", False)
    means, grads = loss.population_grid_value_and_grad(16, 24, RE_BOX, IM_BOX, rows)
    for p in (0, 1, 719, 720, 721, 799):
        m, g = loss.grid_value_and_grad(16, 24, RE_BOX, IM_BOX, rows[p])
        assert torch.equal(means[p], m) and torch.equal(grads[p], g), p
    ev = IterationCounts(9, 1.0, 1e-10, "lower_tri", blas_variant=0)
    crow = np.clip(rows[:3], 0, 1)
    big = np.concatenate([np.tile(crow, (22000, 1)), crow[:1]])  # 66001 rows: two launches of the counts kernel
    pop = ev.population_grid_summary(2, 3, RE_BOX, IM_BOX, big)
    ref = [ev.grid_summary(2, 3, RE_BOX, IM_BOX, r).hist for r in crow]
    for p in (0, 1, 2, 65534, 65535, 65536, 66000):
        assert np.array_equal(pop.hist[p], ref[p % 3]), p


# ---- 4. determinism -------------------------------------------------------------------------------------------------
def test_determinism_and_streams():
    rng = np.random.default_rng(4)
    loss = SpectralRadiusLoss(6, 1.0, "lower_tri")
    rows = _rho_rows(rng, 5, 6, "lower_tri", True)
    ev = IterationCounts(6, 1.0, 1e-10, "lower_tri", blas_variant=0)
    crow = _population(rng, 5, 6, "lower_tri", True, False)
    a = loss.population_grid_value_and_grad(200, 201, RE_BOX, IM_BOX, rows)
    h = ev.population_grid_summary(200, 201, RE_BOX, IM_BOX, crow).hist
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        b = loss.population_grid_value_and_grad(200, 201, RE_BOX, IM_BOX, rows)
        h2 = ev.population_grid_summary(200, 201, RE_BOX, IM_BOX, crow).hist
    torch.cuda.synchronize()
    c = loss.population_grid_value_and_grad(200, 201, RE_BOX, IM_BOX, rows)
    assert all(torch.equal(x, y) and torch.equal(x, z) for x, y, z in zip(a, b, c))
    assert np.array_equal(h, h2)


# ---- 5. distribution ------------------------------------------------------------------------------------------------
def _dist_worker(rank, ws, port, backend, tmp):
    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank if backend == "nccl" else 0)
    dist.init_process_group(backend, rank=rank, world_size=ws)
    try:
        rows = np.array([[0.2, 0.1, 0.15, 0.12, 0.3], [0.0] * 5, [0.1] * 5])
        s = IterationCounts(5, 1.0, 1e-10, "diag", blas_variant=0).population_grid_summary(3, 65, RE_BOX, IM_BOX, rows)
        m, g = SpectralRadiusLoss(5, 1.0, "diag").population_grid_value_and_grad(3, 65, RE_BOX, IM_BOX, rows)
        np.savez(os.path.join(tmp, f"r{rank}.npz"), hist=s.hist, m=m.cpu().numpy(), g=g.cpu().numpy())
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(600)
@pytest.mark.parametrize("backend", ["gloo", "nccl"])
def test_two_rank_population_grid(tmp_path, backend):
    import torch.multiprocessing as mp

    if backend == "nccl" and torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_dist_worker, args=(2, port, backend, str(tmp_path)), nprocs=2, join=True)
    r0, r1 = np.load(tmp_path / "r0.npz"), np.load(tmp_path / "r1.npz")
    rows = np.array([[0.2, 0.1, 0.15, 0.12, 0.3], [0.0] * 5, [0.1] * 5])
    hist = IterationCounts(5, 1.0, 1e-10, "diag", blas_variant=0).population_grid_summary(3, 65, RE_BOX, IM_BOX, rows).hist
    m, g = SpectralRadiusLoss(5, 1.0, "diag").population_grid_value_and_grad(3, 65, RE_BOX, IM_BOX, rows)
    for r in (r0, r1):
        assert np.array_equal(r["hist"], hist)
        # the all-reduced sums add the shards' sums: equal to the single process up to the order of that one addition
        assert np.allclose(r["m"], m.cpu().numpy(), rtol=1e-13) and np.allclose(r["g"], g.cpu().numpy(), rtol=1e-12)
    assert np.array_equal(r0["m"], r1["m"]) and np.array_equal(r0["g"], r1["g"])


# ---- 6. autograd ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cplx", [False, True])
def test_autograd_per_row(cplx):
    rng = np.random.default_rng(6)
    loss = SpectralRadiusLoss(5, 1.0, "lower_tri")
    rows = torch.tensor(_rho_rows(rng, 4, 5, "lower_tri", cplx), device="cuda", requires_grad=True)
    v = loss.population_grid_differentiable(40, 41, RE_BOX, IM_BOX, rows)
    assert v.shape == (4,)
    v.sum().backward()
    lam = rng.uniform(*RE_BOX, 500) + 1j * rng.uniform(*IM_BOX, 500)
    rows2 = rows.detach().clone().requires_grad_(True)
    (loss.population_differentiable(lam, rows2) * torch.arange(1.0, 5.0, device="cuda", dtype=torch.float64)).sum().backward()
    for p in range(4):
        one = rows[p].detach().clone().requires_grad_(True)
        w = loss.grid_differentiable(40, 41, RE_BOX, IM_BOX, one)
        w.backward()
        assert torch.equal(v[p].detach(), w.detach()) and torch.equal(rows.grad[p], one.grad), p
        one2 = rows[p].detach().clone().requires_grad_(True)
        loss.differentiable(lam, one2).backward()
        assert torch.equal(rows2.grad[p], one2.grad * (p + 1)), p


# ---- 7. refusals and memory -----------------------------------------------------------------------------------------
def test_refusals():
    ev = IterationCounts(5, 1.0, 1e-10, "lower_tri", free_action_space=False)
    loss = SpectralRadiusLoss(5, 1.0, "lower_tri")
    lam = _lams(np.random.default_rng(0), 8)
    for bad in (np.zeros((0, 15)), np.zeros((3, 14)), np.zeros(15), np.zeros((2, 3, 15))):
        with pytest.raises(ValueError):
            ev.population_summary(lam, bad)
        with pytest.raises(ValueError):
            ev.population_grid_summary(8, 8, RE_BOX, IM_BOX, bad)
        with pytest.raises(ValueError):
            loss.population_value_and_grad(lam, bad)
        with pytest.raises(ValueError):
            loss.population_grid_value_and_grad(8, 8, RE_BOX, IM_BOX, bad)
    with pytest.raises(TypeError):
        ev.population_summary(lam, np.zeros((3, 15), np.complex128))  # complex rows without free_action_space
    with pytest.raises(TypeError):
        ev.population_summary(lam, np.zeros((3, 15), np.int64))
    with pytest.raises(ValueError):
        IterationCounts(5, 1.0, 1e-10, prec="LU").population_summary(lam, np.zeros((3, 5)))
    with pytest.raises(ValueError):
        SpectralRadiusLoss(5, 1.0, prec="LU").population_value_and_grad(lam, np.zeros((3, 5)))
    with pytest.raises(ValueError):
        ev.population_grid_summary(8, 8, RE_BOX, IM_BOX, np.zeros((3, 15)), rows=(3, 9))
    s = ev.population_summary(np.zeros(0, np.complex128), np.zeros((2, 15)))
    assert len(s) == 2 and not s.hist.any() and (s.mean_niter == 666.0).all() and (s.success_rate == 0.0).all()


def test_peak_memory():
    """P times the single-row scratch plus a small constant"""
    M, pt, P, n = 9, "lower_tri", 64, 1024
    loss = SpectralRadiusLoss(M, 1.0, pt)
    rows = torch.as_tensor(_rho_rows(np.random.default_rng(2), P, M, pt, False), device="cuda")
    single = int(loss._L.sdcgym_spectral_radius_grad_sum_scratch_doubles(M, loss._desc.prec_type, n * n)) * 8
    loss.population_grid_value_and_grad(n, n, RE_BOX, IM_BOX, rows)  # warm-up
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    loss.population_grid_value_and_grad(n, n, RE_BOX, IM_BOX, rows)
    torch.cuda.synchronize()
    assert torch.cuda.max_memory_allocated() - base <= P * single + (1 << 20)
    ev = IterationCounts(M, 1.0, 1e-10, pt, blas_variant=0)
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    ev.population_grid_summary(n, n, RE_BOX, IM_BOX, rows)
    torch.cuda.synchronize()
    assert torch.cuda.max_memory_allocated() - base <= (1 << 20)


# ---- 8. examples ----------------------------------------------------------------------------------------------------
def _load(name):
    import importlib.util

    path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "examples", name)
    spec = importlib.util.spec_from_file_location(name[:-3] + "_population_example", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_examples(capsys):
    hist, theta = _load("train_diag_spectral_radius.py").main(
        ["--M", "5", "--starts", "4", "--grid", "32", "--steps", "5", "--eval-grid", "32"])
    assert theta.shape == (4, 5)
    text = capsys.readouterr().out
    assert "best start" in text and "MIN -- Mean number" in text and "start 3 -- Mean number" in text
    with pytest.raises(SystemExit):
        _load("train_diag_spectral_radius.py").main(["--starts", "2", "--sweeps", "3", "--steps", "1"])
    res = _load("search_niter.py").main(["--M", "5", "--grid", "32", "--generations", "2", "--lam", "6",
                                         "--rho-steps", "3"])
    assert res["best"].shape == (5,)
    text = capsys.readouterr().out
    assert "MIN -- Mean number" in text and "RHO -- Mean number" in text and "ES  -- Mean number" in text

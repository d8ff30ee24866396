"""GPU: iteration counts of the sdc-v0 full solve from the reset state (``full_solve_counts_kernel`` through
``sdcgym_full_solve_counts``, ``IterationCounts``) against the env route ``make("sdc-v0")`` + ``reset(lam)`` +
``step_tensor``, bit for bit, and its summaries against ``test_model``'s formula."""
import os
import socket
from fractions import Fraction

import numpy as np
import pytest
import torch

import sdc_gym_b200
from sdc_gym_b200.iterations import IterationCounts
from sdc_gym_b200.loss import SpectralRadiusLoss
from sdc_gym_b200.precond import num_actions

pytestmark = pytest.mark.gpu

RE_BOX, IM_BOX = (-100.0, 0.0), (-10.0, 0.0)
MAX_ITERS = 50


def _lams(rng, n):
    """random lambdas of the box, plus lambda = 0, lambdas far outside it (err nodes with prec='zeros' / 'EE') and
    -4, -5 (50 sweeps without convergence with prec='zeros')"""
    lam = rng.uniform(*RE_BOX, n) + 1j * rng.uniform(*IM_BOX, n)
    special = [0.0, -1e4, -3e3 + 50j, -4.0, -5.0, -700.0 - 300j, -0.3 - 0.1j, -1.0]
    lam[: min(n, len(special))] = special[: min(n, len(special))]
    return lam


def _rows(rng, n, M, prec_type, cplx, do_scale):
    A = num_actions(M, prec_type)
    if cplx:
        return rng.uniform(0, 0.4, (n, A)) + 1j * rng.uniform(-0.05, 0.05, (n, A))
    return rng.uniform(-1, 1, (n, A)) if do_scale else rng.uniform(0, 0.5, (n, A))


def env_route(M, lam, actions, *, prec=None, prec_type="diag", do_scale=False, free_action_space=True,
              use_doubles=True, blas_variant=0, restol=1e-10, dt=1.0):
    """(niter, residual, flags) numpy of reset(lam) + step_tensor(rows) on an sdc-v0 env of len(lam) envs"""
    n = len(lam)
    kw = dict(prec=prec) if prec else dict(prec_type=prec_type)
    env = sdc_gym_b200.make("sdc-v0", num_envs=n, M=M, dt=dt, restol=restol, do_scale=do_scale,
                            free_action_space=free_action_space, use_doubles=use_doubles, blas_variant=blas_variant,
                            autoreset=False, phased=False, **kw)
    env.reset(lam=lam)
    a = None
    if actions is not None:
        a = torch.as_tensor(actions, device=env.device)
        if a.dim() == 1:
            a = a.expand(n, -1)
    out = env.step_tensor(a)
    res = tuple(out[k].cpu().numpy().copy() for k in ("niter", "residual", "flags"))
    env.close()
    return res


def _np(t):
    return t.cpu().numpy()


def assert_bits(a, b, what):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    if a.dtype == np.float64:
        a, b = a.view(np.int64), b.view(np.int64)
    assert np.array_equal(a, b), what


CONFIGS = [
    dict(prec_type="diag", cplx=False, do_scale=True, free_action_space=False),
    dict(prec_type="diag", cplx=False, do_scale=False, free_action_space=False),
    dict(prec_type="diag", cplx=True),
    dict(prec_type="diag", cplx=False),  # real rows read as complex (free_action_space)
    dict(prec_type="lower_diag", cplx=False, do_scale=False, free_action_space=False),
    dict(prec_type="lower_tri", cplx=True),
    dict(prec_type="strictly_lower_tri", cplx=False, do_scale=False, free_action_space=False),
    dict(prec_type="lower_tri", cplx=False, do_scale=True, free_action_space=False, use_doubles=False),
    dict(prec_type="diag", cplx=True, use_doubles=False),
    dict(prec="LU"), dict(prec="min"), dict(prec="EE"), dict(prec="zeros"),
]


def _split(cfg):
    cfg = dict(cfg)
    cplx = cfg.pop("cplx", False)
    return cplx, cfg


# ---- 1. per node, against the env route ---------------------------------------------------------------------------
@pytest.mark.parametrize("M", range(2, 10))
@pytest.mark.parametrize("variant", [0, 1])
def test_per_node_against_env_route(M, variant):
    rng = np.random.default_rng(100 * M + variant)
    n = 300  # ragged against the 64 / 128-thread blocks
    lam = _lams(rng, n)
    for cfg in CONFIGS:
        cplx, kw = _split(cfg)
        prec = kw.get("prec")
        ev = IterationCounts(M, 1.0, 1e-10, blas_variant=variant, **kw)
        if prec is None:
            rows = _rows(rng, n, M, kw["prec_type"], cplx, kw.get("do_scale", False))
            if kw.get("use_doubles") is False:
                rows = rows.astype(np.complex64 if cplx else np.float32)
            shared = rows[0]
        else:
            rows = shared = None
        for acts in ((rows, shared) if prec is None else (None,)):
            ref = env_route(M, lam, acts, blas_variant=variant, **kw)
            got = tuple(_np(t) for t in ev.solve(lam, None if acts is None else torch.as_tensor(acts)))
            for k, (a, b) in enumerate(zip(got, ref)):
                assert_bits(a, b, f"M={M} {cfg} shared={acts is shared} output {k}")


def test_node_classes_are_covered():
    """the lambdas of the per-node test reach every outcome: converged (lambda = 0 among them), err and exhausted"""
    M = 5
    rng = np.random.default_rng(500)
    lam = _lams(rng, 300)
    seen = set()
    for cfg in CONFIGS:
        cplx, kw = _split(cfg)
        ev = IterationCounts(M, 1.0, 1e-10, blas_variant=0, **kw)
        acts = None if kw.get("prec") else _rows(rng, 300, M, kw["prec_type"], cplx, kw.get("do_scale", False))
        niter, res, flags = (_np(t) for t in ev.solve(lam, acts))
        conv, err = (flags & 2) != 0, (flags & 4) != 0
        seen |= {"conv"} if conv.any() else set()
        seen |= {"err"} if err.any() else set()
        seen |= {"exhausted"} if (~conv & ~err).any() else set()
        assert conv[0] and res[0] == 0.0  # lambda = 0
    assert seen == {"conv", "err", "exhausted"}


# ---- 2. grid --------------------------------------------------------------------------------------------------------
def fma_node(lo, hi, a, n):
    return lo if n <= 1 else float(Fraction(hi - lo) * Fraction(a / (n - 1)) + Fraction(lo))


@pytest.mark.parametrize("pt,cplx", [("diag", False), ("lower_tri", True)])
def test_grid_nodes_and_results(pt, cplx):
    M, n_re, n_im = 5, 37, 41
    rng = np.random.default_rng(7)
    row = _rows(rng, 1, M, pt, cplx, False)[0]
    ev = IterationCounts(M, 1.0, 1e-10, pt, blas_variant=0)
    niter, res, flags, lam = ev.grid(n_re, n_im, RE_BOX, IM_BOX, row, return_lam=True)
    a, b = np.divmod(np.arange(n_re * n_im), n_im)
    ref = np.array([complex(fma_node(*RE_BOX, int(i), n_re), fma_node(*IM_BOX, int(j), n_im)) for i, j in zip(a, b)])
    lam_np = _np(lam).reshape(-1)
    assert_bits(lam_np.view(np.float64), ref.view(np.float64), "grid nodes")
    # the nodes of SpectralRadiusLoss.grid, bit for bit
    sr = SpectralRadiusLoss(M, 1.0, pt)
    assert_bits(_np(sr.spectral_radii(lam_np, row)), _np(sr.grid(n_re, n_im, RE_BOX, IM_BOX, row)).reshape(-1), "rho")
    # grid results are list-mode results on those lambdas, and the env's
    l_niter, l_res, l_flags = (_np(t) for t in ev.solve(lam_np, row))
    assert_bits(_np(niter).reshape(-1), l_niter, "niter")
    assert_bits(_np(res).reshape(-1), l_res, "residual")
    assert_bits(_np(flags).reshape(-1), l_flags, "flags")
    e = env_route(M, lam_np, row, prec_type=pt)
    assert_bits(l_niter, e[0], "env niter")
    assert_bits(l_res, e[1], "env residual")
    assert_bits(l_flags, e[2], "env flags")
    # the corner node is lambda = 0: converged, a success
    assert lam_np[-1] == 0 and l_flags[-1] & 2 and not l_flags[-1] & 4 and l_res[-1] == 0.0 and l_niter[-1] < 50


# ---- 3. summary -----------------------------------------------------------------------------------------------------
def hist_of(niter, flags):
    conv, err = (flags & 2) != 0, (flags & 4) != 0
    h = np.bincount(niter[conv & ~err], minlength=MAX_ITERS + 3)[: MAX_ITERS + 3].astype(np.int64)
    h[MAX_ITERS + 1], h[MAX_ITERS + 2] = err.sum(), (~conv & ~err).sum()
    return h


def reference_test_model(niter, residual, restol):
    """the reference's evaluation (rl_playground.py:147-156): success = niter < 50 and residual < restol"""
    ok = [(int(k), float(r)) for k, r in zip(niter, residual) if k < 50 and r < restol]
    mean = np.mean([k for k, _ in ok]) if ok else 666
    return len(ok) / len(niter), mean


@pytest.mark.parametrize("N", [1, 127, 129, 4099])
@pytest.mark.parametrize("pt", ["diag", "strictly_lower_tri"])
def test_summary_histogram(N, pt):
    M = 9 if pt == "strictly_lower_tri" else 5  # 64-thread blocks at M = 9
    rng = np.random.default_rng(N)
    lam = _lams(rng, N)
    rows = _rows(rng, N, M, pt, False, False)
    ev = IterationCounts(M, 1.0, 1e-10, pt, free_action_space=False, blas_variant=0)
    niter, _, flags = (_np(t) for t in ev.solve(lam, rows))
    s = ev.summary(lam, rows)
    assert np.array_equal(s.hist, hist_of(niter, flags)) and s.count == N
    assert s.n_err == int(((flags & 4) != 0).sum()) and s.n_exhausted == int(s.hist[-1])


def test_summary_is_test_model_including_a_50th_sweep_convergence():
    M, restol = 5, 1e-10
    rng = np.random.default_rng(50)
    ev = IterationCounts(M, 1.0, restol, "diag", blas_variant=0)
    # find nodes that converge exactly on their 50th sweep (a failure for test_model)
    lam = rng.uniform(*RE_BOX, 1 << 18) + 1j * rng.uniform(*IM_BOX, 1 << 18)
    row = np.array([0.2818591930905709, 0.2011358490453793, 0.06274536689514164, 0.11790265267514095, 0.1571629578515223])
    rows = np.clip(row[None] + rng.normal(0, 0.08, (len(lam), M)), 0, 1)
    niter, res, flags = (_np(t) for t in ev.solve(lam, rows))
    at50 = np.flatnonzero((niter == 50) & ((flags & 2) != 0))
    assert len(at50) > 0, "no node converges on its 50th sweep"
    pick = np.concatenate([at50[:8], np.arange(4000)])
    lam, rows = lam[pick], rows[pick]
    e_niter, e_res, _ = env_route(M, lam, rows, restol=restol)
    s = ev.summary(lam, rows)
    rate, mean = reference_test_model(e_niter, e_res, restol)
    assert s.success_rate == rate and s.mean_niter == mean
    assert s.hist[50] >= min(8, len(at50)) and s.success_rate < 1  # converged at niter 50: counted, not a success
    # nothing succeeds: 666
    k = min(8, len(at50))
    s = ev.summary(lam[:k], rows[:k])
    assert s.success_rate == 0.0 and s.mean_niter == 666 == reference_test_model(e_niter[:k], e_res[:k], restol)[1]


def test_grid_summary_memory():
    ev = IterationCounts(5, 1.0, 1e-10, prec="min")
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    s = ev.grid_summary(4096, 4096, RE_BOX, IM_BOX)
    assert s.count == 4096 * 4096
    torch.cuda.synchronize()
    assert torch.cuda.max_memory_allocated() - base < 64 << 20


# ---- 4. sharding ----------------------------------------------------------------------------------------------------
def test_row_ranges_concatenate_to_the_grid():
    ev = IterationCounts(5, 1.0, 1e-10, "lower_tri", blas_variant=0)
    row = _rows(np.random.default_rng(3), 1, 5, "lower_tri", True, False)[0]
    full = ev.grid(50, 33, RE_BOX, IM_BOX, row)
    parts = [ev.grid(50, 33, RE_BOX, IM_BOX, row, rows=r) for r in ((0, 7), (7, 7), (7, 31), (31, 50))]
    for k in range(3):
        assert torch.equal(torch.cat([p[k] for p in parts]), full[k])
    whole = ev.grid_summary(50, 33, RE_BOX, IM_BOX, row)
    hs = [ev.grid_summary(50, 33, RE_BOX, IM_BOX, row, rows=r).hist for r in ((0, 7), (7, 31), (31, 50))]
    assert np.array_equal(sum(hs), whole.hist)
    empty = ev.grid_summary(50, 33, RE_BOX, IM_BOX, row, rows=(9, 9))
    assert not empty.hist.any() and empty.count == 0 and empty.mean_niter == 666
    with pytest.raises(ValueError):
        ev.grid_summary(50, 33, RE_BOX, IM_BOX, row, rows=(3, 51))


def _dist_worker(rank, ws, port, backend, tmp):
    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank if backend == "nccl" else 0)
    dist.init_process_group(backend, rank=rank, world_size=ws)
    try:
        ev = IterationCounts(5, 1.0, 1e-10, prec="LU", blas_variant=0)
        s = ev.grid_summary(3, 65, RE_BOX, IM_BOX)  # 2 + 1 rows
        np.save(os.path.join(tmp, f"r{rank}.npy"), s.hist)
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(600)
@pytest.mark.parametrize("backend", ["gloo", "nccl"])
def test_two_rank_grid_summary(tmp_path, backend):
    """rows=None over two ranks (gloo: both on one device; nccl: one device each) against the single-process call"""
    import torch.multiprocessing as mp

    if backend == "nccl" and torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_dist_worker, args=(2, port, backend, str(tmp_path)), nprocs=2, join=True)
    r0, r1 = np.load(tmp_path / "r0.npy"), np.load(tmp_path / "r1.npy")
    ref = IterationCounts(5, 1.0, 1e-10, prec="LU", blas_variant=0).grid_summary(3, 65, RE_BOX, IM_BOX).hist
    assert np.array_equal(r0, r1) and np.array_equal(r0, ref)


# ---- 5. other -------------------------------------------------------------------------------------------------------
def test_cuda_graph_replay_equals_eager():
    ev = IterationCounts(7, 1.0, 1e-10, "diag", blas_variant=0)
    row = torch.tensor([0.15, 0.12, 0.08, 0.04, 0.1, 0.14, 0.15], dtype=torch.float64, device="cuda")
    eager = ev.grid_summary(96, 80, RE_BOX, IM_BOX, row).hist
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        ev.grid_summary(96, 80, RE_BOX, IM_BOX, row)  # warm-up on the capture stream
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        captured = ev.grid_summary(96, 80, RE_BOX, IM_BOX, row)
    captured.hist_device.fill_(-1)
    g.replay()
    torch.cuda.synchronize()
    assert np.array_equal(captured.hist, eager)


def test_non_current_device():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    lam = _lams(np.random.default_rng(2), 1000)
    a = IterationCounts(5, 1.0, 1e-10, prec="EE", blas_variant=0, device="cuda:0")
    b = IterationCounts(5, 1.0, 1e-10, prec="EE", blas_variant=0, device="cuda:1")
    assert torch.cuda.current_device() == 0
    ra, rb = a.solve(lam), b.solve(lam)
    assert rb[0].device.index == 1
    for x, y in zip(ra, rb):
        assert torch.equal(x, y.to(x.device))
    assert np.array_equal(a.summary(lam).hist, b.summary(lam).hist)


def test_refusals():
    lam = _lams(np.random.default_rng(1), 8)
    ev = IterationCounts(5, 1.0, 1e-10, "lower_tri", free_action_space=False)
    with pytest.raises(ValueError):
        ev.solve(lam)  # actions required
    with pytest.raises(ValueError):
        ev.solve(lam, np.zeros((8, 14)))  # shape
    with pytest.raises(ValueError):
        ev.solve(lam, np.zeros((7, 15)))
    with pytest.raises(TypeError):
        ev.solve(lam, np.zeros((8, 15), np.int64))  # dtype
    with pytest.raises(TypeError):
        ev.solve(lam, np.zeros((8, 15), np.complex128))  # complex rows without free_action_space
    with pytest.raises(ValueError):
        ev.grid(8, 8, RE_BOX, IM_BOX, np.zeros((64, 15)))  # per-node rows in grid mode
    with pytest.raises(ValueError):
        ev.grid_summary(8, 8, RE_BOX, IM_BOX, np.zeros((64, 15)))
    with pytest.raises(ValueError):
        IterationCounts(5, 1.0, 1e-10, prec="LU").solve(lam, np.zeros((8, 5)))  # actions with prec
    with pytest.raises(ValueError):
        IterationCounts(5, 1.0, 1e-10, "upper")
    n, r, f = IterationCounts(5, 1.0, 1e-10, prec="LU").solve(np.zeros(0, np.complex128))
    assert n.numel() == r.numel() == f.numel() == 0
    assert IterationCounts(5, 1.0, 1e-10, prec="LU").summary(np.zeros(0, np.complex128)).count == 0


# ---- 6. examples ----------------------------------------------------------------------------------------------------
def _load(name):
    import importlib.util

    path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "examples", name)
    spec = importlib.util.spec_from_file_location(name[:-3] + "_example", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_examples(tmp_path, capsys):
    out = _load("niter_map.py").main(["--M", "5", "--grid", "48", "--save", str(tmp_path / "m")])
    assert set(out) == {"LU", "MIN", "RL"} and out["LU"].count == 48 * 48
    assert np.load(tmp_path / "m_LU.npy").shape == (48, 48)
    assert "LU  -- Mean number of iterations and success rate:" in capsys.readouterr().out
    _load("train_diag_spectral_radius.py").main(["--M", "5", "--grid", "32", "--steps", "3", "--eval-grid", "40"])
    text = capsys.readouterr().out
    assert "MIN -- Mean number" in text and "RL  -- Mean number" in text

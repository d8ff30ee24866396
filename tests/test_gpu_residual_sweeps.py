"""GPU: ``ResidualLoss.sweeps`` / ``sweeps_differentiable`` (``sdcgym_residual_sweeps``, csrc/residual_sweeps.cuh):
||r_K||_inf after K sweeps and its gradient through every sweep.

- against the 40-digit reference ``tests/mp_sweeps_reference.SweepsRef``, per sample and per entry, with the error model of
  tests/test_residual_sweeps_host.py (tolerances from the float64 twin's error on the same inputs);
- against what the env sweeps (``sdc-v1``, ``restol = 0``), K chained ``take_step`` calls, and a torch-autograd twin;
- the gradient through K >= 2 sweeps is not the last-sweep-only gradient that chained ``take_step`` calls give;
- the autograd wrapper, edge cases and determinism.
"""
import os

import numpy as np
import pytest

import sdc_gym_b200
from sdc_gym_b200.collocation import collocation_matrix
from sdc_gym_b200.precond import fixed_preconditioner, num_actions
from tests.test_loss_reference_host import LAYOUTS, draw
from tests.test_residual_sweeps_host import check_sweeps, random_state

pytestmark = pytest.mark.gpu


def _np(t):
    return t.detach().cpu().numpy()


def _outs(res):
    return tuple(_np(t) for t in res)


@pytest.mark.parametrize("M", range(2, 10))
def test_sweeps_against_mp_reference(M):
    """every layout, real and complex theta, dt = 1 and 0.5, K = 1, 2, 7, 50, from the reset state and a given state"""
    from sdc_gym_b200.loss import ResidualLoss
    rng = np.random.default_rng(2100 + M)
    n_checked, n_left = 0, 0
    for prec_type in LAYOUTS:
        for dt in (1.0, 0.5):
            loss = ResidualLoss(M, dt, prec_type)
            for cplx in (True, False):
                for K in (1, 2, 7, 50):
                    lam, theta = draw(rng, M, prec_type, 2, cplx=cplx)
                    outs = _outs(loss.sweeps(lam, theta, K, with_grad=True))
                    ek, _, lo = check_sweeps(M, prec_type, lam, theta, dt, K, outs, real=not cplx)
                    u0, u, r = random_state(rng, M, 2)
                    outs = _outs(loss.sweeps(lam, theta, K, u0, u, r, with_grad=True))
                    ek2, _, lo2 = check_sweeps(M, prec_type, lam, theta, dt, K, outs, u0=u0, u=u, r=r, real=not cplx)
                    n_checked += len(ek) + len(ek2)
                    n_left += lo + lo2
    assert n_checked >= 0.6 * (n_checked + n_left), (n_checked, n_left)


def test_sweeps_batch_edges_and_broadcast_row():
    """B = 1, 127, 129, 4099 around the 128-thread blocks give the same bits per row and match the reference at the
    block edges; one shared row (not expanded) gives the bits of the expanded rows"""
    from sdc_gym_b200.loss import ResidualLoss
    rng = np.random.default_rng(31)
    for M in (2, 5, 9):
        for prec_type in LAYOUTS:
            loss = ResidualLoss(M, 0.5, prec_type)
            lam, theta = draw(rng, M, prec_type, 4099)
            full = _outs(loss.sweeps(lam, theta, 7, with_grad=True))
            for B in (1, 127, 129):
                part = _outs(loss.sweeps(lam[:B], theta[:B], 7, with_grad=True))
                for x, y in zip(part, full):
                    assert np.array_equal(x, y[:B])
            rows = [0, 126, 127, 128, 4095, 4098]
            check_sweeps(M, prec_type, lam[rows], theta[rows], 0.5, 7, tuple(x[rows] for x in full))
            one = theta[:1]
            a = _outs(loss.sweeps(lam[:300], one[0], 7, with_grad=True))
            b = _outs(loss.sweeps(lam[:300], np.repeat(one, 300, axis=0), 7, with_grad=True))
            for x, y in zip(a, b):
                assert np.array_equal(x, y)
            check_sweeps(M, prec_type, lam[:3], one[0], 0.5, 7, tuple(x[:3] for x in a))


def _tol(u0, C, u):
    """1e-12 of ||u0|| + ||C|| ||u|| per sample"""
    return 1e-12 * (np.max(np.abs(u0), axis=1) + np.max(np.sum(np.abs(C), axis=2), axis=1) * np.max(np.abs(u), axis=1))


@pytest.mark.parametrize("K", [1, 5, 10])
def test_sweeps_measure_what_the_env_sweeps(K):
    """sdc-v1 with complex diagonal actions near MIN (free_action_space, no scaling), lambdas injected by reset, restol
    = 0 and K steps: u, r and ||r|| of the env agree with ``sweeps`` from the reset state"""
    import torch
    from sdc_gym_b200.loss import ResidualLoss
    M, n = 5, 2048
    rng = np.random.default_rng(40 + K)
    lam = rng.uniform(-100, 0, n) + 1j * rng.uniform(-10, 0, n)
    theta = (np.diag(fixed_preconditioner("min", M))[None] + rng.uniform(-0.02, 0.02, (n, M))
             + 1j * rng.uniform(-0.01, 0.01, (n, M)))
    env = sdc_gym_b200.make("sdc-v1", num_envs=n, M=M, dt=1.0, restol=0.0, free_action_space=True, do_scale=False,
                            lambda_real_interval=[-100, 0], lambda_imag_interval=[-10, 0], seed=1)
    env.reset(lam=lam)
    act = torch.as_tensor(theta, device="cuda")
    for _ in range(K):
        out = env.step_tensor(act)
    assert not bool((out["flags"] & sdc_gym_b200._lib.FLAG_ERR).any())
    obs = _np(env.observation_tensor())
    u_env, r_env = obs[:, 0], obs[:, 1]
    u_K, r_K, norms = _outs(ResidualLoss(M, 1.0, "diag").sweeps(lam, theta, K))
    Q = collocation_matrix(M)
    C = np.eye(M)[None] - lam[:, None, None] * Q[None]
    tol = _tol(np.ones((n, M)), C, u_K)
    assert np.all(np.max(np.abs(u_env - u_K), axis=1) <= tol)
    assert np.all(np.max(np.abs(r_env - r_K), axis=1) <= tol)
    assert np.all(np.abs(np.max(np.abs(r_env), axis=1) - norms) <= tol)


@pytest.mark.parametrize("prec_type", LAYOUTS)
def test_sweeps_against_chained_take_step_and_the_truncated_gradient(prec_type):
    """K chained take_step(Cs=None) calls give the same u, r, ||r|| within 1e-12 of ||u0|| + ||C|| ||u||; for K = 1 the
    gradient is take_step's; for K >= 2 it differs from the last sweep's take_step gradient (what summing the chained
    calls' last term gives) by far more than that"""
    from sdc_gym_b200.loss import ResidualLoss
    M, n = 5, 512
    rng = np.random.default_rng(50)
    lam, theta = draw(rng, M, prec_type, n)
    u0, u, r = random_state(rng, M, n)
    loss = ResidualLoss(M, 1.0, prec_type)
    Q = collocation_matrix(M)
    C = np.eye(M)[None] - lam[:, None, None] * Q[None]
    for K in (1, 2, 5, 20):
        u_K, r_K, norms, g = _outs(loss.sweeps(lam, theta, K, u0, u, r, with_grad=True))
        uc, rc = u, r
        for _ in range(K):
            uc, rc, nc, gc = _outs(loss.take_step(lam, theta, None, u0, uc, rc, with_grad=True))
        tol = _tol(u0, C, u_K)
        assert np.all(np.max(np.abs(uc - u_K), axis=1) <= tol)
        assert np.all(np.max(np.abs(rc - r_K), axis=1) <= tol)
        assert np.all(np.abs(nc - norms) <= tol)
        scale = np.max(np.abs(g), axis=1)
        diff = np.max(np.abs(gc - g), axis=1) / scale
        if K == 1:
            assert np.max(diff) <= 1e-10, np.max(diff)
        else:
            assert np.median(diff) > 1e-3, (K, np.median(diff))


def _torch_twin(M, prec_type, dt, lam, theta, K, u0=None, u=None, r=None):
    """the K sweeps as batched complex128 torch ops (triangular solves), differentiated by autograd: (norms, g) with
    g in the kernels' convention d n = Re sum g d theta"""
    import torch
    from tests import mp_reference as R
    dev = torch.device("cuda")
    B = len(lam)
    th = torch.as_tensor(theta, device=dev).to(torch.complex128).requires_grad_(True)
    z = torch.as_tensor(lam * dt, device=dev).to(torch.complex128)
    idx = R.param_index(M, prec_type)
    rows = torch.tensor([a for a, _ in idx], device=dev)
    cols = torch.tensor([c for _, c in idx], device=dev)
    Qd = torch.zeros((B, M, M), dtype=torch.complex128, device=dev)
    Qd = Qd.index_put((torch.arange(B, device=dev)[:, None], rows[None], cols[None]), th)
    Q = torch.as_tensor(collocation_matrix(M), device=dev).to(torch.complex128)
    eye = torch.eye(M, dtype=torch.complex128, device=dev)
    P = eye - z[:, None, None] * Qd
    C = eye - z[:, None, None] * Q
    if u0 is None:
        u0t = torch.ones((B, M), dtype=torch.complex128, device=dev)
        ut = u0t.clone()
        rt = u0t - (C @ ut[..., None])[..., 0]
    else:
        u0t, ut, rt = (torch.as_tensor(x, device=dev) for x in (u0, u, r))
    for _ in range(K):
        dl = torch.linalg.solve_triangular(P, rt[..., None], upper=False)[..., 0]
        ut = ut + dl
        rt = u0t - (C @ ut[..., None])[..., 0]
    n = rt.abs().amax(dim=1)
    n.sum().backward()
    return _np(n), np.conj(_np(th.grad))


@pytest.mark.parametrize("prec_type", LAYOUTS)
def test_sweeps_gradient_against_torch_autograd(prec_type):
    from sdc_gym_b200.loss import ResidualLoss
    rng = np.random.default_rng(60)
    for M in (3, 5, 9):
        lam, theta = draw(rng, M, prec_type, 1000)
        for K in (1, 4, 12):
            _, _, norms, g = _outs(ResidualLoss(M, 1.0, prec_type).sweeps(lam, theta, K, with_grad=True))
            tn, tg = _torch_twin(M, prec_type, 1.0, lam, theta, K)
            ok = np.isfinite(tn) & (tn > 1e-6)
            assert np.all(np.abs(tn - norms)[ok] <= 1e-10 * (1 + tn[ok]))
            err = np.max(np.abs(tg - g), axis=1) / np.max(np.abs(tg), axis=1)
            assert np.percentile(err[ok], 99) <= 1e-9 and np.median(err[ok]) <= 1e-12, (M, K, np.max(err[ok]))


def test_sweeps_differentiable_backward_and_central_difference():
    """backward for per-sample rows and one shared row against g; a central difference along a random direction; real
    rows get a real gradient, complex rows the torch convention"""
    import torch
    from sdc_gym_b200.loss import ResidualLoss
    M, n, K = 5, 256, 6
    rng = np.random.default_rng(70)
    for prec_type in ("diag", "lower_tri"):
        loss = ResidualLoss(M, 1.0, prec_type)
        for cplx in (False, True):
            lam, theta = draw(rng, M, prec_type, n, cplx=cplx)
            _, _, norms, g = loss.sweeps(lam, theta, K, with_grad=True)
            th = torch.as_tensor(theta, device="cuda").requires_grad_(True)
            nd = loss.sweeps_differentiable(lam, th, K)
            assert torch.equal(nd.detach(), norms)
            w = torch.rand(n, dtype=torch.float64, device="cuda")
            (nd * w).sum().backward()
            want = (g * w[:, None]).conj() if cplx else (g.real * w[:, None])
            assert th.grad.dtype == th.dtype and torch.allclose(th.grad, want, rtol=1e-14, atol=0)
            row = torch.as_tensor(theta[0], device="cuda").requires_grad_(True)
            torch.log(loss.sweeps_differentiable(lam, row, K)).mean().backward()
            _, _, n1, g1 = loss.sweeps(lam, theta[0], K, with_grad=True)
            gr = (g1 / n1[:, None]).sum(0) / n
            assert row.grad.shape == row.shape and torch.allclose(row.grad, gr.conj() if cplx else gr.real,
                                                                  rtol=1e-12, atol=0)
            # central difference of mean log n along a random direction of the shared row
            d = rng.normal(size=theta.shape[1]) + (1j * rng.normal(size=theta.shape[1]) if cplx else 0)
            h = 1e-6
            f = lambda s: float(torch.log(loss.sweeps(lam, theta[0] + s * d, K)[2]).mean())  # noqa: E731
            fd = (f(h) - f(-h)) / (2 * h)
            an = float(np.real(np.sum(np.conj(_np(row.grad)) * d))) if cplx else float(np.sum(_np(row.grad) * d))
            assert abs(fd - an) <= 1e-6 * max(1.0, abs(an)), (prec_type, cplx, fd, an)


def test_sweeps_edges_and_determinism():
    """a diverging sample (+inf or NaN, g = 0) next to finite ones, lambda = 0 (norm 0, g = 0), and the same bits on
    two calls and on two streams"""
    import torch
    from sdc_gym_b200.loss import ResidualLoss
    M = 5
    loss = ResidualLoss(M, 1.0, "diag")
    lam = np.array([-50.0, -1e10, 0.0, -30 - 3j], np.complex128)
    theta = np.full((4, M), 0.2)
    theta[1] = 0.0
    _, _, norms, g = _outs(loss.sweeps(lam, theta, 50, with_grad=True))
    assert np.isfinite(norms[[0, 3]]).all() and np.all(np.any(g[[0, 3]] != 0, axis=1))
    assert not np.isfinite(norms[1]) and np.all(g[1] == 0)
    assert norms[2] == 0.0 and np.all(g[2] == 0)
    rng = np.random.default_rng(80)
    lam, theta = draw(rng, M, "lower_tri", 20000)
    loss = ResidualLoss(M, 1.0, "lower_tri")
    a = _outs(loss.sweeps(lam, theta, 20, with_grad=True))
    b = _outs(loss.sweeps(lam, theta, 20, with_grad=True))
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        c = loss.sweeps(lam, theta, 20, with_grad=True)
    s.synchronize()
    c = _outs(c)
    for x, y, w in zip(a, b, c):
        assert np.array_equal(x, y, equal_nan=True) and np.array_equal(x, w, equal_nan=True)


def test_example_with_sweeps_lowers_its_loss():
    import importlib.util
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("train", os.path.join(root, "examples",
                                                                        "train_diag_spectral_radius.py"))
    tr = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(tr)
    hist, theta = tr.main(["--steps", "60", "--batch", "16384", "--sweeps", "5"])
    assert hist[-1] < hist[0] - 0.5 and np.all(np.isfinite(theta))

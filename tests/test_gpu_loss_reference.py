"""GPU: the loss gradients of the device kernels against a 40-digit reference (tests/mp_reference.py), per sample and
per entry - never a batch sum, in which a wrong entry of a few samples disappears.

SpectralRadiusLoss (``rho_grad_kernel``, csrc/specrad.cuh ``spectral_radius_grad_one``): the error model of
tests/test_loss_reference_host.py, per sample,
    rho:  |rho - rho_mp| / rho_mp                  <= 128 eps kappa
    g:    max_k |g_k - g_mp,k| / max_k |g_mp,k|     <= 64 max(twin error, eps kappa)
with the float64 twin of the same formula (numpy inverse, LAPACK zgeev left and right vectors) on the same inputs.
Samples with kappa > 1e6 or a modulus gap below 1e-6 are excluded and counted.

ResidualLoss (``residual_step_kernel``, csrc/vecnorm.cu): u' = u + P^{-1} r, r' = u0 - C u' and the gradient of
||r'||_inf are triangular solves and products, whose float64 error is bounded by eps times the Skeel condition
number s(P) = || |P^{-1}| |P| ||_inf.  Per sample,
    u', g:    max error / max |reference|                       <= 64 max(twin error, M eps s(P))
    r', norm: max error / (max |u0| + || |C| |u'| ||_inf)        <= 64 max(twin error, M eps s(P))
Samples whose two largest |r'_k| are within 1e-6 relative (where the max has no derivative) are left out of the
gradient check and counted.

Run with ``-s`` to see the per-(M, layout) maximum and 99th percentile of the kernel's and the twin's errors.
"""
import numpy as np
import pytest

from sdc_gym_b200.collocation import collocation_matrix
from sdc_gym_b200.precond import fixed_preconditioner, num_actions
from tests import mp_reference as R
from tests.test_loss_reference_host import C_GRAD, EPS, LAYOUTS, check_specrad, draw

pytestmark = pytest.mark.gpu


def _np(t):
    return t.detach().cpu().numpy()


def _stats(name, ek, et, excluded, n):
    if len(ek):
        print(f"\n{name}: n={n} excluded={excluded} kernel max {ek.max():.2e} p99 {np.percentile(ek, 99):.2e} | "
              f"twin max {et.max():.2e} p99 {np.percentile(et, 99):.2e}")


@pytest.mark.parametrize("M", range(2, 10))
def test_spectral_radius_gradient_against_mp_reference(M):
    """radii_and_grads and value_and_grad for every layout: complex outputs at dt = 1 and 0.1, real outputs, real
    lambda with real outputs (K real; its dominant eigenvalue is often a conjugate pair)"""
    import torch
    from sdc_gym_b200.loss import SpectralRadiusLoss
    rng = np.random.default_rng(300 + M)
    for prec_type in LAYOUTS:
        eks, ets, n_ex, n_all = [], [], 0, 0
        for n, dt, cplx, real_lam in ((16, 1.0, True, False), (8, 0.1, True, False), (8, 0.1, False, False),
                                      (8, 1.0, False, True)):
            lam, qd = draw(rng, M, prec_type, n, cplx=cplx, real_lam=real_lam)
            loss = SpectralRadiusLoss(M, dt, prec_type)
            rho_t, g_t = loss.radii_and_grads(lam, qd)
            val, gv = loss.value_and_grad(lam, qd)
            assert torch.equal(gv, g_t / n if cplx else g_t.real / n) and gv.is_complex() == cplx
            assert float(val) == float(loss.mean(rho_t))
            ek, et, ex = check_specrad(M, prec_type, lam, qd, dt, _np(rho_t), _np(g_t), real=not cplx)
            eks.append(ek)
            ets.append(et)
            n_ex += ex
            n_all += n
        _stats(f"rho grad M={M} {prec_type}", np.concatenate(eks), np.concatenate(ets), n_ex, n_all)
        assert n_ex <= 0.05 * n_all


def test_spectral_radius_gradient_edges():
    """lambda = 0 gives rho = 0 and g = 0 exactly; a broadcast output row equals the expanded rows bit for bit;
    B = 1, 127, 129 and 4099 around the 128-thread blocks give the same bits per row and match the reference at the
    block edges; Q_delta within 1e-4 of MIN (K numerically singular) matches the reference"""
    import torch
    from sdc_gym_b200.loss import SpectralRadiusLoss
    rng = np.random.default_rng(77)
    for M in (2, 5, 9):
        for prec_type in LAYOUTS:
            loss = SpectralRadiusLoss(M, 0.5, prec_type)
            lam, qd = draw(rng, M, prec_type, 4099)
            lam[[3, 128, 4098]] = 0.0
            rho, g = loss.radii_and_grads(lam, qd)
            rho, g = _np(rho), _np(g)
            assert np.all(rho[[3, 128, 4098]] == 0.0) and np.all(g[[3, 128, 4098]] == 0.0)
            for B in (1, 127, 129):
                rb, gb = loss.radii_and_grads(lam[:B], qd[:B])
                assert np.array_equal(_np(rb), rho[:B]) and np.array_equal(_np(gb), g[:B])
            rows = [0, 126, 127, 129, 4095, 4096, 4097]
            check_specrad(M, prec_type, lam[rows], qd[rows], 0.5, rho[rows], g[rows])
            one = qd[:1]
            rb, gb = loss.radii_and_grads(lam[:200], one)
            re, ge = loss.radii_and_grads(lam[:200], np.repeat(one, 200, axis=0))
            assert torch.equal(rb, re) and torch.equal(gb, ge)
            assert torch.equal(loss.value_and_grad(lam[:200], torch.as_tensor(one[0], device="cuda"))[1],
                               loss.value_and_grad(lam[:200], np.repeat(one, 200, axis=0))[1])
    n_ex = 0
    for M in (3, 4, 5, 7):
        base = np.diag(fixed_preconditioner("min", M))
        lam = rng.uniform(-100, 0, 16) + 1j * rng.uniform(-10, 0, 16)
        qd = base[None] + rng.uniform(-1e-4, 1e-4, (16, M))
        rho, g = SpectralRadiusLoss(M, 1.0, "diag").radii_and_grads(lam, qd)
        n_ex += check_specrad(M, "diag", lam, qd, 1.0, _np(rho), _np(g), real=True)[2]
    assert n_ex == 0


def _skeel(z, Qd):
    P = np.eye(Qd.shape[0]) - z * Qd
    return np.max(np.sum(np.abs(np.linalg.inv(P)) @ np.abs(P), axis=1))


def _check_residual(M, prec_type, lam, theta, dt, u0, u, r_old, C, outs, *, real, grad=True):
    """per-sample comparison of one ResidualLoss step (u', r', norms, g) with ResidualRef; returns (kernel errors,
    twin errors, number left out of the gradient check)"""
    u_new, r_new, norms, g = outs
    Q = collocation_matrix(M)
    ek, et, left_out = [], [], 0
    for i in range(len(lam)):
        Ci = None if C is None else C[i]
        ref = R.ResidualRef(Q, lam[i], dt, theta[i], prec_type, u0[i], u[i], r_old[i], Ci)
        tu, tr, tn, tg = R.residual_twin(Q, lam[i], dt, theta[i], prec_type, u0[i], u[i], r_old[i], Ci)
        Qd = np.zeros((M, M), np.complex128)
        for k, (r, c) in enumerate(R.param_index(M, prec_type)):
            Qd[r, c] = theta[i][k]
        floor = M * EPS * _skeel(R.z_of(lam[i], dt), Qd)
        Cm = np.eye(M) - R.z_of(lam[i], dt) * Q if Ci is None else Ci
        su = np.max(np.abs(ref.u_new))
        sr = np.max(np.abs(u0[i])) + np.max(np.abs(Cm) @ np.abs(ref.u_new))
        for got, want, twin, scale, what in ((u_new[i], ref.u_new, tu, su, "u'"), (r_new[i], ref.r_new, tr, sr, "r'"),
                                             (norms[i], ref.norm, tn, sr, "norm")):
            e_k, e_t = np.max(np.abs(got - want)) / scale, np.max(np.abs(twin - want)) / scale
            assert e_k <= C_GRAD * max(e_t, floor), (what, M, prec_type, i, e_k, e_t, floor)
        if not grad:
            continue
        if ref.gap2 < 1e-6 or ref.norm == 0:
            left_out += 1
            continue
        gk, gr, gt = (g[i].real, ref.g.real, tg.real) if real else (g[i], ref.g, tg)
        s = np.max(np.abs(gr))
        if s == 0:  # r_old = 0: nothing moves with Q_delta
            assert np.all(gk == 0)
            continue
        e_k, e_t = np.max(np.abs(gk - gr)) / s, np.max(np.abs(gt - gr)) / s
        assert e_k <= C_GRAD * max(e_t, floor), ("g", M, prec_type, i, e_k, e_t, floor)
        ek.append(e_k)
        et.append(e_t)
    return np.array(ek), np.array(et), left_out


def _residual_inputs(rng, M, lam, dt, n):
    Q = collocation_matrix(M)
    z = np.array([R.z_of(l, dt) for l in lam])
    u0 = rng.uniform(0, 1, (n, M)) + 1j * rng.uniform(0, 1, (n, M))
    u = rng.uniform(0, 1, (n, M)) + 1j * rng.uniform(0, 1, (n, M))
    C = np.eye(M)[None] - z[:, None, None] * Q[None]
    C_pert = C + 1e-2 * (rng.normal(size=(n, M, M)) + 1j * rng.normal(size=(n, M, M)))
    r_old = u0 - np.einsum("bij,bj->bi", C, u)
    return u0, u, r_old, C_pert


@pytest.mark.parametrize("M", range(2, 10))
def test_residual_loss_step_and_gradient_against_mp_reference(M):
    """take_step(with_grad=True) and value_and_grad for every layout, real and complex outputs, dt = 0.7, with the
    system matrices given (Cs, here not I - zQ, so a wrong row of Cs shows) and formed on the device (Cs=None);
    rows with r_old = 0 give u' = u and g = 0 exactly"""
    import torch
    from sdc_gym_b200.loss import ResidualLoss
    rng = np.random.default_rng(500 + M)
    dt, n = 0.7, 12
    for prec_type in LAYOUTS:
        loss = ResidualLoss(M, dt, prec_type)
        eks, ets, n_lo = [], [], 0
        for cplx in (True, False):
            lam, theta = draw(rng, M, prec_type, n, cplx=cplx)
            u0, u, r_old, C_pert = _residual_inputs(rng, M, lam, dt, n)
            r_old[5] = 0.0
            for C in (C_pert, None):
                outs_t = loss.take_step(lam, theta, C, u0, u, r_old, with_grad=True)
                outs = tuple(_np(t) for t in outs_t)
                assert np.array_equal(outs[0][5], u[5]) and np.all(outs[3][5] == 0.0)
                assert outs[3].shape == (n, num_actions(M, prec_type)) and np.iscomplexobj(outs[3])
                (val, _, _), gv = loss.value_and_grad(lam, theta, C, u0, u, r_old)
                assert torch.equal(gv, (outs_t[3] if cplx else outs_t[3].real) / n) and gv.is_complex() == cplx
                ek, et, lo = _check_residual(M, prec_type, lam, theta, dt, u0, u, r_old, C, outs, real=not cplx)
                eks.append(ek)
                ets.append(et)
                n_lo += lo
        _stats(f"residual grad M={M} {prec_type}", np.concatenate(eks), np.concatenate(ets), n_lo, 4 * n)
        assert n_lo <= 0.05 * 4 * n


@pytest.mark.parametrize("M", [3, 5, 9])
def test_residual_loss_with_a_fixed_preconditioner_against_mp_reference(M):
    """a fixed prec (LU): values against the reference, and a gradient with no parameters, shape (B, 0)"""
    from sdc_gym_b200.loss import ResidualLoss
    rng = np.random.default_rng(600 + M)
    n, dt = 16, 0.3
    Qd = fixed_preconditioner("LU", M)
    theta = np.tile(Qd[np.tril_indices(M)], (n, 1))
    lam = rng.uniform(-100, 0, n) + 1j * rng.uniform(-10, 0, n)
    u0, u, r_old, C_pert = _residual_inputs(rng, M, lam, dt, n)
    loss = ResidualLoss(M, dt, prec="LU")
    for C in (C_pert, None):
        outs = tuple(_np(t) for t in loss.take_step(lam, None, C, u0, u, r_old, with_grad=True))
        assert outs[3].shape == (n, 0)
        _check_residual(M, "lower_tri", lam, theta, dt, u0, u, r_old, C, outs, real=False, grad=False)

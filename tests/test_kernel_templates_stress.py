"""CPU: kernel templates (host shim) against the C oracle on seeded batches large enough to exercise the
integer band / squared-magnitude / exact-norm decision stages and the single-candidate fast norm."""
import numpy as np
import pytest

from oracle import exact
from sdc_gym_b200.collocation import collocation_matrix
from sdc_gym_b200.precond import fixed_preconditioner, num_actions
from tests import host_shim
from tests.helpers import assert_reward_close, assert_same


def _run(kind, M, n, *, prec=None, prec_type="diag", mode="good", steps=1, strategy="iteration_only", seed=0,
         im_int=(-10, 0), variant=0, entry="shim_step"):
    rng = np.random.default_rng(seed)
    Q = collocation_matrix(M)
    lam = rng.uniform(-100, 0, n) + 1j * rng.uniform(im_int[0], im_int[1], n)
    d = host_shim.make_desc(kind, M, prec=prec, prec_type=prec_type, do_scale=(prec_type == "diag"), strategy=strategy,
                            variant=variant)
    b = host_shim.ShimBatch(d, n, entry=entry)
    u, r = b.reset(lam)
    ou, orr = exact.reset(Q, 1.0, lam, variant)
    assert_same(u, ou); assert_same(r, orr)
    assert_same(b.resnorm[:n], np.abs(orr).max(axis=1), "resnorm after reset")
    rinit, niter = orr.copy(), np.zeros(n, np.int32)
    A = 0 if prec else num_actions(M, prec_type)
    Qd = fixed_preconditioner(prec, M, Q) if prec else None
    alive = np.ones(n, bool)
    for s in range(steps):
        if prec:
            act = None
        elif prec_type == "diag" and mode == "good" and M in (3, 5, 7):
            act = 2 * (np.diag(fixed_preconditioner("min", M))[None] + rng.uniform(-0.03, 0.03, (n, M))) - 1
        elif prec_type == "diag":
            act = rng.uniform(-1, 1, (n, A))
        else:
            act = rng.uniform(0, 0.5, (n, A))
        out = b.step(act)
        o = exact.step(kind, Q, 1.0, lam, ou, orr, niter, rinit, act, prec_type="fixed" if prec else prec_type,
                       Qd_fixed=Qd, do_scale=(prec_type == "diag"), reward_strategy=strategy, variant=variant)
        assert_same(out["u"][alive], ou[alive], f"step {s} u"); assert_same(out["r"][alive], orr[alive], f"step {s} r")
        assert np.array_equal(out["niter"][alive], niter[alive]), f"step {s} niter"
        assert_same(out["residual"][alive], o["resnorm"][alive], f"step {s} residual")
        assert np.array_equal(out["err"][alive], o["err"][alive])
        assert_reward_close(out["reward"][alive], o["reward"][alive])
        if kind == "sdc-v1":
            assert np.array_equal(out["done"][alive], o["done"][alive])
            alive &= ~o["done"]
        else:
            assert np.array_equal(out["conv"][alive], o["done"][alive])
    return niter


@pytest.mark.parametrize("M", [3, 5, 7, 9])
def test_v0_diag_good_and_uniform(M):
    nit = _run("sdc-v0", M, 3000, mode="good", seed=M)
    if M != 9:
        assert (nit < 50).any()
    _run("sdc-v0", M, 1500, mode="uniform", seed=50 + M)


def test_v0_real_lambda_ties_and_variant1():
    _run("sdc-v0", 5, 1500, mode="good", seed=3, im_int=(0, 0))
    _run("sdc-v0", 5, 1500, mode="good", seed=4, variant=1)
    _run("sdc-v0", 3, 1500, mode="good", seed=5, variant=1)


@pytest.mark.parametrize("prec", ["LU", "min", "EE"])
def test_v0_fixed(prec):
    _run("sdc-v0", 5, 1000, prec=prec, seed=7)


def test_v0_lower_tri_and_v1_rollout():
    _run("sdc-v0", 5, 600, prec_type="lower_tri", seed=8)
    _run("sdc-v1", 5, 300, mode="good", steps=50, strategy="residual_change", seed=9)
    _run("sdc-v1", 7, 200, prec="LU", steps=30, strategy="residual_change", seed=10)


def test_philox_draws_curriculum_and_fused_autoreset_on_host():
    """kernel templates on the host: lambda draws equal the numpy restatement (incl. the np.interp curriculum of
    sdc_env.py:287-292), and the fused auto-reset leaves the reset state of the next lambda + terminal planes."""
    from sdc_gym_b200 import rng as host_rng
    n, M = 300, 5
    Q = collocation_matrix(M)
    d = host_shim.make_desc("sdc-v0", M, seed=17, env_offset=1000, autoreset=True, curriculum=(2, 6))
    b = host_shim.ShimBatch(d, n)
    rng = np.random.default_rng(0)
    for ep in range(1, 5):
        u, r = b.reset()
        lo = float(np.interp(ep, [2, 6], [0, -100]))
        lam = host_rng.lambda_stream(17, 1000 + np.arange(n), ep - 1, (-100, 0), (-10, 0), re_lo_override=lo)
        assert_same(b.lam[0, :n] + 1j * b.lam[1, :n], lam, f"draw {ep}")
        ou, orr = exact.reset(Q, 1.0, lam)
        assert_same(u, ou); assert_same(r, orr)
        assert np.all(b.episodes[:n] == ep)
    # one fused step: terminal planes hold the solve, S the next episode
    act = 2 * (np.diag(fixed_preconditioner("min", M))[None] + rng.uniform(-0.03, 0.03, (n, M))) - 1
    out = b.step(act)
    nit = np.zeros(n, np.int32)
    o = exact.step("sdc-v0", Q, 1.0, lam, ou, orr, nit, orr.copy(), act)
    assert_same(out["term_u"], ou); assert_same(out["term_r"], orr)
    assert np.array_equal(out["niter"], nit) and out["done"].all()
    assert_same(out["lam"], lam, "info lam = finished lambda")
    lo = float(np.interp(5, [2, 6], [0, -100]))
    lam2 = host_rng.lambda_stream(17, 1000 + np.arange(n), 4, (-100, 0), (-10, 0), re_lo_override=lo)
    assert_same(b.lam[0, :n] + 1j * b.lam[1, :n], lam2)
    nu, nr = exact.reset(Q, 1.0, lam2)
    assert_same(out["u"], nu); assert_same(out["r"], nr)
    assert np.all(b.episodes[:n] == 5) and np.all(b.niter[:n] == 0)
    assert_same(b.resnorm[:n], np.abs(nr).max(axis=1))


def test_shared_memory_formulation_of_large_dense_kernels():
    """HOLD 5 (inverse work matrix, Pinv and C in the complex side store): same bits as the oracle"""
    _run("sdc-v0", 8, 200, prec_type="lower_tri", seed=21, entry="shim_step_hold5")
    _run("sdc-v0", 9, 100, prec="LU", seed=22, entry="shim_step_hold5")
    _run("sdc-v1", 8, 100, prec_type="strictly_lower_tri", steps=10, seed=23, entry="shim_step_hold5")


def test_spectral_radius_gradient_against_eigenvector_formula_and_finite_differences():
    """host build of the gradient template: analytic reference from scipy's left/right eigenvectors (1e-10 per
    entry; tests/test_loss_reference_host.py pins both against a 40-digit reference) and central finite differences
    (1e-5)"""
    import ctypes
    import scipy.linalg
    from sdc_gym_b200 import _lib
    from sdc_gym_b200.precond import qdmat_from_output
    L = host_shim.shim()
    L.shim_spectral_radius_grad.argtypes = [ctypes.POINTER(_lib.RhoDesc), ctypes.c_int64] + [ctypes.c_void_p] * 4
    rng = np.random.default_rng(0)

    def K_of(Q, lam, Qd):
        M = Q.shape[0]
        return lam * np.linalg.inv(np.eye(M) - lam * Qd) @ (Q - Qd)

    for M in (3, 5, 7):
        Q = collocation_matrix(M)
        for pt, hi in (("diag", 0.4), ("lower_diag", 0.4), ("lower_tri", 0.3), ("strictly_lower_tri", 0.08)):
            A, n = num_actions(M, pt), 24
            lam = rng.uniform(-100, 0, n) + 1j * rng.uniform(-10, 0, n)
            qd = rng.uniform(0.02, hi, (n, A)) + 1j * rng.uniform(-0.05, 0.05, (n, A))
            d = _lib.RhoDesc()
            d.M, d.prec_type, d.dt, d.qd_is_complex = M, _lib.PREC_TYPES[pt], 1.0, 1
            for k, v in enumerate(Q.reshape(-1)):
                d.Q[k] = v
            rho, g = np.zeros(n), np.zeros((n, A), np.complex128)
            assert L.shim_spectral_radius_grad(ctypes.byref(d), n, lam.ctypes.data, qd.ctypes.data, rho.ctypes.data,
                                               g.ctypes.data) == 0
            for i in range(n):
                Qd = qdmat_from_output(qd[i], M, pt)
                K = K_of(Q, lam[i], Qd)
                w, vl, vr = scipy.linalg.eig(K, left=True, right=True)
                k = int(np.argmax(abs(w)))
                mu, x, y = w[k], vr[:, k], vl[:, k]
                assert abs(rho[i] - abs(mu)) <= 1e-10 * abs(mu)
                P = np.eye(M) - lam[i] * Qd
                wv = np.linalg.solve(P.conj().T, y)
                full = np.conj(mu) / abs(mu) * lam[i] * (mu - 1) * np.outer(np.conj(wv), x) / (np.conj(y) @ x)
                ref = np.array([full[r, c] for r in range(M) for c in range(M)
                                if qdmat_from_output(np.arange(1, A + 1), M, pt)[r, c] != 0])
                assert np.allclose(g[i], ref, rtol=1e-10, atol=1e-12 * abs(ref).max()), (M, pt, i)
            # finite differences on one sample
            i, h = 0, 1e-6
            for k in range(A):
                for dirc in (1.0, 1j):
                    qp, qm = qd[i].copy(), qd[i].copy()
                    qp[k] += h * dirc
                    qm[k] -= h * dirc
                    fp = max(abs(np.linalg.eigvals(K_of(Q, lam[i], qdmat_from_output(qp, M, pt)))))
                    fm = max(abs(np.linalg.eigvals(K_of(Q, lam[i], qdmat_from_output(qm, M, pt)))))
                    assert abs((fp - fm) / (2 * h) - (g[i, k] * dirc).real) <= 1e-4 * max(1.0, abs(g[i]).max())


@pytest.mark.parametrize("M", [2, 4, 6, 8])
def test_even_M_on_host(M):
    _run("sdc-v0", M, 400, mode="uniform", seed=70 + M)
    _run("sdc-v0", M, 200, prec="LU", seed=71 + M)
    _run("sdc-v0", M, 200, prec_type="lower_tri", seed=72 + M)
    _run("sdc-v1", M, 100, mode="uniform", steps=12, strategy="residual_change", seed=73 + M)


def test_pinv_in_side_store_formulation():
    """HOLD 9 (M = 8, 9 dense): LU work matrix, then Pinv, in the side store; C re-derived"""
    _run("sdc-v0", 9, 150, prec_type="lower_tri", seed=31, entry="shim_step_hold9")
    _run("sdc-v0", 8, 150, prec="LU", seed=32, entry="shim_step_hold9")
    _run("sdc-v1", 9, 80, prec_type="strictly_lower_tri", steps=10, seed=33, entry="shim_step_hold9")


@pytest.mark.parametrize("M", [3, 5, 7, 9])
def test_spectral_radius_template_against_lapack_incl_singular_iteration_matrices(M):
    """host build of rho_one (csrc/specrad.cuh): Householder-Hessenberg + shifted QR with real-cosine rotations and
    the unshifted first step for numerically singular matrices (MIN, near-MIN, LU make Q - Qd (nearly) singular),
    against numpy's zgeev: 1e-10 relative (dp_playground.py:216-228, sdc_env.py:421-425)."""
    import ctypes
    from sdc_gym_b200 import _lib
    from sdc_gym_b200.precond import fixed_preconditioner, qdmat_from_output
    L = host_shim.shim()
    rng = np.random.default_rng(100 + M)
    Q = collocation_matrix(M)

    def check(prec_type, qd, Qds, lam, fixed=None):
        n = lam.shape[0]
        d = _lib.RhoDesc()
        d.M, d.prec_type, d.dt = M, _lib.PREC_TYPES[prec_type], 1.0
        d.qd_is_complex = int(qd is not None and np.iscomplexobj(qd))
        for k, v in enumerate(Q.reshape(-1)):
            d.Q[k] = v
        if fixed is not None:
            for k, v in enumerate(np.asarray(fixed, dtype=np.float64).reshape(-1)):
                d.Qd_fixed[k] = v
        rho = np.zeros(n)
        qd_ptr = None if qd is None else np.ascontiguousarray(qd).ctypes.data
        keep = None if qd is None else np.ascontiguousarray(qd)
        assert L.shim_spectral_radius(ctypes.byref(d), n, lam.ctypes.data, None if keep is None else keep.ctypes.data,
                                      rho.ctypes.data) == 0
        for i in range(n):
            K = lam[i] * np.linalg.inv(np.eye(M) - lam[i] * Qds[i]) @ (Q - Qds[i])
            ref = max(abs(np.linalg.eigvals(K)))
            assert abs(rho[i] - ref) <= 1e-10 * ref + 1e-14, (M, prec_type, i, rho[i], ref)

    n = 60
    lam = rng.uniform(-100, 0, n) + 1j * rng.uniform(-10, 0, n)
    lam[0] = 0.0
    # fixed preconditioners: MIN (M = 3, 5, 7) and LU give numerically singular Q - Qd
    for prec in ("min", "LU", "EE", "zeros"):
        Qd = fixed_preconditioner(prec, M, Q)
        check("fixed", None, [Qd] * n, lam, fixed=Qd)
    # learned diagonals next to MIN (nearly singular) and generic ones, real and complex
    base = np.diag(fixed_preconditioner("min", M))
    near = base[None] + rng.uniform(-1e-4, 1e-4, (n, M))
    check("diag", near, [np.diag(x) for x in near], lam)
    gen = rng.uniform(0.02, 0.5, (n, M)) + 1j * rng.uniform(-0.05, 0.05, (n, M))
    check("diag", gen, [np.diag(x) for x in gen], lam)
    A = num_actions(M, "lower_tri")
    tri = rng.uniform(0.0, 0.3, (n, A))
    check("lower_tri", tri, [qdmat_from_output(x, M, "lower_tri") for x in tri], lam)

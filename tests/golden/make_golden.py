"""Generates tests/golden/sdc_golden_*.npz by running the UNMODIFIED reference env
(/root/reference/sdc_gym/envs/sdc_env.py, loaded through oracle/ref_loader.py) on seeded inputs.

Run in the build container only (the reference does not exist on the GPU box):

    OPENBLAS_NUM_THREADS=1 python tests/golden/make_golden.py

Every case stores its inputs (M, Q, dt, lambda, actions, constructor kwargs) and the reference outputs per
step (u, r, info['residual'], info['niter'], reward, done).  The non-diagonal *learned* preconditioners
(`lower_diag`, `lower_tri`, `strictly_lower_tri`) have no env path in the reference; for them the reference
env class is subclassed overriding ONLY `_get_prec` with the `get_qdmat` layout of dp_playground.py:194-207
(SURVEY.md 8c) - sweep, inverse, norms, rewards and control flow stay the reference's.

The vectors are specific to the numpy/OpenBLAS build that produced them (numpy 2.3.5, OpenBLAS 0.3.30,
SkylakeX core - recorded in the manifest); tests replay them with blas_variant = SkylakeX.
"""
from __future__ import annotations

import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, REPO)

from oracle import ref_loader  # noqa: E402
from sdc_gym_b200.collocation import collocation_matrix  # noqa: E402
from sdc_gym_b200.precond import num_actions  # noqa: E402

MAX_ITERS = 50


def subclass_with_layout(cls, prec_type):
    class Sub(cls):
        def _get_prec(self, scaled_action):
            M = self.M
            out = np.asarray(scaled_action)
            if self.action_space.dtype in (np.float32, np.complex64):
                # use_doubles=False: same storage rule as the reference's own diagonal branch (sdc_env.py:138-140)
                out = out.astype(self.action_space.dtype)
            if prec_type == "lower_diag":
                return np.diag(out, k=-1)
            Qd = np.zeros((M, M), dtype=out.dtype)
            if prec_type == "lower_tri":
                Qd[np.tril_indices(M)] = out
            else:
                Qd[np.tril_indices(M, k=-1)] = out
            return Qd

    return Sub


MIN_DIAG = {
    3: [0.3203856825077055, 0.1399680686269595, 0.3716708461097372],
    5: [0.2818591930905709, 0.2011358490453793, 0.06274536689514164, 0.11790265267514095, 0.1571629578515223],
    7: [0.15223871397682717, 0.12625448001038536, 0.08210714764924298, 0.03994434742760019,
        0.1052662547386142, 0.14075805578834127, 0.15636085758812895],
}


def run_case(name, kind, M, n, rng, *, prec=None, prec_type="diag", dt=1.0, restol=1e-10, cplx=False, do_scale=True,
             strategy="iteration_only", norm_factor=1, action_mode="uniform", collect=False,
             re_int=(-100, 0), im_int=(-10, 0), step_penalty=0.1, residual_weight=0.5, use_doubles=True):
    mod = ref_loader.load_reference_envs()
    cls = mod.SDC_Full_Env if kind == "sdc-v0" else mod.SDC_Step_Env
    if prec is None and prec_type != "diag":
        cls = subclass_with_layout(cls, prec_type)
    A = num_actions(M, prec_type) if prec is None else 0
    steps_max = 1 if kind == "sdc-v0" else MAX_ITERS
    Q = collocation_matrix(M)
    lam = rng.uniform(re_int[0], re_int[1], n) + 1j * rng.uniform(im_int[0], im_int[1], n)
    act_dtype = np.complex128 if cplx else np.float64
    actions = np.zeros((n, steps_max, max(A, 1)), act_dtype)
    U = np.zeros((n, steps_max, M), np.complex128)
    R = np.zeros((n, steps_max, M), np.complex128)
    u0 = np.zeros((n, M), np.complex128)
    r0 = np.zeros((n, M), np.complex128)
    res = np.zeros((n, steps_max))
    nit = np.zeros((n, steps_max), np.int32)
    rew = np.zeros((n, steps_max))
    done = np.zeros((n, steps_max), bool)
    nsteps = np.zeros(n, np.int32)
    old_states = np.zeros((n, 2 * M, MAX_ITERS), np.complex128) if collect else None
    for e in range(n):
        env = cls(M=M, dt=dt, restol=restol, prec=prec, lambda_real_interval=list(re_int),
                  lambda_imag_interval=list(im_int), reward_iteration_only=None, reward_strategy=strategy,
                  norm_factor=norm_factor, do_scale=do_scale, free_action_space=cplx, collect_states=collect,
                  step_penalty=step_penalty, residual_weight=residual_weight, use_doubles=use_doubles)
        # NB: env.Q stays the reference's own (non-contiguous) view of Qmat.  Handing it a C-contiguous copy
        # would let `scipy.linalg.lu(Q.T, overwrite_a=True)` (sdc_env.py:142-143) overwrite Q in place.
        assert np.array_equal(env.Q, Q)
        env.reset()
        ref_loader.inject_lambda(env, lam[e])
        u0[e], r0[e] = env.state[0], env.state[1]
        for s in range(steps_max):
            if A == 0:
                a = None
            elif cplx:
                a = rng.uniform(0, 0.5, A) + 1j * rng.uniform(-0.1, 0.1, A)
            elif action_mode == "good" and prec_type == "diag" and M in MIN_DIAG:
                a = 2 * (np.array(MIN_DIAG[M]) + rng.uniform(-0.02, 0.02, M)) - 1
            elif do_scale:
                a = rng.uniform(-1, 1, A)
            else:
                a = rng.uniform(0, 0.6, A)
            if a is not None:
                if not use_doubles:  # SB3 hands the env actions in the action-space dtype (float32 / complex64)
                    a = a.astype(env.action_space.dtype)
                actions[e, s] = a  # stored as float64 / complex128 (exact)
            _, reward, d, info = env.step(None if a is None else a.copy())
            U[e, s], R[e, s] = env.state[0], env.state[1]
            res[e, s], nit[e, s], rew[e, s], done[e, s] = info["residual"], info["niter"], reward, d
            nsteps[e] = s + 1
            if d:
                break
        if collect:
            old_states[e] = env.old_states
    out = dict(lam=lam, actions=actions, u=U, r=R, u0=u0, r0=r0, residual=res, niter=nit, reward=rew, done=done,
               nsteps=nsteps, Q=Q)
    if collect:
        out["old_states"] = old_states
    meta = dict(name=name, kind=kind, M=M, n=n, prec=prec, prec_type=prec_type if prec is None else "fixed", dt=dt,
                restol=restol, cplx=cplx, do_scale=do_scale, strategy=strategy, norm_factor=norm_factor,
                collect=collect, step_penalty=step_penalty, residual_weight=residual_weight,
                use_doubles=use_doubles)
    return meta, out


def main():
    rng = np.random.default_rng(20261018)
    cases = []
    arrays = {}

    def add(name, *a, **k):
        meta, out = run_case(name, *a, **k)
        cases.append(meta)
        for key, v in out.items():
            arrays[f"{name}/{key}"] = v

    for kind, nn in (("sdc-v0", 12), ("sdc-v1", 4)):
        tag = kind[-2:]
        for M in (3, 5, 7, 9):
            add(f"{tag}_diag_M{M}_uniform", kind, M, nn, rng)
            if M in MIN_DIAG:
                add(f"{tag}_diag_M{M}_good", kind, M, nn, rng, action_mode="good")
            for prec in ("LU", "min", "EE", "zeros"):
                add(f"{tag}_{prec}_M{M}", kind, M, max(3, nn // 3), rng, prec=prec)
            for pt in ("lower_diag", "lower_tri", "strictly_lower_tri"):
                add(f"{tag}_{pt}_M{M}", kind, M, max(3, nn // 3), rng, prec_type=pt, do_scale=False)
            add(f"{tag}_lower_tri_cplx_M{M}", kind, M, 3, rng, prec_type="lower_tri", do_scale=False, cplx=True)
        add(f"{tag}_diag_cplx_M5", kind, 5, max(3, nn // 2), rng, cplx=True, do_scale=False)
        add(f"{tag}_diag_cplx_M7_dt025", kind, 7, 3, rng, cplx=True, do_scale=False, dt=0.25)
        add(f"{tag}_diag_M5_dt05", kind, 5, max(3, nn // 2), rng, dt=0.5, action_mode="good")
        add(f"{tag}_diag_M5_realonly", kind, 5, max(3, nn // 2), rng, im_int=(0, 0), action_mode="good")
        for strat in ("iteration_only", "residual_change", "gauss_kernel", "fast_convergence",
                      "smooth_fast_convergence", "smoother_fast_convergence"):
            add(f"{tag}_diag_M5_{strat}", kind, 5, max(3, nn // 2), rng, strategy=strat, action_mode="good",
                step_penalty=0.25, residual_weight=0.8)
        add(f"{tag}_diag_M5_residual_change_nf", kind, 5, max(3, nn // 2), rng, strategy="residual_change",
            action_mode="good", norm_factor=3.7)
        add(f"{tag}_diag_M5_collect", kind, 5, 3, rng, action_mode="good", collect=True)
        add(f"{tag}_LU_M5_collect", kind, 5, 2, rng, prec="LU", collect=True)

    # use_doubles=False (float32 / complex64 action space, utils/utils.py:279-280 for SAC): appended with their own
    # generator so the cases above keep their bits
    rng = np.random.default_rng(20261019)
    for kind, nn in (("sdc-v0", 12), ("sdc-v1", 4)):
        tag = kind[-2:]
        for M in (3, 5, 9):
            add(f"{tag}_diag_M{M}_f32", kind, M, nn, rng, use_doubles=False)
        add(f"{tag}_diag_M5_good_f32", kind, 5, nn, rng, use_doubles=False, action_mode="good")
        add(f"{tag}_diag_M5_noscale_f32", kind, 5, 4, rng, use_doubles=False, do_scale=False)
        add(f"{tag}_diag_cplx_M5_c64", kind, 5, 4, rng, use_doubles=False, cplx=True, do_scale=False)
        add(f"{tag}_lower_tri_M5_f32", kind, 5, 4, rng, use_doubles=False, prec_type="lower_tri", do_scale=False)
        add(f"{tag}_lower_tri_M9_f32", kind, 9, 3, rng, use_doubles=False, prec_type="lower_tri", do_scale=False)
        add(f"{tag}_strictly_lower_tri_cplx_M7_c64", kind, 7, 3, rng, use_doubles=False, cplx=True,
            prec_type="strictly_lower_tri", do_scale=False)

    from threadpoolctl import threadpool_info
    blas = [i for i in threadpool_info() if i.get("internal_api") == "openblas"]
    manifest = dict(
        generator="tests/golden/make_golden.py", reference="pancetta/sdc-gym sdc_gym/envs/sdc_env.py (unmodified, stub imports)",
        numpy=np.__version__, openblas=blas[0]["version"] if blas else None,
        openblas_core=blas[0]["architecture"] if blas else None, blas_variant=0, cases=cases)
    write_golden(manifest, arrays)
    print(f"{len(cases)} cases, {sum(v.nbytes for v in arrays.values()) / 1e6:.2f} MB raw")


SHARDS = 4  # the cases go round-robin into this many compressed files, each well under 1 MB


def write_golden(manifest, arrays):
    """sdc_golden_<k>.npz (arrays keyed '<case>/<array>') + sdc_golden.json (manifest; 'file' names each case's npz)"""
    for i, case in enumerate(manifest["cases"]):
        case["file"] = f"sdc_golden_{i % SHARDS}.npz"
    for k in range(SHARDS):
        fname = f"sdc_golden_{k}.npz"
        names = {c["name"] for c in manifest["cases"] if c["file"] == fname}
        np.savez_compressed(os.path.join(HERE, fname), **{key: v for key, v in arrays.items()
                                                          if key.split("/", 1)[0] in names})
    with open(os.path.join(HERE, "sdc_golden.json"), "w") as f:
        json.dump(manifest, f, indent=1)


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""Search a diagonal Q_delta for few sdc-v0 iterations directly, with a derivative-free (mu/mu, lambda) evolution
strategy: the iteration count is what the reference judges a Q_delta by (`test_model`), and it has no gradient.

Objective of a row: the mean over every node of the N x N lambda grid of the box [-100, 0] x [-10, 0] of its sweep
count, an err node or a node that runs out of sweeps counted as 50 (defined here, not in the library).  Each generation
evaluates all lambda candidates in one launch (`IterationCounts.population_grid_summary`).  The search starts from
MIN's diagonal; for comparison a row trained on the mean spectral radius over the same grid (from 0.5, Adam) is
judged too.  Whether the search beats MIN is not known in advance: the script reports what it finds.

    python examples/search_niter.py --M 5 --grid 256 --generations 40 --lam 32
"""
import argparse
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from sdc_gym_b200 import fixed_preconditioner  # noqa: E402
from sdc_gym_b200.iterations import IterationCounts  # noqa: E402

BOX = ((-100.0, 0.0), (-10.0, 0.0))
FAIL_SWEEPS = 50  # what an err node or a node out of sweeps counts as


def objective(hist, max_iters):
    """mean sweep count per node of each histogram row (P, max_iters + 3), failures counted as FAIL_SWEEPS"""
    h = np.asarray(hist, np.float64)
    k = np.arange(max_iters + 1)
    total = h[:, : max_iters + 1] @ k + FAIL_SWEEPS * (h[:, max_iters + 1] + h[:, max_iters + 2])
    return total / h.sum(1)


def summary_line(name, mean_niter, success_rate):
    return f"{name:<3} -- Mean number of iterations and success rate: {mean_niter:4.2f}, {success_rate * 100} %"


def rho_trained_row(M, grid, steps, lr=0.02):
    import torch

    from sdc_gym_b200.loss import SpectralRadiusLoss

    loss_fn = SpectralRadiusLoss(M, 1.0, "diag")
    theta = torch.full((M,), 0.5, dtype=torch.float64, device="cuda", requires_grad=True)
    opt = torch.optim.Adam([theta], lr=lr)
    for _ in range(steps):
        opt.zero_grad()
        loss_fn.grid_differentiable(grid, grid, *BOX, theta).backward()
        opt.step()
    return theta.detach().cpu().numpy()


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--M", type=int, default=5)
    ap.add_argument("--grid", type=int, default=256, help="N: the N x N lambda grid of the box")
    ap.add_argument("--generations", type=int, default=40)
    ap.add_argument("--lam", type=int, default=32, help="candidates per generation")
    ap.add_argument("--mu", type=int, default=0, help="parents per generation (default lam / 4)")
    ap.add_argument("--sigma", type=float, default=0.03, help="initial step size")
    ap.add_argument("--rho-steps", type=int, default=200, help="Adam steps of the rho-trained comparison row")
    ap.add_argument("--seed", type=int, default=0)
    args = ap.parse_args(argv)
    M, n = args.M, args.grid
    mu = args.mu or max(1, args.lam // 4)
    rng = np.random.default_rng(args.seed)
    ev = IterationCounts(M, 1.0, 1e-10, "diag")

    mean = np.diag(fixed_preconditioner("min", M)).astype(np.float64)
    sigma = args.sigma
    best, best_f = mean.copy(), float(objective(ev.population_grid_summary(n, n, *BOX, mean[None]).hist,
                                               ev.max_iters)[0])
    f_min = best_f
    print(f"generation   0  objective of MIN {f_min:.4f}")
    for g in range(1, args.generations + 1):
        cand = np.clip(mean + sigma * rng.standard_normal((args.lam, M)), 0.0, 1.0)
        f = objective(ev.population_grid_summary(n, n, *BOX, cand).hist, ev.max_iters)
        order = np.argsort(f, kind="stable")
        mean = cand[order[:mu]].mean(0)
        # a simple success rule for the step size: shrink when the generation's best does not improve on the best so far
        if f[order[0]] < best_f:
            best, best_f = cand[order[0]].copy(), float(f[order[0]])
            sigma *= 1.1
        else:
            sigma *= 0.85
        print(f"generation {g:3d}  best {f[order[0]]:.4f}  best so far {best_f:.4f}  sigma {sigma:.4f}")

    rho_row = rho_trained_row(M, min(n, 256), args.rho_steps)
    s_min = IterationCounts(M, 1.0, 1e-10, prec="min").grid_summary(n, n, *BOX)
    pop = ev.population_grid_summary(n, n, *BOX, np.stack([rho_row, best]))
    print(summary_line("MIN", s_min.mean_niter, s_min.success_rate))
    print(summary_line("RHO", pop.mean_niter[0], pop.success_rate[0]))
    print(summary_line("ES", pop.mean_niter[1], pop.success_rate[1]))
    f_rho, f_es = objective(pop.hist, ev.max_iters)
    print(f"objective (mean sweeps, failures as {FAIL_SWEEPS}): MIN {f_min:.4f}  RHO {f_rho:.4f}  ES {f_es:.4f}")
    print(f"ES diag {best.round(4)}")
    return {"best": best, "objective": {"MIN": f_min, "RHO": float(f_rho), "ES": float(f_es)}, "rho_row": rho_row}


if __name__ == "__main__":
    main()

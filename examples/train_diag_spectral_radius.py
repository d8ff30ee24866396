#!/usr/bin/env python
"""dp_playground in miniature: learn one diagonal Q_delta (the reference's `Params` "model", dp_playground.py:478-560)
by gradient descent on the mean spectral radius over freshly sampled lambdas, or with --grid N over the N x N
lambda grid of the box [-100, 0] x [-10, 0] - forward and backward both run the hand-written kernels
(`SpectralRadiusLoss.differentiable` / `grid_differentiable`), which reduce the gradient of the one shared row on
the device.  With --sweeps K it minimises instead what K sweeps of the iteration achieve,
mean log(||r_K||_inf / ||r_0||_inf) over the sampled lambdas from the envs' reset state, with the gradient taken
through all K sweeps (`ResidualLoss.sweeps_differentiable`); with --sweeps K --grid N it minimises that mean over the
N x N grid, reduced on the device (`ResidualLoss.sweeps_grid_differentiable`).  With --eval-grid N it then judges the
trained row as the reference does, by sdc-v0 iteration counts and success rate, over the N x N grid next to MIN's
(`IterationCounts.grid_summary`).

    python examples/train_diag_spectral_radius.py --M 5 --steps 300 --batch 65536
    python examples/train_diag_spectral_radius.py --M 5 --steps 200 --grid 256
    python examples/train_diag_spectral_radius.py --M 5 --steps 200 --sweeps 5
    python examples/train_diag_spectral_radius.py --M 5 --steps 200 --sweeps 5 --grid 256
    python examples/train_diag_spectral_radius.py --M 5 --steps 200 --grid 256 --eval-grid 512
    python examples/train_diag_spectral_radius.py --M 5 --steps 200 --grid 256 --starts 16 --eval-grid 512

With --starts P it trains P seeded random diagonals together (multi-start: the mean rho is not convex in the row),
one Adam over the (P, M) tensor - Adam is elementwise, so the rows train independently - with the losses of all P
rows in one launch per step (`SpectralRadiusLoss.population_differentiable` / `population_grid_differentiable`), and
prints the best row; --eval-grid then judges every trained row in one launch (`IterationCounts.population_grid_summary`).
"""
import argparse
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from sdc_gym_b200.collocation import collocation_matrix  # noqa: E402
from sdc_gym_b200.loss import ResidualLoss, SpectralRadiusLoss  # noqa: E402


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--M", type=int, default=5)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--batch", type=int, default=65536)
    ap.add_argument("--lr", type=float, default=0.02)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--grid", type=int, default=0, help="train on the N x N lambda grid instead of sampled lambdas")
    ap.add_argument("--sweeps", type=int, default=0,
                    help="K > 0: minimise mean log(||r_K|| / ||r_0||) after K sweeps instead of the mean rho")
    ap.add_argument("--eval-grid", type=int, default=0,
                    help="N > 0: after training, print the sdc-v0 iteration counts of the row and of MIN on the N x N grid")
    ap.add_argument("--starts", type=int, default=1, help="P > 1: train P seeded random diagonals together")
    args = ap.parse_args(argv)
    if args.starts > 1:
        if args.sweeps:
            ap.error("--starts trains the spectral-radius loss only: the K-sweep loss has no population form")
        return multi_start(args)
    dev = torch.device("cuda")
    gen = torch.Generator(device=dev)
    gen.manual_seed(args.seed)
    loss_fn = SpectralRadiusLoss(args.M, 1.0, "diag")
    if args.sweeps:
        res_fn = ResidualLoss(args.M, 1.0, "diag")
        q1 = float(abs(collocation_matrix(args.M).sum(axis=1)).max())  # ||r_0|| = |lam dt| max_i |(Q 1)_i|
    theta = torch.full((args.M,), 0.5, dtype=torch.float64, device=dev, requires_grad=True)
    opt = torch.optim.Adam([theta], lr=args.lr)
    history = []
    for step in range(args.steps):
        opt.zero_grad()
        if args.sweeps and args.grid:
            loss = res_fn.sweeps_grid_differentiable(args.grid, args.grid, (-100.0, 0.0), (-10.0, 0.0), theta,
                                                     args.sweeps, reduction="log_ratio")
        elif args.sweeps:
            lam = torch.complex(torch.rand(args.batch, dtype=torch.float64, device=dev, generator=gen) * -100.0,
                                torch.zeros(args.batch, dtype=torch.float64, device=dev))
            n = res_fn.sweeps_differentiable(lam, theta, args.sweeps)
            loss = torch.log(n / (lam.abs() * q1)).mean()
        elif args.grid:
            loss = loss_fn.grid_differentiable(args.grid, args.grid, (-100.0, 0.0), (-10.0, 0.0), theta)
        else:
            lam = torch.complex(torch.rand(args.batch, dtype=torch.float64, device=dev, generator=gen) * -100.0,
                                torch.zeros(args.batch, dtype=torch.float64, device=dev))
            loss = loss_fn.differentiable(lam, theta)
        loss.backward()
        opt.step()
        history.append(float(loss.detach()))
        if step % 50 == 0 or step == args.steps - 1:
            what = f"mean log(|r_{args.sweeps}|/|r_0|)" if args.sweeps else "mean rho"
            print(f"step {step:4d}  {what} {history[-1]:.6f}  diag {theta.detach().cpu().numpy().round(4)}")
    if args.eval_grid:
        # the reference's judgement of the trained row: sdc-v0 iteration counts and success rate, here over every
        # lambda of the N x N grid, next to MIN's
        from sdc_gym_b200.iterations import IterationCounts

        n, box = args.eval_grid, ((-100.0, 0.0), (-10.0, 0.0))
        for name, ev, row in (("MIN", IterationCounts(args.M, 1.0, 1e-10, prec="min"), None),
                              ("RL", IterationCounts(args.M, 1.0, 1e-10, "diag"), theta.detach())):
            s = ev.grid_summary(n, n, *box, row)
            print(f"{name:<3} -- Mean number of iterations and success rate: {s.mean_niter:4.2f}, "
                  f"{s.success_rate * 100} %")
    return history, theta.detach().cpu().numpy()


def _summary_line(name, mean_niter, success_rate):
    return f"{name} -- Mean number of iterations and success rate: {mean_niter:4.2f}, {success_rate * 100} %"


def multi_start(args):
    dev = torch.device("cuda")
    gen = torch.Generator(device=dev)
    gen.manual_seed(args.seed)
    box = ((-100.0, 0.0), (-10.0, 0.0))
    loss_fn = SpectralRadiusLoss(args.M, 1.0, "diag")
    theta = torch.rand((args.starts, args.M), dtype=torch.float64, device=dev, generator=gen)
    theta.requires_grad_(True)
    opt = torch.optim.Adam([theta], lr=args.lr)
    history = []
    for step in range(args.steps):
        opt.zero_grad()
        if args.grid:
            losses = loss_fn.population_grid_differentiable(args.grid, args.grid, *box, theta)
        else:
            lam = torch.complex(torch.rand(args.batch, dtype=torch.float64, device=dev, generator=gen) * -100.0,
                                torch.zeros(args.batch, dtype=torch.float64, device=dev))
            losses = loss_fn.population_differentiable(lam, theta)
        losses.sum().backward()
        opt.step()
        history.append(losses.detach().cpu().numpy())
        if step % 50 == 0 or step == args.steps - 1:
            print(f"step {step:4d}  mean rho best {history[-1].min():.6f}  worst {history[-1].max():.6f}")
    rows = theta.detach()
    # the last step's losses belong to the rows before its update: judge the trained rows themselves
    final = (loss_fn.population_grid_value_and_grad(args.grid, args.grid, *box, rows)[0] if args.grid else
             loss_fn.population_value_and_grad(lam, rows)[0]).cpu().numpy()
    best = int(final.argmin())
    print(f"best start {best}: mean rho {final[best]:.6f}  diag {rows[best].cpu().numpy().round(4)}")
    if args.eval_grid:
        from sdc_gym_b200.iterations import IterationCounts

        n = args.eval_grid
        s = IterationCounts(args.M, 1.0, 1e-10, prec="min").grid_summary(n, n, *box)
        print(_summary_line("MIN", s.mean_niter, s.success_rate))
        pop = IterationCounts(args.M, 1.0, 1e-10, "diag").population_grid_summary(n, n, *box, rows)
        for p in range(len(pop)):
            print(_summary_line(f"start {p}", pop.mean_niter[p], pop.success_rate[p]))
    return history, rows.cpu().numpy()


if __name__ == "__main__":
    main()

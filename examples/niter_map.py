#!/usr/bin/env python
"""Iteration counts of the sdc-v0 full solve over a lambda grid, counted on the device (`IterationCounts`): the
reference's evaluation (`test_model`, rl_playground.py:147-156) for LU, MIN and a given diagonal, with every lambda of
an N x N grid of the box instead of drawn lambdas.  Optionally saves each niter map (N, N) as .npy.

    python examples/niter_map.py --M 5 --grid 512 --re -100 0 --im -10 0
    python examples/niter_map.py --M 5 --grid 512 --diag 0.28 0.2 0.06 0.12 0.16 --save /tmp/niter

Prints the reference's summary line per preconditioner:
    LU  -- Mean number of iterations and success rate: 17.13, 100.0 %
"""
import argparse
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from sdc_gym_b200 import fixed_preconditioner  # noqa: E402
from sdc_gym_b200.iterations import IterationCounts  # noqa: E402


def summary_line(name, s):
    return (f"{name:<3} -- Mean number of iterations and success rate: {s.mean_niter:4.2f}, "
            f"{s.success_rate * 100} %")


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--M", type=int, default=5)
    ap.add_argument("--grid", type=int, default=512, help="N: the N x N grid of the box, end points included")
    ap.add_argument("--re", type=float, nargs=2, default=(-100.0, 0.0))
    ap.add_argument("--im", type=float, nargs=2, default=(-10.0, 0.0))
    ap.add_argument("--restol", type=float, default=1e-10)
    ap.add_argument("--diag", type=float, nargs="+", default=None,
                    help="a diagonal Q_delta to evaluate next to LU and MIN (default: the MIN diagonal)")
    ap.add_argument("--save", default=None, help="prefix: write <prefix>_<name>.npy, the (N, N) niter map")
    args = ap.parse_args(argv)
    n = args.grid
    diag = np.asarray(args.diag if args.diag else np.diag(fixed_preconditioner("min", args.M)), np.float64)
    if diag.shape != (args.M,):
        ap.error(f"--diag needs {args.M} values")
    runs = [("LU", IterationCounts(args.M, 1.0, args.restol, prec="LU"), None),
            ("MIN", IterationCounts(args.M, 1.0, args.restol, prec="min"), None),
            ("RL", IterationCounts(args.M, 1.0, args.restol, "diag"), diag)]
    out = {}
    for name, ev, row in runs:
        s = ev.grid_summary(n, n, args.re, args.im, row)
        print(summary_line(name, s))
        out[name] = s
        if args.save:
            niter, _, _ = ev.grid(n, n, args.re, args.im, row)
            np.save(f"{args.save}_{name}.npy", niter.cpu().numpy())
    return out


if __name__ == "__main__":
    main()

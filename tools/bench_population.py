"""Population calls against a Python loop of single-row calls, on the device.

    python tools/bench_population.py --out bench_population.jsonl [--budget 20]

For M = 5 ``diag`` and M = 9 ``lower_tri``, grids 256^2, 1024^2 and 4096^2 and P in {1, 8, 64} rows:
  counts  ``IterationCounts.population_grid_summary`` (one launch) against P calls of ``grid_summary``;
  rho     ``SpectralRadiusLoss.population_grid_value_and_grad`` against P calls of ``grid_value_and_grad``.
Each route is timed from the first call to a device synchronise, after a warm-up call of the same shape, best of
--reps; the peak allocation of each route is recorded, and the two routes' results are compared bit for bit in the
same run.  A route whose single-row time times P exceeds --budget seconds is skipped and recorded as skipped.  The
first line records the card name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from sdc_gym_b200 import fixed_preconditioner  # noqa: E402
from sdc_gym_b200.iterations import IterationCounts  # noqa: E402
from sdc_gym_b200.loss import SpectralRadiusLoss  # noqa: E402
from sdc_gym_b200.precond import num_actions  # noqa: E402

BOX = ((-100.0, 0.0), (-10.0, 0.0))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[torch.cuda.current_device()] if q.returncode == 0 else "unknown"


def timed(fn, reps):
    """(best seconds, peak bytes above the start, result) of fn() ended by a device synchronise"""
    fn()  # warm-up
    torch.cuda.synchronize()
    best, peak, out = float("inf"), 0, None
    for _ in range(reps):
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        best = min(best, time.perf_counter() - t0)
        peak = max(peak, torch.cuda.max_memory_allocated() - base)
    return best, peak, out


def rows_for(M, pt, P, rng):
    A = num_actions(M, pt)
    if pt == "diag":
        base = np.diag(fixed_preconditioner("min", M))
        return np.clip(base + rng.normal(0, 0.03, (P, A)), 0, 1)
    return rng.uniform(0.02, 0.3, (P, A))


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--budget", type=float, default=5.0, help="seconds a route may take at most (estimated)")
    ap.add_argument("--trace", default=None,
                    help="file: torch.profiler table of both counts routes at M = 5, 256^2, P = 8 (a run of its own)")
    ap.add_argument("--grids", type=int, nargs="+", default=[256, 1024, 4096])
    ap.add_argument("--pops", type=int, nargs="+", default=[1, 8, 64])
    args = ap.parse_args(argv)
    rng = np.random.default_rng(0)
    if args.trace:
        return trace(args.trace, rng)
    with open(args.out, "w") as f:
        f.write(json.dumps({"card": card(), "torch": torch.__version__}) + "\n")
        for M, pt in ((5, "diag"), (9, "lower_tri")):
            ev = IterationCounts(M, 1.0, 1e-10, pt)
            loss = SpectralRadiusLoss(M, 1.0, pt)
            for n in args.grids:
                one = {}
                for P in args.pops:
                    rows = torch.as_tensor(rows_for(M, pt, P, rng), device="cuda")
                    for what in ("counts", "rho"):
                        rec = dict(what=what, M=M, prec_type=pt, grid=n, P=P)
                        est = one.get(what, 0.0) * P
                        if est > args.budget:
                            rec.update(skipped=f"estimated {est:.1f} s per call of the loop > budget {args.budget} s")
                            f.write(json.dumps(rec) + "\n")
                            f.flush()
                            continue
                        if what == "counts":
                            pop_fn = lambda: ev.population_grid_summary(n, n, *BOX, rows).hist_device  # noqa: E731
                            loop_fn = lambda: [ev.grid_summary(n, n, *BOX, r).hist_device for r in rows]  # noqa: E731
                        else:
                            pop_fn = lambda: loss.population_grid_value_and_grad(n, n, *BOX, rows)  # noqa: E731
                            loop_fn = lambda: [loss.grid_value_and_grad(n, n, *BOX, r) for r in rows]  # noqa: E731
                        t_loop, m_loop, loop = timed(loop_fn, args.reps)
                        t_pop, m_pop, pop = timed(pop_fn, args.reps)
                        if what == "counts":
                            equal = all(torch.equal(pop[p], loop[p]) for p in range(P))
                        else:
                            equal = all(torch.equal(pop[0][p], loop[p][0]) and torch.equal(pop[1][p], loop[p][1])
                                        for p in range(P))
                        if P == 1:
                            one[what] = t_loop
                        rec.update(loop_ms=t_loop * 1e3, population_ms=t_pop * 1e3, speedup=t_loop / t_pop,
                                   loop_peak_bytes=m_loop, population_peak_bytes=m_pop, bits_equal=bool(equal))
                        print(json.dumps(rec), flush=True)
                        f.write(json.dumps(rec) + "\n")
                        f.flush()


def trace(path, rng):
    from torch.profiler import ProfilerActivity, profile

    ev = IterationCounts(5, 1.0, 1e-10, "diag")
    rows = torch.as_tensor(rows_for(5, "diag", 8, rng), device="cuda")
    n = 256
    ev.population_grid_summary(n, n, *BOX, rows).hist_device
    [ev.grid_summary(n, n, *BOX, r) for r in rows]
    torch.cuda.synchronize()
    with open(path, "w") as f:
        f.write(f"# {card()}\n")
        for name, fn in (("loop of 8 single-row calls", lambda: [ev.grid_summary(n, n, *BOX, r) for r in rows]),
                         ("one population call, P = 8", lambda: ev.population_grid_summary(n, n, *BOX, rows))):
            with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
                fn()
                torch.cuda.synchronize()
            f.write(f"## {name}\n")
            f.write(prof.key_averages().table(sort_by="cuda_time_total", row_limit=12) + "\n")
            events = sorted((e for e in prof.events() if e.device_type.name == "CUDA"), key=lambda e: e.time_range.start)
            if events:
                span = events[-1].time_range.end - events[0].time_range.start
                busy = sum(e.time_range.end - e.time_range.start for e in events)
                f.write(f"device span {span:.1f} us, kernels and copies busy {busy:.1f} us\n\n")


if __name__ == "__main__":
    main()

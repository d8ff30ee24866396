"""sdc-v0 iteration-count histogram over an N x N lambda grid: ``IterationCounts.grid_summary`` (lambdas generated on
the device, ``full_solve_counts_kernel``, histogram counted on chip) against the env route a user has without it:
``make("sdc-v0", num_envs=N*N)``, ``reset(lam=host grid)``, ``step_tensor(row expanded to N*N)`` and ``torch.bincount``
of the outcome classes.  Both routes use the same nodes (the host grid is ``grid(..., return_lam=True)`` copied to the
host once) and must give the same histogram.

One JSON object per line: time per evaluation from CUDA events over --reps evaluations after --warmup (the two routes
measured twice, alternating; the env route's time is reset + step + bincount, its construction excluded), and the
increase of ``torch.cuda.max_memory_allocated`` over what was live before (the env route's includes its planes).  The
GPU's name and power limit are read in the same run."""
import argparse, gc, json, os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import sdc_gym_b200
from sdc_gym_b200.iterations import IterationCounts
from sdc_gym_b200.precond import fixed_preconditioner, num_actions

ap = argparse.ArgumentParser()
ap.add_argument("--grids", type=int, nargs="+", default=[1024, 4096])
ap.add_argument("--reps", type=int, default=3)
ap.add_argument("--warmup", type=int, default=1)
ap.add_argument("--out", default=None, help="also append the lines to this file")
args = ap.parse_args()
dev = torch.device("cuda", 0)
RE, IM = (-100.0, 0.0), (-10.0, 0.0)
MIN5 = np.diag(fixed_preconditioner("min", 5))
# (name, M, prec_type, row): the MIN diagonal as a row, a diagonal as a training run leaves it, a lower-triangular row
CASES = [
    ("M5_diag_min_row", 5, "diag", MIN5),
    ("M5_diag_learned", 5, "diag", np.array([0.31, 0.19, 0.09, 0.12, 0.15])),
    ("M5_lower_tri", 5, "lower_tri", None),
    ("M9_diag", 9, "diag", None),
    ("M9_lower_tri", 9, "lower_tri", None),
]


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = ""
    return out or torch.cuda.get_device_name(dev)


def timed(fn):
    for _ in range(args.warmup):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(args.reps):
        out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / args.reps, out


def env_hist(out):
    f = out["flags"]
    conv, err = (f & 2).ne(0), (f & 4).ne(0)
    bins = torch.where(err, 51, torch.where(conv, out["niter"].long(), 52))
    return torch.bincount(bins, minlength=53)


gpu = gpu_info()
rng = np.random.default_rng(0)
lines = []
for name, M, pt, row in CASES:
    if row is None:
        row = rng.uniform(0.02, 0.3, num_actions(M, pt))
    ev = IterationCounts(M, 1.0, 1e-10, pt, device=dev)
    row_t = torch.tensor(row, dtype=torch.float64, device=dev)
    for n in args.grids:
        N = n * n
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats(dev)
        base = torch.cuda.memory_allocated(dev)
        ms_a, s = timed(lambda: ev.grid_summary(n, n, RE, IM, row_t))
        hist_fused = s.hist.copy()
        mem_fused = torch.cuda.max_memory_allocated(dev) - base
        lam_host = ev.grid(n, n, RE, IM, row_t, return_lam=True)[3].reshape(-1).cpu().numpy()
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats(dev)
        base = torch.cuda.memory_allocated(dev)
        env = sdc_gym_b200.make("sdc-v0", num_envs=N, M=M, dt=1.0, restol=1e-10, prec_type=pt, do_scale=False,
                                free_action_space=True, autoreset=False, keep_terminal=False, device=dev)
        rows = row_t.expand(N, -1)

        def env_route():
            env.reset(lam=lam_host)
            return env_hist(env.step_tensor(rows, want_terminal=False))

        ms_b, h = timed(env_route)
        mem_env = torch.cuda.max_memory_allocated(dev) - base
        ms_a2, _ = timed(lambda: ev.grid_summary(n, n, RE, IM, row_t))
        ms_b2, _ = timed(env_route)
        line = json.dumps({
            "gpu": gpu, "case": name, "M": M, "prec_type": pt, "grid": n, "N": N, "reps": args.reps,
            "grid_summary_ms": [round(ms_a, 3), round(ms_a2, 3)],
            "env_route_ms": [round(ms_b, 3), round(ms_b2, 3)],
            "grid_summary_peak_alloc_MB": round(mem_fused / 2**20, 2),
            "env_route_peak_alloc_MB": round(mem_env / 2**20, 2),
            "same_hist": bool(np.array_equal(hist_fused, h.cpu().numpy())),
            "success_rate": s.success_rate, "mean_niter": s.mean_niter,
        })
        print(line, flush=True)
        lines.append(line)
        env.close()
        del env, rows, lam_host
        gc.collect()  # the env holds reference cycles: free its planes before the next case's baseline
        torch.cuda.empty_cache()
if args.out:
    with open(args.out, "a") as f:
        f.write("\n".join(lines) + "\n")

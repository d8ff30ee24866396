"""K-sweep residual loss and its gradient for ONE shared Q_delta row: the fused call that reduces the gradient on the
device (``ResidualLoss.sweeps_shared_value_and_grad`` / ``sweeps_grid_value_and_grad``, ``residual_sweeps_sum_kernel``)
against the per-sample path (``sweeps(with_grad=True)`` on the shared row, then ``torch.sum`` of the norms and of the
gradient) on the same lambdas, from the envs' reset state, reduction 'mean'.  The grid's lambdas for the per-sample
path are formed on the device with the formula of ``grid_lambda``.  Complex rows.

One JSON object per line: call time from CUDA events over --reps calls after warm-up (the two paths measured twice,
alternating), and the increase of ``torch.cuda.max_memory_allocated`` over the inputs for each path; the GPU's name and
power limit are read in the same run."""
import argparse, json, os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from sdc_gym_b200.loss import ResidualLoss
from sdc_gym_b200.precond import num_actions

ap = argparse.ArgumentParser()
ap.add_argument("--B", type=int, default=1 << 20)
ap.add_argument("--grid", type=int, default=2048)
ap.add_argument("--M", type=int, nargs="+", default=[5, 9])
ap.add_argument("--prec-types", nargs="+", default=["diag", "lower_tri"])
ap.add_argument("--K", type=int, nargs="+", default=[5, 50])
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--warmup", type=int, default=1)
args = ap.parse_args()
dev = torch.device("cuda", 0)
RE, IM = (-100.0, 0.0), (-10.0, 0.0)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = ""
    return out or torch.cuda.get_device_name(dev)


def measure(fn):
    """(ms per call over args.reps calls after args.warmup, peak allocation above what was live before, bytes)"""
    for _ in range(args.warmup):
        fn()
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats(dev)
    base = torch.cuda.memory_allocated(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / args.reps, torch.cuda.max_memory_allocated(dev) - base


def grid_lambdas(n):
    k = torch.arange(n, dtype=torch.float64, device=dev) / (n - 1)
    re, im = RE[0] + (RE[1] - RE[0]) * k, IM[0] + (IM[1] - IM[0]) * k
    return torch.complex(re[:, None].expand(n, n), im[None, :].expand(n, n)).reshape(-1)


gpu = gpu_info()
rng = np.random.default_rng(0)
for M in args.M:
    for pt in args.prec_types:
        A = num_actions(M, pt)
        loss = ResidualLoss(M, 1.0, pt, device=dev)
        row = torch.as_tensor(rng.uniform(0.02, 0.3, A) + 1j * rng.uniform(-0.05, 0.05, A), device=dev)
        for mode in ("batch", "grid"):
            lam = (torch.as_tensor(rng.uniform(*RE, args.B) + 1j * rng.uniform(*IM, args.B), device=dev)
                   if mode == "batch" else grid_lambdas(args.grid))
            N = lam.numel()
            for K in args.K:
                def per_sample():
                    _, _, n, g = loss.sweeps(lam, row, K, with_grad=True)
                    return torch.sum(n) / N, torch.sum(g, 0) / N

                if mode == "batch":
                    def fused():
                        return loss.sweeps_shared_value_and_grad(lam, row, K)
                else:
                    def fused():
                        return loss.sweeps_grid_value_and_grad(args.grid, args.grid, RE, IM, row, K)

                fused_ms, fused_mem = measure(fused)
                ps_ms, ps_mem = measure(per_sample)
                fused_ms2, _ = measure(fused)
                ps_ms2, _ = measure(per_sample)
                v_f, g_f = fused()
                v_p, g_p = per_sample()
                print(json.dumps({
                    "gpu": gpu, "mode": mode, "N": N, "M": M, "prec_type": pt, "K": K, "row": "complex",
                    "reduction": "mean", "reps": args.reps,
                    "fused_ms": [round(fused_ms, 4), round(fused_ms2, 4)],
                    "per_sample_sum_ms": [round(ps_ms, 4), round(ps_ms2, 4)],
                    "fused_peak_alloc_MB": round(fused_mem / 2**20, 2),
                    "per_sample_peak_alloc_MB": round(ps_mem / 2**20, 2),
                    "rel_diff_mean": abs(float(v_f) - float(v_p)) / abs(float(v_p)),
                    "max_rel_diff_grad": float((g_f - g_p).abs().max() / g_p.abs().max()),
                }), flush=True)
            del lam

"""||r_K||_inf after K sweeps, and its gradient through the K sweeps, for B samples with per-sample complex Q_delta rows
from the envs' reset state: ``ResidualLoss.sweeps`` (``residual_sweeps_kernel``) against what a user writes without
it - the same K sweeps as batched torch complex128 ops (``solve_triangular``) differentiated by autograd, and for the
value alone also K chained ``take_step`` calls.

One JSON object per line: time per call from CUDA events over --reps calls after warm-up, the increase of
``torch.cuda.max_memory_allocated`` over the inputs, and the bytes and flops per sample the algorithm needs (computed
from the shapes below, not measured).  The kernel's per-thread local memory for the saved deltas is allocated by the
driver, not by torch, and is not in the peak.  The GPU's name and power limit are read in the same run."""
import argparse, json, os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from sdc_gym_b200.collocation import collocation_matrix
from sdc_gym_b200.loss import ResidualLoss
from sdc_gym_b200.precond import num_actions
from tests.mp_reference import param_index

ap = argparse.ArgumentParser()
ap.add_argument("--B", type=int, default=1 << 20)
ap.add_argument("--M", type=int, nargs="+", default=[5, 9])
ap.add_argument("--prec-types", nargs="+", default=["diag", "lower_tri"])
ap.add_argument("--K", type=int, nargs="+", default=[1, 5, 20, 50])
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--warmup", type=int, default=1)
ap.add_argument("--out", default=None)
args = ap.parse_args()
dev = torch.device("cuda", 0)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = ""
    return out or torch.cuda.get_device_name(dev)


def measure(fn):
    """(ms per call over args.reps calls after args.warmup, peak allocation above what was live before)"""
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


def per_sample(M, prec_type, K, grad):
    """(bytes, flops) per sample: lambda + theta in, norm (+ g) out, plus the K deltas written and re-read for the
    gradient; a complex multiply-add is 8 flops, a real-by-complex one 4"""
    idx = param_index(M, prec_type)
    A, lower = len(idx), sum(1 for r, c in idx if c < r)
    sweep = 8 * lower + 6 * M + 4 * M * M + 6 * M + 4 * M  # substitution, diagonal scale, Q u, z (Q u), updates
    byts, flops = 16 + 16 * A + 8, K * sweep
    if grad:
        byts += 16 * A + 2 * 16 * M * K
        flops += K * (sweep + 8 * A)
    return byts, flops


def torch_twin(M, prec_type, lam, theta, K, grad):
    z = lam
    idx = param_index(M, prec_type)
    B = lam.shape[0]
    th = theta.detach().clone().requires_grad_(grad)
    rows = torch.tensor([a for a, _ in idx], device=dev)
    cols = torch.tensor([c for _, c in idx], device=dev)
    Qd = torch.zeros((B, M, M), dtype=torch.complex128, device=dev)
    Qd = Qd.index_put((torch.arange(B, device=dev)[:, None], rows[None], cols[None]), th)
    Q = torch.as_tensor(collocation_matrix(M), device=dev).to(torch.complex128)
    eye = torch.eye(M, dtype=torch.complex128, device=dev)
    P = eye - z[:, None, None] * Qd
    C = eye - z[:, None, None] * Q
    u0 = torch.ones((B, M), dtype=torch.complex128, device=dev)
    u = u0.clone()
    r = u0 - (C @ u[..., None])[..., 0]
    for _ in range(K):
        dl = torch.linalg.solve_triangular(P, r[..., None], upper=False)[..., 0]
        u = u + dl
        r = u0 - (C @ u[..., None])[..., 0]
    n = r.abs().amax(dim=1)
    if grad:
        n.sum().backward()
        return n, th.grad
    return n, None


info = gpu_info()
out = open(args.out, "a") if args.out else None
rng = np.random.default_rng(0)
for M in args.M:
    for prec_type in args.prec_types:
        A = num_actions(M, prec_type)
        loss = ResidualLoss(M, 1.0, prec_type)
        lam = torch.complex(torch.as_tensor(rng.uniform(-100, 0, args.B), device=dev),
                            torch.as_tensor(rng.uniform(-10, 0, args.B), device=dev))
        theta = torch.complex(torch.as_tensor(rng.uniform(0.02, 0.3, (args.B, A)), device=dev),
                              torch.as_tensor(rng.uniform(-0.05, 0.05, (args.B, A)), device=dev))
        for K in args.K:
            for grad in (False, True):
                rec = dict(gpu=info, M=M, prec_type=prec_type, K=K, B=args.B, grad=grad)
                b, f = per_sample(M, prec_type, K, grad)
                rec.update(bytes_per_sample=b, flops_per_sample=f)
                ms, peak = measure(lambda: loss.sweeps(lam, theta, K, with_grad=grad))
                rec.update(kernel_ms=round(ms, 4), kernel_peak_bytes=peak,
                           kernel_gflops=round(f * args.B / ms / 1e6, 1), kernel_gbytes_s=round(b * args.B / ms / 1e6, 1))
                ms, peak = measure(lambda: torch_twin(M, prec_type, lam, theta, K, grad))
                rec.update(autograd_twin_ms=round(ms, 4), autograd_twin_peak_bytes=peak)
                if not grad:
                    def chained():
                        u0 = torch.ones((args.B, M), dtype=torch.complex128, device=dev)
                        Q = torch.as_tensor(collocation_matrix(M), device=dev).to(torch.complex128)
                        u, r = u0, lam[:, None] * (Q.sum(dim=1)[None])
                        for _ in range(K):
                            u, r, _n = loss.take_step(lam, theta, None, u0, u, r)
                        return _n
                    ms, peak = measure(chained)
                    rec.update(chained_take_step_ms=round(ms, 4), chained_take_step_peak_bytes=peak)
                line = json.dumps(rec)
                print(line, flush=True)
                if out:
                    out.write(line + "\n")
                    out.flush()
                torch.cuda.empty_cache()

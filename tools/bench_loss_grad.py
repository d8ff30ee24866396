"""Times the spectral-radius gradient kernel alone (``rho_grad_kernel`` through ``SpectralRadiusLoss.radii_and_grads``,
CUDA events, 2^20 samples by default) next to the value kernel (``rho_kernel``) on the same inputs.  One JSON object
per line, with the GPU's name and power limit.  SDCGYM_LIB=<experiment build> selects another library, so two builds
can be compared by alternating calls."""
import argparse, json, os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from sdc_gym_b200.loss import SpectralRadiusLoss
from sdc_gym_b200.precond import num_actions

ap = argparse.ArgumentParser()
ap.add_argument("--B", type=int, default=1 << 20)
ap.add_argument("--M", type=int, nargs="+", default=[5, 9])
ap.add_argument("--prec-types", nargs="+", default=["diag", "lower_tri"])
ap.add_argument("--reps", type=int, default=20)
ap.add_argument("--tag", default="")
args = ap.parse_args()
dev = torch.device("cuda", 0)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = ""
    return out or torch.cuda.get_device_name(dev)


def timed(fn, reps, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps  # ms


gpu = gpu_info()
rng = np.random.default_rng(0)
for M in args.M:
    for pt in args.prec_types:
        B, A = args.B, num_actions(M, pt)
        lam = torch.as_tensor(rng.uniform(-100, 0, B) + 1j * rng.uniform(-10, 0, B), device=dev)
        hi = 0.08 if pt == "strictly_lower_tri" else 0.3
        out = torch.as_tensor(rng.uniform(0.02, hi, (B, A)) + 1j * rng.uniform(-0.05, 0.05, (B, A)), device=dev)
        loss = SpectralRadiusLoss(M, 1.0, pt, device=dev)
        grad_ms = timed(lambda: loss.radii_and_grads(lam, out), args.reps)
        rho_ms = timed(lambda: loss.spectral_radii(lam, out), args.reps)
        print(json.dumps({"tag": args.tag, "lib": os.environ.get("SDCGYM_LIB", "in-tree"), "gpu": gpu, "B": B,
                          "M": M, "prec_type": pt, "grad_ms": round(grad_ms, 4), "rho_ms": round(rho_ms, 4)}),
              flush=True)
        del lam, out

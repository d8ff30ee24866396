"""Does the K-sweep residual loss give a diagonal Q_delta that converges in fewer iterations than the spectral-radius
loss?  Trains one real diagonal with ``examples/train_diag_spectral_radius.py`` by rho, by ``--sweeps 5`` and by
``--sweeps 10`` (200 steps each, same seed), then runs the reference's evaluation loop (``evaluate_baselines.test_model``)
on ``sdc-v0`` (M = 5, real lambda in [-100, 0], restol 1e-10) with each learned diagonal passed as the action
(``free_action_space=True, do_scale=False``) and with the MIN diagonal.  One JSON line per diagonal: mean niter over
the successful episodes and the success rate; the GPU's name and power limit are read in the same run."""
import argparse, importlib.util, json, os, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import sdc_gym_b200

ap = argparse.ArgumentParser()
ap.add_argument("--steps", type=int, default=200)
ap.add_argument("--num_envs", type=int, default=100000)
ap.add_argument("--tests", type=int, default=3)
ap.add_argument("--out", default=None)
args = ap.parse_args()


def load(name):
    spec = importlib.util.spec_from_file_location(name, os.path.join(ROOT, "examples", name + ".py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


try:
    info = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True, timeout=30).stdout.strip()
except (OSError, subprocess.SubprocessError):
    info = ""
train, ev = load("train_diag_spectral_radius"), load("evaluate_baselines")
M = 5
diags = {}
for label, extra in (("rho", []), ("sweeps5", ["--sweeps", "5"]), ("sweeps10", ["--sweeps", "10"])):
    hist, theta = train.main(["--M", str(M), "--steps", str(args.steps)] + extra)
    diags[label] = (theta, hist[0], hist[-1])
diags["MIN"] = (np.diag(sdc_gym_b200.fixed_preconditioner("min", M)), None, None)
kw = dict(M=M, dt=1.0, restol=1e-10, lambda_real_interval=[-100, 0], lambda_imag_interval=[0, 0], seed=0)
out = open(args.out, "a") if args.out else None
for label, (theta, l0, l1) in diags.items():
    env = sdc_gym_b200.make("sdc-v0", num_envs=args.num_envs, free_action_space=True, do_scale=False, **kw)
    act = np.tile(np.asarray(theta, np.complex128), (args.num_envs, 1))
    niter, succ = ev.test_model(env, args.tests, label[:3], predict=lambda obs: act)
    rec = dict(gpu=info, trained_by=label, steps=args.steps if l0 is not None else 0, diag=[float(x) for x in theta],
               loss_first=l0, loss_last=l1, mean_niter=niter, success_rate=succ, num_envs=args.num_envs,
               tests=args.tests)
    line = json.dumps(rec)
    print(line, flush=True)
    if out:
        out.write(line + "\n")

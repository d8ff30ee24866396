"""Times the device replay buffer (sdc_gym_b200.replay) on one GPU, CUDA events / synchronised wall clock, each timed
window >= 1 s after warm-up:

* store (pre-step observation copy + replay_store_kernel) of a normalised sdc-v1 step, M = 5, 2^20 envs, in GB/s of
  the bytes it moves, next to a bare device copy of the same number of bytes in the same run (the working set,
  ~0.4 GB a row, is several times the 126 MB L2; the ring's rows rotate);
* sample (gather + normalisation) of B = 256, 2^14, 2^18 transitions from that buffer, in samples/s;
* one collect_transitions step against one collect_rollouts step (8-step collections, same policy, 2^20 envs);
* collect_transitions (8 steps) + sample(256) eagerly against one CUDA-graph replay of both, at 8 and 16 384 envs.

Prints the card's name and power limit first; one JSON object per line.  ``--out FILE`` also writes the lines there."""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import sdc_gym_b200  # noqa: E402
from sdc_gym_b200.replay import ReplayBuffer, collect_transitions  # noqa: E402
from sdc_gym_b200.rollout import collect_rollouts  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--envs", type=int, default=1 << 20)
ap.add_argument("--rows", type=int, default=8)
ap.add_argument("--out", default=None)
ap.add_argument("--min-seconds", type=float, default=1.0)
args = ap.parse_args()

M = 5
KW = dict(M=M, dt=1.0, restol=1e-10, lambda_real_interval=[-100, 0], lambda_imag_interval=[-10, 0], seed=0,
          output="torch", reward_iteration_only=False)
w = torch.linspace(-1.0, 1.0, 4 * M, dtype=torch.float64, device="cuda")
out_f = open(args.out, "w") if args.out else None


def emit(rec):
    line = json.dumps(rec)
    print(line, flush=True)
    if out_f:
        out_f.write(line + "\n")
        out_f.flush()


def policy(obs_planes):  # a dozen torch ops on the observation planes, capturable
    s = torch.tanh((obs_planes * w[:, None]).sum(0))
    return torch.stack([torch.tanh(s * (k + 1) * 0.7) for k in range(M)], dim=1) * 0.9


def policy_onpolicy(obs_planes):
    return policy(obs_planes), None, None


def event_us(fn, min_s):
    """mean device time per call over a window of >= min_s seconds (after a warm-up of 5 calls)"""
    for _ in range(5):
        fn()
    torch.cuda.synchronize()
    reps = 10
    while True:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if ms >= min_s * 1e3:
            return ms / reps * 1e3
        reps = max(reps * 2, int(reps * min_s * 1e3 / max(ms, 1e-3) * 1.1))


def wall_us(fn, min_s):
    for _ in range(5):
        fn()
    torch.cuda.synchronize()
    reps = 10
    while True:
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if dt >= min_s:
            return dt / reps * 1e6
        reps = max(reps * 2, int(reps * min_s / max(dt, 1e-6) * 1.1))


q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                   text=True)
emit({"card": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]})

# ---- store and sample at 2^20 envs ------------------------------------------------------------------------------
N = args.envs
env = sdc_gym_b200.VecNormalize(sdc_gym_b200.make("sdc-v1", num_envs=N, **KW))
env.reset()
venv = env.venv
rb = ReplayBuffer(args.rows * N, env, seed=1)
collect_transitions(env, policy, args.rows + 1, rb)  # fills the ring; also leaves a real step's outputs behind
a = policy(env.current_norm_planes[:, :N])
out = env.step_tensor(a)
P, A = 4 * M, M


def store():
    rb.store_obs(venv.S)
    rb.store(venv, a, out["flags"], out["raw_reward"])


# bytes moved per env: obs planes read + written, next-obs planes read (S or terminal) + written, actions read +
# written, reward read + written, flags read, done written
store_bytes = N * (4 * P * 8 + 2 * A * 8 + 2 * 8 + 1 + 1)
src = torch.empty(store_bytes // 2, dtype=torch.uint8, device="cuda")
dst = torch.empty_like(src)
src.fill_(1)
store_us = event_us(store, args.min_seconds)
copy_us = event_us(lambda: dst.copy_(src), args.min_seconds)
step_us = event_us(lambda: venv.step_tensor(a), args.min_seconds)
emit({"what": "store", "envs": N, "M": M, "rows": rb.rows, "bytes_per_env_step": store_bytes // N,
      "store_us": round(store_us, 2), "store_GBps": round(store_bytes / store_us / 1e3, 1),
      "bare_copy_us": round(copy_us, 2), "bare_copy_GBps": round(store_bytes / copy_us / 1e3, 1),
      "store_over_copy": round(store_us / copy_us, 3), "bare_sdc_v1_step_us": round(step_us, 2)})
del src, dst

for B in (256, 1 << 14, 1 << 18):
    for normalised in (False, True):
        us = event_us(lambda: rb.sample(B, env if normalised else None), args.min_seconds)
        emit({"what": "sample", "envs": N, "rows": rb.rows, "batch": B, "normalised": normalised,
              "us": round(us, 2), "samples_per_s": round(B / us * 1e6, 1)})

# ---- one collection step: off-policy (replay) against on-policy (rollout) ---------------------------------------
T = 8
rbuf = None


def rollout():
    global rbuf
    rbuf = collect_rollouts(env, policy_onpolicy, T, buffer=rbuf)


tr_us = wall_us(lambda: collect_transitions(env, policy, T, rb), args.min_seconds)
ro_us = wall_us(rollout, args.min_seconds)
emit({"what": "collect_step", "envs": N, "n_steps": T, "collect_transitions_us_per_step": round(tr_us / T, 2),
      "collect_rollouts_us_per_step": round(ro_us / T, 2), "ratio": round(tr_us / ro_us, 3)})
del rb, rbuf, env, venv, out, a
torch.cuda.empty_cache()

# ---- eager against CUDA graph at small batches --------------------------------------------------------------------
for n in (8, 16384):
    rec = {"what": "graph", "envs": n, "n_steps": T, "sample_batch": 256}
    for mode in ("eager", "graph"):
        e = sdc_gym_b200.VecNormalize(sdc_gym_b200.make("sdc-v1", num_envs=n, **KW))
        e.reset()
        r = ReplayBuffer(64 * n, e, seed=1)

        def once():
            collect_transitions(e, policy, T, r)
            return r.sample(256, e)

        fn = once
        if mode == "graph":
            for _ in range(2):
                once()
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            g = torch.cuda.CUDAGraph()
            with torch.cuda.stream(side):
                with torch.cuda.graph(g, stream=side):
                    once()
            torch.cuda.current_stream().wait_stream(side)
            fn = g.replay
        us = wall_us(fn, args.min_seconds)
        rec[mode + "_us"] = round(us, 2)
        rec[mode + "_env_steps_per_s"] = round(n * T / us * 1e6, 1)
        del e, r
    rec["speedup"] = round(rec["eager_us"] / rec["graph_us"], 2)
    emit(rec)

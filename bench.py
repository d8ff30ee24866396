#!/usr/bin/env python
"""bench.py - headline benchmark of the SDC env-step hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[1]): batched `sdc-v0` full-solve env, 2^20 envs per GPU, M=5, diagonal Q_delta
from uniform random actions in [-1,1]^5, lambda ~ U[-100,0] + i U[-10,0], restol=1e-10, max 50 sweeps, with the
DummyVecEnv auto-reset fused into the step (every step finishes all episodes and draws new lambdas).
One "step" = one env.step over all envs of all ranks; value = env-steps/s over the whole job (weak scaling:
envs per GPU fixed).  Prints ONE JSON line (rank 0).

Timed regions
  value : K device-resident steps (`SDCVecEnv.step_tensor`, actions already in HBM), CUDA events on the launching
          stream, barrier + synchronize on both sides, max over ranks.
  e2e   : K steps through the drop-in API `SDCVecEnv.step(numpy actions)` with its DEFAULT settings: pinned-host
          actions -> H2D, kernels, obs/reward/done/info -> D2H into the result block whose views are returned
          (caller-owned until dropped), wall clock with synchronize on both sides.  `e2e.variants` adds the same loop
          with `reuse_buffers=True` and with an explicit fresh copy of every output per step; `e2e.pcie_ceiling` is
          the same bytes moved by bare concurrent cudaMemcpyAsync on all ranks (what the box's PCIe allows).
  secondary : bounded (<= ~10 s) measurements of BASELINE configs 3, 4, 5 at this run's rank count.
  cpu_baseline : the reference's own env (oracle/_ref/sdc_env.py, staged unmodified by `make -C oracle ref`; the numpy
          port oracle/sdc_port.py when no reference file is reachable) on one host core, ~10 s sample.
  --impl reference : the same on all host cores (multiprocessing), time-bounded samples.
  --dump-outputs DIR : after the `value` steps, what the last of them returned (reward, flags, niter, residual, lam,
          terminal observation planes) for a fixed sample of rank 0's envs, as float64 .npy files.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
os.environ.setdefault("OPENBLAS_NUM_THREADS", "1")

METRIC = "SDC env-steps/sec (M=5, diag Qdelta)"
UNIT = "env-steps/s"
M = 5
ENVS_PER_GPU = 1 << 20
FLOPS_PER_SWEEP = 4 * M * M + 22 * M  # 210 at M=5, diag Q_delta (SURVEY.md 8d)
FLOPS_SETUP = 15 * M
BYTES_PER_ENV_STEP_V0 = 8 * M + 32 * M + 52  # 252 B algorithmic (SURVEY.md 8d)
WORKLOAD = "sdc-v0 full solve, M=5, diag Qdelta (uniform random actions), 2^20 envs/GPU, restol=1e-10, maxiter=50"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 50 ms while the timed regions (value + e2e) run."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for name, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def _dist_setup(n_gpus):
    import torch

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if os.environ.get("NCCL_DEBUG", "").upper() in ("VERSION", "WARN"):
            os.environ.pop("NCCL_DEBUG")  # both levels print NCCL's version banner to stdout: one JSON line only
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    elif n_gpus > 1:
        raise SystemExit("--gpus N > 1 must be launched with torch.distributed.run (one rank per GPU)")
    else:
        torch.cuda.set_device(0)
    return world, rank, local


def _cpu_ref_worker(args):
    kind, seconds, seed = args
    os.environ["OPENBLAS_NUM_THREADS"] = "1"
    from oracle import ref_bench

    return ref_bench.rollout_throughput(kind, seconds, num_envs=8, M=M, seed=seed)


def _impl_text(impl):
    return ("the UNMODIFIED reference env (sdc_gym/envs/sdc_env.py staged in oracle/_ref, stub gym/pySDC modules)"
            if impl == "reference" else "numpy port of the reference env (oracle/sdc_port.py)")


def cpu_baseline_single(seconds=10.0):
    from oracle import ref_bench

    ref_bench.rollout_throughput("sdc-v0", 0.5, num_envs=8, M=M, seed=99)  # warm-up
    steps, el, sum_niter, impl = ref_bench.rollout_throughput("sdc-v0", seconds, num_envs=8, M=M, seed=0)
    return {"value": steps / el, "unit": UNIT, "cores": 1, "kind": impl,
            "sample": f"{steps} sdc-v0 env-steps (M=5, diag, uniform random actions, 8-env DummyVecEnv loop, "
                      f"mean niter {sum_niter / steps:.1f}) in {el:.1f} s on one host core, {_impl_text(impl)}"}


def cpu_baselines_secondary(seconds=3.0):
    """BASELINE.md 3: the reference's sdc-v1 8-env rollout (configs[0]) and its numpy spectral radius, one core each."""
    from oracle import ref_bench

    s1, e1, _, impl = ref_bench.rollout_throughput("sdc-v1", seconds, num_envs=8, M=M, seed=0, reward_iteration_only=False)
    n, e2, mean_rho, _ = ref_bench.spectral_radius_throughput(seconds, M=M)
    return {"sdc_v1_8env": {"value": s1 / e1, "unit": UNIT, "cores": 1, "kind": impl,
                            "sample": f"{s1} sdc-v1 env-steps (M=5, diag, 8 envs, residual_change reward) in {e1:.1f} s"},
            "spectral_radius_numpy": {"value": n / e2, "unit": "matrices/s", "cores": 1, "kind": impl,
                                      "sample": f"{n} x (np.linalg.inv + np.linalg.eigvals, sdc_env.py:193-201,421-425), "
                                                f"M=5 MIN diag, in {e2:.1f} s; mean rho {mean_rho:.4f}"}}


def cpu_c_oracle_single(envs=16384):
    """Extra context: the plain-C rounding-exact restatement (oracle/sdc_exact.c) on one core - an upper bound for
    what a compiled CPU implementation of the same arithmetic does; the reference itself is the numpy figure."""
    import numpy as np
    from oracle import exact
    from sdc_gym_b200.collocation import collocation_matrix

    rng = np.random.default_rng(0)
    Q = collocation_matrix(M)
    lam = rng.uniform(-100, 0, envs) + 1j * rng.uniform(-10, 0, envs)
    act = rng.uniform(-1, 1, (envs, M))
    u, r = exact.reset(Q, 1.0, lam)
    niter = np.zeros(envs, np.int32)
    t0 = time.perf_counter()
    exact.step("sdc-v0", Q, 1.0, lam, u, r, niter, r.copy(), act)
    el = time.perf_counter() - t0
    return {"value": envs / el, "unit": UNIT, "cores": 1, "kind": "port (plain C, rounding-exact oracle)",
            "sample": f"{envs} sdc-v0 env-steps in {el:.2f} s, mean niter {niter.mean():.1f}"}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on all host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp

    from oracle import ref_bench

    impl = ref_bench.available_impl()
    per_step = max(0.5, min(4.0, 150.0 / max(1, args.steps + args.warmup)))
    if os.environ.get("SDCGYM_BENCH_REF_SECONDS"):  # tests shorten the samples
        per_step = float(os.environ["SDCGYM_BENCH_REF_SECONDS"])
    cores = int(os.environ.get("SDCGYM_BENCH_REF_CORES", os.cpu_count() or 1))
    ctx = mp.get_context("spawn")
    total_steps, total_time = 0, 0.0
    with ctx.Pool(cores) as pool:
        for s in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            res = pool.map(_cpu_ref_worker, [("sdc-v0", per_step, 1000 * s + c) for c in range(cores)])
            el = time.perf_counter() - t0
            if s >= args.warmup:
                total_steps += sum(r[0] for r in res)
                total_time += el
    value = total_steps / total_time
    sample = (f"{args.steps} samples of {per_step:.1f} s on {cores} processes (one per host core), each stepping an "
              f"8-env sdc-v0 DummyVecEnv loop with uniform random actions; {_impl_text(impl)}")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total_time / max(1, args.steps),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": {"workload": WORKLOAD, "host_cores": cores},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": impl, "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def run_secondary(torch, np, dev, rank, world, barrier, max_over_ranks, fp64_peak, hbm_peak, args):
    """BASELINE.json configs 3, 4, 5 at this run's rank count, a few steps each (<= ~10 s in total).  Work per unit and
    the roofline each is held against: SURVEY.md 8(d) / DESIGN.md 4."""
    import sdc_gym_b200
    from sdc_gym_b200 import dist as sdist
    from sdc_gym_b200.loss import SpectralRadiusLoss
    from sdc_gym_b200.precond import fixed_preconditioner, num_actions
    from sdc_gym_b200.rollout import collect_rollouts

    KW = dict(dt=1.0, restol=1e-10, lambda_real_interval=[-100, 0], lambda_imag_interval=[-10, 0], seed=0, device=dev)
    gen = torch.Generator(device=dev)
    gen.manual_seed(100 + rank)

    def timed(fn, steps, warm=2):
        for _ in range(warm):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1)) / steps

    def allsum(x):
        t = torch.tensor([float(x)], dtype=torch.float64, device=dev)
        if world > 1:
            torch.distributed.all_reduce(t)
        return float(t.item())

    out = {"n_gpus": world}
    # ---- config 3: M sweep x {lower_tri, strictly_lower_tri}, sdc-v0, exact np.linalg.inv emulation on the device ----
    Ns = args.secondary_envs
    sweep = []
    for Mx in (3, 5, 7, 9):
        for pt in ("lower_tri", "strictly_lower_tri"):
            A = num_actions(Mx, pt)
            acts = [torch.rand((Ns, A), dtype=torch.float64, device=dev, generator=gen) * 0.3 for _ in range(2)]
            # M <= 7: both launch sequences of the dense full solve (bit-identical results; SDCVecEnv's default times
            # them on the caller's workload and keeps the faster one, which is what `ms_per_step` reports)
            by_launch = {}
            for phased in ((False, True) if Mx <= 7 else (False,)):
                env = sdc_gym_b200.make("sdc-v0", num_envs=Ns, M=Mx, prec_type=pt, do_scale=False, env_offset=rank * Ns,
                                        phased=phased, **KW)
                env.reset()
                k = [0]

                def f():
                    k[0] += 1
                    env.step_tensor(acts[k[0] % 2])

                by_launch["phased" if phased else "single"] = timed(f, 3)
                sum_niter = allsum(env.info_niter[:Ns].double().sum())
                if phased:
                    suspended = [int(c) for c in env.phase_count.cpu().numpy()[:2]]
                del env
            launch = min(by_launch, key=by_launch.get)
            ms = by_launch[launch]
            per_sweep = 8 * Mx * Mx + (18 if pt == "lower_tri" else 12) * Mx
            flops = sum_niter * per_sweep + world * Ns * (15 * Mx + 2 * A)
            tf = flops / (ms * 1e-3) / 1e12
            sweep.append({"M": Mx, "prec_type": pt, "envs_per_gpu": Ns, "ms_per_step": ms,
                          "env_steps_per_s": world * Ns / ms * 1e3, "mean_niter": sum_niter / (world * Ns),
                          "fp64_tflops_algorithmic": tf, "fp64_frac": tf / (world * fp64_peak) if fp64_peak else None,
                          "launch": launch, "ms_by_launch": by_launch,
                          "suspended_per_pass_rank0": suspended if Mx <= 7 else None})
            del acts
            torch.cuda.empty_cache()
    out["config3_dense_qdelta_sweep"] = {
        "workload": "sdc-v0, Q_delta entries ~ U[0, 0.3] (do_scale=False), lambda ~ U[-100,0] + i U[-10,0]", "cases": sweep,
        "flops": "per sweep 8M^2+18M (lower_tri) / 8M^2+12M (strictly_lower_tri), set-up 15M + 2A (SURVEY 8d); the "
                 "bit-exact kernels execute more (the pivoted zgetf2 + ztrsm emulation of np.linalg.inv per step)",
        "launch": "single = one kernel, a warp runs until its last env is done; phased = warps that have thinned out "
                  "hand their stragglers to compacted lists (csrc/step_kernels.cuh step_one PHASE); M >= 8: lane-team kernel"}
    # ---- the certified substitution sweep mode (SDCGYM_SWEEP_CERTIFIED) against the exact mode on the headline workload
    #      and on a workload where half of the envs converge (actions near the MIN preconditioner) ----
    Nc = ENVS_PER_GPU
    xmin = torch.as_tensor(np.ascontiguousarray(np.diag(fixed_preconditioner("min", 5))), device=dev)
    modes = []
    for wl in ("uniform", "near_MIN"):
        if wl == "uniform":
            acts = [torch.rand((Nc, 5), dtype=torch.float64, device=dev, generator=gen) * 2 - 1 for _ in range(2)]
        else:
            acts = [2 * (xmin[None] + (torch.rand((Nc, 5), dtype=torch.float64, device=dev, generator=gen) - 0.5) * 0.04) - 1
                    for _ in range(2)]
        res = {}
        for mode in ("exact", "certified"):
            env = sdc_gym_b200.make("sdc-v0", num_envs=Nc, M=5, env_offset=rank * Nc, sweep_mode=mode, **KW)
            env.reset()
            k = [0]

            def f():
                k[0] += 1
                env.step_tensor(acts[k[0] % 2])

            ms = timed(f, 4)
            fb0 = env.fallback_stats()[1]
            f()
            fb = (env.fallback_stats()[1] - fb0) / Nc
            res[mode] = dict(ms=ms, niter=env.info_niter[:Nc].clone(), flags=env.flags[:Nc].clone(), fb=fb)
            del env
        same = bool(torch.equal(res["exact"]["niter"], res["certified"]["niter"])
                    and torch.equal(res["exact"]["flags"], res["certified"]["flags"]))
        modes.append({"workload": wl, "exact_ms_per_step": res["exact"]["ms"], "certified_ms_per_step": res["certified"]["ms"],
                      "certified_fallback_frac": res["certified"]["fb"], "niter_and_flags_bit_equal": same})
        del acts, res
        torch.cuda.empty_cache()
    out["sweep_modes"] = {
        "envs_per_gpu": Nc, "M": 5, "cases": modes,
        "note": "certified = fp32 certificate kernel + substitution-sweep kernel + exact kernel over the fallback list "
                "(csrc/certify.cuh, fast_kernels.cuh): same iteration counts and flags, u / r within rounding; the "
                "headline `value` is measured in the exact mode"}
    # ---- config 4: spectral-radius loss on a 4096 x 4096 lambda grid, M = 5, MIN diagonal; rows sharded over the ranks ----
    G = args.grid
    loss = SpectralRadiusLoss(5, 1.0, "diag", device=dev)
    x = np.diag(fixed_preconditioner("min", 5))
    lo, cnt = sdist.shard_range(G, rank, world)
    ms = timed(lambda: loss.grid(G, G, [-100, 0], [-10, 0], x, rows=(lo, lo + cnt)), 3)
    rho_flops = 13 * 5 ** 3 * 8  # ~13 kflop per matrix (SURVEY 8d)
    tf = G * G * rho_flops / (ms * 1e-3) / 1e12
    out["config4_spectral_radius_grid"] = {"grid": [G, G], "M": 5, "prec": "MIN diag", "ms": ms, "scaling": "strong",
                                           "matrices_per_s": G * G / ms * 1e3, "fp64_tflops_algorithmic": tf,
                                           "fp64_frac": tf / (world * fp64_peak) if fp64_peak else None,
                                           "flops_per_matrix": rho_flops}
    # ---- config 5: sdc-v1 rollout collection, device VecNormalize (synchronised over the ranks), RolloutBuffer + GAE ----
    Nr, T = 1 << 20, 8
    env = sdc_gym_b200.VecNormalize(
        sdc_gym_b200.make("sdc-v1", num_envs=Nr, M=5, env_offset=rank * Nr, reward_iteration_only=False, **KW),
        norm_obs=True, norm_reward=True, sync=True)
    env.reset()

    def policy(obs_planes):
        a = torch.empty((Nr, 5), dtype=torch.float64, device=dev).uniform_(-1.0, 1.0, generator=gen)
        return a, obs_planes[0], None

    buf = [collect_rollouts(env, policy, T)]

    def roll():
        buf[0] = collect_rollouts(env, policy, T, buffer=buf[0])

    ms = timed(roll, 3, warm=1)
    bytes_step = 8 * 5 + 64 * 5 + 49                   # sdc-v1 env-step (SURVEY 8d): 409 B
    bytes_norm = 3 * 32 * 5 + 40                       # statistics read + apply read/write of the 4M planes, returns/reward
    bytes_buf = 2 * (8 * 5 + 8 + 8 + 1)                # actions, rewards, values, episode starts into the buffer
    bpe = bytes_step + bytes_norm + bytes_buf
    gbs = world * Nr * T * bpe / (ms * 1e-3) / 1e9
    out["config5_normalised_rollout"] = {
        "envs_per_gpu": Nr, "n_steps": T, "env_steps_per_rollout": world * Nr * T, "ms_per_rollout": ms,
        "env_steps_per_s": world * Nr * T / ms * 1e3, "time_for_64M_env_steps_s": (1 << 26) / (world * Nr * T / ms * 1e3),
        "algorithmic_bytes_per_env_step": bpe, "hbm_GBps_algorithmic": gbs, "hbm_frac": gbs / (world * hbm_peak),
        "policy": "uniform random actions drawn on the device", "normaliser_sync": "every step, all ranks"}
    del env, buf
    torch.cuda.empty_cache()
    # ---- the same collection as ONE CUDA-graph replay per rollout (sdc_gym_b200.rollout.GraphedRollout; single rank:
    #      the in-kernel peer exchange is sequenced from the host), at the benchmark size and in the reference's own
    #      regime of 8 envs (BASELINE config 1), where launches and the interpreter are the whole cost ----
    if world == 1:
        from sdc_gym_b200.rollout import GraphedRollout

        graphed = []
        for Ng in (8, 16384, Nr):
            def gpolicy(obs_planes, Ng=Ng):  # default CUDA generator: capturable
                return torch.empty((Ng, 5), dtype=torch.float64, device=dev).uniform_(-1.0, 1.0), obs_planes[0], None

            rec = {"envs": Ng, "n_steps": T}
            for mode in ("eager", "graph"):
                env = sdc_gym_b200.VecNormalize(sdc_gym_b200.make("sdc-v1", num_envs=Ng, M=5, reward_iteration_only=False,
                                                                  output="torch", **KW))
                env.reset()
                gr = GraphedRollout(env, gpolicy, T, warmup=2) if mode == "graph" else None
                b = [None]

                def once():
                    if gr is not None:
                        gr.collect()
                    else:
                        b[0] = collect_rollouts(env, gpolicy, T, buffer=b[0])

                for _ in range(4):
                    once()
                torch.cuda.synchronize()
                reps = 5 if Ng == Nr else 30
                t0 = time.perf_counter()
                for _ in range(reps):
                    once()
                torch.cuda.synchronize()
                ms_g = (time.perf_counter() - t0) / reps * 1e3  # wall clock: the interpreter is what the graph removes
                rec[mode + "_ms_per_rollout"] = ms_g
                rec[mode + "_env_steps_per_s"] = Ng * T / ms_g * 1e3
                del env, gr, b
            graphed.append(rec)
        out["config5_graphed_rollout"] = {
            "cases": graphed, "timing": "wall clock around back-to-back rollouts, synchronised at both ends",
            "note": "bit-identical to the eager collection (tests/test_gpu_normalize_loss.py); BASELINE.md: the reference's "
                    "sdc-v1 8-env rollout runs at ~1.2e4 env-steps/s per host core"}
        torch.cuda.empty_cache()
    return out


DUMP_ENVS = 1 << 17  # sampled envs per dump: 216 B each in float64 (index included), 28.3 MB in all


def dump_outputs(path, out, N):
    """Write what the last timed `step_tensor` returned, for a fixed seeded sample of envs, as float64 .npy files:
    two builds run with the same arguments see the same inputs, so their dumps compare output for output."""
    import numpy as np
    import torch

    idx = np.arange(N) if N <= DUMP_ENVS else np.sort(np.random.default_rng(0).choice(N, DUMP_ENVS, replace=False))
    idx_dev = torch.as_tensor(idx, device=out["reward"].device)
    arrays = {"env_index": idx.astype(np.float64)}
    for name in ("reward", "flags", "niter", "residual"):
        arrays[name] = out[name][idx_dev].double().cpu().numpy()
    arrays["lam"] = torch.view_as_real(out["lam"][idx_dev]).cpu().numpy()  # (n, 2): real, imaginary part
    if "terminal" in out:
        arrays["terminal"] = out["terminal"][:, idx_dev].cpu().numpy()  # (4M, n) planes, as returned
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def run_ours(args):
    import numpy as np
    import torch

    world, rank, local = _dist_setup(args.gpus)
    import sdc_gym_b200
    from sdc_gym_b200 import _lib

    dev = torch.device("cuda", local)
    N = ENVS_PER_GPU if args.envs_per_gpu is None else args.envs_per_gpu
    env = sdc_gym_b200.make("sdc-v0", num_envs=N, M=M, dt=1.0, restol=1e-10, seed=0, env_offset=rank * N,
                            lambda_real_interval=[-100, 0], lambda_imag_interval=[-10, 0], autoreset=True, device=dev)
    gen = torch.Generator(device=dev)
    gen.manual_seed(1 + rank)
    pool = [torch.rand((N, M), dtype=torch.float64, device=dev, generator=gen) * 2 - 1 for _ in range(4)]
    env.reset()

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(x):
        if world > 1:
            t = torch.tensor([x], dtype=torch.float64, device=dev)
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
            return float(t.item())
        return x

    # ---------------- device-resident value ----------------
    for k in range(args.warmup):
        env.step_tensor(pool[k % 4])
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(args.steps):
        out = env.step_tensor(pool[k % 4])
    e1.record()
    barrier()
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out, N)
    launches = args.steps  # one step kernel per step (solve + reward + auto-reset fused)
    # statistics of the last step (per-rollout reduction over NCCL, outside the step path)
    niter = env.info_niter[:N].to(torch.float64)
    flags = env.flags[:N]
    stats = torch.stack([env.reward[:N].sum(), niter.sum(), (flags & 2).ne(0).sum().double(),
                         (flags & 4).ne(0).sum().double()])
    if world > 1:
        torch.distributed.all_reduce(stats)
    stats = stats.cpu().numpy()
    sum_niter_local = float(niter.sum().item())
    value = world * N * args.steps / (ms_total * 1e-3)

    # ---------------- FP64 peak probe (measured live; MEASURED_PEAKS.json has no fp64 entry) ----------------
    L = _lib.load()
    sink = torch.zeros(1, dtype=torch.float64, device=dev)
    stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    flops = ctypes.c_double(0.0)
    best = 0.0
    probe_sampler = ClockSampler(local)  # the denominator's own clock record (the probe runs ~0.6 s)
    if rank == 0:
        probe_sampler.start()
    for _ in range(24):
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p0.record()
        _lib.check(L.sdcgym_fp64_peak_probe(4096, sink.data_ptr(), ctypes.byref(flops), stream), "probe")
        p1.record()
        torch.cuda.synchronize(dev)
        best = max(best, flops.value / (p0.elapsed_time(p1) * 1e-3) / 1e12)
    fp64_peak_tflops = best
    probe_clocks = probe_sampler.stop() if rank == 0 else None

    kernel_ms = ms_total / args.steps  # the step is a single kernel launch
    alg_flops = sum_niter_local * FLOPS_PER_SWEEP + N * FLOPS_SETUP
    achieved_tflops = alg_flops / (kernel_ms * 1e-3) / 1e12
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    hbm_achieved = N * BYTES_PER_ENV_STEP_V0 / (kernel_ms * 1e-3) / 1e9
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            traffic = json.load(f).get("step_kernel_dram_bytes_per_launch")
    except Exception:
        pass

    # ---------------- end-to-end through the drop-in API with host buffers ----------------
    rng = np.random.default_rng(7 + rank)
    host_bufs = [env.pinned_action_buffer(0), env.pinned_action_buffer(1)]
    for b in host_bufs:  # two action sets resident in page-locked host memory, used alternately
        b[:] = rng.uniform(-1, 1, (N, M))

    def e2e_loop(e, steps, copy_outputs=False, read_infos=False):
        checksum = 0.0
        for k in range(min(3, args.warmup)):
            e.step(host_bufs[k % 2])
        barrier()
        t0 = time.perf_counter()
        for k in range(steps):
            obs, rew, done, infos = e.step(host_bufs[k % 2])
            if copy_outputs:  # what a caller pays who must own fresh, contiguous arrays every step
                obs, rew, done = np.array(obs, order="C"), rew.copy(), done.copy()
                keep = (infos.niter.copy(), infos.residual.copy(), infos.lam.copy())  # noqa: F841
            if read_infos:  # a caller that looks at info['niter' / 'residual' / 'lam'] after every step
                checksum += float(infos.niter[0]) + float(infos.residual[0]) + float(infos.lam[0].real)
            checksum += float(rew[0]) + float(obs[0, 1, 0].real) + float(done[0])
        barrier()
        return max_over_ranks(time.perf_counter() - t0), checksum

    e2e_s, checksum = e2e_loop(env, args.steps)  # DEFAULT settings: outputs owned by the caller until dropped
    clocks = sampler.stop() if rank == 0 else None
    e2e_value = world * N * args.steps / e2e_s
    h2d = N * M * 8
    lazy = bool(getattr(env, "lazy_info", False)) and N >= 32768
    d2h_info = N * (4 + 8 + 16)  # niter, residual norm, lambda: fetched when an info dict / array is read (lazy_info)
    d2h = N * (M * 16 + 8 + 1) + (0 if lazy else d2h_info)  # residual row (the u row of sdc-v0's reset state is
    #                                                          constant), reward, flags [+ info arrays]
    host_sets, host_copies = len(env._host["sets"]), env.host_set_copies
    infos_s, _ = e2e_loop(env, args.steps, read_infos=True)
    env.reuse_buffers = True
    reuse_s, _ = e2e_loop(env, args.steps)
    copy_s, _ = e2e_loop(env, max(2, args.steps // 2), copy_outputs=True)
    copy_steps = max(2, args.steps // 2)
    env.reuse_buffers = False

    # ---------------- what the box's PCIe allows for these bytes: bare concurrent copies on every rank -------------
    hb = env._host["sets"][0].blk
    skip = int(env._layout.reward)
    dsrc = env.dev_block
    a_dev, a_host = env.action_dev, env._host["actions"][0]
    s1, s2 = torch.cuda.Stream(dev), torch.cuda.Stream(dev)

    lay = env._layout
    segs = [(int(lay.reward), int(lay.residual)), (int(lay.flags), int(lay.total))] if lazy else [(skip, int(lay.total))]
    moved = sum(b - a for a, b in segs)

    def copies():
        with torch.cuda.stream(s1):
            a_dev.copy_(a_host, non_blocking=True)
        with torch.cuda.stream(s2):
            for a, b in segs:
                hb[a:b].copy_(dsrc[a:b], non_blocking=True)

    for _ in range(3):
        copies()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        copies()
        s1.synchronize()
        s2.synchronize()
    barrier()
    pcie_s = max_over_ranks(time.perf_counter() - t0)
    pcie_value = world * N * args.steps / pcie_s
    pcie = {"value": pcie_value, "unit": UNIT, "ms_per_step": 1e3 * pcie_s / args.steps,
            "d2h_GBps_per_gpu": moved / (pcie_s / args.steps) / 1e9,
            "how": f"{world} rank(s) concurrently: cudaMemcpyAsync of one step's bytes (H2D {h2d} B on one stream, D2H "
                   f"{moved} B on another, page-locked host memory), no kernels",
            "e2e_frac": e2e_value / pcie_value}

    # ---------------- secondary: BASELINE configs 3, 4, 5 (bounded) ----------------
    secondary = None
    if not args.no_secondary:
        secondary = run_secondary(torch, np, dev, rank, world, barrier, max_over_ranks, fp64_peak_tflops, hbm_peak, args)

    cpu, cpu_c, cpu_more = None, None, None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline_single(args.cpu_seconds)
        cpu_c = cpu_c_oracle_single()
        cpu_more = cpu_baselines_secondary(min(3.0, args.cpu_seconds))

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "envs_per_gpu": N, "global_envs": world * N, "M": M,
                       "prec_type": "diag", "sharding": f"envs partitioned over {world} GPU(s), no collective on the "
                       "step path; NCCL all-reduce of rollout statistics only",
                       "l2_policy": "inputs larger than L2 (~600 MB of env state/action/result planes touched per step; "
                                    "4 rotating action sets)",
                       "blas_variant": int(env.blas_variant)},
            "gpu_launches": launches,
            "roofline": {"bound": "fp64", "achieved": achieved_tflops, "peak": fp64_peak_tflops, "unit": "TFLOP/s",
                         "frac": achieved_tflops / fp64_peak_tflops if fp64_peak_tflops else None,
                         "traffic": traffic,
                         "peak_source": "measured live: DFMA-chain probe kernel (sdcgym_fp64_peak_probe), best of 24; "
                                        "MEASURED_PEAKS.json has no fp64 entry (nominal 148 SM x 64 x 2 x 1.965 GHz = 37.2)",
                         "peak_clocks": probe_clocks,
                         "traffic_source": "profiles/traffic.json (dram__bytes_read.sum + dram__bytes_write.sum of one "
                                           "`ncu --set full` capture of this kernel; not re-measured in this run)",
                         "algorithmic_flops_per_launch": alg_flops, "kernel_ms": kernel_ms,
                         "mean_niter": sum_niter_local / N,
                         "note": "bit-exact emulation of the reference's rounding sequence needs 183 FP64 instructions "
                                 "(mul/add/fma, <= 1 FMA each) per 210-flop sweep: instruction-level ceiling of the "
                                 "algorithmic fraction = 210/(2*183) = 0.57, x 0.87 lane efficiency (envs of a warp stop "
                                 "at different sweeps) = 0.49; measured (ncu, profiles/ncu_step_kernel_r01_shipped_summary.json): FP64 pipe 76 % busy, shared-memory/LSU data pipe 81 % (25 LDS.128 of C per sweep) - the two co-limit the kernel",
                         "hbm": {"achieved": hbm_achieved, "peak": hbm_peak, "unit": "GB/s",
                                 "frac": hbm_achieved / hbm_peak, "bytes_per_env_step": BYTES_PER_ENV_STEP_V0,
                                 "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback 6.65 TB/s"}},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": 1e3 * e2e_s / args.steps,
                    "api": "SDCVecEnv.step(numpy actions in pinned memory) -> numpy obs, rewards, dones, infos with the "
                           "DEFAULT settings: results are views of a page-locked result block that is rewritten only "
                           "once the caller has dropped them (terminal observations stay on the device until an info "
                           "dict asks for them; the u row of sdc-v0's returned reset state is constant and not moved)",
                    "host_result_blocks": host_sets, "steps_that_copied": host_copies,
                    "info_arrays": ("niter / residual / lam (28 B per env) stay in the device block until an info dict or "
                                    "array is read (lazy_info, batches >= 32768 envs); variants.reading_infos_every_step "
                                    "pays for them") if lazy else "transferred with every step",
                    "variants": {"reading_infos_every_step": {"value": world * N * args.steps / infos_s, "unit": UNIT,
                                                              "ms_per_step": 1e3 * infos_s / args.steps,
                                                              "d2h_bytes_per_step": d2h + (d2h_info if lazy else 0)},
                                 "reuse_buffers": {"value": world * N * args.steps / reuse_s, "unit": UNIT,
                                                   "ms_per_step": 1e3 * reuse_s / args.steps},
                                 "fresh_copy_of_every_output": {"value": world * N * copy_steps / copy_s, "unit": UNIT,
                                                                "ms_per_step": 1e3 * copy_s / copy_steps}},
                    "pcie_ceiling": pcie},
            "secondary": secondary,
            "cpu_baseline": cpu,
            "cpu_baseline_c_oracle": cpu_c,
            "cpu_baseline_secondary": cpu_more,
            "clocks": clocks,
            "rollout_stats": {"sum_reward": float(stats[0]), "sum_niter": float(stats[1]),
                              "converged": float(stats[2]), "diverged": float(stats[3]),
                              "reduced_over": f"{world} rank(s) via NCCL all-reduce" if world > 1 else "1 rank"},
            "checksum": checksum,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        torch.distributed.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs-per-gpu", type=int, default=None)
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--grid", type=int, default=4096, help="lambda grid edge of the config-4 measurement")
    ap.add_argument("--secondary-envs", type=int, default=1 << 22, help="envs per GPU of the config-3 sweep")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (rank 0, a fixed sample of at most "
                         f"{DUMP_ENVS} envs) as DIR/<name>.npy in float64")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()

"""Builds ``sdc_gym_b200/libsdcgym.so`` (sm_100a) in-tree with nvcc.

``python -m sdc_gym_b200.build`` or ``build_library()``.  The per-M instantiation units are compiled in
parallel.  The .so travels with the repository snapshot to the GPU box (git-ignored, not gpurun-ignored).
"""
from __future__ import annotations

import concurrent.futures
import hashlib
import os
import shutil
import subprocess
import sys

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
OBJ_DIR = os.path.join(_HERE, "_build")
LIB_PATH = os.path.join(_HERE, "libsdcgym.so")
M_VALUES = tuple(range(2, 10))

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-fmad=false",  # never contract a*b+c: every FMA in the kernels is an explicit __fma_rn
    "-Xcompiler", "-fPIC",
]
NVCC_FLAGS += os.environ.get("SDCGYM_EXTRA_NVCC_FLAGS", "").split()  # experiments only


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libsdcgym.so cannot be built (no CPU fallback exists)")


def _sources_digest() -> str:
    h = hashlib.sha256()
    files = sorted(os.listdir(CSRC)) + ["../../include/sdcgym.h"]
    for name in files:
        path = os.path.join(CSRC, name)
        if os.path.isfile(path):
            h.update(name.encode())
            with open(path, "rb") as f:
                h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def _run(cmd):
    proc = subprocess.run(cmd, capture_output=True, text=True)
    if proc.returncode != 0:
        raise RuntimeError("command failed: %s\n%s\n%s" % (" ".join(cmd), proc.stdout, proc.stderr))
    return proc.stdout + proc.stderr


def build_library(force: bool = False, verbose: bool = False) -> str:
    digest = _sources_digest()
    stamp = os.path.join(OBJ_DIR, "digest.txt")
    if not force and os.path.exists(LIB_PATH) and os.path.exists(stamp):
        with open(stamp) as f:
            if f.read().strip() == digest:
                return LIB_PATH
    os.makedirs(OBJ_DIR, exist_ok=True)
    nvcc = _nvcc()
    jobs = []
    for M in M_VALUES:
        jobs.append(([nvcc, *NVCC_FLAGS, f"-DSDCGYM_M={M}", "-c", os.path.join(CSRC, "step_inst.cu"),
                      "-o", os.path.join(OBJ_DIR, f"step_m{M}.o")]))
    for name in ("sdcgym_abi", "specrad", "vecnorm", "hostpipe", "replay", "residual_sweeps", "residual_sweeps_sum"):
        src = os.path.join(CSRC, name + ".cu")
        if os.path.exists(src):
            # the spectral-radius kernel follows no prescribed rounding sequence: let it contract FMAs; the replay
            # sampler is built like vecnorm.cu, whose normalisation (normalize.cuh) it shares, and so is the K-sweep
            # residual loss and its reduced form, whose one-sweep counterpart lives in vecnorm.cu
            contract = ("specrad", "vecnorm", "replay", "residual_sweeps", "residual_sweeps_sum")
            flags = [f for f in NVCC_FLAGS if not (name in contract and f == "-fmad=false")]
            jobs.append([nvcc, *flags, "-c", src, "-o", os.path.join(OBJ_DIR, name + ".o")])
    workers = max(1, min(len(jobs), os.cpu_count() or 1))
    with concurrent.futures.ThreadPoolExecutor(workers) as ex:
        for out in ex.map(_run, jobs):
            if verbose and out.strip():
                print(out)
    objs = [j[-1] for j in jobs]
    _run([nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC", "-o", LIB_PATH, *objs])
    with open(stamp, "w") as f:
        f.write(digest)
    return LIB_PATH


if __name__ == "__main__":
    path = build_library(force="--force" in sys.argv, verbose=True)
    print(path)

"""`bench.py`: the `--impl reference` arm prints exactly one JSON line with the contract's keys (CPU); the arguments
are checked (CPU); `--dump-outputs` writes the same arrays for the same arguments (GPU)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    env = dict(os.environ, SDCGYM_BENCH_REF_SECONDS="0.2", SDCGYM_BENCH_REF_CORES="2", OPENBLAS_NUM_THREADS="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                          "--warmup", "3"], capture_output=True, text=True, env=env, timeout=300)
    assert out.returncode == 0, out.stderr
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "env-steps/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["steps"] == 2 and d["warmup"] == 3 and d["vs_baseline"] is None
    from oracle import ref_loader
    want = "reference" if ref_loader.reference_path() is not None else "port"  # the unmodified env when it is reachable
    assert d["cpu_baseline"]["kind"] == want and d["cpu_baseline"]["cores"] == 2 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["metric"].startswith("SDC env-steps/sec")
    # ranks other than 0 do no work and print nothing
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference"], capture_output=True,
                         text=True, env=dict(env, RANK="1", WORLD_SIZE="2"), timeout=60)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_steps_below_one_are_refused():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True,
                         timeout=120)
    assert out.returncode == 2 and "--steps" in out.stderr


@pytest.mark.gpu
def test_dump_outputs_are_the_same_for_the_same_arguments(tmp_path):
    """`--dump-outputs DIR`: float64 arrays of the last timed step, identical over two runs with the same arguments"""
    import numpy as np

    dumps = []
    for run in ("a", "b"):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--envs-per-gpu", "5000", "--steps", "3",
                              "--warmup", "3", "--no-secondary", "--no-cpu-baseline",
                              "--dump-outputs", str(tmp_path / run)], capture_output=True, text=True, timeout=600)
        assert out.returncode == 0, out.stderr[-2000:]
        lines = [l for l in out.stdout.splitlines() if l.strip()]
        assert len(lines) == 1
        line = json.loads(lines[0])
        assert line["steps"] == 3
        dumps.append({f[:-4]: np.load(tmp_path / run / f) for f in sorted(os.listdir(tmp_path / run))})
        # 5000 envs: the dump holds every env, so it must add up to the statistics the same run took from the env's
        # buffers after its last timed step (a warm-up step, other envs or wrong values would not)
        d, st = dumps[-1], line["rollout_stats"]
        flags = d["flags"].astype(np.uint8)
        assert d["niter"].sum() == st["sum_niter"]
        assert np.isclose(d["reward"].sum(), st["sum_reward"], rtol=1e-12, atol=0)  # summation order differs
        assert (flags & 2).astype(bool).sum() == st["converged"] and (flags & 4).astype(bool).sum() == st["diverged"]
    a, b = dumps
    assert sorted(a) == ["env_index", "flags", "lam", "niter", "residual", "reward", "terminal"]
    assert all(v.dtype == np.float64 for v in a.values())
    assert a["reward"].shape == (5000,) and a["lam"].shape == (5000, 2) and a["terminal"].shape == (20, 5000)
    assert np.array_equal(a["env_index"], np.arange(5000)) and a["niter"].min() >= 1
    assert sorted(b) == sorted(a)
    for k in a:
        assert np.array_equal(a[k].view(np.int64), b[k].view(np.int64)), k

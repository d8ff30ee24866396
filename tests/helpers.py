"""Shared helpers of the parity tests: golden-vector access and bit-level comparisons."""
from __future__ import annotations

import json
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN_DIR = os.path.join(HERE, "golden")
GOLDEN_JSON = os.path.join(GOLDEN_DIR, "sdc_golden.json")

_golden = None


def golden():
    """(manifest, {npz file name: arrays}); the manifest names the file of every case"""
    global _golden
    if _golden is None:
        with open(GOLDEN_JSON) as f:
            manifest = json.load(f)
        files = sorted({c["file"] for c in manifest["cases"]})
        _golden = (manifest, {f: np.load(os.path.join(GOLDEN_DIR, f)) for f in files})
    return _golden


def case_arrays(name):
    _, files = golden()
    arrays = files[case_meta(name)["file"]]
    prefix = name + "/"
    return {k[len(prefix):]: arrays[k] for k in arrays.files if k.startswith(prefix)}


def case_ids():
    manifest, _ = golden()
    return [c["name"] for c in manifest["cases"]]


def case_meta(name):
    manifest, _ = golden()
    return next(c for c in manifest["cases"] if c["name"] == name)


def same(a, b):
    """value-exact equality: every element equal (or both NaN).  +0 == -0 (sign of exact zeros is not pinned)."""
    a, b = np.asarray(a), np.asarray(b)
    if a.shape != b.shape:
        return False
    if np.iscomplexobj(a) or np.iscomplexobj(b):
        return same(a.real, b.real) and same(a.imag, b.imag)
    return bool(np.all((a == b) | (np.isnan(a) & np.isnan(b))))


def assert_same(a, b, what=""):
    a, b = np.asarray(a), np.asarray(b)
    if not same(a, b):
        bad = np.argwhere(~((a == b) | (np.isnan(a) & np.isnan(b)))) if a.shape == b.shape else None
        raise AssertionError(f"{what}: not bit-equal; first mismatches at {None if bad is None else bad[:5].tolist()}\n"
                             f"a={a.ravel()[:6]}\nb={b.ravel()[:6]}")


REWARD_RTOL = 1e-14  # rewards go through libm log/exp: reproducible to ~1 ulp only (SURVEY Appendix A)


def assert_reward_close(a, b, what=""):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    ok = np.abs(a - b) <= REWARD_RTOL * np.maximum(np.abs(a), np.abs(b)) + 0.0
    ok |= (a == b) | (np.isnan(a) & np.isnan(b))
    assert np.all(ok), f"{what}: rewards differ beyond {REWARD_RTOL} rel: {a[~ok][:5]} vs {b[~ok][:5]}"

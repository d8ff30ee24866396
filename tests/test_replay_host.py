"""CPU: the replay sampler's index function (sdc_gym_b200/csrc/replay_index.cuh, the header csrc/replay.cu
includes), compiled for the host, against its numpy restatement (sdc_gym_b200.replay.replay_indices) - the formula
tests/test_gpu_replay.py uses to predict the device's draws."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from sdc_gym_b200.replay import replay_indices

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("replay_shim") / "libreplay_shim.so")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-o", so,
                           os.path.join(HERE, "host_shim", "replay_shim.cpp")])
    L = ctypes.CDLL(so)
    L.shim_replay_indices.argtypes = [ctypes.c_uint64, ctypes.c_uint32, ctypes.c_int64, ctypes.c_uint32,
                                      ctypes.c_uint32, ctypes.c_void_p, ctypes.c_void_p]
    L.shim_replay_indices.restype = None
    return L


@pytest.mark.parametrize("seed", [0, 1, 0xDEADBEEFCAFEF00D])
@pytest.mark.parametrize("call", [0, 1, 77, 0xFFFFFFFF])
@pytest.mark.parametrize("upper,n_envs", [(1, 1), (1, 8), (5, 4096), (3, 33), (1000, 1 << 20), (7, 100003),
                                          ((1 << 32) - 1, (1 << 32) - 1)])
def test_host_build_of_the_index_function_matches_numpy(shim, seed, call, upper, n_envs):
    count = 2048
    rows, envs = np.zeros(count, np.uint32), np.zeros(count, np.uint32)
    shim.shim_replay_indices(seed, call, count, upper, n_envs, rows.ctypes.data, envs.ctypes.data)
    want_rows, want_envs = replay_indices(seed, call, np.arange(count), upper, n_envs)
    assert np.array_equal(rows.astype(np.int64), want_rows)
    assert np.array_equal(envs.astype(np.int64), want_envs)
    assert rows.max() < upper and envs.max() < n_envs
    if upper > 1:
        assert len(np.unique(rows)) > 1


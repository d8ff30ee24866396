"""ctypes binding of ``libsdcgym.so`` (C ABI declared in ``include/sdcgym.h``).

There is no CPU fallback: if the shared library is missing or a call fails, this module raises.
"""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SDCGYM_LIB") or os.path.join(_HERE, "libsdcgym.so")  # (SDCGYM_LIB: experiment builds)

MAX_M = 9
ABI_VERSION = 14

ENV_KINDS = {"sdc-v0": 0, "sdc-v1": 1}
PREC_TYPES = {"diag": 0, "lower_diag": 1, "lower_tri": 2, "strictly_lower_tri": 3, "fixed": 4}
REWARD_STRATEGIES = {
    "iteration_only": 0,
    "residual_change": 1,
    "gauss_kernel": 2,
    "fast_convergence": 3,
    "smooth_fast_convergence": 4,
    "smoother_fast_convergence": 5,
    "spectral_radius": 6,
}
FLAG_DONE, FLAG_CONVERGED, FLAG_ERR = 1, 2, 4
BLAS_SKYLAKEX, BLAS_HASWELL = 0, 1
ACTION_SCALE, ACTION_F32 = 1, 2  # bits of EnvDesc.do_scale (include/sdcgym.h)
SWEEP_MODES = {"exact": 0, "certified": 1}
CERT_PLANES = 8
PHASE_COUNTERS = 8  # SDCGYM_PHASE_COUNTERS

_c_double_p = ctypes.POINTER(ctypes.c_double)


class EnvDesc(ctypes.Structure):
    """struct sdcgym_env_desc"""

    _fields_ = [
        ("M", ctypes.c_int32),
        ("env_kind", ctypes.c_int32),
        ("prec_type", ctypes.c_int32),
        ("action_is_complex", ctypes.c_int32),
        ("do_scale", ctypes.c_int32),
        ("max_iters", ctypes.c_int32),
        ("reward_strategy", ctypes.c_int32),
        ("blas_variant", ctypes.c_int32),
        ("autoreset", ctypes.c_int32),
        ("curriculum", ctypes.c_int32),
        ("sweep_mode", ctypes.c_int32),
        ("reserved0", ctypes.c_int32),
        ("dt", ctypes.c_double),
        ("restol", ctypes.c_double),
        ("step_penalty", ctypes.c_double),
        ("residual_weight", ctypes.c_double),
        ("norm_factor", ctypes.c_double),
        ("lam_re_lo", ctypes.c_double),
        ("lam_re_hi", ctypes.c_double),
        ("lam_im_lo", ctypes.c_double),
        ("lam_im_hi", ctypes.c_double),
        ("interp_x0", ctypes.c_double),
        ("interp_x1", ctypes.c_double),
        ("seed", ctypes.c_uint64),
        ("env_offset", ctypes.c_int64),
        ("Q", ctypes.c_double * (MAX_M * MAX_M)),
        ("Qd_fixed", ctypes.c_double * (MAX_M * MAX_M)),
    ]


class State(ctypes.Structure):
    """struct sdcgym_state (device pointers as integers)"""

    _fields_ = [
        ("N", ctypes.c_int64),
        ("ld", ctypes.c_int64),
        ("lam", ctypes.c_void_p),
        ("S", ctypes.c_void_p),
        ("resnorm", ctypes.c_void_p),
        ("niter", ctypes.c_void_p),
        ("episodes", ctypes.c_void_p),
        ("rng_ctr", ctypes.c_void_p),
        ("norm_init", ctypes.c_void_p),
        ("cert", ctypes.c_void_p),
        ("fallback_list", ctypes.c_void_p),
        ("fallback_count", ctypes.c_void_p),
        ("phase_list", ctypes.c_void_p),
        ("phase_count", ctypes.c_void_p),
        ("phase_pinv", ctypes.c_void_p),
    ]


class StepIO(ctypes.Structure):
    """struct sdcgym_step_io"""

    _fields_ = [
        ("action", ctypes.c_void_p),
        ("action_env_stride", ctypes.c_int64),
        ("action_comp_stride", ctypes.c_int64),
        ("reward", ctypes.c_void_p),
        ("flags", ctypes.c_void_p),
        ("info_residual", ctypes.c_void_p),
        ("info_niter", ctypes.c_void_p),
        ("info_lam", ctypes.c_void_p),
        ("terminal_obs", ctypes.c_void_p),
        ("old_states", ctypes.c_void_p),
    ]


class RhoDesc(ctypes.Structure):
    """struct sdcgym_rho_desc"""

    _fields_ = [
        ("M", ctypes.c_int32),
        ("prec_type", ctypes.c_int32),
        ("qd_is_complex", ctypes.c_int32),
        ("qd_broadcast", ctypes.c_int32),
        ("dt", ctypes.c_double),
        ("Q", ctypes.c_double * (MAX_M * MAX_M)),
        ("Qd_fixed", ctypes.c_double * (MAX_M * MAX_M)),
        ("grid_re", ctypes.c_int64),
        ("grid_im", ctypes.c_int64),
        ("grid_first", ctypes.c_int64),
        ("re_lo", ctypes.c_double),
        ("re_hi", ctypes.c_double),
        ("im_lo", ctypes.c_double),
        ("im_hi", ctypes.c_double),
    ]


class LambdaGrid(ctypes.Structure):
    """struct sdcgym_lambda_grid"""

    _fields_ = [("n_re", ctypes.c_int64), ("n_im", ctypes.c_int64), ("first", ctypes.c_int64),
                ("re_lo", ctypes.c_double), ("re_hi", ctypes.c_double), ("im_lo", ctypes.c_double),
                ("im_hi", ctypes.c_double)]


class HostIO(ctypes.Structure):
    """struct sdcgym_host_io"""

    _fields_ = [
        ("action", ctypes.c_void_p),
        ("obs", ctypes.c_void_p),
        ("reward", ctypes.c_void_p),
        ("flags", ctypes.c_void_p),
        ("niter", ctypes.c_void_p),
        ("residual", ctypes.c_void_p),
        ("lam", ctypes.c_void_p),
    ]


class BlockLayout(ctypes.Structure):
    """struct sdcgym_block_layout"""

    _fields_ = [("N", ctypes.c_int64), ("M", ctypes.c_int32), ("reserved", ctypes.c_int32)] + [
        (k, ctypes.c_uint64) for k in ("obs_u", "reward", "residual", "lam", "niter", "flags", "obs_r", "total")]


class BlockIO(ctypes.Structure):
    """struct sdcgym_block_io"""

    _fields_ = [
        ("dev_block", ctypes.c_void_p),
        ("host_block", ctypes.c_void_p),
        ("action_dev", ctypes.c_void_p),
        ("action_host", ctypes.c_void_p),
        ("terminal_obs", ctypes.c_void_p),
        ("skip_u", ctypes.c_int32),
        ("chunks", ctypes.c_int32),
    ]


class DeviceGuard:
    """Makes ``device`` the current CUDA device for the duration of a ``with`` block (re-entrant, no-op when it
    already is): the C ABI launches on the calling thread's current device, streams and buffers belong to the
    env's device."""

    __slots__ = ("idx", "_stack", "_cuda")

    def __init__(self, device):
        import torch

        self._cuda = torch.cuda
        self.idx = device.index if device.index is not None else torch.cuda.current_device()
        self._stack = []

    def __enter__(self):
        cur = self._cuda.current_device()
        if cur != self.idx:
            self._cuda.set_device(self.idx)
            self._stack.append(cur)
        else:
            self._stack.append(-1)
        return self

    def __exit__(self, *exc):
        prev = self._stack.pop()
        if prev >= 0:
            self._cuda.set_device(prev)
        return False


def on_device(fn):
    """Method decorator: run with ``self._guard`` (a DeviceGuard) held."""
    import functools

    @functools.wraps(fn)
    def wrapper(self, *args, **kwargs):
        with self._guard:
            return fn(self, *args, **kwargs)

    return wrapper


class VecNorm(ctypes.Structure):
    """struct sdcgym_vecnorm"""

    _fields_ = [
        ("norm_obs", ctypes.c_int32), ("norm_reward", ctypes.c_int32), ("training", ctypes.c_int32),
        ("reserved", ctypes.c_int32),
        ("gamma", ctypes.c_double), ("epsilon", ctypes.c_double), ("clip_obs", ctypes.c_double),
        ("clip_reward", ctypes.c_double),
        ("obs_mean", ctypes.c_void_p), ("obs_var", ctypes.c_void_p), ("obs_count2", ctypes.c_void_p),
        ("ret_mean", ctypes.c_void_p), ("ret_var", ctypes.c_void_p), ("ret_count2", ctypes.c_void_p),
        ("returns", ctypes.c_void_p), ("scratch_obs", ctypes.c_void_p), ("scratch_ret", ctypes.c_void_p),
        ("sums_obs", ctypes.c_void_p), ("sums_ret", ctypes.c_void_p), ("out_planes", ctypes.c_void_p),
        ("out_reward", ctypes.c_void_p),
    ]


MAX_RANKS = 16


class Xchg(ctypes.Structure):
    """struct sdcgym_xchg"""

    _fields_ = [("world", ctypes.c_int32), ("rank", ctypes.c_int32), ("slot_doubles", ctypes.c_int32),
                ("reserved", ctypes.c_int32), ("seq", ctypes.c_uint64), ("peers", ctypes.c_void_p * MAX_RANKS)]


class Replay(ctypes.Structure):
    """struct sdcgym_replay"""

    _fields_ = [("P", ctypes.c_int32), ("A", ctypes.c_int32), ("rows", ctypes.c_int64), ("N", ctypes.c_int64),
                ("ld", ctypes.c_int64), ("seed", ctypes.c_uint64)] + [
        (k, ctypes.c_void_p) for k in ("obs", "next_obs", "actions", "rewards", "dones", "counters")]


class SdcGymError(RuntimeError):
    pass


_ERRORS = {-1: "SDCGYM_EINVAL (bad argument)", -2: "SDCGYM_EUNSUPPORTED", -3: "SDCGYM_ENULL (null pointer)",
           -4: "SDCGYM_ENOMEM"}

_lib = None


def load():
    """Load libsdcgym.so; raises if it has not been built (``python -m sdc_gym_b200.build``)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise SdcGymError(
            f"{LIB_PATH} not found: build it with `python -m sdc_gym_b200.build` (needs nvcc). "
            "There is no CPU fallback for the SDC kernels."
        )
    L = ctypes.CDLL(LIB_PATH)
    L.sdcgym_abi_version.restype = ctypes.c_int
    if L.sdcgym_abi_version() != ABI_VERSION:
        raise SdcGymError("libsdcgym.so ABI version mismatch; rebuild")
    vp, i64, dbl = ctypes.c_void_p, ctypes.c_int64, ctypes.c_double
    L.sdcgym_num_actions.argtypes = [ctypes.c_int, ctypes.c_int]
    L.sdcgym_supported.argtypes = [ctypes.c_int, ctypes.c_int]
    L.sdcgym_reset.argtypes = [ctypes.POINTER(EnvDesc), ctypes.POINTER(State), vp, vp, vp, vp]
    L.sdcgym_step.argtypes = [ctypes.POINTER(EnvDesc), ctypes.POINTER(State), ctypes.POINTER(StepIO), vp]
    L.sdcgym_export_obs.argtypes = [ctypes.c_int, i64, i64, vp, vp, vp]
    L.sdcgym_import_obs.argtypes = [ctypes.c_int, i64, i64, vp, vp, vp]
    L.sdcgym_refresh_resnorm.argtypes = [ctypes.c_int, i64, i64, vp, vp, vp]
    L.sdcgym_sum_f64.argtypes = [i64, vp, vp, vp, vp]
    L.sdcgym_sum_scratch_doubles.restype = ctypes.c_int
    L.sdcgym_fp64_peak_probe.argtypes = [i64, vp, _c_double_p, vp]
    if hasattr(L, "sdcgym_spectral_radius"):
        L.sdcgym_spectral_radius.argtypes = [ctypes.POINTER(RhoDesc), i64, vp, vp, vp, vp]
    L.sdcgym_spectral_radius_grad.argtypes = [ctypes.POINTER(RhoDesc), i64, vp, vp, vp, vp, vp]
    L.sdcgym_spectral_radius_grad.restype = ctypes.c_int
    L.sdcgym_spectral_radius_grad_sum_scratch_doubles.argtypes = [ctypes.c_int, ctypes.c_int, i64]
    L.sdcgym_spectral_radius_grad_sum_scratch_doubles.restype = i64
    L.sdcgym_spectral_radius_grad_sum.argtypes = [ctypes.POINTER(RhoDesc), i64, vp, vp, vp, vp, vp, vp]
    L.sdcgym_spectral_radius_grad_sum.restype = ctypes.c_int
    dp_ = ctypes.POINTER(RhoDesc)
    L.sdcgym_residual_step.argtypes = [dp_, i64, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    L.sdcgym_residual_sweeps.argtypes = [dp_, i64, ctypes.c_int, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    L.sdcgym_residual_sweeps_sum.argtypes = [dp_, i64, ctypes.c_int, ctypes.c_int, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    L.sdcgym_full_solve_counts.argtypes = [ctypes.POINTER(EnvDesc), ctypes.POINTER(LambdaGrid), i64, vp, vp, i64, i64,
                                           vp, vp, vp, vp, vp, vp]
    L.sdcgym_full_solve_counts.restype = ctypes.c_int
    L.sdcgym_full_solve_counts_population.argtypes = [ctypes.POINTER(EnvDesc), ctypes.POINTER(LambdaGrid), i64, vp,
                                                      i64, vp, i64, i64, vp, vp]
    L.sdcgym_full_solve_counts_population.restype = ctypes.c_int
    L.sdcgym_spectral_radius_grad_sum_population.argtypes = [dp_, i64, vp, i64, vp, i64, vp, vp, vp]
    L.sdcgym_spectral_radius_grad_sum_population.restype = ctypes.c_int
    L.sdcgym_vecnorm_scratch_doubles.argtypes = [ctypes.c_int]
    L.sdcgym_vecnorm_accumulate.argtypes = [ctypes.c_int, i64, i64, vp, vp, vp, vp, vp]
    L.sdcgym_vecnorm_merge.argtypes = [ctypes.c_int, dbl, vp, vp, vp, vp, vp]
    L.sdcgym_vecnorm_update.argtypes = [ctypes.c_int, i64, i64, vp, vp, vp, vp, vp, vp, vp]
    L.sdcgym_vecnorm_update_returns.argtypes = [i64, vp, dbl, vp, vp, vp, vp, vp, vp, vp]
    L.sdcgym_vecnorm_apply.argtypes = [ctypes.c_int, i64, i64, vp, vp, vp, dbl, dbl, vp, vp]
    L.sdcgym_xchg_bytes.argtypes = [ctypes.c_int, ctypes.c_int]
    L.sdcgym_xchg_bytes.restype = ctypes.c_size_t
    L.sdcgym_vecnorm_update_dist.argtypes = [ctypes.c_int, i64, i64, vp, vp, vp, vp, vp, vp, ctypes.POINTER(Xchg), vp]
    L.sdcgym_vecnorm_update_returns_dist.argtypes = [i64, vp, dbl, vp, vp, vp, vp, vp, vp, ctypes.POINTER(Xchg), vp]
    L.sdcgym_vecnorm_update_both.argtypes = [ctypes.c_int, i64, i64, vp, vp, dbl, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp,
                                             ctypes.POINTER(Xchg), vp]
    L.sdcgym_vecnorm_update_both.restype = ctypes.c_int
    L.sdcgym_ipc_alloc.argtypes = [ctypes.c_size_t, ctypes.POINTER(vp), ctypes.c_char_p]
    L.sdcgym_ipc_open.argtypes = [ctypes.c_char_p, ctypes.POINTER(vp)]
    L.sdcgym_ipc_close.argtypes = [vp]
    L.sdcgym_ipc_free.argtypes = [vp]
    for name in ("sdcgym_vecnorm_update_dist", "sdcgym_vecnorm_update_returns_dist", "sdcgym_ipc_alloc",
                 "sdcgym_ipc_open", "sdcgym_ipc_close", "sdcgym_ipc_free"):
        getattr(L, name).restype = ctypes.c_int
    L.sdcgym_vecnorm_returns.argtypes = [i64, vp, dbl, vp, vp]
    L.sdcgym_vecnorm_reward.argtypes = [i64, vp, vp, vp, dbl, dbl, ctypes.c_int, vp, vp, vp]
    L.sdcgym_pipe_create.argtypes = [ctypes.c_int, ctypes.POINTER(vp)]
    L.sdcgym_pipe_destroy.argtypes = [vp]
    L.sdcgym_pipe_step.argtypes = [vp, ctypes.POINTER(EnvDesc), ctypes.POINTER(State), ctypes.POINTER(StepIO), vp,
                                   ctypes.POINTER(HostIO), ctypes.c_int, vp]
    L.sdcgym_pipe_step_vecnorm.argtypes = [vp, ctypes.POINTER(EnvDesc), ctypes.POINTER(State), ctypes.POINTER(StepIO), vp,
                                           ctypes.POINTER(HostIO), ctypes.POINTER(VecNorm), vp]
    L.sdcgym_export_rows.argtypes = [ctypes.c_int, i64, i64, vp, vp, vp]
    L.sdcgym_block_layout_init.argtypes = [ctypes.c_int, i64, ctypes.POINTER(BlockLayout)]
    L.sdcgym_pipe_step_block.argtypes = [vp, ctypes.POINTER(EnvDesc), ctypes.POINTER(State), ctypes.POINTER(BlockLayout),
                                         ctypes.POINTER(BlockIO), ctypes.POINTER(VecNorm), vp]
    for name in ("sdcgym_export_rows", "sdcgym_block_layout_init", "sdcgym_pipe_step_block"):
        getattr(L, name).restype = ctypes.c_int
    L.sdcgym_host_alloc.argtypes = [ctypes.c_size_t, ctypes.POINTER(vp)]
    L.sdcgym_host_free.argtypes = [vp]
    for name in ("sdcgym_pipe_create", "sdcgym_pipe_destroy", "sdcgym_pipe_step", "sdcgym_pipe_step_vecnorm",
                 "sdcgym_host_alloc", "sdcgym_host_free"):
        getattr(L, name).restype = ctypes.c_int
    L.sdcgym_gae.argtypes = [ctypes.c_int, i64, vp, vp, vp, vp, vp, dbl, dbl, vp, vp, vp]
    L.sdcgym_gae.restype = ctypes.c_int
    rp = ctypes.POINTER(Replay)
    L.sdcgym_replay_store_obs.argtypes = [rp, vp, i64, vp]
    L.sdcgym_replay_store.argtypes = [rp, vp, vp, i64, vp, vp, vp, i64, vp]
    L.sdcgym_replay_sample.argtypes = [rp, i64, vp, vp, vp, dbl, dbl, dbl, vp, vp, vp, vp, vp, vp]
    for name in ("sdcgym_replay_store_obs", "sdcgym_replay_store", "sdcgym_replay_sample"):
        getattr(L, name).restype = ctypes.c_int
    for name in ("sdcgym_residual_step", "sdcgym_residual_sweeps", "sdcgym_residual_sweeps_sum", "sdcgym_vecnorm_scratch_doubles", "sdcgym_vecnorm_accumulate",
                 "sdcgym_vecnorm_merge", "sdcgym_vecnorm_update", "sdcgym_vecnorm_update_returns", "sdcgym_vecnorm_apply", "sdcgym_vecnorm_returns", "sdcgym_vecnorm_reward"):
        getattr(L, name).restype = ctypes.c_int
    for name in ("sdcgym_num_actions", "sdcgym_supported", "sdcgym_reset", "sdcgym_step", "sdcgym_export_obs",
                 "sdcgym_import_obs", "sdcgym_refresh_resnorm", "sdcgym_sum_f64", "sdcgym_fp64_peak_probe",
                 "sdcgym_spectral_radius"):
        if hasattr(L, name):
            getattr(L, name).restype = ctypes.c_int
    _lib = L
    return L


def check(rc: int, what: str):
    if rc == 0:
        return
    if rc < 0:
        raise SdcGymError(f"{what}: {_ERRORS.get(rc, rc)}")
    raise SdcGymError(f"{what}: CUDA error {rc}")


def exported_symbols():
    """Names of all ``sdcgym_*`` entry points declared in include/sdcgym.h (parsed from the header)."""
    import re

    header = os.path.join(os.path.dirname(_HERE), "include", "sdcgym.h")
    with open(header) as f:
        text = f.read()
    return sorted(set(re.findall(r"\b(?:int|int64_t|size_t)\s+(sdcgym_[a-z0-9_]+)\s*\(", text)))

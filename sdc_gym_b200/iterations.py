"""Iteration counts and success rate of the ``sdc-v0`` full solve over a lambda batch or a lambda grid.

The reference judges a Q_delta by ``test_model`` / ``run_tests`` (``rl_playground.py:147-156``,
``dp_playground.py:844-957``): one ``sdc-v0`` episode per lambda, then the mean iteration count over the successful
episodes and the success rate, with success = ``niter < 50 and residual < restol``.  ``IterationCounts`` evaluates
those episodes without an env: ``sdcgym_full_solve_counts`` runs the env's own full-solve kernel body from the reset
state, so each node's ``niter``, ``residual`` and flags are bit-equal to ``make("sdc-v0", ...)`` after
``reset(lam=[lam])`` and ``step_tensor(row)``.  Grid lambdas are generated on the device and are the nodes of
``SpectralRadiusLoss.grid``, bit for bit; the summaries reduce to a histogram on the device.
"""
from __future__ import annotations

import ctypes

import numpy as np

from . import _lib
from .collocation import collocation_matrix
from .precond import PREC_TYPES, fixed_preconditioner, num_actions
from .vec_env import MAX_ITERS, detect_blas_variant


def _torch():
    import torch

    return torch


def count_stats(hist, max_iters):
    """``test_model``'s numbers from histograms ``hist`` (numpy int64 [..., max_iters + 3]), each a numpy array over
    the leading axes: (count, n_err, n_exhausted, n_success, success_rate, mean_niter).  Success is a converged episode
    whose niter is below 50; ``mean_niter`` is 666.0 where nothing succeeds and ``success_rate`` 0.0 for an empty set."""
    h = np.asarray(hist)
    ns = min(MAX_ITERS, max_iters + 1)
    count = h.sum(-1)
    n_success = h[..., :ns].sum(-1)
    rate = np.where(count > 0, n_success / np.maximum(count, 1), 0.0)
    mean = np.where(n_success > 0, np.sum(np.arange(ns) * h[..., :ns], -1) / np.maximum(n_success, 1), 666.0)
    return count, h[..., max_iters + 1], h[..., max_iters + 2], n_success, rate, mean


class CountSummary:
    """What ``test_model`` reports for a set of episodes, from the device histogram ``hist_device`` (int64
    [max_iters + 3]: niter of the converged episodes, then the err count, then the count of episodes that ran out of
    sweeps).  The histogram is copied to the host once, on first use.

    Success is ``niter < 50 and residual < restol``: a converged episode whose niter is below 50.  An episode that
    converges on its 50th sweep is not a success.  ``mean_niter`` is the mean niter of the successes, 666 when there
    are none (the reference's value); ``success_rate`` is 0 for an empty set.  An err episode never counts as a
    success here; the reference's literal test would count one whose residual, after growing 100-fold in one sweep,
    is still below restol, which needs ||r_0|| < restol / 100."""

    def __init__(self, hist_device, max_iters=MAX_ITERS):
        self.hist_device = hist_device
        self.max_iters = int(max_iters)
        self._hist = None

    @property
    def hist(self):
        if self._hist is None:
            self._hist = self.hist_device.cpu().numpy()
        return self._hist

    def _stats(self):
        return count_stats(self.hist, self.max_iters)

    @property
    def n_err(self):
        return int(self._stats()[1])

    @property
    def n_exhausted(self):
        return int(self._stats()[2])

    @property
    def count(self):
        return int(self._stats()[0])

    @property
    def n_success(self):
        return int(self._stats()[3])

    @property
    def success_rate(self):
        return float(self._stats()[4])

    @property
    def mean_niter(self):
        mean = float(self._stats()[5])
        return 666 if self.n_success == 0 else mean

    def __repr__(self):
        return (f"CountSummary(count={self.count}, success_rate={self.success_rate:.6f}, "
                f"mean_niter={self.mean_niter}, n_err={self.n_err}, n_exhausted={self.n_exhausted})")


class PopulationSummary:
    """``CountSummary`` for each of P action rows, from the device histograms ``hist_device`` (int64
    [P, max_iters + 3]), copied to the host once, on first use.  ``count``, ``n_err``, ``n_exhausted``,
    ``n_success``, ``success_rate`` and ``mean_niter`` are numpy arrays (P,) with ``CountSummary``'s rules (666.0
    where nothing succeeds); ``summary[p]`` is row p's ``CountSummary``."""

    def __init__(self, hist_device, max_iters=MAX_ITERS):
        self.hist_device = hist_device
        self.max_iters = int(max_iters)
        self._hist = None

    def __len__(self):
        return int(self.hist_device.shape[0])

    @property
    def hist(self):
        if self._hist is None:
            self._hist = self.hist_device.cpu().numpy()
        return self._hist

    def __getitem__(self, p):
        s = CountSummary(self.hist_device[p], self.max_iters)
        s._hist = self.hist[p]
        return s

    count = property(lambda self: count_stats(self.hist, self.max_iters)[0])
    n_err = property(lambda self: count_stats(self.hist, self.max_iters)[1])
    n_exhausted = property(lambda self: count_stats(self.hist, self.max_iters)[2])
    n_success = property(lambda self: count_stats(self.hist, self.max_iters)[3])
    success_rate = property(lambda self: count_stats(self.hist, self.max_iters)[4])
    mean_niter = property(lambda self: count_stats(self.hist, self.max_iters)[5])

    def __repr__(self):
        return f"PopulationSummary(P={len(self)}, success_rate={self.success_rate}, mean_niter={self.mean_niter})"


class IterationCounts:
    """The ``sdc-v0`` full solve from the reset state for lambdas from a list or a grid (``sdcgym_full_solve_counts``).

    The keywords are ``SDCVecEnv``'s; the defaults are those ``run_tests`` evaluates with (``do_scale=False``,
    ``free_action_space=True``).  ``prec`` ('LU', 'min', 'EE', 'zeros') fixes Q_delta; otherwise every call takes
    action rows in the ``prec_type`` layout, with the dtype rules of ``SDCVecEnv.step_tensor``: complex rows need
    ``free_action_space``, real rows are read as complex with ``free_action_space``, and under ``use_doubles=False``
    the scaled entries are rounded to float32 as the env does.  ``actions`` is (N, n_act), one row per lambda, or one
    row (n_act,) / (1, n_act) shared by every lambda (read in place)."""

    def __init__(self, M, dt, restol, prec_type="diag", *, prec=None, do_scale=False, free_action_space=True,
                 use_doubles=True, blas_variant=None, device=None):
        torch = _torch()
        if prec is None and prec_type not in PREC_TYPES:
            raise ValueError(f"unknown prec_type {prec_type!r}")
        if not torch.cuda.is_available():
            raise _lib.SdcGymError("IterationCounts needs a CUDA device: there is no CPU fallback")
        self._L = _lib.load()
        self.M, self.dt, self.restol = int(M), float(dt), float(restol)
        self.prec = prec
        self.prec_type = "fixed" if prec is not None else prec_type
        if not self._L.sdcgym_supported(self.M, _lib.PREC_TYPES[self.prec_type]):
            raise NotImplementedError(f"M={self.M}, prec_type={self.prec_type} has no compiled kernel")
        self.free_action_space = bool(free_action_space)
        self.n_act = 0 if prec is not None else num_actions(self.M, prec_type)
        self.max_iters = MAX_ITERS
        self.Q = collocation_matrix(self.M)
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        d = _lib.EnvDesc()
        d.M, d.env_kind, d.prec_type = self.M, _lib.ENV_KINDS["sdc-v0"], _lib.PREC_TYPES[self.prec_type]
        d.action_is_complex = int(self.free_action_space)
        d.do_scale = (_lib.ACTION_SCALE if do_scale else 0) | (0 if use_doubles else _lib.ACTION_F32)
        d.max_iters = self.max_iters
        d.reward_strategy = _lib.REWARD_STRATEGIES["iteration_only"]
        d.blas_variant = detect_blas_variant() if blas_variant is None else int(blas_variant)
        d.dt, d.restol, d.norm_factor = self.dt, self.restol, 1.0
        for k, v in enumerate(self.Q.reshape(-1)):
            d.Q[k] = float(v)
        if prec is not None:
            for k, v in enumerate(fixed_preconditioner(prec, self.M, self.Q).reshape(-1)):
                d.Qd_fixed[k] = float(v)
        self.blas_variant = d.blas_variant
        self._desc = d
        self._guard = _lib.DeviceGuard(self.device)

    # ------------------------------------------------------------------ plumbing
    def _stream(self):
        return ctypes.c_void_p(_torch().cuda.current_stream(self.device).cuda_stream)

    def _action_tensor(self, actions):
        torch = _torch()
        t = actions if isinstance(actions, torch.Tensor) else torch.as_tensor(np.array(actions))
        if not (t.is_floating_point() or t.is_complex()):
            raise TypeError(f"actions must be real or complex floating point, not {t.dtype}")
        if t.is_complex() and not self.free_action_space:
            raise TypeError("complex actions need free_action_space=True")
        return t

    def _device_rows(self, t):
        """the rows as step_tensor reads them: complex128 (viewed as pairs) with free_action_space, else float64"""
        torch = _torch()
        t = t.to(self.device)
        return torch.view_as_real(t.to(torch.complex128).contiguous()) if self.free_action_space \
            else t.to(torch.float64).contiguous()

    def _rows(self, actions, N, grid):
        """(tensor kept alive, pointer, env stride, component stride) of the action rows, as step_tensor reads them"""
        if self.prec is not None:
            if actions is not None:
                raise ValueError(f"prec={self.prec!r} fixes Q_delta: no actions")
            return None, None, 0, 0
        if actions is None:
            raise ValueError("actions required (no fixed prec)")
        t = self._action_tensor(actions)
        if t.dim() == 1:
            t = t.reshape(1, -1)
        if t.dim() != 2 or t.shape[1] != self.n_act:
            raise ValueError(f"actions must have shape (N, {self.n_act}) or ({self.n_act},)")
        shared = t.shape[0] == 1
        if not shared and (grid or t.shape[0] != N):
            raise ValueError(f"actions must be one row ({self.n_act},) in grid mode" if grid else
                             f"actions must have shape ({N}, {self.n_act}) or ({self.n_act},)")
        a = self._device_rows(t)
        return a, a.data_ptr(), 0 if shared else a.stride(0), a.stride(1)

    def _population(self, population):
        """(tensor kept alive, row stride, component stride) of P candidate rows (P, n_act)"""
        if self.prec is not None:
            raise ValueError(f"prec={self.prec!r} fixes Q_delta: a population has no rows")
        t = self._action_tensor(population)
        if t.dim() != 2 or t.shape[0] < 1 or t.shape[1] != self.n_act:
            raise ValueError(f"population must have shape (P, {self.n_act}) with P >= 1, not {tuple(t.shape)}")
        a = self._device_rows(t)
        return a, a.stride(0), a.stride(1)

    def _run_population(self, N, lam_r, grid, population):
        """hist (P, max_iters + 3) of sdcgym_full_solve_counts_population"""
        torch = _torch()
        a, rs, cs = self._population(population)
        P = a.shape[0]
        hist = torch.empty((P, self.max_iters + 3), dtype=torch.int64, device=self.device)
        _lib.check(self._L.sdcgym_full_solve_counts_population(
            ctypes.byref(self._desc), None if grid is None else ctypes.byref(grid), N,
            None if lam_r is None else lam_r.data_ptr(), P, a.data_ptr(), rs, cs, hist.data_ptr(), self._stream()),
            "sdcgym_full_solve_counts_population")
        self._keep = (a, lam_r)
        return hist

    def _lams(self, lams):
        torch = _torch()
        lam = lams if isinstance(lams, torch.Tensor) else torch.as_tensor(np.asarray(lams, dtype=np.complex128))
        if not (lam.is_floating_point() or lam.is_complex()):
            lam = lam.to(torch.float64)
        lam = lam.to(self.device).to(torch.complex128).reshape(-1).contiguous()
        return torch.view_as_real(lam)

    def _run(self, N, lam_r, grid, actions, per_node, hist=None, with_lam=False):
        torch = _torch()
        a, aptr, es, cs = self._rows(actions, N, grid is not None)
        dev = self.device
        niter = torch.empty(N, dtype=torch.int32, device=dev) if per_node else None
        res = torch.empty(N, dtype=torch.float64, device=dev) if per_node else None
        flags = torch.empty(N, dtype=torch.uint8, device=dev) if per_node else None
        lam_out = torch.empty((N, 2), dtype=torch.float64, device=dev) if with_lam else None
        ptr = lambda t: None if t is None else t.data_ptr()  # noqa: E731
        _lib.check(self._L.sdcgym_full_solve_counts(
            ctypes.byref(self._desc), None if grid is None else ctypes.byref(grid), N, ptr(lam_r), aptr, es, cs,
            ptr(niter), ptr(res), ptr(flags), ptr(lam_out), ptr(hist), self._stream()), "sdcgym_full_solve_counts")
        self._keep = (a, lam_r)
        return niter, res, flags, lam_out

    @staticmethod
    def _grid(n_re, n_im, re_iv, im_iv, lo):
        g = _lib.LambdaGrid()
        g.n_re, g.n_im, g.first = int(n_re), int(n_im), int(lo) * int(n_im)
        g.re_lo, g.re_hi = float(re_iv[0]), float(re_iv[1])
        g.im_lo, g.im_hi = float(im_iv[0]), float(im_iv[1])
        return g

    def _hist(self):
        torch = _torch()
        return torch.empty(self.max_iters + 3, dtype=torch.int64, device=self.device)

    # ------------------------------------------------------------------ public
    @_lib.on_device
    def solve(self, lams, actions=None):
        """(niter int32, residual float64, flags uint8) CUDA tensors (N,): ``info['niter']``, ``info['residual']`` and
        the env's ``flags`` of one ``sdc-v0`` episode per lambda.  ``lams``: (N,) complex (numpy or torch)."""
        lam_r = self._lams(lams)
        niter, res, flags, _ = self._run(lam_r.shape[0], lam_r, None, actions, True)
        return niter, res, flags

    @_lib.on_device
    def grid(self, n_re, n_im, lambda_real_interval, lambda_imag_interval, action=None, rows=None, return_lam=False):
        """``solve`` on the (n_re x n_im) lambda grid of ``SpectralRadiusLoss.grid`` (same nodes, bit for bit),
        lambdas generated on the device, for ONE action row (or the fixed ``prec``).  Returns (niter, residual,
        flags) maps (n_re, n_im), or (hi - lo, n_im) with ``rows=(lo, hi)``; ``return_lam`` adds the (.., n_im)
        complex128 map of the lambdas the nodes ran with."""
        torch = _torch()
        n_re, n_im = int(n_re), int(n_im)
        lo, hi = (0, n_re) if rows is None else (int(rows[0]), int(rows[1]))
        if not 0 <= lo <= hi <= n_re:
            raise ValueError(f"rows={rows} outside the grid of {n_re} rows")
        N = (hi - lo) * n_im
        g = self._grid(n_re, n_im, lambda_real_interval, lambda_imag_interval, lo)
        niter, res, flags, lam = self._run(N, None, g, action, True, with_lam=return_lam)
        out = tuple(t.reshape(hi - lo, n_im) for t in (niter, res, flags))
        if return_lam:
            out += (torch.view_as_complex(lam).reshape(hi - lo, n_im),)
        return out

    @_lib.on_device
    def summary(self, lams, actions=None):
        """``CountSummary`` of one episode per lambda: the histogram is accumulated on the device, no per-node array is
        written, and reading the summary copies max_iters + 3 integers."""
        lam_r = self._lams(lams)
        hist = self._hist()
        self._run(lam_r.shape[0], lam_r, None, actions, False, hist)
        return CountSummary(hist, self.max_iters)

    def grid_summary(self, n_re, n_im, lambda_real_interval, lambda_imag_interval, action=None, rows=None):
        """``summary`` over the grid of ``grid``.  ``rows=None``: the whole grid, its rows sharded over the ranks of
        the default process group (``dist.shard_range``) and the histogram all-reduced once; ``rows=(lo, hi)``: grid
        rows lo..hi-1 only, no collective call (an empty range gives a zero histogram).  Makes no host
        synchronisation, so a single process can capture it in a CUDA graph."""
        from . import dist as _dist

        @_lib.on_device
        def rows_hist(self, lo, hi):
            hist = self._hist()
            g = self._grid(n_re, n_im, lambda_real_interval, lambda_imag_interval, lo)
            self._run((hi - lo) * int(n_im), None, g, action, False, hist)  # N = 0 zeroes hist
            return hist

        hist, _ = _dist.sharded_rows_sum(n_re, rows, lambda lo, hi: rows_hist(self, lo, hi))
        return CountSummary(hist, self.max_iters)

    @_lib.on_device
    def population_summary(self, lams, population):
        """``summary`` for each row of ``population`` (P, n_act), every row shared by all lambdas, in one launch
        (``sdcgym_full_solve_counts_population``).  Returns a ``PopulationSummary``; row p equals ``summary(lams,
        population[p])``, bit for bit.  The dtype rules are those of ``summary``."""
        lam_r = self._lams(lams)
        return PopulationSummary(self._run_population(lam_r.shape[0], lam_r, None, population), self.max_iters)

    def population_grid_summary(self, n_re, n_im, lambda_real_interval, lambda_imag_interval, population, rows=None):
        """``grid_summary`` for each row of ``population`` (P, n_act) in one launch per shard.  ``rows=None``: grid rows
        sharded over the ranks of the default process group with one all-reduce of the (P, max_iters + 3) histograms;
        ``rows=(lo, hi)``: grid rows lo..hi-1 only, no collective call.  Returns a ``PopulationSummary``."""
        from . import dist as _dist

        @_lib.on_device
        def rows_hist(self, lo, hi):
            g = self._grid(n_re, n_im, lambda_real_interval, lambda_imag_interval, lo)
            return self._run_population((hi - lo) * int(n_im), None, g, population)  # N = 0 zeroes hist

        hist, _ = _dist.sharded_rows_sum(n_re, rows, lambda lo, hi: rows_hist(self, lo, hi))
        return PopulationSummary(hist, self.max_iters)

"""Batched forward values of the ``dp_playground.py`` losses on the device.

``SpectralRadiusLoss(M, dt, prec_type)(lams, outputs)`` mirrors ``dp_playground.py:186-231``: the mean over the
batch of ``rho(lam*dt * inv(I - lam*dt*Qd) @ (Q - Qd))`` with ``Qd = get_qdmat(output)``.  The reference runs
``jnp.linalg.inv`` + ``jnp.linalg.eigvals`` per sample on the CPU (it forces JAX onto the CPU because eigvals
has no GPU kernel, ``dp_playground.py:981-985``); here one thread per sample runs a complex Hessenberg-QR
(``csrc/specrad.cuh``) - 1e-10 relative agreement with LAPACK is the contract, not bit equality.
"""
from __future__ import annotations

import ctypes

import numpy as np

from . import _lib
from .collocation import collocation_matrix
from .precond import PREC_TYPES, fixed_preconditioner, num_actions


class UnknownPrecTypeError(ValueError):
    pass


def _torch():
    import torch

    return torch


class SpectralRadiusLoss:
    def __init__(self, M, dt, prec_type="diag", *, prec=None, Q=None, device=None):
        if prec is None and prec_type not in PREC_TYPES:
            raise UnknownPrecTypeError(prec_type)
        torch = _torch()
        if not torch.cuda.is_available():
            raise _lib.SdcGymError("SpectralRadiusLoss needs a CUDA device: there is no CPU fallback")
        self._L = _lib.load()
        self.M, self.dt = int(M), float(dt)
        self.prec = prec
        self.prec_type = "fixed" if prec is not None else prec_type
        self.Q = collocation_matrix(self.M) if Q is None else np.ascontiguousarray(Q, dtype=np.float64)
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.n_out = 0 if prec is not None else num_actions(self.M, prec_type)
        d = _lib.RhoDesc()
        d.M, d.prec_type, d.dt = self.M, _lib.PREC_TYPES[self.prec_type], self.dt
        for k, v in enumerate(self.Q.reshape(-1)):
            d.Q[k] = float(v)
        if prec is not None:
            for k, v in enumerate(fixed_preconditioner(prec, self.M, self.Q).reshape(-1)):
                d.Qd_fixed[k] = float(v)
        self._desc = d
        self._guard = _lib.DeviceGuard(self.device)

    def _stream(self):
        return ctypes.c_void_p(_torch().cuda.current_stream(self.device).cuda_stream)

    def _outputs_tensor(self, outputs, B):
        torch = _torch()
        if self.prec is not None:
            return None, 0, 0
        t = outputs if isinstance(outputs, torch.Tensor) else torch.as_tensor(np.array(outputs))
        t = t.to(self.device)
        is_c = t.is_complex()
        t = t.to(torch.complex128 if is_c else torch.float64)
        if t.dim() == 1:
            t = t.reshape(1, -1)
        if t.shape[-1] != self.n_out:
            raise ValueError(f"outputs must have {self.n_out} components for prec_type={self.prec_type}")
        broadcast = int(t.shape[0] == 1 and B != 1)
        if not broadcast and t.shape[0] != B:
            raise ValueError("outputs and lams disagree on the batch size")
        t = t.contiguous()
        return (torch.view_as_real(t).contiguous() if is_c else t), int(is_c), broadcast

    @_lib.on_device
    def spectral_radii(self, lams, outputs=None):
        """rho per sample as a CUDA float64 tensor (B,).  ``lams``: (B,) or (B, 1) complex (numpy or torch)."""
        torch = _torch()
        lam = lams if isinstance(lams, torch.Tensor) else torch.as_tensor(np.asarray(lams, dtype=np.complex128))
        lam = lam.to(self.device).to(torch.complex128).reshape(-1).contiguous()
        B = lam.numel()
        if B == 0:  # an empty shard: nothing to launch (a NULL lambda pointer would select grid mode in the ABI)
            return torch.empty(0, dtype=torch.float64, device=self.device)
        qd, is_c, bc = self._outputs_tensor(outputs, B)
        d = self._desc
        d.qd_is_complex, d.qd_broadcast = is_c, bc
        d.grid_re = d.grid_im = 0
        rho = torch.empty(B, dtype=torch.float64, device=self.device)
        lam_r = torch.view_as_real(lam)
        _lib.check(self._L.sdcgym_spectral_radius(ctypes.byref(d), B, lam_r.data_ptr(),
                                                  None if qd is None else qd.data_ptr(), rho.data_ptr(),
                                                  self._stream()), "sdcgym_spectral_radius")
        self._keep = (lam_r, qd)
        return rho

    def __call__(self, lams, outputs=None):
        """mean spectral radius over the batch (``jnp.mean(jax.vmap(...))``, dp_playground.py:230-231)."""
        rho = self.spectral_radii(lams, outputs)
        return self.mean(rho)

    @_lib.on_device
    def radii_and_grads(self, lams, outputs):
        """(rho (B,), g (B, n_out) complex128) with d rho_b = Re(sum_k g_bk d output_bk): per-sample spectral
        radius and its derivative with respect to the Q_delta parameters (left/right eigenvector formula,
        ``csrc/specrad.cuh``).  Valid where the dominant eigenvalue is simple."""
        torch = _torch()
        if self.prec is not None:
            raise ValueError("a fixed preconditioner has no parameters to differentiate")
        lam = lams if isinstance(lams, torch.Tensor) else torch.as_tensor(np.asarray(lams, dtype=np.complex128))
        lam = lam.detach().to(self.device).to(torch.complex128).reshape(-1).contiguous()
        B = lam.numel()
        if B == 0:
            return (torch.empty(0, dtype=torch.float64, device=self.device),
                    torch.empty((0, self.n_out), dtype=torch.complex128, device=self.device))
        out = outputs.detach() if isinstance(outputs, torch.Tensor) else outputs
        qd, is_c, bc = self._outputs_tensor(out, B)
        if bc:
            qd = qd.expand(B, *qd.shape[1:]).contiguous()
        d = self._desc
        d.qd_is_complex, d.qd_broadcast = is_c, 0
        d.grid_re = d.grid_im = 0
        rho = torch.empty(B, dtype=torch.float64, device=self.device)
        grad = torch.empty((B, self.n_out, 2), dtype=torch.float64, device=self.device)
        lam_r = torch.view_as_real(lam)
        _lib.check(self._L.sdcgym_spectral_radius_grad(ctypes.byref(d), B, lam_r.data_ptr(), qd.data_ptr(),
                                                       rho.data_ptr(), grad.data_ptr(), self._stream()),
                   "sdcgym_spectral_radius_grad")
        self._keep = (lam_r, qd)
        return rho, torch.view_as_complex(grad)

    def value_and_grad(self, lams, outputs, convention="jax"):
        """(mean rho, d mean_rho / d outputs) - what ``jax.value_and_grad(loss)`` gives the reference's trainer for
        the loss itself (``dp_playground.py:1038-1073``).  For complex ``outputs`` the gradient follows
        ``convention``: 'jax' (``d/dx - i d/dy``) or 'torch' (its conjugate); for real outputs it is real."""
        torch = _torch()
        rho, g = self.radii_and_grads(lams, outputs)
        g = g / rho.numel()
        is_c = (outputs.is_complex() if isinstance(outputs, torch.Tensor) else np.iscomplexobj(outputs))
        if not is_c:
            g = g.real
        elif convention == "torch":
            g = g.conj()
        elif convention != "jax":
            raise ValueError("convention must be 'jax' or 'torch'")
        return self.mean(rho), g

    def differentiable(self, lams, outputs):
        """Mean spectral radius as a torch scalar that supports ``.backward()`` into ``outputs`` (a CUDA tensor with
        ``requires_grad``) - forward and backward both run the hand-written kernels.  A single parameter row,
        shape (n_out,) or (1, n_out), shared by every lambda goes through ``shared_value_and_grad``."""
        if outputs.ndim == 1 or (outputs.ndim == 2 and outputs.shape[0] == 1):
            return _SharedRowFn.apply(outputs, lambda o, conv: self.shared_value_and_grad(lams, o, conv))
        return _SpectralRadiusFn.apply(outputs, self, lams)

    def _sums_buffers(self, N):
        """(sums (1 + 2 n_out,), scratch) for a device-reduced loss over N samples of ONE parameter row; the scratch
        size is the tile and fold tree's, which ``sdcgym_residual_sweeps_sum`` shares"""
        torch = _torch()
        sums = torch.empty(1 + 2 * self.n_out, dtype=torch.float64, device=self.device)
        n_scratch = int(self._L.sdcgym_spectral_radius_grad_sum_scratch_doubles(self.M, self._desc.prec_type, N))
        if n_scratch < 0:
            _lib.check(n_scratch, "sdcgym_spectral_radius_grad_sum_scratch_doubles")
        return sums, torch.empty(n_scratch, dtype=torch.float64, device=self.device)

    def _grad_sums(self, N, lam_r, qd, is_c):
        """(1 + 2 n_out,) CUDA float64: sum of rho, then sum Re g_k, sum Im g_k (``sdcgym_spectral_radius_grad_sum``)
        over N samples of ONE parameter row; lam_r None selects the grid already set in the descriptor."""
        d = self._desc
        d.qd_is_complex, d.qd_broadcast = is_c, 1
        sums, scratch = self._sums_buffers(N)
        _lib.check(self._L.sdcgym_spectral_radius_grad_sum(
            ctypes.byref(d), N, None if lam_r is None else lam_r.data_ptr(), qd.data_ptr(), None, scratch.data_ptr(),
            sums.data_ptr(), self._stream()), "sdcgym_spectral_radius_grad_sum")
        self._keep = (lam_r, qd, scratch)
        return sums

    def _mean_and_grad(self, sums, count, is_c, convention):
        """(sums[..., 0] / count, g / count) with g in ``convention`` (see ``value_and_grad``); real rows give a real g."""
        torch = _torch()
        if convention not in ("jax", "torch"):
            raise ValueError("convention must be 'jax' or 'torch'")
        # sums (..., 1 + 2 n_out): one row or a population of rows
        pairs = sums[..., 1:].reshape(*sums.shape[:-1], self.n_out, 2) / max(count, 1)  # no samples: zero gradient, NaN mean
        g = torch.view_as_complex(pairs.contiguous())
        if not is_c:
            g = g.real.contiguous()
        elif convention == "torch":
            g = g.conj().resolve_conj()
        return sums[..., 0] / count, g

    def _shared_row(self, output):
        if self.prec is not None:
            raise ValueError("a fixed preconditioner has no parameters to differentiate")
        out = output.detach() if isinstance(output, _torch().Tensor) else np.asarray(output)
        if not (out.ndim == 1 or (out.ndim == 2 and out.shape[0] == 1)):
            raise ValueError(f"output must be one parameter row, shape ({self.n_out},) or (1, {self.n_out})")
        qd, is_c, _ = self._outputs_tensor(out, 1)
        return qd, is_c

    @_lib.on_device
    def shared_value_and_grad(self, lams, output, convention="jax"):
        """(mean rho, d mean_rho / d output) for ONE parameter row ``output`` (shape (n_out,) or (1, n_out)) shared by
        every lambda: ``value_and_grad`` on the row expanded to the batch, reduced on the device without forming the
        per-sample gradient (``sdcgym_spectral_radius_grad_sum``).  ``g`` has shape (n_out,); conventions as in
        ``value_and_grad``.  An empty batch gives (NaN, zeros)."""
        torch = _torch()
        qd, is_c = self._shared_row(output)
        lam = lams if isinstance(lams, torch.Tensor) else torch.as_tensor(np.asarray(lams, dtype=np.complex128))
        lam = lam.detach().to(self.device).to(torch.complex128).reshape(-1).contiguous()
        B = lam.numel()
        if B == 0:  # 0/0, and nothing to launch (a NULL lambda pointer would select grid mode in the ABI)
            sums = torch.zeros(1 + 2 * self.n_out, dtype=torch.float64, device=self.device)
        else:
            d = self._desc
            d.grid_re = d.grid_im = 0
            sums = self._grad_sums(B, torch.view_as_real(lam), qd, is_c)
        return self._mean_and_grad(sums, B, is_c, convention)

    @_lib.on_device
    def _grid_sums(self, n_re, n_im, lambda_real_interval, lambda_imag_interval, lo, hi, sums_of, P=None):
        """sums_of(N) over grid rows lo..hi-1 with the grid set in the descriptor (zeros for an empty range, of shape
        (P, 1 + 2 n_out) for a population of P rows)"""
        torch = _torch()
        N = (hi - lo) * int(n_im)
        if N == 0:  # an empty shard contributes nothing and launches nothing
            shape = (1 + 2 * self.n_out,) if P is None else (P, 1 + 2 * self.n_out)
            return torch.zeros(shape, dtype=torch.float64, device=self.device)
        d = self._desc
        d.grid_re, d.grid_im, d.grid_first = int(n_re), int(n_im), lo * int(n_im)
        d.re_lo, d.re_hi = float(lambda_real_interval[0]), float(lambda_real_interval[1])
        d.im_lo, d.im_hi = float(lambda_imag_interval[0]), float(lambda_imag_interval[1])
        try:
            return sums_of(N)
        finally:
            d.grid_first = 0

    def _sharded_grid_sums(self, n_re, n_im, lambda_real_interval, lambda_imag_interval, rows, sums_of, P=None):
        """(sums, sample count) of sums_of over the grid: ``rows=None`` shards the rows over the ranks of the default
        process group and all-reduces the 1 + 2 n_out sums (of each of P rows); ``rows=(lo, hi)`` takes those rows
        only, no collective."""
        from . import dist as _dist

        n_re, n_im = int(n_re), int(n_im)
        sums, n_rows = _dist.sharded_rows_sum(n_re, rows, lambda lo, hi: self._grid_sums(
            n_re, n_im, lambda_real_interval, lambda_imag_interval, lo, hi, sums_of, P))
        return sums, n_rows * n_im

    def grid_value_and_grad(self, n_re, n_im, lambda_real_interval, lambda_imag_interval, output, rows=None,
                            convention="jax"):
        """(mean rho, d mean_rho / d output) over the (n_re x n_im) lambda grid of ``grid`` for ONE parameter row,
        lambdas generated on the device and the gradient reduced there (``sdcgym_spectral_radius_grad_sum``).
        ``rows=None``: the whole grid, rows sharded over the ranks of the default process group as in ``grid_mean``
        with one all-reduce of 1 + 2 n_out doubles.  ``rows=(lo, hi)``: the mean and gradient over grid rows lo..hi-1
        only, no collective call (an empty range gives (NaN, zeros)).  Conventions as in ``value_and_grad``."""
        qd, is_c = self._shared_row(output)
        sums, count = self._sharded_grid_sums(n_re, n_im, lambda_real_interval, lambda_imag_interval, rows,
                                              lambda N: self._grad_sums(N, None, qd, is_c))
        return self._mean_and_grad(sums, count, is_c, convention)

    def grid_differentiable(self, n_re, n_im, lambda_real_interval, lambda_imag_interval, output):
        """``grid_value_and_grad`` over the whole grid as a torch scalar that supports ``.backward()`` into the
        parameter row ``output``."""
        return _SharedRowFn.apply(output, lambda o, conv: self.grid_value_and_grad(
            n_re, n_im, lambda_real_interval, lambda_imag_interval, o, convention=conv))

    # ---- populations: P parameter rows, each shared by every lambda, in one launch ----
    def _population_rows(self, population):
        """(qd (P, n_out[, 2]) float64 on the device, is_c) of P >= 1 parameter rows"""
        torch = _torch()
        if self.prec is not None:
            raise ValueError("a fixed preconditioner has no parameters to differentiate")
        t = population.detach() if isinstance(population, torch.Tensor) else torch.as_tensor(np.array(population))
        if t.dim() != 2 or t.shape[0] < 1 or t.shape[1] != self.n_out:
            raise ValueError(f"population must have shape (P, {self.n_out}) with P >= 1, not {tuple(t.shape)}")
        qd, is_c, _ = self._outputs_tensor(t, t.shape[0])
        return qd, is_c

    def _population_sums(self, N, lam_r, qd, is_c):
        """(P, 1 + 2 n_out) CUDA float64 (``sdcgym_spectral_radius_grad_sum_population``): ``_grad_sums`` of each row"""
        torch = _torch()
        d = self._desc
        d.qd_is_complex, d.qd_broadcast = is_c, 1
        P = qd.shape[0]
        sums = torch.empty((P, 1 + 2 * self.n_out), dtype=torch.float64, device=self.device)
        n_scratch = int(self._L.sdcgym_spectral_radius_grad_sum_scratch_doubles(self.M, d.prec_type, N))
        if n_scratch < 0:
            _lib.check(n_scratch, "sdcgym_spectral_radius_grad_sum_scratch_doubles")
        scratch = torch.empty(P * n_scratch, dtype=torch.float64, device=self.device)
        _lib.check(self._L.sdcgym_spectral_radius_grad_sum_population(
            ctypes.byref(d), N, None if lam_r is None else lam_r.data_ptr(), P, qd.data_ptr(), qd[0].numel(),
            scratch.data_ptr(), sums.data_ptr(), self._stream()), "sdcgym_spectral_radius_grad_sum_population")
        self._keep = (lam_r, qd, scratch)
        return sums

    @_lib.on_device
    def population_value_and_grad(self, lams, population, convention="jax"):
        """``shared_value_and_grad`` for each row of ``population`` (P, n_out), every row shared by all lambdas, in one
        launch: (means (P,), gradients (P, n_out)); row p equals ``shared_value_and_grad(lams, population[p])`` bit for
        bit.  An empty batch gives (NaN, zeros) per row."""
        torch = _torch()
        qd, is_c = self._population_rows(population)
        lam = lams if isinstance(lams, torch.Tensor) else torch.as_tensor(np.asarray(lams, dtype=np.complex128))
        lam = lam.detach().to(self.device).to(torch.complex128).reshape(-1).contiguous()
        B = lam.numel()
        if B == 0:  # 0/0, and nothing to launch (a NULL lambda pointer would select grid mode in the ABI)
            sums = torch.zeros((qd.shape[0], 1 + 2 * self.n_out), dtype=torch.float64, device=self.device)
        else:
            d = self._desc
            d.grid_re = d.grid_im = 0
            sums = self._population_sums(B, torch.view_as_real(lam), qd, is_c)
        return self._mean_and_grad(sums, B, is_c, convention)

    def population_grid_value_and_grad(self, n_re, n_im, lambda_real_interval, lambda_imag_interval, population,
                                       rows=None, convention="jax"):
        """``grid_value_and_grad`` for each row of ``population`` (P, n_out) in one launch per shard: (means (P,),
        gradients (P, n_out)).  ``rows=None``: the whole grid, rows sharded over the ranks of the default process
        group with one all-reduce of P (1 + 2 n_out) doubles; ``rows=(lo, hi)``: grid rows lo..hi-1 only, no
        collective call (an empty range gives (NaN, zeros) per row)."""
        qd, is_c = self._population_rows(population)
        sums, count = self._sharded_grid_sums(n_re, n_im, lambda_real_interval, lambda_imag_interval, rows,
                                              lambda N: self._population_sums(N, None, qd, is_c), qd.shape[0])
        return self._mean_and_grad(sums, count, is_c, convention)

    def population_differentiable(self, lams, population):
        """``population_value_and_grad`` as a (P,) tensor whose ``.sum().backward()`` gives each row of ``population``
        its own gradient (real rows real, complex rows in the torch convention, as ``differentiable``)"""
        return _SharedRowFn.apply(population, lambda o, conv: self.population_value_and_grad(lams, o, conv))

    def population_grid_differentiable(self, n_re, n_im, lambda_real_interval, lambda_imag_interval, population):
        """``population_grid_value_and_grad`` over the whole grid as a (P,) tensor that supports ``.backward()`` into
        ``population``"""
        return _SharedRowFn.apply(population, lambda o, conv: self.population_grid_value_and_grad(
            n_re, n_im, lambda_real_interval, lambda_imag_interval, o, convention=conv))

    @_lib.on_device
    def _sum(self, rho):
        """deterministic fp64 sum (fixed reduction tree) as a CUDA scalar"""
        torch = _torch()
        out = torch.zeros(1, dtype=torch.float64, device=self.device)
        if rho.numel():
            scratch = torch.empty(self._L.sdcgym_sum_scratch_doubles(), dtype=torch.float64, device=self.device)
            _lib.check(self._L.sdcgym_sum_f64(rho.numel(), rho.data_ptr(), scratch.data_ptr(), out.data_ptr(),
                                              self._stream()), "sdcgym_sum_f64")
        return out[0]

    def mean(self, rho):
        return self._sum(rho) / rho.numel()

    @_lib.on_device
    def grid(self, n_re, n_im, lambda_real_interval, lambda_imag_interval, output=None, rows=None):
        """rho on the (n_re x n_im) tensor grid over the lambda box for ONE Q_delta parameter row (or the fixed
        ``prec``): lambdas are generated from the grid index on the device (0 bytes in, 8 bytes out per matrix).
        ``rows=(lo, hi)`` evaluates only the grid rows lo..hi-1 (real-axis index) - the shard of one rank.
        Returns a CUDA tensor (n_re, n_im) [(hi - lo, n_im) with ``rows``]."""
        torch = _torch()
        qd, is_c, _ = self._outputs_tensor(output, 1) if self.prec is None else (None, 0, 0)
        lo, hi = (0, int(n_re)) if rows is None else (int(rows[0]), int(rows[1]))
        if not 0 <= lo <= hi <= int(n_re):
            raise ValueError(f"rows={rows} outside the grid of {n_re} rows")
        d = self._desc
        d.qd_is_complex, d.qd_broadcast = is_c, 1
        d.grid_re, d.grid_im, d.grid_first = int(n_re), int(n_im), lo * int(n_im)
        d.re_lo, d.re_hi = float(lambda_real_interval[0]), float(lambda_real_interval[1])
        d.im_lo, d.im_hi = float(lambda_imag_interval[0]), float(lambda_imag_interval[1])
        N = (hi - lo) * int(n_im)
        rho = torch.empty(N, dtype=torch.float64, device=self.device)
        _lib.check(self._L.sdcgym_spectral_radius(ctypes.byref(d), N, None, None if qd is None else qd.data_ptr(),
                                                  rho.data_ptr(), self._stream()), "sdcgym_spectral_radius")
        d.grid_first = 0
        self._keep = (qd,)
        return rho.reshape(hi - lo, n_im)

    def grid_mean(self, n_re, n_im, lambda_real_interval, lambda_imag_interval, output=None):
        """Mean of rho over the grid with the rows sharded over the ranks of the default process group (SURVEY 8e):
        every rank evaluates ``dist.shard_range(n_re)`` rows and ONE scalar is all-reduced.  Without an initialised
        process group this is the single-GPU mean.  Returns a CUDA scalar (the same value on every rank)."""
        from . import dist as _dist

        rank, world = _dist.world()
        lo, count = _dist.shard_range(int(n_re), rank, world)
        rho = self.grid(n_re, n_im, lambda_real_interval, lambda_imag_interval, output, rows=(lo, lo + count))
        total = _dist.all_reduce_sum(self._sum(rho.reshape(-1)).reshape(1))[0]
        return total / (int(n_re) * int(n_im))


def _make_autograd_fn():
    torch = _torch()

    class SpectralRadiusFn(torch.autograd.Function):
        @staticmethod
        def forward(ctx, outputs, loss, lams):
            value, g = loss.value_and_grad(lams, outputs, convention="torch")
            ctx.save_for_backward(g)
            ctx.out_shape, ctx.out_dtype = outputs.shape, outputs.dtype
            return value.reshape(())

        @staticmethod
        def backward(ctx, upstream):
            (g,) = ctx.saved_tensors
            return (g * upstream).reshape(ctx.out_shape).to(ctx.out_dtype), None, None

    return SpectralRadiusFn


def _make_shared_row_fn():
    torch = _torch()

    class SharedRowFn(torch.autograd.Function):
        """value_and_grad(row, convention) -> (scalar, g of the row's size): the loss of one shared parameter row; or
        (values (P,), g (P, n_out)): the losses of a population of P rows"""

        @staticmethod
        def forward(ctx, row, value_and_grad):
            value, g = value_and_grad(row, "torch")
            ctx.save_for_backward(g)
            ctx.out_shape, ctx.out_dtype = row.shape, row.dtype
            return value.reshape(value.shape[:1] if value.dim() else ())

        @staticmethod
        def backward(ctx, upstream):
            (g,) = ctx.saved_tensors
            if upstream.dim():  # one upstream value per population row
                upstream = upstream[:, None]
            return (g * upstream).reshape(ctx.out_shape).to(ctx.out_dtype), None

    return SharedRowFn


def _make_sweeps_fn():
    torch = _torch()

    class SweepsFn(torch.autograd.Function):
        """sweeps(outputs) -> (u_K, r_K, norms (B,), g (B, n_out)): per-sample norms, backward through g"""

        @staticmethod
        def forward(ctx, outputs, sweeps):
            _, _, norms, g = sweeps(outputs)
            g = g if outputs.is_complex() else g.real
            ctx.save_for_backward(g.conj() if outputs.is_complex() else g)
            ctx.out_shape, ctx.out_dtype = outputs.shape, outputs.dtype
            return norms

        @staticmethod
        def backward(ctx, upstream):
            (g,) = ctx.saved_tensors
            gu = g * upstream.to(g.dtype)[:, None]
            shared = len(ctx.out_shape) == 1 or (ctx.out_shape[0] == 1 and g.shape[0] != 1)
            if shared:
                gu = gu.sum(0)
            return gu.reshape(ctx.out_shape).to(ctx.out_dtype), None

    return SweepsFn


class _LazyFn:
    def __init__(self, make):
        self._make, self._fn = make, None

    def apply(self, *a):
        if self._fn is None:
            self._fn = self._make()
        return self._fn.apply(*a)


_SpectralRadiusFn = _LazyFn(_make_autograd_fn)
_SharedRowFn = _LazyFn(_make_shared_row_fn)
_SweepsFn = _LazyFn(_make_sweeps_fn)

NormLoss = SpectralRadiusLoss  # the reference keeps this alias (dp_playground.py:233)

SWEEPS_REDUCTIONS = {"mean": 0, "log_ratio": 1}  # SDCGYM_SWEEPS_MEAN, SDCGYM_SWEEPS_LOG_RATIO (include/sdcgym.h)


class ResidualLoss:
    """``dp_playground.py:235-258``: one sweep with the learned Q_delta; loss = mean ||r'||_inf.

    ``__call__(lams, outputs, Cs, u0s, us, old_residuals) -> (mean_norm, us', residuals')`` like the reference.
    ``Cs`` may be ``None`` (the system matrices are then formed from ``lams`` on the device instead of being read).
    """

    def __init__(self, M, dt, prec_type="diag", *, prec=None, Q=None, device=None):
        self._sr = SpectralRadiusLoss(M, dt, prec_type, prec=prec, Q=Q, device=device)
        self.M, self.dt, self.prec_type = self._sr.M, self._sr.dt, self._sr.prec_type
        self.Q, self.device = self._sr.Q, self._sr.device
        self._guard = self._sr._guard

    def _c128(self, x, shape):
        torch = _torch()
        t = x if isinstance(x, torch.Tensor) else torch.as_tensor(np.asarray(x, dtype=np.complex128))
        t = t.to(self.device).to(torch.complex128).reshape(shape).contiguous()
        return torch.view_as_real(t)

    @_lib.on_device
    def take_step(self, lams, outputs, Cs, u0s, us, old_residuals, with_grad=False):
        torch = _torch()
        sr, M = self._sr, self.M
        lam = self._c128(lams, (-1,))
        B = lam.shape[0]
        out = outputs.detach() if isinstance(outputs, torch.Tensor) else outputs
        qd, is_c, bc = sr._outputs_tensor(out, B)
        if bc:
            qd = qd.expand(B, *qd.shape[1:]).contiguous()
        d = sr._desc
        d.qd_is_complex, d.qd_broadcast = is_c, 0
        u0, u, r = (self._c128(x, (B, M)) for x in (u0s, us, old_residuals))
        C = None if Cs is None else self._c128(Cs, (B, M, M))
        u_out = torch.empty((B, M, 2), dtype=torch.float64, device=self.device)
        r_out = torch.empty((B, M, 2), dtype=torch.float64, device=self.device)
        norms = torch.empty(B, dtype=torch.float64, device=self.device)
        grad = torch.empty((B, sr.n_out, 2), dtype=torch.float64, device=self.device) if with_grad else None
        _lib.check(sr._L.sdcgym_residual_step(
            ctypes.byref(d), B, lam.data_ptr(), None if qd is None else qd.data_ptr(),
            None if C is None else C.data_ptr(), u0.data_ptr(), u.data_ptr(), r.data_ptr(), u_out.data_ptr(),
            r_out.data_ptr(), norms.data_ptr(), None if grad is None else grad.data_ptr(), sr._stream()),
            "sdcgym_residual_step")
        self._keep = (lam, qd, C, u0, u, r)
        res = (torch.view_as_complex(u_out), torch.view_as_complex(r_out), norms)
        return res + (torch.view_as_complex(grad),) if with_grad else res

    @_lib.on_device
    def sweeps(self, lams, outputs, K, u0s=None, us=None, residuals=None, with_grad=False):
        """``(u_K, r_K, norms[, g])`` after exactly K (1..50) sweeps of ``take_step``'s iteration with C = I - z Q, no
        early stop (``sdcgym_residual_sweeps``).  Inputs are shaped as in ``take_step``; ``u0s``, ``us`` and
        ``residuals`` all None start from the envs' reset state u0 = u = 1, r = u0 - C 1.  ``outputs`` is (B, n_out),
        or one row (n_out,) / (1, n_out) shared by every lambda.  ``g`` (B, n_out) complex128 is the derivative of
        ``norms`` through all K sweeps, d norm_b = Re(sum_k g_bk d theta_bk) (for a shared row: of each sample's norm
        with respect to that row).  A norm that is 0, +inf or NaN has g = 0."""
        torch = _torch()
        sr, M = self._sr, self.M
        given = [x is not None for x in (u0s, us, residuals)]
        if any(given) and not all(given):
            raise ValueError("give all of u0s, us and residuals, or none of them (the reset state)")
        lam = self._c128(lams, (-1,))
        B = lam.shape[0]
        out = outputs.detach() if isinstance(outputs, torch.Tensor) else outputs
        qd, is_c, bc = sr._outputs_tensor(out, B) if B else (None, 0, 0)
        d = sr._desc
        d.qd_is_complex, d.qd_broadcast = is_c, bc
        u0, u, r = (self._c128(x, (B, M)) for x in (u0s, us, residuals)) if all(given) else (None, None, None)
        u_out = torch.empty((B, M, 2), dtype=torch.float64, device=self.device)
        r_out = torch.empty((B, M, 2), dtype=torch.float64, device=self.device)
        norms = torch.empty(B, dtype=torch.float64, device=self.device)
        grad = torch.zeros((B, sr.n_out, 2), dtype=torch.float64, device=self.device) if with_grad else None
        if B:
            ptr = lambda t: None if t is None else t.data_ptr()  # noqa: E731
            _lib.check(sr._L.sdcgym_residual_sweeps(
                ctypes.byref(d), B, int(K), lam.data_ptr(), ptr(qd), ptr(u0), ptr(u), ptr(r), u_out.data_ptr(),
                r_out.data_ptr(), norms.data_ptr(), ptr(grad), sr._stream()), "sdcgym_residual_sweeps")
        self._keep = (lam, qd, u0, u, r)
        res = (torch.view_as_complex(u_out), torch.view_as_complex(r_out), norms)
        return res + (torch.view_as_complex(grad),) if with_grad else res

    def sweeps_differentiable(self, lams, outputs, K, u0s=None, us=None, residuals=None):
        """Per-sample ``||r_K||_inf`` (B,) of ``sweeps`` as a tensor that supports ``.backward()`` into ``outputs`` (a
        CUDA tensor with ``requires_grad``): forward and backward both run the K-sweep kernel, and the gradient is taken
        through every sweep.  Compose any reduction on top, e.g. ``torch.log(n).mean()``.  Real rows get a real
        gradient, complex rows the torch convention (as ``SpectralRadiusLoss.differentiable``); a single shared row
        gets a gradient of its own shape, summed over the batch."""
        return _SweepsFn.apply(outputs, lambda o: self.sweeps(lams, o, K, u0s, us, residuals, with_grad=True))

    def _sweeps_args(self, K, reduction, u0s, us, residuals):
        if reduction not in SWEEPS_REDUCTIONS:
            raise ValueError(f"reduction must be one of {sorted(SWEEPS_REDUCTIONS)}, not {reduction!r}")
        given = [x is not None for x in (u0s, us, residuals)]
        if any(given) and not all(given):
            raise ValueError("give all of u0s, us and residuals, or none of them (the reset state)")
        return int(K), SWEEPS_REDUCTIONS[reduction]

    def _sweeps_sums(self, N, K, reduction, lam, qd, is_c, u0=None, u=None, r=None):
        """(1 + 2 n_out,) CUDA float64 (``sdcgym_residual_sweeps_sum``) over N samples of ONE parameter row; lam None
        selects the grid already set in the descriptor"""
        sr = self._sr
        d = sr._desc
        d.qd_is_complex, d.qd_broadcast = is_c, 1
        sums, scratch = sr._sums_buffers(N)
        ptr = lambda t: None if t is None else t.data_ptr()  # noqa: E731
        _lib.check(sr._L.sdcgym_residual_sweeps_sum(
            ctypes.byref(d), N, K, reduction, ptr(lam), qd.data_ptr(), ptr(u0), ptr(u), ptr(r), None,
            scratch.data_ptr(), sums.data_ptr(), sr._stream()), "sdcgym_residual_sweeps_sum")
        self._keep = (lam, qd, u0, u, r, scratch)
        return sums

    @_lib.on_device
    def sweeps_shared_value_and_grad(self, lams, output, K, u0s=None, us=None, residuals=None, reduction="mean",
                                     convention="jax"):
        """(mean loss, d mean / d output) after exactly K sweeps (as ``sweeps``) for ONE parameter row ``output``
        (shape (n_out,) or (1, n_out)) shared by every lambda, reduced on the device without forming the per-sample
        gradient, u_K or r_K (``sdcgym_residual_sweeps_sum``).  ``reduction``: 'mean', the mean of n_K = ||r_K||_inf
        (``ResidualLoss``'s own loss), or 'log_ratio', the mean of log(n_K / n_0) with n_0 = ||r_0||_inf of the
        starting residual.  A sample with n_0 = 0 (lambda = 0 from the reset state) adds zeros to the log_ratio value
        and gradient; a sample whose n_K is 0, +inf or NaN adds a zero gradient, and its value (n_K = 0: -inf under
        log_ratio) reaches the mean unchanged.  The mean divides by the batch size.  ``g`` has shape (n_out,);
        conventions as in ``SpectralRadiusLoss.value_and_grad``.  An empty batch gives (NaN, zeros)."""
        torch = _torch()
        K, red = self._sweeps_args(K, reduction, u0s, us, residuals)
        qd, is_c = self._sr._shared_row(output)
        lam = self._c128(lams, (-1,))
        B = lam.shape[0]
        if B == 0:  # 0/0, and nothing to launch (a NULL lambda pointer would select grid mode in the ABI)
            sums = torch.zeros(1 + 2 * self._sr.n_out, dtype=torch.float64, device=self.device)
        else:
            self._sr._desc.grid_re = self._sr._desc.grid_im = 0
            states = (self._c128(x, (B, self.M)) for x in (u0s, us, residuals)) if u0s is not None else ()
            sums = self._sweeps_sums(B, K, red, lam, qd, is_c, *states)
        return self._sr._mean_and_grad(sums, B, is_c, convention)

    def sweeps_grid_value_and_grad(self, n_re, n_im, lambda_real_interval, lambda_imag_interval, output, K,
                                   reduction="mean", rows=None, convention="jax"):
        """``sweeps_shared_value_and_grad`` from the envs' reset state over the (n_re x n_im) lambda grid of
        ``SpectralRadiusLoss.grid``, lambdas generated on the device.  ``rows=None``: the whole grid, rows sharded
        over the ranks of the default process group with one all-reduce of 1 + 2 n_out doubles.  ``rows=(lo, hi)``:
        grid rows lo..hi-1 only, no collective call (an empty range gives (NaN, zeros))."""
        K, red = self._sweeps_args(K, reduction, None, None, None)
        sr = self._sr
        qd, is_c = sr._shared_row(output)
        sums, count = sr._sharded_grid_sums(n_re, n_im, lambda_real_interval, lambda_imag_interval, rows,
                                            lambda N: self._sweeps_sums(N, K, red, None, qd, is_c))
        return sr._mean_and_grad(sums, count, is_c, convention)

    def sweeps_shared_differentiable(self, lams, output, K, u0s=None, us=None, residuals=None, reduction="mean"):
        """``sweeps_shared_value_and_grad`` as a torch scalar that supports ``.backward()`` into the parameter row
        ``output``"""
        return _SharedRowFn.apply(output, lambda o, conv: self.sweeps_shared_value_and_grad(
            lams, o, K, u0s, us, residuals, reduction, conv))

    def sweeps_grid_differentiable(self, n_re, n_im, lambda_real_interval, lambda_imag_interval, output, K,
                                   reduction="mean"):
        """``sweeps_grid_value_and_grad`` over the whole grid as a torch scalar that supports ``.backward()`` into the
        parameter row ``output``"""
        return _SharedRowFn.apply(output, lambda o, conv: self.sweeps_grid_value_and_grad(
            n_re, n_im, lambda_real_interval, lambda_imag_interval, o, K, reduction, convention=conv))

    def __call__(self, lams, outputs, Cs, u0s, us, old_residuals):
        us_new, residuals, norms = self.take_step(lams, outputs, Cs, u0s, us, old_residuals)
        return self._sr.mean(norms), us_new, residuals

    def value_and_grad(self, lams, outputs, Cs, u0s, us, old_residuals, convention="jax"):
        """((loss, us', residuals'), d loss / d outputs): ``jax.value_and_grad(loss, has_aux=True)`` for the residual
        loss (``dp_playground.py:1038-1073``); gradient conventions as in ``SpectralRadiusLoss.value_and_grad``."""
        torch = _torch()
        us_new, residuals, norms, g = self.take_step(lams, outputs, Cs, u0s, us, old_residuals, with_grad=True)
        g = g / norms.numel()
        is_c = (outputs.is_complex() if isinstance(outputs, torch.Tensor) else np.iscomplexobj(outputs))
        if not is_c:
            g = g.real
        elif convention == "torch":
            g = g.conj()
        elif convention != "jax":
            raise ValueError("convention must be 'jax' or 'torch'")
        return (self._sr.mean(norms), us_new, residuals), g

"""Multi-GPU plumbing: env sharding and the (only) collectives of the path.

Envs are independent, so the global env index range is cut into contiguous per-rank slices and every rank steps
its slice with no communication (``SURVEY.md`` 8e).  ``torch.distributed`` (NCCL on GPUs, gloo in the CPU tests)
is used for two tiny all-reduces only: rollout statistics and the normaliser's moment sums.
"""
from __future__ import annotations

import numpy as np


def _dist():
    import torch.distributed as dist

    return dist


def is_distributed() -> bool:
    dist = _dist()
    return dist.is_available() and dist.is_initialized()


def world():
    """(rank, world_size) of the default process group, (0, 1) when not initialised."""
    if is_distributed():
        dist = _dist()
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def shard_range(num_envs_global: int, rank: int, world_size: int):
    """Contiguous slice [offset, offset + count) of the global env index range owned by ``rank``.

    The first ``num_envs_global % world_size`` ranks get one env more; empty slices are allowed.
    """
    if not 0 <= rank < world_size:
        raise ValueError("rank out of range")
    base, extra = divmod(int(num_envs_global), int(world_size))
    count = base + (1 if rank < extra else 0)
    offset = rank * base + min(rank, extra)
    return offset, count


def make_sharded(envname, num_envs_global, **kwargs):
    """This rank's slice of a global batch of ``num_envs_global`` envs (same seeds/lambda streams as one big env)."""
    from . import make

    rank, ws = world()
    offset, count = shard_range(num_envs_global, rank, ws)
    return make(envname, num_envs=count, env_offset=kwargs.pop("env_offset", 0) + offset, **kwargs)


def all_reduce_sum(t):
    """In-place sum all-reduce of a tensor over the default group (no-op when single process)."""
    if is_distributed():
        _dist().all_reduce(t)
    return t


def sharded_rows_sum(n_rows, rows, sums_of):
    """(sums, number of rows summed) of ``sums_of(lo, hi)``, a tensor of sums over the rows lo..hi-1 of a grid of
    ``n_rows`` rows.  ``rows=None``: this rank's ``shard_range`` of the rows, the sums all-reduced over the default
    process group (every rank gets the sums over all rows); ``rows=(lo, hi)``: those rows only, no collective call."""
    n_rows = int(n_rows)
    if rows is None:
        rank, size = world()
        lo, count = shard_range(n_rows, rank, size)
        return all_reduce_sum(sums_of(lo, lo + count)), n_rows
    lo, hi = int(rows[0]), int(rows[1])
    if not 0 <= lo <= hi <= n_rows:
        raise ValueError(f"rows={rows} outside the grid of {n_rows} rows")
    return sums_of(lo, hi), hi - lo


class PeerExchange:
    """Exchange regions for the in-kernel all-reduce of the normaliser moments (include/sdcgym.h ``sdcgym_xchg``):
    every rank allocates one region, the 64-byte CUDA IPC handles travel over the process group (the only use of the
    host-side collective: once, at set-up), every rank maps all the others' regions.  ``struct(seq)`` fills the
    argument block of ``sdcgym_vecnorm_update*_dist``."""

    def __init__(self, slot_doubles: int):
        import ctypes

        from . import _lib

        L = _lib.load()
        dist = _dist()
        self._L = L
        self.rank, self.world = world()
        if self.world > _lib.MAX_RANKS:
            raise _lib.SdcGymError(f"peer exchange supports up to {_lib.MAX_RANKS} ranks")
        self.slot = int(slot_doubles)
        nbytes = L.sdcgym_xchg_bytes(self.world, self.slot)
        ptr = ctypes.c_void_p()
        handle = ctypes.create_string_buffer(64)
        _lib.check(L.sdcgym_ipc_alloc(nbytes, ctypes.byref(ptr), handle), "sdcgym_ipc_alloc")
        self._own = ptr.value
        handles = [None] * self.world
        dist.all_gather_object(handles, bytes(handle.raw))
        self.peers = [None] * self.world
        self._opened = []
        for r, h in enumerate(handles):
            if r == self.rank:
                self.peers[r] = self._own
                continue
            q = ctypes.c_void_p()
            _lib.check(L.sdcgym_ipc_open(h, ctypes.byref(q)), f"sdcgym_ipc_open (rank {r})")
            self.peers[r] = q.value
            self._opened.append(q.value)
        dist.barrier()  # nobody launches an exchange before every region is mapped everywhere
        self.seq = 0
        self._struct = _lib.Xchg()
        self._struct.world, self._struct.rank, self._struct.slot_doubles = self.world, self.rank, self.slot
        for r, q in enumerate(self.peers):
            self._struct.peers[r] = q

    def next(self):
        """The argument struct for the next exchange (sequence numbers 1, 2, 3, ... in lock step on all ranks)."""
        self.seq += 1
        self._struct.seq = self.seq
        return self._struct

    def close(self):
        for q in self._opened:
            self._L.sdcgym_ipc_close(q)
        self._opened = []
        if self._own:
            self._L.sdcgym_ipc_free(self._own)
            self._own = None


def chan_merge(mean, var, count, shifted_sum, shifted_sumsq, batch_count):
    """Host restatement of ``rms_merge_kernel`` (SB3 ``RunningMeanStd.update_from_moments``): the batch is described
    by sums of (x - mean) and (x - mean)^2 over ``batch_count`` samples.  Works on numpy arrays or tensors."""
    if batch_count <= 0:
        return mean, var, count
    d1 = shifted_sum / batch_count
    bvar = shifted_sumsq / batch_count - d1 * d1
    bvar = bvar * (bvar > 0)
    tot = count + batch_count
    m2 = var * count + bvar * batch_count + d1 * d1 * count * batch_count / tot
    return mean + d1 * batch_count / tot, m2 / tot, tot


class RolloutStats:
    """Per-rollout statistics accumulated on the device and reduced once over all ranks:
    env-steps, episodes, sum of rewards, sum of sweeps (niter), converged and diverged episode counts."""

    FIELDS = ("env_steps", "episodes", "sum_reward", "sum_niter", "converged", "diverged")

    def __init__(self, device):
        import torch

        self.acc = torch.zeros(len(self.FIELDS), dtype=torch.float64, device=device)

    def update(self, out):
        """``out``: dict returned by ``SDCVecEnv.step_tensor`` (reward, flags, niter)."""
        import torch

        flags = out["flags"]
        done = (flags & 1).ne(0)
        vals = torch.stack([
            torch.tensor(float(flags.numel()), dtype=torch.float64, device=flags.device),
            done.sum().double(),
            out["reward"].sum(),
            (out["niter"].double() * done.double()).sum(),
            ((flags & 2).ne(0) & done).sum().double(),
            ((flags & 4).ne(0) & done).sum().double(),
        ])
        self.acc += vals

    def reduce(self):
        """All-reduce and return a dict of Python floats (this is the one host sync of a rollout)."""
        t = all_reduce_sum(self.acc.clone())
        return dict(zip(self.FIELDS, (float(v) for v in t.cpu().numpy())))

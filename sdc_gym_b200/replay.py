"""Device-resident replay buffer and transition collection for off-policy learners (SAC / TD3 / DDPG; the reference
selects ``use_doubles=False`` for SAC, ``utils/utils.py:279-280``).

``ReplayBuffer`` reproduces SB3's ``ReplayBuffer`` (``add`` / ``sample``) fed the way
``OffPolicyAlgorithm._store_transition`` feeds it: the un-normalised observation the action was taken on, the
un-normalised reward, and as next observation the new one - or, for an env whose episode just ended, its terminal
observation (the new one is then already the next episode's reset state).  ``sample`` normalises with the
``VecNormalize``'s current statistics, as SB3 does.  Storage and sampling are kernels of ``libsdcgym.so``
(``csrc/replay.cu``); the ring position, the ``full`` flag and the sample-call counter live on the device, so
``collect_transitions`` + ``sample`` can be captured in one CUDA graph and replayed.  Deviations from SB3: DESIGN.md 5.

Several ranks: every rank owns its buffer over its own envs and samples it locally; nothing is exchanged.
"""
from __future__ import annotations

import collections
import ctypes

import numpy as np

from . import _lib
from .rng import philox4x32_10

ReplaySamples = collections.namedtuple("ReplaySamples", "observations actions next_observations dones rewards")

REPLAY_TAG = 0x5250  # kReplayTag, csrc/replay_index.cuh


def _torch():
    import torch

    return torch


def replay_indices(seed, call, j, upper, n_envs):
    """numpy restatement of ``replay_index`` (csrc/replay_index.cuh): (row, env) of sample(s) ``j`` of the
    ``call``-th ``sample`` of a buffer seeded ``seed`` holding ``upper`` rows of ``n_envs`` envs."""
    j = np.asarray(j, dtype=np.uint64)
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    x0, x1, _, _ = philox4x32_10((j & np.uint64(0xFFFFFFFF)).astype(np.uint32), (j >> np.uint64(32)).astype(np.uint32),
                                 np.uint32(int(call) & 0xFFFFFFFF), np.uint32(REPLAY_TAG), seed & 0xFFFFFFFF, seed >> 32)
    row = (x0.astype(np.uint64) * np.uint64(upper)) >> np.uint64(32)
    env = (x1.astype(np.uint64) * np.uint64(n_envs)) >> np.uint64(32)
    return row.astype(np.int64), env.astype(np.int64)


def _check_env(venv):
    if venv.collect_states:
        raise NotImplementedError("ReplayBuffer: collect_states observations ((2M, 50) histories) are not supported")
    if venv._kernel_n_act == 0:
        raise ValueError("ReplayBuffer: the env has a fixed preconditioner (prec=...): there is no action to learn")
    if venv.terminal is None and venv.autoreset:
        raise ValueError("ReplayBuffer: an auto-reset env must keep its terminal observations (keep_terminal=True): "
                         "they are the next observation of every finished episode")


class ReplayBuffer:
    """Ring of ``max(buffer_size // num_envs, 1)`` rows x ``num_envs`` transitions in HBM (SB3 ``ReplayBuffer``).

    Stored per transition: observation and next observation as raw float64 planes (the env's ``S`` layout), the
    action as the policy handed it to ``step_tensor`` (float64, or complex128 with ``free_action_space``), the raw
    reward (float64) and the done flag.  ``env``: the (bare or ``VecNormalize``-wrapped) env the buffer is filled
    from; it fixes the number of envs, the observation planes (4M) and the action width and type."""

    def __init__(self, buffer_size, env, seed=0, device=None):
        torch = _torch()
        venv = getattr(env, "venv", env)
        _check_env(venv)
        self.num_envs, self.M = int(venv.num_envs), int(venv.M)
        self.rows = max(int(buffer_size) // self.num_envs, 1)
        self.buffer_size = self.rows * self.num_envs
        self.P, self.n_act = 4 * self.M, int(venv._kernel_n_act)
        self.action_is_complex = bool(venv.free_action_space)
        self.device = venv.device
        want = None if device is None else torch.device(device)
        if want is not None and (want.type != "cuda" or want.index not in (None, self.device.index)):
            raise ValueError(f"ReplayBuffer: the env's kernels write into the buffer, which must live on {self.device}")
        self.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        self.ld = int(venv.ld)
        self._guard = _lib.DeviceGuard(self.device)
        R, P, N = self.rows, self.P, self.num_envs
        f64 = torch.float64
        with self._guard:
            self.obs_store = torch.zeros((R, P, self.ld), dtype=f64, device=self.device)
            self.next_obs_store = torch.zeros((R, P, self.ld), dtype=f64, device=self.device)
            self.actions = torch.zeros((R, N, self.n_act), dtype=torch.complex128 if self.action_is_complex else f64,
                                       device=self.device)
            self.rewards = torch.zeros((R, N), dtype=f64, device=self.device)
            self.dones = torch.zeros((R, N), dtype=torch.uint8, device=self.device)
            self.counters = torch.zeros(3, dtype=torch.int64, device=self.device)  # pos, full, sample calls
        self.observations = self.obs_store[:, :, :N]  # (rows, 4M, N) views
        self.next_observations = self.next_obs_store[:, :, :N]
        self._desc = _lib.Replay()
        d = self._desc
        d.P, d.A, d.rows, d.N, d.ld, d.seed = P, self.n_act * (2 if self.action_is_complex else 1), R, N, self.ld, self.seed
        d.obs, d.next_obs = self.obs_store.data_ptr(), self.next_obs_store.data_ptr()
        d.actions, d.rewards = self.actions.data_ptr(), self.rewards.data_ptr()
        d.dones, d.counters = self.dones.data_ptr(), self.counters.data_ptr()
        self._L = _lib.load()
        self.venv = venv
        self._stored = False  # a store has been issued (eagerly or into a captured graph): sampling is allowed

    # ---- counters (read back from the device: these synchronise) -------------------------------------------------
    @property
    def pos(self):
        return int(self.counters[0].item())

    @property
    def full(self):
        return bool(self.counters[1].item())

    def size(self):
        c = self.counters.tolist()
        return self.rows if c[1] else c[0]

    # ---- storing ------------------------------------------------------------------------------------------------
    def _stream(self):
        return ctypes.c_void_p(_torch().cuda.current_stream(self.device).cuda_stream)

    def check_env(self, env):
        """Raise unless ``env`` (bare or wrapped) is the kind of env this buffer was built for."""
        venv = getattr(env, "venv", env)
        _check_env(venv)
        if (venv.num_envs, venv.M, venv._kernel_n_act, bool(venv.free_action_space), venv.ld) != (
                self.num_envs, self.M, self.n_act, self.action_is_complex, self.ld):
            raise ValueError(f"ReplayBuffer built for {self.num_envs} envs, M={self.M}, {self.n_act} "
                             f"{'complex' if self.action_is_complex else 'real'} actions; the env has {venv.num_envs} "
                             f"envs, M={venv.M}, {venv._kernel_n_act} "
                             f"{'complex' if venv.free_action_space else 'real'} actions")
        return venv

    def _action_view(self, actions):
        """(N, A) actions -> (N, A) float64 or (N, 2A) (re, im) float64 tensor with contiguous components"""
        torch = _torch()
        if tuple(actions.shape) != (self.num_envs, self.n_act):
            raise ValueError(f"actions must have shape ({self.num_envs}, {self.n_act})")
        if self.action_is_complex:
            a = torch.view_as_real(actions.to(torch.complex128)).reshape(self.num_envs, 2 * self.n_act)
        else:
            if actions.is_complex():
                raise TypeError("complex actions need free_action_space=True")
            a = actions.to(torch.float64)
        if a.stride(1) != 1:
            a = a.contiguous()
        return a

    @_lib.on_device
    def store_obs(self, planes):
        """Row ``pos`` of the observations := ``planes`` (4M, >= N; plane stride ``planes.stride(0)``): the raw
        observation the next action is taken on.  Call before the step overwrites it."""
        torch = _torch()
        if (planes.dim() != 2 or planes.shape[0] != self.P or planes.shape[1] < self.num_envs or planes.stride(1) != 1
                or planes.dtype != torch.float64 or planes.device != self.device):
            raise ValueError(f"observation planes must be a float64 ({self.P}, {self.num_envs}) tensor on {self.device} "
                             "with contiguous planes")
        _lib.check(self._L.sdcgym_replay_store_obs(ctypes.byref(self._desc), planes.data_ptr(), planes.stride(0),
                                                   self._stream()), "sdcgym_replay_store_obs")

    @_lib.on_device
    def store(self, venv, actions, flags, raw_reward):
        """Complete row ``pos`` after the step of ``venv`` and advance: next observation (``venv.terminal`` where the
        episode ended, else ``venv.S``), ``actions``, ``raw_reward``, done flags."""
        a = self._action_view(actions)
        self._keep = a
        term = venv.terminal
        _lib.check(self._L.sdcgym_replay_store(ctypes.byref(self._desc), venv.S.data_ptr(),
                                               None if term is None else term.data_ptr(), venv.S.stride(0),
                                               flags.data_ptr(), raw_reward.data_ptr(), a.data_ptr(), a.stride(0),
                                               self._stream()), "sdcgym_replay_store")
        self._stored = True

    def add(self, obs_planes, actions, step_out):
        """Store one transition of every env of the buffer's env, which has just stepped: ``obs_planes`` (4M, N) is
        the raw observation ``actions`` were taken on (a copy taken before the step), ``step_out`` the dict its
        ``step_tensor`` returned (flags and raw reward are read from it; the next observation and the terminal planes
        from the env's raw planes)."""
        self.store_obs(obs_planes)
        self.store(self.venv, actions, step_out["flags"], step_out.get("raw_reward", step_out["reward"]))

    # ---- sampling -----------------------------------------------------------------------------------------------
    @_lib.on_device
    def sample(self, batch_size, env=None):
        """``batch_size`` transitions drawn uniformly with replacement (SB3 ``ReplayBuffer.sample``).  ``env``: a
        ``VecNormalize`` whose current statistics normalise observations (``norm_obs``) and rewards
        (``norm_reward``), or ``None`` / a bare env for raw values.  Observations are planes (4M, B), actions (B, A),
        rewards and dones (B,) float64.  Every call draws fresh indices (the call counter advances on the device)."""
        torch = _torch()
        B = int(batch_size)
        if B < 0:
            raise ValueError(f"batch_size must be >= 0, got {batch_size}")
        if not self._stored:
            raise ValueError("ReplayBuffer.sample: the buffer is empty")
        dev, f64 = self.device, torch.float64
        obs = torch.empty((self.P, B), dtype=f64, device=dev)
        next_obs = torch.empty((self.P, B), dtype=f64, device=dev)
        act = torch.empty((B, self.n_act), dtype=torch.complex128 if self.action_is_complex else f64, device=dev)
        rew = torch.empty(B, dtype=f64, device=dev)
        done = torch.empty(B, dtype=f64, device=dev)
        norm = env if env is not None and env is not getattr(env, "venv", env) else None
        mean = var = ret_var = None
        eps, clip_obs, clip_rew = 0.0, 0.0, 0.0
        if norm is not None:
            eps, clip_obs, clip_rew = float(norm.epsilon), float(norm.clip_obs), float(norm.clip_reward)
            if norm.P != self.P:
                raise ValueError(f"normaliser statistics are for M={norm.P // 4}, the buffer holds M={self.M}")
            if norm.norm_obs:
                mean, var = norm.obs_rms.mean.data_ptr(), norm.obs_rms.var.data_ptr()
            if norm.norm_reward:
                ret_var = norm.ret_rms.var.data_ptr()
        _lib.check(self._L.sdcgym_replay_sample(ctypes.byref(self._desc), B, mean, var, ret_var, eps, clip_obs, clip_rew,
                                                obs.data_ptr(), next_obs.data_ptr(), act.data_ptr(), rew.data_ptr(),
                                                done.data_ptr(), self._stream()), "sdcgym_replay_sample")
        return ReplaySamples(obs, act, next_obs, done, rew)


def collect_transitions(env, policy, n_steps, replay):
    """Step ``env`` ``n_steps`` times with ``policy`` and store every transition in ``replay`` - the off-policy
    counterpart of ``collect_rollouts``, with no host round trip per step.

    ``env``: ``VecNormalize`` (or bare ``SDCVecEnv``) that has been ``reset()``.  ``policy(obs_planes) -> actions``
    with ``obs_planes`` a (4M, N) CUDA tensor - normalised when ``env`` normalises observations - and ``actions`` a
    (N, A) CUDA tensor.  The buffer receives the raw planes, terminal planes and reward.  Returns ``replay``."""
    venv = replay.check_env(env)
    N = venv.num_envs
    normalised = env is not venv and getattr(env, "norm_obs", False)
    for _ in range(int(n_steps)):
        obs = env.current_norm_planes[:, :N] if normalised else venv.S[:, :N]
        actions = policy(obs)
        replay.store_obs(venv.S)
        out = env.step_tensor(actions)
        replay.store(venv, actions, out["flags"], out.get("raw_reward", out["reward"]))
    return replay

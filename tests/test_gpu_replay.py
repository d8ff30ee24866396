"""GPU: the device replay buffer (sdc_gym_b200.replay) against a numpy restatement of SB3's off-policy storage and
sampling, and captured in a CUDA graph against eager calls.

SB3 is not installed; its semantics are restated here:
* ``OffPolicyAlgorithm._store_transition`` stores the ORIGINAL observation the action was taken on, the ORIGINAL
  reward (``VecNormalize.get_original_reward``) and as next observation the new original one, except for envs that
  are done, whose next observation is ``infos[i]["terminal_observation"]``;
* ``ReplayBuffer.add`` writes row ``pos`` of a ring of ``buffer_size // n_envs`` rows, ``pos`` wraps to 0 and
  ``full`` becomes true on the first wrap;
* ``ReplayBuffer.sample`` draws ``batch_inds ~ U{0 .. (rows if full else pos) - 1}`` and ``env_inds ~ U{0 .. n_envs -
  1}`` with replacement, normalises observations with the env's current ``obs_rms`` and rewards with ``ret_rms`` and
  returns ``dones * (1 - timeouts)`` (= dones here, see DESIGN.md 5).
Deviations (DESIGN.md 5): terminal observations are stored raw, storage keeps the env's float64 / complex128 types,
indices come from the Philox stream restated in ``sdc_gym_b200.replay.replay_indices``."""
import ctypes

import numpy as np
import pytest

import sdc_gym_b200
from sdc_gym_b200 import _lib
from sdc_gym_b200.precond import fixed_preconditioner
from sdc_gym_b200.replay import ReplayBuffer, collect_transitions, replay_indices

pytestmark = pytest.mark.gpu
KW = dict(M=5, dt=1.0, restol=1e-10, lambda_real_interval=[-100, 0], lambda_imag_interval=[-10, 0],
          blas_variant=_lib.BLAS_SKYLAKEX)
XMIN = np.diag(fixed_preconditioner("min", 5))


class NumpyReplay:  # stable_baselines3.common.buffers.ReplayBuffer (optimize_memory_usage=False), restated
    def __init__(self, buffer_size, n_envs, obs_dim, act_dim, act_dtype):
        self.rows = max(buffer_size // n_envs, 1)
        self.observations = np.zeros((self.rows, n_envs, obs_dim))
        self.next_observations = np.zeros((self.rows, n_envs, obs_dim))
        self.actions = np.zeros((self.rows, n_envs, act_dim), act_dtype)
        self.rewards = np.zeros((self.rows, n_envs))
        self.dones = np.zeros((self.rows, n_envs))
        self.pos, self.full = 0, False

    def add(self, obs, next_obs, action, reward, done):
        self.observations[self.pos] = obs
        self.next_observations[self.pos] = next_obs
        self.actions[self.pos] = action
        self.rewards[self.pos] = reward
        self.dones[self.pos] = done
        self.pos += 1
        if self.pos == self.rows:
            self.full, self.pos = True, 0


def store_transition(rb, last_original_obs, new_original_obs, actions, original_reward, dones, infos):
    """OffPolicyAlgorithm._store_transition, restated (observations as (N, 4M) real planes)"""
    next_obs = new_original_obs.copy()
    for i in np.nonzero(dones)[0]:
        next_obs[i] = planes_of(infos[i]["terminal_observation"][None])[0]
    rb.add(last_original_obs, next_obs, actions, original_reward, dones)


def planes_of(obs):  # (N, 2, M) complex -> (N, 4M) real in plane order
    return np.ascontiguousarray(obs).reshape(obs.shape[0], -1).view(np.float64)


def bits(x):
    import torch

    if isinstance(x, torch.Tensor):
        x = x.cpu().numpy()
    x = np.ascontiguousarray(x)
    if x.dtype == np.complex128:
        x = x.view(np.float64)
    return x.view(np.int64) if x.dtype == np.float64 else x


def table_policy(table):
    import torch

    it = iter([torch.as_tensor(a, device="cuda") for a in table])
    return lambda obs: next(it)


def action_table(rng, steps, n, cplx):
    a = [2 * (XMIN[None] + rng.uniform(-0.1, 0.1, (n, 5))) - 1 for _ in range(steps)]
    if cplx:  # free_action_space: Q_delta diagonals taken as given (no scaling), small imaginary parts
        a = [XMIN[None] + rng.uniform(-0.05, 0.05, (n, 5)) + 1j * rng.uniform(-0.02, 0.02, (n, 5)) for _ in range(steps)]
    return a


def check_against_twin(kind, n, steps, buffer_size, normalised, **env_kw):
    """drive one env through collect_transitions into a ReplayBuffer and a bare twin through step(numpy) into the
    numpy restatement; compare the rings bit for bit"""
    import torch

    cplx = env_kw.get("free_action_space", False)
    table = action_table(np.random.default_rng(11), steps, n, cplx)
    env = sdc_gym_b200.make(kind, num_envs=n, seed=3, **env_kw, **KW)
    env = sdc_gym_b200.VecNormalize(env) if normalised else env
    env.reset()
    rb = ReplayBuffer(buffer_size, env, seed=1)
    collect_transitions(env, table_policy(table), steps, rb)

    twin = sdc_gym_b200.make(kind, num_envs=n, seed=3, **env_kw, **KW)
    ref = NumpyReplay(buffer_size, n, 20, 5, np.complex128 if cplx else np.float64)
    last = planes_of(twin.reset()).copy()
    for s in range(steps):
        obs, reward, dones, infos = twin.step(table[s])
        new = planes_of(obs).copy()
        store_transition(ref, last, new, table[s], reward.copy(), dones.copy(), infos)
        last = new
    torch.cuda.synchronize()
    assert rb.pos == ref.pos and rb.full == ref.full and rb.size() == (ref.rows if ref.full else ref.pos)
    assert np.array_equal(bits(rb.observations.permute(0, 2, 1)), bits(ref.observations))
    assert np.array_equal(bits(rb.next_observations.permute(0, 2, 1)), bits(ref.next_observations))
    assert np.array_equal(bits(rb.actions), bits(ref.actions))
    assert np.array_equal(bits(rb.rewards), bits(ref.rewards))
    assert np.array_equal(rb.dones.cpu().numpy(), ref.dones.astype(np.uint8))
    return env, rb, ref


def test_store_matches_sb3_store_transition_sdc_v1_normalised():
    n = 4096
    env, rb, ref = check_against_twin("sdc-v1", n, 12, 5 * n, True, reward_iteration_only=False)
    assert ref.full and ref.pos == 2  # 12 steps over 5 rows: wrapped twice
    assert 0 < ref.dones.sum() < ref.dones.size  # some episodes ended (terminal substitution exercised), not all


@pytest.mark.parametrize("free_action_space,use_doubles", [(False, True), (True, True), (False, False)])
def test_store_matches_sb3_store_transition_sdc_v0(free_action_space, use_doubles):
    """every sdc-v0 transition is terminal: next_obs is the terminal state, the next row's obs a reset state"""
    n = 2048
    env, rb, ref = check_against_twin("sdc-v0", n, 7, 3 * n, False, free_action_space=free_action_space,
                                      use_doubles=use_doubles)
    assert ref.dones.all()
    obs = rb.observations.cpu().numpy()
    assert np.all(obs[:, 0:10:2] == 1.0) and np.all(obs[:, 1:10:2] == 0.0)  # u of a reset state is 1
    assert not np.array_equal(bits(rb.observations), bits(rb.next_observations))


def _filled(n=64, rows=16, steps=20, seed=9, env_seed=4):
    table = action_table(np.random.default_rng(2), steps, n, False)
    env = sdc_gym_b200.VecNormalize(sdc_gym_b200.make("sdc-v1", num_envs=n, seed=env_seed, reward_iteration_only=False,
                                                      **KW))
    env.reset()
    rb = ReplayBuffer(rows * n, env, seed=seed)
    collect_transitions(env, table_policy(table), steps, rb)
    return env, rb


def _gather(rb, rows, envs):
    obs = rb.observations.cpu().numpy()[rows, :, envs].T  # (P, B)
    nxt = rb.next_observations.cpu().numpy()[rows, :, envs].T
    return (obs, rb.actions.cpu().numpy()[rows, envs], nxt, rb.dones.cpu().numpy()[rows, envs].astype(np.float64),
            rb.rewards.cpu().numpy()[rows, envs])


def test_sample_indices_gather_and_normalisation():
    import torch
    from scipy.stats import chisquare

    n, rows = 64, 16
    env, rb = _filled(n, rows, steps=20)
    assert rb.full and rb.pos == 4
    B = 1 << 20
    # raw sample (call 0): every field is the host-predicted gather, bit for bit
    smp = rb.sample(B)
    r_idx, e_idx = replay_indices(rb.seed, 0, np.arange(B), rows, n)
    want = _gather(rb, r_idx, e_idx)
    for got, w in zip(smp, want):
        assert np.array_equal(bits(got), bits(w))
    counts = np.bincount(r_idx * n + e_idx, minlength=rows * n)
    assert chisquare(counts).pvalue > 1e-3
    # normalised sample (call 1): the same bits as the VecNormalize kernels applied to the raw gather
    B2 = 4096
    smp = rb.sample(B2, env)
    r_idx, e_idx = replay_indices(rb.seed, 1, np.arange(B2), rows, n)
    obs, act, nxt, done, rew = _gather(rb, r_idx, e_idx)
    L = _lib.load()
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    mean, var = env.obs_rms.mean.cpu().numpy(), env.obs_rms.var.cpu().numpy()
    for raw, got in ((obs, smp.observations), (nxt, smp.next_observations)):
        x = torch.as_tensor(np.ascontiguousarray(raw), device="cuda")
        y = torch.empty_like(x)
        _lib.check(L.sdcgym_vecnorm_apply(20, B2, B2, x.data_ptr(), env.obs_rms.mean.data_ptr(),
                                          env.obs_rms.var.data_ptr(), env.epsilon, env.clip_obs, y.data_ptr(), stream),
                   "apply")
        assert torch.equal(got.view(torch.int64), y.view(torch.int64))
        w = np.clip((raw - mean[:, None]) / np.sqrt(var[:, None] + env.epsilon), -env.clip_obs, env.clip_obs)
        assert np.allclose(got.cpu().numpy(), w, rtol=1e-10, atol=1e-10)
        assert np.abs(w).max() > 0.5  # the statistics are not trivial
    r = torch.as_tensor(rew, device="cuda")
    ro = torch.empty_like(r)
    _lib.check(L.sdcgym_vecnorm_reward(B2, r.data_ptr(), None, env.ret_rms.var.data_ptr(), env.epsilon, env.clip_reward,
                                       1, ro.data_ptr(), None, stream), "reward")
    assert torch.equal(smp.rewards.view(torch.int64), ro.view(torch.int64))
    ret_var = float(env.ret_rms.var.cpu().numpy()[0])
    assert np.allclose(smp.rewards.cpu().numpy(), np.clip(rew / np.sqrt(ret_var + env.epsilon), -10, 10), rtol=1e-12)
    assert ret_var != 1.0
    assert np.array_equal(bits(smp.actions), bits(act)) and np.array_equal(bits(smp.dones), bits(done))
    assert rb.counters[2].item() == 2


def test_sample_before_the_first_wrap_draws_stored_rows_only():
    n, rows = 64, 16
    env, rb = _filled(n, rows, steps=5)
    assert not rb.full and rb.pos == 5 and rb.size() == 5
    B = 8192
    smp = rb.sample(B)
    r_idx, e_idx = replay_indices(rb.seed, 0, np.arange(B), 5, n)
    assert r_idx.max() == 4 and np.array_equal(np.unique(r_idx), np.arange(5))
    for got, w in zip(smp, _gather(rb, r_idx, e_idx)):
        assert np.array_equal(bits(got), bits(w))
    assert not np.any(smp.next_observations.cpu().numpy()[0:10:2] == 0.0)  # no unwritten (zero) row was drawn


def test_consecutive_calls_differ_and_a_seed_reproduces():
    env, rb = _filled(seed=9)
    a1, a2 = rb.sample(512), rb.sample(512)
    assert not np.array_equal(bits(a1.observations), bits(a2.observations))
    env_b, rb_b = _filled(seed=9)
    b1, b2 = rb_b.sample(512), rb_b.sample(512)
    for x, y in zip(a1 + a2, b1 + b2):
        assert np.array_equal(bits(x), bits(y))
    env_c, rb_c = _filled(seed=10)
    assert not np.array_equal(bits(rb_c.sample(512).observations), bits(a1.observations))


def test_collect_and_sample_captured_in_a_cuda_graph_replay_like_eager_calls():
    """collect_transitions (policy, env steps, statistics, normalisation, stores) + sample captured ONCE and replayed
    three times: buffers, counters, samples, env state and normaliser statistics bit-identical to an eager twin"""
    import torch

    n, k, B = 4096, 4, 2048
    w = torch.linspace(-1.0, 1.0, 20, dtype=torch.float64, device="cuda")

    def policy(obs_planes):  # deterministic and capturable
        s = torch.tanh((obs_planes * w[:, None]).sum(0))
        return torch.stack([torch.tanh(s * (j + 1) * 0.7) for j in range(5)], dim=1) * 0.9

    def make():
        e = sdc_gym_b200.VecNormalize(sdc_gym_b200.make("sdc-v1", num_envs=n, seed=7, output="torch",
                                                        reward_iteration_only=False, **KW))
        e.reset()
        return e, ReplayBuffer(3 * n, e, seed=5)

    (ea, ra), (eb, rb) = make(), make()
    for e, r in ((ea, ra), (eb, rb)):  # eager warm-up of both
        collect_transitions(e, policy, k, r)
        r.sample(B, e)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        with torch.cuda.graph(graph, stream=side):
            collect_transitions(eb, policy, k, rb)
            smp_b = rb.sample(B, eb)
    torch.cuda.current_stream().wait_stream(side)
    for it in range(3):
        collect_transitions(ea, policy, k, ra)
        smp_a = ra.sample(B, ea)
        graph.replay()
        torch.cuda.synchronize()
        for name in ("obs_store", "next_obs_store", "actions", "rewards", "dones", "counters"):
            assert np.array_equal(bits(getattr(ra, name)), bits(getattr(rb, name))), (it, name)
        for x, y in zip(smp_a, smp_b):
            assert np.array_equal(bits(x), bits(y)), it
        assert torch.equal(ea.venv.S.view(torch.int64), eb.venv.S.view(torch.int64))
        assert torch.equal(ea.venv.episodes, eb.venv.episodes)
        for rms in ("obs_rms", "ret_rms"):
            for f in ("mean", "var", "count2"):
                a, b = getattr(getattr(ea, rms), f), getattr(getattr(eb, rms), f)
                assert torch.equal(a.view(torch.int64), b.view(torch.int64)), (it, rms, f)
    assert ra.counters.tolist() == [(k * 4) % 3, 1, 4]  # 16 stores over 3 rows, four sample calls
    assert int(ra.dones.sum()) > 0


def test_refusals_and_empty_batches():
    import torch

    kw = dict(num_envs=64, **KW)
    with pytest.raises(NotImplementedError):
        ReplayBuffer(640, sdc_gym_b200.make("sdc-v0", collect_states=True, **kw))
    with pytest.raises(ValueError, match="fixed preconditioner"):
        ReplayBuffer(640, sdc_gym_b200.make("sdc-v1", prec="LU", **kw))
    with pytest.raises(ValueError, match="keep_terminal"):
        ReplayBuffer(640, sdc_gym_b200.make("sdc-v1", keep_terminal=False, **kw))
    env = sdc_gym_b200.make("sdc-v1", **kw)
    env.reset()
    rb = ReplayBuffer(640, env)
    with pytest.raises(ValueError, match="empty"):
        rb.sample(8)
    zero = lambda obs: torch.zeros((64, 5), dtype=torch.float64, device="cuda")  # noqa: E731
    for other in (sdc_gym_b200.make("sdc-v1", **{**kw, "num_envs": 128}),
                  sdc_gym_b200.make("sdc-v1", **{**kw, "M": 4})):
        other.reset()
        with pytest.raises(ValueError, match="built for"):
            collect_transitions(other, zero, 1, rb)
    collect_transitions(env, zero, 2, rb)
    with pytest.raises(ValueError, match="batch_size"):
        rb.sample(-1)
    e = rb.sample(0)
    assert [tuple(t.shape) for t in e] == [(20, 0), (0, 5), (20, 0), (0,), (0,)]
    assert all(t.dtype == torch.float64 for t in e)
    assert rb.pos == 2 and rb.counters[2].item() == 0  # an empty batch draws nothing

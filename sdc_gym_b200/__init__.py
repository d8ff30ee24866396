"""sdc_gym_b200 - B200-native (sm_100a) implementation of sdc-gym's data-parallel hot path.

Public surface (mirrors the reference's, see DESIGN.md):

* ``make(envname, num_envs=..., **kwargs)`` / ``SDCVecEnv`` - batched ``sdc-v0`` / ``sdc-v1`` envs with the
  DummyVecEnv protocol (reference ``sdc_gym/__init__.py:3-13``, ``utils/utils.py:235-315``); ``sdc-v4``
  (``SDCForceVecEnv``, ``sdc_gym/__init__.py:15-19``) composes the same kernels.
* ``SpectralRadiusLoss`` / ``ResidualLoss`` - batched forward values of the ``dp_playground.py:186-258`` losses.
* ``IterationCounts`` - iteration counts and success rate of the ``sdc-v0`` full solve over a lambda batch or grid
  (the reference's ``test_model`` evaluation), counted on the device.
* ``VecNormalize`` - device-side observation / reward normalisation (SB3 semantics).
* ``RolloutBuffer`` / ``collect_rollouts`` / ``GraphedRollout`` (on-policy) and ``ReplayBuffer`` /
  ``collect_transitions`` (off-policy) - device-resident transition storage.
* ``collocation_matrix`` - the Gauss-Radau-right Q the reference takes from pySDC.

The compute path is ``libsdcgym.so`` (hand-written CUDA, C ABI in ``include/sdcgym.h``); importing this
package does not need a GPU, constructing an env does.
"""
from .collocation import CollGaussRadauRight, collocation_matrix  # noqa: F401
from .precond import fixed_preconditioner, num_actions, qdmat_from_output  # noqa: F401

REGISTRY = {
    # id: (env kind, max_episode_steps)  - sdc_gym/__init__.py:3-13
    "sdc-v0": ("SDC_Full_Env", 1),
    "sdc-v1": ("SDC_Step_Env", 50),
    "sdc-v4": ("SDC_Full_Force_Env", 50),  # sdc_gym/__init__.py:15-19 (force_env.py)
}

__all__ = ["make", "make_env", "SDCVecEnv", "SDCForceVecEnv", "SpectralRadiusLoss", "ResidualLoss", "IterationCounts", "PopulationSummary", "VecNormalize", "VecCheckNan", "RolloutBuffer", "collect_rollouts", "GraphedRollout",
           "ReplayBuffer", "collect_transitions",
           "collocation_matrix", "CollGaussRadauRight", "fixed_preconditioner", "num_actions", "REGISTRY", "register_gym"]


def __getattr__(name):
    # lazy: keep `import sdc_gym_b200` free of torch / CUDA
    if name == "SDCVecEnv":
        from .vec_env import SDCVecEnv
        return SDCVecEnv
    if name == "SDCForceVecEnv":
        from .force_env import SDCForceVecEnv
        return SDCForceVecEnv
    if name in ("SpectralRadiusLoss", "ResidualLoss"):
        from . import loss
        return getattr(loss, name)
    if name in ("IterationCounts", "CountSummary", "PopulationSummary"):
        from . import iterations
        return getattr(iterations, name)
    if name in ("VecNormalize", "VecCheckNan"):
        from . import vec_normalize
        return getattr(vec_normalize, name)
    if name in ("RolloutBuffer", "collect_rollouts", "GraphedRollout"):
        from . import rollout
        return getattr(rollout, name)
    if name in ("ReplayBuffer", "collect_transitions"):
        from . import replay
        return getattr(replay, name)
    raise AttributeError(name)


def make(envname, num_envs=1, **kwargs):
    """``gym.make(envname, **kwargs)`` for a whole batch: returns an ``SDCVecEnv`` with ``num_envs`` envs."""
    if envname not in REGISTRY:
        raise KeyError(f"unknown env id {envname!r}; registered: {sorted(REGISTRY)}")
    if envname == "sdc-v4":
        from .force_env import SDCForceVecEnv
        return SDCForceVecEnv(envname, num_envs=num_envs, **kwargs)
    from .vec_env import SDCVecEnv
    return SDCVecEnv(envname, num_envs=num_envs, **kwargs)


def register_gym(force=False):
    """Optional shim for the reference's scripts: when ``gym`` (or ``gymnasium``) is importable, register the ids of
    ``sdc_gym/__init__.py:3-13`` so that ``gym.make('sdc-v0', **kwargs)`` resolves to this package instead of the
    numpy env.  The entry point builds a single-env ``SDCVecEnv`` (``num_envs=1``) behind a thin ``gym.Env`` adapter;
    batched use goes through ``make`` / ``make_env``, which need no gym at all.  Returns the ids registered (an empty
    list when no gym package is installed - never an error: gym is not a dependency of the path)."""
    done = []
    for modname in ("gym", "gymnasium"):
        try:
            gym = __import__(modname)
            from importlib import import_module
            registration = import_module(modname + ".envs.registration")
        except Exception:
            continue
        registry = getattr(registration, "registry", {})
        specs = getattr(registry, "env_specs", registry)
        for env_id, (_cls, max_steps) in REGISTRY.items():
            if env_id in specs and not force:
                continue
            if env_id in specs:
                try:
                    del specs[env_id]
                except Exception:
                    pass
            gym.register(id=env_id, entry_point="sdc_gym_b200.gym_adapter:make_single",
                         kwargs={"envname": env_id}, max_episode_steps=max_steps)
            done.append(f"{modname}:{env_id}")
    return done


_ENV_ARGS = ("M", "dt", "restol", "lambda_real_interval", "lambda_imag_interval",
             "lambda_real_interpolation_interval", "norm_factor", "residual_weight", "step_penalty",
             "reward_iteration_only", "reward_strategy", "collect_states")


def make_env(args, num_envs=None, include_norm=False, norm_reward=True, **kwargs):
    """Drop-in for the reference's ``utils.make_env`` (``utils/utils.py:235-315``): same argument handling
    (``kwargs`` beat ``args``), returns the batched env, optionally wrapped in the device ``VecNormalize``."""
    if num_envs is None:
        num_envs = args.num_envs
    args_kwargs = {a: kwargs.pop(a, getattr(args, a)) for a in _ENV_ARGS}
    all_kwargs = {**kwargs, **args_kwargs}
    if getattr(args, "model_class", None) == "SAC":
        all_kwargs["use_doubles"] = False
    seed = all_kwargs.pop("seed", getattr(args, "seed", None))
    env = make(args.envname, num_envs=num_envs, seed=seed, **all_kwargs)
    if include_norm:
        from .vec_normalize import VecNormalize
        if getattr(args, "env_path", None) is not None:  # utils/utils.py:296-297: resume a saved normaliser
            env = VecNormalize.load(str(args.env_path), env)
        else:
            model_kwargs = getattr(args, "model_kwargs", None) or {}
            extra = {"gamma": model_kwargs["gamma"]} if "gamma" in model_kwargs else {}
            env = VecNormalize(env, norm_obs=getattr(args, "norm_obs", True), norm_reward=norm_reward, **extra)
    if getattr(args, "debug_nans", False):
        from .vec_normalize import VecCheckNan
        env = VecCheckNan(env, raise_exception=True)
    return env

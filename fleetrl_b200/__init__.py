"""fleetrl_b200 — the FleetRL environment step (FleetEnv.reset/step) as hand-written sm_100a CUDA behind a C ABI.

Only what the path needs lives here: csrc/ (kernels + C ABI), the ctypes binding, and the host-side mirror of
the reference's FleetEnv / SB3 VecEnv interface.
"""
__version__ = "0.1.0"


def __getattr__(name):  # lazy: importing the package must not require torch / CUDA (config and table code is pure NumPy)
    if name in ("FleetVecEnv", "FleetEnv", "LazyInfos"):
        from . import vec_env
        return getattr(vec_env, name)
    if name == "FleetVecNormalize":
        from . import normalize
        return normalize.FleetVecNormalize
    if name in ("FleetRolloutBuffer", "RolloutBufferSamples", "collect_rollouts"):
        from . import rollout
        return getattr(rollout, name)
    if name in ("FleetMlpPolicy", "ppo_loss", "ppo_train"):
        from . import ppo
        return getattr(ppo, name)
    if name in ("build_fleet", "FleetInputs"):
        from . import tables
        return getattr(tables, name)
    raise AttributeError(name)

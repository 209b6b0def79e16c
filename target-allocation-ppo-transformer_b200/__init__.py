"""B200-native batched UAV->target allocation environment (rollout path of
Dingyf717/target-allocation-ppo-transformer), hand-written sm_100a CUDA behind a C ABI.

The directory name carries hyphens (it is fixed by the project layout), so import it through the
repo-root shim:  `import uavenv_b200 as ub`  ->  ub.UAVEnvBatched, ub.UAVEnv, ub.cfg, ub.compute_gae.
Sub-packages mirror the reference tree: configs/, envs/, agents/, networks/.
"""
from .configs.config import Config, cfg, HARD_MODE  # noqa: F401


def __getattr__(name):  # torch / CUDA are only touched when the env classes are asked for
    if name in ("UAVEnvBatched", "UAVEnv"):
        from .envs import uav_env
        return getattr(uav_env, name)
    if name in ("compute_gae", "normalize_advantages", "PPOAgent"):
        from .agents import ppo
        return getattr(ppo, name)
    if name in ("TransformerActorCritic", "TransformerBlock"):
        from .networks import transformer_net
        return getattr(transformer_net, name)
    if name == "FusedPolicyForward":
        from .networks.fused_forward import FusedPolicyForward
        return FusedPolicyForward
    if name == "FusedTrunks":
        from .networks.fused_train import FusedTrunks
        return FusedTrunks
    if name == "train":                      # the submodule itself is callable: ub.train(...) == ub.train.train(...)
        import importlib
        return importlib.import_module(__name__ + ".train")
    if name in ("evaluate", "evaluate_baseline", "EpisodeRecorder", "load_checkpoint"):
        from . import evaluation
        return getattr(evaluation, name)
    if name in ("allocate", "improve_allocation", "upper_bound"):
        from . import allocation
        return getattr(allocation, name)
    if name in ("analyze_environment_difficulty", "record_decisions"):
        from . import diagnostics
        return getattr(diagnostics, name)
    if name == "load_library":
        from ._capi import load
        return load
    raise AttributeError(name)

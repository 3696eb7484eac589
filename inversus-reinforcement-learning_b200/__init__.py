"""inversus_b200 -- B200-native batched INVERSUS simulator (drop-in for the rollout path of
Jason-Hoford/inversus-reinforcement-learning: inversus_rl/env_wrappers.py MultiEnvRunner).

The directory is named `inversus-reinforcement-learning_b200` (not importable as written); the
repo-root module `inversus_b200.py` registers it under the importable name `inversus_b200`.

Public surface
    MultiEnvRunner, SingleInversusRLEnv, discrete_to_action   reference-shaped numpy API
    BatchedInversus                                           tensor-native API (device views)
    InversusCNNPolicy, PPOAgent, DeviceRollout, train_*       GPU-resident PPO around it (next rows)
    evaluate                                                  K episodes per env vs the dummy or another policy
    shard_range, reduce_rollout_stats                         multi-GPU layout helpers
    build_library, library_path                               in-tree nvcc build of the C-ABI .so
"""
from . import constants
from ._build import build_library
from ._capi import InversusError, library_path

__all__ = ["constants", "build_library", "library_path", "InversusError", "BatchedInversus",
           "MultiEnvRunner", "SingleInversusRLEnv", "discrete_to_action", "build_observation", "PlayerId", "InfoList",
           "shard_range", "reduce_rollout_stats", "InversusCNNPolicy", "make_policy_from_env", "PPOAgent",
           "DeviceRollout", "compute_gae", "train_vs_dummy", "train_selfplay", "evaluate"]

_LAZY = {
    "BatchedInversus": ("simulator", "BatchedInversus"),
    "MultiEnvRunner": ("env_wrappers", "MultiEnvRunner"),
    "SingleInversusRLEnv": ("env_wrappers", "SingleInversusRLEnv"),
    "discrete_to_action": ("env_wrappers", "discrete_to_action"),
    "build_observation": ("env_wrappers", "build_observation"),
    "PlayerId": ("env_wrappers", "PlayerId"),
    "InfoList": ("env_wrappers", "InfoList"),
    "InversusCNNPolicy": ("policies", "InversusCNNPolicy"),
    "make_policy_from_env": ("policies", "make_policy_from_env"),
    "PPOAgent": ("ppo_agent", "PPOAgent"),
    "DeviceRollout": ("ppo_agent", "DeviceRollout"),
    "compute_gae": ("ppo_agent", "compute_gae"),
    "train_vs_dummy": ("training", "train_vs_dummy"),
    "train_selfplay": ("training", "train_selfplay"),
    "evaluate": ("evaluate", "evaluate"),
    "shard_range": ("sharding", "shard_range"),
    "reduce_rollout_stats": ("sharding", "reduce_rollout_stats"),
}


def __getattr__(name):  # lazy, like the reference's inversus_rl/__init__.py, so torch loads on demand
    if name in _LAZY:
        import importlib
        mod, attr = _LAZY[name]
        value = getattr(importlib.import_module(f"{__name__}.{mod}"), attr)
        if name == mod:  # importing the submodule bound its name here: keep the function instead
            globals()[name] = value
        return value
    raise AttributeError(f"module {__name__!r} has no attribute {name!r}")

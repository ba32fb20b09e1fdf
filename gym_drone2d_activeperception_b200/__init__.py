"""drone2d-b200: B200-native batched simulator for the per-step hot path of gym-Drone2D-ActivePerception.

Public API (mirrors the reference's names):
    Params            -- reference utils.Params (utils.py:65-171)
    Drone2DVecEnv     -- batched Drone2DEnv2 (envs/drone_v2.py) on one GPU
    generate_world(s) -- host-side world generation from seeds (drone_v2.py:12-117)
"""
from .params import Params, grid_type, state_machine  # noqa: F401
from .world import generate_world, generate_worlds, count_agents, load_static_map, world_key, split_world_key  # noqa: F401


def __getattr__(name):
    # torch / CUDA are imported lazily so that host-only tooling (world generation, Params) works without them
    if name in ("Drone2DVecEnv", "make_config", "oxford_cos_threshold"):
        from . import vec_env
        return getattr(vec_env, name)
    if name in ("Drone2DEnv2", "make"):
        from . import env
        return getattr(env, name)
    raise AttributeError(name)


__version__ = "0.1.0"

"""B200-native batched env step for the hrl_pybullet_envs environments.

    import hrl_pybullet_envs_b200 as hrl
    env = hrl.make('AntGatherBulletEnv-v0')            # gym-style single env (README.md:20-37)
    vec = hrl.VecEnv('AntGatherBulletEnv-v0', 4096)    # step(actions[N,8]) -> torch tensors
"""
from .config import ENV_IDS, HrlConfig  # noqa: F401
from .gym_shim import Box, make, register, registry  # noqa: F401

__all__ = ["ENV_IDS", "HrlConfig", "Box", "make", "register", "registry", "VecEnv", "RolloutBuffer", "RunningNormalizer"]


def __getattr__(name):  # torch is only needed for the CUDA path
    if name in ("VecEnv", "RolloutBuffer"):
        from . import vec_env
        return getattr(vec_env, name)
    if name == "RunningNormalizer":
        from . import normalize
        return normalize.RunningNormalizer
    if name in ("gather_sensor", "sense_walls"):
        from . import vec_env
        return getattr(vec_env, name)
    raise AttributeError(name)

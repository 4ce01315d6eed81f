"""Environment construction (reference: xuance/environment/__init__.py:12-76 ``make_envs``)."""
from .envs import REGISTRY_ENV, XuanCeEnvWrapper, CartPoleEnv, SyntheticAtariEnv, SyntheticMuJoCoEnv
from .ma_envs import SyntheticSMACEnv, XuanCeMultiAgentEnvWrapper
from .vector_envs import (REGISTRY_VEC_ENV, VecEnv, DummyVecEnv, DummyVecEnv_Atari, SubprocVecEnv, SubprocVecEnv_Atari,
                          ShmSubprocVecEnv, ShmSubprocVecEnv_Atari, DummyVecMultiAgentEnv, SubprocVecMultiAgentEnv)
from .tensor_env import TensorEnvWrapper


def make_envs(config):
    """``config.env_id`` selects the raw env, ``config.vectorize`` the vector wrapper, ``config.parallels`` the count.
    Under distributed training every rank builds its own ``parallels / world_size`` envs with rank-distinct seeds
    (the reference hard-codes rank = 1 here, appendix B #15)."""
    import os
    world = int(os.environ.get("WORLD_SIZE", "1")) if getattr(config, "distributed_training", False) else 1
    rank = int(os.environ.get("RANK", "0")) if world > 1 else 0
    n = config.parallels // world
    base_seed = getattr(config, "env_seed", 1) + rank * n
    if getattr(config, "env_name", None) == "StarCraft2":       # SMAC-shaped synthetic multi-agent env (QMIX path)
        kw = {k: getattr(config, k) for k in ("episode_limit", "p_death", "p_mask") if hasattr(config, k)}
        map_name = config.env_id
        fns = [lambda env_seed=None, **_: XuanCeMultiAgentEnvWrapper(SyntheticSMACEnv(seed=env_seed, map_name=map_name, **kw))
               for _ in range(n)]
        vec = getattr(config, "vectorize", "Dummy_StarCraft2")
        vec_cls = REGISTRY_VEC_ENV[vec] if vec in ("SubprocVecMultiAgentEnv", "Subproc_StarCraft2") else DummyVecMultiAgentEnv
        return vec_cls(fns, base_seed)
    env_cls = REGISTRY_ENV[config.env_id]

    def thunk(i):
        return lambda: XuanCeEnvWrapper(env_cls(seed=base_seed + i))

    vec_cls = REGISTRY_VEC_ENV[getattr(config, "vectorize", "DummyVecEnv")]
    return vec_cls([thunk(i) for i in range(n)], base_seed)

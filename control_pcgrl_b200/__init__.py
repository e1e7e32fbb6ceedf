"""control_pcgrl_b200 -- B200-native batched PCGRL environment step (drop-in for control-pcgrl's env path).

Public surface (mirrors the reference's names; see INTEGRATION.md):
    make("binary-narrow-v0", cfg=cfg)      single-env gym façade          (control_pcgrl/__init__.py)
    make_env(cfg)                          wrapped env as rl/envs.py builds it (cfg.multiagent.n_agents: + MultiAgentWrapper)
    BatchedPcgrlEnv(cfg, n_envs)           N grids on one GPU, one fused launch per step
    PcgrlVectorEnv(cfg, num_envs)          vector-env seam with auto-reset and device observations
    make_rllib_vector_env(cfg, num_envs)   ray.rllib VectorEnv (vector_reset / reset_at / vector_step) over one shard
    make_config(...)                       dataclass with the reference's cfg field names
    level_distances / level_knn / level_diversity   Hamming distances between levels, kNN novelty, group diversity
Importing this package never touches CUDA; constructing an env loads libpcgrl_sm100.so and fails
loudly if it (or a GPU) is missing.
"""
from .config import Config, TaskConfig, make_config  # noqa: F401
from .problems import PROBLEM_NAMES, get_spec  # noqa: F401
from .registry import REGISTRY, make, make_batched  # noqa: F401


def __getattr__(name):
    if name in ("BatchedPcgrlEnv", "level_distances", "level_knn", "level_diversity"):
        from . import batched_env
        return getattr(batched_env, name)
    if name in ("PcgrlVectorEnv", "make_rllib_vector_env"):
        from . import vector_env
        return getattr(vector_env, name)
    if name in ("PcgrlEnv", "PcgrlCtrlEnv", "PcgrlEnv3D", "ControlWrapper", "UniformNoiseyTargets", "make_env",
                "CroppedImagePCGRLWrapper", "ActionMapImagePCGRLWrapper", "CAactionWrapper", "MultiAgentWrapper"):
        from . import envs
        return getattr(envs, name)
    raise AttributeError(name)


__version__ = "0.1.0"

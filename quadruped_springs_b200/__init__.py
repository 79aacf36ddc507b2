"""quadruped_springs_b200: B200-native batched simulator for the hot path of
francescovezzi/quadruped-springs (QuadrupedGymEnv.step for N independent Go1s)."""
from .env import (  # noqa: F401
    ActionInterfaceCollection, BatchedQuadruped, BatchedQuadrupedGymEnv, EnvRandomizerCollection,
    MotorInterfaceCollection, SensorCollection, TaskCollection,
)
from .hopf_network import HopfNetwork  # noqa: F401
from . import demo, load_model, ops, stats, substep, vec_env  # noqa: F401
from .substep import SubstepRecorder  # noqa: F401
from .vec_env import BatchedVecEnv, MlpPolicyTorch, VecNormalizeTorch  # noqa: F401

__all__ = ["BatchedQuadrupedGymEnv", "BatchedQuadruped", "HopfNetwork", "ops", "BatchedVecEnv", "VecNormalizeTorch",
           "MlpPolicyTorch", "SubstepRecorder"]

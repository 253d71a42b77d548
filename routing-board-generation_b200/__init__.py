"""B200-native batched routing-board engine: the ParallelRandomWalk / SeedExtension /
Uniform generators and the Jumanji Connector reset / step behind the reference's own
plugin surface.  Host side in Python over a C-ABI CUDA library (include/rbg_b200.h)."""
from . import _lib, engine, sharding  # noqa: F401
from ._lib import RbgError, launch_count  # noqa: F401
from .benchmarking import EvaluateEmptyBoard, PolicyEvaluator, RandomAgentEvaluator  # noqa: F401
from .board_generation import ParallelRandomWalkBoard, SeedExtensionBoard, SequentialRandomWalkBoard  # noqa: F401
from .connector import Connector, DenseRewardFn, MultiToSingleWrapper, VmapAutoResetWrapper, make_random_policy_connector  # noqa: F401
from .engine import PRNGKey, split  # noqa: F401
from .interface import BoardGenerator, BoardName  # noqa: F401
from .offline_generation import BoardDatasetGeneratorJAX  # noqa: F401
from .online_generators import Generator, ParallelRandomWalkGenerator, SeedExtensionGenerator, SequentialRandomWalkGenerator, UniformRandomGenerator  # noqa: F401
from .types import Agent, Observation, State, TimeStep  # noqa: F401

__all__ = [
    "Agent", "BoardDatasetGeneratorJAX", "BoardGenerator", "BoardName", "Connector", "DenseRewardFn", "EvaluateEmptyBoard", "Generator", "MultiToSingleWrapper", "Observation",
    "ParallelRandomWalkBoard", "ParallelRandomWalkGenerator", "PolicyEvaluator", "PRNGKey", "RandomAgentEvaluator", "RbgError", "SeedExtensionBoard", "SeedExtensionGenerator", "SequentialRandomWalkBoard", "SequentialRandomWalkGenerator",
    "State", "TimeStep", "UniformRandomGenerator", "VmapAutoResetWrapper", "engine", "launch_count", "make_random_policy_connector",
    "sharding", "split",
]

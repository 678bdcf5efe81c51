"""neorl_industrial -- B200-native drop-in for the env path of danieleschmidt/neoRL-industrial-gym.

``import neorl_industrial as ni; env = ni.make('ChemicalReactor-v0', num_envs=65536)``. The public names of
the reference's step path are kept (make, evaluate_with_safety, SafetyConstraint, SafetyMetrics, the three
env classes, ``neorl_industrial.safety.SafetyWrapper``); the arithmetic runs in hand-written sm_100a CUDA
kernels behind a C ABI (include/nig_b200.h). No JAX, no Triton, no CPU fallback.
"""
__version__ = "0.1.0+b200"

from .core.types import BatchedSafetyMetrics, DatasetQuality, IndustrialState, SafetyConstraint, SafetyMetrics
from .environments import ChemicalReactorEnv, IndustrialEnv, PowerGridEnv, RobotAssemblyEnv
from .safety import BoundConstraint, SafetyWrapper
from .utils import evaluate_with_safety, make
from .vector import NativeEnv
from .torch_env import TorchIndustrialEnv
from .policies import MLPPolicy
from ._native import build_native

__all__ = [
    "__version__", "DatasetQuality", "IndustrialState", "SafetyConstraint", "SafetyMetrics", "BatchedSafetyMetrics",
    "IndustrialEnv", "ChemicalReactorEnv", "PowerGridEnv", "RobotAssemblyEnv", "SafetyWrapper", "BoundConstraint",
    "make", "evaluate_with_safety", "NativeEnv", "TorchIndustrialEnv", "MLPPolicy", "build_native",
]

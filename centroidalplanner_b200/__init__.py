"""B200-native batched evaluator for CentroidalPlanner's IFOPT problem.

The product is `libcplb.so` (hand-written sm_100a CUDA behind the C ABI in
include/cpl_batched.h); this package is the thin host mirror of the reference's interface.
Importing it never touches oracle/ and never falls back to a CPU evaluation.
"""
from ._cabi import (BLOCK_COM, BLOCK_FORCE, BLOCK_NORMAL, BLOCK_POSITION, COMPONENT_MAJOR, ENV_GROUND, ENV_NONE,
                    ENV_SUPERQUADRIC, INSTANCE_MAJOR, LIB_PATH)
from .autodiff import constraints_and_cost
from .native_solver import NativeInteriorPoint
from .planner import BatchedCentroidalPlanner, BatchedCoMPlanner
from .problem import BatchedCplProblem, EnvironmentClass, Ground, Superquadric

__all__ = ["BatchedCplProblem", "NativeInteriorPoint", "BatchedCentroidalPlanner", "BatchedCoMPlanner", "EnvironmentClass", "Ground", "Superquadric", "INSTANCE_MAJOR", "COMPONENT_MAJOR",
           "ENV_NONE", "ENV_GROUND", "ENV_SUPERQUADRIC", "BLOCK_COM", "BLOCK_FORCE", "BLOCK_POSITION", "BLOCK_NORMAL",
           "LIB_PATH", "constraints_and_cost"]

"""dart_planner_b200 -- B200-native batched SE(3)-MPC solve path for DART-Planner.

Drop-in for `dart_planner.planning.se3_mpc_planner.SE3MPCPlanner` (same plan/config API)
plus a batched entry point (`plan_batch`) that solves thousands of independent problems per
call on hand-written sm_100a kernels through a C ABI (include/dart_se3mpc.h).
There is no CPU fallback.
"""
from .config import SE3MPCConfig, load_planner_config  # noqa: F401
from .types import DroneState, Trajectory  # noqa: F401
from .planner import (BatchSolution, SE3MPCPlanner, extract_batch, plan_batch,  # noqa: F401
                      solve_batch_tensors)
from .mapper import DenseOccupancyGrid, SensorObservation  # noqa: F401
from .mission import BatchedMissionGoals, SemanticWaypoint  # noqa: F401
from .wire import SignedEnvelope  # noqa: F401
from .closed_loop import ClosedLoopSim  # noqa: F401
from .differentiable import plan_batch_differentiable  # noqa: F401
from .sharding import ShardedSolver, replicate_map, shard_range  # noqa: F401

__all__ = ["SE3MPCConfig", "load_planner_config", "DroneState", "Trajectory", "SE3MPCPlanner",
           "BatchSolution", "plan_batch", "plan_batch_differentiable", "extract_batch", "solve_batch_tensors", "DenseOccupancyGrid", "SensorObservation", "ClosedLoopSim",
           "BatchedMissionGoals", "SemanticWaypoint", "SignedEnvelope",
           "ShardedSolver", "replicate_map", "shard_range"]

from .ik_solver import BatchIKResult, IKResult, IKSolver, JacobianIKController, solve_ik  # noqa: F401
from .move import MoveIKSkill, plan_moves, plan_pose_moves  # noqa: F401

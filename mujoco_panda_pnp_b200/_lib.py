"""ctypes binding of libpnp_b200.so (the C ABI in include/pnp_b200.h).

There is no CPU fallback: if the shared library is missing or a call fails this module raises.
The library is built in-tree by ``mujoco_panda_pnp_b200/csrc/build.py`` (nvcc, sm_100a).
"""

from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_int, c_int32, c_int64, c_uint64, c_void_p

from .tree import PnpTreeStruct

LIB_NAME = "libpnp_b200.so"
LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), LIB_NAME)

PNP_KIN_AUTO, PNP_KIN_GENERIC, PNP_KIN_SPECIALIZED, PNP_KIN_SPEC_LANE, PNP_KIN_SPEC_PAIR = 0, 1, 2, 3, 4
PNP_IK_CONVERGED, PNP_IK_SUCCESS = 1, 2
KINEMATICS = {"auto": PNP_KIN_AUTO, "generic": PNP_KIN_GENERIC, "specialized": PNP_KIN_SPECIALIZED,
              "spec_lane": PNP_KIN_SPEC_LANE, "spec_pair": PNP_KIN_SPEC_PAIR}

_ERRNAMES = {-1: "PNP_EINVAL", -2: "PNP_ENOTREE", -3: "PNP_ENODEVICE", -4: "PNP_ENOMEM"}


class PnpIkParams(ctypes.Structure):
    _fields_ = [
        ("max_iters", c_int32),
        ("kinematics", c_int32),
        ("pos_thresh", c_double),
        ("damping", c_double),
        ("step_limit", c_double),
    ]


class PnpRewardParams(ctypes.Structure):
    _fields_ = [
        ("sparse", c_int32),
        ("n_tasks", c_int32),
        ("initial_object_height", c_double),
        ("distance_threshold", c_double),
        ("high_pick_z", c_double),
        ("threshold_report_tol", c_double),
    ]


class PnpMoveParams(ctypes.Structure):
    _fields_ = [
        ("pos_thresh", c_double),
        ("step_size", c_double),
        ("max_traj_points", c_int32),
        ("max_outer", c_int32),
        ("traj_cap", c_int32),
        ("compute_order", c_int32),
    ]


class PnpMovePoseParams(ctypes.Structure):
    _fields_ = [
        ("pos_thresh", c_double),
        ("rot_thresh", c_double),
        ("step_size", c_double),
        ("rot_step", c_double),
        ("ik_rot_thresh", c_double),
        ("ik_rot_weight", c_double),
        ("max_traj_points", c_int32),
        ("traj_cap", c_int32),
    ]


class PnpNormalizeParams(ctypes.Structure):
    _fields_ = [
        ("mean", c_double * 25),
        ("var", c_double * 25),
        ("epsilon", c_double),
        ("clip_obs", c_double),
    ]


class PnpLibraryError(RuntimeError):
    pass


# every exported symbol with its signature; tests/test_capi_symbols.py checks this list against
# include/pnp_b200.h and against the built library
_P = c_void_p
SIGNATURES = {
    "pnp_abi_version": (c_int, []),
    "pnp_last_error": (c_char_p, []),
    "pnp_device_info": (c_int, [POINTER(c_int32), POINTER(c_int32), POINTER(c_int32)]),
    "pnp_set_tree": (c_int, [POINTER(PnpTreeStruct)]),
    "pnp_get_tree": (c_int, [POINTER(PnpTreeStruct)]),
    "pnp_tree_is_specialized": (c_int, []),
    "pnp_get_specialized_tree": (c_int, [POINTER(PnpTreeStruct)]),
    "pnp_fk_jac_f32": (c_int, [_P, c_int64, _P, _P, _P, c_int32, _P]),
    "pnp_fk_jac_f64": (c_int, [_P, c_int64, _P, _P, _P, c_int32, _P]),
    "pnp_ik_solve_f32": (c_int, [_P, _P, c_int32, c_int64, POINTER(PnpIkParams), _P, _P, _P, _P, _P, _P, _P]),
    "pnp_ik_solve_packed_f32": (c_int, [_P, _P, c_int32, c_int64, POINTER(PnpIkParams), _P, _P, _P, _P]),
    "pnp_ik_solve_compact_f32": (c_int, [_P, _P, c_int32, c_int64, POINTER(PnpIkParams), _P, _P, _P]),
    "pnp_ik_solve_f64": (c_int, [_P, _P, c_int32, c_int64, POINTER(PnpIkParams), _P, _P, _P, _P, _P, _P, _P]),
    "pnp_ik_multistart_scratch_bytes": (c_int, [c_int64, POINTER(c_int64)]),
    "pnp_ik_solve_multistart_f32": (c_int, [_P, _P, c_int32, c_int64, _P, c_int32, POINTER(PnpIkParams), _P, _P, _P, _P, _P,
                                            _P, _P, _P, _P, _P]),
    "pnp_ik_solve_multistart_packed_f32": (c_int, [_P, _P, c_int32, c_int64, _P, c_int32, POINTER(PnpIkParams), _P, _P, _P,
                                                   _P, _P, _P, _P]),
    "pnp_ik_solve_multistart_f64": (c_int, [_P, _P, c_int32, c_int64, _P, c_int32, POINTER(PnpIkParams), _P, _P, _P, _P, _P,
                                            _P, _P, _P, _P, _P]),
    "pnp_ik_waypoints_f32": (c_int, [_P, _P, c_int64, c_int32, c_double, POINTER(PnpIkParams), _P, _P, _P, _P, _P, _P]),
    "pnp_ik_pose_solve_f32": (c_int, [_P, _P, _P, c_int32, c_int64, POINTER(PnpIkParams), c_double, c_double,
                                      _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "pnp_ik_pose_solve_f64": (c_int, [_P, _P, _P, c_int32, c_int64, POINTER(PnpIkParams), c_double, c_double,
                                      _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "pnp_ik_pose_solve_multistart_f32": (c_int, [_P, _P, _P, c_int32, c_int64, _P, c_int32, POINTER(PnpIkParams),
                                                 c_double, c_double, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "pnp_ik_pose_solve_multistart_f64": (c_int, [_P, _P, _P, c_int32, c_int64, _P, c_int32, POINTER(PnpIkParams),
                                                 c_double, c_double, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "pnp_move_ik_plan_f32": (c_int, [_P, _P, c_int64, POINTER(PnpMoveParams), POINTER(PnpIkParams), _P, _P, _P, _P, _P, _P, _P]),
    "pnp_move_ik_plan_f64": (c_int, [_P, _P, c_int64, POINTER(PnpMoveParams), POINTER(PnpIkParams), _P, _P, _P, _P, _P, _P, _P]),
    "pnp_move_plan_order_f32": (c_int, [_P, _P, c_int64, _P, c_int32, _P]),
    "pnp_move_plan_order_f64": (c_int, [_P, _P, c_int64, _P, c_int32, _P]),
    "pnp_move_plan_order_check": (c_int, [_P, c_int64, _P, _P, _P]),
    "pnp_move_ik_plan_ordered_f32": (c_int, [_P, _P, _P, c_int64, POINTER(PnpMoveParams), POINTER(PnpIkParams), _P, _P, _P, _P, _P, _P, _P]),
    "pnp_move_ik_plan_sorted_f32": (c_int, [_P, _P, _P, c_int64, POINTER(PnpMoveParams), POINTER(PnpIkParams), _P, _P, _P, _P, _P, _P, _P]),
    "pnp_move_ik_plan_ordered_f64": (c_int, [_P, _P, _P, c_int64, POINTER(PnpMoveParams), POINTER(PnpIkParams), _P, _P, _P, _P, _P, _P, _P]),
    "pnp_move_ik_plan_pose_f32": (c_int, [_P, _P, _P, c_int64, POINTER(PnpMovePoseParams), POINTER(PnpIkParams), _P, _P, _P, _P,
                                          _P, _P, _P, _P, _P]),
    "pnp_move_ik_plan_pose_f64": (c_int, [_P, _P, _P, c_int64, POINTER(PnpMovePoseParams), POINTER(PnpIkParams), _P, _P, _P, _P,
                                          _P, _P, _P, _P, _P]),
    "pnp_reward_f32": (c_int, [_P, _P, _P, _P, _P, _P, c_int64, POINTER(PnpRewardParams), _P, _P, _P, _P]),
    "pnp_reward_f64": (c_int, [_P, _P, _P, _P, _P, _P, c_int64, POINTER(PnpRewardParams), _P, _P, _P, _P]),
    "pnp_get_obs_f32": (c_int, [_P, _P, _P, _P, _P, _P, _P, c_int32, c_int64, c_double, _P, c_int32, _P]),
    "pnp_get_obs_f64": (c_int, [_P, _P, _P, _P, _P, _P, _P, c_int32, c_int64, c_double, _P, c_int32, _P]),
    "pnp_her_relabel_f32": (c_int, [_P, _P, _P, _P, _P, c_int64, POINTER(PnpRewardParams), POINTER(PnpNormalizeParams),
                                    _P, _P, _P, _P, _P, _P]),
    "pnp_her_relabel_table_f32": (c_int, [_P, _P, _P, _P, _P, _P, c_int64, POINTER(PnpRewardParams),
                                          POINTER(PnpNormalizeParams), _P, _P, _P, _P, _P, _P]),
    "pnp_goal_distance_f64": (c_int, [_P, _P, c_int64, _P, _P]),
    "pnp_ik_solve_one_host_f32": (c_int, [c_void_p, _P, _P, POINTER(PnpIkParams), _P]),
    "pnp_host_ctx_create": (c_int, [POINTER(c_void_p), c_int64]),
    "pnp_host_ctx_destroy": (c_int, [c_void_p]),
    "pnp_ik_solve_host_f32": (c_int, [_P, _P, _P, c_int32, c_int64, POINTER(PnpIkParams), _P, _P, _P, _P, _P, _P]),
    "pnp_ik_solve_packed_host_f32": (c_int, [_P, _P, _P, c_int32, c_int64, POINTER(PnpIkParams), _P, _P, _P]),
    "pnp_ik_solve_compact_host_f32": (c_int, [_P, _P, _P, c_int32, c_int64, POINTER(PnpIkParams), _P, _P]),
    "pnp_reward_one_host_f64": (c_int, [_P, _P, _P, _P, _P, c_double, c_int32, POINTER(PnpRewardParams), _P, _P, _P]),
    "pnp_reward_host_f32": (c_int, [_P, _P, _P, _P, _P, _P, _P, c_int64, POINTER(PnpRewardParams), _P, _P, _P]),
    "pnp_reward_host_f64": (c_int, [_P, _P, _P, _P, _P, _P, _P, c_int64, POINTER(PnpRewardParams), _P, _P, _P]),
    "pnp_probe_fp32_peak": (c_int, [POINTER(c_double), POINTER(c_double)]),
    "pnp_launch_count": (c_uint64, []),
}

_lib = None


def load() -> ctypes.CDLL:
    """Load libpnp_b200.so (once).  Raises PnpLibraryError if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PnpLibraryError(
            f"{LIB_PATH} not found: build it with `python -m mujoco_panda_pnp_b200.csrc.build` "
            "(or __graft_entry__.build()).  There is no CPU fallback."
        )
    lib = ctypes.CDLL(LIB_PATH)
    for name, (restype, argtypes) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here means the .so is stale
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc == 0:
        return
    msg = load().pnp_last_error()
    msg = msg.decode("utf-8", "replace") if msg else ""
    name = _ERRNAMES.get(rc, f"cudaError {rc}" if rc > 0 else str(rc))
    if rc == -1:
        raise ValueError(f"{what}: {name}: {msg}")
    raise PnpLibraryError(f"{what}: {name}: {msg}")


def launch_count() -> int:
    return int(load().pnp_launch_count())

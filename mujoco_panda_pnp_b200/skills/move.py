"""MoveIKSkill - GPU drop-in for the reference's adaptive IK trajectory planner.

Mirrors /root/reference/panda_mujoco_gym/skills/move.py:61-208: same constructor, ``reset()``
fills ``pos_traj`` / ``quat_traj`` (the whole planning loop of move.py:76-191 runs in
``move_ik_plan_kernel``), ``step()`` replays the waypoints through the env exactly like the
reference (set_mocap_pose + 5 physics sub-steps; physics itself is the env's, out of scope here).

Additive API: ``plan_moves(model, q_start[N,7], targets[N,3])`` plans N moves in one launch;
``plan_pose_moves(model, q_start, target_pos, target_quat)`` plans N moves to a position AND an orientation
(``move_pose_plan_kernel``, every waypoint a solved pose), and ``MoveIKSkill(..., target_quat=q)`` uses it;
``plan_axis_moves(model, q_start, target_pos, target_axis)`` plans N moves to a position and a direction of the tool
axis, the roll about it free (``move_axis_plan_kernel``), and ``MoveIKSkill(..., target_axis=a)`` uses it.

Difference to the reference, on purpose: the planning loop is bounded (``max_outer`` rounds,
default 4*max_traj_points+64).  The reference loop never terminates for unreachable targets.
"""

from __future__ import annotations

from typing import Any, Optional

import numpy as np
import torch

from .. import engine
from ..tree import KinematicTree


def plan_moves(model: Any, q_start, targets, pos_thresh: float = 0.01, max_traj_points: int = 200,
               step_size: float = 0.01, max_outer: int = 0, traj_cap: Optional[int] = None,
               precision: str = "fp32", site_name: str = "ee_center_site", device=None, tree=None):
    """Plan N MoveIKSkill trajectories at once.  Returns the engine dict (device tensors):
    traj[N,traj_cap,3], traj_len[N], q_final[N,7], n_solves[N], status[N]."""
    if not torch.cuda.is_available():
        raise engine._lib.PnpLibraryError("no CUDA device: plan_moves has no CPU path")
    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    dt = torch.float32 if precision == "fp32" else torch.float64
    tree = tree or KinematicTree.from_mjmodel(model, site_name)
    to = lambda x: (x if isinstance(x, torch.Tensor) else torch.as_tensor(np.asarray(x))).to(device=dev, dtype=dt)  # noqa: E731
    with torch.cuda.device(dev):
        engine.set_tree(tree)
        return engine.move_ik_plan(to(q_start).reshape(-1, 7), to(targets).reshape(-1, 3), engine.ik_params(),
                                   pos_thresh=pos_thresh, max_traj_points=max_traj_points, step_size=step_size,
                                   max_outer=max_outer, traj_cap=traj_cap or max_traj_points + 56)


def plan_pose_moves(model: Any, q_start, target_pos, target_quat, pos_thresh: float = 0.01, rot_thresh: float = 0.05,
                    step_size: float = 0.01, rot_step: float = 0.05, ik_rot_thresh: float = 1e-2, rot_weight: float = 1.0,
                    max_traj_points: int = 200, traj_cap: Optional[int] = None, precision: str = "fp32",
                    site_name: str = "ee_center_site", device=None, tree=None):
    """Plan N moves to target_pos[N,3] and target_quat[N,4] (wxyz) at once (engine.move_ik_plan_pose).  Returns the
    engine dict (device tensors): pos_traj, quat_traj, q_traj, traj_len, q_final, n_solves, status."""
    if not torch.cuda.is_available():
        raise engine._lib.PnpLibraryError("no CUDA device: plan_pose_moves has no CPU path")
    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    dt = torch.float32 if precision == "fp32" else torch.float64
    tree = tree or KinematicTree.from_mjmodel(model, site_name)
    to = lambda x: (x if isinstance(x, torch.Tensor) else torch.as_tensor(np.asarray(x))).to(device=dev, dtype=dt)  # noqa: E731
    with torch.cuda.device(dev):
        engine.set_tree(tree)
        return engine.move_ik_plan_pose(to(q_start).reshape(-1, 7), to(target_pos).reshape(-1, 3),
                                        to(target_quat).reshape(-1, 4), engine.ik_params(), pos_thresh=pos_thresh,
                                        rot_thresh=rot_thresh, step_size=step_size, rot_step=rot_step,
                                        ik_rot_thresh=ik_rot_thresh, rot_weight=rot_weight,
                                        max_traj_points=max_traj_points, traj_cap=traj_cap)


def plan_axis_moves(model: Any, q_start, target_pos, target_axis, tool_axis=(0.0, 0.0, 1.0), pos_thresh: float = 0.01,
                    rot_thresh: float = 0.05, step_size: float = 0.01, rot_step: float = 0.05,
                    ik_rot_thresh: float = 1e-2, rot_weight: float = 1.0, max_traj_points: int = 200,
                    traj_cap: Optional[int] = None, precision: str = "fp32", site_name: str = "ee_center_site",
                    device=None, tree=None):
    """Plan N moves to target_pos[N,3] with the site-frame ``tool_axis`` along target_axis[N,3] (world frame), the
    roll about it free, at once (engine.move_ik_plan_axis).  Returns the engine dict (device tensors): pos_traj,
    axis_traj, quat_traj, q_traj, traj_len, q_final, n_solves, status."""
    if not torch.cuda.is_available():
        raise engine._lib.PnpLibraryError("no CUDA device: plan_axis_moves has no CPU path")
    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    dt = torch.float32 if precision == "fp32" else torch.float64
    tree = tree or KinematicTree.from_mjmodel(model, site_name)
    to = lambda x: (x if isinstance(x, torch.Tensor) else torch.as_tensor(np.asarray(x))).to(device=dev, dtype=dt)  # noqa: E731
    with torch.cuda.device(dev):
        engine.set_tree(tree)
        return engine.move_ik_plan_axis(to(q_start).reshape(-1, 7), to(target_pos).reshape(-1, 3),
                                        to(target_axis).reshape(-1, 3), engine.ik_params(), tool_axis=tool_axis,
                                        pos_thresh=pos_thresh, rot_thresh=rot_thresh, step_size=step_size,
                                        rot_step=rot_step, ik_rot_thresh=ik_rot_thresh, rot_weight=rot_weight,
                                        max_traj_points=max_traj_points, traj_cap=traj_cap)


class MoveIKSkill:
    """Adaptive IK trajectory planning (reference: skills/move.py:61-208).

    With ``target_quat`` (wxyz) the move also turns the gripper to that orientation: ``reset()`` plans with the pose
    planner (plan_pose_moves), every waypoint a solved pose, and keeps its joints in ``q_traj``.  With ``target_axis``
    (world frame) the move turns the site-frame ``tool_axis`` onto that direction and leaves the roll free: ``reset()``
    plans with the axis planner (plan_axis_moves) and fills ``q_traj`` the same way; ``rot_thresh`` and ``rot_step``
    then apply to the axis angle.  At most one of the two may be given.  Without either the move is the reference's
    position-only plan."""

    def __init__(self, env, target_pos: np.ndarray, pos_thresh: float = 0.01,
                 max_traj_points: int = 200, step_size: float = 0.01, *, precision: str = "fp32",
                 target_quat: Optional[np.ndarray] = None, rot_thresh: float = 0.05, rot_step: float = 0.05,
                 target_axis: Optional[np.ndarray] = None, tool_axis=(0.0, 0.0, 1.0)):
        if target_quat is not None and target_axis is not None:
            raise ValueError("give target_quat or target_axis, not both")
        self.env = env
        self.target_pos = np.asarray(target_pos, float)
        self.target_quat = None if target_quat is None else np.asarray(target_quat, float)
        self.target_axis = None if target_axis is None else np.asarray(target_axis, float)
        self.tool_axis = tool_axis
        self.rot_thresh = rot_thresh
        self.rot_step = rot_step
        self.q_traj: list = []
        self.pos_thresh = pos_thresh
        self.max_traj_points = max_traj_points
        self.step_size = step_size
        self.precision = precision
        self.i = 0
        self.done = False
        self.pos_traj: list = []
        self.quat_traj: list = []
        self.status = 0

    def reset(self):
        self.i = 0
        self.done = False
        model = self.env.unwrapped.model  # move.py:81-82
        data = self.env.unwrapped.data
        start_quat = np.asarray(self.env.get_ee_orientation(), dtype=np.float64).copy()  # :92
        q_current = np.asarray(data.qpos[:7], dtype=np.float64).copy()  # :93
        if self.target_quat is not None or self.target_axis is not None:
            if self.target_quat is not None:
                out = plan_pose_moves(model, q_current[None], self.target_pos[None], self.target_quat[None],
                                      self.pos_thresh, self.rot_thresh, self.step_size, self.rot_step,
                                      max_traj_points=self.max_traj_points, precision=self.precision)
            else:
                out = plan_axis_moves(model, q_current[None], self.target_pos[None], self.target_axis[None],
                                      self.tool_axis, self.pos_thresh, self.rot_thresh, self.step_size, self.rot_step,
                                      max_traj_points=self.max_traj_points, precision=self.precision)
            n = min(int(out["traj_len"][0]), out["pos_traj"].shape[1])
            self.status = int(out["status"][0])
            self.pos_traj = list(out["pos_traj"][0, :n].double().cpu().numpy())
            self.quat_traj = list(out["quat_traj"][0, :n].double().cpu().numpy())
            self.q_traj = list(out["q_traj"][0, :n].double().cpu().numpy())
            return
        out = plan_moves(model, q_current[None], self.target_pos[None], self.pos_thresh, self.max_traj_points,
                         self.step_size, precision=self.precision)
        n = int(out["traj_len"][0])
        cap = out["traj"].shape[1]
        traj = out["traj"][0, : min(n, cap)].double().cpu().numpy()
        self.status = int(out["status"][0])
        self.pos_traj = [p.copy() for p in traj]
        self.quat_traj = [start_quat.copy() for _ in traj]  # orientation kept constant (:134)

    def step(self):
        if self.done:
            return self.zero_action()
        if self.i < len(self.pos_traj):  # move.py:199-204
            self.env.set_mocap_pose(self.pos_traj[self.i], self.quat_traj[self.i])
            self._step_sim(n=5)
            self.i += 1
        else:
            self.done = True
        return self.zero_action()

    def is_done(self) -> bool:
        return self.done

    def zero_action(self) -> np.ndarray:  # base.py:35-36
        return np.zeros_like(self.env.action_space.low, dtype=np.float32)

    def _step_sim(self, n: int = 1):  # base.py:39-46 (physics belongs to the env)
        mj = self.env.unwrapped
        for _ in range(n):
            mj._mujoco.mj_step(mj.model, mj.data, nstep=1)
        if hasattr(self.env, "render") and getattr(self.env, "render_mode", None) is not None:
            self.env.render()

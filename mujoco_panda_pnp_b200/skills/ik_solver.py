"""JacobianIKController - GPU drop-in for the reference's IK solver.

Mirrors /root/reference/panda_mujoco_gym/skills/ik_solver.py: same class name, constructor,
``solve`` signature, ``IKResult`` fields and attribute names (model, data, site_id,
joint_ids, lower, upper), so ``MoveIKSkill.reset`` (skills/move.py:85,128,152,168) and
test/ik_test.py:31-38 run unchanged.  The arithmetic of ``solve`` (ik_solver.py:50-101) is the
``ik_solve_kernel`` of libpnp_b200.so; there is no CPU implementation in this package.

Additive API: ``solve_batch`` (N queries in one launch) and ``fk`` (mj_kinematics/mj_jacSite
for the EE site).
"""

from __future__ import annotations

from dataclasses import dataclass
from typing import Any, Optional

import numpy as np
import torch

from .. import engine
from ..engine import BatchIKResult
from ..tree import KinematicTree


@dataclass
class IKResult:
    """Result of IK solving with detailed information (ik_solver.py:16-24)."""

    success: bool  # Whether IK converged successfully
    q: np.ndarray  # Final joint angles (7,)
    final_pos: np.ndarray  # Final end-effector position (3,)
    pos_error: float  # Final position error (distance)
    iterations: int  # Number of iterations used
    converged: bool  # Whether converged within threshold


def _to_tensor(x) -> torch.Tensor:
    return x if isinstance(x, torch.Tensor) else torch.as_tensor(np.asarray(x))


class JacobianIKController:
    def __init__(self, model: Any, data: Any, site_name: str = "ee_center_site", *,
                 device: Optional[Any] = None, precision: str = "fp32", kinematics: str = "auto"):
        """``model`` / ``data``: a live ``mujoco.MjModel`` / ``MjData`` or this package's
        ``KinematicModel`` / ``KinematicData`` (same field names).  Keyword-only extras select
        the CUDA device, the compute precision ("fp32" product path, "fp64" parity path) and
        the kinematics code path ("auto" | "generic" | "specialized")."""
        if precision not in ("fp32", "fp64"):
            raise ValueError("precision must be 'fp32' or 'fp64'")
        self.model = model
        self.data = data
        self.site_id = model.site(site_name).id  # ik_solver.py:30
        self.joint_ids = np.arange(7)  # :31
        self.lower = np.asarray(model.jnt_range[:7, 0], dtype=np.float64).copy()  # :32
        self.upper = np.asarray(model.jnt_range[:7, 1], dtype=np.float64).copy()  # :33
        self.site_name = site_name
        self.precision = precision
        self.kinematics = kinematics
        if not torch.cuda.is_available():
            raise engine._lib.PnpLibraryError("no CUDA device: JacobianIKController has no CPU path")
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        self.tree = KinematicTree.from_mjmodel(model, site_name)
        with torch.cuda.device(self.device):
            self.specialized = engine.set_tree(self.tree)
        # single-query fast path: preallocated staging arrays and cached parameter structs
        self._param_cache = {}
        self._one_in_t = np.empty(3, np.float32)
        self._one_in_q = np.empty(7, np.float32)
        self._one_out = np.empty(12, np.float32)
        self._one_word = self._one_out[11:12].view(np.int32)

    # ------------------------------------------------------------------------------------
    def _dtype(self):
        return torch.float32 if self.precision == "fp32" else torch.float64

    def _params(self, max_iters, pos_thresh, damping, step_limit):
        return engine.ik_params(max_iters, pos_thresh, damping, step_limit, self.kinematics)

    def solve(self, target_pos: np.ndarray, q_init: np.ndarray,
              max_iters: int = 100, pos_thresh: float = 1e-3,
              damping: float = 1e-2, step_limit: float = 0.1, seeds=None) -> IKResult:
        """Same contract as the reference (ik_solver.py:35-101).  Side effect kept: on return
        ``data.qpos[:7] == result.q`` and ``data.site_xpos[site_id] == result.final_pos``.

        ``seeds`` (K, 7), an extension: when the solve from ``q_init`` fails, retry from each seed in turn and return
        the first success (see solve_batch); the call then goes through the batch path."""
        target_pos = np.asarray(target_pos, dtype=np.float64)
        q_init = np.asarray(q_init, dtype=np.float64)
        if target_pos.shape != (3,) or q_init.shape != (7,):
            raise ValueError("solve expects target_pos (3,) and q_init (7,)")
        if self.precision == "fp32" and seeds is None:
            # one C call, no memcpy: the kernel reads the query from and writes the result to a mapped
            # pinned mailbox (pnp_ik_solve_one_host_f32)
            key = (max_iters, pos_thresh, damping, step_limit)
            params = self._param_cache.get(key)
            if params is None:
                params = self._param_cache[key] = self._params(max_iters, pos_thresh, damping, step_limit)
            t32, q32, o = self._one_in_t, self._one_in_q, self._one_out
            t32[:] = target_pos
            q32[:] = q_init
            if torch.cuda.current_device() == self.device.index:
                engine.set_tree(self.tree)
                engine.ik_solve_one_host(t32, q32, params, o)
            else:
                with torch.cuda.device(self.device):
                    engine.set_tree(self.tree)
                    engine.ik_solve_one_host(t32, q32, params, o)
            word = int(self._one_word[0])
            q = o[0:7].astype(np.float64)
            final_pos = o[8:11].astype(np.float64)
            self._write_back(q, final_pos)
            return IKResult(success=bool(word & (2 << 24)), q=q, final_pos=final_pos, pos_error=float(o[7]),
                            iterations=word & 0xFFFFFF, converged=bool(word & (1 << 24)))
        r = self.solve_batch(target_pos[None], q_init[None], max_iters, pos_thresh, damping, step_limit, seeds=seeds)
        q = r.q[0].double().cpu().numpy()
        final_pos = r.final_pos[0].double().cpu().numpy()
        self._write_back(q, final_pos)
        return IKResult(
            success=bool(r.success[0]), q=q, final_pos=final_pos, pos_error=float(r.pos_error[0]),
            iterations=int(r.iterations[0]), converged=bool(r.converged[0]),
        )

    def solve_batch(self, targets, q_init, max_iters: int = 100, pos_thresh: float = 1e-3,
                    damping: float = 1e-2, step_limit: float = 0.1, counters=None, seeds=None) -> BatchIKResult:
        """N independent solves in one launch.  targets (N,3); q_init (N,7) or (7,) broadcast.
        NumPy / CPU inputs are copied to ``self.device``; CUDA tensors are used in place.
        Returns device tensors (BatchIKResult).

        ``seeds`` (K, 7), K <= 255 (e.g. ``engine.ik_restart_seeds(8)``): every query the solve from ``q_init`` does not
        solve is solved again from seeds[0], seeds[1], ... until one succeeds (engine.ik_solve_multistart); the result
        then carries ``attempt`` (0 = from q_init, k = from seeds[k - 1])."""
        dt = self._dtype()
        with torch.cuda.device(self.device):
            engine.set_tree(self.tree)
            t, qi = _to_tensor(targets), _to_tensor(q_init)
            if t.dim() != 2 or t.shape[1] != 3:
                raise ValueError(f"targets must have shape (N, 3), got {tuple(t.shape)}")
            t = t.to(device=self.device, dtype=dt)
            qi = qi.to(device=self.device, dtype=dt)
            params = self._params(max_iters, pos_thresh, damping, step_limit)
            if seeds is not None:
                sd = _to_tensor(seeds).to(device=self.device, dtype=dt)
                return engine.ik_solve_multistart(t, qi, sd, params, counters=counters)
            return engine.ik_solve(t, qi, params, counters=counters)

    def fk(self, q):
        """EE-site position, wxyz quaternion and 6x7 Jacobian [jacp; jacr] at q (N,7)."""
        with torch.cuda.device(self.device):
            engine.set_tree(self.tree)
            qt = _to_tensor(q).to(device=self.device, dtype=self._dtype()).reshape(-1, 7)
            return engine.fk_jac(qt, kinematics=self.kinematics)

    def solve_pose(self, target_pos, target_quat, q_init, max_iters: int = 100, pos_thresh: float = 1e-3,
                   rot_thresh: float = 1e-2, damping: float = 1e-2, step_limit: float = 0.1,
                   rot_weight: float = 1.0, seeds=None) -> dict:
        """Pose-mode IK (EXTENSION, no reference counterpart: see pnp_ik_pose_solve_* in
        include/pnp_b200.h).  target_pos (3,)|(N,3), target_quat wxyz (4,)|(N,4), q_init (7,)|(N,7).
        Returns a dict of device tensors (batched) with q, final_pos, final_quat, pos_error,
        rot_error, iterations, converged, success.

        ``seeds`` (K, 7), K <= 255 (e.g. ``engine.ik_restart_seeds(8)``): every query the solve from ``q_init`` does not
        solve is solved again from seeds[0], seeds[1], ... until one succeeds (engine.ik_pose_solve_multistart); the
        dict then also holds ``attempt`` (0 = from q_init, k = from seeds[k - 1])."""
        dt = self._dtype()
        with torch.cuda.device(self.device):
            engine.set_tree(self.tree)
            tp = _to_tensor(target_pos).to(device=self.device, dtype=dt).reshape(-1, 3)
            tq = _to_tensor(target_quat).to(device=self.device, dtype=dt).reshape(-1, 4)
            qi = _to_tensor(q_init).to(device=self.device, dtype=dt)
            params = self._params(max_iters, pos_thresh, damping, step_limit)
            if seeds is not None:
                sd = _to_tensor(seeds).to(device=self.device, dtype=dt)
                return engine.ik_pose_solve_multistart(tp, tq, qi, sd, params, rot_thresh=rot_thresh,
                                                       rot_weight=rot_weight)
            return engine.ik_pose_solve(tp, tq, qi, params, rot_thresh=rot_thresh, rot_weight=rot_weight)

    def solve_axis(self, target_pos, target_axis, q_init, max_iters: int = 100, pos_thresh: float = 1e-3,
                   damping: float = 1e-2, step_limit: float = 0.1, tool_axis=(0.0, 0.0, 1.0), rot_thresh: float = 1e-2,
                   rot_weight: float = 1.0, seeds=None, cone_angle=None) -> dict:
        """Axis-constrained IK (EXTENSION: see pnp_ik_axis_solve_* in include/pnp_b200.h): the site at target_pos
        with its ``tool_axis`` (site frame; the default +z is the packaged Panda's approach direction) along
        target_axis (world frame), the roll about that axis free - e.g. a top-down grasp is target_axis (0, 0, -1).
        target_pos (3,)|(N,3), target_axis (3,)|(N,3), q_init (7,)|(N,7).  Returns a dict of device tensors (batched)
        with q, final_pos, final_axis, final_quat, pos_error, axis_error (rad), iterations, converged, success.

        ``seeds`` (K, 7), K <= 255: as solve_pose (engine.ik_axis_solve_multistart); the dict then also holds
        ``attempt``.  ``cone_angle`` (rad, in [0, pi]): accept the tool axis anywhere within that angle of target_axis
        (pnp_ik_axis_cone_solve_*), e.g. a top-down grasp that tolerates 15 degrees of tilt; None asks for the exact
        axis."""
        dt = self._dtype()
        with torch.cuda.device(self.device):
            engine.set_tree(self.tree)
            tp = _to_tensor(target_pos).to(device=self.device, dtype=dt).reshape(-1, 3)
            ta = _to_tensor(target_axis).to(device=self.device, dtype=dt).reshape(-1, 3)
            qi = _to_tensor(q_init).to(device=self.device, dtype=dt)
            params = self._params(max_iters, pos_thresh, damping, step_limit)
            kw = dict(tool_axis=tool_axis, rot_thresh=rot_thresh, rot_weight=rot_weight, cone_angle=cone_angle)
            if seeds is not None:
                sd = _to_tensor(seeds).to(device=self.device, dtype=dt)
                return engine.ik_axis_solve_multistart(tp, ta, qi, sd, params, **kw)
            return engine.ik_axis_solve(tp, ta, qi, params, **kw)

    def _write_back(self, q: np.ndarray, final_pos: np.ndarray) -> None:
        d = self.data
        if d is None:
            return
        d.qpos[:7] = q  # ik_solver.py:82
        mj = _mujoco_module()
        if mj is not None and isinstance(d, mj.MjData):  # real MjData: keep the simulator consistent (ik_solver.py:83)
            mj.mj_forward(self.model, d)
            return
        if hasattr(d, "site_xpos"):
            d.site_xpos[self.site_id] = final_pos


_MUJOCO = [False, None]  # [looked up?, module or None]: a failing import on every solve() cost ~25 us


def _mujoco_module():
    if not _MUJOCO[0]:
        try:
            import mujoco

            _MUJOCO[1] = mujoco
        except ImportError:
            _MUJOCO[1] = None
        _MUJOCO[0] = True
    return _MUJOCO[1]


IKSolver = JacobianIKController  # north_star calls the class IKSolver (SURVEY.md D1)


def solve_ik(model, data, site_name, target_pos, target_quat, q_init, seeds=None):
    """The function FrankaEnv.solve_ik tries to import (envs/panda_env.py:399-409) and the reference
    never defined.  Pose-mode DLS IK on the GPU; returns an IKResult for the single query.

    ``seeds`` (K, 7), an extension: when the solve from ``q_init`` fails, retry from each seed in turn and return the
    first success (JacobianIKController.solve_pose)."""
    ctl = JacobianIKController(model, data, site_name)
    r = ctl.solve_pose(np.asarray(target_pos, float), np.asarray(target_quat, float), np.asarray(q_init, float),
                       seeds=seeds)
    q = r["q"][0].double().cpu().numpy()
    final_pos = r["final_pos"][0].double().cpu().numpy()
    ctl._write_back(q, final_pos)
    return IKResult(success=bool(r["success"][0]), q=q, final_pos=final_pos, pos_error=float(r["pos_error"][0]),
                    iterations=int(r["iterations"][0]), converged=bool(r["converged"][0]))

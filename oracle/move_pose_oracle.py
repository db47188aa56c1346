"""ORACLE (test infrastructure) for the pose-mode move planner EXTENSION (pnp_move_ik_plan_pose_*).

The reference has no pose planner: MoveIKSkill.reset (the reference's skills/move.py:76-191) plans the
end-effector position only and keeps the start orientation, and RotateSkill turns the gripper by a mocap SLERP that
never checks reachability.  This module states the semantics the GPU kernel implements, in scalar FP64 over the restated
engine (mj_oracle.py) and the pose solve of pose_ik_oracle.solve_pose.  PARITY UNPINNED (no reference behaviour exists).

It keeps the reference planner's skeleton (warm start from the current q, an adaptive step, a smaller step after a
rejected solve, a 10x smaller fallback) and drops its bookkeeping quirks (the double failure increment, the y-frozen
strategy 2, fallback successes that do not advance the point count), so that every plan terminates.  Per env:

    (p, r) = FK(q_start) (site position, mju_mat2Quat of the site frame); point 0 = (p, r, q_start)
    goal_quat normalised; a non-finite goal component or a zero goal quaternion: BROKE, one point
    round:  d = goal_pos - p, dist = |d|;  w = quat2vel(goal_quat (x) conj(r)), theta = |w|
            dist <= pos_thresh and theta <= rot_thresh: done (status 0)
            points >= max_traj_points: CAPPED
            f = min(1, step_size / dist, rot_step / theta)  (a zero dist or theta drops its term)
            attempts g = f, f / 2, f / 20:  aim = (p + g d, quat(g w) (x) r), or exactly the goal when g == 1
                solve_pose(aim, from q, ik params); a success appends (final_pos, final_quat, q), moves (p, r, q)
                there, counts a point and ends the round
            three rejections: BROKE
    the unreached goal is never appended: every point is a solved pose with its joints.
"""

from __future__ import annotations

import math

import numpy as np

from . import mj_oracle, pose_ik_oracle

BROKE, CAPPED, OVERFLOW = 1, 2, 4
ATTEMPTS = (1.0, 0.5, 0.05)  # fractions of f tried in one round: full step, halved, a tenth of the halved one


def quat_of_rotvec(v):
    """Unit quaternion of the rotation vector v (wxyz); identity for v = 0."""
    th = math.sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2])
    if th == 0.0:
        return np.array([1.0, 0.0, 0.0, 0.0])
    s, c = math.sin(0.5 * th), math.cos(0.5 * th)
    return np.array([c, s * v[0] / th, s * v[1] / th, s * v[2] / th])


def _fk(model, data, sid, q):
    data.qpos[:7] = q
    mj_oracle.mj_forward(model, data)
    r = np.empty(4)
    mj_oracle.mju_mat2Quat(r, data.site_xmat[sid])
    return data.site_xpos[sid].copy(), r


def remaining(p, r, goal_pos, goal_quat):
    """(d, dist, w, theta): the motion left from the pose (p, r) to the goal."""
    d = goal_pos - p
    w = pose_ik_oracle.quat2vel(mj_oracle.mju_mulQuat(goal_quat, np.array([r[0], -r[1], -r[2], -r[3]])))
    return d, float(np.linalg.norm(d)), w, float(np.linalg.norm(w))


def plan_pose(model, q_start, goal_pos, goal_quat, pos_thresh=0.01, rot_thresh=0.05, step_size=0.01, rot_step=0.05,
              ik_rot_thresh=1e-2, rot_weight=1.0, max_traj_points=200, max_iters=100, ik_pos_thresh=1e-3,
              damping=1e-2, step_limit=0.1, site_name="ee_center_site"):
    """One plan.  Returns dict(pos_traj [L,3], quat_traj [L,4], q_traj [L,7], q_final [7], n_solves, status)."""
    sid = model.site(site_name).id
    data = mj_oracle.MjData(model)
    gp = np.asarray(goal_pos, dtype=np.float64)
    gq = np.asarray(goal_quat, dtype=np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        gq = gq / np.linalg.norm(gq)
    q = np.array(q_start, dtype=np.float64)
    p, r = _fk(model, data, sid, q)
    pos_traj, quat_traj, q_traj = [p.copy()], [r.copy()], [q.copy()]
    n_solves = status = points = 0
    if not (np.isfinite(gp).all() and np.isfinite(gq).all()):
        status = BROKE
    while status == 0:
        d, dist, w, th = remaining(p, r, gp, gq)
        if dist <= pos_thresh and th <= rot_thresh:
            break
        if points >= max_traj_points:
            status = CAPPED
            break
        f = 1.0
        if dist > 0.0:
            f = min(f, step_size / dist)
        if th > 0.0:
            f = min(f, rot_step / th)
        for scale in ATTEMPTS:
            g = f * scale
            if g == 1.0:
                aim_p, aim_q = gp, gq
            else:
                aim_p, aim_q = p + g * d, mj_oracle.mju_mulQuat(quat_of_rotvec(g * w), r)
            res = pose_ik_oracle.solve_pose(model, data, aim_p, aim_q, q, max_iters=max_iters, pos_thresh=ik_pos_thresh,
                                            rot_thresh=ik_rot_thresh, damping=damping, step_limit=step_limit,
                                            rot_weight=rot_weight, site_name=site_name)
            n_solves += 1
            if res["success"]:
                p, r, q = res["final_pos"].copy(), res["final_quat"].copy(), res["q"].copy()
                pos_traj.append(p.copy())
                quat_traj.append(r.copy())
                q_traj.append(q.copy())
                points += 1
                break
        else:
            status = BROKE
    return dict(pos_traj=np.array(pos_traj), quat_traj=np.array(quat_traj), q_traj=np.array(q_traj), q_final=q,
                n_solves=n_solves, status=status)


def quat_angle(a, b):
    """Rotation angle (rad) between unit quaternions a and b, rows or single."""
    dot = np.abs(np.sum(np.asarray(a) * np.asarray(b), axis=-1))
    return 2.0 * np.arccos(np.clip(dot, 0.0, 1.0))

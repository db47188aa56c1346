"""ORACLE (test infrastructure) for the axis-mode move planner EXTENSION (pnp_move_ik_plan_axis_*).

A pick-and-place move often fixes where the gripper goes and which way its approach axis points, but not the roll about
that axis: a top-down descent keeps the gripper vertical, a reach into the shelf turns it horizontal.  This module
states what the GPU kernel plans for such a move, in scalar FP64 over the restated engine (mj_oracle.py) and the axis
solve of axis_ik_oracle.solve_axis.  It is the pose planner (move_pose_oracle.plan_pose) with the rotation replaced by
the tilt of one site-frame tool axis t.  PARITY UNPINNED (no reference behaviour exists).  Per env:

    (t, u1, u2) = axis_ik_oracle.tool_basis(tool_axis)  (one per call; ValueError for a zero or non-finite tool_axis)
    (p, R) = FK(q_start), a = R t, r = mat2quat(R); point 0 = (p, a, r, q_start)
    goal_axis normalised; a non-finite goal component or a zero goal axis: BROKE, one point
    round:  d = goal_pos - p, dist = |d|;  c = a x g, s = |c|, theta = atan2(s, a.g)   (as the axis solver evaluates it)
            dist <= pos_thresh and theta <= rot_thresh: done (status 0)
            points >= max_traj_points: CAPPED
            f = min(1, step_size / dist, rot_step / theta)  (a zero dist or theta drops its term)
            m = (g - (a.g) a) / s if s > 0;  -b2 (b2 = R u2) if s == 0 and a.g < 0  (the solver's n = b1: b1 x a = -b2)
            attempts h = f, f / 2, f / 20:  aim = (p + h d, normalize(cos(h theta) a + sin(h theta) m)), or exactly
                the goal when h == 1
                solve_axis(aim, from q, ik params, ik_rot_thresh, rot_weight, tool_axis); a success appends
                (final_pos, final_axis, quat of the final frame, q), moves there, counts a point and ends the round
            three rejections: BROKE
    the unreached goal is never appended: every point is a solved axis task with its joints.

theta is written exactly as the solver writes it (same association order, sqrt and atan2), so a solve aimed at the goal
that converges ends the plan by construction (pos_thresh >= the IK's pos_thresh, rot_thresh >= ik_rot_thresh).
"""

from __future__ import annotations

import math

import numpy as np

from . import axis_ik_oracle, mj_oracle

BROKE, CAPPED, OVERFLOW = 1, 2, 4
ATTEMPTS = (1.0, 0.5, 0.05)  # fractions of f tried in one round: full step, halved, a tenth of the halved one


def _normalize(v):
    """v / |v| with |v| summed left to right, as the kernels normalise a loaded axis (axis_load_target)."""
    n = math.sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2])
    return np.array([v[0] / n, v[1] / n, v[2] / n])


def _frame(model, data, sid, q):
    """(p, R, r) of the site at q: position, frame and quaternion."""
    data.qpos[:7] = q
    mj_oracle.mj_forward(model, data)
    r = np.empty(4)
    mj_oracle.mju_mat2Quat(r, data.site_xmat[sid])
    return data.site_xpos[sid].copy(), np.asarray(data.site_xmat[sid], dtype=np.float64).reshape(3, 3).copy(), r


def tilt(a, g):
    """(s, ad, theta) of the world tool axis a against the unit goal axis g, in the axis solver's operation order."""
    c = (a[1] * g[2] - a[2] * g[1], a[2] * g[0] - a[0] * g[2], a[0] * g[1] - a[1] * g[0])
    s = math.sqrt((c[0] * c[0] + c[1] * c[1]) + c[2] * c[2])
    ad = (a[0] * g[0] + a[1] * g[1]) + a[2] * g[2]
    return s, ad, math.atan2(s, ad)


def aim_axis(a, b2, g, h, theta):
    """The aim axis of the fraction h of the remaining tilt: a turned by h theta toward g."""
    s, ad, _ = tilt(a, g)
    if s > 0.0:
        m = (g - ad * a) / s
    elif ad < 0.0:
        m = -b2
    else:
        m = np.zeros(3)
    return _normalize(math.cos(h * theta) * a + math.sin(h * theta) * m)


def plan_axis(model, q_start, goal_pos, goal_axis, tool_axis=(0.0, 0.0, 1.0), pos_thresh=0.01, rot_thresh=0.05,
              step_size=0.01, rot_step=0.05, ik_rot_thresh=1e-2, rot_weight=1.0, max_traj_points=200, max_iters=100,
              ik_pos_thresh=1e-3, damping=1e-2, step_limit=0.1, site_name="ee_center_site", trace=None):
    """One plan.  Returns dict(pos_traj [L,3], axis_traj [L,3], quat_traj [L,4], q_traj [L,7], q_final [7], n_solves,
    status).  ``trace``, a list, receives (R, goal axis, h, theta, aim axis) of every attempt that is not the goal
    itself, R the site frame of the last point (tests of the aim rule)."""
    t, _, u2 = axis_ik_oracle.tool_basis(tool_axis)
    sid = model.site(site_name).id
    data = mj_oracle.MjData(model)
    gp = np.asarray(goal_pos, dtype=np.float64).reshape(3)
    with np.errstate(divide="ignore", invalid="ignore"):
        g = _normalize(np.asarray(goal_axis, dtype=np.float64).reshape(3))
    q = np.array(q_start, dtype=np.float64)
    p, R, r = _frame(model, data, sid, q)
    a, b2 = R @ t, R @ u2
    pos_traj, axis_traj, quat_traj, q_traj = [p.copy()], [a.copy()], [r.copy()], [q.copy()]
    n_solves = status = points = 0
    if not (np.isfinite(gp).all() and np.isfinite(g).all()):
        status = BROKE
    while status == 0:
        d = gp - p
        dist = math.sqrt((d[0] * d[0] + d[1] * d[1]) + d[2] * d[2])
        _, _, th = tilt(a, g)
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
            h = f * scale
            if h == 1.0:
                aim_p, aim_a = gp, g
            else:
                aim_p, aim_a = p + h * d, aim_axis(a, b2, g, h, th)
                if trace is not None:
                    trace.append((R.copy(), g.copy(), h, th, aim_a.copy()))
            res = axis_ik_oracle.solve_axis(model, data, aim_p, aim_a, q, tool_axis=tool_axis, max_iters=max_iters,
                                            pos_thresh=ik_pos_thresh, rot_thresh=ik_rot_thresh, damping=damping,
                                            step_limit=step_limit, rot_weight=rot_weight, site_name=site_name)
            n_solves += 1
            if res["success"]:
                q = res["q"].copy()
                p, R, r = _frame(model, data, sid, q)
                a, b2 = R @ t, R @ u2
                pos_traj.append(p.copy())
                axis_traj.append(a.copy())
                quat_traj.append(r.copy())
                q_traj.append(q.copy())
                points += 1
                break
        else:
            status = BROKE
    return dict(pos_traj=np.array(pos_traj), axis_traj=np.array(axis_traj), quat_traj=np.array(quat_traj),
                q_traj=np.array(q_traj), q_final=q, n_solves=n_solves, status=status)


def axis_angle(a, b):
    """Angle (rad) between unit vectors a and b, rows or single."""
    dot = np.sum(np.asarray(a) * np.asarray(b), axis=-1)
    return np.arccos(np.clip(dot, -1.0, 1.0))

"""ORACLE (test infrastructure) for the cone-tolerant axis IK EXTENSION.

A pick that accepts the gripper's approach axis anywhere within an angle alpha of a direction: the axis solve of
oracle/axis_ik_oracle.py with one per-call scalar, cone_angle alpha in [0, pi].  This module states what
pnp_ik_axis_cone_solve_* computes, in FP64 NumPy.  PARITY UNPINNED (no reference behaviour exists).

    a, b1, b2, theta, n as in the axis solve
    on = theta > alpha                                          (false for a NaN theta)
    w' = rot_weight if on else 0;  g = theta - alpha if on else 0
    e = [tp - p ; w' g n.b1 ; w' g n.b2],  J = [jacp ; w' b1^T jacr ; w' b2^T jacr]
    dq = J^T solve(J J^T + damping I5, e);  q = clip(q + clip(dq, +-step_limit), lower, upper)
    converged when |tp - p| < pos_thresh and theta - alpha < rot_thresh, tested before the update
    success = converged and |tp - p| < 2 pos_thresh and theta - alpha < 2 rot_thresh

Inside the cone the tilt rows are dropped, not zeroed in the error alone: the 5x5 system is then the position solver's
3x3 plus damping I2, and the step is the damped position step, so the axis is free to move anywhere in the cone.  With
the rows kept and only the error clamped (a deadzone), an axis that enters the cone is frozen where it entered, and
success falls as alpha grows (DESIGN.md 4.9).  alpha = 0 is the axis solve; alpha = pi is the position solve.
axis_error stays theta, the true angle to the target axis.
"""

from __future__ import annotations

import math

import numpy as np

from . import mj_oracle as mujoco
from .axis_ik_oracle import _axis_error, _normalized_axes, tool_basis


def _tilt(theta, alpha, rot_weight):
    """(w', g) of the statement, per row or for a scalar theta."""
    on = np.asarray(theta > alpha)
    return np.where(on, rot_weight, 0.0), np.where(on, theta - alpha, 0.0)


def solve_cone(model, data, target_pos, target_axis, q_init, cone_angle, tool_axis=(0.0, 0.0, 1.0), max_iters=100,
               pos_thresh=1e-3, rot_thresh=1e-2, damping=1e-2, step_limit=0.1, rot_weight=1.0,
               site_name="ee_center_site"):
    """One query on the restated engine (mj_forward / mj_jacSite)."""
    sid = model.site(site_name).id
    lower, upper = model.jnt_range[:7, 0], model.jnt_range[:7, 1]
    t, u1, u2 = tool_basis(tool_axis)
    d = np.asarray(target_axis, dtype=np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        d = d / np.linalg.norm(d)
    tp = np.asarray(target_pos, dtype=np.float64)
    q = np.array(q_init, dtype=np.float64)
    converged, iterations = False, 0
    pe = th = 0.0
    for i in range(max_iters + 1):
        data.qpos[:7] = q
        mujoco.mj_forward(model, data)
        p = data.site_xpos[sid].copy()
        R = np.asarray(data.site_xmat[sid], dtype=np.float64).reshape(3, 3)
        a, b1, b2 = R @ t, R @ u1, R @ u2
        c = np.cross(a, d)
        s = math.sqrt(float(c @ c))
        ad = float(a @ d)
        th = math.atan2(s, ad)
        if s > 0:
            nv = c / s
        elif s == 0 and ad < 0:
            nv = b1
        else:
            nv = np.zeros(3)
        e_pos = tp - p
        pe = float(np.linalg.norm(e_pos))
        if i == max_iters:
            iterations = max_iters
            break
        if pe < pos_thresh and th - cone_angle < rot_thresh:
            converged, iterations = True, i + 1
            break
        w, g = (rot_weight, th - cone_angle) if th > cone_angle else (0.0, 0.0)
        jp, jr = np.zeros((3, model.nv)), np.zeros((3, model.nv))
        mujoco.mj_jacSite(model, data, jp, jr, sid)
        J = np.vstack([jp[:, :7], w * (b1 @ jr[:, :7]), w * (b2 @ jr[:, :7])])
        e = np.concatenate([e_pos, [w * g * float(nv @ b1), w * g * float(nv @ b2)]])
        dq = J.T @ np.linalg.solve(J @ J.T + damping * np.eye(5), e)
        q = np.clip(q + np.clip(dq, -step_limit, step_limit), lower, upper)
    success = converged and pe < 2 * pos_thresh and th - cone_angle < 2 * rot_thresh
    return dict(success=success, converged=converged, q=q, final_pos=p, final_axis=a, axis_error=th,
                pos_error=pe, iterations=iterations)


# ---------------------------------------------------------------------------------------------------------------------
# The same statement over N queries at once, on the C restatement's FK (c_oracle.fk_jac).
# ---------------------------------------------------------------------------------------------------------------------
def solve_cone_batch(chain, target_pos, target_axis, q_init, cone_angle, tool_axis=(0.0, 0.0, 1.0), max_iters=100,
                     pos_thresh=1e-3, rot_thresh=1e-2, damping=1e-2, step_limit=0.1, rot_weight=1.0, nthreads=8,
                     trace=None):
    """solve_cone over N queries: target_pos[N,3], target_axis[N,3] (any norm), q_init[7] or [N,7].

    Returns what axis_ik_oracle.solve_axis_batch returns (axis_error is theta).  ``trace``, a list, receives q of every
    row before each pass (tests of single steps)."""
    from . import c_oracle

    tp = np.ascontiguousarray(target_pos, dtype=np.float64).reshape(-1, 3)
    n = len(tp)
    d = _normalized_axes(np.asarray(target_axis, dtype=np.float64).reshape(-1, 3), n)
    basis = tool_basis(tool_axis)
    q = np.array(np.broadcast_to(np.asarray(q_init, dtype=np.float64), (n, 7)))
    lower, upper = np.array(chain.lower[:]), np.array(chain.upper[:])
    out = dict(final_pos=np.zeros((n, 3)), final_axis=np.zeros((n, 3)), final_mat=np.zeros((n, 3, 3)),
               pos_error=np.zeros(n), axis_error=np.zeros(n), iterations=np.zeros(n, dtype=np.int64),
               converged=np.zeros(n, dtype=bool))
    act = np.arange(n)
    for i in range(max_iters + 1):
        if trace is not None:
            trace.append(q.copy())
        if len(act) == 0:
            break
        qa = q[act]
        p, mat, jac = c_oracle.fk_jac(chain, qa, nthreads=nthreads)
        a, b1, b2, theta, nv = _axis_error(mat, basis, d[act])
        e_pos = tp[act] - p
        pe = np.linalg.norm(e_pos, axis=1)
        last = i == max_iters
        done = np.ones(len(act), dtype=bool) if last else (pe < pos_thresh) & (theta - cone_angle < rot_thresh)
        idx = act[done]
        out["final_pos"][idx], out["final_axis"][idx], out["final_mat"][idx] = p[done], a[done], mat[done]
        out["pos_error"][idx], out["axis_error"][idx] = pe[done], theta[done]
        out["iterations"][idx] = max_iters if last else i + 1
        out["converged"][idx] = not last
        keep = ~done
        if not keep.any():
            break
        w, g = _tilt(theta[keep], cone_angle, rot_weight)
        jr = jac[keep, 3:6]
        J = np.concatenate([jac[keep, 0:3], w[:, None, None] * np.einsum("ni,nij->nj", b1[keep], jr)[:, None],
                            w[:, None, None] * np.einsum("ni,nij->nj", b2[keep], jr)[:, None]], axis=1)
        wt = w * g
        e = np.concatenate([e_pos[keep], (wt * np.einsum("ni,ni->n", nv[keep], b1[keep]))[:, None],
                            (wt * np.einsum("ni,ni->n", nv[keep], b2[keep]))[:, None]], axis=1)
        A = J @ np.swapaxes(J, 1, 2) + damping * np.eye(5)
        dq = (np.swapaxes(J, 1, 2) @ np.linalg.solve(A, e[:, :, None]))[:, :, 0]
        q[act[keep]] = np.clip(qa[keep] + np.clip(dq, -step_limit, step_limit), lower, upper)
        act = act[keep]
    out["q"] = q
    out["success"] = (out["converged"] & (out["pos_error"] < 2 * pos_thresh)
                      & (out["axis_error"] - cone_angle < 2 * rot_thresh))
    return out

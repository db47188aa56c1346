"""ORACLE (test infrastructure) for the axis-constrained IK EXTENSION.

A pick asks for the gripper at a point with its approach axis along a direction, and leaves the roll about that axis
free.  This module states what pnp_ik_axis_solve_* computes, in FP64 NumPy: the position solver's loop with a 5-row
task, 3 position rows and 2 tilt rows.  PARITY UNPINNED (no reference behaviour exists).

    t = normalize(tool_axis) (site frame), (u1, u2, t) the orthonormal basis of tool_basis(t)
    a = R t, b1 = R u1, b2 = R u2;  d = normalize(target_axis);  c = a x d, s = |c|, theta = atan2(s, a.d)
    n = c / s if s > 0;  b1 if s == 0 and a.d < 0;  0 otherwise
    e = [tp - p ; w theta (n.b1) ; w theta (n.b2)],  J = [jacp ; w b1^T jacr ; w b2^T jacr]   (5 x 7)
    dq = J^T solve(J J^T + damping I5, e);  q = clip(q + clip(dq, +-step_limit), lower, upper)
    converged when |tp - p| < pos_thresh and theta < rot_thresh, tested before the update
    success = converged and |tp - p| < 2 pos_thresh and theta < 2 rot_thresh
"""

from __future__ import annotations

import math

import numpy as np

from . import mj_oracle as mujoco


def tool_basis(tool_axis):
    """(t, u1, u2): t = tool_axis normalised, u1 = normalize(t x e_k) with e_k the basis vector of t's smallest-magnitude
    component (lowest index on a tie), u2 = t x u1.  Raises ValueError for a zero or non-finite tool_axis."""
    t = np.asarray(tool_axis, dtype=np.float64).reshape(3)
    nt = float(np.linalg.norm(t))
    if not np.isfinite(t).all() or not nt > 0.0:
        raise ValueError(f"tool_axis must be finite and nonzero, got {t}")
    t = t / nt
    e = np.zeros(3)
    e[int(np.argmin(np.abs(t)))] = 1.0  # argmin returns the lowest index on a tie
    u1 = np.cross(t, e)
    u1 = u1 / np.linalg.norm(u1)
    return t, u1, np.cross(t, u1)


def _normalized_axes(target_axis, n):
    d = np.broadcast_to(np.asarray(target_axis, dtype=np.float64), (n, 3))
    with np.errstate(divide="ignore", invalid="ignore"):
        return d / np.linalg.norm(d, axis=1, keepdims=True)


def _axis_error(mat, basis, d):
    """Per row: a, b1, b2 (world), theta and the tilt direction n of the statement."""
    t, u1, u2 = basis
    a, b1, b2 = mat @ t, mat @ u1, mat @ u2
    c = np.cross(a, d)
    s = np.linalg.norm(c, axis=1)
    ad = np.einsum("ni,ni->n", a, d)
    theta = np.arctan2(s, ad)
    pos = s > 0
    with np.errstate(divide="ignore", invalid="ignore"):
        nv = np.where(pos[:, None], c / np.where(pos, s, 1.0)[:, None], 0.0)
    flip = (s == 0) & (ad < 0)
    nv[flip] = b1[flip]
    return a, b1, b2, theta, nv


def solve_axis(model, data, target_pos, target_axis, q_init, tool_axis=(0.0, 0.0, 1.0), max_iters=100,
               pos_thresh=1e-3, rot_thresh=1e-2, damping=1e-2, step_limit=0.1, rot_weight=1.0,
               site_name="ee_center_site"):
    """One query on the restated engine (mj_forward / mj_jacSite)."""
    sid = model.site(site_name).id
    lower, upper = model.jnt_range[:7, 0], model.jnt_range[:7, 1]
    basis = tool_basis(tool_axis)
    t, u1, u2 = basis
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
        else:  # aligned, or a NaN target axis (theta NaN: NaN error rows)
            nv = np.zeros(3)
        e_pos = tp - p
        pe = float(np.linalg.norm(e_pos))
        if i == max_iters:
            iterations = max_iters
            break
        if pe < pos_thresh and th < rot_thresh:
            converged, iterations = True, i + 1
            break
        jp, jr = np.zeros((3, model.nv)), np.zeros((3, model.nv))
        mujoco.mj_jacSite(model, data, jp, jr, sid)
        J = np.vstack([jp[:, :7], rot_weight * (b1 @ jr[:, :7]), rot_weight * (b2 @ jr[:, :7])])
        e = np.concatenate([e_pos, [rot_weight * th * float(nv @ b1), rot_weight * th * float(nv @ b2)]])
        dq = J.T @ np.linalg.solve(J @ J.T + damping * np.eye(5), e)
        q = np.clip(q + np.clip(dq, -step_limit, step_limit), lower, upper)
    success = converged and pe < 2 * pos_thresh and th < 2 * rot_thresh
    return dict(success=success, converged=converged, q=q, final_pos=p, final_axis=a, axis_error=th,
                pos_error=pe, iterations=iterations)


# ---------------------------------------------------------------------------------------------------------------------
# The same statement over N queries at once, on the C restatement's FK (c_oracle.fk_jac).
# ---------------------------------------------------------------------------------------------------------------------
def axis_eval_batch(chain, q, target_pos, target_axis, tool_axis=(0.0, 0.0, 1.0), nthreads=8):
    """One evaluation of the statement at joint angles q[N,7]: the pass the loop makes before its convergence test.

    Returns final_pos[N,3], final_axis[N,3] (a = R t), axis_error[N] (theta), pos_error[N], mat[N,3,3] (R) and
    s[N] (|a x d|)."""
    from . import c_oracle

    q = np.ascontiguousarray(q, dtype=np.float64).reshape(-1, 7)
    n = len(q)
    p, mat, _ = c_oracle.fk_jac(chain, q, nthreads=nthreads)
    tp = np.broadcast_to(np.asarray(target_pos, dtype=np.float64), (n, 3))
    d = _normalized_axes(target_axis, n)
    a, _, _, theta, _ = _axis_error(mat, tool_basis(tool_axis), d)
    return dict(final_pos=p, final_axis=a, axis_error=theta, pos_error=np.linalg.norm(tp - p, axis=1), mat=mat,
                s=np.linalg.norm(np.cross(a, d), axis=1))


def solve_axis_batch(chain, target_pos, target_axis, q_init, tool_axis=(0.0, 0.0, 1.0), max_iters=100, pos_thresh=1e-3,
                     rot_thresh=1e-2, damping=1e-2, step_limit=0.1, rot_weight=1.0, nthreads=8, trace=None):
    """solve_axis over N queries: target_pos[N,3], target_axis[N,3] (any norm), q_init[7] or [N,7].

    Returns arrays: q, final_pos, final_axis, final_mat (R at the finishing pass), pos_error, axis_error, iterations,
    converged, success.  ``trace``, a list, receives q of every row before each pass (tests of single steps)."""
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
        done = np.ones(len(act), dtype=bool) if last else (pe < pos_thresh) & (theta < rot_thresh)
        idx = act[done]
        out["final_pos"][idx], out["final_axis"][idx], out["final_mat"][idx] = p[done], a[done], mat[done]
        out["pos_error"][idx], out["axis_error"][idx] = pe[done], theta[done]
        out["iterations"][idx] = max_iters if last else i + 1
        out["converged"][idx] = not last
        keep = ~done
        if not keep.any():
            break
        jr = jac[keep, 3:6]
        J = np.concatenate([jac[keep, 0:3], rot_weight * np.einsum("ni,nij->nj", b1[keep], jr)[:, None],
                            rot_weight * np.einsum("ni,nij->nj", b2[keep], jr)[:, None]], axis=1)
        wt = rot_weight * theta[keep]
        e = np.concatenate([e_pos[keep], (wt * np.einsum("ni,ni->n", nv[keep], b1[keep]))[:, None],
                            (wt * np.einsum("ni,ni->n", nv[keep], b2[keep]))[:, None]], axis=1)
        A = J @ np.swapaxes(J, 1, 2) + damping * np.eye(5)
        dq = (np.swapaxes(J, 1, 2) @ np.linalg.solve(A, e[:, :, None]))[:, :, 0]
        q[act[keep]] = np.clip(qa[keep] + np.clip(dq, -step_limit, step_limit), lower, upper)
        act = act[keep]
    out["q"] = q
    out["success"] = out["converged"] & (out["pos_error"] < 2 * pos_thresh) & (out["axis_error"] < 2 * rot_thresh)
    return out

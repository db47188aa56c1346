"""ORACLE (test infrastructure) for the pose-mode IK EXTENSION.

There is no reference arithmetic for this: FrankaEnv.solve_ik(target_pos, target_quat, q_init)
(/root/reference/panda_mujoco_gym/envs/panda_env.py:399-409) imports
``panda_mujoco_gym.skills.ik_solver.solve_ik``, which does not exist.  This module therefore states
the semantics the GPU kernel implements - the reference's position loop (ik_solver.py:50-101)
widened to a 6-row task - in FP64 NumPy on the restated engine (mj_oracle.py), so that the kernel
can be checked iteration for iteration.  PARITY UNPINNED (no reference behaviour exists).

    e = [target_pos - p ; w * quat2vel(target_quat (x) conj(site_quat))]   (mju_quat2Vel, dt = 1)
    J = [jacp ; w * jacr][:, :7];  dq = J^T solve(J J^T + damping I6, e)
    clip(dq, +-step_limit); q = clip(q + dq, lower, upper)
    converged when |e_pos| < pos_thresh and |rotvec| < rot_thresh, tested before the update
"""

from __future__ import annotations

import math

import numpy as np

from . import mj_oracle as mujoco


def quat2vel(q):
    axis = np.array(q[1:4], dtype=np.float64)
    sin_a_2 = math.sqrt(axis[0] ** 2 + axis[1] ** 2 + axis[2] ** 2)
    speed = 2 * math.atan2(sin_a_2, q[0])
    if speed > math.pi:
        speed -= 2 * math.pi
    return axis * (speed / sin_a_2) if sin_a_2 > 0 else np.zeros(3)


def solve_pose(model, data, target_pos, target_quat, q_init, max_iters=100, pos_thresh=1e-3, rot_thresh=1e-2,
               damping=1e-2, step_limit=0.1, rot_weight=1.0, site_name="ee_center_site"):
    sid = model.site(site_name).id
    lower, upper = model.jnt_range[:7, 0], model.jnt_range[:7, 1]
    tq = np.asarray(target_quat, dtype=np.float64)
    tq = tq / np.linalg.norm(tq)
    q = np.array(q_init, dtype=np.float64)
    converged, iterations = False, 0
    pe = re = 0.0
    for i in range(max_iters + 1):
        data.qpos[:7] = q
        mujoco.mj_forward(model, data)
        p = data.site_xpos[sid].copy()
        qc = np.empty(4)
        mujoco.mju_mat2Quat(qc, data.site_xmat[sid])
        conj = np.array([qc[0], -qc[1], -qc[2], -qc[3]])
        rv = quat2vel(mujoco.mju_mulQuat(tq, conj))
        e_pos = np.asarray(target_pos, dtype=np.float64) - p
        pe, re = float(np.linalg.norm(e_pos)), float(np.linalg.norm(rv))
        if i == max_iters:
            iterations = max_iters
            break
        if pe < pos_thresh and re < rot_thresh:
            converged, iterations = True, i + 1
            break
        jp, jr = np.zeros((3, model.nv)), np.zeros((3, model.nv))
        mujoco.mj_jacSite(model, data, jp, jr, sid)
        J = np.vstack([jp[:, :7], rot_weight * jr[:, :7]])
        e = np.concatenate([e_pos, rot_weight * rv])
        dq = J.T @ np.linalg.solve(J @ J.T + damping * np.eye(6), e)
        q = np.clip(q + np.clip(dq, -step_limit, step_limit), lower, upper)
    success = converged and pe < 2 * pos_thresh and re < 2 * rot_thresh
    return dict(success=success, converged=converged, q=q, final_pos=p, final_quat=qc, pos_error=pe, rot_error=re,
                iterations=iterations)


# ---------------------------------------------------------------------------------------------------------------------
# The same statement over N queries at once, on the C restatement's FK (c_oracle.fk_jac).  Every per-query step is the
# scalar one above written with NumPy arrays: mju_mat2Quat's case rule, mju_mulQuat, quat2vel's fold of the angle into
# (-pi, pi], the convergence test before the update, and each query's outputs frozen in the pass it finishes.
# ---------------------------------------------------------------------------------------------------------------------
def mat2quat_batch(mat):
    """mju_mat2Quat of mat[N,9] (row-major) -> (quat[N,4] wxyz, case[N], margin[N]).

    case: 0 positive trace, 1/2/3 m00/m11/m22 the largest diagonal entry (MuJoCo's tie rule).  margin is the smallest
    gap among the comparisons that selected the case (|trace|, and for cases 1-3 the lead of the largest diagonal entry
    over the next), i.e. how far the rotation is from one whose rounded matrix could take another case."""
    m = np.asarray(mat, dtype=np.float64).reshape(-1, 9)
    m0, m4, m8 = m[:, 0], m[:, 4], m[:, 8]
    tr = m0 + m4 + m8
    c0 = tr > 0
    c1 = ~c0 & (m0 > m4) & (m0 > m8)
    c2 = ~c0 & ~c1 & (m4 > m8)
    case = np.where(c0, 0, np.where(c1, 1, np.where(c2, 2, 3)))
    q = np.zeros((len(m), 4))
    with np.errstate(divide="ignore", invalid="ignore"):
        big = np.where(c0, 0.5 * np.sqrt(np.maximum(1 + m0 + m4 + m8, 0.0)), 0.0)
        big = np.where(c1, 0.5 * np.sqrt(np.maximum(1 + m0 - m4 - m8, 0.0)), big)
        big = np.where(c2, 0.5 * np.sqrt(np.maximum(1 - m0 + m4 - m8, 0.0)), big)
        big = np.where(case == 3, 0.5 * np.sqrt(np.maximum(1 - m0 - m4 + m8, 0.0)), big)
        a75, a26, a31 = 0.25 * (m[:, 7] - m[:, 5]) / big, 0.25 * (m[:, 2] - m[:, 6]) / big, 0.25 * (m[:, 3] - m[:, 1]) / big
        b13, b26, b57 = 0.25 * (m[:, 1] + m[:, 3]) / big, 0.25 * (m[:, 2] + m[:, 6]) / big, 0.25 * (m[:, 5] + m[:, 7]) / big
    rows = [(c0, (big, a75, a26, a31)), (c1, (a75, big, b13, b26)), (c2, (a26, b13, big, b57)),
            (case == 3, (a31, b26, b57, big))]
    for sel, comps in rows:
        for i in range(4):
            q[sel, i] = comps[i][sel]
    n = np.sqrt(q[:, 0] * q[:, 0] + q[:, 1] * q[:, 1] + q[:, 2] * q[:, 2] + q[:, 3] * q[:, 3])
    tiny = n < 1e-15  # mju_normalize4
    q = np.where(tiny[:, None], np.array([1.0, 0.0, 0.0, 0.0]), q / np.where(tiny, 1.0, n)[:, None])
    d = np.sort(np.stack([m0, m4, m8], axis=1), axis=1)
    margin = np.where(c0, np.abs(tr), np.minimum(np.abs(tr), d[:, 2] - d[:, 1]))
    return q, case, margin


def mulquat_batch(a, b):
    """mju_mulQuat row-wise."""
    return np.stack([
        a[:, 0] * b[:, 0] - a[:, 1] * b[:, 1] - a[:, 2] * b[:, 2] - a[:, 3] * b[:, 3],
        a[:, 0] * b[:, 1] + a[:, 1] * b[:, 0] + a[:, 2] * b[:, 3] - a[:, 3] * b[:, 2],
        a[:, 0] * b[:, 2] - a[:, 1] * b[:, 3] + a[:, 2] * b[:, 0] + a[:, 3] * b[:, 1],
        a[:, 0] * b[:, 3] + a[:, 1] * b[:, 2] - a[:, 2] * b[:, 1] + a[:, 3] * b[:, 0],
    ], axis=1)


def quat2vel_batch(q):
    """quat2vel row-wise (mju_quat2Vel, dt = 1): angle 2 atan2(|v|, w) folded into (-pi, pi]."""
    axis = q[:, 1:4]
    sin_a_2 = np.sqrt(axis[:, 0] ** 2 + axis[:, 1] ** 2 + axis[:, 2] ** 2)
    speed = 2 * np.arctan2(sin_a_2, q[:, 0])
    speed = np.where(speed > math.pi, speed - 2 * math.pi, speed)
    pos = sin_a_2 > 0
    sc = np.where(pos, speed / np.where(pos, sin_a_2, 1.0), 0.0)
    return axis * sc[:, None]


def _normalized_targets(target_quat, n):
    tq = np.broadcast_to(np.asarray(target_quat, dtype=np.float64), (n, 4))
    with np.errstate(divide="ignore", invalid="ignore"):
        return tq / np.linalg.norm(tq, axis=1, keepdims=True)


def _pose_error(p, mat, tp, tq):
    qc, case, margin = mat2quat_batch(mat.reshape(-1, 9))
    eq = mulquat_batch(tq, qc * np.array([1.0, -1.0, -1.0, -1.0]))
    rv = quat2vel_batch(eq)
    e_pos = tp - p
    return dict(qc=qc, case=case, margin=margin, err_w=eq[:, 0], rv=rv, e_pos=e_pos,
                pe=np.linalg.norm(e_pos, axis=1), re=np.linalg.norm(rv, axis=1))


def pose_eval_batch(chain, q, target_pos, target_quat, nthreads=8):
    """One evaluation of the statement at joint angles q[N,7]: the pass the loop makes before its convergence test.

    Returns final_pos[N,3], final_quat[N,4] (mju_mat2Quat of the site frame), pos_error[N], rot_error[N] (rad),
    case[N] / case_margin[N] (see mat2quat_batch) and err_w[N], the w of target (x) conj(site quat) - negative when the
    angle fold of quat2vel applies."""
    from . import c_oracle

    q = np.ascontiguousarray(q, dtype=np.float64).reshape(-1, 7)
    n = len(q)
    p, mat, _ = c_oracle.fk_jac(chain, q, nthreads=nthreads)
    tp = np.broadcast_to(np.asarray(target_pos, dtype=np.float64), (n, 3))
    ev = _pose_error(p, mat, tp, _normalized_targets(target_quat, n))
    return dict(final_pos=p, final_quat=ev["qc"], pos_error=ev["pe"], rot_error=ev["re"], case=ev["case"],
                case_margin=ev["margin"], err_w=ev["err_w"])


def solve_pose_batch(chain, target_pos, target_quat, q_init, max_iters=100, pos_thresh=1e-3, rot_thresh=1e-2,
                     damping=1e-2, step_limit=0.1, rot_weight=1.0, nthreads=8):
    """solve_pose over N queries: target_pos[N,3], target_quat[N,4] wxyz (any norm), q_init[7] or [N,7].

    Returns arrays: q, final_pos, final_quat, pos_error, rot_error, iterations, converged, success."""
    from . import c_oracle

    tp = np.ascontiguousarray(target_pos, dtype=np.float64).reshape(-1, 3)
    n = len(tp)
    tq = _normalized_targets(np.asarray(target_quat, dtype=np.float64).reshape(-1, 4), n)
    q = np.array(np.broadcast_to(np.asarray(q_init, dtype=np.float64), (n, 7)))
    lower, upper = np.array(chain.lower[:]), np.array(chain.upper[:])
    out = dict(final_pos=np.zeros((n, 3)), final_quat=np.zeros((n, 4)), pos_error=np.zeros(n), rot_error=np.zeros(n),
               iterations=np.zeros(n, dtype=np.int64), converged=np.zeros(n, dtype=bool))
    w6 = np.array([1.0, 1.0, 1.0, rot_weight, rot_weight, rot_weight])
    act = np.arange(n)
    for i in range(max_iters + 1):
        if len(act) == 0:
            break
        qa = q[act]
        p, mat, jac = c_oracle.fk_jac(chain, qa, nthreads=nthreads)
        ev = _pose_error(p, mat, tp[act], tq[act])
        last = i == max_iters
        done = np.ones(len(act), dtype=bool) if last else (ev["pe"] < pos_thresh) & (ev["re"] < rot_thresh)
        idx = act[done]
        out["final_pos"][idx], out["final_quat"][idx] = p[done], ev["qc"][done]
        out["pos_error"][idx], out["rot_error"][idx] = ev["pe"][done], ev["re"][done]
        out["iterations"][idx] = max_iters if last else i + 1
        out["converged"][idx] = not last
        keep = ~done
        if not keep.any():
            break
        J = jac[keep] * w6[None, :, None]
        e = np.concatenate([ev["e_pos"][keep], rot_weight * ev["rv"][keep]], axis=1)
        A = J @ np.swapaxes(J, 1, 2) + damping * np.eye(6)
        dq = (np.swapaxes(J, 1, 2) @ np.linalg.solve(A, e[:, :, None]))[:, :, 0]
        q[act[keep]] = np.clip(qa[keep] + np.clip(dq, -step_limit, step_limit), lower, upper)
        act = act[keep]
    out["q"] = q
    out["success"] = out["converged"] & (out["pos_error"] < 2 * pos_thresh) & (out["rot_error"] < 2 * rot_thresh)
    return out

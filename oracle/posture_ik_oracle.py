"""ORACLE (test infrastructure) for posture-regularised IK (pnp_ik_solve_posture_* / pnp_ik_pose_solve_posture_*).

No reference arithmetic exists for a null-space term: the reference solver (ik_solver.py:50-101) has none (SURVEY App.
D.4).  This module states the semantics the GPU kernels implement, in FP64 NumPy: the position loop of ik_oracle and the
pose loop of pose_ik_oracle with the step alone changed.  PARITY UNPINNED (no reference behaviour exists).

At a pass at q, with J, e and lambda = damping of the plain solver (3 rows; pose: 6 rows, rotation rows * rot_weight):

    z  = gain (q_rest - q)
    y  = (J J^T + lambda I)^-1 (e - J z)
    dq = z + J^T y                        = J+ e + (I - J+ J) z,   J+ = J^T (J J^T + lambda I)^-1
    q <- clip(q + clip(dq, +-step_limit), lower, upper)

Everything else is the plain loop: the convergence test on the TASK error before the update, iterations = i + 1, the
success rule.  gain = 0 gives z = 0, e - J 0 = e and 0 + J^T y = J^T y: the plain solver's iterates.
"""

from __future__ import annotations

import numpy as np

from . import mj_oracle as mujoco
from . import pose_ik_oracle as pio


def posture_step(J, e, q, q_rest, gain, damping):
    """dq of one pass (single query: J[m,7], e[m], q[7]; or batched: J[N,m,7], e[N,m], q[N,7], q_rest[7] / [N,7])."""
    z = gain * (q_rest - q)
    if J.ndim == 2:
        A = J @ J.T + damping * np.eye(J.shape[0])
        y = np.linalg.solve(A, e - J @ z)
        return z + J.T @ y
    A = J @ np.swapaxes(J, 1, 2) + damping * np.eye(J.shape[1])
    y = np.linalg.solve(A, (e - (J @ z[:, :, None])[:, :, 0])[:, :, None])
    return z + (np.swapaxes(J, 1, 2) @ y)[:, :, 0]


# ---------------------------------------------------------------------------------------------------------------------
# Scalar statements over the restated engine (mj_oracle)
# ---------------------------------------------------------------------------------------------------------------------
def solve_position(model, data, target_pos, q_init, q_rest, gain, max_iters=100, pos_thresh=1e-3, damping=1e-2,
                   step_limit=0.1, site_name="ee_center_site", step=posture_step):
    """ik_oracle.JacobianIKController.solve with the posture step.  ``step``: the step formula (the tests pass an
    independent projector form)."""
    sid = model.site(site_name).id
    lower, upper = model.jnt_range[:7, 0], model.jnt_range[:7, 1]
    tp = np.asarray(target_pos, dtype=np.float64)
    q_rest = np.asarray(q_rest, dtype=np.float64)
    q = np.array(q_init, dtype=np.float64)
    hit, n_iter = False, 0
    for k in range(max_iters):
        data.qpos[:7] = q
        mujoco.mj_forward(model, data)
        e = tp - data.site_xpos[sid]
        if np.linalg.norm(e) < pos_thresh:
            hit, n_iter = True, k + 1
            break
        jp, jr = np.zeros((3, model.nv)), np.zeros((3, model.nv))
        mujoco.mj_jacSite(model, data, jp, jr, sid)
        dq = step(jp[:, :7], e, q, q_rest, gain, damping)
        q = np.clip(q + np.clip(dq, -step_limit, step_limit), lower, upper)
        n_iter = k + 1
    data.qpos[:7] = q
    mujoco.mj_forward(model, data)
    p = data.site_xpos[sid].copy()
    err = float(np.linalg.norm(p - tp))
    return dict(success=bool(hit and err < 2 * pos_thresh), converged=hit, q=q, final_pos=p, pos_error=err,
                iterations=n_iter)


def solve_pose(model, data, target_pos, target_quat, q_init, q_rest, gain, max_iters=100, pos_thresh=1e-3,
               rot_thresh=1e-2, damping=1e-2, step_limit=0.1, rot_weight=1.0, site_name="ee_center_site",
               step=posture_step):
    """pose_ik_oracle.solve_pose with the posture step."""
    sid = model.site(site_name).id
    lower, upper = model.jnt_range[:7, 0], model.jnt_range[:7, 1]
    tq = np.asarray(target_quat, dtype=np.float64)
    tq = tq / np.linalg.norm(tq)
    q_rest = np.asarray(q_rest, dtype=np.float64)
    q = np.array(q_init, dtype=np.float64)
    converged, iterations = False, 0
    for i in range(max_iters + 1):
        data.qpos[:7] = q
        mujoco.mj_forward(model, data)
        p = data.site_xpos[sid].copy()
        qc = np.empty(4)
        mujoco.mju_mat2Quat(qc, data.site_xmat[sid])
        rv = pio.quat2vel(mujoco.mju_mulQuat(tq, np.array([qc[0], -qc[1], -qc[2], -qc[3]])))
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
        q = np.clip(q + np.clip(step(J, e, q, q_rest, gain, damping), -step_limit, step_limit), lower, upper)
    success = converged and pe < 2 * pos_thresh and re < 2 * rot_thresh
    return dict(success=success, converged=converged, q=q, final_pos=p, final_quat=qc, pos_error=pe, rot_error=re,
                iterations=iterations)


# ---------------------------------------------------------------------------------------------------------------------
# The same statements over N queries at once, on the C restatement's FK (c_oracle.fk_jac); each query's outputs are
# frozen in the pass it finishes, as in pose_ik_oracle.solve_pose_batch.
# ---------------------------------------------------------------------------------------------------------------------
def _rows(x, n):
    return np.array(np.broadcast_to(np.asarray(x, dtype=np.float64), (n, 7)))


def solve_position_batch(chain, target_pos, q_init, q_rest, gain, max_iters=100, pos_thresh=1e-3, damping=1e-2,
                         step_limit=0.1, nthreads=8):
    """solve_position over N queries: target_pos[N,3], q_init / q_rest [7] or [N,7].
    Returns arrays: q, final_pos, pos_error, iterations, converged, success."""
    from . import c_oracle

    tp = np.ascontiguousarray(target_pos, dtype=np.float64).reshape(-1, 3)
    n = len(tp)
    q, qr = _rows(q_init, n), _rows(q_rest, n)
    lower, upper = np.array(chain.lower[:]), np.array(chain.upper[:])
    out = dict(final_pos=np.zeros((n, 3)), pos_error=np.zeros(n), iterations=np.zeros(n, dtype=np.int64),
               converged=np.zeros(n, dtype=bool))
    act = np.arange(n)
    for i in range(max_iters + 1):
        if len(act) == 0:
            break
        qa = q[act]
        p, _, jac = c_oracle.fk_jac(chain, qa, nthreads=nthreads)
        e = tp[act] - p
        pe = np.linalg.norm(e, axis=1)
        last = i == max_iters
        done = np.ones(len(act), dtype=bool) if last else pe < pos_thresh
        idx = act[done]
        out["final_pos"][idx], out["pos_error"][idx] = p[done], pe[done]
        out["iterations"][idx] = max_iters if last else i + 1
        out["converged"][idx] = not last
        keep = ~done
        if not keep.any():
            break
        dq = posture_step(jac[keep, :3], e[keep], qa[keep], qr[act[keep]], gain, damping)
        q[act[keep]] = np.clip(qa[keep] + np.clip(dq, -step_limit, step_limit), lower, upper)
        act = act[keep]
    out["q"] = q
    out["success"] = out["converged"] & (out["pos_error"] < 2 * pos_thresh)
    return out


def solve_pose_batch(chain, target_pos, target_quat, q_init, q_rest, gain, max_iters=100, pos_thresh=1e-3,
                     rot_thresh=1e-2, damping=1e-2, step_limit=0.1, rot_weight=1.0, nthreads=8):
    """solve_pose over N queries (pose_ik_oracle.solve_pose_batch with the posture step).
    Returns arrays: q, final_pos, final_quat, pos_error, rot_error, iterations, converged, success."""
    from . import c_oracle

    tp = np.ascontiguousarray(target_pos, dtype=np.float64).reshape(-1, 3)
    n = len(tp)
    tq = pio._normalized_targets(np.asarray(target_quat, dtype=np.float64).reshape(-1, 4), n)
    q, qr = _rows(q_init, n), _rows(q_rest, n)
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
        ev = pio._pose_error(p, mat, tp[act], tq[act])
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
        dq = posture_step(J, e, qa[keep], qr[act[keep]], gain, damping)
        q[act[keep]] = np.clip(qa[keep] + np.clip(dq, -step_limit, step_limit), lower, upper)
        act = act[keep]
    out["q"] = q
    out["success"] = out["converged"] & (out["pos_error"] < 2 * pos_thresh) & (out["rot_error"] < 2 * rot_thresh)
    return out


# ---------------------------------------------------------------------------------------------------------------------
# Step-0 statistics of a batch result
# ---------------------------------------------------------------------------------------------------------------------
def limit_margin(q, lower, upper):
    """Smallest normalised joint-limit margin min_j min(q - lo, hi - q) / (hi - lo), per row."""
    lo, hi = np.asarray(lower, dtype=np.float64), np.asarray(upper, dtype=np.float64)
    return (np.minimum(q - lo, hi - q) / (hi - lo)).min(axis=1)


def summarize(out, q_rest, lower, upper):
    """success rate, mean iterations, mean |q - q_rest|, margin mean / 5th percentile, and the fraction of failures that
    end with a joint on its limit."""
    q = out["q"]
    lo, hi = np.asarray(lower, dtype=np.float64), np.asarray(upper, dtype=np.float64)
    m = limit_margin(q, lo, hi)
    fail = ~out["success"]
    on_limit = ((q <= lo) | (q >= hi)).any(axis=1)
    return dict(success=float(out["success"].mean()), mean_iters=float(out["iterations"].mean()),
                rest_dist=float(np.linalg.norm(q - np.asarray(q_rest), axis=1).mean()), margin_mean=float(m.mean()),
                margin_p5=float(np.percentile(m, 5)),
                fail_on_limit=float(on_limit[fail].mean()) if fail.any() else 0.0)


def mid_range(lower, upper):
    """The default rest posture: the middle of each joint's range."""
    return 0.5 * (np.asarray(lower, dtype=np.float64) + np.asarray(upper, dtype=np.float64))


def cold_targets(chain, n, seed=1234):
    """Reachable targets of the cfg5 / W-cold workloads: q* ~ U(joint limits) from synthetic.random_joint_configs (CPU
    generator, FP64); returns (q*, FK position, site quaternion)."""
    import torch

    from mujoco_panda_pnp_b200 import synthetic

    q_star = synthetic.random_joint_configs(n, chain.lower[:], chain.upper[:], seed=seed, dtype=torch.float64).numpy()
    ev = pio.pose_eval_batch(chain, q_star, np.zeros(3), np.array([1.0, 0.0, 0.0, 0.0]))
    return q_star, ev["final_pos"], ev["final_quat"]


def sweep(chain, q_init, n=1 << 16, gains=(0.0, 0.02, 0.05, 0.1, 0.2, 0.5), seed=1234, nthreads=8):
    """The Step-0 table: summarize() of the position and the pose solve of n cold targets from q_init, per gain, with
    q_rest = mid_range of the chain's limits."""
    lo, hi = np.array(chain.lower[:]), np.array(chain.upper[:])
    qr = mid_range(lo, hi)
    _, pos, quat = cold_targets(chain, n, seed)
    rows = []
    for g in gains:
        rp = solve_position_batch(chain, pos, q_init, qr, g, nthreads=nthreads)
        ro = solve_pose_batch(chain, pos, quat, q_init, qr, g, nthreads=nthreads)
        rows.append(dict(gain=g, position=summarize(rp, qr, lo, hi), pose=summarize(ro, qr, lo, hi)))
    return rows

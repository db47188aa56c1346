"""CPU: the FP64 statement of axis-constrained IK (oracle/axis_ik_oracle.py), held against itself in its two
implementations, against the damped projected 6-row form it is equivalent to, and on the A-cold workload: q* uniform
in the joint limits, target (FK(q*), R(q*) t), start NEUTRAL."""
import numpy as np
import pytest
import torch

from conftest import NEUTRAL
from mujoco_panda_pnp_b200 import synthetic
from oracle import axis_ik_oracle, c_oracle, mj_oracle, pose_ik_oracle


def _limits(chain):
    return np.array(chain.lower[:]), np.array(chain.upper[:])


def _a_cold(chain, n, seed=1234, tool=(0.0, 0.0, 1.0)):
    lo, hi = _limits(chain)
    q_star = synthetic.random_joint_configs(n, lo, hi, seed=seed, dtype=torch.float64).numpy()
    p, mat, _ = c_oracle.fk_jac(chain, q_star, nthreads=8)
    return q_star, p, mat @ axis_ik_oracle.tool_basis(tool)[0], mat


def test_tool_basis_rule():
    t, u1, u2 = axis_ik_oracle.tool_basis((0.0, 0.0, 2.0))
    assert np.array_equal(t, [0, 0, 1]) and np.array_equal(u1, [0, 1, 0]) and np.array_equal(u2, [-1, 0, 0])
    rng = np.random.default_rng(3)
    for v in list(rng.normal(size=(64, 3))) + [np.array([1.0, 1.0, 1.0]), np.array([0.0, -3.0, 0.0])]:
        t, u1, u2 = axis_ik_oracle.tool_basis(v)
        B = np.stack([u1, u2, t])
        np.testing.assert_allclose(B @ B.T, np.eye(3), atol=1e-15)
        assert np.linalg.det(B) > 0 and np.allclose(t, v / np.linalg.norm(v), atol=1e-15)
    for bad in ((0.0, 0.0, 0.0), (np.nan, 0.0, 1.0), (np.inf, 0.0, 0.0)):
        with pytest.raises(ValueError):
            axis_ik_oracle.tool_basis(bad)


@pytest.mark.parametrize("tool", [(0.0, 0.0, 1.0), (0.3, -0.2, 0.9)])
def test_scalar_and_batched_statements_agree(oracle_model, oracle_chain, tool):
    q_star, p, ax, _ = _a_cold(oracle_chain, 24, seed=7, tool=tool)
    ref = axis_ik_oracle.solve_axis_batch(oracle_chain, p, ax, NEUTRAL, tool_axis=tool)
    d = mj_oracle.MjData(oracle_model)
    for k in range(len(p)):
        w = axis_ik_oracle.solve_axis(oracle_model, d, p[k], ax[k], NEUTRAL, tool_axis=tool)
        assert w["iterations"] == ref["iterations"][k] and w["converged"] == ref["converged"][k], k
        assert w["success"] == ref["success"][k]
        np.testing.assert_allclose(w["q"], ref["q"][k], atol=1e-9)
        np.testing.assert_allclose(w["final_axis"], ref["final_axis"][k], atol=1e-9)
        assert abs(w["axis_error"] - ref["axis_error"][k]) < 1e-9
    assert ref["converged"].sum() >= 15


def _solve_projected(chain, tp, ta, q_init, tool, max_iters=100, pos_thresh=1e-3, rot_thresh=1e-2, damping=1e-2,
                     step_limit=0.1, rot_weight=1.0):
    """The same task as the damped 6-row system J = [jacp; w (I - a a^T) jacr], e = [tp - p; w theta n], 6x6 solve."""
    n = len(tp)
    t = axis_ik_oracle.tool_basis(tool)[0]
    d = ta / np.linalg.norm(ta, axis=1, keepdims=True)
    q = np.array(np.broadcast_to(q_init, (n, 7)))
    lo, hi = _limits(chain)
    iters = np.full(n, max_iters)
    act = np.ones(n, dtype=bool)
    for i in range(max_iters):
        p, mat, jac = c_oracle.fk_jac(chain, q, nthreads=8)
        a = mat @ t
        c = np.cross(a, d)
        s = np.linalg.norm(c, axis=1)
        th = np.arctan2(s, np.einsum("ni,ni->n", a, d))
        nv = c / s[:, None]
        done = act & (np.linalg.norm(tp - p, axis=1) < pos_thresh) & (th < rot_thresh)
        iters[done] = i + 1
        act &= ~done
        P = np.eye(3)[None] - a[:, :, None] * a[:, None, :]
        J = np.concatenate([jac[:, :3], rot_weight * P @ jac[:, 3:]], axis=1)
        e = np.concatenate([tp - p, rot_weight * th[:, None] * nv], axis=1)
        dq = (np.swapaxes(J, 1, 2) @ np.linalg.solve(J @ np.swapaxes(J, 1, 2) + damping * np.eye(6), e[:, :, None]))[:, :, 0]
        q = np.where(act[:, None], np.clip(q + np.clip(dq, -step_limit, step_limit), lo, hi), q)
    return q, iters


def test_basis_form_equals_projected_six_row_form(oracle_chain, monkeypatch):
    tool = (0.2, 0.5, -0.8)
    _, p, ax, _ = _a_cold(oracle_chain, 512, seed=11, tool=tool)
    ref = axis_ik_oracle.solve_axis_batch(oracle_chain, p, ax, NEUTRAL, tool_axis=tool)
    q6, it6 = _solve_projected(oracle_chain, p, ax, NEUTRAL, tool)
    assert np.array_equal(ref["iterations"], it6)
    assert np.abs(ref["q"] - q6).max() < 1e-9
    # any orthonormal completion (u1, u2) of t gives the same steps: rotate it about t by a random angle
    t, u1, u2 = axis_ik_oracle.tool_basis(tool)
    g = np.random.default_rng(5).uniform(0, 2 * np.pi)
    rot = (t, np.cos(g) * u1 + np.sin(g) * u2, -np.sin(g) * u1 + np.cos(g) * u2)
    monkeypatch.setattr(axis_ik_oracle, "tool_basis", lambda _: rot)
    alt = axis_ik_oracle.solve_axis_batch(oracle_chain, p, ax, NEUTRAL, tool_axis=tool)
    assert np.array_equal(ref["iterations"], alt["iterations"])
    assert np.abs(ref["q"] - alt["q"]).max() < 1e-9
    assert ref["converged"].mean() > 0.8


def test_antiparallel_start_steps_along_b1(oracle_chain):
    """a = -d exactly at the start (s = 0, theta = pi): n = b1, the first step turns the tool about b1."""
    lo, hi = _limits(oracle_chain)
    q = np.random.default_rng(13).uniform(lo, hi, (256, 7))
    _, mat, _ = c_oracle.fk_jac(oracle_chain, q)
    ev = axis_ik_oracle.axis_eval_batch(oracle_chain, q, np.zeros(3), -(mat[:, :, 2]))
    exact = np.nonzero(ev["s"] == 0)[0]
    assert len(exact) >= 8
    k = exact[:8]
    q0, p0, d = q[k], ev["final_pos"][k], -(mat[k, :, 2])
    assert np.all(ev["axis_error"][k] == np.pi)
    trace = []
    axis_ik_oracle.solve_axis_batch(oracle_chain, p0, d, q0, max_iters=1, trace=trace)
    dq = trace[1] - q0
    assert (np.abs(dq).max(axis=1) > 1e-2).all()
    # the DLS step of the error [0, 0, 0, pi, 0]: a pure tilt about b1, no position error
    _, mat0, jac0 = c_oracle.fk_jac(oracle_chain, q0)
    t, u1, u2 = axis_ik_oracle.tool_basis((0, 0, 1))
    J = np.concatenate([jac0[:, :3], np.einsum("ni,nij->nj", mat0 @ u1, jac0[:, 3:])[:, None],
                        np.einsum("ni,nij->nj", mat0 @ u2, jac0[:, 3:])[:, None]], axis=1)
    e = np.tile([0.0, 0.0, 0.0, np.pi, 0.0], (len(k), 1))
    want = (np.swapaxes(J, 1, 2) @ np.linalg.solve(J @ np.swapaxes(J, 1, 2) + 1e-2 * np.eye(5), e[:, :, None]))[:, :, 0]
    np.testing.assert_allclose(trace[1], np.clip(q0 + np.clip(want, -0.1, 0.1), lo, hi), atol=1e-12)
    after = axis_ik_oracle.axis_eval_batch(oracle_chain, trace[1], p0, d)
    assert (after["s"] > 0).all() and (after["axis_error"] < np.pi).all()
    out = axis_ik_oracle.solve_axis_batch(oracle_chain, p0, d, q0, max_iters=100)
    assert np.median(out["axis_error"]) < 1.0, out["axis_error"]


def test_degenerate_target_axis(oracle_model, oracle_chain):
    _, p, ax, _ = _a_cold(oracle_chain, 8, seed=17)
    ax[[1, 4]] = 0.0
    ax[6] = [np.nan, 0.0, 1.0]
    bad = np.zeros(8, dtype=bool)
    bad[[1, 4, 6]] = True
    out = axis_ik_oracle.solve_axis_batch(oracle_chain, p, ax, NEUTRAL, max_iters=30)
    assert not out["converged"][bad].any() and not out["success"][bad].any()
    assert (out["iterations"][bad] == 30).all()
    d = mj_oracle.MjData(oracle_model)
    w = axis_ik_oracle.solve_axis(oracle_model, d, p[1], ax[1], NEUTRAL, max_iters=30)
    assert not w["success"] and w["iterations"] == 30
    clean = axis_ik_oracle.solve_axis_batch(oracle_chain, p[~bad], ax[~bad], NEUTRAL, max_iters=30)
    assert np.array_equal(clean["q"], out["q"][~bad])


def test_a_cold_axis_task_beats_the_pose_task(oracle_chain):
    """4096 A-cold targets from NEUTRAL: the axis task leaves the Panda one more redundant joint than the pose task on
    the same q*, and solves clearly more of them (FP64, default parameters)."""
    q_star, p, ax, mat = _a_cold(oracle_chain, 4096)
    axis = axis_ik_oracle.solve_axis_batch(oracle_chain, p, ax, NEUTRAL)
    quat = pose_ik_oracle.mat2quat_batch(mat.reshape(-1, 9))[0]
    pose = pose_ik_oracle.solve_pose_batch(oracle_chain, p, quat, NEUTRAL)
    sa, sp = axis["success"].mean(), pose["success"].mean()
    assert sa >= 0.85 and sa >= sp + 0.1, (sa, sp)

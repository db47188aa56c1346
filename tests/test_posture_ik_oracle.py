"""CPU checks of the posture-regularised IK statement (oracle/posture_ik_oracle.py) and of its Step-0 finding.

The statement: the plain position / pose loop with the step dq = z + J^T (J J^T + lambda I)^-1 (e - J z),
z = gain (q_rest - q).  Targets are cold: q* ~ U(joint limits), solved from NEUTRAL, q_rest = mid-range."""
import numpy as np
import pytest

from conftest import NEUTRAL
from oracle import ik_oracle, mj_oracle, pose_ik_oracle
from oracle import posture_ik_oracle as pk


def projector_step(J, e, q, q_rest, gain, damping):
    """The damped projector form J+ e + (I - J+ J) z, J+ = J^T (J J^T + lambda I)^-1, with an explicit inverse."""
    jp = J.T @ np.linalg.inv(J @ J.T + damping * np.eye(J.shape[0]))
    z = gain * (np.asarray(q_rest) - q)
    return jp @ e + (np.eye(7) - jp @ J) @ z


@pytest.fixture(scope="module")
def limits(oracle_chain):
    return np.array(oracle_chain.lower[:]), np.array(oracle_chain.upper[:])


@pytest.fixture(scope="module")
def cold(oracle_chain):
    return pk.cold_targets(oracle_chain, 1024, seed=7)


@pytest.mark.parametrize("gain", [0.02, 0.1])
def test_statement_matches_projector_form(oracle_model, limits, cold, gain):
    """Both solvers: the rearranged step and the explicit projector give the same iterations and q to 1e-8."""
    d = mj_oracle.MjData(oracle_model)
    qr = pk.mid_range(*limits)
    _, pos, quat = cold
    for i in range(4):
        a = pk.solve_position(oracle_model, d, pos[i], NEUTRAL, qr, gain)
        b = pk.solve_position(oracle_model, d, pos[i], NEUTRAL, qr, gain, step=projector_step)
        assert a["iterations"] == b["iterations"] and a["converged"] == b["converged"], i
        np.testing.assert_allclose(a["q"], b["q"], atol=1e-8)
        a = pk.solve_pose(oracle_model, d, pos[i], quat[i], NEUTRAL, qr, gain)
        b = pk.solve_pose(oracle_model, d, pos[i], quat[i], NEUTRAL, qr, gain, step=projector_step)
        assert a["iterations"] == b["iterations"] and a["converged"] == b["converged"], i
        np.testing.assert_allclose(a["q"], b["q"], atol=1e-8)


def test_gain_zero_is_the_plain_solver(oracle_model, oracle_chain, limits, cold):
    """gain = 0 reproduces ik_oracle / pose_ik_oracle, scalar and batched."""
    d = mj_oracle.MjData(oracle_model)
    qr = pk.mid_range(*limits)
    _, pos, quat = cold
    ctl = ik_oracle.JacobianIKController(oracle_model, d)
    for i in range(4):
        a = pk.solve_position(oracle_model, d, pos[i], NEUTRAL, qr, 0.0)
        b = ctl.solve(pos[i], NEUTRAL)
        assert a["iterations"] == b.iterations and a["success"] == b.success
        # (ik_oracle forms J J^T and J^T y over all nv columns, finger columns included: other summation order, 1 ulp)
        np.testing.assert_allclose(a["q"], b.q, rtol=0, atol=1e-12)
        a = pk.solve_pose(oracle_model, d, pos[i], quat[i], NEUTRAL, qr, 0.0)
        b = pose_ik_oracle.solve_pose(oracle_model, d, pos[i], quat[i], NEUTRAL)
        assert a["iterations"] == b["iterations"] and a["success"] == b["success"]
        np.testing.assert_array_equal(a["q"], b["q"])
    a = pk.solve_pose_batch(oracle_chain, pos[:256], quat[:256], NEUTRAL, qr, 0.0)
    b = pose_ik_oracle.solve_pose_batch(oracle_chain, pos[:256], quat[:256], NEUTRAL)
    for key in b:
        np.testing.assert_array_equal(a[key], b[key], err_msg=key)
    a = pk.solve_position_batch(oracle_chain, pos[:256], NEUTRAL, qr, 0.0)
    from oracle import c_oracle
    b = c_oracle.ik_solve(oracle_chain, pos[:256], NEUTRAL, nthreads=8)
    np.testing.assert_array_equal(a["iterations"], b["iterations"])
    np.testing.assert_array_equal(a["success"], b["success"])
    np.testing.assert_allclose(a["q"], b["q"], atol=1e-9)


@pytest.mark.parametrize("gain", [0.02, 0.1])
def test_joint7_follows_the_closed_form(oracle_model, oracle_chain, limits, cold, gain):
    """Position mode: joint 7's Jacobian column is zero (the EE site lies on its axis), so dq_7 = z_7 and
    q_7 = q_rest_7 + (1 - gain)^m (q_7^0 - q_rest_7) after m updates while neither clip acts."""
    qr = pk.mid_range(*limits)
    q0 = NEUTRAL.copy()
    assert abs(gain * (qr[6] - q0[6])) < 0.1  # no step clip on joint 7 at any pass
    _, pos, _ = cold
    out = pk.solve_position_batch(oracle_chain, pos[:128], q0, qr, gain)
    m = np.where(out["converged"], out["iterations"] - 1, out["iterations"])  # updates: the test precedes the update
    want = qr[6] + (1.0 - gain) ** m * (q0[6] - qr[6])
    np.testing.assert_allclose(out["q"][:, 6], want, rtol=0, atol=1e-12)
    d = mj_oracle.MjData(oracle_model)
    r = pk.solve_position(oracle_model, d, pos[0], q0, qr, gain)
    m0 = r["iterations"] - 1 if r["converged"] else r["iterations"]
    assert abs(r["q"][6] - (qr[6] + (1.0 - gain) ** m0 * (q0[6] - qr[6]))) < 1e-12


def test_step0_finding_pinned(oracle_chain, limits, cold):
    """Step 0 (DESIGN.md 4.7), pinned as measured on a fixed 1024-target sample: already at the smallest gain of the
    sweep (0.02) the damped projector's task-space leak costs both solvers a large share of their successes, so no gain
    of the sweep qualifies as a default."""
    qr = pk.mid_range(*limits)
    _, pos, quat = cold
    p0 = pk.solve_position_batch(oracle_chain, pos, NEUTRAL, qr, 0.0)
    p1 = pk.solve_position_batch(oracle_chain, pos, NEUTRAL, qr, 0.02)
    o0 = pk.solve_pose_batch(oracle_chain, pos, quat, NEUTRAL, qr, 0.0)
    o1 = pk.solve_pose_batch(oracle_chain, pos, quat, NEUTRAL, qr, 0.02)
    assert p0["success"].mean() > 0.99 and p1["success"].mean() < p0["success"].mean() - 0.10
    assert o0["success"].mean() > 0.65 and o1["success"].mean() < o0["success"].mean() - 0.30
    assert p1["iterations"].mean() > 1.25 * p0["iterations"].mean()
    assert o1["iterations"].mean() > 1.25 * o0["iterations"].mean()


def test_stalled_position_solves_sit_at_the_leak_fixed_point(oracle_chain, limits, cold):
    """Why the solves stall: a pass moves the task error to lambda (J J^T + lambda I)^-1 (e - J z), whose fixed point is
    e* = -lambda (J J^T)^-1 J z - an error of order lambda gain |q_rest - q| / sigma(J), pos_thresh already at gain
    0.02.  The position solves that run out of passes end there."""
    from oracle import c_oracle

    qr = pk.mid_range(*limits)
    _, pos, _ = cold
    gain, damping = 0.02, 1e-2
    out = pk.solve_position_batch(oracle_chain, pos, NEUTRAL, qr, gain)
    lo, hi = limits
    stalled = ~out["converged"] & ~((out["q"] <= lo) | (out["q"] >= hi)).any(axis=1)
    assert stalled.sum() >= 100
    q = out["q"][stalled]
    p, _, jac = c_oracle.fk_jac(oracle_chain, q, nthreads=8)
    J = jac[:, :3]
    e = pos[stalled] - p
    jz = (J @ (gain * (qr - q))[:, :, None])[:, :, 0]
    e_star = -damping * np.linalg.solve(J @ np.swapaxes(J, 1, 2), jz[:, :, None])[:, :, 0]
    rel = np.linalg.norm(e - e_star, axis=1) / np.linalg.norm(e, axis=1)
    assert np.median(rel) < 0.05
    assert np.median(np.linalg.norm(e, axis=1)) > 1e-3  # above pos_thresh: the convergence test never passes

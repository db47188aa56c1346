"""CPU checks of the axis-mode move planner's FP64 statement (oracle/move_axis_oracle.py).

Workload W1: synthetic.reachable_pose_move_envs - start near NEUTRAL, goal (FK(q*), R(q*) t) with q* = NEUTRAL
+- 0.6 rad clipped to the limits and t the tool axis.  Default planner and IK parameters throughout."""
import math

import numpy as np
import pytest
import torch
from scipy.spatial.transform import Rotation

from conftest import NEUTRAL
from mujoco_panda_pnp_b200 import synthetic
from oracle import axis_ik_oracle, move_axis_oracle

IK_POS_THRESH, IK_ROT_THRESH = 1e-3, 1e-2
POS_THRESH, ROT_THRESH, STEP, ROT_STEP, MAX_POINTS = 0.01, 0.05, 0.01, 0.05, 200
Z, OBLIQUE = (0.0, 0.0, 1.0), (1.0, 1.0, 1.0)


def axis_workload(oracle_model, oracle_chain, n, seed=0, tool_axis=Z):
    """(q_start[N,7], goal_pos[N,3], goal_axis[N,3]) of W1, FK by the C restatement."""
    lo, hi = oracle_model.jnt_range[:7, 0], oracle_model.jnt_range[:7, 1]
    e = synthetic.reachable_pose_move_envs(n, lo, hi, seed=seed, dtype=torch.float64)
    ev = axis_ik_oracle.axis_eval_batch(oracle_chain, e["q_goal"].numpy(), np.zeros(3), np.array([0.0, 0.0, 1.0]),
                                        tool_axis=tool_axis)
    return e["q_start"].numpy(), ev["final_pos"], ev["final_axis"]


def neutral_frame(oracle_chain, tool_axis=Z):
    ev = axis_ik_oracle.axis_eval_batch(oracle_chain, NEUTRAL[None], np.zeros(3), np.array([0.0, 0.0, 1.0]),
                                        tool_axis=tool_axis)
    return ev["final_pos"][0], ev["final_axis"][0], ev["mat"][0]


def check_invariants(oracle_model, oracle_chain, plan, goal_pos, goal_axis, fk_pos_tol, fk_rot_tol, tool_axis=Z,
                     max_points=MAX_POINTS):
    """What every plan of the statement satisfies (also applied to the GPU's FP32 plans, with FK tolerances): every
    point is FK(q) of its joints (position to fk_pos_tol, tool axis and quaternion components up to sign to
    fk_rot_tol), the joints are inside the limits, steps and turns are bounded, and an OK plan ends at the goal."""
    pos, axis, quat, qs = plan["pos_traj"], plan["axis_traj"], plan["quat_traj"], plan["q_traj"]
    L = len(pos)
    assert 1 <= L <= max_points + 1 and plan["n_solves"] <= 3 * max_points
    ev = axis_ik_oracle.axis_eval_batch(oracle_chain, qs, np.zeros(3), np.array([0.0, 0.0, 1.0]), tool_axis=tool_axis)
    assert np.abs(ev["final_pos"] - pos).max() <= fk_pos_tol
    assert np.abs(ev["final_axis"] - axis).max() <= fk_rot_tol
    r = Rotation.from_matrix(ev["mat"]).as_quat()[:, [3, 0, 1, 2]]
    dq = np.minimum(np.abs(r - quat).max(axis=1), np.abs(r + quat).max(axis=1))
    assert dq.max() <= fk_rot_tol
    lo, hi = oracle_model.jnt_range[:7, 0], oracle_model.jnt_range[:7, 1]
    assert (qs[1:] >= lo).all() and (qs[1:] <= hi).all()
    if L > 1:
        step = np.linalg.norm(np.diff(pos, axis=0), axis=1)
        turn = move_axis_oracle.axis_angle(axis[1:], axis[:-1])
        assert step.max() <= STEP + 2 * IK_POS_THRESH + fk_pos_tol
        assert turn.max() <= ROT_STEP + 2 * IK_ROT_THRESH + fk_rot_tol
    if plan["status"] == 0:
        g = np.asarray(goal_axis) / np.linalg.norm(goal_axis)
        assert np.linalg.norm(pos[-1] - goal_pos) <= POS_THRESH + fk_pos_tol
        assert move_axis_oracle.axis_angle(axis[-1], g) <= ROT_THRESH + fk_rot_tol


@pytest.fixture(scope="module")
def workload_plans(oracle_model, oracle_chain):
    qs, gp, ga = axis_workload(oracle_model, oracle_chain, 256)
    return gp, ga, [move_axis_oracle.plan_axis(oracle_model, qs[k], gp[k], ga[k]) for k in range(len(qs))]


def test_workload_plans_hold_the_invariants(oracle_model, oracle_chain, workload_plans):
    gp, ga, plans = workload_plans
    for k, plan in enumerate(plans):
        check_invariants(oracle_model, oracle_chain, plan, gp[k], ga[k], 1e-12, 1e-9)
        np.testing.assert_array_equal(plan["q_final"], plan["q_traj"][-1])
    status = np.array([p["status"] for p in plans])
    ok = float((status == 0).mean())
    print(f"axis planner statement: OK rate {ok:.4f} on 256 W1 moves, "
          f"mean points {np.mean([len(p['pos_traj']) for p in plans]):.1f}")
    assert ok >= 0.95


def _rotvec_aim(R, g, h, theta, tool_axis=Z):
    """The aim axis from a second source: a rotated by h theta about the solver's tilt direction n (scipy)."""
    a, _, _, th, nv = axis_ik_oracle._axis_error(R[None], axis_ik_oracle.tool_basis(tool_axis), g[None])
    assert abs(th[0] - theta) <= 1e-14  # np.linalg.norm and np.arctan2 against the solver's scalar order
    return Rotation.from_rotvec(h * theta * nv[0]).apply(a[0])


def test_aim_rule_against_a_rotation_about_the_tilt_direction(oracle_model, oracle_chain):
    qs, gp, ga = axis_workload(oracle_model, oracle_chain, 4, seed=7)
    rounds = 0
    for k in range(len(qs)):
        trace = []
        move_axis_oracle.plan_axis(oracle_model, qs[k], gp[k], ga[k], trace=trace)
        for R, g, h, theta, aim in trace:
            np.testing.assert_allclose(aim, _rotvec_aim(R, g, h, theta), rtol=0, atol=1e-12)
            rounds += 1
    assert rounds > 20


def _antiparallel_start(oracle_chain):
    """A start near NEUTRAL whose tool axis a normalises to itself exactly, so that g = -a gives a x g == 0."""
    rng = np.random.default_rng(0)
    for _ in range(200):
        q = NEUTRAL + rng.uniform(-0.05, 0.05, 7)
        ev = axis_ik_oracle.axis_eval_batch(oracle_chain, q[None], np.zeros(3), np.array([0.0, 0.0, 1.0]))
        a = ev["final_axis"][0]
        if math.sqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2]) == 1.0:
            return q, ev["final_pos"][0], a
    raise AssertionError("no start with a unit tool axis found")


def test_exactly_antiparallel_goal_turns_toward_minus_b2(oracle_model, oracle_chain):
    """s == 0 and a.g < 0: theta = pi and the aim turns a toward -b2, as the solver's own fallback n = b1 does."""
    q, p0, a = _antiparallel_start(oracle_chain)
    trace = []
    plan = move_axis_oracle.plan_axis(oracle_model, q, p0, -a, trace=trace, max_traj_points=3)
    R, g, h, theta, aim = trace[0]
    assert theta == math.pi and move_axis_oracle.tilt(R @ np.array(Z), g)[0] == 0.0
    _, _, u2 = axis_ik_oracle.tool_basis(Z)
    want = math.cos(h * math.pi) * a - math.sin(h * math.pi) * (R @ u2)
    np.testing.assert_allclose(aim, want / np.linalg.norm(want), rtol=0, atol=1e-15)
    np.testing.assert_allclose(aim, _rotvec_aim(R, g, h, theta), rtol=0, atol=1e-12)
    assert abs(h * theta - ROT_STEP) < 1e-15  # dist == 0: the rotation alone sets the step
    assert len(plan["pos_traj"]) > 1  # the first turn is solved


def test_tilt_only_move(oracle_model, oracle_chain):
    """60 degrees of tilt at a fixed position: at least ceil((pi/3) / rot_step) points, the position held within the
    IK tolerances of the fractional aims."""
    p0, a0, R0 = neutral_frame(oracle_chain)
    g = Rotation.from_rotvec(math.pi / 3 * R0[:, 0]).apply(a0)
    plan = move_axis_oracle.plan_axis(oracle_model, NEUTRAL, p0, g)
    assert plan["status"] == 0
    assert len(plan["pos_traj"]) >= math.ceil((math.pi / 3) / ROT_STEP)
    assert np.linalg.norm(plan["pos_traj"] - p0, axis=1).max() <= POS_THRESH + 2 * IK_POS_THRESH


def test_translation_only_move(oracle_model, oracle_chain):
    """A move with the start axis as its goal axis keeps it within the IK's tolerance along the path."""
    p0, a0, _ = neutral_frame(oracle_chain)
    goal = p0 + np.array([0.1, 0.15, -0.1])
    plan = move_axis_oracle.plan_axis(oracle_model, NEUTRAL, goal, a0)
    assert plan["status"] == 0 and len(plan["pos_traj"]) >= math.ceil(np.linalg.norm(goal - p0) / STEP)
    assert move_axis_oracle.axis_angle(plan["axis_traj"], a0).max() <= ROT_THRESH


@pytest.mark.parametrize("goal_pos, goal_axis", [
    ((np.nan, 0.0, 0.5), (0.0, 0.0, -1.0)),
    ((1.0, np.inf, 0.5), (0.0, 0.0, -1.0)),
    ((0.5, 0.0, 0.5), (np.nan, 0.0, -1.0)),
    ((0.5, 0.0, 0.5), (0.0, -np.inf, 0.0)),
    ((0.5, 0.0, 0.5), (0.0, 0.0, 0.0)),
])
def test_broken_goal_ends_at_once(oracle_model, goal_pos, goal_axis):
    plan = move_axis_oracle.plan_axis(oracle_model, NEUTRAL, goal_pos, goal_axis)
    assert plan["status"] == move_axis_oracle.BROKE and len(plan["pos_traj"]) == 1 and plan["n_solves"] == 0


def test_unreachable_goal_caps_and_failed_solves_break(oracle_model, oracle_chain):
    """An unreachable position creeps along the workspace boundary until max_traj_points; a small max_traj_points caps
    with max_traj_points + 1 points; solves that cannot converge (max_iters = 0) end the first round in BROKE."""
    p0, a0, _ = neutral_frame(oracle_chain)
    far = move_axis_oracle.plan_axis(oracle_model, NEUTRAL, (2.0, 0.0, 0.5), a0)
    assert far["status"] == move_axis_oracle.CAPPED and len(far["pos_traj"]) == MAX_POINTS + 1
    assert MAX_POINTS <= far["n_solves"] <= 3 * MAX_POINTS
    capped = move_axis_oracle.plan_axis(oracle_model, NEUTRAL, p0 + np.array([0.2, 0.0, 0.0]), a0, max_traj_points=5)
    assert capped["status"] == move_axis_oracle.CAPPED and len(capped["pos_traj"]) == 6
    broke = move_axis_oracle.plan_axis(oracle_model, NEUTRAL, p0 + np.array([0.2, 0.0, 0.0]), a0, max_iters=0)
    assert broke["status"] == move_axis_oracle.BROKE and len(broke["pos_traj"]) == 1 and broke["n_solves"] == 3


def test_oblique_tool_axis(oracle_model, oracle_chain):
    """The tool axis (1, 1, 1): W1 plans for that axis hold the invariants, with axis_traj = R t for t = (1,1,1)/sqrt 3."""
    qs, gp, ga = axis_workload(oracle_model, oracle_chain, 16, seed=5, tool_axis=OBLIQUE)
    ok = 0
    for k in range(len(qs)):
        plan = move_axis_oracle.plan_axis(oracle_model, qs[k], gp[k], ga[k], tool_axis=OBLIQUE)
        check_invariants(oracle_model, oracle_chain, plan, gp[k], ga[k], 1e-12, 1e-9, tool_axis=OBLIQUE)
        ok += plan["status"] == 0
    assert ok >= 15


@pytest.mark.parametrize("tool_axis", [(0.0, 0.0, 0.0), (np.nan, 0.0, 1.0), (0.0, np.inf, 0.0)])
def test_degenerate_tool_axis_raises(oracle_model, tool_axis):
    with pytest.raises(ValueError):
        move_axis_oracle.plan_axis(oracle_model, NEUTRAL, (0.5, 0.0, 0.5), (0.0, 0.0, -1.0), tool_axis=tool_axis)

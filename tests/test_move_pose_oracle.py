"""CPU checks of the pose-mode move planner's FP64 statement (oracle/move_pose_oracle.py).

Workload: synthetic.reachable_pose_move_envs - start near NEUTRAL, goal pose (FK(q*), quat(q*)) with q* = NEUTRAL
+- 0.6 rad clipped to the limits.  Default planner and IK parameters throughout."""
import math

import numpy as np
import pytest
import torch

from conftest import NEUTRAL
from mujoco_panda_pnp_b200 import synthetic
from oracle import mj_oracle, move_pose_oracle, pose_ik_oracle

IK_POS_THRESH, IK_ROT_THRESH = 1e-3, 1e-2
POS_THRESH, ROT_THRESH, STEP, ROT_STEP, MAX_POINTS = 0.01, 0.05, 0.01, 0.05, 200


def pose_workload(oracle_model, oracle_chain, n, seed=0):
    """(q_start[N,7], goal_pos[N,3], goal_quat[N,4]) of reachable_pose_move_envs, FK by the C restatement."""
    lo, hi = oracle_model.jnt_range[:7, 0], oracle_model.jnt_range[:7, 1]
    e = synthetic.reachable_pose_move_envs(n, lo, hi, seed=seed, dtype=torch.float64)
    ev = pose_ik_oracle.pose_eval_batch(oracle_chain, e["q_goal"].numpy(), np.zeros(3), np.array([1.0, 0.0, 0.0, 0.0]))
    return e["q_start"].numpy(), ev["final_pos"], ev["final_quat"]


def neutral_pose(oracle_chain):
    ev = pose_ik_oracle.pose_eval_batch(oracle_chain, NEUTRAL[None], np.zeros(3), np.array([1.0, 0.0, 0.0, 0.0]))
    return ev["final_pos"][0], ev["final_quat"][0]


def check_invariants(oracle_model, oracle_chain, plan, goal_pos, goal_quat, fk_pos_tol, fk_rot_tol):
    """What every plan of the statement satisfies (also applied to the GPU's FP32 plans, with FK tolerances): every
    point is FK(q) of its joints - position to fk_pos_tol, quaternion components (up to sign) to fk_rot_tol / 2."""
    pos, quat, qs = plan["pos_traj"], plan["quat_traj"], plan["q_traj"]
    L = len(pos)
    assert 1 <= L <= MAX_POINTS + 1 and plan["n_solves"] <= 3 * MAX_POINTS
    ev = pose_ik_oracle.pose_eval_batch(oracle_chain, qs, np.zeros(3), np.array([1.0, 0.0, 0.0, 0.0]))
    assert np.abs(ev["final_pos"] - pos).max() <= fk_pos_tol
    dq = np.minimum(np.abs(ev["final_quat"] - quat).max(axis=1), np.abs(ev["final_quat"] + quat).max(axis=1))
    assert dq.max() <= fk_rot_tol / 2
    lo, hi = oracle_model.jnt_range[:7, 0], oracle_model.jnt_range[:7, 1]
    assert (qs[1:] >= lo).all() and (qs[1:] <= hi).all()
    if L > 1:
        step = np.linalg.norm(np.diff(pos, axis=0), axis=1)
        turn = move_pose_oracle.quat_angle(quat[1:], quat[:-1])
        assert step.max() <= STEP + 2 * IK_POS_THRESH + fk_pos_tol
        assert turn.max() <= ROT_STEP + 2 * IK_ROT_THRESH + fk_rot_tol
    if plan["status"] == 0:
        gq = np.asarray(goal_quat) / np.linalg.norm(goal_quat)
        assert np.linalg.norm(pos[-1] - goal_pos) <= POS_THRESH + fk_pos_tol
        assert move_pose_oracle.quat_angle(quat[-1], gq) <= ROT_THRESH + fk_rot_tol


@pytest.fixture(scope="module")
def workload_plans(oracle_model, oracle_chain):
    qs, gp, gq = pose_workload(oracle_model, oracle_chain, 256)
    return gp, gq, [move_pose_oracle.plan_pose(oracle_model, qs[k], gp[k], gq[k]) for k in range(len(qs))]


def test_workload_plans_hold_the_invariants(oracle_model, oracle_chain, workload_plans):
    gp, gq, plans = workload_plans
    for k, plan in enumerate(plans):
        check_invariants(oracle_model, oracle_chain, plan, gp[k], gq[k], 1e-12, 2e-12)
        np.testing.assert_array_equal(plan["q_final"], plan["q_traj"][-1])
    status = np.array([p["status"] for p in plans])
    ok = float((status == 0).mean())
    print(f"pose planner statement: OK rate {ok:.4f} on 256 reachable pose moves, "
          f"mean points {np.mean([len(p['pos_traj']) for p in plans]):.1f}")
    assert ok >= 0.95  # 1.0 measured (256 of 256)


def test_rotation_only_move(oracle_model, oracle_chain):
    """90 degrees about world z at a fixed position: at least ceil((pi/2) / rot_step) points, and the held position
    drifts by 9.8e-3 m at most along the path (measured; each solve lands anywhere inside its tolerance and the aim
    pulls back only by the fraction f)."""
    p0, r0 = neutral_pose(oracle_chain)
    qz = np.array([math.cos(math.pi / 4), 0.0, 0.0, math.sin(math.pi / 4)])
    plan = move_pose_oracle.plan_pose(oracle_model, NEUTRAL, p0, mj_oracle.mju_mulQuat(qz, r0))
    assert plan["status"] == 0
    assert len(plan["pos_traj"]) >= math.ceil((math.pi / 2) / ROT_STEP)
    drift = np.linalg.norm(plan["pos_traj"] - p0, axis=1).max()
    assert drift <= 2 * 9.8e-3


def test_translation_only_move(oracle_model, oracle_chain):
    """A move with the start orientation as its goal keeps it: the orientation drifts by 1.0e-3 rad at most along the
    path (measured)."""
    p0, r0 = neutral_pose(oracle_chain)
    goal = p0 + np.array([0.1, 0.15, -0.1])
    plan = move_pose_oracle.plan_pose(oracle_model, NEUTRAL, goal, r0)
    assert plan["status"] == 0 and len(plan["pos_traj"]) >= math.ceil(np.linalg.norm(goal - p0) / STEP)
    drift = move_pose_oracle.quat_angle(plan["quat_traj"], r0).max()
    assert drift <= 2 * 1.0e-3


@pytest.mark.parametrize("goal_pos, goal_quat", [
    ((np.nan, 0.0, 0.5), (1.0, 0.0, 0.0, 0.0)),
    ((1.0, 0.0, 0.5), (np.nan, 0.0, 0.0, 0.0)),
    ((1.0, 0.0, np.inf), (1.0, 0.0, 0.0, 0.0)),
    ((1.0, 0.0, 0.5), (0.0, 0.0, 0.0, 0.0)),
])
def test_broken_goal_ends_at_once(oracle_model, goal_pos, goal_quat):
    plan = move_pose_oracle.plan_pose(oracle_model, NEUTRAL, goal_pos, goal_quat)
    assert plan["status"] == move_pose_oracle.BROKE and len(plan["pos_traj"]) == 1 and plan["n_solves"] == 0


def test_unreachable_goal_caps_and_failed_solves_break(oracle_model, oracle_chain):
    """Every plan terminates without a round bound.  An unreachable goal creeps along the workspace boundary on
    shortened steps (rejected full steps included) until max_traj_points; a small max_traj_points caps with
    max_traj_points + 1 points; solves that cannot converge (max_iters = 0) end the first round in BROKE."""
    p0, r0 = neutral_pose(oracle_chain)
    far = move_pose_oracle.plan_pose(oracle_model, NEUTRAL, (2.0, 0.0, 0.5), r0)
    assert far["status"] == move_pose_oracle.CAPPED and len(far["pos_traj"]) == MAX_POINTS + 1
    assert MAX_POINTS < far["n_solves"] <= 3 * MAX_POINTS
    capped = move_pose_oracle.plan_pose(oracle_model, NEUTRAL, p0 + np.array([0.2, 0.0, 0.0]), r0, max_traj_points=5)
    assert capped["status"] == move_pose_oracle.CAPPED and len(capped["pos_traj"]) == 6
    broke = move_pose_oracle.plan_pose(oracle_model, NEUTRAL, p0 + np.array([0.2, 0.0, 0.0]), r0, max_iters=0)
    assert broke["status"] == move_pose_oracle.BROKE and len(broke["pos_traj"]) == 1 and broke["n_solves"] == 3

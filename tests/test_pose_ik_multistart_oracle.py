"""CPU checks of the multi-start pose IK statement and of the default seed table on workspace poses.

W-cold: q* ~ U(joint limits), target (FK(q*), mat2Quat(R(q*))) - every target is reachable - solved from NEUTRAL."""
import numpy as np
import torch

from conftest import NEUTRAL
from mujoco_panda_pnp_b200 import engine
from oracle import mj_oracle, pose_ik_oracle


def solve_pose_multistart(model, data, target_pos, target_quat, q_init, seeds, **kw):
    """Scalar FP64 statement of the multi-start pose solve (pnp_ik_pose_solve_multistart_*): attempt 0 is
    ``pose_ik_oracle.solve_pose`` from q_init; when it is not a success, attempts 1..K solve the same pose from
    seeds[k - 1].  Returns (attempt, result) of the first successful attempt in order 0..K, or of attempt 0 when none
    succeeds."""
    r0 = pose_ik_oracle.solve_pose(model, data, target_pos, target_quat, q_init, **kw)
    if r0["success"]:
        return 0, r0
    for k, s in enumerate(np.asarray(seeds, dtype=np.float64).reshape(-1, 7)):
        r = pose_ik_oracle.solve_pose(model, data, target_pos, target_quat, s, **kw)
        if r["success"]:
            return k + 1, r
    return 0, r0


def solve_pose_multistart_batch(chain, target_pos, target_quat, q_init, seeds, **kw):
    """The same statement over N queries (pose_ik_oracle.solve_pose_batch): solve from q_init, then re-solve the
    still-failed queries from each seed in turn, keeping the first success.  ``kw``: solve_pose_batch's parameters.
    Returns solve_pose_batch's arrays plus attempt[N] (0 = q_init, k = seeds[k - 1])."""
    tp = np.ascontiguousarray(target_pos, dtype=np.float64).reshape(-1, 3)
    tq = np.asarray(target_quat, dtype=np.float64).reshape(-1, 4)
    out = pose_ik_oracle.solve_pose_batch(chain, tp, tq, q_init, **kw)
    out["attempt"] = np.zeros(len(tp), dtype=np.int64)
    left = np.nonzero(~out["success"])[0]
    for k, s in enumerate(np.asarray(seeds, dtype=np.float64).reshape(-1, 7)):
        if not len(left):
            break
        rk = pose_ik_oracle.solve_pose_batch(chain, tp[left], tq[left], s, **kw)
        ok = rk["success"]
        for key in rk:
            out[key][left[ok]] = rk[key][ok]
        out["attempt"][left[ok]] = k + 1
        left = left[~ok]
    return out


def workspace(chain, n, seed=0):
    """W targets: (final_pos[N,3], final_quat[N,4]) of q* ~ U(joint limits) from np.random.default_rng(seed)."""
    rng = np.random.default_rng(seed)
    q_star = rng.uniform(np.array(chain.lower[:]), np.array(chain.upper[:]), (n, 7))
    ev = pose_ik_oracle.pose_eval_batch(chain, q_star, np.zeros(3), np.array([1.0, 0.0, 0.0, 0.0]))
    return ev["final_pos"], ev["final_quat"]


def test_batched_statement_matches_scalar_restarts(oracle_model, oracle_chain):
    """W-cold targets attempt 0 solves, ones a restart rescues, ones no seed rescues, and unreachable poses: the
    batched statement picks the attempt the scalar one picks, with the same iterations and flags."""
    pos, quat = workspace(oracle_chain, 512, seed=3)
    seeds = engine.ik_restart_seeds(4, device="cpu", dtype=torch.float64).numpy()
    full = solve_pose_multistart_batch(oracle_chain, pos, quat, NEUTRAL, seeds)
    pick = np.concatenate([np.nonzero((full["attempt"] == 0) & full["success"])[0][:6],
                           np.nonzero(full["attempt"] > 0)[0][:6], np.nonzero(~full["success"])[0][:2]])
    far_pos = np.array([[2.5, 0.0, 0.5], [0.0, 0.0, 3.0]])
    pos_s = np.concatenate([pos[pick], far_pos])
    quat_s = np.concatenate([quat[pick], quat[:2]])
    got = solve_pose_multistart_batch(oracle_chain, pos_s, quat_s, NEUTRAL, seeds)
    assert (got["attempt"] > 0).sum() >= 4 and not got["success"][-2:].any()
    d = mj_oracle.MjData(oracle_model)
    for i in range(len(pos_s)):
        k, w = solve_pose_multistart(oracle_model, d, pos_s[i], quat_s[i], NEUTRAL, seeds)
        assert k == got["attempt"][i], i
        assert w["iterations"] == got["iterations"][i] and w["success"] == got["success"][i], i
        assert w["converged"] == got["converged"][i], i
        if w["converged"]:  # (a 100-pass walk that never converges amplifies the two statements' rounding differences)
            np.testing.assert_allclose(w["q"], got["q"][i], atol=1e-9)
            np.testing.assert_allclose(w["final_pos"], got["final_pos"][i], atol=1e-9)


def test_default_seed_table_rescues_the_w_cold_failures(oracle_chain):
    """4096 W-cold targets: engine.ik_restart_seeds(8) must rescue at least 93 % of the queries attempt 0 fails on
    (these targets: 1 104 failures, 1 057 rescued, 95.7 %)."""
    pos, quat = workspace(oracle_chain, 4096, seed=0)
    seeds = engine.ik_restart_seeds(8, device="cpu", dtype=torch.float64).numpy()
    out = solve_pose_multistart_batch(oracle_chain, pos, quat, NEUTRAL, seeds)
    rescued = int((out["attempt"] > 0).sum())
    failed0 = rescued + int((~out["success"]).sum())
    assert 0.2 * len(pos) < failed0 < 0.35 * len(pos)  # about a quarter of W-cold fails from NEUTRAL
    assert rescued >= 0.93 * failed0, (rescued, failed0)

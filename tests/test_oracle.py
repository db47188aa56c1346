"""The oracle against the reference's golden vectors (CPU only).

tests/golden/*.npz were produced by oracle/gen_golden.py by running the reference's OWN
ik_solver.py / panda_env.py (third-party natives stubbed).  These tests pin the restatements
(oracle/*.py and oracle/c/pnp_oracle.c) to those outputs before anything trusts them.
"""
import json
import os

import numpy as np

from conftest import GOLDEN, NEUTRAL
from oracle import c_oracle, ik_oracle, mj_oracle, reward_oracle


# ------------------------------------------------------------------ FK / Jacobian
def test_fk_golden_and_home_wpt(oracle_model, golden_fk):
    d = mj_oracle.MjData(oracle_model)
    for k in range(len(golden_fk["q"])):
        pos, mat, quat, jac = ik_oracle.fk_site(oracle_model, d, golden_fk["q"][k])
        np.testing.assert_array_equal(pos, golden_fk["pos"][k])
        np.testing.assert_array_equal(jac, golden_fk["jac"][k])
        np.testing.assert_array_equal(quat, golden_fk["quat"][k])
    # the one real-MuJoCo number in the reference (execute_pnp.py:38): printed to 8 decimals
    assert np.abs(golden_fk["pos"][0] - golden_fk["home_wpt"]).max() < 5e-9


def test_jacobian_matches_central_differences(oracle_model):
    d = mj_oracle.MjData(oracle_model)
    rng = np.random.default_rng(3)
    lo, hi = oracle_model.jnt_range[:7, 0], oracle_model.jnt_range[:7, 1]
    h = 1e-6
    for _ in range(5):
        q = rng.uniform(lo, hi)
        _, _, _, jac = ik_oracle.fk_site(oracle_model, d, q)
        for j in range(7):
            dq = np.zeros(7)
            dq[j] = h
            pp, mp, _, _ = ik_oracle.fk_site(oracle_model, d, q + dq)
            pm, mm, _, _ = ik_oracle.fk_site(oracle_model, d, q - dq)
            np.testing.assert_allclose((pp - pm) / (2 * h), jac[:3, j], atol=2e-9)
            w = (mp - mm) / (2 * h) @ (0.5 * (mp + mm)).T  # skew(omega)
            np.testing.assert_allclose([w[2, 1], w[0, 2], w[1, 0]], jac[3:, j], atol=2e-9)


def test_mat2quat_branches():
    rng = np.random.default_rng(0)
    for k in range(200):
        q = rng.normal(size=4)
        if k % 4 == 1:
            q[0] = 0.01 * q[0]  # force the trace <= 0 branches
        q /= np.linalg.norm(q)
        out = np.empty(4)
        mj_oracle.mju_mat2Quat(out, mj_oracle.mju_quat2Mat(q).reshape(9))
        assert min(np.abs(out - q).max(), np.abs(out + q).max()) < 1e-12


def test_c_oracle_fk_matches_numpy_oracle(oracle_chain, golden_fk):
    pos, mat, jac = c_oracle.fk_jac(oracle_chain, golden_fk["q"])
    np.testing.assert_allclose(pos, golden_fk["pos"], atol=1e-14)
    np.testing.assert_allclose(mat, golden_fk["mat"], atol=1e-14)
    np.testing.assert_allclose(jac, golden_fk["jac"], atol=1e-14)


# ------------------------------------------------------------------ IK
def _case_kwargs(g, k):
    return dict(max_iters=int(g["max_iters"][k]), pos_thresh=float(g["pos_thresh"][k]),
                damping=float(g["damping"][k]), step_limit=float(g["step_limit"][k]))


def test_numpy_ik_oracle_is_bit_identical_to_reference_code(oracle_model, golden_ik):
    g = golden_ik
    ctl = ik_oracle.JacobianIKController(oracle_model, mj_oracle.MjData(oracle_model))
    for k in range(len(g["tag"])):
        r = ctl.solve(g["target"][k], g["q_init"][k], **_case_kwargs(g, k))
        tag = str(g["tag"][k])
        assert r.iterations == g["iterations"][k], tag
        assert r.converged == g["converged"][k] and r.success == g["success"][k], tag
        np.testing.assert_array_equal(r.q, g["q"][k], err_msg=tag)
        np.testing.assert_array_equal(r.final_pos, g["final_pos"][k], err_msg=tag)
        assert r.pos_error == g["pos_error"][k], tag
        # controller side effect (SURVEY 3.1): data mirrors the result
        np.testing.assert_array_equal(ctl.data.qpos[:7], r.q)


def test_golden_covers_the_survey_known_answers(golden_ik):
    g = golden_ik
    tags = [str(t) for t in g["tag"]]
    want = {"cfg1_cube1": 7, "cfg1_cube2": 11, "cfg1_cube3": 8, "cfg1_home": 1, "ik_test": 10}  # SURVEY App. C
    for tag, iters in want.items():
        k = tags.index(tag)
        assert g["iterations"][k] == iters and g["converged"][k]
    k = tags.index("cfg1_cube1")
    np.testing.assert_allclose(g["q"][k], [0, 0.4737271, 0, -1.4312119, 0, 2.63849197, 0.79], atol=5e-8)
    np.testing.assert_allclose(g["final_pos"][k], [1.41469724, 0, 0.73000737], atol=5e-9)
    # loop-exhaustion semantics (App. D.1): 7 iterations needed -> max_iters=6 is not converged,
    # max_iters=7 converges on the last (test-only) pass
    assert not g["converged"][tags.index("max_iters_6_short")] and g["iterations"][tags.index("max_iters_6_short")] == 6
    assert g["converged"][tags.index("max_iters_7_exact")] and g["iterations"][tags.index("max_iters_7_exact")] == 7
    assert not g["converged"][tags.index("unreachable")] and g["iterations"][tags.index("unreachable")] == 100


def test_c_ik_oracle_matches_reference_golden(oracle_chain, golden_ik):
    g = golden_ik
    for k in range(len(g["tag"])):
        r = c_oracle.ik_solve(oracle_chain, g["target"][k][None], g["q_init"][k], **_case_kwargs(g, k))
        tag = str(g["tag"][k])
        assert r["iterations"][0] == g["iterations"][k], tag
        assert r["converged"][0] == g["converged"][k] and r["success"][0] == g["success"][k], tag
        np.testing.assert_allclose(r["q"][0], g["q"][k], atol=1e-9, err_msg=tag)
        np.testing.assert_allclose(r["final_pos"][0], g["final_pos"][k], atol=1e-9, err_msg=tag)


def test_c_ik_oracle_threads_and_per_query_init(oracle_chain):
    rng = np.random.default_rng(11)
    q0 = np.clip(NEUTRAL + rng.uniform(-0.2, 0.2, (257, 7)), np.array(oracle_chain.lower[:]), np.array(oracle_chain.upper[:]))
    tg, _, _ = c_oracle.fk_jac(oracle_chain, q0 + rng.uniform(-0.05, 0.05, q0.shape))
    a = c_oracle.ik_solve(oracle_chain, tg, q0, nthreads=1)
    b = c_oracle.ik_solve(oracle_chain, tg, q0, nthreads=5)
    for k in a:
        np.testing.assert_array_equal(a[k], b[k])
    assert a["converged"].all() and a["iterations"].max() <= 6


# ------------------------------------------------------------------ reward
_ROW_KEYS = ("achieved_goal", "desired_goal", "ee_pos", "ee_quat", "fingers_width", "task_index")


def test_reward_constants(golden_reward):
    np.testing.assert_array_equal(reward_oracle.HORIZONTAL_QUAT, golden_reward["horizontal_quat"])
    np.testing.assert_array_equal(reward_oracle.VERTICAL_QUAT, golden_reward["vertical_quat"])
    assert reward_oracle.HORIZONTAL_QUAT[0] == 0.7071067811865476 and reward_oracle.HORIZONTAL_QUAT[1] == -0.7071067811865475


def test_numpy_reward_oracle_bit_exact_vs_reference_code(golden_reward):
    g = golden_reward
    rows = [g[k] for k in _ROW_KEYS]
    for rt in ("dense", "sparse"):
        got = reward_oracle.compute_reward_rows(*rows, reward_type=rt)
        np.testing.assert_array_equal(got.view(np.uint32), g[f"reward_{rt}"].view(np.uint32))
    succ = np.array([reward_oracle.is_success(a, d) for a, d in zip(g["achieved_goal"], g["desired_goal"])])
    np.testing.assert_array_equal(succ, g["is_success"])
    np.testing.assert_array_equal(reward_oracle.goal_distance(g["achieved_goal"], g["desired_goal"]), g["goal_distance"])


def test_c_reward_oracle_bit_exact_vs_reference_code(oracle_chain, golden_reward):
    g = golden_reward
    rows = [g[k] for k in _ROW_KEYS]
    for rt in ("dense", "sparse"):
        got, succ = c_oracle.reward(*rows, reward_type=rt, nthreads=3)
        np.testing.assert_array_equal(got.view(np.uint32), g[f"reward_{rt}"].view(np.uint32))
        np.testing.assert_array_equal(succ, g["is_success"])


def test_reward_known_answers(golden_reward):
    g = golden_reward
    # SURVEY App. C rows 0..5; row 0 is the real old_reward of the reference's VecNormalize pickle
    bits = [0xBD591687, 0xBCBC6A7F, 0x40DF9581, 0x40E4EAD6, 0x4182900B, 0x411F26E9]
    assert [int(b) for b in g["reward_dense"][:6].view(np.uint32)] == bits
    sparse = g["reward_sparse"][:6].view(np.uint32)
    assert [int(b) for b in sparse] == [0xBF800000] * 4 + [0x80000000] * 2  # -1.0 ... and -0.0 when placed
    with open(os.path.join(GOLDEN, "vecnormalize_stats.json")) as fh:
        stats = json.load(fh)
    assert stats["old_reward_bits"] == ["0xbd591687"] * 4
    # every branch is populated in the fixture
    d = g["reward_dense"]
    assert (d > 9).sum() > 100 and ((d > 1.5) & (d < 5)).sum() > 10 and (d < 0).sum() > 1000
    adj = reward_oracle.threshold_adjacent(g["achieved_goal"], g["desired_goal"], g["ee_pos"])
    assert adj.sum() >= 500


# ------------------------------------------------------------------ _get_obs
def test_obs_oracle_bit_identical_to_reference_code(oracle_model):
    from oracle import obs_oracle

    g = np.load(os.path.join(GOLDEN, "obs_reference_golden.npz"))
    data = mj_oracle.MjData(oracle_model)
    for i in range(len(g["q_arm"])):
        name = f"cube{int(g['obj_index'][i]) + 1}"
        obs_oracle.set_state(oracle_model, data, g["q_arm"][i], g["qvel_arm"][i], g["fingers"][i], name,
                             g["obj_pos"][i], g["obj_quat"][i], g["obj_vel"][i])
        o = obs_oracle.get_obs(oracle_model, data, name, g["goal"][i], dt=float(g["dt"]))
        np.testing.assert_array_equal(o["observation"], g["observation"][i])
        np.testing.assert_array_equal(o["achieved_goal"], g["achieved_goal"][i])
        np.testing.assert_array_equal(o["desired_goal"], g["desired_goal"][i])
    obs = g["observation"]
    assert obs.shape == (256, 19)
    # layout pins (panda_env.py:297): width = f1 + f2 at [6], obj_pos at [7:10] = achieved_goal
    np.testing.assert_array_equal(obs[:, 6], g["fingers"].sum(axis=1))
    np.testing.assert_array_equal(obs[:, 7:10], g["achieved_goal"])
    np.testing.assert_array_equal(obs[:, 13:16], g["obj_vel"][:, :3] * 0.05)
    # ee_vel = jacp @ qvel * dt agrees with a finite difference of FK along qvel
    h = 1e-7
    p0 = ik_oracle.fk_site(oracle_model, data, g["q_arm"][9])[0]
    p1 = ik_oracle.fk_site(oracle_model, data, g["q_arm"][9] + h * g["qvel_arm"][9])[0]
    np.testing.assert_allclose((p1 - p0) / h * 0.05, obs[9, 3:6], atol=1e-7)
    # gimbal rows went through mat2euler's degenerate branch
    assert abs(abs(obs[0, 11]) - np.pi / 2) < 1e-6 and obs[0, 10] == 0.0


# ------------------------------------------------------------------ MoveIKSkill planner
def test_move_planner_oracles_match_reference_code(oracle_model, oracle_chain):
    """tests/golden/move_reference_golden.npz = pos_traj of the reference's own MoveIKSkill.reset
    (skills/move.py:76-191).  The NumPy restatement must be bit-identical on the short cases, the C
    restatement within 1e-9 on all (incl. the ones whose IK solves fail on the way)."""
    from oracle import move_oracle

    g = np.load(os.path.join(GOLDEN, "move_reference_golden.npz"))
    n = len(g["traj_len"])
    assert n >= 18 and g["traj_len"].max() == 202 and g["traj_len"].min() == 1
    r = c_oracle.move_plan(oracle_chain, g["q_start"], g["target"], traj_cap=g["traj"].shape[1], nthreads=4)
    np.testing.assert_array_equal(r["traj_len"], g["traj_len"])
    assert (r["status"] == 0).all()
    for k in range(n):
        L = int(g["traj_len"][k])
        np.testing.assert_allclose(r["traj"][k, :L], g["traj"][k, :L], atol=1e-9)
    assert (r["n_solves"] > r["traj_len"]).sum() >= 4  # the failing-solve cases really failed on the way
    for k in range(6):  # NumPy restatement: bit-identical (kept to the short cases for run time)
        o = move_oracle.plan(oracle_model, g["q_start"][k], g["target"][k])
        np.testing.assert_array_equal(o["pos_traj"], g["traj"][k, : int(g["traj_len"][k])])


def test_move_planner_never_terminates_on_unreachable_targets_without_a_bound(oracle_chain):
    """Reference quirk: for an unreachable target fallback strategy 1 keeps succeeding with ever
    smaller steps and never advances point_count; only an explicit bound stops the loop."""
    r = c_oracle.move_plan(oracle_chain, NEUTRAL[None], np.array([[2.0, 0.0, 0.5]]), max_outer=400, traj_cap=64)
    assert r["status"][0] & 2 and r["status"][0] & 4 and r["traj_len"][0] > 200


def test_pose_ik_statement_agrees_with_an_independent_formulation(oracle_model):
    """oracle/pose_ik_oracle.py states the pose-mode extension (there is no reference code for it, SURVEY 8f-4).  A
    second, independently written formulation must walk the same iterates: the orientation error as SciPy's rotation
    vector of R_target R_site^T (instead of mju_mat2Quat + mju_mulQuat + mju_quat2Vel) and the damped step as the
    least-squares solution of the stacked system [J; sqrt(damping) I] dq = [e; 0] (numpy.linalg.lstsq, instead of
    J^T solve(J J^T + damping I, e)) - two-source evidence for the semantics the GPU kernel is tested against."""
    from scipy.spatial.transform import Rotation

    from oracle import pose_ik_oracle

    model = oracle_model
    sid = model.site("ee_center_site").id
    lower, upper = model.jnt_range[:7, 0], model.jnt_range[:7, 1]
    rng = np.random.default_rng(11)
    d1, d2 = mj_oracle.MjData(model), mj_oracle.MjData(model)
    n_conv = 0
    for case in range(12):
        q_goal = np.clip(NEUTRAL + rng.uniform(-0.5, 0.5, 7), lower, upper)
        p_t, _, quat_t, _ = ik_oracle.fk_site(model, d1, q_goal)
        want = pose_ik_oracle.solve_pose(model, d1, p_t, quat_t, NEUTRAL, damping=1e-2, rot_weight=0.7)
        # ---- independent loop ----------------------------------------------------------------------------
        r_t = Rotation.from_quat([quat_t[1], quat_t[2], quat_t[3], quat_t[0]])  # SciPy is xyzw
        q = NEUTRAL.copy()
        converged, iterations = False, 0
        for i in range(100 + 1):
            d2.qpos[:7] = q
            mj_oracle.mj_forward(model, d2)
            p = d2.site_xpos[sid].copy()
            r_c = Rotation.from_matrix(np.asarray(d2.site_xmat[sid]).reshape(3, 3))
            rv = (r_t * r_c.inv()).as_rotvec()  # world-frame rotation vector, angle in [0, pi]
            e_pos = p_t - p
            if i == 100:
                iterations = 100
                break
            if np.linalg.norm(e_pos) < 1e-3 and np.linalg.norm(rv) < 1e-2:
                converged, iterations = True, i + 1
                break
            jp, jr = np.zeros((3, model.nv)), np.zeros((3, model.nv))
            mj_oracle.mj_jacSite(model, d2, jp, jr, sid)
            J = np.vstack([jp[:, :7], 0.7 * jr[:, :7]])
            e = np.concatenate([e_pos, 0.7 * rv])
            A = np.vstack([J, np.sqrt(1e-2) * np.eye(7)])
            b = np.concatenate([e, np.zeros(7)])
            dq = np.linalg.lstsq(A, b, rcond=None)[0]
            q = np.clip(q + np.clip(dq, -0.1, 0.1), lower, upper)
        assert converged == want["converged"] and iterations == want["iterations"], case
        np.testing.assert_allclose(q, want["q"], atol=1e-8)
        np.testing.assert_allclose(p, want["final_pos"], atol=1e-9)
        n_conv += converged
    assert n_conv >= 10


def test_batched_pose_statement_walks_the_scalar_iterates(oracle_model, oracle_chain):
    """pose_ik_oracle.solve_pose_batch (N queries at once on c_oracle's FK, NumPy mat2Quat / mulQuat / quat2vel, one
    batched 6x6 solve) against the scalar statement solve_pose, query by query: the GPU pose tests run thousands of
    queries against the batched form, so it has to be the same statement.  Half the queries start near their target,
    half at NEUTRAL; the targets span all four mju_mat2Quat cases and a third of the quaternions are given as -q or
    scaled (the statement normalises them and the angle fold makes -q the same rotation)."""
    from oracle import pose_ik_oracle

    rng = np.random.default_rng(5)
    lo, hi = oracle_model.jnt_range[:7, 0], oracle_model.jnt_range[:7, 1]
    # draw from the workspace until each mat2Quat case has 16 targets
    qs = rng.uniform(lo, hi, (400, 7))
    ev = pose_ik_oracle.pose_eval_batch(oracle_chain, qs, np.zeros(3), np.array([1.0, 0.0, 0.0, 0.0]))
    pick = np.concatenate([np.nonzero(ev["case"] == c)[0][:16] for c in range(4)])
    assert len(pick) == 64
    q_star = qs[pick]
    pos, quat = ev["final_pos"][pick], ev["final_quat"][pick].copy()
    quat[1::3] *= -1.0
    quat[2::6] *= 7.5
    quat[5::6] *= 1e-3
    near = np.arange(64) % 2 == 0
    q_init = np.where(near[:, None], np.clip(q_star + rng.uniform(-0.3, 0.3, (64, 7)), lo, hi), NEUTRAL)
    got = pose_ik_oracle.solve_pose_batch(oracle_chain, pos, quat, q_init)
    d = mj_oracle.MjData(oracle_model)
    ties = 0
    for k in range(64):
        w = pose_ik_oracle.solve_pose(oracle_model, d, pos[k], quat[k], q_init[k])
        if got["iterations"][k] != w["iterations"]:
            ties += 1  # FK rounding of the two restatements put one of them exactly on a threshold
            continue
        assert bool(got["converged"][k]) == w["converged"] and bool(got["success"][k]) == w["success"], k
        if w["converged"]:
            np.testing.assert_allclose(got["q"][k], w["q"], atol=1e-9, err_msg=str(k))
            np.testing.assert_allclose(got["final_pos"][k], w["final_pos"], atol=1e-9, err_msg=str(k))
            np.testing.assert_allclose(got["final_quat"][k], w["final_quat"], atol=1e-9, err_msg=str(k))
            assert abs(got["pos_error"][k] - w["pos_error"]) < 1e-9 and abs(got["rot_error"][k] - w["rot_error"]) < 1e-9
    assert ties <= 1, ties
    assert got["converged"][near].all() and got["converged"][~near].mean() > 0.4
    # the single evaluation is the pass the loop makes: at q_init with max_iters = 0
    e0 = pose_ik_oracle.pose_eval_batch(oracle_chain, q_init, pos, quat)
    z = pose_ik_oracle.solve_pose_batch(oracle_chain, pos, quat, q_init, max_iters=0)
    assert (z["iterations"] == 0).all() and not z["converged"].any() and np.array_equal(z["q"], q_init)
    for key in ("final_pos", "final_quat", "pos_error", "rot_error"):
        np.testing.assert_array_equal(z[key], e0[key])
    # both hemispheres of the error quaternion occur, and -q gives the same rotation error as q
    assert (e0["err_w"] < 0).any() and (e0["err_w"] > 0).any()
    e1 = pose_ik_oracle.pose_eval_batch(oracle_chain, q_init, pos, -quat)
    np.testing.assert_allclose(e1["rot_error"], e0["rot_error"], atol=1e-12)

"""GPU parity: batched JacobianIKController.solve vs the oracle / reference golden vectors.

Tolerances (north_star): converged joint solutions must reproduce reference EE poses to
1e-4 m.  The FP64 kernel follows the reference iteration for iteration (identical iteration
counts, q within 1e-9); the FP32 kernel is the product path and is held to the stated EE
tolerance, with iteration-count flips counted and bounded."""
import numpy as np
import pytest
import torch

from conftest import NEUTRAL
from mujoco_panda_pnp_b200 import KinematicData, KinematicTree, engine, synthetic
from mujoco_panda_pnp_b200.skills import IKResult, JacobianIKController
from oracle import c_oracle, ik_oracle, mj_oracle

pytestmark = pytest.mark.gpu

EE_TOL_M = 1e-4  # north_star: converged solutions reproduce reference EE poses to 1e-4 m


@pytest.fixture(scope="module")
def tree(cuda_lib):
    t = KinematicTree.from_mjcf()
    engine.set_tree(t)
    return t


def _kw(g, k):
    return dict(max_iters=int(g["max_iters"][k]), pos_thresh=float(g["pos_thresh"][k]),
                damping=float(g["damping"][k]), step_limit=float(g["step_limit"][k]))


@pytest.mark.parametrize("kin", ["specialized", "generic"])
def test_reference_golden_fp64_is_iteration_exact(kin_model, golden_ik, kin):
    g = golden_ik
    ctl = JacobianIKController(kin_model, KinematicData(kin_model), precision="fp64", kinematics=kin)
    for k in range(len(g["tag"])):
        r = ctl.solve(g["target"][k], g["q_init"][k], **_kw(g, k))
        tag = str(g["tag"][k])
        assert isinstance(r, IKResult)
        assert r.iterations == g["iterations"][k], tag
        assert r.converged == bool(g["converged"][k]) and r.success == bool(g["success"][k]), tag
        # converged solves agree to 1e-9; the non-converged ones sit in a singular stretched-out
        # pose for ~100 steps where the reference's 1e-17 Jacobian noise is amplified to ~1e-7
        tol = 1e-9 if r.converged else 1e-6
        np.testing.assert_allclose(r.q, g["q"][k], atol=tol, err_msg=tag)
        np.testing.assert_allclose(r.final_pos, g["final_pos"][k], atol=tol, err_msg=tag)
        assert abs(r.pos_error - g["pos_error"][k]) < tol, tag


@pytest.mark.parametrize("kin", ["specialized", "generic"])
def test_reference_golden_fp32(kin_model, golden_ik, oracle_chain, kin):
    g = golden_ik
    ctl = JacobianIKController(kin_model, KinematicData(kin_model), kinematics=kin)
    flips = 0
    for k in range(len(g["tag"])):
        r = ctl.solve(g["target"][k], g["q_init"][k], **_kw(g, k))
        tag = str(g["tag"][k])
        assert r.converged == bool(g["converged"][k]), tag
        flips += int(r.iterations != g["iterations"][k])
        if r.converged and r.iterations == g["iterations"][k]:
            # same number of DLS steps -> same joint solution up to FP32 rounding
            np.testing.assert_allclose(r.q, g["q"][k], atol=2e-5, err_msg=tag)
            ee = c_oracle.fk_jac(oracle_chain, r.q[None])[0][0]
            assert np.linalg.norm(ee - g["final_pos"][k]) < EE_TOL_M, tag
        if r.converged:
            assert np.linalg.norm(r.final_pos - g["target"][k]) < g["pos_thresh"][k] + 1e-6
    assert flips <= 2, flips  # threshold-adjacent cases may take one step more or less in FP32


def test_controller_is_a_drop_in(kin_model):
    """Same attributes / side effects as the reference class (ik_solver.py:27-33, SURVEY 3.1)."""
    data = KinematicData(kin_model)
    ctl = JacobianIKController(kin_model, data)
    assert ctl.site_id == kin_model.site("ee_center_site").id
    np.testing.assert_array_equal(ctl.joint_ids, np.arange(7))
    np.testing.assert_array_equal(ctl.lower, kin_model.jnt_range[:7, 0])
    np.testing.assert_array_equal(ctl.upper, kin_model.jnt_range[:7, 1])
    assert ctl.specialized
    r = ctl.solve(np.array([1.415, 0.0, 0.73]), NEUTRAL)  # positional, defaults: move.py:128
    assert r.success and r.converged and r.iterations == 7 and r.q.shape == (7,) and r.q.dtype == np.float64
    np.testing.assert_array_equal(data.qpos[:7], r.q)
    np.testing.assert_array_equal(data.site_xpos[ctl.site_id], r.final_pos)
    assert isinstance(r.pos_error, float) and isinstance(r.iterations, int) and isinstance(r.success, bool)
    # test/ik_test.py:31-38 call pattern (keyword arguments)
    r2 = ctl.solve(target_pos=np.array([1.33843967, 0.0, 0.49740014]), q_init=NEUTRAL, max_iters=100,
                   pos_thresh=1e-4, damping=0.05)
    assert r2.converged and r2.iterations == 10
    with pytest.raises(ValueError):
        ctl.solve(np.zeros(2), NEUTRAL)


ROT_TOL_RAD = 1e-3  # north_star: ... and to 1e-3 rad


def _rot_angle(ra, rb):
    """Angle (rad) of the rotation between rotation matrices ra and rb ([n,3,3]), row-wise."""
    tr = np.einsum("nij,nij->n", ra, rb)  # trace(ra^T rb)
    return np.arccos(np.clip((tr - 1.0) * 0.5, -1.0, 1.0))


def _compare_with_oracle(res, ref, targets, oracle_chain, pos_thresh, flip_budget, rot_budget=0):
    q = res.q.double().cpu().numpy()
    conv = res.converged.cpu().numpy()
    iters = res.iterations.cpu().numpy()
    assert np.array_equal(res.success.cpu().numpy(), conv)  # App. D.2
    flips = int((iters != ref["iterations"]).sum())
    conv_flips = int((conv != ref["converged"]).sum())
    assert flips <= flip_budget, (flips, flip_budget)
    assert conv_flips <= max(1, flip_budget // 4)
    both = conv & ref["converged"]
    same = both & (iters == ref["iterations"])
    # reference FK (position AND orientation) of the GPU's joint solution vs the reference's own final EE pose
    ee, ee_mat, _ = c_oracle.fk_jac(oracle_chain, q, nthreads=8)
    ref_mat = c_oracle.fk_jac(oracle_chain, ref["q"], nthreads=8)[1]
    assert np.linalg.norm(ee[same] - ref["final_pos"][same], axis=1).max() < EE_TOL_M
    rot = _rot_angle(ee_mat, ref_mat)
    # rot_budget: converged queries whose long FP32 walk drifted along the null space of the 7-joint arm (the same
    # position within EE_TOL_M, another orientation); at most that many, and each within 1e-2 rad
    drift = int((rot[same] >= ROT_TOL_RAD).sum())
    assert drift <= rot_budget and rot[same].max() < (1e-2 if rot_budget else ROT_TOL_RAD), (drift, rot[same].max())
    # queries whose iteration count flipped (one side crossed pos_thresh a step earlier): both poses lie in the
    # pos_thresh ball around the target, one DLS step (<= ~pos_thresh of EE travel) apart
    flipped = both & ~same
    if flipped.any():
        assert np.linalg.norm(ee[flipped] - ref["final_pos"][flipped], axis=1).max() <= 2 * pos_thresh
        assert rot[flipped].max() < 1e-2, rot[flipped].max()
    # every converged GPU solution really is within pos_thresh of its target under reference FK
    assert np.linalg.norm(ee[conv] - targets[conv], axis=1).max() < pos_thresh + 1e-5
    # limits respected
    lo, hi = np.array(oracle_chain.lower[:]), np.array(oracle_chain.upper[:])
    assert (q >= lo - 1e-6).all() and (q <= hi + 1e-6).all()
    return flips


@pytest.mark.parametrize("kin", ["specialized", "generic"])
def test_cfg2_4096_cold_targets_vs_oracle(tree, oracle_chain, kin):
    """BASELINE cfg2: 4096 reachable targets, cold start from neutral, defaults."""
    n = 4096
    qstar = synthetic.random_joint_configs(n, tree.lower, tree.upper, seed=0, dtype=torch.float64).numpy()
    targets = c_oracle.fk_jac(oracle_chain, qstar, nthreads=8)[0]
    ref = c_oracle.ik_solve(oracle_chain, targets, NEUTRAL, nthreads=8)
    cnt = torch.zeros(4, dtype=torch.int64, device="cuda")
    res = engine.ik_solve(torch.tensor(targets, dtype=torch.float32, device="cuda"),
                          torch.tensor(NEUTRAL, dtype=torch.float32, device="cuda"),
                          engine.ik_params(kinematics=kin), counters=cnt)
    ref32 = c_oracle.ik_solve(oracle_chain, targets.astype(np.float32).astype(np.float64), NEUTRAL, nthreads=8)
    _compare_with_oracle(res, ref32, targets, oracle_chain, 1e-3, flip_budget=8)
    c = cnt.cpu().numpy()
    assert c[0] == n and c[1] == int(res.converged.sum()) and c[2] == c[1] and c[3] == int(res.iterations.sum())
    # workload statistics of SURVEY 8d (success ~99.7 %, mean iterations ~16)
    assert 0.99 < c[1] / n < 1.0 and 15 < c[3] / n < 17.5
    assert ref["converged"].mean() == pytest.approx(c[1] / n, abs=2e-3)


def test_fp64_kernel_matches_oracle_on_cfg2(tree, oracle_chain):
    n = 4096
    qstar = synthetic.random_joint_configs(n, tree.lower, tree.upper, seed=0, dtype=torch.float64).numpy()
    targets = c_oracle.fk_jac(oracle_chain, qstar, nthreads=8)[0]
    ref = c_oracle.ik_solve(oracle_chain, targets, NEUTRAL, nthreads=8)
    res = engine.ik_solve(torch.tensor(targets, device="cuda"), torch.tensor(NEUTRAL, device="cuda"), engine.ik_params())
    iters = res.iterations.cpu().numpy()
    assert (iters != ref["iterations"]).sum() <= 1  # exact-threshold ties only
    same = iters == ref["iterations"]
    conv = ref["converged"] & same
    np.testing.assert_allclose(res.q.cpu().numpy()[conv], ref["q"][conv], atol=1e-7)
    np.testing.assert_allclose(res.final_pos.cpu().numpy()[conv], ref["final_pos"][conv], atol=1e-8)


def test_per_query_init_ragged_sizes_and_edge_cases(tree, oracle_chain):
    rng = np.random.default_rng(21)
    lo, hi = tree.lower, tree.upper
    for n in (1, 2, 31, 33, 1000):
        q0 = np.clip(NEUTRAL + rng.uniform(-0.3, 0.3, (n, 7)), lo, hi)
        targets = c_oracle.fk_jac(oracle_chain, np.clip(q0 + rng.uniform(-0.1, 0.1, (n, 7)), lo, hi))[0]
        ref = c_oracle.ik_solve(oracle_chain, targets, q0)
        res = engine.ik_solve(torch.tensor(targets, device="cuda"), torch.tensor(q0, device="cuda"), engine.ik_params())
        assert np.array_equal(res.iterations.cpu().numpy(), ref["iterations"])
        np.testing.assert_allclose(res.q.cpu().numpy(), ref["q"], atol=1e-8)
    # empty batch
    res = engine.ik_solve(torch.empty((0, 3), device="cuda"), torch.tensor(NEUTRAL, dtype=torch.float32, device="cuda"),
                          engine.ik_params())
    assert len(res) == 0 and res.iterations.shape == (0,)
    # max_iters = 0: no pass runs, iterations 0, final_pos = FK(q_init), not converged (ik_solver.py:54-57,88)
    res = engine.ik_solve(torch.tensor([[1.3, 0.0, 0.6]], device="cuda", dtype=torch.float64),
                          torch.tensor(NEUTRAL, device="cuda"), engine.ik_params(max_iters=0))
    assert int(res.iterations[0]) == 0 and not bool(res.converged[0])
    np.testing.assert_allclose(res.final_pos[0].cpu().numpy(), [1.23843967, 0, 0.49740014], atol=1e-8)
    np.testing.assert_allclose(res.q[0].cpu().numpy(), NEUTRAL)
    # argument validation
    with pytest.raises(ValueError):
        engine.ik_solve(torch.zeros((4, 3), device="cuda"), torch.zeros((3, 7), device="cuda"), engine.ik_params())
    with pytest.raises(ValueError, match="damping"):
        engine.ik_solve(torch.zeros((4, 3), device="cuda"), torch.zeros(7, device="cuda"), engine.ik_params(damping=0.0))


def test_unreachable_targets_run_out_of_iterations(tree, oracle_chain):
    targets = np.array([[2.5, 0.0, 0.5], [0.6, 0.0, -0.5], [1.415, 0, 0.73]])
    ref = c_oracle.ik_solve(oracle_chain, targets, NEUTRAL, max_iters=40)
    res = engine.ik_solve(torch.tensor(targets, dtype=torch.float32, device="cuda"),
                          torch.tensor(NEUTRAL, dtype=torch.float32, device="cuda"), engine.ik_params(max_iters=40))
    assert res.converged.tolist() == [False, False, True] == ref["converged"].tolist()
    assert res.iterations.tolist() == [40, 40, 7]
    # non-converged solves end in a stretched-out (near-singular) pose after 40 clipped steps: FP32
    # rounding is amplified there; converged solves are held to the tight tolerance elsewhere
    np.testing.assert_allclose(res.pos_error.cpu().numpy(), ref["pos_error"], rtol=2e-5, atol=2e-6)
    np.testing.assert_allclose(res.q.double().cpu().numpy(), ref["q"], atol=1e-3)


def test_large_batch_properties(tree, oracle_chain):
    """2^22 cold targets (cfg5 scale): size-independent properties + a sampled oracle check."""
    n = 1 << 22
    q = synthetic.random_joint_configs(n, tree.lower, tree.upper, seed=1234, device="cuda")
    targets = engine.fk_jac(q, want_quat=False, want_jac=False)[0]
    del q
    neutral = torch.tensor(NEUTRAL, dtype=torch.float32, device="cuda")
    cnt = torch.zeros(4, dtype=torch.int64, device="cuda")
    res = engine.ik_solve(targets, neutral, engine.ik_params(), counters=cnt)
    c = cnt.cpu().numpy()
    assert c[0] == n and c[1] == int(res.converged.sum()) and c[3] == int(res.iterations.long().sum())
    assert 0.995 < c[1] / n < 1.0 and 15.5 < c[3] / n < 16.5
    it = res.iterations
    assert int(it.min()) >= 1 and int(it.max()) == 100
    # the FP32 kernel tests |e|^2 < thresh^2, so the reported sqrt may round onto the threshold itself
    assert bool(((it == 100) | res.converged).all()) and bool((res.pos_error[res.converged] <= 1.0000002e-3).all())
    # final_pos is FK(q) (ik_solver.py:88): recompute with the FK kernel
    fk = engine.fk_jac(res.q, want_quat=False, want_jac=False)[0]
    assert float((fk - res.final_pos).abs().max()) < 2e-6
    # idempotence: a converged solution is a fixed point - re-solving from it takes 1 iteration
    idx = torch.nonzero(res.converged)[:65536, 0]
    again = engine.ik_solve(targets[idx], res.q[idx], engine.ik_params())
    assert bool((again.iterations == 1).all()) and torch.equal(again.q, res.q[idx])
    # determinism despite dynamic lane refill
    res2 = engine.ik_solve(targets, neutral, engine.ik_params())
    assert torch.equal(res.q, res2.q) and torch.equal(res.iterations, res2.iterations)
    # sampled oracle comparison (first 16384 queries)
    m = 16384
    th = targets[:m].double().cpu().numpy()
    ref = c_oracle.ik_solve(oracle_chain, th, NEUTRAL, nthreads=8)
    sub = engine.BatchIKResult(success=res.success[:m], q=res.q[:m], final_pos=res.final_pos[:m],
                               pos_error=res.pos_error[:m], iterations=res.iterations[:m], converged=res.converged[:m])
    flips = _compare_with_oracle(sub, ref, th, oracle_chain, 1e-3, flip_budget=32)
    print(f"iteration-count flips FP32 vs FP64 oracle: {flips}/{m}")


def test_pair_kernel_is_bit_identical_to_lane_kernel(tree, oracle_chain):
    """The two-queries-per-lane kernel (packed FFMA2/FMUL2/FADD2, deferred flush) executes the same
    correctly rounded FP32 operations per query as the one-query-per-lane kernel: every output must be
    bit-identical, whatever the batch size, q_init mode, output layout or which slot a query lands in."""
    neutral = torch.tensor(NEUTRAL, dtype=torch.float32, device="cuda")
    for n in (1, 2, 63, 64, 65, 4097, 300_001, (1 << 21) + 5):
        q = synthetic.random_joint_configs(n, tree.lower, tree.upper, seed=100 + n % 97, device="cuda")
        targets = engine.fk_jac(q, want_quat=False, want_jac=False)[0]
        q0 = (neutral + 0.2 * torch.randn((n, 7), device="cuda")).contiguous()
        # a few unreachable targets (run out of iterations) and queries that converge on the first pass
        # from a q_init OUTSIDE the joint limits (must be returned untouched, ik_solver.py:61-67)
        targets[::97] = torch.tensor([2.5, 0.0, 0.5], device="cuda")
        q_out = q0.clone()
        q_out[::53, 0] = 3.2  # upper limit of joint 1 is 2.8973
        t_out = targets.clone()
        t_out[::53] = engine.fk_jac(q_out[::53].contiguous(), want_quat=False, want_jac=False)[0]
        for qi, tg in ((neutral, targets), (q0, targets), (q_out, t_out)):
            for packed in (True, False):
                cl = torch.zeros(4, dtype=torch.int64, device="cuda")
                cp = torch.zeros(4, dtype=torch.int64, device="cuda")
                a = engine.ik_solve(tg, qi, engine.ik_params(max_iters=60, kinematics="spec_lane"), packed=packed, counters=cl)
                for kin in ("spec_pair",):
                    cp.zero_()
                    b = engine.ik_solve(tg, qi, engine.ik_params(max_iters=60, kinematics=kin), packed=packed, counters=cp)
                    for f in ("q", "final_pos", "pos_error", "iterations", "converged", "success"):
                        assert torch.equal(getattr(a, f), getattr(b, f)), (n, f, packed, kin)
                    assert torch.equal(cl, cp) and int(cl[0]) == n
        first = engine.ik_solve(t_out, q_out, engine.ik_params(kinematics="spec_pair"))
        sel = torch.arange(0, n, 53, device="cuda")
        assert bool((first.iterations[sel] == 1).all()) and torch.equal(first.q[sel], q_out[sel])
    # and the pair kernel against the FP64 oracle on its own
    n = 8192
    qstar = synthetic.random_joint_configs(n, tree.lower, tree.upper, seed=5, dtype=torch.float64).numpy()
    th = c_oracle.fk_jac(oracle_chain, qstar, nthreads=8)[0].astype(np.float32).astype(np.float64)
    ref = c_oracle.ik_solve(oracle_chain, th, NEUTRAL, nthreads=8)
    res = engine.ik_solve(torch.tensor(th, dtype=torch.float32, device="cuda"), neutral, engine.ik_params(kinematics="spec_pair"))
    _compare_with_oracle(res, ref, th, oracle_chain, 1e-3, flip_budget=16)


def test_packed_and_separate_outputs_agree(tree):
    """pnp_ik_solve_packed_f32 (the default) and pnp_ik_solve_f32 write the same results."""
    n = 100_003
    q = synthetic.random_joint_configs(n, tree.lower, tree.upper, seed=77, device="cuda")
    targets = engine.fk_jac(q, want_quat=False, want_jac=False)[0]
    q0 = (torch.tensor(NEUTRAL, dtype=torch.float32, device="cuda") + 0.1 * torch.randn((n, 7), device="cuda")).contiguous()
    for qi in (torch.tensor(NEUTRAL, dtype=torch.float32, device="cuda"), q0):
        a = engine.ik_solve(targets, qi, engine.ik_params(), packed=True)
        b = engine.ik_solve(targets, qi, engine.ik_params(), packed=False)
        assert a.q.shape == (n, 7) and a.final_pos.shape == (n, 3) and a.iterations.dtype == torch.int32
        assert torch.equal(a.q, b.q) and torch.equal(a.final_pos, b.final_pos) and torch.equal(a.pos_error, b.pos_error)
        assert torch.equal(a.iterations, b.iterations) and torch.equal(a.converged, b.converged)
        assert torch.equal(a.success, b.success)
    with pytest.raises(ValueError):
        engine.ik_solve(targets.double(), qi.double(), engine.ik_params(), packed=True)


def test_waypoint_sequences_vs_oracle(tree, oracle_model, oracle_chain):
    """cfg4 (MoveIKSkill inner loop, move.py:106-137) on a few envs vs a NumPy restatement."""
    n, steps = 24, 50
    w = synthetic.waypoint_envs(n, seed=5, dtype=torch.float64)
    q0, goal = w["q_start"].numpy(), w["goal"].numpy()
    out = engine.ik_waypoints(torch.tensor(q0, dtype=torch.float32, device="cuda"),
                              torch.tensor(goal, dtype=torch.float32, device="cuda"), steps, engine.ik_params())
    ctl = ik_oracle.JacobianIKController(oracle_model, mj_oracle.MjData(oracle_model))
    data = mj_oracle.MjData(oracle_model)
    for e in range(n):
        q = q0[e].astype(np.float32).astype(np.float64)
        g = goal[e].astype(np.float32).astype(np.float64)
        pos = ik_oracle.fk_site(oracle_model, data, q)[0]
        accepted = fails = 0
        for _ in range(steps):
            direction = g - pos
            dist = np.linalg.norm(direction)
            if not dist > 0.01:
                break
            step = min(min(0.01, dist * 0.1), 0.02) * (0.5 if fails > 0 else 1.0)
            nxt = pos + direction * step / dist if dist > step else g.copy()
            r = ctl.solve(nxt, q)
            if r.success and r.pos_error < 0.02:
                pos, q, fails = r.final_pos, r.q, 0
                accepted += 1
            else:
                fails += 1
        assert int(out["n_accepted"][e]) == accepted
        np.testing.assert_allclose(out["pos"][e].cpu().numpy(), pos, atol=5e-5)
        np.testing.assert_allclose(out["q"][e].cpu().numpy(), q, atol=2e-3)


def test_waypoint_pair_kernel_is_bit_identical_to_lane_kernel(tree, oracle_chain):
    """ik_waypoints_v_kernel<F2> (two envs per lane, packed FP32) vs <float> (one env per lane): same
    operations per env, so every output is bit-identical; both agree with the scalar-template kernel
    (generic kinematics) within the FP32 tolerance."""
    for n, steps in ((1, 50), (63, 50), (65, 7), (5000, 50), (200_001, 20)):
        w = synthetic.waypoint_envs(n, seed=n % 13, device="cuda")
        outs = {}
        for kin in ("spec_lane", "spec_pair", "generic"):
            cnt = torch.zeros(4, dtype=torch.int64, device="cuda")
            outs[kin] = (engine.ik_waypoints(w["q_start"], w["goal"], steps, engine.ik_params(kinematics=kin), counters=cnt), cnt)
        (a, ca), (b, cb), (g, cg) = outs["spec_lane"], outs["spec_pair"], outs["generic"]
        for f in ("q", "pos", "n_accepted", "iters_total"):
            assert torch.equal(a[f], b[f]), (n, f)
        assert torch.equal(ca, cb)
        same = a["n_accepted"] == g["n_accepted"]
        assert float(same.float().mean()) > 0.999
        diff = (a["pos"][same] - g["pos"][same]).abs().amax(dim=1)
        # the two kernels round differently; a waypoint solve is only converged to pos_thresh = 1e-3, so
        # a rare iteration-count flip moves an end point by up to that much
        assert float((diff < 5e-5).float().mean()) > 0.99 and float(diff.max()) < 2.5e-3
    # an env whose q_start violates a joint limit and already sits at its goal: returned untouched
    q0 = torch.tensor(NEUTRAL, dtype=torch.float32, device="cuda").repeat(64, 1)
    q0[:, 0] = 3.2
    goal = engine.fk_jac(q0, want_quat=False, want_jac=False)[0]
    for kin in ("spec_lane", "spec_pair"):
        r = engine.ik_waypoints(q0, goal, 10, engine.ik_params(kinematics=kin))
        assert torch.equal(r["q"], q0) and int(r["n_accepted"].sum()) == 0


def test_waypoint_fused_pass_is_bit_identical_to_separate_passes(tree, monkeypatch):
    """The pass in which a warm solve is accepted (or the INIT pass) is also the first iteration of the next
    solve: same q, so the same FK and Jacobian, only the target changes (move.py:128-137).  One pass less
    per solve, and every output bit-identical to the kernel that spends a separate pass on it
    (PNP_WAYPOINT_FUSE=0) - including rejected solves, iteration caps of 1 and 2, targets already within
    pos_thresh, and starts outside the joint limits."""
    cases = [(1, 50, {}), (65, 50, {}), (3000, 50, {}), (3000, 12, dict(max_iters=1)), (3000, 12, dict(max_iters=2)),
             (3000, 20, dict(pos_thresh=5e-3, damping=0.05)), (100_001, 30, {})]
    for n, steps, kw in cases:
        w = synthetic.waypoint_envs(n, seed=n % 7 + 1, device="cuda")
        q0 = w["q_start"].clone()
        q0[::5, 0] = 3.1     # beyond joint 1's limit: the first solve starts from it unclipped
        q0[1::9, 3] = 0.2    # beyond joint 4's upper limit
        for kin in ("spec_lane", "spec_pair"):
            outs = []
            for fuse in ("0", "1"):
                monkeypatch.setenv("PNP_WAYPOINT_FUSE", fuse)
                cnt = torch.zeros(4, dtype=torch.int64, device="cuda")
                outs.append((engine.ik_waypoints(q0, w["goal"], steps, engine.ik_params(kinematics=kin, **kw), counters=cnt), cnt))
            (a, ca), (b, cb) = outs
            for f in ("q", "pos", "n_accepted", "iters_total"):
                assert torch.equal(a[f], b[f]), (n, steps, kw, kin, f)
            assert torch.equal(ca, cb) and int(ca[0]) > 0
    monkeypatch.delenv("PNP_WAYPOINT_FUSE")


def test_single_query_mailbox_path_equals_batch_kernel(kin_model, golden_ik, tree):
    """JacobianIKController.solve goes through pnp_ik_solve_one_host_f32 (mapped pinned mailbox, one
    launch, no memcpy); it runs the arithmetic of the batch kernels, so a batch of one gives the same bits."""
    g = golden_ik
    ctl = JacobianIKController(kin_model, KinematicData(kin_model))
    for k in range(0, len(g["tag"]), 3):
        kw = _kw(g, k)
        r = ctl.solve(g["target"][k], g["q_init"][k], **kw)
        b = engine.ik_solve(torch.tensor(g["target"][k][None], dtype=torch.float32, device="cuda"),
                            torch.tensor(g["q_init"][k], dtype=torch.float32, device="cuda"),
                            engine.ik_params(kinematics="spec_lane", **kw))
        assert r.iterations == int(b.iterations[0]) and r.converged == bool(b.converged[0]) and r.success == bool(b.success[0])
        np.testing.assert_array_equal(r.q.astype(np.float32), b.q[0].cpu().numpy())
        np.testing.assert_array_equal(r.final_pos.astype(np.float32), b.final_pos[0].cpu().numpy())
        assert np.float32(r.pos_error) == b.pos_error[0].cpu().numpy()
    # generic tree path of the same entry point
    ctl_g = JacobianIKController(kin_model, KinematicData(kin_model), kinematics="generic")
    r = ctl_g.solve(np.array([1.415, 0.0, 0.73]), NEUTRAL)
    assert r.success and r.iterations == 7 and np.linalg.norm(r.final_pos - [1.415, 0.0, 0.73]) < 1e-3


def test_cfg5_full_size_batch_properties(tree):
    """BASELINE cfg5 at the bench size (2^24 cold targets, one launch): size-independent properties.
    The pair and lane kernels must agree bit for bit on all 16.7 M queries, the counters must equal the
    per-query outputs, every converged query must satisfy the threshold under the FK kernel, and the
    result must not depend on how the dynamic slot refill interleaved the queries (two runs equal)."""
    n = 1 << 24
    targets = torch.empty((n, 3), dtype=torch.float32, device="cuda")
    for off in range(0, n, 1 << 22):
        q = synthetic.random_joint_configs(1 << 22, tree.lower, tree.upper, seed=77 + off, device="cuda")
        targets[off:off + (1 << 22)] = engine.fk_jac(q, want_quat=False, want_jac=False)[0]
        del q
    neutral = torch.tensor(NEUTRAL, dtype=torch.float32, device="cuda")
    cnt = torch.zeros(4, dtype=torch.int64, device="cuda")
    a = engine.ik_solve(targets, neutral, engine.ik_params(kinematics="spec_pair"), counters=cnt)
    c = cnt.cpu().numpy()
    assert c[0] == n and c[1] == int(a.converged.sum()) and c[2] == c[1] and c[3] == int(a.iterations.long().sum())
    assert 0.997 < c[1] / n < 0.999 and 15.7 < c[3] / n < 16.0   # SURVEY 8d workload statistics
    b = engine.ik_solve(targets, neutral, engine.ik_params(kinematics="spec_lane"))
    for f in ("q", "final_pos", "pos_error", "iterations", "converged"):
        assert torch.equal(getattr(a, f), getattr(b, f)), f
    del b
    a2 = engine.ik_solve(targets, neutral, engine.ik_params(kinematics="spec_pair"))
    assert torch.equal(a.q, a2.q) and torch.equal(a.iterations, a2.iterations)
    del a2
    fk = engine.fk_jac(a.q, want_quat=False, want_jac=False)[0]
    assert float((fk - a.final_pos).abs().max()) < 2e-6
    err = (fk - targets).norm(dim=1)
    assert float(err[a.converged].max()) < 1e-3 + 2e-6
    assert bool((a.iterations[~a.converged] == 100).all())


def test_cfg4_full_size_waypoint_properties(tree):
    """BASELINE cfg4 at full size (2^20 envs x 50 warm-started waypoint solves, one launch): the pair and
    lane kernels agree bit for bit on every env; counters equal the per-env outputs; every env ends closer
    to its goal than it started, within the waypoint budget; warm solves take ~2 passes (SURVEY 8d)."""
    n, steps = 1 << 20, 50
    w = synthetic.waypoint_envs(n, seed=0, device="cuda")
    cnt = torch.zeros(4, dtype=torch.int64, device="cuda")
    a = engine.ik_waypoints(w["q_start"], w["goal"], steps, engine.ik_params(kinematics="spec_pair"), counters=cnt)
    b = engine.ik_waypoints(w["q_start"], w["goal"], steps, engine.ik_params(kinematics="spec_lane"))
    for f in ("q", "pos", "n_accepted", "iters_total"):
        assert torch.equal(a[f], b[f]), f
    c = cnt.cpu().numpy()
    assert c[3] == int(a["iters_total"].long().sum()) and c[1] == c[0]       # every warm solve converges
    assert int(a["n_accepted"].max()) <= steps and int(a["n_accepted"].min()) >= 0
    assert c[0] >= int(a["n_accepted"].long().sum())                        # solves >= accepted waypoints
    assert 1.9 < c[3] / c[0] < 2.3
    start = engine.fk_jac(w["q_start"], want_quat=False, want_jac=False)[0]
    d0 = (w["goal"] - start).norm(dim=1)
    d1 = (w["goal"] - a["pos"]).norm(dim=1)
    assert bool((d1 <= d0 + 1e-6).all())
    moved = a["n_accepted"] > 0
    assert bool((d1[moved] < d0[moved]).all())
    # pos is FK(q) of the returned joints
    fk = engine.fk_jac(a["q"], want_quat=False, want_jac=False)[0]
    assert float((fk - a["pos"]).abs().max()) < 2e-6
    # no failed solves in this workload: an env with fewer than `steps` accepted waypoints stopped because
    # it reached its goal (move.py:106, |goal - pos| <= 0.01)
    if c[0] == int(a["n_accepted"].long().sum()):
        early = a["n_accepted"] < steps
        assert float(d1[early].max()) <= 0.01 + 1e-6


def test_solver_parameter_sweep_vs_oracle(tree, oracle_chain):
    """The solve kwargs are part of the reference signature (ik_solver.py:35-37): sweep them - thresholds,
    damping, step limit, iteration budget, warm and cold starts - on all three FP32 kernels (generic tree,
    one query per lane, two per lane) against the FP64 C restatement."""
    rng = np.random.default_rng(99)
    lo, hi = tree.lower, tree.upper
    cases = [dict(max_iters=100, pos_thresh=1e-3, damping=1e-2, step_limit=0.1),     # defaults
             dict(max_iters=100, pos_thresh=1e-4, damping=0.05, step_limit=0.1),     # test/ik_test.py
             dict(max_iters=25, pos_thresh=2e-3, damping=1e-3, step_limit=0.05),
             dict(max_iters=200, pos_thresh=5e-4, damping=0.1, step_limit=0.2),
             dict(max_iters=3, pos_thresh=1e-3, damping=1e-2, step_limit=0.1),       # most queries run out
             dict(max_iters=60, pos_thresh=1e-2, damping=1.0, step_limit=1.0)]
    n = 3000
    for ci, kw in enumerate(cases):
        qstar = rng.uniform(lo, hi, (n, 7))
        targets = c_oracle.fk_jac(oracle_chain, qstar, nthreads=8)[0].astype(np.float32).astype(np.float64)
        warm = ci % 2 == 1
        q0 = np.clip(qstar + rng.uniform(-0.2, 0.2, (n, 7)), lo, hi).astype(np.float32).astype(np.float64) if warm else NEUTRAL
        ref = c_oracle.ik_solve(oracle_chain, targets, q0, nthreads=8, **kw)
        tg = torch.tensor(targets, dtype=torch.float32, device="cuda")
        qi = torch.tensor(q0, dtype=torch.float32, device="cuda")
        for kin in ("generic", "spec_lane", "spec_pair"):
            res = engine.ik_solve(tg, qi, engine.ik_params(kinematics=kin, **kw))
            iters = res.iterations.cpu().numpy()
            conv = res.converged.cpu().numpy()
            flips = int((iters != ref["iterations"]).sum())
            assert flips <= max(6, n // 250), (kw, kin, flips)
            assert int((conv != ref["converged"]).sum()) <= max(3, n // 500), (kw, kin)
            same = conv & ref["converged"] & (iters == ref["iterations"])
            q = res.q.double().cpu().numpy()
            ee = c_oracle.fk_jac(oracle_chain, q, nthreads=8)[0]
            assert np.linalg.norm(ee[same] - ref["final_pos"][same], axis=1).max() < EE_TOL_M, (kw, kin)
            assert np.linalg.norm(ee[conv] - targets[conv], axis=1).max() < kw["pos_thresh"] + 1e-5
            assert (q >= lo - 1e-6).all() and (q <= hi + 1e-6).all() or warm  # cold start stays within limits

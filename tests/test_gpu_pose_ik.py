"""GPU: pose-mode (6-row, 6x6 solve) IK extension vs its FP64 NumPy statement (oracle/pose_ik_oracle.py).
No reference behaviour exists for this entry point (panda_env.py:399-409 imports a missing name).

The workspace tests draw q* uniformly inside the joint limits and ask for the pose (FK(q*), mat2Quat(R(q*))), so the
site frame visits all four mju_mat2Quat cases and both hemispheres of the error quaternion (near NEUTRAL the end
effector points down and every target lands in case 1).  W-near starts at clip(q* + U(+-0.3)), W-cold at NEUTRAL.
The FP64 kernel is held to the batched statement (pose_ik_oracle.solve_pose_batch) iteration for iteration; the FP32
kernel, run against the statement on its FP32-rounded inputs, to a counted number of iteration flips and to poses
re-evaluated with the FP64 FK."""
import ctypes

import numpy as np
import pytest
import torch

from conftest import NEUTRAL
from mujoco_panda_pnp_b200 import KinematicData, KinematicTree, _lib, engine, synthetic
from mujoco_panda_pnp_b200.skills import JacobianIKController, solve_ik
from oracle import c_oracle, ik_oracle, mj_oracle, pose_ik_oracle

pytestmark = pytest.mark.gpu


def _targets(oracle_model, n, seed, spread=0.5):
    rng = np.random.default_rng(seed)
    lo, hi = oracle_model.jnt_range[:7, 0], oracle_model.jnt_range[:7, 1]
    qs = np.clip(NEUTRAL + rng.uniform(-spread, spread, (n, 7)), lo, hi)
    d = mj_oracle.MjData(oracle_model)
    pos, quat = [], []
    for q in qs:
        p, _, qu, _ = ik_oracle.fk_site(oracle_model, d, q)
        pos.append(p), quat.append(qu)
    return np.array(pos), np.array(quat)


@pytest.mark.parametrize("kin", ["specialized", "generic"])
def test_fp64_pose_ik_is_iteration_exact_vs_statement(cuda_lib, oracle_model, kin_model, kin):
    pos, quat = _targets(oracle_model, 48, seed=1)
    ctl = JacobianIKController(kin_model, KinematicData(kin_model), precision="fp64", kinematics=kin)
    out = ctl.solve_pose(pos, quat, NEUTRAL)
    d = mj_oracle.MjData(oracle_model)
    n_conv = 0
    for k in range(len(pos)):
        w = pose_ik_oracle.solve_pose(oracle_model, d, pos[k], quat[k], NEUTRAL)
        assert int(out["iterations"][k]) == w["iterations"], k
        assert bool(out["converged"][k]) == w["converged"] and bool(out["success"][k]) == w["success"]
        tol = 1e-8 if w["converged"] else 1e-5
        np.testing.assert_allclose(out["q"][k].cpu().numpy(), w["q"], atol=tol)
        np.testing.assert_allclose(out["final_pos"][k].cpu().numpy(), w["final_pos"], atol=tol)
        assert abs(float(out["rot_error"][k]) - w["rot_error"]) < tol
        n_conv += w["converged"]
    assert n_conv >= 40


def test_fp32_pose_ik_reaches_the_pose(cuda_lib, oracle_model, oracle_chain, kin_model):
    from oracle import c_oracle

    pos, quat = _targets(oracle_model, 2048 // 8, seed=2)
    ctl = JacobianIKController(kin_model, KinematicData(kin_model))
    out = ctl.solve_pose(pos, quat, NEUTRAL)
    conv = out["converged"].cpu().numpy()
    assert conv.mean() > 0.9
    q = out["q"].double().cpu().numpy()
    ee, mat, _ = c_oracle.fk_jac(oracle_chain, q)
    assert np.linalg.norm(ee[conv] - pos[conv], axis=1).max() < 1e-3 + 1e-5
    # orientation: angle between the reached and the requested frame below rot_thresh (+ FP32 slack)
    for k in np.nonzero(conv)[0][:64]:
        qc = np.empty(4)
        mj_oracle.mju_mat2Quat(qc, mat[k].reshape(9))
        ang = 2 * np.arccos(min(1.0, abs(float(qc @ quat[k]))))
        assert ang < 1e-2 + 1e-4
    # the dangling reference API: solve_ik(model, data, site_name, target_pos, target_quat, q_init)
    data = KinematicData(kin_model)
    r = solve_ik(kin_model, data, "ee_center_site", pos[0], quat[0], NEUTRAL)
    assert r.success and r.q.shape == (7,) and np.array_equal(data.qpos[:7], r.q)
    with pytest.raises(ValueError):
        engine.ik_pose_solve(torch.zeros((2, 3), device="cuda"), torch.zeros((3, 4), device="cuda"),
                             torch.zeros(7, device="cuda"), engine.ik_params())


# ---------------------------------------------------------------------------------------------------------------------
# Workspace tests against the batched FP64 statement
# ---------------------------------------------------------------------------------------------------------------------
IK_BLOCK = 128  # pnp_kernels.cuh: threads per IK block; up to sm_count * IK_BLOCK queries take the small-batch path
KINS = ["specialized", "generic"]
DTYPES = {"fp32": torch.float32, "fp64": torch.float64}
DEFAULTS = dict(max_iters=100, pos_thresh=1e-3, rot_thresh=1e-2, damping=1e-2, step_limit=0.1, rot_weight=1.0)
FP32_POS_TOL, FP32_QUAT_TOL, FP32_ROT_TOL = 1e-5, 1e-5, 2e-5  # FP32 kernel vs FP64 evaluation at the same q
SIGN_MARGIN = 1e-4  # below this mat2Quat case margin an FP32 frame may take the neighbouring case (quaternion -q)


@pytest.fixture(scope="module")
def tree(cuda_lib):
    t = KinematicTree.from_mjcf()
    engine.set_tree(t)
    return t


def _limits(chain):
    return np.array(chain.lower[:]), np.array(chain.upper[:])


def _workspace(chain, n, seed):
    """W: q* uniform inside the joint limits, target (FK(q*), mat2Quat(R(q*))), with the mat2Quat case of each target."""
    rng = np.random.default_rng(seed)
    lo, hi = _limits(chain)
    q_star = rng.uniform(lo, hi, (n, 7))
    ev = pose_ik_oracle.pose_eval_batch(chain, q_star, np.zeros(3), np.array([1.0, 0.0, 0.0, 0.0]))
    return q_star, ev["final_pos"], ev["final_quat"], ev["case"], rng


def _start(chain, q_star, rng, start):
    if start == "near":  # W-near
        lo, hi = _limits(chain)
        return np.clip(q_star + rng.uniform(-0.3, 0.3, q_star.shape), lo, hi)
    return np.tile(NEUTRAL, (len(q_star), 1))  # W-cold


def _assert_cases(case, at_least=100):
    counts = np.bincount(case, minlength=4)
    assert (counts >= at_least).all(), counts


def _rounded(dtype, *arrays):
    """The inputs as the kernel of this precision sees them, in FP64 (the statement runs on these)."""
    if dtype == torch.float32:
        return [np.asarray(a, dtype=np.float32).astype(np.float64) for a in arrays]
    return [np.asarray(a, dtype=np.float64) for a in arrays]


def _split(p):
    p = dict(DEFAULTS, **p)
    return {k: p[k] for k in ("max_iters", "pos_thresh", "damping", "step_limit")}, p["rot_thresh"], p["rot_weight"]


def _solve(tree, dtype, kin, pos, quat, q_init, counters=None, **p):
    engine.set_tree(tree)
    ik, rot_thresh, rot_weight = _split(p)

    def t(a):
        return torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64), device="cuda").to(dtype)

    out = engine.ik_pose_solve(t(pos), t(quat), t(q_init), engine.ik_params(kinematics=kin, **ik),
                               rot_thresh=rot_thresh, rot_weight=rot_weight, counters=counters)
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in out.items()}


def _statement(chain, dtype, pos, quat, q_init, **p):
    pos, quat, q_init = _rounded(dtype, pos, quat, q_init)
    return pose_ik_oracle.solve_pose_batch(chain, pos, quat, q_init, **dict(DEFAULTS, **p))


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint8)


def _assert_quat(got, want, margin, tol, sign_margin):
    """Per component within tol, with the statement's sign wherever its mat2Quat case margin exceeds sign_margin; up
    to sign inside that margin (the two cases give -q and q of one rotation)."""
    got = np.asarray(got, dtype=np.float64)
    d_same = np.abs(got - want).max(axis=1)
    d_any = np.minimum(d_same, np.abs(got + want).max(axis=1))
    strict = margin > sign_margin
    assert d_same[strict].max(initial=0.0) < tol, (d_same[strict].max(), np.argmax(np.where(strict, d_same, 0)))
    assert d_any.max(initial=0.0) < tol, d_any.max()


def _rot_angle(ra, rb):
    tr = np.einsum("nij,nij->n", ra, rb)
    return np.arccos(np.clip((tr - 1.0) * 0.5, -1.0, 1.0))


def _check_fp64(chain, got, ref, pos, quat, tol=1e-8):
    """Iteration-exact: identical iteration counts and flags (at most one query whose FK rounding puts the kernel and
    the statement on opposite sides of a threshold), converged queries within tol in every output."""
    tie = got["iterations"] != ref["iterations"]
    assert tie.sum() <= 1, np.nonzero(tie)[0][:10]
    ok = ~tie
    assert np.array_equal(got["converged"][ok], ref["converged"][ok])
    assert np.array_equal(got["success"][ok], ref["success"][ok])
    c = ok & ref["converged"]
    for key in ("q", "final_pos", "pos_error", "rot_error"):
        d = np.abs(got[key][c] - ref[key][c]).max(initial=0.0)
        assert d < tol, (key, d)
    margin = pose_ik_oracle.pose_eval_batch(chain, ref["q"], pos, quat)["case_margin"]
    _assert_quat(got["final_quat"][c], ref["final_quat"][c], margin[c], tol, 1e-12)
    return int(tie.sum())


def _check_fp32(chain, got, ref, pos, quat, budget, q_budget=2, dq_cap=1e-3, **p):
    """FP32 kernel vs the statement on the FP32-rounded inputs (pos, quat).

    - Iteration flips (one side crosses a threshold a pass earlier) are counted and bounded by ``budget``, converged /
      not-converged flips by 2.  Measured on a B200 (all settings, both kinematics): 0 of 4096 W-near, 1 of 2048
      W-cold, at most 2 of 2048 in the representation test and at most 2 of 512 (0.4 %, pos_thresh = 1e-4) in the
      parameter tests; converged flips at most 1 per batch.  Budgets are max(2, 2x observed).
    - Solves that converge in the same number of passes on both sides agree in q within 2e-5 rad, except for at most
      ``q_budget`` of them, and all of them within ``dq_cap`` (1e-3 rad).  The exceptions are long cold-start walks
      and weak damping, where FP32 rounding early in the walk is amplified: measured |dq|max quantiles (50/99/99.9/100 %)
      W-near
      3.7e-7/2.5e-6/4.2e-6/5.7e-6; W-cold 6.6e-7/1.0e-5/4.9e-5/4.1e-4 (7 and 9 of ~1400 above 2e-5); damping 1e-4
      5.3e-7/1.9e-5/1.6e-4/5.1e-4 (4 and 11 of ~500).  Their FP64-FK poses still agree within 1e-4 m and 1e-4 rad
      (measured at most 6.6e-5 m, 5.8e-5 rad), which is asserted for every one of them.
    - Every converged q reaches the target under the FP64 FK, and the kernel's own reported pose and errors are those
      of its q (tolerances of the one-evaluation probe)."""
    p = dict(DEFAULTS, **p)
    conv, iters = got["converged"], got["iterations"]
    assert np.array_equal(got["success"], conv)
    flips = int((iters != ref["iterations"]).sum())
    conv_flips = int((conv != ref["converged"]).sum())
    assert flips <= budget, (flips, budget)
    assert conv_flips <= 2, conv_flips
    q = got["q"].astype(np.float64)
    same = conv & ref["converged"] & (iters == ref["iterations"])
    dq = np.abs(q[same] - ref["q"][same]).max(axis=1)
    assert (dq > 2e-5).sum() <= q_budget and dq.max(initial=0.0) < dq_cap, (int((dq > 2e-5).sum()), dq.max(initial=0.0))
    ee, mat, _ = c_oracle.fk_jac(chain, q, nthreads=8)
    ref_mat = c_oracle.fk_jac(chain, ref["q"], nthreads=8)[1]
    assert np.linalg.norm(ee[same] - ref["final_pos"][same], axis=1).max(initial=0.0) < 1e-4
    assert _rot_angle(mat, ref_mat)[same].max(initial=0.0) < 1e-4
    ev = pose_ik_oracle.pose_eval_batch(chain, q, pos, quat)
    assert ev["pos_error"][conv].max(initial=0.0) < p["pos_thresh"] + 1e-5
    assert ev["rot_error"][conv].max(initial=0.0) < p["rot_thresh"] + FP32_ROT_TOL
    assert np.abs(got["final_pos"] - ev["final_pos"]).max() < FP32_POS_TOL
    assert np.abs(got["pos_error"] - ev["pos_error"]).max() < FP32_POS_TOL
    assert np.abs(got["rot_error"] - ev["rot_error"]).max() < FP32_ROT_TOL
    _assert_quat(got["final_quat"], ev["final_quat"], ev["case_margin"], FP32_QUAT_TOL, SIGN_MARGIN)
    lo, hi = _limits(chain)
    assert (q >= lo - 1e-6).all() and (q <= hi + 1e-6).all()
    return flips


THETAS = [0.0, 1e-6, 1e-4, 1e-2, 0.3, np.pi / 2, 3.0, np.pi - 1e-4, np.pi]


def _probe_inputs(chain, n=65536, seed=21):
    """q uniform in the limits (5 % of them widened by 0.3 rad past the limits), target quaternions
    delta(theta, random axis) (x) q_ref with q_ref the site quaternion at q - so the error rotation has angle theta -
    each also as -tq, 1e-3 tq and 7.5 tq; every tenth row a uniform random unit quaternion."""
    rng = np.random.default_rng(seed)
    lo, hi = _limits(chain)
    q = rng.uniform(lo, hi, (n, 7))
    wide = rng.random(n) < 0.05
    q[wide] = rng.uniform(lo - 0.3, hi + 0.3, (int(wide.sum()), 7))
    ev = pose_ik_oracle.pose_eval_batch(chain, q, np.zeros(3), np.array([1.0, 0.0, 0.0, 0.0]))
    pos = ev["final_pos"] + rng.uniform(-0.2, 0.2, (n, 3))
    pos[::7] = ev["final_pos"][::7]
    variant = np.arange(n) % 40
    theta = np.array(THETAS)[variant % 9]
    axis = rng.normal(size=(n, 3))
    axis /= np.linalg.norm(axis, axis=1, keepdims=True)
    delta = np.concatenate([np.cos(theta / 2)[:, None], np.sin(theta / 2)[:, None] * axis], axis=1)
    tq = pose_ik_oracle.mulquat_batch(delta, ev["final_quat"])
    rep = np.minimum(variant // 9, 4)  # 0: tq, 1: -tq, 2: 1e-3 tq, 3: 7.5 tq, 4: random unit quaternion
    tq *= np.array([1.0, -1.0, 1e-3, 7.5, 1.0])[rep][:, None]
    rnd = rep == 4
    r = rng.normal(size=(int(rnd.sum()), 4))
    tq[rnd] = r / np.linalg.norm(r, axis=1, keepdims=True)
    return q, pos, tq


@pytest.mark.parametrize("kin", KINS)
@pytest.mark.parametrize("prec", ["fp32", "fp64"])
def test_one_evaluation_probe_vs_statement(tree, oracle_chain, prec, kin):
    """max_iters = 0: the kernel makes one FK, mat2quat_fast, error quaternion and quat2vel_fast at q_init, writes
    every output and stops - a direct test of those device functions over 64 k frames in all four mat2Quat cases and
    both hemispheres of the error quaternion, at error angles from 0 to pi.

    FP32: in the angle fold of quat2vel_fast (opposite-hemisphere target) 2 pi is subtracted from a float near 2 pi,
    which leaves an absolute floor of about 5e-7 rad on rot_error; FP32_ROT_TOL (2e-5 rad) covers it, and at any
    rot_thresh >= 1e-4 it does not change a convergence decision."""
    dtype = DTYPES[prec]
    q, pos, tq = _probe_inputs(oracle_chain)
    got = _solve(tree, dtype, kin, pos, tq, q, max_iters=0)
    qr, posr, tqr = _rounded(dtype, q, pos, tq)
    ref = pose_ik_oracle.pose_eval_batch(oracle_chain, qr, posr, tqr)
    lo, hi = _limits(oracle_chain)
    assert ((qr < lo) | (qr > hi)).any(axis=1).sum() > 1000
    assert (got["iterations"] == 0).all() and not got["converged"].any() and not got["success"].any()
    assert np.array_equal(_bits(got["q"]), _bits(q.astype(got["q"].dtype)))  # returned as given: no clamp, no step
    _assert_cases(ref["case"])
    assert (ref["err_w"] < 0).sum() >= 100 and (ref["err_w"] > 0).sum() >= 100
    if dtype == torch.float32:
        tol_p, tol_q, tol_r, sign_margin = FP32_POS_TOL, FP32_QUAT_TOL, FP32_ROT_TOL, SIGN_MARGIN
    else:
        tol_p, tol_q, tol_r, sign_margin = 1e-12, 1e-12, 1e-11, 1e-12
    assert np.abs(got["final_pos"] - ref["final_pos"]).max() < tol_p
    assert np.abs(got["pos_error"] - ref["pos_error"]).max() < tol_p
    _assert_quat(got["final_quat"], ref["final_quat"], ref["case_margin"], tol_q, sign_margin)
    d = np.abs(got["rot_error"] - ref["rot_error"])
    assert d.max() < tol_r, (d.max(), int(np.argmax(d)))


@pytest.mark.parametrize("kin", KINS)
@pytest.mark.parametrize("start", ["near", "cold"])
def test_fp64_workspace_solves_are_iteration_exact(tree, oracle_chain, start, kin):
    """FP64 kernel, 2048 workspace targets from W-near / W-cold, against the batched statement on c_oracle's FK."""
    q_star, pos, quat, case, rng = _workspace(oracle_chain, 2048, seed=31)
    _assert_cases(case)
    q_init = _start(oracle_chain, q_star, rng, start)
    got = _solve(tree, torch.float64, kin, pos, quat, q_init)
    ref = _statement(oracle_chain, torch.float64, pos, quat, q_init)
    _check_fp64(oracle_chain, got, ref, pos, quat)
    assert ref["converged"].mean() > (0.95 if start == "near" else 0.5)


@pytest.mark.parametrize("kin", KINS)
@pytest.mark.parametrize("start,n", [("near", 4096), ("cold", 2048)])
def test_fp32_workspace_solves_vs_statement(tree, oracle_chain, start, n, kin):
    """FP32 kernel on W-near (4096) / W-cold (2048) against the statement on its FP32-rounded inputs."""
    q_star, pos, quat, case, rng = _workspace(oracle_chain, n, seed=41)
    _assert_cases(case)
    q_init = _start(oracle_chain, q_star, rng, start)
    got = _solve(tree, torch.float32, kin, pos, quat, q_init)
    ref = _statement(oracle_chain, torch.float32, pos, quat, q_init)
    pos32, quat32 = _rounded(torch.float32, pos, quat)
    _check_fp32(oracle_chain, got, ref, pos32, quat32, budget=2, q_budget=2 if start == "near" else 18)
    assert got["converged"].mean() > (0.95 if start == "near" else 0.5)


@pytest.mark.parametrize("kin", KINS)
@pytest.mark.parametrize("prec", ["fp32", "fp64"])
def test_quaternion_representation_invariance(tree, oracle_chain, prec, kin):
    """tq, -tq and 3.7 tq name the same target: the solves must be those of the statement for tq.  A quat2vel that
    does not fold the angle of an opposite-hemisphere error quaternion fails here."""
    dtype = DTYPES[prec]
    q_star, pos, quat, case, rng = _workspace(oracle_chain, 2048, seed=51)
    q_init = _start(oracle_chain, q_star, rng, "near")
    ref = _statement(oracle_chain, dtype, pos, quat, q_init)
    pos_r, quat_r = _rounded(dtype, pos, quat)
    for scale in (1.0, -1.0, 3.7):
        got = _solve(tree, dtype, kin, pos, scale * quat, q_init)
        if dtype == torch.float64:
            tie = got["iterations"] != ref["iterations"]
            assert tie.sum() <= 1, scale
            c = ~tie & ref["converged"]
            assert np.array_equal(got["converged"][~tie], ref["converged"][~tie])
            assert np.abs(got["q"][c] - ref["q"][c]).max() < 1e-9, scale
        else:
            _check_fp32(oracle_chain, got, ref, pos_r, quat_r, budget=4)


SETTINGS = {
    "rot_weight=0.25": dict(rot_weight=0.25),
    "rot_weight=4": dict(rot_weight=4.0),
    "rot_thresh=1e-3": dict(rot_thresh=1e-3),
    "rot_thresh=5e-2": dict(rot_thresh=5e-2),
    "pos_thresh=1e-4": dict(pos_thresh=1e-4),
    "damping=1e-4": dict(damping=1e-4),
    "damping=1e-1": dict(damping=1e-1),
    "step_limit=0.02": dict(step_limit=0.02),
    "step_limit=0": dict(step_limit=0.0),
    "max_iters=1": dict(max_iters=1),
    "max_iters=5": dict(max_iters=5),
}


@pytest.mark.parametrize("kin", KINS)
@pytest.mark.parametrize("prec", ["fp32", "fp64"])
@pytest.mark.parametrize("setting", list(SETTINGS))
def test_parameters_vs_statement(tree, oracle_chain, setting, prec, kin):
    """512 W-near queries per solver parameter: FP64 iteration-exact, FP32 flip-bounded."""
    dtype, p = DTYPES[prec], SETTINGS[setting]
    q_star, pos, quat, case, rng = _workspace(oracle_chain, 512, seed=61)
    q_init = _start(oracle_chain, q_star, rng, "near")
    got = _solve(tree, dtype, kin, pos, quat, q_init, **p)
    ref = _statement(oracle_chain, dtype, pos, quat, q_init, **p)
    if dtype == torch.float64:
        _check_fp64(oracle_chain, got, ref, pos, quat)
    else:
        pos32, quat32 = _rounded(dtype, pos, quat)
        _check_fp32(oracle_chain, got, ref, pos32, quat32, budget=4, q_budget=22 if setting == "damping=1e-4" else 2, **p)
    if p.get("step_limit") == 0.0:  # q never moves
        assert np.array_equal(_bits(got["q"]), _bits(q_init.astype(got["q"].dtype)))
    if "max_iters" in p:
        assert got["iterations"].max() <= p["max_iters"]


@pytest.mark.parametrize("kin", KINS)
@pytest.mark.parametrize("prec", ["fp32", "fp64"])
def test_broadcast_q_init_is_bit_identical_to_per_row(tree, oracle_chain, prec, kin):
    dtype = DTYPES[prec]
    q_star, pos, quat, case, rng = _workspace(oracle_chain, 512, seed=71)
    a = _solve(tree, dtype, kin, pos, quat, NEUTRAL)  # stride 0
    b = _solve(tree, dtype, kin, pos, quat, np.tile(NEUTRAL, (512, 1)))
    for k in a:
        assert np.array_equal(_bits(a[k]), _bits(b[k])), k


def _raw_pose_solve(dtype, kin, tp, tq, qi, outs, counters):
    """pnp_ik_pose_solve_* through the C ABI; outs = (q, final_pos, final_quat, pos_err, rot_err, iters, flags), any
    but q None."""
    lib = _lib.load()
    fn = lib.pnp_ik_pose_solve_f32 if dtype == torch.float32 else lib.pnp_ik_pose_solve_f64
    ptr = [None if t is None else t.data_ptr() for t in outs]
    _lib.check(fn(tp.data_ptr(), tq.data_ptr(), qi.data_ptr(), 7, tp.shape[0], ctypes.byref(engine.ik_params(kinematics=kin)),
                  1e-2, 1.0, *ptr, None if counters is None else counters.data_ptr(),
                  torch.cuda.current_stream().cuda_stream), "pnp_ik_pose_solve")


@pytest.mark.parametrize("kin", KINS)
@pytest.mark.parametrize("prec", ["fp32", "fp64"])
def test_results_do_not_depend_on_batch_shape(tree, oracle_chain, prec, kin):
    """97 witness queries solved one at a time, as one batch (small-batch path: one working warp per block) and at
    scattered rows of batches of sm_count * IK_BLOCK, sm_count * IK_BLOCK + 1 and 2^20 queries (persistent warps with
    lane refill): bit-identical, since no lane's arithmetic depends on where it runs.  The 2^20 batch goes through the
    C ABI into sentinel-filled buffers (every row must be written), with counters, and once more with every nullable
    output NULL."""
    dtype = DTYPES[prec]
    engine.set_tree(tree)
    sm = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    q_star, pos, quat, case, rng = _workspace(oracle_chain, 4096, seed=81)
    q_init = _start(oracle_chain, q_star, rng, "near")
    w = rng.choice(4096, 97, replace=False)
    ref = _solve(tree, dtype, kin, pos[w], quat[w], q_init[w])
    keys = list(ref)
    for k in range(97):
        one = _solve(tree, dtype, kin, pos[w[k]:w[k] + 1], quat[w[k]:w[k] + 1], q_init[w[k]:w[k] + 1])
        for key in keys:
            assert np.array_equal(_bits(one[key][0]), _bits(ref[key][k])), (k, key)
    dev = torch.device("cuda")
    pool = [torch.as_tensor(a, device=dev).to(dtype) for a in (pos, quat, q_init)]
    for n in (sm * IK_BLOCK, sm * IK_BLOCK + 1, 1 << 20):
        idx = rng.integers(0, 4096, n)
        slots = rng.choice(n, 97, replace=False)
        idx[slots] = w
        it = torch.as_tensor(idx, device=dev)
        tp, tq, qi = (a[it].contiguous() for a in pool)
        if n < (1 << 20):
            out = engine.ik_pose_solve(tp, tq, qi, engine.ik_params(kinematics=kin))
            torch.cuda.synchronize()
            for key in keys:
                assert np.array_equal(_bits(out[key][slots].cpu().numpy()), _bits(ref[key])), (n, key)
            continue
        outs = (torch.full((n, 7), float("nan"), dtype=dtype, device=dev),
                torch.full((n, 3), float("nan"), dtype=dtype, device=dev),
                torch.full((n, 4), float("nan"), dtype=dtype, device=dev),
                torch.full((n,), float("nan"), dtype=dtype, device=dev),
                torch.full((n,), float("nan"), dtype=dtype, device=dev),
                torch.full((n,), -1, dtype=torch.int32, device=dev),
                torch.full((n,), 0xFF, dtype=torch.uint8, device=dev))
        counters = torch.zeros(4, dtype=torch.int64, device=dev)
        _raw_pose_solve(dtype, kin, tp, tq, qi, outs, counters)
        torch.cuda.synchronize()
        q, fpos, fquat, perr, rerr, iters, flags = outs
        for t in (q, fpos, fquat, perr, rerr):
            assert torch.isfinite(t).all()
        assert bool(((iters >= 0) & (iters <= 100)).all()) and bool((flags <= 3).all())
        conv, succ = (flags & 1) != 0, (flags & 2) != 0
        assert counters.tolist() == [n, int(conv.sum()), int(succ.sum()), int(iters.long().sum())]
        got = dict(q=q, final_pos=fpos, final_quat=fquat, pos_error=perr, rot_error=rerr, iterations=iters,
                   converged=conv, success=succ)
        for key in keys:
            assert np.array_equal(_bits(got[key][slots].cpu().numpy()), _bits(ref[key])), (n, key)
        q2 = torch.full((n, 7), float("nan"), dtype=dtype, device=dev)
        _raw_pose_solve(dtype, kin, tp, tq, qi, (q2, None, None, None, None, None, None), None)
        torch.cuda.synchronize()
        assert torch.equal(q2.view(torch.uint8), q.view(torch.uint8))
    empty = engine.ik_pose_solve(*(a[:0] for a in pool), engine.ik_params(kinematics=kin))
    assert all(v.shape[0] == 0 for v in empty.values())


@pytest.mark.parametrize("kin", KINS)
@pytest.mark.parametrize("prec", ["fp32", "fp64"])
def test_degenerate_target_quaternions(tree, oracle_chain, prec, kin):
    """A zero or NaN target quaternion has no rotation to reach: the query runs to max_iters unconverged, and its
    neighbours in the batch are untouched."""
    dtype = DTYPES[prec]
    q_star, pos, quat, case, rng = _workspace(oracle_chain, 256, seed=91)
    q_init = _start(oracle_chain, q_star, rng, "near")
    clean = _solve(tree, dtype, kin, pos, quat, q_init)
    bad_quat = np.array([[0.0, 0.0, 0.0, 0.0], [np.nan] * 4, [np.nan, 1.0, 0.0, 0.0], [0.0, 0.0, 0.0, 0.0]])
    at = np.array([0, 37, 130, 255])
    pos2, quat2, qi2 = (np.insert(a, at, a[at], axis=0) for a in (pos, quat, q_init))
    quat2[at + np.arange(len(at))] = bad_quat
    bad = np.zeros(len(pos2), dtype=bool)
    bad[at + np.arange(len(at))] = True
    got = _solve(tree, dtype, kin, pos2, quat2, qi2, max_iters=40)
    assert not got["converged"][bad].any() and not got["success"][bad].any()
    assert (got["iterations"][bad] == 40).all()
    clean40 = _solve(tree, dtype, kin, pos, quat, q_init, max_iters=40)
    for key in clean40:
        assert np.array_equal(_bits(got[key][~bad]), _bits(clean40[key])), key
    assert clean["converged"].mean() > 0.95


@pytest.mark.parametrize("prec", ["fp32", "fp64"])
def test_pose_solve_rejects_invalid_arguments(tree, prec):
    dtype = DTYPES[prec]
    engine.set_tree(tree)
    z = lambda *s: torch.zeros(s, dtype=dtype, device="cuda")  # noqa: E731
    tp, tq, qi, p = z(4, 3), z(4, 4) + 1.0, z(4, 7), engine.ik_params()
    engine.ik_pose_solve(tp, tq, qi, p)  # the valid call
    for kw in (dict(rot_thresh=0.0), dict(rot_thresh=-1e-2), dict(rot_thresh=float("nan")), dict(rot_weight=0.0),
               dict(rot_weight=-1.0), dict(rot_weight=float("nan"))):
        with pytest.raises(ValueError):
            engine.ik_pose_solve(tp, tq, qi, p, **kw)
    for args in ((tp, tq, z(4, 6)), (tp, tq, z(6)), (tp, tq, z(5, 7)), (tp, z(5, 4), qi), (z(4, 4), tq, qi)):
        with pytest.raises(ValueError):
            engine.ik_pose_solve(*args, p)

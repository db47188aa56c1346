"""GPU: the generic-kinematics kernels on arms that are not the packaged Panda, against the FP64 oracles.

``pnp_set_tree`` selects the specialised kernels only for a tree bit-identical to the packaged one, so the generic
build (``GenericKin``, tree in ``__constant__`` memory) serves every other arm: another robot or tool, changed limits
or ``ref`` angles, a live MjModel one ulp off our MJCF reader.  On the packaged Panda (qref = 0, base not rotated, hand
yawed about z) a generic kernel that dropped ``q - qref``, read the packaged limits or base, or ignored ``ee_rot`` would
give the right answer; here it cannot.  Trees:

- PANDA_VARIANT: the Panda with a shifted, 30 degree yawed base; ref = (0.4, -0.3, 0, -1.2, 0, 1.5, 0.785); joint 5
  axis flipped; a joint-3 anchor; joint 2 and joint 6 ranges narrowed / shifted; a longer, tilted tool and a site
  rotated about a skew axis.  The oracle reads it with its own MJCF compile (mj_oracle), bit-equal to ours.
- GENERAL: test_tree's _GENERAL_MJCF (skewed axes, anchors, a ref, Euler / axis-angle frames).  The oracle's reader
  takes quaternions only, so its raw body chain (c_oracle.chain_from_model: no folding) comes from our parse.
- PANDA_ULP: the packaged tree with every double of link_pos, link_rot, ee_pos and ee_rot a few ulp off.

Workloads: q* uniform inside the tree's limits, targets FK(q*) (pose: with mju_mat2Quat of the site frame); "cold"
starts at the middle of the joint ranges, "near" at clip(q* + U(-0.3, 0.3)).  Oracle statistics (CPU, default
parameters; position IK over 4096 targets, pose IK over 2048):

    tree      position cold        position near      pose cold            pose near
              success  mean its    success  its      success  mean its    success  its
    Panda     0.9978   14.5        0.9995   5.6      0.7817   46.7        0.9883   11.1
    variant   0.9910   14.2        0.9998   5.1      0.6504   53.5        0.9927   11.2
    GENERAL   0.9832   18.6        0.9995   6.5      0.4722   74.8        0.9927   17.4

so a cold batch of 4096 has 37 (variant) / 69 (GENERAL) queries that run out of iterations next to thousands that
converge.  Position planner (1024 moves from mid-range +- 0.3 rad to FK(start +- 0.6 rad), every 64th goal moved
1.5 m out of reach, max_outer 300): 1008 plans end at the goal, 16 hit the round bound (status 2), both trees.  With
single-pass solves (max_iters 1, pos_thresh 8e-4, step 0.05) the fallback strategies run out: status 1 on 753 / 608
plans, status 2 on the rest.  Pose planner statement (48 moves from mid-range +- 0.05 rad to the pose at start +- 0.6
rad, max_traj_points 60): CAPPED on 3 (variant) / 0 (GENERAL), OK on the rest.

FP32 budgets are max(2, 2x the count observed on one B200) as in test_gpu_pose_ik.py; OBSERVED records the counts.
Every test leaves the packaged tree uploaded (the other modules' fixtures assume it)."""
import math
from dataclasses import dataclass
from typing import Any

import numpy as np
import pytest
import torch

from conftest import NEUTRAL
from mujoco_panda_pnp_b200 import KinematicData, KinematicModel, KinematicTree, engine, synthetic
from mujoco_panda_pnp_b200.skills import JacobianIKController
from oracle import c_oracle, mj_oracle, move_pose_oracle, pose_ik_oracle
from test_gpu_ik import _compare_with_oracle, _rot_angle
from test_gpu_ik_multistart import FAR, bits, expected
from test_gpu_move_pose import host
from test_gpu_pose_ik import (FP32_POS_TOL, FP32_QUAT_TOL, FP32_ROT_TOL, SIGN_MARGIN, _assert_cases, _assert_quat,
                              _bits, _check_fp32, _check_fp64, _probe_inputs, _rounded, _solve, _start, _statement,
                              _workspace)
from test_ik_multistart_oracle import multistart_batched
from test_move_pose_oracle import check_invariants
from test_tree import _GENERAL_MJCF

pytestmark = pytest.mark.gpu

PANDA_VARIANT = """
<mujoco>
  <compiler angle="radian" autolimits="true"/>
  <default>
    <default class="arm">
      <joint axis="0 0 1" range="-2.8973 2.8973"/>
    </default>
  </default>
  <worldbody>
    <body name="link0" childclass="arm" pos="0.45 -0.12 0.35" quat="0.9659258 0 0 0.2588190">
      <body name="link1" pos="0 0 0.333">
        <joint name="joint1" ref="0.4"/>
        <body name="link2" quat="1 -1 0 0">
          <joint name="joint2" range="-1.5 1.7628" ref="-0.3"/>
          <body name="link3" pos="0 -0.316 0" quat="1 1 0 0">
            <joint name="joint3" pos="0.01 0 0.02"/>
            <body name="link4" pos="0.0825 0 0" quat="1 1 0 0">
              <joint name="joint4" range="-3.0718 -0.0698" ref="-1.2"/>
              <body name="link5" pos="-0.0825 0.384 0" quat="1 -1 0 0">
                <joint name="joint5" axis="0 0 -1"/>
                <body name="link6" quat="1 1 0 0">
                  <joint name="joint6" range="0.2 3.5" ref="1.5"/>
                  <body name="link7" pos="0.088 0 0" quat="1 1 0 0">
                    <joint name="joint7" ref="0.785"/>
                    <body name="hand" pos="0 0 0.107" quat="0.9238795 0 0 -0.3826834">
                      <body name="tool" pos="0.01 -0.005 0.16" quat="0.97 0.17 0.15 0">
                        <site name="ee_center_site" pos="0 0.01 0.02" quat="0.9 0.3 -0.2 0.1"/>
                      </body>
                    </body>
                  </body>
                </body>
              </body>
            </body>
          </body>
        </body>
      </body>
    </body>
  </worldbody>
</mujoco>
"""

FOREIGN = ["variant", "general"]
IK_BLOCK = 128  # pnp_kernels.cuh: up to sm_count * IK_BLOCK queries take the small-batch path

# FP32 counts observed on one B200 (1000 W power limit); each budget is max(2, 2x the count)
OBSERVED = {
    # iteration-count flips of the position solve vs the oracle on the FP32-rounded inputs (4096 / 23040 queries)
    ("variant", "pos", "cold", "small"): 0, ("variant", "pos", "cold", "large"): 3,
    ("variant", "pos", "near", "small"): 1, ("variant", "pos", "near", "large"): 3,
    ("general", "pos", "cold", "small"): 1, ("general", "pos", "cold", "large"): 4,
    ("general", "pos", "near", "small"): 0, ("general", "pos", "near", "large"): 2,
    # position solves converged in the same passes on both sides whose end orientations differ by more than 1e-3 rad
    # (the walk drifted along the arm's null space; the positions agree within 1e-4 m)
    ("variant", "pos_rot", "cold", "large"): 1,
    # multistart attempt indices that differ from the CPU replay of the restart rule
    ("variant", "ms_attempt"): 0, ("general", "ms_attempt"): 0,
    # waypoint envs whose accepted count or end point (5e-5 m) differs from the chained oracle solves
    ("variant", "waypoints"): 0, ("general", "waypoints"): 0,
    # pose solve (2048 queries): iteration flips, and converged solves with |dq| > 2e-5 rad (q_budget of _check_fp32)
    ("variant", "pose", "cold"): 0, ("variant", "pose", "near"): 1,
    ("general", "pose", "cold"): 0, ("general", "pose", "near"): 0,
    ("variant", "pose_dq", "cold"): 17, ("variant", "pose_dq", "near"): 0,
    ("general", "pose_dq", "cold"): 4, ("general", "pose_dq", "near"): 0,
    # planner envs whose status differs from the FP64 oracle's
    ("variant", "plan_status"): 0, ("general", "plan_status"): 0,
}
# largest |dq| (rad) of those pose solves: the variant's cold walks (53 passes on average) go past _check_fp32's 1e-3
POSE_DQ_MAX_OBSERVED = {("variant", "cold"): 2.13e-3}


def budget(*key):
    return max(2, 2 * OBSERVED.get(key, 0))


@dataclass
class Arm:
    name: str
    model: Any    # the product's parse (KinematicModel)
    omodel: Any   # the model the scalar oracles run on
    tree: KinematicTree
    chain: Any    # c_oracle raw body chain
    lo: np.ndarray
    hi: np.ndarray

    @property
    def mid(self):
        return 0.5 * (self.lo + self.hi)


@pytest.fixture(scope="module")
def arms(cuda_lib, tmp_path_factory):
    c_oracle.build()
    out = {}
    for name, xml in (("variant", PANDA_VARIANT), ("general", _GENERAL_MJCF)):
        path = tmp_path_factory.mktemp("trees") / f"{name}.xml"
        path.write_text(xml)
        model = KinematicModel.from_xml_path(str(path))
        omodel = mj_oracle.MjModel.from_xml_path(str(path)) if name == "variant" else model
        chain = c_oracle.chain_from_model(omodel)
        if name == "variant":
            assert bytes(chain) == bytes(c_oracle.chain_from_model(model))  # two independent MJCF compiles agree
        out[name] = Arm(name, model, omodel, KinematicTree.from_mjmodel(model), chain, np.array(chain.lower[:]),
                        np.array(chain.upper[:]))
    return out


@pytest.fixture(params=FOREIGN)
def arm(request, arms):
    """The foreign tree uploaded (AUTO resolves to the generic build); the packaged tree back afterwards."""
    a = arms[request.param]
    try:
        assert engine.set_tree(a.tree) is False
        yield a
    finally:
        engine.set_tree(KinematicTree.from_mjcf())


def gpu(x, dt=torch.float64):
    return torch.as_tensor(np.ascontiguousarray(x, dtype=np.float64), device="cuda").to(dt)


def r32(x):
    return np.asarray(x, dtype=np.float32).astype(np.float64)


def fk(arm, q):
    return c_oracle.fk_jac(arm.chain, q, nthreads=8)[0]


def draw(arm, n, seed, start):
    """q* ~ U(limits), the target FK(q*), the start (cold: mid-range, broadcast; near: clip(q* + U(+-0.3)))."""
    rng = np.random.default_rng(seed)
    q_star = rng.uniform(arm.lo, arm.hi, (n, 7))
    q0 = arm.mid if start == "cold" else np.clip(q_star + rng.uniform(-0.3, 0.3, q_star.shape), arm.lo, arm.hi)
    return q_star, fk(arm, q_star), q0


def batch_size(size):
    sm = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    return 4096 if size == "small" else sm * IK_BLOCK + 4096


# ---------------------------------------------------------------------------------------------------------------------
# FK, Jacobian, quaternion, get_obs
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("prec", ["fp32", "fp64"])
def test_fk_jac_and_obs_over_full_turns(arm, prec):
    """2^16 configurations with q - qref over +-2 pi on every joint: position, Jacobian and site frame vs c_oracle.
    get_obs's end-effector fields (position, velocity J qvel dt) against the same FK: its obs_oracle statement reads
    the Panda scene's object sites, which a bare arm does not have."""
    dt, tol = (torch.float32, 1e-5) if prec == "fp32" else (torch.float64, 1e-12)
    n = 1 << 16
    rng = np.random.default_rng(3)
    q = gpu(arm.tree.qref + rng.uniform(-2 * math.pi, 2 * math.pi, (n, 7)), dt)
    qh = q.double().cpu().numpy()
    assert np.abs(qh - arm.tree.qref).max() > 6.2
    pos, quat, jac = engine.fk_jac(q)
    want_pos, want_mat, want_jac = c_oracle.fk_jac(arm.chain, qh, nthreads=8)
    assert np.abs(pos.double().cpu().numpy() - want_pos).max() < tol
    assert np.abs(jac.double().cpu().numpy() - want_jac).max() < tol
    w, x, y, z = quat.double().cpu().numpy().T
    R = np.stack([1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y),
                  2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x),
                  2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)], axis=1).reshape(n, 3, 3)
    assert np.abs(R - want_mat).max() < 2 * tol
    with pytest.raises(ValueError, match="differs from the build-time"):
        engine.fk_jac(q[:1].contiguous(), kinematics="specialized")
    qvel = rng.uniform(-1.0, 1.0, (n, 7))
    z3 = np.zeros((n, 3))
    obj_quat = np.tile([1.0, 0.0, 0.0, 0.0], (n, 1))
    rows = engine.get_obs(q, gpu(qvel, dt), gpu(np.zeros((n, 2)), dt), gpu(z3, dt), gpu(obj_quat, dt),
                          gpu(np.zeros((n, 6)), dt), gpu([1.0, 0.0, 0.5], dt), dt=0.05)
    rows = rows.double().cpu().numpy()
    qvel = qvel.astype(np.float32).astype(np.float64) if dt == torch.float32 else qvel
    assert np.abs(rows[:, 0:3] - want_pos).max() < tol
    assert np.abs(rows[:, 3:6] - np.einsum("nij,nj->ni", want_jac[:, :3], qvel) * 0.05).max() < tol


# ---------------------------------------------------------------------------------------------------------------------
# Position IK
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("size", ["small", "large"])
@pytest.mark.parametrize("start", ["cold", "near"])
def test_position_ik_fp64_is_iteration_exact(arm, start, size):
    """4096 queries (small-batch path) and sm_count * 128 + 4096 (persistent warps with refill), cold (broadcast
    q_init) and near (per-query q_init): iteration counts of c_oracle.ik_solve but for one threshold tie."""
    q_star, targets, q0 = draw(arm, batch_size(size), seed=11, start=start)
    ref = c_oracle.ik_solve(arm.chain, targets, q0, nthreads=8)
    res = engine.ik_solve(gpu(targets), gpu(q0), engine.ik_params())
    iters = res.iterations.cpu().numpy()
    same = iters == ref["iterations"]
    assert (~same).sum() <= 1
    assert np.array_equal(res.converged.cpu().numpy()[same], ref["converged"][same])
    conv = same & ref["converged"]
    np.testing.assert_allclose(res.q.cpu().numpy()[conv], ref["q"][conv], atol=1e-7)
    np.testing.assert_allclose(res.final_pos.cpu().numpy()[conv], ref["final_pos"][conv], atol=1e-8)
    assert ref["converged"].mean() > 0.97
    if start == "cold":
        assert (~ref["converged"]).sum() >= 20  # both outcomes are tested


@pytest.mark.parametrize("size", ["small", "large"])
@pytest.mark.parametrize("start", ["cold", "near"])
def test_position_ik_fp32_vs_oracle(arm, start, size):
    q_star, targets, q0 = draw(arm, batch_size(size), seed=12, start=start)
    targets, q0 = r32(targets), r32(q0)
    ref = c_oracle.ik_solve(arm.chain, targets, q0, nthreads=8)
    res = engine.ik_solve(gpu(targets, torch.float32), gpu(q0, torch.float32), engine.ik_params())
    flips = int((res.iterations.cpu().numpy() != ref["iterations"]).sum())
    q = res.q.double().cpu().numpy()
    same = res.converged.cpu().numpy() & ref["converged"] & (res.iterations.cpu().numpy() == ref["iterations"])
    rot = _rot_angle(c_oracle.fk_jac(arm.chain, q[same])[1], c_oracle.fk_jac(arm.chain, ref["q"][same])[1])
    print(f"{arm.name} pos {start} {size}: {flips} flips, {(rot >= 1e-3).sum()} orientations > 1e-3 rad apart "
          f"(max {rot.max():.2e}) of {len(targets)}")
    rot_budget = budget(arm.name, "pos_rot", start, size) if (arm.name, "pos_rot", start, size) in OBSERVED else 0
    _compare_with_oracle(res, ref, targets, arm.chain, 1e-3, flip_budget=budget(arm.name, "pos", start, size),
                         rot_budget=rot_budget)


def test_single_query_mailbox_equals_a_batch_of_one(arm):
    """JacobianIKController.solve (ik_solve_one_kernel<false>, the generic branch) and engine.ik_solve on a batch of
    one (ik_solve_kernel<float, GenericKin>) run the same FP32 operations: the same bits, converged or not."""
    ctl = JacobianIKController(arm.model, KinematicData(arm.model))
    assert not ctl.specialized
    _, targets, near = draw(arm, 24, seed=13, start="near")
    starts = [arm.mid if k % 2 else near[k] for k in range(len(targets))]
    cases = [(targets[k], starts[k], {}) for k in range(len(targets))]
    cases += [(targets[k], arm.mid, dict(max_iters=3)) for k in range(4)]              # run out of iterations
    cases += [(np.array([2.5, 0.0, 0.5]), arm.mid, dict(max_iters=20, damping=0.05))]  # unreachable
    n_conv = 0
    for target, q0, kw in cases:
        r = ctl.solve(target, q0, **kw)
        b = engine.ik_solve(gpu(target[None], torch.float32), gpu(q0, torch.float32), engine.ik_params(**kw))
        assert r.iterations == int(b.iterations[0]) and r.converged == bool(b.converged[0]) and r.success == bool(b.success[0])
        np.testing.assert_array_equal(r.q.astype(np.float32), b.q[0].cpu().numpy())
        np.testing.assert_array_equal(r.final_pos.astype(np.float32), b.final_pos[0].cpu().numpy())
        assert np.float32(r.pos_error) == b.pos_error[0].cpu().numpy()
        n_conv += r.converged
    assert 20 <= n_conv < len(cases)


def test_default_restart_seeds_follow_the_uploaded_tree(arm, arms):
    """engine.ik_restart_seeds() without limits draws inside the limits of the tree last uploaded - a foreign tree, a
    controller's, or the packaged one - so that its seeds are starts the solver does not clamp away."""
    kw = dict(dtype=torch.float64, device="cpu")
    seeds = engine.ik_restart_seeds(8, **kw)
    assert torch.equal(seeds, engine.ik_restart_seeds(8, arm.lo, arm.hi, **kw))
    assert bool(((seeds >= torch.as_tensor(arm.lo)) & (seeds <= torch.as_tensor(arm.hi))).all())
    packaged = KinematicTree.from_mjcf()
    engine.set_tree(packaged)
    assert torch.equal(engine.ik_restart_seeds(8, **kw), engine.ik_restart_seeds(8, packaged.lower, packaged.upper, **kw))
    JacobianIKController(arm.model, KinematicData(arm.model))
    assert torch.equal(engine.ik_restart_seeds(8, **kw), seeds)


@pytest.mark.parametrize("prec", ["fp32", "fp64"])
def test_position_multistart(arm, prec):
    """4096 cold targets and 48 unreachable ones with the default seed table (this tree's limits): every row is the
    plain solve from the start its attempt names, bit for bit, and the attempt is that of the CPU replay of the restart
    rule on c_oracle (FP64: but for one threshold tie)."""
    dt = torch.float32 if prec == "fp32" else torch.float64
    packed = dt == torch.float32
    _, targets, _ = draw(arm, 4096, seed=14, start="cold")
    targets = np.concatenate([targets, np.array(FAR * 8)])
    tg, q0 = gpu(targets, dt), gpu(arm.mid, dt)
    seeds = engine.ik_restart_seeds(8, dtype=dt)
    params = engine.ik_params()
    r = engine.ik_solve_multistart(tg, q0, seeds, params, packed=packed)
    attempt, exp, succ = expected(tg, q0, seeds, params, packed)
    got = bits(r)
    for key in exp:
        assert torch.equal(got[key], exp[key]), key
    assert torch.equal(r.attempt.long(), attempt)
    rnd = r32 if dt == torch.float32 else np.asarray
    att_ref, ref = multistart_batched(arm.chain, rnd(targets), rnd(arm.mid), seeds.double().cpu().numpy())
    att = r.attempt.long().cpu().numpy()
    assert (att_ref > 0).sum() >= 20 and not ref["success"][-len(FAR) * 8:].any()
    mism = int((att != att_ref).sum())
    print(f"{arm.name} multistart {prec}: {mism} attempt mismatches, {(att_ref > 0).sum()} rescued")
    assert mism <= (1 if dt == torch.float64 else budget(arm.name, "ms_attempt"))
    if dt == torch.float64:
        same = (att == att_ref) & ref["converged"]
        np.testing.assert_allclose(r.q.cpu().numpy()[same], ref["q"][same], atol=1e-7)


def test_waypoints_vs_chained_oracle_solves(arm):
    """ik_waypoints (FP32) against MoveIKSkill's inner loop replayed on the host with c_oracle solves."""
    n, steps = 48, 50
    rng = np.random.default_rng(15)
    q0 = r32(np.clip(arm.mid + rng.uniform(-0.3, 0.3, (n, 7)), arm.lo, arm.hi))
    goal = r32(fk(arm, np.clip(q0 + rng.uniform(-0.5, 0.5, (n, 7)), arm.lo, arm.hi)))
    out = engine.ik_waypoints(gpu(q0, torch.float32), gpu(goal, torch.float32), steps, engine.ik_params())
    acc_gpu, pos_gpu, q_gpu = (out[k].cpu().numpy() for k in ("n_accepted", "pos", "q"))
    bad = 0
    for e in range(n):
        q, g = q0[e], goal[e]
        pos = fk(arm, q[None])[0]
        accepted = fails = 0
        for _ in range(steps):
            direction = g - pos
            dist = np.linalg.norm(direction)
            if not dist > 0.01:
                break
            step = min(min(0.01, dist * 0.1), 0.02) * (0.5 if fails > 0 else 1.0)
            nxt = pos + direction * step / dist if dist > step else g.copy()
            r = c_oracle.ik_solve(arm.chain, nxt[None], q)
            if r["success"][0] and r["pos_error"][0] < 0.02:
                pos, q, fails = r["final_pos"][0], r["q"][0], 0
                accepted += 1
            else:
                fails += 1
        if acc_gpu[e] != accepted or np.abs(pos_gpu[e] - pos).max() > 5e-5:
            bad += 1
            continue
        np.testing.assert_allclose(q_gpu[e], q, atol=2e-3)
    assert int(acc_gpu.sum()) > 10 * n
    print(f"{arm.name} waypoints: {bad} of {n} envs differ")
    assert bad <= budget(arm.name, "waypoints")


# ---------------------------------------------------------------------------------------------------------------------
# Pose IK
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("prec", ["fp32", "fp64"])
def test_pose_one_evaluation_probe(arm, prec):
    """max_iters = 0 on 64 k frames of this tree (test_gpu_pose_ik's probe): FK, ee_rot, mat2quat and quat2vel at q."""
    dtype = torch.float32 if prec == "fp32" else torch.float64
    q, pos, tq = _probe_inputs(arm.chain)
    got = _solve(arm.tree, dtype, "auto", pos, tq, q, max_iters=0)
    qr, posr, tqr = _rounded(dtype, q, pos, tq)
    ref = pose_ik_oracle.pose_eval_batch(arm.chain, qr, posr, tqr)
    assert (got["iterations"] == 0).all() and not got["converged"].any()
    assert np.array_equal(_bits(got["q"]), _bits(q.astype(got["q"].dtype)))
    _assert_cases(ref["case"])
    if dtype == torch.float32:
        tol_p, tol_q, tol_r, sign_margin = FP32_POS_TOL, FP32_QUAT_TOL, FP32_ROT_TOL, SIGN_MARGIN
    else:
        tol_p, tol_q, tol_r, sign_margin = 1e-12, 1e-12, 1e-11, 1e-12
    assert np.abs(got["final_pos"] - ref["final_pos"]).max() < tol_p
    assert np.abs(got["pos_error"] - ref["pos_error"]).max() < tol_p
    _assert_quat(got["final_quat"], ref["final_quat"], ref["case_margin"], tol_q, sign_margin)
    assert np.abs(got["rot_error"] - ref["rot_error"]).max() < tol_r


def pose_workspace(arm, n, seed, start):
    q_star, _, q0 = draw(arm, n, seed, start)
    ev = pose_ik_oracle.pose_eval_batch(arm.chain, q_star, np.zeros(3), np.array([1.0, 0.0, 0.0, 0.0]))
    return ev["final_pos"], ev["final_quat"], ev["case"], np.broadcast_to(q0, q_star.shape)


@pytest.mark.parametrize("start", ["cold", "near"])
def test_pose_ik_fp64_is_iteration_exact(arm, start):
    pos, quat, case, q0 = pose_workspace(arm, 2048, seed=16, start=start)
    _assert_cases(case)
    got = _solve(arm.tree, torch.float64, "auto", pos, quat, q0)
    ref = _statement(arm.chain, torch.float64, pos, quat, q0)
    _check_fp64(arm.chain, got, ref, pos, quat)
    assert ref["converged"].mean() > (0.95 if start == "near" else 0.4)


@pytest.mark.parametrize("start", ["cold", "near"])
def test_pose_ik_fp32_vs_statement(arm, start):
    pos, quat, case, q0 = pose_workspace(arm, 2048, seed=17, start=start)
    got = _solve(arm.tree, torch.float32, "auto", pos, quat, q0)
    ref = _statement(arm.chain, torch.float32, pos, quat, q0)
    pos32, quat32 = _rounded(torch.float32, pos, quat)
    same = got["converged"] & ref["converged"] & (got["iterations"] == ref["iterations"])
    n_dq = int((np.abs(got["q"].astype(np.float64)[same] - ref["q"][same]).max(axis=1, initial=0.0) > 2e-5).sum())
    flips = int((got["iterations"] != ref["iterations"]).sum())
    print(f"{arm.name} pose {start}: {flips} flips, {n_dq} |dq| > 2e-5 of {len(pos)}")
    dq_cap = 2 * POSE_DQ_MAX_OBSERVED.get((arm.name, start), 5e-4)
    _check_fp32(arm.chain, got, ref, pos32, quat32, budget=budget(arm.name, "pose", start),
                q_budget=budget(arm.name, "pose_dq", start), dq_cap=dq_cap)


@pytest.mark.parametrize("prec", ["fp32", "fp64"])
def test_pose_multistart(arm, prec):
    """512 cold pose queries, four seeds from this tree's limits: every row is the plain pose solve from the start its
    attempt names, bit for bit; FP64 attempts are those of the restart rule replayed on the statement."""
    dtype = torch.float32 if prec == "fp32" else torch.float64
    pos, quat, _, q0 = pose_workspace(arm, 512, seed=18, start="cold")
    seeds = engine.ik_restart_seeds(4, dtype=torch.float64, device="cpu").numpy()
    out = engine.ik_pose_solve_multistart(gpu(pos, dtype), gpu(quat, dtype), gpu(arm.mid, dtype), gpu(seeds, dtype),
                                          engine.ik_params())
    got = {k: v.cpu().numpy() for k, v in out.items()}
    runs = [_solve(arm.tree, dtype, "auto", pos, quat, arm.mid)] + [_solve(arm.tree, dtype, "auto", pos, quat, s) for s in seeds]
    succ = np.stack([r["success"] for r in runs])
    first = np.where(succ.any(axis=0), np.argmax(succ, axis=0), 0)
    assert np.array_equal(got["attempt"], first) and (first > 0).sum() >= 20
    for key in runs[0]:
        want = np.stack([r[key] for r in runs])[first, np.arange(len(pos))]
        assert np.array_equal(_bits(got[key]), _bits(want)), key
    if dtype == torch.float64:
        att = np.zeros(len(pos), dtype=np.int64)
        left = np.nonzero(~_statement(arm.chain, dtype, pos, quat, q0)["success"])[0]
        for k, s in enumerate(seeds):
            ok = _statement(arm.chain, dtype, pos[left], quat[left], s)["success"]
            att[left[ok]] = k + 1
            left = left[~ok]
        assert int((att != got["attempt"]).sum()) <= 1


# ---------------------------------------------------------------------------------------------------------------------
# Position planner
# ---------------------------------------------------------------------------------------------------------------------
PLAN_SETTINGS = {
    "default": (dict(), dict(max_outer=300, traj_cap=256)),
    "fallback": (dict(max_iters=1, pos_thresh=8e-4), dict(step_size=0.05, max_outer=200, traj_cap=256)),
}


def plan_workload(arm, n, seed):
    """Start mid-range +- 0.3 rad, goal FK(start +- 0.6 rad); every 64th goal 1.5 m out of reach."""
    rng = np.random.default_rng(seed)
    q0 = np.clip(arm.mid + rng.uniform(-0.3, 0.3, (n, 7)), arm.lo, arm.hi)
    goal = fk(arm, np.clip(q0 + rng.uniform(-0.6, 0.6, (n, 7)), arm.lo, arm.hi))
    goal[::64] += np.array([1.5, 0.0, 0.0])
    return q0, goal


def oracle_plan(arm, q0, goal, ik, mv):
    okw = dict(max_iters=ik.get("max_iters", 100), ik_pos_thresh=ik.get("pos_thresh", 1e-3))
    return c_oracle.move_plan(arm.chain, q0, goal, nthreads=8, **okw, **mv)


@pytest.mark.parametrize("setting", list(PLAN_SETTINGS))
def test_move_plan_fp64_vs_oracle(arm, setting):
    ik, mv = PLAN_SETTINGS[setting]
    q0, goal = plan_workload(arm, 1024, seed=19)
    out = engine.move_ik_plan(gpu(q0), gpu(goal), engine.ik_params(**ik), **mv)
    ref = oracle_plan(arm, q0, goal, ik, mv)
    st, tl, ns = (out[k].cpu().numpy() for k in ("status", "traj_len", "n_solves"))
    same = (st == ref["status"]) & (tl == ref["traj_len"]) & (ns == ref["n_solves"])
    assert (~same).sum() <= 2, np.nonzero(~same)[0][:10]
    traj = out["traj"].cpu().numpy()
    for k in np.nonzero(same)[0]:
        L = min(int(tl[k]), mv["traj_cap"])
        np.testing.assert_allclose(traj[k, :L], ref["traj"][k, :L], atol=1e-8)
    if setting == "default":
        assert (ref["status"] == 0).sum() > 900 and (ref["status"] & 2).sum() >= 10
    else:
        assert (ref["status"] & 1).sum() > 300 and (ref["status"] & 2).sum() > 100


def test_move_plan_fp32_holds_the_invariants(arm):
    """FP32 plans (default setting): status as the FP64 oracle's on the FP32-rounded inputs but for a counted few; the
    trajectory starts at FK(q_start); steps between accepted points stay within step_size + the accept tolerance; a
    finished plan ends within pos_thresh of the goal; q_final reproduces the last accepted point under FP64 FK; the
    solve counter equals the per-env counts."""
    ik, mv = PLAN_SETTINGS["default"]
    q0, goal = (r32(a) for a in plan_workload(arm, 1024, seed=20))
    cnt = torch.zeros(4, dtype=torch.int64, device="cuda")
    out = engine.move_ik_plan(gpu(q0, torch.float32), gpu(goal, torch.float32), engine.ik_params(), counters=cnt, **mv)
    ref = oracle_plan(arm, q0, goal, ik, mv)
    st, L = out["status"].cpu().numpy(), out["traj_len"].cpu().numpy().astype(np.int64)
    traj = out["traj"].double().cpu().numpy()
    n_bad = int((st != ref["status"]).sum())
    print(f"{arm.name} fp32 planner: {n_bad} status mismatches of {len(st)}")
    assert n_bad <= budget(arm.name, "plan_status")
    assert int(cnt[0]) == int(out["n_solves"].sum())
    assert ((st & ~7) == 0).all() and L.min() >= 1 and L.max() <= mv["traj_cap"]
    assert np.abs(traj[:, 0] - fk(arm, q0)).max() < 1e-5
    idx = np.arange(traj.shape[1])[None, :]
    seg = np.linalg.norm(traj[:, 1:] - traj[:, :-1], axis=2)
    assert seg[idx[:, 1:] < (L[:, None] - 1)].max() < 0.01 + 0.02 + 1e-4
    last = traj[np.arange(len(L)), L - 1]
    ok = st == 0
    assert np.linalg.norm(last[ok] - goal[ok], axis=1).max() <= 0.01 + 1e-5
    appended = (last == goal).all(axis=1) & (L > 1)
    prev = traj[np.arange(len(L)), np.maximum(L - 2, 0)]
    last_accepted = np.where(appended[:, None], prev, last)
    assert np.abs(fk(arm, out["q_final"].double().cpu().numpy()) - last_accepted).max() < 2e-5


@pytest.mark.parametrize("prec", ["fp32", "fp64"])
def test_move_plan_longest_first_order_at_2_16(arm, prec):
    """From 2^16 envs up "auto" orders the plans by |goal - FK(q_start)| (FP32: the gathered-input kernel, FP64:
    PnpMoveParams.compute_order), with the generic FK: the order must follow the oracle's distances, and the plans must
    be bit-identical to index order.  The first 128 FP64 plans are checked against c_oracle as well."""
    dt = torch.float32 if prec == "fp32" else torch.float64
    n = engine.PLAN_ORDER_MIN
    q0, goal = plan_workload(arm, n, seed=21)
    qs, gl = gpu(q0, dt), gpu(goal, dt)
    mv = dict(max_outer=40, traj_cap=64)
    a = engine.move_ik_plan(qs, gl, engine.ik_params(), **mv)
    b = engine.move_ik_plan(qs, gl, engine.ik_params(), order=None, **mv)
    assert ("_scratch48" in a) == (dt == torch.float32)
    for f in ("traj_len", "n_solves", "status", "q_final"):
        assert torch.equal(a[f], b[f]), f
    mask = torch.arange(mv["traj_cap"], device="cuda")[None, :] < a["traj_len"].long().clamp(max=mv["traj_cap"])[:, None]
    assert torch.equal(a["traj"][mask], b["traj"][mask])
    order = engine.move_plan_order(qs, gl).cpu().numpy().astype(np.int64)
    assert np.array_equal(np.sort(order), np.arange(n))
    p0 = engine.fk_jac(qs, want_quat=False, want_jac=False)[0]  # the kernels' own FK, held to c_oracle above
    d0 = (gl - p0).norm(dim=1).cpu().numpy()[order]
    bucket = np.minimum((d0 * 64.0).astype(np.int64), 127)
    assert np.all(np.diff(bucket) <= 1) and np.all(np.diff(bucket.astype(np.float64)).cumsum() <= 1)
    if dt == torch.float64:
        m = 128
        ref = oracle_plan(arm, q0[:m], goal[:m], {}, mv)
        same = (a["traj_len"][:m].cpu().numpy() == ref["traj_len"]) & (a["status"][:m].cpu().numpy() == ref["status"])
        assert (~same).sum() <= 1


# ---------------------------------------------------------------------------------------------------------------------
# Pose planner
# ---------------------------------------------------------------------------------------------------------------------
POSE_PLAN_POINTS = 60  # bounds the scalar statement's cost on the moves that creep along a limit


def pose_plan_workload(arm, n, seed):
    rng = np.random.default_rng(seed)
    q0 = np.clip(arm.mid + rng.uniform(-0.05, 0.05, (n, 7)), arm.lo, arm.hi)
    qg = np.clip(q0 + rng.uniform(-0.6, 0.6, (n, 7)), arm.lo, arm.hi)
    ev = pose_ik_oracle.pose_eval_batch(arm.chain, qg, np.zeros(3), np.array([1.0, 0.0, 0.0, 0.0]))
    return q0, ev["final_pos"], ev["final_quat"]


def test_pose_planner_fp64_vs_statement(arm):
    n = 48
    q0, gp, gq = pose_plan_workload(arm, n, seed=22)
    got = host(engine.move_ik_plan_pose(gpu(q0), gpu(gp), gpu(gq), engine.ik_params(), max_traj_points=POSE_PLAN_POINTS))
    bad, status = 0, []
    for k in range(n):
        w = move_pose_oracle.plan_pose(arm.omodel, q0[k], gp[k], gq[k], max_traj_points=POSE_PLAN_POINTS)
        status.append(w["status"])
        L = len(w["pos_traj"])
        if (int(got["traj_len"][k]), int(got["status"][k]), int(got["n_solves"][k])) != (L, w["status"], w["n_solves"]):
            bad += 1
            continue
        for key in ("pos_traj", "quat_traj", "q_traj"):
            np.testing.assert_allclose(got[key][k, :L], w[key], rtol=0, atol=1e-9, err_msg=key)
        np.testing.assert_allclose(got["q_final"][k], w["q_final"], rtol=0, atol=1e-9)
    status = np.array(status)
    print(f"{arm.name} pose planner statement: status counts {np.bincount(status, minlength=3)}")
    assert bad <= 1 and (status == 0).sum() >= n // 2


def test_pose_planner_fp32_holds_the_invariants(arm):
    n = 1024
    q0, gp, gq = pose_plan_workload(arm, n, seed=23)
    a = host(engine.move_ik_plan_pose(gpu(q0, torch.float32), gpu(gp, torch.float32), gpu(gq, torch.float32),
                                      engine.ik_params(), max_traj_points=POSE_PLAN_POINTS))
    b = host(engine.move_ik_plan_pose(gpu(q0), gpu(gp), gpu(gq), engine.ik_params(), max_traj_points=POSE_PLAN_POINTS))
    agree = float((a["status"] == b["status"]).mean())
    print(f"{arm.name} pose planner fp32 vs fp64: status agreement {agree:.4f}, OK {(a['status'] == 0).mean():.4f}")
    assert agree > 0.95 and (a["status"] == 0).mean() > 0.5
    for k in range(n):
        L = int(a["traj_len"][k])
        qt = a["q_traj"][k, :L]
        assert (qt >= arm.lo - 1e-6).all() and (qt <= arm.hi + 1e-6).all()
        # the FP32 kernel clamps to the limits rounded to float, up to one float ulp outside (GENERAL's -90 degrees)
        plan = dict(pos_traj=a["pos_traj"][k, :L], quat_traj=a["quat_traj"][k, :L], q_traj=np.clip(qt, arm.lo, arm.hi),
                    n_solves=int(a["n_solves"][k]), status=int(a["status"][k]))
        check_invariants(arm.model, arm.chain, plan, gp[k], gq[k], 1e-5, 1e-4)
        assert np.array_equal(a["q_final"][k], a["q_traj"][k, L - 1])


# ---------------------------------------------------------------------------------------------------------------------
# The packaged Panda a few ulp off
# ---------------------------------------------------------------------------------------------------------------------
def panda_ulp():
    """The packaged tree with every double of link_pos, link_rot, ee_pos and ee_rot moved 1-3 ulp (seeded walk)."""
    t = KinematicTree.from_mjcf()
    rng = np.random.default_rng(24)

    def walk(a):
        a = np.array(a, dtype=np.float64)
        flat = a.reshape(-1)
        for i in range(flat.size):
            toward = np.inf if rng.random() < 0.5 else -np.inf
            for _ in range(int(rng.integers(1, 4))):
                flat[i] = np.nextafter(flat[i], toward)
        return a

    u = KinematicTree(link_pos=walk(t.link_pos), link_rot=walk(t.link_rot), ee_pos=walk(t.ee_pos),
                      ee_rot=walk(t.ee_rot), lower=t.lower.copy(), upper=t.upper.copy(), qref=t.qref.copy())
    for f in ("link_pos", "link_rot", "ee_pos", "ee_rot"):
        d = np.abs(getattr(u, f) - getattr(t, f))
        assert (d > 0).all() and (d <= 6 * np.spacing(np.abs(getattr(t, f)))).all(), f
    return u


@pytest.mark.parametrize("prec", ["fp32", "fp64"])
def test_panda_a_few_ulp_off_runs_generic_like_specialised(cuda_lib, oracle_chain, prec):
    """Today the tree match is exact, so AUTO runs the generic build on a tree a few ulp off the packaged one.  Its
    results must be those of the specialised build: FP64 both iteration-exact against c_oracle on the packaged chain,
    FP32 both within test_gpu_ik's cfg2 flip budget (position) and test_gpu_pose_ik's W-near budget (pose)."""
    dt = torch.float32 if prec == "fp32" else torch.float64
    packaged, ulp = KinematicTree.from_mjcf(), panda_ulp()
    qstar = synthetic.random_joint_configs(4096, packaged.lower, packaged.upper, seed=0, dtype=torch.float64).numpy()
    targets = c_oracle.fk_jac(oracle_chain, qstar, nthreads=8)[0]
    w_star, w_pos, w_quat, _, rng = _workspace(oracle_chain, 4096, seed=41)  # test_gpu_pose_ik's FP32 W-near batch
    near = _start(oracle_chain, w_star, rng, "near")
    results = {}
    try:
        for name, tree in (("specialised", packaged), ("generic", ulp)):
            if name == "specialised":
                assert engine.set_tree(tree) is True
            else:
                assert engine.set_tree(tree) is False  # exact match only: a tolerant match makes this `is True`
                with pytest.raises(ValueError, match="differs from the build-time"):
                    engine.fk_jac(torch.zeros((1, 7), dtype=dt, device="cuda"), kinematics="specialized")
            pos_res = engine.ik_solve(gpu(targets, dt), gpu(NEUTRAL, dt), engine.ik_params())
            pose_res = _solve(tree, dt, "auto", w_pos, w_quat, near) if dt == torch.float32 else None
            results[name] = pos_res, pose_res
    finally:
        engine.set_tree(KinematicTree.from_mjcf())
    rnd = r32 if dt == torch.float32 else np.asarray
    ref = c_oracle.ik_solve(oracle_chain, rnd(targets), NEUTRAL, nthreads=8)
    if dt == torch.float32:
        pose_ref = _statement(oracle_chain, dt, w_pos, w_quat, near)
        pos32, quat32 = _rounded(dt, w_pos, w_quat)
    for name, (res, pose) in results.items():
        if dt == torch.float64:
            iters = res.iterations.cpu().numpy()
            assert (iters != ref["iterations"]).sum() <= 1, name
            conv = (iters == ref["iterations"]) & ref["converged"]
            np.testing.assert_allclose(res.q.cpu().numpy()[conv], ref["q"][conv], atol=1e-7)
            np.testing.assert_allclose(res.final_pos.cpu().numpy()[conv], ref["final_pos"][conv], atol=1e-8)
        else:
            _compare_with_oracle(res, ref, r32(targets), oracle_chain, 1e-3, flip_budget=8)
            _check_fp32(oracle_chain, pose, pose_ref, pos32, quat32, budget=2)

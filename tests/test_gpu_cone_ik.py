"""GPU: cone-tolerant axis IK (pnp_ik_axis_cone_solve_*, engine.ik_axis_solve(cone_angle=...),
JacobianIKController.solve_axis(cone_angle=...)) against its FP64 statement (oracle/cone_ik_oracle.py).

Workloads and checkers are test_gpu_axis_ik.py's: A-near / A-cold targets (FK(q*), R(q*) t), the FP64 kernel held to
the batched statement iteration for iteration, the FP32 kernel to counted iteration flips and to its q re-evaluated
with the FP64 FK.  The cone's two ends are held to the axis and the position kernels, and the multistart to
bit-identity with the plain cone solve from the attempt it names."""
import ctypes
import math

import numpy as np
import pytest
import torch

from conftest import NEUTRAL
from mujoco_panda_pnp_b200 import KinematicData, _lib, engine, synthetic
from mujoco_panda_pnp_b200.skills import JacobianIKController
from oracle import c_oracle, cone_ik_oracle
from test_gpu_axis_ik import (DEFAULTS, DTYPES, IK_BLOCK, KEYS, KINS, OBLIQUE, Z, _bits, _ik, _outs, _rounded, _tbits,
                              _tool, assert_rows, check_fp32, check_fp64, expected, ms_workload, tree, workload)  # noqa: F401
from test_gpu_foreign_trees import arm, arms, gpu  # noqa: F401  (fixtures of the foreign arms)

pytestmark = pytest.mark.gpu

DEG = math.pi / 180.0


def solve(dtype, kin, pos, ax, q_init, alpha, tool=Z, counters=None, **p):
    p = dict(DEFAULTS, **p)
    out = engine.ik_axis_solve(gpu(pos, dtype), gpu(ax, dtype), gpu(q_init, dtype),
                               engine.ik_params(kinematics=kin, **_ik(p)), tool_axis=tool, rot_thresh=p["rot_thresh"],
                               rot_weight=p["rot_weight"], counters=counters, cone_angle=alpha)
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in out.items()}


def statement(chain, dtype, pos, ax, q_init, alpha, tool=Z, **p):
    pos, ax, q_init = _rounded(dtype, pos, ax, q_init)
    return cone_ik_oracle.solve_cone_batch(chain, pos, ax, q_init, alpha, tool_axis=tool, **dict(DEFAULTS, **p))


def check_fp32_cone(chain, got, ref, pos, ax, alpha, **kw):
    """check_fp32 with the converged rows' axis bound moved out by the cone: theta < alpha + rot_thresh."""
    check_fp32(chain, got, ref, pos, ax, rot_thresh=alpha + DEFAULTS["rot_thresh"], **kw)


def raw_solve(dtype, kin, tp, ta, qi, stride, n, outs, counters, alpha, tool=Z, rot_thresh=1e-2, rot_weight=1.0):
    """pnp_ik_axis_cone_solve_* through the C ABI; outs as _outs, any entry None."""
    lib = _lib.load()
    fn = lib.pnp_ik_axis_cone_solve_f32 if dtype == torch.float32 else lib.pnp_ik_axis_cone_solve_f64
    ptr = [None if t is None else t.data_ptr() for t in outs]
    return fn(None if tp is None else tp.data_ptr(), ta.data_ptr(), qi.data_ptr(), stride, n,
              ctypes.byref(engine.ik_params(kinematics=kin)), _tool(tool), rot_thresh, alpha, rot_weight, *ptr,
              None if counters is None else counters.data_ptr(), torch.cuda.current_stream().cuda_stream)


# ---------------------------------------------------------------------------------------------------------------------
# Plain solve against the statement and against its two ends
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kin", KINS)
@pytest.mark.parametrize("start", ["near", "cold"])
@pytest.mark.parametrize("deg", [10, 30])
def test_fp64_is_iteration_exact(tree, oracle_chain, deg, start, kin):
    pos, ax, q0 = workload(oracle_chain, 2048, seed=131, start=start)
    got = solve(torch.float64, kin, pos, ax, q0, deg * DEG)
    ref = statement(oracle_chain, torch.float64, pos, ax, q0, deg * DEG)
    check_fp64(got, ref)
    assert ref["converged"].mean() > (0.95 if start == "near" else 0.85)


@pytest.mark.parametrize("kin", KINS)
@pytest.mark.parametrize("start,n", [("near", 4096), ("cold", 2048)])
def test_fp32_vs_statement(tree, oracle_chain, start, n, kin):
    alpha = 20 * DEG
    pos, ax, q0 = workload(oracle_chain, n, seed=141, start=start)
    got = solve(torch.float32, kin, pos, ax, q0, alpha)
    ref = statement(oracle_chain, torch.float32, pos, ax, q0, alpha)
    pos32, ax32 = _rounded(torch.float32, pos, ax)
    check_fp32_cone(oracle_chain, got, ref, pos32, ax32, alpha, budget=4 if start == "near" else 16,
                    q_budget=8 if start == "near" else 60, dq_cap=5e-3 if start == "near" else 2e-2)
    assert got["converged"].mean() > (0.95 if start == "near" else 0.85)


@pytest.mark.parametrize("kin", KINS)
def test_zero_cone_is_the_axis_solve(tree, oracle_chain, kin):
    pos, ax, q0 = workload(oracle_chain, 2048, seed=151, start="cold")
    cone = solve(torch.float64, kin, pos, ax, q0, 0.0)
    axis = solve(torch.float64, kin, pos, ax, q0, None)
    assert np.array_equal(cone["iterations"], axis["iterations"])
    assert np.array_equal(cone["converged"], axis["converged"]) and np.array_equal(cone["success"], axis["success"])
    assert np.abs(cone["q"] - axis["q"]).max() < 1e-9


@pytest.mark.parametrize("kin", KINS)
def test_pi_cone_is_the_position_solve(tree, oracle_chain, kin):
    pos, ax, q0 = workload(oracle_chain, 2048, seed=161, start="cold")
    cone = solve(torch.float64, kin, pos, ax, q0, math.pi)
    r = engine.ik_solve(gpu(pos), gpu(q0), engine.ik_params(kinematics=kin))
    torch.cuda.synchronize()
    assert np.array_equal(cone["iterations"], r.iterations.cpu().numpy())
    assert np.array_equal(cone["converged"], r.converged.cpu().numpy())
    assert np.abs(cone["q"] - r.q.cpu().numpy()).max() < 1e-9
    assert cone["converged"].mean() > 0.9


# ---------------------------------------------------------------------------------------------------------------------
# Layout, replay, degenerate axes, rejected arguments
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kin", KINS)
@pytest.mark.parametrize("prec", ["fp32", "fp64"])
def test_results_do_not_depend_on_batch_shape(tree, oracle_chain, prec, kin):
    """32 witness queries one at a time, as one batch (small-batch path), and at scattered rows of batches of
    sm_count * IK_BLOCK + 1 and 2^18 queries (persistent warps with lane refill): bit-identical.  A broadcast q_init
    gives the bits of a per-row one."""
    dtype, alpha = DTYPES[prec], 15 * DEG
    engine.set_tree(tree)
    sm = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    pos, ax, q0 = workload(oracle_chain, 4096, seed=171, start="cold")
    rng = np.random.default_rng(172)
    w = rng.choice(4096, 32, replace=False)
    ref = solve(dtype, kin, pos[w], ax[w], q0[w], alpha)
    for k in range(32):
        one = solve(dtype, kin, pos[w[k]:w[k] + 1], ax[w[k]:w[k] + 1], q0[w[k]:w[k] + 1], alpha)
        for key in KEYS:
            assert np.array_equal(_bits(one[key][0]), _bits(ref[key][k])), (k, key)
    bc = solve(dtype, kin, pos[w], ax[w], NEUTRAL, alpha)
    for key in KEYS:
        assert np.array_equal(_bits(bc[key]), _bits(ref[key])), key
    pool = [gpu(a, dtype) for a in (pos, ax, q0)]
    for n in (sm * IK_BLOCK + 1, 1 << 18):
        idx = rng.integers(0, 4096, n)
        slots = rng.choice(n, 32, replace=False)
        idx[slots] = w
        it = torch.as_tensor(idx, device="cuda")
        tp, ta, qi = (a[it].contiguous() for a in pool)
        outs = _outs(n, dtype)
        counters = torch.zeros(4, dtype=torch.int64, device="cuda")
        _lib.check(raw_solve(dtype, kin, tp, ta, qi, 7, n, outs, counters, alpha), "pnp_ik_axis_cone_solve")
        torch.cuda.synchronize()
        q, fpos, fax, fquat, perr, aerr, iters, flags = outs
        conv, succ = (flags & 1) != 0, (flags & 2) != 0
        assert counters.tolist() == [n, int(conv.sum()), int(succ.sum()), int(iters.long().sum())]
        got = dict(zip(KEYS, (q, fpos, fax, fquat, perr, aerr, iters, conv, succ)))
        for key in KEYS:
            assert np.array_equal(_bits(got[key][slots].cpu().numpy()), _bits(ref[key])), (n, key)


def test_graph_capture_replays_on_new_inputs(tree, oracle_chain):
    n, alpha = 1 << 14, 20 * DEG
    pos, ax, _ = workload(oracle_chain, n, seed=181, start="cold")
    tp, ta = gpu(pos, torch.float32), gpu(ax, torch.float32)
    q0 = torch.tensor(NEUTRAL, dtype=torch.float32, device="cuda")
    outs = _outs(n, torch.float32)
    counters = torch.zeros(4, dtype=torch.int64, device="cuda")

    def call():
        _lib.check(raw_solve(torch.float32, "auto", tp, ta, q0, 0, n, outs, counters, alpha), "pnp_ik_axis_cone_solve")

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        call()
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        call()
    pos2, ax2, _ = workload(oracle_chain, n, seed=182, start="cold")
    tp.copy_(gpu(pos2, torch.float32)), ta.copy_(gpu(ax2, torch.float32))
    counters.zero_()
    g.replay()
    torch.cuda.synchronize()
    c2 = torch.zeros(4, dtype=torch.int64, device="cuda")
    r = engine.ik_axis_solve(gpu(pos2, torch.float32), gpu(ax2, torch.float32), q0, engine.ik_params(), counters=c2,
                             cone_angle=alpha)
    torch.cuda.synchronize()
    for key, t in zip(KEYS[:7], outs[:7]):
        assert torch.equal(t.view(torch.uint8), r[key].contiguous().view(torch.uint8)), key
    assert torch.equal(outs[7], r["converged"].to(torch.uint8) | (r["success"].to(torch.uint8) << 1))
    assert torch.equal(counters, c2)


@pytest.mark.parametrize("kin", KINS)
@pytest.mark.parametrize("prec", ["fp32", "fp64"])
def test_degenerate_axes(tree, oracle_chain, prec, kin):
    """A zero or NaN target axis runs to max_iters unconverged (its passes are position passes) and leaves its
    neighbours untouched."""
    dtype, alpha = DTYPES[prec], 20 * DEG
    pos, ax, q0 = workload(oracle_chain, 256, seed=191, start="near")
    at = np.array([0, 37, 130, 255])
    pos2, ax2, q2 = (np.insert(a, at, a[at], axis=0) for a in (pos, ax, q0))
    bad = np.zeros(len(pos2), dtype=bool)
    bad[at + np.arange(len(at))] = True
    ax2[bad] = [[0.0, 0.0, 0.0], [np.nan, 0.0, 1.0], [np.nan] * 3, [0.0, 0.0, 0.0]]
    got = solve(dtype, kin, pos2, ax2, q2, alpha, max_iters=40)
    assert not got["converged"][bad].any() and not got["success"][bad].any()
    assert (got["iterations"][bad] == 40).all() and np.isfinite(got["q"]).all()
    clean = solve(dtype, kin, pos, ax, q0, alpha, max_iters=40)
    for key in clean:
        assert np.array_equal(_bits(got[key][~bad]), _bits(clean[key])), key
    if dtype == torch.float64:
        ref = statement(oracle_chain, dtype, pos2[bad], ax2[bad], q2[bad], alpha, max_iters=40)
        assert np.abs(got["q"][bad] - ref["q"]).max() < 1e-9


@pytest.mark.parametrize("prec", ["fp32", "fp64"])
def test_rejected_arguments_leave_outputs_untouched(tree, oracle_chain, prec, cuda_lib):
    dtype = DTYPES[prec]
    n = 256
    pos, ax, q0 = (gpu(a, dtype) for a in workload(oracle_chain, n, seed=195, start="near"))
    outs = _outs(n, dtype, 7.0)
    before = [t.clone() for t in outs]
    bad = (float("nan"), -1e-12, -1.0, math.pi * (1 + 1e-15), 4.0, float("inf"))
    for alpha in bad:
        assert raw_solve(dtype, "auto", pos, ax, q0, 7, n, outs, None, alpha) == -1, alpha
    for c in (dict(tool=None), dict(rot_thresh=0.0), dict(rot_weight=float("nan"))):
        assert raw_solve(dtype, "auto", pos, ax, q0, 7, n, outs, None, 0.1, **c) == -1, c
    assert raw_solve(dtype, "auto", None, ax, q0, 7, n, outs, None, 0.1) == -1
    # the multistart rejects the same angles before its first launch
    nb = ctypes.c_int64()
    assert cuda_lib.pnp_ik_multistart_scratch_bytes(n, ctypes.byref(nb)) == 0
    scratch = torch.zeros(nb.value // 4 + 8, dtype=torch.int32, device="cuda")
    seeds = engine.ik_restart_seeds(4, dtype=dtype)
    attempt = torch.full((n,), 9, dtype=torch.uint8, device="cuda")
    fn = cuda_lib.pnp_ik_axis_cone_solve_multistart_f32 if dtype == torch.float32 else \
        cuda_lib.pnp_ik_axis_cone_solve_multistart_f64
    for alpha in bad:
        rc = fn(pos.data_ptr(), ax.data_ptr(), q0.data_ptr(), 7, n, seeds.data_ptr(), 4, ctypes.byref(engine.ik_params()),
                _tool(), 1e-2, alpha, 1.0, *(t.data_ptr() for t in outs), attempt.data_ptr(), None, None,
                scratch.data_ptr(), torch.cuda.current_stream().cuda_stream)
        assert rc == -1, alpha
    torch.cuda.synchronize()
    for a, b in zip(outs, before):
        assert torch.equal(a, b)
    assert bool((attempt == 9).all())
    assert raw_solve(dtype, "auto", pos, ax, q0, 7, n, outs, None, 0.0) == 0
    assert raw_solve(dtype, "auto", pos, ax, q0, 7, n, outs, None, math.pi) == 0
    with pytest.raises(ValueError):
        engine.ik_axis_solve(pos, ax, q0, engine.ik_params(), cone_angle=-0.5)


# ---------------------------------------------------------------------------------------------------------------------
# Foreign arms, restarts, the controller and the measured gain
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("start", ["cold", "near"])
def test_foreign_arm_vs_statement(arm, start):  # noqa: F811
    alpha = 20 * DEG
    rng = np.random.default_rng(26)
    q_star = rng.uniform(arm.lo, arm.hi, (2048, 7))
    p, mat, _ = c_oracle.fk_jac(arm.chain, q_star, nthreads=8)
    ax = mat[:, :, 2]
    q0 = np.broadcast_to(arm.mid, q_star.shape) if start == "cold" else \
        np.clip(q_star + rng.uniform(-0.3, 0.3, q_star.shape), arm.lo, arm.hi)
    got = solve(torch.float64, "auto", p, ax, q0, alpha)
    check_fp64(got, statement(arm.chain, torch.float64, p, ax, q0, alpha))
    assert got["converged"].mean() > (0.95 if start == "near" else 0.5)
    got32 = solve(torch.float32, "auto", p, ax, q0, alpha)
    ref32 = statement(arm.chain, torch.float32, p, ax, q0, alpha)
    p32, ax32 = _rounded(torch.float32, p, ax)
    check_fp32_cone(arm.chain, got32, ref32, p32, ax32, alpha, budget=16, q_budget=80, dq_cap=2e-2)


@pytest.mark.parametrize("kin", KINS)
@pytest.mark.parametrize("prec", ["fp32", "fp64"])
@pytest.mark.parametrize("tool", ["z", "oblique"])
def test_multistart_rows_are_plain_solves(tree, oracle_chain, prec, kin, tool):
    dt, alpha = DTYPES[prec], 20 * DEG
    t = Z if tool == "z" else OBLIQUE
    tp, ta = ms_workload(oracle_chain, 1 << 13, dt, seed=4321)
    box = np.array(synthetic.SHELF_BOX)  # shelf-horizontal reaches: the cone's own hard case
    ps = box[:, 0] + (box[:, 1] - box[:, 0]) * np.random.default_rng(3).random((2048, 3))
    tp = torch.cat([tp, gpu(ps, dt)])
    ta = torch.cat([ta, gpu(np.tile([1.0, 0.0, 0.0], (2048, 1)), dt)])
    q0 = torch.tensor(NEUTRAL, dtype=dt, device="cuda")
    seeds = engine.ik_restart_seeds(8, dtype=dt)
    params = engine.ik_params(kinematics=kin)
    counters = torch.zeros(4, dtype=torch.int64, device="cuda")
    stats = torch.zeros(3, dtype=torch.int64, device="cuda")
    r = engine.ik_axis_solve_multistart(tp, ta, q0, seeds, params, tool_axis=t, counters=counters, restart_stats=stats,
                                        cone_angle=alpha)
    attempt, exp = expected(tp, ta, q0, seeds, params, tool_axis=t, cone_angle=alpha)
    assert_rows(_tbits(r), exp)
    assert torch.equal(r["attempt"].long(), attempt)
    c = counters.cpu().numpy()
    assert c[0] == len(tp) and c[1] == int(r["converged"].sum()) and c[2] == int(r["success"].sum())
    assert c[3] == int(r["iterations"].long().sum())
    s = stats.cpu().numpy()
    assert s[1] == int((attempt > 0).sum()) and s[1] > 50


def test_controller_solve_axis_with_a_cone(tree, oracle_chain, kin_model):
    data = KinematicData(kin_model)
    seeds = engine.ik_restart_seeds(8)
    pos, ax, _ = workload(oracle_chain, 2048, seed=203, start="cold")
    alpha = 15 * DEG
    for precision in ("fp32", "fp64"):
        ctl = JacobianIKController(kin_model, data, precision=precision)
        dt = torch.float32 if precision == "fp32" else torch.float64
        r = ctl.solve_axis(pos, ax, NEUTRAL, cone_angle=alpha)
        e = engine.ik_axis_solve(gpu(pos, dt), gpu(ax, dt), gpu(NEUTRAL, dt), engine.ik_params(), cone_angle=alpha)
        assert_rows(_tbits(r), _tbits(e), what=precision)
        m = ctl.solve_axis(pos, ax, NEUTRAL, cone_angle=alpha, seeds=seeds)
        em = engine.ik_axis_solve_multistart(gpu(pos, dt), gpu(ax, dt), gpu(NEUTRAL, dt), seeds.to(dt),
                                             engine.ik_params(), cone_angle=alpha)
        assert_rows(_tbits(m), _tbits(em), what=precision)
        assert torch.equal(m["attempt"], em["attempt"]) and int(em["attempt"].count_nonzero()) > 10
        exact = ctl.solve_axis(pos, ax, NEUTRAL)
        assert float(r["success"].float().mean()) > float(exact["success"].float().mean())


def test_cone_solves_more_shelf_and_a_cold_targets(tree):
    """2^16 FP32 queries from NEUTRAL: a 20 degree cone solves more than the exact axis on shelf-horizontal reaches and
    on A-cold targets (DESIGN.md 4.9)."""
    n = 1 << 16
    q = synthetic.random_joint_configs(n, tree.lower, tree.upper, seed=1234, device="cuda", dtype=torch.float64)
    pos, quat, _ = engine.fk_jac(q, want_jac=False)
    w, x, y, z = quat.unbind(1)
    axis = torch.stack([2 * (x * z + w * y), 2 * (y * z - w * x), 1 - 2 * (x * x + y * y)], dim=1)
    box = torch.tensor(synthetic.SHELF_BOX, dtype=torch.float64)
    ps = box[:, 0] + (box[:, 1] - box[:, 0]) * torch.as_tensor(np.random.default_rng(0).random((n, 3)))
    horiz = torch.tensor([1.0, 0.0, 0.0], dtype=torch.float64).expand(n, 3)
    q0 = torch.tensor(NEUTRAL, dtype=torch.float32, device="cuda")
    for name, tp, ta, gain in (("a_cold", pos, axis, 0.03), ("shelf_horizontal", ps, horiz, 0.3)):
        tp, ta = tp.float().cuda().contiguous(), ta.float().cuda().contiguous()
        plain = engine.ik_axis_solve(tp, ta, q0, engine.ik_params())["success"].float().mean().item()
        cone = engine.ik_axis_solve(tp, ta, q0, engine.ik_params(), cone_angle=20 * DEG)["success"].float().mean().item()
        print(f"{name}: axis {plain:.4f}, 20 degree cone {cone:.4f}")
        assert cone > plain + gain, (name, plain, cone)

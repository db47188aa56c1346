"""GPU: axis-constrained IK (pnp_ik_axis_solve_*, engine.ik_axis_solve, JacobianIKController.solve_axis) against its
FP64 statement (oracle/axis_ik_oracle.py).

The workload is A: q* uniform inside the joint limits, target (FK(q*), R(q*) t) for the tool axis t; A-near starts at
clip(q* + U(+-0.3)), A-cold at NEUTRAL.  The FP64 kernel is held to the batched statement iteration for iteration; the
FP32 kernel, run against the statement on its FP32-rounded inputs, to a counted number of iteration flips and to its
q re-evaluated with the FP64 FK.  The multistart is held to bit-identity with the plain solve from the attempt it
names."""
import ctypes

import numpy as np
import pytest
import torch

from conftest import NEUTRAL
from mujoco_panda_pnp_b200 import KinematicData, KinematicTree, _lib, engine
from mujoco_panda_pnp_b200.skills import JacobianIKController
from oracle import axis_ik_oracle, c_oracle, pose_ik_oracle
from test_gpu_foreign_trees import arm, arms, gpu  # noqa: F401  (fixtures of the foreign arms)

pytestmark = pytest.mark.gpu

IK_BLOCK = 128  # pnp_kernels.cuh: up to sm_count * IK_BLOCK queries take the small-batch path
KINS = ["specialized", "generic"]
DTYPES = {"fp32": torch.float32, "fp64": torch.float64}
DEFAULTS = dict(max_iters=100, pos_thresh=1e-3, rot_thresh=1e-2, damping=1e-2, step_limit=0.1, rot_weight=1.0)
Z, OBLIQUE = (0.0, 0.0, 1.0), (0.3, -0.2, 0.9)
FP32_POS_TOL, FP32_AXIS_TOL, FP32_ROT_TOL = 1e-5, 1e-5, 2e-5  # FP32 kernel vs FP64 evaluation at the same q
KEYS = ("q", "final_pos", "final_axis", "final_quat", "pos_error", "axis_error", "iterations", "converged", "success")


@pytest.fixture(scope="module")
def tree(cuda_lib):
    t = KinematicTree.from_mjcf()
    engine.set_tree(t)
    return t


def _limits(chain):
    return np.array(chain.lower[:]), np.array(chain.upper[:])


def workload(chain, n, seed, start, tool=Z):
    """A: q* ~ U(limits), target (FK(q*), R(q*) t), start NEUTRAL (cold) or clip(q* + U(+-0.3)) (near)."""
    rng = np.random.default_rng(seed)
    lo, hi = _limits(chain)
    q_star = rng.uniform(lo, hi, (n, 7))
    p, mat, _ = c_oracle.fk_jac(chain, q_star, nthreads=8)
    ax = mat @ axis_ik_oracle.tool_basis(tool)[0]
    q0 = np.tile(NEUTRAL, (n, 1)) if start == "cold" else np.clip(q_star + rng.uniform(-0.3, 0.3, q_star.shape), lo, hi)
    return p, ax, q0


def _rounded(dtype, *arrays):
    if dtype == torch.float32:
        return [np.asarray(a, dtype=np.float32).astype(np.float64) for a in arrays]
    return [np.asarray(a, dtype=np.float64) for a in arrays]


def _ik(p):
    return {k: p[k] for k in ("max_iters", "pos_thresh", "damping", "step_limit")}


def solve(dtype, kin, pos, ax, q_init, tool=Z, counters=None, **p):
    p = dict(DEFAULTS, **p)
    out = engine.ik_axis_solve(gpu(pos, dtype), gpu(ax, dtype), gpu(q_init, dtype),
                               engine.ik_params(kinematics=kin, **_ik(p)), tool_axis=tool, rot_thresh=p["rot_thresh"],
                               rot_weight=p["rot_weight"], counters=counters)
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in out.items()}


def statement(chain, dtype, pos, ax, q_init, tool=Z, **p):
    pos, ax, q_init = _rounded(dtype, pos, ax, q_init)
    return axis_ik_oracle.solve_axis_batch(chain, pos, ax, q_init, tool_axis=tool, **dict(DEFAULTS, **p))


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint8)


def _quat_close(got, mat, tol):
    """final_quat against mju_mat2Quat of the statement's frame, up to the sign two mat2Quat cases may differ by."""
    want = pose_ik_oracle.mat2quat_batch(mat.reshape(-1, 9))[0]
    got = np.asarray(got, dtype=np.float64)
    d = np.minimum(np.abs(got - want).max(axis=1, initial=0.0), np.abs(got + want).max(axis=1, initial=0.0))
    assert d.max(initial=0.0) < tol, d.max(initial=0.0)


def check_fp64(got, ref, tol=1e-8, ties=1):
    """Iteration-exact: identical iteration counts and flags (at most `ties` queries whose FK rounding puts the kernel
    and the statement on opposite sides of a threshold), converged queries within tol in every output."""
    tie = got["iterations"] != ref["iterations"]
    assert tie.sum() <= ties, np.nonzero(tie)[0][:10]
    ok = ~tie
    assert np.array_equal(got["converged"][ok], ref["converged"][ok])
    assert np.array_equal(got["success"][ok], ref["success"][ok])
    c = ok & ref["converged"]
    for key in ("q", "final_pos", "final_axis", "pos_error", "axis_error"):
        d = np.abs(got[key][c] - ref[key][c]).max(initial=0.0)
        assert d < tol, (key, d)
    _quat_close(got["final_quat"][c], ref["final_mat"][c], tol)


def check_fp32(chain, got, ref, pos, ax, tool=Z, budget=2, q_budget=2, dq_cap=1e-3, **p):
    """FP32 kernel vs the statement on the FP32-rounded inputs: iteration flips bounded by ``budget``, converged flips
    by 2; solves that converge in the same passes on both sides agree in q within 2e-5 rad but for ``q_budget`` of them,
    all within ``dq_cap``; every converged q reaches the target under the FP64 FK, and the reported pose, axis and errors
    are those of the returned q."""
    p = dict(DEFAULTS, **p)
    conv, iters = got["converged"], got["iterations"]
    assert np.array_equal(got["success"], conv)
    flips = int((iters != ref["iterations"]).sum())
    conv_flips = int((conv != ref["converged"]).sum())
    q = got["q"].astype(np.float64)
    same = conv & ref["converged"] & (iters == ref["iterations"])
    dq = np.abs(q[same] - ref["q"][same]).max(axis=1, initial=0.0)
    print(f"fp32 axis: {flips} flips, {conv_flips} converged flips, {int((dq > 2e-5).sum())} |dq| > 2e-5 "
          f"(max {dq.max(initial=0.0):.2e}) of {len(q)}")
    assert flips <= budget, (flips, budget)
    assert conv_flips <= 2, conv_flips
    assert (dq > 2e-5).sum() <= q_budget and dq.max(initial=0.0) < dq_cap, (int((dq > 2e-5).sum()), dq.max(initial=0.0))
    ev = axis_ik_oracle.axis_eval_batch(chain, q, pos, ax, tool_axis=tool)
    assert ev["pos_error"][conv].max(initial=0.0) < p["pos_thresh"] + 1e-5
    assert ev["axis_error"][conv].max(initial=0.0) < p["rot_thresh"] + FP32_ROT_TOL
    assert np.abs(got["final_pos"] - ev["final_pos"]).max() < FP32_POS_TOL
    assert np.abs(got["final_axis"] - ev["final_axis"]).max() < FP32_AXIS_TOL
    assert np.abs(got["pos_error"] - ev["pos_error"]).max() < FP32_POS_TOL
    assert np.abs(got["axis_error"] - ev["axis_error"]).max() < FP32_ROT_TOL
    _quat_close(got["final_quat"], ev["mat"], 1e-5)
    lo, hi = _limits(chain)
    assert (q >= lo - 1e-6).all() and (q <= hi + 1e-6).all()


# ---------------------------------------------------------------------------------------------------------------------
# Plain solve against the statement
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kin", KINS)
@pytest.mark.parametrize("start", ["near", "cold"])
def test_fp64_is_iteration_exact(tree, oracle_chain, start, kin):
    pos, ax, q0 = workload(oracle_chain, 2048, seed=31, start=start)
    got = solve(torch.float64, kin, pos, ax, q0)
    ref = statement(oracle_chain, torch.float64, pos, ax, q0)
    check_fp64(got, ref)
    assert ref["converged"].mean() > (0.95 if start == "near" else 0.8)


@pytest.mark.parametrize("kin", KINS)
@pytest.mark.parametrize("start,n", [("near", 4096), ("cold", 2048)])
def test_fp32_vs_statement(tree, oracle_chain, start, n, kin):
    pos, ax, q0 = workload(oracle_chain, n, seed=41, start=start)
    got = solve(torch.float32, kin, pos, ax, q0)
    ref = statement(oracle_chain, torch.float32, pos, ax, q0)
    pos32, ax32 = _rounded(torch.float32, pos, ax)
    check_fp32(oracle_chain, got, ref, pos32, ax32, budget=2 if start == "near" else 8,
               q_budget=2 if start == "near" else 40, dq_cap=1e-3 if start == "near" else 5e-3)
    assert got["converged"].mean() > (0.95 if start == "near" else 0.8)


SETTINGS = {
    "oblique tool": dict(tool=OBLIQUE),
    "rot_weight=4": dict(rot_weight=4.0),
    "rot_thresh=1e-3": dict(rot_thresh=1e-3),
    "damping=1e-1": dict(damping=1e-1),
    "step_limit=0": dict(step_limit=0.0),
    "max_iters=5": dict(max_iters=5),
}


@pytest.mark.parametrize("kin", KINS)
@pytest.mark.parametrize("prec", ["fp32", "fp64"])
@pytest.mark.parametrize("setting", list(SETTINGS))
def test_parameters_vs_statement(tree, oracle_chain, setting, prec, kin):
    dtype, p = DTYPES[prec], dict(SETTINGS[setting])
    tool = p.pop("tool", Z)
    pos, ax, q0 = workload(oracle_chain, 512, seed=61, start="near", tool=tool)
    got = solve(dtype, kin, pos, ax, q0, tool=tool, **p)
    ref = statement(oracle_chain, dtype, pos, ax, q0, tool=tool, **p)
    if dtype == torch.float64:
        check_fp64(got, ref)
    else:
        pos32, ax32 = _rounded(dtype, pos, ax)
        check_fp32(oracle_chain, got, ref, pos32, ax32, tool=tool, budget=4, **p)
    if p.get("step_limit") == 0.0:
        assert np.array_equal(_bits(got["q"]), _bits(q0.astype(got["q"].dtype)))


@pytest.mark.parametrize("kin", KINS)
@pytest.mark.parametrize("prec", ["fp32", "fp64"])
def test_broadcast_q_init_is_bit_identical_to_per_row(tree, oracle_chain, prec, kin):
    dtype = DTYPES[prec]
    pos, ax, _ = workload(oracle_chain, 512, seed=71, start="cold")
    a = solve(dtype, kin, pos, ax, NEUTRAL)
    b = solve(dtype, kin, pos, ax, np.tile(NEUTRAL, (512, 1)))
    for k in a:
        assert np.array_equal(_bits(a[k]), _bits(b[k])), k


def _outs(n, dt, fill=float("nan")):
    return [torch.full((n, 7), fill, dtype=dt, device="cuda"), torch.full((n, 3), fill, dtype=dt, device="cuda"),
            torch.full((n, 3), fill, dtype=dt, device="cuda"), torch.full((n, 4), fill, dtype=dt, device="cuda"),
            torch.full((n,), fill, dtype=dt, device="cuda"), torch.full((n,), fill, dtype=dt, device="cuda"),
            torch.full((n,), -1, dtype=torch.int32, device="cuda"), torch.full((n,), 0xFF, dtype=torch.uint8, device="cuda")]


def _tool(t=Z):
    return None if t is None else (ctypes.c_double * 3)(*t)


def raw_solve(dtype, kin, tp, ta, qi, stride, n, outs, counters, tool=Z, rot_thresh=1e-2, rot_weight=1.0, params=None):
    """pnp_ik_axis_solve_* through the C ABI; outs as _outs, any entry None."""
    lib = _lib.load()
    fn = lib.pnp_ik_axis_solve_f32 if dtype == torch.float32 else lib.pnp_ik_axis_solve_f64
    ptr = [None if t is None else t.data_ptr() for t in outs]
    return fn(None if tp is None else tp.data_ptr(), ta.data_ptr(), qi.data_ptr(), stride, n,
              ctypes.byref(params or engine.ik_params(kinematics=kin)), _tool(tool), rot_thresh, rot_weight, *ptr,
              None if counters is None else counters.data_ptr(), torch.cuda.current_stream().cuda_stream)


@pytest.mark.parametrize("kin", KINS)
@pytest.mark.parametrize("prec", ["fp32", "fp64"])
def test_results_do_not_depend_on_batch_shape(tree, oracle_chain, prec, kin):
    """48 witness queries solved one at a time, as one batch (small-batch path: one working warp per block) and at
    scattered rows of batches of sm_count * IK_BLOCK, sm_count * IK_BLOCK + 1 and 2^20 queries (persistent warps with
    lane refill): bit-identical.  The 2^20 batch goes through the C ABI into sentinel-filled buffers, with counters, and
    again with every nullable output NULL, and with final_quat alone NULL."""
    dtype = DTYPES[prec]
    engine.set_tree(tree)
    sm = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    pos, ax, q0 = workload(oracle_chain, 4096, seed=81, start="near")
    rng = np.random.default_rng(82)
    w = rng.choice(4096, 48, replace=False)
    ref = solve(dtype, kin, pos[w], ax[w], q0[w])
    for k in range(48):
        one = solve(dtype, kin, pos[w[k]:w[k] + 1], ax[w[k]:w[k] + 1], q0[w[k]:w[k] + 1])
        for key in KEYS:
            assert np.array_equal(_bits(one[key][0]), _bits(ref[key][k])), (k, key)
    pool = [gpu(a, dtype) for a in (pos, ax, q0)]
    for n in (sm * IK_BLOCK, sm * IK_BLOCK + 1, 1 << 20):
        idx = rng.integers(0, 4096, n)
        slots = rng.choice(n, 48, replace=False)
        idx[slots] = w
        it = torch.as_tensor(idx, device="cuda")
        tp, ta, qi = (a[it].contiguous() for a in pool)
        if n < (1 << 20):
            out = engine.ik_axis_solve(tp, ta, qi, engine.ik_params(kinematics=kin))
            torch.cuda.synchronize()
            for key in KEYS:
                assert np.array_equal(_bits(out[key][slots].cpu().numpy()), _bits(ref[key])), (n, key)
            continue
        outs = _outs(n, dtype)
        counters = torch.zeros(4, dtype=torch.int64, device="cuda")
        _lib.check(raw_solve(dtype, kin, tp, ta, qi, 7, n, outs, counters), "pnp_ik_axis_solve")
        torch.cuda.synchronize()
        q, fpos, fax, fquat, perr, aerr, iters, flags = outs
        for t in (q, fpos, fax, fquat, perr, aerr):
            assert torch.isfinite(t).all()
        assert bool(((iters >= 0) & (iters <= 100)).all()) and bool((flags <= 3).all())
        conv, succ = (flags & 1) != 0, (flags & 2) != 0
        assert counters.tolist() == [n, int(conv.sum()), int(succ.sum()), int(iters.long().sum())]
        got = dict(zip(KEYS, (q, fpos, fax, fquat, perr, aerr, iters, conv, succ)))
        for key in KEYS:
            assert np.array_equal(_bits(got[key][slots].cpu().numpy()), _bits(ref[key])), (n, key)
        part = _outs(n, dtype)
        part[3] = None
        _lib.check(raw_solve(dtype, kin, tp, ta, qi, 7, n, part, None), "pnp_ik_axis_solve")
        only_q = [torch.full((n, 7), float("nan"), dtype=dtype, device="cuda")] + [None] * 7
        _lib.check(raw_solve(dtype, kin, tp, ta, qi, 7, n, only_q, None), "pnp_ik_axis_solve")
        torch.cuda.synchronize()
        for a, b in zip(part, outs):
            assert a is None or torch.equal(a.view(torch.uint8), b.view(torch.uint8))
        assert torch.equal(only_q[0].view(torch.uint8), q.view(torch.uint8))
    empty = engine.ik_axis_solve(*(a[:0] for a in pool), engine.ik_params(kinematics=kin))
    assert all(v.shape[0] == 0 for v in empty.values())


@pytest.mark.parametrize("kin", KINS)
@pytest.mark.parametrize("prec", ["fp32", "fp64"])
def test_degenerate_axes(tree, oracle_chain, prec, kin):
    """A zero or NaN target axis runs to max_iters unconverged and leaves its neighbours untouched.  A start whose tool
    axis is exactly opposite the target's (s = 0, theta = pi, taken from the kernel's own evaluation at the start) takes
    a step and leaves theta = pi."""
    dtype = DTYPES[prec]
    pos, ax, q0 = workload(oracle_chain, 256, seed=91, start="near")
    at = np.array([0, 37, 130, 255])
    pos2, ax2, q2 = (np.insert(a, at, a[at], axis=0) for a in (pos, ax, q0))
    bad = np.zeros(len(pos2), dtype=bool)
    bad[at + np.arange(len(at))] = True
    ax2[bad] = [[0.0, 0.0, 0.0], [np.nan, 0.0, 1.0], [np.nan] * 3, [0.0, 0.0, 0.0]]
    got = solve(dtype, kin, pos2, ax2, q2, max_iters=40)
    assert not got["converged"][bad].any() and not got["success"][bad].any()
    assert (got["iterations"][bad] == 40).all()
    clean = solve(dtype, kin, pos, ax, q0, max_iters=40)
    for key in clean:
        assert np.array_equal(_bits(got[key][~bad]), _bits(clean[key])), key
    # antiparallel start: the target axis is minus the kernel's own tool axis at q0
    ev0 = solve(dtype, kin, pos, ax, q0, max_iters=0)
    flip = -ev0["final_axis"].astype(np.float64)
    e0 = solve(dtype, kin, ev0["final_pos"], flip, q0, max_iters=0)
    assert (e0["axis_error"] > np.pi - 1e-3).mean() > 0.9
    one = solve(dtype, kin, ev0["final_pos"], flip, q0, max_iters=1)
    moved = np.abs(one["q"].astype(np.float64) - q0.astype(one["q"].dtype)).max(axis=1)
    assert (moved > 1e-3).all() and np.isfinite(one["q"]).all()
    assert (one["axis_error"] < np.pi - 1e-4).all() and np.median(one["axis_error"]) < np.pi - 1e-2


@pytest.mark.parametrize("kin", KINS)
def test_exactly_antiparallel_start_takes_the_b1_tilt(tree, kin):
    """s == 0 exactly in the kernel: with link rotations exactly 0 / +-1 (the snapped tree: the specialised kernels are
    generated from it, the generic ones read it when it is uploaded) the site's z axis at q = qref is a signed basis
    vector, so with the target axis -a the cross product a x d is exactly zero however it is contracted.  The FP64
    first step must be the DLS step of the error [0, 0, 0, w pi, 0] (n = b1), computed here from the kernel's own
    Jacobian."""
    snapped, tool = tree.snapped(), Z
    try:
        engine.set_tree(tree if kin == "specialized" else snapped)
        q0 = snapped.qref[None].copy()
        ev = solve(torch.float64, kin, np.zeros((1, 3)), np.array([[0.0, 0.0, 1.0]]), q0, tool=tool, max_iters=0)
        a0 = ev["final_axis"][0]
        assert set(np.abs(a0).tolist()) == {0.0, 1.0}, a0  # exact: a x (-a) = 0 in any evaluation order
        p0, d = ev["final_pos"], -a0[None]
        e0 = solve(torch.float64, kin, p0, d, q0, tool=tool, max_iters=0)
        assert e0["axis_error"][0] == np.pi and e0["pos_error"][0] == 0.0
        one = solve(torch.float64, kin, p0, d, q0, tool=tool, max_iters=1)
        _, _, jac = engine.fk_jac(gpu(q0), want_quat=False, kinematics=kin)
        jac = jac[0].cpu().numpy()
        R = np.eye(3)
        for i in range(7):
            R = R @ snapped.link_rot[i]
        R = R @ snapped.ee_rot
        _, u1, u2 = axis_ik_oracle.tool_basis(tool)
        J = np.vstack([jac[:3], (R @ u1) @ jac[3:], (R @ u2) @ jac[3:]])
        dq = J.T @ np.linalg.solve(J @ J.T + 1e-2 * np.eye(5), np.array([0.0, 0.0, 0.0, np.pi, 0.0]))
        want = np.clip(q0[0] + np.clip(dq, -0.1, 0.1), snapped.lower, snapped.upper)
        assert np.abs(one["q"][0] - want).max() < 1e-12, (one["q"][0], want)
        assert np.abs(one["q"][0] - q0[0]).max() > 1e-2
    finally:
        engine.set_tree(tree)


@pytest.mark.parametrize("prec", ["fp32", "fp64"])
def test_rejected_arguments_leave_outputs_untouched(tree, oracle_chain, prec):
    dtype = DTYPES[prec]
    n = 256
    pos, ax, q0 = (gpu(a, dtype) for a in workload(oracle_chain, n, seed=95, start="near"))
    outs = _outs(n, dtype, 7.0)
    before = [t.clone() for t in outs]

    def call(**over):
        kw = dict(tp=pos, n=n, outs=outs, tool=Z, rot_thresh=1e-2, rot_weight=1.0)
        kw.update(over)
        return raw_solve(dtype, "auto", kw["tp"], ax, q0, 7, kw["n"], kw["outs"], None, tool=kw["tool"],
                         rot_thresh=kw["rot_thresh"], rot_weight=kw["rot_weight"])

    cases = [dict(tool=None), dict(tool=(0.0, 0.0, 0.0)), dict(tool=(float("nan"), 0.0, 1.0)),
             dict(tool=(float("inf"), 0.0, 0.0)), dict(rot_thresh=0.0), dict(rot_thresh=-1.0),
             dict(rot_thresh=float("nan")), dict(rot_weight=0.0), dict(rot_weight=float("nan")), dict(tp=None),
             dict(outs=[None] + outs[1:]), dict(n=1 << 31), dict(n=-1)]
    for c in cases:
        assert call(**c) == -1, c
    torch.cuda.synchronize()
    for a, b in zip(outs, before):
        assert torch.equal(a, b)
    assert call() == 0 and call(tool=(1e-300, 0.0, 0.0)) == 0 and call(tool=(1e200, 1e200, 0.0)) == 0
    for kw in (dict(rot_thresh=0.0), dict(rot_weight=-1.0), dict(tool_axis=(0, 0)), dict(tool_axis=(0, 0, 0))):
        with pytest.raises(ValueError):
            engine.ik_axis_solve(pos, ax, q0, engine.ik_params(), **kw)
    with pytest.raises(ValueError):
        engine.ik_axis_solve(pos, ax[:10], q0, engine.ik_params())


def test_graph_capture_replays_on_new_inputs(tree, oracle_chain):
    n = 1 << 14
    pos, ax, _ = workload(oracle_chain, n, seed=101, start="cold")
    tp, ta = gpu(pos, torch.float32), gpu(ax, torch.float32)
    q0 = torch.tensor(NEUTRAL, dtype=torch.float32, device="cuda")
    outs = _outs(n, torch.float32)
    counters = torch.zeros(4, dtype=torch.int64, device="cuda")

    def call():
        _lib.check(raw_solve(torch.float32, "auto", tp, ta, q0, 0, n, outs, counters), "pnp_ik_axis_solve")

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        call()
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        call()
    pos2, ax2, _ = workload(oracle_chain, n, seed=102, start="cold")
    tp.copy_(gpu(pos2, torch.float32)), ta.copy_(gpu(ax2, torch.float32))
    counters.zero_()
    g.replay()
    torch.cuda.synchronize()
    c2 = torch.zeros(4, dtype=torch.int64, device="cuda")
    r = engine.ik_axis_solve(gpu(pos2, torch.float32), gpu(ax2, torch.float32), q0, engine.ik_params(), counters=c2)
    torch.cuda.synchronize()
    for key, t in zip(KEYS[:7], outs[:7]):
        assert torch.equal(t.view(torch.uint8), r[key].contiguous().view(torch.uint8)), key
    assert torch.equal(outs[7], r["converged"].to(torch.uint8) | (r["success"].to(torch.uint8) << 1))
    assert torch.equal(counters, c2)


# ---------------------------------------------------------------------------------------------------------------------
# Foreign arms (test_gpu_foreign_trees.py's builders): the generic kernels against the statement on their chains
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("start", ["cold", "near"])
def test_foreign_arm_vs_statement(arm, start):  # noqa: F811
    rng = np.random.default_rng(16)
    q_star = rng.uniform(arm.lo, arm.hi, (2048, 7))
    p, mat, _ = c_oracle.fk_jac(arm.chain, q_star, nthreads=8)
    ax = mat[:, :, 2]
    q0 = np.broadcast_to(arm.mid, q_star.shape) if start == "cold" else \
        np.clip(q_star + rng.uniform(-0.3, 0.3, q_star.shape), arm.lo, arm.hi)
    got = solve(torch.float64, "auto", p, ax, q0)
    check_fp64(got, statement(arm.chain, torch.float64, p, ax, q0))
    assert got["converged"].mean() > (0.95 if start == "near" else 0.5)
    got32 = solve(torch.float32, "auto", p, ax, q0)
    ref32 = statement(arm.chain, torch.float32, p, ax, q0)
    p32, ax32 = _rounded(torch.float32, p, ax)
    check_fp32(arm.chain, got32, ref32, p32, ax32, budget=8, q_budget=60, dq_cap=1e-2)


# ---------------------------------------------------------------------------------------------------------------------
# Multistart
# ---------------------------------------------------------------------------------------------------------------------
def _tbits(r):
    out = {}
    for k in KEYS:
        t = r[k].contiguous()
        out[k] = t.view(torch.int64 if t.dtype == torch.float64 else torch.int32) if t.is_floating_point() else t.clone()
    return out


def expected(tp, ta, q_init, seeds, params, **kw):
    """The composition of plain calls: one from q_init, one per seed broadcast over all queries."""
    runs = [_tbits(engine.ik_axis_solve(tp, ta, q_init, params, **kw))] + \
           [_tbits(engine.ik_axis_solve(tp, ta, s, params, **kw)) for s in seeds]
    succ = torch.stack([r["success"] for r in runs])
    k1 = torch.arange(len(runs), device=succ.device)[:, None].expand_as(succ)
    first = torch.where(succ, k1, torch.full_like(k1, len(runs))).min(0).values
    attempt = torch.where(first == len(runs), torch.zeros_like(first), first)
    exp = {}
    for key in runs[0]:
        st = torch.stack([r[key] for r in runs])
        idx = attempt.view(1, -1, *([1] * (st.dim() - 2))).expand(1, *st.shape[1:])
        exp[key] = st.gather(0, idx)[0]
    return attempt, exp


def assert_rows(got, exp, what=""):
    for key in exp:
        assert torch.equal(got[key], exp[key]), (what, key)


def ms_workload(chain, n, dt, seed=1234):
    """A-cold targets, then unreachable positions and zero / NaN axes."""
    pos, ax, _ = workload(chain, n, seed=seed, start="cold")
    far = np.array([[2.5, 0.0, 0.5], [0.0, 0.0, 3.0], [-2.0, 1.5, 0.2]] * 4)
    bad_ax = np.array([[0.0, 0.0, 0.0], [np.nan, 0.0, 1.0]])
    pos = np.concatenate([pos, far, pos[:2]])
    ax = np.concatenate([ax, ax[:12], bad_ax])
    return gpu(pos, dt), gpu(ax, dt)


@pytest.mark.parametrize("kin", KINS)
@pytest.mark.parametrize("prec", ["fp32", "fp64"])
@pytest.mark.parametrize("tool", ["z", "oblique"])
def test_multistart_rows_are_plain_solves(tree, oracle_chain, prec, kin, tool):
    dt = DTYPES[prec]
    t = Z if tool == "z" else OBLIQUE
    tp, ta = ms_workload(oracle_chain, 1 << 13, dt)
    q0 = torch.tensor(NEUTRAL, dtype=dt, device="cuda")
    seeds = engine.ik_restart_seeds(8, dtype=dt)
    params = engine.ik_params(kinematics=kin)
    counters = torch.zeros(4, dtype=torch.int64, device="cuda")
    stats = torch.zeros(3, dtype=torch.int64, device="cuda")
    r = engine.ik_axis_solve_multistart(tp, ta, q0, seeds, params, tool_axis=t, counters=counters, restart_stats=stats)
    attempt, exp = expected(tp, ta, q0, seeds, params, tool_axis=t)
    assert_rows(_tbits(r), exp)
    assert torch.equal(r["attempt"].long(), attempt)
    c = counters.cpu().numpy()
    assert c[0] == len(tp) and c[1] == int(r["converged"].sum()) and c[2] == int(r["success"].sum())
    assert c[3] == int(r["iterations"].long().sum())
    s = stats.cpu().numpy()
    assert s[1] == int((attempt > 0).sum()) and s[1] > 100 and s[2] >= int(r["iterations"][attempt > 0].long().sum())
    assert not r["success"][-14:].any() and not r["attempt"][-14:].any()


def test_multistart_fp64_matches_the_statement(tree, oracle_chain):
    pos, ax, _ = workload(oracle_chain, 1024, seed=11, start="cold")
    seeds = engine.ik_restart_seeds(4, dtype=torch.float64)
    r = engine.ik_axis_solve_multistart(gpu(pos), gpu(ax), gpu(NEUTRAL), seeds, engine.ik_params())
    got = {k: v.cpu().numpy() for k, v in r.items()}
    att = np.zeros(len(pos), dtype=np.int64)
    ref = axis_ik_oracle.solve_axis_batch(oracle_chain, pos, ax, NEUTRAL)
    left = np.nonzero(~ref["success"])[0]
    for k, s in enumerate(seeds.cpu().numpy()):
        rk = axis_ik_oracle.solve_axis_batch(oracle_chain, pos[left], ax[left], s)
        for key in ("q", "iterations", "converged", "success"):
            ref[key][left[rk["success"]]] = rk[key][rk["success"]]
        att[left[rk["success"]]] = k + 1
        left = left[~rk["success"]]
    assert (att > 0).sum() > 50
    same = (got["attempt"] == att) & (got["iterations"] == ref["iterations"])
    assert int((~same).sum()) <= 2, np.nonzero(~same)[0]
    c = same & ref["converged"]
    assert np.abs(got["q"][c] - ref["q"][c]).max() < 1e-8


def test_multistart_k0_is_the_plain_solve(tree, oracle_chain):
    tp, ta = ms_workload(oracle_chain, 1 << 12, torch.float32)
    q0 = torch.tensor(NEUTRAL, dtype=torch.float32, device="cuda")
    c0, c1 = (torch.zeros(4, dtype=torch.int64, device="cuda") for _ in range(2))
    n0 = _lib.launch_count()
    p = engine.ik_axis_solve(tp, ta, q0, engine.ik_params(), counters=c0)
    n1 = _lib.launch_count()
    r = engine.ik_axis_solve_multistart(tp, ta, q0, torch.empty((0, 7), device="cuda"), engine.ik_params(), counters=c1)
    n2 = _lib.launch_count()
    assert n2 - n1 == n1 - n0
    assert_rows(_tbits(r), _tbits(p))
    assert torch.equal(c0, c1) and not r["attempt"].any()


def test_multistart_255_seeds(tree, oracle_chain):
    tp, ta = ms_workload(oracle_chain, 512, torch.float32)
    q0 = torch.tensor(NEUTRAL, dtype=torch.float32, device="cuda")
    seeds = engine.ik_restart_seeds(255, seed=7)
    params = engine.ik_params()
    r = engine.ik_axis_solve_multistart(tp, ta, q0, seeds, params)
    attempt, exp = expected(tp, ta, q0, seeds, params)
    assert_rows(_tbits(r), exp)
    assert torch.equal(r["attempt"].long(), attempt) and int(attempt.max()) > 8
    with pytest.raises(ValueError):
        engine.ik_axis_solve_multistart(tp, ta, q0, engine.ik_restart_seeds(256), params)


def test_multistart_rejected_arguments_leave_outputs_untouched(tree, oracle_chain, cuda_lib):
    n = 256
    tp, ta = (gpu(a, torch.float32) for a in workload(oracle_chain, n, seed=5, start="cold")[:2])
    q0 = torch.tensor(NEUTRAL, dtype=torch.float32, device="cuda")
    seeds = engine.ik_restart_seeds(4)
    nb = ctypes.c_int64()
    assert cuda_lib.pnp_ik_multistart_scratch_bytes(n, ctypes.byref(nb)) == 0
    scratch = torch.zeros(nb.value // 4 + 8, dtype=torch.int32, device="cuda")
    outs = _outs(n, torch.float32, 7.0)
    attempt = torch.full((n,), 9, dtype=torch.uint8, device="cuda")
    before = [t.clone() for t in outs] + [attempt.clone()]

    def call(seeds_p=seeds.data_ptr(), k=4, scratch_p=scratch.data_ptr(), tool=Z, flags=True):
        ptr = [t.data_ptr() for t in outs]
        if not flags:
            ptr[7] = None
        return cuda_lib.pnp_ik_axis_solve_multistart_f32(
            tp.data_ptr(), ta.data_ptr(), q0.data_ptr(), 0, n, seeds_p, k, ctypes.byref(engine.ik_params()), _tool(tool),
            1e-2, 1.0, *ptr, attempt.data_ptr(), None, None, scratch_p, torch.cuda.current_stream().cuda_stream)

    cases = [dict(k=-1), dict(k=256), dict(seeds_p=None), dict(scratch_p=None), dict(scratch_p=scratch.data_ptr() + 4),
             dict(flags=False), dict(tool=None), dict(tool=(0.0, 0.0, 0.0)), dict(seeds_p=outs[0].data_ptr(), k=1),
             dict(scratch_p=outs[3].data_ptr()), dict(scratch_p=attempt.data_ptr() - 16)]
    for c in cases:
        assert call(**c) == -1, c
    torch.cuda.synchronize()
    for a, b in zip(outs + [attempt], before):
        assert torch.equal(a, b)
    assert call() == 0


def test_multistart_stream_order_and_graph(tree, oracle_chain):
    """Back-to-back calls without a synchronisation equal the synchronised sequence; a captured multistart replays on
    new inputs."""
    tp, ta = ms_workload(oracle_chain, 1 << 14, torch.float32)
    op, oa = ms_workload(oracle_chain, 1 << 14, torch.float32, seed=11)
    q0 = torch.tensor(NEUTRAL, dtype=torch.float32, device="cuda")
    seeds = engine.ik_restart_seeds(8)
    params = engine.ik_params()

    def sequence(sync):
        a = engine.ik_axis_solve_multistart(tp, ta, q0, seeds, params)
        if sync:
            torch.cuda.synchronize()
        b = engine.ik_axis_solve(tp, ta, a["q"], params)  # warm start from the multistart's q_out
        if sync:
            torch.cuda.synchronize()
        a2 = engine.ik_axis_solve_multistart(op, oa, q0, seeds, params)
        c = engine.ik_axis_solve(op, oa, q0, params)
        torch.cuda.synchronize()
        return [_tbits(x) for x in (a, b, a2, c)], a["attempt"].clone()

    (ref, att), (got, att2) = sequence(True), sequence(False)
    for x, y in zip(ref, got):
        assert_rows(y, x)
    assert torch.equal(att, att2) and int(att.count_nonzero()) > 100
    # graph capture of the engine call, replayed on new inputs
    tp_s, ta_s = tp.clone(), ta.clone()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        engine.ik_axis_solve_multistart(tp_s, ta_s, q0, seeds, params)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        cap = engine.ik_axis_solve_multistart(tp_s, ta_s, q0, seeds, params)
    tp_s.copy_(op), ta_s.copy_(oa)
    g.replay()
    torch.cuda.synchronize()
    assert_rows(_tbits(cap), ref[2])
    assert torch.equal(cap["attempt"], engine.ik_axis_solve_multistart(op, oa, q0, seeds, params)["attempt"])


def test_controller_solve_axis(tree, oracle_chain, kin_model):
    data = KinematicData(kin_model)
    seeds = engine.ik_restart_seeds(8)
    pos, ax, _ = workload(oracle_chain, 2048, seed=3, start="cold")
    for precision in ("fp32", "fp64"):
        ctl = JacobianIKController(kin_model, data, precision=precision)
        dt = torch.float32 if precision == "fp32" else torch.float64
        r = ctl.solve_axis(pos, ax, NEUTRAL, seeds=seeds)
        e = engine.ik_axis_solve_multistart(gpu(pos, dt), gpu(ax, dt), gpu(NEUTRAL, dt), seeds.to(dt), engine.ik_params())
        assert_rows(_tbits(r), _tbits(e), what=precision)
        assert torch.equal(r["attempt"], e["attempt"]) and int(e["attempt"].count_nonzero()) > 20
        p = ctl.solve_axis(pos, ax, NEUTRAL)
        assert "attempt" not in p and torch.equal(p["success"], e["success"] & (e["attempt"] == 0))
        one = ctl.solve_axis(pos[0], ax[0], NEUTRAL, tool_axis=(0, 0, 5))
        assert_rows(_tbits(one), {k: v[:1] for k, v in _tbits(p).items()}, what="one query")

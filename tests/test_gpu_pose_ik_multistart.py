"""GPU: multi-start pose IK (pnp_ik_pose_solve_multistart_*, engine.ik_pose_solve_multistart).

The specification is bit-identity: every returned row equals, bit for bit, the plain pose solve of the same precision
and kinematics from the start ``attempt`` names, and ``attempt`` is the first successful one.  The workload is W-cold
(q* ~ U(joint limits), target (FK(q*), quat(q*)), solved from NEUTRAL): about a quarter of it fails attempt 0."""
import ctypes

import numpy as np
import pytest
import torch

from conftest import NEUTRAL
from mujoco_panda_pnp_b200 import KinematicData, KinematicTree, _lib, engine, synthetic
from mujoco_panda_pnp_b200.skills import JacobianIKController, solve_ik
from test_pose_ik_multistart_oracle import solve_pose_multistart_batch, workspace

pytestmark = pytest.mark.gpu

DTYPES = {"f32": torch.float32, "f64": torch.float64}
FAR = [[2.5, 0.0, 0.5], [0.0, 0.0, 3.0], [-2.0, 1.5, 0.2], [1.0, -2.2, 1.0], [3.0, 3.0, 3.0], [0.0, 2.6, 0.8]]
KEYS = ("q", "final_pos", "final_quat", "pos_error", "rot_error")


@pytest.fixture(scope="module")
def tree(cuda_lib):
    t = KinematicTree.from_mjcf()
    engine.set_tree(t)
    return t


def w_cold(tree, n, seed=1234):
    """W targets (float64 on the device): pose of q* ~ U(joint limits)."""
    qstar = synthetic.random_joint_configs(n, tree.lower, tree.upper, seed=seed, dtype=torch.float64).cuda()
    pos, quat, _ = engine.fk_jac(qstar, want_jac=False)
    return pos, quat


def workload(tree, n=1 << 15):
    """W targets, then unreachable positions, NaN positions, zero and NaN quaternions (float64)."""
    pos, quat = w_cold(tree, n)
    m = len(FAR) * 8
    far = torch.tensor(FAR * 8, dtype=torch.float64, device="cuda")
    bad_pos = torch.cat([pos[:3], torch.full((2, 3), float("nan"), dtype=torch.float64, device="cuda")])
    bad_quat = torch.cat([torch.zeros((2, 4), dtype=torch.float64, device="cuda"),
                          torch.full((1, 4), float("nan"), dtype=torch.float64, device="cuda"), quat[:2]])
    return torch.cat([pos, far, bad_pos]), torch.cat([quat, quat[:m], bad_quat])


def seed_table(tree, dt):
    """seeds[0] = NEUTRAL (the broadcast q_init: never chosen for a query that failed from it), then 7 U(limits)."""
    s = torch.cat([torch.tensor(NEUTRAL, dtype=torch.float64)[None],
                   engine.ik_restart_seeds(7, tree.lower, tree.upper, seed=3, dtype=torch.float64, device="cpu")])
    return s.to(device="cuda", dtype=dt)


def bits(r):
    out = {}
    for k in KEYS:
        t = r[k].contiguous()
        out[k] = t.view(torch.int64 if t.dtype == torch.float64 else torch.int32)
    out["iterations"] = r["iterations"].to(torch.int32)
    out["converged"], out["success"] = r["converged"].clone(), r["success"].clone()
    return out


def plain(tp, tq, q_init, params, **kw):
    return bits(engine.ik_pose_solve(tp, tq, q_init, params, **kw))


def expected(tp, tq, q_init, seeds, params, **kw):
    """The composition of plain calls: one from q_init, one per seed broadcast over all queries."""
    runs = [plain(tp, tq, q_init, params, **kw)] + [plain(tp, tq, s, params, **kw) for s in seeds]
    succ = torch.stack([r["success"] for r in runs])  # [K+1, n]
    k1 = torch.arange(len(runs), device=succ.device)[:, None].expand_as(succ)
    first = torch.where(succ, k1, torch.full_like(k1, len(runs))).min(0).values
    attempt = torch.where(first == len(runs), torch.zeros_like(first), first)
    exp = {}
    for key in runs[0]:
        st = torch.stack([r[key] for r in runs])
        idx = attempt.view(1, -1, *([1] * (st.dim() - 2))).expand(1, *st.shape[1:])
        exp[key] = st.gather(0, idx)[0]
    return attempt, exp, succ


def assert_rows(got, exp, rows=None, what=""):
    for key in exp:
        g, e = (got[key], exp[key]) if rows is None else (got[key][rows], exp[key])
        assert torch.equal(g, e), (what, key)


def check_counters(r, counters):
    c = counters.cpu().numpy()
    assert c[0] == len(r["q"])
    assert c[1] == int(r["converged"].sum()) and c[2] == int(r["success"].sum())
    assert c[3] == int(r["iterations"].to(torch.int64).sum())


@pytest.mark.parametrize("kin", ["specialized", "generic"])
@pytest.mark.parametrize("dtype", list(DTYPES))
@pytest.mark.parametrize("bcast", [True, False])
def test_composition_identity(tree, dtype, kin, bcast):
    dt = DTYPES[dtype]
    tp, tq = (t.to(dt) for t in workload(tree))
    n = len(tp)
    q_init = torch.tensor(NEUTRAL, dtype=dt, device="cuda") if bcast else \
        synthetic.random_joint_configs(n, tree.lower, tree.upper, seed=5, dtype=torch.float64).to("cuda", dt)
    params = engine.ik_params(kinematics=kin)
    seeds = seed_table(tree, dt)
    counters = torch.zeros(4, dtype=torch.int64, device="cuda")
    stats = torch.zeros(3, dtype=torch.int64, device="cuda")
    r = engine.ik_pose_solve_multistart(tp, tq, q_init, seeds, params, counters=counters, restart_stats=stats)
    attempt, exp, succ = expected(tp, tq, q_init, seeds, params)
    assert_rows(bits(r), exp)
    assert torch.equal(r["attempt"].long(), attempt)
    check_counters(r, counters)
    s = stats.cpu().numpy()
    rescued = attempt > 0
    assert s[0] == int((~succ[0]).sum()) and s[1] == int(rescued.sum())
    assert s[2] >= int(r["iterations"][rescued].to(torch.int64).sum())
    assert s[1] > 1000 and int((~r["success"]).sum()) >= len(FAR) * 8 + 5  # rescues; unreachable / NaN rows left
    assert not r["success"][-5:].any() and not r["attempt"][-5:].any()
    if bcast:
        assert not (attempt == 1).any()  # seeds[0] == q_init: fails wherever attempt 0 failed
    # somewhere an earlier seed won over a later one that also succeeds
    tie = torch.zeros_like(rescued)
    for k in range(2, len(seeds)):
        tie |= (attempt == k) & succ[k + 1:].any(0)
    assert tie.any()


def test_fp64_matches_the_statement(tree, oracle_chain):
    """FP64 kernel vs the FP64 statement on 2048 W-cold targets, 8 seeds: the same attempt, iterations and flags
    (except where FK rounding puts the two on opposite sides of a threshold in one of the attempts: at most 2 queries),
    q within 1e-8 where converged."""
    pos, quat = workspace(oracle_chain, 2048, seed=11)
    seeds = engine.ik_restart_seeds(8, dtype=torch.float64)
    r = engine.ik_pose_solve_multistart(torch.as_tensor(pos, device="cuda"), torch.as_tensor(quat, device="cuda"),
                                        torch.tensor(NEUTRAL, dtype=torch.float64, device="cuda"), seeds,
                                        engine.ik_params())
    ref = solve_pose_multistart_batch(oracle_chain, pos, quat, NEUTRAL, seeds.cpu().numpy())
    got = {k: v.cpu().numpy() for k, v in r.items()}
    assert (ref["attempt"] > 0).sum() > 300
    same = (got["attempt"] == ref["attempt"]) & (got["iterations"] == ref["iterations"])
    assert int((~same).sum()) <= 2, np.nonzero(~same)[0]
    assert np.array_equal(got["converged"][same], ref["converged"][same])
    assert np.array_equal(got["success"][same], ref["success"][same])
    c = same & ref["converged"]
    for key in ("q", "final_pos", "pos_error", "rot_error"):
        assert np.abs(got[key][c] - ref[key][c]).max() < 1e-8, key


def test_k0_is_the_plain_solve(tree):
    tp, tq = (t.float() for t in workload(tree, 1 << 14))
    q0 = torch.tensor(NEUTRAL, dtype=torch.float32, device="cuda")
    params = engine.ik_params()
    c0, c1 = (torch.zeros(4, dtype=torch.int64, device="cuda") for _ in range(2))
    n0 = _lib.launch_count()
    p = engine.ik_pose_solve(tp, tq, q0, params, counters=c0)
    n1 = _lib.launch_count()
    r = engine.ik_pose_solve_multistart(tp, tq, q0, torch.empty((0, 7), device="cuda"), params, counters=c1)
    n2 = _lib.launch_count()
    assert n2 - n1 == n1 - n0
    assert_rows(bits(r), bits(p))
    assert torch.equal(c0, c1) and not r["attempt"].any()


@pytest.mark.parametrize("case", ["all_near", "all_unreachable"])
def test_nothing_to_rescue(tree, case):
    g = torch.Generator().manual_seed(1)
    if case == "all_near":
        q = torch.tensor(NEUTRAL)[None] + 0.05 * (torch.rand((4096, 7), generator=g, dtype=torch.float64) - 0.5)
        tp, tq, _ = engine.fk_jac(q.cuda().float(), want_jac=False)
    else:
        tp = torch.tensor(FAR * 700, dtype=torch.float32, device="cuda")
        tq = torch.nn.functional.normalize(torch.randn((len(tp), 4), generator=g), dim=1).cuda()
    q0 = torch.tensor(NEUTRAL, dtype=torch.float32, device="cuda")
    params = engine.ik_params()
    stats = torch.zeros(3, dtype=torch.int64, device="cuda")
    r = engine.ik_pose_solve_multistart(tp, tq, q0, engine.ik_restart_seeds(8), params, restart_stats=stats)
    assert_rows(bits(r), plain(tp, tq, q0, params))
    assert not r["attempt"].any()
    s = stats.cpu().numpy()
    if case == "all_near":
        assert bool(r["success"].all()) and s[0] == 0
    else:
        assert not r["success"].any() and s[0] == len(tp) and s[1] == 0


def test_255_seeds(tree):
    """The most seeds a call takes: every wave of the table runs, and the first success still wins."""
    tp, tq = (t.float() for t in workload(tree, 512))
    q0 = torch.tensor(NEUTRAL, dtype=torch.float32, device="cuda")
    seeds = engine.ik_restart_seeds(255, seed=7)
    params = engine.ik_params()
    stats = torch.zeros(3, dtype=torch.int64, device="cuda")
    r = engine.ik_pose_solve_multistart(tp, tq, q0, seeds, params, restart_stats=stats)
    attempt, exp, succ = expected(tp, tq, q0, seeds, params)
    assert_rows(bits(r), exp)
    assert torch.equal(r["attempt"].long(), attempt)
    assert int(attempt.max()) > 8 and int(stats[1]) == int((attempt > 0).sum())
    with pytest.raises(ValueError):
        engine.ik_pose_solve_multistart(tp, tq, q0, engine.ik_restart_seeds(256), params)


def test_batch_sizes(tree, cuda_lib):
    sm = ctypes.c_int32()
    cuda_lib.pnp_device_info(ctypes.byref(sm), None, None)
    tp, tq = (t.float() for t in workload(tree, 1 << 15))
    perm = torch.randperm(len(tp), generator=torch.Generator().manual_seed(2)).cuda()
    tp, tq = tp[perm], tq[perm]
    seeds = engine.ik_restart_seeds(8)
    params = engine.ik_params()
    q0 = torch.tensor(NEUTRAL, dtype=torch.float32, device="cuda")
    for n in (0, 1, 31, 33, sm.value * 128 - 1, sm.value * 128 + 1):
        a, b = tp[:n].contiguous(), tq[:n].contiguous()
        r = engine.ik_pose_solve_multistart(a, b, q0, seeds, params)
        attempt, exp, _ = expected(a, b, q0, seeds, params)
        assert_rows(bits(r), exp, what=n)
        assert torch.equal(r["attempt"].long(), attempt), n


def test_large_batch(tree):
    """2^20 + 3 W-cold queries in FP32 with engine.ik_restart_seeds(8): rows attempt 0 solves are the plain solve's,
    every other row is its composition of plain calls, and the success rate is at least 0.98 (measured on a B200:
    0.98816 on tools/bench_pose_multistart.py's 2^20 W-cold targets, from 0.73557 for the plain solve)."""
    n = (1 << 20) + 3
    tp, tq = (t.float() for t in w_cold(tree, n, seed=9))
    q0 = torch.tensor(NEUTRAL, dtype=torch.float32, device="cuda")
    seeds = engine.ik_restart_seeds(8)
    params = engine.ik_params()
    counters = torch.zeros(4, dtype=torch.int64, device="cuda")
    r = engine.ik_pose_solve_multistart(tp, tq, q0, seeds, params, counters=counters)
    p = plain(tp, tq, q0, params)
    got = bits(r)
    a = r["attempt"].long()
    keep = ~p["success"]
    assert torch.equal(a[p["success"]], torch.zeros_like(a[p["success"]]))
    assert_rows(got, {k: v[p["success"]] for k, v in p.items()}, p["success"], "attempt 0")
    check_counters(r, counters)
    rows = torch.nonzero(keep).flatten()
    assert len(rows) > 0.2 * n
    sub_p, sub_q = tp[rows].contiguous(), tq[rows].contiguous()
    attempt, exp, _ = expected(sub_p, sub_q, q0, seeds, params)
    assert torch.equal(a[rows], attempt)
    assert_rows(got, exp, rows, "restarted")
    rate = float(r["success"].float().mean())
    assert rate >= 0.98, rate
    r2 = engine.ik_pose_solve_multistart(tp, tq, q0, seeds, params)
    assert_rows(bits(r2), got, what="rerun")
    assert torch.equal(r2["attempt"], r["attempt"])


def _p(t):
    return None if t is None else t.data_ptr()


def _outs(n, dt, fill=7.0):
    return dict(q=torch.full((n, 7), fill, dtype=dt, device="cuda"), fpos=torch.full((n, 3), fill, dtype=dt, device="cuda"),
                fquat=torch.full((n, 4), fill, dtype=dt, device="cuda"), perr=torch.full((n,), fill, dtype=dt, device="cuda"),
                rerr=torch.full((n,), fill, dtype=dt, device="cuda"),
                iters=torch.full((n,), 7, dtype=torch.int32, device="cuda"),
                flags=torch.full((n,), 7, dtype=torch.uint8, device="cuda"),
                attempt=torch.full((n,), 9, dtype=torch.uint8, device="cuda"),
                counters=torch.full((4,), 5, dtype=torch.int64, device="cuda"),
                stats=torch.full((3,), 5, dtype=torch.int64, device="cuda"))


def _scratch(cuda_lib, n, extra=8):
    nb = ctypes.c_int64()
    assert cuda_lib.pnp_ik_multistart_scratch_bytes(n, ctypes.byref(nb)) == 0
    return torch.zeros(nb.value // 4 + extra, dtype=torch.int32, device="cuda"), nb.value


def _call(cuda_lib, dt, tp, tq, q0, stride, n, seeds_p, k, params, o, scratch_p, **over):
    """The C entry point with the outputs of o (an _outs dict); keyword arguments replace a pointer."""
    fn = cuda_lib.pnp_ik_pose_solve_multistart_f32 if dt == torch.float32 else cuda_lib.pnp_ik_pose_solve_multistart_f64
    ptr = {key: over[key] if key in over else _p(v) for key, v in o.items()}
    return fn(_p(tp), _p(tq), _p(q0), stride, n, seeds_p, k, ctypes.byref(params), 1e-2, 1.0, ptr["q"], ptr["fpos"],
              ptr["fquat"], ptr["perr"], ptr["rerr"], ptr["iters"], ptr["flags"], ptr["attempt"], ptr["counters"],
              ptr["stats"], scratch_p, torch.cuda.current_stream().cuda_stream)


@pytest.mark.parametrize("dtype", list(DTYPES))
def test_null_optional_outputs(tree, cuda_lib, dtype):
    """final_pos, final_quat, pos_err, rot_err, iters (attempt 0's iterations then live in scratch), attempt, counters and
    restart_stats may be NULL; the outputs that remain equal those of the full call, and so do the counters."""
    dt = DTYPES[dtype]
    tp, tq = (t.to(dt) for t in workload(tree, 1 << 13))
    n = len(tp)
    q0 = torch.tensor(NEUTRAL, dtype=dt, device="cuda")
    seeds = engine.ik_restart_seeds(8, dtype=dt)
    params = engine.ik_params()
    scratch, _ = _scratch(cuda_lib, n)
    full, part = _outs(n, dt), _outs(n, dt)
    full["counters"].zero_(), part["counters"].zero_(), full["stats"].zero_()
    assert _call(cuda_lib, dt, tp, tq, q0, 0, n, _p(seeds), 8, params, full, _p(scratch)) == 0
    nulls = dict(fpos=None, fquat=None, perr=None, rerr=None, iters=None, attempt=None, stats=None)
    assert _call(cuda_lib, dt, tp, tq, q0, 0, n, _p(seeds), 8, params, part, _p(scratch), **nulls) == 0
    torch.cuda.synchronize()
    for key in ("q", "flags", "counters"):
        assert torch.equal(part[key], full[key]), key
    for key in ("fpos", "fquat", "perr", "rerr", "iters", "attempt", "stats"):
        assert torch.equal(part[key], _outs(n, dt)[key]), key  # untouched
    assert int(full["attempt"].count_nonzero()) > 100
    nulls["counters"] = None  # and only q and flags
    assert _call(cuda_lib, dt, tp, tq, q0, 0, n, _p(seeds), 8, params, part, _p(scratch), **nulls) == 0
    torch.cuda.synchronize()
    assert torch.equal(part["q"], full["q"]) and torch.equal(part["flags"], full["flags"])


@pytest.mark.parametrize("dtype", list(DTYPES))
def test_rejected_arguments_leave_outputs_untouched(tree, cuda_lib, dtype):
    dt = DTYPES[dtype]
    n = 256
    tp, tq = (t.to(dt) for t in w_cold(tree, n))
    q0 = torch.tensor(NEUTRAL, dtype=dt, device="cuda")
    seeds = engine.ik_restart_seeds(4, dtype=dt)
    params = engine.ik_params()
    scratch, _ = _scratch(cuda_lib, n)
    o = _outs(n, dt)
    before = {k: v.clone() for k, v in o.items()}

    def call(seeds_p, k, scratch_p, **over):
        return _call(cuda_lib, dt, tp, tq, q0, 0, n, seeds_p, k, params, o, scratch_p, **over)

    s, sc = _p(seeds), _p(scratch)
    cases = [(s, -1, sc, {}), (s, 256, sc, {}), (None, 4, sc, {}), (s, 4, None, {}), (s, 4, sc + 4, {}),
             (s, 4, sc, dict(flags=None)),
             (_p(o["q"]), 1, sc, {}), (_p(o["fquat"]), 1, sc, {}), (_p(o["rerr"]), 1, sc, {}),
             (_p(o["counters"]), 1, sc, {}), (_p(o["stats"]), 1, sc, {}), (_p(o["iters"]), 1, sc, {}),
             (s, 4, _p(o["q"]), {}), (s, 4, _p(o["fquat"]), {}), (s, 4, _p(o["attempt"]) - 16, {}),
             (s, 4, _p(o["flags"]) - 16, {}), (s, 4, _p(o["counters"]) - 16, {}), (sc + 1024, 4, sc, {})]
    for c in cases:
        assert call(c[0], c[1], c[2], **c[3]) == -1, c
    torch.cuda.synchronize()
    for k, v in before.items():
        assert torch.equal(o[k], v), k
    assert call(s, 4, sc) == 0  # and the same call with valid arguments runs


def test_stream_order_without_synchronisation(tree):
    tp, tq = (t.float() for t in workload(tree))
    op, oq = (t.float() for t in w_cold(tree, len(tp), seed=11))
    q0 = torch.tensor(NEUTRAL, dtype=torch.float32, device="cuda")
    seeds = engine.ik_restart_seeds(8)
    params = engine.ik_params()

    def sequence(sync):
        a = engine.ik_pose_solve_multistart(tp, tq, q0, seeds, params)
        if sync:
            torch.cuda.synchronize()
        b = engine.ik_pose_solve(tp, tq, a["q"], params)  # warm start from the multistart's q_out
        if sync:
            torch.cuda.synchronize()
        a2 = engine.ik_pose_solve_multistart(op, oq, q0, seeds, params)
        c = engine.ik_pose_solve(op, oq, q0, params)  # other buffers: may overlap with the restarts' launches
        torch.cuda.synchronize()
        return [bits(x) for x in (a, b, a2, c)], a["attempt"].clone()

    (ref, att), (got, att2) = sequence(True), sequence(False)
    for x, y in zip(ref, got):
        assert_rows(y, x)
    assert torch.equal(att, att2) and int(att.count_nonzero()) > 1000
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        r = engine.ik_pose_solve_multistart(tp, tq, q0, seeds, params)
    s.synchronize()
    assert_rows(bits(r), ref[0])
    assert torch.equal(r["attempt"], att)


def test_graph_capture_replays_on_new_inputs(tree, cuda_lib):
    tp_s, tq_s = (t.float() for t in workload(tree, 1 << 15))
    n = len(tp_s)
    q0 = torch.tensor(NEUTRAL, dtype=torch.float32, device="cuda")
    seeds = engine.ik_restart_seeds(8)
    params = engine.ik_params()
    scratch, _ = _scratch(cuda_lib, n, 0)
    o = _outs(n, torch.float32)
    o["counters"].zero_()

    def call():
        _lib.check(_call(cuda_lib, torch.float32, tp_s, tq_s, q0, 0, n, _p(seeds), 8, params, o, _p(scratch), stats=None),
                   "pose multistart")

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        call()  # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        call()
    new_p, new_q = (t.float() for t in w_cold(tree, n, seed=21))
    tp_s.copy_(new_p), tq_s.copy_(new_q)
    o["counters"].zero_()
    g.replay()
    torch.cuda.synchronize()
    got = bits(dict(q=o["q"], final_pos=o["fpos"], final_quat=o["fquat"], pos_error=o["perr"], rot_error=o["rerr"],
                    iterations=o["iters"], converged=(o["flags"] & 1) != 0, success=(o["flags"] & 2) != 0))
    got = {k: v.clone() for k, v in got.items()}
    got_attempt, c_graph = o["attempt"].clone(), o["counters"].clone()
    counters = torch.zeros(4, dtype=torch.int64, device="cuda")
    r = engine.ik_pose_solve_multistart(new_p, new_q, q0, seeds, params, counters=counters)
    torch.cuda.synchronize()
    assert int(r["attempt"].count_nonzero()) > 1000
    assert_rows(got, bits(r))
    assert torch.equal(got_attempt, r["attempt"]) and torch.equal(c_graph, counters)


def test_controller_seeds(tree, kin_model):
    data = KinematicData(kin_model)
    seeds = engine.ik_restart_seeds(8)
    tp, tq = workload(tree, 4096)
    for precision in ("fp32", "fp64"):
        ctl = JacobianIKController(kin_model, data, precision=precision)
        dt = torch.float32 if precision == "fp32" else torch.float64
        r = ctl.solve_pose(tp, tq, NEUTRAL, seeds=seeds)
        e = engine.ik_pose_solve_multistart(tp.to(dt), tq.to(dt), torch.tensor(NEUTRAL, dtype=dt, device="cuda"),
                                            seeds.to(dt), engine.ik_params())
        assert_rows(bits(r), bits(e), what=precision)
        assert torch.equal(r["attempt"], e["attempt"])
        p = ctl.solve_pose(tp, tq, NEUTRAL)  # without seeds: the plain solve
        assert "attempt" not in p and torch.equal(p["success"], e["success"] & (e["attempt"] == 0))
    r32 = engine.ik_pose_solve_multistart(tp.float(), tq.float(), torch.tensor(NEUTRAL, device="cuda"), seeds,
                                          engine.ik_params())
    i = int(torch.nonzero(r32["attempt"]).flatten()[0])  # a query a restart rescues (solve_ik runs FP32)
    one = solve_ik(kin_model, data, "ee_center_site", tp[i].cpu().numpy(), tq[i].cpu().numpy(), NEUTRAL,
                   seeds=seeds.cpu().numpy())
    assert one.success and not solve_ik(kin_model, data, "ee_center_site", tp[i].cpu().numpy(),
                                        tq[i].cpu().numpy(), NEUTRAL).success
    one = solve_ik(kin_model, data, "ee_center_site", tp[i].cpu().numpy(), tq[i].cpu().numpy(), NEUTRAL,
                   seeds=seeds.cpu().numpy())
    np.testing.assert_array_equal(one.q, r32["q"][i].double().cpu().numpy())
    np.testing.assert_array_equal(data.qpos[:7], one.q)
    assert one.iterations == int(r32["iterations"][i])

"""GPU: multi-start position IK (pnp_ik_solve_multistart_*, engine.ik_solve_multistart).

The specification is bit-identity: every returned row equals, bit for bit, the plain solve of the same layout,
precision and kinematics from the start ``attempt`` names, and ``attempt`` is the first successful one."""
import ctypes

import numpy as np
import pytest
import torch

from conftest import NEUTRAL
from mujoco_panda_pnp_b200 import KinematicData, KinematicTree, _lib, engine, synthetic
from mujoco_panda_pnp_b200.skills import JacobianIKController
from test_ik_multistart_oracle import multistart_batched

pytestmark = pytest.mark.gpu

LAYOUTS = {"sep32": (torch.float32, False), "packed32": (torch.float32, True), "f64": (torch.float64, False)}
FAR = [[2.5, 0.0, 0.5], [0.0, 0.0, 3.0], [-2.0, 1.5, 0.2], [1.0, -2.2, 1.0], [3.0, 3.0, 3.0], [0.0, 2.6, 0.8]]


@pytest.fixture(scope="module")
def tree(cuda_lib):
    t = KinematicTree.from_mjcf()
    engine.set_tree(t)
    return t


def cfg5(tree, n, seed=1234):
    qstar = synthetic.random_joint_configs(n, tree.lower, tree.upper, seed=seed, dtype=torch.float64).cuda()
    return engine.fk_jac(qstar, want_quat=False, want_jac=False)[0]


def workload(tree, n=1 << 16):
    """cfg5 targets, then unreachable ones and two NaN targets."""
    t = torch.cat([cfg5(tree, n), torch.tensor(FAR * 8, dtype=torch.float64, device="cuda"),
                   torch.full((2, 3), float("nan"), dtype=torch.float64, device="cuda")])
    return t


def seed_table(tree, dt):
    """seeds[0] = NEUTRAL (the broadcast q_init: never chosen for a query that failed from it), then 7 U(limits)."""
    s = torch.cat([torch.tensor(NEUTRAL, dtype=torch.float64)[None],
                   engine.ik_restart_seeds(7, tree.lower, tree.upper, seed=3, dtype=torch.float64, device="cpu")])
    return s.to(device="cuda", dtype=dt)


def bits(r):
    out = {}
    for k in ("q", "final_pos", "pos_error"):
        t = getattr(r, k).contiguous()
        out[k] = t.view(torch.int64 if t.dtype == torch.float64 else torch.int32)
    out["iterations"] = r.iterations.to(torch.int32)
    out["converged"], out["success"] = r.converged.clone(), r.success.clone()
    return out


def plain(targets, q_init, params, packed):
    return bits(engine.ik_solve(targets, q_init, params, packed=packed))


def expected(targets, q_init, seeds, params, packed):
    """The composition of plain calls: one from q_init, one per seed broadcast over all queries."""
    runs = [plain(targets, q_init, params, packed)] + [plain(targets, s, params, packed) for s in seeds]
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


def check_counters(r, counters):
    c = counters.cpu().numpy()
    assert c[0] == len(r.q)
    assert c[1] == int(r.converged.sum()) and c[2] == int(r.success.sum())
    assert c[3] == int(r.iterations.to(torch.int64).sum())


@pytest.mark.parametrize("kin", ["auto", "generic", "spec_lane", "spec_pair"])
@pytest.mark.parametrize("layout", list(LAYOUTS))
@pytest.mark.parametrize("bcast", [True, False])
def test_composition_identity(tree, layout, kin, bcast):
    dt, packed = LAYOUTS[layout]
    targets = workload(tree).to(dt)
    n = len(targets)
    q_init = torch.tensor(NEUTRAL, dtype=dt, device="cuda") if bcast else \
        synthetic.random_joint_configs(n, tree.lower, tree.upper, seed=5, dtype=torch.float64).to("cuda", dt)
    params = engine.ik_params(kinematics=kin)
    seeds = seed_table(tree, dt)
    counters = torch.zeros(4, dtype=torch.int64, device="cuda")
    stats = torch.zeros(3, dtype=torch.int64, device="cuda")
    r = engine.ik_solve_multistart(targets, q_init, seeds, params, counters=counters, restart_stats=stats, packed=packed)
    attempt, exp, succ = expected(targets, q_init, seeds, params, packed)
    got = bits(r)
    for key in exp:
        assert torch.equal(got[key], exp[key]), key
    assert torch.equal(r.attempt.long(), attempt)
    check_counters(r, counters)
    s = stats.cpu().numpy()
    rescued = attempt > 0
    assert s[0] == int((~succ[0]).sum()) and s[1] == int(rescued.sum())
    assert s[2] >= int(r.iterations[rescued].to(torch.int64).sum())
    assert s[1] > 20 and (~r.success).sum() >= len(FAR) * 8 + 2  # failures rescued; unreachable / NaN rows left
    if bcast:
        assert not (attempt == 1).any()  # seeds[0] == q_init: fails wherever attempt 0 failed
    # somewhere an earlier seed won over a later one that also succeeds
    tie = torch.zeros_like(rescued)
    for k in range(2, len(seeds)):
        tie |= (attempt == k) & succ[k + 1:].any(0)
    assert tie.any()


def test_fp64_matches_the_c_statement(tree, oracle_chain):
    """FP64 kernel vs oracle composition (FP64 C statement): the attempt index agrees except where one side crosses
    the threshold a step earlier (at most 1 query); where they agree, converged q agree to 1e-7."""
    targets = cfg5(tree, 1 << 14, seed=77)
    seeds = engine.ik_restart_seeds(8, dtype=torch.float64)
    r = engine.ik_solve_multistart(targets, torch.tensor(NEUTRAL, dtype=torch.float64, device="cuda"), seeds,
                                   engine.ik_params())
    att_ref, ref = multistart_batched(oracle_chain, targets.cpu().numpy(), NEUTRAL, seeds.cpu().numpy())
    att = r.attempt.long().cpu().numpy()
    assert (att_ref > 0).sum() > 10
    assert int((att != att_ref).sum()) <= 1
    same = (att == att_ref) & ref["converged"]
    np.testing.assert_allclose(r.q.cpu().numpy()[same], ref["q"][same], atol=1e-7)
    assert (r.iterations.cpu().numpy()[same] != ref["iterations"][same]).sum() <= 1


def test_k0_is_the_plain_solve(tree):
    targets = workload(tree, 1 << 14).float()
    q0 = torch.tensor(NEUTRAL, dtype=torch.float32, device="cuda")
    params = engine.ik_params()
    c0, c1 = (torch.zeros(4, dtype=torch.int64, device="cuda") for _ in range(2))
    n0 = _lib.launch_count()
    p = engine.ik_solve(targets, q0, params, counters=c0)
    n1 = _lib.launch_count()
    r = engine.ik_solve_multistart(targets, q0, torch.empty((0, 7), device="cuda"), params, counters=c1)
    n2 = _lib.launch_count()
    assert n2 - n1 == n1 - n0
    for key, v in bits(p).items():
        assert torch.equal(bits(r)[key], v), key
    assert torch.equal(c0, c1) and not r.attempt.any()


@pytest.mark.parametrize("case", ["all_succeed", "all_unreachable"])
def test_nothing_to_rescue(tree, case):
    if case == "all_succeed":
        q = torch.tensor(NEUTRAL)[None] + 0.05 * (torch.rand((4096, 7), generator=torch.Generator().manual_seed(1)) - 0.5)
        targets = engine.fk_jac(q.cuda().float(), want_quat=False, want_jac=False)[0]
    else:
        targets = torch.tensor(FAR * 700, dtype=torch.float32, device="cuda")
    q0 = torch.tensor(NEUTRAL, dtype=torch.float32, device="cuda")
    params = engine.ik_params()
    stats = torch.zeros(3, dtype=torch.int64, device="cuda")
    r = engine.ik_solve_multistart(targets, q0, engine.ik_restart_seeds(8), params, restart_stats=stats)
    p = plain(targets, q0, params, True)
    for key, v in p.items():
        assert torch.equal(bits(r)[key], v), key
    assert not r.attempt.any()
    s = stats.cpu().numpy()
    if case == "all_succeed":
        assert bool(r.success.all()) and s[0] == 0
    else:
        assert not r.success.any() and s[0] == len(targets) and s[1] == 0


def test_batch_sizes(tree, cuda_lib):
    sm = ctypes.c_int32()
    cuda_lib.pnp_device_info(ctypes.byref(sm), None, None)
    pool = workload(tree, 1 << 15).float()
    pool = pool[torch.randperm(len(pool), generator=torch.Generator().manual_seed(2)).cuda()]
    seeds = engine.ik_restart_seeds(8)
    params = engine.ik_params()
    q0 = torch.tensor(NEUTRAL, dtype=torch.float32, device="cuda")
    for n in (0, 1, 31, 33, sm.value * 128 - 1, sm.value * 128 + 1):
        t = pool[:n].contiguous()
        r = engine.ik_solve_multistart(t, q0, seeds, params)
        attempt, exp, _ = expected(t, q0, seeds, params, True)
        for key in exp:
            assert torch.equal(bits(r)[key], exp[key]), (n, key)
        assert torch.equal(r.attempt.long(), attempt), n


def test_large_batch_with_drain_hand_over(tree):
    """2^22 queries: attempt 0 runs the pair kernel with its resume launch; check every rescued row and a sample."""
    n = 1 << 22
    targets = cfg5(tree, n, seed=9).float()
    q0 = torch.tensor(NEUTRAL, dtype=torch.float32, device="cuda")
    seeds = engine.ik_restart_seeds(8)
    params = engine.ik_params()
    counters = torch.zeros(4, dtype=torch.int64, device="cuda")
    r = engine.ik_solve_multistart(targets, q0, seeds, params, counters=counters)
    p = plain(targets, q0, params, True)
    got = bits(r)
    a = r.attempt.long()
    keep = a == 0
    for key in p:
        assert torch.equal(got[key][keep], p[key][keep]), key
    check_counters(r, counters)
    rows = torch.nonzero(~p["success"]).flatten()
    assert len(rows) > 1000
    sub = targets[rows].contiguous()
    attempt, exp, _ = expected(sub, q0, seeds, params, True)
    assert torch.equal(a[rows], attempt)
    for key in exp:
        assert torch.equal(got[key][rows], exp[key]), key
    assert int(a.count_nonzero()) >= 0.98 * len(rows)  # the default table rescues nearly every failure
    r2 = engine.ik_solve_multistart(targets, q0, seeds, params)
    for key, v in bits(r2).items():
        assert torch.equal(v, got[key]), key
    assert torch.equal(r2.attempt, r.attempt)


def test_runs_are_bit_identical(tree):
    targets = workload(tree).float()
    q0 = torch.tensor(NEUTRAL, dtype=torch.float32, device="cuda")
    seeds = engine.ik_restart_seeds(8)
    for packed in (True, False):
        a = engine.ik_solve_multistart(targets, q0, seeds, engine.ik_params(), packed=packed)
        b = engine.ik_solve_multistart(targets, q0, seeds, engine.ik_params(), packed=packed)
        for key, v in bits(a).items():
            assert torch.equal(bits(b)[key], v), key
        assert torch.equal(a.attempt, b.attempt)


def _p(t):
    return None if t is None else t.data_ptr()


@pytest.mark.parametrize("layout", list(LAYOUTS))
def test_rejected_arguments_leave_outputs_untouched(tree, cuda_lib, layout):
    dt, packed = LAYOUTS[layout]
    n = 256
    targets = cfg5(tree, n).to(dt)
    q0 = torch.tensor(NEUTRAL, dtype=dt, device="cuda")
    seeds = engine.ik_restart_seeds(4, dtype=dt)
    params = engine.ik_params()
    nb = ctypes.c_int64()
    assert cuda_lib.pnp_ik_multistart_scratch_bytes(n, ctypes.byref(nb)) == 0
    assert cuda_lib.pnp_ik_multistart_scratch_bytes(-1, ctypes.byref(nb)) == -1
    scratch = torch.zeros(nb.value // 4 + 8, dtype=torch.int32, device="cuda")
    if packed:
        outs = dict(q8=torch.full((n, 8), 7.0, device="cuda"), aux=torch.full((n, 4), 7.0, device="cuda"))
    else:
        outs = dict(q=torch.full((n, 7), 7.0, dtype=dt, device="cuda"), fpos=torch.full((n, 3), 7.0, dtype=dt, device="cuda"),
                    err=torch.full((n,), 7.0, dtype=dt, device="cuda"), iters=torch.full((n,), 7, dtype=torch.int32, device="cuda"),
                    flags=torch.full((n,), 7, dtype=torch.uint8, device="cuda"))
    attempt = torch.full((n,), 9, dtype=torch.uint8, device="cuda")
    counters = torch.full((4,), 5, dtype=torch.int64, device="cuda")
    stats = torch.full((3,), 5, dtype=torch.int64, device="cuda")
    before = {k: v.clone() for k, v in {**outs, "attempt": attempt, "counters": counters, "stats": stats}.items()}

    def call(seeds_p, k, scratch_p, flags_p="default"):
        st = torch.cuda.current_stream().cuda_stream
        if packed:
            return cuda_lib.pnp_ik_solve_multistart_packed_f32(
                _p(targets), _p(q0), 0, n, seeds_p, k, ctypes.byref(params), _p(outs["q8"]), _p(outs["aux"]), _p(attempt),
                _p(counters), _p(stats), scratch_p, st)
        fn = cuda_lib.pnp_ik_solve_multistart_f32 if dt == torch.float32 else cuda_lib.pnp_ik_solve_multistart_f64
        fl = _p(outs["flags"]) if flags_p == "default" else flags_p
        return fn(_p(targets), _p(q0), 0, n, seeds_p, k, ctypes.byref(params), _p(outs["q"]), _p(outs["fpos"]), _p(outs["err"]),
                  _p(outs["iters"]), fl, _p(attempt), _p(counters), _p(stats), scratch_p, st)

    first_out = outs["q8"] if packed else outs["q"]
    cases = [(_p(seeds), -1, _p(scratch)), (_p(seeds), 256, _p(scratch)), (None, 4, _p(scratch)), (_p(seeds), 4, None),
             (_p(seeds), 4, _p(scratch) + 4), (_p(first_out), 1, _p(scratch)), (_p(seeds), 4, _p(first_out)),
             (_p(seeds), 4, _p(attempt) - 16 * (nb.value // 16)), (_p(counters), 1, _p(scratch))]
    for c in cases:
        assert call(*c) == -1, c
    if not packed:
        assert call(_p(seeds), 4, _p(scratch), None) == -1
    torch.cuda.synchronize()
    now = {**outs, "attempt": attempt, "counters": counters, "stats": stats}
    for k, v in before.items():
        assert torch.equal(now[k], v), k
    assert call(_p(seeds), 4, _p(scratch)) == 0  # and the same call with valid arguments runs


def test_stream_order_without_synchronisation(tree):
    targets = workload(tree).float()
    other = cfg5(tree, len(targets), seed=11).float()
    q0 = torch.tensor(NEUTRAL, dtype=torch.float32, device="cuda")
    seeds = engine.ik_restart_seeds(8)
    params = engine.ik_params()

    def sequence(sync):
        a = engine.ik_solve_multistart(targets, q0, seeds, params, packed=False)
        if sync:
            torch.cuda.synchronize()
        b = engine.ik_solve(targets, a.q, params)  # warm start from the multistart's q_out
        if sync:
            torch.cuda.synchronize()
        a2 = engine.ik_solve_multistart(other, q0, seeds, params)
        c = engine.ik_solve(other, q0, params)  # other buffers: may overlap with the restarts' launches
        torch.cuda.synchronize()
        return [bits(x) for x in (a, b, a2, c)]

    ref, got = sequence(True), sequence(False)
    for x, y in zip(ref, got):
        for key in x:
            assert torch.equal(x[key], y[key]), key
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        r = engine.ik_solve_multistart(targets, q0, seeds, params, packed=False)
    s.synchronize()
    for key, v in ref[0].items():
        assert torch.equal(bits(r)[key], v), key


def test_graph_capture_replays_on_new_inputs(tree, cuda_lib):
    n = 1 << 15
    t_static = workload(tree, n).float()
    n = len(t_static)
    q0 = torch.tensor(NEUTRAL, dtype=torch.float32, device="cuda")
    seeds = engine.ik_restart_seeds(8)
    params = engine.ik_params()
    nb = ctypes.c_int64()
    cuda_lib.pnp_ik_multistart_scratch_bytes(n, ctypes.byref(nb))
    scratch = torch.empty(nb.value // 4, dtype=torch.int32, device="cuda")
    q8, aux = torch.empty((n, 8), device="cuda"), torch.empty((n, 4), device="cuda")
    attempt = torch.empty(n, dtype=torch.uint8, device="cuda")
    counters = torch.zeros(4, dtype=torch.int64, device="cuda")

    def call():
        _lib.check(cuda_lib.pnp_ik_solve_multistart_packed_f32(
            _p(t_static), _p(q0), 0, n, _p(seeds), 8, ctypes.byref(params), _p(q8), _p(aux), _p(attempt), _p(counters),
            None, _p(scratch), torch.cuda.current_stream().cuda_stream), "multistart")

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        call()  # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        call()
    new = cfg5(tree, n, seed=21).float()
    t_static.copy_(new)
    counters.zero_()
    g.replay()
    torch.cuda.synchronize()
    c_graph = counters.clone()
    q, err, fpos, word = engine.unpack_ik(q8.clone(), aux.clone())
    got = bits(engine.BatchIKResult(q=q, final_pos=fpos, pos_error=err, word=word))
    got_attempt = attempt.clone()
    counters.zero_()
    r = engine.ik_solve_multistart(new, q0, seeds, params, counters=counters)
    torch.cuda.synchronize()
    assert int(r.attempt.count_nonzero()) > 0
    for key, v in bits(r).items():
        assert torch.equal(got[key], v), key
    assert torch.equal(got_attempt, r.attempt) and torch.equal(c_graph, counters)


def test_controller_seeds(tree, kin_model):
    model = kin_model
    data = KinematicData(model)
    seeds = engine.ik_restart_seeds(8)
    targets = workload(tree, 4096).float()
    for precision in ("fp32", "fp64"):
        ctl = JacobianIKController(model, data, precision=precision)
        dt = torch.float32 if precision == "fp32" else torch.float64
        r = ctl.solve_batch(targets, NEUTRAL, seeds=seeds)
        e = engine.ik_solve_multistart(targets.to(dt), torch.tensor(NEUTRAL, dtype=dt, device="cuda"), seeds.to(dt),
                                       engine.ik_params())
        for key, v in bits(e).items():
            assert torch.equal(bits(r)[key], v), key
        assert torch.equal(r.attempt, e.attempt)
        i = int(torch.nonzero(e.attempt).flatten()[0])  # a query rescued by a restart
        one = ctl.solve(targets[i].double().cpu().numpy(), NEUTRAL, seeds=seeds.cpu().numpy())
        assert one.success
        np.testing.assert_array_equal(one.q, e.q[i].double().cpu().numpy())
        np.testing.assert_array_equal(data.qpos[:7], one.q)
        assert one.iterations == int(e.iterations[i])
    a, b = engine.ik_restart_seeds(8, seed=4), engine.ik_restart_seeds(8, seed=4)
    assert a.is_cuda and torch.equal(a, b)
    lo, hi = torch.as_tensor(tree.lower, device="cuda"), torch.as_tensor(tree.upper, device="cuda")
    assert ((a.double() >= lo) & (a.double() <= hi)).all()

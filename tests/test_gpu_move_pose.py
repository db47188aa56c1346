"""GPU: the pose-mode move planner (pnp_move_ik_plan_pose_*, move_pose_plan_kernel) against its FP64 statement
(oracle/move_pose_oracle.py), FP32 against FP64, and the stream / argument / storage rules of the entry point."""
import ctypes
import math
import types

import numpy as np
import pytest
import torch

from conftest import ASSET, NEUTRAL
from mujoco_panda_pnp_b200 import KinematicData, KinematicModel, KinematicTree, _lib, engine
from mujoco_panda_pnp_b200.skills import MoveIKSkill, plan_pose_moves
from oracle import mj_oracle, move_pose_oracle
from test_move_pose_oracle import check_invariants, neutral_pose, pose_workload

pytestmark = pytest.mark.gpu

OUT_KEYS = ("pos_traj", "quat_traj", "q_traj", "traj_len", "q_final", "n_solves", "status")


@pytest.fixture(scope="module")
def tree(cuda_lib):
    t = KinematicTree.from_mjcf()
    engine.set_tree(t)
    return t


def edge_cases(oracle_chain):
    """(q_start, goal_pos, goal_quat) rows: a rotation-only move, a translation-only one, an unreachable goal, a NaN
    goal position, an infinite one, a NaN quaternion and a zero quaternion."""
    p0, r0 = neutral_pose(oracle_chain)
    qz = np.array([math.cos(math.pi / 4), 0.0, 0.0, math.sin(math.pi / 4)])
    rows = [(p0, mj_oracle.mju_mulQuat(qz, r0)), (p0 + np.array([0.1, 0.15, -0.1]), r0), (np.array([2.0, 0.0, 0.5]), r0),
            (np.array([np.nan, 0.0, 0.5]), r0), (np.array([1.0, np.inf, 0.5]), r0),
            (p0, np.array([np.nan, 0.0, 0.0, 0.0])), (p0, np.zeros(4))]
    return (np.tile(NEUTRAL, (len(rows), 1)), np.array([r[0] for r in rows]), np.array([r[1] for r in rows]))


def gpu(x, dt=torch.float64):
    return torch.tensor(np.asarray(x), dtype=dt, device="cuda")


def host(out):
    return {k: (None if out[k] is None else out[k].double().cpu().numpy() if out[k].is_floating_point()
                else out[k].cpu().numpy()) for k in OUT_KEYS}


@pytest.fixture(scope="module")
def fp64_cases(tree, oracle_model, oracle_chain):
    """128 workload envs plus the edge cases, with the statement's plans."""
    qs, gp, gq = pose_workload(oracle_model, oracle_chain, 128, seed=1)
    eq, ep, eg = edge_cases(oracle_chain)
    qs, gp, gq = np.concatenate([qs, eq]), np.concatenate([gp, ep]), np.concatenate([gq, eg])
    want = [move_pose_oracle.plan_pose(oracle_model, qs[k], gp[k], gq[k]) for k in range(len(qs))]
    return qs, gp, gq, want


def assert_matches_statement(got, want):
    for k, w in enumerate(want):
        L = len(w["pos_traj"])
        assert (int(got["traj_len"][k]), int(got["status"][k]), int(got["n_solves"][k])) == (L, w["status"], w["n_solves"]), k
        np.testing.assert_allclose(got["pos_traj"][k, :L], w["pos_traj"], rtol=0, atol=1e-9)
        np.testing.assert_allclose(got["quat_traj"][k, :L], w["quat_traj"], rtol=0, atol=1e-9)
        np.testing.assert_allclose(got["q_traj"][k, :L], w["q_traj"], rtol=0, atol=1e-9)
        np.testing.assert_allclose(got["q_final"][k], w["q_final"], rtol=0, atol=1e-9)


@pytest.mark.parametrize("kin", ["specialized", "generic"])
def test_fp64_kernel_matches_statement(fp64_cases, oracle_model, kin):
    qs, gp, gq, want = fp64_cases
    got = host(engine.move_ik_plan_pose(gpu(qs), gpu(gp), gpu(gq), engine.ik_params(kinematics=kin)))
    assert_matches_statement(got, want)
    # the edge rows end as the statement says: BROKE at once for the broken goals, CAPPED for the unreachable one
    assert list(got["status"][-5:]) == [move_pose_oracle.CAPPED] + [move_pose_oracle.BROKE] * 4
    assert list(got["traj_len"][-4:]) == [1] * 4
    # other parameters: a short cap, and solves that cannot converge (three rejections, BROKE)
    for kw, ik in ((dict(max_traj_points=5), {}), ({}, dict(max_iters=0))):
        sel = slice(0, 16)
        got = host(engine.move_ik_plan_pose(gpu(qs[sel]), gpu(gp[sel]), gpu(gq[sel]), engine.ik_params(kinematics=kin, **ik), **kw))
        want2 = [move_pose_oracle.plan_pose(oracle_model, qs[k], gp[k], gq[k], **kw, **ik) for k in range(16)]
        assert_matches_statement(got, want2)


@pytest.fixture(scope="module")
def fp32_vs_fp64(tree, oracle_model, oracle_chain):
    qs, gp, gq = pose_workload(oracle_model, oracle_chain, 4096, seed=2)
    p32 = engine.move_ik_plan_pose(gpu(qs, torch.float32), gpu(gp, torch.float32), gpu(gq, torch.float32), engine.ik_params())
    p64 = engine.move_ik_plan_pose(gpu(qs), gpu(gp), gpu(gq), engine.ik_params())
    return qs, gp, gq, host(p32), host(p64)


def test_fp32_kernel_against_fp64_kernel(fp32_vs_fp64):
    """Status agreement and the gap between the final poses of plans that are OK in both.  Measured on one B200
    (4096 envs): see the bounds below, each at most twice the observed value."""
    _, _, _, a, b = fp32_vs_fp64
    agree = float((a["status"] == b["status"]).mean())
    ok = (a["status"] == 0) & (b["status"] == 0)
    ka, kb = a["traj_len"][ok] - 1, b["traj_len"][ok] - 1
    rows = np.nonzero(ok)[0]
    gap_p = np.linalg.norm(a["pos_traj"][rows, ka] - b["pos_traj"][rows, kb], axis=1).max()
    gap_r = move_pose_oracle.quat_angle(a["quat_traj"][rows, ka], b["quat_traj"][rows, kb]).max()
    same_len = float((a["traj_len"] == b["traj_len"]).mean())
    print(f"fp32 vs fp64: status agreement {agree:.5f}, same length {same_len:.4f}, OK in both {ok.mean():.4f}, "
          f"final pose gap {gap_p:.3e} m / {gap_r:.3e} rad")
    assert 1.0 - agree <= 2 * DISAGREE_OBSERVED
    assert gap_p <= 2 * GAP_POS_OBSERVED and gap_r <= 2 * GAP_ROT_OBSERVED


# observed on one B200 by test_fp32_kernel_against_fp64_kernel (4096 workload envs, seed 2): every status and every
# plan length agree, all 4096 plans are OK in both, final pose gap 6.96e-4 m / 1.62e-3 rad
DISAGREE_OBSERVED = 0.0
GAP_POS_OBSERVED = 7.0e-4
GAP_ROT_OBSERVED = 1.62e-3


def test_fp32_plans_hold_the_invariants(fp32_vs_fp64, oracle_model, oracle_chain):
    """Every FP32 plan satisfies the statement's invariants, FK taken in FP64 from its q_traj (1e-5 m / 1e-4 rad)."""
    _, gp, gq, a, _ = fp32_vs_fp64
    for k in range(len(gp)):
        L = int(a["traj_len"][k])
        plan = dict(pos_traj=a["pos_traj"][k, :L], quat_traj=a["quat_traj"][k, :L], q_traj=a["q_traj"][k, :L],
                    n_solves=int(a["n_solves"][k]), status=int(a["status"][k]))
        check_invariants(oracle_model, oracle_chain, plan, gp[k], gq[k], 1e-5, 1e-4)
        assert np.array_equal(a["q_final"][k], a["q_traj"][k, L - 1])


def bits_equal(x, y):
    for k in OUT_KEYS:
        if x[k] is None or y[k] is None:
            assert x[k] is None and y[k] is None, k
        else:
            assert torch.equal(x[k], y[k]), k


def test_schedule_independence_and_nullable_joint_path(tree, oracle_model, oracle_chain):
    """An env's FP32 outputs are bit-identical alone, in a batch of 2^16 and in a permuted batch; q_traj = NULL
    leaves every other output bit-identical."""
    n = 1 << 16
    qs, gp, gq = (gpu(x, torch.float32) for x in pose_workload(oracle_model, oracle_chain, n, seed=3))
    pk = engine.ik_params()
    full = engine.move_ik_plan_pose(qs, gp, gq, pk)
    perm = torch.randperm(n, generator=torch.Generator().manual_seed(0)).cuda()
    shuf = engine.move_ik_plan_pose(qs[perm], gp[perm], gq[perm], pk)
    bits_equal({k: full[k][perm] for k in OUT_KEYS}, shuf)
    for e in (0, 1, 4097, n - 1):
        one = engine.move_ik_plan_pose(qs[e:e + 1], gp[e:e + 1], gq[e:e + 1], pk)
        bits_equal({k: full[k][e:e + 1] for k in OUT_KEYS}, one)
    noq = engine.move_ik_plan_pose(qs, gp, gq, pk, want_q_traj=False)
    bits_equal({k: (None if k == "q_traj" else full[k]) for k in OUT_KEYS}, noq)


def raw_call(lib, dt, qs, gp, gq, mp, pk, n, out):
    fn = lib.pnp_move_ik_plan_pose_f32 if dt == torch.float32 else lib.pnp_move_ik_plan_pose_f64
    p = lambda t: None if t is None else t.data_ptr()  # noqa: E731
    return fn(p(qs), p(gp), p(gq), n, mp if mp is None else ctypes.byref(mp), pk if pk is None else ctypes.byref(pk),
              *(p(out[k]) for k in OUT_KEYS), None, torch.cuda.current_stream().cuda_stream)


def test_overflow_writes_nothing_past_the_cap(tree, oracle_model, oracle_chain, cuda_lib):
    """traj_cap < max_traj_points + 1: OVERFLOW on the plans that outgrow it, their first traj_cap points as in an
    uncapped run, and sentinel rows behind the last env's storage untouched."""
    n, cap, pad = 256, 8, 4
    qs, gp, gq = (gpu(x, torch.float32) for x in pose_workload(oracle_model, oracle_chain, n, seed=4))
    pk = engine.ik_params()
    full = engine.move_ik_plan_pose(qs, gp, gq, pk)
    sentinel = -12345.0
    store = {k: torch.full((n * cap + pad, w), sentinel, dtype=torch.float32, device="cuda")
             for k, w in (("pos_traj", 3), ("quat_traj", 4), ("q_traj", 7))}
    out = dict(store, traj_len=torch.empty(n, dtype=torch.int32, device="cuda"), q_final=torch.empty((n, 7), device="cuda"),
               n_solves=torch.empty(n, dtype=torch.int32, device="cuda"), status=torch.empty(n, dtype=torch.int32, device="cuda"))
    mp = _lib.PnpMovePoseParams(0.01, 0.05, 0.01, 0.05, 1e-2, 1.0, 200, cap)
    assert raw_call(cuda_lib, torch.float32, qs, gp, gq, mp, pk, n, out) == 0
    torch.cuda.synchronize()
    for k in ("traj_len", "q_final", "n_solves"):
        assert torch.equal(out[k], full[k]), k
    over = full["traj_len"] > cap
    assert bool(over.any()) and bool((~over).any())
    assert torch.equal((out["status"] & 4) != 0, over) and torch.equal(out["status"] & 3, full["status"])
    for k in ("pos_traj", "quat_traj", "q_traj"):
        got = store[k][: n * cap].view(n, cap, -1)
        L = full["traj_len"].clamp(max=cap)
        mask = torch.arange(cap, device="cuda")[None, :] < L[:, None]
        assert torch.equal(got[mask], full[k][:, :cap][mask]), k
        assert bool((got[~mask] == sentinel).all()), k
        assert bool((store[k][n * cap:] == sentinel).all()), k


def test_rejected_arguments_launch_nothing(tree, cuda_lib):
    n = 4
    qs = gpu(np.tile(NEUTRAL, (n, 1)), torch.float32)
    gp, gq = gpu(np.tile([1.2, 0.0, 0.6], (n, 1)), torch.float32), gpu(np.tile([0.0, 1.0, 0.0, 0.0], (n, 1)), torch.float32)
    base = lambda: _lib.PnpMovePoseParams(0.01, 0.05, 0.01, 0.05, 1e-2, 1.0, 200, 201)  # noqa: E731
    out = {k: torch.full(s, 7.0, device="cuda") for k, s in (("pos_traj", (n, 201, 3)), ("quat_traj", (n, 201, 4)),
                                                              ("q_traj", (n, 201, 7)), ("q_final", (n, 7)))}
    out.update({k: torch.full((n,), 7, dtype=torch.int32, device="cuda") for k in ("traj_len", "n_solves", "status")})
    snapshot = {k: v.clone() for k, v in out.items()}
    cases = []
    for field, value in (("pos_thresh", 5e-4), ("rot_thresh", 5e-3), ("step_size", 0.0), ("rot_step", -0.05),
                         ("ik_rot_thresh", 0.0), ("ik_rot_weight", 0.0), ("traj_cap", 0), ("max_traj_points", -1),
                         ("pos_thresh", float("nan"))):
        mp = base()
        setattr(mp, field, value)
        cases.append((field, mp, engine.ik_params(), n, {}))
    for k in ("pos_traj", "quat_traj", "traj_len", "q_final", "n_solves", "status"):
        cases.append((f"NULL {k}", base(), engine.ik_params(), n, {k: None}))
    cases += [("n >= 2^31", base(), engine.ik_params(), 1 << 31, {}), ("NULL move", None, engine.ik_params(), n, {}),
              ("NULL params", base(), None, n, {}), ("negative n", base(), engine.ik_params(), -1, {})]
    torch.cuda.synchronize()
    launches = cuda_lib.pnp_launch_count()
    for name, mp, pk, nn, swap in cases:
        assert raw_call(cuda_lib, torch.float32, qs, gp, gq, mp, pk, nn, dict(out, **swap)) == -1, name
    torch.cuda.synchronize()
    assert cuda_lib.pnp_launch_count() == launches
    for k in out:
        assert torch.equal(out[k], snapshot[k]), k
    with pytest.raises(ValueError):
        engine.move_ik_plan_pose(qs, gp, gq, engine.ik_params(pos_thresh=0.02))


def test_graph_replay_equals_eager_call(tree, oracle_model, oracle_chain):
    """Captured into a CUDA graph, the call replays exactly what an eager call on a non-default stream computes."""
    n = 4096
    qs, gp, gq = (gpu(x, torch.float32) for x in pose_workload(oracle_model, oracle_chain, n, seed=5))
    pk = engine.ik_params()
    side = torch.cuda.Stream()
    cnt = torch.zeros(4, dtype=torch.int64, device="cuda")
    with torch.cuda.stream(side):
        eager = engine.move_ik_plan_pose(qs, gp, gq, pk, counters=cnt)
    side.synchronize()
    assert int(cnt[0]) == int(eager["n_solves"].sum())
    s_qs, s_gp, s_gq = torch.zeros_like(qs), torch.zeros_like(gp), torch.zeros_like(gq)
    s_gq[:, 0] = 1.0
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        captured = engine.move_ik_plan_pose(s_qs, s_gp, s_gq, pk)
    s_qs.copy_(qs); s_gp.copy_(gp); s_gq.copy_(gq)
    g.replay()
    torch.cuda.synchronize()
    bits_equal(captured, eager)


class StubEnv:
    """The slice of FrankaEnv that MoveIKSkill touches: model / data, the EE orientation, set_mocap_pose."""

    def __init__(self, q):
        self.model = KinematicModel.from_xml_path(ASSET)
        self.data = KinematicData(self.model)
        self.data.qpos[:7] = q
        self.unwrapped = self
        self.sent = []
        self.action_space = types.SimpleNamespace(low=np.zeros(4))
        self._mujoco = types.SimpleNamespace(mj_step=lambda m, d, nstep=1: None)

    def get_ee_orientation(self):
        return np.array([0.0, 1.0, 0.0, 0.0])

    def set_mocap_pose(self, pos, quat):
        self.sent.append((np.array(pos), np.array(quat)))


def test_move_skill_with_target_quat_plans_poses(tree, oracle_chain):
    p0, r0 = neutral_pose(oracle_chain)
    qz = np.array([math.cos(math.pi / 8), 0.0, 0.0, math.sin(math.pi / 8)])
    target_pos, target_quat = p0 + np.array([0.05, -0.05, 0.0]), mj_oracle.mju_mulQuat(qz, r0)
    env = StubEnv(NEUTRAL)
    skill = MoveIKSkill(env, target_pos, target_quat=target_quat)
    skill.reset()
    want = plan_pose_moves(env.model, NEUTRAL[None], target_pos[None], target_quat[None])
    L = int(want["traj_len"][0])
    assert skill.status == int(want["status"][0]) == 0 and len(skill.pos_traj) == L > 1
    for key, got in (("pos_traj", skill.pos_traj), ("quat_traj", skill.quat_traj), ("q_traj", skill.q_traj)):
        assert np.array_equal(np.array(got), want[key][0, :L].double().cpu().numpy()), key
    while not skill.is_done():
        skill.step()
    assert len(env.sent) == L
    for k, (pos, quat) in enumerate(env.sent):
        assert np.array_equal(pos, skill.pos_traj[k]) and np.array_equal(quat, skill.quat_traj[k])
    # without target_quat the skill keeps the position-only plan and the start orientation
    plain = MoveIKSkill(StubEnv(NEUTRAL), target_pos)
    plain.reset()
    assert all(np.array_equal(q, [0.0, 1.0, 0.0, 0.0]) for q in plain.quat_traj)

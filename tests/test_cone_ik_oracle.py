"""CPU: the FP64 statement of cone-tolerant axis IK (oracle/cone_ik_oracle.py), held against itself in its two
implementations, against its two ends (alpha = 0 is the axis solve, alpha = pi the position solve), against one
position pass inside the cone, and on the four workloads of DESIGN.md 4.9, where it is compared with the deadzone form
the statement rejects."""
import math

import numpy as np
import pytest
import torch

from conftest import NEUTRAL
from mujoco_panda_pnp_b200 import synthetic
from oracle import axis_ik_oracle, c_oracle, cone_ik_oracle, mj_oracle


def _limits(chain):
    return np.array(chain.lower[:]), np.array(chain.upper[:])


def _a_cold(chain, n, seed=1234, tool=(0.0, 0.0, 1.0)):
    lo, hi = _limits(chain)
    q_star = synthetic.random_joint_configs(n, lo, hi, seed=seed, dtype=torch.float64).numpy()
    p, mat, _ = c_oracle.fk_jac(chain, q_star, nthreads=8)
    return p, mat @ axis_ik_oracle.tool_basis(tool)[0]


def _workloads(chain, n):
    """A-cold, top-down, shelf top-down and shelf horizontal (tools/cone_ik_cpu_table.py)."""
    p, ax = _a_cold(chain, n)
    box = np.array(synthetic.SHELF_BOX)
    ps = box[:, 0] + (box[:, 1] - box[:, 0]) * np.random.default_rng(0).random((n, 3))
    down, horiz = np.tile([0.0, 0.0, -1.0], (n, 1)), np.tile([1.0, 0.0, 0.0], (n, 1))
    return dict(a_cold=(p, ax), top_down=(p, down), shelf_top_down=(ps, down), shelf_horizontal=(ps, horiz))


@pytest.mark.parametrize("deg", [10.0, 30.0])
@pytest.mark.parametrize("tool", [(0.0, 0.0, 1.0), (0.3, -0.2, 0.9)])
def test_scalar_and_batched_statements_agree(oracle_model, oracle_chain, tool, deg):
    p, ax = _a_cold(oracle_chain, 24, seed=7, tool=tool)
    alpha = math.radians(deg)
    ref = cone_ik_oracle.solve_cone_batch(oracle_chain, p, ax, NEUTRAL, alpha, tool_axis=tool)
    d = mj_oracle.MjData(oracle_model)
    for k in range(len(p)):
        w = cone_ik_oracle.solve_cone(oracle_model, d, p[k], ax[k], NEUTRAL, alpha, tool_axis=tool)
        assert w["iterations"] == ref["iterations"][k] and w["converged"] == ref["converged"][k], k
        assert w["success"] == ref["success"][k]
        np.testing.assert_allclose(w["q"], ref["q"][k], atol=1e-9)
        assert abs(w["axis_error"] - ref["axis_error"][k]) < 1e-9
    assert ref["converged"].sum() >= 15


def test_zero_cone_is_the_axis_solve(oracle_chain):
    p, ax = _a_cold(oracle_chain, 512, seed=21)
    cone = cone_ik_oracle.solve_cone_batch(oracle_chain, p, ax, NEUTRAL, 0.0)
    axis = axis_ik_oracle.solve_axis_batch(oracle_chain, p, ax, NEUTRAL)
    assert np.array_equal(cone["iterations"], axis["iterations"])
    assert np.array_equal(cone["converged"], axis["converged"]) and np.array_equal(cone["success"], axis["success"])
    assert np.abs(cone["q"] - axis["q"]).max() < 1e-12
    assert np.array_equal(cone["axis_error"], axis["axis_error"])


def test_pi_cone_is_the_position_solve(oracle_chain):
    lo, hi = _limits(oracle_chain)
    q_star = synthetic.random_joint_configs(1024, lo, hi, seed=7, dtype=torch.float64).numpy()
    p = c_oracle.fk_jac(oracle_chain, q_star, nthreads=8)[0]
    ax = np.tile([0.0, 0.0, -1.0], (len(p), 1))
    cone = cone_ik_oracle.solve_cone_batch(oracle_chain, p, ax, NEUTRAL, math.pi)
    pos = c_oracle.ik_solve(oracle_chain, p, NEUTRAL, nthreads=8)
    assert np.array_equal(cone["iterations"], pos["iterations"])
    assert np.array_equal(cone["converged"], pos["converged"])
    assert np.abs(cone["q"] - pos["q"]).max() < 1e-9
    assert cone["converged"].mean() > 0.9


def test_pass_inside_the_cone_is_a_position_pass(oracle_chain):
    """One pass from q with theta <= alpha: dq = jacp^T (jacp jacp^T + damping I3)^-1 (tp - p), clipped."""
    lo, hi = _limits(oracle_chain)
    q0 = np.random.default_rng(31).uniform(lo, hi, (64, 7))
    p0, mat0, jac0 = c_oracle.fk_jac(oracle_chain, q0)
    # a target axis 0.1 rad off the tool axis, a cone of 0.2 rad, a target 5 cm away
    off = np.cross(mat0[:, :, 2], mat0[:, :, 0])
    d = np.cos(0.1) * mat0[:, :, 2] + np.sin(0.1) * off / np.linalg.norm(off, axis=1, keepdims=True)
    tp = p0 + np.array([0.03, -0.02, 0.03])
    ev = axis_ik_oracle.axis_eval_batch(oracle_chain, q0, tp, d)
    assert np.allclose(ev["axis_error"], 0.1, atol=1e-12)
    trace = []
    cone_ik_oracle.solve_cone_batch(oracle_chain, tp, d, q0, 0.2, max_iters=1, trace=trace)
    jp = jac0[:, :3]
    want = (np.swapaxes(jp, 1, 2) @ np.linalg.solve(jp @ np.swapaxes(jp, 1, 2) + 1e-2 * np.eye(3),
                                                    (tp - p0)[:, :, None]))[:, :, 0]
    np.testing.assert_allclose(trace[1], np.clip(q0 + np.clip(want, -0.1, 0.1), lo, hi), atol=1e-12)
    # outside the cone the tilt rows are live and the pass is not a position pass
    trace_out = []
    cone_ik_oracle.solve_cone_batch(oracle_chain, tp, d, q0, 0.05, max_iters=1, trace=trace_out)
    assert np.abs(trace_out[1] - trace[1]).max() > 1e-4


def test_degenerate_target_axis(oracle_chain):
    p, ax = _a_cold(oracle_chain, 8, seed=17)
    ax[[1, 4]] = 0.0
    ax[6] = [np.nan, 0.0, 1.0]
    bad = np.zeros(8, dtype=bool)
    bad[[1, 4, 6]] = True
    alpha = math.radians(20)
    out = cone_ik_oracle.solve_cone_batch(oracle_chain, p, ax, NEUTRAL, alpha, max_iters=30)
    assert not out["converged"][bad].any() and not out["success"][bad].any()
    assert (out["iterations"][bad] == 30).all() and np.isfinite(out["q"]).all()
    clean = cone_ik_oracle.solve_cone_batch(oracle_chain, p[~bad], ax[~bad], NEUTRAL, alpha, max_iters=30)
    assert np.array_equal(clean["q"], out["q"][~bad])


def _solve_deadzone(chain, tp, ta, q_init, alpha, max_iters=100, pos_thresh=1e-3, rot_thresh=1e-2, damping=1e-2,
                    step_limit=0.1, w=1.0):
    """The form the statement rejects: the tilt error clamped to w max(theta - alpha, 0), the tilt rows left in J."""
    n = len(tp)
    d = ta / np.linalg.norm(ta, axis=1, keepdims=True)
    basis = axis_ik_oracle.tool_basis((0.0, 0.0, 1.0))
    q = np.array(np.broadcast_to(q_init, (n, 7)))
    lo, hi = _limits(chain)
    conv, pe_o, th_o = np.zeros(n, bool), np.zeros(n), np.zeros(n)
    act = np.arange(n)
    for i in range(max_iters + 1):
        if len(act) == 0:
            break
        qa = q[act]
        p, mat, jac = c_oracle.fk_jac(chain, qa, nthreads=8)
        _, b1, b2, th, nv = axis_ik_oracle._axis_error(mat, basis, d[act])
        pe = np.linalg.norm(tp[act] - p, axis=1)
        g = np.maximum(th - alpha, 0.0)
        last = i == max_iters
        done = np.ones(len(act), bool) if last else (pe < pos_thresh) & (g < rot_thresh)
        pe_o[act[done]], th_o[act[done]], conv[act[done]] = pe[done], g[done], not last
        keep = ~done
        if not keep.any():
            break
        jr = jac[keep, 3:6]
        J = np.concatenate([jac[keep, :3], w * np.einsum("ni,nij->nj", b1[keep], jr)[:, None],
                            w * np.einsum("ni,nij->nj", b2[keep], jr)[:, None]], axis=1)
        e = np.concatenate([(tp[act] - p)[keep], (w * g[keep] * np.einsum("ni,ni->n", nv[keep], b1[keep]))[:, None],
                            (w * g[keep] * np.einsum("ni,ni->n", nv[keep], b2[keep]))[:, None]], axis=1)
        dq = (np.swapaxes(J, 1, 2) @ np.linalg.solve(J @ np.swapaxes(J, 1, 2) + damping * np.eye(5), e[:, :, None]))[:, :, 0]
        q[act[keep]] = np.clip(qa[keep] + np.clip(dq, -step_limit, step_limit), lo, hi)
        act = act[keep]
    return conv & (pe_o < 2 * pos_thresh) & (th_o < 2 * rot_thresh)


def test_cone_success_grows_with_the_angle_and_the_deadzone_does_not(oracle_chain):
    """4096 targets per workload from NEUTRAL (DESIGN.md 4.9): dropping the tilt rows inside the cone never loses a
    workload's success as the cone widens, and gains at least 0.05 at 30 degrees; the deadzone form loses A-cold
    successes at 20 degrees."""
    rates = {}
    for name, (p, ax) in _workloads(oracle_chain, 4096).items():
        base = axis_ik_oracle.solve_axis_batch(oracle_chain, p, ax, NEUTRAL)["success"].mean()
        r = {deg: cone_ik_oracle.solve_cone_batch(oracle_chain, p, ax, NEUTRAL, math.radians(deg))["success"].mean()
             for deg in (10, 20, 30)}
        assert all(v >= base for v in r.values()), (name, base, r)
        assert r[30] >= base + 0.05, (name, base, r)
        rates[name] = (base, r)
        if name == "a_cold":
            dead = _solve_deadzone(oracle_chain, p, ax, NEUTRAL, math.radians(20)).mean()
            assert dead < base, (base, dead)
    assert rates["shelf_horizontal"][1][20] > rates["shelf_horizontal"][0] + 0.3, rates

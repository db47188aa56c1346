"""CPU checks of the multi-start IK statement and of the default seed table."""
import numpy as np
import torch

from conftest import NEUTRAL
from mujoco_panda_pnp_b200 import engine, synthetic
from oracle import c_oracle, ik_oracle, mj_oracle


def solve_multistart(ctl, target_pos, q_init, seeds, **kw):
    """FP64 statement of the multi-start solve (pnp_ik_solve_multistart_*) over the restated controller: attempt 0 is
    ``ctl.solve`` from q_init; when it is not a success, attempts 1..K solve the same target from seeds[k - 1].  Returns
    (attempt, IKResult) of the first successful attempt in order 0..K, or of attempt 0 when none succeeds."""
    r0 = ctl.solve(target_pos, q_init, **kw)
    if r0.success:
        return 0, r0
    for k, s in enumerate(np.asarray(seeds, dtype=np.float64).reshape(-1, 7)):
        r = ctl.solve(target_pos, s, **kw)
        if r.success:
            return k + 1, r
    return 0, r0


def multistart_batched(chain, targets, q_init, seeds, **kw):
    """The batched composition a caller writes: solve, then re-solve the still-failed rows from each seed in turn."""
    r = c_oracle.ik_solve(chain, targets, q_init, nthreads=8, **kw)
    out = {k: v.copy() for k, v in r.items()}
    attempt = np.zeros(len(targets), dtype=np.int64)
    left = np.nonzero(~r["success"])[0]
    for k, s in enumerate(seeds):
        if not len(left):
            break
        rk = c_oracle.ik_solve(chain, targets[left], s, nthreads=8, **kw)
        ok = rk["success"]
        for key in out:
            out[key][left[ok]] = rk[key][ok]
        attempt[left[ok]] = k + 1
        left = left[~ok]
    return attempt, out


def cfg5_targets(chain, lower, upper, n, seed=1234):
    qstar = synthetic.random_joint_configs(n, lower, upper, seed=seed, dtype=torch.float64).numpy()
    return c_oracle.fk_jac(chain, qstar, nthreads=8)[0]


def test_restart_seeds_are_deterministic_and_inside_the_limits(oracle_model):
    lo, hi = oracle_model.jnt_range[:7, 0], oracle_model.jnt_range[:7, 1]
    a = engine.ik_restart_seeds(8, device="cpu", dtype=torch.float64)
    b = engine.ik_restart_seeds(8, lo, hi, seed=0, device="cpu", dtype=torch.float64)
    assert a.shape == (8, 7) and torch.equal(a, b)
    assert not torch.equal(a, engine.ik_restart_seeds(8, seed=1, device="cpu", dtype=torch.float64))
    assert ((a >= torch.as_tensor(lo)) & (a <= torch.as_tensor(hi))).all()
    assert torch.equal(engine.ik_restart_seeds(8, device="cpu"), a.float())


def test_scalar_statement_matches_the_batched_composition(oracle_model, oracle_chain):
    """~300 targets: reachable cfg5 targets that attempt 0 solves, ones it fails on, and unreachable ones."""
    lo, hi = oracle_model.jnt_range[:7, 0], oracle_model.jnt_range[:7, 1]
    pool = cfg5_targets(oracle_chain, lo, hi, 1 << 14)
    r0 = c_oracle.ik_solve(oracle_chain, pool, NEUTRAL, nthreads=8)
    hard = pool[~r0["success"]][:40]
    assert len(hard) >= 20
    easy = pool[r0["success"]][:240]
    far = np.array([[2.5, 0.0, 0.5], [0.0, 0.0, 3.0], [-2.0, 1.5, 0.2], [1.0, -2.2, 1.0], [0.0, 0.0, -2.0],
                    [3.0, 3.0, 3.0], [0.0, 2.6, 0.8], [-2.4, -0.5, 1.4]])
    targets = np.concatenate([easy, hard, far])
    seeds = engine.ik_restart_seeds(8, lo, hi, device="cpu", dtype=torch.float64).numpy()
    attempt, ref = multistart_batched(oracle_chain, targets, NEUTRAL, seeds)
    assert (attempt[len(easy):len(easy) + len(hard)] > 0).any()
    assert (attempt[-len(far):] == 0).all() and not ref["success"][-len(far):].any()
    ctl = ik_oracle.JacobianIKController(oracle_model, mj_oracle.MjData(oracle_model))
    for i, t in enumerate(targets):
        k, r = solve_multistart(ctl, t, NEUTRAL, seeds)
        assert k == attempt[i], i
        assert r.iterations == ref["iterations"][i] and r.success == ref["success"][i], i
        if r.converged:  # (a 100-pass walk that never converges amplifies the two statements' rounding differences)
            np.testing.assert_allclose(r.q, ref["q"][i], atol=1e-9)


def test_default_seed_table_rescues_the_cfg5_failures(oracle_model, oracle_chain):
    """2^18 cfg5 targets (q* ~ U(joint range), seed 1234) cold from NEUTRAL: engine.ik_restart_seeds(8) must rescue
    at least 98 % of the queries attempt 0 fails on."""
    lo, hi = oracle_model.jnt_range[:7, 0], oracle_model.jnt_range[:7, 1]
    targets = cfg5_targets(oracle_chain, lo, hi, 1 << 18)
    seeds = engine.ik_restart_seeds(8, device="cpu", dtype=torch.float64).numpy()
    attempt, out = multistart_batched(oracle_chain, targets, NEUTRAL, seeds)
    failed0 = int((attempt > 0).sum() + (~out["success"]).sum())
    rescued = int((attempt > 0).sum())
    assert failed0 > 300  # ~0.2 % of the batch
    assert rescued >= 0.98 * failed0, (rescued, failed0)

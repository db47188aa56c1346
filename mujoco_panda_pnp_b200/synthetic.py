"""Synthetic workloads of SURVEY.md section 8(d) (cfg2 .. cfg5), generated with torch so the same
code runs on the CPU (tests, golden fixtures) and on the GPU (bench, per-rank seeds).

Nothing here is on the product's compute path: it only manufactures inputs shaped like the
reference's own data.  Distributions come from the reference's VecNormalize statistics
(scripts/checkpoints/tqc_dense_vecnormalize_200000_steps.pkl, extracted into
tests/golden/vecnormalize_stats.json) and scene constants of assets/shelf_pnp.xml:56-77.
"""

from __future__ import annotations

from typing import Dict, Optional

import torch

NEUTRAL_Q = (0.00, 0.41, 0.00, -1.85, 0.00, 2.26, 0.79)  # panda_env.py:64-66

# observation[0:3] (ee_pos), achieved_goal running mean / var from the reference's pickle
EE_POS_MEAN = (1.112, -0.017, 0.499)
EE_POS_VAR = (0.051, 0.100, 0.057)
AG_MEAN = (1.411, 0.457, 0.081)
AG_VAR = (0.028, 0.670, 0.040)
AG_Z_MIN = 0.0199
TARGET_SITES = ((1.0, -0.1, 0.3), (1.0, 0.0, 0.3), (1.0, 0.1, 0.3))  # shelf_pnp.xml:56-58
SHELF_BOX = ((1.0, 1.45), (-0.25, 0.25), (0.3, 1.1))  # cfg4 goal region


def _gen(seed: int, device) -> torch.Generator:
    g = torch.Generator(device=device)
    g.manual_seed(int(seed))
    return g


def random_joint_configs(n: int, lower, upper, seed: int = 0, device="cpu", dtype=torch.float32) -> torch.Tensor:
    """q* ~ U(lower, upper), shape (n, 7) (cfg2 / cfg5: targets are FK(q*), hence reachable)."""
    g = _gen(seed, device)
    lo = torch.as_tensor(lower, dtype=torch.float64, device=device)
    hi = torch.as_tensor(upper, dtype=torch.float64, device=device)
    u = torch.rand((n, 7), generator=g, device=device, dtype=torch.float64)
    return (lo + (hi - lo) * u).to(dtype)


def reward_rows(
    n: int,
    seed: int = 0,
    device="cpu",
    dtype=torch.float32,
    n_adversarial: Optional[int] = None,
    n_tasks: int = 3,
) -> Dict[str, torch.Tensor]:
    """cfg3: HER-relabelled transition rows with every reward branch populated.

    Returns achieved_goal[n,3], desired_goal[n,3], ee_pos[n,3], ee_quat[n,4] (wxyz),
    fingers_width[n], task_index[n] (int32).  Stratification (by row index modulo, so it is
    independent of n): 25 % of rows put the cube in the gripper (ag = ee_pos + N(0, 0.02^2)),
    5 % are placed (dg = ag + N(0, 0.02^2)), 20 % keep one of the three real target sites as
    goal, the rest get a HER "future" goal = another row's achieved_goal.  The last
    ``n_adversarial`` rows (default min(2^16, n // 16)) sit within +-1e-6 of the 0.05
    thresholds on d_place / d_reach: the rows north_star exempts from bit-exactness.
    """
    g = _gen(seed, device)
    f64 = torch.float64
    kw = dict(generator=g, device=device, dtype=f64)
    idx = torch.arange(n, device=device)

    ee = torch.tensor(EE_POS_MEAN, dtype=f64, device=device) + torch.randn((n, 3), **kw) * torch.tensor(
        EE_POS_VAR, dtype=f64, device=device
    ).sqrt()
    ag = torch.tensor(AG_MEAN, dtype=f64, device=device) + torch.randn((n, 3), **kw) * torch.tensor(
        AG_VAR, dtype=f64, device=device
    ).sqrt()
    ag[:, 2].clamp_(min=AG_Z_MIN)
    width = torch.rand((n,), **kw) * 0.08
    quat = torch.randn((n, 4), **kw)
    quat = quat / quat.norm(dim=1, keepdim=True)
    task = torch.randint(0, n_tasks, (n,), generator=g, device=device, dtype=torch.int32)

    # gripped / lifted reachable: cube follows the gripper; half of those with closed fingers
    in_hand = (idx % 4) == 1
    noise = torch.randn((n, 3), **kw) * 0.02
    ag = torch.where(in_hand[:, None], ee + noise, ag)
    closed = in_hand & ((idx % 8) == 1)
    width = torch.where(closed, width * 0.5, width)
    # aligned gripper for a share of the in-hand rows (exercise the alignment bonus)
    aligned = in_hand & ((idx % 16) == 5)
    horiz = torch.tensor([0.7071067811865476, -0.7071067811865475, 0.0, 0.0], dtype=f64, device=device)
    quat = torch.where(aligned[:, None], horiz.expand(n, 4) + torch.randn((n, 4), **kw) * 0.02, quat)
    quat = quat / quat.norm(dim=1, keepdim=True)

    # goals: 20 % real sites, 80 % HER future relabel, 5 % placed
    sites = torch.tensor(TARGET_SITES, dtype=f64, device=device)
    site_goal = sites[torch.randint(0, 3, (n,), generator=g, device=device)]
    future = ag[torch.randint(0, max(n, 1), (n,), generator=g, device=device)]
    dg = torch.where(((idx % 5) == 0)[:, None], site_goal, future)
    placed = (idx % 20) == 7
    dg = torch.where(placed[:, None], ag + torch.randn((n, 3), **kw) * 0.02, dg)

    # adversarial tail: distances within 1e-6 of the thresholds
    if n_adversarial is None:
        n_adversarial = min(1 << 16, n // 16)
    if n_adversarial > 0:
        k = n_adversarial
        d = torch.randn((k, 3), **kw)
        d = d / d.norm(dim=1, keepdim=True)
        eps = (torch.rand((k, 1), **kw) * 2 - 1) * 1e-6
        tail = slice(n - k, n)
        half = k // 2
        dg[tail] = ag[tail] + d * (0.05 + eps)
        # second half: d_reach on the threshold instead (and fingers closed so `gripped` flips)
        ee[n - half :] = ag[n - half :] + d[k - half :] * (0.05 + eps[k - half :])
        width[n - half :] = 0.03

    out = dict(
        achieved_goal=ag.to(dtype),
        desired_goal=dg.to(dtype),
        ee_pos=ee.to(dtype),
        ee_quat=quat.to(dtype),
        fingers_width=width.to(dtype),
        task_index=task,
    )
    return {k: v.contiguous() for k, v in out.items()}


def waypoint_envs(n: int, seed: int = 0, device="cpu", dtype=torch.float32) -> Dict[str, torch.Tensor]:
    """cfg4: per-env start joints (neutral + U(-0.05, 0.05)^7) and goal in the shelf box."""
    g = _gen(seed, device)
    f64 = torch.float64
    q0 = torch.tensor(NEUTRAL_Q, dtype=f64, device=device) + (
        torch.rand((n, 7), generator=g, device=device, dtype=f64) * 0.1 - 0.05
    )
    lo = torch.tensor([b[0] for b in SHELF_BOX], dtype=f64, device=device)
    hi = torch.tensor([b[1] for b in SHELF_BOX], dtype=f64, device=device)
    goal = lo + (hi - lo) * torch.rand((n, 3), generator=g, device=device, dtype=f64)
    return dict(q_start=q0.to(dtype).contiguous(), goal=goal.to(dtype).contiguous())


def reachable_move_envs(n: int, lower, upper, seed: int = 0, device="cpu", dtype=torch.float32, spread: float = 0.6):
    """Planner workload with goals that are reachable by construction: start = neutral +- 0.05 rad,
    goal = FK(q*) with q* = neutral +- ``spread`` rad clipped to the limits (the caller evaluates FK).
    The reference's MoveIKSkill loop never terminates for unreachable goals, so the headline planner
    numbers use this generator; the shelf box of ``waypoint_envs`` contains a few unreachable goals."""
    g = _gen(seed, device)
    f64 = torch.float64
    neutral = torch.tensor(NEUTRAL_Q, dtype=f64, device=device)
    q0 = neutral + (torch.rand((n, 7), generator=g, device=device, dtype=f64) * 0.1 - 0.05)
    qs = neutral + (torch.rand((n, 7), generator=g, device=device, dtype=f64) * 2 - 1) * spread
    lo = torch.as_tensor(lower, dtype=f64, device=device)
    hi = torch.as_tensor(upper, dtype=f64, device=device)
    return dict(q_start=q0.to(dtype).contiguous(), q_goal=torch.minimum(torch.maximum(qs, lo), hi).to(dtype).contiguous())


def reachable_pose_move_envs(n: int, lower, upper, seed: int = 0, device="cpu", dtype=torch.float32, spread: float = 0.6):
    """Pose-planner workload, reachable by construction: start = neutral +- 0.05 rad, goal pose = (FK(q*), quat(q*))
    with q* = neutral +- ``spread`` rad clipped to the limits.  The caller evaluates FK of q_goal for the goal position
    and orientation.  Same draws as reachable_move_envs, so the position planner can run the same starts and goal
    positions."""
    return reachable_move_envs(n, lower, upper, seed=seed, device=device, dtype=dtype, spread=spread)


def her_future_indices(n: int, episode_len: int = 300, seed: int = 0, device="cpu", keep_fraction: float = 0.2,
                       strategy: str = "future") -> torch.Tensor:
    """int32[n] `future_idx` of a HER relabel over a replay buffer that stores its episodes as runs of ``episode_len``
    consecutive transitions (300 = the reference's max_episode_steps, panda_mujoco_gym/__init__.py:15).

    ``future``  (SB3 GoalSelectionStrategy.FUTURE, the default of HerReplayBuffer): the goal of transition t of an episode
                is the achieved goal of a transition drawn uniformly from [t, T-1] of the SAME episode;
    ``uniform`` any transition of the buffer (no locality at all: the worst case for the gather).
    A fraction ``keep_fraction`` of the rows keeps the stored goal (index -1; n_sampled_goal = 4 -> 1 in 5)."""
    g = _gen(seed, device)
    idx = torch.arange(n, device=device, dtype=torch.int64)
    if strategy == "future":
        t = idx % episode_len
        last = torch.clamp(idx - t + (episode_len - 1), max=n - 1)            # last transition of the episode
        span = (last - idx + 1).to(torch.float64)
        fut = idx + torch.clamp((torch.rand(n, generator=g, device=device, dtype=torch.float64) * span).long(), max=episode_len - 1)
        fut = torch.minimum(fut, last)
    elif strategy == "uniform":
        fut = torch.randint(0, max(n, 1), (n,), generator=g, device=device, dtype=torch.int64)
    else:
        raise ValueError("strategy must be 'future' or 'uniform'")
    keep = torch.rand(n, generator=g, device=device) < keep_fraction
    return torch.where(keep, torch.full_like(fut, -1), fut).to(torch.int32)

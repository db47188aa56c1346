"""GPU: the persistent-warp IK-family kernels give every row the same result whatever the launch geometry.

ik_solve (FP64, FP32 generic), ik_waypoints and move_ik_plan switch from the small-batch grid (one working warp per
block, up to sm_count * IK_BLOCK rows) to the persistent grid (occupancy-capped, warps reserving ticket chunks) one row
later, and a batch whose size is no multiple of the chunk ends on a ragged chunk.  Witness rows scattered into such
batches must be bit-identical to a batch of just those rows, every row of sentinel-filled outputs must be written, and
the counters must add up to the outputs."""
import ctypes

import numpy as np
import pytest
import torch

from conftest import NEUTRAL
from mujoco_panda_pnp_b200 import KinematicTree, _lib, engine

pytestmark = pytest.mark.gpu

IK_BLOCK = 128  # pnp_kernels.cuh: up to sm_count * IK_BLOCK rows take the small-batch grid
N_POOL, N_WIT = 4096, 64


@pytest.fixture(scope="module")
def sm(cuda_lib):
    engine.set_tree(KinematicTree.from_mjcf())
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def _sizes(sm):
    # the last switch to the small grid, the first persistent batch, and an odd size (ragged last ticket chunk)
    return (sm * IK_BLOCK, sm * IK_BLOCK + 1, 3 * sm * IK_BLOCK + 37)


def _pool(dtype, seed):
    """q [N_POOL,7] around NEUTRAL and targets [N_POOL,3] in front of the robot (some out of reach) on the GPU."""
    rng = np.random.default_rng(seed)
    q = NEUTRAL + rng.uniform(-0.4, 0.4, (N_POOL, 7))
    tgt = np.stack([rng.uniform(0.25, 0.75, N_POOL), rng.uniform(-0.4, 0.4, N_POOL), rng.uniform(0.0, 0.6, N_POOL)], 1)
    dev = torch.device("cuda")
    return torch.as_tensor(q, dtype=dtype, device=dev), torch.as_tensor(tgt, dtype=dtype, device=dev), rng


def _batch(rng, n, pool, wit):
    """rows of pool drawn at random, the witnesses at N_WIT scattered slots"""
    idx = rng.integers(0, N_POOL, n)
    slots = rng.choice(n, N_WIT, replace=False)
    idx[slots] = wit
    it = torch.as_tensor(idx, device="cuda")
    return [a[it].contiguous() for a in pool], torch.as_tensor(slots, device="cuda")


def _bits(t):
    return t.contiguous().view(torch.uint8).cpu()


def _sentinel(shape, dtype):
    fill = -1 if dtype == torch.int32 else (0xFF if dtype == torch.uint8 else float("nan"))
    return torch.full(shape, fill, dtype=dtype, device="cuda")


def _written(t):
    return bool(torch.isfinite(t).all()) if t.is_floating_point() else bool((t != (0xFF if t.dtype == torch.uint8 else -1)).all())


def _untouched(t):
    return bool(torch.isnan(t).all()) if t.is_floating_point() else bool((t == -1).all())


def _stream():
    return torch.cuda.current_stream().cuda_stream


# ---- ik_solve ---------------------------------------------------------------------------------------------------------
def _ik(dtype, kin, tgt, q0):
    n = tgt.shape[0]
    outs = (_sentinel((n, 7), dtype), _sentinel((n, 3), dtype), _sentinel((n,), dtype), _sentinel((n,), torch.int32),
            _sentinel((n,), torch.uint8))
    counters = torch.zeros(4, dtype=torch.int64, device="cuda")
    lib = _lib.load()
    fn = lib.pnp_ik_solve_f32 if dtype == torch.float32 else lib.pnp_ik_solve_f64
    _lib.check(fn(tgt.data_ptr(), q0.data_ptr(), 7, n, ctypes.byref(engine.ik_params(kinematics=kin)),
                  *(t.data_ptr() for t in outs), counters.data_ptr(), _stream()), "pnp_ik_solve")
    torch.cuda.synchronize()
    return outs, counters


@pytest.mark.parametrize("dtype,kin", [(torch.float64, "auto"), (torch.float64, "generic"), (torch.float32, "generic")])
def test_ik_solve_rows_do_not_depend_on_launch_geometry(sm, dtype, kin):
    q, tgt, rng = _pool(dtype, seed=11)
    wit = rng.choice(N_POOL, N_WIT, replace=False)
    ref, _ = _ik(dtype, kin, tgt[wit].contiguous(), q[wit].contiguous())
    for n in _sizes(sm):
        (qb, tb), slots = _batch(rng, n, (q, tgt), wit)
        outs, counters = _ik(dtype, kin, tb, qb)
        assert all(_written(t) for t in outs), n
        iters, flags = outs[3], outs[4]
        conv, succ = (flags & 1) != 0, (flags & 2) != 0
        assert counters.tolist() == [n, int(conv.sum()), int(succ.sum()), int(iters.long().sum())], n
        for got, want in zip(outs, ref):
            assert torch.equal(_bits(got[slots]), _bits(want)), n


# ---- ik_waypoints -----------------------------------------------------------------------------------------------------
def _waypoints(kin, q0, goal):
    n = q0.shape[0]
    outs = (_sentinel((n, 7), torch.float32), _sentinel((n, 3), torch.float32), _sentinel((n,), torch.int32),
            _sentinel((n,), torch.int32))
    counters = torch.zeros(4, dtype=torch.int64, device="cuda")
    _lib.check(_lib.load().pnp_ik_waypoints_f32(q0.data_ptr(), goal.data_ptr(), n, 20, 0.01,
                                                ctypes.byref(engine.ik_params(kinematics=kin)),
                                                *(t.data_ptr() for t in outs), counters.data_ptr(), _stream()),
               "pnp_ik_waypoints")
    torch.cuda.synchronize()
    return outs, counters


@pytest.mark.parametrize("kin", ["spec_lane", "spec_pair", "generic"])
def test_ik_waypoints_rows_do_not_depend_on_launch_geometry(sm, kin):
    q, tgt, rng = _pool(torch.float32, seed=12)
    wit = rng.choice(N_POOL, N_WIT, replace=False)
    ref, _ = _waypoints(kin, q[wit].contiguous(), tgt[wit].contiguous())
    for n in _sizes(sm):
        (qb, tb), slots = _batch(rng, n, (q, tgt), wit)
        outs, counters = _waypoints(kin, qb, tb)
        assert all(_written(t) for t in outs), n
        assert bool((outs[2] >= 0).all()) and bool((outs[3] >= 0).all())
        # one counter per solve: success == converged, and the iterations add up to iters_total
        assert counters[1] == counters[2] and int(counters[3]) == int(outs[3].long().sum()), n
        for got, want in zip(outs, ref):
            assert torch.equal(_bits(got[slots]), _bits(want)), n


# ---- move_ik_plan -----------------------------------------------------------------------------------------------------
def _plan(dtype, kin, traj_cap, q0, tgt, order=None):
    n = q0.shape[0]
    outs = (_sentinel((n, traj_cap, 3), dtype), _sentinel((n,), torch.int32), _sentinel((n, 7), dtype),
            _sentinel((n,), torch.int32), _sentinel((n,), torch.int32))
    counters = torch.zeros(4, dtype=torch.int64, device="cuda")
    mp = engine.PnpMoveParams(0.01, 0.01, 40, 0, traj_cap, 0)
    lib = _lib.load()
    fn = lib.pnp_move_ik_plan_ordered_f32 if dtype == torch.float32 else lib.pnp_move_ik_plan_ordered_f64
    _lib.check(fn(q0.data_ptr(), tgt.data_ptr(), None if order is None else order.data_ptr(), n, ctypes.byref(mp),
                  ctypes.byref(engine.ik_params(kinematics=kin)), *(t.data_ptr() for t in outs), counters.data_ptr(),
                  _stream()), "pnp_move_ik_plan")
    torch.cuda.synchronize()
    return outs, counters


def _check_plan(outs, counters, rows):
    """rows [bool n]: the envs that must have been planned (the others keep their sentinels)"""
    traj, tlen, qf, solves, status = outs
    for t in (tlen, qf, solves, status):
        assert _written(t[rows]) and _untouched(t[~rows])
    n_pts = torch.clamp(tlen[rows], max=traj.shape[1]).long()
    filled = torch.arange(traj.shape[1], device="cuda")[None, :] < n_pts[:, None]
    assert bool(torch.isfinite(traj[rows]).all(-1)[filled].all())
    assert int(counters[0]) == int(solves[rows].long().sum()) and counters[1] == counters[2]


# (traj_cap % 4 == 0 with an aligned trajectory: the FP32 one-env-per-lane planner stages its points in shared memory)
PLANS = [(torch.float32, "spec_lane", 64), (torch.float32, "spec_lane", 62), (torch.float32, "spec_pair", 64),
         (torch.float32, "generic", 64), (torch.float64, "auto", 64)]


@pytest.mark.parametrize("dtype,kin,traj_cap", PLANS)
def test_move_ik_plan_rows_do_not_depend_on_launch_geometry(sm, dtype, kin, traj_cap):
    q, tgt, rng = _pool(dtype, seed=13)
    wit = rng.choice(N_POOL, N_WIT, replace=False)
    ref, _ = _plan(dtype, kin, traj_cap, q[wit].contiguous(), tgt[wit].contiguous())
    for n in _sizes(sm):
        (qb, tb), slots = _batch(rng, n, (q, tgt), wit)
        outs, counters = _plan(dtype, kin, traj_cap, qb, tb)
        _check_plan(outs, counters, torch.ones(n, dtype=torch.bool, device="cuda"))
        for got, want in zip(outs, ref):
            assert torch.equal(_bits(got[slots]), _bits(want)), n
        # a caller-made order whose out-of-range entries straddle ticket-chunk boundaries: those envs are skipped, the
        # rest are planned exactly as without an order
        perm = torch.as_tensor(rng.permutation(n), dtype=torch.int32, device="cuda")
        keep = torch.ones(n, dtype=torch.bool, device="cuda")
        keep[slots] = False  # witnesses must stay planned
        at = torch.arange(n, device="cuda")
        hole = (((at % 128) >= 120) | ((at % 128) < 8)) & keep[perm.long()]
        dropped = torch.zeros(n, dtype=torch.bool, device="cuda")
        dropped[perm[hole].long()] = True
        order = torch.where(hole, torch.full_like(perm, n + 5), perm)
        outs2, counters2 = _plan(dtype, kin, traj_cap, qb, tb, order)
        _check_plan(outs2, counters2, ~dropped)
        for got, full in zip(outs2, outs):
            assert torch.equal(_bits(got[~dropped]), _bits(full[~dropped])), n

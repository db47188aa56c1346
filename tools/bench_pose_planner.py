"""Time the pose-mode move planner (pnp_move_ik_plan_pose_f32) next to the position planner and next to the torch
composition a caller writes without it.

    python tools/bench_pose_planner.py [--sizes 14 16 18 20] [--composition-sizes 14 16] [--warmup 2] [--iters 5]

Workload: synthetic.reachable_pose_move_envs(seed=0) - start NEUTRAL +- 0.05 rad, goal pose (FK(q*), quat(q*)) with
q* = NEUTRAL +- 0.6 rad clipped to the limits, so every goal is reachable.  FP32, default planner parameters (pos_thresh
0.01 m, rot_thresh 0.05 rad, step_size 0.01 m, rot_step 0.05 rad, 200 points, traj_cap 201), default IK (max_iters 100,
pos_thresh 1e-3, ik_rot_thresh 1e-2).  Columns per size:
  pose planner    one call into preallocated outputs (q_traj included), median of --iters calls, each alone between
                  two CUDA events; plans/s, mean waypoints (traj_len - 1), mean solves, DLS passes/s (the iterations of
                  every waypoint solve, from the counters; the INIT pass of each env is not counted)
  position        engine.move_ik_plan on the same starts and goal positions (its default longest-plan-first path),
                  outputs reused between calls
  composition     the same statement in torch: one engine.ik_pose_solve per round over the envs still planning, and a
                  host synchronisation per round to drop the finished ones (--composition-sizes only)
The calls alternate within each repetition.  Prints one JSON line with the GPU's name, power limit and clock.
"""

from __future__ import annotations

import argparse
import ctypes
import json
import math
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import torch  # noqa: E402

from mujoco_panda_pnp_b200 import KinematicTree, _lib, engine, synthetic  # noqa: E402

PLAN = dict(pos_thresh=0.01, rot_thresh=0.05, step_size=0.01, rot_step=0.05, ik_rot_thresh=1e-2, rot_weight=1.0,
            max_traj_points=200)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else None
    except (OSError, subprocess.SubprocessError):
        return None


def event_ms(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def mulquat(a, b):
    return torch.stack([a[:, 0] * b[:, 0] - a[:, 1] * b[:, 1] - a[:, 2] * b[:, 2] - a[:, 3] * b[:, 3],
                        a[:, 0] * b[:, 1] + a[:, 1] * b[:, 0] + a[:, 2] * b[:, 3] - a[:, 3] * b[:, 2],
                        a[:, 0] * b[:, 2] - a[:, 1] * b[:, 3] + a[:, 2] * b[:, 0] + a[:, 3] * b[:, 1],
                        a[:, 0] * b[:, 3] + a[:, 1] * b[:, 2] - a[:, 2] * b[:, 1] + a[:, 3] * b[:, 0]], dim=1)


def quat2vel(q):
    s = q[:, 1:].norm(dim=1)
    a = 2 * torch.atan2(s, q[:, 0])
    a = torch.where(a > math.pi, a - 2 * math.pi, a)
    return q[:, 1:] * torch.where(s > 0, a / torch.where(s > 0, s, torch.ones_like(s)), torch.zeros_like(s))[:, None]


def composition(qs, gp, gq, params, cap):
    """The planner's statement (oracle/move_pose_oracle.py) with one batched pose solve per round."""
    n, dev = qs.shape[0], qs.device
    gq = gq / gq.norm(dim=1, keepdim=True)
    p, r, _ = engine.fk_jac(qs, want_jac=False)
    q = qs.clone()
    pos_traj = torch.zeros((n, cap, 3), device=dev)
    quat_traj = torch.zeros((n, cap, 4), device=dev)
    q_traj = torch.zeros((n, cap, 7), device=dev)
    pos_traj[:, 0], quat_traj[:, 0], q_traj[:, 0] = p, r, q
    points = torch.zeros(n, dtype=torch.long, device=dev)
    attempt = torch.zeros(n, dtype=torch.long, device=dev)
    status = torch.zeros(n, dtype=torch.int32, device=dev)
    solves = torch.zeros(n, dtype=torch.int32, device=dev)
    scale = torch.tensor([1.0, 0.5, 0.05], device=dev)
    live = torch.arange(n, device=dev)
    while True:
        d = gp[live] - p[live]
        dist = d.norm(dim=1)
        w = quat2vel(mulquat(gq[live], r[live] * torch.tensor([1.0, -1.0, -1.0, -1.0], device=dev)))
        th = w.norm(dim=1)
        first = attempt[live] == 0
        done = first & (dist <= PLAN["pos_thresh"]) & (th <= PLAN["rot_thresh"])
        capped = first & ~done & (points[live] >= PLAN["max_traj_points"])
        status[live[capped]] = 2
        keep = ~(done | capped)
        live, d, dist, w, th = live[keep], d[keep], dist[keep], w[keep], th[keep]
        if live.numel() == 0:  # host synchronisation: one per round
            break
        one = torch.ones_like(dist)
        f = torch.minimum(torch.minimum(one, torch.where(dist > 0, PLAN["step_size"] / dist, one)),
                          torch.where(th > 0, PLAN["rot_step"] / th, one))
        g = f * scale[attempt[live]]
        h = 0.5 * g * th
        k = torch.where(th > 0, torch.sin(h) / torch.where(th > 0, th, one), torch.zeros_like(th))
        aim_q = mulquat(torch.cat([torch.cos(h)[:, None], k[:, None] * w], dim=1), r[live])
        full = (g == 1.0)[:, None]
        aim_p = torch.where(full, gp[live], p[live] + g[:, None] * d)
        aim_q = torch.where(full, gq[live], aim_q)
        res = engine.ik_pose_solve(aim_p.contiguous(), aim_q.contiguous(), q[live].contiguous(), params,
                                   rot_thresh=PLAN["ik_rot_thresh"], rot_weight=PLAN["rot_weight"])
        solves[live] += 1
        ok = res["success"]
        acc = live[ok]
        p[acc], r[acc], q[acc] = res["final_pos"][ok], res["final_quat"][ok], res["q"][ok]
        points[acc] += 1
        slot = points[acc].clamp(max=cap - 1)
        pos_traj[acc, slot], quat_traj[acc, slot], q_traj[acc, slot] = p[acc], r[acc], q[acc]
        attempt[acc] = 0
        rej = live[~ok]
        attempt[rej] += 1
        broke = rej[attempt[rej] == 3]
        status[broke] = 1
        live = live[attempt[live] < 3]
    return dict(pos_traj=pos_traj, quat_traj=quat_traj, q_traj=q_traj, traj_len=(points + 1).int(), q_final=q,
                n_solves=solves, status=status)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[14, 16, 18, 20], help="log2 of the batch sizes")
    ap.add_argument("--composition-sizes", type=int, nargs="*", default=[14, 16])
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--iters", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_pose_planner needs a CUDA device")
    dev = torch.device("cuda", torch.cuda.current_device())
    lib = _lib.load()
    tree = KinematicTree.from_mjcf()
    engine.set_tree(tree)
    params = engine.ik_params()
    cap = PLAN["max_traj_points"] + 1
    mp = _lib.PnpMovePoseParams(PLAN["pos_thresh"], PLAN["rot_thresh"], PLAN["step_size"], PLAN["rot_step"],
                                PLAN["ik_rot_thresh"], PLAN["rot_weight"], PLAN["max_traj_points"], cap)
    result = dict(tool="bench_pose_planner", gpu=gpu_info(), torch=torch.__version__, warmup=args.warmup,
                  iters=args.iters, plan=PLAN, runs={})
    for lg in args.sizes:
        n = 1 << lg
        e = synthetic.reachable_pose_move_envs(n, tree.lower, tree.upper, seed=0, device=dev)
        gp, gq, _ = engine.fk_jac(e["q_goal"], want_jac=False)
        qs = e["q_start"]
        o = dict(pos=torch.empty((n, cap, 3), device=dev), quat=torch.empty((n, cap, 4), device=dev),
                 q=torch.empty((n, cap, 7), device=dev), tlen=torch.empty(n, dtype=torch.int32, device=dev),
                 qf=torch.empty((n, 7), device=dev), solves=torch.empty(n, dtype=torch.int32, device=dev),
                 status=torch.empty(n, dtype=torch.int32, device=dev))
        stream = lambda: torch.cuda.current_stream().cuda_stream  # noqa: E731

        def pose(counters=None):
            _lib.check(lib.pnp_move_ik_plan_pose_f32(
                qs.data_ptr(), gp.data_ptr(), gq.data_ptr(), n, ctypes.byref(mp), ctypes.byref(params),
                *(o[k].data_ptr() for k in ("pos", "quat", "q", "tlen", "qf", "solves", "status")),
                None if counters is None else counters.data_ptr(), stream()), "pose planner")

        position_out = engine.move_ik_plan(qs, gp, params)

        def position():
            engine.move_ik_plan(qs, gp, params, out=position_out)

        def comp():
            return composition(qs, gp, gq, params, cap)

        variants = [pose, position] + ([comp] if lg in args.composition_sizes else [])
        for _ in range(args.warmup):
            for f in variants:
                f()
        torch.cuda.synchronize()
        times = {f.__name__: [] for f in variants}
        for _ in range(args.iters):
            for f in variants:
                times[f.__name__].append(event_ms(f))
        med = {k: statistics.median(v) for k, v in times.items()}
        cnt = torch.zeros(4, dtype=torch.int64, device=dev)
        pose(cnt)
        torch.cuda.synchronize()
        c = cnt.cpu().tolist()
        st = o["status"]
        run = dict(
            n=n,
            pose_ms=med["pose"], pose_ms_min=min(times["pose"]), pose_plans_per_s=n / (med["pose"] * 1e-3),
            pose_ok=float((st == 0).float().mean()), pose_broke=float((st & 1 != 0).float().mean()),
            pose_capped=float((st & 2 != 0).float().mean()),
            pose_mean_waypoints=float((o["tlen"] - 1).float().mean()), pose_mean_solves=float(o["solves"].float().mean()),
            pose_solves=c[0], pose_dls_passes=c[3], pose_dls_passes_per_s=c[3] / (med["pose"] * 1e-3),
            pose_passes_per_solve=c[3] / max(c[0], 1),
            position_ms=med["position"], position_ms_min=min(times["position"]),
            position_plans_per_s=n / (med["position"] * 1e-3),
            position_ok=float((position_out["status"] == 0).float().mean()),
            position_mean_points=float(position_out["traj_len"].float().mean()),
            position_mean_solves=float(position_out["n_solves"].float().mean()),
        )
        if "comp" in med:
            r = comp()
            torch.cuda.synchronize()
            run.update(composition_ms=med["comp"], composition_ms_min=min(times["comp"]),
                       composition_plans_per_s=n / (med["comp"] * 1e-3), composition_over_pose=med["comp"] / med["pose"],
                       composition_ok=float((r["status"] == 0).float().mean()),
                       composition_same_len=float((r["traj_len"] == o["tlen"]).float().mean()),
                       composition_mean_solves=float(r["n_solves"].float().mean()))
        result["runs"][str(lg)] = run
        print(json.dumps(dict(progress=lg, **run)), file=sys.stderr)
        del o, qs, gp, gq, position_out
        torch.cuda.empty_cache()
    print(json.dumps(result))


if __name__ == "__main__":
    main()

"""Time the axis-mode move planner (pnp_move_ik_plan_axis_f32) next to the pose-mode planner on the same moves.

    python tools/bench_axis_planner.py [--sizes 14 16 18 20] [--w2-size 16] [--warmup 2] [--iters 10] [--out FILE]

FP32, default planner parameters (pos_thresh 0.01 m, rot_thresh 0.05 rad, step_size 0.01 m, rot_step 0.05 rad,
200 points, traj_cap 201, q_traj written), default IK (max_iters 100, pos_thresh 1e-3, ik_rot_thresh 1e-2), tool axis
(0, 0, 1).  Workloads:
  W1  synthetic.reachable_pose_move_envs(seed=0): start NEUTRAL +- 0.05 rad, q* = NEUTRAL +- 0.6 rad clipped to the
      limits.  Axis planner: goal (FK(q*), R(q*) t); pose planner: goal (FK(q*), quat(q*)), so both goals are
      reachable by construction and the axis goal leaves the roll free.
  W2  pick-and-place: the same goal positions FK(q*) with a top-down goal axis (0, 0, -1); the pose planner gets the
      NEUTRAL site quaternion as the roll a caller would have to invent.
Each call writes into preallocated outputs and is timed alone between two CUDA events; the two planners alternate within
each repetition and the median of --iters calls is reported.  Per planner: time, plans/s, solver passes/s (every
waypoint solve's DLS passes, from the counters; the INIT pass of each env is not counted), mean points, solves and
passes per solve, and the OK / BROKE / CAPPED shares.  The JSON line carries the GPU's name, power limit and max SM
clock (read in the same process), and the ptxas resource lines of the four axis-planner instantiations when the
build log of this tree is present."""

from __future__ import annotations

import argparse
import ctypes
import json
import os
import re
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
TOOL = (0.0, 0.0, 1.0)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else None
    except (OSError, subprocess.SubprocessError):
        return None


def ptxas_lines():
    """{kernel: 'N registers, S bytes stack, spills'} of move_axis_plan_kernel from the tree's build log, if any."""
    path = os.path.join(ROOT, "mujoco_panda_pnp_b200", "csrc", "build.log")
    if not os.path.exists(path):
        return None
    out, cur = {}, None
    for line in open(path):
        m = re.search(r"Compiling entry function '(_ZN3pnp21move_axis_plan_kernel\w+)'", line)
        if m:
            cur = m.group(1)
            continue
        if cur and ("spill" in line or "Used" in line):
            out[cur] = (out.get(cur, "") + " " + line.split(":", 1)[-1].strip()).strip()
            if "Used" in line:
                cur = None
    return out


def event_ms(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def outputs(n, cap, dev):
    return dict(pos=torch.empty((n, cap, 3), device=dev), axis=torch.empty((n, cap, 3), device=dev),
                quat=torch.empty((n, cap, 4), device=dev), q=torch.empty((n, cap, 7), device=dev),
                tlen=torch.empty(n, dtype=torch.int32, device=dev), qf=torch.empty((n, 7), device=dev),
                solves=torch.empty(n, dtype=torch.int32, device=dev), status=torch.empty(n, dtype=torch.int32, device=dev))


def measure(lib, params, mp, qs, gp, ga, gq, warmup, iters):
    n, dev = qs.shape[0], qs.device
    cap = mp.traj_cap
    oa, op = outputs(n, cap, dev), outputs(n, cap, dev)
    tool = (ctypes.c_double * 3)(*TOOL)
    stream = lambda: torch.cuda.current_stream().cuda_stream  # noqa: E731

    def axis(counters=None):
        _lib.check(lib.pnp_move_ik_plan_axis_f32(
            qs.data_ptr(), gp.data_ptr(), ga.data_ptr(), n, ctypes.byref(mp), ctypes.byref(params), tool,
            *(oa[k].data_ptr() for k in ("pos", "axis", "quat", "q", "tlen", "qf", "solves", "status")),
            None if counters is None else counters.data_ptr(), stream()), "axis planner")

    def pose(counters=None):
        _lib.check(lib.pnp_move_ik_plan_pose_f32(
            qs.data_ptr(), gp.data_ptr(), gq.data_ptr(), n, ctypes.byref(mp), ctypes.byref(params),
            *(op[k].data_ptr() for k in ("pos", "quat", "q", "tlen", "qf", "solves", "status")),
            None if counters is None else counters.data_ptr(), stream()), "pose planner")

    variants = (axis, pose)
    for _ in range(warmup):
        for f in variants:
            f()
    torch.cuda.synchronize()
    times = {f.__name__: [] for f in variants}
    for _ in range(iters):
        for f in variants:
            times[f.__name__].append(event_ms(f))
    run = dict(n=n)
    for f, o in ((axis, oa), (pose, op)):
        name = f.__name__
        med = statistics.median(times[name])
        cnt = torch.zeros(4, dtype=torch.int64, device=dev)
        f(cnt)
        torch.cuda.synchronize()
        c = cnt.cpu().tolist()
        st = o["status"]
        run.update({
            f"{name}_ms": med, f"{name}_ms_min": min(times[name]), f"{name}_plans_per_s": n / (med * 1e-3),
            f"{name}_passes_per_s": c[3] / (med * 1e-3),
            f"{name}_ok": float((st == 0).float().mean()), f"{name}_broke": float((st & 1 != 0).float().mean()),
            f"{name}_capped": float((st & 2 != 0).float().mean()),
            f"{name}_mean_points": float(o["tlen"].float().mean()), f"{name}_mean_solves": float(o["solves"].float().mean()),
            f"{name}_passes_per_solve": c[3] / max(c[0], 1),
        })
    run["pose_over_axis"] = run["pose_ms"] / run["axis_ms"]
    return run


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[14, 16, 18, 20], help="log2 of the W1 batch sizes")
    ap.add_argument("--w2-size", type=int, default=16, help="log2 of the W2 batch size")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_axis_planner needs a CUDA device")
    dev = torch.device("cuda", torch.cuda.current_device())
    lib = _lib.load()
    tree = KinematicTree.from_mjcf()
    engine.set_tree(tree)
    params = engine.ik_params()
    mp = _lib.PnpMovePoseParams(PLAN["pos_thresh"], PLAN["rot_thresh"], PLAN["step_size"], PLAN["rot_step"],
                                PLAN["ik_rot_thresh"], PLAN["rot_weight"], PLAN["max_traj_points"],
                                PLAN["max_traj_points"] + 1)
    result = dict(tool="bench_axis_planner", gpu=gpu_info(), torch=torch.__version__, warmup=args.warmup,
                  iters=args.iters, plan=PLAN, tool_axis=TOOL, ptxas=ptxas_lines(), w1={}, w2={})
    neutral = torch.tensor([synthetic.NEUTRAL_Q], dtype=torch.float32, device=dev)
    _, neutral_quat, _ = engine.fk_jac(neutral, want_jac=False)
    for lg, key in [(lg, "w1") for lg in args.sizes] + [(args.w2_size, "w2")]:
        n = 1 << lg
        e = synthetic.reachable_pose_move_envs(n, tree.lower, tree.upper, seed=0, device=dev)
        gp, gq, _ = engine.fk_jac(e["q_goal"], want_jac=False)
        if key == "w1":
            ga = engine.ik_axis_solve(gp, torch.tensor([[0.0, 0.0, 1.0]], device=dev).expand(n, 3).contiguous(),
                                      e["q_goal"], engine.ik_params(max_iters=0), tool_axis=TOOL)["final_axis"]
        else:
            ga = torch.tensor([[0.0, 0.0, -1.0]], device=dev).expand(n, 3).contiguous()
            gq = neutral_quat.expand(n, 4).contiguous()
        run = measure(lib, params, mp, e["q_start"], gp, ga, gq, args.warmup, args.iters)
        result[key][str(lg)] = run
        print(json.dumps(dict(progress=f"{key} 2^{lg}", **run)), file=sys.stderr)
        torch.cuda.empty_cache()
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()

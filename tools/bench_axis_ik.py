"""Time the axis-constrained IK solve against the pose solve on the same q*, and its multistart.

    python tools/bench_axis_ik.py [--sizes 20 22] [--warmup 3] [--iters 10] [--seeds 8] [--groups 1 2 4]

Workload A-cold, float32, reference defaults (max_iters 100, pos_thresh 1e-3, rot_thresh 1e-2, rot_weight 1), every
query solved from NEUTRAL: q* ~ U(joint range) from the device generator with seed 1234; the axis task is
(FK(q*), R(q*) t) with the tool axis t = site +z, the pose task on the same q* is (FK(q*), quat(q*)).  The plain axis
solve and the plain pose solve alternate within each repetition, each timed alone between two CUDA events; medians
are reported.  At 2^20 queries inputs and outputs about fill the 126 MB L2, at 2^22 they do not.  The multistart runs
with engine.ik_restart_seeds(8); --groups times it once per restart group width, each in a child process with
PNP_MS_AXIS_GROUP set (the library reads it once per process).  The card's name, power limit and max SM clock are read
in the same call, and the registers, stack frame and spills of every axis and pose instantiation are taken from the
build's -Xptxas -v log.  The FP64 (parity) instantiations of both plain solves are timed too, up to --fp64-max.
Prints one JSON line.
"""

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

NEUTRAL = (0.00, 0.41, 0.00, -1.85, 0.00, 2.26, 0.79)
BUILD_LOG = os.path.join(ROOT, "mujoco_panda_pnp_b200", "csrc", "build.log")


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else None
    except (OSError, subprocess.SubprocessError):
        return None


def registers():
    """{kernel instantiation: [registers, stack frame bytes, spill stores, spill loads]} of the axis and pose IK kernels."""
    if not os.path.exists(BUILD_LOG):
        return None
    out, cur = {}, None
    for line in open(BUILD_LOG):
        m = re.search(r"Compiling entry function '(\S+)'", line)
        if m:
            name = m.group(1)
            cur = name if re.search(r"(axis|pose)_(solve|wave)_kernel", name) and "move" not in name else None
            continue
        if cur is None:
            continue
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and cur not in out:  # the entry's own line comes first; callees follow
            out[cur] = [None, int(m.group(1)), int(m.group(2)), int(m.group(3))]
        m = re.search(r"Used (\d+) registers", line)
        if m and cur in out:
            out[cur][0] = int(m.group(1))
            cur = None
    return out


def event_ms(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def targets(tree, n, dev):
    q = synthetic.random_joint_configs(n, tree.lower, tree.upper, seed=1234, device=dev, dtype=torch.float64)
    pos, quat, _ = engine.fk_jac(q, want_jac=False)
    w, x, y, z = quat.unbind(1)
    axis = torch.stack([2 * (x * z + w * y), 2 * (y * z - w * x), 1 - 2 * (x * x + y * y)], dim=1)  # R(q*) e_z
    return pos.float().contiguous(), quat.float().contiguous(), axis.float().contiguous()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[20, 22], help="log2 of the batch sizes")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--seeds", type=int, default=8)
    ap.add_argument("--groups", type=int, nargs="*", default=[1, 2, 4], help="restart group widths to time")
    ap.add_argument("--fp64-max", type=int, default=20, help="largest log2 size the FP64 solves are timed at")
    ap.add_argument("--multistart-only", action="store_true", help="(child process of the group sweep)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_axis_ik needs a CUDA device")
    dev = torch.device("cuda", torch.cuda.current_device())
    lib = _lib.load()
    tree = KinematicTree.from_mjcf()
    engine.set_tree(tree)
    params = engine.ik_params()
    neutral = torch.tensor(NEUTRAL, dtype=torch.float32, device=dev)
    seeds = engine.ik_restart_seeds(args.seeds, tree.lower, tree.upper, device=dev)
    stream = lambda: torch.cuda.current_stream().cuda_stream  # noqa: E731
    tool = (ctypes.c_double * 3)(0.0, 0.0, 1.0)
    group = os.environ.get("PNP_MS_AXIS_GROUP")
    result = dict(tool="bench_axis_ik", gpu=gpu_info(), torch=torch.__version__, k_seeds=args.seeds,
                  warmup=args.warmup, iters=args.iters, group_env=group, runs={})
    if not args.multistart_only:
        result["registers_stack_spill_stores_loads"] = registers()
    for lg in args.sizes:
        n = 1 << lg
        tp, tq, ta = targets(tree, n, dev)
        o = [torch.empty((n, 7), device=dev), torch.empty((n, 3), device=dev), torch.empty((n, 3), device=dev),
             torch.empty((n, 4), device=dev), torch.empty(n, device=dev), torch.empty(n, device=dev),
             torch.empty(n, dtype=torch.int32, device=dev), torch.empty(n, dtype=torch.uint8, device=dev)]
        attempt = torch.empty(n, dtype=torch.uint8, device=dev)
        nb = ctypes.c_int64()
        _lib.check(lib.pnp_ik_multistart_scratch_bytes(n, ctypes.byref(nb)), "scratch_bytes")
        scratch = torch.empty((nb.value + 15) // 16 * 4, dtype=torch.int32, device=dev)
        axis_out = [t.data_ptr() for t in o]
        pose_out = [o[i].data_ptr() for i in (0, 1, 3, 4, 5, 6, 7)]

        def ptr(t):
            return t.data_ptr() if t is not None else None

        def axis(counters=None):
            _lib.check(lib.pnp_ik_axis_solve_f32(tp.data_ptr(), ta.data_ptr(), neutral.data_ptr(), 0, n,
                                                 ctypes.byref(params), tool, 1e-2, 1.0, *axis_out, ptr(counters),
                                                 stream()), "axis")

        def pose(counters=None):
            _lib.check(lib.pnp_ik_pose_solve_f32(tp.data_ptr(), tq.data_ptr(), neutral.data_ptr(), 0, n,
                                                 ctypes.byref(params), 1e-2, 1.0, *pose_out, ptr(counters), stream()),
                       "pose")

        def multi(counters=None, stats=None):
            _lib.check(lib.pnp_ik_axis_solve_multistart_f32(
                tp.data_ptr(), ta.data_ptr(), neutral.data_ptr(), 0, n, seeds.data_ptr(), args.seeds,
                ctypes.byref(params), tool, 1e-2, 1.0, *axis_out, attempt.data_ptr(), ptr(counters), ptr(stats),
                scratch.data_ptr(), stream()), "multistart")

        variants = [multi] if args.multistart_only else [axis, pose, multi]
        for _ in range(args.warmup):
            for f in variants:
                f()
        torch.cuda.synchronize()
        times = {f.__name__: [] for f in variants}
        for _ in range(args.iters):
            for f in variants:
                times[f.__name__].append(event_ms(f))
        med = {k: statistics.median(v) for k, v in times.items()}
        run = dict(n=n, multistart_ms=med["multi"], multistart_ms_min=min(times["multi"]))
        cm = torch.zeros(4, dtype=torch.int64, device=dev)
        stats = torch.zeros(3, dtype=torch.int64, device=dev)
        multi(cm, stats)
        torch.cuda.synchronize()
        cm = cm.cpu().numpy()
        run.update(multistart_success=float(cm[2]) / n,
                   restart_stats=dict(restarted=int(stats[0]), rescued=int(stats[1]), restart_dls_passes=int(stats[2])))
        if not args.multistart_only:
            ca, cp = torch.zeros(4, dtype=torch.int64, device=dev), torch.zeros(4, dtype=torch.int64, device=dev)
            axis(ca)
            pose(cp)
            torch.cuda.synchronize()
            ca, cp = ca.cpu().numpy(), cp.cpu().numpy()
            run.update(axis_ms=med["axis"], axis_ms_min=min(times["axis"]), pose_ms=med["pose"],
                       pose_ms_min=min(times["pose"]), axis_success=float(ca[2]) / n, pose_success=float(cp[2]) / n,
                       axis_mean_passes=float(ca[3]) / n, pose_mean_passes=float(cp[3]) / n,
                       axis_ns_per_pass=med["axis"] * 1e6 / float(ca[3]), pose_ns_per_pass=med["pose"] * 1e6 / float(cp[3]))
        if not args.multistart_only and lg <= args.fp64_max:
            # the FP64 (parity) instantiations: the axis pass is one out-of-line function there
            tp64, tq64, ta64 = (t.double() for t in (tp, tq, ta))
            n64 = neutral.double()
            o64 = [t.double() if t.is_floating_point() else t for t in o]
            a64 = [t.data_ptr() for t in o64]
            p64 = [o64[i].data_ptr() for i in (0, 1, 3, 4, 5, 6, 7)]
            c64a, c64p = (torch.zeros(4, dtype=torch.int64, device=dev) for _ in range(2))

            def axis64(counters=None):
                _lib.check(lib.pnp_ik_axis_solve_f64(tp64.data_ptr(), ta64.data_ptr(), n64.data_ptr(), 0, n,
                                                     ctypes.byref(params), tool, 1e-2, 1.0, *a64, ptr(counters),
                                                     stream()), "axis64")

            def pose64(counters=None):
                _lib.check(lib.pnp_ik_pose_solve_f64(tp64.data_ptr(), tq64.data_ptr(), n64.data_ptr(), 0, n,
                                                     ctypes.byref(params), 1e-2, 1.0, *p64, ptr(counters), stream()),
                           "pose64")

            axis64(c64a), pose64(c64p)
            torch.cuda.synchronize()
            t64 = {"axis64": [], "pose64": []}
            for _ in range(max(3, args.iters // 2)):
                for f in (axis64, pose64):
                    t64[f.__name__].append(event_ms(f))
            c64a, c64p = c64a.cpu().numpy(), c64p.cpu().numpy()
            m64 = {k: statistics.median(v) for k, v in t64.items()}
            run.update(fp64=dict(axis_ms=m64["axis64"], pose_ms=m64["pose64"], axis_success=float(c64a[2]) / n,
                                 pose_success=float(c64p[2]) / n,
                                 axis_ns_per_pass=m64["axis64"] * 1e6 / float(c64a[3]),
                                 pose_ns_per_pass=m64["pose64"] * 1e6 / float(c64p[3])))
            del tp64, tq64, ta64, o64
        result["runs"][f"a_cold_{lg}"] = run
        del tp, tq, ta, o, attempt, scratch
        torch.cuda.empty_cache()
    if not args.multistart_only and args.groups:
        sweep = {}
        for g in args.groups:
            env = dict(os.environ, PNP_MS_AXIS_GROUP=str(g))
            cmd = [sys.executable, os.path.abspath(__file__), "--multistart-only", "--groups", "--sizes",
                   *map(str, args.sizes), "--warmup", str(args.warmup), "--iters", str(args.iters), "--seeds",
                   str(args.seeds)]
            out = subprocess.run(cmd, env=env, capture_output=True, text=True, check=True).stdout.strip().splitlines()
            child = json.loads(out[-1])
            sweep[str(g)] = {k: dict(ms=v["multistart_ms"], ms_min=v["multistart_ms_min"], success=v["multistart_success"])
                             for k, v in child["runs"].items()}
        result["multistart_group_sweep"] = sweep
    print(json.dumps(result))


if __name__ == "__main__":
    main()

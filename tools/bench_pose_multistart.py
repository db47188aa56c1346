"""Time the multi-start pose solve against the plain pose solve and against the torch composition a caller writes today.

    python tools/bench_pose_multistart.py [--sizes 20 22] [--warmup 3] [--iters 10] [--seeds 8] [--workloads w_cold near]

Workloads, float32, reference defaults (max_iters 100, pos_thresh 1e-3, rot_thresh 1e-2), every query solved from
NEUTRAL:
  w_cold  q* ~ U(joint range) from the device generator with seed 1234, target (FK(q*), quat(q*)): every target is
          reachable, about a quarter of them fail attempt 0
  near    q* = clip(NEUTRAL + U(-1, 1), joint range), same seed: about 1 in 400 fails attempt 0
Every call is timed alone between two CUDA events, the three variants alternate within each repetition, and the median
is reported.  At 2^20 queries the inputs and outputs (28 + 89 B per query, 117 MiB) about fill the 126 MB L2; at 2^22
they do not.  `waves_ms_by_k` times the multistart with the first G, 2G, ... seeds of the same table (G = lanes per
restarted query, PNP_MS_POSE_GROUP or the library default): the differences are the cost of each further wave.  Prints
one JSON line.
"""

from __future__ import annotations

import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import torch  # noqa: E402

from mujoco_panda_pnp_b200 import KinematicTree, _lib, engine, synthetic  # noqa: E402

NEUTRAL = (0.00, 0.41, 0.00, -1.85, 0.00, 2.26, 0.79)
DEFAULT_GROUP = 1  # kMsPoseGroup in csrc/pnp_capi.cu


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


def targets(tree, n, workload, dev):
    q = synthetic.random_joint_configs(n, tree.lower, tree.upper, seed=1234, device=dev, dtype=torch.float64)
    if workload == "near":
        lo = torch.as_tensor(tree.lower, dtype=torch.float64, device=dev)
        hi = torch.as_tensor(tree.upper, dtype=torch.float64, device=dev)
        g = torch.Generator(device=dev).manual_seed(1234)
        u = torch.rand((n, 7), generator=g, device=dev, dtype=torch.float64) * 2.0 - 1.0
        q = torch.minimum(torch.maximum(torch.tensor(NEUTRAL, dtype=torch.float64, device=dev) + u, lo), hi)
    pos, quat, _ = engine.fk_jac(q, want_jac=False)
    return pos.float().contiguous(), quat.float().contiguous()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[20, 22], help="log2 of the batch sizes")
    ap.add_argument("--workloads", nargs="+", default=["w_cold", "near"], choices=["w_cold", "near"])
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--seeds", type=int, default=8)
    ap.add_argument("--no-composition", action="store_true", help="skip the torch composition (group-width sweeps)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_pose_multistart needs a CUDA device")
    dev = torch.device("cuda", torch.cuda.current_device())
    lib = _lib.load()
    tree = KinematicTree.from_mjcf()
    engine.set_tree(tree)
    params = engine.ik_params()
    rot_thresh, rot_weight = 1e-2, 1.0
    neutral = torch.tensor(NEUTRAL, dtype=torch.float32, device=dev)
    seeds = engine.ik_restart_seeds(args.seeds, tree.lower, tree.upper, device=dev)
    group = int(os.environ.get("PNP_MS_POSE_GROUP", "0")) or None
    stream = lambda: torch.cuda.current_stream().cuda_stream  # noqa: E731
    result = dict(tool="bench_pose_multistart", gpu=gpu_info(), torch=torch.__version__, k_seeds=args.seeds,
                  warmup=args.warmup, iters=args.iters, group=group or DEFAULT_GROUP, group_override=group, runs={})
    for workload in args.workloads:
        for lg in args.sizes:
            n = 1 << lg
            tp, tq = targets(tree, n, workload, dev)
            o = dict(q=torch.empty((n, 7), device=dev), fpos=torch.empty((n, 3), device=dev),
                     fquat=torch.empty((n, 4), device=dev), perr=torch.empty(n, device=dev),
                     rerr=torch.empty(n, device=dev), iters=torch.empty(n, dtype=torch.int32, device=dev),
                     flags=torch.empty(n, dtype=torch.uint8, device=dev))
            attempt = torch.empty(n, dtype=torch.uint8, device=dev)
            nb = ctypes.c_int64()
            _lib.check(lib.pnp_ik_multistart_scratch_bytes(n, ctypes.byref(nb)), "scratch_bytes")
            scratch = torch.empty((nb.value + 15) // 16 * 4, dtype=torch.int32, device=dev)
            outs = [o[k].data_ptr() for k in ("q", "fpos", "fquat", "perr", "rerr", "iters", "flags")]

            def ptr(t):
                return t.data_ptr() if t is not None else None

            def plain(counters=None):
                _lib.check(lib.pnp_ik_pose_solve_f32(tp.data_ptr(), tq.data_ptr(), neutral.data_ptr(), 0, n,
                                                     ctypes.byref(params), rot_thresh, rot_weight, *outs,
                                                     ptr(counters), stream()), "plain")

            def multi(k=args.seeds, counters=None, stats=None):
                _lib.check(lib.pnp_ik_pose_solve_multistart_f32(
                    tp.data_ptr(), tq.data_ptr(), neutral.data_ptr(), 0, n, seeds.data_ptr(), k, ctypes.byref(params),
                    rot_thresh, rot_weight, *outs, attempt.data_ptr(), ptr(counters), ptr(stats), scratch.data_ptr(),
                    stream()), "multistart")

            def composition():
                # what a caller writes without the multistart entry point: solve, nonzero, gather, re-solve, scatter
                r = engine.ik_pose_solve(tp, tq, neutral, params, rot_thresh=rot_thresh, rot_weight=rot_weight)
                left = torch.nonzero(~r["success"]).flatten()
                for k in range(args.seeds):
                    if left.numel() == 0:
                        break
                    rk = engine.ik_pose_solve(tp.index_select(0, left), tq.index_select(0, left), seeds[k], params,
                                              rot_thresh=rot_thresh, rot_weight=rot_weight)
                    ok = rk["success"]
                    rows = left[ok]
                    for key in ("q", "final_pos", "final_quat", "pos_error", "rot_error", "iterations", "converged",
                                "success"):
                        r[key].index_copy_(0, rows, rk[key][ok])
                    left = left[~ok]
                return r

            variants = [plain, multi] + ([] if args.no_composition else [composition])
            for _ in range(args.warmup):
                for f in variants:
                    f()
            torch.cuda.synchronize()
            times = {f.__name__: [] for f in variants}
            for _ in range(args.iters):
                for f in variants:
                    times[f.__name__].append(event_ms(f))
            # outputs and statistics, outside the timed calls
            c_plain = torch.zeros(4, dtype=torch.int64, device=dev)
            plain(c_plain)
            c_multi = torch.zeros(4, dtype=torch.int64, device=dev)
            stats = torch.zeros(3, dtype=torch.int64, device=dev)
            multi(counters=c_multi, stats=stats)
            torch.cuda.synchronize()
            multi_success_out = float(((o["flags"] >> 1) & 1).float().mean())
            g = group or DEFAULT_GROUP
            waves = {}
            for k in list(range(g, args.seeds, g)) + [args.seeds]:
                for _ in range(2):
                    multi(k)
                waves[str(k)] = statistics.median(event_ms(lambda: multi(k)) for _ in range(max(5, args.iters // 2)))
            cp, cm = c_plain.cpu().numpy(), c_multi.cpu().numpy()
            med = {k: statistics.median(v) for k, v in times.items()}
            run = dict(
                n=n, workload=workload,
                plain_ms=med["plain"], plain_ms_min=min(times["plain"]), plain_success=float(cp[2]) / n,
                multistart_ms=med["multi"], multistart_ms_min=min(times["multi"]),
                multistart_success=float(cm[2]) / n, multistart_success_from_outputs=multi_success_out,
                multistart_over_plain=med["multi"] / med["plain"],
                restart_stats=dict(restarted=int(stats[0]), rescued=int(stats[1]), restart_dls_passes=int(stats[2]),
                                   plain_dls_passes=int(cp[3])),
                waves_ms_by_k=waves,
            )
            if not args.no_composition:
                r = composition()
                torch.cuda.synchronize()
                run.update(composition_ms=med["composition"], composition_ms_min=min(times["composition"]),
                           composition_success=float(r["success"].float().mean()),
                           composition_over_multistart=med["composition"] / med["multi"])
            result["runs"][f"{workload}_{lg}"] = run
            del tp, tq, o, outs, attempt, scratch
            torch.cuda.empty_cache()
    print(json.dumps(result))


if __name__ == "__main__":
    main()

"""Time the cone-tolerant axis IK solve against the exact axis solve on the four workloads of DESIGN.md 4.9.

    python tools/bench_cone_ik.py [--sizes 20 22] [--warmup 3] [--iters 10] [--degrees 10 20 30] [--seeds 8]

float32, reference defaults (max_iters 100, pos_thresh 1e-3, rot_thresh 1e-2, rot_weight 1), tool axis site +z, every
query solved from NEUTRAL.  Workloads: A-cold (q* ~ U(joint range) from the device generator with seed 1234, target
(FK(q*), R(q*) z)); top-down (the same positions, axis world -z); shelf top-down (positions uniform in
synthetic.SHELF_BOX, NumPy default_rng(0), axis -z); shelf horizontal (the same positions, axis world +x).  Per size and
workload, the axis solve and the cone solve at each angle alternate within each repetition, each timed alone between two
CUDA events; medians of --iters repetitions are reported with the success rate, the mean passes and the DLS passes per
second from the solves' counters.  At 2^20 queries inputs and outputs about fill the 126 MB L2, at 2^22 they do not.
The multistart with engine.ik_restart_seeds(--seeds) runs at 20 degrees.  The card's name, power limit and max SM clock
are read in the same call, and the registers, stack frame and spills of the axis and cone kernels are taken from the
build's -Xptxas -v log.  Prints one JSON line.
"""

from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402
import torch  # noqa: E402

from bench_axis_ik import event_ms, gpu_info  # noqa: E402
from mujoco_panda_pnp_b200 import KinematicTree, engine, synthetic  # noqa: E402

NEUTRAL = (0.00, 0.41, 0.00, -1.85, 0.00, 2.26, 0.79)
BUILD_LOG = os.path.join(ROOT, "mujoco_panda_pnp_b200", "csrc", "build.log")


def registers():
    """{kernel instantiation: [registers, stack frame bytes, spill stores, spill loads]} of the axis and cone kernels."""
    import re

    if not os.path.exists(BUILD_LOG):
        return None
    out, cur = {}, None
    for line in open(BUILD_LOG):
        m = re.search(r"Compiling entry function '(\S+)'", line)
        if m:
            name = m.group(1)
            cur = name if re.search(r"axis(_cone)?_(solve|wave)_kernel", name) and "move" not in name else None
            continue
        if cur is None:
            continue
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and cur not in out:
            out[cur] = [None, int(m.group(1)), int(m.group(2)), int(m.group(3))]
        m = re.search(r"Used (\d+) registers", line)
        if m and cur in out:
            out[cur][0] = int(m.group(1))
            cur = None
    return out


def workloads(tree, n, dev):
    q = synthetic.random_joint_configs(n, tree.lower, tree.upper, seed=1234, device=dev, dtype=torch.float64)
    pos, quat, _ = engine.fk_jac(q, want_jac=False)
    w, x, y, z = quat.unbind(1)
    axis = torch.stack([2 * (x * z + w * y), 2 * (y * z - w * x), 1 - 2 * (x * x + y * y)], dim=1)  # R(q*) e_z
    box = np.array(synthetic.SHELF_BOX)
    ps = torch.tensor(box[:, 0] + (box[:, 1] - box[:, 0]) * np.random.default_rng(0).random((n, 3)), device=dev)
    down = torch.tensor([0.0, 0.0, -1.0], device=dev).expand(n, 3)
    horiz = torch.tensor([1.0, 0.0, 0.0], device=dev).expand(n, 3)
    f = lambda t: t.float().contiguous()  # noqa: E731
    return dict(a_cold=(f(pos), f(axis)), top_down=(f(pos), f(down)), shelf_top_down=(f(ps), f(down)),
                shelf_horizontal=(f(ps), f(horiz)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[20, 22], help="log2 of the batch sizes")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--degrees", type=float, nargs="+", default=[10.0, 20.0, 30.0])
    ap.add_argument("--seeds", type=int, default=8)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_cone_ik needs a CUDA device")
    dev = torch.device("cuda", torch.cuda.current_device())
    tree = KinematicTree.from_mjcf()
    engine.set_tree(tree)
    params = engine.ik_params()
    neutral = torch.tensor(NEUTRAL, dtype=torch.float32, device=dev)
    seeds = engine.ik_restart_seeds(args.seeds, tree.lower, tree.upper, device=dev)
    result = dict(tool="bench_cone_ik", gpu=gpu_info(), torch=torch.__version__, warmup=args.warmup, iters=args.iters,
                  k_seeds=args.seeds, registers_stack_spill_stores_loads=registers(), runs={})
    variants = [None] + [math.radians(d) for d in args.degrees]
    names = ["axis"] + [f"cone_{d:g}" for d in args.degrees]
    for lg in args.sizes:
        n = 1 << lg
        for wname, (tp, ta) in workloads(tree, n, dev).items():
            calls = [lambda c=None, a=a: engine.ik_axis_solve(tp, ta, neutral, params, counters=c, cone_angle=a)
                     for a in variants]
            for _ in range(args.warmup):
                for f in calls:
                    f()
            torch.cuda.synchronize()
            times = [[] for _ in calls]
            for _ in range(args.iters):
                for k, f in enumerate(calls):
                    times[k].append(event_ms(f))
            run = {}
            for k, f in enumerate(calls):
                c = torch.zeros(4, dtype=torch.int64, device=dev)
                f(c)
                torch.cuda.synchronize()
                c = c.cpu().numpy()
                ms = statistics.median(times[k])
                run[names[k]] = dict(ms=ms, ms_min=min(times[k]), success=float(c[2]) / n, mean_passes=float(c[3]) / n,
                                     dls_passes_per_s=float(c[3]) / (ms * 1e-3))
            for k in range(1, len(calls)):
                run[names[k]].update(wall_ratio_vs_axis=run[names[k]]["ms"] / run["axis"]["ms"],
                                     pass_rate_ratio_vs_axis=run[names[k]]["dls_passes_per_s"]
                                     / run["axis"]["dls_passes_per_s"])
            if wname in ("a_cold", "shelf_horizontal"):
                alpha = math.radians(20.0)
                multi = lambda c=None, s=None: engine.ik_axis_solve_multistart(  # noqa: E731
                    tp, ta, neutral, seeds, params, counters=c, restart_stats=s, cone_angle=alpha)
                multi()
                torch.cuda.synchronize()
                mt = [event_ms(multi) for _ in range(args.iters)]
                c = torch.zeros(4, dtype=torch.int64, device=dev)
                st = torch.zeros(3, dtype=torch.int64, device=dev)
                multi(c, st)
                torch.cuda.synchronize()
                run["multistart_cone_20"] = dict(ms=statistics.median(mt), success=float(c[2]) / n,
                                                 restart_stats=[int(v) for v in st.cpu().numpy()])
            result["runs"][f"{wname}_{lg}"] = run
            print(json.dumps({f"{wname}_{lg}": run}), file=sys.stderr, flush=True)
        torch.cuda.empty_cache()
    print(json.dumps(result))


if __name__ == "__main__":
    main()

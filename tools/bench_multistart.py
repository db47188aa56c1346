"""Time the multi-start position solve against the plain solve and against the torch composition a caller writes today.

    python tools/bench_multistart.py [--sizes 20 22 24] [--warmup 3] [--iters 20] [--seeds 8]

Workload: bench.py's cfg5 (targets = FK(q*), q* ~ U(joint range) from the device generator with seed 1234, cold from
NEUTRAL, reference defaults), float32 packed outputs.  Every launch is timed alone between two CUDA events (so the plain
solve gets no overlap with a neighbour), the three variants alternate within each repetition, and the median is
reported.  At 2^20 queries the inputs and outputs (12 + 48 B per query, 60 MiB) fit the 126 MB L2 and stay there
between launches; at 2^22 and 2^24 they do not.  `waves_ms` times the multistart with the first G, 2G, ... seeds of the
same table (G = lanes per restarted query): the differences are the cost of each further wave.  Prints one JSON line.
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

import numpy as np  # noqa: E402
import torch  # noqa: E402

from mujoco_panda_pnp_b200 import KinematicTree, _lib, engine, synthetic  # noqa: E402

NEUTRAL = (0.00, 0.41, 0.00, -1.85, 0.00, 2.26, 0.79)


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[20, 22, 24], help="log2 of the batch sizes")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--seeds", type=int, default=8)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_multistart needs a CUDA device")
    dev = torch.device("cuda", torch.cuda.current_device())
    lib = _lib.load()
    tree = KinematicTree.from_mjcf()
    engine.set_tree(tree)
    params = engine.ik_params()
    neutral = torch.tensor(NEUTRAL, dtype=torch.float32, device=dev)
    seeds = engine.ik_restart_seeds(args.seeds, tree.lower, tree.upper, device=dev)
    group = int(os.environ.get("PNP_MS_GROUP", "0")) or None
    stream = lambda: torch.cuda.current_stream().cuda_stream  # noqa: E731
    result = dict(tool="bench_multistart", gpu=gpu_info(), torch=torch.__version__, k_seeds=args.seeds,
                  warmup=args.warmup, iters=args.iters, group_override=group, sizes={})
    for lg in args.sizes:
        n = 1 << lg
        qstar = synthetic.random_joint_configs(n, tree.lower, tree.upper, seed=1234, device=dev)
        targets = engine.fk_jac(qstar, want_quat=False, want_jac=False)[0]
        del qstar
        q8, aux = torch.empty((n, 8), device=dev), torch.empty((n, 4), device=dev)
        attempt = torch.empty(n, dtype=torch.uint8, device=dev)
        nb = ctypes.c_int64()
        _lib.check(lib.pnp_ik_multistart_scratch_bytes(n, ctypes.byref(nb)), "scratch_bytes")
        scratch = torch.empty((nb.value + 15) // 16 * 4, dtype=torch.int32, device=dev)

        def plain(counters=None):
            _lib.check(lib.pnp_ik_solve_packed_f32(targets.data_ptr(), neutral.data_ptr(), 0, n, ctypes.byref(params),
                                                   q8.data_ptr(), aux.data_ptr(),
                                                   counters.data_ptr() if counters is not None else None, stream()), "plain")

        def multi(k=args.seeds, counters=None, stats=None):
            _lib.check(lib.pnp_ik_solve_multistart_packed_f32(
                targets.data_ptr(), neutral.data_ptr(), 0, n, seeds.data_ptr(), k, ctypes.byref(params), q8.data_ptr(),
                aux.data_ptr(), attempt.data_ptr(), counters.data_ptr() if counters is not None else None,
                stats.data_ptr() if stats is not None else None, scratch.data_ptr(), stream()), "multistart")

        def composition():
            # what a caller writes without the multistart entry point: solve, nonzero, gather, re-solve, scatter
            r = engine.ik_solve(targets, neutral, params, out_q8=q8, out_aux4=aux)
            left = torch.nonzero(~r.success).flatten()
            for k in range(args.seeds):
                if left.numel() == 0:
                    break
                m = left.numel()
                q8k, auxk = torch.empty((m, 8), device=dev), torch.empty((m, 4), device=dev)
                ok = engine.ik_solve(targets.index_select(0, left), seeds[k], params, out_q8=q8k, out_aux4=auxk).success
                rows = left[ok]
                q8.index_copy_(0, rows, q8k[ok])
                aux.index_copy_(0, rows, auxk[ok])
                left = left[~ok]

        for _ in range(args.warmup):
            plain(), multi(), composition()
        torch.cuda.synchronize()
        t_plain, t_multi, t_comp = [], [], []
        for _ in range(args.iters):
            t_plain.append(event_ms(plain))
            t_multi.append(event_ms(multi))
            t_comp.append(event_ms(composition))
        # outputs and statistics, outside the timed launches
        c_plain = torch.zeros(4, dtype=torch.int64, device=dev)
        plain(c_plain)
        c_multi = torch.zeros(4, dtype=torch.int64, device=dev)
        stats = torch.zeros(3, dtype=torch.int64, device=dev)
        multi(counters=c_multi, stats=stats)
        torch.cuda.synchronize()
        word = aux[:, 3].view(torch.int32)
        multi_success_out = float(((word >> 25) & 1).float().mean())
        composition()
        torch.cuda.synchronize()
        comp_success = float(((aux[:, 3].view(torch.int32) >> 25) & 1).float().mean())
        # the cost of each wave: the same table cut to the first G, 2G, ... seeds
        g = group or 4
        waves = {}
        for k in list(range(g, args.seeds, g)) + [args.seeds]:
            for _ in range(2):
                multi(k)
            waves[str(k)] = statistics.median(event_ms(lambda: multi(k)) for _ in range(max(5, args.iters // 2)))
        cp, cm = c_plain.cpu().numpy(), c_multi.cpu().numpy()
        result["sizes"][str(lg)] = dict(
            n=n,
            plain_ms=statistics.median(t_plain), plain_ms_min=min(t_plain), plain_success=float(cp[2]) / n,
            multistart_ms=statistics.median(t_multi), multistart_ms_min=min(t_multi),
            multistart_success=float(cm[2]) / n, multistart_success_from_outputs=multi_success_out,
            restart_stats=dict(restarted=int(stats[0]), rescued=int(stats[1]), restart_dls_passes=int(stats[2]),
                               plain_dls_passes=int(cp[3])),
            composition_ms=statistics.median(t_comp), composition_success=comp_success,
            multistart_over_plain=statistics.median(t_multi) / statistics.median(t_plain),
            waves_ms_by_k=waves,
            inputs_in_l2=n * 60 < 126e6,
        )
        del targets, q8, aux, attempt, scratch
        torch.cuda.empty_cache()
    print(json.dumps(result))


if __name__ == "__main__":
    main()

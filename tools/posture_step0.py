"""Step 0 of posture-regularised IK (DESIGN.md 4.7): the FP64 statement of oracle/posture_ik_oracle.py swept over the
null-space gain on the CPU, before any kernel is written.

    python tools/posture_step0.py [--n 65536] [--gains 0 0.02 0.05 0.1 0.2 0.5] [--out profiles/posture_step0.json]

Workloads, both from NEUTRAL with q_rest = the middle of each joint's range and the solvers' default parameters:
  position  cfg5 cold targets: q* ~ U(joint limits) (synthetic.random_joint_configs, seed 1234), target FK(q*)
  pose      W-cold: the same q*, target (FK(q*), site quaternion of q*)
Per gain and workload: success rate, mean iterations, mean |q - q_rest|, mean and 5th percentile of the smallest
normalised joint-limit margin, and the fraction of failures that end with a joint on its limit.  Then the default-gain
rule: the largest gain whose success rate on both workloads is no more than 0.1 point below plain and whose mean
iteration count is at most 1.25x plain (None: no gain above 0 qualifies).
"""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))

from mujoco_panda_pnp_b200 import synthetic  # noqa: E402
from oracle import c_oracle, mj_oracle, posture_ik_oracle  # noqa: E402

ASSET = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "mujoco_panda_pnp_b200", "assets",
                     "panda_shelf_kinematic.xml")


def default_gain(rows):
    plain = rows[0]
    assert plain["gain"] == 0.0
    ok = [r["gain"] for r in rows[1:]
          if all(r[w]["success"] >= plain[w]["success"] - 1e-3 and r[w]["mean_iters"] <= 1.25 * plain[w]["mean_iters"]
                 for w in ("position", "pose"))]
    return max(ok) if ok else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1 << 16)
    ap.add_argument("--gains", type=float, nargs="+", default=[0.0, 0.02, 0.05, 0.1, 0.2, 0.5])
    ap.add_argument("--threads", type=int, default=os.cpu_count() or 8)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    chain = c_oracle.chain_from_model(mj_oracle.MjModel.from_xml_path(ASSET))
    t0 = time.time()
    rows = posture_ik_oracle.sweep(chain, np.array(synthetic.NEUTRAL_Q), n=args.n, gains=tuple(args.gains),
                                   nthreads=args.threads)
    res = dict(tool="posture_step0", n=args.n, precision="fp64 (CPU, oracle/posture_ik_oracle.py)",
               q_rest="mid-range of the joint limits", q_init="NEUTRAL", seed=1234, rows=rows,
               default_gain=default_gain(rows), seconds=round(time.time() - t0, 1))
    for r in rows:
        print(f"gain {r['gain']:<6} " + " | ".join(
            f"{w}: succ {r[w]['success']:.4f} iters {r[w]['mean_iters']:.2f} |q-q_rest| {r[w]['rest_dist']:.3f} "
            f"margin {r[w]['margin_mean']:.4f} p5 {r[w]['margin_p5']:.4f} fail@limit {r[w]['fail_on_limit']:.3f}"
            for w in ("position", "pose")))
    print("default gain:", res["default_gain"])
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
            f.write("\n")


if __name__ == "__main__":
    main()

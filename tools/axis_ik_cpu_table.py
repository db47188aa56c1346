"""The FP64 CPU table of DESIGN.md 4.8: axis task against pose task from NEUTRAL, default parameters, tool axis site +z.

    python tools/axis_ik_cpu_table.py [--n 4096]

Rows (each on the statements of oracle/axis_ik_oracle.py and oracle/pose_ik_oracle.py over the C oracle's FK):
  A-cold     q* ~ U(joint limits) (synthetic.random_joint_configs, seed 1234); axis (FK(q*), R(q*) z), pose
             (FK(q*), quat(q*))
  top-down   the same FK(q*) positions, axis world -z; pose with NEUTRAL's site quaternion
  shelf      positions uniform in synthetic.SHELF_BOX (NumPy default_rng(0)), top-down as above
Prints one JSON line.  Needs no GPU.
"""

from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402
import torch  # noqa: E402

from mujoco_panda_pnp_b200 import synthetic  # noqa: E402
from oracle import axis_ik_oracle, c_oracle, mj_oracle, pose_ik_oracle  # noqa: E402

ASSET = os.path.join(ROOT, "mujoco_panda_pnp_b200", "assets", "panda_shelf_kinematic.xml")


def row(axis, pose):
    return dict(axis_success=float(axis["success"].mean()), axis_mean_passes=float(axis["iterations"].mean()),
                pose_success=float(pose["success"].mean()), pose_mean_passes=float(pose["iterations"].mean()))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=4096)
    n = ap.parse_args().n
    c_oracle.build()
    chain = c_oracle.chain_from_model(mj_oracle.MjModel.from_xml_path(ASSET))
    lo, hi = np.array(chain.lower[:]), np.array(chain.upper[:])
    neutral = np.array(synthetic.NEUTRAL_Q)
    q = synthetic.random_joint_configs(n, lo, hi, seed=1234, dtype=torch.float64).numpy()
    p, mat, _ = c_oracle.fk_jac(chain, q, nthreads=8)
    quat = pose_ik_oracle.mat2quat_batch(mat.reshape(-1, 9))[0]
    out = dict(tool="axis_ik_cpu_table", n=n)
    out["a_cold"] = row(axis_ik_oracle.solve_axis_batch(chain, p, mat[:, :, 2], neutral),
                        pose_ik_oracle.solve_pose_batch(chain, p, quat, neutral))
    qn = pose_ik_oracle.mat2quat_batch(c_oracle.fk_jac(chain, neutral[None])[1].reshape(-1, 9))[0]
    down, qdown = np.tile([0.0, 0.0, -1.0], (n, 1)), np.tile(qn, (n, 1))
    out["top_down"] = row(axis_ik_oracle.solve_axis_batch(chain, p, down, neutral),
                          pose_ik_oracle.solve_pose_batch(chain, p, qdown, neutral))
    box = np.array(synthetic.SHELF_BOX)
    ps = box[:, 0] + (box[:, 1] - box[:, 0]) * np.random.default_rng(0).random((n, 3))
    out["shelf_top_down"] = row(axis_ik_oracle.solve_axis_batch(chain, ps, down, neutral),
                                pose_ik_oracle.solve_pose_batch(chain, ps, qdown, neutral))
    print(json.dumps(out))


if __name__ == "__main__":
    main()

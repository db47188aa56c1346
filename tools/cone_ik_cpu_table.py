"""The FP64 CPU table of DESIGN.md 4.9: cone-tolerant axis IK from NEUTRAL, default parameters, tool axis site +z.

    python tools/cone_ik_cpu_table.py [--n 4096]

Workloads (each on the statement of oracle/cone_ik_oracle.py over the C oracle's FK):
  A-cold            q* ~ U(joint limits) (synthetic.random_joint_configs, seed 1234), target (FK(q*), R(q*) z)
  top-down          the same FK(q*) positions, axis world -z
  shelf top-down    positions uniform in synthetic.SHELF_BOX (NumPy default_rng(0)), axis world -z
  shelf horizontal  the same positions, axis world +x (into the shelf)
Each cell is success rate and mean passes at one cone half-angle; 0 degrees is the axis solve.  The deadzone form
(tilt error w max(theta - alpha, 0), tilt rows kept in J), which the statement rejects, is given for A-cold and
top-down for contrast.  Prints one JSON line.  Needs no GPU.
"""

from __future__ import annotations

import argparse
import json
import math
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402
import torch  # noqa: E402

from mujoco_panda_pnp_b200 import synthetic  # noqa: E402
from oracle import axis_ik_oracle, c_oracle, cone_ik_oracle, mj_oracle  # noqa: E402

ASSET = os.path.join(ROOT, "mujoco_panda_pnp_b200", "assets", "panda_shelf_kinematic.xml")
DEGREES = (0, 5, 10, 15, 20, 30)


def deadzone(chain, tp, ta, q_init, alpha, max_iters=100, pos_thresh=1e-3, rot_thresh=1e-2, damping=1e-2,
             step_limit=0.1, w=1.0):
    """(success rate, mean passes) of the deadzone form: the axis solve with its tilt error clamped to
    w max(theta - alpha, 0) and the tilt rows left in J.  Kept here for contrast only."""
    n = len(tp)
    d = ta / np.linalg.norm(ta, axis=1, keepdims=True)
    basis = axis_ik_oracle.tool_basis((0.0, 0.0, 1.0))
    q = np.array(np.broadcast_to(q_init, (n, 7)))
    lo, hi = np.array(chain.lower[:]), np.array(chain.upper[:])
    it, conv, pe_o, g_o = np.zeros(n, int), np.zeros(n, bool), np.zeros(n), np.zeros(n)
    act = np.arange(n)
    for i in range(max_iters + 1):
        if len(act) == 0:
            break
        qa = q[act]
        p, mat, jac = c_oracle.fk_jac(chain, qa, nthreads=16)
        _, b1, b2, th, nv = axis_ik_oracle._axis_error(mat, basis, d[act])
        pe = np.linalg.norm(tp[act] - p, axis=1)
        g = np.maximum(th - alpha, 0.0)
        last = i == max_iters
        done = np.ones(len(act), bool) if last else (pe < pos_thresh) & (g < rot_thresh)
        idx = act[done]
        pe_o[idx], g_o[idx], conv[idx], it[idx] = pe[done], g[done], not last, max_iters if last else i + 1
        keep = ~done
        if not keep.any():
            break
        jr = jac[keep, 3:6]
        J = np.concatenate([jac[keep, :3], w * np.einsum("ni,nij->nj", b1[keep], jr)[:, None],
                            w * np.einsum("ni,nij->nj", b2[keep], jr)[:, None]], axis=1)
        e = np.concatenate([(tp[act] - p)[keep], (w * g[keep] * np.einsum("ni,ni->n", nv[keep], b1[keep]))[:, None],
                            (w * g[keep] * np.einsum("ni,ni->n", nv[keep], b2[keep]))[:, None]], axis=1)
        dq = (np.swapaxes(J, 1, 2) @ np.linalg.solve(J @ np.swapaxes(J, 1, 2) + damping * np.eye(5), e[:, :, None]))[:, :, 0]
        q[act[keep]] = np.clip(qa[keep] + np.clip(dq, -step_limit, step_limit), lo, hi)
        act = act[keep]
    succ = conv & (pe_o < 2 * pos_thresh) & (g_o < 2 * rot_thresh)
    return dict(success=float(succ.mean()), mean_passes=float(it.mean()))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=4096)
    n = ap.parse_args().n
    c_oracle.build()
    chain = c_oracle.chain_from_model(mj_oracle.MjModel.from_xml_path(ASSET))
    lo, hi = np.array(chain.lower[:]), np.array(chain.upper[:])
    neutral = np.array(synthetic.NEUTRAL_Q)
    q = synthetic.random_joint_configs(n, lo, hi, seed=1234, dtype=torch.float64).numpy()
    p, mat, _ = c_oracle.fk_jac(chain, q, nthreads=16)
    box = np.array(synthetic.SHELF_BOX)
    ps = box[:, 0] + (box[:, 1] - box[:, 0]) * np.random.default_rng(0).random((n, 3))
    down, horiz = np.tile([0.0, 0.0, -1.0], (n, 1)), np.tile([1.0, 0.0, 0.0], (n, 1))
    work = dict(a_cold=(p, mat[:, :, 2]), top_down=(p, down), shelf_top_down=(ps, down), shelf_horizontal=(ps, horiz))
    out = dict(tool="cone_ik_cpu_table", n=n, cone={}, deadzone={})
    for deg in DEGREES:
        row = {}
        for name, (tp, ta) in work.items():
            r = cone_ik_oracle.solve_cone_batch(chain, tp, ta, neutral, math.radians(deg), nthreads=16)
            row[name] = dict(success=float(r["success"].mean()), mean_passes=float(r["iterations"].mean()))
        out["cone"][str(deg)] = row
    for deg in (20, 45):
        out["deadzone"][str(deg)] = {name: deadzone(chain, *work[name], neutral, math.radians(deg))
                                     for name in ("a_cold", "top_down")}
    print(json.dumps(out))


if __name__ == "__main__":
    main()

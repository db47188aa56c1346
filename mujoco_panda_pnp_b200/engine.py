"""Thin Python layer over the C ABI: torch tensors (device memory, streams) in, tensors out.

PyTorch is plumbing here (allocation, current stream); every computation is a kernel of
libpnp_b200.so.  Functions taking CUDA tensors launch on ``torch.cuda.current_stream()`` and
return without synchronising.  Functions with a ``_host`` suffix take NumPy arrays / CPU
tensors and go through the library's own H2D -> kernel -> D2H pipeline (``pnp_*_host``).
"""

from __future__ import annotations

import ctypes
import threading
from typing import Dict, Optional, Tuple

import numpy as np
import torch

from . import _lib
from ._lib import KINEMATICS, PnpIkParams, PnpMoveParams, PnpNormalizeParams, PnpRewardParams
from .tree import KinematicTree, PnpTreeStruct

_uploaded: Dict[int, bytes] = {}  # device index -> bytes of the PnpTree currently in constant memory
_uploaded_obj: Dict[int, tuple] = {}  # device index -> (the KinematicTree object last uploaded, specialised?); trees are
#                                       treated as immutable once uploaded
_host_ctx: Dict[Tuple[int, int], ctypes.c_void_p] = {}


def _require_cuda() -> None:
    if not torch.cuda.is_available():
        raise _lib.PnpLibraryError("no CUDA device: mujoco_panda_pnp_b200 has no CPU path")


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def set_tree(tree: KinematicTree) -> bool:
    """Upload ``tree`` to the current device's constant memory (no-op if already there).

    Returns True when the library will use its build-time specialised kinematics for it."""
    dev = torch.cuda.current_device() if _uploaded_obj else -1
    hit = _uploaded_obj.get(dev)
    if hit is not None and hit[0] is tree:  # same object as last time on this device: nothing to do
        return hit[1]
    _require_cuda()
    dev = torch.cuda.current_device()
    lib = _lib.load()
    s = tree.to_struct()
    blob = bytes(s)
    if _uploaded.get(dev) != blob:
        _lib.check(lib.pnp_set_tree(ctypes.byref(s)), "pnp_set_tree")
        _uploaded[dev] = blob
    spec = bool(lib.pnp_tree_is_specialized())
    _uploaded_obj[dev] = (tree, spec)
    return spec


def specialized_tree() -> KinematicTree:
    """The tree the specialised kernels were generated for (from the library itself)."""
    s = PnpTreeStruct()
    _lib.check(_lib.load().pnp_get_specialized_tree(ctypes.byref(s)), "pnp_get_specialized_tree")
    return KinematicTree(
        link_pos=np.array(s.link_pos[:]).reshape(7, 3),
        link_rot=np.array(s.link_rot[:]).reshape(7, 3, 3),
        ee_pos=np.array(s.ee_pos[:]),
        ee_rot=np.array(s.ee_rot[:]).reshape(3, 3),
        lower=np.array(s.lower[:]),
        upper=np.array(s.upper[:]),
        qref=np.array(s.qref[:]),
    )


def ik_params(max_iters=100, pos_thresh=1e-3, damping=1e-2, step_limit=0.1, kinematics="auto") -> PnpIkParams:
    return PnpIkParams(int(max_iters), KINEMATICS[kinematics], float(pos_thresh), float(damping), float(step_limit))


def reward_params(reward_type="dense", n_tasks=3, initial_object_height=0.001, distance_threshold=0.05,
                  high_pick_z=0.35, threshold_report_tol=1e-6) -> PnpRewardParams:
    if reward_type not in ("dense", "sparse"):
        raise ValueError(f"reward_type must be 'dense' or 'sparse', got {reward_type!r}")
    return PnpRewardParams(int(reward_type == "sparse"), int(n_tasks), float(initial_object_height),
                           float(distance_threshold), float(high_pick_z), float(threshold_report_tol))


def _check_cuda(name: str, t: torch.Tensor, dtype, shape_tail) -> torch.Tensor:
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise ValueError(f"{name} must be a CUDA tensor")
    if t.dtype != dtype:
        raise ValueError(f"{name} must be {dtype}, got {t.dtype}")
    if tuple(t.shape[1:]) != tuple(shape_tail):
        raise ValueError(f"{name} must have shape (N, {', '.join(map(str, shape_tail))}), got {tuple(t.shape)}")
    return t.contiguous()


def _check_out(name: str, t, shape, dtype, device) -> torch.Tensor:
    """A caller-supplied CUDA output buffer goes to the library as a bare pointer: refuse anything that is not exactly
    the buffer the kernel will write (shape, dtype, device, contiguous)."""
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise ValueError(f"{name} must be a CUDA tensor")
    if tuple(t.shape) != tuple(shape) or t.dtype != dtype or t.device != device or not t.is_contiguous():
        raise ValueError(f"{name} must be a contiguous {dtype} tensor of shape {tuple(shape)} on {device}, got "
                         f"{t.dtype} {tuple(t.shape)} on {t.device}{'' if t.is_contiguous() else ' (not contiguous)'}")
    return t


def _check_out_np(name: str, a, shape, dtype) -> np.ndarray:
    """Same for a host output buffer of the host-buffer operators (written by cudaMemcpyAsync)."""
    if not isinstance(a, np.ndarray) or a.shape != tuple(shape) or a.dtype != np.dtype(dtype) or not a.flags["C_CONTIGUOUS"] \
            or not a.flags["WRITEABLE"]:
        raise ValueError(f"{name} must be a writable C-contiguous {np.dtype(dtype)} array of shape {tuple(shape)}")
    return a


def _q_init_arg(q_init: torch.Tensor, n: int, dt, dev) -> Tuple[torch.Tensor, int]:
    """q_init of the device IK entry points and its row stride: (7,) is broadcast to every query (stride 0), (N, 7)
    gives one start per query (stride 7)."""
    if q_init.dim() == 1:
        if q_init.shape != (7,):
            raise ValueError("broadcast q_init must have shape (7,)")
        return q_init.to(device=dev, dtype=dt).contiguous(), 0
    q_init = _check_cuda("q_init", q_init, dt, (7,))
    if q_init.shape[0] != n:
        raise ValueError("q_init and the targets disagree on N")
    return q_init, 7


def _multistart_inputs(seeds, n: int, dt, dev, counters, restart_stats):
    """The seed table (K, 7) of a multistart call in dt on dev, its scratch and its attempt output (uint8[N])."""
    seeds = torch.as_tensor(seeds).to(device=dev, dtype=dt).reshape(-1, 7).contiguous()
    if seeds.shape[0] > 255:
        raise ValueError(f"at most 255 seeds, got {seeds.shape[0]}")
    for name, t, m in (("counters", counters, 4), ("restart_stats", restart_stats, 3)):
        if t is not None and (t.dtype != torch.int64 or t.numel() < m or not t.is_cuda):
            raise ValueError(f"{name} must be a CUDA int64 tensor with >= {m} elements")
    nbytes = ctypes.c_int64()
    _lib.check(_lib.load().pnp_ik_multistart_scratch_bytes(n, ctypes.byref(nbytes)), "pnp_ik_multistart_scratch_bytes")
    with torch.cuda.device(dev):
        scratch = torch.empty(((nbytes.value + 15) // 16, 4), dtype=torch.int32, device=dev)
        attempt = torch.empty((n,), dtype=torch.uint8, device=dev)
    return seeds, scratch, attempt


# ---------------------------------------------------------------------------------------------
# FK + Jacobian
# ---------------------------------------------------------------------------------------------
def fk_jac(q: torch.Tensor, want_quat=True, want_jac=True, kinematics="auto"):
    """q[N,7] (cuda, f32|f64) -> pos[N,3], quat[N,4] wxyz | None, jac[N,6,7] | None."""
    lib = _lib.load()
    if q.dtype not in (torch.float32, torch.float64):
        raise ValueError("q must be float32 or float64")
    q = _check_cuda("q", q, q.dtype, (7,))
    n = q.shape[0]
    pos = torch.empty((n, 3), dtype=q.dtype, device=q.device)
    quat = torch.empty((n, 4), dtype=q.dtype, device=q.device) if want_quat else None
    jac = torch.empty((n, 6, 7), dtype=q.dtype, device=q.device) if want_jac else None
    fn = lib.pnp_fk_jac_f32 if q.dtype == torch.float32 else lib.pnp_fk_jac_f64
    with torch.cuda.device(q.device):
        _lib.check(fn(_ptr(q), n, _ptr(pos), _ptr(quat), _ptr(jac), KINEMATICS[kinematics], _stream()), "pnp_fk_jac")
    return pos, quat, jac


# ---------------------------------------------------------------------------------------------
# batched IK
# ---------------------------------------------------------------------------------------------
class BatchIKResult:
    """Batched IKResult (ik_solver.py:16-24): same fields, one row per query (device tensors).

    With the packed kernel ``q`` / ``final_pos`` / ``pos_error`` are views into the two output
    buffers and ``iterations`` / ``converged`` / ``success`` are decoded lazily from the packed
    word (iterations | flags << 24) on first access, so a solve launches exactly one kernel."""

    def __init__(self, success=None, q=None, final_pos=None, pos_error=None, iterations=None, converged=None,
                 counters=None, word=None, attempt=None):
        self.q, self.final_pos, self.pos_error, self.counters = q, final_pos, pos_error, counters
        self.attempt = attempt  # ik_solve_multistart: uint8[N], the attempt each row is the result of (0 = from q_init)
        self._success, self._iterations, self._converged, self._word = success, iterations, converged, word

    @property
    def iterations(self):
        if self._iterations is None:
            self._iterations = self._word & 0xFFFFFF
        return self._iterations

    @property
    def converged(self):
        if self._converged is None:
            self._converged = (self._word & (1 << 24)) != 0
        return self._converged

    @property
    def success(self):
        if self._success is None:
            self._success = (self._word & (2 << 24)) != 0
        return self._success

    def __len__(self) -> int:
        return int(self.q.shape[0])


class HostIKResult(dict):
    """Host-side result of ik_solve_host: a dict whose derived entries (iterations, flags,
    converged, success) are decoded from the packed word only when first asked for."""

    def __missing__(self, key):
        if dict.__contains__(self, "aux4"):
            word = dict.__getitem__(self, "aux4")[:, 3].view(np.int32)
        else:  # compact records: the word is the 8th column of q8
            word = dict.__getitem__(self, "q8")[:, 7].view(np.int32)
        if key == "iterations":
            val = word & 0xFFFFFF
        elif key == "flags":
            val = (word >> 24).astype(np.uint8)
        elif key == "converged":
            val = (word & (1 << 24)) != 0
        elif key == "success":
            val = (word & (2 << 24)) != 0
        else:
            raise KeyError(key)
        self[key] = val
        return val


def unpack_ik(out_q8, out_aux4):
    """Views into the packed IK outputs (torch tensors or NumPy arrays alike):
    q[N,7], pos_error[N], final_pos[N,3], packed word[N] int32 (iterations | flags << 24)."""
    word = out_aux4[:, 3].view(torch.int32) if isinstance(out_aux4, torch.Tensor) else out_aux4[:, 3].view(np.int32)
    return out_q8[:, :7], out_q8[:, 7], out_aux4[:, :3], word


def ik_solve(targets: torch.Tensor, q_init: torch.Tensor, params: PnpIkParams, counters: Optional[torch.Tensor] = None,
             packed: Optional[bool] = None, out_q8: Optional[torch.Tensor] = None,
             out_aux4: Optional[torch.Tensor] = None, compact: bool = False) -> BatchIKResult:
    """Device path: targets[N,3], q_init[N,7] or [7] (cuda, same float dtype).

    float32 uses the packed-output kernel (pnp_ik_solve_packed_f32) by default: the result fields
    are views into two [N,8] / [N,4] buffers.  ``packed=False`` selects the separate-array entry
    point (pnp_ik_solve_f32); float64 always uses separate arrays.  ``compact=True`` (float32) writes
    one 32-byte record per query - q, iterations, converged, success; ``final_pos`` / ``pos_error`` are None."""
    lib = _lib.load()
    dt = targets.dtype
    if dt not in (torch.float32, torch.float64):
        raise ValueError("targets must be float32 or float64")
    targets = _check_cuda("targets", targets, dt, (3,))
    n = targets.shape[0]
    dev = targets.device
    q_init, stride = _q_init_arg(q_init, n, dt, dev)
    if counters is not None and (counters.dtype != torch.int64 or counters.numel() < 4 or not counters.is_cuda):
        raise ValueError("counters must be a CUDA int64 tensor with >= 4 elements")
    if compact:
        if dt != torch.float32 or packed is False:
            raise ValueError("compact outputs exist for float32 only (and exclude packed=False)")
        packed = True
    if packed is None:
        packed = dt == torch.float32
    if packed and dt != torch.float32:
        raise ValueError("packed outputs exist for float32 only")
    with torch.cuda.device(dev):
        if packed:
            q8 = _check_out("out_q8", out_q8, (n, 8), dt, dev) if out_q8 is not None else torch.empty((n, 8), dtype=dt, device=dev)
            if compact:
                _lib.check(
                    lib.pnp_ik_solve_compact_f32(_ptr(targets), _ptr(q_init), stride, n, ctypes.byref(params), _ptr(q8),
                                                 _ptr(counters), _stream()),
                    "pnp_ik_solve_compact",
                )
                return BatchIKResult(q=q8[:, :7], word=q8[:, 7].view(torch.int32), counters=counters)
            aux = _check_out("out_aux4", out_aux4, (n, 4), dt, dev) if out_aux4 is not None else torch.empty((n, 4), dtype=dt, device=dev)
            _lib.check(
                lib.pnp_ik_solve_packed_f32(_ptr(targets), _ptr(q_init), stride, n, ctypes.byref(params), _ptr(q8),
                                            _ptr(aux), _ptr(counters), _stream()),
                "pnp_ik_solve_packed",
            )
            q, err, fpos, word = unpack_ik(q8, aux)
            return BatchIKResult(q=q, final_pos=fpos, pos_error=err, word=word, counters=counters)
        else:
            q = torch.empty((n, 7), dtype=dt, device=dev)
            fpos = torch.empty((n, 3), dtype=dt, device=dev)
            err = torch.empty((n,), dtype=dt, device=dev)
            iters = torch.empty((n,), dtype=torch.int32, device=dev)
            flags = torch.empty((n,), dtype=torch.uint8, device=dev)
            fn = lib.pnp_ik_solve_f32 if dt == torch.float32 else lib.pnp_ik_solve_f64
            _lib.check(
                fn(_ptr(targets), _ptr(q_init), stride, n, ctypes.byref(params), _ptr(q), _ptr(fpos), _ptr(err),
                   _ptr(iters), _ptr(flags), _ptr(counters), _stream()),
                "pnp_ik_solve",
            )
    return BatchIKResult(
        success=(flags & 2) != 0, q=q, final_pos=fpos, pos_error=err, iterations=iters,
        converged=(flags & 1) != 0, counters=counters,
    )


def ik_restart_seeds(k: int, lower=None, upper=None, seed: int = 0, dtype=torch.float32, device="cuda") -> torch.Tensor:
    """A seed table for ik_solve_multistart: k joint configurations ~ U(lower, upper), shape (k, 7).

    Drawn from a CPU ``torch.Generator`` and then moved to ``device``, so a seed gives the same table on every device.
    ``lower`` / ``upper`` default to the joint limits of the tree set_tree last uploaded to the current device (a
    JacobianIKController uploads its model's tree when it is made), so that the default seeds lie inside the limits the
    solver clamps to; before any upload, and without a CUDA device, they are the packaged tree's."""
    if lower is None or upper is None:
        hit = _uploaded_obj.get(torch.cuda.current_device()) if _uploaded_obj and torch.cuda.is_available() else None
        t = hit[0] if hit is not None else KinematicTree.from_mjcf()
        lower = t.lower if lower is None else lower
        upper = t.upper if upper is None else upper
    from .synthetic import random_joint_configs

    return random_joint_configs(int(k), lower, upper, seed=seed, device="cpu", dtype=torch.float64).to(
        device=device, dtype=dtype).contiguous()


def ik_solve_multistart(targets: torch.Tensor, q_init: torch.Tensor, seeds: torch.Tensor, params: PnpIkParams,
                        counters: Optional[torch.Tensor] = None, restart_stats: Optional[torch.Tensor] = None,
                        packed: Optional[bool] = None) -> BatchIKResult:
    """ik_solve, then every query it did not solve is solved again from the rows of ``seeds`` (K, 7), in order, until
    one succeeds (pnp_ik_solve_multistart_*).  Each row of the result is, bit for bit, the plain ik_solve of that target
    from the start ``result.attempt`` names (0 = q_init, k = seeds[k - 1]); rows no attempt solves keep attempt 0.

    ``counters`` (int64[4]) accumulates over the returned rows like ik_solve's; ``restart_stats`` (int64[3])
    accumulates queries restarted, queries rescued and DLS passes spent on restarts.  Same layouts as ik_solve
    (packed float32 by default, ``packed=False`` / float64: separate arrays).  Never synchronises."""
    lib = _lib.load()
    dt = targets.dtype
    if dt not in (torch.float32, torch.float64):
        raise ValueError("targets must be float32 or float64")
    targets = _check_cuda("targets", targets, dt, (3,))
    n = targets.shape[0]
    dev = targets.device
    q_init, stride = _q_init_arg(q_init, n, dt, dev)
    if packed is None:
        packed = dt == torch.float32
    if packed and dt != torch.float32:
        raise ValueError("packed outputs exist for float32 only")
    seeds, scratch, attempt = _multistart_inputs(seeds, n, dt, dev, counters, restart_stats)
    k = seeds.shape[0]
    with torch.cuda.device(dev):
        if packed:
            q8 = torch.empty((n, 8), dtype=dt, device=dev)
            aux = torch.empty((n, 4), dtype=dt, device=dev)
            _lib.check(
                lib.pnp_ik_solve_multistart_packed_f32(_ptr(targets), _ptr(q_init), stride, n, _ptr(seeds), k,
                                                       ctypes.byref(params), _ptr(q8), _ptr(aux), _ptr(attempt),
                                                       _ptr(counters), _ptr(restart_stats), _ptr(scratch), _stream()),
                "pnp_ik_solve_multistart_packed",
            )
            q, err, fpos, word = unpack_ik(q8, aux)
            return BatchIKResult(q=q, final_pos=fpos, pos_error=err, word=word, counters=counters, attempt=attempt)
        q = torch.empty((n, 7), dtype=dt, device=dev)
        fpos = torch.empty((n, 3), dtype=dt, device=dev)
        err = torch.empty((n,), dtype=dt, device=dev)
        iters = torch.empty((n,), dtype=torch.int32, device=dev)
        flags = torch.empty((n,), dtype=torch.uint8, device=dev)
        fn = lib.pnp_ik_solve_multistart_f32 if dt == torch.float32 else lib.pnp_ik_solve_multistart_f64
        _lib.check(
            fn(_ptr(targets), _ptr(q_init), stride, n, _ptr(seeds), k, ctypes.byref(params), _ptr(q), _ptr(fpos),
               _ptr(err), _ptr(iters), _ptr(flags), _ptr(attempt), _ptr(counters), _ptr(restart_stats), _ptr(scratch),
               _stream()),
            "pnp_ik_solve_multistart",
        )
    return BatchIKResult(
        success=(flags & 2) != 0, q=q, final_pos=fpos, pos_error=err, iterations=iters,
        converged=(flags & 1) != 0, counters=counters, attempt=attempt,
    )


def ik_waypoints(q_start: torch.Tensor, goal: torch.Tensor, n_steps: int, params: PnpIkParams,
                 step_size: float = 0.01, counters: Optional[torch.Tensor] = None):
    """cfg4: per-env warm-started waypoint sequences (float32 device tensors)."""
    lib = _lib.load()
    q_start = _check_cuda("q_start", q_start, torch.float32, (7,))
    goal = _check_cuda("goal", goal, torch.float32, (3,))
    n = q_start.shape[0]
    if goal.shape[0] != n:
        raise ValueError("q_start and goal disagree on N")
    dev = q_start.device
    q = torch.empty((n, 7), dtype=torch.float32, device=dev)
    pos = torch.empty((n, 3), dtype=torch.float32, device=dev)
    acc = torch.empty((n,), dtype=torch.int32, device=dev)
    its = torch.empty((n,), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(
            lib.pnp_ik_waypoints_f32(_ptr(q_start), _ptr(goal), n, int(n_steps), float(step_size),
                                     ctypes.byref(params), _ptr(q), _ptr(pos), _ptr(acc), _ptr(its),
                                     _ptr(counters), _stream()),
            "pnp_ik_waypoints",
        )
    return dict(q=q, pos=pos, n_accepted=acc, iters_total=its)


def ik_pose_solve(target_pos: torch.Tensor, target_quat: torch.Tensor, q_init: torch.Tensor, params: PnpIkParams,
                  rot_thresh: float = 1e-2, rot_weight: float = 1.0, counters: Optional[torch.Tensor] = None) -> dict:
    """Pose-mode IK (extension): target_pos[N,3], target_quat[N,4] wxyz, q_init[N,7] or [7]."""
    lib = _lib.load()
    dt = target_pos.dtype
    if dt not in (torch.float32, torch.float64):
        raise ValueError("target_pos must be float32 or float64")
    target_pos = _check_cuda("target_pos", target_pos, dt, (3,))
    target_quat = _check_cuda("target_quat", target_quat, dt, (4,))
    n = target_pos.shape[0]
    if target_quat.shape[0] != n:
        raise ValueError("target_pos and target_quat disagree on N")
    dev = target_pos.device
    q_init, stride = _q_init_arg(q_init, n, dt, dev)
    q = torch.empty((n, 7), dtype=dt, device=dev)
    fpos = torch.empty((n, 3), dtype=dt, device=dev)
    fquat = torch.empty((n, 4), dtype=dt, device=dev)
    perr = torch.empty((n,), dtype=dt, device=dev)
    rerr = torch.empty((n,), dtype=dt, device=dev)
    iters = torch.empty((n,), dtype=torch.int32, device=dev)
    flags = torch.empty((n,), dtype=torch.uint8, device=dev)
    fn = lib.pnp_ik_pose_solve_f32 if dt == torch.float32 else lib.pnp_ik_pose_solve_f64
    with torch.cuda.device(dev):
        _lib.check(
            fn(_ptr(target_pos), _ptr(target_quat), _ptr(q_init), stride, n, ctypes.byref(params), float(rot_thresh),
               float(rot_weight), _ptr(q), _ptr(fpos), _ptr(fquat), _ptr(perr), _ptr(rerr), _ptr(iters), _ptr(flags),
               _ptr(counters), _stream()),
            "pnp_ik_pose_solve",
        )
    return dict(q=q, final_pos=fpos, final_quat=fquat, pos_error=perr, rot_error=rerr, iterations=iters,
                converged=(flags & 1) != 0, success=(flags & 2) != 0)


def ik_pose_solve_multistart(target_pos: torch.Tensor, target_quat: torch.Tensor, q_init: torch.Tensor,
                             seeds: torch.Tensor, params: PnpIkParams, rot_thresh: float = 1e-2, rot_weight: float = 1.0,
                             counters: Optional[torch.Tensor] = None,
                             restart_stats: Optional[torch.Tensor] = None) -> dict:
    """ik_pose_solve, then every query it did not solve is solved again from the rows of ``seeds`` (K, 7), in order,
    until one succeeds (pnp_ik_pose_solve_multistart_*).  Each row of the result is, bit for bit, the plain
    ik_pose_solve of that target from the start ``attempt`` names (0 = q_init, k = seeds[k - 1]); rows no attempt
    solves keep attempt 0.  Returns ik_pose_solve's dict plus ``attempt`` (uint8[N]).

    ``counters`` (int64[4]) accumulates over the returned rows like ik_pose_solve's; ``restart_stats`` (int64[3])
    accumulates queries restarted, queries rescued and DLS passes spent on restarts.  Never synchronises."""
    lib = _lib.load()
    dt = target_pos.dtype
    if dt not in (torch.float32, torch.float64):
        raise ValueError("target_pos must be float32 or float64")
    target_pos = _check_cuda("target_pos", target_pos, dt, (3,))
    target_quat = _check_cuda("target_quat", target_quat, dt, (4,))
    n = target_pos.shape[0]
    if target_quat.shape[0] != n:
        raise ValueError("target_pos and target_quat disagree on N")
    dev = target_pos.device
    q_init, stride = _q_init_arg(q_init, n, dt, dev)
    seeds, scratch, attempt = _multistart_inputs(seeds, n, dt, dev, counters, restart_stats)
    k = seeds.shape[0]
    fn = lib.pnp_ik_pose_solve_multistart_f32 if dt == torch.float32 else lib.pnp_ik_pose_solve_multistart_f64
    with torch.cuda.device(dev):
        q = torch.empty((n, 7), dtype=dt, device=dev)
        fpos = torch.empty((n, 3), dtype=dt, device=dev)
        fquat = torch.empty((n, 4), dtype=dt, device=dev)
        perr = torch.empty((n,), dtype=dt, device=dev)
        rerr = torch.empty((n,), dtype=dt, device=dev)
        iters = torch.empty((n,), dtype=torch.int32, device=dev)
        flags = torch.empty((n,), dtype=torch.uint8, device=dev)
        _lib.check(
            fn(_ptr(target_pos), _ptr(target_quat), _ptr(q_init), stride, n, _ptr(seeds), k, ctypes.byref(params),
               float(rot_thresh), float(rot_weight), _ptr(q), _ptr(fpos), _ptr(fquat), _ptr(perr), _ptr(rerr),
               _ptr(iters), _ptr(flags), _ptr(attempt), _ptr(counters), _ptr(restart_stats), _ptr(scratch),
               _stream()),
            "pnp_ik_pose_solve_multistart",
        )
    return dict(q=q, final_pos=fpos, final_quat=fquat, pos_error=perr, rot_error=rerr, iterations=iters,
                converged=(flags & 1) != 0, success=(flags & 2) != 0, attempt=attempt)


def _axis_inputs(target_pos, target_axis, tool_axis):
    dt = target_pos.dtype
    if dt not in (torch.float32, torch.float64):
        raise ValueError("target_pos must be float32 or float64")
    target_pos = _check_cuda("target_pos", target_pos, dt, (3,))
    target_axis = _check_cuda("target_axis", target_axis, dt, (3,))
    if target_axis.shape[0] != target_pos.shape[0]:
        raise ValueError("target_pos and target_axis disagree on N")
    tool = np.asarray(tool_axis, dtype=np.float64).reshape(-1)
    if tool.shape != (3,):
        raise ValueError("tool_axis must have 3 components")
    return target_pos, target_axis, (ctypes.c_double * 3)(*tool.tolist())


def _axis_outputs(n, dt, dev):
    return dict(q=torch.empty((n, 7), dtype=dt, device=dev), final_pos=torch.empty((n, 3), dtype=dt, device=dev),
                final_axis=torch.empty((n, 3), dtype=dt, device=dev), final_quat=torch.empty((n, 4), dtype=dt, device=dev),
                pos_error=torch.empty((n,), dtype=dt, device=dev), axis_error=torch.empty((n,), dtype=dt, device=dev),
                iterations=torch.empty((n,), dtype=torch.int32, device=dev),
                flags=torch.empty((n,), dtype=torch.uint8, device=dev))


def _axis_result(o, **extra):
    flags = o.pop("flags")
    return dict(o, converged=(flags & 1) != 0, success=(flags & 2) != 0, **extra)


def _axis_entry(lib, dt, multistart, rot_thresh, cone_angle, rot_weight):
    """(entry point, its name, its arguments after tool_axis up to q_out): the axis solve's, or the cone solve's when
    cone_angle is not None."""
    name = "pnp_ik_axis_solve" if cone_angle is None else "pnp_ik_axis_cone_solve"
    name += ("_multistart" if multistart else "") + ("_f32" if dt == torch.float32 else "_f64")
    angles = (float(rot_thresh),) if cone_angle is None else (float(rot_thresh), float(cone_angle))
    return getattr(lib, name), name, (*angles, float(rot_weight))


def ik_axis_solve(target_pos: torch.Tensor, target_axis: torch.Tensor, q_init: torch.Tensor, params: PnpIkParams,
                  tool_axis=(0.0, 0.0, 1.0), rot_thresh: float = 1e-2, rot_weight: float = 1.0,
                  counters: Optional[torch.Tensor] = None, cone_angle: Optional[float] = None) -> dict:
    """Axis-constrained IK (extension, pnp_ik_axis_solve_*): put the site at target_pos[N,3] with its ``tool_axis``
    (site frame, (3,)) along target_axis[N,3] (world frame, any norm), the roll about that axis free.  q_init[N,7] or
    [7].  Returns q, final_pos, final_axis (the tool axis in the world frame), final_quat, pos_error, axis_error (the
    angle between final_axis and the target axis, rad), iterations, converged, success.

    ``cone_angle`` (rad, in [0, pi]): accept the tool axis anywhere within that angle of the target axis
    (pnp_ik_axis_cone_solve_*); axis_error stays the true angle.  None runs the exact axis solve."""
    lib = _lib.load()
    target_pos, target_axis, tool = _axis_inputs(target_pos, target_axis, tool_axis)
    dt, n, dev = target_pos.dtype, target_pos.shape[0], target_pos.device
    q_init, stride = _q_init_arg(q_init, n, dt, dev)
    fn, name, thr = _axis_entry(lib, dt, False, rot_thresh, cone_angle, rot_weight)
    with torch.cuda.device(dev):
        o = _axis_outputs(n, dt, dev)
        _lib.check(
            fn(_ptr(target_pos), _ptr(target_axis), _ptr(q_init), stride, n, ctypes.byref(params), tool,
               *thr, *(_ptr(t) for t in o.values()), _ptr(counters),
               _stream()),
            name[:-4],
        )
    return _axis_result(o)


def ik_axis_solve_multistart(target_pos: torch.Tensor, target_axis: torch.Tensor, q_init: torch.Tensor,
                             seeds: torch.Tensor, params: PnpIkParams, tool_axis=(0.0, 0.0, 1.0),
                             rot_thresh: float = 1e-2, rot_weight: float = 1.0, counters: Optional[torch.Tensor] = None,
                             restart_stats: Optional[torch.Tensor] = None, cone_angle: Optional[float] = None) -> dict:
    """ik_axis_solve, then every query it did not solve is solved again from the rows of ``seeds`` (K, 7), in order,
    until one succeeds (pnp_ik_axis_solve_multistart_*).  Each row of the result is, bit for bit, the plain
    ik_axis_solve of that target from the start ``attempt`` names (0 = q_init, k = seeds[k - 1]).  Returns
    ik_axis_solve's dict plus ``attempt`` (uint8[N]); ``counters`` / ``restart_stats`` as ik_pose_solve_multistart;
    ``cone_angle`` as ik_axis_solve (pnp_ik_axis_cone_solve_multistart_*).  Never synchronises."""
    lib = _lib.load()
    target_pos, target_axis, tool = _axis_inputs(target_pos, target_axis, tool_axis)
    dt, n, dev = target_pos.dtype, target_pos.shape[0], target_pos.device
    q_init, stride = _q_init_arg(q_init, n, dt, dev)
    seeds, scratch, attempt = _multistart_inputs(seeds, n, dt, dev, counters, restart_stats)
    fn, name, thr = _axis_entry(lib, dt, True, rot_thresh, cone_angle, rot_weight)
    with torch.cuda.device(dev):
        o = _axis_outputs(n, dt, dev)
        _lib.check(
            fn(_ptr(target_pos), _ptr(target_axis), _ptr(q_init), stride, n, _ptr(seeds), seeds.shape[0],
               ctypes.byref(params), tool, *thr,
               *(_ptr(t) for t in o.values()), _ptr(attempt), _ptr(counters), _ptr(restart_stats), _ptr(scratch),
               _stream()),
            name[:-4],
        )
    return _axis_result(o, attempt=attempt)


PLAN_ORDER_MIN = 1 << 16  # below this a launch has fewer envs than lanes: nothing to balance (2^14 measured slower)


def move_plan_order(q_start: torch.Tensor, target: torch.Tensor, kinematics="auto") -> torch.Tensor:
    """order[N] (int32 bit pattern of uint32): env indices by descending |target - FK(q_start)|, i.e. longest
    MoveIKSkill plans first (skills/move.py:106-137); feed to move_ik_plan(order=...)."""
    lib = _lib.load()
    dt = q_start.dtype
    if dt not in (torch.float32, torch.float64):
        raise ValueError("q_start must be float32 or float64")
    q_start = _check_cuda("q_start", q_start, dt, (7,))
    target = _check_cuda("target", target, dt, (3,))
    n = q_start.shape[0]
    if target.shape[0] != n:
        raise ValueError("q_start and target disagree on N")
    order = torch.empty((n,), dtype=torch.int32, device=q_start.device)
    fn = lib.pnp_move_plan_order_f32 if dt == torch.float32 else lib.pnp_move_plan_order_f64
    with torch.cuda.device(q_start.device):
        kin = KINEMATICS[kinematics] if isinstance(kinematics, str) else int(kinematics)
        _lib.check(fn(_ptr(q_start), _ptr(target), n, _ptr(order), kin, _stream()), "pnp_move_plan_order")
    return order


def move_plan_order_check(order: torch.Tensor) -> int:
    """Number of entries of ``order`` (int32[N], CUDA) that are outside [0, N) or repeat an earlier entry; 0 means
    a permutation (pnp_move_plan_order_check).  Synchronises to read the count."""
    lib = _lib.load()
    order = _check_cuda("order", order, torch.int32, ())
    n = order.shape[0]
    dev = order.device
    bitmap = torch.empty(((n + 31) // 32,), dtype=torch.int32, device=dev)
    bad = torch.empty((1,), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.pnp_move_plan_order_check(_ptr(order), n, _ptr(bitmap), _ptr(bad), _stream()), "pnp_move_plan_order_check")
    return int(bad.item())


def move_ik_plan(q_start: torch.Tensor, target: torch.Tensor, params: PnpIkParams, pos_thresh: float = 0.01,
                 max_traj_points: int = 200, step_size: float = 0.01, max_outer: int = 0, traj_cap: int = 256,
                 counters: Optional[torch.Tensor] = None, order="auto", out: Optional[dict] = None,
                 validate_order: bool = True):
    """Batched MoveIKSkill.reset planner (skills/move.py:76-191): CUDA tensors f32 or f64.

    ``order``: "auto" (longest plans first from N = 2^16 up, see move_plan_order), None (index order) or a
    tensor from move_plan_order; it changes the schedule, never the result (a caller-made tensor is checked to be a
    permutation unless ``validate_order=False``).  ``out``: the dict of a previous
    call with the same N / traj_cap / dtype, whose buffers are then reused (trajectory rows beyond traj_len
    keep their old contents); fresh trajectory storage is zero-filled.

    Returns dict(traj[N,traj_cap,3], traj_len[N], q_final[N,7], n_solves[N], status[N]).  With ``order="auto"`` on float32
    batches of >= 2^16 envs the call goes through pnp_move_ik_plan_sorted_f32 (inputs gathered in plan order) and the dict
    also carries ``_scratch48``, the [N,12] int32 scratch of that call, so that ``out=`` reuses it as well."""
    lib = _lib.load()
    dt = q_start.dtype
    if dt not in (torch.float32, torch.float64):
        raise ValueError("q_start must be float32 or float64")
    q_start = _check_cuda("q_start", q_start, dt, (7,))
    target = _check_cuda("target", target, dt, (3,))
    n = q_start.shape[0]
    if target.shape[0] != n:
        raise ValueError("q_start and target disagree on N")
    dev = q_start.device
    mp = PnpMoveParams(float(pos_thresh), float(step_size), int(max_traj_points), int(max_outer), int(traj_cap), 0)
    if out is not None:
        traj, tlen, qf, solves, status = (out[k] for k in ("traj", "traj_len", "q_final", "n_solves", "status"))
        if (traj.shape != (n, traj_cap, 3) or traj.dtype != dt or traj.device != dev or not traj.is_contiguous()
                or tlen.shape != (n,) or qf.shape != (n, 7) or qf.dtype != dt or solves.shape != (n,) or status.shape != (n,)):
            raise ValueError("out does not match N / traj_cap / dtype / device of this call")
    else:
        traj = torch.zeros((n, traj_cap, 3), dtype=dt, device=dev)
        tlen = torch.empty((n,), dtype=torch.int32, device=dev)
        qf = torch.empty((n, 7), dtype=dt, device=dev)
        solves = torch.empty((n,), dtype=torch.int32, device=dev)
        status = torch.empty((n,), dtype=torch.int32, device=dev)
    if isinstance(order, str):
        if order != "auto":
            raise ValueError("order must be 'auto', None or a tensor from move_plan_order")
        order = None
        if n >= PLAN_ORDER_MIN and dt == torch.float32:
            # longest plan first with gathered inputs: 48 B of scratch per env for the call to fill and read
            scratch = out.get("_scratch48") if out is not None else None
            if scratch is None or scratch.shape != (n, 12) or scratch.device != dev:
                scratch = torch.empty((n, 12), dtype=torch.int32, device=dev)
            with torch.cuda.device(dev):
                _lib.check(
                    lib.pnp_move_ik_plan_sorted_f32(_ptr(q_start), _ptr(target), _ptr(scratch), n, ctypes.byref(mp), ctypes.byref(params),
                                                    _ptr(traj), _ptr(tlen), _ptr(qf), _ptr(solves), _ptr(status), _ptr(counters), _stream()),
                    "pnp_move_ik_plan_sorted",
                )
            return dict(traj=traj, traj_len=tlen, q_final=qf, n_solves=solves, status=status, _scratch48=scratch)
        if n >= PLAN_ORDER_MIN:  # scratch for the call to fill and use (PnpMoveParams.compute_order)
            order = torch.empty((n,), dtype=torch.int32, device=dev)
            mp.compute_order = 1
    elif order is not None:
        order = _check_cuda("order", order, torch.int32, ())
        if order.shape[0] != n:
            raise ValueError("order disagrees with q_start on N")
        if validate_order:  # one pass over a bitmap; costs a device->host read of one word
            bad = move_plan_order_check(order)
            if bad:
                raise ValueError(f"order is not a permutation of [0, {n}): {bad} entries are out of range or repeated")
    fn = lib.pnp_move_ik_plan_ordered_f32 if dt == torch.float32 else lib.pnp_move_ik_plan_ordered_f64
    with torch.cuda.device(dev):
        _lib.check(
            fn(_ptr(q_start), _ptr(target), _ptr(order), n, ctypes.byref(mp), ctypes.byref(params), _ptr(traj), _ptr(tlen),
               _ptr(qf), _ptr(solves), _ptr(status), _ptr(counters), _stream()),
            "pnp_move_ik_plan",
        )
    return dict(traj=traj, traj_len=tlen, q_final=qf, n_solves=solves, status=status)


def move_ik_plan_pose(q_start: torch.Tensor, goal_pos: torch.Tensor, goal_quat: torch.Tensor, params: PnpIkParams,
                      pos_thresh: float = 0.01, rot_thresh: float = 0.05, step_size: float = 0.01, rot_step: float = 0.05,
                      ik_rot_thresh: float = 1e-2, rot_weight: float = 1.0, max_traj_points: int = 200,
                      traj_cap: Optional[int] = None, want_q_traj: bool = True,
                      counters: Optional[torch.Tensor] = None) -> dict:
    """Pose-mode move planner (pnp_move_ik_plan_pose_*, extension): plan N moves to a goal position AND orientation,
    every waypoint a solved pose (oracle/move_pose_oracle.py states the semantics).  q_start[N,7], goal_pos[N,3],
    goal_quat[N,4] wxyz, CUDA float32 or float64.  ``params`` is the IK of every waypoint solve; ``pos_thresh`` must be
    >= params.pos_thresh and ``rot_thresh`` >= ``ik_rot_thresh``.  traj_cap defaults to max_traj_points + 1 (never
    overflows).  Never synchronises.

    Returns dict(pos_traj[N,cap,3], quat_traj[N,cap,4], q_traj[N,cap,7] (None unless want_q_traj), traj_len[N],
    q_final[N,7], n_solves[N], status[N]); rows past traj_len are zero."""
    lib = _lib.load()
    dt = q_start.dtype
    if dt not in (torch.float32, torch.float64):
        raise ValueError("q_start must be float32 or float64")
    q_start = _check_cuda("q_start", q_start, dt, (7,))
    goal_pos = _check_cuda("goal_pos", goal_pos, dt, (3,))
    goal_quat = _check_cuda("goal_quat", goal_quat, dt, (4,))
    n = q_start.shape[0]
    if goal_pos.shape[0] != n or goal_quat.shape[0] != n:
        raise ValueError("q_start, goal_pos and goal_quat disagree on N")
    if counters is not None and (counters.dtype != torch.int64 or counters.numel() < 4 or not counters.is_cuda):
        raise ValueError("counters must be a CUDA int64 tensor with >= 4 elements")
    cap = int(traj_cap) if traj_cap is not None else int(max_traj_points) + 1
    mp = _lib.PnpMovePoseParams(float(pos_thresh), float(rot_thresh), float(step_size), float(rot_step),
                                float(ik_rot_thresh), float(rot_weight), int(max_traj_points), cap)
    dev = q_start.device
    with torch.cuda.device(dev):
        pos_traj = torch.zeros((n, max(cap, 0), 3), dtype=dt, device=dev)
        quat_traj = torch.zeros((n, max(cap, 0), 4), dtype=dt, device=dev)
        q_traj = torch.zeros((n, max(cap, 0), 7), dtype=dt, device=dev) if want_q_traj else None
        tlen = torch.empty((n,), dtype=torch.int32, device=dev)
        qf = torch.empty((n, 7), dtype=dt, device=dev)
        solves = torch.empty((n,), dtype=torch.int32, device=dev)
        status = torch.empty((n,), dtype=torch.int32, device=dev)
        fn = lib.pnp_move_ik_plan_pose_f32 if dt == torch.float32 else lib.pnp_move_ik_plan_pose_f64
        _lib.check(
            fn(_ptr(q_start), _ptr(goal_pos), _ptr(goal_quat), n, ctypes.byref(mp), ctypes.byref(params), _ptr(pos_traj),
               _ptr(quat_traj), _ptr(q_traj), _ptr(tlen), _ptr(qf), _ptr(solves), _ptr(status), _ptr(counters),
               _stream()),
            "pnp_move_ik_plan_pose",
        )
    return dict(pos_traj=pos_traj, quat_traj=quat_traj, q_traj=q_traj, traj_len=tlen, q_final=qf, n_solves=solves,
                status=status)


def move_ik_plan_axis(q_start: torch.Tensor, goal_pos: torch.Tensor, goal_axis: torch.Tensor, params: PnpIkParams,
                      tool_axis=(0.0, 0.0, 1.0), pos_thresh: float = 0.01, rot_thresh: float = 0.05,
                      step_size: float = 0.01, rot_step: float = 0.05, ik_rot_thresh: float = 1e-2,
                      rot_weight: float = 1.0, max_traj_points: int = 200, traj_cap: Optional[int] = None,
                      want_q_traj: bool = True, counters: Optional[torch.Tensor] = None) -> dict:
    """Axis-mode move planner (pnp_move_ik_plan_axis_*, extension): plan N moves to a goal position and a goal
    direction goal_axis[N,3] (world frame, any norm) of the site-frame ``tool_axis``, the roll about it free, every
    waypoint a solved axis task (oracle/move_axis_oracle.py states the semantics).  rot_thresh, rot_step, ik_rot_thresh
    and rot_weight apply to the axis angle.  Otherwise as move_ik_plan_pose: ``pos_thresh`` >= params.pos_thresh,
    ``rot_thresh`` >= ``ik_rot_thresh``, traj_cap defaults to max_traj_points + 1.  Never synchronises.

    Returns dict(pos_traj[N,cap,3], axis_traj[N,cap,3] (the world tool axis), quat_traj[N,cap,4], q_traj[N,cap,7] (None
    unless want_q_traj), traj_len[N], q_final[N,7], n_solves[N], status[N]); rows past traj_len are zero."""
    lib = _lib.load()
    dt = q_start.dtype
    if dt not in (torch.float32, torch.float64):
        raise ValueError("q_start must be float32 or float64")
    q_start = _check_cuda("q_start", q_start, dt, (7,))
    goal_pos, goal_axis, tool = _axis_inputs(goal_pos, goal_axis, tool_axis)
    n = q_start.shape[0]
    if goal_pos.dtype != dt or goal_pos.shape[0] != n:
        raise ValueError("q_start, goal_pos and goal_axis disagree on N or dtype")
    if counters is not None and (counters.dtype != torch.int64 or counters.numel() < 4 or not counters.is_cuda):
        raise ValueError("counters must be a CUDA int64 tensor with >= 4 elements")
    cap = int(traj_cap) if traj_cap is not None else int(max_traj_points) + 1
    mp = _lib.PnpMovePoseParams(float(pos_thresh), float(rot_thresh), float(step_size), float(rot_step),
                                float(ik_rot_thresh), float(rot_weight), int(max_traj_points), cap)
    dev = q_start.device
    with torch.cuda.device(dev):
        pos_traj = torch.zeros((n, max(cap, 0), 3), dtype=dt, device=dev)
        axis_traj = torch.zeros((n, max(cap, 0), 3), dtype=dt, device=dev)
        quat_traj = torch.zeros((n, max(cap, 0), 4), dtype=dt, device=dev)
        q_traj = torch.zeros((n, max(cap, 0), 7), dtype=dt, device=dev) if want_q_traj else None
        tlen = torch.empty((n,), dtype=torch.int32, device=dev)
        qf = torch.empty((n, 7), dtype=dt, device=dev)
        solves = torch.empty((n,), dtype=torch.int32, device=dev)
        status = torch.empty((n,), dtype=torch.int32, device=dev)
        fn = lib.pnp_move_ik_plan_axis_f32 if dt == torch.float32 else lib.pnp_move_ik_plan_axis_f64
        _lib.check(
            fn(_ptr(q_start), _ptr(goal_pos), _ptr(goal_axis), n, ctypes.byref(mp), ctypes.byref(params), tool,
               _ptr(pos_traj), _ptr(axis_traj), _ptr(quat_traj), _ptr(q_traj), _ptr(tlen), _ptr(qf), _ptr(solves),
               _ptr(status), _ptr(counters), _stream()),
            "pnp_move_ik_plan_axis",
        )
    return dict(pos_traj=pos_traj, axis_traj=axis_traj, quat_traj=quat_traj, q_traj=q_traj, traj_len=tlen, q_final=qf,
                n_solves=solves, status=status)


# ---------------------------------------------------------------------------------------------
# reward
# ---------------------------------------------------------------------------------------------
def reward(ag, dg, ee_pos, ee_quat, width, task_index, params: PnpRewardParams, want_success=True,
           counters: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None,
           out_success: Optional[torch.Tensor] = None):
    """Device path: rows as CUDA tensors (f32 or f64 storage), reward float32[N]."""
    lib = _lib.load()
    dt = ag.dtype
    if dt not in (torch.float32, torch.float64):
        raise ValueError("achieved_goal must be float32 or float64")
    ag = _check_cuda("achieved_goal", ag, dt, (3,))
    dg = _check_cuda("desired_goal", dg, dt, (3,))
    ee_pos = _check_cuda("ee_pos", ee_pos, dt, (3,))
    ee_quat = _check_cuda("ee_quat", ee_quat, dt, (4,))
    width = _check_cuda("fingers_width", width, dt, ())
    task_index = _check_cuda("task_index", task_index, torch.int32, ())
    n = ag.shape[0]
    for name, t in (("desired_goal", dg), ("ee_pos", ee_pos), ("ee_quat", ee_quat), ("fingers_width", width),
                    ("task_index", task_index)):
        if t.shape[0] != n:
            raise ValueError(f"{name} disagrees with achieved_goal on N")
    dev = ag.device
    rew = _check_out("out", out, (n,), torch.float32, dev) if out is not None else torch.empty((n,), dtype=torch.float32, device=dev)
    succ = _check_out("out_success", out_success, (n,), torch.float32, dev) if out_success is not None else (
        torch.empty((n,), dtype=torch.float32, device=dev) if want_success else None)
    fn = lib.pnp_reward_f32 if dt == torch.float32 else lib.pnp_reward_f64
    with torch.cuda.device(dev):
        _lib.check(
            fn(_ptr(ag), _ptr(dg), _ptr(ee_pos), _ptr(ee_quat), _ptr(width), _ptr(task_index), n,
               ctypes.byref(params), _ptr(rew), _ptr(succ), _ptr(counters), _stream()),
            "pnp_reward",
        )
    return rew, succ


OBS_DIM = 19  # observation width with block_gripper=False (panda_env.py:297)


def get_obs(q_arm, qvel_arm, fingers, obj_pos, obj_quat, obj_vel, goal, dt: float = 0.05, kinematics="auto"):
    """Batched FrankaEnv._get_obs from kinematic state (CUDA tensors, f32 or f64).

    Returns rows[N,25] = observation[19] | achieved_goal[3] | desired_goal[3]."""
    lib = _lib.load()
    dt_ = q_arm.dtype
    if dt_ not in (torch.float32, torch.float64):
        raise ValueError("q_arm must be float32 or float64")
    q_arm = _check_cuda("q_arm", q_arm, dt_, (7,))
    n = q_arm.shape[0]
    qvel_arm = _check_cuda("qvel_arm", qvel_arm, dt_, (7,))
    fingers = _check_cuda("fingers", fingers, dt_, (2,))
    obj_pos = _check_cuda("obj_pos", obj_pos, dt_, (3,))
    obj_quat = _check_cuda("obj_quat", obj_quat, dt_, (4,))
    obj_vel = _check_cuda("obj_vel", obj_vel, dt_, (6,))
    for name, t in (("qvel_arm", qvel_arm), ("fingers", fingers), ("obj_pos", obj_pos), ("obj_quat", obj_quat),
                    ("obj_vel", obj_vel)):
        if t.shape[0] != n:
            raise ValueError(f"{name} disagrees with q_arm on N")
    if goal.dim() == 1:
        if goal.shape != (3,):
            raise ValueError("broadcast goal must have shape (3,)")
        goal, stride = goal.to(device=q_arm.device, dtype=dt_).contiguous(), 0
    else:
        goal, stride = _check_cuda("goal", goal, dt_, (3,)), 3
        if goal.shape[0] != n:
            raise ValueError("goal disagrees with q_arm on N")
    out = torch.empty((n, 25), dtype=dt_, device=q_arm.device)
    fn = lib.pnp_get_obs_f32 if dt_ == torch.float32 else lib.pnp_get_obs_f64
    with torch.cuda.device(q_arm.device):
        _lib.check(
            fn(_ptr(q_arm), _ptr(qvel_arm), _ptr(fingers), _ptr(obj_pos), _ptr(obj_quat), _ptr(obj_vel), _ptr(goal),
               stride, n, float(dt), _ptr(out), KINEMATICS[kinematics], _stream()),
            "pnp_get_obs",
        )
    return out


def normalize_params(mean, var, epsilon: float = 1e-8, clip_obs: float = 10.0) -> PnpNormalizeParams:
    """VecNormalize statistics for the 25-wide row: observation[19] | achieved_goal[3] | desired_goal[3]."""
    mean = np.asarray(mean, dtype=np.float64).reshape(-1)
    var = np.asarray(var, dtype=np.float64).reshape(-1)
    if mean.shape != (25,) or var.shape != (25,):
        raise ValueError("mean and var must have 25 entries (obs19 | ag3 | dg3)")
    p = PnpNormalizeParams()
    p.mean[:] = mean.tolist()
    p.var[:] = var.tolist()
    p.epsilon, p.clip_obs = float(epsilon), float(clip_obs)
    return p


def her_relabel(obs, next_obs, future_idx, ee_quat, task_index, params: PnpRewardParams,
                norm: Optional[PnpNormalizeParams] = None, want_success: bool = True,
                counters: Optional[torch.Tensor] = None, out_obs=None, out_next_obs=None, out_reward=None,
                future_ag: Optional[torch.Tensor] = None):
    """HER relabel + reward + optional VecNormalize over N stored transitions (CUDA float32).

    obs / next_obs: [N,25] rows (observation19 | achieved_goal3 | desired_goal3); future_idx int32[N]
    (row whose next achieved_goal becomes the goal; < 0 or >= N keeps the stored one); ee_quat[N,4];
    task_index int32[N].  ``future_ag`` [N,3] (optional): the next achieved goals as a separate table
    (SB3's ``next_observations["achieved_goal"]``); the goal gather then reads this L2-sized table instead
    of the 100-byte rows.  Returns (out_obs[N,25], out_next_obs[N,25], reward[N], is_success[N] | None)."""
    lib = _lib.load()
    obs = _check_cuda("obs", obs, torch.float32, (25,))
    next_obs = _check_cuda("next_obs", next_obs, torch.float32, (25,))
    future_idx = _check_cuda("future_idx", future_idx, torch.int32, ())
    ee_quat = _check_cuda("ee_quat", ee_quat, torch.float32, (4,))
    task_index = _check_cuda("task_index", task_index, torch.int32, ())
    n = obs.shape[0]
    if future_ag is not None:
        future_ag = _check_cuda("future_ag", future_ag, torch.float32, (3,))
    for name, t in (("next_obs", next_obs), ("future_idx", future_idx), ("ee_quat", ee_quat), ("task_index", task_index),
                    ("future_ag", future_ag)):
        if t is not None and t.shape[0] != n:
            raise ValueError(f"{name} disagrees with obs on N")
    dev = obs.device
    o = _check_out("out_obs", out_obs, (n, 25), torch.float32, dev) if out_obs is not None else torch.empty_like(obs)
    x = _check_out("out_next_obs", out_next_obs, (n, 25), torch.float32, dev) if out_next_obs is not None else torch.empty_like(next_obs)
    r = _check_out("out_reward", out_reward, (n,), torch.float32, dev) if out_reward is not None else torch.empty((n,), dtype=torch.float32, device=dev)
    sc = torch.empty((n,), dtype=torch.float32, device=dev) if want_success else None
    with torch.cuda.device(dev):
        _lib.check(
            lib.pnp_her_relabel_table_f32(_ptr(obs), _ptr(next_obs), _ptr(future_idx), _ptr(future_ag), _ptr(ee_quat),
                                          _ptr(task_index), n, ctypes.byref(params),
                                          ctypes.byref(norm) if norm is not None else None, _ptr(o), _ptr(x), _ptr(r),
                                          _ptr(sc), _ptr(counters), _stream()),
            "pnp_her_relabel",
        )
    return o, x, r, sc


def goal_distance(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    lib = _lib.load()
    a = _check_cuda("a", a, torch.float64, (3,))
    b = _check_cuda("b", b, torch.float64, (3,))
    if a.shape != b.shape:
        raise ValueError("a and b must have the same shape")
    d = torch.empty((a.shape[0],), dtype=torch.float64, device=a.device)
    with torch.cuda.device(a.device):
        _lib.check(lib.pnp_goal_distance_f64(_ptr(a), _ptr(b), a.shape[0], _ptr(d), _stream()), "pnp_goal_distance")
    return d


# ---------------------------------------------------------------------------------------------
# host-buffer path (library-owned copy/compute pipeline)
# ---------------------------------------------------------------------------------------------
def host_ctx(chunk_rows: int = 0) -> ctypes.c_void_p:
    _require_cuda()
    key = (torch.cuda.current_device(), int(chunk_rows))
    if key not in _host_ctx:
        ctx = ctypes.c_void_p()
        _lib.check(_lib.load().pnp_host_ctx_create(ctypes.byref(ctx), int(chunk_rows)), "pnp_host_ctx_create")
        _host_ctx[key] = ctx
    return _host_ctx[key]


def _np_ptr(a: Optional[np.ndarray]) -> Optional[int]:
    return None if a is None else a.ctypes.data


def _as_host(name: str, a, dtype, shape_tail) -> np.ndarray:
    if isinstance(a, torch.Tensor):
        if a.is_cuda:
            raise ValueError(f"{name}: host path got a CUDA tensor")
        a = a.numpy()
    a = np.ascontiguousarray(a, dtype=dtype)
    if a.shape[1:] != tuple(shape_tail):
        raise ValueError(f"{name} must have shape (N, {', '.join(map(str, shape_tail))}), got {a.shape}")
    return a


def ik_solve_host(targets, q_init, params: PnpIkParams, chunk_rows: int = 0, out: Optional[dict] = None,
                  packed: bool = True, compact: bool = False) -> dict:
    """Host path: NumPy / CPU-tensor inputs (float32), NumPy outputs.

    packed=True (default) goes through pnp_ik_solve_packed_host_f32: the device writes two packed
    records per query and the returned q / final_pos / pos_error / iterations are views into the
    host copies ``out["q8"]`` [N,8] and ``out["aux4"]`` [N,4] (preallocate them pinned for full
    copy/compute overlap).  compact=True (pnp_ik_solve_compact_host_f32) brings back ``out["q8"]`` only -
    q, iterations, converged, success in 32 bytes per query; final_pos / pos_error are not computed.
    packed=False uses the separate-array operator."""
    lib = _lib.load()
    targets = _as_host("targets", targets, np.float32, (3,))
    n = targets.shape[0]
    if isinstance(q_init, torch.Tensor):
        q_init = q_init.numpy()
    q_init = np.ascontiguousarray(q_init, dtype=np.float32)
    if q_init.shape == (7,):
        stride = 0
    elif q_init.shape == (n, 7):
        stride = 7
    else:
        raise ValueError(f"q_init must have shape (7,) or ({n}, 7), got {q_init.shape}")
    out = out or {}

    def buf(key, shape, dtype):
        return _check_out_np(f"out[{key!r}]", out[key], shape, dtype) if out.get(key) is not None else np.empty(shape, dtype)

    counters = np.zeros(4, dtype=np.uint64)
    if compact:
        q8 = buf("q8", (n, 8), np.float32)
        _lib.check(
            lib.pnp_ik_solve_compact_host_f32(host_ctx(chunk_rows), _np_ptr(targets), _np_ptr(q_init), stride, n,
                                              ctypes.byref(params), _np_ptr(q8), _np_ptr(counters)),
            "pnp_ik_solve_compact_host",
        )
        return HostIKResult(q=q8[:, :7], q8=q8, counters=counters)  # iterations / converged / success decoded on demand
    if packed:
        q8 = buf("q8", (n, 8), np.float32)
        aux = buf("aux4", (n, 4), np.float32)
        _lib.check(
            lib.pnp_ik_solve_packed_host_f32(host_ctx(chunk_rows), _np_ptr(targets), _np_ptr(q_init), stride, n,
                                             ctypes.byref(params), _np_ptr(q8), _np_ptr(aux), _np_ptr(counters)),
            "pnp_ik_solve_packed_host",
        )
        q, err, fpos, _ = unpack_ik(q8, aux)
        return HostIKResult(q=q, final_pos=fpos, pos_error=err, q8=q8, aux4=aux, counters=counters)
    q = buf("q", (n, 7), np.float32)
    fpos = buf("final_pos", (n, 3), np.float32)
    err = buf("pos_error", (n,), np.float32)
    iters = buf("iterations", (n,), np.int32)
    flags = buf("flags", (n,), np.uint8)
    _lib.check(
        lib.pnp_ik_solve_host_f32(host_ctx(chunk_rows), _np_ptr(targets), _np_ptr(q_init), stride, n,
                                  ctypes.byref(params), _np_ptr(q), _np_ptr(fpos), _np_ptr(err), _np_ptr(iters),
                                  _np_ptr(flags), _np_ptr(counters)),
        "pnp_ik_solve_host",
    )
    return dict(q=q, final_pos=fpos, pos_error=err, iterations=iters, flags=flags,
                converged=(flags & 1).astype(bool), success=(flags & 2).astype(bool), counters=counters)


def ik_solve_one_host(target3: np.ndarray, q_init7: np.ndarray, params: PnpIkParams, out12: Optional[np.ndarray] = None):
    """One query through the mapped-mailbox path (pnp_ik_solve_one_host_f32): float32 arrays in, the 12
    result words out (q0..q6, pos_error, final_pos xyz, iterations | flags << 24)."""
    lib = _lib.load()
    out = out12 if out12 is not None else np.empty(12, np.float32)
    rc = lib.pnp_ik_solve_one_host_f32(host_ctx(0), target3.ctypes.data, q_init7.ctypes.data, ctypes.byref(params),
                                       out.ctypes.data)
    if rc:
        _lib.check(rc, "pnp_ik_solve_one_host")
    return out


_tls = threading.local()


def reward_one_host(ag3: np.ndarray, dg3: np.ndarray, ee_pos3: np.ndarray, ee_quat4: np.ndarray, fingers_width: float,
                    task_index: int, params: PnpRewardParams):
    """One row through the mapped-mailbox path (pnp_reward_one_host_f64): contiguous float64 arrays in,
    (reward np.float32, is_success float, bits int) out - bits = placed | gripped << 1 | threshold_adjacent << 2."""
    lib = _lib.load()
    outs = getattr(_tls, "reward_out", None)
    if outs is None:  # per thread: the C call runs without the GIL
        outs = _tls.reward_out = (ctypes.c_float(), ctypes.c_float(), ctypes.c_uint32())
    r, sc, bits = outs
    rc = lib.pnp_reward_one_host_f64(host_ctx(0), ag3.ctypes.data, dg3.ctypes.data, ee_pos3.ctypes.data,
                                     ee_quat4.ctypes.data, float(fingers_width), int(task_index), ctypes.byref(params),
                                     ctypes.byref(r), ctypes.byref(sc), ctypes.byref(bits))
    if rc:
        _lib.check(rc, "pnp_reward_one_host")
    return np.float32(r.value), sc.value, bits.value


def reward_host(ag, dg, ee_pos, ee_quat, width, task_index, params: PnpRewardParams, want_success=True,
                chunk_rows: int = 0, out: Optional[np.ndarray] = None, out_success: Optional[np.ndarray] = None):
    """Host path: NumPy rows (float32 or float64 storage) -> reward float32[N], success, counters."""
    lib = _lib.load()
    first = ag.numpy() if isinstance(ag, torch.Tensor) else np.asarray(ag)
    dt = np.float32 if first.dtype == np.float32 else np.float64
    ag = _as_host("achieved_goal", ag, dt, (3,))
    dg = _as_host("desired_goal", dg, dt, (3,))
    ee_pos = _as_host("ee_pos", ee_pos, dt, (3,))
    ee_quat = _as_host("ee_quat", ee_quat, dt, (4,))
    width = _as_host("fingers_width", width, dt, ())
    task_index = _as_host("task_index", task_index, np.int32, ())
    n = ag.shape[0]
    for name, t in (("desired_goal", dg), ("ee_pos", ee_pos), ("ee_quat", ee_quat), ("fingers_width", width),
                    ("task_index", task_index)):
        if t.shape[0] != n:
            raise ValueError(f"{name} disagrees with achieved_goal on N")
    rew = _check_out_np("out", out, (n,), np.float32) if out is not None else np.empty((n,), np.float32)
    succ = _check_out_np("out_success", out_success, (n,), np.float32) if out_success is not None else (
        np.empty((n,), np.float32) if want_success else None)
    counters = np.zeros(4, dtype=np.uint64)
    fn = lib.pnp_reward_host_f32 if dt == np.float32 else lib.pnp_reward_host_f64
    _lib.check(
        fn(host_ctx(chunk_rows), _np_ptr(ag), _np_ptr(dg), _np_ptr(ee_pos), _np_ptr(ee_quat), _np_ptr(width),
           _np_ptr(task_index), n, ctypes.byref(params), _np_ptr(rew), _np_ptr(succ), _np_ptr(counters)),
        "pnp_reward_host",
    )
    return rew, succ, counters


def probe_fp32_peak() -> Tuple[float, float]:
    """(TFLOP/s, ms) of the FFMA microbenchmark on the current device."""
    _require_cuda()
    t, ms = ctypes.c_double(), ctypes.c_double()
    _lib.check(_lib.load().pnp_probe_fp32_peak(ctypes.byref(t), ctypes.byref(ms)), "pnp_probe_fp32_peak")
    return t.value, ms.value

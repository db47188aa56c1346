#!/usr/bin/env python
"""bench.py - Panda IK solves/s and HER reward evals/s on B200, beside the host-CPU path.

    python bench.py --gpus N --steps K --warmup W            # our arm (one rank per GPU)
    python bench.py --impl reference --steps K --warmup W    # reference arm = CPU oracle port

Headline line (one JSON object on stdout, rank 0):
  metric  panda_ik_converged_solves_per_s          (BASELINE.json: "Panda IK solves/s ...")
  step    one pass of the IK hot path over the rank's batch: 2^24 cold reachable targets per
          GPU from the neutral pose, reference defaults (BASELINE cfg5 sweep point; the cfg2
          batch of 4096 is a latency case and is reported under "latency").  Weak scaling.
  value   converged solves of all ranks / max-over-ranks device time, inputs resident in HBM
  e2e     same metric through the host-buffer C-ABI operator (pnp_ik_solve_packed_host_f32): pinned host
          inputs -> H2D -> kernel -> D2H of every IKResult field, all inside the timed region;
          e2e.link = the same bytes moved by bare cudaMemcpyAsync in both directions at once, no kernels
          (what the box's PCIe / host side delivers to this many ranks at the same time);
          e2e_compact = the 32-byte-record operator (q + iterations + flags only)
  roofline     IK kernel vs the FP32 CUDA-core peak (measured live by pnp_probe_fp32_peak;
               MEASURED_PEAKS.json has no FP32 entry) - the schema's "hbm"/"tensor" do not apply
  reward       the second half of the metric (HER reward evals/s, cfg3: 16 777 216 rows, FP32
               storage, 64 B/row) with its own value / e2e / HBM roofline / cpu_baseline
  latency      cfg1 (one solve() host to host), cfg2 (4096 cold targets, one launch), one scalar
               compute_reward() - each beside the C port and the NumPy port of the same call
  cpu_baseline the C oracle port on all host cores over a bounded sample of the same workload
  headline     both halves of BASELINE.json's metric once more, last on the line

--dump-outputs DIR writes, after the timed steps, what the last timed IK step and the last timed reward step of rank 0
computed, as DIR/<name>.npy (float32 / float64, about 40 MB): the IKResult fields of a fixed, seeded sample of 2^19
queries, the rewards of a sample of 2^19 rows, and the indices of both samples.  The inputs are seeded, so two builds
run with the same arguments can be compared output for output.
"""

from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the tree may be read-only: leave no __pycache__ behind in it

import numpy as np  # noqa: E402

IK_FLOP_PER_ITER = 500.0  # SURVEY.md 8(d): algorithmic FLOP per DLS iteration (position mode)
IK_FLOP_PER_SOLVE = 216.0  # + one FK per solve
REWARD_BYTES_PER_ROW = 64.0  # 60 B in + 4 B out (FP32 storage)
LOG2_N_IK = 24
LOG2_N_REWARD = 24
REWARD_KEYS = ("achieved_goal", "desired_goal", "ee_pos", "ee_quat", "fingers_width", "task_index")
NEUTRAL = np.array([0.00, 0.41, 0.00, -1.85, 0.00, 2.26, 0.79])
DUMP_SAMPLE = 1 << 19  # rows per --dump-outputs sample: 64 B per IK query + 12 B per reward row, 38 MiB in all


def host_cores() -> int:
    return len(os.sched_getaffinity(0))


def bench_config(world: int, log2_n_ik: int = LOG2_N_IK, log2_n_reward: int = LOG2_N_REWARD) -> dict:
    """What is measured - the same dict in our arm and in the reference arm."""
    return {
        "workload": f"cfg5 cold IK, 2^{log2_n_ik} reachable targets (FK of q* ~ U(joint range)) per GPU from the neutral "
                    "pose, max_iters=100 pos_thresh=1e-3 damping=1e-2 step_limit=0.1",
        "second_half": f"cfg3 dense reward, 2^{log2_n_reward} HER-relabelled rows per GPU, FP32 storage",
        "l2_hygiene": f"inputs+outputs per step {(1 << log2_n_ik) * 60 / 1e6:.0f} MB (IK) / {(1 << log2_n_reward) * 64 / 1e6:.0f} MB "
                      "(reward) > 126 MB L2, no flush needed",
        "parallelism": f"batch-index shards x{world}, NCCL all_reduce of 4 counters",
        "outputs": "two preallocated output sets written alternately (steps are back-to-back launches on one stream)",
    }


# ------------------------------------------------------------------------------------------------
# clocks: sample NVML during the timed regions
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    def __init__(self, gpu_index: int, period_s: float = 0.005):
        self.idx, self.period = gpu_index, period_s
        self.sm, self.reasons = [], set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._thread = None
        self._nvml = None

    def start(self):
        try:
            import pynvml

            pynvml.nvmlInit()
            self._nvml = pynvml
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = self.idx
            if vis:
                ids = [v.strip() for v in vis.split(",") if v.strip()]
                if self.idx < len(ids) and ids[self.idx].isdigit():
                    phys = int(ids[self.idx])
            self._h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
        except Exception as exc:  # pragma: no cover - depends on the box
            self._nvml = None
            self.reasons.add(f"nvml_unavailable:{type(exc).__name__}")
            return self
        self._thread = threading.Thread(target=self._run, daemon=True)
        self._thread.start()
        return self

    def _run(self):
        nv = self._nvml
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
        }
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or getattr(
            nv, "nvmlDeviceGetCurrentClocksThrottleReasons")
        while not self._stop.is_set():
            try:
                self.sm.append(int(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
                mask = int(get_reasons(self._h))
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self) -> dict:
        self._stop.set()
        if self._thread:
            self._thread.join(timeout=2)
        sm = self.sm
        # "under load": drop idle-clock samples from before the first kernel ramps the clocks
        loaded = [x for x in sm if self.max_mhz and x >= 0.5 * self.max_mhz] or sm
        return {
            "sm_mhz": int(statistics.median(loaded)) if loaded else None,
            "sm_max_mhz": self.max_mhz,
            "reasons": sorted(self.reasons),
            "samples": len(sm),
        }


def ncu_traffic(kernel: str, units: int, files=("ncu_traffic_r2d.json", "ncu_traffic_r2.json", "ncu_traffic_r1.json")):
    """DRAM bytes per launch for `kernel` from the committed `ncu --set full` capture
    (profiles/ncu_traffic_r2d.json, else _r2 / _r1: dram__bytes_read.sum + dram__bytes_write.sum per unit, scaled to
    this launch's unit count); None when no capture is on file."""
    for name in files:  # the latest capture on file
        try:
            with open(os.path.join(ROOT, "profiles", name)) as fh:
                return float(json.load(fh)[kernel]["dram_bytes_per_unit"]) * units
        except Exception:
            continue
    return None


def bind_to_gpu_numa_node(gpu_index: int):
    """Pin this rank's threads to the CPUs NVML reports as local to its GPU, so that the pinned host
    buffers of the e2e path are allocated (first touch) on the NUMA node behind the same PCIe root.
    Best effort: returns the CPU count bound to, or None."""
    try:
        import pynvml

        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = gpu_index
        if vis:
            ids = [v.strip() for v in vis.split(",") if v.strip()]
            if gpu_index < len(ids) and ids[gpu_index].isdigit():
                phys = int(ids[gpu_index])
        h = pynvml.nvmlDeviceGetHandleByIndex(phys)
        allowed = os.sched_getaffinity(0)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        local = {64 * w + b for w, word in enumerate(words) for b in range(64) if (int(word) >> b) & 1}
        cpus = allowed & local
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


def measured_peaks() -> dict:
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            d = json.load(fh)
        return {"hbm_gbs": float(d["hbm_gbs"]), "source": "MEASURED_PEAKS.json (burst copy)"}
    return {"hbm_gbs": 6650.0, "source": "fallback (B200_PROFILING.md: 6.65 TB/s)"}


# ------------------------------------------------------------------------------------------------
# CPU path (oracle port) - used only as the reported baseline / reference arm
# ------------------------------------------------------------------------------------------------
def cpu_ik_setup():
    from oracle import c_oracle, mj_oracle

    c_oracle.build()
    asset = os.path.join(ROOT, "mujoco_panda_pnp_b200", "assets", "panda_shelf_kinematic.xml")
    model = mj_oracle.MjModel.from_xml_path(asset)
    return c_oracle, c_oracle.chain_from_model(model), model


def cpu_ik_targets(c_oracle, chain, model, n, seed=1234):
    rng = np.random.default_rng(seed)
    q = rng.uniform(model.jnt_range[:7, 0], model.jnt_range[:7, 1], size=(n, 7))
    return c_oracle.fk_jac(chain, q, nthreads=host_cores())[0]


def cpu_ik_baseline(budget_s: float = 12.0) -> dict:
    """Bounded sample of the bench workload on all host cores (C oracle port, FP64)."""
    c_oracle, chain, model = cpu_ik_setup()
    cores = host_cores()
    calib = cpu_ik_targets(c_oracle, chain, model, 4096 * max(1, cores // 4))
    t0 = time.perf_counter()
    c_oracle.ik_solve(chain, calib, NEUTRAL, nthreads=cores)
    rate = len(calib) / (time.perf_counter() - t0)
    n = int(min(max(rate * budget_s, 8192), 1 << 22))
    targets = cpu_ik_targets(c_oracle, chain, model, n)
    t0 = time.perf_counter()
    r = c_oracle.ik_solve(chain, targets, NEUTRAL, nthreads=cores)
    dt = time.perf_counter() - t0
    out = {
        "value": float(r["converged"].sum() / dt), "unit": "solves/s", "cores": cores, "kind": "port",
        "sample": f"{n} cold targets (same generator as the GPU batch), {dt:.1f} s, FP64 C restatement of "
                  "ik_solver.py:50-101 without mj_forward's collision stages (faster than the real reference)",
        "mean_iterations": float(r["iterations"].mean()),
    }
    # SURVEY 8d (ii): the NumPy restatement on one core - the closest thing here to the reference's own
    # Python (same control flow and NumPy/LAPACK calls, MuJoCo replaced by the restated engine)
    try:
        from oracle import ik_oracle, mj_oracle

        ctl = ik_oracle.JacobianIKController(model, mj_oracle.MjData(model))
        m, t0, conv = 0, time.perf_counter(), 0
        while m < len(targets) and (time.perf_counter() - t0 < 2.0 or m < 8):
            conv += int(ctl.solve(targets[m], NEUTRAL).converged)
            m += 1
        dt1 = time.perf_counter() - t0
        out["numpy_port_1core"] = {"value": conv / dt1, "unit": "solves/s", "cores": 1,
                                   "sample": f"{m} of the same targets, {dt1:.1f} s, oracle/ik_oracle.py"}
    except Exception as exc:  # the C port above is the baseline; this line is informational
        out["numpy_port_1core"] = {"unavailable": repr(exc)}
    return out


def cpu_latency_baselines(targets4096: np.ndarray) -> dict:
    """The CPU side of the three latency configs: the C port and the NumPy port of the same call, timed here."""
    from oracle import c_oracle, ik_oracle, mj_oracle, reward_oracle

    c_oracle, chain, model = cpu_ik_setup()
    cores = host_cores()
    out = {}
    grasp = [np.array(t) for t in [(1.415, 0, 0.73), (1.415, 0, 1.03), (1.415, 0, 0.43)]]
    for t_ in grasp:
        c_oracle.ik_solve(chain, t_[None], NEUTRAL, nthreads=1)
    t0 = time.perf_counter()
    for _ in range(200):
        for t_ in grasp:
            c_oracle.ik_solve(chain, t_[None], NEUTRAL, nthreads=1)
    c_us = (time.perf_counter() - t0) / 600 * 1e6
    ctl = ik_oracle.JacobianIKController(model, mj_oracle.MjData(model))
    t0 = time.perf_counter()
    for t_ in grasp:
        ctl.solve(t_, NEUTRAL)
    np_us = (time.perf_counter() - t0) / 3 * 1e6
    out["cfg1"] = {"c_port_us_per_solve": c_us, "numpy_port_us_per_solve": np_us, "cores": 1,
                   "note": "same 3 grasp poses; C port = one ctypes call per solve, NumPy port = oracle/ik_oracle.py "
                           "(the reference's control flow over the restated engine, no mj_forward collision stages)"}
    c_oracle.ik_solve(chain, targets4096, NEUTRAL, nthreads=cores)
    ts = []
    for _ in range(5):
        t0 = time.perf_counter()
        c_oracle.ik_solve(chain, targets4096, NEUTRAL, nthreads=cores)
        ts.append(time.perf_counter() - t0)
    out["cfg2"] = {"c_port_us_per_batch": min(ts) * 1e6, "cores": cores,
                   "numpy_port_us_per_batch_est": np_us * 4096, "note": "NumPy port: per-solve time x 4096, one core"}
    h = cpu_reward_rows(64)
    c_oracle.reward(*[x[:1] for x in h], nthreads=1)
    t0 = time.perf_counter()
    for _ in range(50):
        for i in range(64):
            c_oracle.reward(*[x[i:i + 1] for x in h], nthreads=1)
    rc_us = (time.perf_counter() - t0) / (50 * 64) * 1e6
    t0 = time.perf_counter()
    for _ in range(20):
        for i in range(64):
            reward_oracle.compute_reward(h[0][i], h[1][i], h[2][i], h[3][i], h[4][i], h[5][i])
    rn_us = (time.perf_counter() - t0) / (20 * 64) * 1e6
    out["reward_scalar"] = {"c_port_us_per_call": rc_us, "numpy_port_us_per_call": rn_us, "cores": 1,
                            "note": "NumPy port = oracle/reward_oracle.compute_reward, the reference's own statements "
                                    "(panda_env.py:205-245) with the simulator getters replaced by arguments"}
    return out


def cpu_reward_rows(n, seed=0):
    import torch

    from mujoco_panda_pnp_b200 import synthetic

    rows = synthetic.reward_rows(n, seed=seed, device="cpu", dtype=torch.float32)
    return [rows[k].double().numpy() if rows[k].dtype != torch.int32 else rows[k].numpy() for k in REWARD_KEYS]


def cpu_reward_baseline(budget_s: float = 8.0) -> dict:
    from oracle import c_oracle

    c_oracle.build()
    cores = host_cores()
    n = 1 << 22
    h = cpu_reward_rows(n)
    c_oracle.reward(*[x[: 1 << 16] for x in h], nthreads=cores)
    reps, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < budget_s or reps == 0:
        c_oracle.reward(*h, reward_type="dense", nthreads=cores)
        reps += 1
    dt = time.perf_counter() - t0
    return {"value": float(n * reps / dt), "unit": "rows/s", "cores": cores, "kind": "port",
            "sample": f"{reps} x {n} rows (first 2^22 of the cfg3 generator), {dt:.1f} s, FP64 C restatement of "
                      "panda_env.py:205-245"}


# ------------------------------------------------------------------------------------------------
# reference arm
# ------------------------------------------------------------------------------------------------
def run_reference(args) -> int:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import torch

    from mujoco_panda_pnp_b200 import synthetic

    c_oracle, chain, model = cpu_ik_setup()
    cores = host_cores()
    calib = cpu_ik_targets(c_oracle, chain, model, 8192)
    t0 = time.perf_counter()
    c_oracle.ik_solve(chain, calib, NEUTRAL, nthreads=cores)
    rate = len(calib) / (time.perf_counter() - t0)
    # Each step = the SAME workload as our arm: 2^24 cold targets of the same generator family (q* ~ U(joint range),
    # target = FK(q*), seed 1234).  Only if the whole K + W run would not end within ~10 minutes on this box's cores is
    # a step cut down to a bounded sample of that batch (said in cpu_baseline.sample; the metric is a rate).
    n_full = 1 << args.log2_n_ik
    budget_s = 600.0 / max(1, args.steps + args.warmup)
    n = n_full if n_full / rate <= budget_s else int(max(rate * budget_s, 4096))
    qstar = synthetic.random_joint_configs(n, model.jnt_range[:7, 0], model.jnt_range[:7, 1], seed=1234, dtype=torch.float64).numpy()
    targets = c_oracle.fk_jac(chain, qstar, nthreads=cores)[0]
    del qstar
    for _ in range(args.warmup):
        c_oracle.ik_solve(chain, targets, NEUTRAL, nthreads=cores)
    conv = 0
    t0 = time.perf_counter()
    for _ in range(args.steps):
        r = c_oracle.ik_solve(chain, targets, NEUTRAL, nthreads=cores)
        conv += int(r["converged"].sum())
    dt = time.perf_counter() - t0
    value = conv / dt
    rw = cpu_reward_baseline(budget_s=5.0)
    sample = (f"each step = {'the full batch of ' if n == n_full else 'a bounded sample of '}{n} cold reachable targets from "
              f"neutral (workload: 2^{args.log2_n_ik} per GPU), {cores} threads, FP64 C restatement of ik_solver.py:50-101")
    line = {
        "impl": "reference", "metric": "panda_ik_converged_solves_per_s", "value": value, "unit": "solves/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": bench_config(args.gpus, args.log2_n_ik, args.log2_n_reward),
        "cpu_baseline": {"value": value, "unit": "solves/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "solves/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "reward": {"metric": "her_reward_evals_per_s", "value": rw["value"], "unit": "rows/s", "cpu_baseline": rw},
        "note": "reference arm = oracle port (C, FP64, all host threads): mujoco is not installable in this image, "
                "see DESIGN.md; it omits mj_forward's collision/constraint work and is faster than the real reference",
        "headline": {"ik_solves_per_s": value, "reward_rows_per_s": rw["value"], "cores": cores},
    }
    emit(line)
    return 0


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def cuda_time_steps(fn, steps, torch, presync=True):
    """Per-launch CUDA-event durations (ms) on the current stream."""
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    if presync:
        torch.cuda.synchronize()
    for e0, e1 in evs:
        e0.record()
        fn()
        e1.record()
    torch.cuda.synchronize()
    total = evs[0][0].elapsed_time(evs[-1][1])  # whole timed region, first launch to last completion
    return total, [e0.elapsed_time(e1) for e0, e1 in evs]


def dump_rows(n: int, seed: int) -> np.ndarray:
    """Ascending row indices of the --dump-outputs sample: all n rows, or a fixed seeded DUMP_SAMPLE of them."""
    if n <= DUMP_SAMPLE:
        return np.arange(n)
    return np.sort(np.random.default_rng(seed).choice(n, DUMP_SAMPLE, replace=False))


def write_dump(out_dir: str, ik_rows, q8, aux4, rw_rows, reward) -> None:
    """The sampled outputs of the last timed steps as out_dir/<name>.npy: what ik_solve's BatchIKResult and reward()
    return for those rows, flags and iteration counts as float32, indices as float64."""
    from mujoco_panda_pnp_b200 import engine

    q, pos_error, final_pos, word = engine.unpack_ik(q8, aux4)
    arrays = {
        "ik_query_index": ik_rows.astype(np.float64),
        "ik_q": q,
        "ik_final_pos": final_pos,
        "ik_pos_error": pos_error,
        "ik_iterations": (word & 0xFFFFFF).astype(np.float32),
        "ik_converged": ((word & (1 << 24)) != 0).astype(np.float32),
        "ik_success": ((word & (2 << 24)) != 0).astype(np.float32),
        "reward_row_index": rw_rows.astype(np.float64),
        "reward": reward,
    }
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))
    print(f"[bench] wrote {len(arrays)} arrays ({sum(a.nbytes for a in arrays.values()) / 2**20:.1f} MiB) to {out_dir}")


def run_ours(args) -> int:
    import torch

    from mujoco_panda_pnp_b200 import KinematicTree, _lib, engine, synthetic
    from mujoco_panda_pnp_b200 import distributed as D

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (there is no CPU fallback; use --impl reference for the CPU arm)")
    rank, local_rank, world = D.init_process_group("nccl")
    if not os.path.exists(_lib.LIB_PATH):  # normally prebuilt by __graft_entry__.build(); never fall back to CPU
        if rank == 0:
            from mujoco_panda_pnp_b200.csrc import build as cuda_build

            cuda_build.build()
        D.barrier()
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torchrun --nproc-per-node {args.gpus}")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = bind_to_gpu_numa_node(local_rank) if world > 1 else None
    lib = _lib.load()
    tree = KinematicTree.from_mjcf()
    specialized = engine.set_tree(tree)
    K, W = args.steps, args.warmup

    # ---------------- inputs, resident in HBM (generated per rank on device) ----------------
    n_ik = 1 << args.log2_n_ik
    qstar = synthetic.random_joint_configs(n_ik, tree.lower, tree.upper, seed=1234 + rank, device=dev)
    targets = engine.fk_jac(qstar, want_quat=False, want_jac=False)[0]
    del qstar
    neutral = torch.tensor(NEUTRAL, dtype=torch.float32, device=dev)
    params = engine.ik_params()
    ik_counters = torch.zeros(4, dtype=torch.int64, device=dev)
    # preallocated outputs (allocation is not part of a step)
    # Two output sets, written alternately - what a consumer that reads step k while step k+1 runs needs anyway.  With
    # nothing between two launches that the second one could clobber, the library makes it a programmatic dependent of
    # the first: its blocks move into the SMs that the first launch's drain (a handful of queries on their way to
    # max_iters) leaves idle.  Every launch still solves all 2^24 queries and writes all its outputs.
    ik_outs = [dict(q8=torch.empty((n_ik, 8), device=dev), aux4=torch.empty((n_ik, 4), device=dev)) for _ in range(2)]
    ik_out = ik_outs[0]
    import ctypes

    stream = torch.cuda.current_stream().cuda_stream
    ik_step_no = [0]

    def ik_step(counters=None):
        o = ik_outs[ik_step_no[0] & 1]
        ik_step_no[0] += 1
        _lib.check(lib.pnp_ik_solve_packed_f32(targets.data_ptr(), neutral.data_ptr(), 0, n_ik, ctypes.byref(params),
                                               o["q8"].data_ptr(), o["aux4"].data_ptr(),
                                               counters.data_ptr() if counters is not None else None, stream), "ik")

    n_rw = 1 << args.log2_n_reward
    rows = synthetic.reward_rows(n_rw, seed=rank, device=dev, dtype=torch.float32)
    rw_args = [rows[k] for k in REWARD_KEYS]
    rw_params = engine.reward_params("dense")
    rw_out = torch.empty(n_rw, dtype=torch.float32, device=dev)
    rw_counters = torch.zeros(4, dtype=torch.int64, device=dev)

    def rw_step(counters=None):
        engine.reward(*rw_args, rw_params, want_success=False, counters=counters, out=rw_out)

    fp32_peak, _ = engine.probe_fp32_peak()
    fp32_peak = max(fp32_peak, engine.probe_fp32_peak()[0])
    peaks = measured_peaks()

    sampler = ClockSampler(local_rank).start()

    # ---------------- IK: device-resident timing ------------------------------------------
    for _ in range(W):
        ik_step()
    ik_step(ik_counters)  # one counted pass (also untimed): per-step workload statistics
    torch.cuda.synchronize()
    D.barrier()
    launches0 = lib.pnp_launch_count()
    # K launches back to back between ONE pair of events (an event record between two launches is a stream operation of
    # its own and would serialise them): the kernel's average duration is the region / K
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(K):
        ik_step()
    ev1.record()
    torch.cuda.synchronize()
    ik_total = ev0.elapsed_time(ev1)
    launches_ik = lib.pnp_launch_count() - launches0
    dump = args.dump_outputs and rank == 0
    if dump:  # the output set the last timed step wrote, before the launches below reuse it
        ik_rows = dump_rows(n_ik, seed=0)
        last = ik_outs[(ik_step_no[0] - 1) & 1]
        ik_dump = {k: last[k].index_select(0, torch.from_numpy(ik_rows).to(dev)).cpu().numpy() for k in ("q8", "aux4")}
    D.barrier()
    ik_ms_total = D.reduce_max(ik_total, dev)
    ik_kernel_ms = ik_total / K
    # for reference, outside the timed region: the same launch alone on an idle device (events around every launch)
    _, t_ik = cuda_time_steps(ik_step, min(K, 5), torch)
    ik_single_ms = statistics.median(t_ik)
    assert all(torch.equal(ik_outs[0][k], ik_outs[1][k]) for k in ("q8", "aux4")), "the two output sets differ"
    c = D.reduce_counters(ik_counters).cpu().numpy()
    c_local = ik_counters.cpu().numpy()
    ik_value = float(c[1]) * K / (ik_ms_total * 1e-3)
    ik_flop_launch = IK_FLOP_PER_ITER * float(c_local[3]) + IK_FLOP_PER_SOLVE * float(c_local[0])
    ik_tflops = ik_flop_launch / (ik_kernel_ms * 1e-3) / 1e12

    # ---------------- reward: device-resident timing --------------------------------------
    for _ in range(W):
        rw_step()
    rw_step(rw_counters)
    torch.cuda.synchronize()
    D.barrier()
    rw_total, t_rw = cuda_time_steps(rw_step, K, torch)
    if dump:
        rw_rows = dump_rows(n_rw, seed=1)
        rw_dump = rw_out.index_select(0, torch.from_numpy(rw_rows).to(dev)).cpu().numpy()
    D.barrier()
    rw_ms_total = D.reduce_max(rw_total, dev)
    rw_kernel_ms = sum(t_rw) / K
    rw_value = float(n_rw) * world * K / (rw_ms_total * 1e-3)
    rw_gbs = REWARD_BYTES_PER_ROW * n_rw / (rw_kernel_ms * 1e-3) / 1e9

    # ---------------- e2e: host buffers through the C-ABI host operators --------------------
    h_targets = targets.cpu().pin_memory()
    h_neutral = NEUTRAL.astype(np.float32)
    h_out = dict(q8=torch.empty((n_ik, 8)).pin_memory().numpy(), aux4=torch.empty((n_ik, 4)).pin_memory().numpy())
    for _ in range(2):
        engine.ik_solve_host(h_targets, h_neutral, params, out=h_out)
    D.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    conv_e2e = 0
    for _ in range(K):
        r = engine.ik_solve_host(h_targets, h_neutral, params, out=h_out)  # blocks until outputs are on the host
        conv_e2e += int(r["counters"][1])
    ik_e2e_s = D.reduce_max(time.perf_counter() - t0, dev)
    conv_e2e_total = int(D.reduce_counters(torch.tensor([conv_e2e, 0, 0, 0], dtype=torch.int64, device=dev))[0])
    ik_e2e = conv_e2e_total / ik_e2e_s
    ik_h2d = n_ik * 12 + 28
    ik_d2h = n_ik * (32 + 16) + 32  # packed records: q0..q6,pos_error | final_pos xyz, iterations|flags

    # the 32-byte-record operator: q + iterations + flags only (final_pos / pos_error not brought back)
    for _ in range(2):
        engine.ik_solve_host(h_targets, h_neutral, params, out=h_out, compact=True)
    D.barrier()
    t0 = time.perf_counter()
    conv_c = 0
    for _ in range(K):
        r = engine.ik_solve_host(h_targets, h_neutral, params, out=h_out, compact=True)
        conv_c += int(r["counters"][1])
    ik_e2e_c_s = D.reduce_max(time.perf_counter() - t0, dev)
    ik_e2e_c = int(D.reduce_counters(torch.tensor([conv_c, 0, 0, 0], dtype=torch.int64, device=dev))[0]) / ik_e2e_c_s
    # what the link delivers: the same bytes per step as bare copies in both directions at once, no kernels, all ranks
    # at the same time (pinned host memory, one cudaMemcpyAsync per direction on its own stream)
    d_up = torch.empty(n_ik * 3, device=dev)
    d_dn = torch.empty(n_ik * 12, device=dev)
    h_up = h_targets.reshape(-1)
    h_dn = torch.empty(n_ik * 12).pin_memory()
    s_up, s_dn = torch.cuda.Stream(), torch.cuda.Stream()

    def raw_copies():
        with torch.cuda.stream(s_up):
            d_up.copy_(h_up, non_blocking=True)
        with torch.cuda.stream(s_dn):
            h_dn.copy_(d_dn, non_blocking=True)
        s_up.synchronize()
        s_dn.synchronize()

    raw_copies()
    D.barrier()
    t0 = time.perf_counter()
    for _ in range(K):
        raw_copies()
    link_s = D.reduce_max(time.perf_counter() - t0, dev) / K
    link = {"h2d_plus_d2h_gbs_all_ranks": (n_ik * 60.0) * world / link_s / 1e9,
            "d2h_gbs_all_ranks": (n_ik * 48.0) * world / link_s / 1e9,
            "ceiling_solves_per_s": float(c[1]) / float(c[0]) * n_ik * world / link_s,
            "how": "bare pinned cudaMemcpyAsync of one step's bytes (12 B/query up, 48 B/query down) on two streams, "
                   "all ranks at once, max over ranks: the e2e value cannot exceed ceiling_solves_per_s on this box"}
    del d_up, d_dn, h_dn

    h_rows = [rows[k].cpu().pin_memory() for k in REWARD_KEYS]
    h_rw = torch.empty(n_rw, dtype=torch.float32).pin_memory().numpy()
    for _ in range(2):
        engine.reward_host(*h_rows, rw_params, want_success=False, out=h_rw)
    D.barrier()
    t0 = time.perf_counter()
    for _ in range(K):
        engine.reward_host(*h_rows, rw_params, want_success=False, out=h_rw)
    rw_e2e_s = D.reduce_max(time.perf_counter() - t0, dev)
    rw_e2e = n_rw * world * K / rw_e2e_s

    # ---------------- side configs (rank 0 only, short) ---------------------------------
    side = {}
    if rank == 0:
        # cfg2 is a latency case (one ~30 us launch): the launches are queued behind a 3 ms device-side sleep so that the
        # CUDA events bracket device time only, not the ~20 us of Python between record() and the launch
        t4096 = targets[:4096].contiguous()
        q8_s, aux_s = torch.empty((4096, 8), device=dev), torch.empty((4096, 4), device=dev)
        f = lambda: engine.ik_solve(t4096, neutral, params, out_q8=q8_s, out_aux4=aux_s)  # noqa: E731
        for _ in range(3):
            f()
        torch.cuda.synchronize()
        torch.cuda._sleep(int(3e-3 * 1.9e9))
        _, ts = cuda_time_steps(f, 20, torch, presync=False)
        side["cfg2"] = {"workload": "4096 cold targets from neutral, 1 launch (ik_solve_small_kernel: one query per lane, one warp per SM)",
                        "ms_per_launch": statistics.median(ts), "us_per_launch": statistics.median(ts) * 1e3,
                        "us_min": min(ts) * 1e3, "solves_per_s": 4096 / (statistics.median(ts) * 1e-3),
                        "bound": "latency: the launch lasts as long as its slowest query, 100 dependent DLS passes (max_iters) "
                                 "of ~500 clocks each on a lone warp"}
        n_env = 1 << 20
        w = synthetic.waypoint_envs(n_env, seed=0, device=dev)
        cnt = torch.zeros(4, dtype=torch.int64, device=dev)
        engine.ik_waypoints(w["q_start"], w["goal"], 50, params, counters=cnt)
        torch.cuda.synchronize()
        cw = cnt.cpu().numpy()
        _, ts = cuda_time_steps(lambda: engine.ik_waypoints(w["q_start"], w["goal"], 50, params), 3, torch)
        side["cfg4"] = {"workload": "2^20 envs x 50 warm-started waypoint solves, 1 launch",
                        "ms_per_launch": min(ts), "warm_solves_per_s": float(cw[0]) / (min(ts) * 1e-3),
                        "mean_iterations": float(cw[3]) / max(1.0, float(cw[0]))}
        # cfg1: single-query latency through the drop-in controller (host in, host out)
        from mujoco_panda_pnp_b200 import KinematicData, KinematicModel
        from mujoco_panda_pnp_b200.skills import JacobianIKController

        kmodel = KinematicModel.from_xml_path(os.path.join(ROOT, "mujoco_panda_pnp_b200", "assets", "panda_shelf_kinematic.xml"))
        ctl = JacobianIKController(kmodel, KinematicData(kmodel))
        grasp = [np.array(t) for t in [(1.415, 0, 0.73), (1.415, 0, 1.03), (1.415, 0, 0.43)]]
        for t_ in grasp:
            ctl.solve(t_, NEUTRAL)
        t0 = time.perf_counter()
        reps = 50
        its = []
        for _ in range(reps):
            for t_ in grasp:
                its.append(ctl.solve(t_, NEUTRAL).iterations)
        side["cfg1"] = {"workload": "single-query solve() to the 3 shelf grasp poses from neutral (test/ik_test.py path)",
                        "us_per_solve_host_to_host": (time.perf_counter() - t0) / (3 * reps) * 1e6,
                        "iterations": its[:3]}
        # one scalar compute_reward(achieved_goal (3,), desired_goal (3,), info) host to host: what FrankaEnv.step pays
        # once per env.step (envs/panda_env.py:176-181), through the mapped mailbox
        from mujoco_panda_pnp_b200.envs import FrankaShelfPNPReward

        renv = FrankaShelfPNPReward("dense")
        hr = [rows[k][:64].double().cpu().numpy() if rows[k].dtype != torch.int32 else rows[k][:64].cpu().numpy() for k in REWARD_KEYS]
        infos = [dict(ee_pos=hr[2][i], ee_quat=hr[3][i], fingers_width=float(hr[4][i]), task_index=int(hr[5][i])) for i in range(64)]
        for i in range(64):
            renv.compute_reward(hr[0][i], hr[1][i], infos[i])
        t0 = time.perf_counter()
        for _ in range(20):
            for i in range(64):
                renv.compute_reward(hr[0][i], hr[1][i], infos[i])
        side["reward_scalar"] = {"workload": "one compute_reward() with (3,) goals, host in -> np.float32 out (pnp_reward_one_host_f64)",
                                 "us_per_call_host_to_host": (time.perf_counter() - t0) / (20 * 64) * 1e6}
        # SURVEY 8f-1: whole MoveIKSkill.reset planner, 2^20 envs in one launch (plans are 40-200 solves long and a lane
        # owns one env at a time: below ~2^20 envs the launch is dominated by load imbalance, 2^18 runs at 0.7 of this rate)
        n_pl = 1 << 20
        wp = synthetic.reachable_move_envs(n_pl, tree.lower, tree.upper, seed=1, device=dev)
        wp["goal"] = engine.fk_jac(wp["q_goal"], want_quat=False, want_jac=False)[0]
        cnt = torch.zeros(4, dtype=torch.int64, device=dev)
        plan = engine.move_ik_plan(wp["q_start"], wp["goal"], params, counters=cnt)
        torch.cuda.synchronize()
        cp = cnt.cpu().numpy()
        # timed: the order kernels (longest plan first) + the planner, into the buffers of the call above
        _, ts = cuda_time_steps(lambda: engine.move_ik_plan(wp["q_start"], wp["goal"], params, out=plan), 2, torch)
        side["move_planner"] = {"workload": "2^20 MoveIKSkill.reset plans, reachable goals FK(neutral +- 0.6 rad), 1 launch",
                                "ms_per_launch": min(ts),
                                "plans_per_s": n_pl / (min(ts) * 1e-3), "ik_solves_per_s": float(cp[0]) / (min(ts) * 1e-3),
                                "mean_solves_per_plan": float(cp[0]) / n_pl}
        del wp, plan
        # SURVEY 8f-2: HER relabel + reward + VecNormalize over stored transitions (464 B/transition).  The headline
        # workload is what HER does ("future" strategy: the goal comes from a later transition of the SAME episode,
        # episodes stored as runs of 300 rows = the reference's max_episode_steps, panda_mujoco_gym/__init__.py:15);
        # the uniform-random gather (any row of the buffer) rides along as the worst case, with and without the goal table
        n_h = 1 << 23
        g = torch.Generator(device=dev)
        g.manual_seed(7)
        h_next = torch.randn((n_h, 25), generator=g, device=dev)
        h_obs = h_next + 0.01
        h_quat = torch.randn((n_h, 4), generator=g, device=dev)
        h_task = torch.randint(0, 3, (n_h,), generator=g, device=dev, dtype=torch.int32)
        h_o, h_x, h_r = torch.empty_like(h_obs), torch.empty_like(h_next), torch.empty(n_h, device=dev)
        nrm = engine.normalize_params(np.zeros(25), np.ones(25))

        def her_line(h_fut, workload, alg_bytes=464.0, traffic=None, **kw):
            f_her = lambda: engine.her_relabel(h_obs, h_next, h_fut, h_quat, h_task, rw_params, norm=nrm, want_success=False,  # noqa: E731
                                               out_obs=h_o, out_next_obs=h_x, out_reward=h_r, **kw)
            for _ in range(3):
                f_her()
            _, ts = cuda_time_steps(f_her, 10, torch)
            ms = statistics.median(ts)
            gbs = alg_bytes * n_h / (ms * 1e-3) / 1e9
            return {"workload": workload, "ms_per_launch": ms, "transitions_per_s": n_h / (ms * 1e-3),
                    "roofline": {"bound": "hbm", "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": gbs / peaks["hbm_gbs"],
                                 "traffic": traffic,
                                 "algorithmic": "%d B/transition (200 read + 200 written + 64 reward stream, SURVEY 8d%s)"
                                                % (alg_bytes, " + the 12-byte gathered goal" if alg_bytes > 464 else ""),
                                 "kernel": "her_relabel_kernel<true>"}}

        fut_ep = synthetic.her_future_indices(n_h, 300, seed=7, device=dev, strategy="future")
        side["her_relabel"] = her_line(fut_ep, "2^23 stored transitions, HER 'future' strategy (goal = achieved goal of a later transition "
                                       "of the same 300-step episode, 1 in 5 keeps its goal): gather, relabel obs/next_obs, reward, VecNormalize",
                                       traffic=ncu_traffic("her_relabel_kernel", n_h, files=("ncu_traffic_r2d.json",)))  # captured on this workload
        del fut_ep
        fut_un = synthetic.her_future_indices(n_h, 300, seed=7, device=dev, strategy="uniform")
        side["her_relabel_uniform_gather"] = her_line(fut_un, "same, goal gathered from ANY row of the buffer (no locality: every 12-byte goal "
                                                      "costs a DRAM burst)", traffic=ncu_traffic("her_relabel_kernel", n_h, files=("ncu_traffic_r2.json",)))  # captured on this one
        h_tab = h_next[:, 19:22].contiguous()
        side["her_relabel_goal_table"] = her_line(fut_un, "uniform gather from a separate [N,3] achieved-goal table (pnp_her_relabel_table_f32)",
                                                  alg_bytes=476.0, future_ag=h_tab)
        del h_tab, fut_un
        del h_next, h_obs, h_o, h_x
        # R4: batched _get_obs from kinematic state (128 B in + 100 B out per env)
        n_o = 1 << 22
        go = torch.Generator(device=dev)
        go.manual_seed(3)
        rnd = lambda *sh: torch.randn(sh, generator=go, device=dev)  # noqa: E731
        o_args = [rnd(n_o, 7), rnd(n_o, 7), rnd(n_o, 2).abs() * 0.02, rnd(n_o, 3), rnd(n_o, 4), rnd(n_o, 6), rnd(n_o, 3)]
        f_obs = lambda: engine.get_obs(*o_args)  # noqa: E731
        for _ in range(3):
            f_obs()
        _, ts = cuda_time_steps(f_obs, 10, torch)
        ms = statistics.median(ts)
        side["get_obs"] = {"workload": "2^22 envs, FrankaEnv._get_obs from kinematic state -> [obs19|ag3|dg3] rows",
                           "ms_per_launch": ms, "envs_per_s": n_o / (ms * 1e-3), "GBps_algorithmic": 228.0 * n_o / (ms * 1e-3) / 1e9,
                           "roofline": {"bound": "hbm", "achieved": 228.0 * n_o / (ms * 1e-3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                        "frac": 228.0 * n_o / (ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
                                        "algorithmic": "228 B/env (128 in + 100 out)", "kernel": "get_obs_bulk_kernel<SpecKin>"}}
        # K3/K4: mj_kinematics + mj_jacSite + mju_mat2Quat for the EE site (28 B in, 12 + 16 + 168 B out per configuration)
        n_f = 1 << 22
        qf = synthetic.random_joint_configs(n_f, tree.lower, tree.upper, seed=9, device=dev)
        f_fk = lambda: engine.fk_jac(qf)  # noqa: E731
        for _ in range(3):
            f_fk()
        _, ts = cuda_time_steps(f_fk, 10, torch)
        ms = statistics.median(ts)
        side["fk_jac"] = {"workload": "2^22 joint configurations -> EE position, wxyz quaternion, 6x7 Jacobian (FP32)",
                          "ms_per_launch": ms, "configs_per_s": n_f / (ms * 1e-3), "GBps_algorithmic": 224.0 * n_f / (ms * 1e-3) / 1e9,
                          "roofline": {"bound": "hbm", "achieved": 224.0 * n_f / (ms * 1e-3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                       "frac": 224.0 * n_f / (ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
                                       "algorithmic": "224 B/configuration (28 in + 12 + 16 + 168 out)", "kernel": "fk_jac_bulk_kernel<SpecKin>"},
                          "note": "includes the torch.empty of the three outputs"}
        del qf
        # SURVEY 8f-4: pose-mode (6x6) IK extension, reachable poses near neutral
        n_p = 1 << 20
        qp = synthetic.reachable_move_envs(n_p, tree.lower, tree.upper, seed=5, device=dev, spread=0.5)["q_goal"]
        ppos, pquat, _ = engine.fk_jac(qp, want_jac=False)
        cntp = torch.zeros(4, dtype=torch.int64, device=dev)
        engine.ik_pose_solve(ppos, pquat, neutral, params, counters=cntp)
        torch.cuda.synchronize()
        cpp = cntp.cpu().numpy()
        _, ts = cuda_time_steps(lambda: engine.ik_pose_solve(ppos, pquat, neutral, params), 3, torch)
        side["pose_ik"] = {"workload": "2^20 pose targets FK(neutral +- 0.5 rad), cold from neutral, 6-row DLS",
                           "ms_per_launch": min(ts), "solves_per_s": n_p / (min(ts) * 1e-3),
                           "converged": float(cpp[1]) / n_p, "mean_iterations": float(cpp[3]) / n_p}
    clocks = sampler.stop()

    # ---------------- CPU baselines (rank 0, N=1 only) ----------------------------------
    cpu_ik = cpu_rw = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_ik = cpu_ik_baseline()
        cpu_rw = cpu_reward_baseline()
        lat = cpu_latency_baselines(targets[:4096].double().cpu().numpy())
        for key in ("cfg1", "cfg2", "reward_scalar"):
            if key in side:
                side[key]["cpu"] = lat[key]
    D.barrier()

    if rank == 0:
        latency = {k: side.pop(k) for k in ("cfg1", "cfg2", "reward_scalar") if k in side}
        ik_roofline = {
            "bound": "fp32", "achieved": ik_tflops, "peak": fp32_peak, "unit": "TFLOP/s",
            "frac": ik_tflops / fp32_peak, "frac_of_nominal_74.4": ik_tflops / 74.4,
            "traffic": ncu_traffic("ik_solve_v_kernel" if specialized else "ik_solve_kernel", n_ik),
            "traffic_note": "DRAM bytes/launch from the ncu capture (48 B/query; algorithmic 60 B, part of the output is still in L2 at kernel end)",
            "kernel": ("ik_solve_v_kernel<F2,packed,bcast> (two queries per lane on FFMA2/FMUL2/FADD2)" if specialized
                       else "ik_solve_kernel<float,GenericKin,packed>"),
            "kernel_ms": ik_kernel_ms,
            "kernel_ms_single_launch": ik_single_ms,
            "kernel_ms_note": "kernel_ms = timed region / steps, launches back to back into alternating output sets (consecutive "
                              "launches overlap drain and ramp, programmatic dependent launch); single_launch = one launch alone",
            "peak_source": "pnp_probe_fp32_peak, measured in this run (no FP32 entry in MEASURED_PEAKS.json; nominal 148 x 128 x 2 x 1.965 GHz = 74.4)",
            "algorithmic": f"{IK_FLOP_PER_ITER:.0f} FLOP x iterations + {IK_FLOP_PER_SOLVE:.0f} per solve (SURVEY 8d)",
        }
        rw_roofline = {"bound": "hbm", "achieved": rw_gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                       "frac": rw_gbs / peaks["hbm_gbs"], "traffic": ncu_traffic("reward_kernel", n_rw),
                       "kernel": "reward_kernel<float,true>", "kernel_ms": rw_kernel_ms, "peak_source": peaks["source"],
                       "algorithmic": "64 B/row (60 in + 4 out)"}
        rw_e2e_d = {"value": rw_e2e, "unit": "rows/s", "h2d_bytes_per_step": n_rw * 60, "d2h_bytes_per_step": n_rw * 4,
                    "api": "pnp_reward_host_f32",
                    "note": "host-resident rows are PCIe bound (64 B/row over a ~57 GB/s link): about the speed of the CPU "
                            "port; the GPU reward pays when the rows are already resident (value, her_relabel)"}
        e2e = {"value": ik_e2e, "unit": "solves/s", "h2d_bytes_per_step": ik_h2d, "d2h_bytes_per_step": ik_d2h,
               "steps": K, "api": "pnp_ik_solve_packed_host_f32 (pinned host buffers, 3-stream chunk pipeline)", "link": link}
        e2e_compact = {"value": ik_e2e_c, "unit": "solves/s", "h2d_bytes_per_step": ik_h2d, "d2h_bytes_per_step": n_ik * 32 + 32,
                       "steps": K, "api": "pnp_ik_solve_compact_host_f32 (q, iterations, converged, success; no final_pos / pos_error)"}
        line = {
            "metric": "panda_ik_converged_solves_per_s", "value": ik_value, "unit": "solves/s", "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": ik_ms_total / K, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": bench_config(world, args.log2_n_ik, args.log2_n_reward),
            "workload_stats": {"kinematics": "specialized" if specialized else "generic",
                               "success_rate": float(c[2]) / float(c[0]), "mean_iterations": float(c[3]) / float(c[0]),
                               "numa_bound_cpus": numa, "threshold_adjacent_reward_rows": int(rw_counters[3].item())},
            "e2e": e2e,
            "e2e_compact": e2e_compact,
            "gpu_launches": int(launches_ik),
            "clocks": clocks,
            "roofline": ik_roofline,
            "cpu_baseline": cpu_ik,
            **side,
            "latency": latency,
            "reward": {
                "metric": "her_reward_evals_per_s", "value": rw_value, "unit": "rows/s",
                "workload": f"cfg3 dense reward, 2^{args.log2_n_reward} HER-relabelled rows per GPU, FP32 storage",
                "ms_per_step": rw_ms_total / K, "e2e": rw_e2e_d, "roofline": rw_roofline, "cpu_baseline": cpu_rw,
            },
            # both halves of BASELINE.json's metric once more, LAST on the line (the driver keeps the tail)
            "headline": {
                "ik": {"solves_per_s": ik_value, "roofline_frac": ik_tflops / fp32_peak, "e2e_solves_per_s": ik_e2e,
                       "e2e_compact_solves_per_s": ik_e2e_c, "e2e_link_ceiling_solves_per_s": link["ceiling_solves_per_s"],
                       "cpu_port_solves_per_s": cpu_ik["value"] if cpu_ik else None, "cpu_cores": cpu_ik["cores"] if cpu_ik else None},
                "reward": {"rows_per_s": rw_value, "roofline_frac": rw_gbs / peaks["hbm_gbs"], "GBps": rw_gbs,
                           "e2e_rows_per_s": rw_e2e, "cpu_port_rows_per_s": cpu_rw["value"] if cpu_rw else None},
                "latency_us": {k: (v.get("us_per_solve_host_to_host") or v.get("us_per_launch") or v.get("us_per_call_host_to_host"))
                               for k, v in latency.items()},
            },
        }
        if dump:
            write_dump(args.dump_outputs, ik_rows, ik_dump["q8"], ik_dump["aux4"], rw_rows, rw_dump)
        emit(line)
    if world > 1:
        import torch.distributed as dist

        dist.destroy_process_group()
    return 0


_JSON_FD = None


def emit(line: dict) -> None:
    """Write the one JSON line to the real stdout (see main(): fd 1 is pointed at stderr meanwhile)."""
    data = (json.dumps(line) + "\n").encode()
    os.write(_JSON_FD if _JSON_FD is not None else 1, data)


def main() -> int:
    global _JSON_FD
    # Libraries write banners to stdout from C (NCCL prints "NCCL version ..." on init).  The
    # contract is ONE JSON line on stdout, so keep a private handle on the real stdout and point
    # fd 1 / sys.stdout at stderr for everything else.
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = sys.stderr
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--log2-n-ik", type=int, default=LOG2_N_IK)
    ap.add_argument("--log2-n-reward", type=int, default=LOG2_N_REWARD)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write a seeded sample of the last timed step's outputs to DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs records the GPU path (--impl ours)")
    if args.warmup < 3:
        args.warmup = 3  # timing rule: at least 3 warm-up steps
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())

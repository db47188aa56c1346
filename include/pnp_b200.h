/*
 * pnp_b200.h - C ABI of libpnp_b200.so: the B200 (sm_100a) implementation of the
 * mujoco-panda-pnp hot path (Panda position IK + goal-conditioned reward).
 *
 * Drop-in boundary.  The reference has no native FFI: its hot path is Python calling
 * MuJoCo / NumPy.  Each entry point below replaces one reference interface:
 *
 *   pnp_set_tree           model data read by JacobianIKController.__init__
 *                          (panda_mujoco_gym/skills/ik_solver.py:27-33) and by MuJoCo inside
 *                          mj_kinematics / mj_jacSite (ik_solver.py:58,72)
 *   pnp_fk_jac_*           mujoco.mj_kinematics + mujoco.mj_jacSite + mju_mat2Quat for the EE
 *                          site (ik_solver.py:58-59,70-72; envs/panda_env.py:337-346)
 *   pnp_ik_solve_*         JacobianIKController.solve (ik_solver.py:35-101), batched
 *   pnp_ik_waypoints_*     the warm-started solve sequence of MoveIKSkill.reset
 *                          (skills/move.py:106-137), fixed number of waypoints per env
 *   pnp_ik_pose_solve_*    FrankaEnv.solve_ik(target_pos, target_quat, q_init) (panda_env.py:399-409;
 *                          dangling in the reference - an extension defined here)
 *   pnp_ik_axis_solve_*    a tool position and approach direction, the roll about the tool axis free (an extension
 *                          defined here)
 *   pnp_ik_axis_cone_solve_*  the same with the approach direction anywhere within a cone (an extension defined here)
 *   pnp_move_ik_plan_*     the whole MoveIKSkill.reset planner (skills/move.py:76-191)
 *   pnp_move_ik_plan_pose_*  the same planner to a goal position and orientation (an extension defined here)
 *   pnp_move_ik_plan_axis_*  the same planner to a goal position and tool-axis direction, the roll free (an
 *                          extension defined here)
 *   pnp_get_obs_*          FrankaEnv._get_obs (envs/panda_env.py:279-301) from kinematic state
 *   pnp_reward_*           FrankaEnv.compute_reward / _is_success / goal_distance
 *                          (envs/panda_env.py:205-245, 303-306, 311-315), row-wise
 *   pnp_her_relabel_f32,   HER goal relabel + reward + VecNormalize over stored transitions
 *   pnp_her_relabel_table_f32   (scripts/train.py:4,68,74-93; SB3 HerReplayBuffer semantics)
 *   pnp_*_host             the same operators taking HOST buffers (what a Python/ctypes
 *                          caller of the reference API holds): chunked H2D -> kernel -> D2H
 *                          pipeline on library-owned streams
 *
 * Conventions
 *   - Plain C types only.  "_dev" style entry points (no suffix) take DEVICE pointers and a
 *     cudaStream_t passed as void*; they never allocate, never synchronise and never throw.
 *   - Every function returns 0 on success or a negative PNP_E* code / positive cudaError_t.
 *     pnp_last_error() returns a thread-local message for the last failure.
 *   - Outputs are overwritten.  `counters` (nullable) is ACCUMULATED with atomics; the caller
 *     zeroes it.  Any output pointer documented "nullable" may be NULL to skip that store.
 *   - _f32 kernels compute in FP32 registers (the product path); _f64 kernels run the same
 *     algorithm in FP64 (used to separate algorithmic parity from FP32 rounding).
 *   - Arm joints are qpos[0:7] (ik_solver.py:31-33,51).  Quaternions are wxyz (MuJoCo).
 */
#ifndef PNP_B200_H_
#define PNP_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PNP_ABI_VERSION 3
#define PNP_NJOINT 7

/* error codes (negative; positive values are cudaError_t) */
#define PNP_OK 0
#define PNP_EINVAL (-1)      /* bad argument (null pointer, negative size, bad enum) */
#define PNP_ENOTREE (-2)     /* pnp_set_tree has not been called on this device */
#define PNP_ENODEVICE (-3)   /* no CUDA device / wrong architecture (needs sm_100) */
#define PNP_ENOMEM (-4)      /* host-API scratch allocation failed */

/* Canonical 7-hinge chain (FP64, host memory).  See mujoco_panda_pnp_b200/tree.py:
 *   frame_0 = I;  A_i = frame_i * Fixed(link_pos[i], link_rot[i]);
 *   frame_{i+1} = A_i * Rz(q_i - qref[i]);  site = frame_7 * Fixed(ee_pos, ee_rot)
 * Rotations are row-major 3x3.  lower/upper = model.jnt_range[:7] (ik_solver.py:32-33). */
typedef struct PnpTree {
  int32_t njoint;   /* must be PNP_NJOINT */
  int32_t reserved;
  double link_pos[PNP_NJOINT * 3];
  double link_rot[PNP_NJOINT * 9];
  double ee_pos[3];
  double ee_rot[9];
  double lower[PNP_NJOINT];
  double upper[PNP_NJOINT];
  double qref[PNP_NJOINT];
} PnpTree;

/* JacobianIKController.solve keyword arguments (ik_solver.py:35-37), same defaults upstream */
typedef struct PnpIkParams {
  int32_t max_iters;   /* 100  */
  int32_t kinematics;  /* PNP_KIN_AUTO / _GENERIC / _SPECIALIZED */
  double pos_thresh;   /* 1e-3 */
  double damping;      /* 1e-2, added un-squared: J J^T + damping * I (ik_solver.py:79) */
  double step_limit;   /* 0.1  */
} PnpIkParams;

#define PNP_KIN_AUTO 0         /* specialised code when the uploaded tree matches it, else generic */
#define PNP_KIN_GENERIC 1      /* always read the tree from __constant__ memory */
#define PNP_KIN_SPECIALIZED 2  /* require the build-time specialised tree (error if mismatch) */
/* FP32 position IK (pnp_ik_solve_f32 / _packed_f32 and the host-buffer variants), pnp_ik_waypoints_f32 and
 * pnp_move_ik_plan*_f32; elsewhere they mean PNP_KIN_SPECIALIZED.  Same arithmetic, bit-identical results,
 * different lane mapping: */
#define PNP_KIN_SPEC_LANE 3    /* one query / env per lane, explicit-FMA specialised code (what AUTO picks for the
                                  waypoint and planner kernels and for small IK batches) */
#define PNP_KIN_SPEC_PAIR 4    /* two queries / envs per lane on packed FFMA2/FMUL2/FADD2 (what AUTO picks for
                                  FP32 IK batches of > 256 queries per SM on the specialised tree) */

/* flags[] bits written by the IK kernels (IKResult.converged / .success, ik_solver.py:92-100) */
#define PNP_IK_CONVERGED 1u
#define PNP_IK_SUCCESS 2u

/* counters[] layout for the IK kernels: the 4 values reduced across GPUs (SURVEY 8e) */
#define PNP_IK_CNT_N 0
#define PNP_IK_CNT_CONVERGED 1
#define PNP_IK_CNT_SUCCESS 2
#define PNP_IK_CNT_ITERATIONS 3

/* env scalars read by compute_reward (panda_env.py:205-245; shelf_pnp.py:17-26) */
typedef struct PnpRewardParams {
  int32_t sparse;                /* reward_type == "sparse" */
  int32_t n_tasks;               /* len(task_sequence) */
  double initial_object_height;  /* panda_env.py:139-141 */
  double distance_threshold;     /* 0.05 */
  double high_pick_z;            /* 0.35 */
  double threshold_report_tol;   /* rows with |d - threshold| < tol are counted (1e-6) */
} PnpRewardParams;

/* counters[] layout for the reward kernels */
#define PNP_RW_CNT_N 0
#define PNP_RW_CNT_PLACED 1
#define PNP_RW_CNT_GRIPPED 2
#define PNP_RW_CNT_THRESHOLD_ADJACENT 3

/* ---- library / device ------------------------------------------------------------------ */
int pnp_abi_version(void);
const char* pnp_last_error(void);
/* sm count, clock (kHz), compute capability major*10+minor of the current device */
int pnp_device_info(int32_t* sm_count, int32_t* clock_khz, int32_t* cc);

/* ---- kinematic tree -------------------------------------------------------------------- */
/* Upload the chain to __constant__ memory of the current device (FP64 and FP32 copies). */
int pnp_set_tree(const PnpTree* host_tree);
int pnp_get_tree(PnpTree* host_tree_out);
/* 1 when the uploaded tree is bit-identical to the build-time specialised one */
int pnp_tree_is_specialized(void);
/* copy of the tree the specialised kernels were generated for */
int pnp_get_specialized_tree(PnpTree* host_tree_out);

/* ---- FK + 6x7 geometric Jacobian (mj_kinematics + mj_jacSite + mju_mat2Quat) ------------- */
/* q[n,7] -> pos[n,3], quat[n,4] (wxyz, nullable), jac[n,6,7] row-major rows 0-2 jacp, 3-5 jacr
 * (nullable).  kinematics: PNP_KIN_*. */
int pnp_fk_jac_f32(const float* q, int64_t n, float* pos, float* quat, float* jac, int32_t kinematics, void* stream);
int pnp_fk_jac_f64(const double* q, int64_t n, double* pos, double* quat, double* jac, int32_t kinematics, void* stream);

/* ---- batched JacobianIKController.solve ------------------------------------------------- */
/* targets[n,3]; q_init[n,7] when q_init_stride == 7 or one broadcast [7] when 0.
 * Outputs: q_out[n,7], final_pos[n,3] (nullable), pos_err[n] (nullable), iters[n] int32
 * (nullable), flags[n] uint8 (nullable), counters[4] uint64 (nullable, accumulated). */
int pnp_ik_solve_f32(const float* targets, const float* q_init, int32_t q_init_stride, int64_t n,
                     const PnpIkParams* params, float* q_out, float* final_pos, float* pos_err,
                     int32_t* iters, uint8_t* flags, unsigned long long* counters, void* stream);
/* FP32 IK kernels evaluate sin/cos of the joint angles by table look-up with a one-term magic-number range reduction:
 * 1.8e-7 absolute inside +-2 pi (the joint range; a q_init outside the joint limits is fine), growing by 2.8e-8 per
 * radian beyond; the index arithmetic needs |q| < 3.2e3 rad.
 * Stream semantics of the FP32 solves on the build-time tree: two consecutive launches of > 128 queries per SM on one
 * stream with nothing between them overlap their drain / ramp (programmatic dependent launch) unless the second one reads
 * or overwrites memory of the first (the library compares the byte ranges and falls back to plain stream order); from
 * 16384 queries per SM up a launch is followed by a small resume launch that finishes its last stragglers.  Neither
 * changes a result bit.  The first such launch on a stream allocates 6 MB of device scratch (cudaMalloc: one device
 * synchronisation).  Captured launches (CUDA graphs) keep plain stream order.  The restart kernels of
 * pnp_ik_solve_multistart_* are plain launches (no programmatic-serialization attribute, no early trigger): an IK launch
 * queued after a multistart call cannot start before the call's last kernel has completed.  See INTEGRATION.md section 4. */
/* Same solve with PACKED outputs (the fast path: 3 x 128-bit stores per query instead of 13):
 *   out_q8  [n][8] float = q0..q6, pos_error
 *   out_aux4[n][4] float = final_pos xyz, then a 32-bit word (iterations | flags << 24)
 * Both 16-byte aligned.  n < 2^31 per call for all IK entry points. */
int pnp_ik_solve_packed_f32(const float* targets, const float* q_init, int32_t q_init_stride, int64_t n,
                            const PnpIkParams* params, float* out_q8, float* out_aux4,
                            unsigned long long* counters, void* stream);
/* COMPACT outputs: one 32-byte record per query, out_q8[n][8] float = q0..q6, then the 32-bit word
 * (iterations | flags << 24).  final_pos / pos_error are not written (final_pos = FK(q): pnp_fk_jac_f32; a converged
 * query lies within pos_thresh of its target by construction).  For callers that want IKResult.q / .success /
 * .converged / .iterations only: 2/3 of the bytes of the packed layout, which is what the host-buffer operator
 * spends its time moving. */
int pnp_ik_solve_compact_f32(const float* targets, const float* q_init, int32_t q_init_stride, int64_t n,
                             const PnpIkParams* params, float* out_q8, unsigned long long* counters, void* stream);
int pnp_ik_solve_f64(const double* targets, const double* q_init, int32_t q_init_stride, int64_t n,
                     const PnpIkParams* params, double* q_out, double* final_pos, double* pos_err,
                     int32_t* iters, uint8_t* flags, unsigned long long* counters, void* stream);
/* ---- multi-start solve: restart the queries that attempt 0 did not solve from a shared seed table ---------------- */
/* Attempt 0 is the plain solve of the same layout (pnp_ik_solve_f32 / _packed_f32 / _f64) from q_init, same params,
 * same kernel choice.  For every query whose attempt 0 is not a success, attempts 1..n_seeds solve the same target from
 * seeds[k - 1] (seeds[n_seeds][7], q_init semantics: may lie outside the limits), same params.  A query returns the
 * record of its FIRST successful attempt in the order 0, 1, ..., n_seeds, or attempt 0's when none succeeds; every output
 * field is bit-identical to the plain entry point's result for that target from that start.  0 <= n_seeds <= 255;
 * n_seeds = 0 is the plain solve (no extra kernel launch).
 *   attempt[n]        uint8 (nullable): the attempt returned
 *   counters[4]       (nullable, accumulated): as pnp_ik_solve_*, over the RETURNED records
 *   restart_stats[3]  (nullable, accumulated): queries that entered restarts, queries rescued, DLS passes run by restart
 *                     attempts (the cost; >= the iterations of the returned restart attempts)
 *   scratch           device memory, 16-byte aligned, pnp_ik_multistart_scratch_bytes(n) bytes; required
 * The separate layouts need flags (non-null: the restarts read attempt 0's success from it).  seeds and scratch must not
 * overlap an output.  The call never synchronises the host (it can be captured in a CUDA graph): the restarts run in
 * ceil(n_seeds / G) waves that read their list lengths on the device.  They are plain launches, so a library IK launch
 * queued after a multistart call on the same stream starts only once the multistart has completed. */
int pnp_ik_multistart_scratch_bytes(int64_t n, int64_t* bytes);
int pnp_ik_solve_multistart_f32(const float* targets, const float* q_init, int32_t q_init_stride, int64_t n,
                                const float* seeds, int32_t n_seeds, const PnpIkParams* params, float* q_out,
                                float* final_pos, float* pos_err, int32_t* iters, uint8_t* flags, uint8_t* attempt,
                                unsigned long long* counters, unsigned long long* restart_stats, void* scratch,
                                void* stream);
int pnp_ik_solve_multistart_packed_f32(const float* targets, const float* q_init, int32_t q_init_stride, int64_t n,
                                       const float* seeds, int32_t n_seeds, const PnpIkParams* params, float* out_q8,
                                       float* out_aux4, uint8_t* attempt, unsigned long long* counters,
                                       unsigned long long* restart_stats, void* scratch, void* stream);
int pnp_ik_solve_multistart_f64(const double* targets, const double* q_init, int32_t q_init_stride, int64_t n,
                                const double* seeds, int32_t n_seeds, const PnpIkParams* params, double* q_out,
                                double* final_pos, double* pos_err, int32_t* iters, uint8_t* flags, uint8_t* attempt,
                                unsigned long long* counters, unsigned long long* restart_stats, void* scratch,
                                void* stream);
/* Launch scratch (the refill ticket of the IK / waypoint / pose / planner kernels, the plan-order histograms) is kept
 * per STREAM: any number of launches may be queued on a stream, and up to 64 distinct streams per device may have
 * library launches in flight at the same time.  A captured CUDA graph keeps the scratch of its capture stream - do
 * not replay it concurrently with other library launches issued on that same stream object. */

/* ---- warm-started waypoint sequences (MoveIKSkill.reset inner loop, move.py:106-137) ----- */
/* Per env: start joints q_start[n,7], goal[n,3].  n_steps times: pos = FK(q); dist = |goal-pos|;
 * step = min(step_size, 0.1*dist, 0.02); next = pos + dir*step/dist (or goal when dist<=step);
 * solve(next, q) with `params`; accept iff success and pos_err < 2*step_size (move.py:131).
 * q is carried in registers across the n_steps solves (one launch).  Outputs: q_out[n,7],
 * pos_out[n,3] final EE position, n_accepted[n] int32 (nullable), iters_total[n] int32
 * (nullable), counters[4] (nullable; N counts solves = n*n_steps). */
int pnp_ik_waypoints_f32(const float* q_start, const float* goal, int64_t n, int32_t n_steps,
                         double step_size, const PnpIkParams* params, float* q_out, float* pos_out,
                         int32_t* n_accepted, int32_t* iters_total, unsigned long long* counters,
                         void* stream);

/* ---- pose-mode IK: 6-row task, 6x6 solve (EXTENSION, fills FrankaEnv.solve_ik, panda_env.py:399-409) */
/* target_pos[n,3], target_quat[n,4] wxyz (normalised on load).  e = [pos error; rot_weight * rotation
 * vector of target (x) conj(site quat)] in the world frame, J = [jacp; rot_weight * jacr],
 * dq = J^T (J J^T + damping I6)^-1 e, same clips and loop semantics as pnp_ik_solve_*; converged
 * when |pos error| < pos_thresh and |rotation vector| < rot_thresh.  The reference has no such
 * function (it imports a missing name), so parity is against this repo's own FP64 restatement.
 * Outputs: q_out[n,7], final_pos[n,3], final_quat[n,4], pos_err[n], rot_err[n] (rad), iters, flags
 * (all but q_out nullable), counters[4] (nullable). */
int pnp_ik_pose_solve_f32(const float* target_pos, const float* target_quat, const float* q_init,
                          int32_t q_init_stride, int64_t n, const PnpIkParams* params, double rot_thresh,
                          double rot_weight, float* q_out, float* final_pos, float* final_quat, float* pos_err,
                          float* rot_err, int32_t* iters, uint8_t* flags, unsigned long long* counters,
                          void* stream);
int pnp_ik_pose_solve_f64(const double* target_pos, const double* target_quat, const double* q_init,
                          int32_t q_init_stride, int64_t n, const PnpIkParams* params, double rot_thresh,
                          double rot_weight, double* q_out, double* final_pos, double* final_quat,
                          double* pos_err, double* rot_err, int32_t* iters, uint8_t* flags,
                          unsigned long long* counters, void* stream);
/* Multi-start pose solve: pnp_ik_pose_solve_* from q_init (attempt 0, unchanged), then, for every query whose attempt 0
 * is not a success, attempts 1..n_seeds solve the same pose from seeds[k - 1] (seeds[n_seeds][7], q_init semantics),
 * same params.  A query returns the record of its FIRST successful attempt in the order 0, 1, ..., n_seeds, or attempt
 * 0's when none succeeds; every output (q_out, final_pos, final_quat, pos_err, rot_err, iters, flags; nullable as in
 * pnp_ik_pose_solve_*) is bit-identical to the plain entry point's for that target from that start.  0 <= n_seeds <= 255;
 * n_seeds = 0 is the plain pose solve plus attempt zeroed (no extra kernel launch).
 *   flags             required (the restarts read attempt 0's success from it)
 *   attempt[n]        uint8 (nullable): the attempt returned
 *   counters[4]       (nullable, accumulated): as pnp_ik_pose_solve_*, over the RETURNED records
 *   restart_stats[3]  (nullable, accumulated): queries that entered restarts, queries rescued, DLS passes run by restart
 *                     attempts (>= the iterations of the returned restart attempts)
 *   scratch           device memory, 16-byte aligned, pnp_ik_multistart_scratch_bytes(n) bytes; required
 * seeds and scratch must not overlap an output or each other.  Like pnp_ik_solve_multistart_*, the call never
 * synchronises the host (it can be captured in a CUDA graph) and its restart waves are plain launches. */
int pnp_ik_pose_solve_multistart_f32(const float* target_pos, const float* target_quat, const float* q_init,
                                     int32_t q_init_stride, int64_t n, const float* seeds, int32_t n_seeds,
                                     const PnpIkParams* params, double rot_thresh, double rot_weight, float* q_out,
                                     float* final_pos, float* final_quat, float* pos_err, float* rot_err, int32_t* iters,
                                     uint8_t* flags, uint8_t* attempt, unsigned long long* counters,
                                     unsigned long long* restart_stats, void* scratch, void* stream);
int pnp_ik_pose_solve_multistart_f64(const double* target_pos, const double* target_quat, const double* q_init,
                                     int32_t q_init_stride, int64_t n, const double* seeds, int32_t n_seeds,
                                     const PnpIkParams* params, double rot_thresh, double rot_weight, double* q_out,
                                     double* final_pos, double* final_quat, double* pos_err, double* rot_err,
                                     int32_t* iters, uint8_t* flags, uint8_t* attempt, unsigned long long* counters,
                                     unsigned long long* restart_stats, void* scratch, void* stream);

/* ---- axis-constrained IK: tool position and approach direction, roll free (EXTENSION) ----- */
/* target_pos[n,3] and target_axis[n,3] (normalised on load) in the world frame; tool_axis[3] (host memory, one per
 * call, e.g. {0, 0, 1}: the packaged Panda's site +z, the approach direction) in the site frame.  The host normalises
 * t = tool_axis and completes it to the site-frame basis (u1, u2, t): u1 = normalize(t x e_k), e_k the basis vector of
 * t's smallest-magnitude component (lowest index on a tie), u2 = t x u1.  Each pass, with R the site frame:
 *   a = R t, b1 = R u1, b2 = R u2;  c = a x d, s = |c|, theta = atan2(s, a.d)   (d = the normalised target axis)
 *   n = c / s if s > 0;  b1 if s == 0 and a.d < 0;  0 otherwise
 *   e = [tp - p ; w theta n.b1 ; w theta n.b2],  J = [jacp ; w b1^T jacr ; w b2^T jacr]  (w = rot_weight)
 *   dq = J^T (J J^T + damping I5)^-1 e, same clips and loop semantics as pnp_ik_pose_solve_*;
 *   converged when |tp - p| < pos_thresh and theta < rot_thresh; success adds |tp - p| < 2 pos_thresh and
 *   theta < 2 rot_thresh.
 * The roll about t is whatever the solve reaches.  Outputs: q_out[n,7], final_pos[n,3], final_axis[n,3] (a),
 * final_quat[n,4] (site frame, wxyz), pos_err[n], axis_err[n] (theta, rad), iters, flags (all but q_out nullable),
 * counters[4] (nullable).  Rejected with PNP_EINVAL before anything is enqueued: a NULL, non-finite or zero tool_axis,
 * rot_thresh or rot_weight not > 0, NULL inputs or q_out, n >= 2^31.  The call never synchronises the host (it can be
 * captured in a CUDA graph).  The statement is oracle/axis_ik_oracle.py. */
int pnp_ik_axis_solve_f32(const float* target_pos, const float* target_axis, const float* q_init, int32_t q_init_stride,
                          int64_t n, const PnpIkParams* params, const double* tool_axis, double rot_thresh,
                          double rot_weight, float* q_out, float* final_pos, float* final_axis, float* final_quat,
                          float* pos_err, float* axis_err, int32_t* iters, uint8_t* flags, unsigned long long* counters,
                          void* stream);
int pnp_ik_axis_solve_f64(const double* target_pos, const double* target_axis, const double* q_init,
                          int32_t q_init_stride, int64_t n, const PnpIkParams* params, const double* tool_axis,
                          double rot_thresh, double rot_weight, double* q_out, double* final_pos, double* final_axis,
                          double* final_quat, double* pos_err, double* axis_err, int32_t* iters, uint8_t* flags,
                          unsigned long long* counters, void* stream);
/* Multi-start axis solve: pnp_ik_axis_solve_* from q_init (attempt 0, unchanged), then the restarts of
 * pnp_ik_pose_solve_multistart_* (same seeds, attempt, counters, restart_stats and scratch contract, flags required):
 * a query returns its FIRST successful attempt in the order 0, 1, ..., n_seeds, or attempt 0's when none succeeds, and
 * every output is bit-identical to the plain entry point's for that target from that start. */
int pnp_ik_axis_solve_multistart_f32(const float* target_pos, const float* target_axis, const float* q_init,
                                     int32_t q_init_stride, int64_t n, const float* seeds, int32_t n_seeds,
                                     const PnpIkParams* params, const double* tool_axis, double rot_thresh,
                                     double rot_weight, float* q_out, float* final_pos, float* final_axis,
                                     float* final_quat, float* pos_err, float* axis_err, int32_t* iters, uint8_t* flags,
                                     uint8_t* attempt, unsigned long long* counters, unsigned long long* restart_stats,
                                     void* scratch, void* stream);
int pnp_ik_axis_solve_multistart_f64(const double* target_pos, const double* target_axis, const double* q_init,
                                     int32_t q_init_stride, int64_t n, const double* seeds, int32_t n_seeds,
                                     const PnpIkParams* params, const double* tool_axis, double rot_thresh,
                                     double rot_weight, double* q_out, double* final_pos, double* final_axis,
                                     double* final_quat, double* pos_err, double* axis_err, int32_t* iters,
                                     uint8_t* flags, uint8_t* attempt, unsigned long long* counters,
                                     unsigned long long* restart_stats, void* scratch, void* stream);

/* ---- cone-tolerant axis IK: the approach direction anywhere within a cone (EXTENSION) -------- */
/* pnp_ik_axis_solve_* with cone_angle alpha in [0, pi] (radians, one per call): the tool axis a may end anywhere within
 * alpha of the target axis d.  With theta, n, b1, b2 as in the axis solve, each pass:
 *   on = theta > alpha (false for a NaN theta);  w' = rot_weight if on, else 0;  g = theta - alpha if on, else 0
 *   e = [tp - p ; w' g n.b1 ; w' g n.b2],  J = [jacp ; w' b1^T jacr ; w' b2^T jacr],  dq as in the axis solve;
 *   converged when |tp - p| < pos_thresh and theta - alpha < rot_thresh; success adds |tp - p| < 2 pos_thresh and
 *   theta - alpha < 2 rot_thresh.
 * Inside the cone the tilt rows are dropped, so the pass is the damped position pass and the axis moves freely within
 * the cone; alpha = 0 is the axis solve and alpha = pi the position solve.  axis_err stays theta, the true angle.
 * Outputs, counters, restarts, seeds and scratch as pnp_ik_axis_solve_* / pnp_ik_axis_solve_multistart_*.  Rejected
 * with PNP_EINVAL before anything is enqueued: everything the axis entry points reject, and a NaN, negative or > pi
 * cone_angle.  The call never synchronises the host (it can be captured in a CUDA graph).  The statement is
 * oracle/cone_ik_oracle.py. */
int pnp_ik_axis_cone_solve_f32(const float* target_pos, const float* target_axis, const float* q_init,
                               int32_t q_init_stride, int64_t n, const PnpIkParams* params, const double* tool_axis,
                               double rot_thresh, double cone_angle, double rot_weight, float* q_out, float* final_pos,
                               float* final_axis, float* final_quat, float* pos_err, float* axis_err, int32_t* iters,
                               uint8_t* flags, unsigned long long* counters, void* stream);
int pnp_ik_axis_cone_solve_f64(const double* target_pos, const double* target_axis, const double* q_init,
                               int32_t q_init_stride, int64_t n, const PnpIkParams* params, const double* tool_axis,
                               double rot_thresh, double cone_angle, double rot_weight, double* q_out,
                               double* final_pos, double* final_axis, double* final_quat, double* pos_err,
                               double* axis_err, int32_t* iters, uint8_t* flags, unsigned long long* counters,
                               void* stream);
int pnp_ik_axis_cone_solve_multistart_f32(const float* target_pos, const float* target_axis, const float* q_init,
                                          int32_t q_init_stride, int64_t n, const float* seeds, int32_t n_seeds,
                                          const PnpIkParams* params, const double* tool_axis, double rot_thresh,
                                          double cone_angle, double rot_weight, float* q_out, float* final_pos,
                                          float* final_axis, float* final_quat, float* pos_err, float* axis_err,
                                          int32_t* iters, uint8_t* flags, uint8_t* attempt, unsigned long long* counters,
                                          unsigned long long* restart_stats, void* scratch, void* stream);
int pnp_ik_axis_cone_solve_multistart_f64(const double* target_pos, const double* target_axis, const double* q_init,
                                          int32_t q_init_stride, int64_t n, const double* seeds, int32_t n_seeds,
                                          const PnpIkParams* params, const double* tool_axis, double rot_thresh,
                                          double cone_angle, double rot_weight, double* q_out, double* final_pos,
                                          double* final_axis, double* final_quat, double* pos_err, double* axis_err,
                                          int32_t* iters, uint8_t* flags, uint8_t* attempt,
                                          unsigned long long* counters, unsigned long long* restart_stats,
                                          void* scratch, void* stream);

/* ---- full MoveIKSkill.reset trajectory planner (skills/move.py:76-191) -------------------- */
typedef struct PnpMoveParams {
  double pos_thresh;        /* 0.01  MoveIKSkill.pos_thresh (move.py:66) */
  double step_size;         /* 0.01  MoveIKSkill.step_size */
  int32_t max_traj_points;  /* 200   MoveIKSkill.max_traj_points */
  int32_t max_outer;        /* bound on planner rounds; 0 = 4*max_traj_points + 64.  The reference
                               has no bound and never returns for unreachable targets. */
  int32_t traj_cap;         /* points of storage per env in traj (>= 2) */
  int32_t compute_order;    /* pnp_move_ik_plan_ordered_* only: 1 = `order` is scratch, fill it first
                               (pnp_move_plan_order_*) and then take the envs in that order; 0 = `order` is an input */
} PnpMoveParams;
#define PNP_MOVE_BROKE 1u      /* fallback strategies exhausted (reference `break`, move.py:178-180);
                                  pose / axis planner: three rejected solves in one round, or a non-finite / zero goal */
#define PNP_MOVE_CAPPED 2u     /* max_outer reached; pose / axis planner: max_traj_points points reached */
#define PNP_MOVE_OVERFLOW 4u   /* more than traj_cap points: extra points dropped, traj_len still counts */
/* Per env: q_start[n,7], target[n,3].  The whole adaptive-waypoint state machine (accept rule,
 * failure counting incl. the double increment, fallback strategies 1-3, final-point append) runs
 * on the device; every IK solve uses `params`.  Outputs: traj[n,traj_cap,3] = MoveIKSkill.pos_traj
 * (first point = FK(q_start)), traj_len[n], q_final[n,7] (= q_current after the loop),
 * n_solves[n] (nullable), status[n] (nullable, PNP_MOVE_* bits), counters[4] (nullable). */
int pnp_move_ik_plan_f32(const float* q_start, const float* target, int64_t n, const PnpMoveParams* move,
                         const PnpIkParams* params, float* traj, int32_t* traj_len, float* q_final,
                         int32_t* n_solves, int32_t* status, unsigned long long* counters, void* stream);
int pnp_move_ik_plan_f64(const double* q_start, const double* target, int64_t n, const PnpMoveParams* move,
                         const PnpIkParams* params, double* traj, int32_t* traj_len, double* q_final,
                         int32_t* n_solves, int32_t* status, unsigned long long* counters, void* stream);
/* Longest plan first.  A plan is 2-200 warm-started solves long (move.py:106-137) and its length follows
 * d0 = |target - FK(q_start)|; a launch that takes its envs in index order ends with most lanes idle behind
 * the last long plans.  pnp_move_plan_order_* writes order[n] = the env indices sorted by descending d0
 * (counting sort on 1/64 m buckets; the order inside a bucket is unspecified), pnp_move_ik_plan_ordered_*
 * takes its envs in that order (order NULL = index order; with move->compute_order = 1 it fills `order`
 * itself first, one call instead of two).  A caller-made `order` must be a permutation of [0, n).  The planner skips
 * an entry outside the batch (nothing is read or written for it); a repeated entry plans that env twice (same
 * outputs) and leaves another env unplanned.  pnp_move_plan_order_check tells: bitmap_scratch[(n + 31) / 32] is
 * device scratch, *n_bad (device, overwritten) = entries that are out of range or repeat an earlier one; 0 = a
 * permutation.  Every output stays indexed by env and is bit-identical to the unordered call; only the time changes. */
int pnp_move_plan_order_check(const uint32_t* order, int64_t n, uint32_t* bitmap_scratch, uint32_t* n_bad, void* stream);
int pnp_move_plan_order_f32(const float* q_start, const float* target, int64_t n, uint32_t* order,
                            int32_t kinematics, void* stream);
int pnp_move_plan_order_f64(const double* q_start, const double* target, int64_t n, uint32_t* order,
                            int32_t kinematics, void* stream);
int pnp_move_ik_plan_ordered_f32(const float* q_start, const float* target, uint32_t* order, int64_t n,
                                 const PnpMoveParams* move, const PnpIkParams* params, float* traj,
                                 int32_t* traj_len, float* q_final, int32_t* n_solves, int32_t* status,
                                 unsigned long long* counters, void* stream);
int pnp_move_ik_plan_ordered_f64(const double* q_start, const double* target, uint32_t* order, int64_t n,
                                 const PnpMoveParams* move, const PnpIkParams* params, double* traj,
                                 int32_t* traj_len, double* q_final, int32_t* n_solves, int32_t* status,
                                 unsigned long long* counters, void* stream);
/* Longest plan first with the inputs gathered: `scratch48` is device scratch of 48 bytes per env (16-byte aligned).
 * The call sorts like pnp_move_plan_order_f32 and writes the i-th env to plan as one record {q_start[7], target[3],
 * env} into it, so a lane that takes its next env does one sequential 48-byte read instead of order[i] ->
 * q_start[env], two dependent random ones (2^20 plans: 1.58 -> 1.34 ms).  Outputs are those of pnp_move_ik_plan_f32,
 * indexed by env, bit for bit.  (On a non-specialised tree the scratch serves as a plain order[n].) */
int pnp_move_ik_plan_sorted_f32(const float* q_start, const float* target, void* scratch48, int64_t n,
                                const PnpMoveParams* move, const PnpIkParams* params, float* traj,
                                int32_t* traj_len, float* q_final, int32_t* n_solves, int32_t* status,
                                unsigned long long* counters, void* stream);

/* ---- pose-mode move planner: plan to a goal position AND orientation (EXTENSION) ------------ */
typedef struct PnpMovePoseParams {
  double pos_thresh;       /* 0.01 m   the plan ends when |goal_pos - p| <= pos_thresh ...                        */
  double rot_thresh;       /* 0.05 rad ... and the remaining rotation angle <= rot_thresh                        */
  double step_size;        /* 0.01 m   largest translation per waypoint                                          */
  double rot_step;         /* 0.05 rad largest rotation per waypoint                                             */
  double ik_rot_thresh;    /* 0.01 rad rot_thresh of every pose solve (pnp_ik_pose_solve_*)                     */
  double ik_rot_weight;    /* 1.0      rot_weight of every pose solve                                            */
  int32_t max_traj_points; /* 200      solved waypoints at most                                                  */
  int32_t traj_cap;        /* >= 1     points of storage per env; max_traj_points + 1 never overflows           */
} PnpMovePoseParams;
/* Per env: q_start[n,7], goal_pos[n,3], goal_quat[n,4] wxyz (normalised on load).  (p, r) = FK(q_start) (site position
 * and quaternion) is point 0.  Each round: d = goal_pos - p, w = rotation vector of goal_quat (x) conj(r) (the pose
 * solver's error, short path).  The plan ends with status 0 when |d| <= pos_thresh and |w| <= rot_thresh, and with
 * PNP_MOVE_CAPPED after max_traj_points points.  Otherwise f = min(1, step_size / |d|, rot_step / |w|) and up to three
 * pose solves (pnp_ik_pose_solve_* from the current q with `params`, ik_rot_thresh, ik_rot_weight) aim at the fractions
 * f, f/2, f/20 of the remaining motion: (p + g d, quat(g w) (x) r), or exactly the goal when g == 1.  The first success
 * appends its (final_pos, final_quat, q) and moves there; three rejections end the plan with PNP_MOVE_BROKE, as does a
 * non-finite goal or a zero goal quaternion (then traj_len = 1).  The unreached goal is never appended: every point is a
 * solved pose, and pos_traj, quat_traj and q_traj line up.  traj_len <= max_traj_points + 1, n_solves <=
 * 3 max_traj_points; points past traj_cap are dropped and set PNP_MOVE_OVERFLOW (traj_len still counts them).
 * Outputs: pos_traj[n,traj_cap,3], quat_traj[n,traj_cap,4], q_traj[n,traj_cap,7] (nullable), traj_len[n], q_final[n,7]
 * (the joints of the last point), n_solves[n], status[n] (PNP_MOVE_* bits), counters[4] (nullable: every pose solve, as
 * pnp_ik_pose_solve_*).  Rejected with PNP_EINVAL before anything is enqueued: pos_thresh < params->pos_thresh or
 * rot_thresh < ik_rot_thresh (a solve converged short of the plan's tolerance would re-aim at the goal forever),
 * step_size or rot_step <= 0, NULL outputs other than q_traj and counters, n >= 2^31.  The call never synchronises the
 * host and can be captured in a CUDA graph.  The oracle is oracle/move_pose_oracle.py. */
int pnp_move_ik_plan_pose_f32(const float* q_start, const float* goal_pos, const float* goal_quat, int64_t n,
                              const PnpMovePoseParams* move, const PnpIkParams* params, float* pos_traj,
                              float* quat_traj, float* q_traj, int32_t* traj_len, float* q_final, int32_t* n_solves,
                              int32_t* status, unsigned long long* counters, void* stream);
int pnp_move_ik_plan_pose_f64(const double* q_start, const double* goal_pos, const double* goal_quat, int64_t n,
                              const PnpMovePoseParams* move, const PnpIkParams* params, double* pos_traj,
                              double* quat_traj, double* q_traj, int32_t* traj_len, double* q_final, int32_t* n_solves,
                              int32_t* status, unsigned long long* counters, void* stream);

/* ---- axis-mode move planner: plan to a goal position and tool-axis direction, roll free (EXTENSION) ---------------- */
/* Per env: q_start[n,7], goal_pos[n,3], goal_axis[n,3] (world frame, normalised on load); tool_axis[3] (host memory,
 * one per call, site frame) with its basis (t, u1, u2) as in pnp_ik_axis_solve_*.  PnpMovePoseParams as for the pose
 * planner, with rot_thresh, rot_step, ik_rot_thresh and ik_rot_weight applying to the axis angle theta.  (p, R) =
 * FK(q_start), a = R t: point 0 is (p, a, quat(R), q_start).  Each round: d = goal_pos - p, theta = atan2(|a x g|, a.g)
 * (g the goal axis, evaluated as the axis solver evaluates its error).  The plan ends with status 0 when |d| <=
 * pos_thresh and theta <= rot_thresh, and with PNP_MOVE_CAPPED after max_traj_points points.  Otherwise f = min(1,
 * step_size / |d|, rot_step / theta) and up to three axis solves (pnp_ik_axis_solve_* from the current q with `params`,
 * tool_axis, ik_rot_thresh, ik_rot_weight) aim at the fractions h = f, f/2, f/20 of the remaining motion:
 * (p + h d, normalize(cos(h theta) a + sin(h theta) m)) with m = (g - (a.g) a) / |a x g| the unit tangent turning a
 * toward g (m = -R u2 when a and g are exactly antiparallel, the solver's own choice of tilt direction), or exactly the
 * goal when h == 1.  The first success appends its (final_pos, final_axis, final_quat, q) and moves there; three
 * rejections end the plan with PNP_MOVE_BROKE, as does a non-finite goal or a zero goal axis (then traj_len = 1).  The
 * roll about t is whatever the solves reach.  The unreached goal is never appended: every point is a solved axis task,
 * and pos_traj, axis_traj, quat_traj and q_traj line up.  traj_len <= max_traj_points + 1, n_solves <=
 * 3 max_traj_points; points past traj_cap are dropped and set PNP_MOVE_OVERFLOW (traj_len still counts them).
 * Outputs: pos_traj[n,traj_cap,3], axis_traj[n,traj_cap,3] (a, world frame), quat_traj[n,traj_cap,4] (site frame,
 * wxyz), q_traj[n,traj_cap,7] (nullable), traj_len[n], q_final[n,7] (the joints of the last point), n_solves[n],
 * status[n] (PNP_MOVE_* bits), counters[4] (nullable: every axis solve, as pnp_ik_axis_solve_*).  Rejected with
 * PNP_EINVAL before anything is enqueued: everything pnp_move_ik_plan_pose_* rejects, a NULL, non-finite or zero
 * tool_axis, NULL outputs other than q_traj and counters.  The call never synchronises the host and can be captured in
 * a CUDA graph.  The oracle is oracle/move_axis_oracle.py. */
int pnp_move_ik_plan_axis_f32(const float* q_start, const float* goal_pos, const float* goal_axis, int64_t n,
                              const PnpMovePoseParams* move, const PnpIkParams* params, const double* tool_axis,
                              float* pos_traj, float* axis_traj, float* quat_traj, float* q_traj, int32_t* traj_len,
                              float* q_final, int32_t* n_solves, int32_t* status, unsigned long long* counters,
                              void* stream);
int pnp_move_ik_plan_axis_f64(const double* q_start, const double* goal_pos, const double* goal_axis, int64_t n,
                              const PnpMovePoseParams* move, const PnpIkParams* params, const double* tool_axis,
                              double* pos_traj, double* axis_traj, double* quat_traj, double* q_traj, int32_t* traj_len,
                              double* q_final, int32_t* n_solves, int32_t* status, unsigned long long* counters,
                              void* stream);

/* ---- compute_reward / _is_success, row-wise --------------------------------------------- */
/* Per row: achieved_goal[n,3], desired_goal[n,3], ee_pos[n,3], ee_quat[n,4] wxyz,
 * fingers_width[n], task_index[n] int32.  Math is FP64 in the reference's operation order
 * without FMA contraction, one final round-to-nearest cast to float (bit-exact).
 * reward[n] float; is_success[n] float (nullable); counters[4] (nullable). */
int pnp_reward_f32(const float* ag, const float* dg, const float* ee_pos, const float* ee_quat,
                   const float* width, const int32_t* task_index, int64_t n,
                   const PnpRewardParams* params, float* reward, float* is_success,
                   unsigned long long* counters, void* stream);
int pnp_reward_f64(const double* ag, const double* dg, const double* ee_pos, const double* ee_quat,
                   const double* width, const int32_t* task_index, int64_t n,
                   const PnpRewardParams* params, float* reward, float* is_success,
                   unsigned long long* counters, void* stream);
/* ---- HER relabel + obs assembly (what scripts/train.py:4 "TQC(+HER)" promises) ------------- */
/* VecNormalize.normalize_obs parameters (scripts/checkpoints/tqc_dense_vecnormalize_*.pkl):
 * rows are clip((x - mean) / sqrt(var + epsilon), +-clip_obs) per column of the 25-wide row. */
typedef struct PnpNormalizeParams {
  double mean[25];
  double var[25];
  double epsilon;   /* 1e-8 */
  double clip_obs;  /* 10.0 */
} PnpNormalizeParams;
/* obs / next_obs: float[n,25] = observation[19] | achieved_goal[3] | desired_goal[3] (the layout
 * pnp_get_obs_* writes).  Per transition i: new goal = next_obs[future_idx[i]].achieved_goal
 * (future_idx[i] < 0 keeps the stored goal); both rows get the new desired_goal; reward[i] =
 * compute_reward(next_obs[i].achieved_goal, new goal) with ee_pos = next_obs[i][0:3],
 * fingers_width = next_obs[i][6], ee_quat[n,4] and task_index[n] from the side arrays (bit-exact,
 * same arithmetic as pnp_reward_f32); is_success (nullable); rows optionally normalised (norm
 * nullable = copy through).  future_idx[i] >= n keeps the stored goal like a negative index.  Outputs must not
 * overlap the inputs or each other (checked by address range).  counters as pnp_reward_*. */
int pnp_her_relabel_f32(const float* obs, const float* next_obs, const int32_t* future_idx, const float* ee_quat,
                        const int32_t* task_index, int64_t n, const PnpRewardParams* params,
                        const PnpNormalizeParams* norm, float* out_obs, float* out_next_obs, float* reward,
                        float* is_success, unsigned long long* counters, void* stream);

/* Same operator with the future goals gathered from a separate table future_ag[n,3] (row j = the
 * achieved goal of next_obs[j]; what SB3's DictReplayBuffer keeps as next_observations["achieved_goal"])
 * instead of out of the 100-byte next_obs rows: the random 12-byte gather then hits a table that fits
 * the L2 instead of costing a 64-128 B DRAM burst per transition.  future_ag == NULL is
 * pnp_her_relabel_f32.  Identical results when the table matches next_obs[:, 19:22]. */
int pnp_her_relabel_table_f32(const float* obs, const float* next_obs, const int32_t* future_idx,
                              const float* future_ag, const float* ee_quat, const int32_t* task_index, int64_t n,
                              const PnpRewardParams* params, const PnpNormalizeParams* norm, float* out_obs,
                              float* out_next_obs, float* reward, float* is_success, unsigned long long* counters,
                              void* stream);

/* goal_distance (panda_env.py:311-315): a[n,3], b[n,3] -> d[n] (FP64 math) */
int pnp_goal_distance_f64(const double* a, const double* b, int64_t n, double* d, void* stream);

/* ---- FrankaEnv._get_obs from kinematic state (envs/panda_env.py:279-301) ------------------ */
/* Per env: q_arm[n,7], qvel_arm[n,7], fingers[n,2] (qpos of finger_joint1/2), the current target
 * cube's free-joint state obj_pos[n,3], obj_quat[n,4] wxyz, obj_vel[n,6] (linear world, angular
 * body-local: MuJoCo's free-joint qvel), goal[n,3] (goal_stride 3) or one goal[3] (stride 0).
 * dt = opt.timestep * n_substeps (0.002 * 25).  out[n,25] = observation[19] (ee_pos3, ee_vel3,
 * fingers_width, obj_pos3, obj_rot3 euler, obj_velp3, obj_velr3) | achieved_goal[3] | desired_goal[3]. */
int pnp_get_obs_f32(const float* q_arm, const float* qvel_arm, const float* fingers, const float* obj_pos,
                    const float* obj_quat, const float* obj_vel, const float* goal, int32_t goal_stride,
                    int64_t n, double dt, float* out, int32_t kinematics, void* stream);
int pnp_get_obs_f64(const double* q_arm, const double* qvel_arm, const double* fingers, const double* obj_pos,
                    const double* obj_quat, const double* obj_vel, const double* goal, int32_t goal_stride,
                    int64_t n, double dt, double* out, int32_t kinematics, void* stream);

/* ---- host-buffer operators (end-to-end path: copies inside) ----------------------------- */
typedef struct PnpHostCtx PnpHostCtx;
/* chunk_rows: rows per pipeline stage (0 = default).  Allocates device scratch + 3 streams. */
int pnp_host_ctx_create(PnpHostCtx** out, int64_t chunk_rows);
int pnp_host_ctx_destroy(PnpHostCtx* ctx);
/* Same arguments as pnp_ik_solve_f32 but every pointer is HOST memory (pinned for full
 * overlap; pageable works).  counters[4] is host memory, overwritten.  Blocks until done. */
int pnp_ik_solve_host_f32(PnpHostCtx* ctx, const float* targets, const float* q_init,
                          int32_t q_init_stride, int64_t n, const PnpIkParams* params, float* q_out,
                          float* final_pos, float* pos_err, int32_t* iters, uint8_t* flags,
                          unsigned long long* counters);
/* Packed-output variant (see pnp_ik_solve_packed_f32): out_q8[n][8], out_aux4[n][4] on the host. */
int pnp_ik_solve_packed_host_f32(PnpHostCtx* ctx, const float* targets, const float* q_init,
                                 int32_t q_init_stride, int64_t n, const PnpIkParams* params,
                                 float* out_q8, float* out_aux4, unsigned long long* counters);
/* ONE query, host in / host out, lowest latency - what JacobianIKController.solve(target_pos, q_init)
 * (ik_solver.py:35) costs when it is called one pose at a time (test/ik_test.py, MoveIKSkill in a BT).
 * No cudaMemcpy: the kernel reads target3 / q_init7 from, and writes the result to, a pinned host
 * mailbox mapped into the device address space; one launch + one stream synchronisation.
 * out12 = q0..q6, pos_error | final_pos xyz, word (iterations | flags << 24): the two packed records of
 * pnp_ik_solve_packed_f32.  FP32; same arithmetic as the batch kernels (bit-identical results on the
 * specialised tree).  One mailbox per ctx: concurrent single-query calls on a ctx are serialised by a lock. */
int pnp_ik_solve_one_host_f32(PnpHostCtx* ctx, const float* target3, const float* q_init7,
                              const PnpIkParams* params, float* out12);
/* Compact-output variant of pnp_ik_solve_packed_host_f32 (see pnp_ik_solve_compact_f32): 32 B per query come back
 * instead of 48. */
int pnp_ik_solve_compact_host_f32(PnpHostCtx* ctx, const float* targets, const float* q_init,
                                  int32_t q_init_stride, int64_t n, const PnpIkParams* params,
                                  float* out_q8, unsigned long long* counters);
/* ONE row, host in / host out, lowest latency - FrankaEnv.compute_reward(achieved_goal (3,), desired_goal (3,), info)
 * as FrankaEnv.step calls it once per env.step (envs/panda_env.py:176-181) and test/reward_test.py:71-72 once per
 * transition.  Same mapped-mailbox path as pnp_ik_solve_one_host_f32: one launch + one stream synchronisation, no
 * cudaMemcpy, no counters.  FP64 storage, bit-exact (same arithmetic as pnp_reward_f64).  is_success and bits
 * (placed | gripped << 1 | threshold_adjacent << 2) are nullable.  Single-query calls on one ctx are serialised by
 * a lock. */
int pnp_reward_one_host_f64(PnpHostCtx* ctx, const double* ag3, const double* dg3, const double* ee_pos3,
                            const double* ee_quat4, double fingers_width, int32_t task_index,
                            const PnpRewardParams* params, float* reward, float* is_success, uint32_t* bits);
int pnp_reward_host_f32(PnpHostCtx* ctx, const float* ag, const float* dg, const float* ee_pos,
                        const float* ee_quat, const float* width, const int32_t* task_index,
                        int64_t n, const PnpRewardParams* params, float* reward, float* is_success,
                        unsigned long long* counters);
int pnp_reward_host_f64(PnpHostCtx* ctx, const double* ag, const double* dg, const double* ee_pos,
                        const double* ee_quat, const double* width, const int32_t* task_index,
                        int64_t n, const PnpRewardParams* params, float* reward, float* is_success,
                        unsigned long long* counters);

/* ---- measurement helpers ---------------------------------------------------------------- */
/* FFMA throughput microbenchmark on the current device: the FP32 roofline denominator
 * (MEASURED_PEAKS.json has none).  Returns TFLOP/s (FMA = 2) and the elapsed ms. */
int pnp_probe_fp32_peak(double* tflops_out, double* ms_out);
/* number of kernel launches issued by this library since load (bench.py's gpu_launches) */
unsigned long long pnp_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* PNP_B200_H_ */

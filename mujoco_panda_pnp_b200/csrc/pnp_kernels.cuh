// Kernels of libpnp_b200.so (sm_100a).  See DESIGN.md for the rooflines and data layout.
#pragma once

#include <type_traits>

#include "pnp_common.cuh"

namespace pnp {

constexpr int IK_BLOCK = 128;  // (forcing 8 blocks/SM = 64 regs was measured: no gain, generic path spills)
constexpr unsigned FULL = 0xffffffffu;
#ifndef IK_PAIR_MIN_BLOCKS
#define IK_PAIR_MIN_BLOCKS 4
#endif

__device__ __forceinline__ unsigned long long warp_sum(unsigned long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
  return v;
}

// =============================================================================================
// FK + Jacobian: one lane per joint configuration.
// =============================================================================================
template <typename T, typename Kin>
__global__ void __launch_bounds__(128) fk_jac_kernel(const T* __restrict__ q, long long n, T* __restrict__ pos,
                                                     T* __restrict__ quat, T* __restrict__ jac) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n;
       i += (long long)gridDim.x * blockDim.x) {
    T s[NJ], c[NJ];
#pragma unroll
    for (int k = 0; k < NJ; ++k) sincos_t(q[i * NJ + k] - Kin::template qref<T>(k), &s[k], &c[k]);
    T p[3], J[42], R[9];
    Kin::template fk_full<T>(s, c, p, J, R);
    pos[i * 3 + 0] = p[0];
    pos[i * 3 + 1] = p[1];
    pos[i * 3 + 2] = p[2];
    if (quat) {
      T qu[4];
      mat2quat<T>(R, qu);
#pragma unroll
      for (int k = 0; k < 4; ++k) quat[i * 4 + k] = qu[k];
    }
    if (jac) {
#pragma unroll
      for (int k = 0; k < 42; ++k) jac[i * 42 + k] = J[k];
    }
  }
}

// =============================================================================================
// FrankaEnv._get_obs from kinematic state (panda_env.py:279-301): one lane per env.
//   ee_pos  = site_xpos(ee_center_site)                       (:285)  FK(q)
//   ee_vel  = (jacp @ qvel) * dt                              (:286)  only arm dofs 0..6 are non-zero
//   obj_pos = cube site = free-joint position                 (:290)
//   obj_rot = mat2euler(site_xmat)                            (:291)  gymnasium_robotics convention
//   obj_velp = free-joint linear velocity * dt                (:292)  site sits at the body origin
//   obj_velr = R(obj_quat) * local angular velocity * dt      (:293)  jacr columns = body axes
//   fingers_width = qpos(finger_joint1) + qpos(finger_joint2) (:296, :348-352)
// Output row [25] = observation[19] | achieved_goal[3] (= obj_pos) | desired_goal[3] (:297-301).
// =============================================================================================
__device__ __forceinline__ float atan2_t(float y, float x) { return atan2f(y, x); }
__device__ __forceinline__ double atan2_t(double y, double x) { return atan2(y, x); }

template <typename T>
struct ObsArgs {
  const T *q_arm, *qvel_arm, *fingers, *obj_pos, *obj_quat, *obj_vel, *goal;
  int goal_stride;  // 3 = per env, 0 = one broadcast goal
  long long n;
  T dt;
  T* out;  // [n][25]
};

// One lane per env, 128 envs per block tile.  The 25-wide output rows (100 B for FP32) are
// assembled in shared memory (row stride 25 words: conflict-free) and written out by the whole
// block as consecutive words, so every store instruction covers 128 contiguous bytes instead of
// 32 rows 100 B apart.
constexpr int OBS_TILE = 128;

template <typename T, typename Kin>
__global__ void __launch_bounds__(OBS_TILE) get_obs_kernel(const ObsArgs<T> a) {
  __shared__ T s_out[OBS_TILE * 25];
  const long long n_tiles = (a.n + OBS_TILE - 1) / OBS_TILE;
  for (long long t = blockIdx.x; t < n_tiles; t += gridDim.x) {
    const long long i = t * OBS_TILE + threadIdx.x;
    if (i < a.n) {
      T s[NJ], c[NJ], qv[NJ];
#pragma unroll
      for (int k = 0; k < NJ; ++k) {
        sincos_t(a.q_arm[i * NJ + k] - Kin::template qref<T>(k), &s[k], &c[k]);
        qv[k] = a.qvel_arm[i * NJ + k];
      }
      T p[3], J[21];
#pragma unroll
      for (int k = 0; k < 21; ++k) J[k] = T(0);
      Kin::template fk_jacp<T>(s, c, p, J);
      T* o = s_out + threadIdx.x * 25;
      o[0] = p[0]; o[1] = p[1]; o[2] = p[2];
#pragma unroll
      for (int r = 0; r < 3; ++r) {
        T acc = T(0);
#pragma unroll
        for (int j = 0; j < NJ; ++j) acc = acc + J[r * 7 + j] * qv[j];
        o[3 + r] = acc * a.dt;
      }
      o[6] = a.fingers[i * 2] + a.fingers[i * 2 + 1];
      // free-joint body pose: mj_kinematics normalises the quaternion, xmat = quat2mat
      T w = a.obj_quat[i * 4], x = a.obj_quat[i * 4 + 1], y = a.obj_quat[i * 4 + 2], z = a.obj_quat[i * 4 + 3];
      const T nrm = sqrt_t(w * w + x * x + y * y + z * z);
      if (nrm < T(1e-15)) { w = T(1); x = y = z = T(0); } else { w = w / nrm; x = x / nrm; y = y / nrm; z = z / nrm; }
      const T q00 = w * w, q01 = w * x, q02 = w * y, q03 = w * z, q11 = x * x, q12 = x * y, q13 = x * z;
      const T q22 = y * y, q23 = y * z, q33 = z * z;
      const T m00 = q00 + q11 - q22 - q33, m01 = T(2) * (q12 - q03), m02 = T(2) * (q13 + q02);
      const T m10 = T(2) * (q12 + q03), m11 = q00 - q11 + q22 - q33, m12 = T(2) * (q23 - q01);
      const T m20 = T(2) * (q13 - q02), m21 = T(2) * (q23 + q01), m22 = q00 - q11 - q22 + q33;
      const T ox = a.obj_pos[i * 3], oy = a.obj_pos[i * 3 + 1], oz = a.obj_pos[i * 3 + 2];
      o[7] = ox; o[8] = oy; o[9] = oz;
      // rotations.mat2euler
      const T cy = sqrt_t(m22 * m22 + m12 * m12);
      const bool cond = cy > T(4.0 * 2.220446049250313e-16);
      o[12] = -atan2_t(cond ? m01 : -m10, cond ? m00 : m11);  // one atan2 on selected arguments
      o[11] = -atan2_t(-m02, cy);
      o[10] = cond ? -atan2_t(m12, m22) : T(0);
      const T vx = a.obj_vel[i * 6], vy = a.obj_vel[i * 6 + 1], vz = a.obj_vel[i * 6 + 2];
      const T wx = a.obj_vel[i * 6 + 3], wy = a.obj_vel[i * 6 + 4], wz = a.obj_vel[i * 6 + 5];
      o[13] = vx * a.dt; o[14] = vy * a.dt; o[15] = vz * a.dt;
      o[16] = (m00 * wx + m01 * wy + m02 * wz) * a.dt;
      o[17] = (m10 * wx + m11 * wy + m12 * wz) * a.dt;
      o[18] = (m20 * wx + m21 * wy + m22 * wz) * a.dt;
      o[19] = ox; o[20] = oy; o[21] = oz;
      const T* g = a.goal + (long long)a.goal_stride * i;
      o[22] = g[0]; o[23] = g[1]; o[24] = g[2];
    }
    __syncthreads();
    const long long rows = (a.n - t * OBS_TILE < OBS_TILE) ? a.n - t * OBS_TILE : OBS_TILE;
    T* dst = a.out + t * OBS_TILE * 25;
    for (int k = threadIdx.x; k < rows * 25; k += OBS_TILE) dst[k] = s_out[k];
    __syncthreads();
  }
}

// =============================================================================================
// Batched JacobianIKController.solve: one LANE per query, persistent warps with lane refill.
// This scalar-template kernel serves FP64 (the parity kernel) and any non-specialised tree; FP32 on the
// specialised tree runs ik_solve_v_kernel below (same control flow, value-type arithmetic).
//
// Every pass of the loop evaluates FK/J/DLS once for all 32 lanes.  A lane whose query
// finished (converged, or max_iters passes done) stores its result and immediately takes the
// next unsolved query from a global ticket (warp-aggregated atomicAdd), so lanes of one warp
// work on queries at different iteration counts and the warp never idles on its slowest
// query.  Control flow per query is exactly ik_solver.py:57-101:
//   pass i (< max_iters): FK -> test -> (converged: iterations=i+1, stop) | update, i+1
//   pass i == max_iters : FK only -> final_pos, converged=false, iterations=max_iters
//
// Output layouts.  kPacked = false: the five separate arrays of pnp_ik_solve_*.  kPacked = true
// (pnp_ik_solve_packed_f32): two 16-byte aligned records per query,
//   out_q8  [n][8] = q0..q6, pos_error            (2 x 128-bit stores)
//   out_aux [n][4] = final_pos xyz, bits(iterations | flags << 24)   (1 x 128-bit store)
// which cuts the per-finish store sequence from 13 STG.32 to 3 STG.128.
// =============================================================================================
template <typename T>
struct IkArgs {
  const T* targets;
  const T* q_init;
  int q_init_stride;  // 0 = broadcast
  unsigned n;         // < 2^31 (checked on the host): 32-bit index arithmetic in the hot loop
  IkConst<T> k;
  T* q_out;           // packed: out_q8
  T* final_pos;       // packed: out_aux
  T* pos_err;
  int32_t* iters;
  uint8_t* flags;
  unsigned long long* counters;
  unsigned* ticket;   // zeroed before launch
  unsigned chunk;     // queries a warp reserves per ticket atomic (>= 32)
  unsigned flush_min; // ik_solve_v_kernel: lanes with a finished slot that trigger a store + refill
  unsigned solo_warp; // small batches: the block has 4 warps to load the 40 KB trig table quickly, only warp 0 solves
                      // (one warp per block spreads a small batch over all SMs); every persistent IK-family kernel
  unsigned tail;      // ik_solve_v_kernel<F2>: finish the block's last stragglers in the one-query-per-lane latency loop
  unsigned guided;    // ik_solve_v_kernel: 0 = fixed ticket chunks; else a reservation is (queries left) / guided, within [32 S, chunk]
  T thresh2;          // pos_thresh^2, squared on the host in T: read straight from the constant bank by the per-pass compare
                      // (computed in the kernel, ptxas re-did the multiply every pass rather than keep it in a register)
  unsigned* ticket_next;  // ik_solve_v_kernel: the ticket of this stream's NEXT launch, zeroed by block 0 (no memset node between
                          // two launches, so the next one can be a programmatic dependent of this one); nullptr = leave it alone
  unsigned pdl;       // ik_solve_v_kernel, programmatic dependent launch (see IK_PDL_*)
  // Hand-over of a launch's unfinished queries to a follow-up launch (see "drain hand-over" at ik_solve_v_kernel).
  //   pair kernel: park_dump / park_list non-null = a warp that sees the pool dry parks ALL its running slots there and leaves
  //   resume kernel (kResume): takes its queries from them; n = *park_slots
  float2* park_dump;      // [lane rows][8]: the q register pairs of every lane that parked a slot (row stride 64 B)
  uint4* park_list;       // [slots]: query index, pass counter, 2 * row + slot
  unsigned* park_lanes;   // rows written   (device counters, zero before the pair launch)
  unsigned* park_slots;   // slots written
  unsigned* zero_next[3]; // resume kernel: the counters the NEXT launch pair of this stream will use, zeroed by block 0
};

// Warp-local pool of reserved query indices [next, end) of the persistent IK-family kernels: one ticket atomic reserves
// `chunk` consecutive queries, lanes then draw from the pool without touching global memory.  (A per-refill atomic on the
// single ticket address serialises in L2 at ~1 op/clk and capped ik_solve_kernel at ~3.3 G solves/s regardless of its
// instruction count.)  ik_solve_v_kernel keeps its own copy: guided chunks, the dry-pool hand-over.
struct WarpPool {
  unsigned next = 0, end = 0;

  // Every slot k of this lane with want[k] draws the next index: ranks are slot-major over the warp (all slot-0 draws,
  // then slot 1), and the warp reserves a fresh chunk when the pool holds fewer indices than it draws.  take(k, idx)
  // runs for each draw below n.  A slot that draws an index >= n sets the lane's `exhausted` latch: the ticket is past
  // the batch, and the caller's want[] stops asking for this lane.
  template <int S, typename Take>
  __device__ __forceinline__ void refill(const bool (&want)[S], bool& exhausted, unsigned n, unsigned* ticket, unsigned chunk,
                                         Take take) {
    const unsigned lane = threadIdx.x & 31u;
    const unsigned lanemask_lt = (1u << lane) - 1u;
    unsigned need[S], count = 0;
#pragma unroll
    for (int k = 0; k < S; ++k) {
      need[k] = __ballot_sync(FULL, want[k]);
      count += (unsigned)__popc(need[k]);
    }
    if (count) {
      bool ran_out = false;
      const unsigned avail = end - next;
      unsigned fresh = 0;
      if (count > avail) {  // warp-uniform
        if (lane == 0) fresh = atomicAdd(ticket, chunk);
        fresh = __shfl_sync(FULL, fresh, 0);
      }
      unsigned before = 0;
#pragma unroll
      for (int k = 0; k < S; ++k) {
        if (want[k]) {
          const unsigned rank = before + (unsigned)__popc(need[k] & lanemask_lt);
          const unsigned idx = rank < avail ? next + rank : fresh + (rank - avail);
          if (idx < n) take(k, idx);
          else ran_out = true;
        }
        before += (unsigned)__popc(need[k]);
      }
      if (count > avail) { next = fresh + (count - avail); end = fresh + chunk; }
      else next += count;
      exhausted = exhausted || ran_out;
    }
  }
};

// End of a persistent IK-family kernel: the warp's query, convergence and iteration counts into counters[] (nullable).
// Every solver here counts success == converged (SURVEY App. D.2).
__device__ __forceinline__ void ik_counters_add(unsigned long long* counters, unsigned long long c_n,
                                                unsigned long long c_conv, unsigned long long c_iter) {
  if (!counters) return;
  c_n = warp_sum(c_n); c_conv = warp_sum(c_conv); c_iter = warp_sum(c_iter);
  if ((threadIdx.x & 31u) == 0) {
    atomicAdd(counters + PNP_IK_CNT_N, c_n);
    atomicAdd(counters + PNP_IK_CNT_CONVERGED, c_conv);
    atomicAdd(counters + PNP_IK_CNT_SUCCESS, c_conv);
    atomicAdd(counters + PNP_IK_CNT_ITERATIONS, c_iter);
  }
}

// Back-to-back launches of ik_solve_v_kernel on one stream overlap the drain of launch k with the ramp of launch k+1
// (programmatic dependent launch).  A launch's last ~0.09 ms are its drain: the ticket pool is dry and every block waits
// for a handful of queries on their way to max_iters.  Each block signals `griddepcontrol.launch_dependents` once ALL its
// warps have seen the pool dry (none of them touches the ticket again), so the next launch's blocks move into the SMs as
// this launch's blocks leave them.  What keeps that safe:
//   * the two launches draw from different tickets (the stream's two tickets alternate; block 0 of launch k zeroes the one
//     launch k+1 will use - launch k-1, its last user, is past its pool by the time launch k starts);
//   * IK_PDL_WAIT_FIRST: the host found that this launch reads or overwrites something the previous launch on the stream
//     writes or reads (same output buffers, q_init = the previous q_out, ...): `griddepcontrol.wait` before the first
//     global access, i.e. plain stream order, nothing overlaps;
//   * IK_PDL_WAIT_AT_DRY: no such overlap: the wait moves to the point where the block's last warp sees the pool dry,
//     right before the block's own launch_dependents - by then the previous launch ended long ago, so it costs nothing, and
//     it bounds the overlap to TWO consecutive launches (launch k+2 cannot start before launch k has completed).
enum { IK_PDL_OFF = 0, IK_PDL_WAIT_FIRST = 1, IK_PDL_WAIT_AT_DRY = 2 };
__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void griddep_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// output layouts of the FP32 IK kernels
enum { IK_OUT_SEPARATE = 0,  // five arrays (pnp_ik_solve_f32)
       IK_OUT_PACKED = 1,    // out_q8[n][8] = q0..q6, pos_error; out_aux[n][4] = final_pos xyz, iterations | flags << 24
       IK_OUT_COMPACT = 2 }; // out_q8[n][8] = q0..q6, iterations | flags << 24   (32 B per query, nothing else)

// convergence test (ik_solver.py:61-64).  FP64 follows the reference literally (sqrt, then
// compare); FP32 compares squared norms and takes the sqrt only when a lane finishes.
__device__ __forceinline__ bool below_thresh(double n2, const IkConst<double>& k) { return sqrt(n2) < k.pos_thresh; }
__device__ __forceinline__ bool below_thresh(float n2, const IkConst<float>& k) { return n2 < k.pos_thresh * k.pos_thresh; }
__device__ __forceinline__ double finish_sqrt(double n2) { return sqrt(n2); }
// sqrt as x * rsqrt(x) on one MUFU.RSQ.  (rsqrtf() wraps the same instruction in a subnormal fix-up - scale by 2^24,
// MUFU, scale by 2^12 - i.e. three more FMA-pipe instructions per call in the store block, where everything on that pipe
// queues behind the packed math.)  The clamp keeps 0 * rsqrt(0) = 0 * inf out: squared distances below 1e-30 m^2 come
// back as n2 * 1e15, i.e. as nothing.
__device__ __forceinline__ float finish_sqrt(float n2) {
  float r;
  asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(fmaxf(n2, 1e-30f)));
  return n2 * r;
}

// The two pieces of a position solve that ik_solve_kernel and the multistart restarts (ms_wave_kernel) share, so that a
// restart attempt runs the plain kernel's arithmetic bit for bit.
// One DLS pass at q (pass number `it`): a lane that is `active` and finishes in this pass calls
// done(p, n2, iterations, conv) with FK(q) and the squared error at the q it finished at.  qn is the DLS step from q
// (:81-85); the caller moves q there, for the lanes it keeps solving.
template <typename T, typename Kin, typename Done>
__device__ __forceinline__ void ik_pass(const IkConst<T>& k, const Trig<T>& trig, const T (&q)[NJ], const T (&tgt)[3],
                                        int it, bool active, T (&qn)[NJ], Done done) {
  T p[3], n2;
  ik_eval_and_step<T, Kin>(q, tgt, k, trig, p, n2, qn);
  const bool last = it >= k.max_iters;             // loop ran out (ik_solver.py:57)
  const bool conv = !last && below_thresh(n2, k);  // :61-64
  if (active && (conv || last)) done(p, n2, conv ? it + 1 : it, conv);  // iterations :66 / :85
}

// Store the record of query idx in layout kOut (:88-92: final_pos = FK(q) = p; final_error = err;
// success = conv && err < 2*thresh).  Separate layout: every output but q_out nullable.
template <int kOut, typename T>
__device__ __forceinline__ void ik_store(const IkArgs<T>& a, unsigned idx, const T (&q)[NJ], const T* p, T n2,
                                         int iterations, bool conv) {
  const T err = finish_sqrt(n2);
  const bool success = conv && (err < a.k.pos_thresh * T(2));
  const unsigned fl = (conv ? PNP_IK_CONVERGED : 0u) | (success ? PNP_IK_SUCCESS : 0u);
  if (kOut == IK_OUT_PACKED) {
    float4* oq = reinterpret_cast<float4*>(a.q_out) + (size_t)idx * 2u;
    oq[0] = make_float4((float)q[0], (float)q[1], (float)q[2], (float)q[3]);
    oq[1] = make_float4((float)q[4], (float)q[5], (float)q[6], (float)err);
    reinterpret_cast<float4*>(a.final_pos)[idx] =
        make_float4((float)p[0], (float)p[1], (float)p[2], __int_as_float((int)((unsigned)iterations | (fl << 24))));
  } else if (kOut == IK_OUT_COMPACT) {
    float4* oq = reinterpret_cast<float4*>(a.q_out) + (size_t)idx * 2u;
    oq[0] = make_float4((float)q[0], (float)q[1], (float)q[2], (float)q[3]);
    oq[1] = make_float4((float)q[4], (float)q[5], (float)q[6], __int_as_float((int)((unsigned)iterations | (fl << 24))));
  } else {
    T* qo = a.q_out + (size_t)idx * NJ;
#pragma unroll
    for (int i = 0; i < NJ; ++i) qo[i] = q[i];
    if (a.final_pos) {
      T* fp = a.final_pos + (size_t)idx * 3u;
      fp[0] = p[0]; fp[1] = p[1]; fp[2] = p[2];
    }
    if (a.pos_err) a.pos_err[idx] = err;
    if (a.iters) a.iters[idx] = iterations;
    if (a.flags) a.flags[idx] = (uint8_t)fl;
  }
}

template <typename T, typename Kin, int kOut>
__global__ void __launch_bounds__(IK_BLOCK) ik_solve_kernel(const IkArgs<T> a) {
  __shared__ __align__(16) T s_q0[8];  // broadcast q_init: refills read it from shared memory
  __shared__ __align__(16) float s_tab[Trig<T>::kUsesTable ? kTrigVWords : 4];
  if (Trig<T>::kUsesTable) load_trigv_table(s_tab);
  if (a.q_init_stride == 0 && threadIdx.x < NJ) s_q0[threadIdx.x] = a.q_init[threadIdx.x];
  __syncthreads();
  if (a.solo_warp && threadIdx.x >= 32) return;  // helper warps of a small-batch block: table loaded, done
  const Trig<T> trig{s_tab};

  T q[NJ], tgt[3];
  int it = 0;
  unsigned idx = 0;
  bool active = false, exhausted = false;
  unsigned c_n = 0, c_conv = 0;  // per lane: < 2^31 queries
  unsigned long long c_iter = 0;
#pragma unroll
  for (int i = 0; i < NJ; ++i) q[i] = T(0);
  tgt[0] = tgt[1] = tgt[2] = T(0);
  WarpPool pool;

  while (true) {
    // ---- refill idle lanes -------------------------------------------------------------
    const bool want[1] = {!active && !exhausted};
    pool.refill(want, exhausted, a.n, a.ticket, a.chunk, [&](int, unsigned i) {
          idx = i;
          const T* tp = a.targets + (size_t)idx * 3u;
          tgt[0] = tp[0]; tgt[1] = tp[1]; tgt[2] = tp[2];
          if (a.q_init_stride == 0) {
#pragma unroll
            for (int j = 0; j < NJ; ++j) q[j] = s_q0[j];
          } else {
            const T* qi = a.q_init + (size_t)idx * NJ;
#pragma unroll
            for (int j = 0; j < NJ; ++j) q[j] = qi[j];
          }
          it = 0;
          active = true;
        });
    if (!__any_sync(FULL, active)) break;

    // ---- one DLS pass for all lanes ----------------------------------------------------
    T qn[NJ];
    ik_pass<T, Kin>(a.k, trig, q, tgt, it, active, qn, [&](const T* p, T n2, int iterations, bool conv) {
      ik_store<kOut>(a, idx, q, p, n2, iterations, conv);
      c_n += 1u;
      c_conv += conv ? 1u : 0u;
      c_iter += (unsigned)iterations;
      active = false;
    });
    // unconditional update: a lane that just finished is idle and gets overwritten by the
    // refill at the top of the next pass (:81-85)
#pragma unroll
    for (int i = 0; i < NJ; ++i) q[i] = qn[i];
    ++it;
  }
  ik_counters_add(a.counters, c_n, c_conv, c_iter);
}

// =============================================================================================
// The same solver over the value types of pnp_vec.cuh (specialised tree, FP32 only):
//   V = float : one query per lane (used for the bit-identity test and small batches)
//   V = F2    : TWO queries per lane.  All FK / Jacobian / J J^T / LDL^T / J^T y arithmetic of the two
//               queries runs on packed FFMA2 / FMUL2 / FADD2 (one issue slot, two FP32 results per
//               lane), which frees issue slots for the per-query clamps, compares, table look-ups
//               and the finish / refill control flow.  Each of the 64 slots of a warp refills
//               independently from the warp's reserved index pool.
// Control flow per query, output layouts and counters are those of ik_solve_kernel above.
// =============================================================================================
template <typename V>
struct Slots;
template <>
struct Slots<float> {
  static constexpr int kN = 1;
  static __device__ __forceinline__ float get(float v, int) { return v; }
  static __device__ __forceinline__ void set(float& v, int, float x) { v = x; }
};
template <>
struct Slots<F2> {
  static constexpr int kN = 2;
  static __device__ __forceinline__ float get(const F2& v, int k) { return k == 0 ? v.v.x : v.v.y; }
  static __device__ __forceinline__ void set(F2& v, int k, float x) { if (k == 0) v.v.x = x; else v.v.y = x; }
};

// Predicated global accesses for the store + refill block of ik_solve_v_kernel: as plain `if`s the
// four per-slot blocks (store slot 0/1, refill slot 0/1) were four divergent branches executed one after
// the other by a handful of lanes (24 % of all warp samples for 15 % of the instructions); predicated,
// the block is straight-line code and the two slots' dependency chains interleave.
__device__ __forceinline__ void stg128_if(bool pred, float* ptr, float x, float y, float z, float w) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %0, 0;\n\t@p st.global.v4.f32 [%1], {%2, %3, %4, %5};\n\t}"
      :: "r"((unsigned)pred), "l"(ptr), "f"(x), "f"(y), "f"(z), "f"(w) : "memory");
}
__device__ __forceinline__ void ldg3_if(bool pred, const float* ptr, float& x, float& y, float& z) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %3, 0;\n\t@p ld.global.nc.f32 %0, [%4];\n\t@p ld.global.nc.f32 %1, [%4+4];\n\t"
      "@p ld.global.nc.f32 %2, [%4+8];\n\t}"
      : "+f"(x), "+f"(y), "+f"(z) : "r"((unsigned)pred), "l"(ptr));
}
__device__ __forceinline__ void lds1_if(bool pred, const float* ptr, float& x) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %1, 0;\n\t@p ld.shared.f32 %0, [%2];\n\t}"
               : "+f"(x) : "r"((unsigned)pred), "r"((unsigned)__cvta_generic_to_shared(ptr)));
}
__device__ __forceinline__ void ldg1_if(bool pred, const float* ptr, float& x) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %1, 0;\n\t@p ld.global.nc.f32 %0, [%2];\n\t}"
               : "+f"(x) : "r"((unsigned)pred), "l"(ptr));
}

// ---------------------------------------------------------------------------------------------
// One query per lane, from a given state to the end: the loop of the small-batch latency kernel, also run by the tail
// phase of the pair kernel.  No refill, no per-slot state machine - the loop body is a single basic block (evaluate,
// test, vote, step).  Same arithmetic as ik_solve_v_kernel (ik_eval_v / ik_step_v).  A finished lane is frozen (step
// limit 0).  `it` is the lane's pass counter on entry (0 for a fresh query).  All 32 lanes must call.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void lane_solve(const IkConst<float>& k, const TrigV& trig, bool valid, int it, float (&q)[NJ],
                                           const float (&q0)[NJ], const float (&tgt)[3], float (&pf)[3], float& n2f, int& iterations,
                                           bool& conv) {
  const float thresh2 = k.pos_thresh * k.pos_thresh;
  bool done = !valid;
  conv = false;
  iterations = 0;
  float tb[3];
  pnp_spec::spec_world_to_base_v<float>(tgt, tb);
  float p[3], e[3], n2, J[21], s0, c0;  // of the last pass
  for (;; ++it) {
    ik_eval_j1_v<float>(q, tb, trig, p, e, n2, J, s0, c0);
    const bool last = it >= k.max_iters;                       // loop ran out (ik_solver.py:57)
    const bool fin = !done && (last || n2 < thresh2);          // :61-64
    if (fin) {
      conv = !last;
      iterations = conv ? it + 1 : it;                         // :66 / :85
    }
    done = done || fin;
    if (__all_sync(FULL, done)) break;
    ik_step_v<float>(q, J, e, k.damping, done ? 0.0f : k.step_limit);  // frozen once finished
  }
  // final_pos / final_error (:88-89).  A finished lane keeps its q (step limit 0) and every pass recomputes the same p / n2
  // from it, so the values of the LAST pass are every lane's final ones - no per-pass copies.  One exception: a query that
  // finished on its FIRST pass returns q (q0: the state it entered with) untouched even outside the joint limits, where the
  // limit clip of the frozen step has moved it: those lanes get their q back and the warp evaluates once more (rare).
  const bool first_pass = valid && iterations == (conv ? 1 : 0);
  if (__any_sync(FULL, first_pass)) {
#pragma unroll
    for (int i = 0; i < NJ; ++i) q[i] = first_pass ? q0[i] : q[i];
    ik_eval_j1_v<float>(q, tb, trig, p, e, n2, J, s0, c0);
  }
  n2f = n2;
  p_world_v<float>(p, s0, c0, pf);
}

// the result record(s) of one query in the layout kOut (see IK_OUT_*)
template <int kOut>
__device__ __forceinline__ void store_lane_result(const IkArgs<float>& a, unsigned id, const float (&q)[NJ], const float (&pf)[3],
                                                  float n2f, int iterations, bool conv) {
  const float err = finish_sqrt(n2f);
  const bool success = conv && (err < a.k.pos_thresh * 2.0f);  // :88-92
  const unsigned fl = (conv ? PNP_IK_CONVERGED : 0u) | (success ? PNP_IK_SUCCESS : 0u);
  const float word = __int_as_float((int)((unsigned)iterations | (fl << 24)));
  if (kOut == IK_OUT_PACKED) {
    float4* oq = reinterpret_cast<float4*>(a.q_out) + (size_t)id * 2u;
    oq[0] = make_float4(q[0], q[1], q[2], q[3]);
    oq[1] = make_float4(q[4], q[5], q[6], err);
    reinterpret_cast<float4*>(a.final_pos)[id] = make_float4(pf[0], pf[1], pf[2], word);
  } else if (kOut == IK_OUT_COMPACT) {
    float4* oq = reinterpret_cast<float4*>(a.q_out) + (size_t)id * 2u;
    oq[0] = make_float4(q[0], q[1], q[2], q[3]);
    oq[1] = make_float4(q[4], q[5], q[6], word);
  } else {
    float* qo = a.q_out + (size_t)id * NJ;
#pragma unroll
    for (int i = 0; i < NJ; ++i) qo[i] = q[i];
    if (a.final_pos) { a.final_pos[(size_t)id * 3u] = pf[0]; a.final_pos[(size_t)id * 3u + 1] = pf[1]; a.final_pos[(size_t)id * 3u + 2] = pf[2]; }
    if (a.pos_err) a.pos_err[id] = err;
    if (a.iters) a.iters[id] = iterations;
    if (a.flags) a.flags[id] = (uint8_t)fl;
  }
}

// Deferred flush: a finished slot is FROZEN (its step limit becomes 0, so qn == q and the next passes
// recompute the same p / n2) instead of being stored and refilled at once; the divergent store +
// refill code runs only when at least `flush_min` lanes hold a finished slot, when nothing is
// running any more, or when a query finished on its very first pass (its q_init may lie outside the
// joint limits, where the limit clip would not leave it untouched - see the store block).  With 64 slots per warp and a
// mean of 16 passes per query some slot finishes on 98 % of the passes; flushing every pass made the
// finish/refill code 45 % of all issued instructions.
//
// kBcast: one q_init for the whole batch (staged in shared memory) vs one per query.  A template
// parameter rather than a run-time branch because ptxas puts the (predicated-off) q_init loads on
// the scoreboard of the target loads, and the first trig FFMA2 of the pass then waited a full
// global-load latency for targets it does not need until mid-pass.
//
// Tail phase (a.tail, pair kernel).  0.2 % of cold queries run into max_iters = 100 while the mean is 16 passes, so when
// the ticket pool runs dry most warps are left holding one or two long-running slots, and a warp with one live slot
// still pays a full two-queries-per-lane pass: the launch time fits a + b n with a = 0.123 ms at max_iters = 100,
// 0.050 ms at 30 and 0.013 ms for targets that take 3 passes (tools/dev/dev_ik_fixed_cost.py) - ~1.1 us per pass of the
// longest query, on every scheduler.  Once a warp has seen the pool dry and is down to <= 8 running slots it parks
// them (query index, pass counter, q) in shared memory and leaves; the LAST warp of the block to get there finishes
// the block's stragglers after the loop, one per lane, in lane_solve().  A query continues from exactly the state it
// was parked in: results do not depend on whether or where it was handed over.
// (First attempt, dropped: the last warp took the list back into its 64 slots through the refill code.  No gain -
// a lone two-queries-per-lane warp needs ~1000 clocks per pass, and a refill that can also read the list put 40
// predicated instructions more into every flush.)
#ifndef IK_TAIL_PER_WARP_N
#define IK_TAIL_PER_WARP_N 8
#endif
// drain hand-over (see ik_solve_v_kernel): a warp hands its running slots to the resume launch once it is down to this many.
// Measured at 2^24 queries, launches back to back / one launch alone: no hand-over 2.392 / 2.433 ms, at <= 8 slots 2.383 /
// 2.428, <= 16: 2.357 / 2.405, <= 32: 2.354 / 2.412, everything at the dry point (64): 2.378 / 2.464.
#ifndef IK_HANDOVER_AT
#define IK_HANDOVER_AT 16
#endif
constexpr int IK_TAIL_PER_WARP = IK_TAIL_PER_WARP_N;         // a warp parks once it is down to this many running slots
constexpr int IK_TAIL_MAX = (IK_BLOCK / 32) * IK_TAIL_PER_WARP;  // the block's stragglers: one per lane, 32 at a time
__device__ __forceinline__ float2 pair_of(float v) { return make_float2(v, 0.0f); }
__device__ __forceinline__ float2 pair_of(const F2& v) { return v.v; }

//
// Drain hand-over (pair kernel, launches that run as programmatic dependents).  A block cannot give its registers and
// shared memory to the next launch while its last warp finishes the block's stragglers, and nearly every block holds a
// query on its way to max_iters - so the overlap of two launches hid only a third of the drain.  With park_dump / park_list
// set, a warp that has seen the ticket pool dry and is down to IK_HANDOVER_AT running slots parks them in GLOBAL memory
// (whole register pairs, like the in-block tail) and leaves; no block waits for a straggler.  The follow-up launch - this kernel as <float, kOut, kBcast,
// kResume = true>, one block per SM, small enough to sit next to four blocks of the NEXT pair launch - resumes the parked
// queries one per lane from exactly the state they were parked in (same arithmetic: no result bit depends on where a query
// finishes) while the next pair launch already runs.  Chain per stream: pair k -> resume k -> pair k+1 -> resume k+1, every
// edge a programmatic one; resume k waits for pair k to complete before it reads the list, and only then lets pair k+1 start.
// kCount = false (the caller passed no counters): the per-slot counter updates drop out of the store block - 8 instructions of
// 158, two of them 64-bit adds whose carries queue on the FMA pipe: 2.351 -> 2.312 ms for 2^24 queries (A/B on one box).
template <typename V, int kOut, bool kBcast, bool kResume = false, bool kCount = true>
__global__ void __launch_bounds__(IK_BLOCK, Slots<V>::kN == 2 ? IK_PAIR_MIN_BLOCKS : 1) ik_solve_v_kernel(const IkArgs<float> a) {
  constexpr int S = Slots<V>::kN;
  static_assert(!kResume || S == 1, "the resume kernel runs one query per lane");
  const unsigned lane = threadIdx.x & 31u;
  __shared__ __align__(16) float s_q0[8];
  __shared__ __align__(16) float s_trig[kTrigVWords];
  __shared__ float2 s_dump[S == 2 ? IK_TAIL_MAX * NJ : 1];         // tail: the q register pairs of the lanes that park a slot
  __shared__ unsigned s_list[S == 2 ? IK_TAIL_MAX * 3 : 1];        // tail: query index, pass counter, owner of each parked slot
  __shared__ unsigned s_list_n, s_live_warps, s_dry_warps;
  load_trigv_table(s_trig);  // (the table is the library's own: nothing a previous launch writes)
  if (a.pdl == IK_PDL_WAIT_FIRST || kResume) griddep_wait();  // resume: the pair launch has completed, its list is final
  if (kBcast && threadIdx.x < NJ) s_q0[threadIdx.x] = a.q_init[threadIdx.x];
  if (threadIdx.x == 0) {
    s_list_n = 0; s_live_warps = IK_BLOCK / 32; s_dry_warps = 0;
    if (blockIdx.x == 0 && a.ticket_next) { atomicExch(a.ticket_next, 0u); __threadfence(); }
    if (kResume && blockIdx.x == 0) {
      // the pair launch before this one has completed, hence (its wait at the dry point) so has the resume launch before
      // that: the counters of the stream's other parity are free, and the next pair launch starts only after this block
      // has let it (below)
#pragma unroll
      for (int i = 0; i < 3; ++i)
        if (a.zero_next[i]) atomicExch(a.zero_next[i], 0u);
      __threadfence();
    }
  }
  __syncthreads();
  if (kResume) griddep_launch_dependents();  // the next pair launch may move in next to this one
  const unsigned n_lim = kResume ? *reinterpret_cast<volatile unsigned*>(a.park_slots) : a.n;
  if (a.solo_warp && threadIdx.x >= 32) return;  // helper warps of a small-batch block: table loaded, done
  const TrigV trig{s_trig};
  const unsigned lanemask_lt = (1u << lane) - 1u;
  const int flush_min = (int)a.flush_min;
  const bool tail = S == 2 && a.tail && !a.solo_warp;  // see the tail phase below the loop
  bool pool_dry = false;   // warp-uniform: a lane of this warp has drawn an index past the end of the batch
  bool last_warp = false;  // this warp was the last of its block to leave the loop
  enum { IDLE = 0, RUN = 1, FIN_CONV = 2, FIN_NOCONV = 3 };

  V q[NJ], tgt[3], slim(0.0f);
  int it[S], st[S];
  unsigned idx[S];
  bool exhausted = false;
  unsigned c_n = 0, c_conv = 0;
  unsigned long long c_iter = 0;
#pragma unroll
  for (int i = 0; i < NJ; ++i) q[i] = V(0.0f);
  tgt[0] = tgt[1] = tgt[2] = V(0.0f);
#pragma unroll
  for (int k = 0; k < S; ++k) { it[k] = 0; idx[k] = 0; st[k] = IDLE; }
  unsigned pool_next = 0, pool_end = 0;  // warp-local pool of reserved query indices
  unsigned my_chunk = a.chunk;           // queries this warp reserves with its next ticket atomic
  bool flush = true;  // first pass: nothing to store, every slot to fill

  while (true) {
    if (flush) {  // warp-uniform
      // ---- refill idle slots (slot-major ranks: all idle slot-0 lanes first, then slot 1) -----------
      unsigned need[S], count = 0;
#pragma unroll
      for (int k = 0; k < S; ++k) {
        need[k] = __ballot_sync(FULL, st[k] == IDLE && !exhausted);
        count += (unsigned)__popc(need[k]);
      }
      if (count) {
        const unsigned avail = pool_end - pool_next;
        unsigned fresh = 0;
        if (count > avail) {  // warp-uniform
          if (pool_dry) {
            fresh = n_lim;  // this warp has seen the end of the batch: it never touches the ticket again (the next launch
                          // of the stream may already have zeroed it for the launch after that, see IK_PDL_*)
          } else {
            if (lane == 0) fresh = atomicAdd(a.ticket, my_chunk);
            fresh = __shfl_sync(FULL, fresh, 0);
          }
        }
        unsigned before = 0;
        bool ran_out = false;
#pragma unroll
        for (int k = 0; k < S; ++k) {  // predicated, no per-slot branch
          const bool want = st[k] == IDLE && !exhausted;
          const unsigned rank = before + (unsigned)__popc(need[k] & lanemask_lt);
          const unsigned id = rank < avail ? pool_next + rank : fresh + (rank - avail);
          const bool ok = want && id < n_lim;
          ran_out = ran_out || (want && !ok);
          unsigned qid = id;   // the query behind ticket `id`
          int it0 = 0;         // and the pass it starts at
          if constexpr (kResume) {
            // ticket `id` is a parked slot: its query, its pass counter, and where its q sits in the dump
            uint4 m = make_uint4(0u, 0u, 0u, 0u);
            if (ok) m = a.park_list[id];
            qid = m.x;
            it0 = (int)m.y;
            const float* src = reinterpret_cast<const float*>(a.park_dump + (size_t)(m.z >> 1) * 8u) + (m.z & 1u);
#pragma unroll
            for (int i = 0; i < NJ; ++i) {
              float qi = Slots<V>::get(q[i], k);
              ldg1_if(ok, src + 2 * i, qi);
              Slots<V>::set(q[i], k, qi);
            }
          }
          float t0 = Slots<V>::get(tgt[0], k), t1 = Slots<V>::get(tgt[1], k), t2 = Slots<V>::get(tgt[2], k);
          ldg3_if(ok, a.targets + (size_t)qid * 3u, t0, t1, t2);
          Slots<V>::set(tgt[0], k, t0);
          Slots<V>::set(tgt[1], k, t1);
          Slots<V>::set(tgt[2], k, t2);
          if constexpr (!kResume) {
#pragma unroll
            for (int i = 0; i < NJ; ++i) {
              float qi = Slots<V>::get(q[i], k);
              if (kBcast) lds1_if(ok, s_q0 + i, qi);   // predicated load: one instruction instead of LDS + select
              else ldg1_if(ok, a.q_init + (size_t)id * NJ + i, qi);
              Slots<V>::set(q[i], k, qi);
            }
          }
          idx[k] = ok ? qid : idx[k];
          it[k] = ok ? it0 : it[k];
          st[k] = ok ? (int)RUN : st[k];
          Slots<V>::set(slim, k, ok ? a.k.step_limit : Slots<V>::get(slim, k));
          before += (unsigned)__popc(need[k]);
        }
        exhausted = exhausted || ran_out;
        if (count > avail) {
          pool_next = fresh + (count - avail);
          pool_end = fresh + my_chunk;
          if (a.guided) {
            // guided self-scheduling: the next reservation shrinks with what is left, so that no warp is still working
            // through a full chunk of 256 when the others have run dry
            const unsigned left = pool_end < a.n ? a.n - pool_end : 0u;
            const unsigned want = (left / a.guided) & ~31u;
            my_chunk = want < 32u * S ? 32u * S : (want > a.chunk ? a.chunk : want);
          }
        } else {
          pool_next += count;
        }
        if (S == 2 || a.pdl) {
          const bool dry_now = __any_sync(FULL, ran_out);
          if (a.pdl && dry_now && !pool_dry) {  // warp-uniform, once per warp: this warp is done with the ticket
            unsigned before_me = 0;
            if (lane == 0) before_me = atomicAdd(&s_dry_warps, 1u);
            before_me = __shfl_sync(FULL, before_me, 0);
            if (before_me + 1u == (a.solo_warp ? 1u : (unsigned)(IK_BLOCK / 32))) {  // the block's last warp to get here
              if (a.pdl == IK_PDL_WAIT_AT_DRY) griddep_wait();
              griddep_launch_dependents();
            }
          }
          pool_dry = pool_dry || dry_now;
        }
      }
      if (S == 2 && tail && pool_dry) {  // warp-uniform
        // ---- nothing left to take: once this warp is down to a few running slots it parks them and leaves ----------
        unsigned run_m[S], n_run = 0;
#pragma unroll
        for (int k = 0; k < S; ++k) {
          run_m[k] = __ballot_sync(FULL, st[k] == RUN);
          n_run += (unsigned)__popc(run_m[k]);
        }
        if (a.park_list && n_run <= (unsigned)(IK_HANDOVER_AT)) {
          // drain hand-over: what is still running goes to the follow-up launch, whole register pairs again
          if (n_run) {
            const unsigned any_m = S == 2 ? (run_m[0] | run_m[S - 1]) : run_m[0];
            unsigned row0 = 0, slot0 = 0;
            if (lane == 0) { row0 = atomicAdd(a.park_lanes, (unsigned)__popc(any_m)); slot0 = atomicAdd(a.park_slots, n_run); }
            row0 = __shfl_sync(FULL, row0, 0);
            slot0 = __shfl_sync(FULL, slot0, 0);
            const unsigned row = row0 + (unsigned)__popc(any_m & lanemask_lt);
            if ((any_m >> lane) & 1u) {
#pragma unroll
              for (int i = 0; i < NJ; ++i) a.park_dump[(size_t)row * 8u + i] = pair_of(q[i]);
            }
            unsigned before = 0;
#pragma unroll
            for (int k = 0; k < S; ++k) {
              if (st[k] == RUN)
                a.park_list[slot0 + before + (unsigned)__popc(run_m[k] & lanemask_lt)] = make_uint4(idx[k], (unsigned)it[k], row * 2u + (unsigned)k, 0u);
              before += (unsigned)__popc(run_m[k]);
            }
          }
          break;
        }
        if (!a.park_list && n_run <= (unsigned)IK_TAIL_PER_WARP) {
          unsigned base = 0;
          if (n_run) {
            if (lane == 0) base = atomicAdd(&s_list_n, n_run);
            base = __shfl_sync(FULL, base, 0);
            // a lane that parks a slot dumps BOTH its slots as whole register pairs: 64-bit stores that never touch a half
            // (reading the halves inside this divergent block made ptxas split the pairs and re-pack them in the hot
            // loop).  At most n_run <= IK_TAIL_PER_WARP lanes per warp do, into rows [base, base + n_run) of the dump.
            const unsigned any_m = S == 2 ? (run_m[0] | run_m[S - 1]) : run_m[0];
            const unsigned row = base + (unsigned)__popc(any_m & lanemask_lt);
            if ((any_m >> lane) & 1u) {
#pragma unroll
              for (int i = 0; i < NJ; ++i) s_dump[row * NJ + i] = pair_of(q[i]);
            }
            unsigned before = 0;
#pragma unroll
            for (int k = 0; k < S; ++k) {
              if (st[k] == RUN) {
                unsigned* e = s_list + (base + before + (unsigned)__popc(run_m[k] & lanemask_lt)) * 3u;
                e[0] = idx[k];
                e[1] = (unsigned)it[k];
                e[2] = row * 2u + (unsigned)k;
              }
              before += (unsigned)__popc(run_m[k]);
            }
          }
          __threadfence_block();  // list and dump are written before this warp is counted out
          unsigned left = 0;
          if (lane == 0) left = atomicSub(&s_live_warps, 1u);
          last_warp = __shfl_sync(FULL, left, 0) == 1u;
          break;
        }
      }
      bool any_run = false;
#pragma unroll
      for (int k = 0; k < S; ++k) any_run = any_run || st[k] == RUN;
      if (!__any_sync(FULL, any_run)) break;  // everything stored, nothing left to take
    }

    // ---- one DLS pass for all slots of all lanes ---------------------------------------------------
    // (the target stays in the world frame in its registers and takes the constant shift into the frame of joint 1's
    //  parent here, two packed adds per pass: converted in the refill, the adds sat right behind the target loads and the
    //  store + refill block waited a global-load latency for them - 6 % of all warp samples)
    V p[3], n2, e[3], J[21], s0, c0, tb[3];  // p: in joint 1's frame
    pnp_spec::spec_world_to_base_v<V>(tgt, tb);
    ik_eval_j1_v<V>(q, tb, trig, p, e, n2, J, s0, c0);
    // per-slot state update in integer arithmetic (0 / 1 flags): as booleans ptxas ran out of predicate registers and
    // spilled them through SEL / LOP pairs, ~45 instructions per pass for the two slots
    int any_fin_i = 0, any_run_i = 0, imm_i = 0;
#pragma unroll
    for (int k = 0; k < S; ++k) {
      const int run = st[k] == RUN ? 1 : 0;
      const int last = it[k] >= a.k.max_iters ? 1 : 0;                           // loop ran out (ik_solver.py:57)
      const int below = Slots<V>::get(n2, k) < a.thresh2 ? 1 : 0;                    // :61-64
      const int newly = run & (last | below);
      imm_i |= newly & (it[k] == 0 ? 1 : 0);                                       // finished on its first pass
      it[k] += run & (last ^ 1);                                                   // iterations = i+1 (:66 / :85), then frozen
      st[k] += newly + (newly & last);                                             // RUN -> FIN_CONV (2) / FIN_NOCONV (3)
      Slots<V>::set(slim, k, newly ? 0.0f : Slots<V>::get(slim, k));               // freeze: the step below leaves q as it is
      any_fin_i |= st[k] >> 1;
      any_run_i |= run & (newly ^ 1);
    }
    const bool any_fin = any_fin_i != 0, any_run = any_run_i != 0, imm = imm_i != 0;
    ik_step_v<V>(q, J, e, a.k.damping, slim);
    const int n_fin = __popc(__ballot_sync(FULL, any_fin));
    const bool any_imm = __any_sync(FULL, imm);
    flush = n_fin >= flush_min || !__any_sync(FULL, any_run) || any_imm;
    if (S == 2 && tail && pool_dry && !flush) {  // warp-uniform; pool dry: flush (store, then park) once few slots still run
      unsigned n_run = 0;
#pragma unroll
      for (int k = 0; k < S; ++k) n_run += (unsigned)__popc(__ballot_sync(FULL, st[k] == RUN));
      flush = n_run <= (unsigned)(a.park_list ? (IK_HANDOVER_AT) : IK_TAIL_PER_WARP);
    }
    if (flush) {  // warp-uniform
      // ---- store finished slots.  A frozen slot keeps its q and recomputes the same p / n2 every pass,
      //      so this pass's values are the query's final ones.  One exception: a query that finished on
      //      its FIRST pass returns q_init untouched (ik_solver.py:61-67 tests before any update) even
      //      when q_init violates the joint limits, where the limit clip of the frozen step has just
      //      moved it: those are flushed in the same pass (imm) and re-read their q_init.  That only ever
      //      happens in a flush such a finish forces itself, so the common flush is a second copy of the block
      //      WITHOUT the reload: no seven predicated-off loads per slot and no copy of q into registers of its own.
      V pw[3];
      p_world_v<V>(p, s0, c0, pw);  // final_pos in the world frame (both slots, packed)
      auto store_finished = [&](auto with_reload) {
#pragma unroll
        for (int k = 0; k < S; ++k) {
          const bool f = st[k] >= FIN_CONV;
          const bool conv = st[k] == FIN_CONV;
          const float err = finish_sqrt(Slots<V>::get(n2, k));
          const int iterations = it[k];
          // :88-92  success = converged && final_error < 2 * pos_thresh: a converged query has |e|^2 < pos_thresh^2, so
          // the second test cannot fail (SURVEY App. D.2) - no compare, no 2 * pos_thresh on the FMA pipe of this block
          const unsigned fl = conv ? (PNP_IK_CONVERGED | PNP_IK_SUCCESS) : 0u;
          const unsigned id = idx[k];
          float qf[NJ];
#pragma unroll
          for (int i = 0; i < NJ; ++i) qf[i] = Slots<V>::get(q[i], k);
          if constexpr (decltype(with_reload)::value) {
            if (f && iterations == (conv ? 1 : 0)) {  // finished on the first pass (non-converged: max_iters == 0); rare
              const float* qi = kBcast ? a.q_init : a.q_init + (size_t)id * NJ;
#pragma unroll
              for (int i = 0; i < NJ; ++i) qf[i] = qi[i];
            }
          }
          const float word = __int_as_float((int)((unsigned)iterations | (fl << 24)));
          if (kOut == IK_OUT_PACKED) {
            float* oq = a.q_out + (size_t)id * 8u;
            stg128_if(f, oq, qf[0], qf[1], qf[2], qf[3]);
            stg128_if(f, oq + 4, qf[4], qf[5], qf[6], err);
            stg128_if(f, a.final_pos + (size_t)id * 4u, Slots<V>::get(pw[0], k), Slots<V>::get(pw[1], k), Slots<V>::get(pw[2], k), word);
          } else if (kOut == IK_OUT_COMPACT) {
            float* oq = a.q_out + (size_t)id * 8u;
            stg128_if(f, oq, qf[0], qf[1], qf[2], qf[3]);
            stg128_if(f, oq + 4, qf[4], qf[5], qf[6], word);
          } else if (f) {
            float* qo = a.q_out + (size_t)id * NJ;
#pragma unroll
            for (int i = 0; i < NJ; ++i) qo[i] = qf[i];
            if (a.final_pos) {
              float* fp = a.final_pos + (size_t)id * 3u;
              fp[0] = Slots<V>::get(pw[0], k); fp[1] = Slots<V>::get(pw[1], k); fp[2] = Slots<V>::get(pw[2], k);
            }
            if (a.pos_err) a.pos_err[id] = err;
            if (a.iters) a.iters[id] = iterations;
            if (a.flags) a.flags[id] = (uint8_t)fl;
          }
          if constexpr (kCount) {
            c_n += f ? 1u : 0u;
            c_conv += (f && conv) ? 1u : 0u;
            c_iter += f ? (unsigned)iterations : 0u;
          }
          st[k] = f ? (int)IDLE : st[k];
        }
      };
      if (any_imm) store_finished(std::true_type{});
      else store_finished(std::false_type{});
    }
  }

  if (S == 2 && last_warp) {
    // ---- tail phase.  Every other warp of the block has parked its last running slots and gone (their fence precedes
    //      their decrement, which precedes ours).  The stragglers of the whole block - a handful of queries on their
    //      way to max_iters - finish here, one per lane, in the latency loop of the small-batch kernel: ~500 clocks
    //      per pass for a lone warp, where four straggler warps sharing a scheduler needed ~2000 per round. -----------
    __threadfence_block();
    const unsigned cnt = *reinterpret_cast<volatile unsigned*>(&s_list_n);  // <= 4 warps x IK_TAIL_PER_WARP
    for (unsigned base = 0; base < cnt; base += 32u) {
      const bool valid = base + lane < cnt;
      const unsigned* e = s_list + (valid ? base + lane : 0u) * 3u;
      const unsigned id = e[0], who = e[2];
      const int it0 = (int)e[1];
      const float* src = reinterpret_cast<const float*>(s_dump + (size_t)(who >> 1) * NJ) + (who & 1u);
      float ql[NJ], q0[NJ], tl[3], pf[3], n2f;
#pragma unroll
      for (int i = 0; i < NJ; ++i) ql[i] = q0[i] = src[2 * i];
#pragma unroll
      for (int i = 0; i < 3; ++i) tl[i] = a.targets[(size_t)id * 3u + i];
      bool conv;
      int iterations;
      lane_solve(a.k, trig, valid, it0, ql, q0, tl, pf, n2f, iterations, conv);  // (a first-pass finish gets q0 back in there)
      if (valid) {
        store_lane_result<kOut>(a, id, ql, pf, n2f, iterations, conv);
        c_n += 1u;
        c_conv += conv ? 1u : 0u;
        c_iter += (unsigned)iterations;
      }
    }
  }
  if (a.counters) {  // (kept in the kCount = false instantiation, which only runs with a.counters == nullptr: compiled out, the same
                     //  kernel was 2 % SLOWER - 2.364 vs 2.312 ms - for no reason visible in the source; A/B three ways on one box)
    const unsigned long long w_n = warp_sum((unsigned long long)c_n), w_conv = warp_sum((unsigned long long)c_conv),
                             w_iter = warp_sum(c_iter);
    if (lane == 0) {
      atomicAdd(a.counters + PNP_IK_CNT_N, w_n);
      atomicAdd(a.counters + PNP_IK_CNT_CONVERGED, w_conv);
      atomicAdd(a.counters + PNP_IK_CNT_SUCCESS, w_conv);  // success == converged (SURVEY App. D.2)
      atomicAdd(a.counters + PNP_IK_CNT_ITERATIONS, w_iter);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Small cold batches, latency bound (BASELINE cfg2: 4096 targets).  A launch of n <= ~one warp per scheduler lasts as
// long as its slowest query - 100 passes for a target that runs into max_iters - so what matters is the latency of
// ONE pass of a lone warp, not throughput.  One query per lane, one working warp per block (the batch spreads over all
// SMs), three helper warps that only load the trig table; no ticket, no refill: lane_solve() above.  Bit-identical to
// ik_solve_v_kernel<float>.
// ---------------------------------------------------------------------------------------------
template <int kOut, bool kBcast>
__global__ void __launch_bounds__(IK_BLOCK) ik_solve_small_kernel(const IkArgs<float> a) {
  __shared__ __align__(16) float s_trig[kTrigVWords];
  load_trigv_table(s_trig);
  __syncthreads();
  if (threadIdx.x >= 32) return;
  const TrigV trig{s_trig};
  const unsigned lane = threadIdx.x;
  const unsigned id = blockIdx.x * 32u + lane;
  const bool valid = id < a.n;
  const unsigned ld = valid ? id : 0u;
  float q[NJ], q0[NJ], tgt[3], pf[3], n2f;
#pragma unroll
  for (int i = 0; i < 3; ++i) tgt[i] = a.targets[(size_t)ld * 3u + i];
  const float* qi = kBcast ? a.q_init : a.q_init + (size_t)ld * NJ;
#pragma unroll
  for (int i = 0; i < NJ; ++i) q[i] = q0[i] = qi[i];
  bool conv;
  int iterations;
  lane_solve(a.k, trig, valid, 0, q, q0, tgt, pf, n2f, iterations, conv);  // (a first-pass finish gets q_init back in there)
  if (a.counters) {  // whole warp (lanes past the end of the batch add zeros)
    const unsigned long long w_n = warp_sum((unsigned long long)(valid ? 1u : 0u)),
                             w_conv = warp_sum((unsigned long long)((valid && conv) ? 1u : 0u)),
                             w_iter = warp_sum((unsigned long long)(valid ? iterations : 0));
    if (lane == 0) {
      atomicAdd(a.counters + PNP_IK_CNT_N, w_n);
      atomicAdd(a.counters + PNP_IK_CNT_CONVERGED, w_conv);
      atomicAdd(a.counters + PNP_IK_CNT_SUCCESS, w_conv);  // success == converged (SURVEY App. D.2)
      atomicAdd(a.counters + PNP_IK_CNT_ITERATIONS, w_iter);
    }
  }
  if (!valid) return;
  store_lane_result<kOut>(a, id, q, pf, n2f, iterations, conv);
}

// ---------------------------------------------------------------------------------------------
// One query, lowest latency (JacobianIKController.solve called from Python, one pose at a time:
// test/ik_test.py, MoveIKSkill stepping through a BT).  `in` and `out` point into a pinned host mailbox
// mapped into the device address space: the kernel reads target + q_init over PCIe and writes the two
// packed result records straight back, so a solve costs one kernel launch and one stream
// synchronisation - no cudaMemcpy, no ticket memset.  Same arithmetic as the batch kernels
// (kSpec: ik_eval_v / ik_step_v, bit-identical to ik_solve_v_kernel; else the generic-tree template).
//   in [10] = target xyz, q_init[7];   out[12] = q0..q6, pos_error | final_pos xyz, iterations|flags<<24
// ---------------------------------------------------------------------------------------------
template <bool kSpec>
__global__ void __launch_bounds__(IK_BLOCK) ik_solve_one_kernel(const float* __restrict__ in, const IkConst<float> k,
                                                                float* __restrict__ out) {
  __shared__ __align__(16) float s_trig[kTrigVWords];
  __shared__ float s_in[10];
  load_trigv_table(s_trig);
  if (threadIdx.x < 10) s_in[threadIdx.x] = in[threadIdx.x];
  __syncthreads();
  if (threadIdx.x != 0) return;
  float q[NJ], tgt[3] = {s_in[0], s_in[1], s_in[2]}, p[3], n2;
#pragma unroll
  for (int i = 0; i < NJ; ++i) q[i] = s_in[3 + i];
  const float thresh2 = k.pos_thresh * k.pos_thresh;
  int it = 0;
  bool conv = false;
  while (true) {
    const bool last = it >= k.max_iters;                       // loop ran out (ik_solver.py:57)
    if (kSpec) {
      const TrigV trig{s_trig};
      float e[3], J[21], s0, c0;
      ik_eval_v<float>(q, tgt, trig, p, e, n2, J, s0, c0);
      conv = !last && n2 < thresh2;                            // :61-64
      if (conv || last) break;
      ik_step_v<float>(q, J, e, k.damping, k.step_limit);
    } else {
      // generic tree: same table trig as the specialised path
      float s[NJ], c[NJ], J[21], A[6];
#pragma unroll
      for (int i = 0; i < NJ; ++i) {
        const TrigV trig{s_trig};
        trig(q[i] - GenericKin::template qref<float>(i), &s[i], &c[i]);
      }
      GenericKin::template fk_jacp<float>(s, c, p, J);
      const float e0 = tgt[0] - p[0], e1 = tgt[1] - p[1], e2 = tgt[2] - p[2];
      n2 = (e0 * e0 + e1 * e1) + e2 * e2;
      conv = !last && n2 < thresh2;
      if (conv || last) break;
      GenericKin::template jjt<float>(J, A);
      const float a00 = A[0] + k.damping, a11 = A[3] + k.damping, a22 = A[5] + k.damping;
      const float i0 = rcp_t(a00);
      const float l10 = A[1] * i0, l20 = A[2] * i0;
      const float d1 = a11 - l10 * A[1];
      const float u12 = A[4] - l10 * A[2];
      const float i1 = rcp_t(d1);
      const float l21 = u12 * i1;
      const float d2 = a22 - l20 * A[2] - l21 * u12;
      const float i2 = rcp_t(d2);
      const float z1 = e1 - l10 * e0;
      const float z2 = e2 - l20 * e0 - l21 * z1;
      float y[3], dq[NJ];
      y[2] = z2 * i2;
      y[1] = z1 * i1 - l21 * y[2];
      y[0] = e0 * i0 - l10 * y[1] - l20 * y[2];
      GenericKin::template jty<float>(J, y, dq);
#pragma unroll
      for (int i = 0; i < NJ; ++i) {
        const float d = clamp_t(dq[i], -k.step_limit, k.step_limit);                                   // :80
        q[i] = clamp_t(q[i] + d, GenericKin::template lower<float>(i), GenericKin::template upper<float>(i));  // :81
      }
    }
    ++it;
  }
  const float err = finish_sqrt(n2);
  const int iterations = conv ? it + 1 : it;                   // :66 / :85
  const bool success = conv && (err < k.pos_thresh * 2.0f);    // :88-92
  const unsigned fl = (conv ? PNP_IK_CONVERGED : 0u) | (success ? PNP_IK_SUCCESS : 0u);
  float4* o = reinterpret_cast<float4*>(out);
  o[0] = make_float4(q[0], q[1], q[2], q[3]);
  o[1] = make_float4(q[4], q[5], q[6], err);
  o[2] = make_float4(p[0], p[1], p[2], __int_as_float((int)((unsigned)iterations | (fl << 24))));
}

// =============================================================================================
// Multi-start position IK (pnp_ik_solve_multistart_*): attempt 0 is the plain solve above, written to the outputs by
// the plain launch path.  For the queries it did not solve, attempts 1..K restart the same target from a shared seed
// table; a query returns the record of its first successful attempt (attempt 0's when none succeeds).
//
//   ms_collect_kernel   appends the index of every query whose attempt 0 failed to a list (one atomic per warp)
//   ms_wave_*_kernel    wave w: each listed query gets a group of G consecutive lanes of one warp that run the seeds
//                       [w G, w G + G) in parallel, each a plain solve from its seed (lane_solve on the specialised tree,
//                       ik_pass everywhere else: the same arithmetic as the plain entry points, so a returned attempt
//                       is bit-identical to the plain solve from that start).  The lowest lane of the
//                       group that succeeds overwrites the query's record; a query without a success goes onto the
//                       next wave's list.
// Every wave is launched whether or not its list is empty: it reads the list length on the device and its blocks leave at
// once when they have nothing to do, so the host never reads a count.  The order of a list is not deterministic, the
// outputs are: each query depends on its own attempts only.
// =============================================================================================
constexpr int MS_BLOCK = 128;
constexpr int MS_COLLECT_BLOCK = 256;
constexpr int MS_MAX_SEEDS = 255;
constexpr int MS_HDR_WORDS = 256;  // list lengths: [0] = failures of attempt 0, [w + 1] = queries still failed after wave w

// The argument block of a restart wave, for either solver: A is attempt 0's argument block (IkArgs<T>, PoseIkArgs<T>)
template <typename A>
struct MsArgs {
  A a;                     // targets and the outputs of attempt 0 (its layout), solver constants
  const std::remove_pointer_t<decltype(A::q_out)>* seeds;  // [n_seeds][7], in the solver's float type
  int n_seeds;
  int wave;                // this launch runs seeds [wave * group, wave * group + group)
  unsigned group;          // lanes per query: a power of two <= 32
  const unsigned* list_in;
  const unsigned* cnt_in;
  unsigned* list_out;      // nullptr: last wave
  unsigned* cnt_out;
  const int32_t* iters0;   // separate layouts: iterations of attempt 0 (the iters output or scratch)
  uint8_t* attempt;        // nullable
  unsigned long long* restart_stats;  // nullable: restarted, rescued, DLS passes of restart attempts
};

// success bit of attempt 0: flags[] (separate layout) or the flag byte of the packed word
template <int kOut>
__global__ void __launch_bounds__(MS_COLLECT_BLOCK) ms_collect_kernel(const uint8_t* __restrict__ flags,
                                                                      const unsigned* __restrict__ aux_words, unsigned n,
                                                                      unsigned* __restrict__ list, unsigned* __restrict__ cnt,
                                                                      unsigned long long* __restrict__ restart_stats) {
  const unsigned lane = threadIdx.x & 31u;
  const unsigned stride = gridDim.x * MS_COLLECT_BLOCK;
  unsigned long long c_fail = 0;
  for (unsigned base = blockIdx.x * MS_COLLECT_BLOCK + (threadIdx.x & ~31u); base < n; base += stride) {  // warp-uniform
    const unsigned i = base + lane;
    bool failed = false;
    if (i < n) {
      const unsigned fl = kOut == IK_OUT_SEPARATE ? (unsigned)flags[i] : aux_words[(size_t)i * 4u + 3u] >> 24;
      failed = (fl & PNP_IK_SUCCESS) == 0u;
    }
    const unsigned fb = __ballot_sync(FULL, failed);
    if (fb) {
      unsigned at = 0;
      if (lane == 0) at = atomicAdd(cnt, (unsigned)__popc(fb));
      at = __shfl_sync(FULL, at, 0);
      if (failed) list[at + (unsigned)__popc(fb & ((1u << lane) - 1u))] = i;
      c_fail += (unsigned)__popc(fb);
    }
  }
  if (restart_stats && lane == 0 && c_fail) atomicAdd(restart_stats + 0, c_fail);
}

// The part of a wave every restart kernel shares (position: both lane mappings and layouts; pose): pick the group's
// first success, store it, queue the unsolved queries.  `solve(valid, id, seed, out...)` runs one attempt per lane and
// stores nothing; `prev(id, fl, it)` reads the flags and iteration count of the record being replaced (attempt 0's),
// `store(id)` writes the lane's record.  Every solver counts success == converged, so the counter correction is the
// same for all.
template <typename A, typename Solve, typename Prev, typename Store>
__device__ __forceinline__ void ms_wave(const MsArgs<A>& m, unsigned cnt, Solve solve, Prev prev, Store store) {
  const unsigned lane = threadIdx.x & 31u;
  const unsigned G = m.group;
  const unsigned gl = lane & (G - 1u);
  const unsigned gmask = (G == 32u ? FULL : ((1u << G) - 1u)) << (lane & ~(G - 1u));
  const unsigned long long lanes_total = (unsigned long long)cnt * G;
  // warps interleaved over the blocks: a short list spreads over as many SMs as possible
  const unsigned warps_total = gridDim.x * (MS_BLOCK / 32);
  const unsigned warp_id = (threadIdx.x >> 5) * gridDim.x + blockIdx.x;
  unsigned long long c_conv = 0, c_iter = 0, c_rescued = 0, c_passes = 0;
  bool worked = false;
  for (unsigned long long base = (unsigned long long)warp_id * 32u; base < lanes_total; base += (unsigned long long)warps_total * 32u) {
    worked = true;
    const unsigned long long L = base + lane;
    const bool listed = L < lanes_total;
    const unsigned id = listed ? m.list_in[L / G] : 0u;
    const int seed = m.wave * (int)G + (int)gl;
    const bool valid = listed && seed < m.n_seeds;
    bool succ;
    int iterations;
    solve(valid, id, valid ? seed : 0, succ, iterations);
    succ = succ && valid;
    c_passes += valid ? (unsigned)iterations : 0u;
    const unsigned sb = __ballot_sync(FULL, succ) & gmask;
    if (sb && lane == (unsigned)(__ffs(sb) - 1)) {
      // the record of attempt 0 leaves the returned set: correct the counters (which counted it) by the difference
      unsigned old_fl, old_it;
      prev(id, old_fl, old_it);
      store(id);
      if (m.attempt) m.attempt[id] = (uint8_t)(seed + 1);
      c_conv += 1ull - (unsigned long long)(old_fl & PNP_IK_CONVERGED);
      c_iter += (unsigned long long)(unsigned)iterations - (unsigned long long)old_it;  // mod 2^64
      c_rescued += 1u;
    }
    const bool push = m.list_out && listed && gl == 0u && !sb;
    const unsigned pb = __ballot_sync(FULL, push);
    if (pb) {
      unsigned at = 0;
      if (lane == 0) at = atomicAdd(m.cnt_out, (unsigned)__popc(pb));
      at = __shfl_sync(FULL, at, 0);
      if (push) m.list_out[at + (unsigned)__popc(pb & ((1u << lane) - 1u))] = id;
    }
  }
  if (!worked) return;
  if (m.a.counters) {
    const unsigned long long w_conv = warp_sum(c_conv), w_iter = warp_sum(c_iter);
    if (lane == 0) {
      atomicAdd(m.a.counters + PNP_IK_CNT_CONVERGED, w_conv);
      atomicAdd(m.a.counters + PNP_IK_CNT_SUCCESS, w_conv);  // success == converged, as the plain kernels count it
      atomicAdd(m.a.counters + PNP_IK_CNT_ITERATIONS, w_iter);
    }
  }
  if (m.restart_stats) {
    const unsigned long long w_res = warp_sum(c_rescued), w_pass = warp_sum(c_passes);
    if (lane == 0) {
      atomicAdd(m.restart_stats + 1, w_res);
      atomicAdd(m.restart_stats + 2, w_pass);
    }
  }
}

// flags and iterations of attempt 0's position record: flags[] / iters0[] (separate layout) or the packed word
template <int kOut, typename A>
__device__ __forceinline__ void ms_ik_prev(const MsArgs<A>& m, unsigned id, unsigned& fl, unsigned& it) {
  if (kOut == IK_OUT_SEPARATE) {
    fl = m.a.flags[id];
    it = (unsigned)m.iters0[id];
  } else {
    const unsigned w = reinterpret_cast<const unsigned*>(m.a.final_pos)[(size_t)id * 4u + 3u];
    fl = w >> 24;
    it = w & 0xFFFFFFu;
  }
}

// FP32 on the specialised tree: lane_solve + store_lane_result, i.e. ik_solve_small_kernel's arithmetic per lane
template <int kOut>
__global__ void __launch_bounds__(MS_BLOCK) ms_wave_v_kernel(const MsArgs<IkArgs<float>> m) {
  const unsigned cnt = *m.cnt_in;
  if ((unsigned long long)blockIdx.x * 32u >= (unsigned long long)cnt * m.group) return;  // no work for any warp of this block
  __shared__ __align__(16) float s_trig[kTrigVWords];
  load_trigv_table(s_trig);
  __syncthreads();
  const TrigV trig{s_trig};
  float q[NJ], pf[3], n2f;
  bool conv;
  int it_kept = 0;
  auto solve = [&](bool valid, unsigned id, int seed, bool& succ, int& iterations) {
    float q0[NJ], tgt[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) tgt[i] = m.a.targets[(size_t)id * 3u + i];
#pragma unroll
    for (int i = 0; i < NJ; ++i) q[i] = q0[i] = m.seeds[seed * NJ + i];
    lane_solve(m.a.k, trig, valid, 0, q, q0, tgt, pf, n2f, iterations, conv);
    succ = conv && (finish_sqrt(n2f) < m.a.k.pos_thresh * 2.0f);  // store_lane_result's success
    it_kept = iterations;
  };
  auto store = [&](unsigned id) { store_lane_result<kOut>(m.a, id, q, pf, n2f, it_kept, conv); };
  ms_wave(m, cnt, solve, [&](unsigned id, unsigned& fl, unsigned& it) { ms_ik_prev<kOut>(m, id, fl, it); }, store);
}

// FP32 on other trees and FP64: per lane ik_pass and ik_store, ik_solve_kernel's pass and store block, no refill
template <typename T, typename Kin, int kOut>
__global__ void __launch_bounds__(MS_BLOCK) ms_wave_kernel(const MsArgs<IkArgs<T>> m) {
  const unsigned cnt = *m.cnt_in;
  if ((unsigned long long)blockIdx.x * 32u >= (unsigned long long)cnt * m.group) return;
  __shared__ __align__(16) float s_tab[Trig<T>::kUsesTable ? kTrigVWords : 4];
  if (Trig<T>::kUsesTable) load_trigv_table(s_tab);
  __syncthreads();
  const Trig<T> trig{s_tab};
  // the finished attempt of this lane: q (which stops moving when the lane finishes), FK(q) and the squared error
  T q[NJ], p[3], n2;
  bool conv;
  int it_kept = 0;
  auto solve = [&](bool valid, unsigned id, int seed, bool& succ, int& iterations) {
    T tgt[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) tgt[i] = m.a.targets[(size_t)id * 3u + i];
#pragma unroll
    for (int i = 0; i < NJ; ++i) q[i] = m.seeds[seed * NJ + i];
    bool active = valid;
    conv = false;
    iterations = 0;
    p[0] = p[1] = p[2] = T(0);
    n2 = T(0);
    for (int it = 0; __any_sync(FULL, active); ++it) {
      T qn[NJ];
      ik_pass<T, Kin>(m.a.k, trig, q, tgt, it, active, qn, [&](const T* pp, T nn2, int its, bool cv) {
        conv = cv;
        iterations = its;
        p[0] = pp[0]; p[1] = pp[1]; p[2] = pp[2];
        n2 = nn2;
        active = false;
      });
      if (active) {
#pragma unroll
        for (int i = 0; i < NJ; ++i) q[i] = qn[i];
      }
    }
    succ = conv && (finish_sqrt(n2) < m.a.k.pos_thresh * T(2));
    it_kept = iterations;
  };
  auto store = [&](unsigned id) { ik_store<kOut>(m.a, id, q, p, n2, it_kept, conv); };
  ms_wave(m, cnt, solve, [&](unsigned id, unsigned& fl, unsigned& it) { ms_ik_prev<kOut>(m, id, fl, it); }, store);
}

// =============================================================================================
// Warm-started waypoint sequences (MoveIKSkill.reset inner loop, skills/move.py:106-137):
// one lane per env, q carried in registers across the n_steps solves.
// =============================================================================================
template <typename T>
struct WaypointArgs {
  const T* q_start;
  const T* goal;
  unsigned n;       // < 2^31 (checked on the host)
  int n_steps;
  T step_size;
  T reach_thresh;  // MoveIKSkill.pos_thresh = 0.01 (move.py:66,106)
  IkConst<T> k;
  T* q_out;
  T* pos_out;
  int32_t* n_accepted;
  int32_t* iters_total;
  unsigned long long* counters;
  unsigned* ticket; // zeroed before launch
  unsigned chunk;   // envs a warp reserves per ticket atomic
  unsigned solo_warp;  // small batches: 4 warps load the trig table, only warp 0 works
};

// The two loop levels (waypoints x DLS passes) are FLATTENED and the lanes are PERSISTENT: every pass
// of the warp loop is one DLS evaluation for all lanes; a lane whose inner solve finished does its
// accept / advance-to-next-waypoint bookkeeping on the spot and starts the next solve in the following
// pass; a lane whose env is finished writes it back and takes the next env (chunked ticket, as in
// ik_solve_kernel).  A fresh env enters in state INIT and gets its start position FK(q_start) from the
// shared DLS pass of that round.  (The first version ran the inner solve as a warp-synchronous loop per
// waypoint inside a grid-stride loop over envs: warm-started solves take 2 passes on average but 3 for
// some lane of nearly every warp, and envs need 10-50 waypoints, so lanes idled for 1/3 of the passes.)
template <typename T, typename Kin>
__global__ void __launch_bounds__(IK_BLOCK) ik_waypoints_kernel(const WaypointArgs<T> a) {
  __shared__ __align__(16) float s_tab[Trig<T>::kUsesTable ? kTrigVWords : 4];
  if (Trig<T>::kUsesTable) load_trigv_table(s_tab);
  __syncthreads();
  if (a.solo_warp && threadIdx.x >= 32) return;  // helper warps of a small-batch block: table loaded, done
  const Trig<T> trig{s_tab};
  enum { IDLE = 0, INIT = 1, RUN = 2 };
  unsigned long long c_n = 0, c_conv = 0, c_iter = 0;
  WarpPool pool;
  bool exhausted = false;
  unsigned e = 0;
  int state = IDLE;
  T q[NJ], qs[NJ], goal[3] = {T(0), T(0), T(0)}, pos[3] = {T(0), T(0), T(0)}, tgt[3] = {T(0), T(0), T(0)};
#pragma unroll
  for (int i = 0; i < NJ; ++i) q[i] = qs[i] = T(0);
  int step = 0, it = 0, accepted = 0, iters_sum = 0, fails = 0;

  // set up the solve of waypoint `step`; false when the env has nothing left to do
  auto next_waypoint = [&]() -> bool {
    if (step >= a.n_steps) return false;
    const T dx = goal[0] - pos[0], dy = goal[1] - pos[1], dz = goal[2] - pos[2];   // :110
    const T d2 = (dx * dx + dy * dy) + dz * dz;
    const T dist = finish_sqrt(d2);                                                // :111 (FP32: d2 * rsqrt(d2))
    if (!(dist > a.reach_thresh)) return false;                                    // :106 (pos no longer changes)
    T stp = fmin(fmin(a.step_size, dist * T(0.1)), T(0.02));                       // :114-117
    if (fails > 0) stp = stp * T(0.5);                                             // :118-119
    if (dist > stp) {                                                              // :122-125
      const T f = stp * rcp_t(dist);
      tgt[0] = pos[0] + dx * f; tgt[1] = pos[1] + dy * f; tgt[2] = pos[2] + dz * f;
    } else {
      tgt[0] = goal[0]; tgt[1] = goal[1]; tgt[2] = goal[2];
    }
#pragma unroll
    for (int i = 0; i < NJ; ++i) qs[i] = q[i];                                     // solve(next_pos, q_current) (:128)
    it = 0;
    return true;
  };

  while (true) {
    // ---- refill idle lanes ------------------------------------------------------------------
    const bool want[1] = {state == IDLE && !exhausted};
    pool.refill(want, exhausted, a.n, a.ticket, a.chunk, [&](int, unsigned idx) {
          e = idx;
#pragma unroll
          for (int i = 0; i < NJ; ++i) q[i] = qs[i] = a.q_start[(size_t)e * NJ + i];
#pragma unroll
          for (int i = 0; i < 3; ++i) goal[i] = a.goal[(size_t)e * 3 + i];
          step = 0; accepted = 0; iters_sum = 0; fails = 0;
          state = INIT;
        });
    if (!__any_sync(FULL, state != IDLE)) break;

    // ---- one DLS pass for all lanes -------------------------------------------------------------
    T n2, qn[NJ], pp[3];
    ik_eval_and_step<T, Kin>(qs, tgt, a.k, trig, pp, n2, qn);
    bool advance = false;
    if (state == INIT) {
      pos[0] = pp[0]; pos[1] = pp[1]; pos[2] = pp[2];               // move.py:91 start_pos = FK(q_start)
      state = RUN;
      advance = true;
    } else if (state == RUN) {
      const bool last = it >= a.k.max_iters;
      const bool conv = !last && below_thresh(n2, a.k);
      if (conv || last) {
        const T err = finish_sqrt(n2);
        const int iters = conv ? it + 1 : it;
        const bool success = conv && (err < a.k.pos_thresh * T(2));
        iters_sum += iters;
        c_n += 1; c_conv += conv ? 1 : 0; c_iter += (unsigned long long)iters;
        if (success && (err < a.step_size * T(2))) {                               // :131-138
#pragma unroll
          for (int i = 0; i < NJ; ++i) q[i] = qs[i];
          pos[0] = pp[0]; pos[1] = pp[1]; pos[2] = pp[2];
          fails = 0;
          ++accepted;
        } else {
          ++fails;                                                                 // :142
        }
        ++step;
        advance = true;
      } else {
#pragma unroll
        for (int i = 0; i < NJ; ++i) qs[i] = qn[i];
        ++it;
      }
    }
    const bool done = advance && !next_waypoint();
    if (done) {
#pragma unroll
      for (int i = 0; i < NJ; ++i) a.q_out[(size_t)e * NJ + i] = q[i];
#pragma unroll
      for (int i = 0; i < 3; ++i) a.pos_out[(size_t)e * 3 + i] = pos[i];
      if (a.n_accepted) a.n_accepted[e] = accepted;
      if (a.iters_total) a.iters_total[e] = iters_sum;
      state = IDLE;
    }
  }
  ik_counters_add(a.counters, c_n, c_conv, c_iter);
}

// ---------------------------------------------------------------------------------------------
// The same waypoint state machine over the value types of pnp_vec.cuh (specialised tree, FP32):
// V = F2 runs TWO envs per lane with all DLS arithmetic on packed FFMA2/FMUL2/FADD2 (the scalar kernel
// above is issue bound at ~500 instructions per pass, 55 % of them FP32 math); V = float is the
// one-env-per-lane instantiation of the same code, bit-identical to the pair kernel.
// A slot whose solve finishes in a pass is frozen for that pass (step limit 0), does its accept /
// advance bookkeeping after the shared step, and starts its next solve in the following pass.  The
// accepted joint vector of each slot lives in shared memory (written on accept, read on a rejected
// solve and at write-back), which keeps the kernel at 4 blocks per SM.
// ---------------------------------------------------------------------------------------------
template <typename V, bool kFuse>
__global__ void __launch_bounds__(IK_BLOCK, Slots<V>::kN == 2 ? IK_PAIR_MIN_BLOCKS : 1) ik_waypoints_v_kernel(const WaypointArgs<float> a) {
  constexpr int S = Slots<V>::kN;
  __shared__ __align__(16) float s_trig[kTrigVWords];
  __shared__ float s_qa[S * NJ * IK_BLOCK];  // accepted q of every slot: [(k * NJ + i) * IK_BLOCK + thread]
  load_trigv_table(s_trig);
  __syncthreads();
  if (a.solo_warp && threadIdx.x >= 32) return;  // helper warps of a small-batch block: table loaded, done
  const TrigV trig{s_trig};
  const float thresh2 = a.k.pos_thresh * a.k.pos_thresh;
  float* const qa = s_qa + threadIdx.x;
  enum { IDLE = 0, INIT = 1, RUN = 2 };

  V qs[NJ], tgt[3], pos[3], goal[3], slim(0.0f);
  int state[S], step[S], it[S], accepted[S], iters_sum[S], fails[S];
  unsigned env[S];
  bool exhausted = false;
  unsigned long long c_n = 0, c_conv = 0, c_iter = 0;
  WarpPool pool;
#pragma unroll
  for (int i = 0; i < NJ; ++i) qs[i] = V(0.0f);
#pragma unroll
  for (int i = 0; i < 3; ++i) tgt[i] = pos[i] = goal[i] = V(0.0f);
#pragma unroll
  for (int k = 0; k < S; ++k) { state[k] = IDLE; step[k] = it[k] = accepted[k] = iters_sum[k] = fails[k] = 0; env[k] = 0; }

  while (true) {
    // ---- refill idle slots ---------------------------------------------------------------------------
    bool want[S];
#pragma unroll
    for (int k = 0; k < S; ++k) want[k] = state[k] == IDLE && !exhausted;
    pool.refill(want, exhausted, a.n, a.ticket, a.chunk, [&](int k, unsigned id) {
          env[k] = id;
#pragma unroll
          for (int i = 0; i < NJ; ++i) {
            const float v = a.q_start[(size_t)id * NJ + i];
            Slots<V>::set(qs[i], k, v);
            qa[(k * NJ + i) * IK_BLOCK] = v;
          }
#pragma unroll
          for (int i = 0; i < 3; ++i) Slots<V>::set(goal[i], k, a.goal[(size_t)id * 3 + i]);
          step[k] = 0; accepted[k] = 0; iters_sum[k] = 0; fails[k] = 0; it[k] = 0;
          state[k] = INIT;
        });
    bool any_live = false;
#pragma unroll
    for (int k = 0; k < S; ++k) any_live = any_live || state[k] != IDLE;
    if (!__any_sync(FULL, any_live)) break;

    // ---- one DLS pass for all slots of all lanes ---------------------------------------------------
    V p[3], pr[3], n2, ev[3], J[21], s0, c0, tb[3];  // pr: FK in joint 1's frame (ik_eval_j1_v); p: the same point in the world
    pnp_spec::spec_world_to_base_v<V>(tgt, tb);
    ik_eval_j1_v<V>(qs, tb, trig, pr, ev, n2, J, s0, c0);
    p_world_v<V>(pr, s0, c0, p);
    bool fin[S], iterating[S], reload[S];
#pragma unroll
    for (int k = 0; k < S; ++k) {
      const bool running = state[k] == RUN;
      fin[k] = running && (it[k] >= a.k.max_iters || Slots<V>::get(n2, k) < thresh2);
      iterating[k] = running && !fin[k];
      Slots<V>::set(slim, k, iterating[k] ? a.k.step_limit : 0.0f);  // INIT / finishing / idle slots: frozen
    }
    // kFuse: the update moves behind the bookkeeping, so that the pass in which a solve is accepted (or the INIT
    // pass) is also the first iteration of the next solve - same q, hence the same p and J, only the target changes
    if (!kFuse) ik_step_v<V>(qs, J, ev, a.k.damping, slim);

    // ---- bookkeeping, branch-free: with ~2 passes per warm solve half of the slots finish a solve in
    //      every pass, so this runs as predicated straight-line code; the waypoint geometry of both
    //      slots (move.py:110-125) is packed arithmetic ---------------------------------------------------
    bool adv[S], fused[S];
#pragma unroll
    for (int k = 0; k < S; ++k) {
      const bool init = state[k] == INIT;
      const bool f = fin[k];
      const bool conv = it[k] < a.k.max_iters;
      const float err = finish_sqrt(Slots<V>::get(n2, k));
      const int iters = it[k] + (conv ? 1 : 0);
      const bool success = conv && (err < a.k.pos_thresh * 2.0f);
      const bool accept = f && success && (err < a.step_size * 2.0f);                // :131-138
      iters_sum[k] += f ? iters : 0;
      c_n += f ? 1u : 0u; c_conv += (f && conv) ? 1u : 0u; c_iter += f ? (unsigned)iters : 0u;
      const bool keep = accept && it[k] > 0;  // qs becomes q_current
      if (keep) {
#pragma unroll
        for (int i = 0; i < NJ; ++i) qa[(k * NJ + i) * IK_BLOCK] = Slots<V>::get(qs[i], k);
      }
      // rejected solve: the next one restarts from q_current; INIT pass / solve accepted on its first
      // pass: q_current itself, reloaded because the frozen limit clip may have moved an out-of-limits q_start
      reload[k] = init || (f && !keep);
      if (!kFuse && reload[k]) {
#pragma unroll
        for (int i = 0; i < NJ; ++i) Slots<V>::set(qs[i], k, qa[(k * NJ + i) * IK_BLOCK]);
      }
      fused[k] = init || accept;  // the next solve starts from the q this pass was evaluated at
      if (init || accept) {                                                          // :91 start_pos / :136
#pragma unroll
        for (int i = 0; i < 3; ++i) Slots<V>::set(pos[i], k, Slots<V>::get(p[i], k));
      }
      accepted[k] += accept ? 1 : 0;
      fails[k] = accept ? 0 : fails[k] + (f ? 1 : 0);                                // :142
      step[k] += f ? 1 : 0;
      adv[k] = init || f;
      it[k] = adv[k] ? 0 : it[k] + 1;
      state[k] = init ? RUN : state[k];
    }
    {
      const V dx = v_sub(goal[0], pos[0]), dy = v_sub(goal[1], pos[1]), dz = v_sub(goal[2], pos[2]);   // :110
      const V d2 = pnp_fma(dz, dz, pnp_fma(dy, dy, pnp_mul(dx, dx)));
      V dist, stp, inv;
#pragma unroll
      for (int k = 0; k < S; ++k) {
        const float dk = finish_sqrt(Slots<V>::get(d2, k));                          // :111
        float sk = fminf(fminf(a.step_size, dk * 0.1f), 0.02f);                      // :114-117
        sk = fails[k] > 0 ? sk * 0.5f : sk;                                          // :118-119
        Slots<V>::set(dist, k, dk);
        Slots<V>::set(stp, k, sk);
        Slots<V>::set(inv, k, rcp_approx(dk));
      }
      const V fr = pnp_mul(stp, inv);
      const V nx = pnp_fma(dx, fr, pos[0]), ny = pnp_fma(dy, fr, pos[1]), nz = pnp_fma(dz, fr, pos[2]);  // :122-125
#pragma unroll
      for (int k = 0; k < S; ++k) {
        const float dk = Slots<V>::get(dist, k);
        const bool far = dk > Slots<V>::get(stp, k);
        const bool moving = step[k] < a.n_steps && dk > a.reach_thresh;              // :106
        if (adv[k]) {
          Slots<V>::set(tgt[0], k, far ? Slots<V>::get(nx, k) : Slots<V>::get(goal[0], k));
          Slots<V>::set(tgt[1], k, far ? Slots<V>::get(ny, k) : Slots<V>::get(goal[1], k));
          Slots<V>::set(tgt[2], k, far ? Slots<V>::get(nz, k) : Slots<V>::get(goal[2], k));
        }
        if (adv[k] && !moving) {  // nothing left to do for this env: write it back (once per env)
          const unsigned id = env[k];
#pragma unroll
          for (int i = 0; i < NJ; ++i) a.q_out[(size_t)id * NJ + i] = qa[(k * NJ + i) * IK_BLOCK];
#pragma unroll
          for (int i = 0; i < 3; ++i) a.pos_out[(size_t)id * 3 + i] = Slots<V>::get(pos[i], k);
          if (a.n_accepted) a.n_accepted[id] = accepted[k];
          if (a.iters_total) a.iters_total[id] = iters_sum[k];
          state[k] = IDLE;
        }
      }
    }
    if (kFuse) {
      // error of the new targets at this pass's p: what the first pass of the next solve would compute
      V en[3], n2n, tbn[3];
      pnp_spec::spec_world_to_base_v<V>(tgt, tbn);
      target_err_j1_v<V>(tbn, pr, s0, c0, en, n2n);
#pragma unroll
      for (int k = 0; k < S; ++k) {
        // a new solve that is already within pos_thresh of its target (or an env that is done, or a rejected
        // solve, which restarts from another q) stays frozen and is handled by the next pass as before
        fused[k] = fused[k] && adv[k] && state[k] == RUN && a.k.max_iters > 0 && !(Slots<V>::get(n2n, k) < thresh2);
        if (fused[k]) {
#pragma unroll
          for (int i = 0; i < 3; ++i) Slots<V>::set(ev[i], k, Slots<V>::get(en[i], k));
          it[k] = 1;
        }
        Slots<V>::set(slim, k, (iterating[k] || fused[k]) ? a.k.step_limit : 0.0f);
      }
      ik_step_v<V>(qs, J, ev, a.k.damping, slim);
#pragma unroll
      for (int k = 0; k < S; ++k) {
        if (reload[k] && !fused[k]) {
#pragma unroll
          for (int i = 0; i < NJ; ++i) Slots<V>::set(qs[i], k, qa[(k * NJ + i) * IK_BLOCK]);
        }
      }
    }
  }
  ik_counters_add(a.counters, c_n, c_conv, c_iter);
}

// =============================================================================================
// Pose-mode IK (SURVEY 8f-4, an EXTENSION: the reference's FrankaEnv.solve_ik(target_pos,
// target_quat, q_init) at envs/panda_env.py:399-409 imports a function that does not exist, so
// there is no reference arithmetic to match).  Same loop as the position solver with a 6-row task:
//   e = [target_pos - p ;  w * rotvec(target_quat (x) conj(site_quat))]      (world frame)
//   J = [jacp ; w * jacr]  (6x7, mj_jacSite),  dq = J^T (J J^T + damping I_6)^-1 e
//   converged  <=>  |e_pos| < pos_thresh  and  |rotvec| < rot_thresh          (tested before update)
// The 6x6 SPD system is solved by an LDL^T factorisation held in registers.  One lane per query.
// =============================================================================================
template <typename T>
struct PoseIkArgs {
  const T* target_pos;
  const T* target_quat;
  const T* q_init;
  int q_init_stride;
  unsigned n;       // < 2^31 (checked on the host)
  IkConst<T> k;
  T rot_thresh, rot_weight;
  T* q_out;
  T* final_pos;
  T* final_quat;
  T* pos_err;
  T* rot_err;
  int32_t* iters;
  uint8_t* flags;
  unsigned long long* counters;
  unsigned* ticket; // zeroed before launch
  unsigned chunk;   // queries a warp reserves per ticket atomic
  unsigned solo_warp;  // small batches: 4 warps load the trig table, only warp 0 works
};

// mju_quat2Vel(res, quat, 1): rotation vector of a unit quaternion, angle folded into (-pi, pi]
template <typename T>
__device__ __forceinline__ void quat2vel(const T* q, T* v) {
  const T sin_a_2 = sqrt_t(q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
  T speed = T(2) * atan2_t(sin_a_2, q[0]);
  if (speed > T(3.14159265358979323846)) speed -= T(6.28318530717958647692);
  const T sc = sin_a_2 > T(0) ? speed / sin_a_2 : T(0);
  v[0] = q[1] * sc; v[1] = q[2] * sc; v[2] = q[3] * sc;
}

// FP32 pose kernel: the same, with x*rsqrt(x) and one rsqrt for the division (the pose extension is held to
// tolerances, not to bit parity - there is no reference arithmetic for it)
__device__ __forceinline__ void quat2vel_fast(const float* q, float* v) {
  const float s2 = q[1] * q[1] + q[2] * q[2] + q[3] * q[3];
  const float r = s2 > 0.0f ? rsqrtf(s2) : 0.0f;
  float speed = 2.0f * atan2f(s2 * r, q[0]);
  if (speed > 3.14159265358979323846f) speed -= 6.28318530717958647692f;
  const float sc = speed * r;
  v[0] = q[1] * sc; v[1] = q[2] * sc; v[2] = q[3] * sc;
}
__device__ __forceinline__ void quat2vel_fast(const double* q, double* v) { quat2vel<double>(q, v); }

// mju_mat2Quat with the case chosen by selects instead of branches (the four cases of random targets diverge)
// and rsqrt for the square roots / divisions; same case rule and formulas as mat2quat<T>
__device__ __forceinline__ void mat2quat_fast(const float* m, float* q) {
  const bool c0 = m[0] + m[4] + m[8] > 0.0f;
  const bool c1 = !c0 && m[0] > m[4] && m[0] > m[8];
  const bool c2 = !c0 && !c1 && m[4] > m[8];
  const float s0 = (c0 || c1) ? m[0] : -m[0];
  const float s1 = (c0 || c2) ? m[4] : -m[4];
  const float s2 = (c0 || (!c1 && !c2)) ? m[8] : -m[8];
  const float t = 1.0f + s0 + s1 + s2;
  const float r = rsqrtf(t);
  const float big = 0.5f * t * r, k = 0.5f * r;
  const float a75 = k * (m[7] - m[5]), a26 = k * (m[2] - m[6]), a31 = k * (m[3] - m[1]);
  const float b13 = k * (m[1] + m[3]), b26 = k * (m[2] + m[6]), b57 = k * (m[5] + m[7]);
  float w = c0 ? big : (c1 ? a75 : (c2 ? a26 : a31));
  float x = c0 ? a75 : (c1 ? big : (c2 ? b13 : b26));
  float y = c0 ? a26 : (c1 ? b13 : (c2 ? big : b57));
  float z = c0 ? a31 : (c1 ? b26 : (c2 ? b57 : big));
  const float inv = rsqrtf(w * w + x * x + y * y + z * z);
  q[0] = w * inv; q[1] = x * inv; q[2] = y * inv; q[3] = z * inv;
}
__device__ __forceinline__ void mat2quat_fast(const double* m, double* q) { mat2quat<double>(m, q); }

// solve the SPD system A y = b, A given by its lower triangle L[i][j] (j <= i), in place (LDL^T)
template <typename T, int N>
__device__ __forceinline__ void ldlt_solve(T (&A)[N][N], T (&b)[N]) {
  T dg[N], dinv[N];
#pragma unroll
  for (int j = 0; j < N; ++j) {
    T d = A[j][j];
#pragma unroll
    for (int k = 0; k < j; ++k) d -= A[j][k] * A[j][k] * dg[k];
    dg[j] = d;
    dinv[j] = rcp_t(d);  // FP32: one MUFU.RCP (1 ulp); FP64: 1.0 / d
#pragma unroll
    for (int i = j + 1; i < N; ++i) {
      T v = A[i][j];
#pragma unroll
      for (int k = 0; k < j; ++k) v -= A[i][k] * A[j][k] * dg[k];
      A[i][j] = v * dinv[j];
    }
  }
#pragma unroll
  for (int i = 0; i < N; ++i)
#pragma unroll
    for (int k = 0; k < i; ++k) b[i] -= A[i][k] * b[k];
#pragma unroll
  for (int i = 0; i < N; ++i) b[i] *= dinv[i];
#pragma unroll
  for (int i = N - 1; i >= 0; --i)
#pragma unroll
    for (int k = i + 1; k < N; ++k) b[i] -= A[k][i] * b[k];
}

// The three pieces of a pose solve that ik_pose_solve_kernel and the multistart restarts (ms_pose_wave_kernel) share,
// so that a restart attempt runs the plain kernel's arithmetic bit for bit.
// Target of query e: its position and its quaternion normalised on load.
template <typename T>
__device__ __forceinline__ void pose_load_target(const PoseIkArgs<T>& a, unsigned e, T (&tp)[3], T (&tq)[4]) {
#pragma unroll
  for (int i = 0; i < 3; ++i) tp[i] = a.target_pos[(size_t)e * 3 + i];
#pragma unroll
  for (int i = 0; i < 4; ++i) tq[i] = a.target_quat[(size_t)e * 4 + i];
  const T nq = sqrt_t(tq[0] * tq[0] + tq[1] * tq[1] + tq[2] * tq[2] + tq[3] * tq[3]);
#pragma unroll
  for (int i = 0; i < 4; ++i) tq[i] = tq[i] / nq;
}

// One 6-row DLS pass at q (pass number `it`): evaluate the pose error and test convergence; a lane that is `active` and
// finishes in this pass calls done(pp, qcur, pe, re, iterations, conv) with the pose and errors at the q it finished
// at (q is still that q during the call).  Then q takes the DLS step - unconditionally: the caller discards the q of a
// lane that has finished.
template <typename T, typename Kin, typename Done>
__device__ __forceinline__ void pose_pass(const PoseIkArgs<T>& a, const Trig<T>& trig, T (&q)[NJ], const T (&tp)[3],
                                          const T (&tq)[4], int it, bool active, Done done) {
  T s[NJ], c[NJ];
#pragma unroll
  for (int i = 0; i < NJ; ++i) trig(q[i] - Kin::template qref<T>(i), &s[i], &c[i]);
  T pp[3], J[42], R[9], qcur[4];
  Kin::template fk_full<T>(s, c, pp, J, R);
  mat2quat_fast(R, qcur);
  // err_quat = target (x) conj(current); rotation vector in the world frame
  const T eq[4] = {tq[0] * qcur[0] + tq[1] * qcur[1] + tq[2] * qcur[2] + tq[3] * qcur[3],
                   -tq[0] * qcur[1] + tq[1] * qcur[0] - tq[2] * qcur[3] + tq[3] * qcur[2],
                   -tq[0] * qcur[2] + tq[1] * qcur[3] + tq[2] * qcur[0] - tq[3] * qcur[1],
                   -tq[0] * qcur[3] - tq[1] * qcur[2] + tq[2] * qcur[1] + tq[3] * qcur[0]};
  T rv[3];
  quat2vel_fast(eq, rv);
  T err[6] = {tp[0] - pp[0], tp[1] - pp[1], tp[2] - pp[2], rv[0] * a.rot_weight, rv[1] * a.rot_weight,
              rv[2] * a.rot_weight};
  const T pe = finish_sqrt((err[0] * err[0] + err[1] * err[1]) + err[2] * err[2]);
  const T re = finish_sqrt((rv[0] * rv[0] + rv[1] * rv[1]) + rv[2] * rv[2]);
  const bool last = it >= a.k.max_iters;
  const bool conv = !last && (pe < a.k.pos_thresh) && (re < a.rot_thresh);
  if (active && (conv || last)) done(pp, qcur, pe, re, conv ? it + 1 : it, conv);
#pragma unroll
  for (int j = 0; j < NJ; ++j) { J[21 + j] *= a.rot_weight; J[28 + j] *= a.rot_weight; J[35 + j] *= a.rot_weight; }
  T A[6][6];
#pragma unroll
  for (int r = 0; r < 6; ++r)
#pragma unroll
    for (int c2 = 0; c2 <= r; ++c2) {
      T acc = T(0);
#pragma unroll
      for (int j = 0; j < NJ; ++j) acc = acc + J[r * 7 + j] * J[c2 * 7 + j];
      A[r][c2] = acc + (r == c2 ? a.k.damping : T(0));
    }
  ldlt_solve<T, 6>(A, err);
#pragma unroll
  for (int j = 0; j < NJ; ++j) {
    T dq = T(0);
#pragma unroll
    for (int r = 0; r < 6; ++r) dq = dq + J[r * 7 + j] * err[r];
    dq = clamp_t(dq, -a.k.step_limit, a.k.step_limit);
    q[j] = clamp_t(q[j] + dq, Kin::template lower<T>(j), Kin::template upper<T>(j));
  }
}

// the success rule of a finished pose solve
template <typename T>
__device__ __forceinline__ bool pose_success(const PoseIkArgs<T>& a, T pe, T re, bool conv) {
  return conv && (pe < a.k.pos_thresh * T(2)) && (re < a.rot_thresh * T(2));
}

// Store the record of query e (every output but q_out nullable)
template <typename T>
__device__ __forceinline__ void pose_store(const PoseIkArgs<T>& a, unsigned e, const T (&q)[NJ], const T* pp,
                                           const T* qcur, T pe, T re, int iterations, bool conv) {
  const bool success = pose_success(a, pe, re, conv);
#pragma unroll
  for (int i = 0; i < NJ; ++i) a.q_out[(size_t)e * NJ + i] = q[i];
  if (a.final_pos) { a.final_pos[(size_t)e * 3] = pp[0]; a.final_pos[(size_t)e * 3 + 1] = pp[1]; a.final_pos[(size_t)e * 3 + 2] = pp[2]; }
  if (a.final_quat) {
#pragma unroll
    for (int i = 0; i < 4; ++i) a.final_quat[(size_t)e * 4 + i] = qcur[i];
  }
  if (a.pos_err) a.pos_err[e] = pe;
  if (a.rot_err) a.rot_err[e] = re;
  if (a.iters) a.iters[e] = iterations;
  if (a.flags) a.flags[e] = (uint8_t)((conv ? PNP_IK_CONVERGED : 0u) | (success ? PNP_IK_SUCCESS : 0u));
}

// Persistent warps with lane refill, like ik_solve_kernel: pose solves take 4-30 passes, and a grid of
// one-shot lanes ran every warp at the pace of its slowest query (25.9 of 32 lanes active per
// instruction, twice the mean pass count).  The FP32 instantiation uses the table trig.
template <typename T, typename Kin>
__global__ void __launch_bounds__(IK_BLOCK) ik_pose_solve_kernel(const PoseIkArgs<T> a) {
  __shared__ __align__(16) float s_tab[Trig<T>::kUsesTable ? kTrigVWords : 4];
  if (Trig<T>::kUsesTable) load_trigv_table(s_tab);
  __syncthreads();
  if (a.solo_warp && threadIdx.x >= 32) return;  // helper warps of a small-batch block: table loaded, done
  const Trig<T> trig{s_tab};
  unsigned long long c_n = 0, c_conv = 0, c_iter = 0;
  WarpPool pool;
  bool exhausted = false, active = false;
  unsigned e = 0;
  int it = 0;
  T q[NJ], tp[3] = {T(0), T(0), T(0)}, tq[4] = {T(1), T(0), T(0), T(0)};
#pragma unroll
  for (int i = 0; i < NJ; ++i) q[i] = T(0);

  while (true) {
    // ---- refill idle lanes -------------------------------------------------------------------
    const bool want[1] = {!active && !exhausted};
    pool.refill(want, exhausted, a.n, a.ticket, a.chunk, [&](int, unsigned idx) {
          e = idx;
          const T* qi = a.q_init + (size_t)a.q_init_stride * e;
#pragma unroll
          for (int i = 0; i < NJ; ++i) q[i] = qi[i];
          pose_load_target(a, e, tp, tq);
          it = 0;
          active = true;
        });
    if (!__any_sync(FULL, active)) break;

    // ---- one 6-row DLS pass for all lanes (a lane that just finished is idle and is overwritten by the next refill) --
    pose_pass<T, Kin>(a, trig, q, tp, tq, it, active,
                      [&](const T* pp, const T* qcur, T pe, T re, int iterations, bool conv) {
                        pose_store(a, e, q, pp, qcur, pe, re, iterations, conv);
                        c_n += 1; c_conv += conv ? 1 : 0; c_iter += (unsigned long long)iterations;
                        active = false;
                      });
    ++it;
  }
  ik_counters_add(a.counters, c_n, c_conv, c_iter);
}

// ---- multi-start pose IK (pnp_ik_pose_solve_multistart_*) ---------------------------------------------------------
// The position multistart's machinery (ms_collect_kernel, ms_wave) on the pose solve: attempt 0 is
// ik_pose_solve_kernel; the collect kernel lists the queries whose flags[] lack PNP_IK_SUCCESS; wave w gives each listed
// query G lanes that run seeds [w G, w G + G) with pose_pass, the plain kernel's pass, from pose_load_target's target.
// The lowest successful lane of a group stores the record with pose_store (every output the caller passed) and the
// attempt; queries without a success go onto the next wave's list.  Attempt 0's flags and iterations are read as in the
// position solver's separate layout (ms_ik_prev).
template <typename T, typename Kin>
__global__ void __launch_bounds__(MS_BLOCK) ms_pose_wave_kernel(const MsArgs<PoseIkArgs<T>> m) {
  const unsigned cnt = *m.cnt_in;
  if ((unsigned long long)blockIdx.x * 32u >= (unsigned long long)cnt * m.group) return;  // no work for any warp of this block
  __shared__ __align__(16) float s_tab[Trig<T>::kUsesTable ? kTrigVWords : 4];
  if (Trig<T>::kUsesTable) load_trigv_table(s_tab);
  __syncthreads();
  const Trig<T> trig{s_tab};
  // the finished attempt of this lane: q, pose and errors at the pass it finished in
  T qk[NJ], pk[3], qck[4], pek = T(0), rek = T(0);
  bool conv = false;
  int it_kept = 0;
  auto solve = [&](bool valid, unsigned id, int seed, bool& succ, int& iterations) {
    T q[NJ], tp[3], tq[4];
    pose_load_target(m.a, id, tp, tq);
#pragma unroll
    for (int i = 0; i < NJ; ++i) q[i] = m.seeds[seed * NJ + i];
    bool active = valid;
    conv = false;
    it_kept = 0;
    for (int it = 0; __any_sync(FULL, active); ++it)
      pose_pass<T, Kin>(m.a, trig, q, tp, tq, it, active,
                        [&](const T* pp, const T* qcur, T pe, T re, int its, bool cv) {
#pragma unroll
                          for (int i = 0; i < NJ; ++i) qk[i] = q[i];
#pragma unroll
                          for (int i = 0; i < 3; ++i) pk[i] = pp[i];
#pragma unroll
                          for (int i = 0; i < 4; ++i) qck[i] = qcur[i];
                          pek = pe; rek = re; it_kept = its; conv = cv;
                          active = false;
                        });
    iterations = it_kept;
    succ = pose_success(m.a, pek, rek, conv);
  };
  auto prev = [&](unsigned id, unsigned& fl, unsigned& it) { ms_ik_prev<IK_OUT_SEPARATE>(m, id, fl, it); };
  auto store = [&](unsigned id) { pose_store(m.a, id, qk, pk, qck, pek, rek, it_kept, conv); };
  ms_wave(m, cnt, solve, prev, store);
}

// =============================================================================================
// MoveIKSkill.reset trajectory planner (skills/move.py:76-191) as a per-lane state machine.
//
// One lane per env.  Every trip of the warp loop is ONE shared, divergence-free DLS pass
// (:128/:152/:168) for all lanes.  A lane whose solve finished in that pass post-processes it by
// state and then picks the IK target its new state asks for - NORMAL: the adaptive waypoint
// (:110-125); FB1: fallback strategy 1, a 10x smaller step (:149-151); FB2: strategy 2, the same
// step with y frozen (:163-167).  Post-processing: accept rule success && err < 2*step_size (:131), failure counter incl. the reference's
// double increment (:142,:183), fallback chaining, `break` when both fallbacks fail (:178-180),
// point_count only advanced on an accepted NORMAL step (:186), final target append (:189-191).
// The reference loop has no bound and spins forever on unreachable targets (fallback 1 keeps
// succeeding with ever smaller steps and never advances point_count); max_outer bounds the number
// of NORMAL rounds here and is reported in status bit 1.
// status bits: 1 = fallbacks exhausted (reference `break`), 2 = max_outer reached,
//              4 = trajectory capacity exceeded (traj_len keeps counting, extra points dropped).
// =============================================================================================
template <typename T>
struct MoveArgs {
  const T* q_start;
  const T* target;
  unsigned n;       // < 2^31 (checked on the host)
  T pos_thresh, step_size;
  int max_traj_points, max_outer, traj_cap;
  IkConst<T> k;
  T* traj;          // [n][traj_cap][3]
  int32_t* traj_len;
  T* q_final;       // [n][7]
  int32_t* n_solves;
  int32_t* status;
  unsigned long long* counters;
  unsigned* ticket; // zeroed before launch
  unsigned chunk;   // envs a warp reserves per ticket atomic
  unsigned solo_warp;  // small batches: 4 warps load the trig table, only warp 0 works
  const unsigned* order;  // nullable: env taken by the i-th ticket (longest plans first, plan_order_* kernels below)
  const float4* records;  // nullable (FP32 value-type kernel): the i-th ticket's inputs as one 48-byte record
                          // {q_start[7], target[3], env, -}, written in plan order by plan_order_scatter_kernel: a refill is
                          // one sequential read instead of order[i] -> q_start[env], two dependent random ones
};

// ---- longest plan first ------------------------------------------------------------------------------
// A plan is 2-200 warm solves long and a lane owns one env at a time, so a launch ends with lanes idle
// while the last long plans finish (2^18 envs in index order: 36 % over the balanced time).  The length of
// a plan is, to 0.997 correlation, a function of d0 = |goal - FK(q_start)| (move.py:110-125: steps of
// step_size, then the geometric tail), so the planner takes its envs in descending d0: a counting sort on
// PLAN_BUCKETS buckets of d0, two small launches (histogram, scatter), FK recomputed instead of stored.
// The order within a bucket is whatever the atomics give; the planner's outputs are indexed by env and do
// not depend on it.
constexpr int PLAN_BUCKETS = 128;     // 1/64 m per bucket, the last one open ended
constexpr int PLAN_ORDER_BLOCK = 256;
constexpr int PLAN_ORDER_PER_THREAD = 1;  // small batches want blocks, not work per thread: the sort sits in front of the planner

template <typename T, typename Kin>
__device__ __forceinline__ int plan_bucket(const T* q_start, const T* target, unsigned e) {
  T q[NJ], p[3];
#pragma unroll
  for (int i = 0; i < NJ; ++i) q[i] = q_start[(size_t)e * NJ + i];
  fk_position<T, Kin>(q, p);
  const T dx = target[(size_t)e * 3] - p[0], dy = target[(size_t)e * 3 + 1] - p[1], dz = target[(size_t)e * 3 + 2] - p[2];
  const float d0 = sqrtf((float)((dx * dx + dy * dy) + dz * dz));
  const float b = fminf(d0 * 64.0f, (float)(PLAN_BUCKETS - 1));  // fminf drops a NaN: it lands with the longest plans
  return PLAN_BUCKETS - 1 - (int)b;                              // bucket 0 = longest plans
}

// work[0..PLAN_BUCKETS) += histogram of the buckets (work zeroed before the launch)
template <typename T, typename Kin>
__global__ void __launch_bounds__(PLAN_ORDER_BLOCK) plan_order_hist_kernel(const T* q_start, const T* target, unsigned n,
                                                                            unsigned* work) {
  __shared__ unsigned s_cnt[PLAN_BUCKETS];
  if (threadIdx.x < PLAN_BUCKETS) s_cnt[threadIdx.x] = 0;
  __syncthreads();
  const unsigned base = blockIdx.x * (PLAN_ORDER_BLOCK * PLAN_ORDER_PER_THREAD);
#pragma unroll
  for (int j = 0; j < PLAN_ORDER_PER_THREAD; ++j) {
    const unsigned e = base + j * PLAN_ORDER_BLOCK + threadIdx.x;
    if (e < n) atomicAdd(&s_cnt[plan_bucket<T, Kin>(q_start, target, e)], 1u);
  }
  __syncthreads();
  if (threadIdx.x < PLAN_BUCKETS && s_cnt[threadIdx.x]) atomicAdd(&work[threadIdx.x], s_cnt[threadIdx.x]);
}

// order[start(bucket) + rank within bucket] = env; work[PLAN_BUCKETS..2*PLAN_BUCKETS) are the bucket cursors
template <typename T, typename Kin>
__global__ void __launch_bounds__(PLAN_ORDER_BLOCK) plan_order_scatter_kernel(const T* q_start, const T* target, unsigned n,
                                                                               unsigned* work, unsigned* order,
                                                                               float4* records = nullptr) {
  __shared__ unsigned s_hist[PLAN_BUCKETS], s_cnt[PLAN_BUCKETS], s_base[PLAN_BUCKETS];
  if (threadIdx.x < PLAN_BUCKETS) { s_hist[threadIdx.x] = work[threadIdx.x]; s_cnt[threadIdx.x] = 0; }
  __syncthreads();
  const unsigned base = blockIdx.x * (PLAN_ORDER_BLOCK * PLAN_ORDER_PER_THREAD);
  int bucket[PLAN_ORDER_PER_THREAD];
  unsigned rank[PLAN_ORDER_PER_THREAD];
#pragma unroll
  for (int j = 0; j < PLAN_ORDER_PER_THREAD; ++j) {
    const unsigned e = base + j * PLAN_ORDER_BLOCK + threadIdx.x;
    bucket[j] = 0; rank[j] = 0;
    if (e < n) {
      bucket[j] = plan_bucket<T, Kin>(q_start, target, e);
      rank[j] = atomicAdd(&s_cnt[bucket[j]], 1u);
    }
  }
  __syncthreads();
  if (threadIdx.x < PLAN_BUCKETS) {
    unsigned start = 0;
    for (int b = 0; b < (int)threadIdx.x; ++b) start += s_hist[b];
    const unsigned c = s_cnt[threadIdx.x];
    s_base[threadIdx.x] = start + (c ? atomicAdd(&work[PLAN_BUCKETS + threadIdx.x], c) : 0u);
  }
  __syncthreads();
#pragma unroll
  for (int j = 0; j < PLAN_ORDER_PER_THREAD; ++j) {
    const unsigned e = base + j * PLAN_ORDER_BLOCK + threadIdx.x;
    if (e < n) {
      const unsigned at = s_base[bucket[j]] + rank[j];
      if (order) order[at] = e;
      if (records) {  // (rows just read by plan_bucket: L1 / L2 hits)
        float v[10];
#pragma unroll
        for (int i = 0; i < NJ; ++i) v[i] = (float)q_start[(size_t)e * NJ + i];
#pragma unroll
        for (int i = 0; i < 3; ++i) v[7 + i] = (float)target[(size_t)e * 3 + i];
        float4* r = records + (size_t)at * 3u;
        r[0] = make_float4(v[0], v[1], v[2], v[3]);
        r[1] = make_float4(v[4], v[5], v[6], v[7]);
        r[2] = make_float4(v[8], v[9], __uint_as_float(e), 0.0f);
      }
    }
  }
}

// Is a caller-made `order` a permutation of [0, n)?  One pass: every entry sets its bit in a zeroed bitmap; an entry
// outside the batch or a bit already set counts as bad.  (The planner itself skips out-of-range entries; a repeated
// entry plans one env twice and leaves another one unplanned - this is how a caller finds out.)
__global__ void __launch_bounds__(256) plan_order_check_kernel(const unsigned* __restrict__ order, unsigned n,
                                                                unsigned* __restrict__ bitmap, unsigned* __restrict__ n_bad) {
  unsigned bad = 0;
  for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const unsigned e = order[i];
    if (e >= n) { ++bad; continue; }
    const unsigned bit = 1u << (e & 31u);
    if (atomicOr(&bitmap[e >> 5], bit) & bit) ++bad;
  }
  bad = (unsigned)warp_sum((unsigned long long)bad);
  if ((threadIdx.x & 31u) == 0 && bad) atomicAdd(n_bad, bad);
}

// The planner's scalar bookkeeping in the two precisions: FP64 follows the reference's operations
// literally (sqrt, a*b/c, (a/c)*b); FP32 - held to the 1e-4 m tolerance, not to bit parity - uses one
// MUFU each (x*rsqrt(x), a*b*rcp(c)): the bookkeeping runs on every pass of the flattened loop, and
// IEEE division / sqrt sequences were a fifth of its instructions.
__device__ __forceinline__ double norm_fast(double d2) { return sqrt(d2); }
__device__ __forceinline__ float norm_fast(float d2) { return finish_sqrt(d2); }
__device__ __forceinline__ double muldiv(double a, double b, double c) { return a * b / c; }
__device__ __forceinline__ float muldiv(float a, float b, float c) { return a * b * rcp_approx(c); }
__device__ __forceinline__ double divmul(double a, double c, double b) { return (a / c) * b; }
__device__ __forceinline__ float divmul(float a, float c, float b) { return a * rcp_approx(c) * b; }

// Persistent warps with lane refill (like ik_solve_kernel): trajectories differ in length (40-200
// rounds), so a lane whose env is finished writes it back and takes the next env instead of idling
// until the longest trajectory of its warp ends.  A fresh env enters in state INIT and gets its
// start position FK(q_start) (move.py:91) from the shared DLS pass of that round - no divergent FK.
// The planner's loop and the solver's loop are FLATTENED: one DLS pass per trip of the warp loop; a
// lane whose solve finished post-processes it (accept rule, fallback transitions) and picks the target
// of its next solve in the same trip.  Lanes therefore never wait for the slowest solve of their warp
// (a failing fallback solve runs 100 passes, a warm accepted one 2), and a batch that mixes reachable
// and unreachable goals no longer runs at the pace of its capped envs.
template <typename T, typename Kin>
__global__ void __launch_bounds__(IK_BLOCK) move_ik_plan_kernel(const MoveArgs<T> a) {
  __shared__ __align__(16) float s_tab[Trig<T>::kUsesTable ? kTrigVWords : 4];
  if (Trig<T>::kUsesTable) load_trigv_table(s_tab);
  __syncthreads();
  if (a.solo_warp && threadIdx.x >= 32) return;  // helper warps of a small-batch block: table loaded, done
  const Trig<T> trig{s_tab};
  enum { NORMAL = 0, FB1 = 1, FB2 = 2, DONE = 3, INIT = 4, IDLE = 5 };
  unsigned long long c_n = 0, c_conv = 0, c_iter = 0;
  WarpPool pool;
  bool exhausted = false;
  unsigned e = 0;
  T q[NJ], qs[NJ], goal[3] = {T(0), T(0), T(0)}, pos[3] = {T(0), T(0), T(0)}, tgt[3] = {T(0), T(0), T(0)};
#pragma unroll
  for (int i = 0; i < NJ; ++i) q[i] = qs[i] = T(0);
  T* traj = a.traj;
  int len = 0, solves = 0, st = 0, state = IDLE, it = 0;
  int point_count = 0, cf = 0, outer = 0;
  T astep = T(0);
  auto append = [&](const T* pt) {
    if (len < a.traj_cap) { traj[len * 3] = pt[0]; traj[len * 3 + 1] = pt[1]; traj[len * 3 + 2] = pt[2]; }
    else st |= 4;
    ++len;
  };

  while (true) {
    // ---- write back finished envs, refill idle lanes -------------------------------------------
    if (state == DONE) {
#pragma unroll
      for (int i = 0; i < NJ; ++i) a.q_final[(size_t)e * NJ + i] = q[i];
      a.traj_len[e] = len;
      if (a.n_solves) a.n_solves[e] = solves;
      if (a.status) a.status[e] = st;
      state = IDLE;
    }
    const bool want[1] = {state == IDLE && !exhausted};
    pool.refill(want, exhausted, a.n, a.ticket, a.chunk, [&](int, unsigned idx) {
          const unsigned eo = a.order ? a.order[idx] : idx;
          if (eo < a.n) {  // an out-of-range entry of a caller-made order is skipped: nothing is read or written for it
            e = eo;
#pragma unroll
            for (int i = 0; i < NJ; ++i) q[i] = qs[i] = a.q_start[(size_t)e * NJ + i];
#pragma unroll
            for (int i = 0; i < 3; ++i) goal[i] = a.target[(size_t)e * 3 + i];
            traj = a.traj + (size_t)e * a.traj_cap * 3;
            len = 0; solves = 0; st = 0; point_count = 0; cf = 0; outer = 0; astep = T(0);
            state = INIT;
          }
        });
    if (!__any_sync(FULL, state != IDLE)) break;

    // ---- one DLS pass for all lanes (ik_solver.py:58-83); INIT lanes only take FK(q_start) from it ----
    T n2, qn[NJ], pp[3];
    ik_eval_and_step<T, Kin>(qs, tgt, a.k, trig, pp, n2, qn);

    bool choose = false;  // this lane starts a new solve: pick its IK target below
    if (state == INIT) {
      pos[0] = pp[0]; pos[1] = pp[1]; pos[2] = pp[2];                                 // :91 start_pos = FK(q_start)
      append(pos);                                                                    // :98
      state = NORMAL;
      choose = true;
    } else if (state == NORMAL || state == FB1 || state == FB2) {
      const bool last = it >= a.k.max_iters;
      const bool conv = !last && below_thresh(n2, a.k);
      if (conv || last) {
        // ---- the solve of this lane finished: post-process by state ------------------------------
        const T err = finish_sqrt(n2);
        const int iters = conv ? it + 1 : it;
        const T dx = goal[0] - pos[0], dy = goal[1] - pos[1], dz = goal[2] - pos[2];  // :110 (pos of this solve)
        const T dist = norm_fast((dx * dx + dy * dy) + dz * dz);                      // :111
        ++solves;
        c_n += 1; c_conv += conv ? 1 : 0; c_iter += (unsigned long long)iters;
        const bool success = conv && (err < a.k.pos_thresh * T(2));                   // ik_solver.py:92
        const bool accept = state == NORMAL ? (success && err < a.step_size * T(2)) : success;  // :131/:154/:170
        if (accept) {
          append(pp);
#pragma unroll
          for (int i = 0; i < NJ; ++i) q[i] = qs[i];
          pos[0] = pp[0]; pos[1] = pp[1]; pos[2] = pp[2];
          cf = 0;
          if (state == NORMAL) ++point_count;                                         // :186 (fallbacks `continue`)
          state = NORMAL;
        } else {
          bool try_fb2 = false;
          if (state == NORMAL) {
            ++cf;                                                                     // :142
            if (cf >= 3) {                                                            // :144
              if (dist > astep * T(0.1)) state = FB1; else try_fb2 = true;            // :150
            } else {
              ++cf;                                                                   // :183
            }
          } else if (state == FB1) {
            try_fb2 = true;
          } else {                                                                    // FB2 failed
            st |= 1;                                                                  // :178-180
            state = DONE;
            if (dist > a.pos_thresh) append(goal);                                    // :189-191
          }
          if (try_fb2) {
            const T an = norm_fast((dx * dx + T(0)) + dz * dz);                       // :165
            if (an > T(0.001)) {
              state = FB2;
            } else {
              st |= 1;
              state = DONE;
              if (dist > a.pos_thresh) append(goal);
            }
          }
        }
        choose = state != DONE;
      } else {
#pragma unroll
        for (int i = 0; i < NJ; ++i) qs[i] = qn[i];
        ++it;
      }
    }

    // ---- choose the IK target of the solve that starts in the next pass ---------------------------
    if (choose) {
      const T dx = goal[0] - pos[0], dy = goal[1] - pos[1], dz = goal[2] - pos[2];    // :110
      const T dist = norm_fast((dx * dx + dy * dy) + dz * dz);                        // :111 (== :106 norm)
      if (state == NORMAL) {
        if (!(dist > a.pos_thresh && point_count < a.max_traj_points)) {              // :106-107
          state = DONE;
        } else if (outer >= a.max_outer) {
          st |= 2;
          state = DONE;
        } else {
          ++outer;
          T stp = fmin(fmin(a.step_size, dist * T(0.1)), T(0.02));                    // :114-117
          if (cf > 0) stp = stp * T(0.5);                                             // :118-119
          astep = stp;
          if (dist > stp) {                                                           // :122-125
            tgt[0] = pos[0] + muldiv(dx, stp, dist); tgt[1] = pos[1] + muldiv(dy, stp, dist); tgt[2] = pos[2] + muldiv(dz, stp, dist);
          } else {
            tgt[0] = goal[0]; tgt[1] = goal[1]; tgt[2] = goal[2];
          }
        }
        if (state == DONE && dist > a.pos_thresh) append(goal);                       // :189-191
      } else if (state == FB1) {
        const T smaller = astep * T(0.1);                                             // :149-151
        tgt[0] = pos[0] + muldiv(dx, smaller, dist); tgt[1] = pos[1] + muldiv(dy, smaller, dist); tgt[2] = pos[2] + muldiv(dz, smaller, dist);
      } else {  // FB2
        const T an = norm_fast((dx * dx + T(0)) + dz * dz);                           // :163-167
        tgt[0] = pos[0] + divmul(dx, an, astep); tgt[1] = pos[1] + divmul(T(0), an, astep); tgt[2] = pos[2] + divmul(dz, an, astep);
      }
#pragma unroll
      for (int i = 0; i < NJ; ++i) qs[i] = q[i];                                      // every solve starts from q_current
      it = 0;
    }
  }
  ik_counters_add(a.counters, c_n, c_conv, c_iter);
}

// =============================================================================================
// Pose-mode move planner (pnp_move_ik_plan_pose_*, an EXTENSION stated in oracle/move_pose_oracle.py): plan a move to
// a goal position AND orientation, every waypoint a solved pose with its joints.
//   round: d = goal_pos - p, w = quat2vel(goal_quat (x) conj(r)); done when |d| <= pos_thresh and |w| <= rot_thresh,
//          CAPPED at max_traj_points points; f = min(1, step_size / |d|, rot_step / |w|)
//   up to three pose solves from q at the fractions f, f/2, f/20 of (d, w) (the goal itself when the fraction is 1);
//   the first success appends (final_pos, final_quat, q) and moves there; three rejections: BROKE.
// Same lane machinery as move_ik_plan_kernel: one env per lane, persistent warps refilled from WarpPool, one shared
// pose_pass per warp trip.  Every waypoint solve is pose_pass / pose_success unchanged, i.e. the plain pose solve of
// that aim from that q (ik_pose_solve_kernel's arithmetic).  A fresh env enters as INIT with its pass number set to
// max_iters: the pass then ends at once and hands the lane FK(q_start) - no divergent FK.
// =============================================================================================
template <typename T>
struct MovePoseArgs {
  PoseIkArgs<T> ik;  // every waypoint's pose solve: k, rot_thresh (= ik_rot_thresh), rot_weight; target_pos /
                     // target_quat = the goals (pose_load_target); n, counters, ticket, chunk, solo_warp
  const T* q_start;
  T pos_thresh, rot_thresh, step_size, rot_step;
  int max_traj_points, traj_cap;
  T* pos_traj;       // [n][traj_cap][3]
  T* quat_traj;      // [n][traj_cap][4]
  T* q_traj;         // [n][traj_cap][7], nullable
  int32_t* traj_len;
  T* q_final;        // [n][7]
  int32_t* n_solves;
  int32_t* status;
};

// a / b: FP64 literally, FP32 on one MUFU.RCP (the planner's bookkeeping, as muldiv / divmul above)
__device__ __forceinline__ double div_fast(double a, double b) { return a / b; }
__device__ __forceinline__ float div_fast(float a, float b) { return a * rcp_approx(b); }

template <typename T, typename Kin>
__global__ void __launch_bounds__(IK_BLOCK) move_pose_plan_kernel(const MovePoseArgs<T> a) {
  __shared__ __align__(16) float s_tab[Trig<T>::kUsesTable ? kTrigVWords : 4];
  if (Trig<T>::kUsesTable) load_trigv_table(s_tab);
  __syncthreads();
  if (a.ik.solo_warp && threadIdx.x >= 32) return;  // helper warps of a small-batch block: table loaded, done
  const Trig<T> trig{s_tab};
  enum { SOLVE = 0, DONE = 1, INIT = 2, IDLE = 3 };
  unsigned long long c_n = 0, c_conv = 0, c_iter = 0;
  WarpPool pool;
  bool exhausted = false, bad_goal = false;
  unsigned e = 0;
  size_t row = 0;  // e * traj_cap
  // q: joints of the last point; qs: the running solve; (p, r): pose of the last point; (tp, tq): the running aim
  T q[NJ], qs[NJ], p[3] = {T(0), T(0), T(0)}, r[4] = {T(1), T(0), T(0), T(0)};
  T gp[3] = {T(0), T(0), T(0)}, gq[4] = {T(1), T(0), T(0), T(0)}, tp[3] = {T(0), T(0), T(0)}, tq[4] = {T(1), T(0), T(0), T(0)};
#pragma unroll
  for (int i = 0; i < NJ; ++i) q[i] = qs[i] = T(0);
  int len = 0, solves = 0, st = 0, state = IDLE, it = 0, points = 0, attempt = 0;
  auto append = [&]() {
    if (len < a.traj_cap) {
      const size_t k = row + (size_t)len;
#pragma unroll
      for (int i = 0; i < 3; ++i) a.pos_traj[k * 3 + i] = p[i];
#pragma unroll
      for (int i = 0; i < 4; ++i) a.quat_traj[k * 4 + i] = r[i];
      if (a.q_traj) {
#pragma unroll
        for (int i = 0; i < NJ; ++i) a.q_traj[k * NJ + i] = q[i];
      }
    } else {
      st |= (int)PNP_MOVE_OVERFLOW;
    }
    ++len;
  };

  while (true) {
    // ---- write back finished envs, refill idle lanes -------------------------------------------
    if (state == DONE) {
#pragma unroll
      for (int i = 0; i < NJ; ++i) a.q_final[(size_t)e * NJ + i] = q[i];
      a.traj_len[e] = len;
      a.n_solves[e] = solves;
      a.status[e] = st;
      state = IDLE;
    }
    const bool want[1] = {state == IDLE && !exhausted};
    pool.refill(want, exhausted, a.ik.n, a.ik.ticket, a.ik.chunk, [&](int, unsigned idx) {
          e = idx;
#pragma unroll
          for (int i = 0; i < NJ; ++i) q[i] = qs[i] = a.q_start[(size_t)e * NJ + i];
          pose_load_target(a.ik, e, gp, gq);
          bad_goal = false;
#pragma unroll
          for (int i = 0; i < 3; ++i) bad_goal = bad_goal || !isfinite(gp[i]);
#pragma unroll
          for (int i = 0; i < 4; ++i) bad_goal = bad_goal || !isfinite(gq[i]);  // a zero quaternion normalises to NaN
#pragma unroll
          for (int i = 0; i < 3; ++i) tp[i] = gp[i];
#pragma unroll
          for (int i = 0; i < 4; ++i) tq[i] = gq[i];
          row = (size_t)e * (size_t)a.traj_cap;
          len = 0; solves = 0; st = 0; points = 0; attempt = 0;
          it = a.ik.k.max_iters;
          state = INIT;
        });
    if (!__any_sync(FULL, state != IDLE)) break;

    // ---- one 6-row DLS pass for all lanes; a lane whose solve ends post-processes it --------------
    bool choose = false;  // this lane starts a new solve: pick its aim below
    pose_pass<T, Kin>(a.ik, trig, qs, tp, tq, it, state != IDLE,
                      [&](const T* pp, const T* qcur, T pe, T re, int iterations, bool conv) {
                        bool accept = true;  // INIT: point 0 = FK(q_start)
                        if (state == SOLVE) {
                          ++solves;
                          c_n += 1; c_conv += conv ? 1 : 0; c_iter += (unsigned long long)iterations;
                          accept = pose_success(a.ik, pe, re, conv);
                          if (accept) {
#pragma unroll
                            for (int i = 0; i < NJ; ++i) q[i] = qs[i];
                            ++points;
                          }
                        }
                        if (accept) {
#pragma unroll
                          for (int i = 0; i < 3; ++i) p[i] = pp[i];
#pragma unroll
                          for (int i = 0; i < 4; ++i) r[i] = qcur[i];
                          append();
                          attempt = 0;
                        } else if (++attempt == 3) {
                          st |= (int)PNP_MOVE_BROKE;
                        }
                        state = attempt == 3 ? DONE : SOLVE;
                        choose = state == SOLVE;
                      });

    // ---- stop tests at the start of a round, then the aim of the next solve ------------------------
    if (choose) {
      const T d[3] = {gp[0] - p[0], gp[1] - p[1], gp[2] - p[2]};
      const T dist = finish_sqrt((d[0] * d[0] + d[1] * d[1]) + d[2] * d[2]);
      // goal (x) conj(r) and its angle, written as pose_pass writes the solver's error: a solve aimed at the goal that
      // converges ends the plan by construction (pos_thresh >= the IK's, rot_thresh >= ik_rot_thresh)
      const T eq[4] = {gq[0] * r[0] + gq[1] * r[1] + gq[2] * r[2] + gq[3] * r[3],
                       -gq[0] * r[1] + gq[1] * r[0] - gq[2] * r[3] + gq[3] * r[2],
                       -gq[0] * r[2] + gq[1] * r[3] + gq[2] * r[0] - gq[3] * r[1],
                       -gq[0] * r[3] - gq[1] * r[2] + gq[2] * r[1] + gq[3] * r[0]};
      T w[3];
      quat2vel_fast(eq, w);
      const T th = finish_sqrt((w[0] * w[0] + w[1] * w[1]) + w[2] * w[2]);
      if (attempt == 0) {
        if (bad_goal) {
          st |= (int)PNP_MOVE_BROKE;
          state = DONE;
        } else if (dist <= a.pos_thresh && th <= a.rot_thresh) {
          state = DONE;
        } else if (points >= a.max_traj_points) {
          st |= (int)PNP_MOVE_CAPPED;
          state = DONE;
        }
      }
      if (state == SOLVE) {
        T f = T(1);
        if (dist > T(0)) f = fmin(f, div_fast(a.step_size, dist));
        if (th > T(0)) f = fmin(f, div_fast(a.rot_step, th));
        const T g = attempt == 0 ? f : f * (attempt == 1 ? T(0.5) : T(0.05));
        if (g == T(1)) {
#pragma unroll
          for (int i = 0; i < 3; ++i) tp[i] = gp[i];
#pragma unroll
          for (int i = 0; i < 4; ++i) tq[i] = gq[i];
        } else {
#pragma unroll
          for (int i = 0; i < 3; ++i) tp[i] = p[i] + g * d[i];
          // aim rotation quat(g w) (x) r, one sincos of the half angle
          T s, c;
          trig(T(0.5) * g * th, &s, &c);
          const T k = th > T(0) ? div_fast(s, th) : T(0);
          const T h[4] = {c, k * w[0], k * w[1], k * w[2]};
          tq[0] = h[0] * r[0] - h[1] * r[1] - h[2] * r[2] - h[3] * r[3];
          tq[1] = h[0] * r[1] + h[1] * r[0] + h[2] * r[3] - h[3] * r[2];
          tq[2] = h[0] * r[2] - h[1] * r[3] + h[2] * r[0] + h[3] * r[1];
          tq[3] = h[0] * r[3] + h[1] * r[2] - h[2] * r[1] + h[3] * r[0];
        }
#pragma unroll
        for (int i = 0; i < NJ; ++i) qs[i] = q[i];  // every solve starts from the joints of the last point
        it = 0;
      }
    } else {
      ++it;
    }
  }
  ik_counters_add(a.ik.counters, c_n, c_conv, c_iter);
}

// =============================================================================================
// compute_reward / _is_success streaming kernel (panda_env.py:205-245, 303-306).
//
// HBM-bound: 60 B in + 4 B out per row (FP32 storage).  Each lane owns kRows consecutive rows
// so that every [n,3] array is read as three 128-bit loads per lane (48 contiguous bytes), the
// quaternion as kRows 128-bit loads, width / task as one vector load: 15 independent 128-bit
// loads in flight per lane, no shared-memory round trip needed for the 12-byte stride.
// Arithmetic: FP64 with explicit _rn intrinsics (never contracted to FMA), the reference's
// operation order, one final round-to-nearest cast -> bit-exact with NumPy/Python float64.
// =============================================================================================
// Host-prepared constants.  The two distance tests of the reference compare a correctly
// rounded FP64 sqrt against a threshold: sqrt_rn(s) < t.  sqrt_rn is monotone, so the test is
// EXACTLY equivalent to s < S with S = min{s : sqrt_rn(s) >= t}, found on the host by a
// nextafter search (pnp_capi.cu: sqrt_preimage).  That removes one FP64 sqrt per row (d_place is
// only ever compared) and makes the other one conditional (d_reach is needed as a value only
// when it is below 0.05).  The +-1e-6 "threshold adjacent" report uses the same trick.
struct RewardConst {
  int sparse;
  int n_bonus;            // entries of bonus[] that are valid (task indices 0..n_bonus-1)
  double n_tasks;
  double h0, high_z;
  double s_place_lt;      // d_place < distance_threshold  <=>  s_place < s_place_lt
  double s_reach_lt;      // d_reach < 0.05                <=>  s_reach < s_reach_lt
  double s_place_adj_lo, s_place_adj_hi;  // |d_place - thr| < tol  <=>  lo <= s_place < hi
  double s_reach_adj_lo, s_reach_adj_hi;
  float width_lt_f32;     // (double)w < 0.045 <=> w < width_lt_f32 for FP32 storage
  double bonus[16];       // 0.5 * (task / n_tasks), evaluated in FP64 on the host (:244)
};

__device__ __forceinline__ double sumsq3_rn(double x, double y, double z) {
  // np.linalg.norm(v, axis=-1)**2 part: add.reduce(v*v) -> ((x*x + y*y) + z*z), separate mul/add
  return __dadd_rn(__dadd_rn(__dmul_rn(x, x), __dmul_rn(y, y)), __dmul_rn(z, z));
}
__device__ __forceinline__ double norm3_rn(double x, double y, double z) { return __dsqrt_rn(sumsq3_rn(x, y, z)); }

__device__ __forceinline__ bool width_closed(float w, const RewardConst& k) { return w < k.width_lt_f32; }
__device__ __forceinline__ bool width_closed(double w, const RewardConst&) { return w < 0.045; }

// One row of panda_env.py:205-245 (+ :303-306).  TIn is the storage type of the row; every
// value is widened to FP64 exactly, all arithmetic uses _rn intrinsics (never contracted).
template <typename TIn>
__device__ __forceinline__ float reward_row(const TIn* ag_, const TIn* dg_, const TIn* ee_, const TIn* eq_, TIn width,
                                            int task, const RewardConst& k, float* success, unsigned& placed_o,
                                            unsigned& gripped_o, unsigned& adjacent_o) {
  const double ag0 = (double)ag_[0], ag1 = (double)ag_[1], ag2 = (double)ag_[2];
  const double s_reach = sumsq3_rn(__dsub_rn((double)ee_[0], ag0), __dsub_rn((double)ee_[1], ag1),
                                   __dsub_rn((double)ee_[2], ag2));                           // :211 (squared)
  const double s_place = sumsq3_rn(__dsub_rn(ag0, (double)dg_[0]), __dsub_rn(ag1, (double)dg_[1]),
                                   __dsub_rn(ag2, (double)dg_[2]));                           // :212 (squared)
  const bool near = s_reach < k.s_reach_lt;                                          // d_reach < 0.05
  const bool placed = s_place < k.s_place_lt;                                        // :220
  const bool gripped = width_closed(width, k) && near;                               // :214-216
  *success = placed ? 1.0f : 0.0f;                                                   // :303-306
  placed_o = placed;
  gripped_o = gripped;
  adjacent_o = ((s_place >= k.s_place_adj_lo) && (s_place < k.s_place_adj_hi)) ||
               ((s_reach >= k.s_reach_adj_lo) && (s_reach < k.s_reach_adj_hi));
  if (k.sparse) return placed ? -0.0f : -1.0f;                                       // :227-228
  // :231-232  reward = -0.003; reward += -min(d_reach, 0.05)
  double r = __dadd_rn(-0.003, near ? -__dsqrt_rn(s_reach) : -0.05);
  if (gripped) {                                                                     // :234-236
    // :223-224 need_q = HORIZONTAL [0.70710678118654757, -0.70710678118654746, 0, 0] if ag.z >
    // high_pick_z else VERTICAL [1, 0, -0, 0]; the z / w products are +-0 for finite inputs and
    // vanish under abs(), so only two components are widened.
    const bool horiz = ag2 > k.high_z;
    const double n0 = horiz ? 0.7071067811865476 : 1.0;
    const double n1 = horiz ? -0.7071067811865475 : 0.0;
    const double dot = __dadd_rn(__dmul_rn((double)eq_[0], n0), __dmul_rn((double)eq_[1], n1));
    const double ori_err = __dsub_rn(1.0, fabs(dot));
    r = __dadd_rn(r, 2.0);
    r = __dadd_rn(r, __dsub_rn(1.0, ori_err));
    if (__dsub_rn(ag2, k.h0) > 0.04) r = __dadd_rn(r, 4.0);                          // :219, :238-239
  }
  if (placed) r = __dadd_rn(r, 10.0);                                                // :241-242
  const double bonus = ((unsigned)task < (unsigned)k.n_bonus)
                           ? k.bonus[task]
                           : __dmul_rn(0.5, __ddiv_rn((double)task, k.n_tasks));     // :244
  r = __dadd_rn(r, bonus);
  return __double2float_rn(r);                                                       // :245
}

template <typename TIn>
struct RewardArgs {
  const TIn *ag, *dg, *ee, *eq, *width;
  const int32_t* task;
  long long n;
  RewardConst k;
  float* reward;
  float* success;
  unsigned long long* counters;
};

template <typename TIn>
struct RowsPerLane {
  static constexpr int value = 16 / sizeof(TIn);  // float: 4 rows, double: 2 rows
};

// 128-bit streaming load (read-once data: do not allocate in L1)
__device__ __forceinline__ uint4 ldg_stream(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}

template <typename TIn, int N>
struct Pack {
  union {
    uint4 v[N * sizeof(TIn) / 16];
    TIn e[N];
  };
};

template <typename TIn, bool kVec>
__global__ void __launch_bounds__(256) reward_kernel(const RewardArgs<TIn> a) {
  constexpr int R = RowsPerLane<TIn>::value;
  const unsigned lane = threadIdx.x & 31u;
  unsigned long long c_placed = 0, c_gripped = 0, c_adj = 0;
  const long long n_groups = (a.n + R - 1) / R;
  for (long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x; g < n_groups;
       g += (long long)gridDim.x * blockDim.x) {
    const long long row0 = g * R;
    TIn ag[R * 3], dg[R * 3], ee[R * 3], eq[R * 4], wd[R];
    int32_t tk[R];
    const bool full = kVec && (row0 + R <= a.n);
    if (full) {
      Pack<TIn, R * 3> pa, pd, pe;
      Pack<TIn, R * 4> pq;
      Pack<TIn, R> pw;
#pragma unroll
      for (int v = 0; v < 3; ++v) {
        pa.v[v] = ldg_stream(reinterpret_cast<const uint4*>(a.ag + row0 * 3) + v);
        pd.v[v] = ldg_stream(reinterpret_cast<const uint4*>(a.dg + row0 * 3) + v);
        pe.v[v] = ldg_stream(reinterpret_cast<const uint4*>(a.ee + row0 * 3) + v);
      }
#pragma unroll
      for (int v = 0; v < 4; ++v) pq.v[v] = ldg_stream(reinterpret_cast<const uint4*>(a.eq + row0 * 4) + v);
      pw.v[0] = ldg_stream(reinterpret_cast<const uint4*>(a.width + row0));
      if constexpr (R == 4) {
        const uint4 t = ldg_stream(reinterpret_cast<const uint4*>(a.task + row0));
        tk[0] = (int)t.x; tk[1] = (int)t.y; tk[2] = (int)t.z; tk[3] = (int)t.w;
      } else {
        const int2 t = *reinterpret_cast<const int2*>(a.task + row0);
        tk[0] = t.x; tk[1] = t.y;
      }
#pragma unroll
      for (int i = 0; i < R * 3; ++i) { ag[i] = pa.e[i]; dg[i] = pd.e[i]; ee[i] = pe.e[i]; }
#pragma unroll
      for (int i = 0; i < R * 4; ++i) eq[i] = pq.e[i];
#pragma unroll
      for (int i = 0; i < R; ++i) wd[i] = pw.e[i];
    } else {
#pragma unroll
      for (int r = 0; r < R; ++r) {
        const long long row = (row0 + r < a.n) ? row0 + r : a.n - 1;
#pragma unroll
        for (int i = 0; i < 3; ++i) {
          ag[r * 3 + i] = a.ag[row * 3 + i];
          dg[r * 3 + i] = a.dg[row * 3 + i];
          ee[r * 3 + i] = a.ee[row * 3 + i];
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) eq[r * 4 + i] = a.eq[row * 4 + i];
        wd[r] = a.width[row];
        tk[r] = a.task[row];
      }
    }
    float rw[R], sc[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
      unsigned pl, gr, ad;
      rw[r] = reward_row<TIn>(ag + r * 3, dg + r * 3, ee + r * 3, eq + r * 4, wd[r], tk[r], a.k, &sc[r], pl, gr, ad);
      if (row0 + r < a.n) { c_placed += pl; c_gripped += gr; c_adj += ad; }
    }
    if (full) {
      if constexpr (R == 4) {
        *reinterpret_cast<float4*>(a.reward + row0) = make_float4(rw[0], rw[1], rw[2], rw[3]);
        if (a.success) *reinterpret_cast<float4*>(a.success + row0) = make_float4(sc[0], sc[1], sc[2], sc[3]);
      } else {
        *reinterpret_cast<float2*>(a.reward + row0) = make_float2(rw[0], rw[1]);
        if (a.success) *reinterpret_cast<float2*>(a.success + row0) = make_float2(sc[0], sc[1]);
      }
    } else {
#pragma unroll
      for (int r = 0; r < R; ++r)
        if (row0 + r < a.n) {
          a.reward[row0 + r] = rw[r];
          if (a.success) a.success[row0 + r] = sc[r];
        }
    }
  }
  if (a.counters) {
    c_placed = warp_sum(c_placed); c_gripped = warp_sum(c_gripped); c_adj = warp_sum(c_adj);
    if (lane == 0) {
      if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(a.counters + PNP_RW_CNT_N, (unsigned long long)a.n);
      atomicAdd(a.counters + PNP_RW_CNT_PLACED, c_placed);
      atomicAdd(a.counters + PNP_RW_CNT_GRIPPED, c_gripped);
      atomicAdd(a.counters + PNP_RW_CNT_THRESHOLD_ADJACENT, c_adj);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// One row, lowest latency: FrankaEnv.step evaluates compute_reward once per env.step (envs/panda_env.py:176-181) and
// test/reward_test.py:71-72 calls it one transition at a time.  `in` / `out` point into the pinned, mapped host mailbox
// of the single-query path (see ik_solve_one_kernel): one launch + one stream synchronisation, no cudaMemcpy, no
// counters memset.  FP64 storage (what the reference hands over), the same reward_row as the streaming kernel.
//   in [15] = achieved_goal3, desired_goal3, ee_pos3, ee_quat4 (wxyz), fingers_width, task_index (as a double)
//   out[3]  = reward, is_success, bits(placed | gripped << 1 | threshold_adjacent << 2)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32) reward_one_kernel(const double* __restrict__ in, const RewardConst k,
                                                        float* __restrict__ out) {
  if (threadIdx.x != 0) return;
  float succ;
  unsigned pl, gr, ad;
  const float r = reward_row<double>(in, in + 3, in + 6, in + 9, in[13], (int)in[14], k, &succ, pl, gr, ad);
  out[0] = r;
  out[1] = succ;
  out[2] = __uint_as_float(pl | (gr << 1) | (ad << 2));
}

// ---------------------------------------------------------------------------------------------
// The planner over the value types of pnp_vec.cuh (specialised tree, FP32): V = float plans one env per
// lane, V = F2 two (packed FFMA2/FMUL2/FADD2) - same operations, bit-identical results.  Same state
// machine and reference line numbers as move_ik_plan_kernel above, restructured so that the COMMON
// transitions run branch-free: with ~2 passes per warm solve half of the slots finish a solve in every
// pass, and as `if` blocks the post-processing was executed divergently on every trip (the scalar kernel
// runs at 0.23 of the FP32 peak, the waypoint kernel with branch-free bookkeeping at 0.50).
//   predicated : INIT, an accepted solve (append the point, q_current = result.q, pos = final_pos), the
//                adaptive waypoint of the next NORMAL solve (packed geometry for both slots)
//   divergent  : a rejected solve and the fallback chain (rare), the end of an env (once per env)
// A slot whose solve finishes in a pass is frozen for that pass (step limit 0); q_current of every slot
// lives in shared memory.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void stg1_if(bool pred, float* ptr, float x) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %0, 0;\n\t@p st.global.f32 [%1], %2;\n\t}"
               :: "r"((unsigned)pred), "l"(ptr), "f"(x) : "memory");
}

//
// kStage (one env per lane, blocks of PLAN_BLOCK = 160 threads, 4 per SM - the same 20 warps as 5 blocks of 128, with
// 12 KB of shared memory per block to spare): the trajectory point of an accepted solve - one per lane on nearly every
// pass - goes into a 4-point (48-byte) row of shared memory and leaves as three 128-bit stores once the row is full.
// Written straight to global memory the three 4-byte stores of a pass hit 32 different 128-byte lines each: 96 L1
// wavefronts per warp pass, 1.5x the algorithmic DRAM bytes in partial-sector write-backs, and 31 % of the launch
// (measured with the appends predicated off).  The last 1-3 points of an env and its final goal point are stored
// directly, once per env.  Needs traj_cap % 4 == 0 and a 16-byte aligned trajectory buffer (the host checks).
constexpr int PLAN_BLOCK = 160;
constexpr int PLAN_STAGE_PTS = 4;
constexpr size_t plan_smem_bytes(int slots, int block, bool stage) {
  return sizeof(float) * ((size_t)kTrigVWords + (size_t)slots * NJ * block + (stage ? (size_t)block * PLAN_STAGE_PTS * 3 : 0));
}
__device__ __forceinline__ void sts1_if(bool pred, float* ptr, float x) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %0, 0;\n\t@p st.shared.f32 [%1], %2;\n\t}"
               :: "r"((unsigned)pred), "r"((unsigned)__cvta_generic_to_shared(ptr)), "f"(x) : "memory");
}

template <typename V, bool kFuse, int kBlock = IK_BLOCK, bool kStage = false>
__global__ void __launch_bounds__(kBlock, (Slots<V>::kN == 2 || kBlock == PLAN_BLOCK) ? IK_PAIR_MIN_BLOCKS : 5) move_ik_plan_v_kernel(const MoveArgs<float> a) {
  constexpr int S = Slots<V>::kN;
  static_assert(!kStage || S == 1, "trajectory staging is written for one env per lane");
  // dynamic shared memory (the staged variant needs 53 KB, above the 48 KB a kernel may declare statically): plan_smem_bytes()
  extern __shared__ __align__(16) unsigned char plan_smem[];
  float* const s_trig = reinterpret_cast<float*>(plan_smem);
  float* const s_qa = s_trig + kTrigVWords;       // q_current of every slot: [(k * NJ + i) * kBlock + thread]
  float* const s_pts = s_qa + S * NJ * kBlock;    // kStage: [thread][point][xyz] (16-byte aligned: every term is a multiple of 16 B)
  load_trigv_table(s_trig);
  __syncthreads();
  if (a.solo_warp && threadIdx.x >= 32) return;  // helper warps of a small-batch block: table loaded, done
  const TrigV trig{s_trig};
  const float thresh2 = a.k.pos_thresh * a.k.pos_thresh;
  float* const qa = s_qa + threadIdx.x;
  enum { NORMAL = 0, FB1 = 1, FB2 = 2, DONE = 3, INIT = 4, IDLE = 5 };

  V qs[NJ], tgt[3], pos[3], goal[3], slim(0.0f);
  int state[S], it[S], len[S], solves[S], st[S], point_count[S], cf[S], outer[S];
  float astep[S];
  unsigned env[S];
  bool exhausted = false;
  unsigned long long c_n = 0, c_conv = 0, c_iter = 0;
  WarpPool pool;
#pragma unroll
  for (int i = 0; i < NJ; ++i) qs[i] = V(0.0f);
#pragma unroll
  for (int i = 0; i < 3; ++i) tgt[i] = pos[i] = goal[i] = V(0.0f);
#pragma unroll
  for (int k = 0; k < S; ++k) {
    state[k] = IDLE; it[k] = len[k] = solves[k] = st[k] = point_count[k] = cf[k] = outer[k] = 0; astep[k] = 0.0f; env[k] = 0;
  }
  int staged = 0, gbase = 0;  // kStage: points of this lane's env waiting in s_pts / already in global memory
  float* const my_pts = s_pts + (kStage ? threadIdx.x * (PLAN_STAGE_PTS * 3) : 0);
  // the point of an accepted solve (move.py:98,135,157,173): staged (kStage) or stored like the others
  auto append_take = [&](bool pred, int k, float x, float y, float z) {
    const bool room = len[k] < a.traj_cap;
    if (kStage) {
      float* sp = my_pts + staged * 3;
      sts1_if(pred && room, sp, x);
      sts1_if(pred && room, sp + 1, y);
      sts1_if(pred && room, sp + 2, z);
      staged += (pred && room) ? 1 : 0;
    } else {
      float* t = a.traj + ((size_t)env[k] * a.traj_cap + (room ? len[k] : 0)) * 3;
      stg1_if(pred && room, t, x);
      stg1_if(pred && room, t + 1, y);
      stg1_if(pred && room, t + 2, z);
    }
    st[k] |= (pred && !room) ? 4 : 0;
    len[k] += pred ? 1 : 0;
  };
  // traj[len] = point (move.py:191 and the failure exits), predicated; beyond traj_cap the point is dropped (status bit 4)
  auto append_if = [&](bool pred, int k, float x, float y, float z) {
    const bool room = len[k] < a.traj_cap;
    float* t = a.traj + ((size_t)env[k] * a.traj_cap + (room ? len[k] : 0)) * 3;
    stg1_if(pred && room, t, x);
    stg1_if(pred && room, t + 1, y);
    stg1_if(pred && room, t + 2, z);
    st[k] |= (pred && !room) ? 4 : 0;
    len[k] += pred ? 1 : 0;
  };

  while (true) {
    // ---- write back finished envs (once per env), refill idle slots ----------------------------------
#pragma unroll
    for (int k = 0; k < S; ++k) {
      if (state[k] == DONE) {
        const unsigned id = env[k];
        if (kStage) {  // the env's last 1-3 staged points (a full row left at the end of its pass)
          float* t = a.traj + ((size_t)id * a.traj_cap + gbase) * 3;
          for (int w = 0; w < staged * 3; ++w) t[w] = my_pts[w];
          staged = 0; gbase = 0;
        }
#pragma unroll
        for (int i = 0; i < NJ; ++i) a.q_final[(size_t)id * NJ + i] = qa[(k * NJ + i) * kBlock];
        a.traj_len[id] = len[k];
        if (a.n_solves) a.n_solves[id] = solves[k];
        if (a.status) a.status[id] = st[k];
        state[k] = IDLE;
      }
    }
    bool want[S];
#pragma unroll
    for (int k = 0; k < S; ++k) want[k] = state[k] == IDLE && !exhausted;
    pool.refill(want, exhausted, a.n, a.ticket, a.chunk, [&](int k, unsigned id) {
          float rec[12];
          unsigned e;
          if (a.records) {  // warp-uniform
            const float4 r0 = a.records[(size_t)id * 3u], r1 = a.records[(size_t)id * 3u + 1], r2 = a.records[(size_t)id * 3u + 2];
            rec[0] = r0.x; rec[1] = r0.y; rec[2] = r0.z; rec[3] = r0.w; rec[4] = r1.x; rec[5] = r1.y; rec[6] = r1.z;
            rec[7] = r1.w; rec[8] = r2.x; rec[9] = r2.y;
            e = __float_as_uint(r2.z);
          } else {
            e = a.order ? a.order[id] : id;
            if (e < a.n) {
#pragma unroll
              for (int i = 0; i < NJ; ++i) rec[i] = a.q_start[(size_t)e * NJ + i];
#pragma unroll
              for (int i = 0; i < 3; ++i) rec[7 + i] = a.target[(size_t)e * 3 + i];
            }
          }
          if (e < a.n) {  // an out-of-range entry of a caller-made order is skipped: nothing is read or written for it
            env[k] = e;
#pragma unroll
            for (int i = 0; i < NJ; ++i) {
              Slots<V>::set(qs[i], k, rec[i]);
              qa[(k * NJ + i) * kBlock] = rec[i];
            }
#pragma unroll
            for (int i = 0; i < 3; ++i) Slots<V>::set(goal[i], k, rec[7 + i]);
            len[k] = 0; solves[k] = 0; st[k] = 0; point_count[k] = 0; cf[k] = 0; outer[k] = 0; astep[k] = 0.0f; it[k] = 0;
            state[k] = INIT;
          }
        });
    bool any_live = false;
#pragma unroll
    for (int k = 0; k < S; ++k) any_live = any_live || state[k] != IDLE;
    if (!__any_sync(FULL, any_live)) break;

    // ---- one DLS pass for all slots of all lanes (ik_solver.py:58-83) ---------------------------------
    V p[3], pr[3], n2, ev[3], J[21], s0, c0, tb[3];  // pr: FK in joint 1's frame (ik_eval_j1_v); p: the same point in the world
    pnp_spec::spec_world_to_base_v<V>(tgt, tb);
    ik_eval_j1_v<V>(qs, tb, trig, pr, ev, n2, J, s0, c0);
    p_world_v<V>(pr, s0, c0, p);
    bool fin[S], iterating[S], reload[S], fused[S];
#pragma unroll
    for (int k = 0; k < S; ++k) {
      const bool solving = state[k] <= FB2;
      fin[k] = solving && (it[k] >= a.k.max_iters || Slots<V>::get(n2, k) < thresh2);
      iterating[k] = solving && !fin[k];
      Slots<V>::set(slim, k, iterating[k] ? a.k.step_limit : 0.0f);  // INIT / finishing / idle slots: frozen
    }
    // kFuse: the update moves behind the post-processing, so that the pass in which a solve is accepted (or the
    // INIT pass) is also the first iteration of the next solve - q_current is the q this pass was evaluated at,
    // hence the same p and J, only the target changes (see ik_waypoints_v_kernel)
    if (!kFuse) ik_step_v<V>(qs, J, ev, a.k.damping, slim);

    // ---- post-processing: common transitions predicated, rejected solves divergent -----------------------
    bool choose[S];  // slot needs the adaptive NORMAL waypoint of its next solve
#pragma unroll
    for (int k = 0; k < S; ++k) {
      const bool init = state[k] == INIT;
      const bool f = fin[k];
      const bool conv = it[k] < a.k.max_iters;
      const float err = finish_sqrt(Slots<V>::get(n2, k));
      const int iters = it[k] + (conv ? 1 : 0);
      const bool success = conv && (err < a.k.pos_thresh * 2.0f);                     // ik_solver.py:92
      const bool acc = f && (state[k] == NORMAL ? (success && err < a.step_size * 2.0f) : success);  // :131/:154/:170
      const bool rej = f && !acc;
      const bool take = init || acc;  // INIT: start_pos = FK(q_start) (:91,:98); accepted solve (:131-138 / :154-160 / :170-176)
      solves[k] += f ? 1 : 0;
      c_n += f ? 1u : 0u; c_conv += (f && conv) ? 1u : 0u; c_iter += f ? (unsigned)iters : 0u;
      const float px = Slots<V>::get(p[0], k), py = Slots<V>::get(p[1], k), pz = Slots<V>::get(p[2], k);
      append_take(take, k, px, py, pz);
      if (take) { Slots<V>::set(pos[0], k, px); Slots<V>::set(pos[1], k, py); Slots<V>::set(pos[2], k, pz); }
      const bool keep = acc && it[k] > 0;  // q_current = result.q
      if (keep) {
#pragma unroll
        for (int i = 0; i < NJ; ++i) qa[(k * NJ + i) * kBlock] = Slots<V>::get(qs[i], k);
      }
      // rejected: the next solve restarts from q_current; INIT / accepted on the first pass: q_current itself
      // (reloaded: the frozen limit clip may have moved an out-of-limits q_start)
      reload[k] = init || (f && !keep);
      fused[k] = take;
      if (!kFuse && reload[k]) {
#pragma unroll
        for (int i = 0; i < NJ; ++i) Slots<V>::set(qs[i], k, qa[(k * NJ + i) * kBlock]);
      }
      point_count[k] += (acc && state[k] == NORMAL) ? 1 : 0;                          // :186 (fallbacks `continue`)
      cf[k] = take ? 0 : cf[k];
      state[k] = take ? (int)NORMAL : state[k];
      choose[k] = take;
      if (rej) {
        // ---- rare: the scalar kernel's logic for a rejected solve, verbatim --------------------------------
        const float qx = Slots<V>::get(pos[0], k), qy = Slots<V>::get(pos[1], k), qz = Slots<V>::get(pos[2], k);
        const float gx = Slots<V>::get(goal[0], k), gy = Slots<V>::get(goal[1], k), gz = Slots<V>::get(goal[2], k);
        const float dx = gx - qx, dy = gy - qy, dz = gz - qz;                          // :110 (pos of this solve)
        const float dist = finish_sqrt((dx * dx + dy * dy) + dz * dz);                // :111
        bool try_fb2 = false;
        if (state[k] == NORMAL) {
          ++cf[k];                                                                    // :142
          if (cf[k] >= 3) {                                                           // :144
            if (dist > astep[k] * 0.1f) state[k] = FB1; else try_fb2 = true;          // :150
          } else {
            ++cf[k];                                                                  // :183
            choose[k] = true;                                                         // stays NORMAL, halved step next
          }
        } else if (state[k] == FB1) {
          try_fb2 = true;
        } else {                                                                      // FB2 failed
          st[k] |= 1;                                                                 // :178-180
          state[k] = DONE;
          append_if(dist > a.pos_thresh, k, gx, gy, gz);                              // :189-191
        }
        if (try_fb2) {
          const float an = finish_sqrt((dx * dx + 0.0f) + dz * dz);                   // :165
          if (an > 0.001f) {
            state[k] = FB2;
          } else {
            st[k] |= 1;
            state[k] = DONE;
            append_if(dist > a.pos_thresh, k, gx, gy, gz);
          }
        }
        if (state[k] == FB1) {
          const float f1 = astep[k] * 0.1f * rcp_approx(dist);                        // :149-151
          Slots<V>::set(tgt[0], k, qx + dx * f1); Slots<V>::set(tgt[1], k, qy + dy * f1); Slots<V>::set(tgt[2], k, qz + dz * f1);
        } else if (state[k] == FB2) {
          const float an = finish_sqrt((dx * dx + 0.0f) + dz * dz);                   // :163-167
          const float f2 = astep[k] * rcp_approx(an);
          Slots<V>::set(tgt[0], k, qx + dx * f2); Slots<V>::set(tgt[1], k, qy + 0.0f * f2); Slots<V>::set(tgt[2], k, qz + dz * f2);
        }
      }
      it[k] = (init || f) ? 0 : it[k] + 1;
    }
    // ---- the adaptive waypoint of the next NORMAL solve (:106-125), both slots in packed arithmetic ------
    {
      const V dx = v_sub(goal[0], pos[0]), dy = v_sub(goal[1], pos[1]), dz = v_sub(goal[2], pos[2]);   // :110
      const V d2 = pnp_fma(dz, dz, pnp_fma(dy, dy, pnp_mul(dx, dx)));
      V dist, stp, inv;
#pragma unroll
      for (int k = 0; k < S; ++k) {
        const float dk = finish_sqrt(Slots<V>::get(d2, k));                           // :111 (== :106 norm)
        float sk = fminf(fminf(a.step_size, dk * 0.1f), 0.02f);                       // :114-117
        sk = cf[k] > 0 ? sk * 0.5f : sk;                                              // :118-119
        Slots<V>::set(dist, k, dk);
        Slots<V>::set(stp, k, sk);
        Slots<V>::set(inv, k, rcp_approx(dk));
      }
      const V fr = pnp_mul(stp, inv);
      const V nx = pnp_fma(dx, fr, pos[0]), ny = pnp_fma(dy, fr, pos[1]), nz = pnp_fma(dz, fr, pos[2]);  // :122-125
#pragma unroll
      for (int k = 0; k < S; ++k) {
        const float dk = Slots<V>::get(dist, k), sk = Slots<V>::get(stp, k);
        const bool loop_ok = dk > a.pos_thresh && point_count[k] < a.max_traj_points;  // :106-107
        const bool capped = loop_ok && outer[k] >= a.max_outer;
        const bool go = choose[k] && loop_ok && !capped;
        const bool far = dk > sk;
        outer[k] += go ? 1 : 0;
        astep[k] = go ? sk : astep[k];
        fused[k] = fused[k] && go;
        if (go) {
          Slots<V>::set(tgt[0], k, far ? Slots<V>::get(nx, k) : Slots<V>::get(goal[0], k));
          Slots<V>::set(tgt[1], k, far ? Slots<V>::get(ny, k) : Slots<V>::get(goal[1], k));
          Slots<V>::set(tgt[2], k, far ? Slots<V>::get(nz, k) : Slots<V>::get(goal[2], k));
        }
        if (choose[k] && !go) {  // end of the env (once per env)
          st[k] |= capped ? 2 : 0;
          state[k] = DONE;
          append_if(dk > a.pos_thresh, k, Slots<V>::get(goal[0], k), Slots<V>::get(goal[1], k), Slots<V>::get(goal[2], k));  // :189-191
        }
      }
    }
    if (kStage) {  // a full row of four points leaves as three 128-bit stores (16-byte aligned: see the host checks)
      const bool full = staged == PLAN_STAGE_PTS;
      const float4* row = reinterpret_cast<const float4*>(my_pts);
      const float4 c0 = row[0], c1 = row[1], c2 = row[2];
      float* t = a.traj + ((size_t)env[0] * a.traj_cap + gbase) * 3;
      stg128_if(full, t, c0.x, c0.y, c0.z, c0.w);
      stg128_if(full, t + 4, c1.x, c1.y, c1.z, c1.w);
      stg128_if(full, t + 8, c2.x, c2.y, c2.z, c2.w);
      gbase += full ? PLAN_STAGE_PTS : 0;
      staged = full ? 0 : staged;
    }
    if (kFuse) {
      // error of the new targets at this pass's p: what the first pass of the next solve would compute
      V en[3], n2n, tbn[3];
      pnp_spec::spec_world_to_base_v<V>(tgt, tbn);
      target_err_j1_v<V>(tbn, pr, s0, c0, en, n2n);
#pragma unroll
      for (int k = 0; k < S; ++k) {
        // a new solve already within pos_thresh of its target stays frozen and is finished by the next pass
        fused[k] = fused[k] && a.k.max_iters > 0 && !(Slots<V>::get(n2n, k) < thresh2);
        if (fused[k]) {
#pragma unroll
          for (int i = 0; i < 3; ++i) Slots<V>::set(ev[i], k, Slots<V>::get(en[i], k));
          it[k] = 1;
        }
        Slots<V>::set(slim, k, (iterating[k] || fused[k]) ? a.k.step_limit : 0.0f);
      }
      ik_step_v<V>(qs, J, ev, a.k.damping, slim);
#pragma unroll
      for (int k = 0; k < S; ++k) {
        if (reload[k] && !fused[k]) {
#pragma unroll
          for (int i = 0; i < NJ; ++i) Slots<V>::set(qs[i], k, qa[(k * NJ + i) * kBlock]);
        }
      }
    }
  }
  ik_counters_add(a.counters, c_n, c_conv, c_iter);
}

// =============================================================================================
// HER relabel + obs assembly (SURVEY 8f-2): what `train.py:4` promises ("TQC(+HER)") and SB3's
// HerReplayBuffer would do per sampled transition - done in one streaming pass:
//   new_goal   = next_obs[future_idx].achieved_goal   (future_idx < 0: keep the stored goal)
//   obs.dg = next_obs.dg = new_goal
//   reward     = compute_reward(next_obs.achieved_goal, new_goal, info)   (bit-exact, reward_row)
//   is_success = ||ag - new_goal|| < distance_threshold
//   rows      -> VecNormalize.normalize_obs: clip((x - mean) / sqrt(var + eps), +-clip_obs)  (optional)
// Rows are the critic-ready layout [observation19 | achieved_goal3 | desired_goal3] in FP32
// (100 B).  ee_pos and fingers_width come from the row itself (observation[0:3], [6]); ee_quat
// and task_index are not part of the observation and ride in side arrays.
//
// Data movement: 100-byte rows are not 16-byte multiples, so tiles of 128 rows (12.8 KB per
// array) are staged through shared memory.  Full tiles use the Blackwell/Hopper bulk-async-copy
// engine (cp.async.bulk global->shared completing on an mbarrier, shared->global bulk store),
// double buffered: one elected thread moves 51 KB per tile while the other 127 only compute.
// Each lane owns one row of the tile in shared memory (stride 25 words: conflict-free).
// Algorithmic traffic 464 B per transition (SURVEY 8d): 200 read + 200 written + 64 reward stream.
// =============================================================================================
constexpr int HER_TILE = 128;
constexpr int HER_ROW = 25;
constexpr int HER_TILE_BYTES = HER_TILE * HER_ROW * 4;  // 12800

struct HerArgs {
  const float* obs;
  const float* next_obs;
  const int32_t* future_idx;
  const float* future_ag;  // optional [n_total][3] table of next achieved goals (what a replay buffer keeps
                           // anyway): the random gather then reads 12 B from a table that fits the L2
                           // instead of 12 B out of a 100-byte row (a 64-128 B DRAM burst each)
  const float* ee_quat;
  const int32_t* task;
  long long n;          // rows handled by this launch
  long long n_total;    // rows addressable through future_idx
  long long row0;       // first row of this launch (tail launches start past the full tiles)
  RewardConst k;
  float* out_obs;
  float* out_next;
  float* reward;
  float* success;
  int normalize;
  float clip;
  float mean_hi[HER_ROW];  // mean = mean_hi + mean_lo (two-float split of the FP64 statistic: the
  float mean_lo[HER_ROW];  // desired_goal columns have var ~1e-9, so x - mean must not lose the low bits)
  float inv_std[HER_ROW];
  unsigned long long* counters;
};

__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra.uni WAIT_DONE;\n"
      "bra.uni WAIT_LOOP;\n"
      "WAIT_DONE:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, unsigned bytes, unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void bulk_s2g(void* dst_gmem, const void* src_smem, unsigned bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem), "r"(smem_u32(src_smem)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read_all() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// relabel + reward + normalise one row held in shared memory (o = obs row, x = next_obs row)
__device__ __forceinline__ void her_row(const HerArgs& a, long long row, float* o, float* x, unsigned& pl, unsigned& gr,
                                        unsigned& ad) {
  const int fi = a.future_idx[row];
  float g[3] = {x[22], x[23], x[24]};
  if (fi >= 0 && (long long)fi < a.n_total) {  // an index past the end keeps the stored goal, like a negative one
    const float* src = a.future_ag ? a.future_ag + (long long)fi * 3
                                   : a.next_obs + (long long)fi * HER_ROW + 19;   // future achieved_goal (original rows)
    g[0] = src[0]; g[1] = src[1]; g[2] = src[2];
  }
  const float ag[3] = {x[19], x[20], x[21]};
  const float ee[3] = {x[0], x[1], x[2]};
  const float4 qv = *reinterpret_cast<const float4*>(a.ee_quat + row * 4);
  const float eq[4] = {qv.x, qv.y, qv.z, qv.w};
  float succ;
  const float r = reward_row<float>(ag, g, ee, eq, x[6], a.task[row], a.k, &succ, pl, gr, ad);
  a.reward[row] = r;
  if (a.success) a.success[row] = succ;
  o[22] = g[0]; o[23] = g[1]; o[24] = g[2];
  x[22] = g[0]; x[23] = g[1]; x[24] = g[2];
  if (a.normalize) {
#pragma unroll
    for (int k = 0; k < HER_ROW; ++k) {
      o[k] = fminf(fmaxf(((o[k] - a.mean_hi[k]) - a.mean_lo[k]) * a.inv_std[k], -a.clip), a.clip);
      x[k] = fminf(fmaxf(((x[k] - a.mean_hi[k]) - a.mean_lo[k]) * a.inv_std[k], -a.clip), a.clip);
    }
  }
}

template <bool kBulk>
__global__ void __launch_bounds__(HER_TILE) her_relabel_kernel(const HerArgs a) {
  extern __shared__ __align__(128) unsigned char her_smem[];
  float* buf = reinterpret_cast<float*>(her_smem);  // [stage][obs|next][HER_TILE*HER_ROW]
  __shared__ unsigned long long bar[2];
  const int tid = threadIdx.x;
  const unsigned lane = tid & 31u;
  unsigned long long c_placed = 0, c_gripped = 0, c_adj = 0;
  const long long n_tiles = (a.n + HER_TILE - 1) / HER_TILE;
  auto stage_ptr = [&](int stage, int which) { return buf + (stage * 2 + which) * (HER_TILE * HER_ROW); };

  if (kBulk) {
    if (tid == 0) { mbar_init(&bar[0], 1); mbar_init(&bar[1], 1); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    __syncthreads();
    long long t = blockIdx.x;
    if (t < n_tiles && tid == 0) {
      const long long r0 = a.row0 + t * HER_TILE;
      mbar_expect_tx(&bar[0], 2 * HER_TILE_BYTES);
      bulk_g2s(stage_ptr(0, 0), a.obs + r0 * HER_ROW, HER_TILE_BYTES, &bar[0]);
      bulk_g2s(stage_ptr(0, 1), a.next_obs + r0 * HER_ROW, HER_TILE_BYTES, &bar[0]);
    }
    for (int it = 0; t < n_tiles; t += gridDim.x, ++it) {
      const int stage = it & 1;
      const long long tn = t + gridDim.x;
      if (tid == 0 && tn < n_tiles) {
        bulk_wait_read_all();  // the store that last read stage^1 has drained its shared-memory reads
        const long long rn = a.row0 + tn * HER_TILE;
        mbar_expect_tx(&bar[stage ^ 1], 2 * HER_TILE_BYTES);
        bulk_g2s(stage_ptr(stage ^ 1, 0), a.obs + rn * HER_ROW, HER_TILE_BYTES, &bar[stage ^ 1]);
        bulk_g2s(stage_ptr(stage ^ 1, 1), a.next_obs + rn * HER_ROW, HER_TILE_BYTES, &bar[stage ^ 1]);
      }
      mbar_wait(&bar[stage], (unsigned)((it >> 1) & 1));
      const long long row = a.row0 + t * HER_TILE + tid;
      unsigned pl, gr, ad;
      her_row(a, row, stage_ptr(stage, 0) + tid * HER_ROW, stage_ptr(stage, 1) + tid * HER_ROW, pl, gr, ad);
      c_placed += pl; c_gripped += gr; c_adj += ad;
      fence_async_smem();  // generic-proxy writes -> visible to the bulk-copy (async) proxy
      __syncthreads();
      if (tid == 0) {
        const long long r0 = a.row0 + t * HER_TILE;
        bulk_s2g(a.out_obs + r0 * HER_ROW, stage_ptr(stage, 0), HER_TILE_BYTES);
        bulk_s2g(a.out_next + r0 * HER_ROW, stage_ptr(stage, 1), HER_TILE_BYTES);
        bulk_commit();
      }
    }
    if (tid == 0) bulk_wait_all();
  } else {
    for (long long t = blockIdx.x; t < n_tiles; t += gridDim.x) {
      const long long r0 = a.row0 + t * HER_TILE;
      const long long rows = (a.row0 + a.n - r0 < HER_TILE) ? a.row0 + a.n - r0 : HER_TILE;
      float* so = stage_ptr(0, 0);
      float* sx = stage_ptr(0, 1);
      for (int i = tid; i < rows * HER_ROW; i += HER_TILE) {
        so[i] = a.obs[r0 * HER_ROW + i];
        sx[i] = a.next_obs[r0 * HER_ROW + i];
      }
      __syncthreads();
      if (tid < rows) {
        unsigned pl, gr, ad;
        her_row(a, r0 + tid, so + tid * HER_ROW, sx + tid * HER_ROW, pl, gr, ad);
        c_placed += pl; c_gripped += gr; c_adj += ad;
      }
      __syncthreads();
      for (int i = tid; i < rows * HER_ROW; i += HER_TILE) {
        a.out_obs[r0 * HER_ROW + i] = so[i];
        a.out_next[r0 * HER_ROW + i] = sx[i];
      }
      __syncthreads();
    }
  }
  if (a.counters) {
    c_placed = warp_sum(c_placed); c_gripped = warp_sum(c_gripped); c_adj = warp_sum(c_adj);
    if (lane == 0) {
      if (blockIdx.x == 0 && tid == 0) atomicAdd(a.counters + PNP_RW_CNT_N, (unsigned long long)a.n);
      atomicAdd(a.counters + PNP_RW_CNT_PLACED, c_placed);
      atomicAdd(a.counters + PNP_RW_CNT_GRIPPED, c_gripped);
      atomicAdd(a.counters + PNP_RW_CNT_THRESHOLD_ADJACENT, c_adj);
    }
  }
}

// =============================================================================================
// get_obs_bulk_kernel: FrankaEnv._get_obs (same row arithmetic as get_obs_kernel, FP32) with ALL data
// movement on the bulk-async-copy engine.  A tile is 128 consecutive envs; its seven input slices
// (q_arm 3584 B, qvel_arm 3584 B, fingers 1024 B, obj_pos 1536 B, obj_quat 2048 B, obj_vel 3072 B,
// goal 1536 B) are contiguous in their arrays, so one elected thread fetches them with seven
// cp.async.bulk copies completing on an mbarrier, double buffered against the compute of the previous
// tile; the 12.8 KB of assembled rows overwrite the tile's own consumed input stage and leave with
// one bulk store.  72 KB of shared memory per block (two stages + the trig table), 3 blocks per SM.  The per-lane strided loads of
// get_obs_kernel left the warps on the long scoreboard for half of their time (ncu: 0.60 of the DRAM
// peak); here no lane ever issues a global load.  Full tiles of 16-byte aligned arrays only; tails and
// unaligned views run get_obs_kernel.
// =============================================================================================
struct ObsTileLayout {  // word offsets of the input slices inside one stage
  static constexpr int q = 0, qv = q + OBS_TILE * 7, fg = qv + OBS_TILE * 7, op = fg + OBS_TILE * 2,
                       oq = op + OBS_TILE * 3, ov = oq + OBS_TILE * 4, gl = ov + OBS_TILE * 6,
                       words = gl + OBS_TILE * 3;  // 4096 words = 16 KB
};
constexpr int OBS_STAGE_BYTES = ObsTileLayout::words * 4;
constexpr int OBS_OUT_BYTES = OBS_TILE * 25 * 4;
constexpr int OBS_BULK_SMEM = 2 * OBS_STAGE_BYTES + kTrigVWords * 4;  // 32 KB of stages (the rows of a tile overwrite its own
                                                                     // consumed input stage) + the 40 KB trig table

template <typename Kin>
__global__ void __launch_bounds__(OBS_TILE) get_obs_bulk_kernel(const ObsArgs<float> a) {
  using L = ObsTileLayout;
  extern __shared__ __align__(128) unsigned char obs_smem[];
  float* buf = reinterpret_cast<float*>(obs_smem);  // [2][L::words]
  float* s_trig = buf + 2 * L::words;               // [kTrigVWords]: the IK kernels' table trig
  __shared__ unsigned long long bar[2];
  load_trigv_table(s_trig);
  const Trig<float> trig{s_trig};
  const int tid = threadIdx.x;
  const long long n_tiles = a.n / OBS_TILE;  // full tiles only
  const bool per_env_goal = a.goal_stride != 0;
  const unsigned tile_bytes = (unsigned)(OBS_STAGE_BYTES - (per_env_goal ? 0 : OBS_TILE * 3 * 4));
  auto fetch = [&](long long t, int stage) {  // elected thread
    float* d = buf + stage * L::words;
    const long long e0 = t * OBS_TILE;
    mbar_expect_tx(&bar[stage], tile_bytes);
    bulk_g2s(d + L::q, a.q_arm + e0 * 7, OBS_TILE * 7 * 4, &bar[stage]);
    bulk_g2s(d + L::qv, a.qvel_arm + e0 * 7, OBS_TILE * 7 * 4, &bar[stage]);
    bulk_g2s(d + L::fg, a.fingers + e0 * 2, OBS_TILE * 2 * 4, &bar[stage]);
    bulk_g2s(d + L::op, a.obj_pos + e0 * 3, OBS_TILE * 3 * 4, &bar[stage]);
    bulk_g2s(d + L::oq, a.obj_quat + e0 * 4, OBS_TILE * 4 * 4, &bar[stage]);
    bulk_g2s(d + L::ov, a.obj_vel + e0 * 6, OBS_TILE * 6 * 4, &bar[stage]);
    if (per_env_goal) bulk_g2s(d + L::gl, a.goal + e0 * 3, OBS_TILE * 3 * 4, &bar[stage]);
  };
  if (tid == 0) { mbar_init(&bar[0], 1); mbar_init(&bar[1], 1); }
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  __syncthreads();
  float g0 = 0.0f, g1 = 0.0f, g2 = 0.0f;
  if (!per_env_goal) { g0 = a.goal[0]; g1 = a.goal[1]; g2 = a.goal[2]; }
  long long t = blockIdx.x;
  if (t < n_tiles && tid == 0) fetch(t, 0);
  for (int it = 0; t < n_tiles; t += gridDim.x, ++it) {
    const int stage = it & 1;
    const long long tn = t + gridDim.x;
    if (tid == 0 && tn < n_tiles) {
      bulk_wait_read_all();  // the store of the previous tile has drained its reads of stage^1
      fetch(tn, stage ^ 1);
    }
    mbar_wait(&bar[stage], (unsigned)((it >> 1) & 1));
    float* in = buf + stage * L::words;
    float o[25];
    {
      float s[NJ], c[NJ], qv[NJ];
#pragma unroll
      for (int k = 0; k < NJ; ++k) {
        trig(in[L::q + tid * 7 + k] - Kin::template qref<float>(k), &s[k], &c[k]);
        qv[k] = in[L::qv + tid * 7 + k];
      }
      float p[3], J[21];
#pragma unroll
      for (int k = 0; k < 21; ++k) J[k] = 0.0f;
      Kin::template fk_jacp<float>(s, c, p, J);
      o[0] = p[0]; o[1] = p[1]; o[2] = p[2];
#pragma unroll
      for (int r = 0; r < 3; ++r) {
        float acc = 0.0f;
#pragma unroll
        for (int j = 0; j < NJ; ++j) acc = acc + J[r * 7 + j] * qv[j];
        o[3 + r] = acc * a.dt;
      }
      o[6] = in[L::fg + tid * 2] + in[L::fg + tid * 2 + 1];
      const float4 qq = *reinterpret_cast<const float4*>(in + L::oq + tid * 4);
      float w = qq.x, x = qq.y, y = qq.z, z = qq.w;
      const float nrm = sqrt_t(w * w + x * x + y * y + z * z);
      if (nrm < 1e-15f) { w = 1.0f; x = y = z = 0.0f; } else { w = w / nrm; x = x / nrm; y = y / nrm; z = z / nrm; }
      const float q00 = w * w, q01 = w * x, q02 = w * y, q03 = w * z, q11 = x * x, q12 = x * y, q13 = x * z;
      const float q22 = y * y, q23 = y * z, q33 = z * z;
      const float m00 = q00 + q11 - q22 - q33, m01 = 2.0f * (q12 - q03), m02 = 2.0f * (q13 + q02);
      const float m10 = 2.0f * (q12 + q03), m11 = q00 - q11 + q22 - q33, m12 = 2.0f * (q23 - q01);
      const float m20 = 2.0f * (q13 - q02), m21 = 2.0f * (q23 + q01), m22 = q00 - q11 - q22 + q33;
      const float ox = in[L::op + tid * 3], oy = in[L::op + tid * 3 + 1], oz = in[L::op + tid * 3 + 2];
      o[7] = ox; o[8] = oy; o[9] = oz;
      const float cy = sqrt_t(m22 * m22 + m12 * m12);
      const bool cond = cy > (float)(4.0 * 2.220446049250313e-16);
      o[12] = -atan2_t(cond ? m01 : -m10, cond ? m00 : m11);  // one atan2 on selected arguments
      o[11] = -atan2_t(-m02, cy);
      o[10] = cond ? -atan2_t(m12, m22) : 0.0f;
      const float* v = in + L::ov + tid * 6;
      o[13] = v[0] * a.dt; o[14] = v[1] * a.dt; o[15] = v[2] * a.dt;
      o[16] = (m00 * v[3] + m01 * v[4] + m02 * v[5]) * a.dt;
      o[17] = (m10 * v[3] + m11 * v[4] + m12 * v[5]) * a.dt;
      o[18] = (m20 * v[3] + m21 * v[4] + m22 * v[5]) * a.dt;
      o[19] = ox; o[20] = oy; o[21] = oz;
      if (per_env_goal) { g0 = in[L::gl + tid * 3]; g1 = in[L::gl + tid * 3 + 1]; g2 = in[L::gl + tid * 3 + 2]; }
      o[22] = g0; o[23] = g1; o[24] = g2;
    }
    __syncthreads();  // every lane has read its inputs: the stage can be overwritten with the rows
#pragma unroll
    for (int k = 0; k < 25; ++k) in[tid * 25 + k] = o[k];
    fence_async_smem();  // generic-proxy writes -> visible to the bulk-copy (async) proxy
    __syncthreads();
    if (tid == 0) {
      bulk_s2g(a.out + t * (OBS_TILE * 25), in, OBS_OUT_BYTES);
      bulk_commit();
    }
  }
  if (tid == 0) bulk_wait_all();
}

// =============================================================================================
// fk_jac_bulk_kernel: fk_jac_kernel's arithmetic (FP32) with coalesced output.  One lane per configuration writes
// its 3 + 4 + 42 output words into shared-memory tiles of 128 configurations (the 168-byte-stride per-lane stores
// of fk_jac_kernel reach 0.12 of the HBM bandwidth); one elected thread sends each tile out with up to three
// cp.async.bulk stores (pos 1.5 KB, quat 2 KB, jac 21 KB), double buffered against the next tile's compute.
// Full tiles of 16-byte aligned outputs only; tails and unaligned views run fk_jac_kernel.
// =============================================================================================
constexpr int FK_TILE = 128;
constexpr int FK_STAGE_WORDS = FK_TILE * (3 + 4 + 42);          // pos | quat | jac
constexpr int FK_BULK_SMEM = 2 * FK_STAGE_WORDS * 4;            // 50176 B

template <typename Kin>
__global__ void __launch_bounds__(FK_TILE) fk_jac_bulk_kernel(const float* __restrict__ q, long long n_tiles,
                                                              float* __restrict__ pos, float* __restrict__ quat,
                                                              float* __restrict__ jac) {
  extern __shared__ __align__(128) unsigned char fk_smem[];
  float* buf = reinterpret_cast<float*>(fk_smem);
  const int tid = threadIdx.x;
  int it = 0;
  for (long long t = blockIdx.x; t < n_tiles; t += gridDim.x, ++it) {
    float* sp = buf + (it & 1) * FK_STAGE_WORDS;
    float* sq = sp + FK_TILE * 3;
    float* sj = sq + FK_TILE * 4;
    const long long i = t * FK_TILE + tid;
    float s[NJ], c[NJ];
#pragma unroll
    for (int k = 0; k < NJ; ++k) sincos_t(q[i * NJ + k] - Kin::template qref<float>(k), &s[k], &c[k]);
    float p[3], J[42], R[9];
    Kin::template fk_full<float>(s, c, p, J, R);
    // the stage written now was read by the bulk stores issued two tiles ago
    if (tid == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
    __syncthreads();
    sp[tid * 3 + 0] = p[0]; sp[tid * 3 + 1] = p[1]; sp[tid * 3 + 2] = p[2];
    if (quat) {
      float qu[4];
      mat2quat<float>(R, qu);
      *reinterpret_cast<float4*>(sq + tid * 4) = make_float4(qu[0], qu[1], qu[2], qu[3]);
    }
    if (jac) {
#pragma unroll
      for (int k = 0; k < 42; ++k) sj[tid * 42 + k] = J[k];
    }
    fence_async_smem();  // generic-proxy writes -> visible to the bulk-copy (async) proxy
    __syncthreads();
    if (tid == 0) {
      bulk_s2g(pos + t * (FK_TILE * 3), sp, FK_TILE * 3 * 4);
      if (quat) bulk_s2g(quat + t * (FK_TILE * 4), sq, FK_TILE * 4 * 4);
      if (jac) bulk_s2g(jac + t * (FK_TILE * 42), sj, FK_TILE * 42 * 4);
      bulk_commit();
    }
  }
  if (tid == 0) bulk_wait_all();
}

// goal_distance (panda_env.py:311-315)
__global__ void goal_distance_kernel(const double* __restrict__ a, const double* __restrict__ b, long long n,
                                     double* __restrict__ d) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n;
       i += (long long)gridDim.x * blockDim.x) {
    d[i] = norm3_rn(__dsub_rn(a[3 * i], b[3 * i]), __dsub_rn(a[3 * i + 1], b[3 * i + 1]),
                    __dsub_rn(a[3 * i + 2], b[3 * i + 2]));
  }
}

// =============================================================================================
// FFMA throughput probe: 8 independent accumulator chains per lane, 3-register-operand FFMAs.
// =============================================================================================
__global__ void __launch_bounds__(256) fp32_peak_kernel(float* out, int iters, float a, float b) {
  float x0 = threadIdx.x * 1e-3f, x1 = x0 + 1.f, x2 = x0 + 2.f, x3 = x0 + 3.f;
  float x4 = x0 + 4.f, x5 = x0 + 5.f, x6 = x0 + 6.f, x7 = x0 + 7.f;
  for (int i = 0; i < iters; ++i) {
#pragma unroll
    for (int u = 0; u < 16; ++u) {
      x0 = fmaf(x0, a, b); x1 = fmaf(x1, a, b); x2 = fmaf(x2, a, b); x3 = fmaf(x3, a, b);
      x4 = fmaf(x4, a, b); x5 = fmaf(x5, a, b); x6 = fmaf(x6, a, b); x7 = fmaf(x7, a, b);
    }
  }
  const float s = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
  if (s == 123.456f) out[0] = s;  // keep the chains alive
}

}  // namespace pnp

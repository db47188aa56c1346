// C ABI of libpnp_b200.so (declared in include/pnp_b200.h).  Host-side glue only: argument
// checks, constant-memory upload, launch geometry, the host-buffer pipeline.
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdarg>
#include <new>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <initializer_list>
#include <mutex>
#include <string>
#include <type_traits>

#include "pnp_kernels.cuh"

namespace {

thread_local std::string g_err;
std::atomic<unsigned long long> g_launches{0};

// Launch scratch (refill ticket, plan-order histograms) is keyed by STREAM: launches on one stream are ordered, so a
// stream's slot is free again by the time its next launch runs, whatever other streams are doing.  (Round 1 handed the
// slots out round-robin per launch: launch k and launch k+64 on different streams could share a live ticket.)
// The slots are allocated once in pnp_set_tree - never inside a launch, so capturing into a CUDA graph works - and a
// stream gets one on first use.  A captured graph keeps the slot of its capture stream: do not replay it concurrently
// with other work that was issued on that same stream object.  kStreamSlots distinct streams per device may have
// library launches in flight at a time; beyond that the least recently assigned slot is handed out again.
constexpr int kMaxDevices = 16;
constexpr int kStreamSlots = 64;

// What the previous ik_solve_v_kernel launch of a stream reads and writes, and which of the stream's two tickets the next
// one takes: the host side of the programmatic-dependent-launch overlap described at IK_PDL_* in pnp_kernels.cuh.
struct ByteRange {
  const char* b = nullptr;
  const char* e = nullptr;
};
struct IkPdlState {
  bool primed = false;      // the previous launch of this stream was an ik_solve_v_kernel that zeroed the ticket `parity`
  unsigned parity = 0;      // ticket the next launch draws from
  ByteRange in[2], out[5];  // of the previous launch (valid while primed)
  // drain hand-over (pair kernel -> resume kernel): two parking areas per stream, allocated on the stream's first big launch
  float2* dump[2] = {nullptr, nullptr};
  uint4* list[2] = {nullptr, nullptr};
  size_t rows_cap = 0;
  bool last_handover = false;  // the previous launch had a resume launch behind it (which zeroed this parity's counters)
};
// per stream and parity: {ticket, parked rows, parked slots, ticket of the resume launch}
constexpr int kIkScratchWords = 4;

struct DeviceState {
  bool have_tree = false;
  bool specialized = false;
  PnpTree tree{};
  int sm_count = 0;
  unsigned* tickets = nullptr;     // kStreamSlots refill tickets
  unsigned* order_work = nullptr;  // kStreamSlots blocks of 2*PLAN_BUCKETS words: plan-order histograms + cursors
  unsigned* ik_sc = nullptr;       // kStreamSlots x 2 parities x kIkScratchWords counters of ik_solve_v_kernel (launches alternate)
  IkPdlState ik_pdl[kStreamSlots];
  cudaStream_t slot_stream[kStreamSlots] = {};
  bool slot_used[kStreamSlots] = {};
  unsigned slot_clock = 0;
};
DeviceState g_dev[kMaxDevices];
std::mutex g_mu;

// the scratch slot of `st` on this device (see above); g_mu held by the caller
int stream_slot_locked(DeviceState* s, cudaStream_t st) {
  for (int i = 0; i < kStreamSlots; ++i)
    if (s->slot_used[i] && s->slot_stream[i] == st) return i;
  int i = 0;
  for (; i < kStreamSlots; ++i)
    if (!s->slot_used[i]) break;
  if (i == kStreamSlots) i = (int)(s->slot_clock++ % kStreamSlots);  // all taken: recycle, oldest assignment first
  s->slot_used[i] = true;
  s->slot_stream[i] = st;
  {  // a new owner: forget the previous stream's launch history, keep the parking areas
    IkPdlState fresh;
    for (int k = 0; k < 2; ++k) { fresh.dump[k] = s->ik_pdl[i].dump[k]; fresh.list[k] = s->ik_pdl[i].list[k]; }
    fresh.rows_cap = s->ik_pdl[i].rows_cap;  // (last_handover = false: the first launch memsets the counters)
    s->ik_pdl[i] = fresh;
  }
  return i;
}
int stream_slot(DeviceState* s, cudaStream_t st) {
  std::lock_guard<std::mutex> lk(g_mu);
  return stream_slot_locked(s, st);
}
ByteRange byte_range(const void* p, size_t bytes) { ByteRange r; if (p) { r.b = (const char*)p; r.e = r.b + bytes; } return r; }
bool ranges_overlap(const ByteRange& x, const ByteRange& y) { return x.b && y.b && x.b < y.e && y.b < x.e; }

int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}

int cuda_fail(cudaError_t e, const char* what) {
  g_err = std::string(what) + ": " + cudaGetErrorString(e);
  return (int)e;
}

#define CUDA_TRY(expr)                                   \
  do {                                                   \
    cudaError_t _e = (expr);                             \
    if (_e != cudaSuccess) return cuda_fail(_e, #expr);  \
  } while (0)

int current_state(DeviceState** out) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return cuda_fail(e, "cudaGetDevice");
  if (dev < 0 || dev >= kMaxDevices) return fail(PNP_ENODEVICE, "device index %d out of range", dev);
  DeviceState* s = &g_dev[dev];
  if (s->sm_count == 0) {
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, dev));
    if (prop.major != 10)
      return fail(PNP_ENODEVICE, "libpnp_b200 is built for sm_100a only; device %d is sm_%d%d", dev, prop.major,
                  prop.minor);
    s->sm_count = prop.multiProcessorCount;
  }
  *out = s;
  return PNP_OK;
}

bool tree_matches_spec(const PnpTree& t) {
  return t.njoint == PNP_NJOINT && !memcmp(t.link_pos, pnp_spec::kLinkPos, sizeof t.link_pos) &&
         !memcmp(t.link_rot, pnp_spec::kLinkRot, sizeof t.link_rot) &&
         !memcmp(t.ee_pos, pnp_spec::kEePos, sizeof t.ee_pos) &&
         !memcmp(t.ee_rot, pnp_spec::kEeRot, sizeof t.ee_rot) &&
         !memcmp(t.lower, pnp_spec::kLower, sizeof t.lower) && !memcmp(t.upper, pnp_spec::kUpper, sizeof t.upper) &&
         !memcmp(t.qref, pnp_spec::kQref, sizeof t.qref);
}

template <typename T>
void fill_tree_dev(const PnpTree& t, pnp::TreeDev<T>* d) {
  for (int i = 0; i < 21; ++i) d->link_pos[i] = (T)t.link_pos[i];
  for (int i = 0; i < 63; ++i) d->link_rot[i] = (T)t.link_rot[i];
  for (int i = 0; i < 3; ++i) d->ee_pos[i] = (T)t.ee_pos[i];
  for (int i = 0; i < 9; ++i) d->ee_rot[i] = (T)t.ee_rot[i];
  for (int i = 0; i < 7; ++i) {
    d->lower[i] = (T)t.lower[i];
    d->upper[i] = (T)t.upper[i];
    d->qref[i] = (T)t.qref[i];
  }
}

// kinematics selector -> use the specialised instantiation?
int pick_kin(const DeviceState* s, int kinematics, bool* use_spec) {
  if (!s->have_tree) return fail(PNP_ENOTREE, "pnp_set_tree has not been called on this device");
  switch (kinematics) {
    case PNP_KIN_AUTO: *use_spec = s->specialized; return PNP_OK;
    case PNP_KIN_GENERIC: *use_spec = false; return PNP_OK;
    case PNP_KIN_SPECIALIZED:
    case PNP_KIN_SPEC_LANE:
    case PNP_KIN_SPEC_PAIR:
      if (!s->specialized) return fail(PNP_EINVAL, "uploaded tree differs from the build-time specialised tree");
      *use_spec = true;
      return PNP_OK;
    default: return fail(PNP_EINVAL, "bad kinematics selector %d", kinematics);
  }
}

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

int grid_for(long long work_items, int block, int sm_count, int blocks_per_sm) {
  long long g = (work_items + block - 1) / block;
  const long long cap = (long long)sm_count * blocks_per_sm;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}

// Raise a kernel's dynamic shared-memory cap above the default 48 KB, once per kernel and device.  Before the kernel's
// occupancy query too: the query only sees the raised cap.
template <auto kKernel>
int max_dynamic_smem(DeviceState* s, size_t bytes) {
  static bool set_on_device[kMaxDevices] = {};
  bool& set = set_on_device[s - g_dev];
  if (!set) {
    CUDA_TRY(cudaFuncSetAttribute(kKernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    set = true;
  }
  return PNP_OK;
}

// Resident blocks per SM of a kernel, queried once per kernel and device (every kernel is launched with one block size
// and one dynamic shared-memory size).  A kernel of which no block fits an SM cannot be launched: an error.
template <auto kKernel>
int occupancy(DeviceState* s, int block, size_t smem, int* out) {
  static int occ_of_device[kMaxDevices] = {};
  int& occ = occ_of_device[s - g_dev];
  if (occ == 0) {
    int o = 0;
    CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o, kKernel, block, smem));
    if (o < 1) return cuda_fail(cudaErrorLaunchOutOfResources, "cudaOccupancyMaxActiveBlocksPerMultiprocessor: 0 blocks per SM");
    occ = o;
  }
  *out = occ;
  return PNP_OK;
}

// Launch geometry of a persistent-warp kernel of the IK family (lanes keep drawing queries from a ticket, S queries per
// lane).  Small batches: one working warp per block - the block's other warps only load the trig table - so that the few
// warps spread over as many SMs as possible.  Otherwise the lanes the batch needs, capped at occ blocks per SM.  A warp
// reserves `chunk` queries per ticket atomic: about 1/div of its share, within [32 S, cap], a multiple of 32.  (For a
// small batch, n <= 32 S grid and n / (warps div) < S: the chunk is the floor 32 S, whichever warp count divides.)
struct PersistentGrid {
  int grid;
  unsigned chunk;
};
PersistentGrid persistent_grid(const DeviceState* s, long long n, int S, int block, int occ, bool small, int div, int cap) {
  const long long lanes = (n + S - 1) / S;
  PersistentGrid g;
  g.grid = small ? (int)((lanes + 31) / 32) : grid_for(lanes, block, s->sm_count, occ);
  long long chunk = n / ((long long)g.grid * (block / 32) * div);
  chunk = chunk < 32 * S ? 32 * S : (chunk > cap ? cap : chunk);
  g.chunk = (unsigned)(chunk & ~31ll);
  return g;
}

// The refill ticket of the stream's scratch slot, zeroed on the stream.
int stream_ticket(DeviceState* s, cudaStream_t st, unsigned** out) {
  unsigned* ticket = s->tickets + stream_slot(s, st);
  CUDA_TRY(cudaMemsetAsync(ticket, 0, sizeof(unsigned), st));
  *out = ticket;
  return PNP_OK;
}

template <typename T>
pnp::IkConst<T> make_ik_const(const PnpIkParams* p) {
  pnp::IkConst<T> k;
  k.pos_thresh = (T)p->pos_thresh;
  k.damping = (T)p->damping;
  k.step_limit = (T)p->step_limit;
  k.max_iters = p->max_iters;
  return k;
}

int check_ik_params(const PnpIkParams* p) {
  if (!p) return fail(PNP_EINVAL, "params is NULL");
  if (p->max_iters < 0) return fail(PNP_EINVAL, "max_iters must be >= 0");
  if (!(p->damping > 0.0)) return fail(PNP_EINVAL, "damping must be > 0 (J J^T + damping I must be SPD)");
  if (!(p->step_limit >= 0.0)) return fail(PNP_EINVAL, "step_limit must be >= 0");
  return PNP_OK;
}

template <typename T>
int fk_jac_impl(const T* q, int64_t n, T* pos, T* quat, T* jac, int32_t kinematics, void* stream) {
  if (n < 0 || (n > 0 && (!q || !pos))) return fail(PNP_EINVAL, "fk_jac: null pointer or negative n");
  DeviceState* s;
  int rc = current_state(&s);
  if (rc) return rc;
  bool spec;
  if ((rc = pick_kin(s, kinematics, &spec))) return rc;
  if (n == 0) return PNP_OK;
  cudaStream_t st = (cudaStream_t)stream;
  // FP32, 16-byte aligned outputs: full 128-configuration tiles go through the kernel with staged, bulk-stored
  // outputs; the ragged tail (and everything else) through the per-lane kernel
  int64_t done = 0;
  if constexpr (std::is_same<T, float>::value) {
    // (position / quaternion only: 12-28 B out per configuration, the per-lane kernel at full occupancy is faster)
    const bool aligned = aligned16(pos) && (!quat || aligned16(quat)) && aligned16(jac);
    if (jac && aligned && n >= pnp::FK_TILE) {
      rc = spec ? max_dynamic_smem<pnp::fk_jac_bulk_kernel<pnp::SpecKin>>(s, pnp::FK_BULK_SMEM)
                : max_dynamic_smem<pnp::fk_jac_bulk_kernel<pnp::GenericKin>>(s, pnp::FK_BULK_SMEM);
      if (rc) return rc;
      const int64_t tiles = n / pnp::FK_TILE;
      const int grid = (int)std::min<int64_t>(tiles, (int64_t)s->sm_count * 4);  // 4 x 49 KB of shared memory per SM
      if (spec)
        pnp::fk_jac_bulk_kernel<pnp::SpecKin><<<grid, pnp::FK_TILE, pnp::FK_BULK_SMEM, st>>>(q, tiles, pos, quat, jac);
      else
        pnp::fk_jac_bulk_kernel<pnp::GenericKin><<<grid, pnp::FK_TILE, pnp::FK_BULK_SMEM, st>>>(q, tiles, pos, quat, jac);
      ++g_launches;
      CUDA_TRY(cudaGetLastError());
      done = tiles * pnp::FK_TILE;
    }
  }
  if (done < n) {
    const int64_t m = n - done;
    const int grid = grid_for(m, 128, s->sm_count, 16);
    T* quat_t = quat ? quat + done * 4 : nullptr;
    T* jac_t = jac ? jac + done * 42 : nullptr;
    if (spec)
      pnp::fk_jac_kernel<T, pnp::SpecKin><<<grid, 128, 0, st>>>(q + done * 7, m, pos + done * 3, quat_t, jac_t);
    else
      pnp::fk_jac_kernel<T, pnp::GenericKin><<<grid, 128, 0, st>>>(q + done * 7, m, pos + done * 3, quat_t, jac_t);
    ++g_launches;
    CUDA_TRY(cudaGetLastError());
  }
  return PNP_OK;
}

template <typename T>
int get_obs_impl(const T* q_arm, const T* qvel_arm, const T* fingers, const T* obj_pos, const T* obj_quat,
                 const T* obj_vel, const T* goal, int32_t goal_stride, int64_t n, double dt, T* out,
                 int32_t kinematics, void* stream) {
  if (n < 0 || (n > 0 && (!q_arm || !qvel_arm || !fingers || !obj_pos || !obj_quat || !obj_vel || !goal || !out)))
    return fail(PNP_EINVAL, "get_obs: null pointer or negative n");
  if (goal_stride != 0 && goal_stride != 3) return fail(PNP_EINVAL, "goal_stride must be 0 or 3");
  DeviceState* s;
  int rc = current_state(&s);
  if (rc) return rc;
  bool spec;
  if ((rc = pick_kin(s, kinematics, &spec))) return rc;
  if (n == 0) return PNP_OK;
  pnp::ObsArgs<T> a;
  a.q_arm = q_arm; a.qvel_arm = qvel_arm; a.fingers = fingers; a.obj_pos = obj_pos; a.obj_quat = obj_quat;
  a.obj_vel = obj_vel; a.goal = goal; a.goal_stride = goal_stride; a.n = n; a.dt = (T)dt; a.out = out;
  cudaStream_t st = (cudaStream_t)stream;
  // FP32, 16-byte aligned arrays: full 128-env tiles go through the bulk-async-copy kernel, the ragged
  // tail (and everything else) through the per-lane kernel
  int64_t done = 0;
  if constexpr (std::is_same<T, float>::value) {
    const bool aligned = aligned16(q_arm) && aligned16(qvel_arm) && aligned16(fingers) && aligned16(obj_pos) &&
                         aligned16(obj_quat) && aligned16(obj_vel) && aligned16(out) && (goal_stride == 0 || aligned16(goal));
    static const bool bulk_enabled = [] { const char* e = getenv("PNP_OBS_BULK"); return !e || atoi(e) != 0; }();
    if (aligned && bulk_enabled && n >= pnp::OBS_TILE) {
      rc = spec ? max_dynamic_smem<pnp::get_obs_bulk_kernel<pnp::SpecKin>>(s, pnp::OBS_BULK_SMEM)
                : max_dynamic_smem<pnp::get_obs_bulk_kernel<pnp::GenericKin>>(s, pnp::OBS_BULK_SMEM);
      if (rc) return rc;
      const int64_t tiles = n / pnp::OBS_TILE;
      const int grid = (int)std::min<int64_t>(tiles, (int64_t)s->sm_count * 3);  // 3 x 72 KB of shared memory per SM
      if (spec)
        pnp::get_obs_bulk_kernel<pnp::SpecKin><<<grid, pnp::OBS_TILE, pnp::OBS_BULK_SMEM, st>>>(a);
      else
        pnp::get_obs_bulk_kernel<pnp::GenericKin><<<grid, pnp::OBS_TILE, pnp::OBS_BULK_SMEM, st>>>(a);
      ++g_launches;
      CUDA_TRY(cudaGetLastError());
      done = tiles * pnp::OBS_TILE;
    }
  }
  if (done < n) {
    a.q_arm += done * 7; a.qvel_arm += done * 7; a.fingers += done * 2; a.obj_pos += done * 3; a.obj_quat += done * 4;
    a.obj_vel += done * 6; a.goal += done * goal_stride; a.out += done * 25; a.n = n - done;
    const int grid = grid_for(a.n, pnp::OBS_TILE, s->sm_count, 8);
    if (spec)
      pnp::get_obs_kernel<T, pnp::SpecKin><<<grid, pnp::OBS_TILE, 0, st>>>(a);
    else
      pnp::get_obs_kernel<T, pnp::GenericKin><<<grid, pnp::OBS_TILE, 0, st>>>(a);
    ++g_launches;
    CUDA_TRY(cudaGetLastError());
  }
  return PNP_OK;
}

int env_int(const char* name, int dflt) {
  const char* e = getenv(name);
  return e ? atoi(e) : dflt;
}

template <typename T, typename Kin, int kOut>
int launch_ik(DeviceState* s, const pnp::IkArgs<T>& a, bool small, cudaStream_t st) {
  int occ;
  const int rc = occupancy<pnp::ik_solve_kernel<T, Kin, kOut>>(s, pnp::IK_BLOCK, 0, &occ);
  if (rc) return rc;
  // queries reserved per ticket atomic: ~1/16 of a warp's share, within [32, 256]
  const PersistentGrid g = persistent_grid(s, a.n, 1, pnp::IK_BLOCK, occ, small, 16, 256);
  pnp::IkArgs<T> args = a;
  args.chunk = g.chunk;
  args.solo_warp = small ? 1u : 0u;
  pnp::ik_solve_kernel<T, Kin, kOut><<<g.grid, pnp::IK_BLOCK, 0, st>>>(args);
  ++g_launches;
  CUDA_TRY(cudaGetLastError());
  return PNP_OK;
}

// Value-type kernels (pnp_vec.cuh): V = float, one query per lane; V = F2, two queries per lane.
template <typename V, int kOut>
int launch_ik_v(DeviceState* s, const pnp::IkArgs<float>& a, bool small, cudaStream_t st) {
  constexpr int S = pnp::Slots<V>::kN;
  // (small batches: a lone warp would need ~5 us to load the 40 KB trig table, hence the helper warps)
  const int block = pnp::IK_BLOCK;
  // the grid of all four variants below follows the instantiation with counters, and the compact layout's follows the
  // packed one's: those use fewer registers, and 5 blocks per SM measured slower than 4 (DESIGN.md 4.1)
  constexpr int kOccOut = kOut == pnp::IK_OUT_SEPARATE ? pnp::IK_OUT_SEPARATE : pnp::IK_OUT_PACKED;
  int occ;
  const int rc = occupancy<pnp::ik_solve_v_kernel<V, kOccOut, true>>(s, block, 0, &occ);
  if (rc) return rc;
  static const int env_occ = env_int("PNP_IK_OCC", 0);
  const int occ_use = env_occ > 0 && env_occ < occ ? env_occ : occ;
  const PersistentGrid g = persistent_grid(s, a.n, S, block, occ_use, small, 16, 256);
  const int grid = g.grid;
  const long long warps = (long long)grid * (block / 32);
  pnp::IkArgs<float> args = a;
  args.solo_warp = small ? 1u : 0u;
  args.chunk = g.chunk;
  {
    // lanes with a finished slot that trigger a store + refill (PNP_IK_FLUSH_MIN overrides, for tuning)
    static const int env_flush = env_int("PNP_IK_FLUSH_MIN", 0);
    const bool oversubscribed = (long long)a.n >= (long long)s->sm_count * 8192;
    args.flush_min = env_flush > 0 ? (unsigned)env_flush : (S == 2 ? (small ? 1u : 10u) : (oversubscribed ? 4u : 1u));
    // tail phase of the pair kernel (PNP_IK_TAIL=0 switches it off, for measurements)
    static const int env_tail = env_int("PNP_IK_TAIL", 1);
    args.tail = (S == 2 && !small && env_tail != 0) ? 1u : 0u;
    // guided ticket chunks: a reservation = (queries left) / (2 x warps) (PNP_IK_GUIDED=0: fixed chunks)
    static const int env_guided = env_int("PNP_IK_GUIDED", 1);
    args.guided = (!small && env_guided != 0) ? (unsigned)(warps * 2) : 0u;
  }
  // (no counters asked for: the instantiation without the counter updates in its store block)
  const bool bc = a.q_init_stride == 0, cnt = a.counters != nullptr;
  auto kernel = bc ? (cnt ? pnp::ik_solve_v_kernel<V, kOut, true, false, true> : pnp::ik_solve_v_kernel<V, kOut, true, false, false>)
                   : (cnt ? pnp::ik_solve_v_kernel<V, kOut, false, false, true> : pnp::ik_solve_v_kernel<V, kOut, false, false, false>);
  static const int env_pdl = env_int("PNP_IK_PDL", 1);  // 0: every launch zeroes its ticket with a memset node (measurements)
  static const int env_handover = env_int("PNP_IK_HANDOVER", 1);  // 0: stragglers finish inside their blocks (measurements)
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  CUDA_TRY(cudaStreamIsCapturing(st, &cap));
  std::lock_guard<std::mutex> lk(g_mu);  // the slot's state changes in the order of the launches on its stream
  const int sl = stream_slot_locked(s, st);
  IkPdlState& ps = s->ik_pdl[sl];
  unsigned* sc = s->ik_sc + (size_t)sl * 2 * kIkScratchWords;
  args.park_dump = nullptr; args.park_list = nullptr; args.park_lanes = nullptr; args.park_slots = nullptr;
  args.zero_next[0] = args.zero_next[1] = args.zero_next[2] = nullptr;
  auto forget = [&]() { ps.primed = false; ps.parity = 0; ps.last_handover = false; };
  if (small || !env_pdl || cap != cudaStreamCaptureStatusNone) {
    // small batches (a launch is one dependent chain: nothing to overlap), captured launches (a replayed node cannot
    // alternate tickets): the launch zeroes its own ticket, plain stream order
    args.ticket = sc;
    args.ticket_next = nullptr;
    args.pdl = pnp::IK_PDL_OFF;
    forget();
    CUDA_TRY(cudaMemsetAsync(args.ticket, 0, sizeof(unsigned), st));
    kernel<<<grid, block, 0, st>>>(args);
    ++g_launches;
    CUDA_TRY(cudaGetLastError());
    return PNP_OK;
  }
  // what this launch reads and writes
  ByteRange in[2], out[5];
  const size_t n = a.n;
  in[0] = byte_range(a.targets, n * 12);
  in[1] = byte_range(a.q_init, a.q_init_stride ? n * 28 : 28);
  if (kOut == pnp::IK_OUT_SEPARATE) {
    out[0] = byte_range(a.q_out, n * 28); out[1] = byte_range(a.final_pos, n * 12); out[2] = byte_range(a.pos_err, n * 4);
    out[3] = byte_range(a.iters, n * 4); out[4] = byte_range(a.flags, n);
  } else {
    out[0] = byte_range(a.q_out, n * 32);
    if (kOut == pnp::IK_OUT_PACKED) out[1] = byte_range(a.final_pos, n * 16);
  }
  bool clash = false;  // with the previous launch of this stream, which may still be draining when this one starts
  if (ps.primed) {
    for (const ByteRange& o : out)
      for (int k = 0; k < 7; ++k) clash = clash || ranges_overlap(o, k < 2 ? ps.in[k] : ps.out[k - 2]);
    for (const ByteRange& i : in)
      for (const ByteRange& po : ps.out) clash = clash || ranges_overlap(i, po);
  }
  // drain hand-over: the pair kernel parks what is still running when its pool runs dry, a resume launch finishes it
  // (from 16384 queries per SM up: a smaller launch timed alone loses more to the resume launch's fixed cost than its blocks
  //  gain by leaving early - 2^20 queries alone 0.241 -> 0.264 ms with it, 2^22 0.679 -> 0.668 ms)
  bool handover = S == 2 && env_handover && args.tail && (long long)a.n >= (long long)s->sm_count * 16384;
  if (handover) {
    const size_t rows = (size_t)grid * (block / 32) * (IK_HANDOVER_AT);  // a warp parks at most IK_HANDOVER_AT slots (<= that many lanes)
    if (ps.rows_cap < rows) {  // first big launch of this stream (cudaMalloc synchronises the device once)
      const size_t most = (size_t)s->sm_count * 8 * (block / 32) * (IK_HANDOVER_AT);
      const size_t cap_rows = most > rows ? most : rows;
      for (int k = 0; k < 2; ++k) {
        if (ps.dump[k]) cudaFree(ps.dump[k]);
        if (ps.list[k]) cudaFree(ps.list[k]);
        ps.dump[k] = nullptr; ps.list[k] = nullptr;
      }
      ps.rows_cap = 0;
      bool ok = true;
      for (int k = 0; k < 2 && ok; ++k)
        ok = cudaMalloc(&ps.dump[k], cap_rows * 8 * sizeof(float2)) == cudaSuccess &&
             cudaMalloc(&ps.list[k], cap_rows * sizeof(uint4)) == cudaSuccess;
      if (ok) ps.rows_cap = cap_rows;
      else { (void)cudaGetLastError(); handover = false; }  // no memory for it: stragglers finish in their blocks
      forget();  // (the synchronising allocation ended whatever was in flight)
    }
  }
  const unsigned p = ps.parity;
  unsigned* scp = sc + p * kIkScratchWords;
  unsigned* scn = sc + (p ^ 1u) * kIkScratchWords;
  args.ticket = scp + 0;
  args.ticket_next = scn + 0;
  args.pdl = clash ? pnp::IK_PDL_WAIT_FIRST : pnp::IK_PDL_WAIT_AT_DRY;
  if (handover) {
    args.park_dump = ps.dump[p]; args.park_list = ps.list[p];
    args.park_lanes = scp + 1; args.park_slots = scp + 2;
  }
  // (a hand-over launch after one without: no resume launch has zeroed this parity's parking counters)
  if (!ps.primed || (handover && !ps.last_handover)) CUDA_TRY(cudaMemsetAsync(sc, 0, 2 * kIkScratchWords * sizeof(unsigned), st));
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3((unsigned)block);
  cfg.dynamicSmemBytes = 0;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, args);
  ++g_launches;
  if (e != cudaSuccess) {
    forget();
    return cuda_fail(e, "cudaLaunchKernelEx(ik_solve_v_kernel)");
  }
  if (handover) {
    // the resume launch: one block per SM (it shares the SMs with the next pair launch), one query per lane
    pnp::IkArgs<float> r = args;
    r.ticket = scp + 3;
    r.ticket_next = nullptr;
    r.pdl = pnp::IK_PDL_OFF;
    r.zero_next[0] = scn + 1; r.zero_next[1] = scn + 2; r.zero_next[2] = scn + 3;
    r.chunk = 32; r.flush_min = 1; r.solo_warp = 0; r.tail = 0; r.guided = 0;
    auto resume = bc ? (cnt ? pnp::ik_solve_v_kernel<float, kOut, true, true, true> : pnp::ik_solve_v_kernel<float, kOut, true, true, false>)
                     : (cnt ? pnp::ik_solve_v_kernel<float, kOut, false, true, true> : pnp::ik_solve_v_kernel<float, kOut, false, true, false>);
    cfg.gridDim = dim3((unsigned)s->sm_count);
    e = cudaLaunchKernelEx(&cfg, resume, r);
    ++g_launches;
    if (e != cudaSuccess) {
      forget();
      return cuda_fail(e, "cudaLaunchKernelEx(ik_solve_v_kernel, resume)");
    }
  } else {
    // no resume launch will zero the other parity's hand-over counters: nothing uses them in this mode
  }
  ps.primed = true;
  ps.last_handover = handover;
  ps.parity ^= 1u;
  for (int k = 0; k < 2; ++k) ps.in[k] = in[k];
  for (int k = 0; k < 5; ++k) ps.out[k] = out[k];
  return PNP_OK;
}

// Small cold batches (at most one working warp per scheduler): the single-basic-block latency kernel, no ticket.
template <int kOut>
int launch_ik_small(const pnp::IkArgs<float>& a, cudaStream_t st) {
  const int grid = (int)((a.n + 31u) / 32u);
  if (a.q_init_stride == 0)
    pnp::ik_solve_small_kernel<kOut, true><<<grid, pnp::IK_BLOCK, 0, st>>>(a);
  else
    pnp::ik_solve_small_kernel<kOut, false><<<grid, pnp::IK_BLOCK, 0, st>>>(a);
  ++g_launches;
  CUDA_TRY(cudaGetLastError());
  return PNP_OK;
}

// FP32 on the specialised tree always runs the value-type arithmetic (ik_eval_v / ik_step_v: a batch gives
// bit-identical results whichever kernel is picked).  AUTO / SPECIALIZED:
//   n <= 128 queries per SM          ik_solve_small_kernel (latency bound: the launch lasts as long as its slowest query)
//   n > 256 queries per SM           two queries per lane (packed FFMA2/FMUL2/FADD2): measured faster than one per lane from
//                                    2^16 queries up (0.071 vs 0.093 ms; 2^19: 0.167 vs 0.192 ms), slower at 2^15 (0.077 vs 0.071 ms)
//   in between                       one query per lane with refill
template <int kOut>
int launch_ik_spec_f32(DeviceState* s, const pnp::IkArgs<float>& a, int kinematics, bool small, cudaStream_t st) {
  const bool big = (long long)a.n > (long long)s->sm_count * pnp::IK_BLOCK * 2;
  if (kinematics == PNP_KIN_SPEC_PAIR || (kinematics != PNP_KIN_SPEC_LANE && big))
    return launch_ik_v<pnp::F2, kOut>(s, a, (long long)a.n <= (long long)s->sm_count * pnp::IK_BLOCK * 2, st);
  return launch_ik_v<float, kOut>(s, a, small, st);
}

template <typename T, int kOut>
int ik_solve_impl(const T* targets, const T* q_init, int32_t q_init_stride, int64_t n, const PnpIkParams* params,
                  T* q_out, T* final_pos, T* pos_err, int32_t* iters, uint8_t* flags, unsigned long long* counters,
                  void* stream, pnp::IkArgs<T>* args_out = nullptr) {
  int rc = check_ik_params(params);
  if (rc) return rc;
  if (n < 0 || (n > 0 && (!targets || !q_init || !q_out))) return fail(PNP_EINVAL, "ik_solve: null pointer or negative n");
  if (n >= (int64_t(1) << 31)) return fail(PNP_EINVAL, "ik_solve: n must be < 2^31 per call (split the batch)");
  if (q_init_stride != 0 && q_init_stride != PNP_NJOINT) return fail(PNP_EINVAL, "q_init_stride must be 0 or 7");
  if (kOut == pnp::IK_OUT_PACKED && n > 0 && (!final_pos || !aligned16(q_out) || !aligned16(final_pos)))
    return fail(PNP_EINVAL, "ik_solve_packed: out_q8 / out_aux must be non-null and 16-byte aligned");
  if (kOut == pnp::IK_OUT_COMPACT && n > 0 && !aligned16(q_out))
    return fail(PNP_EINVAL, "ik_solve_compact: out_q8 must be 16-byte aligned");
  DeviceState* s;
  if ((rc = current_state(&s))) return rc;
  bool spec;
  if ((rc = pick_kin(s, params->kinematics, &spec))) return rc;
  if (n == 0) return PNP_OK;
  cudaStream_t st = (cudaStream_t)stream;

  pnp::IkArgs<T> a;
  a.targets = targets; a.q_init = q_init; a.q_init_stride = q_init_stride; a.n = (unsigned)n;
  a.k = make_ik_const<T>(params);
  a.q_out = q_out; a.final_pos = final_pos; a.pos_err = pos_err; a.iters = iters; a.flags = flags;
  a.counters = counters; a.ticket = nullptr; a.chunk = 32; a.flush_min = 1; a.solo_warp = 0; a.tail = 0; a.guided = 0;
  a.ticket_next = nullptr; a.pdl = 0;
  a.park_dump = nullptr; a.park_list = nullptr; a.park_lanes = nullptr; a.park_slots = nullptr;
  a.zero_next[0] = a.zero_next[1] = a.zero_next[2] = nullptr;
  a.thresh2 = a.k.pos_thresh * a.k.pos_thresh;
  if (args_out) *args_out = a;  // the multistart's restarts use this block
  const bool small = n <= (long long)s->sm_count * pnp::IK_BLOCK;
  if constexpr (std::is_same<T, float>::value) {
    // the latency kernel needs no ticket: skip the memset node as well
    static const int env_small = env_int("PNP_IK_SMALL", 1);
    if (spec && small && env_small && (params->kinematics == PNP_KIN_AUTO || params->kinematics == PNP_KIN_SPECIALIZED))
      return launch_ik_small<kOut>(a, st);
  }
  if (spec) {
    if constexpr (std::is_same<T, float>::value) return launch_ik_spec_f32<kOut>(s, a, params->kinematics, small, st);  // own tickets
  }
  if ((rc = stream_ticket(s, st, &a.ticket))) return rc;
  if (spec) {
    if constexpr (!std::is_same<T, float>::value) {
      return launch_ik<T, pnp::SpecKin, kOut>(s, a, small, st);
    }
  }
  return launch_ik<T, pnp::GenericKin, kOut>(s, a, small, st);
}

// ---- multistart (see ms_collect_kernel / ms_wave* in pnp_kernels.cuh) ----------------------------------------------
// Lanes per restarted query: the seeds a wave runs in parallel.
// Position solver: a wave lasts as long as its slowest attempt (up to max_iters passes) whatever its width, so fewer,
// wider waves cost less until the lanes no longer fit the SMs at once; see DESIGN.md 4.1 for the measurement.
// PNP_MS_GROUP overrides it (1, 2, 4 or 8), for measurements.
constexpr int kMsGroup = 4;
// Pose solver: about a quarter of a cold workspace batch enters the first wave, and a failing attempt runs all
// max_iters passes, so a wave costs about its lane count times max_iters: the narrowest group, which spends no attempt
// on a query an earlier seed already rescues, measured fastest (DESIGN.md 4.6: 2^22 W-cold poses with 8 seeds in
// 14.7 ms at G = 1, 16.0 / 20.3 / 30.8 ms at G = 2 / 4 / 8).  PNP_MS_POSE_GROUP overrides it (1, 2, 4 or 8), for
// measurements.
constexpr int kMsPoseGroup = 1;
constexpr size_t kMsHdrBytes = pnp::MS_HDR_WORDS * sizeof(unsigned);
size_t ms_list_bytes(int64_t n) { return ((size_t)n * sizeof(unsigned) + 15u) & ~(size_t)15u; }
// header | list A | list B | iterations of attempt 0 (separate layout without an iters output)
size_t ms_scratch_bytes(int64_t n) { return kMsHdrBytes + 3 * ms_list_bytes(n); }

// one restart wave
template <auto kKernel, typename M>
int launch_ms_wave(DeviceState* s, const M& m, cudaStream_t st) {
  int occ;
  const int rc = occupancy<kKernel>(s, pnp::MS_BLOCK, 0, &occ);
  if (rc) return rc;
  kKernel<<<s->sm_count * occ, pnp::MS_BLOCK, 0, st>>>(m);
  ++g_launches;
  CUDA_TRY(cudaGetLastError());
  return PNP_OK;
}

// The multistart of either solver; A is its argument block (IkArgs<T>, PoseIkArgs<T>), `who` names it in messages.
// kCollect is where attempt 0's success and iterations are read: IK_OUT_SEPARATE (flags[] required, iterations from
// iters or scratch) or IK_OUT_PACKED (the packed word of a.final_pos).  `outputs` are the byte ranges of the solver's
// outputs.  attempt0(iters0, a) runs the plain solve with iters0 as its iterations output and leaves its argument
// block in `a`; wave(s, spec, m, st) launches the restart kernel of one wave.  Every argument is checked before the
// first launch.
template <typename A, int kCollect, typename T, typename Attempt0, typename Wave>
int multistart_impl(const char* who, int64_t n, const T* seeds, int32_t n_seeds, const PnpIkParams* params,
                    const uint8_t* flags, int32_t* iters, uint8_t* attempt, unsigned long long* counters,
                    unsigned long long* restart_stats, void* scratch, std::initializer_list<ByteRange> outputs,
                    int group_default, const char* group_env, void* stream, Attempt0 attempt0, Wave wave) {
  if (n_seeds < 0 || n_seeds > pnp::MS_MAX_SEEDS) return fail(PNP_EINVAL, "%s: n_seeds must be in [0, 255]", who);
  if (n_seeds > 0 && !seeds) return fail(PNP_EINVAL, "%s: seeds is NULL", who);
  if (!scratch || !aligned16(scratch)) return fail(PNP_EINVAL, "%s: scratch must be non-null and 16-byte aligned", who);
  if (kCollect == pnp::IK_OUT_SEPARATE && n > 0 && !flags)
    return fail(PNP_EINVAL, "%s: flags must be non-null (the restarts read attempt 0's success from it)", who);
  if (n > 0) {
    // seeds (read by every wave) and scratch (written) must not share memory with an output or with each other
    const ByteRange in[2] = {byte_range(seeds, (size_t)n_seeds * PNP_NJOINT * sizeof(T)), byte_range(scratch, ms_scratch_bytes(n))};
    const ByteRange more[3] = {byte_range(attempt, (size_t)n), byte_range(counters, 4 * sizeof(unsigned long long)),
                               byte_range(restart_stats, 3 * sizeof(unsigned long long))};
    bool clash = false;
    for (const ByteRange& o : outputs) clash = clash || ranges_overlap(o, in[0]) || ranges_overlap(o, in[1]);
    for (const ByteRange& o : more) clash = clash || ranges_overlap(o, in[0]) || ranges_overlap(o, in[1]);
    if (clash) return fail(PNP_EINVAL, "%s: seeds and scratch must not overlap an output", who);
    if (ranges_overlap(in[0], in[1])) return fail(PNP_EINVAL, "%s: seeds and scratch must not overlap", who);
  }
  unsigned* hdr = static_cast<unsigned*>(scratch);
  unsigned* list[2] = {reinterpret_cast<unsigned*>((char*)scratch + kMsHdrBytes),
                       reinterpret_cast<unsigned*>((char*)scratch + kMsHdrBytes + ms_list_bytes(n))};
  int32_t* iters0 = iters;
  if (kCollect == pnp::IK_OUT_SEPARATE && !iters0 && n_seeds > 0)  // the restarts need attempt 0's iterations for the counters
    iters0 = reinterpret_cast<int32_t*>((char*)scratch + kMsHdrBytes + 2 * ms_list_bytes(n));
  // attempt 0: the plain entry point, unchanged
  pnp::MsArgs<A> m;
  int rc = attempt0(iters0, m.a);
  if (rc || n == 0) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  if (attempt) CUDA_TRY(cudaMemsetAsync(attempt, 0, (size_t)n, st));
  if (n_seeds == 0) return PNP_OK;
  DeviceState* s;
  if ((rc = current_state(&s))) return rc;
  bool spec;
  if ((rc = pick_kin(s, params->kinematics, &spec))) return rc;

  CUDA_TRY(cudaMemsetAsync(hdr, 0, kMsHdrBytes, st));
  {
    const int grid = grid_for(n, pnp::MS_COLLECT_BLOCK, s->sm_count, 8);
    const unsigned* aux_words = kCollect == pnp::IK_OUT_SEPARATE ? nullptr : reinterpret_cast<const unsigned*>(m.a.final_pos);
    pnp::ms_collect_kernel<kCollect><<<grid, pnp::MS_COLLECT_BLOCK, 0, st>>>(m.a.flags, aux_words, (unsigned)n, list[0],
                                                                              hdr, restart_stats);
    ++g_launches;
    CUDA_TRY(cudaGetLastError());
  }
  static const int env_group = env_int(group_env, 0);  // (one instantiation per solver and layout: one variable each)
  const int G = (env_group == 1 || env_group == 2 || env_group == 4 || env_group == 8) ? env_group : group_default;
  m.seeds = seeds; m.n_seeds = n_seeds; m.group = (unsigned)G;
  m.iters0 = iters0; m.attempt = attempt; m.restart_stats = restart_stats;
  const int waves = (n_seeds + G - 1) / G;
  for (int w = 0; w < waves; ++w) {
    m.wave = w;
    m.list_in = list[w & 1]; m.cnt_in = hdr + w;
    m.list_out = w + 1 < waves ? list[(w + 1) & 1] : nullptr; m.cnt_out = hdr + w + 1;
    if ((rc = wave(s, spec, m, st))) return rc;
  }
  return PNP_OK;
}

template <typename T, int kOut>
int ik_multistart_impl(const T* targets, const T* q_init, int32_t q_init_stride, int64_t n, const T* seeds, int32_t n_seeds,
                       const PnpIkParams* params, T* q_out, T* final_pos, T* pos_err, int32_t* iters, uint8_t* flags,
                       uint8_t* attempt, unsigned long long* counters, unsigned long long* restart_stats, void* scratch,
                       void* stream) {
  const size_t m = (size_t)n;
  const bool sep = kOut == pnp::IK_OUT_SEPARATE;  // else packed: out_q8 in q_out, out_aux4 in final_pos
  return multistart_impl<pnp::IkArgs<T>, kOut>(
      "ik_multistart", n, seeds, n_seeds, params, flags, iters, attempt, counters, restart_stats, scratch,
      {byte_range(q_out, m * (sep ? PNP_NJOINT * sizeof(T) : 8 * sizeof(float))),
       byte_range(final_pos, m * (sep ? 3 * sizeof(T) : 4 * sizeof(float))), byte_range(pos_err, m * sizeof(T)),
       byte_range(iters, m * sizeof(int32_t)), byte_range(flags, m)},
      kMsGroup, "PNP_MS_GROUP", stream,
      [&](int32_t* iters0, pnp::IkArgs<T>& a) {
        return ik_solve_impl<T, kOut>(targets, q_init, q_init_stride, n, params, q_out, final_pos, pos_err, iters0, flags,
                                      counters, stream, &a);
      },
      [&](DeviceState* s, bool spec, const auto& m, cudaStream_t st) {
        if constexpr (std::is_same<T, float>::value) {
          if (spec && params->kinematics != PNP_KIN_GENERIC) return launch_ms_wave<pnp::ms_wave_v_kernel<kOut>>(s, m, st);
          return launch_ms_wave<pnp::ms_wave_kernel<float, pnp::GenericKin, kOut>>(s, m, st);
        } else {
          return spec ? launch_ms_wave<pnp::ms_wave_kernel<double, pnp::SpecKin, kOut>>(s, m, st)
                      : launch_ms_wave<pnp::ms_wave_kernel<double, pnp::GenericKin, kOut>>(s, m, st);
        }
      });
}

// Smallest double s >= 0 with sqrt(s) >= t (sqrt is correctly rounded, hence monotone): the
// reference's `sqrt(s) < t` is exactly `s < sqrt_preimage(t)`.
double sqrt_preimage(double t) {
  if (!(t > 0.0)) return 0.0;  // sqrt(s) < t is never true for t <= 0 (or NaN)
  if (std::isinf(t)) return t;
  double s = t * t;
  while (s > 0.0 && std::sqrt(s) >= t) s = std::nextafter(s, -INFINITY);
  while (std::sqrt(s) < t) s = std::nextafter(s, INFINITY);
  return s;
}

// [lo, hi) in the squared domain such that  |fl(d - thr)| < tol  <=>  lo <= d*d(rounded sum) < hi
void adjacency_window(double thr, double tol, double* lo, double* hi) {
  if (!(tol > 0.0) || !(thr > 0.0)) { *lo = INFINITY; *hi = -INFINITY; return; }
  double d_lo = thr - tol, d_hi = thr + tol;
  // walk to the exact first / last doubles satisfying the reference-style predicate
  for (int i = 0; i < 64 && std::fabs(std::nextafter(d_lo, -INFINITY) - thr) < tol; ++i) d_lo = std::nextafter(d_lo, -INFINITY);
  for (int i = 0; i < 64 && !(std::fabs(d_lo - thr) < tol); ++i) d_lo = std::nextafter(d_lo, INFINITY);
  for (int i = 0; i < 64 && std::fabs(std::nextafter(d_hi, INFINITY) - thr) < tol; ++i) d_hi = std::nextafter(d_hi, INFINITY);
  for (int i = 0; i < 64 && !(std::fabs(d_hi - thr) < tol); ++i) d_hi = std::nextafter(d_hi, -INFINITY);
  *lo = sqrt_preimage(d_lo);
  *hi = sqrt_preimage(std::nextafter(d_hi, INFINITY));
}

pnp::RewardConst make_reward_const(const PnpRewardParams* p) {
  pnp::RewardConst k;
  k.sparse = p->sparse;
  k.n_tasks = (double)p->n_tasks;
  k.h0 = p->initial_object_height;
  k.high_z = p->high_pick_z;
  k.s_place_lt = sqrt_preimage(p->distance_threshold);
  k.s_reach_lt = sqrt_preimage(0.05);
  adjacency_window(p->distance_threshold, p->threshold_report_tol, &k.s_place_adj_lo, &k.s_place_adj_hi);
  adjacency_window(0.05, p->threshold_report_tol, &k.s_reach_adj_lo, &k.s_reach_adj_hi);
  // (double)w < 0.045  <=>  w < W, W = smallest float whose value is >= 0.045
  float w = (float)0.045;
  if ((double)w < 0.045) w = std::nextafterf(w, INFINITY);
  k.width_lt_f32 = w;
  k.n_bonus = p->n_tasks < 16 ? p->n_tasks : 16;
  for (int i = 0; i < 16; ++i) k.bonus[i] = 0.5 * ((double)i / (double)p->n_tasks);  // panda_env.py:244
  return k;
}

template <typename TIn>
int reward_impl(const TIn* ag, const TIn* dg, const TIn* ee, const TIn* eq, const TIn* width, const int32_t* task,
                int64_t n, const PnpRewardParams* params, float* reward, float* success,
                unsigned long long* counters, void* stream) {
  if (!params) return fail(PNP_EINVAL, "params is NULL");
  if (params->n_tasks <= 0) return fail(PNP_EINVAL, "n_tasks must be > 0");
  if (n < 0 || (n > 0 && (!ag || !dg || !ee || !eq || !width || !task || !reward)))
    return fail(PNP_EINVAL, "reward: null pointer or negative n");
  DeviceState* s;
  int rc = current_state(&s);
  if (rc) return rc;
  if (n == 0) return PNP_OK;
  pnp::RewardArgs<TIn> a;
  a.ag = ag; a.dg = dg; a.ee = ee; a.eq = eq; a.width = width; a.task = task; a.n = n;
  a.k = make_reward_const(params);
  a.reward = reward; a.success = success; a.counters = counters;
  constexpr int R = pnp::RowsPerLane<TIn>::value;
  const bool vec = aligned16(ag) && aligned16(dg) && aligned16(ee) && aligned16(eq) && aligned16(width) &&
                   aligned16(task) && aligned16(reward) && (!success || aligned16(success));
  const long long groups = (n + R - 1) / R;
  const int grid = grid_for(groups, 256, s->sm_count, 8);
  cudaStream_t st = (cudaStream_t)stream;
  if (vec)
    pnp::reward_kernel<TIn, true><<<grid, 256, 0, st>>>(a);
  else
    pnp::reward_kernel<TIn, false><<<grid, 256, 0, st>>>(a);
  ++g_launches;
  CUDA_TRY(cudaGetLastError());
  return PNP_OK;
}

}  // namespace

// ================================================================================================
extern "C" {

int pnp_abi_version(void) { return PNP_ABI_VERSION; }
const char* pnp_last_error(void) { return g_err.c_str(); }
unsigned long long pnp_launch_count(void) { return g_launches.load(); }

int pnp_device_info(int32_t* sm_count, int32_t* clock_khz, int32_t* cc) {
  int dev = 0;
  CUDA_TRY(cudaGetDevice(&dev));
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, dev));
  if (sm_count) *sm_count = prop.multiProcessorCount;
  if (clock_khz) *clock_khz = prop.clockRate;
  if (cc) *cc = prop.major * 10 + prop.minor;
  return PNP_OK;
}

int pnp_set_tree(const PnpTree* t) {
  if (!t) return fail(PNP_EINVAL, "tree is NULL");
  if (t->njoint != PNP_NJOINT) return fail(PNP_EINVAL, "tree.njoint must be %d", PNP_NJOINT);
  DeviceState* s;
  int rc = current_state(&s);
  if (rc) return rc;
  pnp::TreeDev<float> tf;
  pnp::TreeDev<double> td;
  fill_tree_dev(*t, &tf);
  fill_tree_dev(*t, &td);
  // Replacing a tree that kernels on any stream (torch side streams, the host operators' non-blocking streams) may
  // still be reading: cudaMemcpyToSymbol orders against none of them, so wait for the device first.  (The first
  // upload and a re-upload of the same tree have nothing to wait for.)
  if (s->have_tree && memcmp(&s->tree, t, sizeof *t) != 0) CUDA_TRY(cudaDeviceSynchronize());
  CUDA_TRY(cudaMemcpyToSymbol(pnp::c_tree_f32, &tf, sizeof tf));
  CUDA_TRY(cudaMemcpyToSymbol(pnp::c_tree_f64, &td, sizeof td));
  if (!s->tickets) {
    CUDA_TRY(cudaMalloc(&s->tickets, kStreamSlots * sizeof(unsigned)));
    CUDA_TRY(cudaMalloc(&s->ik_sc, 2 * kIkScratchWords * kStreamSlots * sizeof(unsigned)));
    CUDA_TRY(cudaMalloc(&s->order_work, (size_t)kStreamSlots * 2 * pnp::PLAN_BUCKETS * sizeof(unsigned)));
    // sin(k * 2*pi/8192), k < 8192 + 2048, for the FP32 IK kernels' first-order table trig, evaluated in FP64
    static float tabv[pnp::kTrigVWords];
    for (int k = 0; k < pnp::kTrigVWords; ++k)
      tabv[k] = (float)std::sin((double)k * (6.283185307179586476925286766559 / pnp::kTrigVN));
    CUDA_TRY(cudaMemcpyToSymbol(pnp::g_trigv_tab, tabv, sizeof tabv));
  }
  s->tree = *t;
  s->have_tree = true;
  s->specialized = tree_matches_spec(*t);
  return PNP_OK;
}

int pnp_get_tree(PnpTree* out) {
  if (!out) return fail(PNP_EINVAL, "out is NULL");
  DeviceState* s;
  int rc = current_state(&s);
  if (rc) return rc;
  if (!s->have_tree) return fail(PNP_ENOTREE, "pnp_set_tree has not been called on this device");
  *out = s->tree;
  return PNP_OK;
}

int pnp_tree_is_specialized(void) {
  DeviceState* s;
  if (current_state(&s)) return 0;
  return s->have_tree && s->specialized ? 1 : 0;
}

int pnp_get_specialized_tree(PnpTree* out) {
  if (!out) return fail(PNP_EINVAL, "out is NULL");
  memset(out, 0, sizeof *out);
  out->njoint = PNP_NJOINT;
  memcpy(out->link_pos, pnp_spec::kLinkPos, sizeof out->link_pos);
  memcpy(out->link_rot, pnp_spec::kLinkRot, sizeof out->link_rot);
  memcpy(out->ee_pos, pnp_spec::kEePos, sizeof out->ee_pos);
  memcpy(out->ee_rot, pnp_spec::kEeRot, sizeof out->ee_rot);
  memcpy(out->lower, pnp_spec::kLower, sizeof out->lower);
  memcpy(out->upper, pnp_spec::kUpper, sizeof out->upper);
  memcpy(out->qref, pnp_spec::kQref, sizeof out->qref);
  return PNP_OK;
}

int pnp_fk_jac_f32(const float* q, int64_t n, float* pos, float* quat, float* jac, int32_t kin, void* stream) {
  return fk_jac_impl<float>(q, n, pos, quat, jac, kin, stream);
}
int pnp_fk_jac_f64(const double* q, int64_t n, double* pos, double* quat, double* jac, int32_t kin, void* stream) {
  return fk_jac_impl<double>(q, n, pos, quat, jac, kin, stream);
}

int pnp_ik_solve_f32(const float* targets, const float* q_init, int32_t q_init_stride, int64_t n,
                     const PnpIkParams* params, float* q_out, float* final_pos, float* pos_err, int32_t* iters,
                     uint8_t* flags, unsigned long long* counters, void* stream) {
  return ik_solve_impl<float, pnp::IK_OUT_SEPARATE>(targets, q_init, q_init_stride, n, params, q_out, final_pos, pos_err, iters,
                                     flags, counters, stream);
}
int pnp_ik_solve_packed_f32(const float* targets, const float* q_init, int32_t q_init_stride, int64_t n,
                            const PnpIkParams* params, float* out_q8, float* out_aux4,
                            unsigned long long* counters, void* stream) {
  return ik_solve_impl<float, pnp::IK_OUT_PACKED>(targets, q_init, q_init_stride, n, params, out_q8, out_aux4, nullptr, nullptr,
                                    nullptr, counters, stream);
}
int pnp_ik_solve_compact_f32(const float* targets, const float* q_init, int32_t q_init_stride, int64_t n,
                             const PnpIkParams* params, float* out_q8, unsigned long long* counters, void* stream) {
  return ik_solve_impl<float, pnp::IK_OUT_COMPACT>(targets, q_init, q_init_stride, n, params, out_q8, nullptr, nullptr,
                                                   nullptr, nullptr, counters, stream);
}
int pnp_ik_solve_f64(const double* targets, const double* q_init, int32_t q_init_stride, int64_t n,
                     const PnpIkParams* params, double* q_out, double* final_pos, double* pos_err, int32_t* iters,
                     uint8_t* flags, unsigned long long* counters, void* stream) {
  return ik_solve_impl<double, pnp::IK_OUT_SEPARATE>(targets, q_init, q_init_stride, n, params, q_out, final_pos, pos_err, iters,
                                      flags, counters, stream);
}

int pnp_ik_multistart_scratch_bytes(int64_t n, int64_t* bytes) {
  if (n < 0 || !bytes) return fail(PNP_EINVAL, "ik_multistart_scratch_bytes: negative n or NULL bytes");
  *bytes = (int64_t)ms_scratch_bytes(n);
  return PNP_OK;
}
int pnp_ik_solve_multistart_f32(const float* targets, const float* q_init, int32_t q_init_stride, int64_t n, const float* seeds,
                                int32_t n_seeds, const PnpIkParams* params, float* q_out, float* final_pos, float* pos_err,
                                int32_t* iters, uint8_t* flags, uint8_t* attempt, unsigned long long* counters,
                                unsigned long long* restart_stats, void* scratch, void* stream) {
  return ik_multistart_impl<float, pnp::IK_OUT_SEPARATE>(targets, q_init, q_init_stride, n, seeds, n_seeds, params, q_out,
                                                         final_pos, pos_err, iters, flags, attempt, counters, restart_stats,
                                                         scratch, stream);
}
int pnp_ik_solve_multistart_packed_f32(const float* targets, const float* q_init, int32_t q_init_stride, int64_t n,
                                       const float* seeds, int32_t n_seeds, const PnpIkParams* params, float* out_q8,
                                       float* out_aux4, uint8_t* attempt, unsigned long long* counters,
                                       unsigned long long* restart_stats, void* scratch, void* stream) {
  return ik_multistart_impl<float, pnp::IK_OUT_PACKED>(targets, q_init, q_init_stride, n, seeds, n_seeds, params, out_q8,
                                                       out_aux4, nullptr, nullptr, nullptr, attempt, counters, restart_stats,
                                                       scratch, stream);
}
int pnp_ik_solve_multistart_f64(const double* targets, const double* q_init, int32_t q_init_stride, int64_t n,
                                const double* seeds, int32_t n_seeds, const PnpIkParams* params, double* q_out,
                                double* final_pos, double* pos_err, int32_t* iters, uint8_t* flags, uint8_t* attempt,
                                unsigned long long* counters, unsigned long long* restart_stats, void* scratch, void* stream) {
  return ik_multistart_impl<double, pnp::IK_OUT_SEPARATE>(targets, q_init, q_init_stride, n, seeds, n_seeds, params, q_out,
                                                          final_pos, pos_err, iters, flags, attempt, counters, restart_stats,
                                                          scratch, stream);
}

int pnp_ik_waypoints_f32(const float* q_start, const float* goal, int64_t n, int32_t n_steps, double step_size,
                         const PnpIkParams* params, float* q_out, float* pos_out, int32_t* n_accepted,
                         int32_t* iters_total, unsigned long long* counters, void* stream) {
  int rc = check_ik_params(params);
  if (rc) return rc;
  if (n < 0 || n_steps < 0 || (n > 0 && (!q_start || !goal || !q_out || !pos_out)))
    return fail(PNP_EINVAL, "ik_waypoints: null pointer or negative size");
  DeviceState* s;
  if ((rc = current_state(&s))) return rc;
  bool spec;
  if ((rc = pick_kin(s, params->kinematics, &spec))) return rc;
  if (n == 0) return PNP_OK;
  if (n >= (int64_t(1) << 31)) return fail(PNP_EINVAL, "ik_waypoints: n must be < 2^31 per call");
  cudaStream_t st = (cudaStream_t)stream;
  pnp::WaypointArgs<float> a;
  if ((rc = stream_ticket(s, st, &a.ticket))) return rc;
  a.q_start = q_start; a.goal = goal; a.n = (unsigned)n; a.n_steps = n_steps;
  a.step_size = (float)step_size; a.reach_thresh = 0.01f;
  a.k = make_ik_const<float>(params);
  a.q_out = q_out; a.pos_out = pos_out; a.n_accepted = n_accepted; a.iters_total = iters_total;
  a.counters = counters;
  const bool small = n <= (long long)s->sm_count * pnp::IK_BLOCK;
  const int block = pnp::IK_BLOCK;
  // specialised tree: the value-type kernels (same arithmetic in both), one env per lane unless two are asked
  // for (with the fused accept / first-iteration pass the bookkeeping weighs more than the packed arithmetic
  // saves: 2^20 envs x 50, 0.81 ms against 0.87); other trees: the scalar-template kernel
  const bool pair = spec && params->kinematics == PNP_KIN_SPEC_PAIR;
  int occ;  // (the fused instantiation's, for both)
  rc = !spec ? occupancy<pnp::ik_waypoints_kernel<float, pnp::GenericKin>>(s, block, 0, &occ)
       : pair ? occupancy<pnp::ik_waypoints_v_kernel<pnp::F2, true>>(s, block, 0, &occ)
              : occupancy<pnp::ik_waypoints_v_kernel<float, true>>(s, block, 0, &occ);
  if (rc) return rc;
  // envs reserved per ticket atomic: ~1/8 of a warp's share within [32 S, 128] (keeps the tail short)
  const PersistentGrid g = persistent_grid(s, n, pair ? 2 : 1, block, occ, small, 8, 128);
  const int grid = g.grid;
  a.chunk = g.chunk;
  a.solo_warp = small ? 1u : 0u;
  if (!spec)
    pnp::ik_waypoints_kernel<float, pnp::GenericKin><<<grid, block, 0, st>>>(a);
  else {
    // PNP_WAYPOINT_FUSE=0 (read per call; tests and measurements only): the accepting pass of a solve is not also
    // the first iteration of the next one - one pass more per solve, bit-identical results
    const char* fe = getenv("PNP_WAYPOINT_FUSE");
    const bool fuse = !fe || atoi(fe) != 0;
    if (pair && fuse) pnp::ik_waypoints_v_kernel<pnp::F2, true><<<grid, block, 0, st>>>(a);
    else if (pair) pnp::ik_waypoints_v_kernel<pnp::F2, false><<<grid, block, 0, st>>>(a);
    else if (fuse) pnp::ik_waypoints_v_kernel<float, true><<<grid, block, 0, st>>>(a);
    else pnp::ik_waypoints_v_kernel<float, false><<<grid, block, 0, st>>>(a);
  }
  ++g_launches;
  CUDA_TRY(cudaGetLastError());
  return PNP_OK;
}

}  // extern "C"

namespace {
template <typename T>
int pose_solve_impl(const T* tpos, const T* tquat, const T* q_init, int32_t q_init_stride, int64_t n,
                    const PnpIkParams* params, double rot_thresh, double rot_weight, T* q_out, T* final_pos,
                    T* final_quat, T* pos_err, T* rot_err, int32_t* iters, uint8_t* flags,
                    unsigned long long* counters, void* stream, pnp::PoseIkArgs<T>* args_out = nullptr) {
  int rc = check_ik_params(params);
  if (rc) return rc;
  if (!(rot_thresh > 0.0) || !(rot_weight > 0.0)) return fail(PNP_EINVAL, "rot_thresh and rot_weight must be > 0");
  if (n < 0 || (n > 0 && (!tpos || !tquat || !q_init || !q_out)))
    return fail(PNP_EINVAL, "ik_pose_solve: null pointer or negative n");
  if (q_init_stride != 0 && q_init_stride != PNP_NJOINT) return fail(PNP_EINVAL, "q_init_stride must be 0 or 7");
  DeviceState* s;
  if ((rc = current_state(&s))) return rc;
  bool spec;
  if ((rc = pick_kin(s, params->kinematics, &spec))) return rc;
  if (n == 0) return PNP_OK;
  if (n >= (int64_t(1) << 31)) return fail(PNP_EINVAL, "ik_pose_solve: n must be < 2^31 per call");
  cudaStream_t st = (cudaStream_t)stream;
  pnp::PoseIkArgs<T> a;
  if ((rc = stream_ticket(s, st, &a.ticket))) return rc;
  a.target_pos = tpos; a.target_quat = tquat; a.q_init = q_init; a.q_init_stride = q_init_stride; a.n = (unsigned)n;
  a.k = make_ik_const<T>(params);
  a.rot_thresh = (T)rot_thresh; a.rot_weight = (T)rot_weight;
  a.q_out = q_out; a.final_pos = final_pos; a.final_quat = final_quat; a.pos_err = pos_err; a.rot_err = rot_err;
  a.iters = iters; a.flags = flags; a.counters = counters;
  const bool small = n <= (long long)s->sm_count * pnp::IK_BLOCK;
  const int block = pnp::IK_BLOCK;
  int occ;
  rc = spec ? occupancy<pnp::ik_pose_solve_kernel<T, pnp::SpecKin>>(s, block, 0, &occ)
            : occupancy<pnp::ik_pose_solve_kernel<T, pnp::GenericKin>>(s, block, 0, &occ);
  if (rc) return rc;
  const PersistentGrid g = persistent_grid(s, n, 1, block, occ, small, 16, 256);
  a.chunk = g.chunk;
  a.solo_warp = small ? 1u : 0u;
  if (args_out) *args_out = a;  // the multistart's restarts use this block
  if (spec)
    pnp::ik_pose_solve_kernel<T, pnp::SpecKin><<<g.grid, block, 0, st>>>(a);
  else
    pnp::ik_pose_solve_kernel<T, pnp::GenericKin><<<g.grid, block, 0, st>>>(a);
  ++g_launches;
  CUDA_TRY(cudaGetLastError());
  return PNP_OK;
}

// Multi-start pose solve: pose_solve_impl, then the restart waves of ms_pose_wave_kernel (see multistart_impl).
template <typename T>
int pose_multistart_impl(const T* tpos, const T* tquat, const T* q_init, int32_t q_init_stride, int64_t n, const T* seeds,
                         int32_t n_seeds, const PnpIkParams* params, double rot_thresh, double rot_weight, T* q_out,
                         T* final_pos, T* final_quat, T* pos_err, T* rot_err, int32_t* iters, uint8_t* flags,
                         uint8_t* attempt, unsigned long long* counters, unsigned long long* restart_stats, void* scratch,
                         void* stream) {
  const size_t m = (size_t)n;
  return multistart_impl<pnp::PoseIkArgs<T>, pnp::IK_OUT_SEPARATE>(
      "ik_pose_multistart", n, seeds, n_seeds, params, flags, iters, attempt, counters, restart_stats, scratch,
      {byte_range(q_out, m * PNP_NJOINT * sizeof(T)), byte_range(final_pos, m * 3 * sizeof(T)),
       byte_range(final_quat, m * 4 * sizeof(T)), byte_range(pos_err, m * sizeof(T)), byte_range(rot_err, m * sizeof(T)),
       byte_range(iters, m * sizeof(int32_t)), byte_range(flags, m)},
      kMsPoseGroup, "PNP_MS_POSE_GROUP", stream,
      [&](int32_t* iters0, pnp::PoseIkArgs<T>& a) {
        return pose_solve_impl<T>(tpos, tquat, q_init, q_init_stride, n, params, rot_thresh, rot_weight, q_out, final_pos,
                                  final_quat, pos_err, rot_err, iters0, flags, counters, stream, &a);
      },
      [&](DeviceState* s, bool spec, const auto& m, cudaStream_t st) {
        return spec ? launch_ms_wave<pnp::ms_pose_wave_kernel<T, pnp::SpecKin>>(s, m, st)
                    : launch_ms_wave<pnp::ms_pose_wave_kernel<T, pnp::GenericKin>>(s, m, st);
      });
}

template <typename T>
int plan_order_impl(const T* q_start, const T* target, int64_t n, uint32_t* order, int32_t kinematics, void* stream,
                    float4* records = nullptr) {
  if (n < 0 || (n > 0 && (!q_start || !target || (!order && !records)))) return fail(PNP_EINVAL, "move_plan_order: null pointer or negative n");
  DeviceState* s;
  int rc = current_state(&s);
  if (rc) return rc;
  bool spec;
  if ((rc = pick_kin(s, kinematics, &spec))) return rc;
  if (n == 0) return PNP_OK;
  if (n >= (int64_t(1) << 31)) return fail(PNP_EINVAL, "move_plan_order: n must be < 2^31 per call");
  cudaStream_t st = (cudaStream_t)stream;
  unsigned* work = s->order_work + (size_t)stream_slot(s, st) * 2 * pnp::PLAN_BUCKETS;
  CUDA_TRY(cudaMemsetAsync(work, 0, 2 * pnp::PLAN_BUCKETS * sizeof(unsigned), st));
  const int per_block = pnp::PLAN_ORDER_BLOCK * pnp::PLAN_ORDER_PER_THREAD;
  const int grid = (int)((n + per_block - 1) / per_block);
  if (spec) {
    pnp::plan_order_hist_kernel<T, pnp::SpecKin><<<grid, pnp::PLAN_ORDER_BLOCK, 0, st>>>(q_start, target, (unsigned)n, work);
    pnp::plan_order_scatter_kernel<T, pnp::SpecKin><<<grid, pnp::PLAN_ORDER_BLOCK, 0, st>>>(q_start, target, (unsigned)n, work, order, records);
  } else {
    pnp::plan_order_hist_kernel<T, pnp::GenericKin><<<grid, pnp::PLAN_ORDER_BLOCK, 0, st>>>(q_start, target, (unsigned)n, work);
    pnp::plan_order_scatter_kernel<T, pnp::GenericKin><<<grid, pnp::PLAN_ORDER_BLOCK, 0, st>>>(q_start, target, (unsigned)n, work, order, records);
  }
  g_launches += 2;
  CUDA_TRY(cudaGetLastError());
  return PNP_OK;
}

template <typename T>
int move_plan_impl(const T* q_start, const T* target, int64_t n, const PnpMoveParams* mp, const PnpIkParams* params,
                   T* traj, int32_t* traj_len, T* q_final, int32_t* n_solves, int32_t* status,
                   unsigned long long* counters, uint32_t* order, void* stream, float4* records = nullptr) {
  int rc = check_ik_params(params);
  if (rc) return rc;
  if (!mp) return fail(PNP_EINVAL, "move params is NULL");
  if (records) {
    // pnp_move_ik_plan_sorted_f32: `records` is scratch of 48 B per env.  The FP32 value-type planner of the specialised
    // tree reads its envs from it (filled here, longest plan first); every other kernel takes the same scratch as a
    // plain order[n]
    DeviceState* s0;
    bool spec0;
    if ((rc = current_state(&s0)) || (rc = pick_kin(s0, params->kinematics, &spec0))) return rc;
    if (!(std::is_same<T, float>::value && spec0)) { order = reinterpret_cast<uint32_t*>(records); records = nullptr; }
    if ((rc = plan_order_impl<T>(q_start, target, n, order, params->kinematics, stream, records))) return rc;
  } else if (order && mp->compute_order) {
    if ((rc = plan_order_impl<T>(q_start, target, n, order, params->kinematics, stream))) return rc;
  }
  if (mp->traj_cap < 2 || mp->max_traj_points < 0 || !(mp->step_size > 0.0) || !(mp->pos_thresh >= 0.0))
    return fail(PNP_EINVAL, "move params: need traj_cap >= 2, max_traj_points >= 0, step_size > 0, pos_thresh >= 0");
  if (n < 0 || (n > 0 && (!q_start || !target || !traj || !traj_len || !q_final)))
    return fail(PNP_EINVAL, "move_ik_plan: null pointer or negative n");
  DeviceState* s;
  if ((rc = current_state(&s))) return rc;
  bool spec;
  if ((rc = pick_kin(s, params->kinematics, &spec))) return rc;
  if (n == 0) return PNP_OK;
  if (n >= (int64_t(1) << 31)) return fail(PNP_EINVAL, "move_ik_plan: n must be < 2^31 per call");
  cudaStream_t st = (cudaStream_t)stream;
  pnp::MoveArgs<T> a;
  if ((rc = stream_ticket(s, st, &a.ticket))) return rc;
  a.q_start = q_start; a.target = target; a.n = (unsigned)n;
  a.pos_thresh = (T)mp->pos_thresh; a.step_size = (T)mp->step_size;
  a.max_traj_points = mp->max_traj_points;
  a.max_outer = mp->max_outer > 0 ? mp->max_outer : 4 * mp->max_traj_points + 64;
  a.traj_cap = mp->traj_cap;
  a.k = make_ik_const<T>(params);
  a.traj = traj; a.traj_len = traj_len; a.q_final = q_final; a.n_solves = n_solves; a.status = status;
  a.counters = counters;
  a.order = order;
  a.records = records;
  const bool small = n <= (long long)s->sm_count * pnp::IK_BLOCK;
  int block = pnp::IK_BLOCK;
  int occ;
  if constexpr (std::is_same<T, float>::value) {
    if (spec) {
      // specialised tree, FP32: the value-type kernels (same arithmetic in both, branch-free common path)
      const bool pair = params->kinematics == PNP_KIN_SPEC_PAIR;
      const int S = pair ? 2 : 1;
      // PNP_WAYPOINT_FUSE=0 (read per call; tests and measurements only): a separate pass for the first
      // iteration of every solve, bit-identical results
      const char* fe = getenv("PNP_WAYPOINT_FUSE");
      const bool fuse = !fe || atoi(fe) != 0;
      // trajectory points staged in shared memory, blocks of 160 threads (PNP_PLAN_STAGE=0: direct stores, measurements)
      static const int env_stage = env_int("PNP_PLAN_STAGE", 1);
      const bool stage = env_stage && !pair && !small && mp->traj_cap % 4 == 0 && aligned16(traj);
      if (stage) block = pnp::PLAN_BLOCK;
      const size_t smem = pnp::plan_smem_bytes(S, block, stage);
      // (the fused instantiation's occupancy, for both; the staged kernels need 53 KB of dynamic shared memory)
      if (stage) {
        if ((rc = max_dynamic_smem<pnp::move_ik_plan_v_kernel<float, true, pnp::PLAN_BLOCK, true>>(s, smem)) ||
            (rc = max_dynamic_smem<pnp::move_ik_plan_v_kernel<float, false, pnp::PLAN_BLOCK, true>>(s, smem)))
          return rc;
      }
      rc = pair    ? occupancy<pnp::move_ik_plan_v_kernel<pnp::F2, true>>(s, block, smem, &occ)
           : stage ? occupancy<pnp::move_ik_plan_v_kernel<float, true, pnp::PLAN_BLOCK, true>>(s, block, smem, &occ)
                   : occupancy<pnp::move_ik_plan_v_kernel<float, true>>(s, block, smem, &occ);
      if (rc) return rc;
      const PersistentGrid g = persistent_grid(s, n, S, block, occ, small, 8, 128);
      const int gridv = g.grid;
      a.chunk = g.chunk;
      a.solo_warp = small ? 1u : 0u;
      if (pair && fuse) pnp::move_ik_plan_v_kernel<pnp::F2, true><<<gridv, block, smem, st>>>(a);
      else if (pair) pnp::move_ik_plan_v_kernel<pnp::F2, false><<<gridv, block, smem, st>>>(a);
      else if (stage && fuse) pnp::move_ik_plan_v_kernel<float, true, pnp::PLAN_BLOCK, true><<<gridv, block, smem, st>>>(a);
      else if (stage) pnp::move_ik_plan_v_kernel<float, false, pnp::PLAN_BLOCK, true><<<gridv, block, smem, st>>>(a);
      else if (fuse) pnp::move_ik_plan_v_kernel<float, true><<<gridv, block, smem, st>>>(a);
      else pnp::move_ik_plan_v_kernel<float, false><<<gridv, block, smem, st>>>(a);
      ++g_launches;
      CUDA_TRY(cudaGetLastError());
      return PNP_OK;
    }
  }
  rc = spec ? occupancy<pnp::move_ik_plan_kernel<T, pnp::SpecKin>>(s, block, 0, &occ)
            : occupancy<pnp::move_ik_plan_kernel<T, pnp::GenericKin>>(s, block, 0, &occ);
  if (rc) return rc;
  // envs reserved per ticket atomic: ~1/8 of a warp's share within [32, 128] (keeps the tail short)
  const PersistentGrid g = persistent_grid(s, n, 1, block, occ, small, 8, 128);
  a.chunk = g.chunk;
  a.solo_warp = small ? 1u : 0u;
  if (spec)
    pnp::move_ik_plan_kernel<T, pnp::SpecKin><<<g.grid, block, 0, st>>>(a);
  else
    pnp::move_ik_plan_kernel<T, pnp::GenericKin><<<g.grid, block, 0, st>>>(a);
  ++g_launches;
  CUDA_TRY(cudaGetLastError());
  return PNP_OK;
}

// Pose-mode planner: every argument is checked before anything is enqueued on the stream.
template <typename T>
int move_pose_plan_impl(const T* q_start, const T* goal_pos, const T* goal_quat, int64_t n, const PnpMovePoseParams* mp,
                        const PnpIkParams* params, T* pos_traj, T* quat_traj, T* q_traj, int32_t* traj_len, T* q_final,
                        int32_t* n_solves, int32_t* status, unsigned long long* counters, void* stream) {
  int rc = check_ik_params(params);
  if (rc) return rc;
  if (!mp) return fail(PNP_EINVAL, "move_pose params is NULL");
  if (mp->traj_cap < 1 || mp->max_traj_points < 0)
    return fail(PNP_EINVAL, "move_pose params: need traj_cap >= 1 and max_traj_points >= 0");
  if (!(mp->step_size > 0.0) || !(mp->rot_step > 0.0))
    return fail(PNP_EINVAL, "move_pose params: step_size and rot_step must be > 0");
  if (!(mp->ik_rot_thresh > 0.0) || !(mp->ik_rot_weight > 0.0))
    return fail(PNP_EINVAL, "move_pose params: ik_rot_thresh and ik_rot_weight must be > 0");
  // a plan whose last solve converged short of the planner's tolerance would re-aim at the goal forever
  if (!(mp->pos_thresh >= params->pos_thresh) || !(mp->rot_thresh >= mp->ik_rot_thresh))
    return fail(PNP_EINVAL, "move_pose params: need pos_thresh >= params->pos_thresh and rot_thresh >= ik_rot_thresh");
  if (n < 0 || (n > 0 && (!q_start || !goal_pos || !goal_quat || !pos_traj || !quat_traj || !traj_len || !q_final ||
                          !n_solves || !status)))
    return fail(PNP_EINVAL, "move_ik_plan_pose: null pointer or negative n");
  if (n >= (int64_t(1) << 31)) return fail(PNP_EINVAL, "move_ik_plan_pose: n must be < 2^31 per call");
  DeviceState* s;
  if ((rc = current_state(&s))) return rc;
  bool spec;
  if ((rc = pick_kin(s, params->kinematics, &spec))) return rc;
  if (n == 0) return PNP_OK;
  const bool small = n <= (long long)s->sm_count * pnp::IK_BLOCK;
  const int block = pnp::IK_BLOCK;
  int occ;
  rc = spec ? occupancy<pnp::move_pose_plan_kernel<T, pnp::SpecKin>>(s, block, 0, &occ)
            : occupancy<pnp::move_pose_plan_kernel<T, pnp::GenericKin>>(s, block, 0, &occ);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  pnp::MovePoseArgs<T> a{};
  if ((rc = stream_ticket(s, st, &a.ik.ticket))) return rc;
  a.ik.target_pos = goal_pos; a.ik.target_quat = goal_quat; a.ik.n = (unsigned)n;
  a.ik.k = make_ik_const<T>(params);
  a.ik.rot_thresh = (T)mp->ik_rot_thresh; a.ik.rot_weight = (T)mp->ik_rot_weight;
  a.ik.counters = counters;
  a.q_start = q_start;
  a.pos_thresh = (T)mp->pos_thresh; a.rot_thresh = (T)mp->rot_thresh;
  a.step_size = (T)mp->step_size; a.rot_step = (T)mp->rot_step;
  a.max_traj_points = mp->max_traj_points; a.traj_cap = mp->traj_cap;
  a.pos_traj = pos_traj; a.quat_traj = quat_traj; a.q_traj = q_traj;
  a.traj_len = traj_len; a.q_final = q_final; a.n_solves = n_solves; a.status = status;
  // the position planner's geometry: plans differ in length, so warps reserve ~1/8 of their share within [32, 128]
  const PersistentGrid g = persistent_grid(s, n, 1, block, occ, small, 8, 128);
  a.ik.chunk = g.chunk;
  a.ik.solo_warp = small ? 1u : 0u;
  if (spec)
    pnp::move_pose_plan_kernel<T, pnp::SpecKin><<<g.grid, block, 0, st>>>(a);
  else
    pnp::move_pose_plan_kernel<T, pnp::GenericKin><<<g.grid, block, 0, st>>>(a);
  ++g_launches;
  CUDA_TRY(cudaGetLastError());
  return PNP_OK;
}
}  // namespace

extern "C" {

int pnp_ik_pose_solve_f32(const float* target_pos, const float* target_quat, const float* q_init,
                          int32_t q_init_stride, int64_t n, const PnpIkParams* params, double rot_thresh,
                          double rot_weight, float* q_out, float* final_pos, float* final_quat, float* pos_err,
                          float* rot_err, int32_t* iters, uint8_t* flags, unsigned long long* counters, void* stream) {
  return pose_solve_impl<float>(target_pos, target_quat, q_init, q_init_stride, n, params, rot_thresh, rot_weight, q_out,
                                final_pos, final_quat, pos_err, rot_err, iters, flags, counters, stream);
}
int pnp_ik_pose_solve_f64(const double* target_pos, const double* target_quat, const double* q_init,
                          int32_t q_init_stride, int64_t n, const PnpIkParams* params, double rot_thresh,
                          double rot_weight, double* q_out, double* final_pos, double* final_quat, double* pos_err,
                          double* rot_err, int32_t* iters, uint8_t* flags, unsigned long long* counters, void* stream) {
  return pose_solve_impl<double>(target_pos, target_quat, q_init, q_init_stride, n, params, rot_thresh, rot_weight, q_out,
                                 final_pos, final_quat, pos_err, rot_err, iters, flags, counters, stream);
}

int pnp_ik_pose_solve_multistart_f32(const float* target_pos, const float* target_quat, const float* q_init,
                                     int32_t q_init_stride, int64_t n, const float* seeds, int32_t n_seeds,
                                     const PnpIkParams* params, double rot_thresh, double rot_weight, float* q_out,
                                     float* final_pos, float* final_quat, float* pos_err, float* rot_err, int32_t* iters,
                                     uint8_t* flags, uint8_t* attempt, unsigned long long* counters,
                                     unsigned long long* restart_stats, void* scratch, void* stream) {
  return pose_multistart_impl<float>(target_pos, target_quat, q_init, q_init_stride, n, seeds, n_seeds, params, rot_thresh,
                                     rot_weight, q_out, final_pos, final_quat, pos_err, rot_err, iters, flags, attempt,
                                     counters, restart_stats, scratch, stream);
}
int pnp_ik_pose_solve_multistart_f64(const double* target_pos, const double* target_quat, const double* q_init,
                                     int32_t q_init_stride, int64_t n, const double* seeds, int32_t n_seeds,
                                     const PnpIkParams* params, double rot_thresh, double rot_weight, double* q_out,
                                     double* final_pos, double* final_quat, double* pos_err, double* rot_err,
                                     int32_t* iters, uint8_t* flags, uint8_t* attempt, unsigned long long* counters,
                                     unsigned long long* restart_stats, void* scratch, void* stream) {
  return pose_multistart_impl<double>(target_pos, target_quat, q_init, q_init_stride, n, seeds, n_seeds, params,
                                      rot_thresh, rot_weight, q_out, final_pos, final_quat, pos_err, rot_err, iters, flags,
                                      attempt, counters, restart_stats, scratch, stream);
}

int pnp_move_plan_order_f32(const float* q_start, const float* target, int64_t n, uint32_t* order, int32_t kinematics,
                            void* stream) {
  return plan_order_impl<float>(q_start, target, n, order, kinematics, stream);
}
int pnp_move_plan_order_f64(const double* q_start, const double* target, int64_t n, uint32_t* order, int32_t kinematics,
                            void* stream) {
  return plan_order_impl<double>(q_start, target, n, order, kinematics, stream);
}

int pnp_move_plan_order_check(const uint32_t* order, int64_t n, uint32_t* bitmap_scratch, uint32_t* n_bad, void* stream) {
  if (n < 0 || (n > 0 && (!order || !bitmap_scratch)) || !n_bad) return fail(PNP_EINVAL, "move_plan_order_check: null pointer or negative n");
  if (n >= (int64_t(1) << 31)) return fail(PNP_EINVAL, "move_plan_order_check: n must be < 2^31");
  DeviceState* s;
  int rc = current_state(&s);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  CUDA_TRY(cudaMemsetAsync(n_bad, 0, sizeof(uint32_t), st));
  if (n == 0) return PNP_OK;
  CUDA_TRY(cudaMemsetAsync(bitmap_scratch, 0, (size_t)((n + 31) / 32) * sizeof(uint32_t), st));
  pnp::plan_order_check_kernel<<<grid_for(n, 256, s->sm_count, 8), 256, 0, st>>>(order, (unsigned)n, bitmap_scratch, n_bad);
  ++g_launches;
  CUDA_TRY(cudaGetLastError());
  return PNP_OK;
}

int pnp_move_ik_plan_f32(const float* q_start, const float* target, int64_t n, const PnpMoveParams* mp,
                         const PnpIkParams* params, float* traj, int32_t* traj_len, float* q_final,
                         int32_t* n_solves, int32_t* status, unsigned long long* counters, void* stream) {
  return move_plan_impl<float>(q_start, target, n, mp, params, traj, traj_len, q_final, n_solves, status, counters, nullptr,
                               stream);
}
int pnp_move_ik_plan_ordered_f32(const float* q_start, const float* target, uint32_t* order, int64_t n,
                                 const PnpMoveParams* mp, const PnpIkParams* params, float* traj, int32_t* traj_len,
                                 float* q_final, int32_t* n_solves, int32_t* status, unsigned long long* counters,
                                 void* stream) {
  return move_plan_impl<float>(q_start, target, n, mp, params, traj, traj_len, q_final, n_solves, status, counters, order,
                               stream);
}
int pnp_move_ik_plan_sorted_f32(const float* q_start, const float* target, void* scratch48, int64_t n,
                                const PnpMoveParams* mp, const PnpIkParams* params, float* traj, int32_t* traj_len,
                                float* q_final, int32_t* n_solves, int32_t* status, unsigned long long* counters, void* stream) {
  if (n > 0 && (!scratch48 || !aligned16(scratch48))) return fail(PNP_EINVAL, "move_ik_plan_sorted: scratch must be non-null and 16-byte aligned");
  return move_plan_impl<float>(q_start, target, n, mp, params, traj, traj_len, q_final, n_solves, status, counters, nullptr,
                               stream, reinterpret_cast<float4*>(scratch48));
}
int pnp_move_ik_plan_f64(const double* q_start, const double* target, int64_t n, const PnpMoveParams* mp,
                         const PnpIkParams* params, double* traj, int32_t* traj_len, double* q_final,
                         int32_t* n_solves, int32_t* status, unsigned long long* counters, void* stream) {
  return move_plan_impl<double>(q_start, target, n, mp, params, traj, traj_len, q_final, n_solves, status, counters, nullptr,
                                stream);
}
int pnp_move_ik_plan_ordered_f64(const double* q_start, const double* target, uint32_t* order, int64_t n,
                                 const PnpMoveParams* mp, const PnpIkParams* params, double* traj, int32_t* traj_len,
                                 double* q_final, int32_t* n_solves, int32_t* status, unsigned long long* counters,
                                 void* stream) {
  return move_plan_impl<double>(q_start, target, n, mp, params, traj, traj_len, q_final, n_solves, status, counters, order,
                                stream);
}

int pnp_move_ik_plan_pose_f32(const float* q_start, const float* goal_pos, const float* goal_quat, int64_t n,
                              const PnpMovePoseParams* move, const PnpIkParams* params, float* pos_traj, float* quat_traj,
                              float* q_traj, int32_t* traj_len, float* q_final, int32_t* n_solves, int32_t* status,
                              unsigned long long* counters, void* stream) {
  return move_pose_plan_impl<float>(q_start, goal_pos, goal_quat, n, move, params, pos_traj, quat_traj, q_traj, traj_len,
                                    q_final, n_solves, status, counters, stream);
}
int pnp_move_ik_plan_pose_f64(const double* q_start, const double* goal_pos, const double* goal_quat, int64_t n,
                              const PnpMovePoseParams* move, const PnpIkParams* params, double* pos_traj,
                              double* quat_traj, double* q_traj, int32_t* traj_len, double* q_final, int32_t* n_solves,
                              int32_t* status, unsigned long long* counters, void* stream) {
  return move_pose_plan_impl<double>(q_start, goal_pos, goal_quat, n, move, params, pos_traj, quat_traj, q_traj, traj_len,
                                     q_final, n_solves, status, counters, stream);
}

int pnp_reward_f32(const float* ag, const float* dg, const float* ee_pos, const float* ee_quat, const float* width,
                   const int32_t* task_index, int64_t n, const PnpRewardParams* params, float* reward,
                   float* is_success, unsigned long long* counters, void* stream) {
  return reward_impl<float>(ag, dg, ee_pos, ee_quat, width, task_index, n, params, reward, is_success, counters, stream);
}
int pnp_reward_f64(const double* ag, const double* dg, const double* ee_pos, const double* ee_quat,
                   const double* width, const int32_t* task_index, int64_t n, const PnpRewardParams* params,
                   float* reward, float* is_success, unsigned long long* counters, void* stream) {
  return reward_impl<double>(ag, dg, ee_pos, ee_quat, width, task_index, n, params, reward, is_success, counters,
                             stream);
}

int pnp_get_obs_f32(const float* q_arm, const float* qvel_arm, const float* fingers, const float* obj_pos,
                    const float* obj_quat, const float* obj_vel, const float* goal, int32_t goal_stride, int64_t n,
                    double dt, float* out, int32_t kinematics, void* stream) {
  return get_obs_impl<float>(q_arm, qvel_arm, fingers, obj_pos, obj_quat, obj_vel, goal, goal_stride, n, dt, out,
                             kinematics, stream);
}
int pnp_get_obs_f64(const double* q_arm, const double* qvel_arm, const double* fingers, const double* obj_pos,
                    const double* obj_quat, const double* obj_vel, const double* goal, int32_t goal_stride,
                    int64_t n, double dt, double* out, int32_t kinematics, void* stream) {
  return get_obs_impl<double>(q_arm, qvel_arm, fingers, obj_pos, obj_quat, obj_vel, goal, goal_stride, n, dt, out,
                              kinematics, stream);
}

int pnp_her_relabel_f32(const float* obs, const float* next_obs, const int32_t* future_idx, const float* ee_quat,
                        const int32_t* task_index, int64_t n, const PnpRewardParams* params,
                        const PnpNormalizeParams* norm, float* out_obs, float* out_next_obs, float* reward,
                        float* is_success, unsigned long long* counters, void* stream) {
  return pnp_her_relabel_table_f32(obs, next_obs, future_idx, nullptr, ee_quat, task_index, n, params, norm, out_obs,
                                   out_next_obs, reward, is_success, counters, stream);
}

int pnp_her_relabel_table_f32(const float* obs, const float* next_obs, const int32_t* future_idx, const float* future_ag,
                              const float* ee_quat, const int32_t* task_index, int64_t n, const PnpRewardParams* params,
                              const PnpNormalizeParams* norm, float* out_obs, float* out_next_obs, float* reward,
                              float* is_success, unsigned long long* counters, void* stream) {
  if (!params) return fail(PNP_EINVAL, "params is NULL");
  if (params->n_tasks <= 0) return fail(PNP_EINVAL, "n_tasks must be > 0");
  if (n < 0 || (n > 0 && (!obs || !next_obs || !future_idx || !ee_quat || !task_index || !out_obs || !out_next_obs || !reward)))
    return fail(PNP_EINVAL, "her_relabel: null pointer or negative n");
  if (n > 0) {
    const size_t bytes = (size_t)n * pnp::HER_ROW * sizeof(float);
    auto overlap = [bytes](const float* x, const float* y) {
      const uintptr_t a0 = (uintptr_t)x, b0 = (uintptr_t)y;
      return a0 < b0 + bytes && b0 < a0 + bytes;
    };
    if (overlap(out_obs, obs) || overlap(out_obs, next_obs) || overlap(out_next_obs, obs) || overlap(out_next_obs, next_obs) ||
        overlap(out_obs, out_next_obs))
      return fail(PNP_EINVAL, "her_relabel: outputs must not alias or overlap the inputs or each other (future goals are gathered from next_obs)");
  }
  if (n > 0 && !aligned16(ee_quat)) return fail(PNP_EINVAL, "her_relabel: ee_quat must be 16-byte aligned");
  DeviceState* s;
  int rc = current_state(&s);
  if (rc) return rc;
  if (n == 0) return PNP_OK;
  pnp::HerArgs a;
  a.obs = obs; a.next_obs = next_obs; a.future_idx = future_idx; a.future_ag = future_ag; a.ee_quat = ee_quat;
  a.task = task_index;
  a.n_total = n; a.k = make_reward_const(params);
  a.out_obs = out_obs; a.out_next = out_next_obs; a.reward = reward; a.success = is_success; a.counters = counters;
  a.normalize = norm ? 1 : 0;
  a.clip = norm ? (float)norm->clip_obs : 0.f;
  for (int k = 0; k < pnp::HER_ROW; ++k) {
    a.mean_hi[k] = norm ? (float)norm->mean[k] : 0.f;
    a.mean_lo[k] = norm ? (float)(norm->mean[k] - (double)a.mean_hi[k]) : 0.f;
    a.inv_std[k] = norm ? (float)(1.0 / std::sqrt(norm->var[k] + norm->epsilon)) : 1.f;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const size_t smem_bulk = 2 * 2 * pnp::HER_TILE_BYTES, smem_plain = 2 * pnp::HER_TILE_BYTES;
  if ((rc = max_dynamic_smem<pnp::her_relabel_kernel<true>>(s, smem_bulk))) return rc;
  const bool bulk_ok = aligned16(obs) && aligned16(next_obs) && aligned16(out_obs) && aligned16(out_next_obs);
  const int64_t full = bulk_ok ? (n / pnp::HER_TILE) * pnp::HER_TILE : 0;
  if (full > 0) {
    a.row0 = 0; a.n = full;
    const int grid = grid_for(full, pnp::HER_TILE, s->sm_count, 4);
    pnp::her_relabel_kernel<true><<<grid, pnp::HER_TILE, smem_bulk, st>>>(a);
    ++g_launches;
    CUDA_TRY(cudaGetLastError());
  }
  if (n - full > 0) {  // ragged tail (< 128 rows) or unaligned buffers: plain staged copies
    pnp::HerArgs t = a;
    t.row0 = full; t.n = n - full;  // each launch adds its own row count to counters[N]
    const int grid = grid_for(n - full, pnp::HER_TILE, s->sm_count, 8);
    pnp::her_relabel_kernel<false><<<grid, pnp::HER_TILE, smem_plain, st>>>(t);
    ++g_launches;
    CUDA_TRY(cudaGetLastError());
  }
  return PNP_OK;
}

int pnp_goal_distance_f64(const double* a, const double* b, int64_t n, double* d, void* stream) {
  if (n < 0 || (n > 0 && (!a || !b || !d))) return fail(PNP_EINVAL, "goal_distance: null pointer or negative n");
  DeviceState* s;
  int rc = current_state(&s);
  if (rc) return rc;
  if (n == 0) return PNP_OK;
  pnp::goal_distance_kernel<<<grid_for(n, 256, s->sm_count, 8), 256, 0, (cudaStream_t)stream>>>(a, b, n, d);
  ++g_launches;
  CUDA_TRY(cudaGetLastError());
  return PNP_OK;
}

int pnp_probe_fp32_peak(double* tflops_out, double* ms_out) {
  DeviceState* s;
  int rc = current_state(&s);
  if (rc) return rc;
  float* d_out = nullptr;
  CUDA_TRY(cudaMalloc(&d_out, sizeof(float)));
  cudaEvent_t e0, e1;
  CUDA_TRY(cudaEventCreate(&e0));
  CUDA_TRY(cudaEventCreate(&e1));
  const int blocks = s->sm_count * 8, threads = 256, iters = 4096;
  pnp::fp32_peak_kernel<<<blocks, threads>>>(d_out, 64, 0.999f, 0.001f);  // warm-up
  CUDA_TRY(cudaEventRecord(e0));
  pnp::fp32_peak_kernel<<<blocks, threads>>>(d_out, iters, 0.999f, 0.001f);
  CUDA_TRY(cudaEventRecord(e1));
  CUDA_TRY(cudaEventSynchronize(e1));
  g_launches += 2;
  float ms = 0.f;
  CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));
  const double flop = 2.0 * 8 * 16 * (double)iters * (double)blocks * threads;
  if (tflops_out) *tflops_out = flop / (ms * 1e-3) / 1e12;
  if (ms_out) *ms_out = ms;
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(d_out);
  return PNP_OK;
}

}  // extern "C"

#include "pnp_host_api.inc"

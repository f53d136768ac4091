// cs_api.cu — the C ABI of include/coreslam_b200.h over the kernels in cs_kernels.cuh.
//
// One cs_processor replaces one CoreSLAMProcessor (CoreSLAM/CoreSLAMProcessor.cs): it owns the
// device-resident HoleMap, the pinned staging block the scan is written into, one CUDA stream and a
// mapped result slot the finalize kernel stores the pose into.  No CPU fallback exists: every compute
// entry point launches kernels or fails.
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>  // header-only: ranges cost a pointer test unless a profiler is attached

#include <chrono>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <limits>
#include <cstring>
#include <atomic>
#include <exception>
#include <memory>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/coreslam_b200.h"
#include "cs_kernels.cuh"
#include "cs_obstacle.cuh"
#include "cs_lattice.cuh"
#include "cs_bnb.cuh"
#include "cs_wedge.cuh"

static_assert(sizeof(CsDevResult) == sizeof(cs_result), "cs_result layout");
static_assert(sizeof(cs_config) == 72, "cs_config layout (ctypes / P/Invoke mirror it)");
static_assert(sizeof(CsStepHeader) == 48, "CsStepHeader");
static_assert(sizeof(cs_lattice) == 36 && sizeof(cs_lattice_hit) == 20, "cs_lattice layout (ctypes / P/Invoke mirror it)");
static_assert(sizeof(cs_relocalize_stats) == 40, "cs_relocalize_stats layout (ctypes / P/Invoke mirror it)");
static_assert(CS_LAT_SEQ_MAX == CS_SEQUENCE_MAX_SCANS && CS_SEQUENCE_MAX_SCANS <= CS_LAT_THREADS, "one thread per scan of a sequence");

namespace {

thread_local std::string g_create_error;

constexpr size_t kHdrBytes = 64;
// NVTX range over one C-ABI call (SURVEY section 5): shows up as a named span in Nsight Systems / ncu --nvtx
struct NvtxRange {
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
};

constexpr int kRayCopies = 8;  // copies of the per-ray draw parameters of a stand-alone session (see CsSession::rays)

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// Owners of the CUDA resources a handle allocates: released when the owner goes, so a failed create, a destroy and an
// early return all give back what was allocated.  The descriptors copied to the device (CsSession, CsObstacle,
// CsStepArgs) hold plain pointers into these blocks.
struct DevFree { void operator()(void* p) const { cudaFree(p); } };
struct HostFree { void operator()(void* p) const { cudaFreeHost(p); } };  // pinned, plain or mapped
struct StreamDestroy { void operator()(cudaStream_t s) const { cudaStreamDestroy(s); } };
struct EventDestroy { void operator()(cudaEvent_t e) const { cudaEventDestroy(e); } };
template <typename T> using DevBuf = std::unique_ptr<T[], DevFree>;
template <typename T> using HostBuf = std::unique_ptr<T[], HostFree>;
using Stream = std::unique_ptr<CUstream_st, StreamDestroy>;
using Event = std::unique_ptr<CUevent_st, EventDestroy>;

// `count` elements of T into an empty owner.
template <typename T> cudaError_t alloc(DevBuf<T>& buf, size_t count) {
  T* p = nullptr;
  const cudaError_t e = cudaMalloc(&p, count * sizeof(T));
  buf.reset(p);
  return e;
}
template <typename T> cudaError_t alloc(HostBuf<T>& buf, size_t count, unsigned flags = cudaHostAllocDefault) {
  T* p = nullptr;
  const cudaError_t e = cudaHostAlloc(&p, count * sizeof(T), flags);
  buf.reset(p);
  return e;
}
// a scratch block of at least `count` elements (kept when big enough; its contents do not survive a call)
template <typename T> cudaError_t grow(DevBuf<T>& buf, size_t& cap, size_t count) {
  if (cap >= count) return cudaSuccess;
  buf.reset();
  cap = 0;
  const cudaError_t e = alloc(buf, count);
  if (e == cudaSuccess) cap = count;
  return e;
}
cudaError_t create(Stream& s) {
  cudaStream_t p = nullptr;
  const cudaError_t e = cudaStreamCreateWithFlags(&p, cudaStreamNonBlocking);
  s.reset(p);
  return e;
}
cudaError_t create(Event& ev, unsigned flags = cudaEventDisableTiming) {
  cudaEvent_t p = nullptr;
  const cudaError_t e = cudaEventCreateWithFlags(&p, flags);
  ev.reset(p);
  return e;
}

struct Timing {
  Event ev[5];
};

}  // namespace

// Production mode (on-device Philox candidates): the candidates of scan k+1 are a function of (seed, k+1) alone, so their sort
// is queued right behind the draw kernel of scan k and runs in its shadow; the search of scan k+1 then starts without a sort
// in front.  The same holds for the replay of a device-resident scan log with candidate tables (cs_replay): the next scan's
// table is already in HBM.  (Not for cs_update with a host table: it arrives with the scan.)  The descriptor says what was
// sorted into which half of CsSession::s2_sorted; a step that asks for anything else (another candidate mode, table, slice or
// scan number, another upload of the log) sorts as usual and overwrites it.
struct Presort {
  bool valid = false;
  unsigned scan_index = 0;
  int cand_first = 0, cand_count = 0, slot = 0;
  int cand_mode = 0;
  const float* cand = nullptr;  // replay of a device-resident log with candidate tables: the table that was sorted ...
  uint64_t tag = 0;             // ... and the upload of the log it belongs to
};

// Host mirror of the deterministic parts of the state machine.  A batch steps all its sessions together, so one mirror
// serves one processor or a whole batch.
struct StepState {
  int parity = 0;      // which CsSession::state / key slot is current
  int scan_count = 0;  // CoreSLAMProcessor.cs:34 (saturates at PositionSearchBeginning)
  int search_begin = 5;
  unsigned update_count = 0;  // Philox scan index
  unsigned step_counter = 0;  // source of CsStepArgs::step_id
  int w_slot = 0;             // which third of CsSession::w_top the next drawn step counts into
  int s2_toggle = 0;          // which half of CsSession::s2_sorted the next sort writes

  bool searches() const { return scan_count >= search_begin; }  // :726
  // after an Update has been enqueued
  void advance(bool searched) {
    parity ^= 1;
    update_count++;
    if (!searched) scan_count++;  // :741
  }
};

// What a processor (one session) and a batch (n sessions of the same shape) both have and mean alike.
struct CsHost {
  int device = 0;
  cudaStream_t stream = nullptr;
  Stream own_stream;  // the stream above when the library created it (never one the caller passed in cfg.stream)
  bool tiled = true;
  int size = 0, pitch_tiles = 0, n_cand = 0;
  float scale = 0.f;
  size_t map_cells = 0;  // allocated cells of one map (tiled: pitch_tiles^2 * 64)
  DevBuf<CsSession> d_sess;
  DevBuf<uint16_t> d_linear;  // lazily allocated row-major scratch for upload/download
  DevBuf<unsigned long long> d_checksum;
  // ray and wedge scratch of all sessions (CsSession::rays .. w_top, alloc_ray_scratch)
  DevBuf<int4> d_rays;
  DevBuf<int> d_batch_max;
  DevBuf<unsigned long long> d_prep_words;
  DevBuf<int2> d_w_rk;
  DevBuf<float2> d_w_bkey;
  DevBuf<int> d_w_top;
  // ObstacleMaps (cfg.obstacle_map_size > 0), one per session, all of the geometry `ho` (alloc_obstacle_maps): session j's
  // pixels, bitmap and touched counter are the j-th pieces of the three blocks, described by d_obst[j] (host mirrors: a
  // processor's `ho` itself, a batch's cs_batch::obst)
  CsObstacle ho{};
  DevBuf<CsObstacle> d_obst;
  DevBuf<int8_t> d_obst_pixels;
  DevBuf<uint32_t> d_obst_no_hit;
  DevBuf<long long> d_obst_touched;
  int s2_cap = 0;                // slab-search capacity of one session (0: no slab-search scratch)
  StepState step;
  // stuck-poll word (CsSpin) in pinned+mapped memory, and its device address: a processor's lies in its result slot, a
  // batch allocates its own under CS_FLAG_DEBUG_BOUNDED_SPIN (NULL otherwise)
  uint8_t* h_stuck = nullptr;
  uint8_t* d_stuck = nullptr;
  uint64_t launches = 0;
  std::string error;
  bool poisoned = false;
};

struct cs_processor : CsHost {
  cs_config cfg{};
  int max_points = 0;

  CsSession hs{};            // host mirror of the session descriptor
  DevBuf<uint16_t> d_map;
  DevBuf<uint8_t> d_packed;
  DevBuf<int> d_ray_dbg;
  DevBuf<int> d_distances;
  DevBuf<unsigned long long> d_spec;  // glue table (CsStepArgs::spec): 8 words per flat candidate
  DevBuf<long long> d_ring_cycles;

  // slab search scratch (CsSession::s2_*), allocated when the handle has enough candidates for it to pay
  DevBuf<float4> d_s2_sorted;
  DevBuf<float4> d_s2_tmp;
  DevBuf<unsigned long long> d_s2_meta;
  DevBuf<unsigned long long> d_s2_acc;
  DevBuf<unsigned> d_s2_ghist;
  Presort presort;

  // ObstacleMap (cfg.obstacle_map_size > 0; CoreSLAM/ObstacleMap.cs, CoreSLAMProcessor.cs:53, :132-133): CsHost::ho is the
  // host mirror of its descriptor
  int unmapped_obstacle_hits = -5;  // :98

  // asynchronous map export (cs_map_export_begin / _wait): snapshot on the main stream, D2H on a side stream
  Stream export_stream;
  Event ev_export_snap, ev_export_done;
  bool export_busy = false;
  DevBuf<int8_t> d_obst_snap;

  DevBuf<float2> d_cloud;  // scan points computed on the device from raw segments (cs_update_segments)

  // cs_relocalize: the scan (allocated on first use), the distance volume and the top-k lists (both grow on demand)
  DevBuf<float2> d_lat_points;
  DevBuf<int> d_lat_volume;
  size_t lat_volume_cap = 0;
  DevBuf<unsigned long long> d_lat_lists;
  size_t lat_lists_cap = 0;
  // cs_relocalize_bounded (cs_bnb.cuh): the min-window grids, the top-level seeds, two node lists, the per-tile slot index
  // and its counters; the distances of the evaluated tiles go to d_lat_volume, the top-k lists to d_lat_lists
  DevBuf<uint16_t> d_bnb_grids;
  size_t bnb_grids_cap = 0;
  DevBuf<int> d_bnb_seeds;
  size_t bnb_seeds_cap = 0;
  DevBuf<int4> d_bnb_nodes;
  size_t bnb_nodes_cap = 0;
  DevBuf<int> d_bnb_slot;
  size_t bnb_slot_cap = 0;
  DevBuf<unsigned long long> d_bnb_counters;
  // cs_relocalize_sequence*: the concatenated scans (grow on demand), the odometry and scan_first as passed, and the
  // per-scan records the kernels read (CS_SEQUENCE_MAX_SCANS each, allocated on first use)
  DevBuf<float2> d_seq_points;
  size_t seq_points_cap = 0;
  DevBuf<float> d_seq_odometry;
  DevBuf<int> d_seq_first;
  DevBuf<CsSeqScan> d_seq_scans;

  // staging: [hdr 64][points][cand][cand_cs]; segments path: [hdr 64][rays][seg_first][seg_poses][cand]
  size_t stage_bytes = 0;
  HostBuf<uint8_t> h_stage;  // pinned
  DevBuf<uint8_t> d_stage;
  // cs_update's staging runs ahead of the stream: the H2D copy of scan k goes through a copy stream into the buffer scan
  // k-1 is NOT using (d_stage / d_stage_b alternate), so it overlaps the integration of scan k-1 instead of queueing
  // behind it; the main stream only waits for the copy's event.  ev_stage_free[i]: last step that reads buffer i is enqueued.
  DevBuf<uint8_t> d_stage_b;
  Stream copy_stream;
  Event ev_copy, ev_stage_free[2];
  int stage_flip = 0, stage_cur = 0;

  // mapped result slot
  HostBuf<uint8_t> h_slot;  // pinned+mapped: CsDevResult at 0, seq flag at 64, stuck-poll word (CsSpin) at 96
  uint8_t* d_slot = nullptr;
  unsigned seq = 0;

  // split-phase update in flight (cs_update_begin ... cs_update_finish)
  bool pending = false;
  CsStepArgs pending_args{};
  int pending_points = 0, pending_rings = 0;

  // candidate-split group (cs_group_*): this rank's exchange table and the (peer-mapped) tables of all ranks
  int group_rank = 0, group_world = 0;
  bool group_shares_device = false;  // another rank of the group runs on this handle's device (same process)
  unsigned xchg_seq = 0;
  DevBuf<unsigned long long> d_xchg;
  unsigned long long* xchg_peer[CS_GROUP_MAX] = {};
  bool xchg_ipc[CS_GROUP_MAX] = {};  // opened with cudaIpcOpenMemHandle (to be closed on detach)

  Timing tm;
  cs_timing last_timing{};

  // The owners release after this: on the handle's device, once every stream the handle queues work on has drained (the
  // export stream's copy writes caller memory) and the peers' exchange tables are unmapped.
  ~cs_processor() {
    cudaSetDevice(device);
    for (cudaStream_t s : {stream, copy_stream.get(), export_stream.get()})
      if (s) cudaStreamSynchronize(s);
    for (int p = 0; p < CS_GROUP_MAX; p++)
      if (xchg_ipc[p] && xchg_peer[p]) cudaIpcCloseMemHandle(xchg_peer[p]);
  }
};

struct cs_scanlog {
  int device = 0, n_scans = 0, max_points = 0, n_offsets = 0;
  std::vector<CsStepHeader> h_hdr;
  std::vector<float> h_points;   // n_scans * max_points * 2
  std::vector<float> h_offsets;  // n_scans * n_offsets * 3
  std::vector<double> h_max_range;  // per scan, sizes the update kernel's grid
  DevBuf<CsStepHeader> d_hdr;
  DevBuf<float2> d_points;
  DevBuf<float> d_offsets;
  DevBuf<CsDevResult> d_results;
  bool uploaded = false;
  uint64_t generation = 0;  // counts the uploads: what a handle sorted ahead from this log is only good for the same upload

  ~cs_scanlog() { cudaSetDevice(device); }  // (the owners release on the log's device)
};

namespace {

cs_status fail(CsHost* h, cs_status code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (h) {
    h->error = buf;
    if (code == CS_ERR_CUDA) h->poisoned = true;
  } else {
    g_create_error = buf;
  }
  return code;
}

#define CS_CUDA(h, expr)                                                                         \
  do {                                                                                           \
    cudaError_t _e = (expr);                                                                     \
    if (_e != cudaSuccess)                                                                       \
      return fail((h), CS_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)

// CS_FLAG_DEBUG_BOUNDED_SPIN: a device-side poll of an earlier step gave up (CsSpin, cs_kernels.cuh): the handle fails
const char* stuck_site_name(unsigned w) {
  switch (w & 0xffu) {
    case CS_STUCK_POSE: return "the pose of the step (search kernel / set-up kernel never published it)";
    case CS_STUCK_RAYS: return "the rays of the step (a preparing block never arrived)";
    case CS_STUCK_HANDOFF: return "the hand-off word of a contested cell";
    default: return "an unknown word";
  }
}
#define CS_CHECK_STUCK(h)                                                                                        \
  do {                                                                                                           \
    const unsigned _w = (h)->h_stuck ? *reinterpret_cast<volatile unsigned*>((h)->h_stuck) : 0u;                \
    if (_w)                                                                                                      \
      return fail((h), CS_ERR_CUDA, "bounded polls: block %u of the draw kernel gave up waiting for %s", _w >> 8, \
                  stuck_site_name(_w));                                                                          \
  } while (0)

#define CS_CHECK_HANDLE(h)                                                          \
  do {                                                                              \
    if (!(h)) return CS_ERR_INVALID_ARGUMENT;                                       \
    if ((h)->poisoned) return CS_ERR_CUDA;                                          \
    CS_CHECK_STUCK(h);                                                              \
    cudaError_t _e = cudaSetDevice((h)->device);                                    \
    if (_e != cudaSuccess) return fail((h), CS_ERR_CUDA, "cudaSetDevice: %s", cudaGetErrorString(_e)); \
  } while (0)

// In cs_create / cs_batch_create: a failed call records its message and returns through the function's `bail`, which
// destroys the half-built handle.
#define CS_CREATE_CUDA(h, expr)                                                                              \
  do {                                                                                                       \
    cudaError_t _e = (expr);                                                                                 \
    if (_e != cudaSuccess) {                                                                                 \
      const cs_status _st = _e == cudaErrorMemoryAllocation ? CS_ERR_OUT_OF_MEMORY : CS_ERR_CUDA;            \
      fail((h), _st, "%s failed: %s", #expr, cudaGetErrorString(_e));                                        \
      return bail(_st);                                                                                      \
    }                                                                                                        \
  } while (0)

cs_status push_session(cs_processor* h) {
  CS_CUDA(h, cudaMemcpyAsync(h->d_sess.get(), &h->hs, sizeof(CsSession), cudaMemcpyHostToDevice, h->stream));
  return CS_OK;
}

// session fields the host owns; state/key/x1.. are device-owned, so properties are patched individually
cs_status patch_session(cs_processor* h, size_t offset, const void* src, size_t bytes) {
  CS_CUDA(h, cudaMemcpyAsync(reinterpret_cast<uint8_t*>(h->d_sess.get()) + offset, src, bytes, cudaMemcpyHostToDevice,
                             h->stream));
  CS_CUDA(h, cudaStreamSynchronize(h->stream));  // src may be a stack temporary
  return CS_OK;
}

template <typename F>
void dispatch_layout(bool tiled, F&& f) {
  if (tiled) f(std::true_type{});
  else f(std::false_type{});
}

cs_status launch_fill(cs_processor* h, uint16_t value) {
  cs_fill_kernel<<<148 * 4, 256, 0, h->stream>>>(h->d_map.get(), h->map_cells, value);
  h->launches++;
  CS_CUDA(h, cudaGetLastError());
  return CS_OK;
}

struct StagePlan {
  size_t off_points, off_cand, off_cs, total;
};

StagePlan plan_stage(int n_points, int n_cand_floats3, bool with_cs) {
  StagePlan p;
  p.off_points = kHdrBytes;
  p.off_cand = align_up(p.off_points + (size_t)n_points * 8, 16);
  p.off_cs = align_up(p.off_cand + (size_t)n_cand_floats3 * 12, 16);
  p.total = align_up(p.off_cs + (with_cs ? (size_t)(n_cand_floats3 + 1) * 8 : 0), 16);
  return p;
}

// Wedge integration (cs_wedge.cuh): levels a ray of a size x size map can reach, and the words of one half of CsSession::w_top.
int wedge_levels(int size) {
  const int k = size > 1 ? size - 1 : 1;
  int L = 0;
  if (k < 64) { while ((2 << L) <= k) L++; } else L = 5 + (k >> 6);
  return L + 1;
}
size_t wedge_top_words(int size) { return (size_t)wedge_levels(size) * (CS_W_SECTORS + 1); }

// The host-owned constants of a session (the defaults of CoreSLAMProcessor.cs:82-92); the caller adds its scratch pointers.
void init_session(CsSession& s, const CsHost& h, const cs_config& cfg, uint16_t* map) {
  memset(&s, 0, sizeof(s));
  s.map = map;
  s.size = h.size;
  s.pitch_tiles = h.pitch_tiles;
  s.scale = h.scale;
  s.sigma_xy = cfg.sigma_xy;
  s.sigma_theta = cfg.sigma_theta;
  s.iters = cfg.iterations_per_thread;
  s.threads = cfg.num_search_threads;
  s.n_cand = h.n_cand;
  s.quality = 50;        // :82
  s.hole_width = 0.6f;   // :87
  s.search_begin = 5;    // :92
  s.seed = cfg.seed;
  s.w_levels = wedge_levels(h.size);
}

// The device-owned state of a session after Reset (CoreSLAMProcessor.cs:167-175): the start pose, scan count 0
// (lastOdometryPose = 0, :173-174), no search or integration in flight.
void reset_session(CsSession& s, const float start_pose[3]) {
  memset(s.state, 0, sizeof(s.state));
  for (int k = 0; k < 3; k++) s.state[0].pose[k] = start_pose[k];  // :172
  s.key[0] = s.key[1] = ~0ull;
  s.search_done = 0;
  s.visits_slot[0] = s.visits_slot[1] = 0;
  s.ring_ticket[0] = s.ring_ticket[1] = 0;
  memset(s.ll_pose, 0, sizeof(s.ll_pose));
}

// Upper bound on the ring count of a scan: |rotated, scaled point| + half the hole width, plus rounding slack.
int rings_hint_of(int size, float scale, float hole_width, double max_range) {
  if (!(max_range == max_range) || max_range > 1e30) return size;
  double cells = max_range * (double)scale * 1.00001 + 0.5 * (double)hole_width * (double)scale + 4.0;
  if (cells >= (double)size) return size;
  return (int)cells + 1;
}
int rings_hint(const cs_processor* h, double max_range) { return rings_hint_of(h->size, h->scale, h->hs.hole_width, max_range); }

// Largest range of a scan (for the rings hint: an upper bound on the rings the scan can reach; NaN sticks, overflow gives
// +inf, both mean "all rings").  Four independent running maxima: a batch update calls this for every session on one host
// thread (1024 x 360 points per cfg5 step), where a single dependent chain cost as much as the staging copy itself.
double max_range_of(const float* points, int n) {
  float m0 = 0.f, m1 = 0.f, m2 = 0.f, m3 = 0.f;
  bool nan_seen = false;
  int i = 0;
  for (; i + 4 <= n; i += 4) {
    const float* p = points + 2 * (size_t)i;
    const float r0 = p[0] * p[0] + p[1] * p[1], r1 = p[2] * p[2] + p[3] * p[3];
    const float r2 = p[4] * p[4] + p[5] * p[5], r3 = p[6] * p[6] + p[7] * p[7];
    nan_seen |= (r0 != r0) | (r1 != r1) | (r2 != r2) | (r3 != r3);
    m0 = r0 > m0 ? r0 : m0;
    m1 = r1 > m1 ? r1 : m1;
    m2 = r2 > m2 ? r2 : m2;
    m3 = r3 > m3 ? r3 : m3;
  }
  for (; i < n; i++) {
    const float r = points[2 * i] * points[2 * i] + points[2 * i + 1] * points[2 * i + 1];
    nan_seen |= (r != r);
    m0 = r > m0 ? r : m0;
  }
  if (nan_seen) return std::numeric_limits<double>::quiet_NaN();
  const float m = std::fmax(std::fmax(m0, m1), std::fmax(m2, m3));
  return std::sqrt((double)m) * 1.000001;  // float rounding of r^2 (2^-24 relative) stays inside the bound
}

// The test hooks of the bounded polls (CS_FLAG_DEBUG_BOUNDED_SPIN), read from the environment once per process.
struct Tune {
  int spin_ms = 0, fault = 0;
  Tune() {
    auto geti = [](const char* name) { const char* v = getenv(name); return v ? atoi(v) : 0; };
    spin_ms = geti("CS_TUNE_SPIN_MS");  // milliseconds a device-side poll lasts (default 2000)
    fault = geti("CS_TUNE_FAULT");      // 1 = the draw kernel waits for a pose tag nobody publishes
  }
};
const Tune& tune() { static Tune t; return t; }

int device_sm_count(int device) {
  static int cache[64] = {0};
  if (device < 0 || device >= 64) return 148;
  if (!cache[device]) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || n <= 0) n = 148;
    cache[device] = n;
  }
  return cache[device];
}

// Warps (= candidates) per block of the search kernel.  All blocks of one scan are resident at once, and a
// warp's run time is fixed by the scan, so the kernel ends when the SM with the most warps ends: pick the
// block size whose busiest SM carries the fewest warps (4097 candidates on 148 SMs: 8 warps -> 4 blocks = 32
// warps on some SMs against 27.7 on average; 4 warps -> 7 blocks = 28).  Bigger blocks win ties (the scan is
// staged once per block).
int cs_search_warps(long long cand_count, int n_sessions, int num_sms) {
  const long long total = cand_count * (long long)n_sessions;
  if (total > (long long)num_sms * 40) return CS_SEARCH_WARPS;  // more than one wave anyway
  int best = CS_SEARCH_WARPS;
  long long best_cost = -1;
  for (int w = CS_SEARCH_WARPS; w >= 2; w >>= 1) {
    const long long blocks = ((cand_count + w - 1) / w) * n_sessions;
    const long long per_sm = (blocks + num_sms - 1) / num_sms;
    if (per_sm > 16) continue;  // keep the whole grid resident (shared memory: 16 x 16 KB)
    const long long cost = per_sm * w;
    if (best_cost < 0 || cost < best_cost) { best_cost = cost; best = w; }
  }
  return best;
}

// Slab search (cs_sort_kernel + cs_search2_kernel) instead of the warp-per-candidate kernel: one session alone whose
// candidate count fills the machine with slabs.  Block (c, s) = points [c*points, ...) x sorted candidates [s*threads, ...).
constexpr int kS2MinCand = 1024;
constexpr int kS2MinCandBatch = 256;
struct S2Plan {
  int points = 0, threads = 0, clusters = 0, slabs = 0;
};
int cs_s2_min_cand(uint32_t flags, int n_sessions = 1) {  // fewest candidates (searchPose included) the slab search is used for; 0 = never
  if (flags & CS_FLAG_SEARCH_WARP) return 0;
  if (flags & CS_FLAG_SEARCH_SLAB) return 1;
  // a batch fills the machine with its sessions; what the slabs need is enough candidates to amortise a block's set-up
  return n_sessions > 1 ? kS2MinCandBatch : kS2MinCand;
}
bool cs_plan_search2(int n_sessions, int s2_cap, int min_cand, long long cand_count, int n_points, int num_sms, S2Plan* p,
                     int max_threads = CS_S2_MAX_THREADS) {
  if (min_cand <= 0 || n_sessions < 1 || s2_cap <= 0 || cand_count > s2_cap || n_points < 1) return false;
  if (cand_count < min_cand) return false;
  if (n_sessions > 1 && (cand_count > CS_SORT_THREADS * CS_SORT_REG || n_sessions > 65535)) return false;  // batches: one sort block per session
  // the plan depends on (candidates, points, SMs) only: remember the last one (a replay asks for the same every scan)
  struct Memo { long long cand = -1; int points = -1, sms = -1, sessions = -1, max_threads = -1; bool ok = false; S2Plan plan; };
  static thread_local Memo memo;
  if (memo.cand == cand_count && memo.points == n_points && memo.sms == num_sms && memo.sessions == n_sessions && memo.max_threads == max_threads) {
    *p = memo.plan;
    return memo.ok;
  }
  memo.cand = cand_count; memo.points = n_points; memo.sms = num_sms; memo.sessions = n_sessions; memo.max_threads = max_threads; memo.ok = false;
  // Launch shape: the kernel is one resident wave of blocks (clusters x slabs) and ends when the busiest SM ends.  A lane
  // pays a fixed set-up (candidate pose, cos/sin: ~kSetup instruction slots) plus ~kLookup per point of its cluster, in
  // whole batches of CS_S2_BATCH; a block's cost is that times its warps, and an SM issues about kIpcPerWarp
  // instructions per clock and resident warp, up to kIpcMax.  Pick the (points, threads) pair with the shortest busiest SM.
  constexpr double kSetup = 450.0, kLookup = 26.0, kIpcPerWarp = 0.12, kIpcMax = 3.0;
  int best_points = 0, best_threads = 0;
  double best_cost = 0.0;
  for (int points = CS_S2_BATCH; points <= CS_S2_MAX_POINTS; points += 4) {
    const long long clusters = (n_points + points - 1) / points;
    if (clusters > CS_S2_MAX_CLUSTERS) continue;
    const int batches = ((int)((n_points + clusters - 1) / clusters) + CS_S2_BATCH - 1) / CS_S2_BATCH;  // of the fullest cluster
    for (int threads = max_threads; threads >= 64; threads -= 32) {  // bigger blocks win ties: one cluster's lines shared by more warps
      const long long slabs = (cand_count + threads - 1) / threads;
      if (slabs > 65535) continue;
      const long long blocks = clusters * slabs * n_sessions;
      const long long per_sm = (blocks + num_sms - 1) / num_sms;
      const double warps = (double)per_sm * (threads / 32);
      const double resident = warps < 48.0 ? warps : 48.0;
      const double ipc = resident * kIpcPerWarp < kIpcMax ? resident * kIpcPerWarp : kIpcMax;
      const double cost = warps * (kSetup + kLookup * CS_S2_BATCH * batches) / ipc;
      if (best_points == 0 || cost < best_cost * 0.999) { best_cost = cost; best_points = points; best_threads = threads; }
    }
  }
  if (best_points == 0) return false;
  const long long clusters = (n_points + best_points - 1) / best_points;
  const long long slabs = (cand_count + best_threads - 1) / best_threads;
  if (slabs > 65535 || clusters > CS_S2_MAX_CLUSTERS) return false;
  // even out: the same number of blocks with the smallest equal shares
  p->clusters = (int)clusters;
  p->points = (int)((n_points + clusters - 1) / clusters);
  p->slabs = (int)slabs;
  p->threads = (int)(((cand_count + slabs - 1) / slabs + 31) / 32 * 32);
  memo.plan = *p;
  memo.ok = true;
  return true;
}

// What a step is launched on: one processor (n_sessions = 1) or a batch of independent sessions
// (grid.y = n_sessions; every kernel indexes its session by blockIdx.y).
struct LaunchCtx {
  int s2_cap = 0;            // capacity of the slab-search scratch (0: none)
  int s2_min_cand = 0;       // cs_s2_min_cand of the handle
  Presort* presort = nullptr;  // one session alone: the sort queued ahead for the next scan, if any
  const float* next_cand = nullptr;  // cs_replay with tables: the next scan's table (nullptr: none) and the log's upload number
  uint64_t log_tag = 0;
  const CsSession* hs = nullptr;  // host mirror of the (first) session (host-owned constants for the slab kernels)
  int num_sms = 0;
  cudaStream_t stream = nullptr;
  CsSession* d_sess = nullptr;
  bool tiled = true;
  int n_sessions = 1;
  uint64_t* launches = nullptr;
  StepState* step = nullptr;  // step_counter, w_slot and s2_toggle advance with every launch
  long long* diag = nullptr;
  int diag_rings = 0;
  volatile unsigned* stuck_dev = nullptr;  // CS_FLAG_DEBUG_BOUNDED_SPIN: device address of the mapped-host word (CsSpin)
  unsigned long long* spec = nullptr;      // glue table of the handle (one session alone)
  cudaEvent_t ev_pose = nullptr;  // optional: recorded once the pose is out
  cudaEvent_t ev_done = nullptr;  // optional: recorded after the draw kernel

  // what a step of either handle is launched on; launch_step adds what only a processor has
  LaunchCtx(CsHost* h, uint32_t flags, int sessions, const CsSession* host_sessions)
      : s2_cap(h->s2_cap), s2_min_cand(cs_s2_min_cand(flags, sessions)), hs(host_sessions), num_sms(device_sm_count(h->device)),
        stream(h->stream), d_sess(h->d_sess.get()), tiled(h->tiled), n_sessions(sessions), launches(&h->launches), step(&h->step) {
    if (flags & CS_FLAG_DEBUG_BOUNDED_SPIN) stuck_dev = reinterpret_cast<volatile unsigned*>(h->d_stuck);
  }
};

enum { CS_PHASE_SEARCH = 1, CS_PHASE_FINISH = 2, CS_PHASE_ALL = 3 };

// One step on the stream: [search kernel, whose last block publishes the pose] or [set-up kernel] -> draw
// kernel (cs_wedge_kernel, whose first blocks prepare the rays).  Split phases (multi-GPU candidate split):
// SEARCH launches only the search over this GPU's candidate slice and leaves the packed arg-min in
// CsSession::key[parity]; FINISH — after the caller's 8-byte min exchange — launches the set-up kernel
// (which decodes the reduced key) and the draw kernel.
// Launch with the programmatic-stream-serialization attribute: the kernel may become resident while its
// predecessor in the stream drains; every kernel here calls cs_pdl_wait() before it reads anything the
// predecessor wrote.
// One-shot: the next launch_pdl on this thread is a plain (fully serialised) launch.  Set after a kernel that PRODUCES
// inputs of the step (cs_cloud_kernel writes the scan points): the step's first kernel reads its inputs before its
// dependency wait, which is only sound when they were complete before it could start.
thread_local bool g_next_launch_plain = false;

template <typename... KArgs, typename... Args>
cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args... args) {
  if (g_next_launch_plain) {
    g_next_launch_plain = false;
    kernel<<<grid, block, smem, stream>>>(args...);
    return cudaGetLastError();
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, args...);
}

// The candidate sort of a step (a.s2_* set): one block sorts a table of up to 8192 candidates out of its registers; generated
// (Philox) candidates are spread over the SMs, one per thread, as soon as there are more than one block's threads of them
// (batches: one block per session).  warm: one session alone with a tiled map — the sort grid's other blocks (or the
// histogram kernel's threads) pull the map within reach of the step into L2 beside the sort.
cudaError_t launch_sort(const LaunchCtx& c, CsStepArgs& a, bool warm) {
  cudaError_t e = cudaSuccess;
  warm = warm && c.n_sessions == 1 && c.tiled;
  const bool one_block = a.cand_count <= CS_SORT_THREADS * CS_SORT_REG &&
                         (a.cand_mode != CS_CAND_PHILOX || a.cand_count <= CS_SORT_THREADS || c.n_sessions > 1);
  if (warm) a.w_prefetch = 1;
  if (one_block) {
    e = launch_pdl(a.cand_mode == CS_CAND_PHILOX ? cs_sort_kernel<true> : cs_sort_kernel<false>,
                   dim3(warm ? 1u + (unsigned)c.num_sms : 1u, (unsigned)c.n_sessions), dim3(CS_SORT_THREADS), 0, c.stream, c.d_sess, a);
    if (e != cudaSuccess) return e;
    (*c.launches)++;
  } else {
    const unsigned sort_blocks = (unsigned)((a.cand_count + CS_SORT_MB_CHUNK - 1) / CS_SORT_MB_CHUNK);
    e = launch_pdl(a.cand_mode == CS_CAND_PHILOX ? cs_sort_hist_kernel<true> : cs_sort_hist_kernel<false>, dim3(sort_blocks),
                   dim3(CS_SORT_THREADS), 0, c.stream, c.d_sess, a);
    if (e != cudaSuccess) return e;
    e = launch_pdl(cs_sort_scatter_kernel, dim3(sort_blocks), dim3(CS_SORT_THREADS), 0, c.stream, c.d_sess, a);
    if (e != cudaSuccess) return e;
    (*c.launches) += 2;
  }
  return e;
}

cudaError_t launch_step_ctx(const LaunchCtx& c, CsStepArgs a, int n_points, int rings, int phases) {
  // An empty cloud (Update with segments that carry no rays): CalculateDistance returns int.MaxValue for every pose (:251-258),
  // so searchPose wins (:630-648, strict <) without a single lookup: no search kernel, the glue decodes (MaxValue, index 0).
  // (a.empty_cloud is set by the caller that knows the scan: stage_update.)
  const bool searching = (a.step_mode != CS_STEP_INTEGRATE_ONLY) && a.do_search && !a.empty_cloud;
  const bool draws = a.step_mode != CS_STEP_SEARCH_ONLY && n_points > 0;
  const bool fused = searching && phases == CS_PHASE_ALL;
  a.fuse_publish = fused ? 1 : 0;
  a.max_ring_hint = rings - 1;
  a.w_prefetch = 0;  // the map around the pose goes to L2 ahead of its use (one session alone; batches hide the latency)
  a.diag = c.diag;
  a.diag_rings = c.diag_rings;
  a.spec = (fused && draws && a.step_mode == CS_STEP_UPDATE) ? c.spec : nullptr;
  a.stuck_flag = c.stuck_dev;
  a.spin_ns = c.stuck_dev ? (long long)(tune().spin_ms > 0 ? tune().spin_ms : 2000) * 1000000ll : 0;
  if (phases & CS_PHASE_FINISH) {  // a call that publishes a pose takes the next step id: never 0, alternating parity
    if (++c.step->step_counter == 0) c.step->step_counter = 2;
    a.step_id = c.step->step_counter;
  }
  cudaError_t e = cudaSuccess;
  S2Plan s2;
  bool used_s2 = false;
  if ((phases & CS_PHASE_SEARCH) && searching &&
      cs_plan_search2(c.n_sessions, c.s2_cap, c.s2_min_cand, a.cand_count, a.s2_host_points, c.num_sms, &s2,
                      a.spec ? CS_S2_MAX_THREADS - 32 : CS_S2_MAX_THREADS)) {  // (the glue table's service warp rides along)
    used_s2 = true;
    a.s2_points = s2.points;
    a.s2_slab = s2.threads;
    a.s2_slot = (c.step->s2_toggle ^= 1);
    a.s2_batch = c.n_sessions > 1 ? 1 : 0;
    // (Measured and dropped: letting the candidate sort — the first kernel of the step, one block — prefetch the map around
    // the search pose: 65 k prefetches from one SM take 40 us.)
    a.s2_map = c.hs->map;
    a.s2_sorted = c.hs->s2_sorted + (size_t)a.s2_slot * c.hs->s2_cap;
    a.s2_tmp = c.hs->s2_tmp;
    a.s2_meta = c.hs->s2_meta;
    a.s2_acc = c.hs->s2_acc;
    a.s2_ghist = c.hs->s2_ghist;
    a.s2_seed = c.hs->seed;
    a.s2_size = c.hs->size;
    a.s2_pitch_tiles = c.hs->pitch_tiles;
    a.s2_scale = c.hs->scale;
    a.s2_sigma_xy = c.hs->sigma_xy;
    a.s2_sigma_theta = c.hs->sigma_theta;
    // (Measured and dropped: a warm-up kernel in front of the sort, one block per SM loading the map within reach of the step while
    // the one-block sort runs: one more link in the dependency chain costs more than the cold lookups — cfg2 41.8 -> 42.6 us.)
    const bool presorted = c.presort && c.presort->valid && !c.ev_done /* (CS_FLAG_TIMING measures the whole stage) */ && c.presort->cand_mode == a.cand_mode && c.presort->scan_index == a.scan_index &&
                           c.presort->cand_first == a.cand_first && c.presort->cand_count == a.cand_count && c.presort->slot == a.s2_slot &&
                           (a.cand_mode == CS_CAND_PHILOX || (a.cand_mode == CS_CAND_OFFSETS && c.presort->cand == a.cand && c.presort->tag == c.log_tag && c.log_tag != 0));
    if (c.presort) c.presort->valid = false;
    if (!presorted) {
      e = launch_sort(c, a, /*warm=*/true);
      if (e != cudaSuccess) return e;
    }
    dispatch_layout(c.tiled, [&](auto T) {
      e = launch_pdl(cs_search2_kernel<decltype(T)::value>, dim3((unsigned)s2.clusters, (unsigned)s2.slabs, (unsigned)c.n_sessions),
                     dim3(s2.threads + (a.spec ? 32 : 0)), 0, c.stream, c.d_sess, a);
    });
    if (e != cudaSuccess) return e;
    (*c.launches)++;
  } else if ((phases & CS_PHASE_SEARCH) && searching) {
    a.spec = nullptr;  // (the glue table is filled by the slab search's service warps)
    const int warps = cs_search_warps(a.cand_count, c.n_sessions, c.num_sms);
    dim3 grid((unsigned)((a.cand_count + warps - 1) / warps), (unsigned)c.n_sessions);
    int chunk = (n_points + 1) & ~1;  // even: the staging loop moves two points per 16-byte load
    if (chunk > CS_SEARCH_CHUNK) chunk = CS_SEARCH_CHUNK;
    if (chunk < 2) chunk = 2;
    a.search_chunk = chunk;
    dispatch_layout(c.tiled, [&](auto T) {
      e = launch_pdl(cs_search_kernel<decltype(T)::value>, grid, dim3(warps * 32), (size_t)chunk * sizeof(float2), c.stream,
                     c.d_sess, a);
    });
    if (e != cudaSuccess) return e;
    (*c.launches)++;
  }
  if (!(phases & CS_PHASE_FINISH)) return cudaGetLastError();
  if (!fused) {
    e = launch_pdl(cs_setup_kernel, dim3(1, (unsigned)c.n_sessions), dim3(CS_SETUP_THREADS), 0, c.stream, c.d_sess, a);
    if (e != cudaSuccess) return e;
    (*c.launches)++;
  }
  // the pose is out once this kernel has finished
  if (c.ev_pose) cudaEventRecord(c.ev_pose, c.stream);
  if (draws) {
    // The wedge kernel: (ring range x angular wedge) tasks, one warp each (cs_wedge.cuh).  The first blocks prepare the rays,
    // 128 each (big scans: bigger groups, so that at most 64 blocks prepare); every warp of the grid then takes tasks (small
    // scans: by block tickets; otherwise round-robin).  One session alone gets a resident wave — three blocks per SM of the
    // 80-register instance for a small scan, four of the 64-register one for a big scan — a session of a batch four blocks.
    int group = (((n_points + 63) / 64) + 31) / 32 * 32;
    if (group < 128) group = 128;
    if (group > CS_W_THREADS) group = CS_W_THREADS;  // one ray per thread of a preparing block
    a.prep_group = group;
    const int nprep = (n_points + group - 1) / group;
    // (one small scan alone: the 80-register instance, three blocks per SM; see cs_wedge_kernel)
    const bool latency = c.n_sessions == 1 && n_points <= 2048;
    int blocks = c.n_sessions == 1 ? (latency ? 3 : 4) * c.num_sms : 4;
    if (blocks < nprep) blocks = nprep;
    // A rank of a candidate-split group that shares its device with another rank (several handles of one process on one GPU)
    // must not keep a grid of polling blocks resident while its search kernel waits for the other ranks' keys — the ranks
    // would starve each other: its draw kernel starts after the search.  Ranks on devices of their own overlap as usual.
    if (a.xchg_world > 1 && a.xchg_serial_draw) g_next_launch_plain = true;
    {  // the counters rotate through three thirds: counted into now / counted into by the previous drawn step / zeroed now
      const int d = c.step->w_slot++;
      a.w_slot = d % 3;
      // The previous scan's counts size this scan's wedges (the table is then ready before the pose) where a scan is a latency
      // chain; a big scan is throughput, its wedges are narrow (a few degrees of heading change between scans would
      // overfill some) and it builds the table from its own counts.
      a.w_prev = (d > 0 && n_points <= 2048) ? (d + 2) % 3 : -1;
      a.w_zero = (d + 1) % 3;
      if (c.step->w_slot >= 3000) c.step->w_slot -= 2997;  // (keeps d > 0 and d mod 3)
    }
    if (a.w_prefetch == 0 && c.n_sessions == 1 && c.tiled) a.w_prefetch = 2;
    // (Measured and dropped: in batches, the preparing thread of a ray prefetching the tiles along it — cfg5 2.01 -> 2.08 ms
    // per step: the draw tasks of a batch already keep the memory system busy.)
    CsStepArgs draw_args = a;
    if (tune().fault == 1 && c.stuck_dev) draw_args.step_id ^= 0x40000000u;  // (fault injection: a pose tag nobody publishes)
    dispatch_layout(c.tiled, [&](auto T) {
      e = launch_pdl(latency ? cs_wedge_kernel<decltype(T)::value, 3> : cs_wedge_kernel<decltype(T)::value, 4>,
                     dim3((unsigned)blocks, (unsigned)c.n_sessions), dim3(CS_W_THREADS), 0, c.stream, c.d_sess, draw_args);
    });
    if (e != cudaSuccess) return e;
    (*c.launches)++;
  }
  // ---- production mode: the next scan's candidate sort, queued in the shadow of this scan's draw kernel (see Presort).  Not
  // under CS_FLAG_TIMING (the events around the stages would count it to the wrong one).
  const bool ahead_table = a.cand_mode == CS_CAND_OFFSETS && c.next_cand != nullptr && c.log_tag != 0 && !a.cand_cs;
  if (c.presort && used_s2 && fused && draws && (a.cand_mode == CS_CAND_PHILOX || ahead_table) && c.n_sessions == 1 &&
      !c.ev_done) {
    CsStepArgs b = a;
    if (ahead_table) b.cand = c.next_cand;
    b.scan_index = a.scan_index + 1;
    b.s2_slot = a.s2_slot ^ 1;
    b.s2_sorted = c.hs->s2_sorted + (size_t)b.s2_slot * c.hs->s2_cap;
    b.w_prefetch = 0;  // (the next scan's header is not known yet: its draw kernel's blocks warm the map themselves)
    e = launch_sort(c, b, /*warm=*/false);
    if (e != cudaSuccess) return e;
    c.presort->valid = true;
    c.presort->scan_index = b.scan_index;
    c.presort->cand_first = a.cand_first;
    c.presort->cand_count = a.cand_count;
    c.presort->slot = b.s2_slot;
    c.presort->cand_mode = a.cand_mode;
    c.presort->cand = ahead_table ? c.next_cand : nullptr;
    c.presort->tag = ahead_table ? c.log_tag : 0;
  }
  if (c.ev_done) cudaEventRecord(c.ev_done, c.stream);
  return cudaGetLastError();
}

// UpdateObstacleMap (CoreSLAMProcessor.cs:540-593) for n_sessions sessions: the ray kernel (hits + no-hit marks), then the
// sweep over the marked tiles.  Plain stream order: both follow the draw kernel of the same step.
cudaError_t launch_obstacle_update(cudaStream_t stream, const CsSession* d_sess, const CsObstacle* d_obst, const CsObstacle& ho,
                                   const CsStepArgs& a, int n_points, int n_sessions, int num_sms, uint64_t* launches) {
  const int warps = CS_OBST_RAY_THREADS / 32;
  int blocks = (n_points + warps - 1) / warps;
  if (blocks > num_sms * 8) blocks = num_sms * 8;
  if (blocks < 1) blocks = 1;
  cs_obstacle_rays_kernel<<<dim3((unsigned)blocks, (unsigned)n_sessions), CS_OBST_RAY_THREADS, 0, stream>>>(d_sess, d_obst, a);
  (*launches)++;
  const int n_words = ho.words_per_row * (ho.rows / 4);
  int sblocks = (n_words + 255) / 256;
  if (sblocks > num_sms * 8) sblocks = num_sms * 8;
  cs_obstacle_sweep_kernel<<<dim3((unsigned)sblocks, (unsigned)n_sessions), 256, 0, stream>>>(d_obst);
  (*launches)++;
  return cudaGetLastError();
}

// An ObstacleMap of `size` pixels per edge (ObstacleMap.cs:17-22, :103) without its buffers: rows padded to whole 8-cell
// words and the row count to whole 4-row tiles of the no-hit bitmap.
CsObstacle obstacle_geometry(int size, float physical_map_size) {
  CsObstacle o{};
  o.size = size;
  o.pitch = (size + 7) / 8 * 8;
  o.rows = (size + 3) / 4 * 4;
  o.words_per_row = o.pitch / 8;
  o.scale = (float)size / physical_map_size;  // ObstacleMap.cs:20
  o.max_hits = 10;                            // :103
  return o;
}
size_t obstacle_pixel_bytes(const CsObstacle& o) { return (size_t)o.pitch * o.rows; }
size_t obstacle_bitmap_words(const CsObstacle& o) { return (size_t)o.words_per_row * (o.rows / 4); }

// ArrayEx.Fill(ObstacleMap.Pixels, v) (:170) of n_sessions maps of the geometry `ho`: with `values`, session j's map gets
// values[j] (device array), otherwise every map gets `value`.
cudaError_t launch_obstacle_fill(cudaStream_t stream, const CsObstacle* d_obst, const int* values, int value, const CsObstacle& ho,
                                 int n_sessions, uint64_t* launches) {
  size_t blocks = (obstacle_pixel_bytes(ho) / 8 + 255) / 256;
  if (blocks > 148 * 2) blocks = 148 * 2;
  cs_obstacle_fill_kernel<<<dim3((unsigned)blocks, (unsigned)n_sessions), 256, 0, stream>>>(d_obst, values, value);
  (*launches)++;
  return cudaGetLastError();
}

// Pixels of one ObstacleMap out to `pixels` (Size * Size sbyte, [y, x]); returns once the copy is complete.
cs_status download_obstacle_map(CsHost* h, const CsObstacle& o, int8_t* pixels) {
  CS_CUDA(h, cudaMemcpy2DAsync(pixels, (size_t)o.size, o.pixels, (size_t)o.pitch, (size_t)o.size, (size_t)o.size,
                               cudaMemcpyDeviceToHost, h->stream));
  CS_CUDA(h, cudaStreamSynchronize(h->stream));
  return CS_OK;
}

cs_status launch_step(cs_processor* h, CsStepArgs a, int n_points, int rings, bool timing, int ev_base, int phases = CS_PHASE_ALL,
                      const float* next_cand = nullptr, uint64_t log_tag = 0) {
  LaunchCtx c(h, h->cfg.flags, 1, &h->hs);
  c.presort = &h->presort;
  c.next_cand = next_cand;
  c.log_tag = log_tag;
  c.spec = h->d_spec.get();
  c.diag = h->d_ring_cycles.get();
  c.diag_rings = h->size;
  a.hdr_stride = 1;
  const bool want_pose_event = timing || (a.seq_flag && (h->cfg.flags & CS_FLAG_NO_HOST_SPIN));
  c.ev_pose = (want_pose_event && (phases & CS_PHASE_FINISH)) ? h->tm.ev[ev_base + 0].get() : nullptr;
  c.ev_done = (timing && (phases & CS_PHASE_FINISH)) ? h->tm.ev[ev_base + 1].get() : nullptr;
  CS_CUDA(h, launch_step_ctx(c, a, n_points, rings, phases));
  if (h->d_obst && (phases & CS_PHASE_FINISH) && a.step_mode != CS_STEP_SEARCH_ONLY && n_points > 0) {
    // UpdateObstacleMap (:751) follows UpdateHoleMap (:750): same pose (CsSession::cur_pose), same cloud
    CS_CUDA(h, launch_obstacle_update(c.stream, h->d_sess.get(), h->d_obst.get(), h->ho, a, n_points, 1, c.num_sms, &h->launches));
  }
  if (c.ev_done) cudaEventRecord(h->tm.ev[ev_base + 2].get(), h->stream);
  CS_CUDA(h, cudaEventRecord(h->ev_stage_free[h->stage_cur].get(), h->stream));  // this step's readers of its staging buffer are enqueued
  return CS_OK;
}

// A handle that belongs to a candidate-split group evaluates its slice of the flat candidate indices and exchanges the
// arg-min inside the search kernel (cs_exchange_min); the exchange number advances with every searched scan, identically on
// every rank.
void apply_group(cs_processor* h, CsStepArgs& a) {
  if (h->group_world <= 1 || !a.do_search || a.empty_cloud) return;
  const long long n_flat = (long long)h->n_cand + 1;
  const long long lo = (long long)h->group_rank * n_flat / h->group_world, hi = (long long)(h->group_rank + 1) * n_flat / h->group_world;
  a.cand_first = (int)lo;
  a.cand_count = (int)(hi - lo);
  a.xchg_world = h->group_world;
  a.xchg_serial_draw = h->group_shares_device ? 1 : 0;
  a.xchg_rank = h->group_rank;
  a.xchg_seq = ++h->xchg_seq;
  for (int p = 0; p < h->group_world; p++) a.xchg_peer[p] = h->xchg_peer[p];
}

cs_status wait_for_pose(cs_processor* h, unsigned seq, cudaEvent_t fallback_event) {
  auto t0 = std::chrono::steady_clock::now();
  if (h->cfg.flags & CS_FLAG_NO_HOST_SPIN) {
    CS_CUDA(h, cudaEventSynchronize(fallback_event));
  } else {
    volatile unsigned* flag = reinterpret_cast<volatile unsigned*>(h->h_slot.get() + 64);
    unsigned spins = 0;
    while (*flag != seq) {
      if ((++spins & 0x3fff) == 0) {
        cudaError_t e = cudaStreamQuery(h->stream);
        if (e != cudaSuccess && e != cudaErrorNotReady)
          return fail(h, CS_ERR_CUDA, "stream error while waiting for the pose: %s", cudaGetErrorString(e));
        if (e == cudaSuccess && *flag != seq)
          return fail(h, CS_ERR_CUDA, "stream drained but the pose flag was never written");
      }
#if defined(__x86_64__)
      __builtin_ia32_pause();
#endif
    }
  }
  std::atomic_thread_fence(std::memory_order_acquire);
  auto t1 = std::chrono::steady_clock::now();
  h->last_timing.host_wait_ms = std::chrono::duration<double, std::milli>(t1 - t0).count();
  return CS_OK;
}

void copy_result(cs_result* out, const CsDevResult* r) {
  out->pose[0] = r->pose[0]; out->pose[1] = r->pose[1]; out->pose[2] = r->pose[2];
  out->distance = r->distance;
  out->index = r->index;
  out->searched = r->searched;
  out->visits = r->visits;
}

// The result records of an Update, for the caller: the visits are counted on the device while the integration runs
// (cs_get_visits after cs_sync), so they read -1 here.
void copy_update_results(cs_result* out, const CsDevResult* r, int n) {
  for (int j = 0; j < n; j++) {
    copy_result(out + j, r + j);
    out[j].visits = -1;
  }
}

// The arguments of an Update step (CoreSLAMProcessor.Update, :717-752) that follow from the handle's step state; the caller
// adds its inputs, outputs and strides.
CsStepArgs update_args(const CsHost& h, bool with_offsets, int n_points) {
  CsStepArgs a{};
  a.scan_index = h.step.update_count;
  a.cand_mode = with_offsets ? CS_CAND_OFFSETS : CS_CAND_PHILOX;
  a.step_mode = CS_STEP_UPDATE;
  a.parity = h.step.parity;
  a.do_search = h.step.searches() ? 1 : 0;
  a.n_cand = h.n_cand;
  a.cand_first = 0;
  a.cand_count = h.n_cand + 1;
  a.s2_host_points = n_points;
  return a;
}

cs_status ensure_linear(CsHost* h) {
  if (!h->d_linear) CS_CUDA(h, alloc(h->d_linear, (size_t)h->size * h->size));
  return CS_OK;
}

// A row-major copy of `map` in d_linear, queued on the handle's stream.
cs_status relayout_to_linear(CsHost* h, uint16_t* map) {
  cs_status st = ensure_linear(h);
  if (st != CS_OK) return st;
  dispatch_layout(h->tiled, [&](auto T) {
    cs_relayout_kernel<decltype(T)::value><<<148 * 8, 256, 0, h->stream>>>(map, h->d_linear.get(), h->size, h->pitch_tiles, 0);
  });
  h->launches++;
  return CS_OK;
}

// ... and copied out to `pixels` (size * size, row-major); returns once the copy is complete.
cs_status download_map(CsHost* h, uint16_t* map, uint16_t* pixels) {
  cs_status st = relayout_to_linear(h, map);
  if (st != CS_OK) return st;
  CS_CUDA(h, cudaMemcpyAsync(pixels, h->d_linear.get(), (size_t)h->size * h->size * 2, cudaMemcpyDeviceToHost, h->stream));
  CS_CUDA(h, cudaStreamSynchronize(h->stream));
  return CS_OK;
}

cs_status collect_timing(cs_processor* h, bool had_h2d) {
  CS_CUDA(h, cudaEventSynchronize(h->tm.ev[4].get()));
  float ms = 0;
  cs_timing& t = h->last_timing;
  if (had_h2d) { cudaEventElapsedTime(&ms, h->tm.ev[0].get(), h->tm.ev[1].get()); t.h2d_ms = ms; } else t.h2d_ms = 0;
  cudaEventElapsedTime(&ms, h->tm.ev[1].get(), h->tm.ev[2].get()); t.search_ms = ms;
  cudaEventElapsedTime(&ms, h->tm.ev[2].get(), h->tm.ev[3].get()); t.integrate_ms = ms;  // the draw kernel
  t.finalize_ms = 0.f;
  cudaEventElapsedTime(&ms, h->tm.ev[0].get(), h->tm.ev[4].get()); t.total_device_ms = ms;
  t.obstacle_ms = 0.f;
  if (h->d_obst) { cudaEventElapsedTime(&ms, h->tm.ev[3].get(), h->tm.ev[4].get()); t.obstacle_ms = ms; }
  return CS_OK;
}

bool finite3(const float* p) { return p[0] == p[0] && p[1] == p[1] && p[2] == p[2]; }

// What cs_create and cs_batch_create both require of a configuration (of a batch: of its first session's).  On success,
// the candidates per scan (T*I) and the point capacity.
cs_status check_config(const cs_config& cfg, long long* n_cand, int* max_points) {
  if (cfg.hole_map_size < 8 || cfg.hole_map_size > 16384)
    return fail(nullptr, CS_ERR_INVALID_ARGUMENT, "hole_map_size must be in [8, 16384], got %d", cfg.hole_map_size);
  if (!(cfg.physical_map_size > 0.f))
    return fail(nullptr, CS_ERR_INVALID_ARGUMENT, "physical_map_size must be positive");
  if (cfg.iterations_per_thread < 0) return fail(nullptr, CS_ERR_INVALID_ARGUMENT, "iterations_per_thread out of range");
  const int threads = cfg.num_search_threads > 0 ? cfg.num_search_threads : 1;
  *n_cand = (long long)threads * cfg.iterations_per_thread;
  if (*n_cand > (1ll << 26)) return fail(nullptr, CS_ERR_INVALID_ARGUMENT, "too many candidates per scan");
  *max_points = cfg.max_points > 0 ? cfg.max_points : 16384;
  if (*max_points > 65536) return fail(nullptr, CS_ERR_INVALID_ARGUMENT, "max_points must be <= 65536");
  if (cfg.obstacle_map_size < 0 || cfg.obstacle_map_size > 16384)
    return fail(nullptr, CS_ERR_INVALID_ARGUMENT, "obstacle_map_size must be 0 (no ObstacleMap) or in [1, 16384], got %d",
                cfg.obstacle_map_size);
  const int ndev = cs_device_count();
  if (ndev <= 0)
    return fail(nullptr, CS_ERR_NO_DEVICE, "no CUDA device: this library has no CPU path (cudaGetDeviceCount = 0)");
  if (cfg.device < 0 || cfg.device >= ndev)
    return fail(nullptr, CS_ERR_INVALID_ARGUMENT, "device %d out of range (have %d)", cfg.device, ndev);
  return CS_OK;
}

// The ray and wedge scratch of the n sessions sess[0..n) (CsSession::rays .. w_top), each session pointed at its slice:
// `copies` copies of ray_stride rays and of batch_stride batch maxima, and the wedge tables of ray_stride rays on a map of
// h.size.  The words a step expects zeroed are zeroed.
cudaError_t alloc_ray_scratch(CsHost& h, CsSession* sess, int n, int copies, int ray_stride, int batch_stride) {
  const size_t rays = (size_t)copies * ray_stride, maxima = (size_t)copies * batch_stride, prep = (size_t)2 * copies * 16;
  const size_t bkeys = (size_t)(ray_stride / 32 + 1), top = 3 * wedge_top_words(h.size);
  cudaError_t e = alloc(h.d_rays, rays * n);
  if (e == cudaSuccess) e = alloc(h.d_batch_max, maxima * n);
  if (e == cudaSuccess) e = alloc(h.d_prep_words, prep * n);
  if (e == cudaSuccess) e = cudaMemset(h.d_prep_words.get(), 0, prep * n * sizeof(unsigned long long));
  if (e == cudaSuccess) e = alloc(h.d_w_rk, (size_t)ray_stride * n);
  if (e == cudaSuccess) e = alloc(h.d_w_bkey, bkeys * n);
  if (e == cudaSuccess) e = alloc(h.d_w_top, top * n);
  if (e == cudaSuccess) e = cudaMemset(h.d_w_top.get(), 0, top * n * sizeof(int));
  if (e != cudaSuccess) return e;
  for (int j = 0; j < n; j++) {
    CsSession& s = sess[j];
    s.rays = h.d_rays.get() + j * rays;
    s.batch_max = h.d_batch_max.get() + j * maxima;
    s.ray_copies = copies;
    s.ray_stride = ray_stride;
    s.batch_stride = batch_stride;
    s.prep_words = h.d_prep_words.get() + j * prep;
    s.w_rk = h.d_w_rk.get() + (size_t)j * ray_stride;
    s.w_bkey = h.d_w_bkey.get() + j * bkeys;
    s.w_top = h.d_w_top.get() + j * top;
  }
  return cudaSuccess;
}

// n ObstacleMaps of `size` pixels per edge (:132-133): h.ho becomes their geometry, and desc[0..n) the host descriptors of
// the maps, each with its pieces of the pixel, no-hit bitmap and touched-counter blocks.  The device descriptor array
// d_obst is allocated; the caller uploads desc into it.
cudaError_t alloc_obstacle_maps(CsHost& h, CsObstacle* desc, int n, int size, float physical_map_size) {
  h.ho = obstacle_geometry(size, physical_map_size);
  const size_t px = obstacle_pixel_bytes(h.ho), words = obstacle_bitmap_words(h.ho);
  cudaError_t e = alloc(h.d_obst_pixels, px * n);
  if (e == cudaSuccess) e = alloc(h.d_obst_no_hit, words * n);
  if (e == cudaSuccess) e = alloc(h.d_obst_touched, (size_t)n);
  if (e == cudaSuccess) e = alloc(h.d_obst, (size_t)n);
  if (e != cudaSuccess) return e;
  for (int j = 0; j < n; j++) {
    CsObstacle& o = desc[j];
    o = h.ho;
    o.pixels = h.d_obst_pixels.get() + j * px;
    o.no_hit = h.d_obst_no_hit.get() + j * words;
    o.touched = h.d_obst_touched.get() + j;
  }
  return cudaSuccess;
}

}  // namespace

// =====================================================================================================
extern "C" {

int32_t cs_abi_version(void) { return CS_ABI_VERSION; }

const char* cs_last_error(const cs_processor* h) { return h ? h->error.c_str() : g_create_error.c_str(); }

int32_t cs_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

cs_status cs_create(const cs_config* cfg, cs_processor** out) {
  if (!cfg || !out) return fail(nullptr, CS_ERR_INVALID_ARGUMENT, "cs_create: null argument");
  *out = nullptr;
  if (cfg->iterations_per_thread > (1 << 24)) return fail(nullptr, CS_ERR_INVALID_ARGUMENT, "iterations_per_thread out of range");
  long long n_cand = 0;
  int max_points = 0;
  const cs_status cst = check_config(*cfg, &n_cand, &max_points);
  if (cst != CS_OK) return cst;

  cs_processor* h = new cs_processor();
  h->cfg = *cfg;
  h->device = cfg->device;
  h->tiled = !(cfg->flags & CS_FLAG_ROW_MAJOR_MAP);
  h->size = cfg->hole_map_size;
  h->pitch_tiles = (h->size + 7) / 8;
  h->max_points = max_points;
  h->n_cand = (int)n_cand;
  h->scale = (float)cfg->hole_map_size / cfg->physical_map_size;  // HoleMap.cs:20
  h->map_cells = h->tiled ? (size_t)h->pitch_tiles * h->pitch_tiles * 64 : (size_t)h->size * h->size;

  auto bail = [&](cs_status st) {
    g_create_error = h->error;
    cs_destroy(h);
    return st;
  };
  CS_CREATE_CUDA(h, cudaSetDevice(h->device));
  if (cfg->stream) {
    h->stream = (cudaStream_t)cfg->stream;
  } else {
    CS_CREATE_CUDA(h, create(h->own_stream));
    h->stream = h->own_stream.get();
  }
  CS_CREATE_CUDA(h, alloc(h->d_map, h->map_cells));
  CS_CREATE_CUDA(h, alloc(h->d_sess, 1));
  CsSession& s = h->hs;
  init_session(s, *h, *cfg, h->d_map.get());
  if (cfg->flags & CS_FLAG_DEBUG_RAYS) CS_CREATE_CUDA(h, alloc(h->d_ray_dbg, (size_t)max_points * 6));
  const int ray_stride = (max_points + 31) / 32 * 32;
  const int batch_stride = (ray_stride / 32 + 31) / 32 * 32;  // whole 128-byte lines per copy
  CS_CREATE_CUDA(h, alloc_ray_scratch(*h, &s, 1, kRayCopies, ray_stride, batch_stride));
  CS_CREATE_CUDA(h, alloc(h->d_spec, ((size_t)n_cand + 1) * 8));
  CS_CREATE_CUDA(h, cudaMemset(h->d_spec.get(), 0, ((size_t)n_cand + 1) * 8 * sizeof(unsigned long long)));  // (tag 0 is never a step's)
  CS_CREATE_CUDA(h, alloc(h->d_distances, (size_t)n_cand + 1));
  CS_CREATE_CUDA(h, alloc(h->d_checksum, 1));
  if (cs_s2_min_cand(cfg->flags) > 0 && n_cand + 1 >= cs_s2_min_cand(cfg->flags)) {
    h->s2_cap = (int)n_cand + 1;
    const size_t cap = (size_t)h->s2_cap;
    CS_CREATE_CUDA(h, alloc(h->d_s2_sorted, 2 * cap));
    CS_CREATE_CUDA(h, alloc(h->d_s2_tmp, cap));
    CS_CREATE_CUDA(h, alloc(h->d_s2_meta, cap));
    CS_CREATE_CUDA(h, alloc(h->d_s2_acc, cap));
    CS_CREATE_CUDA(h, cudaMemsetAsync(h->d_s2_acc.get(), 0, cap * sizeof(unsigned long long), h->stream));
    CS_CREATE_CUDA(h, alloc(h->d_s2_ghist, (size_t)CS_SORT_BINS + 1));
    CS_CREATE_CUDA(h, cudaMemsetAsync(h->d_s2_ghist.get(), 0, (size_t)(CS_SORT_BINS + 1) * sizeof(unsigned), h->stream));
  }
  h->stage_bytes = plan_stage(max_points, (int)n_cand, true).total + 16 * ((size_t)max_points + 1) + 64;  // + segment tables
  CS_CREATE_CUDA(h, alloc(h->d_cloud, (size_t)max_points));
  CS_CREATE_CUDA(h, alloc(h->h_stage, h->stage_bytes));
  CS_CREATE_CUDA(h, alloc(h->d_stage, h->stage_bytes));
  CS_CREATE_CUDA(h, alloc(h->d_stage_b, h->stage_bytes));
  CS_CREATE_CUDA(h, create(h->copy_stream));
  CS_CREATE_CUDA(h, create(h->ev_copy));
  for (Event& e : h->ev_stage_free) CS_CREATE_CUDA(h, create(e));
  CS_CREATE_CUDA(h, alloc(h->h_slot, 128, cudaHostAllocMapped));
  CS_CREATE_CUDA(h, cudaHostGetDevicePointer((void**)&h->d_slot, h->h_slot.get(), 0));
  memset(h->h_slot.get(), 0, 128);
  h->h_stuck = h->h_slot.get() + 96;
  h->d_stuck = h->d_slot + 96;
  for (Event& e : h->tm.ev) CS_CREATE_CUDA(h, create(e, cudaEventDefault));
  if (cfg->obstacle_map_size > 0) {  // :132-133
    CS_CREATE_CUDA(h, alloc_obstacle_maps(*h, &h->ho, 1, cfg->obstacle_map_size, cfg->physical_map_size));
    // (in stream order: the fill kernel of cs_reset below reads the descriptor on the handle's stream)
    CS_CREATE_CUDA(h, cudaMemcpyAsync(h->d_obst.get(), &h->ho, sizeof(CsObstacle), cudaMemcpyHostToDevice, h->stream));
  }

  // Optional L2 persistence window over the map (the gathers are served from L2 either way when the
  // map fits the 126 MB L2; the window only matters next to other L2-hungry work).
  {
    cudaDeviceProp prop;
    if ((cfg->flags & CS_FLAG_L2_PERSIST) && cudaGetDeviceProperties(&prop, h->device) == cudaSuccess &&
        prop.persistingL2CacheMaxSize > 0) {
      size_t bytes = h->map_cells * sizeof(uint16_t);
      size_t win = bytes < (size_t)prop.accessPolicyMaxWindowSize ? bytes : (size_t)prop.accessPolicyMaxWindowSize;
      size_t carve = win < (size_t)prop.persistingL2CacheMaxSize ? win : (size_t)prop.persistingL2CacheMaxSize;
      if (cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, carve) == cudaSuccess) {
        cudaStreamAttrValue attr{};
        attr.accessPolicyWindow.base_ptr = h->d_map.get();
        attr.accessPolicyWindow.num_bytes = win;
        attr.accessPolicyWindow.hitRatio = win <= carve ? 1.0f : (float)carve / (float)win;
        attr.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
        attr.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
        cudaStreamSetAttribute(h->stream, cudaStreamAttributeAccessPolicyWindow, &attr);
      }
      cudaGetLastError();
    }
  }

  s.s2_sorted = h->d_s2_sorted.get();
  s.s2_tmp = h->d_s2_tmp.get();
  s.s2_meta = h->d_s2_meta.get();
  s.s2_acc = h->d_s2_acc.get();
  s.s2_ghist = h->d_s2_ghist.get();
  s.s2_cap = h->s2_cap;
  s.ray_dbg = h->d_ray_dbg.get();
  s.distances = (cfg->flags & CS_FLAG_KEEP_DISTANCES) ? h->d_distances.get() : nullptr;
  cs_status st = cs_reset(h);
  if (st != CS_OK) return bail(st);
  *out = h;
  return CS_OK;
}

cs_status cs_destroy(cs_processor* h) {
  if (!h) return CS_OK;
  delete h;  // ~cs_processor drains the handle's streams; then every owner releases
  cudaGetLastError();
  return CS_OK;
}

cs_status cs_reset(cs_processor* h) {  // CoreSLAMProcessor.cs:167-175
  CS_CHECK_HANDLE(h);
  reset_session(h->hs, h->cfg.start_pose);
  h->step.parity = 0;
  h->step.scan_count = 0;
  h->step.update_count = 0;
  h->step.search_begin = h->hs.search_begin;
  cs_status st = push_session(h);
  if (st != CS_OK) return st;
  st = launch_fill(h, (uint16_t)((CS_TS_OBSTACLE + CS_TS_NO_OBSTACLE) / 2));  // :169
  if (st != CS_OK) return st;
  if (h->d_obst)  // :170 ArrayEx.Fill(ObstacleMap.Pixels, UnmappedObstacleHits)
    CS_CUDA(h, launch_obstacle_fill(h->stream, h->d_obst.get(), nullptr, h->unmapped_obstacle_hits, h->ho, 1, &h->launches));
  CS_CUDA(h, cudaStreamSynchronize(h->stream));
  return CS_OK;
}

// ---- ObstacleMap (CoreSLAM/ObstacleMap.cs; CoreSLAMProcessor.cs:53, :98, :103) --------------------------
#define CS_NEED_OBSTACLE(h)                                                                                  \
  do {                                                                                                       \
    if (!(h)->d_obst) return fail((h), CS_ERR_STATE, "the handle was created without an ObstacleMap (obstacle_map_size = 0)"); \
  } while (0)

cs_status cs_set_unmapped_obstacle_hits(cs_processor* h, int32_t hits) {
  CS_CHECK_HANDLE(h);
  if (hits < -128 || hits > 127) return fail(h, CS_ERR_INVALID_ARGUMENT, "UnmappedObstacleHits is an sbyte");
  h->unmapped_obstacle_hits = hits;  // takes effect at the next Reset, as in the reference (:96)
  return CS_OK;
}

cs_status cs_set_max_obstacle_hits(cs_processor* h, int32_t hits) {
  CS_CHECK_HANDLE(h);
  if (hits < -128 || hits > 127) return fail(h, CS_ERR_INVALID_ARGUMENT, "MaxObstacleHits is an sbyte");
  h->ho.max_hits = hits;
  if (!h->d_obst) return CS_OK;
  CS_CUDA(h, cudaMemcpyAsync(reinterpret_cast<uint8_t*>(h->d_obst.get()) + offsetof(CsObstacle, max_hits), &h->ho.max_hits, sizeof(int),
                             cudaMemcpyHostToDevice, h->stream));
  CS_CUDA(h, cudaStreamSynchronize(h->stream));
  return CS_OK;
}

cs_status cs_get_obstacle_map_info(const cs_processor* h, int32_t* size, float* scale) {
  if (!h) return CS_ERR_INVALID_ARGUMENT;
  if (size) *size = h->ho.size;
  if (scale) *scale = h->ho.scale;
  return CS_OK;
}

cs_status cs_obstacle_map_download(cs_processor* h, int8_t* pixels) {
  CS_CHECK_HANDLE(h);
  CS_NEED_OBSTACLE(h);
  if (!pixels) return fail(h, CS_ERR_INVALID_ARGUMENT, "null pixels");
  return download_obstacle_map(h, h->ho, pixels);
}

cs_status cs_obstacle_map_upload(cs_processor* h, const int8_t* pixels) {
  CS_CHECK_HANDLE(h);
  CS_NEED_OBSTACLE(h);
  if (!pixels) return fail(h, CS_ERR_INVALID_ARGUMENT, "null pixels");
  const CsObstacle& o = h->ho;
  CS_CUDA(h, cudaMemcpy2DAsync(o.pixels, (size_t)o.pitch, pixels, (size_t)o.size, (size_t)o.size, (size_t)o.size,
                               cudaMemcpyHostToDevice, h->stream));
  CS_CUDA(h, cudaStreamSynchronize(h->stream));
  return CS_OK;
}

cs_status cs_obstacle_map_fill(cs_processor* h, int32_t value) {
  CS_CHECK_HANDLE(h);
  CS_NEED_OBSTACLE(h);
  if (value < -128 || value > 127) return fail(h, CS_ERR_INVALID_ARGUMENT, "ObstacleMap pixels are sbyte");
  CS_CUDA(h, launch_obstacle_fill(h->stream, h->d_obst.get(), nullptr, value, h->ho, 1, &h->launches));
  return CS_OK;
}

cs_status cs_get_obstacle_visits(cs_processor* h, int64_t* touched) {
  CS_CHECK_HANDLE(h);
  CS_NEED_OBSTACLE(h);
  if (!touched) return fail(h, CS_ERR_INVALID_ARGUMENT, "null out");
  long long v = 0;
  CS_CUDA(h, cudaMemcpyAsync(&v, h->ho.touched, sizeof(v), cudaMemcpyDeviceToHost, h->stream));
  CS_CUDA(h, cudaStreamSynchronize(h->stream));
  *touched = v;
  return CS_OK;
}

cs_status cs_set_quality(cs_processor* h, int32_t quality) {
  CS_CHECK_HANDLE(h);
  if (quality < 1 || quality > 255) return fail(h, CS_ERR_INVALID_ARGUMENT, "Quality must be 1..255 (CoreSLAMProcessor.cs:76-82)");
  h->hs.quality = quality;
  return patch_session(h, offsetof(CsSession, quality), &h->hs.quality, sizeof(int));
}

cs_status cs_set_hole_width(cs_processor* h, float metres) {
  CS_CHECK_HANDLE(h);
  if (!(metres >= 0.f) || !(metres * h->scale < 60000.f))
    return fail(h, CS_ERR_INVALID_ARGUMENT, "HoleWidth*Scale must be in [0, 60000) cells");
  h->hs.hole_width = metres;
  return patch_session(h, offsetof(CsSession, hole_width), &h->hs.hole_width, sizeof(float));
}

cs_status cs_set_position_search_beginning(cs_processor* h, int32_t scans) {
  CS_CHECK_HANDLE(h);
  h->hs.search_begin = scans;
  h->step.search_begin = scans;
  return patch_session(h, offsetof(CsSession, search_begin), &h->hs.search_begin, sizeof(int));
}

cs_status cs_get_pose(cs_processor* h, float pose[3]) {
  CS_CHECK_HANDLE(h);
  if (!pose) return fail(h, CS_ERR_INVALID_ARGUMENT, "null pose");
  CsState st;
  CS_CUDA(h, cudaMemcpyAsync(&st, reinterpret_cast<uint8_t*>(h->d_sess.get()) + offsetof(CsSession, state) + h->step.parity * sizeof(CsState),
                             sizeof(CsState), cudaMemcpyDeviceToHost, h->stream));
  CS_CUDA(h, cudaStreamSynchronize(h->stream));
  pose[0] = st.pose[0]; pose[1] = st.pose[1]; pose[2] = st.pose[2];
  return CS_OK;
}

cs_status cs_set_pose(cs_processor* h, const float pose[3], const float last_odometry[3], int32_t scan_count) {
  CS_CHECK_HANDLE(h);
  if (!pose || !last_odometry) return fail(h, CS_ERR_INVALID_ARGUMENT, "null pose");
  CsState st{};
  for (int k = 0; k < 3; k++) { st.pose[k] = pose[k]; st.last_odo[k] = last_odometry[k]; }
  st.scan_count = scan_count;
  h->step.scan_count = scan_count;
  return patch_session(h, offsetof(CsSession, state) + h->step.parity * sizeof(CsState), &st, sizeof(CsState));
}

cs_status cs_get_map_info(const cs_processor* h, int32_t* size, float* scale) {
  if (!h) return CS_ERR_INVALID_ARGUMENT;
  if (size) *size = h->size;
  if (scale) *scale = h->scale;
  return CS_OK;
}

// -----------------------------------------------------------------------------------------------------
cs_status cs_search(cs_processor* h, const float* points, int32_t n_points, const float search_pose[3],
                    const float* cand_poses, const float* cand_cs, int32_t n_cand, uint32_t scan_index,
                    cs_result* best, int32_t* distances) {
  NvtxRange nvtx_range("cs_search");
  CS_CHECK_HANDLE(h);
  if (!points || !search_pose || !best || n_points <= 0) return fail(h, CS_ERR_INVALID_ARGUMENT, "cs_search: bad argument");
  if (n_points > h->max_points) return fail(h, CS_ERR_CAPACITY, "n_points %d > max_points %d", n_points, h->max_points);
  if (n_cand < 0 || n_cand > h->n_cand) return fail(h, CS_ERR_CAPACITY, "n_cand %d > T*I = %d", n_cand, h->n_cand);
  if (!cand_poses && n_cand != h->n_cand) return fail(h, CS_ERR_INVALID_ARGUMENT, "Philox mode evaluates exactly T*I candidates");

  StagePlan sp = plan_stage(n_points, n_cand, cand_cs != nullptr);
  h->stage_cur = 0;
  CsStepHeader* hdr = reinterpret_cast<CsStepHeader*>(h->h_stage.get());
  memset(hdr, 0, kHdrBytes);
  hdr->odo[0] = search_pose[0]; hdr->odo[1] = search_pose[1]; hdr->odo[2] = search_pose[2];
  hdr->n_points = n_points;
  memcpy(h->h_stage.get() + sp.off_points, points, (size_t)n_points * 8);
  if (cand_poses) memcpy(h->h_stage.get() + sp.off_cand, cand_poses, (size_t)n_cand * 12);
  if (cand_cs) memcpy(h->h_stage.get() + sp.off_cs, cand_cs, (size_t)(n_cand + 1) * 8);
  CS_CUDA(h, cudaMemcpyAsync(h->d_stage.get(), h->h_stage.get(), sp.total, cudaMemcpyHostToDevice, h->stream));

  // distances requested: point the session at the buffer for this call
  int* dist_ptr = distances ? h->d_distances.get() : h->hs.distances;
  if (dist_ptr != h->hs.distances) {
    CS_CUDA(h, cudaMemcpyAsync(reinterpret_cast<uint8_t*>(h->d_sess.get()) + offsetof(CsSession, distances), &dist_ptr,
                               sizeof(int*), cudaMemcpyHostToDevice, h->stream));
  }

  CsStepArgs a{};
  a.hdr = reinterpret_cast<const CsStepHeader*>(h->d_stage.get());
  a.points = reinterpret_cast<const float2*>(h->d_stage.get() + sp.off_points);
  a.cand = cand_poses ? reinterpret_cast<const float*>(h->d_stage.get() + sp.off_cand) : nullptr;
  a.cand_cs = cand_cs ? reinterpret_cast<const float*>(h->d_stage.get() + sp.off_cs) : nullptr;
  a.result = reinterpret_cast<CsDevResult*>(h->d_slot);
  a.seq_flag = reinterpret_cast<volatile unsigned*>(h->d_slot + 64);
  a.seq_value = ++h->seq;
  a.scan_index = scan_index;
  a.cand_mode = cand_poses ? CS_CAND_ABSOLUTE : CS_CAND_PHILOX;
  a.step_mode = CS_STEP_SEARCH_ONLY;
  a.parity = h->step.parity;
  a.do_search = 1;
  a.n_cand = n_cand;
  a.cand_first = 0;
  a.cand_count = n_cand + 1;
  a.s2_host_points = n_points;
  cs_status st = launch_step(h, a, 0, 0, false, 0);
  if (st != CS_OK) return st;
  if (distances) {
    CS_CUDA(h, cudaMemcpyAsync(distances, h->d_distances.get(), (size_t)(n_cand + 1) * sizeof(int), cudaMemcpyDeviceToHost,
                               h->stream));
    int* restore = h->hs.distances;
    CS_CUDA(h, cudaMemcpyAsync(reinterpret_cast<uint8_t*>(h->d_sess.get()) + offsetof(CsSession, distances), &restore,
                               sizeof(int*), cudaMemcpyHostToDevice, h->stream));
  }
  CS_CUDA(h, cudaStreamSynchronize(h->stream));
  copy_result(best, reinterpret_cast<const CsDevResult*>(h->h_slot.get()));
  best->visits = 0;
  return CS_OK;
}

// -----------------------------------------------------------------------------------------------------
// Relocalisation (no reference counterpart): the distance of every pose of a lattice (cs_lattice_kernel), then the k best
// window minima (select + merge kernels, see cs_lattice.cuh).  Reads the map as the stream leaves it; writes only its own
// scratch.

// The scans of a relocalisation: one scan (cs_relocalize, cs_relocalize_bounded) or a sequence of n_scans whose points
// are back to back, scan k owning [scan_first[k], scan_first[k+1]), with the odometry pose of each
// (cs_relocalize_sequence*; n_points is set from scan_first by check_relocalize).
struct RelocScans {
  bool seq;
  const float* points;
  int32_t n_points;
  const int32_t* scan_first;
  const float* odometry;
  int32_t n_scans;
};

// The argument checks of the relocalisation calls; *total: the poses of the lattice (counting stops past max_poses).
static cs_status check_relocalize(cs_processor* h, const char* name, RelocScans& sc, const cs_lattice* lattice,
                                  int32_t window, int32_t k, const cs_lattice_hit* hits, const int32_t* n_hits, long long max_poses,
                                  const char* max_name, long long* total) {
  const bool seq = sc.seq;
  if (!sc.points || !lattice || !hits || !n_hits || (!seq && sc.n_points <= 0)) return fail(h, CS_ERR_INVALID_ARGUMENT, "%s: bad argument", name);
  long long most = sc.n_points;  // points of the largest scan
  if (seq) {
    if (!sc.scan_first || !sc.odometry) return fail(h, CS_ERR_INVALID_ARGUMENT, "%s: bad argument", name);
    if (sc.n_scans < 1 || sc.n_scans > CS_SEQUENCE_MAX_SCANS)
      return fail(h, CS_ERR_INVALID_ARGUMENT, "%s: n_scans %d outside 1..%d", name, sc.n_scans, CS_SEQUENCE_MAX_SCANS);
    if (sc.scan_first[0] != 0) return fail(h, CS_ERR_INVALID_ARGUMENT, "%s: scan_first[0] = %d != 0", name, sc.scan_first[0]);
    most = 0;
    for (int s = 0; s < sc.n_scans; s++) {
      const long long n = (long long)sc.scan_first[s + 1] - sc.scan_first[s];
      if (n < 1) return fail(h, CS_ERR_INVALID_ARGUMENT, "%s: scan %d has %lld points", name, s, n);
      most = std::max(most, n);
    }
    for (int i = 0; i < 3 * sc.n_scans; i++)
      if (!std::isfinite(sc.odometry[i])) return fail(h, CS_ERR_INVALID_ARGUMENT, "%s: odometry[%d][%d] not finite", name, i / 3, i % 3);
  }
  if (window < 0) return fail(h, CS_ERR_INVALID_ARGUMENT, "%s: window %d < 0", name, window);
  if (k < 1 || k > CS_LATTICE_MAX_HITS)
    return fail(h, CS_ERR_INVALID_ARGUMENT, "%s: k %d outside 1..%d", name, k, CS_LATTICE_MAX_HITS);
  long long t = 1;
  for (int a = 0; a < 3; a++) {
    if (lattice->count[a] < 1) return fail(h, CS_ERR_INVALID_ARGUMENT, "%s: count[%d] = %d < 1", name, a, lattice->count[a]);
    if (!std::isfinite(lattice->origin[a])) return fail(h, CS_ERR_INVALID_ARGUMENT, "%s: origin[%d] not finite", name, a);
    if (lattice->count[a] > 1 && !(std::isfinite(lattice->step[a]) && lattice->step[a] > 0.f))
      return fail(h, CS_ERR_INVALID_ARGUMENT, "%s: step[%d] must be finite and > 0", name, a);
    t *= lattice->count[a];
    if (t > max_poses) break;
  }
  if (most > h->max_points) return fail(h, CS_ERR_CAPACITY, "n_points %lld > max_points %d", most, h->max_points);
  if (t > max_poses) return fail(h, CS_ERR_CAPACITY, "%s: more than %s = %lld poses", name, max_name, max_poses);
  if (seq) sc.n_points = sc.scan_first[sc.n_scans];
  // one scan sits at the lattice pose itself (its offset is +-0 and its heading change +0, which changes no cell): the
  // single-scan kernels give the same distances bit for bit, without the sequence's set-up
  if (seq && sc.n_scans == 1) sc.seq = false;
  *total = t;
  return CS_OK;
}

// The scans to the device: a single scan to d_lat_points, a sequence to d_seq_points with its records in d_seq_scans
// (cs_seq_offsets_kernel).  Sets the points and sequence fields of *a.
static cs_status upload_reloc_scans(cs_processor* h, const char* name, const RelocScans& sc, CsLatticeArgs* a) {
  const bool seq = sc.seq;
  {
    cudaError_t e = cudaSuccess;
    if (!seq && !h->d_lat_points) e = alloc(h->d_lat_points, (size_t)h->max_points);
    if (seq) {
      e = grow(h->d_seq_points, h->seq_points_cap, (size_t)sc.n_points);
      if (e == cudaSuccess && !h->d_seq_scans) e = alloc(h->d_seq_odometry, 3 * CS_SEQUENCE_MAX_SCANS);
      if (e == cudaSuccess && !h->d_seq_scans) e = alloc(h->d_seq_first, CS_SEQUENCE_MAX_SCANS + 1);
      if (e == cudaSuccess && !h->d_seq_scans) e = alloc(h->d_seq_scans, CS_SEQUENCE_MAX_SCANS);
    }
    if (e != cudaSuccess) {
      cudaGetLastError();  // (an allocation failure is not sticky: the handle stays usable)
      return fail(h, CS_ERR_OUT_OF_MEMORY, "%s: scratch allocation failed: %s", name, cudaGetErrorString(e));
    }
  }
  float2* points = seq ? h->d_seq_points.get() : h->d_lat_points.get();
  CS_CUDA(h, cudaMemcpyAsync(points, sc.points, (size_t)sc.n_points * sizeof(float2), cudaMemcpyHostToDevice, h->stream));
  a->points = points;
  a->n_points = sc.n_points;
  a->seq = CsSeqArgs{nullptr, sc.n_scans};
  if (seq) {
    CS_CUDA(h, cudaMemcpyAsync(h->d_seq_odometry.get(), sc.odometry, (size_t)sc.n_scans * 3 * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    CS_CUDA(h, cudaMemcpyAsync(h->d_seq_first.get(), sc.scan_first, (size_t)(sc.n_scans + 1) * sizeof(int), cudaMemcpyHostToDevice, h->stream));
    cs_seq_offsets_kernel<<<1, CS_SEQUENCE_MAX_SCANS, 0, h->stream>>>(h->d_seq_odometry.get(), h->d_seq_first.get(), sc.n_scans, h->d_seq_scans.get());
    h->launches++;
    CS_CUDA(h, cudaGetLastError());
    a->seq.scans = h->d_seq_scans.get();
  }
  return CS_OK;
}

// cs_lattice_kernel's arguments for the handle's map and the lattice (no scans or output set: upload_reloc_scans)
static CsLatticeArgs lattice_args(const cs_processor* h, const cs_lattice* lattice) {
  CsLatticeArgs a{};
  a.map = h->d_map.get();
  a.size = h->size;
  a.pitch_tiles = h->pitch_tiles;
  a.scale = h->scale;
  for (int q = 0; q < 3; q++) {
    a.origin[q] = lattice->origin[q];
    a.step[q] = lattice->count[q] > 1 ? lattice->step[q] : 0.f;  // (a single point sits at the origin whatever the step)
    a.count[q] = lattice->count[q];
  }
  a.tiles_x = (lattice->count[0] - 1) / CS_LAT_TILE_X + 1;
  a.tiles_y = (lattice->count[1] - 1) / CS_LAT_TILE_Y + 1;
  return a;
}

// n_lists sorted lists of k keys at `lists` -> one, by merge kernels ping-ponging with `other`; `lists` ends at the result
static cs_status merge_lattice_lists(cs_processor* h, unsigned long long*& lists, unsigned long long* other, int n_lists, int k) {
  for (; n_lists > 1; n_lists = (n_lists + CS_LAT_MERGE_LISTS - 1) / CS_LAT_MERGE_LISTS) {
    const unsigned blocks = (unsigned)((n_lists + CS_LAT_MERGE_LISTS - 1) / CS_LAT_MERGE_LISTS);
    cs_lattice_merge_kernel<<<blocks, CS_LAT_THREADS, 0, h->stream>>>(lists, n_lists, k, other);
    h->launches++;
    CS_CUDA(h, cudaGetLastError());
    std::swap(lists, other);
  }
  return CS_OK;
}

// the keys (distance << 32 | flat index, ~0 = none) of a merged list -> hits; returns how many
static int lattice_hits(const CsLatticeArgs& a, const unsigned long long* keys, int k, cs_lattice_hit* hits) {
  int n = 0;
  for (; n < k && keys[n] != ~0ull; n++) {
    const unsigned idx = (unsigned)keys[n];
    const unsigned c0 = (unsigned)a.count[0], c1 = (unsigned)a.count[1];
    const int ix = (int)(idx % c0), iy = (int)(idx / c0 % c1), it = (int)(idx / (c0 * c1));
    hits[n].pose[0] = cs_lattice_coord(a.origin[0], a.step[0], ix);
    hits[n].pose[1] = cs_lattice_coord(a.origin[1], a.step[1], iy);
    hits[n].pose[2] = cs_lattice_coord(a.origin[2], a.step[2], it);
    hits[n].distance = (int32_t)(keys[n] >> 32);
    hits[n].index = (int32_t)idx;
  }
  return n;
}

// select-kernel blocks over n poses, and the keys of their lists plus the merge kernels' first output
static int lattice_sel_blocks(long long n) { return (int)((n + CS_LAT_THREADS * CS_LAT_SEL_PER - 1) / (CS_LAT_THREADS * CS_LAT_SEL_PER)); }
static size_t lattice_list_keys(int sel_blocks, int k) {
  return (size_t)sel_blocks * k + (size_t)((sel_blocks + CS_LAT_MERGE_LISTS - 1) / CS_LAT_MERGE_LISTS) * k;
}

// The exhaustive search of cs_relocalize and cs_relocalize_sequence
static cs_status relocalize(cs_processor* h, const char* name, RelocScans sc, const cs_lattice* lattice, int32_t window, int32_t k,
                            cs_lattice_hit* hits, int32_t* n_hits, int32_t* distances) {
  CS_CHECK_HANDLE(h);
  long long total = 0;
  if (cs_status st = check_relocalize(h, name, sc, lattice, window, k, hits, n_hits, CS_LATTICE_MAX_POSES, "CS_LATTICE_MAX_POSES", &total))
    return st;

  const int c0 = lattice->count[0], c1 = lattice->count[1], c2 = lattice->count[2];
  const int sel_blocks = lattice_sel_blocks(total);
  const size_t list_keys = (size_t)sel_blocks * k;
  {
    cudaError_t e = grow(h->d_lat_volume, h->lat_volume_cap, (size_t)total);
    if (e == cudaSuccess) e = grow(h->d_lat_lists, h->lat_lists_cap, lattice_list_keys(sel_blocks, k));
    if (e != cudaSuccess) {
      cudaGetLastError();  // (an allocation failure is not sticky: the handle stays usable)
      return fail(h, CS_ERR_OUT_OF_MEMORY, "%s: scratch allocation failed: %s", name, cudaGetErrorString(e));
    }
  }
  CsLatticeArgs a = lattice_args(h, lattice);
  if (cs_status st = upload_reloc_scans(h, name, sc, &a)) return st;
  a.volume = h->d_lat_volume.get();
  const unsigned lat_blocks = (unsigned)((long long)a.tiles_x * a.tiles_y * c2);
  dispatch_layout(h->tiled, [&](auto T) {
    if (sc.seq) cs_lattice_kernel<decltype(T)::value, false, true><<<lat_blocks, CS_LAT_THREADS, 0, h->stream>>>(a);
    else cs_lattice_kernel<decltype(T)::value><<<lat_blocks, CS_LAT_THREADS, 0, h->stream>>>(a);
  });
  h->launches++;
  CS_CUDA(h, cudaGetLastError());

  unsigned long long* lists = h->d_lat_lists.get();
  const int win = std::min(window, std::max(c0, std::max(c1, c2)));  // (a wider box is the whole lattice; keeps ix + win in range)
  cs_lattice_select_kernel<<<(unsigned)sel_blocks, CS_LAT_THREADS, 0, h->stream>>>(a.volume, c0, c1, c2, win, k, lists);
  h->launches++;
  CS_CUDA(h, cudaGetLastError());
  if (cs_status st = merge_lattice_lists(h, lists, lists + list_keys, sel_blocks, k)) return st;

  unsigned long long keys[CS_LATTICE_MAX_HITS];
  CS_CUDA(h, cudaMemcpyAsync(keys, lists, (size_t)k * sizeof(unsigned long long), cudaMemcpyDeviceToHost, h->stream));
  if (distances)
    CS_CUDA(h, cudaMemcpyAsync(distances, a.volume, (size_t)total * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
  CS_CUDA(h, cudaStreamSynchronize(h->stream));
  *n_hits = lattice_hits(a, keys, k, hits);
  return CS_OK;
}

cs_status cs_relocalize(cs_processor* h, const float* points, int32_t n_points, const cs_lattice* lattice, int32_t window,
                        int32_t k, cs_lattice_hit* hits, int32_t* n_hits, int32_t* distances) {
  NvtxRange nvtx_range("cs_relocalize");
  return relocalize(h, "cs_relocalize", RelocScans{false, points, n_points, nullptr, nullptr, 0}, lattice, window, k, hits, n_hits, distances);
}

cs_status cs_relocalize_sequence(cs_processor* h, const float* points, const int32_t* scan_first, const float* odometry,
                                 int32_t n_scans, const cs_lattice* lattice, int32_t window, int32_t k, cs_lattice_hit* hits,
                                 int32_t* n_hits, int32_t* distances) {
  NvtxRange nvtx_range("cs_relocalize_sequence");
  return relocalize(h, "cs_relocalize_sequence", RelocScans{true, points, 0, scan_first, odometry, n_scans}, lattice, window, k, hits, n_hits,
                    distances);
}

// Branch and bound over the lattice (cs_bnb.cuh, DESIGN section 4): min-window grids of the map, U from one exact pose
// per top-level node, then per pass a descent from the top level (nodes of up to 128 x 128 poses) to the 16 x 8 patches
// of 32 x 32 tiles, the exact distances of the surviving tiles and the window test over them.  The host reads the
// survivors' count after each level (the next launch's size).  Serves cs_relocalize_bounded and
// cs_relocalize_sequence_bounded.
static cs_status relocalize_bounded(cs_processor* h, const char* name, RelocScans sc, const cs_lattice* lattice, int32_t window,
                                    int32_t k, cs_lattice_hit* hits, int32_t* n_hits, cs_relocalize_stats* stats) {
  CS_CHECK_HANDLE(h);
  long long total = 0;
  if (cs_status st = check_relocalize(h, name, sc, lattice, window, k, hits, n_hits, CS_LATTICE_MAX_POSES_BOUNDED,
                                      "CS_LATTICE_MAX_POSES_BOUNDED", &total))
    return st;

  const int c0 = lattice->count[0], c1 = lattice->count[1], c2 = lattice->count[2];
  CsLatticeArgs a = lattice_args(h, lattice);
  if (c0 > (1 << 30) || c1 > (1 << 30))  // (the last tile's indices must stay ints)
    return fail(h, CS_ERR_CAPACITY, "%s: count[0] = %d or count[1] = %d > 2^30", name, c0, c1);
  const long long n_tiles = (long long)a.tiles_x * a.tiles_y * c2;
  if (n_tiles > (1ll << 28))
    return fail(h, CS_ERR_CAPACITY, "%s: %lld tiles of 32 x 32 poses > 2^28 (count[0], count[1] too small for %d headings)",
                name, n_tiles, c2);
  // top level: the smallest power-of-two node (32 .. 128 poses a side) that covers the lattice's x and y, or 128
  int top = CS_BNB_LEAF_LEVEL;
  while (top < 7 && (c0 > (1 << top) || c1 > (1 << top))) top++;
  const int top_x = ((c0 - 1) >> top) + 1, top_y = ((c1 - 1) >> top) + 1;
  const long long n_top = (long long)top_x * top_y * c2;
  // grids G_0 .. G_max_grid: windows as wide as the cell span of the top level's children (wider spans bound by 0)
  const double span = (double)((1 << (top - 1)) - 1) * std::max(a.step[0], a.step[1]) * h->scale + 2.0;
  int max_grid = 0;
  while (max_grid < CS_BNB_MAX_GRID && (double)(1 << max_grid) < span + 1.0) max_grid++;
  const size_t cells = (size_t)h->size * h->size;
  const size_t node_cap = (size_t)std::min<long long>(n_tiles, CS_LATTICE_BOUNDED_MAX_NODES);
  const int seed_blocks = lattice_sel_blocks(n_top);
  {
    cudaError_t e = h->d_bnb_counters ? cudaSuccess : alloc(h->d_bnb_counters, 4);
    if (e == cudaSuccess) e = grow(h->d_bnb_grids, h->bnb_grids_cap, (size_t)(max_grid + 1) * cells);
    if (e == cudaSuccess) e = grow(h->d_bnb_seeds, h->bnb_seeds_cap, (size_t)n_top);
    if (e == cudaSuccess) e = grow(h->d_bnb_nodes, h->bnb_nodes_cap, 2 * node_cap);
    if (e == cudaSuccess) e = grow(h->d_bnb_slot, h->bnb_slot_cap, (size_t)n_tiles);
    if (e == cudaSuccess) e = grow(h->d_lat_lists, h->lat_lists_cap, lattice_list_keys(seed_blocks, k));
    if (e != cudaSuccess) {
      cudaGetLastError();  // (an allocation failure is not sticky: the handle stays usable)
      return fail(h, CS_ERR_OUT_OF_MEMORY, "%s: scratch allocation failed: %s", name, cudaGetErrorString(e));
    }
  }
  if (cs_status st = upload_reloc_scans(h, name, sc, &a)) return st;

  // the grids, rebuilt from the map as the stream leaves it
  uint16_t* grids = h->d_bnb_grids.get();
  const unsigned grid_blocks = (unsigned)std::min<size_t>((cells + CS_LAT_THREADS - 1) / CS_LAT_THREADS, 148 * 8);
  dispatch_layout(h->tiled, [&](auto T) {
    cs_bnb_grid0_kernel<decltype(T)::value><<<grid_blocks, CS_LAT_THREADS, 0, h->stream>>>(h->d_map.get(), h->size, h->pitch_tiles, grids);
  });
  h->launches++;
  CS_CUDA(h, cudaGetLastError());
  for (int j = 1; j <= max_grid; j++) {
    cs_bnb_grid_kernel<<<grid_blocks, CS_LAT_THREADS, 0, h->stream>>>(grids + (j - 1) * cells, h->size, 1 << (j - 1), grids + j * cells);
    h->launches++;
    CS_CUDA(h, cudaGetLastError());
  }

  CsBnbArgs b{};
  b.grids = grids;
  b.size = h->size;
  b.max_grid = max_grid;
  b.scale = h->scale;
  b.points = a.points;
  b.n_points = a.n_points;
  for (int q = 0; q < 3; q++) b.origin[q] = a.origin[q], b.step[q] = a.step[q], b.count[q] = a.count[q];
  b.top_x = top_x;
  b.top_y = top_y;
  b.counters = h->d_bnb_counters.get();

  // first U: the k-th smallest exact distance of the top-level nodes' first poses (INT32_MAX - 1 when fewer than k are finite)
  unsigned long long keys[CS_LATTICE_MAX_HITS];
  {
    b.level = top;
    (sc.seq ? cs_bnb_seed_kernel<true> : cs_bnb_seed_kernel<false>)<<<(unsigned)n_top, CS_LAT_THREADS, 0, h->stream>>>(b, h->d_bnb_seeds.get(), a.seq);
    h->launches++;
    CS_CUDA(h, cudaGetLastError());
    unsigned long long* lists = h->d_lat_lists.get();
    cs_lattice_select_kernel<<<(unsigned)seed_blocks, CS_LAT_THREADS, 0, h->stream>>>(h->d_bnb_seeds.get(), (int)n_top, 1, 1, 0, k, lists);
    h->launches++;
    CS_CUDA(h, cudaGetLastError());
    if (cs_status st = merge_lattice_lists(h, lists, lists + (size_t)seed_blocks * k, seed_blocks, k)) return st;
    CS_CUDA(h, cudaMemcpyAsync(keys, lists, (size_t)k * sizeof(unsigned long long), cudaMemcpyDeviceToHost, h->stream));
    CS_CUDA(h, cudaStreamSynchronize(h->stream));
  }
  const int kMaxU = 2147483646;
  int upper = keys[k - 1] != ~0ull ? (int)(keys[k - 1] >> 32) : kMaxU;

  const int win = std::min(window, std::max(c0, std::max(c1, c2)));  // (as cs_relocalize)
  cs_relocalize_stats st{};
  st.poses = total;
  st.levels = top - CS_BNB_LEAF_LEVEL + 1;
  int4* node_buf[2] = {h->d_bnb_nodes.get(), h->d_bnb_nodes.get() + node_cap};
  unsigned long long counters[4];
  for (;;) {
    st.passes++;
    st.upper_bound = upper;
    b.upper = upper;
    // descent: level `top` (every node of the lattice) down to the tiles
    b.in = nullptr;
    long long n_in = n_top, n_leaves = 0;
    for (int level = top, flip = 0; n_in > 0; level--, flip ^= 1) {
      CS_CUDA(h, cudaMemsetAsync(b.counters, 0, 4 * sizeof(unsigned long long), h->stream));
      b.level = level;
      b.out = node_buf[flip];
      b.out_cap = (int)node_cap;
      const bool leaf = level == CS_BNB_LEAF_LEVEL;
      if (sc.seq) (leaf ? cs_bnb_bound_kernel<true, true> : cs_bnb_bound_kernel<false, true>)<<<(unsigned)n_in, CS_LAT_THREADS, 0, h->stream>>>(b, a.seq);
      else (leaf ? cs_bnb_bound_kernel<true> : cs_bnb_bound_kernel<false>)<<<(unsigned)n_in, CS_LAT_THREADS, 0, h->stream>>>(b, a.seq);
      h->launches++;
      CS_CUDA(h, cudaGetLastError());
      CS_CUDA(h, cudaMemcpyAsync(counters, b.counters, 3 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, h->stream));
      CS_CUDA(h, cudaStreamSynchronize(h->stream));
      st.bounded += (int64_t)counters[1];
      st.evaluated += (int64_t)counters[2];
      if (counters[0] > node_cap)
        return fail(h, CS_ERR_CAPACITY, "%s: %llu nodes of %d x %d poses survive, more than CS_LATTICE_BOUNDED_MAX_NODES = %d",
                    name, counters[0], 1 << (level - 1), 1 << (level - 1), CS_LATTICE_BOUNDED_MAX_NODES);
      n_in = (long long)counters[0];
      b.in = node_buf[flip];
      if (level == CS_BNB_LEAF_LEVEL) {
        n_leaves = n_in;
        break;
      }
    }

    // the surviving tiles' exact distances, the window test over them and the k best
    unsigned long long passed = 0;
    if (n_leaves == 0) {
      for (int i = 0; i < k; i++) keys[i] = ~0ull;
    } else {
      const int sel_blocks = lattice_sel_blocks(n_leaves * CS_LAT_TILE_X * CS_LAT_TILE_Y);
      {
        cudaError_t e = grow(h->d_lat_volume, h->lat_volume_cap, (size_t)n_leaves * CS_LAT_TILE_X * CS_LAT_TILE_Y);
        if (e == cudaSuccess) e = grow(h->d_lat_lists, h->lat_lists_cap, lattice_list_keys(sel_blocks, k));
        if (e != cudaSuccess) {
          cudaGetLastError();
          return fail(h, CS_ERR_OUT_OF_MEMORY, "%s: scratch allocation failed: %s", name, cudaGetErrorString(e));
        }
      }
      CS_CUDA(h, cudaMemsetAsync(h->d_bnb_slot.get(), 0xff, (size_t)n_tiles * sizeof(int), h->stream));
      CS_CUDA(h, cudaMemsetAsync(b.counters, 0, 4 * sizeof(unsigned long long), h->stream));
      a.volume = h->d_lat_volume.get();
      a.tiles = b.in;
      a.tile_slot = h->d_bnb_slot.get();
      dispatch_layout(h->tiled, [&](auto T) {
        if (sc.seq) cs_lattice_kernel<decltype(T)::value, true, true><<<(unsigned)n_leaves, CS_LAT_THREADS, 0, h->stream>>>(a);
        else cs_lattice_kernel<decltype(T)::value, true><<<(unsigned)n_leaves, CS_LAT_THREADS, 0, h->stream>>>(a);
      });
      h->launches++;
      CS_CUDA(h, cudaGetLastError());
      unsigned long long* lists = h->d_lat_lists.get();
      cs_lattice_select_tiles_kernel<<<(unsigned)sel_blocks, CS_LAT_THREADS, 0, h->stream>>>(
          a.volume, a.tiles, a.tile_slot, (int)n_leaves, c0, c1, c2, a.tiles_x, a.tiles_y, win, k, upper, b.counters + 3, lists);
      h->launches++;
      CS_CUDA(h, cudaGetLastError());
      if (cs_status s = merge_lattice_lists(h, lists, lists + (size_t)sel_blocks * k, sel_blocks, k)) return s;
      CS_CUDA(h, cudaMemcpyAsync(keys, lists, (size_t)k * sizeof(unsigned long long), cudaMemcpyDeviceToHost, h->stream));
      CS_CUDA(h, cudaMemcpyAsync(&passed, b.counters + 3, sizeof(unsigned long long), cudaMemcpyDeviceToHost, h->stream));
      CS_CUDA(h, cudaStreamSynchronize(h->stream));
    }
    // k true minima with distance <= U are the k best of the lattice; at U = INT32_MAX - 1 nothing finite was pruned
    if (passed >= (unsigned long long)k || upper == kMaxU) break;
    // else the k-th candidate found (distance > U) as the next U, and after three passes the last resort
    upper = (keys[k - 1] != ~0ull && st.passes < 3) ? std::max(upper + 1, (int)(keys[k - 1] >> 32)) : kMaxU;
  }
  *n_hits = lattice_hits(a, keys, k, hits);
  if (stats) *stats = st;
  return CS_OK;
}

cs_status cs_relocalize_bounded(cs_processor* h, const float* points, int32_t n_points, const cs_lattice* lattice,
                                int32_t window, int32_t k, cs_lattice_hit* hits, int32_t* n_hits, cs_relocalize_stats* stats) {
  NvtxRange nvtx_range("cs_relocalize_bounded");
  return relocalize_bounded(h, "cs_relocalize_bounded", RelocScans{false, points, n_points, nullptr, nullptr, 0}, lattice, window, k,
                            hits, n_hits, stats);
}

cs_status cs_relocalize_sequence_bounded(cs_processor* h, const float* points, const int32_t* scan_first, const float* odometry,
                                         int32_t n_scans, const cs_lattice* lattice, int32_t window, int32_t k,
                                         cs_lattice_hit* hits, int32_t* n_hits, cs_relocalize_stats* stats) {
  NvtxRange nvtx_range("cs_relocalize_sequence_bounded");
  return relocalize_bounded(h, "cs_relocalize_sequence_bounded", RelocScans{true, points, 0, scan_first, odometry, n_scans}, lattice,
                            window, k, hits, n_hits, stats);
}

cs_status cs_integrate(cs_processor* h, const float* points, int32_t n_points, const float pose[3],
                       const float* pose_cs, int64_t* visits) {
  NvtxRange nvtx_range("cs_integrate");
  CS_CHECK_HANDLE(h);
  if (!points || !pose || n_points < 0) return fail(h, CS_ERR_INVALID_ARGUMENT, "cs_integrate: bad argument");
  if (n_points > h->max_points) return fail(h, CS_ERR_CAPACITY, "n_points %d > max_points %d", n_points, h->max_points);
  // No sync needed before refilling the pinned block: the previous call returned only after its pose
  // flag, which the device writes after that call's H2D copy completed; the device-side block is
  // protected by stream order.
  StagePlan sp = plan_stage(n_points, 0, false);
  h->stage_cur = 0;
  CsStepHeader* hdr = reinterpret_cast<CsStepHeader*>(h->h_stage.get());
  memset(hdr, 0, kHdrBytes);
  hdr->odo[0] = pose[0]; hdr->odo[1] = pose[1]; hdr->odo[2] = pose[2];
  hdr->n_points = n_points;
  if (pose_cs) { hdr->cs[0] = pose_cs[0]; hdr->cs[1] = pose_cs[1]; hdr->has_cs = 1; }
  memcpy(h->h_stage.get() + sp.off_points, points, (size_t)n_points * 8);
  CS_CUDA(h, cudaMemcpyAsync(h->d_stage.get(), h->h_stage.get(), sp.total, cudaMemcpyHostToDevice, h->stream));
  CsStepArgs a{};
  a.hdr = reinterpret_cast<const CsStepHeader*>(h->d_stage.get());
  a.points = reinterpret_cast<const float2*>(h->d_stage.get() + sp.off_points);
  a.result = reinterpret_cast<CsDevResult*>(h->d_slot);
  a.step_mode = CS_STEP_INTEGRATE_ONLY;
  a.parity = h->step.parity;
  cs_status st = launch_step(h, a, n_points, rings_hint(h, max_range_of(points, n_points)), false, 0);
  if (st != CS_OK) return st;
  if (visits) {
    long long v = 0;
    CS_CUDA(h, cudaMemcpyAsync(&v, reinterpret_cast<uint8_t*>(h->d_sess.get()) + offsetof(CsSession, visits_slot) + (h->step.step_counter & 1u) * sizeof(long long), sizeof(v),
                               cudaMemcpyDeviceToHost, h->stream));
    CS_CUDA(h, cudaStreamSynchronize(h->stream));
    *visits = v;
  }
  return CS_OK;
}

// Stages one scan and fills the step arguments of an Update; shared by cs_update and cs_update_begin.
// Raw scan segments of one Update (cs_update_segments): the cloud is computed on the device.
struct SegInput {
  const float* rays;        // n_points * (angle, radius)
  const int32_t* seg_first; // n_segments + 1
  const float* seg_poses;   // n_segments * 3
  int n_segments;
};

static cs_status launch_cloud(cs_processor* h, const uint8_t* d_rays, const uint8_t* d_first, const uint8_t* d_poses, int n_rays,
                              int n_segments, const float odo[3]) {
  cs_cloud_kernel<<<(n_rays + CS_CLOUD_THREADS - 1) / CS_CLOUD_THREADS, CS_CLOUD_THREADS, 0, h->stream>>>(
      reinterpret_cast<const float2*>(d_rays), reinterpret_cast<const int*>(d_first), reinterpret_cast<const float*>(d_poses),
      n_segments, n_rays, odo[0], odo[1], odo[2], h->d_cloud.get());
  h->launches++;
  CS_CUDA(h, cudaGetLastError());
  return CS_OK;
}

static cs_status check_segments(cs_processor* h, const float* rays, const int32_t* seg_first, const float* seg_poses, int32_t n_rays,
                                int32_t n_segments) {
  // n_rays == 0 is legal: segments whose Rays lists are empty still advance the processor state (:719-747, every distance
  // is int.MaxValue and searchPose wins); only a negative count or missing tables are argument errors
  if ((!rays && n_rays > 0) || !seg_first || !seg_poses || n_rays < 0) return fail(h, CS_ERR_INVALID_ARGUMENT, "segments: bad argument");
  if (n_segments <= 0) return fail(h, CS_ERR_INVALID_ARGUMENT, "Sequence contains no elements (segments.Last(), CoreSLAMProcessor.cs:719)");
  if (n_rays > h->max_points) return fail(h, CS_ERR_CAPACITY, "n_rays %d > max_points %d", n_rays, h->max_points);
  if (n_segments > h->max_points) return fail(h, CS_ERR_CAPACITY, "n_segments %d > max_points %d", n_segments, h->max_points);
  if (seg_first[0] != 0 || seg_first[n_segments] != n_rays) return fail(h, CS_ERR_INVALID_ARGUMENT, "seg_first must run from 0 to n_rays");
  for (int s = 0; s < n_segments; s++)
    if (seg_first[s + 1] < seg_first[s]) return fail(h, CS_ERR_INVALID_ARGUMENT, "seg_first must be non-decreasing");
  return CS_OK;
}

// upper bound of |point| over the cloud of the segments: |segment.Pose - odometry| + |radius|
static double max_range_of_segments(const float* rays, const int32_t* seg_first, const float* seg_poses, int n_segments, const float odo[3]) {
  double m = 0.0;
  bool nan_seen = false;  // a NaN radius or segment pose: "all rings" (rings_hint_of), whatever the other rays reach
  for (int s = 0; s < n_segments; s++) {
    const double dx = (double)seg_poses[3 * s] - odo[0], dy = (double)seg_poses[3 * s + 1] - odo[1];
    const double d0 = std::sqrt(dx * dx + dy * dy);
    for (int i = seg_first[s]; i < seg_first[s + 1]; i++) {
      const double r = d0 + std::fabs((double)rays[2 * i + 1]);
      if (r != r) nan_seen = true;
      else if (r > m) m = r;
    }
  }
  return nan_seen ? std::numeric_limits<double>::quiet_NaN() : m;
}

static cs_status stage_update(cs_processor* h, const float* points, int32_t n_points, const float odometry_pose[3],
                              const float* cand_offsets, bool timing, CsStepArgs* out_args, const SegInput* seg = nullptr,
                              bool split_phase = false) {
  if ((!points && !seg && n_points > 0) || !odometry_pose || n_points < 0) return fail(h, CS_ERR_INVALID_ARGUMENT, "cs_update: bad argument");
  if (n_points > h->max_points) return fail(h, CS_ERR_CAPACITY, "n_points %d > max_points %d", n_points, h->max_points);
  if (!finite3(odometry_pose)) return fail(h, CS_ERR_INVALID_ARGUMENT, "odometry pose is NaN");
  if (h->pending) return fail(h, CS_ERR_STATE, "a split-phase update is in flight: call cs_update_finish first");

  // The previous call's integration may still be running: the pinned block is free again (its H2D copy
  // finished before that call's pose flag), the device block is protected by stream order.
  const bool do_search = h->step.searches();
  const bool with_offsets = cand_offsets != nullptr && do_search;
  StagePlan sp = plan_stage(n_points, with_offsets ? h->n_cand : 0, false);
  CsStepHeader* hdr = reinterpret_cast<CsStepHeader*>(h->h_stage.get());
  memset(hdr, 0, kHdrBytes);
  hdr->odo[0] = odometry_pose[0]; hdr->odo[1] = odometry_pose[1]; hdr->odo[2] = odometry_pose[2];
  hdr->n_points = n_points;
  size_t off_first = 0, off_poses = 0;
  if (seg) {  // the points slot carries the raw rays; the segment tables go behind the candidate table
    if (n_points > 0) memcpy(h->h_stage.get() + sp.off_points, seg->rays, (size_t)n_points * 8);
    off_first = sp.total;
    off_poses = align_up(off_first + (size_t)(seg->n_segments + 1) * 4, 16);
    sp.total = align_up(off_poses + (size_t)seg->n_segments * 12, 16);
    memcpy(h->h_stage.get() + off_first, seg->seg_first, (size_t)(seg->n_segments + 1) * 4);
    memcpy(h->h_stage.get() + off_poses, seg->seg_poses, (size_t)seg->n_segments * 12);
  } else if (n_points > 0) {
    memcpy(h->h_stage.get() + sp.off_points, points, (size_t)n_points * 8);
  }
  if (with_offsets) memcpy(h->h_stage.get() + sp.off_cand, cand_offsets, (size_t)h->n_cand * 12);

  if (timing) cudaEventRecord(h->tm.ev[0].get(), h->stream);
  // run ahead of the stream: copy into the buffer the scan in flight is not reading, behind nothing but that buffer's
  // last readers (two scans ago); the main stream picks the copy up through its event
  h->stage_cur = (h->stage_flip ^= 1);
  uint8_t* d_base = h->stage_cur ? h->d_stage_b.get() : h->d_stage.get();
  CS_CUDA(h, cudaStreamWaitEvent(h->copy_stream.get(), h->ev_stage_free[h->stage_cur].get(), 0));
  CS_CUDA(h, cudaMemcpyAsync(d_base, h->h_stage.get(), sp.total, cudaMemcpyHostToDevice, h->copy_stream.get()));
  CS_CUDA(h, cudaEventRecord(h->ev_copy.get(), h->copy_stream.get()));
  CS_CUDA(h, cudaStreamWaitEvent(h->stream, h->ev_copy.get(), 0));
  if (seg && n_points > 0) {  // ScanSegmentsToCloud (:723) on the device; the step's first kernel must not start before it is complete
    cs_status cst = launch_cloud(h, d_base + sp.off_points, d_base + off_first, d_base + off_poses, n_points,
                                 seg->n_segments, odometry_pose);
    if (cst != CS_OK) return cst;
    g_next_launch_plain = true;
  }
  if (timing) cudaEventRecord(h->tm.ev[1].get(), h->stream);

  CsStepArgs a = update_args(*h, with_offsets, n_points);
  a.hdr = reinterpret_cast<const CsStepHeader*>(d_base);
  a.points = seg ? h->d_cloud.get() : reinterpret_cast<const float2*>(d_base + sp.off_points);
  a.cand = with_offsets ? reinterpret_cast<const float*>(d_base + sp.off_cand) : nullptr;
  a.result = reinterpret_cast<CsDevResult*>(h->d_slot);
  a.seq_flag = reinterpret_cast<volatile unsigned*>(h->d_slot + 64);
  a.seq_value = ++h->seq;
  a.empty_cloud = (do_search && n_points == 0) ? 1 : 0;
  if (!split_phase) apply_group(h, a);  // (cs_update_begin / _finish: the caller exchanges the key between the phases)
  *out_args = a;
  return CS_OK;
}

// Host-side bookkeeping after an Update has been enqueued, the wait for the pose, and the result copy.
static cs_status complete_update(cs_processor* h, const CsStepArgs& a, bool timing, cs_result* out) {
  h->step.advance(a.do_search);
  cs_status st = wait_for_pose(h, a.seq_value, h->tm.ev[2].get());
  if (st != CS_OK) return st;
  if (timing) {
    st = collect_timing(h, true);
    if (st != CS_OK) return st;
  }
  CS_CHECK_STUCK(h);
  if (reinterpret_cast<const CsDevResult*>(h->h_slot.get())->searched < 0)
    return fail(h, CS_ERR_NCCL, "candidate-split group: a rank never delivered its arg-min (exchange timed out after %.1f s)",
                (double)CS_XCHG_TIMEOUT_NS * 1e-9);
  if (out) {
    copy_update_results(out, reinterpret_cast<const CsDevResult*>(h->h_slot.get()), 1);
    if (timing) {
      long long v = 0;
      CS_CUDA(h, cudaMemcpyAsync(&v, reinterpret_cast<uint8_t*>(h->d_sess.get()) + offsetof(CsSession, visits_slot) + (h->step.step_counter & 1u) * sizeof(long long), sizeof(v),
                                 cudaMemcpyDeviceToHost, h->stream));
      CS_CUDA(h, cudaStreamSynchronize(h->stream));
      out->visits = v;
    }
  }
  return CS_OK;
}

cs_status cs_update(cs_processor* h, const float* points, int32_t n_points, const float odometry_pose[3],
                    const float* cand_offsets, cs_result* out) {
  NvtxRange nvtx_range("cs_update");
  CS_CHECK_HANDLE(h);
  const bool timing = (h->cfg.flags & CS_FLAG_TIMING) != 0;
  CsStepArgs a{};
  cs_status st = stage_update(h, points, n_points, odometry_pose, cand_offsets, timing, &a);
  if (st != CS_OK) return st;
  st = launch_step(h, a, n_points, rings_hint(h, max_range_of(points, n_points)), timing, 2);
  if (st != CS_OK) return st;
  return complete_update(h, a, timing, out);
}

// CoreSLAMProcessor.Update(List<ScanSegment>) whole (:717-752): ScanSegmentsToCloud included (SURVEY 8f row 2).
cs_status cs_update_segments(cs_processor* h, const float* rays, const int32_t* seg_first, const float* seg_poses, int32_t n_rays,
                             int32_t n_segments, const float* cand_offsets, cs_result* out) {
  NvtxRange nvtx_range("cs_update_segments");
  CS_CHECK_HANDLE(h);
  cs_status st = check_segments(h, rays, seg_first, seg_poses, n_rays, n_segments);
  if (st != CS_OK) return st;
  const float* odo = seg_poses + 3 * (size_t)(n_segments - 1);  // :719 odoPose = segments.Last().Pose
  const bool timing = (h->cfg.flags & CS_FLAG_TIMING) != 0;
  SegInput seg{rays, seg_first, seg_poses, n_segments};
  CsStepArgs a{};
  st = stage_update(h, nullptr, n_rays, odo, cand_offsets, timing, &a, &seg);
  if (st != CS_OK) { g_next_launch_plain = false; return st; }
  st = launch_step(h, a, n_rays, rings_hint(h, max_range_of_segments(rays, seg_first, seg_poses, n_segments, odo)), timing, 2);
  g_next_launch_plain = false;
  if (st != CS_OK) return st;
  return complete_update(h, a, timing, out);
}

cs_status cs_segments_to_cloud(cs_processor* h, const float* rays, const int32_t* seg_first, const float* seg_poses, int32_t n_rays,
                               int32_t n_segments, const float odometry_pose[3], float* points_out) {
  CS_CHECK_HANDLE(h);
  cs_status st = check_segments(h, rays, seg_first, seg_poses, n_rays, n_segments);
  if (st != CS_OK) return st;
  if (!odometry_pose || !points_out) return fail(h, CS_ERR_INVALID_ARGUMENT, "cs_segments_to_cloud: null argument");
  if (h->pending) return fail(h, CS_ERR_STATE, "a split-phase update is in flight: call cs_update_finish first");
  const size_t off_rays = kHdrBytes;
  const size_t off_first = align_up(off_rays + (size_t)n_rays * 8, 16);
  const size_t off_poses = align_up(off_first + (size_t)(n_segments + 1) * 4, 16);
  const size_t total = align_up(off_poses + (size_t)n_segments * 12, 16);
  memcpy(h->h_stage.get() + off_rays, rays, (size_t)n_rays * 8);
  memcpy(h->h_stage.get() + off_first, seg_first, (size_t)(n_segments + 1) * 4);
  memcpy(h->h_stage.get() + off_poses, seg_poses, (size_t)n_segments * 12);
  CS_CUDA(h, cudaMemcpyAsync(h->d_stage.get(), h->h_stage.get(), total, cudaMemcpyHostToDevice, h->stream));
  st = launch_cloud(h, h->d_stage.get() + off_rays, h->d_stage.get() + off_first, h->d_stage.get() + off_poses, n_rays, n_segments, odometry_pose);
  if (st != CS_OK) return st;
  CS_CUDA(h, cudaMemcpyAsync(points_out, h->d_cloud.get(), (size_t)n_rays * 8, cudaMemcpyDeviceToHost, h->stream));
  CS_CUDA(h, cudaStreamSynchronize(h->stream));
  return CS_OK;
}

// ---- multi-GPU candidate split (SURVEY 8e, BASELINE cfg4) ---------------------------------------------
cs_status cs_update_begin(cs_processor* h, const float* points, int32_t n_points, const float odometry_pose[3],
                          const float* cand_offsets, int32_t cand_first, int32_t cand_count, uint64_t** key_device) {
  NvtxRange nvtx_range("cs_update_begin");
  CS_CHECK_HANDLE(h);
  if (cand_first < 0 || cand_count < 0 || (long long)cand_first + cand_count > (long long)h->n_cand + 1)
    return fail(h, CS_ERR_INVALID_ARGUMENT, "candidate slice [%d, %d) outside [0, T*I+1 = %d)", cand_first,
                cand_first + cand_count, h->n_cand + 1);
  CsStepArgs a{};
  cs_status st = stage_update(h, points, n_points, odometry_pose, cand_offsets, false, &a, nullptr, true);
  if (st != CS_OK) return st;
  a.cand_first = cand_first;
  a.cand_count = cand_count;
  const int rings = rings_hint(h, max_range_of(points, n_points));
  if (cand_count > 0) {
    st = launch_step(h, a, n_points, rings, false, 2, CS_PHASE_SEARCH);
    if (st != CS_OK) return st;
  }
  h->pending = true;
  h->pending_args = a;
  h->pending_points = n_points;
  h->pending_rings = rings;
  if (key_device)  // NULL when this scan runs no search (:726): nothing to exchange
    *key_device = (a.do_search && cand_count > 0)
                      ? reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(h->d_sess.get()) + offsetof(CsSession, key) +
                                                    sizeof(unsigned long long) * (size_t)a.parity)
                      : nullptr;
  return CS_OK;
}

cs_status cs_update_finish(cs_processor* h, cs_result* out) {
  NvtxRange nvtx_range("cs_update_finish");
  CS_CHECK_HANDLE(h);
  if (!h->pending) return fail(h, CS_ERR_STATE, "cs_update_finish without cs_update_begin");
  h->pending = false;
  const CsStepArgs a = h->pending_args;
  cs_status st = launch_step(h, a, h->pending_points, h->pending_rings, false, 2, CS_PHASE_FINISH);
  if (st != CS_OK) return st;
  return complete_update(h, a, false, out);
}

// ---- candidate-split group with the exchange inside the search kernel (SURVEY 8b "cs_group_create", 8e) ------------------
static cs_status group_table(cs_processor* h) {
  if (!h->d_xchg) {
    const size_t words = (size_t)2 * CS_GROUP_MAX * 2;
    CS_CUDA(h, alloc(h->d_xchg, words));
    CS_CUDA(h, cudaMemset(h->d_xchg.get(), 0, words * sizeof(unsigned long long)));
  }
  return CS_OK;
}

cs_status cs_group_export(cs_processor* h, cs_ipc_handle* out) {
  CS_CHECK_HANDLE(h);
  if (!out) return fail(h, CS_ERR_INVALID_ARGUMENT, "cs_group_export: null out");
  cs_status st = group_table(h);
  if (st != CS_OK) return st;
  static_assert(sizeof(cudaIpcMemHandle_t) <= sizeof(cs_ipc_handle), "cs_ipc_handle too small");
  cudaIpcMemHandle_t mh;
  CS_CUDA(h, cudaIpcGetMemHandle(&mh, h->d_xchg.get()));
  memset(out, 0, sizeof(*out));
  memcpy(out, &mh, sizeof(mh));
  return CS_OK;
}

cs_status cs_group_detach(cs_processor* h) {
  CS_CHECK_HANDLE(h);
  CS_CUDA(h, cudaStreamSynchronize(h->stream));
  for (int p = 0; p < CS_GROUP_MAX; p++) {
    if (h->xchg_ipc[p] && h->xchg_peer[p]) cudaIpcCloseMemHandle(h->xchg_peer[p]);
    h->xchg_peer[p] = nullptr;
    h->xchg_ipc[p] = false;
  }
  h->group_world = 0;
  h->group_rank = 0;
  h->group_shares_device = false;
  h->xchg_seq = 0;
  if (h->d_xchg) CS_CUDA(h, cudaMemset(h->d_xchg.get(), 0, (size_t)2 * CS_GROUP_MAX * 2 * sizeof(unsigned long long)));
  cudaGetLastError();
  return CS_OK;
}

static cs_status group_check(cs_processor* h, int32_t rank, int32_t world) {
  if (world < 1 || world > CS_GROUP_MAX || rank < 0 || rank >= world)
    return fail(h, CS_ERR_INVALID_ARGUMENT, "group: rank %d of %d (at most %d ranks)", rank, world, CS_GROUP_MAX);
  if ((long long)h->n_cand + 1 < world) return fail(h, CS_ERR_INVALID_ARGUMENT, "group: fewer candidates than ranks");
  if (h->pending) return fail(h, CS_ERR_STATE, "a split-phase update is in flight");
  return CS_OK;
}

cs_status cs_group_attach(cs_processor* h, int32_t rank, int32_t world, const cs_ipc_handle* handles) {
  CS_CHECK_HANDLE(h);
  cs_status st = group_check(h, rank, world);
  if (st != CS_OK) return st;
  if (!handles && world > 1) return fail(h, CS_ERR_INVALID_ARGUMENT, "cs_group_attach: null handles");
  st = cs_group_detach(h);
  if (st == CS_OK) st = group_table(h);
  if (st != CS_OK) return st;
  for (int p = 0; p < world; p++) {
    if (p == rank) { h->xchg_peer[p] = h->d_xchg.get(); continue; }
    cudaIpcMemHandle_t mh;
    memcpy(&mh, &handles[p], sizeof(mh));
    void* ptr = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&ptr, mh, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
      cudaGetLastError();
      cs_group_detach(h);
      return fail(h, CS_ERR_NCCL, "cs_group_attach: cudaIpcOpenMemHandle(rank %d) failed: %s", p, cudaGetErrorString(e));
    }
    h->xchg_peer[p] = static_cast<unsigned long long*>(ptr);
    h->xchg_ipc[p] = true;
  }
  h->group_rank = rank;
  h->group_world = world;
  return CS_OK;
}

cs_status cs_group_attach_local(cs_processor* h, int32_t rank, int32_t world, cs_processor* const* peers) {
  CS_CHECK_HANDLE(h);
  cs_status st = group_check(h, rank, world);
  if (st != CS_OK) return st;
  if (!peers && world > 1) return fail(h, CS_ERR_INVALID_ARGUMENT, "cs_group_attach_local: null peers");
  st = cs_group_detach(h);
  if (st == CS_OK) st = group_table(h);
  if (st != CS_OK) return st;
  for (int p = 0; p < world; p++) {
    cs_processor* q = (p == rank) ? h : peers[p];
    if (!q) { cs_group_detach(h); return fail(h, CS_ERR_INVALID_ARGUMENT, "cs_group_attach_local: peer %d is null", p); }
    if (q != h) {
      if (cudaSetDevice(q->device) != cudaSuccess || group_table(q) != CS_OK) {
        cudaSetDevice(h->device);
        cs_group_detach(h);
        return fail(h, CS_ERR_CUDA, "cs_group_attach_local: peer %d has no exchange table", p);
      }
      cudaSetDevice(h->device);
      if (q->device == h->device) h->group_shares_device = true;
      if (q->device != h->device) {
        cudaError_t e = cudaDeviceEnablePeerAccess(q->device, 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) {
          cudaGetLastError();
          cs_group_detach(h);
          return fail(h, CS_ERR_NCCL, "cs_group_attach_local: no peer access to device %d: %s", q->device, cudaGetErrorString(e));
        }
        cudaGetLastError();
      }
    }
    h->xchg_peer[p] = q->d_xchg.get();
  }
  h->group_rank = rank;
  h->group_world = world;
  return CS_OK;
}

cs_status cs_sync(cs_processor* h) {
  CS_CHECK_HANDLE(h);
  CS_CUDA(h, cudaStreamSynchronize(h->stream));
  return CS_OK;
}

// -----------------------------------------------------------------------------------------------------
static cs_status export_wait(cs_processor* h) {
  if (h->export_busy) {
    CS_CUDA(h, cudaEventSynchronize(h->ev_export_done.get()));
    h->export_busy = false;
  }
  return CS_OK;
}

cs_status cs_map_download(cs_processor* h, uint16_t* pixels) {
  NvtxRange nvtx_range("cs_map_download");
  CS_CHECK_HANDLE(h);
  if (!pixels) return fail(h, CS_ERR_INVALID_ARGUMENT, "null pixels");
  cs_status st = export_wait(h);  // d_linear may still be read by an export's D2H copy
  if (st != CS_OK) return st;
  return download_map(h, h->d_map.get(), pixels);
}

cs_status cs_map_upload(cs_processor* h, const uint16_t* pixels) {
  NvtxRange nvtx_range("cs_map_upload");
  CS_CHECK_HANDLE(h);
  if (!pixels) return fail(h, CS_ERR_INVALID_ARGUMENT, "null pixels");
  cs_status st = export_wait(h);  // d_linear may still be read by an export's D2H copy
  if (st == CS_OK) st = ensure_linear(h);
  if (st != CS_OK) return st;
  CS_CUDA(h, cudaMemcpyAsync(h->d_linear.get(), pixels, (size_t)h->size * h->size * 2, cudaMemcpyHostToDevice, h->stream));
  dispatch_layout(h->tiled, [&](auto T) {
    cs_relayout_kernel<decltype(T)::value><<<148 * 8, 256, 0, h->stream>>>(h->d_map.get(), h->d_linear.get(), h->size, h->pitch_tiles, 1);
  });
  h->launches++;
  CS_CUDA(h, cudaStreamSynchronize(h->stream));
  return CS_OK;
}

cs_status cs_map_fill(cs_processor* h, uint16_t value) {
  CS_CHECK_HANDLE(h);
  cs_status st = launch_fill(h, value);
  if (st != CS_OK) return st;
  CS_CUDA(h, cudaStreamSynchronize(h->stream));
  return CS_OK;
}

cs_status cs_map_packed(cs_processor* h, uint8_t* packed) {
  CS_CHECK_HANDLE(h);
  if (!packed) return fail(h, CS_ERR_INVALID_ARGUMENT, "null packed");
  {
    cs_status wst = export_wait(h);
    if (wst != CS_OK) return wst;
  }
  size_t n = ((size_t)h->size * h->size) / 2;
  if (!h->d_packed) CS_CUDA(h, alloc(h->d_packed, n));
  dispatch_layout(h->tiled, [&](auto T) {
    cs_pack_kernel<decltype(T)::value><<<148 * 8, 256, 0, h->stream>>>(h->d_map.get(), h->size, h->pitch_tiles, h->d_packed.get());
  });
  h->launches++;
  CS_CUDA(h, cudaMemcpyAsync(packed, h->d_packed.get(), n, cudaMemcpyDeviceToHost, h->stream));
  CS_CUDA(h, cudaStreamSynchronize(h->stream));
  return CS_OK;
}

// Map export without stalling the update stream (SURVEY 8f row 3): the viewer formats of the reference — Gray16
// (MainWindow.xaml.cs:227-229 writes HoleMap.Pixels into a Gray16 bitmap), 4-bpp packed (HoleMap.GetPackedPixels,
// HoleMap.cs:44-55) and the ObstacleMap's sbyte grid — are snapshotted by a short kernel in stream order (after the
// last integration, before the next), and the device-to-host copy of the snapshot runs on a side stream while the next
// Updates proceed.
cs_status cs_map_export_begin(cs_processor* h, int32_t format, void* dst) {
  CS_CHECK_HANDLE(h);
  if (!dst) return fail(h, CS_ERR_INVALID_ARGUMENT, "cs_map_export_begin: null destination");
  if (format < CS_EXPORT_GRAY16 || format > CS_EXPORT_OBSTACLE_I8) return fail(h, CS_ERR_INVALID_ARGUMENT, "unknown export format %d", format);
  if (format == CS_EXPORT_OBSTACLE_I8 && !h->d_obst) return fail(h, CS_ERR_STATE, "this processor has no ObstacleMap");
  if (!h->export_stream) {
    CS_CUDA(h, create(h->export_stream));
    CS_CUDA(h, create(h->ev_export_snap));
    CS_CUDA(h, create(h->ev_export_done));
  }
  // the previous export's copy must be through with the snapshot buffers before they are overwritten (device-side wait)
  if (h->export_busy) CS_CUDA(h, cudaStreamWaitEvent(h->stream, h->ev_export_done.get(), 0));
  const size_t cells = (size_t)h->size * h->size;
  const void* src = nullptr;
  size_t bytes = 0;
  if (format == CS_EXPORT_GRAY16) {
    cs_status st = relayout_to_linear(h, h->d_map.get());
    if (st != CS_OK) return st;
    src = h->d_linear.get(); bytes = cells * 2;
  } else if (format == CS_EXPORT_PACKED4) {
    if (!h->d_packed) CS_CUDA(h, alloc(h->d_packed, cells / 2));
    dispatch_layout(h->tiled, [&](auto T) {
      cs_pack_kernel<decltype(T)::value><<<148 * 8, 256, 0, h->stream>>>(h->d_map.get(), h->size, h->pitch_tiles, h->d_packed.get());
    });
    h->launches++;
    src = h->d_packed.get(); bytes = cells / 2;
  } else {
    const CsObstacle& o = h->ho;
    bytes = (size_t)o.size * o.size;
    if (!h->d_obst_snap) CS_CUDA(h, alloc(h->d_obst_snap, bytes));
    CS_CUDA(h, cudaMemcpy2DAsync(h->d_obst_snap.get(), (size_t)o.size, o.pixels, (size_t)o.pitch, (size_t)o.size, (size_t)o.size,
                                 cudaMemcpyDeviceToDevice, h->stream));
    src = h->d_obst_snap.get();
  }
  CS_CUDA(h, cudaGetLastError());
  CS_CUDA(h, cudaEventRecord(h->ev_export_snap.get(), h->stream));
  CS_CUDA(h, cudaStreamWaitEvent(h->export_stream.get(), h->ev_export_snap.get(), 0));
  CS_CUDA(h, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, h->export_stream.get()));
  CS_CUDA(h, cudaEventRecord(h->ev_export_done.get(), h->export_stream.get()));
  h->export_busy = true;
  return CS_OK;
}

cs_status cs_map_export_wait(cs_processor* h) {
  CS_CHECK_HANDLE(h);
  return export_wait(h);
}

// Queues the checksum of `map` (cs_host_map_checksum of its row-major pixels) into *out; the caller synchronises.
static cs_status queue_map_checksum(CsHost* h, const uint16_t* map, int blocks, uint64_t* out) {
  CS_CUDA(h, cudaMemsetAsync(h->d_checksum.get(), 0, sizeof(unsigned long long), h->stream));
  dispatch_layout(h->tiled, [&](auto T) {
    cs_checksum_kernel<decltype(T)::value><<<blocks, 256, 0, h->stream>>>(map, h->size, h->pitch_tiles, h->d_checksum.get());
  });
  h->launches++;
  CS_CUDA(h, cudaMemcpyAsync(out, h->d_checksum.get(), sizeof(unsigned long long), cudaMemcpyDeviceToHost, h->stream));
  return CS_OK;
}

cs_status cs_map_checksum(cs_processor* h, uint64_t* checksum) {
  CS_CHECK_HANDLE(h);
  if (!checksum) return fail(h, CS_ERR_INVALID_ARGUMENT, "null checksum");
  cs_status st = queue_map_checksum(h, h->d_map.get(), 148 * 8, checksum);
  if (st != CS_OK) return st;
  CS_CUDA(h, cudaStreamSynchronize(h->stream));
  return CS_OK;
}

uint64_t cs_host_map_checksum(const uint16_t* pixels, int32_t size) {
  unsigned long long acc = 0;
  const size_t n = (size_t)size * (size_t)size;
  for (size_t i = 0; i < n; i++) acc += ((unsigned long long)pixels[i] + 1ull) * cs_mix64((unsigned long long)i);
  return acc;
}

uint64_t cs_host_obstacle_checksum(const int8_t* pixels, int32_t size) {
  unsigned long long acc = 0;
  const size_t n = size > 0 ? (size_t)size * (size_t)size : 0;
  for (size_t i = 0; i < n; i++) acc += ((unsigned long long)(uint8_t)pixels[i] + 1ull) * cs_mix64((unsigned long long)i);
  return acc;
}

// -----------------------------------------------------------------------------------------------------
cs_status cs_get_timing(cs_processor* h, cs_timing* t) {
  if (!h || !t) return CS_ERR_INVALID_ARGUMENT;
  *t = h->last_timing;
  return CS_OK;
}

cs_status cs_get_distances(cs_processor* h, int32_t* distances, int32_t count) {
  CS_CHECK_HANDLE(h);
  if (!h->hs.distances) return fail(h, CS_ERR_STATE, "handle was created without CS_FLAG_KEEP_DISTANCES");
  if (!distances || count < 0 || count > h->n_cand + 1) return fail(h, CS_ERR_INVALID_ARGUMENT, "bad count");
  CS_CUDA(h, cudaMemcpyAsync(distances, h->d_distances.get(), (size_t)count * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  CS_CUDA(h, cudaStreamSynchronize(h->stream));
  return CS_OK;
}

cs_status cs_get_rays(cs_processor* h, int32_t* rays, int32_t n_points) {
  CS_CHECK_HANDLE(h);
  if (!h->d_ray_dbg) return fail(h, CS_ERR_STATE, "handle was created without CS_FLAG_DEBUG_RAYS");
  if (!rays || n_points < 0 || n_points > h->max_points) return fail(h, CS_ERR_INVALID_ARGUMENT, "bad n_points");
  CS_CUDA(h, cudaMemcpyAsync(rays, h->d_ray_dbg.get(), (size_t)n_points * 6 * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  CS_CUDA(h, cudaStreamSynchronize(h->stream));
  return CS_OK;
}

cs_status cs_get_visits(cs_processor* h, int64_t* visits) {
  CS_CHECK_HANDLE(h);
  if (!visits) return fail(h, CS_ERR_INVALID_ARGUMENT, "null visits");
  long long v = 0;
  CS_CUDA(h, cudaMemcpyAsync(&v, reinterpret_cast<uint8_t*>(h->d_sess.get()) + offsetof(CsSession, visits_slot) + (h->step.step_counter & 1u) * sizeof(long long), sizeof(v),
                             cudaMemcpyDeviceToHost, h->stream));
  CS_CUDA(h, cudaStreamSynchronize(h->stream));
  *visits = v;
  return CS_OK;
}

cs_status cs_get_ring_cycles(cs_processor* h, int64_t* cycles, int32_t count) {
  CS_CHECK_HANDLE(h);
  const size_t slots = ((size_t)h->size + CS_DIAG_SEARCH_BLOCKS) * 8;
  if (count < 0 || (size_t)count > slots) return fail(h, CS_ERR_INVALID_ARGUMENT, "bad count");
  if (!h->d_ring_cycles) {  // first call switches the diagnostics on
    CS_CUDA(h, alloc(h->d_ring_cycles, slots));
    CS_CUDA(h, cudaMemsetAsync(h->d_ring_cycles.get(), 0, slots * sizeof(long long), h->stream));
    h->hs.ring_cycles = h->d_ring_cycles.get();
    return patch_session(h, offsetof(CsSession, ring_cycles), &h->hs.ring_cycles, sizeof(long long*));
  }
  if (cycles && count > 0) {
    CS_CUDA(h, cudaMemcpyAsync(cycles, h->d_ring_cycles.get(), (size_t)count * sizeof(long long), cudaMemcpyDeviceToHost, h->stream));
    CS_CUDA(h, cudaStreamSynchronize(h->stream));
  }
  return CS_OK;
}

cs_status cs_get_search_plan(cs_processor* h, int32_t n_points, int32_t n_cand, int32_t plan[5]) {
  CS_CHECK_HANDLE(h);
  if (!plan || n_points < 1 || n_cand < 0) return fail(h, CS_ERR_INVALID_ARGUMENT, "cs_get_search_plan: bad argument");
  const int sms = device_sm_count(h->device);
  S2Plan s2;
  // (as cs_update launches it: a block carries the glue table's service warp beside the slab's threads)
  const int cap = h->d_spec ? CS_S2_MAX_THREADS - 32 : CS_S2_MAX_THREADS;
  if (cs_plan_search2(1, h->s2_cap, cs_s2_min_cand(h->cfg.flags), (long long)n_cand + 1, n_points, sms, &s2, cap)) {
    plan[0] = 1; plan[1] = s2.clusters; plan[2] = s2.slabs; plan[3] = s2.threads; plan[4] = s2.points;
  } else {
    const int warps = cs_search_warps((long long)n_cand + 1, 1, sms);
    plan[0] = 0; plan[1] = (int)(((long long)n_cand + 1 + warps - 1) / warps); plan[2] = 1; plan[3] = warps * 32; plan[4] = n_points;
  }
  return CS_OK;
}

cs_status cs_get_launch_count(cs_processor* h, uint64_t* launches) {
  if (!h || !launches) return CS_ERR_INVALID_ARGUMENT;
  *launches = h->launches;
  return CS_OK;
}

cs_status cs_pinned_alloc(void** ptr, uint64_t bytes) {
  if (!ptr) return CS_ERR_INVALID_ARGUMENT;
  cudaError_t e = cudaHostAlloc(ptr, bytes, cudaHostAllocDefault);
  if (e != cudaSuccess) {
    fail(nullptr, CS_ERR_OUT_OF_MEMORY, "cudaHostAlloc(%llu): %s", (unsigned long long)bytes, cudaGetErrorString(e));
    cudaGetLastError();
    return CS_ERR_OUT_OF_MEMORY;
  }
  return CS_OK;
}

cs_status cs_pinned_free(void* ptr) {
  if (ptr) HostFree()(ptr);
  return CS_OK;
}

// -----------------------------------------------------------------------------------------------------
cs_status cs_scanlog_create(int32_t device, int32_t n_scans, int32_t max_points, int32_t n_offsets, cs_scanlog** out) {
  if (!out || n_scans <= 0 || max_points <= 0 || n_offsets < 0 || max_points > 65536)
    return fail(nullptr, CS_ERR_INVALID_ARGUMENT, "cs_scanlog_create: bad argument");
  *out = nullptr;
  if (cs_device_count() <= device) return fail(nullptr, CS_ERR_NO_DEVICE, "no such CUDA device");
  std::unique_ptr<cs_scanlog> log;  // (a failed create releases what it allocated)
  try {  // a file header with a huge n_scans must come back as a status, not as std::bad_alloc through the C boundary
    log.reset(new cs_scanlog());
    log->device = device;
    log->n_scans = n_scans;
    log->max_points = (max_points + 1) & ~1;  // keep every scan's points 16-byte aligned
    log->n_offsets = n_offsets;
    log->h_hdr.assign((size_t)n_scans, CsStepHeader{});
    log->h_points.assign((size_t)n_scans * log->max_points * 2, 0.f);
    log->h_offsets.assign((size_t)n_scans * n_offsets * 3, 0.f);
    log->h_max_range.assign((size_t)n_scans, 0.0);
  } catch (const std::exception&) {  // bad_alloc, length_error
    return fail(nullptr, CS_ERR_OUT_OF_MEMORY, "cs_scanlog_create: host allocation failed (%d scans x %d points, %d offsets)", n_scans,
                max_points, n_offsets);
  }
  cudaSetDevice(device);
  const bool ok = alloc(log->d_hdr, (size_t)n_scans) == cudaSuccess &&
                  alloc(log->d_points, (size_t)n_scans * log->max_points) == cudaSuccess &&
                  alloc(log->d_offsets, 3 * (size_t)n_scans * (n_offsets > 0 ? n_offsets : 1)) == cudaSuccess &&
                  alloc(log->d_results, (size_t)n_scans) == cudaSuccess;
  if (!ok) {
    cudaGetLastError();
    return fail(nullptr, CS_ERR_OUT_OF_MEMORY, "cs_scanlog_create: device allocation failed");
  }
  *out = log.release();
  return CS_OK;
}

cs_status cs_scanlog_set(cs_scanlog* log, int32_t scan, const float* points, int32_t n_points,
                         const float odometry_pose[3], const float* cand_offsets) {
  if (!log || !points || !odometry_pose || scan < 0 || scan >= log->n_scans || n_points <= 0 || n_points > log->max_points)
    return CS_ERR_INVALID_ARGUMENT;
  CsStepHeader& hd = log->h_hdr[scan];
  memset(&hd, 0, sizeof(hd));
  hd.odo[0] = odometry_pose[0]; hd.odo[1] = odometry_pose[1]; hd.odo[2] = odometry_pose[2];
  hd.n_points = n_points;
  memcpy(&log->h_points[(size_t)scan * log->max_points * 2], points, (size_t)n_points * 8);
  log->h_max_range[scan] = max_range_of(points, n_points);
  if (cand_offsets && log->n_offsets > 0)
    memcpy(&log->h_offsets[(size_t)scan * log->n_offsets * 3], cand_offsets, (size_t)log->n_offsets * 12);
  log->uploaded = false;
  return CS_OK;
}

cs_status cs_scanlog_upload(cs_scanlog* log) {
  if (!log) return CS_ERR_INVALID_ARGUMENT;
  cudaSetDevice(log->device);
  bool ok = cudaMemcpy(log->d_hdr.get(), log->h_hdr.data(), sizeof(CsStepHeader) * log->n_scans, cudaMemcpyHostToDevice) == cudaSuccess &&
            cudaMemcpy(log->d_points.get(), log->h_points.data(), log->h_points.size() * sizeof(float), cudaMemcpyHostToDevice) == cudaSuccess;
  if (ok && log->n_offsets > 0)
    ok = cudaMemcpy(log->d_offsets.get(), log->h_offsets.data(), log->h_offsets.size() * sizeof(float), cudaMemcpyHostToDevice) == cudaSuccess;
  if (!ok) return fail(nullptr, CS_ERR_CUDA, "cs_scanlog_upload: %s", cudaGetErrorString(cudaGetLastError()));
  log->uploaded = true;
  static std::atomic<uint64_t> g_log_generation{1};
  log->generation = g_log_generation.fetch_add(1);
  return CS_OK;
}

// ---- scan-log files (SURVEY 8f row 4) ---------------------------------------------------------------
// The reference has no log format (the simulator generates scans live, MainWindow.xaml.cs:380-407); this one lets a
// recorded drive be replayed through both implementations.  Little-endian, see include/coreslam_b200.h.
namespace {
struct CslgHeader {
  char magic[4];
  uint32_t version, n_scans, max_points, n_offsets, reserved[3];
};
static_assert(sizeof(CslgHeader) == 32, "CSLG header");

struct FileCloser {
  FILE* f;
  ~FileCloser() { if (f) fclose(f); }
};

cs_status cslg_open(const char* path, FILE** f, CslgHeader* hd) {
  if (!path) return fail(nullptr, CS_ERR_INVALID_ARGUMENT, "scan log: null path");
  *f = fopen(path, "rb");
  if (!*f) return fail(nullptr, CS_ERR_INVALID_ARGUMENT, "scan log: cannot open %s", path);
  if (fread(hd, sizeof(*hd), 1, *f) != 1 || memcmp(hd->magic, "CSLG", 4) != 0 || hd->version != 1 || hd->n_scans == 0 ||
      hd->max_points == 0 || hd->max_points > 65536 || hd->n_offsets > (1u << 26)) {
    fclose(*f);
    *f = nullptr;
    return fail(nullptr, CS_ERR_INVALID_ARGUMENT, "scan log: %s is not a CSLG version 1 file", path);
  }
  return CS_OK;
}

// reads the next record; points/offsets may be NULL to skip their payload
cs_status cslg_read_record(FILE* f, const CslgHeader& hd, int32_t* n_points, float odo[3], float* points, float* offsets) {
  uint32_t n = 0;
  if (fread(&n, 4, 1, f) != 1 || n == 0 || n > hd.max_points || fread(odo, 4, 3, f) != 3)
    return fail(nullptr, CS_ERR_INVALID_ARGUMENT, "scan log: truncated or corrupt record");
  *n_points = (int32_t)n;
  const long pts_bytes = (long)n * 8, off_bytes = (long)hd.n_offsets * 12;
  bool ok = points ? fread(points, 8, n, f) == n : fseek(f, pts_bytes, SEEK_CUR) == 0;
  if (ok && hd.n_offsets) ok = offsets ? fread(offsets, 12, hd.n_offsets, f) == hd.n_offsets : fseek(f, off_bytes, SEEK_CUR) == 0;
  return ok ? CS_OK : fail(nullptr, CS_ERR_INVALID_ARGUMENT, "scan log: truncated record");
}
}  // namespace

cs_status cs_scanlog_save(const cs_scanlog* log, const char* path) {
  if (!log || !path) return fail(nullptr, CS_ERR_INVALID_ARGUMENT, "cs_scanlog_save: null argument");
  FILE* f = fopen(path, "wb");
  if (!f) return fail(nullptr, CS_ERR_INVALID_ARGUMENT, "cs_scanlog_save: cannot create %s", path);
  FileCloser closer{f};
  CslgHeader hd{};
  memcpy(hd.magic, "CSLG", 4);
  hd.version = 1; hd.n_scans = (uint32_t)log->n_scans; hd.max_points = (uint32_t)log->max_points; hd.n_offsets = (uint32_t)log->n_offsets;
  bool ok = fwrite(&hd, sizeof(hd), 1, f) == 1;
  for (int k = 0; ok && k < log->n_scans; k++) {
    const CsStepHeader& sh = log->h_hdr[k];
    if (sh.n_points <= 0) return fail(nullptr, CS_ERR_STATE, "cs_scanlog_save: scan %d was never set", k);
    const uint32_t n = (uint32_t)sh.n_points;
    ok = fwrite(&n, 4, 1, f) == 1 && fwrite(sh.odo, 4, 3, f) == 3 &&
         fwrite(&log->h_points[(size_t)k * log->max_points * 2], 8, n, f) == n;
    if (ok && log->n_offsets > 0)
      ok = fwrite(&log->h_offsets[(size_t)k * log->n_offsets * 3], 12, (size_t)log->n_offsets, f) == (size_t)log->n_offsets;
  }
  return ok ? CS_OK : fail(nullptr, CS_ERR_INVALID_ARGUMENT, "cs_scanlog_save: write to %s failed", path);
}

cs_status cs_scanlog_file_info(const char* path, int32_t* n_scans, int32_t* max_points, int32_t* n_offsets) {
  FILE* f = nullptr;
  CslgHeader hd;
  cs_status st = cslg_open(path, &f, &hd);
  if (st != CS_OK) return st;
  fclose(f);
  if (n_scans) *n_scans = (int32_t)hd.n_scans;
  if (max_points) *max_points = (int32_t)hd.max_points;
  if (n_offsets) *n_offsets = (int32_t)hd.n_offsets;
  return CS_OK;
}

cs_status cs_scanlog_file_read(const char* path, int32_t scan, float* points, int32_t* n_points, float odometry_pose[3],
                               float* cand_offsets) {
  if (!n_points || !odometry_pose || scan < 0) return fail(nullptr, CS_ERR_INVALID_ARGUMENT, "cs_scanlog_file_read: bad argument");
  FILE* f = nullptr;
  CslgHeader hd;
  cs_status st = cslg_open(path, &f, &hd);
  if (st != CS_OK) return st;
  FileCloser closer{f};
  if ((uint32_t)scan >= hd.n_scans) return fail(nullptr, CS_ERR_INVALID_ARGUMENT, "cs_scanlog_file_read: scan %d of %u", scan, hd.n_scans);
  for (int k = 0; k <= scan; k++) {
    const bool want = k == scan;
    st = cslg_read_record(f, hd, n_points, odometry_pose, want ? points : nullptr, want ? cand_offsets : nullptr);
    if (st != CS_OK) return st;
  }
  return CS_OK;
}

cs_status cs_scanlog_load(int32_t device, const char* path, cs_scanlog** out) {
  if (!out) return fail(nullptr, CS_ERR_INVALID_ARGUMENT, "cs_scanlog_load: null out");
  *out = nullptr;
  FILE* f = nullptr;
  CslgHeader hd;
  cs_status st = cslg_open(path, &f, &hd);
  if (st != CS_OK) return st;
  FileCloser closer{f};
  cs_scanlog* log = nullptr;
  st = cs_scanlog_create(device, (int32_t)hd.n_scans, (int32_t)hd.max_points, (int32_t)hd.n_offsets, &log);
  if (st != CS_OK) return st;
  std::vector<float> pts, off;
  try {
    pts.resize((size_t)hd.max_points * 2);
    off.resize((size_t)hd.n_offsets * 3);
  } catch (const std::exception&) {
    cs_scanlog_destroy(log);
    return fail(nullptr, CS_ERR_OUT_OF_MEMORY, "cs_scanlog_load: host allocation failed");
  }
  for (uint32_t k = 0; k < hd.n_scans; k++) {
    int32_t n = 0;
    float odo[3];
    st = cslg_read_record(f, hd, &n, odo, pts.data(), hd.n_offsets ? off.data() : nullptr);
    if (st == CS_OK) st = cs_scanlog_set(log, (int32_t)k, pts.data(), n, odo, hd.n_offsets ? off.data() : nullptr);
    if (st != CS_OK) {
      cs_scanlog_destroy(log);
      return st;
    }
  }
  st = cs_scanlog_upload(log);
  if (st != CS_OK) {
    cs_scanlog_destroy(log);
    return st;
  }
  *out = log;
  return CS_OK;
}

cs_status cs_scanlog_destroy(cs_scanlog* log) {
  if (!log) return CS_OK;
  delete log;
  cudaGetLastError();
  return CS_OK;
}

cs_status cs_replay(cs_processor* h, const cs_scanlog* log, int32_t first, int32_t count, cs_result* results) {
  NvtxRange nvtx_range("cs_replay");
  CS_CHECK_HANDLE(h);
  if (!log || !log->uploaded) return fail(h, CS_ERR_STATE, "scan log not uploaded");
  if (log->device != h->device) return fail(h, CS_ERR_INVALID_ARGUMENT, "scan log lives on another device");
  if (first < 0 || count < 0 || first + count > log->n_scans) return fail(h, CS_ERR_INVALID_ARGUMENT, "scan range");
  if (log->n_offsets > 0 && log->n_offsets != h->n_cand)
    return fail(h, CS_ERR_INVALID_ARGUMENT, "scan log carries %d offsets per scan, handle needs T*I = %d", log->n_offsets, h->n_cand);
  if (log->max_points > h->max_points) return fail(h, CS_ERR_CAPACITY, "scan log max_points exceeds the handle's");
  const bool timing = (h->cfg.flags & CS_FLAG_TIMING) != 0;
  const bool per_kernel = timing && count == 1;
  if (timing) {
    cudaEventRecord(h->tm.ev[0].get(), h->stream);
    if (per_kernel) cudaEventRecord(h->tm.ev[1].get(), h->stream);
  }
  for (int i = 0; i < count; i++) {
    const int sidx = first + i;
    CsStepArgs a = update_args(*h, log->n_offsets > 0, log->h_hdr[sidx].n_points);
    a.hdr = log->d_hdr.get() + sidx;
    a.points = log->d_points.get() + (size_t)sidx * log->max_points;
    a.cand = log->n_offsets > 0 ? log->d_offsets.get() + (size_t)sidx * log->n_offsets * 3 : nullptr;
    a.result = log->d_results.get() + sidx;
    a.visits_out = reinterpret_cast<long long*>(reinterpret_cast<uint8_t*>(log->d_results.get() + sidx) + offsetof(CsDevResult, visits));
    apply_group(h, a);
    // (the next scan's table, if the log has one: its sort is queued behind this scan's draw kernel, see Presort)
    const float* next_cand = (log->n_offsets > 0 && sidx + 1 < log->n_scans) ? log->d_offsets.get() + (size_t)(sidx + 1) * log->n_offsets * 3 : nullptr;
    cs_status st = launch_step(h, a, log->h_hdr[sidx].n_points, rings_hint(h, log->h_max_range[sidx]), per_kernel, 2, CS_PHASE_ALL,
                               next_cand, log->generation);
    if (st != CS_OK) return st;
    h->step.advance(a.do_search);
  }
  if (timing && !per_kernel) cudaEventRecord(h->tm.ev[4].get(), h->stream);
  if (results && count > 0) {
    static_assert(sizeof(cs_result) == sizeof(CsDevResult), "");
    CS_CUDA(h, cudaMemcpyAsync(results, log->d_results.get() + first, sizeof(CsDevResult) * count, cudaMemcpyDeviceToHost, h->stream));
  }
  // results == NULL: fire and forget — the scans stay queued on the stream (cs_sync / cs_get_pose wait for them)
  if (results || timing) CS_CUDA(h, cudaStreamSynchronize(h->stream));
  if (per_kernel) {
    cs_status st = collect_timing(h, false);
    if (st != CS_OK) return st;
  } else if (timing) {
    float ms = 0;
    cudaEventElapsedTime(&ms, h->tm.ev[0].get(), h->tm.ev[4].get());
    h->last_timing = cs_timing{};
    h->last_timing.total_device_ms = ms;
  }
  return CS_OK;
}

// =====================================================================================================
// Batches of independent sessions on one GPU (SURVEY 8e "sessions", BASELINE cfg5): one launch per
// kernel for all sessions (grid.y = session), every session with its own map, pose, parameters and
// Philox stream.  No data-path communication between sessions or GPUs.
// =====================================================================================================
}  // extern "C"

struct cs_batch : CsHost {
  int n = 0;
  int max_points = 0;
  int user_max_points = 0;  // the caller's cfg.max_points: stride of the caller's `points` array (max_points above is the
                            // internal stride of the staging / device blocks, rounded up to even for 16-byte alignment)
  std::vector<CsSession> hs;
  DevBuf<uint16_t> d_maps;
  // slab-search scratch of all sessions (CsSession::s2_*): per session 2*cap sorted + cap tmp entries, cap meta + cap acc words
  DevBuf<float4> d_s2_entries;
  DevBuf<unsigned long long> d_s2_words;
  uint32_t flags = 0;
  // staging: [n headers][n * max_points points][n * n_cand offsets]
  size_t off_points = 0, off_cand = 0, stage_bytes = 0;
  HostBuf<uint8_t> h_stage;
  DevBuf<uint8_t> d_stage;
  DevBuf<CsDevResult> d_results;
  HostBuf<CsDevResult> h_results;
  HostBuf<uint8_t> stuck_word;  // CS_FLAG_DEBUG_BOUNDED_SPIN: the block CsHost::h_stuck / d_stuck point into
  // cs_batch_submit / cs_batch_collect: two staging + result slots, so that the host stages step k+1 while step k runs
  struct PipeSlot {
    HostBuf<uint8_t> h_stage;
    DevBuf<uint8_t> d_stage;
    DevBuf<CsDevResult> d_results;
    HostBuf<CsDevResult> h_results;
    Event done;
  } pipe[2];
  unsigned pipe_submitted = 0, pipe_collected = 0;
  std::vector<float> start_poses;  // n * 3: cfgs[j].start_pose, the Pose of session j after cs_batch_reset (:172)

  std::vector<CsObstacle> obst;  // host descriptors of the sessions' ObstacleMaps (CsHost::d_obst)
  std::vector<int> unmapped_obstacle_hits;  // per session, :98; the fill values of the next cs_batch_reset
  DevBuf<int> d_obst_fill;                  // ... as the fill kernel reads them
  DevBuf<unsigned long long> d_obst_sums;   // cs_batch_obstacle_checksums

  ~cs_batch() {  // the owners release after this, on the batch's device, once its stream has drained
    cudaSetDevice(device);
    if (stream) cudaStreamSynchronize(stream);
  }
};

namespace {
// The maps of Reset (:169-170) for every session: HoleMap := 32750, ObstacleMap := the session's UnmappedObstacleHits (with
// its no-hit bitmap and touched counter cleared).  Queued on the stream; the caller synchronises.
cs_status batch_fill_maps(cs_batch* b) {
  cs_fill_kernel<<<148 * 8, 256, 0, b->stream>>>(b->d_maps.get(), b->map_cells * (size_t)b->n, (uint16_t)((CS_TS_OBSTACLE + CS_TS_NO_OBSTACLE) / 2));
  b->launches++;
  CS_CUDA(b, cudaGetLastError());
  if (b->d_obst) {
    CS_CUDA(b, cudaMemcpyAsync(b->d_obst_fill.get(), b->unmapped_obstacle_hits.data(), sizeof(int) * (size_t)b->n, cudaMemcpyHostToDevice,
                               b->stream));
    CS_CUDA(b, launch_obstacle_fill(b->stream, b->d_obst.get(), b->d_obst_fill.get(), 0, b->ho, b->n, &b->launches));
  }
  return CS_OK;
}

// The host-owned descriptors of all sessions' ObstacleMaps to the device (in stream order).
cs_status batch_push_obstacles(cs_batch* b) {
  CS_CUDA(b, cudaMemcpyAsync(b->d_obst.get(), b->obst.data(), sizeof(CsObstacle) * (size_t)b->n, cudaMemcpyHostToDevice, b->stream));
  return CS_OK;
}
}  // namespace

extern "C" {

const char* cs_batch_last_error(const cs_batch* b) { return b ? b->error.c_str() : g_create_error.c_str(); }

cs_status cs_batch_create(const cs_config* cfgs, int32_t n_sessions, cs_batch** out) {
  if (!cfgs || !out || n_sessions <= 0 || n_sessions > 65535)
    return fail(nullptr, CS_ERR_INVALID_ARGUMENT, "cs_batch_create: bad argument (1..65535 sessions)");
  *out = nullptr;
  const cs_config& c0 = cfgs[0];
  for (int j = 1; j < n_sessions; j++) {
    const cs_config& c = cfgs[j];
    if (c.hole_map_size != c0.hole_map_size || c.physical_map_size != c0.physical_map_size ||
        c.iterations_per_thread != c0.iterations_per_thread || c.num_search_threads != c0.num_search_threads ||
        c.device != c0.device || c.max_points != c0.max_points || c.flags != c0.flags || c.obstacle_map_size != c0.obstacle_map_size)
      return fail(nullptr, CS_ERR_INVALID_ARGUMENT,
                   "cs_batch_create: session %d differs in map size / iterations / threads / device / max_points / flags / "
                   "obstacle_map_size (only start_pose, sigma_xy, sigma_theta and seed may vary)", j);
  }
  long long n_cand = 0;
  int max_points = 0;
  const cs_status cst = check_config(c0, &n_cand, &max_points);
  if (cst != CS_OK) return cst;

  cs_batch* b = new cs_batch();
  b->device = c0.device;
  b->n = n_sessions;
  b->tiled = !(c0.flags & CS_FLAG_ROW_MAJOR_MAP);
  b->size = c0.hole_map_size;
  b->pitch_tiles = (b->size + 7) / 8;
  b->user_max_points = max_points;
  b->max_points = (max_points + 1) & ~1;
  b->n_cand = (int)n_cand;
  b->scale = (float)c0.hole_map_size / c0.physical_map_size;
  b->flags = c0.flags;
  b->map_cells = b->tiled ? (size_t)b->pitch_tiles * b->pitch_tiles * 64 : (size_t)b->size * b->size;
  b->hs.assign((size_t)n_sessions, CsSession{});
  b->off_points = align_up(sizeof(CsStepHeader) * (size_t)n_sessions, 16);
  b->off_cand = align_up(b->off_points + (size_t)n_sessions * b->max_points * 8, 16);
  b->stage_bytes = align_up(b->off_cand + (size_t)n_sessions * (size_t)n_cand * 12, 16);

  auto bail = [&](cs_status st) {
    g_create_error = b->error;
    cs_batch_destroy(b);
    return st;
  };
  CS_CREATE_CUDA(b, cudaSetDevice(b->device));
  if (c0.stream) {
    b->stream = (cudaStream_t)c0.stream;
  } else {
    CS_CREATE_CUDA(b, create(b->own_stream));
    b->stream = b->own_stream.get();
  }
  CS_CREATE_CUDA(b, alloc(b->d_maps, b->map_cells * (size_t)n_sessions));
  CS_CREATE_CUDA(b, alloc(b->d_sess, (size_t)n_sessions));
  for (int j = 0; j < n_sessions; j++) init_session(b->hs[j], *b, cfgs[j], b->d_maps.get() + (size_t)j * b->map_cells);
  // (a session of a batch has few blocks: one copy of its rays, nothing to spread)
  CS_CREATE_CUDA(b, alloc_ray_scratch(*b, b->hs.data(), n_sessions, 1, b->max_points, b->max_points / 32 + 1));
  CS_CREATE_CUDA(b, alloc(b->d_checksum, 1));
  const int min_cand = cs_s2_min_cand(b->flags, n_sessions);
  if (n_sessions > 1 && min_cand > 0 && n_cand + 1 >= min_cand && n_cand + 1 <= CS_SORT_THREADS * CS_SORT_REG) {
    b->s2_cap = n_cand + 1;
    const size_t cap = (size_t)b->s2_cap;
    CS_CREATE_CUDA(b, alloc(b->d_s2_entries, (size_t)n_sessions * 3 * cap));
    CS_CREATE_CUDA(b, alloc(b->d_s2_words, (size_t)n_sessions * 2 * cap));
    CS_CREATE_CUDA(b, cudaMemsetAsync(b->d_s2_words.get(), 0, (size_t)n_sessions * 2 * cap * sizeof(unsigned long long), b->stream));
  }
  CS_CREATE_CUDA(b, alloc(b->h_stage, b->stage_bytes));
  CS_CREATE_CUDA(b, alloc(b->d_stage, b->stage_bytes));
  CS_CREATE_CUDA(b, alloc(b->d_results, (size_t)n_sessions));
  CS_CREATE_CUDA(b, alloc(b->h_results, (size_t)n_sessions));
  if (b->flags & CS_FLAG_DEBUG_BOUNDED_SPIN) {
    CS_CREATE_CUDA(b, alloc(b->stuck_word, 64, cudaHostAllocMapped));
    b->h_stuck = b->stuck_word.get();
    CS_CREATE_CUDA(b, cudaHostGetDevicePointer((void**)&b->d_stuck, b->h_stuck, 0));
    memset(b->h_stuck, 0, 64);
  }
  for (int j = 0; j < n_sessions; j++) {
    CsSession& s = b->hs[j];
    if (b->s2_cap > 0) {
      const size_t cap = (size_t)b->s2_cap;
      s.s2_sorted = b->d_s2_entries.get() + (size_t)j * 3 * cap;
      s.s2_tmp = s.s2_sorted + 2 * cap;
      s.s2_meta = b->d_s2_words.get() + (size_t)j * 2 * cap;
      s.s2_acc = s.s2_meta + cap;
      s.s2_cap = b->s2_cap;
    }
    reset_session(s, cfgs[j].start_pose);
  }
  b->start_poses.resize((size_t)n_sessions * 3);
  for (int j = 0; j < n_sessions; j++)
    for (int k = 0; k < 3; k++) b->start_poses[3 * (size_t)j + k] = cfgs[j].start_pose[k];
  if (c0.obstacle_map_size > 0) {  // :132-133, per session
    b->obst.resize((size_t)n_sessions);
    CS_CREATE_CUDA(b, alloc_obstacle_maps(*b, b->obst.data(), n_sessions, c0.obstacle_map_size, c0.physical_map_size));
    CS_CREATE_CUDA(b, alloc(b->d_obst_fill, (size_t)n_sessions));
    CS_CREATE_CUDA(b, alloc(b->d_obst_sums, (size_t)n_sessions));
    b->unmapped_obstacle_hits.assign((size_t)n_sessions, -5);  // :98
    const cs_status st = batch_push_obstacles(b);
    if (st != CS_OK) return bail(st);
  }
  const cs_status st = batch_fill_maps(b);
  if (st != CS_OK) return bail(st);
  CS_CREATE_CUDA(b, cudaMemcpyAsync(b->d_sess.get(), b->hs.data(), sizeof(CsSession) * (size_t)n_sessions, cudaMemcpyHostToDevice, b->stream));
  CS_CREATE_CUDA(b, cudaStreamSynchronize(b->stream));
  *out = b;
  return CS_OK;
}

cs_status cs_batch_destroy(cs_batch* b) {
  if (!b) return CS_OK;
  delete b;  // ~cs_batch drains the stream; then every owner releases
  cudaGetLastError();
  return CS_OK;
}

int32_t cs_batch_size(const cs_batch* b) { return b ? b->n : 0; }

// session < 0: all sessions.  Quality 1..255 (:76-82), HoleWidth metres (:87).
cs_status cs_batch_set_params(cs_batch* b, int32_t session, int32_t quality, float hole_width) {
  CS_CHECK_HANDLE(b);
  if (session >= b->n) return fail(b, CS_ERR_INVALID_ARGUMENT, "session %d out of range", session);
  if (quality < 1 || quality > 255) return fail(b, CS_ERR_INVALID_ARGUMENT, "Quality must be 1..255");
  if (!(hole_width >= 0.f) || !(hole_width * b->scale < 60000.f)) return fail(b, CS_ERR_INVALID_ARGUMENT, "HoleWidth out of range");
  CS_CUDA(b, cudaStreamSynchronize(b->stream));
  for (int j = (session < 0 ? 0 : session); j < (session < 0 ? b->n : session + 1); j++) {
    b->hs[j].quality = quality;
    b->hs[j].hole_width = hole_width;
    CS_CUDA(b, cudaMemcpyAsync(reinterpret_cast<uint8_t*>(b->d_sess.get() + j) + offsetof(CsSession, quality), &b->hs[j].quality,
                                sizeof(int), cudaMemcpyHostToDevice, b->stream));
    CS_CUDA(b, cudaMemcpyAsync(reinterpret_cast<uint8_t*>(b->d_sess.get() + j) + offsetof(CsSession, hole_width), &b->hs[j].hole_width,
                                sizeof(float), cudaMemcpyHostToDevice, b->stream));
  }
  CS_CUDA(b, cudaStreamSynchronize(b->stream));
  return CS_OK;
}

static float batch_max_hole_width(const cs_batch* b) {
  float w = 0.f;
  for (const CsSession& s : b->hs) w = s.hole_width > w ? s.hole_width : w;
  return w;
}

// One CoreSLAMProcessor.Update (:717-752) for every session of the batch.
//   points        n_sessions * max_points * (x, y); session j uses the first n_points[j]
//   odometry      n_sessions * (x, y, theta)
//   cand_offsets  n_sessions * T*I * (dx, dy, dtheta) verification tables, or NULL: per-session Philox streams
//   results       optional, n_sessions records (blocks until the poses are back)
namespace {
// UpdateObstacleMap (:751) of every session behind the draw kernel of the step `a` (same pose, same cloud, as launch_step
// does for one processor): one launch of each obstacle kernel for all sessions.  Nothing without ObstacleMaps or points.
cs_status batch_obstacle_update(cs_batch* b, const CsStepArgs& a, int n_points) {
  if (!b->d_obst || n_points <= 0) return CS_OK;
  CS_CUDA(b, launch_obstacle_update(b->stream, b->d_sess.get(), b->d_obst.get(), b->ho, a, n_points, b->n, device_sm_count(b->device), &b->launches));
  return CS_OK;
}

// Stages one Update of every session into (h_stage -> d_stage) and launches its kernels; the result records go to d_results.
cs_status batch_stage_and_launch(cs_batch* b, uint8_t* h_stage, uint8_t* d_stage, CsDevResult* d_results, const float* points,
                                 const int32_t* n_points, const float* odometry, const float* cand_offsets) {
  const bool with_offsets = cand_offsets != nullptr && b->step.searches();
  int max_n = 0;
  double max_range = 0.0;
  bool range_nan = false;  // a NaN point anywhere in the batch: every ring is launched (NaN does not order, so it is tracked apart)
  for (int j = 0; j < b->n; j++) {
    const int np = n_points[j];
    if (np <= 0 || np > b->user_max_points)
      return fail(b, CS_ERR_CAPACITY, "session %d: n_points %d outside 1..%d", j, np, b->user_max_points);
    const float* odo = odometry + 3 * (size_t)j;
    if (!finite3(odo)) return fail(b, CS_ERR_INVALID_ARGUMENT, "session %d: odometry pose is NaN", j);
    CsStepHeader* hdr = reinterpret_cast<CsStepHeader*>(h_stage) + j;
    memset(hdr, 0, sizeof(CsStepHeader));
    hdr->odo[0] = odo[0]; hdr->odo[1] = odo[1]; hdr->odo[2] = odo[2];
    hdr->n_points = np;
    const float* src = points + (size_t)j * b->user_max_points * 2;  // the caller's stride is the caller's cfg.max_points
    memcpy(h_stage + b->off_points + (size_t)j * b->max_points * 8, src, (size_t)np * 8);
    const double r = max_range_of(src, np);
    if (r != r) range_nan = true;
    else if (r > max_range) max_range = r;
    if (np > max_n) max_n = np;
  }
  if (range_nan) max_range = std::numeric_limits<double>::quiet_NaN();
  if (with_offsets) memcpy(h_stage + b->off_cand, cand_offsets, (size_t)b->n * b->n_cand * 12);
  const size_t bytes = with_offsets ? b->stage_bytes : b->off_cand;
  CS_CUDA(b, cudaMemcpyAsync(d_stage, h_stage, bytes, cudaMemcpyHostToDevice, b->stream));

  CsStepArgs a = update_args(*b, with_offsets, max_n);
  a.hdr = reinterpret_cast<const CsStepHeader*>(d_stage);
  a.hdr_stride = 1;
  a.points = reinterpret_cast<const float2*>(d_stage + b->off_points);
  a.points_stride = (size_t)b->max_points;
  a.cand = with_offsets ? reinterpret_cast<const float*>(d_stage + b->off_cand) : nullptr;
  a.cand_stride = (size_t)b->n_cand * 3;
  a.result = d_results;
  a.result_stride = 1;
  CS_CUDA(b, launch_step_ctx(LaunchCtx(b, b->flags, b->n, b->hs.data()), a, max_n,
                             rings_hint_of(b->size, b->scale, batch_max_hole_width(b), max_range), CS_PHASE_ALL));
  cs_status st = batch_obstacle_update(b, a, max_n);
  if (st != CS_OK) return st;
  b->step.advance(a.do_search);
  return CS_OK;
}
}  // namespace

cs_status cs_batch_update(cs_batch* b, const float* points, const int32_t* n_points, const float* odometry,
                          const float* cand_offsets, cs_result* results) {
  NvtxRange nvtx_range("cs_batch_update");
  CS_CHECK_HANDLE(b);
  if (!points || !n_points || !odometry) return fail(b, CS_ERR_INVALID_ARGUMENT, "cs_batch_update: null argument");
  // the pinned block may still be the source of the previous call's copy
  CS_CUDA(b, cudaStreamSynchronize(b->stream));
  cs_status st = batch_stage_and_launch(b, b->h_stage.get(), b->d_stage.get(), b->d_results.get(), points, n_points, odometry, cand_offsets);
  if (st != CS_OK) return st;
  if (results) {
    CS_CUDA(b, cudaMemcpyAsync(b->h_results.get(), b->d_results.get(), sizeof(CsDevResult) * (size_t)b->n, cudaMemcpyDeviceToHost, b->stream));
    CS_CUDA(b, cudaStreamSynchronize(b->stream));
    copy_update_results(results, b->h_results.get(), b->n);
  }
  return CS_OK;
}

// The same Update, pipelined: cs_batch_submit stages and queues a step and returns; cs_batch_collect waits for the oldest
// submitted step and hands out its result records.  At most two steps may be waiting for their collect, so a caller that
// alternates submit(k+1), collect(k) has the host staging of step k+1 (pinned copy, range scan, H2D) running while the device
// works on step k, and consecutive steps stay chained on the stream (no host round trip between them).
cs_status cs_batch_submit(cs_batch* b, const float* points, const int32_t* n_points, const float* odometry,
                          const float* cand_offsets) {
  NvtxRange nvtx_range("cs_batch_submit");
  CS_CHECK_HANDLE(b);
  if (!points || !n_points || !odometry) return fail(b, CS_ERR_INVALID_ARGUMENT, "cs_batch_submit: null argument");
  if (b->pipe_submitted - b->pipe_collected >= 2u)
    return fail(b, CS_ERR_STATE, "cs_batch_submit: two submitted steps are waiting for cs_batch_collect");
  cs_batch::PipeSlot& p = b->pipe[b->pipe_submitted & 1u];
  if (!p.done) {  // first use of the slot: all five resources or none (the event, created last, is the guard)
    cs_batch::PipeSlot fresh;
    cudaError_t e = alloc(fresh.h_stage, b->stage_bytes);
    if (e == cudaSuccess) e = alloc(fresh.d_stage, b->stage_bytes);
    if (e == cudaSuccess) e = alloc(fresh.d_results, (size_t)b->n);
    if (e == cudaSuccess) e = alloc(fresh.h_results, (size_t)b->n);
    if (e == cudaSuccess) e = create(fresh.done);
    if (e != cudaSuccess) {
      cudaGetLastError();
      return fail(b, e == cudaErrorMemoryAllocation ? CS_ERR_OUT_OF_MEMORY : CS_ERR_CUDA, "cs_batch_submit: staging slot: %s",
                   cudaGetErrorString(e));
    }
    p = std::move(fresh);
  }
  // The slot's pinned block was the source of the copy two submits ago; that step has been collected (its `done` event,
  // recorded after the copy, was waited for), so the block is free.  The device block is protected by stream order.
  cs_status st = batch_stage_and_launch(b, p.h_stage.get(), p.d_stage.get(), p.d_results.get(), points, n_points, odometry, cand_offsets);
  if (st != CS_OK) return st;
  CS_CUDA(b, cudaMemcpyAsync(p.h_results.get(), p.d_results.get(), sizeof(CsDevResult) * (size_t)b->n, cudaMemcpyDeviceToHost,
                             b->stream));
  CS_CUDA(b, cudaEventRecord(p.done.get(), b->stream));
  b->pipe_submitted++;
  return CS_OK;
}

cs_status cs_batch_collect(cs_batch* b, cs_result* results /* n_sessions records, or NULL to only wait */) {
  NvtxRange nvtx_range("cs_batch_collect");
  CS_CHECK_HANDLE(b);
  if (b->pipe_collected == b->pipe_submitted) return fail(b, CS_ERR_STATE, "cs_batch_collect: nothing was submitted");
  const cs_batch::PipeSlot& p = b->pipe[b->pipe_collected & 1u];
  CS_CUDA(b, cudaEventSynchronize(p.done.get()));
  if (results) copy_update_results(results, p.h_results.get(), b->n);
  b->pipe_collected++;
  return CS_OK;
}

// Parameter sweep: every session consumes the same device-resident scan log (its own map, pose, parameters
// and — when the log carries no candidate tables — its own Philox stream).  results: optional, the
// n_sessions records of the LAST scan replayed.
cs_status cs_batch_replay(cs_batch* b, const cs_scanlog* log, int32_t first, int32_t count, cs_result* results) {
  NvtxRange nvtx_range("cs_batch_replay");
  CS_CHECK_HANDLE(b);
  if (!log || !log->uploaded) return fail(b, CS_ERR_STATE, "scan log not uploaded");
  if (log->device != b->device) return fail(b, CS_ERR_INVALID_ARGUMENT, "scan log lives on another device");
  if (first < 0 || count < 0 || first + count > log->n_scans) return fail(b, CS_ERR_INVALID_ARGUMENT, "scan range");
  if (log->n_offsets > 0 && log->n_offsets != b->n_cand) return fail(b, CS_ERR_INVALID_ARGUMENT, "scan log offsets != T*I");
  if (log->max_points > b->max_points) return fail(b, CS_ERR_CAPACITY, "scan log max_points exceeds the batch's");
  const float hw = batch_max_hole_width(b);
  for (int i = 0; i < count; i++) {
    const int sidx = first + i;
    CsStepArgs a = update_args(*b, log->n_offsets > 0, log->h_hdr[sidx].n_points);
    a.hdr = log->d_hdr.get() + sidx;
    a.hdr_stride = 0;
    a.points = log->d_points.get() + (size_t)sidx * log->max_points;
    a.points_stride = 0;
    a.cand = log->n_offsets > 0 ? log->d_offsets.get() + (size_t)sidx * log->n_offsets * 3 : nullptr;
    a.cand_stride = 0;
    a.result = b->d_results.get();
    a.result_stride = 1;
    CS_CUDA(b, launch_step_ctx(LaunchCtx(b, b->flags, b->n, b->hs.data()), a, log->h_hdr[sidx].n_points,
                               rings_hint_of(b->size, b->scale, hw, log->h_max_range[sidx]), CS_PHASE_ALL));
    cs_status st = batch_obstacle_update(b, a, log->h_hdr[sidx].n_points);
    if (st != CS_OK) return st;
    b->step.advance(a.do_search);
  }
  if (results && count > 0) {
    CS_CUDA(b, cudaMemcpyAsync(b->h_results.get(), b->d_results.get(), sizeof(CsDevResult) * (size_t)b->n, cudaMemcpyDeviceToHost, b->stream));
    CS_CUDA(b, cudaStreamSynchronize(b->stream));
    copy_update_results(results, b->h_results.get(), b->n);
  }  // results == NULL: fire and forget (cs_batch_sync waits)
  return CS_OK;
}

cs_status cs_batch_sync(cs_batch* b) {
  CS_CHECK_HANDLE(b);
  CS_CUDA(b, cudaStreamSynchronize(b->stream));
  return CS_OK;
}

cs_status cs_batch_get_poses(cs_batch* b, float* poses /* n_sessions * 3 */) {
  CS_CHECK_HANDLE(b);
  if (!poses) return fail(b, CS_ERR_INVALID_ARGUMENT, "null poses");
  std::vector<CsSession> tmp((size_t)b->n);
  CS_CUDA(b, cudaMemcpyAsync(tmp.data(), b->d_sess.get(), sizeof(CsSession) * (size_t)b->n, cudaMemcpyDeviceToHost, b->stream));
  CS_CUDA(b, cudaStreamSynchronize(b->stream));
  for (int j = 0; j < b->n; j++)
    for (int k = 0; k < 3; k++) poses[3 * j + k] = tmp[j].state[b->step.parity].pose[k];
  return CS_OK;
}

cs_status cs_batch_map_download(cs_batch* b, int32_t session, uint16_t* pixels) {
  CS_CHECK_HANDLE(b);
  if (!pixels || session < 0 || session >= b->n) return fail(b, CS_ERR_INVALID_ARGUMENT, "cs_batch_map_download: bad argument");
  return download_map(b, b->hs[session].map, pixels);
}

cs_status cs_batch_map_checksums(cs_batch* b, uint64_t* checksums /* n_sessions */) {
  CS_CHECK_HANDLE(b);
  if (!checksums) return fail(b, CS_ERR_INVALID_ARGUMENT, "null checksums");
  for (int j = 0; j < b->n; j++) {
    cs_status st = queue_map_checksum(b, b->hs[j].map, 148 * 4, checksums + j);
    if (st != CS_OK) return st;
  }
  CS_CUDA(b, cudaStreamSynchronize(b->stream));
  return CS_OK;
}

cs_status cs_batch_get_launch_count(cs_batch* b, uint64_t* launches) {
  if (!b || !launches) return CS_ERR_INVALID_ARGUMENT;
  *launches = b->launches;
  return CS_OK;
}

// CoreSLAMProcessor.Reset (:167-175) of every session: the batch steps all sessions with one step state, so they reset together.
cs_status cs_batch_reset(cs_batch* b) {
  CS_CHECK_HANDLE(b);
  if (b->pipe_submitted != b->pipe_collected)
    return fail(b, CS_ERR_STATE, "cs_batch_reset: submitted steps are waiting for cs_batch_collect");
  CS_CUDA(b, cudaStreamSynchronize(b->stream));  // the host mirrors are the source of the uploads below
  for (int j = 0; j < b->n; j++) reset_session(b->hs[j], &b->start_poses[3 * (size_t)j]);  // :172-174
  b->step.parity = 0;
  b->step.scan_count = 0;
  b->step.update_count = 0;
  CS_CUDA(b, cudaMemcpyAsync(b->d_sess.get(), b->hs.data(), sizeof(CsSession) * (size_t)b->n, cudaMemcpyHostToDevice, b->stream));
  cs_status st = batch_fill_maps(b);  // :169-170
  if (st != CS_OK) return st;
  CS_CUDA(b, cudaStreamSynchronize(b->stream));
  return CS_OK;
}

// ---- the sessions' ObstacleMaps (cfg.obstacle_map_size > 0; CoreSLAM/ObstacleMap.cs, CoreSLAMProcessor.cs:98, :103) ----
// session < 0: all sessions.  MaxObstacleHits applies from the next step, UnmappedObstacleHits from the next cs_batch_reset.
cs_status cs_batch_set_obstacle_params(cs_batch* b, int32_t session, int32_t unmapped_hits, int32_t max_hits) {
  CS_CHECK_HANDLE(b);
  CS_NEED_OBSTACLE(b);
  if (session >= b->n) return fail(b, CS_ERR_INVALID_ARGUMENT, "session %d out of range", session);
  if (unmapped_hits < -128 || unmapped_hits > 127) return fail(b, CS_ERR_INVALID_ARGUMENT, "UnmappedObstacleHits is an sbyte");
  if (max_hits < -128 || max_hits > 127) return fail(b, CS_ERR_INVALID_ARGUMENT, "MaxObstacleHits is an sbyte");
  for (int j = (session < 0 ? 0 : session); j < (session < 0 ? b->n : session + 1); j++) {
    b->unmapped_obstacle_hits[j] = unmapped_hits;
    b->obst[j].max_hits = max_hits;
  }
  cs_status st = batch_push_obstacles(b);  // in stream order: steps already queued keep the values they were queued with
  if (st != CS_OK) return st;
  CS_CUDA(b, cudaStreamSynchronize(b->stream));
  return CS_OK;
}

cs_status cs_batch_obstacle_map_download(cs_batch* b, int32_t session, int8_t* pixels) {
  CS_CHECK_HANDLE(b);
  CS_NEED_OBSTACLE(b);
  if (!pixels || session < 0 || session >= b->n)
    return fail(b, CS_ERR_INVALID_ARGUMENT, "cs_batch_obstacle_map_download: bad argument");
  return download_obstacle_map(b, b->obst[session], pixels);
}

cs_status cs_batch_obstacle_checksums(cs_batch* b, uint64_t* checksums /* n_sessions */) {
  CS_CHECK_HANDLE(b);
  CS_NEED_OBSTACLE(b);
  if (!checksums) return fail(b, CS_ERR_INVALID_ARGUMENT, "null checksums");
  const unsigned cells = (unsigned)b->ho.size * (unsigned)b->ho.size;
  const int sms = device_sm_count(b->device);
  unsigned blocks = (unsigned)((sms * 8 + b->n - 1) / b->n);  // about eight blocks per SM over all sessions
  if (blocks > (cells + 255) / 256) blocks = (cells + 255) / 256;
  CS_CUDA(b, cudaMemsetAsync(b->d_obst_sums.get(), 0, sizeof(unsigned long long) * (size_t)b->n, b->stream));
  cs_obstacle_checksum_kernel<<<dim3(blocks, (unsigned)b->n), 256, 0, b->stream>>>(b->d_obst.get(), b->d_obst_sums.get());
  b->launches++;
  CS_CUDA(b, cudaGetLastError());
  CS_CUDA(b, cudaMemcpyAsync(checksums, b->d_obst_sums.get(), sizeof(unsigned long long) * (size_t)b->n, cudaMemcpyDeviceToHost, b->stream));
  CS_CUDA(b, cudaStreamSynchronize(b->stream));
  return CS_OK;
}

cs_status cs_batch_get_obstacle_visits(cs_batch* b, int64_t* touched /* n_sessions */) {
  CS_CHECK_HANDLE(b);
  CS_NEED_OBSTACLE(b);
  if (!touched) return fail(b, CS_ERR_INVALID_ARGUMENT, "null out");
  static_assert(sizeof(long long) == sizeof(int64_t), "touched counters");
  CS_CUDA(b, cudaMemcpyAsync(touched, b->d_obst_touched.get(), sizeof(long long) * (size_t)b->n, cudaMemcpyDeviceToHost, b->stream));
  CS_CUDA(b, cudaStreamSynchronize(b->stream));
  return CS_OK;
}

cs_status cs_set_flags(cs_processor* h, uint32_t flags) {
  CS_CHECK_HANDLE(h);
  const uint32_t fixed = CS_FLAG_ROW_MAJOR_MAP | CS_FLAG_L2_PERSIST | CS_FLAG_DEBUG_RAYS | CS_FLAG_SEARCH_WARP | CS_FLAG_SEARCH_SLAB;
  if ((flags & fixed) != (h->cfg.flags & fixed))
    return fail(h, CS_ERR_INVALID_ARGUMENT, "map layout / L2 window / debug rays / search kernel choice are fixed at creation");
  h->cfg.flags = flags;
  int* dist = (flags & CS_FLAG_KEEP_DISTANCES) ? h->d_distances.get() : nullptr;
  h->hs.distances = dist;
  return patch_session(h, offsetof(CsSession, distances), &dist, sizeof(int*));
}

// Random 2-byte gather micro-benchmark: the measured ceiling the search kernel's lookup rate is
// compared with (SURVEY.md 8d).  Every thread issues `per_thread` independent loads at hashed cell
// indices of a table of `cells` uint16 (L2-resident when it fits), eight in flight at a time.
__global__ void cs_gather_peak_kernel(const uint16_t* __restrict__ table, unsigned mask, int per_thread,
                                      unsigned long long* __restrict__ sink) {
  unsigned tid = blockIdx.x * blockDim.x + threadIdx.x;
  unsigned long long z = cs_mix64(tid);
  unsigned acc = 0;
  for (int i = 0; i < per_thread; i += 8) {
    unsigned v[8];
#pragma unroll
    for (int k = 0; k < 8; k++) {
      z = z * 6364136223846793005ull + 1442695040888963407ull;
      v[k] = __ldg(table + ((unsigned)(z >> 33) & mask));
    }
#pragma unroll
    for (int k = 0; k < 8; k++) acc += v[k];
  }
  if (acc == 0xffffffffu) atomicAdd(sink, 1ull);
}

int32_t cs_rings_hint(int32_t size_pixels, float size_meters, float hole_width, const float* points, int32_t n_points) {
  if (size_pixels <= 0 || !points || n_points < 0) return 0;
  const float scale = (float)size_pixels / size_meters;  // HoleMap.cs:20
  return rings_hint_of(size_pixels, scale, hole_width, max_range_of(points, n_points));
}

cs_status cs_gather_peak(int32_t device, int64_t cells, int32_t per_thread, int32_t repeats, double* lookups_per_s) {
  if (!lookups_per_s || cells < 1024 || per_thread < 8 || repeats < 1) return CS_ERR_INVALID_ARGUMENT;
  if (cs_device_count() <= device) return fail(nullptr, CS_ERR_NO_DEVICE, "no such CUDA device");
  cudaSetDevice(device);
  unsigned pow2 = 1024;
  while ((int64_t)pow2 * 2 <= cells && pow2 < (1u << 30)) pow2 *= 2;
  DevBuf<uint16_t> table;
  DevBuf<unsigned long long> sink;
  Event e0, e1;
  if (alloc(table, pow2) != cudaSuccess || alloc(sink, 1) != cudaSuccess) {
    cudaGetLastError();
    return fail(nullptr, CS_ERR_OUT_OF_MEMORY, "cs_gather_peak: allocation failed");
  }
  cudaMemset(table.get(), 1, (size_t)pow2 * 2);
  cudaMemset(sink.get(), 0, 8);
  create(e0, cudaEventDefault);
  create(e1, cudaEventDefault);
  const int blocks = 148 * 8, threads = 256;
  double best = 0;
  for (int r = 0; r < repeats + 2; r++) {
    cudaEventRecord(e0.get());
    cs_gather_peak_kernel<<<blocks, threads>>>(table.get(), pow2 - 1, per_thread, sink.get());
    cudaEventRecord(e1.get());
    cudaEventSynchronize(e1.get());
    float ms = 0;
    cudaEventElapsedTime(&ms, e0.get(), e1.get());
    double rate = (double)blocks * threads * (double)(per_thread / 8 * 8) / (ms * 1e-3);
    if (r >= 2 && rate > best) best = rate;
  }
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(nullptr, CS_ERR_CUDA, "cs_gather_peak: %s", cudaGetErrorString(e));
  *lookups_per_s = best;
  return CS_OK;
}

// -----------------------------------------------------------------------------------------------------
void cs_philox_offsets(uint64_t seed, uint32_t scan_index, int32_t n, float sigma_xy, float sigma_theta, float* offsets) {
  for (int32_t i = 0; i < n; i++) cs_gauss3(seed, scan_index, (uint32_t)i, sigma_xy, sigma_theta, offsets + 3 * (size_t)i);
}

void cs_host_sincos(const float* angles, int32_t n, float* cos_out, float* sin_out) {
  for (int32_t i = 0; i < n; i++) {
    if (cos_out) cos_out[i] = cs_cosf(angles[i]);
    if (sin_out) sin_out[i] = cs_sinf(angles[i]);
  }
}

float cs_host_normalize_angle(float a) { return cs_normalize_angle(a); }

cs_status cs_device_sincos(int32_t device, const float* angles, int32_t n, float* cos_out, float* sin_out) {
  if (!angles || !cos_out || !sin_out || n <= 0) return CS_ERR_INVALID_ARGUMENT;
  if (cs_device_count() <= device) return fail(nullptr, CS_ERR_NO_DEVICE, "no such CUDA device");
  cudaSetDevice(device);
  DevBuf<float> d_in, d_c, d_s;
  size_t bytes = (size_t)n * sizeof(float);
  bool ok = alloc(d_in, (size_t)n) == cudaSuccess && alloc(d_c, (size_t)n) == cudaSuccess && alloc(d_s, (size_t)n) == cudaSuccess &&
            cudaMemcpy(d_in.get(), angles, bytes, cudaMemcpyHostToDevice) == cudaSuccess;
  if (ok) {
    cs_sincos_kernel<<<(n + 255) / 256, 256>>>(d_in.get(), n, d_c.get(), d_s.get());
    ok = cudaMemcpy(cos_out, d_c.get(), bytes, cudaMemcpyDeviceToHost) == cudaSuccess &&
         cudaMemcpy(sin_out, d_s.get(), bytes, cudaMemcpyDeviceToHost) == cudaSuccess;
  }
  if (!ok) return fail(nullptr, CS_ERR_CUDA, "cs_device_sincos: %s", cudaGetErrorString(cudaGetLastError()));
  return CS_OK;
}

}  // extern "C"

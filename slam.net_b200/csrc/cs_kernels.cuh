// cs_kernels.cuh — sm_100a kernels of the CoreSLAM scan-to-map hot path.
//
//   cs_search_kernel     CalculateDistanceSISD + MonteCarloSearch + ParallelMonteCarloSearch arg-min
//                        (CoreSLAM/CoreSLAMProcessor.cs:226-259, 624-653, 674-710)
//                        The last block to finish also runs the Update glue (:717-752: gate, searchPose,
//                        NormalizeAngle, state) and publishes the pose, so the pose leaves the device at
//                        the end of the search kernel itself.
//   cs_sort_kernel,      the slab search: the same arg-min over candidates sorted by heading (many candidates)
//   cs_search2_kernel
//   cs_setup_kernel      the same glue on its own, for steps without a search kernel that publishes
//
// The draw kernel that follows (UpdateHoleMap / ClipRay / DrawLaserRayOnHoleMap, :496-534, 320-345,
// 359-443) is cs_wedge_kernel in cs_wedge.cuh; the closed-form ray set-up it calls (cs_ray_from_point) is here.
//
// No tensor cores: nothing here is a contraction.  The search is a 2-byte gather per (candidate, point)
// out of an L2-resident map; the integration is an ordered 2-byte read-modify-write per visited cell.
// Compile with -fmad=false: every float operation below must round once, like RyuJIT's scalar SSE code.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "cs_math.h"

#define CS_TS_NO_OBSTACLE 65500  // CoreSLAMProcessor.cs:21
#define CS_TS_OBSTACLE 0         // CoreSLAMProcessor.cs:22

#define CS_GROUP_MAX 8                      // most GPUs of a candidate-split group (one NVSwitch box)
#define CS_XCHG_TIMEOUT_NS 2000000000ll     // a rank that waits this long for the others' keys gives up (searched = -1)

enum CsCandMode { CS_CAND_PHILOX = 0, CS_CAND_OFFSETS = 1, CS_CAND_ABSOLUTE = 2 };
enum CsStepMode { CS_STEP_UPDATE = 0, CS_STEP_SEARCH_ONLY = 1, CS_STEP_INTEGRATE_ONLY = 2 };

struct CsState {  // CoreSLAMProcessor.cs:34-35, 106
  float pose[3];
  float last_odo[3];
  int scan_count;
  int pad;
};

struct CsStepHeader {  // per-scan input, 48 B
  float odo[3];        // odometry pose (UPDATE) or explicit pose (SEARCH_ONLY / INTEGRATE_ONLY)
  int n_points;
  float cs[2];         // optional host (cos, sin) of the explicit pose
  int has_cs;
  int pad[5];
};

struct CsRay {  // 32 B: everything the draw loop needs to know about one ray, in closed form
  int dxc, dyc;   // clipped extents along the major / minor axis (:370-371 after the :383-385 swap)
  int a0, b0;     // pixval descends for major steps a0..b0 (:406-416); ascends from max(a0, b0+1) (:418-427)
  int incv;       // :398
  int kc;         // how many of the ascending steps take the +1 carry (:422-426)
  int nd_total;   // number of descending steps once past b0
  int flags;      // bit0 valid, bit1 steep (major axis = y), bit2 major step negative, bit3 minor step negative
};

// 16-byte form kept in global memory (every field fits: sizes <= 16384, |incv| <= 65500)
__device__ __forceinline__ int4 cs_pack_ray(const CsRay& r) {
  int4 q;
  q.x = r.dxc | (r.dyc << 14) | (r.flags << 28);
  q.y = r.a0 | ((r.b0 + 1) << 15);
  q.z = (-r.incv) | (r.nd_total << 16);
  q.w = r.kc;
  return q;
}
__device__ __forceinline__ CsRay cs_unpack_ray(const int4 q) {
  CsRay r;
  r.dxc = q.x & 0x3fff; r.dyc = (q.x >> 14) & 0x3fff; r.flags = (int)((unsigned)q.x >> 28);
  r.a0 = q.y & 0x7fff; r.b0 = ((q.y >> 15) & 0x7fff) - 1;
  r.incv = -(q.z & 0xffff); r.nd_total = (int)((unsigned)q.z >> 16);
  r.kc = q.w;
  return r;
}

struct CsDevResult {  // device twin of cs_result (include/coreslam_b200.h)
  float pose[3];
  int distance;
  int index;
  int searched;
  long long visits;
};

struct CsSession {  // one CoreSLAMProcessor, device resident
  uint16_t* map;    // HoleMap.Pixels; tiled: 8x8-cell tiles of 128 B (one line), rows of 8 cells inside, 8x2 cells per 32 B sector
  int size;         // HoleMap.Size
  int pitch_tiles;  // tiles per tile-row (tiled layout)
  float scale;      // HoleMap.Scale
  float sigma_xy, sigma_theta;
  int iters, threads, n_cand;  // n_cand = max(threads,1) * iters random candidates (+1 for searchPose)
  int quality;       // :82
  float hole_width;  // :87
  int search_begin;  // :92
  unsigned long long seed;
  CsState state[2];            // state[parity] is current; an Update writes state[parity^1] and the host flips parity
  unsigned long long key[2];   // packed (distance << 32 | flat index) arg-min; key[parity] belongs to the current step
  int4* rays;                  // packed per-ray draw parameters of the current integration: ray_copies copies of
                               // ray_stride entries each (every SM reads the copy smid % ray_copies, so the lines the
                               // whole grid wants at the same instant are spread over several L2 slices)
  int* batch_max;              // per 32 consecutive rays: largest dxc of a valid ray, -1 if none; ray_copies copies of
                               // batch_stride entries
  int ray_copies, ray_stride, batch_stride, pad1;
  unsigned long long* prep_words;  // [2 slots][ray_copies] words, 128 B apart: preparing blocks of the draw kernel that are
                                   // done; slot = step id & 1, re-armed for the next step by this step's publishing thread
  int* ray_dbg;                // optional 6 ints per ray (x1,y1,x2,y2,xp,yp), CS_FLAG_DEBUG_RAYS
  int* distances;              // optional n_cand+1
  long long* ring_cycles;      // set by cs_get_ring_cycles but read by no kernel (they record through CsStepArgs::diag);
                               // kept so that the polled words below stay where they are relative to 128-byte lines
  float cur_pose[3];           // pose the current integration draws from (Pose after :745-747)
  float cur_cs[2];             // its (cos, sin), unscaled
  unsigned search_done;        // blocks of the running search kernel that have finished
  unsigned pad0;
  // The pose the current integration draws from, published without a fence: five 8-byte words {float bits, step id},
  // each single-copy atomic — x, y, theta (Pose after :745-747), cos, sin (unscaled).  The draw kernel's blocks are
  // resident before the search ends and poll the words for their step id.
  unsigned long long ll_pose[5];
  unsigned long long pad2;
  long long visits_slot[2];    // cells written by the integration of step id & 1 = sum over valid rays of dxc+1
  unsigned ring_ticket[2];     // block tickets of the draw kernel (small scans); slot = step id & 1, re-armed for the next
                               // step by the publishing thread of this step
  // ---- scratch of the slab search (cs_sort_kernel + cs_search2_kernel; one session alone, many candidates)
  float4* s2_sorted;            // [2][s2_cap]: this step's candidates in ascending order of heading offset, as
                                // (x, y, theta [offsets or absolute pose], flat index bits); slot = CsStepArgs::s2_slot
  float4* s2_tmp;               // [s2_cap] the same entries in flat order (scratch of the running sort)
  unsigned long long* s2_meta;  // [s2_cap] heading bin << 32 | rank inside the bin (scratch of the running sort)
  unsigned long long* s2_acc;   // [s2_cap] per sorted position: cell sum | in-bounds count << 32 | clusters arrived << 49; zero between steps
  int s2_cap, pad3;
  unsigned* s2_ghist;           // [CS_SORT_BINS + 1] histogram of the multi-block sort + its arrival counter; zero between steps
  // ---- scratch of the wedge integration (cs_wedge.cuh)
  int2* w_rk;                   // per ray: (angular key as float bits, dxc or -1 for a ray that draws nothing)
  float2* w_bkey;               // per 32 consecutive rays: (smallest, largest) key of a valid ray
  int* w_top;                   // [3][w_levels * (CS_W_SECTORS + 1)]: valid rays that reach (level, key sector) and that reach each
                                // level; the thirds rotate: CsStepArgs::w_slot / w_prev / w_zero
  int w_levels, pad4;           // levels a ray of this map can reach (cs_w_level_of(size - 1) + 1)
};

struct CsStepArgs {  // by-value kernel argument; session j uses element j of every array
  const CsStepHeader* hdr; size_t hdr_stride;    // 1: one header per session, 0: every session reads hdr[0] (shared scan log)
  const float2* points;  size_t points_stride;   // stride in float2 between sessions
  const float* cand;     size_t cand_stride;     // offsets or absolute poses, 3 floats per candidate
  const float* cand_cs;                          // optional (n_cand+1)*2 host cos/sin
  CsDevResult* result;   size_t result_stride;   // where finalize writes (device or mapped host memory)
  volatile unsigned* seq_flag;                   // optional mapped-host flag, set to seq_value when the pose is out
  unsigned seq_value;
  unsigned scan_index;
  int cand_mode;   // CsCandMode
  int step_mode;   // CsStepMode
  int parity;      // state[parity]/key[parity] are read; an UPDATE step writes state[parity^1] and arms key[parity^1]
  int do_search;   // host mirror of scanCount >= PositionSearchBeginning (:726)
  int n_cand;      // random candidates evaluated this step (excludes searchPose)
  int cand_first;  // first flat index evaluated by this GPU (multi-GPU candidate split), normally 0
  int cand_count;  // number of flat indices evaluated by this GPU, normally n_cand+1
  int fuse_publish;  // search kernel: its last block runs the Update glue and publishes the pose
  int max_ring_hint; // rings the host launched blocks for, minus one
  int prep_group;    // rays prepared by each of the first blocks of the draw kernel (multiple of 32)
  int search_chunk;  // points staged in shared memory per pass of the search kernel (<= CS_SEARCH_CHUNK)
  unsigned step_id;  // nonzero, different for consecutive steps on the same session(s): tags ll_pose, selects the counter slots
  long long* visits_out;  // optional device slot that receives the visit count
  volatile unsigned* stuck_flag;  // CS_FLAG_DEBUG_BOUNDED_SPIN: mapped-host word that receives the CsStuckSite of a poll
  long long spin_ns;              // that gave up after spin_ns nanoseconds (0: polls are unbounded, the normal build of a step)
  long long* diag;        // optional diagnostics buffer (8 values per task of the draw kernel, then 8 per block of
                          // the search kernel), see cs_get_ring_cycles
  int diag_rings;         // records reserved for the draw kernel in diag
  // slab search (cs_search2_kernel): block (c, s) evaluates points [c*s2_points, ...) for sorted candidates [s*s2_slab, ...)
  int s2_points;          // points per cluster (<= CS_S2_MAX_POINTS)
  int s2_slab;            // candidates per slab (multiple of 32, = threads per block)
  int s2_slot;            // which half of CsSession::s2_sorted this step uses
  int s2_host_points;     // the host's copy of hdr.n_points (0: unknown, the slab search is not used)
  // host-owned session constants by value, so that the slab kernels' first instructions do not wait for a (cold)
  // read of the session descriptor: CsSession::map, size, pitch_tiles, scale, sigmas, seed, and the scratch pointers
  const uint16_t* s2_map;
  float4* s2_sorted;             // this step's half of CsSession::s2_sorted
  float4* s2_tmp;
  unsigned long long* s2_meta;
  unsigned long long* s2_acc;
  unsigned* s2_ghist;            // CS_SORT_BINS + 1 words, zero between steps (multi-block sort)
  unsigned long long s2_seed;
  int s2_size, s2_pitch_tiles;
  float s2_scale, s2_sigma_xy, s2_sigma_theta;
  // candidate split over a group of GPUs with the arg-min exchanged inside the search kernel (cs_group_attach): rank r's
  // table holds, per half (exchange number & 1) and rank, two words {packed key, tag}; every rank writes its key into every
  // table over peer-mapped memory and waits for the world's keys in its own
  // glue table (one session alone, slab search): entry idx = the pose and (cos, sin) an UPDATE step ends on if flat candidate
  // idx wins, as five words {step tag << 32 | float bits} (the format of CsSession::ll_pose) in a 64-byte slot.  Every block
  // of the slab search carries one extra warp that looks nothing up: at the start of the kernel it writes the entries of its
  // share of the slab's candidates.  The publishing thread then copies the winner's entry instead of running the glue
  // arithmetic (candidate pose, NormalizeAngle, cos, sin: ~1000 dependent instructions of cold code) at the very end of the
  // step's critical path.  An entry whose tags are not this step's is ignored and the glue computed as before (the winner
  // of a candidate-split group may be another rank's candidate): nothing depends on timing.
  unsigned long long* spec;      // nullptr: no table
  int xchg_world;                // 0 / 1: no exchange
  int xchg_rank;
  unsigned xchg_seq;             // exchange number, the same on every rank
  int xchg_serial_draw;          // 1: another rank shares this device: the draw kernel must not be resident during the exchange
  unsigned long long* xchg_peer[CS_GROUP_MAX];
  int w_slot;                    // which third of CsSession::w_top this step counts into (rotates per drawn step)
  int w_prev;                    // the third the previous drawn step counted into (its counts size this step's wedges); -1: none
  int w_zero;                    // the third the next drawn step will count into (zeroed by this step)
  int w_prefetch;                // the map around the pose is pulled into L2 — 1: by the candidate sort, 2: by the draw kernel's
                                 // blocks while they wait
  int empty_cloud;               // 1: the scan has no points and the step searches: no search kernel ran, the arg-min is
                                 // (int.MaxValue, searchPose) by definition (:251-258, :630-648)
  int s2_batch;                  // 1: a batch of sessions (session = blockIdx.z of the search, blockIdx.y of the sort): the values
                                 // above come from CsSession instead, hdr / points / cand / result are strided per session
};

// ---------------------------------------------------------------------------------------------------
// map addressing
// ---------------------------------------------------------------------------------------------------
template <bool TILED>
__device__ __forceinline__ uint32_t cs_cell_offset(int x, int y, int size, int pitch_tiles) {
  if (TILED) {
    // tile (y>>3, x>>3) * 64 + (y&7)*8 + (x&7), written so that it costs two AND, one shift-add and two multiply-adds:
    // x + 7*(x & ~7) = (x&7) + 64*(x>>3);  8*y + (y & ~7)*(8*pitch - 8) = 64*pitch*(y>>3) + 8*(y&7)
    const uint32_t ux = (uint32_t)x, uy = (uint32_t)y;
    const uint32_t xx = (ux & ~7u) * 7u + ux;
    return (uy & ~7u) * ((uint32_t)pitch_tiles * 8u - 8u) + (uy << 3) + xx;
  } else {
    return (uint32_t)y * (uint32_t)size + (uint32_t)x;
  }
}

// programmatic dependent launch: a kernel launched with the stream-serialization attribute may start while its
// predecessor drains; it must not touch the predecessor's results before cs_pdl_wait()
__device__ __forceinline__ void cs_pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void cs_pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// diagnostics only (a.diag != nullptr): wall-clock stamps and the SM a block ran on
__device__ __forceinline__ long long cs_globaltimer() { long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t) :: "memory"); return t; }
__device__ __forceinline__ int cs_smid() { int v; asm volatile("mov.u32 %0, %%smid;" : "=r"(v)); return v; }

// Bounded polls (CS_FLAG_DEBUG_BOUNDED_SPIN).  The kernels of a step talk to each other through words they poll (the pose
// out of the search kernel, the arrival count of the preparing blocks, the hand-off word of a contested cell); the polls
// rely on co-residency arguments (DESIGN.md section 4) and normally have no way out.  With CsStepArgs::spin_ns set every
// poll looks at the clock once in 1024 turns, gives up after spin_ns, and reports where through the mapped-host word: the
// block leaves the kernel (its partners' polls then run out too, so the grid drains), and the host turns the word into
// CS_ERR_CUDA on the handle's next call instead of a hang.
enum CsStuckSite { CS_STUCK_NONE = 0, CS_STUCK_POSE = 1, CS_STUCK_RAYS = 2, CS_STUCK_HANDOFF = 3 };
struct CsSpin {
  long long t0 = 0;
  unsigned turns = 0;
  __device__ __forceinline__ bool expired(const CsStepArgs& a, unsigned site) {
    if (a.spin_ns == 0 || (++turns & 1023u) != 0u) return false;
    const long long t = cs_globaltimer();
    if (t0 == 0) { t0 = t; return false; }
    if (t - t0 < a.spin_ns) return false;
    if (a.stuck_flag) { *a.stuck_flag = site | ((unsigned)blockIdx.x << 8); __threadfence_system(); }
    return true;
  }
};
#define CS_DIAG_SEARCH_BLOCKS 8192  // search-kernel timeline records kept after the per-ring records

// wrapping int32 arithmetic (C# unchecked)
__device__ __forceinline__ int cs_wadd(int a, int b) { return (int)((unsigned)a + (unsigned)b); }
__device__ __forceinline__ int cs_wsub(int a, int b) { return (int)((unsigned)a - (unsigned)b); }
__device__ __forceinline__ int cs_wmul(int a, int b) { return (int)((unsigned)a * (unsigned)b); }
__device__ __forceinline__ int cs_wabs(int a) { return a < 0 ? cs_wsub(0, a) : a; }
__device__ __forceinline__ int cs_sign(int a) { return (a > 0) - (a < 0); }
__device__ __forceinline__ int cs_wdiv(int a, int b) { return (b == 0 || (a == (int)0x80000000 && b == -1)) ? 0 : a / b; }

// ---------------------------------------------------------------------------------------------------
// candidate enumeration: flat index 0 = searchPose, 1 + t*I + i = thread t's i-th candidate
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ void cs_search_pose(const CsSession& S, const CsStepHeader& h, const CsStepArgs& a,
                                               float sp[3]) {
  if (a.step_mode == CS_STEP_UPDATE) {
    const CsState& st = S.state[a.parity];
#pragma unroll
    for (int k = 0; k < 3; k++) sp[k] = __fadd_rn(st.pose[k], __fsub_rn(h.odo[k], st.last_odo[k]));  // :728
  } else {
    sp[0] = h.odo[0]; sp[1] = h.odo[1]; sp[2] = h.odo[2];
  }
}

// Pulls the part of the map a scan can reach into L2: the tiles within `max_ring_hint` (+ the reach of the search) of the
// pose the step starts from, one 32-byte sector per iteration, thread t of nt.  Called in the shadow of other work (the
// candidate sort, the wait for the pose); where the map is L2-resident already the prefetches hit.  The state may be one step
// old when this runs ahead of the previous step's end: good enough for a prefetch.
__device__ __forceinline__ void cs_prefetch_disc(const CsSession& S, const CsStepHeader& hdr, const CsStepArgs& a, int t, int nt) {
  float sp[3];
  if (a.step_mode == CS_STEP_UPDATE && a.do_search) cs_search_pose(S, hdr, a, sp);
  else { sp[0] = hdr.odo[0]; sp[1] = hdr.odo[1]; sp[2] = hdr.odo[2]; }
  const int size = S.size, pitch_tiles = S.pitch_tiles;
  const float scale = S.scale;
  const int cx = cs_cvt_i32(__fmul_rn(sp[0], scale)), cy = cs_cvt_i32(__fmul_rn(sp[1], scale));
  const int R = a.max_ring_hint + 16 + (int)(4.0f * S.sigma_xy * scale);
  if (!(cx > -R && cy > -R && cx < size + R && cy < size + R)) return;  // (NaN / far-off poses: nothing to fetch)
  const int tx0 = max(cx - R, 0) >> 3, tx1 = min(cx + R, size - 1) >> 3;
  const int ty0 = max(cy - R, 0) >> 3, ty1 = min(cy + R, size - 1) >> 3;
  const int tw = tx1 - tx0 + 1, th = ty1 - ty0 + 1;
  const long long r2 = (long long)(R + 8) * (R + 8);
  // (Plain loads whose results nobody uses, one per 32-byte sector: `prefetch.global.L2` changed nothing measurable —
  // cfg2 flushed 42.6 us per step with it, 42.5 without — while loads from the same idle threads take the step to 41.7.)
  for (int i = t; i < tw * th * 4; i += nt) {
    const int tile = i >> 2, ty = ty0 + tile / tw, tx = tx0 + tile % tw;
    const long long dx = tx * 8 + 4 - cx, dy = ty * 8 + 4 - cy;
    if (dx * dx + dy * dy <= r2) {
      const uint16_t* sector = S.map + ((size_t)ty * pitch_tiles + tx) * 64 + (i & 3) * 16;
      unsigned unused;
      asm volatile("ld.global.cg.u32 %0, [%1];" : "=r"(unused) : "l"(sector));
    }
  }
}

__device__ __forceinline__ void cs_candidate_pose(const CsSession& S, const CsStepArgs& a, const float* cand,
                                                  const float sp[3], int idx, float pose[3]) {
  if (idx == 0) {
    pose[0] = sp[0]; pose[1] = sp[1]; pose[2] = sp[2];
    return;
  }
  if (a.cand_mode == CS_CAND_ABSOLUTE) {
    const float* p = cand + 3 * (size_t)(idx - 1);
    pose[0] = p[0]; pose[1] = p[1]; pose[2] = p[2];
    return;
  }
  float off[3];
  if (a.cand_mode == CS_CAND_OFFSETS) {
    const float* p = cand + 3 * (size_t)(idx - 1);
    off[0] = p[0]; off[1] = p[1]; off[2] = p[2];
  } else {
    cs_gauss3(S.seed, a.scan_index, (uint32_t)(idx - 1), S.sigma_xy, S.sigma_theta, off);
  }
  pose[0] = __fadd_rn(sp[0], off[0]);  // :635-637
  pose[1] = __fadd_rn(sp[1], off[1]);
  pose[2] = __fadd_rn(sp[2], off[2]);
}

// ---------------------------------------------------------------------------------------------------
// ray set-up (ClipRay :320-345 and the prologue of DrawLaserRayOnHoleMap :361-402)
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool cs_clip_ray(int size, int& xyc, int& yxc, int xy, int yx) {
  if (xyc < 0) {
    if (xyc == xy) return false;
    yxc = cs_wadd(yxc, cs_wdiv(cs_wmul(cs_wsub(yxc, yx), cs_wsub(0, xyc)), cs_wsub(xyc, xy)));
    xyc = 0;
  }
  if (xyc >= size) {
    if (xyc == xy) return false;
    yxc = cs_wadd(yxc, cs_wdiv(cs_wmul(cs_wsub(yxc, yx), cs_wsub(size - 1, xyc)), cs_wsub(xyc, xy)));
    xyc = size - 1;
  }
  return true;
}

__device__ __forceinline__ CsRay cs_make_ray(int size, int x1, int y1, int x2, int y2, int xp, int yp) {
  CsRay r;
  r.dxc = 0; r.dyc = 0; r.a0 = 0; r.b0 = -1; r.incv = 0; r.kc = 0; r.nd_total = 0; r.flags = 0;
  int x2c = x2, y2c = y2;
  if (!cs_clip_ray(size, x2c, y2c, x1, y1)) return r;  // :365
  if (!cs_clip_ray(size, y2c, x2c, y1, x1)) return r;  // :366
  int dx = cs_wabs(cs_wsub(x2, x1)), dy = cs_wabs(cs_wsub(y2, y1));        // :368-369
  int dxc = cs_wabs(cs_wsub(x2c, x1)), dyc = cs_wabs(cs_wsub(y2c, y1));    // :370-371
  int sx = cs_sign(cs_wsub(x2, x1)), sy = cs_sign(cs_wsub(y2, y1));        // :372-373
  int D, smaj, smin;
  bool steep;
  if (dx > dy) {  // :377
    steep = false;
    D = cs_wabs(cs_wsub(xp, x2));
    smaj = sx; smin = sy;
  } else {
    steep = true;
    dx = dy;
    int t = dxc; dxc = dyc; dyc = t;
    D = cs_wabs(cs_wsub(yp, y2));
    smaj = sy; smin = sx;
  }
  if (D == 0) return r;  // :389-392
  // the walk below never leaves the box [start, clipped end]; reject anything a wrapped clip produced
  if (dxc >= size || dyc >= size || D < 0) return r;
  const int value = CS_TS_OBSTACLE;
  int incv = (value - CS_TS_NO_OBSTACLE) / D;                     // :398
  int rem = -(value - CS_TS_NO_OBSTACLE - cs_wmul(D, incv));      // -incerrorv >= 0, :399
  // zone thresholds in 64 bit: descending while t2 < x <= t1, ascending while x > t2 and x > t1 (:406-408)
  long long t2 = (long long)cs_wsub(dx, cs_wmul(2, D)) + 1;       // first x with x > dx - 2*derrorv
  long long t1 = (long long)cs_wsub(dx, D);
  long long a0 = t2 > 0 ? t2 : 0;
  long long lim = (long long)size + 1;                            // beyond any x <= dxc
  if (a0 > lim) a0 = lim;
  if (t1 > lim) t1 = lim;
  if (t1 < -1) t1 = -1;
  long long nd_total = t1 - a0 + 1;
  if (nd_total < 0) nd_total = 0;
  long long e0 = (long long)(D / 2) - nd_total * (long long)rem;  // errorv entering the ascending zone (:397, :411)
  long long need = -e0 - (long long)rem;
  long long kc = 0;
  if (need > 0) {
    const long long knum = need + (long long)rem + (long long)D - 1, kden = (long long)rem + (long long)D;
    kc = (knum < 0x7fffffffLL) ? (long long)((unsigned)knum / (unsigned)kden) : knum / kden;  // 32-bit in practice
  }
  if (kc > lim) kc = lim;
  r.dxc = dxc; r.dyc = dyc;
  r.a0 = (int)a0; r.b0 = (int)t1;
  r.incv = incv; r.kc = (int)kc; r.nd_total = (int)nd_total;
  r.flags = 1 | (steep ? 2 : 0) | (smaj < 0 ? 4 : 0) | (smin < 0 ? 8 : 0);
  return r;
}

// pixval written at major step x of ray r (closed form of :402-428)
__device__ __forceinline__ int cs_ray_pixval(const CsRay& r, int x) {
  if (x <= r.b0) {
    int nd = x - r.a0 + 1;
    nd = nd > 0 ? nd : 0;
    return CS_TS_NO_OBSTACLE + nd * r.incv;
  }
  int c0 = max(r.a0, r.b0 + 1);
  if (x < c0) return CS_TS_NO_OBSTACLE;
  int j = x - c0 + 1;
  return CS_TS_NO_OBSTACLE + (r.nd_total - j) * r.incv + min(j, r.kc);
}

// minor-axis offset after x major steps (closed form of the Bresenham error walk :394-396, 433-441)
__device__ __forceinline__ int cs_ray_minor(const CsRay& r, int x) {
  if (x == 0) return 0;
  // floor(num / den) with num < 2^30, den <= 2^15: a float estimate is within +-1, fixed up exactly
  const int num = 2 * r.dyc * x + r.dxc - 1;
  const int den = 2 * r.dxc;
  int q = __float2int_rz(__fmul_rz(__int2float_rz(num), __frcp_rz(__int2float_rz(den))));
  int rem = num - q * den;
  if (rem < 0) { q--; rem += den; }
  if (rem >= den) q++;
  return min(q, x);
}



// ---------------------------------------------------------------------------------------------------
// Update glue (:717-752) — run by ONE thread.  cs_glue_pose decodes the arg-min, applies the search gate
// and normalises the angle; cs_glue_publish stores state / result / flag and leaves the pose and its
// (cos, sin) in the session's cur_pose / cur_cs for the kernels that follow.
// ---------------------------------------------------------------------------------------------------
struct CsGlue {
  float pose[3];
  float cs[2];
  int dist, index, searched;
};

// pure part: which pose does this step end on (no side effects)
__device__ __forceinline__ void cs_glue_pose(CsSession& S, const CsStepHeader& hdr, const CsStepArgs& a, const float* cand,
                                             unsigned long long key, CsGlue& g) {
  g.dist = 2147483647; g.index = 0; g.searched = 0;
  bool have_cs = false;
  if (a.step_mode == CS_STEP_INTEGRATE_ONLY) {
    g.pose[0] = hdr.odo[0]; g.pose[1] = hdr.odo[1]; g.pose[2] = hdr.odo[2];
    if (hdr.has_cs) { have_cs = true; g.cs[0] = hdr.cs[0]; g.cs[1] = hdr.cs[1]; }
  } else {
    float sp[3];
    cs_search_pose(S, hdr, a, sp);
    if (a.do_search) {
      g.dist = (int)(unsigned)(key >> 32);
      g.index = (int)(unsigned)(key & 0xffffffffu);
      g.searched = 1;
      cs_candidate_pose(S, a, cand, sp, g.index, g.pose);
    } else {
      g.pose[0] = hdr.odo[0]; g.pose[1] = hdr.odo[1]; g.pose[2] = hdr.odo[2];  // :742
    }
    if (a.step_mode == CS_STEP_UPDATE) g.pose[2] = cs_normalize_angle(g.pose[2]);  // :746
  }
  if (!have_cs) { g.cs[0] = cs_cosf(g.pose[2]); g.cs[1] = cs_sinf(g.pose[2]); }
}

// side effects: processor state, arg-min re-arm, result record + flag, session scratch for the integration
__device__ __forceinline__ void cs_glue_publish(CsSession& S, const CsStepHeader& hdr, const CsStepArgs& a,
                                                CsDevResult* result, const CsGlue& g, long long* d = nullptr) {
  // device-side consumers first: the draw kernel of this step is already resident and polls these words (nothing it reads
  // besides them is written below; the state is for the next step, which a kernel boundary orders behind this one)
  {
    const unsigned long long tag = (unsigned long long)a.step_id << 32;
    volatile unsigned long long* ll = S.ll_pose;
    ll[0] = tag | __float_as_uint(g.pose[0]);
    ll[1] = tag | __float_as_uint(g.pose[1]);
    ll[2] = tag | __float_as_uint(g.pose[2]);
    ll[3] = tag | __float_as_uint(g.cs[0]);
    ll[4] = tag | __float_as_uint(g.cs[1]);
  }
  if (d) d[2] = cs_globaltimer();
  if (a.step_mode == CS_STEP_UPDATE) {
    const CsState& st0 = S.state[a.parity];
    CsState& st1 = S.state[a.parity ^ 1];
    st1.pose[0] = g.pose[0]; st1.pose[1] = g.pose[1]; st1.pose[2] = g.pose[2];                   // :747
    st1.last_odo[0] = hdr.odo[0]; st1.last_odo[1] = hdr.odo[1]; st1.last_odo[2] = hdr.odo[2];   // :745
    st1.scan_count = st0.scan_count + (a.do_search ? 0 : 1);                                     // :741
    S.key[a.parity ^ 1] = ~0ull;  // arm the next step's arg-min
  } else if (a.step_mode == CS_STEP_SEARCH_ONLY) {
    S.key[a.parity] = ~0ull;  // re-arm in place
  }
  S.cur_pose[0] = g.pose[0]; S.cur_pose[1] = g.pose[1]; S.cur_pose[2] = g.pose[2];
  S.cur_cs[0] = g.cs[0]; S.cur_cs[1] = g.cs[1];
  // re-arm the NEXT step's counters (kernel boundaries order this before that step's draw kernel; this step's
  // were re-armed by the previous step's publisher, or are zero from the start)
  {
    const unsigned nslot = (a.step_id + 1u) & 1u;
    S.ring_ticket[nslot] = 0u;
    S.visits_slot[nslot] = 0;
    for (int c = 0; c < S.ray_copies; c++) S.prep_words[((size_t)nslot * S.ray_copies + c) * 16] = 0ull;
  }
  if (result) {
    result->pose[0] = g.pose[0]; result->pose[1] = g.pose[1]; result->pose[2] = g.pose[2];
    result->distance = g.dist;
    result->index = g.index;
    result->searched = g.searched;
    result->visits = 0;
    if (a.seq_flag) {
      __threadfence_system();
      *a.seq_flag = a.seq_value;
    }
  }
}

// The pose-dependent constants of UpdateHoleMap (:499-512), shared by every ray of the scan.
struct CsRayFrame {
  float px, py, c, s, hw, scale;
  int x1, y1, size;
  bool on_map;
};
__device__ __forceinline__ CsRayFrame cs_ray_frame(const CsSession& S, const float pose[3], const float cs[2]) {
  CsRayFrame f;
  f.scale = S.scale;
  f.size = S.size;
  f.px = __fadd_rn(__fmul_rn(pose[0], f.scale), 0.5f);  // :499
  f.py = __fadd_rn(__fmul_rn(pose[1], f.scale), 0.5f);  // :500
  f.c = __fmul_rn(cs[0], f.scale);                       // :501
  f.s = __fmul_rn(cs[1], f.scale);                       // :502
  f.x1 = cs_cvt_i32(f.px); f.y1 = cs_cvt_i32(f.py);      // :505-506
  f.on_map = !(f.x1 < 0 || f.x1 >= f.size || f.y1 < 0 || f.y1 >= f.size);  // :509-512
  f.hw = S.hole_width;
  return f;
}

// One ray of UpdateHoleMap (:517-530) + ClipRay + the prologue of DrawLaserRayOnHoleMap; d6 (optional) receives
// (x1,y1,x2,y2,xp,yp).
__device__ __forceinline__ CsRay cs_ray_from_point(const CsRayFrame& f, const float2 p, int* d6) {
  CsRay r;
  r.dxc = 0; r.dyc = 0; r.a0 = 0; r.b0 = -1; r.incv = 0; r.kc = 0; r.nd_total = 0; r.flags = 0;
  int x2 = 0, y2 = 0, xp = 0, yp = 0;
  if (f.on_map) {
    float x2p = __fsub_rn(__fmul_rn(f.c, p.x), __fmul_rn(f.s, p.y));  // :519
    float y2p = __fadd_rn(__fmul_rn(f.s, p.x), __fmul_rn(f.c, p.y));  // :520
    xp = cs_cvt_i32(__fadd_rn(f.px, x2p));                            // :521
    yp = cs_cvt_i32(__fadd_rn(f.py, y2p));                            // :522
    float dist = __fsqrt_rn(__fadd_rn(__fmul_rn(x2p, x2p), __fmul_rn(y2p, y2p)));  // :524
    float add = __fdiv_rn(__fdiv_rn(__fmul_rn(f.hw, f.scale), 2.0f), dist);        // :525
    float k1 = __fadd_rn(1.0f, add);
    x2p = __fmul_rn(x2p, k1);                                         // :527
    y2p = __fmul_rn(y2p, k1);                                         // :528
    x2 = cs_cvt_i32(__fadd_rn(f.px, x2p));                            // :529
    y2 = cs_cvt_i32(__fadd_rn(f.py, y2p));                            // :530
    r = cs_make_ray(f.size, f.x1, f.y1, x2, y2, xp, yp);
  }
  if (d6) { d6[0] = f.x1; d6[1] = f.y1; d6[2] = x2; d6[3] = y2; d6[4] = xp; d6[5] = yp; }
  return r;
}

// The one exchange step of the candidate split (SURVEY 8e), run by the publishing thread: this rank's packed arg-min goes
// into every rank's table (8-byte stores over NVLink / peer-mapped memory, key first, then the tag behind a system fence),
// then the thread waits until its own table holds the world's keys of this exchange and takes their minimum — the same
// value on every rank.  Two halves by exchange parity: a rank that runs ahead writes the next exchange into the other half.
__device__ __forceinline__ unsigned long long cs_exchange_min(const CsStepArgs& a, unsigned long long key, bool& timed_out) {
  const size_t half = (size_t)(a.xchg_seq & 1u) * CS_GROUP_MAX * 2;
  const unsigned long long tag = 0x100000000ull | (unsigned long long)a.xchg_seq;  // never 0
  for (int p = 0; p < a.xchg_world; p++) {
    volatile unsigned long long* slot = a.xchg_peer[p] + half + (size_t)a.xchg_rank * 2;
    slot[0] = key;
  }
  __threadfence_system();
  for (int p = 0; p < a.xchg_world; p++) {
    volatile unsigned long long* slot = a.xchg_peer[p] + half + (size_t)a.xchg_rank * 2;
    slot[1] = tag;
  }
  volatile unsigned long long* mine = a.xchg_peer[a.xchg_rank] + half;
  unsigned long long best = ~0ull;
  const long long t0 = cs_globaltimer();
  for (int r = 0; r < a.xchg_world; r++) {
    while (mine[2 * r + 1] != tag) {
      if (cs_globaltimer() - t0 > CS_XCHG_TIMEOUT_NS) { timed_out = true; return key; }
    }
    __threadfence_system();
    best = min(best, mine[2 * r]);
  }
  return best;
}

// Glue + publish by one thread (the rays are prepared by the first blocks of the draw kernel).
__device__ __forceinline__ void cs_publish(CsSession& S, const CsStepHeader& hdr, const CsStepArgs& a, const float* cand,
                                           CsDevResult* result, bool have_guess = false, unsigned long long guess = 0ull) {
  long long* d = a.diag ? a.diag + ((size_t)a.diag_rings + CS_DIAG_SEARCH_BLOCKS - 1) * 8 : nullptr;  // (diagnostics: one session)
  if (d) d[0] = cs_globaltimer();
  const bool need_key = a.step_mode != CS_STEP_INTEGRATE_ONLY && a.do_search;
  // the winner's entry of the glue table (see CsStepArgs::spec): fetched for the arg-min as this thread last saw it — almost
  // always the final one — together with the read of the final key, and again only if the two differ
  const bool use_table = a.spec && need_key && a.step_mode == CS_STEP_UPDATE;
  unsigned long long w[5] = {0ull, 0ull, 0ull, 0ull, 0ull};
  unsigned widx = 0xffffffffu;
  if (use_table && have_guess) {
    widx = (unsigned)(guess & 0xffffffffull);
    const unsigned long long* e = a.spec + (size_t)widx * 8;
#pragma unroll
    for (int i = 0; i < 5; i++) w[i] = __ldcg(e + i);
  }
  unsigned long long key = 0ull;
  if (need_key) key = a.empty_cloud ? (0x7fffffffull << 32) : atomicAdd(&S.key[a.parity], 0ull);  // L2 read: sees every block's atomicMin
  bool timed_out = false;
  const bool exchange = need_key && a.xchg_world > 1 && !a.empty_cloud;
  if (exchange) key = cs_exchange_min(a, key, timed_out);
  CsGlue g;
  bool from_table = false;
  if (use_table) {
    if ((unsigned)(key & 0xffffffffull) != widx) {
      const unsigned long long* e = a.spec + (size_t)(unsigned)(key & 0xffffffffull) * 8;
#pragma unroll
      for (int i = 0; i < 5; i++) w[i] = __ldcg(e + i);
    }
    const unsigned long long tag = (unsigned long long)a.step_id << 32;
    from_table = true;
#pragma unroll
    for (int i = 0; i < 5; i++) from_table = from_table && (w[i] & 0xffffffff00000000ull) == tag;
    if (from_table) {
      g.pose[0] = __uint_as_float((unsigned)w[0]); g.pose[1] = __uint_as_float((unsigned)w[1]); g.pose[2] = __uint_as_float((unsigned)w[2]);
      g.cs[0] = __uint_as_float((unsigned)w[3]); g.cs[1] = __uint_as_float((unsigned)w[4]);
      g.dist = (int)(unsigned)(key >> 32); g.index = (int)(unsigned)(key & 0xffffffffu); g.searched = 1;
    }
  }
  if (from_table) {
  } else if (have_guess && need_key && !exchange) {
    // The arg-min as this thread last saw it is almost always the final one: the glue arithmetic runs on it while
    // the read above is in flight, and is redone only if the final key differs.
    cs_glue_pose(S, hdr, a, cand, guess, g);
    if (key != guess) cs_glue_pose(S, hdr, a, cand, key, g);
  } else {
    cs_glue_pose(S, hdr, a, cand, key, g);
  }
  if (d) { d[1] = cs_globaltimer(); d[4] = from_table ? 1 : 0; }
  if (timed_out) g.searched = -1;  // the host turns this into CS_ERR_NCCL: a rank of the group never delivered its key
  cs_glue_publish(S, hdr, a, result, g, d);
  if (d) d[3] = cs_globaltimer();
}

// ---------------------------------------------------------------------------------------------------
// search: one warp per candidate pose, lanes stride over the scan in 32-point strips
// ---------------------------------------------------------------------------------------------------
#define CS_SEARCH_WARPS 8     // most warps (= candidates) per block; the host picks 2, 4 or 8 (see cs_search_warps)
#define CS_SEARCH_CHUNK 2048  // most points staged in shared memory per pass (16 KB); dynamic: 8 B x min(P, chunk)

template <bool TILED>
__global__ void __launch_bounds__(CS_SEARCH_WARPS * 32)
cs_search_kernel(CsSession* __restrict__ sessions, CsStepArgs a) {
  extern __shared__ float4 cs_search_smem[];
  float2* s_pts = reinterpret_cast<float2*>(cs_search_smem);  // a.search_chunk points
  __shared__ unsigned long long s_key[CS_SEARCH_WARPS];
  const int nwarps = blockDim.x >> 5;
  const int chunk = a.search_chunk;

  // This grid depends on the previous step's draw kernel (cs_pdl_wait below); the next kernel of this step may
  // become resident once every block here is past that wait.
  long long* tl = nullptr;  // timeline record of this block (diagnostics)
  if (a.diag && blockIdx.y == 0 && blockIdx.x < CS_DIAG_SEARCH_BLOCKS && threadIdx.x == 0) {
    tl = a.diag + ((size_t)a.diag_rings + blockIdx.x) * 8;
    tl[0] = cs_smid(); tl[1] = cs_globaltimer(); tl[7] = 0;
  }
  const int sj = blockIdx.y;
  CsSession& S = sessions[sj];
  const CsStepHeader& hdr = a.hdr[(size_t)sj * a.hdr_stride];
  const float2* __restrict__ points = a.points + (size_t)sj * a.points_stride;
  const float* cand = a.cand ? a.cand + (size_t)sj * a.cand_stride : nullptr;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int local = blockIdx.x * nwarps + warp;
  const int idx = a.cand_first + local;  // flat candidate index
  const bool valid = local < a.cand_count;

  // ---- everything that does not depend on the previous step goes first: the step's inputs (scan, header,
  // candidate table) were uploaded before the kernels in front, and size / scale / seed / sigmas are host-owned
  // constants.  When this grid becomes resident early (programmatic dependent launch) all of it overlaps the tail
  // of the previous step's draw kernel.
  const int P = hdr.n_points;
  const int size = S.size, pitch_tiles = S.pitch_tiles;
  const uint16_t* __restrict__ map = S.map;
  const float scale = S.scale;
  {  // first chunk of the scan -> shared memory, asynchronously (two points per 16-byte copy).  Through L1 (.ca):
     // every block of the grid reads the same few KB, and the blocks of one SM should share one L2 fetch.
    const int n0 = min(chunk, P);
    const float4* src4 = reinterpret_cast<const float4*>(points);
    const unsigned dst = (unsigned)__cvta_generic_to_shared(s_pts);
    for (int i = threadIdx.x; i < (n0 >> 1); i += blockDim.x)
      asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(dst + 16u * (unsigned)i), "l"(src4 + i) : "memory");
    asm volatile("cp.async.commit_group;" ::: "memory");
    if ((n0 & 1) && threadIdx.x == 0) s_pts[n0 - 1] = points[n0 - 1];
  }
  float off[3] = {0.f, 0.f, 0.f};  // candidate offset (or absolute pose) of this warp
  float ct = 0.f, st = 0.f;
  if (valid) {
    if (idx > 0) {
      if (a.cand_mode == CS_CAND_PHILOX) {
        cs_gauss3(S.seed, a.scan_index, (uint32_t)(idx - 1), S.sigma_xy, S.sigma_theta, off);
      } else {
        const float* p = cand + 3 * (size_t)(idx - 1);
        off[0] = p[0]; off[1] = p[1]; off[2] = p[2];
      }
    }
    if (a.cand_cs) {
      ct = a.cand_cs[2 * (size_t)idx];
      st = a.cand_cs[2 * (size_t)idx + 1];
    }
  }

  cs_pdl_wait();  // the previous step (its draw kernel: map, and through it the search kernel: state) is complete
  // Only now may this step's draw kernel become resident: it does not wait for this grid as a whole but polls
  // counters that the previous step's publishing thread re-armed, so it must not run ahead of that step's end.
  cs_pdl_launch_dependents();
  if (tl) tl[2] = cs_globaltimer();

  float px = 0.f, py = 0.f, c = 0.f, s = 0.f;
  if (valid) {
    float sp[3], pose[3];
    cs_search_pose(S, hdr, a, sp);
    if (idx == 0) {
      pose[0] = sp[0]; pose[1] = sp[1]; pose[2] = sp[2];
    } else if (a.cand_mode == CS_CAND_ABSOLUTE) {
      pose[0] = off[0]; pose[1] = off[1]; pose[2] = off[2];
    } else {
      pose[0] = __fadd_rn(sp[0], off[0]);  // :635-637
      pose[1] = __fadd_rn(sp[1], off[1]);
      pose[2] = __fadd_rn(sp[2], off[2]);
    }
    if (!a.cand_cs) {
      ct = cs_cosf(pose[2]);
      st = cs_sinf(pose[2]);
    }
    px = __fadd_rn(__fmul_rn(pose[0], scale), 0.5f);  // :232
    py = __fadd_rn(__fmul_rn(pose[1], scale), 0.5f);  // :233
    c = __fmul_rn(ct, scale);                         // :234
    s = __fmul_rn(st, scale);                         // :235
  }

  unsigned sum = 0;  // <= 65535 * 65536 < 2^32 (max_points <= 65536)
  unsigned nb = 0;
  for (int base = 0; base < P; base += chunk) {
    const int n = min(chunk, P - base);
    if (base == 0) {
      asm volatile("cp.async.wait_group 0;" ::: "memory");
      __syncthreads();
    } else {
      __syncthreads();
      // vectorised staging: two points per 16-byte load
      const float4* src4 = reinterpret_cast<const float4*>(points + base);
      float4* dst4 = reinterpret_cast<float4*>(s_pts);
      for (int i = threadIdx.x; i < (n >> 1); i += blockDim.x) dst4[i] = __ldg(src4 + i);
      if ((n & 1) && threadIdx.x == 0) s_pts[n - 1] = points[base + n - 1];
      __syncthreads();
    }
    if (tl && base == 0) tl[3] = cs_globaltimer();
    if (valid) {
#pragma unroll 8
      for (int i = lane; i < n; i += 32) {
        const float2 p = s_pts[i];
        // :240-241, left-associative, one rounding per operation
        float fx = __fsub_rn(__fadd_rn(px, __fmul_rn(c, p.x)), __fmul_rn(s, p.y));
        float fy = __fadd_rn(__fadd_rn(py, __fmul_rn(s, p.x)), __fmul_rn(c, p.y));
        // (int) cast + bounds test (:244).  fmaxf drops NaN to -2 (out of bounds, like cvttss2si's
        // 0x80000000); +overflow saturates to INT_MAX, also out of bounds.
        int x = __float2int_rz(fmaxf(fx, -2.0f));
        int y = __float2int_rz(fmaxf(fy, -2.0f));
        bool in = ((unsigned)x < (unsigned)size) && ((unsigned)y < (unsigned)size);
        if (in) {
          sum += (unsigned)__ldg(map + cs_cell_offset<TILED>(x, y, size, pitch_tiles));  // :246
          nb++;
        }
      }
    }
  }

#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    sum += __shfl_xor_sync(0xffffffffu, sum, o);
    nb += __shfl_xor_sync(0xffffffffu, nb, o);
  }

  unsigned long long key = ~0ull;
  if (valid) {
    int d = nb > 0 ? (int)(((unsigned long long)sum * 1024ull) / (unsigned long long)P) : 2147483647;  // :251-258
    key = ((unsigned long long)(unsigned)d << 32) | (unsigned)idx;
    if (lane == 0 && S.distances) S.distances[idx] = d;
  }
  if (tl) tl[4] = cs_globaltimer();  // warp 0 is through its candidate
  if (lane == 0) s_key[warp] = key;
  __syncthreads();
  if (tl) tl[5] = cs_globaltimer();    // every warp of the block is
  if (threadIdx.x != 0) return;
  unsigned long long k = s_key[0];
  for (int w = 1; w < nwarps; w++) k = min(k, s_key[w]);
  unsigned long long seen = ~0ull;
  if (k != ~0ull) seen = atomicMin(&S.key[a.parity], k);
  if (!a.fuse_publish) return;
  // ---- the last block to finish owns the complete arg-min: Update glue, pose out.  Every block counts itself
  // after its atomicMin is performed (fence); the one that sees the full count reads the final key.
  const unsigned long long guess = min(seen, k);  // the arg-min as of this block's own contribution
  __threadfence();
  const bool last = atomicAdd(&S.search_done, 1u) == gridDim.x - 1;
  if (!last) return;
  S.search_done = 0;
  CsDevResult* result = a.result ? a.result + (size_t)sj * a.result_stride : nullptr;
  cs_publish(S, hdr, a, cand, result, guess != ~0ull, guess);
  if (tl) { tl[6] = cs_globaltimer(); tl[7] = 1; }
}

// ---------------------------------------------------------------------------------------------------
// slab search: the same arithmetic as cs_search_kernel, laid out for cache locality instead of one warp per
// candidate.  Used for one session alone with many candidates (the host decides, see cs_use_search2).
//
// A candidate's lookups land where the search pose's would, displaced by its offsets: (dx, dy) moves a point by a
// few cells, dtheta by range x dtheta — tens to hundreds of cells.  So candidates with nearly the same heading
// offset read nearly the same cells for the same point.  cs_sort_kernel orders the step's candidates by heading
// offset (a counting sort over fixed bins of width sigma_theta / 256: only locality depends on it, the arg-min is
// decided by (distance, flat index) whatever the evaluation order).  cs_search2_kernel then gives every LANE one
// candidate of the sorted order and walks a cluster of consecutive scan points (broadcast from shared memory):
//   * the 32 lanes of a warp look the same point up under 32 neighbouring headings: a handful of 128-byte tiles
//     per request instead of one per lane (the L1 tag stage handles one line per clock);
//   * a block = one slab of consecutive sorted candidates x one cluster of consecutive points sweeps a compact
//     piece of the map, which its SM's L1 keeps: L2 sees each tile about once per block instead of once per lookup;
//   * no warp reduction: a lane owns its candidate's partial sum and adds it (cells << 0 | in-bounds count << 40)
//     to the candidate's 64-bit accumulator with one RED per cluster.
// The cluster that arrives last at a slab turns the slab's sums into distances (:251-258) and arg-mins them; the slab
// that finishes last runs the Update glue exactly like the last block of cs_search_kernel.
// ---------------------------------------------------------------------------------------------------
#define CS_S2_MAX_POINTS 128   // most points per cluster (1 KB of shared memory)
#define CS_S2_BATCH 16         // lookups a lane has in flight: the cluster is walked in batches of this many points
#define CS_S2_MAX_THREADS 512  // most candidates per slab
#define CS_S2_ARRIVAL_SHIFT 49 // accumulator word: cells (bits 0-31) | in-bounds count (32-48) | clusters arrived (49-63)
#define CS_S2_MAX_CLUSTERS 16384
#define CS_SORT_BINS 2048      // heading bins: [-4 sigma, 4 sigma) in steps of sigma / 256, clamped
#define CS_SORT_THREADS 1024
#define CS_SORT_REG 8          // candidates a thread of the one-block sort keeps in registers between its two passes
#define CS_SORT_MB_CHUNK 1024  // candidates per block of the two-kernel sort

// heading bin of a candidate whose heading differs from the search pose's by `rel`
__device__ __forceinline__ unsigned cs_sort_bin(float rel, float inv) {
  return (unsigned)(int)fminf(fmaxf(rel * inv + (float)(CS_SORT_BINS / 2), 0.f), (float)(CS_SORT_BINS - 1));  // NaN -> 0
}

// Block-wide exclusive scan of s_hist[CS_SORT_BINS] in place (CS_SORT_THREADS threads, two bins each); `c0`, `c1` are
// this thread's two counts.
__device__ __forceinline__ void cs_sort_scan(unsigned* s_hist, unsigned* s_warp, unsigned c0, unsigned c1) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  unsigned v = c0 + c1;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned t = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v += t;
  }
  if (lane == 31) s_warp[warp] = v;
  __syncthreads();
  if (warp == 0) {
    const unsigned w0 = s_warp[lane];
    unsigned w = w0;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned t = __shfl_up_sync(0xffffffffu, w, o);
      if (lane >= o) w += t;
    }
    s_warp[lane] = w - w0;  // exclusive over warps
  }
  __syncthreads();
  const unsigned excl = v - (c0 + c1) + s_warp[warp];
  s_hist[2 * tid] = excl;
  s_hist[2 * tid + 1] = excl + c0;
  __syncthreads();
}

// One block sorts up to CS_SORT_THREADS * CS_SORT_REG candidates.  PHILOX = false: the candidates come from a table
// (offsets or absolute poses); every load of the pass is in flight at once, everything stays in registers.  PHILOX =
// true: the deviates are generated here, one candidate at a time (the generator is long; unrolling it eight times
// would cost more in instruction fetch than it saves), parked in global scratch between the two passes.
template <bool PHILOX>
__global__ void __launch_bounds__(CS_SORT_THREADS)
cs_sort_kernel(CsSession* __restrict__ sessions, CsStepArgs a) {
  __shared__ unsigned s_hist[CS_SORT_BINS];
  __shared__ unsigned s_warp[CS_SORT_THREADS / 32];
  // Nothing here depends on the previous step (inputs of this step and host-owned constants only), so no wait in
  // front; the wait at the end keeps completion transitive: "this grid done" must imply "the grid in front done" for
  // the search kernel behind.
  cs_pdl_launch_dependents();
  const int tid = threadIdx.x;
  const int n = a.cand_count;
  // a batch of sessions: one block per session, everything per session comes from its descriptor
  const int sj = blockIdx.y;
  const CsSession& S = sessions[sj];
  if (blockIdx.x > 0) {
    // One session alone: the sort is this grid's block 0, on one SM, for ~5 us.  The other blocks meanwhile load the sectors of
    // the map within reach of the step — what the search is about to gather from and the draw kernel to blend into — so that a
    // step whose map is not in L2 (the first scan after a pause, bench.py's flushed default line, maps beyond the L2) pays the
    // HBM latency here, beside the sort, and not in the lookups.  Where the map is L2-resident the loads hit.
    cs_prefetch_disc(S, a.hdr[(size_t)sj * a.hdr_stride], a, (int)(blockIdx.x - 1) * CS_SORT_THREADS + tid, (int)(gridDim.x - 1) * CS_SORT_THREADS);
    cs_pdl_wait();
    return;
  }
  const float* cand = a.cand ? a.cand + (size_t)sj * a.cand_stride : nullptr;
  float4* __restrict__ out = a.s2_batch ? S.s2_sorted + (size_t)a.s2_slot * S.s2_cap : a.s2_sorted;
  float4* __restrict__ tmp = a.s2_batch ? S.s2_tmp : a.s2_tmp;
  unsigned long long* __restrict__ meta = a.s2_batch ? S.s2_meta : a.s2_meta;
  const float sigma_theta = a.s2_batch ? S.sigma_theta : a.s2_sigma_theta;
  const float sigma_xy = a.s2_batch ? S.sigma_xy : a.s2_sigma_xy;
  const unsigned long long seed = a.s2_batch ? S.seed : a.s2_seed;
  for (int i = tid; i < CS_SORT_BINS; i += CS_SORT_THREADS) s_hist[i] = 0u;
  __syncthreads();
  const float inv = sigma_theta > 0.f ? 256.0f / sigma_theta : 0.f;
  if (PHILOX) {
#pragma unroll 1
    for (int i = tid; i < n; i += CS_SORT_THREADS) {
      const int idx = a.cand_first + i;
      float off[3] = {0.f, 0.f, 0.f};
      if (idx > 0) cs_gauss3(seed, a.scan_index, (uint32_t)(idx - 1), sigma_xy, sigma_theta, off);
      const unsigned bin = cs_sort_bin(off[2], inv);
      const unsigned rank = atomicAdd(&s_hist[bin], 1u);
      tmp[i] = make_float4(off[0], off[1], off[2], __int_as_float(idx));
      meta[i] = ((unsigned long long)bin << 32) | rank;
    }
    __syncthreads();
    cs_sort_scan(s_hist, s_warp, s_hist[2 * tid], s_hist[2 * tid + 1]);
#pragma unroll 1
    for (int i = tid; i < n; i += CS_SORT_THREADS) {
      const unsigned long long m = meta[i];
      out[s_hist[(unsigned)(m >> 32)] + (unsigned)m] = tmp[i];
    }
  } else {
    const float ref = a.cand_mode == CS_CAND_ABSOLUTE ? a.hdr[(size_t)sj * a.hdr_stride].odo[2] : 0.f;  // headings are binned relative to the search pose
    float ex[CS_SORT_REG], ey[CS_SORT_REG], ez[CS_SORT_REG];
    unsigned met[CS_SORT_REG];  // bin << 16 | rank inside the bin (< 8192)
#pragma unroll
    for (int k = 0; k < CS_SORT_REG; k++) {
      const int i = tid + k * CS_SORT_THREADS;
      const int idx = a.cand_first + i;
      ex[k] = 0.f; ey[k] = 0.f; ez[k] = 0.f;
      if (i < n && idx > 0) {
        const float* p = cand + 3 * (size_t)(idx - 1);
        ex[k] = __ldg(p); ey[k] = __ldg(p + 1); ez[k] = __ldg(p + 2);
      }
    }
#pragma unroll
    for (int k = 0; k < CS_SORT_REG; k++) {
      const int i = tid + k * CS_SORT_THREADS;
      const unsigned bin = cs_sort_bin((a.cand_first + i) > 0 ? ez[k] - ref : 0.f, inv);
      met[k] = bin << 16;
      if (i < n) met[k] |= atomicAdd(&s_hist[bin], 1u);
    }
    __syncthreads();
    cs_sort_scan(s_hist, s_warp, s_hist[2 * tid], s_hist[2 * tid + 1]);
#pragma unroll
    for (int k = 0; k < CS_SORT_REG; k++) {
      const int i = tid + k * CS_SORT_THREADS;
      if (i < n) out[s_hist[met[k] >> 16] + (met[k] & 0xffffu)] = make_float4(ex[k], ey[k], ez[k], __int_as_float(a.cand_first + i));
    }
  }
  cs_pdl_wait();
}

// Candidate sets too big for one block: the same counting sort over several blocks and two kernels.
// cs_sort_hist_kernel: every block bins its CS_SORT_MB_CHUNK candidates (one per thread: the blocks spread over the SMs), reserves a run inside each bin of the
// global histogram (one atomicAdd per non-empty bin and block, the returned value is the block's base rank in that bin)
// and parks entry and (bin, rank) in global scratch.  cs_sort_scatter_kernel: every block scans the complete histogram
// and moves its candidates to their final positions; the last block re-arms the histogram.
template <bool PHILOX>
__global__ void __launch_bounds__(CS_SORT_THREADS)
cs_sort_hist_kernel(CsSession* __restrict__ sessions, CsStepArgs a) {
  __shared__ unsigned s_hist[CS_SORT_BINS];
  cs_pdl_launch_dependents();
  const int tid = threadIdx.x;
  const int n = a.cand_count;
  if (a.w_prefetch == 1) cs_prefetch_disc(sessions[0], a.hdr[0], a, blockIdx.x * CS_SORT_THREADS + tid, gridDim.x * CS_SORT_THREADS);
  const int base_i = blockIdx.x * (CS_SORT_MB_CHUNK);
  const int end_i = min(n, base_i + CS_SORT_MB_CHUNK);
  for (int i = tid; i < CS_SORT_BINS; i += CS_SORT_THREADS) s_hist[i] = 0u;
  __syncthreads();
  const float inv = a.s2_sigma_theta > 0.f ? 256.0f / a.s2_sigma_theta : 0.f;
  const float ref = (!PHILOX && a.cand_mode == CS_CAND_ABSOLUTE) ? a.hdr[0].odo[2] : 0.f;
#pragma unroll 1
  for (int i = base_i + tid; i < end_i; i += CS_SORT_THREADS) {
    const int idx = a.cand_first + i;
    float off[3] = {0.f, 0.f, 0.f};
    float rel = 0.f;
    if (idx > 0) {
      if (PHILOX) {
        cs_gauss3(a.s2_seed, a.scan_index, (uint32_t)(idx - 1), a.s2_sigma_xy, a.s2_sigma_theta, off);
        rel = off[2];
      } else {
        const float* p = a.cand + 3 * (size_t)(idx - 1);
        off[0] = __ldg(p); off[1] = __ldg(p + 1); off[2] = __ldg(p + 2);
        rel = off[2] - ref;
      }
    }
    const unsigned bin = cs_sort_bin(rel, inv);
    const unsigned rank = atomicAdd(&s_hist[bin], 1u);
    a.s2_tmp[i] = make_float4(off[0], off[1], off[2], __int_as_float(idx));
    a.s2_meta[i] = ((unsigned long long)bin << 32) | rank;
  }
  __syncthreads();
  for (int b = tid; b < CS_SORT_BINS; b += CS_SORT_THREADS) {
    const unsigned cnt = s_hist[b];
    s_hist[b] = cnt ? atomicAdd(&a.s2_ghist[b], cnt) : 0u;  // this block's base rank inside bin b
  }
  __syncthreads();
#pragma unroll 1
  for (int i = base_i + tid; i < end_i; i += CS_SORT_THREADS) {
    const unsigned long long m = a.s2_meta[i];  // this thread's own store
    a.s2_meta[i] = m + s_hist[(unsigned)(m >> 32)];
  }
  cs_pdl_wait();  // completion stays transitive (see cs_sort_kernel)
}

__global__ void __launch_bounds__(CS_SORT_THREADS)
cs_sort_scatter_kernel(CsSession* __restrict__ sessions, CsStepArgs a) {
  __shared__ unsigned s_hist[CS_SORT_BINS];
  __shared__ unsigned s_warp[CS_SORT_THREADS / 32];
  __shared__ int s_last;
  cs_pdl_wait();  // the histogram is complete
  cs_pdl_launch_dependents();
  const int tid = threadIdx.x;
  const int n = a.cand_count;
  const int base_i = blockIdx.x * (CS_SORT_MB_CHUNK);
  cs_sort_scan(s_hist, s_warp, __ldcg(&a.s2_ghist[2 * tid]), __ldcg(&a.s2_ghist[2 * tid + 1]));
  for (int i = base_i + tid; i < min(n, base_i + CS_SORT_MB_CHUNK); i += CS_SORT_THREADS) {
    const unsigned long long m = __ldcg(&a.s2_meta[i]);
    a.s2_sorted[s_hist[(unsigned)(m >> 32)] + (unsigned)m] = __ldcg(&a.s2_tmp[i]);
  }
  // the last block to get here re-arms the histogram for the next step (every block has read it by then)
  __syncthreads();
  if (tid == 0) s_last = atomicAdd(&a.s2_ghist[CS_SORT_BINS], 1u) == gridDim.x - 1;
  __syncthreads();
  if (s_last)
    for (int b = tid; b <= CS_SORT_BINS; b += CS_SORT_THREADS) a.s2_ghist[b] = 0u;
}

template <bool TILED>
__global__ void __launch_bounds__(CS_S2_MAX_THREADS)
cs_search2_kernel(CsSession* __restrict__ sessions, CsStepArgs a) {
  __shared__ float2 s_pts[CS_S2_MAX_POINTS];
  const int sj = blockIdx.z;  // session of a batch (0 for a session alone)
  CsSession& S = sessions[sj];
  const CsStepHeader& hdr = a.hdr[(size_t)sj * a.hdr_stride];
  const float2* __restrict__ points = a.points + (size_t)sj * a.points_stride;
  const float* cand = a.cand ? a.cand + (size_t)sj * a.cand_stride : nullptr;
  const int tid = threadIdx.x, lane = tid & 31;
  const int cluster = blockIdx.x, slab = blockIdx.y;
  const unsigned n_clusters = gridDim.x;

  // ---- before the dependency wait: this step's inputs and host-owned constants only
  const int P = a.s2_batch ? hdr.n_points : a.s2_host_points;  // = hdr.n_points (the sessions of a batch may differ)
  const int p0 = cluster * a.s2_points;
  const int np = max(0, min(a.s2_points, P - p0));
  const int np_pad = (np + CS_S2_BATCH - 1) / CS_S2_BATCH * CS_S2_BATCH;
  // the last batch is padded with NaN points: they fail the bounds test like any NaN point does (:244)
  for (int i = tid; i < np_pad; i += blockDim.x) s_pts[i] = i < np ? __ldg(points + p0 + i) : make_float2(__int_as_float(0x7fc00000), 0.f);
  const int size = a.s2_batch ? S.size : a.s2_size, pitch_tiles = a.s2_batch ? S.pitch_tiles : a.s2_pitch_tiles;
  const uint16_t* __restrict__ map = a.s2_batch ? S.map : a.s2_map;
  const float scale = a.s2_batch ? S.scale : a.s2_scale;
  const float4* __restrict__ sorted = a.s2_batch ? S.s2_sorted + (size_t)a.s2_slot * S.s2_cap : a.s2_sorted;
  unsigned long long* __restrict__ acc = a.s2_batch ? S.s2_acc : a.s2_acc;
  int* const distances = S.distances;
  const int pos = slab * a.s2_slab + tid;  // position in the sorted order
  const bool valid = tid < a.s2_slab && pos < a.cand_count;  // (threads beyond the slab: the service warp, see below)

  long long* tl = nullptr;  // timeline record of this block (diagnostics)
  if (a.diag && tid == 0 && (int)(blockIdx.y * gridDim.x + blockIdx.x) < CS_DIAG_SEARCH_BLOCKS - 2) {
    tl = a.diag + ((size_t)a.diag_rings + blockIdx.y * gridDim.x + blockIdx.x) * 8;
    tl[0] = cs_smid(); tl[1] = cs_globaltimer(); tl[7] = 0;
  }
  cs_pdl_wait();  // the sort of this step — and through it the previous step — is complete
  cs_pdl_launch_dependents();
  if (tl) tl[2] = cs_globaltimer();

  float px = 0.f, py = 0.f, c = 0.f, s = 0.f;
  int idx = 0;
  if (valid) {
    const float4 e = __ldcg(sorted + pos);
    idx = __float_as_int(e.w);
    float sp[3], pose[3];
    cs_search_pose(S, hdr, a, sp);
    if (idx == 0) {
      pose[0] = sp[0]; pose[1] = sp[1]; pose[2] = sp[2];
    } else if (a.cand_mode == CS_CAND_ABSOLUTE) {
      pose[0] = e.x; pose[1] = e.y; pose[2] = e.z;
    } else {
      pose[0] = __fadd_rn(sp[0], e.x);  // :635-637
      pose[1] = __fadd_rn(sp[1], e.y);
      pose[2] = __fadd_rn(sp[2], e.z);
    }
    float ct, st;
    if (a.cand_cs) {
      ct = a.cand_cs[2 * (size_t)idx];
      st = a.cand_cs[2 * (size_t)idx + 1];
    } else {
      ct = cs_cosf(pose[2]);
      st = cs_sinf(pose[2]);
    }
    px = __fadd_rn(__fmul_rn(pose[0], scale), 0.5f);  // :232
    py = __fadd_rn(__fmul_rn(pose[1], scale), 0.5f);  // :233
    c = __fmul_rn(ct, scale);                         // :234
    s = __fmul_rn(st, scale);                         // :235
  }
  __syncthreads();  // s_pts
  if (a.spec && tid >= a.s2_slab) {
    // ---- the service warp: glue-table entries (CsStepArgs::spec) of this block's share of the slab's candidates — one in
    // n_clusters, the blocks of a slab between them cover it — while the other warps look up
    const unsigned long long tag = (unsigned long long)a.step_id << 32;
    float sp[3];
    cs_search_pose(S, hdr, a, sp);
    for (int q = cluster + lane * (int)n_clusters; q < a.s2_slab; q += 32 * (int)n_clusters) {
      const int p = slab * a.s2_slab + q;
      if (p >= a.cand_count) break;
      const float4 e = __ldcg(sorted + p);
      const int ei = __float_as_int(e.w);
      float pz[3];
      if (ei == 0) { pz[0] = sp[0]; pz[1] = sp[1]; pz[2] = sp[2]; }
      else if (a.cand_mode == CS_CAND_ABSOLUTE) { pz[0] = e.x; pz[1] = e.y; pz[2] = e.z; }
      else { pz[0] = __fadd_rn(sp[0], e.x); pz[1] = __fadd_rn(sp[1], e.y); pz[2] = __fadd_rn(sp[2], e.z); }  // :635-637
      pz[2] = cs_normalize_angle(pz[2]);  // :746 (the table is only used by UPDATE steps)
      unsigned long long* w = a.spec + (size_t)ei * 8;
      __stcg(w + 0, tag | __float_as_uint(pz[0]));
      __stcg(w + 1, tag | __float_as_uint(pz[1]));
      __stcg(w + 2, tag | __float_as_uint(pz[2]));
      __stcg(w + 3, tag | __float_as_uint(cs_cosf(pz[2])));
      __stcg(w + 4, tag | __float_as_uint(cs_sinf(pz[2])));
    }
    return;
  }
  const unsigned act = __ballot_sync(0xffffffffu, valid);  // lanes of this warp that own a candidate
  if (!valid) return;

  unsigned sum = 0, nb = 0;  // sum <= 65535 * 128
#pragma unroll 1
  for (int i0 = 0; i0 < np_pad; i0 += CS_S2_BATCH) {
    unsigned cell[CS_S2_BATCH];
    unsigned v[CS_S2_BATCH];
#pragma unroll
    for (int j = 0; j < CS_S2_BATCH; j++) {
      const float2 p = s_pts[i0 + j];  // broadcast
      float fx = __fsub_rn(__fadd_rn(px, __fmul_rn(c, p.x)), __fmul_rn(s, p.y));  // :240
      float fy = __fadd_rn(__fadd_rn(py, __fmul_rn(s, p.x)), __fmul_rn(c, p.y));  // :241
      int x = __float2int_rz(fmaxf(fx, -2.0f));  // see cs_search_kernel
      int y = __float2int_rz(fmaxf(fy, -2.0f));
      const bool in = ((unsigned)x < (unsigned)size) && ((unsigned)y < (unsigned)size);  // :244
      cell[j] = in ? cs_cell_offset<TILED>(x, y, size, pitch_tiles) : 0xffffffffu;
    }
#pragma unroll
    for (int j = 0; j < CS_S2_BATCH; j++) {
      v[j] = 0u;
      if (cell[j] != 0xffffffffu) v[j] = (unsigned)__ldg(map + cell[j]);  // :246
    }
#pragma unroll
    for (int j = 0; j < CS_S2_BATCH; j++) {
      sum += v[j];
      nb += cell[j] != 0xffffffffu;
    }
  }

  // ---- one atomic per (candidate, cluster): adds the partial sums and counts the arrival.  The cluster that arrives
  // last at a candidate sees every other cluster's contribution in the returned word (single-address atomics are
  // totally ordered), so it owns the candidate's complete sum: distance (:251-258), arg-min, and the word goes back to
  // zero for the next step.  No fence, no block-wide wait.
  if (tl) tl[4] = cs_globaltimer();  // warp 0 is through its lookups
  const unsigned long long mine = (1ull << CS_S2_ARRIVAL_SHIFT) | ((unsigned long long)nb << 32) | (unsigned long long)sum;
  const unsigned long long old = atomicAdd(&acc[pos], mine);
  const bool fin = (unsigned)(old >> CS_S2_ARRIVAL_SHIFT) == n_clusters - 1u;
  unsigned long long key = ~0ull;
  if (fin) {
    const unsigned long long tot = old + mine;
    const unsigned long long cells = tot & 0xffffffffull, cnt = (tot >> 32) & 0x1ffffull;
    const int d = cnt > 0 ? (int)((cells * 1024ull) / (unsigned long long)P) : 2147483647;  // :251-258
    key = ((unsigned long long)(unsigned)d << 32) | (unsigned)idx;
    if (distances) distances[idx] = d;
    acc[pos] = 0ull;
  }
  if (tl) tl[5] = cs_globaltimer();  // ... and has its atomic back
  const unsigned fin_mask = __ballot_sync(act, fin);
  if (fin_mask == 0u) return;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long other = __shfl_xor_sync(act, key, o);
    if (act >> (lane ^ o) & 1u) key = min(key, other);
  }
  if (lane != (int)(__ffs(act) - 1)) return;
  const unsigned long long seen = atomicMin(&S.key[a.parity], key);
  if (!a.fuse_publish) return;
  // ---- the warp that completes the last candidates owns the complete arg-min: Update glue, pose out (as the last block
  // of cs_search_kernel does).  Its own atomicMin has returned, so it is performed; the fence orders it before the count.
  const unsigned long long guess = min(seen, key);
  __threadfence();
  const unsigned nfin = (unsigned)__popc(fin_mask);
  const bool last = atomicAdd(&S.search_done, nfin) + nfin == (unsigned)a.cand_count;
  if (!last) return;
  S.search_done = 0;
  cs_publish(S, hdr, a, cand, a.result ? a.result + (size_t)sj * a.result_stride : nullptr, true, guess);
}

// ---------------------------------------------------------------------------------------------------
// set-up kernel: the Update glue without a search kernel in front (map-only scans, cs_integrate, multi-GPU
// searches whose arg-min is reduced between the kernels).  One thread per session.
// ---------------------------------------------------------------------------------------------------
#define CS_SETUP_THREADS 32

__global__ void __launch_bounds__(CS_SETUP_THREADS)
cs_setup_kernel(CsSession* __restrict__ sessions, CsStepArgs a) {
  cs_pdl_wait();
  cs_pdl_launch_dependents();  // after the wait: see cs_search_kernel
  const int sj = blockIdx.y;
  if (threadIdx.x != 0) return;
  CsSession& S = sessions[sj];
  const CsStepHeader& hdr = a.hdr[(size_t)sj * a.hdr_stride];
  const float* cand = a.cand ? a.cand + (size_t)sj * a.cand_stride : nullptr;
  CsDevResult* result = a.result ? a.result + (size_t)sj * a.result_stride : nullptr;
  cs_publish(S, hdr, a, cand, result);
}

// ---------------------------------------------------------------------------------------------------
// ScanSegmentsToCloud (CoreSLAMProcessor.cs:187-207) on the device: one thread per ray.  rays = (angle, radius) of all
// segments back to back; seg_first[s] = index of segment s's first ray (n_seg + 1 entries); seg_poses = (x, y, theta)
// per segment; (ox, oy, oz) = the odometry pose the cloud is relative to (the last segment's pose, :719).
// Same operations in the same order as the C#: pose = segment.Pose - odometryPose (:194), then
// pose.X + r.Radius * MathF.Cos(r.Angle + pose.Z) (:200-201), one rounding each, libm-identical cosf/sinf.
// ---------------------------------------------------------------------------------------------------
#define CS_CLOUD_THREADS 128
__global__ void __launch_bounds__(CS_CLOUD_THREADS)
cs_cloud_kernel(const float2* __restrict__ rays, const int* __restrict__ seg_first, const float* __restrict__ seg_poses, int n_seg,
                int n_rays, float ox, float oy, float oz, float2* __restrict__ points) {
  const int i = blockIdx.x * CS_CLOUD_THREADS + threadIdx.x;
  if (i >= n_rays) return;
  int lo = 0, hi = n_seg - 1;  // last segment whose first ray is <= i (empty segments are skipped by the search)
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (__ldg(seg_first + mid) <= i) lo = mid; else hi = mid - 1;
  }
  const float px = __fsub_rn(__ldg(seg_poses + 3 * lo), ox);      // :194
  const float py = __fsub_rn(__ldg(seg_poses + 3 * lo + 1), oy);
  const float pz = __fsub_rn(__ldg(seg_poses + 3 * lo + 2), oz);
  const float2 r = __ldg(rays + i);
  const float ang = __fadd_rn(r.x, pz);
  points[i] = make_float2(__fadd_rn(px, __fmul_rn(r.y, cs_cosf(ang))),   // :200
                          __fadd_rn(py, __fmul_rn(r.y, cs_sinf(ang))));  // :201
}

// ---------------------------------------------------------------------------------------------------
// map helpers
// ---------------------------------------------------------------------------------------------------
__global__ void cs_fill_kernel(uint16_t* __restrict__ map, size_t n_cells, uint16_t value) {
  // 8 cells per 16-byte store
  const uint32_t v2 = (uint32_t)value | ((uint32_t)value << 16);
  const uint4 v = make_uint4(v2, v2, v2, v2);
  size_t n16 = n_cells / 8;
  uint4* p = reinterpret_cast<uint4*>(map);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (size_t)gridDim.x * blockDim.x) p[i] = v;
  if (blockIdx.x == 0 && threadIdx.x == 0)
    for (size_t i = n16 * 8; i < n_cells; i++) map[i] = value;
}

// row-major <-> device layout; to_device != 0: linear -> map
template <bool TILED>
__global__ void cs_relayout_kernel(uint16_t* __restrict__ map, uint16_t* __restrict__ linear, int size, int pitch_tiles,
                                   int to_device) {
  const size_t n = (size_t)size * (size_t)size;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    int y = (int)(i / (size_t)size), x = (int)(i % (size_t)size);
    uint32_t o = cs_cell_offset<TILED>(x, y, size, pitch_tiles);
    if (to_device) map[o] = linear[i];
    else linear[i] = map[o];
  }
}

__device__ __host__ __forceinline__ unsigned long long cs_mix64(unsigned long long z) {
  z += 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

// checksum = sum over cells of (value+1) * mix64(row-major index), mod 2^64 — order independent
template <bool TILED>
__global__ void cs_checksum_kernel(const uint16_t* __restrict__ map, int size, int pitch_tiles,
                                   unsigned long long* __restrict__ out) {
  const size_t n = (size_t)size * (size_t)size;
  unsigned long long acc = 0;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    int y = (int)(i / (size_t)size), x = (int)(i % (size_t)size);
    unsigned long long v = map[cs_cell_offset<TILED>(x, y, size, pitch_tiles)];
    acc += (v + 1ull) * cs_mix64((unsigned long long)i);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) atomicAdd(out, acc);
}

// HoleMap.GetPackedPixels (HoleMap.cs:44-55): two cells per byte, top 4 bits each
template <bool TILED>
__global__ void cs_pack_kernel(const uint16_t* __restrict__ map, int size, int pitch_tiles, uint8_t* __restrict__ out) {
  const size_t n = ((size_t)size * (size_t)size) / 2;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    size_t i0 = 2 * i, i1 = 2 * i + 1;
    unsigned a = map[cs_cell_offset<TILED>((int)(i0 % size), (int)(i0 / size), size, pitch_tiles)];
    unsigned b = map[cs_cell_offset<TILED>((int)(i1 % size), (int)(i1 / size), size, pitch_tiles)];
    out[i] = (uint8_t)(((a >> 12) << 4) | (b >> 12));
  }
}

__global__ void cs_sincos_kernel(const float* __restrict__ in, int n, float* __restrict__ c, float* __restrict__ s) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    c[i] = cs_cosf(in[i]);
    s[i] = cs_sinf(in[i]);
  }
}

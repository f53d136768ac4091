// cs_obstacle.cuh — the ObstacleMap half of CoreSLAMProcessor.Update on the device (SURVEY 8f row 1).
//
//   cs_obstacle_rays_kernel    UpdateObstacleMap's ray loop (CoreSLAM/CoreSLAMProcessor.cs:540-571) with
//                              DrawLaserRayOnObstacleMap (:456-490): one warp per ray, lanes over the steps
//   cs_obstacle_sweep_kernel   the no-hit sweep (:576-592), only over the cells the rays marked
//   cs_obstacle_fill_kernel    Reset's fill (:170) and cs_obstacle_map_fill
//   cs_obstacle_checksum_kernel  a hash of each map (session batches: all sessions in one launch)
// Every kernel takes an array of CsObstacle descriptors and works on descriptor blockIdx.y: a processor launches them with
// one, a session batch with one per session.
//
// The reference walks each ray with a loop-carried error term and finishes with an O(Size^2) pass over a
// bool[,] noHitMap.  Here
//  * the walk is evaluated in closed form per (ray, step): with major = max(dx, dy), minor = min(dx, dy) and
//    h = major / 2, the minor coordinate after k steps is max(0, ceil((k*minor - h) / major)) and the major one
//    is k (dx > dy: x is the major axis, otherwise y — the rosettacode variant steps both axes in one iteration);
//    tests/test_oracle_obstacle.py::test_closed_form_matches_the_loop checks it against the loop;
//  * the ray starts inside the map and is monotone in both axes, so "cell k is inside the map" alone decides
//    whether the loop got that far (:465-469);
//  * noHitMap is a bitmap of 8x4-cell tiles, one 32-bit word per tile (a ray's 32 consecutive steps fall into a
//    few words whichever way it runs); lanes on the same word merge their bits and one of them issues the atomic OR;
//  * hits (:474-477) are saturating increments, commutative, done with a CAS on the byte's word; every hit of a
//    scan precedes the sweep (kernel boundary), as in the reference where the sweep follows the ray loop;
//  * the sweep visits bitmap words, not cells: a thread owns the 8x4 tile of its word, steps the marked cells
//    towards zero with 8-byte row accesses and clears the word, so the bitmap is zero again for the next scan.
// Integer-only after the float->cell transform, which is the same left-associated, singly rounded arithmetic
// as the search kernel's (:566-567).
#pragma once
#include "cs_kernels.cuh"

struct CsObstacle {      // one ObstacleMap (CoreSLAM/ObstacleMap.cs:11-44), device resident
  int8_t* pixels;        // row-major, `pitch` bytes per row (multiple of 8), `rows` rows (multiple of 4)
  uint32_t* no_hit;      // words_per_row * rows/4 words; bit (y&3)*8 + (x&7) of word (y>>2)*words_per_row + (x>>3)
  long long* touched;    // cells the rays have touched since the last Reset (no-hit marks + hits), measurement only
  int size;              // ObstacleMap.Size
  int pitch, rows, words_per_row;
  float scale;           // ObstacleMap.Scale
  int max_hits;          // MaxObstacleHits (:103)
};

#define CS_OBST_RAY_THREADS 256

// minor-axis offset after k major steps; k < 2^14
__device__ __forceinline__ int cs_obst_minor(int k, int minor, int major, int h) {
  if (major < 65536) {  // k*minor < 2^30
    const int num = k * minor - h;
    return num <= 0 ? 0 : (int)(((unsigned)num + (unsigned)major - 1u) / (unsigned)major);
  }
  const long long num = (long long)k * minor - h;
  return num <= 0 ? 0 : (int)((num + major - 1) / major);
}

__global__ void __launch_bounds__(CS_OBST_RAY_THREADS)
cs_obstacle_rays_kernel(const CsSession* __restrict__ sessions, const CsObstacle* __restrict__ obstacles, CsStepArgs a) {
  const CsSession& S = sessions[blockIdx.y];
  const CsObstacle O = obstacles[blockIdx.y];
  const CsStepHeader& hdr = a.hdr[blockIdx.y * a.hdr_stride];
  const float2* __restrict__ points = a.points + blockIdx.y * a.points_stride;
  const int n = hdr.n_points;
  const int lane = threadIdx.x & 31;
  const int warps_per_block = blockDim.x >> 5;
  const int size = O.size;

  const float scale = O.scale;
  const float px = __fadd_rn(__fmul_rn(S.cur_pose[0], scale), 0.5f);  // :545
  const float py = __fadd_rn(__fmul_rn(S.cur_pose[1], scale), 0.5f);  // :546
  const float c = __fmul_rn(S.cur_cs[0], scale);                      // :547
  const float s = __fmul_rn(S.cur_cs[1], scale);                      // :548
  const int x1 = cs_cvt_i32(px), y1 = cs_cvt_i32(py);                  // :553-554
  if (x1 < 0 || x1 >= size || y1 < 0 || y1 >= size) return;           // :557-560 (the bitmap is already clear)

  long long touched = 0;
  for (int ray = blockIdx.x * warps_per_block + (threadIdx.x >> 5); ray < n; ray += gridDim.x * warps_per_block) {
    const float2 p = points[ray];
    const int x2 = cs_cvt_i32(__fsub_rn(__fadd_rn(px, __fmul_rn(c, p.x)), __fmul_rn(s, p.y)));  // :566
    const int y2 = cs_cvt_i32(__fadd_rn(__fadd_rn(py, __fmul_rn(s, p.x)), __fmul_rn(c, p.y)));  // :567
    const int ddx = cs_wsub(x2, x1), ddy = cs_wsub(y2, y1);
    if (ddx == (int)0x80000000 || ddy == (int)0x80000000) continue;  // Math.Abs(int.MinValue) throws in the reference
    const int dx = ddx < 0 ? -ddx : ddx, dy = ddy < 0 ? -ddy : ddy;  // :458-459
    const int sx = cs_sign(ddx), sy = cs_sign(ddy);
    const bool xmajor = dx > dy;                                      // :460 picks the sign of err the same way
    const int major = xmajor ? dx : dy, minor = xmajor ? dy : dx;
    const int h = major / 2;
    const int last = min(major, size - 1);  // the major coordinate moves one cell per step: at most size-1 steps stay inside
    for (int k0 = 0; k0 <= last; k0 += 32) {
      const int k = k0 + lane;
      bool inside = false;
      int x = 0, y = 0;
      if (k <= last) {
        const int m = cs_obst_minor(k, minor, major, h);
        x = xmajor ? x1 + sx * k : x1 + sx * m;
        y = xmajor ? y1 + sy * m : y1 + sy * k;
        inside = x >= 0 && x < size && y >= 0 && y < size;  // :465-466
      }
      const unsigned live = __ballot_sync(0xffffffffu, inside);
      if (live == 0u) break;  // monotone: once outside, outside for good
      const unsigned marking = __ballot_sync(0xffffffffu, inside && k != major);
      touched += __popc(live);
      if (inside) {
        if (k == major) {  // :471-479 the hit: ObstacleMap.Pixels[y1, x1] < MaxObstacleHits -> ++
          const size_t byte = (size_t)y * O.pitch + x;
          unsigned* w = reinterpret_cast<unsigned*>(O.pixels + (byte & ~(size_t)3));
          const int sh = (int)(byte & 3) * 8;
          unsigned old = *reinterpret_cast<volatile unsigned*>(w);
          for (;;) {
            const int v = (int)(signed char)((old >> sh) & 0xffu);
            if (v >= O.max_hits) break;
            const unsigned nw = (old & ~(0xffu << sh)) | (((unsigned)(v + 1) & 0xffu) << sh);
            const unsigned seen = atomicCAS(w, old, nw);
            if (seen == old) break;
            old = seen;
          }
        } else {  // :483 noHitMap[y1, x1] = true
          const unsigned word = (unsigned)(y >> 2) * (unsigned)O.words_per_row + (unsigned)(x >> 3);
          const unsigned bit = 1u << (((y & 3) << 3) | (x & 7));
          const unsigned peers = __match_any_sync(marking, word);
          const unsigned bits = __reduce_or_sync(peers, bit);
          if (lane == __ffs(peers) - 1) {
            // skip the atomic when another ray has marked all of these cells already (the stretch near the robot
            // is shared by every ray of the scan)
            const unsigned seen = *reinterpret_cast<volatile unsigned*>(O.no_hit + word);
            if ((seen & bits) != bits) atomicOr(O.no_hit + word, bits);
          }
        }
      }
    }
  }
  if (O.touched) {
    // every lane counted the same ballots: lane 0 reports
    if (lane == 0 && touched) atomicAdd(reinterpret_cast<unsigned long long*>(O.touched), (unsigned long long)touched);
  }
}

// One thread per bitmap word = per 8x4-cell tile.
__global__ void __launch_bounds__(256)
cs_obstacle_sweep_kernel(const CsObstacle* __restrict__ obstacles) {
  const CsObstacle O = obstacles[blockIdx.y];
  const int n_words = O.words_per_row * (O.rows >> 2);
  for (int w = blockIdx.x * blockDim.x + threadIdx.x; w < n_words; w += gridDim.x * blockDim.x) {
    const unsigned bits = O.no_hit[w];
    if (bits == 0u) continue;
    O.no_hit[w] = 0u;  // ArrayEx.Fill(noHitMap, false) of the next update (:542)
    const int ty = w / O.words_per_row, tx = w - ty * O.words_per_row;
#pragma unroll
    for (int r = 0; r < 4; r++) {
      const unsigned row = (bits >> (8 * r)) & 0xffu;
      if (row == 0u) continue;
      unsigned long long* q = reinterpret_cast<unsigned long long*>(O.pixels + (size_t)(ty * 4 + r) * O.pitch + tx * 8);
      unsigned long long v = *q;
#pragma unroll
      for (int b = 0; b < 8; b++) {
        if (row & (1u << b)) {  // :580-590: negative cells count up to 0, positive ones down to 0
          const int px = (int)(signed char)((v >> (8 * b)) & 0xffull);
          const int nx = px < 0 ? px + 1 : (px > 0 ? px - 1 : 0);
          v = (v & ~(0xffull << (8 * b))) | ((unsigned long long)((unsigned)nx & 0xffu) << (8 * b));
        }
      }
      *q = v;
    }
  }
}

// ArrayEx.Fill(ObstacleMap.Pixels, v) (:170), with the no-hit bitmap and the touched counter cleared: one ObstacleMap per
// blockIdx.y, filled with values[blockIdx.y] (a batch's per-session UnmappedObstacleHits) or, without values, with `value`.
__global__ void cs_obstacle_fill_kernel(const CsObstacle* __restrict__ obstacles, const int* __restrict__ values, int value) {
  const CsObstacle O = obstacles[blockIdx.y];
  if (values) value = values[blockIdx.y];
  const size_t n8 = (size_t)O.pitch * O.rows / 8;
  const unsigned long long b = (unsigned long long)((unsigned)value & 0xffu) * 0x0101010101010101ull;
  unsigned long long* q = reinterpret_cast<unsigned long long*>(O.pixels);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (size_t)gridDim.x * blockDim.x) q[i] = b;
  const size_t nw = (size_t)O.words_per_row * (O.rows >> 2);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nw; i += (size_t)gridDim.x * blockDim.x) O.no_hit[i] = 0u;
  if (blockIdx.x == 0 && threadIdx.x == 0 && O.touched) *O.touched = 0;
}

// Position-dependent hash of every ObstacleMap, one per blockIdx.y: out[blockIdx.y] += sum over the row-major cells i of
// ((uint8_t)pixel + 1) * cs_mix64(i), mod 2^64 (cs_host_obstacle_checksum; the caller zeroes `out`).
__global__ void __launch_bounds__(256)
cs_obstacle_checksum_kernel(const CsObstacle* __restrict__ obstacles, unsigned long long* __restrict__ out) {
  const CsObstacle O = obstacles[blockIdx.y];
  const unsigned size = (unsigned)O.size, n = size * size;  // size <= 16384: n < 2^32
  unsigned long long acc = 0;
  for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const unsigned y = i / size, x = i - y * size;
    const unsigned long long v = (unsigned char)O.pixels[(size_t)y * O.pitch + x];
    acc += (v + 1ull) * cs_mix64((unsigned long long)i);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0 && acc) atomicAdd(out + blockIdx.y, acc);
}

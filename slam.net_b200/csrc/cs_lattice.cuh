// cs_lattice.cuh — relocalisation on an existing map (cs_relocalize): the reference's distance function
// (CalculateDistanceSISD, CoreSLAM/CoreSLAMProcessor.cs:226-259) at every pose of a regular (x, y, theta) lattice, then
// the lattice poses that are strict local minima of (distance, flat index) within a window, best first.
//
//   cs_lattice_kernel         distance of every lattice pose -> a volume of int32 (flat index (it*count1 + iy)*count0 + ix);
//                             or (LIST) of the poses of listed 32 x 32 tiles -> 1024 values per tile (cs_relocalize_bounded);
//                             or (SEQ) the sum over a scan sequence, each scan placed by its odometry relative to the last
//                             (cs_relocalize_sequence)
//   cs_seq_offsets_kernel     the odometry of a scan sequence -> each scan's offset from the anchor (the last scan)
//   cs_lattice_select_kernel  window test of every pose; the k best local minima of each block's poses -> one sorted list
//   cs_lattice_select_tiles_kernel  the same over the listed tiles only (cs_relocalize_bounded, see cs_bnb.cuh)
//   cs_lattice_merge_kernel   CS_LAT_MERGE_LISTS sorted lists -> one, until one list remains
// All are plain stream-ordered launches that poll nothing: the state of the handle (map, pose, step chain) is only read.
//
// Why a lattice is cheaper per lookup than a candidate search: the reference computes x = (int)((px + c*X) - s*Y) and
// y = (int)((py + s*X) + c*Y) (:240-241), every product rounded by itself.  The four products c*X, s*Y, s*X, c*Y of a point
// depend on the heading alone, so a block takes one heading, stages the products of a chunk of points in shared memory
// (one float4 per point) and every (x, y) pose of that heading reuses them: bit-identical to the search kernels.  A thread
// holds CS_LAT_PY poses that share their x and differ in y, so the x coordinate of a point is also shared: per lookup
// that leaves 2 FADD + FMNMX + F2I + bounds + address + LDG + IADD, plus a quarter of the x part.
#pragma once
#include "cs_kernels.cuh"

#define CS_LAT_THREADS 256
#define CS_LAT_PY 4             // poses per thread: one x, CS_LAT_PY values of y
#define CS_LAT_TILE_X 32        // poses of a block along x: a warp covers 16 x 8 poses, the 8 warps 2 x 4 warp patches
#define CS_LAT_TILE_Y 32
#define CS_LAT_CHUNK 1024       // points staged per pass (16 KB of products)
#define CS_LAT_SEL_PER 16       // poses per thread of the select kernel
#define CS_LAT_MERGE_LISTS 32   // lists merged by one block of the merge kernel
#define CS_LAT_MERGE_PER 8      // keys per thread of the merge kernel (CS_LAT_MERGE_LISTS * 64 / CS_LAT_THREADS)
#define CS_LAT_SEQ_MAX 32       // scans of a sequence (CS_SEQUENCE_MAX_SCANS)

// One scan of a sequence: its points [first, first + count) of the concatenated scans, and its odometry pose relative to
// the anchor's (the last scan's), in the anchor's frame: with ca, sa = cosf, sinf(anchor theta), e = o - anchor,
// dx = ca*ex + sa*ey, dy = ca*ey - sa*ex, dtheta = o.theta - anchor.theta (cs_seq_offsets_kernel).
struct CsSeqScan {
  int first, count;
  float dx, dy, dtheta;
};
// the scans of a sequence (points index the concatenated scans)
struct CsSeqArgs {
  const CsSeqScan* scans;
  int n_scans;
};

struct CsLatticeArgs {
  const uint16_t* map;
  int size, pitch_tiles;
  float scale;
  const float2* points;
  int n_points;
  float origin[3], step[3];
  int count[3];
  int tiles_x, tiles_y;
  int* volume;
  const int4* tiles;  // LIST: the tiles to evaluate, {it, tile x, tile y, mask of the warp patches to evaluate}
  int* tile_slot;     // LIST: dense per-tile index of the lattice ((it*tiles_y + tile y)*tiles_x + tile x) -> list position
  CsSeqArgs seq;      // SEQ: the scans of the sequence
};

// odometry[3k .. 3k+2] and scan_first[0 .. n_scans] -> out[k]; one thread per scan, one rounding per operation
__global__ void cs_seq_offsets_kernel(const float* __restrict__ odometry, const int* __restrict__ scan_first, int n_scans,
                                      CsSeqScan* __restrict__ out) {
  const int k = threadIdx.x;
  if (k >= n_scans) return;
  const float* o = odometry + 3 * k;
  const float* an = odometry + 3 * (n_scans - 1);
  const float ca = cs_cosf(an[2]), sa = cs_sinf(an[2]);
  const float ex = __fsub_rn(o[0], an[0]), ey = __fsub_rn(o[1], an[1]);
  CsSeqScan q;
  q.first = scan_first[k];
  q.count = scan_first[k + 1] - q.first;
  q.dx = __fadd_rn(__fmul_rn(ca, ex), __fmul_rn(sa, ey));
  q.dy = __fsub_rn(__fmul_rn(ca, ey), __fmul_rn(sa, ex));
  q.dtheta = __fsub_rn(o[2], an[2]);
  out[k] = q;
}

// pose coordinate of lattice point i along one axis: origin + (float)i * step, two roundings, no FMA
__host__ __device__ __forceinline__ float cs_lattice_coord(float origin, float step, int i) {
#ifdef __CUDA_ARCH__
  return __fadd_rn(origin, __fmul_rn((float)i, step));
#else
  const float t = (float)i * step;
  return origin + t;
#endif
}

// The reference's arithmetic of one lookup (:232-244), shared by every kernel that evaluates or bounds lattice distances:
// the pose x (or y) in map units, the four per-point products and the (int) cast of the cell coordinates, each operation
// one rounding.  x is non-decreasing in px and y in py (cs_bnb.cuh relies on it).
__device__ __forceinline__ float cs_map_p(float coord, float scale) { return __fadd_rn(__fmul_rn(coord, scale), 0.5f); }  // :232-233
__device__ __forceinline__ float cs_lattice_p(float origin, float step, int i, float scale) {
  return cs_map_p(cs_lattice_coord(origin, step, i), scale);
}
__device__ __forceinline__ float4 cs_lattice_products(float c, float s, float2 p) {
  return make_float4(__fmul_rn(c, p.x), __fmul_rn(s, p.y), __fmul_rn(s, p.x), __fmul_rn(c, p.y));
}
__device__ __forceinline__ int cs_lattice_cell_x(float px, float4 q) { return __float2int_rz(fmaxf(__fsub_rn(__fadd_rn(px, q.x), q.y), -2.0f)); }
__device__ __forceinline__ int cs_lattice_cell_y(float py, float4 q) { return __float2int_rz(fmaxf(__fadd_rn(__fadd_rn(py, q.z), q.w), -2.0f)); }

// Scan q of a sequence at a lattice pose of heading theta (c0, s0 = cosf, sinf(theta), unscaled): its (c, s) scaled as in
// :234-235 at theta + dtheta, and the offset (ox, oy) = (c0*dx - s0*dy, s0*dx + c0*dy) its pose adds to the lattice x, y.
// The offset is the same for every (x, y) pose of the heading, so the cell of a point stays non-decreasing in ix and iy.
struct CsSeqPose {
  float c, s, ox, oy;
};
__device__ __forceinline__ CsSeqPose cs_seq_pose(float theta, float c0, float s0, float scale, const CsSeqScan& q) {
  const float t = __fadd_rn(theta, q.dtheta);
  CsSeqPose p;
  p.c = __fmul_rn(cs_cosf(t), scale);
  p.s = __fmul_rn(cs_sinf(t), scale);
  p.ox = __fsub_rn(__fmul_rn(c0, q.dx), __fmul_rn(s0, q.dy));
  p.oy = __fadd_rn(__fmul_rn(s0, q.dx), __fmul_rn(c0, q.dy));
  return p;
}

// Every scan's CsSeqPose at lattice heading theta into s_pose, one scan per thread, then a barrier.
__device__ __forceinline__ void cs_seq_poses(float theta, float scale, const CsSeqArgs& seq, CsSeqPose* s_pose) {
  if ((int)threadIdx.x < seq.n_scans) s_pose[threadIdx.x] = cs_seq_pose(theta, cs_cosf(theta), cs_sinf(theta), scale, seq.scans[threadIdx.x]);
  __syncthreads();
}

// int.MaxValue when no point was in bounds, else floor(1024 * sum / n) (:251-258)
__device__ __forceinline__ int cs_lattice_distance(bool any, unsigned sum, int n) {
  return any ? (int)(((unsigned long long)sum * 1024ull) / (unsigned)n) : 2147483647;
}

// The sums of one scan's points over a thread's CS_LAT_PY poses (one x, the rows py), staged in chunks through s_prod.
template <bool TILED>
__device__ __forceinline__ void cs_lattice_sums(const CsLatticeArgs& a, float4* s_prod, const float2* __restrict__ points, int n_points,
                                                float c, float s, float px, const float (&py)[CS_LAT_PY], bool active,
                                                unsigned (&sum)[CS_LAT_PY], unsigned& in_any) {
  const int size = a.size, pitch_tiles = a.pitch_tiles;
  const uint16_t* __restrict__ map = a.map;
  for (int base = 0; base < n_points; base += CS_LAT_CHUNK) {
    const int n = min(CS_LAT_CHUNK, n_points - base);
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += CS_LAT_THREADS) {
      s_prod[i] = cs_lattice_products(c, s, points[base + i]);
    }
    __syncthreads();
    if (!active) continue;
#pragma unroll 4
    for (int i = 0; i < n; i++) {
      const float4 q = s_prod[i];
      // :240-241, left-associative, one rounding per operation; the (int) cast + bounds test of cs_search_kernel (:244)
      const int x = cs_lattice_cell_x(px, q);
      const bool xin = (unsigned)x < (unsigned)size;
#pragma unroll
      for (int j = 0; j < CS_LAT_PY; j++) {
        const int y = cs_lattice_cell_y(py[j], q);
        if (xin && (unsigned)y < (unsigned)size) {
          sum[j] += (unsigned)__ldg(map + cs_cell_offset<TILED>(x, y, size, pitch_tiles));  // :246
          in_any |= 1u << j;
        }
      }
    }
  }
}

// One block takes one 32 x 32 tile of poses of one heading: the tile blockIdx.x of the lattice, or with LIST the tile
// a.tiles[blockIdx.x], whose warps evaluate only the 16 x 8 patches (warp w: x half w & 1, rows 8 * (w >> 1)) set in its
// mask and write int.MaxValue for the others.  LIST writes the tile's 1024 poses (row-major, 32 per row) at
// a.volume + 1024 * blockIdx.x and records the slot in a.tile_slot.  SEQ: the distance of a pose is the sum over the scans
// a.seq.scans[0 .. n_scans) of each scan's distance at the pose the scan's offset and heading change give it, int.MaxValue when
// any scan has no point in bounds (<= 32 * 1024 * 65535 < 2^31 otherwise).
template <bool TILED, bool LIST = false, bool SEQ = false>
__global__ void __launch_bounds__(CS_LAT_THREADS) cs_lattice_kernel(CsLatticeArgs a) {
  __shared__ float4 s_prod[CS_LAT_CHUNK];  // (c*X, s*Y, s*X, c*Y) of the chunk's points
  int it, tile_x, tile_y;
  unsigned mask = 0xffu;
  if (LIST) {
    const int4 e = a.tiles[blockIdx.x];
    it = e.x, tile_x = e.y, tile_y = e.z, mask = (unsigned)e.w;
    if (threadIdx.x == 0) a.tile_slot[((size_t)it * a.tiles_y + tile_y) * a.tiles_x + tile_x] = (int)blockIdx.x;
  } else {
    const int tiles_xy = a.tiles_x * a.tiles_y;
    it = (int)(blockIdx.x / (unsigned)tiles_xy);
    const int tile = (int)(blockIdx.x % (unsigned)tiles_xy);
    tile_x = tile % a.tiles_x, tile_y = tile / a.tiles_x;
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ix = tile_x * CS_LAT_TILE_X + (warp & 1) * 16 + (lane & 15);
  const int iy0 = tile_y * CS_LAT_TILE_Y + (warp >> 1) * 8 + (lane >> 4);  // + 2j, j < CS_LAT_PY

  const float theta = cs_lattice_coord(a.origin[2], a.step[2], it);
  float c = 0.f, s = 0.f, px = 0.f, py[CS_LAT_PY];
  if (!SEQ) {
    c = __fmul_rn(cs_cosf(theta), a.scale);  // :234
    s = __fmul_rn(cs_sinf(theta), a.scale);  // :235
    px = cs_lattice_p(a.origin[0], a.step[0], ix, a.scale);  // :232
#pragma unroll
    for (int j = 0; j < CS_LAT_PY; j++) py[j] = cs_lattice_p(a.origin[1], a.step[1], iy0 + 2 * j, a.scale);  // :233
  }
  const bool inside = ix < a.count[0] && iy0 < a.count[1];
  const bool active = inside && ((mask >> warp) & 1u);

  unsigned sum[CS_LAT_PY];  // <= 65535 * 65536 < 2^32 (max_points <= 65536)
  unsigned in_any = 0;      // bit j: some point of pose j was in bounds
#pragma unroll
  for (int j = 0; j < CS_LAT_PY; j++) sum[j] = 0;
  unsigned total[CS_LAT_PY];  // SEQ: the sum of the scans' distances (< 2^31), or >= 2^31 once a scan had no point in bounds
  if (SEQ) {
    __shared__ CsSeqPose s_pose[CS_LAT_SEQ_MAX];
    cs_seq_poses(theta, a.scale, a.seq, s_pose);
    const float x = cs_lattice_coord(a.origin[0], a.step[0], ix);
    float y[CS_LAT_PY];
#pragma unroll
    for (int j = 0; j < CS_LAT_PY; j++) y[j] = cs_lattice_coord(a.origin[1], a.step[1], iy0 + 2 * j), total[j] = 0;
    for (int k = 0; k < a.seq.n_scans; k++) {
      const CsSeqScan q = a.seq.scans[k];
      const CsSeqPose p = s_pose[k];
      px = cs_map_p(__fadd_rn(x, p.ox), a.scale);
#pragma unroll
      for (int j = 0; j < CS_LAT_PY; j++) py[j] = cs_map_p(__fadd_rn(y[j], p.oy), a.scale), sum[j] = 0;
      in_any = 0;
      cs_lattice_sums<TILED>(a, s_prod, a.points + q.first, q.count, p.c, p.s, px, py, active, sum, in_any);
#pragma unroll
      for (int j = 0; j < CS_LAT_PY; j++) total[j] = (in_any >> j) & 1u ? total[j] + (unsigned)cs_lattice_distance(true, sum[j], q.count) : 0x80000000u;
    }
  } else {
    cs_lattice_sums<TILED>(a, s_prod, a.points, a.n_points, c, s, px, py, active, sum, in_any);
  }
  if (!inside) return;
  const size_t plane = (size_t)it * a.count[1];
#pragma unroll
  for (int j = 0; j < CS_LAT_PY; j++) {
    const int iy = iy0 + 2 * j;
    if (iy < a.count[1]) {
      const int d = SEQ ? (int)min(total[j], 2147483647u) : cs_lattice_distance((in_any >> j) & 1u, sum[j], a.n_points);
      if (LIST)
        a.volume[(size_t)blockIdx.x * (CS_LAT_TILE_X * CS_LAT_TILE_Y) + (iy - tile_y * CS_LAT_TILE_Y) * CS_LAT_TILE_X + (ix - tile_x * CS_LAT_TILE_X)] = d;
      else
        a.volume[(plane + iy) * a.count[0] + ix] = d;
    }
  }
}

// The PER keys each thread of the block holds (~0 = none) -> the k smallest of the block, ascending, into out[0..k)
// (padded with ~0).  Keys are unique, so one extraction per output removes exactly one key.
template <int PER>
__device__ __forceinline__ void cs_lattice_block_topk(unsigned long long (&key)[PER], int k, unsigned long long* __restrict__ out) {
  __shared__ unsigned long long s_min[CS_LAT_THREADS / 32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int r = 0; r < k; r++) {
    unsigned long long m = key[0];
#pragma unroll
    for (int j = 1; j < PER; j++) m = min(m, key[j]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = min(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (lane == 0) s_min[warp] = m;
    __syncthreads();
    m = s_min[0];
#pragma unroll
    for (int w = 1; w < CS_LAT_THREADS / 32; w++) m = min(m, s_min[w]);
    __syncthreads();  // (s_min is rewritten by the next round)
    if (threadIdx.x == 0) out[r] = m;
    if (m == ~0ull) {  // fewer than k keys: pad
      for (int q = r + 1 + (int)threadIdx.x; q < k; q += CS_LAT_THREADS) out[q] = ~0ull;
      return;
    }
#pragma unroll
    for (int j = 0; j < PER; j++)
      if (key[j] == m) key[j] = ~0ull;
  }
}

// key of a pose: distance << 32 | flat index (distance >= 0, so the order is (distance, index))
__device__ __forceinline__ unsigned long long cs_lattice_key(int d, unsigned idx) { return ((unsigned long long)(unsigned)d << 32) | idx; }

// A pose is a candidate when its distance is < int.MaxValue and its key is below the key of every other pose within
// +-window steps on each axis (the box clipped at the lattice edges, theta not wrapped).  dist(n, t, y, x) reads the
// distance of pose n = (t*c1 + y)*c0 + x.
template <class Dist>
__device__ __forceinline__ bool cs_lattice_window_min(const Dist& dist, unsigned long long mine, unsigned idx, int ix, int iy, int it,
                                                      int c0, int c1, int c2, int window) {
  const int x0 = max(ix - window, 0), x1 = min(ix + window, c0 - 1);
  const int y0 = max(iy - window, 0), y1 = min(iy + window, c1 - 1);
  const int t0 = max(it - window, 0), t1 = min(it + window, c2 - 1);
  bool best = true;
  for (int t = t0; t <= t1 && best; t++)
    for (int y = y0; y <= y1 && best; y++) {
      const unsigned row = ((unsigned)t * (unsigned)c1 + (unsigned)y) * (unsigned)c0;
      for (int x = x0; x <= x1; x++) {
        const unsigned n = row + (unsigned)x;
        if (n != idx && cs_lattice_key(dist(n, t, y, x), n) < mine) { best = false; break; }
      }
    }
  return best;
}

// Block b takes the poses [b * CS_LAT_THREADS * CS_LAT_SEL_PER, ...) and writes its k best candidates to lists[b * k ...].
__global__ void __launch_bounds__(CS_LAT_THREADS)
cs_lattice_select_kernel(const int* __restrict__ volume, int c0, int c1, int c2, int window, int k, unsigned long long* __restrict__ lists) {
  const unsigned total = (unsigned)c0 * (unsigned)c1 * (unsigned)c2;
  const auto dist = [&](unsigned n, int, int, int) { return __ldg(volume + n); };
  unsigned long long key[CS_LAT_SEL_PER];
#pragma unroll
  for (int j = 0; j < CS_LAT_SEL_PER; j++) {
    key[j] = ~0ull;
    const unsigned idx = (blockIdx.x * CS_LAT_SEL_PER + j) * CS_LAT_THREADS + threadIdx.x;
    if (idx >= total) continue;
    const int d = __ldg(volume + idx);
    if (d == 2147483647) continue;
    const unsigned long long mine = cs_lattice_key(d, idx);
    const int ix = (int)(idx % (unsigned)c0), iy = (int)(idx / (unsigned)c0 % (unsigned)c1), it = (int)(idx / ((unsigned)c0 * (unsigned)c1));
    if (cs_lattice_window_min(dist, mine, idx, ix, iy, it, c0, c1, c2, window)) key[j] = mine;
  }
  cs_lattice_block_topk(key, k, lists + (size_t)blockIdx.x * k);
}

// cs_lattice_select_kernel over the poses of the tiles cs_lattice_kernel<., true> evaluated: tile s of `tiles` holds its
// 1024 distances at buf + 1024 * s, tile_slot maps a tile of the lattice to s (-1: not evaluated).  A pose of a tile
// that was not evaluated reads int.MaxValue, so it is larger than any candidate's key and is never one itself.  Also
// counts into *passed the candidates whose distance is <= upper.
__global__ void __launch_bounds__(CS_LAT_THREADS)
cs_lattice_select_tiles_kernel(const int* __restrict__ buf, const int4* __restrict__ tiles, const int* __restrict__ tile_slot, int n_tiles,
                               int c0, int c1, int c2, int tiles_x, int tiles_y, int window, int k, int upper,
                               unsigned long long* __restrict__ passed, unsigned long long* __restrict__ lists) {
  constexpr int TILE = CS_LAT_TILE_X * CS_LAT_TILE_Y;
  const auto dist = [&](unsigned, int t, int y, int x) {
    const int s = __ldg(tile_slot + ((size_t)t * tiles_y + y / CS_LAT_TILE_Y) * tiles_x + x / CS_LAT_TILE_X);
    return s < 0 ? 2147483647 : __ldg(buf + (size_t)s * TILE + (y % CS_LAT_TILE_Y) * CS_LAT_TILE_X + x % CS_LAT_TILE_X);
  };
  const unsigned total = (unsigned)n_tiles * TILE;
  unsigned long long key[CS_LAT_SEL_PER];
  unsigned n_passed = 0;
#pragma unroll
  for (int j = 0; j < CS_LAT_SEL_PER; j++) {
    key[j] = ~0ull;
    const unsigned p = (blockIdx.x * CS_LAT_SEL_PER + j) * CS_LAT_THREADS + threadIdx.x;
    if (p >= total) continue;
    const int4 e = __ldg(tiles + p / TILE);
    const int ix = e.y * CS_LAT_TILE_X + (int)(p % CS_LAT_TILE_X), iy = e.z * CS_LAT_TILE_Y + (int)(p % TILE / CS_LAT_TILE_X);
    if (ix >= c0 || iy >= c1) continue;
    const int d = __ldg(buf + p);
    if (d == 2147483647) continue;
    const unsigned idx = ((unsigned)e.x * (unsigned)c1 + (unsigned)iy) * (unsigned)c0 + (unsigned)ix;
    const unsigned long long mine = cs_lattice_key(d, idx);
    if (cs_lattice_window_min(dist, mine, idx, ix, iy, e.x, c0, c1, c2, window)) {
      key[j] = mine;
      n_passed += d <= upper;
    }
  }
  if (n_passed) atomicAdd(passed, (unsigned long long)n_passed);
  cs_lattice_block_topk(key, k, lists + (size_t)blockIdx.x * k);
}

// Block b merges the sorted lists [b * CS_LAT_MERGE_LISTS, ...) of k keys each (of n_lists) into out[b * k ...].
__global__ void __launch_bounds__(CS_LAT_THREADS)
cs_lattice_merge_kernel(const unsigned long long* __restrict__ in, int n_lists, int k, unsigned long long* __restrict__ out) {
  const int first = blockIdx.x * CS_LAT_MERGE_LISTS;
  const int n_keys = min(CS_LAT_MERGE_LISTS, n_lists - first) * k;
  const unsigned long long* src = in + (size_t)first * k;
  unsigned long long key[CS_LAT_MERGE_PER];
#pragma unroll
  for (int j = 0; j < CS_LAT_MERGE_PER; j++) {
    const int i = j * CS_LAT_THREADS + (int)threadIdx.x;
    key[j] = i < n_keys ? src[i] : ~0ull;
  }
  cs_lattice_block_topk(key, k, out + (size_t)blockIdx.x * k);
}

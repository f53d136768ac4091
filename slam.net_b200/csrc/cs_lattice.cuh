// cs_lattice.cuh — relocalisation on an existing map (cs_relocalize): the reference's distance function
// (CalculateDistanceSISD, CoreSLAM/CoreSLAMProcessor.cs:226-259) at every pose of a regular (x, y, theta) lattice, then
// the lattice poses that are strict local minima of (distance, flat index) within a window, best first.
//
//   cs_lattice_kernel         distance of every lattice pose -> a volume of int32 (flat index (it*count1 + iy)*count0 + ix)
//   cs_lattice_select_kernel  window test of every pose; the k best local minima of each block's poses -> one sorted list
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
};

// pose coordinate of lattice point i along one axis: origin + (float)i * step, two roundings, no FMA
__host__ __device__ __forceinline__ float cs_lattice_coord(float origin, float step, int i) {
#ifdef __CUDA_ARCH__
  return __fadd_rn(origin, __fmul_rn((float)i, step));
#else
  const float t = (float)i * step;
  return origin + t;
#endif
}

template <bool TILED>
__global__ void __launch_bounds__(CS_LAT_THREADS) cs_lattice_kernel(CsLatticeArgs a) {
  __shared__ float4 s_prod[CS_LAT_CHUNK];  // (c*X, s*Y, s*X, c*Y) of the chunk's points
  const int tiles_xy = a.tiles_x * a.tiles_y;
  const int it = (int)(blockIdx.x / (unsigned)tiles_xy);
  const int tile = (int)(blockIdx.x % (unsigned)tiles_xy);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ix = (tile % a.tiles_x) * CS_LAT_TILE_X + (warp & 1) * 16 + (lane & 15);
  const int iy0 = (tile / a.tiles_x) * CS_LAT_TILE_Y + (warp >> 1) * 8 + (lane >> 4);  // + 2j, j < CS_LAT_PY

  const float theta = cs_lattice_coord(a.origin[2], a.step[2], it);
  const float c = __fmul_rn(cs_cosf(theta), a.scale);  // :234
  const float s = __fmul_rn(cs_sinf(theta), a.scale);  // :235
  const float px = __fadd_rn(__fmul_rn(cs_lattice_coord(a.origin[0], a.step[0], ix), a.scale), 0.5f);  // :232
  float py[CS_LAT_PY];
#pragma unroll
  for (int j = 0; j < CS_LAT_PY; j++)
    py[j] = __fadd_rn(__fmul_rn(cs_lattice_coord(a.origin[1], a.step[1], iy0 + 2 * j), a.scale), 0.5f);  // :233
  const bool active = ix < a.count[0] && iy0 < a.count[1];

  const int size = a.size, pitch_tiles = a.pitch_tiles;
  const uint16_t* __restrict__ map = a.map;
  unsigned sum[CS_LAT_PY];  // <= 65535 * 65536 < 2^32 (max_points <= 65536)
  unsigned in_any = 0;      // bit j: some point of pose j was in bounds
#pragma unroll
  for (int j = 0; j < CS_LAT_PY; j++) sum[j] = 0;

  for (int base = 0; base < a.n_points; base += CS_LAT_CHUNK) {
    const int n = min(CS_LAT_CHUNK, a.n_points - base);
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += CS_LAT_THREADS) {
      const float2 p = a.points[base + i];
      s_prod[i] = make_float4(__fmul_rn(c, p.x), __fmul_rn(s, p.y), __fmul_rn(s, p.x), __fmul_rn(c, p.y));
    }
    __syncthreads();
    if (!active) continue;
#pragma unroll 4
    for (int i = 0; i < n; i++) {
      const float4 q = s_prod[i];
      // :240-241, left-associative, one rounding per operation; the (int) cast + bounds test of cs_search_kernel (:244)
      const int x = __float2int_rz(fmaxf(__fsub_rn(__fadd_rn(px, q.x), q.y), -2.0f));
      const bool xin = (unsigned)x < (unsigned)size;
#pragma unroll
      for (int j = 0; j < CS_LAT_PY; j++) {
        const int y = __float2int_rz(fmaxf(__fadd_rn(__fadd_rn(py[j], q.z), q.w), -2.0f));
        if (xin && (unsigned)y < (unsigned)size) {
          sum[j] += (unsigned)__ldg(map + cs_cell_offset<TILED>(x, y, size, pitch_tiles));  // :246
          in_any |= 1u << j;
        }
      }
    }
  }
  if (!active) return;
  const size_t plane = (size_t)it * a.count[1];
#pragma unroll
  for (int j = 0; j < CS_LAT_PY; j++) {
    const int iy = iy0 + 2 * j;
    if (iy < a.count[1]) {
      const int d = ((in_any >> j) & 1u) ? (int)(((unsigned long long)sum[j] * 1024ull) / (unsigned)a.n_points) : 2147483647;  // :251-258
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
// +-window steps on each axis (the box clipped at the lattice edges, theta not wrapped).  Block b takes the poses
// [b * CS_LAT_THREADS * CS_LAT_SEL_PER, ...) and writes its k best candidates to lists[b * k ...].
__global__ void __launch_bounds__(CS_LAT_THREADS)
cs_lattice_select_kernel(const int* __restrict__ volume, int c0, int c1, int c2, int window, int k, unsigned long long* __restrict__ lists) {
  const unsigned total = (unsigned)c0 * (unsigned)c1 * (unsigned)c2;
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
    const int x0 = max(ix - window, 0), x1 = min(ix + window, c0 - 1);
    const int y0 = max(iy - window, 0), y1 = min(iy + window, c1 - 1);
    const int t0 = max(it - window, 0), t1 = min(it + window, c2 - 1);
    bool best = true;
    for (int t = t0; t <= t1 && best; t++)
      for (int y = y0; y <= y1 && best; y++) {
        const unsigned row = ((unsigned)t * (unsigned)c1 + (unsigned)y) * (unsigned)c0;
        for (int x = x0; x <= x1; x++) {
          const unsigned n = row + (unsigned)x;
          if (n != idx && cs_lattice_key(__ldg(volume + n), n) < mine) { best = false; break; }
        }
      }
    if (best) key[j] = mine;
  }
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

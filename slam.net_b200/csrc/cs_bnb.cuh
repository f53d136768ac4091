// cs_bnb.cuh — branch and bound over a pose lattice (cs_relocalize_bounded): lower bounds of the lattice distance
// (cs_lattice.cuh) over blocks of poses, from min-window grids of the HoleMap, so that most of a fine lattice is never
// evaluated.  DESIGN section 4 has the exactness argument.
//
//   cs_bnb_grid0_kernel   G_0: a row-major copy of the HoleMap (either layout)
//   cs_bnb_grid_kernel    G_j[y][x] = min of the HoleMap over [x, x+2^j) x [y, y+2^j) clipped to the map, from G_{j-1}
//   cs_bnb_seed_kernel    exact distance of the first pose of every top-level node (the first guess of the upper bound)
//   cs_bnb_bound_kernel   one node -> the bounds of its children; the children with bound <= upper are appended to the
//                         next level's list (at the last level: the node's 32 x 32 tile, with a mask of its 16 x 8 patches)
// All are plain stream-ordered launches that poll nothing.  The SEQ instances of the seed and bound kernels do the same
// for a scan sequence (cs_relocalize_sequence_bounded): the seed is the exact sum over the scans, and a child's bound the
// sum of the scans' bounds, each scan's rectangles taken at its own offset and heading.
//
// The bound.  For one heading, a point's cell is x = (int)((px + c*X) - s*Y), px = (origin + (float)ix*step)*Scale + 0.5f,
// every operation a rounded f32 add or multiply by a positive factor, then a truncation: x is non-decreasing in ix, and y
// in iy.  Over the poses [ix0, ix1] x [iy0, iy1] of one heading the point therefore stays in the cell rectangle
// [x(ix0), x(ix1)] x [y(iy0), y(iy1)] (four exact evaluations).  Its term is >= the minimum of the map over any window
// holding that rectangle when the rectangle lies on the map, >= 0 otherwise (an off-map point adds nothing), and the
// node's poses all have distance int.MaxValue when every rectangle lies wholly off the map.  floor(1024 * sum / P) is
// non-decreasing in the sum, so the bound is <= the distance of every pose of the node.  A scan of a sequence adds a
// constant offset to px (and py) for one heading and rotates by a constant angle: its cells stay non-decreasing in ix and
// iy, and the sum of the scans' bounds is <= the sum of their distances.
#pragma once
#include "cs_lattice.cuh"

#define CS_BNB_MAX_GRID 10   // G_0 .. G_10: windows up to 1024 cells
#define CS_BNB_LEAF_LEVEL 5  // the descent ends at the 32 x 32 tiles of cs_lattice_kernel (CS_LAT_TILE_X = CS_LAT_TILE_Y = 32)

template <bool TILED>
__global__ void __launch_bounds__(CS_LAT_THREADS) cs_bnb_grid0_kernel(const uint16_t* __restrict__ map, int size, int pitch_tiles, uint16_t* __restrict__ g0) {
  const size_t cells = (size_t)size * size;
  for (size_t i = (size_t)blockIdx.x * CS_LAT_THREADS + threadIdx.x; i < cells; i += (size_t)gridDim.x * CS_LAT_THREADS) {
    const int x = (int)(i % (unsigned)size), y = (int)(i / (unsigned)size);
    g0[i] = __ldg(map + cs_cell_offset<TILED>(x, y, size, pitch_tiles));
  }
}

// window doubling: [x, x+2h) = [x, x+h) u [x+h, x+2h), clipped to the map, on both axes
__global__ void __launch_bounds__(CS_LAT_THREADS) cs_bnb_grid_kernel(const uint16_t* __restrict__ prev, int size, int h, uint16_t* __restrict__ out) {
  const size_t cells = (size_t)size * size;
  for (size_t i = (size_t)blockIdx.x * CS_LAT_THREADS + threadIdx.x; i < cells; i += (size_t)gridDim.x * CS_LAT_THREADS) {
    const int x = (int)(i % (unsigned)size), y = (int)(i / (unsigned)size);
    const bool xr = x + h < size, yd = y + h < size;
    unsigned m = __ldg(prev + i);
    if (xr) m = min(m, (unsigned)__ldg(prev + i + h));
    if (yd) m = min(m, (unsigned)__ldg(prev + i + (size_t)h * size));
    if (xr && yd) m = min(m, (unsigned)__ldg(prev + i + (size_t)h * size + h));
    out[i] = (uint16_t)m;
  }
}

struct CsBnbArgs {
  const uint16_t* grids;  // G_0 .. G_max_grid, size*size cells each, row-major
  int size, max_grid;
  float scale;
  const float2* points;
  int n_points;
  float origin[3], step[3];
  int count[3];
  int level;           // the nodes of this launch are 2^level x 2^level poses of one heading
  int top_x, top_y;    // nodes per heading along x, y when `in` is NULL (the top level: every node of the lattice)
  const int4* in;      // the nodes: {it, node x, node y, 0}
  int4* out;           // the surviving children: {it, child x, child y, 0}, or at level CS_BNB_LEAF_LEVEL the node's tile
  int out_cap;         //   {it, tile x, tile y, mask of its surviving 16 x 8 patches}
  int upper;           // children with bound > upper are pruned
  unsigned long long* counters;  // [0] children appended (also past out_cap), [1] bounds computed, [2] poses of the tiles' patches
};

__device__ __forceinline__ int4 cs_bnb_node(const CsBnbArgs& a) {
  if (a.in) return a.in[blockIdx.x];
  const unsigned per_heading = (unsigned)a.top_x * (unsigned)a.top_y, r = blockIdx.x % per_heading;
  return make_int4((int)(blockIdx.x / per_heading), (int)(r % (unsigned)a.top_x), (int)(r / (unsigned)a.top_x), 0);
}

// c = cos(theta)*Scale, s = sin(theta)*Scale of heading it (:234-235)
__device__ __forceinline__ float2 cs_bnb_heading(const CsBnbArgs& a, int it) {
  const float theta = cs_lattice_coord(a.origin[2], a.step[2], it);
  return make_float2(__fmul_rn(cs_cosf(theta), a.scale), __fmul_rn(cs_sinf(theta), a.scale));
}

// The exact sum of the points' map values at one pose, on thread 0 as floor(1024 * sum / n_points), int.MaxValue when no
// point is in bounds (:251-258).  s_sum, s_any: block scratch, free again when thread 0 returns.
__device__ __forceinline__ int cs_bnb_pose_distance(const CsBnbArgs& a, const float2* __restrict__ points, int n_points, float c, float s,
                                                    float px, float py, unsigned* s_sum, unsigned& s_any) {
  if (threadIdx.x == 0) s_any = 0;
  unsigned sum = 0;
  bool any = false;
  for (int i = threadIdx.x; i < n_points; i += CS_LAT_THREADS) {
    const float4 q = cs_lattice_products(c, s, points[i]);
    const int x = cs_lattice_cell_x(px, q), y = cs_lattice_cell_y(py, q);
    if ((unsigned)x < (unsigned)a.size && (unsigned)y < (unsigned)a.size) {
      sum += __ldg(a.grids + (size_t)y * a.size + x);
      any = true;
    }
  }
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  const bool warp_any = __any_sync(0xffffffffu, any);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) {
    s_sum[threadIdx.x >> 5] = sum;
    if (warp_any) s_any = 1;
  }
  __syncthreads();
  int d = 0;
  if (threadIdx.x == 0) {
    unsigned long long t = 0;
    for (int w = 0; w < CS_LAT_THREADS / 32; w++) t += s_sum[w];
    d = s_any ? (int)(t * 1024ull / (unsigned)n_points) : 2147483647;  // :251-258
  }
  return d;
}

// seeds[node] = the exact distance of the node's first pose (the top level: in == NULL)
template <bool SEQ = false>
__global__ void __launch_bounds__(CS_LAT_THREADS) cs_bnb_seed_kernel(CsBnbArgs a, int* __restrict__ seeds, CsSeqArgs seq) {
  __shared__ unsigned s_sum[CS_LAT_THREADS / 32];
  __shared__ unsigned s_any;
  const int4 node = cs_bnb_node(a);
  if (SEQ) {
    __shared__ CsSeqPose s_pose[CS_LAT_SEQ_MAX];
    cs_seq_poses(cs_lattice_coord(a.origin[2], a.step[2], node.x), a.scale, seq, s_pose);
    const float x = cs_lattice_coord(a.origin[0], a.step[0], node.y << a.level);
    const float y = cs_lattice_coord(a.origin[1], a.step[1], node.z << a.level);
    unsigned total = 0;
    bool off = false;
    for (int k = 0; k < seq.n_scans; k++) {
      const CsSeqScan q = seq.scans[k];
      const CsSeqPose p = s_pose[k];
      const int d = cs_bnb_pose_distance(a, a.points + q.first, q.count, p.c, p.s, cs_map_p(__fadd_rn(x, p.ox), a.scale),
                                         cs_map_p(__fadd_rn(y, p.oy), a.scale), s_sum, s_any);
      off |= d == 2147483647;
      total += (unsigned)d;
    }
    if (threadIdx.x == 0) seeds[blockIdx.x] = off ? 2147483647 : (int)total;
  } else {
    const float2 cs = cs_bnb_heading(a, node.x);
    const float px = cs_lattice_p(a.origin[0], a.step[0], node.y << a.level, a.scale);
    const float py = cs_lattice_p(a.origin[1], a.step[1], node.z << a.level, a.scale);
    const int d = cs_bnb_pose_distance(a, a.points, a.n_points, cs.x, cs.y, px, py, s_sum, s_any);
    if (threadIdx.x == 0) seeds[blockIdx.x] = d;
  }
}

// The lower-bound sums of one scan's points over the NX x NY children whose first and last poses map to pxl/pxh, pyl/pyh
// (c, s: the scan's scaled heading) into s_sum[warp][child], and per warp the children some point's rectangle of which
// touches the map into s_any[warp]; ends with a barrier after which thread 0 may read them.
template <int NX, int NY>
__device__ __forceinline__ void cs_bnb_child_sums(const CsBnbArgs& a, const float2* __restrict__ points, int n_points, float2 cs,
                                                  const float (&pxl)[NX], const float (&pxh)[NX], const float (&pyl)[NY],
                                                  const float (&pyh)[NY], unsigned (*s_sum)[NX * NY], unsigned* s_any) {
  constexpr int NC = NX * NY;
  const int size = a.size;
  const size_t cells = (size_t)size * size;
  unsigned sum[NC];
#pragma unroll
  for (int c = 0; c < NC; c++) sum[c] = 0;
  unsigned any = 0;  // bit c: some point's rectangle of child c touches the map
  for (int i = threadIdx.x; i < n_points; i += CS_LAT_THREADS) {
    const float4 q = cs_lattice_products(cs.x, cs.y, points[i]);
    int xl[NX], xh[NX], yl[NY], yh[NY];
#pragma unroll
    for (int j = 0; j < NX; j++) xl[j] = cs_lattice_cell_x(pxl[j], q), xh[j] = cs_lattice_cell_x(pxh[j], q);
#pragma unroll
    for (int j = 0; j < NY; j++) yl[j] = cs_lattice_cell_y(pyl[j], q), yh[j] = cs_lattice_cell_y(pyh[j], q);
#pragma unroll
    for (int c = 0; c < NC; c++) {
      const int x_lo = xl[c % NX], x_hi = xh[c % NX], y_lo = yl[c / NX], y_hi = yh[c / NX];
      if (x_hi < 0 || x_lo >= size || y_hi < 0 || y_lo >= size) continue;  // wholly off the map: adds 0 at every pose
      any |= 1u << c;
      if (x_lo < 0 || x_hi >= size || y_lo < 0 || y_hi >= size) continue;  // partly off: bounded by 0
      const int j = 32 - __clz(max(x_hi - x_lo, y_hi - y_lo));             // 2^j >= span + 1
      if (j <= a.max_grid) sum[c] += __ldg(a.grids + (size_t)j * cells + (size_t)y_lo * size + x_lo);
    }
  }
#pragma unroll
  for (int c = 0; c < NC; c++)
    for (int o = 16; o > 0; o >>= 1) sum[c] += __shfl_xor_sync(0xffffffffu, sum[c], o);
  for (int o = 16; o > 0; o >>= 1) any |= __shfl_xor_sync(0xffffffffu, any, o);
  const int warp = threadIdx.x >> 5;
  if ((threadIdx.x & 31) == 0) {
#pragma unroll
    for (int c = 0; c < NC; c++) s_sum[warp][c] = sum[c];
    s_any[warp] = any;
  }
  __syncthreads();
}

// One block per node: the bounds of its NX x NY children, each point's rectangle looked up in the grid whose window
// covers it (2^j >= span + 1; a wider span bounds the term by 0).  TILE: the node is a 32 x 32 tile and its children are
// the 16 x 8 patches of cs_lattice_kernel's warps (patch w: column w & 1, row w >> 1); otherwise the four quadrants.
// SEQ: a child's bound is the sum of the scans' bounds, and a child where some scan lies wholly off the map is dropped.
template <bool TILE, bool SEQ = false>
__global__ void __launch_bounds__(CS_LAT_THREADS) cs_bnb_bound_kernel(CsBnbArgs a, CsSeqArgs seq) {
  constexpr int NX = 2, NY = TILE ? 4 : 2, NC = NX * NY;
  __shared__ unsigned s_sum[CS_LAT_THREADS / 32][NC];
  __shared__ unsigned s_any[CS_LAT_THREADS / 32];
  const int4 node = cs_bnb_node(a);
  const int side = 1 << a.level, wx = side / NX, wy = side / NY;
  const int x0 = node.y * side, y0 = node.z * side;  // < count[0], count[1]
  float2 cs = make_float2(0.f, 0.f);
  if (!SEQ) cs = cs_bnb_heading(a, node.x);
  // children's first and last pose along each axis (a child that starts past the lattice edge does not exist)
  float pxl[NX], pxh[NX], pyl[NY], pyh[NY];
  int ixl[NX], ixh[NX], iyl[NY], iyh[NY];  // (SEQ: their lattice indices)
  unsigned exists = 0;
#pragma unroll
  for (int i = 0; i < NX; i++) {
    const int lo = x0 + min(i * wx, a.count[0] - 1 - x0), hi = x0 + min((i + 1) * wx - 1, a.count[0] - 1 - x0);
    ixl[i] = lo, ixh[i] = hi;
    if (!SEQ) pxl[i] = cs_lattice_p(a.origin[0], a.step[0], lo, a.scale), pxh[i] = cs_lattice_p(a.origin[0], a.step[0], hi, a.scale);
  }
#pragma unroll
  for (int i = 0; i < NY; i++) {
    const int lo = y0 + min(i * wy, a.count[1] - 1 - y0), hi = y0 + min((i + 1) * wy - 1, a.count[1] - 1 - y0);
    iyl[i] = lo, iyh[i] = hi;
    if (!SEQ) pyl[i] = cs_lattice_p(a.origin[1], a.step[1], lo, a.scale), pyh[i] = cs_lattice_p(a.origin[1], a.step[1], hi, a.scale);
  }
#pragma unroll
  for (int c = 0; c < NC; c++)
    if ((c % NX) * wx < a.count[0] - x0 && (c / NX) * wy < a.count[1] - y0) exists |= 1u << c;

  unsigned alive = ~0u;  // SEQ, thread 0, bit c: every scan has some point whose rectangle of child c touches the map
  long long bound[NC];   // SEQ, thread 0: the sum of the scans' bounds
  if (SEQ) {
    __shared__ CsSeqPose s_pose[CS_LAT_SEQ_MAX];
    cs_seq_poses(cs_lattice_coord(a.origin[2], a.step[2], node.x), a.scale, seq, s_pose);
#pragma unroll
    for (int c = 0; c < NC; c++) bound[c] = 0;
    for (int k = 0; k < seq.n_scans; k++) {
      const CsSeqScan q = seq.scans[k];
      const CsSeqPose p = s_pose[k];
      const auto at = [&](int axis, int i, float o) { return cs_map_p(__fadd_rn(cs_lattice_coord(a.origin[axis], a.step[axis], i), o), a.scale); };
#pragma unroll
      for (int i = 0; i < NX; i++) pxl[i] = at(0, ixl[i], p.ox), pxh[i] = at(0, ixh[i], p.ox);
#pragma unroll
      for (int i = 0; i < NY; i++) pyl[i] = at(1, iyl[i], p.oy), pyh[i] = at(1, iyh[i], p.oy);
      if (k) __syncthreads();  // (thread 0 has read the previous scan's sums)
      cs_bnb_child_sums<NX, NY>(a, a.points + q.first, q.count, make_float2(p.c, p.s), pxl, pxh, pyl, pyh, s_sum, s_any);
      if (threadIdx.x == 0) {
        unsigned all_any = 0;
        for (int w = 0; w < CS_LAT_THREADS / 32; w++) all_any |= s_any[w];
        alive &= all_any;
        for (int c = 0; c < NC; c++) {
          unsigned long long t = 0;
          for (int w = 0; w < CS_LAT_THREADS / 32; w++) t += s_sum[w][c];
          bound[c] += (long long)(t * 1024ull / (unsigned)q.count);
        }
      }
    }
  } else {
    cs_bnb_child_sums<NX, NY>(a, a.points, a.n_points, cs, pxl, pxh, pyl, pyh, s_sum, s_any);
  }
  if (threadIdx.x != 0) return;
  unsigned keep = 0, all_any = 0;
  if (SEQ) all_any = alive;
  else
    for (int w = 0; w < CS_LAT_THREADS / 32; w++) all_any |= s_any[w];
  long long poses = 0;
  for (int c = 0; c < NC; c++) {
    if (!((exists >> c) & 1u) || !((all_any >> c) & 1u)) continue;  // no such child, or only int.MaxValue poses
    long long b;
    if (SEQ) {
      b = bound[c];
    } else {
      unsigned long long t = 0;
      for (int w = 0; w < CS_LAT_THREADS / 32; w++) t += s_sum[w][c];
      b = (long long)(t * 1024ull / (unsigned)a.n_points);
    }
    if (b > (long long)a.upper) continue;  // strictly above: ties survive
    keep |= 1u << c;
    const int cx = x0 + (c % NX) * wx, cy = y0 + (c / NX) * wy;
    poses += (long long)min(wx, a.count[0] - cx) * min(wy, a.count[1] - cy);
  }
  atomicAdd(a.counters + 1, (unsigned long long)__popc(exists));
  if (!keep) return;
  if (TILE) {
    atomicAdd(a.counters + 2, (unsigned long long)poses);
    const unsigned long long slot = atomicAdd(a.counters, 1ull);
    if (slot < (unsigned long long)a.out_cap) a.out[slot] = make_int4(node.x, node.y, node.z, (int)keep);
  } else {
    const unsigned long long slot = atomicAdd(a.counters, (unsigned long long)__popc(keep));
    int n = 0;
    for (int c = 0; c < NC; c++)
      if ((keep >> c) & 1u) {
        if (slot + n < (unsigned long long)a.out_cap) a.out[slot + n] = make_int4(node.x, 2 * node.y + c % NX, 2 * node.z + c / NX, 0);
        n++;
      }
  }
}

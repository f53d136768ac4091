// cs_wedge.cuh — the draw loop of DrawLaserRayOnHoleMap (CoreSLAM/CoreSLAMProcessor.cs:404-442) as independent
// (ring range x angular wedge) tasks, one warp per task, no block-wide synchronisation in the draw loop.
//
// Why it is exact.  Every ray of a scan starts in the same cell (x1,y1) and advances one cell along its major axis per
// step, so its step k lies on the square ring of Chebyshev radius k; rings never share a cell.  On ring k ray r sits at
// position  p = c*k + g*m(k)  along the ring (c in {1,3,5,7} the side, g = +-1), and the Bresenham walk :394-396, 433-441
// has the closed form  m(k) = min(k, ceil(k*s - 1/2)),  s = dyc/dxc  — so  |p - k*kappa| <= 1/2  with the ray's angular
// key  kappa = c + g*s  in [0, 8].  A wedge is a key interval [beta_w, beta_w+1); on ring k it OWNS the positions
// ceil(k*beta_w) <= p < ceil(k*beta_w+1)  (every position of every ring belongs to exactly one wedge, whatever the
// boundaries are), and only rays with  beta_w - 1/(2k) <= kappa < beta_w+1 + 1/(2k)  can land there.  A task therefore
// filters its candidate rays by key (conservatively, in float), keeps them in RAY ORDER, decides ownership of every visit
// exactly (integers), and applies the visits of one cell in ray order: all visitors of a cell are candidates of the one
// task that owns the cell, so the reference's order (foreach over cloud.Points, :517) is kept without atomics, sorting or
// a slot table, for any ray order.  tools/wedge_model.py is the host model of this decomposition.
//
// Two paths per task, chosen by the candidate count:
//   fast     <= 32 candidates: one ray per lane, Bresenham state carried in registers from ring to ring (no per-ring
//            division), visits of one cell inside the warp found with match.any and applied by the lowest lane in lane
//            (= ray) order; rings go four at a time in three passes (walk + ownership, the four match.any back to back, the
//            leaders' four map loads), with an instance for groups of rings on which no lane is inside its hole profile.
//   general  any number of candidates (dense levels, where the margins alone exceed a warp; clustered or multi-turn
//            scans): the wedge's cells of up to 8 rings are staged in shared memory, the batches of 32 rays that can hold
//            candidates are walked in ray order with the next batch's rays in flight, same-cell groups fold into the
//            staged values (uniform groups as a count with the exact fixed-point early-out), then the touched cells go back.
// Rings 0 .. CS_W_CENTER - 1, which every ray crosses, are drawn by one block as shared-memory counts (cs_w_center).
// The first blocks prepare the rays (cs_ray_from_point: UpdateHoleMap, ClipRay, the prologue of the draw loop), plus each
// ray's key, the key range of every 32 rays, and per level and key sector the number of rays that reach it (which sizes
// the wedges: ~26 candidates each, cut at the quantiles of the level's rays).  DESIGN.md section 4 has the scheduling and
// the measurements.
#pragma once
#include "cs_kernels.cuh"

#define CS_W_THREADS 256
#define CS_W_WARPS (CS_W_THREADS / 32)
#define CS_W_LEVELS 264   // rings [1,1] [2,3] [4,7] [8,15] [16,31] [32,63], then 64 rings each: ring 16383 is level 260
#define CS_W_FIX 14       // wedge boundaries are multiples of 2^-14 (keys span [0, 8])
#define CS_W_CAP 256      // cells of a wedge staged per pass of the general path
#define CS_W_G 4            // rings in flight per lane on the fast path
#define CS_W_H 4            // ... handled in parts of this many (cs_w_fast_group)
#define CS_W_MAX_WEDGES 8192
#define CS_W_SECTORS 64   // key sectors of width 1/8: the rays that reach a level are counted per sector, and each sector is
                          // cut into wedges of its own (long rays cluster in a few directions: a uniform cut would leave some
                          // wedges with several times the candidates a warp holds)
#define CS_W_OWN 26       // candidates a wedge is sized for (own rays + the rays of its margins)

__device__ __forceinline__ int cs_w_level_first(int L) { return L < 6 ? (1 << L) : 64 * (L - 5); }
__device__ __forceinline__ int cs_w_level_last(int L) { return L < 6 ? (2 << L) - 1 : 64 * (L - 5) + 63; }
__device__ __forceinline__ int cs_w_level_of(int k) { return k < 64 ? 31 - __clz(k) : 5 + (k >> 6); }  // k >= 1

// wedges of a level reached by `alive` rays whose first ring is k0: about 26 candidates per wedge, of which
// alive / (8 k0) come from the +-1/(2 k0) margins; where the margins alone exceed that (the centre) a wedge is as wide
// as its margins.  Never more wedges than ring k0 has cells.
__device__ __forceinline__ int cs_w_wedges(int alive, int k0) {
  if (alive <= 0) return 0;
  const int halo2 = alive / (8 * k0);
  const int own = halo2 > 13 ? halo2 : 26 - halo2;
  int W = (alive + own - 1) / own;
  W = min(W, min(8 * k0, CS_W_MAX_WEDGES));
  return max(W, 1);
}
__device__ __forceinline__ unsigned cs_w_beta(int w, int W) { return (unsigned)(((unsigned)w * (8u << CS_W_FIX)) / (unsigned)W); }
__device__ __forceinline__ int cs_w_bound(int k, unsigned beta) { return (int)(((unsigned)k * beta + ((1u << CS_W_FIX) - 1u)) >> CS_W_FIX); }

// side constant c and minor sign g of  p = c*k + g*m  (cs_ring_visit's position, before the 8k -> 0 wrap)
__device__ __forceinline__ void cs_w_side(int flags, int& c, int& g) {
  const bool steep = (flags & 2) != 0, majneg = (flags & 4) != 0, minneg = (flags & 8) != 0;
  c = steep ? (majneg ? 7 : 3) : (majneg ? 5 : 1);
  g = ((steep != majneg) ? -1 : 1) * (minneg ? -1 : 1);
}

struct CsWTask {
  int k0, k1;          // rings, inclusive
  unsigned blo, bhi;   // wedge boundaries (fixed point)
  float flo, fhi;      // key range a candidate must fall in (margins included)
  float wrap_lo;       // wedge 0 also takes keys >= wrap_lo (positions 8k wrap to 0); 9 = no
};

// ---- ray preparation by the first blocks (UpdateHoleMap :517-530, ClipRay, the prologue of DrawLaserRayOnHoleMap), one ray
// per lane: packed ray, (key, dxc), the warp's key range and largest dxc.  Returns what cs_w_count needs.
struct CsWPrepared {
  float key;
  int dxc;     // -1: the ray draws nothing
  int bm;      // largest dxc of the warp's rays
};
__device__ __forceinline__ CsWPrepared cs_w_prepare(CsSession& S, const CsRayFrame& f, const float2 p, int i, bool in_range,
                                                    long long& visits) {
  const unsigned full = 0xffffffffu;
  CsRay r;
  r.dxc = 0; r.dyc = 0; r.a0 = 0; r.b0 = -1; r.incv = 0; r.kc = 0; r.nd_total = 0; r.flags = 0;
  if (in_range) r = cs_ray_from_point(f, p, S.ray_dbg ? S.ray_dbg + 6 * (size_t)i : nullptr);
  const bool valid = (r.flags & 1) != 0;
  float key = 0.f;
  if (valid) {
    visits += (long long)r.dxc + 1;
    int c, g;
    cs_w_side(r.flags, c, g);
    const float s = r.dxc > 0 ? __fdiv_rn((float)min(r.dyc, r.dxc), (float)r.dxc) : 0.f;
    key = (float)c + (float)g * s;
  }
  if (in_range) {
    S.rays[i] = cs_pack_ray(r);
    S.w_rk[i] = make_int2(__float_as_int(key), valid ? r.dxc : -1);
  }
  const int lane = threadIdx.x & 31;
  const int bm = __reduce_max_sync(full, valid ? r.dxc : -1);
  // keys are in [0, 8]: order-preserving as unsigned bit patterns
  const unsigned kmin = __reduce_min_sync(full, valid ? __float_as_uint(key) : 0x7f800000u);
  const unsigned kmax = __reduce_max_sync(full, valid ? __float_as_uint(key) : 0u);
  if (lane == 0 && in_range) {
    S.batch_max[i >> 5] = bm;
    S.w_bkey[i >> 5] = make_float2(__uint_as_float(kmin), __uint_as_float(kmax));
  }
  CsWPrepared out;
  out.key = key; out.dxc = valid ? r.dxc : -1; out.bm = bm;
  return out;
}

// Counts for sizing the wedges: per level the rays that reach it, in all and per key sector.  The lanes of a sector add as
// one (the 32 consecutive rays of a warp span a sector or two of a lidar scan).  Only the balance of the task table depends
// on these numbers, never a result.
__device__ __forceinline__ void cs_w_count(const CsSession& S, const CsWPrepared& q, int* top) {
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  int* tot = top + (size_t)S.w_levels * CS_W_SECTORS;
  const bool counted = q.dxc >= 1;
  const unsigned cm = __ballot_sync(full, counted);
  if (cm) {
    const int sector = min(CS_W_SECTORS - 1, (int)(q.key * (CS_W_SECTORS / 8.0f)));
    unsigned same = 0u;
    if (counted) same = __match_any_sync(cm, sector);
    const bool leader = counted && lane == __ffs(same) - 1;
    const int top_level = cs_w_level_of(max(q.bm, 1));
#pragma unroll 4
    for (int L = 0; L <= top_level; L++) {
      const unsigned here = __ballot_sync(full, counted && q.dxc >= cs_w_level_first(L));
      if (leader && (here & same)) atomicAdd(&top[L * CS_W_SECTORS + sector], (int)__popc(here & same));
      if (lane == 0 && here) atomicAdd(&tot[L], (int)__popc(here));
    }
  }
}

// The batches of 32 consecutive rays that can hold a candidate of task t (by their key range and largest dxc), as a bitmap
// in shared memory (bit b of word b / 32); returns the number of words in use.
#define CS_W_BMAP_WORDS 64  // 65536 rays / 32 / 32
__device__ __forceinline__ int cs_w_batch_map(const CsSession& S, const CsWTask& t, int n, unsigned* s_bmap) {
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const int nb = (n + 31) >> 5;
  const int nw = (nb + 31) >> 5;
  __syncwarp();  // (readers of the previous map are done)
  for (int w0 = 0; w0 < nw; w0 += 4) {  // four words per round trip
    int bm[4];
    float2 kk[4];
#pragma unroll
    for (int u = 0; u < 4; u++) {
      const int bi = (w0 + u) * 32 + lane;
      bm[u] = -1;
      kk[u] = make_float2(0.f, 0.f);
      if (bi < nb) { bm[u] = S.batch_max[bi]; kk[u] = S.w_bkey[bi]; }
    }
#pragma unroll
    for (int u = 0; u < 4; u++) {
      const bool ov = bm[u] >= t.k0 && ((kk[u].y >= t.flo && kk[u].x < t.fhi) || kk[u].y >= t.wrap_lo);
      const unsigned om = __ballot_sync(full, ov);
      if (lane == 0 && w0 + u < nw) s_bmap[w0 + u] = om;
    }
  }
  __syncwarp();
  return nw;
}
// next batch at or after `from` in the bitmap, or -1
__device__ __forceinline__ int cs_w_next_batch(const unsigned* s_bmap, int nw, int from) {
  int w = from >> 5;
  if (w >= nw) return -1;
  unsigned m = s_bmap[w] & (0xffffffffu << (from & 31));
  while (m == 0u) {
    if (++w >= nw) return -1;
    m = s_bmap[w];
  }
  return w * 32 + __ffs(m) - 1;
}
__device__ __forceinline__ bool cs_w_is_candidate(const CsWTask& t, const int2 rk) {
  const float key = __int_as_float(rk.x);
  return rk.y >= t.k0 && ((key >= t.flo && key < t.fhi) || key >= t.wrap_lo);
}

// one blend of the draw loop; CsBlendState applies a run of them with the exact fixed-point early-out
__device__ __forceinline__ int cs_blend(int old, int pixval, int alpha) {
  return (int)(uint16_t)(((256 - alpha) * old + alpha * pixval) >> 8);  // :431
}

struct CsBlendState {
  int val, last_pv;
  bool fixed;  // val is a fixed point of blending with last_pv: more of the same changes nothing (exact)
  __device__ __forceinline__ void apply(int pv, int alpha) {
    if (fixed && pv == last_pv) return;
    const int nv = cs_blend(val, pv, alpha);
    fixed = (nv == val);
    last_pv = pv;
    val = nv;
  }
  __device__ __forceinline__ void apply_n(int pv, int cnt, int alpha) {
    while (cnt-- > 0) {
      const int nv = cs_blend(val, pv, alpha);
      if (nv == val) break;  // fixed point of this pixval
      val = nv;
    }
  }
};

// One visit: ray r at ring k.  pos = the cell's index along the ring (0 .. 8k-1, one value per cell:
// side s of the square contributes (2s+1)k +- minor, the corner 8k wraps to 0).
template <bool TILED>
__device__ __forceinline__ bool cs_ring_visit(const CsRay& r, int k, int x1, int y1, int size, int pitch_tiles, int& pos,
                                              uint32_t& cell, int& pv) {
  if (!(r.flags & 1) || k > r.dxc) return false;
  const int m = cs_ray_minor(r, k);
  const int dmaj = (r.flags & 4) ? -k : k;
  const int dmin = (r.flags & 8) ? -m : m;
  const bool steep = (r.flags & 2) != 0;
  const int ox = steep ? dmin : dmaj;
  const int oy = steep ? dmaj : dmin;
  const int x = x1 + ox, y = y1 + oy;
  if ((unsigned)x >= (unsigned)size || (unsigned)y >= (unsigned)size) return false;  // cannot happen for a clipped ray
  int p;
  if (!steep) p = (r.flags & 4) ? 5 * k - oy : k + oy;
  else p = (r.flags & 4) ? 7 * k + ox : 3 * k - ox;
  pos = (p == 8 * k) ? 0 : p;
  cell = cs_cell_offset<TILED>(x, y, size, pitch_tiles);
  pv = cs_ray_pixval(r, k);
  return true;
}

// cell of position p on ring k around (x1, y1) (inverse of cs_ring_visit's position)
__device__ __forceinline__ void cs_w_pos_to_xy(int p, int k, int x1, int y1, int& x, int& y) {
  if (p <= 2 * k) { x = x1 + k; y = y1 + (p - k); }
  else if (p <= 4 * k) { y = y1 + k; x = x1 + (3 * k - p); }
  else if (p <= 6 * k) { x = x1 - k; y = y1 + (5 * k - p); }
  else { y = y1 - k; x = x1 + (p - 7 * k); }
}

// One ray's walk, carried from ring to ring: the incremental form of cs_ring_visit (cell, position on the ring) and the
// closed form of the pixval.  init(k) puts the state ON ring k (k >= 0); step() advances it by one ring.
struct CsWWalk {
  int dxc;            // last ring of the ray; -1: this lane has no ray
  int den2, dy2, rem; // Bresenham: (2 dyc k + dxc - 1) = q * 2 dxc + rem
  int x, y, pos, k;
  int cside, g, dxM, dyM, dxN, dyN;
  int a0, b0, c0, incv, kc, ndt;
  __device__ __forceinline__ void init(const CsRay& r, bool have, int k_, int x1, int y1) {
    dxc = have ? r.dxc : -1;
    const int dyc = min(r.dyc, r.dxc);  // a clipped dyc > dxc walks the diagonal (m = k), like dyc = dxc
    den2 = 2 * max(dxc, 1); dy2 = 2 * max(dyc, 0);
    cs_w_side(r.flags, cside, g);
    const bool steep = (r.flags & 2) != 0;
    const int smaj = (r.flags & 4) ? -1 : 1, smin = (r.flags & 8) ? -1 : 1;
    dxM = steep ? 0 : smaj; dyM = steep ? smaj : 0;  // per ring
    dxN = steep ? smin : 0; dyN = steep ? 0 : smin;  // per minor step
    k = k_;
    int q = (k == 0 || dxc < 1) ? 0 : cs_ray_minor(r, k);
    rem = dy2 * k + max(dxc, 1) - 1 - q * den2;
    x = x1 + dxM * k + dxN * q; y = y1 + dyM * k + dyN * q;
    pos = cside * k + g * q;
    a0 = r.a0; b0 = r.b0; c0 = max(r.a0, r.b0 + 1); incv = r.incv; kc = r.kc; ndt = r.nd_total;
  }
  __device__ __forceinline__ void step() {
    k++;
    rem += dy2;
    if (rem >= den2) { rem -= den2; x += dxN; y += dyN; pos += g; }
    x += dxM; y += dyM; pos += cside;
  }
  __device__ __forceinline__ int posn() const { return pos == 8 * k ? 0 : pos; }  // the corner 8k is position 0
  __device__ __forceinline__ int pixval() const {  // closed form of :402-428 (cs_ray_pixval), without branches
    const int nd = max(k - a0 + 1, 0);               // descending steps taken so far (k <= b0)
    const int j = max(k - c0 + 1, 0);                // ascending steps taken so far (k >= c0); 0 in the flat zone between
    const int steps = (k <= b0) ? nd : ((j > 0) ? ndt - j : 0);
    return CS_TS_NO_OBSTACLE + steps * incv + ((k <= b0) ? 0 : min(j, kc));
  }
};

// ---- the centre: rings 0 .. CS_W_CENTER - 1, drawn by ONE block for all rays.  Every ray crosses every one of these rings,
// and almost every visit there carries the free-space pixval (the hole profile starts a hole width before the hit): blends
// of one pixval commute with themselves, so a cell visited n times with that pixval alone just needs n — counted with
// shared-memory atomics, one thread per ray — and the exact fixed-point early-out.  A cell that also sees another pixval
// (an obstacle within a few cells of the sensor) is flagged and redone exactly, in ray order, by one warp.
#define CS_W_CENTER 16
#define CS_W_CENTER_CELLS (1 + 4 * CS_W_CENTER * (CS_W_CENTER - 1))  // ring 0: 1 cell, ring k: 8k cells
__device__ __forceinline__ int cs_w_center_index(int k, int posn) { return k == 0 ? 0 : 1 + 4 * k * (k - 1) + posn; }

// one cell of ring k (position p), exactly: every ray in ray order (one warp; all lanes keep the running value)
template <bool TILED>
__device__ void cs_w_cell_exact(const CsSession& S, uint16_t* __restrict__ map, int n, int k, int p, int x1, int y1, int size,
                                int pitch_tiles, int alpha) {
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  int x, y;
  cs_w_pos_to_xy(p, k, x1, y1, x, y);
  if ((unsigned)x >= (unsigned)size || (unsigned)y >= (unsigned)size) return;
  const uint32_t cell = cs_cell_offset<TILED>(x, y, size, pitch_tiles);
  CsBlendState st;
  st.val = (int)__ldcg(map + cell); st.last_pv = -1; st.fixed = false;
  for (int base = 0; base < n; base += 32) {
    const int i = base + lane;
    int pv = 0, pos = 0;
    uint32_t c2 = 0;
    bool hit = false;
    if (i < n) {
      const CsRay r = cs_unpack_ray(S.rays[i]);
      hit = cs_ring_visit<TILED>(r, k, x1, y1, size, pitch_tiles, pos, c2, pv) && pos == p;
    }
    unsigned act = __ballot_sync(full, hit);
    while (act) {
      const int l = __ffs(act) - 1;
      act &= act - 1;
      st.apply(__shfl_sync(full, pv, l), alpha);
    }
  }
  if (lane == 0) __stcg(map + cell, (uint16_t)st.val);
}

template <bool TILED>
__device__ void cs_w_center(const CsSession& S, uint16_t* __restrict__ map, int n, int x1, int y1, int size, int pitch_tiles, int alpha,
                            unsigned* s_cnt /* CS_W_CENTER_CELLS */, int* s_flagged /* 1 + CS_W_CENTER_CELLS */) {
  const int tid = threadIdx.x, warp = tid >> 5;
  for (int i = tid; i < CS_W_CENTER_CELLS; i += CS_W_THREADS) s_cnt[i] = 0u;
  if (tid == 0) s_flagged[0] = 0;
  __syncthreads();
  for (int i = tid; i < n; i += CS_W_THREADS) {
    const CsRay r = cs_unpack_ray(S.rays[i]);
    if (!(r.flags & 1)) continue;
    CsWWalk w;
    w.init(r, true, 0, x1, y1);
#pragma unroll
    for (int k = 0; k < CS_W_CENTER; k++) {
      if (k > 0) w.step();
      if (k <= w.dxc) {
        const int idx = cs_w_center_index(k, w.posn());
        atomicAdd(&s_cnt[idx], 1u);
        if (w.pixval() != CS_TS_NO_OBSTACLE) atomicOr(&s_cnt[idx], 0x80000000u);
      }
    }
  }
  __syncthreads();
  for (int c = tid; c < CS_W_CENTER_CELLS; c += CS_W_THREADS) {
    const unsigned wd = s_cnt[c];
    const int cnt = (int)(wd & 0x7fffffffu);
    if (cnt == 0) continue;
    if (wd >> 31) { s_flagged[1 + atomicAdd(&s_flagged[0], 1)] = c; continue; }
    int k = 0;
#pragma unroll
    for (int kk = 1; kk < CS_W_CENTER; kk++) if (c >= 1 + 4 * kk * (kk - 1)) k = kk;
    const int p = k == 0 ? 0 : c - (1 + 4 * k * (k - 1));
    int x, y;
    cs_w_pos_to_xy(p, k, x1, y1, x, y);
    if ((unsigned)x >= (unsigned)size || (unsigned)y >= (unsigned)size) continue;  // (cannot happen for clipped rays)
    const uint32_t cell = cs_cell_offset<TILED>(x, y, size, pitch_tiles);
    CsBlendState st;
    st.val = (int)__ldcg(map + cell); st.last_pv = -1; st.fixed = false;
    st.apply_n(CS_TS_NO_OBSTACLE, cnt, alpha);
    __stcg(map + cell, (uint16_t)st.val);
  }
  __syncthreads();
  const int nf = s_flagged[0];
  for (int f = warp; f < nf; f += CS_W_WARPS) {
    const int c = s_flagged[1 + f];
    int k = 0;
#pragma unroll
    for (int kk = 1; kk < CS_W_CENTER; kk++) if (c >= 1 + 4 * kk * (kk - 1)) k = kk;
    cs_w_cell_exact<TILED>(S, map, n, k, k == 0 ? 0 : c - (1 + 4 * k * (k - 1)), x1, y1, size, pitch_tiles, alpha);
  }
}

// Folds the visits of one ring held by the lanes of a warp (inw lanes: position posn, pixval pv) into the staged cells:
// lanes on one cell form a group, its lowest lane applies the group in lane (= ray) order — as a count when the group has
// one pixval (blends of one value commute with themselves; exact fixed-point early-out).
__device__ __forceinline__ void cs_w_fold(bool inw, int posn, int pv, int slot, unsigned* s_val, int alpha) {
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const unsigned act = __ballot_sync(full, inw);
  if (!act) return;
  unsigned rest = 0u;  // leaders of groups with several pixvals: the other members, applied in lane order below
  bool lead = false;
  int v = 0;
  if (inw) {
    const unsigned grp = __match_any_sync(act, posn);
    lead = (grp & ((1u << lane) - 1u)) == 0u;
    unsigned same = grp;
    const bool multi = (grp & (grp - 1u)) != 0u;  // every lane of a group sees the same grp
    const unsigned mm = __ballot_sync(act, multi);
    if (multi) same = __match_any_sync(mm, ((unsigned long long)(unsigned)posn << 32) | (unsigned)pv);
    if (lead) {
      v = (int)(s_val[slot] & 0xffffu);
      if (same == grp) {  // one pixval: blends of one value commute with themselves — a count, exact fixed-point early-out
        CsBlendState st;
        st.val = v; st.last_pv = -1; st.fixed = false;
        st.apply_n(pv, __popc(grp), alpha);
        v = st.val;
      } else {
        v = cs_blend(v, pv, alpha);
        rest = grp & ~(1u << lane);
      }
    }
  }
  while (__any_sync(full, rest != 0u)) {  // warp-uniform: every leader with members left fetches its next one
    const int src = rest ? __ffs(rest) - 1 : lane;
    const int pvj = __shfl_sync(full, pv, src);
    if (rest) { v = cs_blend(v, pvj, alpha); rest &= rest - 1; }
  }
  if (lead) s_val[slot] = (unsigned)v | 0x10000u;  // touched
}

// ---- general path: any number of candidates.  The rings of the task are taken a few at a time (as many as fit the staged
// cells, at most CS_W_CHUNK): the wedge's cells of those rings go to shared memory, then the batches of 32 consecutive rays
// that can hold candidates are walked in ray order — each lane carries its ray through the rings of the chunk — and fold
// into the staged cells; the touched cells go back at the end of the chunk.  The next batch's rays are in flight while the
// current one is walked.
#define CS_W_CHUNK 8
template <bool TILED>
__device__ void cs_w_general(const CsSession& S, uint16_t* __restrict__ map, const CsWTask& t, int n, int x1, int y1, int size,
                             int pitch_tiles, int alpha, unsigned* s_val, uint32_t* s_cell, unsigned* s_bmap, int nw) {
  const int lane = threadIdx.x & 31;
  int ka = t.k0;
  while (ka <= t.k1) {
    // rings ka .. kb of this chunk and where their cells start in the staging arrays
    int off[CS_W_CHUNK + 1];
    int kb = ka - 1, cells = 0;
    off[0] = 0;
#pragma unroll
    for (int j = 0; j < CS_W_CHUNK; j++) {
      const int k = ka + j;
      int cnt = 0;
      if (k <= t.k1 && kb == k - 1) {
        cnt = cs_w_bound(k, t.bhi) - cs_w_bound(k, t.blo);
        if (off[j] + cnt <= CS_W_CAP || j == 0) kb = k;
        else cnt = 0;
      }
      off[j + 1] = off[j] + cnt;
      cells += cnt;
    }
    // (a single ring wider than the staging arrays is taken in pieces of CS_W_CAP positions)
    const int first_lo = cs_w_bound(ka, t.blo);
    const int pieces = (kb == ka && off[1] > CS_W_CAP) ? (off[1] + CS_W_CAP - 1) / CS_W_CAP : 1;
    for (int piece = 0; piece < pieces; piece++) {
      const int p_lo = piece * CS_W_CAP;                       // positions [p_lo, p_hi) of the (single) ring, relative to first_lo
      const int total = pieces > 1 ? min(CS_W_CAP, off[1] - p_lo) : cells;
      for (int i = lane; i < total; i += 32) {  // stage the cells
        int j = 0, obase = 0;
#pragma unroll
        for (int jj = 1; jj < CS_W_CHUNK; jj++)
          if (pieces == 1 && jj <= kb - ka && i >= off[jj]) { j = jj; obase = off[jj]; }
        const int k = ka + j;
        const int p = (pieces > 1) ? first_lo + p_lo + i : cs_w_bound(k, t.blo) + (i - obase);
        int x, y;
        cs_w_pos_to_xy(p, k, x1, y1, x, y);
        const bool on = (unsigned)x < (unsigned)size && (unsigned)y < (unsigned)size;
        const uint32_t cell = on ? cs_cell_offset<TILED>(x, y, size, pitch_tiles) : 0xffffffffu;
        s_cell[i] = cell;
        s_val[i] = on ? (unsigned)__ldcg(map + cell) : 0u;
      }
      __syncwarp();
      int b = cs_w_next_batch(s_bmap, nw, 0);
      int2 rk_next = make_int2(0, -1);
      int4 q_next = make_int4(0, 0, 0, 0);
      if (b >= 0 && b * 32 + lane < n) { rk_next = S.w_rk[b * 32 + lane]; q_next = S.rays[b * 32 + lane]; }
      while (b >= 0) {
        const int2 rk = rk_next;
        const int4 q = q_next;
        const int i = b * 32 + lane;
        b = cs_w_next_batch(s_bmap, nw, b + 1);
        rk_next = make_int2(0, -1);
        if (b >= 0 && b * 32 + lane < n) { rk_next = S.w_rk[b * 32 + lane]; q_next = S.rays[b * 32 + lane]; }
        const bool cand = i < n && cs_w_is_candidate(t, rk);
        if (__ballot_sync(0xffffffffu, cand) == 0u) continue;
        const CsRay r = cs_unpack_ray(q);
        CsWWalk w;
        w.init(r, cand, ka - 1, x1, y1);
        unsigned accl = (unsigned)(ka - 1) * t.blo, acch = (unsigned)(ka - 1) * t.bhi;
#pragma unroll
        for (int j = 0; j < CS_W_CHUNK; j++) {
          if (ka + j <= kb) {  // warp-uniform
            w.step();
            accl += t.blo; acch += t.bhi;
            int lo = (int)((accl + ((1u << CS_W_FIX) - 1u)) >> CS_W_FIX), hi = (int)((acch + ((1u << CS_W_FIX) - 1u)) >> CS_W_FIX);
            if (pieces > 1) { lo += p_lo; hi = min(hi, lo + CS_W_CAP); }
            const int posn = w.posn();
            const bool inw = w.k <= w.dxc && posn >= lo && posn < hi && (unsigned)w.x < (unsigned)size && (unsigned)w.y < (unsigned)size;
            cs_w_fold(inw, posn, w.pixval(), (pieces > 1 ? 0 : off[j]) + posn - lo, s_val, alpha);
          }
        }
        __syncwarp();  // the next batch may touch the same cells
      }
      for (int i = lane; i < total; i += 32) {
        const unsigned v = s_val[i];
        if (v & 0x10000u) __stcg(map + s_cell[i], (uint16_t)(v & 0xffffu));
      }
      __syncwarp();
    }
    ka = kb + 1;
  }
}

// ---- fast path: at most 32 candidates (s_list, in ray order), one per lane; rings four at a time so that four map loads per
// lane are in flight; visits of one cell inside the warp are found with match.any and applied by the lowest lane in lane order.
// One group of CS_W_G rings.  FREE: no lane is inside its hole profile on these rings (k < a0 for every ray, decided by the
// caller with one vote): every visit carries the free-space pixval, which is then a constant — no pixval evaluation, and
// same-cell visits are a count.
template <bool TILED, bool FREE>
__device__ __forceinline__ void cs_w_fast_group(uint16_t* __restrict__ map, CsWWalk& w, const CsWTask& t, int kb, int last, unsigned& accl,
                                                unsigned& acch, int size, int pitch_tiles, int alpha) {
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const unsigned lt_mask = (1u << lane) - 1u;
  uint32_t cell[CS_W_G];
  int pv[CS_W_G], val[CS_W_G];
  unsigned grp[CS_W_G], act[CS_W_G];
  unsigned inwbits = 0u, leadbits = 0u, cfbits = 0u, freebits = 0u;
  // (In parts of CS_W_H rings — all CS_W_G of them: halves measured slower — three passes each: the walk and the ownership
  // test, then the match.any of the part back to back — ~40 cycles each, and the intrinsic inside a branch would be
  // serialised by the copy the compiler puts behind it: hence all lanes take part, the lanes that do not visit with ONE
  // shared key no cell has (the cost of a match grows with its distinct keys) — then the leaders' map loads.)
#pragma unroll
  for (int h = 0; h < CS_W_G; h += CS_W_H) {
#pragma unroll
    for (int j = h; j < h + CS_W_H; j++) {
      const int k = kb + j;  // (warp-uniform)
      w.step();
      accl += t.blo; acch += t.bhi;
      const int lo = (int)((accl + ((1u << CS_W_FIX) - 1u)) >> CS_W_FIX), hi = (int)((acch + ((1u << CS_W_FIX) - 1u)) >> CS_W_FIX);
      const int posn = (w.pos == 8 * k) ? 0 : w.pos;
      const bool inw = k <= last && posn >= lo && posn < hi && (unsigned)w.x < (unsigned)size && (unsigned)w.y < (unsigned)size;
      pv[j] = FREE ? CS_TS_NO_OBSTACLE : w.pixval();
      cell[j] = cs_cell_offset<TILED>(w.x, w.y, size, pitch_tiles);  // (one value per cell of the map: the key of the match)
      if (inw) inwbits |= 1u << j;
      act[j] = __ballot_sync(full, inw);
    }
#pragma unroll
    for (int j = h; j < h + CS_W_H; j++)
      grp[j] = __match_any_sync(full, ((inwbits >> j) & 1u) ? cell[j] : 0xffffffffu);
#pragma unroll
    for (int j = h; j < h + CS_W_H; j++) {
      const bool inw = (inwbits >> j) & 1u;
      const bool lead = inw && (grp[j] & lt_mask) == 0u;
      val[j] = 0;
      if (lead) { val[j] = (int)__ldcg(map + cell[j]); leadbits |= 1u << j; }
      if (act[j] != 0u && __any_sync(full, inw && !lead)) {  // some cell of this ring has several visitors in this warp
        cfbits |= 1u << j;
        if (FREE || !__any_sync(full, inw && pv[j] != CS_TS_NO_OBSTACLE)) freebits |= 1u << j;  // ... all in free space
      }
    }
  }
#pragma unroll
  for (int j = 0; j < CS_W_G; j++) {
    const bool lead = (leadbits >> j) & 1u;
    int v = cs_blend(val[j], pv[j], alpha);
    if ((freebits >> j) & 1u) {  // warp-uniform: one pixval everywhere — blends of one value commute: a count per cell
      int more = lead ? __popc(grp[j]) - 1 : 0;
      while (more-- > 0) {
        const int nv = cs_blend(v, CS_TS_NO_OBSTACLE, alpha);
        if (nv == v) break;  // fixed point of this pixval (exact)
        v = nv;
      }
    } else if (!FREE && ((cfbits >> j) & 1u)) {  // warp-uniform: every leader fetches its members' pixvals in lane (= ray) order
      unsigned rest = lead ? (grp[j] & ~(1u << lane)) : 0u;
      const int apv = alpha * pv[j];  // (the member's half of the blend :431, so that the leader's chain is one multiply-add)
      for (int turns = __reduce_max_sync(full, __popc(rest)); turns > 0; turns--) {
        const int apvj = __shfl_sync(full, apv, __ffs(rest) - 1);  // (rest == 0: lane 31's, unused)
        if (rest) { v = (int)(uint16_t)(((256 - alpha) * v + apvj) >> 8); rest &= rest - 1; }
      }
    }
    if (lead) __stcg(map + cell[j], (uint16_t)v);
  }
}

template <bool TILED>
__device__ void cs_w_fast(const CsSession& S, uint16_t* __restrict__ map, const CsWTask& t, int ncand, const int* s_list,
                          const int4* s_rays /* the candidates' rays, already fetched by the filter; or nullptr */, int x1, int y1,
                          int size, int pitch_tiles, int alpha) {
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  CsRay r;
  r.dxc = -1; r.dyc = 0; r.a0 = 0; r.b0 = -1; r.incv = 0; r.kc = 0; r.nd_total = 0; r.flags = 0;
  if (lane < ncand) r = cs_unpack_ray(s_rays ? s_rays[lane] : S.rays[s_list[lane]]);
  CsWWalk w;
  w.init(r, lane < ncand, t.k0 - 1, x1, y1);
  const int last = min(w.dxc, t.k1);  // this lane's last ring in the task (-1: none)
  unsigned accl = (unsigned)(t.k0 - 1) * t.blo, acch = (unsigned)(t.k0 - 1) * t.bhi;

  for (int kb = t.k0; kb <= t.k1; kb += CS_W_G) {
    const bool hot = kb <= last && kb + CS_W_G - 1 >= w.a0;  // this lane's hole profile (:402-428) starts at ring a0
    if (!__any_sync(full, hot))
      cs_w_fast_group<TILED, true>(map, w, t, kb, last, accl, acch, size, pitch_tiles, alpha);
    else
      cs_w_fast_group<TILED, false>(map, w, t, kb, last, accl, acch, size, pitch_tiles, alpha);
  }
}

// Runs one task — rings ka .. kb of a level whose first ring is k0 (the wedge was sized for k0; the margins follow ka): while
// the wedge holds more candidates than a warp has lanes it is cut in halves (left part first) as long as halving can help
// (the wedge is wider than its margins); what cannot be cut takes the general path.
// PRELOAD: the filter fetches every ray it looks at together with its (key, dxc) and parks the candidates' rays in shared
// memory (the general path's cell staging, idle on the fast path): one trip to L2 less in front of the first ring, for the
// price of fetching the rays of the non-candidates of the batches looked at — the latency instance of the kernel does it.
template <bool TILED, bool PRELOAD>
__device__ void cs_w_run(const CsSession& S, uint16_t* __restrict__ map, int ka, int kb, unsigned blo, unsigned bhi, int n, int x1,
                         int y1, int size, int pitch_tiles, int alpha, unsigned* s_val, uint32_t* s_cell, int* s_list,
                         unsigned* s_bmap, long long* tl) {
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  int tl_pieces = 0, tl_cand = 0, tl_mode = 0;
  const float eps = 0.5f / (float)ka + 1e-4f;
  const unsigned min_width = (unsigned)(4.0f * eps * (float)(1 << CS_W_FIX)) + 2u;
  unsigned lo = blo;
  while (lo < bhi) {
    unsigned hi = bhi;
    CsWTask t;
    int ncand, kmax, nw;
    for (;;) {
      t.k0 = ka;
      t.k1 = kb;
      t.blo = lo;
      t.bhi = hi;
      t.flo = (float)lo * (1.0f / (float)(1 << CS_W_FIX)) - eps;
      t.fhi = (float)hi * (1.0f / (float)(1 << CS_W_FIX)) + eps;
      t.wrap_lo = (lo == 0u) ? 8.0f - eps : 9.0f;
      // candidates, in ray order; the largest dxc among them bounds the rings of the task
      ncand = 0; kmax = 0;
      nw = cs_w_batch_map(S, t, n, s_bmap);
      int b = cs_w_next_batch(s_bmap, nw, 0);
      int2 rk_next = make_int2(0, -1);
      int4 ray_next = make_int4(0, 0, 0, 0);
      if (b >= 0 && b * 32 + lane < n) {
        rk_next = S.w_rk[b * 32 + lane];
        if (PRELOAD) ray_next = S.rays[b * 32 + lane];
      }
      while (b >= 0) {
        const int2 rk = rk_next;
        const int4 ray = ray_next;
        const int i = b * 32 + lane;
        b = cs_w_next_batch(s_bmap, nw, b + 1);
        rk_next = make_int2(0, -1);
        if (b >= 0 && b * 32 + lane < n) {
          rk_next = S.w_rk[b * 32 + lane];
          if (PRELOAD) ray_next = S.rays[b * 32 + lane];
        }
        const bool cand = i < n && cs_w_is_candidate(t, rk);
        const unsigned m = __ballot_sync(full, cand);
        if (cand) {
          const int at = ncand + __popc(m & ((1u << lane) - 1u));
          if (at < 32) {
            s_list[at] = i;
            if (PRELOAD) reinterpret_cast<int4*>(s_cell)[at] = ray;
          }
        }
        ncand += __popc(m);
        kmax = max(kmax, __reduce_max_sync(full, cand ? rk.y : 0));
      }
      if (ncand <= 32 || hi - lo < min_width) break;
      hi = lo + (hi - lo) / 2u;
    }
    if (tl && lane == 0 && tl_pieces == 0) tl[1] = cs_globaltimer();
    tl_pieces++;
    tl_cand = max(tl_cand, ncand);
    if (ncand > 32) tl_mode = 1;
    if (ncand > 0) {
      t.k1 = min(t.k1, kmax);
      __syncwarp();
      if (ncand <= 32)
        cs_w_fast<TILED>(S, map, t, ncand, s_list, PRELOAD ? reinterpret_cast<const int4*>(s_cell) : nullptr, x1, y1, size, pitch_tiles, alpha);
      else
        cs_w_general<TILED>(S, map, t, n, x1, y1, size, pitch_tiles, alpha, s_val, s_cell, s_bmap, nw);
      __syncwarp();
    }
    lo = hi;
  }
  if (tl && lane == 0) { tl[2] = cs_globaltimer(); tl[3] = (long long)tl_cand | ((long long)tl_mode << 16) | ((long long)tl_pieces << 20) | ((long long)ka << 32); }
}

// Two instances per layout.  RESIDENT = 4 (64 registers, a few spills): the most warps per SM — batches of sessions and big
// scans, which are throughput.  RESIDENT = 3 (80 registers, no spills): one small scan alone, a latency chain, where a
// shorter instruction stream per ring and fewer polling blocks beside the search kernel are worth more than the warps
// (cfg2 43.6 -> 42.4 us per step, cfg1 36.4 -> 35.2; cfg5 the other way, 2.00 -> 2.08 ms).
template <bool TILED, int RESIDENT>
__global__ void __launch_bounds__(CS_W_THREADS, RESIDENT)
cs_wedge_kernel(CsSession* __restrict__ sessions, CsStepArgs a) {
  __shared__ int s_first[CS_W_LEVELS + 2];   // first (sub-)task of each level; s_first[nlev] = their number
  __shared__ int s_uniform[CS_W_LEVELS];     // > 0: the level is cut into this many equal wedges (the dense centre)
  __shared__ int s_tot[CS_W_LEVELS];         // tasks of each level
  __shared__ int s_T[CS_W_LEVELS];           // rays per wedge of a level cut by its sector counts
  __shared__ int s_split[CS_W_LEVELS];       // warps that share the rings of one task of the level
  __shared__ int s_nlev;
  __shared__ int s_ticket;
  __shared__ float sh_pose[5];
  __shared__ long long sh_vis[CS_W_WARPS];
  __shared__ unsigned s_val[CS_W_WARPS][CS_W_CAP];
  __shared__ __align__(16) uint32_t s_cell[CS_W_WARPS][CS_W_CAP];
  __shared__ int s_list[CS_W_WARPS][32];
  __shared__ unsigned s_bmap[CS_W_WARPS][CS_W_BMAP_WORDS];
  __shared__ unsigned s_center[CS_W_CENTER_CELLS];
  __shared__ int s_flagged[1 + CS_W_CENTER_CELLS];

  const unsigned full = 0xffffffffu;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const long long t_start = a.diag ? cs_globaltimer() : 0;  // diagnostics (cs_get_ring_cycles): block start, rays ready, table ready
  cs_pdl_launch_dependents();  // the next step's search may become resident once every block here has started
  // No griddepcontrol.wait in front: this kernel is resident before the search in front has ended; its preparing blocks
  // poll the pose words (CsSession::ll_pose), everybody else the preparing blocks' count (CsSession::prep_words).

  const int sj = blockIdx.y;
  CsSession& S = sessions[sj];
  const CsStepHeader& hdr = a.hdr[(size_t)sj * a.hdr_stride];
  const int n = hdr.n_points;
  const int size = S.size, pitch_tiles = S.pitch_tiles;
  const float scale = S.scale;
  const int alpha = S.quality;
  uint16_t* __restrict__ map = S.map;
  const int copies = S.ray_copies;
  const int NL = S.w_levels;
  const unsigned slot = a.step_id & 1u;
  const unsigned long long ll_tag = (unsigned long long)a.step_id << 32;
  const size_t top_words = (size_t)NL * (CS_W_SECTORS + 1);  // per (level, sector), then per level
  int* top = S.w_top + (size_t)a.w_slot * top_words;           // this scan's counts (sizes the NEXT scan's wedges)
  // The task table is built from the counts of the scan BEFORE this one when there is one (a.w_prev >= 0): scans follow each
  // other closely, any cut of the circle into wedges is correct (only the balance depends on it), and the table is then
  // ready before the pose is out.  The first scan of a handle builds it from its own counts, after its rays are ready.
  const int* tab = S.w_top + (size_t)(a.w_prev >= 0 ? a.w_prev : a.w_slot) * top_words;

  auto build_table = [&]() {
    const int* tot_tab = tab + (size_t)NL * CS_W_SECTORS;
    // wedges per level.  Where the margins of ring k0 alone hold more rays than a wedge is sized for (the centre) the level is
    // cut into equal wedges as wide as the margins; elsewhere into wedges of T rays each by the sector counts (boundaries at
    // the T-quantiles of the level's rays, interpolated inside a sector: long rays cluster in a few directions, and equal
    // wedges would leave some with several times the candidates a warp holds).
    for (int L = tid; L < NL; L += CS_W_THREADS) {
      const int k0 = cs_w_level_first(L);
      const int alive = k0 >= CS_W_CENTER ? tot_tab[L] : 0;  // (the rings of the centre are drawn by cs_w_center)
      int tot = 0, uni = 0, T = 0;
      // a level the previous scan did not reach still gets a task (one wedge, the whole circle): this scan may reach it
      if (alive <= 0 && k0 >= CS_W_CENTER && a.w_prev >= 0) { uni = 1; tot = 1; }
      if (alive > 0 && alive / (8 * k0) > CS_W_OWN / 2) {
        uni = cs_w_wedges(alive, k0);
        tot = uni;
      } else if (alive > 0) {
        T = CS_W_OWN - alive / (8 * k0);  // the margins of a wedge, 1 / k0 wide in all, hold alive / (8 k0) rays on average
        tot = (alive + T - 1) / T;
      }
      s_tot[L] = tot; s_uniform[L] = uni; s_T[L] = T;
    }
    __syncthreads();
    if (warp == 0) {
      // How many warps share the rings of one task.  The wedges of the dense levels (equal wedges as wide as their margins:
      // several passes of 32 rays per ring, the long tasks of a big scan) are always split ring by ring, up to 8 ways; the
      // others into sub-tasks of r rings, r the shortest of 4, 8, 16, 32, 64 (= whole levels) at which the table still holds at
      // most one sub-task per warp of the grid — a small scan is a latency chain: shorter tasks end it sooner, and equal lengths
      // keep the 64-ring outer levels from ending it; a big scan is throughput: whole levels amortise a task's set-up.
      const int slots = (int)gridDim.x * CS_W_WARPS;
      int rlen = 64;
      for (int r = 4; r < 64; r *= 2) {
        int cnt = 0;
        for (int L0 = 0; L0 < NL; L0 += 32) {
          const int L = L0 + lane;
          if (L < NL) {
            const int len = cs_w_level_last(L) - cs_w_level_first(L) + 1;
            cnt += s_tot[L] * (s_uniform[L] > 1 ? min(8, len) : (len + r - 1) / r);
          }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(full, cnt, o);
        if (cnt <= slots) { rlen = r; break; }
      }
      int total = 0, nlev = 0;
      for (int L0 = 0; L0 < NL; L0 += 32) {
        const int L = L0 + lane;
        int split = 1;
        if (L < NL) {
          const int len = cs_w_level_last(L) - cs_w_level_first(L) + 1;
          split = s_uniform[L] > 1 ? min(8, len) : (len + rlen - 1) / rlen;
          s_split[L] = split;
        }
        const int W = L < NL ? s_tot[L] * split : 0;
        int incl = W;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int u = __shfl_up_sync(full, incl, o);
          if (lane >= o) incl += u;
        }
        if (L < NL) s_first[L] = total + incl - W;
        const unsigned has = __ballot_sync(full, W > 0);
        if (has) nlev = L0 + 32 - __clz(has);
        total += __shfl_sync(full, incl, 31);
      }
      if (lane == 0) { s_first[nlev] = total; s_nlev = nlev; }
    }
    __syncthreads();
  };

  // ---- while the pose is not out yet: pull the part of the map the scan can reach into L2.  The centre is the pose the
  // step starts from (searchPose :728, or the given pose), the radius the ring count the host launched for plus the reach
  // of the search; one 128-byte tile per thread.  (Harmless where the map is L2-resident already: the prefetch hits.)
  if (TILED && a.w_prefetch == 2) cs_prefetch_disc(S, hdr, a, (int)blockIdx.x * CS_W_THREADS + tid, (int)gridDim.x * CS_W_THREADS);

  // ---- ray preparation: the first nprep blocks take a.prep_group rays each, one ray per thread
  const int group = a.prep_group;
  const int nprep = (n + group - 1) / group;
  const bool preparing = (int)blockIdx.x < nprep;
  if (!preparing && a.w_prev >= 0) build_table();  // (the preparing blocks build theirs after the rays: the pose comes first)
  if (preparing) {
    const float2* __restrict__ points = a.points + (size_t)sj * a.points_stride;
    const int g_begin = blockIdx.x * group, g_end = min(n, g_begin + group);
    if (blockIdx.x == 0) {  // the third of the counters that the NEXT scan will count into is this step's to re-arm
      int* other = S.w_top + (size_t)a.w_zero * top_words;
      for (int i = tid; i < (int)top_words; i += CS_W_THREADS) other[i] = 0;
    }
    // (at most CS_W_THREADS rays per block: a.prep_group <= CS_W_THREADS is what the host launches)
    const bool my_warp = g_begin + warp * 32 < g_end;  // whole warps: the warp reductions need every lane
    const int my_i = g_begin + tid;
    const bool in_range = my_warp && my_i < g_end;
    const float2 my_p = in_range ? __ldg(points + my_i) : make_float2(1.f, 0.f);  // in flight while the pose is awaited
    bool stuck = false;
    if (tid < 5) {
      volatile unsigned long long* ll = S.ll_pose + tid;
      unsigned long long w;
      CsSpin spin;
      while (((w = *ll) & 0xffffffff00000000ull) != ll_tag)
        if (spin.expired(a, CS_STUCK_POSE)) { stuck = true; break; }
      sh_pose[tid] = __uint_as_float((unsigned)w);
    }
    if (__syncthreads_or(stuck)) return;  // (bounded polls only: the pose never came)
    const float pose[3] = {sh_pose[0], sh_pose[1], sh_pose[2]};
    const float cs[2] = {sh_pose[3], sh_pose[4]};
    const CsRayFrame f = cs_ray_frame(S, pose, cs);
    long long vis = 0;
    CsWPrepared q;
    q.key = 0.f; q.dxc = -1; q.bm = -1;
    if (my_warp) {
      q = cs_w_prepare(S, f, my_p, my_i, in_range, vis);
      if (a.w_prev < 0) cs_w_count(S, q, top);  // this scan's own table needs the counts before the rays are announced
    }
    __threadfence();  // this thread's stores (and counts) are visible device-wide before the block's arrival is counted
    __syncthreads();
    if (tid < copies) atomicAdd(S.prep_words + ((size_t)slot * copies + tid) * 16, 1ull);
    // off the critical path: the counts that size the next scan's wedges, and the visit count
    if (my_warp && a.w_prev >= 0) cs_w_count(S, q, top);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) vis += __shfl_xor_sync(full, vis, o);
    if (lane == 0) sh_vis[warp] = vis;
    __syncthreads();
    if (tid == 0) {
      for (int w = 1; w < CS_W_WARPS; w++) vis += sh_vis[w];
      if (vis) {
        atomicAdd((unsigned long long*)&S.visits_slot[slot], (unsigned long long)vis);
        if (a.visits_out) atomicAdd((unsigned long long*)a.visits_out, (unsigned long long)vis);
      }
    }
    if (a.w_prev >= 0) build_table();
  }
  // ---- everybody: wait for the preparing blocks — as late as possible: with the table at hand (built from the previous
  // scan's counts) a block first draws its ticket and every warp works out its wedge, and only then are this scan's rays
  // needed.
  bool have_rays = false;
  int x1 = 0, y1 = 0;
  long long t_prep = 0;
  auto wait_rays = [&]() -> bool {  // (whole block); false: the rays never came (bounded polls only)
    bool stuck = false;
    if (tid == 0) {
      volatile unsigned long long* pw = S.prep_words + ((size_t)slot * copies + (cs_smid() % copies)) * 16;
      CsSpin spin;
      while (*pw != (unsigned long long)nprep)
        if (spin.expired(a, CS_STUCK_RAYS)) { stuck = true; break; }
      __threadfence();
    } else if (!preparing && (tid == 32 || tid == 64)) {
      // the pose words are out long before the rays are (the preparing blocks work from them): two more threads fetch x and
      // y meanwhile, instead of one more trip to L2 after the arrival
      volatile unsigned long long* ll = S.ll_pose + (tid >> 6);
      unsigned long long w;
      CsSpin spin;
      while (((w = *ll) & 0xffffffff00000000ull) != ll_tag)
        if (spin.expired(a, CS_STUCK_POSE)) { stuck = true; break; }
      sh_pose[tid >> 6] = __uint_as_float((unsigned)w);
    }
    if (__syncthreads_or(stuck)) return false;
    have_rays = true;
    if (a.diag) t_prep = cs_globaltimer();
    const float pose_x = sh_pose[0], pose_y = sh_pose[1];  // (the preparing blocks have theirs from their own poll)
    x1 = cs_cvt_i32(__fadd_rn(__fmul_rn(pose_x, scale), 0.5f));  // :499, :505
    y1 = cs_cvt_i32(__fadd_rn(__fmul_rn(pose_y, scale), 0.5f));  // :500, :506
    return true;
  };
  if (a.w_prev < 0) {  // this scan's own counts: the table needs the rays first
    if (!wait_rays()) return;
    build_table();
  }
  const long long t_sched = a.diag ? cs_globaltimer() : 0;
  const int nlev = s_nlev;
  const int n_tasks = s_first[nlev];

  // wedge and rings of (sub-)task stask; false: nothing to do
  auto decode = [&](int stask, int& ka, int& kb, unsigned& blo, unsigned& bhi) -> bool {
      int L = 0;  // level of the task: last L with s_first[L] <= stask
      {
        int lo = 0, hi = nlev - 1;
        while (lo < hi) {
          const int mid = (lo + hi + 1) >> 1;
          if (s_first[mid] <= stask) lo = mid; else hi = mid - 1;
        }
        L = lo;
      }
      const int sub = s_split[L];
      const int r = (stask - s_first[L]) / sub;
      const int sub_j = (stask - s_first[L]) % sub;
      if (s_uniform[L] > 0) {
        const int W = s_uniform[L];
        if (r >= W) return false;
        blo = cs_w_beta(r, W);
        bhi = cs_w_beta(r + 1, W);
      } else {
        // wedge r of the level holds the rays number r T .. (r + 1) T - 1 in key order (by the sector counts)
        const int c0 = tab[L * CS_W_SECTORS + lane], c1 = tab[L * CS_W_SECTORS + 32 + lane];
        int p0 = c0, p1 = c1;  // inclusive prefix sums over the 64 sectors
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int u0 = __shfl_up_sync(full, p0, o), u1 = __shfl_up_sync(full, p1, o);
          if (lane >= o) { p0 += u0; p1 += u1; }
        }
        p1 += __shfl_sync(full, p0, 31);
        const int T = s_T[L], W = s_tot[L];
        if (r >= W) return false;
        unsigned bnd[2];
#pragma unroll
        for (int e = 0; e < 2; e++) {
          const int x = (r + e) * T;  // key below which x rays of the level lie
          const unsigned b0 = __ballot_sync(full, p0 >= x), b1 = __ballot_sync(full, p1 >= x);
          unsigned v = 8u << CS_W_FIX;
          if (x <= 0) v = 0u;
          else if (b0 | b1) {
            const int sec = b0 ? __ffs(b0) - 1 : 32 + __ffs(b1) - 1;
            const int incl = sec < 32 ? __shfl_sync(full, p0, sec) : __shfl_sync(full, p1, sec - 32);
            const int cs_ = sec < 32 ? __shfl_sync(full, c0, sec) : __shfl_sync(full, c1, sec - 32);
            v = ((unsigned)sec << (CS_W_FIX - 3)) + (((unsigned)(x - (incl - cs_))) << (CS_W_FIX - 3)) / (unsigned)cs_;
          }
          bnd[e] = v;
        }
        blo = bnd[0];
        bhi = (r == W - 1) ? (8u << CS_W_FIX) : bnd[1];
      }
      // this warp's share of the level's rings
      const int k0 = cs_w_level_first(L), k1 = cs_w_level_last(L);
      const int per = (k1 - k0 + sub) / sub;
      ka = k0 + sub_j * per; kb = min(k1, ka + per - 1);
      if (ka > k1) return false;
      return true;
  };

  // ---- tasks.  The table counts sub-tasks: a task's rings split over s_split[level] warps; inner levels come first.
  const int n_sub_tasks = n_tasks;
  const int n_tickets = (n_sub_tasks + CS_W_WARPS - 1) / CS_W_WARPS;
  if (n_tickets < (int)gridDim.x) {
    // A scan with at most a ticket per block (a latency chain).  Blocks draw tickets: ticket t is the sub-tasks t,
    // t + n_tickets, t + 2 n_tickets ... — one per warp, from all over the table — and the ticket behind the last one is the
    // centre.  Blocks that become resident late (an SM the search kernel left late) find the tickets gone instead of
    // holding the scan up with tasks of their own.
    for (;;) {
      __syncthreads();  // (the previous ticket's readers are done; all warps are through their tasks)
      if (tid == 0) s_ticket = (int)atomicAdd(&S.ring_ticket[slot], 1u);
      __syncthreads();
      const int ticket = s_ticket;
      if (ticket > n_tickets) break;
      int ka = 0, kb = -1;
      unsigned blo = 0u, bhi = 0u;
      const int stask = ticket + n_tickets * warp;
      const bool ok = ticket < n_tickets && stask < n_sub_tasks && decode(stask, ka, kb, blo, bhi);
      if (!have_rays && !wait_rays()) return;
      if (ticket == n_tickets) {  // (block-uniform branch: cs_w_center has barriers)
        cs_w_center<TILED>(S, map, n, x1, y1, size, pitch_tiles, alpha, s_center, s_flagged);
        continue;
      }
      if (!ok) continue;
      long long* tl = (a.diag && sj == 0 && stask < a.diag_rings) ? a.diag + (size_t)stask * 8 : nullptr;
      if (tl && lane == 0) { tl[0] = cs_globaltimer(); tl[4] = t_start; tl[5] = t_prep; tl[6] = t_sched; tl[7] = cs_smid() | ((long long)blockIdx.x << 16); }
      cs_w_run<TILED, RESIDENT == 3>(S, map, ka, kb, blo, bhi, n, x1, y1, size, pitch_tiles, alpha, s_val[warp], s_cell[warp],
                      s_list[warp], s_bmap[warp], tl);
    }
  } else {
    // A big scan or a session of a batch (throughput): static round-robin over the warps of the session's blocks, consecutive
    // sub-tasks to different blocks, the blocks that prepared rays last; the centre to the block whose tasks come last.
    if (!have_rays && !wait_rays()) return;
    const int nblocks = (int)gridDim.x;
    int rb = (int)blockIdx.x - min(nprep, nblocks - 1);
    if (rb < 0) rb += nblocks;
    if (rb == nblocks - 1) cs_w_center<TILED>(S, map, n, x1, y1, size, pitch_tiles, alpha, s_center, s_flagged);
    for (int stask = rb + nblocks * warp; stask < n_sub_tasks; stask += nblocks * CS_W_WARPS) {
      int ka = 0, kb = -1;
      unsigned blo = 0u, bhi = 0u;
      if (!decode(stask, ka, kb, blo, bhi)) continue;
      long long* tl = (a.diag && sj == 0 && stask < a.diag_rings) ? a.diag + (size_t)stask * 8 : nullptr;
      if (tl && lane == 0) { tl[0] = cs_globaltimer(); tl[4] = t_start; tl[5] = t_prep; tl[6] = t_sched; tl[7] = cs_smid() | ((long long)blockIdx.x << 16); }
      cs_w_run<TILED, RESIDENT == 3>(S, map, ka, kb, blo, bhi, n, x1, y1, size, pitch_tiles, alpha, s_val[warp], s_cell[warp],
                      s_list[warp], s_bmap[warp], tl);
    }
  }
  cs_pdl_wait();  // the kernel in front has long finished; this only makes "this grid done" imply "that grid done"
}

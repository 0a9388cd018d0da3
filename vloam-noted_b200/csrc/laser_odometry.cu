// laser_odometry.cu -- LaserOdometry::solveLO (laser_odometry.cpp:199-584) as CUDA.
//
// Per outer pass (2 per frame, LO.cpp:224):
//   lo_assoc<false>  sharp points  -> 1-NN in cornerLast + ring-window scan -> LidarEdgeFactor slots
//   lo_assoc<true>   flat points   -> 1-NN in surfLast  + ring-window scan -> LidarPlaneFactor slots
//   vl_solve         5 evaluation kernels (lm_solver.cu) on para_q / para_t
// then lo_accumulate (LO.cpp:524-525) and the cloud swap (LO.cpp:558-564, a pointer flip).
//
// The 1-NN is exact brute force: a CTA takes 8 queries and streams the target cloud
// once through registers (8 distances per loaded point), so L2 traffic is 1/8 of a
// query-per-CTA scan; ties resolve by (d2, index) like the oracle.  The ring-window
// scans follow the reference's visit order literally (forward ascending, then backward
// descending, strict <), one warp per query, 128 points per step, with the `break`
// position found by ballot so nothing is assumed about the monotonicity of
// int(intensity) (SURVEY 7.2 item 3).
#include "common.cuh"

#define LO_QPB 8  // queries per block == warps per block

struct Best { float d; int j; };

__device__ __forceinline__ Best best_min_lo(Best a, Best b) {  // smaller d, then smaller index
  return (b.d < a.d || (b.d == a.d && b.j < a.j)) ? b : a;
}
__device__ __forceinline__ Best best_min_hi(Best a, Best b) {  // smaller d, then larger index (descending visit order)
  return (b.d < a.d || (b.d == a.d && b.j > a.j)) ? b : a;
}
__device__ __forceinline__ Best warp_best(Best v, bool preferLow) {
  for (int d = 16; d > 0; d >>= 1) {
    Best o; o.d = __shfl_xor_sync(0xffffffffu, v.d, d); o.j = __shfl_xor_sync(0xffffffffu, v.j, d);
    v = preferLow ? best_min_lo(v, o) : best_min_hi(v, o);
  }
  return v;
}

// LO.cpp:319-322: ((tx-sx)^2 + (ty-sy)^2) + (tz-sz)^2 in f32
__device__ __forceinline__ float lo_sqdis(const float4 t, float sx, float sy, float sz) {
  const float dx = __fsub_rn(t.x, sx), dy = __fsub_rn(t.y, sy), dz = __fsub_rn(t.z, sz);
  return __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
}

#define LO_TBL 144  // ring-value table: first index whose int(intensity) >= v, v in [0, LO_TBL)

// int(intensity) is the ring id and the "last" clouds are ring-major, so the `break` positions of
// the reference's scans are table look-ups -- provided the sequence really is non-decreasing.  This
// kernel builds the table and verifies that; a cloud that fails the check (a negative relTime makes
// int(intensity) = ring - 1, SURVEY 7.2 item 3) takes the ballot path that assumes nothing.
// tbl layout per cloud: [0, LO_TBL) first-index table, [LO_TBL] = 1 if monotone.
__global__ void __launch_bounds__(256) lo_ring_table(const float4* __restrict__ corner, int nc, const float4* __restrict__ surf, int ns,
                                                     int* __restrict__ tbl) {
  VL_PDL_WAIT();

  const int which = blockIdx.y;
  const float4* cl = which ? surf : corner;
  const int n = which ? ns : nc;
  int* t = tbl + which * (LO_TBL + 1);
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (n == 0) { if (j <= LO_TBL) t[j] = j == LO_TBL ? 1 : 0; return; }
  if (j >= n) return;
  const int v = min(max((int)cl[j].w, 0), LO_TBL - 1);
  const int raw = (int)cl[j].w;
  if (j == 0) { for (int q = 0; q <= v; ++q) t[q] = 0; if (raw < 0 || raw > 255) t[LO_TBL] = 0; }
  else {
    const int rawp = (int)cl[j - 1].w;
    const int vp = min(max(rawp, 0), LO_TBL - 1);
    if (raw < rawp || raw < 0 || raw > 255) t[LO_TBL] = 0;  // not monotone (or outside the packed byte): tables unusable
    for (int q = vp + 1; q <= v; ++q) t[q] = j;
  }
  if (j == n - 1) for (int q = v + 1; q < LO_TBL; ++q) t[q] = n;
}
__global__ void lo_ring_table_init(int* __restrict__ tbl) {
  VL_PDL_WAIT();
 if (threadIdx.x < 2) tbl[threadIdx.x * (LO_TBL + 1) + LO_TBL] = 1; }

template <bool SURF>
__global__ void __launch_bounds__(LO_QPB * 32) lo_assoc(const float4* __restrict__ query, int nq, const float4* __restrict__ target, int nt,
                                                        const double* __restrict__ pose, const int* __restrict__ tbl, int* __restrict__ outIdx,
                                                        double* __restrict__ factors, int* __restrict__ valid, int slotBase, double* __restrict__ factorS) {
  VL_PDL_WAIT();

  const int deskew = factorS != nullptr;
  __shared__ float sq[LO_QPB][3];
  __shared__ Best sbest[LO_QPB][LO_QPB];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q0 = blockIdx.x * LO_QPB;
  if (threadIdx.x < LO_QPB) {
    const int qi = q0 + threadIdx.x;
    float sx = 0.f, sy = 0.f, sz = 0.f;
    if (qi < nq) vl_transform_to_start(pose, query[qi], deskew, sx, sy, sz);  // TransformToStart (LO.cpp:152-173): f64 math, f32 store
    sq[threadIdx.x][0] = sx; sq[threadIdx.x][1] = sy; sq[threadIdx.x][2] = sz;
  }
  __syncthreads();
  // ---- phase 1: exact 1-NN for the block's 8 queries (kdtree nearestKSearch k = 1)
  float qx[LO_QPB], qy[LO_QPB], qz[LO_QPB];
  Best b[LO_QPB];
#pragma unroll
  for (int k = 0; k < LO_QPB; ++k) { qx[k] = sq[k][0]; qy[k] = sq[k][1]; qz[k] = sq[k][2]; b[k].d = 3.0e38f; b[k].j = -1; }
#pragma unroll 4
  for (int j = threadIdx.x; j < nt; j += LO_QPB * 32) {
    const float4 t = __ldg(&target[j]);
#pragma unroll
    for (int k = 0; k < LO_QPB; ++k) {
      const float d = vl_dist2(qx[k], qy[k], qz[k], t.x, t.y, t.z);
      if (d < b[k].d) { b[k].d = d; b[k].j = j; }
    }
  }
#pragma unroll
  for (int k = 0; k < LO_QPB; ++k) {
    if (b[k].j < 0) b[k].j = 0x7fffffff;
    const Best w = warp_best(b[k], true);
    if (lane == 0) sbest[k][warp] = w;
  }
  __syncthreads();
  // ---- phase 2: warp `warp` owns query q0 + warp
  const int qi = q0 + warp;
  if (qi >= nq) return;
  Best nn = sbest[warp][0];
#pragma unroll
  for (int w = 1; w < LO_QPB; ++w) nn = best_min_lo(nn, sbest[warp][w]);
  const float sx = sq[warp][0], sy = sq[warp][1], sz = sq[warp][2];
  int closest = -1, ind2 = -1, ind3 = -1;
  if (nt > 0 && nn.j != 0x7fffffff && (double)nn.d < 25.0) {  // DISTANCE_SQ_THRESHOLD (LO.cpp:299, 397)
    closest = nn.j;
    const int id = (int)target[closest].w;  // closestPointScanID
    Best f2{25.0f, -1}, f3{25.0f, -1};
    Best g2{25.0f, -1}, g3{25.0f, -1};
    if (tbl[LO_TBL]) {
      // monotone ring values: the scans stop at table positions, every point in between is visited
      const int F = tbl[min(id + 3, LO_TBL - 1)];            // first j with int(intensity) >= id + 3  (> id + 2.5)
      const int Bq = id - 2 <= 0 ? 0 : tbl[min(id - 2, LO_TBL - 1)];  // points below it have int(intensity) <= id - 3
#pragma unroll 4
      for (int j = closest + 1 + lane; j < F; j += 32) {   // LO.cpp:309-331, 407-430
        const float4 t = __ldg(&target[j]);
        const int v = (int)t.w;
        const float d = lo_sqdis(t, sx, sy, sz);
        if (SURF) {
          if (v <= id) { if (d < f2.d) { f2.d = d; f2.j = j; } }
          else if (d < f3.d) { f3.d = d; f3.j = j; }
        } else if (v > id) { if (d < f2.d) { f2.d = d; f2.j = j; } }
      }
#pragma unroll 4
      for (int j = closest - 1 - lane; j >= Bq; j -= 32) {  // LO.cpp:334-355, 433-456
        const float4 t = __ldg(&target[j]);
        const int v = (int)t.w;
        const float d = lo_sqdis(t, sx, sy, sz);
        if (SURF) {
          if (v >= id) { if (d < g2.d) { g2.d = d; g2.j = j; } }
          else if (d < g3.d) { g3.d = d; g3.j = j; }
        } else if (v < id) { if (d < g2.d) { g2.d = d; g2.j = j; } }
      }
    } else {
    // forward: j = closest+1 .. ; break at the first int(intensity) > id + 2.5 (LO.cpp:309-331, 407-430)
    for (int base = closest + 1; base < nt; base += 128) {
      bool stop = false;
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int j = base + u * 32 + lane;
        const bool in = j < nt;
        const float4 t = in ? __ldg(&target[j]) : make_float4(0.f, 0.f, 0.f, 0.f);
        const int v = (int)t.w;
        const bool brk = in && (double)v > (double)id + 2.5;
        const unsigned bb = __ballot_sync(0xffffffffu, brk);
        const bool live = in && (bb == 0 || lane < __ffs(bb) - 1);
        if (live) {
          const float d = lo_sqdis(t, sx, sy, sz);
          if (SURF) {
            if (v <= id) { if (d < f2.d) { f2.d = d; f2.j = j; } }
            else if (d < f3.d) { f3.d = d; f3.j = j; }
          } else if (v > id) { if (d < f2.d) { f2.d = d; f2.j = j; } }
        }
        if (bb != 0 || base + (u + 1) * 32 >= nt) { stop = true; break; }
      }
      if (stop) break;
    }
    // backward: j = closest-1 .. 0 ; break at the first int(intensity) < id - 2.5 (LO.cpp:334-355, 433-456)
    for (int base = closest - 1; base >= 0; base -= 128) {
      bool stop = false;
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int j = base - u * 32 - lane;
        const bool in = j >= 0;
        const float4 t = in ? __ldg(&target[j]) : make_float4(0.f, 0.f, 0.f, 0.f);
        const int v = (int)t.w;
        const bool brk = in && (double)v < (double)id - 2.5;
        const unsigned bb = __ballot_sync(0xffffffffu, brk);
        const bool live = in && (bb == 0 || lane < __ffs(bb) - 1);
        if (live) {
          const float d = lo_sqdis(t, sx, sy, sz);
          if (SURF) {
            if (v >= id) { if (d < g2.d) { g2.d = d; g2.j = j; } }
            else if (d < g3.d) { g3.d = d; g3.j = j; }
          } else if (v < id) { if (d < g2.d) { g2.d = d; g2.j = j; } }
        }
        if (bb != 0 || base - (u + 1) * 32 < 0) { stop = true; break; }
      }
      if (stop) break;
    }
    }
    f2 = warp_best(f2, true);
    g2 = warp_best(g2, false);
    if (SURF) { f3 = warp_best(f3, true); g3 = warp_best(g3, false); }
    // forward candidates were visited first: backward wins only when strictly nearer
    ind2 = (g2.j >= 0 && g2.d < f2.d) ? g2.j : f2.j;
    if (ind2 < 0 && g2.j >= 0) ind2 = g2.j;
    if (SURF) { ind3 = (g3.j >= 0 && g3.d < f3.d) ? g3.j : f3.j; if (ind3 < 0 && g3.j >= 0) ind3 = g3.j; }
  }
  if (lane != 0) return;
  const int slot = slotBase + qi;
  double* f = factors + (size_t)slot * 10;
  const float4 cp = query[qi];
  if (deskew) factorS[slot] = vl_point_s(cp.w);
  if (SURF) {
    outIdx[qi * 3] = closest; outIdx[qi * 3 + 1] = ind2; outIdx[qi * 3 + 2] = ind3;
    const bool ok = closest >= 0 && ind2 >= 0 && ind3 >= 0;
    valid[slot] = ok ? 1 : 0;
    if (ok) {  // LidarPlaneFactor ctor (LF.hpp:73-74): ljm_norm = normalize((j-l) x (j-m))
      const float4 J = target[closest], L = target[ind2], M = target[ind3];
      const double u[3] = {(double)J.x - (double)L.x, (double)J.y - (double)L.y, (double)J.z - (double)L.z};
      const double w[3] = {(double)J.x - (double)M.x, (double)J.y - (double)M.y, (double)J.z - (double)M.z};
      double n[3] = {u[1] * w[2] - u[2] * w[1], u[2] * w[0] - u[0] * w[2], u[0] * w[1] - u[1] * w[0]};
      const double n2 = n[0] * n[0] + n[1] * n[1] + n[2] * n[2];
      if (n2 > 0.0) { const double nn2 = sqrt(n2); n[0] /= nn2; n[1] /= nn2; n[2] /= nn2; }
      f[0] = 1.0; f[1] = cp.x; f[2] = cp.y; f[3] = cp.z;
      f[4] = J.x; f[5] = J.y; f[6] = J.z; f[7] = n[0]; f[8] = n[1]; f[9] = n[2];
    }
  } else {
    outIdx[qi * 2] = closest; outIdx[qi * 2 + 1] = ind2;
    const bool ok = ind2 >= 0;
    valid[slot] = ok ? 1 : 0;
    if (ok) {  // LidarEdgeFactor(curr, a = closest, b = second, s = 1) (LO.cpp:360-381)
      const float4 A = target[closest], B = target[ind2];
      f[0] = 0.0; f[1] = cp.x; f[2] = cp.y; f[3] = cp.z;
      f[4] = A.x; f[5] = A.y; f[6] = A.z; f[7] = B.x; f[8] = B.y; f[9] = B.z;
    }
  }
}


// ---- uniform grid over the "last" clouds -----------------------------------------------------------
// The reference rebuilds two KD-trees per frame (LO.cpp:573-574).  Here both last clouds are counting-
// sorted once per frame into 1.28 m cells (256 x 256 x 32 cells per cloud).  A search visits the 27 cells
// around the query first: they contain every point closer than 1.28 m, so a minimum below (1.25 m)^2 is
// already the global one; otherwise the 5x5x5 block (everything within 2.56 m) and, failing that, the
// 9x9x9 block (>= 5.12 m around the query, i.e. everything inside the 5 m acceptance radius of
// LO.cpp:299/397) are visited.  The less-flat cloud puts ~150 points into a 2.56 m cell near the sensor:
// with cells that large a query warp spent 20 us filtering ~4000 candidates per pass.  Entries are {x, y, z, bits(index |
// int(intensity) << 24)}.  Coordinates outside the grid are clamped, which keeps neighbours neighbours
// (clamping is monotone), so the search stays exact.
#define LOG_NX 256
#define LOG_NY 256
#define LOG_NZ 32
#define LOG_NCELL (LOG_NX * LOG_NY * LOG_NZ)
#define LOG_INV 0.78125f     // 1 / 1.28
#define LOG_NEAR1 1.5625f    // (1.25 m)^2 < cell^2: a minimum below this found in the 3x3x3 block is global
#define LOG_NEAR2 6.25f      // (2.5 m)^2 < (2 cells)^2: same for the 5x5x5 block; the 9x9x9 block covers the 5 m gate
#define LOG_OX (-163.84f)
#define LOG_OZ (-10.24f)

__device__ __forceinline__ int log_cx(float v) { return min(max((int)floorf((v - LOG_OX) * LOG_INV), 0), LOG_NX - 1); }
__device__ __forceinline__ int log_cz(float v) { return min(max((int)floorf((v - LOG_OZ) * LOG_INV), 0), LOG_NZ - 1); }
__device__ __forceinline__ int log_cell(float x, float y, float z) { return log_cx(x) + LOG_NX * (log_cx(y) + LOG_NY * log_cz(z)); }

// Round 1 counted into -- and scanned -- a dense array of 2 x 2.1M cells for ~56k points (16.8 MB read + zeroing + write per
// sweep to index 0.9 MB of points).  Now only the occupied part of the grid exists: a row of the grid (fixed y, z) is cut into
// GROUPS of 8 consecutive x-cells, and the occupied groups (~10k) live in an open-addressing hash table of H >= points slots.
// A slot is one 64-byte line {group id, start[0..8]}: the points of the group are contiguous in the cell-sorted copy, sub-cell
// after sub-cell, so the row segment [x - R, x + R] the search visits is ONE range per group it touches (<= 2 groups for
// R <= 4) and a look-up is one dependent memory access after the probe (same line).  (A hash of single cells needed 27 / 125 /
// 729 look-ups per query for R = 1 / 2 / 4; corner queries often reach R = 4 and the kernel took 64 us instead of 35.)
// Build: lo_grid_count (probe / claim the slot, count per sub-cell), lo_grid_alloc (one thread per slot: a contiguous range for
// the group from a bump counter -- one atomic per CTA -- and the nine starts), lo_grid_fill.  No scan.
// Layout of one set (ints): LoSlot[H] | cnt[8 H] | top[4]
#define LOG_EMPTY 0xffffffffu
#define LOG_G 8
#define LOG_NGX (LOG_NX / LOG_G)
#define LOG_NGROUP (LOG_NCELL / LOG_G)
struct __align__(64) LoSlot { unsigned key; int start[LOG_G + 1]; int pad[6]; };
struct LoHash { const LoSlot* slot; int mask; };
__device__ __forceinline__ unsigned log_hash(unsigned id) { id ^= id >> 15; id *= 0x9E3779B1u; id ^= id >> 13; return id; }

__global__ void __launch_bounds__(256) lo_grid_count(const float4* __restrict__ corner, int nc, const float4* __restrict__ surf, int ns,
                                                     LoSlot* __restrict__ slots, int* __restrict__ cnt, int mask, int* __restrict__ subOf) {
  VL_PDL_WAIT();

  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= nc + ns) return;
  const int which = g >= nc;
  const float4 p = which ? surf[g - nc] : corner[g];
  const int cx = log_cx(p.x);
  const unsigned id = (unsigned)(which * LOG_NGROUP + (cx >> 3) + LOG_NGX * (log_cx(p.y) + LOG_NY * log_cz(p.z)));
  unsigned h = log_hash(id) & (unsigned)mask;
  for (;;) {
    const unsigned prev = atomicCAS(&slots[h].key, LOG_EMPTY, id);
    if (prev == LOG_EMPTY || prev == id) break;
    h = (h + 1) & (unsigned)mask;
  }
  const int so = (int)h * LOG_G + (cx & 7);
  subOf[g] = so;
  atomicAdd(&cnt[so], 1);
}
// one thread per slot: the group's range in the sorted copy and the starts of its sub-cells; the counters become the fill cursors
__global__ void __launch_bounds__(256) lo_grid_alloc(LoSlot* __restrict__ slots, int* __restrict__ cnt, int* __restrict__ top) {
  VL_PDL_WAIT();

  __shared__ int ws[32];
  __shared__ int sBase;
  const int h = blockIdx.x * blockDim.x + threadIdx.x;
  const bool used = slots[h].key != LOG_EMPTY;
  int4 a = make_int4(0, 0, 0, 0), b = a;
  if (used) { a = *reinterpret_cast<const int4*>(cnt + (size_t)h * LOG_G); b = *reinterpret_cast<const int4*>(cnt + (size_t)h * LOG_G + 4); }
  const int total = a.x + a.y + a.z + a.w + b.x + b.y + b.z + b.w;
  int blockTotal = 0;
  const int ex = vl_block_excl_scan<256>(total, ws, &blockTotal);
  if (threadIdx.x == 0) sBase = blockTotal > 0 ? atomicAdd(top, blockTotal) : 0;
  __syncthreads();
  if (!used) return;
  int st = sBase + ex;
  int* o = slots[h].start;
  o[0] = st; st += a.x; o[1] = st; st += a.y; o[2] = st; st += a.z; o[3] = st; st += a.w;
  o[4] = st; st += b.x; o[5] = st; st += b.y; o[6] = st; st += b.z; o[7] = st; st += b.w; o[8] = st;
  *reinterpret_cast<int4*>(cnt + (size_t)h * LOG_G) = make_int4(0, 0, 0, 0);
  *reinterpret_cast<int4*>(cnt + (size_t)h * LOG_G + 4) = make_int4(0, 0, 0, 0);
}
__global__ void __launch_bounds__(256) lo_grid_fill(const float4* __restrict__ corner, int nc, const float4* __restrict__ surf, int ns,
                                                    const int* __restrict__ subOf, const LoSlot* __restrict__ slots,
                                                    int* __restrict__ fill, float4* __restrict__ sorted) {
  VL_PDL_WAIT();

  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= nc + ns) return;
  const int which = g >= nc;
  const int j = which ? g - nc : g;
  const float4 p = which ? surf[j] : corner[j];
  const int so = subOf[g];
  const int pos = slots[so >> 3].start[so & 7] + atomicAdd(&fill[so], 1);
  const unsigned v = (unsigned)min(max((int)p.w, 0), 255);
  sorted[pos] = make_float4(p.x, p.y, p.z, __uint_as_float((unsigned)j | (v << 24)));
}
// point range of sub-cells [lo, hi] of one group (empty when the group holds nothing)
__device__ __forceinline__ void log_lookup(const LoHash& H, unsigned id, int lo, int hi, int& beg, int& len) {
  unsigned h = log_hash(id) & (unsigned)H.mask;
  for (;;) {
    const LoSlot* sl = H.slot + h;
    const unsigned k = __ldg(&sl->key);
    if (k == id) { beg = __ldg(&sl->start[lo]); len = __ldg(&sl->start[hi + 1]) - beg; return; }
    if (k == LOG_EMPTY) { beg = 0; len = 0; return; }
    h = (h + 1) & (unsigned)H.mask;
  }
}

__device__ __forceinline__ Best warp_best_v(Best v, unsigned& tag, bool preferLow) {
  for (int d = 16; d > 0; d >>= 1) {
    Best o; o.d = __shfl_xor_sync(0xffffffffu, v.d, d); o.j = __shfl_xor_sync(0xffffffffu, v.j, d);
    const unsigned ot = __shfl_xor_sync(0xffffffffu, tag, d);
    const bool take = preferLow ? (o.d < v.d || (o.d == v.d && o.j < v.j)) : (o.d < v.d || (o.d == v.d && o.j > v.j));
    if (take) { v = o; tag = ot; }
  }
  return v;
}

// Association over the grid (valid when int(intensity) of the target cloud is non-decreasing: the
// reference's forward scan then visits exactly {j > closest : ring_j <= id + 2} and the backward scan
// {j < closest : ring_j >= id - 2}; candidates farther than 5 m can never win because the running
// minima start at DISTANCE_SQ_THRESHOLD = 25).  One warp per query, two passes over its 27 cells.
// Visit the (2R+1)^3 block of cells around (cx, cy, cz), R = 1, 2 or 4.  A block is (2R+1)^2 rows; the cells [cx - R, cx + R]
// of a row lie in one or two groups of the hash: lane l looks up (row l / 2, group l % 2) -- all look-ups of a round in ~two
// memory latencies (probe, starts on the same line); R = 1 takes one round, R = 2 two, R = 4 six -- and VL_WARP_VISIT_FLAT
// spreads the candidates of all ranges over the lanes.  A larger block simply revisits the smaller one: every update in the
// bodies below is an idempotent minimum, and escalation only happens where the inner block was nearly empty.  BODY sees float4 t.
#define LOG_VISIT(R, BODY)                                                                                   \
  do {                                                                                                       \
    const int side_ = 2 * (R) + 1;                                                                           \
    const int xs_ = max(cx - (R), 0), xe_ = min(cx + (R), LOG_NX - 1);                                       \
    const int g0_ = xs_ >> 3, g1_ = xe_ >> 3;                                                                \
    for (int r0_ = 0; r0_ < 2 * side_ * side_; r0_ += 32) {                                                  \
      const int it_ = r0_ + lane, rr_ = it_ >> 1, part_ = it_ & 1;                                           \
      int beg_ = 0, len_ = 0;                                                                                \
      if (rr_ < side_ * side_ && (part_ == 0 || g1_ != g0_)) {                                               \
        const int zz_ = cz + rr_ / side_ - (R), yy_ = cy + rr_ % side_ - (R);                                \
        if (zz_ >= 0 && zz_ < LOG_NZ && yy_ >= 0 && yy_ < LOG_NY) {                                          \
          const int g_ = part_ ? g1_ : g0_;                                                                  \
          log_lookup(H, (unsigned)(groupBase + g_ + LOG_NGX * (yy_ + LOG_NY * zz_)), part_ ? 0 : (xs_ & 7),  \
                     g_ == g1_ ? (xe_ & 7) : 7, beg_, len_);                                                 \
        }                                                                                                    \
      }                                                                                                      \
      VL_WARP_VISIT_FLAT(beg_, len_, lane, sorted, BODY);                                                    \
    }                                                                                                        \
  } while (0)

// Association over the grid (valid when int(intensity) of the target cloud is non-decreasing: the
// reference's forward scan then visits exactly {j > closest : ring_j <= id + 2} and the backward scan
// {j < closest : ring_j >= id - 2}; candidates farther than 5 m can never win because the running
// minima start at DISTANCE_SQ_THRESHOLD = 25).  One warp per query.
__constant__ int* g_lo_trace = nullptr;  // debug: per query warp {cycles, flags: 1 = shell in the NN pass, 2 = shell in the second pass}

template <bool SURF>
__device__ __forceinline__ void lo_assoc_grid_dev(int qi, int lane, const float4* __restrict__ query, const float4* __restrict__ target,
                                                  const float4* __restrict__ sorted, const LoHash H,
                                                  const double* __restrict__ pose, int* __restrict__ outIdx,
                                                  double* __restrict__ factors, int* __restrict__ valid, int slotBase, double* __restrict__ factorS) {
  const long long tr0 = g_lo_trace ? clock64() : 0;
  int trFlags = 0;
  const float4 cp = query[qi];
  float sx, sy, sz;
  vl_transform_to_start(pose, cp, factorS != nullptr, sx, sy, sz);  // TransformToStart (LO.cpp:152-173)
  const int cx = log_cx(sx), cy = log_cx(sy), cz = log_cz(sz);
  const int groupBase = SURF ? LOG_NGROUP : 0;
  // ---- pass A: exact nearest neighbour, ties by index
  Best nn{3.0e38f, 0x7fffffff};
  unsigned nnv = 0;
#define LOG_NN_BODY                                                                      \
  {                                                                                      \
    const float d = vl_dist2(sx, sy, sz, t.x, t.y, t.z);                                 \
    const unsigned bits = __float_as_uint(t.w);                                          \
    const int j = (int)(bits & 0xffffffu);                                               \
    if (d < nn.d || (d == nn.d && j < nn.j)) { nn.d = d; nn.j = j; nnv = bits >> 24; }   \
  }
  LOG_VISIT(1, LOG_NN_BODY);
  nn = warp_best_v(nn, nnv, true);
  if (!(nn.d < LOG_NEAR1)) {  // nothing within 1.25 m: widen the block (warp-uniform branches)
    trFlags |= 1;
    LOG_VISIT(2, LOG_NN_BODY);
    nn = warp_best_v(nn, nnv, true);
    if (!(nn.d < LOG_NEAR2)) {
      trFlags |= 8;
      LOG_VISIT(4, LOG_NN_BODY);
      nn = warp_best_v(nn, nnv, true);
    }
  }
  int closest = -1, ind2 = -1, ind3 = -1;
  if (nn.j != 0x7fffffff && (double)nn.d < 25.0) {  // LO.cpp:299, 397
    closest = nn.j;
    const int id = (int)nnv;
    Best f2{25.0f, 0x7fffffff}, f3{25.0f, 0x7fffffff}, g2{25.0f, -1}, g3{25.0f, -1};
#define LOG_B_BODY                                                                                        \
  {                                                                                                       \
    const unsigned bits = __float_as_uint(t.w);                                                           \
    const int j = (int)(bits & 0xffffffu);                                                                \
    const int v = (int)(bits >> 24);                                                                      \
    /* ring band first: with non-decreasing rings every class below lies in [id - 2, id + 2], and ~90 % */ \
    /* of the candidates of a 64-beam cloud fail this two-instruction test before any distance is formed */ \
    if (v >= id - 2 && v <= id + 2) {                                                                     \
    const float d = lo_sqdis(t, sx, sy, sz);                                                              \
    if (d < 25.0f) { /* the running minima start at DISTANCE_SQ_THRESHOLD; only strict < replaces them */ \
      if (j > closest) { /* forward scan LO.cpp:309-331 / 407-430 */                                      \
        if (v <= id + 2) {                                                                                \
          if (SURF) {                                                                                     \
            if (v <= id) { if (d < f2.d || (d == f2.d && j < f2.j)) { f2.d = d; f2.j = j; } }             \
            else if (d < f3.d || (d == f3.d && j < f3.j)) { f3.d = d; f3.j = j; }                         \
          } else if (v > id) { if (d < f2.d || (d == f2.d && j < f2.j)) { f2.d = d; f2.j = j; } }         \
        }                                                                                                 \
      } else if (j < closest) { /* backward scan LO.cpp:334-355 / 433-456 */                              \
        if (v >= id - 2) {                                                                                \
          if (SURF) {                                                                                     \
            if (v >= id) { if (d < g2.d || (d == g2.d && j > g2.j)) { g2.d = d; g2.j = j; } }             \
            else if (d < g3.d || (d == g3.d && j > g3.j)) { g3.d = d; g3.j = j; }                         \
          } else if (v < id) { if (d < g2.d || (d == g2.d && j > g2.j)) { g2.d = d; g2.j = j; } }         \
        }                                                                                                 \
      }                                                                                                   \
    }                                                                                                     \
    }                                                                                                     \
  }
    LOG_VISIT(1, LOG_B_BODY);
    Best F2 = warp_best(f2, true), G2 = warp_best(g2, false), F3 = f3, G3 = g3;
    if (SURF) { F3 = warp_best(f3, true); G3 = warp_best(g3, false); }
    // a class whose best candidate is nearer than the radius the visited block guarantees is settled
    if (!(fminf(F2.d, G2.d) < LOG_NEAR1) || (SURF && !(fminf(F3.d, G3.d) < LOG_NEAR1))) {
      trFlags |= 2;
      LOG_VISIT(2, LOG_B_BODY);
      F2 = warp_best(f2, true); G2 = warp_best(g2, false);
      if (SURF) { F3 = warp_best(f3, true); G3 = warp_best(g3, false); }
      if (!(fminf(F2.d, G2.d) < LOG_NEAR2) || (SURF && !(fminf(F3.d, G3.d) < LOG_NEAR2))) {
        trFlags |= 16;
        LOG_VISIT(4, LOG_B_BODY);
        F2 = warp_best(f2, true); G2 = warp_best(g2, false);
        if (SURF) { F3 = warp_best(f3, true); G3 = warp_best(g3, false); }
      }
    }
    // forward candidates were visited first: backward wins only when strictly nearer
    if (F2.j == 0x7fffffff) F2.j = -1;
    ind2 = (G2.j >= 0 && G2.d < F2.d) ? G2.j : F2.j;
    if (SURF) {
      if (F3.j == 0x7fffffff) F3.j = -1;
      ind3 = (G3.j >= 0 && G3.d < F3.d) ? G3.j : F3.j;
    }
  }
  if (lane != 0) return;
  const int slot = slotBase + qi;
  if (g_lo_trace) { g_lo_trace[2 * slot] = (int)(clock64() - tr0); g_lo_trace[2 * slot + 1] = trFlags | (SURF ? 4 : 0); }
  double* f = factors + (size_t)slot * 10;
  if (factorS) factorS[slot] = vl_point_s(cp.w);
  if (SURF) {
    outIdx[qi * 3] = closest; outIdx[qi * 3 + 1] = ind2; outIdx[qi * 3 + 2] = ind3;
    const bool ok = closest >= 0 && ind2 >= 0 && ind3 >= 0;
    valid[slot] = ok ? 1 : 0;
    if (ok) {  // LidarPlaneFactor ctor (LF.hpp:73-74)
      const float4 J = target[closest], L = target[ind2], M = target[ind3];
      const double u[3] = {(double)J.x - (double)L.x, (double)J.y - (double)L.y, (double)J.z - (double)L.z};
      const double w[3] = {(double)J.x - (double)M.x, (double)J.y - (double)M.y, (double)J.z - (double)M.z};
      double n[3] = {u[1] * w[2] - u[2] * w[1], u[2] * w[0] - u[0] * w[2], u[0] * w[1] - u[1] * w[0]};
      const double n2 = n[0] * n[0] + n[1] * n[1] + n[2] * n[2];
      if (n2 > 0.0) { const double nn2 = sqrt(n2); n[0] /= nn2; n[1] /= nn2; n[2] /= nn2; }
      f[0] = 1.0; f[1] = cp.x; f[2] = cp.y; f[3] = cp.z;
      f[4] = J.x; f[5] = J.y; f[6] = J.z; f[7] = n[0]; f[8] = n[1]; f[9] = n[2];
    }
  } else {
    outIdx[qi * 2] = closest; outIdx[qi * 2 + 1] = ind2;
    const bool ok = ind2 >= 0;
    valid[slot] = ok ? 1 : 0;
    if (ok) {  // LidarEdgeFactor (LO.cpp:360-381)
      const float4 A = target[closest], B = target[ind2];
      f[0] = 0.0; f[1] = cp.x; f[2] = cp.y; f[3] = cp.z;
      f[4] = A.x; f[5] = A.y; f[6] = A.z; f[7] = B.x; f[8] = B.y; f[9] = B.z;
    }
  }
}

template <bool SURF>
__global__ void __launch_bounds__(256) lo_assoc_grid(const float4* __restrict__ query, int nq, const float4* __restrict__ target,
                                                     const float4* __restrict__ sorted, const LoHash H,
                                                     const double* __restrict__ pose, int* __restrict__ outIdx,
                                                     double* __restrict__ factors, int* __restrict__ valid, int slotBase, double* __restrict__ factorS) {
  VL_PDL_WAIT();

  const int lane = threadIdx.x & 31;
  const int qi = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (qi >= nq) return;
  lo_assoc_grid_dev<SURF>(qi, lane, query, target, sorted, H, pose, outIdx, factors, valid, slotBase, factorS);
}

// sharp and flat queries in one launch: warps [0, nS) run the corner association, [nS, nS + nF) the surf one
__global__ void __launch_bounds__(256) lo_assoc_grid_both(const float4* __restrict__ sharp, const float4* __restrict__ flat, int slotBound,
                                                          const SrScalars* __restrict__ srs, const float4* __restrict__ cornerLast, const float4* __restrict__ surfLast,
                                                          const float4* __restrict__ sorted, const LoHash H,
                                                          const double* __restrict__ pose, int* __restrict__ cornerIdx, int* __restrict__ surfIdx,
                                                          double* __restrict__ factors, int* __restrict__ valid, double* __restrict__ factorS) {
  VL_PDL_WAIT(); vl_chain_stamp(11);

  const int lane = threadIdx.x & 31;
  const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nS = srs->nSharp, nF = srs->nFlat;  // device-side counts: the host may not know them yet
  if (w >= nS + nF) { if (w < slotBound && lane == 0) valid[w] = 0; return; }
  if (w < nS) lo_assoc_grid_dev<false>(w, lane, sharp, cornerLast, sorted, H, pose, cornerIdx, factors, valid, 0, factorS);
  else if (w < nS + nF) lo_assoc_grid_dev<true>(w - nS, lane, flat, surfLast, sorted, H, pose, surfIdx, factors, valid, nS, factorS);
}

__global__ void lo_accumulate(LoScalars* s) {
  VL_PDL_WAIT();
  // LO.cpp:524-525
  if (threadIdx.x != 0) return;
  double r[3];
  vl_qrot(s->q_w, s->para_t[0], s->para_t[1], s->para_t[2], r);
  s->t_w[0] = s->t_w[0] + r[0]; s->t_w[1] = s->t_w[1] + r[1]; s->t_w[2] = s->t_w[2] + r[2];
  double qn[4];
  vl_qmul(s->q_w, s->para_q, qn);
  for (int k = 0; k < 4; ++k) s->q_w[k] = qn[k];
}

// LO.cpp:537-556 (VLOAM_FLAG_TRANSFORM_TO_END): every point of a[0, na) followed by b[0, nb) through TransformToEnd with
// pose = {q_last_curr, t_last_curr}, out of place.  na / nb are device counts (a look-ahead solve is queued before the host knows
// them); na == nullptr takes the host count naHost.
__global__ void __launch_bounds__(256) lo_transform_to_end(const float4* __restrict__ a, const int* __restrict__ na, int naHost, float4* __restrict__ ea,
                                                           const float4* __restrict__ b, const int* __restrict__ nb, float4* __restrict__ eb,
                                                           const double* __restrict__ pose, int deskew) {
  VL_PDL_WAIT();
  const int n0 = na ? *na : naHost, n1 = nb ? *nb : 0;
  const double P[7] = {pose[0], pose[1], pose[2], pose[3], pose[4], pose[5], pose[6]};
  for (int g = blockIdx.x * blockDim.x + threadIdx.x; g < n0 + n1; g += gridDim.x * blockDim.x) {
    if (g < n0) ea[g] = vl_transform_to_end(P, a[g], deskew);
    else eb[g - n0] = vl_transform_to_end(P, b[g - n0], deskew);
  }
}

// This sweep's less-sharp / less-flat clouds (generation c->cur of the scan-registration set swapped in) into the end buffers of
// the same generation, with the odometry state c->los, on the current stream.  Raw clouds stay readable; a discarded look-ahead
// result only ever wrote the end buffers of its own generation.
static int lo_queue_to_end(vloam_b200_ctx* c) {
  const int g = c->cur;
  VL_TRY(vl_reserve(c, c->endSharp[g], max(c->lessSharp[g].cap, (size_t)1)));
  VL_TRY(vl_reserve(c, c->endFlat[g], max(c->lessFlat[g].cap, (size_t)1)));
  VL_BYTES(32.0 * ((double)c->nLessSharp + c->nLessFlat));  // (last known counts)
  VL_LAUNCH(lo_transform_to_end, c->num_sms * 4, 256, 0, (const float4*)c->lessSharp[g].p, (const int*)&c->srs->nLessSharp, 0, c->endSharp[g].p,
            (const float4*)c->lessFlat[g].p, (const int*)&c->srs->nLessFlat, c->endFlat[g].p, (const double*)c->los->para_q, vl_distortion(c) ? 1 : 0);
  VL_CUDA(cudaGetLastError());
  return VLOAM_OK;
}
// the full-resolution cloud (n points, host count) through the same TransformToEnd, on the context's main stream
int vl_lo_to_end_cloud(vloam_b200_ctx* c, const float4* d_in, int n, float4* d_out) {
  VL_BYTES(32.0 * n);
  VL_LAUNCH(lo_transform_to_end, c->num_sms * 4, 256, 0, d_in, (const int*)nullptr, n, d_out, (const float4*)nullptr, (const int*)nullptr,
            (float4*)nullptr, (const double*)c->los->para_q, vl_distortion(c) ? 1 : 0);
  VL_CUDA(cudaGetLastError());
  return VLOAM_OK;
}

__global__ void lo_set_prior(LoScalars* s, const double* __restrict__ prior) {
  VL_PDL_WAIT();
  // LO.cpp:237-250
  if (threadIdx.x < 4) s->para_q[threadIdx.x] = prior[threadIdx.x];
  else if (threadIdx.x < 7) s->para_t[threadIdx.x - 4] = prior[threadIdx.x];
}

// Per-frame structures over the clouds that just became "last" (the reference rebuilds its KD-trees at
// this point, LO.cpp:573-574): ring tables + monotonicity flags, and the search grid.  The two flags are
// copied to pinned host memory; the next frame's first sync point makes them readable.
int vl_lo_build_last(vloam_b200_ctx* c, int set, const float4* corner, int nc, const float4* surf, int ns) {
  const int n = nc + ns;
  cudaStream_t st = VL_STREAM(c);  // (the caller selects the side stream through vl_tls_stream: the helper thread may be the one issuing this)
  // set `set` was searched by the odometry solve before the current one: rebuild it only behind the solves queued so far
  if (!c->sideWaitsIssued) VL_CUDA(cudaStreamWaitEvent(st, c->evLoSolve, 0));
  int* tbl = c->loRingTbl + set * 2 * (LO_TBL + 1);
  VL_LAUNCH(lo_ring_table_init, 1, 32, 0, tbl);
  VL_LAUNCH(lo_ring_table, dim3(vl_div_up(max(max(nc, ns), LO_TBL + 1), 256), 2), 256, 0, corner, nc, surf, ns, tbl);
  VL_CUDA(cudaMemcpyAsync(&c->h_vScalars[8 + 2 * set], tbl + LO_TBL, sizeof(int), cudaMemcpyDeviceToHost, st));
  VL_CUDA(cudaMemcpyAsync(&c->h_vScalars[9 + 2 * set], tbl + (LO_TBL + 1) + LO_TBL, sizeof(int), cudaMemcpyDeviceToHost, st));
  // hash of occupied 8-cell row groups: H >= points slots of 16 ints, then 8 H sub-cell counters and the bump counter
  int H = 1 << 15; while (H < n) H <<= 1;
  VL_TRY(vl_reserve(c, c->loGridCells[set], (size_t)24 * H + 4));
  c->loGridMask[set] = H - 1;
  VL_TRY(vl_reserve(c, c->loGridCellOf, (size_t)max(n, 1), false, (size_t)n / 2));
  VL_TRY(vl_reserve(c, c->loGridSorted[set], (size_t)max(n, 1), false, (size_t)n / 2));
  if (n > 0 && n < (1 << 24)) {
    LoSlot* slots = reinterpret_cast<LoSlot*>(c->loGridCells[set].p); int* cnt = c->loGridCells[set].p + (size_t)16 * H; int* top = cnt + (size_t)8 * H;
    VL_CUDA(cudaMemsetAsync(slots, 0xff, sizeof(LoSlot) * H, st));                 // every key = LOG_EMPTY
    VL_CUDA(cudaMemsetAsync(cnt, 0, sizeof(int) * ((size_t)8 * H + 4), st));      // counters and the bump counter
    VL_BYTES(16.0 * n);  // SURVEY 8(d) B_lo: the clouds that become "last" are read once to build their search structure
    VL_LAUNCH(lo_grid_count, vl_div_up(n, 256), 256, 0, corner, nc, surf, ns, slots, cnt, H - 1, c->loGridCellOf.p);
    VL_LAUNCH(lo_grid_alloc, H / 256, 256, 0, slots, cnt, top);
    VL_BYTES(32.0 * n);
    VL_LAUNCH(lo_grid_fill, vl_div_up(n, 256), 256, 0, corner, nc, surf, ns, c->loGridCellOf.p, (const LoSlot*)slots, cnt, c->loGridSorted[set].p);
    c->loGridValid[set] = true;
  } else c->loGridValid[set] = false;
  VL_CUDA(cudaGetLastError());
  return VLOAM_OK;
}

// upper bounds on the query counts that hold before the host has read them (SR.cpp:386-400, 452)
static inline int lo_sharp_bound(const vloam_b200_ctx* c) { return c->prm.n_scans * VL_SECTORS * 2; }
static inline int lo_flat_bound(const vloam_b200_ctx* c) { return c->prm.n_scans * VL_SECTORS * 4; }

static int lo_associate(vloam_b200_ctx* c, const double* d_pose, const float4* cornerLast, int nCL, const float4* surfLast, int nSL) {
  const int nS = c->sr_counts_valid ? c->nSharp : lo_sharp_bound(c), nF = c->sr_counts_valid ? c->nFlat : lo_flat_bound(c);
  VL_TRY(vl_reserve(c, c->loCornerIdx, (size_t)max(nS, 1) * 2));
  VL_TRY(vl_reserve(c, c->loSurfIdx, (size_t)max(nF, 1) * 3));
  VL_TRY(vl_reserve(c, c->loFactors, (size_t)max(nS + nF, 1) * 10));
  VL_TRY(vl_reserve(c, c->loFactorValid, (size_t)max(nS + nF, 1)));
  if (vl_distortion(c)) VL_TRY(vl_reserve(c, c->factorS, (size_t)max(nS + nF, 1)));
  double* fS = vl_distortion(c) ? c->factorS.p : nullptr;
  // h_vScalars[8/9]: int(intensity) of the corner / surf cloud is non-decreasing (read after a sync point)
  const int set = c->lastSet;
  const bool gridC = c->loGridValid[set] && (c->loAssumeMonotone || c->h_vScalars[8 + 2 * set] != 0);
  const bool gridS = c->loGridValid[set] && (c->loAssumeMonotone || c->h_vScalars[9 + 2 * set] != 0);
  LoHash start;  // (hash of the occupied row groups of set `set`)
  start.slot = reinterpret_cast<const LoSlot*>(c->loGridCells[set].p); start.mask = c->loGridMask[set];
  const float4* gsorted = c->loGridSorted[set].p;
  const int* rtbl = c->loRingTbl + set * 2 * (LO_TBL + 1);
  if (gridC && gridS && nS + nF > 0) {
    VL_BYTES(16.0 * ((double)c->nSharp + c->nFlat + nCL + nSL));  // SURVEY 8(d) B_lo, one pass: every query and every point of the two last clouds once
    VL_LAUNCH(lo_assoc_grid_both, vl_div_up((long long)(nS + nF) * 32, 256), 256, 0, c->sharp.p, c->flat.p, nS + nF, c->srs, cornerLast, surfLast,
              gsorted, start, d_pose, c->loCornerIdx.p, c->loSurfIdx.p, c->loFactors.p, c->loFactorValid.p, fS);
    VL_CUDA(cudaGetLastError());
    return VLOAM_OK;
  }
  if (nS > 0) {
    if (gridC)
      VL_LAUNCH(lo_assoc_grid<false>, vl_div_up((long long)nS * 32, 256), 256, 0, c->sharp.p, nS, cornerLast, gsorted, start, d_pose,
                c->loCornerIdx.p, c->loFactors.p, c->loFactorValid.p, 0, fS);
    else
      VL_LAUNCH(lo_assoc<false>, vl_div_up(nS, LO_QPB), LO_QPB * 32, 0, c->sharp.p, nS, cornerLast, nCL, d_pose, rtbl, c->loCornerIdx.p,
                c->loFactors.p, c->loFactorValid.p, 0, fS);
  }
  if (nF > 0) {
    if (gridS) {
      VL_BYTES(16.0 * ((double)nF + nSL));
      VL_LAUNCH(lo_assoc_grid<true>, vl_div_up((long long)nF * 32, 256), 256, 0, c->flat.p, nF, surfLast, gsorted, start, d_pose,
                c->loSurfIdx.p, c->loFactors.p, c->loFactorValid.p, nS, fS);
    } else
      VL_LAUNCH(lo_assoc<true>, vl_div_up(nF, LO_QPB), LO_QPB * 32, 0, c->flat.p, nF, surfLast, nSL, d_pose, rtbl + (LO_TBL + 1), c->loSurfIdx.p,
                c->loFactors.p, c->loFactorValid.p, nS, fS);
  }
  VL_CUDA(cudaGetLastError());
  return VLOAM_OK;
}

int vl_chain_trace_arm_lo(void* dev) { return cudaMemcpyToSymbol(g_chain_trace, &dev, sizeof(void*)) == cudaSuccess ? VLOAM_OK : VLOAM_E_CUDA; }
int vl_lo_preload(vloam_b200_ctx* c) {  // see vl_sr_set_attrs: load every kernel of this file when a context is created
  cudaFuncAttributes fa_;
  VL_CUDA(cudaFuncGetAttributes(&fa_, lo_ring_table)); VL_CUDA(cudaFuncGetAttributes(&fa_, lo_ring_table_init));
  VL_CUDA(cudaFuncGetAttributes(&fa_, lo_assoc<false>)); VL_CUDA(cudaFuncGetAttributes(&fa_, lo_assoc<true>));
  VL_CUDA(cudaFuncGetAttributes(&fa_, lo_grid_count)); VL_CUDA(cudaFuncGetAttributes(&fa_, lo_grid_alloc)); VL_CUDA(cudaFuncGetAttributes(&fa_, lo_grid_fill));
  VL_CUDA(cudaFuncGetAttributes(&fa_, lo_assoc_grid<false>)); VL_CUDA(cudaFuncGetAttributes(&fa_, lo_assoc_grid<true>));
  VL_CUDA(cudaFuncGetAttributes(&fa_, lo_assoc_grid_both)); VL_CUDA(cudaFuncGetAttributes(&fa_, lo_accumulate));
  VL_CUDA(cudaFuncGetAttributes(&fa_, lo_set_prior)); VL_CUDA(cudaFuncGetAttributes(&fa_, lo_transform_to_end));
  return VLOAM_OK;
}

extern bool vl_debug_capture(const vloam_b200_ctx* c);

// debug: the first call arms the per-warp trace of the grid association; later calls copy it out (n ints)
int vl_lo_trace(vloam_b200_ctx* c, int* out, int n) {
  static int* d_buf = nullptr;
  const int cap = 2 * 8192;
  if (!d_buf) {
    VL_CUDA(cudaMalloc(&d_buf, sizeof(int) * cap));
    VL_CUDA(cudaMemset(d_buf, 0, sizeof(int) * cap));
    VL_CUDA(cudaMemcpyToSymbol(g_lo_trace, &d_buf, sizeof(int*)));
  }
  VL_CUDA(cudaStreamSynchronize(c->stream));
  VL_CUDA(cudaMemcpy(out, d_buf, sizeof(int) * min(n, cap), cudaMemcpyDeviceToHost));
  return VLOAM_OK;
}

// The two association + solve passes (LO.cpp:224-553) and the pose accumulation, queued on the current stream against
// the context's current scan-registration set and odometry state (c->los).
static int lo_queue_solve(vloam_b200_ctx* c, const double* prior_q, const double* prior_t, int use_prior) {
  double* d_pose = c->los->para_q;  // para_q[4] + para_t[3] are contiguous
    const float4* cornerLast = c->cornerLastPtr; const float4* surfLast = c->surfLastPtr;
    double* d_prior = reinterpret_cast<double*>(c->vScalars + 32);  // 8-byte aligned scratch (7 doubles)
    if (use_prior) {
      double h[7] = {prior_q[0], prior_q[1], prior_q[2], prior_q[3], prior_t[0], prior_t[1], prior_t[2]};
      VL_CUDA(cudaMemcpyAsync(d_prior, h, sizeof h, cudaMemcpyHostToDevice, VL_STREAM(c)));
      VL_CUDA(cudaStreamSynchronize(VL_STREAM(c)));  // h is a stack buffer
    }
    for (int pass = 0; pass < 2; ++pass) {  // LO.cpp:224
      if (use_prior) VL_LAUNCH(lo_set_prior, 1, 32, 0, c->los, d_prior);
      VL_TRY(lo_associate(c, d_pose, cornerLast, c->nCornerLast, surfLast, c->nSurfLast));
      if (vl_debug_capture(c)) {
        VL_TRY(vl_reserve(c, c->dbgLoCorner[pass], (size_t)max(c->nSharp, 1) * 2));
        VL_TRY(vl_reserve(c, c->dbgLoSurf[pass], (size_t)max(c->nFlat, 1) * 3));
        VL_CUDA(cudaMemcpyAsync(c->dbgLoCorner[pass].p, c->loCornerIdx.p, sizeof(int) * 2 * c->nSharp, cudaMemcpyDeviceToDevice, VL_STREAM(c)));
        VL_CUDA(cudaMemcpyAsync(c->dbgLoSurf[pass].p, c->loSurfIdx.p, sizeof(int) * 3 * c->nFlat, cudaMemcpyDeviceToDevice, VL_STREAM(c)));
      }
      const int nslots = c->sr_counts_valid ? c->nSharp + c->nFlat : lo_sharp_bound(c) + lo_flat_bound(c);
      VL_TRY(vl_solve_buf(c, c->loFactors.p, c->loFactorValid.p, nslots, &c->srs->nQueries, d_pose, vl_debug_capture(c) ? &c->dbgLoCost[pass * 2] : nullptr,
                          c->nSharp + c->nFlat, vl_distortion(c) ? c->factorS.p : nullptr, 8));
    }
    VL_LAUNCH(lo_accumulate, 1, 32, 0, c->los);
    if (vl_to_end(c)) VL_TRY(lo_queue_to_end(c));  // LO.cpp:537-556, before the swap: evLoSolve / evLoNext cover it
  VL_CUDA(cudaEventRecord(c->evLoSolve, VL_STREAM(c)));
  return VLOAM_OK;
}

// Look-ahead odometry.  Called by the mapping stage just before it waits at sync point S2: when the next sweep's scan
// registration is already in flight (vl_launch_lookahead), its odometry solve depends on nothing the host still has to
// decide -- the "last" clouds and their search structures are this sweep's (evLast), the counts are read on the
// device -- so it is queued now, behind this sweep's mapping, on a COPY of the odometry state.  The next
// laser_odometry call adopts the copy if it is for that sweep and ignores it otherwise.
// Part 1 (vl_lo_lookahead_solve) queues the solve; part 2 (vl_lo_lookahead_stacks), called after sync point S2 has been recorded, issues the next
// sweep's stack filters if its scan registration finishes before this sweep's mapping does.
static bool lo_lookahead_possible(const vloam_b200_ctx* c) {
  static const bool off = getenv("VLOAM_NO_LO_LOOKAHEAD") != nullptr;
  return !off && c->srNextValid && c->lo_inited && !c->prof_name[0] && !vl_debug_capture(c) && c->loGridValid[c->lastSet];
}
// It runs on its own stream, BESIDE this sweep's mapping (own factor slots): it needs this sweep's odometry result (evLoSolve),
// the structures over this sweep's clouds (evLast) and the next sweep's features (evSRfeat) -- nothing of the mapping.
static int lo_lookahead_waits(vloam_b200_ctx* c) {
  VL_CUDA(cudaStreamWaitEvent(c->streamLO, c->evLoSolve, 0));
  VL_CUDA(cudaStreamWaitEvent(c->streamLO, c->evLast, 0));
  // (sharp + flat of the next sweep: not its per-ring voxel filter -- unless its TransformToEnd reads the less-flat cloud as well)
  VL_CUDA(cudaStreamWaitEvent(c->streamLO, vl_to_end(c) ? c->srNext->evSR : c->srNext->evSRfeat, 0));
  return VLOAM_OK;
}
int vl_lo_lookahead_solve(vloam_b200_ctx* c, bool flush, bool waitsIssued) {
  c->loNextValid = false; c->loNextQueued = false;
  if (flush) VL_TRY(vl_lo_flush_deferred(c));  // (records evLast)
  // The structures over this sweep's clouds may still be being built on the side stream: wait for them on the DEVICE and
  // assume what the host cannot know yet -- that both clouds have monotone ring ids, i.e. the grid search applies.
  // The flags are checked when the result is adopted; a wrong guess only discards the look-ahead.
  if (!lo_lookahead_possible(c)) return VLOAM_OK;
  const int set = c->lastSet;
  if (!waitsIssued) VL_TRY(lo_lookahead_waits(c));
  if (c->timing) cudaEventRecord(c->evx[9], c->streamLO);
  VL_CUDA(cudaMemcpyAsync(c->losNext, c->los, sizeof(LoScalars), cudaMemcpyDeviceToDevice, c->streamLO));
  const int curNow = c->cur;
  vl_sr_swap(c, *c->srNext);
  { LoScalars* t_ = c->los; c->los = c->losNext; c->losNext = t_; }
  c->loAssumeMonotone = true;
  vl_tls_stream = c->streamLO;
  int r = lo_queue_solve(c, nullptr, nullptr, 0);  // (host counts of that sweep not known yet: bounds, the kernels read the counts on the device)
  vl_tls_stream = nullptr;
  if (r == VLOAM_OK && cudaEventRecord(c->evLoNext, c->streamLO) != cudaSuccess) r = VLOAM_E_CUDA;
  if (c->timing) cudaEventRecord(c->evx[6], c->streamLO);
  c->loAssumeMonotone = false;
  { LoScalars* t_ = c->los; c->los = c->losNext; c->losNext = t_; }
  vl_sr_swap(c, *c->srNext);
  c->cur = curNow;
  if (r != VLOAM_OK) return r;
  c->loNextQueued = true; c->loNextSet = set;
  return VLOAM_OK;
}
int vl_lo_lookahead_stacks(vloam_b200_ctx* c) {
  if (!c->loNextQueued) return VLOAM_OK;
  c->loNextQueued = false;
  // The host only waits for S2 from here on.  If the look-ahead scan registration finishes before this sweep's mapping
  // does, the next sweep's stack filters (LM.cpp:492-500) are issued now as well, into the spare stack buffers.
  const bool mapNext = ((c->lo_frameCount + 1) % c->prm.mapping_skip_frame) == 0;
  static const bool noStacksNext = getenv("VLOAM_NO_STACKS_LOOKAHEAD") != nullptr;
  bool srDone = false;
  int r = VLOAM_OK;
  // Under VLOAM_FLAG_TRANSFORM_TO_END the next sweep's stacks come from its end clouds, i.e. from the look-ahead solve queued just
  // now, which may still be discarded: they are filtered in the plain order, after that solve is adopted (vl_lo_run).
  if (mapNext && !noStacksNext && !vl_to_end(c)) {
    for (;;) {
      cudaError_t e = cudaEventQuery(c->srNext->evSR);
      if (e == cudaSuccess) { srDone = true; break; }
      if (e != cudaErrorNotReady) break;                  // a real error: the next checked call reports it
      e = cudaEventQuery(c->evS2);
      if (e != cudaErrorNotReady) break;                  // mapping finished first: never hold the pose back for the stacks
    }
    (void)cudaGetLastError();  // (cudaErrorNotReady is a status, not a failure: do not leave it for the next cudaGetLastError check)
  }
  if (srDone) {
    const int curNow = c->cur;
    vl_sr_swap(c, *c->srNext);
    r = vl_sr_sync_counts(c);
    const float4* nCorner = c->lessSharp[c->cur].p; const int nNc = c->nLessSharp; const float4* nSurf = c->lessFlat[c->cur].p; const int nNs = c->nLessFlat;
    vl_sr_swap(c, *c->srNext);
    c->cur = curNow;
    if (r == VLOAM_OK) r = vl_lm_enqueue_stacks_next(c, nCorner, nNc, nSurf, nNs);
  }
  if (r != VLOAM_OK) return r;
  c->loNextValid = true;
  return VLOAM_OK;
}

// The side-stream work a look-ahead replay defers out of the odometry call: the registered next sweep's upload + scan
// registration (streamSR) and the search structures over this sweep's clouds (stream2).  Thread-agnostic: the helper thread runs it
// while the caller queues the mapping stage (vl_lo_submit_side), or the caller itself (vl_lo_flush_deferred).
int vl_lo_side_work(vloam_b200_ctx* c) {
  int r = VLOAM_OK;
  // One sweep ahead: its scan registration heads the chain SR -> odometry and goes first.  Two sweeps ahead: the next sweep's scan
  // registration is done; when its odometry is queued already (sideWaitsIssued) nothing waits for the builds and the upload +
  // scan registration of the sweep after next, the longest chain, goes first; otherwise that odometry waits for the structures over
  // this sweep's clouds and they go first.
  if (c->earlyLoArmed) {  // the next sweep's odometry: its stream waits were issued by the caller before anything below re-records their events
    c->earlyLoArmed = false;
    r = vl_lo_lookahead_solve(c, false, true);
    if (r != VLOAM_OK) { c->sideWaitsIssued = false; return r; }
  }
  const bool srFirst = c->srDeferred && (!c->srNextValid || c->sideWaitsIssued);
  if (srFirst) { c->srDeferred = false; r = vl_launch_lookahead(c); }
  if (r == VLOAM_OK && (c->loDeferred || c->preDeferred)) {
    cudaStream_t prev = vl_tls_stream;
    vl_tls_stream = c->stream2;
    if (c->loDeferred) { c->loDeferred = false; r = vl_lo_build_last(c, c->defSet, c->defCorner, c->defNc, c->defSurf, c->defNs); }
    if (r == VLOAM_OK && c->preDeferred) {  // the structures of the NEXT sweep, into the set this sweep's odometry searched
      c->preDeferred = false;
      r = vl_lo_build_last(c, c->preSet, c->preCorner, c->preNc, c->preSurf, c->preNs);
      c->loPreValid = r == VLOAM_OK;
    }
    vl_tls_stream = prev;
    if (r != VLOAM_OK) { c->sideWaitsIssued = false; return r; }
    VL_CUDA(cudaEventRecord(c->evLast, c->stream2));
    if (c->timing) VL_CUDA(cudaEventRecord(c->evx[5], c->stream2));
  }
  if (r == VLOAM_OK && c->srDeferred) { c->srDeferred = false; r = vl_launch_lookahead(c); }
  c->sideWaitsIssued = false;
  return r;
}
// Plan the pre-build (caller thread, before the side work is submitted): the next sweep's clouds and counts are known when its
// scan registration has finished.  Set lastSet ^ 1 is the one this sweep's odometry searched.
int vl_lo_plan_prebuild(vloam_b200_ctx* c) {
  c->preDeferred = false;
  static const bool off = getenv("VLOAM_NO_PREBUILD") != nullptr;
  // (under VLOAM_FLAG_TRANSFORM_TO_END the next sweep's "last" clouds are its end clouds, which do not exist before its own
  // odometry solve: nothing to pre-build, its structures are built in the plain order)
  if (off || vl_to_end(c) || !c->srNextValid || c->loPreValid || cudaEventQuery(c->srNext->evSR) != cudaSuccess) { (void)cudaGetLastError(); return VLOAM_OK; }
  vl_sr_swap(c, *c->srNext);
  const int r = vl_sr_sync_counts(c);
  c->preCorner = c->lessSharp[c->cur].p; c->preNc = c->nLessSharp; c->preSurf = c->lessFlat[c->cur].p; c->preNs = c->nLessFlat;
  vl_sr_swap(c, *c->srNext);
  if (r != VLOAM_OK) return r;
  c->preSet = c->lastSet ^ 1;
  c->preDeferred = true;
  return VLOAM_OK;
}
// Early look-ahead (two sweeps ahead, structures pre-built): the next sweep's odometry is queued BEFORE this sweep's mapping
// launches -- its inputs are complete -- and the side streams are ordered behind the odometry solves queued so far first, because
// the solve queued here re-records evLoSolve (the side work must wait for this sweep's solve, not for the next one's).
// Only the stream WAITS are issued here (they capture the events' current records: evLast before the side work re-records it,
// evLoSolve before the solve itself does); the launches follow once the first mapping pass is queued (vl_lo_lookahead_solve with
// waitsIssued), so the mapping's first kernels are not held back by ~20 us of launch calls.
int vl_lo_early_lookahead(vloam_b200_ctx* c, bool* armed) {
  *armed = false;
  if (c->loDeferred || c->sideSubmitted || !c->srAdopted || !lo_lookahead_possible(c)) return VLOAM_OK;  // (loDeferred: the structures over this sweep's clouds are not built yet)
  VL_CUDA(cudaStreamWaitEvent(c->streamSR, c->evLoSolve, 0));
  VL_CUDA(cudaStreamWaitEvent(c->stream2, c->evLoSolve, 0));
  c->sideWaitsIssued = true;
  VL_TRY(lo_lookahead_waits(c));
  *armed = true; c->earlyLoArmed = true;
  return VLOAM_OK;
}
int vl_lo_submit_side(vloam_b200_ctx* c) {
  if (!c->srDeferred && !c->loDeferred && !c->preDeferred && !c->earlyLoArmed) { c->sideWaitsIssued = false; return VLOAM_OK; }
  VL_TRY(vl_lm_submit_task(c, vl_lo_side_work));
  c->sideSubmitted = true;
  return VLOAM_OK;
}
int vl_lo_flush_deferred(vloam_b200_ctx* c) {
  if (c->sideSubmitted) { c->sideSubmitted = false; VL_TRY(vl_lm_join(c)); }  // the helper thread has it: wait until it is issued
  return vl_lo_side_work(c);
}

int vl_lo_run(vloam_b200_ctx* c, const double* prior_q, const double* prior_t, int use_prior) {
  VL_TRY(vl_lo_flush_deferred(c));
  VL_CUDA(cudaStreamWaitEvent(c->stream, c->evLoNext, 0));  // a look-ahead solve (adopted below, or stale) owns the odometry's factor slots until it is done
  VL_CUDA(cudaEventSynchronize(c->evLast));  // set [lastSet] (built underneath the previous frame) and its flags are complete
  // The grid kernels read the query counts on the device, so the odometry can be queued before the host
  // has them (sync point S1 then costs no GPU idle time).  The ballot fallback and the debug snapshots
  // need host counts first.
  const int set = c->lastSet;
  const bool early = c->loGridValid[set] && c->h_vScalars[8 + 2 * set] != 0 && c->h_vScalars[9 + 2 * set] != 0 && !vl_debug_capture(c);
  if (!early) VL_TRY(vl_sr_sync_counts(c));
  // Scan registration already complete when the sweep arrived (look-ahead): sync point S1 is free, and the stack
  // filters of this sweep go to the helper thread now instead of behind the odometry launches.
  const bool mapThisFrame = ((c->lo_frameCount + 1) % c->prm.mapping_skip_frame) == 0;  // LO.cpp:668
  bool stacksQueued = false;
  c->stacksAdopted = false;
  if (c->stacksNextReady) {  // this sweep's stacks were filtered underneath the previous sweep's mapping
    c->stacksNextReady = false;
    if (c->srAdopted && mapThisFrame) { VL_TRY(vl_sr_sync_counts(c)); VL_TRY(vl_lm_adopt_stacks_next(c)); stacksQueued = true; c->stacksAdopted = true; }
  }
  const bool toEnd = vl_to_end(c);
  // (under VLOAM_FLAG_TRANSFORM_TO_END the stacks are filtered from the end clouds: queued below, once this sweep's solve is)
  if (!toEnd && !stacksQueued && early && mapThisFrame && cudaEventQuery(c->evSR) == cudaSuccess) {
    VL_TRY(vl_sr_sync_counts(c));
    VL_TRY(vl_lm_enqueue_stacks(c, c->lessSharp[c->cur].p, c->nLessSharp, c->lessFlat[c->cur].p, c->nLessFlat, true));
    stacksQueued = true;
  }
  // The solve of this sweep was queued behind the previous sweep's mapping (vl_lo_lookahead_solve) into the spare state:
  // adopting it is a pointer swap.  Anything that could make it stale clears loNextValid.
  const bool adoptLO = c->loNextValid && c->srAdopted && !use_prior && early && c->lo_inited && c->loNextSet == set;  // (early: grid valid, both flags set, no capture)
  c->loNextValid = false;
  if (adoptLO) { LoScalars* t_ = c->los; c->los = c->losNext; c->losNext = t_; }
  else if (c->lo_inited) VL_TRY(lo_queue_solve(c, prior_q, prior_t, use_prior));  // LO.cpp:209-217: the first frame only initialises
  else if (toEnd) {  // ... but LO.cpp:537-556 runs on it too, with q_last_curr = identity, t_last_curr = 0
    VL_TRY(lo_queue_to_end(c));
    VL_CUDA(cudaEventRecord(c->evLoSolve, VL_STREAM(c)));
  }
  // this sweep's clouds as LaserOdometry hands them on: in the sweep-end frame under the flag (the main stream is behind the
  // transform here: queued above, or waited for through evLoNext when the look-ahead solve was adopted)
  const float4* outCorner = toEnd ? c->endSharp[c->cur].p : c->lessSharp[c->cur].p;
  const float4* outSurf = toEnd ? c->endFlat[c->cur].p : c->lessFlat[c->cur].p;
  if (toEnd) {
    VL_CUDA(cudaEventRecord(c->evEnd, c->stream));
    if (early && mapThisFrame && cudaEventQuery(c->evSR) == cudaSuccess) {
      VL_TRY(vl_sr_sync_counts(c));
      VL_TRY(vl_lm_enqueue_stacks(c, outCorner, c->nLessSharp, outSurf, c->nLessFlat, true));
      stacksQueued = true;
    }
  }
  // With the solve adopted, the stacks queued and the mapping stage following in the same call, nothing on the pose
  // chain depends on the search structures of the next "last" clouds: they are queued by the mapping stage right after
  // its own launches (vl_lo_flush_deferred).
  const bool defer = adoptLO && stacksQueued && c->inProcessFrame && mapThisFrame;
  if (defer) c->srDeferred = c->srPendCount > 0;  // ... and so is the next sweep's scan registration: the helper thread issues both while the caller queues the mapping
  else VL_TRY(vl_launch_lookahead(c));  // the next sweep's scan registration, if one is registered, goes to its side stream now
  VL_HOST_MARK(2);
  VL_TRY(vl_sr_sync_counts(c));  // sync point S1 (event after scan registration; the odometry above is already queued)
  if (mapThisFrame && !stacksQueued)
    VL_TRY(vl_lm_enqueue_stacks(c, outCorner, c->nLessSharp, outSurf, c->nLessFlat));
  // built during the previous sweep (two sweeps registered ahead)?
  const bool preHit = c->loPreValid && c->srAdopted && c->preSet == (c->lastSet ^ 1) && c->preCorner == c->lessSharp[c->cur].p && c->preNc == c->nLessSharp &&
                      c->preSurf == c->lessFlat[c->cur].p && c->preNs == c->nLessFlat && c->loGridValid[c->lastSet ^ 1];
  c->loPreValid = false;
  if (preHit) {
    // nothing to build: evLast was recorded behind that build
  } else if (defer) {
    c->loDeferred = true; c->defSet = c->lastSet ^ 1;
    c->defCorner = outCorner; c->defNc = c->nLessSharp; c->defSurf = outSurf; c->defNs = c->nLessFlat;
  } else {  // LO.cpp:573-574 (setInputCloud on both KD-trees) for the clouds that become "last" after this solve:
     // they are this frame's less-sharp / less-flat clouds, final since scan registration, so the side
     // stream builds them while the odometry still searches the previous set (end clouds: behind this solve, evLoSolve)
    vl_tls_stream = c->stream2;
    const int r = vl_lo_build_last(c, c->lastSet ^ 1, outCorner, c->nLessSharp, outSurf, c->nLessFlat);
    vl_tls_stream = nullptr;
    if (r != VLOAM_OK) return r;
    VL_CUDA(cudaEventRecord(c->evLast, c->stream2));
    if (c->timing) VL_CUDA(cudaEventRecord(c->evx[5], c->stream2));
  }
  c->lo_inited = true;
  // LO.cpp:558-574: this frame's less-sharp / less-flat clouds become the "last" clouds
  c->cornerLastPtr = const_cast<float4*>(outCorner); c->surfLastPtr = const_cast<float4*>(outSurf);
  c->nCornerLast = c->nLessSharp; c->nSurfLast = c->nLessFlat;
  c->lastSet ^= 1;
  c->lo_frameCount++;
  c->skip_frame = (c->lo_frameCount % c->prm.mapping_skip_frame) != 0;  // LO.cpp:668-678
  VL_CUDA(cudaGetLastError());
  return VLOAM_OK;
}

// Association only, at an explicit pose; nothing in the context's odometry state changes.
int vl_lo_associate_only(vloam_b200_ctx* c, const double* x, int* corner_idx, int* surf_idx) {
  VL_TRY(vl_sr_sync_counts(c));
  double* d_x = reinterpret_cast<double*>(c->vScalars + 32);
  VL_CUDA(cudaMemcpyAsync(d_x, x, 7 * sizeof(double), cudaMemcpyHostToDevice, c->stream));
  VL_CUDA(cudaStreamSynchronize(c->stream));
  VL_TRY(lo_associate(c, d_x, c->cornerLastPtr, c->nCornerLast, c->surfLastPtr, c->nSurfLast));
  if (corner_idx && c->nSharp) VL_CUDA(cudaMemcpyAsync(corner_idx, c->loCornerIdx.p, sizeof(int) * 2 * c->nSharp, cudaMemcpyDeviceToHost, c->stream));
  if (surf_idx && c->nFlat) VL_CUDA(cudaMemcpyAsync(surf_idx, c->loSurfIdx.p, sizeof(int) * 3 * c->nFlat, cudaMemcpyDeviceToHost, c->stream));
  VL_CUDA(cudaStreamSynchronize(c->stream));
  return VLOAM_OK;
}

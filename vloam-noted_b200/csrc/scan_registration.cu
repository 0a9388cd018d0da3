// scan_registration.cu -- ScanRegistration::input (scan_registration.cpp:144-513) as CUDA.
//
// Data flow per sweep (all on c->stream, no host round trip inside):
//   sr_find_bounds   first / last point surviving the NaN + range filter -> startOri / endOri
//   sr_classify      per point: filter, ring id, -atan2f, first-half trigger, per-block ring histogram
//   sr_ring_scan     per-ring exclusive scan over blocks (+ ring starts, last-block-done)
//   sr_scatter       stable ring-major scatter + relTime / intensity (halfPassed == index > trigger)
//   sr_curvature     11-tap literal left fold
//   sr_pick          one CTA per ring: 6 sector sorts + greedy sharp / less-sharp / flat walks
//   sr_ring_voxel    one CTA per ring: select label<=0, pcl::VoxelGrid(0.2) restated
//   sr_offsets       prefix sums of the per-(ring,sector) pick counts and per-ring DS counts
//   sr_gather        compaction into the four feature clouds in the reference's push order
//
// Parity notes: every f32 expression is evaluated with explicitly rounded ops in the
// reference's order (the TU is also built with -fmad=false); atanf / atan2f are the
// fdlibm routines of exact_math.h, bit-identical to glibc 2.39.
#include <limits.h>
#include <math_constants.h>
#include "common.cuh"
#include "exact_math.h"
extern bool vl_debug_capture(const vloam_b200_ctx* c);
#include "bitonic.cuh"

#define SR_BLOCK 256
#define SR_PICK_THREADS 512  // sr_pick / sr_ring_voxel: one CTA per ring, the sorts want the threads
#define SR_SECT_CAP 1024   // sector keys sorted in shared memory up to this size
#define SR_RING_CAP 8192   // picked flags kept in shared memory up to this ring length
#define SR_VOX_CAP 4096    // ring voxel keys sorted in shared memory up to this size
#define VL_PI 3.14159265358979323846

__device__ __forceinline__ void sr_load(const float* in, int i, int stride, bool vec4, float& x, float& y, float& z) {
  if (vec4) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(in) + i);
    x = v.x; y = v.y; z = v.z;
  } else {
    const float* p = in + (size_t)i * stride;
    x = __ldg(p); y = __ldg(p + 1); z = __ldg(p + 2);
  }
}

// pcl::removeNaNFromPointCloud + removeClosedPointCloud (SR.cpp:107-141, 174-176)
__device__ __forceinline__ bool sr_valid1(float x, float y, float z, float thres2) {
  if (!isfinite(x) || !isfinite(y) || !isfinite(z)) return false;
  const float d2 = __fadd_rn(__fadd_rn(__fmul_rn(x, x), __fmul_rn(y, y)), __fmul_rn(z, z));
  return !(d2 < thres2);
}

// Ring id (SR.cpp:217-259) with the C++ promotion rules spelled out; -1 = rejected.
__device__ __forceinline__ int sr_ring_of(float x, float y, float z, int nscans) {
  const float h = __fsqrt_rn(__fadd_rn(__fmul_rn(x, x), __fmul_rn(y, y)));
  const float a180 = __fmul_rn(vlx::atanf_exact(__fdiv_rn(z, h)), 180.0f);
  const float angle = (float)__ddiv_rn((double)a180, VL_PI);
  int scanID;
  if (nscans == 16) {
    const float t = __fdiv_rn(__fadd_rn(angle, 15.0f), 2.0f);
    scanID = (int)__dadd_rn((double)t, 0.5);
    if (scanID > 15 || scanID < 0) return -1;
  } else if (nscans == 32) {
    const double t = __ddiv_rn(__dmul_rn(__dadd_rn((double)angle, 92.0 / 3.0), 3.0), 4.0);
    scanID = (int)t;
    if (scanID > 31 || scanID < 0) return -1;
  } else if (nscans == 64) {
    if ((double)angle >= -8.83) scanID = (int)__dadd_rn(__dmul_rn((double)__fsub_rn(2.0f, angle), 3.0), 0.5);
    else scanID = 32 + (int)__dadd_rn(__dmul_rn(__dsub_rn(-8.83, (double)angle), 2.0), 0.5);
    if (angle > 2.0f || (double)angle < -24.33 || scanID > 50 || scanID < 0) return -1;
  } else {  // 128-beam builder extension (oracle_stages.cpp, SURVEY 8d)
    const double v = __dadd_rn(__ddiv_rn(__dadd_rn((double)angle, 22.5), 45.0 / 127.0), 0.5);
    scanID = (int)v;
    if (v < 0.0 || scanID > 127) return -1;
  }
  return scanID;
}

__device__ __forceinline__ float sr_ori_first(float ori, float startOri) {  // SR.cpp:267-274
  if ((double)ori < __dsub_rn((double)startOri, VL_PI / 2)) ori = (float)__dadd_rn((double)ori, 2 * VL_PI);
  else if ((double)ori > __dadd_rn((double)startOri, VL_PI * 3 / 2)) ori = (float)__dsub_rn((double)ori, 2 * VL_PI);
  return ori;
}

__global__ void __launch_bounds__(1024) sr_find_bounds(const float* __restrict__ in, int n, int stride, int vec4, float thres2,
                                                       SrScalars* __restrict__ s) {
  VL_PDL_WAIT();

  __shared__ int found;
  int first = -1, last = -1;
  for (int base = 0; base < n; base += blockDim.x) {
    if (threadIdx.x == 0) found = INT_MAX;
    __syncthreads();
    const int i = base + threadIdx.x;
    if (i < n) { float x, y, z; sr_load(in, i, stride, vec4, x, y, z); if (sr_valid1(x, y, z, thres2)) atomicMin(&found, i); }
    __syncthreads();
    const int f = found;
    __syncthreads();
    if (f != INT_MAX) { first = f; break; }
  }
  for (int top = n; top > 0; top -= blockDim.x) {
    if (threadIdx.x == 0) found = -1;
    __syncthreads();
    const int i = top - 1 - (int)threadIdx.x;
    if (i >= 0) { float x, y, z; sr_load(in, i, stride, vec4, x, y, z); if (sr_valid1(x, y, z, thres2)) atomicMax(&found, i); }
    __syncthreads();
    const int f = found;
    __syncthreads();
    if (f >= 0) { last = f; break; }
  }
  if (threadIdx.x == 0) {
    s->firstValid = first; s->lastValid = last; s->trigger = INT_MAX; s->blocksDone = 0;
    s->count = 0; s->nSharp = s->nLessSharp = s->nFlat = s->nLessFlat = 0; s->nQueries = 0;
    float so = 0.f, eo = 0.f;
    if (first >= 0) {
      float x, y, z;
      sr_load(in, first, stride, vec4, x, y, z);
      so = -vlx::atan2f_exact(y, x);                                       // SR.cpp:185
      sr_load(in, last, stride, vec4, x, y, z);
      eo = (float)__dadd_rn((double)(-vlx::atan2f_exact(y, x)), 2 * VL_PI);  // SR.cpp:187
      if ((double)__fsub_rn(eo, so) > 3 * VL_PI) eo = (float)__dsub_rn((double)eo, 2 * VL_PI);
      else if ((double)__fsub_rn(eo, so) < VL_PI) eo = (float)__dadd_rn((double)eo, 2 * VL_PI);
    }
    s->startOri = so; s->endOri = eo;
  }
}

__global__ void __launch_bounds__(SR_BLOCK) sr_classify(const float* __restrict__ in, int n, int stride, int vec4, float thres2,
                                                        int nscans, SrScalars* __restrict__ s, int* __restrict__ ring,
                                                        float* __restrict__ oriOut, int* __restrict__ blockHist, int numBlocks) {
  VL_PDL_WAIT();

  __shared__ int hist[VL_MAX_RINGS];
  for (int t = threadIdx.x; t < VL_MAX_RINGS; t += blockDim.x) hist[t] = 0;
  __syncthreads();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  int r = -1; float ori = 0.f; bool trig = false;
  if (i < n) {
    float x, y, z; sr_load(in, i, stride, vec4, x, y, z);
    if (sr_valid1(x, y, z, thres2)) {
      r = sr_ring_of(x, y, z, nscans);
      if (r >= 0) {
        ori = -vlx::atan2f_exact(y, x);  // SR.cpp:263
        const float so = s->startOri;
        const float o1 = sr_ori_first(ori, so);
        trig = (double)__fsub_rn(o1, so) > VL_PI;  // SR.cpp:276
        atomicAdd(&hist[r], 1);
      }
    }
    ring[i] = r; oriOut[i] = ori;
  }
  const unsigned b = __ballot_sync(0xffffffffu, trig);
  if (b && (threadIdx.x & 31) == __ffs(b) - 1) atomicMin(&s->trigger, i);
  __syncthreads();
  for (int t = threadIdx.x; t < nscans; t += blockDim.x) blockHist[(size_t)t * numBlocks + blockIdx.x] = hist[t];
}

// One warp per ring: exclusive scan of that ring's per-block counts.  The last CTA
// to finish turns the ring totals into ring starts (SR.cpp:308-315).
__global__ void __launch_bounds__(256) sr_ring_scan(int* __restrict__ blockHist, int numBlocks, int nscans, int* __restrict__ ringCount,
                                                    int* __restrict__ ringStart, SrScalars* __restrict__ s) {
  VL_PDL_WAIT();

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int r = blockIdx.x * 8 + warp;
  if (r < nscans) {
    int* h = blockHist + (size_t)r * numBlocks;
    int carry = 0;
    for (int base = 0; base < numBlocks; base += 32) {
      const int b = base + lane;
      const int v = b < numBlocks ? h[b] : 0;
      int inc = v;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) { const int t = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += t; }
      if (b < numBlocks) h[b] = carry + inc - v;
      carry += __shfl_sync(0xffffffffu, inc, 31);
    }
    if (lane == 0) ringCount[r] = carry;
  }
  __shared__ int isLast;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) isLast = (atomicAdd(&s->blocksDone, 1) == (int)gridDim.x - 1);
  __syncthreads();
  if (isLast && warp == 0) {
    __threadfence();
    int carry = 0;
    for (int base = 0; base < nscans; base += 32) {
      const int rr = base + lane;
      const int v = rr < nscans ? ((volatile int*)ringCount)[rr] : 0;
      int inc = v;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) { const int t = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += t; }
      if (rr < nscans) ringStart[rr] = carry + inc - v;
      carry += __shfl_sync(0xffffffffu, inc, 31);
    }
    if (lane == 0) { ringStart[nscans] = carry; s->count = carry; }
  }
}

__global__ void __launch_bounds__(SR_BLOCK) sr_scatter(const float* __restrict__ in, int n, int stride, int vec4, int nscans,
                                                       const SrScalars* __restrict__ s, const int* __restrict__ ring,
                                                       const float* __restrict__ oriIn, const int* __restrict__ blockOff, int numBlocks,
                                                       const int* __restrict__ ringStart, float4* __restrict__ cloud) {
  VL_PDL_WAIT();

  __shared__ int warpCnt[SR_BLOCK / 32][VL_MAX_RINGS];
  for (int t = threadIdx.x; t < (SR_BLOCK / 32) * VL_MAX_RINGS; t += blockDim.x) (&warpCnt[0][0])[t] = 0;
  __syncthreads();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int r = i < n ? ring[i] : -1;
  const int key = r >= 0 ? r : (-1 - lane);  // rejected lanes never match anyone
  const unsigned m = __match_any_sync(0xffffffffu, key);
  const int rankInWarp = __popc(m & ((1u << lane) - 1u));
  if (r >= 0 && rankInWarp == 0) warpCnt[warp][r] = __popc(m);
  __syncthreads();
  if (r < 0) return;
  int before = 0;
  for (int w = 0; w < warp; ++w) before += warpCnt[w][r];
  const int dst = ringStart[r] + blockOff[(size_t)r * numBlocks + blockIdx.x] + before + rankInWarp;
  float x, y, z; sr_load(in, i, stride, vec4, x, y, z);
  const float so = s->startOri, eo = s->endOri;
  float ori = oriIn[i];
  if (i <= s->trigger) {  // halfPassed still false when this point is processed (SR.cpp:265-280)
    ori = sr_ori_first(ori, so);
  } else {                // SR.cpp:281-292
    ori = (float)__dadd_rn((double)ori, 2 * VL_PI);
    if ((double)ori < __dsub_rn((double)eo, VL_PI * 3 / 2)) ori = (float)__dadd_rn((double)ori, 2 * VL_PI);
    else if ((double)ori > __dadd_rn((double)eo, VL_PI / 2)) ori = (float)__dsub_rn((double)ori, 2 * VL_PI);
  }
  const float relTime = __fdiv_rn(__fsub_rn(ori, so), __fsub_rn(eo, so));       // SR.cpp:294
  const float inten = (float)__dadd_rn((double)r, __dmul_rn(0.1, (double)relTime));  // SR.cpp:296
  cloud[dst] = make_float4(x, y, z, inten);
}

__global__ void __launch_bounds__(SR_BLOCK) sr_curvature(const float4* __restrict__ cloud, const SrScalars* __restrict__ s,
                                                         float* __restrict__ curv, int* __restrict__ label,
                                                         unsigned char* __restrict__ picked) {
  VL_PDL_WAIT();

  __shared__ float4 tile[SR_BLOCK + 10];
  const int count = s->count;
  const int base = blockIdx.x * blockDim.x;
  if (base >= count) return;
  for (int t = threadIdx.x; t < SR_BLOCK + 10; t += blockDim.x) {
    const int g = base - 5 + t;
    tile[t] = (g >= 0 && g < count) ? cloud[g] : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  __syncthreads();
  const int i = base + threadIdx.x;
  if (i >= count) return;
  float cv = 0.f;
  if (i >= 5 && i < count - 5) {  // SR.cpp:323-339, strict left fold
    const float4* p = &tile[threadIdx.x + 5];
#define SR_FOLD(f)                                                                                         \
  __fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(__fsub_rn(__fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(     \
      p[-5].f, p[-4].f), p[-3].f), p[-2].f), p[-1].f), __fmul_rn(10.0f, p[0].f)), p[1].f), p[2].f), p[3].f), p[4].f), p[5].f)
    const float dx = SR_FOLD(x), dy = SR_FOLD(y), dz = SR_FOLD(z);
#undef SR_FOLD
    cv = __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
  }
  curv[i] = cv; label[i] = 0; picked[i] = 0;
}

__device__ __forceinline__ float sr_gap2(const float4* __restrict__ cloud, int a, int b) {  // SR.cpp:408-411
  const float4 p = cloud[a], q = cloud[b];
  const float dx = __fsub_rn(p.x, q.x), dy = __fsub_rn(p.y, q.y), dz = __fsub_rn(p.z, q.z);
  return __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
}

// Mark ind and its +-5 neighbours until a gap > 0.05 (SR.cpp:403-429); warp-cooperative.
// gb[k] (ring-local) = squared gap between points k and k-1 exceeds 0.05, precomputed for the ring.
// Only positions in [lo, hi] are written; forward marks beyond hi are returned as a bit mask
// (bit b = position hi + 1 + b), backward marks below lo are dropped (that sector is already final).
__device__ __forceinline__ unsigned sr_mark(const unsigned char* gb, unsigned char* pk, int loc, int lane, int lo, int hi) {
  bool brk = false;
  if (lane < 5) brk = gb[loc + lane + 1] != 0;            // l = lane+1: gap(ind+l, ind+l-1)
  else if (lane < 10) brk = gb[loc - (lane - 4) + 1] != 0;  // l = -(lane-4): gap(ind+l, ind+l+1)
  const unsigned bb = __ballot_sync(0xffffffffu, brk);
  const unsigned f = bb & 31u, w = (bb >> 5) & 31u;
  const int nf = f ? __ffs(f) - 1 : 5, nb = w ? __ffs(w) - 1 : 5;
  if (lane == 0) pk[loc] = 1;
  if (lane < nf && loc + lane + 1 <= hi) pk[loc + lane + 1] = 1;
  if (lane >= 5 && lane - 5 < nb && loc - (lane - 4) >= lo) pk[loc - (lane - 4)] = 1;
  unsigned spill = 0;
  const int over = loc + nf - hi;  // forward marks that land beyond hi: positions hi+1 .. loc+nf
  if (over > 0) spill = ((1u << over) - 1u) << max(loc + 1 - (hi + 1), 0);
  __syncwarp();
  return spill;
}

__device__ __forceinline__ int sr_sp(int start, int end, int j) { return start + (end - start) * j / 6; }          // SR.cpp:360
__device__ __forceinline__ int sr_ep(int start, int end, int j) { return start + (end - start) * (j + 1) / 6 - 1; }  // SR.cpp:361

// Greedy walks of one sector (SR.cpp:371-483), warp-cooperative: 32 sorted candidates per ballot.
// pre: marks already present on the first five points of the sector (bit b = point sp + b);
// [lo, hi]: ring-local range this walk may mark.  Returns the forward spill of its marks beyond hi.
__device__ __forceinline__ unsigned sr_walk_sector(int j, int r, int start, int end, int rs, const unsigned long long* __restrict__ ks,
                                                   const unsigned char* gb, unsigned char* pk, int* __restrict__ label,
                                                   int* __restrict__ provSharp, int* __restrict__ provLess, int* __restrict__ provFlat,
                                                   int* __restrict__ cntSharp, int* __restrict__ cntLess, int* __restrict__ cntFlat, int lane,
                                                   unsigned pre, int lo, int hi) {
  const int spj = sr_sp(start, end, j), epj = sr_ep(start, end, j);
  const int m = epj - spj + 1;
  const int slot = r * VL_SECTORS + j;
  unsigned spill = 0;
  if (lane < 5 && ((pre >> lane) & 1u) && lane < m) pk[spj - rs + lane] = 1;
  __syncwarp();
  // ---- descending walk: sharp (<=2) then less sharp (<=20 total), SR.cpp:371-431
  int cnt = 0, pos = m - 1;
  while (pos >= 0 && cnt < 20) {
    const int k = pos - lane;
    const bool valid = k >= 0;
    const unsigned long long key = valid ? ks[k] : 0ull;
    const int ind = (int)(unsigned)(key & 0xffffffffull);
    const bool big = valid && (double)__uint_as_float((unsigned)(key >> 32)) > 0.1;
    const bool cand = big && pk[ind - rs] == 0;
    const unsigned bc = __ballot_sync(0xffffffffu, cand);
    if (bc == 0) {
      const unsigned bv = __ballot_sync(0xffffffffu, valid), bb = __ballot_sync(0xffffffffu, big);
      if (bb != bv) break;  // reached curvature <= 0.1: nothing further can qualify
      pos -= 32;
      continue;
    }
    const int first = __ffs(bc) - 1;
    const int pind = __shfl_sync(0xffffffffu, ind, first);
    cnt++;
    if (lane == 0) {
      if (cnt <= 2) { label[pind] = 2; provSharp[slot * 2 + cnt - 1] = pind; }
      else label[pind] = 1;
      provLess[slot * 20 + cnt - 1] = pind;
    }
    spill |= sr_mark(gb, pk, pind - rs, lane, lo, hi);
    pos = pos - first - 1;
  }
  if (lane == 0) { cntSharp[slot] = min(cnt, 2); cntLess[slot] = cnt; }
  // ---- ascending walk: flat (<=4; the 4th is not marked), SR.cpp:439-483
  cnt = 0; pos = 0;
  while (pos < m && cnt < 4) {
    const int k = pos + lane;
    const bool valid = k < m;
    const unsigned long long key = valid ? ks[k] : 0ull;
    const int ind = (int)(unsigned)(key & 0xffffffffull);
    const bool small = valid && (double)__uint_as_float((unsigned)(key >> 32)) < 0.1;
    const bool cand = small && pk[ind - rs] == 0;
    const unsigned bc = __ballot_sync(0xffffffffu, cand);
    if (bc == 0) {
      const unsigned bv = __ballot_sync(0xffffffffu, valid), bs = __ballot_sync(0xffffffffu, small);
      if (bs != bv) break;
      pos += 32;
      continue;
    }
    const int first = __ffs(bc) - 1;
    const int pind = __shfl_sync(0xffffffffu, ind, first);
    cnt++;
    if (lane == 0) { label[pind] = -1; provFlat[slot * 4 + cnt - 1] = pind; }
    if (cnt >= 4) break;
    spill |= sr_mark(gb, pk, pind - rs, lane, lo, hi);
    pos = pos + first + 1;
  }
  if (lane == 0) cntFlat[slot] = cnt;
  __syncwarp();
  return spill;
}

__device__ long long* g_sr_trace = nullptr;  // debug: clock64 phase stamps, 8 per CTA of sr_pick then 8 per CTA of sr_ring_voxel
#define SR_TRACE(slot) do { if (g_sr_trace && threadIdx.x == 0) g_sr_trace[(TRACE_BASE + blockIdx.x) * 8 + (slot)] = clock64(); } while (0)
#define TRACE_BASE 0
// ---- sector walk on per-lane sorted lists ------------------------------------------------------------
// The greedy walks only ever need "the largest (smallest) curvature among the points not yet vetoed", at
// most 20 + 4 times per sector.  A sector of up to 32 * SR_REG_SLOTS points is dealt out to one warp
// (element e lives in lane e % 32, slot e / 32).  Every lane sorts its <= 16 (curvature bits, slot) keys
// once in registers (bitonic network, compile-time indices) and parks the sorted list in shared memory
// together with the inverse permutation; `live` is a bit mask over SORTED positions.  A pick is then: the
// highest (lowest) live position of each lane (one clz / ffs and one shared-memory read), the largest
// curvature over the warp and the largest element holding it (two hardware warp reductions: the
// (curvature, index) order of SURVEY Appendix B), and the +-5 marks as bit clears in the owning lanes
// (the marked window is <= 11 elements, so each lane owns at most one).  No global sort, no candidate
// list: ~3 us per sector instead of an 18 us bitonic sort of all six sectors followed by a 10 us walk.
#define SR_REG_SLOTS 16
struct SrLaneLists {                       // per warp
  unsigned bits[SR_REG_SLOTS][32];         // [sorted position][lane]: curvature bits, ascending
  unsigned char slot[SR_REG_SLOTS][32];    // [sorted position][lane]: element slot held there
  unsigned char pos[SR_REG_SLOTS][32];     // [slot][lane]: sorted position of that slot
};

__device__ __forceinline__ unsigned sr_walk_sector_reg(int j, int r, int start, int end, int rs, const float* __restrict__ curv,
                                                       const unsigned char* gb, SrLaneLists& L, int* __restrict__ label, int* __restrict__ provSharp,
                                                       int* __restrict__ provLess, int* __restrict__ provFlat, int* __restrict__ cntSharp,
                                                       int* __restrict__ cntLess, int* __restrict__ cntFlat, int lane, unsigned pre) {
  const int spj = sr_sp(start, end, j), epj = sr_ep(start, end, j);
  const int m = epj - spj + 1;
  const int slot = r * VL_SECTORS + j;
  // per-lane ascending sort of (curvature bits, slot); absent elements sort to the top and stay dead
  unsigned long long key[SR_REG_SLOTS];
#pragma unroll
  for (int q = 0; q < SR_REG_SLOTS; ++q) {
    const int e = q * 32 + lane;
    key[q] = e < m ? (((unsigned long long)__float_as_uint(curv[spj + e]) << 32) | (unsigned)q) : (0xffffffff00000000ull | (unsigned)q);
  }
#pragma unroll
  for (int k = 2; k <= SR_REG_SLOTS; k <<= 1) {
#pragma unroll
    for (int jj = k >> 1; jj > 0; jj >>= 1) {
#pragma unroll
      for (int i = 0; i < SR_REG_SLOTS; ++i) {
        const int l = i ^ jj;
        if (l > i) {
          const bool up = (i & k) == 0;
          const unsigned long long a = key[i], b = key[l];
          const bool sw = (a > b) == up;
          key[i] = sw ? b : a; key[l] = sw ? a : b;
        }
      }
    }
  }
  unsigned live = 0, big = 0, small = 0;  // over sorted positions
#pragma unroll
  for (int p = 0; p < SR_REG_SLOTS; ++p) {
    const unsigned bits = (unsigned)(key[p] >> 32);
    const int q = (int)(key[p] & 0xffu);
    L.bits[p][lane] = bits; L.slot[p][lane] = (unsigned char)q; L.pos[q][lane] = (unsigned char)p;
    if (q * 32 + lane < m) {
      live |= 1u << p;
      const float cv = __uint_as_float(bits);
      if ((double)cv > 0.1) big |= 1u << p;    // SR.cpp:375
      if ((double)cv < 0.1) small |= 1u << p;  // SR.cpp:443
    }
  }
  __syncwarp();
  SR_TRACE(6);
  if (lane < 5 && ((pre >> lane) & 1u)) live &= ~(1u << L.pos[0][lane]);  // incoming marks sit on elements 0..4 = slot 0 of lanes 0..4
  unsigned spill = 0;
  // mark element e and its +-5 neighbours until a gap > 0.05 (SR.cpp:403-429).  The marked window
  // [e - nb, e + nf] is at most 11 elements long, so every lane owns at most one element of it.
  auto mark = [&](int e) {
    const int loc = spj - rs + e;
    bool brk = false;
    if (lane < 5) brk = gb[loc + lane + 1] != 0;
    else if (lane < 10) brk = gb[loc - (lane - 4) + 1] != 0;
    const unsigned bb = __ballot_sync(0xffffffffu, brk);
    const unsigned f = bb & 31u, w = (bb >> 5) & 31u;
    const int nf = f ? __ffs(f) - 1 : 5, nb = w ? __ffs(w) - 1 : 5;
    const int first = e - nb;
    const int d = (lane - first) & 31;  // offset of this lane's element inside the window, if it has one
    const int pe = first + d;
    if (d <= nb + nf && pe >= 0 && pe < m) live &= ~(1u << L.pos[pe >> 5][lane]);
    const int over = e + nf - (m - 1);  // forward marks beyond the sector: elements m .. e + nf
    if (over > 0) spill |= (1u << over) - 1u;
  };
  // ---- descending walk: sharp (<=2) then less sharp (<=20 total), SR.cpp:371-431
  int cnt = 0;
  while (cnt < 20) {
    const unsigned cand = live & big;
    unsigned lb = 0u, le = 0u;
    if (cand) {
      const int p = 31 - __clz(cand);  // ascending lists: the highest live position is this lane's largest (curvature, element)
      lb = L.bits[p][lane];
      le = (unsigned)(L.slot[p][lane] * 32 + lane + 1);
    }
    const unsigned gmax = __reduce_max_sync(0xffffffffu, lb);
    if (gmax == 0u) break;  // curvature > 0.1 has non-zero bits
    const int e = (int)__reduce_max_sync(0xffffffffu, (lb == gmax) ? le : 0u) - 1;
    const int pind = spj + e;
    cnt++;
    if (lane == 0) {
      if (cnt <= 2) { label[pind] = 2; provSharp[slot * 2 + cnt - 1] = pind; }
      else label[pind] = 1;
      provLess[slot * 20 + cnt - 1] = pind;
    }
    mark(e);
  }
  if (lane == 0) { cntSharp[slot] = min(cnt, 2); cntLess[slot] = cnt; }
  SR_TRACE(7);
  // ---- ascending walk: flat (<=4; the 4th is not marked), SR.cpp:439-483
  cnt = 0;
  while (cnt < 4) {
    const unsigned cand = live & small;
    unsigned lb = 0xffffffffu, le = 0xffffffffu;
    if (cand) {
      const int p = __ffs(cand) - 1;  // the lowest live position: smallest (curvature, element)
      lb = L.bits[p][lane];
      le = (unsigned)(L.slot[p][lane] * 32 + lane);
    }
    const unsigned gmin = __reduce_min_sync(0xffffffffu, lb);
    if (gmin == 0xffffffffu) break;
    const int e = (int)__reduce_min_sync(0xffffffffu, (lb == gmin) ? le : 0xffffffffu);
    const int pind = spj + e;
    cnt++;
    if (lane == 0) { label[pind] = -1; provFlat[slot * 4 + cnt - 1] = pind; }
    if (cnt >= 4) break;
    mark(e);
  }
  if (lane == 0) cntFlat[slot] = cnt;
  __syncwarp();
  return spill;
}


// One CTA per ring.  All six sectors are sorted together (batched bitonic on
// (curvature bits, index) keys -- the canonical tie order of SURVEY Appendix B), then
// warp 0 walks the sectors in order because +-5 marks spill into the next sector.
__global__ void __launch_bounds__(SR_PICK_THREADS) sr_pick(const float4* __restrict__ cloud, const float* __restrict__ curv,
                                                    int* __restrict__ label, unsigned char* __restrict__ pickedG,
                                                    unsigned char* __restrict__ gapG, unsigned long long* __restrict__ scratch, const int* __restrict__ ringStart,
                                                    const int* __restrict__ ringCount, int* __restrict__ provSharp,
                                                    int* __restrict__ provLess, int* __restrict__ provFlat, int* __restrict__ cntSharp,
                                                    int* __restrict__ cntLess, int* __restrict__ cntFlat) {
  VL_PDL_WAIT();

  extern __shared__ unsigned long long smem[];
  SR_TRACE(0);
  const int r = blockIdx.x;
  const int rs = ringStart[r], rc = ringCount[r];
  const int start = rs + 5, end = rs + rc - 6;  // scanStartInd / scanEndInd (SR.cpp:310-314)
  if (threadIdx.x < VL_SECTORS) { cntSharp[r * VL_SECTORS + threadIdx.x] = 0; cntLess[r * VL_SECTORS + threadIdx.x] = 0; cntFlat[r * VL_SECTORS + threadIdx.x] = 0; }
  if (end - start < 6) return;  // SR.cpp:355-356
  int maxLen = 0, minLen0 = INT_MAX;
#pragma unroll
  for (int j = 0; j < VL_SECTORS; ++j) {
    const int len = sr_ep(start, end, j) - sr_sp(start, end, j) + 1;
    maxLen = max(maxLen, len); minLen0 = min(minLen0, len);
  }
  if (maxLen <= 32 * SR_REG_SLOTS && minLen0 >= 6 && rc <= SR_RING_CAP) {
    // ---- register path (every sensor of the reference: <= 512 points per sector) ----
    unsigned char* gbs = reinterpret_cast<unsigned char*>(smem);
    for (int t = threadIdx.x; t < rc; t += blockDim.x)
      gbs[t] = (t > 0 && (double)sr_gap2(cloud, rs + t, rs + t - 1) > 0.05) ? 1 : 0;  // SR.cpp:408-411
    __syncthreads();
    SR_TRACE(1); SR_TRACE(2);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    __shared__ unsigned spillReg[VL_SECTORS];
    __shared__ SrLaneLists lists[VL_SECTORS];
    // Six warps, six sectors.  Round 0: every sector is walked blind to its predecessor's marks.  A pre-marked
    // point changes a walk only if that walk had picked it (a mark does nothing but veto a pick), so in the
    // following rounds sector j keeps its result while (a) every mark it was walked with is still in its
    // predecessor's spill and (b) no NEW spill mark sits on one of its picks; otherwise it is walked again with
    // the current spill.  Sector j is final after round j at the latest (sector 0 never changes); nearly always
    // one round with one or two re-walks, all of them in parallel.
    unsigned used = 0u;  // marks this warp's sector was last walked with
    if (warp < VL_SECTORS) {
      const unsigned so = sr_walk_sector_reg(warp, r, start, end, rs, curv, gbs, lists[warp], label, provSharp, provLess, provFlat, cntSharp, cntLess, cntFlat, lane, 0u);
      if (lane == 0) spillReg[warp] = so;
    }
    SR_TRACE(3);
    for (int round = 1; round < VL_SECTORS; ++round) {
      __syncthreads();
      if (round == 1) SR_TRACE(4);
      bool need = false;
      unsigned in = 0u;
      int pind = -1;
      if (warp >= 1 && warp < VL_SECTORS) {
        in = spillReg[warp - 1];
        const int spj = sr_sp(start, end, warp);
        const int slot = r * VL_SECTORS + warp;
        const int nl = cntLess[slot], nfl = cntFlat[slot];
        if (lane < nl) pind = provLess[slot * 20 + lane];
        else if (lane >= 20 && lane - 20 < nfl) pind = provFlat[slot * 4 + lane - 20];
        const unsigned fresh = in & ~used;
        const bool hit = pind >= 0 && pind - spj < 5 && ((fresh >> (pind - spj)) & 1u);
        need = (used & ~in) != 0u || __ballot_sync(0xffffffffu, hit) != 0u;
      }
      if (!__syncthreads_or(need ? 1 : 0)) break;  // (also orders the reads of spillReg above before the writes below)
      if (need) {
        if (pind >= 0) label[pind] = 0;  // undo this sector's previous walk
        __syncwarp();
        const unsigned so = sr_walk_sector_reg(warp, r, start, end, rs, curv, gbs, lists[warp], label, provSharp, provLess, provFlat, cntSharp, cntLess, cntFlat, lane, in);
        used = in;
        if (lane == 0) spillReg[warp] = so;
      }
    }
    SR_TRACE(5);
    return;
  }
  int P = 32; while (P < maxLen) P <<= 1;
  const bool inSmem = P <= SR_SECT_CAP;
  // sector j keys live at keys + j*P; the global fallback uses 2*count entries per ring (6P <= 12*len/6*... bounded by 2*rc+384)
  unsigned long long* keys = inSmem ? smem : scratch + (size_t)2 * rs + (size_t)r * 6 * 64;
  unsigned char* pk = (rc <= SR_RING_CAP) ? reinterpret_cast<unsigned char*>(smem + VL_SECTORS * SR_SECT_CAP) : pickedG + rs;
  unsigned char* gb = (rc <= SR_RING_CAP) ? pk + SR_RING_CAP : gapG + rs;
  for (int t = threadIdx.x; t < rc; t += blockDim.x) {
    pk[t] = 0;
    gb[t] = (t > 0 && (double)sr_gap2(cloud, rs + t, rs + t - 1) > 0.05) ? 1 : 0;  // SR.cpp:408-411
  }
  for (int t = threadIdx.x; t < VL_SECTORS * P; t += blockDim.x) {
    const int j = t / P, k = t - j * P;
    const int idx = sr_sp(start, end, j) + k;
    const int last = sr_ep(start, end, j);
    keys[t] = (idx <= last) ? (((unsigned long long)__float_as_uint(curv[idx]) << 32) | (unsigned)idx) : ~0ull;
  }
  __syncthreads();
  SR_TRACE(1);
  bt_sort_batched<SR_PICK_THREADS>(keys, P, VL_SECTORS);
  SR_TRACE(2);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int minLen = INT_MAX;
#pragma unroll
  for (int j = 0; j < VL_SECTORS; ++j) minLen = min(minLen, sr_ep(start, end, j) - sr_sp(start, end, j) + 1);
  if (minLen < 6) {  // tiny ring: marks may cross more than one sector boundary -- walk the sectors in order
    if (warp != 0) return;
    for (int j = 0; j < VL_SECTORS; ++j)
      sr_walk_sector(j, r, start, end, rs, keys + j * P, gb, pk, label, provSharp, provLess, provFlat, cntSharp, cntLess, cntFlat, lane, 0u, 0, INT_MAX);
    return;
  }
  // The sectors only interact through the <= 5 marks a pick near the end of sector j leaves on the first
  // points of sector j+1 (SR.cpp:403-417).  Six warps walk the six sectors at once, each confined to its
  // own range and reporting that spill as a bit mask; a pre-marked point changes a sector's walk only if
  // the walk had picked that very point (a mark does nothing but veto a pick), so afterwards warp 0 checks
  // the sectors in order and re-walks the few whose picks collide with the final spill of their predecessor.
  __shared__ unsigned spillOut[VL_SECTORS];
  if (warp < VL_SECTORS) {
    const int j = warp;
    const unsigned so = sr_walk_sector(j, r, start, end, rs, keys + j * P, gb, pk, label, provSharp, provLess, provFlat, cntSharp, cntLess, cntFlat, lane, 0u,
                                       sr_sp(start, end, j) - rs, sr_ep(start, end, j) - rs);
    if (lane == 0) spillOut[j] = so;
  }
  SR_TRACE(3);
  __syncthreads();
  SR_TRACE(4);
  if (warp != 0) return;
  for (int j = 1; j < VL_SECTORS; ++j) {
    const unsigned in = spillOut[j - 1];
    if (in == 0) continue;
    const int spj = sr_sp(start, end, j), epj = sr_ep(start, end, j);
    const int slot = r * VL_SECTORS + j;
    const int nl = cntLess[slot], nfl = cntFlat[slot];
    int pind = -1;
    if (lane < nl) pind = provLess[slot * 20 + lane];
    else if (lane >= 20 && lane - 20 < nfl) pind = provFlat[slot * 4 + lane - 20];
    const bool hit = pind >= 0 && pind - spj < 5 && ((in >> (pind - spj)) & 1u);
    if (__ballot_sync(0xffffffffu, hit) == 0) continue;  // the spill vetoes nothing this sector picked
    if (pind >= 0) label[pind] = 0;                       // undo the speculative walk of sector j ...
    for (int t = spj - rs + lane; t <= epj - rs; t += 32) pk[t] = 0;
    __syncwarp();
    const unsigned so = sr_walk_sector(j, r, start, end, rs, keys + j * P, gb, pk, label, provSharp, provLess, provFlat, cntSharp, cntLess, cntFlat, lane, in,
                                       spj - rs, epj - rs);  // ... and repeat it with the incoming marks in place
    if (lane == 0) spillOut[j] = so;
    __syncwarp();
  }
  SR_TRACE(5);
}
#undef TRACE_BASE

// ---- per-ring pcl::VoxelGrid(0.2) of the label<=0 points (SR.cpp:486-503) -------------
struct VoxBox { int minb[3], mul1, mul2, guard; float inv; };

__device__ __forceinline__ unsigned vox_idx(const float4 p, const VoxBox& b) {
  const int i0 = (int)__fsub_rn(floorf(__fmul_rn(p.x, b.inv)), (float)b.minb[0]);
  const int i1 = (int)__fsub_rn(floorf(__fmul_rn(p.y, b.inv)), (float)b.minb[1]);
  const int i2 = (int)__fsub_rn(floorf(__fmul_rn(p.z, b.inv)), (float)b.minb[2]);
  return (unsigned)(i0 + i1 * b.mul1 + i2 * b.mul2);
}

__device__ __forceinline__ void vox_make_box(const float mn[3], const float mx[3], float leaf, VoxBox* b) {
  const float inv = __fdiv_rn(1.0f, leaf);
  b->inv = inv;
  const long long dx = (long long)__fmul_rn(__fsub_rn(mx[0], mn[0]), inv) + 1;
  const long long dy = (long long)__fmul_rn(__fsub_rn(mx[1], mn[1]), inv) + 1;
  const long long dz = (long long)__fmul_rn(__fsub_rn(mx[2], mn[2]), inv) + 1;
  b->guard = (dx * dy * dz > (long long)INT_MAX) ? 1 : 0;
  int maxb[3];
  for (int a = 0; a < 3; ++a) {
    b->minb[a] = (int)floorf(__fmul_rn(mn[a], inv));
    maxb[a] = (int)floorf(__fmul_rn(mx[a], inv));
  }
  const int d0 = maxb[0] - b->minb[0] + 1, d1 = maxb[1] - b->minb[1] + 1;
  b->mul1 = d0; b->mul2 = d0 * d1;
}

__global__ void __launch_bounds__(SR_PICK_THREADS) sr_ring_voxel(const float4* __restrict__ cloud, const int* __restrict__ label,
                                                          const int* __restrict__ ringStart, const int* __restrict__ ringCount,
                                                          int* __restrict__ sel, unsigned long long* __restrict__ scratch,
                                                          float4* __restrict__ outProv, int* __restrict__ dsCount, float leaf) {
  VL_PDL_WAIT();

#define TRACE_BASE 128
  SR_TRACE(0);
  extern __shared__ unsigned long long vsm[];  // [SR_VOX_CAP] keys, then [SR_VOX_CAP] float4 points
  unsigned long long* skeys = vsm;
  float4* spts = reinterpret_cast<float4*>(vsm + SR_VOX_CAP);
  __shared__ int warpSum[SR_PICK_THREADS / 32];
  __shared__ float red[6][SR_PICK_THREADS / 32];
  __shared__ VoxBox box;
  const int r = blockIdx.x;
  const int rs = ringStart[r], rc = ringCount[r];
  const int start = rs + 5, end = rs + rc - 6;
  if (end - start < 6) { if (threadIdx.x == 0) dsCount[r] = 0; return; }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int* mySel = sel + rs;
  // 1. ordered selection + bounding box
  float mn[3] = {CUDART_INF_F, CUDART_INF_F, CUDART_INF_F}, mx[3] = {-CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F};
  int total = 0;
  for (int base = start; base < end; base += SR_PICK_THREADS) {
    const int k = base + threadIdx.x;
    const bool f = k < end && label[k] <= 0;
    const unsigned b = __ballot_sync(0xffffffffu, f);
    if (lane == 0) warpSum[warp] = __popc(b);
    __syncthreads();
    int before = 0, all = 0;
    for (int w = 0; w < SR_PICK_THREADS / 32; ++w) { const int v = warpSum[w]; if (w < warp) before += v; all += v; }
    if (f) {
      mySel[total + before + __popc(b & ((1u << lane) - 1u))] = k;
      const float4 p = cloud[k];
      mn[0] = fminf(mn[0], p.x); mx[0] = fmaxf(mx[0], p.x);
      mn[1] = fminf(mn[1], p.y); mx[1] = fmaxf(mx[1], p.y);
      mn[2] = fminf(mn[2], p.z); mx[2] = fmaxf(mx[2], p.z);
    }
    total += all;
    __syncthreads();
  }
  const int m = total;
  if (m == 0) { if (threadIdx.x == 0) dsCount[r] = 0; return; }
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    float lo = mn[a], hi = mx[a];
    for (int d = 16; d > 0; d >>= 1) { lo = fminf(lo, __shfl_xor_sync(0xffffffffu, lo, d)); hi = fmaxf(hi, __shfl_xor_sync(0xffffffffu, hi, d)); }
    if (lane == 0) { red[a][warp] = lo; red[3 + a][warp] = hi; }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    float lo[3], hi[3];
    for (int a = 0; a < 3; ++a) {
      lo[a] = red[a][0]; hi[a] = red[3 + a][0];
      for (int w = 1; w < SR_PICK_THREADS / 32; ++w) { lo[a] = fminf(lo[a], red[a][w]); hi[a] = fmaxf(hi[a], red[3 + a][w]); }
    }
    vox_make_box(lo, hi, leaf, &box);
  }
  __syncthreads();
  float4* out = outProv + rs;
  if (box.guard) {  // leaf too small for the extent: pcl returns the input unchanged
    for (int t = threadIdx.x; t < m; t += SR_PICK_THREADS) out[t] = cloud[mySel[t]];
    if (threadIdx.x == 0) dsCount[r] = m;
    return;
  }
  SR_TRACE(1);
  // 2. (voxel idx, local index) keys, bitonic sort
  int P = 32; while (P < m) P <<= 1;
  unsigned long long* keys = (P <= SR_VOX_CAP) ? skeys : scratch + (size_t)2 * rs + (size_t)r * 6 * 64;
  const bool ptsInSmem = m <= SR_VOX_CAP;
  for (int t = threadIdx.x; t < P; t += SR_PICK_THREADS) {
    unsigned long long key = ~0ull;
    if (t < m) {
      const float4 p = cloud[mySel[t]];
      if (ptsInSmem) spts[t] = p;
      key = ((unsigned long long)vox_idx(p, box) << 32) | (unsigned)t;
    }
    keys[t] = key;
  }
  __syncthreads();
  SR_TRACE(2);
  if (P <= SR_VOX_CAP) bt_smem_sort<SR_PICK_THREADS>(skeys, P);  // (P >= 32) the usual case: LDS / STS, register rounds
  else bt_sort_batched<SR_PICK_THREADS>(keys, P, 1);
  SR_TRACE(3);
  // 3. run heads -> ordered output slots; the head thread folds its run in f32, in index order
  total = 0;
  for (int base = 0; base < m; base += SR_PICK_THREADS) {
    const int t = base + threadIdx.x;
    const bool head = t < m && (t == 0 || (unsigned)(keys[t] >> 32) != (unsigned)(keys[t - 1] >> 32));
    const unsigned b = __ballot_sync(0xffffffffu, head);
    if (lane == 0) warpSum[warp] = __popc(b);
    __syncthreads();
    int before = 0, all = 0;
    for (int w = 0; w < SR_PICK_THREADS / 32; ++w) { const int v = warpSum[w]; if (w < warp) before += v; all += v; }
    if (head) {
      const unsigned vox = (unsigned)(keys[t] >> 32);
      float sx = 0.f, sy = 0.f, sz = 0.f, si = 0.f; int nrun = 0;
      for (int q = t; q < m && (unsigned)(keys[q] >> 32) == vox; ++q) {
        const int li = (int)(unsigned)(keys[q] & 0xffffffffull);
        const float4 p = ptsInSmem ? spts[li] : cloud[mySel[li]];
        sx = __fadd_rn(sx, p.x); sy = __fadd_rn(sy, p.y); sz = __fadd_rn(sz, p.z); si = __fadd_rn(si, p.w);
        ++nrun;
      }
      const float fn = (float)nrun;
      out[total + before + __popc(b & ((1u << lane) - 1u))] =
          make_float4(__fdiv_rn(sx, fn), __fdiv_rn(sy, fn), __fdiv_rn(sz, fn), __fdiv_rn(si, fn));
    }
    total += all;
    __syncthreads();
  }
  if (threadIdx.x == 0) dsCount[r] = total;
  SR_TRACE(4);
#undef TRACE_BASE
}

// Exclusive scans of the pick counts (ring-major, sector, pick order = the reference's
// push_back order) and of the per-ring DS counts.
// phase 1: the three pick-based clouds (all the odometry of this sweep needs: it may start before the per-ring voxel filter
// has run); phase 2: the per-ring downsampled less-flat cloud.
__global__ void __launch_bounds__(1024) sr_offsets(int nscans, int phase, const int* __restrict__ cntSharp, const int* __restrict__ cntLess,
                                                   const int* __restrict__ cntFlat, const int* __restrict__ dsCount,
                                                   int* __restrict__ offSharp, int* __restrict__ offLess, int* __restrict__ offFlat,
                                                   int* __restrict__ dsOff, SrScalars* __restrict__ s) {
  VL_PDL_WAIT();

  __shared__ int ws[32];
  const int t = threadIdx.x;
  const int nslots = nscans * VL_SECTORS;
  if (phase == 1) {
    const int own[3] = {t < nslots ? cntSharp[t] : 0, t < nslots ? cntLess[t] : 0, t < nslots ? cntFlat[t] : 0};
    int ex[3], tot[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) ex[a] = vl_block_excl_scan<1024>(own[a], ws, &tot[a]);
    if (t < nslots) { offSharp[t] = ex[0]; offLess[t] = ex[1]; offFlat[t] = ex[2]; }
    if (t == 0) { s->nSharp = tot[0]; s->nLessSharp = tot[1]; s->nFlat = tot[2]; s->nQueries = tot[0] + tot[2]; }
  } else {
    int tot = 0;
    const int ex = vl_block_excl_scan<1024>(t < nscans ? dsCount[t] : 0, ws, &tot);
    if (t < nscans) dsOff[t] = ex;
    if (t == 0) s->nLessFlat = tot;
  }
}

__global__ void __launch_bounds__(SR_BLOCK) sr_gather(const float4* __restrict__ cloud, int nscans, int phase, const SrScalars* __restrict__ s,
                                                      const int* __restrict__ provSharp, const int* __restrict__ provLess,
                                                      const int* __restrict__ provFlat, const int* __restrict__ cntSharp,
                                                      const int* __restrict__ cntLess, const int* __restrict__ cntFlat,
                                                      const int* __restrict__ offSharp, const int* __restrict__ offLess,
                                                      const int* __restrict__ offFlat, const int* __restrict__ ringStart,
                                                      const int* __restrict__ dsCount, const int* __restrict__ dsOff,
                                                      const float4* __restrict__ lessFlatProv, float4* __restrict__ sharp,
                                                      float4* __restrict__ lessSharp, float4* __restrict__ flat, float4* __restrict__ lessFlat) {
  VL_PDL_WAIT();

  int t = blockIdx.x * blockDim.x + threadIdx.x;
  const int nslots = nscans * VL_SECTORS;
  if (phase == 1) {
    if (t < nslots * 2) { const int sl = t / 2, k = t - sl * 2; if (k < cntSharp[sl]) sharp[offSharp[sl] + k] = cloud[provSharp[t]]; return; }
    t -= nslots * 2;
    if (t < nslots * 20) { const int sl = t / 20, k = t - sl * 20; if (k < cntLess[sl]) lessSharp[offLess[sl] + k] = cloud[provLess[t]]; return; }
    t -= nslots * 20;
    if (t < nslots * 4) { const int sl = t / 4, k = t - sl * 4; if (k < cntFlat[sl]) flat[offFlat[sl] + k] = cloud[provFlat[t]]; }
    return;
  }
  if (t >= s->count) return;
  int lo = 0, hi = nscans;  // ring of position t: largest r with ringStart[r] <= t
  while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (ringStart[mid] <= t) lo = mid; else hi = mid; }
  const int k = t - ringStart[lo];
  if (k < dsCount[lo]) lessFlat[dsOff[lo] + k] = lessFlatProv[t];
}

// vloam_b200_exact_math: the DEVICE compile of exact_math.h on caller-supplied inputs (tests compare it with glibc bit for bit)
__global__ void __launch_bounds__(256) sr_exact_math(const float* __restrict__ y, const float* __restrict__ x, int n, float* __restrict__ oAtan,
                                                     float* __restrict__ oAtan2) {
  VL_PDL_WAIT();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  oAtan[i] = vlx::atanf_exact(x[i]);
  oAtan2[i] = vlx::atan2f_exact(y[i], x[i]);
}
int vl_sr_exact_math(vloam_b200_ctx* c, const float* d_y, const float* d_x, int n, float* d_atan, float* d_atan2) {
  VL_LAUNCH(sr_exact_math, vl_div_up(n, 256), 256, 0, d_y, d_x, n, d_atan, d_atan2);
  VL_CUDA(cudaGetLastError());
  return VLOAM_OK;
}

// ---------------------------------------------------------------------------------
int vl_sr_run(vloam_b200_ctx* c, const float* d_xyz, int n, int stride) {
  const int R = c->prm.n_scans;
  c->sr_counts_valid = false;
  c->n_in = n; c->stride = stride;
  c->cur = (c->cur + 1) % 3;  // this sweep's lessSharp / lessFlat: neither the "last" clouds' buffer nor the sweep before that
  if (n <= 0) {
    VL_CUDA(cudaMemsetAsync(c->srs, 0, sizeof(SrScalars), VL_STREAM(c)));
    VL_CUDA(cudaMemsetAsync(c->ringCount, 0, sizeof(int) * VL_MAX_RINGS, VL_STREAM(c)));
    VL_CUDA(cudaMemsetAsync(c->ringStart, 0, sizeof(int) * (VL_MAX_RINGS + 1), VL_STREAM(c)));
    VL_CUDA(cudaEventRecord(c->evSRfeat, VL_STREAM(c)));
    VL_CUDA(cudaEventRecord(c->evSR, VL_STREAM(c)));
    return VLOAM_OK;
  }
  // (a previous run of this set may have left its tail on the side stream: it reads buffers this run rewrites)
  if (vl_tls_stream == nullptr) VL_CUDA(cudaStreamWaitEvent(c->stream, c->evSR, 0));
  const int numBlocks = vl_div_up(n, SR_BLOCK);
  VL_TRY(vl_reserve(c, c->ring, n));
  VL_TRY(vl_reserve(c, c->ori, n));
  VL_TRY(vl_reserve(c, c->blockHist, (size_t)R * numBlocks));
  VL_TRY(vl_reserve(c, c->cloud, n));
  VL_TRY(vl_reserve(c, c->curv, n));
  VL_TRY(vl_reserve(c, c->label, n));
  VL_TRY(vl_reserve(c, c->picked, (size_t)2 * n));
  VL_TRY(vl_reserve(c, c->sortScratch, (size_t)2 * n + (size_t)VL_MAX_RINGS * 6 * 64 + 64));
  VL_TRY(vl_reserve(c, c->lessFlatProv, n));
  VL_TRY(vl_reserve(c, c->selIdx, n));
  VL_TRY(vl_reserve(c, c->sharp, (size_t)R * VL_SECTORS * 2));
  VL_TRY(vl_reserve(c, c->flat, (size_t)R * VL_SECTORS * 4));
  VL_TRY(vl_reserve(c, c->lessSharp[c->cur], (size_t)R * VL_SECTORS * 20));
  VL_TRY(vl_reserve(c, c->lessFlat[c->cur], n));
  const int vec4 = (stride == 4 && (reinterpret_cast<uintptr_t>(d_xyz) & 15) == 0) ? 1 : 0;
  const float thres = c->prm.minimum_range;
  const float thres2 = thres * thres;

  VL_LAUNCH(sr_find_bounds, 1, 1024, 0, d_xyz, n, stride, vec4, thres2, c->srs);
  VL_BYTES((4.0 * stride + 8.0) * n);
  VL_LAUNCH(sr_classify, numBlocks, SR_BLOCK, 0, d_xyz, n, stride, vec4, thres2, R, c->srs, c->ring.p, c->ori.p, c->blockHist.p, numBlocks);
  VL_LAUNCH(sr_ring_scan, vl_div_up(R, 8), 256, 0, c->blockHist.p, numBlocks, R, c->ringCount, c->ringStart, c->srs);
  VL_BYTES((4.0 * stride + 8.0 + 16.0) * n);
  VL_LAUNCH(sr_scatter, numBlocks, SR_BLOCK, 0, d_xyz, n, stride, vec4, R, c->srs, c->ring.p, c->ori.p, c->blockHist.p, numBlocks,
            c->ringStart, c->cloud.p);
  VL_BYTES(25.0 * n);
  VL_LAUNCH(sr_curvature, numBlocks, SR_BLOCK, 0, c->cloud.p, c->srs, c->curv.p, c->label.p, c->picked.p);
  const size_t pickSmem = (size_t)VL_SECTORS * SR_SECT_CAP * sizeof(unsigned long long) + 2 * SR_RING_CAP;
  VL_BYTES(40.0 * n);  // 2 points + curvature per ring point in, labels + picks out (upper bound: n kept)
  VL_LAUNCH(sr_pick, R, SR_PICK_THREADS, pickSmem, c->cloud.p, c->curv.p, c->label.p, c->picked.p, c->picked.p + n, c->sortScratch.p, c->ringStart, c->ringCount,
            c->provSharp, c->provLess, c->provFlat, c->cntSharp, c->cntLess, c->cntFlat);
  // sharp / less-sharp / flat are complete here: the odometry of this sweep waits on evSRfeat, not on the per-ring voxel filter below
  VL_LAUNCH(sr_offsets, 1, 1024, 0, R, 1, c->cntSharp, c->cntLess, c->cntFlat, c->ringDsCount, c->offSharp, c->offLess, c->offFlat,
            c->ringDsOff, c->srs);
  VL_LAUNCH(sr_gather, vl_div_up(R * VL_SECTORS * 26, SR_BLOCK), SR_BLOCK, 0, c->cloud.p, R, 1, c->srs, c->provSharp, c->provLess, c->provFlat,
            c->cntSharp, c->cntLess, c->cntFlat, c->offSharp, c->offLess, c->offFlat, c->ringStart, c->ringDsCount, c->ringDsOff,
            c->lessFlatProv.p, c->sharp.p, c->lessSharp[c->cur].p, c->flat.p, c->lessFlat[c->cur].p);
  VL_CUDA(cudaEventRecord(c->evSRfeat, VL_STREAM(c)));
  if (c->timing && VL_STREAM(c) == c->streamSR) cudaEventRecord(c->evx[8], c->streamSR);
  // One sweep at a time (this run is on the pose chain's stream): the odometry that follows needs nothing of what comes below --
  // the per-ring voxel filter of the less-flat cloud, ~40 us -- so that tail goes to the side stream behind evSRfeat and the
  // odometry starts at once.  Everything that reads the less-flat cloud or the counts waits for evSR anyway (sync point S1, the
  // stack filters and search structures issued behind it, the getters).
  const bool tailAside = vl_tls_stream == nullptr && !c->prof_name[0] && !vl_debug_capture(c);
  struct TlsRestore { cudaStream_t prev; bool on; ~TlsRestore() { if (on) vl_tls_stream = prev; } } tlsRestore{vl_tls_stream, tailAside};
  if (tailAside) { VL_CUDA(cudaStreamWaitEvent(c->streamSR, c->evSRfeat, 0)); vl_tls_stream = c->streamSR; }
  const size_t voxSmem = (size_t)SR_VOX_CAP * (sizeof(unsigned long long) + sizeof(float4));
  VL_BYTES(36.0 * n);
  VL_LAUNCH(sr_ring_voxel, R, SR_PICK_THREADS, voxSmem, c->cloud.p, c->label.p, c->ringStart, c->ringCount, c->selIdx.p, c->sortScratch.p,
            c->lessFlatProv.p, c->ringDsCount, 0.2f);
  VL_LAUNCH(sr_offsets, 1, 1024, 0, R, 2, c->cntSharp, c->cntLess, c->cntFlat, c->ringDsCount, c->offSharp, c->offLess, c->offFlat,
            c->ringDsOff, c->srs);
  VL_LAUNCH(sr_gather, vl_div_up(n, SR_BLOCK), SR_BLOCK, 0, c->cloud.p, R, 2, c->srs, c->provSharp, c->provLess, c->provFlat,
            c->cntSharp, c->cntLess, c->cntFlat, c->offSharp, c->offLess, c->offFlat, c->ringStart, c->ringDsCount, c->ringDsOff,
            c->lessFlatProv.p, c->sharp.p, c->lessSharp[c->cur].p, c->flat.p, c->lessFlat[c->cur].p);
  VL_CUDA(cudaMemcpyAsync(c->h_srs, c->srs, sizeof(SrScalars), cudaMemcpyDeviceToHost, VL_STREAM(c)));
  VL_CUDA(cudaEventRecord(c->evSR, VL_STREAM(c)));
  if (c->timing && VL_STREAM(c) == c->streamSR) cudaEventRecord(c->evx[10], c->streamSR);
  VL_CUDA(cudaGetLastError());
  return VLOAM_OK;
}

// Sync point S1: the host learns the feature counts.  It waits on the event recorded right after scan
// registration, not on the stream, so odometry kernels queued behind it keep the GPU busy meanwhile.
// function attributes are per device: set when a context is created on it (vloam_b200_create)
int vl_sr_set_attrs(vloam_b200_ctx* c) {
  VL_CUDA(cudaFuncSetAttribute(sr_pick, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               (int)((size_t)VL_SECTORS * SR_SECT_CAP * sizeof(unsigned long long) + 2 * SR_RING_CAP)));
  VL_CUDA(cudaFuncSetAttribute(sr_ring_voxel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               (int)((size_t)SR_VOX_CAP * (sizeof(unsigned long long) + sizeof(float4)))));
  // lazy module loading would otherwise charge each kernel's first launch (~1 ms apiece) to the first sweeps
  cudaFuncAttributes fa_;
  VL_CUDA(cudaFuncGetAttributes(&fa_, sr_find_bounds));
  VL_CUDA(cudaFuncGetAttributes(&fa_, sr_classify));
  VL_CUDA(cudaFuncGetAttributes(&fa_, sr_ring_scan));
  VL_CUDA(cudaFuncGetAttributes(&fa_, sr_scatter));
  VL_CUDA(cudaFuncGetAttributes(&fa_, sr_curvature));
  VL_CUDA(cudaFuncGetAttributes(&fa_, sr_pick));
  VL_CUDA(cudaFuncGetAttributes(&fa_, sr_ring_voxel));
  VL_CUDA(cudaFuncGetAttributes(&fa_, sr_offsets));
  VL_CUDA(cudaFuncGetAttributes(&fa_, sr_gather));
  return VLOAM_OK;
}

// debug: the first call arms the phase trace of sr_pick / sr_ring_voxel; later calls copy it out (256 x 8 stamps)
int vl_sr_trace(vloam_b200_ctx* c, long long* out, int n) {
  static long long* d_buf = nullptr;
  const int cap = 256 * 8;
  if (!d_buf) {
    VL_CUDA(cudaMalloc(&d_buf, sizeof(long long) * cap));
    VL_CUDA(cudaMemset(d_buf, 0, sizeof(long long) * cap));
    VL_CUDA(cudaMemcpyToSymbol(g_sr_trace, &d_buf, sizeof(long long*)));
  }
  VL_CUDA(cudaStreamSynchronize(c->stream));
  VL_CUDA(cudaMemcpy(out, d_buf, sizeof(long long) * min(n, cap), cudaMemcpyDeviceToHost));
  return VLOAM_OK;
}

int vl_sr_sync_counts(vloam_b200_ctx* c) {
  if (c->sr_counts_valid) return VLOAM_OK;
  VL_CUDA(cudaEventSynchronize(c->evSR));
  if (c->n_in <= 0) { c->nKept = c->nSharp = c->nLessSharp = c->nFlat = c->nLessFlat = 0; }
  else {
    c->nKept = c->h_srs->count; c->nSharp = c->h_srs->nSharp; c->nLessSharp = c->h_srs->nLessSharp;
    c->nFlat = c->h_srs->nFlat; c->nLessFlat = c->h_srs->nLessFlat;
  }
  c->sr_counts_valid = true;
  return VLOAM_OK;
}

// laser_mapping.cu -- LaserMapping::input / solveMapping (laser_mapping.cpp:178-814) as CUDA.
//
// Map layout in HBM.  The reference keeps 2 x 4851 per-cube PCL clouds (LM.h:117-150).
// Here each cube of each kind (corner / surf) is a segment [start, start+count) of one
// big float4 pool plus a `sorted` length: the prefix whose voxel keys are strictly
// increasing (what a previous VoxelGrid pass left behind); anything after it is an
// unsorted tail (raw appends to cubes outside the 5x5x3 window).  Rolling the 21x21x11
// window (LM.cpp:252-444) permutes the 4851-entry table, it never moves points.
//
// Per frame:
//   lm_prepare        input() + centre cube + roll + valid-cube list + gather offsets
//   lm_gather         the 75 valid cubes -> contiguous cornerFromMap / surfFromMap (canonical kNN ids)
//   vl_voxel_grid     current less-sharp / less-flat -> cornerStack / surfStack (LM.cpp:492-500)
//   [sync S2: Mc, Ms, Qc, Qs, tail sizes]
//   grid build        counting sort of both sub-maps into 2 m cells over the 250x250x150 m window
//   2 x { lm_knn (5-NN), lm_fit (PCA line / QR plane -> factor slots), vl_solve }
//   lm_transform_update, then the map update:
//   rf_*              VoxelGrid re-filter of the valid cubes (LM.cpp:795-808) WITHOUT re-sorting the
//                     map: only tails + this frame's points are sorted, then merged into the
//                     already-ordered prefixes (exact: a prefix has one point per voxel and
//                     the lowest point indices, so every run is [prefix point?] + tail points)
#include <limits.h>
#include <float.h>
#include <math_constants.h>
#include <cooperative_groups.h>
#include "common.cuh"
#include "bitonic.cuh"
#include "lm_grid.cuh"
namespace cg = cooperative_groups;
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <thread>

// ---- helper thread ------------------------------------------------------------------------------------
// After sync point S2 the caller has its pose; what remains of the frame is issuing ~25 launches of the map
// update and of the next frame's speculative sub-map on stream3 -- ~100 us of host time during which neither
// the caller nor the next sweep's scan registration made progress.  One helper thread per context issues
// them instead.  It spins for a millisecond after each task (a replay hands it work every ~0.4 ms) and
// sleeps on a condition variable otherwise (a live 10 Hz feed must not burn a core).
thread_local cudaStream_t vl_tls_stream = nullptr;

struct VlWorker {
  std::thread th;
  std::mutex m;
  std::condition_variable cv;
  std::function<int()> task;
  std::atomic<int> state{0};   // 0 idle, 1 task posted, 2 running
  std::atomic<bool> sleeping{false};
  bool quit = false;
  int rc = VLOAM_OK;
  int device = 0;
};

static void lm_worker_main(VlWorker* w) {
  cudaSetDevice(w->device);
  for (;;) {
    const auto t0 = std::chrono::steady_clock::now();
    while (w->state.load(std::memory_order_acquire) != 1) {
      if (std::chrono::steady_clock::now() - t0 > std::chrono::milliseconds(1)) {
        std::unique_lock<std::mutex> lk(w->m);
        w->sleeping.store(true);
        w->cv.wait(lk, [&] { return w->state.load(std::memory_order_acquire) == 1 || w->quit; });
        w->sleeping.store(false);
        if (w->quit) return;
        break;
      }
      // busy-wait briefly, then give the core away between polls: with one process per GPU on a 16-core box the
      // helper threads of eight ranks must not starve the threads that feed them
      if (std::chrono::steady_clock::now() - t0 > std::chrono::microseconds(50)) std::this_thread::yield();
#if defined(__x86_64__)
      else __builtin_ia32_pause();
#endif
    }
    w->state.store(2, std::memory_order_relaxed);
    w->rc = w->task();
    w->state.store(0, std::memory_order_release);
  }
}

int vl_lm_join(vloam_b200_ctx* c) {
  VlWorker* w = c->worker;
  if (!w) return VLOAM_OK;
  while (w->state.load(std::memory_order_acquire) != 0) {
#if defined(__x86_64__)
    __builtin_ia32_pause();
#endif
  }
  const int rc = w->rc;
  w->rc = VLOAM_OK;
  return rc;
}

void vl_lm_shutdown(vloam_b200_ctx* c) {
  VlWorker* w = c->worker;
  if (!w) return;
  vl_lm_join(c);
  { std::lock_guard<std::mutex> lk(w->m); w->quit = true; }
  w->cv.notify_all();
  // a spinning worker notices quit only through the condition variable path: post nothing, it falls asleep within 1 ms
  w->th.join();
  delete w;
  c->worker = nullptr;
}

int vl_lm_submit_task(vloam_b200_ctx* c, int (*fn)(vloam_b200_ctx*));
static int lm_submit(vloam_b200_ctx* c, std::function<int()> f) {
  if (!c->worker) {
    VlWorker* w = new VlWorker();
    w->device = c->device;
    w->th = std::thread(lm_worker_main, w);
    c->worker = w;
  }
  VlWorker* w = c->worker;
  VL_TRY(vl_lm_join(c));
  w->task = std::move(f);
  // Publish under the worker's mutex and always notify: a worker that is between its last poll of `state` and
  // cv.wait() holds the mutex, so it either sees state == 1 in the wait predicate or receives this notification
  // (checking `sleeping` without the lock could miss both: the store and the load may be reordered on x86).
  { std::lock_guard<std::mutex> lk(w->m); w->state.store(1, std::memory_order_seq_cst); }
  w->cv.notify_one();
  return VLOAM_OK;
}

int vl_lm_submit_task(vloam_b200_ctx* c, int (*fn)(vloam_b200_ctx*)) { return lm_submit(c, [c, fn]() -> int { return fn(c); }); }

#define LM_CELL 2.0f
#define LM_GX 125
#define LM_GY 125
#define LM_GZ 75
#define LM_NCELL (LM_GX * LM_GY * LM_GZ)
#define LM_NSEG 250  // (kind, valid slot)

struct RfWork {
  int slotOfCube[VL_CUBE_NUM];          // valid slot of a cube index or -1
  int gatherOff[2][VL_MAX_VALID + 1];   // exclusive offsets of the valid cubes inside fromMap
  int tailOff[LM_NSEG + 1];             // exclusive offsets of existing-tail keys
  int prefOff[LM_NSEG + 1];             // exclusive offsets of prefix points
  int tailBegin[LM_NSEG + 1];           // per segment range in the sorted key array
  int segCount[LM_NSEG + 1];            // keys per segment (histogram of rf_keys; zeroed by lm_prepare)
  int segFill[LM_NSEG + 1];             // scatter cursors
  int outOff[LM_NSEG + 1];              // staging offsets
  int outCount[LM_NSEG];
  int firstViolation[LM_NSEG];
  int nKeysValid;
  int nq;                               // Qc + Qs when the optimisation runs, else 0
  float gridOrigin[3];
};

// Everything the sub-map gather and the search grid need to know about one valid-cube window.  Two
// copies live on the device: `real`, written by lm_prepare from this frame's pose, and `spec`, written
// right after the previous frame's map update for the window that frame used (lm_spec_prepare).
struct LmSub {
  int validNum, Mc, Ms;
  int cI, cJ, cK, cenW, cenH, cenD;     // window centre and laserCloudCen* it was built for
  int ok;                               // spec: the descriptor (and the structures built from it) is complete
  float gridOrigin[3];
  int validInd[VL_MAX_VALID];
  int gatherOff[2][VL_MAX_VALID + 1];
};

__device__ __forceinline__ int lm_cube_of(float v, int cen) {  // LM.cpp:747-756
  const double t = (double)v + 25.0;
  int c = (int)(t / 50.0) + cen;
  if (t < 0) c--;
  return c;
}

// voxel key of a map point inside cube (ci,cj,ck): 10 bits per axis, (iz, iy, ix) order ==
// ascending pcl::VoxelGrid linear index inside any bounding box of that cube's points.
__device__ __forceinline__ unsigned lm_vox_key(const float4 p, float inv, int ci, int cj, int ck, int cenW, int cenH, int cenD) {
  const int bx = (int)floorf(__fmul_rn((float)(50 * (ci - cenW) - 25), inv)) - 2;
  const int by = (int)floorf(__fmul_rn((float)(50 * (cj - cenH) - 25), inv)) - 2;
  const int bz = (int)floorf(__fmul_rn((float)(50 * (ck - cenD) - 25), inv)) - 2;
  const int ix = min(max((int)floorf(__fmul_rn(p.x, inv)) - bx, 0), 1023);
  const int iy = min(max((int)floorf(__fmul_rn(p.y, inv)) - by, 0), 1023);
  const int iz = min(max((int)floorf(__fmul_rn(p.z, inv)) - bz, 0), 1023);
  return ((unsigned)iz << 20) | ((unsigned)iy << 10) | (unsigned)ix;
}
__device__ __forceinline__ unsigned lm_vox_key_cube(const float4 p, float inv, int cube, const LmScalars* s) {
  const int ci = cube % VL_CUBE_W, cj = (cube / VL_CUBE_W) % VL_CUBE_H, ck = cube / (VL_CUBE_W * VL_CUBE_H);
  return lm_vox_key(p, inv, ci, cj, ck, s->cenW, s->cenH, s->cenD);
}

__device__ __forceinline__ float lm_leaf_inv(const vloam_b200_params& p, int kind) { return __fdiv_rn(1.0f, kind ? p.plane_res : p.line_res); }

// exclusive scan of one int per thread over the first 256 threads of the block (all threads must call)
__device__ __forceinline__ int lm_scan256(int v, int* buf, int* total) {
  // exclusive scan over threads 0..255 (block of 256 or 1024 threads; every thread must call): warp shuffles, then
  // the eight warp totals through shared memory -- two barriers instead of the eighteen of a Hillis-Steele ladder
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  int inc = t < 256 ? v : 0;
  for (int d = 1; d < 32; d <<= 1) { const int u = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += u; }
  if (t < 256 && lane == 31) buf[warp] = inc;
  __syncthreads();
  int before = 0, all = 0;
#pragma unroll
  for (int w = 0; w < 8; ++w) { const int sw = buf[w]; if (w < warp) before += sw; all += sw; }
  if (total) *total = all;
  __syncthreads();
  return t < 256 ? before + inc - v : 0;
}

// ---- LaserMapping::input (LM.cpp:178-209) + centre cube / roll / valid list (LM.cpp:228-466)
__global__ void __launch_bounds__(1024) lm_prepare(LmScalars* __restrict__ s, const LoScalars* __restrict__ lo, MapCubeTable* __restrict__ tc,
                                                   MapCubeTable* __restrict__ ts, RfWork* __restrict__ w, int skip, int resetValid,
                                                   LmSub* __restrict__ real) {
  VL_PDL_WAIT();

  __shared__ int shift[3];
  __shared__ int center[3];
  if (threadIdx.x == 0) {
    s->needSlow = 0;
    if (resetValid) s->validNum = 0;  // LaserMapping::reset (LM.cpp:132-136)
    for (int k = 0; k < 4; ++k) s->q_wodom[k] = lo->q_w[k];
    for (int k = 0; k < 3; ++k) s->t_wodom[k] = lo->t_w[k];
    double r[3];
    vl_qrot(s->q_wmap_wodom, s->t_wodom[0], s->t_wodom[1], s->t_wodom[2], r);
    if (skip) {
      vl_qmul(s->q_wmap_wodom, s->q_wodom, s->q_hf);
      for (int k = 0; k < 3; ++k) s->t_hf[k] = r[k] + s->t_wmap_wodom[k];
    } else {
      double qn[4];
      vl_qmul(s->q_wmap_wodom, s->q_wodom, qn);
      for (int k = 0; k < 4; ++k) s->pose[k] = qn[k];
      for (int k = 0; k < 3; ++k) s->pose[4 + k] = r[k] + s->t_wmap_wodom[k];
    }
    int cI = (int)((s->pose[4] + 25.0) / 50.0) + s->cenW;
    int cJ = (int)((s->pose[5] + 25.0) / 50.0) + s->cenH;
    int cK = (int)((s->pose[6] + 25.0) / 50.0) + s->cenD;
    if (s->pose[4] + 25.0 < 0) cI--;
    if (s->pose[5] + 25.0 < 0) cJ--;
    if (s->pose[6] + 25.0 < 0) cK--;
    int sI = 0, sJ = 0, sK = 0;
    if (!skip) {  // net effect of the six while loops: contents move by +s along an axis
      while (cI < 3) { cI++; sI++; }
      while (cI >= VL_CUBE_W - 3) { cI--; sI--; }
      while (cJ < 3) { cJ++; sJ++; }
      while (cJ >= VL_CUBE_H - 3) { cJ--; sJ--; }
      while (cK < 3) { cK++; sK++; }
      while (cK >= VL_CUBE_D - 3) { cK--; sK--; }
      s->cenW += sI; s->cenH += sJ; s->cenD += sK;
    }
    shift[0] = sI; shift[1] = sJ; shift[2] = sK;
    center[0] = cI; center[1] = cJ; center[2] = cK;
  }
  __syncthreads();
  if (skip) return;  // (a skipped frame neither consumes nor invalidates the speculative sub-map)
  const int sI = shift[0], sJ = shift[1], sK = shift[2];
  if (sI != 0 || sJ != 0 || sK != 0) {
    // new[i,j,k] = old[i-sI, j-sJ, k-sK]; entries whose source wrapped are the cleared slabs (they
    // keep the storage of the entry that fell off the other side).
    int v[5][8]; bool wrap[5];
    for (int q = 0; q < 5; ++q) {
      const int d = threadIdx.x + q * 1024;
      if (d >= VL_CUBE_NUM) break;
      const int i = d % VL_CUBE_W, j = (d / VL_CUBE_W) % VL_CUBE_H, k = d / (VL_CUBE_W * VL_CUBE_H);
      const int si = i - sI, sj = j - sJ, sk = k - sK;
      wrap[q] = si < 0 || si >= VL_CUBE_W || sj < 0 || sj >= VL_CUBE_H || sk < 0 || sk >= VL_CUBE_D;
      // saturating modulo: multi-cube jumps still give a bijection
      const int mi = ((si % VL_CUBE_W) + VL_CUBE_W) % VL_CUBE_W, mj = ((sj % VL_CUBE_H) + VL_CUBE_H) % VL_CUBE_H,
                mk = ((sk % VL_CUBE_D) + VL_CUBE_D) % VL_CUBE_D;
      const int src = mi + VL_CUBE_W * mj + VL_CUBE_W * VL_CUBE_H * mk;
      v[q][0] = tc->start[src]; v[q][1] = tc->count[src]; v[q][2] = tc->cap[src]; v[q][3] = tc->sorted[src];
      v[q][4] = ts->start[src]; v[q][5] = ts->count[src]; v[q][6] = ts->cap[src]; v[q][7] = ts->sorted[src];
    }
    __syncthreads();
    for (int q = 0; q < 5; ++q) {
      const int d = threadIdx.x + q * 1024;
      if (d >= VL_CUBE_NUM) break;
      tc->start[d] = v[q][0]; tc->count[d] = wrap[q] ? 0 : v[q][1]; tc->cap[d] = v[q][2]; tc->sorted[d] = wrap[q] ? 0 : v[q][3];
      ts->start[d] = v[q][4]; ts->count[d] = wrap[q] ? 0 : v[q][5]; ts->cap[d] = v[q][6]; ts->sorted[d] = wrap[q] ? 0 : v[q][7];
    }
  }
  __shared__ int sTot[2];
  if (threadIdx.x < 2) sTot[threadIdx.x] = 0;
  __syncthreads();
  if (threadIdx.x <= LM_NSEG) { w->segCount[threadIdx.x] = 0; w->segFill[threadIdx.x] = 0; }  // histogram / bucket cursors of this frame's update keys
  int myC = 0, myS = 0;
  for (int d = threadIdx.x; d < VL_CUBE_NUM; d += 1024) { w->slotOfCube[d] = -1; myC += tc->count[d]; myS += ts->count[d]; }
  for (int o = 16; o > 0; o >>= 1) { myC += __shfl_xor_sync(0xffffffffu, myC, o); myS += __shfl_xor_sync(0xffffffffu, myS, o); }
  if ((threadIdx.x & 31) == 0) { atomicAdd(&sTot[0], myC); atomicAdd(&sTot[1], myS); }
  __shared__ int sbuf[256];
  __shared__ int snv;
  __syncthreads();
  if (threadIdx.x == 0) { s->totalC = sTot[0]; s->totalS = sTot[1]; }
  if (threadIdx.x == 0) {
    const int cI = center[0], cJ = center[1], cK = center[2];
    int nv = s->validNum;  // LaserMapping::reset zeroes it once per frame (LM.cpp:132-136)
    for (int i = cI - 2; i <= cI + 2; i++)
      for (int j = cJ - 2; j <= cJ + 2; j++)
        for (int k = cK - 1; k <= cK + 1; k++)
          if (i >= 0 && i < VL_CUBE_W && j >= 0 && j < VL_CUBE_H && k >= 0 && k < VL_CUBE_D && nv < VL_MAX_VALID)
            s->validInd[nv++] = i + VL_CUBE_W * j + VL_CUBE_W * VL_CUBE_H * k;
    s->validNum = nv;
    snv = nv;
    w->gridOrigin[0] = (float)(50 * (cI - 2 - s->cenW) - 25);
    w->gridOrigin[1] = (float)(50 * (cJ - 2 - s->cenH) - 25);
    w->gridOrigin[2] = (float)(50 * (cK - 1 - s->cenD) - 25);
    real->validNum = nv; real->cI = cI; real->cJ = cJ; real->cK = cK; real->cenW = s->cenW; real->cenH = s->cenH; real->cenD = s->cenD;
    for (int k = 0; k < 3; ++k) real->gridOrigin[k] = w->gridOrigin[k];
  }
  __syncthreads();
  const int nv = snv;
  const int t = threadIdx.x;
  // thread t < 250 owns segment (kind, slot) = (t / 125, t % 125)
  const int kind = t / VL_MAX_VALID, slot = t % VL_MAX_VALID;
  int cnt = 0, srt = 0;
  if (t < LM_NSEG && slot < nv) {
    const int cb = s->validInd[slot];
    const MapCubeTable* tb = kind ? ts : tc;
    cnt = tb->count[cb]; srt = tb->sorted[cb];
    if (kind == 0) w->slotOfCube[cb] = slot;
  }
  int total = 0;
  const int offCnt = lm_scan256(cnt, sbuf, &total);          // corner segments first, then surf
  __shared__ int sMc;
  if (t == VL_MAX_VALID) sMc = offCnt;                        // exclusive offset of the first surf segment == Mc
  __syncthreads();
  if (t < LM_NSEG) { w->gatherOff[kind][slot] = kind ? offCnt - sMc : offCnt; real->gatherOff[kind][slot] = kind ? offCnt - sMc : offCnt; }
  if (t < VL_MAX_VALID) real->validInd[t] = t < nv ? s->validInd[t] : 0;
  if (t == 0) {
    s->Mc = sMc; s->Ms = total - sMc; w->gatherOff[0][VL_MAX_VALID] = sMc; w->gatherOff[1][VL_MAX_VALID] = total - sMc;
    real->Mc = sMc; real->Ms = total - sMc; real->gatherOff[0][VL_MAX_VALID] = sMc; real->gatherOff[1][VL_MAX_VALID] = total - sMc; real->ok = 1;
  }
  int tailTotal = 0, prefTotal = 0;
  const int tl = cnt - srt;
  const int offTail = lm_scan256(tl, sbuf, &tailTotal);
  const int offPref = lm_scan256(srt, sbuf, &prefTotal);
  if (t < LM_NSEG) { w->tailOff[t] = offTail; w->prefOff[t] = offPref; }
  __shared__ int sTailC;
  if (t == VL_MAX_VALID) sTailC = offTail;
  __syncthreads();
  if (t == 0) { w->tailOff[LM_NSEG] = tailTotal; w->prefOff[LM_NSEG] = prefTotal; s->tailC = sTailC; s->tailS = tailTotal - sTailC; }
}

// The window the next frame will most likely use is the one this frame used (a cube is 50 m wide): right
// after the map update, on the update's stream, its descriptor is rebuilt from the updated cube tables.
__global__ void __launch_bounds__(256) lm_spec_prepare(const LmSub* __restrict__ last, const MapCubeTable* __restrict__ tc,
                                                       const MapCubeTable* __restrict__ ts, LmSub* __restrict__ spec) {
  VL_PDL_WAIT();

  __shared__ int sbuf[256];
  __shared__ int snv;
  if (threadIdx.x == 0) {
    const int cI = last->cI, cJ = last->cJ, cK = last->cK;
    int nv = 0;
    for (int i = cI - 2; i <= cI + 2; i++)  // LM.cpp:448-466, on a freshly reset list
      for (int j = cJ - 2; j <= cJ + 2; j++)
        for (int k = cK - 1; k <= cK + 1; k++)
          if (i >= 0 && i < VL_CUBE_W && j >= 0 && j < VL_CUBE_H && k >= 0 && k < VL_CUBE_D && nv < VL_MAX_VALID)
            spec->validInd[nv++] = i + VL_CUBE_W * j + VL_CUBE_W * VL_CUBE_H * k;
    spec->validNum = nv; snv = nv;
    spec->cI = cI; spec->cJ = cJ; spec->cK = cK; spec->cenW = last->cenW; spec->cenH = last->cenH; spec->cenD = last->cenD;
    spec->gridOrigin[0] = (float)(50 * (cI - 2 - last->cenW) - 25);
    spec->gridOrigin[1] = (float)(50 * (cJ - 2 - last->cenH) - 25);
    spec->gridOrigin[2] = (float)(50 * (cK - 1 - last->cenD) - 25);
  }
  __syncthreads();
  const int nv = snv, t = threadIdx.x;
  const int kind = t / VL_MAX_VALID, slot = t % VL_MAX_VALID;
  int cnt = 0;
  if (t < LM_NSEG && slot < nv) cnt = (kind ? ts : tc)->count[spec->validInd[slot]];
  int total = 0;
  const int offCnt = lm_scan256(cnt, sbuf, &total);
  __shared__ int sMc;
  if (t == VL_MAX_VALID) sMc = offCnt;
  __syncthreads();
  if (t < LM_NSEG) spec->gatherOff[kind][slot] = kind ? offCnt - sMc : offCnt;
  if (t == 0) { spec->Mc = sMc; spec->Ms = total - sMc; spec->gatherOff[0][VL_MAX_VALID] = sMc; spec->gatherOff[1][VL_MAX_VALID] = total - sMc; spec->ok = 1; }
}

// LM.cpp:476-485: concatenate the valid cubes (loop order of LM.cpp:448-452) into the sub-map clouds.
// skip (may be null): device flag "the speculative build already produced exactly this" -> nothing to do.
__device__ __forceinline__ void lm_dev_gather(const LmSub* __restrict__ sub, const MapCubeTable* __restrict__ tc, const MapCubeTable* __restrict__ ts,
                                              const float4* __restrict__ poolC, const float4* __restrict__ poolS,
                                              float4* __restrict__ outC, float4* __restrict__ outS) {
  const int nv = sub->validNum, mc = sub->Mc, total = sub->Mc + sub->Ms;
  for (int g = blockIdx.x * blockDim.x + threadIdx.x; g < total; g += gridDim.x * blockDim.x) {
    const int kind = g >= mc;
    const int e = kind ? g - mc : g;
    const int* off = sub->gatherOff[kind];
    int lo = 0, hi = nv;
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (off[mid] <= e) lo = mid; else hi = mid; }
    const int cb = sub->validInd[lo];
    if (kind) outS[e] = poolS[ts->start[cb] + (e - off[lo])];
    else outC[e] = poolC[tc->start[cb] + (e - off[lo])];
  }
}
// 2 m search cells over the 250 x 250 x 150 m window
__device__ __forceinline__ int lm_cell_coord(float v, float o, int n) {
  const int cidx = (int)floorf(__fmul_rn(__fsub_rn(v, o), 1.0f / LM_CELL));
  return min(max(cidx, 0), n - 1);
}
// ---- persistent voxel-hash grid (lm_grid.cuh): rebuild from the cube pools ------------------------------------------
__device__ __forceinline__ int lg_cell_of(const float4 p, const float* o) {
  return lm_cell_coord(p.x, o[0], LM_GX) + LM_GX * (lm_cell_coord(p.y, o[1], LM_GY) + LM_GY * lm_cell_coord(p.z, o[2], LM_GZ));
}
// empty directory, reset chunk allocator, header <- the window `sub` describes
__global__ void __launch_bounds__(256) lg_zero(LgGrid g, const LmSub* __restrict__ sub) {
  VL_PDL_WAIT();
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < 2 * LM_NCELL; i += gridDim.x * blockDim.x) g.dir[i] = make_int2(0, -1);
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    *g.top = 0;
    LgHeader* h = g.hdr;
    h->valid = 1; h->dirty = 0; h->dead = 0; h->nOps = 0;
    h->cI = sub->cI; h->cJ = sub->cJ; h->cK = sub->cK; h->cenW = sub->cenW; h->cenH = sub->cenH; h->cenD = sub->cenD;
    h->validNum = sub->validNum; h->count[0] = sub->Mc; h->count[1] = sub->Ms;
    for (int k = 0; k < VL_MAX_VALID; ++k) h->validInd[k] = k < sub->validNum ? sub->validInd[k] : 0;
    for (int k = 0; k < 3; ++k) h->origin[k] = sub->gridOrigin[k];
  }
}
// every point of the valid cubes (loop order of LM.cpp:448-452) -> its cell; key = (slot, voxel key) for the filtered prefix,
// (slot, TAIL | position) for unfiltered tail points (they make the grid `dirty`: the next update must take the pool path)
__global__ void __launch_bounds__(256) lg_rebuild(LgGrid g, const LmSub* __restrict__ sub, const LmScalars* __restrict__ s, vloam_b200_params prm,
                                                  const MapCubeTable* __restrict__ tc, const MapCubeTable* __restrict__ ts,
                                                  const float4* __restrict__ poolC, const float4* __restrict__ poolS) {
  VL_PDL_WAIT();
  const int nv = sub->validNum, mc = sub->Mc, total = sub->Mc + sub->Ms;
  const float o[3] = {sub->gridOrigin[0], sub->gridOrigin[1], sub->gridOrigin[2]};
  for (int gi = blockIdx.x * blockDim.x + threadIdx.x; gi < total; gi += gridDim.x * blockDim.x) {
    const int kind = gi >= mc;
    const int e = kind ? gi - mc : gi;
    const int* off = sub->gatherOff[kind];
    int lo = 0, hi = nv;
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (off[mid] <= e) lo = mid; else hi = mid; }
    const int cb = sub->validInd[lo];
    const MapCubeTable* tb = kind ? ts : tc;
    const int pos = e - off[lo];
    const float4 p = (kind ? poolS : poolC)[tb->start[cb] + pos];
    unsigned low;
    if (pos >= tb->sorted[cb]) { low = LG_TAIL | (unsigned)pos; g.hdr->dirty = 1; }
    else low = lm_vox_key_cube(p, lm_leaf_inv(prm, kind), cb, s);
    lg_insert(g, kind * LM_NCELL + lg_cell_of(p, o), p, lg_key(lo, low), pos);
  }
}

// LaserMapping::input (LM.cpp:178-209) + the window test of the in-place path: when the centre cube did not move, nothing
// rolls, the valid list was reset (LM.cpp:132-136) and the grid is clean, this sweep's sub-map IS the grid: no table
// is touched.  Otherwise needSlow is raised: every later kernel of the sweep returns at once and the host repeats the
// mapping stage through lm_prepare (the pool path).  The pose arithmetic is lm_prepare's, statement for statement.
// qc != null: lm_set_counts' work is done here as well (in-place path: one launch fewer on the pose chain; the stacks are filtered
// long before the odometry result arrives).
__global__ void __launch_bounds__(256) lm_prepare_fast(LmScalars* __restrict__ s, const LoScalars* __restrict__ lo, RfWork* __restrict__ w,
                                                       LgHeader* __restrict__ gh, int skip, int resetValid, const int* __restrict__ qc = nullptr,
                                                       const int* __restrict__ qs = nullptr, const int* __restrict__ gridTop = nullptr) {
  VL_PDL_WAIT(); vl_chain_stamp(1);
  if (threadIdx.x <= LM_NSEG && !skip) { w->segCount[threadIdx.x] = 0; w->segFill[threadIdx.x] = 0; }
  if (threadIdx.x != 0) return;
  for (int k = 0; k < 4; ++k) s->q_wodom[k] = lo->q_w[k];
  for (int k = 0; k < 3; ++k) s->t_wodom[k] = lo->t_w[k];
  double r[3];
  vl_qrot(s->q_wmap_wodom, s->t_wodom[0], s->t_wodom[1], s->t_wodom[2], r);
  if (skip) {
    vl_qmul(s->q_wmap_wodom, s->q_wodom, s->q_hf);
    for (int k = 0; k < 3; ++k) s->t_hf[k] = r[k] + s->t_wmap_wodom[k];
    return;
  }
  double qn[4];
  vl_qmul(s->q_wmap_wodom, s->q_wodom, qn);
  for (int k = 0; k < 4; ++k) s->pose[k] = qn[k];
  for (int k = 0; k < 3; ++k) s->pose[4 + k] = r[k] + s->t_wmap_wodom[k];
  int cI = (int)((s->pose[4] + 25.0) / 50.0) + s->cenW;
  int cJ = (int)((s->pose[5] + 25.0) / 50.0) + s->cenH;
  int cK = (int)((s->pose[6] + 25.0) / 50.0) + s->cenD;
  if (s->pose[4] + 25.0 < 0) cI--;
  if (s->pose[5] + 25.0 < 0) cJ--;
  if (s->pose[6] + 25.0 < 0) cK--;
  const bool roll = cI < 3 || cI >= VL_CUBE_W - 3 || cJ < 3 || cJ >= VL_CUBE_H - 3 || cK < 3 || cK >= VL_CUBE_D - 3;
  // (a freshly reset valid list refilled for the same centre cube IS the grid's list: validInd is left as the last pool-path sweep wrote it)
  const bool same = gh->valid && !gh->dirty && !roll && resetValid && cI == gh->cI && cJ == gh->cJ && cK == gh->cK && s->cenW == gh->cenW &&
                    s->cenH == gh->cenH && s->cenD == gh->cenD;
  s->needSlow = same ? 0 : 1;
  if (same) { s->validNum = gh->validNum; s->Mc = gh->count[0]; s->Ms = gh->count[1]; gh->nOps = 0; }
  if (qc) {  // == lm_set_counts
    s->gridTop = *gridTop; s->gridDirty = gh->dirty; s->gridDead = gh->dead; s->gridCount = gh->count[0] + gh->count[1]; s->gridCountC = gh->count[0];
    s->Qc = *qc; s->Qs = *qs;
    s->optimized = (s->Mc > 10 && s->Ms > 50 && *qc + *qs > 0 && !s->needSlow) ? 1 : 0;
    w->nq = s->optimized ? *qc + *qs : 0;
  }
}

// One warp per downsampled feature: 5-NN in the 3x3x3 cell neighbourhood of the voxel-hash grid (exact inside the 1 m
// acceptance ball, SURVEY A.2), ordered by (d2, key) == (d2, canonical id).  Lane r < 27 looks up cell r's directory entry
// (one memory latency for all 27), then the chunks of all cells are visited with every lane busy (VL_WARP_VISIT_FLAT); cells
// with more than LG_C points take further rounds along their chunk chains.
__global__ void __launch_bounds__(256) lg_knn(const LmScalars* __restrict__ s, LgGrid g, const float4* __restrict__ stackC,
                                              const float4* __restrict__ stackS, float4* __restrict__ knnPts, float* __restrict__ knnD2,
                                              unsigned long long* __restrict__ knnKey) {
  VL_PDL_WAIT(); vl_chain_stamp(2);

  const int lane = threadIdx.x & 31;
  const int Qc = s->Qc, Qs = s->Qs, opt = s->optimized;
  double pose[7];  // loaded with the counts: one memory latency instead of two
#pragma unroll
  for (int k = 0; k < 7; ++k) pose[k] = s->pose[k];
  const float ox = g.hdr->origin[0], oy = g.hdr->origin[1], oz = g.hdr->origin[2];
  if (!opt) return;
  const int nWarps = (gridDim.x * blockDim.x) >> 5;
  for (int qi = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; qi < Qc + Qs; qi += nWarps) {
    const int kind = qi >= Qc;
    const float4 po = kind ? stackS[qi - Qc] : stackC[qi];
    double r[3];
    vl_qrot(pose, (double)po.x, (double)po.y, (double)po.z, r);  // pointAssociateToMap (LM.cpp:154-164)
    const float sx = (float)(r[0] + pose[4]), sy = (float)(r[1] + pose[5]), sz = (float)(r[2] + pose[6]);
    const int cx = (int)floorf(__fmul_rn(__fsub_rn(sx, ox), 1.0f / LM_CELL));
    const int cy = (int)floorf(__fmul_rn(__fsub_rn(sy, oy), 1.0f / LM_CELL));
    const int cz = (int)floorf(__fmul_rn(__fsub_rn(sz, oz), 1.0f / LM_CELL));
    float bd[5]; int br[5];
#pragma unroll
    for (int k = 0; k < 5; ++k) { bd[k] = CUDART_INF_F; br[k] = -1; }
    int cnt = 0, head = -1;
    if (lane < 27) {
      const int xx = cx - 1 + lane % 3, yy = cy - 1 + (lane / 3) % 3, zz = cz - 1 + lane / 9;
      if (xx >= 0 && xx < LM_GX && yy >= 0 && yy < LM_GY && zz >= 0 && zz < LM_GZ) {
        const int2 d = g.dir[kind * LM_NCELL + xx + LM_GX * (yy + LM_GY * zz)];
        cnt = d.x; head = d.y;
      }
    }
    while (__any_sync(0xffffffffu, cnt > 0)) {
      const int rb = cnt > 0 ? head * LG_C : 0, rl = min(max(cnt, 0), LG_C);
      VL_WARP_VISIT_FLAT(rb, rl, lane, g.pts, {
        const float d = vl_dist2(sx, sy, sz, t.x, t.y, t.z);
        if (d < bd[4] || (d == bd[4] && d < CUDART_INF_F && lg_key_less(g, p, br[4]))) {  // insertion into the lane-local sorted top-5
          bd[4] = d; br[4] = p;
#pragma unroll
          for (int k = 4; k > 0; --k)
            if (bd[k] < bd[k - 1] || (bd[k] == bd[k - 1] && lg_key_less(g, br[k], br[k - 1]))) {
              const float td = bd[k]; bd[k] = bd[k - 1]; bd[k - 1] = td;
              const int ti = br[k]; br[k] = br[k - 1]; br[k - 1] = ti;
            }
        }
      });
      cnt -= LG_C;
      if (cnt > 0) head = g.next[head];
    }
    // merge the 32 lane-local lists: pop the global minimum of (d2, key) five times.  d2 >= 0, so its bit pattern orders
    // like the value: one hardware warp reduction per pop; equal distances (rare) are resolved on the 64-bit keys
    float nd[5]; int nr[5];
#pragma unroll
    for (int k = 0; k < 5; ++k) {
      const unsigned hb = __float_as_uint(bd[0]);  // +inf (empty list) sorts last
      const unsigned gmin = __reduce_min_sync(0xffffffffu, hb);
      unsigned tie = __ballot_sync(0xffffffffu, hb == gmin && br[0] >= 0);
      int win = -1;
      if (tie) {
        if (__popc(tie) > 1) {
          const unsigned long long ky = (hb == gmin && br[0] >= 0) ? g.key[br[0]] : LG_DEAD;
          const unsigned khi = __reduce_min_sync(0xffffffffu, (unsigned)(ky >> 32));
          const unsigned klo = __reduce_min_sync(0xffffffffu, (unsigned)(ky >> 32) == khi ? (unsigned)ky : 0xffffffffu);
          tie = __ballot_sync(0xffffffffu, ky == (((unsigned long long)khi << 32) | klo));
        }
        win = __ffs(tie) - 1;
      }
      nd[k] = win >= 0 ? __uint_as_float(gmin) : CUDART_INF_F;
      nr[k] = win >= 0 ? __shfl_sync(0xffffffffu, br[0], win) : -1;
      if (lane == win) {
#pragma unroll
        for (int q = 0; q < 4; ++q) { bd[q] = bd[q + 1]; br[q] = br[q + 1]; }
        bd[4] = CUDART_INF_F; br[4] = -1;
      }
    }
#pragma unroll
    for (int k = 0; k < 5; ++k) {
      if (lane == k) {
        knnPts[qi * 5 + k] = nr[k] >= 0 ? g.pts[nr[k]] : make_float4(0.f, 0.f, 0.f, 0.f);
        knnD2[qi * 5 + k] = nd[k];
        if (knnKey) knnKey[qi * 5 + k] = nr[k] >= 0 ? g.key[nr[k]] : LG_DEAD;
      }
    }
  }
}

// debug capture: key -> canonical id of the concatenated sub-map cloud (LM.cpp:476-485); needs the pools in step with the grid
__global__ void __launch_bounds__(256) lg_keys_to_ids(const unsigned long long* __restrict__ keys, int n, int Qc, const LmSub* __restrict__ sub,
                                                      const LmScalars* __restrict__ s, vloam_b200_params prm, const MapCubeTable* __restrict__ tc,
                                                      const MapCubeTable* __restrict__ ts, const float4* __restrict__ poolC,
                                                      const float4* __restrict__ poolS, int* __restrict__ ids) {
  VL_PDL_WAIT();
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const unsigned long long key = keys[t];
  if (key == LG_DEAD) { ids[t] = -1; return; }
  const int kind = (t / 5) >= Qc;
  const int slot = lg_key_slot(key);
  const unsigned low = (unsigned)key;
  const int cb = sub->validInd[slot];
  const MapCubeTable* tb = kind ? ts : tc;
  int pos;
  if (low & LG_TAIL) pos = (int)(low & ~LG_TAIL);
  else {
    const float4* pool = (kind ? poolS : poolC) + tb->start[cb];
    const float inv = lm_leaf_inv(prm, kind);
    int lo = 0, hi = tb->sorted[cb];
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (lm_vox_key_cube(pool[mid], inv, cb, s) < low) lo = mid + 1; else hi = mid; }
    pos = lo;
  }
  ids[t] = sub->gatherOff[kind][slot] + pos;
}
// debug capture: the concatenated sub-map clouds themselves (LM.cpp:476-485)
__global__ void __launch_bounds__(256) lm_gather(const LmSub* __restrict__ sub, const MapCubeTable* __restrict__ tc, const MapCubeTable* __restrict__ ts,
                                                 const float4* __restrict__ poolC, const float4* __restrict__ poolS, float4* __restrict__ outC,
                                                 float4* __restrict__ outS) {
  VL_PDL_WAIT();
  lm_dev_gather(sub, tc, ts, poolC, poolS, outC, outS);
}

// ---- fits -------------------------------------------------------------------------------------
// Eigen::SelfAdjointEigenSolver<Matrix3d> contract (ascending eigenvalues, unit eigenvectors) by the cyclic Jacobi method: branch-light
// and register-resident.  The oracle restates Eigen's own tridiagonal-QR algorithm (oracle_math.cpp), so the two are independent witnesses.
__device__ void lm_sym_eig3(double a[3][3], double evals[3], double evecs[3][3]) {
  double v[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}};
  for (int sweep = 0; sweep < 30; ++sweep) {
    const double off = fabs(a[0][1]) + fabs(a[0][2]) + fabs(a[1][2]);
    if (off == 0.0) break;
    for (int p = 0; p < 2; ++p)
      for (int q = p + 1; q < 3; ++q) {
        if (a[p][q] == 0.0) continue;
        const double theta = (a[q][q] - a[p][p]) / (2.0 * a[p][q]);
        const double t = (theta >= 0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
        const double cs = 1.0 / sqrt(t * t + 1.0), sn = t * cs;
        const double apq = a[p][q];
        a[p][p] -= t * apq;
        a[q][q] += t * apq;
        a[p][q] = a[q][p] = 0.0;
        const int r = 3 - p - q;
        const double arp = a[r][p], arq = a[r][q];
        a[r][p] = a[p][r] = cs * arp - sn * arq;
        a[r][q] = a[q][r] = sn * arp + cs * arq;
        for (int k = 0; k < 3; ++k) {
          const double vkp = v[k][p], vkq = v[k][q];
          v[k][p] = cs * vkp - sn * vkq;
          v[k][q] = sn * vkp + cs * vkq;
        }
      }
  }
  int ord[3] = {0, 1, 2};  // stable insertion sort by eigenvalue (matches std::sort on 3 distinct keys)
  for (int i = 1; i < 3; ++i) for (int j = i; j > 0 && a[ord[j]][ord[j]] < a[ord[j - 1]][ord[j - 1]]; --j) { const int t = ord[j]; ord[j] = ord[j - 1]; ord[j - 1] = t; }
  for (int cidx = 0; cidx < 3; ++cidx) {
    evals[cidx] = a[ord[cidx]][ord[cidx]];
    for (int r = 0; r < 3; ++r) evecs[r][cidx] = v[r][ord[cidx]];
  }
}

// ColPivHouseholderQR<5x3>::solve restated exactly as oracle_math.cpp does.
__device__ void lm_qr_solve_5x3(double A[5][3], double b[5], double x[3]) {
  int perm[3] = {0, 1, 2};
  double maxpivot = 0.0, diag[3] = {0, 0, 0};
  for (int k = 0; k < 3; ++k) {
    int best = k; double bestn = -1.0;
    for (int j = k; j < 3; ++j) { double n2 = 0; for (int i = k; i < 5; ++i) n2 += A[i][j] * A[i][j]; if (n2 > bestn) { bestn = n2; best = j; } }
    if (best != k) { for (int i = 0; i < 5; ++i) { const double t = A[i][k]; A[i][k] = A[i][best]; A[i][best] = t; } const int t = perm[k]; perm[k] = perm[best]; perm[best] = t; }
    double tail2 = 0; for (int i = k + 1; i < 5; ++i) tail2 += A[i][k] * A[i][k];
    const double c0 = A[k][k];
    double beta, tau, v[5] = {0, 0, 0, 0, 0};
    if (tail2 <= DBL_MIN) { tau = 0; beta = c0; }
    else {
      beta = sqrt(c0 * c0 + tail2);
      if (c0 >= 0) beta = -beta;
      for (int i = k + 1; i < 5; ++i) v[i] = A[i][k] / (c0 - beta);
      tau = (beta - c0) / beta;
    }
    v[k] = 1.0;
    if (tau != 0) {
      for (int j = k + 1; j < 3; ++j) {
        double sm = 0; for (int i = k; i < 5; ++i) sm += v[i] * A[i][j];
        sm *= tau; for (int i = k; i < 5; ++i) A[i][j] -= sm * v[i];
      }
      double sm = 0; for (int i = k; i < 5; ++i) sm += v[i] * b[i];
      sm *= tau; for (int i = k; i < 5; ++i) b[i] -= sm * v[i];
    }
    A[k][k] = beta; for (int i = k + 1; i < 5; ++i) A[i][k] = 0;
    diag[k] = beta;
    if (fabs(beta) > maxpivot) maxpivot = fabs(beta);
  }
  int rank = 0;
  for (int k = 0; k < 3; ++k) if (fabs(diag[k]) > DBL_EPSILON * 3.0 * maxpivot) ++rank;
  double y[3] = {0, 0, 0};
  for (int k = rank - 1; k >= 0; --k) { double sm = b[k]; for (int j = k + 1; j < rank; ++j) sm -= A[k][j] * y[j]; y[k] = sm / A[k][k]; }
  for (int k = 0; k < 3; ++k) x[perm[k]] = y[k];
}

// The two fits of LM.cpp:559-603 / 637-680 on five neighbours (f64 from f32 coordinates).  o6: edge -> {a, b} (the two
// synthetic line points), plane -> {unit normal, d, 0, 0}.  Returns the accept flag.
__device__ __forceinline__ bool lm_fit_one(int kind, double P[5][3], double o6[6]) {
  if (!kind) {  // LM.cpp:559-603: PCA line test
    double cen[3] = {0, 0, 0};
    for (int j = 0; j < 5; ++j) for (int k = 0; k < 3; ++k) cen[k] = cen[k] + P[j][k];
    for (int k = 0; k < 3; ++k) cen[k] = cen[k] / 5.0;
    double cov[3][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}};
    for (int j = 0; j < 5; ++j) {
      const double z[3] = {P[j][0] - cen[0], P[j][1] - cen[1], P[j][2] - cen[2]};
      for (int a = 0; a < 3; ++a) for (int b = 0; b < 3; ++b) cov[a][b] = cov[a][b] + z[a] * z[b];
    }
    double ev[3], evec[3][3];
    lm_sym_eig3(cov, ev, evec);
    if (!(ev[2] > 3 * ev[1])) return false;
    for (int k = 0; k < 3; ++k) { const double u = evec[k][2]; o6[k] = 0.1 * u + cen[k]; o6[3 + k] = -0.1 * u + cen[k]; }
    return true;
  }
  // LM.cpp:637-680: least-squares plane n.p + 1 = 0, 0.2 m flatness check
  double A[5][3], B[5] = {-1, -1, -1, -1, -1}, nrm[3];
  for (int j = 0; j < 5; ++j) for (int k = 0; k < 3; ++k) A[j][k] = P[j][k];
  lm_qr_solve_5x3(A, B, nrm);
  const double nn = sqrt(nrm[0] * nrm[0] + nrm[1] * nrm[1] + nrm[2] * nrm[2]);
  const double d = 1 / nn;
  if (nn > 0) { nrm[0] /= nn; nrm[1] /= nn; nrm[2] /= nn; }
  for (int j = 0; j < 5; ++j)
    if (fabs(nrm[0] * P[j][0] + nrm[1] * P[j][1] + nrm[2] * P[j][2] + d) > 0.2) return false;
  o6[0] = nrm[0]; o6[1] = nrm[1]; o6[2] = nrm[2]; o6[3] = d; o6[4] = 0; o6[5] = 0;
  return true;
}

// Line / plane fit of one feature per THREAD (the f64 eigen / QR work of 32 features shares a warp's
// issue slots instead of idling 31 lanes behind lane 0 of the search kernel).
__global__ void __launch_bounds__(128) lm_fit(const LmScalars* __restrict__ s, const float4* __restrict__ stackC, const float4* __restrict__ stackS,
                                              const float4* __restrict__ knnPts, const float* __restrict__ knnD2, int* __restrict__ knnOk,
                                              double* __restrict__ factors, int* __restrict__ valid) {
  VL_PDL_WAIT(); vl_chain_stamp(3);

  const int Qc = s->Qc, Qs = s->Qs, opt = s->optimized;  // (one round trip for the three)
  if (!opt) return;
  for (int qi = blockIdx.x * blockDim.x + threadIdx.x; qi < Qc + Qs; qi += gridDim.x * blockDim.x) {
  const int kind = qi >= Qc;
  // every load of the query is issued before any of them is used: the neighbours are read whether or not the fifth distance
  // passes the gate (lg_knn wrote all five slots of every query), one round trip instead of three
  const float d4 = knnD2[qi * 5 + 4];  // +inf when fewer than five neighbours were found
  float4 nb[5];
#pragma unroll
  for (int j = 0; j < 5; ++j) nb[j] = knnPts[qi * 5 + j];
  const float4 po = kind ? stackS[qi - Qc] : stackC[qi];
  bool ok = false;
  double* f = factors + (size_t)qi * 10;
  if ((double)d4 < 1.0) {
    double P[5][3];
#pragma unroll
    for (int j = 0; j < 5; ++j) { const float4 t = nb[j]; P[j][0] = t.x; P[j][1] = t.y; P[j][2] = t.z; }
    double o6[6];
    ok = lm_fit_one(kind, P, o6);
    if (ok) {
      f[0] = kind ? 2.0 : 0.0; f[1] = po.x; f[2] = po.y; f[3] = po.z;
#pragma unroll
      for (int k = 0; k < 6; ++k) f[4 + k] = o6[k];
    }
  }
  valid[qi] = ok ? 1 : 0;
  knnOk[qi] = ok ? 1 : 0;
  }
}

// vloam_b200_fit: the same fits on caller-supplied five-point sets (parity tests against an independent witness)
__global__ void __launch_bounds__(128) lm_fit_sets(const float* __restrict__ near, int n, int kind, int* __restrict__ ok, double* __restrict__ prm) {
  VL_PDL_WAIT();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double P[5][3], o6[6] = {0, 0, 0, 0, 0, 0};
  for (int j = 0; j < 5; ++j) for (int k = 0; k < 3; ++k) P[j][k] = near[(size_t)i * 15 + j * 3 + k];
  const bool a = lm_fit_one(kind, P, o6);
  ok[i] = a ? 1 : 0;
  for (int k = 0; k < 6; ++k) prm[(size_t)i * 6 + k] = a ? o6[k] : 0.0;
}
int vl_lm_fit_sets(vloam_b200_ctx* c, const float* d_near, int n, int kind, int* d_ok, double* d_prm) {
  VL_LAUNCH(lm_fit_sets, vl_div_up(max(n, 1), 128), 128, 0, d_near, n, kind, d_ok, d_prm);
  VL_CUDA(cudaGetLastError());
  return VLOAM_OK;
}

// hostLmm != null (in-place path): sync point S2 without a copy engine round trip -- the warp writes both scalar structs straight
// into pinned host memory (UVA) and then the frame's sequence number; the host spins on that word.  (Two cudaMemcpyAsync + an
// event cost ~20 us between the final pose and the caller seeing it, which is host turn-around the next sweep's mapping waits for.)
__global__ void lm_transform_update(LmScalars* s, const LgHeader* __restrict__ gh, const int* __restrict__ gridTop, const LoScalars* __restrict__ los,
                                    LmScalars* hostLmm, LoScalars* hostLos, volatile unsigned* hostFlag, unsigned seq) {
  VL_PDL_WAIT(); vl_chain_stamp(5);
  // LM.cpp:147-151
  if (threadIdx.x == 0) {
    if (gh) { s->gridTop = *gridTop; s->gridDirty = gh->dirty; s->gridDead = gh->dead; s->gridCount = gh->count[0] + gh->count[1]; s->gridCountC = gh->count[0]; }
    if (!s->needSlow) vl_transform_update(s->pose, s->q_wodom, s->t_wodom, s->q_wmap_wodom, s->t_wmap_wodom);  // (needSlow: the sweep is repeated on the pool path: leave the state untouched)
  }
  if (!hostLmm) return;
  __syncwarp();
  static_assert(sizeof(LmScalars) % 8 == 0 && sizeof(LoScalars) % 8 == 0, "scalar structs are copied as 8-byte words");
  const unsigned long long* a = reinterpret_cast<const unsigned long long*>(s);
  unsigned long long* ha = reinterpret_cast<unsigned long long*>(hostLmm);
  for (int k = threadIdx.x; k < (int)(sizeof(LmScalars) / 8); k += 32) ha[k] = a[k];
  const unsigned long long* b = reinterpret_cast<const unsigned long long*>(los);
  unsigned long long* hb = reinterpret_cast<unsigned long long*>(hostLos);
  for (int k = threadIdx.x; k < (int)(sizeof(LoScalars) / 8); k += 32) hb[k] = b[k];
  __threadfence_system();
  __syncwarp();
  if (threadIdx.x == 0) *hostFlag = seq;
}

// ---- map update: insert (LM.cpp:741-788) + per-cube VoxelGrid re-filter (LM.cpp:795-808) -------
// sort key: [63:56] segment (kind*125 + valid slot) | [55:26] voxel (iz,iy,ix) | [25:0] order
// order: existing tail point -> its position in the cube; new point -> RF_NEW + its index in the new points.
// (The map publication's keys carry the index of the collected grid entry in `order`, without RF_NEW.)
#define RF_SEG_SHIFT 56
#define RF_VOX_SHIFT 26
#define RF_NEW (1u << 25)
#define RF_NO_KEY (~0ull)  // unused key slot: sorts last, counted in no segment
__device__ __forceinline__ unsigned long long rf_key(int sg, unsigned vk, unsigned ord) {
  return ((unsigned long long)sg << RF_SEG_SHIFT) | ((unsigned long long)vk << RF_VOX_SHIFT) | (unsigned long long)ord;
}
__device__ __forceinline__ unsigned long long rf_key_new(int sg, unsigned vk, int i) { return rf_key(sg, vk, RF_NEW + (unsigned)i); }
__device__ __forceinline__ int rf_key_seg(unsigned long long key) { return (int)(key >> RF_SEG_SHIFT); }
__device__ __forceinline__ unsigned rf_key_vox(unsigned long long key) { return (unsigned)((key >> RF_VOX_SHIFT) & 0x3fffffffull); }
__device__ __forceinline__ unsigned rf_key_ord(unsigned long long key) { return (unsigned)(key & 0x3ffffffull); }
__device__ __forceinline__ bool rf_key_is_new(unsigned long long key) { return rf_key_ord(key) >= RF_NEW; }
__device__ __forceinline__ int rf_key_new_idx(unsigned long long key) { return (int)(rf_key_ord(key) - RF_NEW); }

__global__ void __launch_bounds__(256) rf_keys(const LmScalars* __restrict__ s, RfWork* __restrict__ w, vloam_b200_params prm,
                                               const MapCubeTable* __restrict__ tc, const MapCubeTable* __restrict__ ts,
                                               const float4* __restrict__ poolC, const float4* __restrict__ poolS,
                                               const float4* __restrict__ stackC, const float4* __restrict__ stackS,
                                               float4* __restrict__ newPts, int* __restrict__ newCube,
                                               unsigned long long* __restrict__ keys, int P) {
  VL_PDL_WAIT();

  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= P) return;
  const int tailTotal = w->tailOff[LM_NSEG];
  const int Qc = s->Qc, Qs = s->Qs;
  unsigned long long key = RF_NO_KEY;
  if (g < tailTotal) {  // an existing tail point of a valid cube
    int lo = 0, hi = LM_NSEG;
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (w->tailOff[mid] <= g) lo = mid; else hi = mid; }
    const int kind = lo / VL_MAX_VALID, slot = lo % VL_MAX_VALID;
    const int cb = s->validInd[slot];
    const MapCubeTable* t = kind ? ts : tc;
    const int pos = t->sorted[cb] + (g - w->tailOff[lo]);
    const float4 p = (kind ? poolS : poolC)[t->start[cb] + pos];
    const unsigned vk = lm_vox_key_cube(p, lm_leaf_inv(prm, kind), cb, s);
    key = rf_key(lo, vk, (unsigned)pos);
  } else if (g < tailTotal + Qc + Qs) {  // this frame's point i of the stacks
    const int i = g - tailTotal;
    const int kind = i >= Qc;
    const float4 po = kind ? stackS[i - Qc] : stackC[i];
    double r[3];
    vl_qrot(s->pose, (double)po.x, (double)po.y, (double)po.z, r);
    const float4 p = make_float4((float)(r[0] + s->pose[4]), (float)(r[1] + s->pose[5]), (float)(r[2] + s->pose[6]), po.w);
    const int ci = lm_cube_of(p.x, s->cenW), cj = lm_cube_of(p.y, s->cenH), ck = lm_cube_of(p.z, s->cenD);
    int cb = -1;
    if (ci >= 0 && ci < VL_CUBE_W && cj >= 0 && cj < VL_CUBE_H && ck >= 0 && ck < VL_CUBE_D) cb = ci + VL_CUBE_W * cj + VL_CUBE_W * VL_CUBE_H * ck;
    newPts[i] = p;
    const int slot = cb >= 0 ? w->slotOfCube[cb] : -1;
    newCube[i] = (cb >= 0 && slot < 0) ? cb : -1;  // only cubes outside the window need the raw append path
    if (slot >= 0) {
      const unsigned vk = lm_vox_key(p, lm_leaf_inv(prm, kind), ci, cj, ck, s->cenW, s->cenH, s->cenD);
      key = rf_key_new(kind * VL_MAX_VALID + slot, vk, i);
    }
  }
  keys[g] = key;
  if (key != RF_NO_KEY) atomicAdd(&w->segCount[rf_key_seg(key)], 1);
}

// ---- segmented sort of the update keys ----------------------------------------------------------------
// The keys are (segment | voxel | order) and every later step works per segment (one segment = one valid cube
// of one kind).  Instead of one bitonic network over all keys (37 us for 8k keys: ~48 barrier rounds of a
// 1024-thread CTA pair), the keys are bucketed by segment -- histogram in rf_keys, a 250-entry scan that IS the
// per-segment range table, one scatter -- and each bucket is sorted by its own CTA in shared memory.
// Every block of the scatter scans the 250 counts for itself (one 256-thread scan, ~1 us) instead of waiting for a
// separate single-block launch; block 0 publishes the range table for the later steps.  segFill is zeroed by lm_prepare.
__global__ void __launch_bounds__(256) rf_seg_scatter(const unsigned long long* __restrict__ in, int n, RfWork* __restrict__ w,
                                                      unsigned long long* __restrict__ out) {
  VL_PDL_WAIT();

  __shared__ int sb[256];
  __shared__ int sBegin[256];
  const int t = threadIdx.x;
  const int cnt = t < LM_NSEG ? w->segCount[t] : 0;
  int total = 0;
  const int off = lm_scan256(cnt, sb, &total);
  sBegin[t] = off;
  if (blockIdx.x == 0) {
    if (t < LM_NSEG) { w->tailBegin[t] = off; w->firstViolation[t] = INT_MAX; }
    if (t == 0) { w->tailBegin[LM_NSEG] = total; w->nKeysValid = total; }
  }
  __syncthreads();
  const int g = blockIdx.x * blockDim.x + t;
  if (g >= n) return;
  const unsigned long long key = in[g];
  if (key == RF_NO_KEY) return;
  const int sg = rf_key_seg(key);
  out[sBegin[sg] + atomicAdd(&w->segFill[sg], 1)] = key;
}
#define RF_SEG_THREADS 512
#define RF_SEG_CAP 8192  // keys of one segment sorted in shared memory; larger segments use `scratch` (global)
__global__ void __launch_bounds__(RF_SEG_THREADS) rf_seg_sort(unsigned long long* __restrict__ keys, const RfWork* __restrict__ w,
                                                              unsigned long long* __restrict__ scratch, int cap) {
  VL_PDL_WAIT();

  extern __shared__ unsigned long long sk[];
  const int sg = blockIdx.x;
  const int beg = w->tailBegin[sg], n = w->tailBegin[sg + 1] - beg;
  if (n <= 1) return;
  int P = 8; while (P < n) P <<= 1;
  if (P <= cap) {
    for (int t = threadIdx.x; t < P; t += RF_SEG_THREADS) sk[t] = t < n ? keys[beg + t] : RF_NO_KEY;
    __syncthreads();
    bt_smem_sort<RF_SEG_THREADS>(sk, P);
    for (int t = threadIdx.x; t < n; t += RF_SEG_THREADS) keys[beg + t] = sk[t];
  } else {  // P <= 2 n - 1: the segments' scratch areas [2 beg, 2 beg + P) do not overlap
    unsigned long long* g = scratch + (size_t)2 * beg;
    for (int t = threadIdx.x; t < P; t += RF_SEG_THREADS) g[t] = t < n ? keys[beg + t] : RF_NO_KEY;
    __syncthreads();
    bt_sort_batched<RF_SEG_THREADS>(g, P, 1);
    for (int t = threadIdx.x; t < n; t += RF_SEG_THREADS) keys[beg + t] = g[t];
  }
}

__device__ __forceinline__ float4 rf_key_point(unsigned long long key, const LmScalars* s, const MapCubeTable* tc, const MapCubeTable* ts,
                                               const float4* poolC, const float4* poolS, const float4* newPts) {
  if (rf_key_is_new(key)) return newPts[rf_key_new_idx(key)];
  const int sg = rf_key_seg(key);
  const int kind = sg / VL_MAX_VALID, cb = s->validInd[sg % VL_MAX_VALID];
  return (kind ? poolS : poolC)[(kind ? ts : tc)->start[cb] + (int)rf_key_ord(key)];
}

// For each sorted tail key: is it the head of a run that no prefix point owns?
__global__ void __launch_bounds__(256) rf_match(const unsigned long long* __restrict__ keys, const LmScalars* __restrict__ s,
                                                const RfWork* __restrict__ w, vloam_b200_params prm, const MapCubeTable* __restrict__ tc,
                                                const MapCubeTable* __restrict__ ts, const float4* __restrict__ poolC,
                                                const float4* __restrict__ poolS, int* __restrict__ unmatchedHead) {
  VL_PDL_WAIT();

  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= w->nKeysValid) return;
  const unsigned long long key = keys[t];
  const int sg = rf_key_seg(key);
  const unsigned vk = rf_key_vox(key);
  const bool head = (t == w->tailBegin[sg]) || rf_key_vox(keys[t - 1]) != vk;
  int um = 0;
  if (head) {
    const int kind = sg / VL_MAX_VALID, cb = s->validInd[sg % VL_MAX_VALID];
    const MapCubeTable* tb = kind ? ts : tc;
    const float4* pool = (kind ? poolS : poolC) + tb->start[cb];
    const float inv = lm_leaf_inv(prm, kind);
    int lo = 0, hi = tb->sorted[cb];
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (lm_vox_key_cube(pool[mid], inv, cb, s) < vk) lo = mid + 1; else hi = mid; }
    const bool matched = lo < tb->sorted[cb] && lm_vox_key_cube(pool[lo], inv, cb, s) == vk;
    um = matched ? 0 : 1;
  }
  unmatchedHead[t] = um;
}

__global__ void __launch_bounds__(1024) rf_scan_layout(int* __restrict__ unmatched, const LmScalars* __restrict__ s, RfWork* __restrict__ w,
                                                       const MapCubeTable* __restrict__ tc, const MapCubeTable* __restrict__ ts) {
  VL_PDL_WAIT();

  // exclusive scan of unmatched[0..n) in place, unmatched[n] = total; 8 consecutive flags per thread and round
  __shared__ int ws[32];
  const int n = w->nKeysValid;
  int carry = 0;  // the same value in every thread
  for (int base = 0; base < n; base += 8192) {
    const int b = base + threadIdx.x * 8;
    int v[8];
    if (b + 7 < n) {
      const int4 lo = *reinterpret_cast<const int4*>(unmatched + b), hi = *reinterpret_cast<const int4*>(unmatched + b + 4);
      v[0] = lo.x; v[1] = lo.y; v[2] = lo.z; v[3] = lo.w; v[4] = hi.x; v[5] = hi.y; v[6] = hi.z; v[7] = hi.w;
    } else {
#pragma unroll
      for (int k = 0; k < 8; ++k) v[k] = b + k < n ? unmatched[b + k] : 0;
    }
    int own = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) own += v[k];
    int tot = 0;
    int run = carry + vl_block_excl_scan<1024>(own, ws, &tot);
#pragma unroll
    for (int k = 0; k < 8; ++k) { const int t = v[k]; v[k] = run; run += t; }
    if (b + 7 < n) {
      *reinterpret_cast<int4*>(unmatched + b) = make_int4(v[0], v[1], v[2], v[3]);
      *reinterpret_cast<int4*>(unmatched + b + 4) = make_int4(v[4], v[5], v[6], v[7]);
    } else {
#pragma unroll
      for (int k = 0; k < 8; ++k) if (b + k < n) unmatched[b + k] = v[k];
    }
    carry += tot;
  }
  if (threadIdx.x == 0) unmatched[n] = carry;
  __syncthreads();
  __shared__ int sb2[256];
  const int sg = threadIdx.x;
  int cnt = 0;
  if (sg < LM_NSEG) {
    const int kind = sg / VL_MAX_VALID, slot = sg % VL_MAX_VALID;
    if (slot < s->validNum) {
      const int cb = s->validInd[slot];
      cnt = (kind ? ts : tc)->sorted[cb] + (unmatched[w->tailBegin[sg + 1]] - unmatched[w->tailBegin[sg]]);
    }
  }
  int tot = 0;
  const int off = lm_scan256(cnt, sb2, &tot);
  if (sg < LM_NSEG) { w->outOff[sg] = off; w->outCount[sg] = cnt; }
  if (sg == 0) w->outOff[LM_NSEG] = tot;
}

__device__ __forceinline__ float4 rf_fold(float4 acc, const float4 p) {
  return make_float4(__fadd_rn(acc.x, p.x), __fadd_rn(acc.y, p.y), __fadd_rn(acc.z, p.z), __fadd_rn(acc.w, p.w));
}
__device__ __forceinline__ float4 rf_centroid(const float4 acc, int n) {
  const float fn = (float)n;
  return make_float4(__fdiv_rn(acc.x, fn), __fdiv_rn(acc.y, fn), __fdiv_rn(acc.z, fn), __fdiv_rn(acc.w, fn));
}

// new voxels: runs of tail keys that no prefix point owns
__device__ __forceinline__ void rf_dev_emit_new(int blk, const unsigned long long* __restrict__ keys, const int* __restrict__ uScan,
                                                const LmScalars* __restrict__ s, const RfWork* __restrict__ w, const vloam_b200_params& prm,
                                                const MapCubeTable* __restrict__ tc, const MapCubeTable* __restrict__ ts,
                                                const float4* __restrict__ poolC, const float4* __restrict__ poolS,
                                                const float4* __restrict__ newPts, float4* __restrict__ staging) {
  const int t = blk * blockDim.x + threadIdx.x;
  const int n = w->nKeysValid;
  if (t >= n) return;
  if (uScan[t + 1] == uScan[t]) return;  // not an unmatched head
  const unsigned long long key = keys[t];
  const int sg = rf_key_seg(key);
  const unsigned vk = rf_key_vox(key);
  const int segEnd = w->tailBegin[sg + 1];
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  int cnt = 0;
  for (int q = t; q < segEnd && rf_key_vox(keys[q]) == vk; ++q) { acc = rf_fold(acc, rf_key_point(keys[q], s, tc, ts, poolC, poolS, newPts)); ++cnt; }
  const int kind = sg / VL_MAX_VALID, cb = s->validInd[sg % VL_MAX_VALID];
  const MapCubeTable* tb = kind ? ts : tc;
  const float4* pool = (kind ? poolS : poolC) + tb->start[cb];
  const float inv = lm_leaf_inv(prm, kind);
  int lo = 0, hi = tb->sorted[cb];
  while (lo < hi) { const int mid = (lo + hi) >> 1; if (lm_vox_key_cube(pool[mid], inv, cb, s) < vk) lo = mid + 1; else hi = mid; }
  staging[w->outOff[sg] + lo + (uScan[t] - uScan[w->tailBegin[sg]])] = rf_centroid(acc, cnt);
}

// prefix points: shifted by the new voxels that sort before them; absorb a matching tail run
__device__ __forceinline__ void rf_dev_emit_prefix(int blk, int nblk, const unsigned long long* __restrict__ keys, const int* __restrict__ uScan,
                                                   const LmScalars* __restrict__ s, const RfWork* __restrict__ w, const vloam_b200_params& prm,
                                                   const MapCubeTable* __restrict__ tc, const MapCubeTable* __restrict__ ts,
                                                   const float4* __restrict__ poolC, const float4* __restrict__ poolS,
                                                   const float4* __restrict__ newPts, float4* __restrict__ staging) {
  const int total = w->prefOff[LM_NSEG];
  for (int g = blk * blockDim.x + threadIdx.x; g < total; g += nblk * blockDim.x) {
    int lo = 0, hi = LM_NSEG;
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (w->prefOff[mid] <= g) lo = mid; else hi = mid; }
    const int sg = lo, i = g - w->prefOff[sg];
    const int kind = sg / VL_MAX_VALID, cb = s->validInd[sg % VL_MAX_VALID];
    const MapCubeTable* tb = kind ? ts : tc;
    const float4 p = (kind ? poolS : poolC)[tb->start[cb] + i];
    const unsigned vk = lm_vox_key_cube(p, lm_leaf_inv(prm, kind), cb, s);
    int a = w->tailBegin[sg], b = w->tailBegin[sg + 1];
    const int segBegin = a, segEnd = b;
    while (a < b) { const int mid = (a + b) >> 1; if (rf_key_vox(keys[mid]) < vk) a = mid + 1; else b = mid; }
    float4 acc = rf_fold(make_float4(0.f, 0.f, 0.f, 0.f), p);
    int cnt = 1;
    for (int q = a; q < segEnd && rf_key_vox(keys[q]) == vk; ++q) { acc = rf_fold(acc, rf_key_point(keys[q], s, tc, ts, poolC, poolS, newPts)); ++cnt; }
    staging[w->outOff[sg] + i + (uScan[a] - uScan[segBegin])] = rf_centroid(acc, cnt);
  }
}

// Both emitters in one launch: they write disjoint staging entries and neither reads what the other writes, so the
// first nbNew blocks handle the new voxels (a few long per-run loops) while the rest stream the prefix points.
__global__ void __launch_bounds__(256) rf_emit(int nbNew, const unsigned long long* __restrict__ keys, const int* __restrict__ uScan,
                                               const LmScalars* __restrict__ s, const RfWork* __restrict__ w, vloam_b200_params prm,
                                               const MapCubeTable* __restrict__ tc, const MapCubeTable* __restrict__ ts,
                                               const float4* __restrict__ poolC, const float4* __restrict__ poolS,
                                               const float4* __restrict__ newPts, float4* __restrict__ staging) {
  VL_PDL_WAIT();

  if ((int)blockIdx.x < nbNew) rf_dev_emit_new(blockIdx.x, keys, uScan, s, w, prm, tc, ts, poolC, poolS, newPts, staging);
  else rf_dev_emit_prefix(blockIdx.x - nbNew, gridDim.x - nbNew, keys, uScan, s, w, prm, tc, ts, poolC, poolS, newPts, staging);
}

// grow cube storage where the re-filtered cloud no longer fits (bump allocation from the pool top;
// a block scan keeps the layout deterministic)
__global__ void __launch_bounds__(256) rf_alloc(LmScalars* __restrict__ s, const RfWork* __restrict__ w, MapCubeTable* __restrict__ tc,
                                                MapCubeTable* __restrict__ ts, int poolCapC, int poolCapS) {
  VL_PDL_WAIT();

  __shared__ int sb[256];
  const int sg = threadIdx.x;
  const int kind = sg / VL_MAX_VALID, slot = sg % VL_MAX_VALID;
  int ncapC = 0, ncapS = 0, cb = -1;
  if (sg < LM_NSEG && slot < s->validNum) {
    cb = s->validInd[slot];
    const MapCubeTable* tb = kind ? ts : tc;
    const int need = w->outCount[sg];
    if (need > tb->cap[cb]) { if (kind) ncapS = max(2 * need, 256); else ncapC = max(2 * need, 256); }
  }
  int totC = 0, totS = 0;
  const int offC = lm_scan256(ncapC, sb, &totC);
  const int offS = lm_scan256(ncapS, sb, &totS);
  const int topC = s->poolTopC, topS = s->poolTopS;
  const bool okC = topC + totC <= poolCapC, okS = topS + totS <= poolCapS;
  if (ncapC > 0 && okC) { tc->start[cb] = topC + offC; tc->cap[cb] = ncapC; }
  if (ncapS > 0 && okS) { ts->start[cb] = topS + offS; ts->cap[cb] = ncapS; }
  __syncthreads();
  if (sg == 0) {
    if (okC) s->poolTopC = topC + totC; else s->overflow = 1;
    if (okS) s->poolTopS = topS + totS; else s->overflow = 1;
  }
}

__global__ void __launch_bounds__(256) rf_commit(const float4* __restrict__ staging, LmScalars* __restrict__ s, RfWork* __restrict__ w,
                                                 vloam_b200_params prm, MapCubeTable* __restrict__ tc, MapCubeTable* __restrict__ ts,
                                                 float4* __restrict__ poolC, float4* __restrict__ poolS) {
  VL_PDL_WAIT();

  const int total = w->outOff[LM_NSEG];
  for (int g = blockIdx.x * blockDim.x + threadIdx.x; g < total; g += gridDim.x * blockDim.x) {
    int lo = 0, hi = LM_NSEG;
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (w->outOff[mid] <= g) lo = mid; else hi = mid; }
    const int sg = lo, k = g - w->outOff[sg];
    const int kind = sg / VL_MAX_VALID, cb = s->validInd[sg % VL_MAX_VALID];
    MapCubeTable* tb = kind ? ts : tc;
    if (w->outCount[sg] > tb->cap[cb]) continue;  // pool exhausted (overflow flag is set)
    const float4 p = staging[g];
    (kind ? poolS : poolC)[tb->start[cb] + k] = p;
    if (k > 0) {  // does the re-filtered cloud keep one point per voxel in ascending order?
      const float inv = lm_leaf_inv(prm, kind);
      if (lm_vox_key_cube(staging[g - 1], inv, cb, s) >= lm_vox_key_cube(p, inv, cb, s)) atomicMin(&w->firstViolation[sg], k);
    }
  }
}

__global__ void rf_finish(LmScalars* __restrict__ s, const RfWork* __restrict__ w, MapCubeTable* __restrict__ tc, MapCubeTable* __restrict__ ts) {
  VL_PDL_WAIT();

  const int sg = threadIdx.x;
  if (sg >= LM_NSEG) return;
  const int kind = sg / VL_MAX_VALID, slot = sg % VL_MAX_VALID;
  if (slot >= s->validNum) return;
  const int cb = s->validInd[slot];
  MapCubeTable* tb = kind ? ts : tc;
  if (w->outCount[sg] > tb->cap[cb]) return;
  tb->count[cb] = w->outCount[sg];
  tb->sorted[cb] = min(w->outCount[sg], w->firstViolation[sg]);
}

// Points that land in a cube outside the 5x5x3 window are appended raw, in stack order (LM.cpp:762, 786).
// One CTA walks the stacks in chunks of 1024: outside points are compacted in order, ranked among
// the points of the same (kind, cube) inside the chunk, cube storage is grown where needed, and every
// point is written to count + rank.  The common case (no outside point at all) is one pass of flags.
__global__ void __launch_bounds__(1024) rf_append_outside(LmScalars* __restrict__ s, const float4* __restrict__ newPts,
                                                          const int* __restrict__ newCube, MapCubeTable* __restrict__ tc,
                                                          MapCubeTable* __restrict__ ts, float4* __restrict__ poolC, float4* __restrict__ poolS,
                                                          int poolCapC, int poolCapS, const int* __restrict__ anyOutside) {
  VL_PDL_WAIT();

  // in-place path: mu_keys left {a point fell outside the window, points, needSlow, Qc} of ITS sweep in anyOutside[0..3] -- the next
  // sweep's lm_prepare_fast may be rewriting LmScalars while this kernel runs (the pose chain does not wait for it)
  if (anyOutside && (anyOutside[2] || !*anyOutside)) return;
  const int Qc = anyOutside ? anyOutside[3] : s->Qc, total = anyOutside ? anyOutside[1] : s->Qc + s->Qs;
  __shared__ int lIdx[1024], lKey[1024];
  __shared__ int gKey[1024], gOld[1024], gNew[1024], gCnt[1024];
  __shared__ int warpSum[32];
  __shared__ int nGrow;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int any = 0, outC = 0, outS = 0;
  for (int i = threadIdx.x; i < total; i += 1024) if (newCube[i] >= 0) { any = 1; if (i < Qc) ++outC; else ++outS; }
  if (__syncthreads_or(any) == 0) return;
  if (outC) atomicAdd(&s->outsideC, outC);  // (the host's bound on the map size follows these counts, read at the next S2)
  if (outS) atomicAdd(&s->outsideS, outS);
  for (int base = 0; base < total; base += 1024) {
    const int i = base + threadIdx.x;
    const int cb = i < total ? newCube[i] : -1;
    const bool f = cb >= 0;
    const unsigned bal = __ballot_sync(0xffffffffu, f);
    if (lane == 0) warpSum[warp] = __popc(bal);
    if (threadIdx.x == 0) nGrow = 0;
    __syncthreads();
    int before = 0, n = 0;
    for (int w = 0; w < 32; ++w) { const int v = warpSum[w]; if (w < warp) before += v; n += v; }
    if (f) { const int pos = before + __popc(bal & ((1u << lane) - 1u)); lIdx[pos] = i; lKey[pos] = (i >= Qc ? VL_CUBE_NUM : 0) + cb; }
    __syncthreads();
    if (n == 0) continue;
    // rank inside the chunk among entries of the same (kind, cube); the first one is the leader
    const int e = threadIdx.x;
    int key = -1, rank = 0, tot = 0;
    if (e < n) {
      key = lKey[e];
      for (int q = 0; q < n; ++q) { const bool same = lKey[q] == key; rank += (same && q < e); tot += same; }
      if (rank == 0) {
        const int kind = key >= VL_CUBE_NUM, c2 = key - kind * VL_CUBE_NUM;
        const MapCubeTable* tb = kind ? ts : tc;
        if (tb->count[c2] + tot > tb->cap[c2]) { const int g = atomicAdd(&nGrow, 1); gKey[g] = key; gCnt[g] = tb->count[c2] + tot; }
      }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      for (int g = 0; g < nGrow; ++g) {
        const int kind = gKey[g] >= VL_CUBE_NUM, c2 = gKey[g] - kind * VL_CUBE_NUM;
        MapCubeTable* tb = kind ? ts : tc;
        const int ncap = max(2 * gCnt[g], 256);
        int& top = kind ? s->poolTopS : s->poolTopC;
        gOld[g] = tb->start[c2];
        if (top + ncap > (kind ? poolCapS : poolCapC)) { s->overflow = 1; gNew[g] = -1; continue; }
        gNew[g] = top; tb->start[c2] = top; tb->cap[c2] = ncap; top += ncap;
      }
    }
    __syncthreads();
    for (int g = 0; g < nGrow; ++g) {
      if (gNew[g] < 0) continue;
      const int kind = gKey[g] >= VL_CUBE_NUM, c2 = gKey[g] - kind * VL_CUBE_NUM;
      float4* pool = kind ? poolS : poolC;
      const int cnt = (kind ? ts : tc)->count[c2];
      for (int q = threadIdx.x; q < cnt; q += 1024) pool[gNew[g] + q] = pool[gOld[g] + q];
    }
    __syncthreads();
    if (e < n) {
      const int kind = key >= VL_CUBE_NUM, c2 = key - kind * VL_CUBE_NUM;
      MapCubeTable* tb = kind ? ts : tc;
      if (tb->count[c2] + tot <= tb->cap[c2]) (kind ? poolS : poolC)[tb->start[c2] + tb->count[c2] + rank] = newPts[lIdx[e]];
    }
    __syncthreads();
    if (e < n && rank == 0) {
      const int kind = key >= VL_CUBE_NUM, c2 = key - kind * VL_CUBE_NUM;
      MapCubeTable* tb = kind ? ts : tc;
      if (tb->count[c2] + tot <= tb->cap[c2]) tb->count[c2] += tot;
    }
    __syncthreads();
  }
}

// ---- in-place map update on the voxel-hash grid (LM.cpp:741-808 without touching the other ~1M points) -------------------
// pcl::VoxelGrid over [cube cloud ; this sweep's points] changes only the voxels the new points fall into.  Two launches:
//   mu_keys   every new point: world transform (LM.cpp:744, 768), cube, voxel key; points of the same (cube, voxel) meet in a
//             small open-addressing hash table: the point that claims the slot leads the group and looks the map point of that
//             voxel up IN THE GRID -- it lies inside the voxel's box, i.e. in one of the <= 2x2x2 cells the box overlaps --
//             and every point appends itself to the slot's member list
//   mu_apply  every leader: the fold exactly as VoxelGrid does it: map point first (it has the lower index), then the members
//             in stack order, f32 sums, one division.  The centroid is stored back in place, or appended to its cell
//             when the voxel is new or the centroid left its 2 m cell (the old entry is tombstoned).
// No sort: round 1's update sorted (segment | voxel | order) keys, 30 us for the one cube that holds most of a sweep.
// A centroid that no longer maps to its own voxel (f32 rounding at a voxel face) is legal -- the next VoxelGrid pass re-keys
// it -- but outside the in-place scheme: it raises `dirty`, and the next sweep runs the pool path on materialised cubes.
#define MU_CAP 16           // members of a voxel group kept in its slot (a world voxel collects at most the points of the ~8 lidar-frame
                            // voxels it overlaps -- the stacks are voxel-filtered at the same leaf; more: the leader walks the stack)
struct MuWork {            // device scratch of one update (sized by the host for nq points)
  unsigned long long* hkey;  // [H] hash table: (segment << 32 | voxel key) or empty
  int* cnt;                  // [H] points of the group
  int H;                     // power of two >= 4 nq
  int* slotOf;               // [nq] hash slot of point i (| MU_LEAD for the point that claimed the slot), -1: not in a valid cube
  int* found;                // [nq] leaders: grid entry of the voxel's map point (-1: new voxel), and the cell it sits in
  int* foundCell;            // [nq]
  int* members;              // [H * MU_CAP] stack indices, in arrival order
  int* anyOutside;           // a point fell into a cube outside the 5x5x3 window (rf_append_outside has work)
};
#define MU_LEAD 0x40000000
__device__ __forceinline__ unsigned mu_hash(unsigned long long k) { k ^= k >> 31; k *= 0x9E3779B97F4A7C15ull; k ^= k >> 29; return (unsigned)k; }

// where the grid holds the map point of voxel (slot, vk) of kind `kind`: entry index and cell, -1 when the voxel is empty.
// Called while nothing modifies the grid (mu_keys: the previous update is complete, this one inserts only in mu_apply).
__device__ __forceinline__ void mu_lookup(const LmScalars* __restrict__ s, const vloam_b200_params& prm, const LgGrid& g, int sg, unsigned vk,
                                          int& foundOut, int& foundCellOut) {
  const int kind = sg / VL_MAX_VALID, slot = sg % VL_MAX_VALID, cb = s->validInd[slot];
  const float leaf = kind ? prm.plane_res : prm.line_res;
  const float inv = lm_leaf_inv(prm, kind);
  const int ci = cb % VL_CUBE_W, cj = (cb / VL_CUBE_W) % VL_CUBE_H, ck = cb / (VL_CUBE_W * VL_CUBE_H);
  // world voxel index of the run: inverse of lm_vox_key
  const int gx = (int)(vk & 1023u) + (int)floorf(__fmul_rn((float)(50 * (ci - s->cenW) - 25), inv)) - 2;
  const int gy = (int)((vk >> 10) & 1023u) + (int)floorf(__fmul_rn((float)(50 * (cj - s->cenH) - 25), inv)) - 2;
  const int gz = (int)(vk >> 20) + (int)floorf(__fmul_rn((float)(50 * (ck - s->cenD) - 25), inv)) - 2;
  const float* o = g.hdr->origin;
  const float eps = 0.02f * leaf;  // p * inv is rounded: a point of voxel gx may sit a few ulp outside [gx, gx + 1) * leaf
  const int x0 = lm_cell_coord((float)gx * leaf - eps, o[0], LM_GX), x1 = lm_cell_coord((float)(gx + 1) * leaf + eps, o[0], LM_GX);
  const int y0 = lm_cell_coord((float)gy * leaf - eps, o[1], LM_GY), y1 = lm_cell_coord((float)(gy + 1) * leaf + eps, o[1], LM_GY);
  const int z0 = lm_cell_coord((float)gz * leaf - eps, o[2], LM_GZ), z1 = lm_cell_coord((float)(gz + 1) * leaf + eps, o[2], LM_GZ);
  const unsigned long long want = lg_key(slot, vk);
  int found = -1, foundCell = -1;
  if (x1 - x0 <= 1 && y1 - y0 <= 1 && z1 - z0 <= 1) {
    // leaf <= 2 m: the box spans at most 2 x 2 x 2 cells.  All directory entries, then the first chunk of every cell, are
    // loaded without waiting for one another (a serial walk is ~20 dependent L2 round trips per voxel)
    int cellId[8]; int2 dd[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const int xx = x0 + (q & 1), yy = y0 + ((q >> 1) & 1), zz = z0 + (q >> 2);
      const bool on = xx <= x1 && yy <= y1 && zz <= z1;
      cellId[q] = kind * LM_NCELL + xx + LM_GX * (yy + LM_GY * zz);
      dd[q] = on ? __ldcg(&g.dir[cellId[q]]) : make_int2(0, -1);  // (L2: other voxels' appends to these cells may be in flight)
    }
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      if (dd[q].x <= 0 || dd[q].y < 0) continue;
      const ulonglong2* kp = reinterpret_cast<const ulonglong2*>(g.key + (size_t)dd[q].y * LG_C);
      const int m = min(dd[q].x, LG_C);
#pragma unroll
      for (int i = 0; i < LG_C / 2; ++i) {
        const ulonglong2 kk = __ldcg(&kp[i]);
        if (2 * i < m && kk.x == want) { found = dd[q].y * LG_C + 2 * i; foundCell = cellId[q]; }
        if (2 * i + 1 < m && kk.y == want) { found = dd[q].y * LG_C + 2 * i + 1; foundCell = cellId[q]; }
      }
    }
    if (found < 0) {
#pragma unroll
      for (int q = 0; q < 8; ++q) {  // longer chains (> LG_C points in a cell)
        int chunk = dd[q].y;
        for (int left = dd[q].x - LG_C; left > 0 && found < 0 && chunk >= 0; left -= LG_C) {
          chunk = __ldcg(&g.next[chunk]);
          if (chunk < 0) break;  // (another voxel's append is still extending this chain: nothing of ours can be beyond)
          const int m = min(left, LG_C);
          const ulonglong2* kp = reinterpret_cast<const ulonglong2*>(g.key + (size_t)chunk * LG_C);
#pragma unroll
          for (int i = 0; i < LG_C / 2; ++i) {  // all 16 keys of the chunk in flight at once (a scalar loop with an early exit is 16 dependent L2 round trips)
            const ulonglong2 kk = __ldcg(&kp[i]);
            if (2 * i < m && kk.x == want) { found = chunk * LG_C + 2 * i; foundCell = cellId[q]; }
            if (2 * i + 1 < m && kk.y == want) { found = chunk * LG_C + 2 * i + 1; foundCell = cellId[q]; }
          }
        }
      }
    }
  } else {
    for (int zz = z0; zz <= z1 && found < 0; ++zz)
      for (int yy = y0; yy <= y1 && found < 0; ++yy)
        for (int xx = x0; xx <= x1 && found < 0; ++xx) {
          const int cell = kind * LM_NCELL + xx + LM_GX * (yy + LM_GY * zz);
          const int2 d = __ldcg(&g.dir[cell]);
          int chunk = d.y;
          for (int left = d.x; left > 0 && found < 0 && chunk >= 0; left -= LG_C, chunk = left > 0 ? __ldcg(&g.next[chunk]) : -1) {
            const int m = min(left, LG_C);
            for (int i = 0; i < m; ++i)
              if (__ldcg(&g.key[chunk * LG_C + i]) == want) { found = chunk * LG_C + i; foundCell = cell; break; }
          }
        }
  }
  foundOut = found; foundCellOut = foundCell;
}

// Grouping AND look-up in one launch: the point that claims a voxel's hash slot (CAS winner) becomes the group's leader and looks
// the voxel's map point up in the grid right away -- its two dependent L2 round trips overlap the other points' hashing --
// and every point, the leader included, appends itself to the slot's member list.  (Round 2's first version elected the lowest
// stack index with atomicMin and needed a second launch, mu_group, before anybody knew the leader.)
__global__ void __launch_bounds__(256) mu_keys(const LmScalars* __restrict__ s, const RfWork* __restrict__ w, vloam_b200_params prm, LgGrid g,
                                               const float4* __restrict__ stackC, const float4* __restrict__ stackS, float4* __restrict__ newPts,
                                               int* __restrict__ newCube, MuWork m) {
  VL_PDL_WAIT(); vl_chain_stamp(6);
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int Qc = s->Qc, Qs = s->Qs;
  if (i == 0) { m.anyOutside[1] = s->needSlow ? 0 : Qc + Qs; m.anyOutside[2] = s->needSlow; m.anyOutside[3] = Qc; }  // (for rf_append_outside)
  if (s->needSlow || i >= Qc + Qs) return;  // (queued before the host knows whether the sweep stays on the in-place path, and with a bound on the count)
  const int kind = i >= Qc;
  const float4 po = kind ? stackS[i - Qc] : stackC[i];
  double r[3];
  vl_qrot(s->pose, (double)po.x, (double)po.y, (double)po.z, r);
  const float4 p = make_float4((float)(r[0] + s->pose[4]), (float)(r[1] + s->pose[5]), (float)(r[2] + s->pose[6]), po.w);
  const int ci = lm_cube_of(p.x, s->cenW), cj = lm_cube_of(p.y, s->cenH), ck = lm_cube_of(p.z, s->cenD);
  int cb = -1;
  if (ci >= 0 && ci < VL_CUBE_W && cj >= 0 && cj < VL_CUBE_H && ck >= 0 && ck < VL_CUBE_D) cb = ci + VL_CUBE_W * cj + VL_CUBE_W * VL_CUBE_H * ck;
  newPts[i] = p;
  const int slot = cb >= 0 ? w->slotOfCube[cb] : -1;
  newCube[i] = (cb >= 0 && slot < 0) ? cb : -1;  // only cubes outside the window need the raw append path
  int hs = -1;
  if (slot >= 0) {
    const unsigned vk = lm_vox_key(p, lm_leaf_inv(prm, kind), ci, cj, ck, s->cenW, s->cenH, s->cenD);
    const int sg = kind * VL_MAX_VALID + slot;
    const unsigned long long key = ((unsigned long long)sg << 32) | vk;
    unsigned h = mu_hash(key) & (unsigned)(m.H - 1);
    bool won = false;
    for (;;) {
      const unsigned long long prev = atomicCAS(&m.hkey[h], ~0ull, key);
      if (prev == ~0ull) { won = true; break; }
      if (prev == key) break;
      h = (h + 1) & (unsigned)(m.H - 1);
    }
    const int pos = atomicAdd(&m.cnt[h], 1);
    if (pos < MU_CAP) m.members[(size_t)h * MU_CAP + pos] = i;
    hs = (int)h;
    if (won) {
      hs |= MU_LEAD;
      int f, fc;
      mu_lookup(s, prm, g, sg, vk, f, fc);
      m.found[i] = f; m.foundCell[i] = fc;
    }
  } else if (cb >= 0) *m.anyOutside = 1;
  m.slotOf[i] = hs;
}
__global__ void __launch_bounds__(128) mu_apply(const LmScalars* __restrict__ s, vloam_b200_params prm, LgGrid g, const float4* __restrict__ newPts,
                                                MuWork mw) {
  VL_PDL_WAIT(); vl_chain_stamp(7);
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  const int soRaw = mw.slotOf[t];  // (in bounds for every launched thread: the grid covers the host bound the buffer was sized for; issued with the scalars)
  const int nq = s->needSlow ? 0 : s->Qc + s->Qs;
  const int so = t < nq ? soRaw : -1;
  int bornKind = -1, died = 0;  // bookkeeping of this thread's voxel, added up per warp at the end (thousands of atomics on ONE address cost ~50 us)
  if (so >= 0 && (so & MU_LEAD)) {  // the leader of its voxel
  const int hs = so & ~MU_LEAD;
  const int found = mw.found[t], foundCell = mw.foundCell[t];
  const int nm = mw.cnt[hs];
  int mem[MU_CAP];
#pragma unroll
  for (int q = 0; q < MU_CAP; ++q) mem[q] = q < nm ? mw.members[(size_t)hs * MU_CAP + q] : 0x7fffffff;
  const unsigned long long hk = mw.hkey[hs];
  const int sg = (int)(hk >> 32);
  const unsigned vk = (unsigned)hk;
  const int kind = sg / VL_MAX_VALID, slot = sg % VL_MAX_VALID, cb = s->validInd[slot];
  const float inv = lm_leaf_inv(prm, kind);
  const int ci = cb % VL_CUBE_W, cj = (cb / VL_CUBE_W) % VL_CUBE_H, ck = cb / (VL_CUBE_W * VL_CUBE_H);
  const float* o = g.hdr->origin;
  const unsigned long long want = lg_key(slot, vk);
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  int cnt = 0;
  if (found >= 0) { acc = rf_fold(acc, g.pts[found]); cnt = 1; }
  if (nm <= MU_CAP) {
    // arrival order is arbitrary: take the members in stack order (nm is 1..3 for nearly every voxel)
    int last = -1;
    for (int q = 0; q < nm; ++q) {
      int best = 0x7fffffff;
#pragma unroll
      for (int r = 0; r < MU_CAP; ++r) { const int v = mem[r]; if (v > last && v < best) best = v; }
      acc = rf_fold(acc, newPts[best]); ++cnt;
      last = best;
    }
  } else {
    for (int j = 0; j < nq; ++j) if ((mw.slotOf[j] & ~MU_LEAD) == hs && mw.slotOf[j] >= 0) { acc = rf_fold(acc, newPts[j]); ++cnt; }  // (more members than slots: walk the stack)
  }
  const float4 c = rf_centroid(acc, cnt);
  if (lm_vox_key(c, inv, ci, cj, ck, s->cenW, s->cenH, s->cenD) != vk) g.hdr->dirty = 1;  // drifted across a voxel face: pool path next sweep
  const int cell = kind * LM_NCELL + lg_cell_of(c, o);
  // The entry stays where it is even when the centroid slid into the neighbouring 2 m cell, as long as leaf <= 0.95 m: it cannot leave
  // its voxel's box (checked above), so it stays within `leaf` of the cell that lists it, and a query that accepts it (d2 < 1 m^2) is
  // then closer than 2 m to that cell, i.e. still visits it (27-cell search).  Voxels that straddle a cell boundary used to be
  // tombstoned and re-appended every time their centroid crossed it: ~500 per sweep, 10 % dead entries after 200 sweeps, and the
  // sweeps before a window move ran 15-20 % slower than the ones after its rebuild (profiles/r2_long_run_1000_sweeps.txt).
  const float leafK = kind ? prm.plane_res : prm.line_res;
  if (found >= 0 && (cell == foundCell || leafK <= 0.95f)) g.pts[found] = c;
  else {
    int pos = -1;
    if (found >= 0) { pos = g.posOf[found]; g.pts[found].x = CUDART_INF_F; *(volatile unsigned long long*)&g.key[found] = LG_DEAD; died = 1; }
    else bornKind = kind;
    lg_insert(g, cell, c, want, pos);
  }
  }
  const unsigned b0 = __ballot_sync(0xffffffffu, bornKind == 0), b1 = __ballot_sync(0xffffffffu, bornKind == 1), bd = __ballot_sync(0xffffffffu, died);
  if ((threadIdx.x & 31) == 0) {
    if (b0) atomicAdd(&g.hdr->count[0], __popc(b0));
    if (b1) atomicAdd(&g.hdr->count[1], __popc(b1));
    if (bd) atomicAdd(&g.hdr->dead, __popc(bd));
  }
}

// ---- grid -> cube pools (the pools are the exchange format: export, window moves, the pool-path update) ----------------------
// In-place updates leave the valid cubes' pool segments behind in two ways: coordinates of voxels that absorbed new points, and
// voxels that did not exist when the grid was built.  mz_collect walks the grid once: an entry that came from the pools writes
// its current coordinates back to its old position (the filtered prefix keeps its order: voxel keys do not change); a voxel
// created since becomes a "new point" of ONE ordinary pool-path merge (rf_seg_scatter ... rf_finish with no stack points):
// unique voxel keys, so the merge only moves each of them to its sorted position -- the cubes come out exactly as
// pcl::VoxelGrid leaves them (LM.cpp:795-808), through the same code the pool path runs every sweep.
__global__ void __launch_bounds__(256) mz_layout_for_grid(LmScalars* __restrict__ s, RfWork* __restrict__ w, LgHeader* __restrict__ gh,
                                                          const MapCubeTable* __restrict__ tc, const MapCubeTable* __restrict__ ts) {
  VL_PDL_WAIT();
  __shared__ int sbuf[256];
  const int t = threadIdx.x;
  const int nv = gh->validNum;
  if (t < VL_MAX_VALID && t < nv) s->validInd[t] = gh->validInd[t];  // the merge below addresses cubes through the context's list
  if (t == 0) { s->validNum = nv; gh->nOps = 0; }
  if (t <= LM_NSEG) { w->segCount[t] = 0; w->segFill[t] = 0; }
  const int kind = t / VL_MAX_VALID, slot = t % VL_MAX_VALID;
  int cnt = 0, srt = 0;
  if (t < LM_NSEG && slot < nv) {
    const MapCubeTable* tb = kind ? ts : tc;
    cnt = tb->count[gh->validInd[slot]]; srt = tb->sorted[gh->validInd[slot]];
  }
  int tailTotal = 0, prefTotal = 0;
  const int offTail = lm_scan256(cnt - srt, sbuf, &tailTotal);
  const int offPref = lm_scan256(srt, sbuf, &prefTotal);
  if (t < LM_NSEG) { w->tailOff[t] = offTail; w->prefOff[t] = offPref; }
  if (t == 0) { w->tailOff[LM_NSEG] = tailTotal; w->prefOff[LM_NSEG] = prefTotal; }
}
__global__ void __launch_bounds__(256) mz_collect(LgGrid g, RfWork* __restrict__ w, const MapCubeTable* __restrict__ tc, const MapCubeTable* __restrict__ ts,
                                                  float4* __restrict__ poolC, float4* __restrict__ poolS, float4* __restrict__ newPts,
                                                  int* __restrict__ newCube, unsigned long long* __restrict__ keys, int cap) {
  VL_PDL_WAIT();
  lg_for_each_live(g, LM_NCELL, [&](int e, unsigned long long key, int kind) {
    const int slot = lg_key_slot(key), cb = g.hdr->validInd[slot];
    const int pos = g.posOf[e];
    if (pos >= 0) { (kind ? poolS : poolC)[(kind ? ts : tc)->start[cb] + pos] = g.pts[e]; return; }
    const int j = atomicAdd(&g.hdr->nOps, 1);
    if (j >= cap) { g.hdr->dirty = 1; return; }  // (the host bounds the voxels created since the last build: cannot happen)
    const int sg = kind * VL_MAX_VALID + slot;
    newPts[j] = g.pts[e]; newCube[j] = -1;
    keys[j] = rf_key_new(sg, lg_key_vox(key), j);
    atomicAdd(&w->segCount[sg], 1);
  });
}

// after an import: longest strictly increasing voxel-key prefix of every cube
__global__ void __launch_bounds__(256) lm_scan_sorted(const LmScalars* __restrict__ s, vloam_b200_params prm, MapCubeTable* __restrict__ t,
                                                      const float4* __restrict__ pool, int kind) {
  VL_PDL_WAIT();

  const int cb = blockIdx.x;
  __shared__ int firstBad;
  if (threadIdx.x == 0) firstBad = INT_MAX;
  __syncthreads();
  const int n = t->count[cb];
  const float inv = lm_leaf_inv(prm, kind);
  const float4* p = pool + t->start[cb];
  for (int k = 1 + threadIdx.x; k < n; k += blockDim.x)
    if (lm_vox_key_cube(p[k - 1], inv, cb, s) >= lm_vox_key_cube(p[k], inv, cb, s)) atomicMin(&firstBad, k);
  __syncthreads();
  if (threadIdx.x == 0) t->sorted[cb] = min(n, firstBad);
}

// gh != null (in-place path): the grid's bookkeeping for the host (read at S2) is taken HERE, before this sweep's in-place update can
// touch it -- that update starts the moment the pose is final, beside lm_transform_update.
__global__ void lm_set_counts(LmScalars* s, RfWork* w, const int* qc, const int* qs, const LgHeader* __restrict__ gh, const int* __restrict__ gridTop) {
  VL_PDL_WAIT();

  if (threadIdx.x != 0) return;
  if (gh) { s->gridTop = *gridTop; s->gridDirty = gh->dirty; s->gridDead = gh->dead; s->gridCount = gh->count[0] + gh->count[1]; s->gridCountC = gh->count[0]; }
  s->Qc = *qc; s->Qs = *qs;
  // LM.cpp:514: optimise only against a sub-map with > 10 corner and > 50 surf points
  s->optimized = (s->Mc > 10 && s->Ms > 50 && *qc + *qs > 0 && !s->needSlow) ? 1 : 0;
  w->nq = s->optimized ? *qc + *qs : 0;  // factor slots the solver looks at
}

// ---- LaserMapping::publish: laserCloudMap (LM.cpp:884-899) assembled on the device, without touching the map -------------------
// Output: for cube i = 0 .. 4850 in table order, corner cube i then surf cube i -- segment q = 2 i + kind -- each cube's points in
// the order the pools hold them after a pool-path sweep (pcl::VoxelGrid's order, raw appends after it).  Where a segment's points
// are taken from:
//   * the pools, for every cube when they are current, and for the cubes outside the grid's window otherwise;
//   * the grid, for the grid window's valid cubes after in-place updates (the pools are stale there).  The live entries of such a
//     segment, in ascending voxel key, are what lm_materialize would write: an entry from the build keeps its rank in the stale
//     (key-ordered) pool prefix, shifted by the voxels created since with a smaller key; a voxel created since goes to the number
//     of prefix points with a smaller key (binary search, as rf_match) plus its rank among the new voxels of its segment (sorted
//     per segment with rf_seg_scatter / rf_seg_sort).  One scatter then writes every point to its final slot.
// Nothing here writes pools, cube tables, the grid or LmScalars; the merge scratch is the assembly's own.
#define MP_NSEG (2 * VL_CUBE_NUM)
#define MP_INTS (2 * MP_NSEG + 2)
#define MP_CNT (MP_NSEG + 1)   // pubInt[MP_CNT]: voxels created since the grid was built (collected)
#define MP_SRC (MP_NSEG + 2)   // pubInt[MP_SRC + q]: pool start of segment q, -1 = from the grid

// every live grid entry created since the build (posOf < 0) -> (segment | voxel key | j) and its entry index
__global__ void __launch_bounds__(256) mp_collect(LgGrid g, RfWork* __restrict__ w, unsigned long long* __restrict__ keys, int* __restrict__ ent,
                                                  int* __restrict__ counter, int cap) {
  VL_PDL_WAIT();
  lg_for_each_live(g, LM_NCELL, [&](int e, unsigned long long key, int kind) {
    if (g.posOf[e] >= 0) return;
    const int j = atomicAdd(counter, 1);
    if (j >= cap) return;  // (the host bounds the voxels created since the build; vl_lm_get_map reports a violation)
    const int sg = kind * VL_MAX_VALID + lg_key_slot(key);
    keys[j] = rf_key(sg, lg_key_vox(key), (unsigned)j);
    ent[j] = e;
    atomicAdd(&w->segCount[sg], 1);
  });
}

// points per output segment -> exclusive offsets (pubInt[0 .. MP_NSEG]) and where each segment comes from (pubInt[MP_SRC + q])
__global__ void __launch_bounds__(1024) mp_layout(const LgHeader* __restrict__ gh, const RfWork* __restrict__ w, const MapCubeTable* __restrict__ tc,
                                                  const MapCubeTable* __restrict__ ts, int fromGrid, int* __restrict__ pub) {
  VL_PDL_WAIT();
  __shared__ int slotOf[VL_CUBE_NUM];
  __shared__ int ws[32];
  for (int i = threadIdx.x; i < VL_CUBE_NUM; i += 1024) slotOf[i] = -1;
  __syncthreads();
  if (fromGrid && (int)threadIdx.x < gh->validNum) slotOf[gh->validInd[threadIdx.x]] = threadIdx.x;
  __syncthreads();
  constexpr int PER = (MP_NSEG + 1023) / 1024;
  const int q0 = threadIdx.x * PER;
  int cnt[PER], own = 0;
#pragma unroll
  for (int k = 0; k < PER; ++k) {
    const int q = q0 + k;
    cnt[k] = 0;
    if (q >= MP_NSEG) continue;
    const int cb = q >> 1, kind = q & 1;
    const MapCubeTable* tb = kind ? ts : tc;
    const int slot = slotOf[cb];
    cnt[k] = tb->count[cb] + (slot >= 0 ? w->segCount[kind * VL_MAX_VALID + slot] : 0);
    pub[MP_SRC + q] = slot >= 0 ? -1 : tb->start[cb];
    own += cnt[k];
  }
  int tot = 0;
  int run = vl_block_excl_scan<1024>(own, ws, &tot);
#pragma unroll
  for (int k = 0; k < PER; ++k) if (q0 + k < MP_NSEG) { pub[q0 + k] = run; run += cnt[k]; }
  if (threadIdx.x == 0) pub[MP_NSEG] = tot;
}

// segments taken from the pools: one thread per output point
__global__ void __launch_bounds__(256) mp_copy_pools(const int* __restrict__ pub, const float4* __restrict__ poolC, const float4* __restrict__ poolS,
                                                     float4* __restrict__ out, int outCap) {
  VL_PDL_WAIT();
  const int total = min(pub[MP_NSEG], outCap);
  for (int g = blockIdx.x * blockDim.x + threadIdx.x; g < total; g += gridDim.x * blockDim.x) {
    int lo = 0, hi = MP_NSEG;
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (pub[mid] <= g) lo = mid; else hi = mid; }
    const int src = pub[MP_SRC + lo];
    if (src >= 0) out[g] = ((lo & 1) ? poolS : poolC)[src + g - pub[lo]];
  }
}

// segments taken from the grid, entries that existed when it was built: stale pool rank + new voxels of the segment with a smaller key
__global__ void __launch_bounds__(256) mp_grid_old(LgGrid g, const RfWork* __restrict__ w, const unsigned long long* __restrict__ sorted,
                                                   const int* __restrict__ pub, float4* __restrict__ out, int outCap) {
  VL_PDL_WAIT();
  lg_for_each_live(g, LM_NCELL, [&](int e, unsigned long long key, int kind) {
    const int pos = g.posOf[e];
    if (pos < 0) return;
    const int slot = lg_key_slot(key), sg = kind * VL_MAX_VALID + slot;
    const unsigned vk = lg_key_vox(key);
    const int base = pub[2 * g.hdr->validInd[slot] + kind] + pos;
    int a = w->tailBegin[sg], b = w->tailBegin[sg + 1];
    const int segBegin = a;
    while (a < b) { const int mid = (a + b) >> 1; if (rf_key_vox(sorted[mid]) < vk) a = mid + 1; else b = mid; }
    const int o = base + (a - segBegin);
    if (o < outCap) out[o] = g.pts[e];
  });
}

// segments taken from the grid, voxels created since the build (sorted per segment): prefix points with a smaller key + rank
__global__ void __launch_bounds__(256) mp_grid_new(LgGrid g, const RfWork* __restrict__ w, const unsigned long long* __restrict__ sorted,
                                                   const int* __restrict__ ent, vloam_b200_params prm, const MapCubeTable* __restrict__ tc,
                                                   const MapCubeTable* __restrict__ ts, const float4* __restrict__ poolC,
                                                   const float4* __restrict__ poolS, const int* __restrict__ pub, float4* __restrict__ out, int outCap) {
  VL_PDL_WAIT();
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= w->nKeysValid) return;
  const unsigned long long key = sorted[t];
  const int sg = rf_key_seg(key);
  const int kind = sg / VL_MAX_VALID, slot = sg % VL_MAX_VALID;
  const unsigned vk = rf_key_vox(key);
  const LgHeader* h = g.hdr;
  const int cb = h->validInd[slot];
  const int ci = cb % VL_CUBE_W, cj = (cb / VL_CUBE_W) % VL_CUBE_H, ck = cb / (VL_CUBE_W * VL_CUBE_H);
  const MapCubeTable* tb = kind ? ts : tc;
  const float4* pool = (kind ? poolS : poolC) + tb->start[cb];
  const float inv = lm_leaf_inv(prm, kind);
  int lo = 0, hi = tb->count[cb];  // (every point of a grid-window cube is in its filtered prefix: a tail would have kept the grid dirty)
  while (lo < hi) { const int mid = (lo + hi) >> 1; if (lm_vox_key(pool[mid], inv, ci, cj, ck, h->cenW, h->cenH, h->cenD) < vk) lo = mid + 1; else hi = mid; }
  const int o = pub[2 * cb + kind] + lo + (t - w->tailBegin[sg]);
  if (o < outCap) out[o] = g.pts[ent[rf_key_ord(key)]];
}

// -----------------------------------------------------------------------------------------------
#define LM_POOL_C (16 << 20)
#define LM_POOL_S (48 << 20)

struct LmDevice {  // extra device state owned by this file
  RfWork* work;
  DBuf<float4> newPts; DBuf<int> newCube;
  DBuf<int> unmatched;
  int* dQ;          // 2 x two device ints: Qc, Qs from the voxel filters (pair ctx::stackSel is current)
  long long hMapUpperC, hMapUpperS;  // host upper bounds on the total map size
  LmSub* subReal; LmSub* subSpec;    // sub-map window descriptors (lm_prepare's / the one rebuilt after a pool-path update)
  // ---- the persistent voxel-hash grid (lm_grid.cuh)
  LgGrid grid;                       // device pointers (dir, chunks, allocator, header)
  DBuf<unsigned long long> muKey; DBuf<int> muInt;  // scratch of the in-place update (MuWork: hash table, groups)
  DBuf<int> knnIds;                  // debug capture: canonical ids of the neighbours
  bool gridEnabled;                  // VLOAM_NO_GRID unset: in-place updates and the post-update rebuild are on
  bool noWorker;                     // VLOAM_NO_WORKER set: the caller issues everything itself (no helper thread)
  bool gridValid;                    // host: the grid was (re)built behind the last map update and nothing edited the map since
  bool poolsStale;                   // host: the valid cubes' pools are behind the grid (in-place updates since the last materialisation)
  long long gridTopUpper;            // host bound on the chunks in use
  long long newVoxUpper;             // host bound on the voxels created by in-place updates since the grid was built
  long long builtCount;              // live points the grid held when it was built
  long long builtCountC;             // ... of them corner points
  long long baseC, baseS;            // bound on the map size (all cubes) when the grid was built, and the raw appends outside the window
  long long outBaseC, outBaseS;      // counted until then: the bound of every later sweep follows the DEVICE counts from there (no drift)
  long long paths[2];                // mapped sweeps since create that took the in-place path / the pool path ("lm.paths")
  // ---- map publication (LaserMapping::publish's laserCloudMap, vl_lm_publish_map)
  cudaStream_t pubStream;            // the assembly runs here, behind the last map update; every later map edit waits for evPub
  cudaEvent_t evPub;
  RfWork* pubWork;                   // the assembly's own merge scratch (the update's `work` may be in use by the next sweep)
  int* pubInt;                       // [MP_NSEG + 1] output offsets (last: points) | new-voxel counter | [MP_NSEG] pool start or -1 (grid)
  DBuf<unsigned long long> pubKeys; DBuf<int> pubEnt;  // new voxels: sort keys (unsorted | sorted | scratch) and their grid entries
  DBuf<float4> pubOut;               // the published cloud
  bool pubDone;                      // something was published since create
  long long pubNewCap, pubOutCap;    // bounds the last assembly was sized for (checked by vl_lm_get_map)
  // ---- prior maps (vloam_b200_load_map / set_map_update / get_map_kind); the buffers are reserved by the first call
  bool mapUpdate;                    // LM.cpp:741-808 runs on mapped sweeps (vloam_b200_set_map_update; default on)
  DBuf<float4> ldIn[2];              // the caller's corner / surf clouds, packed
  DBuf<unsigned long long> ldKeys;   // (cube | voxel | input index) keys of both kinds
  DBuf<int> ldInt;                   // LD_SCALARS scalars | per-cube output offsets of both kinds | per-tile run heads of both kinds
  DBuf<int> pubKindOff;              // get_map_kind: output offset of every cube's segment of one kind (+ total)
  DBuf<float4> pubKind;              // ... and the cloud
};

// chunk pool of the grid: P points occupy at most min(P, cells) + P / LG_C chunks (every cell ends in one partly filled chunk)
// (+ P / 4: chunks leaked by lost CAS races while many threads open the same cell at once)
static long long lg_chunk_bound(long long points) { return (points < 2LL * LM_NCELL ? points : 2LL * LM_NCELL) + points / LG_C + points / 4 + 4096; }
static int lg_reserve(vloam_b200_ctx* c, LmDevice* d, long long chunks) {
  if (chunks <= d->grid.cap) return VLOAM_OK;
  long long ncap = d->grid.cap ? d->grid.cap : (1LL << 20);
  while (ncap < chunks) ncap *= 2;
  VL_CUDA(cudaStreamSynchronize(VL_STREAM(c)));  // (only ever called right before a full rebuild: the old contents are dead)
  if (d->pubStream) VL_CUDA(cudaEventSynchronize(d->evPub));  // ... but a map publication may still be reading them
  if (d->grid.pts) { cudaFree(d->grid.pts); cudaFree(d->grid.key); cudaFree(d->grid.next); cudaFree(d->grid.posOf); }
  __atomic_fetch_add(&c->regrows, 1LL, __ATOMIC_RELAXED);
  VL_CUDA(cudaMalloc(&d->grid.pts, (size_t)ncap * LG_C * sizeof(float4)));
  VL_CUDA(cudaMalloc(&d->grid.key, (size_t)ncap * LG_C * sizeof(unsigned long long)));
  VL_CUDA(cudaMalloc(&d->grid.next, (size_t)ncap * sizeof(int)));
  VL_CUDA(cudaMalloc(&d->grid.posOf, (size_t)ncap * LG_C * sizeof(int)));
  d->grid.cap = (int)ncap;
  return VLOAM_OK;
}

int vl_lm_init(vloam_b200_ctx* c) {
  LmDevice* d = new LmDevice();
  c->lm = d;
  VL_CUDA(cudaMalloc(&d->work, sizeof(RfWork)));
  VL_CUDA(cudaMemset(d->work, 0, sizeof(RfWork)));
  VL_CUDA(cudaMalloc(&d->dQ, sizeof(int) * 4));
  VL_CUDA(cudaMemset(d->dQ, 0, sizeof(int) * 4));
  VL_CUDA(cudaMalloc(&d->subReal, sizeof(LmSub))); VL_CUDA(cudaMemset(d->subReal, 0, sizeof(LmSub)));
  VL_CUDA(cudaMalloc(&d->subSpec, sizeof(LmSub))); VL_CUDA(cudaMemset(d->subSpec, 0, sizeof(LmSub)));
  memset(&d->grid, 0, sizeof d->grid);
  VL_CUDA(cudaMalloc(&d->grid.dir, sizeof(int2) * 2 * LM_NCELL));
  VL_CUDA(cudaMalloc(&d->grid.top, sizeof(int)));
  VL_CUDA(cudaMemset(d->grid.top, 0, sizeof(int)));
  VL_CUDA(cudaMalloc(&d->grid.hdr, sizeof(LgHeader)));
  VL_CUDA(cudaMemset(d->grid.hdr, 0, sizeof(LgHeader)));
  VL_TRY(lg_reserve(c, d, 1 << 21));  // 2 Mi chunks (~0.8 GB of the 180 GB): a ~30M-point sub-map before the first regrow
  VL_CUDA(cudaStreamCreateWithFlags(&d->pubStream, cudaStreamNonBlocking));  // (default = lowest priority: the assembly is never on the pose chain)
  VL_CUDA(cudaEventCreateWithFlags(&d->evPub, cudaEventDisableTiming));
  VL_CUDA(cudaMalloc(&d->pubWork, sizeof(RfWork)));
  VL_CUDA(cudaMalloc(&d->pubInt, sizeof(int) * MP_INTS));
  VL_CUDA(cudaMemset(d->pubInt, 0, sizeof(int) * MP_INTS));
  d->gridEnabled = getenv("VLOAM_NO_GRID") == nullptr;
  d->noWorker = getenv("VLOAM_NO_WORKER") != nullptr;
  d->gridValid = false; d->poolsStale = false; d->gridTopUpper = 0; d->newVoxUpper = 0; d->builtCount = 0; d->mapUpdate = true;
  VL_CUDA(cudaFuncSetAttribute(rf_seg_sort, cudaFuncAttributeMaxDynamicSharedMemorySize, RF_SEG_CAP * 8));
  d->hMapUpperC = d->hMapUpperS = 0;
  // Map pools: bump allocation with doubling per cube; when a pool is half full it is doubled (copy) at sync point
  // S2, so a long drive degrades into a rare ~ms stall instead of VLOAM_E_CAPACITY.  VLOAM_POOL_POINTS: initial
  // size of the corner pool in points (the surf pool gets 3x), for tests of the growth path.
  const char* pp = getenv("VLOAM_POOL_POINTS");
  if (pp) {  // exact sizes (vl_reserve rounds small requests up)
    const size_t pc = (size_t)max(atoll(pp), 4096LL);
    VL_CUDA(cudaMalloc(&c->poolC.p, pc * sizeof(float4))); c->poolC.cap = pc;
    VL_CUDA(cudaMalloc(&c->poolS.p, 3 * pc * sizeof(float4))); c->poolS.cap = 3 * pc;
  } else {
    VL_TRY(vl_reserve(c, c->poolC, LM_POOL_C));
    VL_TRY(vl_reserve(c, c->poolS, LM_POOL_S));
  }
  VL_CUDA(cudaMemset(c->cubeC, 0, sizeof(MapCubeTable)));
  VL_CUDA(cudaMemset(c->cubeS, 0, sizeof(MapCubeTable)));
  LmScalars h;
  memset(&h, 0, sizeof h);
  h.cenW = 10; h.cenH = 10; h.cenD = 5;  // LM.h:75-78
  h.pose[3] = 1.0; h.q_wmap_wodom[3] = 1.0; h.q_wodom[3] = 1.0; h.q_hf[3] = 1.0;
  VL_CUDA(cudaMemcpy(c->lmm, &h, sizeof h, cudaMemcpyHostToDevice));
  *c->h_lmm = h;
  return VLOAM_OK;
}

void vl_lm_free(vloam_b200_ctx* c) {  // everything vl_lm_init and this file's reserves own (the pools are freed by capi.cu)
  LmDevice* d = c->lm;
  if (!d) return;
  if (d->pubStream) { cudaStreamSynchronize(d->pubStream); cudaStreamDestroy(d->pubStream); }
  if (d->evPub) cudaEventDestroy(d->evPub);
  void* dev[] = {d->work, d->dQ, d->subReal, d->subSpec, d->newPts.p, d->newCube.p, d->unmatched.p, d->grid.dir, d->grid.top, d->grid.hdr,
                 d->grid.pts, d->grid.key, d->grid.next, d->grid.posOf, d->muKey.p, d->muInt.p, d->knnIds.p,
                 d->pubWork, d->pubInt, d->pubKeys.p, d->pubEnt.p, d->pubOut.p, d->ldIn[0].p, d->ldIn[1].p, d->ldKeys.p, d->ldInt.p,
                 d->pubKindOff.p, d->pubKind.p};
  for (void* p : dev) vl_dev_free(c, p);
  delete d;
  c->lm = nullptr;
}

extern bool vl_debug_capture(const vloam_b200_ctx* c);

// LM.cpp:492-500: VoxelGrid of this frame's less-sharp / less-flat clouds.  They depend on scan
// registration only, so the odometry stage enqueues them on the side stream right after its first sync
// point and they run underneath the odometry kernels; solveMapping waits on evStacks.
// The filters only conflict with the previous map update through rf_keys, the one kernel that reads the previous
// stacks (evKeys), not with the rest of the update or the speculative sub-map behind it.
// early = true (the counts were known when the sweep arrived: look-ahead scan registration): the helper thread
// issues the ~14 launches while the caller queues the odometry, so the stacks are ready well before the mapping
// front needs them; whoever needs evStacks joins the helper first (vl_lm_run does).
static int lm_issue_stacks(vloam_b200_ctx* c, const float4* corner, int nc, const float4* surf, int ns, bool toNext) {
  LmDevice* d = c->lm;
  struct Restore { cudaStream_t prev; ~Restore() { vl_tls_stream = prev; } } restore{vl_tls_stream};
  DBuf<float4>& dstS = toNext ? c->stackSN : c->stackS;
  DBuf<float4>& dstC = toNext ? c->stackCN : c->stackC;
  int* dq = d->dQ + 2 * (toNext ? c->stackSel ^ 1 : c->stackSel);
  // surf filter on stream2 (scratch lane 0), corner filter beside it on stream4 (scratch lane 1)
  vl_tls_stream = c->stream2;
  // the buffers about to be overwritten were last read by rf_keys of the update that used this pair (stream3)
  const int pairW = toNext ? c->stackSel ^ 1 : c->stackSel;
  cudaStreamWaitEvent(c->stream2, toNext ? c->evKeysSel[pairW] : c->evKeys, 0);
  int r = vl_reserve(c, dstS, (size_t)max(ns, 1));
  if (r == VLOAM_OK) r = vl_voxel_grid_device(c, surf, ns, nullptr, c->prm.plane_res, dstS.p, dq + 1, 0);
  if (c->timing) cudaEventRecord(c->evx[3], c->stream2);
  vl_tls_stream = c->stream4;
  cudaStreamWaitEvent(c->stream4, toNext ? c->evKeysSel[pairW] : c->evKeys, 0);
  if (r == VLOAM_OK) r = vl_reserve(c, dstC, (size_t)max(nc, 1));
  if (r == VLOAM_OK) r = vl_voxel_grid_device(c, corner, nc, nullptr, c->prm.line_res, dstC.p, dq, 1);
  if (c->timing) cudaEventRecord(c->evx[4], c->stream4);
  if (r != VLOAM_OK) return r;
  VL_CUDA(cudaEventRecord(c->evStacks, c->stream2));
  VL_CUDA(cudaEventRecord(c->evStacksC, c->stream4));
  if (!toNext) c->stacksReady = true;
  return VLOAM_OK;
}
int vl_lm_enqueue_stacks(vloam_b200_ctx* c, const float4* corner, int nc, const float4* surf, int ns, bool early, bool ownClouds) {
  VL_TRY(vl_lm_join(c));  // evKeys of the previous frame's update must have been recorded before it is waited on
  if (!ownClouds) {  // the caller's clouds (vloam_b200_laser_mapping_input): behind their upload, and behind any filter of this sweep's own
    VL_CUDA(cudaStreamWaitEvent(c->stream2, c->evIn, 0));
    VL_CUDA(cudaStreamWaitEvent(c->stream4, c->evIn, 0));
  } else if (vl_to_end(c)) {  // the clouds are this sweep's end clouds (LO.cpp:537-556): filter them behind its TransformToEnd
    VL_CUDA(cudaStreamWaitEvent(c->stream2, c->evEnd, 0));
    VL_CUDA(cudaStreamWaitEvent(c->stream4, c->evEnd, 0));
  }
  if (early && !c->lm->noWorker && !c->prof_name[0] && !vl_debug_capture(c))
    return lm_submit(c, [=]() -> int { return lm_issue_stacks(c, corner, nc, surf, ns, false); });
  return lm_issue_stacks(c, corner, nc, surf, ns, false);
}
// The next sweep's stacks, filtered while this sweep's mapping still runs (its scan registration finished early): they
// go to the spare buffers and the spare pair of counts, so nothing of this sweep is disturbed -- this sweep's mapping has
// been queued already (it holds its own wait on evStacks), its map update reads the current buffers.
int vl_lm_enqueue_stacks_next(vloam_b200_ctx* c, const float4* corner, int nc, const float4* surf, int ns) {
  c->stacksNextReady = false;
  if (c->lm->noWorker) VL_TRY(lm_issue_stacks(c, corner, nc, surf, ns, true));
  else VL_TRY(lm_submit(c, [=]() -> int { return lm_issue_stacks(c, corner, nc, surf, ns, true); }));
  c->stacksNextReady = true;
  return VLOAM_OK;
}
int vl_lm_adopt_stacks_next(vloam_b200_ctx* c) {
  VL_TRY(vl_lm_join(c));  // the helper may still be issuing them (it owns the spare DBufs until it is done)
  { DBuf<float4> t_ = c->stackC; c->stackC = c->stackCN; c->stackCN = t_; }
  { DBuf<float4> t_ = c->stackS; c->stackS = c->stackSN; c->stackSN = t_; }
  c->stackSel ^= 1;
  c->stacksReady = true;
  return VLOAM_OK;
}

// ---- host side of the voxel-hash grid ------------------------------------------------------------------------------------
// (re)build the grid for the window `sub` describes from the cube pools, on the calling thread's stream
static int lg_rebuild_launch(vloam_b200_ctx* c, LmDevice* d, const LmSub* sub, long long pointsBound) {
  VL_TRY(lg_reserve(c, d, lg_chunk_bound(pointsBound)));
  const int gsGrid = c->num_sms * 8;
  VL_BYTES(16.0 * LM_NCELL);
  VL_LAUNCH(lg_zero, gsGrid, 256, 0, d->grid, sub);
  VL_BYTES(16.0 * (double)pointsBound);  // SURVEY 8(d) B_lm: the sub-map is read once to build the search structure
  VL_LAUNCH(lg_rebuild, gsGrid, 256, 0, d->grid, sub, c->lmm, c->prm, c->cubeC, c->cubeS, c->poolC.p, c->poolS.p);
  d->gridTopUpper = lg_chunk_bound(pointsBound);
  d->newVoxUpper = 0; d->builtCount = -1;  // (-1: taken from the device count at the next sync point S2)
  return VLOAM_OK;
}

// Pool head room: a cube that outgrows its segment gets a new one of twice its new size, so one pass over the valid cubes
// allocates at most 2 x (points + inserts) + 256 per touched cube.  When that no longer fits the pool is doubled (copy) --
// only ever called where the previous update is complete and the next one has not been issued.
static int lm_pool_headroom(vloam_b200_ctx* c, long long totalC, long long totalS, int Qc, int Qs) {
  const size_t needC = 2 * ((size_t)totalC + Qc) + 256 * (size_t)(VL_MAX_VALID + min(Qc, VL_CUBE_NUM));
  const size_t needS = 2 * ((size_t)totalS + Qs) + 256 * (size_t)(VL_MAX_VALID + min(Qs, VL_CUBE_NUM));
  const bool growC = (size_t)c->h_lmm->poolTopC + needC > c->poolC.cap, growS = (size_t)c->h_lmm->poolTopS + needS > c->poolS.cap;
  if (growC || growS) VL_CUDA(cudaEventSynchronize(c->lm->evPub));  // a map publication in flight reads the pool that is replaced
  if ((size_t)c->h_lmm->poolTopC + needC > c->poolC.cap) VL_TRY(vl_reserve(c, c->poolC, 2 * ((size_t)c->h_lmm->poolTopC + needC), true));
  if ((size_t)c->h_lmm->poolTopS + needS > c->poolS.cap) VL_TRY(vl_reserve(c, c->poolS, 2 * ((size_t)c->h_lmm->poolTopS + needS), true));
  return VLOAM_OK;
}

// ---- the pool path's merge (LM.cpp:795-808): keys of tail points and new points merged into the filtered prefixes of the valid cubes
#define LG_NEWVOX_MAX (1 << 20)  // voxels the in-place updates may create before the pools are brought up to date (bounds the merge's buffers)
// key array of a merge: [0, N) unsorted keys | [N, 2N) bucketed + sorted | [2N, 4N) scratch for oversize segments
static size_t lm_merge_stride(long long keys) { return ((size_t)keys + 255) & ~(size_t)255; }

// Buffers of one merge: `keys` keys, `newPoints` new points, filtered prefixes of at most `prefix` points.  The per-sweep sizes follow
// the map and ask for slack; the one-off pre-sizing for the largest grid -> pools merge (a first window move must not stall on five
// cudaMallocs) asks for none.
static int lm_reserve_merge(vloam_b200_ctx* c, LmDevice* d, long long keys, long long newPoints, long long prefix, bool slack = true) {
  const size_t N = lm_merge_stride(keys);
  VL_TRY(vl_reserve(c, c->tailKeys, 4 * N, false, slack ? 4 * N : 0));
  VL_TRY(vl_reserve(c, d->newPts, (size_t)newPoints));
  VL_TRY(vl_reserve(c, d->newCube, (size_t)newPoints));
  VL_TRY(vl_reserve(c, d->unmatched, (size_t)keys + 2, false, slack ? (size_t)keys + (1 << 16) : 0));
  VL_TRY(vl_reserve(c, c->staging, (size_t)prefix + keys + 1, false, (size_t)prefix / 2 + (1 << 20)));
  return VLOAM_OK;
}

// The merge of the nKeys keys in tailKeys, on the calling thread's stream: bucketed and sorted per segment (one valid cube of one
// kind), every run matched against its cube's filtered prefix, laid out, emitted, cube storage grown, committed.  emitPts / commitPts:
// points the emit and the commit step read and write (algorithmic bytes, VL_BYTES).
static int lm_queue_merge(vloam_b200_ctx* c, LmDevice* d, int nKeys, double emitPts, double commitPts) {
  const size_t N = lm_merge_stride(nKeys);
  unsigned long long* keysIn = c->tailKeys.p;
  unsigned long long* keysSorted = c->tailKeys.p + N;
  const int gsGrid = c->num_sms * 8, nb = vl_div_up(nKeys, 256);
  static const int segCap = getenv("VLOAM_SEG_CAP") ? max(8, min(atoi(getenv("VLOAM_SEG_CAP")), RF_SEG_CAP)) : RF_SEG_CAP;  // tests force the global path
  VL_LAUNCH(rf_seg_scatter, nb, 256, 0, keysIn, nKeys, d->work, keysSorted);
  VL_BYTES(16.0 * nKeys);
  VL_LAUNCH(rf_seg_sort, LM_NSEG, RF_SEG_THREADS, (size_t)RF_SEG_CAP * 8, keysSorted, d->work, c->tailKeys.p + 2 * N, segCap);
  VL_LAUNCH(rf_match, nb, 256, 0, keysSorted, c->lmm, d->work, c->prm, c->cubeC, c->cubeS, c->poolC.p, c->poolS.p, d->unmatched.p);
  VL_LAUNCH(rf_scan_layout, 1, 1024, 0, d->unmatched.p, c->lmm, d->work, c->cubeC, c->cubeS);
  VL_BYTES(32.0 * emitPts);
  VL_LAUNCH(rf_emit, nb + gsGrid, 256, 0, nb, keysSorted, d->unmatched.p, c->lmm, d->work, c->prm, c->cubeC, c->cubeS, c->poolC.p, c->poolS.p,
            d->newPts.p, c->staging.p);
  VL_LAUNCH(rf_alloc, 1, 256, 0, c->lmm, d->work, c->cubeC, c->cubeS, (int)c->poolC.cap, (int)c->poolS.cap);
  VL_BYTES(32.0 * commitPts);
  VL_LAUNCH(rf_commit, gsGrid, 256, 0, c->staging.p, c->lmm, d->work, c->prm, c->cubeC, c->cubeS, c->poolC.p, c->poolS.p);
  VL_LAUNCH(rf_finish, 1, 256, 0, c->lmm, d->work, c->cubeC, c->cubeS);
  return VLOAM_OK;
}

// grid -> pools for the valid cubes of the grid's window (the in-place updates left those pools behind); on the calling thread's stream
static int lm_materialize(vloam_b200_ctx* c, LmDevice* d) {
  const long long total = d->hMapUpperC + d->hMapUpperS;
  const int P = (int)max(min(d->newVoxUpper, (long long)LG_NEWVOX_MAX), 1LL);   // bound on the voxels created since the grid was built
  VL_TRY(lm_pool_headroom(c, d->hMapUpperC, d->hMapUpperS, 0, 0));
  VL_TRY(lm_reserve_merge(c, d, P, P, total));
  const int gsGrid = c->num_sms * 8;
  VL_CUDA(cudaStreamWaitEvent(VL_STREAM(c), d->evPub, 0));  // a map publication may still read the stale pools and the grid
  VL_CUDA(cudaMemsetAsync(c->tailKeys.p, 0xff, lm_merge_stride(P) * sizeof(unsigned long long), VL_STREAM(c)));  // unused key slots read as "no key"
  VL_LAUNCH(mz_layout_for_grid, 1, 256, 0, c->lmm, d->work, d->grid.hdr, c->cubeC, c->cubeS);
  VL_BYTES(32.0 * (double)total);
  VL_LAUNCH(mz_collect, gsGrid, 256, 0, d->grid, d->work, c->cubeC, c->cubeS, c->poolC.p, c->poolS.p, d->newPts.p, d->newCube.p, c->tailKeys.p, P);
  VL_TRY(lm_queue_merge(c, d, P, (double)total, (double)total));
  d->poolsStale = false;
  d->gridValid = false;  // (the entries' pool positions are no longer the pools': the grid is rebuilt before its next use)
  d->newVoxUpper = 0;
  VL_CUDA(cudaGetLastError());
  return VLOAM_OK;
}

// make the cube pools current (export, import, external edits): nothing to do unless in-place updates ran since
int vl_lm_sync_pools(vloam_b200_ctx* c) {
  LmDevice* d = c->lm;
  if (!d || !d->poolsStale) return VLOAM_OK;
  VL_TRY(vl_lm_join(c));
  VL_CUDA(cudaStreamWaitEvent(c->stream, c->evMap, 0));
  VL_CUDA(cudaMemcpyAsync(c->h_lmm, c->lmm, sizeof(LmScalars), cudaMemcpyDeviceToHost, c->stream));  // poolTop for the head-room check
  VL_CUDA(cudaStreamSynchronize(c->stream));
  VL_TRY(lm_materialize(c, d));
  VL_CUDA(cudaStreamSynchronize(c->stream));
  return VLOAM_OK;
}

// the two association + solve passes of LM.cpp:526-717 and transformUpdate (LM.cpp:737) over the sub-map of d->subReal; every kernel
// reads its sizes on the device.  The caller has ordered the main stream behind this sweep's stacks and set the counts.
// losPub != null (in-place path): the pose is final after the passes (evPose), and lm_transform_update hands both scalar structs --
// the odometry state from losPub -- to the host for sync point S2 itself.
// afterHead (may be empty): host work that is not on the pose chain -- arranging and submitting the side work -- runs once the first
// kNN + fit are queued, so the device already has ~35 us of work when the host turns to it.
static int lm_queue_passes(vloam_b200_ctx* c, LmDevice* d, int nqBound, bool capture, const LoScalars* losPub,
                           const std::function<int()>& afterHead = std::function<int()>()) {
  const bool earlyPose = losPub != nullptr;
  if (c->timing) VL_CUDA(cudaEventRecord(c->evx[1], c->stream));
  int Qc = 0, Qs = 0;
  if (capture) {  // debug snapshots need host counts first
    VL_CUDA(cudaMemcpyAsync(c->h_lmm, c->lmm, sizeof(LmScalars), cudaMemcpyDeviceToHost, c->stream));
    VL_CUDA(cudaStreamSynchronize(c->stream));
    Qc = c->h_lmm->Qc; Qs = c->h_lmm->Qs;
    VL_TRY(vl_reserve(c, c->knnKey, (size_t)nqBound * 5));
    VL_TRY(vl_reserve(c, d->knnIds, (size_t)nqBound * 5));
  }
  for (int pass = 0; pass < 2; ++pass) {  // LM.cpp:526
    VL_BYTES(16.0 * (double)max(c->h_lmm->Qc + c->h_lmm->Qs, 1) * 6);  // query + 5 neighbours (SURVEY 8d), last known Qc + Qs
    VL_LAUNCH(lg_knn, c->num_sms * 8, 256, 0, c->lmm, d->grid, c->stackC.p, c->stackS.p, c->knnPts.p, c->knnD2.p, capture ? c->knnKey.p : (unsigned long long*)nullptr);
    VL_BYTES((16.0 * 6 + 24.0 + 84.0) * (double)max(c->h_lmm->Qc + c->h_lmm->Qs, 1));
    VL_LAUNCH(lm_fit, c->num_sms, 128, 0, c->lmm, c->stackC.p, c->stackS.p, c->knnPts.p, c->knnD2.p, c->knnOk.p, c->factors.p, c->factorValid.p);
    if (pass == 0 && afterHead) VL_TRY(afterHead());
    if (capture) {
      const int nq = Qc + Qs;
      if (nq > 0) VL_LAUNCH(lg_keys_to_ids, vl_div_up(nq * 5, 256), 256, 0, c->knnKey.p, nq * 5, Qc, d->subReal, c->lmm, c->prm, c->cubeC, c->cubeS, c->poolC.p, c->poolS.p, d->knnIds.p);
      for (int kind = 0; kind < 2; ++kind) {
        const int n = kind ? Qs : Qc, off = kind ? Qc : 0;
        VL_TRY(vl_reserve(c, c->dbgKnnIdx[pass][kind], (size_t)max(n, 1) * 5));
        VL_TRY(vl_reserve(c, c->dbgKnnD2[pass][kind], (size_t)max(n, 1) * 5));
        VL_TRY(vl_reserve(c, c->dbgKnnOk[pass][kind], (size_t)max(n, 1)));
        if (n == 0) continue;
        VL_CUDA(cudaMemcpyAsync(c->dbgKnnIdx[pass][kind].p, d->knnIds.p + (size_t)off * 5, sizeof(int) * 5 * n, cudaMemcpyDeviceToDevice, c->stream));
        VL_CUDA(cudaMemcpyAsync(c->dbgKnnD2[pass][kind].p, c->knnD2.p + (size_t)off * 5, sizeof(float) * 5 * n, cudaMemcpyDeviceToDevice, c->stream));
        VL_CUDA(cudaMemcpyAsync(c->dbgKnnOk[pass][kind].p, c->knnOk.p + off, sizeof(int) * n, cudaMemcpyDeviceToDevice, c->stream));
      }
    }
    VL_TRY(vl_solve(c, nqBound, &d->work->nq, c->lmm->pose, capture ? &c->dbgLmCost[pass * 2] : nullptr, c->h_lmm->Qc + c->h_lmm->Qs));
    if (c->timing && pass == 0) VL_CUDA(cudaEventRecord(c->evx[2], c->stream));
  }
  // in-place path: the pose is final HERE -- the map update (own stream) does not wait for transformUpdate
  if (earlyPose) { VL_CUDA(cudaEventRecord(c->evPose, c->stream)); c->s2seq++; }
  VL_LAUNCH(lm_transform_update, 1, 32, 0, c->lmm, (const LgHeader*)(earlyPose ? nullptr : d->grid.hdr), (const int*)d->grid.top, losPub,
            earlyPose ? c->h_lmm : (LmScalars*)nullptr, earlyPose ? c->h_los : (LoScalars*)nullptr, (volatile unsigned*)c->h_s2flag, c->s2seq);  // LM.cpp:737 (runs even when the optimisation was skipped)
  return VLOAM_OK;
}

// sync point S2: the pose is final; sizes for the map update.  While the device finishes this sweep's mapping, the next sweep's
// odometry solve is queued (replays with a registered look-ahead sweep) -- once per call of vl_lm_run.
static int lm_sync_s2(vloam_b200_ctx* c, bool capture, bool* lookaheadDone, bool published = false) {
  if (c->sideSubmitted) { c->sideSubmitted = false; VL_TRY(vl_lm_join(c)); }  // (see vl_lm_run: the helper must be done with the context's fields)
  if (!published) {
    VL_CUDA(cudaEventRecord(c->evPose, c->stream));
    VL_CUDA(cudaMemcpyAsync(c->h_los, c->los, sizeof(LoScalars), cudaMemcpyDeviceToHost, c->stream));
    VL_CUDA(cudaMemcpyAsync(c->h_lmm, c->lmm, sizeof(LmScalars), cudaMemcpyDeviceToHost, c->stream));
  }
  VL_CUDA(cudaEventRecord(c->evS2, c->stream));
  VL_HOST_MARK(5);
  if (!*lookaheadDone) {
    VL_TRY(vl_lo_flush_deferred(c));
    if (!capture) VL_TRY(vl_lo_lookahead_solve(c));
    *lookaheadDone = true;
  }
  if (!capture) VL_TRY(vl_lo_lookahead_stacks(c));  // (no-op unless a look-ahead solve was queued in this call)
  if (published) {
    // lm_transform_update wrote both structs and then this sweep's sequence number into pinned memory: spin on the word; the
    // event is looked at now and then so that a failed launch cannot hang the caller
    volatile unsigned* flag = c->h_s2flag;
    for (unsigned spin = 1; *flag != c->s2seq; ++spin) {
      if ((spin & 1023u) == 0) {
        const cudaError_t e = cudaEventQuery(c->evS2);
        if (e == cudaSuccess) break;  // (complete: its writes are visible)
        if (e != cudaErrorNotReady) { snprintf(c->err, sizeof c->err, "%s:%d S2: %s", __FILE__, __LINE__, cudaGetErrorString(e)); return VLOAM_E_CUDA; }
        (void)cudaGetLastError();
      }
#if defined(__x86_64__)
      __builtin_ia32_pause();
#endif
    }
    __atomic_thread_fence(__ATOMIC_ACQUIRE);
  } else VL_CUDA(cudaEventSynchronize(c->evS2));
  c->s2Done = true;
  VL_HOST_MARK(6);
  if (c->h_lmm->overflow) { snprintf(c->err, sizeof c->err, "map pool exhausted"); return VLOAM_E_CAPACITY; }
  return VLOAM_OK;
}

// The in-place path: the grid describes this sweep's sub-map unless lm_prepare_fast finds the window moved or the grid dirty.  The
// passes and the in-place map update are queued, then the host waits at S2 and updates its bounds.  *fellBack: lm_prepare_fast raised
// needSlow -- nothing of this sweep's mapping was applied (every kernel returned at once) and the caller repeats it on the pool path.
static int lm_run_in_place(vloam_b200_ctx* c, LmDevice* d, const LoScalars* lo, int nqBound, int resetValid, bool inlineUpdate, bool* fellBack) {
  *fellBack = false;
  bool lookaheadDone = false;
  // stacks filtered a sweep ago (look-ahead): the counts are set by lm_prepare_fast itself, one launch fewer on the pose chain
  const bool countsSet = c->stacksAdopted;
  // the odometry state S2 hands to the host (h_los) is always the context's own, also when `lo` is the caller's pose
  const LoScalars* const losNow = c->los;  // (read before the helper thread may swap the odometry states)
  if (countsSet) {
    VL_CUDA(cudaStreamWaitEvent(c->stream, c->evStacks, 0));
    VL_CUDA(cudaStreamWaitEvent(c->stream, c->evStacksC, 0));
    VL_LAUNCH(lm_prepare_fast, 1, 256, 0, c->lmm, lo, d->work, d->grid.hdr, 0, resetValid, (const int*)(d->dQ + 2 * c->stackSel),
              (const int*)(d->dQ + 2 * c->stackSel + 1), (const int*)d->grid.top);
  } else {
    VL_LAUNCH(lm_prepare_fast, 1, 256, 0, c->lmm, lo, d->work, d->grid.hdr, 0, resetValid, (const int*)nullptr, (const int*)nullptr, (const int*)nullptr);
  }
  if (c->timing) VL_CUDA(cudaEventRecord(c->evx[0], c->stream));
  VL_HOST_MARK(8);
  if (!countsSet) {
    VL_CUDA(cudaStreamWaitEvent(c->stream, c->evStacks, 0));   // only now are this frame's downsampled stacks needed (side streams)
    VL_CUDA(cudaStreamWaitEvent(c->stream, c->evStacksC, 0));
    VL_LAUNCH(lm_set_counts, 1, 32, 0, c->lmm, d->work, d->dQ + 2 * c->stackSel, d->dQ + 2 * c->stackSel + 1, (const LgHeader*)d->grid.hdr,
              (const int*)d->grid.top);
  }
  // The helper thread issues the next sweep's odometry (two sweeps ahead, structures pre-built), the look-ahead scan registration
  // and the next odometry structures while the caller queues the rest of the mapping stage.  It swaps scan-registration sets and the
  // odometry state in and out of the context while it does: it is handed the work only after the launch above has read c->los
  // (and, to keep the head of the pose chain short, after the first kNN + fit are queued) and joined before lm_sync_s2 reads it again.
  auto sideWork = [&]() -> int {
    VL_HOST_MARK(9);
    VL_TRY(vl_lo_early_lookahead(c, &lookaheadDone));
    VL_TRY(vl_lo_plan_prebuild(c));
    const int rs = vl_lo_submit_side(c);
    VL_HOST_MARK(10);
    return rs;
  };
  VL_TRY(lm_queue_passes(c, d, nqBound, false, losNow, inlineUpdate ? std::function<int()>() : std::function<int()>(sideWork)));
  VL_HOST_MARK(11);
  // The in-place map update is queued NOW, behind the pose (evPose) on its own stream, before the host waits at S2: its kernels
  // read the counts and the needSlow flag on the device (sizes here are bounds), so the device runs it the moment the pose is
  // final instead of waiting for S2 -> host -> helper thread -> launch (~45 us on the chain the next sweep's mapping waits for).
  // the next sweep's odometry solve goes to its own stream first: its inputs are ready long before this sweep's pose is
  if (!lookaheadDone) {
    VL_TRY(vl_lo_flush_deferred(c));
    VL_TRY(vl_lo_lookahead_solve(c));
    lookaheadDone = true;
  }
  // (points outside the window are appended raw to their cubes' pool segments: room for them is checked BEFORE the append is queued,
  // with the bound, against the pool top of the last S2)
  if (d->mapUpdate) VL_TRY(lm_pool_headroom(c, 0, 0, nqBound, nqBound));
  if (!d->mapUpdate) {  // frozen map: no insert, no re-filter, no raw append -- the update's events are recorded behind the pose all the same
    vl_tls_stream = c->stream3;
    struct Restore { ~Restore() { vl_tls_stream = nullptr; } } restore;
    VL_CUDA(cudaStreamWaitEvent(c->stream3, c->evAux, 0));  // (a previous sweep's raw appends: evAux keeps covering them)
    VL_CUDA(cudaStreamWaitEvent(c->stream3, c->evPose, 0));
    VL_CUDA(cudaEventRecord(c->evKeys, c->stream3));
    VL_CUDA(cudaEventRecord(c->evKeysSel[c->stackSel], c->stream3));
    VL_CUDA(cudaEventRecord(c->evUpd, c->stream3));
    VL_CUDA(cudaEventRecord(c->evAux, c->stream3));
    VL_CUDA(cudaEventRecord(c->evMap, c->stream3));
    if (c->timing) VL_CUDA(cudaEventRecord(c->evx[7], c->stream3));
  } else {
    const int nq = nqBound;
    const float4* const stackCp = c->stackC.p; const float4* const stackSp = c->stackS.p;
    vl_tls_stream = c->stream3;
    struct Restore { ~Restore() { vl_tls_stream = nullptr; } } restore;
    int H = 1024; while (H < 4 * nq) H <<= 1;
    VL_TRY(vl_reserve(c, d->newPts, (size_t)nq));
    VL_TRY(vl_reserve(c, d->newCube, (size_t)nq));
    VL_TRY(vl_reserve(c, d->muKey, (size_t)H));
    VL_TRY(vl_reserve(c, d->muInt, (size_t)H * (1 + MU_CAP) + (size_t)nq * 3 + 4));
    MuWork mw;
    mw.hkey = d->muKey.p; mw.H = H; mw.cnt = d->muInt.p; mw.anyOutside = mw.cnt + H; mw.slotOf = mw.anyOutside + 4; mw.found = mw.slotOf + nq;
    mw.foundCell = mw.found + nq; mw.members = mw.foundCell + nq;
    // (the scratch is cleared behind the previous update, on its stream, BEFORE the wait for this sweep's pose: off the chain)
    VL_CUDA(cudaStreamWaitEvent(c->stream3, c->evAux, 0));                // (anyOutside is read by the previous sweep's append on streamAux)
    // a map publication queued since the last update reads the grid and the pools that mu_apply and rf_append_outside (behind evUpd) edit
    VL_CUDA(cudaStreamWaitEvent(c->stream3, d->evPub, 0));
    VL_CUDA(cudaMemsetAsync(mw.hkey, 0xff, (size_t)H * 8, c->stream3));   // empty slots
    VL_CUDA(cudaMemsetAsync(mw.cnt, 0, (size_t)(H + 4) * 4, c->stream3));  // group sizes and the anyOutside flag behind them
    VL_CUDA(cudaStreamWaitEvent(c->stream3, c->evPose, 0));
    VL_BYTES(16.0 * max(c->h_lmm->Qc + c->h_lmm->Qs, 1));  // SURVEY 8(d) B_lm insert term: every new point once (last known count)
    VL_LAUNCH(mu_keys, vl_div_up(nq, 256), 256, 0, c->lmm, d->work, c->prm, d->grid, stackCp, stackSp, d->newPts.p, d->newCube.p, mw);
    VL_CUDA(cudaEventRecord(c->evKeys, c->stream3));  // nothing below reads the stacks any more: the next sweep's filters may overwrite them
    VL_CUDA(cudaEventRecord(c->evKeysSel[c->stackSel], c->stream3));
    // points outside the 5x5x3 window go to cubes the grid does not hold: appended raw to their pool segments beside the in-place update
    VL_CUDA(cudaEventRecord(c->evUpd, c->stream3));
    VL_CUDA(cudaStreamWaitEvent(c->streamAux, c->evUpd, 0));
    vl_tls_stream = c->streamAux;
    VL_LAUNCH(rf_append_outside, 1, 1024, 0, c->lmm, d->newPts.p, d->newCube.p, c->cubeC, c->cubeS, c->poolC.p, c->poolS.p, (int)c->poolC.cap,
              (int)c->poolS.cap, (const int*)mw.anyOutside);
    vl_tls_stream = c->stream3;
    VL_CUDA(cudaEventRecord(c->evAux, c->streamAux));
    VL_BYTES(2.0 * 32.0 * max(c->h_lmm->Qc + c->h_lmm->Qs, 1));  // read + write of the map points that change (SURVEY 8(d) re-filter term restricted to what changes)
    VL_LAUNCH(mu_apply, vl_div_up(nq, 128), 128, 0, c->lmm, c->prm, d->grid, d->newPts.p, mw);
    VL_CUDA(cudaEventRecord(c->evMap, c->stream3));
    if (c->timing) VL_CUDA(cudaEventRecord(c->evx[7], c->stream3));
  }
  VL_HOST_MARK(12);
  VL_TRY(lm_sync_s2(c, false, &lookaheadDone, true));
  VL_HOST_MARK(13);
  if (c->h_lmm->needSlow) { *fellBack = true; return VLOAM_OK; }
  const int Qc = c->h_lmm->Qc, Qs = c->h_lmm->Qs, nq = Qc + Qs;
  if (d->builtCount < 0) {  // first in-place sweep after a rebuild: nothing created yet
    d->builtCount = c->h_lmm->gridCount; d->builtCountC = c->h_lmm->gridCountC;
    d->baseC = d->hMapUpperC; d->baseS = d->hMapUpperS; d->outBaseC = c->h_lmm->outsideC; d->outBaseS = c->h_lmm->outsideS;
  }
  c->lm_optimized = c->h_lmm->optimized;
  if (d->mapUpdate) {  // (a frozen map grows no bound)
    d->gridTopUpper = (long long)c->h_lmm->gridTop + nq;  // chunks in use before this update + at most one new chunk per new voxel
    // map size after this update <= size at the build + voxels created in the grid + raw appends outside the window (device counts
    // at this S2: everything up to the previous update) + this sweep's points.  (Adding Qc + Qs per sweep drifts by ~15k points a
    // sweep -- most of them merge into existing voxels -- and made the next window move regrow the grid and the merge buffers.)
    d->hMapUpperC = d->baseC + (c->h_lmm->gridCountC - d->builtCountC) + (c->h_lmm->outsideC - d->outBaseC) + Qc;
    d->hMapUpperS = d->baseS + ((c->h_lmm->gridCount - c->h_lmm->gridCountC) - (d->builtCount - d->builtCountC)) + (c->h_lmm->outsideS - d->outBaseS) + Qs;
    d->newVoxUpper = (long long)c->h_lmm->gridCount - d->builtCount + nq;  // voxels created so far (device count at S2) + at most nq by this update
    if (nq > 0) d->poolsStale = true;
  }
  d->paths[0]++;
  c->lm_frameCount++;
  VL_HOST_MARK(7);
  VL_CUDA(cudaGetLastError());
  return VLOAM_OK;
}

// What the pool path's map update takes from sync point S2 (the next sweep may swap the stack buffers while the helper issues it).
struct LmPoolUpdate {
  int tailTotal;                      // unsorted tail points of the valid cubes
  int Qc, Qs, Mc, Ms;                 // this sweep's stacks and sub-map
  long long totalC, totalS;           // points in all cubes before the update
  const float4* stackC; const float4* stackS; int stackSel;
  bool rebuildAfter;                  // rebuild the grid behind the update (in-place path next sweep)
  bool update;                        // LmDevice::mapUpdate when the sweep was mapped
};

// ---- map update (LM.cpp:741-808) of the pool path on stream3: the caller reads the pose, and the next frame's scan registration +
// odometry start, while the map is brought up to date.
static int lm_pool_update(vloam_b200_ctx* c, LmDevice* d, const LmPoolUpdate& u) {
  vl_tls_stream = c->stream3;  // every launch helper below issues on the update's stream, whichever thread runs this
  struct Restore { ~Restore() { vl_tls_stream = nullptr; } } restore;
  VL_CUDA(cudaStreamWaitEvent(c->stream3, c->evPose, 0));
  const int nq = u.Qc + u.Qs, nKeys = u.tailTotal + nq;
  if (!u.update) {  // frozen map: no insert, no re-filter, no raw append (the window roll of lm_prepare still cleared what left the grid)
    VL_CUDA(cudaEventRecord(c->evKeys, c->stream3));
    VL_CUDA(cudaEventRecord(c->evKeysSel[u.stackSel], c->stream3));
  } else if (nKeys > 0) {
    VL_TRY(lm_reserve_merge(c, d, nKeys, max(nq, 1), (long long)u.Mc + u.Ms));
    VL_LAUNCH(rf_keys, vl_div_up(nKeys, 256), 256, 0, c->lmm, d->work, c->prm, c->cubeC, c->cubeS, c->poolC.p, c->poolS.p, u.stackC, u.stackS,
              d->newPts.p, d->newCube.p, c->tailKeys.p, nKeys);
    VL_CUDA(cudaEventRecord(c->evKeys, c->stream3));  // nothing below reads the stacks any more: the next sweep's filters may overwrite them
    VL_CUDA(cudaEventRecord(c->evKeysSel[u.stackSel], c->stream3));
    VL_TRY(lm_queue_merge(c, d, nKeys, (double)u.Mc + u.Ms, (double)u.Mc + u.Ms + nq));  // (read every prefix point once, write it once to staging; staging -> pool copy)
    if (nq > 0) {
      // Points that fell outside the 5x5x3 window go to cubes the sub-map never reads: this single-CTA
      // kernel (~20 us) runs beside the grid rebuild; the next solveMapping waits on both (evMap, evAux).
      VL_CUDA(cudaEventRecord(c->evUpd, c->stream3));
      VL_CUDA(cudaStreamWaitEvent(c->streamAux, c->evUpd, 0));
      vl_tls_stream = c->streamAux;
      VL_LAUNCH(rf_append_outside, 1, 1024, 0, c->lmm, d->newPts.p, d->newCube.p, c->cubeC, c->cubeS, c->poolC.p, c->poolS.p, (int)c->poolC.cap,
                (int)c->poolS.cap, (const int*)nullptr);
      vl_tls_stream = c->stream3;
    }
  }
  VL_CUDA(cudaEventRecord(c->evAux, c->streamAux));
  // the map after this frame's update holds at most the points it held before plus this frame's inserts
  d->hMapUpperC = u.totalC + (u.update ? u.Qc : 0); d->hMapUpperS = u.totalS + (u.update ? u.Qs : 0);
  // ---- the grid of the NEXT sweep: rebuilt here, behind the update on its side stream, for the window this sweep used (a cube
  // is 50 m wide, so the next sweep almost always uses the same one and runs the in-place path; lm_prepare_fast checks).
  // Debug snapshots keep the pool path every sweep.
  if (u.rebuildAfter) {
    VL_LAUNCH(lm_spec_prepare, 1, 256, 0, d->subReal, c->cubeC, c->cubeS, d->subSpec);
    VL_TRY(lg_rebuild_launch(c, d, d->subSpec, d->hMapUpperC + d->hMapUpperS));
    d->gridValid = true;
  }
  VL_CUDA(cudaEventRecord(c->evMap, c->stream3));
  return VLOAM_OK;
}

// The pool path (round 1's): cube tables, sorted pools; the grid is rebuilt for the window lm_prepare finds.  lookaheadDone: the
// in-place path fell back after its sync point S2 had already queued the next sweep's odometry.
static int lm_run_pool(vloam_b200_ctx* c, LmDevice* d, const LoScalars* lo, int nqBound, int resetValid, bool capture, bool inlineUpdate,
                       bool lookaheadDone) {
  VL_CUDA(cudaStreamWaitEvent(c->stream, c->evAux, 0));  // (the previous sweep's raw appends outside the window edit the cube tables)
  // a map publication queued since the last update: lm_prepare rolls the cube tables it reads, and this stream's evPose orders the
  // update, the speculative rebuild and the appends (stream3, streamAux) behind it as well
  VL_CUDA(cudaStreamWaitEvent(c->stream, d->evPub, 0));
  if (d->poolsStale) VL_TRY(lm_materialize(c, d));  // the in-place updates since the last pool-path sweep, written back first (main stream)
  d->paths[1]++;
  VL_LAUNCH(lm_prepare, 1, 1024, 0, c->lmm, lo, c->cubeC, c->cubeS, d->work, 0, resetValid, d->subReal);
  const long long totalBound = d->hMapUpperC + d->hMapUpperS;
  if (d->gridEnabled) VL_TRY(lm_reserve_merge(c, d, LG_NEWVOX_MAX, LG_NEWVOX_MAX, totalBound, false));
  VL_TRY(lg_rebuild_launch(c, d, d->subReal, totalBound));
  if (c->timing) VL_CUDA(cudaEventRecord(c->evx[0], c->stream));
  if (capture) {  // the debug getters read the concatenated sub-map clouds (LM.cpp:476-485)
    VL_TRY(vl_reserve(c, c->fromMapC, (size_t)max(d->hMapUpperC, 1LL), false, (size_t)d->hMapUpperC / 2 + (1 << 20)));
    VL_TRY(vl_reserve(c, c->fromMapS, (size_t)max(d->hMapUpperS, 1LL), false, (size_t)d->hMapUpperS / 2 + (1 << 20)));
    VL_LAUNCH(lm_gather, c->num_sms * 8, 256, 0, d->subReal, c->cubeC, c->cubeS, c->poolC.p, c->poolS.p, c->fromMapC.p, c->fromMapS.p);
  }
  VL_CUDA(cudaStreamWaitEvent(c->stream, c->evStacks, 0));   // only now are this frame's downsampled stacks needed (side streams)
  VL_CUDA(cudaStreamWaitEvent(c->stream, c->evStacksC, 0));
  VL_LAUNCH(lm_set_counts, 1, 32, 0, c->lmm, d->work, d->dQ + 2 * c->stackSel, d->dQ + 2 * c->stackSel + 1, (const LgHeader*)nullptr, (const int*)d->grid.top);
  VL_TRY(lm_queue_passes(c, d, nqBound, capture, nullptr));
  VL_TRY(lm_sync_s2(c, capture, &lookaheadDone));
  const LmScalars* h = c->h_lmm;
  // the previous update is complete (this stream waited on evMap), the next one has not been issued, and a pool copy keeps every cube's offset valid
  VL_TRY(lm_pool_headroom(c, h->totalC, h->totalS, h->Qc, h->Qs));
  c->lm_optimized = h->optimized;
  const LmPoolUpdate u = {h->tailC + h->tailS, h->Qc, h->Qs, h->Mc, h->Ms, h->totalC, h->totalS, c->stackC.p, c->stackS.p, c->stackSel,
                          d->gridEnabled && !capture, d->mapUpdate};
  d->gridValid = false;
  c->lm_frameCount++;
  // otherwise the helper thread issues the update while the caller returns with its pose (whoever needs the map next joins it first: vl_lm_join)
  if (inlineUpdate) VL_TRY(lm_pool_update(c, d, u));
  else VL_TRY(lm_submit(c, [c, d, u]() -> int { return lm_pool_update(c, d, u); }));
  VL_HOST_MARK(7);
  VL_CUDA(cudaGetLastError());
  return VLOAM_OK;
}

int vl_lm_run(vloam_b200_ctx* c, const VlLmInput& in) {
  LmDevice* d = c->lm;
  VL_HOST_MARK(3);
  VL_TRY(vl_lm_join(c));  // the previous frame's map update has been issued (evMap recorded, host bounds updated)
  VL_HOST_MARK(4);
  const int resetValid = c->lm_reset_pending ? 1 : 0;
  c->lm_reset_pending = false;
  VL_CUDA(cudaStreamWaitEvent(c->stream, c->evMap, 0));  // the previous frame's map update (stream3) must be complete
  // ... its raw appends to cubes OUTSIDE the window (streamAux) touch pool segments only: nothing of the in-place path reads them
  // (a single CTA that takes 20-60 us when the sensor nears a window edge: it used to sit on the next sweep's pose chain);
  // the pool path waits for them before it reads the cube tables.
  if (in.skip) {  // LM.cpp:197-201: only the high-frequency pose is propagated
    c->rlReady = false;
    if (in.caller) c->stacksReady = false;  // (stacks this sweep's odometry may have filtered are not used)
    VL_LAUNCH(lm_prepare_fast, 1, 256, 0, c->lmm, in.los, d->work, d->grid.hdr, 1, resetValid, (const int*)nullptr, (const int*)nullptr, (const int*)nullptr);
    VL_TRY(vl_lo_flush_deferred(c)); VL_CUDA(cudaGetLastError());
    return VLOAM_OK;
  }
  if (in.caller) {  // filtered again from the caller's clouds into the pair the update reads, on the same side streams as any first filter
    VL_TRY(vl_lm_enqueue_stacks(c, in.corner, in.nc, in.surf, in.ns, false, false));
  } else if (!c->stacksReady) {  // laser_mapping called without this frame's laser_odometry having queued them
    VL_CUDA(cudaStreamSynchronize(c->stream));
    VL_TRY(vl_lm_enqueue_stacks(c, in.corner, in.nc, in.surf, in.ns));
  }
  c->stacksReady = false;
  const bool capture = vl_debug_capture(c);
  const int nqBound = max(in.nc + in.ns, 1);  // a voxel filter never grows a cloud
  VL_TRY(vl_reserve(c, c->knnPts, (size_t)nqBound * 5));
  VL_TRY(vl_reserve(c, c->knnD2, (size_t)nqBound * 5));
  VL_TRY(vl_reserve(c, c->knnOk, (size_t)nqBound));
  VL_TRY(vl_reserve(c, c->factors, (size_t)nqBound * 10));
  VL_TRY(vl_reserve(c, c->factorValid, (size_t)nqBound));
  const bool inlineUpdate = d->noWorker || capture || c->prof_name[0];  // profiling and debug snapshots serialise everything
  bool fellBack = false;
  c->rlReady = true;
  if (d->gridEnabled && d->gridValid && !capture && d->gridTopUpper + 2LL * nqBound <= d->grid.cap && d->newVoxUpper + nqBound <= LG_NEWVOX_MAX) {
    VL_TRY(lm_run_in_place(c, d, in.los, nqBound, resetValid, inlineUpdate, &fellBack));
    if (!fellBack) return VLOAM_OK;
  }
  return lm_run_pool(c, d, in.los, nqBound, resetValid, capture, inlineUpdate, fellBack);
}

// LM.cpp:901-905 (LaserMapping::publish): laserCloudFullRes through pointAssociateToMap.  lo != nullptr
// (VLOAM_FLAG_TRANSFORM_TO_END): laserCloudFullRes is the end-frame cloud LaserOdometry hands over, TransformToEnd with
// lo = {q_last_curr, t_last_curr} of this sweep (LO.cpp:537-556), stored as float before the map transform.
__global__ void __launch_bounds__(256) lm_register_full(const float4* __restrict__ in, int n, const LmScalars* __restrict__ s, int skip,
                                                        float4* __restrict__ out, const double* __restrict__ lo, int deskew) {
  VL_PDL_WAIT();

  const double* q = skip ? s->q_hf : s->pose;
  const double* t = skip ? s->t_hf : s->pose + 4;
  const double pose[7] = {q[0], q[1], q[2], q[3], t[0], t[1], t[2]};
  double L[7] = {0, 0, 0, 1, 0, 0, 0};
  if (lo) for (int k = 0; k < 7; ++k) L[k] = lo[k];
  for (int g = blockIdx.x * blockDim.x + threadIdx.x; g < n; g += gridDim.x * blockDim.x) {
    const float4 p = lo ? vl_transform_to_end(L, in[g], deskew) : in[g];
    double r[3];
    vl_qrot(pose, (double)p.x, (double)p.y, (double)p.z, r);  // LM.cpp:154-164
    out[g] = make_float4((float)(r[0] + pose[4]), (float)(r[1] + pose[5]), (float)(r[2] + pose[6]), p.w);
  }
}

int vl_lm_register_full(vloam_b200_ctx* c, const float4* d_in, int n, float4* d_out, int skip, bool toEnd) {
  VL_BYTES(32.0 * n);
  // (c->los is this sweep's odometry state: a look-ahead solve of the next sweep writes the spare state, losNext)
  VL_LAUNCH(lm_register_full, c->num_sms * 4, 256, 0, d_in, n, c->lmm, skip, d_out, toEnd ? (const double*)c->los->para_q : (const double*)nullptr,
            vl_distortion(c) ? 1 : 0);
  VL_CUDA(cudaGetLastError());
  return VLOAM_OK;
}

int vl_lm_rescan_sorted(vloam_b200_ctx* c) {
  c->lm->gridValid = false;  // the state behind the grid was edited from outside
  VL_LAUNCH(lm_scan_sorted, VL_CUBE_NUM, 256, 0, c->lmm, c->prm, c->cubeC, c->poolC.p, 0);
  VL_LAUNCH(lm_scan_sorted, VL_CUBE_NUM, 256, 0, c->lmm, c->prm, c->cubeS, c->poolS.p, 1);
  VL_CUDA(cudaStreamSynchronize(c->stream));
  return VLOAM_OK;
}

// blob = int32 counts[4851] followed by the points of all cubes in cube-index order
int vl_lm_export_map(vloam_b200_ctx* c, int which, void* out, long cap, long* bytes) {
  VL_TRY(vl_lm_sync_pools(c));  // in-place grid updates leave the valid cubes' pools behind: write them back first
  MapCubeTable h;
  VL_CUDA(cudaStreamSynchronize(c->stream));
  VL_CUDA(cudaMemcpy(&h, which ? c->cubeS : c->cubeC, sizeof h, cudaMemcpyDeviceToHost));
  long total = 0;
  for (int i = 0; i < VL_CUBE_NUM; ++i) total += h.count[i];
  *bytes = (long)VL_CUBE_NUM * 4 + total * 16;
  if (!out || cap < *bytes) return VLOAM_OK;
  memcpy(out, h.count, (size_t)VL_CUBE_NUM * 4);
  char* p = (char*)out + (size_t)VL_CUBE_NUM * 4;
  const float4* pool = which ? c->poolS.p : c->poolC.p;
  for (int i = 0; i < VL_CUBE_NUM; ++i) {
    if (h.count[i] == 0) continue;
    VL_CUDA(cudaMemcpy(p, pool + h.start[i], (size_t)h.count[i] * 16, cudaMemcpyDeviceToHost));
    p += (size_t)h.count[i] * 16;
  }
  return VLOAM_OK;
}

// The map is replaced from outside (a debug import, vloam_b200_load_map): the helper thread has issued the last update and the last
// publication has finished reading the old map; the grid is rebuilt by the next mapped sweep (pool path), the pools are no longer
// behind it, and the host bounds restart from the new contents (the caller sets hMapUpper*).
static int lm_map_replaced(vloam_b200_ctx* c) {
  LmDevice* d = c->lm;
  VL_TRY(vl_lm_join(c));
  VL_TRY(vl_lm_pub_sync(c));
  d->gridValid = false; d->poolsStale = false;
  d->newVoxUpper = 0; d->gridTopUpper = 0;
  c->rlReady = false;  // (the stacks belong to a sweep mapped in the old map)
  return VLOAM_OK;
}

int vl_lm_import_map(vloam_b200_ctx* c, int which, const void* data, long bytes) {
  LmDevice* d = c->lm;
  if (bytes < (long)VL_CUBE_NUM * 4) { snprintf(c->err, sizeof c->err, "map blob too short"); return VLOAM_E_INVALID; }
  const int* counts = (const int*)data;
  long long total = 0;
  for (int i = 0; i < VL_CUBE_NUM; ++i) total += counts[i];
  if (bytes != (long)VL_CUBE_NUM * 4 + total * 16) { snprintf(c->err, sizeof c->err, "map blob size mismatch"); return VLOAM_E_INVALID; }
  VL_TRY(lm_map_replaced(c));
  DBuf<float4>& pool = which ? c->poolS : c->poolC;
  // fresh layout: every cube gets 25 % head room (at least 256 points)
  MapCubeTable h;
  memset(&h, 0, sizeof h);
  long long top = 0;
  for (int i = 0; i < VL_CUBE_NUM; ++i) {
    if (counts[i] == 0) continue;
    h.start[i] = (int)top; h.count[i] = counts[i]; h.cap[i] = counts[i] + counts[i] / 4 + 256;
    top += h.cap[i];
  }
  VL_CUDA(cudaStreamSynchronize(c->stream));
  if ((size_t)top * 2 > pool.cap) VL_TRY(vl_reserve(c, pool, (size_t)top * 2));  // (contents are replaced below)
  const char* p = (const char*)data + (size_t)VL_CUBE_NUM * 4;
  for (int i = 0; i < VL_CUBE_NUM; ++i) {
    if (counts[i] == 0) continue;
    VL_CUDA(cudaMemcpy(pool.p + h.start[i], p, (size_t)counts[i] * 16, cudaMemcpyHostToDevice));
    p += (size_t)counts[i] * 16;
  }
  MapCubeTable* dt = which ? c->cubeS : c->cubeC;
  VL_CUDA(cudaMemcpy(dt, &h, sizeof h, cudaMemcpyHostToDevice));
  LmScalars hs;
  VL_CUDA(cudaMemcpy(&hs, c->lmm, sizeof hs, cudaMemcpyDeviceToHost));
  if (which) hs.poolTopS = (int)top; else hs.poolTopC = (int)top;
  VL_CUDA(cudaMemcpy(c->lmm, &hs, sizeof hs, cudaMemcpyHostToDevice));
  VL_LAUNCH(lm_scan_sorted, VL_CUBE_NUM, 256, 0, c->lmm, c->prm, dt, pool.p, which);
  VL_CUDA(cudaStreamSynchronize(c->stream));
  if (which) d->hMapUpperS = total; else d->hMapUpperC = total;
  return VLOAM_OK;
}

// LaserMapping::publish (LM.cpp:884-899): queue the assembly of laserCloudMap on the publication stream, behind the last map
// update (evMap) and its raw appends (evAux).  The host does not wait; every later edit of the map waits for evPub on the device
// (vl_lm_run, lm_materialize), and the host waits for it before it replaces a buffer the assembly reads (lm_pool_headroom,
// lg_reserve, vl_lm_pub_sync before imports and destroy).
int vl_lm_publish_map(vloam_b200_ctx* c) {
  LmDevice* d = c->lm;
  VL_TRY(vl_lm_join(c));  // the helper thread has issued the last update (evMap, evAux recorded; poolsStale / newVoxUpper / hMapUpper* current)
  struct Restore { cudaStream_t prev; ~Restore() { vl_tls_stream = prev; } } restore{vl_tls_stream};
  vl_tls_stream = d->pubStream;
  const bool fromGrid = d->poolsStale;
  const long long bound = d->hMapUpperC + d->hMapUpperS;
  // buffers first, while this stream holds nothing but earlier publications: a regrow syncs the stream, and behind the waits
  // below that would make the host wait for the map update in flight
  VL_TRY(vl_reserve(c, d->pubOut, (size_t)max(bound, 1LL), false, (size_t)bound / 2 + (1 << 20)));
  if (fromGrid) {
    VL_TRY(vl_reserve(c, d->pubKeys, (size_t)4 * LG_NEWVOX_MAX));  // sized once for the largest bound: [0, N) unsorted | [N, 2N) sorted | [2N, 4N) scratch
    VL_TRY(vl_reserve(c, d->pubEnt, (size_t)LG_NEWVOX_MAX));
  }
  VL_CUDA(cudaStreamWaitEvent(d->pubStream, c->evMap, 0));
  VL_CUDA(cudaStreamWaitEvent(d->pubStream, c->evAux, 0));
  d->pubOutCap = (long long)d->pubOut.cap;
  const int gsGrid = c->num_sms * 8;
  const int outCap = (int)min(d->pubOutCap, (long long)INT_MAX);
  int* pub = d->pubInt;
  VL_CUDA(cudaMemsetAsync(d->pubWork, 0, sizeof(RfWork), d->pubStream));
  VL_CUDA(cudaMemsetAsync(pub + MP_CNT, 0, sizeof(int), d->pubStream));
  const int P = fromGrid ? (int)max(min(d->newVoxUpper, (long long)LG_NEWVOX_MAX), 1LL) : 0;
  const size_t N = lm_merge_stride(P);
  unsigned long long* keysIn = nullptr; unsigned long long* keysSorted = nullptr;
  if (fromGrid) {
    keysIn = d->pubKeys.p; keysSorted = d->pubKeys.p + N;
    VL_CUDA(cudaMemsetAsync(keysIn, 0xff, N * sizeof(unsigned long long), d->pubStream));
    VL_BYTES(16.0 * LM_NCELL + 12.0 * bound);
    VL_LAUNCH(mp_collect, gsGrid, 256, 0, d->grid, d->pubWork, keysIn, d->pubEnt.p, pub + MP_CNT, P);
    VL_LAUNCH(rf_seg_scatter, vl_div_up(P, 256), 256, 0, keysIn, P, d->pubWork, keysSorted);
    VL_LAUNCH(rf_seg_sort, LM_NSEG, RF_SEG_THREADS, (size_t)RF_SEG_CAP * 8, keysSorted, d->pubWork, d->pubKeys.p + 2 * N, RF_SEG_CAP);
  }
  d->pubNewCap = P;
  VL_LAUNCH(mp_layout, 1, 1024, 0, (const LgHeader*)d->grid.hdr, (const RfWork*)d->pubWork, (const MapCubeTable*)c->cubeC, (const MapCubeTable*)c->cubeS,
            fromGrid ? 1 : 0, pub);
  VL_BYTES(32.0 * bound);  // every point read once and written once (upper bound: the grid's share is moved by the kernels below)
  VL_LAUNCH(mp_copy_pools, gsGrid, 256, 0, (const int*)pub, (const float4*)c->poolC.p, (const float4*)c->poolS.p, d->pubOut.p, outCap);
  if (fromGrid) {
    VL_LAUNCH(mp_grid_old, gsGrid, 256, 0, d->grid, (const RfWork*)d->pubWork, (const unsigned long long*)keysSorted, (const int*)pub, d->pubOut.p, outCap);
    VL_LAUNCH(mp_grid_new, vl_div_up(P, 256), 256, 0, d->grid, (const RfWork*)d->pubWork, (const unsigned long long*)keysSorted, (const int*)d->pubEnt.p,
              c->prm, (const MapCubeTable*)c->cubeC, (const MapCubeTable*)c->cubeS, (const float4*)c->poolC.p, (const float4*)c->poolS.p, (const int*)pub,
              d->pubOut.p, outCap);
  }
  VL_CUDA(cudaEventRecord(d->evPub, d->pubStream));
  VL_CUDA(cudaGetLastError());
  d->pubDone = true;
  return VLOAM_OK;
}

// wait for the last publication and copy its cloud out (out == NULL: size query)
int vl_lm_get_map(vloam_b200_ctx* c, float* out, int cap_points) {
  LmDevice* d = c->lm;
  if (!d->pubDone) { snprintf(c->err, sizeof c->err, "get_map: nothing was published"); return VLOAM_E_INVALID; }
  VL_CUDA(cudaStreamWaitEvent(c->stream, d->evPub, 0));
  int h[2] = {0, 0};  // {points, voxels created since the grid was built}
  VL_CUDA(cudaMemcpyAsync(h, d->pubInt + MP_NSEG, sizeof h, cudaMemcpyDeviceToHost, c->stream));
  VL_CUDA(cudaStreamSynchronize(c->stream));
  if (h[1] > d->pubNewCap || h[0] > d->pubOutCap) {
    snprintf(c->err, sizeof c->err, "get_map: the published map exceeded its bounds (%d points / %lld, %d new voxels / %lld)", h[0], d->pubOutCap, h[1], d->pubNewCap);
    return VLOAM_E_CAPACITY;
  }
  if (!out || h[0] == 0) return h[0];
  if (cap_points < h[0]) { snprintf(c->err, sizeof c->err, "map buffer too small (%d < %d)", cap_points, h[0]); return VLOAM_E_CAPACITY; }
  VL_CUDA(cudaMemcpyAsync(out, d->pubOut.p, (size_t)h[0] * 16, cudaMemcpyDeviceToHost, c->stream));
  VL_CUDA(cudaStreamSynchronize(c->stream));
  return h[0];
}

// host wait for the last publication (before the map is replaced from the host, and in vloam_b200_synchronize)
int vl_lm_pub_sync(vloam_b200_ctx* c) {
  LmDevice* d = c->lm;
  if (d && d->pubStream) VL_CUDA(cudaStreamSynchronize(d->pubStream));
  return VLOAM_OK;
}

// ---- vloam_b200_load_map: world-frame clouds -> the cube map -----------------------------------------------------------------------
// Every point goes to its cube by the insert formula (LM.cpp:747-761, lm_cube_of) at the context's current laserCloudCen*; every
// non-empty cube is then pcl::VoxelGrid-filtered (LM.cpp:795-808) over its points in input order.  One device-wide sort of the keys
//   [63:51] cube | [50:21] voxel (lm_vox_key: ascending == pcl's linear voxel index) | [20:0] input index
// buckets the points by cube, orders each cube by voxel and keeps input order inside a voxel -- the tie order of SURVEY Appendix B --
// so that a dense cube of ~100k points is sorted by the multi-CTA kernels like any other (no per-segment single-CTA sort).
#define LD_IDX_BITS 21
#define LD_CUBE_SHIFT 51
#define LD_NO_KEY (~0ull)
#define LD_TILE 256
#define LD_SCALARS 8  // ldInt[0..7]: {points, pool top} of corner, of surf, dropped corner, dropped surf
__device__ __forceinline__ unsigned long long ld_run(unsigned long long key) { return key >> LD_IDX_BITS; }  // (cube, voxel)
__device__ __forceinline__ bool ld_head(const unsigned long long* keys, int i, unsigned long long key) {
  return key != LD_NO_KEY && (i == 0 || ld_run(keys[i - 1]) != ld_run(key));
}

// finite check, cube (LM.cpp:747-756) and inside-grid check (LM.cpp:758-761), voxel key; dropped points are counted per kind
__global__ void __launch_bounds__(256) ld_keys(const float4* __restrict__ in, int n, int P, int kind, const LmScalars* __restrict__ s,
                                               vloam_b200_params prm, unsigned long long* __restrict__ keys, int* __restrict__ dropped) {
  VL_PDL_WAIT();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  unsigned long long key = LD_NO_KEY;
  bool drop = false;
  if (i < n) {
    const float4 p = in[i];
    drop = true;
    // (|v| < 1e9: the int conversion of lm_cube_of cannot overflow; such a point is outside any window anyway)
    if (fabsf(p.x) < 1e9f && fabsf(p.y) < 1e9f && fabsf(p.z) < 1e9f) {
      const int ci = lm_cube_of(p.x, s->cenW), cj = lm_cube_of(p.y, s->cenH), ck = lm_cube_of(p.z, s->cenD);
      if (ci >= 0 && ci < VL_CUBE_W && cj >= 0 && cj < VL_CUBE_H && ck >= 0 && ck < VL_CUBE_D) {
        const unsigned vk = lm_vox_key(p, lm_leaf_inv(prm, kind), ci, cj, ck, s->cenW, s->cenH, s->cenD);
        const int cb = ci + VL_CUBE_W * cj + VL_CUBE_W * VL_CUBE_H * ck;
        key = ((unsigned long long)cb << LD_CUBE_SHIFT) | ((unsigned long long)vk << LD_IDX_BITS) | (unsigned long long)i;
        drop = false;
      }
    }
  }
  if (i < P) keys[i] = key;
  const unsigned b = __ballot_sync(0xffffffffu, drop);
  if ((threadIdx.x & 31) == 0 && b) atomicAdd(dropped + kind, __popc(b));
}

// run heads (one per occupied voxel) per tile of LD_TILE sorted keys, and per cube (the cube table's count, zeroed before)
__global__ void __launch_bounds__(LD_TILE) ld_heads(const unsigned long long* __restrict__ keys, int P, MapCubeTable* __restrict__ t,
                                                    int* __restrict__ tileCnt) {
  VL_PDL_WAIT();
  __shared__ int ws[LD_TILE / 32];
  const int i = blockIdx.x * LD_TILE + threadIdx.x;
  const unsigned long long key = i < P ? keys[i] : LD_NO_KEY;
  const bool head = ld_head(keys, i, key);
  const int cb = head ? (int)(key >> LD_CUBE_SHIFT) : -1;
  const unsigned same = __match_any_sync(0xffffffffu, cb);  // heads of a warp nearly always share their cube: one atomic per cube
  if (head && (__ffs(same) - 1) == (int)(threadIdx.x & 31)) atomicAdd(&t->count[cb], __popc(same));
  const unsigned bal = __ballot_sync(0xffffffffu, head);
  if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = __popc(bal);
  __syncthreads();
  if (threadIdx.x == 0) { int sum = 0; for (int w = 0; w < LD_TILE / 32; ++w) sum += ws[w]; tileCnt[blockIdx.x] = sum; }
}

// tile offsets (in place), and the pool layout of a fresh import: every cube count + count / 4 + 256 points of room (as
// vl_lm_import_map), sorted = count; output offset of every cube's first centroid, pool top, totals
__global__ void __launch_bounds__(1024) ld_layout(int* __restrict__ tileCnt, int nTiles, MapCubeTable* __restrict__ t, int* __restrict__ cubeOff,
                                                  LmScalars* __restrict__ s, int kind, int* __restrict__ tot) {
  VL_PDL_WAIT();
  __shared__ int ws[32];
  int carry = 0;  // the same value in every thread
  for (int base = 0; base < nTiles; base += 1024) {
    const int b = base + threadIdx.x;
    const int own = b < nTiles ? tileCnt[b] : 0;
    int sum = 0;
    const int ex = vl_block_excl_scan<1024>(own, ws, &sum);
    if (b < nTiles) tileCnt[b] = carry + ex;
    carry += sum;
  }
  constexpr int PER = (VL_CUBE_NUM + 1023) / 1024;
  const int c0 = threadIdx.x * PER;
  int cnt[PER], cap[PER], ownN = 0, ownCap = 0;
#pragma unroll
  for (int k = 0; k < PER; ++k) {
    cnt[k] = c0 + k < VL_CUBE_NUM ? t->count[c0 + k] : 0;
    cap[k] = cnt[k] ? cnt[k] + cnt[k] / 4 + 256 : 0;
    ownN += cnt[k]; ownCap += cap[k];
  }
  int totN = 0, totCap = 0;
  int runN = vl_block_excl_scan<1024>(ownN, ws, &totN);
  int runC = vl_block_excl_scan<1024>(ownCap, ws, &totCap);
#pragma unroll
  for (int k = 0; k < PER; ++k) {
    const int cb = c0 + k;
    if (cb >= VL_CUBE_NUM) continue;
    cubeOff[cb] = runN; t->start[cb] = cap[k] ? runC : 0; t->cap[cb] = cap[k]; t->sorted[cb] = cnt[k];
    runN += cnt[k]; runC += cap[k];
  }
  if (threadIdx.x == 0) {
    tot[2 * kind] = totN; tot[2 * kind + 1] = totCap;
    if (kind) s->poolTopS = totCap; else s->poolTopC = totCap;
  }
}

// one thread per run head: the voxel's points in input order, f32 sums, one division (rf_fold / rf_centroid), to its place in the pool
__global__ void __launch_bounds__(LD_TILE) ld_fold(const float4* __restrict__ in, const unsigned long long* __restrict__ keys, int P,
                                                   const int* __restrict__ tileOff, const int* __restrict__ cubeOff,
                                                   const MapCubeTable* __restrict__ t, float4* __restrict__ pool) {
  VL_PDL_WAIT();
  __shared__ int ws[LD_TILE / 32];
  const int i = blockIdx.x * LD_TILE + threadIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned long long key = i < P ? keys[i] : LD_NO_KEY;
  const bool head = ld_head(keys, i, key);
  const unsigned bal = __ballot_sync(0xffffffffu, head);
  if (lane == 0) ws[warp] = __popc(bal);
  __syncthreads();
  if (!head) return;
  int before = 0;
  for (int w = 0; w < warp; ++w) before += ws[w];
  const unsigned long long run = ld_run(key);
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  int cnt = 0;
  for (int q = i; q < P && ld_run(keys[q]) == run; ++q) { acc = rf_fold(acc, in[(int)(keys[q] & ((1ull << LD_IDX_BITS) - 1))]); ++cnt; }
  const int cb = (int)(key >> LD_CUBE_SHIFT);
  const int rank = tileOff[blockIdx.x] + before + __popc(bal & ((1u << lane) - 1u));
  pool[t->start[cb] + rank - cubeOff[cb]] = rf_centroid(acc, cnt);
}

int vl_lm_load_map(vloam_b200_ctx* c, const float* corner, int nc, const float* surf, int ns, int stride, int w_offset, bool device,
                   long long dropped[2]) {
  LmDevice* d = c->lm;
  if (nc >= (1 << LD_IDX_BITS) || ns >= (1 << LD_IDX_BITS)) {
    snprintf(c->err, sizeof c->err, "load_map: at most %d points per kind", (1 << LD_IDX_BITS) - 1);
    return VLOAM_E_CAPACITY;
  }
  VL_TRY(lm_map_replaced(c));
  // the last map update and its raw appends (stream3, streamAux) edit the tables and pools rewritten below
  VL_CUDA(cudaStreamWaitEvent(c->stream, c->evMap, 0));
  VL_CUDA(cudaStreamWaitEvent(c->stream, c->evAux, 0));
  const int n[2] = {nc, ns};
  int P[2], nTiles[2];
  for (int k = 0; k < 2; ++k) {
    P[k] = 0;
    if (n[k] > 0) { P[k] = 2; while (P[k] < n[k]) P[k] <<= 1; }
    nTiles[k] = vl_div_up(P[k], LD_TILE);
    VL_TRY(vl_reserve(c, d->ldIn[k], (size_t)max(n[k], 1)));
  }
  VL_TRY(vl_reserve(c, d->ldKeys, (size_t)max(P[0] + P[1], 1)));
  VL_TRY(vl_reserve(c, d->ldInt, (size_t)LD_SCALARS + 2 * VL_CUBE_NUM + nTiles[0] + nTiles[1]));
  const VlCloudIn cl[2] = {{corner, nc, d->ldIn[0].p}, {surf, ns, d->ldIn[1].p}};
  VL_TRY(vl_pack_clouds(c, cl, 2, stride, w_offset, device));
  int* tot = d->ldInt.p;
  int* cubeOff[2] = {tot + LD_SCALARS, tot + LD_SCALARS + VL_CUBE_NUM};
  int* tiles[2] = {tot + LD_SCALARS + 2 * VL_CUBE_NUM, tot + LD_SCALARS + 2 * VL_CUBE_NUM + nTiles[0]};
  unsigned long long* keys[2] = {d->ldKeys.p, d->ldKeys.p + P[0]};
  MapCubeTable* tab[2] = {c->cubeC, c->cubeS};
  VL_CUDA(cudaMemsetAsync(tot, 0, LD_SCALARS * sizeof(int), c->stream));
  for (int k = 0; k < 2; ++k) {
    VL_CUDA(cudaMemsetAsync(tab[k], 0, sizeof(MapCubeTable), c->stream));
    if (n[k] > 0) {
      VL_BYTES(24.0 * P[k]);
      VL_LAUNCH(ld_keys, vl_div_up(P[k], 256), 256, 0, (const float4*)d->ldIn[k].p, n[k], P[k], k, (const LmScalars*)c->lmm, c->prm, keys[k], tot + 4);
      VL_TRY(vl_sort_u64(c, keys[k], P[k]));
      VL_LAUNCH(ld_heads, nTiles[k], LD_TILE, 0, (const unsigned long long*)keys[k], P[k], tab[k], tiles[k]);
    }
    VL_LAUNCH(ld_layout, 1, 1024, 0, tiles[k], nTiles[k], tab[k], cubeOff[k], c->lmm, k, tot);
  }
  int h[LD_SCALARS];
  VL_CUDA(cudaMemcpyAsync(h, tot, sizeof h, cudaMemcpyDeviceToHost, c->stream));
  VL_CUDA(cudaStreamSynchronize(c->stream));
  for (int k = 0; k < 2; ++k) {
    DBuf<float4>& pool = k ? c->poolS : c->poolC;
    if ((size_t)h[2 * k + 1] * 2 > pool.cap) VL_TRY(vl_reserve(c, pool, (size_t)h[2 * k + 1] * 2));  // (contents are replaced below)
    if (n[k] > 0) {
      VL_BYTES(32.0 * P[k]);
      VL_LAUNCH(ld_fold, nTiles[k], LD_TILE, 0, (const float4*)d->ldIn[k].p, (const unsigned long long*)keys[k], P[k], (const int*)tiles[k],
                (const int*)cubeOff[k], (const MapCubeTable*)tab[k], pool.p);
    }
  }
  // whatever reads the map next on another stream (a publication, the next update) waits for these
  VL_CUDA(cudaEventRecord(c->evMap, c->stream));
  VL_CUDA(cudaEventRecord(c->evAux, c->stream));
  VL_CUDA(cudaGetLastError());
  d->hMapUpperC = h[0]; d->hMapUpperS = h[2];
  c->h_lmm->poolTopC = h[1]; c->h_lmm->poolTopS = h[3];
  if (dropped) { dropped[0] = h[4]; dropped[1] = h[5]; }
  return VLOAM_OK;
}

// vloam_b200_set_map_pose: q_wmap_wodom / t_wmap_wodom (LM.cpp:147-151) on the main stream, behind the last transformUpdate
struct LmMapPose { double q[4], t[3]; };
__global__ void lm_set_map_pose(LmScalars* __restrict__ s, LmMapPose p) {
  VL_PDL_WAIT();
  for (int k = 0; k < 4; ++k) s->q_wmap_wodom[k] = p.q[k];
  for (int k = 0; k < 3; ++k) s->t_wmap_wodom[k] = p.t[k];
}
int vl_lm_set_map_pose(vloam_b200_ctx* c, const double q[4], const double t[3]) {
  VL_TRY(vl_lm_join(c));
  LmMapPose p;
  memcpy(p.q, q, sizeof p.q); memcpy(p.t, t, sizeof p.t);
  VL_LAUNCH(lm_set_map_pose, 1, 1, 0, c->lmm, p);
  VL_CUDA(cudaGetLastError());
  return VLOAM_OK;
}

void vl_lm_set_map_update(vloam_b200_ctx* c, bool enabled) { c->lm->mapUpdate = enabled; }

// vloam_b200_get_map_kind: the segments of one kind of the published cloud (pubInt: segment q = 2 cube + kind), in cube order
__global__ void __launch_bounds__(1024) mp_kind_layout(const int* __restrict__ pub, int kind, int* __restrict__ off) {
  VL_PDL_WAIT();
  __shared__ int ws[32];
  constexpr int PER = (VL_CUBE_NUM + 1023) / 1024;
  const int c0 = threadIdx.x * PER;
  int cnt[PER], own = 0;
#pragma unroll
  for (int k = 0; k < PER; ++k) {
    const int q = 2 * (c0 + k) + kind;
    cnt[k] = c0 + k < VL_CUBE_NUM ? pub[q + 1] - pub[q] : 0;
    own += cnt[k];
  }
  int tot = 0;
  int run = vl_block_excl_scan<1024>(own, ws, &tot);
#pragma unroll
  for (int k = 0; k < PER; ++k) if (c0 + k < VL_CUBE_NUM) { off[c0 + k] = run; run += cnt[k]; }
  if (threadIdx.x == 0) off[VL_CUBE_NUM] = tot;
}
__global__ void __launch_bounds__(256) mp_kind_copy(const int* __restrict__ pub, const int* __restrict__ off, int kind, const float4* __restrict__ cloud,
                                                    float4* __restrict__ out) {
  VL_PDL_WAIT();
  const int total = off[VL_CUBE_NUM];
  for (int g = blockIdx.x * blockDim.x + threadIdx.x; g < total; g += gridDim.x * blockDim.x) {
    int lo = 0, hi = VL_CUBE_NUM;
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (off[mid] <= g) lo = mid; else hi = mid; }
    out[g] = cloud[pub[2 * lo + kind] + (g - off[lo])];
  }
}
int vl_lm_get_map_kind(vloam_b200_ctx* c, int which, float* out, int cap_points) {
  LmDevice* d = c->lm;
  const int n = vl_lm_get_map(c, nullptr, 0);  // waits for the publication; its errors
  if (n < 0) return n;
  VL_TRY(vl_reserve(c, d->pubKindOff, (size_t)VL_CUBE_NUM + 1));
  VL_LAUNCH(mp_kind_layout, 1, 1024, 0, (const int*)d->pubInt, which, d->pubKindOff.p);
  int m = 0;
  VL_CUDA(cudaMemcpyAsync(&m, d->pubKindOff.p + VL_CUBE_NUM, sizeof m, cudaMemcpyDeviceToHost, c->stream));
  VL_CUDA(cudaStreamSynchronize(c->stream));
  if (!out || m == 0) return m;
  if (cap_points < m) { snprintf(c->err, sizeof c->err, "map buffer too small (%d < %d)", cap_points, m); return VLOAM_E_CAPACITY; }
  VL_TRY(vl_reserve(c, d->pubKind, (size_t)m));
  VL_BYTES(32.0 * m);
  VL_LAUNCH(mp_kind_copy, min(vl_div_up(m, 256), c->num_sms * 8), 256, 0, (const int*)d->pubInt, (const int*)d->pubKindOff.p, which,
            (const float4*)d->pubOut.p, d->pubKind.p);
  VL_CUDA(cudaMemcpyAsync(out, d->pubKind.p, (size_t)m * 16, cudaMemcpyDeviceToHost, c->stream));
  VL_CUDA(cudaStreamSynchronize(c->stream));
  return m;
}

void vl_lm_paths(vloam_b200_ctx* c, long long out[2]) { const LmDevice* d = c->lm; out[0] = d->paths[0]; out[1] = d->paths[1]; }

int vl_chain_trace_arm_lm(void* dev) { return cudaMemcpyToSymbol(g_chain_trace, &dev, sizeof(void*)) == cudaSuccess ? VLOAM_OK : VLOAM_E_CUDA; }
int vl_lm_preload(vloam_b200_ctx* c) {  // see vl_sr_set_attrs: load every kernel of this file when a context is created
  cudaFuncAttributes fa_;
  VL_CUDA(cudaFuncGetAttributes(&fa_, lm_prepare));
  VL_CUDA(cudaFuncGetAttributes(&fa_, lm_spec_prepare));
  VL_CUDA(cudaFuncGetAttributes(&fa_, lm_fit));
  VL_CUDA(cudaFuncGetAttributes(&fa_, lg_zero)); VL_CUDA(cudaFuncGetAttributes(&fa_, lg_rebuild)); VL_CUDA(cudaFuncGetAttributes(&fa_, lm_prepare_fast));
  VL_CUDA(cudaFuncGetAttributes(&fa_, lg_knn)); VL_CUDA(cudaFuncGetAttributes(&fa_, lg_keys_to_ids)); VL_CUDA(cudaFuncGetAttributes(&fa_, lm_gather));
  VL_CUDA(cudaFuncGetAttributes(&fa_, mu_apply)); VL_CUDA(cudaFuncGetAttributes(&fa_, mu_keys)); VL_CUDA(cudaFuncGetAttributes(&fa_, mz_collect));
  VL_CUDA(cudaFuncGetAttributes(&fa_, mz_layout_for_grid));
  VL_CUDA(cudaFuncGetAttributes(&fa_, lm_fit_sets));
  VL_CUDA(cudaFuncGetAttributes(&fa_, lm_transform_update));
  VL_CUDA(cudaFuncGetAttributes(&fa_, rf_keys));
  VL_CUDA(cudaFuncGetAttributes(&fa_, rf_seg_scatter));
  VL_CUDA(cudaFuncGetAttributes(&fa_, rf_seg_sort));
  VL_CUDA(cudaFuncGetAttributes(&fa_, rf_match));
  VL_CUDA(cudaFuncGetAttributes(&fa_, rf_scan_layout));
  VL_CUDA(cudaFuncGetAttributes(&fa_, rf_emit));
  VL_CUDA(cudaFuncGetAttributes(&fa_, rf_alloc));
  VL_CUDA(cudaFuncGetAttributes(&fa_, rf_commit));
  VL_CUDA(cudaFuncGetAttributes(&fa_, rf_finish));
  VL_CUDA(cudaFuncGetAttributes(&fa_, rf_append_outside));
  VL_CUDA(cudaFuncGetAttributes(&fa_, lm_scan_sorted));
  VL_CUDA(cudaFuncGetAttributes(&fa_, lm_set_counts));
  VL_CUDA(cudaFuncGetAttributes(&fa_, lm_register_full));
  VL_CUDA(cudaFuncGetAttributes(&fa_, mp_collect)); VL_CUDA(cudaFuncGetAttributes(&fa_, mp_layout)); VL_CUDA(cudaFuncGetAttributes(&fa_, mp_copy_pools));
  VL_CUDA(cudaFuncGetAttributes(&fa_, mp_grid_old)); VL_CUDA(cudaFuncGetAttributes(&fa_, mp_grid_new));
  return VLOAM_OK;
}

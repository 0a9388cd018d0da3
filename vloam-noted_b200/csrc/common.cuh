// common.cuh -- context, device buffers and launch helpers shared by the stage files.
//
// Everything on the hot path runs as hand-written CUDA on the context's single
// stream.  The host side only orders launches and reads back a handful of
// counts at explicit sync points; it never computes on point data.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include "vloam_b200.h"

#define VL_MAX_RINGS 128
#define VL_SECTORS 6
#define VL_CUBE_W 21
#define VL_CUBE_H 21
#define VL_CUBE_D 11
#define VL_CUBE_NUM (VL_CUBE_W * VL_CUBE_H * VL_CUBE_D)
#define VL_MAX_VALID 125  // laserCloudValidInd[125], laser_mapping.h:127
#define VL_PROF_MAX 4096

// ---- device-resident scalars (one struct per context, also mirrored in pinned host memory)
struct SrScalars {
  int firstValid, lastValid;  // first / last point surviving the NaN + range filter
  int trigger;                // input index of the first point that sets halfPassed (INT_MAX if none)
  float startOri, endOri;     // scan_registration.cpp:185-197
  int count;                  // kept points == laserCloud size
  int nSharp, nLessSharp, nFlat, nLessFlat;
  int blocksDone;             // last-block-done counter for the ring scan
  int nQueries;               // nSharp + nFlat: odometry factor slots
};

struct LmSolveState {  // trust-region LM state, lives on the device (lm_solver.cu)
  double x[7];         // current iterate {qx,qy,qz,qw,tx,ty,tz}
  double xc[7];        // candidate
  double best[7];
  double scale[6];     // Jacobi scaling, computed once at iteration 0
  double diag[6];
  double H[21], g[6];  // accepted-point normal equations (unscaled, robustified)
  double cost, cand_cost, min_cost, model_cost_change;
  double radius, decrease_factor, x_norm, gmax;
  int reuse_diagonal, done, iter, last_successful, have_candidate, nfactors;
  double initial_cost, final_cost;
};

struct EvalOut {  // one robustified evaluation: 21 upper-triangular H, 6 g, cost
  double v[28];
};

struct MapCubeTable {  // per cube slot: where its points live in the pool
  int start[VL_CUBE_NUM];
  int count[VL_CUBE_NUM];
  int cap[VL_CUBE_NUM];
  int sorted[VL_CUBE_NUM];  // length of the prefix whose voxel keys are strictly increasing
};

struct LmScalars {
  int cenW, cenH, cenD;             // laserCloudCen{Width,Height,Depth}
  int validNum;
  int validInd[VL_MAX_VALID];
  int Mc, Ms;                       // sub-map sizes
  int Qc, Qs;                       // downsampled stack sizes
  int tailC, tailS;                 // unsorted tail points in the valid cubes (incl. this frame's inserts)
  int poolTopC, poolTopS;
  int overflow;                     // set when a pool / buffer bound was hit
  int optimized;
  int totalC, totalS;               // points in all 4851 cubes before this frame's update (bounds the next sub-map)
  int needSlow;                     // lm_prepare_fast: this sweep cannot use the in-place grid path (window moved / grid dirty): the host repeats it on the pool path
  int gridCount;                    // live points in the grid (both kinds)
  int gridCountC;                   // ... of them corner points
  int outsideC, outsideS;           // points appended raw to cubes outside the 5x5x3 window so far (rf_append_outside), per kind
  int gridTop, gridDirty, gridDead; // voxel-hash grid: chunks in use, dirty flag, tombstones (copied by lm_transform_update for the host's bookkeeping)
  double pose[7];                   // q_w_curr, t_w_curr (parameters[7], laser_mapping.h:156)
  double q_wmap_wodom[4], t_wmap_wodom[3];
  double q_wodom[4], t_wodom[3];
  double q_hf[4], t_hf[3];
};

struct LoScalars {
  double para_q[4], para_t[3];  // q_last_curr, t_last_curr (laser_odometry.h:127-131)
  double q_w[4], t_w[3];        // q_w_curr, t_w_curr
  int corner_correspondence, plane_correspondence;
};

template <typename T>
struct DBuf {  // growable device buffer
  T* p = nullptr;
  size_t cap = 0;  // elements
};

// Launch helpers take their stream from here: the map update of a frame is issued by a helper thread
// (laser_mapping.cu) while the calling thread already queues the next sweep, so "the current stream" is a
// per-thread notion.  Non-null: this thread's launches go there instead of c->stream.
#include <chrono>
static inline double vl_now_us() { return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now().time_since_epoch()).count(); }
#define VL_HOST_MARK(k) do { c->hostT[k] = vl_now_us(); } while (0)  // (a clock read: ~20 ns)
extern thread_local cudaStream_t vl_tls_stream;
#define VL_STREAM(c) (vl_tls_stream ? vl_tls_stream : (c)->stream)
struct VlWorker;

struct vloam_b200_ctx {
  vloam_b200_params prm;
  int device;
  cudaStream_t stream;
  cudaStream_t stream2;       // side stream: work that is independent of the odometry solve overlaps it
  cudaStream_t stream4;       // second side stream: the corner stack filter runs beside the surf one
  cudaEvent_t evStacksC;
  cudaStream_t streamAux;     // map-update work that is off the chain update -> speculative sub-map (zeroing, outside appends)
  cudaEvent_t evAux, evAuxZero, evUpd;
  cudaStream_t stream3;       // map update of frame k runs here while frame k+1's scan registration / odometry run on `stream`
  cudaEvent_t evSR;           // scan registration of this frame finished and its counts are in h_srs
  cudaEvent_t evSRfeat;       // ... its sharp / less-sharp / flat clouds are complete (the per-ring voxel filter of the less-flat cloud may still run)
  cudaEvent_t evStacks;       // this frame's downsampled stacks are ready
  cudaEvent_t evLast;         // search structures over the next "last" clouds are built
  cudaEvent_t evPose;         // solveMapping's pose is final (the map update may start)
  cudaEvent_t evMap;          // the map update has finished (the next solveMapping may start)
  cudaEvent_t evKeys;         // the map update has read the stacks (rf_keys): the next sweep's stack filters may start
  cudaEvent_t evKeysSel[2];   // same, per stack buffer pair (index = stackSel the update read): the look-ahead filters wait on the pair they overwrite
  bool stacksReady;
  bool lm_reset_pending;      // LaserMapping::reset was called since the last solveMapping
  char err[512];
  long long launches;         // updated with __atomic_fetch_add (two issuing threads)
  long long regrows;          // device buffer (re)allocations after creation (vl_reserve): each one stalls a stream for ~ms
  // One device arena per context, allocated in create: vl_reserve carves the ~60 per-sweep buffers out of it with a bump pointer.
  // (A cudaMalloc costs 2-35 ms on a B200 box with a driver that has >1 GB mapped: the first sweep of a context spent 210 ms in
  // 56 of them, and every later regrow stalled a sweep by several ms.)  Requests that do not fit fall back to cudaMalloc.
  char* arena; size_t arenaCap; size_t arenaTop;
  VlWorker* worker;           // helper thread that issues the map update (created on first use)
  int num_sms;
  bool timing;
  cudaEvent_t ev[4];
  double hostT[16];     // timing mode only: host clock (us) at marks inside a frame (see "timing.host" in capi.cu)
  cudaEvent_t evx[12]; // timing mode only: finer marks (see "timing.detail" in capi.cu)
  float stage_ms[3];

  // ---- scan registration
  DBuf<float> in;            // raw input (n * stride floats)
  int n_in, stride;
  DBuf<int> ring;            // per input point ring id or -1
  DBuf<float> ori;           // per input point -atan2f(y,x)
  DBuf<int> blockHist;       // [ring][block] counts -> exclusive offsets
  int* ringCount;            // [VL_MAX_RINGS]
  int* ringStart;            // [VL_MAX_RINGS + 1]
  SrScalars* srs;            // device
  SrScalars* h_srs;          // pinned host mirror
  DBuf<float4> cloud;        // laserCloud
  DBuf<float> curv;
  DBuf<int> label;
  DBuf<unsigned char> picked;
  DBuf<unsigned long long> sortScratch;  // oversize sector / ring sorts
  int* provSharp; int* provLess; int* provFlat;  // provisional picks (indices) per (ring, sector)
  int* cntSharp; int* cntLess; int* cntFlat;     // per (ring, sector)
  int* offSharp; int* offLess; int* offFlat;     // exclusive offsets
  DBuf<float4> lessFlatProv;  // per-ring downsampled points at ringStart[r]
  int* ringDsCount; int* ringDsOff;
  DBuf<int> selIdx;           // per-ring compacted selection (original indices)
  DBuf<float4> sharp, flat;
  DBuf<float4> lessSharp[3], lessFlat[3];  // three generations: the "last" clouds, this frame's ([cur]) and the look-ahead's
  DBuf<float4> endSharp[3], endFlat[3];    // VLOAM_FLAG_TRANSFORM_TO_END: generation g's clouds in the sweep-end frame (lo_transform_to_end)
  cudaEvent_t evEnd;                       // ... this sweep's end clouds are written (recorded by vl_lo_run; the stack filters wait on it)
  int cur;                   // index of this frame's lessSharp / lessFlat buffer
  int nKept, nSharp, nLessSharp, nFlat, nLessFlat;  // host copies (valid after the SR sync point)
  bool sr_counts_valid;
  // look-ahead scan registration (vloam_b200_prefetch_scan[_device]): a second set of every field above (VL_SR_FIELDS)
  // ... and a third one: a replay may register TWO sweeps ahead.  While sweep k is mapped, sweep k+1's set (srNext, filled during
  // sweep k-1) feeds the look-ahead odometry and stack filters, and sweep k+2's upload + scan registration run into srNext2; when
  // sweep k+1 is processed its set is swapped into the context and srNext2 becomes srNext.
  struct SrSet* srNext;       // spare set; holds the results for srNextKey when srNextValid
  const float* srNextKey; int srNextN, srNextStride; bool srNextValid;
  struct SrSet* srNext2;      // second spare set (the sweep after srNextKey)
  const float* srNext2Key; int srNext2N, srNext2Stride; bool srNext2Valid;
  struct SrPend { const float* key; int n, stride; bool dev; } srPend[2];  // registered, not yet launched (in order)
  int srPendCount;
  cudaStream_t streamSR;

  // ---- laser odometry
  LoScalars* los; LoScalars* h_los;
  LoScalars* losNext;         // odometry state after the look-ahead odometry of sweep srNextKey (valid when loNextValid)
  bool loNextValid, loNextQueued, srAdopted, s2Done;
  int loNextSet;              // the "last" set the look-ahead odometry searched (it assumed monotone rings: checked at adoption)
  bool loAssumeMonotone;      // lo_associate: take the grid path without the host flags (look-ahead only)
  bool inProcessFrame;        // inside process_frame: mapping follows the odometry in the same call
  bool srDeferred, sideSubmitted;  // the registered look-ahead scan registration is issued with the deferred structures; that side work is with the helper thread
  bool loDeferred; int defSet, defNc, defNs; const float4* defCorner; const float4* defSurf;  // side-stream work of the odometry stage queued after the mapping
  // Two sweeps registered ahead: the search structures over the NEXT sweep's clouds (its scan registration finished a sweep ago)
  // are built during THIS sweep, into the set this sweep's odometry searched; the next call finds them (loPreValid + the keys below)
  // and its look-ahead odometry can be queued at once.  preDeferred: that build is part of the deferred side work of this call.
  bool preDeferred, loPreValid; int preSet, preNc, preNs; const float4* preCorner; const float4* preSurf;
  bool stacksAdopted;         // this sweep's stacks were filtered during the previous sweep (look-ahead) and adopted
  bool earlyLoArmed;          // the next sweep's look-ahead odometry is the first item of the side work (its stream waits are issued)
  bool sideWaitsIssued;       // the caller already ordered streamSR / stream2 behind the last odometry solve (before queuing the next one)
  cudaEvent_t evS2;           // sync point S2 (pose + sizes copied to the host)
  unsigned* h_s2flag; unsigned s2seq;  // in-place path: lm_transform_update writes the structs + this sequence number into pinned memory
  cudaStream_t streamLO;      // the look-ahead odometry of the NEXT sweep runs here, beside this sweep's mapping (own factor buffers)
  cudaEvent_t evLoNext;       // that look-ahead solve has finished (its result is in losNext)
  cudaEvent_t evLoSolve;      // the last queued odometry solve (and every one before it) has finished reading the "last" clouds and their grids
  int nCornerLast, nSurfLast;  // host counts of the "last" clouds (= other buffer of the pair)
  bool lo_inited; int lo_frameCount;
  float4* cornerLastPtr; float4* surfLastPtr;  // after solveLO's swap
  // search structures over the "last" clouds, double-buffered: set [lastSet] serves this frame's odometry
  // while the side stream builds set [lastSet ^ 1] from this frame's clouds
  int* loRingTbl;                     // 2 sets x 2 clouds x (144 + 1) ints: ring-value -> first index tables
  DBuf<int> loGridCells[2], loGridCellOf; DBuf<float4> loGridSorted[2]; bool loGridValid[2]; int loGridMask[2];  // hash of occupied 1.28 m cells per set
  int lastSet;
  DBuf<int> loCornerIdx, loSurfIdx;   // association results (2 / 3 ints per query)
  DBuf<double> factors;               // 10 doubles per factor slot (mapping stage, C-ABI evaluate / solve)
  DBuf<double> loFactors; DBuf<int> loFactorValid;  // the odometry stage's own factor slots: its look-ahead solve overlaps the mapping solve
  DBuf<double> factorS;               // DISTORTION only: interpolation ratio s of every odometry factor slot (LO.cpp:368-372, 472-476)
  DBuf<int> factorValid;
  DBuf<EvalOut> evalPartials;
  EvalOut* evalOut;
  LmSolveState* lms; LmSolveState* h_lms;
  DBuf<int> dbgLoCorner[2], dbgLoSurf[2];
  double dbgLoCost[4];
  bool skip_frame;

  // ---- laser mapping
  LmScalars* lmm; LmScalars* h_lmm;
  MapCubeTable* cubeC; MapCubeTable* cubeS;  // device
  DBuf<float4> poolC, poolS;
  DBuf<float4> stackC, stackS;
  DBuf<float4> stackCN, stackSN;  // the NEXT sweep's stacks (filtered during this sweep when its scan registration finished early); swapped in at adoption
  int stackSel; bool stacksNextReady;  // which pair of device counts (LmDevice::dQ) belongs to stackC / stackS
  DBuf<float4> fromMapC, fromMapS;
  int lm_frameCount;
  int lm_optimized;  // host copy: did the last solveMapping run the optimisation (LM.cpp:514)
  DBuf<float> knnD2; DBuf<int> knnOk;
  DBuf<float4> knnPts; DBuf<unsigned long long> knnKey;  // the five neighbours themselves (the grid has no stable point ids) and their keys (debug capture)
  DBuf<int> dbgKnnIdx[2][2]; DBuf<float> dbgKnnD2[2][2]; DBuf<int> dbgKnnOk[2][2];
  double dbgLmCost[4];
  struct LmDevice* lm;  // the mapping stage's own state (laser_mapping.cu: vl_lm_init)
  // voxel filter scratch
  DBuf<unsigned long long> vKeys, vKeys2; DBuf<int> vHead; DBuf<int> vScan, vScan2;  // two scratch lanes: the corner and surf filters run concurrently
  DBuf<float4> vOut; DBuf<float4> vIn;
  DBuf<float4> regOut;  // full-resolution cloud registered into the map frame
  int* vScalars;  // device scratch ints
  int* h_vScalars;
  // refilter scratch
  DBuf<unsigned long long> tailKeys; DBuf<float4> staging;
  // caller-supplied stage inputs (vloam_b200_laser_odometry_input / vloam_b200_laser_mapping_input, stage_inputs.cu); everything here
  // is reserved by the first input call, a context that never makes one holds none of it
  DBuf<float> inStage;                  // host clouds with stride != 4 or w_offset != 3, uploaded as they are, before vl_pack_xyzi
  DBuf<float4> miCorner, miSurf, miFull;  // LaserMapping::input's laserCloudCornerLast / laserCloudSurfLast / laserCloudFullRes
  LoScalars* miLos;                     // device: the caller's q_wodom_curr / t_wodom_curr in q_w / t_w (never c->los)
  cudaEvent_t evIn;                     // the caller's clouds are on the device (the stack filters of the side streams wait on it)
  int miNc, miNs, miNfull;
  bool miPending;                       // a mapping input waits for the next vloam_b200_laser_mapping call of this frame
  bool miUsed;                          // the mapping call of this frame consumed one (register_full_cloud and the pose follow it)
  bool miSkip;                          // its skip_frame
  // vloam_b200_relocalize (relocalize.cu): its state is created by the first call
  struct RlState* rl;
  bool rlReady;                         // the last laser_mapping call mapped a sweep, and no map was loaded since (its stacks are the query)
  // per-kernel timing (vloam_b200_profile_kernel): CUDA events around the launches of one named kernel
  char prof_name[64];                 // kernel to time, or "*" for every launch
  cudaEvent_t prof_ev[VL_PROF_MAX][2];
  const char* prof_kname[VL_PROF_MAX];
  double prof_kbytes[VL_PROF_MAX];
  cudaStream_t prof_kstream[VL_PROF_MAX];
  int prof_n, prof_created;
  double prof_bytes, prof_next_bytes;
};

// Every per-sweep field of the scan-registration stage (names as in vloam_b200_ctx).  The look-ahead keeps a second
// set: it is swapped into the context while its kernels are queued and swapped back afterwards, and swapped in for
// good when the sweep it belongs to is processed.  (The kernels captured the pointers at launch; swapping is host
// bookkeeping only.)
#define VL_SR_FIELDS(X)                                                                                              \
  X(DBuf<float>, in) X(int, n_in) X(int, stride) X(DBuf<int>, ring) X(DBuf<float>, ori) X(DBuf<int>, blockHist)        \
  X(int*, ringCount) X(int*, ringStart) X(SrScalars*, srs) X(SrScalars*, h_srs) X(DBuf<float4>, cloud) X(DBuf<float>, curv) \
  X(DBuf<int>, label) X(DBuf<unsigned char>, picked) X(DBuf<unsigned long long>, sortScratch)                        \
  X(int*, provSharp) X(int*, provLess) X(int*, provFlat) X(int*, cntSharp) X(int*, cntLess) X(int*, cntFlat)          \
  X(int*, offSharp) X(int*, offLess) X(int*, offFlat) X(DBuf<float4>, lessFlatProv) X(int*, ringDsCount) X(int*, ringDsOff) \
  X(DBuf<int>, selIdx) X(DBuf<float4>, sharp) X(DBuf<float4>, flat) X(int, cur)                                      \
  X(int, nKept) X(int, nSharp) X(int, nLessSharp) X(int, nFlat) X(int, nLessFlat) X(bool, sr_counts_valid) X(cudaEvent_t, evSR) X(cudaEvent_t, evSRfeat)
struct SrSet {
#define VL_X(type, name) type name{};
  VL_SR_FIELDS(VL_X)
#undef VL_X
};
static inline void vl_sr_swap(vloam_b200_ctx* c, SrSet& s) {
#define VL_X(type, name) { type t_ = c->name; c->name = s.name; s.name = t_; }
  VL_SR_FIELDS(VL_X)
#undef VL_X
}

// ---- error handling ---------------------------------------------------------
#define VL_CUDA(call)                                                                     \
  do {                                                                                    \
    cudaError_t e_ = (call);                                                              \
    if (e_ != cudaSuccess) {                                                              \
      snprintf(c->err, sizeof c->err, "%s:%d %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); \
      return VLOAM_E_CUDA;                                                                \
    }                                                                                     \
  } while (0)

#define VL_TRY(call)            \
  do {                          \
    int r_ = (call);            \
    if (r_ != VLOAM_OK) return r_; \
  } while (0)

// Every kernel is launched with programmatic stream serialisation allowed and starts with VL_PDL_WAIT()
// (griddepcontrol.wait): the next grid of a dependent chain is already resident when its predecessor
// drains, which removes most of the launch gap between the ~45 dependent kernels of a frame.
#define VL_PDL_WAIT() cudaGridDependencySynchronize()
// debug: device-side timeline of the pose chain (tests/gpu_chain_trace.py).  Each traced kernel stamps %globaltimer when its first
// thread passes the dependency wait (= its predecessor in the stream has finished and this grid runs); one pointer per
// translation unit (no relocatable device code), armed by vloam_b200_debug_get("chain.trace").
#ifdef __CUDACC__
struct VlChainTrace { unsigned long long n; unsigned long long rec[4096][2]; };
static __constant__ VlChainTrace* g_chain_trace = nullptr;  // (__constant__: the check costs one LDC, not a global-memory round trip at the start of every kernel)
__device__ __forceinline__ void vl_chain_stamp(int id) {
  if (g_chain_trace && blockIdx.x == 0 && threadIdx.x == 0) {
    unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    const unsigned long long k = atomicAdd(&g_chain_trace->n, 1ull);
    if (k < 4096) { g_chain_trace->rec[k][0] = (unsigned long long)id; g_chain_trace->rec[k][1] = t; }
  }
}
int vl_chain_trace_arm_lm(void* dev);      // laser_mapping.cu's copy of the pointer
int vl_chain_trace_arm_solver(void* dev);  // lm_solver.cu's
int vl_chain_trace_arm_lo(void* dev);      // laser_odometry.cu's
#endif
#define VL_LAUNCH(kernel, grid, block, smem, ...)                                              \
  do {                                                                                         \
    const bool prof_ = c->prof_name[0] && vl_prof_match(c, #kernel) && c->prof_n < VL_PROF_MAX; \
    if (prof_) cudaEventRecord(c->prof_ev[c->prof_n][0], VL_STREAM(c));                        \
    cudaLaunchConfig_t cfg_ = {};                                                              \
    cfg_.gridDim = dim3(grid); cfg_.blockDim = dim3(block); cfg_.dynamicSmemBytes = (smem); cfg_.stream = VL_STREAM(c); \
    cudaLaunchAttribute at_[1];                                                                \
    at_[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;                            \
    at_[0].val.programmaticStreamSerializationAllowed = 1;                                     \
    cfg_.attrs = at_; cfg_.numAttrs = 1;                                                       \
    cudaLaunchKernelEx(&cfg_, kernel, __VA_ARGS__);                                            \
    if (prof_) { cudaEventRecord(c->prof_ev[c->prof_n][1], VL_STREAM(c)); c->prof_kname[c->prof_n] = #kernel; c->prof_kbytes[c->prof_n] = c->prof_next_bytes; c->prof_kstream[c->prof_n] = VL_STREAM(c); \
                 c->prof_n++; c->prof_bytes += c->prof_next_bytes; } \
    c->prof_next_bytes = 0;                                                                    \
    __atomic_fetch_add(&c->launches, 1LL, __ATOMIC_RELAXED);                                   \
  } while (0)

// algorithmic bytes of the next launch (DESIGN.md roofline table), consumed by VL_LAUNCH when that kernel is profiled
#define VL_BYTES(b) (c->prof_next_bytes = (double)(b))

static inline bool vl_prof_match(const vloam_b200_ctx* c, const char* k) {
  // template kernels show up as "lo_assoc<true>": compare the prefix
  if (c->prof_name[0] == '*') return true;
  const size_t n = strlen(c->prof_name);
  return strncmp(c->prof_name, k, n) == 0 && (k[n] == 0 || k[n] == '<');
}

// cudaFree for anything vl_reserve handed out: blocks inside the arena are released with it
static inline void vl_dev_free(vloam_b200_ctx* c, void* p) {
  if (!p) return;
  if (c->arena && (char*)p >= c->arena && (char*)p < c->arena + c->arenaCap) return;
  cudaFree(p);
}

// Grows (never shrinks).  cudaMalloc / cudaFree stall the stream for milliseconds, so buffers whose
// size follows the map ask for `slack` extra elements: growth then happens once per ~hundreds of frames.
template <typename T>
static inline int vl_reserve(vloam_b200_ctx* c, DBuf<T>& b, size_t n, bool keep = false, size_t slack = 0) {
  if (n <= b.cap) return VLOAM_OK;
  n += slack;
  size_t ncap = b.cap ? b.cap : ((size_t)1 << 17);  // a regrow stalls the pipeline for ~1 ms: start above any per-sweep feature count
  while (ncap < n) ncap *= 2;
  if (ncap * sizeof(T) <= ((size_t)32 << 20)) ncap *= 2;  // HBM is plentiful: head room so a count hovering at a power of two never regrows
  T* np = nullptr;
  __atomic_fetch_add(&c->regrows, 1LL, __ATOMIC_RELAXED);
  const size_t bytes_ = (ncap * sizeof(T) + 511) & ~(size_t)511;
  if (c->arena && bytes_ <= c->arenaCap / 4) {  // bump allocation from the context's arena (grown-out blocks are not reused: they are few and small)
    const size_t at = __atomic_fetch_add(&c->arenaTop, bytes_, __ATOMIC_RELAXED);
    if (at + bytes_ <= c->arenaCap) np = reinterpret_cast<T*>(c->arena + at);
  }
  if (np) {
    if (keep && b.p && b.cap) VL_CUDA(cudaMemcpyAsync(np, b.p, b.cap * sizeof(T), cudaMemcpyDeviceToDevice, VL_STREAM(c)));
    if (b.p) { VL_CUDA(cudaStreamSynchronize(VL_STREAM(c))); vl_dev_free(c, b.p); }
    b.p = np; b.cap = ncap;
    return VLOAM_OK;
  }
  static const bool trace = getenv("VLOAM_TRACE_ALLOC") != nullptr;
  const double t0_ = trace ? vl_now_us() : 0.0;
  VL_CUDA(cudaMalloc(&np, ncap * sizeof(T)));
  if (trace) fprintf(stderr, "[vloam_b200] grow buffer to %zu x %zu B (frame %d): cudaMalloc %.0f us\n", ncap, sizeof(T), c->lo_frameCount, vl_now_us() - t0_);
  if (keep && b.p && b.cap) VL_CUDA(cudaMemcpyAsync(np, b.p, b.cap * sizeof(T), cudaMemcpyDeviceToDevice, VL_STREAM(c)));
  if (b.p) { VL_CUDA(cudaStreamSynchronize(VL_STREAM(c))); vl_dev_free(c, b.p); }
  b.p = np; b.cap = ncap;
  return VLOAM_OK;
}

static inline int vl_div_up(long long a, long long b) { return (int)((a + b - 1) / b); }

// ---- stage entry points (one per .cu file) ------------------------------------
int vl_sr_run(vloam_b200_ctx* c, const float* d_xyz, int n, int stride);
int vl_sr_sync_counts(vloam_b200_ctx* c);
int vl_sr_exact_math(vloam_b200_ctx* c, const float* d_y, const float* d_x, int n, float* d_atan, float* d_atan2);
int vl_lo_run(vloam_b200_ctx* c, const double* prior_q, const double* prior_t, int use_prior);
int vl_lo_associate_only(vloam_b200_ctx* c, const double* x, int* corner_idx, int* surf_idx);
int vl_lo_build_last(vloam_b200_ctx* c, int set, const float4* corner, int nc, const float4* surf, int ns);
// What one solveMapping reads (LaserMapping::input, LM.cpp:178-209): the context's own odometry output, or the caller's
// (vloam_b200_laser_mapping_input).  los: device block whose q_w / t_w are q_wodom_curr / t_wodom_curr.
struct VlLmInput {
  const float4* corner; int nc;
  const float4* surf; int ns;
  const LoScalars* los;
  int skip;
  bool caller;  // the clouds are the caller's: filter them into the stacks here, superseding any filtered from the context's own
};
int vl_lm_run(vloam_b200_ctx* c, const VlLmInput& in);
// early: see laser_mapping.cu; ownClouds: the clouds are this sweep's odometry output (under VLOAM_FLAG_TRANSFORM_TO_END the filters wait for evEnd)
int vl_lm_enqueue_stacks(vloam_b200_ctx* c, const float4* corner, int nc, const float4* surf, int ns, bool early = false, bool ownClouds = true);
int vl_lm_enqueue_stacks_next(vloam_b200_ctx* c, const float4* corner, int nc, const float4* surf, int ns);  // into the spare stack buffers (helper thread)
int vl_lm_adopt_stacks_next(vloam_b200_ctx* c);  // make the spare stack buffers current
int vl_lm_publish_map(vloam_b200_ctx* c);         // queue the assembly of laserCloudMap (LM.cpp:884-899) on the publication stream
int vl_lm_get_map(vloam_b200_ctx* c, float* out, int cap_points);  // wait for it and copy it out
int vl_lm_pub_sync(vloam_b200_ctx* c);            // host wait for the last publication
void vl_lm_paths(vloam_b200_ctx* c, long long out[2]);  // mapped sweeps on the in-place / pool path since create
int vl_lm_init(vloam_b200_ctx* c);
void vl_lm_free(vloam_b200_ctx* c);
extern "C" int vl_launch_lookahead(vloam_b200_ctx* c);  // capi.cu: queue the registered look-ahead scan registration (no-op without one)
int vl_sr_set_attrs(vloam_b200_ctx* c);
int vl_sort_set_attrs(vloam_b200_ctx* c);
int vl_solver_set_attrs(vloam_b200_ctx* c);
int vl_lo_preload(vloam_b200_ctx* c);
int vl_lo_lookahead_solve(vloam_b200_ctx* c, bool flush = true, bool waitsIssued = false);   // part 1: queue the next sweep's odometry solve on its own stream (flush: issue the deferred side work first)
int vl_lo_plan_prebuild(vloam_b200_ctx* c);     // two sweeps ahead: plan the build of the next sweep's search structures as part of this call's side work
int vl_lo_early_lookahead(vloam_b200_ctx* c, bool* armed);  // ... and queue the next sweep's odometry before this sweep's mapping when its structures are pre-built
int vl_lo_lookahead_stacks(vloam_b200_ctx* c);  // part 2 (after S2 is recorded): the next sweep's stack filters, if its scan registration is done
int vl_lo_flush_deferred(vloam_b200_ctx* c);  // queue the deferred side-stream work of the last odometry call (look-ahead scan registration, next search structures)
int vl_vg_preload(vloam_b200_ctx* c);
int vl_lm_preload(vloam_b200_ctx* c);
int vl_lm_register_full(vloam_b200_ctx* c, const float4* d_in, int n, float4* d_out, int skip, bool toEnd);
// stage_inputs.cu: up to VL_PACK_MAX caller clouds of (stride, w_offset) float records into float4 buffers, on the main stream
#define VL_PACK_MAX 5
struct VlCloudIn { const float* src; int n; float4* dst; };
int vl_pack_clouds(vloam_b200_ctx* c, const VlCloudIn* clouds, int k, int stride, int w_offset, bool device);
int vl_lm_fit_sets(vloam_b200_ctx* c, const float* d_near, int n, int kind, int* d_ok, double* d_prm);  // vloam_b200_fit
int vl_lm_join(vloam_b200_ctx* c);      // wait until the helper thread has issued the pending map update; returns its status
int vl_lm_submit_task(vloam_b200_ctx* c, int (*fn)(vloam_b200_ctx*));  // hand a launch-issuing task to the helper thread (joins the previous one first)
int vl_lo_side_work(vloam_b200_ctx* c);  // the deferred side-stream work of the odometry stage (look-ahead scan registration, next search structures)
int vl_lo_submit_side(vloam_b200_ctx* c);  // ... issued by the helper thread while the caller queues the mapping
void vl_lm_shutdown(vloam_b200_ctx* c);  // stop the helper thread
int vl_lm_export_map(vloam_b200_ctx* c, int which, void* out, long cap, long* bytes);
int vl_lm_sync_pools(vloam_b200_ctx* c);  // write the in-place grid updates back to the cube pools (no-op when they are current)
int vl_lm_import_map(vloam_b200_ctx* c, int which, const void* data, long bytes);
// prior maps (vloam_b200_load_map, set_map_pose, set_map_update, get_map_kind)
int vl_lm_load_map(vloam_b200_ctx* c, const float* corner, int nc, const float* surf, int ns, int stride, int w_offset, bool device,
                   long long dropped[2]);
int vl_lm_set_map_pose(vloam_b200_ctx* c, const double q[4], const double t[3]);
void vl_lm_set_map_update(vloam_b200_ctx* c, bool enabled);
int vl_lm_get_map_kind(vloam_b200_ctx* c, int which, float* out, int cap_points);
// relocalization (relocalize.cu): vloam_b200_relocalize on a drained context, its debug getters (rl.*) and its state
int vl_rl_run(vloam_b200_ctx* c, const vloam_b200_reloc_params& p, const double q_c[4], const double t_c[3], vloam_b200_reloc_result* res);
long vl_rl_debug(vloam_b200_ctx* c, const char* name, void* out, long cap);
void vl_rl_free(vloam_b200_ctx* c);

// sort / voxel primitives (voxel_grid.cu)
int vl_sort_u64(vloam_b200_ctx* c, unsigned long long* d_keys, int n_pow2);
// pcl::VoxelGrid of d_in[0..n) -> d_out, count written to *d_count (device int); n is a host bound,
// d_n (device int, may be null) is the actual count.
int vl_voxel_grid_device(vloam_b200_ctx* c, const float4* d_in, int n, const int* d_n, float leaf, float4* d_out, int* d_count, int lane = 0);

// solver (lm_solver.cu): evaluates factor slots [0, nslots) with validity flags.
// nslots: host bound on the factor slots; d_nslots (device, may be null): actual count, min() of both is used
// d_s (device, may be null): per-slot interpolation ratio; non-null = the functors slerp q by s and scale t by s (DISTORTION)
int vl_solve(vloam_b200_ctx* c, int nslots, const int* d_nslots, double* d_x_inout, double* costs2 /* host, may be null */,
             int hint = 0 /* last known actual slot count, 0 = none */, const double* d_s = nullptr);
int vl_solve_buf(vloam_b200_ctx* c, const double* d_factors, const int* d_valid, int nslots, const int* d_nslots, double* d_x_inout, double* costs2, int hint,
                 const double* d_s, int ncta = 16);  // same on explicit factor buffers; ncta: CTAs of the solver's cluster (8 or 16: it fixes the summation order), on the calling thread's current stream (VL_STREAM)
int vl_evaluate_once(vloam_b200_ctx* c, int nslots, const double* d_x, EvalOut* d_out, const double* d_s = nullptr);
static inline bool vl_distortion(const vloam_b200_ctx* c) { return (c->prm.reserved & 1) != 0; }  // LaserOdometry::DISTORTION (LO.h:90)
static inline bool vl_to_end(const vloam_b200_ctx* c) { return (c->prm.reserved & VLOAM_FLAG_TRANSFORM_TO_END) != 0; }  // LO.cpp:537-556 enabled
int vl_lo_to_end_cloud(vloam_b200_ctx* c, const float4* d_in, int n, float4* d_out);  // TransformToEnd of n points with this sweep's q/t_last_curr

// ---- shared device helpers -----------------------------------------------------
#ifdef __CUDACC__
// Eigen quaternion * vector (no normalisation): uv = u x v; uv += uv; v + w*uv + u x uv.
__device__ __forceinline__ void vl_qrot(const double q[4], double vx, double vy, double vz, double o[3]) {
  const double ux = q[0], uy = q[1], uz = q[2], w = q[3];
  double uvx = uy * vz - uz * vy;
  double uvy = uz * vx - ux * vz;
  double uvz = ux * vy - uy * vx;
  uvx += uvx; uvy += uvy; uvz += uvz;
  const double cx = uy * uvz - uz * uvy;
  const double cy = uz * uvx - ux * uvz;
  const double cz = ux * uvy - uy * uvx;
  o[0] = (vx + w * uvx) + cx;
  o[1] = (vy + w * uvy) + cy;
  o[2] = (vz + w * uvz) + cz;
}
__device__ __forceinline__ void vl_qmul(const double a[4], const double b[4], double o[4]) {
  const double ax = a[0], ay = a[1], az = a[2], aw = a[3];
  const double bx = b[0], by = b[1], bz = b[2], bw = b[3];
  const double w = aw * bw - ax * bx - ay * by - az * bz;
  const double x = aw * bx + ax * bw + ay * bz - az * by;
  const double y = aw * by + ay * bw + az * bx - ax * bz;
  const double z = aw * bz + az * bw + ax * by - ay * bx;
  o[0] = x; o[1] = y; o[2] = z; o[3] = w;
}
// transformUpdate (LM.cpp:147-151): q_wmap_wodom = q_w_curr * q_wodom_curr.inverse() (Eigen's conjugate / squaredNorm),
// t_wmap_wodom = t_w_curr - q_wmap_wodom * t_wodom_curr; pose = {q_w_curr, t_w_curr}
__device__ __forceinline__ void vl_transform_update(const double pose[7], const double q_wodom[4], const double t_wodom[3], double q_out[4], double t_out[3]) {
  const double* q = q_wodom;
  const double n2 = q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3];
  const double qi[4] = {-q[0] / n2, -q[1] / n2, -q[2] / n2, q[3] / n2};
  vl_qmul(pose, qi, q_out);
  double r[3];
  vl_qrot(q_out, t_wodom[0], t_wodom[1], t_wodom[2], r);
  for (int k = 0; k < 3; ++k) t_out[k] = pose[4 + k] - r[k];
}
// Eigen::Quaterniond::Identity().slerp(t, q) (Eigen/src/Geometry/Quaternion.h), used by TransformToStart and the odometry
// functors when DISTORTION is on (LO.cpp:163, LF.hpp:29-33, 86-90): d = w; |d| >= 1 - eps -> (1 - t) I + t q, else
// theta = acos(|d|), scale0 = sin((1 - t) theta) / sin(theta), scale1 = sin(t theta) / sin(theta); d < 0 flips scale1.
__device__ __forceinline__ void vl_slerp_identity(double t, const double q[4], double out[4]) {
  const double one = 1.0 - 2.220446049250313e-16;
  const double d = q[3], absD = fabs(d);
  double scale0, scale1;
  if (absD >= one) { scale0 = 1.0 - t; scale1 = t; }
  else {
    const double theta = acos(absD), sinTheta = sin(theta);
    scale0 = sin((1.0 - t) * theta) / sinTheta;
    scale1 = sin(t * theta) / sinTheta;
  }
  if (d < 0.0) scale1 = -scale1;
  out[0] = scale1 * q[0]; out[1] = scale1 * q[1]; out[2] = scale1 * q[2]; out[3] = scale0 + scale1 * q[3];
}
// interpolation ratio of a point: (intensity - int(intensity)) is a float, SCAN_PERIOD a double (LO.cpp:156-160)
__device__ __forceinline__ double vl_point_s(float intensity) { return (double)__fsub_rn(intensity, (float)(int)intensity) / 0.1; }
// TransformToStart (LO.cpp:152-173): pose = {q_last_curr, t_last_curr}; deskew: slerp(s, q), s * t with s from the point
__device__ __forceinline__ void vl_transform_to_start(const double* pose, const float4 p, int deskew, float& sx, float& sy, float& sz) {
  double r[3];
  if (deskew) {
    const double s = vl_point_s(p.w);
    double qs[4];
    vl_slerp_identity(s, pose, qs);
    vl_qrot(qs, (double)p.x, (double)p.y, (double)p.z, r);
    sx = (float)(r[0] + s * pose[4]); sy = (float)(r[1] + s * pose[5]); sz = (float)(r[2] + s * pose[6]);
  } else {
    vl_qrot(pose, (double)p.x, (double)p.y, (double)p.z, r);
    sx = (float)(r[0] + pose[4]); sy = (float)(r[1] + pose[5]); sz = (float)(r[2] + pose[6]);
  }
}
// TransformToEnd (LO.cpp:176-193): un = TransformToStart(p) stored as float, then q_last_curr.inverse() * (un - t_last_curr) in
// double, stored as float; intensity = int(intensity).  inverse() is Eigen's conjugate / squaredNorm (q is not exactly unit after
// the solver's update), `*` Eigen's _transformVector (vl_qrot).
__device__ __forceinline__ float4 vl_transform_to_end(const double* pose, const float4 p, int deskew) {
  float ux, uy, uz;
  vl_transform_to_start(pose, p, deskew, ux, uy, uz);
  const double n2 = pose[0] * pose[0] + pose[1] * pose[1] + pose[2] * pose[2] + pose[3] * pose[3];
  const double qi[4] = {-pose[0] / n2, -pose[1] / n2, -pose[2] / n2, pose[3] / n2};
  double r[3];
  vl_qrot(qi, (double)ux - pose[4], (double)uy - pose[5], (double)uz - pose[6], r);
  return make_float4((float)r[0], (float)r[1], (float)r[2], (float)(int)p.w);
}

// Visit every element of up to 32 index ranges of ARRAY (float4) with all lanes busy, 128 elements per step.
// Lane r owns range [myBeg, myBeg + myLen) (myLen = 0 when it has none), so the look-ups that produced
// the ranges were issued together (one memory latency, not one per range).  Non-empty ranges are compacted
// onto lanes 0..nr-1 with their exclusive prefix; the range owning each of the 32 consecutive flattened
// positions of a sub-step then follows from one ballot (ranges starting at or before the sub-step) and
// one warp OR-reduction (bit i: a range starts at position base + i) -- registers only, no search.  The
// four loads of a step are issued before any is used: a query warp has few sibling warps to hide the L2
// latency behind.  BODY sees `const float4 t` and `const int p` (its index in ARRAY).
#define VL_WARP_VISIT_FLAT(myBeg, myLen, lane, ARRAY, BODY)                                                    \
  do {                                                                                                         \
    int inc_ = (myLen);                                                                                        \
    for (int d_ = 1; d_ < 32; d_ <<= 1) { const int t_ = __shfl_up_sync(0xffffffffu, inc_, d_); if ((lane) >= d_) inc_ += t_; } \
    const int total_ = __shfl_sync(0xffffffffu, inc_, 31);                                                     \
    if (total_ <= 0) break;                                                                                    \
    const unsigned ne_ = __ballot_sync(0xffffffffu, (myLen) > 0);                                              \
    const int nr_ = __popc(ne_);                                                                               \
    const int src_ = (lane) < nr_ ? (int)__fns(ne_, 0, (lane) + 1) : 0;                                        \
    const int cbeg_ = __shfl_sync(0xffffffffu, (myBeg), src_);                                                 \
    int cexc_ = __shfl_sync(0xffffffffu, inc_ - (myLen), src_);                                                \
    if ((lane) >= nr_) cexc_ = 0x7fffffff;                                                                     \
    const int safe_ = __shfl_sync(0xffffffffu, cbeg_, 0);                                                      \
    for (int base_ = 0; base_ < total_; base_ += 128) {                                                        \
      int p4_[4]; bool ok4_[4];                                                                                \
      _Pragma("unroll")                                                                                        \
      for (int u_ = 0; u_ < 4; ++u_) {                                                                         \
        const int b_ = base_ + 32 * u_;                                                                        \
        const int cnt0_ = __popc(__ballot_sync(0xffffffffu, cexc_ <= b_));                                     \
        const unsigned st_ = __reduce_or_sync(0xffffffffu, (cexc_ > b_ && cexc_ < b_ + 32) ? (1u << (cexc_ - b_)) : 0u); \
        const int k_ = max(cnt0_ - 1 + __popc(st_ & ((2u << (lane)) - 1u)), 0) & 31;                           \
        const int rb_ = __shfl_sync(0xffffffffu, cbeg_, k_), ro_ = __shfl_sync(0xffffffffu, cexc_, k_);        \
        const int idx_ = b_ + (lane);                                                                          \
        ok4_[u_] = idx_ < total_;                                                                              \
        p4_[u_] = ok4_[u_] ? rb_ + (idx_ - ro_) : safe_;                                                       \
      }                                                                                                        \
      const float4 t0_ = __ldg(&(ARRAY)[p4_[0]]), t1_ = __ldg(&(ARRAY)[p4_[1]]);                               \
      const float4 t2_ = __ldg(&(ARRAY)[p4_[2]]), t3_ = __ldg(&(ARRAY)[p4_[3]]);                               \
      if (ok4_[0]) { const float4 t = t0_; const int p = p4_[0]; (void)p; BODY }                               \
      if (ok4_[1]) { const float4 t = t1_; const int p = p4_[1]; (void)p; BODY }                               \
      if (ok4_[2]) { const float4 t = t2_; const int p = p4_[2]; (void)p; BODY }                               \
      if (ok4_[3]) { const float4 t = t3_; const int p = p4_[3]; (void)p; BODY }                               \
    }                                                                                                          \
  } while (0)

// Exclusive scan of one int per thread over a block of T threads (T a multiple of 32, <= 1024; every thread calls):
// warp shuffles, the T/32 warp totals through `ws` (>= 32 ints of shared memory) and a second shuffle scan by warp 0:
// three barriers, where a Hillis-Steele ladder over 1024 entries takes twenty.  *total (may be null) = block sum.
template <int T>
__device__ __forceinline__ int vl_block_excl_scan(int v, int* ws, int* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int inc = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) { const int u = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += u; }
  if (lane == 31) ws[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    int x = lane < T / 32 ? ws[lane] : 0;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const int u = __shfl_up_sync(0xffffffffu, x, d); if (lane >= d) x += u; }
    ws[lane] = x;
  }
  __syncthreads();
  const int before = warp > 0 ? ws[warp - 1] : 0;
  if (total) *total = ws[T / 32 - 1];
  __syncthreads();
  return before + inc - v;
}

// FLANN L2_Simple<float>: acc = 0; acc += d*d over x, y, z (f32, no FMA: -fmad=false).
__device__ __forceinline__ float vl_dist2(float qx, float qy, float qz, float px, float py, float pz) {
  float acc = 0.f, d;
  d = qx - px; acc += d * d;
  d = qy - py; acc += d * d;
  d = qz - pz; acc += d * d;
  return acc;
}
#endif

// capi.cu -- the C ABI of include/vloam_b200.h on top of the stage files.
#include <stdlib.h>
#include <string>
#include <vector>
#include "common.cuh"

static bool g_capture_default = false;
// stage files ask through this hook whether to keep per-pass association snapshots
bool vl_debug_capture(const vloam_b200_ctx* c) { return c->h_vScalars && c->h_vScalars[0] != 0; }
int vl_lm_rescan_sorted(vloam_b200_ctx* c);
int vl_solver_trace(vloam_b200_ctx* c, long long* out16);
int vl_lo_trace(vloam_b200_ctx* c, int* out, int n);
int vl_sr_trace(vloam_b200_ctx* c, long long* out, int n);

extern "C" {

void vloam_b200_default_params(vloam_b200_params* p) {
  p->n_scans = 64; p->minimum_range = 5.0f; p->line_res = 0.4f; p->plane_res = 0.8f; p->mapping_skip_frame = 1; p->reserved = 0;
}

const char* vloam_b200_last_error(const vloam_b200_ctx* c) { return c ? c->err : "null context"; }

#define VL_CUDA_CREATE(call)                                                                                       \
  do {                                                                                                             \
    cudaError_t e_ = (call);                                                                                       \
    if (e_ != cudaSuccess) { fprintf(stderr, "vloam_b200_create: %s: %s\n", #call, cudaGetErrorString(e_)); return VLOAM_E_CUDA; } \
  } while (0)

// fixed-size arrays, counters and the completion event of one scan-registration field set (VL_SR_FIELDS)
static int alloc_sr_fixed(vloam_b200_ctx* c) {
  const int R = VL_MAX_RINGS, S = VL_MAX_RINGS * VL_SECTORS;
  VL_CUDA_CREATE(cudaEventCreateWithFlags(&c->evSR, cudaEventDisableTiming));
  VL_CUDA_CREATE(cudaEventCreateWithFlags(&c->evSRfeat, cudaEventDisableTiming));
  VL_CUDA_CREATE(cudaMalloc(&c->ringCount, sizeof(int) * R));
  VL_CUDA_CREATE(cudaMalloc(&c->ringStart, sizeof(int) * (R + 1)));
  VL_CUDA_CREATE(cudaMemset(c->ringCount, 0, sizeof(int) * R));
  VL_CUDA_CREATE(cudaMemset(c->ringStart, 0, sizeof(int) * (R + 1)));
  VL_CUDA_CREATE(cudaMalloc(&c->srs, sizeof(SrScalars)));
  VL_CUDA_CREATE(cudaMemset(c->srs, 0, sizeof(SrScalars)));
  VL_CUDA_CREATE(cudaMallocHost(&c->h_srs, sizeof(SrScalars)));
  memset(c->h_srs, 0, sizeof(SrScalars));
  VL_CUDA_CREATE(cudaMalloc(&c->provSharp, sizeof(int) * S * 2));
  VL_CUDA_CREATE(cudaMalloc(&c->provLess, sizeof(int) * S * 20));
  VL_CUDA_CREATE(cudaMalloc(&c->provFlat, sizeof(int) * S * 4));
  int** smalls[] = {&c->cntSharp, &c->cntLess, &c->cntFlat, &c->offSharp, &c->offLess, &c->offFlat};
  for (int** q : smalls) { VL_CUDA_CREATE(cudaMalloc(q, sizeof(int) * S)); VL_CUDA_CREATE(cudaMemset(*q, 0, sizeof(int) * S)); }
  VL_CUDA_CREATE(cudaMalloc(&c->ringDsCount, sizeof(int) * R));
  VL_CUDA_CREATE(cudaMalloc(&c->ringDsOff, sizeof(int) * R));
  c->sr_counts_valid = false; c->n_in = 0; c->nKept = c->nSharp = c->nLessSharp = c->nFlat = c->nLessFlat = 0;
  return VLOAM_OK;
}
static void free_sr_set(vloam_b200_ctx* c) {  // the set currently swapped into the context
  void* dev[] = {c->ringCount, c->ringStart, c->srs, c->provSharp, c->provLess, c->provFlat, c->cntSharp, c->cntLess, c->cntFlat, c->offSharp,
                 c->offLess, c->offFlat, c->ringDsCount, c->ringDsOff, c->in.p, c->ring.p, c->ori.p, c->blockHist.p, c->cloud.p, c->curv.p,
                 c->label.p, c->picked.p, c->sortScratch.p, c->lessFlatProv.p, c->selIdx.p, c->sharp.p, c->flat.p};
  for (void* p : dev) vl_dev_free(c, p);
  if (c->h_srs) cudaFreeHost(c->h_srs);
  if (c->evSR) cudaEventDestroy(c->evSR);
  if (c->evSRfeat) cudaEventDestroy(c->evSRfeat);
}

static int create_impl(vloam_b200_ctx* c, const vloam_b200_params* p, int device);

int vloam_b200_create(const vloam_b200_params* p, int device, vloam_b200_ctx** out) {
  if (!p || !out) return VLOAM_E_INVALID;
  *out = nullptr;
  // SR.cpp:58-61, 255-259: only 16 / 32 / 64 beams (128 = builder extension)
  if (p->n_scans != 16 && p->n_scans != 32 && p->n_scans != 64 && p->n_scans != 128) return VLOAM_E_INVALID;
  if (!(p->line_res >= 0.05f) || !(p->plane_res >= 0.05f) || p->mapping_skip_frame < 1) return VLOAM_E_INVALID;
  if (p->reserved & ~(VLOAM_FLAG_DISTORTION | VLOAM_FLAG_TRANSFORM_TO_END)) return VLOAM_E_INVALID;
  VL_CUDA_CREATE(cudaSetDevice(device));
  vloam_b200_ctx* c = new vloam_b200_ctx();  // value-initialised: every pointer / handle starts out null
  const int r = create_impl(c, p, device);
  if (r != VLOAM_OK) { vloam_b200_destroy(c); (void)cudaGetLastError(); return r; }  // destroy tolerates a half-built context: nothing leaks
  *out = c;
  return VLOAM_OK;
}

static int create_impl(vloam_b200_ctx* c, const vloam_b200_params* p, int device) {
  c->prm = *p; c->device = device; c->err[0] = 0; c->launches = 0; c->worker = nullptr; c->timing = false; c->cur = 0;
  c->sr_counts_valid = false; c->n_in = 0; c->lo_inited = false; c->lo_frameCount = 0; c->lm_frameCount = 0; c->lm_optimized = 0; c->skip_frame = false;
  c->nKept = c->nSharp = c->nLessSharp = c->nFlat = c->nLessFlat = 0; c->nCornerLast = c->nSurfLast = 0;
  c->cornerLastPtr = nullptr; c->surfLastPtr = nullptr;
  for (int k = 0; k < 4; ++k) c->dbgLoCost[k] = c->dbgLmCost[k] = 0;
  for (int k = 0; k < 3; ++k) c->stage_ms[k] = 0;
  c->prof_name[0] = 0; c->prof_n = 0; c->prof_created = 0; c->prof_bytes = 0; c->prof_next_bytes = 0;
  {  // the arena behind vl_reserve (common.cuh); VLOAM_ARENA_MB = 0 turns it off (every buffer its own cudaMalloc)
    const char* e = getenv("VLOAM_ARENA_MB");
    const size_t mb = e ? (size_t)max(atoll(e), 0LL) : 1024;
    c->arena = nullptr; c->arenaCap = 0; c->arenaTop = 0;
    if (mb) { VL_CUDA_CREATE(cudaMalloc(&c->arena, mb << 20)); c->arenaCap = mb << 20; }
  }
  cudaDeviceProp prop;
  VL_CUDA_CREATE(cudaGetDeviceProperties(&prop, device));
  c->num_sms = prop.multiProcessorCount;
  // Stream priorities: the pose chain (main stream) goes first, the stack filters it waits on next, and the work
  // that only has to be ready for the NEXT sweep (map update, speculative sub-map, look-ahead scan registration)
  // last -- when SMs free up, blocks of the solver's 16-CTA cluster are placed before the streaming grids' blocks.
  // VLOAM_NO_PRIORITIES=1: all streams at the default priority.
  int prLow = 0, prHigh = 0;
  VL_CUDA_CREATE(cudaDeviceGetStreamPriorityRange(&prLow, &prHigh));
  // (round 2: the in-place map update is ~3 short kernels the NEXT sweep's mapping waits for directly: it runs at the pose chain's priority)
  // ... and so does the look-ahead scan registration: the NEXT sweep's odometry (own stream, beside this sweep's mapping) starts when it is done
  int lv[4] = {2, 1, 2, 2};  // levels above the lowest priority: main | stack filters | map update | look-ahead scan registration
  int lvLO = 2;                // the look-ahead odometry stream
  if (const char* e = getenv("VLOAM_PRIO")) sscanf(e, "%d,%d,%d,%d,%d", &lv[0], &lv[1], &lv[2], &lv[3], &lvLO);
  if (getenv("VLOAM_NO_PRIORITIES")) lv[0] = lv[1] = lv[2] = lv[3] = lvLO = 0;
  int pr[5];
  for (int k = 0; k < 4; ++k) pr[k] = max(prLow - lv[k], prHigh);  // (numerically lower = more urgent)
  pr[4] = max(prLow - lvLO, prHigh);
  VL_CUDA_CREATE(cudaStreamCreateWithPriority(&c->stream, cudaStreamNonBlocking, pr[0]));
  VL_CUDA_CREATE(cudaStreamCreateWithPriority(&c->stream2, cudaStreamNonBlocking, pr[1]));
  VL_CUDA_CREATE(cudaStreamCreateWithPriority(&c->stream3, cudaStreamNonBlocking, pr[2]));
  VL_CUDA_CREATE(cudaStreamCreateWithPriority(&c->stream4, cudaStreamNonBlocking, pr[1]));
  VL_CUDA_CREATE(cudaEventCreateWithFlags(&c->evStacksC, cudaEventDisableTiming));
  VL_CUDA_CREATE(cudaStreamCreateWithPriority(&c->streamAux, cudaStreamNonBlocking, pr[2]));
  VL_CUDA_CREATE(cudaEventCreateWithFlags(&c->evAux, cudaEventDisableTiming));
  VL_CUDA_CREATE(cudaEventCreateWithFlags(&c->evAuxZero, cudaEventDisableTiming));
  VL_CUDA_CREATE(cudaEventCreateWithFlags(&c->evUpd, cudaEventDisableTiming));
  VL_CUDA_CREATE(cudaEventCreateWithFlags(&c->evStacks, cudaEventDisableTiming));
  VL_CUDA_CREATE(cudaEventCreateWithFlags(&c->evLast, cudaEventDisableTiming));
  VL_CUDA_CREATE(cudaEventCreateWithFlags(&c->evPose, cudaEventDisableTiming));
  VL_CUDA_CREATE(cudaEventCreateWithFlags(&c->evMap, cudaEventDisableTiming));
  VL_CUDA_CREATE(cudaEventCreateWithFlags(&c->evKeys, cudaEventDisableTiming));
  for (int k = 0; k < 2; ++k) VL_CUDA_CREATE(cudaEventCreateWithFlags(&c->evKeysSel[k], cudaEventDisableTiming));
  c->stacksReady = false; c->lm_reset_pending = true; c->lastSet = 0; c->loGridValid[0] = c->loGridValid[1] = false;
  for (int k = 0; k < 4; ++k) VL_CUDA_CREATE(cudaEventCreate(&c->ev[k]));
  for (int k = 0; k < 12; ++k) { VL_CUDA_CREATE(cudaEventCreate(&c->evx[k])); VL_CUDA_CREATE(cudaEventRecord(c->evx[k], c->stream)); }
  VL_TRY(alloc_sr_fixed(c));
  c->srNext = new SrSet();
  vl_sr_swap(c, *c->srNext);      // the spare set gets its own fixed-size arrays, counters and event
  { const int r_ = alloc_sr_fixed(c); vl_sr_swap(c, *c->srNext); if (r_ != VLOAM_OK) return r_; }
  c->srNext2 = new SrSet();
  vl_sr_swap(c, *c->srNext2);
  { const int r_ = alloc_sr_fixed(c); vl_sr_swap(c, *c->srNext2); if (r_ != VLOAM_OK) return r_; }
  c->srNextKey = c->srNext2Key = nullptr; c->srNextValid = c->srNext2Valid = false; c->srPendCount = 0;
  VL_CUDA_CREATE(cudaStreamCreateWithPriority(&c->streamSR, cudaStreamNonBlocking, pr[3]));
  VL_CUDA_CREATE(cudaMalloc(&c->los, sizeof(LoScalars)));
  VL_CUDA_CREATE(cudaMalloc(&c->losNext, sizeof(LoScalars)));
  VL_CUDA_CREATE(cudaEventCreateWithFlags(&c->evS2, cudaEventDisableTiming));
  VL_CUDA_CREATE(cudaMallocHost(&c->h_s2flag, 64)); *c->h_s2flag = 0; c->s2seq = 0;
  VL_CUDA_CREATE(cudaEventCreateWithFlags(&c->evLoSolve, cudaEventDisableTiming));
  VL_CUDA_CREATE(cudaEventCreateWithFlags(&c->evLoNext, cudaEventDisableTiming));
  VL_CUDA_CREATE(cudaEventCreateWithFlags(&c->evEnd, cudaEventDisableTiming));
  VL_CUDA_CREATE(cudaStreamCreateWithPriority(&c->streamLO, cudaStreamNonBlocking, pr[4]));
  c->loNextValid = c->loNextQueued = c->srAdopted = c->s2Done = false; c->loAssumeMonotone = c->inProcessFrame = c->loDeferred = false; c->srDeferred = c->sideSubmitted = false; c->preDeferred = c->loPreValid = c->sideWaitsIssued = c->earlyLoArmed = c->stacksAdopted = false; c->loNextSet = 0; c->stackSel = 0; c->stacksNextReady = false;
  VL_CUDA_CREATE(cudaMallocHost(&c->h_los, sizeof(LoScalars)));
  LoScalars hl; memset(&hl, 0, sizeof hl); hl.para_q[3] = 1.0; hl.q_w[3] = 1.0;  // LO.cpp:81-91
  VL_CUDA_CREATE(cudaMemcpy(c->los, &hl, sizeof hl, cudaMemcpyHostToDevice));
  *c->h_los = hl;
  VL_CUDA_CREATE(cudaMalloc(&c->loRingTbl, sizeof(int) * 4 * 160));
  VL_CUDA_CREATE(cudaMalloc(&c->evalOut, sizeof(EvalOut)));
  VL_CUDA_CREATE(cudaMalloc(&c->lms, sizeof(LmSolveState)));
  VL_CUDA_CREATE(cudaMemset(c->lms, 0, sizeof(LmSolveState)));
  VL_CUDA_CREATE(cudaMallocHost(&c->h_lms, sizeof(LmSolveState)));
  VL_CUDA_CREATE(cudaMalloc(&c->lmm, sizeof(LmScalars)));
  VL_CUDA_CREATE(cudaMallocHost(&c->h_lmm, sizeof(LmScalars)));
  memset(c->h_lmm, 0, sizeof(LmScalars));
  VL_CUDA_CREATE(cudaMalloc(&c->cubeC, sizeof(MapCubeTable)));
  VL_CUDA_CREATE(cudaMalloc(&c->cubeS, sizeof(MapCubeTable)));
  VL_CUDA_CREATE(cudaMalloc(&c->vScalars, sizeof(int) * 256));
  VL_CUDA_CREATE(cudaMemset(c->vScalars, 0, sizeof(int) * 256));
  VL_CUDA_CREATE(cudaMallocHost(&c->h_vScalars, sizeof(int) * 256));
  memset(c->h_vScalars, 0, sizeof(int) * 256);
  c->h_vScalars[0] = g_capture_default ? 1 : 0;
  int r = vl_lm_init(c);
  if (r == VLOAM_OK) r = vl_sr_set_attrs(c);
  if (r == VLOAM_OK) r = vl_sort_set_attrs(c);
  if (r == VLOAM_OK) r = vl_solver_set_attrs(c);
  if (r == VLOAM_OK) r = vl_lo_preload(c);
  if (r == VLOAM_OK) r = vl_vg_preload(c);
  if (r == VLOAM_OK) r = vl_lm_preload(c);
  if (r != VLOAM_OK) { fprintf(stderr, "vloam_b200_create: %s\n", c->err); return r; }
  VL_CUDA_CREATE(cudaDeviceSynchronize());
  return VLOAM_OK;
}

void vloam_b200_destroy(vloam_b200_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  vl_lm_shutdown(c);
  cudaStreamSynchronize(c->stream); cudaStreamSynchronize(c->stream2); cudaStreamSynchronize(c->stream3); cudaStreamSynchronize(c->stream4);
  // Device memory is released wholesale: contexts live for a whole replay (MAIN.cpp:118-124).
  cudaStreamSynchronize(c->streamSR);
  free_sr_set(c);
  if (c->srNext) { vl_sr_swap(c, *c->srNext); free_sr_set(c); delete c->srNext; c->srNext = nullptr; }
  if (c->srNext2) { vl_sr_swap(c, *c->srNext2); free_sr_set(c); delete c->srNext2; c->srNext2 = nullptr; }
  cudaStreamDestroy(c->streamSR);
  vl_lm_free(c);
  if (c->streamLO) { cudaStreamSynchronize(c->streamLO); cudaStreamDestroy(c->streamLO); }
  cudaEventDestroy(c->evS2); cudaEventDestroy(c->evLoSolve); cudaEventDestroy(c->evLoNext); if (c->evEnd) cudaEventDestroy(c->evEnd);
  void* singles[] = {c->los, c->losNext, c->evalOut, c->lms, c->lmm, c->cubeC, c->cubeS, c->vScalars, c->loRingTbl, c->loGridCells[0].p, c->loGridCells[1].p,
                     c->loGridCellOf.p, c->loGridSorted[0].p, c->loGridSorted[1].p, c->dbgLoCorner[0].p, c->dbgLoCorner[1].p, c->dbgLoSurf[0].p,
                     c->dbgLoSurf[1].p, c->dbgKnnIdx[0][0].p, c->dbgKnnIdx[0][1].p, c->dbgKnnIdx[1][0].p, c->dbgKnnIdx[1][1].p, c->dbgKnnD2[0][0].p,
                     c->dbgKnnD2[0][1].p, c->dbgKnnD2[1][0].p, c->dbgKnnD2[1][1].p, c->dbgKnnOk[0][0].p, c->dbgKnnOk[0][1].p, c->dbgKnnOk[1][0].p,
                     c->dbgKnnOk[1][1].p};
  for (void* p : singles) vl_dev_free(c, p);
  void* bufs[] = {c->lessSharp[0].p, c->lessSharp[1].p, c->lessSharp[2].p, c->lessFlat[0].p, c->lessFlat[1].p, c->lessFlat[2].p, c->endSharp[0].p, c->endSharp[1].p, c->endSharp[2].p, c->endFlat[0].p, c->endFlat[1].p, c->endFlat[2].p, c->loCornerIdx.p, c->loSurfIdx.p, c->factors.p, c->factorS.p, c->factorValid.p, c->loFactors.p, c->loFactorValid.p, c->evalPartials.p,
                  c->poolC.p, c->poolS.p, c->stackC.p, c->stackS.p, c->stackCN.p, c->stackSN.p, c->fromMapC.p, c->fromMapS.p, c->knnD2.p, c->knnOk.p,
                  c->vKeys.p, c->vKeys2.p, c->vHead.p, c->vScan.p, c->vScan2.p, c->vOut.p, c->vIn.p, c->regOut.p, c->tailKeys.p, c->staging.p};
  for (void* p : bufs) vl_dev_free(c, p);
  if (c->h_s2flag) cudaFreeHost(c->h_s2flag);
  cudaFreeHost(c->h_los); cudaFreeHost(c->h_lms); cudaFreeHost(c->h_lmm); cudaFreeHost(c->h_vScalars);
  for (int k = 0; k < 4; ++k) cudaEventDestroy(c->ev[k]);
  for (int k = 0; k < 12; ++k) cudaEventDestroy(c->evx[k]);
  cudaStreamSynchronize(c->stream2); cudaStreamSynchronize(c->stream3);
  cudaEventDestroy(c->evStacks); cudaEventDestroy(c->evLast); cudaEventDestroy(c->evPose); cudaEventDestroy(c->evMap); cudaEventDestroy(c->evKeys); cudaEventDestroy(c->evKeysSel[0]); cudaEventDestroy(c->evKeysSel[1]);
  cudaEventDestroy(c->evStacksC);
  cudaStreamSynchronize(c->streamAux); cudaEventDestroy(c->evAux); cudaEventDestroy(c->evAuxZero); cudaEventDestroy(c->evUpd); cudaStreamDestroy(c->streamAux);
  cudaStreamDestroy(c->stream2); cudaStreamDestroy(c->stream3); cudaStreamDestroy(c->stream4);
  cudaStreamDestroy(c->stream);
  if (c->arena) cudaFree(c->arena);
  delete c;
}

int vloam_b200_begin_frame(vloam_b200_ctx* c) {
  if (!c) return VLOAM_E_INVALID;  // ABI boundary: a null context is the caller's error, not a crash
  VL_CUDA(cudaSetDevice(c->device));
  c->lm_reset_pending = true;  // applied by the next solveMapping (the map update of the previous frame may still be reading the list)
  return VLOAM_OK;
}

// Look-ahead for replays: register the NEXT sweep -- or the next TWO sweeps, in order -- (device or host pointer).  The upload
// and scan registration of a registered sweep are queued on a side stream from inside the processing of the current sweep, into
// a spare field set, so they run underneath this sweep's odometry and mapping; the scan_registration / process_frame call that
// comes with the same (pointer, n, stride) finds the work done.  With two sweeps registered, the odometry of sweep k+1 (whose
// scan registration ran during sweep k-1) starts at once beside the mapping of sweep k while sweep k+2 is uploaded and
// registered: nothing of the chain upload -> scan registration -> odometry is left on the critical path.  A call with any other
// buffer drops what was registered.  A registered buffer must stay valid and unchanged until the call that processes it;
// registering a buffer that is already registered is a no-op.  No reference counterpart: the bag player hands over one sweep at
// a time (MAIN.cpp:143).
static int register_pending(vloam_b200_ctx* c, const float* key, int n, int stride, bool dev) {
  if (n <= 0 || stride < 3 || !key) { snprintf(c->err, sizeof c->err, "bad cloud shape"); return VLOAM_E_INVALID; }
  if (c->srNextValid && key == c->srNextKey && n == c->srNextN && stride == c->srNextStride) return VLOAM_OK;
  if (c->srNext2Valid && key == c->srNext2Key && n == c->srNext2N && stride == c->srNext2Stride) return VLOAM_OK;
  for (int k = 0; k < c->srPendCount; ++k)
    if (c->srPend[k].key == key && c->srPend[k].n == n && c->srPend[k].stride == stride) return VLOAM_OK;
  if (c->srPendCount == 2) c->srPendCount = 1;  // more than two ahead: the newest registration replaces the last one
  c->srPend[c->srPendCount].key = key; c->srPend[c->srPendCount].n = n; c->srPend[c->srPendCount].stride = stride; c->srPend[c->srPendCount].dev = dev;
  c->srPendCount++;
  return VLOAM_OK;
}
int vloam_b200_prefetch_scan_device(vloam_b200_ctx* c, const float* d_xyz, int n, int stride) {
  if (!c) return VLOAM_E_INVALID;  // ABI boundary: a null context is the caller's error, not a crash
  return register_pending(c, d_xyz, n, stride, true);
}
int vloam_b200_prefetch_scan(vloam_b200_ctx* c, const float* xyz, int n, int stride) {
  if (!c) return VLOAM_E_INVALID;  // ABI boundary: a null context is the caller's error, not a crash
  return register_pending(c, xyz, n, stride, false);
}

// queue the registered look-ahead sweeps: spare set swapped in, upload + scan registration on streamSR, set swapped back out.
// Called by the odometry stage once its own kernels are queued (the host would only wait at S1 otherwise): issuing
// these ~10 launches before the odometry delays the sweep that is being processed.
int vl_launch_lookahead(vloam_b200_ctx* c) {
  int r = VLOAM_OK;
  while (r == VLOAM_OK && c->srPendCount > 0) {
    const int slot = !c->srNextValid ? 0 : (!c->srNext2Valid ? 1 : -1);
    if (slot < 0) break;  // both spare sets hold sweeps that have not been processed yet: the registration waits
    const vloam_b200_ctx::SrPend pd = c->srPend[0];
    c->srPend[0] = c->srPend[1]; c->srPendCount--;
    SrSet* S = slot ? c->srNext2 : c->srNext;
    const int curNow = c->cur;
    vl_sr_swap(c, *S);
    c->cur = (curNow + slot) % 3;  // vl_sr_run advances it: the look-ahead writes the generation after this sweep's (slot 1: the one after that,
                                   // i.e. the generation of the sweep BEFORE this one, dead once this sweep's odometry solve is done)
    vl_tls_stream = c->streamSR;
    // The generation of the less-sharp / less-flat clouds this run overwrites was the "last" cloud of an odometry solve that is
    // queued already (the previous sweep's, or this sweep's): order the overwrite behind the solves queued so far on the DEVICE
    // (a caller that never syncs -- skipped mapping frames with pose_out == NULL -- gives no host-side guarantee).
    if (!c->sideWaitsIssued) cudaStreamWaitEvent(c->streamSR, c->evLoSolve, 0);
    const float* d_xyz = pd.key;
    if (!pd.dev) {
      r = vl_reserve(c, c->in, (size_t)pd.n * pd.stride);
      if (r == VLOAM_OK && cudaMemcpyAsync(c->in.p, pd.key, (size_t)pd.n * pd.stride * sizeof(float), cudaMemcpyHostToDevice, c->streamSR) != cudaSuccess) r = VLOAM_E_CUDA;
      d_xyz = c->in.p;
    }
    if (r == VLOAM_OK) r = vl_sr_run(c, d_xyz, pd.n, pd.stride);
    vl_tls_stream = nullptr;
    vl_sr_swap(c, *S);  // (the context's own `cur` comes back with its set)
    if (slot) { c->srNext2Valid = r == VLOAM_OK; c->srNext2Key = pd.key; c->srNext2N = pd.n; c->srNext2Stride = pd.stride; }
    else { c->srNextValid = r == VLOAM_OK; c->srNextKey = pd.key; c->srNextN = pd.n; c->srNextStride = pd.stride; }
  }
  return r;
}

// Drop every look-ahead result (the sweep that arrived is not the registered one, or the state they were computed from was
// edited).  Their kernels may still be running on streamSR, writing generations the fresh run is about to use: wait for them.
void vl_drop_lookahead(vloam_b200_ctx* c) {
  if (c->sideSubmitted) { c->sideSubmitted = false; vl_lm_join(c); }  // (the helper thread may still be issuing side work that sets these flags)
  if (c->srNextValid || c->srNext2Valid) cudaStreamSynchronize(c->streamSR);
  c->srNextValid = c->srNext2Valid = false;
  c->loNextValid = false;
  c->loPreValid = false;
}

// this sweep was registered ahead: adopt the spare set (its kernels may still be running on streamSR)
static bool adopt_lookahead(vloam_b200_ctx* c, const float* key, int n, int stride) {
  if (!c->srNextValid || key != c->srNextKey || n != c->srNextN || stride != c->srNextStride) return false;
  vl_sr_swap(c, *c->srNext);
  // the set of the sweep after this one moves up; the set that just came out of the context is the free one
  { SrSet* t_ = c->srNext; c->srNext = c->srNext2; c->srNext2 = t_; }
  c->srNextValid = c->srNext2Valid; c->srNextKey = c->srNext2Key; c->srNextN = c->srNext2N; c->srNextStride = c->srNext2Stride;
  c->srNext2Valid = false;
  cudaStreamWaitEvent(c->stream, c->evSR, 0);
  return true;
}

int vloam_b200_scan_registration_device(vloam_b200_ctx* c, const float* d_xyz, int n, int stride) {
  if (!c) return VLOAM_E_INVALID;  // ABI boundary: a null context is the caller's error, not a crash
  if (n < 0 || stride < 3) { snprintf(c->err, sizeof c->err, "bad cloud shape"); return VLOAM_E_INVALID; }
  if (c->timing) VL_CUDA(cudaEventRecord(c->ev[0], c->stream));
  c->srAdopted = adopt_lookahead(c, d_xyz, n, stride);
  if (!c->srAdopted) {
    vl_drop_lookahead(c);  // a look-ahead result for another sweep targets the generation this run is about to write
    VL_TRY(vl_sr_run(c, d_xyz, n, stride));
  }
  if (c->timing) VL_CUDA(cudaEventRecord(c->ev[1], c->stream));
  return VLOAM_OK;
}

int vloam_b200_scan_registration(vloam_b200_ctx* c, const float* xyz, int n, int stride) {
  if (!c) return VLOAM_E_INVALID;  // ABI boundary: a null context is the caller's error, not a crash
  if (n < 0 || stride < 3 || (n > 0 && !xyz)) { snprintf(c->err, sizeof c->err, "bad cloud shape"); return VLOAM_E_INVALID; }
  if (c->timing) VL_CUDA(cudaEventRecord(c->ev[0], c->stream));
  c->srAdopted = adopt_lookahead(c, xyz, n, stride);
  if (!c->srAdopted) {
    vl_drop_lookahead(c);
    VL_TRY(vl_reserve(c, c->in, (size_t)max(n, 1) * stride));
    if (n > 0) VL_CUDA(cudaMemcpyAsync(c->in.p, xyz, (size_t)n * stride * sizeof(float), cudaMemcpyHostToDevice, c->stream));
    VL_TRY(vl_sr_run(c, c->in.p, n, stride));
  }
  if (c->timing) VL_CUDA(cudaEventRecord(c->ev[1], c->stream));
  return VLOAM_OK;
}

int vloam_b200_get_cloud(vloam_b200_ctx* c, int which, float* out, int cap_points) {
  if (!c) return VLOAM_E_INVALID;  // ABI boundary: a null context is the caller's error, not a crash
  VL_TRY(vl_sr_sync_counts(c));
  const float4* src = nullptr; int n = 0;
  switch (which) {
    case VLOAM_CLOUD_FULL: src = c->cloud.p; n = c->nKept; break;
    case VLOAM_CLOUD_SHARP: src = c->sharp.p; n = c->nSharp; break;
    case VLOAM_CLOUD_LESS_SHARP: src = c->lessSharp[c->cur].p; n = c->nLessSharp; break;
    case VLOAM_CLOUD_FLAT: src = c->flat.p; n = c->nFlat; break;
    case VLOAM_CLOUD_LESS_FLAT: src = c->lessFlat[c->cur].p; n = c->nLessFlat; break;
    case VLOAM_CLOUD_CORNER_LAST: src = c->cornerLastPtr; n = c->nCornerLast; break;
    case VLOAM_CLOUD_SURF_LAST: src = c->surfLastPtr; n = c->nSurfLast; break;
    case VLOAM_CLOUD_FULL_RES:  // LaserOdometry::output's laserCloudFullRes: the end-frame cloud under VLOAM_FLAG_TRANSFORM_TO_END
      src = c->cloud.p; n = c->nKept;
      if (vl_to_end(c) && out && n > 0 && cap_points >= n) {
        VL_TRY(vl_reserve(c, c->regOut, (size_t)n));
        VL_TRY(vl_lo_to_end_cloud(c, c->cloud.p, n, c->regOut.p));
        src = c->regOut.p;
      }
      break;
    default: snprintf(c->err, sizeof c->err, "unknown cloud id %d", which); return VLOAM_E_INVALID;
  }
  if (out && n > 0) {
    if (cap_points < n) { snprintf(c->err, sizeof c->err, "cloud buffer too small (%d < %d)", cap_points, n); return VLOAM_E_CAPACITY; }
    VL_CUDA(cudaMemcpyAsync(out, src, (size_t)n * 16, cudaMemcpyDeviceToHost, c->stream));
    VL_CUDA(cudaStreamSynchronize(c->stream));
  }
  return n;
}

int vloam_b200_laser_odometry(vloam_b200_ctx* c, const double* prior_q, const double* prior_t, int use_prior, double* q_w, double* t_w,
                              double* q_lc, double* t_lc, int* skip_frame) {
  if (!c) return VLOAM_E_INVALID;  // ABI boundary: a null context is the caller's error, not a crash
  if (use_prior && (!prior_q || !prior_t)) { snprintf(c->err, sizeof c->err, "use_prior without a prior"); return VLOAM_E_INVALID; }
  VL_TRY(vl_lo_run(c, prior_q, prior_t, use_prior));
  if (c->timing) VL_CUDA(cudaEventRecord(c->ev[2], c->stream));
  if (q_w || t_w || q_lc || t_lc) {
    VL_CUDA(cudaMemcpyAsync(c->h_los, c->los, sizeof(LoScalars), cudaMemcpyDeviceToHost, c->stream));
    VL_CUDA(cudaStreamSynchronize(c->stream));
    if (q_w) memcpy(q_w, c->h_los->q_w, 32);
    if (t_w) memcpy(t_w, c->h_los->t_w, 24);
    if (q_lc) memcpy(q_lc, c->h_los->para_q, 32);
    if (t_lc) memcpy(t_lc, c->h_los->para_t, 24);
  }
  if (skip_frame) *skip_frame = c->skip_frame ? 1 : 0;
  return VLOAM_OK;
}

int vloam_b200_laser_mapping(vloam_b200_ctx* c, double* q_w, double* t_w) {
  if (!c) return VLOAM_E_INVALID;  // ABI boundary: a null context is the caller's error, not a crash
  VL_TRY(vl_lm_run(c));
  if (c->timing) VL_CUDA(cudaEventRecord(c->ev[3], c->stream));
  if (q_w || t_w) {
    VL_CUDA(cudaMemcpyAsync(c->h_lmm, c->lmm, sizeof(LmScalars), cudaMemcpyDeviceToHost, c->stream));
    VL_CUDA(cudaStreamSynchronize(c->stream));
    if (c->h_lmm->overflow) { snprintf(c->err, sizeof c->err, "map pool exhausted"); return VLOAM_E_CAPACITY; }
    const double* q = c->skip_frame ? c->h_lmm->q_hf : c->h_lmm->pose;
    const double* t = c->skip_frame ? c->h_lmm->t_hf : c->h_lmm->pose + 4;
    if (q_w) memcpy(q_w, q, 32);
    if (t_w) memcpy(t_w, t, 24);
  }
  return VLOAM_OK;
}

int vloam_b200_register_full_cloud(vloam_b200_ctx* c, float* out, int cap_points) {
  if (!c) return VLOAM_E_INVALID;  // ABI boundary: a null context is the caller's error, not a crash
  VL_TRY(vl_sr_sync_counts(c));
  const int n = c->nKept;
  if (!out || n == 0) return n;
  if (cap_points < n) { snprintf(c->err, sizeof c->err, "cloud buffer too small (%d < %d)", cap_points, n); return VLOAM_E_CAPACITY; }
  VL_TRY(vl_reserve(c, c->regOut, (size_t)n));
  VL_TRY(vl_lm_register_full(c, c->cloud.p, n, c->regOut.p));
  VL_CUDA(cudaMemcpyAsync(out, c->regOut.p, (size_t)n * 16, cudaMemcpyDeviceToHost, c->stream));
  VL_CUDA(cudaStreamSynchronize(c->stream));
  return n;
}

static int process_common(vloam_b200_ctx* c, double* pose_out) {
  VL_HOST_MARK(1);
  c->inProcessFrame = true;
  const int rlo = vloam_b200_laser_odometry(c, nullptr, nullptr, 0, nullptr, nullptr, nullptr, nullptr, nullptr);
  c->inProcessFrame = false;
  if (rlo != VLOAM_OK) return rlo;
  if (pose_out) {
    c->s2Done = false;
    VL_TRY(vl_lm_run(c));
    if (c->timing) VL_CUDA(cudaEventRecord(c->ev[3], c->stream));
    if (!c->s2Done) {  // (mapping skipped on this frame) -- otherwise sync point S2 already brought both structs over
      VL_CUDA(cudaMemcpyAsync(c->h_los, c->los, sizeof(LoScalars), cudaMemcpyDeviceToHost, c->stream));
      VL_CUDA(cudaMemcpyAsync(c->h_lmm, c->lmm, sizeof(LmScalars), cudaMemcpyDeviceToHost, c->stream));
      VL_CUDA(cudaStreamSynchronize(c->stream));
    }
    if (c->h_lmm->overflow) { snprintf(c->err, sizeof c->err, "map pool exhausted"); return VLOAM_E_CAPACITY; }
    memcpy(pose_out, c->h_los->q_w, 32); memcpy(pose_out + 4, c->h_los->t_w, 24);
    memcpy(pose_out + 7, c->skip_frame ? c->h_lmm->q_hf : c->h_lmm->pose, 32);
    memcpy(pose_out + 11, c->skip_frame ? c->h_lmm->t_hf : c->h_lmm->pose + 4, 24);
    return VLOAM_OK;
  }
  return vloam_b200_laser_mapping(c, nullptr, nullptr);
}

int vloam_b200_process_frame(vloam_b200_ctx* c, const float* xyz, int n, int stride, double* pose_out) {
  if (!c) return VLOAM_E_INVALID;  // ABI boundary: a null context is the caller's error, not a crash
  VL_HOST_MARK(0);
  VL_TRY(vloam_b200_begin_frame(c));
  VL_TRY(vloam_b200_scan_registration(c, xyz, n, stride));
  return process_common(c, pose_out);
}
int vloam_b200_process_frame_device(vloam_b200_ctx* c, const float* d_xyz, int n, int stride, double* pose_out) {
  if (!c) return VLOAM_E_INVALID;  // ABI boundary: a null context is the caller's error, not a crash
  VL_HOST_MARK(0);
  VL_TRY(vloam_b200_begin_frame(c));
  VL_TRY(vloam_b200_scan_registration_device(c, d_xyz, n, stride));
  return process_common(c, pose_out);
}

int vloam_b200_synchronize(vloam_b200_ctx* c) {
  if (!c) return VLOAM_E_INVALID;  // ABI boundary: a null context is the caller's error, not a crash
  VL_TRY(vl_lo_flush_deferred(c));
  VL_TRY(vl_lm_join(c));
  VL_CUDA(cudaStreamSynchronize(c->streamSR));
  VL_CUDA(cudaStreamSynchronize(c->streamLO));
  VL_CUDA(cudaStreamSynchronize(c->streamAux));
  VL_CUDA(cudaStreamSynchronize(c->stream)); VL_CUDA(cudaStreamSynchronize(c->stream2)); VL_CUDA(cudaStreamSynchronize(c->stream3));
  VL_CUDA(cudaStreamSynchronize(c->stream4));
  VL_TRY(vl_lm_pub_sync(c));
  return VLOAM_OK;
}

int vloam_b200_publish_map(vloam_b200_ctx* c) {
  if (!c) return VLOAM_E_INVALID;  // ABI boundary: a null context is the caller's error, not a crash
  return vl_lm_publish_map(c);
}
int vloam_b200_get_map(vloam_b200_ctx* c, float* out_xyzi, int cap_points) {
  if (!c) return VLOAM_E_INVALID;  // ABI boundary: a null context is the caller's error, not a crash
  if (cap_points < 0) return VLOAM_E_INVALID;
  return vl_lm_get_map(c, out_xyzi, cap_points);
}
void* vloam_b200_stream(vloam_b200_ctx* c) { if (!c) return nullptr; return (void*)c->stream; }
long long vloam_b200_kernel_launches(const vloam_b200_ctx* c) { if (!c) return 0; return c->launches; }
int vloam_b200_set_timing(vloam_b200_ctx* c, int enabled) { if (!c) return VLOAM_E_INVALID; c->timing = enabled != 0; return VLOAM_OK; }
int vloam_b200_stage_ms(vloam_b200_ctx* c, float* ms3) {
  if (!c) return VLOAM_E_INVALID;  // ABI boundary: a null context is the caller's error, not a crash
  if (!c->timing) { snprintf(c->err, sizeof c->err, "timing is off"); return VLOAM_E_INVALID; }
  VL_CUDA(cudaStreamSynchronize(c->stream));
  for (int k = 0; k < 3; ++k) VL_CUDA(cudaEventElapsedTime(&ms3[k], c->ev[k], c->ev[k + 1]));
  return VLOAM_OK;
}

// Time one named kernel: CUDA events are recorded around each of its launches on the context's stream.
int vloam_b200_profile_kernel(vloam_b200_ctx* c, const char* name) {
  if (!c) return VLOAM_E_INVALID;  // ABI boundary: a null context is the caller's error, not a crash
  VL_TRY(vl_lm_join(c));
  VL_CUDA(cudaStreamSynchronize(c->stream));
  if (!c->prof_created) {
    for (int k = 0; k < VL_PROF_MAX; ++k) { VL_CUDA(cudaEventCreate(&c->prof_ev[k][0])); VL_CUDA(cudaEventCreate(&c->prof_ev[k][1])); }
    c->prof_created = 1;
  }
  c->prof_n = 0; c->prof_bytes = 0;
  if (name) { strncpy(c->prof_name, name, sizeof c->prof_name - 1); c->prof_name[sizeof c->prof_name - 1] = 0; }
  else c->prof_name[0] = 0;
  return VLOAM_OK;
}
int vloam_b200_profile_result(vloam_b200_ctx* c, int* launches, double* total_ms, double* total_bytes) {
  if (!c) return VLOAM_E_INVALID;  // ABI boundary: a null context is the caller's error, not a crash
  VL_CUDA(cudaStreamSynchronize(c->stream));
  double ms = 0;
  for (int k = 0; k < c->prof_n; ++k) { float t = 0; VL_CUDA(cudaEventElapsedTime(&t, c->prof_ev[k][0], c->prof_ev[k][1])); ms += t; }
  *launches = c->prof_n; *total_ms = ms; *total_bytes = c->prof_bytes;
  return VLOAM_OK;
}

// Per-kernel table of the launches timed since vloam_b200_profile_kernel(c, "*"): writes lines
// "name count total_ms total_bytes\n" into buf (NUL-terminated); returns the number of distinct kernels.
int vloam_b200_profile_table(vloam_b200_ctx* c, char* buf, int cap) {
  if (!c) return VLOAM_E_INVALID;  // ABI boundary: a null context is the caller's error, not a crash
  VL_TRY(vloam_b200_synchronize(c));
  std::vector<std::string> names; std::vector<int> cnt; std::vector<double> ms, by;
  for (int k = 0; k < c->prof_n; ++k) {
    float t = 0; VL_CUDA(cudaEventElapsedTime(&t, c->prof_ev[k][0], c->prof_ev[k][1]));
    std::string nm(c->prof_kname[k]);
    const size_t lt = nm.find('<'); if (lt != std::string::npos) nm = nm.substr(0, lt);
    size_t i = 0; for (; i < names.size(); ++i) if (names[i] == nm) break;
    if (i == names.size()) { names.push_back(nm); cnt.push_back(0); ms.push_back(0); by.push_back(0); }
    cnt[i]++; ms[i] += t; by[i] += c->prof_kbytes[k];
  }
  std::string out;
  for (size_t i = 0; i < names.size(); ++i) { char line[256]; snprintf(line, sizeof line, "%s %d %.6f %.1f\n", names[i].c_str(), cnt[i], ms[i], by[i]); out += line; }
  if ((int)out.size() + 1 > cap) { snprintf(c->err, sizeof c->err, "profile table buffer too small"); return VLOAM_E_CAPACITY; }
  memcpy(buf, out.c_str(), out.size() + 1);
  return (int)names.size();
}

// Timeline of the launches timed since vloam_b200_profile_kernel(c, "*"): lines "name stream start_us end_us\n",
// times relative to the first recorded launch, stream = 0 (main) .. 3.  Event pairs around every launch
// serialise neighbouring launches a little (no programmatic overlap across an event), so this shows the
// dependency structure and the gaps, not the exact production schedule.
int vloam_b200_profile_timeline(vloam_b200_ctx* c, char* buf, int cap) {
  if (!c) return VLOAM_E_INVALID;  // ABI boundary: a null context is the caller's error, not a crash
  VL_TRY(vloam_b200_synchronize(c));
  std::string out;
  const cudaStream_t ss[7] = {c->stream, c->stream2, c->stream3, c->stream4, c->streamSR, c->streamAux, c->streamLO};
  for (int k = 0; k < c->prof_n; ++k) {
    float t0 = 0, t1 = 0;
    VL_CUDA(cudaEventElapsedTime(&t0, c->prof_ev[0][0], c->prof_ev[k][0]));
    VL_CUDA(cudaEventElapsedTime(&t1, c->prof_ev[0][0], c->prof_ev[k][1]));
    int si = 0; for (int q = 0; q < 7; ++q) if (ss[q] == c->prof_kstream[k]) si = q;
    char line[256]; snprintf(line, sizeof line, "%s %d %.3f %.3f\n", c->prof_kname[k], si, t0 * 1e3, t1 * 1e3);
    out += line;
  }
  if ((int)out.size() + 1 > cap) { snprintf(c->err, sizeof c->err, "timeline buffer too small"); return VLOAM_E_CAPACITY; }
  memcpy(buf, out.c_str(), out.size() + 1);
  return c->prof_n;
}

int vloam_b200_lo_associate(vloam_b200_ctx* c, const double* x, int* corner_idx, int* surf_idx) { if (!c) return VLOAM_E_INVALID; return vl_lo_associate_only(c, x, corner_idx, surf_idx); }

// ---- name-keyed state access ----------------------------------------------------------------
static long put_dev(vloam_b200_ctx* c, const void* dsrc, size_t bytes, void* out, long cap) {
  if (out && bytes && (long)bytes <= cap) {
    if (cudaMemcpyAsync(out, dsrc, bytes, cudaMemcpyDeviceToHost, c->stream) != cudaSuccess || cudaStreamSynchronize(c->stream) != cudaSuccess) {
      snprintf(c->err, sizeof c->err, "debug_get copy failed"); return VLOAM_E_CUDA;
    }
  }
  return (long)bytes;
}
static long put_host(const void* src, size_t bytes, void* out, long cap) { if (out && (long)bytes <= cap && bytes) memcpy(out, src, bytes); return (long)bytes; }

long vloam_b200_debug_get(vloam_b200_ctx* c, const char* name, void* out, long cap) {
  if (!c) return VLOAM_E_INVALID;  // ABI boundary: a null context is the caller's error, not a crash
  const std::string n(name);
  if (n.rfind("sr.", 0) == 0 || n.rfind("lo.", 0) == 0) { if (vl_sr_sync_counts(c) != VLOAM_OK) return VLOAM_E_CUDA; }
  if (vloam_b200_synchronize(c) != VLOAM_OK) return VLOAM_E_CUDA;
  if (n == "sr.laserCloud") return put_dev(c, c->cloud.p, (size_t)c->nKept * 16, out, cap);
  if (n == "sr.sharp") return put_dev(c, c->sharp.p, (size_t)c->nSharp * 16, out, cap);
  if (n == "sr.lessSharp") return put_dev(c, c->lessSharp[c->cur].p, (size_t)c->nLessSharp * 16, out, cap);
  if (n == "sr.flat") return put_dev(c, c->flat.p, (size_t)c->nFlat * 16, out, cap);
  if (n == "sr.lessFlat") return put_dev(c, c->lessFlat[c->cur].p, (size_t)c->nLessFlat * 16, out, cap);
  if (n == "sr.curvature") return put_dev(c, c->curv.p, (size_t)c->nKept * 4, out, cap);
  if (n == "sr.label") return put_dev(c, c->label.p, (size_t)c->nKept * 4, out, cap);
  if (n == "sr.scanStartInd" || n == "sr.scanEndInd") {
    std::vector<int> rs(VL_MAX_RINGS + 1), rc(VL_MAX_RINGS);
    cudaMemcpy(rs.data(), c->ringStart, sizeof(int) * (VL_MAX_RINGS + 1), cudaMemcpyDeviceToHost);
    cudaMemcpy(rc.data(), c->ringCount, sizeof(int) * VL_MAX_RINGS, cudaMemcpyDeviceToHost);
    std::vector<int> v(c->prm.n_scans);
    for (int r = 0; r < c->prm.n_scans; ++r) v[r] = n == "sr.scanStartInd" ? rs[r] + 5 : rs[r] + rc[r] - 6;
    return put_host(v.data(), v.size() * 4, out, cap);
  }
  if (n == "lo.cornerLast") return put_dev(c, c->cornerLastPtr, (size_t)c->nCornerLast * 16, out, cap);
  if (n == "lo.surfLast") return put_dev(c, c->surfLastPtr, (size_t)c->nSurfLast * 16, out, cap);
  if (n == "lo.pose") {
    LoScalars h; cudaMemcpy(&h, c->los, sizeof h, cudaMemcpyDeviceToHost);
    double v[14]; memcpy(v, h.q_w, 32); memcpy(v + 4, h.t_w, 24); memcpy(v + 7, h.para_q, 32); memcpy(v + 11, h.para_t, 24);
    return put_host(v, sizeof v, out, cap);
  }
  for (int k = 0; k < 2; ++k) {
    const std::string s = std::to_string(k);
    if (n == "lo.assoc.corner" + s) return put_dev(c, c->dbgLoCorner[k].p, (size_t)c->nSharp * 8, out, cap);
    if (n == "lo.assoc.surf" + s) return put_dev(c, c->dbgLoSurf[k].p, (size_t)c->nFlat * 12, out, cap);
    if (n.rfind("lm.knn.", 0) == 0 && n.back() == ('0' + k)) {
      const std::string kind = n.substr(7, n.size() - 8);
      const int Qc = c->h_lmm->Qc, Qs = c->h_lmm->Qs;
      if (kind == "cidx") return put_dev(c, c->dbgKnnIdx[k][0].p, (size_t)Qc * 20, out, cap);
      if (kind == "sidx") return put_dev(c, c->dbgKnnIdx[k][1].p, (size_t)Qs * 20, out, cap);
      if (kind == "cd2") return put_dev(c, c->dbgKnnD2[k][0].p, (size_t)Qc * 20, out, cap);
      if (kind == "sd2") return put_dev(c, c->dbgKnnD2[k][1].p, (size_t)Qs * 20, out, cap);
      if (kind == "cok") return put_dev(c, c->dbgKnnOk[k][0].p, (size_t)Qc * 4, out, cap);
      if (kind == "sok") return put_dev(c, c->dbgKnnOk[k][1].p, (size_t)Qs * 4, out, cap);
    }
  }
  if (n == "timing.host") {  // timing mode: host clock in us since process_frame was entered
    // {SR queued / adopted, odometry queued (+ look-ahead), S1 passed + side streams queued, helper joined, mapping queued, S2 passed}
    // ..., [7..12] finer marks of the in-place mapping path: prepare queued, first kNN + fit queued, side work submitted, passes queued,
    //      update queued, lm_sync_s2 returned
    double v[15];
    for (int k = 0; k < 15; ++k) v[k] = c->hostT[k + 1] - c->hostT[0];
    return put_host(v, sizeof v, out, cap);
  }
  if (n == "timing.detail") {  // timing mode: ms since the start of the frame's scan registration
    // {SR end, LO end, LM end, sub-map build end, stacks awaited + counts set, first solve end, surf stack ready, corner stack ready, next LO grid ready}
    // ..., look-ahead odometry of the NEXT sweep finished (streamLO), map update of this sweep finished (stream3)}
    // ..., next sweep's sharp / flat features ready (streamSR), look-ahead odometry started (streamLO), next sweep's scan registration complete}
    float v[15] = {0};
    if (!c->timing) { snprintf(c->err, sizeof c->err, "timing is off"); return VLOAM_E_INVALID; }
    for (int k = 0; k < 3; ++k) cudaEventElapsedTime(&v[k], c->ev[0], c->ev[k + 1]);
    for (int k = 0; k < 12; ++k) cudaEventElapsedTime(&v[3 + k], c->ev[0], c->evx[k]);
    return put_host(v, sizeof v, out, cap);
  }
  if (n == "sr.trace") {  // clock64 phase stamps of the last sr_pick (CTAs 0..127) and sr_ring_voxel (128..255) launches
    static long long v[256 * 8];
    if (vl_sr_trace(c, v, 256 * 8) != VLOAM_OK) return VLOAM_E_CUDA;
    return put_host(v, sizeof v, out, cap);
  }
  if (n == "lo.trace") {  // per query warp of the last grid association: {cycles, flags}
    static int v[2 * 8192];
    if (vl_lo_trace(c, v, 2 * 8192) != VLOAM_OK) return VLOAM_E_CUDA;
    return put_host(v, sizeof v, out, cap);
  }
  if (n == "solver.trace") {  // clock64 stamps of the last lm_solve_cluster launch (first call arms the trace)
    long long v[16];
    if (vl_solver_trace(c, v) != VLOAM_OK) return VLOAM_E_CUDA;
    return put_host(v, sizeof v, out, cap);
  }
  if (n == "chain.trace") {  // first call arms the device-side timeline of the pose chain; later calls copy it out and reset it
    static VlChainTrace* d_tr = nullptr;
    if (!d_tr) {
      VL_CUDA(cudaMalloc(&d_tr, sizeof(VlChainTrace)));
      VL_CUDA(cudaMemset(d_tr, 0, sizeof(VlChainTrace)));
      VL_TRY(vl_chain_trace_arm_lm(d_tr)); VL_TRY(vl_chain_trace_arm_solver(d_tr)); VL_TRY(vl_chain_trace_arm_lo(d_tr));
      return 0;
    }
    VL_TRY(vloam_b200_synchronize(c));
    if (!out || cap < (long)sizeof(VlChainTrace)) return (long)sizeof(VlChainTrace);
    VL_CUDA(cudaMemcpy(out, d_tr, sizeof(VlChainTrace), cudaMemcpyDeviceToHost));
    VL_CUDA(cudaMemset(d_tr, 0, 8));
    return (long)sizeof(VlChainTrace);
  }
  if (n == "lm.grid") {  // bookkeeping of the voxel-hash grid as of the last S2: {chunks in use, live points, tombstones, dirty}
    const int v[4] = {c->h_lmm->gridTop, c->h_lmm->gridCount, c->h_lmm->gridDead, c->h_lmm->gridDirty};
    return put_host(v, sizeof v, out, cap);
  }
  if (n == "alloc.count") { const long long v = c->regrows; return put_host(&v, sizeof v, out, cap); }  // device buffer (re)allocations so far
  if (n == "lm.paths") { long long v[2]; vl_lm_paths(c, v); return put_host(v, sizeof v, out, cap); }  // mapped sweeps since create: {in-place, pool path}
  if (n == "lo.costs") return put_host(c->dbgLoCost, sizeof c->dbgLoCost, out, cap);
  if (n == "lm.costs") return put_host(c->dbgLmCost, sizeof c->dbgLmCost, out, cap);
  if (n == "lm.pose" || n == "lm.state" || n == "lm.validInd") {
    LmScalars h; cudaMemcpy(&h, c->lmm, sizeof h, cudaMemcpyDeviceToHost);
    if (n == "lm.pose") { double v[14]; memcpy(v, h.pose, 56); memcpy(v + 7, h.q_wmap_wodom, 32); memcpy(v + 11, h.t_wmap_wodom, 24); return put_host(v, sizeof v, out, cap); }
    if (n == "lm.state") { int v[5] = {h.cenW, h.cenH, h.cenD, c->lm_frameCount, c->lm_optimized}; return put_host(v, sizeof v, out, cap); }
    return put_host(h.validInd, (size_t)h.validNum * 4, out, cap);
  }
  if (n == "lm.cornerStack") return put_dev(c, c->stackC.p, (size_t)c->h_lmm->Qc * 16, out, cap);
  if (n == "lm.surfStack") return put_dev(c, c->stackS.p, (size_t)c->h_lmm->Qs * 16, out, cap);
  if (n == "lm.cornerFromMap") return put_dev(c, c->fromMapC.p, (size_t)c->h_lmm->Mc * 16, out, cap);
  if (n == "lm.surfFromMap") return put_dev(c, c->fromMapS.p, (size_t)c->h_lmm->Ms * 16, out, cap);
  if (n == "lm.cornerMap" || n == "lm.surfMap") {
    long bytes = 0;
    if (vl_lm_export_map(c, n == "lm.surfMap", out, cap, &bytes) != VLOAM_OK) return VLOAM_E_CUDA;
    return bytes;
  }
  snprintf(c->err, sizeof c->err, "unknown buffer name '%s'", name);
  return VLOAM_E_NAME;
}

int vloam_b200_debug_set(vloam_b200_ctx* c, const char* name, const void* data, long bytes) {
  if (!c) return VLOAM_E_INVALID;  // ABI boundary: a null context is the caller's error, not a crash
  const std::string n(name);
  VL_TRY(vloam_b200_synchronize(c));
  if (n.rfind("lm.", 0) == 0) VL_TRY(vl_lm_sync_pools(c));  // edits of the mapping state work on the cube pools
  c->loNextValid = false;  // whatever is set below may change what the next odometry solve starts from
  if (n == "debug.capture") { c->h_vScalars[0] = (bytes >= 4 && *(const int*)data) ? 1 : 0; return VLOAM_OK; }
  if (n == "lo.last") {  // blob: int nc, int ns, corner points, surf points  (the state solveLO swaps in, LO.cpp:558-574)
    const int* hdr = (const int*)data;
    if (bytes < 8 || bytes != 8 + ((long)hdr[0] + hdr[1]) * 16) { snprintf(c->err, sizeof c->err, "lo.last blob size mismatch"); return VLOAM_E_INVALID; }
    const int o = (c->cur + 1) % 3;  // (cur becomes o below, so the next sweep's scan registration writes (o + 1) % 3)
    vl_drop_lookahead(c);          // a look-ahead result was computed into buffer o: drop it
    VL_TRY(vl_reserve(c, c->lessSharp[o], (size_t)max(hdr[0], 1)));
    VL_TRY(vl_reserve(c, c->lessFlat[o], (size_t)max(hdr[1], 1)));
    const char* p = (const char*)data + 8;
    if (hdr[0]) VL_CUDA(cudaMemcpy(c->lessSharp[o].p, p, (size_t)hdr[0] * 16, cudaMemcpyHostToDevice));
    if (hdr[1]) VL_CUDA(cudaMemcpy(c->lessFlat[o].p, p + (size_t)hdr[0] * 16, (size_t)hdr[1] * 16, cudaMemcpyHostToDevice));
    // make that buffer the current one so the next frame (cur = (cur + 1) % 3) writes the generation after it
    c->cur = o;
    c->cornerLastPtr = c->lessSharp[o].p; c->surfLastPtr = c->lessFlat[o].p;
    c->nCornerLast = hdr[0]; c->nSurfLast = hdr[1];
    c->lo_inited = true;
    VL_TRY(vl_lo_build_last(c, c->lastSet, c->cornerLastPtr, c->nCornerLast, c->surfLastPtr, c->nSurfLast));
    VL_CUDA(cudaStreamSynchronize(c->stream));
    return VLOAM_OK;
  }
  if (n == "lo.pose") {
    if (bytes != 14 * 8) return VLOAM_E_INVALID;
    const double* v = (const double*)data;
    LoScalars h; VL_CUDA(cudaMemcpy(&h, c->los, sizeof h, cudaMemcpyDeviceToHost));
    memcpy(h.q_w, v, 32); memcpy(h.t_w, v + 4, 24); memcpy(h.para_q, v + 7, 32); memcpy(h.para_t, v + 11, 24);
    VL_CUDA(cudaMemcpy(c->los, &h, sizeof h, cudaMemcpyHostToDevice));
    return VLOAM_OK;
  }
  if (n == "lm.pose" || n == "lm.state") {
    LmScalars h; VL_CUDA(cudaMemcpy(&h, c->lmm, sizeof h, cudaMemcpyDeviceToHost));
    if (n == "lm.pose") {
      if (bytes != 14 * 8) return VLOAM_E_INVALID;
      const double* v = (const double*)data;
      memcpy(h.pose, v, 56); memcpy(h.q_wmap_wodom, v + 7, 32); memcpy(h.t_wmap_wodom, v + 11, 24);
    } else {
      if (bytes < 16) return VLOAM_E_INVALID;
      const int* v = (const int*)data;
      h.cenW = v[0]; h.cenH = v[1]; h.cenD = v[2]; c->lm_frameCount = v[3];
    }
    VL_CUDA(cudaMemcpy(c->lmm, &h, sizeof h, cudaMemcpyHostToDevice));
    if (n == "lm.state") VL_TRY(vl_lm_rescan_sorted(c));  // voxel keys are relative to the cube origin
    return VLOAM_OK;
  }
  if (n == "lm.cornerMap") return vl_lm_import_map(c, 0, data, bytes);
  if (n == "lm.surfMap") return vl_lm_import_map(c, 1, data, bytes);
  snprintf(c->err, sizeof c->err, "unknown buffer name '%s'", name);
  return VLOAM_E_NAME;
}

int vloam_b200_voxel_grid(vloam_b200_ctx* c, const float* in, int n, float leaf, float* out, int cap_points) {
  if (!c) return VLOAM_E_INVALID;  // ABI boundary: a null context is the caller's error, not a crash
  if (n < 0 || !(leaf > 0.f)) return VLOAM_E_INVALID;
  VL_TRY(vloam_b200_synchronize(c));  // look-ahead stack filters of a registered sweep may still be using the filter scratch
  VL_TRY(vl_reserve(c, c->vIn, (size_t)max(n, 1)));
  VL_TRY(vl_reserve(c, c->vOut, (size_t)max(n, 1)));
  if (n) VL_CUDA(cudaMemcpyAsync(c->vIn.p, in, (size_t)n * 16, cudaMemcpyHostToDevice, c->stream));
  int* d_count = c->vScalars + 16;
  VL_TRY(vl_voxel_grid_device(c, c->vIn.p, n, nullptr, leaf, c->vOut.p, d_count));
  int m = 0;
  VL_CUDA(cudaMemcpyAsync(&m, d_count, 4, cudaMemcpyDeviceToHost, c->stream));
  VL_CUDA(cudaStreamSynchronize(c->stream));
  if (m > cap_points) { snprintf(c->err, sizeof c->err, "voxel_grid output buffer too small"); return VLOAM_E_CAPACITY; }
  if (m && out) { VL_CUDA(cudaMemcpyAsync(out, c->vOut.p, (size_t)m * 16, cudaMemcpyDeviceToHost, c->stream)); VL_CUDA(cudaStreamSynchronize(c->stream)); }
  return m;
}

static int upload_factors(vloam_b200_ctx* c, const double* factors, int nf) {
  VL_TRY(vl_reserve(c, c->factors, (size_t)max(nf, 1) * 10));
  VL_TRY(vl_reserve(c, c->factorValid, (size_t)max(nf, 1)));
  if (nf) {
    VL_CUDA(cudaMemcpyAsync(c->factors.p, factors, (size_t)nf * 80, cudaMemcpyHostToDevice, c->stream));
    std::vector<int> ones(nf, 1);
    VL_CUDA(cudaMemcpyAsync(c->factorValid.p, ones.data(), (size_t)nf * 4, cudaMemcpyHostToDevice, c->stream));
    VL_CUDA(cudaStreamSynchronize(c->stream));
  }
  return VLOAM_OK;
}

static int upload_s(vloam_b200_ctx* c, const double* s, int nf) {
  VL_TRY(vl_reserve(c, c->factorS, (size_t)max(nf, 1)));
  if (nf) { VL_CUDA(cudaMemcpyAsync(c->factorS.p, s, (size_t)nf * 8, cudaMemcpyHostToDevice, c->stream)); VL_CUDA(cudaStreamSynchronize(c->stream)); }
  return VLOAM_OK;
}

int vloam_b200_evaluate_deskew(vloam_b200_ctx* c, const double* factors, const double* s, int nf, const double* x, double* cost, double* H, double* g) {
  if (!c) return VLOAM_E_INVALID;
  VL_TRY(vloam_b200_synchronize(c));
  VL_TRY(upload_factors(c, factors, nf));
  if (s) VL_TRY(upload_s(c, s, nf));
  double* d_x = reinterpret_cast<double*>(c->vScalars + 32);
  VL_CUDA(cudaMemcpyAsync(d_x, x, 56, cudaMemcpyHostToDevice, c->stream));
  VL_TRY(vl_evaluate_once(c, nf, d_x, c->evalOut, s ? c->factorS.p : nullptr));
  EvalOut h;
  VL_CUDA(cudaMemcpyAsync(&h, c->evalOut, sizeof h, cudaMemcpyDeviceToHost, c->stream));
  VL_CUDA(cudaStreamSynchronize(c->stream));
  int t = 0;
  for (int i = 0; i < 6; ++i) for (int j = i; j < 6; ++j) { H[i * 6 + j] = h.v[t]; H[j * 6 + i] = h.v[t]; ++t; }
  for (int i = 0; i < 6; ++i) g[i] = h.v[21 + i];
  *cost = h.v[27];
  return VLOAM_OK;
}
int vloam_b200_evaluate(vloam_b200_ctx* c, const double* factors, int nf, const double* x, double* cost, double* H, double* g) {
  return vloam_b200_evaluate_deskew(c, factors, nullptr, nf, x, cost, H, g);
}

int vloam_b200_solve_deskew(vloam_b200_ctx* c, const double* factors, const double* s, int nf, double* x, double* log4) {
  if (!c) return VLOAM_E_INVALID;
  VL_TRY(vloam_b200_synchronize(c));
  VL_TRY(upload_factors(c, factors, nf));
  if (s) VL_TRY(upload_s(c, s, nf));
  double* d_x = reinterpret_cast<double*>(c->vScalars + 32);
  VL_CUDA(cudaMemcpyAsync(d_x, x, 56, cudaMemcpyHostToDevice, c->stream));
  double costs[2] = {0, 0};
  VL_TRY(vl_solve(c, nf, nullptr, d_x, costs, 0, s ? c->factorS.p : nullptr));
  VL_CUDA(cudaMemcpyAsync(x, d_x, 56, cudaMemcpyDeviceToHost, c->stream));
  VL_CUDA(cudaStreamSynchronize(c->stream));
  if (log4) { log4[0] = nf ? c->h_lms->iter : 0; log4[1] = 0; log4[2] = costs[0]; log4[3] = costs[1]; }
  return VLOAM_OK;
}
int vloam_b200_solve(vloam_b200_ctx* c, const double* factors, int nf, double* x, double* log4) {
  return vloam_b200_solve_deskew(c, factors, nullptr, nf, x, log4);
}

// n five-point sets (float32[n][5][3]) through the line (kind 0, LM.cpp:559-603) or plane (kind 1, LM.cpp:637-680) fit of the
// mapping stage: accept flags ok[n] and parameters params[n][6] ({a, b} of the edge factor / {unit normal, d, 0, 0}).
int vloam_b200_fit(vloam_b200_ctx* c, const float* near, int n, int kind, int* ok, double* params) {
  if (!c) return VLOAM_E_INVALID;
  if (n < 0 || (kind != 0 && kind != 1) || (n > 0 && (!near || !ok || !params))) return VLOAM_E_INVALID;
  if (n == 0) return VLOAM_OK;
  VL_TRY(vloam_b200_synchronize(c));
  float* d_near = nullptr; int* d_ok = nullptr; double* d_prm = nullptr;
  int r = VLOAM_OK;
  if (cudaMalloc(&d_near, (size_t)n * 60) != cudaSuccess || cudaMalloc(&d_ok, (size_t)n * 4) != cudaSuccess || cudaMalloc(&d_prm, (size_t)n * 48) != cudaSuccess) r = VLOAM_E_CUDA;
  if (r == VLOAM_OK && cudaMemcpyAsync(d_near, near, (size_t)n * 60, cudaMemcpyHostToDevice, c->stream) != cudaSuccess) r = VLOAM_E_CUDA;
  if (r == VLOAM_OK) r = vl_lm_fit_sets(c, d_near, n, kind, d_ok, d_prm);
  if (r == VLOAM_OK && (cudaMemcpyAsync(ok, d_ok, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream) != cudaSuccess ||
                        cudaMemcpyAsync(params, d_prm, (size_t)n * 48, cudaMemcpyDeviceToHost, c->stream) != cudaSuccess ||
                        cudaStreamSynchronize(c->stream) != cudaSuccess)) r = VLOAM_E_CUDA;
  if (r == VLOAM_E_CUDA) snprintf(c->err, sizeof c->err, "vloam_b200_fit: %s", cudaGetErrorString(cudaGetLastError()));
  cudaFree(d_near); cudaFree(d_ok); cudaFree(d_prm);
  return r;
}

// atanf(x[i]) and atan2f(y[i], x[i]) as the scan-registration kernels evaluate them ON THE DEVICE (exact_math.h; SR.cpp:185-187, 217,
// 263 call glibc's): host arrays in, host arrays out.
int vloam_b200_exact_math(vloam_b200_ctx* c, const float* y, const float* x, int n, float* atan_x, float* atan2_yx) {
  if (!c) return VLOAM_E_INVALID;
  if (n < 0 || (n > 0 && (!y || !x || !atan_x || !atan2_yx))) return VLOAM_E_INVALID;
  if (n == 0) return VLOAM_OK;
  VL_TRY(vloam_b200_synchronize(c));
  float* d = nullptr;
  int r = VLOAM_OK;
  const size_t B = (size_t)n * sizeof(float);
  if (cudaMalloc(&d, 4 * B) != cudaSuccess) r = VLOAM_E_CUDA;
  if (r == VLOAM_OK && (cudaMemcpyAsync(d, y, B, cudaMemcpyHostToDevice, c->stream) != cudaSuccess ||
                        cudaMemcpyAsync(d + n, x, B, cudaMemcpyHostToDevice, c->stream) != cudaSuccess)) r = VLOAM_E_CUDA;
  if (r == VLOAM_OK) r = vl_sr_exact_math(c, d, d + n, n, d + 2 * (size_t)n, d + 3 * (size_t)n);
  if (r == VLOAM_OK && (cudaMemcpyAsync(atan_x, d + 2 * (size_t)n, B, cudaMemcpyDeviceToHost, c->stream) != cudaSuccess ||
                        cudaMemcpyAsync(atan2_yx, d + 3 * (size_t)n, B, cudaMemcpyDeviceToHost, c->stream) != cudaSuccess ||
                        cudaStreamSynchronize(c->stream) != cudaSuccess)) r = VLOAM_E_CUDA;
  if (r == VLOAM_E_CUDA) snprintf(c->err, sizeof c->err, "vloam_b200_exact_math: %s", cudaGetErrorString(cudaGetLastError()));
  if (d) cudaFree(d);
  return r;
}

}  // extern "C"

// relocalize.cu -- vloam_b200_relocalize: exact correlative search of the last mapped sweep's stacks in the loaded map, by branch and
// bound over translation (Hess et al., "Real-Time Loop Closure in 2D LIDAR SLAM", 2016) made level-synchronous for the GPU.
//
// The search space and its scores are defined in include/vloam_b200.h (and restated in tests/relocalize_ref.py):
//   rl_select   query points u = R_c p of the stacks (range gate, every k-th), their |u_z| extent and the map's size (one block)
//   rl_cells    per yaw j and point the base cell c_j(p) = floor((Rz(theta_j) u + t_c - o) / r)
//   rl_occ      level-0 occupancy: byte 1 at the cell of every map point of the cubes that overlap the grid
//   rl_pool     level h = max of level h-1 over the x, then the y shifts {0, 2^(h-1)}: level h at cell x is the max of level 0 over
//               [x, x + 2^h)^2, so the bound of a node covering 2^h x 2^h offsets is one look-up per point at its corner cell
//   rl_top      bound of every coarsest node (one per yaw and z offset); rl_greedy descends each to a leaf (initial lower bound)
//   rl_seed / rl_expand  the frontier, level by level: a child is kept when its bound >= the best leaf score so far (ties are
//               kept, so the lowest index among equal scores survives); leaves raise the bound and the winner is a 64-bit
//               (score, ~index) max.  The runner-up is the same search with the exclusion zone around the winner bounded by -1.
// Scores are integer counts after the per-yaw step, so the result does not depend on the order of the atomics.
#include <math.h>
#include <string>
#include <vector>
#include "common.cuh"

#define RL_MAX_LEVELS 16  // S = 2 N + 1 translation offsets per axis < 2^15 (node corners are packed in 16 bits)

struct RlSpace {                // one search, by value into every kernel
  const int4* cells;            // [nJ][m] base cells (w unused)
  const unsigned char* occ;     // level h at occ + h * levelCells
  size_t levelCells;
  int Gx, Gy, Gz;
  int m, nJ, nZ, S, N, Nz, H, full;
  double dtheta, r, exclM, exclRad;
};

struct RlDev {                  // device results of both passes (0: best, 1: runner-up)
  unsigned long long key[2];    // (score << 32) | ~index, 0 = none
  int L[2];                     // best leaf score so far
  long long evals[2];           // node bounds computed
  int nFront[2][RL_MAX_LEVELS]; // frontier nodes kept per level (level H: the seeds)
};

struct RlSelectOut { int m, nKept, mapPoints, pad; double zmax; };

struct RlState {                // first vloam_b200_relocalize call: nothing of this exists in a context that never calls it
  DBuf<int> kept; DBuf<double> u; DBuf<int4> cells; DBuf<double2> yaw; DBuf<unsigned char> occ; DBuf<int> topB;
  DBuf<int2> front[2];
  RlDev* dev; RlDev* h_dev; RlSelectOut* sel; RlSelectOut* h_sel;
  cudaEvent_t ev[3];
  // host copies of the last search for the debug getters (rl.points, rl.occ, rl.yaw, rl.levels, rl.ms)
  int m, Gx, Gy, Gz; double o[3]; std::vector<double> yawTab; RlDev last; float ms[2];
};

__device__ __forceinline__ int rl_lookup(const RlSpace& s, const unsigned char* occ, int x, int y, int z, int span) {
  // level-h value of window [x, x + span)^2: a window that starts below the grid is bounded by the one at 0 (it covers the part inside)
  if (x < 0) { if (x <= -span) return 0; x = 0; }
  if (y < 0) { if (y <= -span) return 0; y = 0; }
  if (x >= s.Gx || y >= s.Gy || z < 0 || z >= s.Gz) return 0;
  return occ[((size_t)z * s.Gy + y) * s.Gx + x];
}

// the node (jj, ax0.., ay0..) of span `span` lies entirely inside the exclusion zone around pass 0's winner
__device__ __forceinline__ bool rl_excluded(const RlSpace& s, const RlDev* d, int pass, int jj, int ax0, int ay0, int span) {
  if (pass == 0) return false;
  const unsigned long long kb = d->key[0];
  const long long lin = (long long)(unsigned)~(unsigned)(kb & 0xffffffffull);
  const long long per = (long long)s.nZ * s.S * s.S;
  const int jb = (int)(lin / per), ayb = (int)((lin / s.S) % s.S), axb = (int)(lin % s.S);
  int dj = abs(jj - jb);
  if (s.full) dj = min(dj, s.nJ - dj);
  if (!((double)dj * s.dtheta < s.exclRad)) return false;
  const int ax1 = min(ax0 + span, s.S) - 1, ay1 = min(ay0 + span, s.S) - 1;
  const int dx = max(abs(ax0 - axb), abs(ax1 - axb)), dy = max(abs(ay0 - ayb), abs(ay1 - ayb));
  return (double)dx * s.r < s.exclM && (double)dy * s.r < s.exclM;
}

__device__ __forceinline__ int rl_warp_sum(int v) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// bounds of the four children (level hc) of a node at level hc + 1 with corner (ax0, ay0); children past S get -2, excluded ones -1
__device__ __forceinline__ void rl_children(const RlSpace& s, const RlDev* d, int pass, int jz, int ax0, int ay0, int hc, int lane, int b[4]) {
  const int jj = jz / s.nZ, izz = jz - jj * s.nZ, span = 1 << hc;
  const unsigned char* occ = s.occ + (size_t)hc * s.levelCells;
  const int4* cells = s.cells + (size_t)jj * s.m;
  int cnt[4] = {0, 0, 0, 0};
  for (int p = lane; p < s.m; p += 32) {
    const int4 c = __ldg(&cells[p]);
    const int x = c.x + ax0 - s.N, y = c.y + ay0 - s.N, z = c.z + izz - s.Nz;
#pragma unroll
    for (int k = 0; k < 4; ++k) cnt[k] += rl_lookup(s, occ, x + (k & 1) * span, y + (k >> 1) * span, z, span);
  }
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int ax = ax0 + (k & 1) * span, ay = ay0 + (k >> 1) * span;
    const int sum = rl_warp_sum(cnt[k]);
    b[k] = (ax >= s.S || ay >= s.S) ? -2 : rl_excluded(s, d, pass, jj, ax, ay, span) ? -1 : sum;
  }
}

__device__ __forceinline__ void rl_leaf(const RlSpace& s, RlDev* d, int pass, int jz, int ax, int ay, int score) {
  const long long lin = ((long long)jz * s.S + ay) * s.S + ax;
  atomicMax(&d->L[pass], score);
  atomicMax(&d->key[pass], ((unsigned long long)(unsigned)score << 32) | (unsigned long long)(~(unsigned)lin));
}

// query points: stackC then stackS, range <= max_range in order, every k-th of the n kept (k = ceil(n / max_points)), u = R_c p
struct RlRot { double R[9]; };
__global__ void __launch_bounds__(1024) rl_select(const float4* __restrict__ sc, int nc, const float4* __restrict__ ss, int ns, RlRot rot,
                                                  double maxR2, int maxPoints, const MapCubeTable* __restrict__ tc,
                                                  const MapCubeTable* __restrict__ ts, int* __restrict__ kept, double* __restrict__ u,
                                                  RlSelectOut* __restrict__ out) {
  VL_PDL_WAIT();
  __shared__ int ws[32];
  __shared__ double zs[32];
  __shared__ int mapPts;
  if (threadIdx.x == 0) mapPts = 0;
  __syncthreads();
  int base = 0;
  for (int b0 = 0; b0 < nc + ns; b0 += 1024) {
    const int i = b0 + threadIdx.x;
    bool keep = false;
    if (i < nc + ns) {
      const float4 p = i < nc ? sc[i] : ss[i - nc];
      const double x = p.x, y = p.y, z = p.z;
      keep = x * x + y * y + z * z <= maxR2;
    }
    int tot = 0;
    const int at = vl_block_excl_scan<1024>(keep ? 1 : 0, ws, &tot);
    if (keep) kept[base + at] = i;
    base += tot;
  }
  __syncthreads();
  const int n = base, k = n > 0 ? (n + maxPoints - 1) / maxPoints : 1, m = (n + k - 1) / k;
  double zmax = 0.0;
  for (int q = threadIdx.x; q < m; q += 1024) {
    const int i = kept[q * k];
    const float4 p = i < nc ? sc[i] : ss[i - nc];
    const double px = p.x, py = p.y, pz = p.z;
    const double* R = rot.R;
    const double ux = R[0] * px + R[1] * py + R[2] * pz, uy = R[3] * px + R[4] * py + R[5] * pz, uz = R[6] * px + R[7] * py + R[8] * pz;
    u[3 * q] = ux; u[3 * q + 1] = uy; u[3 * q + 2] = uz;
    zmax = fmax(zmax, fabs(uz));
  }
  int own = 0;
  for (int cb = threadIdx.x; cb < VL_CUBE_NUM; cb += 1024) own += tc->count[cb] + ts->count[cb];
  for (int o = 16; o > 0; o >>= 1) { zmax = fmax(zmax, __shfl_xor_sync(0xffffffffu, zmax, o)); own += __shfl_xor_sync(0xffffffffu, own, o); }
  if ((threadIdx.x & 31) == 0) { zs[threadIdx.x >> 5] = zmax; atomicAdd(&mapPts, own); }
  __syncthreads();
  if (threadIdx.x == 0) {
    double z = 0.0;
    for (int w = 0; w < 32; ++w) z = fmax(z, zs[w]);
    out->m = m; out->nKept = n; out->mapPoints = mapPts; out->zmax = z;
  }
}

struct RlGrid { double tc[3], o[3], r; };
__global__ void __launch_bounds__(256) rl_cells(const double* __restrict__ u, int m, int nJ, const double2* __restrict__ yaw, RlGrid g,
                                                int4* __restrict__ cells) {
  VL_PDL_WAIT();
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < (long long)m * nJ; i += (long long)gridDim.x * blockDim.x) {
    const int j = (int)(i / m), p = (int)(i - (long long)j * m);
    const double c = yaw[j].x, s = yaw[j].y, ux = u[3 * p], uy = u[3 * p + 1], uz = u[3 * p + 2];
    const double vx = c * ux - s * uy, vy = s * ux + c * uy;
    cells[i] = make_int4((int)floor((vx + g.tc[0] - g.o[0]) / g.r), (int)floor((vy + g.tc[1] - g.o[1]) / g.r),
                         (int)floor((uz + g.tc[2] - g.o[2]) / g.r), 0);
  }
}

// one block per cube and kind; cubes whose 50 m box (with 1 m margin for the insert formula's rounding) misses the grid are skipped
__global__ void __launch_bounds__(256) rl_occ(const LmScalars* __restrict__ s, const MapCubeTable* __restrict__ tc, const MapCubeTable* __restrict__ ts,
                                              const float4* __restrict__ pc, const float4* __restrict__ ps, RlGrid g, int Gx, int Gy, int Gz,
                                              unsigned char* __restrict__ occ) {
  VL_PDL_WAIT();
  const int cube = blockIdx.x, kind = blockIdx.y;
  const MapCubeTable* t = kind ? ts : tc;
  const int n = t->count[cube];
  if (n == 0) return;
  const int ci = cube % VL_CUBE_W, cj = (cube / VL_CUBE_W) % VL_CUBE_H, ck = cube / (VL_CUBE_W * VL_CUBE_H);
  const int off[3] = {ci - s->cenW, cj - s->cenH, ck - s->cenD};
  const int G[3] = {Gx, Gy, Gz};
  for (int a = 0; a < 3; ++a) {
    const double lo = 50.0 * off[a] - 26.0, hi = 50.0 * off[a] + 26.0;
    if (hi < g.o[a] || lo > g.o[a] + g.r * G[a]) return;
  }
  const float4* pool = (kind ? ps : pc) + t->start[cube];
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const float4 p = pool[i];
    const double x = floor(((double)p.x - g.o[0]) / g.r), y = floor(((double)p.y - g.o[1]) / g.r), z = floor(((double)p.z - g.o[2]) / g.r);
    if (x < 0.0 || y < 0.0 || z < 0.0 || x >= (double)Gx || y >= (double)Gy || z >= (double)Gz) continue;
    occ[((size_t)z * Gy + (size_t)y) * Gx + (size_t)x] = 1;
  }
}

// dst = max(src, src shifted by d along x (axis 0) or y (axis 1)); cells past the grid read 0
__global__ void __launch_bounds__(256) rl_pool(const unsigned char* __restrict__ src, unsigned char* __restrict__ dst, int Gx, int Gy, size_t cells,
                                               int d, int axis) {
  VL_PDL_WAIT();
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < cells; i += (size_t)gridDim.x * blockDim.x) {
    const int x = (int)(i % Gx), y = (int)((i / Gx) % Gy);
    unsigned char v = src[i];
    if (axis == 0 ? x + d < Gx : y + d < Gy) v = max(v, src[axis == 0 ? i + d : i + (size_t)d * Gx]);
    dst[i] = v;
  }
}

// one warp per coarsest node (yaw, z offset; corner (0, 0) at level H): its bound, or -1 inside the exclusion zone
__global__ void __launch_bounds__(256) rl_top(RlSpace s, RlDev* __restrict__ d, int pass, int* __restrict__ topB) {
  VL_PDL_WAIT();
  const int jz = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (jz >= s.nJ * s.nZ) return;
  const int jj = jz / s.nZ, izz = jz - jj * s.nZ, span = 1 << s.H;
  const unsigned char* occ = s.occ + (size_t)s.H * s.levelCells;
  const int4* cells = s.cells + (size_t)jj * s.m;
  int cnt = 0;
  for (int p = lane; p < s.m; p += 32) {
    const int4 c = __ldg(&cells[p]);
    cnt += rl_lookup(s, occ, c.x - s.N, c.y - s.N, c.z + izz - s.Nz, span);
  }
  cnt = rl_warp_sum(cnt);
  if (lane) return;
  const int b = rl_excluded(s, d, pass, jj, 0, 0, span) ? -1 : cnt;
  topB[jz] = b;
  atomicAdd((unsigned long long*)&d->evals[pass], 1ull);
  if (s.H == 0 && b >= 0) rl_leaf(s, d, pass, jz, 0, 0, b);  // (one offset per axis: the coarsest nodes are the leaves)
}

// initial lower bound: every coarsest node descends to a leaf through its best child (ties: the lowest index)
__global__ void __launch_bounds__(256) rl_greedy(RlSpace s, RlDev* __restrict__ d, int pass, const int* __restrict__ topB) {
  VL_PDL_WAIT();
  const int jz = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (jz >= s.nJ * s.nZ || topB[jz] < 0) return;
  int ax0 = 0, ay0 = 0;
  for (int hc = s.H - 1; hc >= 0; --hc) {
    int b[4];
    rl_children(s, d, pass, jz, ax0, ay0, hc, lane, b);
    int kb = -1;
    for (int k = 0; k < 4; ++k) if (b[k] >= 0 && (kb < 0 || b[k] > b[kb])) kb = k;
    if (lane == 0) atomicAdd((unsigned long long*)&d->evals[pass], 4ull);
    if (kb < 0) return;
    ax0 += (kb & 1) << hc; ay0 += (kb >> 1) << hc;
    if (hc == 0 && lane == 0) rl_leaf(s, d, pass, jz, ax0, ay0, b[kb]);
  }
}

// level-H frontier: the coarsest nodes whose bound reaches the greedy lower bound
__global__ void __launch_bounds__(256) rl_seed(RlSpace s, RlDev* __restrict__ d, int pass, const int* __restrict__ topB, int2* __restrict__ out) {
  VL_PDL_WAIT();
  const int jz = blockIdx.x * blockDim.x + threadIdx.x;
  if (jz >= s.nJ * s.nZ) return;
  if (topB[jz] >= 0 && topB[jz] >= d->L[pass]) out[atomicAdd(&d->nFront[pass][s.H], 1)] = make_int2(jz, 0);
}

// expand the level-h frontier (persistent warps, one node at a time): children at level h - 1 whose bound reaches the current lower
// bound go to the next frontier; at h = 1 the children are leaves
__global__ void __launch_bounds__(256) rl_expand(RlSpace s, RlDev* __restrict__ d, int pass, int h, const int2* __restrict__ in, int2* __restrict__ out) {
  VL_PDL_WAIT();
  const int lane = threadIdx.x & 31;
  const int n = d->nFront[pass][h];
  const int hc = h - 1;
  for (int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < n; w += (gridDim.x * blockDim.x) >> 5) {
    const int2 node = in[w];
    const int ax0 = node.y & 0xffff, ay0 = node.y >> 16;
    int b[4];
    rl_children(s, d, pass, node.x, ax0, ay0, hc, lane, b);
    if (lane) continue;
    const int L = *(volatile int*)&d->L[pass];
    int nv = 0;
    for (int k = 0; k < 4; ++k) {
      if (b[k] == -2) continue;
      ++nv;
      if (b[k] < 0 || b[k] < L) continue;
      const int ax = ax0 + ((k & 1) << hc), ay = ay0 + ((k >> 1) << hc);
      if (hc == 0) rl_leaf(s, d, pass, node.x, ax, ay, b[k]);
      else out[atomicAdd(&d->nFront[pass][hc], 1)] = make_int2(node.x, ax | (ay << 16));
    }
    atomicAdd((unsigned long long*)&d->evals[pass], (unsigned long long)nv);
  }
}

// transformUpdate (LM.cpp:147-151) with the found pose as q_w_curr / t_w_curr and the last mapped sweep's odometry pose
struct RlPose { double v[7]; };
__global__ void rl_apply(LmScalars* __restrict__ s, RlPose p) {
  VL_PDL_WAIT();
  vl_transform_update(p.v, s->q_wodom, s->t_wodom, s->q_wmap_wodom, s->t_wmap_wodom);
}

// ---- host --------------------------------------------------------------------------------------------------------------------------
static int rl_fail(vloam_b200_ctx* c, int code, const char* msg) {
  snprintf(c->err, sizeof c->err, "relocalize: %s", msg);
  return code;
}

static void rl_qmul(const double a[4], const double b[4], double o[4]) {  // vl_qmul on the host (same operations)
  const double ax = a[0], ay = a[1], az = a[2], aw = a[3];
  const double bx = b[0], by = b[1], bz = b[2], bw = b[3];
  o[3] = aw * bw - ax * bx - ay * by - az * bz;
  o[0] = aw * bx + ax * bw + ay * bz - az * by;
  o[1] = aw * by + ay * bw + az * bx - ax * bz;
  o[2] = aw * bz + az * bw + ax * by - ay * bx;
}

void vl_rl_free(vloam_b200_ctx* c) {
  RlState* r = c->rl;
  if (!r) return;
  void* dev[] = {r->kept.p, r->u.p, r->cells.p, r->yaw.p, r->occ.p, r->topB.p, r->front[0].p, r->front[1].p, r->dev, r->sel};
  for (void* p : dev) vl_dev_free(c, p);
  if (r->h_dev) cudaFreeHost(r->h_dev);
  if (r->h_sel) cudaFreeHost(r->h_sel);
  for (int k = 0; k < 3; ++k) if (r->ev[k]) cudaEventDestroy(r->ev[k]);
  delete r;
  c->rl = nullptr;
}

static int rl_init(vloam_b200_ctx* c) {
  if (c->rl) return VLOAM_OK;
  RlState* r = new RlState();
  c->rl = r;
  VL_CUDA(cudaMalloc(&r->dev, sizeof(RlDev)));
  VL_CUDA(cudaMalloc(&r->sel, sizeof(RlSelectOut)));
  VL_CUDA(cudaMallocHost(&r->h_dev, sizeof(RlDev)));
  VL_CUDA(cudaMallocHost(&r->h_sel, sizeof(RlSelectOut)));
  __atomic_fetch_add(&c->regrows, 2LL, __ATOMIC_RELAXED);
  for (int k = 0; k < 3; ++k) VL_CUDA(cudaEventCreate(&r->ev[k]));
  return VLOAM_OK;
}

// The caller has drained the context (vloam_b200_synchronize) and checked the parameters.
int vl_rl_run(vloam_b200_ctx* c, const vloam_b200_reloc_params& P, const double qc_in[4], const double tc[3], vloam_b200_reloc_result* res) {
  if (!c->rlReady) return rl_fail(c, VLOAM_E_INVALID, "no mapped sweep since the context was created or its map was loaded");
  VL_TRY(vl_lm_sync_pools(c));  // in-place updates since the pools were last current are written back first
  VL_TRY(rl_init(c));
  RlState* R = c->rl;
  cudaStream_t st = c->stream;
  // R_c: the normalised quaternion through Eigen's toRotationMatrix (Quaternion.h)
  const double nq = sqrt(((qc_in[0] * qc_in[0] + qc_in[1] * qc_in[1]) + qc_in[2] * qc_in[2]) + qc_in[3] * qc_in[3]);
  const double q[4] = {qc_in[0] / nq, qc_in[1] / nq, qc_in[2] / nq, qc_in[3] / nq};
  const double tx = 2 * q[0], ty = 2 * q[1], tz = 2 * q[2], twx = tx * q[3], twy = ty * q[3], twz = tz * q[3];
  const double txx = tx * q[0], txy = ty * q[0], txz = tz * q[0], tyy = ty * q[1], tyz = tz * q[1], tzz = tz * q[2];
  const RlRot rot = {{1 - (tyy + tzz), txy - twz, txz + twy, txy + twz, 1 - (txx + tzz), tyz - twx, txz - twy, tyz + twx, 1 - (txx + tyy)}};
  const int Qc = c->h_lmm->Qc, Qs = c->h_lmm->Qs;
  VL_TRY(vl_reserve(c, R->kept, (size_t)max(Qc + Qs, 1)));
  VL_TRY(vl_reserve(c, R->u, (size_t)3 * P.max_points));
  VL_CUDA(cudaEventRecord(R->ev[0], st));
  VL_LAUNCH(rl_select, 1, 1024, 0, (const float4*)c->stackC.p, Qc, (const float4*)c->stackS.p, Qs, rot, P.max_range * P.max_range, P.max_points,
            (const MapCubeTable*)c->cubeC, (const MapCubeTable*)c->cubeS, R->kept.p, R->u.p, R->sel);
  VL_CUDA(cudaMemcpyAsync(R->h_sel, R->sel, sizeof(RlSelectOut), cudaMemcpyDeviceToHost, st));
  VL_CUDA(cudaStreamSynchronize(st));
  const RlSelectOut sel = *R->h_sel;
  if (sel.mapPoints == 0) return rl_fail(c, VLOAM_E_INVALID, "the map is empty");
  if (sel.m == 0) return rl_fail(c, VLOAM_E_INVALID, "no point of the last mapped sweep lies within max_range");
  // the discretisation (include/vloam_b200.h)
  const double r = P.resolution;
  const double dth = P.yaw_step_deg > 0 ? P.yaw_step_deg * M_PI / 180.0 : r / P.max_range;
  const int full = P.half_yaw_deg >= 180.0;
  const double nJd = full ? ceil(2.0 * M_PI / dth - 1e-9) : 2.0 * floor(P.half_yaw_deg * M_PI / 180.0 / dth + 1e-9) + 1.0;
  const double Nd = floor(P.half_xy / r), Nzd = floor(P.half_z / r);
  const double Sd = 2.0 * Nd + 1.0, nZd = 2.0 * Nzd + 1.0;
  const double Gxd = 2.0 * (ceil(P.max_range / r) + Nd + 1.0), Gzd = 2.0 * (ceil(sel.zmax / r) + Nzd + 1.0);
  if (Sd >= 32768.0) return rl_fail(c, VLOAM_E_CAPACITY, "at most 16383 translation steps per side (half_xy / resolution)");
  if (nJd * nZd * Sd * Sd > 2147483647.0) return rl_fail(c, VLOAM_E_CAPACITY, "more than 2^31 - 1 candidates (yaws x z offsets x xy offsets)");
  if (Gxd * Gxd * Gzd > 2147483647.0) return rl_fail(c, VLOAM_E_CAPACITY, "occupancy grid above 2^31 - 1 cells (max_range, half_xy, half_z)");
  RlSpace s;
  s.nJ = (int)nJd; s.N = (int)Nd; s.Nz = (int)Nzd; s.S = (int)Sd; s.nZ = (int)nZd; s.m = sel.m; s.full = full;
  s.Gx = s.Gy = (int)Gxd; s.Gz = (int)Gzd;
  s.H = 0; while ((1 << s.H) < s.S) ++s.H;
  s.levelCells = (size_t)s.Gx * s.Gy * s.Gz;
  s.dtheta = dth; s.r = r; s.exclM = P.exclusion_m; s.exclRad = P.exclusion_deg * M_PI / 180.0;
  const long long nTop = (long long)s.nJ * s.nZ;
  const long long frontCap = nTop * (long long)((s.S + 1) / 2) * ((s.S + 1) / 2);  // the full node count of level 1, the largest stored level
  RlGrid g;
  for (int a = 0; a < 3; ++a) g.tc[a] = tc[a];
  g.o[0] = tc[0] - r * (double)(s.Gx / 2); g.o[1] = tc[1] - r * (double)(s.Gy / 2); g.o[2] = tc[2] - r * (double)(s.Gz / 2);
  g.r = r;
  R->yawTab.resize((size_t)2 * s.nJ);
  const int j0 = full ? 0 : s.nJ / 2;
  for (int j = 0; j < s.nJ; ++j) { const double th = (double)(j - j0) * dth; R->yawTab[2 * j] = cos(th); R->yawTab[2 * j + 1] = sin(th); }
  VL_TRY(vl_reserve(c, R->yaw, (size_t)s.nJ));
  VL_TRY(vl_reserve(c, R->cells, (size_t)s.nJ * s.m));
  VL_TRY(vl_reserve(c, R->occ, s.levelCells * (s.H + 2)));  // levels 0..H and the separable passes' scratch
  VL_TRY(vl_reserve(c, R->topB, (size_t)nTop));
  if (s.H > 0) for (int k = 0; k < 2; ++k) VL_TRY(vl_reserve(c, R->front[k], (size_t)max(frontCap, 1LL)));
  VL_CUDA(cudaMemcpyAsync(R->yaw.p, R->yawTab.data(), (size_t)s.nJ * sizeof(double2), cudaMemcpyHostToDevice, st));
  VL_CUDA(cudaMemsetAsync(R->occ.p, 0, s.levelCells, st));
  VL_CUDA(cudaMemsetAsync(R->dev, 0, sizeof(RlDev), st));
  VL_LAUNCH(rl_cells, min(vl_div_up((long long)s.nJ * s.m, 256), c->num_sms * 16), 256, 0, (const double*)R->u.p, s.m, s.nJ,
            (const double2*)R->yaw.p, g, R->cells.p);
  VL_LAUNCH(rl_occ, dim3(VL_CUBE_NUM, 2), 256, 0, (const LmScalars*)c->lmm, (const MapCubeTable*)c->cubeC, (const MapCubeTable*)c->cubeS,
            (const float4*)c->poolC.p, (const float4*)c->poolS.p, g, s.Gx, s.Gy, s.Gz, R->occ.p);
  const int gsCells = (int)min((long long)vl_div_up((long long)s.levelCells, 256), (long long)c->num_sms * 16);
  unsigned char* tmp = R->occ.p + (size_t)(s.H + 1) * s.levelCells;
  for (int h = 1; h <= s.H; ++h) {
    const int d = 1 << (h - 1);
    VL_LAUNCH(rl_pool, gsCells, 256, 0, (const unsigned char*)(R->occ.p + (size_t)(h - 1) * s.levelCells), tmp, s.Gx, s.Gy, s.levelCells, d, 0);
    VL_LAUNCH(rl_pool, gsCells, 256, 0, (const unsigned char*)tmp, R->occ.p + (size_t)h * s.levelCells, s.Gx, s.Gy, s.levelCells, d, 1);
  }
  VL_CUDA(cudaEventRecord(R->ev[1], st));
  s.cells = R->cells.p; s.occ = R->occ.p;
  const int warpBlocks = vl_div_up(nTop * 32, 256);
  for (int pass = 0; pass < 2; ++pass) {
    VL_LAUNCH(rl_top, warpBlocks, 256, 0, s, R->dev, pass, R->topB.p);
    if (s.H == 0) continue;
    VL_LAUNCH(rl_greedy, warpBlocks, 256, 0, s, R->dev, pass, (const int*)R->topB.p);
    VL_LAUNCH(rl_seed, vl_div_up(nTop, 256), 256, 0, s, R->dev, pass, (const int*)R->topB.p, R->front[s.H & 1].p);
    for (int h = s.H; h >= 1; --h)
      VL_LAUNCH(rl_expand, c->num_sms * 8, 256, 0, s, R->dev, pass, h, (const int2*)R->front[h & 1].p, R->front[(h - 1) & 1].p);
  }
  VL_CUDA(cudaEventRecord(R->ev[2], st));
  VL_CUDA(cudaMemcpyAsync(R->h_dev, R->dev, sizeof(RlDev), cudaMemcpyDeviceToHost, st));
  VL_CUDA(cudaStreamSynchronize(st));
  VL_CUDA(cudaGetLastError());
  const RlDev out = *R->h_dev;
  R->last = out; R->m = s.m; R->Gx = s.Gx; R->Gy = s.Gy; R->Gz = s.Gz;
  for (int a = 0; a < 3; ++a) R->o[a] = g.o[a];
  VL_CUDA(cudaEventElapsedTime(&R->ms[0], R->ev[0], R->ev[2]));
  VL_CUDA(cudaEventElapsedTime(&R->ms[1], R->ev[0], R->ev[1]));
  // candidate index -> pose: R = Rz(theta_j) R_c as the quaternion product qz(theta_j) * q_c, t = t_c + r (ix, iy, iz)
  auto pose = [&](unsigned long long key, double qo[4], double to[3], long long* idx) -> int {
    if (key == 0) { for (int k = 0; k < 4; ++k) qo[k] = 0; for (int k = 0; k < 3; ++k) to[k] = 0; *idx = -1; return -1; }
    const long long lin = (long long)(unsigned)~(unsigned)(key & 0xffffffffull);
    const int ax = (int)(lin % s.S), ay = (int)((lin / s.S) % s.S), izz = (int)((lin / ((long long)s.S * s.S)) % s.nZ);
    const int jj = (int)(lin / ((long long)s.S * s.S * s.nZ));
    const double th = (double)(jj - j0) * dth;
    const double qz[4] = {0.0, 0.0, sin(th / 2.0), cos(th / 2.0)};
    rl_qmul(qz, q, qo);
    to[0] = tc[0] + r * (double)(ax - s.N); to[1] = tc[1] + r * (double)(ay - s.N); to[2] = tc[2] + r * (double)(izz - s.Nz);
    *idx = lin;
    return (int)(key >> 32);
  };
  res->score = pose(out.key[0], res->q, res->t, &res->index);
  res->runner_score = pose(out.key[1], res->runner_q, res->runner_t, &res->runner_index);
  res->n_points = s.m;
  res->found = (double)res->score >= P.min_score * (double)s.m ? 1 : 0;
  res->candidates = nTop * s.S * s.S;
  res->nodes = out.evals[0] + out.evals[1];
  if (P.apply && res->found) {
    RlPose p;
    for (int k = 0; k < 4; ++k) p.v[k] = res->q[k];
    for (int k = 0; k < 3; ++k) p.v[4 + k] = res->t[k];
    VL_LAUNCH(rl_apply, 1, 1, 0, c->lmm, p);
    VL_CUDA(cudaStreamSynchronize(st));
  }
  VL_CUDA(cudaGetLastError());
  return VLOAM_OK;
}

// debug getters of the last search: rl.points, rl.occ, rl.yaw, rl.levels, rl.ms (capi.cu's vloam_b200_debug_get)
long vl_rl_debug(vloam_b200_ctx* c, const char* name, void* out, long cap) {
  const std::string n(name);
  RlState* R = c->rl;
  if (!R || R->m == 0) { snprintf(c->err, sizeof c->err, "%s: no relocalize call yet", n.c_str()); return VLOAM_E_INVALID; }
  std::vector<char> buf;
  if (n == "rl.points") {
    buf.resize((size_t)R->m * 24);
    VL_CUDA(cudaMemcpy(buf.data(), R->u.p, buf.size(), cudaMemcpyDeviceToHost));
  } else if (n == "rl.occ") {  // double origin[3], int64 dims[3] (x fastest), then the level-0 bytes
    const size_t cells = (size_t)R->Gx * R->Gy * R->Gz;
    buf.resize(48 + cells);
    const long long dims[3] = {R->Gx, R->Gy, R->Gz};
    memcpy(buf.data(), R->o, 24); memcpy(buf.data() + 24, dims, 24);
    VL_CUDA(cudaMemcpy(buf.data() + 48, R->occ.p, cells, cudaMemcpyDeviceToHost));
  } else if (n == "rl.yaw") {
    buf.resize(R->yawTab.size() * 8);
    memcpy(buf.data(), R->yawTab.data(), buf.size());
  } else if (n == "rl.levels") {  // int64 [2][RL_MAX_LEVELS] frontier nodes kept per level (pass 0: best, 1: runner-up), then evals[2]
    long long v[2 * RL_MAX_LEVELS + 2];
    for (int p = 0; p < 2; ++p) for (int h = 0; h < RL_MAX_LEVELS; ++h) v[p * RL_MAX_LEVELS + h] = R->last.nFront[p][h];
    v[2 * RL_MAX_LEVELS] = R->last.evals[0]; v[2 * RL_MAX_LEVELS + 1] = R->last.evals[1];
    buf.resize(sizeof v); memcpy(buf.data(), v, sizeof v);
  } else if (n == "rl.ms") {  // device time of the last call {whole search, occupancy + pyramid} in ms
    buf.resize(sizeof R->ms); memcpy(buf.data(), R->ms, sizeof R->ms);
  } else {
    snprintf(c->err, sizeof c->err, "unknown buffer name '%s'", n.c_str());
    return VLOAM_E_NAME;
  }
  if (out && cap >= (long)buf.size()) memcpy(out, buf.data(), buf.size());
  return (long)buf.size();
}

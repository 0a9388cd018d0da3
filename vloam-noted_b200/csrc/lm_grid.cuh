// lm_grid.cuh -- the laserMapping sub-map as a PERSISTENT device voxel-hash grid (north star: "map held as a device
// voxel-hash grid"; VERDICT r1 "missing" 4 / "next" 5).
//
// The reference rebuilds two KD-trees over the ~1M-point sub-map every sweep (LM.cpp:519-520) and re-filters all 75 valid
// cubes (LM.cpp:795-808); round 1 did the GPU analogue (gather + counting sort of 1M points, rewrite of every cube) per
// sweep: ~120 MB of DRAM traffic for ~15k points that actually change.  Here the points of the 75 valid cubes live in
// a search structure that is UPDATED IN PLACE:
//
//   cell directory   dir[kind][125 x 125 x 75]  {count, head chunk}    2 m cells over the 250 x 250 x 150 m window
//   chunks           16 entries each: pts[] (x, y, z, intensity), key[] ((valid slot << 32) | voxel key), next[]
//
// kNN visits the 27 cells around a query exactly as before (SURVEY A.2: exact inside the 1 m acceptance ball); ties are
// ordered by key = (valid-cube slot, voxel key), which is the order of the canonical point ids (position in the
// concatenated sub-map cloud, LM.cpp:476-485) because a filtered cube is sorted by voxel key.  The per-sweep map update
// (LM.cpp:741-808) becomes: group the ~7-15k new points by (cube, voxel) in a small hash table (no sort), find the map point of
// each voxel IN THE GRID (it lies in one of the <= 8 cells the voxel's box overlaps), fold the group in the reference's order (map
// point first, then the new points in stack order, f32), and store the centroid back -- in place, or as a new entry; an entry stays
// listed in its cell when its centroid slides into the neighbouring one (exact for leaf <= 0.95 m, see mu_apply).  The per-cube
// sorted pools of laser_mapping.cu stay the exchange format (export, window moves, raw tails): they are brought up to date from
// the grid only when needed -- every entry remembers its position in its cube's pool segment (refreshed in place), the
// voxels created since go through ONE pass of the pool path's merge (rf_*), which puts them at their sorted positions.
//
// Anything the in-place update does not handle exactly -- a window move, a cube with an unfiltered tail, a centroid
// that rounds across its voxel boundary (the next VoxelGrid pass then re-keys it: LM.cpp:795-808 on a drifted point) --
// raises `dirty` / a window mismatch, and that sweep takes the pool path of round 1 (bit-identical by construction,
// test_speculative_submap_equals_inline_build / test_grid_update_equals_pool_update).
#pragma once
#include <cuda_runtime.h>

#define LG_C 16                    // entries per chunk
#define LG_TAIL (1u << 31)         // key low word: unfiltered tail point, ordered by its position in the cube
#define LG_DEAD (~0ull)            // tombstone (pts.x = +inf as well: never a neighbour, never a match)

struct LgHeader {  // device: which window / map state the grid describes
  int valid;                         // built and in step with the map
  int dirty;                         // an entry needs the pool path (tail point, drifted centroid) or a chunk allocation failed
  int cI, cJ, cK, cenW, cenH, cenD;  // window centre cube and laserCloudCen* it was built for
  int validNum;                      // the valid-cube list the keys' slots refer to (LM.cpp:448-466 for that centre)
  int validInd[125];
  int count[2];                      // live points per kind (== Mc, Ms of LM.cpp:476-485)
  int dead;                          // tombstoned entries since the last rebuild
  int nOps;                          // pending inserts of the running update
  float origin[3];
};

struct LgGrid {  // passed by value to kernels
  int2* dir;                    // [2 * LM_NCELL] {count, head}
  float4* pts;                  // [cap * LG_C]
  unsigned long long* key;      // [cap * LG_C]
  int* next;                    // [cap]
  int* posOf;                   // [cap * LG_C] position of the entry in its cube's pool segment when the grid was built, -1 = voxel created since
  int* top;                     // chunk bump pointer
  int cap;                      // chunks
  LgHeader* hdr;
};

// Append one entry to a cell.  The position is claimed with one atomic; the chain is extended with a CAS (a thread that
// loses the race leaks its chunk: the bump allocator is reset at the next rebuild).  A new chunk is filled with tombstone
// keys BEFORE it is published, so a thread that scans a cell while another one appends to it reads either a dead key or
// a finished one (8-byte stores are atomic): the in-place update can look voxels up and insert new ones in one kernel.
__device__ __forceinline__ int lg_insert(const LgGrid& g, int cell, const float4 p, unsigned long long key, int poolPos) {
  int2* d = &g.dir[cell];
  const int pos = atomicAdd(&d->x, 1);
  const int k = pos / LG_C;
  int* link = &d->y;
  int chunk = -1;
  for (int j = 0; j <= k; ++j) {
    int cur = *(volatile int*)link;
    if (cur < 0) {
      const int nw = atomicAdd(g.top, 1);
      if (nw >= g.cap) { g.hdr->dirty = 1; return -1; }  // cannot happen when the host sized the chunk pool (it bounds the demand before every launch);
                                                         // the claimed slot stays unwritten, `dirty` forces a rebuild before the next read
      g.next[nw] = -1;
      ulonglong2* kk = reinterpret_cast<ulonglong2*>(g.key + (size_t)nw * LG_C);
#pragma unroll
      for (int q = 0; q < LG_C / 2; ++q) kk[q] = make_ulonglong2(LG_DEAD, LG_DEAD);
      __threadfence();
      const int old = atomicCAS(link, -1, nw);
      cur = old < 0 ? nw : old;
    }
    chunk = cur;
    link = &g.next[cur];
  }
  const int e = chunk * LG_C + (pos % LG_C);
  g.pts[e] = p;
  g.posOf[e] = poolPos;
  // (no fence: a concurrent scanner only ever reads pts[] of the entry whose key it was looking for, and this key is another voxel's)
  *(volatile unsigned long long*)&g.key[e] = key;
  return e;
}

// entry key: (valid slot << 32) | voxel key, or | (LG_TAIL | position in the cube) for an unfiltered tail point
__device__ __forceinline__ unsigned long long lg_key(int slot, unsigned low) { return ((unsigned long long)slot << 32) | low; }
__device__ __forceinline__ int lg_key_slot(unsigned long long key) { return (int)(key >> 32); }
__device__ __forceinline__ unsigned lg_key_vox(unsigned long long key) { return (unsigned)key & 0x3fffffffu; }

// Every live entry of both kinds' cells (ncell per kind), one cell per thread of a grid-stride loop: f(entry, key, kind).
template <typename F>
__device__ __forceinline__ void lg_for_each_live(const LgGrid& g, int ncell, F f) {
  for (int cell = blockIdx.x * blockDim.x + threadIdx.x; cell < 2 * ncell; cell += gridDim.x * blockDim.x) {
    const int2 d = g.dir[cell];
    const int kind = cell >= ncell;
    int chunk = d.y;
    for (int left = d.x; left > 0; left -= LG_C, chunk = left > 0 ? g.next[chunk] : -1) {
      const int m = min(left, LG_C);
      for (int i = 0; i < m; ++i) {
        const int e = chunk * LG_C + i;
        const unsigned long long key = g.key[e];
        if (key != LG_DEAD) f(e, key, kind);
      }
    }
  }
}

// key order == canonical id order; refs < 0 (empty list slot) sort last
__device__ __forceinline__ bool lg_key_less(const LgGrid& g, int a, int b) {
  if (b < 0) return a >= 0;
  if (a < 0) return false;
  return g.key[a] < g.key[b];
}

// LiDAR/radar hard voxelizer, VFE mean and pillar scatter (sm_100a).
//
// Reference contract being replaced (third-party, reached through models/bev_depth.py:181-183 of
// the reference; semantics restated in SURVEY.md Appendix A from mmcv-full 1.7.0 /
// mmdet3d 1.0.0rc4): `hard_voxelize` is *serial in point order* -- a voxel is created at the
// first in-range point of its cell, at most max_voxels voxels exist (later cells are dropped
// entirely), and the first max_points points of a voxel are kept in order.
//
// Two pipelines with identical outputs: grids of up to 2^26 cells per batch (every pillar / voxel grid of the reference) take
// the DENSE-TABLE path further down (first-point table, tickets + eviction, cooperative finalize, dense canvas); larger grids
// take the hash path described here.
// Parallel formulation with bit-identical results (hash path):
//   1. warp-cooperative hash insert of (sample, cell) keys; per slot atomicMin of the point
//      index  -> first-occurrence point of every cell (order independent)
//   2. flag "point is the first of its cell" -> exclusive scan in point order = voxel id
//      (mmcv's voxel numbering), capped at max_voxels
//   3. per voxel, the max_points smallest point indices via a chain of atomicMin on a sorted
//      slot list (each slot ends up holding the r-th smallest index whatever the interleaving)
//   4. gather: every row of voxels / num_points / coors / mean is written, rows beyond the voxel
//      count as zeros; optional fused VFE mean (HardSimpleVFE) and its canvas (live rows only)
// mmcv's own deterministic CUDA path needs an O(N^2) predecessor scan and a single-thread
// numbering kernel for the same result.
#include "common.cuh"
#include "scan.cuh"
#include "tma.cuh"

#include <cstdlib>

namespace bevpool {

constexpr unsigned long long kEmptyKey = ~0ull;
constexpr int32_t kEmptyIdx = 0x7f7f7f7f;   // what cudaMemset(0x7f) writes

struct VoxGeom {
  float vx, vy, vz, xmin, ymin, zmin;
  int gx, gy, gz;
  float ivx, ivy, ivz;                       // 1 / voxel size, rounded to float (point_to_cell_fast)
};

// IEEE float32 subtract, true division, floor -- exactly mmcv's `floor((p - min) / voxel_size)`.
// NaN and out-of-int-range values compare false / out of range and are dropped.
__device__ __forceinline__ bool point_to_cell(const float *p, const VoxGeom &g, int &x, int &y, int &z) {
  const float fx = floorf(__fdiv_rn(__fsub_rn(p[0], g.xmin), g.vx));
  const float fy = floorf(__fdiv_rn(__fsub_rn(p[1], g.ymin), g.vy));
  const float fz = floorf(__fdiv_rn(__fsub_rn(p[2], g.zmin), g.vz));
  const bool ok = fx >= 0.f && fx < (float)g.gx && fy >= 0.f && fy < (float)g.gy && fz >= 0.f && fz < (float)g.gz;
  x = ok ? (int)fx : -1;
  y = ok ? (int)fy : -1;
  z = ok ? (int)fz : -1;
  return ok;
}

// The same result with ONE rare branch instead of three IEEE divisions.  q' = (p - min) * (1 / v) differs from the
// correctly rounded quotient by less than 7.3e-4 while |q'| < 4096 (two roundings of 2^-24 on q', one on the quotient):
// when q' is farther than 1e-3 from every integer both floor to the same value; otherwise -- and for huge or NaN
// coordinates, which compare false -- the exact expression decides.
__device__ __forceinline__ bool point_to_cell_fast(const float *p, const VoxGeom &g, int &x, int &y, int &z) {
  const float tx = __fsub_rn(p[0], g.xmin), ty = __fsub_rn(p[1], g.ymin), tz = __fsub_rn(p[2], g.zmin);
  const float qx = __fmul_rn(tx, g.ivx), qy = __fmul_rn(ty, g.ivy), qz = __fmul_rn(tz, g.ivz);
  const float dx = fabsf(qx - rintf(qx)), dy = fabsf(qy - rintf(qy)), dz = fabsf(qz - rintf(qz));
  const float big = fmaxf(fmaxf(fabsf(qx), fabsf(qy)), fabsf(qz));
  float fx, fy, fz;
  if (fminf(fminf(dx, dy), dz) > 1e-3f && big < 4096.f) {
    fx = floorf(qx); fy = floorf(qy); fz = floorf(qz);
  } else {
    fx = floorf(__fdiv_rn(tx, g.vx)); fy = floorf(__fdiv_rn(ty, g.vy)); fz = floorf(__fdiv_rn(tz, g.vz));
  }
  const bool ok = fx >= 0.f && fx < (float)g.gx && fy >= 0.f && fy < (float)g.gy && fz >= 0.f && fz < (float)g.gz;
  x = ok ? (int)fx : -1;
  y = ok ? (int)fy : -1;
  z = ok ? (int)fz : -1;
  return ok;
}

__device__ __forceinline__ uint32_t hash_u64(unsigned long long k) {
  k ^= k >> 33;
  k *= 0xff51afd7ed558ccdull;
  k ^= k >> 33;
  return (uint32_t)k;
}

// ---- 1. hash insert --------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
vox_insert_kernel(const float *__restrict__ points, const int32_t *__restrict__ offsets, int F, VoxGeom g,
                  unsigned long long *__restrict__ keys, int32_t *__restrict__ first, uint32_t hmask,
                  int32_t *__restrict__ point_slot) {
  const int b = blockIdx.y;
  const int begin = offsets[b], end = offsets[b + 1];
  const int i = begin + blockIdx.x * blockDim.x + threadIdx.x;
  const bool in = i < end;
  int x, y, z;
  unsigned long long key = kEmptyKey;
  if (in && point_to_cell(points + (int64_t)i * F, g, x, y, z))
    key = (unsigned long long)b * ((unsigned long long)g.gx * g.gy * g.gz) +
          ((unsigned long long)z * g.gy + y) * g.gx + x;
  // one probe sequence per distinct key in the warp; the lowest lane holds the lowest index
  const unsigned peers = __match_any_sync(0xffffffffu, key);
  const int lane = threadIdx.x & 31;
  const int leader = __ffs(peers) - 1;
  int slot = -1;
  if (key != kEmptyKey && lane == leader) {
    uint32_t s = hash_u64(key) & hmask;
    while (true) {
      const unsigned long long prev = atomicCAS(keys + s, kEmptyKey, key);
      if (prev == kEmptyKey || prev == key) break;
      s = (s + 1) & hmask;
    }
    atomicMin(first + s, i);
    slot = (int)s;
  }
  slot = __shfl_sync(0xffffffffu, slot, leader);
  if (in) point_slot[i] = key != kEmptyKey ? slot : -1;
}

// ---- 2. first-occurrence flags (scanned afterwards) -----------------------------------------------
__global__ void vox_flag_kernel(const int32_t *__restrict__ point_slot, const int32_t *__restrict__ first,
                                int64_t n, uint32_t *__restrict__ flags) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i > n) return;
  uint32_t f = 0;
  if (i < n) {
    const int s = point_slot[i];
    f = (s >= 0 && first[s] == (int32_t)i) ? 1u : 0u;
  }
  flags[i] = f;   // element n stays 0: the scan leaves the grand total there
}

// per-sample voxel counts (capped) and output row bases; B is small, one thread is enough
__global__ void vox_base_kernel(const uint32_t *__restrict__ prefix, const int32_t *__restrict__ offsets,
                                int batch, int max_voxels, int32_t *__restrict__ voxel_base) {
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    int run = 0;
    for (int b = 0; b < batch; ++b) {
      voxel_base[b] = run;
      const int distinct = (int)(prefix[offsets[b + 1]] - prefix[offsets[b]]);
      run += distinct < max_voxels ? distinct : max_voxels;
    }
    voxel_base[batch] = run;
  }
}

// ---- 3. assign points to voxel slots (first max_points indices, ascending) ---------------------------
__global__ void __launch_bounds__(256)
vox_assign_kernel(const float *__restrict__ points, const int32_t *__restrict__ offsets, int F, VoxGeom g,
                  const int32_t *__restrict__ point_slot, const int32_t *__restrict__ first,
                  const uint32_t *__restrict__ prefix, const int32_t *__restrict__ voxel_base, int max_voxels,
                  int max_points, int32_t *__restrict__ lists, int32_t *__restrict__ counts,
                  int32_t *__restrict__ coors) {
  const int b = blockIdx.y;
  const int begin = offsets[b], end = offsets[b + 1];
  const int i = begin + blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= end) return;
  const int s = point_slot[i];
  if (s < 0) return;
  const int f = first[s];
  const int vid = (int)(prefix[f] - prefix[begin]);
  if (vid >= max_voxels) return;                       // voxel cap: the whole cell is dropped
  const int row = voxel_base[b] + vid;
  if (i == f) {                                        // the creating point records the coordinates
    int x, y, z;
    point_to_cell(points + (int64_t)i * F, g, x, y, z);
    reinterpret_cast<int4 *>(coors)[row] = make_int4(b, z, y, x);
  }
  atomicAdd(counts + row, 1);
  int32_t *list = lists + (int64_t)row * max_points;
  // hint: once the last slot holds a smaller index this point can never enter the list
  if (*reinterpret_cast<volatile int32_t *>(list + max_points - 1) < i) return;
  int v = i;
  for (int r = 0; r < max_points; ++r) {
    const int old = atomicMin(list + r, v);
    if (old == kEmptyIdx) break;
    v = old > v ? old : v;                              // carry the larger one to the next slot
  }
}

// ---- 4. gather ---------------------------------------------------------------------------------
// one warp per row of the padded output (batch * max_voxels rows): copies max_points x F floats (zeros for unused
// slots), writes num_points and, optionally, the mean of the first `mean_features` columns (HardSimpleVFE) and its
// canvas cells (batch, mean_features, gz, gy, gx), zero-filled before.  Rows >= voxel_base[batch] are written as zeros
// (voxels, num_points, coors, mean) and never reach the canvas.
__global__ void __launch_bounds__(256)
vox_gather_kernel(const float *__restrict__ points, int F, const int32_t *__restrict__ lists,
                  const int32_t *__restrict__ counts, const int32_t *__restrict__ voxel_base, int batch,
                  int64_t total_rows, int max_points, float *__restrict__ voxels, int32_t *__restrict__ num_points,
                  int32_t *__restrict__ coors, float *__restrict__ voxel_mean, int mean_features, VoxGeom g,
                  float *__restrict__ canvas) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= total_rows) return;
  const bool live = row < voxel_base[batch];
  const int32_t *list = lists + (int64_t)row * max_points;
  const int cnt = live ? min(counts[row], max_points) : 0;
  float *vout = voxels + (int64_t)row * max_points * F;
  const int total = max_points * F;
  for (int e = lane; e < total; e += 32) {
    const int t = e / F, c = e - t * F;
    float v = 0.f;
    if (t < cnt) v = __ldg(points + (int64_t)list[t] * F + c);
    vout[e] = v;
  }
  if (lane == 0) {
    num_points[row] = cnt;
    if (!live) reinterpret_cast<int4 *>(coors)[row] = make_int4(0, 0, 0, 0);   // (live rows: vox_assign_kernel)
  }
  if ((voxel_mean || canvas) && lane < mean_features) {
    float m = 0.f;
    if (live) {
      float s = 0.f;
      for (int t = 0; t < cnt; ++t) s += __ldg(points + (int64_t)list[t] * F + lane);   // sequential, slot order
      m = s / (float)cnt;
    }
    if (voxel_mean) voxel_mean[(int64_t)row * mean_features + lane] = m;
    if (canvas && live) {
      const int4 c = reinterpret_cast<const int4 *>(coors)[row];                        // (b, z, y, x)
      canvas[((((int64_t)c.x * mean_features + lane) * g.gz + c.y) * g.gy + c.z) * g.gx + c.w] = m;
    }
  }
}

// ---- dynamic voxelization: per-point (z, y, x) or -1 -----------------------------------------------
__global__ void vox_dynamic_kernel(const float *__restrict__ points, int64_t n, int F, VoxGeom g,
                                   int32_t *__restrict__ coors) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int x, y, z;
  point_to_cell(points + i * F, g, x, y, z);
  coors[i * 3 + 0] = z;
  coors[i * 3 + 1] = y;
  coors[i * 3 + 2] = x;
}

// ---- pillar scatter --------------------------------------------------------------------------------
__global__ void scatter_index_kernel(const int32_t *__restrict__ coors, int64_t M, int batch, int nz, int ny,
                                     int nx, int32_t *__restrict__ index_map) {
  const int64_t m = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= M) return;
  const int4 c = reinterpret_cast<const int4 *>(coors)[m];   // (b, z, y, x)
  if (c.x < 0 || c.x >= batch || c.y < 0 || c.y >= nz || c.z < 0 || c.z >= ny || c.w < 0 || c.w >= nx) return;
  // duplicates cannot come from hard voxelization; if a caller has them, the highest row wins (deterministic)
  atomicMax(index_map + (((int64_t)c.x * nz + c.y) * ny + c.z) * nx + c.w, (int)m);
}

// canvas (B, C, nz, ny, nx): every element written exactly once (feature or zero), coalesced along x
template <typename T>
__global__ void __launch_bounds__(256)
scatter_canvas_kernel(const T *__restrict__ feats, const int32_t *__restrict__ index_map, int C,
                      int64_t cells_per_sample, T *__restrict__ canvas) {
  const int b = blockIdx.y;
  const int64_t cell = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (cell >= cells_per_sample) return;
  const int m = index_map[(int64_t)b * cells_per_sample + cell];
  T *out = canvas + (int64_t)b * C * cells_per_sample + cell;
  if (m < 0) {
    const T z = T(0.f);
    for (int c = 0; c < C; ++c) out[(int64_t)c * cells_per_sample] = z;
  } else {
    const T *row = feats + (int64_t)m * C;
    for (int c = 0; c < C; ++c) out[(int64_t)c * cells_per_sample] = row[c];
  }
}

template <typename T>
__global__ void scatter_backward_kernel(const T *__restrict__ grad_canvas, const int32_t *__restrict__ coors,
                                        int64_t M, int C, int batch, int nz, int ny, int nx,
                                        T *__restrict__ grad_feats) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= M * C) return;
  const int64_t m = e / C;
  const int c = (int)(e - m * C);
  const int4 co = reinterpret_cast<const int4 *>(coors)[m];
  T v = T(0.f);
  if (co.x >= 0 && co.x < batch && co.y >= 0 && co.y < nz && co.z >= 0 && co.z < ny && co.w >= 0 && co.w < nx) {
    const int64_t cells = (int64_t)nz * ny * nx;
    v = grad_canvas[((int64_t)co.x * C + c) * cells + ((int64_t)co.y * ny + co.z) * nx + co.w];
  }
  grad_feats[e] = v;
}

// ==== dense-grid path (grids that fit a per-cell table: the aiMotive pillar grid is 2048 x 256 x 1) =================
// The hash table is replaced by what mmcv's own CPU kernel uses, a dense cell -> first-point table, and the
// pipeline is 6 kernels for the whole batch, with no per-voxel index lists and no per-point prefix array:
//   A vox_cell_kernel      a tile of 1024 points = one contiguous span of the cloud brought into shared memory by ONE
//                          TMA bulk copy (a point row is F*4 = 20 bytes: no wider aligned per-thread access exists),
//                          global cell id per point, warp-aggregated atomicMin -> first point of every cell
//   B vox_scan_kernel      per sample: "first point of its cell" flags computed on the fly + decoupled look-back scan
//                          = voxel numbering in point order; the creating point overwrites its cell's entry of the
//                          first-point table with ~vid (one table serves both lookups) and publishes
//                          cell_of_vid[sample][vid]
//   C vox_claim_kernel     per kept point: cell -> voxel number -> a ticket from the voxel's arrival counter; tickets
//     vox_evict_kernel     below max_points are slots of the voxel's list (words = 0x7fffffff - index), later arrivals go
//                          to the tile's overflow segment and are swapped in by compare-and-swap when they are earlier
//                          than the row's latest point (see the kernels).  The lists are a compact array that stays in
//                          L2 -- atomics on the padded voxel tensor itself (15 x F floats per row, far larger than L2)
//                          ran at DRAM random-access speed, 4x slower
//   D vox_finalize_*       one warp per 32 voxel rows: slot words sorted in registers -> point rows gathered into a
//                          shared-memory tile that leaves as one contiguous, coalesced span of the padded voxel
//                          tensor (93 % of it is zeros: written once, by this kernel, at streaming-store speed);
//                          count, coordinates, HardSimpleVFE mean in slot order
//   E vox_canvas_dense_kernel  the pillar scatter of that mean as ONE in-order pass over the canvas (no zero fill, no
//                          scattered stores); without a mean output the canvas is zero-filled on a side stream and the
//                          finalize kernel scatters into it
// The clouds may be given as one concatenated tensor or as a device array of per-sample pointers (no torch.cat).
constexpr int kVcThreads = 256;
constexpr int kVoxMaxF = 16;
constexpr int32_t kVoxIdxBias = 0x7fffffff;          // slot word = kVoxIdxBias - point index  (> 0; 0 = empty)

struct VoxPoints {                                   // point i of sample b (i global, begin = offsets[b])
  const float *cat;                                  // concatenated (total, F), or
  const float *const *per_sample;                    // device array of B base pointers
  __device__ __forceinline__ const float *row(int b, int begin, int i, int F) const {
    return per_sample ? per_sample[b] + (int64_t)(i - begin) * F : cat + (int64_t)i * F;
  }
};

constexpr int kVcPer = 4;                          // points per thread: independent chains in flight, 4x fewer CTAs
constexpr int kVcTile = kVcThreads * kVcPer;       // points per tile (the claim / evict kernels use the same tiles)
// One tile per CTA, 8 resident CTAs per SM at the pillar shape.  (Tried: persistent CTAs over the tiles with two buffers,
// the bulk copy of the next tile in flight behind the current one -- the same 48-50 us: with one tile of prefetch per
// CTA the copy latency is no better hidden than by the neighbouring CTAs.)
__global__ void __launch_bounds__(kVcThreads)
vox_cell_kernel(VoxPoints pts, const int32_t *__restrict__ offsets, int F, VoxGeom g, int64_t cells,
                int32_t *__restrict__ first, int32_t *__restrict__ point_gcell, int l2_hints) {
  extern __shared__ __align__(16) float s_pts[];   // kVcTile * F floats
  __shared__ __align__(8) uint64_t s_bar;
  const int b = blockIdx.y;
  const int begin = offsets[b], end = offsets[b + 1];
  const int tile0 = begin + blockIdx.x * kVcTile;
  if (tile0 >= end) return;
  const int npts = min(kVcTile, end - tile0);
  const float *src = pts.row(b, begin, tile0, F);
  // the tile is one contiguous span of the cloud: ONE bulk copy (TMA, SASS UBLKCP) when its address and size are
  // multiples of 16 bytes (always for full tiles of a 16-byte aligned cloud), else 4-byte loads (a point row is F*4 = 20
  // bytes: no wider aligned per-thread access exists)
  const uint32_t bytes = (uint32_t)npts * (uint32_t)F * 4u;
  if (((reinterpret_cast<uintptr_t>(src) | bytes) & 15u) == 0) {
    if (threadIdx.x == 0) {
      mbar_init(&s_bar, 1);
      fence_mbar_init();
      mbar_expect_tx(&s_bar, bytes);
      if (l2_hints & 4) tma_load_1d_hint(s_pts, src, bytes, &s_bar, l2_policy_evict_first());   // (re-read by the gather, much later)
      else tma_load_1d(s_pts, src, bytes, &s_bar);
    }
    __syncthreads();                               // (the barrier is initialised before anybody polls it)
    mbar_wait(&s_bar, 0);
  } else {
    for (int e = threadIdx.x; e < npts * F; e += kVcThreads) s_pts[e] = ldg_stream_f32(src + e);
    __syncthreads();
  }
  // the table is visited at random by three kernels of the call: evict_last keeps its lines ahead of the streams
  const uint64_t pol = (l2_hints & 1) ? l2_policy_evict_last() : l2_policy_evict_normal();
  int gcell[kVcPer];
#pragma unroll
  for (int k = 0; k < kVcPer; ++k) {
    const int p = k * kVcThreads + threadIdx.x;     // consecutive lanes = consecutive points
    gcell[k] = -1;
    if (p < npts) {
      int x, y, z;
      if (point_to_cell_fast(s_pts + p * F, g, x, y, z)) gcell[k] = (int)((int64_t)b * cells + ((int64_t)z * g.gy + y) * g.gx + x);
      point_gcell[tile0 + p] = gcell[k];
    }
  }
  // first point of every cell: one fire-and-forget red.min per kept point.  (Aggregating the points of a warp that share
  // a cell with __match_any_sync first saved few atomics -- a sweep is sparse -- and cost four MATCH round trips per
  // thread: a quarter of the kernel's stall samples.)
#pragma unroll
  for (int k = 0; k < kVcPer; ++k)
    if (gcell[k] >= 0) red_min_l2hint_i32(first + gcell[k], tile0 + k * kVcThreads + (int)threadIdx.x, pol);
}

// Per SAMPLE (blockIdx.y) exclusive scan, in point order, of flag(i) = "i is the first point of its cell" = the voxel
// number of every cell-creating point, which publishes it: first[global cell] = ~vid (the entry held the point's own
// index until then; other points of the cell only test it against THEIR index) and cell_of_vid[b][vid] = global cell
// (vid < max_voxels only).  The sample's number of distinct cells goes to totals[b].  One decoupled
// look-back chain per sample (a single chain over the whole batch is latency-bound on its tile hand-offs).
static __global__ void __launch_bounds__(kScanThreads)
vox_scan_kernel(const int32_t *__restrict__ offsets, const int32_t *__restrict__ point_gcell,
                int32_t *first, int32_t *__restrict__ cell_of_vid,
                int max_voxels, uint32_t *__restrict__ totals, unsigned long long *status, unsigned int *tickets,
                int tiles_per_sample, int l2_hints) {
  __shared__ uint32_t s_warp[kScanThreads / 32];
  const uint64_t pol = (l2_hints & 1) ? l2_policy_evict_last() : l2_policy_evict_normal();
  __shared__ uint32_t s_tile, s_prefix;
  const int b = blockIdx.y;
  const int begin = offsets[b], n = offsets[b + 1] - begin;
  if (n == 0) {
    if (blockIdx.x == 0 && threadIdx.x == 0) totals[b] = 0u;
    return;
  }
  if ((int64_t)blockIdx.x * kScanTile >= n) return;      // tiles beyond this sample
  if (threadIdx.x == 0) s_tile = atomicAdd(tickets + b, 1u);
  __syncthreads();
  const uint32_t tile = s_tile;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned long long *st_b = status + (int64_t)b * tiles_per_sample;
  const int warp_base = (int)tile * kScanTile + warp * 512;
  int gcs[4][4];
  uint4 v[4];
  uint32_t excl[4];
  uint32_t run = 0;
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int idx = warp_base + r * 128 + lane * 4;
#pragma unroll
    for (int k = 0; k < 4; ++k) gcs[r][k] = idx + k < n ? point_gcell[begin + idx + k] : -1;
  }
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int idx = warp_base + r * 128 + lane * 4;
    uint32_t f[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) f[k] = (gcs[r][k] >= 0 && ld_l2hint_i32(first + gcs[r][k], pol) == begin + idx + k) ? 1u : 0u;
    v[r] = make_uint4(f[0], f[1], f[2], f[3]);
    const uint32_t s = f[0] + f[1] + f[2] + f[3];
    uint32_t incl = s;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    excl[r] = run + incl - s;
    run += __shfl_sync(0xffffffffu, incl, 31);
  }
  if (lane == 0) s_warp[warp] = run;
  __syncthreads();
  if (warp == 0) {
    const uint32_t w = lane < kScanThreads / 32 ? s_warp[lane] : 0u;
    uint32_t incl = w;
#pragma unroll
    for (int o = 1; o < kScanThreads / 32; o <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    const uint32_t total = __shfl_sync(0xffffffffu, incl, kScanThreads / 32 - 1);
    if (lane < kScanThreads / 32) s_warp[lane] = incl - w;
    uint32_t exclusive = 0;
    if (tile == 0) {
      if (lane == 0) st_volatile_u64(st_b, kScanPrefix | total);
    } else {
      if (lane == 0) st_volatile_u64(st_b + tile, kScanAggregate | total);
      int64_t look = (int64_t)tile - 1;
      while (true) {
        const int64_t idx = look - lane;
        unsigned long long st;
        do {
          st = idx >= 0 ? ld_volatile_u64(st_b + idx) : kScanPrefix;
        } while (__any_sync(0xffffffffu, (st >> 32) == 0ull));
        const unsigned pm = __ballot_sync(0xffffffffu, (st >> 32) == 2ull);
        const int firstp = pm ? __ffs(pm) - 1 : 32;
        uint32_t contrib = lane <= firstp ? (uint32_t)(st & 0xffffffffull) : 0u;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) contrib += __shfl_xor_sync(0xffffffffu, contrib, o);
        exclusive += contrib;
        if (pm) break;
        look -= 32;
      }
      if (lane == 0) st_volatile_u64(st_b + tile, kScanPrefix | (uint64_t)(exclusive + total));
    }
    if (lane == 0) {
      s_prefix = exclusive;
      if ((int64_t)(tile + 1) * kScanTile >= n) totals[b] = exclusive + total;      // the sample's last tile
    }
  }
  __syncthreads();
  const uint32_t base = s_prefix + s_warp[warp];
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    uint32_t o[4];
    o[0] = base + excl[r];
    o[1] = o[0] + v[r].x;
    o[2] = o[1] + v[r].y;
    o[3] = o[2] + v[r].z;
    const uint32_t fl[4] = {v[r].x, v[r].y, v[r].z, v[r].w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      if (fl[k]) {                                        // a creating point: o[k] is its cell's voxel number
        st_l2hint_i32(first + gcs[r][k], ~(int32_t)o[k], pol);   // (readers compare with their own index: either value differs)
        if (o[k] < (uint32_t)max_voxels) cell_of_vid[(int64_t)b * max_voxels + o[k]] = gcs[r][k];
      }
    }
  }
}

// voxel_base[b] = rows of the samples before b (their voxel counts capped at max_voxels); one warp
__global__ void vox_dense_base_kernel(const uint32_t *__restrict__ totals, int batch, int max_voxels,
                                      int32_t *__restrict__ voxel_base) {
  int run = 0;                                          // (lane 0 keeps the running base; batch is small)
  for (int b0 = 0; b0 < batch; b0 += 32) {
    const int b = b0 + (int)threadIdx.x;
    const int v = b < batch ? min((int)totals[b], max_voxels) : 0;
    int incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, incl, o);
      if ((int)threadIdx.x >= o) incl += t;
    }
    if (b < batch) voxel_base[b] = run + incl - v;
    run += __shfl_sync(0xffffffffu, incl, 31);
  }
  if (threadIdx.x == 0) voxel_base[batch] = run;
}

// Slot lists.  A voxel's row holds words = kVoxIdxBias - index (> 0), padded to a multiple of 4 words (16-byte
// aligned); it ends up holding the max_points SMALLEST point indices of the voxel as an UNSORTED set, whatever the
// interleaving -- vox_finalize_kernel sorts the (at most max_points) words of a row in registers.  Two kernels:
//   C1 vox_claim_kernel   every kept point takes a ticket from its voxel's arrival counter (one atomicAdd, no chain);
//                         tickets below max_points are slots: the word is stored there.  Later arrivals append
//                         (row, word) to an overflow list (one warp-aggregated atomic per warp).  87 % of the voxels
//                         never overflow: for them this is already the result.
//   C2 vox_evict_kernel   one thread per overflow entry (3.6 % of the points of a sweep: near-range cells receive
//                         thousands of points).  The row is full by now; the entry reads it (16-byte L2 loads), finds
//                         the slot holding the LATEST point and, if it is earlier itself, swaps itself in by
//                         compare-and-swap.  Slot words only ever grow, so a successful swap proves the victim still
//                         was the row's minimum at that moment: with max_points earlier points in the row it can never
//                         be part of the result and is dropped.  A failed swap re-reads the row (somebody else made
//                         progress); an entry that finds the row full of earlier points is done after the loads.
// The sorted-insert formulation this replaces carried the displaced word down the row with one dependent atomicMax
// round trip per slot (71 % of that kernel's stall samples: a sample's 196 CTAs run concurrently, so the points of a
// near-range cell arrive in random order and most arrivals shifted half a row).
__device__ __forceinline__ int4 ld_cg_i4(const int *p) {
  int4 v;
  asm volatile("ld.global.cg.v4.s32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
  return v;
}
__host__ __device__ inline int vox_list_stride(int max_points) { return (max_points + 3) & ~3; }

__global__ void __launch_bounds__(256)
vox_claim_kernel(const int32_t *__restrict__ offsets, const int32_t *__restrict__ point_gcell,
                 const int32_t *__restrict__ vid_of_cell, const int32_t *__restrict__ voxel_base, int max_voxels,
                 int max_points, int32_t *__restrict__ lists, uint32_t *__restrict__ arrivals,
                 int2 *__restrict__ overflow, uint32_t *__restrict__ tile_overflow, int tiles_cap, int l2_hints) {
  __shared__ uint32_t s_over;                                     // overflow entries of this tile so far
  const uint64_t pol = (l2_hints & 1) ? l2_policy_evict_last() : l2_policy_evict_normal();
  const uint64_t pol_lists = (l2_hints & 2) ? l2_policy_evict_last() : l2_policy_evict_normal();
  // grid = (samples, tiles): CTAs are dispatched tile-major, so the tiles of a sample take their tickets roughly in point
  // order -- a near-range voxel's slots are then mostly taken by its earliest points already and the late arrivals in
  // its overflow list lose at their first look at the row (no compare-and-swap rounds)
  const int b = blockIdx.x, tile = blockIdx.y;
  const int begin = offsets[b], end = offsets[b + 1];
  const int tile0 = begin + tile * (256 * kVcPer);
  if (tile0 >= end) return;
  const int i0 = tile0 + threadIdx.x;
  if (threadIdx.x == 0) s_over = 0u;
  __syncthreads();
  const int base = voxel_base[b];
  const int LS = vox_list_stride(max_points);
  const int lane = threadIdx.x & 31;
  int gc[kVcPer], row[kVcPer];
  uint32_t pos[kVcPer];
#pragma unroll
  for (int k = 0; k < kVcPer; ++k) gc[k] = i0 + 256 * k < end ? point_gcell[i0 + 256 * k] : -1;
#pragma unroll
  for (int k = 0; k < kVcPer; ++k) {
    const int vid = gc[k] >= 0 ? ~ld_l2hint_i32(vid_of_cell + gc[k], pol) : max_voxels;
    row[k] = vid < max_voxels ? base + vid : -1;                 // (voxel cap: the whole cell is dropped)
  }
#pragma unroll
  for (int k = 0; k < kVcPer; ++k) pos[k] = row[k] >= 0 ? atom_add_l2hint_u32(arrivals + row[k], 1u, pol_lists) : 0u;
  // Late arrivals go to the TILE's segment of the overflow list (the tile's own points bound its length): positions come
  // from a shared-memory counter.  One global counter for the whole batch -- the first version -- made every second warp
  // wait for the return value of an atomic on a single address (75 % of this kernel's stall samples).
#pragma unroll
  for (int k = 0; k < kVcPer; ++k) {
    const int w = kVoxIdxBias - (i0 + 256 * k);
    const bool over = row[k] >= 0 && pos[k] >= (uint32_t)max_points;
    if (row[k] >= 0 && !over) st_l2hint_i32(lists + (int64_t)row[k] * LS + pos[k], w, pol_lists);
    const unsigned bal = __ballot_sync(0xffffffffu, over);
    if (bal) {
      uint32_t at = 0;
      if (lane == __ffs(bal) - 1) at = atomicAdd(&s_over, (uint32_t)__popc(bal));
      at = __shfl_sync(0xffffffffu, at, __ffs(bal) - 1);
      if (over) overflow[(int64_t)tile0 + at + __popc(bal & ((1u << lane) - 1u))] = make_int2(row[k], w);
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) tile_overflow[(int64_t)b * tiles_cap + tile] = s_over;
}

// word of slot t of a row held as LQ quads (t a compile-time constant after unrolling)
template <int LQ>
__device__ __forceinline__ int vox_quad_word(const int4 (&q)[LQ], int t) {
  const int4 qq = q[t >> 2];
  return (t & 3) == 0 ? qq.x : (t & 3) == 1 ? qq.y : (t & 3) == 2 ? qq.z : qq.w;
}

template <int LQ>                                        // row = 4 * LQ words (max_points <= 16); LQ = 0: any length
__global__ void __launch_bounds__(128)
vox_evict_kernel(const int32_t *__restrict__ offsets, const int2 *__restrict__ overflow_all,
                 const uint32_t *__restrict__ tile_overflow, int tiles_cap, int max_points, int32_t *__restrict__ lists) {
  // one CTA per tile of the claim kernel: its overflow entries sit at the tile's first point index
  const int b = blockIdx.x, tile = blockIdx.y;              // (tile-major like the claim kernel: the earliest candidates first)
  const int begin = offsets[b], end = offsets[b + 1];
  const int tile0 = begin + tile * (256 * kVcPer);
  if (tile0 >= end) return;
  const uint32_t n = tile_overflow[(int64_t)b * tiles_cap + tile];
  const int2 *overflow = overflow_all + tile0;
  const int LS = vox_list_stride(max_points);
  for (uint32_t e = threadIdx.x; e < n; e += blockDim.x) {
    const int2 ent = overflow[e];
    int *row = lists + (int64_t)ent.x * LS;
    int w = ent.y;
    if constexpr (LQ > 0) {
      // The victim is the slot holding the LATEST point (then the displaced point is later than the 14 others and the
      // new one: dropped at once).  On a near-range row hundreds of entries race for that one slot and every swap sends
      // all the others back to re-read the row: the rounds, not the work, were this kernel's time.  An entry that lost
      // a race therefore picks a pseudo-random slot among those holding later points and CARRIES the point it displaces
      // (which may still belong to the result) as its new candidate.  Invariant: row + candidates in flight contain the
      // max_points earliest points; slot words only grow, so a candidate that finds every slot earlier than itself can
      // never enter and is dropped.  Every swap raises the sum of the row's words: the loop ends.
      bool spread = false;
      uint32_t rnd = ((uint32_t)tile0 + e) * 2654435761u + 12345u;
      while (true) {
        int4 q[LQ];
#pragma unroll
        for (int j = 0; j < LQ; ++j) q[j] = ld_cg_i4(row + 4 * j);
        int mw = 0x7fffffff, ms = 0, later = 0;
#pragma unroll
        for (int t = 0; t < 4 * LQ; ++t) {
          const int ww = vox_quad_word<LQ>(q, t);
          if (t < max_points) {
            later += ww < w;
            if (ww < mw) { mw = ww; ms = t; }
          }
        }
        if (later == 0) break;                              // the row is full of earlier points
        bool is_min = true;
        if (spread && later > 1) {
          rnd = rnd * 1664525u + 1013904223u;
          const int pick = (int)((rnd >> 16) % (uint32_t)later);
          const int min_slot = ms;
          int seen = 0;
#pragma unroll
          for (int t = 0; t < 4 * LQ; ++t) {
            const int ww = vox_quad_word<LQ>(q, t);
            if (t < max_points && ww < w) {
              if (seen == pick) { mw = ww; ms = t; }
              ++seen;
            }
          }
          is_min = ms == min_slot;
        }
        if (atomicCAS(row + ms, mw, w) == mw) {
          if (is_min) break;                                // (others only grew since the read: it still was the minimum)
          w = mw;                                           // carry the displaced point
        } else {
          spread = true;
        }
      }
    } else {
      while (true) {
        int mw = 0x7fffffff, ms = 0;
        for (int t4 = 0; t4 < LS; t4 += 4) {
          const int4 qq = ld_cg_i4(row + t4);
          const int ww[4] = {qq.x, qq.y, qq.z, qq.w};
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (t4 + j < max_points && ww[j] < mw) { mw = ww[j]; ms = t4 + j; }
        }
        if (w < mw) break;                                  // the row is full of earlier points
        if (atomicCAS(row + ms, mw, w) == mw) break;
      }
    }
  }
}

// Batcher's merge-exchange network on 16 registers (63 compare-exchanges, every index a compile-time constant)
__device__ __forceinline__ void vox_sort16_desc(int (&w)[16]) {
#pragma unroll
  for (int p = 1; p < 16; p <<= 1) {
#pragma unroll
    for (int k = p; k >= 1; k >>= 1) {
#pragma unroll
      for (int j = k % p; j <= 16 - 1 - k; j += 2 * k) {
#pragma unroll
        for (int i = 0; i < k; ++i) {
          if (i <= 16 - j - k - 1 && (i + j) / (p * 2) == (i + j + k) / (p * 2)) {
            const int a = w[i + j], c = w[i + j + k];
            w[i + j] = max(a, c);
            w[i + j + k] = min(a, c);
          }
        }
      }
    }
  }
}

// One LANE per row of the padded output (batch * max_voxels rows), one warp per 32 consecutive rows.  A live row finds its
// sample (binary search in voxel_base) and its coordinates (cell_of_vid) and walks its slot list: index word -> point
// row, gathered into the warp's shared-memory tile [32 rows][max_points * F] (zero-initialised: the padding);
// running sums for the HardSimpleVFE mean in slot order, count = number of filled slots.  The tile then leaves as ONE
// contiguous span of 32 * max_points * F floats written with 16-byte stores -- every element of `voxels` is written
// exactly once, coalesced (no memset of the 93 %-padding tensor, no 20-byte scattered stores).  Rows beyond the voxel
// count are written as zeros (voxels, num_points, coors, mean).
constexpr int kFinWarps = 4;
template <int FM>                                       // FM >= F: bound of the per-point register arrays (8 or 16)
__global__ void __launch_bounds__(kFinWarps * 32)
vox_finalize_kernel(VoxPoints pts, const int32_t *__restrict__ offsets, int F, VoxGeom g, int64_t cells,
                    const int32_t *__restrict__ cell_of_vid, int32_t *__restrict__ lists, const uint32_t *__restrict__ arrivals,
                    int batch, int max_voxels, int max_points, float *__restrict__ voxels, int32_t *__restrict__ num_points, int32_t *__restrict__ coors,
                    const int32_t *__restrict__ voxel_base, float *__restrict__ voxel_mean, int mean_features,
                    float *__restrict__ canvas) {
  extern __shared__ __align__(16) float s_fin[];          // [kFinWarps][32][TF] floats, then voxel_base (batch + 1 ints)
  const int TF = max_points * F;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float *tile = s_fin + (size_t)warp * 32 * TF;
  int *s_vb = reinterpret_cast<int *>(s_fin + (size_t)kFinWarps * 32 * TF);
  for (int k = threadIdx.x; k <= batch; k += blockDim.x) s_vb[k] = voxel_base[k];
  for (int e = lane; e < 32 * TF / 4; e += 32) reinterpret_cast<float4 *>(tile)[e] = make_float4(0.f, 0.f, 0.f, 0.f);
  __syncthreads();
  const int64_t total_rows = (int64_t)batch * max_voxels;
  const int64_t row0 = ((int64_t)blockIdx.x * kFinWarps + warp) * 32;
  if (row0 >= total_rows) return;
  const int64_t row = row0 + lane;
  if (row < total_rows) {
    int cnt = 0;
    if (row < s_vb[batch]) {
      int lo = 0, hi = batch;                             // sample b: s_vb[b] <= row < s_vb[b + 1]
      while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (s_vb[mid] <= row) lo = mid; else hi = mid;
      }
      const int b = lo;
      const int begin = offsets[b];
      const int LS = vox_list_stride(max_points);
      int32_t *list = lists + row * LS;
      // the row's slot words first (16-byte loads of the padded row: one round trip), then its points four at a time
      int words[16];
#pragma unroll
      for (int t4 = 0; t4 < 4; ++t4) {
        int4 w4 = make_int4(0, 0, 0, 0);
        if (4 * t4 < LS) w4 = reinterpret_cast<const int4 *>(list)[t4];               // (padding words are 0)
        words[4 * t4 + 0] = w4.x; words[4 * t4 + 1] = w4.y; words[4 * t4 + 2] = w4.z; words[4 * t4 + 3] = w4.w;
      }
      // the claim kernels leave an unsorted set in the first `filled` slots (the rest was never written):
      // descending words = ascending point index, empty slots (0) last
      const int filled = (int)min(arrivals[row], (uint32_t)max_points);
#pragma unroll
      for (int t = 0; t < 16; ++t) words[t] = t < filled ? words[t] : 0;
      if (max_points <= 16) {
        vox_sort16_desc(words);
      } else {                                             // long rows: insertion sort in place (this lane owns the row)
        for (int t = 1; t < filled; ++t) {
          const int w = list[t];
          int u = t - 1;
          while (u >= 0 && list[u] < w) { list[u + 1] = list[u]; --u; }
          list[u + 1] = w;
        }
#pragma unroll
        for (int t = 0; t < 16; ++t) words[t] = t < filled ? list[t] : 0;
      }
      const int gc = cell_of_vid[(int64_t)b * max_voxels + (row - s_vb[b])];
      const int64_t c = (int64_t)gc - (int64_t)b * cells;
      const int x = (int)(c % g.gx), y = (int)((c / g.gx) % g.gy), z = (int)(c / ((int64_t)g.gx * g.gy));
      reinterpret_cast<int4 *>(coors)[row] = make_int4(b, z, y, x);
      float *trow = tile + (size_t)lane * TF;
      float sum[FM];
#pragma unroll
      for (int k = 0; k < FM; ++k) sum[k] = 0.f;
      auto word_at = [&](int t) { return t < 16 ? words[t & 15] : (t < filled ? list[t] : 0); };
      for (int t0 = 0; t0 < max_points; t0 += 4) {
        int wq[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          int w = 0;
          if (t0 + j < 16) {
#pragma unroll
            for (int q = 0; q < 16; ++q) w = (q == t0 + j) ? words[q] : w;      // (register array: no dynamic indexing)
          } else {
            w = word_at(t0 + j);
          }
          wq[j] = w;
        }
        if (wq[0] == 0) break;                             // filled slots are a prefix
        float val[4][FM];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float *src = pts.row(b, begin, kVoxIdxBias - (wq[j] ? wq[j] : wq[0]), F);
#pragma unroll
          for (int k = 0; k < FM; ++k)
            if (k < F) val[j][k] = __ldg(src + k);
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          if (wq[j] == 0) break;
          float *dst = trow + cnt * F;
          ++cnt;
#pragma unroll
          for (int k = 0; k < FM; ++k) {
            if (k < F) dst[k] = val[j][k];
            if (k < mean_features) sum[k] += val[j][k];
          }
        }
      }
      if (voxel_mean || canvas) {
#pragma unroll
        for (int k = 0; k < FM; ++k) {
          if (k >= mean_features) break;
          const float m = sum[k] / (float)cnt;
          if (voxel_mean) voxel_mean[row * mean_features + k] = m;
          if (canvas) canvas[((((int64_t)b * mean_features + k) * g.gz + z) * g.gy + y) * g.gx + x] = m;
        }
      }
    } else {                                               // padding row: zero coordinates and mean
      reinterpret_cast<int4 *>(coors)[row] = make_int4(0, 0, 0, 0);
      if (voxel_mean)
        for (int k = 0; k < mean_features; ++k) voxel_mean[row * mean_features + k] = 0.f;
    }
    num_points[row] = cnt;
  }
  __syncwarp();
  // the warp's 32 rows are one contiguous span of the output
  const int64_t nrows = min((int64_t)32, total_rows - row0);
  float *out = voxels + row0 * TF;
  const int n4 = (int)(nrows * TF / 4);                    // row0 * TF * 4 bytes is a multiple of 16 (row0 % 32 == 0)
  for (int e = lane; e < n4; e += 32) stg_stream_f4(reinterpret_cast<float4 *>(out) + e, reinterpret_cast<const float4 *>(tile)[e]);
  for (int e = n4 * 4 + lane; e < nrows * TF; e += 32) out[e] = tile[e];
}

// Rows of at most 16 slots (every pillar / voxel configuration of the reference): same output as vox_finalize_kernel, but
// the point gather is shared by the warp.  With one lane walking its own row the warp runs as long as its fullest row
// (13 % of the rows of a long-range sweep are full: practically every warp went through all four rounds of four slots)
// while the mean row holds 1.7 points.  Here a lane reads, masks and sorts its row's words; the warp lists its (row, slot)
// pairs behind an exclusive scan of the counts and lane p fetches pair p -- every point row of the 32 voxels is in flight
// within two rounds for a typical warp.  The mean is summed by the row's lane from the shared-memory tile in slot order
// (bit-identical to the serial sum).
// The tile holds 16 rows: the warp's 32 rows leave in two passes (gather, mean, write-out per half) -- 8 KB of shared
// memory per warp instead of 13 KB at the pillar shape, 28 resident warps per SM instead of 16 (the kernel is bound by
// instruction issue and latency, not by DRAM).
constexpr int kFinTileRows = 16;
__host__ __device__ inline size_t vox_fin_coop_warp_bytes(int max_points, int F) {   // tile + words + pair map + row sources
  return (size_t)kFinTileRows * 4 * max_points * F + 2048 + 1024 + 256;
}
template <int FM>
__global__ void __launch_bounds__(kFinWarps * 32, FM <= 8 ? 5 : 3)
vox_finalize_coop_kernel(VoxPoints pts, const int32_t *__restrict__ offsets, int F, VoxGeom g, int64_t cells,
                         const int32_t *__restrict__ cell_of_vid, const int32_t *__restrict__ lists,
                         const uint32_t *__restrict__ arrivals, int batch, int max_voxels, int max_points,
                         float *__restrict__ voxels, int32_t *__restrict__ num_points, int32_t *__restrict__ coors,
                         const int32_t *__restrict__ voxel_base, float *__restrict__ voxel_mean, int mean_features,
                         float *__restrict__ canvas) {
  extern __shared__ __align__(128) unsigned char s_finc[];
  const int TF = max_points * F;
  const size_t warp_bytes = vox_fin_coop_warp_bytes(max_points, F);
  const size_t tile_bytes = (size_t)kFinTileRows * 4 * TF;                              // (a multiple of 64)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned char *wb = s_finc + (size_t)warp * warp_bytes;
  float *tile = reinterpret_cast<float *>(wb);                                          // [16][TF]
  int *s_words = reinterpret_cast<int *>(wb + tile_bytes);                              // [32][16] sorted slot words
  uint16_t *s_map = reinterpret_cast<uint16_t *>(wb + tile_bytes + 2048);               // pair p -> row * 16 + slot
  const float **s_src = reinterpret_cast<const float **>(wb + tile_bytes + 3072);       // row -> point 0 of its cloud
  int *s_vb = reinterpret_cast<int *>(s_finc + (size_t)kFinWarps * warp_bytes);
  for (int k = threadIdx.x; k <= batch; k += blockDim.x) s_vb[k] = voxel_base[k];
  __syncthreads();
  const int64_t total_rows = (int64_t)batch * max_voxels;
  const int64_t row0 = ((int64_t)blockIdx.x * kFinWarps + warp) * 32;
  if (row0 >= total_rows) return;
  const int64_t row = row0 + lane;
  const bool live = row < total_rows && row < s_vb[batch];
  const int64_t lrow = live ? row : 0;                       // (dead lanes read row 0: no divergence around the sort)
  int lo = 0, hi = batch;                                    // sample b: s_vb[b] <= row < s_vb[b + 1]
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (s_vb[mid] <= lrow) lo = mid; else hi = mid;
  }
  const int b = lo;
  const int LS = vox_list_stride(max_points);
  const int4 *list = reinterpret_cast<const int4 *>(lists + lrow * LS);
  const int cnt = live ? (int)min(arrivals[lrow], (uint32_t)max_points) : 0;
  const int gc = cell_of_vid[(int64_t)b * max_voxels + (lrow - s_vb[b])];
  const int begin = offsets[b];
  int4 q[4];
#pragma unroll
  for (int t4 = 0; t4 < 4; ++t4) {
    q[t4] = make_int4(0, 0, 0, 0);
    if (4 * t4 < cnt) q[t4] = ldg_stream_i4(list + t4);     // (last use of the row; cnt <= max_points <= LS)
  }
  int words[16];
#pragma unroll
  for (int t4 = 0; t4 < 4; ++t4) {
    words[4 * t4 + 0] = 4 * t4 + 0 < cnt ? q[t4].x : 0;
    words[4 * t4 + 1] = 4 * t4 + 1 < cnt ? q[t4].y : 0;
    words[4 * t4 + 2] = 4 * t4 + 2 < cnt ? q[t4].z : 0;
    words[4 * t4 + 3] = 4 * t4 + 3 < cnt ? q[t4].w : 0;
  }
  // the claim kernels leave an unsorted set in the first `cnt` slots: descending words = ascending point index
  vox_sort16_desc(words);
  int x = 0, y = 0, z = 0;
  if (live) {
    const uint32_t c = (uint32_t)((int64_t)gc - (int64_t)b * cells);      // (dense mode: a sample has < 2^26 cells)
    const uint32_t cy = c / (uint32_t)g.gx;
    x = (int)(c - cy * (uint32_t)g.gx);
    z = (int)(cy / (uint32_t)g.gy);
    y = (int)(cy - (uint32_t)z * (uint32_t)g.gy);
    reinterpret_cast<int4 *>(coors)[row] = make_int4(b, z, y, x);
  } else if (row < total_rows) {
    reinterpret_cast<int4 *>(coors)[row] = make_int4(0, 0, 0, 0);        // padding row (its mean: below)
  }
  if (row < total_rows) num_points[row] = cnt;
  s_src[lane] = pts.per_sample ? pts.per_sample[b] - (int64_t)begin * F : pts.cat;
  int incl = cnt;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  const int total = __shfl_sync(0xffffffffu, incl, 31), off = incl - cnt;
  const int split = __shfl_sync(0xffffffffu, off, kFinTileRows);           // pairs of rows 0..15 come first
#pragma unroll
  for (int t4 = 0; t4 < 4; ++t4)
    *reinterpret_cast<int4 *>(s_words + lane * 16 + 4 * t4) = make_int4(words[4 * t4], words[4 * t4 + 1], words[4 * t4 + 2], words[4 * t4 + 3]);
#pragma unroll
  for (int t = 0; t < 16; ++t)
    if (t < cnt) s_map[off + t] = (uint16_t)(lane * 16 + t);
  // canvas coordinates of the other half-warp's rows are needed by the lanes that share their mean work (below)
  const int64_t canvas_cell = (((int64_t)b * mean_features * g.gz + z) * g.gy + y) * g.gx + x;   // channel 0 of the row's cell
  const int64_t canvas_plane = (int64_t)g.gz * g.gy * g.gx;
#pragma unroll 1
  for (int half = 0; half < 2; ++half) {
    const int64_t hrow0 = row0 + half * kFinTileRows;
    if (hrow0 >= total_rows) break;
    for (int e = lane; e < kFinTileRows * TF / 4; e += 32) reinterpret_cast<float4 *>(tile)[e] = make_float4(0.f, 0.f, 0.f, 0.f);
    __syncwarp();
    const int pbeg = half ? split : 0, pend = half ? total : split;
    for (int p0 = pbeg; p0 < pend; p0 += 64) {                // two point rows per lane in flight
      float val[2][FM];
      int dst[2];
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const int p = p0 + 32 * j + lane;
        dst[j] = -1;
        if (p < pend) {
          const int m = s_map[p], r = m >> 4;
          const float *src = s_src[r] + (int64_t)(kVoxIdxBias - s_words[m]) * F;
#pragma unroll
          for (int k = 0; k < FM; ++k)
            if (k < F) val[j][k] = __ldg(src + k);
          dst[j] = (r & (kFinTileRows - 1)) * TF + (m & 15) * F;
        }
      }
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        if (dst[j] >= 0) {
#pragma unroll
          for (int k = 0; k < FM; ++k)
            if (k < F) tile[dst[j] + k] = val[j][k];
        }
      }
    }
    __syncwarp();
    if (voxel_mean || canvas) {
      // HardSimpleVFE mean of the half's 16 rows, summed in slot order from the tile.  Both half-warps work: lane l and
      // lane l + 16 share row (l & 15) of the half, the first takes the even features, the second the odd ones.
      const int rl = lane & (kFinTileRows - 1), owner = half * kFinTileRows + rl, par = lane >> 4;
      const int rcnt = __shfl_sync(0xffffffffu, cnt, owner);
      const int64_t rcell = __shfl_sync(0xffffffffu, canvas_cell, owner);
      if (rcnt > 0) {
        float sum[(FM + 1) / 2];
#pragma unroll
        for (int k = 0; k < (FM + 1) / 2; ++k) sum[k] = 0.f;
        const float *trow = tile + (size_t)rl * TF + par;
        for (int t = 0; t < rcnt; ++t) {
#pragma unroll
          for (int k = 0; k < (FM + 1) / 2; ++k)
            if (2 * k + par < mean_features) sum[k] += trow[t * F + 2 * k];
        }
        const int64_t orow = hrow0 + rl;
#pragma unroll
        for (int k = 0; k < (FM + 1) / 2; ++k) {
          const int f = 2 * k + par;
          if (f >= mean_features) break;
          const float m = sum[k] / (float)rcnt;
          if (voxel_mean) voxel_mean[orow * mean_features + f] = m;
          if (canvas) canvas[rcell + (int64_t)f * canvas_plane] = m;
        }
      } else if (voxel_mean && hrow0 + rl < total_rows) {   // padding row (live rows hold at least one point)
        for (int f = par; f < mean_features; f += 2) voxel_mean[(hrow0 + rl) * mean_features + f] = 0.f;
      }
    }
    // the half's 16 rows are one contiguous span of the output
    const int64_t nrows = min((int64_t)kFinTileRows, total_rows - hrow0);
    float *out = voxels + hrow0 * TF;
    const int n4 = (int)(nrows * TF / 4);                    // hrow0 * TF * 4 bytes is a multiple of 16 (hrow0 % 16 == 0)
    for (int e = lane; e < n4; e += 32) stg_stream_f4(reinterpret_cast<float4 *>(out) + e, reinterpret_cast<const float4 *>(tile)[e]);
    for (int e = n4 * 4 + lane; e < nrows * TF; e += 32) out[e] = tile[e];
    __syncwarp();
  }
}

// Dense canvas of the fused HardSimpleVFE mean, written ONCE and in order: a thread owns 4 consecutive cells, reads their
// entries of the voxel-number table (16 bytes), fetches the mean row of the occupied ones (5 % of the cells of a
// long-range sweep) and writes mean_features coalesced 16-byte streaming stores.  This replaces a DRAM-speed zero fill of
// the canvas plus mean_features scattered 4-byte stores per voxel from the finalize kernel -- each of those a
// read-modify-write of a 32-byte sector at a random address, 40 % of that kernel's sector traffic -- by one sequential
// read of the table.
template <int FM>
__global__ void __launch_bounds__(256)
vox_canvas_dense_kernel(const int32_t *__restrict__ vid_of_cell, const int32_t *__restrict__ voxel_base,
                        const float *__restrict__ voxel_mean, int mean_features, int max_voxels, int64_t cells,
                        float *__restrict__ canvas) {
  const int b = blockIdx.y;
  const int64_t c4 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (c4 >= cells) return;
  const int4 e4 = ldg_stream_i4(reinterpret_cast<const int4 *>(vid_of_cell + (int64_t)b * cells + c4));
  const int e[4] = {e4.x, e4.y, e4.z, e4.w};
  const int base = voxel_base[b];
  float m[4][FM];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int vid = e[j] < 0 ? ~e[j] : max_voxels;           // (empty cells hold 0x7f7f7f7f; cells beyond the cap are dropped)
    const bool ok = vid < max_voxels;
    const float *src = voxel_mean + (int64_t)(base + (ok ? vid : 0)) * mean_features;
#pragma unroll
    for (int k = 0; k < FM; ++k) m[j][k] = (ok && k < mean_features) ? __ldg(src + k) : 0.f;
  }
#pragma unroll
  for (int k = 0; k < FM; ++k) {
    if (k >= mean_features) break;
    stg_stream_f4(reinterpret_cast<float4 *>(canvas + ((int64_t)b * mean_features + k) * cells + c4),
                  make_float4(m[0][k], m[1][k], m[2][k], m[3][k]));
  }
}

// pillar scatter for UNIQUE coordinates (what hard voxelization produces): canvas pre-zeroed, one thread per element
template <typename T>
__global__ void scatter_unique_kernel(const T *__restrict__ feats, const int32_t *__restrict__ coors, int64_t M, int C,
                                      int batch, int nz, int ny, int nx, T *__restrict__ canvas) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= M * C) return;
  const int64_t m = e / C;
  const int c = (int)(e - m * C);
  const int4 co = reinterpret_cast<const int4 *>(coors)[m];
  if (co.x < 0 || co.x >= batch || co.y < 0 || co.y >= nz || co.z < 0 || co.z >= ny || co.w < 0 || co.w >= nx) return;
  canvas[((((int64_t)co.x * C + c) * nz + co.y) * ny + co.z) * nx + co.w] = feats[e];
}

struct VoxTemp {
  size_t off_scan, off_counts, zero_bytes;   // [0, zero_bytes) memset 0
  size_t off_keys;                           // memset 0xff
  size_t off_first, off_lists, fill7f_bytes; // [off_first, off_first + fill7f_bytes) memset 0x7f
  size_t off_slot, off_flags, bytes;
  uint32_t hash_slots;
};

static VoxTemp vox_temp_layout(int batch, int64_t total_points, int max_voxels, int max_points) {
  VoxTemp L{};
  uint32_t h = 1024;
  while ((double)h < 1.25 * (double)total_points) h <<= 1;
  L.hash_slots = h;
  const size_t rows = (size_t)batch * max_voxels;
  size_t o = 0;
  L.off_scan = o;   o += scan_workspace_bytes(total_points + 1);
  L.off_counts = o; o = align_up(o + rows * 4, 256);
  L.zero_bytes = o;
  L.off_keys = o;   o = align_up(o + (size_t)h * 8, 256);
  L.off_first = o;  o = align_up(o + (size_t)h * 4, 256);
  L.off_lists = o;  o = align_up(o + rows * max_points * 4, 256);
  L.fill7f_bytes = o - L.off_first;
  L.off_slot = o;   o = align_up(o + (size_t)total_points * 4, 256);
  L.off_flags = o;  o = align_up(o + (size_t)(total_points + 1) * 4, 256);
  L.bytes = o;
  return L;
}

// dense mode: first-point table + voxel-number table over all cells of the batch (int32 each), point -> global cell ids
struct VoxDenseTemp {
  size_t off_status, off_tickets, off_arrivals, zero_bytes;   // [0, zero_bytes) memset 0 (scan status words, tickets, arrival counters)
  size_t off_tile_overflow;                     // per (sample, claim tile) overflow counts (written by every live tile)
  int tiles_cap;
  size_t off_lists, off_overflow;
  size_t off_first, first_bytes;                // memset 0x7f
  size_t off_gcell, off_cell_of_vid, off_totals, bytes;
  int tiles_per_sample;
};
constexpr int64_t kVoxDenseMaxCells = 1ll << 26;          // cells of the whole batch (2 x 256 MB of tables); larger grids hash
static bool vox_dense_ok(int batch, const int *grid) {
  const int64_t cells = (int64_t)grid[0] * grid[1] * grid[2];
  const char *e = std::getenv("BEVVOX_FORCE_HASH");          // tests: exercise the hash path on small grids
  const bool forced_hash = e && e[0] == '1';
  return !forced_hash && cells > 0 && (int64_t)batch * cells <= kVoxDenseMaxCells;
}
static VoxDenseTemp vox_dense_layout(int batch, int64_t total_points, int max_voxels, int max_points, const int *grid) {
  VoxDenseTemp L{};
  const size_t cells = (size_t)grid[0] * grid[1] * grid[2];
  L.tiles_per_sample = (int)scan_num_tiles(total_points > 0 ? total_points : 1);    // (the largest sample is bounded by the total)
  size_t o = 0;
  L.off_status = o;  o = align_up(o + (size_t)batch * L.tiles_per_sample * 8, 256);
  L.off_tickets = o; o = align_up(o + (size_t)batch * 4, 256);
  L.off_arrivals = o; o = align_up(o + (size_t)batch * max_voxels * 4, 256);
  L.zero_bytes = o;
  L.tiles_cap = (int)ceil_div64(total_points > 0 ? total_points : 1, kVcThreads * kVcPer);   // (bounds every sample's tile count)
  L.off_tile_overflow = o; o = align_up(o + (size_t)batch * L.tiles_cap * 4, 256);
  L.off_lists = o;   o = align_up(o + (size_t)batch * max_voxels * vox_list_stride(max_points) * 4, 256);   // (never read beyond a row's arrival count)
  L.off_overflow = o; o = align_up(o + (size_t)total_points * 8, 256);
  L.off_first = o;  L.first_bytes = align_up((size_t)batch * cells * 4, 256); o += L.first_bytes;
  L.off_gcell = o;  o = align_up(o + (size_t)total_points * 4, 256);
  L.off_cell_of_vid = o; o = align_up(o + (size_t)batch * max_voxels * 4, 256);
  L.off_totals = o; o = align_up(o + (size_t)batch * 4, 256);
  L.bytes = o > 256 ? o : 256;
  return L;
}

static int check_vox_args(int batch, int64_t total_points, int F, int max_voxels, int max_points) {
  if (batch <= 0 || batch > 65535 || total_points < 0 || F < 3 || F > kVoxMaxF || max_voxels <= 0 || max_points <= 0) return BEVPOOL_E_ARG;
  if (total_points >= 0x7f7f7f7f || (int64_t)batch * max_voxels * (max_points + 3) >= INT32_MAX) return BEVPOOL_E_RANGE;
  return BEVPOOL_OK;
}

static VoxGeom make_geom(const float *vs, const float *range, const int *grid) {
  VoxGeom g;
  g.vx = vs[0]; g.vy = vs[1]; g.vz = vs[2];
  g.xmin = range[0]; g.ymin = range[1]; g.zmin = range[2];
  g.gx = grid[0]; g.gy = grid[1]; g.gz = grid[2];
  g.ivx = 1.0f / g.vx; g.ivy = 1.0f / g.vy; g.ivz = 1.0f / g.vz;
  return g;
}

}  // namespace bevpool

using namespace bevpool;

extern "C" int bevvox_temp_bytes(int batch, int64_t total_points, const int *grid_host, int max_voxels, int max_points,
                                 size_t *temp_bytes) {
  int rc = check_vox_args(batch, total_points, 3, max_voxels, max_points);
  if (rc) return rc;
  if (!temp_bytes || !grid_host) return BEVPOOL_E_ARG;
  *temp_bytes = vox_dense_ok(batch, grid_host) ? vox_dense_layout(batch, total_points, max_voxels, max_points, grid_host).bytes
                                               : vox_temp_layout(batch, total_points, max_voxels, max_points).bytes;
  return BEVPOOL_OK;
}

// bit 0: first-point / voxel-number table evict_last, bit 1: slot lists + arrival counters evict_last, bit 2: point stream
// evict_first (BEVVOX_L2_HINTS, read once; default below)
static int vox_l2_hints() {
  static const int v = [] {
    const char *e = std::getenv("BEVVOX_L2_HINTS");
    return e && e[0] ? std::atoi(e) : 5;
  }();
  return v;
}
static bool vox_overlap_enabled() {
  static const bool on = [] {
    const char *e = std::getenv("BEVVOX_CANVAS_OVERLAP");
    return !(e && e[0] == '0');
  }();
  return on;
}
// one non-blocking side stream per device, created on first use (host object only: no device memory)
static cudaStream_t vox_side_stream() {
  static cudaStream_t streams[64] = {nullptr};
  static std::atomic<int> lock{0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
  if (!streams[dev]) {
    while (lock.exchange(1)) {}
    if (!streams[dev]) {
      cudaStream_t s = nullptr;
      if (cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking) == cudaSuccess) streams[dev] = s;
    }
    lock.store(0);
  }
  return streams[dev];
}

static int hard_voxelize_dense(VoxPoints pts, const int32_t *sample_offsets, int batch, int64_t total_points,
                               int64_t max_sample_points, int F, const VoxGeom &g, const int *grid, int max_points,
                               int max_voxels, float *voxels, int32_t *coors, int32_t *num_points, int32_t *voxel_base,
                               float *voxel_mean, int mean_features, float *canvas, void *temp, cudaStream_t stream,
                               bool fill_canvas) {
  const VoxDenseTemp L = vox_dense_layout(batch, total_points, max_voxels, max_points, grid);
  int32_t *lists = reinterpret_cast<int32_t *>(static_cast<char *>(temp) + L.off_lists);
  const int tps = (int)scan_num_tiles(max_sample_points > 0 ? max_sample_points : 1);   // <= L.tiles_per_sample
  char *tb = static_cast<char *>(temp);
  int32_t *first = reinterpret_cast<int32_t *>(tb + L.off_first);
  const int32_t *vid_of_cell = first;                   // after the scan: ~(voxel number of the cell)
  int32_t *gcell = reinterpret_cast<int32_t *>(tb + L.off_gcell);
  int32_t *cell_of_vid = reinterpret_cast<int32_t *>(tb + L.off_cell_of_vid);
  uint32_t *totals = reinterpret_cast<uint32_t *>(tb + L.off_totals);
  const int64_t cells = (int64_t)grid[0] * grid[1] * grid[2];
  const size_t rows = (size_t)batch * max_voxels;
  // The canvas fill (335 MB per 32 sweeps of pure DRAM-write work) does not depend on anything the first four kernels do,
  // and those are latency bound: it runs on a side stream (fork here, join before the kernel that scatters into it).
  // Event fork / join is legal under stream capture; the side stream is created once per device.
  // With a mean output to read from (and 16-byte aligned cell rows) the canvas is written densely by its own kernel after
  // the finalize kernel; otherwise it is zero-filled here, on the side stream, and the finalize kernel scatters into it.
  const bool dense_canvas = canvas && fill_canvas && voxel_mean && mean_features > 0 && (cells & 3) == 0 &&
                            ((reinterpret_cast<uintptr_t>(canvas) | reinterpret_cast<uintptr_t>(first)) & 15u) == 0;
  cudaEvent_t ev_join = nullptr;
  if (canvas && fill_canvas && !dense_canvas) {
    const size_t cbytes = (size_t)batch * mean_features * g.gx * g.gy * g.gz * sizeof(float);
    cudaStream_t side = vox_overlap_enabled() ? vox_side_stream() : nullptr;
    if (side) {
      cudaEvent_t ev_fork = nullptr;
      BEVPOOL_RETURN_IF_CUDA(cudaEventCreateWithFlags(&ev_fork, cudaEventDisableTiming));
      BEVPOOL_RETURN_IF_CUDA(cudaEventCreateWithFlags(&ev_join, cudaEventDisableTiming));
      BEVPOOL_RETURN_IF_CUDA(cudaEventRecord(ev_fork, stream));
      BEVPOOL_RETURN_IF_CUDA(cudaStreamWaitEvent(side, ev_fork, 0));
      BEVPOOL_RETURN_IF_CUDA(cudaMemsetAsync(canvas, 0, cbytes, side));
      BEVPOOL_RETURN_IF_CUDA(cudaEventRecord(ev_join, side));
      cudaEventDestroy(ev_fork);                            // (released once the recorded work has completed)
    } else {
      BEVPOOL_RETURN_IF_CUDA(cudaMemsetAsync(canvas, 0, cbytes, stream));
    }
  }
  BEVPOOL_RETURN_IF_CUDA(cudaMemsetAsync(tb, 0, L.zero_bytes, stream));
  // (Tried: running fill -> cell -> scan -> base -> claim per group of 8 or 16 samples so that a group's 2 MB-per-sample
  // first-point table stays in L2 between the three kernels that visit it at random -- no gain at 16, slower at 8: the
  // extra launches and tails cost more than the L2 hits return.)
  uint32_t *arrivals = reinterpret_cast<uint32_t *>(tb + L.off_arrivals);
  int2 *overflow = reinterpret_cast<int2 *>(tb + L.off_overflow);
  uint32_t *tile_overflow = reinterpret_cast<uint32_t *>(tb + L.off_tile_overflow);
  const unsigned ptiles = (unsigned)ceil_div64(max_sample_points > 0 ? max_sample_points : 1, kVcThreads * kVcPer);
  const dim3 pgrid(ptiles, (unsigned)batch);
  if (ptiles > 65535u) return BEVPOOL_E_RANGE;            // (the claim kernel walks the tiles in grid.y: 67 M points per sample)
  BEVPOOL_RETURN_IF_CUDA(cudaMemsetAsync(first, 0x7f, L.first_bytes, stream));
  if (total_points > 0) {
    const size_t cell_smem = (size_t)kVcTile * F * sizeof(float);
    if (cell_smem + 64 > 48 * 1024)                       // point rows of 12 floats and more: beyond the default limit
      BEVPOOL_RETURN_IF_CUDA(cudaFuncSetAttribute(vox_cell_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cell_smem));
    vox_cell_kernel<<<pgrid, kVcThreads, cell_smem, stream>>>(pts, sample_offsets, F, g, cells, first, gcell, vox_l2_hints());
    BEVPOOL_LAUNCH_CHECK();
  }
  vox_scan_kernel<<<dim3((unsigned)tps, (unsigned)batch), kScanThreads, 0, stream>>>(
      sample_offsets, gcell, first, cell_of_vid, max_voxels, totals,
      reinterpret_cast<unsigned long long *>(tb + L.off_status), reinterpret_cast<unsigned int *>(tb + L.off_tickets),
      L.tiles_per_sample, vox_l2_hints());
  BEVPOOL_LAUNCH_CHECK();
  vox_dense_base_kernel<<<1, 32, 0, stream>>>(totals, batch, max_voxels, voxel_base);
  BEVPOOL_LAUNCH_CHECK();
  if (total_points > 0) {
    vox_claim_kernel<<<dim3((unsigned)batch, ptiles), 256, 0, stream>>>(sample_offsets, gcell, vid_of_cell, voxel_base, max_voxels, max_points, lists,
                                                arrivals, overflow, tile_overflow, L.tiles_cap, vox_l2_hints());
    BEVPOOL_LAUNCH_CHECK();
  }
  if (total_points > 0) {
    const dim3 egrid((unsigned)batch, ptiles);
    switch (max_points <= 16 ? vox_list_stride(max_points) / 4 : 0) {
      case 1: vox_evict_kernel<1><<<egrid, 128, 0, stream>>>(sample_offsets, overflow, tile_overflow, L.tiles_cap, max_points, lists); break;
      case 2: vox_evict_kernel<2><<<egrid, 128, 0, stream>>>(sample_offsets, overflow, tile_overflow, L.tiles_cap, max_points, lists); break;
      case 3: vox_evict_kernel<3><<<egrid, 128, 0, stream>>>(sample_offsets, overflow, tile_overflow, L.tiles_cap, max_points, lists); break;
      case 4: vox_evict_kernel<4><<<egrid, 128, 0, stream>>>(sample_offsets, overflow, tile_overflow, L.tiles_cap, max_points, lists); break;
      default: vox_evict_kernel<0><<<egrid, 128, 0, stream>>>(sample_offsets, overflow, tile_overflow, L.tiles_cap, max_points, lists); break;
    }
    BEVPOOL_LAUNCH_CHECK();
  }
  static const bool coop_on = [] { const char *e = std::getenv("BEVVOX_FIN_COOP"); return !(e && e[0] == '0'); }();
  const bool coop = coop_on && max_points <= 16;
  const size_t fin_smem = (coop ? (size_t)kFinWarps * vox_fin_coop_warp_bytes(max_points, F)
                                : (size_t)kFinWarps * 32 * max_points * F * sizeof(float)) + (size_t)(batch + 1) * sizeof(int);
  if (fin_smem > 200 * 1024) return BEVPOOL_E_RANGE;       // max_points * F beyond ~390 floats: not a pillar configuration
  if (ev_join) {
    BEVPOOL_RETURN_IF_CUDA(cudaStreamWaitEvent(stream, ev_join, 0));
    cudaEventDestroy(ev_join);
  }
  float *fin_canvas = dense_canvas ? nullptr : canvas;
  const uint32_t *arrivals_c = reinterpret_cast<const uint32_t *>(tb + L.off_arrivals);
  const dim3 cgrid((unsigned)ceil_div64(cells / 4, 256), (unsigned)batch);
  auto launch_canvas = [&](cudaStream_t cs) {
    if (mean_features <= 8)
      vox_canvas_dense_kernel<8><<<cgrid, 256, 0, cs>>>(vid_of_cell, voxel_base, voxel_mean, mean_features, max_voxels, cells, canvas);
    else
      vox_canvas_dense_kernel<16><<<cgrid, 256, 0, cs>>>(vid_of_cell, voxel_base, voxel_mean, mean_features, max_voxels, cells, canvas);
  };
  // (Tried: the finalize kernel in 2-4 launches over row ranges, each range's samples written to the canvas on a side
  // stream beside the next range -- 359 / 373 / 385 us per 32 sweeps against 344 us back to back: the DRAM-write stream
  // slows the finalize kernel's own streaming stores by more than the overlap returns.)
#define BEVVOX_FIN_ARGS pts, sample_offsets, F, g, cells, cell_of_vid, lists, arrivals_c, batch, \
                        max_voxels, max_points, voxels, num_points, coors, voxel_base, voxel_mean, mean_features, fin_canvas
#define BEVVOX_FIN_LAUNCH(KERNEL, GRID, THREADS)                                                                           \
  do {                                                                                                                     \
    if (fin_smem > 48 * 1024)                                                                                              \
      BEVPOOL_RETURN_IF_CUDA(cudaFuncSetAttribute(KERNEL, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fin_smem));    \
    KERNEL<<<GRID, THREADS, fin_smem, stream>>>(BEVVOX_FIN_ARGS);                                                          \
  } while (0)
  {
    const unsigned fin_grid = (unsigned)ceil_div64((int64_t)rows, kFinWarps * 32);
    if (coop) {
      if (F <= 8) BEVVOX_FIN_LAUNCH(vox_finalize_coop_kernel<8>, fin_grid, kFinWarps * 32);
      else BEVVOX_FIN_LAUNCH(vox_finalize_coop_kernel<16>, fin_grid, kFinWarps * 32);
    } else if (F <= 8) BEVVOX_FIN_LAUNCH(vox_finalize_kernel<8>, fin_grid, kFinWarps * 32);
    else BEVVOX_FIN_LAUNCH(vox_finalize_kernel<16>, fin_grid, kFinWarps * 32);
  }
#undef BEVVOX_FIN_LAUNCH
#undef BEVVOX_FIN_ARGS
  BEVPOOL_LAUNCH_CHECK();
  if (dense_canvas) {
    launch_canvas(stream);
    BEVPOOL_LAUNCH_CHECK();
  }
  return BEVPOOL_OK;
}

static int hard_voxelize_impl(const float *points, const float *const *sample_ptrs, const int32_t *sample_offsets, int batch, int64_t total_points,
                              int64_t max_sample_points, int num_features, const float *voxel_size_host,
                              const float *range_host, const int *grid_host, int max_points, int max_voxels,
                              float *voxels, int32_t *coors, int32_t *num_points, int32_t *voxel_base,
                              float *voxel_mean, int mean_features, float *canvas, void *temp, void *stream_,
                              bool canvas_prezeroed = false) {
  int rc = check_vox_args(batch, total_points, num_features, max_voxels, max_points);
  if (rc) return rc;
  if (!sample_offsets || !voxel_size_host || !range_host || !grid_host || !voxels || !coors || !num_points ||
      !voxel_base || !temp)
    return BEVPOOL_E_ARG;
  if (total_points > 0 && !points && !sample_ptrs) return BEVPOOL_E_ARG;
  if ((voxel_mean || canvas) && (mean_features <= 0 || mean_features > num_features || mean_features > 16)) return BEVPOOL_E_ARG;
  if (!aligned16(temp) || !aligned16(coors) || !aligned16(voxels)) return BEVPOOL_E_ALIGN;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const VoxGeom g = make_geom(voxel_size_host, range_host, grid_host);
  if (g.gx <= 0 || g.gy <= 0 || g.gz <= 0) return BEVPOOL_E_ARG;
  if (vox_dense_ok(batch, grid_host)) {
    // dense BEV canvas of the fused HardSimpleVFE mean: (batch, mean_features, gz, gy, gx), zero-filled by the call unless the caller did
    return hard_voxelize_dense(VoxPoints{points, sample_ptrs}, sample_offsets, batch, total_points, max_sample_points, num_features, g, grid_host,
                               max_points, max_voxels, voxels, coors, num_points, voxel_base, voxel_mean, mean_features,
                               canvas, temp, stream, !canvas_prezeroed);
  }
  if (sample_ptrs) return BEVPOOL_E_RANGE;          // per-sample pointers exist on the dense-grid path only
  if (canvas && !canvas_prezeroed)                  // the gather kernel stores the occupied cells
    BEVPOOL_RETURN_IF_CUDA(cudaMemsetAsync(canvas, 0, (size_t)batch * mean_features * g.gx * g.gy * g.gz * sizeof(float), stream));
  const VoxTemp L = vox_temp_layout(batch, total_points, max_voxels, max_points);
  char *tb = static_cast<char *>(temp);
  int32_t *counts = reinterpret_cast<int32_t *>(tb + L.off_counts);
  unsigned long long *keys = reinterpret_cast<unsigned long long *>(tb + L.off_keys);
  int32_t *first = reinterpret_cast<int32_t *>(tb + L.off_first);
  int32_t *lists = reinterpret_cast<int32_t *>(tb + L.off_lists);
  int32_t *point_slot = reinterpret_cast<int32_t *>(tb + L.off_slot);
  uint32_t *flags = reinterpret_cast<uint32_t *>(tb + L.off_flags);

  BEVPOOL_RETURN_IF_CUDA(cudaMemsetAsync(tb, 0, L.zero_bytes, stream));
  BEVPOOL_RETURN_IF_CUDA(cudaMemsetAsync(keys, 0xff, (size_t)L.hash_slots * 8, stream));
  BEVPOOL_RETURN_IF_CUDA(cudaMemsetAsync(first, 0x7f, L.fill7f_bytes, stream));

  const dim3 pgrid((unsigned)ceil_div64(max_sample_points > 0 ? max_sample_points : 1, 256), (unsigned)batch);
  if (total_points > 0) {
    vox_insert_kernel<<<pgrid, 256, 0, stream>>>(points, sample_offsets, num_features, g, keys, first,
                                                L.hash_slots - 1, point_slot);
    BEVPOOL_LAUNCH_CHECK();
  }
  vox_flag_kernel<<<(unsigned)ceil_div64(total_points + 1, 256), 256, 0, stream>>>(point_slot, first, total_points, flags);
  BEVPOOL_LAUNCH_CHECK();
  rc = launch_scan_exclusive(flags, flags, total_points + 1, tb + L.off_scan, stream);
  if (rc) return rc;
  vox_base_kernel<<<1, 32, 0, stream>>>(flags, sample_offsets, batch, max_voxels, voxel_base);
  BEVPOOL_LAUNCH_CHECK();
  if (total_points > 0) {
    vox_assign_kernel<<<pgrid, 256, 0, stream>>>(points, sample_offsets, num_features, g, point_slot, first, flags,
                                                voxel_base, max_voxels, max_points, lists, counts, coors);
    BEVPOOL_LAUNCH_CHECK();
  }
  const int64_t rows = (int64_t)batch * max_voxels;
  vox_gather_kernel<<<(unsigned)ceil_div64(rows, 8), 256, 0, stream>>>(points, num_features, lists, counts, voxel_base,
                                                                      batch, rows, max_points, voxels, num_points, coors,
                                                                      voxel_mean, mean_features, g, canvas);
  BEVPOOL_LAUNCH_CHECK();
  return BEVPOOL_OK;
}

extern "C" int bevvox_hard_voxelize(const float *points, const int32_t *sample_offsets, int batch,
                                    int64_t total_points, int64_t max_sample_points, int num_features,
                                    const float *voxel_size_host, const float *range_host,
                                    const int *grid_host, int max_points, int max_voxels, float *voxels,
                                    int32_t *coors, int32_t *num_points, int32_t *voxel_base,
                                    float *voxel_mean, int mean_features, void *temp, void *stream_) {
  return hard_voxelize_impl(points, nullptr, sample_offsets, batch, total_points, max_sample_points, num_features, voxel_size_host,
                            range_host, grid_host, max_points, max_voxels, voxels, coors, num_points, voxel_base, voxel_mean,
                            mean_features, nullptr, temp, stream_);
}

// voxelize + HardSimpleVFE + pillar scatter in one call (models/bev_depth.py:181-183 with a dense-scatter middle
// encoder).  The clouds are given either concatenated (`points`) or, on the dense-grid path, as a DEVICE array of
// `batch` per-sample base pointers (`sample_ptrs`, points == NULL): the list of tensors the reference passes, without a
// torch.cat.  canvas (batch, mean_features, gz, gy, gx) may be NULL (no scatter).
extern "C" int bevvox_hard_voxelize_scatter(const float *points, const float *const *sample_ptrs,
                                            const int32_t *sample_offsets, int batch, int64_t total_points,
                                            int64_t max_sample_points, int num_features, const float *voxel_size_host,
                                            const float *range_host, const int *grid_host, int max_points,
                                            int max_voxels, float *voxels, int32_t *coors, int32_t *num_points,
                                            int32_t *voxel_base, float *voxel_mean, int mean_features, float *canvas,
                                            int canvas_is_zeroed, void *temp, void *stream_) {
  return hard_voxelize_impl(points, sample_ptrs, sample_offsets, batch, total_points, max_sample_points, num_features,
                            voxel_size_host, range_host, grid_host, max_points, max_voxels, voxels, coors, num_points,
                            voxel_base, voxel_mean, mean_features, canvas, temp, stream_, canvas_is_zeroed != 0);
}

extern "C" int bevvox_dynamic_voxelize(const float *points, int64_t num_points, int num_features,
                                       const float *voxel_size_host, const float *range_host,
                                       const int *grid_host, int32_t *coors, void *stream_) {
  if (num_points < 0 || num_features < 3 || !voxel_size_host || !range_host || !grid_host) return BEVPOOL_E_ARG;
  if (num_points == 0) return BEVPOOL_OK;
  if (!points || !coors) return BEVPOOL_E_ARG;
  const VoxGeom g = make_geom(voxel_size_host, range_host, grid_host);
  vox_dynamic_kernel<<<(unsigned)ceil_div64(num_points, 256), 256, 0, static_cast<cudaStream_t>(stream_)>>>(
      points, num_points, num_features, g, coors);
  BEVPOOL_LAUNCH_CHECK();
  return BEVPOOL_OK;
}

extern "C" int pillar_scatter_forward(const void *voxel_features, const int32_t *coors, int64_t num_voxels,
                                      int channels, int dtype, int batch, int nz, int ny, int nx,
                                      void *canvas, int32_t *index_map, void *stream_) {
  if (num_voxels < 0 || channels <= 0 || batch <= 0 || batch > 65535 || nz <= 0 || ny <= 0 || nx <= 0) return BEVPOOL_E_ARG;
  if (!canvas || (num_voxels > 0 && (!voxel_features || !coors))) return BEVPOOL_E_ARG;
  if (num_voxels > 0 && !aligned16(coors)) return BEVPOOL_E_ALIGN;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const int64_t cells = (int64_t)nz * ny * nx;
  if (!index_map) {
    // UNIQUE coordinates promised by the caller (the output of hard voxelization): DRAM-speed zero fill of the canvas +
    // one store per (voxel, channel); with duplicate coordinates the winner would be arbitrary -- pass index_map then.
    const size_t esz = dtype == BEVPOOL_F32 ? 4 : 2;
    if (dtype != BEVPOOL_F32 && dtype != BEVPOOL_F16 && dtype != BEVPOOL_BF16) return BEVPOOL_E_DTYPE;
    BEVPOOL_RETURN_IF_CUDA(cudaMemsetAsync(canvas, 0, (size_t)batch * channels * cells * esz, stream));
    if (num_voxels == 0) return BEVPOOL_OK;
    const unsigned grid = (unsigned)ceil_div64(num_voxels * channels, 256);
    if (dtype == BEVPOOL_F32)
      scatter_unique_kernel<float><<<grid, 256, 0, stream>>>(static_cast<const float *>(voxel_features), coors, num_voxels, channels, batch, nz, ny, nx, static_cast<float *>(canvas));
    else
      scatter_unique_kernel<uint16_t><<<grid, 256, 0, stream>>>(static_cast<const uint16_t *>(voxel_features), coors, num_voxels, channels, batch, nz, ny, nx, static_cast<uint16_t *>(canvas));
    BEVPOOL_LAUNCH_CHECK();
    return BEVPOOL_OK;
  }
  BEVPOOL_RETURN_IF_CUDA(cudaMemsetAsync(index_map, 0xff, (size_t)batch * cells * 4, stream));
  if (num_voxels > 0) {
    scatter_index_kernel<<<(unsigned)ceil_div64(num_voxels, 256), 256, 0, stream>>>(coors, num_voxels, batch, nz, ny, nx, index_map);
    BEVPOOL_LAUNCH_CHECK();
  }
  const dim3 grid((unsigned)ceil_div64(cells, 256), (unsigned)batch);
  switch (dtype) {
    case BEVPOOL_F32:
      scatter_canvas_kernel<float><<<grid, 256, 0, stream>>>(static_cast<const float *>(voxel_features), index_map, channels, cells, static_cast<float *>(canvas));
      break;
    case BEVPOOL_F16:
      scatter_canvas_kernel<__half><<<grid, 256, 0, stream>>>(static_cast<const __half *>(voxel_features), index_map, channels, cells, static_cast<__half *>(canvas));
      break;
    case BEVPOOL_BF16:
      scatter_canvas_kernel<__nv_bfloat16><<<grid, 256, 0, stream>>>(static_cast<const __nv_bfloat16 *>(voxel_features), index_map, channels, cells, static_cast<__nv_bfloat16 *>(canvas));
      break;
    default: return BEVPOOL_E_DTYPE;
  }
  BEVPOOL_LAUNCH_CHECK();
  return BEVPOOL_OK;
}

extern "C" int pillar_scatter_backward(const void *grad_canvas, const int32_t *coors, int64_t num_voxels,
                                       int channels, int dtype, int batch, int nz, int ny, int nx,
                                       void *grad_voxel_features, void *stream_) {
  if (num_voxels < 0 || channels <= 0 || batch <= 0 || nz <= 0 || ny <= 0 || nx <= 0) return BEVPOOL_E_ARG;
  if (num_voxels == 0) return BEVPOOL_OK;
  if (!grad_canvas || !coors || !grad_voxel_features) return BEVPOOL_E_ARG;
  if (!aligned16(coors)) return BEVPOOL_E_ALIGN;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const unsigned grid = (unsigned)ceil_div64(num_voxels * channels, 256);
  switch (dtype) {
    case BEVPOOL_F32:
      scatter_backward_kernel<float><<<grid, 256, 0, stream>>>(static_cast<const float *>(grad_canvas), coors, num_voxels, channels, batch, nz, ny, nx, static_cast<float *>(grad_voxel_features));
      break;
    case BEVPOOL_F16:
      scatter_backward_kernel<__half><<<grid, 256, 0, stream>>>(static_cast<const __half *>(grad_canvas), coors, num_voxels, channels, batch, nz, ny, nx, static_cast<__half *>(grad_voxel_features));
      break;
    case BEVPOOL_BF16:
      scatter_backward_kernel<__nv_bfloat16><<<grid, 256, 0, stream>>>(static_cast<const __nv_bfloat16 *>(grad_canvas), coors, num_voxels, channels, batch, nz, ny, nx, static_cast<__nv_bfloat16 *>(grad_voxel_features));
      break;
    default: return BEVPOOL_E_DTYPE;
  }
  BEVPOOL_LAUNCH_CHECK();
  return BEVPOOL_OK;
}

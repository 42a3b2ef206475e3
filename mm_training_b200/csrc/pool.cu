// BEV voxel pooling kernels (sm_100a): deterministic sorted-interval segmented
// reduction (forward) and gather (backward), for both the drop-in op and the fused
// depth (x) context entry point.
//
// Reference behaviour being replaced:
//   forward  : ops/voxel_pooling/src/voxel_pooling_forward_cuda.cu:30-34 (C scalar fp32
//              atomicAdd per point) and, for the fused entry, the materialised outer
//              product of layers/backbones/lss_fpn.py:441-463
//   backward : ops/voxel_pooling/voxel_pooling.py:58-69 (mask + advanced-index gather)
//
// HBM-bound gather/scatter with <= 2 flop/byte: no tensor cores.  Every output
// element is written exactly once by exactly one thread, in a fixed order, so results
// are bit-stable run to run (the reference's are not).
#include "common.cuh"
#include "pool_g8.cuh"
#include "tma.cuh"

#include <cstdio>
#include <cstdlib>
#include <type_traits>

namespace bevpool {

// BEVPOOL_DISABLE_G8=1 forces the generic float4-per-lane kernels (used by the tests to cover both paths)
static bool g8_enabled() {
  const char *e = std::getenv("BEVPOOL_DISABLE_G8");
  return !(e && e[0] == '1');
}

// ---- element access: 4 consecutive channels <-> float4 -------------------------------
template <typename T> struct Vec4;
template <> struct Vec4<float> {
  static __device__ __forceinline__ float4 load(const float *p) { return __ldg(reinterpret_cast<const float4 *>(p)); }
  static __device__ __forceinline__ float4 load_stream(const float *p) { return ldg_stream_f4(reinterpret_cast<const float4 *>(p)); }
  static __device__ __forceinline__ void store(float *p, const float4 &v) { stg_stream_f4(reinterpret_cast<float4 *>(p), v); }
  static __device__ __forceinline__ float to_float(float v) { return v; }
  static __device__ __forceinline__ float from_float(float v) { return v; }
};
template <> struct Vec4<__half> {
  static __device__ __forceinline__ float4 load(const __half *p) {
    const uint2 u = __ldg(reinterpret_cast<const uint2 *>(p));
    const float2 a = __half22float2(*reinterpret_cast<const __half2 *>(&u.x));
    const float2 b = __half22float2(*reinterpret_cast<const __half2 *>(&u.y));
    return make_float4(a.x, a.y, b.x, b.y);
  }
  static __device__ __forceinline__ float4 load_stream(const __half *p) { return load(p); }
  static __device__ __forceinline__ void store(__half *p, const float4 &v) {
    __half2 a = __floats2half2_rn(v.x, v.y), b = __floats2half2_rn(v.z, v.w);
    uint2 u;
    u.x = *reinterpret_cast<unsigned *>(&a);
    u.y = *reinterpret_cast<unsigned *>(&b);
    *reinterpret_cast<uint2 *>(p) = u;
  }
  static __device__ __forceinline__ float to_float(__half v) { return __half2float(v); }
  static __device__ __forceinline__ __half from_float(float v) { return __float2half_rn(v); }
};
template <> struct Vec4<__nv_bfloat16> {
  static __device__ __forceinline__ float4 load(const __nv_bfloat16 *p) {
    const uint2 u = __ldg(reinterpret_cast<const uint2 *>(p));
    // bf16 -> f32 is a 16-bit shift
    return make_float4(__uint_as_float(u.x << 16), __uint_as_float(u.x & 0xffff0000u),
                       __uint_as_float(u.y << 16), __uint_as_float(u.y & 0xffff0000u));
  }
  static __device__ __forceinline__ float4 load_stream(const __nv_bfloat16 *p) { return load(p); }
  static __device__ __forceinline__ void store(__nv_bfloat16 *p, const float4 &v) {
    __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y), b = __floats2bfloat162_rn(v.z, v.w);
    uint2 u;
    u.x = *reinterpret_cast<unsigned *>(&a);
    u.y = *reinterpret_cast<unsigned *>(&b);
    *reinterpret_cast<uint2 *>(p) = u;
  }
  static __device__ __forceinline__ float to_float(__nv_bfloat16 v) { return __bfloat162float(v); }
  static __device__ __forceinline__ __nv_bfloat16 from_float(float v) { return __float2bfloat16_rn(v); }
};

constexpr int kPoolThreads = 256;
constexpr int kPoolWarps = kPoolThreads / 32;
constexpr int kUnroll = 8;     // feature rows in flight per warp
constexpr int kFwdTile = 32;   // BEV cells per CTA (contiguous rows of the NHWC output)

// ---- forward: CTA = 32 consecutive BEV cells, warps pull cells from a shared counter ----
// kFused = false: rows = feature rows (B*Np, C), streamed from HBM once.
// kFused = true : rows = context rows (B*N*H*W, C) (L1/L2 resident), scaled by depth[p].
// A cell's points are visited in ascending point order (stable plan) with separate multiply
// and add (no FMA contraction), so the fp32 result is bit-identical to a sequential
// scatter-add over the materialised tensor.  Empty tiles are zero-filled with coalesced stores.
template <typename T, int CPL, bool kFused, bool kGuard>
__device__ __forceinline__ void accum_batch(float4 (&acc)[CPL], const T *__restrict__ rows, int my_row,
                                            float my_d, int j, int n, int lane, int C, int C4) {
  float4 v[kUnroll][CPL];
  float d[kUnroll];
#pragma unroll
  for (int u = 0; u < kUnroll; ++u) {
    const int row = __shfl_sync(0xffffffffu, my_row, j + u);
    d[u] = __shfl_sync(0xffffffffu, my_d, j + u);
    if (!kGuard || j + u < n) {
      const T *rp = rows + (int64_t)row * C;
#pragma unroll
      for (int k = 0; k < CPL; ++k) {
        const int ch = lane + 32 * k;
        if (ch < C4) v[u][k] = kFused ? Vec4<T>::load(rp + ch * 4) : Vec4<T>::load_stream(rp + ch * 4);
      }
    }
  }
#pragma unroll
  for (int u = 0; u < kUnroll; ++u) {
    if (!kGuard || j + u < n) {
#pragma unroll
      for (int k = 0; k < CPL; ++k) {
        if (kFused) {
          acc[k].x = __fadd_rn(acc[k].x, __fmul_rn(d[u], v[u][k].x));
          acc[k].y = __fadd_rn(acc[k].y, __fmul_rn(d[u], v[u][k].y));
          acc[k].z = __fadd_rn(acc[k].z, __fmul_rn(d[u], v[u][k].z));
          acc[k].w = __fadd_rn(acc[k].w, __fmul_rn(d[u], v[u][k].w));
        } else {
          acc[k].x += v[u][k].x;
          acc[k].y += v[u][k].y;
          acc[k].z += v[u][k].z;
          acc[k].w += v[u][k].w;
        }
      }
    }
  }
}

template <typename T, int CPL, bool kFused>
__global__ void __launch_bounds__(kPoolThreads)
pool_forward_kernel(const int32_t *__restrict__ cell_start, const int32_t *__restrict__ sorted_ids,
                    const T *__restrict__ rows, const T *__restrict__ depth, T *__restrict__ out,
                    int64_t total_cells, int C, int dhw, int hw) {
  __shared__ int s_start[kFwdTile + 1];
  __shared__ int s_next;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t tile0 = (int64_t)blockIdx.x * kFwdTile;
  const int ncell = (int)min((int64_t)kFwdTile, total_cells - tile0);
  const int C4 = C >> 2;
  if (threadIdx.x <= ncell) s_start[threadIdx.x] = cell_start[tile0 + threadIdx.x];
  if (threadIdx.x == 0) s_next = kPoolWarps;
  __syncthreads();
  T *tile_out = out + tile0 * C;
  if (s_start[ncell] == s_start[0]) {   // nothing lands in this tile
    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int i = threadIdx.x; i < ncell * C4; i += kPoolThreads) Vec4<T>::store(tile_out + i * 4, z);
    return;
  }
  int c = warp;                          // first cell is static, later ones come from the counter
  while (c < ncell) {
    const int start = s_start[c], end = s_start[c + 1];
    float4 acc[CPL];
#pragma unroll
    for (int k = 0; k < CPL; ++k) acc[k] = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int base = start; base < end; base += 32) {
      const int n = min(32, end - base);
      int my_row = 0;
      float my_d = 0.f;
      if (lane < n) {
        const int gp = sorted_ids[base + lane];
        if (kFused) {
          my_d = Vec4<T>::to_float(depth[gp]);
          my_row = (gp / dhw) * hw + gp % hw;   // pixel row: (b*N+n)*H*W + h*W + w
        } else {
          my_row = gp;
        }
      }
      int j = 0;
      for (; j + kUnroll <= n; j += kUnroll)
        accum_batch<T, CPL, kFused, false>(acc, rows, my_row, my_d, j, n, lane, C, C4);
      if (j < n) accum_batch<T, CPL, kFused, true>(acc, rows, my_row, my_d, j, n, lane, C, C4);
    }
    T *op = tile_out + (int64_t)c * C;
#pragma unroll
    for (int k = 0; k < CPL; ++k) {
      const int ch = lane + 32 * k;
      if (ch < C4) Vec4<T>::store(op + ch * 4, acc[k]);
    }
    if (lane == 0) c = atomicAdd(&s_next, 1);
    c = __shfl_sync(0xffffffffu, c, 0);
  }
}

// ---- backward of the drop-in op: point-centric gather ---------------------------------
// grad_features[p, :] = kept(p) ? grad_out_nhwc[b, cell(p), :] : 0 ; each row written once.
constexpr int kBwdPoints = 64;  // points per CTA
template <typename T>
__global__ void __launch_bounds__(kPoolThreads)
pool_backward_kernel(const int32_t *__restrict__ cell_of_point, const T *__restrict__ grad_nhwc,
                     T *__restrict__ grad_rows, int64_t total_points, int64_t num_points,
                     int64_t cells_per_sample, int C) {
  __shared__ int64_t s_row[kBwdPoints];
  const int C4 = C >> 2;
  const int64_t gp0 = (int64_t)blockIdx.x * kBwdPoints;
  if (threadIdx.x < kBwdPoints) {
    const int64_t gp = gp0 + threadIdx.x;
    int64_t row = -1;
    if (gp < total_points) {
      const int cell = cell_of_point[gp];
      if (cell >= 0) row = (gp / num_points) * cells_per_sample + cell;
    }
    s_row[threadIdx.x] = row;
  }
  __syncthreads();
  const int npts = (int)min((int64_t)kBwdPoints, total_points - gp0);
  const int work = npts * C4;
  for (int i = threadIdx.x; i < work; i += kPoolThreads) {
    const int pl = i / C4, ch = i - pl * C4;
    const int64_t row = s_row[pl];
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (row >= 0) v = Vec4<T>::load(grad_nhwc + row * C + ch * 4);
    Vec4<T>::store(grad_rows + (gp0 + pl) * C + ch * 4, v);
  }
}

// ---- backward of the fused op: pixel-centric, no atomics, no sort ----------------------
// One warp owns one pixel (camera image bn, row h, column w) at a time and walks its ray:
//   grad_depth[d, pix]  = <grad_out[cell(d, pix), :], context[pix, :]>
//   grad_context[pix,:] = sum_d depth[d, pix] * grad_out[cell(d, pix), :]
// The warps of a CTA are the rows h of the same image columns: all rows of a column project
// to (nearly) the same BEV cells, so the CTA's warps gather the same gradient rows and all
// but the first hit L1.  Depth bins are taken 32 at a time (lane = bin); dropped bins are
// skipped; the 32 per-bin partial dot products are reduced with one lane-transposing butterfly
// (31 shuffles per 32 bins instead of 5 per bin).
constexpr int kBwdTileW = 4;     // image columns per CTA
constexpr int kBwdMaxWarps = 8;  // image rows per CTA

__device__ __forceinline__ float transpose_reduce32(float (&p)[32], int lane) {
#pragma unroll
  for (int w = 16; w >= 1; w >>= 1) {
    const bool hi = (lane & w) != 0;
#pragma unroll
    for (int i = 0; i < w; ++i) {
      const float send = hi ? p[i] : p[i + w];
      const float keep = hi ? p[i + w] : p[i];
      p[i] = keep + __shfl_xor_sync(0xffffffffu, send, w);
    }
  }
  return p[0];   // lane l now holds the sum over lanes of the original p[l]
}

template <typename T, int CPL>
__global__ void __launch_bounds__(kBwdMaxWarps * 32)
fused_backward_kernel(const int32_t *__restrict__ cell_of_point, const T *__restrict__ grad_nhwc,
                      const T *__restrict__ depth, const T *__restrict__ ctx_nhwc,
                      T *__restrict__ grad_depth, T *__restrict__ grad_ctx_nhwc, int num_cams, int D,
                      int H, int W, int C, int64_t cells_per_sample) {
  const int lane = threadIdx.x & 31;
  const int bn = blockIdx.z;
  const int h = blockIdx.y * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (h >= H) return;
  const int HW = H * W, C4 = C >> 2;
  const int64_t img_base = (int64_t)bn * D * HW;   // first global point id of this image
  const T *gbase = grad_nhwc + (int64_t)(bn / num_cams) * cells_per_sample * C;
  const int w_end = min(W, (int)(blockIdx.x + 1) * kBwdTileW);

  for (int w = blockIdx.x * kBwdTileW; w < w_end; ++w) {
    const int hw = h * W + w;
    float4 cx[CPL], gacc[CPL];
#pragma unroll
    for (int k = 0; k < CPL; ++k) {
      const int ch = lane + 32 * k;
      gacc[k] = make_float4(0.f, 0.f, 0.f, 0.f);
      cx[k] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (ch < C4) cx[k] = Vec4<T>::load(ctx_nhwc + ((int64_t)bn * HW + hw) * C + ch * 4);
    }
    for (int d0 = 0; d0 < D; d0 += 32) {
      const int d = d0 + lane;
      const int64_t gp = img_base + (int64_t)d * HW + hw;
      int cell = -1;
      float dv = 0.f;
      if (d < D) {
        cell = __ldg(cell_of_point + gp);
        dv = Vec4<T>::to_float(__ldg(depth + gp));
      }
      const unsigned mask = __ballot_sync(0xffffffffu, cell >= 0);
      float result = 0.f;
      if (mask) {
        float part[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) part[i] = 0.f;
        unsigned m = mask;
#pragma unroll
        for (int j0 = 0; j0 < 32; j0 += 4) {
          if (m == 0) break;
          float4 g[4][CPL];
          float dvu[4];
          bool on[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            on[q] = m != 0;
            const int u = on[q] ? __ffs(m) - 1 : 0;
            m &= m - 1;
            const int cu = __shfl_sync(0xffffffffu, cell, u);
            dvu[q] = __shfl_sync(0xffffffffu, dv, u);
#pragma unroll
            for (int k = 0; k < CPL; ++k) {
              const int ch = lane + 32 * k;
              g[q][k] = make_float4(0.f, 0.f, 0.f, 0.f);
              if (on[q] && ch < C4) g[q][k] = Vec4<T>::load(gbase + (int64_t)cu * C + ch * 4);
            }
          }
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            if (on[q]) {
              float dot = 0.f;
#pragma unroll
              for (int k = 0; k < CPL; ++k) {
                dot += g[q][k].x * cx[k].x + g[q][k].y * cx[k].y + g[q][k].z * cx[k].z + g[q][k].w * cx[k].w;
                gacc[k].x += dvu[q] * g[q][k].x;
                gacc[k].y += dvu[q] * g[q][k].y;
                gacc[k].z += dvu[q] * g[q][k].z;
                gacc[k].w += dvu[q] * g[q][k].w;
              }
              part[j0 + q] = dot;
            }
          }
        }
        // lane r holds the dot product of the r-th kept bin; route it to the lane owning that bin
        const float red = transpose_reduce32(part, lane);
        const int rank = __popc(mask & ((1u << lane) - 1u));
        result = __shfl_sync(0xffffffffu, red, rank);
        if (cell < 0) result = 0.f;
      }
      if (d < D) grad_depth[gp] = Vec4<T>::from_float(result);
    }
#pragma unroll
    for (int k = 0; k < CPL; ++k) {
      const int ch = lane + 32 * k;
      if (ch < C4) Vec4<T>::store(grad_ctx_nhwc + ((int64_t)bn * HW + hw) * C + ch * 4, gacc[k]);
    }
  }
}

// ---- gradient rows: NCHW grad_out -> (B, Y, X, C) rows, occupied cells only ---------------
// The backward kernels only ever read the rows of cells that received at least one point, so
// tiles of 32 cells with no kept point are skipped entirely (about 80 % of the aiMotive grid)
// and inside a tile only occupied rows are written.  E = raw element type (uint32_t / uint16_t).
constexpr int kGrTilesPerCta = 8;   // consecutive 32-cell tiles per CTA: empty tiles cost a flag test, not a CTA launch
template <typename E>
__global__ void __launch_bounds__(256)
grad_rows_kernel(const int32_t *__restrict__ cell_start, const E *__restrict__ grad_nchw,
                 E *__restrict__ rows, int64_t G, int C) {
  pdl_wait();
  pdl_trigger();
  extern __shared__ __align__(16) unsigned char smem_raw[];
  E *tile = reinterpret_cast<E *>(smem_raw);   // [32][C + 1]
  __shared__ unsigned s_occ[kGrTilesPerCta];
  const int b = blockIdx.y;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // occupancy masks of this CTA's tiles: warp w tests tile w
  if (warp < kGrTilesPerCta) {
    const int64_t cell0 = ((int64_t)blockIdx.x * kGrTilesPerCta + warp) * 32;
    unsigned m = 0u;
    if (cell0 < G) {
      const int ncell = (int)min((int64_t)32, G - cell0);
      const int64_t gc = (int64_t)b * G + cell0 + lane;
      const bool occ = lane < ncell && cell_start[gc + 1] > cell_start[gc];
      m = __ballot_sync(0xffffffffu, occ);
    }
    if (lane == 0) s_occ[warp] = m;
  }
  __syncthreads();
  const int ld = C + 1;
  for (int k = 0; k < kGrTilesPerCta; ++k) {
    const unsigned occ = s_occ[k];
    if (occ == 0) continue;                       // CTA-uniform
    const int64_t cell0 = ((int64_t)blockIdx.x * kGrTilesPerCta + k) * 32;
    const int ncell = (int)min((int64_t)32, G - cell0);
    // a warp takes every 8th channel; 10 independent 128-byte row loads in flight per lane (80 channels per round)
    const E *src = grad_nchw + (int64_t)b * C * G + cell0 + lane;
    for (int c0 = warp; c0 < C; c0 += 80) {
      E v[10];
#pragma unroll
      for (int k = 0; k < 10; ++k) {
        const int ch = c0 + 8 * k;
        v[k] = (ch < C && lane < ncell) ? src[(int64_t)ch * G] : E(0);
      }
#pragma unroll
      for (int k = 0; k < 10; ++k) {
        const int ch = c0 + 8 * k;
        if (ch < C) tile[lane * ld + ch] = v[k];
      }
    }
    __syncthreads();
    for (int j = warp; j < ncell; j += 8) {
      if (!((occ >> j) & 1u)) continue;
      E *rp = rows + ((int64_t)b * G + cell0 + j) * C;
      for (int c = lane; c < C; c += 32) rp[c] = tile[j * ld + c];
    }
    __syncthreads();
  }
}

// ---- gradient rows, fp32, TMA version ---------------------------------------------------------------
// Same contract as grad_rows_kernel (rows of occupied 32-cell tiles only).  A tile of 32 consecutive cells of
// one BEV row is ONE tensor-map box of the NCHW gradient -- 32 x-cells x C channels, 128-byte rows -- landing in
// shared memory as [channel][cell]; it is turned into [cell][channel] by a diagonal walk (lane l moves element
// (channel c0 + l/2, cell l): reads hit 32 distinct banks, writes (16*cell + channel) mod 32 do too at C = 80) and
// leaves as ONE contiguous bulk store of 32 rows (32 * C * 4 bytes: the tile's rows are adjacent in the NHWC
// buffer).  No LSU traffic to global memory at all.  A CTA owns every gridDim-th tile: it first finds the
// occupied ones among them in ONE parallel round of cell_start loads (80 % of the aiMotive grid is empty), then
// streams them through a 2-deep ring: the box of tile i+1 is in flight while tile i is transposed and stored.
constexpr int kGtCells = 32;
constexpr int kGtThreads = 128;
constexpr int kGtStages = 2;
template <int C>
__global__ void __launch_bounds__(kGtThreads)
grad_rows_tma_kernel(const __grid_constant__ CUtensorMap grad_map, const int32_t *__restrict__ cell_start,
                     float *__restrict__ rows, int X, int Y, int batch, int tiles_x) {
  pdl_wait();
  pdl_trigger();
  extern __shared__ __align__(128) unsigned char gt_raw[];
  float *s_in = reinterpret_cast<float *>(gt_raw);                 // [stage][C][32]
  float *s_out = s_in + kGtStages * C * kGtCells;                  // [stage][32][C]
  uint64_t *s_bar = reinterpret_cast<uint64_t *>(s_out + kGtStages * C * kGtCells);   // [stage]
  int *s_list = reinterpret_cast<int *>(s_bar + kGtStages);        // occupied tiles of this CTA (as k: tile = blockIdx.x + k * gridDim.x)
  __shared__ int s_count;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t tiles = (int64_t)batch * Y * tiles_x;
  if (tid == 0) {
    for (int i = 0; i < kGtStages; ++i) mbar_init(s_bar + i, 1);
    fence_proxy_async();
    s_count = 0;
  }
  __syncthreads();
  // ---- occupied tiles of this CTA, in ascending order (a warp-ordered compaction)
  const int per_cta = (int)((tiles - blockIdx.x + gridDim.x - 1) / gridDim.x);
  for (int k0 = 0; k0 < per_cta; k0 += kGtThreads) {
    const int k = k0 + tid;
    bool occ = false;
    if (k < per_cta) {
      const int64_t t = blockIdx.x + (int64_t)k * gridDim.x;
      const int tx = (int)(t % tiles_x);
      const int64_t c0 = (t / tiles_x) * X + (int64_t)tx * kGtCells;
      const int ncell = min(kGtCells, X - tx * kGtCells);
      occ = __ldg(cell_start + c0 + ncell) != __ldg(cell_start + c0);
    }
    const unsigned m = __ballot_sync(0xffffffffu, occ);
    for (int w = 0; w < kGtThreads / 32; ++w) {                    // warps append in order
      if (w == warp) {
        const int base = s_count;
        if (occ) s_list[base + __popc(m & ((1u << lane) - 1u))] = k;
        __syncwarp();
        if (lane == 0) s_count = base + __popc(m);
      }
      __syncthreads();
    }
  }
  const int n = s_count;
  auto issue = [&](int i) {                                        // box of the i-th occupied tile -> stage i % 2
    if (i < n && tid == 0) {
      const int64_t t = blockIdx.x + (int64_t)s_list[i] * gridDim.x;
      const int tx = (int)(t % tiles_x);
      const int64_t by = t / tiles_x;
      const int st = i % kGtStages;
      mbar_expect_tx(s_bar + st, (uint32_t)(C * kGtCells * 4));
      tma_load_4d(s_in + st * C * kGtCells, &grad_map, tx * kGtCells, (int)(by % Y), 0, (int)(by / Y), s_bar + st);
    }
  };
  issue(0);
  for (int i = 0; i < n; ++i) {
    const int st = i % kGtStages;
    issue(i + 1);                                                  // its stage was drained in iteration i - 1
    const int64_t t = blockIdx.x + (int64_t)s_list[i] * gridDim.x;
    const int tx = (int)(t % tiles_x);
    const int64_t c0 = (t / tiles_x) * X + (int64_t)tx * kGtCells;
    const int ncell = min(kGtCells, X - tx * kGtCells);
    mbar_wait(s_bar + st, (uint32_t)((i / kGtStages) & 1));
    // the bulk store that last read this output stage (iteration i - 2) must have drained it
    if (tid == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
    __syncthreads();
    const float *in = s_in + st * C * kGtCells;
    float *outp = s_out + st * C * kGtCells;
    for (int cb = warp; cb < C; cb += kGtThreads / 32) {           // diagonal transpose
      int c = cb + (lane >> 1);
      c = c >= C ? c - C : c;
      outp[lane * C + c] = in[c * kGtCells + lane];
    }
    fence_proxy_async();
    __syncthreads();                                               // s_out[st] complete; s_in[st] free for tile i + 2
    if (tid == 0) {
      tma_store_1d(rows + c0 * C, outp, (uint32_t)(ncell * C * 4));
      tma_store_commit();
    }
  }
  if (tid == 0) tma_store_wait_read();                             // shared memory must outlive the stores reading it
}

// ---- (batch, R, Cc) -> (batch, Cc, R) tiled transpose ----------------------------------
template <typename T>
__global__ void __launch_bounds__(256)
transpose_kernel(const T *__restrict__ in, T *__restrict__ out, int64_t R, int64_t Cc) {
  pdl_wait();
  pdl_trigger();
  __shared__ T tile[32][33];
  const int64_t batch_off = (int64_t)blockIdx.z * R * Cc;
  const int64_t c0 = (int64_t)blockIdx.x * 32, r0 = (int64_t)blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
#pragma unroll
  for (int i = ty; i < 32; i += 8) {
    const int64_t r = r0 + i, c = c0 + tx;
    if (r < R && c < Cc) tile[i][tx] = in[batch_off + r * Cc + c];
  }
  __syncthreads();
#pragma unroll
  for (int i = ty; i < 32; i += 8) {
    const int64_t c = c0 + i, r = r0 + tx;
    if (r < R && c < Cc) out[batch_off + c * R + r] = tile[tx][i];
  }
}

// ---- launchers ----------------------------------------------------------------------------
static size_t forward_workspace_bytes(int C) {
  // head + tail partial rows of every slice of the largest grid the forward may launch
  return (size_t)2 * 4 * kFwWarpsPerCta * kFwMaxCtasPerSm * sm_count() * (size_t)C * sizeof(float);
}

template <typename T, bool kFused>
static int launch_forward(const PlanView &pv, const T *rows, const T *depth, T *out, void *workspace,
                          int64_t total_cells, int C, int dhw, int hw, cudaStream_t s) {
  const unsigned grid = (unsigned)ceil_div64(total_cells, kFwdTile);
  const int C4 = C >> 2;
  if constexpr (std::is_same<T, float>::value) {
    if (g8_supported(C) && g8_enabled()) {
      if (!workspace) return BEVPOOL_E_ARG;
      if (!aligned16(workspace)) return BEVPOOL_E_ALIGN;
      const FastDiv fd_dhw = make_fastdiv((uint32_t)dhw), fd_hw = make_fastdiv((uint32_t)hw);
      static const int cps_env = env_int("BEVPOOL_FW_CPS", 6), u = env_int("BEVPOOL_FW_U", 4);   // read once
      const int cps = cps_env < 2 ? 2 : (cps_env > kFwMaxCtasPerSm ? kFwMaxCtasPerSm : cps_env);   // CTAs per SM: cps-1 reduce + 1 zero-fill
      const unsigned ctas = (unsigned)(sm_count() * cps);
      const int slices = (int)(ctas - ctas / cps) * kFwWarpsPerCta * 4;
      float *ws_head = static_cast<float *>(workspace);
      float *ws_tail = ws_head + (size_t)slices * C;
      if (u == 2) {
        BEVPOOL_G8_DISPATCH(C, (pool_forward_share_kernel<NV2, kFused, 2><<<ctas, kFwWarpsPerCta * 32, 0, s>>>(
                                   pv.cell_start, pv.sorted_ids, pv.sorted_cells, rows, depth, out, ws_head, ws_tail,
                                   (int64_t)0, total_cells, fd_dhw, fd_hw, cps, (int64_t)INT32_MAX, (int64_t)C)));
      } else {
        BEVPOOL_G8_DISPATCH(C, (pool_forward_share_kernel<NV2, kFused, 4><<<ctas, kFwWarpsPerCta * 32, 0, s>>>(
                                   pv.cell_start, pv.sorted_ids, pv.sorted_cells, rows, depth, out, ws_head, ws_tail,
                                   (int64_t)0, total_cells, fd_dhw, fd_hw, cps, (int64_t)INT32_MAX, (int64_t)C)));
      }
      BEVPOOL_LAUNCH_CHECK();
      BEVPOOL_G8_DISPATCH(C, (pool_forward_fixup_kernel<NV2><<<(unsigned)ceil_div64((int64_t)slices * 8, 128), 128, 0, s>>>(
                                 pv.cell_start, pv.sorted_cells, ws_head, ws_tail, out, (int64_t)0, total_cells, slices, (int64_t)INT32_MAX, (int64_t)C)));
      BEVPOOL_LAUNCH_CHECK();
      return BEVPOOL_OK;
    }
  }
  if (C4 <= 32)
    pool_forward_kernel<T, 1, kFused><<<grid, kPoolThreads, 0, s>>>(pv.cell_start, pv.sorted_ids, rows, depth, out, total_cells, C, dhw, hw);
  else if (C4 <= 64)
    pool_forward_kernel<T, 2, kFused><<<grid, kPoolThreads, 0, s>>>(pv.cell_start, pv.sorted_ids, rows, depth, out, total_cells, C, dhw, hw);
  else
    pool_forward_kernel<T, 4, kFused><<<grid, kPoolThreads, 0, s>>>(pv.cell_start, pv.sorted_ids, rows, depth, out, total_cells, C, dhw, hw);
  BEVPOOL_LAUNCH_CHECK();
  return BEVPOOL_OK;
}

template <typename T, int CPL>
static int launch_fused_backward_cpl(const PlanView &pv, const T *grad, const T *depth, const T *ctx,
                                     T *gdepth, T *gctx, int batch, int N, int D, int H, int W, int C,
                                     int64_t cells, cudaStream_t s) {
  const int warps = H < kBwdMaxWarps ? H : kBwdMaxWarps;
  if ((int64_t)batch * N > 65535 || ceil_div64(H, warps) > 65535) return BEVPOOL_E_RANGE;
  const dim3 grid((unsigned)ceil_div64(W, kBwdTileW), (unsigned)ceil_div64(H, warps), (unsigned)(batch * N));
  fused_backward_kernel<T, CPL><<<grid, warps * 32, 0, s>>>(pv.cell_of_point, grad, depth, ctx, gdepth, gctx,
                                                          N, D, H, W, C, cells);
  BEVPOOL_LAUNCH_CHECK();
  return BEVPOOL_OK;
}

static int check_channels(int C) {
  if (C <= 0 || (C & 3) != 0 || C > 512) return BEVPOOL_E_CHANNELS;
  return BEVPOOL_OK;
}

template <typename T>
static int forward_t(const void *plan, const void *feats, void *out, void *ws, int B, int64_t Np, int C, int X,
                     int Y, cudaStream_t s) {
  const PlanView pv = plan_view(plan, B, Np, X, Y);
  return launch_forward<T, false>(pv, static_cast<const T *>(feats), nullptr, static_cast<T *>(out), ws,
                                  (int64_t)B * X * Y, C, 1, 1, s);
}
template <typename T>
static int backward_t(const void *plan, const void *grad, void *gfeats, int B, int64_t Np, int C, int X,
                      int Y, cudaStream_t s) {
  const PlanView pv = plan_view(plan, B, Np, X, Y);
  const int64_t total = (int64_t)B * Np;
  pool_backward_kernel<T><<<(unsigned)ceil_div64(total, kBwdPoints), kPoolThreads, 0, s>>>(
      pv.cell_of_point, static_cast<const T *>(grad), static_cast<T *>(gfeats), total, Np,
      (int64_t)X * Y, C);
  BEVPOOL_LAUNCH_CHECK();
  return BEVPOOL_OK;
}
template <typename T>
static int fused_forward_t(const void *plan, const void *depth, const void *ctx, void *out, void *ws, int B, int N,
                           int D, int H, int W, int C, int X, int Y, cudaStream_t s) {
  const int64_t Np = (int64_t)N * D * H * W;
  const PlanView pv = plan_view(plan, B, Np, X, Y);
  return launch_forward<T, true>(pv, static_cast<const T *>(ctx), static_cast<const T *>(depth),
                                 static_cast<T *>(out), ws, (int64_t)B * X * Y, C, D * H * W, H * W, s);
}
// pixel-row context on any plan: tile kernel (pool_bwd.cu; fp32, C <= 96), else the generic kernel
template <typename T>
static int fused_backward_t(const void *plan, const void *grad, const void *depth, const void *ctx,
                            void *gdepth, void *gctx, int B, int N, int D, int H, int W, int C, int X,
                            int Y, cudaStream_t s) {
  const int64_t Np = (int64_t)N * D * H * W;
  const PlanView pv = plan_view(plan, B, Np, X, Y);
  const int C4 = C >> 2;
  const T *g = static_cast<const T *>(grad), *dp = static_cast<const T *>(depth), *cx = static_cast<const T *>(ctx);
  T *gd = static_cast<T *>(gdepth), *gc = static_cast<T *>(gctx);
  const int64_t cells = (int64_t)X * Y;
  if constexpr (std::is_same<T, float>::value) {
    if (g8_supported(C) && g8_enabled() && fused_backward_tile_supported(C))
      return launch_fused_backward_tile(pv.cell_of_point, g, dp, cx, gd, gc, B, N, D, H, W, C, cells, s);
  }
  if (C4 <= 32) return launch_fused_backward_cpl<T, 1>(pv, g, dp, cx, gd, gc, B, N, D, H, W, C, cells, s);
  if (C4 <= 64) return launch_fused_backward_cpl<T, 2>(pv, g, dp, cx, gd, gc, B, N, D, H, W, C, cells, s);
  return launch_fused_backward_cpl<T, 4>(pv, g, dp, cx, gd, gc, B, N, D, H, W, C, cells, s);
}

}  // namespace bevpool

using namespace bevpool;

#define BEVPOOL_DISPATCH_DTYPE(dtype, CALL)                        \
  switch (dtype) {                                                 \
    case BEVPOOL_F32: { using T = float; return CALL; }            \
    case BEVPOOL_F16: { using T = __half; return CALL; }           \
    case BEVPOOL_BF16: { using T = __nv_bfloat16; return CALL; }   \
    default: return BEVPOOL_E_DTYPE;                               \
  }

extern "C" int bevpool_forward_workspace_bytes(int channels, size_t *bytes) {
  if (!bytes || channels <= 0) return BEVPOOL_E_ARG;
  *bytes = forward_workspace_bytes(channels);
  return BEVPOOL_OK;
}

extern "C" int bevpool_forward(const void *plan, const void *features, void *out_nhwc, int dtype,
                               int batch, int64_t num_points, int channels, int X, int Y, void *workspace,
                               void *stream) {
  int rc = check_plan_dims(batch, num_points, X, Y);
  if (rc) return rc;
  if ((rc = check_channels(channels))) return rc;
  if (!plan || !features || !out_nhwc) return BEVPOOL_E_ARG;
  if (!aligned16(features) || !aligned16(out_nhwc)) return BEVPOOL_E_ALIGN;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  BEVPOOL_DISPATCH_DTYPE(dtype, (forward_t<T>(plan, features, out_nhwc, workspace, batch, num_points, channels, X, Y, s)));
}

extern "C" int bevpool_backward(const void *plan, const void *grad_out_nhwc, void *grad_features,
                                int dtype, int batch, int64_t num_points, int channels, int X, int Y,
                                void *stream) {
  int rc = check_plan_dims(batch, num_points, X, Y);
  if (rc) return rc;
  if ((rc = check_channels(channels))) return rc;
  if (!plan || !grad_out_nhwc || !grad_features) return BEVPOOL_E_ARG;
  if (!aligned16(grad_out_nhwc) || !aligned16(grad_features)) return BEVPOOL_E_ALIGN;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  BEVPOOL_DISPATCH_DTYPE(dtype, (backward_t<T>(plan, grad_out_nhwc, grad_features, batch, num_points, channels, X, Y, s)));
}

extern "C" int bevpool_fused_forward(const void *plan, const void *depth, const void *context_nhwc,
                                     void *out_nhwc, int dtype, int batch, int num_cams, int depth_bins,
                                     int feat_h, int feat_w, int channels, int X, int Y, void *workspace,
                                     void *stream) {
  int rc = check_frustum_dims(batch, num_cams, depth_bins, feat_h, feat_w, X, Y);
  if (rc) return rc;
  if ((rc = check_channels(channels))) return rc;
  if (!plan || !depth || !context_nhwc || !out_nhwc) return BEVPOOL_E_ARG;
  if (!aligned16(context_nhwc) || !aligned16(out_nhwc)) return BEVPOOL_E_ALIGN;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  BEVPOOL_DISPATCH_DTYPE(dtype, (fused_forward_t<T>(plan, depth, context_nhwc, out_nhwc, workspace, batch, num_cams, depth_bins, feat_h, feat_w, channels, X, Y, s)));
}

extern "C" int bevpool_fused_backward(const void *plan, const void *grad_out_nhwc, const void *depth,
                                      const void *context_nhwc, void *grad_depth, void *grad_context_nhwc,
                                      int dtype, int batch, int num_cams, int depth_bins, int feat_h,
                                      int feat_w, int channels, int X, int Y, void *stream) {
  int rc = check_frustum_dims(batch, num_cams, depth_bins, feat_h, feat_w, X, Y);
  if (rc) return rc;
  if ((rc = check_channels(channels))) return rc;
  if (!plan || !grad_out_nhwc || !depth || !context_nhwc || !grad_depth || !grad_context_nhwc) return BEVPOOL_E_ARG;
  if (!aligned16(grad_out_nhwc) || !aligned16(context_nhwc) || !aligned16(grad_context_nhwc)) return BEVPOOL_E_ALIGN;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  BEVPOOL_DISPATCH_DTYPE(dtype, (fused_backward_t<T>(plan, grad_out_nhwc, depth, context_nhwc, grad_depth, grad_context_nhwc, batch, num_cams, depth_bins, feat_h, feat_w, channels, X, Y, s)));
}

// The run-plan backward behind both entry points below: the gradient row of cell c starts at grad_rows + c * grad_row_stride
// floats.  col_args: the entry point takes only what the column kernel reads (W % 4 == 0, 16-byte aligned depth and
// grad_depth) whatever the layout.  Column kernel (pool_bwd2.cu; pair records); BEVPOOL_BW_KERNEL=1 picks the pixel-row
// kernels where they can run: NCHW context and strided gradient rows exist only on the column kernel.
static int fused_backward_runs(const void *plan, const void *grad_rows, int64_t grad_row_stride, const void *depth,
                               const void *context, void *grad_depth, void *grad_context, bool nchw, bool col_args,
                               int dtype, int batch, int num_cams, int depth_bins, int feat_h, int feat_w, int channels,
                               int X, int Y, void *stream) {
  int rc = check_frustum_dims(batch, num_cams, depth_bins, feat_h, feat_w, X, Y);
  if (rc) return rc;
  if (dtype != BEVPOOL_F32) return BEVPOOL_E_DTYPE;
  if (!g8_supported(channels)) return BEVPOOL_E_CHANNELS;
  if (!plan || !grad_rows || !depth || !context || !grad_depth || !grad_context) return BEVPOOL_E_ARG;
  if (grad_row_stride < channels || (grad_row_stride % 4) != 0) return BEVPOOL_E_ARG;
  if (!aligned16(grad_rows) || !aligned16(context) || !aligned16(grad_context)) return BEVPOOL_E_ALIGN;
  if ((nchw || col_args) && ((feat_w % 4) != 0 || !aligned16(depth) || !aligned16(grad_depth))) return BEVPOOL_E_ALIGN;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const PlanView pv = plan_view(plan, batch, (int64_t)num_cams * depth_bins * feat_h * feat_w, X, Y);
  const float *dp = static_cast<const float *>(depth);
  float *gd = static_cast<float *>(grad_depth);
  const bool strided = grad_row_stride != channels;
  if (g8_enabled()) {
    static const int which = env_int("BEVPOOL_BW_KERNEL", 2);
    if ((which == 2 || nchw || strided) && fused_backward_col_supported(channels, feat_w, dp, gd, pv.cell_of_point))
      return launch_fused_backward_col(pv.cell_of_point, pv.pair_rec, static_cast<const float *>(grad_rows), dp,
                                       static_cast<const float *>(context), gd, static_cast<float *>(grad_context), nchw,
                                       batch, num_cams, depth_bins, feat_h, feat_w, channels, (int64_t)X * Y, s,
                                       grad_row_stride);
    if (strided) return BEVPOOL_E_ALIGN;
  }
  if (nchw) return BEVPOOL_E_CHANNELS;
  return fused_backward_t<float>(plan, grad_rows, depth, context, grad_depth, grad_context, batch, num_cams, depth_bins,
                                 feat_h, feat_w, channels, X, Y, s);
}

extern "C" int bevpool_fused_backward_runs(const void *plan, const void *grad_out_nhwc, const void *depth,
                                           const void *context, void *grad_depth, void *grad_context,
                                           int context_is_nchw, int dtype, int batch, int num_cams, int depth_bins,
                                           int feat_h, int feat_w, int channels, int X, int Y, void *stream) {
  return fused_backward_runs(plan, grad_out_nhwc, channels, depth, context, grad_depth, grad_context, context_is_nchw != 0,
                             false, dtype, batch, num_cams, depth_bins, feat_h, feat_w, channels, X, Y, stream);
}

// gradient rows inside a wider channels-last buffer (the gradient of a concatenated BEV feature map)
extern "C" int bevpool_fused_backward_runs_from(const void *plan, const void *grad_rows, int64_t grad_row_stride,
                                                const void *depth, const void *context, void *grad_depth,
                                                void *grad_context, int context_is_nchw, int dtype, int batch,
                                                int num_cams, int depth_bins, int feat_h, int feat_w, int channels,
                                                int X, int Y, void *stream) {
  return fused_backward_runs(plan, grad_rows, grad_row_stride, depth, context, grad_depth, grad_context,
                             context_is_nchw != 0, true, dtype, batch, num_cams, depth_bins, feat_h, feat_w, channels, X,
                             Y, stream);
}

extern "C" int bevpool_grad_rows(const void *plan, const void *grad_out_nchw, void *rows_nhwc, int dtype,
                                 int batch, int64_t num_points, int channels, int X, int Y, void *stream) {
  int rc = check_plan_dims(batch, num_points, X, Y);
  if (rc) return rc;
  if (!plan || !grad_out_nchw || !rows_nhwc || channels <= 0) return BEVPOOL_E_ARG;
  if (batch > 65535) return BEVPOOL_E_RANGE;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const PlanView pv = plan_view(plan, batch, num_points, X, Y);
  const int64_t G = (int64_t)X * Y;
  const dim3 grid((unsigned)ceil_div64(G, 32 * kGrTilesPerCta), (unsigned)batch);
  static const int use_tma = env_int("BEVPOOL_GRAD_ROWS_TMA", 1);
  if (dtype == BEVPOOL_F32 && use_tma && g8_supported(channels) && (X % 4) == 0 && aligned16(grad_out_nchw) &&
      aligned16(rows_nhwc)) {
    CUtensorMap gmap{};
    const uint64_t dims[4] = {(uint64_t)X, (uint64_t)Y, (uint64_t)channels, (uint64_t)batch};
    const uint64_t strides[3] = {(uint64_t)X * 4, (uint64_t)G * 4, (uint64_t)channels * G * 4};
    const uint32_t box[4] = {kGtCells, 1, (uint32_t)channels, 1};
    if ((rc = make_tensor_map_f32(&gmap, grad_out_nchw, 4, dims, strides, box))) return rc;
    const int tiles_x = (int)ceil_div64(X, kGtCells);
    const int64_t tiles = (int64_t)batch * Y * tiles_x;
    const int per_sm_cap = (int)((size_t)220 * 1024 / ((size_t)2 * kGtStages * channels * kGtCells * 4 + 2048));
    const int per_sm = per_sm_cap < 1 ? 1 : (per_sm_cap > 8 ? 8 : per_sm_cap);
    int64_t ctas = (int64_t)sm_count() * per_sm;
    ctas = ctas > tiles ? tiles : ctas;
    const int64_t list_len = ceil_div64(tiles, ctas);
    const size_t smem = (size_t)2 * kGtStages * channels * kGtCells * 4 + kGtStages * 8 + (size_t)list_len * 4 + 16;
    cudaError_t le = cudaSuccess;
#define BEVPOOL_GT_LAUNCH(CC)                                                                                          \
    do {                                                                                                               \
      if (smem > 48 * 1024)                                                                                            \
        BEVPOOL_RETURN_IF_CUDA(cudaFuncSetAttribute(grad_rows_tma_kernel<CC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
      le = launch_pdl(grad_rows_tma_kernel<CC>, dim3((unsigned)ctas), dim3(kGtThreads), smem, s, gmap, pv.cell_start,  \
                      static_cast<float *>(rows_nhwc), X, Y, batch, tiles_x);                                          \
    } while (0)
    switch (channels) {
      case 32: BEVPOOL_GT_LAUNCH(32); break;
      case 64: BEVPOOL_GT_LAUNCH(64); break;
      case 80: BEVPOOL_GT_LAUNCH(80); break;
      case 96: BEVPOOL_GT_LAUNCH(96); break;
      case 128: BEVPOOL_GT_LAUNCH(128); break;
      default: return BEVPOOL_E_CHANNELS;
    }
#undef BEVPOOL_GT_LAUNCH
    BEVPOOL_RETURN_IF_CUDA(le);
  } else if (dtype == BEVPOOL_F32) {
    const size_t smem = (size_t)32 * (channels + 1) * 4;
    if (smem > 48 * 1024)
      BEVPOOL_RETURN_IF_CUDA(cudaFuncSetAttribute(grad_rows_kernel<uint32_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    BEVPOOL_RETURN_IF_CUDA(launch_pdl(grad_rows_kernel<uint32_t>, grid, dim3(256), smem, s, pv.cell_start,
                                      static_cast<const uint32_t *>(grad_out_nchw), static_cast<uint32_t *>(rows_nhwc), G, channels));
  } else if (dtype == BEVPOOL_F16 || dtype == BEVPOOL_BF16) {
    const size_t smem = (size_t)32 * (channels + 1) * 2;
    grad_rows_kernel<uint16_t><<<grid, 256, smem, s>>>(pv.cell_start, static_cast<const uint16_t *>(grad_out_nchw),
                                                      static_cast<uint16_t *>(rows_nhwc), G, channels);
  } else {
    return BEVPOOL_E_DTYPE;
  }
  BEVPOOL_LAUNCH_CHECK();
  return BEVPOOL_OK;
}

extern "C" int bevpool_transpose(const void *in, void *out, int dtype, int batch, int64_t rows,
                                 int64_t cols, void *stream) {
  if (!in || !out || batch <= 0 || rows <= 0 || cols <= 0) return BEVPOOL_E_ARG;
  if (batch > 65535 || ceil_div64(rows, 32) > 65535) return BEVPOOL_E_RANGE;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const dim3 grid((unsigned)ceil_div64(cols, 32), (unsigned)ceil_div64(rows, 32), (unsigned)batch);
  if (dtype == BEVPOOL_F32) {
    BEVPOOL_RETURN_IF_CUDA(launch_pdl(transpose_kernel<float>, grid, dim3(256), 0, s, static_cast<const float *>(in),
                                      static_cast<float *>(out), rows, cols));
  } else if (dtype == BEVPOOL_F16 || dtype == BEVPOOL_BF16) {
    transpose_kernel<uint16_t><<<grid, 256, 0, s>>>(static_cast<const uint16_t *>(in), static_cast<uint16_t *>(out), rows, cols);
  } else {
    return BEVPOOL_E_DTYPE;
  }
  BEVPOOL_LAUNCH_CHECK();
  return BEVPOOL_OK;
}


// ==== the reference's own native entry point =========================================================================
// ops/voxel_pooling/src/voxel_pooling_forward.cpp:21-22 declares, and :34 calls,
//   void voxel_pooling_forward_kernel_launcher(int batch_size, int num_points, int num_channels, int num_voxel_x,
//        int num_voxel_y, int num_voxel_z, const int *geom_xyz, const float *input_features,
//        float *output_features, int *pos_memo, cudaStream_t stream);
// (defined at voxel_pooling_forward_cuda.cu:38-56).  Exporting the same C++ symbol lets the reference's extension
// link against this library instead of its own .cu with no source change.  One call = plan + pos_memo + forward.
// The signature has no workspace argument, so the scratch buffers come from the stream-ordered allocator
// (cudaMallocAsync / cudaFreeAsync: no synchronisation, capturable) -- the one place the library allocates.
// Differences from the reference launcher: every cell of output_features is WRITTEN (the reference accumulates into
// a buffer the caller pre-zeroes: identical result for the reference's caller, voxel_pooling.py:37-38), every row of
// pos_memo is written ((b, y, x) or -1; the reference leaves the caller's -1 prefill), and a CUDA error is returned
// / printed instead of exit(-1) (voxel_pooling_forward_cuda.cu:52-55).
extern "C" int bevpool_voxel_pooling_forward_launcher(int batch_size, int num_points, int num_channels, int num_voxel_x,
                                                      int num_voxel_y, int num_voxel_z, const int *geom_xyz,
                                                      const float *input_features, float *output_features, int *pos_memo,
                                                      void *stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  size_t plan_bytes = 0, temp_bytes = 0, ws_bytes = 0;
  int rc = bevpool_plan_sizes(batch_size, num_points, num_voxel_x, num_voxel_y, &plan_bytes, &temp_bytes);
  if (rc) return rc;
  if ((rc = bevpool_forward_workspace_bytes(num_channels, &ws_bytes))) return rc;
  const size_t a_plan = 0, a_temp = align_up(plan_bytes, 256), a_ws = a_temp + align_up(temp_bytes, 256);
  char *scratch = nullptr;
  BEVPOOL_RETURN_IF_CUDA(cudaMallocAsync(reinterpret_cast<void **>(&scratch), a_ws + align_up(ws_bytes, 256), stream));
  rc = bevpool_plan_build(geom_xyz, batch_size, num_points, num_voxel_x, num_voxel_y, num_voxel_z, scratch + a_plan,
                          scratch + a_temp, stream);
  if (!rc && pos_memo) rc = bevpool_plan_pos_memo(scratch + a_plan, batch_size, num_points, num_voxel_x, num_voxel_y, pos_memo, stream);
  if (!rc) rc = bevpool_forward(scratch + a_plan, input_features, output_features, BEVPOOL_F32, batch_size, num_points,
                                num_channels, num_voxel_x, num_voxel_y, scratch + a_ws, stream);
  const cudaError_t fe = cudaFreeAsync(scratch, stream);
  return rc ? rc : (int)fe;
}

void voxel_pooling_forward_kernel_launcher(int batch_size, int num_points, int num_channels, int num_voxel_x,
                                           int num_voxel_y, int num_voxel_z, const int *geom_xyz,
                                           const float *input_features, float *output_features, int *pos_memo,
                                           cudaStream_t stream) {
  const int rc = bevpool_voxel_pooling_forward_launcher(batch_size, num_points, num_channels, num_voxel_x, num_voxel_y,
                                                        num_voxel_z, geom_xyz, input_features, output_features, pos_memo, stream);
  if (rc) std::fprintf(stderr, "libbevpool_sm100: voxel_pooling_forward_kernel_launcher failed: %s (code %d)\n",
                       bevpool_error_string(rc), rc);
}

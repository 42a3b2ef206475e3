// Fused lift-splat backward, column kernel (sm_100a, fp32, g8 channel counts).
//
//   grad_depth[d, pix]   = < grad_out[cell(d, pix), :], context[pix, :] >
//   grad_context[pix, :] = sum_d depth[d, pix] * grad_out[cell(d, pix), :]
// (the gradient of layers/backbones/lss_fpn.py:441-464 + ops/voxel_pooling/voxel_pooling.py:58-69 of the
// reference, without the (B, N, D, H, W, C) tensor).  Pixel-centric, no sort, no atomics, every sum in
// ascending-d order (bit-stable).
//
// Why a second kernel (ncu of fused_backward_tile_kernel, profiles/r01zz_ncu_kernels.txt): that kernel is
// bound by instruction issue and dependent-instruction latency, not by HBM -- 81 M warp instructions per 32
// frames of which 12 M are FFMA2, 117 registers, 24 % occupancy.  A lane there owns ONE pixel x C/4 channels, so
// every gradient-row quarter it reads from shared memory (5 LDS.128) feeds only 20 FFMA2, the per-bin
// bookkeeping (scalar fetches, find-first-set walk, shuffle reduction) is paid per 8 pixels, and every chunk
// starts with 8 ballots + 8 shuffles per thread to find the primary cells.  Here
//  * the per-pair bookkeeping comes from the PLAN: one 16-byte pair record per (bin, column) -- primary cell,
//    mask of the rows in it, mask of kept rows elsewhere (common.cuh) -- instead of 16 rows of cell_of_point and
//    a vote; the staging threads only transpose the depths;
//  * warp = one image column x all 16 rows; lane = (4 consecutive rows, channel eighth): a gradient-row
//    eighth (2 LDS.128 + 1 LDS.64 at C = 80, the same addresses for the four row groups = one wavefront
//    each) feeds 40 FFMA2, and the depths arrive transposed ([bin][column][row]: one LDS.128 per lane);
//  * the cross-lane half of the dot products is taken out of the FMA loop: a lane parks its four partial
//    sums in shared memory (one STS.128 per bin) and, once per 4 bins, the warp sums them with independent
//    LDS.128 + FADD and a single exchange (phase B) -- no dependent shuffle chain per bin, so the FFMA2 of
//    consecutive bins overlap;
//  * 128-thread CTAs, 3 per SM;
//  * context is read from the caller's NCHW tensor and the context gradient written back NCHW through
//    TMA tensor maps (cp.async.bulk.tensor, boxes of 4 columns x 16 rows x C channels): the two layout
//    passes (bevpool_transpose, 15 us each per 32 frames) are gone.
// Correct for any geometry: rows of a (bin, column) that do not fall into its primary cell (tilted
// cameras, random geometry) gather their own gradient row from global memory (their cell comes from
// cell_of_point).  Needs a RUN plan (pair records).
#include "common.cuh"
#include "pool_g8.cuh"
#include "tma.cuh"

#include <cstdlib>

namespace bevpool {

constexpr int kBcTW = 4;                            // image columns per CTA = warps per CTA
constexpr int kBcTH = 16;                           // image rows per CTA = one 16-row block of the plan's pair records
constexpr int kBcDC = 16;                           // depth bins per chunk
constexpr int kBcMC = 4;                            // depth bins per mini-chunk (partial dot products parked in shared memory)
constexpr int kBcThreads = 32 * kBcTW;
constexpr int kBcDepStride = kBcTW * kBcTH + 16;    // floats per bin of the transposed depth stage (+16: the two
                                                    // half-warps of a staging warp hit disjoint banks)
constexpr int kBcPartStride = 36;                   // floats per (bin, row group) of the partial-dot buffer: 8 lanes x 4
                                                    // rows + 4 of padding, so the 8 groups a quarter-warp reads differ in bank
static_assert(kBcTH == kRunHB, "the backward tile is one row block of the plan");

template <int NV2>
struct BcSmem {
  static constexpr int C = 16 * NV2;
  static constexpr size_t kRowFloats = (size_t)kBcDC * kBcTW * C;                  // one stage of gradient rows
  static constexpr size_t off_g = 0;                                                  // [2][bin][column][channel]; also the context / context-gradient TMA box
  static constexpr size_t off_dep = off_g + 2 * kRowFloats * 4;                       // float4 [2][bin][row]   (4 columns), as copied
  static constexpr size_t off_rec = off_dep + 2 * kBcDC * kBcTH * 16;                 // int4   [2][bin][column] pair records
  static constexpr size_t off_depT = off_rec + 2 * kBcDC * kBcTW * 16;                // float  [2][bin][kBcDepStride], masked + transposed
  static constexpr size_t off_part = off_depT + 2 * kBcDC * kBcDepStride * 4;         // float  [warp][bin of mini-chunk][row group][kBcPartStride]
  static constexpr size_t off_res = off_part + kBcTW * kBcMC * 4 * kBcPartStride * 4; // float  [bin][kBcDepStride] = [bin][column][row]: grad_depth of the chunk
  static constexpr size_t off_mask = off_res + kBcDC * kBcDepStride * 4;              // uint32 [2][bin][column]: the records' row masks, copied by prep
  static constexpr size_t off_bar = off_mask + 2 * kBcDC * kBcTW * 4;
  static constexpr size_t bytes = off_bar + 16;
};

__device__ __forceinline__ uint32_t opaque_u32(uint32_t v) {
  asm volatile("" : "+r"(v));
  return v;
}
__device__ __forceinline__ float4 lds_f4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ float2 lds_f2(uint32_t addr) {
  float2 v;
  asm volatile("ld.shared.v2.f32 {%0,%1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(addr));
  return v;
}
__device__ __forceinline__ void sts_f4(uint32_t addr, float4 v) {
  asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

// one pixel row of a 16-bit context in the g8 layout (channels of g8_channel), widened to fp32 / rounded from fp32
template <int NV2, typename TC>
__device__ __forceinline__ void g8_load_row_half(const TC *row, int l8, float (&v)[2 * NV2]) {
  constexpr int NF4 = NV2 / 2, NF2 = NV2 & 1;
#pragma unroll
  for (int k = 0; k < NF4; ++k) {
    const uint2 u = __ldg(reinterpret_cast<const uint2 *>(row + 32 * k + 4 * l8));
    const float2 a = CtxType<TC>::to_float2(u.x), b = CtxType<TC>::to_float2(u.y);
    v[4 * k + 0] = a.x; v[4 * k + 1] = a.y; v[4 * k + 2] = b.x; v[4 * k + 3] = b.y;
  }
  if (NF2) {
    const float2 a = CtxType<TC>::to_float2(__ldg(reinterpret_cast<const unsigned *>(row + 32 * NF4 + 2 * l8)));
    v[4 * NF4 + 0] = a.x; v[4 * NF4 + 1] = a.y;
  }
}
template <int NV2, typename TC>
__device__ __forceinline__ void g8_store_row_half(TC *row, int l8, const float (&v)[2 * NV2]) {
  constexpr int NF4 = NV2 / 2, NF2 = NV2 & 1;
#pragma unroll
  for (int k = 0; k < NF4; ++k)
    *reinterpret_cast<uint2 *>(row + 32 * k + 4 * l8) =
        make_uint2(CtxType<TC>::from_float2(v[4 * k], v[4 * k + 1]), CtxType<TC>::from_float2(v[4 * k + 2], v[4 * k + 3]));
  if (NF2) *reinterpret_cast<uint32_t *>(row + 32 * NF4 + 2 * l8) = CtxType<TC>::from_float2(v[4 * NF4], v[4 * NF4 + 1]);
}

// TC: element type of context and grad_context (fp32, or fp16 / bf16 under autocast).  A 16-bit context is widened to
// fp32 where it is loaded and the fp32 context gradient is rounded once where it is stored, so grad_depth and
// grad_context equal the fp32 kernel's on context.float(), the latter rounded to TC.  The NCHW box of a 16-bit context
// is 8 columns wide (a tensor-map box row is at least 16 bytes), of which the CTA uses its 4; its gradient leaves in
// 8-byte stores (4 columns of one channel row), which no 4-column tensor-map box could write.
template <int NV2, bool kNchw, bool kStaticBins, typename TC = float>
__global__ void __launch_bounds__(kBcThreads, (NV2 <= 5 ? 3 : 2))
fused_backward_col_kernel(const __grid_constant__ CUtensorMap ctx_map, const __grid_constant__ CUtensorMap gctx_map,
                          const int32_t *__restrict__ cell_of_point, const int4 *__restrict__ pair_rec,
                          const float *__restrict__ grad_rows, const float *__restrict__ depth,
                          const TC *__restrict__ ctx_nhwc, float *__restrict__ grad_depth,
                          TC *__restrict__ grad_ctx_nhwc, int num_cams, int D, int H, int W,
                          int64_t cells_per_sample, int tiles_h, int tiles_w, int64_t g_stride) {
  pdl_wait();
  pdl_trigger();
  using S = BcSmem<NV2>;
  constexpr int C = S::C, C4 = C / 4, NREG = 2 * NV2;
  constexpr unsigned kFull = 0xffffffffu;
  constexpr int kRowFloats = (int)S::kRowFloats;
  extern __shared__ __align__(128) unsigned char s_raw[];
  float *s_g = reinterpret_cast<float *>(s_raw + S::off_g);
  float4 (*s_dep)[kBcDC][kBcTH] = reinterpret_cast<float4 (*)[kBcDC][kBcTH]>(s_raw + S::off_dep);
  int4 (*s_rec)[kBcDC][kBcTW] = reinterpret_cast<int4 (*)[kBcDC][kBcTW]>(s_raw + S::off_rec);
  float *s_depT = reinterpret_cast<float *>(s_raw + S::off_depT);
  float *s_part = reinterpret_cast<float *>(s_raw + S::off_part);
  float *s_res = reinterpret_cast<float *>(s_raw + S::off_res);
  uint32_t *s_mask = reinterpret_cast<uint32_t *>(s_raw + S::off_mask);
  uint64_t *s_bar = reinterpret_cast<uint64_t *>(s_raw + S::off_bar);

  constexpr int kBoxW = 16 / (int)sizeof(TC);                       // columns of the NCHW context box
  const int tid = threadIdx.x, lane = tid & 31, wl = tid >> 5;      // warp = image column of the tile
  const int l8 = lane & 7, rg = lane >> 3;                          // lane = (rows 4*rg .. 4*rg+3, channel eighth)
  int bid = blockIdx.x;
  const int th = bid % tiles_h; bid /= tiles_h;
  const int tw = bid % tiles_w;
  const int bn = bid / tiles_w;
  const int h0 = th * kBcTH, w0 = tw * kBcTW;
  const int HW = H * W;
  const int64_t img_base = (int64_t)bn * D * HW;
  const float *gbase = grad_rows + (int64_t)(bn / num_cams) * cells_per_sample * g_stride;   // rows may sit in a wider buffer
  const int nchunks = (D + kBcDC - 1) / kBcDC;
  // pair records of this tile: index (((bn * D + d) * tiles_h + th) * W + w0 + column)
  const int4 *rec_base = pair_rec + ((int64_t)bn * D * tiles_h + th) * W + w0;
  const int64_t rec_bin_stride = (int64_t)tiles_h * W;

  // ---- context tile: TMA box [channel][row][4 columns] of the NCHW tensor (rows beyond H read as zeros)
  if (kNchw) {
    if (tid == 0) {
      mbar_init(s_bar, 1);
      fence_proxy_async();
    }
    __syncthreads();
    if (tid == 0) {
      mbar_expect_tx(s_bar, (uint32_t)(kBcTH * C * 16));                   // box rows are 16 bytes
      tma_load_4d(s_g, &ctx_map, sizeof(TC) == 4 ? w0 : (w0 & ~(kBoxW - 1)), h0, 0, bn, s_bar);
    }
  }

  // staging role: a half-warp = the 16 rows of one bin; a thread stages bins sd and sd + 8.  Threads 0..63 also
  // fetch the chunk's 16 x 4 pair records.
  const int sh = tid & 15, sd = tid >> 4;
  const bool srow = h0 + sh < H;
  const int64_t sbase = img_base + (int64_t)(h0 + sh) * W + w0;

  auto issue_meta = [&](int c) {             // depth segments + pair records of chunk c -> stage c & 1
    if (c < nchunks) {
#pragma unroll
      for (int pass = 0; pass < 2; ++pass) {
        const int bin = sd + 8 * pass, d = c * kBcDC + bin;
        float4 *dd = &s_dep[c & 1][bin][sh];
        if (srow && d < D) cp_async16(dd, depth + sbase + (int64_t)d * HW);
        else *dd = make_float4(0.f, 0.f, 0.f, 0.f);
      }
      if (tid < kBcDC * kBcTW) {
        const int bin = tid >> 2, col = tid & 3, d = c * kBcDC + bin;
        int4 *dr = &s_rec[c & 1][bin][col];
        if (d < D && w0 + col < W) cp_async16(dr, rec_base + (int64_t)d * rec_bin_stride + col);
        else *dr = make_int4(-1, 0, -1, 0);
      }
    }
    cp_async_commit();
  };
  // depths of chunk c transposed to [bin][column][row], zero for rows outside the pair's primary cell, and the row
  // masks copied out of the record stage (which the copies of chunk c + 2 overwrite while chunk c is being reduced);
  // returns whether this thread saw a kept pair
  auto prep = [&](int c) -> int {
    if (c >= nchunks) return 0;
    const int st = c & 1;
    int any = 0;
    if (tid < kBcDC * kBcTW) s_mask[st * kBcDC * kBcTW + tid] = (uint32_t)s_rec[st][tid >> 2][tid & 3].y;
#pragma unroll
    for (int pass = 0; pass < 2; ++pass) {
      const int bin = sd + 8 * pass;
      const float4 pd = s_dep[st][bin][sh];
      const int m0 = s_rec[st][bin][0].y, m1 = s_rec[st][bin][1].y, m2 = s_rec[st][bin][2].y, m3 = s_rec[st][bin][3].y;
      float *dT = s_depT + (st * kBcDC + bin) * kBcDepStride + sh;
      dT[0 * kBcTH] = (m0 >> sh) & 1 ? pd.x : 0.f;
      dT[1 * kBcTH] = (m1 >> sh) & 1 ? pd.y : 0.f;
      dT[2 * kBcTH] = (m2 >> sh) & 1 ? pd.z : 0.f;
      dT[3 * kBcTH] = (m3 >> sh) & 1 ? pd.w : 0.f;
      any |= (m0 | m1 | m2 | m3);
    }
    return any;
  };
  // gradient rows of chunk c's primary cells -> row stage c & 1.  Thread = (row slot tid >> 3 of 16, eighth tid & 7):
  // for each of its 4 rows (slot, slot + 16, ...) the float4s eighth, eighth + 8, eighth + 16 of the row (< C/4).
  auto issue_rows = [&](int c, int live) {
    if (c < nchunks && live) {
      const int4 *recs = &s_rec[c & 1][0][0];
      float *dst0 = s_g + (c & 1) * kRowFloats;
      const int rs = tid >> 3, e8 = tid & 7;
#pragma unroll
      for (int k = 0; k < kBcDC * kBcTW / 16; ++k) {
        const int row = rs + 16 * k;
        const int cell = recs[row].x;
        if (cell >= 0) {
          const float4 *src = reinterpret_cast<const float4 *>(gbase + (int64_t)cell * g_stride) + e8;
          float4 *dst = reinterpret_cast<float4 *>(dst0 + row * C) + e8;
#pragma unroll
          for (int v = 0; v < (C4 + 7) / 8; ++v)
            if (e8 + 8 * v < C4) cp_async16(dst + 8 * v, src + 8 * v);
        }
      }
    }
    cp_async_commit();
  };

  issue_meta(0);
  issue_meta(1);

  // ---- this lane's context rows: 4 pixels (rows 4*rg + j of column wl) x NREG channels
  float cx[4][NREG], gacc[4][NREG];
#pragma unroll
  for (int j = 0; j < 4; ++j)
#pragma unroll
    for (int r = 0; r < NREG; ++r) cx[j][r] = gacc[j][r] = 0.f;
  if (kNchw) {
    mbar_wait(s_bar, 0);
    const TC *box = reinterpret_cast<const TC *>(s_g);
    const int col = (sizeof(TC) == 4 ? 0 : (w0 & (kBoxW - 1))) + wl;
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int r = 0; r < NREG; ++r) cx[j][r] = CtxType<TC>::to_float(box[(g8_channel<NV2>(r, l8) * kBcTH + 4 * rg + j) * kBoxW + col]);
  } else {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int h = h0 + 4 * rg + j;
      if (h < H && w0 + wl < W) {
        if constexpr (sizeof(TC) == 4)
          g8_load_row<NV2, true>(reinterpret_cast<const char *>(ctx_nhwc + ((int64_t)bn * HW + h * W + w0 + wl) * C), l8, cx[j]);
        else
          g8_load_row_half<NV2, TC>(ctx_nhwc + ((int64_t)bn * HW + h * W + w0 + wl) * C, l8, cx[j]);
      }
    }
  }
  for (int i = tid; i < kBcDC * kBcDepStride; i += kBcThreads) s_res[i] = 0.f;

  cp_async_wait_1();
  __syncthreads();                           // meta(0) visible; the context box is no longer needed
  prep(0);
  issue_rows(0, 1);

  float *part_w = s_part + wl * (kBcMC * 4 * kBcPartStride);          // this warp's partial-dot buffer
  for (int c = 0; c < nchunks; ++c) {
    // in flight here: meta(c+1), rows(c)
    cp_async_wait_all();
    __syncthreads();
    prep(c + 1);                             // (its outputs are read after the next iteration's barrier)
    issue_rows(c + 1, 1);
    issue_meta(c + 2);                       // into the stage prep(c) consumed an iteration ago

    {
      const int st = c & 1;
      // masks of the chunk's 16 bins for this warp's column: lane b holds bin b's
      const uint32_t m_lane = lane < kBcDC ? s_mask[(st * kBcDC + lane) * kBcTW + wl] : 0u;
      uint32_t live = __ballot_sync(kFull, m_lane != 0u);
      if (live) {                                                     // warp-uniform
        // ONE copy of the loop body walks the kept bins (accumulators stay in place across the back edge); the
        // operands of the next kept bin are fetched from shared memory before the current bin's 40 FFMA2 are issued.
        // Every 4 bins (and at the end) phase B turns the parked partial sums into grad_depth values.
        // Shared-memory operands are addressed through two per-lane byte addresses kept opaque to the compiler
        // (it otherwise re-derives them from the thread index inside the loop to save registers).
        const uint32_t g_addr = opaque_u32(smem_u32(s_g + st * kRowFloats + wl * C) + 16u * l8);
        const uint32_t g_addr2 = opaque_u32(smem_u32(s_g + st * kRowFloats + wl * C + 32 * (NV2 / 2)) + 8u * l8);
        const uint32_t d_addr = opaque_u32(smem_u32(s_depT + st * kBcDC * kBcDepStride + wl * kBcTH + 4 * rg));
        const uint32_t p_addr = opaque_u32(smem_u32(part_w + rg * kBcPartStride + 4 * l8));
        uint32_t binpack = 0u;
        int nslot = 0;
        auto fetch = [&](int b, float (&g)[NREG], float4 &dp4) {
          const uint32_t ga = g_addr + (uint32_t)b * (kBcTW * C * 4);
#pragma unroll
          for (int k = 0; k < NV2 / 2; ++k) {
            const float4 t = lds_f4(ga + 128 * k);
            g[4 * k + 0] = t.x; g[4 * k + 1] = t.y; g[4 * k + 2] = t.z; g[4 * k + 3] = t.w;
          }
          if (NV2 & 1) {
            const float2 t = lds_f2(g_addr2 + (uint32_t)b * (kBcTW * C * 4));
            g[4 * (NV2 / 2) + 0] = t.x; g[4 * (NV2 / 2) + 1] = t.y;
          }
          dp4 = lds_f4(d_addr + (uint32_t)b * (kBcDepStride * 4));
        };
        // phase B: the parked partial sums of up to 4 bins -> grad_depth values.  `bins`: the bin of every slot, packed 4 bits
        // each; `nb`: slots in use.
        auto phase_b = [&](uint32_t bins, int nb) {
          __syncwarp();
          const int pair = lane >> 1, half = lane & 1, kk = pair >> 2, prg = pair & 3;
          const int bq = (int)((bins >> (4 * kk)) & 0xfu);
          const uint32_t mq = __shfl_sync(kFull, m_lane, bq);
          const float4 *pp = reinterpret_cast<const float4 *>(part_w + pair * kBcPartStride + 16 * half);
          const float4 p0 = pp[0], p1 = pp[1], p2 = pp[2], p3 = pp[3];
          float4 t;
          t.x = (p0.x + p1.x) + (p2.x + p3.x);
          t.y = (p0.y + p1.y) + (p2.y + p3.y);
          t.z = (p0.z + p1.z) + (p2.z + p3.z);
          t.w = (p0.w + p1.w) + (p2.w + p3.w);
          t.x += __shfl_xor_sync(kFull, t.x, 1);
          t.y += __shfl_xor_sync(kFull, t.y, 1);
          t.z += __shfl_xor_sync(kFull, t.z, 1);
          t.w += __shfl_xor_sync(kFull, t.w, 1);
          if (half == 0 && kk < nb && (mq & 0xffffu)) {            // (a slot of a dead bin holds stale sums: never stored)
            const uint32_t keep = (mq >> (4 * prg)) & 0xfu;         // rows of this group lying in the bin's primary cell
            t.x = (keep & 1u) ? t.x : 0.f;
            t.y = (keep & 2u) ? t.y : 0.f;
            t.z = (keep & 4u) ? t.z : 0.f;
            t.w = (keep & 8u) ? t.w : 0.f;
            *reinterpret_cast<float4 *>(s_res + bq * kBcDepStride + wl * kBcTH + 4 * prg) = t;
          }
          __syncwarp();
        };
        // body: reduce bin b into partial-sum slot `slot`.  Branch-free over the rows: dot products of rows outside the
        // primary cell are computed and never stored, and their staged depth is 0, so their accumulators receive +-0
        // (exact for finite gradients).
        auto body = [&](int slot, const float (&g)[NREG], const float4 &dp4) {
          const float dp[4] = {dp4.x, dp4.y, dp4.z, dp4.w};
          float sv[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            float2 da = make_float2(0.f, 0.f);                      // (one chain per row: the four rows interleave)
#pragma unroll
            for (int r = 0; r < NREG; r += 2)
              da = __ffma2_rn(make_float2(g[r], g[r + 1]), make_float2(cx[j][r], cx[j][r + 1]), da);
            axpy_row<NREG>(gacc[j], dp[j], g);
            sv[j] = da.x + da.y;
          }
          sts_f4(p_addr + (uint32_t)slot * (4 * kBcPartStride * 4), make_float4(sv[0], sv[1], sv[2], sv[3]));
        };
        const uint32_t slow_bins = __ballot_sync(kFull, (m_lane >> 16) != 0u);
        float ga[NREG], gb[NREG];
        float4 da4, db4;
        if constexpr (kStaticBins) {
          // All 16 bins of the chunk in program order, dead ones skipped by a warp-uniform branch: every shared-memory
          // address is base + immediate, a bin's partial-sum slot is (bin & 3), phase B runs after bins 3, 7, 11, 15 --
          // no find-first-set chain, address arithmetic or slot bookkeeping per bin (the searching loop below spends 47
          // instructions per bin beside its 40 FFMA2, and its FLO -> IMAD -> LDS chain shows up in the stall samples).
          if (live & 1u) fetch(0, ga, da4);
#pragma unroll
          for (int b = 0; b < kBcDC; ++b) {
            if (b + 1 < kBcDC && ((live >> (b + 1)) & 1u)) {
              if (b & 1) fetch(b + 1, ga, da4); else fetch(b + 1, gb, db4);
            }
            if ((live >> b) & 1u) {
              if (b & 1) body(b & 3, gb, db4); else body(b & 3, ga, da4);
            }
            if ((b & 3) == 3 && ((live >> (b - 3)) & 0xfu))
              phase_b((uint32_t)(b - 3) | ((uint32_t)(b - 2) << 4) | ((uint32_t)(b - 1) << 8) | ((uint32_t)b << 12), 4);
          }
        } else {
          int ba = __ffs(live) - 1, bb = ba;
          live &= live - 1u;
          fetch(ba, ga, da4);
          while (true) {                                                // warp-uniform; two roles, no register rotation
            const bool more_a = live != 0u;
            if (more_a) {
              bb = __ffs(live) - 1;
              live &= live - 1u;
              fetch(bb, gb, db4);
            }
            body(nslot, ga, da4);
            binpack |= (uint32_t)ba << (4 * nslot);
            ++nslot;
            if (nslot == kBcMC || !more_a) { phase_b(binpack, nslot); binpack = 0u; nslot = 0; }
            if (!more_a) break;
            const bool more_b = live != 0u;
            if (more_b) {
              ba = __ffs(live) - 1;
              live &= live - 1u;
              fetch(ba, ga, da4);
            }
            body(nslot, gb, db4);
            binpack |= (uint32_t)bb << (4 * nslot);
            ++nslot;
            if (nslot == kBcMC || !more_b) { phase_b(binpack, nslot); binpack = 0u; nslot = 0; }
            if (!more_b) break;
          }
        }
        // ---- kept rows outside their pair's primary cell (tilted cameras, random geometry; none for a level
        // camera): every such row gathers its own gradient row from global memory.  After the loop above, so that
        // phase B's zeros for these rows are already in place.
        for (uint32_t sl = slow_bins; sl; sl &= sl - 1u) {            // warp-uniform
          const int b = __ffs(sl) - 1;
          const uint32_t slow = __shfl_sync(kFull, m_lane, b) >> 16;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            if (((slow >> j) & 0x1111u) == 0u) continue;              // warp-uniform
            const bool p = (slow >> (4 * rg + j)) & 1u;
            float dot = 0.f;
            if (p) {
              const int64_t gp = img_base + (int64_t)(c * kBcDC + b) * HW + (int64_t)(h0 + 4 * rg + j) * W + w0 + wl;
              const int cell = __ldg(cell_of_point + gp);
              const float dv = __ldg(depth + gp);
              float gs[NREG];
              g8_load_row<NV2, false>(reinterpret_cast<const char *>(gbase + (int64_t)cell * g_stride), l8, gs);
              float2 da = make_float2(0.f, 0.f);
#pragma unroll
              for (int r = 0; r < NREG; r += 2)
                da = __ffma2_rn(make_float2(gs[r], gs[r + 1]), make_float2(cx[j][r], cx[j][r + 1]), da);
              dot = da.x + da.y;
              axpy_row<NREG>(gacc[j], dv, gs);
            }
            dot += __shfl_xor_sync(kFull, dot, 4);
            dot += __shfl_xor_sync(kFull, dot, 2);
            dot += __shfl_xor_sync(kFull, dot, 1);
            if (p && l8 == 0) s_res[b * kBcDepStride + wl * kBcTH + 4 * rg + j] = dot;
          }
        }
      }
    }
    __syncthreads();
    // ---- grad_depth of the chunk: one 16-byte segment per (bin, row)
#pragma unroll
    for (int pass = 0; pass < 2; ++pass) {
      const int bin = sd + 8 * pass, d = c * kBcDC + bin;
      float *rp = s_res + bin * kBcDepStride + sh;
      if (srow && d < D)
        stg_stream_f4(reinterpret_cast<float4 *>(grad_depth + sbase + (int64_t)d * HW),
                      make_float4(rp[0], rp[kBcTH], rp[2 * kBcTH], rp[3 * kBcTH]));
      rp[0] = rp[kBcTH] = rp[2 * kBcTH] = rp[3 * kBcTH] = 0.f;
    }
  }
  cp_async_wait_all();

  // ---- context gradient
  if constexpr (kNchw && sizeof(TC) == 2) {
    __syncthreads();                         // every copy into the row stages has landed and been consumed
    TC *s_gc = reinterpret_cast<TC *>(s_g);  // [channel][row][4 columns], rounded once
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int r = 0; r < NREG; ++r) s_gc[(g8_channel<NV2>(r, l8) * kBcTH + 4 * rg + j) * kBcTW + wl] = CtxType<TC>::from_float(gacc[j][r]);
    __syncthreads();
    for (int i = tid; i < C * kBcTH; i += kBcThreads) {                // (channel, row) = (i / 16, i % 16)
      const int h = h0 + (i & (kBcTH - 1));
      if (h < H)
        *reinterpret_cast<uint2 *>(grad_ctx_nhwc + (((int64_t)bn * C + i / kBcTH) * H + h) * W + w0) =
            *reinterpret_cast<const uint2 *>(s_gc + i * kBcTW);
    }
  } else if (kNchw) {
    __syncthreads();                         // every copy into the row stages has landed and been consumed
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int r = 0; r < NREG; ++r) s_g[(g8_channel<NV2>(r, l8) * kBcTH + 4 * rg + j) * kBcTW + wl] = gacc[j][r];
    fence_proxy_async();
    __syncthreads();
    if (tid == 0) {
      tma_store_4d(&gctx_map, w0, h0, 0, bn, s_g);
      tma_store_commit();
      tma_store_wait_read();
    }
  } else {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int h = h0 + 4 * rg + j;
      if (h < H && w0 + wl < W) {
        if constexpr (sizeof(TC) == 4)
          g8_store_row<NV2>(reinterpret_cast<char *>(grad_ctx_nhwc + ((int64_t)bn * HW + h * W + w0 + wl) * C), l8, gacc[j]);
        else
          g8_store_row_half<NV2, TC>(grad_ctx_nhwc + ((int64_t)bn * HW + h * W + w0 + wl) * C, l8, gacc[j]);
      }
    }
  }
}

template <int NV2, bool kNchw, bool kStaticBins, typename TC = float>
static int launch_bc(const CUtensorMap &ctx_map, const CUtensorMap &gctx_map, const int32_t *cell_of_point,
                     const int4 *pair_rec, const float *grad_rows, const float *depth, const void *ctx, float *grad_depth,
                     void *grad_ctx, int num_cams, int D, int H, int W, int64_t cells_per_sample, int64_t ctas,
                     int tiles_h, int tiles_w, int64_t g_stride, cudaStream_t s) {
  constexpr size_t smem = BcSmem<NV2>::bytes;
  const TC *ctx_nhwc = static_cast<const TC *>(ctx);
  TC *grad_ctx_nhwc = static_cast<TC *>(grad_ctx);
  BEVPOOL_RETURN_IF_CUDA(cudaFuncSetAttribute(fused_backward_col_kernel<NV2, kNchw, kStaticBins, TC>,
                                              cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  BEVPOOL_RETURN_IF_CUDA(launch_pdl(fused_backward_col_kernel<NV2, kNchw, kStaticBins, TC>, dim3((unsigned)ctas), dim3(kBcThreads), smem, s,
                                    ctx_map, gctx_map, cell_of_point, pair_rec, grad_rows, depth, ctx_nhwc, grad_depth, grad_ctx_nhwc,
                                    num_cams, D, H, W, cells_per_sample, tiles_h, tiles_w, g_stride));
  BEVPOOL_LAUNCH_CHECK();
  return BEVPOOL_OK;
}

bool fused_backward_col_supported(int C, int W, const void *depth, const void *grad_depth, const void *cell_of_point) {
  return g8_supported(C) && (W % 4 == 0) && aligned16(depth) && aligned16(grad_depth) && aligned16(cell_of_point);
}

// context / grad_context: NCHW (B*N, C, H, W) when `nchw`, else pixel rows (B*N, H, W, C); elements of ctx_dtype.  A 16-bit
// context always takes the static-bins loop: both loops give the same bits.
int launch_fused_backward_col(const int32_t *cell_of_point, const int4 *pair_rec, const float *grad_rows, const float *depth,
                              const void *ctx, float *grad_depth, void *grad_ctx, bool nchw, int batch, int num_cams,
                              int D, int H, int W, int C, int64_t cells_per_sample, cudaStream_t s, int64_t grad_row_stride,
                              int ctx_dtype) {
  if (grad_row_stride <= 0) grad_row_stride = C;
  const int64_t tiles_h = ceil_div64(H, kBcTH), tiles_w = ceil_div64(W, kBcTW);
  const int64_t ctas = (int64_t)batch * num_cams * tiles_h * tiles_w;
  if (ctas >= (int64_t)INT32_MAX) return BEVPOOL_E_RANGE;
  CUtensorMap ctx_map{}, gctx_map{};
  if (ctx_dtype != BEVPOOL_F32) {
    const bool f16 = ctx_dtype == BEVPOOL_F16;
    if (nchw) {
      const uint64_t dims[4] = {(uint64_t)W, (uint64_t)H, (uint64_t)C, (uint64_t)batch * num_cams};
      const uint64_t strides[3] = {(uint64_t)W * 2, (uint64_t)H * W * 2, (uint64_t)C * H * W * 2};
      const uint32_t box[4] = {8, kBcTH, (uint32_t)C, 1};
      const int rc = make_tensor_map(&ctx_map, f16 ? CtxType<__half>::kMap : CtxType<__nv_bfloat16>::kMap, ctx, 4, dims, strides, box);
      if (rc) return rc;
    }
    int rc = BEVPOOL_OK;
#define BEVPOOL_BC_ARGS ctx_map, gctx_map, cell_of_point, pair_rec, grad_rows, depth, ctx, grad_depth, grad_ctx, num_cams, D, H, W, \
                        cells_per_sample, ctas, (int)tiles_h, (int)tiles_w, grad_row_stride, s
    if (f16 && nchw) { BEVPOOL_G8_DISPATCH(C, (rc = launch_bc<NV2, true, true, __half>(BEVPOOL_BC_ARGS))); }
    else if (f16) { BEVPOOL_G8_DISPATCH(C, (rc = launch_bc<NV2, false, true, __half>(BEVPOOL_BC_ARGS))); }
    else if (nchw) { BEVPOOL_G8_DISPATCH(C, (rc = launch_bc<NV2, true, true, __nv_bfloat16>(BEVPOOL_BC_ARGS))); }
    else { BEVPOOL_G8_DISPATCH(C, (rc = launch_bc<NV2, false, true, __nv_bfloat16>(BEVPOOL_BC_ARGS))); }
#undef BEVPOOL_BC_ARGS
    return rc;
  }
  if (nchw) {
    const uint64_t dims[4] = {(uint64_t)W, (uint64_t)H, (uint64_t)C, (uint64_t)batch * num_cams};
    const uint64_t strides[3] = {(uint64_t)W * 4, (uint64_t)H * W * 4, (uint64_t)C * H * W * 4};
    const uint32_t box[4] = {kBcTW, kBcTH, (uint32_t)C, 1};
    int rc = make_tensor_map_f32(&ctx_map, ctx, 4, dims, strides, box);
    if (rc) return rc;
    if ((rc = make_tensor_map_f32(&gctx_map, grad_ctx, 4, dims, strides, box))) return rc;
  }
  int rc = BEVPOOL_OK;
#define BEVPOOL_BC_ARGS ctx_map, gctx_map, cell_of_point, pair_rec, grad_rows, depth, ctx, grad_depth, grad_ctx, num_cams, D, H, W, \
                        cells_per_sample, ctas, (int)tiles_h, (int)tiles_w, grad_row_stride, s
  static const bool static_bins = [] { const char *e = std::getenv("BEVPOOL_BW_STATIC"); return !(e && e[0] == '0'); }();
  if (static_bins) {
    if (nchw) { BEVPOOL_G8_DISPATCH(C, (rc = launch_bc<NV2, true, true>(BEVPOOL_BC_ARGS))); }
    else { BEVPOOL_G8_DISPATCH(C, (rc = launch_bc<NV2, false, true>(BEVPOOL_BC_ARGS))); }
  } else {
    if (nchw) { BEVPOOL_G8_DISPATCH(C, (rc = launch_bc<NV2, true, false>(BEVPOOL_BC_ARGS))); }
    else { BEVPOOL_G8_DISPATCH(C, (rc = launch_bc<NV2, false, false>(BEVPOOL_BC_ARGS))); }
  }
#undef BEVPOOL_BC_ARGS
  return rc;
}

}  // namespace bevpool

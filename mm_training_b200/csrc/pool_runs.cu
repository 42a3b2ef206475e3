// Fused lift-splat forward on a RUN plan (sm_100a, fp32, g8 channel layout).
//
// Replaces the materialised outer product + scatter of layers/backbones/lss_fpn.py:441-464 and
// ops/voxel_pooling/src/voxel_pooling_forward_cuda.cu:30-34.  A run (common.cuh) is a set of
// vertically adjacent frustum points -- same image, depth bin and column -- that land in the same BEV
// cell; for a level camera that is every kept point of a (depth bin, column) pair (11 points per run at
// the aiMotive shape).  Two stages, no atomics, every sum in a fixed order (bit-stable):
//
//   A  frustum_reduce_kernel   run_rows[slot] = sum_h depth[d, h, w] * context[h, w, :]
//        pixel-centric: a CTA owns (image, 4 columns x 16 rows, 32 depth bins); its 64 context rows sit
//        in shared memory (staged once, coalesced) and every depth (x) context product reads them from
//        there -- the forward issues NO data-dependent global gather at all.
//        The context tile arrives by TMA bulk copies (cp.async.bulk + mbarrier, one elected thread), and
//        the empty BEV cells (80 % of the grid) are zero-filled by TMA bulk stores from a zeroed
//        shared-memory buffer that every CTA issues for its share of the grid before it starts
//        reducing: the DRAM-write-bound fill runs in the copy engine behind the issue-bound reduction.
//   B  pool_forward_share_kernel<kIdent>   out[cell] = sum of the cell's run rows (contiguous: the slot
//        order IS the cell order) -- the even-share segmented reduction of pool_g8.cuh over 11x fewer
//        entries; every output row written exactly once.
//
// The point-sorted kernel this replaces gathered one 320-byte context row per kept point through L2
// (1.5 GB per 32 frames, L2->SM fabric bound); here the only per-run traffic is one row written and
// read back through L2 (11x fewer rows), processed a few frames at a time so it never leaves L2.
#include "common.cuh"
#include "pool_g8.cuh"
#include "tma.cuh"

namespace bevpool {

constexpr int kRaTW = 4;                     // image columns per CTA = warps per CTA = one 16-byte depth segment
constexpr int kRaDC = 16;                    // depth bins per staged chunk: 4 groups x 4 bins per warp
constexpr int kRaStages = 3;                 // chunks of (depth, records) in shared memory: one reduced, two in flight
constexpr int kRaThreads = 32 * kRaTW;
constexpr int kRaZeroCells = 32;             // cells covered by the zeroed shared-memory buffer
constexpr int kRaDepStride = kRaTW * kRunHB + 8;    // floats per bin of the transposed depth stage: the four groups of a warp read
                                                    // bins grp, grp + 4, ... -> 16-byte segments 8 banks apart, no conflicts

template <int NV2>
struct RaSmem {
  static constexpr int C = 16 * NV2;
  static constexpr size_t off_ctx = 0;                                                   // float [row][column][channel]
  static constexpr size_t off_dep = off_ctx + (size_t)kRunHB * kRaTW * C * 4;            // float4 [stage][bin][row] (4 columns), as copied
  static constexpr size_t off_rec = off_dep + (size_t)kRaStages * kRaDC * kRunHB * 16;   // int4 [stage][bin][column] pair records
  static constexpr size_t off_depT = off_rec + (size_t)kRaStages * kRaDC * kRaTW * 16;   // float [bin][kRaDepStride]: masked, [column][row]
  static constexpr size_t off_zero = off_depT + (size_t)kRaDC * kRaDepStride * 4;        // kRaZeroCells * C zeros
  static constexpr size_t off_bar = off_zero + (size_t)kRaZeroCells * C * 4;
  static constexpr size_t bytes = off_bar + 16;
};

// In-place layout change of a TMA box of the NCHW context tensor, [channel][16 rows][16 bytes of columns], into fp32
// pixel rows [row][column][channel], through registers (all threads read, barrier, all threads write).  Element e of
// the thread walks the channels fastest with the row rotated by the channel, so the transposed writes are
// conflict-free and the fp32 reads 4-way conflicted at worst (once per CTA: ~1 % of its lifetime).  A box row is
// 16 bytes (the tensor-map minimum): the CTA's 4 columns for fp32; for fp16 / bf16 the 8 columns from w0 & ~7, of
// which the CTA's 4 are converted.
template <int C, typename TC>
__device__ __forceinline__ void nchw_box_to_rows(float *s_ctx, int tid, int w0) {
  constexpr int kElems = kRunHB * kRaTW * C, kPer = (kElems + kRaThreads - 1) / kRaThreads;
  constexpr int kBoxW = 16 / (int)sizeof(TC);
  const int col0 = sizeof(TC) == 4 ? 0 : (w0 & (kBoxW - 1));
  const TC *box = reinterpret_cast<const TC *>(s_ctx);
  float v[kPer];
#pragma unroll
  for (int k = 0; k < kPer; ++k) {
    const int e = k * kRaThreads + tid;
    if (e < kElems) {
      const int c = e % C, rest = e / C, w = rest & (kRaTW - 1), h = ((rest >> 2) + c) & (kRunHB - 1);
      v[k] = CtxType<TC>::to_float(box[(c * kRunHB + h) * kBoxW + col0 + w]);
    }
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < kPer; ++k) {
    const int e = k * kRaThreads + tid;
    if (e < kElems) {
      const int c = e % C, rest = e / C, w = rest & (kRaTW - 1), h = ((rest >> 2) + c) & (kRunHB - 1);
      s_ctx[(h * kRaTW + w) * C + c] = v[k];
    }
  }
  __syncthreads();
}

// fp16 / bf16 pixel rows [row][column][channel], as the bulk copies left them at the start of the tile buffer, widened
// in place to the fp32 rows the reduction reads (same index, twice the bytes); a thread moves element pairs.
template <int C, typename TC>
__device__ __forceinline__ void half_rows_to_f32(float *s_ctx, int tid) {
  constexpr int kPairs = kRunHB * kRaTW * C / 2, kPer = kPairs / kRaThreads;
  static_assert(kPairs % kRaThreads == 0, "whole pairs per thread");
  const uint32_t *src = reinterpret_cast<const uint32_t *>(s_ctx);
  float2 v[kPer];
#pragma unroll
  for (int k = 0; k < kPer; ++k) v[k] = CtxType<TC>::to_float2(src[k * kRaThreads + tid]);
  __syncthreads();
#pragma unroll
  for (int k = 0; k < kPer; ++k) reinterpret_cast<float2 *>(s_ctx)[k * kRaThreads + tid] = v[k];
  __syncthreads();
}

// ---- stage A ----------------------------------------------------------------------------------
// CTA = (image, 4 columns x one 16-row block, one of `d_split` depth ranges), walked in chunks of 16 depth bins;
// 128 threads.  warp = image column; every 8-lane group reduces FOUR (bin, column) pairs at once (bins grp + 4p), lane = channel
// eighth: one shared-memory read of a context row eighth (2 LDS.128 + 1 LDS.64 at C = 80; the four groups read the
// same addresses = one wavefront each) feeds 20 FFMA2.  Everything per-pair comes from the plan's 16-byte PAIR
// RECORD (kept-row masks, slot of the pair's run, number of runs): the kernel reads no per-point index array and
// does no voting.  The staging threads transpose the depths to [bin][column][row] and zero the rows that are not
// kept, so the reduction loop is branch-free over the rows (4 depths = one LDS.128).  Pairs holding several runs
// (tilted cameras, random geometry) take a per-row path that reads run_code from global memory.
// kLogits: `depth` holds the DepthNet LOGITS (lss_fpn.py:423 folded in): consecutive images are dep_img_stride floats
// apart (a channel slice of depth_feature needs no copy) and `stats` holds {max, 1 / sum exp(l - max)} per pixel
// (depth_stats_kernel below); the staging threads turn a logit into its probability while they transpose it.
// TC: element type of the context (fp32, or fp16 / bf16 under autocast).  A 16-bit context arrives in the first half
// of the tile buffer and is widened to fp32 rows before the first chunk is reduced (exactly: every fp16 / bf16 value
// is an fp32 value), so the reduction and its summation order are those of the fp32 kernel.
// TO: element type of `out`, which this stage only zero-fills: fp32, or uint16_t for an fp16 / bf16 output (a zero
// has the same bits in both).  The run rows stay fp32.
template <int NV2, bool kNchw, bool kLogits = false, typename TC = float, typename TO = float>
__global__ void __launch_bounds__(kRaThreads, 4)
frustum_reduce_kernel(const __grid_constant__ CUtensorMap ctx_map, const int32_t *__restrict__ run_code,
                      const int4 *__restrict__ pair_rec, const float *__restrict__ depth,
                      const TC *__restrict__ ctx_nhwc, float *__restrict__ run_rows,
                      const int32_t *__restrict__ cell_start, TO *__restrict__ out, int32_t *__restrict__ status,
                      int img0, int64_t cell_base, int64_t num_cells, int D, int H, int W, int d_split, int d_per_cta,
                      int tiles_h, int tiles_w, int64_t capacity, int vec, int fill, int hints, int64_t out_stride,
                      int64_t dep_img_stride, const float2 *__restrict__ stats) {
  pdl_wait();
  pdl_trigger();
  using S = RaSmem<NV2>;
  constexpr int C = 16 * NV2, NREG = 2 * NV2;
  constexpr unsigned kFull = 0xffffffffu;
  extern __shared__ __align__(128) unsigned char s_raw[];
  float *s_ctx = reinterpret_cast<float *>(s_raw + S::off_ctx);
  float4 (*s_dep)[kRaDC][kRunHB] = reinterpret_cast<float4 (*)[kRaDC][kRunHB]>(s_raw + S::off_dep);
  int4 (*s_rec)[kRaDC][kRaTW] = reinterpret_cast<int4 (*)[kRaDC][kRaTW]>(s_raw + S::off_rec);
  float *s_depT = reinterpret_cast<float *>(s_raw + S::off_depT);
  float *s_zero = reinterpret_cast<float *>(s_raw + S::off_zero);
  uint64_t *s_bar = reinterpret_cast<uint64_t *>(s_raw + S::off_bar);
  const int tid = threadIdx.x, lane = tid & 31, l8 = lane & 7, grp = lane >> 3, wl = tid >> 5;
  int bid = blockIdx.x;
  const int ts = bid % d_split; bid /= d_split;
  const int th = bid % tiles_h; bid /= tiles_h;
  const int tw = bid % tiles_w;
  const int bn = img0 + bid / tiles_w;
  const int h0 = th * kRunHB, w0 = tw * kRaTW;
  const int d_begin = ts * d_per_cta, d_end = min(D, d_begin + d_per_cta);
  const int HW = H * W;
  const int rows_here = min(kRunHB, H - h0), cols_here = min(kRaTW, W - w0);

  // ---- context tile by TMA.  Pixel rows (B*N, H, W, C): one bulk copy per image row (cols_here * C contiguous
  // floats).  NCHW (the reference's layout, lss_fpn.py:441-443): ONE tensor-map box of 4 columns x 16 rows x C
  // channels, landing as [channel][row][column] and turned into pixel rows in place below (rows beyond H arrive
  // as zeros).
  if (tid == 0) {
    mbar_init(s_bar, 1);
    fence_proxy_async();
  }
  if (fill) {
    for (int i = tid; i < kRaZeroCells * C / 4; i += kRaThreads) reinterpret_cast<float4 *>(s_zero)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  if (!kNchw && (rows_here < kRunHB || cols_here < kRaTW)) {       // ragged tile: rows / columns the copies do not cover read as zeros
    for (int i = tid; i < kRunHB * kRaTW * C / 4; i += kRaThreads) reinterpret_cast<float4 *>(s_ctx)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  fence_proxy_async();
  __syncthreads();
  if (tid == 0) {
    if (kNchw) {
      mbar_expect_tx(s_bar, (uint32_t)(kRunHB * C * 16));                  // box rows are 16 bytes
      tma_load_4d(s_ctx, &ctx_map, sizeof(TC) == 4 ? w0 : (w0 & ~(16 / (int)sizeof(TC) - 1)), h0, 0, bn, s_bar);
    } else {
      const uint32_t row_bytes = (uint32_t)(cols_here * C * sizeof(TC));
      mbar_expect_tx(s_bar, row_bytes * rows_here);
      for (int r = 0; r < rows_here; ++r)
        tma_load_1d(reinterpret_cast<TC *>(s_ctx) + r * (kRaTW * C), ctx_nhwc + (((int64_t)bn * H + h0 + r) * W + w0) * C, row_bytes, s_bar);
    }
  }

  // staging role: a half-warp = the 16 rows of one bin; a thread stages bins sd and sd + 8.  Threads 0..63 also
  // fetch the chunk's 16 x 4 pair records.
  const int sh = tid & 15, sd = tid >> 4;
  const bool srow = h0 + sh < H;
  const int64_t sbase = (int64_t)bn * dep_img_stride + (int64_t)(h0 + sh) * W + w0;
  float smax[4] = {0.f, 0.f, 0.f, 0.f}, srcp[4] = {0.f, 0.f, 0.f, 0.f};     // kLogits: softmax statistics of this thread's 4 pixels
  if (kLogits && srow) {
#pragma unroll
    for (int c = 0; c < 4; ++c)
      if (w0 + c < W) {
        const float2 st = __ldg(stats + (int64_t)bn * HW + (int64_t)(h0 + sh) * W + w0 + c);
        smax[c] = st.x;
        srcp[c] = st.y;
      }
  }
  const int nchunks = (d_end - d_begin + kRaDC - 1) / kRaDC;
  const int4 *rec_base = pair_rec + ((int64_t)bn * D * tiles_h + th) * W + w0;
  const int64_t rec_bin_stride = (int64_t)tiles_h * W;

  auto issue_chunk = [&](int cidx) {         // depth segments + pair records of chunk cidx -> stage cidx % 3
    if (cidx < nchunks) {
      const int st = cidx % kRaStages;
#pragma unroll
      for (int pass = 0; pass < 2; ++pass) {
        const int bin = sd + 8 * pass, d = d_begin + cidx * kRaDC + bin;
        float4 *dd = &s_dep[st][bin][sh];
        if (srow && d < d_end) {
          const int64_t gp = sbase + (int64_t)d * HW;
          if (vec) {
            cp_async16(dd, depth + gp);
          } else {
            float4 pd = make_float4(0.f, 0.f, 0.f, 0.f);
            if (w0 + 0 < W) pd.x = __ldg(depth + gp + 0);
            if (w0 + 1 < W) pd.y = __ldg(depth + gp + 1);
            if (w0 + 2 < W) pd.z = __ldg(depth + gp + 2);
            if (w0 + 3 < W) pd.w = __ldg(depth + gp + 3);
            *dd = pd;
          }
        } else {
          *dd = make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
      if (tid < kRaDC * kRaTW) {
        const int bin = tid >> 2, col = tid & 3, d = d_begin + cidx * kRaDC + bin;
        int4 *dr = &s_rec[st][bin][col];
        if (d < d_end && w0 + col < W) cp_async16(dr, rec_base + (int64_t)d * rec_bin_stride + col);
        else *dr = make_int4(-1, 0, -1, 0);
      }
    }
    cp_async_commit();
  };

  const int64_t slot0 = __ldg(cell_start + cell_base);
  const float *ctx_col = s_ctx + wl * C;
  const uint64_t pol_rows = l2_policy_evict_last();
  auto store_run = [&](int64_t slot, const float (&acc)[NREG]) {
    if (slot >= 0 && slot < capacity) {
      if (hints) g8_store_row_hint<NV2>(run_rows + slot * C, l8, acc, pol_rows);
      else g8_store_row_plain<NV2>(run_rows + slot * C, l8, acc);
    } else if (slot >= capacity && l8 == 0) {
      *status = kPlanStatusRowOverflow;      // the caller's run_rows scratch is smaller than the run count (stale max_runs hint)
    }
  };

  issue_chunk(0);
  issue_chunk(1);

  // ---- zero-fill of this CTA's share of the empty BEV cells (after the first chunks' copies are in flight, so
  // that its own dependent loads overlap with them).  A block of 32 cells that is entirely empty (most of the
  // grid) is ONE 10-KB TMA bulk store from the zero buffer; a mixed block is written with ordinary 16-byte stores
  // (many small bulk copies would serialise in the copy engine and delay the context tiles queued behind them).
  // A warp takes every 4th block of the CTA's share; the cell_start entries of up to 4 of its blocks are fetched
  // before the first is examined.
  bool issued_bulk = false;
  if (fill) {
    constexpr int kWarps = kRaThreads / 32, C4 = C / 4, kAhead = 4;
    const int64_t blocks = (num_cells + kRaZeroCells - 1) / kRaZeroCells;
    const int64_t per_cta = (blocks + gridDim.x - 1) / gridDim.x;
    const int64_t blk_begin = (int64_t)blockIdx.x * per_cta, blk_end = min(blocks, blk_begin + per_cta);
    for (int64_t blk0 = blk_begin + wl; blk0 < blk_end; blk0 += kWarps * kAhead) {
      int cs[kAhead], ce[kAhead];
#pragma unroll
      for (int a = 0; a < kAhead; ++a) {
        const int64_t blk = blk0 + (int64_t)a * kWarps;
        cs[a] = ce[a] = 0;
        if (blk < blk_end) {
          const int64_t off = blk * kRaZeroCells;
          const int ncell = (int)min((int64_t)kRaZeroCells, num_cells - off);
          cs[a] = __ldg(cell_start + cell_base + off + min(lane, ncell));
          ce[a] = __ldg(cell_start + cell_base + off + min(lane + 1, ncell));
        }
      }
#pragma unroll
      for (int a = 0; a < kAhead; ++a) {
        const int64_t blk = blk0 + (int64_t)a * kWarps;
        if (blk >= blk_end) break;                           // warp-uniform
        const int64_t off = blk * kRaZeroCells;
        const int ncell = (int)min((int64_t)kRaZeroCells, num_cells - off);
        const int64_t c0 = cell_base + off;
        const unsigned em = __ballot_sync(kFull, lane < ncell && ce[a] == cs[a]);
        if (ncell == kRaZeroCells && em == kFull && out_stride == C) {
          if (lane == 0) {
            if (hints) tma_store_1d_hint(out + c0 * C, s_zero, kRaZeroCells * C * sizeof(TO), l2_policy_evict_first());
            else tma_store_1d(out + c0 * C, s_zero, kRaZeroCells * C * sizeof(TO));
            issued_bulk = true;
          }
        } else if (em) {
          if (out_stride == C) {
#pragma unroll 4
            for (int i = lane; i < ncell * C4; i += 32)
              if ((em >> (i / C4)) & 1u) st_zero4(out + c0 * C, i);
          } else {                                           // rows inside a wider (concatenated) buffer: C elements every out_stride
#pragma unroll 4
            for (int i = lane; i < ncell * C4; i += 32)
              if ((em >> (i / C4)) & 1u) st_zero4(out + (c0 + i / C4) * out_stride, i % C4);
          }
        }
      }
    }
    if (issued_bulk) tma_store_commit();
  }

  bool ctx_ready = false;
  for (int cidx = 0; cidx < nchunks; ++cidx) {
    asm volatile("cp.async.wait_group 1;" ::: "memory");   // chunk cidx has landed (cidx + 1 may still be in flight)
    __syncthreads();                                        // ... for every thread; and chunk cidx - 1 is fully reduced
    issue_chunk(cidx + 2);                                  // into the stage chunk cidx - 1 just left
    const int st = cidx % kRaStages;
    // depths of the chunk transposed to [bin][column][row], zero for rows that are not kept
#pragma unroll
    for (int pass = 0; pass < 2; ++pass) {
      const int bin = sd + 8 * pass;
      float4 pd = s_dep[st][bin][sh];
      if (kLogits) {                                         // softmax(l) = exp(l - max) * (1 / sum); rows / bins beyond the tensor are masked below
        pd.x = expf(pd.x - smax[0]) * srcp[0];
        pd.y = expf(pd.y - smax[1]) * srcp[1];
        pd.z = expf(pd.z - smax[2]) * srcp[2];
        pd.w = expf(pd.w - smax[3]) * srcp[3];
      }
      const unsigned m0 = (unsigned)s_rec[st][bin][0].y, m1 = (unsigned)s_rec[st][bin][1].y;
      const unsigned m2 = (unsigned)s_rec[st][bin][2].y, m3 = (unsigned)s_rec[st][bin][3].y;
      float *dT = s_depT + bin * kRaDepStride + sh;
      dT[0 * kRunHB] = ((m0 | (m0 >> 16)) >> sh) & 1u ? pd.x : 0.f;
      dT[1 * kRunHB] = ((m1 | (m1 >> 16)) >> sh) & 1u ? pd.y : 0.f;
      dT[2 * kRunHB] = ((m2 | (m2 >> 16)) >> sh) & 1u ? pd.z : 0.f;
      dT[3 * kRunHB] = ((m3 | (m3 >> 16)) >> sh) & 1u ? pd.w : 0.f;
    }
    if (!ctx_ready) {                                       // first chunk: the context tile must have landed
      mbar_wait(s_bar, 0);
      ctx_ready = true;
      if constexpr (kNchw) nchw_box_to_rows<C, TC>(s_ctx, tid, w0);
      else if constexpr (sizeof(TC) == 2) half_rows_to_f32<C, TC>(s_ctx, tid);
    }
    __syncthreads();                                        // transposed depths visible

    // this group's four pairs: bins grp, grp + 4, grp + 8, grp + 12 of column wl
    int4 rec[4];
    unsigned km[4];
#pragma unroll
    for (int p = 0; p < 4; ++p) {
      rec[p] = s_rec[st][grp + 4 * p][wl];
      km[p] = ((unsigned)rec[p].y | ((unsigned)rec[p].y >> 16)) & 0xffffu;
    }
    unsigned any = km[0] | km[1] | km[2] | km[3];
    any |= __shfl_xor_sync(kFull, any, 8);
    any |= __shfl_xor_sync(kFull, any, 16);
    if (any == 0u) continue;                                // warp-uniform: nothing kept in this column's 16 bins
    const bool single = rec[0].w <= 1 && rec[1].w <= 1 && rec[2].w <= 1 && rec[3].w <= 1;
    const float *dT = s_depT + grp * kRaDepStride + wl * kRunHB;       // pair p: + 4 * p * kRaDepStride
    if (__all_sync(kFull, single)) {
      // fast path (level camera): one run per pair.  Branch-free over the rows: the depth of a row that is not kept is 0.
      float acc[4][NREG];
#pragma unroll
      for (int p = 0; p < 4; ++p)
#pragma unroll
        for (int r = 0; r < NREG; ++r) acc[p][r] = 0.f;
#pragma unroll
      for (int k = 0; k < kRunHB / 4; ++k) {
        if (((any >> (4 * k)) & 0xfu) == 0u) continue;      // warp-uniform
        float4 dp[4];
#pragma unroll
        for (int p = 0; p < 4; ++p) dp[p] = *reinterpret_cast<const float4 *>(dT + 4 * p * kRaDepStride + 4 * k);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int h = 4 * k + j;
          if (!((any >> h) & 1u)) continue;                 // warp-uniform
          float v[NREG];
          g8_lds_row<NV2>(ctx_col + h * (kRaTW * C), l8, v);
#pragma unroll
          for (int p = 0; p < 4; ++p)
            axpy_row<NREG>(acc[p], j == 0 ? dp[p].x : (j == 1 ? dp[p].y : (j == 2 ? dp[p].z : dp[p].w)), v);
        }
      }
#pragma unroll
      for (int p = 0; p < 4; ++p)
        if (km[p]) store_run((int64_t)rec[p].z - slot0, acc[p]);
    } else {
      // general geometry: several runs per pair; walk the rows of one pair at a time with the run boundaries
      // from run_code (first row of a run: its slot; continuation: kRunCont)
#pragma unroll 1
      for (int p = 0; p < 4; ++p) {
        unsigned kmp = km[p];
        unsigned any_p = kmp | __shfl_xor_sync(kFull, kmp, 8);
        any_p |= __shfl_xor_sync(kFull, any_p, 16);
        if (any_p == 0u) continue;                          // warp-uniform
        const int d = d_begin + cidx * kRaDC + grp + 4 * p;
        const int64_t gp0 = (int64_t)bn * D * HW + (int64_t)d * HW + (int64_t)h0 * W + w0 + wl;
        float acc[NREG];
#pragma unroll
        for (int r = 0; r < NREG; ++r) acc[r] = 0.f;
        int64_t slot = -1;
#pragma unroll
        for (int h = 0; h < kRunHB; ++h) {
          if (!((any_p >> h) & 1u)) continue;               // warp-uniform
          if ((kmp >> h) & 1u) {
            const int cv = __ldg(run_code + gp0 + (int64_t)h * W);
            const float dv = dT[4 * p * kRaDepStride + h];
            if (cv >= 0) {                                   // first row of a run
              store_run(slot, acc);
              if (slot >= 0) {
#pragma unroll
                for (int r = 0; r < NREG; ++r) acc[r] = 0.f;
              }
              slot = (int64_t)cv - slot0;
            }
            float v[NREG];
            g8_lds_row<NV2>(ctx_col + h * (kRaTW * C), l8, v);
            axpy_row<NREG>(acc, dv, v);
          }
        }
        store_run(slot, acc);
      }
    }
  }
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  if (!ctx_ready) mbar_wait(s_bar, 0);                   // (empty depth range) never leave a copy in flight
  if (issued_bulk) tma_store_wait_read();                // the zero buffer must outlive the bulk stores reading it
}

// softmax statistics per pixel: {max_d l, 1 / sum_d exp(l - max)}; thread = pixel, one streaming read of the logits
__global__ void __launch_bounds__(256)
depth_stats_kernel(const float *__restrict__ logits, int64_t img_stride, int D, int HW, float2 *__restrict__ stats) {
  const int pix = blockIdx.x * blockDim.x + threadIdx.x;
  if (pix >= HW) return;
  const float *lp = logits + (int64_t)blockIdx.y * img_stride + pix;
  float m = -INFINITY, s = 0.f;
  for (int d = 0; d < D; ++d) {
    const float l = __ldg(lp + (int64_t)d * HW);
    if (l > m) {
      s = s * expf(m - l);
      m = l;
    }
    s += (l == -INFINITY) ? 0.f : expf(l - m);             // a leading -inf (m still -inf) would add expf(NaN)
  }
  stats[(int64_t)blockIdx.y * HW + pix] = make_float2(m, 1.0f / s);
}

}  // namespace bevpool

using namespace bevpool;

template <int NV2, bool kNchw, bool kLogits = false, typename TC = float, typename TO = float>
static int launch_stage_a(const CUtensorMap &ctx_map, const PlanView &pv, const float *dp, const TC *cx, float *rr,
                          TO *out, int32_t *status, int img0, int64_t cell_base, int64_t num_cells, int nb, int num_cams,
                          int D, int H, int W, int64_t capacity, int vec, int fill, int hints, int d_split, int64_t out_stride,
                          cudaStream_t s, int64_t dep_img_stride = 0, const float2 *stats = nullptr) {
  if (dep_img_stride <= 0) dep_img_stride = (int64_t)D * H * W;
  constexpr int C = 16 * NV2;
  const int tiles_h = (int)ceil_div64(H, kRunHB), tiles_w = (int)ceil_div64(W, kRaTW);
  const int d_per_cta = (int)(ceil_div64(ceil_div64(D, d_split), kRaDC) * kRaDC);      // whole chunks per CTA
  const int splits = (int)ceil_div64(D, d_per_cta);
  const int64_t ctas = (int64_t)nb * num_cams * tiles_w * tiles_h * splits;
  if (ctas >= (int64_t)INT32_MAX) return BEVPOOL_E_RANGE;
  (void)C;
  const size_t smem = RaSmem<NV2>::bytes;
  if (smem > 48 * 1024)
    BEVPOOL_RETURN_IF_CUDA(cudaFuncSetAttribute(frustum_reduce_kernel<NV2, kNchw, kLogits, TC, TO>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  BEVPOOL_RETURN_IF_CUDA(launch_pdl_if(pdl_forward_enabled(), frustum_reduce_kernel<NV2, kNchw, kLogits, TC, TO>, dim3((unsigned)ctas), dim3(kRaThreads), smem, s,
      ctx_map, pv.run_code, pv.pair_rec, dp, cx, rr, pv.cell_start, out, status, img0, cell_base, num_cells, D, H, W, splits, d_per_cta, tiles_h,
      tiles_w, capacity, vec, fill, hints, out_stride, dep_img_stride, stats));
  BEVPOOL_LAUNCH_CHECK();
  return BEVPOOL_OK;
}

// tuning knobs, read once per process (defaults = the measured best; scripts/README.md)
struct RunKnobs {
  int chunk, fill, hints, cps_b, d_split;
};
static const RunKnobs &run_knobs() {
  static const RunKnobs k = [] {
    RunKnobs r;
    r.chunk = env_int("BEVPOOL_RUN_CHUNK", 0);            // frames per (stage A, stage B) pair; 0 = all
    r.fill = env_int("BEVPOOL_RUN_FILL", 1) != 0;         // 0: stage B fills the empty cells itself
    r.hints = env_int("BEVPOOL_RUN_HINTS", 1) != 0;       // L2 eviction-priority hints on the fill / run-row stores
    r.cps_b = env_int("BEVPOOL_RUN_CPSB", 5);             // stage B CTAs per SM (4 warps each)
    r.cps_b = r.cps_b < 1 ? 1 : (r.cps_b > kFwMaxCtasPerSm - 1 ? kFwMaxCtasPerSm - 1 : r.cps_b);
    r.d_split = env_int("BEVPOOL_RUN_DSPLIT", 0);
    return r;
  }();
  return k;
}

// stage A of one frame group without logits, for a context of element type TC; TO as in frustum_reduce_kernel
template <typename TC, typename TO>
static int launch_stage_a_typed(bool nchw, const CUtensorMap &ctx_map, const PlanView &pv, const float *dp, const void *cx,
                                float *rr, TO *out, int32_t *status, int img0, int64_t cell_base, int64_t num_cells, int nb,
                                int num_cams, int D, int H, int W, int C, int64_t capacity, int vec, int fill, int hints,
                                int d_split, int64_t out_stride, cudaStream_t s) {
  const TC *c = static_cast<const TC *>(cx);
  int rc = BEVPOOL_OK;
  if (nchw) {
    BEVPOOL_G8_DISPATCH(C, (rc = launch_stage_a<NV2, true, false, TC, TO>(ctx_map, pv, dp, c, rr, out, status, img0, cell_base, num_cells,
                                                                          nb, num_cams, D, H, W, capacity, vec, fill, hints, d_split,
                                                                          out_stride, s)));
  } else {
    BEVPOOL_G8_DISPATCH(C, (rc = launch_stage_a<NV2, false, false, TC, TO>(ctx_map, pv, dp, c, rr, out, status, img0, cell_base, num_cells,
                                                                           nb, num_cams, D, H, W, capacity, vec, fill, hints, d_split,
                                                                           out_stride, s)));
  }
  return rc;
}

// stage A of one frame group: every context type, and the logits variant (fp32 output only)
template <typename TO>
static int launch_stage_a_any(int ctx_dtype, bool nchw, const float2 *stats, const CUtensorMap &ctx_map, const PlanView &pv,
                              const float *dp, const void *cx, float *rr, TO *out, int32_t *status, int img0, int64_t cell_base,
                              int64_t num_cells, int nb, int num_cams, int D, int H, int W, int C, int64_t capacity, int vec,
                              int fill, int hints, int d_split, int64_t out_stride, int64_t dep_img_stride, cudaStream_t s) {
  int rc = BEVPOOL_OK;
  if (ctx_dtype == BEVPOOL_F16)
    return launch_stage_a_typed<__half>(nchw, ctx_map, pv, dp, cx, rr, out, status, img0, cell_base, num_cells, nb, num_cams, D, H,
                                        W, C, capacity, vec, fill, hints, d_split, out_stride, s);
  if (ctx_dtype == BEVPOOL_BF16)
    return launch_stage_a_typed<__nv_bfloat16>(nchw, ctx_map, pv, dp, cx, rr, out, status, img0, cell_base, num_cells, nb, num_cams,
                                               D, H, W, C, capacity, vec, fill, hints, d_split, out_stride, s);
  if constexpr (sizeof(TO) == 4) {
    if (nchw && stats) {
      BEVPOOL_G8_DISPATCH(C, (rc = launch_stage_a<NV2, true, true>(ctx_map, pv, dp, static_cast<const float *>(cx), rr, out, status, img0,
                                                                   cell_base, num_cells, nb, num_cams, D, H, W, capacity, vec, fill,
                                                                   hints, d_split, out_stride, s, dep_img_stride, stats)));
      return rc;
    }
  }
  return launch_stage_a_typed<float>(nchw, ctx_map, pv, dp, cx, rr, out, status, img0, cell_base, num_cells, nb, num_cams, D, H, W,
                                     C, capacity, vec, fill, hints, d_split, out_stride, s);
}

// stage B of one frame group: even-share segmented sum of the run rows (identity ids) into `out`, rounded once per
// element where TO is 16-bit; fill CTAs only if stage A did not fill
template <typename TO>
static int launch_stage_b(const PlanView &pv, const float *rr, TO *out, float *workspace, int64_t cell_base, int64_t ncells,
                          int C, int64_t capacity, int period_b, int cps_b, int64_t out_stride, cudaStream_t s) {
  const FastDiv one = make_fastdiv(1u);
  const unsigned ctas_b = (unsigned)(sm_count() * (period_b ? period_b : cps_b));
  const int slices = (int)(period_b ? ctas_b - ctas_b / period_b : ctas_b) * kFwWarpsPerCta * 4;
  float *ws_head = workspace;
  float *ws_tail = ws_head + (size_t)slices * C;
  cudaError_t le = cudaSuccess;
  BEVPOOL_G8_DISPATCH(C, (le = launch_pdl_if(pdl_forward_enabled(), pool_forward_share_kernel<NV2, false, 4, true, TO>, dim3(ctas_b),
                                             dim3(kFwWarpsPerCta * 32), 0, s, pv.cell_start, (const int32_t *)nullptr,
                                             pv.sorted_cells, rr, (const float *)nullptr, out, ws_head, ws_tail, cell_base,
                                             ncells, one, one, period_b, capacity, out_stride)));
  BEVPOOL_RETURN_IF_CUDA(le);
  BEVPOOL_LAUNCH_CHECK();
  BEVPOOL_G8_DISPATCH(C, (le = launch_pdl_if(pdl_forward_enabled(), pool_forward_fixup_kernel<NV2, TO>,
                                             dim3((unsigned)ceil_div64((int64_t)slices * 8, 128)), dim3(128), 0, s,
                                             pv.cell_start, pv.sorted_cells, (const float *)ws_head, (const float *)ws_tail, out,
                                             cell_base, ncells, slices, capacity, out_stride)));
  BEVPOOL_RETURN_IF_CUDA(le);
  BEVPOOL_LAUNCH_CHECK();
  return BEVPOOL_OK;
}

// ctx_dtype: element type of `context` (BEVPOOL_F32 / F16 / BF16); depth and run rows are fp32 (`dtype`); out_dtype:
// element type of the output rows (BEVPOOL_F32, or F16 / BF16: every value still computed in fp32, rounded once)
static int fused_forward_runs_impl(const void *plan, const void *depth, const void *context, bool nchw, void *out_nhwc,
                                   int dtype, int batch, int num_cams, int depth_bins, int feat_h, int feat_w,
                                   int channels, int X, int Y, void *run_rows, int64_t run_rows_capacity,
                                   void *workspace, void *stream, int64_t out_stride = 0, int64_t dep_img_stride = 0,
                                   const float2 *stats = nullptr, int64_t ctx_img_stride = 0, bool prezeroed = false,
                                   int ctx_dtype = BEVPOOL_F32, int out_dtype = BEVPOOL_F32) {
  if (ctx_img_stride <= 0) ctx_img_stride = (int64_t)channels * feat_h * feat_w;
  if (out_stride == 0) out_stride = channels;
  if (stats && !nchw) return BEVPOOL_E_ARG;                   // the logits entry point exists for the NCHW layout only
  if (dep_img_stride != 0 && ((dep_img_stride % 4) != 0 || dep_img_stride < (int64_t)depth_bins * feat_h * feat_w)) return BEVPOOL_E_ARG;
  if (out_stride < channels || (out_stride % 4) != 0) return BEVPOOL_E_ARG;
  int rc = check_frustum_dims(batch, num_cams, depth_bins, feat_h, feat_w, X, Y);
  if (rc) return rc;
  const int64_t np = (int64_t)num_cams * depth_bins * feat_h * feat_w;
  if (dtype != BEVPOOL_F32) return BEVPOOL_E_DTYPE;
  if (ctx_dtype != BEVPOOL_F32 && ctx_dtype != BEVPOOL_F16 && ctx_dtype != BEVPOOL_BF16) return BEVPOOL_E_DTYPE;
  if (out_dtype != BEVPOOL_F32 && out_dtype != BEVPOOL_F16 && out_dtype != BEVPOOL_BF16) return BEVPOOL_E_DTYPE;
  if (!g8_supported(channels)) return BEVPOOL_E_CHANNELS;
  if (!plan || !depth || !context || !out_nhwc || !run_rows || !workspace || run_rows_capacity <= 0) return BEVPOOL_E_ARG;
  if (!aligned16(context) || !aligned16(out_nhwc) || !aligned16(run_rows) || !aligned16(workspace)) return BEVPOOL_E_ALIGN;
  const int esz = ctx_dtype == BEVPOOL_F32 ? 4 : 2;
  if (nchw && (feat_w * esz) % 16 != 0) return BEVPOOL_E_ALIGN;      // the tensor-map rows must be multiples of 16 bytes
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const PlanView pv = plan_view(plan, batch, np, X, Y);
  int32_t *status = plan_status(const_cast<void *>(plan));
  const int64_t G = (int64_t)X * Y;
  const int vec = (feat_w % 4 == 0) && aligned16(depth);
  const RunKnobs &kn = run_knobs();
  int fpc = kn.chunk;
  if (fpc <= 0 || fpc > batch) fpc = batch;
  // prezeroed: the caller zero-filled the output itself (e.g. on a side stream, behind the plan build): nobody fills
  const int fill = prezeroed ? 0 : kn.fill, hints = kn.hints, cps_b = kn.cps_b;
  const float *dp = static_cast<const float *>(depth), *cx = static_cast<const float *>(context);
  float *rr = static_cast<float *>(run_rows);
  CUtensorMap ctx_map{};
  if (nchw) {
    const uint64_t dims[4] = {(uint64_t)feat_w, (uint64_t)feat_h, (uint64_t)channels, (uint64_t)batch * num_cams};
    const uint64_t strides[3] = {(uint64_t)feat_w * esz, (uint64_t)feat_h * feat_w * esz, (uint64_t)ctx_img_stride * esz};
    if (ctx_dtype == BEVPOOL_F32) {
      const uint32_t box[4] = {kRaTW, kRunHB, (uint32_t)channels, 1};
      if ((rc = make_tensor_map_f32(&ctx_map, cx, 4, dims, strides, box))) return rc;
    } else {                                                      // 16-byte box rows: 8 columns, the CTA uses 4 of them
      const uint32_t box[4] = {8, kRunHB, (uint32_t)channels, 1};
      const CUtensorMapDataType t = ctx_dtype == BEVPOOL_F16 ? CtxType<__half>::kMap : CtxType<__nv_bfloat16>::kMap;
      if ((rc = make_tensor_map(&ctx_map, t, context, 4, dims, strides, box))) return rc;
    }
  }
  for (int b0 = 0; b0 < batch; b0 += fpc) {
    const int nb = batch - b0 < fpc ? batch - b0 : fpc;
    const int64_t cell_base = (int64_t)b0 * G, ncells = (int64_t)nb * G;
    // depth ranges per tile: enough CTAs for >= ~4 waves of 4 resident CTAs per SM
    const int64_t tiles = (int64_t)nb * num_cams * ceil_div64(feat_w, kRaTW) * ceil_div64(feat_h, kRunHB);
    int d_split = kn.d_split;
    if (d_split <= 0) {
      d_split = (int)ceil_div64((int64_t)16 * sm_count(), tiles);
      const int max_split = (int)ceil_div64(depth_bins, kRaDC);
      d_split = d_split < 1 ? 1 : (d_split > max_split ? max_split : d_split);
    }
    const int img0 = b0 * num_cams;
    if (out_dtype == BEVPOOL_F32)
      rc = launch_stage_a_any(ctx_dtype, nchw, stats, ctx_map, pv, dp, context, rr, static_cast<float *>(out_nhwc), status, img0,
                              cell_base, ncells, nb, num_cams, depth_bins, feat_h, feat_w, channels, run_rows_capacity, vec, fill,
                              hints, d_split, out_stride, dep_img_stride, s);
    else
      rc = launch_stage_a_any(ctx_dtype, nchw, stats, ctx_map, pv, dp, context, rr, static_cast<uint16_t *>(out_nhwc), status, img0,
                              cell_base, ncells, nb, num_cams, depth_bins, feat_h, feat_w, channels, run_rows_capacity, vec, fill,
                              hints, d_split, out_stride, dep_img_stride, s);
    if (rc) return rc;
    const int period_b = (fill || prezeroed) ? 0 : cps_b + 1;
    float *ws = static_cast<float *>(workspace);
    if (out_dtype == BEVPOOL_F32)
      rc = launch_stage_b(pv, rr, static_cast<float *>(out_nhwc), ws, cell_base, ncells, channels, run_rows_capacity, period_b, cps_b,
                          out_stride, s);
    else if (out_dtype == BEVPOOL_F16)
      rc = launch_stage_b(pv, rr, static_cast<__half *>(out_nhwc), ws, cell_base, ncells, channels, run_rows_capacity, period_b, cps_b,
                          out_stride, s);
    else
      rc = launch_stage_b(pv, rr, static_cast<__nv_bfloat16 *>(out_nhwc), ws, cell_base, ncells, channels, run_rows_capacity, period_b,
                          cps_b, out_stride, s);
    if (rc) return rc;
  }
  return BEVPOOL_OK;
}

extern "C" int bevpool_fused_forward_runs(const void *plan, const void *depth, const void *context_nhwc,
                                          void *out_nhwc, int dtype, int batch, int num_cams, int depth_bins,
                                          int feat_h, int feat_w, int channels, int X, int Y, void *run_rows,
                                          int64_t run_rows_capacity, void *workspace, void *stream) {
  return fused_forward_runs_impl(plan, depth, context_nhwc, false, out_nhwc, dtype, batch, num_cams, depth_bins, feat_h,
                                 feat_w, channels, X, Y, run_rows, run_rows_capacity, workspace, stream);
}

extern "C" int bevpool_fused_forward_runs_nchw(const void *plan, const void *depth, const void *context_nchw,
                                               void *out_nhwc, int dtype, int batch, int num_cams, int depth_bins,
                                               int feat_h, int feat_w, int channels, int X, int Y, void *run_rows,
                                               int64_t run_rows_capacity, void *workspace, void *stream) {
  return fused_forward_runs_impl(plan, depth, context_nchw, true, out_nhwc, dtype, batch, num_cams, depth_bins, feat_h,
                                 feat_w, channels, X, Y, run_rows, run_rows_capacity, workspace, stream);
}

// Concat epilogue (models/bev_depth.py:187-189: `torch.cat([img_bev, lidar_bev], dim=1)`): the pooled rows are written
// straight into a wider channels-last buffer -- out points at the first camera channel of cell 0, consecutive cells are
// out_row_stride floats apart -- so neither lss_fpn.py:466's `.contiguous()` nor the cat copies the camera half.
extern "C" int bevpool_fused_forward_runs_into(const void *plan, const void *depth, const void *context,
                                               int context_is_nchw /* flags: bit 0 NCHW context, bit 1 output pre-zeroed */, void *out_rows, int64_t out_row_stride, int dtype,
                                               int batch, int num_cams, int depth_bins, int feat_h, int feat_w,
                                               int channels, int X, int Y, void *run_rows, int64_t run_rows_capacity,
                                               void *workspace, void *stream) {
  if (out_row_stride <= 0) return BEVPOOL_E_ARG;
  return fused_forward_runs_impl(plan, depth, context, (context_is_nchw & 1) != 0, out_rows, dtype, batch, num_cams, depth_bins,
                                 feat_h, feat_w, channels, X, Y, run_rows, run_rows_capacity, workspace, stream, out_row_stride,
                                 0, nullptr, 0, (context_is_nchw & 2) != 0);
}

// Autocast: fp32 depth (the softmax runs in fp32) with the fp16 / bf16 context slice of DepthNet's output.  The context
// is widened to fp32 where stage A loads it, so the output equals that of ..._runs_into on context.float(), bit for bit.
extern "C" int bevpool_fused_forward_runs_mixed(const void *plan, const void *depth, const void *context, int context_dtype,
                                                int flags, void *out_rows, int64_t out_row_stride, int batch, int num_cams,
                                                int depth_bins, int feat_h, int feat_w, int channels, int X, int Y,
                                                void *run_rows, int64_t run_rows_capacity, void *workspace, void *stream) {
  if (out_row_stride <= 0) return BEVPOOL_E_ARG;
  return fused_forward_runs_impl(plan, depth, context, (flags & 1) != 0, out_rows, BEVPOOL_F32, batch, num_cams, depth_bins,
                                 feat_h, feat_w, channels, X, Y, run_rows, run_rows_capacity, workspace, stream, out_row_stride,
                                 0, nullptr, 0, (flags & 2) != 0, context_dtype);
}

// 16-bit concat under autocast: ..._runs_mixed writing fp16 / bf16 rows (out_dtype).  Every value is computed in fp32 as
// there; the only rounding is the one RNE rounding of each output element where stage B stores it, so the rows equal the
// fp32 call's rows `.to(out_dtype)` bit for bit.
extern "C" int bevpool_fused_forward_runs_into16(const void *plan, const void *depth, const void *context, int context_dtype,
                                                 int flags, void *out_rows, int64_t out_row_stride, int out_dtype, int batch,
                                                 int num_cams, int depth_bins, int feat_h, int feat_w, int channels, int X, int Y,
                                                 void *run_rows, int64_t run_rows_capacity, void *workspace, void *stream) {
  if (out_row_stride <= 0) return BEVPOOL_E_ARG;
  if (out_dtype != BEVPOOL_F16 && out_dtype != BEVPOOL_BF16) return BEVPOOL_E_DTYPE;
  return fused_forward_runs_impl(plan, depth, context, (flags & 1) != 0, out_rows, BEVPOOL_F32, batch, num_cams, depth_bins,
                                 feat_h, feat_w, channels, X, Y, run_rows, run_rows_capacity, workspace, stream, out_row_stride,
                                 0, nullptr, 0, (flags & 2) != 0, context_dtype, out_dtype);
}

// lss_fpn.py:423 + :441-443 folded into the forward: the kernel reads DepthNet's output tensor itself -- depth_feature
// (B*N, feature_channels, H, W) fp32 NCHW, logits in channels [0, depth_bins), context in channels
// [context_channel_offset, context_channel_offset + channels) -- no softmax output, no channel-slice copies.
// stats: scratch of 8 * B*N * H * W bytes (softmax max / normaliser per pixel, written by a small pre-pass).
extern "C" int bevpool_fused_forward_runs_logits(const void *plan, const void *depth_feature, int feature_channels,
                                                 int context_channel_offset, void *stats, void *out_rows,
                                                 int64_t out_row_stride, int dtype, int batch, int num_cams,
                                                 int depth_bins, int feat_h, int feat_w, int channels, int X, int Y,
                                                 void *run_rows, int64_t run_rows_capacity, void *workspace,
                                                 void *stream) {
  if (!depth_feature || !stats || num_cams <= 0 || batch <= 0 || depth_bins <= 0 || feat_h <= 0 || feat_w <= 0) return BEVPOOL_E_ARG;
  if (context_channel_offset < 0 || context_channel_offset + channels > feature_channels || depth_bins > feature_channels) return BEVPOOL_E_ARG;
  if (dtype != BEVPOOL_F32) return BEVPOOL_E_DTYPE;
  if (!aligned16(depth_feature) || (feat_w % 4) != 0) return BEVPOOL_E_ALIGN;
  const int HW = feat_h * feat_w;
  const int64_t img_stride = (int64_t)feature_channels * HW;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const float *base = static_cast<const float *>(depth_feature);
  depth_stats_kernel<<<dim3((unsigned)((HW + 255) / 256), (unsigned)(batch * num_cams)), 256, 0, s>>>(
      base, img_stride, depth_bins, HW, static_cast<float2 *>(stats));
  BEVPOOL_LAUNCH_CHECK();
  return fused_forward_runs_impl(plan, base, base + (int64_t)context_channel_offset * HW, true, out_rows, dtype, batch, num_cams,
                                 depth_bins, feat_h, feat_w, channels, X, Y, run_rows, run_rows_capacity, workspace, stream,
                                 out_row_stride, img_stride, static_cast<const float2 *>(stats), img_stride);
}

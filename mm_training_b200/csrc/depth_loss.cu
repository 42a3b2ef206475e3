// Depth loss of the camera branch (sm_100a): binary cross-entropy between the depth distribution and the LiDAR depth
// labels, averaged over the foreground pixels, forward and backward.
//
// Reference being replaced (exps/mm_training_aim.py:163-176, get_depth_loss):
//   preds = depth_preds.permute(0, 2, 3, 1).contiguous().view(-1, D)          full copy of (B*N, D, H, W)
//   fg    = torch.max(labels, dim=1).values > 0.0                             a row holding a NaN is background
//   loss  = 3 * F.binary_cross_entropy(preds[fg], labels[fg], 'none').sum() / max(1.0, fg.sum())
// Two boolean gathers (nonzero: a host sync each), the host-side max(1.0, tensor), and a device assert that aborts the
// CUDA context on a NaN probability.  Here the foreground count stays on the device, so a step is graph-capturable.
//
// Layout.  The probabilities are (B*N, D, H, W): for a fixed bin, consecutive pixels are contiguous.  The dense label
// rows are (B*N*H*W, D): for a fixed pixel, consecutive bins are contiguous.  A CTA owns a TILE of 32 consecutive
// global pixels (a tile may cross an image boundary) and stages the tile's label span -- one contiguous run of 32*D
// floats -- into shared memory with coalesced loads, row r at s[r * Dp], Dp = D | 1 (odd, so the 32 lanes reading
// s[lane * Dp + d] hit 32 distinct banks).  Lane = pixel, warp w takes the bins d = w, w + 8, ...: the probability and
// gradient accesses of a warp are 32 consecutive floats of one bin.  With int32 bins (DepthLabelGenerator's
// return_bins) the tile stages 32 ints instead and a label is (d == bin); everything else is the same template, so
// one-hot labels give the same bits in both forms.
//
// Arithmetic (torch's CUDA kernels, aten/src/ATen/native/cuda/Loss.cu, in fp32, logf / log1pf, never fast intrinsics):
//   forward  e = (t - 1) * max(log1p(-p), -100) - t * max(log(p), -100)   (max keeps a NaN, like std::max)
//            the two products are rounded before the subtraction (no FMA contraction); exact for t in {0, 1}
//            pixel sum: fp32, ascending d; tile sums: fp64, in a fixed order per CTA, then over CTAs in a second
//            launch; S rounded once to fp32.  L = fl(3 * fl(S / fl(max(cnt, 1)))).  No floating-point atomics.
//   backward g' = fl(fl(g * 3) / fl(max(cnt, 1)))  (MulBackward, then DivBackward)
//            grad = +0 + g' * (p - t) / fmaxf((1 - p) * p, 1e-12)   foreground ("+0 +": index_put into zeros)
//            grad = +0                                              background
#include <algorithm>

#include "common.cuh"

namespace bevpool {

constexpr int kLossTile = 32;                          // consecutive global pixels per tile: one lane each
constexpr int kLossThreads = 256;                      // the 8 warps split the bins of a tile
constexpr int kLossWarps = kLossThreads / 32;
constexpr int kLossMaxBins = 1536;                     // 32 rows of D | 1 floats must fit in shared memory
constexpr int kLossFwdGrid = kSMs * 8;                 // persistent forward grid: one fp64 partial per CTA
constexpr int kLossBwdGrid = kSMs * 16;

inline int loss_fwd_grid(int64_t px) { return (int)std::min<int64_t>(ceil_div64(px, kLossTile), kLossFwdGrid); }
inline int loss_bwd_grid(int64_t px) { return (int)std::min<int64_t>(ceil_div64(px, kLossTile), kLossBwdGrid); }
// [sbin: kLossTile ints][flags: kLossWarps x kLossTile ints][rows: kLossTile x (D | 1) floats, if `rows`]
inline size_t loss_smem_bytes(int D, bool rows) {
  return (size_t)(kLossWarps + 1) * kLossTile * 4 + (rows ? (size_t)kLossTile * (D | 1) * 4 : 0);
}
inline size_t loss_ws_cnt_offset(int grid) { return align_up((size_t)grid * 8, 256); }

// one BCE term, torch's expression; std::max(x, -100) is (x < -100 ? -100 : x), so a NaN passes through
__device__ __forceinline__ float bce_term(float p, float t) {
  float lp = logf(p), l1 = log1pf(-p);
  lp = lp < -100.f ? -100.f : lp;
  l1 = l1 < -100.f ? -100.f : l1;
  return __fsub_rn(__fmul_rn(__fsub_rn(t, 1.f), l1), __fmul_rn(t, lp));
}

// foreground gradient element: torch's binary_cross_entropy_backward, then the accumulate of index_put into zeros
__device__ __forceinline__ float bce_grad(float p, float t, float gs) {
  const float den = fmaxf(__fmul_rn(__fsub_rn(1.f, p), p), 1e-12f);
  return __fadd_rn(0.f, __fdiv_rn(__fmul_rn(gs, __fsub_rn(p, t)), den));
}

// Stages the labels of the tile [p0, p0 + n): the dense span (n * D contiguous floats) into rows of Dp floats, or the
// n bins.  Coalesced 4-byte loads, 8 in flight per thread.
template <bool kBins>
__device__ __forceinline__ void stage_tile(const float *__restrict__ labels, const int32_t *__restrict__ bins,
                                           int64_t p0, int n, int D, FastDiv fd, float *s, int *sbin) {
  if constexpr (kBins) {
    if (threadIdx.x < n) sbin[threadIdx.x] = ldg_stream_i32(bins + p0 + threadIdx.x);
  } else {
    const int Dp = D | 1;
    const float *src = labels + p0 * D;
    const int count = n * D;
    for (int i0 = threadIdx.x; i0 < count; i0 += 8 * kLossThreads) {
      float v[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int i = i0 + j * kLossThreads;
        v[j] = i < count ? ldg_stream_f32(src + i) : 0.f;
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int i = i0 + j * kLossThreads;
        if (i < count) {
          const int r = (int)fastdiv((uint32_t)i, fd);
          s[r * Dp + (i - r * D)] = v[j];
        }
      }
    }
  }
}

template <bool kBins>
__device__ __forceinline__ float tile_label(const float *row, int bin, int d) {
  if constexpr (kBins) return d == bin ? 1.f : 0.f;
  else return row[d];
}

// grid: loss_fwd_grid(px); dynamic smem: loss_smem_bytes(D, true)
template <bool kBins>
__global__ void __launch_bounds__(kLossThreads)
depth_loss_forward_kernel(const float *__restrict__ prob, const float *__restrict__ labels,
                          const int32_t *__restrict__ bins, int64_t px, int D, int64_t HW, FastDiv fd,
                          double *__restrict__ part_sum, int *__restrict__ part_cnt) {
  extern __shared__ int smem[];
  const int Dp = D | 1;
  int *sbin = smem;                                          // [kLossTile] (bins only)
  int *flags = sbin + kLossTile;                             // [kLossWarps][kLossTile]: bit 0 t > 0, bit 1 t NaN
  float *s = reinterpret_cast<float *>(flags + kLossWarps * kLossTile);  // [kLossTile][Dp]: labels, then the terms
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t tiles = ceil_div64(px, kLossTile);
  double acc = 0.0;                                          // warp 0: this lane's pixels, in tile order
  int cnt = 0;
  for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    const int64_t p0 = tile * kLossTile;
    const int n = (int)std::min<int64_t>(kLossTile, px - p0);
    stage_tile<kBins>(labels, bins, p0, n, D, fd, s, sbin);
    __syncthreads();
    int f = 0;
    if (lane < n) {
      const int64_t r = p0 + lane, bn = r / HW;
      const float *pp = prob + bn * D * HW + (r - bn * HW);
      float *row = s + lane * Dp;
      const int bin = kBins ? sbin[lane] : 0;
#pragma unroll 2
      for (int d = warp; d < D; d += kLossWarps) {
        const float t = tile_label<kBins>(row, bin, d);
        f |= (t > 0.f ? 1 : 0) | (t != t ? 2 : 0);
        row[d] = bce_term(ldg_stream_f32(pp + (int64_t)d * HW), t);
      }
    }
    flags[warp * kLossTile + lane] = f;
    __syncthreads();
    if (warp == 0 && lane < n) {
      int fl = 0;
#pragma unroll
      for (int w = 0; w < kLossWarps; ++w) fl |= flags[w * kLossTile + lane];
      const float *row = s + lane * Dp;
      float sum = 0.f;
      for (int d = 0; d < D; ++d) sum += row[d];             // ascending d
      if (fl == 1) {                                         // max > 0 and no NaN (torch.max gives NaN)
        acc += (double)sum;
        ++cnt;
      }
    }
    __syncthreads();                                         // s, flags and sbin are reused by the next tile
  }
  if (warp == 0) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      acc += __shfl_xor_sync(0xffffffffu, acc, o);
      cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    }
    if (lane == 0) {
      part_sum[blockIdx.x] = acc;
      part_cnt[blockIdx.x] = cnt;
    }
  }
}

// one CTA: fixed-order sum of the per-CTA partials, then torch's scalar op order
__global__ void __launch_bounds__(256)
depth_loss_finalize_kernel(const double *__restrict__ part_sum, const int *__restrict__ part_cnt, int parts,
                           float *__restrict__ loss, int32_t *__restrict__ fg_count) {
  __shared__ double ss[256];
  __shared__ int sc[256];
  const int t = threadIdx.x;
  double a = 0.0;
  int c = 0;
  for (int i = t; i < parts; i += 256) {
    a += part_sum[i];
    c += part_cnt[i];
  }
  ss[t] = a;
  sc[t] = c;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (t < o) {
      ss[t] += ss[t + o];
      sc[t] += sc[t + o];
    }
    __syncthreads();
  }
  if (t == 0) {
    const int n = sc[0];
    const float S = __double2float_rn(ss[0]);
    loss[0] = __fmul_rn(__fdiv_rn(S, __int2float_rn(max(n, 1))), 3.f);
    fg_count[0] = n;
  }
}

// grid: loss_bwd_grid(px); dynamic smem: loss_smem_bytes(D, !kBins)
template <bool kBins>
__global__ void __launch_bounds__(kLossThreads)
depth_loss_backward_kernel(const float *__restrict__ prob, const float *__restrict__ labels,
                           const int32_t *__restrict__ bins, const float *__restrict__ grad_loss,
                           const int32_t *__restrict__ fg_count, int64_t px, int D, int64_t HW, FastDiv fd,
                           float *__restrict__ grad_prob) {
  extern __shared__ int smem[];
  const int Dp = D | 1;
  int *sbin = smem;
  int *flags = sbin + kLossTile;
  float *s = reinterpret_cast<float *>(flags + kLossWarps * kLossTile);  // dense labels only
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const float gs = __fdiv_rn(__fmul_rn(__ldg(grad_loss), 3.f), __int2float_rn(max(__ldg(fg_count), 1)));
  const int64_t tiles = ceil_div64(px, kLossTile);
  for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    const int64_t p0 = tile * kLossTile;
    const int n = (int)std::min<int64_t>(kLossTile, px - p0);
    stage_tile<kBins>(labels, bins, p0, n, D, fd, s, sbin);
    __syncthreads();
    const float *row = s + lane * Dp;
    const int bin = (kBins && lane < n) ? sbin[lane] : 0;
    if constexpr (!kBins) {                                  // the foreground test needs the whole row first
      int f = 0;
      if (lane < n)
        for (int d = warp; d < D; d += kLossWarps) {
          const float t = row[d];
          f |= (t > 0.f ? 1 : 0) | (t != t ? 2 : 0);
        }
      flags[warp * kLossTile + lane] = f;
      __syncthreads();
    }
    if (lane < n) {
      bool fg;
      if constexpr (kBins) {
        fg = (unsigned)bin < (unsigned)D;
      } else {
        int fl = 0;
#pragma unroll
        for (int w = 0; w < kLossWarps; ++w) fl |= flags[w * kLossTile + lane];
        fg = fl == 1;
      }
      const int64_t r = p0 + lane, bn = r / HW;
      const int64_t base = bn * D * HW + (r - bn * HW);
      const float *pp = prob + base;
      float *gp = grad_prob + base;
#pragma unroll 2
      for (int d = warp; d < D; d += kLossWarps) {
        const int64_t o = (int64_t)d * HW;
        gp[o] = fg ? bce_grad(ldg_stream_f32(pp + o), tile_label<kBins>(row, bin, d), gs) : 0.f;
      }
    }
    __syncthreads();
  }
}

inline bool aligned4(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 3u) == 0; }

inline int loss_check_dims(int num_images, int depth_bins, int feat_h, int feat_w) {
  if (num_images <= 0 || depth_bins <= 0 || feat_h <= 0 || feat_w <= 0) return BEVPOOL_E_ARG;
  if ((int64_t)num_images * feat_h * feat_w >= (int64_t)INT32_MAX) return BEVPOOL_E_RANGE;
  if (depth_bins > kLossMaxBins) return BEVPOOL_E_CHANNELS;
  return BEVPOOL_OK;
}

template <typename K>
inline int loss_smem_opt_in(K kernel, size_t smem) {
  if (smem > 48 * 1024)
    BEVPOOL_RETURN_IF_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  return BEVPOOL_OK;
}

}  // namespace bevpool

using namespace bevpool;

extern "C" int bevdepth_loss_workspace_bytes(int num_images, int depth_bins, int feat_h, int feat_w, size_t *bytes) {
  if (!bytes) return BEVPOOL_E_ARG;
  if (int rc = loss_check_dims(num_images, depth_bins, feat_h, feat_w)) return rc;
  const int grid = loss_fwd_grid((int64_t)num_images * feat_h * feat_w);
  *bytes = loss_ws_cnt_offset(grid) + (size_t)grid * 4;
  return BEVPOOL_OK;
}

extern "C" int bevdepth_loss_forward(const float *prob, const float *labels, const int32_t *bins, int num_images,
                                     int depth_bins, int feat_h, int feat_w, void *workspace, float *loss,
                                     int32_t *fg_count, void *stream) {
  if (!prob || !workspace || !loss || !fg_count || (!labels == !bins)) return BEVPOOL_E_ARG;
  if (int rc = loss_check_dims(num_images, depth_bins, feat_h, feat_w)) return rc;
  if (!aligned4(prob) || !aligned4(labels) || !aligned4(bins) || !aligned4(loss) || !aligned4(fg_count) ||
      (reinterpret_cast<uintptr_t>(workspace) & 7u))
    return BEVPOOL_E_ALIGN;
  const int64_t HW = (int64_t)feat_h * feat_w, px = (int64_t)num_images * HW;
  const int grid = loss_fwd_grid(px);
  const size_t smem = loss_smem_bytes(depth_bins, true);                 // the terms go through the rows
  const FastDiv fd = make_fastdiv((uint32_t)depth_bins);
  double *part_sum = static_cast<double *>(workspace);
  int *part_cnt = reinterpret_cast<int *>(static_cast<char *>(workspace) + loss_ws_cnt_offset(grid));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (bins) {
    if (int rc = loss_smem_opt_in(depth_loss_forward_kernel<true>, smem)) return rc;
    depth_loss_forward_kernel<true><<<grid, kLossThreads, smem, s>>>(prob, nullptr, bins, px, depth_bins, HW, fd,
                                                                     part_sum, part_cnt);
  } else {
    if (int rc = loss_smem_opt_in(depth_loss_forward_kernel<false>, smem)) return rc;
    depth_loss_forward_kernel<false><<<grid, kLossThreads, smem, s>>>(prob, labels, nullptr, px, depth_bins, HW, fd,
                                                                      part_sum, part_cnt);
  }
  BEVPOOL_LAUNCH_CHECK();
  depth_loss_finalize_kernel<<<1, 256, 0, s>>>(part_sum, part_cnt, grid, loss, fg_count);
  BEVPOOL_LAUNCH_CHECK();
  return BEVPOOL_OK;
}

extern "C" int bevdepth_loss_backward(const float *prob, const float *labels, const int32_t *bins,
                                      const float *grad_loss, const int32_t *fg_count, int num_images, int depth_bins,
                                      int feat_h, int feat_w, float *grad_prob, void *stream) {
  if (!prob || !grad_loss || !fg_count || !grad_prob || (!labels == !bins)) return BEVPOOL_E_ARG;
  if (int rc = loss_check_dims(num_images, depth_bins, feat_h, feat_w)) return rc;
  if (!aligned4(prob) || !aligned4(labels) || !aligned4(bins) || !aligned4(grad_loss) || !aligned4(fg_count) ||
      !aligned4(grad_prob))
    return BEVPOOL_E_ALIGN;
  const int64_t HW = (int64_t)feat_h * feat_w, px = (int64_t)num_images * HW;
  const int grid = loss_bwd_grid(px);
  const size_t smem = loss_smem_bytes(depth_bins, !bins);
  const FastDiv fd = make_fastdiv((uint32_t)depth_bins);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (bins) {
    if (int rc = loss_smem_opt_in(depth_loss_backward_kernel<true>, smem)) return rc;
    depth_loss_backward_kernel<true><<<grid, kLossThreads, smem, s>>>(prob, nullptr, bins, grad_loss, fg_count, px,
                                                                      depth_bins, HW, fd, grad_prob);
  } else {
    if (int rc = loss_smem_opt_in(depth_loss_backward_kernel<false>, smem)) return rc;
    depth_loss_backward_kernel<false><<<grid, kLossThreads, smem, s>>>(prob, labels, nullptr, grad_loss, fg_count, px,
                                                                       depth_bins, HW, fd, grad_prob);
  }
  BEVPOOL_LAUNCH_CHECK();
  return BEVPOOL_OK;
}

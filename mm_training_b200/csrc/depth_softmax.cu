// Depth distribution of the lift-splat camera branch in one pass (sm_100a): softmax over the D depth logits of every
// pixel and, when a LiDAR depth oracle is supplied, the overwrite of the pixels that have a LiDAR return.
//
// Reference being replaced (layers/backbones/lss_fpn.py): `depth = depth_feature[:, :D].softmax(1)` :423 and the
// oracle branch :427-434 -- max over D of the oracle, two permute + contiguous copies of (B*N, D, H, W) tensors, a
// boolean-mask index_put and a permuted view that the outer product then reads with a stride.  Here a thread owns one
// pixel; for a fixed depth bin the 32 pixels of a warp are contiguous (one 128-byte line per bin), the logits are
// streamed twice (running max + sum of exponentials, then the normalised write; the second pass hits L1/L2) and both
// outputs -- the probabilities the depth loss needs and the distribution the pooling consumes -- are written once,
// in the (B*N, D, H, W) layout the fused pooling kernels read.
//
// Backward: grad_logits = p * (g - sum_d p * g), g = grad wrt the probabilities + (pixel has no oracle ? grad wrt the
// consumed distribution : 0).
#include "common.cuh"

namespace bevpool {

template <typename T> __device__ __forceinline__ float to_f32(T v);
template <> __device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f32<__half>(__half v) { return __half2float(v); }
template <> __device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }

// grid: (ceil(HW / 256), BN)
template <typename T>
__global__ void __launch_bounds__(256)
depth_softmax_kernel(const T *__restrict__ logits, int64_t logits_img_stride, const float *__restrict__ oracle, int D,
                     int HW, float *__restrict__ prob, float *__restrict__ used) {
  const int pix = blockIdx.x * blockDim.x + threadIdx.x;
  if (pix >= HW) return;
  const int64_t bn = blockIdx.y;
  const T *lp = logits + bn * logits_img_stride + pix;
  float m = -INFINITY, s = 0.f;
  for (int d = 0; d < D; ++d) {                            // online max / sum (one streaming read)
    const float l = to_f32(lp[(int64_t)d * HW]);
    if (l > m) {
      s = s * expf(m - l);
      m = l;
    }
    s += (l == -INFINITY) ? 0.f : expf(l - m);             // a leading -inf (m still -inf) would add expf(NaN)
  }
  bool fg = false;
  const float *op = nullptr;
  if (oracle) {
    op = oracle + (bn * D) * HW + pix;
    float om = -INFINITY;
    for (int d = 0; d < D; ++d) om = fmaxf(om, __ldg(op + (int64_t)d * HW));
    fg = om > 0.0f;                                         // lss_fpn.py:428
  }
  float *pp = prob + (bn * D) * HW + pix;
  float *up = used ? used + (bn * D) * HW + pix : nullptr;
  for (int d = 0; d < D; ++d) {
    const float p = expf(to_f32(lp[(int64_t)d * HW]) - m) / s;
    pp[(int64_t)d * HW] = p;
    if (up) up[(int64_t)d * HW] = fg ? __ldg(op + (int64_t)d * HW) : p;
  }
}

template <typename T>
__global__ void __launch_bounds__(256)
depth_softmax_backward_kernel(const float *__restrict__ prob, const float *__restrict__ grad_prob,
                              const float *__restrict__ grad_used, const float *__restrict__ oracle, int D, int HW,
                              T *__restrict__ grad_logits) {
  const int pix = blockIdx.x * blockDim.x + threadIdx.x;
  if (pix >= HW) return;
  const int64_t base = ((int64_t)blockIdx.y * D) * HW + pix;
  bool fg = false;
  if (oracle && grad_used) {
    float om = -INFINITY;
    for (int d = 0; d < D; ++d) om = fmaxf(om, __ldg(oracle + base + (int64_t)d * HW));
    fg = om > 0.0f;
  }
  const bool use_u = grad_used && !fg;
  float dot = 0.f;
  for (int d = 0; d < D; ++d) {
    const int64_t o = base + (int64_t)d * HW;
    const float g = (grad_prob ? grad_prob[o] : 0.f) + (use_u ? grad_used[o] : 0.f);
    dot += prob[o] * g;
  }
  for (int d = 0; d < D; ++d) {
    const int64_t o = base + (int64_t)d * HW;
    const float g = (grad_prob ? grad_prob[o] : 0.f) + (use_u ? grad_used[o] : 0.f);
    const float v = prob[o] * (g - dot);
    if constexpr (sizeof(T) == 4) grad_logits[o] = v;
    else grad_logits[o] = T(v);
  }
}

}  // namespace bevpool

using namespace bevpool;

extern "C" int bevdepth_softmax_forward(const void *logits, int dtype, int64_t logits_image_stride, const float *oracle,
                                        int num_images, int depth_bins, int feat_h, int feat_w, float *prob, float *used,
                                        void *stream) {
  if (!logits || !prob || num_images <= 0 || depth_bins <= 0 || feat_h <= 0 || feat_w <= 0) return BEVPOOL_E_ARG;
  if (oracle && !used) return BEVPOOL_E_ARG;
  const int HW = feat_h * feat_w;
  if (logits_image_stride < (int64_t)depth_bins * HW) return BEVPOOL_E_ARG;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  dim3 grid((unsigned)((HW + 255) / 256), (unsigned)num_images);
  switch (dtype) {
    case BEVPOOL_F32:
      depth_softmax_kernel<float><<<grid, 256, 0, s>>>(static_cast<const float *>(logits), logits_image_stride, oracle, depth_bins, HW, prob, used);
      break;
    case BEVPOOL_F16:
      depth_softmax_kernel<__half><<<grid, 256, 0, s>>>(static_cast<const __half *>(logits), logits_image_stride, oracle, depth_bins, HW, prob, used);
      break;
    case BEVPOOL_BF16:
      depth_softmax_kernel<__nv_bfloat16><<<grid, 256, 0, s>>>(static_cast<const __nv_bfloat16 *>(logits), logits_image_stride, oracle, depth_bins, HW, prob, used);
      break;
    default:
      return BEVPOOL_E_DTYPE;
  }
  BEVPOOL_LAUNCH_CHECK();
  return BEVPOOL_OK;
}

extern "C" int bevdepth_softmax_backward(const float *prob, const float *grad_prob, const float *grad_used,
                                         const float *oracle, int num_images, int depth_bins, int feat_h, int feat_w,
                                         void *grad_logits, int dtype, void *stream) {
  if (!prob || !grad_logits || (!grad_prob && !grad_used) || num_images <= 0 || depth_bins <= 0 || feat_h <= 0 || feat_w <= 0)
    return BEVPOOL_E_ARG;
  const int HW = feat_h * feat_w;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  dim3 grid((unsigned)((HW + 255) / 256), (unsigned)num_images);
  switch (dtype) {
    case BEVPOOL_F32:
      depth_softmax_backward_kernel<float><<<grid, 256, 0, s>>>(prob, grad_prob, grad_used, oracle, depth_bins, HW, static_cast<float *>(grad_logits));
      break;
    case BEVPOOL_F16:
      depth_softmax_backward_kernel<__half><<<grid, 256, 0, s>>>(prob, grad_prob, grad_used, oracle, depth_bins, HW, static_cast<__half *>(grad_logits));
      break;
    case BEVPOOL_BF16:
      depth_softmax_backward_kernel<__nv_bfloat16><<<grid, 256, 0, s>>>(prob, grad_prob, grad_used, oracle, depth_bins, HW, static_cast<__nv_bfloat16 *>(grad_logits));
      break;
    default:
      return BEVPOOL_E_DTYPE;
  }
  BEVPOOL_LAUNCH_CHECK();
  return BEVPOOL_OK;
}

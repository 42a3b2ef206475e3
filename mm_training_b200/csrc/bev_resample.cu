// Nearest resampling of the LiDAR BEV into the concatenated BEV rows: F.interpolate(x, size=(dst_h, dst_w),
// mode='nearest') followed by torch.cat([camera_half, .], 1), as models/bev_depth.py prepares the LiDAR half of the
// fused BEV map -- and its adjoint.
//
// Index rule per axis (torch's compute_scales_value<float> + nearest_neighbor_compute_source_index, ATen/native/
// UpSample.h):  src(d) = min(floor(float(d) * (float(in) / float(out))), in - 1).
// src() is monotone in d, so the preimage of source index s is the interval [first(s), first(s + 1)), first(s) being
// the smallest d with src(d) >= s.  The backward finds those bounds with src() itself, so it is the exact adjoint of
// the forward also where torch's separate backward formula (nearest_neighbor_bw_compute_source_index) could differ.
//
//   forward   out[b, y, x, :]  = float(src[b, :, src_y(y), src_x(x)])            (a copy: bit-equal to the stock ops)
//   backward  gsrc[b, :, sy, sx] = sum over y in pre(sy) ascending, x in pre(sx) ascending, of g[b, y, x, :]
// The backward sums in fp32 from +0 in torch's upsample_nearest2d_backward order and rounds once to the source dtype;
// it is a gather over source cells (no atomics), every element written once (empty preimages give zeros).
//
// Two layouts of the source / its gradient:
//  * NCHW: one CTA per 32-cell x-run of one row.  Lane = cell for the global side (a warp reads / writes one channel
//    of 32 neighbouring cells), lane = channel for the row side; a padded shared tile turns one into the other.  The
//    cells of a run map to a ratio-dependent, non-uniform set of source columns, so the gather is done by the lanes
//    themselves rather than by a fixed-size tensor-map box (which would read every column of the span: 4x the bytes
//    at a 4x down-sample).
//  * channels_last: 8 lanes per row, 16-byte vectors of the destination (pool_g8.cuh's layout), converting on the way.
#include "common.cuh"

#include <math.h>

namespace bevpool {
namespace {

constexpr int kRsThreads = 256;
constexpr int kRsCells = 32;        // cells of one NCHW tile
constexpr int kRsChunk = 128;       // channels per pass through the shared tile of the NCHW kernels
constexpr int kRsVec = 2;           // float4 chunks per lane per pass of the row backward: 8 * 2 * 4 = 64 channels (no spills)

__host__ __device__ __forceinline__ int nearest_src(int d, int in, int out) {
  const float scale = (float)in / (float)out;
  const int s = (int)floorf((float)d * scale);
  return s < in - 1 ? s : in - 1;
}

// smallest d in [0, out] with nearest_src(d) >= s (out when there is none)
__host__ __device__ __forceinline__ int nearest_first_dst(int s, int in, int out) {
  if (s <= 0) return 0;
  if (s >= in) return out;
  int64_t e = ((int64_t)s * out + in - 1) / in;           // the real-arithmetic answer; float rounding moves it by a few
  int d = (int)(e > out ? out : e);
  while (d > 0 && nearest_src(d - 1, in, out) >= s) --d;
  while (d < out && nearest_src(d, in, out) < s) ++d;
  return d;
}

__device__ __forceinline__ float to_f32(float v) { return v; }
__device__ __forceinline__ float to_f32(__half v) { return __half2float(v); }
__device__ __forceinline__ float to_f32(__nv_bfloat16 v) { return __bfloat162float(v); }
template <typename E> __device__ __forceinline__ E from_f32(float v);
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ __half from_f32<__half>(float v) { return __float2half_rn(v); }
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

// 4 consecutive elements <-> float4 (16 bytes of fp32, 8 bytes of a 16-bit type)
__device__ __forceinline__ float4 load4(const float *p) { return __ldg(reinterpret_cast<const float4 *>(p)); }
template <typename E2, typename E>
__device__ __forceinline__ float4 load4_16(const E *p) {
  const uint2 u = __ldg(reinterpret_cast<const uint2 *>(p));
  const E2 a = *reinterpret_cast<const E2 *>(&u.x), b = *reinterpret_cast<const E2 *>(&u.y);
  return make_float4(to_f32(a.x), to_f32(a.y), to_f32(b.x), to_f32(b.y));
}
__device__ __forceinline__ float4 load4(const __half *p) { return load4_16<__half2>(p); }
__device__ __forceinline__ float4 load4(const __nv_bfloat16 *p) { return load4_16<__nv_bfloat162>(p); }

__device__ __forceinline__ void store4(float *p, const float4 &v) { stg_stream_f4(reinterpret_cast<float4 *>(p), v); }
template <typename E>
__device__ __forceinline__ void store4(E *p, const float4 &v) {
  E e[4] = {from_f32<E>(v.x), from_f32<E>(v.y), from_f32<E>(v.z), from_f32<E>(v.w)};
  *reinterpret_cast<uint2 *>(p) = *reinterpret_cast<const uint2 *>(e);
}

__device__ __forceinline__ void add4(float4 &a, const float4 &v) {
  a.x += v.x;
  a.y += v.y;
  a.z += v.z;
  a.w += v.w;
}

// ---- forward, NCHW source: CTA = (b, y, 32-cell x-run); every element of the run's C destination rows written once
template <typename E>
__global__ void __launch_bounds__(kRsThreads)
resize_nearest_fwd_nchw_kernel(const E *__restrict__ src, float *__restrict__ out, int64_t out_stride, int C, int Hs,
                               int Ws, int Hd, int Wd, int tiles_x) {
  pdl_wait();
  pdl_trigger();
  __shared__ float tile[kRsCells][kRsChunk + 1];          // [cell][channel]: conflict-free both ways
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int tx = (int)(blockIdx.x % tiles_x);
  const int64_t by = blockIdx.x / tiles_x;                  // b * Hd + y
  const int y = (int)(by % Hd), b = (int)(by / Hd);
  const int x0 = tx * kRsCells, ncell = min(kRsCells, Wd - x0);
  const int64_t plane = (int64_t)Hs * Ws;
  // lanes past the run's end re-read its last cell (never stored)
  const E *s = src + (int64_t)b * C * plane + (int64_t)nearest_src(y, Hs, Hd) * Ws +
               nearest_src(x0 + min(lane, ncell - 1), Ws, Wd);
  float *o = out + (by * Wd + x0) * out_stride;
  for (int c0 = 0; c0 < C; c0 += kRsChunk) {
    const int ck = min(kRsChunk, C - c0);
#pragma unroll 4
    for (int cc = warp; cc < ck; cc += kRsThreads / 32) tile[lane][cc] = to_f32(s[(int64_t)(c0 + cc) * plane]);
    __syncthreads();
    for (int j = warp; j < ncell; j += kRsThreads / 32)
      for (int cc = lane; cc < ck; cc += 32) o[(int64_t)j * out_stride + c0 + cc] = tile[j][cc];
    __syncthreads();
  }
}

// ---- forward, channels_last source: 8 lanes per destination row
template <typename E>
__global__ void __launch_bounds__(kRsThreads)
resize_nearest_fwd_rows_kernel(const E *__restrict__ src, float *__restrict__ out, int64_t out_stride, int batch, int C,
                               int Hs, int Ws, int Hd, int Wd) {
  pdl_wait();
  pdl_trigger();
  const int64_t cell = ((int64_t)blockIdx.x * kRsThreads + threadIdx.x) >> 3;
  const int l8 = threadIdx.x & 7;
  const int64_t dst_cells = (int64_t)Hd * Wd;
  if (cell >= (int64_t)batch * dst_cells) return;
  const int b = (int)(cell / dst_cells);
  const int rem = (int)(cell - (int64_t)b * dst_cells);
  const int y = rem / Wd, x = rem - y * Wd;
  const E *s = src + (((int64_t)b * Hs + nearest_src(y, Hs, Hd)) * Ws + nearest_src(x, Ws, Wd)) * C;
  float *o = out + cell * out_stride;
#pragma unroll 4
  for (int q = 4 * l8; q < C; q += 32) store4(o + q, load4(s + q));
}

// ---- backward, NCHW gradient: CTA = (b, sy, 32-cell sx-run); a warp sums the preimage rows of one source cell at a
// time (lane = channel), the tile is then written out one channel at a time (lane = cell)
template <typename E>
__global__ void __launch_bounds__(kRsThreads)
resize_nearest_bwd_nchw_kernel(const float *__restrict__ g, int64_t g_stride, E *__restrict__ gsrc, int C, int Hs,
                               int Ws, int Hd, int Wd, int tiles_x) {
  pdl_wait();
  pdl_trigger();
  __shared__ float tile[kRsCells][kRsChunk + 1];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int tx = (int)(blockIdx.x % tiles_x);
  const int64_t bs = blockIdx.x / tiles_x;                  // b * Hs + sy
  const int sy = (int)(bs % Hs), b = (int)(bs / Hs);
  const int sx0 = tx * kRsCells, ncell = min(kRsCells, Ws - sx0);
  const int y_lo = nearest_first_dst(sy, Hs, Hd), y_hi = nearest_first_dst(sy + 1, Hs, Hd);
  const float *gb = g + (int64_t)b * Hd * Wd * g_stride;
  const int64_t plane = (int64_t)Hs * Ws;
  E *o = gsrc + (int64_t)b * C * plane + (int64_t)sy * Ws + sx0;
  for (int c0 = 0; c0 < C; c0 += kRsChunk) {
    const int ck = min(kRsChunk, C - c0);
    for (int j = warp; j < ncell; j += kRsThreads / 32) {
      const int x_lo = nearest_first_dst(sx0 + j, Ws, Wd), x_hi = nearest_first_dst(sx0 + j + 1, Ws, Wd);
      float acc[kRsChunk / 32];
#pragma unroll
      for (int k = 0; k < kRsChunk / 32; ++k) acc[k] = 0.f;
      for (int y = y_lo; y < y_hi; ++y)
        for (int x = x_lo; x < x_hi; ++x) {
          const float *row = gb + ((int64_t)y * Wd + x) * g_stride + c0;
#pragma unroll
          for (int k = 0; k < kRsChunk / 32; ++k)
            if (lane + 32 * k < ck) acc[k] += __ldg(row + lane + 32 * k);
        }
#pragma unroll
      for (int k = 0; k < kRsChunk / 32; ++k)
        if (lane + 32 * k < ck) tile[j][lane + 32 * k] = acc[k];
    }
    __syncthreads();
    if (lane < ncell)
      for (int cc = warp; cc < ck; cc += kRsThreads / 32) o[(int64_t)(c0 + cc) * plane + lane] = from_f32<E>(tile[lane][cc]);
    __syncthreads();
  }
}

// ---- backward, channels_last gradient: 8 lanes per source row
template <typename E>
__global__ void __launch_bounds__(kRsThreads)
resize_nearest_bwd_rows_kernel(const float *__restrict__ g, int64_t g_stride, E *__restrict__ gsrc, int batch, int C,
                               int Hs, int Ws, int Hd, int Wd) {
  pdl_wait();
  pdl_trigger();
  const int64_t cell = ((int64_t)blockIdx.x * kRsThreads + threadIdx.x) >> 3;
  const int l8 = threadIdx.x & 7;
  const int64_t src_cells = (int64_t)Hs * Ws;
  if (cell >= (int64_t)batch * src_cells) return;
  const int b = (int)(cell / src_cells);
  const int rem = (int)(cell - (int64_t)b * src_cells);
  const int sy = rem / Ws, sx = rem - sy * Ws;
  const int y_lo = nearest_first_dst(sy, Hs, Hd), y_hi = nearest_first_dst(sy + 1, Hs, Hd);
  const int x_lo = nearest_first_dst(sx, Ws, Wd), x_hi = nearest_first_dst(sx + 1, Ws, Wd);
  const float *gb = g + (int64_t)b * Hd * Wd * g_stride;
  E *o = gsrc + cell * C;
  for (int c0 = 4 * l8; c0 < C; c0 += 32 * kRsVec) {
    float4 acc[kRsVec];
#pragma unroll
    for (int k = 0; k < kRsVec; ++k) acc[k] = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int y = y_lo; y < y_hi; ++y)
      for (int x = x_lo; x < x_hi; ++x) {
        const float *row = gb + ((int64_t)y * Wd + x) * g_stride;
#pragma unroll
        for (int k = 0; k < kRsVec; ++k)
          if (c0 + 32 * k < C) add4(acc[k], load4(row + c0 + 32 * k));
      }
#pragma unroll
    for (int k = 0; k < kRsVec; ++k)
      if (c0 + 32 * k < C) store4(o + c0 + 32 * k, acc[k]);
  }
}

int check_resize_args(const void *src, const void *rows, int64_t row_stride, int dtype, int src_is_nchw, int batch,
                      int channels, int src_h, int src_w, int dst_h, int dst_w) {
  if (!src || !rows || batch < 1 || channels < 1 || src_h < 1 || src_w < 1 || dst_h < 1 || dst_w < 1) return BEVPOOL_E_ARG;
  if (dtype != BEVPOOL_F32 && dtype != BEVPOOL_F16 && dtype != BEVPOOL_BF16) return BEVPOOL_E_DTYPE;
  if ((channels % 4) != 0) return BEVPOOL_E_CHANNELS;
  if (row_stride < channels || (row_stride % 4) != 0) return BEVPOOL_E_ARG;
  if ((int64_t)batch * src_h * src_w >= (int64_t)INT32_MAX || (int64_t)batch * dst_h * dst_w >= (int64_t)INT32_MAX)
    return BEVPOOL_E_RANGE;
  if (!aligned16(rows) || (!src_is_nchw && (reinterpret_cast<uintptr_t>(src) & (dtype == BEVPOOL_F32 ? 15u : 7u))))
    return BEVPOOL_E_ALIGN;
  return BEVPOOL_OK;
}

template <typename E>
int launch_resize_fwd(const void *src, int src_is_nchw, int batch, int C, int Hs, int Ws, int Hd, int Wd, float *out,
                      int64_t out_stride, cudaStream_t s) {
  const E *p = static_cast<const E *>(src);
  if (src_is_nchw) {
    const int tiles_x = (int)ceil_div64(Wd, kRsCells);
    BEVPOOL_RETURN_IF_CUDA(launch_pdl(resize_nearest_fwd_nchw_kernel<E>, dim3((unsigned)((int64_t)batch * Hd * tiles_x)),
                                      dim3(kRsThreads), 0, s, p, out, out_stride, C, Hs, Ws, Hd, Wd, tiles_x));
  } else {
    const int64_t threads = (int64_t)batch * Hd * Wd * 8;
    BEVPOOL_RETURN_IF_CUDA(launch_pdl(resize_nearest_fwd_rows_kernel<E>, dim3((unsigned)ceil_div64(threads, kRsThreads)),
                                      dim3(kRsThreads), 0, s, p, out, out_stride, batch, C, Hs, Ws, Hd, Wd));
  }
  BEVPOOL_LAUNCH_CHECK();
  return BEVPOOL_OK;
}

template <typename E>
int launch_resize_bwd(const float *g, int64_t g_stride, void *gsrc, int src_is_nchw, int batch, int C, int Hs, int Ws,
                      int Hd, int Wd, cudaStream_t s) {
  E *p = static_cast<E *>(gsrc);
  if (src_is_nchw) {
    const int tiles_x = (int)ceil_div64(Ws, kRsCells);
    BEVPOOL_RETURN_IF_CUDA(launch_pdl(resize_nearest_bwd_nchw_kernel<E>, dim3((unsigned)((int64_t)batch * Hs * tiles_x)),
                                      dim3(kRsThreads), 0, s, g, g_stride, p, C, Hs, Ws, Hd, Wd, tiles_x));
  } else {
    const int64_t threads = (int64_t)batch * Hs * Ws * 8;
    BEVPOOL_RETURN_IF_CUDA(launch_pdl(resize_nearest_bwd_rows_kernel<E>, dim3((unsigned)ceil_div64(threads, kRsThreads)),
                                      dim3(kRsThreads), 0, s, g, g_stride, p, batch, C, Hs, Ws, Hd, Wd));
  }
  BEVPOOL_LAUNCH_CHECK();
  return BEVPOOL_OK;
}

}  // namespace
}  // namespace bevpool

using namespace bevpool;

extern "C" int bevpool_resize_nearest_index(int in_size, int out_size, int32_t *src_of_dst_host,
                                            int32_t *first_dst_host) {
  if (in_size < 1 || out_size < 1) return BEVPOOL_E_ARG;
  if (src_of_dst_host)
    for (int d = 0; d < out_size; ++d) src_of_dst_host[d] = nearest_src(d, in_size, out_size);
  if (first_dst_host)
    for (int s = 0; s <= in_size; ++s) first_dst_host[s] = nearest_first_dst(s, in_size, out_size);
  return BEVPOOL_OK;
}

extern "C" int bevpool_resize_nearest_into(const void *src, int dtype, int src_is_nchw, int batch, int channels,
                                           int src_h, int src_w, int dst_h, int dst_w, float *out_rows,
                                           int64_t out_row_stride, void *stream) {
  const int rc = check_resize_args(src, out_rows, out_row_stride, dtype, src_is_nchw, batch, channels, src_h, src_w,
                                   dst_h, dst_w);
  if (rc) return rc;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (dtype == BEVPOOL_F32)
    return launch_resize_fwd<float>(src, src_is_nchw, batch, channels, src_h, src_w, dst_h, dst_w, out_rows, out_row_stride, s);
  if (dtype == BEVPOOL_F16)
    return launch_resize_fwd<__half>(src, src_is_nchw, batch, channels, src_h, src_w, dst_h, dst_w, out_rows, out_row_stride, s);
  return launch_resize_fwd<__nv_bfloat16>(src, src_is_nchw, batch, channels, src_h, src_w, dst_h, dst_w, out_rows,
                                          out_row_stride, s);
}

extern "C" int bevpool_resize_nearest_backward_from(const float *grad_rows, int64_t grad_row_stride, void *grad_src,
                                                    int dtype, int src_is_nchw, int batch, int channels, int src_h,
                                                    int src_w, int dst_h, int dst_w, void *stream) {
  const int rc = check_resize_args(grad_src, grad_rows, grad_row_stride, dtype, src_is_nchw, batch, channels, src_h,
                                   src_w, dst_h, dst_w);
  if (rc) return rc;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (dtype == BEVPOOL_F32)
    return launch_resize_bwd<float>(grad_rows, grad_row_stride, grad_src, src_is_nchw, batch, channels, src_h, src_w,
                                    dst_h, dst_w, s);
  if (dtype == BEVPOOL_F16)
    return launch_resize_bwd<__half>(grad_rows, grad_row_stride, grad_src, src_is_nchw, batch, channels, src_h, src_w,
                                     dst_h, dst_w, s);
  return launch_resize_bwd<__nv_bfloat16>(grad_rows, grad_row_stride, grad_src, src_is_nchw, batch, channels, src_h,
                                          src_w, dst_h, dst_w, s);
}

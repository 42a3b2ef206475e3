// BEV augmentation warp: kornia.geometry.transform.warp_affine(src, M, dsize, mode='bilinear', padding_mode='zeros',
// align_corners=True), as models/bev_depth.py's bev_augment_image applies it with the BDA matrix.
//
// The caller passes theta = the (B, 2, 3) matrix kornia hands to F.affine_grid (normalised destination -> normalised
// source, computed from M in torch: ops/bev_augment.py).  The kernels evaluate affine_grid + grid_sample themselves,
// in float32 with torch's formulas (warp_taps below), on channels-last rows:
//   forward   out[d]  = sum over the taps t of d, in the order nw, ne, sw, se, of w_t(d) * src[tap_t(d)]
//   backward  gsrc[s] = sum over the destination pixels d that have s as a tap, in ascending d, of w_t(d) * g[d]
// The backward is a gather over source cells, not a scatter: no atomics, the result is a pure function of the inputs.
// It enumerates a window of candidate destination pixels per source cell and decides membership with warp_taps, the
// function the forward uses, so it is the exact adjoint of the forward tap for tap (also where floor() of a coordinate
// that sits on an integer could go either way).
//
// Optional cell_start (a pooling plan's CSR, B*H*W + 1 entries): source cells with cell_start[c + 1] == cell_start[c]
// are known to be zero rows.  The forward skips such taps without reading the row (adding w * 0, w >= +0, never
// changes the accumulator's value, so the result equals reading a zero row -- by value: an accumulator at -0 from an
// underflowed negative product stays -0 where the zero row would make it +0); the backward writes gradient rows for
// occupied cells only and leaves the others untouched.
#include "common.cuh"
#include "tma.cuh"

#include <math.h>
#include <type_traits>

namespace bevpool {
namespace {

constexpr int kWarpThreads = 256;     // 32 groups of 8 lanes: one destination pixel (forward) / source cell (backward)
constexpr int kWarpChunks = 4;        // float4 chunks per lane per pass: a pass covers 8 * 4 * 4 = 128 channels

struct WarpTaps {
  int x0, y0;                         // the nw tap; ne = (x0 + 1, y0), sw = (x0, y0 + 1), se = (x0 + 1, y0 + 1)
  float w[4];                         // weights in the order nw, ne, sw, se
  unsigned valid;                     // bit t: tap t lies inside the source grid
};

// torch.linspace(-1, 1, n) in float32 as torch's CUDA kernel computes it (the base grid of F.affine_grid)
__device__ __forceinline__ float linspace_m1p1(int i, int n) {
  const float step = 2.f / (float)(n - 1);
  return i < n / 2 ? fmaf(step, (float)i, -1.f) : fmaf(-step, (float)(n - 1 - i), 1.f);
}

// affine_grid (align_corners=True) + grid_sampler_2d's bilinear taps for destination pixel (dx, dy).
// A non-finite coordinate, or one so far outside that no tap can touch the grid, gives no valid tap.
__device__ __forceinline__ WarpTaps warp_taps(const float (&th)[6], int dx, int dy, int Wd, int Hd, int Ws, int Hs) {
  const float xn = linspace_m1p1(dx, Wd), yn = linspace_m1p1(dy, Hd);
  const float gx = fmaf(th[0], xn, fmaf(th[1], yn, th[2]));
  const float gy = fmaf(th[3], xn, fmaf(th[4], yn, th[5]));
  const float ix = ((gx + 1.f) * 0.5f) * (float)(Ws - 1);       // grid_sampler_unnormalize, align_corners
  const float iy = ((gy + 1.f) * 0.5f) * (float)(Hs - 1);
  WarpTaps t;
  t.x0 = t.y0 = 0;
  t.w[0] = t.w[1] = t.w[2] = t.w[3] = 0.f;
  t.valid = 0u;
  if (!(ix > -2.f && ix < (float)Ws + 1.f && iy > -2.f && iy < (float)Hs + 1.f)) return t;
  const float fx = floorf(ix), fy = floorf(iy);
  t.x0 = (int)fx;
  t.y0 = (int)fy;
  const float ex = (fx + 1.f) - ix, wx = ix - fx, ey = (fy + 1.f) - iy, wy = iy - fy;
  t.w[0] = ex * ey;
  t.w[1] = wx * ey;
  t.w[2] = ex * wy;
  t.w[3] = wx * wy;
  const bool x0in = t.x0 >= 0 && t.x0 < Ws, x1in = t.x0 + 1 >= 0 && t.x0 + 1 < Ws;
  const bool y0in = t.y0 >= 0 && t.y0 < Hs, y1in = t.y0 + 1 >= 0 && t.y0 + 1 < Hs;
  t.valid = (x0in && y0in ? 1u : 0u) | (x1in && y0in ? 2u : 0u) | (x0in && y1in ? 4u : 0u) | (x1in && y1in ? 8u : 0u);
  return t;
}

__device__ __forceinline__ void load_theta(const float *theta, int b, float (&th)[6]) {
#pragma unroll
  for (int i = 0; i < 6; ++i) th[i] = __ldg(theta + 6 * b + i);
}

// Candidate window of source cell (sx, sy): destination pixels whose footprint can touch it.  A footprint touches the
// cell iff the pixel's source coordinate lies in [sx - 1, sx + 1) x [sy - 1, sy + 1); the window is the bounding box
// of that square's preimage under the (double precision) destination -> source pixel map, the square first widened by
// a bound on the float32 error of the kernel's coordinates (a flat one-pixel margin dropped taps at magnifications
// around 10^5), clipped to the grid.  Empty when theta is not finite (then no destination pixel has a finite
// coordinate); the whole grid when the map is singular.
__device__ __forceinline__ void warp_window(const float (&th)[6], int sx, int sy, int Ws, int Hs, int Wd, int Hd,
                                            int &x_lo, int &x_hi, int &y_lo, int &y_hi) {
  bool finite = true;
#pragma unroll
  for (int i = 0; i < 6; ++i) finite = finite && isfinite(th[i]);
  if (!finite) {
    x_lo = y_lo = 0;
    x_hi = y_hi = -1;
    return;
  }
  x_lo = y_lo = 0;
  x_hi = Wd - 1;
  y_hi = Hd - 1;
  const double hx = 0.5 * (Ws - 1), hy = 0.5 * (Hs - 1), kx = 2.0 / (Wd - 1), ky = 2.0 / (Hd - 1);
  const double a00 = hx * th[0] * kx, a01 = hx * th[1] * ky, a10 = hy * th[3] * kx, a11 = hy * th[4] * ky;
  const double b0 = hx * ((double)th[2] + 1.0 - th[0] - th[1]), b1 = hy * ((double)th[5] + 1.0 - th[3] - th[4]);
  const double det = a00 * a11 - a01 * a10;
  if (!(fabs(det) > 0.0) || !isfinite(det)) return;
  const double i00 = a11 / det, i01 = -a01 / det, i10 = -a10 / det, i11 = a00 / det;
  const double u = sx - b0, v = sy - b1;
  const double cx = i00 * u + i01 * v, cy = i10 * u + i11 * v;
  // float32 error of warp_taps' coordinates, in source pixels: |ix - exact| <= (Ws - 1) u (3 S + 1) with
  // S = |th0| + |th1| + |th2| and u = 2^-24 (2u from linspace, one rounding per fmaf / add / multiply); taken
  // as (Ws - 1) 2^-22 (S + 1), then mapped to destination pixels through |A^-1|
  const double dx = (Ws - 1) * 0x1p-22 * (fabs((double)th[0]) + fabs((double)th[1]) + fabs((double)th[2]) + 1.0);
  const double dy = (Hs - 1) * 0x1p-22 * (fabs((double)th[3]) + fabs((double)th[4]) + fabs((double)th[5]) + 1.0);
  const double ex = fabs(i00) * (1.0 + dx) + fabs(i01) * (1.0 + dy), ey = fabs(i10) * (1.0 + dx) + fabs(i11) * (1.0 + dy);
  const double xl = floor(cx - ex), xh = ceil(cx + ex), yl = floor(cy - ey), yh = ceil(cy + ey);
  if (!(isfinite(xl) && isfinite(xh) && isfinite(yl) && isfinite(yh))) return;
  x_lo = (int)fmin(fmax(xl, 0.0), (double)Wd);
  x_hi = (int)fmax(fmin(xh, Wd - 1.0), -1.0);
  y_lo = (int)fmin(fmax(yl, 0.0), (double)Hd);
  y_hi = (int)fmax(fmin(yh, Hd - 1.0), -1.0);
}

// A chunk of 4 consecutive row elements: a float4 of fp32 rows, 8 bytes (uint2) of fp16 / bf16 rows.  ld4 widens a
// chunk exactly to fp32; st4 rounds each element once to nearest even (fp16 beyond 65504: +-inf, as torch's `.to(dtype)`).
template <typename T> using Chunk4 = typename std::conditional<sizeof(T) == 4, float4, uint2>::type;
template <typename T>
__device__ __forceinline__ float4 ld4(const Chunk4<T> *p) {
  if constexpr (sizeof(T) == 4) {
    return __ldg(p);
  } else {
    const uint2 u = __ldg(p);
    const float2 a = CtxType<T>::to_float2(u.x), b = CtxType<T>::to_float2(u.y);
    return make_float4(a.x, a.y, b.x, b.y);
  }
}
template <typename T>
__device__ __forceinline__ void st4(Chunk4<T> *p, const float4 &v) {
  if constexpr (sizeof(T) == 4) stg_stream_f4(p, v);
  else *p = make_uint2(CtxType<T>::from_float2(v.x, v.y), CtxType<T>::from_float2(v.z, v.w));
}

__device__ __forceinline__ void fma4(float4 &acc, const float4 &v, float w) {
  acc.x = fmaf(v.x, w, acc.x);
  acc.y = fmaf(v.y, w, acc.y);
  acc.z = fmaf(v.z, w, acc.z);
  acc.w = fmaf(v.w, w, acc.w);
}

// One 8-lane group per destination pixel; lane l8 owns the float4 chunks l8, l8 + 8, ... of the row.  Every element of
// every destination row is written exactly once, zeros included.  TO: element type of the destination rows (fp32, or
// fp16 / bf16: the fp32 sum of the taps rounded once where it is stored).
template <typename TO = float>
__global__ void __launch_bounds__(kWarpThreads)
warp_affine_fwd_kernel(const float *__restrict__ theta, const float *__restrict__ src, int64_t src_stride,
                       TO *__restrict__ out, int64_t out_stride, const int32_t *__restrict__ cell_start, int batch,
                       int C, int Hs, int Ws, int Hd, int Wd) {
  pdl_wait();
  pdl_trigger();
  const int64_t pix = ((int64_t)blockIdx.x * kWarpThreads + threadIdx.x) >> 3;
  const int l8 = threadIdx.x & 7;
  const int64_t dst_cells = (int64_t)Hd * Wd;
  if (pix >= (int64_t)batch * dst_cells) return;
  const int b = (int)(pix / dst_cells);
  const int rem = (int)(pix - (int64_t)b * dst_cells);
  const int dy = rem / Wd, dx = rem - dy * Wd;
  float th[6];
  load_theta(theta, b, th);
  const WarpTaps t = warp_taps(th, dx, dy, Wd, Hd, Ws, Hs);
  const int64_t cbase = (int64_t)b * Hs * Ws;
  int64_t cell[4];
  unsigned use = 0u;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    cell[k] = cbase + (int64_t)(t.y0 + (k >> 1)) * Ws + (t.x0 + (k & 1));
    if ((t.valid >> k) & 1u) {
      if (!cell_start || __ldg(cell_start + cell[k] + 1) != __ldg(cell_start + cell[k])) use |= 1u << k;
    }
  }
  const int C4 = C >> 2;
  const float4 *s4 = reinterpret_cast<const float4 *>(src);
  Chunk4<TO> *o4 = reinterpret_cast<Chunk4<TO> *>(out + pix * out_stride);
  const int64_t s4_stride = src_stride >> 2;
  for (int c0 = 0; c0 < C4; c0 += 8 * kWarpChunks) {
    float4 acc[kWarpChunks];
#pragma unroll
    for (int j = 0; j < kWarpChunks; ++j) acc[j] = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      if (!((use >> k) & 1u)) continue;
      const float4 *row = s4 + cell[k] * s4_stride;
#pragma unroll
      for (int j = 0; j < kWarpChunks; ++j) {
        const int q = c0 + 8 * j + l8;
        if (q < C4) fma4(acc[j], __ldg(row + q), t.w[k]);
      }
    }
#pragma unroll
    for (int j = 0; j < kWarpChunks; ++j) {
      const int q = c0 + 8 * j + l8;
      if (q < C4) st4<TO>(o4 + q, acc[j]);
    }
  }
}

// One 8-lane group per source cell.  The lanes test 8 candidates of the window at a time (row-major order = ascending
// destination index); the group then adds the matches in that order, each lane for its own channel chunks.  TG: element
// type of the gradient rows (fp32, or fp16 / bf16 widened exactly where they are loaded); grad_src is fp32.
template <typename TG = float>
__global__ void __launch_bounds__(kWarpThreads)
warp_affine_bwd_kernel(const float *__restrict__ theta, const TG *__restrict__ grad_out, int64_t grad_out_stride,
                       float *__restrict__ grad_src, int64_t grad_src_stride, const int32_t *__restrict__ cell_start,
                       int batch, int C, int Hs, int Ws, int Hd, int Wd) {
  pdl_wait();
  pdl_trigger();
  const int64_t cell = ((int64_t)blockIdx.x * kWarpThreads + threadIdx.x) >> 3;
  const int lane = threadIdx.x & 31, l8 = lane & 7, gshift = lane & 24;
  const unsigned gmask = 0xffu << gshift;
  const int64_t src_cells = (int64_t)Hs * Ws;
  if (cell >= (int64_t)batch * src_cells) return;
  if (cell_start && __ldg(cell_start + cell + 1) == __ldg(cell_start + cell)) return;
  const int b = (int)(cell / src_cells);
  const int rem = (int)(cell - (int64_t)b * src_cells);
  const int sy = rem / Ws, sx = rem - sy * Ws;
  float th[6];
  load_theta(theta, b, th);
  int x_lo, x_hi, y_lo, y_hi;
  warp_window(th, sx, sy, Ws, Hs, Wd, Hd, x_lo, x_hi, y_lo, y_hi);
  const int bw = x_hi - x_lo + 1, bh = y_hi - y_lo + 1;
  const int64_t nc = (bw > 0 && bh > 0) ? (int64_t)bw * bh : 0;
  const int C4 = C >> 2;
  const Chunk4<TG> *g4 = reinterpret_cast<const Chunk4<TG> *>(grad_out) + (int64_t)b * Hd * Wd * (grad_out_stride >> 2);
  const int64_t g4_stride = grad_out_stride >> 2;
  float4 *o4 = reinterpret_cast<float4 *>(grad_src + cell * grad_src_stride);
  for (int c0 = 0; c0 < C4; c0 += 8 * kWarpChunks) {
    float4 acc[kWarpChunks];
#pragma unroll
    for (int j = 0; j < kWarpChunks; ++j) acc[j] = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int64_t j0 = 0; j0 < nc; j0 += 8) {
      const int64_t j = j0 + l8;
      bool hit = false;
      float w = 0.f;
      int d = 0;
      if (j < nc) {
        const int dy = y_lo + (int)(j / bw), dx = x_lo + (int)(j % bw);
        const WarpTaps t = warp_taps(th, dx, dy, Wd, Hd, Ws, Hs);
        const int tx = sx - t.x0, ty = sy - t.y0;
        if (tx >= 0 && tx <= 1 && ty >= 0 && ty <= 1) {
          const int k = 2 * ty + tx;
          hit = (t.valid >> k) & 1u;
          w = k == 0 ? t.w[0] : k == 1 ? t.w[1] : k == 2 ? t.w[2] : t.w[3];   // (no local-memory indexing)
          d = dy * Wd + dx;
        }
      }
      unsigned m = (__ballot_sync(gmask, hit) >> gshift) & 0xffu;
      while (m) {
        const int k = __ffs(m) - 1;
        m &= m - 1;
        const float wk = __shfl_sync(gmask, w, k, 8);
        const int dk = __shfl_sync(gmask, d, k, 8);
        const Chunk4<TG> *row = g4 + (int64_t)dk * g4_stride;
#pragma unroll
        for (int jj = 0; jj < kWarpChunks; ++jj) {
          const int q = c0 + 8 * jj + l8;
          if (q < C4) fma4(acc[jj], ld4<TG>(row + q), wk);
        }
      }
    }
#pragma unroll
    for (int j = 0; j < kWarpChunks; ++j) {
      const int q = c0 + 8 * j + l8;
      if (q < C4) stg_stream_f4(o4 + q, acc[j]);
    }
  }
}

// Camera slice of a 16-bit concatenated gradient -> packed fp32 (B, Y, X, C) rows (exact), occupied cells only; one
// 8-lane group per cell.
template <typename TG>
__global__ void __launch_bounds__(kWarpThreads)
grad_rows_widen_kernel(const int32_t *__restrict__ cell_start, const TG *__restrict__ grad, int64_t grad_stride,
                       float *__restrict__ rows, int64_t cells, int C) {
  pdl_wait();
  pdl_trigger();
  const int64_t cell = ((int64_t)blockIdx.x * kWarpThreads + threadIdx.x) >> 3;
  const int l8 = threadIdx.x & 7;
  if (cell >= cells || __ldg(cell_start + cell + 1) == __ldg(cell_start + cell)) return;
  const Chunk4<TG> *g = reinterpret_cast<const Chunk4<TG> *>(grad + cell * grad_stride);
  float4 *o = reinterpret_cast<float4 *>(rows + cell * C);
  for (int q = l8; q < C / 4; q += 8) stg_stream_f4(o + q, ld4<TG>(g + q));
}

int check_warp_args(const void *theta, const void *in, int64_t in_stride, const void *out, int64_t out_stride,
                    int batch, int channels, int src_h, int src_w, int dst_h, int dst_w) {
  if (!theta || !in || !out || batch <= 0 || channels <= 0) return BEVPOOL_E_ARG;
  if (src_h < 2 || src_w < 2 || dst_h < 2 || dst_w < 2) return BEVPOOL_E_ARG;
  if ((channels % 4) != 0) return BEVPOOL_E_CHANNELS;
  if (in_stride < channels || (in_stride % 4) != 0 || out_stride < channels || (out_stride % 4) != 0) return BEVPOOL_E_ARG;
  if ((int64_t)batch * src_h * src_w >= (int64_t)INT32_MAX || (int64_t)batch * dst_h * dst_w >= (int64_t)INT32_MAX)
    return BEVPOOL_E_RANGE;
  if (!aligned16(in) || !aligned16(out)) return BEVPOOL_E_ALIGN;
  return BEVPOOL_OK;
}

}  // namespace
}  // namespace bevpool

using namespace bevpool;

extern "C" int bevpool_warp_affine_forward(const float *theta, const void *src_rows, int64_t src_row_stride,
                                           void *out_rows, int64_t out_row_stride, const int32_t *cell_start,
                                           int batch, int channels, int src_h, int src_w, int dst_h, int dst_w,
                                           void *stream) {
  int rc = check_warp_args(theta, src_rows, src_row_stride, out_rows, out_row_stride, batch, channels, src_h, src_w,
                           dst_h, dst_w);
  if (rc) return rc;
  const int64_t threads = (int64_t)batch * dst_h * dst_w * 8;
  BEVPOOL_RETURN_IF_CUDA(launch_pdl(warp_affine_fwd_kernel<float>, dim3((unsigned)ceil_div64(threads, kWarpThreads)),
                                    dim3(kWarpThreads), 0, static_cast<cudaStream_t>(stream), theta,
                                    static_cast<const float *>(src_rows), src_row_stride, static_cast<float *>(out_rows),
                                    out_row_stride, cell_start, batch, channels, src_h, src_w, dst_h, dst_w));
  BEVPOOL_LAUNCH_CHECK();
  return BEVPOOL_OK;
}

extern "C" int bevpool_warp_affine_backward(const float *theta, const void *grad_out_rows, int64_t grad_out_row_stride,
                                            void *grad_src_rows, int64_t grad_src_row_stride, const int32_t *cell_start,
                                            int batch, int channels, int src_h, int src_w, int dst_h, int dst_w,
                                            void *stream) {
  int rc = check_warp_args(theta, grad_out_rows, grad_out_row_stride, grad_src_rows, grad_src_row_stride, batch, channels,
                           src_h, src_w, dst_h, dst_w);
  if (rc) return rc;
  const int64_t threads = (int64_t)batch * src_h * src_w * 8;
  BEVPOOL_RETURN_IF_CUDA(launch_pdl(warp_affine_bwd_kernel<float>, dim3((unsigned)ceil_div64(threads, kWarpThreads)),
                                    dim3(kWarpThreads), 0, static_cast<cudaStream_t>(stream), theta,
                                    static_cast<const float *>(grad_out_rows), grad_out_row_stride,
                                    static_cast<float *>(grad_src_rows), grad_src_row_stride, cell_start, batch, channels,
                                    src_h, src_w, dst_h, dst_w));
  BEVPOOL_LAUNCH_CHECK();
  return BEVPOOL_OK;
}

// The BDA warp between the fp32 pooled scratch and the fp16 / bf16 concatenated rows (out_dtype / grad_dtype: BEVPOOL_F16
// or BEVPOOL_BF16, else BEVPOOL_E_DTYPE).  Same taps, order and cell_start skipping as the fp32 entry points: the
// forward's destination rows equal theirs `.to(out_dtype)` bit for bit, and the backward's fp32 gradient rows equal
// theirs on the widened gradient.
extern "C" int bevpool_warp_affine_forward16(const float *theta, const void *src_rows, int64_t src_row_stride, void *out_rows,
                                             int64_t out_row_stride, int out_dtype, const int32_t *cell_start, int batch,
                                             int channels, int src_h, int src_w, int dst_h, int dst_w, void *stream) {
  int rc = check_warp_args(theta, src_rows, src_row_stride, out_rows, out_row_stride, batch, channels, src_h, src_w,
                           dst_h, dst_w);
  if (rc) return rc;
  if (out_dtype != BEVPOOL_F16 && out_dtype != BEVPOOL_BF16) return BEVPOOL_E_DTYPE;
  const dim3 grid((unsigned)ceil_div64((int64_t)batch * dst_h * dst_w * 8, kWarpThreads));
  const float *src = static_cast<const float *>(src_rows);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (out_dtype == BEVPOOL_F16)
    BEVPOOL_RETURN_IF_CUDA(launch_pdl(warp_affine_fwd_kernel<__half>, grid, dim3(kWarpThreads), 0, s, theta, src, src_row_stride,
                                      static_cast<__half *>(out_rows), out_row_stride, cell_start, batch, channels, src_h, src_w,
                                      dst_h, dst_w));
  else
    BEVPOOL_RETURN_IF_CUDA(launch_pdl(warp_affine_fwd_kernel<__nv_bfloat16>, grid, dim3(kWarpThreads), 0, s, theta, src,
                                      src_row_stride, static_cast<__nv_bfloat16 *>(out_rows), out_row_stride, cell_start, batch,
                                      channels, src_h, src_w, dst_h, dst_w));
  BEVPOOL_LAUNCH_CHECK();
  return BEVPOOL_OK;
}

extern "C" int bevpool_warp_affine_backward16(const float *theta, const void *grad_out_rows, int64_t grad_out_row_stride,
                                              int grad_dtype, void *grad_src_rows, int64_t grad_src_row_stride,
                                              const int32_t *cell_start, int batch, int channels, int src_h, int src_w,
                                              int dst_h, int dst_w, void *stream) {
  int rc = check_warp_args(theta, grad_out_rows, grad_out_row_stride, grad_src_rows, grad_src_row_stride, batch, channels,
                           src_h, src_w, dst_h, dst_w);
  if (rc) return rc;
  if (grad_dtype != BEVPOOL_F16 && grad_dtype != BEVPOOL_BF16) return BEVPOOL_E_DTYPE;
  const dim3 grid((unsigned)ceil_div64((int64_t)batch * src_h * src_w * 8, kWarpThreads));
  float *gsrc = static_cast<float *>(grad_src_rows);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (grad_dtype == BEVPOOL_F16)
    BEVPOOL_RETURN_IF_CUDA(launch_pdl(warp_affine_bwd_kernel<__half>, grid, dim3(kWarpThreads), 0, s, theta,
                                      static_cast<const __half *>(grad_out_rows), grad_out_row_stride, gsrc, grad_src_row_stride,
                                      cell_start, batch, channels, src_h, src_w, dst_h, dst_w));
  else
    BEVPOOL_RETURN_IF_CUDA(launch_pdl(warp_affine_bwd_kernel<__nv_bfloat16>, grid, dim3(kWarpThreads), 0, s, theta,
                                      static_cast<const __nv_bfloat16 *>(grad_out_rows), grad_out_row_stride, gsrc,
                                      grad_src_row_stride, cell_start, batch, channels, src_h, src_w, dst_h, dst_w));
  BEVPOOL_LAUNCH_CHECK();
  return BEVPOOL_OK;
}

// Without a BDA warp the pooling backward reads the camera slice of the concatenated gradient directly; a 16-bit one is
// first widened into fp32 rows here, for the cells the plan's cell_start marks occupied (the only rows that backward
// reads; the others are left untouched).
extern "C" int bevpool_grad_rows_widen(const int32_t *cell_start, const void *grad_rows, int64_t grad_row_stride,
                                       int grad_dtype, float *rows, int batch, int channels, int num_voxel_x,
                                       int num_voxel_y, void *stream) {
  if (!cell_start || !grad_rows || !rows || batch <= 0 || num_voxel_x <= 0 || num_voxel_y <= 0) return BEVPOOL_E_ARG;
  if (channels <= 0 || (channels % 4) != 0) return BEVPOOL_E_CHANNELS;
  if (grad_row_stride < channels || (grad_row_stride % 4) != 0) return BEVPOOL_E_ARG;
  if (grad_dtype != BEVPOOL_F16 && grad_dtype != BEVPOOL_BF16) return BEVPOOL_E_DTYPE;
  const int64_t cells = (int64_t)batch * num_voxel_x * num_voxel_y;
  if (cells >= (int64_t)INT32_MAX) return BEVPOOL_E_RANGE;
  if (!aligned16(grad_rows) || !aligned16(rows)) return BEVPOOL_E_ALIGN;
  const dim3 grid((unsigned)ceil_div64(cells * 8, kWarpThreads));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (grad_dtype == BEVPOOL_F16)
    BEVPOOL_RETURN_IF_CUDA(launch_pdl(grad_rows_widen_kernel<__half>, grid, dim3(kWarpThreads), 0, s, cell_start,
                                      static_cast<const __half *>(grad_rows), grad_row_stride, rows, cells, channels));
  else
    BEVPOOL_RETURN_IF_CUDA(launch_pdl(grad_rows_widen_kernel<__nv_bfloat16>, grid, dim3(kWarpThreads), 0, s, cell_start,
                                      static_cast<const __nv_bfloat16 *>(grad_rows), grad_row_stride, rows, cells, channels));
  BEVPOOL_LAUNCH_CHECK();
  return BEVPOOL_OK;
}

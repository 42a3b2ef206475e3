// Shared helpers for libbevpool_sm100 (sm_100a only; no torch headers).
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <cstdlib>

#include "../../include/bevpool_sm100.h"

#define BEVPOOL_RETURN_IF_CUDA(expr)              \
  do {                                            \
    cudaError_t _e = (expr);                      \
    if (_e != cudaSuccess) return (int)_e;        \
  } while (0)

// placed after every kernel launch: counts it (bevpool_launch_count) and surfaces launch errors
#define BEVPOOL_LAUNCH_CHECK()                    \
  do {                                            \
    ++::bevpool::g_kernel_launches;               \
    cudaError_t _e = cudaPeekAtLastError();       \
    if (_e != cudaSuccess) return (int)_e;        \
  } while (0)

#include <atomic>

namespace bevpool {

extern std::atomic<long long> g_kernel_launches;   // defined in plan.cu

constexpr int kSMs = 148;  // B200: 2 dies x 74 SMs

__host__ __device__ inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
__host__ __device__ inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }

inline bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// ---- 128-bit global access with cache hints --------------------------------------
// streaming read: data touched once (feature rows of the drop-in op): do not pollute L1
__device__ __forceinline__ float4 ldg_stream_f4(const float4 *p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ int4 ldg_stream_i4(const int4 *p) {
  int4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ int ldg_stream_i32(const int *p) {
  int r;
  asm volatile("ld.global.nc.L1::no_allocate.s32 %0, [%1];" : "=r"(r) : "l"(p));
  return r;
}
__device__ __forceinline__ float ldg_stream_f32(const float *p) {
  float r;
  asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(r) : "l"(p));
  return r;
}
// reused read: gathers that hit L1/L2 (context rows, gradient rows)
__device__ __forceinline__ float4 ldg_f4(const float4 *p) { return __ldg(p); }
// streaming store: outputs written exactly once
__device__ __forceinline__ void stg_stream_f4(float4 *p, const float4 &v) {
  asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};"
               :: "l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

// ---- programmatic dependent launch (PDL) -----------------------------------------------------------
// The step is a chain of ~12 short dependent kernels; a plain stream edge costs 2-3 us per link (the next
// grid is only scheduled after the previous one has drained).  Kernels of the fused path are launched with
// the programmatic-stream-serialization attribute: every CTA signals "dependents may be scheduled" at its
// very top, so the next grid's CTAs take the SM slots the last wave frees and sit in pdl_wait() -- which
// returns only when the whole previous grid has completed and its writes are visible.  pdl_wait() is the
// FIRST statement of every such kernel (before any early return), so completion stays transitive along the
// chain.  Both instructions are no-ops for a kernel launched without the attribute.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

bool pdl_enabled();     // plan.cu: BEVPOOL_PDL != 0

bool pdl_forward_enabled();   // plan.cu: BEVPOOL_PDL_FWD == 1 (off by default: measured slower for stage A -> stage B)

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl_if(bool allow, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem,
                                 cudaStream_t s, Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = (allow && pdl_enabled()) ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s,
                              Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

struct FastDiv {          // exact n / d for 0 <= n < 2^31 (round-up magic, 64-bit product)
  uint32_t mul, shift, div;
};
inline FastDiv make_fastdiv(uint32_t d) {
  FastDiv f;
  uint32_t s = 0;
  while ((1ull << s) < d) ++s;
  f.shift = 31 + s;
  f.mul = (uint32_t)((1ull << f.shift) / d + 1ull);
  f.div = d;
  return f;
}
__device__ __forceinline__ uint32_t fastdiv(uint32_t n, const FastDiv &f) {
  return (uint32_t)(((uint64_t)n * f.mul) >> f.shift);
}

// ---- plan layout -------------------------------------------------------------------
// A plan is one caller-owned buffer:
//   header (256 B: PlanHeader) | cell_of_point int32[B*Np] | cell_start int32[B*G+1] | sorted_ids int32[B*Np]
//   | sorted_cells int32[B*Np]
// sorted_ids[k] is the global point id of the k-th kept point in (cell, point id) order and
// sorted_cells[k] its global output row b*G + cell; only the first K = cell_start[B*G] entries
// of both are defined.
struct PlanLayout {
  size_t off_cell_of_point, off_cell_start, off_sorted_ids, off_sorted_cells, off_run_code, off_pair_rec, bytes;
};
struct PlanHeader {       // first 256 bytes of a plan buffer, written by the builders (one thread of the key kernel)
  int32_t magic, kind, status, batch, num_voxel_x, num_voxel_y, num_voxel_z, reserved;
  int64_t num_points;
};
constexpr int32_t kPlanKindPoints = 1, kPlanKindRuns = 2;
// status word: 0 = ok.  Raised on the device by a consumer kernel, read back by bevpool_plan_status().
constexpr int32_t kPlanStatusRowOverflow = 1;   // run_rows scratch smaller than the plan's run count
inline int32_t *plan_status(void *plan) { return &static_cast<PlanHeader *>(plan)->status; }
constexpr int32_t kPlanMagic = 0x42455631;  // "BEV1"

// Run plan (fused op only): the sorted entries are RUNS, not points.  A run is a maximal set of
// vertically adjacent frustum points (same image, depth bin and column, consecutive rows h inside one
// block of kRunHB rows) that fall into the same BEV cell; for a level camera that is every kept point
// of a (depth bin, column) pair.  run_code int32[B*Np]: slot (position in the sorted run list) for
// the first point of a run, kRunCont for its continuation points, kRunDropped for dropped points.
constexpr int kRunHB = 16;
constexpr int32_t kRunDropped = -1, kRunCont = -2;

// Run plans also carry one PAIR RECORD per (image, depth bin, 16-row block, column) -- int4 {primary cell, masks,
// primary slot, number of runs}: the in-sample cell of the pair's first kept row (-1: nothing kept), the rows lying
// in that cell (bits 0..15) and the kept rows lying elsewhere (bits 16..31), the slot of the run that starts at the
// first kept row, and how many runs the pair holds.  For a level camera (one run per pair) the record is all the
// fused kernels need per pair: they read 16 bytes per 16 points instead of cell_of_point / run_code (128 bytes)
// and do no per-row voting; pairs with stray rows fall back to the per-point arrays.
__host__ __device__ inline int64_t plan_num_pairs(int num_cams, int D, int H, int W) {
  return (int64_t)num_cams * D * ((H + kRunHB - 1) / kRunHB) * W;
}
__host__ __device__ inline PlanLayout plan_layout(int batch, int64_t num_points, int X, int Y, bool runs = false,
                                                  int64_t pairs_per_sample = 0) {
  PlanLayout L;
  const size_t P = (size_t)batch * (size_t)num_points;
  const size_t G = (size_t)batch * (size_t)X * (size_t)Y;
  size_t o = 256;
  L.off_cell_of_point = o; o = align_up(o + P * 4, 256);
  L.off_cell_start = o;    o = align_up(o + (G + 1) * 4, 256);
  L.off_sorted_ids = o;    o = align_up(o + P * 4, 256);
  L.off_sorted_cells = o;  o = align_up(o + P * 4 + 64, 256);   // + slack: readers prefetch a batch past K
  L.off_run_code = o;
  if (runs) o = align_up(o + P * 4, 256);
  L.off_pair_rec = align_up(L.off_run_code + P * 4, 256);       // (run plans only; position independent of its size)
  if (runs) o = align_up(L.off_pair_rec + (size_t)batch * (size_t)pairs_per_sample * 16, 256);
  L.bytes = o;
  return L;
}

struct PlanView {
  const int32_t *cell_of_point, *cell_start, *sorted_ids, *sorted_cells, *run_code;
  const int4 *pair_rec;
};
inline PlanView plan_view(const void *plan, int batch, int64_t num_points, int X, int Y) {
  PlanLayout L = plan_layout(batch, num_points, X, Y);
  const char *b = static_cast<const char *>(plan);
  return PlanView{reinterpret_cast<const int32_t *>(b + L.off_cell_of_point),
                  reinterpret_cast<const int32_t *>(b + L.off_cell_start),
                  reinterpret_cast<const int32_t *>(b + L.off_sorted_ids),
                  reinterpret_cast<const int32_t *>(b + L.off_sorted_cells),
                  reinterpret_cast<const int32_t *>(b + L.off_run_code),
                  reinterpret_cast<const int4 *>(b + L.off_pair_rec)};
}

// pool_bwd2.cu: column kernel of the fused backward (fp32, g8 channel counts, W % 4 == 0); reads context and writes
// the context gradient either as pixel rows (B*N, H, W, C) or, through TMA tensor maps, as NCHW (B*N, C, H, W)
int launch_fused_backward_col(const int32_t *cell_of_point, const int4 *pair_rec, const float *grad_rows, const float *depth,
                              const float *ctx, float *grad_depth, float *grad_ctx, bool nchw, int batch, int num_cams,
                              int D, int H, int W, int C, int64_t cells_per_sample, cudaStream_t s,
                              int64_t grad_row_stride = 0);     // floats between consecutive cells' gradient rows (0: C)
bool fused_backward_col_supported(int C, int W, const void *depth, const void *grad_depth, const void *cell_of_point);

// pool_bwd.cu: tile kernel of the fused backward (fp32, g8 channel counts; any W)
int launch_fused_backward_tile(const int32_t *cell_of_point, const float *grad_rows, const float *depth,
                               const float *ctx_nhwc, float *grad_depth, float *grad_ctx_nhwc, int batch,
                               int num_cams, int D, int H, int W, int C, int64_t cells_per_sample,
                               cudaStream_t s);
bool fused_backward_tile_supported(int C);

inline int check_plan_dims(int batch, int64_t num_points, int X, int Y) {
  if (batch <= 0 || num_points <= 0 || X <= 0 || Y <= 0) return BEVPOOL_E_ARG;
  if ((int64_t)batch * num_points >= (int64_t)INT32_MAX) return BEVPOOL_E_RANGE;
  if ((int64_t)batch * X * Y >= (int64_t)INT32_MAX) return BEVPOOL_E_RANGE;
  return BEVPOOL_OK;
}
// the fused entry points: the frustum (num_cams, D, H, W) of every sample, and the plan it implies
inline int check_frustum_dims(int batch, int num_cams, int D, int H, int W, int X, int Y) {
  if (num_cams <= 0 || D <= 0 || H <= 0 || W <= 0) return BEVPOOL_E_ARG;
  return check_plan_dims(batch, (int64_t)num_cams * D * H * W, X, Y);
}

// tuning knobs for experiments; each caller keeps the value in a static, so a knob is read once per process
inline int env_int(const char *name, int dflt) {
  const char *e = std::getenv(name);
  return e && e[0] ? std::atoi(e) : dflt;
}

inline int sm_count() {                     // per device (a process may drive several GPUs)
  int dev = 0, n = 0;
  static int cached[64] = {0};
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return kSMs;
  if (cached[dev] == 0)
    cached[dev] = (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0) ? n : kSMs;
  return cached[dev];
}

}  // namespace bevpool

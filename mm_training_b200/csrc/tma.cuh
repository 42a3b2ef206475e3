// TMA (tensor memory accelerator) + mbarrier helpers for libbevpool_sm100 (sm_100a).
//
// Two flavours are used by the pooling kernels:
//  * 1-D bulk copies (cp.async.bulk, SASS UBLKCP): contiguous rows in either direction;
//  * tensor-map copies (cp.async.bulk.tensor, SASS UTMALDG / UTMASTG): boxes of a strided tensor -- this is
//    how the kernels read the reference's NCHW tensors (context (B*N, C, H, W), layers/backbones/
//    lss_fpn.py:441-443; the incoming gradient (B, C, Y, X), ops/voxel_pooling/voxel_pooling.py:58-69) and
//    write the NCHW context gradient without a separate layout pass.
// The tensor maps are encoded on the host per call (cuTensorMapEncodeTiled through the runtime's driver
// entry point: no link-time dependency on libcuda) and passed as __grid_constant__ kernel parameters.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <cstdio>
#include <cstdlib>

#include "common.cuh"

namespace bevpool {

// ---- host side ---------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline EncodeTiledFn tensor_map_encoder() {
  static EncodeTiledFn fn = [] {
    void *p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      p = nullptr;
    return reinterpret_cast<EncodeTiledFn>(p);
  }();
  return fn;
}

// tensor of `rank` dims (fastest first) with elements of `type`; strides in BYTES for dims 1..rank-1 (multiples of 16),
// box[0] * element size a multiple of 16 bytes.  Out-of-bounds elements of a box read as zero and are not written by stores.
inline int make_tensor_map(CUtensorMap *map, CUtensorMapDataType type, const void *base, int rank, const uint64_t *dims,
                           const uint64_t *strides_bytes, const uint32_t *box) {
  EncodeTiledFn enc = tensor_map_encoder();
  if (!enc) return (int)cudaErrorNotSupported;
  // The encoder is a driver entry point and wants the primary context current on the calling thread; a thread that
  // has only used the runtime lazily (autograd's backward threads) may not have bound it yet.
  static thread_local bool context_bound = false;
  if (!context_bound) {
    cudaFree(nullptr);
    context_bound = true;
  }
  cuuint64_t gd[5], gs[4];
  cuuint32_t bx[5], es[5];
  for (int i = 0; i < rank; ++i) { gd[i] = dims[i]; bx[i] = box[i]; es[i] = 1; }
  for (int i = 0; i + 1 < rank; ++i) gs[i] = strides_bytes[i];
  const CUresult r = enc(map, type, (cuuint32_t)rank, const_cast<void *>(base), gd, gs, bx, es,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    static const bool debug = [] { const char *e = std::getenv("BEVPOOL_DEBUG"); return e && e[0] == '1'; }();
    if (debug) {
      std::fprintf(stderr, "[bevpool] cuTensorMapEncodeTiled failed (%d): base %p rank %d", (int)r, base, rank);
      for (int i = 0; i < rank; ++i) std::fprintf(stderr, " dim%d=%llu box%d=%u", i, (unsigned long long)gd[i], i, bx[i]);
      for (int i = 0; i + 1 < rank; ++i) std::fprintf(stderr, " stride%d=%llu", i, (unsigned long long)gs[i]);
      std::fprintf(stderr, "\n");
    }
    return (int)cudaErrorInvalidValue;
  }
  return BEVPOOL_OK;
}

inline int make_tensor_map_f32(CUtensorMap *map, const void *base, int rank, const uint64_t *dims,
                               const uint64_t *strides_bytes, const uint32_t *box) {
  return make_tensor_map(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, base, rank, dims, strides_bytes, box);
}

// element type and tensor-map type of a context tensor: fp32, or fp16 / bf16 converted to fp32 where it is loaded
template <typename T> struct CtxType;
template <> struct CtxType<float> {
  static constexpr CUtensorMapDataType kMap = CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
  static __device__ __forceinline__ float to_float(float v) { return v; }
};
// 16-bit types: a pair of elements travels as one 32-bit word; every conversion to 16 bits rounds to nearest even
// (fp16 beyond 65504 becomes +-inf), as torch's `.to(dtype)` does
template <> struct CtxType<__half> {
  static constexpr CUtensorMapDataType kMap = CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
  static __device__ __forceinline__ float to_float(__half v) { return __half2float(v); }
  static __device__ __forceinline__ float2 to_float2(uint32_t u) { return __half22float2(*reinterpret_cast<const __half2 *>(&u)); }
  static __device__ __forceinline__ __half from_float(float v) { return __float2half_rn(v); }
  static __device__ __forceinline__ uint32_t from_float2(float a, float b) {
    const __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<const uint32_t *>(&h);
  }
};
template <> struct CtxType<__nv_bfloat16> {
  static constexpr CUtensorMapDataType kMap = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  static __device__ __forceinline__ float to_float(__nv_bfloat16 v) { return __bfloat162float(v); }
  static __device__ __forceinline__ float2 to_float2(uint32_t u) { return make_float2(__uint_as_float(u << 16), __uint_as_float(u & 0xffff0000u)); }
  static __device__ __forceinline__ __nv_bfloat16 from_float(float v) { return __float2bfloat16_rn(v); }
  static __device__ __forceinline__ uint32_t from_float2(float a, float b) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<const uint32_t *>(&h);
  }
};

// ---- device side -------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra WAIT_DONE;\n"
      "bra WAIT_LOOP;\n"
      "WAIT_DONE:\n"
      "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }

// 1-D bulk copies (16-byte aligned addresses and sizes)
__device__ __forceinline__ void tma_load_1d(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tma_store_1d(void *dst_gmem, const void *src_smem, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
               ::"l"(dst_gmem), "r"(smem_u32(src_smem)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_store_1d_hint(void *dst_gmem, const void *src_smem, uint32_t bytes, uint64_t pol) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;"
               ::"l"(dst_gmem), "r"(smem_u32(src_smem)), "r"(bytes), "l"(pol) : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// tensor-map copies: box at coordinates (c0 fastest ... c3), smem destination / source 128-byte aligned
__device__ __forceinline__ void tma_load_4d(void *dst_smem, const CUtensorMap *map, int c0, int c1, int c2, int c3,
                                            uint64_t *bar) {
  asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];"
               ::"r"(smem_u32(dst_smem)), "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tma_store_4d(const CUtensorMap *map, int c0, int c1, int c2, int c3, const void *src_smem) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.tile.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
               ::"l"(map), "r"(smem_u32(src_smem)), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void tma_prefetch_map(const CUtensorMap *map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}

// L2 eviction-priority policies
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  return p;
}

__device__ __forceinline__ uint64_t l2_policy_evict_normal() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(p));
  return p;
}
// 4-byte accesses carrying an L2 eviction-priority policy (tables that several kernels of one call re-visit at random)
__device__ __forceinline__ int ld_l2hint_i32(const int *p, uint64_t pol) {
  int v;
  asm volatile("ld.global.L2::cache_hint.s32 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol) : "memory");
  return v;
}
__device__ __forceinline__ void st_l2hint_i32(int *p, int v, uint64_t pol) {
  asm volatile("st.global.L2::cache_hint.s32 [%0], %1, %2;" ::"l"(p), "r"(v), "l"(pol) : "memory");
}
__device__ __forceinline__ void red_min_l2hint_i32(int *p, int v, uint64_t pol) {
  asm volatile("red.global.min.L2::cache_hint.s32 [%0], %1, %2;" ::"l"(p), "r"(v), "l"(pol) : "memory");
}
__device__ __forceinline__ uint32_t atom_add_l2hint_u32(uint32_t *p, uint32_t v, uint64_t pol) {
  uint32_t r;
  asm volatile("atom.global.add.L2::cache_hint.u32 %0, [%1], %2, %3;" : "=r"(r) : "l"(p), "r"(v), "l"(pol) : "memory");
  return r;
}
__device__ __forceinline__ void tma_load_1d_hint(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar, uint64_t pol) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
               ::"r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)), "l"(pol) : "memory");
}

__device__ __forceinline__ void cp_async16(void *dst_smem, const void *src_gmem) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst_smem)), "l"(src_gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_1() { asm volatile("cp.async.wait_group 1;" ::: "memory"); }

}  // namespace bevpool

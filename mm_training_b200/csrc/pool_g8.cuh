// fp32 fast path of the pooling kernels: 8 lanes per feature row ("g8" layout).
//
// A row of C = 16*NV2 floats (C = 80 -> NV2 = 5) is owned by a group of 8 lanes; lane l holds
// channels [32k + 4l, +4) for k < NV2/2 (float4 loads) plus, when NV2 is odd, the float2 at
// [32*(NV2/2) + 2l, +2).  A warp therefore works on 4 rows per instruction with all 32 lanes
// busy (the generic float4-per-lane layout keeps 20 of 32 lanes busy at C = 80 and spends
// more than half of its issue slots on addressing and predicates).
//
// Same numerics contract as the generic kernels: per-cell sums run in ascending point order
// with separate multiply and add, so the forward is bit-identical to a sequential scatter-add.
#pragma once
#include "common.cuh"

namespace bevpool {


__device__ __forceinline__ float4 ld_stream_or_cached_f4(const char *p, bool stream) {
  return stream ? ldg_stream_f4(reinterpret_cast<const float4 *>(p)) : __ldg(reinterpret_cast<const float4 *>(p));
}

// Row addressing: base pointer made opaque to the optimiser (otherwise it folds the per-sample
// offset back into every row address as a 64-bit multiply chain) + one IMAD.WIDE.U32 per row.
__device__ __forceinline__ const char *opaque_ptr(const void *p) {
  unsigned long long v = reinterpret_cast<unsigned long long>(p);
  asm volatile("" : "+l"(v));
  return reinterpret_cast<const char *>(v);
}
template <int kRowBytes>
__device__ __forceinline__ const char *row_ptr(const char *base, unsigned row) {
  return base + (unsigned long long)row * (unsigned)kRowBytes;
}

// loads the NREG floats of one row for lane l8; `row` points at the row's first byte
template <int NV2, bool kStream>
__device__ __forceinline__ void g8_load_row(const char *row, int l8, float (&v)[2 * NV2]) {
  constexpr int NF4 = NV2 / 2, NF2 = NV2 & 1;
#pragma unroll
  for (int k = 0; k < NF4; ++k) {
    const float4 t = ld_stream_or_cached_f4(row + 128 * k + 16 * l8, kStream);
    v[4 * k + 0] = t.x; v[4 * k + 1] = t.y; v[4 * k + 2] = t.z; v[4 * k + 3] = t.w;
  }
  if (NF2) {
    const float2 t = __ldg(reinterpret_cast<const float2 *>(row + 128 * NF4 + 8 * l8));
    v[4 * NF4 + 0] = t.x; v[4 * NF4 + 1] = t.y;
  }
}

template <int NV2>
__device__ __forceinline__ void g8_store_row(char *row, int l8, const float (&v)[2 * NV2]) {
  constexpr int NF4 = NV2 / 2, NF2 = NV2 & 1;
#pragma unroll
  for (int k = 0; k < NF4; ++k)
    stg_stream_f4(reinterpret_cast<float4 *>(row + 128 * k + 16 * l8),
                  make_float4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]));
  if (NF2) *reinterpret_cast<float2 *>(row + 128 * NF4 + 8 * l8) = make_float2(v[4 * NF4], v[4 * NF4 + 1]);
}

// channel index of register r of lane l8 (for the NCHW context accesses of the backward)
template <int NV2>
__device__ __forceinline__ int g8_channel(int r, int l8) {
  constexpr int NF4 = NV2 / 2;
  return r < 4 * NF4 ? 32 * (r >> 2) + 4 * l8 + (r & 3) : 32 * NF4 + 2 * l8 + (r - 4 * NF4);
}

// ---- shared-memory row access and hinted stores (g8 layout) -------------------------------------
__device__ __forceinline__ void stg_hint_f4(float *p, float4 v, uint64_t pol) {
  asm volatile("st.global.L2::cache_hint.v4.f32 [%0], {%1,%2,%3,%4}, %5;"
               ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "l"(pol) : "memory");
}
__device__ __forceinline__ void stg_hint_f2(float *p, float2 v, uint64_t pol) {
  asm volatile("st.global.L2::cache_hint.v2.f32 [%0], {%1,%2}, %3;" ::"l"(p), "f"(v.x), "f"(v.y), "l"(pol) : "memory");
}

template <int NV2>
__device__ __forceinline__ void g8_lds_row(const float *row, int l8, float (&v)[2 * NV2]) {
  constexpr int NF4 = NV2 / 2, NF2 = NV2 & 1;
#pragma unroll
  for (int k = 0; k < NF4; ++k) {
    const float4 t = *reinterpret_cast<const float4 *>(row + 32 * k + 4 * l8);
    v[4 * k + 0] = t.x; v[4 * k + 1] = t.y; v[4 * k + 2] = t.z; v[4 * k + 3] = t.w;
  }
  if (NF2) {
    const float2 t = *reinterpret_cast<const float2 *>(row + 32 * NF4 + 2 * l8);
    v[4 * NF4 + 0] = t.x; v[4 * NF4 + 1] = t.y;
  }
}

template <int NV2>
__device__ __forceinline__ void g8_store_row_hint(float *row, int l8, const float (&v)[2 * NV2], uint64_t pol) {
  constexpr int NF4 = NV2 / 2, NF2 = NV2 & 1;
#pragma unroll
  for (int k = 0; k < NF4; ++k)
    stg_hint_f4(row + 32 * k + 4 * l8, make_float4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]), pol);
  if (NF2) stg_hint_f2(row + 32 * NF4 + 2 * l8, make_float2(v[4 * NF4], v[4 * NF4 + 1]), pol);
}

template <int NV2>
__device__ __forceinline__ void g8_store_row_plain(float *row, int l8, const float (&v)[2 * NV2]) {
  constexpr int NF4 = NV2 / 2, NF2 = NV2 & 1;
#pragma unroll
  for (int k = 0; k < NF4; ++k)
    *reinterpret_cast<float4 *>(row + 32 * k + 4 * l8) = make_float4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]);
  if (NF2) *reinterpret_cast<float2 *>(row + 32 * NF4 + 2 * l8) = make_float2(v[4 * NF4], v[4 * NF4 + 1]);
}

// two fp32 values rounded to nearest even into one 32-bit word of fp16 / bf16 (fp16: +-inf beyond 65504)
__device__ __forceinline__ uint32_t pack2_rn(__half, float a, float b) {
  const __half2 h = __floats2half2_rn(a, b);
  return *reinterpret_cast<const uint32_t *>(&h);
}
__device__ __forceinline__ uint32_t pack2_rn(__nv_bfloat16, float a, float b) {
  const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<const uint32_t *>(&h);
}

// A finished output row (the only place an output element is rounded): fp32 stored as it is (g8_store_row), fp16 / bf16
// rounded once to nearest even -- lane l8 writes 8 bytes per float4 chunk and 4 bytes for the float2 tail.
template <int NV2, typename TO>
__device__ __forceinline__ void g8_store_out(TO *row, int l8, const float (&v)[2 * NV2]) {
  if constexpr (sizeof(TO) == 4) {
    g8_store_row<NV2>(reinterpret_cast<char *>(row), l8, v);
  } else {
    constexpr int NF4 = NV2 / 2, NF2 = NV2 & 1;
#pragma unroll
    for (int k = 0; k < NF4; ++k)
      *reinterpret_cast<uint2 *>(row + 32 * k + 4 * l8) =
          make_uint2(pack2_rn(TO(), v[4 * k], v[4 * k + 1]), pack2_rn(TO(), v[4 * k + 2], v[4 * k + 3]));
    if (NF2) *reinterpret_cast<uint32_t *>(row + 32 * NF4 + 2 * l8) = pack2_rn(TO(), v[4 * NF4], v[4 * NF4 + 1]);
  }
}

// zeros into elements [4q, 4q + 4) of an output row: one float4, or 8 bytes of a 16-bit type (all-zero bits either way)
template <typename TO>
__device__ __forceinline__ void st_zero4(TO *row, int64_t q) {
  if constexpr (sizeof(TO) == 4) stg_stream_f4(reinterpret_cast<float4 *>(row) + q, make_float4(0.f, 0.f, 0.f, 0.f));
  else reinterpret_cast<uint2 *>(row)[q] = make_uint2(0u, 0u);
}

// ---- packed fp32 math (Blackwell FFMA2 / FADD2: two fp32 lanes per instruction) ---------------
template <int NREG>
__device__ __forceinline__ void axpy_row(float (&acc)[NREG], float a, const float (&v)[NREG]) {
  const float2 a2 = make_float2(a, a);
#pragma unroll
  for (int r = 0; r < NREG; r += 2) {
    const float2 t = __ffma2_rn(a2, make_float2(v[r], v[r + 1]), make_float2(acc[r], acc[r + 1]));
    acc[r] = t.x;
    acc[r + 1] = t.y;
  }
}
template <int NREG>
__device__ __forceinline__ void add_row(float (&acc)[NREG], const float (&v)[NREG]) {
#pragma unroll
  for (int r = 0; r < NREG; r += 2) {
    const float2 t = __fadd2_rn(make_float2(acc[r], acc[r + 1]), make_float2(v[r], v[r + 1]));
    acc[r] = t.x;
    acc[r + 1] = t.y;
  }
}

// ---- forward: even-share segmented reduction over the plan's sorted point list ----------------
// The K kept points, sorted by (cell, point id), are cut into S equal slices (S = 4 x the number
// of warps of a grid that is exactly resident: no scheduling rounds, no tail, and near-camera
// cells that hold 100x the median cannot unbalance anything).  An 8-lane group walks one slice,
// 8 list entries per batch: point id and output row are prefetched two batches ahead, the depth
// gather (whose address needs the id) one batch ahead, 4 context rows are in flight per group.
// A cell whose points all lie inside the slice is stored directly; the partial sums of the (at
// most two) cells cut by the slice's ends go to a workspace and are combined, in slice order,
// by pool_forward_fixup_kernel.  The partition is a pure function of the plan, so the result is
// bit-stable run to run.  Empty cells are zero-filled by the same warps (even share of the grid,
// coalesced 16-byte stores): every output element is written exactly once, no memset.
constexpr int kFwWarpsPerCta = 4;
constexpr int kFwMaxCtasPerSm = 8;

__host__ __device__ __forceinline__ int fwd_slice_len(int K, int num_slices) {
  int L = (int)(((int64_t)K + num_slices - 1) / num_slices);
  L = (L + 7) & ~7;
  return L < 8 ? 8 : L;
}

// kIdent (run plans, stage B): entry k of the list IS row k - e0 of `rows` (the run rows are stored in
// slot order), so no id array is read.  The kernel works on the cells [cell_base, cell_base + total_cells)
// and on the list entries [cell_start[cell_base], cell_start[cell_base + total_cells)); fill_period == 0
// launches no zero-fill CTAs (the caller filled the empty cells elsewhere).
// TO: element type of `out` (fp32, or fp16 / bf16 for run plans: each finished cell is rounded once where it is stored;
// the partial sums in the workspace stay fp32).
template <int NV2, bool kFused, int U, bool kIdent = false, typename TO = float>
__global__ void __launch_bounds__(kFwWarpsPerCta * 32)
pool_forward_share_kernel(const int32_t *__restrict__ cell_start, const int32_t *__restrict__ sorted_ids,
                          const int32_t *__restrict__ sorted_cells, const float *__restrict__ rows,
                          const float *__restrict__ depth, TO *__restrict__ out,
                          float *__restrict__ ws_head, float *__restrict__ ws_tail, int64_t cell_base,
                          int64_t total_cells, FastDiv div_dhw, FastDiv div_hw, int fill_period,
                          int64_t row_capacity, int64_t out_stride) {
  pdl_wait();
  pdl_trigger();
  constexpr int C = 16 * NV2, NREG = 2 * NV2, C4 = C / 4;
  constexpr unsigned kFull = 0xffffffffu;
  const int lane = threadIdx.x & 31, l8 = lane & 7, grp = lane >> 3, warp = threadIdx.x >> 5;
  // Roles: every `fill_period`-th CTA zero-fills the empty cells of the grid (DRAM-write bound) while
  // the other CTAs, co-resident on the same SMs, run the latency-bound reduction.
  const int bid = blockIdx.x;
  if (fill_period > 0 && bid % fill_period == fill_period - 1) {
    const int fwarp = (bid / fill_period) * kFwWarpsPerCta + warp;
    const int nfw = (gridDim.x / fill_period) * kFwWarpsPerCta;
    const int64_t per_warp = ((total_cells + nfw - 1) / nfw + 31) & ~(int64_t)31;
    const int64_t c_begin = cell_base + fwarp * per_warp, c_end = min(cell_base + total_cells, c_begin + per_warp);
    auto load_cs = [&](int64_t c0, int &cs, int &ce) {
      cs = ce = 0;
      if (c0 < c_end) {
        const int ncell = (int)min((int64_t)32, c_end - c0);
        cs = __ldg(cell_start + c0 + min(lane, ncell));
        ce = __ldg(cell_start + c0 + min(lane + 1, ncell));
      }
    };
    int cs, ce, cs_n, ce_n;
    load_cs(c_begin, cs, ce);
    for (int64_t c0 = c_begin; c0 < c_end; c0 += 32) {
      load_cs(c0 + 32, cs_n, ce_n);            // next block's offsets: in flight behind this block's stores
      const int ncell = (int)min((int64_t)32, c_end - c0);
      const unsigned occ = __ballot_sync(kFull, ce > cs);
      if (occ != kFull) {
        if (out_stride == C) {
#pragma unroll 4
          for (int i = lane; i < ncell * C4; i += 32)
            if (!((occ >> (i / C4)) & 1u)) st_zero4(out + c0 * C, i);
        } else {                               // rows inside a wider buffer (concatenated BEV features)
#pragma unroll 4
          for (int i = lane; i < ncell * C4; i += 32)
            if (!((occ >> (i / C4)) & 1u)) st_zero4(out + (c0 + i / C4) * out_stride, i % C4);
        }
      }
      cs = cs_n;
      ce = ce_n;
    }
    return;
  }
  const int rid = fill_period > 0 ? bid - bid / fill_period : bid;
  const int wglobal = rid * kFwWarpsPerCta + warp;
  const int nwarps = (fill_period > 0 ? gridDim.x - gridDim.x / fill_period : gridDim.x) * kFwWarpsPerCta;

  // ---- my slice of the sorted list (entries [e0, K) of it)
  const int e0 = __ldg(cell_start + cell_base);
  // kIdent: never walk past the rows the caller allocated (a stale max_runs hint; stage A raised the plan's status word)
  const int K = (int)min((int64_t)__ldg(cell_start + cell_base + total_cells), kIdent ? (int64_t)e0 + row_capacity : (int64_t)INT32_MAX);
  const int L = fwd_slice_len(K - e0, nwarps * 4);
  const int s = wglobal * 4 + grp;
  const int lo = (int)min((int64_t)e0 + (int64_t)s * L, (int64_t)K), hi = min(lo + L, K);
  const int n0 = __shfl_sync(kFull, hi - lo, 0);            // group 0 has the warp's longest slice
  if (n0 <= 0) return;
  const bool guard = __any_sync(kFull, hi - lo != L);       // only the warp(s) at the very end of the list
  const int nb = (n0 + 7) >> 3;

  const char *rows_b = opaque_ptr(rows);
  auto load_id = [&](int idx) -> int { return idx < K ? (kIdent ? idx - e0 : ldg_stream_i32(sorted_ids + idx)) : -1; };
  auto load_key = [&](int idx) -> int { return idx < K ? ldg_stream_i32(sorted_cells + idx) : -1; };
  auto finish_entry = [&](int id, unsigned &erow, float &ed) {
    erow = 0u;
    ed = 0.f;
    if (id >= 0) {
      const unsigned gp = (unsigned)id;
      if (kFused) {
        const unsigned img = fastdiv(gp, div_dhw);                  // b*N + n
        const unsigned rem = gp - fastdiv(gp, div_hw) * div_hw.div; // h*W + w
        erow = img * div_hw.div + rem;                             // context row of the point's pixel
        ed = ldg_stream_f32(depth + gp);
      } else {
        erow = gp;
      }
    }
  };

  float acc[NREG];
#pragma unroll
  for (int r = 0; r < NREG; ++r) acc[r] = 0.f;

  unsigned row_c, row_n;
  float d_c, d_n;
  int key_c = load_key(lo + l8), key_n = load_key(lo + 8 + l8), key_nn;
  int id_n = load_id(lo + 8 + l8), id_nn;
  finish_entry(load_id(lo + l8), row_c, d_c);
  const int prev_key = lo > e0 ? __ldg(sorted_cells + lo - 1) : -1;
  const int first_key = __shfl_sync(kFull, key_c, 0, 8);   // (all lanes: never short-circuit around a shuffle)
  bool in_head = hi > lo && prev_key == first_key;         // slice starts inside a cell
  unsigned last_gm = 0u;
  float *head_row = ws_head + (size_t)s * C, *tail_row = ws_tail + (size_t)s * C;

  for (int b = 0; b < nb; ++b) {
    const int pos = lo + 8 * b;
    finish_entry(id_n, row_n, d_n);            // batch b+1: its id arrived during batch b-1
    id_nn = load_id(pos + 16 + l8);            // batch b+2
    key_nn = load_key(pos + 16 + l8);
    // entry j closes its cell when the next list entry belongs to another cell
    int nk = __shfl_down_sync(kFull, key_c, 1, 8);
    const int k0n = __shfl_sync(kFull, key_n, 0, 8);
    if (l8 == 7) nk = k0n;
    const bool fl = key_c != nk && (!guard || pos + l8 < hi);
    const unsigned gm = (__ballot_sync(kFull, fl) >> (8 * grp)) & 0xffu;
    if (pos < hi) last_gm = gm;
#pragma unroll
    for (int j0 = 0; j0 < 8; j0 += U) {
      float v[U][NREG];
      float d[U];
      int kk[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const unsigned row = __shfl_sync(kFull, row_c, j0 + u, 8);
        d[u] = __shfl_sync(kFull, d_c, j0 + u, 8);
        kk[u] = __shfl_sync(kFull, key_c, j0 + u, 8);
        if (!guard || pos + j0 + u < hi) {
          g8_load_row<NV2, !kFused>(row_ptr<C * 4>(rows_b, row), l8, v[u]);
        } else {
#pragma unroll
          for (int r = 0; r < NREG; ++r) v[u][r] = 0.f;
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        if (kFused) axpy_row<NREG>(acc, d[u], v[u]); else add_row<NREG>(acc, v[u]);
        if ((gm >> (j0 + u)) & 1u) {
          if (in_head) {
            g8_store_row<NV2>(reinterpret_cast<char *>(head_row), l8, acc);
            in_head = false;
          } else {
            g8_store_out<NV2>(out + (size_t)kk[u] * out_stride, l8, acc);
          }
#pragma unroll
          for (int r = 0; r < NREG; ++r) acc[r] = 0.f;
        }
      }
    }
    row_c = row_n; d_c = d_n; key_c = key_n;
    id_n = id_nn; key_n = key_nn;
  }
  // the last cell continues in the next slice: park the partial sum
  if (hi > lo && !((last_gm >> ((hi - lo - 1) & 7)) & 1u))
    g8_store_row<NV2>(reinterpret_cast<char *>(in_head ? head_row : tail_row), l8, acc);
}

// Combines the partial sums of cells cut by slice boundaries: the slice where such a cell
// begins owns it and adds, in slice order, the head partials of the slices it continues into.
template <int NV2, typename TO = float>
__global__ void __launch_bounds__(128)
pool_forward_fixup_kernel(const int32_t *__restrict__ cell_start, const int32_t *__restrict__ sorted_cells,
                          const float *__restrict__ ws_head, const float *__restrict__ ws_tail,
                          TO *__restrict__ out, int64_t cell_base, int64_t total_cells, int num_slices,
                          int64_t row_capacity, int64_t out_stride) {
  pdl_wait();
  pdl_trigger();
  constexpr int C = 16 * NV2, NREG = 2 * NV2;
  const int s = (blockIdx.x * blockDim.x + threadIdx.x) >> 3, l8 = threadIdx.x & 7;
  if (s >= num_slices) return;
  const int e0 = __ldg(cell_start + cell_base);
  const int K = (int)min((int64_t)__ldg(cell_start + cell_base + total_cells), (int64_t)e0 + row_capacity);
  const int L = fwd_slice_len(K - e0, num_slices);
  const int lo = (int)min((int64_t)e0 + (int64_t)s * L, (int64_t)K), hi = min(lo + L, K);
  if (hi <= lo || hi >= K) return;
  const int key = __ldg(sorted_cells + hi - 1);
  if (key != __ldg(sorted_cells + hi)) return;                      // slice ends on a cell boundary
  if (lo > e0 && __ldg(sorted_cells + lo - 1) == key) return;       // cell began in an earlier slice
  float acc[NREG], v[NREG];
  g8_load_row<NV2, false>(reinterpret_cast<const char *>(ws_tail + (size_t)s * C), l8, acc);
  for (int t = s + 1; t < num_slices; ++t) {
    const int tlo = e0 + t * L, thi = min(tlo + L, K);              // tlo < K because slice t-1 ended mid-cell
    g8_load_row<NV2, false>(reinterpret_cast<const char *>(ws_head + (size_t)t * C), l8, v);
#pragma unroll
    for (int r = 0; r < NREG; ++r) acc[r] += v[r];
    if (!(thi < K && __ldg(sorted_cells + thi - 1) == key && __ldg(sorted_cells + thi) == key)) break;
  }
  g8_store_out<NV2>(out + (size_t)key * out_stride, l8, acc);
}

inline bool g8_supported(int C) {
  return C == 32 || C == 64 || C == 80 || C == 96 || C == 128;
}

#define BEVPOOL_G8_DISPATCH(C, CALL)                    \
  switch (C) {                                          \
    case 32: { constexpr int NV2 = 2; CALL; break; }    \
    case 64: { constexpr int NV2 = 4; CALL; break; }    \
    case 80: { constexpr int NV2 = 5; CALL; break; }    \
    case 96: { constexpr int NV2 = 6; CALL; break; }    \
    case 128: { constexpr int NV2 = 8; CALL; break; }   \
    default: return BEVPOOL_E_CHANNELS;                 \
  }

}  // namespace bevpool

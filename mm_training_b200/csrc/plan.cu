// Pooling plan: per-point BEV cell index + deterministic (stable) sort of the kept
// points by cell, giving a CSR (cell_start, sorted_ids) that every reduction kernel
// walks in a fixed order.  Replaces the index half of the reference kernel
// (ops/voxel_pooling/src/voxel_pooling_forward_cuda.cu:19-29) and removes the need
// for its atomicAdd (:30-34).
//
// Algorithm: per-sample LSD radix sort on the in-sample cell id (y*X + x), 2 passes
// for grids up to 2^20 cells.  Dropped points are compacted away in pass 0, so the
// sort moves K (kept) pairs, not P.  Each pass = tile histogram -> one decoupled
// look-back scan over [sample][digit][tile] -> stable scatter (warp match-any ranks).
// The sort is stable, so points of one cell stay in ascending point order: the same
// order the reference test's golden loop and torch.index_add_ visit them in.
#include "common.cuh"
#include "scan.cuh"

#include <cstdlib>

namespace bevpool {

std::atomic<long long> g_kernel_launches{0};

bool pdl_forward_enabled() {
  static const bool on = [] { const char *e = std::getenv("BEVPOOL_PDL_FWD"); return e && e[0] == '1'; }();
  return on;
}

bool pdl_enabled() {
  static const bool on = [] { const char *e = std::getenv("BEVPOOL_PDL"); return !(e && e[0] == '0'); }();
  return on;
}

static PlanHeader make_plan_header(int32_t kind, int batch, int64_t num_points, int X, int Y, int Z) {
  PlanHeader h{};
  h.magic = kPlanMagic; h.kind = kind; h.status = 0; h.batch = batch;
  h.num_voxel_x = X; h.num_voxel_y = Y; h.num_voxel_z = Z; h.num_points = num_points;
  return h;
}

constexpr int kSortThreads = 256;
constexpr int kSortWarps = kSortThreads / 32;
constexpr int kSortItems = 8;
constexpr int kSortTile = kSortThreads * kSortItems;  // 2048 keys per CTA
constexpr int kMaxPasses = 3;

struct SortConfig {
  int npass;
  int bits[kMaxPasses];
  int shift[kMaxPasses];
  bool msd;            // bits[0] = low (finished per bucket in shared memory), bits[1] = high (global pass)
};

static SortConfig sort_config(int64_t cells_per_sample) {
  int nbits = 1;
  while ((1ll << nbits) < cells_per_sample) ++nbits;
  SortConfig c;
  c.msd = false;
  if (nbits > 8 && nbits <= 18) {
    c.msd = true;
    c.npass = 2;
    c.bits[0] = 8;          c.shift[0] = 0;
    c.bits[1] = nbits - 8;  c.shift[1] = 8;
    c.bits[2] = 0;          c.shift[2] = nbits;
    return c;
  }
  c.npass = (nbits + 9) / 10;
  const int per = (nbits + c.npass - 1) / c.npass;
  int shift = 0;
  for (int p = 0; p < kMaxPasses; ++p) {
    c.bits[p] = p < c.npass ? (nbits - shift < per ? nbits - shift : per) : 0;
    if (p < c.npass && c.bits[p] < 1) c.bits[p] = 1;
    c.shift[p] = shift;
    shift += c.bits[p];
  }
  return c;
}

struct TempLayout {
  size_t off_scan[kMaxPasses + 1];  // scan workspaces: one per pass + cell counts
  size_t off_hist[kMaxPasses];      // tile histograms [sample][digit][tile] (+1 total)
  size_t zero_bytes;                // everything above is memset to 0 per build
  size_t off_keys[2], off_ids[2];   // ping-pong buffers for passes before the last
  size_t bytes;
  int64_t hist_n[kMaxPasses];
  int tiles_per_sample;
};

static TempLayout temp_layout(int batch, int64_t num_points, int X, int Y) {
  const SortConfig sc = sort_config((int64_t)X * Y);
  TempLayout L{};
  L.tiles_per_sample = (int)ceil_div64(num_points, kSortTile);
  size_t o = 0;
  for (int p = 0; p < kMaxPasses; ++p) {
    L.hist_n[p] = p < sc.npass ? (int64_t)batch * (1ll << sc.bits[p]) * L.tiles_per_sample + 1 : 0;
  }
  if (sc.msd) {   // one global pass, over the HIGH bits; the low bits never get a global histogram
    L.hist_n[0] = (int64_t)batch * (1ll << sc.bits[1]) * L.tiles_per_sample + 1;
    L.hist_n[1] = 1;
  }
  for (int p = 0; p < sc.npass; ++p) {
    L.off_scan[p] = o;
    o += scan_workspace_bytes(L.hist_n[p]);
  }
  L.off_scan[kMaxPasses] = o;
  o += scan_workspace_bytes((int64_t)batch * X * Y + 1);
  for (int p = 0; p < sc.npass; ++p) {
    L.off_hist[p] = o;
    o = align_up(o + (size_t)L.hist_n[p] * 4, 256);
  }
  L.zero_bytes = o;
  const size_t P = (size_t)batch * (size_t)num_points;
  const int nbuf = sc.npass >= 3 ? 2 : (sc.npass == 2 ? 1 : 0);
  for (int i = 0; i < 2; ++i) {
    L.off_keys[i] = o;
    if (i < nbuf) o = align_up(o + P * 4, 256);
    L.off_ids[i] = o;
    if (i < nbuf) o = align_up(o + P * 4, 256);
  }
  L.bytes = o > 256 ? o : 256;
  return L;
}

// ---- kernel 1: cell index, per-cell counts, pass-0 tile histogram --------------------
__global__ void __launch_bounds__(kSortThreads)
plan_key_kernel(const int32_t *__restrict__ geom, int64_t num_points, int X, int Y, int Z,
                int32_t *__restrict__ cell_of_point, uint32_t *__restrict__ cell_count,
                uint32_t *__restrict__ hist, int bins, int tiles_per_sample, PlanHeader *hdr, PlanHeader hv) {
  extern __shared__ uint32_t s_hist[];
  const int b = blockIdx.y, tile = blockIdx.x;
  if (b == 0 && tile == 0 && threadIdx.x == 0) *hdr = hv;
  for (int i = threadIdx.x; i < bins; i += kSortThreads) s_hist[i] = 0u;
  __syncthreads();
  const int64_t sample_base = (int64_t)b * num_points;
  const int64_t cells = (int64_t)X * Y;
  const int64_t tile_base = (int64_t)tile * kSortTile;
#pragma unroll
  for (int i = 0; i < kSortItems; ++i) {
    const int64_t p = tile_base + i * kSortThreads + threadIdx.x;
    if (p < num_points) {
      const int64_t gp = sample_base + p;
      const int x = __ldg(geom + gp * 3 + 0);
      const int y = __ldg(geom + gp * 3 + 1);
      const int z = __ldg(geom + gp * 3 + 2);
      // reference bounds test, voxel_pooling_forward_cuda.cu:24; z gates only (:32-33)
      const bool kept = x >= 0 && x < X && y >= 0 && y < Y && z >= 0 && z < Z;
      const int cell = kept ? y * X + x : -1;
      cell_of_point[gp] = cell;
      if (kept) {
        atomicAdd(cell_count + (int64_t)b * cells + cell, 1u);
        atomicAdd(s_hist + (cell & (bins - 1)), 1u);
      }
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < bins; i += kSortThreads)
    hist[((int64_t)b * bins + i) * tiles_per_sample + tile] = s_hist[i];
}

// ---- tile histogram of a later pass (input already compacted per sample) ---------------
__global__ void __launch_bounds__(kSortThreads)
sort_hist_kernel(const int32_t *__restrict__ keys, const uint32_t *__restrict__ scanned0, int bins0,
                 int shift, int bins, int tiles_per_sample, uint32_t *__restrict__ hist) {
  extern __shared__ uint32_t s_hist[];
  const int b = blockIdx.y, tile = blockIdx.x;
  const int64_t seg_begin = scanned0[(int64_t)b * bins0 * tiles_per_sample];
  const int64_t seg_end = scanned0[(int64_t)(b + 1) * bins0 * tiles_per_sample];
  const int64_t tile_begin = seg_begin + (int64_t)tile * kSortTile;
  if (tile_begin >= seg_end) return;
  for (int i = threadIdx.x; i < bins; i += kSortThreads) s_hist[i] = 0u;
  __syncthreads();
#pragma unroll
  for (int i = 0; i < kSortItems; ++i) {
    const int64_t idx = tile_begin + i * kSortThreads + threadIdx.x;
    if (idx < seg_end) atomicAdd(s_hist + ((keys[idx] >> shift) & (bins - 1)), 1u);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < bins; i += kSortThreads)
    hist[((int64_t)b * bins + i) * tiles_per_sample + tile] = s_hist[i];
}

// ---- stable scatter of one radix pass ---------------------------------------------------
// Element order inside a CTA is (warp, round, lane) == ascending input index, so ranks
// handed out in that order keep the sort stable.
template <bool kFirst>
__global__ void __launch_bounds__(kSortThreads)
sort_scatter_kernel(const int32_t *__restrict__ in_keys, const int32_t *__restrict__ in_ids,
                    int32_t *__restrict__ out_keys, int32_t *__restrict__ out_ids,
                    int32_t *__restrict__ out_rows, int32_t cells_per_sample,
                    const uint32_t *__restrict__ scanned, const uint32_t *__restrict__ scanned0,
                    int bins0, int64_t num_points, int shift, int bins, int tiles_per_sample) {
  extern __shared__ uint32_t s_cnt[];  // [kSortWarps][bins]
  const int b = blockIdx.y, tile = blockIdx.x;
  int64_t seg_begin, seg_end;
  if (kFirst) {
    seg_begin = (int64_t)b * num_points;
    seg_end = seg_begin + num_points;
  } else {
    seg_begin = scanned0[(int64_t)b * bins0 * tiles_per_sample];
    seg_end = scanned0[(int64_t)(b + 1) * bins0 * tiles_per_sample];
  }
  const int64_t tile_begin = seg_begin + (int64_t)tile * kSortTile;
  if (tile_begin >= seg_end) return;

  for (int i = threadIdx.x; i < kSortWarps * bins; i += kSortThreads) s_cnt[i] = 0u;
  __syncthreads();

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t *cnt = s_cnt + warp * bins;
  const int64_t warp_begin = tile_begin + warp * (kSortItems * 32);
  int32_t key[kSortItems], id[kSortItems];
  uint32_t rank[kSortItems];
#pragma unroll
  for (int r = 0; r < kSortItems; ++r) {
    const int64_t idx = warp_begin + r * 32 + lane;
    const bool in_range = idx < seg_end;
    key[r] = in_range ? in_keys[idx] : -1;
    id[r] = kFirst ? (int32_t)idx : (in_range ? in_ids[idx] : -1);
  }
#pragma unroll
  for (int r = 0; r < kSortItems; ++r) {
    const bool valid = key[r] >= 0;
    const uint32_t digit = valid ? (uint32_t)((key[r] >> shift) & (bins - 1)) : (uint32_t)bins;
    const unsigned peers = __match_any_sync(0xffffffffu, digit);
    const int leader = __ffs(peers) - 1;
    uint32_t base = 0;
    if (valid && lane == leader) {
      base = cnt[digit];
      cnt[digit] = base + __popc(peers);
    }
    base = __shfl_sync(0xffffffffu, base, leader);
    rank[r] = base + __popc(peers & ((1u << lane) - 1u));
    __syncwarp();
  }
  __syncthreads();
  for (int bin = threadIdx.x; bin < bins; bin += kSortThreads) {
    uint32_t run = scanned[((int64_t)b * bins + bin) * tiles_per_sample + tile];
#pragma unroll
    for (int w = 0; w < kSortWarps; ++w) {
      const uint32_t t = s_cnt[w * bins + bin];
      s_cnt[w * bins + bin] = run;
      run += t;
    }
  }
  __syncthreads();
#pragma unroll
  for (int r = 0; r < kSortItems; ++r) {
    if (key[r] >= 0) {
      const uint32_t digit = (uint32_t)((key[r] >> shift) & (bins - 1));
      const uint32_t pos = cnt[digit] + rank[r];
      out_ids[pos] = id[r];
      if (out_keys) out_keys[pos] = key[r];
      if (out_rows) out_rows[pos] = b * cells_per_sample + key[r];   // last pass: global output row
    }
  }
}

// ==== MSD fast path (grids of 2^9 .. 2^16 cells per sample) ====================================
// pass A (plan_key_msd_kernel): cell index of every point + tile histogram of the HIGH key bits
// pass B (sort_scatter_kernel<true>): stable scatter of the kept (cell, id) pairs into buckets of
//         2^low consecutive cells (one look-back scan over [sample][bucket][tile] in between)
// pass C (bucket_sort_kernel): one CTA per (sample, bucket) finishes the sort locally -- histogram of
//         the low bits in shared memory, CSR offsets of its 2^low cells, stable placement -- so the
//         second global histogram, its scan, the per-cell atomics and the CSR scan of the LSD path
//         are not needed.
// geom is read as 16-byte vectors: a thread owns 4 consecutive points = 48 bytes.
__global__ void __launch_bounds__(kSortThreads)
plan_key_msd_kernel(const int32_t *__restrict__ geom, int64_t num_points, int X, int Y, int Z,
                    int32_t *__restrict__ cell_of_point, uint32_t *__restrict__ hist, int low_bits,
                    int bins, int tiles_per_sample, PlanHeader *hdr, PlanHeader hv) {
  extern __shared__ uint32_t s_hist[];
  const int b = blockIdx.y, tile = blockIdx.x;
  if (b == 0 && tile == 0 && threadIdx.x == 0) *hdr = hv;
  for (int i = threadIdx.x; i < bins; i += kSortThreads) s_hist[i] = 0u;
  __syncthreads();
  const int64_t sample_base = (int64_t)b * num_points;
  const int64_t tile_base = (int64_t)tile * kSortTile;
  const bool vec = ((sample_base + tile_base) & 3) == 0;   // 16-byte alignment of the quad loads
#pragma unroll
  for (int q = 0; q < kSortItems / 4; ++q) {
    const int64_t p0 = tile_base + ((int64_t)q * kSortThreads + threadIdx.x) * 4;
    if (p0 >= num_points) continue;
    const int64_t gp0 = sample_base + p0;
    int c[12];
    if (vec && p0 + 3 < num_points) {
      const int4 *src = reinterpret_cast<const int4 *>(geom + gp0 * 3);
      const int4 a0 = ldg_stream_i4(src), a1 = ldg_stream_i4(src + 1), a2 = ldg_stream_i4(src + 2);
      c[0] = a0.x; c[1] = a0.y; c[2] = a0.z; c[3] = a0.w; c[4] = a1.x; c[5] = a1.y;
      c[6] = a1.z; c[7] = a1.w; c[8] = a2.x; c[9] = a2.y; c[10] = a2.z; c[11] = a2.w;
    } else {
#pragma unroll
      for (int k = 0; k < 12; ++k) c[k] = (p0 + k / 3 < num_points) ? __ldg(geom + gp0 * 3 + k) : -1;
    }
    int cell[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int x = c[3 * k], y = c[3 * k + 1], z = c[3 * k + 2];
      // reference bounds test, voxel_pooling_forward_cuda.cu:24; z gates only (:32-33)
      const bool kept = x >= 0 && x < X && y >= 0 && y < Y && z >= 0 && z < Z && p0 + k < num_points;
      cell[k] = kept ? y * X + x : -1;
      if (kept) atomicAdd(s_hist + (cell[k] >> low_bits), 1u);
    }
    if (vec && p0 + 3 < num_points) {
      *reinterpret_cast<int4 *>(cell_of_point + gp0) = make_int4(cell[0], cell[1], cell[2], cell[3]);
    } else {
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (p0 + k < num_points) cell_of_point[gp0 + k] = cell[k];
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < bins; i += kSortThreads)
    hist[((int64_t)b * bins + i) * tiles_per_sample + tile] = s_hist[i];
}

// ==== run plans ===================================================================================
// Points are enumerated (n, d, h, w); the vertical predecessor of point p is p - W.  A kept point starts
// a run when it is the first row of a kRunHB-row block or its predecessor lies in another cell (or was
// dropped).  Only run heads are sorted -- 11x fewer entries than kept points at the aiMotive shape -- and
// with so few entries a radix sort is mostly launch and latency overhead.  Instead:
//   K1 plan_key_runs_kernel   cell index, run_code, per-cell run counts (integer atomicAdd), and every
//                             warp's run heads compacted into its own slice of a (cell, id) list
//   K2 scan_exclusive_kernel  counts -> cell_start (CSR over runs)
//   K3 run_place_kernel       head -> some position of its cell's segment (atomic cursor: arbitrary order)
//   K4 run_finish_kernel      one thread per cell: orders the segment by point id (median 2 runs per cell),
//                             writes sorted_ids / sorted_cells and each head's slot into run_code
// The result does not depend on the order the atomics happened in: a deterministic, stable sort.
__device__ __forceinline__ int cell_of_xyz(int x, int y, int z, int X, int Y, int Z) {
  // reference bounds test, voxel_pooling_forward_cuda.cu:24; z gates only (:32-33).  0 <= v < N as ONE unsigned compare.
  const bool kept = ((unsigned)x < (unsigned)X) & ((unsigned)y < (unsigned)Y) & ((unsigned)z < (unsigned)Z);
  return kept ? y * X + x : -1;
}

// ==== run plan straight from the camera rig (no geom_xyz tensor) ===================================
// Replaces layers/backbones/lss_fpn.py:328-361 (get_geometry) + :461-462 (quantisation) of the reference as
// the producer of the cell indices: the (B, N, D, H, W, 3) float and int32 tensors are never written or read.
// What stays in torch is what is tiny: combine = sensor2ego @ inverse(intrin) (B*N matrices), the frustum
// axes and the two 3-vectors of the quantisation.  Per point, op for op what the reference's ATen ops do:
//   p = (x*d, y*d, d, 1)                                   (:351-353, float32 multiply)
//   e = combine @ p                                        (:355, rows 0..2; the 4-term dot product in the
//                                                           accumulation order selected by kVariant)
//   q = ((e - (voxel_coord - voxel_size/2)) / voxel_size).int()   (:461-462: IEEE subtract, TRUE division,
//                                                           truncation toward zero)
// Which accumulation order reproduces the reference's batched matmul bit for bit depends on the BLAS kernel
// behind it; the host picks the variant by comparing against torch on the device in use (and falls back to
// the geom_xyz path if none matches): mm_training_b200/ops/voxel_pooling/rig.py.
// Thread = one (image, depth bin, 16-row block, column) pair, walking its rows top to bottom, so run heads
// are found without re-deriving the row above; lanes = consecutive columns (coalesced 4-byte stores).
struct RigParams {
  const float *combine;          // (B*N, 4, 4) row-major
  const float *fx, *fy, *fd;     // frustum axes: x[W], y[H], d[D]  (lss_fpn.py:308-326)
  float lo[3], vs[3], inv_vs[3]; // voxel_coord - voxel_size/2, voxel_size, 1/voxel_size (fast path only)
};

template <int kVariant>
__device__ __forceinline__ float rig_dot4(const float (&m)[4], float px, float py, float pz) {
  // the homogeneous coordinate is exactly 1.0f, so m[3] * 1 == m[3]
  if (kVariant == 0) {          // ascending k, fused multiply-add
    float a = __fmul_rn(m[0], px);
    a = __fmaf_rn(m[1], py, a);
    a = __fmaf_rn(m[2], pz, a);
    return __fadd_rn(a, m[3]);
  } else if (kVariant == 1) {   // descending k, fused multiply-add
    float a = __fmaf_rn(m[2], pz, m[3]);
    a = __fmaf_rn(m[1], py, a);
    return __fmaf_rn(m[0], px, a);
  } else if (kVariant == 2) {   // two k-slices (0,1) + (2,3), each an ascending fused chain that starts from a rounded product
    const float a = __fmaf_rn(m[1], py, __fmul_rn(m[0], px));
    const float b = __fadd_rn(__fmul_rn(m[2], pz), m[3]);
    return __fadd_rn(a, b);
  } else if (kVariant == 3) {   // ascending k, separate multiply and add
    return __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(m[0], px), __fmul_rn(m[1], py)), __fmul_rn(m[2], pz)), m[3]);
  } else if (kVariant == 4) {   // even / odd k-slices (0,2) + (1,3)
    const float a = __fmaf_rn(m[2], pz, __fmul_rn(m[0], px));
    const float b = __fadd_rn(__fmul_rn(m[1], py), m[3]);
    return __fadd_rn(a, b);
  } else {                      // pairwise with the translation fused into the second product
    const float a = __fmaf_rn(m[1], py, __fmul_rn(m[0], px));
    const float b = __fmaf_rn(m[2], pz, m[3]);
    return __fadd_rn(a, b);
  }
}

// trunc((e - lo) / vs) with IEEE semantics; a NaN, infinite or int32-overflowing quotient gives INT_MIN, which every
// bounds test drops.  q' = (e - lo) * fl(1 / vs) differs from the correctly rounded quotient by at most 3 * 2^-24 |q|
// (one rounding each on 1 / vs, on q' and on the quotient), i.e. by less than 7.3e-4 while |q'| < 4096: when q' is
// farther than 1e-3 from every integer both truncate to the same value; otherwise (a fraction of a percent of the
// points at shipped shapes, and every quotient from 4096 up) the exact division decides.  rig_quantise3 does the three
// coordinates of a point with ONE branch to the exact path.
__device__ __forceinline__ int rig_trunc_exact(float t, float vs) {
  const float q = __fdiv_rn(t, vs);
  return fabsf(q) < 2147483648.f ? __float2int_rz(q) : INT_MIN;     // NaN compares false
}
__device__ __forceinline__ int rig_quantise(float e, float lo, float vs, float inv_vs) {
  const float t = __fsub_rn(e, lo);
  const float qf = __fmul_rn(t, inv_vs);
  const float fr = fabsf(qf - rintf(qf));
  if (fr > 1e-3f && fabsf(qf) < 4096.f) return __float2int_rz(qf);   // NaN / inf q' give a NaN fr: exact path
  return rig_trunc_exact(t, vs);
}
__device__ __forceinline__ void rig_quantise3(float ex, float ey, float ez, const RigParams &rp, int &ix, int &iy, int &iz) {
  const float tx = __fsub_rn(ex, rp.lo[0]), ty = __fsub_rn(ey, rp.lo[1]), tz = __fsub_rn(ez, rp.lo[2]);
  const float qx = __fmul_rn(tx, rp.inv_vs[0]), qy = __fmul_rn(ty, rp.inv_vs[1]), qz = __fmul_rn(tz, rp.inv_vs[2]);
  const float fx = fabsf(qx - rintf(qx)), fy = fabsf(qy - rintf(qy)), fz = fabsf(qz - rintf(qz));
  const float big = fmaxf(fmaxf(fabsf(qx), fabsf(qy)), fabsf(qz));
  // A NaN or infinite q' has a NaN fraction.  fminf / fmaxf drop a NaN operand, so each fraction is compared on its
  // own: a NaN fails its comparison and the point takes the exact path.
  if (fx > 1e-3f && fy > 1e-3f && fz > 1e-3f && big < 4096.f) {
    ix = __float2int_rz(qx);
    iy = __float2int_rz(qy);
    iz = __float2int_rz(qz);
  } else {
    ix = rig_trunc_exact(tx, rp.vs[0]);
    iy = rig_trunc_exact(ty, rp.vs[1]);
    iz = rig_trunc_exact(tz, rp.vs[2]);
  }
}

constexpr int kRigThreads = 256;

// kVariant >= 0: cells from the rig (RigParams); kVariant == -1: cells from the caller's geom_xyz tensor (same walk:
// lanes = consecutive columns, so the 12-byte points of a row are read as one 384-byte span per warp).
template <int kVariant>
__global__ void __launch_bounds__(kRigThreads)
plan_key_rig_kernel(RigParams rp, const int32_t *__restrict__ geom, int num_cams, int D, int H, int W, int HB, int X, int Y,
                    int Z, int64_t num_points,
                    int32_t *__restrict__ cell_of_point, int32_t *__restrict__ run_code, uint32_t *__restrict__ counts,
                    int32_t *__restrict__ head_cells, int32_t *__restrict__ head_ids, int32_t *__restrict__ warp_count,
                    uint32_t *__restrict__ sample_total, int warps_per_sample, int slot_cap, int4 *__restrict__ pair_rec,
                    PlanHeader *hdr, PlanHeader hv) {
  pdl_wait();
  pdl_trigger();
  const int b = blockIdx.y;
  if (b == 0 && blockIdx.x == 0 && threadIdx.x == 0) *hdr = hv;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t pairs = (int64_t)num_cams * D * HB * W;
  const int64_t q = (int64_t)blockIdx.x * kRigThreads + threadIdx.x;
  const bool valid = q < pairs;
  int w = 0, hb = 0, d = 0, n = 0;
  if (valid) {
    int64_t t = q;
    w = (int)(t % W); t /= W;
    hb = (int)(t % HB); t /= HB;
    d = (int)(t % D);
    n = (int)(t / D);
  }
  float m0[4] = {0.f, 0.f, 0.f, 0.f}, m1[4] = {0.f, 0.f, 0.f, 0.f}, m2[4] = {0.f, 0.f, 0.f, 0.f};
  float dd = 0.f, px = 0.f;
  if (kVariant >= 0) {
    const float4 *mp = reinterpret_cast<const float4 *>(rp.combine + ((int64_t)b * num_cams + n) * 16);
    const float4 r0 = __ldg(mp), r1 = __ldg(mp + 1), r2 = __ldg(mp + 2);
    m0[0] = r0.x; m0[1] = r0.y; m0[2] = r0.z; m0[3] = r0.w;
    m1[0] = r1.x; m1[1] = r1.y; m1[2] = r1.z; m1[3] = r1.w;
    m2[0] = r2.x; m2[1] = r2.y; m2[2] = r2.z; m2[3] = r2.w;
    dd = __ldg(rp.fd + d);
    px = __fmul_rn(__ldg(rp.fx + w), dd);
  }
  const int64_t cells = (int64_t)X * Y;
  const int64_t region = ((int64_t)b * warps_per_sample + (int64_t)blockIdx.x * (kRigThreads / 32) + warp) * slot_cap;
  const int col_base = (int)((int64_t)b * num_points + ((int64_t)n * D + d) * H * W + w);     // B * Np < 2^31 (host check)
  const unsigned lt = (1u << lane) - 1u;
  uint32_t filled = 0;                 // heads this warp has written so far (warp-uniform)
  int prev = -2, primary = -1, nheads = 0;
  uint32_t fastm = 0u, keptm = 0u;

  // ---- level-camera fast path (rig plans).  Every coordinate of a point is a weakly MONOTONE function of its image
  // row h: py = fy[h] * d enters each dot product once, and fl(.) of a monotone function is monotone through every
  // rounding step (multiply, fused multiply-add, add, subtract, divide by a constant, truncate).  So when the x and y
  // cell indices agree at the first and the last row of a pair they agree on every row in between (a level camera:
  // m[.][1] == 0 for x and y), and the rows whose z index lies in [0, Z) form ONE interval, found by two binary
  // searches on z alone: ~10 coordinate evaluations per pair instead of 48, one head, no per-row voting.  Bit-identical
  // to the per-row walk below by construction; it needs fy sorted (checked per CTA) and end points below 1e30.  A warp
  // takes it only when all its pairs qualify; tilted cameras and geom_xyz plans walk the rows.
  bool warp_fast = false;
  if (kVariant >= 0) {
    __shared__ int s_unsorted;
    if (threadIdx.x == 0) s_unsorted = 0;
    __syncthreads();
    for (int i = threadIdx.x; i + 1 < H; i += kRigThreads)
      if (!(__ldg(rp.fy + i) <= __ldg(rp.fy + i + 1))) s_unsorted = 1;
    __syncthreads();
    const int rows_here = valid ? min(kRunHB, H - hb * kRunHB) : 0;
    constexpr int V = kVariant < 0 ? 0 : kVariant;
    int ix0 = 0, iy0 = 0, iz0 = 0, ix1 = 0, iy1 = 0, iz1 = 0;
    bool fast = s_unsorted == 0;
    if (valid && fast) {
      const float pya = __fmul_rn(__ldg(rp.fy + hb * kRunHB), dd), pyb = __fmul_rn(__ldg(rp.fy + hb * kRunHB + rows_here - 1), dd);
      const float ea0 = rig_dot4<V>(m0, px, pya, dd), ea1 = rig_dot4<V>(m1, px, pya, dd), ea2 = rig_dot4<V>(m2, px, pya, dd);
      const float eb0 = rig_dot4<V>(m0, px, pyb, dd), eb1 = rig_dot4<V>(m1, px, pyb, dd), eb2 = rig_dot4<V>(m2, px, pyb, dd);
      const float big = fmaxf(fmaxf(fmaxf(fabsf(ea0), fabsf(ea1)), fmaxf(fabsf(ea2), fabsf(eb0))), fmaxf(fabsf(eb1), fabsf(eb2)));
      rig_quantise3(ea0, ea1, ea2, rp, ix0, iy0, iz0);
      rig_quantise3(eb0, eb1, eb2, rp, ix1, iy1, iz1);
      // big < 1e30f sends end points that overflowed to +-inf down the walk; fmaxf drops a NaN operand, so it does not
      // see NaN.  A NaN end point gets INT_MIN from rig_quantise3 instead.  A NaN or inf needs a non-finite entry in
      // its combine row, which makes that coordinate non-finite -- INT_MIN -- on every row, so the pair is dropped
      // here exactly as the walk drops each row.
      fast = big < 1e30f && ix0 == ix1 && iy0 == iy1;
    }
    warp_fast = __all_sync(0xffffffffu, fast);
    if (warp_fast) {
      int lo = 0, hi = 0;                                       // kept rows of the pair: [lo, hi)
      const bool xy_ok = valid && ((unsigned)ix0 < (unsigned)X) && ((unsigned)iy0 < (unsigned)Y);
      if (xy_ok) {
        if (iz0 == iz1) {
          if ((unsigned)iz0 < (unsigned)Z) hi = rows_here;
        } else {
          const bool asc = iz0 < iz1;                           // z index as a function of the row: ascending or descending
          auto zi = [&](int k) {                                // ascending view: k-th row from the low-z end
            const int r = asc ? k : rows_here - 1 - k;
            const float py = __fmul_rn(__ldg(rp.fy + hb * kRunHB + r), dd);
            return rig_quantise(rig_dot4<V>(m2, px, py, dd), rp.lo[2], rp.vs[2], rp.inv_vs[2]);
          };
          auto lower_bound = [&](int thr) {                     // first k with zi(k) >= thr (zi(0) = min end, zi(rows-1) = max end)
            int a = 0, e = rows_here;
            while (a < e) {
              const int mid = (a + e) >> 1;
              if (zi(mid) >= thr) e = mid; else a = mid + 1;
            }
            return a;
          };
          const int ka = lower_bound(0), kb = lower_bound(Z);   // kept (ascending view) = [ka, kb)
          if (asc) { lo = ka; hi = kb; } else { lo = rows_here - kb; hi = rows_here - ka; }
        }
      }
      const bool has = hi > lo;
      const int cell = has ? iy0 * X + ix0 : -1;
      if (valid) {
#pragma unroll 4
        for (int r = 0; r < rows_here; ++r) {
          const int gp = col_base + (hb * kRunHB + r) * W;
          const bool kept = r >= lo && r < hi;
          cell_of_point[gp] = kept ? cell : -1;
          run_code[gp] = kept ? (r == lo ? cell : kRunCont) : kRunDropped;     // the head: overwritten with its slot by K4
        }
      }
      const unsigned bal = __ballot_sync(0xffffffffu, has);
      if (has) {
        const int64_t pos = region + __popc(bal & lt);
        head_cells[pos] = cell;
        head_ids[pos] = (col_base + (hb * kRunHB + lo) * W) | (int32_t)0x80000000;   // first kept row of its pair
        atomicAdd(counts + (int64_t)b * cells + cell, 1u);
        primary = cell;
        keptm = fastm = ((hi - lo >= 32 ? 0u : (1u << (hi - lo))) - 1u) << lo;
        nheads = 1;
      }
      filled = __popc(bal);
    }
  }
  if (!warp_fast) {
#pragma unroll 4
  for (int r = 0; r < kRunHB; ++r) {
    const int h = hb * kRunHB + r;
    const bool act = valid && h < H;
    int cell = -1, code = kRunDropped;
    if (act) {
      const int gp = col_base + h * W;
      int ix, iy, iz;
      if (kVariant >= 0) {
        const float py = __fmul_rn(__ldg(rp.fy + h), dd);
        rig_quantise3(rig_dot4<(kVariant < 0 ? 0 : kVariant)>(m0, px, py, dd), rig_dot4<(kVariant < 0 ? 0 : kVariant)>(m1, px, py, dd),
                      rig_dot4<(kVariant < 0 ? 0 : kVariant)>(m2, px, py, dd), rp, ix, iy, iz);
      } else {
        const int32_t *g = geom + (int64_t)gp * 3;
        ix = __ldg(g);
        iy = __ldg(g + 1);
        iz = __ldg(g + 2);
      }
      cell = cell_of_xyz(ix, iy, iz, X, Y, Z);
      code = cell < 0 ? kRunDropped : (cell != prev ? cell : kRunCont);
      prev = cell;
      cell_of_point[gp] = cell;
      run_code[gp] = code;          // heads: overwritten with their slot by K4
      if (cell >= 0) {
        if (primary < 0) primary = cell;
        keptm |= 1u << r;
        if (cell == primary) fastm |= 1u << r;
        nheads += code >= 0;
      }
    }
    const bool head = code >= 0;
    const unsigned bal = __ballot_sync(0xffffffffu, head);
    if (head) {
      const int64_t pos = region + filled + __popc(bal & lt);
      head_cells[pos] = code;
      // bit 31: this head is the first kept row of its pair (K4 then records its slot in the pair record)
      head_ids[pos] = (col_base + h * W) | (keptm == (1u << r) ? (int32_t)0x80000000 : 0);
      atomicAdd(counts + (int64_t)b * cells + code, 1u);
    }
    filled += __popc(bal);
  }
  }
  if (valid) pair_rec[(int64_t)b * pairs + q] = make_int4(primary, (int)(fastm | ((keptm & ~fastm) << 16)), -1, nheads);
  __shared__ uint32_t s_cta_total;
  if (threadIdx.x == 0) s_cta_total = 0u;
  __syncthreads();
  if (lane == 0) {
    warp_count[(int64_t)b * warps_per_sample + (int64_t)blockIdx.x * (kRigThreads / 32) + warp] = (int32_t)filled;
    if (filled) atomicAdd(&s_cta_total, filled);
  }
  __syncthreads();
  if (threadIdx.x == 0 && s_cta_total) atomicAdd(sample_total + b, s_cta_total);   // one global atomic per CTA
}

// the cell index alone (diagnostics / the variant self-test): geom_xyz int32 (B, N, D, H, W, 3) as the reference makes it
template <int kVariant>
__global__ void __launch_bounds__(256)
rig_geom_kernel(RigParams rp, int num_cams, int D, int H, int W, int64_t total, int32_t *__restrict__ geom) {
  const int64_t gp = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (gp >= total) return;
  int64_t t = gp;
  const int w = (int)(t % W); t /= W;
  const int h = (int)(t % H); t /= H;
  const int d = (int)(t % D); t /= D;            // t = b * num_cams + n
  const float *mp = rp.combine + t * 16;
  float m0[4], m1[4], m2[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) { m0[k] = __ldg(mp + k); m1[k] = __ldg(mp + 4 + k); m2[k] = __ldg(mp + 8 + k); }
  const float dd = __ldg(rp.fd + d);
  const float px = __fmul_rn(__ldg(rp.fx + w), dd), py = __fmul_rn(__ldg(rp.fy + h), dd);
  geom[gp * 3 + 0] = rig_quantise(rig_dot4<kVariant>(m0, px, py, dd), rp.lo[0], rp.vs[0], rp.inv_vs[0]);
  geom[gp * 3 + 1] = rig_quantise(rig_dot4<kVariant>(m1, px, py, dd), rp.lo[1], rp.vs[1], rp.inv_vs[1]);
  geom[gp * 3 + 2] = rig_quantise(rig_dot4<kVariant>(m2, px, py, dd), rp.lo[2], rp.vs[2], rp.inv_vs[2]);
}

// K2: exclusive scan of the per-cell run counts, one independent look-back chain per SAMPLE (a single
// chain over B*G cells is latency-bound on its 250 tile hand-offs); a sample's base offset is the sum
// of the run totals of the samples before it (accumulated by K1).  Same tile scheme as scan.cuh.
__global__ void __launch_bounds__(kScanThreads)
run_csr_scan_kernel(const uint32_t *__restrict__ counts, uint32_t *__restrict__ cell_start, int64_t cells,
                    const uint32_t *__restrict__ sample_total, int batch, unsigned long long *status,
                    unsigned int *tickets, int tiles_per_sample) {
  pdl_wait();
  pdl_trigger();
  __shared__ uint32_t s_warp[kScanThreads / 32];
  __shared__ uint32_t s_tile, s_prefix, s_base;
  const int b = blockIdx.y;
  if (threadIdx.x == 0) s_tile = atomicAdd(tickets + b, 1u);
  __syncthreads();
  const uint32_t tile = s_tile;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t *in = counts + (int64_t)b * cells;
  uint32_t *out = cell_start + (int64_t)b * cells;
  unsigned long long *st_b = status + (int64_t)b * tiles_per_sample;
  const int64_t warp_base = (int64_t)tile * kScanTile + warp * 512;

  uint4 v[4];
  uint32_t excl[4];
  uint32_t run = 0;
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int64_t idx = warp_base + r * 128 + lane * 4;
    if (idx + 3 < cells) {
      v[r] = *reinterpret_cast<const uint4 *>(in + idx);
    } else {
      v[r].x = idx < cells ? in[idx] : 0u;
      v[r].y = idx + 1 < cells ? in[idx + 1] : 0u;
      v[r].z = idx + 2 < cells ? in[idx + 2] : 0u;
      v[r].w = 0u;
    }
    const uint32_t s = v[r].x + v[r].y + v[r].z + v[r].w;
    uint32_t incl = s;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    excl[r] = run + incl - s;
    run += __shfl_sync(0xffffffffu, incl, 31);
  }
  if (lane == 0) s_warp[warp] = run;
  __syncthreads();

  if (warp == 0) {
    const uint32_t w = lane < kScanThreads / 32 ? s_warp[lane] : 0u;
    uint32_t incl = w;
#pragma unroll
    for (int o = 1; o < kScanThreads / 32; o <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    const uint32_t total = __shfl_sync(0xffffffffu, incl, kScanThreads / 32 - 1);
    if (lane < kScanThreads / 32) s_warp[lane] = incl - w;
    // base of this sample = runs of all earlier samples
    uint32_t base = 0;
    for (int i = lane; i < b; i += 32) base += sample_total[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) base += __shfl_xor_sync(0xffffffffu, base, o);

    uint32_t exclusive = 0;
    if (tile == 0) {
      if (lane == 0) st_volatile_u64(st_b, kScanPrefix | total);
      if (b == batch - 1 && lane == 0) cell_start[(int64_t)batch * cells] = base + sample_total[b];
    } else {
      if (lane == 0) st_volatile_u64(st_b + tile, kScanAggregate | total);
      int64_t look = (int64_t)tile - 1;
      while (true) {
        const int64_t idx = look - lane;
        unsigned long long st;
        do {
          st = idx >= 0 ? ld_volatile_u64(st_b + idx) : kScanPrefix;
        } while (__any_sync(0xffffffffu, (st >> 32) == 0ull));
        const unsigned pm = __ballot_sync(0xffffffffu, (st >> 32) == 2ull);
        const int first = pm ? __ffs(pm) - 1 : 32;
        uint32_t contrib = lane <= first ? (uint32_t)(st & 0xffffffffull) : 0u;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) contrib += __shfl_xor_sync(0xffffffffu, contrib, o);
        exclusive += contrib;
        if (pm) break;
        look -= 32;
      }
      if (lane == 0) st_volatile_u64(st_b + tile, kScanPrefix | (uint64_t)(exclusive + total));
    }
    if (lane == 0) { s_prefix = exclusive; s_base = base; }
  }
  __syncthreads();

  const uint32_t base = s_base + s_prefix + s_warp[warp];
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int64_t idx = warp_base + r * 128 + lane * 4;
    uint4 o;
    o.x = base + excl[r];
    o.y = o.x + v[r].x;
    o.z = o.y + v[r].y;
    o.w = o.z + v[r].z;
    if (idx + 3 < cells) {
      *reinterpret_cast<uint4 *>(out + idx) = o;
    } else {
      if (idx < cells) out[idx] = o.x;
      if (idx + 1 < cells) out[idx + 1] = o.y;
      if (idx + 2 < cells) out[idx + 2] = o.z;
    }
  }
}

// K3: eight lanes per K1 warp slice (a slice holds 11 heads on average)
__global__ void __launch_bounds__(256)
run_place_kernel(const int32_t *__restrict__ head_cells, const int32_t *__restrict__ head_ids,
                 const int32_t *__restrict__ warp_count, const uint32_t *__restrict__ cell_start,
                 uint32_t *__restrict__ counts, int32_t *__restrict__ placed_ids,
                 int32_t *__restrict__ placed_cells, int64_t num_slices, int slices_per_sample,
                 int64_t cells_per_sample, int slot_cap) {
  pdl_wait();
  pdl_trigger();
  const int64_t slice = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 3;
  const int l8 = threadIdx.x & 7;
  if (slice >= num_slices) return;
  const int n = warp_count[slice];
  const int64_t cell_base = (slice / slices_per_sample) * cells_per_sample;
  for (int i = l8; i < n; i += 8) {
    const int64_t gc = cell_base + head_cells[slice * slot_cap + i];
    const uint32_t left = atomicSub(counts + gc, 1u);          // the per-cell count doubles as the cursor
    const uint32_t pos = cell_start[gc] + left - 1u;
    placed_ids[pos] = head_ids[slice * slot_cap + i];
    placed_cells[pos] = (int32_t)gc;
  }
}

// K4: one thread per run head; rank of a head = number of heads of its cell with a smaller point id (the
// cell's segment is a handful of consecutive ints: L1 hits).  Cells with more than kRunSmallCell runs
// (none for camera rigs: the aiMotive shapes peak at 54 runs per cell) are queued for K5 by the thread
// that holds the segment's first entry, so no thread ever walks a long segment.
constexpr uint32_t kRunSmallCell = 64;

struct PairDims {            // how a global point id decomposes into (sample, image*bin, row, column)
  FastDiv div_w, div_h, div_np;
  int HB, W;
  int64_t pairs_per_sample;
};
// head point `id` got `slot`: if it is the first kept row of its pair, record the slot there
__device__ __forceinline__ void record_primary_slot(int4 *__restrict__ pair_rec, const PairDims &pd, int32_t id, int32_t slot) {
  const uint32_t b = fastdiv((uint32_t)id, pd.div_np);
  const uint32_t p = (uint32_t)id - b * pd.div_np.div;          // point inside the sample
  const uint32_t rowi = fastdiv(p, pd.div_w);                   // (n*D + d) * H + h
  const uint32_t w = p - rowi * pd.div_w.div;
  const uint32_t nd = fastdiv(rowi, pd.div_h);
  const uint32_t h = rowi - nd * pd.div_h.div;
  const int64_t q = (int64_t)b * pd.pairs_per_sample + ((int64_t)nd * pd.HB + h / kRunHB) * pd.W + w;
  pair_rec[q].z = slot;
}
constexpr int32_t kHeadIdMask = 0x7fffffff;       // head ids carry "first kept row of its pair" in bit 31
__global__ void __launch_bounds__(256)
run_finish_kernel(const uint32_t *__restrict__ cell_start, const int32_t *__restrict__ placed_ids,
                  const int32_t *__restrict__ placed_cells, int64_t total_cells, int32_t *__restrict__ sorted_ids,
                  int32_t *__restrict__ sorted_cells, int32_t *__restrict__ run_code, int32_t *__restrict__ big_list,
                  uint32_t *__restrict__ big_count, int4 *__restrict__ pair_rec, PairDims pd) {
  pdl_wait();
  pdl_trigger();
  const uint32_t total = cell_start[total_cells];
  for (uint32_t pos = blockIdx.x * blockDim.x + threadIdx.x; pos < total; pos += gridDim.x * blockDim.x) {
    const int32_t gc = placed_cells[pos];
    const uint32_t s = cell_start[gc], e = cell_start[gc + 1];
    if (e - s > kRunSmallCell) {
      if (pos == s) big_list[atomicAdd(big_count, 1u)] = gc;     // (order of the queue is irrelevant)
      continue;
    }
    const int32_t idf = placed_ids[pos], id = idf & kHeadIdMask;
    uint32_t rank = 0;
    for (uint32_t j = s; j < e; ++j) rank += (placed_ids[j] & kHeadIdMask) < id;
    sorted_ids[s + rank] = id;
    sorted_cells[s + rank] = gc;
    run_code[id] = (int32_t)(s + rank);
    if (idf < 0) record_primary_slot(pair_rec, pd, id, (int32_t)(s + rank));
  }
}

// K5: one CTA per queued cell, same rank rule with the ids staged through shared memory
__global__ void __launch_bounds__(256)
run_finish_big_kernel(const uint32_t *__restrict__ cell_start, const int32_t *__restrict__ placed_ids,
                      const int32_t *__restrict__ big_list, const uint32_t *__restrict__ big_count,
                      int32_t *__restrict__ sorted_ids, int32_t *__restrict__ sorted_cells,
                      int32_t *__restrict__ run_code, int4 *__restrict__ pair_rec, PairDims pd) {
  pdl_wait();
  pdl_trigger();
  constexpr int kTile = 2048;
  __shared__ int32_t s_ids[kTile];
  const uint32_t nbig = *big_count;
  for (uint32_t q = blockIdx.x; q < nbig; q += gridDim.x) {
    const int64_t gc = big_list[q];
    const uint32_t s = cell_start[gc], n = cell_start[gc + 1] - s;
    for (uint32_t i0 = 0; i0 < n; i0 += blockDim.x) {
      const uint32_t i = i0 + threadIdx.x;
      const int32_t idf = i < n ? placed_ids[s + i] : INT32_MAX, id = idf & kHeadIdMask;
      uint32_t rank = 0;
      for (uint32_t j0 = 0; j0 < n; j0 += kTile) {
        __syncthreads();
        const uint32_t m = min((uint32_t)kTile, n - j0);
        for (uint32_t j = threadIdx.x; j < m; j += blockDim.x) s_ids[j] = placed_ids[s + j0 + j] & kHeadIdMask;
        __syncthreads();
        for (uint32_t j = 0; j < m; ++j) rank += s_ids[j] < id;
      }
      if (i < n) {
        sorted_ids[s + rank] = id;
        sorted_cells[s + rank] = (int32_t)gc;
        run_code[id] = (int32_t)(s + rank);
        if (idf < 0) record_primary_slot(pair_rec, pd, id, (int32_t)(s + rank));
      }
    }
  }
}

__global__ void __launch_bounds__(kSortThreads)
bucket_sort_kernel(const int32_t *__restrict__ keys, const int32_t *__restrict__ ids,
                   const uint32_t *__restrict__ scanned, int bins_hi, int tiles_per_sample, int low_bits,
                   int32_t cells_per_sample, int batch, int32_t *__restrict__ cell_start,
                   int32_t *__restrict__ sorted_ids, int32_t *__restrict__ sorted_cells,
                   int32_t *__restrict__ slot_of_id /* run plans: run_code[first point] = slot, else NULL */) {
  __shared__ uint32_t s_run[256];                  // next output position of every low-bits bin
  __shared__ uint32_t s_cnt[kSortWarps][256];      // per-warp counts of the current chunk
  __shared__ uint32_t s_warp_tot[kSortWarps];
  const int h = blockIdx.x, b = blockIdx.y;
  const int nlow = 1 << low_bits, lmask = nlow - 1;
  const int64_t slot = ((int64_t)b * bins_hi + h) * tiles_per_sample;
  const uint32_t begin = scanned[slot], end = scanned[slot + tiles_per_sample];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

  // (i) histogram of the low bits over the whole bucket
  s_run[threadIdx.x] = 0u;
  __syncthreads();
  for (uint32_t i = begin + threadIdx.x; i < end; i += kSortThreads) atomicAdd(&s_run[keys[i] & lmask], 1u);
  __syncthreads();
  // (ii) exclusive scan of the 256 bins (one element per thread) -> CSR offsets of the bucket's cells
  {
    const uint32_t v = s_run[threadIdx.x];
    uint32_t incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    if (lane == 31) s_warp_tot[warp] = incl;
    __syncthreads();
    uint32_t base = begin;
    for (int w = 0; w < warp; ++w) base += s_warp_tot[w];
    const uint32_t excl = base + incl - v;
    __syncthreads();
    s_run[threadIdx.x] = excl;
    const int cell = (h << low_bits) + threadIdx.x;
    if ((int)threadIdx.x < nlow && cell < cells_per_sample) cell_start[(int64_t)b * cells_per_sample + cell] = (int32_t)excl;
    if (h == 0 && b == 0 && threadIdx.x == 0)
      cell_start[(int64_t)batch * cells_per_sample] = (int32_t)scanned[(int64_t)batch * bins_hi * tiles_per_sample];
  }
  __syncthreads();
  // (iii) stable placement, one chunk of kSortTile elements at a time, element order (warp, round, lane)
  for (uint32_t chunk = begin; chunk < end; chunk += kSortTile) {
    for (int i = threadIdx.x; i < kSortWarps * 256; i += kSortThreads) (&s_cnt[0][0])[i] = 0u;
    __syncthreads();
    uint32_t *cnt = s_cnt[warp];
    const uint32_t warp_begin = chunk + warp * (kSortItems * 32);
    int32_t key[kSortItems], id[kSortItems];
    uint32_t rank[kSortItems];
#pragma unroll
    for (int r = 0; r < kSortItems; ++r) {
      const uint32_t idx = warp_begin + r * 32 + lane;
      const bool in_range = idx < end;
      key[r] = in_range ? keys[idx] : -1;
      id[r] = in_range ? ids[idx] : -1;
    }
#pragma unroll
    for (int r = 0; r < kSortItems; ++r) {
      const bool valid = key[r] >= 0;
      const uint32_t digit = valid ? (uint32_t)(key[r] & lmask) : 256u;
      const unsigned peers = __match_any_sync(0xffffffffu, digit);
      const int leader = __ffs(peers) - 1;
      uint32_t base = 0;
      if (valid && lane == leader) {
        base = cnt[digit];
        cnt[digit] = base + __popc(peers);
      }
      base = __shfl_sync(0xffffffffu, base, leader);
      rank[r] = base + __popc(peers & ((1u << lane) - 1u));
      __syncwarp();
    }
    __syncthreads();
    {   // per-bin: turn the warps' counts into starting positions, advance the running offset
      const int bin = threadIdx.x;
      uint32_t run = s_run[bin];
#pragma unroll
      for (int w = 0; w < kSortWarps; ++w) {
        const uint32_t t = s_cnt[w][bin];
        s_cnt[w][bin] = run;
        run += t;
      }
      s_run[bin] = run;
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < kSortItems; ++r) {
      if (key[r] >= 0) {
        const uint32_t pos = cnt[key[r] & lmask] + rank[r];
        sorted_ids[pos] = id[r];
        sorted_cells[pos] = b * cells_per_sample + key[r];
        if (slot_of_id) slot_of_id[id[r]] = (int32_t)pos;
      }
    }
    __syncthreads();
  }
}

__global__ void pos_memo_kernel(const int32_t *__restrict__ cell_of_point, int64_t num_points,
                                int64_t total, int X, int32_t *__restrict__ pos_memo) {
  const int64_t gp = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (gp >= total) return;
  const int cell = cell_of_point[gp];
  int b = -1, y = -1, x = -1;
  if (cell >= 0) {
    b = (int)(gp / num_points);
    y = cell / X;
    x = cell - y * X;
  }
  pos_memo[gp * 3 + 0] = b;
  pos_memo[gp * 3 + 1] = y;
  pos_memo[gp * 3 + 2] = x;
}

}  // namespace bevpool

using namespace bevpool;

extern "C" int bevpool_plan_sizes(int batch, int64_t num_points, int X, int Y, size_t *plan_bytes,
                                  size_t *temp_bytes) {
  int rc = check_plan_dims(batch, num_points, X, Y);
  if (rc) return rc;
  if (!plan_bytes || !temp_bytes) return BEVPOOL_E_ARG;
  *plan_bytes = plan_layout(batch, num_points, X, Y).bytes;
  *temp_bytes = temp_layout(batch, num_points, X, Y).bytes;
  return BEVPOOL_OK;
}

extern "C" int bevpool_plan_build(const int32_t *geom, int batch, int64_t num_points, int X, int Y,
                                  int Z, void *plan, void *temp, void *stream_) {
  int rc = check_plan_dims(batch, num_points, X, Y);
  if (rc) return rc;
  if (!geom || !plan || !temp || Z <= 0) return BEVPOOL_E_ARG;
  if (!aligned16(plan) || !aligned16(temp)) return BEVPOOL_E_ALIGN;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const int64_t cells = (int64_t)X * Y;
  const SortConfig sc = sort_config(cells);
  const PlanLayout PL = plan_layout(batch, num_points, X, Y);
  const TempLayout TL = temp_layout(batch, num_points, X, Y);
  char *pb = static_cast<char *>(plan), *tb = static_cast<char *>(temp);
  int32_t *cell_of_point = reinterpret_cast<int32_t *>(pb + PL.off_cell_of_point);
  uint32_t *cell_start = reinterpret_cast<uint32_t *>(pb + PL.off_cell_start);
  int32_t *sorted_ids = reinterpret_cast<int32_t *>(pb + PL.off_sorted_ids);
  int32_t *sorted_cells = reinterpret_cast<int32_t *>(pb + PL.off_sorted_cells);
  uint32_t *hist[kMaxPasses];
  for (int p = 0; p < sc.npass; ++p) hist[p] = reinterpret_cast<uint32_t *>(tb + TL.off_hist[p]);
  int32_t *keys[2] = {reinterpret_cast<int32_t *>(tb + TL.off_keys[0]),
                      reinterpret_cast<int32_t *>(tb + TL.off_keys[1])};
  int32_t *ids[2] = {reinterpret_cast<int32_t *>(tb + TL.off_ids[0]),
                     reinterpret_cast<int32_t *>(tb + TL.off_ids[1])};
  const int T = TL.tiles_per_sample;
  const dim3 grid(T, batch);

  BEVPOOL_RETURN_IF_CUDA(cudaMemsetAsync(tb, 0, TL.zero_bytes, stream));
  const PlanHeader hv = make_plan_header(kPlanKindPoints, batch, num_points, X, Y, Z);

  if (sc.msd) {
    const int low = sc.bits[0], bins_hi = 1 << sc.bits[1];
    plan_key_msd_kernel<<<grid, kSortThreads, bins_hi * 4, stream>>>(geom, num_points, X, Y, Z, cell_of_point,
                                                                    hist[0], low, bins_hi, T, static_cast<PlanHeader *>(plan), hv);
    BEVPOOL_LAUNCH_CHECK();
    rc = launch_scan_exclusive(hist[0], hist[0], TL.hist_n[0], tb + TL.off_scan[0], stream);
    if (rc) return rc;
    sort_scatter_kernel<true><<<grid, kSortThreads, kSortWarps * bins_hi * 4, stream>>>(
        cell_of_point, nullptr, keys[0], ids[0], nullptr, (int32_t)cells, hist[0], hist[0], bins_hi, num_points,
        low, bins_hi, T);
    BEVPOOL_LAUNCH_CHECK();
    bucket_sort_kernel<<<dim3(bins_hi, batch), kSortThreads, 0, stream>>>(
        keys[0], ids[0], hist[0], bins_hi, T, low, (int32_t)cells, batch, reinterpret_cast<int32_t *>(cell_start),
        sorted_ids, sorted_cells, nullptr);
    BEVPOOL_LAUNCH_CHECK();
    return BEVPOOL_OK;
  }
  BEVPOOL_RETURN_IF_CUDA(cudaMemsetAsync(cell_start, 0, ((size_t)batch * cells + 1) * 4, stream));

  const int bins0 = 1 << sc.bits[0];
  plan_key_kernel<<<grid, kSortThreads, bins0 * 4, stream>>>(
      geom, num_points, X, Y, Z, cell_of_point, cell_start, hist[0], bins0, T, static_cast<PlanHeader *>(plan), hv);
  BEVPOOL_LAUNCH_CHECK();
  rc = launch_scan_exclusive(hist[0], hist[0], TL.hist_n[0], tb + TL.off_scan[0], stream);
  if (rc) return rc;
  {
    const bool last = sc.npass == 1;
    sort_scatter_kernel<true><<<grid, kSortThreads, kSortWarps * bins0 * 4, stream>>>(
        cell_of_point, nullptr, last ? nullptr : keys[0], last ? sorted_ids : ids[0],
        last ? sorted_cells : nullptr, (int32_t)cells, hist[0], hist[0], bins0, num_points, sc.shift[0], bins0, T);
    BEVPOOL_LAUNCH_CHECK();
  }
  for (int p = 1; p < sc.npass; ++p) {
    const int bins = 1 << sc.bits[p];
    const bool last = p == sc.npass - 1;
    const int src = (p - 1) & 1, dst = p & 1;
    sort_hist_kernel<<<grid, kSortThreads, bins * 4, stream>>>(keys[src], hist[0], bins0,
                                                               sc.shift[p], bins, T, hist[p]);
    BEVPOOL_LAUNCH_CHECK();
    rc = launch_scan_exclusive(hist[p], hist[p], TL.hist_n[p], tb + TL.off_scan[p], stream);
    if (rc) return rc;
    sort_scatter_kernel<false><<<grid, kSortThreads, kSortWarps * bins * 4, stream>>>(
        keys[src], ids[src], last ? nullptr : keys[dst], last ? sorted_ids : ids[dst],
        last ? sorted_cells : nullptr, (int32_t)cells, hist[p], hist[0], bins0, num_points, sc.shift[p], bins, T);
    BEVPOOL_LAUNCH_CHECK();
  }
  rc = launch_scan_exclusive(cell_start, cell_start, (int64_t)batch * cells + 1,
                             tb + TL.off_scan[kMaxPasses], stream);
  return rc;
}

extern "C" int bevpool_plan_pos_memo(const void *plan, int batch, int64_t num_points, int X, int Y,
                                     int32_t *pos_memo, void *stream_) {
  int rc = check_plan_dims(batch, num_points, X, Y);
  if (rc) return rc;
  if (!plan || !pos_memo) return BEVPOOL_E_ARG;
  const PlanView v = plan_view(plan, batch, num_points, X, Y);
  const int64_t total = (int64_t)batch * num_points;
  pos_memo_kernel<<<(unsigned)ceil_div64(total, 256), 256, 0, static_cast<cudaStream_t>(stream_)>>>(
      v.cell_of_point, num_points, total, X, pos_memo);
  BEVPOOL_LAUNCH_CHECK();
  return BEVPOOL_OK;
}

extern "C" int bevpool_plan_views(const void *plan, int batch, int64_t num_points, int X, int Y,
                                  const int32_t **cell_of_point, const int32_t **cell_start,
                                  const int32_t **sorted_ids) {
  int rc = check_plan_dims(batch, num_points, X, Y);
  if (rc) return rc;
  if (!plan) return BEVPOOL_E_ARG;
  const PlanView v = plan_view(plan, batch, num_points, X, Y);
  if (cell_of_point) *cell_of_point = v.cell_of_point;
  if (cell_start) *cell_start = v.cell_start;
  if (sorted_ids) *sorted_ids = v.sorted_ids;
  return BEVPOOL_OK;
}

// ---- run plan (fused op): see common.cuh and the K1..K4 kernels above ----
struct RunTempLayout {
  size_t off_scan, off_counts, zero_bytes;     // [0, zero_bytes) is memset to 0 per build
  size_t off_big_count, off_sample_total, off_tickets, off_status;   // (inside the zeroed part)
  size_t off_head_cells, off_head_ids, off_warp_count, off_placed, off_placed_cells, off_big_list, bytes;
  int slices_per_sample, slot_cap;             // K1 warp slices of the head lists and their capacity
};
static RunTempLayout run_temp_layout(int batch, int64_t num_points, int X, int Y, int slices_per_sample, int slot_cap) {
  RunTempLayout L{};
  L.slices_per_sample = slices_per_sample;
  L.slot_cap = slot_cap;
  const size_t G1 = (size_t)batch * X * Y + 1;
  const size_t slices = (size_t)batch * slices_per_sample;
  size_t o = 0;
  L.off_scan = o;        o += scan_workspace_bytes((int64_t)G1);
  L.off_counts = o;      o = align_up(o + G1 * 4, 256);
  L.off_big_count = o;   o += 256;
  L.off_sample_total = o; o = align_up(o + (size_t)batch * 4, 256);
  L.off_tickets = o;     o = align_up(o + (size_t)batch * 4, 256);
  L.off_status = o;      o = align_up(o + (size_t)batch * scan_num_tiles((int64_t)X * Y) * 8, 256);
  L.zero_bytes = o;
  L.off_head_cells = o;  o = align_up(o + slices * slot_cap * 4, 256);
  L.off_head_ids = o;    o = align_up(o + slices * slot_cap * 4, 256);
  L.off_warp_count = o;  o = align_up(o + slices * 4, 256);
  L.off_placed = o;      o = align_up(o + (size_t)batch * num_points * 4, 256);
  L.off_placed_cells = o; o = align_up(o + (size_t)batch * num_points * 4, 256);
  L.off_big_list = o;    o = align_up(o + ((size_t)batch * num_points / 16 + 1) * 4, 256);
  L.bytes = o;
  return L;
}
static RunTempLayout run_temp_layout_rig(int batch, int N, int D, int H, int W, int X, int Y) {
  const int HB = (int)ceil_div64(H, kRunHB);
  const int64_t pairs = (int64_t)N * D * HB * W;
  return run_temp_layout(batch, (int64_t)N * D * H * W, X, Y, (int)ceil_div64(pairs, kRigThreads) * (kRigThreads / 32),
                         32 * (H < kRunHB ? H : kRunHB));
}

extern "C" int bevpool_runplan_sizes(int batch, int num_cams, int depth_bins, int feat_h, int feat_w, int X, int Y,
                                     size_t *plan_bytes, size_t *temp_bytes) {
  if (num_cams <= 0 || depth_bins <= 0 || feat_h <= 0 || feat_w <= 0) return BEVPOOL_E_ARG;
  const int64_t num_points = (int64_t)num_cams * depth_bins * feat_h * feat_w;
  int rc = check_plan_dims(batch, num_points, X, Y);
  if (rc) return rc;
  if (!plan_bytes || !temp_bytes) return BEVPOOL_E_ARG;
  *plan_bytes = plan_layout(batch, num_points, X, Y, true, plan_num_pairs(num_cams, depth_bins, feat_h, feat_w)).bytes;
  *temp_bytes = run_temp_layout_rig(batch, num_cams, depth_bins, feat_h, feat_w, X, Y).bytes;
  return BEVPOOL_OK;
}

extern "C" int bevpool_runplan_rig_sizes(int batch, int num_cams, int depth_bins, int feat_h, int feat_w, int X, int Y,
                                         size_t *plan_bytes, size_t *temp_bytes) {
  if (num_cams <= 0 || depth_bins <= 0 || feat_h <= 0 || feat_w <= 0) return BEVPOOL_E_ARG;
  const int64_t num_points = (int64_t)num_cams * depth_bins * feat_h * feat_w;
  int rc = check_plan_dims(batch, num_points, X, Y);
  if (rc) return rc;
  if (!plan_bytes || !temp_bytes) return BEVPOOL_E_ARG;
  *plan_bytes = plan_layout(batch, num_points, X, Y, true, plan_num_pairs(num_cams, depth_bins, feat_h, feat_w)).bytes;
  *temp_bytes = run_temp_layout_rig(batch, num_cams, depth_bins, feat_h, feat_w, X, Y).bytes;
  return BEVPOOL_OK;
}

// K2..K5 of a run plan: per-cell run counts + per-warp head lists (K1's output) -> CSR, sorted run list, slots
static int run_plan_finish(const RunTempLayout &TL, const PlanLayout &PL, int batch, int64_t cells, int num_cams, int D,
                           int H, int W, char *pb, char *tb, cudaStream_t stream) {
  const int64_t total_cells = (int64_t)batch * cells;
  int4 *pair_rec = reinterpret_cast<int4 *>(pb + PL.off_pair_rec);
  PairDims pd;
  pd.div_w = make_fastdiv((uint32_t)W);
  pd.div_h = make_fastdiv((uint32_t)H);
  pd.div_np = make_fastdiv((uint32_t)((int64_t)num_cams * D * H * W));
  pd.HB = (H + kRunHB - 1) / kRunHB;
  pd.W = W;
  pd.pairs_per_sample = plan_num_pairs(num_cams, D, H, W);
  uint32_t *cell_start = reinterpret_cast<uint32_t *>(pb + PL.off_cell_start);
  int32_t *sorted_ids = reinterpret_cast<int32_t *>(pb + PL.off_sorted_ids);
  int32_t *sorted_cells = reinterpret_cast<int32_t *>(pb + PL.off_sorted_cells);
  int32_t *run_code = reinterpret_cast<int32_t *>(pb + PL.off_run_code);
  uint32_t *counts = reinterpret_cast<uint32_t *>(tb + TL.off_counts);
  int32_t *head_cells = reinterpret_cast<int32_t *>(tb + TL.off_head_cells);
  int32_t *head_ids = reinterpret_cast<int32_t *>(tb + TL.off_head_ids);
  int32_t *warp_count = reinterpret_cast<int32_t *>(tb + TL.off_warp_count);
  int32_t *placed = reinterpret_cast<int32_t *>(tb + TL.off_placed);
  int32_t *placed_cells = reinterpret_cast<int32_t *>(tb + TL.off_placed_cells);
  uint32_t *sample_total = reinterpret_cast<uint32_t *>(tb + TL.off_sample_total);
  if ((cells & 3) == 0) {            // per-sample chains (16-byte aligned sample segments)
    const int tps = (int)scan_num_tiles(cells);
    BEVPOOL_RETURN_IF_CUDA(launch_pdl(run_csr_scan_kernel, dim3(tps, batch), dim3(kScanThreads), 0, stream,
        counts, cell_start, cells, sample_total, batch, reinterpret_cast<unsigned long long *>(tb + TL.off_status),
        reinterpret_cast<unsigned int *>(tb + TL.off_tickets), tps));
    BEVPOOL_LAUNCH_CHECK();
  } else {
    int rc = launch_scan_exclusive(counts, cell_start, total_cells + 1, tb + TL.off_scan, stream);
    if (rc) return rc;
  }
  const int64_t slices = (int64_t)batch * TL.slices_per_sample;
  BEVPOOL_RETURN_IF_CUDA(launch_pdl(run_place_kernel, dim3((unsigned)ceil_div64(slices * 8, 256)), dim3(256), 0, stream,
      head_cells, head_ids, warp_count, cell_start, counts, placed, placed_cells, slices, TL.slices_per_sample, cells,
      TL.slot_cap));
  BEVPOOL_LAUNCH_CHECK();
  int32_t *big_list = reinterpret_cast<int32_t *>(tb + TL.off_big_list);
  uint32_t *big_count = reinterpret_cast<uint32_t *>(tb + TL.off_big_count);
  BEVPOOL_RETURN_IF_CUDA(launch_pdl(run_finish_kernel, dim3(kSMs * 8), dim3(256), 0, stream,
      cell_start, placed, placed_cells, total_cells, sorted_ids, sorted_cells, run_code, big_list, big_count, pair_rec, pd));
  BEVPOOL_LAUNCH_CHECK();
  BEVPOOL_RETURN_IF_CUDA(launch_pdl(run_finish_big_kernel, dim3(kSMs * 2), dim3(256), 0, stream,
                                    cell_start, placed, big_list, big_count, sorted_ids, sorted_cells, run_code, pair_rec, pd));
  BEVPOOL_LAUNCH_CHECK();
  return BEVPOOL_OK;
}

extern "C" int bevpool_runplan_build(const int32_t *geom, int batch, int num_cams, int depth_bins, int feat_h,
                                     int feat_w, int X, int Y, int Z, void *plan, void *temp, void *stream_) {
  if (num_cams <= 0 || depth_bins <= 0 || feat_h <= 0 || feat_w <= 0) return BEVPOOL_E_ARG;
  const int64_t num_points = (int64_t)num_cams * depth_bins * feat_h * feat_w;
  int rc = check_plan_dims(batch, num_points, X, Y);
  if (rc) return rc;
  if (!geom || !plan || !temp || Z <= 0) return BEVPOOL_E_ARG;
  if (!aligned16(plan) || !aligned16(temp)) return BEVPOOL_E_ALIGN;
  if (batch > 65535) return BEVPOOL_E_RANGE;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const int64_t cells = (int64_t)X * Y;
  const int64_t pairs = plan_num_pairs(num_cams, depth_bins, feat_h, feat_w);
  const PlanLayout PL = plan_layout(batch, num_points, X, Y, true, pairs);
  const RunTempLayout TL = run_temp_layout_rig(batch, num_cams, depth_bins, feat_h, feat_w, X, Y);
  char *pb = static_cast<char *>(plan), *tb = static_cast<char *>(temp);
  const int HB = (int)ceil_div64(feat_h, kRunHB);
  const dim3 grid((unsigned)ceil_div64(pairs, kRigThreads), (unsigned)batch);
  BEVPOOL_RETURN_IF_CUDA(cudaMemsetAsync(tb, 0, TL.zero_bytes, stream));
  BEVPOOL_RETURN_IF_CUDA(launch_pdl(plan_key_rig_kernel<-1>, grid, dim3(kRigThreads), 0, stream, RigParams{}, geom, num_cams,
      depth_bins, feat_h, feat_w, HB, X, Y, Z, num_points, reinterpret_cast<int32_t *>(pb + PL.off_cell_of_point),
      reinterpret_cast<int32_t *>(pb + PL.off_run_code), reinterpret_cast<uint32_t *>(tb + TL.off_counts),
      reinterpret_cast<int32_t *>(tb + TL.off_head_cells), reinterpret_cast<int32_t *>(tb + TL.off_head_ids),
      reinterpret_cast<int32_t *>(tb + TL.off_warp_count), reinterpret_cast<uint32_t *>(tb + TL.off_sample_total),
      TL.slices_per_sample, TL.slot_cap, reinterpret_cast<int4 *>(pb + PL.off_pair_rec), static_cast<PlanHeader *>(plan),
      make_plan_header(kPlanKindRuns, batch, num_points, X, Y, Z)));
  BEVPOOL_LAUNCH_CHECK();
  return run_plan_finish(TL, PL, batch, cells, num_cams, depth_bins, feat_h, feat_w, pb, tb, stream);
}

constexpr int kRigVariants = 6;
extern "C" int bevpool_rig_num_variants(void) { return kRigVariants; }

static int make_rig_params(RigParams *rp, const float *combine, const float *fx, const float *fy, const float *fd,
                           const float *lower_host, const float *voxel_size_host) {
  if (!combine || !fx || !fy || !fd || !lower_host || !voxel_size_host) return BEVPOOL_E_ARG;
  if (!aligned16(combine)) return BEVPOOL_E_ALIGN;
  rp->combine = combine; rp->fx = fx; rp->fy = fy; rp->fd = fd;
  for (int i = 0; i < 3; ++i) {
    if (!(voxel_size_host[i] != 0.f)) return BEVPOOL_E_ARG;
    rp->lo[i] = lower_host[i];
    rp->vs[i] = voxel_size_host[i];
    rp->inv_vs[i] = 1.0f / voxel_size_host[i];
  }
  return BEVPOOL_OK;
}

#define BEVPOOL_RIG_DISPATCH(variant, CALL)                 \
  switch (variant) {                                        \
    case 0: { constexpr int V = 0; CALL; break; }           \
    case 1: { constexpr int V = 1; CALL; break; }           \
    case 2: { constexpr int V = 2; CALL; break; }           \
    case 3: { constexpr int V = 3; CALL; break; }           \
    case 4: { constexpr int V = 4; CALL; break; }           \
    case 5: { constexpr int V = 5; CALL; break; }           \
    default: return BEVPOOL_E_ARG;                          \
  }

extern "C" int bevpool_runplan_build_rig(const float *combine, const float *frustum_x, const float *frustum_y,
                                         const float *frustum_d, const float *lower_host, const float *voxel_size_host,
                                         int variant, int batch, int num_cams, int depth_bins, int feat_h, int feat_w,
                                         int X, int Y, int Z, void *plan, void *temp, void *stream_) {
  if (num_cams <= 0 || depth_bins <= 0 || feat_h <= 0 || feat_w <= 0) return BEVPOOL_E_ARG;
  const int64_t num_points = (int64_t)num_cams * depth_bins * feat_h * feat_w;
  int rc = check_plan_dims(batch, num_points, X, Y);
  if (rc) return rc;
  if (!plan || !temp || Z <= 0) return BEVPOOL_E_ARG;
  if (!aligned16(plan) || !aligned16(temp)) return BEVPOOL_E_ALIGN;
  if (batch > 65535) return BEVPOOL_E_RANGE;
  RigParams rp;
  if ((rc = make_rig_params(&rp, combine, frustum_x, frustum_y, frustum_d, lower_host, voxel_size_host))) return rc;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const int64_t cells = (int64_t)X * Y;
  const PlanLayout PL = plan_layout(batch, num_points, X, Y, true, plan_num_pairs(num_cams, depth_bins, feat_h, feat_w));
  const RunTempLayout TL = run_temp_layout_rig(batch, num_cams, depth_bins, feat_h, feat_w, X, Y);
  char *pb = static_cast<char *>(plan), *tb = static_cast<char *>(temp);
  const int HB = (int)ceil_div64(feat_h, kRunHB);
  const int64_t pairs = (int64_t)num_cams * depth_bins * HB * feat_w;
  const dim3 grid((unsigned)ceil_div64(pairs, kRigThreads), (unsigned)batch);
  BEVPOOL_RETURN_IF_CUDA(cudaMemsetAsync(tb, 0, TL.zero_bytes, stream));
  cudaError_t le = cudaSuccess;
  BEVPOOL_RIG_DISPATCH(variant, (le = launch_pdl(plan_key_rig_kernel<V>, grid, dim3(kRigThreads), 0, stream, rp, (const int32_t *)nullptr, num_cams,
      depth_bins, feat_h, feat_w, HB, X, Y, Z, num_points, reinterpret_cast<int32_t *>(pb + PL.off_cell_of_point),
      reinterpret_cast<int32_t *>(pb + PL.off_run_code), reinterpret_cast<uint32_t *>(tb + TL.off_counts),
      reinterpret_cast<int32_t *>(tb + TL.off_head_cells), reinterpret_cast<int32_t *>(tb + TL.off_head_ids),
      reinterpret_cast<int32_t *>(tb + TL.off_warp_count), reinterpret_cast<uint32_t *>(tb + TL.off_sample_total),
      TL.slices_per_sample, TL.slot_cap, reinterpret_cast<int4 *>(pb + PL.off_pair_rec), static_cast<PlanHeader *>(plan),
      make_plan_header(kPlanKindRuns, batch, num_points, X, Y, Z))));
  BEVPOOL_RETURN_IF_CUDA(le);
  BEVPOOL_LAUNCH_CHECK();
  return run_plan_finish(TL, PL, batch, cells, num_cams, depth_bins, feat_h, feat_w, pb, tb, stream);
}

extern "C" int bevpool_rig_geom(const float *combine, const float *frustum_x, const float *frustum_y,
                                const float *frustum_d, const float *lower_host, const float *voxel_size_host, int variant,
                                int batch, int num_cams, int depth_bins, int feat_h, int feat_w, int32_t *geom_xyz,
                                void *stream_) {
  if (batch <= 0 || num_cams <= 0 || depth_bins <= 0 || feat_h <= 0 || feat_w <= 0 || !geom_xyz) return BEVPOOL_E_ARG;
  RigParams rp;
  int rc = make_rig_params(&rp, combine, frustum_x, frustum_y, frustum_d, lower_host, voxel_size_host);
  if (rc) return rc;
  const int64_t total = (int64_t)batch * num_cams * depth_bins * feat_h * feat_w;
  if (total >= (int64_t)INT32_MAX) return BEVPOOL_E_RANGE;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  BEVPOOL_RIG_DISPATCH(variant, (rig_geom_kernel<V><<<(unsigned)ceil_div64(total, 256), 256, 0, stream>>>(
                                    rp, num_cams, depth_bins, feat_h, feat_w, total, geom_xyz)));
  BEVPOOL_LAUNCH_CHECK();
  return BEVPOOL_OK;
}

// the plan's status word (0 = ok, BEVPOOL_PLAN_ROW_OVERFLOW = a consumer found the run_rows scratch too small);
// synchronises `stream`
extern "C" int bevpool_plan_status(const void *plan, int *status_host, void *stream_) {
  if (!plan || !status_host) return BEVPOOL_E_ARG;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  int32_t v = 0;
  BEVPOOL_RETURN_IF_CUDA(cudaMemcpyAsync(&v, plan_status(const_cast<void *>(plan)), 4, cudaMemcpyDeviceToHost, stream));
  BEVPOOL_RETURN_IF_CUDA(cudaStreamSynchronize(stream));
  *status_host = (int)v;
  return BEVPOOL_OK;
}

extern "C" int bevpool_runplan_views(const void *plan, int batch, int64_t num_points, int X, int Y,
                                     const int32_t **cell_of_point, const int32_t **cell_start,
                                     const int32_t **sorted_ids, const int32_t **sorted_cells,
                                     const int32_t **run_code) {
  int rc = check_plan_dims(batch, num_points, X, Y);
  if (rc) return rc;
  if (!plan) return BEVPOOL_E_ARG;
  const PlanView v = plan_view(plan, batch, num_points, X, Y);
  if (cell_of_point) *cell_of_point = v.cell_of_point;
  if (cell_start) *cell_start = v.cell_start;
  if (sorted_ids) *sorted_ids = v.sorted_ids;
  if (sorted_cells) *sorted_cells = v.sorted_cells;
  if (run_code) *run_code = v.run_code;
  return BEVPOOL_OK;
}

extern "C" int bevpool_runplan_pair_records(const void *plan, int batch, int64_t num_points, int X, int Y,
                                            const void **pair_rec) {
  int rc = check_plan_dims(batch, num_points, X, Y);
  if (rc) return rc;
  if (!plan || !pair_rec) return BEVPOOL_E_ARG;
  *pair_rec = plan_view(plan, batch, num_points, X, Y).pair_rec;
  return BEVPOOL_OK;
}

extern "C" int bevpool_abi_version(void) { return BEVPOOL_ABI_VERSION; }

extern "C" int64_t bevpool_launch_count(void) { return (int64_t)g_kernel_launches.load(); }

extern "C" const char *bevpool_error_string(int code) {
  switch (code) {
    case BEVPOOL_OK: return "ok";
    case BEVPOOL_E_ARG: return "invalid argument (null pointer or non-positive size)";
    case BEVPOOL_E_RANGE: return "problem too large for 32-bit point/cell indices";
    case BEVPOOL_E_CHANNELS: return "unsupported channel count";
    case BEVPOOL_E_ALIGN: return "pointer must be 16-byte aligned";
    case BEVPOOL_E_DTYPE: return "unknown dtype code";
    default: return code > 0 ? cudaGetErrorString((cudaError_t)code) : "unknown error";
  }
}

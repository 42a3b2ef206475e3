/* libbevpool_sm100 -- C ABI of the B200-native BEV projection hot path.
 *
 * Drop-in boundary for the native side of aimotive/mm_training's voxel pooling
 * (reference: ops/voxel_pooling/src/voxel_pooling_forward.cpp:24-37, the pybind
 * function `voxel_pooling_forward_wrapper`, and its launcher
 * ops/voxel_pooling/src/voxel_pooling_forward_cuda.cu:38-56) and for the
 * third-party voxelizer / pillar scatter the reference reaches through
 * models/bev_depth.py:181-183 (mmcv `hard_voxelize_forward`, mmdet3d
 * `HardSimpleVFE`, `PointPillarsScatter` / `SparseConvTensor.dense()`).
 *
 * Conventions (same ownership rules as the reference, SURVEY.md section 8b):
 *   - every pointer is a DEVICE pointer unless its name ends in `_host`;
 *   - the caller owns all buffers including workspaces (sizes come from the
 *     *_sizes queries); the library never allocates or frees device memory;
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*),
 *     uses the current device, and is CUDA-graph capturable;
 *   - return value: 0 on success, a positive cudaError_t, or a negative
 *     BEVPOOL_E_* argument error.  The library never calls exit() (the
 *     reference does: voxel_pooling_forward_cuda.cu:52-55).
 */
#ifndef BEVPOOL_SM100_H_
#define BEVPOOL_SM100_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BEVPOOL_ABI_VERSION 2

#define BEVPOOL_OK            0
#define BEVPOOL_E_ARG        -1   /* null pointer / non-positive size            */
#define BEVPOOL_E_RANGE      -2   /* B*Np or B*X*Y does not fit 31 bits          */
#define BEVPOOL_E_CHANNELS   -3   /* channel count unsupported by this build     */
#define BEVPOOL_E_ALIGN      -4   /* pointer not 16-byte aligned                 */
#define BEVPOOL_E_DTYPE      -5   /* unknown dtype code                          */

/* plan status word (bevpool_plan_status) */
#define BEVPOOL_PLAN_OK            0
#define BEVPOOL_PLAN_ROW_OVERFLOW  1   /* run_rows scratch smaller than the plan's run count: results invalid */

/* element types of feature tensors (accumulation is always fp32) */
#define BEVPOOL_F32  0
#define BEVPOOL_F16  1
#define BEVPOOL_BF16 2

int         bevpool_abi_version(void);
const char *bevpool_error_string(int code);
/* number of CUDA kernels this library has launched in this process (memsets not counted) */
int64_t     bevpool_launch_count(void);

/* ---- plan: cell index + stable sort of kept points by BEV cell -------------------
 * Replaces the per-call index work of voxel_pooling_forward_cuda.cu:19-29 (bounds
 * test, z-collapse, pos_memo).  geom_xyz: int32 (B, Np, 3) contiguous, voxel_num
 * = [X, Y, Z].  A plan depends only on geom_xyz and can be reused while the camera
 * geometry is unchanged.                                                          */
int bevpool_plan_sizes(int batch, int64_t num_points, int num_voxel_x, int num_voxel_y,
                       size_t *plan_bytes, size_t *temp_bytes);
int bevpool_plan_build(const int32_t *geom_xyz, int batch, int64_t num_points,
                       int num_voxel_x, int num_voxel_y, int num_voxel_z,
                       void *plan, void *temp, void *stream);
/* the reference's pos_memo (voxel_pooling.py:40, .cu:27-29): int32 (B, Np, 3) = (b, y, x) or -1 */
int bevpool_plan_pos_memo(const void *plan, int batch, int64_t num_points, int num_voxel_x,
                          int num_voxel_y, int32_t *pos_memo, void *stream);
/* status word of a plan (point or run plan): 0, or BEVPOOL_PLAN_* raised on the device by a consumer kernel.
 * Synchronises `stream`. */
int bevpool_plan_status(const void *plan, int *status_host, void *stream);
/* device pointers into a built plan (for tests / diagnostics) */
int bevpool_plan_views(const void *plan, int batch, int64_t num_points, int num_voxel_x,
                       int num_voxel_y, const int32_t **cell_of_point,
                       const int32_t **cell_start, const int32_t **sorted_ids);

/* ---- drop-in op: voxel_pooling(geom_xyz, input_features, voxel_num) --------------
 * forward  (voxel_pooling.py:10-55 + .cu:9-36): features (B, Np, C) -> out (B, Y, X, C),
 *          every cell written exactly once (no pre-zeroing needed), deterministic.
 *          `workspace`: bevpool_forward_workspace_bytes() bytes of scratch (partial sums of
 *          cells cut by the even-share partition of the point list); contents are don't-care.
 * backward (voxel_pooling.py:58-69): grad_out given as (B, Y, X, C) rows ->
 *          grad_features (B, Np, C), dropped points get zeros.                      */
int bevpool_forward_workspace_bytes(int channels, size_t *bytes);   /* for both forward entry points */
int bevpool_forward(const void *plan, const void *features, void *out_nhwc, int dtype,
                    int batch, int64_t num_points, int channels, int num_voxel_x,
                    int num_voxel_y, void *workspace, void *stream);
int bevpool_backward(const void *plan, const void *grad_out_nhwc, void *grad_features,
                     int dtype, int batch, int64_t num_points, int channels,
                     int num_voxel_x, int num_voxel_y, void *stream);

/* The reference's native entry point in one call: same argument list as
 * voxel_pooling_forward_kernel_launcher (ops/voxel_pooling/src/voxel_pooling_forward_cuda.cu:38-42, declared at
 * voxel_pooling_forward.cpp:21-22) = plan + pos_memo + forward.  Scratch comes from cudaMallocAsync on `stream`
 * (the one entry point that allocates: the reference signature has no workspace argument).  The library also
 * exports the C++ symbol `voxel_pooling_forward_kernel_launcher(int x6, const int*, const float*, float*, int*,
 * cudaStream_t)` itself, so the reference's voxel_pooling_forward.cpp links against libbevpool_sm100 unchanged.
 * output_features (B, Y, X, C) is fully written (no pre-zeroing needed), pos_memo (B, Np, 3) fully written.        */
int bevpool_voxel_pooling_forward_launcher(int batch_size, int num_points, int num_channels, int num_voxel_x,
                                           int num_voxel_y, int num_voxel_z, const int *geom_xyz,
                                           const float *input_features, float *output_features, int *pos_memo,
                                           void *stream);

/* ---- fused op: depth (x) context outer product never materialised ----------------
 * Replaces layers/backbones/lss_fpn.py:441-464 + the op.  Points are enumerated
 * (b, n, d, h, w) like the reference's (B, N, D, H, W, C) tensor, Np = N*D*H*W.
 * depth (B*N, D, H, W); context_nhwc / grad_context_nhwc (B*N, H, W, C): pixel rows of C
 * contiguous channels (channels_last); bevpool_transpose converts from / to (B*N, C, H, W).   */
int bevpool_fused_forward(const void *plan, const void *depth, const void *context_nhwc,
                          void *out_nhwc, int dtype, int batch, int num_cams, int depth_bins,
                          int feat_h, int feat_w, int channels, int num_voxel_x,
                          int num_voxel_y, void *workspace, void *stream);
int bevpool_fused_backward(const void *plan, const void *grad_out_nhwc, const void *depth,
                           const void *context_nhwc, void *grad_depth, void *grad_context_nhwc,
                           int dtype, int batch, int num_cams, int depth_bins, int feat_h,
                           int feat_w, int channels, int num_voxel_x, int num_voxel_y,
                           void *stream);

/* ---- fused op on a RUN plan (fp32, channels in {32, 64, 80, 96, 128}) -------------------------
 * Same replacement as above (lss_fpn.py:441-464 + the op), restructured around the frustum: a RUN is
 * a set of vertically adjacent frustum points (same image, depth bin and column; consecutive rows
 * inside one block of 16 rows) that fall into the same BEV cell -- for a level camera every kept
 * point of a (depth bin, column) pair.  The plan sorts runs, not points (an order of magnitude fewer),
 * and the forward never gathers context rows from global memory:
 *   stage A  run_rows[slot] = sum over the run's rows h of depth[d,h,w] * context[h,w,:]
 *            (context rows of a 16x4-pixel tile staged in shared memory)
 *   stage B  out[cell]      = sum of the cell's run rows in slot order (zeros for empty cells, written
 *            by spare CTAs of stage A while it runs)
 * bevpool_runplan_build: geom_xyz int32 (B, N, D, H, W, 3); the plan buffer has the layout of a point
 * plan (cell_of_point is identical; cell_start / sorted_ids / sorted_cells describe RUNS: the first
 * point of each run, ordered by (cell, point id)) plus run_code int32[B*Np]: the run's slot for the
 * first point of a run, -2 for its continuation points, -1 for dropped points.
 * Any grid size.  run_rows: caller-owned scratch of run_rows_capacity rows of `channels` floats;
 * capacity must be >= the largest number of runs in any group of BEVPOOL_RUN_CHUNK (default 8)
 * consecutive samples (default: all) -- the total run count cell_start[B*X*Y] always suffices.
 * workspace: bevpool_forward_workspace_bytes(channels) bytes, as for the other forward entry points.
 * The backward entry points above accept a run plan unchanged (they only read cell_of_point).   */
int bevpool_runplan_sizes(int batch, int num_cams, int depth_bins, int feat_h, int feat_w, int num_voxel_x,
                          int num_voxel_y, size_t *plan_bytes, size_t *temp_bytes);
int bevpool_runplan_build(const int32_t *geom_xyz, int batch, int num_cams, int depth_bins, int feat_h,
                          int feat_w, int num_voxel_x, int num_voxel_y, int num_voxel_z, void *plan,
                          void *temp, void *stream);
int bevpool_runplan_views(const void *plan, int batch, int64_t num_points, int num_voxel_x,
                          int num_voxel_y, const int32_t **cell_of_point, const int32_t **cell_start,
                          const int32_t **sorted_ids, const int32_t **sorted_cells,
                          const int32_t **run_code);
/* pair records of a run plan: int32x4 per (sample, image, depth bin, 16-row block, column), in that order --
 * {in-sample cell of the pair's first kept row or -1, rows in that cell (bits 0..15) | kept rows elsewhere (bits
 * 16..31), slot of the run starting at the first kept row, number of runs in the pair}.  The fused kernels read
 * these 16 bytes per 16 points instead of cell_of_point / run_code wherever a pair holds a single run.          */
int bevpool_runplan_pair_records(const void *plan, int batch, int64_t num_points, int num_voxel_x,
                                 int num_voxel_y, const void **pair_rec);
int bevpool_fused_forward_runs(const void *plan, const void *depth, const void *context_nhwc,
                               void *out_nhwc, int dtype, int batch, int num_cams, int depth_bins,
                               int feat_h, int feat_w, int channels, int num_voxel_x, int num_voxel_y,
                               void *run_rows, int64_t run_rows_capacity, void *workspace, void *stream);

/* The same two operators on the reference's own tensor layout: context and its gradient as (B*N, C, H, W)
 * (what DepthNet produces, layers/backbones/lss_fpn.py:441-443).  The kernels read / write the NCHW tensors
 * through TMA tensor maps (boxes of 4 columns x 16 rows x C channels), so no layout pass is needed.
 * fp32, channels in {32, 64, 80, 96, 128}, feat_w % 4 == 0 (else BEVPOOL_E_ALIGN: use the pixel-row entry points).
 * run_rows_capacity may be smaller than the run count only by mistake: the kernels then never touch memory
 * beyond the scratch, the output is invalid and the plan's status word is raised.                          */
int bevpool_fused_forward_runs_nchw(const void *plan, const void *depth, const void *context_nchw,
                                    void *out_nhwc, int dtype, int batch, int num_cams, int depth_bins,
                                    int feat_h, int feat_w, int channels, int num_voxel_x, int num_voxel_y,
                                    void *run_rows, int64_t run_rows_capacity, void *workspace, void *stream);
/* Concat epilogue (models/bev_depth.py:187-189, `torch.cat([img_bev, lidar_bev], dim=1)`; also replaces the
 * `.contiguous()` of lss_fpn.py:466 for channels-last consumers): the same forward, writing its rows into a wider
 * channels-last buffer (B, Y, X, C_total).  out_rows = address of the first camera channel of cell 0; consecutive
 * cells are out_row_stride floats apart (>= channels, multiple of 4); the other channels of a row are not touched.  */
#define BEVPOOL_FWD_NCHW_CONTEXT   1   /* context is (B*N, C, H, W); else pixel rows (B*N, H, W, C)                    */
#define BEVPOOL_FWD_OUT_PREZEROED  2   /* the kernels write the rows of occupied cells only and leave the others as    */
                                       /* they are: for output rows the caller zero-filled (e.g. on a side stream      */
                                       /* while the plan was being built) or whose empty cells are never read          */
int bevpool_fused_forward_runs_into(const void *plan, const void *depth, const void *context, int flags,
                                    void *out_rows, int64_t out_row_stride, int dtype, int batch, int num_cams,
                                    int depth_bins, int feat_h, int feat_w, int channels, int num_voxel_x,
                                    int num_voxel_y, void *run_rows, int64_t run_rows_capacity, void *workspace,
                                    void *stream);
/* Softmax folded into the forward (lss_fpn.py:423 + :441-443): the kernel reads DepthNet's output tensor itself --
 * depth_feature (B*N, feature_channels, H, W) fp32 NCHW, logits in channels [0, depth_bins), context in channels
 * [context_channel_offset, +channels) -- so neither the probability tensor nor the channel slices are ever made.
 * stats: scratch of 8 * B*N * feat_h * feat_w bytes.  out_rows / out_row_stride as in ..._runs_into (0 = channels).  */
int bevpool_fused_forward_runs_logits(const void *plan, const void *depth_feature, int feature_channels,
                                      int context_channel_offset, void *stats, void *out_rows, int64_t out_row_stride,
                                      int dtype, int batch, int num_cams, int depth_bins, int feat_h, int feat_w,
                                      int channels, int num_voxel_x, int num_voxel_y, void *run_rows,
                                      int64_t run_rows_capacity, void *workspace, void *stream);
/* backward on a RUN plan (pair records): context / grad_context as pixel rows (B*N, H, W, C) or, with
 * context_is_nchw != 0, as (B*N, C, H, W).  bevpool_fused_backward above accepts any plan (point plans included). */
int bevpool_fused_backward_runs(const void *plan, const void *grad_out_nhwc, const void *depth,
                                const void *context, void *grad_depth, void *grad_context, int context_is_nchw,
                                int dtype, int batch, int num_cams, int depth_bins, int feat_h, int feat_w,
                                int channels, int num_voxel_x, int num_voxel_y, void *stream);

/* ... and its counterpart for the gradient of a concatenated buffer: the gradient row of cell c starts at
 * grad_rows + c * grad_row_stride floats (>= channels, multiple of 4).  Needs feat_w % 4 == 0.                     */
int bevpool_fused_backward_runs_from(const void *plan, const void *grad_rows, int64_t grad_row_stride,
                                     const void *depth, const void *context, void *grad_depth, void *grad_context,
                                     int context_is_nchw, int dtype, int batch, int num_cams, int depth_bins,
                                     int feat_h, int feat_w, int channels, int num_voxel_x, int num_voxel_y,
                                     void *stream);

/* ---- run plan straight from the camera rig: no geom_xyz tensor -------------------------------------
 * Replaces layers/backbones/lss_fpn.py:328-361 (get_geometry) + :461-462 (index quantisation) as the
 * producer of the cell indices.  Inputs (all device pointers unless *_host):
 *   combine      float32 (B*N, 4, 4) row-major = sensor2ego @ inverse(intrin)  (lss_fpn.py:354, left in torch)
 *   frustum_x/y/d  the frustum axes of lss_fpn.py:308-326: x[W], y[H], d[D]
 *   lower_host[3]  = voxel_coord - voxel_size / 2 ; voxel_size_host[3]          (lss_fpn.py:461-462)
 *   variant      accumulation order of the 4-term dot products of `combine @ point`
 *                (0 .. bevpool_rig_num_variants()-1); the host picks the one that reproduces torch's batched
 *                matmul bit for bit on the device in use (mm_training_b200/ops/voxel_pooling/rig.py)
 * The plan has exactly the layout bevpool_runplan_build produces.  bevpool_rig_geom writes the int32
 * (B, N, D, H, W, 3) tensor the reference would have made (diagnostics and the variant self-test).       */
int bevpool_rig_num_variants(void);
int bevpool_runplan_rig_sizes(int batch, int num_cams, int depth_bins, int feat_h, int feat_w,
                              int num_voxel_x, int num_voxel_y, size_t *plan_bytes, size_t *temp_bytes);
int bevpool_runplan_build_rig(const float *combine, const float *frustum_x, const float *frustum_y,
                              const float *frustum_d, const float *lower_host, const float *voxel_size_host,
                              int variant, int batch, int num_cams, int depth_bins, int feat_h, int feat_w,
                              int num_voxel_x, int num_voxel_y, int num_voxel_z, void *plan, void *temp,
                              void *stream);
int bevpool_rig_geom(const float *combine, const float *frustum_x, const float *frustum_y,
                     const float *frustum_d, const float *lower_host, const float *voxel_size_host, int variant,
                     int batch, int num_cams, int depth_bins, int feat_h, int feat_w, int32_t *geom_xyz,
                     void *stream);

/* ---- gradient layout: grad_out (B, C, Y, X) contiguous -> rows (B, Y, X, C) --------------
 * Only rows of cells that received a point are written (the backward kernels read no
 * others); the rest of `rows_nhwc` is left untouched.                                 */
int bevpool_grad_rows(const void *plan, const void *grad_out_nchw, void *rows_nhwc, int dtype,
                      int batch, int64_t num_points, int channels, int num_voxel_x,
                      int num_voxel_y, void *stream);

/* ---- layout helper: (batch, rows, cols) -> (batch, cols, rows), e.g. NCHW <-> NHWC */
int bevpool_transpose(const void *in, void *out, int dtype, int batch, int64_t rows,
                      int64_t cols, void *stream);

/* ---- BEV augmentation warp: kornia warp_affine(src, M, dsize, 'bilinear', 'zeros', align_corners=True) -------------
 * What models/bev_depth.py's bev_augment_image applies to the pooled camera BEV with the BDA matrix.  fp32 rows of
 * `channels` floats (channels % 4 == 0), channels-last: source cell (b, y, x) at src_rows + ((b*src_h + y)*src_w + x)
 * * src_row_stride floats, destination pixels likewise with out_row_stride (strides >= channels, multiples of 4; the
 * rows may sit inside a wider buffer such as the concatenated BEV features).  All sizes >= 2.
 *   theta   device float32 (batch, 2, 3): kornia's normalised destination -> normalised source matrix, i.e.
 *           inverse(N(dst) @ [M; 0 0 1] @ inverse(N(src)))[:, :2] with N(h, w) = [[2/(w-1), 0, -1], [0, 2/(h-1), -1],
 *           [0, 0, 1]] (computed from M in torch: mm_training_b200/ops/bev_augment.py)
 *   cell_start  optional (NULL or a pooling plan's CSR, batch*src_h*src_w + 1 entries): source cells with
 *           cell_start[c + 1] == cell_start[c] are zero rows.  Forward: never read (same result, bit for bit, as a row
 *           of zeros).  Backward: gradient rows are written for occupied cells only; the others are left untouched.
 * forward  every destination element is written once (zeros included).  Taps are summed in the order nw, ne, sw, se.
 * backward grad_src = adjoint of the forward, gathered per source cell in ascending destination order: no atomics,
 *          bit-stable.  Its cost per cell grows with 4 / |det A| (A: the destination -> source pixel map), i.e. with
 *          the magnification of the warp.  A non-finite theta gives zero rows in both directions.                     */
int bevpool_warp_affine_forward(const float *theta, const void *src_rows, int64_t src_row_stride, void *out_rows,
                                int64_t out_row_stride, const int32_t *cell_start, int batch, int channels, int src_h,
                                int src_w, int dst_h, int dst_w, void *stream);
int bevpool_warp_affine_backward(const float *theta, const void *grad_out_rows, int64_t grad_out_row_stride,
                                 void *grad_src_rows, int64_t grad_src_row_stride, const int32_t *cell_start, int batch,
                                 int channels, int src_h, int src_w, int dst_h, int dst_w, void *stream);

/* ---- nearest resampling of the LiDAR BEV into the concatenated rows: F.interpolate(src, size=(dst_h, dst_w),
 * mode='nearest') + torch.cat([camera_half, .], 1) ---------------------------------------------------------------------
 * What models/bev_depth.py does to the LiDAR BEV before the concat with the camera BEV, any pair of sizes (up or down).
 * Per axis src(d) = min(floor(float(d) * (float(in) / float(out))), in - 1), torch's float32 rule (ATen/native/
 * UpSample.h); the y and x maps are separable.
 *   src / grad_src  (batch, channels, src_h, src_w) of element type `dtype` (BEVPOOL_F32 / F16 / BF16): NCHW-contiguous
 *           when src_is_nchw != 0, else channels_last (pixel rows of `channels` elements, 16-byte aligned for fp32,
 *           8-byte for 16-bit types)
 *   out_rows / grad_rows  fp32 rows of the concatenated buffer: destination cell (b, y, x) at + ((b*dst_h + y)*dst_w + x)
 *           * row_stride floats (row_stride >= channels, multiple of 4; 16-byte aligned), i.e. the address of the first
 *           LiDAR channel of cell 0.  Other channels of a row are not touched.
 *   channels % 4 == 0; all sizes >= 1.
 * forward  every destination element is an exact fp32 copy of one source element (bit-equal to the stock ops).
 * backward grad_src = adjoint of the forward's own index maps: per source cell the sum over its preimage (ascending y,
 *          then ascending x: torch's CUDA upsample_nearest2d_backward order), fp32 from +0, rounded once to `dtype`.
 *          A gather (no atomics, bit-stable); every element written once, zeros for empty preimages (down-sampling).
 * bevpool_resize_nearest_index (host only, no device work): the maps the kernels use -- src_of_dst_host[d] for d <
 * out_size and first_dst_host[s] for s <= in_size (preimage of s = [first_dst[s], first_dst[s + 1])); either may be NULL. */
int bevpool_resize_nearest_into(const void *src, int dtype, int src_is_nchw, int batch, int channels, int src_h,
                                int src_w, int dst_h, int dst_w, float *out_rows, int64_t out_row_stride, void *stream);
int bevpool_resize_nearest_backward_from(const float *grad_rows, int64_t grad_row_stride, void *grad_src, int dtype,
                                         int src_is_nchw, int batch, int channels, int src_h, int src_w, int dst_h,
                                         int dst_w, void *stream);
int bevpool_resize_nearest_index(int in_size, int out_size, int32_t *src_of_dst_host, int32_t *first_dst_host);

/* ==== LiDAR / radar branch ==========================================================
 * Replaces what the reference reaches through models/bev_depth.py:181-183:
 *   mmcv `hard_voxelize_forward` (via mmdet3d `MVXTwoStageDetector.voxelize`), mmdet3d
 *   `HardSimpleVFE`, and the scatter-to-dense step of `PointPillarsScatter` /
 *   `SparseConvTensor.dense()`.  Semantics: SURVEY.md Appendix A (mmcv-full 1.7.0).
 *
 * bevvox_hard_voxelize -- a whole batch in one call.
 *   points          (total_points, F) float32, the samples' clouds concatenated in order
 *   sample_offsets  device int32[batch + 1], row offsets of each sample in `points`
 *   max_sample_points  largest per-sample point count (host value, sizes the launch)
 *   voxel_size_host[3], range_host[6] = [xmin,ymin,zmin,xmax,ymax,zmax], grid_host[3] = [gx,gy,gz]
 *   outputs are packed like mmdet3d's concatenation: rows of sample b start at voxel_base[b]
 *     voxels     (batch*max_voxels, max_points, F) float32   rows >= voxel_base[batch] untouched
 *     coors      (batch*max_voxels, 4) int32 [b, z, y, x]
 *     num_points (batch*max_voxels) int32
 *     voxel_base device int32[batch + 1] (written): row offsets; [batch] = total voxel count M
 *     voxel_mean optional (batch*max_voxels, mean_features) float32 = HardSimpleVFE, or NULL
 *   temp: bevvox_temp_bytes() bytes of scratch.
 * Grids of up to 2^26 cells per batch (the aiMotive pillar grid has 2^19 per sample) use a dense first-point table
 * like mmcv's CPU kernel, larger ones a hash table; the outputs are identical.  `voxels` and `num_points` are fully
 * overwritten (rows beyond voxel_base[batch] are zero on the dense path).  mean_features <= 16.
 * bevvox_hard_voxelize_scatter (dense path only) takes the clouds either concatenated or as a DEVICE array of `batch`
 * per-sample base pointers (points == NULL; the reference passes a list of tensors: no concatenation pass) and, with
 * canvas != NULL, also writes the dense canvas (batch, mean_features, gz, gy, gx) of the fused HardSimpleVFE mean --
 * voxelize -> VFE -> scatter of models/bev_depth.py:181-183 in one call.  canvas_is_zeroed == 0: the call writes every
 * element of the canvas (with a voxel_mean output: one in-order pass over the canvas after the voxels are final, no
 * fill; without: a zero fill on a side stream + scattered stores); != 0: the caller zero-filled it already and only the
 * occupied cells are stored.                                                                                          */
int bevvox_temp_bytes(int batch, int64_t total_points, const int *grid_host, int max_voxels, int max_points,
                      size_t *temp_bytes);
int bevvox_hard_voxelize(const float *points, const int32_t *sample_offsets, int batch,
                         int64_t total_points, int64_t max_sample_points, int num_features,
                         const float *voxel_size_host, const float *range_host,
                         const int *grid_host, int max_points, int max_voxels, float *voxels,
                         int32_t *coors, int32_t *num_points, int32_t *voxel_base,
                         float *voxel_mean, int mean_features, void *temp, void *stream);
int bevvox_hard_voxelize_scatter(const float *points, const float *const *sample_ptrs,
                                 const int32_t *sample_offsets, int batch, int64_t total_points,
                                 int64_t max_sample_points, int num_features, const float *voxel_size_host,
                                 const float *range_host, const int *grid_host, int max_points, int max_voxels,
                                 float *voxels, int32_t *coors, int32_t *num_points, int32_t *voxel_base,
                                 float *voxel_mean, int mean_features, float *canvas, int canvas_is_zeroed, void *temp,
                                 void *stream);
/* mmcv dynamic voxelization: coors (num_points, 3) int32 [z, y, x], -1 for out-of-range points */
int bevvox_dynamic_voxelize(const float *points, int64_t num_points, int num_features,
                            const float *voxel_size_host, const float *range_host,
                            const int *grid_host, int32_t *coors, void *stream);

/* pillar scatter: voxel_features (M, C), coors (M, 4) [b, z, y, x] -> canvas (B, C, nz, ny, nx)
 * (== (B, C*nz, ny, nx)); every canvas element is written exactly once (no pre-zeroing).
 * index_map: scratch int32 (B*nz*ny*nx), or NULL when the caller guarantees unique coordinates (the output of hard
 * voxelization): then the canvas is zero-filled at DRAM speed and every (voxel, channel) is one store.
 * backward = gather of grad_canvas at coors.                                                 */
int pillar_scatter_forward(const void *voxel_features, const int32_t *coors, int64_t num_voxels,
                           int channels, int dtype, int batch, int nz, int ny, int nx,
                           void *canvas, int32_t *index_map, void *stream);
int pillar_scatter_backward(const void *grad_canvas, const int32_t *coors, int64_t num_voxels,
                            int channels, int dtype, int batch, int nz, int ny, int nx,
                            void *grad_voxel_features, void *stream);

/* ==== depth labels for the depth loss ================================================
 * Replaces exps/mm_training_aim.py:115-162 (get_depth_labels / get_depth_image: python loop over batch x sweep x
 * camera, projection of the LiDAR cloud into every image, `depth_map[v, u] = depth`) and :180-215
 * (get_downsampled_gt_depth: min over each downsample x downsample block, bin index, one_hot).
 *   sample_ptrs     DEVICE array of `batch` pointers to the samples' clouds, (Np_b, num_features) float32, xyz first
 *   sample_counts   device int32[batch]: Np_b;  max_points = largest Np_b (host value, sizes the launch)
 *   bda_inv         (batch, 3, 3) float32 = inverse(bda_mat[:3,:3]) (:126-127; the cloud is un-augmented with it)
 *   extrinsics / intrinsics  (batch * images_per_sample, 4, 4) float32, images ordered (sweep, camera) like :120-125
 *   bin_offset = d_bound[0] - d_bound[2], bin_step = d_bound[2] (as float32, :207-208)
 *   labels          (batch * images_per_sample * (img_h/ds) * (img_w/ds), depth_channels) float32 one-hot, written once
 *   bins            optional int32 per cell: the bin index (0 = no return / out of range); may be NULL
 *   scratch         bevlabel_scratch_bytes(): one 64-bit word per full-resolution pixel.  The call leaves it zeroed;
 *                   pass scratch_is_clean != 0 on later calls with the same buffer to skip the memset.
 * Several points in one pixel: the LAST point in cloud order wins (the reference's CPU behaviour; its CUDA
 * index_put_ picks an arbitrary one).  Arithmetic order: see csrc/depth_labels.cu.                                   */
int bevlabel_scratch_bytes(int num_images, int img_h, int img_w, size_t *bytes);
int bevlabel_depth_labels(const float *const *sample_ptrs, const int32_t *sample_counts, int num_features,
                          int batch, int images_per_sample, int64_t max_points, const float *bda_inv,
                          const float *extrinsics, const float *intrinsics, int img_h, int img_w,
                          int downsample, float bin_offset, float bin_step, int depth_channels,
                          float *labels, int32_t *bins, void *scratch, int scratch_is_clean, void *stream);

/* ==== depth distribution: softmax over D + depth-oracle overwrite in one pass ==========
 * Replaces layers/backbones/lss_fpn.py:423 (`depth_feature[:, :D].softmax(1)`) and the oracle branch :427-434
 * (max over D, two permute + contiguous copies, masked index_put, permuted view).
 *   logits   (num_images, >= depth_bins, H, W): the first depth_bins channels of DepthNet's output, element type
 *            `dtype`; consecutive images are logits_image_stride ELEMENTS apart (so the channel slice needs no copy)
 *   oracle   optional float32 (num_images, depth_bins, H, W): pixels whose max over D is > 0 take the oracle's
 *            distribution (:428-432); NULL = plain softmax
 *   prob     float32 (num_images, depth_bins, H, W): the softmax (what the depth loss consumes, :466)
 *   used     float32, same shape: the distribution the pooling consumes (required iff oracle != NULL)
 * backward: grad_logits = prob * (g - sum_d prob * g), g = grad_prob + (pixel not overwritten ? grad_used : 0);
 *           either gradient may be NULL; grad_logits (num_images, depth_bins, H, W) contiguous, element type `dtype`. */
int bevdepth_softmax_forward(const void *logits, int dtype, int64_t logits_image_stride, const float *oracle,
                             int num_images, int depth_bins, int feat_h, int feat_w, float *prob, float *used,
                             void *stream);
int bevdepth_softmax_backward(const float *prob, const float *grad_prob, const float *grad_used,
                              const float *oracle, int num_images, int depth_bins, int feat_h, int feat_w,
                              void *grad_logits, int dtype, void *stream);

/* ---- depth loss: binary cross-entropy of the depth distribution against the LiDAR depth labels --------------------
 * Replaces exps/mm_training_aim.py:163-176 (get_depth_loss): permute + contiguous copy of the predictions, max over D
 * of the labels, two boolean-mask gathers, F.binary_cross_entropy, sum / max(1.0, fg.sum()) -- with no host sync.
 *   prob     float32 (num_images, depth_bins, H, W) contiguous (what bevdepth_softmax_forward writes)
 *   labels   float32 (num_images * H * W, depth_bins) rows, pixel r = (image * H + y) * W + x; OR
 *   bins     int32 (num_images * H * W): bin b in [0, depth_bins) is the one-hot row of b, anything else a zero row
 *            (bevlabel_depth_labels' `bins`).  Exactly one of labels / bins is non-NULL.  One-hot labels give the same
 *            bits in both forms.
 *   A pixel is foreground when the max of its label row is > 0 (a row holding a NaN is background, as in torch.max).
 *   Per element, fp32 (torch's CUDA kernel): e = (t - 1) * max(log1p(-p), -100) - t * max(log(p), -100); per pixel the
 *   fp32 sum in ascending bin order; over the foreground pixels an fp64 sum in a fixed order, rounded once to S.
 * forward  loss[0] = fl(3 * fl(S / fl(max(cnt, 1)))), fg_count[0] = cnt (device scalars).  workspace:
 *          bevdepth_loss_workspace_bytes() bytes, contents don't-care.  Bit-stable: no floating-point atomics.
 * backward g' = fl(fl(grad_loss[0] * 3) / fl(max(fg_count[0], 1))) read on the device; grad_prob (same shape as prob)
 *          = +0 + g' * (p - t) / max((1 - p) * p, 1e-12) on foreground pixels, +0 elsewhere; every element written.
 * depth_bins <= 1536 (else BEVPOOL_E_CHANNELS); pointers 4-byte aligned, the workspace 8-byte (else BEVPOOL_E_ALIGN). */
int bevdepth_loss_workspace_bytes(int num_images, int depth_bins, int feat_h, int feat_w, size_t *bytes);
int bevdepth_loss_forward(const float *prob, const float *labels, const int32_t *bins, int num_images, int depth_bins,
                          int feat_h, int feat_w, void *workspace, float *loss, int32_t *fg_count, void *stream);
int bevdepth_loss_backward(const float *prob, const float *labels, const int32_t *bins, const float *grad_loss,
                           const int32_t *fg_count, int num_images, int depth_bins, int feat_h, int feat_w,
                           float *grad_prob, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* BEVPOOL_SM100_H_ */

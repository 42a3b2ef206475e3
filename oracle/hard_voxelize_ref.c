/* CPU oracle for LiDAR/radar hard voxelization.  TEST INFRASTRUCTURE -- not product code.
 *
 * PARITY UNPINNED: the arithmetic the reference uses lives in mmcv-full==1.7.0
 * (`mmcv/ops/csrc/pytorch/cpu/voxelization.cpp`: dynamic_voxelize_forward_cpu_kernel,
 * hard_voxelize_forward_cpu_kernel) reached through mmdet3d==1.0.0rc4; neither is
 * vendored under the reference (call sites: models/bev_depth.py:154,181;
 * config exps/conf_aim.py:192-197) nor installed here.  This file restates the
 * published serial algorithm (SURVEY.md Appendix A.2) and is anchored by the
 * hand-derived known-answer test of Appendix A.4 (tests/test_oracle_voxelize.py).
 *
 * Semantics, strictly in point order:
 *   c_j = floor((p_j - range_min_j) / voxel_size_j)   float32 sub, float32 true division
 *   point invalid if any c_j < 0 or c_j >= grid_j
 *   a voxel is created at the first valid point of its cell unless max_voxels are
 *   already in use (then that point, and every later point of the cell, is skipped)
 *   the first max_points points of a voxel are stored in order; the rest are dropped
 *   coors are stored (z, y, x)
 *
 * Build: see oracle/Makefile  (gcc -O2 -shared -fPIC, no -ffast-math).
 */
#include <math.h>
#include <stdlib.h>
#include <string.h>

/* Returns the number of voxels produced, or -1 on allocation failure.
 * voxels: (max_voxels, max_points, F) float32, zero-initialised by the caller
 * coors:  (max_voxels, 3) int32 [z, y, x], zero-initialised by the caller
 * num_points_per_voxel: (max_voxels,) int32, zero-initialised by the caller
 * grid: [gx, gy, gz];  range: [xmin, ymin, zmin, xmax, ymax, zmax]           */
int hard_voxelize_ref(const float *points, int num_points, int num_features,
                      const float *voxel_size, const float *range, const int *grid,
                      int max_points, int max_voxels, float *voxels, int *coors,
                      int *num_points_per_voxel) {
  /* cell -> voxel id + 1 (0: no voxel yet), indexed in 64 bits: grids of 2^31 cells and more are valid.  calloc'd
   * pages are zero until written, so such a grid costs memory only where the cloud has points. */
  const long gx = grid[0], gy = grid[1], gz = grid[2];
  int *coor_to_voxelidx = (int *)calloc((size_t)gx * (size_t)gy * (size_t)gz, sizeof(int));
  if (!coor_to_voxelidx) return -1;

  int voxel_num = 0;
  for (int i = 0; i < num_points; ++i) {
    const float *p = points + (size_t)i * num_features;
    int coor[3]; /* (z, y, x) */
    int failed = 0;
    for (int j = 0; j < 3; ++j) {
      volatile float diff = p[j] - range[j];          /* keep f32 rounding of each step */
      volatile float quot = diff / voxel_size[j];
      int c = (int)floorf(quot);
      if (c < 0 || c >= grid[j]) { failed = 1; break; }
      coor[2 - j] = c;
    }
    if (failed) continue;
    long cell = ((long)coor[0] * gy + coor[1]) * gx + coor[2];
    int vid = coor_to_voxelidx[cell] - 1;
    if (vid == -1) {
      if (max_voxels != -1 && voxel_num >= max_voxels) continue;
      vid = voxel_num++;
      coor_to_voxelidx[cell] = vid + 1;
      coors[vid * 3 + 0] = coor[0];
      coors[vid * 3 + 1] = coor[1];
      coors[vid * 3 + 2] = coor[2];
    }
    int n = num_points_per_voxel[vid];
    if (max_points == -1 || n < max_points) {
      memcpy(voxels + ((size_t)vid * max_points + n) * num_features, p,
             sizeof(float) * (size_t)num_features);
      num_points_per_voxel[vid] = n + 1;
    }
  }
  free(coor_to_voxelidx);
  return voxel_num;
}

/* Dynamic voxelization (per-point coordinates only): coors (Np, 3) [z, y, x] or -1. */
void dynamic_voxelize_ref(const float *points, int num_points, int num_features,
                          const float *voxel_size, const float *range, const int *grid,
                          int *coors) {
  for (int i = 0; i < num_points; ++i) {
    const float *p = points + (size_t)i * num_features;
    int coor[3];
    int failed = 0;
    for (int j = 0; j < 3; ++j) {
      volatile float diff = p[j] - range[j];
      volatile float quot = diff / voxel_size[j];
      int c = (int)floorf(quot);
      if (c < 0 || c >= grid[j]) { failed = 1; break; }
      coor[2 - j] = c;
    }
    for (int k = 0; k < 3; ++k) coors[i * 3 + k] = failed ? -1 : coor[k];
  }
}

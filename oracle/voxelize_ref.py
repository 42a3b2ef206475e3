"""CPU oracle for the LiDAR/radar hard voxelizer, VFE mean and pillar scatter.
TEST INFRASTRUCTURE -- never imported by the product.

PARITY UNPINNED: mmcv-full==1.7.0 / mmdet3d==1.0.0rc4 / spconv are neither vendored
in the reference nor installed; nothing in the reference's ``test/`` exercises this
path.  The restatement follows SURVEY.md Appendix A (mmcv's serial CPU kernel is the
normative definition) and is anchored by the hand-derived KAT of Appendix A.4.
Call sites in the reference: ``models/bev_depth.py:181-183``; configuration
``exps/conf_aim.py:192-212``.

Two implementations of the same algorithm are kept so they can check each other:
``hard_voxelize_c`` (ctypes -> ``oracle/hard_voxelize_ref.c``) and
``hard_voxelize_numpy`` (vectorised first-occurrence formulation).
"""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


def _lib():
    global _LIB
    if _LIB is None:
        path = os.path.join(_HERE, 'libhard_voxelize_ref.so')
        if not os.path.exists(path):
            subprocess.check_call(['make', '-C', _HERE, os.path.join(_HERE, 'libhard_voxelize_ref.so')])
        lib = ctypes.CDLL(path)
        fp = ctypes.POINTER(ctypes.c_float)
        ip = ctypes.POINTER(ctypes.c_int)
        lib.hard_voxelize_ref.restype = ctypes.c_int
        lib.hard_voxelize_ref.argtypes = [fp, ctypes.c_int, ctypes.c_int, fp, fp, ip,
                                          ctypes.c_int, ctypes.c_int, fp, ip, ip]
        lib.dynamic_voxelize_ref.restype = None
        lib.dynamic_voxelize_ref.argtypes = [fp, ctypes.c_int, ctypes.c_int, fp, fp, ip, ip]
        _LIB = lib
    return _LIB


def grid_size_ref(voxel_size, point_cloud_range):
    """mmcv ``Voxelization.__init__``: float32 ``round((max - min) / voxel_size)`` -> [gx, gy, gz]."""
    r = np.asarray(point_cloud_range, dtype=np.float32)
    v = np.asarray(voxel_size, dtype=np.float32)
    return np.round((r[3:] - r[:3]) / v).astype(np.int64)


def _as_f32(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.float32))


def _ptr(a, ct):
    return a.ctypes.data_as(ctypes.POINTER(ct))


def hard_voxelize_c(points, voxel_size, point_cloud_range, max_points, max_voxels):
    """Serial C restatement.  points (Np, F) float32 ->
    (voxels (M, T, F) f32, coors (M, 3) int32 [z,y,x], num_points (M,) int32)."""
    pts = _as_f32(points)
    n, f = pts.shape if pts.ndim == 2 else (0, 0)
    vs, rng = _as_f32(voxel_size), _as_f32(point_cloud_range)
    grid = np.ascontiguousarray(grid_size_ref(voxel_size, point_cloud_range).astype(np.int32))
    voxels = np.zeros((max_voxels, max_points, f), dtype=np.float32)
    coors = np.zeros((max_voxels, 3), dtype=np.int32)
    num = np.zeros((max_voxels,), dtype=np.int32)
    m = _lib().hard_voxelize_ref(_ptr(pts, ctypes.c_float), n, f, _ptr(vs, ctypes.c_float),
                                 _ptr(rng, ctypes.c_float), _ptr(grid, ctypes.c_int),
                                 max_points, max_voxels, _ptr(voxels, ctypes.c_float),
                                 _ptr(coors, ctypes.c_int), _ptr(num, ctypes.c_int))
    assert m >= 0
    return voxels[:m], coors[:m], num[:m]


def point_coors_numpy(points, voxel_size, point_cloud_range):
    """Per-point (z, y, x) cell coordinates or -1 (mmcv dynamic voxelization):
    float32 subtract, float32 true division, floor."""
    pts = _as_f32(points)
    vs, rng = _as_f32(voxel_size), _as_f32(point_cloud_range)
    grid = grid_size_ref(voxel_size, point_cloud_range)
    c = np.floor((pts[:, :3] - rng[None, :3]) / vs[None, :])          # float32 throughout
    # first failing axis decides nothing here: a point is invalid if ANY axis fails
    valid = np.all((c >= 0) & (c < grid[None, :].astype(np.float32)), axis=1)
    ci = np.where(valid[:, None], c, -1).astype(np.int32)
    return ci[:, ::-1].copy(), valid                                     # (z, y, x)


def hard_voxelize_numpy(points, voxel_size, point_cloud_range, max_points, max_voxels):
    """Vectorised formulation of the same semantics (the one the CUDA kernels use):
    voxel id = rank of the cell's first-occurrence point index; cap on voxel id;
    in-voxel slot = number of earlier points of the same cell; cap on slot."""
    pts = _as_f32(points)
    n, f = pts.shape
    zyx, valid = point_coors_numpy(pts, voxel_size, point_cloud_range)
    gx, gy, gz = (int(v) for v in grid_size_ref(voxel_size, point_cloud_range))
    key = (zyx[:, 0].astype(np.int64) * gy + zyx[:, 1]) * gx + zyx[:, 2]
    idx = np.nonzero(valid)[0]
    if idx.size == 0:
        return (np.zeros((0, max_points, f), np.float32), np.zeros((0, 3), np.int32),
                np.zeros((0,), np.int32))
    k = key[idx]
    order = np.argsort(k, kind='stable')                 # groups cells, keeps point order inside
    ks, ids = k[order], idx[order]
    head = np.ones(ks.size, dtype=bool)
    head[1:] = ks[1:] != ks[:-1]
    seg = np.cumsum(head) - 1                            # segment id of each sorted element
    seg_start = np.nonzero(head)[0]
    first_idx = ids[seg_start]                           # first-occurrence point of each cell
    vid_of_seg = np.empty(seg_start.size, dtype=np.int64)
    vid_of_seg[np.argsort(first_idx, kind='stable')] = np.arange(seg_start.size)
    rank = np.arange(ks.size) - seg_start[seg]
    vid = vid_of_seg[seg]
    m = int(min(seg_start.size, max_voxels)) if max_voxels != -1 else seg_start.size
    keep = (vid < m) & (rank < max_points)
    voxels = np.zeros((m, max_points, f), dtype=np.float32)
    voxels[vid[keep], rank[keep]] = pts[ids[keep]]
    coors = np.zeros((m, 3), dtype=np.int32)
    sel = vid_of_seg < m
    coors[vid_of_seg[sel]] = zyx[first_idx[sel]]
    counts = np.diff(np.append(seg_start, ks.size))
    num = np.zeros((m,), dtype=np.int32)
    num[vid_of_seg[sel]] = np.minimum(counts[sel], max_points)
    return voxels, coors, num


def voxelize_batch_ref(points_list, voxel_size, point_cloud_range, max_points, max_voxels,
                       impl=hard_voxelize_c):
    """mmdet3d ``MVXTwoStageDetector.voxelize`` (SURVEY.md Appendix A.3): per sample, then
    concatenate; coors get the batch index prepended -> (voxels, num_points, coors (M,4)
    [b, z, y, x]) -- the unpack order used at ``models/bev_depth.py:181``."""
    vs, ns, cs = [], [], []
    for b, pts in enumerate(points_list):
        v, c, n = impl(np.asarray(pts), voxel_size, point_cloud_range, max_points, max_voxels)
        vs.append(v)
        ns.append(n)
        cs.append(np.concatenate([np.full((c.shape[0], 1), b, np.int32), c], axis=1))
    return np.concatenate(vs, 0), np.concatenate(ns, 0), np.concatenate(cs, 0)


def hard_simple_vfe_ref(voxels, num_points, num_features=5):
    """mmdet3d ``HardSimpleVFE``: ``voxels[:, :, :nf].sum(1) / num_points[:, None]``
    (``models/bev_depth.py:182``, ``exps/conf_aim.py:198-201``)."""
    s = voxels[:, :, :num_features].astype(np.float32).sum(axis=1, dtype=np.float32)
    return s / num_points.astype(np.float32)[:, None]


def vfe_mean_exact(voxels, num_points, nf):
    """The HardSimpleVFE mean exactly as every finalize and gather kernel of ``csrc/voxelize.cu`` computes it, in numpy
    float32: a sum that starts from +0.0f, adds the ``cnt`` filled slots one at a time in slot order (= ascending point
    index), then ONE IEEE division by ``float(cnt)``.  Rows with ``cnt == 0`` (the padding rows) are +0.  Unlike
    ``hard_simple_vfe_ref`` (numpy's pairwise ``sum``, the statement of mmdet3d's op) the summation order is fixed, so
    the kernels' means can be compared bit for bit."""
    v = np.asarray(voxels, dtype=np.float32)
    cnt = np.asarray(num_points).astype(np.int64)
    m = v.shape[0]
    s = np.zeros((m, nf), np.float32)
    out = np.zeros((m, nf), np.float32)
    full = cnt > 0
    with np.errstate(invalid='ignore', over='ignore'):     # (NaN / inf inputs propagate, as on the GPU)
        for t in range(v.shape[1]):
            live = (t < cnt)[:, None]
            s = np.where(live, s + v[:, t, :nf], s)        # (slots >= cnt are not added: -0 + +0 would be +0)
        out[full] = s[full] / cnt[full].astype(np.float32)[:, None]
    return out


def canvas_exact(voxels, num_points, coors, nf, batch_size, grid_zyx):
    """Dense canvas (B, nf*nz, ny, nx) of ``vfe_mean_exact`` at ``coors`` [b, z, y, x]: what the fused
    ``voxelize(..., scatter=True)`` writes."""
    return pillar_scatter_ref(vfe_mean_exact(voxels, num_points, nf), coors, batch_size, grid_zyx)


def pillar_scatter_ref(voxel_features, coors, batch_size, grid_zyx):
    """Scatter (M, C) voxel features to a dense zero canvas at ``coors`` [b, z, y, x]
    -> (B, C*nz, ny, nx): PointPillarsScatter for nz == 1, ``SparseConvTensor.dense()``
    + ``view(N, C*D, H, W)`` in general (SURVEY.md Appendix A.3;
    call site ``models/bev_depth.py:183``)."""
    nz, ny, nx = (int(v) for v in grid_zyx)
    vf = np.asarray(voxel_features)
    c = vf.shape[1]
    canvas = np.zeros((batch_size, c, nz, ny, nx), dtype=vf.dtype)
    co = np.asarray(coors).astype(np.int64)
    canvas[co[:, 0], :, co[:, 1], co[:, 2], co[:, 3]] = vf
    return canvas.reshape(batch_size, c * nz, ny, nx)


def pillar_scatter_backward_ref(grad_canvas, coors, grid_zyx):
    """Gradient of the scatter w.r.t. the voxel features: a gather."""
    nz, ny, nx = (int(v) for v in grid_zyx)
    b = grad_canvas.shape[0]
    g = np.asarray(grad_canvas).reshape(b, -1, nz, ny, nx)
    co = np.asarray(coors).astype(np.int64)
    return g[co[:, 0], :, co[:, 1], co[:, 2], co[:, 3]]

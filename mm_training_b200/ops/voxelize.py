"""LiDAR/radar hard voxelizer, VFE mean and pillar scatter on libbevpool_sm100.

Drop-in for the third-party pieces the reference calls at ``models/bev_depth.py:181-183``
(configuration ``exps/conf_aim.py:192-212``); names, argument order and return order follow
mmcv-full 1.7.0 / mmdet3d 1.0.0rc4 (SURVEY.md Appendix A), so a model can swap them in:

* ``Voxelization(voxel_size, point_cloud_range, max_num_points, max_voxels, deterministic)``
  -- ``mmcv.ops.Voxelization``: ``forward(points (Np, F)) -> (voxels, coors [z,y,x], num_points)``
* ``voxelize(points_list, layer) -> (voxels, num_points, coors [b,z,y,x])``
  -- ``MVXTwoStageDetector.voxelize`` (the unpack order used at ``bev_depth.py:181``); the
  whole batch runs in ONE native call instead of a per-sample python loop
* ``HardSimpleVFE(num_features)`` -- mean of the first ``num_features`` columns over valid points
* ``PointPillarsScatter(in_channels, output_shape)`` / ``pillar_scatter`` -- dense BEV canvas;
  with ``nz > 1`` it is ``SparseConvTensor.dense()`` + ``view(N, C*D, H, W)``.

Voxelizer parity is against our restatement of mmcv 1.7.0 semantics (``oracle/``); the reference
repo pins nothing here.  No CPU fallback: CPU tensors raise.
"""
from __future__ import annotations

import ctypes
import os
from typing import List, Optional, Sequence, Tuple, Union

import torch
from torch import nn
from torch.autograd import Function

from .. import _lib


def _f32_array(vals):
    return (ctypes.c_float * len(vals))(*[float(v) for v in vals])


def _i32_array(vals):
    return (ctypes.c_int * len(vals))(*[int(v) for v in vals])


def _grid_size(voxel_size, point_cloud_range) -> List[int]:
    """mmcv: ``torch.round((range[3:] - range[:3]) / voxel_size).long()`` in float32 -> [gx, gy, gz]."""
    r = torch.tensor(point_cloud_range, dtype=torch.float32)
    v = torch.tensor(voxel_size, dtype=torch.float32)
    return torch.round((r[3:] - r[:3]) / v).long().tolist()


_OFFSETS_CACHE = {}


def _offsets_tensor(offs: tuple, dev) -> torch.Tensor:
    """Device copy of the samples' row offsets, cached per (device, point counts): repeated calls with the same cloud
    sizes (and calls under CUDA-graph capture, where a pageable H2D copy is not allowed) reuse it."""
    key = (str(dev), offs)
    t = _OFFSETS_CACHE.get(key)
    if t is None:
        if len(_OFFSETS_CACHE) > 256:
            _OFFSETS_CACHE.clear()
        t = torch.tensor(offs, dtype=torch.int32).to(dev)
        _OFFSETS_CACHE[key] = t
    return t


_PTR_CACHE = {}


def _pointer_table(ptrs: tuple, dev) -> torch.Tensor:
    """Device array of the samples' base pointers (int64), cached per pointer tuple (see ``_offsets_tensor``)."""
    key = (str(dev), ptrs)
    t = _PTR_CACHE.get(key)
    if t is None:
        if len(_PTR_CACHE) > 256:
            _PTR_CACHE.clear()
        t = torch.tensor(ptrs, dtype=torch.int64).to(dev)
        _PTR_CACHE[key] = t
    return t


def hard_voxelize_batch(points_list: Sequence[torch.Tensor], voxel_size, point_cloud_range,
                        max_num_points: int, max_voxels: int, mean_features: int = 0, padded: bool = False,
                        scatter: bool = False):
    """Voxelizes a list of (Np_i, F) float32 CUDA clouds in one native call.

    Returns ``(voxels (M, T, F), num_points (M,), coors (M, 4) [b,z,y,x], voxel_base (B+1,), voxel_mean
    (M, mean_features) or None)`` with the samples' voxels concatenated in order (mmdet3d's packing).  M is
    data dependent, so the exact-size result costs ONE D2H sync (mmcv pays one per sample) and ``voxel_base`` comes
    back on the CPU.  ``padded=True`` skips the sync (CUDA-graph capturable): the tensors keep their ``B *
    max_voxels`` rows -- every row >= voxel_base[B] of ``voxels``, ``num_points``, ``coors`` and ``voxel_mean`` is zero,
    on the dense-table and the hash pipeline alike -- and ``voxel_base`` stays on the device.
    ``scatter=True`` (needs ``mean_features``) appends the dense BEV canvas ``(B, mean_features * gz, gy, gx)`` of the
    fused HardSimpleVFE mean: voxelize -> VFE -> scatter of ``models/bev_depth.py:181-183`` in one call.  Only the live
    rows reach it.  The mean is mmdet3d's, summed in float32 from +0 over the voxel's points in point order and divided
    once by the count (``oracle.voxelize_ref.vfe_mean_exact``), bit for bit on every pipeline.
    """
    assert len(points_list) > 0
    _lib.require_cuda(*points_list)
    dev = points_list[0].device
    F = int(points_list[0].shape[1])
    counts = [int(p.shape[0]) for p in points_list]
    for p in points_list:
        if p.dtype != torch.float32 or p.dim() != 2 or p.shape[1] != F:
            raise TypeError('points must be float32 (Np, F) tensors with the same F')
    B = len(points_list)
    total = sum(counts)
    offs = [0]
    for c in counts:
        offs.append(offs[-1] + c)
    grid = _grid_size(voxel_size, point_cloud_range)
    grid_c = _i32_array(grid)
    L = _lib.lib()
    tb = ctypes.c_size_t()
    _lib.check(L.bevvox_temp_bytes(B, total, grid_c, max_voxels, max_num_points, ctypes.byref(tb)), 'bevvox_temp_bytes')
    assert not scatter or mean_features > 0, 'scatter=True needs mean_features'
    gx, gy, gz = grid
    dense = B * gx * gy * gz <= (1 << 26) and os.environ.get('BEVVOX_FORCE_HASH', '0') != '1'
    with torch.cuda.device(dev):
        offsets = _offsets_tensor(tuple(offs), dev)
        points_list = [p.contiguous() for p in points_list]
        if dense and B > 1:          # the kernels read the list through a device array of base pointers: no torch.cat
            points, sample_ptrs = None, _pointer_table(tuple(p.data_ptr() for p in points_list), dev)
        else:
            points, sample_ptrs = (points_list[0] if B == 1 else torch.cat(points_list, 0)), None
        rows = B * max_voxels
        voxels = torch.empty(rows, max_num_points, F, dtype=torch.float32, device=dev)
        coors = torch.empty(rows, 4, dtype=torch.int32, device=dev)
        num_points = torch.empty(rows, dtype=torch.int32, device=dev)
        voxel_base = torch.empty(B + 1, dtype=torch.int32, device=dev)
        mean = torch.empty(rows, mean_features, dtype=torch.float32, device=dev) if mean_features > 0 else None
        temp = torch.empty(tb.value, dtype=torch.uint8, device=dev)
        tail = [offsets.data_ptr(), B, total, max(counts), F,
                _f32_array(voxel_size), _f32_array(point_cloud_range), grid_c, max_num_points, max_voxels,
                voxels.data_ptr(), coors.data_ptr(), num_points.data_ptr(), voxel_base.data_ptr(),
                mean.data_ptr() if mean is not None else None, mean_features]
        # (the canvas takes only the voxel_base[B] live rows, counted on the device, on both paths)
        canvas = torch.empty(B, mean_features * gz, gy, gx, dtype=torch.float32, device=dev) if scatter else None
        _lib.check(L.bevvox_hard_voxelize_scatter(
            points.data_ptr() if (points is not None and total > 0) else None,
            sample_ptrs.data_ptr() if sample_ptrs is not None else None, *tail,
            canvas.data_ptr() if canvas is not None else None, 0, temp.data_ptr(), _lib.stream_ptr(dev)),
            'bevvox_hard_voxelize_scatter')
        if padded:
            out = (voxels, num_points, coors, voxel_base, mean)
            return out + (canvas,) if scatter else out
        base = voxel_base.cpu()
    M = int(base[-1])
    out = (voxels[:M], num_points[:M], coors[:M], base, (mean[:M] if mean is not None else None))
    return out + (canvas,) if scatter else out


def dynamic_voxelize(points: torch.Tensor, voxel_size, point_cloud_range) -> torch.Tensor:
    """mmcv dynamic voxelization: (Np, 3) int32 [z, y, x], -1 for out-of-range points."""
    _lib.require_cuda(points)
    if points.dtype != torch.float32 or points.dim() != 2:
        raise TypeError('points must be a float32 (Np, F) tensor')
    points = points.contiguous()
    coors = torch.empty(points.shape[0], 3, dtype=torch.int32, device=points.device)
    with torch.cuda.device(points.device):
        _lib.check(_lib.lib().bevvox_dynamic_voxelize(
            points.data_ptr() if points.shape[0] else None, points.shape[0], points.shape[1], _f32_array(voxel_size),
            _f32_array(point_cloud_range), _i32_array(_grid_size(voxel_size, point_cloud_range)),
            coors.data_ptr() if points.shape[0] else None, _lib.stream_ptr(points.device)), 'bevvox_dynamic_voxelize')
    return coors


class Voxelization(nn.Module):
    """``mmcv.ops.Voxelization`` (SURVEY.md Appendix A.1).  ``deterministic`` is accepted for
    signature compatibility; this implementation is always deterministic."""

    def __init__(self, voxel_size, point_cloud_range, max_num_points, max_voxels=20000, deterministic=True):
        super().__init__()
        self.voxel_size = list(voxel_size)
        self.point_cloud_range = list(point_cloud_range)
        self.max_num_points = max_num_points
        self.max_voxels = max_voxels if isinstance(max_voxels, (tuple, list)) else (max_voxels, max_voxels)
        self.deterministic = deterministic
        gx, gy, gz = _grid_size(voxel_size, point_cloud_range)
        self.grid_size = torch.tensor([gx, gy, gz])
        self.pcd_shape = [gx, gy, gz][::-1]          # [z, y, x] like mmcv (input_feat_shape + [1])[::-1]

    def _max_voxels(self) -> int:
        return self.max_voxels[0] if self.training else self.max_voxels[1]

    def forward(self, points: torch.Tensor):
        max_voxels = self._max_voxels()
        if self.max_num_points == -1 or max_voxels == -1:
            return dynamic_voxelize(points, self.voxel_size, self.point_cloud_range)
        voxels, num_points, coors, _, _ = hard_voxelize_batch([points], self.voxel_size, self.point_cloud_range,
                                                              self.max_num_points, max_voxels)
        return voxels, coors[:, 1:].contiguous(), num_points

    def __repr__(self):
        return (f'{self.__class__.__name__}(voxel_size={self.voxel_size}, point_cloud_range='
                f'{self.point_cloud_range}, max_num_points={self.max_num_points}, max_voxels={self.max_voxels}, '
                f'deterministic={self.deterministic})')


@torch.no_grad()
def voxelize(points: Sequence[torch.Tensor], layer: Voxelization, mean_features: int = 0, padded: bool = False,
             scatter: bool = False):
    """``MVXTwoStageDetector.voxelize``: ``(voxels, num_points, coors_batch [b,z,y,x])`` -- the order
    unpacked at ``models/bev_depth.py:181``.  With ``mean_features`` > 0 a fourth element, the fused
    HardSimpleVFE output, is appended; with ``scatter`` a fifth, the dense canvas of that mean.  ``padded`` skips the
    voxel-count read-back (see ``hard_voxelize_batch``) and appends the device ``voxel_base`` as the last element."""
    res = hard_voxelize_batch(points, layer.voxel_size, layer.point_cloud_range, layer.max_num_points,
                              layer._max_voxels(), mean_features, padded, scatter)
    voxels, num_points, coors, base, mean = res[:5]
    out = [voxels, num_points, coors]
    if mean_features > 0:
        out.append(mean)
    if scatter:
        out.append(res[5])
    if padded:
        out.append(base)
    return tuple(out)


class HardSimpleVFE(nn.Module):
    """mmdet3d ``HardSimpleVFE``: ``features[:, :, :nf].sum(1) / num_points`` (``conf_aim.py:198-201``).
    A few dozen bytes per voxel of dense math: plain torch, or free when fused into the voxelizer
    (``voxelize(..., mean_features=nf)``)."""

    def __init__(self, num_features: int = 4):
        super().__init__()
        self.num_features = num_features

    def forward(self, features, num_points, coors=None):
        points_mean = features[:, :, :self.num_features].sum(dim=1, keepdim=False) / \
            num_points.type_as(features).view(-1, 1)
        return points_mean.contiguous()


class _PillarScatter(Function):
    @staticmethod
    def forward(ctx, voxel_features, coors, batch_size, grid_zyx, unique_coors=False):
        _lib.require_cuda(voxel_features, coors)
        nz, ny, nx = (int(v) for v in grid_zyx)
        feats = voxel_features.contiguous()
        co = coors.contiguous()
        if co.dtype != torch.int32:
            co = co.int()
        M, C = feats.shape
        assert co.shape == (M, 4)
        dev = feats.device
        with torch.cuda.device(dev):
            canvas = torch.empty(batch_size, C, nz, ny, nx, dtype=feats.dtype, device=dev)
            index_map = None if unique_coors else torch.empty(batch_size * nz * ny * nx, dtype=torch.int32, device=dev)
            _lib.check(_lib.lib().pillar_scatter_forward(
                feats.data_ptr() if M else None, co.data_ptr() if M else None, M, C, _lib.dtype_code(feats),
                batch_size, nz, ny, nx, canvas.data_ptr(), index_map.data_ptr() if index_map is not None else None,
                _lib.stream_ptr(dev)), 'pillar_scatter_forward')
        ctx.save_for_backward(co)
        ctx.dims = (M, C, batch_size, nz, ny, nx)
        return canvas.view(batch_size, C * nz, ny, nx)

    @staticmethod
    def backward(ctx, grad_canvas):
        (co,) = ctx.saved_tensors
        M, C, B, nz, ny, nx = ctx.dims
        g = grad_canvas.contiguous()
        grad_feats = torch.empty(M, C, dtype=g.dtype, device=g.device)
        with torch.cuda.device(g.device):
            _lib.check(_lib.lib().pillar_scatter_backward(
                g.data_ptr(), co.data_ptr() if M else None, M, C, _lib.dtype_code(g), B, nz, ny, nx,
                grad_feats.data_ptr() if M else None, _lib.stream_ptr(g.device)), 'pillar_scatter_backward')
        return grad_feats, None, None, None, None


def pillar_scatter(voxel_features: torch.Tensor, coors: torch.Tensor, batch_size: int, grid_zyx,
                   unique_coors: bool = False) -> torch.Tensor:
    """(M, C) voxel features at ``coors`` [b, z, y, x] -> dense (B, C*nz, ny, nx); differentiable
    w.r.t. the features.  ``unique_coors=True`` (true for the output of hard voxelization) takes the fast path:
    zero fill + one store per element; with duplicate coordinates the default path lets the highest row win."""
    return _PillarScatter.apply(voxel_features, coors, batch_size, tuple(grid_zyx), unique_coors)


class PointPillarsScatter(nn.Module):
    """mmdet3d ``PointPillarsScatter(in_channels, output_shape=(ny, nx))``: the scatter-to-dense step only.
    The reference's ``pts_middle_encoder`` (``models/bev_depth.py:183``, ``exps/conf_aim.py:202-212``) is a
    ``SparseEncoder``: spconv sparse 3-D convolutions (5 -> 128 channels) FOLLOWED by ``.dense()``.  The sparse
    convolution stack is out of scope here; this module replaces the ``.dense()`` / pillar-scatter step after it
    (same ``(voxel_features, coors, batch_size)`` call signature), it is not a functional replacement of the encoder."""

    def __init__(self, in_channels: int, output_shape, nz: int = 1):
        super().__init__()
        self.in_channels = in_channels
        self.ny, self.nx = int(output_shape[0]), int(output_shape[1])
        self.nz = nz

    def forward(self, voxel_features, coors, batch_size=None):
        if batch_size is None:
            batch_size = int(coors[:, 0].max().item()) + 1 if coors.shape[0] else 1
        return pillar_scatter(voxel_features, coors, batch_size, (self.nz, self.ny, self.nx))

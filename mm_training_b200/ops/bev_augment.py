"""BEV data augmentation warp on libbevpool_sm100: kornia's ``warp_affine`` as ``bev_augment_image`` applies it
(``models/bev_depth.py:69-84``) to the pooled camera BEV with the BDA matrix (a random rotation, scale and flip).

``warp_affine(src, M, dsize)`` equals ``kornia.geometry.transform.warp_affine(src, M, dsize, mode='bilinear',
padding_mode='zeros', align_corners=True)``.  The matrix kornia hands to ``F.affine_grid`` is computed from ``M`` here
with the same torch ops (``warp_theta``); the kernels (``csrc/bev_warp.cu``) evaluate ``affine_grid`` + ``grid_sample``
themselves on channels-last rows.  Unlike ``grid_sample``'s CUDA backward (floating-point atomics, refused under
``torch.use_deterministic_algorithms(True)``) the backward is a gather: bit-stable run to run.

Scope: bilinear, zeros padding, ``align_corners=True`` (kornia's defaults), float32 with a channel count divisible
by 4, no gradient with respect to ``M``.  Anything else raises; there is no stock fallback.
"""
from __future__ import annotations

from typing import Optional, Sequence

import torch
from torch.autograd import Function

from .. import _lib
from .voxel_pooling.voxel_pooling import _strided_rows, _transpose


def _normal_transform_pixel(h: int, w: int, like: torch.Tensor) -> torch.Tensor:
    """kornia's ``normal_transform_pixel``: pixel -> [-1, 1] coordinates (align_corners=True), (3, 3)."""
    n = torch.eye(3, dtype=like.dtype, device=like.device)
    n[0, 0].fill_(2.0 / (w - 1))          # fill_ with a python scalar: no host -> device copy (CUDA-graph capturable)
    n[1, 1].fill_(2.0 / (h - 1))
    n[:2, 2].fill_(-1.0)
    return n


def warp_theta(M: torch.Tensor, src_hw: Sequence[int], dsize: Sequence[int]) -> torch.Tensor:
    """(B, 2, 3) float32: the normalised destination -> source matrix kornia's ``warp_affine`` passes to
    ``F.affine_grid``, computed on ``M``'s device with kornia's ops (``inv_ex`` for its ``inverse``: the same LU values
    without a host synchronisation).  Always in fp32 or fp64, autocast off: under bf16 autocast the products would round
    the matrix to bf16 (moving the warp by whole cells) and ``inv_ex`` takes no 16-bit input."""
    with torch.autocast(device_type=M.device.type, enabled=False):
        return _warp_theta(M, src_hw, dsize)


def _warp_theta(M: torch.Tensor, src_hw: Sequence[int], dsize: Sequence[int]) -> torch.Tensor:
    H, W = (int(v) for v in src_hw)
    Hd, Wd = (int(v) for v in dsize)
    if M.dim() != 3 or tuple(M.shape[1:]) != (2, 3):
        raise ValueError(f'M must be (B, 2, 3), got {tuple(M.shape)}')
    if min(H, W, Hd, Wd) < 2:
        raise ValueError(f'source {H}x{W} and destination {Hd}x{Wd} must both be at least 2x2')
    if M.requires_grad:
        raise ValueError('warp_affine has no gradient with respect to M; pass M.detach()')
    m = M if M.dtype in (torch.float32, torch.float64) else M.float()
    m3 = torch.eye(3, dtype=m.dtype, device=m.device).repeat(m.shape[0], 1, 1)
    m3[:, :2] = m                                                   # convert_affinematrix_to_homography
    src_pix_from_norm = torch.linalg.inv_ex(_normal_transform_pixel(H, W, m), check_errors=False).inverse
    dst_norm_from_src_norm = _normal_transform_pixel(Hd, Wd, m) @ (m3 @ src_pix_from_norm)
    theta = torch.linalg.inv_ex(dst_norm_from_src_norm, check_errors=False).inverse[:, :2, :]
    return theta.float().contiguous()


def _rows(x: torch.Tensor):
    """(B, C, H, W) float32 -> (tensor whose data_ptr is the first row, row stride): zero-copy when ``x`` already is
    channels-last rows, else one tiled transpose of an NCHW copy."""
    S = _strided_rows(x)
    if S is not None:
        return x, S
    B, C, H, W = x.shape
    return _transpose(x.contiguous(), B, C, H * W), C


def warp_forward_rows(theta: torch.Tensor, src, src_stride: int, out, out_stride: int,
                      cell_start: Optional[torch.Tensor], B: int, C: int, src_hw, dsize) -> None:
    """fp32 ``src`` rows -> ``out`` rows; an fp16 / bf16 ``out`` gets the fp32 result rounded once per element."""
    H, W = src_hw
    Hd, Wd = dsize
    if out.dtype != torch.float32:
        _lib.check(_lib.lib().bevpool_warp_affine_forward16(
            theta.data_ptr(), src.data_ptr(), src_stride, out.data_ptr(), out_stride, _lib.dtype_code(out),
            None if cell_start is None else cell_start.data_ptr(), B, C, H, W, Hd, Wd, _lib.stream_ptr(theta.device)),
            'bevpool_warp_affine_forward16')
        return
    _lib.check(_lib.lib().bevpool_warp_affine_forward(
        theta.data_ptr(), src.data_ptr(), src_stride, out.data_ptr(), out_stride,
        None if cell_start is None else cell_start.data_ptr(), B, C, H, W, Hd, Wd, _lib.stream_ptr(theta.device)),
        'bevpool_warp_affine_forward')


def warp_backward_rows(theta: torch.Tensor, grad_out, grad_out_stride: int, grad_src, grad_src_stride: int,
                       cell_start: Optional[torch.Tensor], B: int, C: int, src_hw, dsize) -> None:
    """``grad_out`` rows -> fp32 ``grad_src`` rows; an fp16 / bf16 ``grad_out`` is widened exactly where it is read."""
    H, W = src_hw
    Hd, Wd = dsize
    if grad_out.dtype != torch.float32:
        _lib.check(_lib.lib().bevpool_warp_affine_backward16(
            theta.data_ptr(), grad_out.data_ptr(), grad_out_stride, _lib.dtype_code(grad_out), grad_src.data_ptr(),
            grad_src_stride, None if cell_start is None else cell_start.data_ptr(), B, C, H, W, Hd, Wd,
            _lib.stream_ptr(theta.device)), 'bevpool_warp_affine_backward16')
        return
    _lib.check(_lib.lib().bevpool_warp_affine_backward(
        theta.data_ptr(), grad_out.data_ptr(), grad_out_stride, grad_src.data_ptr(), grad_src_stride,
        None if cell_start is None else cell_start.data_ptr(), B, C, H, W, Hd, Wd, _lib.stream_ptr(theta.device)),
        'bevpool_warp_affine_backward')


def check_warp_input(src: torch.Tensor) -> None:
    _lib.require_cuda(src)
    if src.dim() != 4:
        raise ValueError(f'src must be (B, C, H, W), got {tuple(src.shape)}')
    if src.dtype != torch.float32:
        raise TypeError(f'warp_affine runs on float32 only (got {src.dtype})')
    if src.shape[1] % 4 != 0:
        raise ValueError(f'warp_affine needs a channel count divisible by 4 (got {src.shape[1]})')


class WarpAffine(Function):
    @staticmethod
    def forward(ctx, src, M, dsize):
        B, C, H, W = src.shape
        Hd, Wd = dsize
        with torch.cuda.device(src.device):
            theta = warp_theta(M, (H, W), dsize).to(src.device)
            rows, stride = _rows(src)
            out = torch.empty(B, Hd, Wd, C, dtype=torch.float32, device=src.device)
            warp_forward_rows(theta, rows, stride, out, C, None, B, C, (H, W), (Hd, Wd))
        ctx.save_for_backward(theta)
        ctx.src_hw = (H, W)
        return out.permute(0, 3, 1, 2)

    @staticmethod
    def backward(ctx, grad_out):
        (theta,) = ctx.saved_tensors
        B, C, Hd, Wd = grad_out.shape
        H, W = ctx.src_hw
        with torch.cuda.device(grad_out.device):
            rows, stride = _rows(grad_out.float())
            grad_src = torch.empty(B, H, W, C, dtype=torch.float32, device=grad_out.device)
            warp_backward_rows(theta, rows, stride, grad_src, C, None, B, C, (H, W), (Hd, Wd))
        return grad_src.permute(0, 3, 1, 2), None, None


def warp_affine(src: torch.Tensor, M: torch.Tensor, dsize: Sequence[int], mode: str = 'bilinear',
                padding_mode: str = 'zeros', align_corners: bool = True) -> torch.Tensor:
    """``kornia.geometry.transform.warp_affine`` with its defaults.  ``src`` (B, C, H, W) float32 CUDA, C % 4 == 0
    (a permuted channels-last view such as ``voxel_pooling_fused``'s output is read in place); ``M`` (B, 2, 3) maps
    source pixels (x = column, y = row) to destination pixels and gets no gradient; ``dsize`` = (H', W').  Returns
    (B, C, H', W') as a permuted view of (B, H', W', C) rows, like the pooling ops.  A singular ``M`` gives zeros."""
    if mode != 'bilinear' or padding_mode != 'zeros' or align_corners is not True:
        raise ValueError(f'warp_affine supports mode="bilinear", padding_mode="zeros", align_corners=True only '
                         f'(got {mode!r}, {padding_mode!r}, {align_corners!r})')
    check_warp_input(src)
    dsize = tuple(int(v) for v in dsize)
    if len(dsize) != 2:
        raise ValueError(f'dsize must be (H, W), got {dsize}')
    if M.shape[0] != src.shape[0]:
        raise ValueError(f'M has {M.shape[0]} matrices for a batch of {src.shape[0]}')
    return WarpAffine.apply(src, M, dsize)

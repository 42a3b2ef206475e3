"""Depth loss of the camera branch: binary cross-entropy of the depth distribution against the LiDAR depth labels, in
native kernels (csrc/depth_loss.cu), differentiable wrt the predictions.

Drop-in for ``get_depth_loss`` (``exps/mm_training_aim.py:163-176``)::

    depth_preds = depth_preds.permute(0, 2, 3, 1).contiguous().view(-1, D)
    fg_mask = torch.max(depth_labels, dim=1).values > 0.0
    loss = F.binary_cross_entropy(depth_preds[fg_mask], depth_labels[fg_mask], reduction='none').sum() \\
           / max(1.0, fg_mask.sum())
    return 3.0 * loss

``depth_loss(depth_labels, depth_preds) -> 0-dim float32 tensor``.  Unlike the reference it makes no copy of the
predictions and no host sync (the foreground count stays on the device, so a training step can be graph-captured), and
a NaN probability gives a NaN loss instead of a device assert.  The forward sum is bit-stable (fp64, fixed order); the
gradient has the bits of torch's CUDA autograd of the reference.

* ``depth_preds``: float32 (B*N, D, H, W), the probabilities ``depth_distribution`` returns.  Always fp32, whatever
  autocast is active (the reference computes the loss under ``autocast(enabled=False)``).
* ``depth_labels``: float32 holding B*N*H*W rows of D (``DepthLabelGenerator``'s labels, any shape that views as
  ``(-1, D)``), or int32 bins of B*N*H*W elements (``DepthLabelGenerator(..., return_bins=True)``): bin b in [0, D) is
  the one-hot row of b, anything else a zero row.  One-hot labels give the same bits in both forms.  Labels get no
  gradient, as in the reference.
No CPU fallback.
"""
from __future__ import annotations

import ctypes
import functools

import torch
from torch.autograd import Function

from .. import _lib


@functools.lru_cache(maxsize=64)
def _workspace_bytes(BN: int, D: int, H: int, W: int) -> int:
    n = ctypes.c_size_t()
    _lib.check(_lib.lib().bevdepth_loss_workspace_bytes(BN, D, H, W, ctypes.byref(n)), 'bevdepth_loss_workspace_bytes')
    return n.value


def _label_ptrs(labels: torch.Tensor):
    p = labels.data_ptr()
    return (p, None) if labels.dtype == torch.float32 else (None, p)


class _DepthLoss(Function):
    @staticmethod
    def forward(ctx, labels, prob):
        BN, D, H, W = prob.shape
        dev = prob.device
        dense, bins = _label_ptrs(labels)
        with torch.cuda.device(dev):
            ws = torch.empty(_workspace_bytes(BN, D, H, W), dtype=torch.uint8, device=dev)
            loss = torch.empty((), dtype=torch.float32, device=dev)
            cnt = torch.empty(1, dtype=torch.int32, device=dev)
            _lib.check(_lib.lib().bevdepth_loss_forward(
                prob.data_ptr(), dense, bins, BN, D, H, W, ws.data_ptr(), loss.data_ptr(), cnt.data_ptr(),
                _lib.stream_ptr(dev)), 'bevdepth_loss_forward')
        ctx.save_for_backward(labels, prob, cnt)
        return loss

    @staticmethod
    def backward(ctx, grad_loss):
        labels, prob, cnt = ctx.saved_tensors
        BN, D, H, W = prob.shape
        dev = prob.device
        dense, bins = _label_ptrs(labels)
        g = grad_loss.float().contiguous()
        with torch.cuda.device(dev):
            grad_prob = torch.empty_like(prob)              # (B*N, D, H, W) contiguous: what depth_distribution reads
            _lib.check(_lib.lib().bevdepth_loss_backward(
                prob.data_ptr(), dense, bins, g.data_ptr(), cnt.data_ptr(), BN, D, H, W, grad_prob.data_ptr(),
                _lib.stream_ptr(dev)), 'bevdepth_loss_backward')
        return None, grad_prob


def _validate(depth_labels: torch.Tensor, depth_preds: torch.Tensor):
    """Raises before any device work; returns the labels as a contiguous (-1, D) / (-1,) tensor and the predictions."""
    _lib.require_cuda(depth_labels, depth_preds)
    if depth_preds.dtype != torch.float32:
        raise TypeError(f'depth_loss: depth_preds must be float32 (depth_distribution returns float32), '
                        f'got {depth_preds.dtype}')
    if depth_labels.dtype not in (torch.float32, torch.int32):
        raise TypeError(f'depth_loss: depth_labels must be float32 rows or int32 bins, got {depth_labels.dtype}')
    if depth_preds.dim() != 4:
        raise ValueError(f'depth_loss: depth_preds must be (B*N, D, H, W), got shape {tuple(depth_preds.shape)}')
    if depth_labels.device != depth_preds.device:
        raise ValueError(f'depth_loss: labels on {depth_labels.device}, predictions on {depth_preds.device}')
    BN, D, H, W = depth_preds.shape
    px = BN * H * W
    if px == 0 or D == 0:
        raise ValueError(f'depth_loss: empty predictions {tuple(depth_preds.shape)}')
    want = px * D if depth_labels.dtype == torch.float32 else px
    if depth_labels.numel() != want:
        kind = f'{px} rows of {D}' if depth_labels.dtype == torch.float32 else f'{px} bins'
        raise ValueError(f'depth_loss: depth_labels {tuple(depth_labels.shape)} do not hold {kind} '
                         f'for depth_preds {tuple(depth_preds.shape)}')
    if depth_labels.requires_grad:
        raise ValueError('depth_loss: depth_labels require grad, but the loss has no gradient wrt the labels '
                         '(the reference gives them none either); pass depth_labels.detach()')
    labels = depth_labels.reshape(-1, D) if depth_labels.dtype == torch.float32 else depth_labels.reshape(-1)
    return labels.contiguous(), depth_preds.contiguous()


def depth_loss(depth_labels: torch.Tensor, depth_preds: torch.Tensor) -> torch.Tensor:
    """``get_depth_loss(depth_labels, depth_preds)``: 3 * sum of the BCE over the foreground pixels / max(1, their
    count), as a 0-dim float32 tensor; D is ``depth_preds.shape[1]``."""
    labels, prob = _validate(depth_labels, depth_preds)
    return _DepthLoss.apply(labels, prob)

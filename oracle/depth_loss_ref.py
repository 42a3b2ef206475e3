"""CPU oracle of the depth loss (csrc/depth_loss.cu, ``mm_training_b200.ops.depth_loss``).  TEST INFRASTRUCTURE --
never imported by the product.

Restates ``get_depth_loss`` (``exps/mm_training_aim.py:163-176``; ``bench_train.depth_loss_ref``) from the float32 inputs:

* ``foreground``      -- ``torch.max(row) > 0`` per label row; a row holding a NaN has a NaN max: background.
* ``loss_ref``        -- the loss in float64, with the -100 clamps and the ``max(1, cnt)`` rule; returns (L, cnt).
* ``grad_ref``        -- its gradient wrt the probabilities in float64: ``g' (p - t) / max((1 - p) p, 1e-12)`` on
  foreground rows, 0 elsewhere, ``g' = 3 g / max(cnt, 1)``; the 1e-12 is torch's float ``1e-12f`` (``EPS``).
* ``loss_f32_emulate`` -- numpy float32 emulation of the kernels' order: fp32 terms (correctly rounded logs), fp32 sum
  per pixel in ascending d, fp64 sum over pixels rounded once, then ``fl(3 * fl(S / fl(max(cnt, 1))))``.
* ``forward_bound``   -- error bound of the kernels' float32 loss against ``loss_ref``.
"""
from __future__ import annotations

import numpy as np
import torch

U32 = 2.0 ** -24                 # unit roundoff of float32
U64 = 2.0 ** -53
FLT_TRUE_MIN = 2.0 ** -149
EPS = float(np.float32(1e-12))   # torch's EPSILON is the float 1e-12f, also in its float64 kernels


def rows(depth_labels: torch.Tensor, depth_preds: torch.Tensor):
    """(labels (P, D), preds (P, D)) in the reference's pixel order (``permute(0, 2, 3, 1)``); int32 bins become
    one-hot rows (a bin outside [0, D) a zero row)."""
    D = depth_preds.shape[1]
    p = depth_preds.permute(0, 2, 3, 1).reshape(-1, D)
    if depth_labels.dtype == torch.int32:
        b = depth_labels.reshape(-1).long()
        t = torch.zeros(b.numel(), D, dtype=torch.float32)
        ok = (b >= 0) & (b < D)
        t[ok.nonzero().view(-1), b[ok]] = 1.0
    else:
        t = depth_labels.reshape(-1, D)
    return t, p


def foreground(t: torch.Tensor) -> torch.Tensor:
    """(P, D) -> (P,) bool: ``torch.max(t, 1).values > 0``, which is False for a row holding a NaN."""
    return (t > 0).any(1) & ~torch.isnan(t).any(1)


def _terms64(t64: torch.Tensor, p64: torch.Tensor):
    a = torch.clamp_min(torch.log1p(-p64), -100.0)      # clamp_min keeps a NaN, like std::max(x, -100)
    b = torch.clamp_min(torch.log(p64), -100.0)
    return (t64 - 1) * a - t64 * b, (t64 - 1).abs() * a.abs() + t64.abs() * b.abs()


def loss_ref(depth_labels: torch.Tensor, depth_preds: torch.Tensor):
    """-> (L float64 0-dim tensor, cnt int)."""
    t, p = rows(depth_labels, depth_preds)
    fg = foreground(t)
    e, _ = _terms64(t[fg].double(), p[fg].double())
    cnt = int(fg.sum())
    return 3.0 * (e.sum() / max(1, cnt)), cnt


def grad_ref(depth_labels: torch.Tensor, depth_preds: torch.Tensor, g: float = 1.0) -> torch.Tensor:
    """float64 (B*N, D, H, W) gradient of ``g * L`` wrt the predictions."""
    t, p = rows(depth_labels, depth_preds)
    fg = foreground(t)
    gs = 3.0 * g / max(1, int(fg.sum()))
    t64, p64 = t.double(), p.double()
    gr = gs * (p64 - t64) / torch.clamp_min((1 - p64) * p64, EPS)
    gr = torch.where(fg[:, None], gr, torch.zeros_like(gr))
    BN, D, H, W = depth_preds.shape
    return gr.view(BN, H, W, D).permute(0, 3, 1, 2).contiguous()


def loss_f32_emulate(depth_labels: torch.Tensor, depth_preds: torch.Tensor) -> np.float32:
    """The kernels' float32 loss, with correctly rounded logs (the kernels' logf / log1pf are within 1 ulp)."""
    f32 = np.float32
    t, p = rows(depth_labels, depth_preds)
    fg = foreground(t).numpy()
    t = t.numpy().astype(f32)
    p = p.numpy().astype(f32)
    with np.errstate(invalid='ignore', divide='ignore', over='ignore', under='ignore'):
        lp = np.log(p.astype(np.float64)).astype(f32)
        l1 = np.log1p(-p.astype(np.float64)).astype(f32)
        lp = np.where(lp < f32(-100), f32(-100), lp)
        l1 = np.where(l1 < f32(-100), f32(-100), l1)
        e = ((t - f32(1)) * l1).astype(f32) - (t * lp).astype(f32)
        s = np.zeros(t.shape[0], dtype=f32)
        for d in range(t.shape[1]):
            s = (s + e[:, d]).astype(f32)
        S = f32(np.sum(s[fg].astype(np.float64)))
        cnt = int(fg.sum())
        return f32(f32(S / f32(max(cnt, 1))) * f32(3))


def gamma(n: int, u: float = U32) -> float:
    return n * u / (1 - n * u)


def forward_bound(depth_labels: torch.Tensor, depth_preds: torch.Tensor) -> float:
    """|kernel loss - loss_ref| <= this, for finite loss_ref.

    Per term e = (t - 1) a - t b: the logs carry at most 1 ulp <= 2u relative (the -100 clamp is 1-Lipschitz and |log|
    <= 104 where it acts, so 2.1u of the clamped value; 4u covers it and subnormal results add 2^-149), t - 1, the two
    products and the subtraction one rounding each; the D-term fp32 sum of a pixel adds gamma_{D-1}.  With
    mag = |t - 1| |a| + |t| |b| per term (= |e| for t in [0, 1]) the pixel sum is within
    (gamma_{D+3} + 4u) * sum_d mag + (D + 2) 2^-149.  The fp64 sum over P pixels adds gamma^{(64)}_P of the magnitudes;
    rounding S to fp32, the division and the product by 3 add 3u |L| (4u with second-order terms):

        3 / max(cnt, 1) * [sum_fg ((gamma_{D+3} + 4u) sum_d mag + (D + 2) 2^-149) + gamma64_P sum_fg sum_d mag] + 4u |L|
    widened by 2^-20 (relative) for the fp64 reference's own rounding."""
    t, p = rows(depth_labels, depth_preds)
    fg = foreground(t)
    D = t.shape[1]
    _, mag = _terms64(t[fg].double(), p[fg].double())
    m = mag.sum(1)
    cnt = int(fg.sum())
    L, _ = loss_ref(depth_labels, depth_preds)
    pix = ((gamma(D + 3) + 4 * U32) * m + (D + 2) * FLT_TRUE_MIN).sum() + gamma(max(cnt, 1), U64) * m.sum()
    return float((3.0 / max(1, cnt) * pix + 4 * U32 * L.abs()) * (1 + 2.0 ** -20))

"""CPU oracle of the depth distribution (csrc/depth_softmax.cu and the statistics pre-pass ``depth_stats_kernel`` of
csrc/pool_runs.cu).  TEST INFRASTRUCTURE -- never imported by the product.

Restates ``layers/backbones/lss_fpn.py:423`` (``depth_feature[:, :D].softmax(1)``) and ``:427-434`` (the depth-oracle
overwrite) in float64, plus what the tests need to hold the float32 kernels to it:

* ``softmax_ref``          -- fp64 softmax of the fp32 value of every logit (fp16 / bf16 upcast exactly); same NaN
  pattern as ``torch.softmax`` for rows holding -inf only, +inf or NaN.
* ``overwrite_ref``        -- pixels whose oracle has a positive entry take the oracle's row.
* ``softmax_backward_ref`` -- ``p * (g - sum_d p * g)`` in fp64 from the kernel's OWN fp32 probabilities, with the
  magnitude that bounds the kernel's float32 rounding.
* ``online_softmax_f32``   -- numpy float32 emulation of the kernels' loop order (online max / sum, then normalise),
  the same idea as ``depth_labels_ref.depth_labels_exact``; ``skip_neg_inf=False`` restates the loop as it was before
  a leading -inf was special-cased (it yields NaN for such rows).
* ``forward_rel_bound``    -- per-element relative error bound of the kernels' float32 softmax.
* ``sum_bound`` / ``round_bracket`` -- error bound of an fp32 sum of n terms and the interval a value within that
  bound must land in once rounded to fp16 / bf16.
"""
from __future__ import annotations

import numpy as np
import torch

U32 = 2.0 ** -24                 # unit roundoff of float32
FLT_MIN = 2.0 ** -126            # smallest normal float32
FLT_TRUE_MIN = 2.0 ** -149       # smallest subnormal float32


def softmax_ref(logits: torch.Tensor, D: int) -> torch.Tensor:
    """(BN, >= D, H, W) logits of any float dtype -> (BN, D, H, W) float64 softmax over the first D channels."""
    x = logits[:, :D].float().double()
    m = x.amax(1, keepdim=True)                  # NaN if the row holds a NaN, -inf if it holds -inf only
    e = torch.exp(x - m)                         # a +inf or NaN max, or an all -inf row, gives NaN here
    return e / e.sum(1, keepdim=True)


def foreground(oracle: torch.Tensor) -> torch.Tensor:
    """(BN, 1, H, W) bool: the pixel has a LiDAR return (``lss_fpn.py:428``: ``max_d oracle > 0``; -0.0 is not)."""
    return oracle.amax(1, keepdim=True) > 0


def overwrite_ref(prob: torch.Tensor, oracle: torch.Tensor) -> torch.Tensor:
    """``lss_fpn.py:427-434``: foreground pixels take the oracle's row, the others keep ``prob``."""
    return torch.where(foreground(oracle), oracle.to(prob.dtype), prob)


def softmax_backward_ref(prob32: torch.Tensor, grad_prob, grad_used, oracle=None):
    """Gradient wrt the logits from the kernel's own fp32 probabilities, in fp64.

    ``g = grad_prob + (pixel is foreground ? 0 : grad_used)`` (either gradient may be None), result ``p * (g - S)``
    with ``S = sum_d p * g``.  Also returns ``mag = p * (|g| + sum_d p * |g|)``: the float32 kernel (one rounding in
    g, a D-term dot product, one subtraction, one product) is within ``sum_bound(D + 3, mag)`` of the result."""
    p = prob32.double()
    g = torch.zeros_like(p)
    if grad_prob is not None:
        g = g + grad_prob.double()
    if grad_used is not None:
        gu = grad_used.double()
        if oracle is not None:
            gu = torch.where(foreground(oracle), torch.zeros_like(gu), gu)
        g = g + gu
    dot = (p * g).sum(1, keepdim=True)
    mag = p * (g.abs() + (p * g.abs()).sum(1, keepdim=True))
    return p * (g - dot), mag


def online_softmax_f32(logits: np.ndarray, skip_neg_inf: bool = True) -> np.ndarray:
    """(P, D) logits -> (P, D) float32 probabilities, in the kernels' order: one pass keeping the running max m and
    sum s (``if l > m: s *= exp(m - l); m = l``, then ``s += exp(l - m)``), then ``exp(l - m) / s``."""
    f32 = np.float32
    x = np.asarray(logits, dtype=f32)
    P, D = x.shape
    m = np.full(P, -np.inf, dtype=f32)
    s = np.zeros(P, dtype=f32)
    with np.errstate(invalid='ignore', over='ignore', under='ignore', divide='ignore'):
        for d in range(D):
            l = x[:, d]
            up = l > m
            s = np.where(up, s * np.exp(m - l), s).astype(f32)
            m = np.where(up, l, m).astype(f32)
            t = np.exp(l - m).astype(f32)
            if skip_neg_inf:
                t = np.where(l == -np.inf, f32(0), t).astype(f32)
            s = (s + t).astype(f32)
        return (np.exp(x - m[:, None]).astype(f32) / s[:, None]).astype(f32)


def forward_rel_bound(logits: torch.Tensor, D: int) -> torch.Tensor:
    """(BN, D, H, W) float64 relative error bound of the kernels' float32 probabilities against ``softmax_ref``
    (rows with a finite result; masked bins are exact zeros and get bound 0).

    Per pixel, m = max l, R = number of times the running max rises after the first finite logit, E = sum_j p_j (m - l_j).
    Each term exp(l_j - m) reaches the sum through argument roundings totalling (m - l_j) u (the gaps telescope over
    the rescales), one expf (2 ulp = 4u) and, per rescale, one more expf and one product (5u); the D additions of
    positive terms add D u.  So the sum is within (E + 4 + 5R + D) u, and the probability (one more subtraction,
    expf and division) within (|l - m| + E + 5R + D + 9) u; +1 u covers second-order terms."""
    x = logits[:, :D].float().double()
    m = x.amax(1, keepdim=True)
    p = softmax_ref(logits, D)
    gap = torch.where(x == -torch.inf, torch.zeros_like(x), m - x)
    E = torch.where(p > 0, p * gap, torch.zeros_like(p)).sum(1, keepdim=True)
    cm = torch.cummax(x, 1).values
    R = ((cm[:, 1:] > cm[:, :-1]) & (cm[:, :-1] > -torch.inf)).sum(1, keepdim=True).double()
    return (gap + E + 5 * R + D + 10) * U32


def sum_bound(n, mag):
    """Error bound of any float32 evaluation of a sum / dot product of n terms whose magnitudes sum to ``mag``:
    gamma_n = n u / (1 - n u), widened by 2^-20 (relative) for the fp64 reference's own rounding, plus n subnormal
    ulps for underflow."""
    g = n * U32 / (1 - n * U32)
    return g * (1 + 2.0 ** -20) * mag + n * FLT_TRUE_MIN


def round_bracket(ref64: torch.Tensor, err, dtype: torch.dtype):
    """(lo, hi) in ``dtype``: ``ref64 -/+ err`` rounded to float32, then to ``dtype``.  Both roundings are monotone, so
    a float32 value within ``err`` of ``ref64``, rounded once to ``dtype``, lies in [lo, hi]."""
    lo = (ref64 - err).float().to(dtype)
    hi = (ref64 + err).float().to(dtype)
    return lo, hi


def in_bracket(x: torch.Tensor, lo: torch.Tensor, hi: torch.Tensor) -> torch.Tensor:
    """Elementwise lo <= x <= hi (compared in float32; -0.0 == +0.0)."""
    x = x.float()
    return (lo.float() <= x) & (x <= hi.float())

"""CPU oracle of the BEV augmentation warp.  TEST INFRASTRUCTURE -- never imported by the product.

``bev_augment_image`` (``models/bev_depth.py:69-84`` of the reference) calls
``kornia.geometry.transform.warp_affine(src, M, dsize, mode='bilinear', padding_mode='zeros', align_corners=True)``.
Kornia is not installed here; its sequence (kornia >= 0.6, as documented) is restated with torch ops:

    M3 = [[M], [0, 0, 1]]                                             # convert_affinematrix_to_homography
    N(h, w) = [[2/(w-1), 0, -1], [0, 2/(h-1), -1], [0, 0, 1]]           # normal_transform_pixel
    dst_norm_T_src_norm = N(H', W') @ (M3 @ inverse(N(H, W)))          # normalize_homography
    theta = inverse(dst_norm_T_src_norm)[:, :2, :]
    out = F.grid_sample(src, F.affine_grid(theta, [B, C, H', W'], align_corners=True), 'bilinear', 'zeros',
                        align_corners=True)

in float32 or float64.  Parity status: pinned by restatement + known answers (tests/test_oracle_warp_affine.py:
identity, flips, integer and half-pixel shifts, a hand-worked 90 degree rotation); kornia itself is not available.
"""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F


def normal_transform_pixel(h: int, w: int, dtype=torch.float64) -> torch.Tensor:
    return torch.tensor([[2.0 / (w - 1), 0.0, -1.0], [0.0, 2.0 / (h - 1), -1.0], [0.0, 0.0, 1.0]], dtype=dtype)


def theta_ref(M: torch.Tensor, src_hw, dsize, dtype=torch.float64) -> torch.Tensor:
    """(B, 2, 3): kornia's normalised destination -> normalised source matrix, computed in ``dtype`` on the CPU."""
    m = M.detach().cpu().to(dtype)
    B = m.shape[0]
    m3 = torch.cat([m, torch.tensor([0.0, 0.0, 1.0], dtype=dtype).expand(B, 1, 3)], dim=1)
    H, W = src_hw
    dst_norm_T_src_norm = normal_transform_pixel(*dsize, dtype=dtype) @ (m3 @ torch.inverse(normal_transform_pixel(H, W, dtype)))
    return torch.linalg.inv_ex(dst_norm_T_src_norm).inverse[:, :2, :]


def warp_affine_ref(src: torch.Tensor, M: torch.Tensor, dsize, dtype=torch.float64) -> torch.Tensor:
    """kornia's warp_affine (bilinear, zeros, align_corners=True) in ``dtype`` on ``src``'s device; differentiable in
    ``src``."""
    B, C, H, W = src.shape
    theta = theta_ref(M, (H, W), dsize, dtype).to(src.device)
    grid = F.affine_grid(theta, [B, C, int(dsize[0]), int(dsize[1])], align_corners=True)
    return F.grid_sample(src.to(dtype), grid, mode='bilinear', padding_mode='zeros', align_corners=True)


def tap_sum_ref(values: torch.Tensor, M: torch.Tensor, dsize, eps: float = 1e-3) -> torch.Tensor:
    """(B, C, H', W') float64: sum of ``values`` (pass |src|) over the in-grid bilinear taps of every destination
    pixel, weights not applied -- the scale of the error a float32 coordinate puts into the output through its
    weights.  A coordinate within ``eps`` of an integer counts the taps of both sides (float32 may floor it the other
    way).  Linear and differentiable in ``values``: its adjoint at |grad| bounds the backward the same way."""
    B, C, H, W = values.shape
    dev = values.device
    theta = theta_ref(M, (H, W), dsize).to(dev)
    grid = F.affine_grid(theta, [B, C, int(dsize[0]), int(dsize[1])], align_corners=True)
    ix = (grid[..., 0] + 1) / 2 * (W - 1)
    iy = (grid[..., 1] + 1) / 2 * (H - 1)
    ok = torch.isfinite(ix) & torch.isfinite(iy)
    ix = torch.where(ok, ix, torch.full_like(ix, -10.0)).clamp(-10, W + 10)
    iy = torch.where(ok, iy, torch.full_like(iy, -10.0)).clamp(-10, H + 10)
    x0, x1 = (ix - eps).floor().long(), (ix + eps).floor().long() + 1
    y0, y1 = (iy - eps).floor().long(), (iy + eps).floor().long() + 1
    a = values.double().reshape(B, C, H * W)
    out = torch.zeros(B, C, *grid.shape[1:3], dtype=torch.float64, device=dev)
    for ty in (0, 1, 2):
        for tx in (0, 1, 2):
            x, y = x0 + tx, y0 + ty
            inside = (x >= 0) & (x < W) & (y >= 0) & (y < H) & (x <= x1) & (y <= y1)
            flat = (y.clamp(0, H - 1) * W + x.clamp(0, W - 1)).view(B, 1, -1).expand(B, C, -1)
            v = a.gather(2, flat).view_as(out)
            out = out + torch.where(inside[:, None], v, torch.zeros_like(v))
    return out


# ---------------------------------------------------------------------------------------------- test matrices
def about_centre(lin: torch.Tensor, H: int, W: int) -> torch.Tensor:
    """(B, 2, 2) linear parts -> (B, 2, 3) pixel maps that keep the grid centre in place."""
    c = torch.tensor([(W - 1) / 2, (H - 1) / 2], dtype=torch.float64)
    return torch.cat([lin, (c - lin @ c)[..., None]], -1)


def bda_matrices(B: int, H: int, W: int, seed: int = 0) -> torch.Tensor:
    """Random BDA: rotation +-22.5 deg, scale 0.95..1.05, random x / y flips, about the grid centre."""
    g = torch.Generator().manual_seed(seed)
    a = (torch.rand(B, generator=g, dtype=torch.float64) * 2 - 1) * math.pi / 8
    s = 0.95 + 0.1 * torch.rand(B, generator=g, dtype=torch.float64)
    fx = torch.where(torch.rand(B, generator=g) < 0.5, -1.0, 1.0).double()
    fy = torch.where(torch.rand(B, generator=g) < 0.5, -1.0, 1.0).double()
    rot = torch.stack([torch.stack([a.cos(), -a.sin()], -1), torch.stack([a.sin(), a.cos()], -1)], -2)
    lin = s[:, None, None] * rot @ torch.diag_embed(torch.stack([fx, fy], -1))
    return about_centre(lin, H, W).float()

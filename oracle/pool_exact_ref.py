"""Integer oracle of the fp32 pooling kernels on dyadic inputs.  TEST INFRASTRUCTURE -- never imported by the product.

The inputs are small dyadic numbers: ``depth = a 2^-4`` (a in [1, amax]), ``context = b 2^-4`` (|b| in [1, bmax]) and
``grad_out = g 2^-4`` (|g| in [0, gmax]).  Every product of two inputs is then an integer multiple of 2^-8, and so is
every partial sum of such products.  A partial sum of the terms of one output element is at most the element's sum of
term magnitudes, so when that sum is below 2^24 units every partial sum is an integer below 2^24 units: a float32
holds it exactly, in any summation order, with or without FMA, however the terms are split into runs, slices and
fix-ups.  The kernels' fp32 outputs must then equal the integer results here BIT FOR BIT; a dropped, duplicated or
misplaced term changes them, however small it is.  ``*_exact`` functions return the integer result together with
the per-element sum of term magnitudes, and ``holds`` checks that sum against 2^24 (the precondition is asserted by
the tests, never assumed).  Given float64 inputs instead, ``forward_exact`` and ``grads_exact`` compute the fp64
reference and magnitudes of general inputs (for ``depth_softmax_ref.sum_bound``).

The softmax-folded route (``voxel_pooling_fused_logits``) is exact too: logits of 0 on k in {1, 2, 4, 8} live bins
of a pixel and -inf on the others give p = expf(0) / k = 1 / k exactly, i.e. a = 16 / k in the units above.

Everything runs image by image on the device the inputs are on, grouping the points of an image by (cell, pixel)
before the channel dimension is touched: no (B, N, D, H, W, C) tensor is made, so CFG-2 at 32 frames stays cheap.
"""
from __future__ import annotations

import torch

SHIFT = 4                        # fractional bits of every input
LIMIT = 1 << 24                  # every partial sum of fewer units than this is exact in float32
_CHUNK = 1 << 18                 # (cell, pixel) keys per gathered block


def _ints(gen, shape, lo, hi, signed, device):
    v = torch.randint(lo, hi + 1, shape, generator=gen)
    if signed:
        v = torch.where(torch.rand(shape, generator=gen) < 0.5, -v, v)
    return v.to(device)


def dyadic_inputs(seed, B, N, D, H, W, C, voxel_num, amax=15, bmax=15, gmax=15, device='cpu'):
    """int64 ``a`` (B*N, D, H, W) in [1, amax], ``b`` (B*N, C, H, W) in +-[1, bmax], ``g`` (B, C, Y, X) in +-[0, gmax]."""
    X, Y, _ = voxel_num
    gen = torch.Generator().manual_seed(seed)
    a = _ints(gen, (B * N, D, H, W), 1, amax, False, device)
    b = _ints(gen, (B * N, C, H, W), 1, bmax, True, device)
    g = _ints(gen, (B, C, Y, X), 0, gmax, True, device)
    return a, b, g


def to_float(v: torch.Tensor, shift: int = SHIFT) -> torch.Tensor:
    """Integer multiple of 2^-shift -> float32 (exact for |v| < 2^24)."""
    return (v.double() * 2.0 ** -shift).float()


def masked_logits(seed, BN, D, H, W, device='cpu', ks=(1, 2, 4, 8)):
    """Logits (BN, D, H, W) float32: 0 on k live bins of every pixel (k drawn from ``ks``, k <= D), -inf elsewhere;
    and ``a`` int64 = 16 / k on the live bins, 0 elsewhere (the probabilities in units of 2^-4)."""
    gen = torch.Generator().manual_seed(seed)
    ks = torch.tensor([k for k in ks if k <= D])
    k = ks[torch.randint(0, len(ks), (BN, 1, H, W), generator=gen)]
    rank = torch.rand(BN, D, H, W, generator=gen).argsort(1).argsort(1)       # a random permutation of the bins per pixel
    live = rank < k
    logits = torch.where(live, torch.tensor(0.0), torch.tensor(float('-inf')))
    a = torch.where(live, 16 // k, torch.zeros_like(rank))
    return logits.to(device), a.to(device)


def depth_feature(logits: torch.Tensor, context: torch.Tensor, extra: int = 0, seed: int = 0) -> torch.Tensor:
    """DepthNet's output tensor: logits in channels [0, D), context in [D, D + C), then ``extra`` random channels."""
    parts = [logits, context]
    if extra:
        gen = torch.Generator().manual_seed(seed)
        BN, _, H, W = logits.shape
        parts.append(torch.randn(BN, extra, H, W, generator=gen).to(logits.device))
    return torch.cat(parts, 1).contiguous()


def frustum_geom(seed, B, N, D, H, W, voxel_num, coherent):
    """int32 geom_xyz (B, N, D, H, W, 3).  coherent: a level camera -- every row of an (image, bin, column) lands in one
    cell, with a dropped prefix of rows (z = -1) and ~3 % of the rows straying into another cell; else every point its
    own random cell, some dropped."""
    g = torch.Generator().manual_seed(seed)
    X, Y, Z = voxel_num
    if coherent:
        x = torch.randint(-1, X + 1, (B, N, D, 1, W), generator=g).expand(B, N, D, H, W)
        y = torch.randint(-1, Y + 1, (B, N, D, 1, W), generator=g).expand(B, N, D, H, W)
        z = torch.where(torch.arange(H).view(1, 1, 1, H, 1) >= torch.randint(0, H, (B, N, D, 1, W), generator=g), 0, -1)
        z = z + torch.randint(0, Z, (B, N, D, H, W), generator=g) * (z >= 0)
        stray = torch.rand(B, N, D, H, W, generator=g) < 0.03
        x = torch.where(stray, torch.randint(0, X, (B, N, D, H, W), generator=g), x)
    else:
        x = torch.randint(-2, X + 2, (B, N, D, H, W), generator=g)
        y = torch.randint(-2, Y + 2, (B, N, D, H, W), generator=g)
        z = torch.randint(-1, Z + 1, (B, N, D, H, W), generator=g)
    return torch.stack([x, y, z], -1).int().contiguous()


def cells(geom_xyz: torch.Tensor, voxel_num) -> torch.Tensor:
    """int64 (B, Np): global output row b*Y*X + y*X + x of every point, -1 where the reference drops it
    (``voxel_pooling_forward_cuda.cu:19-29``: x, y, z outside [0, num_voxel))."""
    X, Y, Z = voxel_num
    B = geom_xyz.shape[0]
    g = geom_xyz.reshape(B, -1, 3).long()
    gx, gy, gz = g[..., 0], g[..., 1], g[..., 2]
    kept = (gx >= 0) & (gx < X) & (gy >= 0) & (gy < Y) & (gz >= 0) & (gz < Z)
    lin = torch.arange(B, device=g.device).view(B, 1) * (X * Y) + gy * X + gx
    return torch.where(kept, lin, torch.full_like(lin, -1))


def _images(cell: torch.Tensor, BN: int, DHW: int, HW: int):
    """Per image: (image index, global rows and pixels of the distinct (cell, pixel) keys, key of every kept point,
    flat (d, h, w) index of every kept point)."""
    flat = cell.reshape(BN, DHW)
    for i in range(BN):
        idx = (flat[i] >= 0).nonzero().squeeze(1)
        key = flat[i, idx] * HW + idx % HW
        uk, inv = torch.unique(key, return_inverse=True)
        yield i, uk // HW, uk % HW, inv, idx


def forward_exact(cell, a, b, voxel_num):
    """Fused forward: ``out[cell, c] = sum over kept points p of the cell of a[p] * b[c, pixel(p)]``.
    Returns ``out`` (B, Y, X, C) int64 in units of 2^-8, ``mag`` (the same sum of |terms|) and ``terms``
    (B, Y, X) int64: the number of points in each cell."""
    X, Y, _ = voxel_num
    BN, D, H, W = a.shape
    C = b.shape[1]
    B = cell.shape[0]
    out = torch.zeros(B * Y * X, C, dtype=b.dtype, device=a.device)
    mag = torch.zeros_like(out)
    terms = torch.bincount(cell[cell >= 0], minlength=B * Y * X)
    for i, uc, up, inv, idx in _images(cell, BN, D * H * W, H * W):
        av = a[i].reshape(-1)[idx]
        A = torch.zeros(uc.numel(), dtype=a.dtype, device=a.device).index_add_(0, inv, av)
        Aabs = torch.zeros_like(A).index_add_(0, inv, av.abs())
        bb = b[i].reshape(C, H * W)
        for s in range(0, uc.numel(), _CHUNK):
            rows = bb[:, up[s:s + _CHUNK]].t()
            out.index_add_(0, uc[s:s + _CHUNK], rows * A[s:s + _CHUNK, None])
            mag.index_add_(0, uc[s:s + _CHUNK], rows.abs() * Aabs[s:s + _CHUNK, None])
    return out.view(B, Y, X, C), mag.view(B, Y, X, C), terms.view(B, Y, X)


def grads_exact(cell, a, b, g):
    """Fused backward in units of 2^-8: ``gd[p] = sum_c g[cell(p), c] * b[c, pixel(p)]`` (0 for dropped points) and
    ``gc[c, pixel] = sum_d a[d, pixel] * g[cell(d, pixel), c]``; each with its sum of |terms|."""
    BN, D, H, W = a.shape
    C = b.shape[1]
    rows_g = g.permute(0, 2, 3, 1).reshape(-1, C)
    gd = torch.zeros(BN, D * H * W, dtype=b.dtype, device=a.device)
    gd_mag = torch.zeros_like(gd)
    gc = torch.zeros(BN, H * W, C, dtype=b.dtype, device=a.device)
    gc_mag = torch.zeros_like(gc)
    for i, uc, up, inv, idx in _images(cell, BN, D * H * W, H * W):
        av = a[i].reshape(-1)[idx]
        A = torch.zeros(uc.numel(), dtype=a.dtype, device=a.device).index_add_(0, inv, av)
        Aabs = torch.zeros_like(A).index_add_(0, inv, av.abs())
        bb = b[i].reshape(C, H * W)
        V = torch.empty(uc.numel(), dtype=b.dtype, device=a.device)
        Vabs = torch.empty_like(V)
        for s in range(0, uc.numel(), _CHUNK):
            G = rows_g[uc[s:s + _CHUNK]]
            ctx = bb[:, up[s:s + _CHUNK]].t()
            V[s:s + _CHUNK] = (G * ctx).sum(1)
            Vabs[s:s + _CHUNK] = (G.abs() * ctx.abs()).sum(1)
            gc[i].index_add_(0, up[s:s + _CHUNK], G * A[s:s + _CHUNK, None])
            gc_mag[i].index_add_(0, up[s:s + _CHUNK], G.abs() * Aabs[s:s + _CHUNK, None])
        gd[i, idx] = V[inv]
        gd_mag[i, idx] = Vabs[inv]
    shape_c = lambda t: t.view(BN, H, W, C).permute(0, 3, 1, 2).contiguous()
    return gd.view(BN, D, H, W), gd_mag.view(BN, D, H, W), shape_c(gc), shape_c(gc_mag)


def logit_grad_exact(a, gd):
    """Gradient wrt the logits of ``softmax`` from the probabilities ``a`` (units of 2^-4, a = 16 / k) and the gradient
    wrt them ``gd`` (units of 2^-8): ``p (g - sum_j p_j g_j)`` in units of 2^-16.  The magnitude returned bounds every
    intermediate of that evaluation (the dot product in units of 2^-12, ``g - dot`` and the final product)."""
    dot = (a * gd).sum(1, keepdim=True)
    dot_abs = (a * gd.abs()).sum(1, keepdim=True)
    mag = a.clamp(min=1) * (16 * gd.abs() + dot_abs)
    return a * (16 * gd - dot), mag


def dropin_forward_exact(cell, f, voxel_num):
    """Drop-in op (``voxel_pooling``): ``out[cell] = sum of the kept rows f[p]`` (integer units); sum of |terms|."""
    X, Y, _ = voxel_num
    B, C = cell.shape[0], f.shape[-1]
    k = cell.reshape(-1) >= 0
    rows = f.reshape(-1, C)[k]
    out = torch.zeros(B * Y * X, C, dtype=torch.int64, device=f.device).index_add_(0, cell.reshape(-1)[k], rows)
    mag = torch.zeros_like(out).index_add_(0, cell.reshape(-1)[k], rows.abs())
    return out.view(B, Y, X, C), mag.view(B, Y, X, C)


def dropin_backward_exact(cell, g):
    """Drop-in backward: kept rows receive ``g[b, :, y, x]``, dropped rows 0; (B, Np, C)."""
    C = g.shape[1]
    rows = g.permute(0, 2, 3, 1).reshape(-1, C)
    c = cell.reshape(-1)
    out = torch.where((c >= 0)[:, None], rows[c.clamp(min=0)], torch.zeros((), dtype=rows.dtype, device=rows.device))
    return out.view(*cell.shape, C)


def holds(mag: torch.Tensor) -> bool:
    """Every element's sum of |terms| is below 2^24 units: its float32 evaluation is exact in any order."""
    return mag.numel() == 0 or int(mag.max()) < LIMIT

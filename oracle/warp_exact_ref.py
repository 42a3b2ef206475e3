"""Float32 emulation of the BDA warp kernels.  TEST INFRASTRUCTURE -- never imported by the product.

``csrc/bev_warp.cu`` is deterministic float32 code with no freedom left to the compiler: ``linspace_m1p1`` and the
grid coordinates use explicit ``fmaf``, the unnormalisation is an add and two multiplies, the weights are plain
products and the channel sums are ``fmaf(v, w, acc)`` in a fixed order (the SASS is FFMA / FADD / FMUL / FRND.FLOOR
in that order, no FTZ).  Every step is restated here on numpy float32 arrays, with a correctly rounded ``fmaf``, so
the kernels must equal these functions BIT FOR BIT -- a tap dropped, counted twice, given the wrong weight or summed
out of order shows up however small its weight is.

* ``warp_taps``            -- the device function: per destination pixel, the nw corner and the four weights / validity
  bits (order nw, ne, sw, se).
* ``warp_forward_exact``   -- per destination pixel and channel ``acc = fmaf(v, w, acc)`` from +0 over the valid taps
  in order; with ``cell_start`` the taps on empty cells are skipped (the kernel never reads those rows).
* ``warp_backward_exact``  -- per source cell and channel, the (destination pixel, tap) pairs whose valid tap lands on
  the cell, zero weights included, in ascending destination index.  The pairs come from the forward's taps, not from a
  search window: a pair the kernel's window misses is a mismatch.  With ``cell_start`` only occupied cells get a row.

``theta`` is always the float32 (B, 2, 3) matrix the kernels receive (``bev_augment.warp_theta`` read back, or a
hand-made one passed through the C ABI).  Rows are channels-last: (B, H, W, C).
"""
from __future__ import annotations

from typing import NamedTuple, Optional

import numpy as np

f32 = np.float32
_OVERFLOW_TIE = 2.0 ** 128 - 2.0 ** 103          # halfway between FLT_MAX and 2^128: the float32 overflow threshold


def fmaf(a, b, c) -> np.ndarray:
    """Correctly rounded float32 fused multiply-add (round to nearest even), elementwise with broadcasting.

    The product of two float32 values is exact in float64; ``s = fl64(p + c)`` plus the TwoSum error ``e`` is the
    exact sum.  Rounding ``s`` to float32 is then correct except where ``s`` sits exactly on a float32 midpoint and
    ``e != 0`` (double rounding): there the exact sum lies on ``e``'s side of the midpoint."""
    a, b, c = np.broadcast_arrays(np.asarray(a, f32), np.asarray(b, f32), np.asarray(c, f32))
    with np.errstate(all='ignore'):
        p = a.astype(np.float64) * b.astype(np.float64)
        c64 = c.astype(np.float64)
        s = p + c64
        bv = s - p
        e = (p - (s - bv)) + (c64 - bv)
        r = s.astype(f32)
        fix = np.isfinite(s) & (e != 0) & (s != r.astype(np.float64))
        if not fix.any():
            return r
        s_, e_, r_ = s[fix], e[fix], r[fix]
        out = r_.copy()
        big = np.isinf(r_)                                              # s rounded past FLT_MAX
        tie_big = big & (np.abs(s_) == _OVERFLOW_TIE)
        out[tie_big] = np.where(np.sign(e_[tie_big]) == np.sign(s_[tie_big]), r_[tie_big],
                                np.copysign(np.finfo(f32).max, s_[tie_big]).astype(f32))
        fin = ~big
        nb = np.nextafter(r_[fin], np.copysign(f32(np.inf), (s_[fin] - r_[fin].astype(np.float64))).astype(f32))
        mid = (r_[fin].astype(np.float64) + nb.astype(np.float64)) * 0.5
        tie = (mid == s_[fin]) & np.isfinite(nb)
        pick = tie & (np.sign(nb.astype(np.float64) - r_[fin].astype(np.float64)) == np.sign(e_[fin]))
        sub = out[fin]
        sub[pick] = nb[pick]
        out[fin] = sub
        r = r.copy()
        r[fix] = out
    return r


def linspace_m1p1(i, n: int) -> np.ndarray:
    """``torch.linspace(-1, 1, n)[i]`` in float32 as the kernel computes it (two-sided, one fmaf)."""
    i = np.asarray(i, dtype=np.int64)
    step = f32(2) / f32(n - 1)
    lo = fmaf(step, i.astype(f32), f32(-1))
    hi = fmaf(-step, (n - 1 - i).astype(f32), f32(1))
    return np.where(i < n // 2, lo, hi)


class Taps(NamedTuple):
    x0: np.ndarray          # (B, Hd, Wd) int64: the nw tap's column (0 where the pixel has no tap)
    y0: np.ndarray          # (B, Hd, Wd) int64
    w: np.ndarray           # (B, Hd, Wd, 4) float32, order nw, ne, sw, se
    valid: np.ndarray       # (B, Hd, Wd, 4) bool: the tap lies inside the source grid


def _theta(theta) -> np.ndarray:
    th = np.asarray(theta, dtype=f32)
    if th.dtype != f32:
        raise TypeError('theta must be float32')
    return th.reshape(-1, 6)


def warp_taps(theta, Hs: int, Ws: int, Hd: int, Wd: int) -> Taps:
    """``warp_taps`` of ``csrc/bev_warp.cu`` for every destination pixel of every sample, step by step in float32."""
    th = _theta(theta)
    t = [th[:, k, None, None] for k in range(6)]
    xn = linspace_m1p1(np.arange(Wd), Wd)[None, None, :]
    yn = linspace_m1p1(np.arange(Hd), Hd)[None, :, None]
    gx = fmaf(t[0], xn, fmaf(t[1], yn, t[2]))
    gy = fmaf(t[3], xn, fmaf(t[4], yn, t[5]))
    with np.errstate(all='ignore'):
        ix = ((gx + f32(1)) * f32(0.5)) * f32(Ws - 1)
        iy = ((gy + f32(1)) * f32(0.5)) * f32(Hs - 1)
        inside = (ix > f32(-2)) & (ix < f32(Ws) + f32(1)) & (iy > f32(-2)) & (iy < f32(Hs) + f32(1))
    ix = np.where(inside, ix, f32(0))
    iy = np.where(inside, iy, f32(0))
    fx, fy = np.floor(ix), np.floor(iy)
    x0, y0 = fx.astype(np.int64), fy.astype(np.int64)
    ex, wx = (fx + f32(1)) - ix, ix - fx
    ey, wy = (fy + f32(1)) - iy, iy - fy
    w = np.stack([ex * ey, wx * ey, ex * wy, wx * wy], -1)
    w = np.where(inside[..., None], w, f32(0))
    x0in, x1in = (x0 >= 0) & (x0 < Ws), (x0 + 1 >= 0) & (x0 + 1 < Ws)
    y0in, y1in = (y0 >= 0) & (y0 < Hs), (y0 + 1 >= 0) & (y0 + 1 < Hs)
    valid = np.stack([x0in & y0in, x1in & y0in, x0in & y1in, x1in & y1in], -1) & inside[..., None]
    return Taps(np.where(inside, x0, 0), np.where(inside, y0, 0), w, valid)


def _occupied(cell_start, B: int, cells: int) -> Optional[np.ndarray]:
    if cell_start is None:
        return None
    cs = np.asarray(cell_start, dtype=np.int64)
    if cs.shape != (B * cells + 1,):
        raise ValueError(f'cell_start must hold B*H*W + 1 = {B * cells + 1} entries, got {cs.shape}')
    return (np.diff(cs) != 0).reshape(B, cells)


def _pairs(taps: Taps, b: int, Ws: int):
    """(source cell, destination pixel, weight) of every valid tap of sample b, destination-major."""
    cells, dsts, ws = [], [], []
    nd = taps.x0[b].size
    d = np.arange(nd)
    for k in range(4):
        v = taps.valid[b, ..., k].ravel()
        cell = ((taps.y0[b] + (k >> 1)) * Ws + taps.x0[b] + (k & 1)).ravel()
        cells.append(cell[v])
        dsts.append(d[v])
        ws.append(taps.w[b, ..., k].ravel()[v])
    return np.concatenate(cells), np.concatenate(dsts), np.concatenate(ws)


def warp_forward_exact(theta, src_rows, dsize, cell_start=None) -> np.ndarray:
    """(B, Hs, Ws, C) float32 source rows -> (B, Hd, Wd, C) float32, bit for bit the forward kernel."""
    src = np.asarray(src_rows, dtype=f32)
    B, Hs, Ws, C = src.shape
    Hd, Wd = (int(v) for v in dsize)
    taps = warp_taps(theta, Hs, Ws, Hd, Wd)
    occ = _occupied(cell_start, B, Hs * Ws)
    out = np.empty((B, Hd * Wd, C), dtype=f32)
    for b in range(B):
        flat = src[b].reshape(Hs * Ws, C)
        acc = np.zeros((Hd * Wd, C), dtype=f32)
        for k in range(4):
            use = taps.valid[b, ..., k].ravel().copy()
            cell = ((taps.y0[b] + (k >> 1)) * Ws + taps.x0[b] + (k & 1)).ravel()
            if occ is not None:
                use &= occ[b, np.where(use, cell, 0)]
            i = np.nonzero(use)[0]
            acc[i] = fmaf(flat[cell[i]], taps.w[b, ..., k].ravel()[i, None], acc[i])
        out[b] = acc
    return out.reshape(B, Hd, Wd, C)


def warp_backward_exact(theta, grad_rows, src_hw, cell_start=None, out=None) -> np.ndarray:
    """(B, Hd, Wd, C) float32 gradient rows -> (B, Hs, Ws, C) float32, bit for bit the backward kernel.

    With ``cell_start`` only the rows of occupied cells are computed; the others are taken from ``out`` (zeros when
    it is not given), as the kernel leaves them untouched.  Sums run in rounds -- round r adds the r-th pair (in
    ascending destination index) of every cell that has one -- so a 64x magnification costs a few thousand small steps
    rather than a Python loop over cells."""
    g = np.asarray(grad_rows, dtype=f32)
    B, Hd, Wd, C = g.shape
    Hs, Ws = (int(v) for v in src_hw)
    taps = warp_taps(theta, Hs, Ws, Hd, Wd)
    occ = _occupied(cell_start, B, Hs * Ws)
    res = np.zeros((B, Hs * Ws, C), dtype=f32) if out is None else np.array(out, dtype=f32).reshape(B, Hs * Ws, C)
    for b in range(B):
        cell, dst, w = _pairs(taps, b, Ws)
        if occ is not None:
            keep = occ[b, cell]
            cell, dst, w = cell[keep], dst[keep], w[keep]
        order = np.lexsort((dst, cell))
        cell, dst, w = cell[order], dst[order], w[order]
        first = np.searchsorted(cell, cell, side='left')
        rank = np.arange(cell.size) - first
        by_round = np.argsort(rank, kind='stable')
        bounds = np.searchsorted(rank[by_round], np.arange(int(rank.max(initial=-1)) + 2))
        gb = g[b].reshape(Hd * Wd, C)
        acc = np.zeros((Hs * Ws, C), dtype=f32)
        for r in range(len(bounds) - 1):
            sel = by_round[bounds[r]:bounds[r + 1]]
            acc[cell[sel]] = fmaf(gb[dst[sel]], w[sel, None], acc[cell[sel]])
        rows = np.ones(Hs * Ws, dtype=bool) if occ is None else occ[b]
        res[b, rows] = acc[rows]
    return res.reshape(B, Hs, Ws, C)


def operator_matrix(theta, Hs: int, Ws: int, Hd: int, Wd: int, value: float = 1.0) -> np.ndarray:
    """(B, Hd*Wd, Hs*Ws) float32: the forward of one sample applied to ``value`` times each unit source vector, i.e.
    entry (d, s) = fmaf(value, w, +0) for the pair (d, s) and +0 where there is none.  ``value = inf`` marks the
    zero-weight pairs with NaN."""
    th = _theta(theta)
    n = Hs * Ws
    basis = np.zeros((th.shape[0], Hs, Ws, n), dtype=f32)
    basis.reshape(th.shape[0], n, n)[:, np.arange(n), np.arange(n)] = f32(value)
    return warp_forward_exact(th, basis, (Hd, Wd)).reshape(th.shape[0], Hd * Wd, n)

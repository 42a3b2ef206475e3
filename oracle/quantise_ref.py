"""float32 restatement of the two cell-quantisation rules and of the kernels' shortcuts for them.  TEST INFRASTRUCTURE
-- never imported by the product.

* ``ieee_trunc_index``: the camera path's ``((e - lo) / vs).int()`` (``lss_fpn.py:461-462``): IEEE subtract, true
  division, truncation toward zero.  A NaN, infinite or int32-overflowing quotient gives INT_MIN (what the rig kernels
  return, and what torch's CPU ``.int()`` gives on x86 -- defined here, not borrowed from torch).
* ``ieee_floor_cell``: mmcv's voxelizer rule ``floor((p - min) / vs)``, kept when 0 <= cell < n, else -1.
* ``rig_quantise_fast`` / ``point_to_cell_fast``: ``csrc/plan.cu`` and ``csrc/voxelize.cu`` take q' = t * fl(1 / vs)
  instead of the division when q' is farther than 1e-3 from every integer and below a bound; the emulations follow
  them op for op, with ``1.0f / vs`` as the host computes it and CUDA's ``fminf`` / ``fmaxf``, which drop a NaN operand
  (``np.fmin`` / ``np.fmax``).

numpy float32 arithmetic is IEEE round-to-nearest-even, one rounding per operation, like the ``__f*_rn`` intrinsics.
"""
from __future__ import annotations

import numpy as np

f32 = np.float32
INT_MIN = -(1 << 31)
_TWO31 = f32(2147483648.0)
_MARGIN = f32(1e-3)


def _trunc_or_int_min(q):
    q = np.asarray(q, dtype=f32)
    with np.errstate(invalid='ignore'):
        ok = np.abs(q) < _TWO31                           # NaN compares false
    out = np.full(q.shape, INT_MIN, np.int32)
    out[ok] = np.trunc(q[ok]).astype(np.int32)
    return out


def ieee_trunc_index(e, lo, vs):
    """int32 ``trunc(fl(fl(e - lo) / vs))``; INT_MIN for a NaN, +-inf or |quotient| >= 2^31."""
    with np.errstate(invalid='ignore', over='ignore', divide='ignore'):
        t = np.subtract(np.asarray(e, f32), np.asarray(lo, f32), dtype=f32)
        q = np.divide(t, f32(vs), dtype=f32)
    return _trunc_or_int_min(q)


def ieee_floor_cell(p, pmin, vs, n):
    """int32 ``floor(fl(fl(p - min) / vs))`` where it lies in [0, n), else -1 (NaN compares false: -1)."""
    with np.errstate(invalid='ignore', over='ignore', divide='ignore'):
        c = np.floor(np.divide(np.subtract(np.asarray(p, f32), f32(pmin), dtype=f32), f32(vs), dtype=f32))
        ok = (c >= 0) & (c < f32(n))
    out = np.full(c.shape, -1, np.int32)
    out[ok] = c[ok].astype(np.int32)
    return out


def rig_quantise_fast(t, vs, bound):
    """``rig_quantise`` of ``csrc/plan.cu`` on t = fl(e - lo): the reciprocal shortcut while
    fraction > 1e-3 and |q'| < ``bound``, else the exact rule (``ieee_trunc_index`` of t)."""
    t = np.asarray(t, f32)
    inv = np.divide(f32(1.0), f32(vs), dtype=f32)
    with np.errstate(invalid='ignore', over='ignore'):
        q = np.multiply(t, inv, dtype=f32)
        fr = np.abs(np.subtract(q, np.rint(q), dtype=f32))
        fast = (fr > _MARGIN) & (np.abs(q) < f32(bound))
    return np.where(fast, _trunc_or_int_min(np.where(fast, q, f32(0))), ieee_trunc_index(t, 0.0, vs))


def point_to_cell_fast(p, pmin, vs, n):
    """``point_to_cell_fast`` of ``csrc/voxelize.cu``: p (Np, 3) -> int32 (Np, 3) [x, y, z], every coordinate -1 when
    the point is dropped.  ONE branch for the three coordinates, taken when min(fractions) > 1e-3 and
    max(|q'|) < 4096 with NaN-dropping min / max."""
    p = np.asarray(p, f32)
    pmin, vs = np.asarray(pmin, f32), np.asarray(vs, f32)
    inv = np.divide(f32(1.0), vs, dtype=f32)
    with np.errstate(invalid='ignore', over='ignore', divide='ignore'):
        t = np.subtract(p, pmin[None, :], dtype=f32)
        q = np.multiply(t, inv[None, :], dtype=f32)
        d = np.abs(np.subtract(q, np.rint(q), dtype=f32))
        big = np.fmax(np.fmax(np.abs(q[:, 0]), np.abs(q[:, 1])), np.abs(q[:, 2]))
        fast = (np.fmin(np.fmin(d[:, 0], d[:, 1]), d[:, 2]) > _MARGIN) & (big < f32(4096))
        c = np.where(fast[:, None], np.floor(q), np.floor(np.divide(t, vs[None, :], dtype=f32)))
        ok = np.all((c >= 0) & (c < np.asarray(n, f32)[None, :]), axis=1)
    out = np.full(c.shape, -1, np.int32)
    out[ok] = c[ok].astype(np.int32)
    return out


def ieee_cells(p, pmin, vs, n):
    """mmcv's per-point rule on p (Np, 3): int32 (Np, 3) [x, y, z], every coordinate -1 when any axis drops the point."""
    p = np.asarray(p, f32)
    c = np.stack([ieee_floor_cell(p[:, j], pmin[j], vs[j], n[j]) for j in range(3)], 1)
    return np.where(np.all(c >= 0, axis=1)[:, None], c, -1).astype(np.int32)


def _step(x, k):
    """x moved by k ulp (k > 0 toward +inf, k < 0 toward -inf)."""
    x = np.asarray(x, f32)
    to = f32(np.inf) if k > 0 else f32(-np.inf)
    for _ in range(abs(k)):
        x = np.nextafter(x, to).astype(f32)
    return x


def near_boundaries(lo, vs, ks, ulps, min_near=0.5):
    """float32 e values around every cell boundary k in ``ks``: e0 = fl(lo + k vs) moved by -ulps..ulps ulp, so
    that the IEEE quotient fl(fl(e - lo) / vs) lies within a few ulp of k.  ``lo`` is a scalar or one value per k.
    Asserts that at least ``min_near`` of the quotients lie within 1e-3 of an integer (the window where the shortcuts
    hand over to the division), so a weak input set cannot pass silently.  Returns (e, lo per e, number of quotients
    within 1e-3 of an integer)."""
    ks = np.asarray(ks, np.float64)
    lo = np.broadcast_to(np.asarray(lo, f32), ks.shape)
    e0 = (lo.astype(np.float64) + ks * np.float64(f32(vs))).astype(f32)
    e = np.concatenate([_step(e0, k) for k in range(-ulps, ulps + 1)])
    lo = np.tile(lo, 2 * ulps + 1)
    with np.errstate(invalid='ignore', over='ignore'):
        q = np.divide(np.subtract(e, lo, dtype=f32), f32(vs), dtype=f32)
        near = int(np.count_nonzero(np.abs(np.subtract(q, np.rint(q), dtype=f32)) <= _MARGIN))
    assert near >= min_near * e.size, f'only {near} of {e.size} quotients lie within 1e-3 of an integer'
    return e, lo, near

"""CPU: the reciprocal shortcuts of the two cell quantisations (``csrc/plan.cu`` rig_quantise, ``csrc/voxelize.cu``
point_to_cell_fast), emulated in float32, against the IEEE rules they replace -- on quotients within a few ulp of a
cell boundary, where a shortcut that is subtly wrong truncates or floors to the neighbouring cell."""
import numpy as np
import pytest

from oracle import quantise_ref as qr

f32 = np.float32
SHIPPED_VS = [0.8, 0.2, 8.0, 0.4, 0.05]
VOXEL_SIZES = [f32(v) for v in SHIPPED_VS] + [f32(v) for v in np.random.default_rng(7).uniform(0.01, 10.0, 32)]
PER_BAND = 10_000_000             # near-boundary quotients per band and rule, over all voxel sizes and both signs
ULPS = 3
BANDS = {                          # band -> (cell boundaries k >= 0 to aim at, least share of quotients within 1e-3)
    'below-1': (lambda rng, n: rng.integers(0, 2, n), 0.9),
    '4096': (lambda rng, n: rng.integers(4096 - 512, 4096 + 512, n), 0.3),
    '16384': (lambda rng, n: rng.integers(16384 - 2048, 16384 + 2048, n), 0.1),
    '2^20': (lambda rng, n: rng.integers((1 << 20) - 4096, (1 << 20) + 4096, n), 0.1),
    '2^22': (lambda rng, n: rng.integers((1 << 22) - 10, (1 << 22) + 11, n), 0.1),
}
BIG = 1 << 24                      # grid length of the voxelizer cases: every positive quotient of the bands is in range


def _band(name, vs, rng, lo=None):
    """(e, lo) near the boundaries of band ``name`` for voxel size vs, half of them with negative quotients.  lo (a
    grid's lower corner) is random per value unless given, so that e - lo rounds differently for every target."""
    ks_of, min_near = BANDS[name]
    n = -(-PER_BAND // (len(VOXEL_SIZES) * 2 * (2 * ULPS + 1)))
    ks = np.concatenate([ks_of(rng, n), -ks_of(rng, n)])
    if lo is None:
        lo = rng.uniform(-60.0, 0.0, ks.size).astype(f32)
    e, lo, _ = qr.near_boundaries(lo, vs, ks, ULPS, min_near)
    return e, lo


@pytest.mark.parametrize('band', list(BANDS))
def test_rig_shortcut_with_the_4096_bound_equals_ieee_truncation(band):
    rng = np.random.default_rng(list(BANDS).index(band))
    total = 0
    for vs in VOXEL_SIZES:
        e, lo = _band(band, vs, rng)
        t = np.subtract(e, lo, dtype=f32)
        want = qr.ieee_trunc_index(e, lo, vs)
        got = qr.rig_quantise_fast(t, vs, 4096)
        bad = np.flatnonzero(got != want)
        assert bad.size == 0, (band, float(vs), bad.size, float(t[bad[0]]), int(got[bad[0]]), int(want[bad[0]]))
        total += e.size
    assert total >= PER_BAND


@pytest.mark.parametrize('band', list(BANDS))
def test_voxelizer_shortcut_equals_ieee_floor(band):
    rng = np.random.default_rng(100 + list(BANDS).index(band))
    n = np.array([BIG] * 3)
    total = 0
    for vs in VOXEL_SIZES:
        pmin = rng.uniform(-60.0, 0.0, 3).astype(f32)
        # every coordinate of a point near a boundary: the shortcut's ONE branch sees three close calls at once
        axes = [_band(band, vs, rng, lo=pmin[j])[0] for j in range(3)]
        p = np.stack([axes[0], np.roll(axes[1], 1), np.roll(axes[2], 2)], 1)
        vsv = np.array([vs] * 3, f32)
        got = qr.point_to_cell_fast(p, pmin, vsv, n)
        want = qr.ieee_cells(p, pmin, vsv, n)
        bad = np.flatnonzero(np.any(got != want, axis=1))
        assert bad.size == 0, (band, float(vs), bad.size, p[bad[0]].tolist(), got[bad[0]].tolist(), want[bad[0]].tolist())
        total += p.shape[0]
    assert total >= PER_BAND


def test_the_2_pow_22_rig_bound_mis_truncates():
    # Why the rig shortcut's bound is 4096 (the bound point_to_cell_fast derives) and no longer 2^22: q' = t * fl(1/vs)
    # is off by up to 3 * 2^-24 |q|, more than the 1e-3 margin from |q| = 5592 up.  vs = 0.16: q' = 16390.998 takes the
    # shortcut and truncates to 16390, the true quotient is 16391.0.
    vs, t = f32(0.16), f32(2622.559814453125)
    assert np.divide(t, vs, dtype=f32) == f32(16391.0)
    assert np.multiply(t, np.divide(f32(1), vs, dtype=f32), dtype=f32) == f32(16390.998046875)
    assert int(qr.ieee_trunc_index(t, 0.0, vs)) == 16391
    assert int(qr.rig_quantise_fast(t, vs, 1 << 22)) == 16390
    assert int(qr.rig_quantise_fast(t, vs, 4096)) == 16391


@pytest.mark.parametrize('vs', [f32(0.8), f32(0.2), f32(0.16), f32(0.3)])
def test_quotients_in_minus_one_to_zero_truncate_to_zero(vs):
    # (-1, 0) truncates to cell 0, which the camera path keeps (mmcv's floor drops it: cell -1)
    t = np.concatenate([-np.geomspace(1e-30, 0.999, 1000), [-float(np.nextafter(vs, f32(0)))]]).astype(f32)
    t = t[np.divide(t, vs, dtype=f32) > f32(-1)]
    assert t.size >= 900
    assert np.all(qr.ieee_trunc_index(t, 0.0, vs) == 0)
    assert np.all(qr.rig_quantise_fast(t, vs, 4096) == 0)
    assert np.all(qr.ieee_floor_cell(t, 0.0, vs, 16) == -1)


def test_non_finite_zero_subnormal_and_overflowing_quotients():
    vs = f32(0.2)
    sub = np.array([1e-45, -1e-45, 1e-39, -1e-39], f32)                  # subnormal t
    t = np.concatenate([[np.nan, np.inf, -np.inf, 0.0, -0.0], sub,
                        [4.4e8, -4.4e8, 4.2e8, 3.0e38]]).astype(f32)
    want = np.array([qr.INT_MIN] * 3 + [0, 0] + [0, 0, 0, 0]
                    + [qr.INT_MIN, qr.INT_MIN, int(np.trunc(np.divide(t[11], vs, dtype=f32))), qr.INT_MIN], np.int32)
    assert 2.0 ** 30 < float(want[11]) < 2.0 ** 31                         # |q| of +-4.4e8 / 0.2 is above 2^31
    for bound in (4096, 1 << 22):
        assert np.array_equal(qr.rig_quantise_fast(t, vs, bound), want)
    assert np.array_equal(qr.ieee_trunc_index(t, 0.0, vs), want)
    # the voxelizer: NaN / inf / overflow on one axis drops the point; +-0 and positive subnormals are cell 0
    n = np.array([8, 8, 8])
    vsv = np.array([vs] * 3, f32)
    p = np.zeros((t.size, 3), f32)
    p[:, 0] = t
    want_x = np.array([-1, -1, -1, 0, 0, 0, -1, 0, -1, -1, -1, -1, -1], np.int32)
    for fn in (qr.point_to_cell_fast, qr.ieee_cells):
        c = fn(p, np.zeros(3, f32), vsv, n)
        assert np.array_equal(c[:, 0], want_x)
        assert np.array_equal(c[:, 1], np.where(want_x < 0, -1, 0))
    # one NaN coordinate next to two comfortable ones: fminf / fmaxf drop the NaN, so the shortcut's branch is taken
    # with q'x = NaN -- and floor(NaN) still fails the range test
    q = np.array([[np.nan, 0.5, 0.5]], f32)
    assert np.array_equal(qr.point_to_cell_fast(q, np.zeros(3, f32), vsv, n), [[-1, -1, -1]])

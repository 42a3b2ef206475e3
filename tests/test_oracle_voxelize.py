"""CPU checks of the voxelizer / VFE / pillar-scatter oracle.  PARITY UNPINNED by the
reference (mmcv/mmdet3d absent): anchored on the hand-derived KAT (SURVEY.md A.4) and on
agreement between the serial C restatement and the vectorised numpy formulation."""
import hashlib
import json
import os

import numpy as np
import pytest

from mm_training_b200 import synthetic
from mm_training_b200.configs import CFG_3
from oracle import voxelize_ref as vz

GOLDEN = os.path.join(os.path.dirname(__file__), 'golden')
IMPLS = [vz.hard_voxelize_c, vz.hard_voxelize_numpy]


@pytest.mark.parametrize('impl', IMPLS)
def test_known_answer_appendix_a4(impl):
    kat = json.load(open(os.path.join(GOLDEN, 'voxelize_kat.json')))
    pts = np.asarray(kat['points'], np.float32)
    v, c, n = impl(pts, kat['voxel_size'], kat['point_cloud_range'], kat['max_num_points'],
                   kat['max_voxels'])
    assert c.tolist() == kat['coors'] and n.tolist() == kat['num_points']
    for vid, ids in enumerate(kat['voxel_point_ids']):
        for slot, pid in enumerate(ids):
            exp = pts[pid] if pid >= 0 else np.zeros(3, np.float32)
            assert np.array_equal(v[vid, slot], exp)
    _, _, cb = vz.voxelize_batch_ref([pts], kat['voxel_size'], kat['point_cloud_range'],
                                     kat['max_num_points'], kat['max_voxels'], impl=impl)
    assert cb.tolist() == kat['coors_batch0']


def test_config3_sweep_matches_digest_and_numpy():
    d = json.load(open(os.path.join(GOLDEN, 'voxelize_sweep_digest.json')))
    pts = synthetic.lidar_sweep(CFG_3.points_per_sweep, 5, seed=2)
    assert hashlib.sha256(pts.tobytes()).hexdigest() == d['points_sha256']
    a = vz.hard_voxelize_c(pts, CFG_3.voxel_size, CFG_3.point_cloud_range, CFG_3.max_num_points,
                           CFG_3.max_voxels)
    b = vz.hard_voxelize_numpy(pts, CFG_3.voxel_size, CFG_3.point_cloud_range, CFG_3.max_num_points,
                               CFG_3.max_voxels)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
    v, c, n = a
    assert v.shape[0] == d['num_voxels'] == CFG_3.max_voxels          # the cap binds (SURVEY 8d)
    assert int(n.sum()) == d['stored_points'] and int(n.max()) == d['max_points']
    assert hashlib.sha256(c.tobytes()).hexdigest() == d['coors_sha256']
    assert hashlib.sha256(n.tobytes()).hexdigest() == d['num_sha256']
    assert hashlib.sha256(v.tobytes()).hexdigest() == d['voxels_sha256']


@pytest.mark.parametrize('seed', range(6))
def test_c_and_numpy_agree_on_random_small(seed):
    rng = np.random.default_rng(seed)
    n = int(rng.integers(0, 400))
    f = int(rng.integers(3, 9))
    pts = rng.uniform(-1.5, 5.5, size=(n, f)).astype(np.float32)
    if n > 10:                                   # duplicates and on-boundary points
        pts[5] = pts[2]
        pts[7, :3] = [0.0, 0.0, 0.0]
        pts[8, :3] = [4.0, 1.0, 0.5]
    args = ([0.5, 0.25, 1.0], [0, 0, 0, 4, 4, 2], int(rng.integers(1, 5)), int(rng.integers(1, 40)))
    a, b = vz.hard_voxelize_c(pts, *args), vz.hard_voxelize_numpy(pts, *args)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)


@pytest.mark.parametrize('impl', IMPLS)
def test_edge_cases(impl):
    rngargs = ([1, 1, 1], [0, 0, 0, 4, 4, 1])
    # empty input
    v, c, n = impl(np.zeros((0, 4), np.float32), *rngargs, 3, 5)
    assert v.shape == (0, 3, 4) and c.shape == (0, 3) and n.shape == (0,)
    # all points in one voxel: first max_points kept in order
    pts = np.tile(np.array([[0.5, 0.5, 0.5, 0]], np.float32), (50, 1))
    pts[:, 3] = np.arange(50)
    v, c, n = impl(pts, *rngargs, 4, 5)
    assert n.tolist() == [4] and v[0, :, 3].tolist() == [0, 1, 2, 3]
    # exactly max_voxels + 1 distinct voxels: last one dropped
    pts = np.array([[x + 0.5, y + 0.5, 0.5] for y in range(2) for x in range(3)], np.float32)
    v, c, n = impl(pts, *rngargs, 2, 5)
    assert v.shape[0] == 5 and c[-1].tolist() == [0, 1, 1]
    # bounds: min is inside, max is outside (floor semantics); negative epsilon is outside
    pts = np.array([[0, 0, 0], [4, 0, 0], [-1e-6, 0, 0], [3.9999, 3.9999, 0.9999]], np.float32)
    v, c, n = impl(pts, *rngargs, 2, 5)
    assert c.tolist() == [[0, 0, 0], [0, 3, 3]]


def test_vfe_and_pillar_scatter_oracle():
    rng = np.random.default_rng(0)
    pts = synthetic.lidar_sweep(5000, 8, seed=5)
    vox, num, coors = vz.voxelize_batch_ref([pts, pts[::-1].copy()], CFG_3.voxel_size,
                                            CFG_3.point_cloud_range, 15, 25000)
    feats = vz.hard_simple_vfe_ref(vox, num, 5)
    assert feats.shape == (vox.shape[0], 5)
    m = 17
    manual = vox[m, :num[m], :5].sum(0) / num[m]
    assert np.allclose(feats[m], manual, rtol=1e-6)
    canvas = vz.pillar_scatter_ref(feats, coors, 2, (1, 256, 2048))
    assert canvas.shape == (2, 5, 256, 2048)
    b, z, y, x = coors[m]
    assert np.array_equal(canvas[b, :, y, x], feats[m])
    assert int((np.abs(canvas).sum(1) > 0).sum()) <= vox.shape[0]
    g = rng.random(canvas.shape).astype(np.float32)
    gb = vz.pillar_scatter_backward_ref(g, coors, (1, 256, 2048))
    assert np.array_equal(gb[m], g[b, :, y, x])


def test_reciprocal_cell_index_rule_equals_the_exact_division():
    """csrc/voxelize.cu::point_to_cell_fast in numpy float32: q' = (p - min) * fl(1 / v) decides floor(fl((p - min) / v))
    whenever q' is farther than 1e-3 from every integer and |q'| < 4096; otherwise the exact expression is used.  Checked
    on random coordinates, on coordinates placed within a few ulps of every cell boundary, and for awkward voxel sizes."""
    rng = np.random.default_rng(0)
    for v in (0.2, 0.1, 0.05, 0.075, 0.8, 1.0 / 3.0, 0.16, 2.5):
        v32 = np.float32(v)
        inv = np.float32(1.0) / v32
        lo = np.float32(-204.8 if v < 1 else -37.3)
        cells = np.arange(0, 4096, dtype=np.float64)
        edges = (np.float64(lo) + cells * np.float64(v32)).astype(np.float32)
        near = np.concatenate([np.nextafter(edges, np.float32(np.inf)), np.nextafter(edges, np.float32(-np.inf)), edges])
        for k in range(1, 6):                                        # a few more ulps around every boundary
            up = near.copy()
            for _ in range(k):
                up = np.nextafter(up, np.float32(np.inf))
            near = np.concatenate([near, up])
        p = np.concatenate([near, rng.uniform(float(lo) - 5, float(lo) + 4096 * v + 5, 2_000_000).astype(np.float32)])
        t = (p - lo).astype(np.float32)
        exact = np.floor((t / v32).astype(np.float32))
        q = (t * inv).astype(np.float32)
        fast_ok = (np.abs(q - np.rint(q)) > np.float32(1e-3)) & (np.abs(q) < np.float32(4096.0))
        assert np.array_equal(np.floor(q)[fast_ok], exact[fast_ok]), v
        ordinary = np.arange(p.size) >= near.size                    # the uniformly drawn coordinates
        ordinary &= (q > 0) & (q < 4000)
        assert fast_ok[ordinary].mean() > 0.99                       # (the exact path is the rare one on ordinary data)


# ---- the VFE mean as the kernels compute it (oracle.voxelize_ref.vfe_mean_exact) -------------------------------------
def _rows(rows, width=None):
    """(M, T, 1) voxels and counts from ragged rows of a single feature column."""
    t = width or max(len(r) for r in rows)
    v = np.zeros((len(rows), t, 1), np.float32)
    for i, r in enumerate(rows):
        v[i, :len(r), 0] = r
    return v, np.array([len(r) for r in rows], np.int32)


def test_vfe_mean_exact_sums_in_slot_order():
    two24 = np.float32(2 ** 24)
    v, n = _rows([[2 ** 24, 1, 1], [1e8, 3, -1e8], [1, 1, 2 ** 24]])
    m = vz.vfe_mean_exact(v, n, 1)[:, 0]
    # 2^24 + 1 rounds back to 2^24 (ties to even) twice: fl(2^24 / 3), not fl((2^24 + 2) / 3)
    assert m[0] == two24 / np.float32(3) and m[0] != np.float32(2 ** 24 + 2) / np.float32(3)
    # 1e8 + 3 rounds to 1e8 (ulp 8), the -1e8 cancels it: +0, where the exact mean is 1
    assert m[1] == 0.0 and not np.signbit(m[1])
    # the other order keeps both ones: 2 + 2^24 is exact
    assert m[2] == np.float32(2 ** 24 + 2) / np.float32(3)


def test_vfe_mean_exact_signed_zero_and_non_finite():
    nan, inf = np.float32(np.nan), np.float32(np.inf)
    v, n = _rows([[-0.0], [-0.0, -0.0], [1.0, nan, 2.0], [inf, 1.0], [-inf, 5.0], [inf, -inf], [3e38, 3e38]], width=4)
    v[:, 2:, 0] = -0.0                                     # (slots beyond the count must not be added)
    m = vz.vfe_mean_exact(v, n, 1)[:, 0]
    assert m[0] == 0.0 and not np.signbit(m[0])           # +0 + -0 = +0, and +0 / 1 = +0
    assert m[1] == 0.0 and not np.signbit(m[1])
    assert np.isnan(m[2]) and m[3] == inf and m[4] == -inf and np.isnan(m[5])
    assert m[6] == inf                                    # the float32 sum overflows before the division
    # a padding row (count 0) is +0, not 0 / 0
    z = vz.vfe_mean_exact(np.zeros((2, 3, 2), np.float32), np.zeros(2, np.int32), 2)
    assert np.array_equal(z.view(np.int32), np.zeros((2, 2), np.int32))


@pytest.mark.parametrize('T', [1, 3, 15, 35])
def test_vfe_mean_exact_error_bound(T):
    # sequential float32 summation then one rounding of the division: |m - mean| <= gamma_cnt * sum|v| / cnt
    rng = np.random.default_rng(T)
    M, nf = 4000, 5
    v = (rng.standard_normal((M, T, nf)) * 10.0 ** rng.integers(-3, 6, (M, T, 1))).astype(np.float32)
    n = rng.integers(1, T + 1, M).astype(np.int32)
    m = vz.vfe_mean_exact(v, n, nf).astype(np.float64)
    live = (np.arange(T)[None, :] < n[:, None])[:, :, None]
    v64 = np.where(live, v.astype(np.float64), 0.0)
    exact = v64.sum(1) / n[:, None]
    u = 2.0 ** -24
    gamma = (n * u / (1 - n * u))[:, None]
    assert np.all(np.abs(m - exact) <= gamma * np.abs(v64).sum(1) / n[:, None])


def test_vfe_mean_exact_differs_from_numpy_pairwise_sum():
    # numpy's float32 sum of a contiguous row runs eight partial sums: on this row it keeps the ones the serial sum loses,
    # so a test comparing against it could not tell the kernels' summation order from another one
    row = np.concatenate([[2 ** 24], np.ones(15)]).astype(np.float32)
    v, n = _rows([row])
    serial = vz.vfe_mean_exact(v, n, 1)[0, 0]
    pairwise = np.float32(np.sum(row, dtype=np.float32)) / np.float32(16)
    assert serial == np.float32(2 ** 24) / np.float32(16) and serial != pairwise


def test_canvas_exact_places_the_exact_mean():
    pts = synthetic.lidar_sweep(3000, 5, seed=6)
    vox, num, coors = vz.voxelize_batch_ref([pts, pts[::-1].copy()], CFG_3.voxel_size, CFG_3.point_cloud_range, 15, 2000)
    canvas = vz.canvas_exact(vox, num, coors, 4, 2, (1, 256, 2048))
    mean = vz.vfe_mean_exact(vox, num, 4)
    assert canvas.shape == (2, 4, 256, 2048)
    got = canvas[coors[:, 0], :, coors[:, 2], coors[:, 3]]
    assert np.array_equal(got.view(np.int32), mean.view(np.int32))
    assert int((canvas != 0).any(1).sum()) <= vox.shape[0]


def test_c_and_numpy_agree_beyond_2_to_the_31_cells():
    # 65536 x 32769 x 1 = 2^31 + 2^16 cells: cell ids past 2^31 must not wrap in either oracle
    vs, rg = [1.0, 1.0, 1.0], [0, 0, 0, 65536, 32769, 1]
    assert int(np.prod(vz.grid_size_ref(vs, rg))) > 2 ** 31
    rng = np.random.default_rng(7)
    n = 3000
    x = np.concatenate([rng.integers(0, 65536, n), [65535, 0, 65535, 3]])
    y = np.concatenate([rng.choice([0, 1, 32767, 32768], n), [32768, 32768, 0, 32768]])
    pts = np.stack([x + 0.5, y + 0.25, np.full(x.size, 0.5), np.arange(x.size)], 1).astype(np.float32)
    pts = np.concatenate([pts, pts[:50]])                   # revisits: slots beyond the first
    a = vz.hard_voxelize_c(pts, vs, rg, 3, 10 ** 6)
    b = vz.hard_voxelize_numpy(pts, vs, rg, 3, 10 ** 6)
    for p, q in zip(a, b):
        assert np.array_equal(p, q)
    cells = np.unique(y.astype(np.int64) * 65536 + x)
    assert a[0].shape[0] == cells.size and cells.max() >= 2 ** 31
    assert [0, 32768, 65535] in a[1].tolist()              # (z, y, x) of cell 2^31 + 65535

"""GPU: the cell quantisation of the rig plan (``csrc/plan.cu``) and of the voxelizer (``csrc/voxelize.cu``) at voxel
boundaries, on wide grids and on non-finite geometry, against the IEEE rules of ``oracle/quantise_ref.py``.

The rig kernels evaluate e = combine @ (x d, y d, d, 1) in one of six accumulation orders.  Rows with a single unit
entry on x d or y d plus a constant, and power-of-two depths, make e = fl(f d + c) in every order, so e -- and hence
the exact cell index -- is known on the CPU without knowing the order."""
import numpy as np
import pytest
import torch

from mm_training_b200 import _lib, synthetic
from mm_training_b200.configs import CFG_2, CFG_3
from mm_training_b200.ops.voxel_pooling import (LiftSplatGeometry, PoolingPlan, rig_variant, voxel_pooling_fused,
                                                voxel_pooling_rig)
from mm_training_b200.ops.voxelize import dynamic_voxelize, hard_voxelize_batch
from oracle import pool_exact_ref as px
from oracle import quantise_ref as qr
from oracle import voxelize_ref as vz

pytestmark = pytest.mark.gpu
DEV = 'cuda'
f32 = np.float32
INT_MIN = qr.INT_MIN
OLD_BOUND = 1 << 22               # the shortcut's bound before it was derived (mis-truncates from |q| ~ 16384 up)


def _variant():
    v = rig_variant(DEV)
    if v is None:
        pytest.skip('no proven variant on this device')
    return v


def _near(lo, vs, ks, n_rest, seed):
    """float32 e values within 3 ulp of the boundaries ks: every one the 2^22-bound shortcut mis-truncates, plus
    ``n_rest`` others, in random order."""
    e, _, _ = qr.near_boundaries(lo, vs, ks, 3, min_near=0.05)
    t = np.subtract(e, f32(lo), dtype=f32)
    wrong = qr.rig_quantise_fast(t, vs, OLD_BOUND) != qr.ieee_trunc_index(e, lo, vs)
    rng = np.random.default_rng(seed)
    rest = rng.choice(np.flatnonzero(~wrong), min(n_rest, int((~wrong).sum())), replace=False)
    pick = np.concatenate([np.flatnonzero(wrong), rest])
    return e[rng.permutation(pick)], int(wrong.sum())


def _band_ks(rng, n, wide=4):
    """cell boundaries of every band of the CPU tests, both signs: below 1, 4096, 16384, 2^20, 2^22 +- 10.  The two
    bands where the 2^22 bound mis-truncates (about one near-boundary quotient in 10^3) get ``wide`` times more."""
    ks = [rng.integers(0, 2, n), rng.integers(4096 - 64, 4096 + 64, n), rng.integers(16384 - 512, 16384 + 512, wide * n),
          rng.integers((1 << 20) - 512, (1 << 20) + 512, wide * n), rng.integers((1 << 22) - 10, (1 << 22) + 11, n)]
    ks = np.concatenate(ks)
    return np.concatenate([ks, -ks])


def _lsg(vs, lo, D, H, W, Xn=64, Yn=8, Zn=4, vs_yz=None):
    """LiftSplatGeometry with a D x H x W frustum (d bound (1, D + 1, 1), final_dim (H, W), downsample 1)."""
    vs = float(vs)
    vy, vz = vs_yz if vs_yz is not None else (vs, vs)
    return LiftSplatGeometry((lo[0], lo[0] + Xn * vs, vs), (lo[1], lo[1] + Yn * vy, vy), (lo[2], lo[2] + Zn * vz, vz),
                             (1.0, D + 1.0, 1.0), (H, W), 1, DEV)


def _set_axes(lsg, fx, fy, fd):
    for name, v, n in (('fx', fx, lsg.W), ('fy', fy, lsg.H), ('fd', fd, lsg.D)):
        v = np.asarray(v, f32)
        assert v.shape == (n,), (name, v.shape, n)
        setattr(lsg, name, torch.from_numpy(v).to(DEV).contiguous())


# rows of combine: ('x', c) -> [1, 0, 0, c], ('y', c) -> [0, 1, 0, c], ('c', c) -> [0, 0, 0, c]
def _combine(rows):
    """(B, N, 4, 4) float32 from rows[b][n] = three (axis, constant) pairs."""
    unit = {'x': [1.0, 0.0, 0.0], 'y': [0.0, 1.0, 0.0], 'c': [0.0, 0.0, 0.0]}
    m = np.zeros((len(rows), len(rows[0]), 4, 4), f32)
    for b, img in enumerate(rows):
        for n, r in enumerate(img):
            for j, (ax, c) in enumerate(r):
                m[b, n, j, :3] = unit[ax]
                m[b, n, j, 3] = c
            m[b, n, 3, 3] = 1.0
    return m


def _e(rows, fx, fy, fd):
    """float32 (B, N, D, H, W, 3): e = fl(f d + c) of every point, f = the column's x, the row's y or 0."""
    fx, fy, fd = (np.asarray(v, f32) for v in (fx, fy, fd))
    D, H, W = fd.size, fy.size, fx.size
    B, N = len(rows), len(rows[0])
    px_ = np.multiply(fx[None, None, :], fd[:, None, None], dtype=f32)
    py_ = np.multiply(fy[None, :, None], fd[:, None, None], dtype=f32)
    e = np.zeros((B, N, D, H, W, 3), f32)
    for b, img in enumerate(rows):
        for n, r in enumerate(img):
            for j, (ax, c) in enumerate(r):
                f = {'x': px_, 'y': py_, 'c': np.zeros((1, 1, 1), f32)}[ax]
                e[b, n, ..., j] = np.broadcast_to(np.add(f, f32(c), dtype=f32), (D, H, W))
    return e


def _ieee_geom(lsg, e):
    lo, vs = lsg.lower.cpu().numpy(), lsg.voxel_size.cpu().numpy()
    return np.stack([qr.ieee_trunc_index(e[..., j], lo[j], vs[j]) for j in range(3)], -1)


# ---------------------------------------------------------------- rig indices, every accumulation order
# voxel size -> whether the 2^22-bound shortcut mis-truncates some of this case's near-boundary values.  Whether it
# does depends on how fl(1 / vs) rounds: for the shipped sizes it happens not to, on these inputs.
RIG_VS = {f32(0.16): True, f32(0.32): True, f32(0.02): True, f32(0.137): True,
          f32(0.2): False, f32(0.8): False, f32(0.05): False, f32(0.3): False, f32(8.0): False, f32(1.9): False}


@pytest.mark.parametrize('vs', list(RIG_VS))
def test_rig_indices_equal_ieee_truncation_in_every_variant(vs):
    rng = np.random.default_rng(int(vs * 1000))
    lo0 = float(f32(rng.uniform(-60.0, 0.0)))
    D, H = 4, 20                                                           # H % 16 != 0: a ragged row block
    lsg0 = _lsg(vs, (lo0,) * 3, 1, 1, 1)
    lo = float(lsg0.lower[0])                                              # voxel_coord - vs / 2, as the reference makes it
    fx, n_wrong = _near(lo, vs, _band_ks(rng, 64, wide=128), 2000, 1)
    fy, _ = _near(lo, vs, _band_ks(rng, 2), H, 2)
    fy = fy[:H]
    W = fx.size
    lsg = _lsg(vs, (lo0,) * 3, D, H, W)
    fd = np.array([1.0, 1.0, 0.5, 2.0], f32)
    _set_axes(lsg, fx, fy, fd)
    cz = [float(v) for v in _near(lo, vs, _band_ks(rng, 1), 4, 3)[0][:4]]
    rows = [[[('x', 0.0), ('y', 0.0), ('x', 0.0)], [('y', 0.0), ('x', 0.0), ('c', cz[0])],
             [('c', cz[1]), ('c', cz[2]), ('y', 0.0)], [('x', cz[3]), ('c', 0.0), ('c', -cz[3])]]]
    want = torch.from_numpy(_ieee_geom(lsg, _e(rows, fx, fy, fd)))
    assert (n_wrong > 0) == RIG_VS[vs], (float(vs), n_wrong)
    combine = torch.from_numpy(_combine(rows)).to(DEV)
    for v in range(_lib.lib().bevpool_rig_num_variants()):
        got = lsg.rig_geom(combine, v).cpu()
        bad = (got != want).nonzero()
        assert bad.shape[0] == 0, (float(vs), v, bad.shape[0], bad[0].tolist(), int(got[tuple(bad[0])]),
                                   int(want[tuple(bad[0])]))


# ---------------------------------------------------------------- rig plans on a grid wider than 16384 cells
WIDE_VS = f32(0.16)


def _wide_case(level):
    """A plan on X = 20000 cells of 0.16 m, Y = 4, Z = 4, with near-boundary x quotients from 8192 to 20000.
    level: x from the column, y constant, z from the row (the level-camera path); else x from the row (the walk)."""
    rng = np.random.default_rng(5 if level else 6)
    D = 3
    fd = np.array([1.0, 1.0, 0.5], f32)
    probe = _lsg(WIDE_VS, (0.0, 0.0, -2.0), 1, 1, 1, Xn=20000, Yn=4, Zn=4, vs_yz=(0.5, 1.0))
    lo = float(probe.lower[0])
    xs, n_wrong = _near(lo, WIDE_VS, rng.integers(16384, 20000, 4000), 600, 4)
    if level:
        H, W = 20, xs.size
        fx, fy = xs, np.arange(H, dtype=f32) * f32(0.25)                  # sorted rows: z rises with the row
        rows = [[[('x', 0.0), ('c', 0.7), ('y', -3.0)], [('x', 0.0), ('c', 1.2), ('y', -2.5)]],
                [[('x', 0.0), ('c', 0.2), ('y', -2.0)], [('x', 0.0), ('c', 1.9), ('y', -3.5)]]]
    else:
        H, W = xs.size, 8
        fx, fy = np.arange(W, dtype=f32) * f32(0.5), xs
        rows = [[[('y', 0.0), ('c', 0.7), ('x', -2.0)], [('y', 0.0), ('c', 1.2), ('x', -1.5)]],
                [[('y', 0.0), ('c', 0.2), ('x', 0.0)], [('y', 0.0), ('c', 1.9), ('x', -1.0)]]]
    lsg = _lsg(WIDE_VS, (0.0, 0.0, -2.0), D, H, W, Xn=20000, Yn=4, Zn=4, vs_yz=(0.5, 1.0))
    assert lsg.voxel_num == (20000, 4, 4)
    _set_axes(lsg, fx, fy, fd)
    e = _e(rows, fx, fy, fd)
    geom = _ieee_geom(lsg, e)
    assert n_wrong > 0
    return lsg, rows, e, geom


def _pairs_take_fast_path(geom, e):
    """Per (image, bin, 16-row block, column): does the level-camera test hold (x and y index equal at the block's first
    and last row, finite end points)?  fy is sorted in both cases."""
    B, N, D, H, W, _ = geom.shape
    out = []
    for hb in range(0, H, 16):
        a, b = geom[:, :, :, hb], geom[:, :, :, min(hb + 15, H - 1)]
        fin = np.isfinite(e[:, :, :, hb]).all(-1) & np.isfinite(e[:, :, :, min(hb + 15, H - 1)]).all(-1)
        out.append((a[..., 0] == b[..., 0]) & (a[..., 1] == b[..., 1]) & fin)
    return np.stack(out, 3)


@pytest.mark.parametrize('level', [True, False], ids=['level-camera-path', 'row-walk'])
def test_wide_grid_rig_plan_equals_ieee_plan(level):
    v = _variant()
    lsg, rows, e, geom = _wide_case(level)
    fast = _pairs_take_fast_path(geom, e)
    # by construction: every pair (so every warp) takes the level-camera path, or none does
    assert fast.all() if level else not fast.any()
    if level:
        kept_x = (geom[..., 0] >= 16384) & (geom[..., 0] < 20000)
        assert kept_x.any() and ((geom[..., 2] >= 0) & (geom[..., 2] < 4)).any() and (geom[..., 2] < 0).any()
    B, N = len(rows), len(rows[0])
    D, H, W = lsg.D, lsg.H, lsg.W
    combine = torch.from_numpy(_combine(rows)).to(DEV)
    ref = PoolingPlan(torch.from_numpy(geom).to(DEV).contiguous(), lsg.voxel_num, frustum=(N, D, H, W))
    plan = PoolingPlan.from_rig(lsg, combine, v)
    assert plan.mode == ref.mode == 'runs'
    assert plan.status() == 0
    for name in ('cell_of_point', 'run_code', 'cell_start', 'sorted_ids', 'sorted_cells'):
        a, b = getattr(plan, name), getattr(ref, name)
        bad = (a != b).nonzero() if a.shape == b.shape else None
        assert a.shape == b.shape and bad.shape[0] == 0, (name, a.shape, b.shape, None if bad is None else bad.shape[0])
    assert int((plan.cell_of_point >= 0).sum()) > 1000
    # pooling on dyadic inputs against the integer oracle
    vn = lsg.voxel_num
    C = 32
    cell = px.cells(torch.from_numpy(geom).to(DEV), vn)
    a, b, _ = px.dyadic_inputs(7, B, N, D, H, W, C, vn, 15, 15, 0, device=DEV)
    want, mag, _ = px.forward_exact(cell, a, b, vn)
    assert px.holds(mag)
    out = voxel_pooling_fused(None, px.to_float(a), px.to_float(b), vn, plan)
    assert torch.equal(out.permute(0, 2, 3, 1), px.to_float(want, 8))


# ---------------------------------------------------------------- non-finite geometry
BAD = (1, 2)                                       # (sample, camera) of the bad image


def _rig(kind, B):
    cfg = CFG_2
    if kind == 'level':
        gen = torch.Generator().manual_seed(3)
        s2e = torch.stack([torch.stack([synthetic.cam2ego(y + float(torch.rand(1, generator=gen)) * 10 - 5)
                                        for y in cfg.cam_yaws_deg]) for _ in range(B)])
        k = torch.eye(4)
        k[0, 0] = k[1, 1] = cfg.focal_px
        k[0, 2], k[1, 2] = cfg.final_dim[1] / 2, cfg.final_dim[0] / 2
        intrin = k[None, None].repeat(B, cfg.num_cams, 1, 1)
    else:
        from mm_training_b200.ops.voxel_pooling.rig import _random_rigs
        s2e, intrin = _random_rigs(B, cfg.num_cams, torch.Generator().manual_seed(9))
    return s2e.to(DEV), intrin.to(DEV)


def _corrupt(case, s2e, intrin):
    s2e, intrin = s2e.clone(), intrin.clone()
    b, n = BAD
    if case == 'nan-row':
        s2e[b, n, 1, :] = float('nan')
    elif case == 'inf-translation':
        s2e[b, n, 0, 3] = float('inf')
        s2e[b, n, 2, 3] = float('-inf')
    elif case == 'singular-intrinsic':
        intrin[b, n, 1, :] = 0.0
    return s2e, intrin


@pytest.mark.parametrize('case', ['nan-row', 'inf-translation', 'singular-intrinsic', 'all-nan-combine'])
@pytest.mark.parametrize('kind', ['level', 'tilted'])
def test_non_finite_geometry_drops_the_image(kind, case):
    v = _variant()
    cfg, B = CFG_2, 2
    lsg = LiftSplatGeometry.from_config(cfg, DEV)
    s2e, intrin = _rig(kind, B)
    N = cfg.num_cams
    b, n = BAD
    bad_s2e, bad_k = _corrupt(case, s2e, intrin)
    combine = lsg.combine(bad_s2e, bad_k)
    if case == 'all-nan-combine':
        combine[b, n] = float('nan')
    assert not bool(torch.isfinite(combine[b, n]).all())
    assert bool(torch.isfinite(combine[1 - b]).all()) and bool(torch.isfinite(combine[b, :n]).all())
    # rig_geom: INT_MIN in every coordinate whose combine row has a non-finite entry (then e is non-finite at every
    # point), the reference's indices everywhere else
    geom = lsg.geom_xyz(s2e, intrin)                   # the good rig through the reference's ops
    got = lsg.rig_geom(combine, v)
    rows_bad = ~torch.isfinite(combine[b, n, :3]).all(1)
    assert bool(rows_bad.any())
    for j in range(3):
        if rows_bad[j]:
            assert bool((got[b, n, ..., j] == INT_MIN).all()), j
    keep = torch.ones(B, N, dtype=torch.bool)
    keep[b, n] = False
    assert torch.equal(got[keep.to(DEV)], geom[keep.to(DEV)])
    # the plan: the bad image dropped, every other entry as in a plan built without it
    geom_wo = geom.clone()
    geom_wo[b, n] = -1
    ref = PoolingPlan(geom_wo, lsg.voxel_num, frustum=(N, lsg.D, lsg.H, lsg.W))
    plan = PoolingPlan.from_rig(lsg, combine, v) if case == 'all-nan-combine' else lsg.plan(bad_s2e, bad_k)
    assert plan.mode == 'runs' and plan.status() == 0
    Np1 = lsg.D * lsg.H * lsg.W
    sl = slice(n * Np1, (n + 1) * Np1)
    assert bool((plan.cell_of_point[b, sl] == -1).all()) and bool((plan.run_code[b, sl] == -1).all())
    for name in ('cell_of_point', 'run_code', 'cell_start', 'sorted_ids', 'sorted_cells'):
        assert torch.equal(getattr(plan, name), getattr(ref, name)), name
    # pooling: equal to the pooling without the bad image's points; zero depth gradient for the bad image
    depth, ctx, go = synthetic.camera_features(cfg, B, device=DEV)
    d, c = depth.clone().requires_grad_(True), ctx.clone().requires_grad_(True)
    if case == 'all-nan-combine':
        out = voxel_pooling_fused(None, d, c, lsg.voxel_num, plan)
    else:
        out = voxel_pooling_rig(lsg, bad_s2e, bad_k, d, c)
    want = voxel_pooling_fused(None, depth, ctx, lsg.voxel_num, ref)
    assert torch.equal(out, want)
    out.backward(go)
    gd = d.grad.view(B, N, *d.grad.shape[1:])
    assert bool((gd[b, n] == 0).all())
    assert bool((gd[1 - b] != 0).any())
    assert plan.status() == 0


# ---------------------------------------------------------------- voxelizer at voxel boundaries
VOX_GRIDS = {
    'cfg3': (CFG_3.voxel_size, CFG_3.point_cloud_range),
    'non-dyadic': ((0.3, 0.15, 0.075), (0.0, -15.0, 0.0, 60.0, 15.0, 6.0)),
    'gx-8192': ((0.05, 0.05, 8.0), (-204.8, -25.6, -5.0, 204.8, 25.6, 3.0)),
}


def _boundary_cloud(vs, pcr, seed):
    """(Np, 4) float32: points at -4..4 ulp of every x / y / z boundary and of the range ends (the other coordinates
    random in range), points near boundaries on all three axes, -0.0 and subnormal offsets from the lower corner where
    it is 0, and one NaN coordinate next to finite ones.  Column 3 is the point index."""
    rng = np.random.default_rng(seed)
    vs, pcr = np.asarray(vs, f32), np.asarray(pcr, f32)
    grid = vz.grid_size_ref(vs, pcr)
    near = []
    for j in range(3):
        b0 = (np.float64(pcr[j]) + np.arange(grid[j] + 1) * np.float64(vs[j])).astype(f32)
        b0 = np.concatenate([b0, pcr[[j, j + 3]]])
        near.append(np.concatenate([qr._step(b0, k) for k in range(-4, 5) if k]))
    pts = []
    for j in range(3):
        p = rng.uniform(pcr[:3], pcr[3:], (near[j].size, 3)).astype(f32)
        p[:, j] = near[j]
        pts.append(p)
    m = max(a.size for a in near)
    pts.append(np.stack([rng.choice(near[j], m) for j in range(3)], 1))
    special = []
    for j in range(3):
        if pcr[j] == 0:
            for val in (-0.0, 0.0, 1e-45, -1e-45, 1e-40, -1e-40, 1.2e-38, -1.2e-38):
                p = rng.uniform(pcr[:3], pcr[3:], 3).astype(f32)
                p[j] = val
                special.append(p)
        p = rng.uniform(pcr[:3], pcr[3:], 3).astype(f32)
        p[j] = np.nan
        special.append(p)
        p = rng.uniform(pcr[:3], pcr[3:], 3).astype(f32)
        p[j] = -0.0
        special.append(p)
    pts.append(np.asarray(special, f32))
    p = np.concatenate(pts)
    p = p[rng.permutation(p.shape[0])]
    return np.concatenate([p, np.arange(p.shape[0], dtype=f32)[:, None]], 1)


def _check_vox(points_list, vs, pcr, T, M):
    voxels, num, coors, base, _ = hard_voxelize_batch([torch.from_numpy(p).to(DEV) for p in points_list], vs, pcr, T, M)
    rv, rn, rc = vz.voxelize_batch_ref(points_list, vs, pcr, T, M)
    assert np.array_equal(coors.cpu().numpy(), rc)
    assert np.array_equal(num.cpu().numpy(), rn)
    got = voxels.cpu().numpy()
    assert got.shape == rv.shape and np.array_equal(got.view(np.int32), rv.view(np.int32))     # bit for bit (NaN too)


@pytest.mark.parametrize('hash_path', [False, True], ids=['dense', 'hash'])
@pytest.mark.parametrize('grid', list(VOX_GRIDS))
def test_voxelizer_at_voxel_boundaries(grid, hash_path, monkeypatch):
    monkeypatch.setenv('BEVVOX_FORCE_HASH', '1' if hash_path else '0')
    vs, pcr = VOX_GRIDS[grid]
    clouds = [_boundary_cloud(vs, pcr, 1), _boundary_cloud(vs, pcr, 2)[::-1].copy()]
    # the reference itself: the clouds straddle boundaries (both sides kept and dropped)
    zyx, valid = vz.point_coors_numpy(clouds[0], vs, pcr)
    assert 0.05 < valid.mean() < 0.99
    total = sum(c.shape[0] for c in clouds)
    _check_vox(clouds, vs, pcr, 4, total)
    _check_vox(clouds, vs, pcr, 2, total // 20)           # voxel cap reached: the first-point order decides
    for c in clouds:
        got = dynamic_voxelize(torch.from_numpy(c).to(DEV), vs, pcr).cpu().numpy()
        assert np.array_equal(got, vz.point_coors_numpy(c, vs, pcr)[0])


def test_voxelizer_shortcut_branch_is_exercised_by_the_boundary_clouds():
    # the gx = 8192 grid puts x quotients above 4096, where point_to_cell_fast's |q'| < 4096 test hands over to the
    # division; the other grids stay below it, where the 1e-3 margin decides
    for grid, (vs, pcr) in VOX_GRIDS.items():
        c = _boundary_cloud(vs, pcr, 1)[:, :3]
        pmin = np.asarray(pcr[:3], f32)
        q = np.divide(np.subtract(c, pmin, dtype=f32), np.asarray(vs, f32), dtype=f32)
        close = np.abs(q - np.rint(q)) <= 1e-3
        assert close.any(1).mean() > 0.3, grid
        assert (np.nanmax(np.abs(q[:, 0])) >= 4096) == (grid == 'gx-8192'), grid
        fast = qr.point_to_cell_fast(c, pmin, vs, vz.grid_size_ref(vs, pcr))
        assert np.array_equal(fast, qr.ieee_cells(c, pmin, np.asarray(vs, f32), vz.grid_size_ref(vs, pcr))), grid

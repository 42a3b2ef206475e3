"""GPU tests: the BEV augmentation warp kernels (csrc/bev_warp.cu) are BIT-EQUAL to their float32 emulation
oracle/warp_exact_ref.py -- forward and backward, on every map class (rotations, shear, anisotropic and extreme scales,
near-singular and off-centre maps, off-grid translation, coordinates on integers, singular / non-finite theta in a
mixed batch), on grids from 2 x 2 to CFG-2, on one and two channel passes with and without a partial tail, through
row strides, with a pooling plan's ``cell_start``, on inf / NaN data and through the concat epilogue.

Every comparison is on the int32 view (``torch.equal`` calls -0 and +0 equal); NaN positions must match, NaN payloads
are not compared (the device's canonical NaN is not numpy's)."""
import math

import numpy as np
import pytest
import torch

from mm_training_b200 import synthetic
from mm_training_b200.configs import CFG_2
from mm_training_b200.ops import warp_affine
from mm_training_b200.ops.bev_augment import warp_backward_rows, warp_forward_rows, warp_theta
from mm_training_b200.ops.voxel_pooling import build_plan, voxel_pooling_fused, voxel_pooling_fused_concat
from oracle import warp_exact_ref as we
from oracle.warp_affine_ref import about_centre, bda_matrices

pytestmark = pytest.mark.gpu
DEV = 'cuda'
f32 = np.float32
POISON = 0x7FC0DEAD                         # a NaN the kernels never produce: an untouched element keeps these bits


def _np(t):
    return t.detach().float().cpu().contiguous().numpy() if isinstance(t, torch.Tensor) else np.asarray(t, f32)


def assert_bits(name, got, ref):
    got, ref = _np(got), _np(ref)
    assert got.shape == ref.shape, (name, got.shape, ref.shape)
    nan = np.isnan(ref)
    assert np.array_equal(np.isnan(got), nan), f'{name}: NaN pattern differs at {int((np.isnan(got) != nan).sum())} elements'
    diff = got.view(np.int32) != ref.view(np.int32)
    diff &= ~nan
    if diff.any():
        i = np.argwhere(diff)[0]
        raise AssertionError(f'{name}: {int(diff.sum())} of {diff.size} elements differ in bits; first at {tuple(i)}: '
                             f'{got[tuple(i)]!r} vs {ref[tuple(i)]!r}')


def values(shape, seed):
    """Signed full-mantissa float32 values over a few binades, one in 64 a subnormal."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(*shape, generator=g) * torch.exp2(torch.randint(-6, 7, shape, generator=g).float())
    sub = torch.randint(1, 1 << 23, shape, generator=g, dtype=torch.int32).view(torch.float32)
    sub = torch.where(torch.rand(shape, generator=g) < 0.5, -sub, sub)
    return torch.where(torch.rand(shape, generator=g) < 1 / 64, sub, x)


# ---------------------------------------------------------------------------------------------- map classes
def _rot(a):
    return torch.tensor([[math.cos(a), -math.sin(a)], [math.sin(a), math.cos(a)]], dtype=torch.float64)


def _lin(L, B):
    return L.expand(B, 2, 2)


def _scaled(m):
    """Magnification (m > 1) or minification about the source centre, onto a destination scaled with it."""
    return lambda B, Hs, Ws, Hd, Wd: about_centre(_lin(m * torch.eye(2, dtype=torch.float64), B), Hs, Ws)


def _near_singular(k):
    # M = R1 diag(1, 1/k) R2: det / |M|^2 = k; the destination grid sees a sliver of the source a fraction k wide,
    # and every source cell's candidate window is a long strip clipped to the grid
    L = _rot(0.3) @ torch.diag(torch.tensor([1.0, 1.0 / k], dtype=torch.float64)) @ _rot(1.1)
    return lambda B, Hs, Ws, Hd, Wd: about_centre(_lin(L, B), Hs, Ws)


def _off_centre(m):
    # magnification m about a point near the bottom-right corner: theta's translation is about +-(1 - 1/m), so
    # fma(th0, xn, fma(th1, yn, th2)) cancels to small coordinates near that corner
    def f(B, Hs, Ws, Hd, Wd):
        L = m * torch.eye(2, dtype=torch.float64)
        c = torch.tensor([Ws - 1.3, Hs - 1.3], dtype=torch.float64)
        return torch.cat([L, (c - L @ c)[:, None]], -1).expand(B, 2, 3).clone()
    return f


def _mats(kind, B, Hs, Ws, Hd, Wd):
    eye = torch.eye(2, dtype=torch.float64)
    if kind == 'bda':
        return bda_matrices(B, Hs, Ws, seed=B + Hs)
    if kind == 'singular':
        return torch.zeros(B, 2, 3)
    fixed = {
        'identity': eye, 'rot90': torch.tensor([[0.0, -1.0], [1.0, 0.0]], dtype=torch.float64),
        'rot45': _rot(math.pi / 4), 'rot135': _rot(3 * math.pi / 4), 'rot_random': _rot(2.2437),
        'shear': torch.tensor([[1.0, 0.7], [0.0, 1.0]], dtype=torch.float64),
        'aniso': torch.diag(torch.tensor([3.0, 0.3], dtype=torch.float64)),
    }
    if kind in fixed:
        return about_centre(_lin(fixed[kind], B), Hs, Ws)
    if kind == 'flips':
        f = torch.tensor([[-1.0, 1.0], [1.0, -1.0], [-1.0, -1.0]], dtype=torch.float64)[torch.arange(B) % 3]
        return about_centre(torch.diag_embed(f), Hs, Ws)
    if kind == 'translate':
        m = about_centre(_lin(eye, B), Hs, Ws)
        m[:, 0, 2], m[:, 1, 2] = 3.0, -2.0
        return m
    if kind == 'off_grid':                                    # the whole destination lands beyond the source
        m = about_centre(_lin(eye, B), Hs, Ws)
        m[:, 0, 2] += Wd + 3.0
        return m
    if kind == 'half_pixel':                                  # destination x samples source x - 0.5: weights 1/2, 0
        m = about_centre(_lin(eye, B), Hs, Ws)
        m[:, 0, 2] += 0.5
        return m
    table = {'mag2': _scaled(2.0), 'mag4': _scaled(4.0), 'mag16': _scaled(16.0), 'mag64': _scaled(64.0),
             'min05': _scaled(0.5), 'min025': _scaled(0.25), 'min01': _scaled(0.1),
             'near_singular_1e-2': _near_singular(1e-2), 'near_singular_1e-4': _near_singular(1e-4),
             'off_centre_16': _off_centre(16.0), 'off_centre_1000': _off_centre(1000.0)}
    return table[kind](B, Hs, Ws, Hd, Wd)


MAPS = ['bda', 'identity', 'flips', 'translate', 'rot90', 'mag2', 'min05', 'singular', 'rot45', 'rot135', 'rot_random',
        'shear', 'aniso', 'mag4', 'mag16', 'mag64', 'min025', 'min01', 'near_singular_1e-2', 'near_singular_1e-4',
        'off_centre_16', 'off_centre_1000', 'off_grid', 'half_pixel']
# (B, C, Hs, Ws, (Hd, Wd))
SHAPES = {'cfg2': (8, 80, 64, 512, (64, 512)), 'g2x2': (2, 4, 2, 2, (2, 2)), 'g2x1024': (2, 8, 2, 1024, (2, 1024)),
          'larger': (2, 12, 9, 14, (23, 31)), 'smaller': (2, 12, 40, 36, (11, 17))}
BIG_MAGNIFICATION = {'mag16', 'mag64', 'off_centre_1000'}     # small grids only: the window grows as m^2


def _theta(M, src_hw, dsize):
    return warp_theta(M.float().to(DEV), src_hw, dsize)


def _forward(theta, src, dsize, cell_start=None):
    B, Hs, Ws, C = src.shape
    out = torch.empty(B, *dsize, C, device=DEV)
    warp_forward_rows(theta, src, C, out, C, cell_start, B, C, (Hs, Ws), dsize)
    return out


def _backward(theta, g, src_hw, cell_start=None, out=None):
    B, Hd, Wd, C = g.shape
    gs = torch.empty(B, *src_hw, C, device=DEV) if out is None else out
    warp_backward_rows(theta, g, C, gs, C, cell_start, B, C, src_hw, (Hd, Wd))
    return gs


def _check_both(name, theta, x_rows, g_rows, src_hw, dsize):
    th = theta.cpu().numpy()
    out = _forward(theta, x_rows, dsize)
    assert_bits(f'{name} forward', out, we.warp_forward_exact(th, _np(x_rows), dsize))
    gs = _backward(theta, g_rows, src_hw)
    assert_bits(f'{name} backward', gs, we.warp_backward_exact(th, _np(g_rows), src_hw))
    return out, gs


@pytest.mark.parametrize('kind', MAPS)
@pytest.mark.parametrize('shape', list(SHAPES))
def test_op_forward_and_backward_bit_equal_to_the_emulation(shape, kind):
    B, C, Hs, Ws, dsize = SHAPES[shape]
    if kind in BIG_MAGNIFICATION and shape == 'cfg2':
        pytest.skip('extreme magnifications run on the small grids')
    M = _mats(kind, B, Hs, Ws, *dsize).float().to(DEV)
    x = values((B, C, Hs, Ws), seed=100 * MAPS.index(kind) + list(SHAPES).index(shape)).to(DEV)
    go = values((B, C, *dsize), seed=7).to(DEV)
    xs = x.clone().requires_grad_(True)
    out = warp_affine(xs, M, dsize)                                   # the op: theta on the device, NCHW in
    out.backward(go)
    th = warp_theta(M, (Hs, Ws), dsize).cpu().numpy()
    ref = we.warp_forward_exact(th, _np(x.permute(0, 2, 3, 1)), dsize)
    assert_bits('forward', out.permute(0, 2, 3, 1), ref)
    gref = we.warp_backward_exact(th, _np(go.permute(0, 2, 3, 1)), (Hs, Ws))
    assert_bits('backward', xs.grad.permute(0, 2, 3, 1), gref)
    if kind == 'singular':                                            # no tap: zeros both ways
        assert not ref.any() and not gref.any()
    if kind in ('min025', 'min01') and shape == 'cfg2':              # most source cells get no gradient at all
        assert (np.abs(gref).sum(-1) == 0).mean() > 0.5


def test_extreme_magnification_next_to_an_integer():
    # 2e5x about a point 4e-4 px right of source column 510 on the CFG-2 grid: the destination pixels near column 390
    # sample coordinates within float32 error of 510, and that error (~1e-5 px) is over 3 destination pixels here.
    # A backward window widened by a flat one pixel instead of the error bound missed 256 of these pairs.
    Hs, Ws, C = 64, 512, 8
    L = 2e5 * torch.eye(2, dtype=torch.float64)
    c = torch.tensor([Ws - 2 + 4e-4, (Hs - 1) / 2], dtype=torch.float64)
    theta = _theta(torch.cat([L, (c - L @ c)[:, None]], -1)[None], (Hs, Ws), (Hs, Ws))
    taps = we.warp_taps(theta.cpu().numpy(), Hs, Ws, Hs, Ws)
    assert np.unique(taps.x0[taps.valid[..., 0]]).tolist() == [Ws - 3, Ws - 2]     # the coordinates straddle 510
    _check_both('2e5x', theta, values((1, Hs, Ws, C), 16).to(DEV), values((1, Hs, Ws, C), 17).to(DEV), (Hs, Ws), (Hs, Ws))


def test_mixed_batch_with_singular_and_non_finite_theta():
    B, C, Hs, Ws, dsize = 5, 16, 20, 28, (24, 24)
    M = bda_matrices(B, Hs, Ws, seed=3).to(DEV)
    theta = warp_theta(M, (Hs, Ws), dsize)
    theta[1] = 0.0                                                    # singular: every pixel samples the centre
    theta[2, 0, 1] = float('nan')
    theta[3, 1, 2] = float('inf')
    x = values((B, Hs, Ws, C), 1).to(DEV)
    g = values((B, *dsize, C), 2).to(DEV)
    out, gs = _check_both('mixed', theta, x, g, (Hs, Ws), dsize)
    assert not bool(out[2:4].any()) and not bool(gs[2:4].any())
    for b in (0, 4):                                                  # the regular samples are unaffected
        o1 = _forward(theta[b:b + 1].contiguous(), x[b:b + 1].contiguous(), dsize)
        g1 = _backward(theta[b:b + 1].contiguous(), g[b:b + 1].contiguous(), (Hs, Ws))
        assert_bits(f'sample {b} forward', out[b:b + 1], o1)
        assert_bits(f'sample {b} backward', gs[b:b + 1], g1)


@pytest.mark.parametrize('C', [4, 128, 132, 256])
@pytest.mark.parametrize('kind', ['rot_random', 'mag4'])
def test_channel_passes(C, kind):
    # a pass of the kernels' channel loop covers 8 lanes x 4 float4 = 128 channels: one pass, exactly one, a second
    # pass with a partial tail, two full passes
    B, Hs, Ws, dsize = 2, 24, 40, (30, 36)
    theta = _theta(_mats(kind, B, Hs, Ws, *dsize), (Hs, Ws), dsize)
    _check_both(f'C={C}', theta, values((B, Hs, Ws, C), C).to(DEV), values((B, *dsize, C), C + 1).to(DEV), (Hs, Ws), dsize)


@pytest.mark.parametrize('C', [80, 132])
def test_row_strides_through_the_abi(C):
    B, Hs, Ws, dsize = 2, 24, 40, (30, 36)
    S = C + 12
    theta = _theta(_mats('rot_random', B, Hs, Ws, *dsize), (Hs, Ws), dsize)
    th = theta.cpu().numpy()
    poison = lambda *shape: torch.full(shape, POISON, dtype=torch.int32, device=DEV).view(torch.float32)
    x = values((B, Hs, Ws, C), 5).to(DEV)
    src = poison(B, Hs, Ws, S)
    src[..., :C] = x
    out = poison(B, *dsize, S)
    warp_forward_rows(theta, src, S, out, S, None, B, C, (Hs, Ws), dsize)
    assert_bits('strided forward', out[..., :C], we.warp_forward_exact(th, _np(x), dsize))
    assert bool((out[..., C:].view(torch.int32) == POISON).all())
    g = values((B, *dsize, C), 6).to(DEV)
    gbuf = poison(B, *dsize, S)
    gbuf[..., :C] = g
    gs = poison(B, Hs, Ws, S)
    warp_backward_rows(theta, gbuf, S, gs, S, None, B, C, (Hs, Ws), dsize)
    assert_bits('strided backward', gs[..., :C], we.warp_backward_exact(th, _np(g), (Hs, Ws)))
    assert bool((gs[..., C:].view(torch.int32) == POISON).all())


# ---------------------------------------------------------------------------------------------- cell_start
def _synthetic_cell_start(B, Hs, Ws, seed):
    """CSR with about half the cells empty, in runs next to occupied ones (1 to 3 entries per occupied cell)."""
    g = torch.Generator().manual_seed(seed)
    counts = torch.randint(1, 4, (B * Hs * Ws,), generator=g) * (torch.rand(B * Hs * Ws, generator=g) < 0.5)
    return torch.cat([torch.zeros(1, dtype=torch.int64), counts.cumsum(0)]).int()


def _camera_plan(B, seed=8):
    geom, vn_t = synthetic.camera_rig(CFG_2, B, device=DEV, yaw_jitter_deg=5.0, seed=seed)
    vn = tuple(int(v) for v in vn_t.tolist())
    plan = build_plan(geom, vn, frustum=tuple(geom.shape[1:5]))
    return geom, vn, plan


@pytest.mark.parametrize('csr', ['plan', 'synthetic'])
def test_cell_start_skips_empty_cells_and_writes_only_occupied_rows(csr):
    if csr == 'plan':
        B, C = 2, 80
        _, (X, Y, _), plan = _camera_plan(B)
        Hs, Ws, cs = Y, X, plan.cell_start
    else:
        B, C, Hs, Ws = 3, 132, 30, 44
        cs = _synthetic_cell_start(B, Hs, Ws, 4).to(DEV)
    dsize = (Hs, Ws)
    occ = (cs[1:] != cs[:-1]).view(B, Hs, Ws)
    assert 0 < int(occ.sum()) < occ.numel()
    theta = _theta(_mats('bda', B, Hs, Ws, *dsize), (Hs, Ws), dsize)
    th, cs_np = theta.cpu().numpy(), cs.cpu().numpy()
    x = values((B, Hs, Ws, C), 9).to(DEV)
    x[~occ] = float('nan')                                            # an empty cell's row is never read
    out = _forward(theta, x, dsize, cs)
    assert_bits('forward, cell_start', out, we.warp_forward_exact(th, _np(x), dsize, cell_start=cs_np))
    g = values((B, *dsize, C), 10).to(DEV)
    gs = torch.full((B, Hs, Ws, C), POISON, dtype=torch.int32, device=DEV).view(torch.float32)
    gs = _backward(theta, g, (Hs, Ws), cs, out=gs)
    assert_bits('backward, occupied rows', gs[occ], we.warp_backward_exact(th, _np(g), (Hs, Ws), cell_start=cs_np)[_np(occ) > 0])
    assert bool((gs[~occ].view(torch.int32) == POISON).all())


def test_skipping_empty_cells_equals_reading_zero_rows_by_value_not_by_sign():
    # Even source rows occupied, odd rows empty; occupied values -2^-149 (the smallest subnormal).  A product with a
    # weight <= 1/2 underflows to -0, so a pixel whose nw / ne taps are occupied ends at -0 when its sw / se taps are
    # skipped, and at +0 (-0 + w * 0) when they read the zero rows: equal values, different sign bits.
    B, C, Hs, Ws = 2, 8, 32, 48
    dsize = (Hs, Ws)
    occ = torch.zeros(B, Hs, Ws, dtype=torch.bool)
    occ[:, 0::2] = True
    cs = torch.cat([torch.zeros(1, dtype=torch.int64), occ.reshape(-1).long().cumsum(0)]).int().to(DEV)
    x = torch.where(occ[..., None], torch.tensor(-2.0 ** -149), torch.tensor(0.0)).expand(B, Hs, Ws, C).contiguous().to(DEV)
    theta = _theta(_mats('rot_random', B, Hs, Ws, *dsize), (Hs, Ws), dsize)
    th = theta.cpu().numpy()
    skipped, read = _forward(theta, x, dsize, cs.to(DEV)), _forward(theta, x, dsize)
    assert_bits('skipped', skipped, we.warp_forward_exact(th, _np(x), dsize, cell_start=cs.cpu().numpy()))
    assert_bits('read', read, we.warp_forward_exact(th, _np(x), dsize))
    assert torch.equal(skipped, read)                                # same values ...
    neg = lambda t: int(torch.signbit(t).sum())
    assert neg(skipped) > neg(read)                                   # ... but skipping keeps -0 where reading gives +0


# ---------------------------------------------------------------------------------------------- non-finite data
@pytest.mark.parametrize('kind', ['identity', 'half_pixel', 'bda', 'mag4'])
def test_inf_and_nan_data_give_the_emulated_nan_pattern(kind):
    # identity and half_pixel put valid zero-weight taps everywhere: fmaf(inf, 0, acc) is NaN there
    B, C, Hs, Ws = 2, 12, 20, 30
    dsize = (Hs, Ws)
    theta = _theta(_mats(kind, B, Hs, Ws, *dsize), (Hs, Ws), dsize)
    gen = torch.Generator().manual_seed(12)

    def sprinkle(t):
        r = torch.rand(t.shape, generator=gen)
        t = torch.where(r < 0.01, torch.tensor(float('inf')), t)
        t = torch.where((r >= 0.01) & (r < 0.02), torch.tensor(float('-inf')), t)
        return torch.where((r >= 0.02) & (r < 0.025), torch.tensor(float('nan')), t)
    x = sprinkle(values((B, Hs, Ws, C), 13)).to(DEV)
    g = sprinkle(values((B, *dsize, C), 14)).to(DEV)
    out, gs = _check_both(kind, theta, x, g, (Hs, Ws), dsize)
    assert bool(out.isnan().any()) and bool(gs.isnan().any())


# ---------------------------------------------------------------------------------------------- the concat epilogue
def test_concat_with_bda_bit_equal_to_the_emulated_warp_of_the_pooled_rows():
    B = 8
    geom, vn, plan = _camera_plan(B, seed=6)
    X, Y, _ = vn
    depth, ctx, _ = synthetic.camera_features(CFG_2, B, device=DEV, seed=6)
    C = ctx.shape[1]
    gen = torch.Generator().manual_seed(6)
    other = torch.randn(B, 16, Y, X, generator=gen).to(DEV)
    go = values((B, C + 16, Y, X), 15).to(DEV).contiguous(memory_format=torch.channels_last)
    M = bda_matrices(B, Y, X, seed=6).to(DEV)
    th = warp_theta(M, (Y, X), (Y, X)).cpu().numpy()
    cs = plan.cell_start.cpu().numpy()
    d, c, o = (t.clone().requires_grad_(True) for t in (depth, ctx, other))
    out = voxel_pooling_fused_concat(d, c, o, vn, plan, bda_affine=M)
    out.backward(go)
    # forward: the emulated warp (empty cells skipped) of the pooled rows, which the pooling gives bit for bit
    pooled = voxel_pooling_fused(None, depth, ctx, vn, plan)
    ref = we.warp_forward_exact(th, _np(pooled.permute(0, 2, 3, 1)), (Y, X), cell_start=cs)
    assert_bits('camera half', out[:, :C].permute(0, 2, 3, 1), ref)
    # backward: the pooling backward fed the emulated warp backward of the camera slice of the gradient
    gp = we.warp_backward_exact(th, _np(go[:, :C].permute(0, 2, 3, 1)), (Y, X), cell_start=cs)
    d2, c2 = (t.clone().requires_grad_(True) for t in (depth, ctx))
    pooled = voxel_pooling_fused(None, d2, c2, vn, plan)
    pooled.backward(torch.from_numpy(gp).to(DEV).permute(0, 3, 1, 2))
    assert_bits('grad depth', d.grad, d2.grad)
    assert_bits('grad context', c.grad, c2.grad)

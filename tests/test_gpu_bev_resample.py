"""GPU tests of the LiDAR BEV nearest resampling (csrc/bev_resample.cu) and of the concat epilogue with it
(``voxel_pooling_fused_concat(..., resize_other='nearest')``).  Oracle: torch's own ``F.interpolate(mode='nearest')``
(the forward is a copy, so bit-equal), its CUDA autograd (bit-equal on integer ratios in fp32: same sums, same order)
and its fp64 autograd on the CPU as the adjoint.

Gradient tolerance, per element: |got - ref64| <= k * 2^-24 * S + u * (|ref64| + k * 2^-24 * S), k the largest preimage
(terms summed per source cell), S the sum of |terms|, u the unit roundoff of the source dtype (0 for fp32)."""

import pytest
import torch
import torch.nn.functional as F

from mm_training_b200 import _lib, synthetic
from mm_training_b200.configs import CFG_2
from mm_training_b200.ops import warp_affine
from mm_training_b200.ops.voxel_pooling import build_plan, voxel_pooling_fused, voxel_pooling_fused_concat
from oracle.warp_affine_ref import bda_matrices as bda_mats

pytestmark = pytest.mark.gpu
DEV = 'cuda'
DTYPES = [torch.float32, torch.bfloat16, torch.float16]
UNIT = {torch.float32: 0.0, torch.bfloat16: 2.0 ** -8, torch.float16: 2.0 ** -11}

# name: (src (Yl, Xl), dst (Y, X), batch, channel counts)
SHAPES = {
    'up2': ((32, 256), (64, 512), 2, (4, 256, 384)),
    'down4': ((256, 2048), (64, 512), 1, (4, 256)),
    'identity': ((64, 512), (64, 512), 2, (4, 256, 384)),
    'frac48x200': ((48, 200), (64, 512), 2, (4, 256, 384)),
    'frac100x700': ((100, 700), (64, 512), 2, (4, 256)),
    'odd_dst': ((40, 50), (37, 45), 2, (4, 384)),            # destination width not a multiple of 32
    'from1': ((1, 3), (5, 70), 3, (4,)),
}
INTEGER_RATIOS = ('up2', 'down4', 'identity')
CASES = [(n, c2) for n, s in SHAPES.items() for c2 in s[3]]


def _other(B, C2, hw, dtype, channels_last, seed=0):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, C2, *hw, generator=g).to(dtype).to(DEV)
    return x.contiguous(memory_format=torch.channels_last) if channels_last else x


def _native_into(other, dst, C):
    """The forward kernel into a (B, Y, X, C + C2) buffer whose camera channels hold NaN (they must stay untouched)."""
    B, C2, Yl, Xl = other.shape
    buf = torch.full((B, *dst, C + C2), float('nan'), device=DEV)
    nchw = 1 if other.is_contiguous() else 0
    _lib.check(_lib.lib().bevpool_resize_nearest_into(other.data_ptr(), _lib.dtype_code(other), nchw, B, C2, Yl, Xl,
                                                      dst[0], dst[1], buf.data_ptr() + 4 * C, C + C2,
                                                      _lib.stream_ptr(DEV)), 'resize_into')
    return buf


def _native_backward(g_rows, C, like):
    B, C2, Yl, Xl = like.shape
    _, Y, X, Ct = g_rows.shape
    nchw = 1 if like.is_contiguous() else 0
    out = torch.empty_like(like)
    _lib.check(_lib.lib().bevpool_resize_nearest_backward_from(g_rows.data_ptr() + 4 * C, Ct, out.data_ptr(),
                                                               _lib.dtype_code(like), nchw, B, C2, Yl, Xl, Y, X,
                                                               _lib.stream_ptr(DEV)), 'resize_backward_from')
    return out


def _adjoint64(g, src_hw):
    x = torch.zeros(*g.shape[:2], *src_hw, dtype=torch.float64, requires_grad=True)
    F.interpolate(x, size=g.shape[2:], mode='nearest').backward(g.double().cpu())
    return x.grad


def _check_grad(got, g_lidar, other_shape, dtype):
    """got against the fp64 CPU autograd of F.interpolate for the incoming LiDAR gradient g_lidar (B, C2, Y, X).
    Channels are independent: of a large source only the first and last 8 are checked here (the integer-ratio cases
    compare every channel with torch's CUDA autograd)."""
    if got.numel() > 2 ** 25:
        got = torch.cat([got[:, :8], got[:, -8:]], 1)
        g_lidar = torch.cat([g_lidar[:, :8], g_lidar[:, -8:]], 1)
    src_hw = other_shape[2:]
    ref, S = _adjoint64(g_lidar, src_hw), _adjoint64(g_lidar.abs(), src_hw)
    k = float(_adjoint64(torch.ones(1, 1, *g_lidar.shape[2:]), src_hw).max())
    e32 = k * 2.0 ** -24 * S
    tol = e32 + UNIT[dtype] * (ref.abs() + e32) + (2.0 ** -24 if dtype == torch.float16 else 0.0)
    err = (got.double().cpu() - ref).abs()
    assert bool((err <= tol).all()), f'max excess {float((err - tol).max())}'


@pytest.mark.parametrize('channels_last', [False, True], ids=['nchw', 'cl'])
@pytest.mark.parametrize('dtype', DTYPES, ids=str)
@pytest.mark.parametrize('name,C2', CASES)
def test_kernels_against_torch(name, C2, dtype, channels_last):
    src, dst, B, _ = SHAPES[name]
    C = 16
    other = _other(B, C2, src, dtype, channels_last)
    buf = _native_into(other, dst, C)
    ref = F.interpolate(other, size=dst, mode='nearest').float()
    assert torch.equal(buf[..., C:].permute(0, 3, 1, 2), ref)
    assert bool(buf[..., :C].isnan().all())
    g = torch.randn(B, *dst, C + C2, generator=torch.Generator().manual_seed(1)).to(DEV)
    got = _native_backward(g, C, other)
    assert got.dtype == other.dtype and got.is_contiguous() == other.is_contiguous()
    g_lidar = g[..., C:].permute(0, 3, 1, 2)
    if dtype == torch.float32 and name in INTEGER_RATIOS:
        o = other.clone().requires_grad_(True)
        F.interpolate(o, size=dst, mode='nearest').backward(g_lidar)
        assert torch.equal(got, o.grad)
    _check_grad(got, g_lidar, other.shape, dtype)
    assert torch.equal(_native_backward(g, C, other), got)                  # bit-stable


# ---------------------------------------------------------------- the concat epilogue
@pytest.fixture(scope='module')
def camera():
    B = 2
    geom, vn_t = synthetic.camera_rig(CFG_2, B, device=DEV, yaw_jitter_deg=5.0, seed=8)
    vn = tuple(int(v) for v in vn_t.tolist())
    depth, ctx, _ = synthetic.camera_features(CFG_2, B, device=DEV, seed=8)
    plan = build_plan(geom, vn, frustum=tuple(geom.shape[1:5]))
    assert plan.mode == 'runs'
    X, Y, _ = vn
    return dict(geom=geom, vn=vn, depth=depth, ctx=ctx, plan=plan, M=bda_mats(B, Y, X, seed=8).to(DEV), B=B)


def _go(cam, C2, seed=2, channels_last=True):
    X, Y, _ = cam['vn']
    go = torch.rand(cam['B'], CFG_2.output_channels + C2, Y, X, generator=torch.Generator().manual_seed(seed)).to(DEV)
    return go.contiguous(memory_format=torch.channels_last) if channels_last else go


def _run(cam, other, go, plan=None, M=None, resize='nearest'):
    d, c, o = (t.clone().requires_grad_(True) for t in (cam['depth'], cam['ctx'], other))
    out = voxel_pooling_fused_concat(d, c, o, cam['vn'], plan or cam['plan'], bda_affine=M, resize_other=resize)
    out.backward(go)
    return out.detach(), d.grad, c.grad, o.grad


def _stock(cam, other, go, plan=None, M=None):
    """camera half (the native ops) + F.interpolate(...).float(), autograd through torch for the LiDAR half"""
    X, Y, _ = cam['vn']
    d, c, o = (t.clone().requires_grad_(True) for t in (cam['depth'], cam['ctx'], other))
    cam_half = voxel_pooling_fused(None, d, c, cam['vn'], plan or cam['plan'])
    if M is not None:
        cam_half = warp_affine(cam_half, M, (Y, X))
    out = torch.cat([cam_half, F.interpolate(o, size=(Y, X), mode='nearest').float()], 1)
    out.backward(go)
    return out.detach(), d.grad, c.grad, o.grad


OP_CASES = [('up2', 256, torch.float32, False), ('up2', 256, torch.bfloat16, True), ('down4', 4, torch.float32, True),
            ('down4', 4, torch.float16, False), ('frac48x200', 384, torch.float32, False),
            ('frac100x700', 4, torch.bfloat16, True), ('up2', 384, torch.float16, True)]


@pytest.mark.parametrize('bda', [False, True], ids=['plain', 'bda'])
@pytest.mark.parametrize('name,C2,dtype,channels_last', OP_CASES)
def test_concat_with_resize_equals_the_stock_composition(camera, name, C2, dtype, channels_last, bda):
    src = SHAPES[name][0]
    X, Y, _ = camera['vn']
    C = CFG_2.output_channels
    other = _other(camera['B'], C2, src, dtype, channels_last, seed=3)
    go = _go(camera, C2)
    M = camera['M'] if bda else None
    out, gd, gc, go_ = _run(camera, other, go, M=M)
    ref = _stock(camera, other, go, M=M)
    assert out.permute(0, 2, 3, 1).is_contiguous()
    assert torch.equal(out, ref[0])
    # the camera gradients are those of the call without resize_other (on the pre-resampled LiDAR BEV)
    pre = F.interpolate(other, size=(Y, X), mode='nearest')
    plain = _run(camera, pre, go, M=M, resize=None)
    assert torch.equal(gd, plain[1]) and torch.equal(gc, plain[2])
    assert go_.dtype == other.dtype and go_.shape == other.shape
    assert go_.is_contiguous() == other.is_contiguous()
    assert go_.permute(0, 2, 3, 1).is_contiguous() == other.permute(0, 2, 3, 1).is_contiguous()
    if dtype == torch.float32 and name in INTEGER_RATIOS:
        assert torch.equal(go_, ref[3])
    _check_grad(go_, go[:, C:], other.shape, dtype)
    # an NCHW incoming gradient (the copying path) gives the same values
    nchw = _run(camera, other, go.contiguous(), M=M)
    for a, b in zip(nchw, (out, gd, gc, go_)):
        assert torch.equal(a, b)
    # bit-stable run to run
    again = _run(camera, other, go, M=M)
    for a, b in zip(again, (out, gd, gc, go_)):
        assert torch.equal(a, b)


@pytest.mark.parametrize('channels_last', [False, True], ids=['nchw', 'cl'])
@pytest.mark.parametrize('bda', [False, True], ids=['plain', 'bda'])
def test_same_size_resize_equals_no_resize(camera, bda, channels_last):
    X, Y, _ = camera['vn']
    other = _other(camera['B'], 256, (Y, X), torch.float32, channels_last, seed=4)
    go = _go(camera, 256)
    M = camera['M'] if bda else None
    a = _run(camera, other, go, M=M)
    b = _run(camera, other, go, M=M, resize=None)
    for u, v in zip(a, b):
        assert torch.equal(u, v)
    assert torch.equal(a[0], _stock(camera, other, go, M=M)[0])


@pytest.mark.parametrize('bda', [False, True], ids=['plain', 'bda'])
def test_concat_with_resize_replays_in_a_cuda_graph(camera, bda):
    geom, vn = camera['geom'], camera['vn']
    fr = tuple(geom.shape[1:5])
    n = camera['plan'].num_sorted
    other = _other(camera['B'], 256, (32, 256), torch.bfloat16, False, seed=5)
    go = _go(camera, 256)
    M = camera['M'] if bda else None
    eager = _run(camera, other, go, M=M)
    d, c, o = (t.clone().requires_grad_(True) for t in (camera['depth'], camera['ctx'], other))

    def step():
        plan = build_plan(geom, vn, frustum=fr, max_runs=n)
        out = voxel_pooling_fused_concat(d, c, o, vn, plan, bda_affine=M, resize_other='nearest')
        return (out,) + torch.autograd.grad(out, (d, c, o), go)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        step()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        captured = step()
    for t in captured:
        t.detach().fill_(float('nan'))
    graph.replay()
    torch.cuda.synchronize()
    for a, b in zip(captured, eager):
        assert torch.equal(a.detach(), b)


@pytest.mark.parametrize('bda', [False, True], ids=['plain', 'bda'])
def test_fallbacks_equal_the_stock_composition(camera, bda):
    M = camera['M'] if bda else None
    # a point plan
    point_plan = build_plan(camera['geom'], camera['vn'])
    assert point_plan.mode == 'points'
    other = _other(camera['B'], 8, (32, 256), torch.float32, False, seed=6)
    go = _go(camera, 8)
    for a, b in zip(_run(camera, other, go, plan=point_plan, M=M), _stock(camera, other, go, plan=point_plan, M=M)):
        assert torch.equal(a, b)
    # C2 % 4 != 0
    other = _other(camera['B'], 6, (32, 256), torch.float32, True, seed=7)
    go = _go(camera, 6)
    for a, b in zip(_run(camera, other, go, M=M), _stock(camera, other, go, M=M)):
        assert torch.equal(a, b)

"""GPU tests of the BEV augmentation warp (csrc/bev_warp.cu, ops/bev_augment.py) and of the concat epilogue with the
BDA warp (``voxel_pooling_fused_concat(..., bda_affine=M)``).  Oracle: oracle/warp_affine_ref.py (kornia's sequence
restated with torch ops) in float64, and torch's own float32 affine_grid + grid_sample on the same device.

Tolerance, per element: |out - ref64| <= 1e-5 |ref64| + 8 * 2^-23 * max(H, W) * S, S = sum of |value| over the taps.
A float32 pixel coordinate near 512 is only good to about 6e-5 px, so every bilinear weight -- however small -- carries
an absolute error of that order, and the output error is bounded by it times the magnitudes the weights multiply
(torch's float32 kernel has the same error).  The gradient uses the same form, with S the adjoint tap sum of |grad|."""
import importlib
import math

import pytest
import torch

from mm_training_b200 import synthetic
from mm_training_b200.configs import CFG_2
from mm_training_b200.ops import warp_affine
from mm_training_b200.ops.voxel_pooling import build_plan, voxel_pooling_fused, voxel_pooling_fused_concat
from oracle import voxel_pool_ref as vp
from oracle import warp_affine_ref as wr
from oracle.warp_affine_ref import about_centre as _about_centre, bda_matrices as bda_mats

vp_mod = importlib.import_module('mm_training_b200.ops.voxel_pooling.voxel_pooling')
pytestmark = pytest.mark.gpu
DEV = 'cuda'

# (B, C, H, W, dsize): the CFG-2 BEV grid, the 128^2 sweep grid, an odd small grid, a destination of another size
SHAPES = {'cfg2': (8, 80, 64, 512, (64, 512)), 'sweep128': (2, 80, 128, 128, (128, 128)),
          'odd7x9': (2, 4, 7, 9, (7, 9)), 'resize': (2, 16, 48, 40, (56, 36))}
MATS = ['bda', 'identity', 'flips', 'translate', 'rot90', 'mag2', 'min05', 'singular']


def make_mats(kind: str, B: int, H: int, W: int) -> torch.Tensor:
    eye = torch.eye(2, dtype=torch.float64).expand(B, 2, 2)
    if kind == 'bda':
        return bda_mats(B, H, W)
    if kind == 'identity':
        return _about_centre(eye, H, W).float()
    if kind == 'flips':
        f = torch.tensor([[-1.0, 1.0], [1.0, -1.0], [-1.0, -1.0]], dtype=torch.float64)[torch.arange(B) % 3]
        return _about_centre(torch.diag_embed(f), H, W).float()
    if kind == 'translate':
        m = _about_centre(eye, H, W)
        m[:, 0, 2], m[:, 1, 2] = 3.0, -2.0
        return m.float()
    if kind == 'rot90':
        return _about_centre(torch.tensor([[0.0, -1.0], [1.0, 0.0]], dtype=torch.float64).expand(B, 2, 2), H, W).float()
    if kind == 'mag2':
        return _about_centre(2 * eye, H, W).float()
    if kind == 'min05':
        return _about_centre(0.5 * eye, H, W).float()
    if kind == 'singular':
        return torch.zeros(B, 2, 3)
    raise KeyError(kind)


def _bound(ref64, S, H, W):
    return 1e-5 * ref64.abs() + 8 * 2.0 ** -23 * max(H, W) * S + 1e-30


def _check(name, got, ref64, bound, factor=1.0):
    err = (got.double() - ref64).abs()
    bad = err > factor * bound
    assert not bool(bad.any()), f'{name}: {int(bad.sum())} elements out of bound, max err {float(err.max()):.3g}'


@pytest.mark.parametrize('kind', MATS)
@pytest.mark.parametrize('shape', list(SHAPES))
def test_forward_backward_against_fp64_oracle_and_torch(shape, kind):
    B, C, H, W, dsize = SHAPES[shape]
    g = torch.Generator().manual_seed(11)
    x = (torch.rand(B, C, H, W, generator=g) - 0.5).to(DEV)
    go = (torch.rand(B, C, *dsize, generator=g) - 0.5).to(DEV)
    M = make_mats(kind, B, H, W).to(DEV)
    xs = x.clone().requires_grad_(True)
    out = warp_affine(xs, M, dsize)
    assert out.shape == (B, C, *dsize) and out.permute(0, 2, 3, 1).is_contiguous()
    out.backward(go)
    if kind == 'singular':                              # non-finite theta: zeros both ways, no fault
        assert bool((out == 0).all()) and bool((xs.grad == 0).all())
        return
    x64 = x.double().requires_grad_(True)
    ref64 = wr.warp_affine_ref(x64, M, dsize)
    ref64.backward(go.double())
    S = wr.tap_sum_ref(x.abs(), M, dsize)
    a = torch.zeros(B, C, H, W, dtype=torch.float64, device=DEV, requires_grad=True)
    (Sb,) = torch.autograd.grad(wr.tap_sum_ref(a, M, dsize), a, go.abs().double())
    fb, bb = _bound(ref64.detach(), S, H, W), _bound(x64.grad, Sb, H, W)
    _check('forward vs fp64', out.detach(), ref64.detach(), fb)
    _check('backward vs fp64', xs.grad, x64.grad, bb)
    # torch's float32 kernels on the same device carry the same error: twice the bound between the two
    x32 = x.clone().requires_grad_(True)
    ref32 = wr.warp_affine_ref(x32, M, dsize, dtype=torch.float32)
    ref32.backward(go)
    _check('forward vs torch fp32', out.detach(), ref32.detach().double(), fb, 2.0)
    _check('backward vs torch fp32', xs.grad, x32.grad.double(), bb, 2.0)


@pytest.mark.parametrize('kind', ['identity', 'flips', 'translate', 'rot90'])
@pytest.mark.parametrize('shape', ['cfg2', 'odd7x9', 'sweep128'])
def test_backward_is_the_adjoint_of_the_forward(shape, kind):
    """<warp(x), g> == <x, warp_bwd(g)> in float64: a (destination, tap) pair the backward's candidate window dropped
    would carry a weight of about 1 in these cases."""
    B, C, H, W, dsize = SHAPES[shape]
    g = torch.Generator().manual_seed(5)
    x = torch.rand(B, C, H, W, generator=g).to(DEV).requires_grad_(True)
    go = torch.rand(B, C, *dsize, generator=g).to(DEV)
    M = make_mats(kind, B, H, W).to(DEV)
    out = warp_affine(x, M, dsize)
    out.backward(go)
    lhs = (out.detach().double() * go.double()).sum()
    rhs = (x.detach().double() * x.grad.double()).sum()
    assert float((lhs - rhs).abs()) <= 1e-6 * float(lhs.abs()), (float(lhs), float(rhs))


def test_deterministic_and_allowed_under_deterministic_algorithms():
    B, C, H, W, dsize = SHAPES['cfg2']
    g = torch.Generator().manual_seed(9)
    x = torch.randn(B, C, H, W, generator=g).to(DEV)
    go = torch.randn(B, C, *dsize, generator=g).to(DEV)
    M = bda_mats(B, H, W, seed=4).to(DEV)
    runs = []
    prev = torch.are_deterministic_algorithms_enabled()
    try:
        torch.use_deterministic_algorithms(True)
        for _ in range(2):
            xs = x.clone().requires_grad_(True)
            out = warp_affine(xs, M, dsize)
            out.backward(go)
            runs.append((out.detach().clone(), xs.grad.clone()))
    finally:
        torch.use_deterministic_algorithms(prev)
    assert torch.equal(runs[0][0], runs[1][0]) and torch.equal(runs[0][1], runs[1][1])


def test_nchw_and_channels_last_inputs_agree():
    B, C, H, W, dsize = SHAPES['resize']
    x = torch.randn(B, C, H, W, generator=torch.Generator().manual_seed(2)).to(DEV)
    M = bda_mats(B, H, W, seed=2).to(DEV)
    a = warp_affine(x, M, dsize)
    b = warp_affine(x.contiguous(memory_format=torch.channels_last), M, dsize)
    assert torch.equal(a, b)


# ---------------------------------------------------------------- the concat epilogue with the BDA warp
def _camera_case(B, seed=8, c2=64):
    cfg = CFG_2
    geom, vn_t = synthetic.camera_rig(cfg, B, device=DEV, yaw_jitter_deg=5.0, seed=seed)
    vn = tuple(int(v) for v in vn_t.tolist())
    depth, ctx, _ = synthetic.camera_features(cfg, B, device=DEV, seed=seed)
    X, Y, _ = vn
    g = torch.Generator().manual_seed(seed)
    other = torch.randn(B, c2, Y, X, generator=g).to(DEV)
    go = torch.rand(B, cfg.output_channels + c2, Y, X, generator=g).to(DEV).contiguous(memory_format=torch.channels_last)
    M = bda_mats(B, Y, X, seed=seed).to(DEV)
    return geom, vn, depth, ctx, other, go, M


def _leaves(*ts):
    return [t.clone().requires_grad_(True) for t in ts]


def _composite(depth, ctx, other, vn, plan, M, go):
    d, c, o = _leaves(depth, ctx, other)
    out = voxel_pooling_fused_concat(d, c, o, vn, plan, bda_affine=M)
    out.backward(go)
    return out.detach(), d.grad, c.grad, o.grad


def test_concat_with_bda_equals_the_composition_of_the_native_ops(monkeypatch):
    B = 4
    geom, vn, depth, ctx, other, go, M = _camera_case(B)
    X, Y, _ = vn
    plan = build_plan(geom, vn, frustum=tuple(geom.shape[1:5]))
    assert plan.mode == 'runs'
    fused = _composite(depth, ctx, other, vn, plan, M, go)
    assert fused[0].permute(0, 2, 3, 1).is_contiguous()
    d, c, o = _leaves(depth, ctx, other)
    ref = torch.cat([warp_affine(voxel_pooling_fused(None, d, c, vn, plan), M, (Y, X)), o], dim=1)
    ref.backward(go)
    assert torch.equal(fused[0], ref.detach())                   # same kernels, same order: bit-equal
    assert torch.equal(fused[1], d.grad) and torch.equal(fused[2], c.grad) and torch.equal(fused[3], o.grad)
    # NaN in every row of the scratch between pooling and warp: nothing but occupied rows is ever read
    monkeypatch.setattr(vp_mod, '_warp_scratch', lambda B_, Y_, X_, C_, dev: torch.full((B_, Y_, X_, C_), float('nan'), device=dev))
    poisoned = _composite(depth, ctx, other, vn, plan, M, go)
    for a, b in zip(poisoned, fused):
        assert torch.equal(a, b)
    # without a BDA matrix: today's output
    monkeypatch.undo()
    d, c, o = _leaves(depth, ctx, other)
    plain = voxel_pooling_fused_concat(d, c, o, vn, plan)
    assert torch.equal(plain, torch.cat([voxel_pooling_fused(None, depth, ctx, vn, plan), other], dim=1))


def test_concat_with_bda_against_the_fp64_oracle_chain():
    B = 1
    geom, vn, depth, ctx, other, go, M = _camera_case(B, seed=3)
    X, Y, _ = vn
    C = ctx.shape[1]
    plan = build_plan(geom, vn, frustum=tuple(geom.shape[1:5]))
    out, gd, gc, _ = _composite(depth, ctx, other, vn, plan, M, go)
    gcpu, dcpu, ccpu = geom.cpu(), depth.cpu(), ctx.cpu()
    pooled = vp.voxel_pooling_fused_ref(gcpu, dcpu, ccpu, vn, acc_dtype=torch.float64).requires_grad_(True)
    ref = wr.warp_affine_ref(pooled, M, (Y, X))
    g_cam = go[:, :C].cpu().double()
    ref.backward(g_cam)
    gd64, gc64 = vp.voxel_pooling_fused_grads_ref(gcpu, dcpu, ccpu, vn, pooled.grad)
    # error scale: the same chains on magnitudes, with the warp's unweighted tap sums
    pooled_abs = vp.voxel_pooling_fused_ref(gcpu, dcpu.abs(), ccpu.abs(), vn, acc_dtype=torch.float64)
    S = wr.tap_sum_ref(pooled_abs, M, (Y, X))
    a = torch.zeros_like(pooled_abs, requires_grad=True)
    (Sb,) = torch.autograd.grad(wr.tap_sum_ref(a, M, (Y, X)), a, g_cam.abs())
    gd_abs, gc_abs = vp.voxel_pooling_fused_grads_ref(gcpu, dcpu.abs(), ccpu.abs(), vn, Sb)
    _check('forward', out[:, :C].cpu(), ref.detach(), _bound(ref.detach(), S, Y, X))
    _check('grad depth', gd.cpu(), gd64, _bound(gd64, gd_abs, Y, X))
    _check('grad context', gc.cpu(), gc64, _bound(gc64, gc_abs, Y, X))


def test_concat_with_bda_replays_in_a_cuda_graph():
    B = 2
    geom, vn, depth, ctx, other, go, M = _camera_case(B, seed=5)
    fr = tuple(geom.shape[1:5])
    first = build_plan(geom, vn, frustum=fr)
    n = first.num_sorted
    eager = _composite(depth, ctx, other, vn, first, M, go)
    d, c, o = _leaves(depth, ctx, other)

    def step():
        plan = build_plan(geom, vn, frustum=fr, max_runs=n)
        out = voxel_pooling_fused_concat(d, c, o, vn, plan, bda_affine=M)
        return (out,) + torch.autograd.grad(out, (d, c, o), go)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        step()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        captured = step()
    for t in captured[:3]:                              # (the LiDAR gradient is a view of `go` itself)
        t.detach().fill_(float('nan'))
    graph.replay()
    torch.cuda.synchronize()
    for a, b in zip(captured, eager):
        assert torch.equal(a.detach(), b)

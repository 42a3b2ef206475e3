"""Fused pooling under autocast: fp32 depth (the softmax runs in fp32) with the fp16 / bf16 context slice of DepthNet's
output.  The contract is the call on ``context.float()`` (the upcast route): the output and ``grad_depth`` must equal it
bit for bit, and ``grad_context`` must equal its fp32 gradient rounded once to the context's dtype, in the context's
memory format.  CPU part: the argument errors of the two C entry points.  GPU part: ``torch.equal`` throughout."""

import pytest
import torch

from mm_training_b200 import _lib, build, synthetic
from mm_training_b200.configs import CFG_2
from mm_training_b200.ops.voxel_pooling import (LiftSplatGeometry, build_plan, voxel_pooling_fused,
                                                voxel_pooling_fused_concat, voxel_pooling_rig)
from mm_training_b200.ops.voxel_pooling.voxel_pooling import RUN_CHANNELS, _route, context_rows_nhwc
from oracle.warp_affine_ref import bda_matrices

DEV = 'cuda'
HALF = (torch.bfloat16, torch.float16)

# ---- CPU: argument errors come back as codes before any device work (fake pointers) --------------------------------
_P, _MISALIGNED = 0x10000, 0x10004
E_ARG, E_CHANNELS, E_ALIGN, E_DTYPE = -1, -3, -4, -5
_PARAMS = {
    'bevpool_fused_forward_runs_mixed': 'plan depth ctx cdtype flags out stride B N D H W C X Y rows cap ws stream',
    'bevpool_fused_backward_runs_mixed': 'plan grad stride depth ctx gdepth gctx nchw cdtype B N D H W C X Y stream',
}
_VALID = dict(plan=_P, depth=_P, ctx=_P, out=_P, grad=_P, gdepth=_P, gctx=_P, ws=_P, rows=_P, stream=None, cdtype=2,
              B=2, N=2, D=8, H=4, W=8, C=80, X=16, Y=16, cap=64, flags=0, stride=128, nchw=0)
_COMMON = [(dict(cdtype=3), E_DTYPE), (dict(cdtype=-1), E_DTYPE), (dict(plan=None), E_ARG), (dict(depth=None), E_ARG),
           (dict(ctx=None), E_ARG), (dict(N=0), E_ARG), (dict(C=84), E_CHANNELS), (dict(C=48), E_CHANNELS),
           (dict(ctx=_MISALIGNED), E_ALIGN), (dict(stride=76), E_ARG), (dict(stride=82), E_ARG)]
_ERRORS = {
    'bevpool_fused_forward_runs_mixed': _COMMON + [
        (dict(out=None), E_ARG), (dict(rows=None), E_ARG), (dict(ws=None), E_ARG), (dict(cap=0), E_ARG),
        (dict(stride=0), E_ARG), (dict(stride=-4), E_ARG), (dict(out=_MISALIGNED), E_ALIGN),
        (dict(flags=1, W=44), E_ALIGN), (dict(flags=3, W=44, cdtype=1), E_ALIGN), (dict(flags=1, W=6, cdtype=0), E_ALIGN)],
    'bevpool_fused_backward_runs_mixed': _COMMON + [
        (dict(grad=None), E_ARG), (dict(gdepth=None), E_ARG), (dict(gctx=None), E_ARG), (dict(stride=-4), E_ARG),
        (dict(gctx=_MISALIGNED), E_ALIGN), (dict(grad=_MISALIGNED), E_ALIGN), (dict(nchw=1, W=44), E_ALIGN),
        (dict(nchw=1, W=44, cdtype=1, stride=0), E_ALIGN), (dict(W=6), E_ALIGN), (dict(stride=0, W=6), E_ALIGN),
        (dict(depth=_MISALIGNED), E_ALIGN), (dict(gdepth=_MISALIGNED), E_ALIGN)],
}


@pytest.fixture(scope='module')
def L():
    build.build()
    return _lib.lib()


@pytest.mark.parametrize('name', sorted(_PARAMS))
def test_mixed_entry_point_argument_errors(L, name):
    assert name in _lib.EXPORTED_SYMBOLS and hasattr(L, name)
    params = _PARAMS[name].split()
    for change, code in _ERRORS[name]:
        args = dict(_VALID, **change)
        assert getattr(L, name)(*[args[p] for p in params]) == code, (name, change)


# ---- GPU ---------------------------------------------------------------------------------------------------------
def _geometry(seed, B, N, D, H, W, vn):
    """A level-camera-like geometry: the rows of an (image, bin, column) share a cell, except dropped rows and a few
    strays (the kernels' fast path with masks and their per-row path)."""
    g = torch.Generator().manual_seed(seed)
    X, Y, Z = vn
    x = torch.randint(-1, X + 1, (B, N, D, 1, W), generator=g).expand(B, N, D, H, W).clone()
    y = torch.randint(-1, Y + 1, (B, N, D, 1, W), generator=g).expand(B, N, D, H, W).clone()
    z = torch.where(torch.rand(B, N, D, H, W, generator=g) < 0.8, torch.randint(0, Z, (B, N, D, H, W), generator=g), -1)
    stray = torch.rand(B, N, D, H, W, generator=g) < 0.03
    x = torch.where(stray, torch.randint(0, X, (B, N, D, H, W), generator=g), x)
    return torch.stack([x, y, z], -1).int().contiguous().to(DEV)


def _inputs(seed, B, N, D, H, W, C, vn, dtype):
    """depth: softmax probabilities; context: U(-0.5, 0.5) with fp16 subnormals and values near 65504 mixed in;
    grad_out: U(0, 1) with a few cells large enough to overflow an fp16 context gradient."""
    g = torch.Generator().manual_seed(seed)
    X, Y, _ = vn
    depth = torch.rand(B * N, D, H, W, generator=g).softmax(1)
    ctx = torch.rand(B * N, C, H, W, generator=g) - 0.5
    pick = torch.rand(B * N, C, H, W, generator=g)
    sign = torch.where(torch.rand(B * N, C, H, W, generator=g) < 0.5, -1.0, 1.0)
    ctx = torch.where(pick < 0.01, sign * 6e-8, ctx)                  # fp16 subnormals (bf16: normal)
    ctx = torch.where((pick >= 0.01) & (pick < 0.015), sign * 65504.0, ctx)
    ctx = torch.where((pick >= 0.015) & (pick < 0.02), sign * 1e-41, ctx)   # fp32 / bf16 subnormals, fp16 zero
    go = torch.rand(B, C, Y, X, generator=g)
    go = torch.where(torch.rand(B, 1, Y, X, generator=g) < 0.05, go * 3e6, go)
    return depth.to(DEV), ctx.to(DEV, dtype), go.to(DEV)


def _run(fn, depth, ctx, go, upcast):
    """(out, grad_depth, grad_context) of fn(depth, ctx) with the gradients as the op returns them (autograd.grad
    applies no layout contract); ``upcast``: the reference route, fn(depth, ctx.float())."""
    d, c = depth.clone().requires_grad_(True), ctx.detach().clone(memory_format=torch.preserve_format).requires_grad_(True)
    out = fn(d, c.float() if upcast else c)
    gd, gc = torch.autograd.grad(out, (d, c), go)
    return out.detach(), gd, gc


def _assert_same(mixed, upcast, ctx):
    out, gd, gc = mixed
    out_u, gd_u, gc_u = upcast
    assert out.dtype == torch.float32 and torch.equal(out, out_u)
    assert gd.dtype == torch.float32 and torch.equal(gd, gd_u)
    assert gc.dtype == ctx.dtype and gc.stride() == ctx.stride() and gc_u.stride() == ctx.stride()
    assert torch.equal(gc, gc_u)


def _expected_route(ctx, W):
    return 'nchw' if ctx.is_contiguous() and W % 8 == 0 else 'rows'


@pytest.mark.gpu
@pytest.mark.parametrize('W', [16, 44])
@pytest.mark.parametrize('layout', ['nchw', 'channels_last'])
@pytest.mark.parametrize('dtype', HALF, ids=['bf16', 'fp16'])
@pytest.mark.parametrize('C', RUN_CHANNELS)
def test_mixed_equals_upcast_route(C, dtype, layout, W):
    B, N, D, H, vn = 2, 2, 24, 20, (24, 20, 3)
    geom = _geometry(C + W, B, N, D, H, W, vn)
    depth, ctx, go = _inputs(C * W, B, N, D, H, W, C, vn, dtype)
    if layout == 'channels_last':
        ctx = ctx.contiguous(memory_format=torch.channels_last)
    plan = build_plan(geom, vn, frustum=(N, D, H, W))
    assert plan.mode == 'runs' and _route('runs', ctx, depth) == _expected_route(ctx, W)
    fn = lambda d, c: voxel_pooling_fused(None, d, c, vn, plan)
    mixed = _run(fn, depth, ctx, go, False)
    _assert_same(mixed, _run(fn, depth, ctx, go, True), ctx)
    assert torch.equal(mixed[0], _run(fn, depth, ctx, go, False)[0])           # bit-stable
    if dtype == torch.float16:
        assert bool(torch.isinf(mixed[2]).any()) and bool(torch.isfinite(mixed[2]).any())   # overflow rounds to inf


@pytest.mark.gpu
@pytest.mark.parametrize('dtype', HALF, ids=['bf16', 'fp16'])
def test_context_rows_of_a_half_nchw_context(dtype):
    """The rows route of an NCHW half context goes through the library's transpose, in the context's dtype."""
    ctx = (torch.rand(3, 80, 16, 44, device=DEV) - 0.5).to(dtype)
    rows = context_rows_nhwc(ctx)
    assert rows.dtype == dtype and rows.is_contiguous() and torch.equal(rows, ctx.permute(0, 2, 3, 1))
    cl = ctx.contiguous(memory_format=torch.channels_last)
    assert context_rows_nhwc(cl).data_ptr() == cl.data_ptr()


def _rig(B, seed=3):
    lsg = LiftSplatGeometry.from_config(CFG_2, DEV)
    s2e, intrin = synthetic.camera_rig_mats(CFG_2, B, DEV, yaw_jitter_deg=4.0, seed=seed)
    return lsg, s2e, intrin


def _depth_feature(B, seed, dtype=torch.bfloat16):
    cfg = CFG_2
    g = torch.Generator().manual_seed(seed)
    h, w = cfg.feat_hw
    feat = torch.randn(B * cfg.num_cams, cfg.depth_bins + cfg.output_channels + 8, h, w, generator=g) * 2
    return feat.to(DEV, dtype)


@pytest.mark.gpu
@pytest.mark.parametrize('op', ['rig', 'concat_bda', 'concat_resize'])
def test_autocast_chain_from_depth_feature(op):
    """DepthNet's bf16 output under autocast: softmax of the first D channels (fp32), the context slice (bf16),
    pooled; the gradient reaching depth_feature equals that of the upcast route."""
    cfg, B = CFG_2, 2
    D, C = cfg.depth_bins, cfg.output_channels
    lsg, s2e, intrin = _rig(B)
    feat = _depth_feature(B, 7)
    X, Y, _ = lsg.voxel_num
    g = torch.Generator().manual_seed(11)
    plan = lsg.plan(s2e, intrin)
    assert plan.mode == 'runs'
    if op == 'rig':
        go = torch.rand(B, C, Y, X, generator=g).to(DEV)
        pool = lambda d, c: voxel_pooling_rig(lsg, s2e, intrin, d, c)
    else:
        other = torch.randn(B, 16, Y // 2, X // 2, generator=g).to(DEV) if op == 'concat_resize' else \
            torch.randn(B, 16, Y, X, generator=g).to(DEV)
        go = torch.rand(B, C + 16, Y, X, generator=g).to(DEV).contiguous(memory_format=torch.channels_last)
        M = bda_matrices(B, Y, X, seed=5).to(DEV) if op == 'concat_bda' else None
        resize = 'nearest' if op == 'concat_resize' else None
        pool = lambda d, c: voxel_pooling_fused_concat(d, c, other, lsg.voxel_num, plan, bda_affine=M, resize_other=resize)

    def step(upcast):
        f = feat.clone().requires_grad_(True)
        with torch.autocast('cuda', dtype=torch.bfloat16):
            depth = f[:, :D].softmax(1)
            ctx = f[:, D:D + C]
            assert depth.dtype == torch.float32 and ctx.dtype == torch.bfloat16
            out = pool(depth, ctx.float() if upcast else ctx)
        (gf,) = torch.autograd.grad(out, (f,), go)
        return out.detach(), gf

    out, gf = step(False)
    out_u, gf_u = step(True)
    assert out.dtype == torch.float32 and torch.equal(out, out_u)
    assert gf.dtype == torch.bfloat16 and torch.equal(gf, gf_u)
    assert bool(gf[:, D:D + C].ne(0).any())


@pytest.mark.gpu
@pytest.mark.parametrize('overlap', ['0', '1'])
@pytest.mark.parametrize('W', [16, 44])
def test_cold_call_from_geom_xyz(monkeypatch, W, overlap):
    """No plan given: the op builds a run plan from the 6-d geom_xyz (the cold path; with BEVPOOL_COLD_OVERLAP=1 the
    output is zero-filled behind the plan build and the kernels write occupied cells only)."""
    monkeypatch.setenv('BEVPOOL_COLD_OVERLAP', overlap)
    B, N, D, H, C, vn = 2, 2, 24, 20, 80, (24, 20, 3)
    geom = _geometry(W, B, N, D, H, W, vn)
    depth, ctx, go = _inputs(W + 1, B, N, D, H, W, C, vn, torch.bfloat16)
    fn = lambda d, c: voxel_pooling_fused(geom, d, c, vn)
    _assert_same(_run(fn, depth, ctx, go, False), _run(fn, depth, ctx, go, True), ctx)


@pytest.mark.gpu
@pytest.mark.parametrize('dtype', HALF, ids=['bf16', 'fp16'])
def test_graph_capture_with_max_runs(dtype):
    """Forward + backward of a mixed call captured in a CUDA graph (plan rebuilt with a max_runs hint inside the
    graph): every replay gives the eager bits."""
    B, N, D, H, W, C, vn = 2, 2, 24, 20, 16, 64, (24, 20, 3)
    geom = _geometry(5, B, N, D, H, W, vn)
    depth, ctx, go = _inputs(6, B, N, D, H, W, C, vn, dtype)
    fr = (N, D, H, W)
    n = build_plan(geom, vn, frustum=fr).num_sorted
    d, c = depth.clone().requires_grad_(True), ctx.clone().requires_grad_(True)

    def chain():
        out = voxel_pooling_fused(None, d, c, vn, build_plan(geom, vn, frustum=fr, max_runs=n))
        return (out, *torch.autograd.grad(out, (d, c), go))
    eager = [t.detach().clone() for t in chain()]
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        chain()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        captured = chain()
    for _ in range(2):
        for t in captured:
            t.detach().fill_(float('nan'))
        graph.replay()
        torch.cuda.synchronize()
        assert all(torch.equal(a.detach(), b) for a, b in zip(captured, eager))
    _assert_same(eager, _run(lambda a, b: voxel_pooling_fused(None, a, b, vn, build_plan(geom, vn, frustum=fr)),
                             depth, ctx, go, True), ctx)


@pytest.mark.gpu
@pytest.mark.parametrize('case', ['point_plan', 'channels_48', 'disable_g8', 'width_6'])
def test_mixed_calls_off_the_run_kernels_pool_the_upcast(monkeypatch, case):
    """Mixed calls no run kernel takes do not assert: they pool context.float(), so they equal the upcast route."""
    B, N, D, H, W, C, vn = 2, 2, 24, 20, 16, 80, (24, 20, 3)
    if case == 'channels_48':
        C = 48
    if case == 'width_6':
        W = 6
    if case == 'disable_g8':
        monkeypatch.setenv('BEVPOOL_DISABLE_G8', '1')
    geom = _geometry(9, B, N, D, H, W, vn)
    depth, ctx, go = _inputs(10, B, N, D, H, W, C, vn, torch.bfloat16)
    if case == 'point_plan':
        plan = build_plan(geom, vn)
        fn = lambda d, c: voxel_pooling_fused(None, d, c, vn, plan)
    elif case == 'width_6':
        plan = build_plan(geom, vn, frustum=(N, D, H, W))
        assert plan.mode == 'runs' and _route('runs', ctx, depth) == 'points'
        fn = lambda d, c: voxel_pooling_fused(None, d, c, vn, plan)
    else:
        fn = lambda d, c: voxel_pooling_fused(geom, d, c, vn)
    _assert_same(_run(fn, depth, ctx, go, False), _run(fn, depth, ctx, go, True), ctx)

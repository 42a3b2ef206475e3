"""The fused camera + LiDAR BEV concat in bf16 / fp16 (``voxel_pooling_fused_concat(..., dtype=...)``).

Contract: the output equals the float32 call's output ``.to(dtype)`` bit for bit, and the gradients of ``depth``,
``context`` and ``other_bev`` for a 16-bit gradient ``g`` equal those of the float32 call fed ``g.float()`` bit for bit,
in the same dtypes and memory formats.  CPU part: argument errors of the new C entry points and the ``dtype`` check.
GPU part: ``torch.equal`` throughout (NaN positions compared as positions, where an fp16 overflow meets a zero)."""

import importlib
import itertools
import os
import random
import subprocess
import sys

import pytest
import torch

from mm_training_b200 import _lib, build
from mm_training_b200.ops.voxel_pooling import build_plan, voxel_pooling_fused_concat
from oracle.warp_affine_ref import bda_matrices

vp_mod = importlib.import_module('mm_training_b200.ops.voxel_pooling.voxel_pooling')

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHILD = os.environ.get('BEVPOOL_CONCAT_HALF_CHILD') == '1'
DEV = 'cuda'
HALF = (torch.bfloat16, torch.float16)

# ---- CPU: argument errors come back as codes before any device work (fake pointers) --------------------------------
_P, _MISALIGNED = 0x10000, 0x10004
E_ARG, E_CHANNELS, E_ALIGN, E_DTYPE = -1, -3, -4, -5
F32, F16, BF16 = 0, 1, 2
_PARAMS = {
    'bevpool_fused_forward_runs_into16': 'plan depth ctx cdtype flags out stride odtype B N D H W C X Y rows cap ws stream',
    'bevpool_warp_affine_forward16': 'theta src sstride out ostride odtype cs B C Hs Ws Hd Wd stream',
    'bevpool_warp_affine_backward16': 'theta grad gstride gdtype gsrc sstride cs B C Hs Ws Hd Wd stream',
    'bevpool_resize_nearest_into16': 'src sdtype nchw B C Hs Ws Hd Wd out stride odtype stream',
    'bevpool_resize_nearest_backward_from16': 'grad gstride gdtype gsrc sdtype nchw B C Hs Ws Hd Wd stream',
    'bevpool_grad_rows_widen': 'cs grad gstride gdtype rows B C X Y stream',
}
_VALID = dict(plan=_P, depth=_P, ctx=_P, out=_P, rows=_P, ws=_P, theta=_P, src=_P, grad=_P, gsrc=_P, cs=None, stream=None,
              cdtype=F32, odtype=BF16, gdtype=F16, sdtype=F32, flags=0, nchw=1, stride=96, sstride=80, ostride=96,
              gstride=96, B=2, N=2, D=8, H=4, W=8, C=80, X=16, Y=16, cap=64, Hs=8, Ws=8, Hd=8, Wd=8)
_ERRORS = {
    'bevpool_fused_forward_runs_into16': [
        (dict(odtype=F32), E_DTYPE), (dict(odtype=3), E_DTYPE), (dict(cdtype=3), E_DTYPE), (dict(plan=None), E_ARG),
        (dict(out=None), E_ARG), (dict(rows=None), E_ARG), (dict(cap=0), E_ARG), (dict(stride=0), E_ARG),
        (dict(stride=82), E_ARG), (dict(stride=76), E_ARG), (dict(N=0), E_ARG), (dict(C=84), E_CHANNELS),
        (dict(C=48), E_CHANNELS), (dict(out=_MISALIGNED), E_ALIGN), (dict(ctx=_MISALIGNED), E_ALIGN),
        (dict(flags=1, W=6), E_ALIGN)],
    'bevpool_warp_affine_forward16': [
        (dict(odtype=F32), E_DTYPE), (dict(odtype=7), E_DTYPE), (dict(theta=None), E_ARG), (dict(out=None), E_ARG),
        (dict(sstride=76), E_ARG), (dict(ostride=94), E_ARG), (dict(Hs=1), E_ARG), (dict(C=82), E_CHANNELS),
        (dict(out=_MISALIGNED), E_ALIGN), (dict(src=_MISALIGNED), E_ALIGN)],
    'bevpool_warp_affine_backward16': [
        (dict(gdtype=F32), E_DTYPE), (dict(gdtype=-1), E_DTYPE), (dict(theta=None), E_ARG), (dict(grad=None), E_ARG),
        (dict(gstride=78), E_ARG), (dict(sstride=0), E_ARG), (dict(Wd=1), E_ARG), (dict(C=82), E_CHANNELS),
        (dict(grad=_MISALIGNED), E_ALIGN), (dict(gsrc=_MISALIGNED), E_ALIGN)],
    'bevpool_resize_nearest_into16': [
        (dict(odtype=F32), E_DTYPE), (dict(odtype=5), E_DTYPE), (dict(sdtype=3), E_DTYPE), (dict(src=None), E_ARG),
        (dict(out=None), E_ARG), (dict(stride=94), E_ARG), (dict(Hs=0), E_ARG), (dict(C=6), E_CHANNELS),
        (dict(out=_MISALIGNED), E_ALIGN), (dict(nchw=0, src=_MISALIGNED), E_ALIGN)],
    'bevpool_resize_nearest_backward_from16': [
        (dict(gdtype=F32), E_DTYPE), (dict(gdtype=4), E_DTYPE), (dict(sdtype=3), E_DTYPE), (dict(grad=None), E_ARG),
        (dict(gsrc=None), E_ARG), (dict(gstride=90), E_ARG), (dict(B=0), E_ARG), (dict(C=6), E_CHANNELS),
        (dict(grad=_MISALIGNED), E_ALIGN), (dict(nchw=0, gsrc=_MISALIGNED), E_ALIGN)],
    'bevpool_grad_rows_widen': [
        (dict(cs=None), E_ARG), (dict(grad=None), E_ARG), (dict(rows=None), E_ARG), (dict(X=0), E_ARG),
        (dict(gstride=78), E_ARG), (dict(gstride=76), E_ARG), (dict(gdtype=F32), E_DTYPE), (dict(gdtype=3), E_DTYPE),
        (dict(C=6), E_CHANNELS), (dict(C=0), E_CHANNELS), (dict(grad=_MISALIGNED), E_ALIGN),
        (dict(rows=_MISALIGNED), E_ALIGN)],
}


@pytest.fixture(scope='module')
def L():
    build.build()
    return _lib.lib()


def _declared():
    import re
    text = open(os.path.join(ROOT, 'include', 'bevpool_sm100.h')).read()
    return set(re.findall(r'\b(bevpool_[a-z0-9_]+)\s*\(', re.sub(r'/\*.*?\*/', '', text, flags=re.S)))


@pytest.mark.parametrize('name', sorted(_PARAMS))
def test_half_entry_point_argument_errors(L, name):
    assert name in _lib.EXPORTED_SYMBOLS and name in _declared() and hasattr(L, name)
    params = _PARAMS[name].split()
    for change, code in _ERRORS[name]:
        args = dict(_VALID, cs=_P if name == 'bevpool_grad_rows_widen' else None)
        args.update(change)
        assert getattr(L, name)(*[args[p] for p in params]) == code, (name, change)


@pytest.mark.parametrize('dtype', [torch.float64, torch.int32, torch.float8_e4m3fn])
def test_other_dtypes_raise(dtype):
    z = torch.zeros(1)
    with pytest.raises(ValueError, match='dtype'):
        voxel_pooling_fused_concat(z, z, z, (4, 4, 1), None, dtype=dtype)


# ---- GPU ---------------------------------------------------------------------------------------------------------
B, N, D, H, C = 2, 2, 24, 20, 80
VN = (32, 24, 3)                                    # X, Y, Z: even, so that a 2x up-sampled LiDAR BEV exists
C2 = 16
RESIZE = {'none': None, 'up2': (VN[1] // 2, VN[0] // 2), 'identity': (VN[1], VN[0]), 'down4': (4 * VN[1], 4 * VN[0])}


def _geometry(seed, W):
    """Level-camera-like geometry (as test_gpu_pool_mixed.py): the rows of an (image, bin, column) share a cell, except
    dropped rows and a few strays (the fast path with masks and the per-row path of stage A)."""
    g = torch.Generator().manual_seed(seed)
    X, Y, Z = VN
    x = torch.randint(-1, X + 1, (B, N, D, 1, W), generator=g).expand(B, N, D, H, W).clone()
    y = torch.randint(-1, Y + 1, (B, N, D, 1, W), generator=g).expand(B, N, D, H, W).clone()
    z = torch.where(torch.rand(B, N, D, H, W, generator=g) < 0.8, torch.randint(0, Z, (B, N, D, H, W), generator=g), -1)
    stray = torch.rand(B, N, D, H, W, generator=g) < 0.03
    x = torch.where(stray, torch.randint(0, X, (B, N, D, H, W), generator=g), x)
    return torch.stack([x, y, z], -1).int().contiguous().to(DEV)


def _inputs(seed, W, ctx_dtype, ctx_layout, other_dtype, other_layout, other_hw, out_dtype, grad_layout, c2=C2):
    """depth: softmax probabilities; context: U(-0.5, 0.5) with fp16 subnormals, +-65504 and fp32 subnormals mixed in
    (test_gpu_pool_mixed.py's recipe); LiDAR BEV: N(0, 1) with 1e5 (beyond fp16) mixed in; gradient: U(0, 1) with 5 % of the cells
    scaled by 3e6 (beyond fp16: +-inf in an fp16 gradient), in out_dtype."""
    g = torch.Generator().manual_seed(seed)
    X, Y, _ = VN
    depth = torch.rand(B * N, D, H, W, generator=g).softmax(1)
    ctx = torch.rand(B * N, C, H, W, generator=g) - 0.5
    pick = torch.rand(B * N, C, H, W, generator=g)
    sign = torch.where(torch.rand(B * N, C, H, W, generator=g) < 0.5, -1.0, 1.0)
    ctx = torch.where(pick < 0.01, sign * 6e-8, ctx)
    ctx = torch.where((pick >= 0.01) & (pick < 0.015), sign * 65504.0, ctx)
    ctx = torch.where((pick >= 0.015) & (pick < 0.02), sign * 1e-41, ctx)
    other = torch.randn(B, c2, *other_hw, generator=g)
    other = torch.where(torch.rand(B, c2, *other_hw, generator=g) < 0.01, 1e5, other)
    go = torch.rand(B, C + c2, Y, X, generator=g)
    go = torch.where(torch.rand(B, 1, Y, X, generator=g) < 0.05, go * 3e6, go)
    ctx = ctx.to(DEV, ctx_dtype)
    if ctx_layout == 'channels_last':
        ctx = ctx.contiguous(memory_format=torch.channels_last)
    other = other.to(DEV, other_dtype)
    if other_layout == 'channels_last':
        other = other.contiguous(memory_format=torch.channels_last)
    go = go.to(DEV, out_dtype)
    if grad_layout == 'channels_last':
        go = go.contiguous(memory_format=torch.channels_last)
    return depth.to(DEV), ctx, other, go


def _run(depth, ctx, other, plan, M, resize, dtype, go):
    """(out, grad_depth, grad_context, grad_other) of one call; the float32 call (dtype None) is fed go.float()."""
    d = depth.clone().requires_grad_(True)
    c = ctx.detach().clone(memory_format=torch.preserve_format).requires_grad_(True)
    o = other.detach().clone(memory_format=torch.preserve_format).requires_grad_(True)
    out = voxel_pooling_fused_concat(d, c, o, VN, plan, bda_affine=M, resize_other=resize, dtype=dtype)
    grads = torch.autograd.grad(out, (d, c, o), go if dtype is not None else go.float())
    return (out.detach(), *grads)


def _layout(t):
    return 'channels_last' if t.stride(1) == 1 else ('nchw' if t.stride(3) == 1 else tuple(t.stride()))


def _same(a, b, what):
    """Bit-for-bit equal values (torch.equal), NaN where the other has NaN (an fp16 inf gradient times a zero)."""
    assert a.dtype == b.dtype and a.shape == b.shape, (what, a.dtype, b.dtype)
    na, nb = a.isnan(), b.isnan()
    assert torch.equal(na, nb), what
    assert torch.equal(a.masked_fill(na, 0), b.masked_fill(nb, 0)), what


def _check(half, ref, dtype, ctx, other, native=True):
    out, gd, gc, go_ = half
    out_r, gd_r, gc_r, go_r = ref
    assert out.dtype == dtype and out.shape == out_r.shape
    if native:
        assert out.permute(0, 2, 3, 1).is_contiguous()              # a channels-last view of one (B, Y, X, C + C2) buffer
    _same(out, out_r.to(dtype), 'out')
    _same(gd, gd_r, 'grad_depth')
    _same(gc, gc_r, 'grad_context')
    _same(go_, go_r, 'grad_other')
    assert gc.dtype == ctx.dtype and _layout(gc) == _layout(gc_r)
    assert go_.dtype == other.dtype and _layout(go_) == _layout(go_r)


def _cases(n, seed):
    """A seeded subset of out dtype x context dtype x BDA x resize x LiDAR dtype x LiDAR layout (+ context and gradient
    layouts) in which every value of every axis appears."""
    axes = [('bf16', 'fp16'), ('fp32', 'bf16', 'fp16'), ('nobda', 'bda'), tuple(RESIZE), ('fp32', 'bf16'),
            ('nchw', 'channels_last'), ('nchw', 'channels_last'), ('channels_last', 'nchw')]
    full = list(itertools.product(*axes))
    picked = random.Random(seed).sample(full, n)
    for i, values in enumerate(axes):
        assert {p[i] for p in picked} == set(values)
    return ['-'.join(p) for p in picked]


_DT = {'fp32': torch.float32, 'bf16': torch.bfloat16, 'fp16': torch.float16}


def _matrix_case(case, W, seed):
    out_s, ctx_s, bda_s, resize_s, other_s, other_l, ctx_l, grad_l = case.split('-')
    dtype = _DT[out_s]
    geom = _geometry(seed, W)
    plan = build_plan(geom, VN, frustum=(N, D, H, W))
    assert plan.mode == 'runs'
    X, Y, _ = VN
    hw = RESIZE[resize_s] or (Y, X)
    depth, ctx, other, go = _inputs(seed + 1, W, _DT[ctx_s], ctx_l, _DT[other_s], other_l, hw, dtype, grad_l)
    M = bda_matrices(B, Y, X, seed=seed).to(DEV) if bda_s == 'bda' else None
    resize = None if RESIZE[resize_s] is None else 'nearest'
    return depth, ctx, other, go, plan, M, resize, dtype


@pytest.mark.gpu
@pytest.mark.parametrize('W', [44, 16])
@pytest.mark.parametrize('case', _cases(40, 7))
def test_core_matrix_equals_the_fp32_call_cast(case, W):
    """W = 44 (CFG-2 width: 16-bit contexts take pixel rows) and W = 16 (an NCHW 16-bit context is read through its
    tensor map)."""
    depth, ctx, other, go, plan, M, resize, dtype = _matrix_case(case, W, seed=len(case) + W)
    ref = _run(depth, ctx, other, plan, M, resize, None, go)
    half = _run(depth, ctx, other, plan, M, resize, dtype, go)
    _check(half, ref, dtype, ctx, other)
    assert torch.equal(half[0], _run(depth, ctx, other, plan, M, resize, dtype, go)[0])       # bit-stable


@pytest.mark.gpu
@pytest.mark.parametrize('ctx_s', ['fp32', 'fp16'])
@pytest.mark.parametrize('bda', [False, True])
def test_core_fp16_overflow(bda, ctx_s):
    """fp16 output of contexts near 65504 (depth weights scaled by 64) and LiDAR values of 1e5: cells beyond the fp16
    range round to +-inf in both halves, as `.to(float16)` does; fp16 gradients of 3e6 are +-inf, and the gradients
    still equal the float32 call's on g.float()."""
    case = f'fp16-{ctx_s}-{"bda" if bda else "nobda"}-none-fp32-nchw-nchw-channels_last'
    depth, ctx, other, go, plan, M, resize, dtype = _matrix_case(case, 44, seed=3)
    depth = depth * 64
    ref = _run(depth, ctx, other, plan, M, resize, None, go)
    half = _run(depth, ctx, other, plan, M, resize, dtype, go)
    _check(half, ref, dtype, ctx, other)
    for part in (half[0][:, :C], half[0][:, C:]):
        assert bool(part.isinf().any()) and bool(part.isfinite().any())
    assert bool(go.isinf().any())


@pytest.mark.gpu
@pytest.mark.parametrize('bda', [False, True])
def test_no_uninitialised_reads(monkeypatch, bda):
    """The warp scratch and the widened gradient rows are NaN-filled before use: only occupied rows are read."""
    case = f'bf16-bf16-{"bda" if bda else "nobda"}-down4-bf16-channels_last-channels_last-channels_last'
    depth, ctx, other, go, plan, M, resize, dtype = _matrix_case(case, 44, seed=11)
    clean = _run(depth, ctx, other, plan, M, resize, dtype, go)
    calls = []

    def poisoned(B_, Y_, X_, C_, dev):
        calls.append(1)
        return torch.full((B_, Y_, X_, C_), float('nan'), device=dev)
    monkeypatch.setattr(vp_mod, '_warp_scratch', poisoned)
    dirty = _run(depth, ctx, other, plan, M, resize, dtype, go)
    assert len(calls) == (2 if bda else 1)
    for a, b in zip(clean, dirty):
        assert torch.equal(a, b)


@pytest.mark.gpu
@pytest.mark.parametrize('dtype', HALF, ids=['bf16', 'fp16'])
def test_no_host_sync(dtype):
    """Python-int voxel_num and a max_runs plan: forward + backward with BDA and a resize never synchronise."""
    W = 44
    geom = _geometry(5, W)
    fr = (N, D, H, W)
    n = build_plan(geom, VN, frustum=fr).num_sorted
    plan = build_plan(geom, VN, frustum=fr, max_runs=n)
    X, Y, _ = VN
    depth, ctx, other, go = _inputs(6, W, torch.bfloat16, 'nchw', torch.bfloat16, 'nchw', (Y // 2, X // 2), dtype,
                                    'channels_last')
    M = bda_matrices(B, Y, X, seed=5).to(DEV)
    d, c, o = depth.clone().requires_grad_(True), ctx.clone().requires_grad_(True), other.clone().requires_grad_(True)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode('error')
    try:
        out = voxel_pooling_fused_concat(d, c, o, list(VN), plan, bda_affine=M, resize_other='nearest', dtype=dtype)
        grads = torch.autograd.grad(out, (d, c, o), go)
    finally:
        torch.cuda.set_sync_debug_mode('default')
    ref = _run(depth, ctx, other, build_plan(geom, VN, frustum=fr), M, 'nearest', None, go)
    _check((out.detach(), *grads), ref, dtype, ctx, other)


@pytest.mark.gpu
@pytest.mark.parametrize('dtype', HALF, ids=['bf16', 'fp16'])
def test_identity_lidar_gradient_is_a_view(dtype):
    depth, ctx, other, go, plan, M, resize, _ = _matrix_case(
        f'{"bf16" if dtype == torch.bfloat16 else "fp16"}-fp32-nobda-none-fp32-nchw-nchw-channels_last', 44, seed=2)
    other = other.to(dtype)
    o = other.clone().requires_grad_(True)
    out = voxel_pooling_fused_concat(depth, ctx, o, VN, plan, dtype=dtype)
    (g,) = torch.autograd.grad(out, (o,), go)
    assert g.dtype == dtype and g.data_ptr() == go[:, C:].data_ptr()


@pytest.mark.gpu
@pytest.mark.parametrize('case', ['point_plan', 'c2_6'])
@pytest.mark.parametrize('dtype', HALF, ids=['bf16', 'fp16'])
def test_fallback_equals_the_fp32_call_cast(case, dtype):
    """No native path (point plan, C2 % 4 != 0): the stock ops, cast with .to(dtype)."""
    W = 44
    geom = _geometry(13, W)
    c2 = 6 if case == 'c2_6' else C2
    X, Y, _ = VN
    depth, ctx, other, go = _inputs(14, W, torch.float32, 'nchw', torch.float32, 'nchw', (Y, X), dtype, 'channels_last',
                                    c2=c2)
    plan = build_plan(geom, VN) if case == 'point_plan' else build_plan(geom, VN, frustum=(N, D, H, W))
    ref = _run(depth, ctx, other, plan, None, None, None, go)
    half = _run(depth, ctx, other, plan, None, None, dtype, go)
    _check(half, ref, dtype, ctx, other, native=False)


@pytest.mark.gpu
def test_float32_dtype_is_the_default_path():
    depth, ctx, other, go, plan, M, resize, _ = _matrix_case('bf16-fp32-bda-up2-fp32-nchw-nchw-channels_last', 44, 4)
    a = _run(depth, ctx, other, plan, M, resize, None, go)
    b = _run(depth, ctx, other, plan, M, resize, torch.float32, go.float())
    for x, y in zip(a, b):
        assert x.dtype == y.dtype and torch.equal(x, y)


# ---- the knob matrix: the `core` tests in a fresh process per knob (each is read once per process) ----------------
KNOBS = ['BEVPOOL_RUN_FILL=0', 'BEVPOOL_RUN_HINTS=0', 'BEVPOOL_RUN_CPSB=1']


@pytest.mark.gpu
@pytest.mark.skipif(CHILD, reason='inside a knob child')
@pytest.mark.parametrize('knob', KNOBS)
def test_knob_matrix(knob):
    key, value = knob.split('=')
    env = dict(os.environ, BEVPOOL_CONCAT_HALF_CHILD='1', **{key: value})
    res = subprocess.run([sys.executable, '-m', 'pytest', os.path.abspath(__file__), '-q', '-m', 'gpu', '-k', 'core',
                          '-p', 'no:cacheprovider'], cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout[-4000:] + res.stderr[-2000:]
    assert ' passed' in res.stdout and ' skipped' not in res.stdout, res.stdout[-2000:]

"""Every fp32 pooling route pinned BIT FOR BIT to the integer oracle (oracle/pool_exact_ref.py) on dyadic inputs, at
production shapes and under every tuning knob, plus a rigorous per-element bound on general inputs.

On dyadic inputs whose per-element sum of |terms| is below 2^24 units every float32 evaluation is exact in any order,
so the kernels must return the integer result exactly (``torch.equal``): a dropped, duplicated or misplaced term fails,
however small it is, whatever the summation order.  Each case proves which kernels it ran from a torch.profiler trace
(CUDA activity).  ``test_knob_matrix`` re-runs the ``core`` cases of this file in a child process per knob setting (the
knobs are read once per process).  The bound tests check every route against the fp64 oracle within
``sum_bound(n, sum |terms|)`` per element, valid for any summation tree."""
import json
import math
import os
import re
import subprocess
import sys
import tempfile

import pytest
import torch
from torch.profiler import ProfilerActivity, profile

from mm_training_b200 import synthetic
from mm_training_b200.configs import CFG_2, CFG_AIM
from mm_training_b200.ops.voxel_pooling import (LiftSplatGeometry, build_plan, rig_variant, voxel_pooling,
                                                voxel_pooling_fused, voxel_pooling_fused_concat,
                                                voxel_pooling_fused_logits, voxel_pooling_rig)
from mm_training_b200.ops.voxel_pooling.voxel_pooling import RUN_CHANNELS, VoxelPoolingFused
from oracle import pool_exact_ref as px
from oracle.depth_softmax_ref import sum_bound

pytestmark = pytest.mark.gpu
DEV = 'cuda'
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHILD = os.environ.get('BEVPOOL_EXACT_CHILD') == '1'
_env = lambda k, d: os.environ.get(k, d) or d


# ---------------------------------------------------------------- kernel traces
def _trace(fn):
    """fn() under torch.profiler (CUDA activity); returns (result, [(kernel name, grid)]).  No trace is a failure."""
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        r = fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, 'trace.json')
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)['traceEvents']
    events = sorted((e for e in events if e.get('cat') == 'kernel'), key=lambda e: e['ts'])
    ks = [(e['name'], tuple(e.get('args', {}).get('grid', ()))) for e in events]
    assert ks, 'the profiler recorded no CUDA kernel'
    return r, ks


def _targ(s):
    s = re.sub(r'^\(\w+\)', '', s.strip())
    return {'true': 1, 'false': 0}.get(s, int(s) if re.fullmatch(r'-?\d+', s) else s)


def _launches(ks, kernel):
    """[(template arguments, grid)] of every launch of ``kernel`` (bools as 0 / 1)."""
    out = []
    for name, grid in ks:
        m = re.search(r'\b' + kernel + r'(?:<([^<>]*)>)?\(', name)
        if m:
            out.append(([_targ(t) for t in m.group(1).split(',')] if m.group(1) else [], grid))
    return out


def _ran(ks, kernel, **at):
    """``kernel`` ran, with template argument i == v for every ``a<i>=v`` given."""
    ls = _launches(ks, kernel)
    assert ls, f'{kernel} did not run; kernels: {sorted({n[:80] for n, _ in ks})}'
    for key, v in at.items():
        assert all(t[int(key[1:])] == v for t, _ in ls), (kernel, key, v, ls)
    return ls


def _not_ran(ks, kernel):
    assert not _launches(ks, kernel), f'{kernel} ran'


def _bw_runs(ks, nchw_ctx, W, C, strided=False):
    """Backward kernel of a run plan: the column kernel (W % 4 == 0; with BEVPOOL_BW_KERNEL=1 only where nothing else
    can run), else the tile kernel (C <= 96, scalar variant when W % 4 != 0) or the generic one."""
    if W % 4 == 0 and (_env('BEVPOOL_BW_KERNEL', '2') == '2' or nchw_ctx or strided):
        _ran(ks, 'fused_backward_col_kernel', a1=int(nchw_ctx))
        _not_ran(ks, 'fused_backward_tile_kernel')
    elif C <= 96:
        _ran(ks, 'fused_backward_tile_kernel', a1=int(W % 4 == 0))
        _not_ran(ks, 'fused_backward_col_kernel')
    else:
        _ran(ks, 'fused_backward_kernel')


def _grad_rows(ks, X, go_nchw):
    if not go_nchw:                                     # the permuted NHWC view is read in place
        _not_ran(ks, 'grad_rows_tma_kernel')
        _not_ran(ks, 'grad_rows_kernel')
    elif X % 4 == 0 and _env('BEVPOOL_GRAD_ROWS_TMA', '1') != '0':
        _ran(ks, 'grad_rows_tma_kernel')
    else:
        _ran(ks, 'grad_rows_kernel')


def _stage_a(B, N, D, H, W):
    """Grid of every stage-A launch and the depth chunks a CTA walks, as fused_forward_runs_impl picks them."""
    fpc = int(_env('BEVPOOL_RUN_CHUNK', '0'))
    fpc = B if fpc <= 0 or fpc > B else fpc
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    grids, chunks = [], []
    for b0 in range(0, B, fpc):
        tiles = min(fpc, B - b0) * N * math.ceil(W / 4) * math.ceil(H / 16)
        ds = int(_env('BEVPOOL_RUN_DSPLIT', '0'))
        if ds <= 0:
            ds = min(max(math.ceil(16 * sms / tiles), 1), math.ceil(D / 16))
        dpc = math.ceil(math.ceil(D / ds) / 16) * 16
        grids.append(tiles * math.ceil(D / dpc))
        chunks.append(dpc // 16)
    return grids, chunks


def _fw_runs(ks, nchw_ctx, B, N, D, H, W, logits=False):
    ls = _ran(ks, 'frustum_reduce_kernel', a1=int(nchw_ctx), a2=int(logits))
    grids, _ = _stage_a(B, N, D, H, W)
    assert [g[0] for _, g in ls] == grids, (ls, grids)
    _ran(ks, 'pool_forward_share_kernel', a1=0, a3=1)
    _ran(ks, 'pool_forward_fixup_kernel')


# ---------------------------------------------------------------- exact inputs and comparison
RANGES = [(15, 15, 15), (7, 7, 7), (3, 3, 3), (1, 1, 1)]


def _exact(geom, vn, N, C, seed):
    """Dyadic (depth, context, grad_out) on the device and the oracle's (out (B, Y, X, C), grad_depth, grad_context)
    as float32; the widest value ranges for which every element meets the precondition."""
    B, _, D, H, W, _ = geom.shape
    cell = px.cells(geom.to(DEV), vn)
    for amax, bmax, gmax in RANGES:
        a, b, g = px.dyadic_inputs(seed, B, N, D, H, W, C, vn, amax, bmax, gmax, device=DEV)
        out, mag, _ = px.forward_exact(cell, a, b, vn)
        if px.holds(mag):
            break
    gd, gdm, gc, gcm = px.grads_exact(cell, a, b, g)
    assert px.holds(mag) and px.holds(gdm) and px.holds(gcm)
    return ((px.to_float(a), px.to_float(b), px.to_float(g)),
            (px.to_float(out, 8), px.to_float(gd, 8), px.to_float(gc, 8)))


def _equal(got, want, what):
    for name, x, y in zip(('out', 'grad_depth', 'grad_context', 'grad_extra')[:len(got)], got, want):
        assert x.shape == y.shape, (what, name, x.shape, y.shape)
        if not torch.equal(x, y):
            bad = (x != y).nonzero()
            raise AssertionError(f'{what}: {name} differs at {bad.shape[0]} of {x.numel()} elements, first {bad[0].tolist()}: '
                                 f'{float(x[tuple(bad[0])])} vs {float(y[tuple(bad[0])])}')


def _layout(t, channels_last):
    return t.contiguous(memory_format=torch.channels_last) if channels_last else t.contiguous()


def _fused(geom, depth, ctx, go, vn, plan=None, go_nchw=True):
    """voxel_pooling_fused forward + backward under the profiler: ((out (B, Y, X, C), grad_depth, grad_context), trace)."""
    d, c = depth.detach().clone().requires_grad_(True), ctx.detach().clone().requires_grad_(True)
    g = go.contiguous() if go_nchw else go.permute(0, 2, 3, 1).contiguous().permute(0, 3, 1, 2)

    def step():
        out = voxel_pooling_fused(geom, d, c, vn, plan)
        out.backward(g)
        return out.detach().permute(0, 2, 3, 1)
    out, ks = _trace(step)
    return (out, d.grad, c.grad), ks


# ---------------------------------------------------------------- run plans
RUN_CASES = [  # B, N, D, H, W, C, vn, coherent
    (2, 2, 64, 16, 8, 80, (32, 16, 1), True),       # 4 depth chunks: the stage-A ring wraps when one CTA walks them all
    (1, 3, 17, 44, 12, 32, (40, 12, 1), True),      # H = 44: ragged last row block
    (2, 1, 15, 17, 4, 64, (8, 8, 2), False),        # Z = 2, a one-row block, every point its own run
    (10, 1, 16, 15, 4, 96, (16, 16, 1), True),      # more frames than one stage-A / B chunk of BEVPOOL_RUN_CHUNK
    (1, 2, 112, 1, 4, 128, (64, 8, 1), True),       # H = 1
    (1, 1, 1, 16, 44, 80, (64, 64, 1), False),      # D = 1
    (1, 2, 409, 16, 80, 80, (128, 32, 1), True),    # D = 409, W = 80
]
RAGGED_CASES = [  # W % 4 != 0: NCHW context through the transpose and pixel rows
    (1, 2, 17, 16, 5, 80, (24, 12, 1), True),
    (2, 1, 33, 15, 3, 32, (16, 8, 1), True),
    (1, 1, 16, 17, 1, 64, (8, 8, 1), False),
    (1, 1, 64, 44, 5, 128, (32, 16, 1), True),      # C = 128: generic backward
    (1, 2, 112, 16, 5, 96, (40, 16, 1), False),
]
LAYOUTS = ['nchw', 'nchw-grad-nhwc', 'channels_last']
assert {c[5] for c in RUN_CASES} == set(RUN_CHANNELS)


def _check_runs(case, layout, seed=11):
    B, N, D, H, W, C, vn, coherent = case
    geom = px.frustum_geom(seed, B, N, D, H, W, vn, coherent).to(DEV)
    (depth, ctx, go), want = _exact(geom, vn, N, C, seed)
    cl = layout == 'channels_last'
    got, ks = _fused(geom, depth, _layout(ctx, cl), go, vn, go_nchw=layout != 'nchw-grad-nhwc')
    _equal(got, want, (case, layout))
    direct = W % 4 == 0 and not cl and _env('BEVPOOL_NCHW_DIRECT', '1') != '0'
    _fw_runs(ks, direct, B, N, D, H, W)
    if not direct and not cl:
        _ran(ks, 'transpose_kernel')
    _bw_runs(ks, direct, W, C)
    _grad_rows(ks, vn[0], layout != 'nchw-grad-nhwc')


@pytest.mark.parametrize('layout', LAYOUTS)
@pytest.mark.parametrize('case', RUN_CASES + RAGGED_CASES)
def test_run_plan_routes_are_exact(case, layout):
    _check_runs(case, layout)


@pytest.mark.parametrize('layout', LAYOUTS)
@pytest.mark.parametrize('case', [RUN_CASES[0], RUN_CASES[3], RAGGED_CASES[0], RAGGED_CASES[3]])
def test_core_run_plan(case, layout):
    _check_runs(case, layout)


def test_core_nchw_direct_off(monkeypatch):
    monkeypatch.setenv('BEVPOOL_NCHW_DIRECT', '0')          # W % 4 == 0, but the transpose + pixel-row route
    _check_runs(RUN_CASES[0], 'nchw')


def test_core_big_cells_and_an_empty_sample():
    """4 cells of ~1000 runs each (the plan's queued-cell kernel; each cell spans many even-share slices) and a second
    sample whose points are all dropped."""
    B, N, D, H, W, C, vn = 2, 2, 30, 8, 8, 32, (2, 2, 1)
    g = torch.Generator().manual_seed(5)
    geom = torch.stack([torch.randint(0, 2, (B, N, D, H, W), generator=g), torch.randint(0, 2, (B, N, D, H, W), generator=g),
                        torch.randint(-1, 1, (B, N, D, H, W), generator=g)], -1).int()
    geom[1, ..., 2] = -1
    geom = geom.contiguous().to(DEV)
    (depth, ctx, go), want = _exact(geom, vn, N, C, 12)
    plan = build_plan(geom, vn, frustum=(N, D, H, W))
    cs = plan.cell_start.cpu()
    assert int((cs[1:] - cs[:-1]).max()) > 64 and int(cs[-1] - cs[4]) == 0
    for cl in (False, True):
        got, ks = _fused(None, depth, _layout(ctx, cl), go, vn, plan=plan)
        _equal(got, want, ('big cells', cl))
        _fw_runs(ks, not cl, B, N, D, H, W)
    assert float(want[0][1].abs().sum()) == 0.0


def test_core_knob_launches():
    """The stage-A grid and launch count follow BEVPOOL_RUN_DSPLIT / BEVPOOL_RUN_CHUNK (10 frames, D = 64)."""
    case = (10, 1, 64, 16, 8, 80, (16, 16, 1), True)
    _check_runs(case, 'nchw')
    grids, chunks = _stage_a(10, 1, 64, 16, 8)
    fpc = int(_env('BEVPOOL_RUN_CHUNK', '0'))
    assert len(grids) == (math.ceil(10 / fpc) if fpc > 0 else 1)
    if int(_env('BEVPOOL_RUN_DSPLIT', '0')) == 1:
        assert chunks == [4] * len(chunks)                  # every CTA walks all 4 chunks: the 3-stage ring wraps


# ---------------------------------------------------------------- production shapes
@pytest.mark.parametrize('channels_last', [False, True])
@pytest.mark.parametrize('cfg,B', [(CFG_2, 32), (CFG_AIM, 4)], ids=['cfg2-b32', 'aim-b4'])
def test_production_shapes_are_exact(cfg, B, channels_last):
    geom, vn = synthetic.camera_rig(cfg, B, device=DEV, yaw_jitter_deg=5.0, seed=3)
    vn = tuple(int(v) for v in vn.tolist())
    N, D, (H, W), C = cfg.num_cams, cfg.depth_bins, cfg.feat_hw, cfg.output_channels
    _, chunks = _stage_a(B, N, D, H, W)
    if not CHILD:
        assert min(chunks) >= 4, chunks                     # the bench's launch shape reuses the cp.async ring
    (depth, ctx, go), want = _exact(geom, vn, N, C, 21)
    got, ks = _fused(geom, depth, _layout(ctx, channels_last), go, vn)
    _equal(got, want, (cfg.name, B, channels_last))
    _fw_runs(ks, not channels_last, B, N, D, H, W)
    _bw_runs(ks, not channels_last, W, C)


# ---------------------------------------------------------------- point plans and the generic kernels
POINT_CASES = [  # B, N, D, H, W, C, vn, coherent
    (2, 2, 17, 16, 8, 32, (24, 12, 1), True),
    (1, 3, 15, 17, 5, 64, (16, 16, 2), False),
    (2, 1, 16, 15, 4, 80, (32, 8, 1), True),
    (1, 2, 33, 44, 3, 96, (20, 20, 1), True),
    (1, 1, 64, 16, 4, 128, (12, 12, 1), False),
]


def _check_points(case, channels_last, generic=False):
    B, N, D, H, W, C, vn, coherent = case
    geom = px.frustum_geom(13, B, N, D, H, W, vn, coherent).to(DEV)
    (depth, ctx, go), want = _exact(geom, vn, N, C, 14)
    plan = build_plan(geom, vn)
    assert plan.mode == 'points'
    got, ks = _fused(None, depth, _layout(ctx, channels_last), go, vn, plan=plan)
    _equal(got, want, (case, channels_last, generic))
    _not_ran(ks, 'frustum_reduce_kernel')
    if generic:
        _ran(ks, 'pool_forward_kernel', a2=1)
        _ran(ks, 'fused_backward_kernel')
        return
    _ran(ks, 'pool_forward_share_kernel', a1=1, a3=0)
    _ran(ks, 'pool_forward_fixup_kernel')
    if C <= 96:
        _ran(ks, 'fused_backward_tile_kernel', a1=int(W % 4 == 0))
    else:
        _ran(ks, 'fused_backward_kernel')


@pytest.mark.parametrize('channels_last', [False, True])
@pytest.mark.parametrize('case', POINT_CASES)
def test_point_plan_routes_are_exact(case, channels_last):
    _check_points(case, channels_last)


def test_core_point_plan():
    _check_points(POINT_CASES[2], False)
    _check_points(POINT_CASES[4], True)


@pytest.mark.parametrize('C', [4, 8, 132, 260, 512])
def test_generic_channel_counts_are_exact(C):
    _check_points((1, 2, 17, 5, 6, C, (12, 10, 1), True), C % 8 == 0, generic=True)


def test_core_disable_g8(monkeypatch):
    monkeypatch.setenv('BEVPOOL_DISABLE_G8', '1')
    _check_points(POINT_CASES[2], False, generic=True)
    B, N, D, H, W, C, vn, coherent = RUN_CASES[0]           # a 6-d geom_xyz builds a point plan without the g8 kernels
    geom = px.frustum_geom(11, B, N, D, H, W, vn, coherent).to(DEV)
    (depth, ctx, go), want = _exact(geom, vn, N, C, 11)
    got, ks = _fused(geom, depth, ctx, go, vn)
    _equal(got, want, 'disable g8')
    _ran(ks, 'pool_forward_kernel')
    _ran(ks, 'fused_backward_kernel')
    _not_ran(ks, 'frustum_reduce_kernel')


# ---------------------------------------------------------------- concat epilogue, cold forward, logits, rig, host
@pytest.mark.parametrize('channels_last', [False, True])
def test_core_concat_epilogue(channels_last):
    B, N, D, H, W, C, vn, coherent = RUN_CASES[0]
    geom = px.frustum_geom(15, B, N, D, H, W, vn, coherent).to(DEV)
    (depth, ctx, go), want = _exact(geom, vn, N, C, 15)
    X, Y, _ = vn
    gen = torch.Generator().manual_seed(16)
    other = torch.randn(B, 4, Y // 2 + 1, X + 3, generator=gen).to(DEV)
    g_cat = torch.cat([go, torch.randn(B, 4, Y, X, generator=gen).to(DEV)], 1).contiguous(memory_format=torch.channels_last)
    plan = build_plan(geom, vn, frustum=(N, D, H, W))
    d, c = depth.clone().requires_grad_(True), _layout(ctx, channels_last).requires_grad_(True)

    def step():
        out = voxel_pooling_fused_concat(d, c, other, vn, plan, resize_other='nearest')
        out.backward(g_cat)
        return out.detach()[:, :C].permute(0, 2, 3, 1)
    out, ks = _trace(step)
    _equal((out, d.grad, c.grad), want, ('concat', channels_last))
    _fw_runs(ks, not channels_last, B, N, D, H, W)
    _bw_runs(ks, not channels_last, W, C, strided=True)


def test_core_cold_forward_prezeroed(monkeypatch):
    monkeypatch.setenv('BEVPOOL_COLD_OVERLAP', '1')
    B, N, D, H, W, C, vn, coherent = RUN_CASES[0]
    geom = px.frustum_geom(17, B, N, D, H, W, vn, coherent).to(DEV)
    (depth, ctx, go), want = _exact(geom, vn, N, C, 17)
    got, ks = _fused(geom, depth, ctx, go, vn)
    _equal(got, want, 'cold')
    _fw_runs(ks, True, B, N, D, H, W)


def test_plan_builder_forward_runs_once():
    """A plan builder handed to the op (the camera rig's route) that returns a point plan: the pooling forward runs once,
    with the kernels and grids of the call that is given that plan."""
    B, N, D, H, W, C, vn, coherent = RUN_CASES[0]                 # fp32 NCHW context, C = 80, W % 4 == 0
    geom = px.frustum_geom(27, B, N, D, H, W, vn, coherent).to(DEV)
    (depth, ctx, _), want = _exact(geom, vn, N, C, 27)
    forward = re.compile(r'\b(pool_forward_\w+|frustum_reduce_kernel)\b')
    runs = []
    for plan, make_plan in ((None, lambda: build_plan(geom, vn)), (build_plan(geom, vn), None)):
        out, ks = _trace(lambda: VoxelPoolingFused.apply(None, depth, ctx, vn, plan, make_plan, B))
        _equal((out.permute(0, 2, 3, 1),), want[:1], ('plan builder', plan is None))
        runs.append([k for k in ks if forward.search(k[0])])
    assert len(_launches(runs[0], 'pool_forward_share_kernel')) == 1, runs[0]
    assert runs[0] == runs[1]


@pytest.mark.parametrize('extra', [0, 3])
@pytest.mark.parametrize('case', [(2, 2, 64, 16, 8, 80, (32, 16, 1)), (1, 2, 17, 44, 12, 32, (40, 12, 1))])
def test_core_logits_route(case, extra):
    """Masked logits (p = 1 / k exactly), the context at channel offset D, ``extra`` further channels."""
    B, N, D, H, W, C, vn = case
    geom = px.frustum_geom(18, B, N, D, H, W, vn, True).to(DEV)
    cell = px.cells(geom, vn)
    logits, a = px.masked_logits(19, B * N, D, H, W, device=DEV)
    _, b, g = px.dyadic_inputs(20, B, N, D, H, W, C, vn, device=DEV)
    out, mag, _ = px.forward_exact(cell, a, b, vn)
    gd, gdm, gc, gcm = px.grads_exact(cell, a, b, g)
    gl, glm = px.logit_grad_exact(a, gd)
    assert all(px.holds(m) for m in (mag, gdm, gcm, glm))
    feat = px.depth_feature(logits, px.to_float(b), extra, seed=21).requires_grad_(True)
    plan = build_plan(geom, vn, frustum=(N, D, H, W))

    def step():
        o = voxel_pooling_fused_logits(feat, D, C, vn, plan)
        o.backward(px.to_float(g))
        return o.detach().permute(0, 2, 3, 1)
    o, ks = _trace(step)
    grad = feat.grad
    _equal((o, grad[:, :D], grad[:, D:D + C], grad[:, D + C:]),
           (px.to_float(out, 8), px.to_float(gl, 16), px.to_float(gc, 8), torch.zeros_like(grad[:, D + C:])), ('logits', case))
    _ran(ks, 'depth_stats_kernel')
    _fw_runs(ks, True, B, N, D, H, W, logits=True)
    _bw_runs(ks, True, W, C)


@pytest.mark.parametrize('tilted', [False, True])
def test_rig_plan_is_exact(tilted):
    if rig_variant(DEV) is None:
        pytest.skip('no accumulation order of the rig plan kernel is proven on this device')
    from mm_training_b200.ops.voxel_pooling.rig import _random_rigs
    cfg, B = CFG_2, 3
    lsg = LiftSplatGeometry.from_config(cfg, DEV)
    if tilted:
        s2e, k = _random_rigs(B, cfg.num_cams, torch.Generator().manual_seed(9))
    else:
        s2e, k = synthetic.camera_rig_mats(cfg, B, yaw_jitter_deg=5.0, seed=9)
    s2e, k = s2e.to(DEV), k.to(DEV)
    geom = lsg.geom_xyz(s2e, k)
    vn = lsg.voxel_num
    (depth, ctx, go), want = _exact(geom, vn, cfg.num_cams, cfg.output_channels, 22)
    got, ks = _fused(None, depth, ctx, go, vn, plan=lsg.plan(s2e, k))
    _equal(got, want, ('rig', tilted))
    _fw_runs(ks, True, B, cfg.num_cams, cfg.depth_bins, *cfg.feat_hw)
    d, c = depth.clone().requires_grad_(True), ctx.clone().requires_grad_(True)
    o = voxel_pooling_rig(lsg, s2e, k, d, c)
    o.backward(go)
    _equal((o.detach().permute(0, 2, 3, 1), d.grad, c.grad), want, ('voxel_pooling_rig', tilted))


def test_host_pipeline_is_exact():
    from mm_training_b200.ops.voxel_pooling.host_pipeline import HostPoolingPipeline
    cfg, B = CFG_2, 5                                        # chunks of 2 frames: a ragged last chunk
    geom, vn = synthetic.camera_rig(cfg, B, device=DEV, yaw_jitter_deg=5.0, seed=23)
    vn = tuple(int(v) for v in vn.tolist())
    N, C = cfg.num_cams, cfg.output_channels
    (depth, ctx, go), (out, gd, gc) = _exact(geom, vn, N, C, 23)
    pin = lambda t: t.cpu().contiguous().pin_memory()
    pipe = HostPoolingPipeline(N, geom.shape, depth.shape, ctx.shape, vn, chunk_frames=2, device=DEV)
    X, Y, _ = vn
    h_out = torch.empty(B, C, Y, X).pin_memory()
    h_gd, h_gc = torch.empty(depth.shape).pin_memory(), torch.empty(ctx.shape).pin_memory()
    pipe.run(pin(geom), pin(depth), pin(ctx), pin(go), h_out, h_gd, h_gc)
    _equal((h_out.permute(0, 2, 3, 1), h_gd, h_gc), (out.cpu(), gd.cpu(), gc.cpu()), 'host pipeline')


# ---------------------------------------------------------------- the drop-in op
@pytest.mark.parametrize('C', [80, 12])
def test_core_dropin(C):
    B, P, vn = 2, 5000, (40, 24, 2)
    g = torch.Generator().manual_seed(24)
    geom = torch.stack([torch.randint(-2, 42, (B, P), generator=g), torch.randint(-1, 25, (B, P), generator=g),
                        torch.randint(-1, 3, (B, P), generator=g)], -1).int()
    geom[:, :1500] = torch.tensor([3, 4, 0], dtype=torch.int32)          # a hot cell
    geom = geom.contiguous().to(DEV)
    cell = px.cells(geom, vn)
    f = px._ints(g, (B, P, C), 1, 225, True, DEV)
    gi = px._ints(g, (B, C, vn[1], vn[0]), 0, 15, True, DEV)
    out, mag = px.dropin_forward_exact(cell, f, vn)
    assert px.holds(mag)
    feats = px.to_float(f, 8).requires_grad_(True)

    def step():
        o = voxel_pooling(geom, feats, vn)
        o.backward(px.to_float(gi))
        return o.detach().permute(0, 2, 3, 1)
    o, ks = _trace(step)
    _equal((o, feats.grad), (px.to_float(out, 8), px.to_float(px.dropin_backward_exact(cell, gi))), ('drop-in', C))
    if C % 16 == 0:
        _ran(ks, 'pool_forward_share_kernel', a1=0, a3=0)
    else:
        _ran(ks, 'pool_forward_kernel', a2=0)
    _ran(ks, 'pool_backward_kernel')


# ---------------------------------------------------------------- rigorous bound on general inputs
def _wide(seed, B, N, D, H, W, C, vn):
    """Wide dynamic range: per-bin depth scales, per-pixel context scales and per-cell grad_out scales of 2^U(-30, 30)."""
    X, Y, _ = vn
    g = torch.Generator().manual_seed(seed)
    sc = lambda *s: torch.exp2(torch.rand(*s, generator=g) * 60 - 30)
    depth = torch.rand(B * N, D, H, W, generator=g) * sc(B * N, D, 1, 1)
    ctx = (torch.rand(B * N, C, H, W, generator=g) - 0.5) * sc(B * N, 1, H, W)
    go = (torch.rand(B, C, Y, X, generator=g) - 0.5) * sc(B, 1, Y, X)
    return depth.to(DEV), ctx.to(DEV), go.to(DEV)


def _within(x, ref, n, mag, what):
    err = (x.double() - ref).abs()
    bound = sum_bound(n, mag)
    assert bool((err <= bound).all()), (what, float((err - bound).max()))


@pytest.mark.parametrize('route', ['nchw', 'channels_last', 'ragged', 'points', 'generic'])
def test_bound_on_wide_range_inputs(route):
    C = 132 if route == 'generic' else 80
    W = 5 if route == 'ragged' else 8
    B, N, D, H, vn = 2, 2, 40, 17, (16, 12, 1)
    geom = px.frustum_geom(25, B, N, D, H, W, vn, True).to(DEV)
    depth, ctx, go = _wide(26, B, N, D, H, W, C, vn)
    cell = px.cells(geom, vn)
    ref, mag, terms = px.forward_exact(cell, depth.double(), ctx.double(), vn)
    gd, gdm, gc, gcm = px.grads_exact(cell, depth.double(), ctx.double(), go.double())
    plan = build_plan(geom, vn) if route in ('points', 'generic') else None
    (out, d, c), ks = _fused(None if plan is not None else geom, depth, _layout(ctx, route == 'channels_last'), go, vn, plan=plan)
    _ran(ks, 'frustum_reduce_kernel' if plan is None else ('pool_forward_kernel' if route == 'generic' else 'pool_forward_share_kernel'))
    _within(out, ref, terms[..., None] + 1, mag, (route, 'out'))
    _within(d, gd, C + 1, gdm, (route, 'grad_depth'))
    _within(c, gc, D + 1, gcm, (route, 'grad_context'))


# ---------------------------------------------------------------- the knob matrix
KNOBS = ['BEVPOOL_RUN_DSPLIT=1', 'BEVPOOL_RUN_DSPLIT=3', 'BEVPOOL_RUN_CHUNK=1', 'BEVPOOL_RUN_CHUNK=3', 'BEVPOOL_RUN_FILL=0',
         'BEVPOOL_RUN_CPSB=1', 'BEVPOOL_RUN_HINTS=0', 'BEVPOOL_BW_KERNEL=1', 'BEVPOOL_BW_OCC=3', 'BEVPOOL_BW_STATIC=0',
         'BEVPOOL_GRAD_ROWS_TMA=0', 'BEVPOOL_FW_CPS=2', 'BEVPOOL_FW_U=2', 'BEVPOOL_PDL=0', 'BEVPOOL_PDL_FWD=1']


@pytest.mark.skipif(CHILD, reason='inside a knob child')
@pytest.mark.parametrize('knob', KNOBS)
def test_knob_matrix(knob):
    """The core cases of this file in a fresh process with one knob set (each knob is read once per process)."""
    key, value = knob.split('=')
    env = dict(os.environ, BEVPOOL_EXACT_CHILD='1', **{key: value})
    res = subprocess.run([sys.executable, '-m', 'pytest', os.path.abspath(__file__), '-q', '-m', 'gpu', '-k', 'core',
                          '-p', 'no:cacheprovider'], cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-4000:] + res.stderr[-2000:]
    assert ' passed' in res.stdout and ' skipped' not in res.stdout, res.stdout[-2000:]

"""GPU parity tests of the pooling path: CUDA kernels (through the python ops, which call the
C ABI) against the CPU oracle, the committed golden fixture and the reference's own CUDA kernel
(oracle/_ref).  Integer results must match bit-exactly.  fp32 forward sums of the generic kernels
are bit-identical to the sequential oracle by construction (same visiting order, no FMA
contraction); the fast (g8) forward cuts a cell's points at fixed, plan-determined positions and
combines the partial sums in a fixed order, so it is bit-stable run to run and held to rtol 1e-5
against the fp64 oracle with an atol that scales with the magnitude of the summed terms, as are
the gradients of the fused op (SURVEY.md section 7, hard part 3).  fp16 / bf16 forward sums are the fp32 oracle
rounded once, bit for bit, and their gradients lie in the rounding bracket of the fp64 result
(tests/test_gpu_pool_half.py covers more shapes and edge values)."""
import os

import numpy as np
import pytest
import torch

from mm_training_b200 import synthetic
from mm_training_b200.configs import CFG_2, CFG_AIM, sweep_grid_config
from mm_training_b200.ops.voxel_pooling import build_plan, voxel_pooling, voxel_pooling_fused
from oracle import ref_cuda_op
from oracle import voxel_pool_ref as vp
from oracle.depth_softmax_ref import in_bracket, round_bracket, sum_bound

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True, params=['g8', 'generic'])
def kernel_path(request, monkeypatch):
    """Every test runs twice: with the fp32 8-lanes-per-row fast path (default) and with the
    generic float4-per-lane kernels forced (the library reads BEVPOOL_DISABLE_G8 per call)."""
    monkeypatch.setenv('BEVPOOL_DISABLE_G8', '1' if request.param == 'generic' else '0')
    return request.param

GOLDEN = os.path.join(os.path.dirname(__file__), 'golden')
DEV = 'cuda'
G8_CHANNELS = (32, 64, 80, 96, 128)


def _assert_forward(out, ref32, ref64, abs64, exact):
    """``exact``: same bits as the sequential fp32 oracle.  Otherwise rtol 1e-5 against the fp64
    oracle plus 1e-6 of the per-cell sum of magnitudes (a few ulps of the largest partial sum)."""
    out = out.detach().cpu()
    if exact:
        assert torch.equal(out, ref32)
    else:
        err = (out.double() - ref64).abs()
        assert bool((err <= 1e-5 * ref64.abs() + 1e-6 * abs64 + 1e-30).all()), float(err.max())
        assert bool((out[abs64 == 0] == 0).all())              # empty cells are exact zeros


def _check_dropin_forward(out, geom, feats, vn, kernel_path):
    C = feats.shape[-1]
    exact = kernel_path == 'generic' or C not in G8_CHANNELS or feats.dtype != torch.float32
    _assert_forward(out, vp.voxel_pooling_ref(geom, feats, vn),
                    vp.voxel_pooling_ref(geom, feats, vn, acc_dtype=torch.float64),
                    vp.voxel_pooling_ref(geom, feats.abs(), vn, acc_dtype=torch.float64), exact)


def _rand_case(seed, B, Np, C, vn, lo=-3, hi_pad=3, dtype=torch.float32):
    g = torch.Generator().manual_seed(seed)
    X, Y, Z = vn
    geom = torch.stack([torch.randint(lo, X + hi_pad, (B, Np), generator=g),
                        torch.randint(lo, Y + hi_pad, (B, Np), generator=g),
                        torch.randint(-1, Z + 1, (B, Np), generator=g)], -1).int()
    feats = (torch.rand(B, Np, C, generator=g) - 0.5).to(dtype)
    return geom, feats


# ---------------------------------------------------------------- reference's own KAT
def test_reference_unit_test_recipe(kernel_path):
    # test/test_ops/test_voxel_pooling.py:15-37, verbatim recipe and tolerance
    geom_xyz, features = vp.reference_test_inputs()
    gold = vp.python_loop_golden(geom_xyz, features, (128, 128, 1))
    out = voxel_pooling(geom_xyz.cuda().int(), features.cuda(),
                        torch.tensor([128, 128, 1], dtype=torch.int, device='cuda'))
    assert out.shape == (2, 80, 128, 128)
    assert torch.allclose(gold.cuda(), out, rtol=1e-3)
    _check_dropin_forward(out, geom_xyz.int(), features, (128, 128, 1), kernel_path)
    fx = np.load(os.path.join(GOLDEN, 'voxel_pool_reftest.npz'))
    rows = out.permute(0, 2, 3, 1).reshape(-1, 80)[torch.from_numpy(fx['probe_cells']).cuda()]
    if kernel_path == 'generic':                          # stronger: same order, same bits
        assert torch.equal(gold.cuda(), out)
        assert np.array_equal(rows.cpu().numpy(), fx['probe_rows'])
    else:
        assert np.allclose(rows.cpu().numpy(), fx['probe_rows'], rtol=1e-5, atol=2e-6)


def test_against_reference_cuda_kernel():
    if not ref_cuda_op.available():
        pytest.skip('oracle/_ref not built: needs a checkout of the reference (make -C oracle ref REF=<checkout>)')
    geom_xyz, features = vp.reference_test_inputs()
    g, f = geom_xyz.cuda().int(), features.cuda()
    ref_out, ref_pos = ref_cuda_op.ref_forward_with_pos_memo(g, f, [128, 128, 1])
    plan = build_plan(g, [128, 128, 1])
    assert torch.equal(plan.pos_memo(), ref_pos)          # integer indices: bit-exact
    out = voxel_pooling(g, f, [128, 128, 1], plan)
    assert torch.allclose(ref_out, out, rtol=1e-3)
    assert torch.allclose(ref_out, out, rtol=1e-5, atol=2e-6)
    # backward against the reference autograd wrapper
    f1 = f.clone().requires_grad_(True)
    f2 = f.clone().requires_grad_(True)
    go = torch.rand(2, 80, 128, 128, device=DEV)
    ref_cuda_op.ref_voxel_pooling(g, f1, [128, 128, 1]).backward(go)
    voxel_pooling(g, f2, [128, 128, 1]).backward(go)
    assert torch.equal(f1.grad, f2.grad)


# ---------------------------------------------------------------- plan (integer work)
@pytest.mark.parametrize('B,Np,vn', [(1, 1, (1, 1, 1)), (2, 5000, (16, 8, 2)), (3, 4097, (128, 128, 1)),
                                      (2, 30000, (512, 64, 1)), (1, 70000, (2048, 1024, 1)),
                                      (5, 2048, (37, 29, 3))])
def test_plan_is_a_stable_sort_by_cell(B, Np, vn):
    geom, _ = _rand_case(1, B, Np, 4, vn)
    plan = build_plan(geom.cuda(), vn)
    kept, lin, pos = vp.cell_index_ref(geom, vn)
    X, Y, Z = vn
    cop = plan.cell_of_point.cpu()
    exp_cell = torch.where(kept, (lin - torch.arange(B).view(B, 1) * X * Y), torch.tensor(-1)).int()
    assert torch.equal(cop, exp_cell)
    assert torch.equal(plan.pos_memo().cpu(), pos)
    counts = torch.bincount(lin[kept], minlength=B * X * Y)
    cs = plan.cell_start.cpu().long()
    assert torch.equal(cs[1:] - cs[:-1], counts) and int(cs[0]) == 0
    ids = plan.sorted_ids.cpu().long()
    gid = torch.arange(B * Np).view(B, Np)
    exp_ids = gid[kept][torch.sort(lin[kept], stable=True).indices]
    assert torch.equal(ids, exp_ids)                       # grouped by cell, ascending inside


def test_plan_all_dropped_and_all_in_one_cell():
    geom = torch.full((2, 3000, 3), -5, dtype=torch.int32)
    plan = build_plan(geom.cuda(), (8, 8, 1))
    assert int(plan.cell_start[-1]) == 0 and bool((plan.cell_of_point == -1).all())
    out = voxel_pooling(geom.cuda(), torch.ones(2, 3000, 8, device=DEV), (8, 8, 1))
    assert float(out.abs().sum()) == 0.0
    geom = torch.zeros((2, 5000, 3), dtype=torch.int32)
    geom[..., 0] = 3
    geom[..., 1] = 2
    feats = torch.rand(2, 5000, 8) - 0.5
    out = voxel_pooling(geom.cuda(), feats.cuda(), (8, 8, 1))
    assert torch.equal(out.cpu(), vp.voxel_pooling_ref(geom, feats, (8, 8, 1)))


# ---------------------------------------------------------------- drop-in op
@pytest.mark.parametrize('B,Np,C,vn', [(2, 6000, 80, (128, 128, 1)), (1, 777, 4, (5, 7, 2)),
                                        (3, 10000, 128, (64, 32, 1)), (2, 3000, 132, (16, 16, 1)),
                                        (1, 2500, 260, (16, 8, 1)), (4, 20000, 64, (512, 64, 1))])
def test_dropin_forward_backward_fp32(B, Np, C, vn, kernel_path):
    geom, feats = _rand_case(2, B, Np, C, vn)
    X, Y, Z = vn
    f = feats.cuda().requires_grad_(True)
    out = voxel_pooling(geom.cuda(), f, torch.tensor(vn, device=DEV))
    ref = vp.voxel_pooling_ref(geom, feats, vn)
    assert out.shape == ref.shape == (B, C, Y, X)
    assert out.permute(0, 2, 3, 1).is_contiguous()         # permuted view like voxel_pooling.py:55
    _check_dropin_forward(out, geom, feats, vn, kernel_path)
    go = torch.rand(B, C, Y, X)
    out.backward(go.cuda())                                # NCHW-contiguous grad -> transpose path
    gref = vp.voxel_pooling_backward_ref(geom, go, vn, feats.shape)
    assert f.grad.shape == feats.shape and torch.equal(f.grad.cpu(), gref)
    f.grad = None
    out2 = voxel_pooling(geom.cuda(), f, vn)
    (out2 * go.cuda()).sum().backward()                    # grad arrives as permuted NHWC view
    assert torch.equal(f.grad.cpu(), gref)


def test_dropin_keeps_caller_shape_and_asserts():
    geom, feats = _rand_case(3, 2, 6 * 5 * 4 * 3, 8, (16, 16, 1))
    g6 = geom.view(2, 6, 5, 4, 3, 3).cuda()
    f6 = feats.view(2, 6, 5, 4, 3, 8).cuda().requires_grad_(True)
    out = voxel_pooling(g6, f6, (16, 16, 1))
    out.sum().backward()
    assert f6.grad.shape == f6.shape
    with pytest.raises(AssertionError):
        voxel_pooling(g6, f6.detach().transpose(1, 2), (16, 16, 1))
    with pytest.raises(TypeError):
        voxel_pooling(g6.long(), f6.detach(), (16, 16, 1))
    with pytest.raises(ValueError):
        voxel_pooling(g6[..., :3], torch.rand(2, 360, 6, device=DEV), (16, 16, 1))   # C % 4 != 0


@pytest.mark.parametrize('dtype', [torch.float16, torch.bfloat16])
def test_dropin_half_precision(dtype):
    geom, feats = _rand_case(4, 2, 8000, 80, (64, 16, 1), dtype=dtype)
    f = feats.cuda().requires_grad_(True)
    out = voxel_pooling(geom.cuda(), f, (64, 16, 1))
    assert out.dtype == dtype
    ref = vp.voxel_pooling_ref(geom, feats.float(), (64, 16, 1))       # fp32 oracle on the upcast inputs
    assert torch.equal(out.cpu(), ref.to(dtype))                        # same fp32 sums, rounded once
    go = torch.rand(2, 80, 16, 64).to(dtype)
    out.backward(go.cuda())
    gref = vp.voxel_pooling_backward_ref(geom, go, (64, 16, 1), feats.shape)
    assert torch.equal(f.grad.cpu(), gref)                              # a gather: exact in any dtype


def test_run_to_run_bit_stability():
    geom, feats = _rand_case(5, 2, 50000, 80, (32, 8, 1))               # ~200 points per cell
    g, f = geom.cuda(), feats.cuda()
    outs = [voxel_pooling(g, f, (32, 8, 1)).clone() for _ in range(5)]
    assert all(torch.equal(outs[0], o) for o in outs[1:])


# ---------------------------------------------------------------- fused op
def _fused_case(seed, B, N, D, H, W, C, vn, dtype=torch.float32):
    g = torch.Generator().manual_seed(seed)
    X, Y, Z = vn
    geom = torch.stack([torch.randint(-2, X + 2, (B, N, D, H, W), generator=g),
                        torch.randint(-2, Y + 2, (B, N, D, H, W), generator=g),
                        torch.randint(0, Z + 1, (B, N, D, H, W), generator=g)], -1).int()
    depth = torch.rand(B * N, D, H, W, generator=g).softmax(1).to(dtype)
    ctx = (torch.rand(B * N, C, H, W, generator=g) - 0.5).to(dtype)
    go = torch.rand(B, C, Y, X, generator=g).to(dtype)
    return geom, depth, ctx, go


def _check_fused(geom, depth, ctx, go, vn, channels_last=False, kernel_path='generic'):
    d = depth.cuda().requires_grad_(True)
    c = ctx.cuda()
    if channels_last:
        c = c.contiguous(memory_format=torch.channels_last)
    c.requires_grad_(True)
    out = voxel_pooling_fused(geom.cuda(), d, c, vn)
    ref = vp.voxel_pooling_fused_ref(geom, depth, ctx, vn)
    assert out.shape == ref.shape
    exact = kernel_path == 'generic' or ctx.shape[1] not in G8_CHANNELS   # bit-exact vs materialise + index_add_
    B, N = geom.shape[0], geom.shape[1]
    feats = vp.materialise_features_ref(depth, ctx, B, N)
    _assert_forward(out, ref, vp.voxel_pooling_ref(geom, feats, vn, acc_dtype=torch.float64),
                    vp.voxel_pooling_ref(geom, feats.abs(), vn, acc_dtype=torch.float64), exact)
    out.backward(go.cuda())
    gd, gc = vp.voxel_pooling_fused_grads_ref(geom, depth, ctx, vn, go)          # fp64
    # atol: eps_f32 * (number of summed terms) * magnitude of the terms
    C, D = ctx.shape[1], depth.shape[1]
    atol_d = 1.2e-7 * C * float(go.abs().max() * ctx.abs().max())
    atol_c = 1.2e-7 * D * float(go.abs().max() * depth.abs().max())
    assert torch.allclose(d.grad.double().cpu(), gd, rtol=1e-5, atol=atol_d)
    assert torch.allclose(c.grad.double().cpu(), gc, rtol=1e-5, atol=atol_c)
    return out


@pytest.mark.parametrize('shape', [(2, 2, 5, 3, 4, 8, (6, 5, 3)), (1, 4, 30, 6, 10, 80, (32, 16, 1)),
                                   (2, 1, 7, 5, 9, 132, (8, 8, 2)), (3, 2, 59, 4, 11, 64, (40, 12, 1)),
                                   (1, 1, 1, 1, 1, 4, (1, 1, 1))])
@pytest.mark.parametrize('channels_last', [False, True])
def test_fused_forward_backward_random(shape, channels_last, kernel_path):
    B, N, D, H, W, C, vn = shape
    _check_fused(*_fused_case(7, B, N, D, H, W, C, vn), vn, channels_last, kernel_path)


@pytest.mark.parametrize('cfg,B', [(CFG_2, 2), (sweep_grid_config(128), 1)])
def test_fused_on_camera_rig(cfg, B, kernel_path):
    geom, vn = synthetic.camera_rig(cfg, B, yaw_jitter_deg=5.0)
    depth, ctx, go = synthetic.camera_features(cfg, B)
    out = _check_fused(geom, depth, ctx, go, vn.tolist(), False, kernel_path)
    # the materialised drop-in path: same bits with the generic kernels (separate multiply and add in
    # point order); the fast path contracts multiply-add (FFMA2), so it agrees to rounding
    feats = vp.materialise_features_ref(depth, ctx, B, cfg.num_cams).cuda()
    mat = voxel_pooling(geom.cuda(), feats, vn.cuda())
    if kernel_path == 'generic':
        assert torch.equal(mat, out)
    else:
        assert torch.allclose(mat, out, rtol=1e-5, atol=1e-6)


def test_fused_full_size_aim_properties():
    # shipped aiMotive shape (P = 2.88 M points/frame): size-independent properties
    cfg, B = CFG_AIM, 1
    geom, vn = synthetic.camera_rig(cfg, B, device=DEV)
    depth, ctx, go = synthetic.camera_features(cfg, B, device=DEV)
    depth.requires_grad_(True)
    ctx.requires_grad_(True)
    plan = build_plan(geom, vn)
    out = voxel_pooling_fused(None, depth, ctx, vn, plan)
    # (1) linearity in context; (2) total mass: sum_cells out = sum_kept depth*ctx
    out2 = voxel_pooling_fused(None, depth, 2 * ctx, vn, plan)
    assert torch.allclose(out2, 2 * out, rtol=1e-6, atol=1e-7)
    kept = (plan.cell_of_point >= 0).view(B * cfg.num_cams, cfg.depth_bins, *cfg.feat_hw)
    mass = torch.einsum('ndhw,nchw->c', (depth * kept).double(), ctx.double())
    assert torch.allclose(out.double().sum(dim=(0, 2, 3)), mass, rtol=1e-6, atol=1e-6)
    # (3) adjoint identity <out, go> == <depth, grad_depth> == <ctx, grad_ctx>  (bilinear op)
    out.backward(go)
    lhs = (out.double() * go.double()).sum()
    assert torch.allclose(lhs, (depth.double() * depth.grad.double()).sum(), rtol=1e-5)
    assert torch.allclose(lhs, (ctx.double() * ctx.grad.double()).sum(), rtol=1e-5)
    # (4) dropped points get exactly zero depth gradient
    assert float(depth.grad[~kept].abs().max()) == 0.0
    # (5) bit-stable
    assert torch.equal(out, voxel_pooling_fused(None, depth, ctx, vn, plan))


@pytest.mark.parametrize('dtype', [torch.float16, torch.bfloat16])
def test_fused_half_precision(dtype):
    vn = (32, 16, 1)
    geom, depth, ctx, go = _fused_case(9, 2, 2, 20, 6, 10, 80, vn, dtype=dtype)
    d = depth.cuda().requires_grad_(True)
    c = ctx.cuda().requires_grad_(True)
    out = voxel_pooling_fused(geom.cuda(), d, c, vn)
    ref = vp.voxel_pooling_fused_ref(geom, depth.float(), ctx.float(), vn)
    assert out.dtype == dtype
    assert torch.equal(out.cpu(), ref.to(dtype))                        # same fp32 sums, rounded once
    out.backward(go.cuda())
    gd, gc = vp.voxel_pooling_fused_grads_ref(geom, depth.float(), ctx.float(), vn, go.float())
    md, mc = vp.voxel_pooling_fused_grads_ref(geom, depth.float().abs(), ctx.float().abs(), vn, go.float().abs())
    # fp32 sums of C (grad_depth) / D (grad_context) products, rounded once
    lo, hi = round_bracket(gd, sum_bound(80, md), dtype)
    assert bool(in_bracket(d.grad.cpu(), lo, hi).all())
    lo, hi = round_bracket(gc, sum_bound(20, mc), dtype)
    assert bool(in_bracket(c.grad.cpu(), lo, hi).all())


def test_plan_reuse_and_stream_capture():
    vn = (32, 16, 1)
    geom, depth, ctx, go = _fused_case(11, 2, 2, 20, 6, 10, 80, vn)
    g, d, c = geom.cuda(), depth.cuda(), ctx.cuda()
    plan = build_plan(g, vn)
    eager = voxel_pooling_fused(None, d, c, vn, plan).clone()
    # the whole call chain is capturable in a CUDA graph (no syncs, caller-owned memory)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        voxel_pooling_fused(g, d, c, vn)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        captured = voxel_pooling_fused(g, d, c, vn)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(captured, eager)

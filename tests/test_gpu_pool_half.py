"""GPU tests of the fp16 / bf16 pooling kernels (the generic kernels of csrc/pool.cu, which every half-precision call
goes through) against the CPU oracle of oracle/voxel_pool_ref.py.

The forward kernels upcast every input to fp32 exactly, sum a cell's points in plan (point) order with a separate
multiply and add, and round once on the store: the output must be BIT-EQUAL to the fp32 oracle (the same sums in the
same order) rounded once to the dtype -- empty cells, a cell of thousands of points, fp16 cells that overflow to inf
included.  The fused backward sums n fp32 products (n = C for grad_depth, D for grad_context) and rounds once, so each
gradient must lie in ``round_bracket(fp64 result, gamma_n * sum |terms|)``; both layouts of the context and of
grad_out are covered, and the two grad_out layouts must give identical bits."""
import pytest
import torch

from mm_training_b200.ops.voxel_pooling import voxel_pooling, voxel_pooling_fused
from oracle import voxel_pool_ref as vp
from oracle.depth_softmax_ref import in_bracket, round_bracket, sum_bound

pytestmark = pytest.mark.gpu
DEV = 'cuda'
HALF = [torch.float16, torch.bfloat16]


def _bits(t):
    return t.contiguous().view(torch.int16)


# ---------------------------------------------------------------- drop-in op
@pytest.mark.parametrize('C', [4, 80, 132, 260, 512])
@pytest.mark.parametrize('dtype', HALF)
def test_dropin_forward_is_the_fp32_oracle_rounded_once(C, dtype):
    B, Np, vn = 2, 6000, (24, 16, 2)
    X, Y, Z = vn
    g = torch.Generator().manual_seed(C)
    geom = torch.stack([torch.randint(-3, X + 3, (B, Np), generator=g), torch.randint(-3, Y + 3, (B, Np), generator=g),
                        torch.randint(-1, Z + 1, (B, Np), generator=g)], -1).int()
    geom[..., 0] = torch.where(geom[..., 0] == 5, 6, geom[..., 0])          # column x = 5 stays empty
    geom[0, :4000] = torch.tensor([3, 2, 0], dtype=torch.int32)             # one dense cell of 4000 points
    feats = ((torch.rand(B, Np, C, generator=g) - 0.5) * 4).to(dtype)
    f = feats.cuda().requires_grad_(True)
    out = voxel_pooling(geom.cuda(), f, vn)
    ref = vp.voxel_pooling_ref(geom, feats.float(), vn)
    assert out.dtype == dtype and out.shape == (B, C, Y, X)
    assert torch.equal(out.cpu(), ref.to(dtype))
    assert float(out[:, :, :, 5].detach().abs().max()) == 0.0
    go = torch.rand(B, C, Y, X, generator=g).to(dtype)
    out.backward(go.cuda())
    assert torch.equal(f.grad.cpu(), vp.voxel_pooling_backward_ref(geom, go, vn, feats.shape))   # a gather: exact


def test_fp16_cell_sums_past_65504_round_to_inf():
    B, Np, C, vn = 1, 12000, 8, (4, 2, 1)
    geom = torch.zeros(B, Np, 3, dtype=torch.int32)
    feats = torch.full((B, Np, C), 30.0)
    geom[0, 3000:6000, 0] = 1
    feats[0, 3000:6000] = -30.0                                             # cell 1: -90000 -> -inf
    geom[0, 6000:, 0] = 2
    feats[0, 9000:] = -30.0                                                 # cell 2: up to 90000, then back to 0 in fp32
    feats = feats.half()
    out = voxel_pooling(geom.cuda(), feats.cuda(), vn)
    ref = vp.voxel_pooling_ref(geom, feats.float(), vn)
    assert float(ref[0, 0, 0, 0]) == 90000.0 and float(ref[0, 0, 0, 2]) == 0.0
    assert torch.equal(out.cpu(), ref.half())
    assert out[0, :, 0, 0].isposinf().all() and out[0, :, 0, 1].isneginf().all() and bool((out[0, :, 0, 2] == 0).all())


# ---------------------------------------------------------------- fused op
FUSED_SHAPES = [(2, 2, 5, 3, 4, 8, (6, 5, 3)), (1, 4, 30, 6, 10, 80, (32, 16, 1)), (2, 1, 7, 5, 9, 132, (8, 8, 2)),
                (3, 2, 59, 4, 11, 64, (40, 12, 1)), (1, 1, 1, 1, 1, 4, (1, 1, 1)), (1, 2, 33, 5, 7, 512, (16, 8, 1)),
                (2, 1, 59, 3, 6, 260, (9, 7, 1))]


def _fused_case(seed, B, N, D, H, W, C, vn, dtype):
    g = torch.Generator().manual_seed(seed)
    X, Y, Z = vn
    geom = torch.stack([torch.randint(-2, X + 2, (B, N, D, H, W), generator=g),
                        torch.randint(-2, Y + 2, (B, N, D, H, W), generator=g),
                        torch.randint(0, Z + 1, (B, N, D, H, W), generator=g)], -1).int()
    depth = torch.rand(B * N, D, H, W, generator=g).softmax(1).to(dtype)
    ctx = (torch.rand(B * N, C, H, W, generator=g) - 0.5).to(dtype)
    go = torch.rand(B, C, Y, X, generator=g).to(dtype)
    return geom, depth, ctx, go


@pytest.mark.parametrize('layout', ['nchw', 'channels_last'])
@pytest.mark.parametrize('shape', FUSED_SHAPES)
@pytest.mark.parametrize('dtype', HALF)
def test_fused_forward_bit_equal_and_gradients_in_the_bracket(dtype, shape, layout):
    B, N, D, H, W, C, vn = shape
    geom, depth, ctx, go = _fused_case(7, B, N, D, H, W, C, vn, dtype)
    d = depth.cuda().requires_grad_(True)
    c = ctx.cuda()
    if layout == 'channels_last':
        c = c.contiguous(memory_format=torch.channels_last)
    c.requires_grad_(True)
    out = voxel_pooling_fused(geom.cuda(), d, c, vn)
    assert out.dtype == dtype
    assert torch.equal(out.cpu(), vp.voxel_pooling_fused_ref(geom, depth.float(), ctx.float(), vn).to(dtype))
    grads = []
    for go_dev in (go.cuda(), go.cuda().contiguous(memory_format=torch.channels_last)):
        d.grad = c.grad = None
        out.backward(go_dev, retain_graph=True)
        grads.append((d.grad.clone(), c.grad.clone()))
    assert torch.equal(_bits(grads[0][0]), _bits(grads[1][0]))              # grad_out layout: same bits
    assert torch.equal(_bits(grads[0][1]), _bits(grads[1][1]))
    gd_dev, gc_dev = grads[0]
    assert gc_dev.shape == ctx.shape
    gd, gc = vp.voxel_pooling_fused_grads_ref(geom, depth.float(), ctx.float(), vn, go.float())
    md, mc = vp.voxel_pooling_fused_grads_ref(geom, depth.float().abs(), ctx.float().abs(), vn, go.float().abs())
    lo, hi = round_bracket(gd, sum_bound(C, md), dtype)
    assert bool(in_bracket(gd_dev.cpu(), lo, hi).all())
    lo, hi = round_bracket(gc, sum_bound(D, mc), dtype)
    assert bool(in_bracket(gc_dev.cpu(), lo, hi).all())
    kept = vp.cell_index_ref(geom, vn)[0].view(B * N, D, H, W)
    assert bool((gd_dev.cpu()[~kept] == 0).all())                             # dropped points: exactly no gradient

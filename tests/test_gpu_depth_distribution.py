"""GPU parity tests of the one-pass depth distribution (csrc/depth_softmax.cu, ops/depth_distribution.py) against
the reference's torch ops restated verbatim (layers/backbones/lss_fpn.py:423,427-434): rtol 1e-5 (+ atol 1e-7) in
fp32, 1e-2 for fp16 / bf16 logits; the overwritten pixels must equal the oracle bit for bit.  The half-precision test
also holds the probabilities to the fp64 bound of oracle/depth_softmax_ref.py and the fp16 / bf16 gradients to the
rounding bracket of the fp64 backward; tests/test_gpu_depth_softmax_edges.py does so at every shape, dtype and edge
value (masked bins, underflow, non-finite rows)."""
import pytest
import torch

from mm_training_b200.ops.depth_distribution import depth_distribution
from oracle import depth_softmax_ref as ds

pytestmark = pytest.mark.gpu
DEV = 'cuda'


def _reference(depth_feature, D, depth_oracle):
    """lss_fpn.py:423,427-434, the reference's ops in the reference's order."""
    depth = depth_feature[:, :D].softmax(1)
    if depth_oracle is None:
        return depth, depth
    b, c, h, w = depth.shape
    fg_mask = (torch.max(depth_oracle, dim=1).values > 0.0).view(-1)
    depth_flattened = depth.permute(0, 2, 3, 1).contiguous().view(-1, c)
    depth_oracle_flattened = depth_oracle.permute(0, 2, 3, 1).contiguous().view(-1, c)
    depth_updated = depth_flattened
    depth_updated[fg_mask] = depth_oracle_flattened[fg_mask]
    depth_updated = depth_updated.view(b, h, w, c).permute(0, 3, 1, 2)
    return depth, depth_updated


def _case(BN, D, C, H, W, seed, dtype=torch.float32, oracle=True):
    g = torch.Generator().manual_seed(seed)
    feat = (torch.randn(BN, D + C, H, W, generator=g) * 3).to(dtype)
    orc = None
    if oracle:
        idx = torch.randint(0, D, (BN, H, W), generator=g)
        orc = torch.nn.functional.one_hot(idx, D).permute(0, 3, 1, 2).float()
        orc = orc * (torch.rand(BN, 1, H, W, generator=g) < 0.4)              # 40 % of the pixels have a LiDAR return
    return feat, orc


@pytest.mark.parametrize('shape', [(8, 112, 80, 16, 44), (2, 409, 80, 44, 80), (3, 7, 5, 3, 5)])
@pytest.mark.parametrize('oracle', [False, True])
def test_forward_and_backward_match_the_reference_ops(shape, oracle):
    BN, D, C, H, W = shape
    feat, orc = _case(BN, D, C, H, W, seed=BN + D, oracle=oracle)
    a = feat.to(DEV).requires_grad_(True)
    b = feat.to(DEV).requires_grad_(True)
    o = orc.to(DEV) if orc is not None else None
    depth, used = depth_distribution(a, D, o)
    rdepth, rused = _reference(b, D, o)
    assert depth.is_contiguous() and used.is_contiguous() and depth.dtype == torch.float32
    assert torch.allclose(depth, rdepth, rtol=1e-5, atol=1e-7)
    assert torch.allclose(used, rused, rtol=1e-5, atol=1e-7)
    if oracle:
        fg = (o.max(1, keepdim=True).values > 0).expand_as(o)
        assert torch.equal(used[fg], o[fg])                                        # overwritten pixels: the oracle, bit for bit
    g = torch.Generator().manual_seed(1)
    w1 = torch.rand(depth.shape, generator=g).to(DEV)
    w2 = torch.rand(depth.shape, generator=g).to(DEV)
    ((depth * w1).sum() + (used * w2).sum()).backward()
    ((rdepth * w1).sum() + (rused * w2).sum()).backward()
    assert float(a.grad[:, D:].abs().sum()) == 0.0                                 # context channels: no gradient from here
    assert torch.allclose(a.grad, b.grad, rtol=1e-4, atol=1e-6)


@pytest.mark.parametrize('dtype', [torch.float16, torch.bfloat16])
def test_half_precision_logits(dtype):
    feat, orc = _case(4, 112, 80, 16, 44, seed=3, dtype=dtype)
    a = feat.to(DEV).requires_grad_(True)
    o = orc.to(DEV)
    depth, used = depth_distribution(a, 112, o)
    rdepth, rused = _reference(feat.to(DEV).float(), 112, o)
    assert torch.allclose(depth, rdepth, rtol=1e-2, atol=1e-6) and torch.allclose(used, rused, rtol=1e-2, atol=1e-6)
    ref = ds.softmax_ref(a.detach(), 112)
    assert bool(((depth.double() - ref).abs() <= ds.forward_rel_bound(a.detach(), 112) * ref + ds.FLT_MIN).all())
    used.sum().backward()
    assert a.grad.dtype == dtype and bool(torch.isfinite(a.grad).all())
    gref, mag = ds.softmax_backward_ref(depth.detach(), None, torch.ones_like(used), o)
    lo, hi = ds.round_bracket(gref, ds.sum_bound(112 + 3, mag), dtype)
    assert bool(ds.in_bracket(a.grad[:, :112], lo, hi).all())


def test_feeds_the_fused_pooling_without_a_copy():
    from mm_training_b200 import synthetic
    from mm_training_b200.configs import CFG_2
    from mm_training_b200.ops.voxel_pooling import voxel_pooling_fused
    cfg, B = CFG_2, 2
    geom, vn = synthetic.camera_rig(cfg, B, device=DEV)
    feat, orc = _case(B * cfg.num_cams, cfg.depth_bins, cfg.output_channels, *cfg.feat_hw, seed=4)
    a = feat.to(DEV).requires_grad_(True)
    b = feat.to(DEV).requires_grad_(True)
    depth, used = depth_distribution(a, cfg.depth_bins, orc.to(DEV))
    out = voxel_pooling_fused(geom, used, a[:, cfg.depth_bins:].contiguous(), vn)
    rdepth, rused = _reference(b, cfg.depth_bins, orc.to(DEV))
    ref = voxel_pooling_fused(geom, rused.contiguous(), b[:, cfg.depth_bins:].contiguous(), vn)
    assert torch.allclose(out, ref, rtol=1e-5, atol=1e-6)
    go = torch.rand_like(out)
    (out * go).sum().backward()
    (ref * go).sum().backward()
    assert torch.allclose(a.grad, b.grad, rtol=1e-4, atol=1e-5)


def test_cpu_tensors_raise():
    with pytest.raises(RuntimeError):
        depth_distribution(torch.zeros(1, 4, 2, 2), 3)


# ---------------------------------------------------------------- softmax folded into the forward (SURVEY.md 8f, N4)
@pytest.mark.parametrize('cfg_name,B,extra', [('cfg2', 3, 0), ('cfg2', 1, 8), ('aim', 1, 0)])
def test_forward_from_logits_equals_softmax_then_pooling(cfg_name, B, extra):
    from mm_training_b200 import synthetic
    from mm_training_b200.configs import CFG_2, CFG_AIM
    from mm_training_b200.ops.voxel_pooling import build_plan, voxel_pooling_fused, voxel_pooling_fused_logits
    cfg = CFG_2 if cfg_name == 'cfg2' else CFG_AIM
    D, C = cfg.depth_bins, cfg.output_channels
    geom, vn_t = synthetic.camera_rig(cfg, B, device=DEV, yaw_jitter_deg=5.0, seed=6)
    vn = tuple(int(v) for v in vn_t.tolist())
    g = torch.Generator().manual_seed(B + extra)
    feat = (torch.randn(B * cfg.num_cams, D + C + extra, *cfg.feat_hw, generator=g) * 2).to(DEV)
    plan = build_plan(geom, vn, frustum=tuple(geom.shape[1:5]))
    a = feat.clone().requires_grad_(True)
    b = feat.clone().requires_grad_(True)
    out = voxel_pooling_fused_logits(a, D, C, vn, plan)
    ref = voxel_pooling_fused(None, b[:, :D].softmax(1).contiguous(), b[:, D:D + C].contiguous(), vn, plan)
    # same sums in the same order over probabilities that differ by float32 rounding of exp / normaliser
    scale = voxel_pooling_fused(None, b[:, :D].softmax(1).contiguous().detach(), b[:, D:D + C].abs().contiguous().detach(), vn, plan)
    assert bool(((out - ref).abs() <= 1e-5 * ref.abs() + 2e-6 * scale).all())
    assert bool((out[scale == 0] == 0).all())
    go = torch.rand(out.shape, generator=g).to(DEV)
    out.backward(go)
    ref.backward(go)
    assert torch.allclose(a.grad, b.grad, rtol=1e-4, atol=1e-5)
    if extra:
        assert float(a.grad[:, D + C:].abs().sum()) == 0.0

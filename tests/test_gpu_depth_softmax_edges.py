"""GPU tests of the depth distribution (csrc/depth_softmax.cu, and the statistics pre-pass of
``voxel_pooling_fused_logits`` in csrc/pool_runs.cu) against the fp64 oracle of oracle/depth_softmax_ref.py, at the
shapes and values where a per-pixel softmax goes wrong: D from 1 to 409, images whose pixel count leaves a ragged
256-thread tail, logits given as a channel slice of DepthNet's output, fp32 / fp16 / bf16, logits spread over +-80
(probabilities that underflow), constant rows, masked (-inf) bins -- leading, trailing, interleaved, all but one --
and non-finite rows (same NaN pattern as torch.softmax).

Bounds (derived in ``depth_softmax_ref.forward_rel_bound`` / ``sum_bound``): every finite probability within
(|l - m| + E + 5R + D + 10) * 2^-24 of the fp64 value relative, + FLT_MIN absolute for underflow; masked bins exactly 0;
constant rows exactly fp32(1 / D).  Gradients: fp32 within gamma_{D+3} * p * (|g| + sum p |g|) of the fp64 result
computed from the kernel's own probabilities; fp16 / bf16 inside the rounding bracket of that bound.  The oracle
overwrite is compared bit for bit."""
import math

import pytest
import torch

from mm_training_b200 import _lib
from mm_training_b200.ops.depth_distribution import depth_distribution
from oracle import depth_softmax_ref as ds

pytestmark = pytest.mark.gpu
DEV = 'cuda'
DS = [1, 2, 31, 32, 33, 112, 409]
HWS = [(1, 1), (3, 5), (17, 15), (257, 1), (16, 44), (44, 80)]
BNS = [1, 3, 8]
DTYPES = [torch.float32, torch.float16, torch.bfloat16]
REGIMES = ['randn3', 'spread80', 'constant', 'lead_mask', 'trail_mask', 'interleaved_mask', 'one_left', 'non_finite']
FINITE = len(REGIMES) - 1                     # regimes [0, FINITE) give finite distributions


def _bits(t):
    return t.view({4: torch.int32, 2: torch.int16}[t.element_size()])


def _logits(BN, D, H, W, seed, regimes=len(REGIMES)):
    """(BN, D, H, W) float32 logits, pixel i following REGIMES[(i + seed) % regimes]; returns (logits, regime map)."""
    g = torch.Generator().manual_seed(seed)
    P = BN * H * W
    reg = (torch.arange(P) + seed) % regimes
    x = torch.randn(P, D, generator=g) * 3
    spread = (torch.rand(P, D, generator=g) * 2 - 1) * 80
    x = torch.where((reg == 1).view(P, 1), spread, x)
    x = torch.where((reg == 2).view(P, 1), (torch.rand(P, 1, generator=g) * 20 - 10).expand(P, D), x)
    d = torch.arange(D).view(1, D)
    k = torch.randint(1, max(D, 2), (P, 1), generator=g)           # 1 <= k <= D - 1 masked bins (none when D = 1)
    lead = (reg == 3).view(P, 1) & (d < k) & (D > 1)
    trail = (reg == 4).view(P, 1) & (d >= D - k) & (D > 1)
    keep = torch.randint(0, D, (P, 1), generator=g)
    inter = (reg == 5).view(P, 1) & (torch.rand(P, D, generator=g) < 0.5) & (d != keep)
    one = (reg == 6).view(P, 1) & (d != keep)
    x = x.masked_fill(lead | trail | inter | one, -math.inf)
    # non-finite rows, in turn: all -inf, one +inf, one NaN (with a -inf beside it when D > 1)
    nf = (reg == 7).nonzero().view(-1)
    for j, p in enumerate(nf.tolist()):
        kind = j % 3
        if kind == 0:
            x[p] = -math.inf
        else:
            x[p, int(keep[p])] = math.inf if kind == 1 else math.nan
            if D > 1:
                x[p, (int(keep[p]) + 1) % D] = -math.inf
    x = x.view(BN, H, W, D).permute(0, 3, 1, 2).contiguous()
    return x, reg.view(BN, 1, H, W)


def _feature(x, dtype, sliced, extra=3):
    """Logits as a contiguous tensor, or as the first D channels of a (BN, D + C + extra, H, W) feature map."""
    if not sliced:
        return x.to(dtype).to(DEV)
    BN, D, H, W = x.shape
    feat = torch.randn(BN, D + 8 + extra, H, W).to(dtype)
    feat[:, :D] = x.to(dtype)
    return feat.to(DEV)


def _check_forward(p, feat, D, reg):
    """p: the kernel's (BN, D, H, W) float32 probabilities for the logits feat[:, :D]."""
    x = feat[:, :D].float()
    ref = ds.softmax_ref(feat, D)
    nan_ref = torch.isnan(ref)
    assert torch.equal(torch.isnan(p), nan_ref)                               # non-finite rows: torch's NaN pattern
    assert bool(nan_ref.any(1).eq(nan_ref.all(1)).all())                     # a row is all NaN or has none
    fin = ~nan_ref
    bound = ds.forward_rel_bound(feat, D) * ref + ds.FLT_MIN
    err = (p.double() - ref).abs()
    assert bool((err[fin] <= bound[fin]).all()), float((err - bound)[fin].max())
    assert bool((p[fin & (x == -math.inf)] == 0).all())                       # masked bins: exact zeros
    const = (reg == 2).expand_as(p).to(p.device)
    assert bool((p[const] == torch.tensor(1.0, dtype=torch.float32) / D).all())   # exactly fp32(1 / D)
    if D == 1:
        assert bool((p[fin] == 1).all())


@pytest.mark.parametrize('sliced', [False, True], ids=['contiguous', 'channel_slice'])
@pytest.mark.parametrize('dtype', DTYPES)
@pytest.mark.parametrize('D', DS)
def test_forward_within_the_fp64_bound(D, dtype, sliced):
    for i, (H, W) in enumerate(HWS):
        BN = BNS[(i + D) % 3]
        x, reg = _logits(BN, D, H, W, seed=i + D)
        feat = _feature(x, dtype, sliced)
        depth, used = depth_distribution(feat, D)
        assert depth is used and depth.is_contiguous() and depth.shape == (BN, D, H, W)
        _check_forward(depth, feat, D, reg)


def _oracle_rows(BN, D, H, W, seed):
    """Depth oracle with, in turn per pixel: a one-hot row, a soft row in (0, 1) (one entry -0.0), an all-zero row,
    a row of negative entries and zeros, and an all -0.0 row.  Only the first two are foreground."""
    g = torch.Generator().manual_seed(seed)
    P = BN * H * W
    kind = (torch.arange(P) + seed) % 5
    o = torch.zeros(P, D)
    o[kind == 0, :] = torch.nn.functional.one_hot(torch.randint(0, D, (P,), generator=g), D).float()[kind == 0]
    soft = torch.rand(P, D, generator=g) * 0.98 + 0.01
    if D > 1:
        soft[:, 0] = -0.0
    o = torch.where((kind == 1).view(P, 1), soft, o)
    neg = -torch.rand(P, D, generator=g) * (torch.rand(P, D, generator=g) < 0.7)
    o = torch.where((kind == 3).view(P, 1), neg, o)
    o = torch.where((kind == 4).view(P, 1), torch.full_like(o, -0.0), o)
    return o.view(BN, H, W, D).permute(0, 3, 1, 2).contiguous()


@pytest.mark.parametrize('dtype', DTYPES)
@pytest.mark.parametrize('D', [1, 2, 33, 112])
def test_oracle_overwrite_is_bit_exact(D, dtype):
    for i, (H, W) in enumerate(HWS[1:]):
        BN = BNS[i % 3]
        x, reg = _logits(BN, D, H, W, seed=7 + i, regimes=FINITE)
        feat = _feature(x, dtype, sliced=bool(i % 2))
        orc = _oracle_rows(BN, D, H, W, seed=i).to(DEV)
        depth, used = depth_distribution(feat, D, orc)
        _check_forward(depth, feat, D, reg)
        fg = ds.foreground(orc)
        assert bool(fg.any()) and bool((~fg).any())
        assert torch.equal(_bits(used), _bits(torch.where(fg, orc, depth)))     # fg: the oracle, else: depth, bit for bit
        assert torch.equal(_bits(used[fg.expand_as(used)]), _bits(orc[fg.expand_as(orc)]))


@pytest.mark.parametrize('through', ['depth', 'used', 'both'])
@pytest.mark.parametrize('dtype', DTYPES)
@pytest.mark.parametrize('D', DS)
def test_backward_within_the_fp64_bound(D, dtype, through):
    for i, (H, W) in enumerate(HWS):
        BN = BNS[(i + D + 1) % 3]
        x, _ = _logits(BN, D, H, W, seed=100 + i + D, regimes=FINITE)
        feat = _feature(x, dtype, sliced=bool(i % 2)).requires_grad_(True)
        orc = None if through == 'depth' else _oracle_rows(BN, D, H, W, seed=i).to(DEV)
        depth, used = depth_distribution(feat, D, orc)
        g = torch.Generator().manual_seed(i)
        w1 = (torch.randn(depth.shape, generator=g) if through != 'used' else None)
        w2 = (torch.randn(depth.shape, generator=g) if through != 'depth' else None)
        w1 = w1.to(DEV) if w1 is not None else None
        w2 = w2.to(DEV) if w2 is not None else None
        loss = 0
        if w1 is not None:
            loss = loss + (depth * w1).sum()
        if w2 is not None:
            loss = loss + (used * w2).sum()
        loss.backward()
        assert feat.grad.dtype == dtype
        grad = feat.grad[:, :D]
        ref, mag = ds.softmax_backward_ref(depth.detach(), w1, w2, orc)
        err = ds.sum_bound(D + 3, mag)
        if dtype == torch.float32:
            assert bool(((grad.double() - ref).abs() <= err).all()), float(((grad.double() - ref).abs() - err).max())
        else:
            lo, hi = ds.round_bracket(ref, err, dtype)
            assert bool(ds.in_bracket(grad, lo, hi).all())
        assert bool((grad[x.to(DEV) == -math.inf] == 0).all())                  # masked bins: exactly no gradient
        if D == 1:
            assert bool((grad == 0).all())
        assert float(feat.grad[:, D:].abs().sum()) == 0.0                       # channels past D: untouched


@pytest.mark.parametrize('dtype', DTYPES)
def test_null_gradient_pointers_equal_zero_gradients(dtype):
    """Through the C ABI: grad_prob = NULL or grad_used = NULL gives the bits of passing zeros."""
    BN, D, H, W = 3, 33, 17, 15
    x, _ = _logits(BN, D, H, W, seed=5, regimes=FINITE)
    orc = _oracle_rows(BN, D, H, W, seed=5).to(DEV)
    prob, _ = depth_distribution(_feature(x, dtype, sliced=False), D, orc)
    g = torch.Generator().manual_seed(5)
    gp = torch.randn(prob.shape, generator=g).to(DEV)
    gu = torch.randn(prob.shape, generator=g).to(DEV)
    z = torch.zeros_like(prob)
    L = _lib.lib()

    def run(grad_prob, grad_used, oracle):
        out = torch.full(prob.shape, math.nan, dtype=dtype, device=DEV)
        ptr = (lambda t: t.data_ptr() if t is not None else None)
        rc = L.bevdepth_softmax_backward(prob.data_ptr(), ptr(grad_prob), ptr(grad_used), ptr(oracle), BN, D, H, W,
                                         out.data_ptr(), _lib.dtype_code(out), _lib.stream_ptr(prob.device))
        _lib.check(rc, 'bevdepth_softmax_backward')
        return out

    for oracle in (None, orc):
        a = run(None, gu, oracle)
        assert not bool(torch.isnan(a).any())
        assert torch.equal(_bits(a), _bits(run(z, gu, oracle)))
        b = run(gp, None, oracle)
        assert torch.equal(_bits(b), _bits(run(gp, z, oracle)))
    assert L.bevdepth_softmax_backward(prob.data_ptr(), None, None, None, BN, D, H, W, z.data_ptr(),
                                       _lib.dtype_code(z), _lib.stream_ptr(prob.device)) != 0


# ---------------------------------------------------------------- masked leading bins through the folded forward
@pytest.mark.parametrize('extra', [0, 8])
def test_fused_logits_with_masked_leading_bins(extra):
    from mm_training_b200 import synthetic
    from mm_training_b200.configs import CFG_2
    from mm_training_b200.ops.voxel_pooling import build_plan, voxel_pooling_fused, voxel_pooling_fused_logits
    cfg, B = CFG_2, 1
    D, C = cfg.depth_bins, cfg.output_channels
    H, W = cfg.feat_hw
    geom, vn_t = synthetic.camera_rig(cfg, B, device=DEV, yaw_jitter_deg=5.0, seed=6)
    vn = tuple(int(v) for v in vn_t.tolist())
    BN = B * cfg.num_cams
    g = torch.Generator().manual_seed(11 + extra)
    feat = torch.randn(BN, D + C + extra, H, W, generator=g) * 2
    # restrict the depth range: camera n masks its first k_n bins, and a random third of the pixels a random number more
    k = torch.tensor([0, 1, 5, D // 3, D - 1, D // 2] * BN)[:BN].view(BN, 1, 1, 1)
    k = torch.where(torch.rand(BN, 1, H, W, generator=g) < 0.33, torch.randint(0, D, (BN, 1, H, W), generator=g), k)
    masked = torch.arange(D).view(1, D, 1, 1) < k
    feat[:, :D] = feat[:, :D].masked_fill(masked, -math.inf)
    feat, masked = feat.to(DEV), masked.to(DEV)
    plan = build_plan(geom, vn, frustum=tuple(geom.shape[1:5]))
    a = feat.clone().requires_grad_(True)
    b = feat.clone().requires_grad_(True)
    out = voxel_pooling_fused_logits(a, D, C, vn, plan)
    assert 'VoxelPoolingFusedLogits' in type(out.grad_fn).__name__            # the native folded forward ran
    assert bool(torch.isfinite(out).all())
    prob, _ = depth_distribution(b, D)
    ref = voxel_pooling_fused(None, prob, b[:, D:D + C].contiguous(), vn, plan)
    scale = voxel_pooling_fused(None, prob.detach(), b[:, D:D + C].abs().contiguous().detach(), vn, plan)
    assert bool(((out - ref).abs() <= 1e-5 * ref.abs() + 2e-6 * scale).all())
    assert bool((out[scale == 0] == 0).all())
    go = torch.rand(out.shape, generator=g).to(DEV)
    out.backward(go)
    ref.backward(go)
    assert bool(torch.isfinite(a.grad).all())
    assert torch.allclose(a.grad, b.grad, rtol=1e-4, atol=1e-5)
    assert bool((a.grad[:, :D][masked] == 0).all())
    if extra:
        assert float(a.grad[:, D + C:].abs().sum()) == 0.0

"""GPU tests of the native depth loss (csrc/depth_loss.cu, ops/depth_loss.py).

The gradient must have the bits of torch's CUDA autograd of the reference (``bench_train.depth_loss_ref``), the loss
must lie within ``depth_loss_ref.forward_bound`` of the fp64 oracle, bins and one-hot rows must give the same bits, and
the op must be bit-stable, autocast-neutral and graph-capturable.  torch's CUDA binary_cross_entropy asserts on inputs
outside [0, 1] (a NaN included) and that assert aborts the CUDA context, so such inputs are compared with the fp64
oracle only."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import bench_train
from mm_training_b200.ops import depth_loss
from mm_training_b200.ops.depth_distribution import depth_distribution
from mm_training_b200.ops.depth_labels import depth_labels as make_depth_labels
from oracle import depth_labels_ref as dl
from oracle import depth_loss_ref as ref

pytestmark = pytest.mark.gpu
DEV = 'cuda'

SHAPES = {'cfg2': (4, 112, 16, 44), 'cfg_aim': (2, 409, 44, 80), 'd1': (3, 1, 5, 7), 'd3': (3, 3, 5, 7),
          'd5': (2, 5, 9, 11), 'd64': (3, 64, 5, 7), 'd113': (2, 113, 6, 9), 'd409': (2, 409, 3, 7),
          'one_pixel': (5, 64, 1, 1)}
EDGE_P = [0.0, 1.0, 1e-30, 1.0 - 2.0 ** -24, 2.0 ** -149, 0.5, 1e-7, 0.999]


def _probs(BN, D, H, W, seed, mask_leading=True):
    """depth_distribution of random logits; with mask_leading, the first two bins of every third pixel are -inf
    (exact zeros)."""
    g = torch.Generator().manual_seed(seed)
    logits = 3 * torch.randn(BN, D, H, W, generator=g)
    if mask_leading and D >= 3:
        m = (torch.arange(BN * H * W) % 3 == 0).view(BN, 1, H, W)
        logits[:, :2] = logits[:, :2].masked_fill(m, float('-inf'))
    p, _ = depth_distribution(logits.to(DEV), D)
    return p.detach()


def _labels(kind, BN, D, H, W, seed):
    g = torch.Generator().manual_seed(seed)
    P = BN * H * W
    bins = torch.randint(0, D, (P,), generator=g)
    zero = torch.rand(P, generator=g) < 0.25
    if kind == 'onehot_zero_rows':
        t = F.one_hot(bins, D).float()
        t[zero] = 0
        return t.to(DEV)
    if kind == 'soft':
        t = torch.rand(P, D, generator=g)
        t[zero] = 0
        return t.to(DEV)
    if kind == 'bins':
        b = bins.int()
        b[zero] = torch.where(torch.rand(int(zero.sum()), generator=g) < 0.5, -1, D).int()
        return b.to(DEV)
    raise ValueError(kind)


def _dense(labels, D):
    t, _ = ref.rows(labels.cpu(), torch.empty(1, D, 1, 1))
    return t.to(DEV)


def _native(labels, prob):
    x = prob.clone().requires_grad_(True)
    L = depth_loss(labels, x)
    (gx,) = torch.autograd.grad(L, (x,))
    return L.detach(), gx


def _torch(labels, prob):
    x = prob.clone().requires_grad_(True)
    L = bench_train.depth_loss_ref(labels, x, prob.shape[1])
    (gx,) = torch.autograd.grad(L, (x,))
    return L.detach(), gx


def _check(labels, prob, against_torch=True):
    L, g = _native(labels, prob)
    L64, cnt = ref.loss_ref(labels.cpu(), prob.cpu())
    bound = ref.forward_bound(labels.cpu(), prob.cpu())
    assert abs(float(L) - float(L64)) <= bound, (float(L), float(L64), bound)
    D = prob.shape[1]
    fg = ref.foreground(_dense(labels, D).cpu())
    g_rows = g.permute(0, 2, 3, 1).reshape(-1, D)[fg.to(DEV).logical_not()]
    assert bool((g_rows.view(torch.int32) == 0).all())                   # background: exactly +0
    if against_torch:
        dense = labels if labels.dtype == torch.float32 else _dense(labels, D)
        Lt, gt = _torch(dense, prob)
        assert torch.equal(g, gt)
        assert abs(float(L) - float(Lt)) <= 2 * bound + 4 * ref.U32 * abs(float(Lt))
    return L, g


@pytest.mark.parametrize('shape', list(SHAPES))
@pytest.mark.parametrize('kind', ['onehot_zero_rows', 'soft', 'bins'])
def test_loss_and_gradient(shape, kind):
    BN, D, H, W = SHAPES[shape]
    prob = _probs(BN, D, H, W, seed=list(SHAPES).index(shape))
    labels = _labels(kind, BN, D, H, W, seed=7)
    L, g = _check(labels, prob)
    if kind == 'bins':                                                  # bins == the one-hot rows, bit for bit
        L2, g2 = _native(_dense(labels, D), prob)
        assert torch.equal(L, L2) and torch.equal(g, g2)
    if D == 1:
        assert bool((prob == 1).all())


def test_depth_label_generator_output():
    """DepthLabelGenerator's rows are all foreground (a cell with no return gets bin 0: the reference's quirk)."""
    D, hw = 112, (256, 704)
    case = dl.synthetic_case(batch=2, sweeps=1, cams=2, num_points=60000, image_hw=hw, seed=5)
    clouds, ext, intr, bda = case
    onehot, bins = make_depth_labels([c.to(DEV) for c in clouds], ext.to(DEV), intr.to(DEV), bda.to(DEV), hw, 16,
                                     (2.0, 58.0, 0.5), D, return_bins=True)
    BN = onehot.shape[0] // (16 * 44)
    prob = _probs(BN, D, 16, 44, seed=3)
    L, g = _check(onehot, prob)
    assert float(ref.foreground(onehot.cpu()).float().mean()) == 1.0
    Lb, gb = _native(bins, prob)
    assert torch.equal(L, Lb) and torch.equal(g, gb)


@pytest.mark.parametrize('kind', ['onehot_zero_rows', 'soft', 'bins'])
def test_hand_placed_probabilities(kind):
    BN, D, H, W = 2, 37, 5, 9
    vals = torch.tensor(EDGE_P)
    g = torch.Generator().manual_seed(11)
    prob = vals[torch.randint(0, len(EDGE_P), (BN, D, H, W), generator=g)].to(DEV)
    labels = _labels(kind, BN, D, H, W, seed=12)
    _check(labels, prob)


@pytest.mark.parametrize('case', ['all_background', 'one_foreground'])
def test_count_edge_cases(case):
    BN, D, H, W = 2, 16, 3, 5
    prob = _probs(BN, D, H, W, seed=1)
    labels = torch.zeros(BN * H * W, D, device=DEV)
    if case == 'one_foreground':
        labels[7, 3] = 1.0
    L, g = _check(labels, prob)
    if case == 'all_background':
        assert float(L) == 0.0 and bool((g.view(torch.int32) == 0).all())


def test_nan_probability_and_nan_label_rows_against_the_oracle():
    """Compared with the fp64 oracle only: torch's CUDA BCE would assert on these."""
    BN, D, H, W = 2, 9, 4, 5
    prob = _probs(BN, D, H, W, seed=2)
    labels = _labels('onehot_zero_rows', BN, D, H, W, seed=3)
    labels[0] = 0
    labels[0, 4] = 1.0                                                  # pixel 0 is foreground
    labels[5, 2] = float('nan')                                         # pixel 5 is background
    L, g = _native(labels, prob)
    L64, cnt = ref.loss_ref(labels.cpu(), prob.cpu())
    assert abs(float(L) - float(L64)) <= ref.forward_bound(labels.cpu(), prob.cpu())
    assert bool((g[0, :, 1, 0].view(torch.int32) == 0).all())         # the NaN row (pixel 5 = image 0, y 1, x 0): +0
    bad = prob.clone()
    bad[0, 3, 0, 0] = float('nan')                                      # a NaN in a foreground row
    Lb, gb = _native(labels, bad)
    assert np.isnan(float(Lb)) and np.isnan(float(ref.loss_ref(labels.cpu(), bad.cpu())[0]))
    assert bool(torch.isnan(gb[0, 3, 0, 0]))
    bad = prob.clone()
    bad[0, 3, 1, 0] = float('nan')                                      # ... in the NaN-label (background) row
    Lc, _ = _native(labels, bad)
    assert torch.equal(Lc, L)


def test_two_calls_give_identical_bits():
    BN, D, H, W = SHAPES['cfg2']
    prob = _probs(BN, D, H, W, seed=4)
    labels = _labels('soft', BN, D, H, W, seed=5)
    a, b = _native(labels, prob), _native(labels, prob)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


def test_autocast_does_not_change_the_bits():
    BN, D, H, W = SHAPES['cfg2']
    prob = _probs(BN, D, H, W, seed=6)
    labels = _labels('onehot_zero_rows', BN, D, H, W, seed=7)
    a = _native(labels, prob)
    with torch.autocast('cuda', dtype=torch.bfloat16):
        b = _native(labels, prob)
    assert b[0].dtype == torch.float32 and torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


@pytest.mark.parametrize('kind', ['onehot_zero_rows', 'bins'])
def test_cuda_graph_replay_equals_eager(kind):
    """Capture forward + backward (a host sync would make the capture fail), replay on new inputs."""
    BN, D, H, W = SHAPES['cfg2']
    prob_s = _probs(BN, D, H, W, seed=8).clone()
    lab_s = _labels(kind, BN, D, H, W, seed=9).clone()

    def step():
        x = prob_s.detach().requires_grad_(True)
        L = depth_loss(lab_s, x)
        (gx,) = torch.autograd.grad(L, (x,))
        return L, gx

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            step()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = step()
    for seed in (10, 11):
        p_new, l_new = _probs(BN, D, H, W, seed=seed), _labels(kind, BN, D, H, W, seed=seed + 1)
        prob_s.copy_(p_new)
        lab_s.copy_(l_new)
        graph.replay()
        torch.cuda.synchronize()
        want = _native(l_new, p_new)
        assert torch.equal(out[0], want[0]) and torch.equal(out[1], want[1])


@pytest.mark.parametrize('shape', ['cfg2', 'd113'])
def test_chain_to_the_logits(shape):
    """depth_distribution -> depth_loss -> backward to the logits, against depth_distribution fed torch's gradient."""
    BN, D, H, W = SHAPES[shape]
    g = torch.Generator().manual_seed(13)
    logits = (3 * torch.randn(BN, D + 5, H, W, generator=g)).to(DEV)    # a channel slice, like DepthNet's output
    labels = _labels('onehot_zero_rows', BN, D, H, W, seed=14)
    grads = []
    for loss_fn in (lambda t, p: depth_loss(t, p), lambda t, p: bench_train.depth_loss_ref(t, p, D)):
        x = logits.clone().requires_grad_(True)
        p, _ = depth_distribution(x, D)
        (gx,) = torch.autograd.grad(loss_fn(labels, p), (x,))
        grads.append(gx)
    assert torch.equal(grads[0], grads[1])

"""CPU checks of the depth-loss oracle (oracle/depth_loss_ref.py) against torch's own binary_cross_entropy, of the
float32 emulation of the kernels' order against the derived bound, and of the argument checks of the C ABI and of
``mm_training_b200.ops.depth_loss`` (no device is touched)."""
import ctypes

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import bench_train
from mm_training_b200 import _lib, build
from mm_training_b200.ops.depth_loss import depth_loss
from oracle import depth_loss_ref as ref

EDGE_P = [0.0, 1.0, 1e-30, 1.0 - 2.0 ** -24, 2.0 ** -149, 0.5, 1e-7]


def _softmax_preds(BN, D, H, W, seed, spread=4.0):
    g = torch.Generator().manual_seed(seed)
    return torch.softmax(spread * torch.randn(BN, D, H, W, generator=g), 1)


def _onehot(BN, D, H, W, seed, zero_frac=0.0):
    g = torch.Generator().manual_seed(seed)
    b = torch.randint(0, D, (BN * H * W,), generator=g)
    t = F.one_hot(b, D).float()
    if zero_frac:
        t[torch.rand(t.shape[0], generator=g) < zero_frac] = 0
    return t


def _torch_loss(labels, preds):
    """``bench_train.depth_loss_ref`` in float64 (the reference's ops; its ``.float()`` would round to fp32)."""
    D = preds.shape[1]
    labels = labels.double().reshape(-1, D)
    preds = preds.double().permute(0, 2, 3, 1).contiguous().view(-1, D)
    fg_mask = torch.max(labels, dim=1).values > 0.0
    loss = F.binary_cross_entropy(preds[fg_mask], labels[fg_mask], reduction='none').sum() / max(1.0, fg_mask.sum())
    return 3.0 * loss


def test_float64_restatement_is_the_reference():
    labels, preds = _cases()['zero_rows']
    assert float(_torch_loss(labels, preds)) == pytest.approx(float(bench_train.depth_loss_ref(labels, preds, 7)),
                                                              rel=1e-6)


def _cases():
    BN, D, H, W = 2, 7, 3, 5
    P = BN * H * W
    p = _softmax_preds(BN, D, H, W, 0)
    edge = p.clone().permute(0, 2, 3, 1).reshape(-1, D)
    vals = torch.tensor(EDGE_P, dtype=torch.float32)
    edge[:, :] = vals[torch.arange(P * D) % len(EDGE_P)].view(P, D)
    edge = edge.view(BN, H, W, D).permute(0, 3, 1, 2).contiguous()
    g = torch.Generator().manual_seed(3)
    soft = torch.rand(P, D, generator=g)
    soft[::3] = 0                                                   # zero rows among soft rows
    one_fg = torch.zeros(P, D)
    one_fg[4, 2] = 1.0
    return {
        'onehot': (_onehot(BN, D, H, W, 1), p),
        'onehot_edge_p': (_onehot(BN, D, H, W, 2), edge),
        'soft_edge_p': (soft, edge),
        'zero_rows': (_onehot(BN, D, H, W, 4, zero_frac=0.5), p),
        'all_background': (torch.zeros(P, D), p),
        'one_foreground': (one_fg, edge),
        'labels_4d': (_onehot(BN, D, H, W, 5).view(BN, H, W, D), p),
    }


@pytest.mark.parametrize('name', list(_cases()))
def test_oracle_equals_torch_bce(name):
    labels, preds = _cases()[name]
    L, cnt = ref.loss_ref(labels, preds)
    want = _torch_loss(labels, preds)
    assert torch.allclose(L, want, rtol=1e-14, atol=0), (float(L), float(want))
    assert cnt == int((torch.max(labels.reshape(-1, preds.shape[1]), 1).values > 0).sum())
    if name == 'all_background':
        assert float(L) == 0.0


@pytest.mark.parametrize('name', list(_cases()))
def test_oracle_gradient_equals_fp64_autograd(name):
    labels, preds = _cases()[name]
    x = preds.double().requires_grad_(True)
    (2.5 * _torch_loss(labels, x)).backward()
    got = ref.grad_ref(labels, preds, g=2.5)
    assert torch.allclose(got, x.grad, rtol=1e-14, atol=0)
    fg = ref.foreground(labels.reshape(-1, preds.shape[1]))
    bg_rows = got.permute(0, 2, 3, 1).reshape(-1, preds.shape[1])[~fg]
    assert bool((bg_rows == 0).all())


def test_bins_are_the_one_hot_rows():
    BN, D, H, W = 2, 9, 3, 4
    g = torch.Generator().manual_seed(0)
    bins = torch.randint(-2, D + 2, (BN * H * W,), generator=g).int()
    preds = _softmax_preds(BN, D, H, W, 1)
    t, _ = ref.rows(bins, preds)
    ok = (bins >= 0) & (bins < D)
    assert torch.equal(t[ok], F.one_hot(bins[ok].long(), D).float())
    assert bool((t[~ok] == 0).all())
    L, cnt = ref.loss_ref(bins, preds)
    L2, cnt2 = ref.loss_ref(t, preds)
    assert float(L) == float(L2) and cnt == cnt2 == int(ok.sum())


def test_nan_rows_follow_torch_max():
    t = torch.tensor([[0.0, 1.0, float('nan')], [float('nan'), 0.0, 0.0], [0.0, 0.0, 0.0], [0.0, 0.2, 0.0],
                      [-1.0, 0.0, 0.0], [-0.0, 0.0, 0.0], [float('inf'), 0.0, 0.0]])
    assert torch.equal(ref.foreground(t), torch.max(t, 1).values > 0)
    assert ref.foreground(t).tolist() == [False, False, False, True, False, False, True]


def test_nan_probability_in_a_foreground_row_gives_nan():
    BN, D, H, W = 1, 4, 2, 2
    p = _softmax_preds(BN, D, H, W, 0)
    t = _onehot(BN, D, H, W, 1)
    p[0, 2, 1, 1] = float('nan')
    assert np.isnan(float(ref.loss_ref(t, p)[0])) and np.isnan(ref.loss_f32_emulate(t, p))
    t2 = t.clone()
    t2[3] = float('nan')                                   # the same pixel's label row holds a NaN: background
    L, cnt = ref.loss_ref(t2, p)
    assert np.isfinite(float(L)) and cnt == 3 and np.isfinite(ref.loss_f32_emulate(t2, p))


def _bound_cases():
    out = []
    for seed, (BN, D, H, W) in enumerate([(2, 1, 3, 5), (2, 3, 4, 4), (1, 113, 4, 8), (2, 409, 2, 8), (1, 64, 5, 7)]):
        p = _softmax_preds(BN, D, H, W, seed, spread=2.0 + 4 * seed)
        out.append((f'random_onehot_D{D}', _onehot(BN, D, H, W, seed, zero_frac=0.2), p))
        g = torch.Generator().manual_seed(100 + seed)
        out.append((f'random_soft_D{D}', torch.rand(BN * H * W, D, generator=g), p))
    # adversarial: one term of 100 (clamped log) then many tiny terms that the fp32 pixel sum absorbs
    BN, D, H, W = 1, 409, 2, 16
    p = torch.full((BN, D, H, W), 1e-7)
    p[:, 0] = 0.0
    t = torch.zeros(BN * H * W, D)
    t[:, 0] = 1.0
    out.append(('adversarial_absorption', t, p))
    # adversarial: logs right at the -100 clamp, and p a hair below 1 with a zero label
    p = torch.full((1, 5, 4, 8), float(np.exp(np.float32(-100.0))))
    p[:, 1] = 1.0 - 2.0 ** -24
    p[:, 2] = float(np.float32(np.exp(-99.99)))
    t = torch.zeros(32, 5)
    t[:, 0] = 1.0
    t[::2, 3] = 0.37
    out.append(('adversarial_clamp', t, p))
    # adversarial: soft labels with p near 0 and 1 everywhere
    g = torch.Generator().manual_seed(7)
    p = torch.where(torch.rand(2, 113, 3, 4, generator=g) < 0.5, torch.tensor(1e-30), torch.tensor(1.0 - 2.0 ** -24))
    out.append(('adversarial_extremes', torch.rand(24, 113, generator=g), p))
    return out


@pytest.mark.parametrize('name,labels,preds', _bound_cases(), ids=[c[0] for c in _bound_cases()])
def test_float32_emulation_lies_inside_the_bound(name, labels, preds):
    L64, _ = ref.loss_ref(labels, preds)
    got = float(ref.loss_f32_emulate(labels, preds))
    bound = ref.forward_bound(labels, preds)
    assert abs(got - float(L64)) <= bound, (got, float(L64), bound)
    assert bound <= 1e-4 * abs(float(L64)) + 1e-30            # and it is not vacuous


# ---------------------------------------------------------------------------------------------- argument errors
@pytest.fixture(scope='module')
def L():
    build.build()
    return _lib.lib()


def test_abi_argument_errors_are_codes_not_crashes(L):
    p = ctypes.c_void_p(256)                               # never dereferenced: every call below fails its argument check
    n = ctypes.c_size_t()
    assert L.bevdepth_loss_workspace_bytes(4, 112, 16, 44, ctypes.byref(n)) == 0 and n.value > 0
    assert L.bevdepth_loss_workspace_bytes(4, 112, 16, 44, None) == -1
    assert L.bevdepth_loss_workspace_bytes(0, 112, 16, 44, ctypes.byref(n)) == -1
    assert L.bevdepth_loss_workspace_bytes(2 ** 16, 112, 256, 256, ctypes.byref(n)) == -2

    fwd = lambda prob, lab, bins, bn, d, h, w, ws=p, out=p, cnt=p: L.bevdepth_loss_forward(
        prob, lab, bins, bn, d, h, w, ws, out, cnt, None)
    bwd = lambda prob, lab, bins, bn, d, h, w, ws=p, out=p, cnt=p: L.bevdepth_loss_backward(
        prob, lab, bins, p, cnt, bn, d, h, w, out, None)
    for fn in (fwd, bwd):
        assert fn(None, p, None, 4, 112, 16, 44) == -1                     # null probabilities
        assert fn(p, None, None, 4, 112, 16, 44) == -1                     # neither labels nor bins
        assert fn(p, p, p, 4, 112, 16, 44) == -1                           # both
        assert fn(p, p, None, 4, 112, 16, 44, out=None) == -1              # null output
        assert fn(p, p, None, 4, 112, 16, 44, cnt=None) == -1              # null count
        assert fn(p, p, None, 0, 112, 16, 44) == -1                        # empty batch
        assert fn(p, p, None, 4, 0, 16, 44) == -1                          # no bins
        assert fn(p, None, p, 4, 112, -1, 44) == -1                        # negative height
        assert fn(p, p, None, 4, 112, 16, 0) == -1                         # empty width
        assert fn(p, p, None, 2 ** 16, 112, 256, 256) == -2                # pixels do not fit 31 bits
        assert fn(p, p, None, 4, 4096, 16, 44) == -3                       # too many bins for shared memory
        assert fn(ctypes.c_void_p(258), p, None, 4, 112, 16, 44) == -4     # misaligned probabilities
        assert fn(p, ctypes.c_void_p(257), None, 4, 112, 16, 44) == -4     # misaligned labels
        assert fn(p, None, ctypes.c_void_p(262), 4, 112, 16, 44) == -4     # misaligned bins
    assert fwd(p, p, None, 4, 112, 16, 44, ws=None) == -1                  # null workspace
    assert fwd(p, p, None, 4, 112, 16, 44, ws=ctypes.c_void_p(260)) == -4  # workspace not 8-byte aligned


def test_python_validation_raises_before_device_work():
    preds = torch.rand(2, 5, 3, 4)
    labels = torch.zeros(24, 5)
    with pytest.raises(RuntimeError, match='CUDA tensors only'):
        depth_loss(labels, preds)
    # everything below fails on a "meta" tensor check before the CUDA check could matter: use fake CUDA-ness
    class FakeCuda(torch.Tensor):
        @property
        def is_cuda(self):
            return True

        @classmethod
        def __torch_function__(cls, func, types, args=(), kwargs=None):
            return super().__torch_function__(func, types, args, kwargs or {})

    fc = lambda t: t.as_subclass(FakeCuda)
    with pytest.raises(TypeError, match='float32'):
        depth_loss(fc(labels), fc(preds.half()))
    with pytest.raises(TypeError, match='float32 rows or int32 bins'):
        depth_loss(fc(labels.double()), fc(preds))
    with pytest.raises(TypeError, match='float32 rows or int32 bins'):
        depth_loss(fc(labels.long()), fc(preds))
    with pytest.raises(ValueError, match='do not hold'):
        depth_loss(fc(torch.zeros(23, 5)), fc(preds))
    with pytest.raises(ValueError, match='do not hold'):
        depth_loss(fc(torch.zeros(25, dtype=torch.int32)), fc(preds))
    with pytest.raises(ValueError, match=r'\(B\*N, D, H, W\)'):
        depth_loss(fc(labels), fc(preds[0]))
    with pytest.raises(ValueError, match='require grad'):
        depth_loss(fc(labels.clone().requires_grad_(True)), fc(preds))

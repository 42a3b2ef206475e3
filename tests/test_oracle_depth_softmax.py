"""CPU checks of the depth-distribution oracle (oracle/depth_softmax_ref.py): the float32 emulation of the kernels'
online softmax against torch.softmax on masked and non-finite rows, known answers, the fp64 backward against fp64
autograd of the reference composition, and the soundness of the fp16 / bf16 rounding bracket."""
import math

import numpy as np
import pytest
import torch

from oracle import depth_softmax_ref as ds

NINF, PINF, NAN = -math.inf, math.inf, math.nan


def _rows(rows):
    return np.array(rows, dtype=np.float32)


def _same_nan_pattern_and_close(ours, ref, rtol=2e-6):
    ours = torch.from_numpy(np.asarray(ours)).double()
    assert torch.equal(torch.isnan(ours), torch.isnan(ref))
    ok = ~torch.isnan(ref)
    assert torch.allclose(ours[ok], ref[ok], rtol=rtol, atol=ds.FLT_MIN)        # fp32 underflow: e^-160 -> 0


MASKED = [
    [NINF, 1.0, 2.0, 0.5],                 # leading -inf (near bins masked)
    [NINF, NINF, NINF, 0.25],              # all but one masked: the survivor is exactly 1
    [0.5, 1.0, NINF, NINF],                # trailing
    [NINF, 3.0, NINF, -2.0],               # interleaved
    [1.0, NINF, 2.0, NINF],
    [-80.0, NINF, 80.0, 0.0],              # wide range: underflow to 0 next to a -inf
]
NON_FINITE = [
    [NINF, NINF, NINF, NINF],              # all masked: NaN everywhere (0 / 0), as torch
    [PINF, 1.0, 2.0, 3.0],                 # +inf anywhere: NaN row
    [1.0, 2.0, PINF, NINF],
    [NINF, PINF, NINF, NINF],
    [NAN, 1.0, 2.0, 3.0],                  # NaN anywhere: NaN row
    [1.0, 2.0, 3.0, NAN],
    [NINF, NAN, NINF, 0.0],
]


@pytest.mark.parametrize('rows', [MASKED, NON_FINITE], ids=['masked', 'non_finite'])
def test_emulation_matches_torch_softmax(rows):
    x = _rows(rows)
    torch_ref = torch.softmax(torch.from_numpy(x).double(), 1)
    _same_nan_pattern_and_close(ds.online_softmax_f32(x), torch_ref)
    ref = ds.softmax_ref(torch.from_numpy(x).view(len(rows), 4, 1, 1), 4).view(len(rows), 4)
    assert torch.equal(torch.isnan(ref), torch.isnan(torch_ref))
    ok = ~torch.isnan(ref)
    assert torch.allclose(ref[ok], torch_ref[ok], rtol=4 * 2.0 ** -53, atol=0)    # fp64 rounding of exp / sum


def test_masked_bins_are_exact_zeros_and_a_single_survivor_is_one():
    p = ds.online_softmax_f32(_rows(MASKED))
    assert np.all(p[np.isneginf(_rows(MASKED))] == 0)
    assert p[1].tolist() == [0.0, 0.0, 0.0, 1.0]
    assert not np.isnan(p).any()
    assert np.isnan(ds.online_softmax_f32(_rows(NON_FINITE))).all()


def test_loop_without_the_neg_inf_guard_turns_a_leading_mask_into_nan():
    # the reason for the guard: with m still -inf, exp(l - m) = exp(-inf + inf) = exp(NaN) poisons the sum
    x = _rows([[NINF, 1.0, 2.0], [1.0, NINF, 2.0]])
    old = ds.online_softmax_f32(x, skip_neg_inf=False)
    assert np.isnan(old[0]).all()
    assert not np.isnan(old[1]).any()                       # only a LEADING -inf broke the loop
    new = ds.online_softmax_f32(x)
    assert np.allclose(new[0], [0.0, 0.26894142, 0.73105858], rtol=1e-6, atol=0)


@pytest.mark.parametrize('D', [1, 2, 3, 7, 112, 409])
def test_constant_logits_give_exactly_one_over_d(D):
    x = np.full((3, D), [[-5.0], [0.0], [17.25]], dtype=np.float32)
    p = ds.online_softmax_f32(x)
    assert np.array_equal(p, np.full_like(p, np.float32(1.0) / np.float32(D)))


def test_single_bin_gives_one_and_no_gradient():
    x = torch.tensor([[-3.0], [0.0], [50.0]]).view(3, 1, 1, 1)
    assert ds.online_softmax_f32(x.view(3, 1).numpy()).tolist() == [[1.0], [1.0], [1.0]]
    p = ds.softmax_ref(x, 1)
    assert torch.equal(p, torch.ones_like(p))
    g, mag = ds.softmax_backward_ref(p.float(), torch.randn(3, 1, 1, 1), torch.randn(3, 1, 1, 1))
    assert torch.equal(g, torch.zeros_like(g))


def test_zero_and_ln3_give_a_quarter_and_three_quarters():
    x = _rows([[0.0, math.log(3.0)]])
    assert np.allclose(ds.online_softmax_f32(x), [[0.25, 0.75]], rtol=3e-7, atol=0)
    p = ds.softmax_ref(torch.from_numpy(x).view(1, 2, 1, 1), 2).view(2)
    assert torch.allclose(p, torch.tensor([0.25, 0.75], dtype=torch.float64), rtol=1e-7, atol=0)


def test_emulation_is_within_the_forward_bound():
    g = torch.Generator().manual_seed(0)
    x = torch.cat([torch.randn(200, 409, generator=g) * 3, (torch.rand(200, 409, generator=g) * 2 - 1) * 80,
                   torch.linspace(-20, 20, 409).expand(4, 409)])           # increasing rows: the max rises every step
    x[::7, :50] = NINF
    p = torch.from_numpy(ds.online_softmax_f32(x.numpy())).double()
    x4 = x.view(*x.shape, 1, 1)
    ref = ds.softmax_ref(x4, 409).view(-1, 409)
    bound = ds.forward_rel_bound(x4, 409).view(-1, 409)
    assert bool(((p - ref).abs() <= bound * ref + ds.FLT_MIN).all())


@pytest.mark.parametrize('with_oracle', [False, True])
def test_backward_matches_fp64_autograd_of_the_reference_composition(with_oracle):
    g = torch.Generator().manual_seed(1)
    BN, D, H, W = 3, 17, 4, 5
    logits = (torch.randn(BN, D, H, W, generator=g, dtype=torch.float64) * 3)
    logits[0, :4] = NINF
    oracle = None
    if with_oracle:
        oracle = torch.nn.functional.one_hot(torch.randint(0, D, (BN, H, W), generator=g), D).permute(0, 3, 1, 2).double()
        oracle = oracle * (torch.rand(BN, 1, H, W, generator=g, dtype=torch.float64) < 0.5)
        oracle[1, :, 0, 0] = -0.0
        oracle[1, :3, 1, 1] = -1.0
    w1 = torch.randn(BN, D, H, W, generator=g, dtype=torch.float64)
    w2 = torch.randn(BN, D, H, W, generator=g, dtype=torch.float64)
    x = logits.clone().requires_grad_(True)
    p = torch.softmax(x, 1)
    used = ds.overwrite_ref(p, oracle) if with_oracle else p
    ((p * w1).sum() + (used * w2).sum()).backward()
    ours, mag = ds.softmax_backward_ref(p.detach(), w1, w2, oracle)
    assert torch.allclose(ours, x.grad, rtol=1e-12, atol=1e-15)
    assert bool((ours[0, :4] == 0).all()) and bool((mag >= ours.abs()).all())


# ---------------------------------------------------------------------------------------------- rounding bracket
def _grid_near(values):
    """fp32 values at, and one and two fp32 ulps on either side of, each of ``values``."""
    v = torch.tensor(values, dtype=torch.float32)
    out = [v]
    for direction in (math.inf, -math.inf):
        w = v
        for _ in range(2):
            w = torch.nextafter(w, torch.full_like(w, direction))
            out.append(w)
    return torch.cat(out)


def _ties(dtype):
    """Midpoints between consecutive ``dtype`` numbers (ties of the fp32 -> dtype rounding), normal and subnormal."""
    fi = torch.finfo(dtype)
    base = torch.tensor([1.0, 1.5, 3.0, 1000.0, fi.tiny, fi.tiny * 3, fi.max / 2, fi.smallest_normal * 0.5,
                         fi.tiny * 0.25], dtype=torch.float32).to(dtype)
    nxt = torch.nextafter(base, torch.full_like(base, math.inf))
    ties = (base.float() + nxt.float()) / 2                     # exact in fp32: dtype has fewer mantissa bits
    return (ties.tolist() + [-t for t in ties.tolist()]
            + [2.0 ** -24, 2.0 ** -25, 3 * 2.0 ** -26, 2.0 ** -133, 2.0 ** -134, 2.0 ** -149])


@pytest.mark.parametrize('dtype', [torch.float16, torch.bfloat16])
def test_round_bracket_contains_every_fp32_value_within_err(dtype):
    extra = [65504.0, 65519.0, 65520.0, 65536.0, -65520.0] if dtype == torch.float16 else [3.3895e38]
    vals = _grid_near(_ties(dtype) + extra)                    # candidate kernel values (fp32)
    g = torch.Generator().manual_seed(2)
    for _ in range(20):
        # references within err of each value: at the value, and shifted by up to err either way
        err = vals.double().abs() * float(torch.rand(1, generator=g)) * 2.0 ** -22 + ds.FLT_TRUE_MIN
        shift = (torch.rand(vals.shape, generator=g, dtype=torch.float64) * 2 - 1) * err
        ref = vals.double() + shift
        lo, hi = ds.round_bracket(ref, err, dtype)
        assert bool(ds.in_bracket(vals.to(dtype), lo, hi).all())
    # exact references bracket to a single value; fp16 overflow lands on inf on both sides
    lo, hi = ds.round_bracket(vals.double(), 0.0, dtype)
    assert torch.equal(lo, vals.to(dtype)) and torch.equal(hi, vals.to(dtype))
    if dtype == torch.float16:
        lo, hi = ds.round_bracket(torch.tensor([65520.0, 65519.0], dtype=torch.float64), 0.0, dtype)
        assert lo.tolist() == hi.tolist() == [math.inf, 65504.0]


@pytest.mark.parametrize('dtype', [torch.float16, torch.bfloat16])
def test_round_bracket_rejects_a_value_off_by_one_half_ulp(dtype):
    x = torch.tensor([1.0, 3.0, 1000.0, 0.0078125], dtype=torch.float64)
    lo, hi = ds.round_bracket(x, x * 2.0 ** -20, dtype)
    assert torch.equal(lo, hi)                                 # a tight error keeps the bracket to one value
    off = torch.nextafter(x.to(dtype), torch.full_like(x, math.inf).to(dtype))
    assert not bool(ds.in_bracket(off, lo, hi).any())


def test_sum_bound_is_gamma_n():
    assert ds.sum_bound(0, 5.0) == 0.0
    b = ds.sum_bound(80, 1.0)
    assert 80 * 2.0 ** -24 < b < 80.01 * 2.0 ** -24

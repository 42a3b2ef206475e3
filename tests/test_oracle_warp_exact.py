"""CPU checks of the float32 emulation of the BDA warp kernels (oracle/warp_exact_ref.py): its ``fmaf`` equals exact
rational rounding, its forward lies within the fp64 bound of tests/test_gpu_bev_warp.py, its backward is the exact
transpose of its forward, and known answers on singular / non-finite theta and on coordinates that sit on integers."""
import math
from fractions import Fraction

import numpy as np
import pytest
import torch

from oracle import warp_affine_ref as wr
from oracle import warp_exact_ref as we
from oracle.warp_affine_ref import about_centre, bda_matrices

f32 = np.float32
FLT_MAX = float(np.finfo(f32).max)


# ---------------------------------------------------------------------------------------------- fmaf
def _round_f32(x: Fraction, zero_sign: float) -> float:
    """Round an exact rational to float32, nearest even, with subnormals and overflow; ``zero_sign`` is the sign an
    exact zero takes."""
    if x == 0:
        return math.copysign(0.0, zero_sign)
    sign, m = (-1.0 if x < 0 else 1.0), abs(x)
    e = m.numerator.bit_length() - m.denominator.bit_length()
    if Fraction(2) ** e > m:
        e -= 1
    q = Fraction(2) ** (max(e, -126) - 23)                  # spacing of float32 values in m's binade
    n = m / q
    k = n.numerator // n.denominator
    rem = n - k
    if rem > Fraction(1, 2) or (rem == Fraction(1, 2) and k % 2 == 1):
        k += 1
    v = k * q
    if v >= Fraction(2) ** 128:
        return sign * math.inf
    return sign * float(v)


def _fma_exact(a, b, c) -> float:
    a, b, c = float(a), float(b), float(c)
    if not (math.isfinite(a) and math.isfinite(b) and math.isfinite(c)):
        return float(np.float64(a) * np.float64(b) + np.float64(c))          # inf / NaN follow IEEE, no rounding
    p, s = Fraction(a) * Fraction(b), Fraction(a) * Fraction(b) + Fraction(c)
    p_neg = math.copysign(1.0, a) * math.copysign(1.0, b) < 0
    zero_sign = -1.0 if (p == 0 and p_neg and math.copysign(1.0, c) < 0) else 1.0
    return _round_f32(s, zero_sign)


def _assert_fma_matches(a, b, c):
    a, b, c = (np.asarray(v, dtype=f32).ravel() for v in (a, b, c))
    got = we.fmaf(a, b, c)
    ref = np.array([_fma_exact(x, y, z) for x, y, z in zip(a, b, c)], dtype=np.float64).astype(f32)
    nan = np.isnan(ref)
    assert np.array_equal(np.isnan(got), nan)
    bad = np.nonzero(got.view(np.int32)[~nan] != ref.view(np.int32)[~nan])[0]
    assert bad.size == 0, [(a[~nan][i], b[~nan][i], c[~nan][i], got[~nan][i], ref[~nan][i]) for i in bad[:5]]


def _bits(n, gen, lo=0, hi=0xFF):
    """Random float32 values with full mantissas and exponents drawn in [lo, hi] (biased), both signs."""
    man = gen.integers(0, 1 << 23, n, dtype=np.int64)
    exp = gen.integers(lo, hi + 1, n, dtype=np.int64)
    sgn = gen.integers(0, 2, n, dtype=np.int64)
    v = ((sgn << 31) | (exp << 23) | man).astype(np.uint32).view(f32)
    return np.where(np.isfinite(v), v, f32(1.5))


def test_fmaf_random_triples():
    gen = np.random.default_rng(1)
    n = 20000
    _assert_fma_matches(_bits(n, gen, 100, 150), _bits(n, gen, 100, 150), _bits(n, gen, 90, 160))
    _assert_fma_matches(_bits(n, gen, 1, 254), _bits(n, gen, 1, 254), _bits(n, gen, 0, 254))
    x = gen.standard_normal((3, n)).astype(f32)
    _assert_fma_matches(*x)


def test_fmaf_adversarial_triples():
    gen = np.random.default_rng(2)
    n = 4000
    a = _bits(n, gen, 120, 135)
    b = _bits(n, gen, 120, 135)
    p = a.astype(np.float64) * b.astype(np.float64)
    hi = p.astype(f32)
    # catastrophic cancellation: c = -fl32(a*b), the result is the product's rounding error (exact)
    _assert_fma_matches(a, b, -hi)
    # exact ties: a*b with a 25-bit significand added to 0 sits halfway between two floats
    odd = (gen.integers(1 << 23, 1 << 24, n) | 1).astype(f32)
    _assert_fma_matches(odd, np.full(n, 0.5, f32), np.zeros(n, f32))
    _assert_fma_matches(odd, np.full(n, 0.5, f32), -np.zeros(n, f32))
    # one tiny addend past a tie: the tie must break toward the addend (the double-rounding case)
    tiny = np.ldexp(np.ones(n, f32), gen.integers(-140, -60, n)).astype(f32)
    _assert_fma_matches(odd, np.full(n, 0.5, f32), tiny)
    _assert_fma_matches(odd, np.full(n, 0.5, f32), -tiny)
    # a product whose float64 sum with c rounds onto a float32 midpoint although the exact sum is not one
    big = (odd * f32(2 ** 20)).astype(f32)
    _assert_fma_matches(big, np.full(n, 2.0 ** -21, f32), np.ldexp(np.ones(n), -60).astype(f32))
    # underflow: subnormal results, ties between subnormals, results that round to +-0
    sa = _bits(n, gen, 50, 80)
    sb = _bits(n, gen, 50, 80)
    _assert_fma_matches(sa, sb, np.zeros(n, f32))
    _assert_fma_matches(sa, sb, _bits(n, gen, 0, 3))
    _assert_fma_matches(np.full(n, 2.0 ** -75, f32), np.full(n, 2.0 ** -75, f32), -_bits(n, gen, 0, 0))
    _assert_fma_matches(odd, np.full(n, 2.0 ** -173, f32), np.zeros(n, f32))             # ties at 2^-150
    _assert_fma_matches(-sa, np.abs(sb) * f32(2 ** -40), np.zeros(n, f32))              # -> -0
    _assert_fma_matches(-sa, np.abs(sb) * f32(2 ** -40), -np.zeros(n, f32))
    # overflow: products past FLT_MAX, the FLT_MAX / inf tie with a nudge either way, signed zeros
    _assert_fma_matches(_bits(n, gen, 190, 200), _bits(n, gen, 190, 200), _bits(n, gen, 100, 254))
    m = f32(FLT_MAX)
    half_ulp = f32(2.0 ** 103)
    _assert_fma_matches([m, m, m, -m, m, m], [1, 1, 1, 1, 1, -1],
                        [half_ulp, np.nextafter(half_ulp, f32(0)), -half_ulp, -half_ulp, 0, 0])
    _assert_fma_matches([1.5, 2 ** 64, 2 ** 64, 2 ** 64], [2.0 ** 127, 2 ** 64, 2 ** 64, -(2 ** 64)],
                        [0, -(2.0 ** 103), 2.0 ** 103 * 1.5, 2.0 ** 103])
    _assert_fma_matches([0, -0.0, 0, -0.0, 0], [1, 1, -1, 1, 5], [-0.0, -0.0, -0.0, 0, -0.0])
    got = we.fmaf([np.inf, np.inf, np.nan, 1], [0, 1, 1, 1], [0, -np.inf, 0, np.inf])
    assert np.isnan(got[:3]).all() and got[3] == np.inf


# ---------------------------------------------------------------------------------------------- taps and forward
SHAPES = {'cfg2': (8, 80, 64, 512, (64, 512)), 'sweep128': (2, 80, 128, 128, (128, 128)),
          'odd7x9': (2, 4, 7, 9, (7, 9)), 'resize': (2, 16, 48, 40, (56, 36))}
MATS = ['bda', 'identity', 'flips', 'translate', 'rot90', 'mag2', 'min05', 'singular']


def make_mats(kind: str, B: int, H: int, W: int) -> torch.Tensor:
    eye = torch.eye(2, dtype=torch.float64).expand(B, 2, 2)
    if kind == 'bda':
        return bda_matrices(B, H, W)
    if kind == 'singular':
        return torch.zeros(B, 2, 3)
    lin = {'identity': eye, 'mag2': 2 * eye, 'min05': 0.5 * eye,
           'flips': torch.diag_embed(torch.tensor([[-1.0, 1.0], [1.0, -1.0], [-1.0, -1.0]], dtype=torch.float64)[torch.arange(B) % 3]),
           'translate': eye, 'rot90': torch.tensor([[0.0, -1.0], [1.0, 0.0]], dtype=torch.float64).expand(B, 2, 2)}[kind]
    m = about_centre(lin, H, W)
    if kind == 'translate':
        m[:, 0, 2], m[:, 1, 2] = 3.0, -2.0
    return m.float()


def _theta32(M, src_hw, dsize) -> np.ndarray:
    from mm_training_b200.ops.bev_augment import warp_theta
    return warp_theta(M, src_hw, dsize).numpy()


@pytest.mark.parametrize('kind', MATS)
@pytest.mark.parametrize('shape', list(SHAPES))
def test_emulated_forward_lies_within_the_fp64_bound(shape, kind):
    B, C, H, W, dsize = SHAPES[shape]
    if shape == 'cfg2':
        B, C = 2, 8
    g = torch.Generator().manual_seed(11)
    x = torch.rand(B, C, H, W, generator=g) - 0.5
    M = make_mats(kind, B, H, W)
    th = _theta32(M, (H, W), dsize)
    out = torch.from_numpy(we.warp_forward_exact(th, x.permute(0, 2, 3, 1).numpy(), dsize)).permute(0, 3, 1, 2)
    if kind == 'singular':
        assert not np.isfinite(th).all() and bool((out == 0).all())
        return
    ref64 = wr.warp_affine_ref(x.double(), M, dsize)
    S = wr.tap_sum_ref(x.abs(), M, dsize)
    bound = 1e-5 * ref64.abs() + 8 * 2.0 ** -23 * max(H, W) * S + 1e-30
    err = (out.double() - ref64).abs()
    assert bool((err <= bound).all()), float(err.max())


def _rot(a):
    return torch.tensor([[math.cos(a), -math.sin(a)], [math.sin(a), math.cos(a)]], dtype=torch.float64)


SMALL = [((5, 7), (5, 7)), ((4, 6), (9, 5)), ((2, 2), (7, 6)), ((6, 5), (2, 3))]
LINEAR = {'rot37': _rot(0.65), 'shear': torch.tensor([[1.0, 0.8], [0.0, 1.0]], dtype=torch.float64),
          'aniso': torch.tensor([[3.0, 0.0], [0.0, 0.3]], dtype=torch.float64), 'mag3': 3 * torch.eye(2, dtype=torch.float64),
          'near_singular': _rot(0.3) @ torch.diag(torch.tensor([1.0, 100.0], dtype=torch.float64)) @ _rot(1.1),
          'half_pixel': torch.eye(2, dtype=torch.float64)}


@pytest.mark.parametrize('kind', list(LINEAR))
@pytest.mark.parametrize('hw', SMALL)
def test_emulated_backward_is_the_transpose_of_the_emulated_forward(hw, kind):
    (Hs, Ws), (Hd, Wd) = hw
    M = about_centre(LINEAR[kind][None], Hs, Ws)
    if kind == 'half_pixel':
        M[0, 0, 2] += 0.5
    th = _theta32(M.float(), (Hs, Ws), (Hd, Wd))
    n_s, n_d = Hs * Ws, Hd * Wd
    for value in (1.0, math.inf):                          # inf: zero-weight pairs become NaN on both sides
        fwd = we.operator_matrix(th, Hs, Ws, Hd, Wd, value)[0]                                  # (n_d, n_s)
        basis = np.zeros((1, Hd, Wd, n_d), dtype=f32)
        basis.reshape(n_d, n_d)[np.arange(n_d), np.arange(n_d)] = f32(value)
        bwd = we.warp_backward_exact(th, basis, (Hs, Ws)).reshape(n_s, n_d)
        assert np.array_equal(np.isnan(fwd.T), np.isnan(bwd))
        ok = ~np.isnan(bwd)
        assert np.array_equal(fwd.T[ok].view(np.int32), bwd[ok].view(np.int32))
    if hw == SMALL[0]:                                     # same grids, centre fixed: the map has taps to compare
        assert np.count_nonzero(fwd) > 0


# ---------------------------------------------------------------------------------------------- known answers
@pytest.mark.parametrize('th', [np.zeros(6), [np.nan, 0, 0, 0, 1, 0], [1, 0, np.inf, 0, 1, 0], [1, 0, 0, 0, 1, -np.inf],
                                [np.inf, 0, 0, 0, 1, 0]])
def test_singular_or_non_finite_theta_gives_no_taps(th):
    th = np.asarray(th, dtype=f32).reshape(1, 2, 3)
    taps = we.warp_taps(th, 5, 6, 7, 8)
    if not np.isfinite(th).all():
        assert not taps.valid.any()
    else:                                                       # all-zero theta: every pixel samples the centre
        assert taps.valid.all() and bool((taps.x0 == 2).all()) and bool((taps.y0 == 2).all())
    src = np.full((1, 5, 6, 4), np.inf, dtype=f32)
    out = we.warp_forward_exact(th, src, (7, 8))
    assert (not np.isfinite(th).all()) == bool((out == 0).all())


def test_coordinate_on_an_integer_keeps_both_taps_one_with_weight_zero():
    # identity: every coordinate is an integer, so ne / sw / se carry weight 0 but stay valid inside the grid
    th = np.array([[[1, 0, 0], [0, 1, 0]]], dtype=f32)
    taps = we.warp_taps(th, 5, 9, 5, 9)
    assert np.array_equal(taps.x0[0], np.broadcast_to(np.arange(9), (5, 9)))
    assert bool((taps.w[..., 0] == 1).all()) and bool((taps.w[..., 1:] == 0).all())
    assert taps.valid[0, :4, :8].all() and not taps.valid[0, 4, :, 2:].any() and not taps.valid[0, :, 8, 1::2].any()
    assert np.signbit(taps.w[..., 1:]).sum() == 0                            # +0, never -0
    # half-pixel shift along x (x = d - 0.5 exactly on a 5x5 grid): both x taps at 0.5, on an integer in y
    th = np.array([[[1, 0, -0.25], [0, 1, 0]]], dtype=f32)
    taps = we.warp_taps(th, 5, 5, 5, 5)
    assert np.array_equal(taps.x0[0], np.broadcast_to(np.arange(-1, 4), (5, 5)))
    assert bool((taps.w[0, :, 1:, :2] == 0.5).all()) and bool((taps.w[0, :, 1:, 2:] == 0).all())
    # an inf source value on a zero-weight tap is NaN (fmaf(inf, 0, acc)), on the full-weight tap inf
    src = np.zeros((1, 5, 9, 4), dtype=f32)
    src[0, 2, 3] = np.inf
    out = we.warp_forward_exact(np.array([[[1, 0, 0], [0, 1, 0]]], dtype=f32), src, (5, 9))
    assert np.isinf(out[0, 2, 3]).all() and np.isnan(out[0, 2, 2]).all() and np.isnan(out[0, 1, 3]).all()
    assert np.isnan(out[0, 1, 2]).all() and np.count_nonzero(np.isnan(out)) == 12


def test_skipping_an_empty_cell_keeps_a_negative_zero_reading_it_does_not():
    # a negative value times a tiny weight underflows to -0; the next tap on a zero row gives +0 (-0 + 0 = +0), while
    # skipping that tap (the cell is empty) keeps -0: equal values, different bits
    Hs, Ws = 3, 4
    th = np.array([[[1, 0, -3e-7], [0, 1, 0]]], dtype=f32)        # x just below an integer: the nw weight is tiny
    taps = we.warp_taps(th, Hs, Ws, Hs, Ws)
    d = (1, 1)
    w = taps.w[0, d[0], d[1]]
    assert taps.valid[0, d[0], d[1]].all() and 0 < w[0] < 1e-5 and w[1] > 0.99
    src = np.zeros((1, Hs, Ws, 4), dtype=f32)
    x0, y0 = taps.x0[0, d[0], d[1]], taps.y0[0, d[0], d[1]]
    src[0, y0, x0] = -np.float32(2.0 ** -140)                                    # nw: -tiny * tiny -> -0
    cs = np.zeros(Hs * Ws + 1, dtype=np.int32)
    cs[1 + y0 * Ws + x0:] = 1                                                     # only the nw cell is occupied
    skipped = we.warp_forward_exact(th, src, (Hs, Ws), cell_start=cs)[0, d[0], d[1]]
    read = we.warp_forward_exact(th, src, (Hs, Ws))[0, d[0], d[1]]
    assert bool((skipped == 0).all()) and bool((read == 0).all())
    assert np.signbit(skipped).all() and not np.signbit(read).any()

"""CPU checks of the BEV augmentation warp: the kornia restatement in oracle/warp_affine_ref.py is pinned by known
answers (kornia is not installed), the op's own theta equals the oracle's, and the C ABI / Python op reject bad
arguments without touching a device."""
import ctypes

import pytest
import torch

from mm_training_b200 import _lib, build
from mm_training_b200.ops.bev_augment import warp_theta
from oracle import warp_affine_ref as wr

DTYPES = [torch.float32, torch.float64]


def _m(rows, B=1):
    return torch.tensor(rows, dtype=torch.float64).expand(B, 2, 3).clone()


def _x(B, C, H, W, dtype, seed=0):
    return torch.rand(B, C, H, W, generator=torch.Generator().manual_seed(seed), dtype=torch.float64).to(dtype)


def _close(a, b, dtype):
    tol = 1e-5 if dtype == torch.float32 else 1e-12
    return torch.allclose(a.double(), b.double(), rtol=tol, atol=tol)


@pytest.mark.parametrize('dtype', DTYPES)
def test_identity_gives_the_input(dtype):
    x = _x(2, 3, 5, 7, dtype)
    assert _close(wr.warp_affine_ref(x, _m([[1, 0, 0], [0, 1, 0]], 2), (5, 7), dtype), x, dtype)


@pytest.mark.parametrize('dtype', DTYPES)
def test_flips(dtype):
    B, C, H, W = 2, 3, 5, 7
    x = _x(B, C, H, W, dtype)
    assert _close(wr.warp_affine_ref(x, _m([[-1, 0, W - 1], [0, 1, 0]], B), (H, W), dtype), torch.flip(x, [-1]), dtype)
    assert _close(wr.warp_affine_ref(x, _m([[1, 0, 0], [0, -1, H - 1]], B), (H, W), dtype), torch.flip(x, [-2]), dtype)


@pytest.mark.parametrize('dtype', DTYPES)
def test_integer_translation_shifts_with_zero_fill(dtype):
    H, W, tx, ty = 6, 8, 3, -2
    x = _x(1, 2, H, W, dtype)
    out = wr.warp_affine_ref(x, _m([[1, 0, tx], [0, 1, ty]]), (H, W), dtype)
    ref = torch.zeros_like(x)
    ref[..., max(ty, 0):H + min(ty, 0), max(tx, 0):W + min(tx, 0)] = x[..., max(-ty, 0):H - max(ty, 0), max(-tx, 0):W - max(tx, 0)]
    assert _close(out, ref, dtype)


@pytest.mark.parametrize('dtype', DTYPES)
def test_half_pixel_shift_is_the_mean_of_the_two_neighbours(dtype):
    x = _x(1, 2, 4, 6, dtype)
    out = wr.warp_affine_ref(x, _m([[1, 0, 0.5], [0, 1, 0]]), (4, 6), dtype)   # destination x samples source x - 0.5
    assert _close(out[..., 1:], (x[..., :-1] + x[..., 1:]) / 2, dtype)
    assert _close(out[..., 0], x[..., 0] / 2, dtype)                            # the other neighbour is zero padding


@pytest.mark.parametrize('dtype', DTYPES)
def test_rotation_by_90_degrees_about_the_centre(dtype):
    # M maps source pixel (x, y) to destination (2 - y, x) on a 3x3 grid: the top-right source pixel (2, 0) lands at the
    # bottom-right (2, 2), i.e. dst[y'][x'] = src[2 - x'][y'] -- a clockwise quarter turn as the image is displayed.
    src = torch.arange(9, dtype=dtype).view(1, 1, 3, 3)
    hand = torch.tensor([[6, 3, 0], [7, 4, 1], [8, 5, 2]], dtype=dtype).view(1, 1, 3, 3)
    out = wr.warp_affine_ref(src, _m([[0, -1, 2], [1, 0, 0]]), (3, 3), dtype)
    assert _close(out, hand, dtype)
    assert torch.equal(torch.rot90(src, -1, [-2, -1]), hand)
    n = 6
    x = _x(2, 3, n, n, dtype)
    assert _close(wr.warp_affine_ref(x, _m([[0, -1, n - 1], [1, 0, 0]], 2), (n, n), dtype), torch.rot90(x, -1, [-2, -1]), dtype)


@pytest.mark.parametrize('dtype', DTYPES)
def test_op_theta_equals_the_oracle_theta(dtype):
    g = torch.Generator().manual_seed(3)
    M = torch.randn(4, 2, 3, generator=g, dtype=torch.float64).to(dtype)
    M[:, :, 2] *= 20
    for src_hw, dsize in [((64, 512), (64, 512)), ((7, 9), (11, 5))]:
        ours = warp_theta(M, src_hw, dsize)
        assert ours.dtype == torch.float32 and ours.shape == (4, 2, 3)
        assert torch.allclose(ours.double(), wr.theta_ref(M, src_hw, dsize), rtol=1e-5, atol=1e-5)


def test_tap_sum_counts_in_grid_taps():
    x = torch.ones(1, 1, 4, 5, dtype=torch.float64)
    s = wr.tap_sum_ref(x, _m([[1, 0, 0.5], [0, 1, 0.5]]), (4, 5))
    assert s[0, 0, 2, 2] == 4 and s[0, 0, 0, 0] == 1 and s[0, 0, 0, 2] == 2


# ---------------------------------------------------------------------------------------------- argument errors
@pytest.fixture(scope='module')
def L():
    build.build()
    return _lib.lib()


def test_abi_argument_errors_are_codes_not_crashes(L):
    p = ctypes.c_void_p(256)                           # never dereferenced: every call below fails its argument check
    for fn in (L.bevpool_warp_affine_forward, L.bevpool_warp_affine_backward):
        assert fn(None, p, 80, p, 80, None, 2, 80, 64, 512, 64, 512, None) == -1        # null theta
        assert fn(p, None, 80, p, 80, None, 2, 80, 64, 512, 64, 512, None) == -1        # null input
        assert fn(p, p, 80, None, 80, None, 2, 80, 64, 512, 64, 512, None) == -1        # null output
        assert fn(p, p, 82, p, 82, None, 2, 82, 64, 512, 64, 512, None) == -3           # C % 4 != 0
        assert fn(p, p, 78, p, 80, None, 2, 80, 64, 512, 64, 512, None) == -1           # stride < C
        assert fn(p, p, 80, p, 90, None, 2, 80, 64, 512, 64, 512, None) == -1           # stride not a multiple of 4
        assert fn(p, p, 80, p, 80, None, 2, 80, 1, 512, 64, 512, None) == -1            # a 1-row grid
        assert fn(p, p, 80, p, 80, None, 0, 80, 64, 512, 64, 512, None) == -1           # empty batch
        assert fn(p, p, 80, p, 80, None, 2 ** 20, 80, 64, 512, 64, 512, None) == -2     # cells do not fit 31 bits
        assert fn(p, ctypes.c_void_p(260), 80, p, 80, None, 2, 80, 64, 512, 64, 512, None) == -4   # misaligned rows


def test_python_op_refuses_bad_arguments():
    from mm_training_b200.ops import warp_affine
    x, M = torch.zeros(1, 4, 3, 3), _m([[1, 0, 0], [0, 1, 0]]).float()
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        warp_affine(x, M, (3, 3))
    for kw in ({'mode': 'nearest'}, {'padding_mode': 'border'}, {'align_corners': False}):
        with pytest.raises(ValueError):
            warp_affine(x, M, (3, 3), **kw)
    with pytest.raises(ValueError, match='gradient'):
        warp_theta(M.clone().requires_grad_(True), (3, 3), (3, 3))
    with pytest.raises(ValueError):
        warp_theta(M, (1, 3), (3, 3))

"""CPU checks of the LiDAR BEV nearest resampling (csrc/bev_resample.cu): the library's index maps equal torch's
F.interpolate(mode='nearest') maps, its preimage bounds are the adjoint of those maps, and the C ABI / Python op reject
bad arguments without touching a device."""
import ctypes
import random
import types

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from mm_training_b200 import _lib, build
from mm_training_b200.ops.voxel_pooling import voxel_pooling_fused_concat

PAIRS = [(32, 64), (256, 512), (256, 64), (2048, 512), (64, 64), (48, 64), (200, 512), (700, 512), (300, 64), (1, 64),
         (64, 1), (100, 64), (48, 64), (2048, 1), (1, 1), (3, 2048)]


def _sweep(n=300, seed=0):
    r = random.Random(seed)
    return [(r.randint(1, 2048), r.randint(1, 2048)) for _ in range(n)]


@pytest.fixture(scope='module')
def L():
    build.build()
    return _lib.lib()


def _maps(L, n_in, n_out):
    src = (ctypes.c_int32 * n_out)()
    first = (ctypes.c_int32 * (n_in + 1))()
    assert L.bevpool_resize_nearest_index(n_in, n_out, src, first) == 0
    return np.frombuffer(src, dtype=np.int32).copy(), np.frombuffer(first, dtype=np.int32).copy()


def _torch_map(n_in, n_out, axis):
    """Source index of every destination position along one axis, as F.interpolate picks it (values are exact in fp32)."""
    if axis == 'x':
        x = torch.arange(n_in, dtype=torch.float32).view(1, 1, 1, n_in)
        return F.interpolate(x, size=(1, n_out), mode='nearest').view(-1).long().numpy()
    x = torch.arange(n_in, dtype=torch.float32).view(1, 1, n_in, 1)
    return F.interpolate(x, size=(n_out, 1), mode='nearest').view(-1).long().numpy()


@pytest.mark.parametrize('axis', ['x', 'y'])
def test_index_maps_equal_torch_nearest(L, axis):
    for n_in, n_out in PAIRS + _sweep():
        src, _ = _maps(L, n_in, n_out)
        assert np.array_equal(src, _torch_map(n_in, n_out, axis)), (n_in, n_out)


def test_preimages_are_the_adjoint_of_the_map(L):
    for n_in, n_out in PAIRS + _sweep(seed=1):
        src, first = _maps(L, n_in, n_out)
        # preimage of s = [first[s], first[s + 1]): exactly the destinations the forward maps to s
        assert np.array_equal(first, np.searchsorted(src, np.arange(n_in + 1), side='left')), (n_in, n_out)
        assert first[0] == 0 and first[-1] == n_out and np.all(np.diff(first) >= 0)


def test_preimage_of_a_ratio_pair_matches_torch_backward(L):
    """On integer ratios torch's backward (a scatter through the same forward map) and the gather agree cell for cell:
    the adjoint of F.interpolate, in fp64 autograd, counts each source cell's preimage."""
    for n_in, n_out in [(32, 64), (256, 512), (256, 64), (2048, 512), (64, 64), (48, 64), (200, 512), (700, 512)]:
        _, first = _maps(L, n_in, n_out)
        x = torch.zeros(1, 1, 1, n_in, dtype=torch.float64, requires_grad=True)
        F.interpolate(x, size=(1, n_out), mode='nearest').sum().backward()
        assert np.array_equal(x.grad.view(-1).long().numpy(), np.diff(first)), (n_in, n_out)


def test_index_helper_rejects_empty_sizes(L):
    assert L.bevpool_resize_nearest_index(0, 4, None, None) == -1
    assert L.bevpool_resize_nearest_index(4, 0, None, None) == -1


# ---------------------------------------------------------------------------------------------- argument errors
def test_abi_argument_errors_are_codes_not_crashes(L):
    p = ctypes.c_void_p(256)                           # never dereferenced: every call below fails its argument check
    fwd = lambda src, dt, nchw, b, c, sh, sw, dh, dw, out, st: L.bevpool_resize_nearest_into(
        src, dt, nchw, b, c, sh, sw, dh, dw, out, st, None)
    bwd = lambda src, dt, nchw, b, c, sh, sw, dh, dw, out, st: L.bevpool_resize_nearest_backward_from(
        out, st, src, dt, nchw, b, c, sh, sw, dh, dw, None)
    for fn in (fwd, bwd):
        assert fn(None, 0, 1, 2, 256, 32, 256, 64, 512, p, 336) == -1                 # null source / gradient
        assert fn(p, 0, 1, 2, 256, 32, 256, 64, 512, None, 336) == -1                 # null rows
        assert fn(p, 0, 1, 0, 256, 32, 256, 64, 512, p, 336) == -1                    # empty batch
        assert fn(p, 0, 1, 2, 0, 32, 256, 64, 512, p, 336) == -1                      # no channels
        assert fn(p, 0, 1, 2, 256, 0, 256, 64, 512, p, 336) == -1                     # empty source
        assert fn(p, 0, 1, 2, 256, 32, 256, 64, 0, p, 336) == -1                      # empty destination
        assert fn(p, 3, 1, 2, 256, 32, 256, 64, 512, p, 336) == -5                    # unknown dtype
        assert fn(p, 0, 1, 2, 6, 32, 256, 64, 512, p, 86) == -3                       # C % 4 != 0
        assert fn(p, 0, 1, 2, 256, 32, 256, 64, 512, p, 252) == -1                    # stride < C
        assert fn(p, 0, 1, 2, 256, 32, 256, 64, 512, p, 338) == -1                    # stride not a multiple of 4
        assert fn(p, 0, 1, 2 ** 17, 256, 32, 256, 64, 512, p, 336) == -2              # cells do not fit 31 bits
        assert fn(p, 0, 1, 2, 256, 32, 256, 64, 512, ctypes.c_void_p(260), 336) == -4  # misaligned rows
        assert fn(ctypes.c_void_p(264), 0, 0, 2, 256, 32, 256, 64, 512, p, 336) == -4  # misaligned fp32 pixel rows
        assert fn(ctypes.c_void_p(260), 2, 0, 2, 256, 32, 256, 64, 512, p, 336) == -4  # misaligned bf16 pixel rows


def test_resize_other_is_validated_before_any_device_work():
    x = torch.zeros(2, 4, 3, 3)
    for bad in ('nearest-exact', 'bilinear', 'NEAREST', 'area', True):
        with pytest.raises(ValueError, match='resize_other'):
            voxel_pooling_fused_concat(x, x, x, (3, 3, 1), None, resize_other=bad)


def test_batch_mismatch_of_other_bev_raises():
    x = torch.zeros(2, 4, 3, 3)
    plan = types.SimpleNamespace(batch=2, voxel_num=(3, 3, 1), mode='runs')
    for mode in (None, 'nearest'):
        with pytest.raises(ValueError, match='batch'):
            voxel_pooling_fused_concat(x, x, torch.zeros(3, 4, 3, 3), (3, 3, 1), plan, resize_other=mode)

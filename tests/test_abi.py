"""CPU checks of the C-ABI boundary: the library builds, loads, exports every symbol that
``include/bevpool_sm100.h`` declares, and argument errors come back as codes (no compute)."""
import ctypes
import os
import re

import pytest

from mm_training_b200 import _lib, build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope='module')
def L():
    build.build()
    return _lib.lib()


def _declared_symbols():
    text = open(os.path.join(ROOT, 'include', 'bevpool_sm100.h')).read()
    text = re.sub(r'/\*.*?\*/', '', text, flags=re.S)
    return sorted(set(re.findall(r'\b((?:bevpool|bevvox|bevlabel|bevdepth|pillar)_[a-z0-9_]+)\s*\(', text)))


def test_every_declared_symbol_is_exported(L):
    names = _declared_symbols()
    assert 'bevpool_forward' in names and 'bevpool_fused_backward' in names
    for n in names:
        assert hasattr(L, n), f'{n} declared in include/bevpool_sm100.h but not exported'
    for n in _lib.EXPORTED_SYMBOLS:
        assert n in names, f'{n} bound in _lib.py but not declared in the header'


def test_reference_launcher_symbol_is_exported(L):
    """ops/voxel_pooling/src/voxel_pooling_forward.cpp:21-22 links against this C++ symbol (Itanium mangling of
    voxel_pooling_forward_kernel_launcher(int x6, const int*, const float*, float*, int*, cudaStream_t))."""
    assert hasattr(L, '_Z37voxel_pooling_forward_kernel_launcheriiiiiiPKiPKfPfPiP11CUstream_st')


def test_abi_version_and_error_strings(L):
    assert L.bevpool_abi_version() == 2
    assert L.bevpool_error_string(0) == b'ok'
    assert b'channel' in L.bevpool_error_string(-3)


def test_argument_errors_are_codes_not_crashes(L):
    pb, tb = ctypes.c_size_t(), ctypes.c_size_t()
    assert L.bevpool_plan_sizes(0, 10, 4, 4, ctypes.byref(pb), ctypes.byref(tb)) == -1
    assert L.bevpool_plan_sizes(4, 2 ** 30, 4, 4, ctypes.byref(pb), ctypes.byref(tb)) == -2
    assert L.bevpool_plan_sizes(2, 6000, 128, 128, ctypes.byref(pb), ctypes.byref(tb)) == 0
    assert pb.value > 2 * 6000 * 8 and tb.value > 0
    # null pointers / bad channel counts are rejected before any launch
    assert L.bevpool_forward(None, None, None, 0, 2, 6000, 80, 128, 128, None, None) == -1
    assert L.bevpool_forward(None, None, None, 0, 2, 6000, 81, 128, 128, None, None) == -3
    assert L.bevpool_transpose(None, None, 0, 1, 4, 4, None) == -1


# The eight fused entry points: parameter names in ABI order.  Every case below breaks one argument of an otherwise
# valid call and must come back with its code before the library touches the device (the pointers are fake).
_FUSED_PARAMS = {
    'bevpool_fused_forward': 'plan depth ctx out dtype B N D H W C X Y ws stream',
    'bevpool_fused_backward': 'plan grad depth ctx gdepth gctx dtype B N D H W C X Y stream',
    'bevpool_fused_forward_runs': 'plan depth ctx out dtype B N D H W C X Y rows cap ws stream',
    'bevpool_fused_forward_runs_nchw': 'plan depth ctx out dtype B N D H W C X Y rows cap ws stream',
    'bevpool_fused_forward_runs_into': 'plan depth ctx flags out stride dtype B N D H W C X Y rows cap ws stream',
    'bevpool_fused_forward_runs_logits': 'plan feat Cf offset stats out stride dtype B N D H W C X Y rows cap ws stream',
    'bevpool_fused_backward_runs': 'plan grad depth ctx gdepth gctx nchw dtype B N D H W C X Y stream',
    'bevpool_fused_backward_runs_from': 'plan grad stride depth ctx gdepth gctx nchw dtype B N D H W C X Y stream',
}
_P, _MISALIGNED = 0x10000, 0x10004
_VALID = dict(plan=_P, depth=_P, ctx=_P, out=_P, grad=_P, gdepth=_P, gctx=_P, ws=_P, rows=_P, feat=_P, stats=_P,
              stream=None, dtype=0, B=2, N=2, D=8, H=4, W=8, C=80, X=16, Y=16, cap=64, flags=0, stride=128, nchw=0,
              Cf=96, offset=8)
E_ARG, E_RANGE, E_CHANNELS, E_ALIGN, E_DTYPE = -1, -2, -3, -4, -5
_COMMON = [(dict(plan=None), E_ARG), (dict(N=0), E_ARG), (dict(W=0), E_ARG), (dict(B=1, X=65536, Y=65536), E_RANGE)]
_RUNS = _COMMON + [(dict(C=84), E_CHANNELS), (dict(C=48), E_CHANNELS), (dict(dtype=1), E_DTYPE), (dict(dtype=2), E_DTYPE),
                   (dict(ctx=_MISALIGNED), E_ALIGN)]
_FUSED_ERRORS = {
    'bevpool_fused_forward': _COMMON + [(dict(C=81), E_CHANNELS), (dict(C=516), E_CHANNELS), (dict(dtype=7), E_DTYPE),
                                        (dict(ctx=_MISALIGNED), E_ALIGN), (dict(out=_MISALIGNED), E_ALIGN)],
    'bevpool_fused_backward': _COMMON + [(dict(C=81), E_CHANNELS), (dict(C=0), E_CHANNELS), (dict(dtype=7), E_DTYPE),
                                         (dict(gdepth=None), E_ARG), (dict(grad=_MISALIGNED), E_ALIGN),
                                         (dict(gctx=_MISALIGNED), E_ALIGN)],
    'bevpool_fused_forward_runs': _RUNS + [(dict(rows=None), E_ARG), (dict(cap=0), E_ARG), (dict(ws=None), E_ARG),
                                           (dict(rows=_MISALIGNED), E_ALIGN)],
    'bevpool_fused_forward_runs_nchw': _RUNS + [(dict(W=5), E_ALIGN), (dict(cap=0), E_ARG)],
    'bevpool_fused_forward_runs_into': _RUNS + [(dict(stride=0), E_ARG), (dict(stride=-4), E_ARG), (dict(stride=76), E_ARG),
                                                (dict(stride=82), E_ARG), (dict(flags=1, W=5), E_ALIGN),
                                                (dict(flags=3, W=6), E_ALIGN), (dict(out=_MISALIGNED), E_ALIGN)],
    'bevpool_fused_forward_runs_logits': [(dict(feat=None), E_ARG), (dict(stats=None), E_ARG), (dict(N=0), E_ARG),
                                          (dict(offset=-1), E_ARG), (dict(offset=17), E_ARG), (dict(Cf=87, offset=8), E_ARG),
                                          (dict(D=97, offset=0, C=16), E_ARG), (dict(dtype=1), E_DTYPE),
                                          (dict(feat=_MISALIGNED), E_ALIGN), (dict(W=6), E_ALIGN)],
    'bevpool_fused_backward_runs': _RUNS + [(dict(gctx=None), E_ARG), (dict(grad=_MISALIGNED), E_ALIGN),
                                            (dict(nchw=1, W=5), E_ALIGN), (dict(nchw=1, depth=_MISALIGNED), E_ALIGN),
                                            (dict(nchw=1, gdepth=_MISALIGNED), E_ALIGN)],
    'bevpool_fused_backward_runs_from': _RUNS + [(dict(stride=0), E_ARG), (dict(stride=-80), E_ARG), (dict(stride=76), E_ARG),
                                                 (dict(stride=82), E_ARG), (dict(W=5), E_ALIGN), (dict(nchw=1, W=5), E_ALIGN),
                                                 (dict(depth=_MISALIGNED), E_ALIGN), (dict(gdepth=_MISALIGNED), E_ALIGN),
                                                 (dict(grad=_MISALIGNED), E_ALIGN)],
}


@pytest.mark.parametrize('name', sorted(_FUSED_PARAMS))
def test_fused_entry_point_argument_errors(L, name):
    params = _FUSED_PARAMS[name].split()
    for change, code in _FUSED_ERRORS[name]:
        args = dict(_VALID, **change)
        assert getattr(L, name)(*[args[p] for p in params]) == code, (name, change)


def test_python_ops_refuse_cpu_tensors():
    import torch
    from mm_training_b200.ops.voxel_pooling import voxel_pooling
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        voxel_pooling(torch.zeros(1, 4, 3, dtype=torch.int32), torch.zeros(1, 4, 8), [2, 2, 1])


def _bench_module():
    import importlib.util
    spec = importlib.util.spec_from_file_location('bench_mod', os.path.join(ROOT, 'bench.py'))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    return bench


def test_bench_byte_model_matches_the_survey():
    """bench.py's roofline numerator is SURVEY.md section 8(d), row (B): 32.5 MB per CFG-2 frame."""
    bench = _bench_module()
    from mm_training_b200.configs import CFG_2, CFG_AIM
    b = bench.algorithmic_bytes(CFG_2, 150442)
    assert abs(b['step'] - 32.5e6) < 0.1e6
    assert b['fused_forward'] + b['fused_backward'] < b['step'] * 1.05
    assert abs(bench.algorithmic_bytes(CFG_AIM, 738884)['step'] - 108e6) < 1.5e6


def test_bench_dump_outputs_is_a_fixed_bounded_sample(tmp_path):
    """bench.py --dump-outputs: float32 .npy files; small arrays whole, large ones as the same seeded sample every run."""
    import numpy as np
    import torch
    bench = _bench_module()
    n = bench.DUMP_MAX_ELEMENTS
    big = torch.arange(n + 1000, dtype=torch.float64)          # element value == flat position
    small = torch.rand(2, 3, 4)
    for d in ('a', 'b'):
        bench.dump_outputs(str(tmp_path / d), {'big': big, 'small': small})
    a, b = np.load(tmp_path / 'a' / 'big.npy'), np.load(tmp_path / 'b' / 'big.npy')
    assert a.dtype == np.float32 and np.array_equal(a, b)
    assert a.size == n and bool((np.diff(a) > 0).all())       # distinct positions, in order
    s = np.load(tmp_path / 'a' / 'small.npy')
    assert s.dtype == np.float32 and np.array_equal(s, small.numpy())

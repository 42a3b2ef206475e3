"""ctypes binding of ``libbevpool_sm100.so`` (the C ABI declared in ``include/bevpool_sm100.h``).

There is no CPU or PyTorch fallback: if the library is missing or a call fails the caller
gets an exception.  The library is built in-tree by ``python -m mm_training_b200.build``.
"""
from __future__ import annotations

import ctypes
import os
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libbevpool_sm100.so')

F32, F16, BF16 = 0, 1, 2
_DTYPE_CODE = {torch.float32: F32, torch.float16: F16, torch.bfloat16: BF16}

_lock = threading.Lock()
_lib = None

_vp = ctypes.c_void_p
_i = ctypes.c_int
_i64 = ctypes.c_int64
_szp = ctypes.POINTER(ctypes.c_size_t)
_fp = ctypes.POINTER(ctypes.c_float)
_ip = ctypes.POINTER(ctypes.c_int)

# name -> argtypes; every function returns int (0 = ok) except the two noted below
_SIGNATURES = {
    'bevpool_plan_sizes': [_i, _i64, _i, _i, _szp, _szp],
    'bevpool_plan_build': [_vp, _i, _i64, _i, _i, _i, _vp, _vp, _vp],
    'bevpool_plan_pos_memo': [_vp, _i, _i64, _i, _i, _vp, _vp],
    'bevpool_plan_views': [_vp, _i, _i64, _i, _i, ctypes.POINTER(_vp), ctypes.POINTER(_vp), ctypes.POINTER(_vp)],
    'bevpool_forward_workspace_bytes': [_i, _szp],
    'bevpool_forward': [_vp, _vp, _vp, _i, _i, _i64, _i, _i, _i, _vp, _vp],
    'bevpool_backward': [_vp, _vp, _vp, _i, _i, _i64, _i, _i, _i, _vp],
    'bevpool_voxel_pooling_forward_launcher': [_i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp],
    'bevpool_fused_forward': [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _vp],
    'bevpool_fused_backward': [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp],
    'bevpool_runplan_sizes': [_i, _i, _i, _i, _i, _i, _i, _szp, _szp],
    'bevpool_runplan_pair_records': [_vp, _i, _i64, _i, _i, ctypes.POINTER(_vp)],
    'bevpool_runplan_build': [_vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp],
    'bevpool_runplan_views': [_vp, _i, _i64, _i, _i] + [ctypes.POINTER(_vp)] * 5,
    'bevpool_fused_forward_runs': [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _i64, _vp, _vp],
    'bevpool_fused_forward_runs_nchw': [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _i64, _vp, _vp],
    'bevpool_fused_forward_runs_into': [_vp, _vp, _vp, _i, _vp, _i64, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _i64, _vp, _vp],
    'bevpool_fused_forward_runs_logits': [_vp, _vp, _i, _i, _vp, _vp, _i64, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _i64, _vp, _vp],
    'bevpool_fused_backward_runs': [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp],
    'bevpool_fused_backward_runs_from': [_vp, _vp, _i64, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp],
    'bevpool_plan_status': [_vp, _ip, _vp],
    'bevpool_runplan_rig_sizes': [_i, _i, _i, _i, _i, _i, _i, _szp, _szp],
    'bevpool_runplan_build_rig': [_vp, _vp, _vp, _vp, _fp, _fp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp],
    'bevpool_rig_geom': [_vp, _vp, _vp, _vp, _fp, _fp, _i, _i, _i, _i, _i, _i, _vp, _vp],
    'bevpool_grad_rows': [_vp, _vp, _vp, _i, _i, _i64, _i, _i, _i, _vp],
    'bevpool_transpose': [_vp, _vp, _i, _i, _i64, _i64, _vp],
    'bevpool_warp_affine_forward': [_vp, _vp, _i64, _vp, _i64, _vp, _i, _i, _i, _i, _i, _i, _vp],
    'bevpool_warp_affine_backward': [_vp, _vp, _i64, _vp, _i64, _vp, _i, _i, _i, _i, _i, _i, _vp],
    'bevpool_resize_nearest_into': [_vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _i64, _vp],
    'bevpool_resize_nearest_backward_from': [_vp, _i64, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp],
    'bevpool_resize_nearest_index': [_i, _i, _vp, _vp],
    'bevvox_temp_bytes':[_i, _i64, _ip, _i, _i, _szp],
    'bevvox_hard_voxelize_scatter': [_vp, _vp, _vp, _i, _i64, _i64, _i, _fp, _fp, _ip, _i, _i, _vp, _vp, _vp, _vp, _vp, _i, _vp, _i, _vp, _vp],
    'bevvox_hard_voxelize': [_vp, _vp, _i, _i64, _i64, _i, _fp, _fp, _ip, _i, _i, _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp],
    'bevvox_dynamic_voxelize': [_vp, _i64, _i, _fp, _fp, _ip, _vp, _vp],
    'pillar_scatter_forward': [_vp, _vp, _i64, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp],
    'pillar_scatter_backward': [_vp, _vp, _i64, _i, _i, _i, _i, _i, _i, _vp, _vp],
    'bevdepth_softmax_forward': [_vp, _i, _i64, _vp, _i, _i, _i, _i, _vp, _vp, _vp],
    'bevdepth_softmax_backward': [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _i, _vp],
    'bevdepth_loss_workspace_bytes': [_i, _i, _i, _i, _szp],
    'bevdepth_loss_forward': [_vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp],
    'bevdepth_loss_backward': [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp],
    'bevlabel_scratch_bytes': [_i, _i, _i, _szp],
    'bevlabel_depth_labels': [_vp, _vp, _i, _i, _i, _i64, _vp, _vp, _vp, _i, _i, _i, ctypes.c_float, ctypes.c_float, _i,
                              _vp, _vp, _vp, _i, _vp],
}
EXPORTED_SYMBOLS = ['bevpool_abi_version', 'bevpool_error_string', 'bevpool_launch_count', 'bevpool_rig_num_variants',
                    *_SIGNATURES]


class BevPoolError(RuntimeError):
    pass


def lib() -> ctypes.CDLL:
    """Loads the native library once; raises if it has not been built."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise BevPoolError(
                        f'{LIB_PATH} not found: build it with `python -m mm_training_b200.build` '
                        '(there is no CPU / PyTorch fallback for this path)')
                l = ctypes.CDLL(LIB_PATH)
                l.bevpool_abi_version.restype = _i
                l.bevpool_abi_version.argtypes = []
                l.bevpool_error_string.restype = ctypes.c_char_p
                l.bevpool_error_string.argtypes = [_i]
                l.bevpool_launch_count.restype = _i64
                l.bevpool_launch_count.argtypes = []
                l.bevpool_rig_num_variants.restype = _i
                l.bevpool_rig_num_variants.argtypes = []
                for name, argtypes in _SIGNATURES.items():
                    fn = getattr(l, name)
                    fn.restype = _i
                    fn.argtypes = argtypes
                _lib = l
    return _lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib().bevpool_error_string(rc).decode()
        exc = ValueError if rc < 0 else BevPoolError
        raise exc(f'{what} failed: {msg} (code {rc})')


def dtype_code(t: torch.Tensor) -> int:
    try:
        return _DTYPE_CODE[t.dtype]
    except KeyError:
        raise TypeError(f'unsupported dtype {t.dtype}: expected float32, float16 or bfloat16') from None


def stream_ptr(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def require_cuda(*tensors: torch.Tensor) -> None:
    for t in tensors:
        if not t.is_cuda:
            raise RuntimeError('mm_training_b200 ops run on CUDA tensors only (no CPU fallback); '
                               f'got a tensor on {t.device}')


def launch_count() -> int:
    """Kernels launched by the native library so far in this process."""
    return int(lib().bevpool_launch_count())

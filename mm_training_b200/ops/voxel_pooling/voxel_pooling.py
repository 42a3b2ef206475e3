"""Drop-in ``voxel_pooling`` autograd op and its fused sibling, on libbevpool_sm100.

Mirrors ``ops/voxel_pooling/voxel_pooling.py`` of the reference:

* ``voxel_pooling(geom_xyz, input_features, voxel_num) -> (B, C, Y, X)`` --
  ``VoxelPooling.forward`` :10-55 / ``.backward`` :58-69 / ``voxel_pooling = VoxelPooling.apply`` :72.
  Same asserts (contiguous inputs, matching point counts), same output (a permuted view of a
  (B, Y, X, C) buffer), gradient only w.r.t. ``input_features`` in the caller's shape.
* ``voxel_pooling_fused(geom_xyz, depth, context, voxel_num)`` replaces the materialised outer
  product of ``layers/backbones/lss_fpn.py:441-464``: ``depth`` (B*N, D, H, W), ``context``
  (B*N, C, H, W); gradients flow to both.

Differences, all deliberate (SURVEY.md section 8b): fp16/bf16 are accepted (fp32 accumulation);
``voxel_num`` may be a tensor on any device or a python sequence; the backward allocates a fresh
gradient instead of mutating a tensor saved in forward; errors raise instead of ``exit(-1)``.
"""
from __future__ import annotations

import ctypes
import os
from typing import Optional, Sequence, Tuple, Union

import torch
from torch.autograd import Function

from ... import _lib

VoxelNum = Union[torch.Tensor, Sequence[int]]

def _voxel_num_ints(voxel_num: VoxelNum) -> Tuple[int, int, int]:
    """[X, Y, Z] as python ints.  A CUDA tensor costs one D2H sync per call (the reference pays
    >= 5, voxel_pooling.py:37-38,45-47); pass python ints or a CPU tensor to avoid it."""
    if isinstance(voxel_num, torch.Tensor):
        voxel_num = voxel_num.tolist()
    x, y, z = (int(v) for v in voxel_num)
    return x, y, z


RUN_CHANNELS = (32, 64, 80, 96, 128)     # channel counts of the fp32 run-plan kernels (csrc/pool_runs.cu)


class PoolingPlan:
    """Cell index of every point + the kept points sorted by BEV cell (CSR).  Depends only on
    ``geom_xyz`` and ``voxel_num``: reuse it while the camera geometry is unchanged.

    ``frustum=(N, D, H, W)`` asks for a RUN plan (fused op only): vertically adjacent points of one
    (image, depth bin, column) that share a BEV cell are sorted as one entry -- 11x fewer entries at
    the aiMotive shape -- and ``run_code`` maps every point to its run.  Any grid size; ``mode`` says which
    kind was built ('runs', or 'points' when ``geom_xyz`` is not 16-byte aligned).
    ``max_runs``: the caller's upper bound of the run count; it sizes the scratch rows of the fused forward
    without reading the count back (no host sync: what a CUDA-graph capture needs).  It is only valid for the
    SAME ``geom_xyz`` (or a rig known to produce no more runs): if the real count is larger the kernels stay
    inside the scratch, the output is invalid and ``status()`` returns BEVPOOL_PLAN_ROW_OVERFLOW (1) -- call
    ``raise_if_overflowed()`` at a point where a sync is acceptable.  Without it the first fused forward reads
    the exact count back (one D2H sync)."""

    def __init__(self, geom_xyz: Optional[torch.Tensor], voxel_num: VoxelNum, frustum: Optional[Sequence[int]] = None,
                 max_runs: Optional[int] = None, _rig=None):
        self.voxel_num = _voxel_num_ints(voxel_num)
        self.mode = 'points'
        self.frustum = None
        self._num_runs = max_runs
        self.hinted = max_runs is not None
        X, Y, Z = self.voxel_num
        L = _lib.lib()
        pb, tb = ctypes.c_size_t(), ctypes.c_size_t()
        if _rig is not None:                       # built from the camera rig (rig.py): no geom_xyz tensor exists
            lsg, combine, variant = _rig
            _lib.require_cuda(combine)
            assert combine.dtype == torch.float32 and combine.is_contiguous() and combine.shape[-2:] == (4, 4)
            self.batch, N = int(combine.shape[0]), int(combine.shape[1])
            D, H, W = lsg.D, lsg.H, lsg.W
            self.num_points = N * D * H * W
            self.device = combine.device
            self.mode, self.frustum = 'runs', (N, D, H, W)
            _lib.check(L.bevpool_runplan_rig_sizes(self.batch, N, D, H, W, X, Y, ctypes.byref(pb), ctypes.byref(tb)),
                       'bevpool_runplan_rig_sizes')
            with torch.cuda.device(self.device):
                self.buffer = torch.empty(pb.value, dtype=torch.uint8, device=self.device)
                temp = torch.empty(tb.value, dtype=torch.uint8, device=self.device)
                _lib.check(L.bevpool_runplan_build_rig(combine.data_ptr(), lsg.fx.data_ptr(), lsg.fy.data_ptr(),
                                                       lsg.fd.data_ptr(), lsg._lower_c, lsg._vs_c, variant, self.batch,
                                                       N, D, H, W, X, Y, Z, self.buffer.data_ptr(), temp.data_ptr(),
                                                       _lib.stream_ptr(self.device)), 'bevpool_runplan_build_rig')
            return
        _lib.require_cuda(geom_xyz)
        if geom_xyz.dtype != torch.int32:
            raise TypeError(f'geom_xyz must be int32 (got {geom_xyz.dtype})')
        assert geom_xyz.is_contiguous()
        assert geom_xyz.shape[-1] == 3
        self.batch = int(geom_xyz.shape[0])
        self.num_points = int(geom_xyz.numel() // (3 * self.batch))
        self.device = geom_xyz.device
        if frustum is not None:
            N, D, H, W = (int(v) for v in frustum)
            assert N * D * H * W == self.num_points, 'frustum shape does not match geom_xyz'
            if geom_xyz.data_ptr() % 16 == 0:
                _lib.check(L.bevpool_runplan_sizes(self.batch, N, D, H, W, X, Y, ctypes.byref(pb), ctypes.byref(tb)),
                           'bevpool_runplan_sizes')
                self.mode, self.frustum = 'runs', (N, D, H, W)
        if self.mode == 'points':
            _lib.check(L.bevpool_plan_sizes(self.batch, self.num_points, X, Y, ctypes.byref(pb), ctypes.byref(tb)),
                       'bevpool_plan_sizes')
        with torch.cuda.device(self.device):
            self.buffer = torch.empty(pb.value, dtype=torch.uint8, device=self.device)
            temp = torch.empty(tb.value, dtype=torch.uint8, device=self.device)
            if self.mode == 'runs':
                N, D, H, W = self.frustum
                _lib.check(L.bevpool_runplan_build(geom_xyz.data_ptr(), self.batch, N, D, H, W, X, Y, Z,
                                                   self.buffer.data_ptr(), temp.data_ptr(),
                                                   _lib.stream_ptr(self.device)), 'bevpool_runplan_build')
            else:
                _lib.check(L.bevpool_plan_build(geom_xyz.data_ptr(), self.batch, self.num_points, X, Y, Z,
                                                self.buffer.data_ptr(), temp.data_ptr(),
                                                _lib.stream_ptr(self.device)), 'bevpool_plan_build')
        # temp is released to the caching allocator here; stream-ordered reuse keeps this safe

    @classmethod
    def from_rig(cls, lsg, combine: torch.Tensor, variant: int, max_runs: Optional[int] = None) -> 'PoolingPlan':
        """Run plan from ``combine = sensor2ego @ inverse(intrin)`` (B, N, 4, 4) and the frustum axes of ``lsg``
        (``rig.LiftSplatGeometry``): the geometry / index tensors of ``lss_fpn.py:328-361,461-462`` are never made."""
        return cls(None, lsg.voxel_num, None, max_runs, _rig=(lsg, combine, variant))

    def status(self) -> int:
        """The plan's device status word (0 = ok, 1 = run-row scratch overflow).  Synchronises the stream."""
        v = ctypes.c_int(0)
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().bevpool_plan_status(self.ptr, ctypes.byref(v), _lib.stream_ptr(self.device)),
                       'bevpool_plan_status')
        return int(v.value)

    def raise_if_overflowed(self) -> None:
        if self.status() == 1:
            raise RuntimeError(f'PoolingPlan: max_runs={self._num_runs} is smaller than the run count of this geometry '
                               '(the hint is only valid for the geom_xyz it was measured on); the pooled output of the '
                               'forward calls that used this plan is invalid')

    @property
    def ptr(self) -> int:
        return self.buffer.data_ptr()

    def _views(self):
        X, Y, _ = self.voxel_num
        ptrs = [ctypes.c_void_p() for _ in range(5)]
        _lib.check(_lib.lib().bevpool_runplan_views(self.ptr, self.batch, self.num_points, X, Y,
                                                    *[ctypes.byref(q) for q in ptrs]), 'bevpool_runplan_views')
        base = self.ptr
        as_i32 = self.buffer.view(torch.int32)
        P, G = self.batch * self.num_points, self.batch * X * Y
        o = lambda q: (q.value - base) // 4
        a, b, c, d, e = ptrs
        views = [as_i32[o(a):o(a) + P], as_i32[o(b):o(b) + G + 1], as_i32[o(c):o(c) + P], as_i32[o(d):o(d) + P]]
        views.append(as_i32[o(e):o(e) + P] if self.mode == 'runs' else None)
        return views

    @property
    def cell_of_point(self) -> torch.Tensor:
        """int32 (B, Np): in-sample cell id y*X + x, or -1 for dropped points."""
        return self._views()[0].view(self.batch, self.num_points)

    @property
    def cell_start(self) -> torch.Tensor:
        """int32 (B*Y*X + 1,): CSR offsets into ``sorted_ids``."""
        return self._views()[1]

    @property
    def sorted_ids(self) -> torch.Tensor:
        """int32 (K,): global point ids (b*Np + p) of kept points (run plans: of the first point of every
        run), grouped by cell, ascending inside a cell."""
        ids = self._views()[2]
        return ids[:int(self.cell_start[-1].item())]

    @property
    def num_sorted(self) -> int:
        """Number of sorted entries K = cell_start[-1]: kept points of a point plan, runs of a run plan.
        Read back from the device once (a sync) unless ``max_runs`` was given."""
        if self._num_runs is None:
            self._num_runs = int(self.cell_start[-1].item())
        return self._num_runs

    @property
    def sorted_cells(self) -> torch.Tensor:
        """int32 (K,): global output row b*Y*X + cell of every sorted entry."""
        return self._views()[3][:int(self.cell_start[-1].item())]

    @property
    def run_code(self) -> torch.Tensor:
        """run plans: int32 (B, Np) -- slot of the run for its first point, -2 continuation, -1 dropped."""
        assert self.mode == 'runs'
        return self._views()[4].view(self.batch, self.num_points)

    @property
    def pair_records(self) -> torch.Tensor:
        """run plans: int32 (B, N, D, ceil(H/16), W, 4) = {primary cell | -1, rows in it | kept rows elsewhere << 16,
        slot of the run that starts at the first kept row, number of runs} per (image, bin, 16-row block, column)."""
        assert self.mode == 'runs'
        N, D, H, W = self.frustum
        HB = (H + 15) // 16
        X, Y, _ = self.voxel_num
        q = ctypes.c_void_p()
        _lib.check(_lib.lib().bevpool_runplan_pair_records(self.ptr, self.batch, self.num_points, X, Y, ctypes.byref(q)),
                   'bevpool_runplan_pair_records')
        o = (q.value - self.ptr) // 4
        n = self.batch * N * D * HB * W * 4
        return self.buffer.view(torch.int32)[o:o + n].view(self.batch, N, D, HB, W, 4)

    def pos_memo(self) -> torch.Tensor:
        """The reference's ``pos_memo`` (voxel_pooling.py:40): int32 (B, Np, 3) = (b, y, x) or -1."""
        X, Y, _ = self.voxel_num
        out = torch.empty(self.batch, self.num_points, 3, dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().bevpool_plan_pos_memo(self.ptr, self.batch, self.num_points, X, Y,
                                                        out.data_ptr(), _lib.stream_ptr(self.device)),
                       'bevpool_plan_pos_memo')
        return out


def build_plan(geom_xyz: torch.Tensor, voxel_num: VoxelNum, frustum: Optional[Sequence[int]] = None,
               max_runs: Optional[int] = None) -> PoolingPlan:
    return PoolingPlan(geom_xyz, voxel_num, frustum, max_runs)


def runs_supported(channels: int, dtype: torch.dtype) -> bool:
    """fp32 fast-path channel counts; BEVPOOL_DISABLE_G8=1 (tests) forces the generic point kernels."""
    return (dtype == torch.float32 and channels in RUN_CHANNELS
            and os.environ.get('BEVPOOL_DISABLE_G8', '0') != '1')


def _transpose(x: torch.Tensor, batch: int, rows: int, cols: int) -> torch.Tensor:
    """(batch, rows, cols) -> (batch, cols, rows) with the library's tiled transpose."""
    with torch.cuda.device(x.device):
        out = torch.empty(batch, cols, rows, dtype=x.dtype, device=x.device)
        _lib.check(_lib.lib().bevpool_transpose(x.data_ptr(), out.data_ptr(), _lib.dtype_code(x), batch, rows, cols,
                                                _lib.stream_ptr(x.device)), 'bevpool_transpose')
    return out


def _strided_rows(x: torch.Tensor) -> Optional[int]:
    """(B, C, H, W) view of channels-last rows -> the row stride in elements, or None.  Zero-copy for the output of the
    pooling ops and for a channel slice of a concatenated channels-last buffer."""
    B, C, H, W = x.shape
    s = x.stride()
    S = s[3]
    if (s[1] == 1 and S >= C and S % 4 == 0 and s[2] == W * S and (B == 1 or s[0] == H * W * S)
            and x.data_ptr() % 16 == 0):
        return S
    return None


def _grad_rows_nhwc(grad_out: torch.Tensor, plan: PoolingPlan) -> torch.Tensor:
    """grad_out arrives as (B, C, Y, X) with arbitrary strides; the kernels want (B, Y, X, C) rows.
    Zero-copy when it already is a permuted NHWC buffer (what autograd hands back for the
    permuted view we return).  Otherwise one pass that transposes only the tiles holding an
    occupied cell -- rows of empty cells are never read by the backward kernels and stay
    uninitialised."""
    B, C, Y, X = grad_out.shape
    nhwc = grad_out.permute(0, 2, 3, 1)
    if nhwc.is_contiguous():
        return nhwc
    if not grad_out.is_contiguous():
        grad_out = grad_out.contiguous()
    with torch.cuda.device(grad_out.device):
        rows = torch.empty(B, Y, X, C, dtype=grad_out.dtype, device=grad_out.device)
        _lib.check(_lib.lib().bevpool_grad_rows(plan.ptr, grad_out.data_ptr(), rows.data_ptr(),
                                                _lib.dtype_code(grad_out), B, plan.num_points, C, X, Y,
                                                _lib.stream_ptr(grad_out.device)), 'bevpool_grad_rows')
    return rows


def _forward_workspace(channels: int, device) -> torch.Tensor:
    """Scratch for the forward kernels (partial sums of cells cut by the even-share partition)."""
    nbytes = ctypes.c_size_t()
    _lib.check(_lib.lib().bevpool_forward_workspace_bytes(channels, ctypes.byref(nbytes)),
               'bevpool_forward_workspace_bytes')
    return torch.empty(nbytes.value, dtype=torch.uint8, device=device)


def _run_scratch(plan: PoolingPlan, channels: int, device):
    """Scratch of a run-plan forward: ``(run_rows, capacity, workspace)`` -- one float32 row per run (sized by the plan's
    run count or its ``max_runs`` hint) and the workspace of stage B."""
    cap = max(1, plan.num_sorted)
    run_rows = torch.empty(cap, channels, dtype=torch.float32, device=device)
    return run_rows, cap, _forward_workspace(channels, device)


def pool_forward(plan: PoolingPlan, input_features: torch.Tensor) -> torch.Tensor:
    """features (B, ..., C) -> (B, Y, X, C); every cell written once, no pre-zeroing."""
    X, Y, _ = plan.voxel_num
    B, C = plan.batch, input_features.shape[-1]
    assert plan.mode == 'points', 'the drop-in op sums arbitrary per-point rows: it needs a point plan'
    with torch.cuda.device(input_features.device):
        out = torch.empty(B, Y, X, C, dtype=input_features.dtype, device=input_features.device)
        ws = _forward_workspace(C, out.device)
        _lib.check(_lib.lib().bevpool_forward(plan.ptr, input_features.data_ptr(), out.data_ptr(),
                                              _lib.dtype_code(input_features), B, plan.num_points, C, X, Y,
                                              ws.data_ptr(), _lib.stream_ptr(out.device)), 'bevpool_forward')
    return out


def pool_backward(plan: PoolingPlan, grad_output: torch.Tensor, input_shape) -> torch.Tensor:
    """grad_output (B, C, Y, X), any strides -> grad_features in ``input_shape``."""
    X, Y, _ = plan.voxel_num
    B, C = grad_output.shape[0], grad_output.shape[1]
    rows = _grad_rows_nhwc(grad_output, plan)
    with torch.cuda.device(rows.device):
        grad_in = torch.empty(input_shape, dtype=rows.dtype, device=rows.device)
        _lib.check(_lib.lib().bevpool_backward(plan.ptr, rows.data_ptr(), grad_in.data_ptr(),
                                               _lib.dtype_code(rows), B, plan.num_points, C, X, Y,
                                               _lib.stream_ptr(rows.device)), 'bevpool_backward')
    return grad_in


def context_rows_nhwc(context: torch.Tensor) -> torch.Tensor:
    """context (B*N, C, H, W), NCHW or channels_last -> (B*N, H, W, C) contiguous rows.  Zero-copy for
    channels_last; NCHW costs one small tiled transpose (C*H*W elements per image)."""
    BN, C, H, W = context.shape
    rows = context.permute(0, 2, 3, 1)
    if not rows.is_contiguous():
        rows = _transpose(context.contiguous(), BN, C, H * W).view(BN, H, W, C)
    return rows


def _nchw_direct(context: torch.Tensor, depth: torch.Tensor, channels: Optional[int] = None) -> bool:
    """NCHW-contiguous fp32 context whose rows are multiples of 16 bytes: the kernels read it through a TMA
    tensor map, no layout pass.  ``channels``: C, when ``context`` holds more channels (DepthNet's output)."""
    C = context.shape[1] if channels is None else channels
    return (context.is_contiguous() and context.dtype == torch.float32 and context.shape[3] % 4 == 0
            and runs_supported(C, context.dtype) and context.data_ptr() % 16 == 0 and depth.data_ptr() % 16 == 0
            and os.environ.get('BEVPOOL_NCHW_DIRECT', '1') != '0')


def _mixed(depth: torch.Tensor, context: torch.Tensor) -> bool:
    """The autocast pair: fp32 depth (softmax runs in fp32) with an fp16 / bf16 context.  Pooled in fp32."""
    return depth.dtype == torch.float32 and context.dtype in (torch.float16, torch.bfloat16)


def _mixed_route(context: torch.Tensor, depth: torch.Tensor, context_rows: Optional[torch.Tensor]) -> str:
    """``_route`` of a mixed call on a run plan.  The 16-bit context kernels exist for the column backward only, which
    needs W % 4 == 0 and a 16-byte aligned contiguous depth; a tensor-map row of a 16-bit NCHW context is 16 bytes
    only when W % 8 == 0, so W = 44 (CFG-2) takes pixel rows."""
    W = depth.shape[3]
    if W % 4 != 0 or not depth.is_contiguous() or depth.data_ptr() % 16 != 0 or context.data_ptr() % 16 != 0:
        return 'points'
    if (context_rows is None and context.is_contiguous() and W % 8 == 0
            and os.environ.get('BEVPOOL_NCHW_DIRECT', '1') != '0'):
        return 'nchw'
    return 'rows'


def _route(plan_mode: str, context: torch.Tensor, depth: torch.Tensor, context_rows: Optional[torch.Tensor] = None,
           channels: Optional[int] = None) -> str:
    """The kernels that pool ``context`` on a plan of ``plan_mode``: 'nchw' (run plan, ``_nchw_direct``), 'rows' (run
    plan; pixel rows, ``context_rows`` or ``context_rows_nhwc(context)``) or 'points' (point plan, or no run kernel for
    the dtype / channel count).  A mixed call (``_mixed``) on 'points' pools ``context.float()``."""
    if plan_mode != 'runs' or not runs_supported(context.shape[1] if channels is None else channels, depth.dtype):
        return 'points'
    if _mixed(depth, context):
        return _mixed_route(context, depth, context_rows)
    return 'nchw' if context_rows is None and _nchw_direct(context, depth, channels) else 'rows'


def fused_forward(plan: PoolingPlan, depth: torch.Tensor, context: torch.Tensor,
                  context_rows: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None,
                  prezeroed: bool = False) -> torch.Tensor:
    """depth (B*N, D, H, W), context (B*N, C, H, W) NCHW or channels_last -> (B, Y, X, C).  ``out``: a caller-provided
    (B, Y, X, C) buffer; on a run plan also rows at a uniform cell stride, such as ``buf[..., :C]`` of a wider
    channels-last ``buf``.  ``prezeroed`` (run plans): the kernels write the rows of occupied cells only and leave the
    others as they are -- for an ``out`` that already holds zeros (``fused_forward_cold``) or whose empty cells are never
    read (the BDA warp's scratch).  A point plan writes every cell either way.  fp32 ``depth`` with an fp16 / bf16
    ``context`` (autocast) gives fp32 rows equal, bit for bit, to the call on ``context.float()``.  An fp16 / bf16 ``out``
    (run plans) receives the fp32 rows rounded once, bit for bit ``.to(out.dtype)`` of what an fp32 ``out`` receives."""
    BN, D, H, W = depth.shape
    C = context.shape[1]
    X, Y, _ = plan.voxel_num
    B = plan.batch
    N = BN // B
    mixed = _mixed(depth, context)
    assert context.shape == (BN, C, H, W) and (depth.dtype == context.dtype or mixed)
    assert B * N == BN and plan.num_points == N * D * H * W
    route = _route(plan.mode, context, depth, context_rows)
    if mixed and route == 'points':             # no run kernel takes it: pool context.float(), the call it stands for
        context, context_rows, mixed = context.float(), None, False
        route = _route(plan.mode, context, depth)
    with torch.cuda.device(depth.device):
        if out is None:
            out, prezeroed = torch.empty(B, Y, X, C, dtype=depth.dtype, device=depth.device), False
        half_out = out.dtype in (torch.float16, torch.bfloat16) and depth.dtype == torch.float32
        assert out.shape == (B, Y, X, C) and (out.dtype == depth.dtype or half_out)
        stride = C if out.is_contiguous() else _strided_rows(out.permute(0, 3, 1, 2))
        assert stride is not None, 'out must be (B, Y, X, C) rows at a uniform cell stride'
        if route == 'points' and half_out:
            raise ValueError(f'an {out.dtype} out needs a run plan and a run kernel for C={C}')
        if route == 'points':
            if plan.mode == 'runs':
                raise ValueError(f'run plans need float32 and C in {RUN_CHANNELS}; build a point plan for C={C}, {depth.dtype}')
            if stride != C:
                raise ValueError('a point plan writes packed (B, Y, X, C) rows: out must be contiguous')
            ctx_nhwc = context_rows_nhwc(context) if context_rows is None else context_rows
            ws = _forward_workspace(C, out.device)
            _lib.check(_lib.lib().bevpool_fused_forward(plan.ptr, depth.data_ptr(), ctx_nhwc.data_ptr(),
                                                        out.data_ptr(), _lib.dtype_code(depth), B, N, D, H, W,
                                                        C, X, Y, ws.data_ptr(), _lib.stream_ptr(depth.device)),
                       'bevpool_fused_forward')
            return out
        assert plan.frustum == (N, D, H, W)
        run_rows, cap, ws = _run_scratch(plan, C, depth.device)
        nchw = route == 'nchw'
        ctx_arg = context if nchw else (context_rows_nhwc(context) if context_rows is None else context_rows)
        flags = (1 if nchw else 0) | (2 if prezeroed else 0)
        if half_out:
            _lib.check(_lib.lib().bevpool_fused_forward_runs_into16(
                plan.ptr, depth.data_ptr(), ctx_arg.data_ptr(), _lib.dtype_code(context), flags, out.data_ptr(), stride,
                _lib.dtype_code(out), B, N, D, H, W, C, X, Y, run_rows.data_ptr(), cap, ws.data_ptr(),
                _lib.stream_ptr(depth.device)), 'bevpool_fused_forward_runs_into16')
            return out
        if mixed:
            _lib.check(_lib.lib().bevpool_fused_forward_runs_mixed(
                plan.ptr, depth.data_ptr(), ctx_arg.data_ptr(), _lib.dtype_code(context), flags, out.data_ptr(), stride,
                B, N, D, H, W, C, X, Y, run_rows.data_ptr(), cap, ws.data_ptr(), _lib.stream_ptr(depth.device)),
                'bevpool_fused_forward_runs_mixed')
            return out
        _lib.check(_lib.lib().bevpool_fused_forward_runs_into(
            plan.ptr, depth.data_ptr(), ctx_arg.data_ptr(), flags, out.data_ptr(),
            stride, _lib.dtype_code(depth), B, N, D, H, W, C, X, Y, run_rows.data_ptr(), cap, ws.data_ptr(),
            _lib.stream_ptr(depth.device)), 'bevpool_fused_forward_runs_into')
    return out


_SIDE_STREAMS = {}


def _side_stream(device) -> torch.cuda.Stream:
    key = torch.device(device).index if torch.device(device).index is not None else torch.cuda.current_device()
    if key not in _SIDE_STREAMS:
        _SIDE_STREAMS[key] = torch.cuda.Stream(device)
    return _SIDE_STREAMS[key]


def fused_forward_cold(make_plan, batch: int, voxel_num: VoxelNum, depth: torch.Tensor, context: torch.Tensor):
    """Plan build + fused forward of a COLD call (geometry changed: the plan is rebuilt); returns ``(plan, out (B, Y, X,
    C))``.  With ``BEVPOOL_COLD_OVERLAP=1`` the output is zero-filled on a side stream WHILE ``make_plan()`` runs on the
    caller's stream (fork / join with events: CUDA-graph capturable) and the forward then writes occupied cells only.
    MEASURED SLOWER than the default (B200, CFG-2, 32 frames: 401 us vs 390 us per step): stage A already hides its fill
    -- one TMA bulk store per empty 32-cell block, issued by the copy engine behind the issue-bound reduction -- while a
    separate fill kernel competes with the plan kernels for SM slots and adds a fork / join.  Kept as an option (and
    tested) because the balance shifts for grids that are mostly empty AND large (512 x 512)."""
    X, Y, _ = _voxel_num_ints(voxel_num)
    C = context.shape[1]
    dev = depth.device
    if not runs_supported(C, depth.dtype) or os.environ.get('BEVPOOL_COLD_OVERLAP', '0') != '1':
        plan = make_plan()
        return plan, fused_forward(plan, depth, context)
    with torch.cuda.device(dev):
        cur, side = torch.cuda.current_stream(dev), _side_stream(dev)
        out = torch.empty(batch, Y, X, C, dtype=depth.dtype, device=dev)
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            out.zero_()
        plan = make_plan()
        cur.wait_stream(side)          # (every later use of `out`, its free included, is ordered behind this join)
        return plan, fused_forward(plan, depth, context, out=out, prezeroed=True)


def _fused_backward_rows(plan: PoolingPlan, route: str, grad_rows: torch.Tensor, row_stride: Optional[int],
                         depth: torch.Tensor, context: torch.Tensor, context_rows: Optional[torch.Tensor]):
    """Fused backward on ``route`` (``_route``) -> (grad_depth, grad_context).  ``row_stride`` None: ``grad_rows`` are
    packed (B, Y, X, C) rows (``_grad_rows_nhwc``); else the row of cell c starts ``c * row_stride`` floats after the
    first (run plans with W % 4 == 0 only).  grad_context has the memory format of ``context``: channels_last in ->
    channels_last out (zero-copy), NCHW in -> NCHW out (written NCHW on the 'nchw' route, else one tiled transpose).
    A mixed call (``_mixed``) returns grad_context in the dtype of ``context``: the fp32 gradient of the call on
    ``context.float()`` rounded once, as autograd's cast would round it."""
    BN, D, H, W = depth.shape
    C = context.shape[1]
    X, Y, _ = plan.voxel_num
    B = plan.batch
    N = BN // B
    mixed = _mixed(depth, context)
    if mixed and route == 'points':
        upcast = context.float()                    # as in fused_forward
        grad_depth, grad_context = _fused_backward_rows(plan, _route(plan.mode, upcast, depth), grad_rows, row_stride,
                                                        depth, upcast, None)
        return grad_depth, grad_context.to(context.dtype)
    nchw = route == 'nchw'
    assert row_stride is None or route != 'points'
    grad_depth = torch.empty_like(depth)
    if nchw:
        ctx_arg, grad_ctx_arg = context, torch.empty_like(context)
    else:
        ctx_arg = context_rows_nhwc(context) if context_rows is None else context_rows
        grad_ctx_arg = torch.empty(BN, H, W, C, dtype=context.dtype, device=context.device)
    args = (depth.data_ptr(), ctx_arg.data_ptr(), grad_depth.data_ptr(), grad_ctx_arg.data_ptr())
    dims = (_lib.dtype_code(depth), B, N, D, H, W, C, X, Y, _lib.stream_ptr(depth.device))
    L = _lib.lib()
    if mixed:
        _lib.check(L.bevpool_fused_backward_runs_mixed(plan.ptr, grad_rows.data_ptr(), row_stride or 0, *args, int(nchw),
                                                       _lib.dtype_code(context), *dims[1:]), 'bevpool_fused_backward_runs_mixed')
    elif route == 'points':
        _lib.check(L.bevpool_fused_backward(plan.ptr, grad_rows.data_ptr(), *args, *dims), 'bevpool_fused_backward')
    elif row_stride is None:
        _lib.check(L.bevpool_fused_backward_runs(plan.ptr, grad_rows.data_ptr(), *args, int(nchw), *dims),
                   'bevpool_fused_backward_runs')
    else:
        _lib.check(L.bevpool_fused_backward_runs_from(plan.ptr, grad_rows.data_ptr(), row_stride, *args, int(nchw), *dims),
                   'bevpool_fused_backward_runs_from')
    if nchw:
        return grad_depth, grad_ctx_arg
    if context.permute(0, 2, 3, 1).is_contiguous():
        return grad_depth, grad_ctx_arg.permute(0, 3, 1, 2)
    return grad_depth, _transpose(grad_ctx_arg, BN, H * W, C).view(BN, C, H, W)


def fused_backward(plan: PoolingPlan, grad_output: torch.Tensor, depth: torch.Tensor,
                   context: torch.Tensor, context_rows: Optional[torch.Tensor] = None):
    """grad_output (B, C, Y, X), any strides -> (grad_depth, grad_context) in the memory format of ``context``
    (``_fused_backward_rows``)."""
    with torch.cuda.device(depth.device):
        rows = _grad_rows_nhwc(grad_output, plan)
        return _fused_backward_rows(plan, _route(plan.mode, context, depth, context_rows), rows, None, depth, context,
                                    context_rows)


class VoxelPooling(Function):
    @staticmethod
    def forward(ctx, geom_xyz: torch.Tensor, input_features: torch.Tensor, voxel_num: VoxelNum,
                plan: Optional[PoolingPlan] = None) -> torch.Tensor:
        _lib.require_cuda(geom_xyz, input_features)
        assert geom_xyz.is_contiguous()
        assert input_features.is_contiguous()
        B, C = input_features.shape[0], input_features.shape[-1]
        num_points = input_features.numel() // (B * C)
        assert geom_xyz.numel() // (3 * geom_xyz.shape[0]) == num_points and geom_xyz.shape[0] == B
        X, Y, Z = _voxel_num_ints(voxel_num)
        with torch.cuda.device(input_features.device):
            if plan is None:
                plan = PoolingPlan(geom_xyz, (X, Y, Z))
            else:
                assert (plan.batch, plan.num_points, plan.voxel_num) == (B, num_points, (X, Y, Z))
            out = pool_forward(plan, input_features)
        ctx.plan = plan
        ctx.input_shape = input_features.shape
        return out.permute(0, 3, 1, 2)

    @staticmethod
    def backward(ctx, grad_output_features: torch.Tensor):
        with torch.cuda.device(grad_output_features.device):
            grad_in = pool_backward(ctx.plan, grad_output_features, ctx.input_shape)
        return None, grad_in, None, None


def voxel_pooling(geom_xyz: torch.Tensor, input_features: torch.Tensor, voxel_num: VoxelNum,
                  plan: Optional[PoolingPlan] = None) -> torch.Tensor:
    """Scatter-sum per-point C-vectors into the BEV grid; returns (B, C, Y, X)."""
    return VoxelPooling.apply(geom_xyz, input_features, voxel_num, plan)


class VoxelPoolingFused(Function):
    @staticmethod
    def forward(ctx, geom_xyz, depth, context, voxel_num, plan, make_plan=None, batch=None):
        _lib.require_cuda(depth, context)
        assert depth.is_contiguous()
        X, Y, Z = _voxel_num_ints(voxel_num)
        with torch.cuda.device(depth.device):
            out = None
            if plan is None:
                runs = True                   # a caller-supplied builder (the camera rig) makes run plans
                if make_plan is None:
                    assert geom_xyz.is_contiguous()
                    # (a run plan reads its run count back once to size the scratch rows: not while capturing)
                    runs = (geom_xyz.dim() == 6 and runs_supported(context.shape[1], depth.dtype)
                            and not torch.cuda.is_current_stream_capturing())
                    frustum = tuple(geom_xyz.shape[1:5]) if runs else None      # (N, D, H, W): sort runs, not points
                    make_plan, batch = (lambda: PoolingPlan(geom_xyz, (X, Y, Z), frustum)), geom_xyz.shape[0]
                if runs and _route('runs', context, depth) == 'nchw':
                    # cold call: the zero fill of the output may overlap the plan build
                    plan, out = fused_forward_cold(make_plan, int(batch), (X, Y, Z), depth, context)
                else:
                    plan = make_plan()
            assert plan.voxel_num == (X, Y, Z)
            route = _route(plan.mode, context, depth)
            # reused by backward; a mixed call on 'points' pools context.float() and makes its own rows
            upcast = route == 'points' and _mixed(depth, context)
            context_rows = None if route == 'nchw' or upcast else context_rows_nhwc(context)
            if out is None:
                out = fused_forward(plan, depth, context, context_rows)
        ctx.plan, ctx.route = plan, route
        ctx.save_for_backward(depth, context, context_rows)
        return out.permute(0, 3, 1, 2)

    @staticmethod
    def backward(ctx, grad_out):
        depth, context, context_rows = ctx.saved_tensors
        with torch.cuda.device(grad_out.device):
            rows = _grad_rows_nhwc(grad_out, ctx.plan)
            grad_depth, grad_context = _fused_backward_rows(ctx.plan, ctx.route, rows, None, depth, context, context_rows)
        return None, grad_depth, grad_context, None, None, None, None


def voxel_pooling_fused(geom_xyz: Optional[torch.Tensor], depth: torch.Tensor, context: torch.Tensor,
                        voxel_num: VoxelNum, plan: Optional[PoolingPlan] = None) -> torch.Tensor:
    """Lift-splat pooling without materialising depth (x) context.

    geom_xyz: int32 (B, N, D, H, W, 3) (ignored when ``plan`` is given); depth (B*N, D, H, W)
    softmax probabilities; context (B*N, C, H, W), NCHW or channels_last.  Returns (B, C, Y, X)
    as a permuted view of a (B, Y, X, C) buffer, like the reference op.

    Under autocast (fp32 ``depth``, fp16 / bf16 ``context``) the result is fp32 and equals, bit for bit, the call on
    ``context.float()``; so do ``grad_depth`` and ``grad_context`` (in the dtype and memory format of ``context``).  On a
    run plan the kernels read the 16-bit context themselves; other cases pool ``context.float()``."""
    return VoxelPoolingFused.apply(geom_xyz, depth, context, voxel_num, plan, None, None)


def _warp_scratch(B: int, Y: int, X: int, C: int, device) -> torch.Tensor:
    """Uninitialised (B, Y, X, C) float32 rows between the pooling and the BDA warp.  Only the rows of occupied cells
    are ever written or read (tests substitute a NaN-filled buffer to prove it)."""
    return torch.empty(B, Y, X, C, dtype=torch.float32, device=device)


def _other_layout(other_bev: torch.Tensor) -> Optional[int]:
    """1 for an NCHW-contiguous ``other_bev``, 0 for channels_last, None for a layout / dtype / alignment the resampling
    kernels do not take (csrc/bev_resample.cu: fp32 / bf16 / fp16, rows of C2 % 4 == 0 elements, vector-aligned)."""
    if other_bev.dtype not in (torch.float32, torch.bfloat16, torch.float16) or other_bev.shape[1] % 4 != 0:
        return None
    if other_bev.is_contiguous():
        return 1
    if other_bev.permute(0, 2, 3, 1).is_contiguous() and other_bev.data_ptr() % 16 == 0:
        return 0
    return None


class VoxelPoolingFusedConcat(Function):
    """``torch.cat([voxel_pooling_fused(...), other_bev], dim=1)`` without the copies of the camera half; with ``theta``
    the camera half is ``warp_affine(voxel_pooling_fused(...), M, (Y, X))`` (``theta`` = ``bev_augment.warp_theta(M)``);
    with ``resize`` the other half is ``F.interpolate(other_bev, size=(Y, X), mode='nearest')``.  The other half is
    written by ``bevpool_resize_nearest_into`` in either case (identity maps when the sizes agree).  ``dtype`` fp16 /
    bf16: the buffer holds the fp32 values rounded once, and the backward reads the 16-bit gradient as it comes (camera
    rows widened to fp32 for occupied cells only, by the warp backward or ``bevpool_grad_rows_widen``)."""

    @staticmethod
    def forward(ctx, depth, context, other_bev, voxel_num, plan, theta=None, resize=False, dtype=torch.float32):
        _lib.require_cuda(depth, context, other_bev)
        X, Y, _ = _voxel_num_ints(voxel_num)
        C = context.shape[1]
        B = plan.batch
        assert other_bev.shape[0] == B and (resize or tuple(other_bev.shape[2:]) == (Y, X))
        C2, Yl, Xl = other_bev.shape[1:]
        other_nchw = _other_layout(other_bev)
        assert other_nchw is not None
        Ct = C + C2
        route = _route(plan.mode, context, depth)
        with torch.cuda.device(depth.device):
            rows = None if route == 'nchw' else context_rows_nhwc(context)
            buf = torch.empty(B, Y, X, Ct, dtype=dtype, device=depth.device)
            if theta is None:
                fused_forward(plan, depth, context, rows, out=buf[..., :C])
            else:
                # the pooled rows go to a scratch first, occupied cells only (no zero fill): the warp skips the taps of
                # empty cells through the plan's cell_start
                from ..bev_augment import warp_forward_rows
                pooled = fused_forward(plan, depth, context, rows, out=_warp_scratch(B, Y, X, C, depth.device),
                                       prezeroed=True)
                warp_forward_rows(theta, pooled, C, buf, Ct, plan.cell_start, B, C, (Y, X), (Y, X))
            # the other half (resampled or not): the one copy a cat cannot avoid
            if dtype == torch.float32:
                _lib.check(_lib.lib().bevpool_resize_nearest_into(
                    other_bev.data_ptr(), _lib.dtype_code(other_bev), other_nchw, B, C2, Yl, Xl, Y, X,
                    buf[..., C:].data_ptr(), Ct, _lib.stream_ptr(depth.device)), 'bevpool_resize_nearest_into')
            else:
                _lib.check(_lib.lib().bevpool_resize_nearest_into16(
                    other_bev.data_ptr(), _lib.dtype_code(other_bev), other_nchw, B, C2, Yl, Xl, Y, X,
                    buf[..., C:].data_ptr(), Ct, _lib.dtype_code(buf), _lib.stream_ptr(depth.device)),
                    'bevpool_resize_nearest_into16')
        ctx.plan, ctx.route, ctx.C, ctx.other_dtype, ctx.theta = plan, route, C, other_bev.dtype, theta
        ctx.other_shape, ctx.other_nchw, ctx.other_code = (B, C2, Yl, Xl), other_nchw, _lib.dtype_code(other_bev)
        ctx.half = dtype != torch.float32
        ctx.save_for_backward(depth, context, rows)
        return buf.permute(0, 3, 1, 2)

    @staticmethod
    def backward(ctx, grad_cat):
        plan, C = ctx.plan, ctx.C
        depth, context, rows = ctx.saved_tensors
        B = plan.batch
        X, Y, _ = plan.voxel_num
        g = grad_cat.permute(0, 2, 3, 1)
        half = ctx.half
        if half:                                    # read in its own dtype; only a layout other than channels_last is copied
            if not g.is_contiguous() or g.data_ptr() % 16 != 0:
                g = g.contiguous()
        elif not g.is_contiguous() or g.dtype != torch.float32:           # channels_last gradients (the usual case) pass as they are
            g = g.float().contiguous()
        Ct = g.shape[-1]
        with torch.cuda.device(depth.device):
            grad_rows, stride = g[..., :C], Ct
            if ctx.theta is not None:
                # gradient of the pooled rows = warp backward of the camera half of grad_cat, occupied cells only (the
                # pooling backward reads no other row)
                from ..bev_augment import warp_backward_rows
                grad_rows, stride = _warp_scratch(B, Y, X, C, depth.device), C
                warp_backward_rows(ctx.theta, g, Ct, grad_rows, C, plan.cell_start, B, C, (Y, X), (Y, X))
            elif half:
                # the camera slice widened to fp32 rows, occupied cells only: the rows the column backward reads
                grad_rows, stride = _warp_scratch(B, Y, X, C, depth.device), C
                _lib.check(_lib.lib().bevpool_grad_rows_widen(
                    plan.cell_start.data_ptr(), g.data_ptr(), Ct, _lib.dtype_code(g), grad_rows.data_ptr(), B, C, X, Y,
                    _lib.stream_ptr(depth.device)), 'bevpool_grad_rows_widen')
            grad_depth, grad_context = _fused_backward_rows(plan, ctx.route, grad_rows, stride, depth, context, rows)
            _, C2, Yl, Xl = ctx.other_shape
            if (Yl, Xl) == (Y, X):
                grad_other = g[..., C:].permute(0, 3, 1, 2).to(ctx.other_dtype)      # identity maps: a view
            elif not ctx.needs_input_grad[2]:
                grad_other = None
            else:
                # adjoint gather straight out of the concatenated gradient; the layout of other_bev
                if ctx.other_nchw:
                    grad_other = torch.empty(B, C2, Yl, Xl, dtype=ctx.other_dtype, device=depth.device)
                else:
                    grad_other = torch.empty(B, Yl, Xl, C2, dtype=ctx.other_dtype, device=depth.device).permute(0, 3, 1, 2)
                if half:
                    _lib.check(_lib.lib().bevpool_resize_nearest_backward_from16(
                        g[..., C:].data_ptr(), Ct, _lib.dtype_code(g), grad_other.data_ptr(), ctx.other_code, ctx.other_nchw,
                        B, C2, Yl, Xl, Y, X, _lib.stream_ptr(depth.device)), 'bevpool_resize_nearest_backward_from16')
                else:
                    _lib.check(_lib.lib().bevpool_resize_nearest_backward_from(
                        g[..., C:].data_ptr(), Ct, grad_other.data_ptr(), ctx.other_code, ctx.other_nchw, B, C2,
                        Yl, Xl, Y, X, _lib.stream_ptr(depth.device)), 'bevpool_resize_nearest_backward_from')
        return grad_depth, grad_context, grad_other, None, None, None, None, None


def voxel_pooling_fused_concat(depth: torch.Tensor, context: torch.Tensor, other_bev: torch.Tensor, voxel_num: VoxelNum,
                               plan: PoolingPlan, *, bda_affine: Optional[torch.Tensor] = None,
                               resize_other: Optional[str] = None, dtype: Optional[torch.dtype] = None) -> torch.Tensor:
    """Concat epilogue of the camera branch (``models/bev_depth.py:187-189``): returns
    ``torch.cat([voxel_pooling_fused(None, depth, context, voxel_num, plan), other_bev], dim=1)`` as a float32
    channels-last tensor.  On a run plan (fp32, W % 4 == 0) the pooled rows are written straight into the concatenated
    buffer and the backward reads its gradient rows straight out of the concatenated gradient -- neither
    ``lss_fpn.py:466``'s ``.contiguous()`` nor the cat copies the camera half; other cases compose the two stock ops.

    ``bda_affine``: the BDA matrix as ``bev_augment_image`` passes it to kornia, (B, 2, 3), no gradient.  The camera
    half is then ``warp_affine(voxel_pooling_fused(...), bda_affine, (Y, X))`` (``ops/bev_augment.py``).  On a run plan
    the pooled map is never zero-filled: the warp skips the empty cells the plan knows of, and its backward produces
    gradient rows for occupied cells only.

    ``resize_other='nearest'``: ``other_bev`` (B, C2, Yl, Xl), any Yl, Xl >= 1, is resampled to the camera grid first --
    the other half is ``F.interpolate(other_bev, size=(Y, X), mode='nearest').float()`` (``bev_depth.py:188-190``), bit
    for bit.  On the native path (fp32 / bf16 / fp16, NCHW or channels_last, C2 % 4 == 0) the resampled rows are written
    straight into the concatenated buffer, and the gradient of ``other_bev`` is gathered straight out of the concatenated
    gradient: the exact adjoint of the forward's index maps, summed in fp32 in torch's order (ascending y, then x) and
    rounded once, in the dtype and memory format of ``other_bev``; no atomics.  ``None`` (default): ``other_bev`` must
    already be (B, C2, Y, X).  Other modes raise ``ValueError``.

    ``dtype``: ``None`` / ``torch.float32`` (default) returns the float32 buffer above.  ``torch.bfloat16`` /
    ``torch.float16`` (what the first conv casts to under autocast) returns that dtype, equal bit for bit to the float32
    result ``.to(dtype)``: every value is still computed in fp32, and each output element is rounded once where it is
    stored (fp16 overflow gives +-inf).  Its backward takes the 16-bit gradient as it comes, in any memory format, and
    gives ``depth``, ``context`` and ``other_bev`` the gradients the float32 call gives for ``grad.float()``, bit for bit,
    in the same dtypes and layouts; with identical grid sizes the gradient of an ``other_bev`` of that dtype is a view.
    On the native path the result is a channels-last view of one (B, Y, X, C + C2) buffer, and no float32 copy of the
    buffer or of its gradient is made; elsewhere the float32 result is cast.  Other dtypes raise ``ValueError``."""
    if resize_other not in (None, 'nearest'):
        raise ValueError(f"resize_other must be None or 'nearest' (got {resize_other!r})")
    if dtype not in (None, torch.float32, torch.float16, torch.bfloat16):
        raise ValueError(f'dtype must be None, torch.float32, torch.float16 or torch.bfloat16 (got {dtype})')
    half = dtype in (torch.float16, torch.bfloat16)
    if other_bev.shape[0] != plan.batch:
        raise ValueError(f'other_bev has batch {other_bev.shape[0]}, the plan {plan.batch}')
    X, Y, _ = plan.voxel_num
    fast = (_route(plan.mode, context, depth) != 'points' and depth.shape[3] % 4 == 0
            and _other_layout(other_bev) is not None and depth.is_contiguous())
    resize = resize_other is not None
    if bda_affine is not None and bda_affine.shape[0] != plan.batch:
        raise ValueError(f'bda_affine has {bda_affine.shape[0]} matrices for a batch of {plan.batch}')
    if fast:
        theta = None
        if bda_affine is not None:
            from ..bev_augment import warp_theta
            theta = warp_theta(bda_affine, (Y, X), (Y, X)).to(depth.device)
        if half:
            return VoxelPoolingFusedConcat.apply(depth, context, other_bev, voxel_num, plan, theta, resize, dtype)
        return VoxelPoolingFusedConcat.apply(depth, context, other_bev, voxel_num, plan, theta, resize)
    camera = voxel_pooling_fused(None, depth, context, voxel_num, plan)
    if bda_affine is not None:
        from ..bev_augment import warp_affine
        camera = warp_affine(camera, bda_affine, (Y, X))
    if resize:
        other_bev = torch.nn.functional.interpolate(other_bev, size=(Y, X), mode='nearest')
    out = torch.cat([camera, other_bev.to(camera.dtype)], dim=1)
    return out.to(dtype) if half else out


class VoxelPoolingFusedLogits(Function):
    """Pooling straight from DepthNet's output tensor: softmax over the depth logits (``lss_fpn.py:423``) and the
    channel slices of ``:441-443`` happen inside the forward kernel."""

    @staticmethod
    def forward(ctx, depth_feature, depth_channels, channels, voxel_num, plan):
        _lib.require_cuda(depth_feature)
        X, Y, _ = _voxel_num_ints(voxel_num)
        BN, Ct, H, W = depth_feature.shape
        D, C = int(depth_channels), int(channels)
        B = plan.batch
        N = BN // B
        assert plan.mode == 'runs' and plan.frustum == (N, D, H, W) and depth_feature.is_contiguous()
        dev = depth_feature.device
        with torch.cuda.device(dev):
            out = torch.empty(B, Y, X, C, dtype=torch.float32, device=dev)
            stats = torch.empty(BN, H, W, 2, dtype=torch.float32, device=dev)
            run_rows, cap, ws = _run_scratch(plan, C, dev)
            _lib.check(_lib.lib().bevpool_fused_forward_runs_logits(
                plan.ptr, depth_feature.data_ptr(), Ct, D, stats.data_ptr(), out.data_ptr(), 0, _lib.dtype_code(depth_feature),
                B, N, D, H, W, C, X, Y, run_rows.data_ptr(), cap, ws.data_ptr(), _lib.stream_ptr(dev)),
                'bevpool_fused_forward_runs_logits')
        ctx.plan, ctx.D, ctx.C = plan, D, C
        ctx.save_for_backward(depth_feature)
        return out.permute(0, 3, 1, 2)

    @staticmethod
    def backward(ctx, grad_out):
        from ..depth_distribution import _backward as softmax_backward, _forward as softmax_forward
        (depth_feature,) = ctx.saved_tensors
        D, C = ctx.D, ctx.C
        with torch.cuda.device(grad_out.device):
            prob, _, _ = softmax_forward(depth_feature[:, :D], None)          # recomputed: the forward never stored it
            context = depth_feature[:, D:D + C].contiguous()
            rows = _grad_rows_nhwc(grad_out, ctx.plan)
            # the route the gate admitted: prob and the context copy are fresh NCHW tensors of the same width
            grad_depth, grad_context = _fused_backward_rows(ctx.plan, 'nchw', rows, None, prob, context, None)
            grad_logits = softmax_backward(prob, None, grad_depth, None, depth_feature.dtype)
            grad_feature = torch.zeros_like(depth_feature) if depth_feature.shape[1] > D + C else torch.empty_like(depth_feature)
            grad_feature[:, :D] = grad_logits
            grad_feature[:, D:D + C] = grad_context
        return grad_feature, None, None, None, None


def voxel_pooling_fused_logits(depth_feature: torch.Tensor, depth_channels: int, channels: int, voxel_num: VoxelNum,
                               plan: PoolingPlan) -> torch.Tensor:
    """``depth_feature`` (B*N, >= D + C, H, W): DepthNet's output (``lss_fpn.py:415-423``) -- depth logits in channels
    [0, D), context in [D, D + C).  Equals ``voxel_pooling_fused(None, depth_feature[:, :D].softmax(1),
    depth_feature[:, D:D+C], voxel_num, plan)`` without the probability tensor or the slice copies (run plan, fp32,
    W % 4 == 0, C in RUN_CHANNELS; other cases compose the stock ops).  For training runs that also need the
    probabilities (depth loss) use ``depth_distribution`` + ``voxel_pooling_fused``."""
    D, C = int(depth_channels), int(channels)
    if _route(plan.mode, depth_feature, depth_feature, channels=C) == 'nchw':
        return VoxelPoolingFusedLogits.apply(depth_feature, D, C, voxel_num, plan)
    return voxel_pooling_fused(None, depth_feature[:, :D].softmax(1).contiguous(), depth_feature[:, D:D + C].contiguous(),
                               voxel_num, plan)

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


def _nchw_direct(context: torch.Tensor, depth: torch.Tensor) -> bool:
    """NCHW-contiguous fp32 context whose rows are multiples of 16 bytes: the kernels read it through a TMA
    tensor map, no layout pass."""
    return (context.is_contiguous() and context.dtype == torch.float32 and context.shape[3] % 4 == 0
            and context.shape[1] in RUN_CHANNELS and context.data_ptr() % 16 == 0 and depth.data_ptr() % 16 == 0
            and os.environ.get('BEVPOOL_DISABLE_G8', '0') != '1' and os.environ.get('BEVPOOL_NCHW_DIRECT', '1') != '0')


def fused_forward(plan: PoolingPlan, depth: torch.Tensor, context: torch.Tensor,
                  context_rows: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None,
                  prezeroed: bool = False) -> torch.Tensor:
    """depth (B*N, D, H, W), context (B*N, C, H, W) NCHW or channels_last -> (B, Y, X, C).  ``out``: a caller-provided
    (B, Y, X, C) buffer; ``prezeroed``: it already holds zeros (run plans only: the kernels then write occupied cells
    only -- see ``fused_forward_cold``)."""
    BN, D, H, W = depth.shape
    C = context.shape[1]
    X, Y, _ = plan.voxel_num
    B = plan.batch
    N = BN // B
    assert context.shape == (BN, C, H, W) and depth.dtype == context.dtype
    assert B * N == BN and plan.num_points == N * D * H * W
    with torch.cuda.device(depth.device):
        if out is None:
            out = torch.empty(B, Y, X, C, dtype=depth.dtype, device=depth.device)
            prezeroed = False
        assert out.shape == (B, Y, X, C) and out.is_contiguous() and out.dtype == depth.dtype
        if plan.mode == 'runs':
            if not runs_supported(C, depth.dtype):
                raise ValueError(f'run plans need float32 and C in {RUN_CHANNELS}; build a point plan for C={C}, {depth.dtype}')
            assert plan.frustum == (N, D, H, W)
            cap = max(1, plan.num_sorted)
            run_rows = torch.empty(cap, C, dtype=torch.float32, device=depth.device)
            ws = _forward_workspace(C, out.device)
            nchw = context_rows is None and _nchw_direct(context, depth)
            ctx_arg = context if nchw else (context_rows_nhwc(context) if context_rows is None else context_rows)
            _lib.check(_lib.lib().bevpool_fused_forward_runs_into(
                plan.ptr, depth.data_ptr(), ctx_arg.data_ptr(), (1 if nchw else 0) | (2 if prezeroed else 0), out.data_ptr(), C,
                _lib.dtype_code(depth), B, N, D, H, W, C, X, Y, run_rows.data_ptr(), cap, ws.data_ptr(),
                _lib.stream_ptr(depth.device)), 'bevpool_fused_forward_runs_into')
            return out
        ctx_nhwc = context_rows_nhwc(context) if context_rows is None else context_rows
        ws = _forward_workspace(C, out.device)
        _lib.check(_lib.lib().bevpool_fused_forward(plan.ptr, depth.data_ptr(), ctx_nhwc.data_ptr(),
                                                    out.data_ptr(), _lib.dtype_code(depth), B, N, D, H, W,
                                                    C, X, Y, ws.data_ptr(), _lib.stream_ptr(depth.device)),
                   'bevpool_fused_forward')
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
        if plan.mode != 'runs':
            return plan, fused_forward(plan, depth, context, out=out)
        return plan, fused_forward(plan, depth, context, out=out, prezeroed=True)


def fused_backward(plan: PoolingPlan, grad_output: torch.Tensor, depth: torch.Tensor,
                   context: torch.Tensor, context_rows: Optional[torch.Tensor] = None):
    """grad_output (B, C, Y, X), any strides -> (grad_depth, grad_context).  grad_context has the
    memory format of ``context``: channels_last in -> channels_last out (zero-copy), NCHW in ->
    NCHW out (written NCHW by the kernel through a TMA tensor map; one tiled transpose on the generic path)."""
    BN, D, H, W = depth.shape
    C = context.shape[1]
    X, Y, _ = plan.voxel_num
    B = plan.batch
    N = BN // B
    with torch.cuda.device(depth.device):
        rows = _grad_rows_nhwc(grad_output, plan)
        grad_depth = torch.empty_like(depth)
        runs = plan.mode == 'runs' and runs_supported(C, depth.dtype)
        if runs and context_rows is None and _nchw_direct(context, depth):
            grad_context = torch.empty_like(context)
            _lib.check(_lib.lib().bevpool_fused_backward_runs(
                plan.ptr, rows.data_ptr(), depth.data_ptr(), context.data_ptr(), grad_depth.data_ptr(),
                grad_context.data_ptr(), 1, _lib.dtype_code(depth), B, N, D, H, W, C, X, Y,
                _lib.stream_ptr(depth.device)), 'bevpool_fused_backward_runs')
            return grad_depth, grad_context
        channels_last = context.permute(0, 2, 3, 1).is_contiguous()
        ctx_nhwc = context_rows_nhwc(context) if context_rows is None else context_rows
        grad_ctx_nhwc = torch.empty(BN, H, W, C, dtype=context.dtype, device=context.device)
        if runs:
            _lib.check(_lib.lib().bevpool_fused_backward_runs(
                plan.ptr, rows.data_ptr(), depth.data_ptr(), ctx_nhwc.data_ptr(), grad_depth.data_ptr(),
                grad_ctx_nhwc.data_ptr(), 0, _lib.dtype_code(depth), B, N, D, H, W, C, X, Y,
                _lib.stream_ptr(depth.device)), 'bevpool_fused_backward_runs')
        else:
            _lib.check(_lib.lib().bevpool_fused_backward(
                plan.ptr, rows.data_ptr(), depth.data_ptr(), ctx_nhwc.data_ptr(), grad_depth.data_ptr(),
                grad_ctx_nhwc.data_ptr(), _lib.dtype_code(depth), B, N, D, H, W, C, X, Y,
                _lib.stream_ptr(depth.device)), 'bevpool_fused_backward')
        if channels_last:
            grad_context = grad_ctx_nhwc.permute(0, 3, 1, 2)
        else:
            grad_context = _transpose(grad_ctx_nhwc, BN, H * W, C).view(BN, C, H, W)
    return grad_depth, grad_context


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
            if plan is None and make_plan is not None:
                # cold call with a caller-supplied plan builder (e.g. from the camera rig): fill overlapped with the build
                if _nchw_direct(context, depth):
                    plan, out = fused_forward_cold(make_plan, int(batch), (X, Y, Z), depth, context)
                    if plan.mode == 'runs':
                        ctx.plan, ctx.direct = plan, True
                        ctx.save_for_backward(depth, context)
                        return out.permute(0, 3, 1, 2)
                else:
                    plan = make_plan()
            if plan is None:
                assert geom_xyz.is_contiguous()
                frustum = None
                # (a run plan reads its run count back once to size the scratch rows: not while capturing)
                if (geom_xyz.dim() == 6 and runs_supported(context.shape[1], depth.dtype)
                        and not torch.cuda.is_current_stream_capturing()):
                    frustum = tuple(geom_xyz.shape[1:5])      # (N, D, H, W): sort runs, not points
                if frustum is not None and _nchw_direct(context, depth):
                    # cold call: zero fill of the output overlapped with the plan build
                    plan, out = fused_forward_cold(lambda: PoolingPlan(geom_xyz, (X, Y, Z), frustum), int(geom_xyz.shape[0]),
                                                   (X, Y, Z), depth, context)
                    ctx.plan, ctx.direct = plan, True
                    ctx.save_for_backward(depth, context)
                    return out.permute(0, 3, 1, 2)
                plan = PoolingPlan(geom_xyz, (X, Y, Z), frustum)
            assert plan.voxel_num == (X, Y, Z)
            direct = plan.mode == 'runs' and _nchw_direct(context, depth)
            context_rows = None if direct else context_rows_nhwc(context)
            out = fused_forward(plan, depth, context, context_rows)
        ctx.plan = plan
        ctx.direct = direct
        if direct:
            ctx.save_for_backward(depth, context)
        else:
            ctx.save_for_backward(depth, context, context_rows)   # the rows are reused by backward
        return out.permute(0, 3, 1, 2)

    @staticmethod
    def backward(ctx, grad_out):
        if ctx.direct:
            (depth, context), context_rows = ctx.saved_tensors, None
        else:
            depth, context, context_rows = ctx.saved_tensors
        with torch.cuda.device(grad_out.device):
            grad_depth, grad_context = fused_backward(ctx.plan, grad_out, depth, context, context_rows)
        return None, grad_depth, grad_context, None, None, None, None


def voxel_pooling_fused(geom_xyz: Optional[torch.Tensor], depth: torch.Tensor, context: torch.Tensor,
                        voxel_num: VoxelNum, plan: Optional[PoolingPlan] = None) -> torch.Tensor:
    """Lift-splat pooling without materialising depth (x) context.

    geom_xyz: int32 (B, N, D, H, W, 3) (ignored when ``plan`` is given); depth (B*N, D, H, W)
    softmax probabilities; context (B*N, C, H, W), NCHW or channels_last.  Returns (B, C, Y, X)
    as a permuted view of a (B, Y, X, C) buffer, like the reference op."""
    return VoxelPoolingFused.apply(geom_xyz, depth, context, voxel_num, plan, None, None)


def _warp_scratch(B: int, Y: int, X: int, C: int, device) -> torch.Tensor:
    """Uninitialised (B, Y, X, C) float32 rows between the pooling and the BDA warp.  Only the rows of occupied cells
    are ever written or read (tests substitute a NaN-filled buffer to prove it)."""
    return torch.empty(B, Y, X, C, dtype=torch.float32, device=device)


class VoxelPoolingFusedConcat(Function):
    """``torch.cat([voxel_pooling_fused(...), other_bev], dim=1)`` without the copies of the camera half; with ``theta``
    the camera half is ``warp_affine(voxel_pooling_fused(...), M, (Y, X))`` (``theta`` = ``bev_augment.warp_theta(M)``)."""

    @staticmethod
    def forward(ctx, depth, context, other_bev, voxel_num, plan, theta=None):
        _lib.require_cuda(depth, context, other_bev)
        X, Y, _ = _voxel_num_ints(voxel_num)
        BN, D, H, W = depth.shape
        C = context.shape[1]
        B = plan.batch
        N = BN // B
        assert other_bev.shape[0] == B and tuple(other_bev.shape[2:]) == (Y, X)
        C2 = other_bev.shape[1]
        Ct = C + C2
        nchw = _nchw_direct(context, depth)
        rows = None if nchw else context_rows_nhwc(context)
        with torch.cuda.device(depth.device):
            buf = torch.empty(B, Y, X, Ct, dtype=torch.float32, device=depth.device)
            cap = max(1, plan.num_sorted)
            run_rows = torch.empty(cap, C, dtype=torch.float32, device=depth.device)
            ws = _forward_workspace(C, depth.device)
            # with the warp, the pooled rows go to a scratch first -- occupied cells only (no zero fill): the warp skips
            # the taps of empty cells through the plan's cell_start
            pooled, stride = (buf, Ct) if theta is None else (_warp_scratch(B, Y, X, C, depth.device), C)
            _lib.check(_lib.lib().bevpool_fused_forward_runs_into(
                plan.ptr, depth.data_ptr(), (context if nchw else rows).data_ptr(),
                (1 if nchw else 0) | (0 if theta is None else 2), pooled.data_ptr(), stride,
                _lib.dtype_code(depth), B, N, D, H, W, C, X, Y, run_rows.data_ptr(), cap, ws.data_ptr(),
                _lib.stream_ptr(depth.device)), 'bevpool_fused_forward_runs_into')
            if theta is not None:
                from ..bev_augment import warp_forward_rows
                warp_forward_rows(theta, pooled, C, buf, Ct, plan.cell_start, B, C, (Y, X), (Y, X))
            buf[..., C:].copy_(other_bev.permute(0, 2, 3, 1))          # the other half: the one copy a cat cannot avoid
        ctx.plan, ctx.nchw, ctx.C, ctx.other_dtype, ctx.theta = plan, nchw, C, other_bev.dtype, theta
        if nchw:
            ctx.save_for_backward(depth, context)
        else:
            ctx.save_for_backward(depth, context, rows)
        return buf.permute(0, 3, 1, 2)

    @staticmethod
    def backward(ctx, grad_cat):
        plan, C = ctx.plan, ctx.C
        if ctx.nchw:
            (depth, context), rows = ctx.saved_tensors, None
        else:
            depth, context, rows = ctx.saved_tensors
        BN, D, H, W = depth.shape
        B = plan.batch
        N = BN // B
        X, Y, _ = plan.voxel_num
        g = grad_cat.permute(0, 2, 3, 1)
        if not g.is_contiguous() or g.dtype != torch.float32:           # channels_last gradients (the usual case) pass as they are
            g = g.float().contiguous()
        Ct = g.shape[-1]
        with torch.cuda.device(depth.device):
            grad_rows, stride = g, Ct
            if ctx.theta is not None:
                # gradient of the pooled rows = warp backward of the camera half of grad_cat, occupied cells only (the
                # pooling backward reads no other row)
                from ..bev_augment import warp_backward_rows
                grad_rows, stride = _warp_scratch(B, Y, X, C, depth.device), C
                warp_backward_rows(ctx.theta, g, Ct, grad_rows, C, plan.cell_start, B, C, (Y, X), (Y, X))
            grad_depth = torch.empty_like(depth)
            if ctx.nchw:
                grad_context = torch.empty_like(context)
                gc_arg = grad_context
            else:
                gc_arg = torch.empty(BN, H, W, C, dtype=context.dtype, device=context.device)
            _lib.check(_lib.lib().bevpool_fused_backward_runs_from(
                plan.ptr, grad_rows.data_ptr(), stride, depth.data_ptr(), (context if ctx.nchw else rows).data_ptr(),
                grad_depth.data_ptr(), gc_arg.data_ptr(), 1 if ctx.nchw else 0, _lib.dtype_code(depth), B, N, D, H, W, C, X, Y,
                _lib.stream_ptr(depth.device)), 'bevpool_fused_backward_runs_from')
            if not ctx.nchw:
                if context.permute(0, 2, 3, 1).is_contiguous():
                    grad_context = gc_arg.permute(0, 3, 1, 2)
                else:
                    grad_context = _transpose(gc_arg, BN, H * W, C).view(BN, C, H, W)
        grad_other = g[..., C:].permute(0, 3, 1, 2).to(ctx.other_dtype)
        return grad_depth, grad_context, grad_other, None, None, None


def voxel_pooling_fused_concat(depth: torch.Tensor, context: torch.Tensor, other_bev: torch.Tensor, voxel_num: VoxelNum,
                               plan: PoolingPlan, *, bda_affine: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Concat epilogue of the camera branch (``models/bev_depth.py:187-189``): returns
    ``torch.cat([voxel_pooling_fused(None, depth, context, voxel_num, plan), other_bev], dim=1)`` as a float32
    channels-last tensor.  On a run plan (fp32, W % 4 == 0) the pooled rows are written straight into the concatenated
    buffer and the backward reads its gradient rows straight out of the concatenated gradient -- neither
    ``lss_fpn.py:466``'s ``.contiguous()`` nor the cat copies the camera half; other cases compose the two stock ops.

    ``bda_affine``: the BDA matrix as ``bev_augment_image`` passes it to kornia, (B, 2, 3), no gradient.  The camera
    half is then ``warp_affine(voxel_pooling_fused(...), bda_affine, (Y, X))`` (``ops/bev_augment.py``).  On a run plan
    the pooled map is never zero-filled: the warp skips the empty cells the plan knows of, and its backward produces
    gradient rows for occupied cells only."""
    C = context.shape[1]
    fast = (plan.mode == 'runs' and runs_supported(C, depth.dtype) and depth.shape[3] % 4 == 0
            and other_bev.shape[1] % 4 == 0 and depth.is_contiguous())
    if bda_affine is None:
        if fast:
            return VoxelPoolingFusedConcat.apply(depth, context, other_bev, voxel_num, plan, None)
        return torch.cat([voxel_pooling_fused(None, depth, context, voxel_num, plan), other_bev.to(depth.dtype)], dim=1)
    from ..bev_augment import warp_affine, warp_theta
    X, Y, _ = plan.voxel_num
    if bda_affine.shape[0] != plan.batch:
        raise ValueError(f'bda_affine has {bda_affine.shape[0]} matrices for a batch of {plan.batch}')
    if fast:
        theta = warp_theta(bda_affine, (Y, X), (Y, X)).to(depth.device)
        return VoxelPoolingFusedConcat.apply(depth, context, other_bev, voxel_num, plan, theta)
    pooled = voxel_pooling_fused(None, depth, context, voxel_num, plan)
    return torch.cat([warp_affine(pooled, bda_affine, (Y, X)), other_bev.to(pooled.dtype)], dim=1)


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
            cap = max(1, plan.num_sorted)
            run_rows = torch.empty(cap, C, dtype=torch.float32, device=dev)
            ws = _forward_workspace(C, dev)
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
            grad_depth, grad_context = fused_backward(ctx.plan, grad_out, prob, context)
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
    if (plan.mode == 'runs' and runs_supported(C, depth_feature.dtype) and depth_feature.shape[3] % 4 == 0
            and depth_feature.is_contiguous() and depth_feature.data_ptr() % 16 == 0
            and os.environ.get('BEVPOOL_NCHW_DIRECT', '1') != '0'):
        return VoxelPoolingFusedLogits.apply(depth_feature, D, C, voxel_num, plan)
    return voxel_pooling_fused(None, depth_feature[:, :D].softmax(1).contiguous(), depth_feature[:, D:D + C].contiguous(),
                               voxel_num, plan)

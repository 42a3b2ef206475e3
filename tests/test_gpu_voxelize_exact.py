"""The voxelizer's float outputs bit for bit: the fused HardSimpleVFE mean and its canvas against
``oracle.voxelize_ref.vfe_mean_exact`` / ``canvas_exact`` (a float32 sum from +0 in slot order, one IEEE division), on
every finalize, gather and canvas route; the padded-output contract (every row >= voxel_base[B] zero, only live rows on
the canvas) on both pipelines; the hash pipeline at the grid sizes that select it; unaligned and ragged clouds; every
tuning knob; and the pillar scatter's duplicate / out-of-range rules.

Float tensors are compared as int32 bit patterns.  Means and canvases may hold NaN, whose payload the GPU canonicalises:
there the NaN positions must agree and every other element must be bit-equal."""
import contextlib
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from mm_training_b200 import _lib, synthetic
from mm_training_b200.configs import CFG_3
from mm_training_b200.ops import voxelize as vzmod
from mm_training_b200.ops.voxelize import PointPillarsScatter, dynamic_voxelize, hard_voxelize_batch, pillar_scatter
from oracle import voxelize_ref as vz

pytestmark = pytest.mark.gpu
DEV = 'cuda'
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHILD = os.environ.get('BEVVOX_EXACT_CHILD') == '1'
NAN, INF = np.float32(np.nan), np.float32(np.inf)

VS = [1.0, 1.0, 1.0]
RG_EVEN = [0, 0, 0, 8, 8, 2]          # 8 x 8 x 2 = 128 cells (a multiple of 4: the dense canvas kernel)
RG_ODD = [0, 0, 0, 9, 9, 1]           # 81 cells: the canvas is zero-filled and the finalize kernel scatters into it


# ---- helpers ------------------------------------------------------------------------------------------------------
@contextlib.contextmanager
def _poisoned(pattern):
    """While active, every CUDA float32 tensor from ``torch.empty`` is NaN and every int32 one holds ``pattern`` (an
    in-range coordinate: what a previous call's buffers may hold).  The voxelizer's uint8 scratch is left alone."""
    real = torch.empty

    def empty(*args, **kwargs):
        t = real(*args, **kwargs)
        if t.is_cuda and t.dtype == torch.float32:
            t.fill_(float('nan'))
        elif t.is_cuda and t.dtype == torch.int32:
            t.fill_(pattern)
        return t

    torch.empty = empty
    try:
        yield
    finally:
        torch.empty = real


@pytest.fixture(params=[0, 1], ids=['poison0', 'poison1'])
def poisoned(request):
    """``with poisoned(): ...`` runs the block with poisoned output allocations (see ``_poisoned``)."""
    return lambda: _poisoned(request.param)


def _bits(a):
    if isinstance(a, torch.Tensor):
        t = a.detach().cpu().contiguous()
        return t.view(torch.int32 if t.element_size() == 4 else torch.int16).numpy()
    a = np.ascontiguousarray(a)
    return a.view(np.int32 if a.dtype.itemsize == 4 else np.int16)


def _same_bits(got, exp, what=''):
    """Bit-equal, NaN positions included (NaN payloads are not compared)."""
    g = got.detach().float().cpu().numpy() if isinstance(got, torch.Tensor) else np.asarray(got, np.float32)
    e = np.asarray(exp, np.float32)
    assert g.shape == e.shape, (what, g.shape, e.shape)
    gn, en = np.isnan(g), np.isnan(e)
    assert np.array_equal(gn, en), (what, 'NaN positions', int((gn != en).sum()))
    bad = np.nonzero(_bits(g)[~gn] != _bits(e)[~en])[0]
    assert bad.size == 0, (what, int(bad.size), g[~gn][bad[:4]], e[~en][bad[:4]])


def _zero_rows(n, *tensors):
    for t in tensors:
        if t is not None:
            assert int((t[n:].reshape(-1).view(torch.int32) != 0).sum()) == 0, 'padding rows not zero'


def _grid(vs, rg):
    return [int(v) for v in vz.grid_size_ref(vs, rg)]


def _over_the_finalize_limit(path, T, F, B):
    """The dense path's per-lane finalize stages 128 rows of T x F floats in shared memory, at most 200 KB."""
    return path == 'dense' and T > 16 and 4 * 128 * T * F + 4 * (B + 1) > 200 * 1024


def _check_exact(clouds_np, vs, rg, T, M, mf, clouds=None, impl=vz.hard_voxelize_c, pattern=0):
    """Padded fused call (poisoned allocations) against the oracle: integer outputs and point rows bit-exact, mean and
    canvas bit-equal to the float32 emulation, every padding row zero."""
    B = len(clouds_np)
    clouds = clouds if clouds is not None else [torch.from_numpy(c).to(DEV) for c in clouds_np]
    if _over_the_finalize_limit('dense' if os.environ.get('BEVVOX_FORCE_HASH') != '1' else 'hash', T,
                                clouds_np[0].shape[1], B):
        with pytest.raises(ValueError, match='too large'):                        # a documented limit, not a fallback
            hard_voxelize_batch(clouds, vs, rg, T, M, mean_features=mf, padded=True, scatter=True)
        return None
    with _poisoned(pattern):
        out = hard_voxelize_batch(clouds, vs, rg, T, M, mean_features=mf, padded=True, scatter=True)
    voxels, num, coors, base, mean, canvas = out
    rv, rn, rc = vz.voxelize_batch_ref(clouds_np, vs, rg, T, M, impl=impl)
    n = rv.shape[0]
    assert int(base[-1]) == n
    assert np.array_equal(_bits(voxels[:n]), _bits(rv)), 'voxels'
    assert np.array_equal(num[:n].cpu().numpy(), rn) and np.array_equal(coors[:n].cpu().numpy(), rc)
    _same_bits(mean[:n], vz.vfe_mean_exact(rv, rn, mf), 'mean')
    gx, gy, gz = _grid(vs, rg)
    _same_bits(canvas, vz.canvas_exact(rv, rn, rc, mf, B, (gz, gy, gx)), 'canvas')
    _zero_rows(n, voxels, num, coors, mean)
    return out


def _crafted(F, T, seed, rg):
    """A cloud on a small grid whose per-cell point order makes the summation order visible: cells holding every count
    from 1 to T, rows [2^24, 1, 1, ...] and [1e8, 3, -1e8], -0.0 rows, NaN / inf intensities and full cells with hundreds
    of late arrivals.  The special values go in the xyz-independent columns; the points of all cells are interleaved,
    in order inside each cell."""
    rng = np.random.default_rng(seed)
    gx, gy, gz = (int(v) for v in rg[3:])
    E = F - 3
    seqs = [rng.standard_normal((c, E)) * 10.0 ** rng.integers(-2, 4, (c, 1)) for c in range(1, T + 1)]
    seqs += [rng.standard_normal((T + 300, E)) for _ in range(2)]                  # late arrivals
    for s in ([2.0 ** 24] + [1.0] * (T + 1), [1e8, 3.0, -1e8], [-0.0] * 3, [-0.0], [0.5, NAN, 1.0],
              [INF, 1.0], [-INF, 2.0, INF], [3e38, 3e38]):
        seqs.append(np.asarray(s, np.float64)[:, None] * 2.0 ** np.arange(E)[None, :])
    cells = rng.permutation(gx * gy * gz)[:len(seqs)]
    if 0 not in cells:                                     # (cell 0 is where zeroed coordinates would scatter to)
        cells[rng.integers(len(seqs))] = 0
    owner = np.repeat(np.arange(len(seqs)), [len(s) for s in seqs])
    owner = owner[rng.permutation(owner.size)]
    pts = np.zeros((owner.size, F), np.float32)
    taken = np.zeros(len(seqs), np.int64)
    with np.errstate(over='ignore'):                       # (3e38 * 2^j is +inf in float32: one more inf row)
        for i, k in enumerate(owner):
            c = cells[k]
            pts[i, :3] = [c % gx, (c // gx) % gy, c // (gx * gy)]
            pts[i, 3:] = seqs[k][taken[k]]
            taken[k] += 1
    pts[:, :3] += rng.uniform(0.01, 0.99, (owner.size, 3)).astype(np.float32)
    return pts


PAIRS = [(3, 1), (3, 2), (3, 3), (4, 3), (5, 5), (8, 7), (8, 8), (9, 9), (12, 12), (16, 16), (16, 5)]


# ---- mean and canvas on every route (the `core` tests also run under every knob, below) -------------------------------
@pytest.mark.parametrize('path', ['dense', 'hash'])
@pytest.mark.parametrize('T', [1, 7, 16, 20, 35])
@pytest.mark.parametrize('F,mf', PAIRS)
def test_core_mean_and_canvas_bit_exact(F, mf, T, path, monkeypatch):
    # T <= 16: the cooperative finalize (the per-lane one under BEVVOX_FIN_COOP=0), T > 16: the per-lane finalize; F <= 8
    # and F > 8: their FM = 8 / 16 builds; mf <= 8 / > 8: the dense canvas kernel's; path 'hash': the hash gather
    monkeypatch.setenv('BEVVOX_FORCE_HASH', '1' if path == 'hash' else '0')
    clouds = [_crafted(F, T, 10 * F + T, RG_EVEN), np.zeros((0, F), np.float32), _crafted(F, T, 10 * F + T + 1, RG_EVEN)]
    _check_exact(clouds, VS, RG_EVEN, T, 60, mf, pattern=T % 2)


@pytest.mark.parametrize('path', ['dense', 'hash'])
@pytest.mark.parametrize('F,mf,T', [(5, 5, 15), (8, 3, 4), (16, 12, 24), (9, 9, 35)])
def test_core_fill_and_scatter_canvas(F, mf, T, path, monkeypatch):
    # 9 x 9 x 1 cells: not a multiple of 4, so the canvas is zero-filled (side stream) and scattered by the finalize kernel
    monkeypatch.setenv('BEVVOX_FORCE_HASH', '1' if path == 'hash' else '0')
    clouds = [_crafted(F, T, 7 + T, RG_ODD), _crafted(F, T, 8 + T, RG_ODD)]
    _check_exact(clouds, VS, RG_ODD, T, 50, mf)


def _abi(clouds_np, vs, rg, T, M, mf, pattern, with_mean=True, with_canvas=False):
    """The C ABI with output buffers poisoned beforehand (NaN floats, ``pattern`` ints): independent of the allocator."""
    B, F = len(clouds_np), clouds_np[0].shape[1]
    counts = [c.shape[0] for c in clouds_np]
    offs = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
    grid = _grid(vs, rg)
    gx, gy, gz = grid
    L = _lib.lib()
    tb = ctypes.c_size_t()
    _lib.check(L.bevvox_temp_bytes(B, int(offs[-1]), vzmod._i32_array(grid), M, T, ctypes.byref(tb)), 'bevvox_temp_bytes')
    pts = torch.from_numpy(np.concatenate(clouds_np)).to(DEV)
    offsets = torch.from_numpy(offs).to(DEV)
    voxels = torch.full((B * M, T, F), float('nan'), device=DEV)
    coors = torch.full((B * M, 4), pattern, dtype=torch.int32, device=DEV)
    num = torch.full((B * M,), pattern, dtype=torch.int32, device=DEV)
    base = torch.full((B + 1,), pattern, dtype=torch.int32, device=DEV)
    mean = torch.full((B * M, mf), float('nan'), device=DEV) if with_mean else None
    canvas = torch.full((B, mf * gz, gy, gx), float('nan'), device=DEV) if with_canvas else None
    temp = torch.empty(tb.value, dtype=torch.uint8, device=DEV)
    head = [pts.data_ptr(), offsets.data_ptr(), B, int(offs[-1]), max(counts), F, vzmod._f32_array(vs),
            vzmod._f32_array(rg), vzmod._i32_array(grid), T, M, voxels.data_ptr(), coors.data_ptr(), num.data_ptr(),
            base.data_ptr(), mean.data_ptr() if mean is not None else None, mf]
    stream = _lib.stream_ptr(torch.device(DEV))
    if with_canvas:
        _lib.check(L.bevvox_hard_voxelize_scatter(head[0], None, *head[1:], canvas.data_ptr(), 0, temp.data_ptr(), stream),
                   'bevvox_hard_voxelize_scatter')
    else:
        _lib.check(L.bevvox_hard_voxelize(*head, temp.data_ptr(), stream), 'bevvox_hard_voxelize')
    torch.cuda.synchronize()
    rv, rn, rc = vz.voxelize_batch_ref(clouds_np, vs, rg, T, M)
    n = rv.shape[0]
    assert int(base[-1]) == n
    assert np.array_equal(_bits(voxels[:n]), _bits(rv))
    assert np.array_equal(num[:n].cpu().numpy(), rn) and np.array_equal(coors[:n].cpu().numpy(), rc)
    if mean is not None:
        _same_bits(mean[:n], vz.vfe_mean_exact(rv, rn, mf), 'mean')
    if canvas is not None:
        _same_bits(canvas, vz.canvas_exact(rv, rn, rc, mf, B, (gz, gy, gx)), 'canvas')
    _zero_rows(n, voxels, num, coors, mean)


@pytest.mark.parametrize('path', ['dense', 'hash'])
@pytest.mark.parametrize('rg', [RG_EVEN, RG_ODD], ids=['even', 'odd'])
def test_core_abi_canvas_without_a_mean_output(rg, path, monkeypatch):
    # voxel_mean == NULL with a canvas: the fill-and-scatter route whatever the cell count
    monkeypatch.setenv('BEVVOX_FORCE_HASH', '1' if path == 'hash' else '0')
    _abi([_crafted(5, 15, 3, rg), _crafted(5, 15, 4, rg)], VS, rg, 15, 60, 5, pattern=0, with_mean=False, with_canvas=True)


@pytest.mark.parametrize('pattern', [0, 1])
@pytest.mark.parametrize('path', ['dense', 'hash'])
@pytest.mark.parametrize('T', [4, 15, 20])
def test_padded_contract_through_the_abi(T, path, pattern, monkeypatch):
    monkeypatch.setenv('BEVVOX_FORCE_HASH', '1' if path == 'hash' else '0')
    clouds = [_crafted(8, T, 30 + T, RG_EVEN), np.zeros((0, 8), np.float32), _crafted(8, T, 31 + T, RG_EVEN)]
    _abi(clouds, VS, RG_EVEN, T, 70, 6, pattern)
    _abi(clouds, VS, RG_EVEN, T, 70, 6, pattern, with_canvas=True)


# ---- the padded contract on sweeps ------------------------------------------------------------------------------------
@pytest.mark.parametrize('path', ['dense', 'hash'])
def test_padded_rows_are_zero_and_only_live_rows_reach_the_canvas(path, poisoned, monkeypatch):
    # rows >= voxel_base[B] of voxels, num_points, coors and the mean are zero on both pipelines; the canvas holds
    # exactly the exact means of the live rows (stale coordinates in dead rows must not scatter)
    monkeypatch.setenv('BEVVOX_FORCE_HASH', '1' if path == 'hash' else '0')
    clouds_np = [synthetic.lidar_sweep(n, 5, seed=50 + i) for i, n in enumerate([40000, 3, 25000])]
    clouds = [torch.from_numpy(c).to(DEV) for c in clouds_np]
    T, M, mf = 15, 25000, 5
    with poisoned():
        voxels, num, coors, base, mean, canvas = hard_voxelize_batch(clouds, CFG_3.voxel_size, CFG_3.point_cloud_range,
                                                                     T, M, mean_features=mf, padded=True, scatter=True)
    rv, rn, rc = vz.voxelize_batch_ref(clouds_np, CFG_3.voxel_size, CFG_3.point_cloud_range, T, M)
    n = rv.shape[0]
    assert int(base[-1]) == n < 3 * M
    assert np.array_equal(num[:n].cpu().numpy(), rn) and np.array_equal(coors[:n].cpu().numpy(), rc)
    _same_bits(mean[:n], vz.vfe_mean_exact(rv, rn, mf), 'mean')
    gx, gy, gz = _grid(CFG_3.voxel_size, CFG_3.point_cloud_range)
    _same_bits(canvas, vz.canvas_exact(rv, rn, rc, mf, 3, (gz, gy, gx)), 'canvas')
    _zero_rows(n, voxels, num, coors, mean)


def test_hash_canvas_after_a_denser_call(monkeypatch):
    # a training loop: the second call's buffers are likely the first call's, whose live rows held real coordinates
    # and means.  The second (sparser) call's canvas must hold its own voxels only.
    monkeypatch.setenv('BEVVOX_FORCE_HASH', '1')
    T, M, mf = 15, 20000, 5
    dense_np = [synthetic.lidar_sweep(150000, 5, seed=60 + i) for i in range(2)]
    first = hard_voxelize_batch([torch.from_numpy(c).to(DEV) for c in dense_np], CFG_3.voxel_size,
                                CFG_3.point_cloud_range, T, M, mean_features=mf, padded=True, scatter=True)
    assert int(first[3][-1]) > 30000
    del first
    sparse_np = [synthetic.lidar_sweep(n, 5, seed=62 + i) for i, n in enumerate([2000, 500])]
    voxels, num, coors, base, mean, canvas = hard_voxelize_batch(
        [torch.from_numpy(c).to(DEV) for c in sparse_np], CFG_3.voxel_size, CFG_3.point_cloud_range, T, M,
        mean_features=mf, padded=True, scatter=True)
    rv, rn, rc = vz.voxelize_batch_ref(sparse_np, CFG_3.voxel_size, CFG_3.point_cloud_range, T, M)
    gx, gy, gz = _grid(CFG_3.voxel_size, CFG_3.point_cloud_range)
    _same_bits(canvas, vz.canvas_exact(rv, rn, rc, mf, 2, (gz, gy, gx)), 'canvas')
    _zero_rows(rv.shape[0], voxels, num, coors, mean)


@pytest.mark.parametrize('case', ['sweeps', 'crafted'])
def test_dense_and_hash_pipelines_are_equal(case, monkeypatch):
    if case == 'sweeps':
        clouds = [synthetic.lidar_sweep(60000, 8, seed=70), synthetic.lidar_sweep(30000, 8, seed=71)]
        geom, T, M = (CFG_3.voxel_size, CFG_3.point_cloud_range), 15, 25000
    else:
        clouds = [_crafted(8, 20, 72, RG_EVEN), _crafted(8, 20, 73, RG_EVEN)]
        geom, T, M = (VS, RG_EVEN), 20, 60
    clouds = [torch.from_numpy(c).to(DEV) for c in clouds]
    outs = []
    for path in ('0', '1'):
        monkeypatch.setenv('BEVVOX_FORCE_HASH', path)
        with _poisoned(int(path)):
            outs.append(hard_voxelize_batch(clouds, *geom, T, M, mean_features=7, padded=True, scatter=True))
    for a, b in zip(*outs):
        assert torch.equal(a.view(torch.int32) if a.dtype == torch.float32 else a,
                           b.view(torch.int32) if b.dtype == torch.float32 else b)


# ---- the hash pipeline where it is selected by size (no environment variable) -----------------------------------------
def _check_large(clouds_np, vs, rg, T, M, mf):
    """Like ``_check_exact``, but the multi-GB canvas is checked on the GPU: the exact means at the oracle's cells and
    zeros everywhere else."""
    B = len(clouds_np)
    with _poisoned(0):
        voxels, num, coors, base, mean, canvas = hard_voxelize_batch([torch.from_numpy(c).to(DEV) for c in clouds_np],
                                                                     vs, rg, T, M, mean_features=mf, padded=True,
                                                                     scatter=True)
    rv, rn, rc = vz.voxelize_batch_ref(clouds_np, vs, rg, T, M, impl=vz.hard_voxelize_numpy)
    n = rv.shape[0]
    assert int(base[-1]) == n
    assert np.array_equal(_bits(voxels[:n]), _bits(rv))
    assert np.array_equal(num[:n].cpu().numpy(), rn) and np.array_equal(coors[:n].cpu().numpy(), rc)
    exact = vz.vfe_mean_exact(rv, rn, mf)
    _same_bits(mean[:n], exact, 'mean')
    _zero_rows(n, voxels, num, coors, mean)
    gx, gy, gz = _grid(vs, rg)
    cv = canvas.view(B, mf, gz, gy, gx)
    idx = torch.from_numpy(rc.astype(np.int64)).to(DEV)
    at = cv[idx[:, 0], :, idx[:, 1], idx[:, 2], idx[:, 3]]                      # (n, mf)
    _same_bits(at, exact, 'canvas at the voxels')
    assert int((canvas.view(torch.int32) != 0).sum()) == int((at.view(torch.int32) != 0).sum()), 'canvas elsewhere'


def test_hash_pipeline_at_real_size():
    # 0.05 x 0.05 x 0.2 on [-51.2, 51.2]^2 x [-5, 3]: 2048 x 2048 x 40 cells, 2.5x the dense table's limit at B = 1
    vs, rg = [0.05, 0.05, 0.2], [-51.2, -51.2, -5.0, 51.2, 51.2, 3.0]
    assert np.prod(_grid(vs, rg)) == 2048 * 2048 * 40
    pts = synthetic.lidar_sweep(200000, 5, seed=80)
    pts[:, :2] *= 0.25                                       # (most of the sweep inside the +-51.2 m range)
    _check_large([pts], vs, rg, 10, 200000, 4)                # (the cap does not bind: padding rows)
    coors = dynamic_voxelize(torch.from_numpy(pts).to(DEV), vs, rg)
    assert np.array_equal(coors.cpu().numpy(), vz.point_coors_numpy(pts, vs, rg)[0])


@pytest.mark.parametrize('B', [1, 2])
def test_dense_table_limit(B):
    # 8192 x 8192 x 1 = 2^26 cells: the dense table at B = 1, the hash table at B = 2
    vs, rg = [0.0125, 0.0125, 8.0], [-51.2, -51.2, -5.0, 51.2, 51.2, 3.0]
    assert np.prod(_grid(vs, rg)) == 1 << 26
    clouds = [synthetic.lidar_sweep(60000, 5, seed=90 + b) * np.float32([0.25, 0.25, 1, 1, 1]) for b in range(B)]
    _check_large(clouds, vs, rg, 5, 70000, 5)                 # (more rows than points: padding rows)


def test_hash_keys_beyond_2_to_the_31():
    # 33 samples on a 2^26-cell grid: the keys b * cells + cell of the last samples pass 2^31
    vs, rg = [0.0125, 0.0125, 8.0], [-51.2, -51.2, -5.0, 51.2, 51.2, 3.0]
    clouds_np = [synthetic.lidar_sweep(2000, 5, seed=100 + b) * np.float32([0.25, 0.25, 1, 1, 1]) for b in range(33)]
    voxels, num, coors, base, mean = hard_voxelize_batch([torch.from_numpy(c).to(DEV) for c in clouds_np], vs, rg, 5,
                                                         3000, mean_features=5)
    rv, rn, rc = vz.voxelize_batch_ref(clouds_np, vs, rg, 5, 3000, impl=vz.hard_voxelize_numpy)
    assert (rc[:, 0] == 32).sum() > 0
    assert np.array_equal(_bits(voxels), _bits(rv)) and np.array_equal(num.cpu().numpy(), rn)
    assert np.array_equal(coors.cpu().numpy(), rc)
    _same_bits(mean, vz.vfe_mean_exact(rv, rn, 5), 'mean')


# ---- unaligned and ragged clouds --------------------------------------------------------------------------------------
def _offset_view(a, k):
    """``a`` on the GPU as a contiguous view k floats into a buffer (base address 4k bytes past 16-byte alignment)."""
    n, F = a.shape
    buf = torch.empty(n * F + k + 4, device=DEV)
    v = buf[k:k + n * F].view(n, F)
    v.copy_(torch.from_numpy(a))
    assert v.is_contiguous() and v.data_ptr() % 16 == 4 * k
    return v


@pytest.mark.parametrize('B', [1, 3])
@pytest.mark.parametrize('k', [0, 1, 2, 3])
@pytest.mark.parametrize('F', [3, 5, 7])
def test_unaligned_and_ragged_clouds(F, k, B):
    # B = 1: the cloud itself is read (concatenated path); B > 1: through the per-sample pointer table.  Counts with a
    # last tile of 1024-point tiles whose byte count is not a multiple of 16: the scalar loads of vox_cell_kernel
    clouds_np = [synthetic.lidar_sweep(n, F, seed=110 + F + b) for b, n in enumerate([5003, 2049, 1025][:B])]
    for c in clouds_np:
        c[:, 3:] = np.random.default_rng(F).standard_normal((c.shape[0], F - 3)).astype(np.float32)
    clouds = [_offset_view(c, k) for c in clouds_np]
    _check_exact(clouds_np, CFG_3.voxel_size, CFG_3.point_cloud_range, 15, 25000, min(F, 5), clouds=clouds)


# ---- the knob matrix --------------------------------------------------------------------------------------------------
KNOBS = ['BEVVOX_FIN_COOP=0', 'BEVVOX_CANVAS_OVERLAP=0', 'BEVVOX_L2_HINTS=0', 'BEVVOX_L2_HINTS=3', 'BEVVOX_L2_HINTS=7']


@pytest.mark.skipif(CHILD, reason='inside a knob child')
@pytest.mark.parametrize('knob', KNOBS)
def test_knob_matrix(knob):
    """The `core` tests of this file in a fresh process with one knob set (each is read once per process): the same
    bits as the emulation, hence as the default.  BEVVOX_FIN_COOP=0 runs the per-lane finalize for max_points <= 16."""
    key, value = knob.split('=')
    env = dict(os.environ, BEVVOX_EXACT_CHILD='1', **{key: value})
    res = subprocess.run([sys.executable, '-m', 'pytest', os.path.abspath(__file__), '-q', '-m', 'gpu', '-k', 'core',
                          '-p', 'no:cacheprovider'], cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout[-4000:] + res.stderr[-2000:]
    assert ' passed' in res.stdout and ' skipped' not in res.stdout, res.stdout[-2000:]


# ---- pillar scatter ---------------------------------------------------------------------------------------------------
def _scatter_case(seed, M=3000, C=6, B=3, nz=2, ny=24, nx=40):
    rng = np.random.default_rng(seed)
    coors = np.stack([rng.integers(0, B, M), rng.integers(0, nz, M), rng.integers(0, ny, M), rng.integers(0, nx, M)], 1)
    dup = rng.random(M) < 0.3                                                            # many duplicates
    coors[dup] = coors[rng.integers(0, M // 4, int(dup.sum()))]
    bad = rng.random(M) < 0.05                                                           # out of range, every axis
    coors[bad] = np.array([[B, 0, 0, 0], [-1, 0, 0, 0], [0, nz, 0, 0], [0, 0, -1, 0], [0, 0, ny, 0], [0, 0, 0, nx],
                           [0, -1, 0, 0], [0, 0, 0, -1]])[rng.integers(0, 8, int(bad.sum()))]
    return coors.astype(np.int32), (B, nz, ny, nx)


def _in_range(coors, dims):
    B, nz, ny, nx = dims
    return np.all((coors >= 0) & (coors < np.array([B, nz, ny, nx])), 1)


@pytest.mark.parametrize('dtype', [torch.float32, torch.float16, torch.bfloat16])
def test_pillar_scatter_duplicates_out_of_range_and_gradient(dtype):
    coors, dims = _scatter_case(1)
    B, nz, ny, nx = dims
    M, C = coors.shape[0], 6
    feats = torch.randn(M, C).to(dtype)
    ok = _in_range(coors, dims)
    # forward: the highest row wins at a shared cell, rows outside the grid are dropped
    exp = torch.zeros(B, C, nz, ny, nx, dtype=dtype)
    for m in np.nonzero(ok)[0]:                                                          # ascending: the last write wins
        b, z, y, x = coors[m]
        exp[b, :, z, y, x] = feats[m]
    f = feats.to(DEV).requires_grad_(True)
    canvas = pillar_scatter(f, torch.from_numpy(coors).to(DEV), B, (nz, ny, nx))
    assert np.array_equal(_bits(canvas.detach().view(B, C, nz, ny, nx)), _bits(exp))
    # backward: a gather for EVERY row, duplicates included; rows outside the grid get zero.  That is the gradient torch's
    # index_put autograd gives mmdet3d's `canvas[:, indices] = voxels.t()`, whichever duplicate the forward kept.
    g = torch.randn(B, C * nz, ny, nx).to(dtype)
    canvas.backward(g.to(DEV))
    ref_f = feats[ok].clone().requires_grad_(True)
    c = coors[ok].astype(np.int64)
    flat = torch.from_numpy(((c[:, 1] * ny + c[:, 2]) * nx + c[:, 3]))
    ref_grad = torch.zeros(M, C, dtype=dtype)
    for b in range(B):
        sel = torch.from_numpy(c[:, 0] == b)
        cv = torch.zeros(C, nz * ny * nx, dtype=dtype)
        rows = ref_f[sel]
        cv = cv.index_put((torch.arange(C)[:, None], flat[sel][None, :]), rows.t())   # canvas[:, indices] = voxels.t()
        (gb,) = torch.autograd.grad(cv, rows, g.view(B, C, -1)[b])
        ref_grad[torch.from_numpy(np.nonzero(ok)[0])[sel]] = gb
    assert np.array_equal(_bits(f.grad), _bits(ref_grad))
    assert int((f.grad[torch.from_numpy(~ok).to(DEV)] != 0).sum()) == 0


def test_pillar_scatter_unique_path_drops_out_of_range_rows():
    coors, dims = _scatter_case(2)
    B, nz, ny, nx = dims
    ok = _in_range(coors, dims)
    _, first = np.unique(coors[ok], axis=0, return_index=True)           # unique coordinates, plus the invalid rows
    keep = np.concatenate([np.nonzero(ok)[0][first], np.nonzero(~ok)[0]])
    co, feats = coors[keep], torch.randn(keep.size, 4)
    canvas = pillar_scatter(feats.to(DEV), torch.from_numpy(co).to(DEV), B, (nz, ny, nx), unique_coors=True)
    ref = vz.pillar_scatter_ref(feats.numpy()[:first.size], co[:first.size], B, (nz, ny, nx))
    assert np.array_equal(_bits(canvas), _bits(ref))


def test_pillar_scatter_empty_and_batch_size_inference():
    f = torch.zeros(0, 5, device=DEV, requires_grad=True)
    canvas = pillar_scatter(f, torch.zeros(0, 4, dtype=torch.int32, device=DEV), 2, (1, 8, 16))
    assert canvas.shape == (2, 5, 8, 16) and int((canvas != 0).sum()) == 0
    canvas.sum().backward()
    assert f.grad.shape == (0, 5)
    # PointPillarsScatter(batch_size=None): the batch is max(b) + 1 (mmdet3d reads coors[-1, 0] + 1 on sorted rows)
    coors = torch.tensor([[0, 0, 1, 2], [2, 0, 3, 4], [1, 0, 7, 15]], dtype=torch.int32, device=DEV)
    feats = torch.arange(15, dtype=torch.float32, device=DEV).view(3, 5)
    bev = PointPillarsScatter(5, (8, 16))(feats, coors)
    assert bev.shape == (3, 5, 8, 16)
    assert torch.equal(bev[2, :, 3, 4], feats[1]) and torch.equal(bev[1, :, 7, 15], feats[2])
    assert int((bev != 0).sum()) == int((feats != 0).sum())
    assert PointPillarsScatter(5, (8, 16))(feats[:0], coors[:0]).shape == (1, 5, 8, 16)

"""GPU parity tests of the RUN plan and the two-stage fused forward built on it
(csrc/plan.cu ``plan_key_runs_kernel``, csrc/pool_runs.cu).  Integer plan contents are compared
bit-exactly with ``oracle.voxel_pool_ref.run_plan_ref``; the forward is held to rtol 1e-5 against the
fp64 oracle plus 1e-6 of the per-cell sum of magnitudes (the run-wise summation order differs from
the reference's point order, SURVEY.md section 7 hard part 3), and must be bit-stable run to run."""
import pytest
import torch

from mm_training_b200 import synthetic
from mm_training_b200.configs import CFG_2, CFG_AIM, sweep_grid_config
from mm_training_b200.ops.voxel_pooling import build_plan, fused_backward, fused_forward, voxel_pooling_fused
from oracle import voxel_pool_ref as vp

pytestmark = pytest.mark.gpu
DEV = 'cuda'


def _random_geom(seed, B, N, D, H, W, vn, column_coherent):
    """column_coherent: all rows of a (depth bin, column) share x, y (a level camera) and z varies."""
    g = torch.Generator().manual_seed(seed)
    X, Y, Z = vn
    shape = (B, N, D, 1, W) if column_coherent else (B, N, D, H, W)
    x = torch.randint(-2, X + 2, shape, generator=g).expand(B, N, D, H, W)
    y = torch.randint(-2, Y + 2, shape, generator=g).expand(B, N, D, H, W)
    z = torch.randint(-1, Z + 1, (B, N, D, H, W), generator=g)
    if column_coherent:                                    # make z mostly in range, with a dropped prefix
        z = torch.where(torch.arange(H).view(1, 1, 1, H, 1) >= torch.randint(0, H, (B, N, D, 1, W), generator=g), 0, -1)
    return torch.stack([x, y, z], -1).int().contiguous()


def _features(seed, B, N, D, H, W, C, vn):
    g = torch.Generator().manual_seed(seed)
    depth = torch.rand(B * N, D, H, W, generator=g).softmax(1)
    ctx = torch.rand(B * N, C, H, W, generator=g) - 0.5
    go = torch.rand(B, C, vn[1], vn[0], generator=g)
    return depth, ctx, go


def _assert_plan(plan, geom, vn):
    head, code, cs, ids = vp.run_plan_ref(geom, vn)
    assert plan.mode == 'runs'
    B = geom.shape[0]
    X, Y, Z = vn
    kept, lin, _ = vp.cell_index_ref(geom, vn)
    exp_cell = torch.where(kept, lin - torch.arange(B).view(B, 1) * X * Y, torch.tensor(-1)).int()
    assert torch.equal(plan.cell_of_point.cpu(), exp_cell)
    assert torch.equal(plan.cell_start.cpu().long(), cs)
    assert torch.equal(plan.sorted_ids.cpu().long(), ids)
    assert torch.equal(plan.run_code.cpu(), code)
    assert torch.equal(plan.sorted_cells.cpu().long(), lin.reshape(-1)[ids])
    assert plan.num_sorted == ids.numel()


def _assert_forward(out_nhwc, geom, depth, ctx, vn):
    B, N = geom.shape[0], geom.shape[1]
    feats = vp.materialise_features_ref(depth, ctx, B, N)
    ref64 = vp.voxel_pooling_ref(geom, feats, vn, acc_dtype=torch.float64)
    abs64 = vp.voxel_pooling_ref(geom, feats.abs(), vn, acc_dtype=torch.float64)
    out = out_nhwc.permute(0, 3, 1, 2).cpu()
    err = (out.double() - ref64).abs()
    assert bool((err <= 1e-5 * ref64.abs() + 1e-6 * abs64 + 1e-30).all()), float(err.max())
    assert bool((out[abs64 == 0] == 0).all())              # empty cells are exact zeros


CASES = [
    # B, N, D, H, W, C, vn, column_coherent
    (2, 2, 9, 16, 8, 80, (32, 16, 1), True),      # vectorised loads, one row block
    (2, 2, 9, 16, 8, 80, (32, 16, 1), False),     # every point its own run
    (1, 3, 33, 44, 12, 80, (64, 32, 2), True),    # three row blocks (16 + 16 + 12), two depth tiles
    (1, 1, 40, 21, 10, 64, (40, 13, 1), True),    # W % 4 != 0: scalar loads, ragged column tile
    (3, 1, 5, 7, 5, 32, (512, 64, 1), False),     # aiMotive grid, tiny frustum
    (10, 1, 6, 16, 4, 96, (32, 16, 1), True),     # more samples than one stage-A/B chunk (8)
    (1, 2, 4, 3, 4, 128, (512, 512, 1), False),   # 2^18 cells per sample
    (1, 1, 3, 4, 4, 32, (8, 8, 1), False),        # 64 cells
]


@pytest.mark.parametrize('case', CASES)
def test_run_plan_and_forward(case):
    B, N, D, H, W, C, vn, coherent = case
    geom = _random_geom(3, B, N, D, H, W, vn, coherent)
    depth, ctx, go = _features(4, B, N, D, H, W, C, vn)
    plan = build_plan(geom.cuda(), vn, frustum=(N, D, H, W))
    _assert_plan(plan, geom, vn)
    out = fused_forward(plan, depth.cuda(), ctx.cuda())
    _assert_forward(out, geom, depth, ctx, vn)
    assert torch.equal(out, fused_forward(plan, depth.cuda(), ctx.cuda()))      # bit-stable
    # the backward kernels accept a run plan unchanged (they read cell_of_point only)
    gd, gc = fused_backward(plan, go.cuda(), depth.cuda(), ctx.cuda())
    rd, rc = vp.voxel_pooling_fused_grads_ref(geom, depth, ctx, vn, go)
    assert torch.allclose(gd.double().cpu(), rd, rtol=1e-5, atol=1.2e-7 * C)
    assert torch.allclose(gc.double().cpu(), rc, rtol=1e-5, atol=1.2e-7 * D)


def test_run_plan_tiny_grid_big_cells_and_shape_check():
    # 4 cells and 2 400 points: every cell holds far more runs than the per-thread ordering handles
    # (the queued-cell kernel takes over); a frustum that does not match geom_xyz is refused
    vn = (2, 2, 1)
    g = torch.Generator().manual_seed(5)
    geom = torch.stack([torch.randint(0, 2, (1, 2, 30, 8, 5), generator=g), torch.randint(0, 2, (1, 2, 30, 8, 5), generator=g),
                        torch.randint(-1, 1, (1, 2, 30, 8, 5), generator=g)], -1).int().contiguous()
    depth, ctx, go = _features(6, 1, 2, 30, 8, 5, 32, vn)
    plan = build_plan(geom.cuda(), vn, frustum=(2, 30, 8, 5))
    _assert_plan(plan, geom, vn)
    cs = plan.cell_start.cpu()
    assert int((cs[1:] - cs[:-1]).max()) > 64
    _assert_forward(fused_forward(plan, depth.cuda(), ctx.cuda()), geom, depth, ctx, vn)
    with pytest.raises(AssertionError):
        build_plan(geom.cuda(), vn, frustum=(3, 30, 8, 5))


@pytest.mark.parametrize('cfg,B', [(CFG_2, 2), (sweep_grid_config(256), 1)])
def test_camera_rig_runs_match_points(cfg, B):
    geom, vn = synthetic.camera_rig(cfg, B, yaw_jitter_deg=5.0)
    vn = vn.tolist()
    depth, ctx, go = synthetic.camera_features(cfg, B)
    g, d, c = geom.cuda(), depth.cuda(), ctx.cuda()
    runs = build_plan(g, vn, frustum=tuple(geom.shape[1:5]))
    _assert_plan(runs, geom, vn)
    out_r = fused_forward(runs, d, c)
    _assert_forward(out_r, geom, depth, ctx, vn)
    out_p = fused_forward(build_plan(g, vn), d, c)                               # point plan, same op
    assert torch.allclose(out_r, out_p, rtol=1e-5, atol=1e-6)
    # the autograd op picks the run plan by itself for a 6-d geom_xyz
    d.requires_grad_(True)
    c.requires_grad_(True)
    out = voxel_pooling_fused(g, d, c, vn)
    assert torch.equal(out.permute(0, 2, 3, 1), out_r)
    out.backward(go.cuda())
    rd, rc = vp.voxel_pooling_fused_grads_ref(geom, depth, ctx, vn, go)
    assert torch.allclose(d.grad.double().cpu(), rd, rtol=1e-5, atol=1e-5)
    assert torch.allclose(c.grad.double().cpu(), rc, rtol=1e-5, atol=1e-5)


def test_full_size_aim_properties_on_run_plan():
    cfg, B = CFG_AIM, 1                                     # shipped shape: 2.88 M points / frame, H = 44
    geom, vn = synthetic.camera_rig(cfg, B, device=DEV)
    depth, ctx, go = synthetic.camera_features(cfg, B, device=DEV)
    plan = build_plan(geom, vn, frustum=tuple(geom.shape[1:5]))
    assert plan.mode == 'runs'
    out = fused_forward(plan, depth, ctx)
    assert torch.allclose(fused_forward(plan, depth, 2 * ctx), 2 * out, rtol=1e-6, atol=1e-7)   # linear
    kept = (plan.cell_of_point >= 0).view(B * cfg.num_cams, cfg.depth_bins, *cfg.feat_hw)
    mass = torch.einsum('ndhw,nchw->c', (depth * kept).double(), ctx.double())                  # total mass
    assert torch.allclose(out.double().sum(dim=(0, 1, 2)), mass, rtol=1e-6, atol=1e-6)
    assert torch.equal(out, fused_forward(plan, depth, ctx))                                     # bit-stable
    code = plan.run_code
    assert bool(((code >= 0) | (code == -2)).view_as(kept).eq(kept).all())
    assert int((code >= 0).sum()) == plan.num_sorted


def test_max_runs_hint_makes_the_chain_capturable():
    cfg, B = CFG_2, 2
    geom, vn = synthetic.camera_rig(cfg, B, device=DEV)
    vn = vn.tolist()
    depth, ctx, _ = synthetic.camera_features(cfg, B, device=DEV)
    fr = tuple(geom.shape[1:5])
    first = build_plan(geom, vn, frustum=fr)
    eager = fused_forward(first, depth, ctx).clone()
    n = first.num_sorted

    def chain():
        return fused_forward(build_plan(geom, vn, frustum=fr, max_runs=n), depth, ctx)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        chain()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        captured = chain()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(captured, eager)


def test_cold_forward_with_overlapped_fill_equals_plain_forward_and_is_capturable(monkeypatch):
    """fused_forward_cold with BEVPOOL_COLD_OVERLAP=1: output zero-filled on a side stream while the plan is built,
    forward writes occupied cells only -- bit-equal to the plain sequence, eagerly and inside a CUDA graph."""
    from mm_training_b200.ops.voxel_pooling import fused_forward_cold
    monkeypatch.setenv('BEVPOOL_COLD_OVERLAP', '1')
    cfg, B = CFG_2, 3
    geom, vn_t = synthetic.camera_rig(cfg, B, device=DEV, yaw_jitter_deg=5.0, seed=12)
    vn = tuple(int(v) for v in vn_t.tolist())
    depth, ctx, _ = synthetic.camera_features(cfg, B, device=DEV, seed=12)
    fr = tuple(geom.shape[1:5])
    ref_plan = build_plan(geom, vn, frustum=fr)
    ref = fused_forward(ref_plan, depth, ctx)
    n = ref_plan.num_sorted
    plan, out = fused_forward_cold(lambda: build_plan(geom, vn, frustum=fr, max_runs=n), B, vn, depth, ctx)
    assert torch.equal(out, ref) and plan.status() == 0
    cl = ctx.contiguous(memory_format=torch.channels_last)
    assert torch.equal(fused_forward_cold(lambda: build_plan(geom, vn, frustum=fr, max_runs=n), B, vn, depth, cl)[1], ref)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        fused_forward_cold(lambda: build_plan(geom, vn, frustum=fr, max_runs=n), B, vn, depth, ctx)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        _, captured = fused_forward_cold(lambda: build_plan(geom, vn, frustum=fr, max_runs=n), B, vn, depth, ctx)
    for _ in range(3):
        captured.fill_(float('nan'))
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(captured, ref)
    # the autograd op takes the same path when it builds the plan itself
    d, c = depth.clone().requires_grad_(True), ctx.clone().requires_grad_(True)
    o = voxel_pooling_fused(geom, d, c, vn)
    assert torch.equal(o.permute(0, 2, 3, 1), ref)


def test_bench_dump_outputs_are_the_timed_step_outputs(tmp_path):
    """bench.py --dump-outputs writes what the timed step returned: the captured outputs refilled by the last graph
    replay (or the last eager step), the forward permuted to (B, C, Y, X), on the seeded inputs of rank 0."""
    import importlib.util
    import json
    import os
    import subprocess
    import sys
    import numpy as np
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for mode in ('graph', 'eager'):
        cmd = [sys.executable, os.path.join(root, 'bench.py'), '--gpus', '1', '--batch', '2', '--steps', '3', '--warmup', '1',
               '--no-extras', '--dump-outputs', str(tmp_path / mode)] + (['--no-graph'] if mode == 'eager' else [])
        res = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
        assert res.returncode == 0, res.stderr[-2000:]
        line = json.loads(res.stdout.strip().splitlines()[-1])
        assert line['steps'] == 3 and line['config']['launch'] == ('cuda_graph_replay' if mode == 'graph' else 'eager')
    spec = importlib.util.spec_from_file_location('bench_mod', os.path.join(root, 'bench.py'))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    geom, vn = synthetic.camera_rig(CFG_2, 2, device=DEV, yaw_jitter_deg=5.0, seed=1)
    depth, ctx, go = synthetic.camera_features(CFG_2, 2, device=DEV, seed=1)
    d, c = depth.requires_grad_(True), ctx.requires_grad_(True)
    out = voxel_pooling_fused(geom, d, c, vn.tolist())                         # (B, C, Y, X)
    out.backward(go)
    bench.dump_outputs(str(tmp_path / 'expect'), {'bev_features': out, 'grad_depth': d.grad, 'grad_context': c.grad})
    for name, tol in (('bev_features', 1e-6), ('grad_depth', 1e-5), ('grad_context', 1e-5)):
        want = np.load(tmp_path / 'expect' / f'{name}.npy')
        graph, eager = (np.load(tmp_path / m / f'{name}.npy') for m in ('graph', 'eager'))
        assert graph.shape == want.shape and np.array_equal(graph, eager)
        assert np.allclose(graph, want, rtol=1e-5, atol=tol), name

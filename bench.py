#!/usr/bin/env python
"""Benchmark of the BEV-projection hot path (BASELINE.json metric: BEV pool fwd+bwd frames/s
and fraction of HBM peak).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One *step* = one pass of the camera pooling path over one batch of synthetic frames on each
GPU: plan build (cell index + stable sort) -> fused voxel-pool forward -> fused backward into
the depth and context gradients.  The workload is BASELINE.json configs[1] (CFG-2: aiMotive
4-cam rig, D=112, 16x44 feature map, C=80, fp32, BEV grid 512x64).  The path shards by sample:
every rank processes its own frames, there is no collective on the data path ("weak" scaling).

Prints ONE JSON line on rank 0.  See DESIGN.md section "Measurement" for the byte accounting.

``--dump-outputs DIR``: after the timed steps, rank 0 writes what its last step returned -- the pooled BEV features
(B, C, Y, X), the depth gradient and the context gradient -- as ``DIR/<name>.npy`` (float32).  The inputs are seeded,
so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from mm_training_b200 import synthetic                      # noqa: E402
from mm_training_b200.configs import CFG_2, CFG_AIM          # noqa: E402

METRIC = 'bev_pool_fwd_bwd_frames_per_s'
UNIT = 'frames/s'


# ------------------------------------------------------------------------------------------
def algorithmic_bytes(cfg, kept_per_frame: float, s: int = 4):
    """SURVEY.md section 8(d), row (B): compulsory traffic of the fused op per frame."""
    P = cfg.points_per_frame
    h, w = cfg.feat_hw
    S = cfg.num_cams * h * w
    C = cfg.output_channels
    x, y, _ = cfg.voxel_num
    G = x * y
    K = kept_per_frame
    fwd_kernel = s * K + 4 * K + 4 * G + s * C * S + s * C * G       # depth+ids of kept, CSR, ctx, out
    bwd_kernel = s * C * G + s * P + 4 * P + s * C * S + s * P + s * C * S
    step = 16 * P + 3 * s * P + 3 * s * C * S + 2 * s * C * G       # formula of section 8(d)
    return dict(fused_forward=fwd_kernel, fused_backward=bwd_kernel, step=step)


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (B200_PROFILING.md).  The timed region
    of this bench is tens of milliseconds, shorter than one `nvidia-smi -lms` period, so the sampler polls
    NVML directly from a thread (a few hundred microseconds per sample); nvidia-smi is the fallback."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
         'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')
    NVML_REASONS = {0x8: 'hw_slowdown', 0x40: 'hw_thermal_slowdown', 0x20: 'sw_thermal_slowdown', 0x4: 'sw_power_cap'}

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []
        self.samples, self.stop, self.thread, self.nvml, self.max_mhz = [], False, None, None, None

    def _poll(self, handle):
        import pynvml
        while not self.stop:
            try:
                mhz = pynvml.nvmlDeviceGetClockInfo(handle, pynvml.NVML_CLOCK_SM)
                reasons = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(handle)
                self.samples.append((mhz, reasons))
            except Exception:                                   # pragma: no cover
                break
            time.sleep(0.0005)

    def __enter__(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get('CUDA_VISIBLE_DEVICES')
            phys = int(vis.split(',')[self.index]) if vis and vis.split(',')[self.index].isdigit() else self.index
            handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(handle, pynvml.NVML_CLOCK_SM)
            self.nvml = pynvml
            self.thread = threading.Thread(target=self._poll, args=(handle,), daemon=True)
            self.thread.start()
            return self
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                                          '-lms', '100', '-i', str(self.index)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True)
            self.t.start()
        except OSError:
            self.proc = None
        return self

    def __exit__(self, *a):
        if self.thread is not None:
            self.stop = True
            self.thread.join(timeout=2)
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            self.t.join(timeout=2)

    def summary(self):
        if self.nvml is not None and self.samples:
            sm = [s[0] for s in self.samples]
            bits = 0
            for s in self.samples:
                bits |= s[1]
            reasons = sorted(n for b, n in self.NVML_REASONS.items() if bits & b)
            return {'sm_mhz': statistics.median(sm), 'sm_max_mhz': self.max_mhz, 'reasons': reasons,
                    'samples': len(sm), 'source': 'nvml, polled during the timed region'}
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for ln in self.lines:
            f = [x.strip() for x in ln.split(',')]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith('active'):
                    reasons.add(n)
        if not sm:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'samples': 0}
        return {'sm_mhz': statistics.median(sm), 'sm_max_mhz': max(mx), 'reasons': sorted(reasons),
                'samples': len(sm), 'source': 'nvidia-smi -lms 100'}


def time_cuda(fn, iters, warmup):
    """median / min ms of ``fn`` with CUDA events on the current stream."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return statistics.median(ts), min(ts)


DUMP_MAX_ELEMENTS = 1 << 22          # per array: the three float32 outputs of a step stay under 64 MB


def dump_outputs(out_dir: str, arrays: dict, seed: int = 0) -> None:
    """Writes every array as ``out_dir/<name>.npy`` in float32.  An array of more than DUMP_MAX_ELEMENTS elements is
    written as a 1-D sample of its flattened (row-major) elements: one position from each of DUMP_MAX_ELEMENTS equal
    slices, drawn with a fixed seed, hence the same positions in every run with the same shapes."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach().float()
        n, k = t.numel(), DUMP_MAX_ELEMENTS
        if n > k:
            gen = torch.Generator().manual_seed(seed)
            lo = torch.arange(k, dtype=torch.int64) * n // k
            width = torch.arange(1, k + 1, dtype=torch.int64) * n // k - lo
            idx = lo + (torch.rand(k, generator=gen, dtype=torch.float64) * width).long()
            t = t.reshape(-1)[idx.to(t.device)]
        np.save(os.path.join(out_dir, name + '.npy'), t.cpu().numpy())


# ------------------------------------------------------------------------------------------
def cpu_pipeline_fwd_bwd(geom, depth, ctx, go, vn):
    """CPU path = the oracle port: materialised outer product + index_add_ forward, autograd
    backward to depth/context (pure torch; this is the ONE place bench.py executes oracle/)."""
    from oracle import voxel_pool_ref as vp
    d = depth.detach().requires_grad_(True)
    c = ctx.detach().requires_grad_(True)
    B, N = geom.shape[0], geom.shape[1]
    X, Y, Z = vn
    C = c.shape[1]
    feats = vp.materialise_features_ref(d, c, B, N).reshape(-1, C)
    kept, lin, _ = vp.cell_index_ref(geom, vn)
    k = kept.reshape(-1)
    out = torch.zeros(B * Y * X, C).index_add(0, lin.reshape(-1)[k], feats[k])
    out = out.view(B, Y, X, C).permute(0, 3, 1, 2)
    out.backward(go)
    return out.detach(), d.grad, c.grad


def run_cpu_baseline(cfg, frames: int, iters: int):
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    geom, vn = synthetic.camera_rig(cfg, frames, yaw_jitter_deg=5.0)
    depth, ctx, go = synthetic.camera_features(cfg, frames)
    vn = vn.tolist()
    cpu_pipeline_fwd_bwd(geom, depth, ctx, go, vn)                      # warm-up
    ts = []
    for _ in range(iters):
        t = time.perf_counter()
        cpu_pipeline_fwd_bwd(geom, depth, ctx, go, vn)
        ts.append(time.perf_counter() - t)
    best = statistics.median(ts)
    return {'value': frames / best, 'unit': UNIT, 'cores': torch.get_num_threads(), 'kind': 'port',
            'sample': f'{frames} frames of {cfg.name} x {iters} iterations (median), pure-torch '
                      f'materialise + index_add_ forward + autograd backward', 'ms_per_frame': best / frames * 1e3}


def _graph_step_ms(step, iters=20, warmup=3, flush_l2=False):
    """Capture ``step`` as one CUDA graph and time its replay (median ms, CUDA events).  ``flush_l2``: a 256 MB fill runs
    before every timed replay, outside the events (a kernel replayed alone would otherwise find its previous launch's
    operands in the 126 MB L2, which it never does inside the step)."""
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        step()
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        keep = step()                                           # noqa: F841
    if not flush_l2:
        med, mn = time_cuda(g.replay, iters, warmup)
    else:
        scrub = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')
        for _ in range(warmup):
            g.replay()
        ts = []
        for _ in range(iters):
            scrub.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            g.replay()
            b.record()
            b.synchronize()
            ts.append(a.elapsed_time(b))
        med, mn = statistics.median(ts), min(ts)
        del scrub
    del g, keep
    return med, mn


def run_sweep(dev, peak_gbs, seed=7, full=False, ref_arms=False):
    """BASELINE.json configs[4]: batch x grid sweep of the same step (cold plan from geom_xyz + fused forward +
    backward, NCHW layouts), one CUDA graph per point, this rank's GPU.  Default: a miniature (batch 1/8/64 on the
    aiMotive grid, the three square grids at batch 8, the shipped CFG-AIM shape at batch 4); ``full``: batch
    1..64 x {128,256,512}^2.  ``ref_arms``: the reference's CUDA pipeline (oracle/_ref) on the same inputs beside
    every point, and the CPU port on a bounded sample (batch <= 2)."""
    from mm_training_b200.configs import sweep_grid_config
    from mm_training_b200.ops.voxel_pooling import build_plan, fused_backward, fused_forward_cold
    if full:
        points = [(sweep_grid_config(g), b) for g in (128, 256, 512) for b in (1, 2, 4, 8, 16, 32, 64)]
    else:
        points = [(CFG_2, 1), (CFG_2, 8), (CFG_2, 64)] + [(sweep_grid_config(g), 8) for g in (128, 256, 512)] + [(CFG_AIM, 4)]
    rows_out = []
    for cfg, B in points:
        geom, vn_t = synthetic.camera_rig(cfg, B, device=dev, yaw_jitter_deg=5.0, seed=seed)
        vn = tuple(int(v) for v in vn_t.tolist())
        depth, ctx, go = synthetic.camera_features(cfg, B, device=dev, seed=seed)
        fr = tuple(geom.shape[1:5])
        n = build_plan(geom, vn, frustum=fr).num_sorted

        def step():
            plan, out = fused_forward_cold(lambda: build_plan(geom, vn, frustum=fr, max_runs=n), B, vn, depth, ctx)
            return out, fused_backward(plan, go, depth, ctx)
        med, _ = _graph_step_ms(step)
        kept = int((build_plan(geom, vn).cell_of_point >= 0).sum().item()) / B
        gbs = algorithmic_bytes(cfg, kept)['step'] * B / (med * 1e-3) / 1e9
        row = {'workload': cfg.name, 'frames_per_step': B, 'ms_per_step': med,
               'frames_per_s': B / (med * 1e-3), 'frac_of_hbm_peak': gbs / peak_gbs}
        if ref_arms:
            from oracle import ref_cuda_op
            if ref_cuda_op.available():
                d_r, c_r = depth.detach().requires_grad_(True), ctx.detach().requires_grad_(True)

                def ref_step():
                    d_r.grad = None
                    c_r.grad = None
                    ref_cuda_op.ref_pipeline(geom, d_r, c_r, vn).backward(go)
                rmed, _ = time_cuda(ref_step, 3, 1)
                row['ref_cuda_frames_per_s'] = B / (rmed * 1e-3)
                del d_r, c_r
            if B <= 2:
                row['cpu_port_frames_per_s'] = run_cpu_baseline(cfg, B, 1)['value']
        rows_out.append(row)
        del geom, depth, ctx, go
        torch.cuda.empty_cache()
    return rows_out


def run_dropin_op(dev, peak_gbs, cfg=CFG_2, B=8, seed=5):
    """Row (A) of SURVEY.md 8(d): the drop-in op ``voxel_pooling(geom_xyz, input_features, voxel_num)`` on
    PRE-MATERIALISED features (B, N, D, H, W, C), forward + autograd backward w.r.t. the features, NCHW-contiguous
    incoming gradient (what lss_fpn.py:466 hands back) -- beside the reference's own CUDA op on the same tensors."""
    from mm_training_b200.ops.voxel_pooling import voxel_pooling
    from oracle import ref_cuda_op
    geom, vn_t = synthetic.camera_rig(cfg, B, device=dev, yaw_jitter_deg=5.0, seed=seed)
    vn = tuple(int(v) for v in vn_t.tolist())
    depth, ctx, go = synthetic.camera_features(cfg, B, device=dev, seed=seed)
    N = cfg.num_cams
    f = depth.unsqueeze(1) * ctx.unsqueeze(2)                                        # lss_fpn.py:441-460
    feats = f.reshape(B, N, *f.shape[1:]).permute(0, 1, 3, 4, 5, 2).contiguous().requires_grad_(True)
    del f

    def ours():
        feats.grad = None
        voxel_pooling(geom, feats, vn).backward(go)
    ours()
    torch.cuda.synchronize()
    from mm_training_b200.ops.voxel_pooling import build_plan
    kept = int((build_plan(geom, vn).cell_of_point >= 0).sum().item()) / B
    P, C = cfg.points_per_frame, cfg.output_channels
    G = vn[0] * vn[1]
    bytes_frame = 12 * P + 4 * C * kept + 4 * C * G + 4 * C * G + 4 * P + 4 * C * P
    med, mn = time_cuda(ours, 10, 3)
    res = {'what': 'drop-in op voxel_pooling(geom_xyz, input_features, voxel_num).backward(grad): cold point plan + '
                   'forward + backward per call, through the autograd Function (eager), pre-materialised features',
           'workload': cfg.name, 'frames_per_step': B, 'ms_per_step': med, 'frames_per_s': B / (med * 1e-3),
           'algorithmic_bytes_per_frame': bytes_frame,
           'roofline': {'bound': 'hbm', 'achieved': bytes_frame * B / (med * 1e-3) / 1e9, 'peak': peak_gbs, 'unit': 'GB/s',
                        'frac': bytes_frame * B / (med * 1e-3) / 1e9 / peak_gbs}}
    if ref_cuda_op.available():
        def ref():
            feats.grad = None
            ref_cuda_op.ref_voxel_pooling(geom, feats, vn).backward(go)
        rmed, _ = time_cuda(ref, 5, 2)
        res['ref_cuda_op'] = {'what': 'the reference op (its CUDA kernel + voxel_pooling.py autograd wrapper) on the same tensors',
                              'ms_per_step': rmed, 'frames_per_s': B / (rmed * 1e-3)}
        res['speedup_vs_ref_cuda_op'] = rmed / med
    return res


def run_half_precision_side(dev, cfg=CFG_2, B=8, seed=5):
    """fp16 / bf16 inputs (north star: features and gradients within 1e-2): the fused op on half-precision depth, context and
    incoming gradient, cold POINT plan + forward + backward (the run-plan fast path is fp32 only; the generic kernels
    accumulate in fp32), CUDA events, beside the fp32 step on the same frames and the worst relative error against it."""
    from mm_training_b200.ops.voxel_pooling import build_plan, fused_backward, fused_forward
    geom, vn_t = synthetic.camera_rig(cfg, B, device=dev, yaw_jitter_deg=5.0, seed=seed)
    vn = tuple(int(v) for v in vn_t.tolist())
    depth, ctx, go = synthetic.camera_features(cfg, B, device=dev, seed=seed)
    fr = tuple(geom.shape[1:5])

    def step32():
        plan = build_plan(geom, vn, frustum=fr)
        return fused_forward(plan, depth, ctx), fused_backward(plan, go, depth, ctx)
    out32, (gd32, gc32) = step32()
    res = {'workload': cfg.name, 'frames_per_step': B, 'fp32_run_plan_ms_per_step': time_cuda(step32, 10, 3)[0],
           'what': 'cold plan + fused forward + fused backward through the functional API, eager'}
    for name, dt in (('bf16', torch.bfloat16), ('fp16', torch.float16)):
        d16, c16, g16 = depth.to(dt), ctx.to(dt), go.to(dt)

        def step16():
            plan = build_plan(geom, vn)
            return fused_forward(plan, d16, c16), fused_backward(plan, g16, d16, c16)
        out16, (gd16, gc16) = step16()
        rel = lambda a, b: float((a.float() - b).abs().max() / b.abs().max())
        res[name] = {'ms_per_step': time_cuda(step16, 10, 3)[0],
                     'max_err_over_max_abs': {'out': rel(out16, out32), 'grad_depth': rel(gd16, gd32), 'grad_context': rel(gc16, gc32)}}
        res[name]['frames_per_s'] = B / (res[name]['ms_per_step'] * 1e-3)
        del d16, c16, g16, out16, gd16, gc16
    return res


def run_depth_labels_side(dev, peak_gbs, B=4):
    """Side measurement (SURVEY.md 8f, N3): depth labels for the depth loss at the shipped shape (704 x 1280 images, 2
    cameras, 200 k LiDAR points per frame, 16 x 16 min-pool, 409 bins): the native two-launch path beside the
    reference's python loop of torch ops (exps/mm_training_aim.py:115-215, restated in oracle/) on the same GPU and on
    the host cores (one frame)."""
    from mm_training_b200.ops.depth_labels import DepthLabelGenerator
    from oracle import depth_labels_ref as dl
    cfg = CFG_AIM
    hw, D = cfg.final_dim, cfg.depth_bins
    case = dl.synthetic_case(batch=B, sweeps=1, cams=cfg.num_cams, num_points=200_000, image_hw=hw, seed=21)
    clouds, ext, intr, bda = case
    g_clouds, g_ext, g_intr, g_bda = [c.to(dev) for c in clouds], ext.to(dev), intr.to(dev), bda.to(dev)
    gen = DepthLabelGenerator(hw, cfg.downsample_factor, cfg.d_bound, D)
    labels, bins = gen(g_clouds, g_ext, g_intr, g_bda, return_bins=True, bda_inv=torch.linalg.inv(bda[:, :3, :3].float()))
    _, ref_bins = dl.depth_labels_exact([clouds[0]], ext[:1], intr[:1], bda[:1], hw, cfg.downsample_factor, cfg.d_bound, D)
    n0 = ref_bins.numel()
    assert torch.equal(bins[:n0].cpu().long(), ref_bins), 'depth labels differ from the oracle'
    med, mn = time_cuda(lambda: gen(g_clouds, g_ext, g_intr, g_bda), 20, 3)
    ref_gpu, _ = time_cuda(lambda: dl.depth_labels_torch(g_clouds, g_ext, g_intr, g_bda, hw, cfg.downsample_factor, cfg.d_bound, D), 3, 1)
    t0 = time.perf_counter()
    dl.depth_labels_torch([clouds[0]], ext[:1], intr[:1], bda[:1], hw, cfg.downsample_factor, cfg.d_bound, D)
    cpu_s = time.perf_counter() - t0
    cells = bins.numel()
    # compulsory bytes: every point read once per image it is projected into (12 B) + the one-hot rows written once
    alg = sum(int(c.shape[0]) for c in clouds) * 12 * cfg.num_cams + cells * D * 4
    return {'workload': f'depth_labels_{hw[0]}x{hw[1]}_2cam_200kpts_D{D}', 'frames_per_step': B, 'ms_per_step': med,
            'frames_per_s': B / (med * 1e-3), 'algorithmic_bytes_per_step': alg,
            'roofline': {'bound': 'hbm', 'achieved': alg / (med * 1e-3) / 1e9, 'peak': peak_gbs, 'unit': 'GB/s',
                         'frac': alg / (med * 1e-3) / 1e9 / peak_gbs,
                         'note': 'the full-resolution winner map (8 B/pixel, read + cleared) is scratch traffic, not counted'},
            'reference_torch_loop_same_gpu': {'ms_per_step': ref_gpu, 'frames_per_s': B / (ref_gpu * 1e-3)},
            'speedup_vs_reference_torch_loop': ref_gpu / med,
            'cpu_port': {'frames_per_s': 1.0 / cpu_s, 'cores': torch.get_num_threads(), 'kind': 'port', 'sample': '1 frame'},
            'parity': 'bin indices bit-exact vs oracle/depth_labels_ref.py::depth_labels_exact (checked in this run)'}


def run_lidar_side(dev, peak_gbs, sweeps: int = 32):
    """Side measurement (not the headline metric; BASELINE.json configs[2]): ``sweeps`` synthetic 200k-point long-range
    sweeps (SURVEY.md 8d) through hard voxelization + fused HardSimpleVFE mean + pillar scatter.  Three ways:
    the mmdet3d-style call (exact-size tensors: one D2H sync for the voxel counts), the same work with padded
    outputs (no sync) eagerly, and that replayed as one CUDA graph (the headline of this block); plus the serial
    CPU restatement of mmcv's hard_voxelize on one sweep (mmcv's CPU kernel is single-threaded)."""
    from mm_training_b200.configs import CFG_3
    from mm_training_b200.ops.voxelize import Voxelization, pillar_scatter, voxelize
    v = CFG_3
    clouds_np = [synthetic.lidar_sweep(v.points_per_sweep, v.num_point_features, seed=2 + i) for i in range(sweeps)]
    clouds = [torch.from_numpy(a).to(dev) for a in clouds_np]
    layer = Voxelization(list(v.voxel_size), list(v.point_cloud_range), v.max_num_points, v.max_voxels).eval()
    gx, gy, gz = (int(g) for g in layer.grid_size.tolist())

    def run_exact():                                      # mmdet3d semantics: exact-size tensors (one D2H sync)
        voxels, num_points, coors, mean = voxelize(clouds, layer, mean_features=v.vfe_features)
        canvas = pillar_scatter(mean, coors, sweeps, (gz, gy, gx), unique_coors=True)
        return voxels, canvas

    def run_padded():                                     # no sync: padded outputs + fused scatter
        return voxelize(clouds, layer, mean_features=v.vfe_features, padded=True, scatter=True)
    voxels, canvas = run_exact()
    pad = run_padded()
    torch.cuda.synchronize()
    assert torch.equal(pad[4], canvas) and torch.equal(pad[0][:voxels.shape[0]], voxels)
    M = voxels.shape[0] / sweeps
    exact_med, _ = time_cuda(run_exact, 10, 3)
    eager_med, _ = time_cuda(run_padded, 10, 3)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        run_padded()
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        keep = run_padded()                               # noqa: F841
    med, mn = time_cuda(g.replay, 20, 3)
    F, T = v.num_point_features, v.max_num_points
    vox_bytes = 4 * F * v.points_per_sweep + 4 * F * T * M + 20 * M
    sc_bytes = 4 * v.vfe_features * M + 16 * M + 4 * v.vfe_features * gz * gy * gx
    gbs = (vox_bytes + sc_bytes) * sweeps / (med * 1e-3) / 1e9
    from oracle import voxelize_ref as vr
    t0 = time.perf_counter()
    vr.hard_voxelize_c(clouds_np[0], list(v.voxel_size), list(v.point_cloud_range), T, v.max_voxels)
    cpu_s = time.perf_counter() - t0
    del g, keep
    return {'workload': v.name, 'sweeps_per_step': sweeps, 'ms_per_step': med, 'sweeps_per_s': sweeps / (med * 1e-3),
            'points_per_s': sweeps * v.points_per_sweep / (med * 1e-3), 'voxels_per_sweep': M,
            'algorithmic_bytes_per_sweep': vox_bytes + sc_bytes, 'achieved_gbs': gbs, 'frac_of_hbm_peak': gbs / peak_gbs,
            'roofline': {'bound': 'hbm', 'achieved': gbs, 'peak': peak_gbs, 'unit': 'GB/s', 'frac': gbs / peak_gbs,
                         'bytes': 'SURVEY.md 8(d): 4*F*Np + 4*F*T*M + 20*M (voxelizer) + 4*Cv*M + 16*M + 4*Cv*gz*gy*gx (scatter) per sweep'},
            'what': 'voxelize(list of sweeps, mean_features=5, padded=True, scatter=True): hard voxelization + HardSimpleVFE mean '
                    '+ pillar scatter to (B, 5, 256, 2048) in one native call, no host sync, CUDA graph replay',
            'eager_no_sync_ms': eager_med, 'mmdet3d_style_exact_size_ms': exact_med,
            'parity': 'bit-exact vs oracle/hard_voxelize_ref.c (our restatement of mmcv 1.7.0; parity unpinned by the reference)',
            'cpu_hard_voxelize': {'sweeps_per_s': 1.0 / cpu_s, 'cores': 1, 'kind': 'port',
                                  'sample': '1 sweep, serial C restatement of mmcv hard_voxelize (oracle/)'}}


# ------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=50)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='native', choices=['native', 'reference'])
    ap.add_argument('--batch', type=int, default=32, help='frames per GPU per step')
    ap.add_argument('--workload', default='cfg2', choices=['cfg2', 'aim', 'train'],
                    help="'train': BASELINE.json configs[3], the fusion training step (bench_train.py), bf16 autocast + DDP")
    ap.add_argument('--train-cfg', default='aim', choices=['aim', 'cfg2'], help='camera shape of --workload train')
    ap.add_argument('--e2e-chunk', type=int, default=4, help='frames per chunk of the host-buffer pipeline')
    ap.add_argument('--plan', default='runs', choices=['runs', 'points'],
                    help="what the plan sorts: 'runs' (vertical point runs, two-stage forward) or 'points'")
    ap.add_argument('--geometry', default='auto', choices=['auto', 'rig', 'geom'],
                    help="where the plan's cell indices come from: 'rig' = built on the device from sensor2ego @ inv(intrin) "
                         "(no geom_xyz tensor; needs an accumulation order proven bit-exact on this device), 'geom' = from the "
                         "reference's int32 geom_xyz tensor, 'auto' = rig when proven")
    ap.add_argument('--no-graph', action='store_true', help='launch eagerly instead of replaying a CUDA graph')
    ap.add_argument('--no-extras', action='store_true', help='skip e2e / cpu / reference-CUDA side measurements')
    ap.add_argument('--sweep', default='mini', choices=['mini', 'full'],
                    help="'full': BASELINE.json configs[4] batch 1..64 x {128,256,512}^2 with both reference arms per point")
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write the outputs of the last timed step to DIR/<name>.npy (float32; a fixed seeded sample of '
                         f'arrays above {DUMP_MAX_ELEMENTS} elements).  Only the native camera pooling step '
                         '(--impl native with --workload cfg2 or aim) dumps: it is the path two builds of the kernels '
                         'are compared on; the CPU port and the training harness are refused')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and (args.impl != 'native' or args.workload == 'train'):
        ap.error('--dump-outputs covers the native camera pooling step only (--impl native, --workload cfg2 or aim)')
    args.batch_given = any(a == '--batch' or a.startswith('--batch=') for a in sys.argv[1:])
    cfg = CFG_AIM if args.workload == 'aim' else CFG_2
    if args.workload == 'aim' and not args.batch_given:
        args.batch = 4

    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local_rank = int(os.environ.get('LOCAL_RANK', 0))

    workload = dict(workload=cfg.name, frames_per_gpu_per_step=args.batch, op='plan_build+fused_forward+fused_backward',
                    points_per_frame=cfg.points_per_frame, channels=cfg.output_channels,
                    voxel_num=list(cfg.voxel_num), sharding='by sample, no collective',
                    cache='inputs+outputs per step exceed the 126 MB L2 (no flush needed)')

    if args.impl == 'reference':
        # CPU arm: the reference's path on the host cores (pure-torch scatter-add port), rank 0 only
        if rank != 0:
            return
        frames = 2
        res = run_cpu_baseline(cfg, frames, args.steps)
        v = res['value']
        line = {'metric': METRIC, 'value': v, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps,
                'warmup': 1, 'ms_per_step': frames / v * 1e3, 'higher_is_better': True, 'scaling': 'weak',
                'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic', 'impl': 'reference',
                'config': dict(workload, frames_per_gpu_per_step=frames, device='cpu'),
                'cpu_baseline': res,
                'e2e': {'value': v, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
                'gpu_launches': 0}
        print(json.dumps(line), flush=True)
        return

    # ---------------------------------------------------------------- native arm
    import torch.distributed as dist
    from mm_training_b200 import _lib
    from mm_training_b200.ops.voxel_pooling import (build_plan, context_rows_nhwc, fused_backward,
                                                    fused_forward, voxel_pooling_fused)
    assert torch.cuda.is_available(), 'bench.py needs a CUDA device (no CPU fallback)'
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    # stdout must carry exactly ONE JSON line: libraries (NCCL prints its version banner with printf) get
    # stderr as their stdout; the result line is written to the saved descriptor at the end
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    _lib.lib()
    if args.workload == 'train':
        import bench_train
        bench_train.run_train(args, rank, world, local_rank, json_fd)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    B = args.batch
    geom, vn_t = synthetic.camera_rig(cfg, B, device=dev, yaw_jitter_deg=5.0, seed=1 + rank)
    vn = tuple(int(v) for v in vn_t.tolist())
    depth, ctx, go = synthetic.camera_features(cfg, B, device=dev, seed=1 + rank)

    frustum = tuple(geom.shape[1:5]) if args.plan == 'runs' else None
    probe = build_plan(geom, vn, frustum=frustum)      # eager, once: the run count sizes the scratch rows
    max_runs = probe.num_sorted if probe.mode == 'runs' else None
    plan_mode = probe.mode

    # geometry source of the plan (SURVEY.md 8f, N1): the rig path replaces lss_fpn.py:328-361,461-462 as well --
    # the (B, N, D, H, W, 3) tensors are never made; combine = sensor2ego @ inverse(intrin) (B*N 4x4 matrices) stays in
    # torch, outside the captured step (torch.inverse is not capturable), everything per point is in the key kernel
    from mm_training_b200.ops.voxel_pooling import LiftSplatGeometry, PoolingPlan, rig_variant
    variant, rig_exact, lsg, combine = None, None, None, None
    if args.geometry != 'geom' and plan_mode == 'runs':
        variant = rig_variant(dev)
        if variant is None and args.geometry == 'rig':
            raise SystemExit('no rig variant reproduces torch on this device')
    if variant is not None:
        lsg = LiftSplatGeometry.from_config(cfg, dev)
        s2e, intrin = synthetic.camera_rig_mats(cfg, B, device=dev, yaw_jitter_deg=5.0, seed=1 + rank)
        combine = lsg.combine(s2e, intrin)
        rp = PoolingPlan.from_rig(lsg, combine, variant)
        rig_exact = bool(torch.equal(rp.cell_of_point, probe.cell_of_point) and torch.equal(rp.sorted_ids, probe.sorted_ids)
                         and torch.equal(rp.run_code, probe.run_code))
        assert rig_exact, 'rig plan differs from the geom_xyz plan'
        del rp
    del probe

    def make_plan():
        # cold plan every step: cell index + sort are redone (no sync: max_runs is known)
        if variant is not None:
            return PoolingPlan.from_rig(lsg, combine, variant, max_runs)
        return build_plan(geom, vn, frustum=frustum, max_runs=max_runs)

    from mm_training_b200.ops.voxel_pooling import fused_forward_cold

    def step():
        # cold call: plan build, then forward (BEVPOOL_COLD_OVERLAP=1: zero fill on a side stream behind the plan build)
        plan, out = fused_forward_cold(make_plan, B, vn, depth, ctx)      # NCHW context read through a TMA tensor map
        gd, gc = fused_backward(plan, go, depth, ctx)  # NCHW incoming gradient; grad_context written NCHW like ctx
        return plan, out, gd, gc

    plan, out, gd, gc = step()
    torch.cuda.synchronize()
    kept_per_frame = int((plan.cell_of_point >= 0).sum().item()) / B
    bytes_ = algorithmic_bytes(cfg, kept_per_frame)

    l0 = _lib.launch_count()
    step()
    launches_per_step = _lib.launch_count() - l0

    use_graph = not args.no_graph
    graph = None
    if use_graph:
        try:
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                step()
            torch.cuda.current_stream().wait_stream(s)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                keep = step()                                   # noqa: F841  (outputs stay alive in the pool)
            run = graph.replay
        except Exception as e:                                  # pragma: no cover
            print(f'[bench] CUDA graph capture failed ({e}); launching eagerly', file=sys.stderr)
            graph, run = None, step
    else:
        run = step

    for _ in range(max(3, args.warmup)):
        run()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    last = None
    with ClockSampler(local_rank) as clocks:
        ev0.record()
        for _ in range(args.steps):
            last = run()
        ev1.record()
        torch.cuda.synchronize()
    if args.dump_outputs and rank == 0:
        _, out_last, gd_last, gc_last = keep if graph is not None else last   # a replay refills the captured outputs
        dump_outputs(args.dump_outputs, {'bev_features': out_last.permute(0, 3, 1, 2), 'grad_depth': gd_last,
                                         'grad_context': gc_last})
        del out_last, gd_last, gc_last
    if world > 1:
        dist.barrier()
    from mm_training_b200.sharding import aggregate_throughput
    value, total_ms, total_frames = aggregate_throughput(B * args.steps, ev0.elapsed_time(ev1), device=dev)
    ms_per_step = total_ms / args.steps

    # ---- e2e on EVERY rank (host pinned buffers in/out, PCIe inside the timed region), max over ranks
    e2e = None
    if not args.no_extras:
        from mm_training_b200.ops.voxel_pooling.host_pipeline import HostPoolingPipeline
        # geometry as the data loader holds it: the rig matrices (4 KB/frame) when the on-device index path is
        # proven on this GPU, else the reference's int32 geom_xyz tensor (3.8 MB/frame)
        e2e_rig = variant is not None
        pin = lambda t: t.cpu().contiguous().pin_memory()
        h_depth, h_ctx, h_go = pin(depth), pin(ctx), pin(go)
        if e2e_rig:
            h_s2e, h_k, h_geom = pin(s2e), pin(intrin), None
        else:
            h_s2e, h_k, h_geom = None, None, pin(geom)
        X, Y, _ = vn
        h_out = torch.empty(B, cfg.output_channels, Y, X).pin_memory()
        h_gd, h_gc = torch.empty_like(h_depth).pin_memory(), torch.empty_like(h_ctx).pin_memory()
        pipe = HostPoolingPipeline(cfg.num_cams, geom.shape, depth.shape, ctx.shape, vn,
                                   chunk_frames=max(1, min(args.e2e_chunk, B)), device=dev, rig=lsg if e2e_rig else None)
        e2e_iters = max(5, min(args.steps, 20))
        run_e2e = lambda: pipe.run(h_geom, h_depth, h_ctx, h_go, h_out, h_gd, h_gc, h_sensor2ego=h_s2e, h_intrin=h_k)
        for _ in range(3):
            run_e2e()                                   # returns with the results in host memory, plans validated
        assert torch.allclose(h_out.to(dev), out.permute(0, 3, 1, 2), rtol=1e-5, atol=1e-6)   # same results as the device path
        if world > 1:
            dist.barrier()
        ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ea.record()
        for _ in range(e2e_iters):
            run_e2e()
        eb.record()
        torch.cuda.synchronize()
        e2e_value, e2e_total_ms, _ = aggregate_throughput(B * e2e_iters, ea.elapsed_time(eb), device=dev)
        h_in = [t for t in (h_geom, h_s2e, h_k, h_depth, h_ctx, h_go) if t is not None]
        h2d = sum(t.numel() * t.element_size() for t in h_in)
        d2h = sum(t.numel() * t.element_size() for t in (h_out, h_gd, h_gc)) + 4 * ((B + pipe.chunk - 1) // pipe.chunk)
        e2e = {'value': e2e_value, 'unit': UNIT, 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
               'ms_per_step': e2e_total_ms / e2e_iters, 'steps': e2e_iters,
               'api': 'HostPoolingPipeline.run: voxel_pooling_fused(...).backward(...) on pinned host tensors, '
                      f'{pipe.chunk}-frame chunks on 3 streams (H2D | run plan + fwd + bwd | D2H), results in host memory and '
                      'plan status checked before every call returns; bytes are per GPU',
               'geometry_input': 'sensor2ego + intrin matrices (plan built on the device)' if e2e_rig else 'int32 geom_xyz tensor',
               'scratch_reruns': pipe.reruns,
               'pcie_gbs_per_gpu': (h2d + d2h) / (e2e_total_ms / e2e_iters * 1e-3) / 1e9,
               'h2d_gbs_per_gpu': h2d / (e2e_total_ms / e2e_iters * 1e-3) / 1e9,
               'd2h_gbs_per_gpu': d2h / (e2e_total_ms / e2e_iters * 1e-3) / 1e9}
        del pipe, h_geom, h_s2e, h_k, h_depth, h_ctx, h_go, h_out, h_gd, h_gc

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except OSError:
        pass
    peak_gbs = float(peaks.get('hbm_gbs', 6650.0))
    peak_src = 'measured (MEASURED_PEAKS.json)' if peaks else 'fallback (B200_PROFILING.md)'

    # ---- per-kernel timing (CUDA events on the launching stream), same inputs, warm
    stages = {}
    stages['plan_build'] = time_cuda(make_plan, 20, 3)
    stages['plan_build_from_geom_xyz'] = time_cuda(lambda: build_plan(geom, vn, frustum=frustum, max_runs=max_runs), 20, 3)
    stages['fused_forward(+ctx transpose)'] = time_cuda(lambda: fused_forward(plan, depth, ctx), 20, 3)
    stages['fused_backward(+grad transpose)'] = time_cuda(lambda: fused_backward(plan, go, depth, ctx), 20, 3)
    ctx_nhwc = ctx.permute(0, 2, 3, 1).contiguous().permute(0, 3, 1, 2)
    go_nhwc = go.permute(0, 2, 3, 1).contiguous().permute(0, 3, 1, 2)
    # the fused kernels alone, launched the way the timed step launches them (one CUDA graph each: no host launch gaps
    # between stage A, stage B and the fix-up); eager events if the capture fails
    kernel_timing = ('CUDA events around the replay of a CUDA graph holding the kernel(s) alone (launched as in the timed step), '
                     'L2 flushed by a 256 MB fill before every replay')
    try:
        k_fwd = _graph_step_ms(lambda: fused_forward(plan, depth, ctx_nhwc), flush_l2=True)
        k_bwd = _graph_step_ms(lambda: fused_backward(plan, go_nhwc, depth, ctx_nhwc), flush_l2=True)
    except Exception as e:                                      # pragma: no cover
        print(f'[bench] per-kernel graph capture failed ({e}); eager timing', file=sys.stderr)
        kernel_timing = 'CUDA events around eager launches'
        k_fwd = time_cuda(lambda: fused_forward(plan, depth, ctx_nhwc), 20, 3)
        k_bwd = time_cuda(lambda: fused_backward(plan, go_nhwc, depth, ctx_nhwc), 20, 3)
    stages['fused_forward_kernel'] = k_fwd
    stages['fused_backward_kernel'] = k_bwd
    # ---- the same step when the caller keeps context and gradient channels_last (zero-copy layouts: no
    # context / context-gradient transposes, no gradient-row pass); reported beside the headline, not as it
    def step_cl():
        p, o = fused_forward_cold(make_plan, B, vn, depth, ctx_nhwc)
        return o, fused_backward(p, go_nhwc, depth, ctx_nhwc)
    cl_ms = None
    try:
        s2 = torch.cuda.Stream()
        s2.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s2):
            step_cl()
        torch.cuda.current_stream().wait_stream(s2)
        g2 = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g2):
            keep2 = step_cl()                                   # noqa: F841
        cl_ms = time_cuda(g2.replay, 20, 3)
    except Exception as e:                                      # pragma: no cover
        print(f'[bench] channels_last side measurement failed ({e})', file=sys.stderr)
    # ---- the public autograd op, eager, no hints (what INTEGRATION.md section 1 shows a user calling)
    def op_step_geom():
        d_, c_ = depth.detach().requires_grad_(True), ctx.detach().requires_grad_(True)
        voxel_pooling_fused(geom, d_, c_, vn).backward(go)
    stages['autograd_op_eager: voxel_pooling_fused(geom_xyz, depth, context, voxel_num).backward(g)'] = time_cuda(op_step_geom, 20, 3)
    if variant is not None:
        from mm_training_b200.ops.voxel_pooling import voxel_pooling_rig

        def op_step_rig():
            d_, c_ = depth.detach().requires_grad_(True), ctx.detach().requires_grad_(True)
            voxel_pooling_rig(lsg, s2e, intrin, d_, c_).backward(go)
        stages['autograd_op_eager: voxel_pooling_rig(lsg, sensor2ego, intrin, depth, context).backward(g)'] = time_cuda(op_step_rig, 20, 3)
    # ---- sustained: the headline graph replayed for >= 1 s (clocks / power settle), this rank
    sustained = None
    if graph is not None and not args.no_extras:
        n_sus = int(1200.0 / max(ms_per_step, 1e-3)) + 1
        with ClockSampler(local_rank) as clk_s:
            sa, sb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            sa.record()
            for _ in range(n_sus):
                run()
            sb.record()
            torch.cuda.synchronize()
        sus_ms = sa.elapsed_time(sb)
        sustained = {'steps': n_sus, 'seconds': sus_ms * 1e-3, 'ms_per_step': sus_ms / n_sus,
                     'frames_per_s': B * n_sus / (sus_ms * 1e-3), 'clocks': clk_s.summary()}
    dom_name, dom = ('fused_backward', k_bwd) if k_bwd[0] >= k_fwd[0] else ('fused_forward', k_fwd)
    achieved = bytes_[dom_name] * B / (dom[0] * 1e-3) / 1e9
    traffic = None                      # dram__bytes_read+write per launch of that kernel, from the committed ncu capture
    try:
        tj = json.load(open(os.path.join(ROOT, 'profiles', 'ncu_traffic.json')))
        ent = tj.get(dom_name + '_kernel')
        if ent and ent.get('frames_per_launch') == B and ent.get('workload') == cfg.name:
            traffic = ent['dram_bytes_per_launch']
    except (OSError, ValueError):
        pass
    roofline = {'bound': 'hbm', 'kernel': dom_name + '_kernel', 'achieved': achieved, 'peak': peak_gbs,
                'unit': 'GB/s', 'frac': achieved / peak_gbs, 'peak_source': peak_src, 'traffic': traffic,
                'algorithmic_bytes_per_frame': bytes_[dom_name], 'kernel_ms': dom[0],
                'frac_of_nominal_8TBps': achieved / 8000.0, 'timing': kernel_timing}
    # both fused kernels against the same peak (the dominant one above is whichever is slower in this run)
    roofline['kernels'] = []
    for nm, kt in (('fused_forward', k_fwd), ('fused_backward', k_bwd)):
        gbs = bytes_[nm] * B / (kt[0] * 1e-3) / 1e9
        ent = None
        try:
            ent = json.load(open(os.path.join(ROOT, 'profiles', 'ncu_traffic.json'))).get(nm + '_kernel')
        except (OSError, ValueError):
            pass
        roofline['kernels'].append({'kernel': nm + '_kernel', 'kernel_ms': kt[0], 'algorithmic_bytes_per_frame': bytes_[nm],
                                    'achieved': gbs, 'frac': gbs / peak_gbs,
                                    'traffic': ent['dram_bytes_per_launch'] if ent and ent.get('frames_per_launch') == B else None})
    step_gbs = bytes_['step'] * B / (ms_per_step * 1e-3) / 1e9
    line = {'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps,
            'warmup': max(3, args.warmup), 'ms_per_step': ms_per_step, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': dict(workload, launch='cuda_graph_replay' if graph is not None else 'eager',
                           kept_points_per_frame=kept_per_frame, plan=plan_mode,
                           geometry=('rig: cell indices derived on the device from sensor2ego @ inv(intrin), variant %d, bit-exact '
                                     'vs the reference ops (checked in this run)' % variant) if variant is not None
                           else 'geom_xyz: int32 tensor made by the reference ops',
                           sorted_entries_per_frame=(max_runs / B if max_runs else kept_per_frame)),
            'roofline': roofline,
            'step_roofline': {'algorithmic_bytes_per_frame': bytes_['step'], 'achieved': step_gbs, 'unit': 'GB/s',
                              'frac': step_gbs / peak_gbs, 'frac_of_nominal_8TBps': step_gbs / 8000.0},
            'stages_ms': {k: {'median': v[0], 'min': v[1]} for k, v in stages.items()},
            'channels_last_step': (None if cl_ms is None else
                                   {'what': 'same step with channels_last context and incoming gradient (zero-copy '
                                            'layouts: no transposes, no gradient-row pass), CUDA graph replay, this rank',
                                    'ms_per_step': cl_ms[0], 'frames_per_s': B / (cl_ms[0] * 1e-3)}),
            'sustained': sustained,
            'tolerance': 'integer work bit-exact; fp32 features/gradients rtol 1e-5 vs the fp64 oracle + 1e-6 x sum|terms| of the '
                         'cell (a few ulps of the partial sums; the reference itself is not run-to-run stable: fp32 atomicAdd order)',
            'gpu_launches': launches_per_step * args.steps,
            'clocks': clocks.summary()}

    line['e2e'] = e2e
    if not args.no_extras and world == 1:
        # ---- the reference's own CUDA op on the same GPU (oracle/_ref), same inputs
        try:
            from oracle import ref_cuda_op
            if ref_cuda_op.available():
                rb = min(B, 8)
                g_r, d_r, c_r, go_r = geom[:rb], depth[:rb * cfg.num_cams], ctx[:rb * cfg.num_cams], go[:rb]
                d_r = d_r.detach().requires_grad_(True)
                c_r = c_r.detach().requires_grad_(True)

                def ref_step():
                    d_r.grad = None
                    c_r.grad = None
                    ref_cuda_op.ref_pipeline(g_r, d_r, c_r, vn).backward(go_r)
                med, mn = time_cuda(ref_step, 5, 2)
                line['ref_cuda'] = {'what': 'reference pipeline lss_fpn.py:441-466 with its own CUDA kernel '
                                            '(compiled for sm_100a) + autograd backward, same GPU',
                                    'frames_per_step': rb, 'ms_per_step': med, 'value': rb / (med * 1e-3),
                                    'unit': UNIT}
        except Exception as e:                                  # pragma: no cover
            line['ref_cuda'] = {'error': repr(e)}

        # ---- CPU baseline: oracle port on the host cores, bounded sample
        line['cpu_baseline'] = run_cpu_baseline(cfg, 2, 3)

        # ---- batch / grid sweep (BASELINE.json configs[4], single GPU)
        try:
            line['sweep'] = run_sweep(dev, peak_gbs, full=args.sweep == 'full', ref_arms=args.sweep == 'full')
        except Exception as e:                                  # pragma: no cover
            line['sweep'] = {'error': repr(e)}

        # ---- drop-in op (A) on pre-materialised features beside the reference's CUDA op
        try:
            line['dropin_op'] = run_dropin_op(dev, peak_gbs)
        except Exception as e:                                  # pragma: no cover
            line['dropin_op'] = {'error': repr(e)}

        # ---- fp16 / bf16 inputs (generic kernels, fp32 accumulation)
        try:
            line['half_precision'] = run_half_precision_side(dev)
        except Exception as e:                                  # pragma: no cover
            line['half_precision'] = {'error': repr(e)}

        # ---- depth labels for the depth loss (SURVEY.md 8f, N3)
        try:
            line['depth_labels'] = run_depth_labels_side(dev, peak_gbs)
        except Exception as e:                                  # pragma: no cover
            line['depth_labels'] = {'error': repr(e)}

        # ---- LiDAR branch (BASELINE.json configs[2]): hard voxelization + HardSimpleVFE mean + pillar scatter
        try:
            line['lidar'] = run_lidar_side(dev, peak_gbs)
        except Exception as e:                                  # pragma: no cover
            line['lidar'] = {'error': repr(e)}

    sys.stdout.flush()
    os.write(json_fd, (json.dumps(line) + '\n').encode())
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == '__main__':
    main()

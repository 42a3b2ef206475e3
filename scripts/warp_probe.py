#!/usr/bin/env python
"""BDA warp measurement on one GPU (CFG-2, 32 frames): the native warp (csrc/bev_warp.cu) against kornia's sequence
run through torch's own kernels, alone and inside the camera step.

    python scripts/warp_probe.py [--frames 32] [--rounds 3] [--out FILE]

(a) warp forward + backward on a (32, 80, 64, 512) fp32 map: ``warp_affine`` (channels-last rows, as the pooling ops
    return them) vs ``F.affine_grid`` + ``F.grid_sample`` on the NCHW map, with the same theta.
(b) the camera step, forward + backward to depth / context / LiDAR BEV: rig plan + ``voxel_pooling_fused_concat(...,
    bda_affine=M)`` vs ``voxel_pooling_fused`` -> ``.contiguous()`` -> stock warp -> ``torch.cat``, and vs today's
    step without BDA (``voxel_pooling_fused_concat`` without a matrix).
Every arm is one CUDA graph, timed by ``bench._graph_step_ms`` (CUDA events around the replay, L2 flushed by a 256 MB
fill before every replay); the arms alternate for ``--rounds`` rounds and the JSON keeps every round.  Bytes per second
come from the byte model below, over the peak bench.py uses (MEASURED_PEAKS.json when present, else 6650 GB/s).
"""
from __future__ import annotations

import argparse
import importlib.util
import json
import os
import statistics
import subprocess
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def _bench():
    spec = importlib.util.spec_from_file_location('bench_mod', os.path.join(ROOT, 'bench.py'))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def warp_bytes(B, C, G_src, G_dst, occupancy=1.0):
    """Compulsory DRAM traffic of warp forward + backward: the forward reads every occupied source row once and writes
    every destination row; the backward reads every destination gradient row and writes every occupied source row."""
    return 4 * C * B * (2 * occupancy * G_src + 2 * G_dst)


def gpu_info():
    info = {'name': torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info['nvidia_smi'] = q
    except (OSError, subprocess.SubprocessError) as e:
        info['nvidia_smi'] = f'unavailable: {e}'
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--frames', type=int, default=32)
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--lidar-channels', type=int, default=256)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('warp_probe.py measures on a CUDA device; none is visible')
    bench = _bench()
    from mm_training_b200 import synthetic
    from mm_training_b200.configs import CFG_2
    from mm_training_b200.ops import warp_affine
    from mm_training_b200.ops.bev_augment import warp_theta
    from mm_training_b200.ops.voxel_pooling import (LiftSplatGeometry, PoolingPlan, build_plan, rig_variant,
                                                    voxel_pooling_fused, voxel_pooling_fused_concat)
    from oracle.warp_affine_ref import bda_matrices

    dev = torch.device('cuda:0')
    cfg, B, C2 = CFG_2, args.frames, args.lidar_channels
    C = cfg.output_channels
    geom, vn_t = synthetic.camera_rig(cfg, B, device=dev, yaw_jitter_deg=5.0, seed=1)
    vn = tuple(int(v) for v in vn_t.tolist())
    X, Y, _ = vn
    G = X * Y
    depth, ctx, _ = synthetic.camera_features(cfg, B, device=dev, seed=1)
    g = torch.Generator().manual_seed(1)
    lidar = torch.randn(B, C2, Y, X, generator=g).to(dev)
    go = torch.rand(B, C + C2, Y, X, generator=g).to(dev).contiguous(memory_format=torch.channels_last)
    M = bda_matrices(B, Y, X, seed=1).to(dev)

    fr = tuple(geom.shape[1:5])
    probe = build_plan(geom, vn, frustum=fr)
    max_runs = probe.num_sorted
    occupancy = float((probe.cell_start[1:] != probe.cell_start[:-1]).float().mean())
    kept = int((probe.cell_of_point >= 0).sum().item()) / B
    variant = rig_variant(dev)
    if variant is not None:
        lsg = LiftSplatGeometry.from_config(cfg, dev)
        s2e, intrin = synthetic.camera_rig_mats(cfg, B, device=dev, yaw_jitter_deg=5.0, seed=1)
        combine = lsg.combine(s2e, intrin)                 # outside the graphs, as in bench.py
        make_plan = lambda: PoolingPlan.from_rig(lsg, combine, variant, max_runs)
    else:
        make_plan = lambda: build_plan(geom, vn, frustum=fr, max_runs=max_runs)

    # ---- (a) the warp alone
    pooled = voxel_pooling_fused(None, depth, ctx, vn, probe).detach()            # channels-last rows
    pooled_nchw = pooled.contiguous()
    go_cam = go[:, :C].contiguous(memory_format=torch.channels_last)
    xa = pooled.clone().requires_grad_(True)
    xs = pooled_nchw.clone().requires_grad_(True)

    def warp_native():
        out = warp_affine(xa, M, (Y, X))
        return (out,) + torch.autograd.grad(out, (xa,), go_cam)

    def warp_stock():
        theta = warp_theta(M, (Y, X), (Y, X))
        out = F.grid_sample(xs, F.affine_grid(theta, [B, C, Y, X], align_corners=True), mode='bilinear',
                            padding_mode='zeros', align_corners=True)
        return (out,) + torch.autograd.grad(out, (xs,), go_cam)

    # ---- (b) the camera step
    d = depth.clone().requires_grad_(True)
    c = ctx.clone().requires_grad_(True)
    o = lidar.clone().requires_grad_(True)

    def step_bda_native():
        out = voxel_pooling_fused_concat(d, c, o, vn, make_plan(), bda_affine=M)
        return (out,) + torch.autograd.grad(out, (d, c, o), go)

    def step_bda_stock():
        plan = make_plan()
        p = voxel_pooling_fused(None, d, c, vn, plan).contiguous()                  # lss_fpn.py:466
        theta = warp_theta(M, (Y, X), (Y, X))
        w = F.grid_sample(p, F.affine_grid(theta, [B, C, Y, X], align_corners=True), mode='bilinear',
                          padding_mode='zeros', align_corners=True)
        out = torch.cat([w, o], 1)
        return (out,) + torch.autograd.grad(out, (d, c, o), go)

    def step_nobda():
        out = voxel_pooling_fused_concat(d, c, o, vn, make_plan())
        return (out,) + torch.autograd.grad(out, (d, c, o), go)

    arms = {'a_warp_native': warp_native, 'a_warp_stock': warp_stock, 'b_step_bda_native': step_bda_native,
            'b_step_bda_stock': step_bda_stock, 'b_step_no_bda': step_nobda}
    # outputs of the native and stock arms, eagerly: same results within float32 rounding
    agree = {}
    for a_, b_ in (('a_warp_native', 'a_warp_stock'), ('b_step_bda_native', 'b_step_bda_stock')):
        ra, rb = arms[a_](), arms[b_]()
        agree[f'{a_} vs {b_}'] = [float((u.detach().float() - v.detach().float()).abs().max() / v.detach().float().abs().max().clamp_min(1e-30))
                                  for u, v in zip(ra, rb)]
        del ra, rb
    torch.cuda.synchronize()

    step_bytes = bench.algorithmic_bytes(cfg, kept)['step'] * B + 8 * C2 * G * B                   # pooling + LiDAR half
    bda_extra = 16 * C * G * B * occupancy          # pooled rows written + read, gradient rows written + read
    model = {'a_warp_native': warp_bytes(B, C, G, G), 'a_warp_stock': warp_bytes(B, C, G, G),
             'b_step_bda_native': step_bytes + bda_extra, 'b_step_bda_stock': step_bytes + bda_extra,
             'b_step_no_bda': step_bytes}
    rounds = {k: [] for k in arms}
    errors = {}
    for _ in range(args.rounds):
        for k, fn in arms.items():
            if k in errors:
                continue
            try:
                rounds[k].append(bench._graph_step_ms(fn, iters=20, warmup=3, flush_l2=True)[0])
            except Exception as e:                                              # noqa: BLE001
                errors[k] = repr(e)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except OSError:
        pass
    peak_gbs = float(peaks.get('hbm_gbs', 6650.0))
    res = {'device': gpu_info(), 'config': cfg.name, 'frames': B, 'grid': [Y, X], 'channels': C, 'lidar_channels': C2,
           'occupied_cell_fraction': occupancy, 'plan': 'rig' if variant is not None else 'geom_xyz',
           'timing': 'median of 20 replays of one CUDA graph per arm (CUDA events), L2 flushed before each replay; '
                     f'arms alternated over {args.rounds} rounds',
           'byte_model': {'a': '4 B * C * B * (2 * H*W + 2 * H\'*W\'): warp reads the map, writes the warped map; backward '
                                'reads its gradient, writes the map gradient',
                          'b': 'bench.algorithmic_bytes(CFG-2)["step"] per frame + 8 B * C_lidar * Y*X per frame (LiDAR half '
                               'read + written into the concatenated buffer); BDA arms + 16 B * C * Y*X * occupancy per '
                               'frame (pooled rows written + read by the warp, their gradient rows written + read)'},
           'peak_gbs': peak_gbs,
           'peak_source': 'measured (MEASURED_PEAKS.json)' if peaks else 'fallback 6650 GB/s (no MEASURED_PEAKS.json)',
           'output_agreement_max_rel': agree, 'errors': errors, 'arms': {}}
    for k in arms:
        if not rounds[k]:
            continue
        ms = statistics.median(rounds[k])
        gbs = model[k] / (ms * 1e-3) / 1e9
        res['arms'][k] = {'ms_rounds': rounds[k], 'ms': ms, 'frames_per_s': B / (ms * 1e-3), 'model_bytes': model[k],
                          'gb_per_s': gbs, 'fraction_of_peak': gbs / peak_gbs}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(json.dumps(res, indent=1) + '\n')


if __name__ == '__main__':
    main()

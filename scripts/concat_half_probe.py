#!/usr/bin/env python
"""The 16-bit concat on one GPU (CFG-2, bf16 256-channel LiDAR BEV, autocast pair: fp32 depth + bf16 context):
``voxel_pooling_fused_concat(..., dtype=torch.bfloat16)`` against the float32 concat followed by ``.to(torch.bfloat16)``
(what autocast's first conv does to it today), forward + backward to depth, context and the LiDAR BEV with a bf16
gradient.

    python scripts/concat_half_probe.py [--frames 32] [--rounds 3] [--out FILE]

Scenarios: no BDA with the LiDAR BEV on the camera grid; BDA (``bda_matrices``) on the camera grid; no BDA with a 4x
down-sampled LiDAR BEV (``resize_other='nearest'``).  Every arm is one CUDA graph on a fixed run plan, timed by
``bench._graph_step_ms`` (CUDA events, 256 MB L2 flush before every replay); the two arms of a scenario alternate over
``--rounds`` rounds.  Reported per arm: ms per step, the shape-derived byte model of the buffer traffic (``byte_model``),
and per scenario whether the two arms' outputs and gradients are bit-equal.  Harness and device query come from
scripts/warp_probe.py.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from warp_probe import _bench, gpu_info   # noqa: E402

SCENARIOS = {'nobda_identity': (False, 1), 'bda_identity': (True, 1), 'nobda_down4': (False, 4)}


def byte_model(G, occ, C, C2, G_src, bda, half):
    """Estimated DRAM bytes per frame of what differs between the arms (the pooling's own traffic is common to both and
    left out): the camera and LiDAR halves of the buffer, the cast and its backward, the camera gradient rows and the
    LiDAR gradient.  G cells, occ occupied cells, G_src LiDAR source cells (bf16)."""
    Ct = C + C2
    resized = G_src != G
    if not half:
        fwd = G * C * 4 + G_src * C2 * 2 + G * C2 * 4 + G * Ct * 4 + G * Ct * 2           # rows, LiDAR, cast
        bwd = G * Ct * 2 + G * Ct * 4                                                   # cast backward
        bwd += (G * C * 4 if bda else 0) + occ * C * 4                                  # warp reads / column kernel reads
        bwd += G * C2 * 4 + G_src * C2 * 2                                              # LiDAR gradient (.to or adjoint)
    else:
        fwd = G * C * 2 + G_src * C2 * 2 + G * C2 * 2
        bwd = (G * C * 2 if bda else occ * C * 2 + occ * C * 4) + occ * C * 4          # warp / widen, column kernel reads
        bwd += (G * C2 * 2 + G_src * C2 * 2) if resized else 0                          # identity: a view
    if bda:
        fwd += occ * C * 4                                                              # the warp reads the pooled scratch
        bwd += occ * C * 4                                                              # ... and writes its gradient rows
    return {'forward': fwd, 'backward': bwd, 'step': fwd + bwd}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--frames', type=int, default=32)
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--lidar-channels', type=int, default=256)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('concat_half_probe.py measures on a CUDA device; none is visible')
    bench = _bench()
    from mm_training_b200 import synthetic
    from mm_training_b200.configs import CFG_2
    from mm_training_b200.ops.voxel_pooling import build_plan, voxel_pooling_fused_concat
    from oracle.warp_affine_ref import bda_matrices

    dev = torch.device('cuda:0')
    cfg, B, C2 = CFG_2, args.frames, args.lidar_channels
    C = cfg.output_channels
    Ct = C + C2
    bf16 = torch.bfloat16
    geom, vn_t = synthetic.camera_rig(cfg, B, device=dev, yaw_jitter_deg=5.0, seed=1)
    vn = tuple(int(v) for v in vn_t.tolist())
    X, Y, _ = vn
    G = X * Y
    fr = tuple(geom.shape[1:5])
    n = build_plan(geom, vn, frustum=fr).num_sorted
    plan = build_plan(geom, vn, frustum=fr, max_runs=n)
    occ = float((plan.cell_start[1:] != plan.cell_start[:-1]).float().sum()) / B
    depth, ctx, _ = synthetic.camera_features(cfg, B, device=dev, seed=1)
    gen = torch.Generator().manual_seed(1)
    go = torch.rand(B, Ct, Y, X, generator=gen).to(dev, bf16).contiguous(memory_format=torch.channels_last)
    M = bda_matrices(B, Y, X, seed=1).to(dev)
    d = depth.clone().requires_grad_(True)
    c = ctx.to(bf16).requires_grad_(True)

    arms, model, pairs = {}, {}, []
    for name, (bda, k) in SCENARIOS.items():
        o = torch.randn(B, C2, k * Y, k * X, generator=gen).to(dev, bf16).requires_grad_(True)
        Mk = M if bda else None
        resize = 'nearest' if k != 1 else None

        def fp32_cast(o=o, Mk=Mk, resize=resize):
            out = voxel_pooling_fused_concat(d, c, o, vn, plan, bda_affine=Mk, resize_other=resize).to(bf16)
            return (out,) + torch.autograd.grad(out, (d, c, o), go)

        def half(o=o, Mk=Mk, resize=resize):
            out = voxel_pooling_fused_concat(d, c, o, vn, plan, bda_affine=Mk, resize_other=resize, dtype=bf16)
            return (out,) + torch.autograd.grad(out, (d, c, o), go)

        arms[name + '_fp32_then_cast'], arms[name + '_bf16'] = fp32_cast, half
        for key, h in ((name + '_fp32_then_cast', False), (name + '_bf16', True)):
            model[key] = {p: v * B for p, v in byte_model(G, occ, C, C2, k * k * G, bda, h).items()}
        pairs.append((name + '_bf16', name + '_fp32_then_cast'))

    agree = {}
    for a_, b_ in pairs:
        ra = [t.detach().clone() for t in arms[a_]()]
        rb = [t.detach().clone() for t in arms[b_]()]
        agree[a_.rsplit('_', 1)[0]] = {'out_grad_depth_grad_context_grad_lidar_bit_equal':
                                       [bool(torch.equal(u, v)) for u, v in zip(ra, rb)]}
        del ra, rb
    torch.cuda.synchronize()

    rounds = {k: [] for k in arms}
    for _ in range(args.rounds):
        for a_, b_ in pairs:
            for key in (a_, b_):
                rounds[key].append(bench._graph_step_ms(arms[key], iters=20, warmup=3, flush_l2=True)[0])
    res = {'device': gpu_info(), 'config': cfg.name, 'frames': B, 'grid': [Y, X], 'channels': C, 'lidar_channels': C2,
           'context': 'bf16 (fp32 depth)', 'lidar_dtype': 'bf16', 'gradient': 'bf16 channels_last',
           'occupied_cells_per_frame': occ,
           'timing': 'median of 20 replays of one CUDA graph per arm (CUDA events), L2 flushed before each replay; '
                     f'arms alternated over {args.rounds} rounds; fixed run plan',
           'byte_model': byte_model.__doc__.strip() + ' Estimates from shapes, not measured traffic.',
           'bit_equal': agree, 'arms': {}}
    for k in arms:
        ms = statistics.median(rounds[k])
        res['arms'][k] = {'ms_rounds': rounds[k], 'us_per_step': ms * 1e3, 'model_bytes': model[k]}
    res['bf16_over_fp32_then_cast'] = {a_.rsplit('_', 1)[0]: res['arms'][a_]['us_per_step'] / res['arms'][b_]['us_per_step']
                                       for a_, b_ in pairs}
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(json.dumps(res, indent=1) + '\n')


if __name__ == '__main__':
    main()

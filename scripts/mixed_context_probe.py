#!/usr/bin/env python
"""Autocast pooling measurement on one GPU: the mixed call (fp32 depth, bf16 context read by the kernels) against the
upcast route (``context.float()``, the fp32 kernels, autograd's cast of the context gradient back to bf16).

    python scripts/mixed_context_probe.py [--frames 32] [--aim-frames 4] [--rounds 3] [--out FILE]

Shapes: CFG-2 (W = 44: a bf16 NCHW row is 88 bytes, not a tensor-map row, so the mixed call takes pixel rows) and
CFG_AIM (W = 80: the mixed call reads the NCHW context through a bf16 tensor map).  Each arm is forward + backward to
depth and context on a fixed run plan, captured as one CUDA graph and timed by ``bench._graph_step_ms`` (CUDA events,
256 MB L2 flush before every replay); arms alternate for ``--rounds`` rounds.  Both arms' outputs and gradients are
compared bit for bit first.
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


def context_bytes(n, route):
    """Context-side DRAM traffic per step for n context elements (depth, plan and output traffic is the same in every
    arm and left out).  upcast: the fp32 copy (read 2 B, write 4 B), the kernels' fp32 read in forward and backward
    (4 B + 4 B), the fp32 gradient write (4 B) and the cast to bf16 (read 4 B, write 2 B).  mixed: the kernels read 2 B
    twice and write the 2-B gradient; the pixel-rows route adds a transpose each way (read 2 B, write 2 B)."""
    if route == 'upcast':
        return n * (2 + 4 + 4 + 4 + 4 + 4 + 2)
    return n * (2 + 2 + 2 + (8 if route == 'rows' else 0))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--frames', type=int, default=32)
    ap.add_argument('--aim-frames', type=int, default=4)
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('mixed_context_probe.py measures on a CUDA device; none is visible')
    bench = _bench()
    from mm_training_b200 import synthetic
    from mm_training_b200.configs import CFG_2, CFG_AIM
    from mm_training_b200.ops.voxel_pooling import build_plan, voxel_pooling_fused
    from mm_training_b200.ops.voxel_pooling.voxel_pooling import _route

    dev = torch.device('cuda:0')
    arms, model, meta, agree = {}, {}, {}, {}
    for cfg, B in ((CFG_2, args.frames), (CFG_AIM, args.aim_frames)):
        geom, vn_t = synthetic.camera_rig(cfg, B, device=dev, yaw_jitter_deg=5.0, seed=1)
        vn = tuple(int(v) for v in vn_t.tolist())
        plan = build_plan(geom, vn, frustum=tuple(geom.shape[1:5]))
        del geom
        depth, ctx, go = synthetic.camera_features(cfg, B, device=dev, seed=1)
        d = depth.requires_grad_(True)
        c = ctx.to(torch.bfloat16).requires_grad_(True)
        route = _route(plan.mode, c, d)

        def mixed(d=d, c=c, go=go, vn=vn, plan=plan):
            out = voxel_pooling_fused(None, d, c, vn, plan)
            return (out,) + torch.autograd.grad(out, (d, c), go)

        def upcast(d=d, c=c, go=go, vn=vn, plan=plan):
            out = voxel_pooling_fused(None, d, c.float(), vn, plan)
            return (out,) + torch.autograd.grad(out, (d, c), go)

        name = cfg.name.split('_')[0]
        arms[f'{name}_mixed'], arms[f'{name}_upcast'] = mixed, upcast
        n = c.numel()
        model[f'{name}_mixed'], model[f'{name}_upcast'] = context_bytes(n, route), context_bytes(n, 'upcast')
        meta[name] = {'config': cfg.name, 'frames': B, 'feat_hw': list(cfg.feat_hw), 'depth_bins': cfg.depth_bins,
                      'channels': cfg.output_channels, 'context_elements': n, 'mixed_route': route}
        ra, rb = [t.detach().clone() for t in mixed()], [t.detach().clone() for t in upcast()]
        agree[name] = [bool(torch.equal(u, v)) for u, v in zip(ra, rb)]
        del ra, rb
    torch.cuda.synchronize()

    rounds = {k: [] for k in arms}
    for _ in range(args.rounds):
        for k, fn in arms.items():
            rounds[k].append(bench._graph_step_ms(fn, iters=20, warmup=3, flush_l2=True)[0])
    res = {'device': gpu_info(), 'shapes': meta,
           'timing': 'median of 20 replays of one CUDA graph per arm (CUDA events), L2 flushed before each replay; '
                     f'arms alternated over {args.rounds} rounds',
           'byte_model': context_bytes.__doc__.strip(),
           'bit_equal_out_grad_depth_grad_context': agree, 'arms': {}}
    for k in arms:
        ms = statistics.median(rounds[k])
        res['arms'][k] = {'us_per_step': round(ms * 1000, 1), 'rounds_us': [round(t * 1000, 1) for t in rounds[k]],
                          'context_bytes_model_MB': round(model[k] / 1e6, 1)}
    for name in meta:
        m, u = res['arms'][f'{name}_mixed']['us_per_step'], res['arms'][f'{name}_upcast']['us_per_step']
        print(f'{name}: mixed {m} us  upcast {u} us  ({meta[name]["mixed_route"]} route; context bytes '
              f'{res["arms"][f"{name}_mixed"]["context_bytes_model_MB"]} vs '
              f'{res["arms"][f"{name}_upcast"]["context_bytes_model_MB"]} MB; bit-equal {agree[name]})', flush=True)
    text = json.dumps(res, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(text + '\n')
    print(text)


if __name__ == '__main__':
    main()

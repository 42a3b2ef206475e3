#!/usr/bin/env python
"""LiDAR BEV resampling measurement on one GPU (CFG-2 grid, 256 LiDAR channels): the native nearest resampling into
the concatenated rows (csrc/bev_resample.cu) against ``F.interpolate`` + the concat copy, alone and inside the camera
step with BDA.

    python scripts/concat_probe.py [--frames 32] [--rounds 3] [--out FILE]

(a) LiDAR half alone, forward + backward, for three source grids (2x up from 32 x 256, the identity 64 x 512, 4x down
    from 256 x 2048), fp32 and bf16, NCHW and channels_last:
      native  ``bevpool_resize_nearest_into`` into the (B, Y, X, 80 + 256) rows, ``bevpool_resize_nearest_backward_from``
              out of the channels-last concatenated gradient;
      stock   ``F.interpolate(...).float()`` copied into the same rows (what the concat did before), torch's nearest
              backward on the LiDAR slice of the same gradient.
(b) the camera step with BDA, forward + backward to depth / context / LiDAR BEV (2x up, fp32 and bf16, NCHW): rig plan +
    ``voxel_pooling_fused_concat(..., bda_affine=M, resize_other='nearest')`` vs ``F.interpolate`` then
    ``voxel_pooling_fused_concat(..., bda_affine=M)``.
Harness, graph timing, L2 flush and device query come from scripts/warp_probe.py: every arm is one CUDA graph timed by
``bench._graph_step_ms`` (CUDA events, 256 MB L2 flush before every replay); arms alternate for ``--rounds`` rounds.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from warp_probe import ROOT, _bench, gpu_info   # noqa: E402

SOURCES = {'up2': (32, 256), 'identity': (64, 512), 'down4': (256, 2048)}
# frames per source in (a): a quarter of --frames at 4x down (its fp32 source and source gradient are 537 MB each per
# frame; the 12 arms' inputs and graph pools must fit together)
FRAME_DIV = {'up2': 1, 'identity': 1, 'down4': 4}


def lidar_bytes(B, C2, G_src, G_dst, elem):
    """Compulsory DRAM traffic of the LiDAR half, forward + backward: read the source, write the fp32 rows; read the
    gradient rows, write the source gradient.  The stock arm moves more (the interpolated copy is written and read
    again in the forward; a 16-bit source adds a conversion pass each way); its time is set against the same model."""
    return B * C2 * (G_src * elem + 4 * G_dst + 4 * G_dst + G_src * elem)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--frames', type=int, default=32)
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--lidar-channels', type=int, default=256)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('concat_probe.py measures on a CUDA device; none is visible')
    bench = _bench()
    from mm_training_b200 import _lib, synthetic
    from mm_training_b200.configs import CFG_2
    from mm_training_b200.ops.voxel_pooling import (LiftSplatGeometry, PoolingPlan, build_plan, rig_variant,
                                                    voxel_pooling_fused_concat)
    from oracle.warp_affine_ref import bda_matrices

    dev = torch.device('cuda:0')
    cfg, B, C2 = CFG_2, args.frames, args.lidar_channels
    C = cfg.output_channels
    Ct = C + C2
    geom, vn_t = synthetic.camera_rig(cfg, B, device=dev, yaw_jitter_deg=5.0, seed=1)
    vn = tuple(int(v) for v in vn_t.tolist())
    X, Y, _ = vn
    G = X * Y
    gen = torch.Generator().manual_seed(1)
    go = torch.rand(B, Ct, Y, X, generator=gen).to(dev).contiguous(memory_format=torch.channels_last)
    L = _lib.lib()
    stream = lambda: _lib.stream_ptr(dev)

    arms, model, pairs = {}, {}, []
    # ---- (a) the LiDAR half alone
    for sname, (Yl, Xl) in SOURCES.items():
        Bs = max(1, B // FRAME_DIV[sname])
        gos = go[:Bs]
        for dtype in (torch.float32, torch.bfloat16):
            for layout in ('nchw', 'cl'):
                src = torch.randn(Bs, C2, Yl, Xl, generator=gen).to(dtype).to(dev)
                if layout == 'cl':
                    src = src.contiguous(memory_format=torch.channels_last)
                nchw = 1 if layout == 'nchw' else 0
                code = _lib.dtype_code(src)
                buf = torch.empty(Bs, Y, X, Ct, device=dev)
                xs = src.clone().requires_grad_(True)

                def native(src=src, nchw=nchw, code=code, buf=buf, Yl=Yl, Xl=Xl, Bs=Bs, gos=gos):
                    _lib.check(L.bevpool_resize_nearest_into(src.data_ptr(), code, nchw, Bs, C2, Yl, Xl, Y, X,
                                                             buf.data_ptr() + 4 * C, Ct, stream()), 'into')
                    gsrc = torch.empty_like(src)
                    _lib.check(L.bevpool_resize_nearest_backward_from(gos.data_ptr() + 4 * C, Ct, gsrc.data_ptr(), code,
                                                                      nchw, Bs, C2, Yl, Xl, Y, X, stream()), 'backward_from')
                    return buf, gsrc

                def stock(xs=xs, buf=buf, gos=gos):
                    lid = F.interpolate(xs, size=(Y, X), mode='nearest').float()
                    buf[..., C:].copy_(lid.detach().permute(0, 2, 3, 1))
                    (gsrc,) = torch.autograd.grad(lid, (xs,), gos[:, C:])
                    return buf, gsrc

                key = f'a_{sname}_{str(dtype)[6:]}_{layout}'
                arms[key + '_native'], arms[key + '_stock'] = native, stock
                m = lidar_bytes(Bs, C2, Yl * Xl, G, src.element_size())
                model[key + '_native'] = model[key + '_stock'] = m
                pairs.append((key + '_native', key + '_stock'))
                if sname == 'identity':
                    # the forward alone against the concat's former copy_ (the identity backward is a view either way)
                    def fwd_native(src=src, nchw=nchw, code=code, buf=buf, Bs=Bs):
                        _lib.check(L.bevpool_resize_nearest_into(src.data_ptr(), code, nchw, Bs, C2, Y, X, Y, X,
                                                                 buf.data_ptr() + 4 * C, Ct, stream()), 'into')
                        return (buf,)

                    def fwd_copy(src=src, buf=buf):
                        buf[..., C:].copy_(src.permute(0, 2, 3, 1))
                        return (buf,)
                    arms[key + '_fwd_native'], arms[key + '_fwd_copy'] = fwd_native, fwd_copy
                    model[key + '_fwd_native'] = model[key + '_fwd_copy'] = Bs * C2 * G * (src.element_size() + 4)
                    pairs.append((key + '_fwd_native', key + '_fwd_copy'))

    # ---- (b) the camera step with BDA
    depth, ctx, _ = synthetic.camera_features(cfg, B, device=dev, seed=1)
    M = bda_matrices(B, Y, X, seed=1).to(dev)
    fr = tuple(geom.shape[1:5])
    probe = build_plan(geom, vn, frustum=fr)
    max_runs = probe.num_sorted
    kept = int((probe.cell_of_point >= 0).sum().item()) / B
    occupancy = float((probe.cell_start[1:] != probe.cell_start[:-1]).float().mean())
    variant = rig_variant(dev)
    if variant is not None:
        lsg = LiftSplatGeometry.from_config(cfg, dev)
        s2e, intrin = synthetic.camera_rig_mats(cfg, B, device=dev, yaw_jitter_deg=5.0, seed=1)
        combine = lsg.combine(s2e, intrin)
        make_plan = lambda: PoolingPlan.from_rig(lsg, combine, variant, max_runs)
    else:
        make_plan = lambda: build_plan(geom, vn, frustum=fr, max_runs=max_runs)
    d = depth.clone().requires_grad_(True)
    c = ctx.clone().requires_grad_(True)
    Yl, Xl = SOURCES['up2']
    for dtype in (torch.float32, torch.bfloat16):
        o = torch.randn(B, C2, Yl, Xl, generator=gen).to(dtype).to(dev).requires_grad_(True)

        def step_native(o=o):
            out = voxel_pooling_fused_concat(d, c, o, vn, make_plan(), bda_affine=M, resize_other='nearest')
            return (out,) + torch.autograd.grad(out, (d, c, o), go)

        def step_stock(o=o):
            out = voxel_pooling_fused_concat(d, c, F.interpolate(o, size=(Y, X), mode='nearest'), vn, make_plan(),
                                             bda_affine=M)
            return (out,) + torch.autograd.grad(out, (d, c, o), go)

        key = f'b_step_bda_up2_{str(dtype)[6:]}'
        arms[key + '_native'], arms[key + '_stock'] = step_native, step_stock
        step_bytes = (bench.algorithmic_bytes(cfg, kept)['step'] + 16 * C * G * occupancy) * B
        model[key + '_native'] = model[key + '_stock'] = step_bytes + lidar_bytes(B, C2, Yl * Xl, G, o.element_size())
        pairs.append((key + '_native', key + '_stock'))

    # outputs of each native / stock pair, eagerly on the same inputs
    agree = {}
    for a_, b_ in pairs:
        ra, rb = arms[a_](), arms[b_]()
        ra, rb = [t.detach().clone() for t in ra], [t.detach().clone() for t in rb]
        agree[f'{a_} vs {b_}'] = {
            'outputs_bit_equal': [bool(torch.equal(u, v)) for u, v in zip(ra, rb)],
            'max_rel': [float((u.float() - v.float()).abs().max() / v.float().abs().max().clamp_min(1e-30))
                        for u, v in zip(ra, rb)]}
        del ra, rb
    torch.cuda.synchronize()

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
           'sources': SOURCES,
           'frames_a': {k: max(1, B // FRAME_DIV[k]) for k in SOURCES}, 'occupied_cell_fraction': occupancy, 'plan': 'rig' if variant is not None else 'geom_xyz',
           'timing': 'median of 20 replays of one CUDA graph per arm (CUDA events), L2 flushed before each replay; '
                     f'arms alternated over {args.rounds} rounds',
           'byte_model': {'a': lidar_bytes.__doc__.strip(),
                          'b': 'bench.algorithmic_bytes(CFG-2)["step"] + 16 B * C * Y*X * occupancy (BDA scratch rows) per '
                               'frame, + the LiDAR half of (a)'},
           'peak_gbs': peak_gbs,
           'peak_source': 'measured (MEASURED_PEAKS.json)' if peaks else 'fallback 6650 GB/s (no MEASURED_PEAKS.json)',
           'output_agreement': agree, 'errors': errors, 'arms': {}}
    for k in arms:
        if not rounds[k]:
            continue
        ms = statistics.median(rounds[k])
        gbs = model[k] / (ms * 1e-3) / 1e9
        res['arms'][k] = {'ms_rounds': rounds[k], 'ms': ms, 'model_bytes': model[k], 'gb_per_s': gbs,
                          'fraction_of_peak': gbs / peak_gbs}
    res['native_over_stock'] = {a_: res['arms'][a_]['ms'] / res['arms'][b_]['ms'] for a_, b_ in pairs
                                if a_ in res['arms'] and b_ in res['arms']}
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(json.dumps(res, indent=1) + '\n')


if __name__ == '__main__':
    main()

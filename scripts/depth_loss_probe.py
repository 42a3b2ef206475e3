#!/usr/bin/env python
"""Depth loss measurement on one GPU: the native ``depth_loss`` (csrc/depth_loss.cu) against the reference's
``get_depth_loss`` (``bench_train.depth_loss_ref``), alone and with the depth softmax in front.

    python scripts/depth_loss_probe.py [--rounds 3] [--out FILE]

Workloads: CFG-2 with 32 frames (D 112, 16 x 44, 4 cameras), CFG-AIM with 4 frames (D 409, 44 x 80, 2 cameras).
(1) loss forward + backward to the probabilities: native with dense fp32 label rows, native with int32 bins, and the
    reference eagerly (its boolean gathers sync the host, so it cannot be captured); the native arms are timed both as
    one CUDA graph and eagerly, for a like-for-like figure.
(2) the depth chain, forward + backward to the logits: ``depth_distribution`` + ``depth_loss`` (graph and eager) against
    ``torch.softmax`` + the reference (eager).
Labels: one-hot rows of random bins with a quarter zero rows.  Harness, L2 flush and device query come from
scripts/warp_probe.py: graph arms are timed by ``bench._graph_step_ms`` (CUDA events, 256 MB L2 flush before every
replay), eager arms the same way around a direct call; arms alternate for ``--rounds`` rounds.  Host syncs per step
are counted with ``torch.cuda.set_sync_debug_mode('warn')``.  The chain arms start from different probabilities
(``depth_distribution`` against ``torch.softmax``), so their gradients are not expected to share bits; the chain's bit
equality with depth_distribution fed torch's gradient is a GPU test (tests/test_gpu_depth_loss.py).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import warnings

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from warp_probe import _bench, gpu_info   # noqa: E402

WORKLOADS = {'cfg2_32f': ('CFG_2', 32), 'aim_4f': ('CFG_AIM', 4)}


def loss_bytes(E, Px, bins):
    """Compulsory DRAM traffic of the loss, forward + backward.  Dense: read prob + labels (8 E), then read prob +
    labels and write the gradient (12 E).  Bins: 4 E + 4 Px, then 8 E + 4 Px."""
    return (12 * E + 8 * Px) if bins else 20 * E


def softmax_bytes(E):
    """depth_distribution forward (read logits, write prob) + backward (read prob and its gradient, write the logits'
    gradient): 2 E + 3 E floats."""
    return 20 * E


def _eager_ms(fn, iters=20, warmup=3):
    scrub = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        scrub.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    del scrub
    return statistics.median(ts)


def _syncs(fn):
    """Host syncs of one call after a warm-up call (first-call initialisation is not part of a step)."""
    fn()
    torch.cuda.synchronize()
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter('always')
        torch.cuda.set_sync_debug_mode('warn')
        try:
            fn()
        finally:
            torch.cuda.set_sync_debug_mode('default')
    torch.cuda.synchronize()
    return sum('synchroniz' in str(x.message) for x in w)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('depth_loss_probe.py measures on a CUDA device; none is visible')
    bench = _bench()
    import bench_train
    from mm_training_b200 import configs
    from mm_training_b200.ops import depth_loss
    from mm_training_b200.ops.depth_distribution import depth_distribution

    dev = torch.device('cuda:0')
    gen = torch.Generator().manual_seed(1)
    arms, kind, model, pairs, syncs, agree, shapes = {}, {}, {}, [], {}, {}, {}
    for wname, (cname, frames) in WORKLOADS.items():
        cfg = getattr(configs, cname)
        D = cfg.depth_bins
        H, W = cfg.feat_hw
        BN = frames * cfg.num_cams
        E, Px = BN * D * H * W, BN * H * W
        shapes[wname] = {'config': cfg.name, 'frames': frames, 'shape': [BN, D, H, W], 'E': E, 'pixels': Px}
        logits = (3 * torch.randn(BN, D, H, W, generator=gen)).to(dev)
        prob = torch.softmax(logits, 1)
        b = torch.randint(0, D, (Px,), generator=gen)
        zero = torch.rand(Px, generator=gen) < 0.25
        bins = b.int().masked_fill(zero, -1).to(dev)
        dense = F.one_hot(b, D).float().masked_fill(zero[:, None], 0.0).to(dev)

        def loss_step(fn, labels, prob=prob):
            def step():
                x = prob.detach().requires_grad_(True)
                L = fn(labels, x)
                return (L.detach(),) + torch.autograd.grad(L, (x,))
            return step

        def chain_step(fn, soft, logits=logits, dense=dense):
            def step():
                x = logits.detach().requires_grad_(True)
                p = soft(x)
                L = fn(dense, p)
                return (L.detach(),) + torch.autograd.grad(L, (x,))
            return step

        ref = lambda t, p, D=D: bench_train.depth_loss_ref(t, p, D)
        native_soft = lambda x, D=D: depth_distribution(x, D)[0]
        steps = {
            f'{wname}_loss_native_dense': (loss_step(depth_loss, dense), loss_bytes(E, Px, False)),
            f'{wname}_loss_native_bins': (loss_step(depth_loss, bins), loss_bytes(E, Px, True)),
            f'{wname}_loss_reference': (loss_step(ref, dense), loss_bytes(E, Px, False)),
            f'{wname}_chain_native': (chain_step(depth_loss, native_soft), loss_bytes(E, Px, False) + softmax_bytes(E)),
            f'{wname}_chain_reference': (chain_step(ref, lambda x: torch.softmax(x, 1)),
                                         loss_bytes(E, Px, False) + softmax_bytes(E)),
        }
        for k, (fn, m) in steps.items():
            native = 'native' in k
            for mode in (('graph', 'eager') if native else ('eager',)):
                arms[f'{k}_{mode}'] = fn
                kind[f'{k}_{mode}'] = mode
                model[f'{k}_{mode}'] = m
            syncs[k] = _syncs(fn)
        for a_, b_ in [(f'{wname}_loss_native_dense', f'{wname}_loss_reference'),
                       (f'{wname}_loss_native_bins', f'{wname}_loss_reference'),
                       (f'{wname}_loss_native_bins', f'{wname}_loss_native_dense'),
                       (f'{wname}_chain_native', f'{wname}_chain_reference')]:
            ra, rb = steps[a_][0](), steps[b_][0]()
            agree[f'{a_} vs {b_}'] = {
                'loss_rel_diff': float((ra[0].double() - rb[0].double()).abs() / rb[0].double().abs()),
                'gradient_bit_equal': bool(torch.equal(ra[1], rb[1]))}
            del ra, rb
        for k in steps:
            if 'native' in k:
                ref_k = k.replace('native_dense', 'reference').replace('native_bins', 'reference').replace(
                    'chain_native', 'chain_reference')
                pairs += [(f'{k}_graph', f'{ref_k}_eager'), (f'{k}_eager', f'{ref_k}_eager')]
    torch.cuda.synchronize()

    rounds = {k: [] for k in arms}
    errors = {}
    for _ in range(args.rounds):
        for k, fn in arms.items():
            if k in errors:
                continue
            try:
                if kind[k] == 'graph':
                    rounds[k].append(bench._graph_step_ms(fn, iters=20, warmup=3, flush_l2=True)[0])
                else:
                    rounds[k].append(_eager_ms(fn))
            except Exception as e:                                              # noqa: BLE001
                errors[k] = repr(e)
    res = {'device': gpu_info(), 'workloads': shapes,
           'timing': 'median of 20 calls per arm (CUDA events), L2 flushed (256 MB fill) before each; graph arms replay '
                     f'one CUDA graph, eager arms call the step directly; arms alternated over {args.rounds} rounds',
           'byte_model': {'loss': loss_bytes.__doc__.strip(), 'chain': 'loss + ' + softmax_bytes.__doc__.strip()},
           'labels': 'one-hot rows of random bins, 25 % zero rows (bins: -1)',
           'host_syncs_per_step': syncs, 'output_agreement': agree, 'errors': errors, 'arms': {}}
    for k in arms:
        if not rounds[k]:
            continue
        ms = statistics.median(rounds[k])
        res['arms'][k] = {'ms_rounds': rounds[k], 'ms': ms, 'model_bytes': model[k],
                          'gb_per_s': model[k] / (ms * 1e-3) / 1e9}
    res['native_over_reference'] = {f'{a_} / {b_}': res['arms'][a_]['ms'] / res['arms'][b_]['ms'] for a_, b_ in pairs
                                    if a_ in res['arms'] and b_ in res['arms']}
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(json.dumps(res, indent=1) + '\n')


if __name__ == '__main__':
    main()

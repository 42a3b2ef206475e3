"""Builds ``libbevpool_sm100.so`` in-tree with nvcc (sm_100a only, no torch headers).

    python -m mm_training_b200.build [--force] [--verbose]

The library is git-ignored but travels to the GPU box with the repo snapshot.
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
LIB_PATH = os.path.join(HERE, 'libbevpool_sm100.so')
SOURCES = ['plan.cu', 'pool.cu', 'pool_runs.cu', 'pool_bwd.cu', 'pool_bwd2.cu', 'voxelize.cu', 'depth_labels.cu', 'depth_softmax.cu',
           'depth_loss.cu', 'bev_warp.cu', 'bev_resample.cu']
NVCC_FLAGS = ['-O3', '-std=c++17', '-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo',
              '-Xcompiler', '-fPIC', '--expt-relaxed-constexpr']
# never --use_fast_math: index arithmetic (voxelizer floor/div) must stay IEEE


def _sources():
    return [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


def _stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(('.cu', '.cuh'))] + \
           [os.path.join(os.path.dirname(HERE), 'include', 'bevpool_sm100.h'), os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not _stale():
        return LIB_PATH
    nvcc = os.environ.get('NVCC', 'nvcc')
    objs = []
    procs = []
    for src in _sources():
        obj = os.path.join(CSRC, os.path.basename(src).replace('.cu', '.o'))
        cmd = [nvcc, *NVCC_FLAGS, '-c', src, '-o', obj]
        if verbose:
            cmd.insert(1, '-Xptxas=-v')
            print(' '.join(cmd), flush=True)
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    for src, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode:
            sys.stderr.write(out)
        if p.returncode:
            raise RuntimeError(f'nvcc failed on {src}')
    cmd = [nvcc, '-shared', '-gencode', 'arch=compute_100a,code=sm_100a', '-o', LIB_PATH, *objs]
    subprocess.check_call(cmd)
    return LIB_PATH


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='--verbose' in sys.argv))

"""Build libbpv.so in-tree with nvcc for sm_100a (no torch, no JIT cache).

    python -m bpv.build            # from bp-from-video_b200/
"""
from __future__ import annotations

import concurrent.futures
import glob
import os
import subprocess
import sys

PKG = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(PKG, 'csrc')
OBJ = os.path.join(PKG, 'build')
LIB = os.path.join(PKG, 'libbpv.so')
NVCC = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17',
         '-Xcompiler', '-fPIC', '--use_fast_math', '-Xptxas', '-v']
# --use_fast_math only affects fp32 intrinsics choices; every fp64 path is IEEE.
# BPV_NVCC_EXTRA (extra nvcc flags, e.g. "-Xptxas -warn-spills") is appended for development builds.
FLAGS += os.environ.get('BPV_NVCC_EXTRA', '').split()


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJ, exist_ok=True)
    srcs = sorted(glob.glob(os.path.join(CSRC, '*.cu')))
    hdrs = glob.glob(os.path.join(CSRC, '*.cuh')) + glob.glob(os.path.join(PKG, '..', 'include', '*.h'))
    jobs = []
    for s in srcs:
        o = os.path.join(OBJ, os.path.basename(s)[:-3] + '.o')
        if force or _stale(o, [s] + hdrs):
            jobs.append((s, o))

    def cc(job):
        s, o = job
        r = subprocess.run([NVCC, *FLAGS, '-c', s, '-o', o], capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f'nvcc failed for {s}:\n{r.stdout}\n{r.stderr}')
        with open(o[:-2] + '.ptxas.txt', 'w') as f:
            f.write(r.stderr)
        return s, r.stderr

    with concurrent.futures.ThreadPoolExecutor(max_workers=os.cpu_count() or 4) as ex:
        for s, log in ex.map(cc, jobs):
            if verbose:
                print(f'--- {os.path.basename(s)}\n{log}')
    objs = [os.path.join(OBJ, os.path.basename(s)[:-3] + '.o') for s in srcs]
    if force or jobs or _stale(LIB, objs):
        r = subprocess.run([NVCC, '-shared', '-o', LIB, *objs, '-gencode', 'arch=compute_100a,code=sm_100a'],
                           capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f'link failed:\n{r.stdout}\n{r.stderr}')
    return LIB


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose=True))

"""
Builds libpbvi_b200.so (the C-ABI engine, include/pbvi_b200.h) in-tree with nvcc for sm_100a.

    python -m pomdp_pbvi_exploration_b200.build [--force] [--verbose]

The library is git-ignored but travels to the GPU box with the repo snapshot.  There is no CPU
fallback: if the library is missing, `_native` raises.
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
LIB = os.environ.get('PBVI_B200_LIB', os.path.join(HERE, 'libpbvi_b200.so'))
SOURCES = ['model.cu', 'backup.cu', 'belief.cu', 'misc.cu', 'hostpack.cu', 'comm.cu', 'hsvi.cu', 'prune_lp.cu']
HOST_SOURCES = ['hostpack_host.cpp']
HEADERS = ['pbvi_common.cuh', 'score_kernel.cuh', os.path.join('..', '..', 'include', 'pbvi_b200.h')]
NVCC = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-lineinfo', '-std=c++17', '-Xcompiler', '-fPIC',
         '-Xcompiler', '-fvisibility=hidden', '--use_fast_math=false', '-fmad=true']


def _stale() -> bool:
    if not os.path.isfile(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HOST_SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build_library(force: bool = False, verbose: bool = False) -> str:
    if not force and not _stale():
        return LIB
    objs = []
    os.makedirs(os.path.join(HERE, '_build'), exist_ok=True)
    flags = [f for f in FLAGS if not f.startswith('--use_fast_math')] + os.environ.get('PBVI_B200_DEFS', '').split()
    if verbose:
        flags += ['-Xptxas', '-v']
    procs = []
    for src in SOURCES:
        obj = os.path.join(HERE, '_build', os.path.basename(LIB).replace('.so', '_') + src.replace('.cu', '.o'))
        objs.append(obj)
        cmd = [NVCC, *flags, '-c', os.path.join(CSRC, src), '-o', obj]
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for src in HOST_SOURCES:                      # plain C++ (host-only code paths of the C ABI)
        obj = os.path.join(HERE, '_build', os.path.basename(LIB).replace('.so', '_') + src.replace('.cpp', '.o'))
        objs.append(obj)
        cmd = [os.environ.get('CXX', 'g++'), '-O3', '-std=c++17', '-fPIC', '-fvisibility=hidden', '-c', os.path.join(CSRC, src), '-o', obj]
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for cmd, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode:
            print(out)
        if p.returncode:
            raise RuntimeError('compilation failed: ' + ' '.join(cmd))
    cmd = [NVCC, '-shared', '-o', LIB, *objs, '-cudart', 'static', '-ldl']
    subprocess.run(cmd, check=True)
    return LIB


if __name__ == '__main__':
    print(build_library(force='--force' in sys.argv, verbose='--verbose' in sys.argv))

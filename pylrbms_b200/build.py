"""In-tree build of ``liblrbms_sm100.so`` (hand-written sm_100a CUDA + the C ABI of ``include/lrbms_sm100.h``).

``python -m pylrbms_b200.build`` or ``pylrbms_b200.build.build()``.  nvcc cross-compiles without a GPU.  The
shared object is git-ignored but travels with the repository snapshot to the GPU box.
"""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
LIB = os.path.join(HERE, 'liblrbms_sm100.so')
SOURCES = ['context.cu', 'project.cu', 'online.cu', 'band.cu', 'pcg.cu', 'symbolic.cpp']
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-lineinfo', '-std=c++17', '-Xcompiler', '-fPIC',
              '-Xcompiler', '-fvisibility=default']
if os.environ.get('LRBMS_DEVTOOLS', '0') not in ('', '0'):
    # developer build: in-kernel cycle counters of the solve kernel (tools/solve_timing.py); never the shipped library
    NVCC_FLAGS.append('-DLRBMS_DEVTOOLS')


def _nvcc():
    for cand in (os.environ.get('NVCC'), '/usr/local/cuda/bin/nvcc', 'nvcc'):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError('nvcc not found')


def _stamp():
    h = hashlib.sha256()
    for root in (CSRC, os.path.join(HERE, '..', 'include')):
        for name in sorted(os.listdir(root)):
            if name.endswith(('.cu', '.cuh', '.cpp', '.h')):
                with open(os.path.join(root, name), 'rb') as f:
                    h.update(name.encode())
                    h.update(f.read())
    h.update(' '.join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force=False, verbose=False):
    """Compile every CUDA source for sm_100a and link the shared library.  Returns the library path."""
    stamp_file = LIB + '.stamp'
    stamp = _stamp()
    if not force and os.path.exists(LIB) and os.path.exists(stamp_file) and open(stamp_file).read() == stamp:
        return LIB
    nvcc = _nvcc()
    objdir = os.path.join(HERE, 'build')
    os.makedirs(objdir, exist_ok=True)

    def compile_one(src):
        obj = os.path.join(objdir, os.path.splitext(src)[0] + '.o')
        cmd = [nvcc] + NVCC_FLAGS + (['-Xptxas', '-v'] if verbose else []) + ['-c', os.path.join(CSRC, src), '-o', obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError('nvcc failed for {}:\n{}\n{}'.format(src, r.stdout, r.stderr))
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=4) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    cmd = [nvcc, '-shared', '-o', LIB] + objs + ['-gencode', 'arch=compute_100a,code=sm_100a', '-lcudart']
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError('link failed:\n{}\n{}'.format(r.stdout, r.stderr))
    with open(stamp_file, 'w') as f:
        f.write(stamp)
    return LIB


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='-v' in sys.argv))

"""In-tree build of libnanowrap.so (nvcc, sm_100a only).  ``python -m ch_shrinkwrap_b200.build``."""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
LIB = os.path.join(HERE, 'libnanowrap.so')
ARCH = ['-gencode', 'arch=compute_100a,code=sm_100a']
COMMON = ['-O3', '-std=c++17', '-lineinfo', '-Xcompiler', '-fPIC', '--expt-relaxed-constexpr'] + os.environ.get('NW_EXTRA_FLAGS', '').split()
# curvature.cu, quality.cu, surface.cu and intersect.cu need one IEEE operation per source operation (see their headers)
SOURCES = {'api.cu': [], 'points.cu': [], 'tree.cu': [], 'sweep.cu': [], 'mesh_ops.cu': [], 'comm.cu': [],
           'ring.cu': [], 'benchhook.cu': [], 'xfer.cu': [], 'curvature.cu': ['-fmad=false'], 'quality.cu': ['-fmad=false'],
           'surface.cu': ['-fmad=false'], 'intersect.cu': ['-fmad=false']}


def _nvcc():
    for c in (os.environ.get('NVCC'), '/usr/local/cuda/bin/nvcc', 'nvcc'):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    raise RuntimeError('nvcc not found')


def build(force=False, verbose=False):
    nvcc = _nvcc()
    srcs = [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    deps = srcs + [os.path.join(CSRC, 'common.cuh'), os.path.join(HERE, '..', 'include', 'nanowrap.h')]
    if not force and os.path.exists(LIB) and all(os.path.getmtime(d) <= os.path.getmtime(LIB) for d in deps):
        return LIB
    objdir = os.path.join(HERE, 'build')
    os.makedirs(objdir, exist_ok=True)

    def compile_one(src):
        name = os.path.basename(src)
        obj = os.path.join(objdir, name + '.o')
        hdr_new = max(os.path.getmtime(d) for d in deps[len(srcs):])
        if not force and os.path.exists(obj) and os.path.getmtime(obj) >= max(os.path.getmtime(src), hdr_new):
            return obj
        cmd = [nvcc] + ARCH + COMMON + SOURCES[name] + (['-Xptxas', '-v'] if verbose else []) + ['-c', src, '-o', obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if verbose:
            sys.stderr.write(r.stderr)
        if r.returncode != 0:
            raise RuntimeError('nvcc failed for %s:\n%s' % (name, r.stderr[-6000:]))
        return obj

    with ThreadPoolExecutor(max_workers=8) as ex:
        objs = list(ex.map(compile_one, srcs))
    cmd = [nvcc] + ARCH + ['-shared', '-o', LIB] + objs + ['-ldl']
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError('link failed:\n' + r.stderr[-4000:])
    return LIB


if __name__ == '__main__':
    print(build(force='-f' in sys.argv, verbose='-v' in sys.argv))

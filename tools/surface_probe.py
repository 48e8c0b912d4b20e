"""Exact point-to-surface distance at C3 (nw_surface_distance): call time for the 10^7 resident localisations against the fitted
501 762-vertex mesh, and the two-way Hausdorff distance of two C3 fits.

Every time is a host clock around calls that end in a stream synchronise (each nw_surface_distance call does), so it is
device time plus the call's small host overhead: the median and the minimum of `reps` calls after two warm-up calls.
  python tools/surface_probe.py [--reps 10] [--out FILE.json]"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
from ch_shrinkwrap_b200 import evaluation_utils as eu, minimesh  # noqa: E402
from ch_shrinkwrap_b200.mesh_conj_grad import ShrinkwrapMeshConjGrad  # noqa: E402


def timed(fn, reps):
    for _ in range(2):
        fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(1e3 * (time.perf_counter() - t0))
    return {'median_ms': float(np.median(ts)), 'min_ms': float(np.min(ts)), 'reps': reps}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=10)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    gpu = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                         capture_output=True, text=True).stdout.strip()
    mesh, pts, sig, cfg = bench.build_workload('c3', 1234)
    P, M = len(pts), len(mesh._vertices)
    s_inv = np.ascontiguousarray((1.0 / sig).ravel(), dtype=np.float32)
    cg = ShrinkwrapMeshConjGrad(mesh, pts)
    mesh.cg = cg
    cg.search(pts, lams=[10.0], num_iters=5, sigma_inv=s_inv)
    fit_a = minimesh.MiniMesh(mesh._vertices['position'].copy(), mesh.faces)
    cg.search(pts, lams=[10.0], num_iters=5, sigma_inv=s_inv)
    fit_b = minimesh.MiniMesh(mesh._vertices['position'].copy(), mesh.faces)
    h = cg._h
    summary = np.empty(3)
    dist = np.empty(P)
    res = {'gpu': gpu, 'workload': 'c3', 'P': P, 'M': M, 'F': int(len(mesh.faces))}
    # the triangle-bounded boxes are rebuilt by every call: a call with no queries is that rebuild alone
    res['box_rebuild_only'] = timed(lambda: h.call('nw_surface_distance', ctypes.c_void_p(pts.ctypes.data), 0, 0, None, None, None,
                                                   None), args.reps)
    res['resident_summary_only'] = timed(lambda: h.call('nw_surface_distance', None, 0, P, None, None, None, eu._lib.dptr(summary)),
                                         args.reps)
    res['resident_dist_readback'] = timed(lambda: h.call('nw_surface_distance', None, 0, P, eu._lib.dptr(dist), None, None, None),
                                          args.reps)
    res['explicit_float32_summary_only'] = timed(lambda: h.call('nw_surface_distance', ctypes.c_void_p(pts.ctypes.data), 0, P, None,
                                                                None, None, eu._lib.dptr(summary)), args.reps)
    res['resident_summary_nm'] = {'max': summary[0], 'mean': summary[1], 'rms': summary[2]}
    aux = eu._lib.Handle(0)
    t0 = time.perf_counter()
    r = eu.hausdorff_distance(fit_a, fit_b, dx_min=5, handle=aux)
    res['hausdorff_c3_fits_after_5_and_10_iterations'] = dict(r._asdict(), call_ms=1e3 * (time.perf_counter() - t0),
                                                              dx_min=5)
    res['hausdorff_repeat'] = timed(lambda: eu.hausdorff_distance(fit_a, fit_b, dx_min=5, handle=aux), 3)
    aux.close()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()

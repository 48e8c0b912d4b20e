"""Self-intersection check at C3 (nw_self_intersections): call time on the bench's 501 762-vertex, 1 003 520-face mesh, in two
cases -- the first call right after an upload of the mesh (nw_set_topology), and repeated calls on the handle of a fit after
5 CG iterations (nothing uploaded).  Also the pair count and statistics of both meshes.

Every time is a host clock around calls that end in a stream synchronise (each nw_self_intersections call does), so it is
device time plus the call's small host overhead: the median and the minimum of `reps` calls after two warm-up calls.
  python tools/intersect_probe.py [--reps 10] [--out FILE.json]"""
import argparse
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


def timed(fn, reps, setup=None):
    """Median and minimum of `reps` timed calls of fn after two warm-up calls; `setup` (untimed) runs before every call."""
    for _ in range(2):
        if setup:
            setup()
        fn()
    ts = []
    for _ in range(reps):
        if setup:
            setup()
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
    s_inv = np.ascontiguousarray((1.0 / sig).ravel(), dtype=np.float32)
    res = {'gpu': gpu, 'workload': 'c3', 'M': int(len(mesh._vertices)), 'F': int(len(mesh.faces))}
    start = minimesh.MiniMesh(mesh._vertices['position'].copy(), mesh.faces)
    aux = eu._lib.Handle(0)
    try:
        pairs, st = eu.self_intersections(start, aux, return_stats=True)
        res['start_mesh'] = {'pairs': int(len(pairs)), 'stats': st._asdict()}
        res['first_call_after_upload'] = timed(lambda: eu._self_intersections(aux), args.reps,
                                               setup=lambda: eu._upload_surface(aux, start))
        res['repeat_after_upload'] = timed(lambda: eu._self_intersections(aux), args.reps)
    finally:
        aux.close()
    cg = ShrinkwrapMeshConjGrad(mesh, pts)
    mesh.cg = cg
    t0 = time.perf_counter()
    cg.search(pts, lams=[10.0], num_iters=5, sigma_inv=s_inv)
    res['search_5_iterations_ms'] = 1e3 * (time.perf_counter() - t0)
    pairs, st = cg.self_intersections(return_stats=True)
    res['fitted_mesh'] = {'pairs': int(len(pairs)), 'stats': st._asdict()}
    res['fitted_handle'] = timed(lambda: cg.self_intersections(), args.reps)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()

"""Exact point-to-surface distance at C3 (nw_surface_distance): call time for the 10^7 resident localisations against the fitted
501 762-vertex mesh, and the two-way Hausdorff distance of two C3 fits.  With --signed, also the signed distance
(nw_surface_signed_distance): a call with no queries just after an upload (twin table, vertex CSR, pseudonormals, volume) and
repeated (pseudonormals and volume), and the 10^7 resident localisations signed and unsigned, alternating call by call.
With --bounds, also the certified bounds of the Hausdorff distance between the two C3 fits (nw_hausdorff_bounds, both ways,
tol = 0.01 nm) against the sampled hausdorff_distance at dx_min = 5, alternating call by call on one auxiliary handle.
With --mean-bounds, the certified bounds of the area-weighted mean and RMS distances between the same two fits
(nw_mean_distance_bounds, both ways, tol = 0.01 nm, the default budget), alternating with hausdorff_distance(dx_min = 5)
and with the reference's average_squared_distance of two points_from_mesh(dx_min = 5) sample clouds (sampling included).

Every time is a host clock around calls that end in a stream synchronise (each nw_surface_distance call does), so it is
device time plus the call's small host overhead: the median and the minimum of `reps` calls after two warm-up calls.
  python tools/surface_probe.py [--reps 10] [--signed] [--bounds] [--mean-bounds] [--out FILE.json]"""
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


def timed_alternating(fns, reps, setup=None):
    """timed() of several calls, one of each in turn per repetition; `setup` (untimed) runs before every timed call."""
    for _ in range(2):
        for fn in fns.values():
            if setup:
                setup()
            fn()
    ts = {k: [] for k in fns}
    for _ in range(reps):
        for k, fn in fns.items():
            if setup:
                setup()
            t0 = time.perf_counter()
            fn()
            ts[k].append(1e3 * (time.perf_counter() - t0))
    return {k: {'median_ms': float(np.median(v)), 'min_ms': float(np.min(v)), 'reps': reps} for k, v in ts.items()}


def signed_legs(h, fit, P, reps):
    """nw_surface_signed_distance against nw_surface_distance on the fit's handle `h`; `fit` (the same mesh) on a second
    handle for the calls that need a fresh upload."""
    lib = eu._lib
    summary, dist, sdist, vol = np.empty(3), np.empty(P), np.empty(P), ctypes.c_double()
    one = np.zeros((1, 3), np.float32)
    res = {}
    aux = lib.Handle(0)
    try:
        q0 = lambda hh: hh.call('nw_surface_signed_distance', ctypes.c_void_p(one.ctypes.data), 0, 0, None, None, None,
                                ctypes.byref(vol))
        res['signed_q0_first_after_upload'] = timed_alternating({'call': lambda: q0(aux)}, reps,
                                                                setup=lambda: eu._upload_surface(aux, fit))['call']
        res['signed_q0_repeat'] = timed(lambda: q0(aux), reps)
        res['volume_nm3'] = vol.value
    finally:
        aux.close()
    res['resident_no_per_query_output'] = timed_alternating({
        'unsigned_summary_only': lambda: h.call('nw_surface_distance', None, 0, P, None, None, None, lib.dptr(summary)),
        'signed_volume_only': lambda: h.call('nw_surface_signed_distance', None, 0, P, None, None, None, ctypes.byref(vol))}, reps)
    res['resident_distance_readback'] = timed_alternating({
        'unsigned': lambda: h.call('nw_surface_distance', None, 0, P, lib.dptr(dist), None, None, None),
        'signed': lambda: h.call('nw_surface_signed_distance', None, 0, P, lib.dptr(sdist), None, None, None)}, reps)
    res['resident_inside_fraction'] = float((sdist < 0).mean())
    res['resident_abs_signed_equals_unsigned'] = bool(np.array_equal(np.abs(sdist), dist))
    return res


def bounds_legs(fit_a, fit_b, reps):
    """hausdorff_bounds(fit_a, fit_b, tol=0.01) against hausdorff_distance(dx_min=5), alternating on one auxiliary handle."""
    aux = eu._lib.Handle(0)
    try:
        r, s01, s10 = eu.hausdorff_bounds(fit_a, fit_b, tol=0.01, handle=aux, return_stats=True)
        hd = eu.hausdorff_distance(fit_a, fit_b, dx_min=5, handle=aux)
        res = {'tol': 0.01, 'lower01': r.lower01, 'upper01': r.upper01, 'lower10': r.lower10, 'upper10': r.upper10,
               'converged': r.converged,
               'witness01': [r.witness01[0].tolist(), r.witness01[1], r.witness01[2]],
               'witness10': [r.witness10[0].tolist(), r.witness10[1], r.witness10[2]],
               'stats_keys': ['levels', 'entries_bounded', 'point_walks', 'faces_skipped', 'converged'],
               'stats01': [int(x) for x in s01], 'stats10': [int(x) for x in s10],
               'hausdorff_distance_dx5': {'h01': hd.h01, 'h10': hd.h10},
               'upper01_ge_6.21': r.upper01 >= 6.21, 'upper10_ge_71.17': r.upper10 >= 71.17,
               'sampled_le_upper': hd.h01 <= r.upper01 and hd.h10 <= r.upper10}
        res['times'] = timed_alternating({
            'hausdorff_bounds_tol0.01': lambda: eu.hausdorff_bounds(fit_a, fit_b, tol=0.01, handle=aux),
            'hausdorff_distance_dx5': lambda: eu.hausdorff_distance(fit_a, fit_b, dx_min=5, handle=aux)}, reps)
    finally:
        aux.close()
    return res


def mean_bounds_legs(fit_a, fit_b, reps):
    """mean_distance_bounds(fit_a, fit_b, tol=0.01) against hausdorff_distance(dx_min=5) and average_squared_distance of
    points_from_mesh samples, alternating; the first two on one auxiliary handle."""
    aux = eu._lib.Handle(0)

    def sampled():
        return eu.average_squared_distance(eu.points_from_mesh(fit_a, dx_min=5), eu.points_from_mesh(fit_b, dx_min=5))
    try:
        r, s01, s10 = eu.mean_distance_bounds(fit_a, fit_b, tol=0.01, handle=aux, return_stats=True)
        hd = eu.hausdorff_distance(fit_a, fit_b, dx_min=5, handle=aux)
        np.random.seed(0)
        asd = sampled()
        res = dict(r._asdict(), tol=0.01, max_queries=eu.HAUSDORFF_MAX_QUERIES,
                   stats_keys=['levels', 'entries_bounded', 'point_walks', 'candidate_faces', 'faces_nonfinite', 'faces_zero_area',
                               'converged'],
                   stats01=[int(x) for x in s01], stats10=[int(x) for x in s10],
                   hausdorff_distance_dx5={'mean01': hd.mean01, 'mean10': hd.mean10},
                   average_squared_distance_dx5=[float(x) for x in np.ravel(asd)])
        res['times'] = timed_alternating({
            'mean_distance_bounds_tol0.01': lambda: eu.mean_distance_bounds(fit_a, fit_b, tol=0.01, handle=aux),
            'hausdorff_distance_dx5': lambda: eu.hausdorff_distance(fit_a, fit_b, dx_min=5, handle=aux),
            'points_from_mesh_dx5_average_squared_distance': sampled}, reps)
    finally:
        aux.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=10)
    ap.add_argument('--signed', action='store_true')
    ap.add_argument('--bounds', action='store_true')
    ap.add_argument('--mean-bounds', action='store_true')
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
    if args.signed:
        res['signed'] = signed_legs(h, fit_b, P, args.reps)
    if args.bounds:
        res['bounds'] = bounds_legs(fit_a, fit_b, args.reps)
    if args.mean_bounds:
        res['mean_bounds'] = mean_bounds_legs(fit_a, fit_b, args.reps)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()

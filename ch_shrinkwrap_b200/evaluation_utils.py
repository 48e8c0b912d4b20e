"""GPU versions of the reference's mesh-quality helpers (``ch_shrinkwrap/evaluation_utils.py:35-180``), same names,
arguments and return values:

* ``points_from_mesh(mesh, dx_min=5, p=1.0, return_normals=False)`` -- the per-triangle Python loop becomes one kernel
  (``nw_points_from_mesh``); the samples are bit-identical to the reference's ``d`` array.  The reference returns them in a
  random order (``np.random.choice`` without replacement, :137); here the order is random too, drawn from
  ``np.random`` exactly like the reference, so seeding ``np.random`` gives the same permutation for the same count.
* ``average_squared_distance(points0, points1)`` -- the two ``cKDTree`` builds + queries become two nearest-point
  searches in the solver's hierarchy (``nw_set_point_targets``); distances are the same float64 numbers.
* ``nearest_point_distance(targets, queries)`` -- the building block, also used by the hole-punch candidate search.

Not in the reference (its surface metrics compare sample clouds, so their answer depends on ``dx_min``):

* ``surface_distance(mesh, points)`` -- exact distance from each point to the closed triangles of a mesh
  (``nw_surface_distance``).
* ``surface_distance(mesh, points, signed=True)`` -- the same distance, negative inside a closed mesh and positive outside
  (``nw_surface_signed_distance``: the angle-weighted pseudonormal of the nearest feature, oriented by the signed volume).
* ``enclosed_volume(mesh)`` -- the volume a closed mesh encloses.
* ``self_intersections(mesh)`` -- the pairs of faces that cross or touch beyond their shared vertices and edges, exactly
  (``nw_self_intersections``); none means the mesh is embedded, which the two calls above assume.
* ``hausdorff_distance(mesh0, mesh1, dx_min)`` -- one-sided and symmetric Hausdorff and mean distances between two meshes,
  from exact point-to-surface distances of each mesh's samples.
* ``hausdorff_bounds(mesh0, mesh1, tol)`` -- certified bounds of the one-sided and symmetric Hausdorff distances, with the
  points that attain the lower bounds (``nw_hausdorff_bounds``).
* ``mean_distance_bounds(mesh0, mesh1, tol)`` -- certified bounds of the area-weighted mean and RMS distances between two
  meshes, both ways (``nw_mean_distance_bounds``): the continuous counterpart of ``average_squared_distance``.

No CPU fallback: these raise if libnanowrap.so or the GPU is missing.
"""
from __future__ import annotations

import ctypes
from collections import namedtuple

import numpy as np

from . import _lib


def _xyz(a):
    a = np.asarray(a)
    if a.ndim != 2 or a.shape[1] != 3:
        raise ValueError('expected an (N,3) array')
    if a.dtype == np.float32:
        return np.ascontiguousarray(a), 0
    return np.ascontiguousarray(a, dtype=np.float64), 1


def nearest_point_distance(targets, queries, handle=None, return_index=False):
    """``scipy.spatial.cKDTree(targets).query(queries, k=1)``: float64 distances (and indices) of the nearest target."""
    t, t64 = _xyz(targets)
    q, q64 = _xyz(queries)
    h = handle if handle is not None else _lib.Handle(0)
    try:
        dist = np.empty(len(q), np.float64)
        idx = np.empty(len(q), np.int32)
        if len(q) == 0:
            return (dist, idx) if return_index else dist
        if len(t) == 0:
            raise ValueError('no target points')
        h.call('nw_set_point_targets', ctypes.c_void_p(t.ctypes.data), t64, len(t))
        h.call('nw_set_points', ctypes.c_void_p(q.ctypes.data), q64, len(q), None, 1.0, None)
        h.call('nw_compute_weights')
        h.call('nw_get_weights', None, None, _lib.dptr(dist), _lib.iptr(idx))
    finally:
        if handle is None:
            h.close()
    return (dist, idx) if return_index else dist


def average_squared_distance(points0, points1, handle=None):
    """evaluation_utils.py:147-180: (mean squared distance of points1 to their nearest points0, and the converse)."""
    points0_err = nearest_point_distance(points0, points1, handle)          # :175
    points1_err = nearest_point_distance(points1, points0, handle)          # :176
    points0_mse = np.nansum(points0_err ** 2) / len(points0_err)            # :178
    points1_mse = np.nansum(points1_err ** 2) / len(points1_err)            # :179
    return points0_mse, points1_mse


def mesh_samples(mesh, dx_min=5, handle=None):
    """The reference's ``d`` array (evaluation_utils.py:59-135) before its random permutation: (n,3) float64."""
    pos = _lib.as_f32(mesh._vertices['position'])
    faces = np.ascontiguousarray(mesh.faces, dtype=np.int32)
    h = handle if handle is not None else _lib.Handle(0)
    try:
        n = ctypes.c_int64(0)
        h.call('nw_points_from_mesh', _lib.fptr(pos), _lib.iptr(faces), len(pos), len(faces), float(dx_min), None, 0, ctypes.byref(n))
        d = np.empty((n.value, 3), np.float64)
        if n.value:
            h.call('nw_points_from_mesh', _lib.fptr(pos), _lib.iptr(faces), len(pos), len(faces), float(dx_min), _lib.dptr(d), n.value,
                   ctypes.byref(n))
    finally:
        if handle is None:
            h.close()
    return d


def _surface_call(h, queries, n_resident=0, want_dist=True, want_face=False, want_closest=False, want_summary=False,
                  signed=False):
    """nw_surface_distance, or with ``signed`` nw_surface_signed_distance, on handle `h`: queries None = the handle's
    `n_resident` resident points, else an (N,3) array.  Returns (dist, face, closest, extra), None for what was not asked
    for; extra is the summary (max, mean, RMS) of the unsigned call (``want_summary``), the enclosed volume of the signed
    one.  A signed call with a length-0 ``queries`` checks the mesh and measures its volume only."""
    if queries is None:
        q, q64, Q = None, 0, int(n_resident)
    else:
        q, q64 = _xyz(queries)
        Q = len(q)
        if Q == 0:
            q = np.zeros((1, 3), q.dtype)              # q must not be NULL: that would mean the resident points
    qp = None if q is None else ctypes.c_void_p(q.ctypes.data)
    dist = np.empty(Q, np.float64) if want_dist else None
    face = np.empty(Q, np.int32) if want_face else None
    closest = np.empty((Q, 3), np.float64) if want_closest else None
    if signed:
        volume = ctypes.c_double(0.0)
        h.call('nw_surface_signed_distance', qp, q64, Q, _lib.dptr(dist), _lib.iptr(face), _lib.dptr(closest),
               ctypes.byref(volume))
        return dist, face, closest, volume.value
    summary = np.empty(3, np.float64) if want_summary else None
    h.call('nw_surface_distance', qp, q64, Q, _lib.dptr(dist), _lib.iptr(face), _lib.dptr(closest), _lib.dptr(summary))
    return dist, face, closest, summary


def _signed_call(h, queries, n_resident=0, want_dist=True, want_face=False, want_closest=False):
    """``_surface_call(..., signed=True)``: (sdist, face, closest, volume)."""
    return _surface_call(h, queries, n_resident, want_dist, want_face, want_closest, signed=True)


def _surface_distances(h, queries, n_resident, signed, return_face, return_closest):
    """The return value of the ``surface_distance`` methods: dist, or (dist[, face][, closest])."""
    dist, face, closest, _ = _surface_call(h, queries, n_resident, True, return_face, return_closest, signed=signed)
    if not (return_face or return_closest):
        return dist
    return (dist,) + ((face,) if return_face else ()) + ((closest,) if return_closest else ())


def _upload_surface(h, mesh):
    """The mesh as the handle's topology (vertex positions as float32, faces = rows of ``mesh.faces``).  Normals and neighbour
    tables do not enter the distance; a mesh without them gets zeros and -1 tables."""
    pos = _lib.as_f32(mesh._vertices['position'])
    faces = np.ascontiguousarray(mesh.faces, dtype=np.int32)
    if len(pos) == 0 or len(faces) == 0:
        raise ValueError('the mesh has no vertices or no faces')
    nrm = getattr(mesh, 'vertex_normals', None)
    nrm = np.zeros_like(pos) if nrm is None else _lib.as_f32(nrm)
    nbr = np.full((len(pos), 20), -1, np.int32)
    if 'neighbors' in (mesh._vertices.dtype.names or ()) and hasattr(mesh, '_halfedges'):
        nb = np.asarray(mesh._vertices['neighbors'])
        nbr = np.where(nb >= 0, np.asarray(mesh._halfedges['vertex'])[np.maximum(nb, 0)], -1).astype(np.int32)
    h.call('nw_set_topology', _lib.fptr(pos), _lib.fptr(nrm), _lib.iptr(faces), _lib.iptr(nbr), None, len(pos), len(faces))


def surface_distance(mesh, points, handle=None, return_face=False, return_closest=False, signed=False):
    """Exact Euclidean distance from each point to the closed triangles of `mesh` (float64, the points' order).

    ``signed=True``: negative inside the solid the mesh bounds, positive outside, 0 on the surface; NaN where the side is
    undecidable (the offset from the closest point is orthogonal to the pseudonormal there).  The magnitude, face and closest
    point are those of the unsigned call.  The side comes from the angle-weighted pseudonormal of the nearest face, edge or
    vertex, and "inside" from the sign of the mesh's signed volume, so either winding gives the same answer.  The mesh must
    be closed, edge-manifold and consistently oriented (ValueError with the defect counts otherwise); a mesh whose separate
    components are oriented against each other is not supported.  It must also be embedded: on a mesh whose faces cross or
    fold over each other the signs are meaningless, and no check here sees that; ``self_intersections`` does.

    ``return_face``: also the row of ``mesh.faces`` of the nearest triangle (int32; exact fp64 ties go to the lowest row);
    ``return_closest``: also the closest point on it ((N,3) float64).  Float32 points are used exactly, float64 points as
    given.  A non-finite point gets NaN, face -1; faces with a non-finite corner are ignored.  Unlike the solver's nearest
    face, which is the nearest face CENTROID (mesh_conj_grad.py:451-454), this is the distance to the surface itself."""
    h = handle if handle is not None else _lib.Handle(0)
    try:
        _upload_surface(h, mesh)
        return _surface_distances(h, points, 0, signed, return_face, return_closest)
    finally:
        if handle is None:
            h.close()


def enclosed_volume(mesh, handle=None):
    """The volume enclosed by a closed, edge-manifold, consistently oriented mesh (float64, either winding): the absolute
    value of the signed volume sum_f dot(a - o, (b - o) x (c - o)) / 6 over the faces (a, b, c), reduced on the GPU in a
    fixed order.  Raises ValueError for a mesh that does not bound a solid, as ``surface_distance(signed=True)`` does.  A
    self-intersecting mesh passes those checks and gets a meaningless volume; ``self_intersections`` is the check."""
    h = handle if handle is not None else _lib.Handle(0)
    try:
        _upload_surface(h, mesh)
        return _signed_call(h, np.zeros((0, 3), np.float32), want_dist=False)[3]
    finally:
        if handle is None:
            h.close()


IntersectionStats = namedtuple('IntersectionStats', 'candidates exact degenerate non_finite')


def _self_intersections(h, return_stats=False, capacity=1024):
    """nw_self_intersections on handle `h`: (n, 2) int32 face-row pairs f < g sorted by (f, g)[, IntersectionStats].  Calls
    again with the exact capacity only when the first guess was too small."""
    n = ctypes.c_int64(0)
    stats = np.zeros(4, np.int64)
    sp = stats.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))
    pairs = np.empty((capacity, 2), np.int32)
    h.call('nw_self_intersections', _lib.iptr(pairs), capacity, ctypes.byref(n), sp)
    if n.value > capacity:
        pairs = np.empty((n.value, 2), np.int32)
        h.call('nw_self_intersections', _lib.iptr(pairs), n.value, ctypes.byref(n), sp)
    pairs = np.ascontiguousarray(pairs[:n.value])
    return (pairs, IntersectionStats(*(int(x) for x in stats))) if return_stats else pairs


def self_intersections(mesh, handle=None, return_stats=False):
    """The pairs of faces of `mesh` that intersect: an (n, 2) int32 array of rows of ``mesh.faces``, f < g, sorted by (f, g).

    Two faces intersect when their closed triangles share a point that their shared vertex indices do not explain: faces with
    no common vertex must not touch at all; faces sharing one vertex must meet only there; faces sharing an edge are reported
    when they are coplanar and fold over each other; faces with the same three vertices always.  Degenerate faces (collinear
    corners, a repeated vertex included) and faces with a non-finite corner are not tested.  The answer is exact for the
    float32 positions (every decision is the exactly evaluated sign of an orientation determinant), so it does not depend on
    the winding, the order of the faces or a power-of-two scale.  The mesh need not be closed or manifold.

    ``return_stats``: also an ``IntersectionStats(candidates, exact, degenerate, non_finite)``: the face pairs whose boxes
    overlapped, the orientation signs that needed the exact stage, and the faces left out.  An empty result means the mesh is
    embedded, which ``surface_distance(signed=True)`` and ``enclosed_volume`` assume."""
    h = handle if handle is not None else _lib.Handle(0)
    try:
        _upload_surface(h, mesh)
        return _self_intersections(h, return_stats)
    finally:
        if handle is None:
            h.close()


HausdorffResult = namedtuple('HausdorffResult', 'h01 h10 hausdorff mean01 mean10')


def _surface_samples(mesh, dx_min, h):
    pos = np.asarray(mesh._vertices['position'], np.float64)
    if 'halfedge' in (mesh._vertices.dtype.names or ()):
        pos = pos[mesh._vertices['halfedge'] != -1]                # a deleted vertex keeps its row
    return np.concatenate([pos, mesh_samples(mesh, dx_min, h)], 0)


def hausdorff_distance(mesh0, mesh1, dx_min=5, handle=None):
    """Distances between two triangle meshes, both ways.

    The samples of a mesh are its vertices plus ``mesh_samples(mesh, dx_min)`` (every triangle sampled on a dx_min grid in
    its own plane).  ``h01`` is the largest exact distance from a sample of mesh0 to the surface of mesh1, ``mean01`` the
    mean of those distances; ``h10`` and ``mean10`` the same the other way; ``hausdorff = max(h01, h10)``.

    Each one-sided value is exact on its sample set, so it is a lower bound of the continuous one-sided Hausdorff distance
    (the supremum over the whole surface) and converges to it as ``dx_min -> 0``; ``hausdorff_bounds`` brackets the
    continuous value itself.  ``mean01`` and ``mean10`` weight every sample alike, not by area, and their error depends on
    ``dx_min``; ``mean_distance_bounds`` brackets the area-weighted mean and RMS distances.  The reductions run on the GPU in a fixed
    order: repeated calls give identical numbers, and swapping the meshes swaps h01 / h10 and mean01 / mean10 exactly.
    Returns a ``HausdorffResult(h01, h10, hausdorff, mean01, mean10)``."""
    h = handle if handle is not None else _lib.Handle(0)
    try:
        s0, s1 = _surface_samples(mesh0, dx_min, h), _surface_samples(mesh1, dx_min, h)
        _upload_surface(h, mesh1)
        r01 = _surface_call(h, s0, want_dist=False, want_summary=True)[3]
        _upload_surface(h, mesh0)
        r10 = _surface_call(h, s1, want_dist=False, want_summary=True)[3]
    finally:
        if handle is None:
            h.close()
    return HausdorffResult(float(r01[0]), float(r10[0]), max(float(r01[0]), float(r10[0])), float(r01[1]), float(r10[1]))


HausdorffBounds = namedtuple('HausdorffBounds', 'lower01 upper01 lower10 upper10 lower upper converged witness01 witness10')
HAUSDORFF_MAX_QUERIES = 1 << 25


def _hausdorff_bounds(h, mesh, tol, max_queries):
    """nw_hausdorff_bounds from `mesh` to the handle's mesh: (lower, upper, witness, stats)."""
    pos = _lib.as_f32(mesh._vertices['position'])
    faces = np.ascontiguousarray(mesh.faces, dtype=np.int32)
    bounds, point, wf, stats = np.zeros(2), np.zeros(3), np.zeros(2, np.int32), np.zeros(5, np.int64)
    h.call('nw_hausdorff_bounds', _lib.fptr(pos), len(pos), _lib.iptr(faces), len(faces), float(tol), int(max_queries),
           _lib.dptr(bounds), _lib.dptr(point), _lib.iptr(wf), stats.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)))
    return float(bounds[0]), float(bounds[1]), (point, int(wf[0]), int(wf[1])), stats


def hausdorff_bounds(mesh0, mesh1, tol=0.01, max_queries=HAUSDORFF_MAX_QUERIES, handle=None, return_stats=False):
    """Certified bounds of the Hausdorff distances between two triangle meshes, both ways.

    h01 = max over the points p of mesh0's closed triangles of the exact distance from p to mesh1's closed triangles (the
    quantity ``surface_distance`` measures), h10 the same the other way.  ``lower01 - eps <= h01 <= upper01``, eps = 2^-40 x
    the sum over the axes of the largest |coordinate| of both meshes' used vertices (about 1e-9 nm for a micrometre-sized
    cell); likewise for h10, and ``lower = max(lower01, lower10)``, ``upper = max(upper01, upper10)`` bracket the symmetric
    distance.  Each lower bound is attained: ``witness01 = (point (3,) float64, face row of mesh0 it lies on, its nearest
    face row of mesh1)``, and ``surface_distance(mesh1, point[None])`` is ``lower01`` bit for bit; likewise ``witness10``.

    A branch and bound over the triangles on the GPU: bounds from the convexity of the distance to single faces and from
    its 1-Lipschitz continuity, triangles split at their edge midpoints until every bound is within ``tol`` (mesh units) of
    the lower bound (``converged``: ``upper - lower <= tol`` both ways) or until the next level would take more than
    ``max_queries`` point walks in one direction (``converged`` False; the bounds are still valid).  Faces with a non-finite
    corner are skipped.  Repeated calls give identical numbers, and swapping the meshes swaps the 01 and 10 fields.
    ``return_stats``: also the two stats arrays (levels, triangles bounded, point walks, faces skipped, converged) of
    ``nw_hausdorff_bounds``.  ValueError for a mesh with no finite face, a face index out of range or ``tol < 0``."""
    h = handle if handle is not None else _lib.Handle(0)
    try:
        _upload_surface(h, mesh1)
        lo01, up01, w01, st01 = _hausdorff_bounds(h, mesh0, tol, max_queries)
        _upload_surface(h, mesh0)
        lo10, up10, w10, st10 = _hausdorff_bounds(h, mesh1, tol, max_queries)
    finally:
        if handle is None:
            h.close()
    r = HausdorffBounds(lo01, up01, lo10, up10, max(lo01, lo10), max(up01, up10), bool(st01[4] and st10[4]), w01, w10)
    return (r, st01, st10) if return_stats else r


MeanDistanceBounds = namedtuple('MeanDistanceBounds', 'mean01_lower mean01_upper rms01_lower rms01_upper mean10_lower '
                                                     'mean10_upper rms10_lower rms10_upper area0 area1 converged')


def _mean_distance_bounds(h, mesh, tol, max_queries):
    """nw_mean_distance_bounds from `mesh` to the handle's mesh: (out (5,) float64, stats (7,) int64)."""
    pos = _lib.as_f32(mesh._vertices['position'])
    faces = np.ascontiguousarray(mesh.faces, dtype=np.int32)
    out, stats = np.zeros(5), np.zeros(7, np.int64)
    h.call('nw_mean_distance_bounds', _lib.fptr(pos), len(pos), _lib.iptr(faces), len(faces), float(tol), int(max_queries),
           _lib.dptr(out), stats.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)))
    return out, stats


def mean_distance_bounds(mesh0, mesh1, tol=0.01, max_queries=HAUSDORFF_MAX_QUERIES, handle=None, return_stats=False):
    """Certified bounds of the area-weighted mean and RMS distances between two triangle meshes, both ways.

    mean01 = (1/|A|) x the integral over mesh0's finite faces A of d_1, the exact distance to mesh1's closed triangles (the
    quantity ``surface_distance`` measures), and rms01 = sqrt((1/|A|) x the integral of d_1^2): the continuous counterparts
    of the reference's ``average_squared_distance`` of two sample clouds, independent of any sampling step.  mean10 and
    rms10 the same the other way.  ``mean01_lower - eps <= mean01 <= mean01_upper + eps`` and likewise for the other three,
    eps = 2^-40 x the sum over the axes of the largest |coordinate| of both meshes' used vertices; ``area0`` and ``area1``
    are the total areas of the finite faces.

    The same branch and bound over the triangles as ``hausdorff_bounds``: each triangle's integrals are bracketed from above
    by the convexity of the distance to single faces and from below by concavity and by support planes of every face of the
    other mesh that can be nearest on it, so a triangle lying over the inside of one face is settled without a split.
    ``converged`` when both gaps are at most ``tol`` (mesh units) both ways; a call that would pass ``max_queries`` point walks
    in one direction stops early with valid, wider brackets.  Faces with a non-finite corner are skipped and counted, faces
    of zero area counted.  Repeated calls give identical numbers, and swapping the meshes swaps the 01 and 10 fields.
    ``return_stats``: also the two stats arrays (levels, triangles bounded, point walks, candidate faces evaluated, faces
    skipped as non-finite, zero-area faces, converged) of ``nw_mean_distance_bounds``.  ValueError for a mesh with no finite
    face or zero total area, a face index out of range, ``tol < 0`` or too small a ``max_queries``."""
    h = handle if handle is not None else _lib.Handle(0)
    try:
        _upload_surface(h, mesh1)
        o01, st01 = _mean_distance_bounds(h, mesh0, tol, max_queries)
        _upload_surface(h, mesh0)
        o10, st10 = _mean_distance_bounds(h, mesh1, tol, max_queries)
    finally:
        if handle is None:
            h.close()
    r = MeanDistanceBounds(*(float(x) for x in o01[1:]), *(float(x) for x in o10[1:]), float(o01[0]), float(o10[0]),
                           bool(st01[6] and st10[6]))
    return (r, st01, st10) if return_stats else r


def points_from_mesh(mesh, dx_min=5, p=1.0, return_normals=False):
    """evaluation_utils.py:35-145."""
    h = _lib.Handle(0)
    try:
        d = mesh_samples(mesh, dx_min, h)
        subsamp = np.random.choice(np.arange(d.shape[0]), size=int(p * d.shape[0]), replace=False)      # :137
        if return_normals:
            # nearest face centroid of every sample (:143-149): the solver's own nearest-face search with the samples as points
            face_centers = mesh._vertices['position'][mesh.faces].mean(1)
            _, faces = nearest_point_distance(face_centers, d, h, return_index=True)
            normals = mesh._faces['normal'][mesh._faces['halfedge'] != -1][faces]
            return d[subsamp], normals[subsamp]
        return d[subsamp]
    finally:
        h.close()

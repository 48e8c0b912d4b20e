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
    (the supremum over the whole surface) and converges to it as ``dx_min -> 0``.  The reductions run on the GPU in a fixed
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

"""nw_surface_distance (exact point-to-surface distance) and the Hausdorff metric on the GPU.

Distances, closest points and faces are compared bit for bit with the numpy restatement
(tests/surface_oracle.py: surface_nearest), ties included."""
import ctypes
import os
import sys

import numpy as np
import pytest

from ch_shrinkwrap_b200 import _lib, minimesh, synth
from ch_shrinkwrap_b200 import evaluation_utils as eu
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import surface_oracle as orc  # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def lobed():
    """Two-lobed star mesh: 16 002 vertices, 32 000 faces, and a localisation cloud on the shape."""
    shape = synth.two_lobed()
    mesh = synth.star_mesh(shape, 40)
    pts, sig = synth.smlm_cloud(shape, 4000, seed=11)
    return mesh, pts, sig


def mixed_queries(mesh, pts, seed=0):
    """The cloud, far points, the mesh's own vertices and edge midpoints (float32)."""
    rng = np.random.default_rng(seed)
    v, f = mesh._vertices['position'], mesh.faces
    far = rng.normal(0.0, 1.0, (300, 3))
    far *= (rng.uniform(2e3, 2e4, 300) / np.sqrt((far * far).sum(1)))[:, None]
    mids = (v[f[:, 0]] + v[f[:, 1]]) * np.float32(0.5)
    mids = mids[rng.choice(len(mids), 4000, replace=False)]
    return np.concatenate([pts, far.astype(np.float32), v, mids]).astype(np.float32)


def assert_matches_oracle(mesh, q):
    d, f, c = eu.surface_distance(mesh, q, return_face=True, return_closest=True)
    od, of, oc = orc.surface_nearest(q, mesh._vertices['position'], mesh.faces)
    assert np.array_equal(f, of), 'faces differ at %s' % np.flatnonzero(f != of)[:10]
    assert np.array_equal(d, od), 'distances differ at %s' % np.flatnonzero(d != od)[:10]
    assert np.array_equal(c, oc)
    return d


@pytest.mark.parametrize('dtype', [np.float32, np.float64])
def test_bit_identical_to_oracle(lobed, dtype):
    mesh, pts, _ = lobed
    q = mixed_queries(mesh, pts)
    if dtype == np.float64:        # values a float32 cannot hold
        q = q.astype(np.float64) + np.random.default_rng(1).normal(0.0, 1e-3, q.shape)
    d = assert_matches_oracle(mesh, q)
    nv = len(mesh._vertices)
    if dtype == np.float32:
        assert np.all(d[len(pts) + 300:len(pts) + 300 + nv] == 0.0)       # a vertex lies on the surface


def _resident_handle(mesh, pts):
    h = _lib.Handle(0)
    eu._upload_surface(h, mesh)
    h.call('nw_set_points', ctypes.c_void_p(pts.ctypes.data), int(pts.dtype == np.float64), len(pts), None, 1.0, None)
    return h


@pytest.mark.parametrize('dtype', [np.float32, np.float64])
def test_resident_points_equal_explicit_points(lobed, dtype):
    mesh, pts, _ = lobed
    pts = np.ascontiguousarray(pts, dtype=dtype)
    if dtype == np.float64:
        pts = pts + np.random.default_rng(2).normal(0.0, 1e-3, pts.shape)
    h = _resident_handle(mesh, pts)
    try:
        explicit = eu._surface_call(h, pts, 0, True, True, True, True)
        cold = eu._surface_call(h, None, len(pts), True, True, True, True)       # no seeds yet: greedy descent
        h.call('nw_compute_weights')                                           # nearest-centroid slots become the seeds
        warm = eu._surface_call(h, None, len(pts), True, True, True, True)
    finally:
        h.close()
    for r in (cold, warm):
        for a, b in zip(r, explicit):
            assert np.array_equal(a, b)
    od, of, _ = orc.surface_nearest(pts, mesh._vertices['position'], mesh.faces)
    assert np.array_equal(explicit[0], od) and np.array_equal(explicit[1], of)
    d = explicit[0]
    assert explicit[3][0] == d.max()
    np.testing.assert_allclose(explicit[3][1:], [d.mean(), np.sqrt((d * d).mean())], rtol=1e-12)


def _fit(mesh, pts, sig, probe):
    """Two nw_search calls of 4 iterations on a fresh handle; with `probe`, nw_surface_distance runs between them."""
    h = _lib.Handle(0)
    try:
        eu._upload_surface(h, mesh)
        s_inv = np.ascontiguousarray(1.0 / sig, dtype=np.float32)
        h.call('nw_set_points', ctypes.c_void_p(pts.ctypes.data), 0, len(pts), _lib.fptr(s_inv), 1.0, None)
        out, hists = [], []
        for k in range(2):
            pos = np.empty((len(mesh._vertices), 3), np.float32)
            hist = [np.zeros(4) for _ in range(5)]
            n = ctypes.c_int(0)
            prev = np.concatenate([x[0] for x in hists]) if hists else np.zeros(0)
            h.call('nw_search', 10.0, 4, 1, _lib.dptr(prev) if len(prev) else None, len(prev), _lib.fptr(pos),
                   *[_lib.dptr(a) for a in hist], ctypes.byref(n))
            out.append(pos)
            hists.append(hist)
            if probe and k == 0:
                eu._surface_call(h, None, len(pts), True, True, True, True)
                eu._surface_call(h, pts[::7] * np.float32(3.0), 0, True, True, True, True)
        return out, hists
    finally:
        h.close()


def test_no_side_effects_on_the_fit(lobed):
    mesh, pts, sig = lobed
    a_pos, a_hist = _fit(mesh, pts, sig, probe=False)
    b_pos, b_hist = _fit(mesh, pts, sig, probe=True)
    for x, y in zip(a_pos, b_pos):
        assert np.array_equal(x, y)
    for x, y in zip(a_hist, b_hist):
        for u, v in zip(x, y):
            assert np.array_equal(u, v)


@pytest.mark.parametrize('dtype', [np.float32, np.float64])
def test_far_queries_take_their_slack_from_the_queries(lobed, dtype):
    mesh, pts, _ = lobed
    rng = np.random.default_rng(4)
    u = rng.normal(0.0, 1.0, (2000, 3))
    u /= np.sqrt((u * u).sum(1))[:, None]
    q = (u * rng.uniform(4e5, 6e5, 2000)[:, None] + rng.normal(0.0, 1.0, u.shape)).astype(dtype)   # ~1000x the mesh's size
    d = assert_matches_oracle(mesh, q)
    assert d.min() > 3e5


def test_hausdorff_parallel_planes_are_exactly_d_apart():
    m0 = minimesh.planar_mesh(100.0, 20)
    v = m0._vertices['position'].copy()
    v[:, 2] += np.float32(0.5)
    m1 = minimesh.MiniMesh(v, m0.faces)
    r = eu.hausdorff_distance(m0, m1, dx_min=3.0)
    assert r == (0.5, 0.5, 0.5, 0.5, 0.5)


def test_hausdorff_of_a_mesh_with_itself_is_zero():
    m = minimesh.sphere_mesh(500.0, 16)
    assert np.all(eu.surface_distance(m, m._vertices['position']) == 0.0)
    # the in-plane samples are built on float32 triangle frames (mesh_samples, as the reference does), so they lie off their
    # own triangle by float32 rounding of the coordinates: ~1e-7 of the radius
    r = eu.hausdorff_distance(m, m, dx_min=10.0)
    assert r.h01 == r.h10 and r.hausdorff <= 1e-6 * 500.0 and r.mean01 <= 1e-7 * 500.0


def _max_circumradius(mesh):
    v = mesh._vertices['position'].astype(np.float64)[mesh.faces]
    a, b, c = (np.sqrt(((v[:, i] - v[:, j]) ** 2).sum(1)) for i, j in ((0, 1), (1, 2), (2, 0)))
    area = 0.5 * np.sqrt((np.cross(v[:, 1] - v[:, 0], v[:, 2] - v[:, 0]) ** 2).sum(1))
    return float((a * b * c / (4.0 * area)).max())


def test_hausdorff_of_concentric_spheres_is_within_the_sagitta_bound():
    r0, r1 = 500.0, 530.0
    m0, m1 = minimesh.sphere_mesh(r0, 12), minimesh.sphere_mesh(r1, 16)
    # each inscribed polyhedron lies between its sphere and the sphere through its face planes: radius sqrt(R^2 - rc^2)
    s0 = r0 - np.sqrt(r0 ** 2 - _max_circumradius(m0) ** 2)
    s1 = r1 - np.sqrt(r1 ** 2 - _max_circumradius(m1) ** 2)
    r = eu.hausdorff_distance(m0, m1, dx_min=10.0)
    for x in (r.h01, r.h10, r.mean01, r.mean10):
        assert (r1 - r0) - s1 - 1e-3 <= x <= (r1 - r0) + s0 + 1e-3, (x, s0, s1)


def test_hausdorff_is_symmetric_and_repeatable(lobed):
    m0 = minimesh.sphere_mesh(450.0, 20)
    m1 = lobed[0]
    r, s = eu.hausdorff_distance(m0, m1, dx_min=15.0), eu.hausdorff_distance(m1, m0, dx_min=15.0)
    assert (r.h01, r.h10, r.mean01, r.mean10, r.hausdorff) == (s.h10, s.h01, s.mean10, s.mean01, s.hausdorff)
    assert eu.hausdorff_distance(m0, m1, dx_min=15.0) == r


def test_c3_mesh_with_a_million_queries_matches_the_oracle_on_a_sample():
    """The bench's C3 mesh (501 762 vertices, two-lobed) and 10^6 localisations on it."""
    v, f = minimesh.geodesic_sphere(224)
    v, f = minimesh.spatially_sorted(v, f)
    r = synth.radial_surface(synth.two_lobed(), v, n_bisect=32)
    mesh = minimesh.MiniMesh(v * (1.2 * r)[:, None], f)
    assert len(mesh._vertices) == 501762
    pts, _ = synth.mesh_surface_cloud(v * r[:, None], f, 1_000_000, seed=3)
    d, face = eu.surface_distance(mesh, pts, return_face=True)
    pick = np.random.default_rng(0).choice(len(pts), 400, replace=False)
    od, of, _ = orc.surface_nearest(pts[pick], mesh._vertices['position'], mesh.faces)
    assert np.array_equal(d[pick], od) and np.array_equal(face[pick], of)
    assert np.all(np.isfinite(d)) and np.all(face >= 0)


def test_point_surface_distance_after_a_fit_measures_the_fitted_surface():
    """MembraneMesh.point_surface_distance(): the fit's resident localisations against the fitted mesh on the fit's handle."""
    from ch_shrinkwrap_b200.membrane_mesh import MembraneMesh
    from ch_shrinkwrap_b200.mesh_conj_grad import ShrinkwrapMeshConjGrad
    shape = synth.Sphere(500.0)
    pts, sig = synth.smlm_cloud(shape, 20000, seed=7)
    mesh = MembraneMesh(mesh=synth.star_mesh(shape, 8, scale=1.2), kc=1.0, step_size=20.0)
    mesh.cg = ShrinkwrapMeshConjGrad(mesh, pts)
    mesh.cg.search(pts, lams=[10.0], num_iters=5, sigma_inv=(1.0 / sig.ravel()).astype(np.float32))
    d, face = mesh.point_surface_distance(return_face=True)
    fitted = minimesh.MiniMesh(mesh._vertices['position'].copy(), mesh.faces)
    od, of = eu.surface_distance(fitted, pts, return_face=True)
    assert np.array_equal(d, od) and np.array_equal(face, of)
    assert np.array_equal(mesh.point_surface_distance(pts[:100]), od[:100])

"""nw_surface_signed_distance (signed point-to-surface distance and enclosed volume) on the GPU.

Magnitudes, faces and closest points are compared bit for bit with nw_surface_distance; the side with the numpy restatement
(tests/signed_oracle.py) wherever that is not within rounding of undecidable, and with the generalised winding number."""
import ctypes
import os
import re
import sys

import numpy as np
import pytest

from ch_shrinkwrap_b200 import _lib, minimesh, synth
from ch_shrinkwrap_b200 import evaluation_utils as eu
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import signed_oracle as so  # noqa: E402
import surface_oracle as orc  # noqa: E402

pytestmark = pytest.mark.gpu
MARGIN = 1e-9


class Raw:
    """Just what _upload_surface reads: positions and face rows (no neighbour tables, so any face list goes up)."""

    def __init__(self, v, f):
        self._vertices = np.zeros(len(v), [('position', np.float32, 3)])
        self._vertices['position'] = v
        self.faces = np.ascontiguousarray(f, np.int32)


@pytest.fixture(scope='module')
def lobed():
    shape = synth.two_lobed()
    mesh = synth.star_mesh(shape, 40)
    pts, sig = synth.smlm_cloud(shape, 4000, seed=11)
    return mesh, pts, sig


def mixed_queries(mesh, pts, seed=0):
    """The cloud, far points, the mesh's own vertices and edge midpoints, and points just off the vertices (float32)."""
    rng = np.random.default_rng(seed)
    v, f = mesh._vertices['position'], mesh.faces
    far = rng.normal(0.0, 1.0, (300, 3))
    far *= (rng.uniform(2e3, 2e4, 300) / np.sqrt((far * far).sum(1)))[:, None]
    mids = (v[f[:, 0]] + v[f[:, 1]]) * np.float32(0.5)
    mids = mids[rng.choice(len(mids), 4000, replace=False)]
    near = v[rng.choice(len(v), 4000, replace=False)] + rng.normal(0.0, 2.0, (4000, 3))
    return np.concatenate([pts, far.astype(np.float32), v, mids, near.astype(np.float32)]).astype(np.float32)


def both(h, q):
    """(signed, unsigned) results on handle h: each (dist, face, closest, volume / summary)."""
    return eu._signed_call(h, q, 0, True, True, True), eu._surface_call(h, q, 0, True, True, True)


def check_against_restatement(sd, face, q, v, f):
    """The sign equals the restatement's wherever its margin holds; returns how many fall under the margin."""
    osd, oface, _, _, margin, _ = so.signed_distance(q, v, f)
    assert np.array_equal(face, oface)
    ok = margin >= MARGIN
    assert np.array_equal(np.sign(sd[ok]), np.sign(osd[ok])), np.flatnonzero(np.sign(sd) != np.sign(osd))[:10]
    zero = osd == 0.0
    assert np.array_equal(sd[zero], osd[zero])
    return int((~ok & ~zero & np.isfinite(osd)).sum())


@pytest.mark.parametrize('dtype', [np.float32, np.float64])
def test_magnitudes_equal_the_unsigned_call_and_signs_the_restatement(lobed, dtype):
    mesh, pts, _ = lobed
    q = mixed_queries(mesh, pts)
    if dtype == np.float64:
        q = q.astype(np.float64) + np.random.default_rng(1).normal(0.0, 1e-3, q.shape)
    h = _lib.Handle(0)
    try:
        eu._upload_surface(h, mesh)
        (sd, sf, sc, vol), (d, f, c, _) = both(h, q)
    finally:
        h.close()
    assert np.array_equal(np.abs(sd), d) and np.array_equal(sf, f) and np.array_equal(sc, c)
    nv = len(mesh._vertices)
    if dtype == np.float32:
        assert np.all(sd[len(pts) + 300:len(pts) + 300 + nv] == 0.0)
    off = (sd != 0.0).sum()                        # the vertices and edge midpoints lie on the surface
    assert (sd < 0).sum() > 0.2 * off and (sd > 0).sum() > 0.2 * off
    under = check_against_restatement(sd, sf, q, mesh._vertices['position'], mesh.faces)
    print('%s: %d of %d queries under the %.0e margin' % (np.dtype(dtype).name, under, len(q), MARGIN))
    assert under * 1e4 < 10 * len(q)
    V = so.signed_distance(q[:1], mesh._vertices['position'], mesh.faces)[3]
    assert abs(vol - V) <= 1e-12 * V


SOLIDS = {'tetrahedron': so.tetrahedron, 'prism': so.prism, 'cube': so.cube, 'l_polycube': so.l_polycube,
          'sphere': so.sphere, 'torus': so.torus}


def _truth_check(h, v, f, q):
    sd, face, _, vol = eu._signed_call(h, q, 0, True, True, False)
    inside = np.abs(so.winding_number(q, v, f)) > 0.5
    far = np.abs(sd) > 1e-6 * float((v.max(0) - v.min(0)).max())
    assert far.sum() > 0.9 * len(q)
    assert np.array_equal((sd < 0)[far], inside[far]), np.flatnonzero((sd < 0) != inside)[:10]
    return sd, face, vol


@pytest.fixture
def handle():
    h = _lib.Handle(0)
    yield h
    h.close()


@pytest.mark.parametrize('name', sorted(SOLIDS))
def test_sign_matches_the_winding_number_and_either_winding(handle, name):
    v, f = SOLIDS[name]()
    q = so.feature_queries(v, f)
    eu._upload_surface(handle, Raw(v, f))
    sd, face, vol = _truth_check(handle, v, f, q)
    check_against_restatement(sd, face, q, v, f)
    fr = np.ascontiguousarray(f[:, [0, 2, 1]])
    eu._upload_surface(handle, Raw(v, fr))
    sr, _, volr = _truth_check(handle, v, fr, q)
    assert volr == vol
    assert abs(vol - so.signed_distance(q[:1], v, f)[3]) <= 1e-12 * vol
    assert np.array_equal(np.abs(sr), eu._surface_call(handle, q, 0)[0])         # the reversed mesh's unsigned distances
    margin = so.signed_distance(q, v, f)[4]
    ok = margin >= MARGIN
    assert np.array_equal(np.sign(sr[ok]), np.sign(sd[ok]))


def test_lobed_mesh_winding_number_on_a_subset(handle, lobed):
    mesh, pts, _ = lobed
    q = mixed_queries(mesh, pts)
    nv = len(mesh._vertices)
    off = np.r_[0:len(pts) + 300, len(pts) + 300 + nv + 4000:len(q)]       # the cloud, far points, points near vertices
    q = q[np.random.default_rng(3).choice(off, 2000, replace=False)]
    eu._upload_surface(handle, mesh)
    _truth_check(handle, mesh._vertices['position'], mesh.faces, q)


def test_reversed_winding_keeps_volume_magnitudes_and_sides(handle, lobed):
    mesh, pts, _ = lobed
    q = mixed_queries(mesh, pts, seed=5)
    v, f = mesh._vertices['position'], mesh.faces
    eu._upload_surface(handle, mesh)
    sd, _, _, vol = eu._signed_call(handle, q)
    fr = np.ascontiguousarray(f[:, [0, 2, 1]])
    eu._upload_surface(handle, Raw(v, fr))
    (sr, _, _, volr), (dr, _, _, _) = both(handle, q)
    assert volr == vol
    assert abs(vol - so.signed_distance(q[:1], v, f)[3]) <= 1e-12 * vol
    assert np.array_equal(np.abs(sr), dr)
    ok = so.signed_distance(q, v, f)[4] >= MARGIN
    assert np.array_equal(np.sign(sr[ok]), np.sign(sd[ok]))


def _counts(msg):
    m = re.search(r'(\d+) boundary edges, (\d+) edges on more than two faces, (\d+) edges whose two faces traverse them the same '
                  r'way, (\d+) faces that repeat a vertex, (\d+) vertices whose faces form more than one fan', msg)
    assert m, msg
    return [int(x) for x in m.groups()]


def _defect_cases():
    import test_oracle_signed as tos
    out = [(c[0], c[1], c[2]) for c in tos.defect_meshes()]
    v, f = so.sphere(4)
    g = f.copy()
    g[3, 2] = g[3, 1]
    out.append(('repeated_vertex', v, g))
    return out


@pytest.mark.parametrize('case', _defect_cases(), ids=lambda c: c[0])
def test_meshes_that_do_not_bound_a_solid_are_refused(handle, case):
    _, v, f = case
    want = so.tables(f, len(v))[3]
    assert any(want)
    eu._upload_surface(handle, Raw(v, f))
    q = (np.asarray(v, np.float64)[:50] + 0.3).astype(np.float32)
    with pytest.raises(ValueError) as e:
        eu._signed_call(handle, q)
    assert _counts(str(e.value)) == want
    with pytest.raises(ValueError):
        eu.enclosed_volume(Raw(v, f), handle)
    d, face, c, _ = eu._surface_call(handle, q, 0, True, True, True)
    od, of, oc = orc.surface_nearest(q, v, f)
    assert np.array_equal(d, od) and np.array_equal(face, of) and np.array_equal(c, oc)


def test_tables_follow_the_topology_and_pseudonormals_the_positions(lobed):
    mesh, pts, _ = lobed
    a = mesh
    bv, bf = so.torus(300.0, 100.0, 48, 24)
    b = Raw(bv, bf)
    q = mixed_queries(mesh, pts)[::5]

    def fresh(m, pos=None):
        h = _lib.Handle(0)
        try:
            eu._upload_surface(h, m)
            if pos is not None:
                h.call('nw_set_positions', _lib.fptr(pos))
            return eu._signed_call(h, q, 0, True, True, True)
        finally:
            h.close()
    h = _lib.Handle(0)
    try:
        eu._upload_surface(h, a)
        ra = eu._signed_call(h, q, 0, True, True, True)
        eu._upload_surface(h, b)
        rb = eu._signed_call(h, q, 0, True, True, True)
        pos = np.ascontiguousarray(bv * np.float32(1.5) + np.float32(20.0))
        h.call('nw_set_positions', _lib.fptr(pos))
        rc = eu._signed_call(h, q, 0, True, True, True)
    finally:
        h.close()
    for got, want in ((ra, fresh(a)), (rb, fresh(b)), (rc, fresh(b, pos))):
        for x, y in zip(got[:3], want[:3]):
            assert np.array_equal(x, y)
        assert got[3] == want[3]
    assert rc[3] != rb[3]


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
        explicit = eu._signed_call(h, pts, 0, True, True, True)
        cold = eu._signed_call(h, None, len(pts), True, True, True)
        h.call('nw_compute_weights')
        warm = eu._signed_call(h, None, len(pts), True, True, True)
    finally:
        h.close()
    for r in (cold, warm):
        for a, b in zip(r[:3], explicit[:3]):
            assert np.array_equal(a, b)
        assert r[3] == explicit[3]


def _fit(mesh, pts, sig, probe):
    """Two nw_search calls of 4 iterations on a fresh handle; with `probe`, signed calls run between them."""
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
                eu._signed_call(h, None, len(pts), True, True, True)
                eu._signed_call(h, pts[::7] * np.float32(3.0), 0, True, True, True)
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


def test_point_surface_distance_signed_after_a_fit():
    from ch_shrinkwrap_b200.membrane_mesh import MembraneMesh
    from ch_shrinkwrap_b200.mesh_conj_grad import ShrinkwrapMeshConjGrad
    shape = synth.Sphere(500.0)
    pts, sig = synth.smlm_cloud(shape, 20000, seed=7)
    mesh = MembraneMesh(mesh=synth.star_mesh(shape, 8, scale=1.2), kc=1.0, step_size=20.0)
    mesh.cg = ShrinkwrapMeshConjGrad(mesh, pts)
    mesh.cg.search(pts, lams=[10.0], num_iters=5, sigma_inv=(1.0 / sig.ravel()).astype(np.float32))
    sd, face = mesh.point_surface_distance(return_face=True, signed=True)
    d = mesh.point_surface_distance()
    fitted = minimesh.MiniMesh(mesh._vertices['position'].copy(), mesh.faces)
    od, of = eu.surface_distance(fitted, pts, return_face=True, signed=True)
    assert np.array_equal(sd, od) and np.array_equal(face, of) and np.array_equal(np.abs(sd), d)
    v, f = fitted._vertices['position'], fitted.faces
    pick = np.random.default_rng(1).choice(len(pts), 2000, replace=False)
    inside = np.abs(so.winding_number(pts[pick], v, f)) > 0.5
    far = np.abs(sd[pick]) > 1e-6 * float((v.max(0) - v.min(0)).max())
    assert np.array_equal((sd[pick] < 0)[far], inside[far])
    V = eu.enclosed_volume(fitted)
    assert abs(V - so.signed_distance(pts[:1], v, f)[3]) <= 1e-12 * V


def test_c3_mesh_with_a_million_queries():
    """The bench's C3 mesh (501 762 vertices) and 10^6 localisations on it."""
    v, f = minimesh.geodesic_sphere(224)
    v, f = minimesh.spatially_sorted(v, f)
    r = synth.radial_surface(synth.two_lobed(), v, n_bisect=32)
    mesh = minimesh.MiniMesh(v * (1.2 * r)[:, None], f)
    assert len(mesh._vertices) == 501762
    pts, _ = synth.mesh_surface_cloud(v * r[:, None], f, 1_000_000, seed=3)
    h = _lib.Handle(0)
    try:
        eu._upload_surface(h, mesh)
        (sd, sf, sc, vol), (d, df, dc, _) = both(h, pts)
    finally:
        h.close()
    assert np.array_equal(np.abs(sd), d) and np.array_equal(sf, df) and np.array_equal(sc, dc)
    pick = np.random.default_rng(0).choice(len(pts), 10_000, replace=False)
    under = check_against_restatement(sd[pick], sf[pick], pts[pick], mesh._vertices['position'], mesh.faces)
    print('C3: %d of 10^4 under the margin, volume %.6g, %.3f of the queries inside' % (under, vol, (sd < 0).mean()))
    assert under < 10

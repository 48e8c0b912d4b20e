"""nw_self_intersections (exact self-intersection pairs of a triangle mesh) on the GPU, against the rational restatement
tests/intersect_oracle.py."""
import ctypes
import os
import sys

import numpy as np
import pytest

from ch_shrinkwrap_b200 import _lib, minimesh, synth
from ch_shrinkwrap_b200 import evaluation_utils as eu
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import intersect_oracle as io  # noqa: E402
import signed_oracle as so  # noqa: E402

pytestmark = pytest.mark.gpu


class Raw:
    """Just what _upload_surface reads: positions and face rows (no neighbour tables, so any face list goes up)."""

    def __init__(self, v, f):
        self._vertices = np.zeros(len(v), [('position', np.float32, 3)])
        self._vertices['position'] = v
        self.faces = np.ascontiguousarray(f, np.int32)


@pytest.fixture(scope='module')
def handle():
    h = _lib.Handle(0)
    yield h
    h.close()


def gpu(handle, v, f, stats=False):
    return eu.self_intersections(Raw(v, f), handle, return_stats=stats)


def check(handle, v, f, subset=None):
    """The GPU list equals the oracle's; returns the GPU stats."""
    got, st = gpu(handle, v, f, stats=True)
    want, deg, nf = io.self_intersections(v, f, subset)
    if subset is not None:
        s = set(int(x) for x in subset)
        got_s = got[[a in s or b in s for a, b in got.tolist()]] if len(got) else got
        assert np.array_equal(got_s, want)
        assert len(got_s) == len(got), 'pairs outside the faces of interest'
    else:
        assert np.array_equal(got, want), (got[:10], want[:10])
        assert (st.degenerate, st.non_finite) == (deg, nf)
    assert got.dtype == np.int32 and (len(got) == 0 or np.all(got[:, 0] < got[:, 1]))
    return got, st


SOLIDS = {'tetrahedron': so.tetrahedron, 'prism': so.prism, 'cube': so.cube, 'l_polycube': so.l_polycube,
          'sphere': so.sphere, 'torus': so.torus}


@pytest.mark.parametrize('name', sorted(SOLIDS))
def test_solids_are_embedded(handle, name):
    v, f = SOLIDS[name]()
    got, st = gpu(handle, v, f, stats=True)
    assert len(got) == 0 and st.degenerate == 0 and st.non_finite == 0 and st.candidates > 0


@pytest.mark.parametrize('n', [4, 8, 16])
def test_star_meshes_and_the_lobed_mesh_are_embedded(handle, n):
    for shape in (synth.Sphere(500.0), synth.two_lobed()):
        m = synth.star_mesh(shape, n)
        assert len(eu.self_intersections(m, handle)) == 0
    m = synth.star_mesh(synth.two_lobed(), 40)           # the mesh of the signed-distance tests
    assert len(eu.self_intersections(m, handle)) == 0


def two_spheres():
    a = minimesh.sphere_mesh(100.0, 8)
    b = minimesh.sphere_mesh(80.0, 8, centre=(120.0, 30.0, 10.0))
    va, vb = a._vertices['position'], b._vertices['position']
    return np.concatenate([va, vb]).astype(np.float32), np.concatenate([a.faces, b.faces + len(va)]).astype(np.int32)


def test_two_overlapping_spheres(handle):
    v, f = two_spheres()
    got, _ = check(handle, v, f)
    assert len(got) > 50


def spiked_star(n=8, k=4, seed=0):
    m = synth.star_mesh(synth.Sphere(500.0), n)
    v = m._vertices['position'].copy()
    moved = np.random.default_rng(seed).choice(len(v), k, replace=False)
    v[moved] *= np.float32(-1.5)
    return v, m.faces.astype(np.int32), moved


def test_star_mesh_with_spikes_through_the_opposite_side(handle):
    v, f, _ = spiked_star()
    got, _ = check(handle, v, f)
    assert len(got) > 0


def test_planar_fold_over_gives_one_pair(handle):
    m = minimesh.planar_mesh(10.0, 6)
    v, f = m._vertices['position'].copy(), m.faces.astype(np.int32)
    assert len(gpu(handle, v, f)) == 0
    # a corner with a single face (c, a, b): pull c across edge ab into the face on its other side
    cnt = np.bincount(f.ravel(), minlength=len(v))
    c = int(np.flatnonzero(cnt == 1)[0])
    fc = int(np.flatnonzero((f == c).any(1))[0])
    a, b = [int(x) for x in f[fc] if x != c]
    g = [r for r in range(len(f)) if r != fc and a in f[r] and b in f[r]][0]
    d = int([x for x in f[g] if x not in (a, b)][0])
    mid = (v[a] + v[b]) * np.float32(0.5)
    v[c] = mid + (v[d] - mid) * np.float32(0.25)
    got, _ = check(handle, v, f)
    assert got.tolist() == [sorted([fc, g])]


def test_two_cubes_touching_face_to_face(handle):
    v, f = so.cube()
    v = np.asarray(v, np.float32)
    w = v[:, 0].max() - v[:, 0].min()
    v2 = np.concatenate([v, v + np.array([w, 0, 0], np.float32)])
    f2 = np.concatenate([f, f + len(v)]).astype(np.int32)
    got, _ = check(handle, v2, f2)
    assert len(got) > 0
    assert len(gpu(handle, np.concatenate([v, v + np.array([w * 1.01, 0, 0], np.float32)]), f2)) == 0


def tilted_grid(n=6):
    """A planar grid on z = x + y (integer coordinates: exactly coplanar in float32, but not axis-aligned)."""
    m = minimesh.planar_mesh(float(n), n)
    v = m._vertices['position'].astype(np.float32).copy()
    v[:, 2] = v[:, 0] + v[:, 1]
    return v, m.faces.astype(np.int32)


def test_the_exact_stage_runs_on_coplanar_and_near_coplanar_folds(handle):
    v, f = tilted_grid()
    got, st = check(handle, v, f)
    assert len(got) == 0 and st.exact > 0
    # fold an interior vertex across the diagonal of its neighbourhood, in the plane
    cnt = np.bincount(f.ravel(), minlength=len(v))
    c = int(np.flatnonzero(cnt == 6)[0])
    w = v.copy()
    w[c, :2] += np.float32(1.5)
    w[c, 2] = w[c, 0] + w[c, 1]
    got, st = check(handle, w, f)
    assert len(got) > 0 and st.exact > 0
    for z in (np.nextafter(w[c, 2], np.float32(1e9)), np.nextafter(w[c, 2], np.float32(-1e9))):
        u = w.copy()
        u[c, 2] = z
        _, st = check(handle, u, f)
        assert st.exact > 0


def test_invariance_under_winding_permutation_and_scale(handle):
    v, f = two_spheres()
    want = gpu(handle, v, f)
    assert len(want) > 0
    assert np.array_equal(gpu(handle, v, f[:, [0, 2, 1]]), want)
    for k in (60, -60):
        assert np.array_equal(gpu(handle, v * np.float32(2.0 ** k), f), want)
    perm = np.random.default_rng(1).permutation(len(f))
    got = gpu(handle, v, f[perm])
    mapped = np.sort(perm[got], 1)
    mapped = mapped[np.lexsort((mapped[:, 1], mapped[:, 0]))]
    assert np.array_equal(mapped, want)


def test_repeated_calls_and_capacity(handle):
    v, f, _ = spiked_star(seed=3)
    eu._upload_surface(handle, Raw(v, f))
    a, sa = eu._self_intersections(handle, True)
    b, sb = eu._self_intersections(handle, True, capacity=1)
    assert np.array_equal(a, b) and sa == sb and len(a) > 2
    n = ctypes.c_int64(-1)
    handle.call('nw_self_intersections', None, 0, ctypes.byref(n), None)
    assert n.value == len(a)
    part = np.full((2, 2), -7, np.int32)
    handle.call('nw_self_intersections', _lib.iptr(part), 2, ctypes.byref(n), None)
    assert n.value == len(a) and np.array_equal(part, a[:2])
    with pytest.raises(ValueError):
        handle.call('nw_self_intersections', None, 4, ctypes.byref(n), None)


def test_points_mode_is_refused(handle):
    t = np.random.default_rng(0).normal(size=(100, 3)).astype(np.float32)
    eu.nearest_point_distance(t, t[:10], handle)
    n = ctypes.c_int64(0)
    with pytest.raises(ValueError):
        handle.call('nw_self_intersections', None, 0, ctypes.byref(n), None)


def test_non_finite_and_degenerate_faces_are_counted(handle):
    v, f = two_spheres()
    v = v.copy()
    v[5] = np.nan
    f = np.concatenate([f, [[0, 0, 1], [1, 2, 1]]]).astype(np.int32)
    _, st = check(handle, v, f)
    assert st.degenerate == 2 and st.non_finite == int((f == 5).any(1).sum())


def _fit(mesh, pts, sig, probe):
    """Two nw_search calls of 4 iterations on a fresh handle; with `probe`, self-intersection calls run between them."""
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
                eu._self_intersections(h, True)
                eu._self_intersections(h, False, capacity=1)
        return out, hists
    finally:
        h.close()


def test_no_side_effects_on_the_fit():
    shape = synth.two_lobed()
    mesh = synth.star_mesh(shape, 40)
    pts, sig = synth.smlm_cloud(shape, 4000, seed=11)
    a_pos, a_hist = _fit(mesh, pts, sig, probe=False)
    b_pos, b_hist = _fit(mesh, pts, sig, probe=True)
    for x, y in zip(a_pos, b_pos):
        assert np.array_equal(x, y)
    for x, y in zip(a_hist, b_hist):
        for u, v in zip(x, y):
            assert np.array_equal(u, v)


def test_self_intersections_after_a_fit():
    from ch_shrinkwrap_b200.membrane_mesh import MembraneMesh
    from ch_shrinkwrap_b200.mesh_conj_grad import ShrinkwrapMeshConjGrad
    shape = synth.Sphere(500.0)
    pts, sig = synth.smlm_cloud(shape, 20000, seed=7)
    mesh = MembraneMesh(mesh=synth.star_mesh(shape, 8, scale=1.2), kc=1.0, step_size=20.0)
    mesh.cg = ShrinkwrapMeshConjGrad(mesh, pts)
    mesh.cg.search(pts, lams=[10.0], num_iters=5, sigma_inv=(1.0 / sig.ravel()).astype(np.float32))
    got, st = mesh.self_intersections(return_stats=True)
    fitted = minimesh.MiniMesh(mesh._vertices['position'].copy(), mesh.faces)
    want, wst = eu.self_intersections(fitted, return_stats=True)
    assert np.array_equal(got, want) and st == wst
    assert np.array_equal(got, io.self_intersections(fitted._vertices['position'], fitted.faces)[0])


def test_c3_mesh_embedded_then_spiked():
    """The bench's C3 mesh (1 003 520 faces): embedded by construction (every face stays inside the cone of its vertex
    directions), then about 100 vertices moved to -1.5 v."""
    v, f = minimesh.geodesic_sphere(224)
    v, f = minimesh.spatially_sorted(v, f)
    r = synth.radial_surface(synth.two_lobed(), v, n_bisect=32)
    pos = (v * (1.2 * r)[:, None]).astype(np.float32)
    f = f.astype(np.int32)
    assert len(f) == 1003520
    h = _lib.Handle(0)
    try:
        got, st = gpu(h, pos, f, stats=True)
        assert len(got) == 0 and st.degenerate == 0 and st.non_finite == 0
        moved = np.random.default_rng(5).choice(len(pos), 100, replace=False)
        pos[moved] *= np.float32(-1.5)
        subset = np.flatnonzero(np.isin(f, moved).any(1))
        got, st = check(h, pos, f, subset)
        print('C3 spiked: %d pairs, %d candidates, %d exact' % (len(got), st.candidates, st.exact))
        assert len(got) > 100
    finally:
        h.close()

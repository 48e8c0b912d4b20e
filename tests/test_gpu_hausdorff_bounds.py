"""nw_hausdorff_bounds: certified bounds of the one-sided Hausdorff distance between two triangle meshes, on the GPU.

Known answers (walls, a tube, one triangle, a mesh and its copy, concentric spheres), the witness against the numpy
restatement (tests/surface_oracle.py), dense barycentric samples (tests/hausdorff_oracle.py) below the upper bound, the
sampled metric hausdorff_distance below it too, determinism, symmetry, the query budget and the refused inputs."""
import ctypes
import os
import sys

import numpy as np
import pytest

from ch_shrinkwrap_b200 import _lib, minimesh, synth
from ch_shrinkwrap_b200 import evaluation_utils as eu
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import hausdorff_oracle as hor  # noqa: E402
import surface_oracle as orc  # noqa: E402

pytestmark = pytest.mark.gpu


def eps_of(m0, m1):
    return 2.0 * hor.rounding_allowance(m0._vertices['position'], m1._vertices['position'])


def quad(p0, p1, p2, p3):
    return np.array([p0, p1, p2, p3], np.float32), np.array([[0, 1, 2], [0, 2, 3]], np.int32)


def union(*parts):
    vs, fs, n = [], [], 0
    for v, f in parts:
        vs.append(v)
        fs.append(f + n)
        n += len(v)
    return minimesh.MiniMesh(np.concatenate(vs), np.concatenate(fs))


def walls(xs=(-1.0, 1.0), ys=()):
    """Squares in the planes x = c (c in xs) and y = c (c in ys), spanning [-10, 10] in the other two coordinates."""
    parts = [quad((c, -10, -10), (c, 10, -10), (c, 10, 10), (c, -10, 10)) for c in xs]
    parts += [quad((-10, c, -10), (10, c, -10), (10, c, 10), (-10, c, 10)) for c in ys]
    return union(*parts)


def triangle(a, b, c):
    return minimesh.MiniMesh(np.array([a, b, c], np.float32), np.array([[0, 1, 2]], np.int32))


def check_witness(r, m0, m1):
    """Each lower bound is the oracle's distance of its witness, bit for bit, with the oracle's nearest face."""
    for lower, (p, fa, fb), a, b in ((r.lower01, r.witness01, m0, m1), (r.lower10, r.witness10, m1, m0)):
        d, f, _ = orc.surface_nearest(p[None], b._vertices['position'], b.faces)
        assert d[0] == lower and f[0] == fb
        # the witness lies on its face of the source mesh, up to the rounding of the midpoints
        dd = orc.surface_nearest(p[None], a._vertices['position'], a.faces[fa:fa + 1])[0]
        assert dd[0] <= 1e-9 * (1.0 + np.abs(p).sum())


def test_interior_maximum_between_two_walls():
    m0, m1 = triangle((-1, -1, 0), (1, -1, 0), (0.3, 2, 0)), walls()
    e, tol = eps_of(m0, m1), 0.01
    r, s01, _ = eu.hausdorff_bounds(m0, m1, tol=tol, return_stats=True)
    assert abs(r.lower01 - 1.0) <= e and r.upper01 - 1.0 <= tol + e and s01[4] == 1
    assert s01[0] >= 2                                  # the corners give 0.7; the first split measures (0, -1, 0)
    check_witness(r, m0, m1)
    assert eu.hausdorff_distance(m0, m1, dx_min=0.05).h01 <= r.upper01


def test_interior_maximum_inside_a_tube():
    m0 = triangle((-0.9, -0.8, 0), (0.85, -0.6, 0), (-0.1, 0.95, 0))
    m1 = walls((-1.0, 1.0), (-1.0, 1.0))
    e, tol = eps_of(m0, m1), 0.01
    r = eu.hausdorff_bounds(m0, m1, tol=tol)
    assert r.lower01 - e <= 1.0 <= r.upper01 and r.upper01 - r.lower01 <= tol and r.converged
    assert r.lower01 > 0.95
    check_witness(r, m0, m1)
    assert eu.hausdorff_distance(m0, m1, dx_min=0.05).h01 <= r.upper01


def test_convex_target_needs_no_split():
    m0 = minimesh.planar_mesh(100.0, 12)
    v = m0._vertices['position'].astype(np.float64)
    m0 = minimesh.MiniMesh(v @ np.array([[0.8, 0.6, 0.0], [-0.6, 0.8, 0.0], [0.0, 0.0, 1.0]]) + [3.0, -7.0, 25.0], m0.faces)
    m1 = triangle((-40, -30, 0), (60, -20, 5), (10, 70, -5))
    e = eps_of(m0, m1)
    r, s01, _ = eu.hausdorff_bounds(m0, m1, return_stats=True)
    vd = orc.surface_nearest(m0._vertices['position'], m1._vertices['position'], m1.faces)[0]
    assert r.lower01 == vd.max() and r.upper01 - r.lower01 <= e
    assert s01[0] == 1 and s01[1] == len(m0.faces) and s01[4] == 1
    check_witness(r, m0, m1)


def test_a_mesh_against_itself_and_an_offset_copy():
    m = minimesh.sphere_mesh(500.0, 8)
    e, tol = eps_of(m, m), 0.01
    r = eu.hausdorff_bounds(m, m, tol=tol)
    assert r.lower <= e and r.upper <= tol + e and r.converged
    p0 = minimesh.planar_mesh(100.0, 20)
    v = p0._vertices['position'].copy()
    v[:, 2] += np.float32(0.5)
    p1 = minimesh.MiniMesh(v, p0.faces)
    e = eps_of(p0, p1)
    r = eu.hausdorff_bounds(p0, p1, tol=tol)
    for lo, up in ((r.lower01, r.upper01), (r.lower10, r.upper10)):
        assert abs(lo - 0.5) <= e and up <= 0.5 + tol + e
    assert r.converged


def _max_circumradius(mesh):
    v = mesh._vertices['position'].astype(np.float64)[mesh.faces]
    a, b, c = (np.sqrt(((v[:, i] - v[:, j]) ** 2).sum(1)) for i, j in ((0, 1), (1, 2), (2, 0)))
    area = 0.5 * np.sqrt((np.cross(v[:, 1] - v[:, 0], v[:, 2] - v[:, 0]) ** 2).sum(1))
    return float((a * b * c / (4.0 * area)).max())


def test_concentric_spheres_are_within_the_sagitta_bound():
    r0, r1, tol = 500.0, 530.0, 0.01
    m0, m1 = minimesh.sphere_mesh(r0, 12), minimesh.sphere_mesh(r1, 16)
    s0 = r0 - np.sqrt(r0 ** 2 - _max_circumradius(m0) ** 2)
    s1 = r1 - np.sqrt(r1 ** 2 - _max_circumradius(m1) ** 2)
    r = eu.hausdorff_bounds(m0, m1, tol=tol)
    for x in (r.lower01, r.upper01, r.lower10, r.upper10):
        assert (r1 - r0) - s1 - tol <= x <= (r1 - r0) + s0 + tol, (x, s0, s1)
    hd = eu.hausdorff_distance(m0, m1, dx_min=10.0)
    assert hd.h01 <= r.upper01 and hd.h10 <= r.upper10 and r.converged


@pytest.fixture(scope='module')
def lobed_pair():
    shape = synth.two_lobed()
    m0 = synth.star_mesh(shape, 24)
    v = m0._vertices['position'] + np.random.default_rng(5).normal(0.0, 2.0, m0._vertices['position'].shape)
    return m0, minimesh.MiniMesh(v, m0.faces), synth.star_mesh(shape, 17, scale=1.21)


@pytest.mark.parametrize('which', ['perturbed', 'resolution'])
def test_lobed_mesh_against_a_copy(lobed_pair, which):
    m0, mp, mr = lobed_pair
    m1 = mp if which == 'perturbed' else mr
    e = eps_of(m0, m1)
    r = eu.hausdorff_bounds(m0, m1)
    assert r.converged and r.upper01 - r.lower01 <= 0.01 and r.upper10 - r.lower10 <= 0.01
    check_witness(r, m0, m1)
    for a, b, lo, up in ((m0, m1, r.lower01, r.upper01), (m1, m0, r.lower10, r.upper10)):
        va, vb = a._vertices['position'], b._vertices['position']
        assert hor.max_sample_distance(va, a.faces, vb, b.faces) <= up + e
        assert orc.surface_nearest(va, vb, b.faces)[0].max() <= lo
    for dx in (1.0, 5.0):
        hd = eu.hausdorff_distance(m0, m1, dx_min=dx)
        assert hd.h01 <= r.upper01 and hd.h10 <= r.upper10 and hd.hausdorff <= r.upper


def test_deterministic_and_symmetric(lobed_pair):
    m0, m1, _ = lobed_pair
    r = eu.hausdorff_bounds(m0, m1)
    again = eu.hausdorff_bounds(m0, m1)
    swapped = eu.hausdorff_bounds(m1, m0)

    def flat(x):
        return [x.lower01, x.upper01, x.lower10, x.upper10, x.lower, x.upper, x.converged,
                x.witness01[0].tobytes(), x.witness01[1:], x.witness10[0].tobytes(), x.witness10[1:]]
    assert flat(r) == flat(again)
    assert (swapped.lower01, swapped.upper01, swapped.lower10, swapped.upper10) == (r.lower10, r.upper10, r.lower01, r.upper01)
    assert swapped.witness01[0].tobytes() == r.witness10[0].tobytes() and swapped.witness01[1:] == r.witness10[1:]
    assert swapped.witness10[0].tobytes() == r.witness01[0].tobytes() and swapped.witness10[1:] == r.witness01[1:]
    assert (swapped.lower, swapped.upper, swapped.converged) == (r.lower, r.upper, r.converged)


def test_a_small_budget_stops_early_with_valid_bounds(lobed_pair):
    m0, _, m1 = lobed_pair
    n_used = len(np.unique(m0.faces))
    r, s01, _ = eu.hausdorff_bounds(m0, m1, tol=1e-6, max_queries=n_used + 100, return_stats=True)
    assert not r.converged and s01[4] == 0 and s01[2] <= n_used + 100
    e = eps_of(m0, m1)
    va, vb = m0._vertices['position'], m1._vertices['position']
    assert hor.max_sample_distance(va, m0.faces, vb, m1.faces) <= r.upper01 + e
    assert r.lower01 <= r.upper01
    with pytest.raises(ValueError, match='max_queries'):
        eu.hausdorff_bounds(m0, m1, max_queries=n_used - 1)


class RawMesh:
    """Positions and face rows only (no topology checks), for inputs a MiniMesh would not build."""

    def __init__(self, v, f):
        self._vertices = np.zeros(len(v), [('position', np.float32, 3)])
        self._vertices['position'] = v
        self.faces = np.asarray(f, np.int32)


def test_refused_inputs_and_skipped_faces():
    m1 = walls()
    m0 = triangle((-1, -1, 0), (1, -1, 0), (0.3, 2, 0))
    with pytest.raises(ValueError, match='tol'):
        eu.hausdorff_bounds(m0, m1, tol=-1.0)
    with pytest.raises(ValueError, match='outside'):
        eu.hausdorff_bounds(RawMesh(m0._vertices['position'], [[0, 1, 3]]), m1)
    nan = RawMesh(np.array([[0, 0, 0], [1, 0, 0], [np.nan, 1, 0]], np.float32), [[0, 1, 2]])
    with pytest.raises(ValueError, match='no face with finite corners'):
        eu.hausdorff_bounds(nan, m1)
    h = _lib.Handle(0)
    try:
        eu._upload_surface(h, m1)
        with pytest.raises(ValueError, match='no face with finite corners'):
            eu._hausdorff_bounds(h, nan, 0.01, 1000)
        eu._upload_surface(h, nan)
        with pytest.raises(ValueError, match="handle's mesh has no face"):
            eu._hausdorff_bounds(h, m0, 0.01, 1000)
        t = np.random.default_rng(0).normal(size=(50, 3)).astype(np.float32)
        h.call('nw_set_point_targets', ctypes.c_void_p(t.ctypes.data), 0, len(t))
        with pytest.raises(ValueError, match='point targets'):
            eu._hausdorff_bounds(h, m0, 0.01, 1000)
    finally:
        h.close()
    # a face with a NaN corner is skipped and counted; its other vertices are not measured unless a finite face uses them
    v = np.concatenate([m0._vertices['position'], [[np.nan, 0, 0], [50.0, 50.0, 50.0]]]).astype(np.float32)
    mixed = RawMesh(v, [[0, 1, 2], [3, 4, 0]])
    r, s01, _ = eu.hausdorff_bounds(mixed, m1, return_stats=True)
    ref = eu.hausdorff_bounds(m0, m1)
    assert s01[3] == 1 and (r.lower01, r.upper01) == (ref.lower01, ref.upper01)

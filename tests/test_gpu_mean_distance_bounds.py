"""nw_mean_distance_bounds: certified bounds of the area-weighted mean and RMS distances between two triangle meshes.

Known answers (parallel squares, a crossing plane, a mesh against itself), the Lipschitz bracket of
tests/mean_distance_oracle.py on a tube, lobed meshes and random triangle soups, the Hausdorff bounds above the RMS, the
area against numpy, determinism, symmetry, the query budget, refused inputs, counted faces and no effect on a fit."""
import ctypes
import os
import sys

import numpy as np
import pytest
from scipy.spatial import Delaunay

from ch_shrinkwrap_b200 import _lib, minimesh, synth
from ch_shrinkwrap_b200 import evaluation_utils as eu
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import hausdorff_oracle as hor  # noqa: E402
import mean_distance_oracle as mo  # noqa: E402

pytestmark = pytest.mark.gpu


class RawMesh:
    """Positions and face rows only (no topology checks): soups, NaN corners and repeated vertices."""

    def __init__(self, v, f):
        self._vertices = np.zeros(len(v), [('position', np.float32, 3)])
        self._vertices['position'] = v
        self.faces = np.asarray(f, np.int32)


def eps_of(m0, m1):
    """The allowance of the call (2^-40 x the L1 coordinate bound), with a factor of 4 for the final divisions."""
    return 4.0 * hor.rounding_allowance(m0._vertices['position'], m1._vertices['position'])


def irregular_square(n=60, seed=3):
    """The unit square at z = 0, Delaunay-triangulated over its corners and n random points."""
    p = np.random.default_rng(seed).uniform(0.02, 0.98, (n, 2))
    p = np.concatenate([[[0, 0], [1, 0], [1, 1], [0, 1]], p])
    f = Delaunay(p).simplices.astype(np.int32)
    return RawMesh(np.concatenate([p, np.zeros((len(p), 1))], 1).astype(np.float32), f)


def big_quad(z_of_x):
    """[-8, 12]^2 as two triangles split along x + y = 4, which misses the unit square; height z_of_x(x)."""
    xy = np.array([[-8, -8], [12, -8], [12, 12], [-8, 12]], np.float64)
    v = np.concatenate([xy, z_of_x(xy[:, :1])], 1).astype(np.float32)
    return RawMesh(v, [[1, 2, 3], [1, 3, 0]])


def oracle(a, b, n):
    return mo.mean_distance_bracket(a._vertices['position'], a.faces, b._vertices['position'], b.faces, n)


def check_oracle(r, m0, m1, n=6, narrower=True):
    """Both brackets are valid, so they overlap; the GPU's is the narrower one."""
    e = eps_of(m0, m1)
    for a, b, got in ((m0, m1, r[0:4]), (m1, m0, r[4:8])):
        _, mean, rms = oracle(a, b, n)
        for (lo, hi), (olo, ohi) in (((got[0], got[1]), mean), ((got[2], got[3]), rms)):
            assert lo <= hi and lo - e <= ohi and olo <= hi + e, (lo, hi, olo, ohi)
            if narrower:
                assert hi - lo <= ohi - olo
    assert r.mean01_lower <= r.rms01_upper and r.mean10_lower <= r.rms10_upper


def test_parallel_squares_are_exact_in_one_level():
    a, delta = irregular_square(), 0.25
    b = big_quad(lambda x: np.full_like(x, delta))
    e = eps_of(a, b)
    r, s01, _ = eu.mean_distance_bounds(a, b, return_stats=True)
    for x in (r.mean01_lower, r.mean01_upper, r.rms01_lower, r.rms01_upper):
        assert abs(x - delta) <= e
    assert abs(r.area0 - 1.0) <= 1e-12 and r.area1 == 400.0
    assert s01[0] == 1 and s01[2] == len(a._vertices) and s01[3] > 0 and s01[6] == 1


def test_a_crossing_plane():
    a, tol = irregular_square(), 0.01
    b = big_quad(lambda x: x - 0.5)
    e = eps_of(a, b)
    r, s01, _ = eu.mean_distance_bounds(a, b, tol=tol, return_stats=True)
    mean, rms = 1.0 / (4.0 * np.sqrt(2.0)), np.sqrt(1.0 / 24.0)
    assert r.mean01_lower - e <= mean <= r.mean01_upper + e and r.mean01_upper - r.mean01_lower <= tol
    assert r.rms01_lower - e <= rms <= r.rms01_upper + e and r.rms01_upper - r.rms01_lower <= tol
    assert s01[6] == 1 and s01[0] > 1 and s01[2] > len(a._vertices)


def test_a_mesh_against_itself():
    m = minimesh.sphere_mesh(500.0, 8)
    e = eps_of(m, m)
    r = eu.mean_distance_bounds(m, m)
    assert all(0.0 <= x <= e for x in r[:8]) and r.converged


def test_a_triangle_inside_a_tube():
    m0 = minimesh.MiniMesh(np.array([(-0.9, -0.8, 0), (0.85, -0.6, 0), (-0.1, 0.95, 0)], np.float32), np.array([[0, 1, 2]], np.int32))
    parts = []
    for c in (-1.0, 1.0):
        parts.append(np.array([(c, -10, -10), (c, 10, -10), (c, 10, 10), (c, -10, 10)], np.float32))
        parts.append(np.array([(-10, c, -10), (10, c, -10), (10, c, 10), (-10, c, 10)], np.float32))
    m1 = RawMesh(np.concatenate(parts), np.concatenate([np.array([[0, 1, 2], [0, 2, 3]]) + 4 * k for k in range(4)]))
    r = eu.mean_distance_bounds(m0, m1, tol=1e-3)
    assert r.converged
    e = eps_of(m0, m1)
    _, mean, rms = oracle(m0, m1, 32)
    assert r.mean01_lower - e <= mean[1] and mean[0] <= r.mean01_upper + e
    assert r.rms01_lower - e <= rms[1] and rms[0] <= r.rms01_upper + e


@pytest.fixture(scope='module')
def lobed_pair():
    shape = synth.two_lobed()
    m0 = synth.star_mesh(shape, 12)
    v = m0._vertices['position'] + np.random.default_rng(5).normal(0.0, 2.0, m0._vertices['position'].shape)
    return m0, minimesh.MiniMesh(v, m0.faces), synth.star_mesh(shape, 9, scale=1.21)


@pytest.mark.parametrize('which', ['perturbed', 'resolution'])
def test_lobed_mesh_against_a_copy(lobed_pair, which):
    m0, mp, mr = lobed_pair
    m1 = mp if which == 'perturbed' else mr
    r = eu.mean_distance_bounds(m0, m1)
    assert r.converged
    check_oracle(r, m0, m1)
    hb = eu.hausdorff_bounds(m0, m1)
    e = eps_of(m0, m1)
    assert r.rms01_lower <= hb.upper01 + e and r.rms10_lower <= hb.upper10 + e
    for m, area in ((m0, r.area0), (m1, r.area1)):
        want = mo.face_areas(m._vertices['position'], m.faces).sum()
        assert abs(area - want) <= 1e-12 * want


def test_deterministic_and_symmetric(lobed_pair):
    m0, m1, _ = lobed_pair
    r = eu.mean_distance_bounds(m0, m1)
    assert tuple(r) == tuple(eu.mean_distance_bounds(m0, m1))
    s = eu.mean_distance_bounds(m1, m0)
    assert tuple(s[4:8]) == tuple(r[0:4]) and tuple(s[0:4]) == tuple(r[4:8])
    assert (s.area0, s.area1, s.converged) == (r.area1, r.area0, r.converged)


def test_a_small_budget_gives_a_wider_valid_bracket(lobed_pair):
    m0, _, m1 = lobed_pair
    n_used = len(np.unique(m0.faces))
    r = eu.mean_distance_bounds(m0, m1)
    small, s01, _ = eu.mean_distance_bounds(m0, m1, tol=1e-6, max_queries=n_used + 100, return_stats=True)
    assert not small.converged and s01[6] == 0 and s01[2] <= n_used + 100
    e = eps_of(m0, m1)
    for k in (0, 2):
        assert small[k] <= r[k] + e and r[k + 1] <= small[k + 1] + e
    with pytest.raises(ValueError, match='max_queries'):
        eu.mean_distance_bounds(m0, m1, max_queries=n_used - 1)


def test_random_soups(lobed_pair):
    rng = np.random.default_rng(17)
    for k in range(4):
        ca, cb = rng.uniform(-3, 3, (12, 3)), rng.uniform(-3, 3, (18, 3))
        a = RawMesh((ca[:, None] + rng.normal(0, 1.0, (12, 3, 3))).reshape(-1, 3).astype(np.float32), np.arange(36).reshape(12, 3))
        b = RawMesh((cb[:, None] + rng.normal(0, 1.0, (18, 3, 3))).reshape(-1, 3).astype(np.float32), np.arange(54).reshape(18, 3))
        r, s01, s10 = eu.mean_distance_bounds(a, b, tol=1e-3, return_stats=True)
        assert r.converged and s01[3] > 0 and s10[3] > 0
        check_oracle(r, a, b, n=24)


def test_refused_inputs_and_counted_faces():
    b = big_quad(lambda x: np.full_like(x, 0.25))
    a = irregular_square()
    with pytest.raises(ValueError, match='tol'):
        eu.mean_distance_bounds(a, b, tol=-1.0)
    with pytest.raises(ValueError, match='outside'):
        eu.mean_distance_bounds(RawMesh(a._vertices['position'], [[0, 1, 9999]]), b)
    nan = RawMesh(np.array([[0, 0, 0], [1, 0, 0], [np.nan, 1, 0]], np.float32), [[0, 1, 2]])
    with pytest.raises(ValueError, match='no face with finite corners'):
        eu.mean_distance_bounds(nan, b)
    flat = RawMesh(np.array([[0, 0, 0], [1, 0, 0], [2, 0, 0]], np.float32), [[0, 1, 2], [0, 0, 1]])
    with pytest.raises(ValueError, match='zero total area'):
        eu.mean_distance_bounds(flat, b)
    h = _lib.Handle(0)
    try:
        t = np.random.default_rng(0).normal(size=(50, 3)).astype(np.float32)
        h.call('nw_set_point_targets', ctypes.c_void_p(t.ctypes.data), 0, len(t))
        with pytest.raises(ValueError, match='point targets'):
            eu._mean_distance_bounds(h, a, 0.01, 1000)
    finally:
        h.close()
    # a NaN-cornered face is skipped and a repeated-vertex face counted; neither changes the brackets
    v = np.concatenate([a._vertices['position'], [[np.nan, 0, 0]]]).astype(np.float32)
    mixed = RawMesh(v, np.concatenate([a.faces, [[len(v) - 1, 0, 1], [0, 0, 1]]]))
    r, s01, _ = eu.mean_distance_bounds(mixed, b, return_stats=True)
    ref = eu.mean_distance_bounds(a, b)
    assert s01[4] == 1 and s01[5] == 1 and tuple(r[0:4]) == tuple(ref[0:4]) and r.area0 == ref.area0


def _fit(mesh, pts, sig, probe):
    """Two nw_search calls of 4 iterations on a fresh handle; with `probe`, mean-distance calls run between them."""
    h = _lib.Handle(0)
    try:
        eu._upload_surface(h, mesh)
        s_inv = np.ascontiguousarray(1.0 / sig, dtype=np.float32)
        h.call('nw_set_points', ctypes.c_void_p(pts.ctypes.data), 0, len(pts), _lib.fptr(s_inv), 1.0, None)
        out = []
        for k in range(2):
            pos = np.empty((len(mesh._vertices), 3), np.float32)
            hist = [np.zeros(4) for _ in range(5)]
            n = ctypes.c_int(0)
            h.call('nw_search', 10.0, 4, 1, None, 0, _lib.fptr(pos), *[_lib.dptr(x) for x in hist], ctypes.byref(n))
            out.append((pos, hist))
            if probe and k == 0:
                eu._mean_distance_bounds(h, synth.star_mesh(synth.two_lobed(), 10), 0.01, 1 << 22)
        return out
    finally:
        h.close()


def test_no_side_effects_on_the_fit():
    shape = synth.two_lobed()
    mesh = synth.star_mesh(shape, 40)
    pts, sig = synth.smlm_cloud(shape, 4000, seed=11)
    for (pa, ha), (pb, hb) in zip(_fit(mesh, pts, sig, False), _fit(mesh, pts, sig, True)):
        assert np.array_equal(pa, pb)
        for x, y in zip(ha, hb):
            assert np.array_equal(x, y)

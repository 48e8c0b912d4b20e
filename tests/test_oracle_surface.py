"""The numpy exact point-to-triangle distance that nw_surface_distance is compared with (tests/surface_oracle.py), on cases
whose answer is known in closed form, and its candidate restriction against plain brute force.  CPU only."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import surface_oracle as orc  # noqa: E402

A, B, C = (0.0, 0.0, 0.0), (1.0, 0.0, 0.0), (0.0, 1.0, 0.0)


def closest(p, a=A, b=B, c=C):
    row = lambda v: np.asarray([v], np.float64)
    return orc.closest_point_triangle(row(p), row(a), row(b), row(c))[0]


@pytest.mark.parametrize('p, want', [
    ((0.25, 0.25, 2.0), (0.25, 0.25, 0.0)),      # above the interior
    ((0.25, 0.25, -3.0), (0.25, 0.25, 0.0)),     # below it
    ((-1.0, -1.0, 0.5), A),                      # vertex regions
    ((2.0, -0.5, 0.0), B),
    ((-0.5, 2.0, 1.0), C),
    ((0.5, -1.0, 0.0), (0.5, 0.0, 0.0)),         # beyond edge ab
    ((-1.0, 0.5, 3.0), (0.0, 0.5, 0.0)),         # beyond edge ca
    ((1.0, 1.0, 0.0), (0.5, 0.5, 0.0)),          # beyond edge bc
    (B, B),                                      # on a vertex
    ((0.5, 0.0, 0.0), (0.5, 0.0, 0.0)),          # on an edge
    ((0.125, 0.5, 0.0), (0.125, 0.5, 0.0)),      # in the triangle
])
def test_regions(p, want):
    assert np.array_equal(closest(p), np.asarray(want))


def test_degenerate_triangles_are_their_closest_edge():
    # collinear corners: the union of the segments is [0, 2] on the x axis
    assert np.array_equal(closest((3.0, 1.0, 0.0), (0.0, 0.0, 0.0), (2.0, 0.0, 0.0), (1.0, 0.0, 0.0)), [2.0, 0.0, 0.0])
    assert np.array_equal(closest((1.5, 0.0, 4.0), (0.0, 0.0, 0.0), (2.0, 0.0, 0.0), (1.0, 0.0, 0.0)), [1.5, 0.0, 0.0])
    # two equal corners
    assert np.array_equal(closest((0.5, -2.0, 0.0), (0.0, 0.0, 0.0), (1.0, 0.0, 0.0), (1.0, 0.0, 0.0)), [0.5, 0.0, 0.0])
    # a point triangle
    assert np.array_equal(closest((1.0, 2.0, 4.0), (1.0, 2.0, 3.0), (1.0, 2.0, 3.0), (1.0, 2.0, 3.0)), [1.0, 2.0, 3.0])


def test_surface_nearest_ties_go_to_the_lowest_face_row():
    verts = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [1, 1, 0], [0.5, 0.5, 5]], np.float32)
    faces = np.array([[0, 1, 2], [1, 3, 2]], np.int32)
    q = np.array([[0.5, 0.5, 1.0], [0.5, 0.5, -1.0], [1.0, 0.0, 0.0]])   # on the shared edge's normal; on a shared corner
    for order in (faces, faces[::-1].copy()):
        d, f, c = orc.surface_nearest(q, verts, order)
        assert np.array_equal(d, [1.0, 1.0, 0.0])
        assert np.array_equal(f, [0, 0, 0])
        assert np.array_equal(c, [[0.5, 0.5, 0.0], [0.5, 0.5, 0.0], [1.0, 0.0, 0.0]])


def test_surface_nearest_skips_non_finite_faces_and_queries():
    verts = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [np.nan, 0, 0], [0, 0, 10]], np.float32)
    faces = np.array([[0, 1, 3], [0, 1, 2], [0, 2, 4]], np.int32)
    d, f, c = orc.surface_nearest(np.array([[0.25, 0.25, -2.0], [np.inf, 0.0, 0.0]]), verts, faces)
    assert f.tolist() == [1, -1] and d[0] == 2.0 and np.isnan(d[1]) and np.isnan(c[1]).all()


def test_candidate_restriction_matches_brute_force():
    from ch_shrinkwrap_b200 import minimesh
    rng = np.random.default_rng(5)
    v, f = minimesh.geodesic_sphere(6)
    v = (v * 100.0 + rng.normal(0.0, 3.0, v.shape)).astype(np.float32)
    q = np.concatenate([rng.normal(0.0, 80.0, (300, 3)), rng.normal(0.0, 1000.0, (50, 3))])
    d, face, c = orc.surface_nearest(q, v, f)
    # every (query, face) pair
    v64 = v.astype(np.float64)
    qi, fi = np.repeat(np.arange(len(q)), len(f)), np.tile(np.arange(len(f)), len(q))
    cl = orc.closest_point_triangle(q[qi], v64[f[fi, 0]], v64[f[fi, 1]], v64[f[fi, 2]])
    d2 = orc._dist2(q[qi], cl).reshape(len(q), len(f))
    best = np.argmin(d2, 1)                         # first minimum = lowest row
    assert np.array_equal(face, best)
    assert np.array_equal(d, np.sqrt(d2[np.arange(len(q)), best]))
    assert np.array_equal(c, cl.reshape(len(q), len(f), 3)[np.arange(len(q)), best])

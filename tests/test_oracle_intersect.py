"""Known answers of the self-intersection restatement (tests/intersect_oracle.py), on the CPU."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import intersect_oracle as io  # noqa: E402
import signed_oracle as so  # noqa: E402


def pairs(v, f):
    return io.self_intersections(np.asarray(v, np.float32), np.asarray(f))[0].tolist()


T = [[0, 0, 0], [4, 0, 0], [0, 4, 0]]                     # a triangle in z = 0


def two(t1, t2):
    return np.array(t1 + t2, np.float32), [[0, 1, 2], [3, 4, 5]]


def test_crossing_triangles():
    assert pairs(*two(T, [[1, 1, -1], [1, 1, 1], [3, 3, 1]])) == [[0, 1]]
    assert pairs(*two(T, [[5, 5, -1], [5, 5, 1], [7, 7, 1]])) == []          # its line crosses the plane outside


@pytest.mark.parametrize('name,other,want', [
    ('point', [[1, 1, 0], [1, 1, 2], [3, 1, 2]], 1),              # a corner on the interior
    ('edge_on_edge', [[1, 0, 0], [3, 0, 0], [2, 0, 2]], 1),       # along an edge
    ('t_junction', [[1, 0, 0], [1, 0, 2], [3, 0, 2]], 1),         # a corner on an edge
    ('just_above', [[1, 1, 1e-3], [1, 1, 2], [3, 1, 2]], 0),
    ('corner_on_corner', [[4, 0, 0], [5, 0, 2], [5, 1, 2]], 1),   # same position, different vertex indices
])
def test_touching_counts(name, other, want):
    assert len(pairs(*two(T, other))) == want


def test_coplanar_overlap_and_disjoint():
    assert pairs(*two(T, [[1, 1, 0], [5, 1, 0], [1, 5, 0]])) == [[0, 1]]
    assert pairs(*two(T, [[3, 3, 0], [6, 3, 0], [3, 6, 0]])) == []              # beyond the hypotenuse
    assert pairs(*two(T, [[1, 1, 0], [2, 1, 0], [1, 2, 0]])) == [[0, 1]]        # inside, no edge crossing
    assert pairs(*two(T, [[2, 2, 0], [5, 2, 0], [2, 5, 0]])) == [[0, 1]]        # touches the hypotenuse at (2, 2)


def test_shared_edge_fold_over_versus_open():
    v = np.array([[0, 0, 0], [4, 0, 0], [0, 4, 0], [1, 1, 0], [4, 4, 0]], np.float32)
    assert pairs(v, [[0, 1, 2], [1, 2, 3]]) == [[0, 1]]       # (1,1,0) lies on the same side of edge 12 as vertex 0
    assert pairs(v, [[0, 1, 2], [1, 2, 4]]) == []             # planar, opposite sides: an ordinary flat edge
    w = v.copy()
    w[4, 2] = 1.0
    assert pairs(w, [[0, 1, 2], [1, 2, 4]]) == []             # a dihedral angle: not coplanar
    w = v.copy()
    w[3, 2] = 1e-3
    assert pairs(w, [[0, 1, 2], [1, 2, 3]]) == []             # folded, but not onto the plane: they meet only on the edge


def test_shared_vertex():
    v = np.array([[0, 0, 0], [4, 0, 0], [0, 4, 0], [1, 1, -1], [1, 1, 3]], np.float32)
    # the edge of the second face opposite the shared vertex 0 pierces the first
    assert pairs(v, [[0, 1, 2], [0, 3, 4]]) == [[0, 1]]
    v2 = v.copy()
    v2[3] = [-1, -1, -1]
    v2[4] = [-1, -2, 3]
    assert pairs(v2, [[0, 1, 2], [0, 3, 4]]) == []            # a fan around the shared vertex
    v3 = np.array([[0, 0, 0], [4, 0, 0], [0, 4, 0], [2, 1, 0], [1, 2, 0]], np.float32)
    assert pairs(v3, [[0, 1, 2], [0, 3, 4]]) == [[0, 1]]      # coplanar, one inside the other


def test_duplicate_faces_and_degenerate_faces():
    v = np.array([[0, 0, 0], [4, 0, 0], [0, 4, 0], [2, 0, 0], [1, 1, 0]], np.float32)
    assert pairs(v, [[0, 1, 2], [2, 0, 1]]) == [[0, 1]]       # three shared vertices
    p, deg, nf = io.self_intersections(v, np.array([[0, 1, 2], [0, 3, 1], [4, 4, 2]]))
    assert p.tolist() == [] and deg == 2 and nf == 0        # collinear corners, a repeated vertex
    w = v.copy()
    w[4] = [np.nan, 0, 0]
    p, deg, nf = io.self_intersections(w, np.array([[0, 1, 2], [4, 1, 2]]))
    assert p.tolist() == [] and deg == 0 and nf == 1


def test_one_ulp_near_coplanar():
    """A corner of the second triangle 1 ulp above / below / on the first's plane z = 1, touching its interior."""
    base = [[0, 0, 1], [4, 0, 1], [0, 4, 1]]
    one = np.float32(1)
    for z, want in ((np.nextafter(one, np.float32(2)), 0), (np.nextafter(one, np.float32(0)), 1), (one, 1)):
        v = np.array(base + [[1, 1, z], [1, 1, 3], [3, 1, 3]], np.float32)
        assert len(pairs(v, [[0, 1, 2], [3, 4, 5]])) == want, z


def test_one_ulp_fold_over_on_a_tilted_plane():
    """On the plane z = x + y (exact in float32 for these values) a shared-edge fold-over counts only while exactly coplanar."""
    v = np.array([[0, 0, 0], [4, 0, 4], [0, 4, 4], [1, 1, 2]], np.float32)
    f = [[0, 1, 2], [1, 2, 3]]
    assert pairs(v, f) == [[0, 1]]
    w = v.copy()
    w[3, 2] = np.nextafter(np.float32(2), np.float32(3))
    assert pairs(w, f) == []


def test_tiny_and_huge_coordinates():
    s, b = np.float32(1e-30), np.float32(1e30)
    v = np.array([[0, 0, 0], [b, 0, 0], [0, b, 0], [s, s, -s], [s, s, s], [2 * s, 3 * s, s]], np.float32)
    assert pairs(v, [[0, 1, 2], [3, 4, 5]]) == [[0, 1]]       # a tiny triangle through a huge one
    v[3, 2] = s / 2
    assert pairs(v, [[0, 1, 2], [3, 4, 5]]) == []             # now entirely above it
    v[3, 2] = 0.0
    assert pairs(v, [[0, 1, 2], [3, 4, 5]]) == [[0, 1]]       # touching it at one corner


def test_scale_permutation_and_winding_invariance():
    v, f = so.sphere(3)
    v = np.concatenate([v, v + np.float32(15.0)]).astype(np.float32)
    f = np.concatenate([f, f + len(v) // 2])
    want = pairs(v, f)
    assert len(want) > 0
    for k in (60, -60):
        assert pairs(v * np.float32(2.0 ** k), f) == want
    assert pairs(v, f[:, [0, 2, 1]]) == want
    perm = np.random.default_rng(0).permutation(len(f))
    got = pairs(v, f[perm])
    mapped = sorted(sorted((int(perm[i]), int(perm[j]))) for i, j in got)
    assert mapped == want


SOLIDS = {'tetrahedron': so.tetrahedron, 'prism': so.prism, 'cube': so.cube, 'l_polycube': so.l_polycube,
          'sphere': so.sphere, 'torus': so.torus}


@pytest.mark.parametrize('name', sorted(SOLIDS))
def test_solids_are_embedded(name):
    v, f = SOLIDS[name]()
    p, deg, nf = io.self_intersections(v, f)
    assert p.tolist() == [] and deg == 0 and nf == 0

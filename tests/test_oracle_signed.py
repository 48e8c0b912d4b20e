"""The numpy signed distance that nw_surface_signed_distance is compared with (tests/signed_oracle.py), against the
generalised winding number on closed solids with sharp, concave and saddle features, and its defect counts on meshes that do
not bound a solid.  CPU only."""
import collections
import math
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import signed_oracle as so  # noqa: E402

SOLIDS = {'tetrahedron': so.tetrahedron, 'prism': so.prism, 'cube': so.cube, 'l_polycube': so.l_polycube,
          'sphere': so.sphere, 'torus': so.torus}


def _check_against_winding(v, f, seed=0):
    q = so.feature_queries(v, f, seed=seed)
    sd, face, _, V, margin, region = so.signed_distance(q, v, f)
    inside = np.abs(so.winding_number(q, v, f)) > 0.5
    far = np.abs(sd) > 1e-6 * float((v.max(0) - v.min(0)).max())
    assert far.sum() > 0.9 * len(q)
    assert np.array_equal((sd < 0)[far], inside[far])
    return q, sd, face, V, margin, region, inside, far


@pytest.mark.parametrize('name', sorted(SOLIDS))
@pytest.mark.parametrize('reverse', [False, True])
def test_sign_matches_the_winding_number(name, reverse):
    v, f = SOLIDS[name]()
    if reverse:
        f = np.ascontiguousarray(f[:, [0, 2, 1]])
    assert so.tables(f, len(v))[3] == [0, 0, 0, 0, 0]
    _, sd, *_ = _check_against_winding(v, f)
    assert not np.isnan(sd).any()


@pytest.mark.parametrize('name', ['tetrahedron', 'prism'])
def test_sharp_solids_need_the_pseudonormal(name):
    """Dihedral angles under 90 degrees: queries near corners and edges land in vertex and edge regions, and the winning
    face's own normal puts some of them on the wrong side."""
    v, f = SOLIDS[name]()
    q, sd, face, _, _, region, inside, far = _check_against_winding(v, f)
    assert ((region >= so.CORNER) & (region < so.EDGE)).sum() > 0 and (region >= so.EDGE).sum() > 0
    naive = so.face_normal_side(q, v, f, face)
    assert (((naive < 0) != inside) & far).sum() > 0


@pytest.mark.parametrize('name', sorted(SOLIDS))
def test_reversed_winding_keeps_the_volume_and_the_sides(name):
    v, f = SOLIDS[name]()
    q = so.feature_queries(v, f, seed=1)
    sd, _, _, V, margin, _ = so.signed_distance(q, v, f)
    sr, _, _, Vr, _, _ = so.signed_distance(q, v, np.ascontiguousarray(f[:, [0, 2, 1]]))
    assert V == Vr
    ok = margin >= 1e-9
    assert np.array_equal(np.sign(sd[ok]), np.sign(sr[ok]))


@pytest.mark.parametrize('name', sorted(SOLIDS))
def test_volume_is_the_sum_of_its_terms(name):
    v, f = SOLIDS[name]()
    t = so.volume_terms(v, f)
    V = so.fixed_order_sum(t)
    assert abs(V - math.fsum(t)) <= 1e-12 * abs(math.fsum(t))
    want = {'cube': 1000.0, 'l_polycube': 5000.0, 'tetrahedron': 8000.0 / 3.0}.get(name)   # 10^3 per cell; (2*10)^3 / 3
    if want is not None:
        assert abs(V - want) <= 1e-12 * want


def test_surface_points_are_zero_and_the_far_field_is_outside():
    v, f = so.sphere()
    q = np.concatenate([v.astype(np.float64), [[0.0, 0.0, 0.0], [1e4, 0.0, 0.0]]])
    sd, face, *_ = so.signed_distance(q, v, f)
    assert np.all(sd[:len(v)] == 0.0) and sd[-2] < 0.0 and sd[-1] > 0.0


def test_torus_hole_is_outside():
    v, f = so.torus()
    sd, *_ = so.signed_distance(np.array([[0.0, 0.0, 0.0], [0.0, 0.0, 5.0], [30.0, 0.0, 0.0]]), v, f)
    assert sd[0] > 0.0 and sd[1] > 0.0 and sd[2] < 0.0


def _boundary_edges(f):
    c = collections.Counter(tuple(sorted(e)) for row in f.tolist() for e in zip(row, row[1:] + row[:1]))
    return sum(1 for n in c.values() if n == 1)


def defect_meshes():
    """(name, vertices, faces, expected counts) for meshes that do not bound a solid."""
    from ch_shrinkwrap_b200 import minimesh
    v, f = so.sphere(4)
    out = [('open', v, f[1:], [3, 0, 0, 0, 0])]
    g = f.copy()
    g[7] = g[7, [0, 2, 1]]
    out.append(('flipped', v, g, [0, 0, 3, 0, 0]))
    a, b = f[0, 0], f[0, 1]
    vf = np.concatenate([v, [v[a] * 1.5]]).astype(np.float32)
    out.append(('fin', vf, np.concatenate([f, [[a, b, len(v)]]]).astype(np.int32), [2, 1, 0, 0, 0]))
    tv, tf = so.tetrahedron()
    t2v = np.concatenate([tv, -tv[1:] + 2 * tv[0]]).astype(np.float32)     # the second one mirrored through vertex 0
    t2f = np.where(tf == 0, 0, tf + 3)[:, [0, 2, 1]]
    out.append(('shared_vertex', t2v, np.concatenate([tf, t2f]).astype(np.int32), [0, 0, 0, 0, 1]))
    pm = minimesh.planar_mesh(100.0, 6)
    out.append(('planar', pm._vertices['position'], pm.faces, [_boundary_edges(pm.faces), 0, 0, 0, 0]))
    return out


@pytest.mark.parametrize('case', defect_meshes(), ids=lambda c: c[0])
def test_defect_counts_are_exact(case):
    _, v, f, want = case
    assert so.tables(f, len(v))[3] == want
    if case[0] == 'planar':
        assert want[0] == 4 * 6


def test_twins_and_csr_of_a_closed_mesh():
    v, f = so.sphere(3)
    twin, voff, vface, _ = so.tables(f, len(v))
    for r in range(len(f)):
        for k in range(3):
            g = twin[r, k]
            u, w = f[r, k], f[r, (k + 1) % 3]
            assert g != r and any((f[g, j], f[g, (j + 1) % 3]) == (w, u) for j in range(3))
    for vi in range(len(v)):
        rows = vface[voff[vi]:voff[vi + 1]]
        assert np.array_equal(rows, np.flatnonzero((f == vi).any(1)))

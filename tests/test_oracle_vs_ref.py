"""Live check of the oracle restatement against the reference itself (only where oracle/refharness.py can import it)."""
import copy

import numpy as np
import pytest

from conftest import make_case

pytestmark = pytest.mark.needs_reference


def test_search_bitwise_vs_reference():
    from oracle import nanowrap_oracle as orc
    from oracle import refharness
    mesh, pts, sig = make_case(n_points=2000, n_geo=4, seed=31)
    m_ref, m_orc = copy.deepcopy(mesh), copy.deepcopy(mesh)
    s = (1.0 / sig.ravel()).astype(np.float32)
    cg = refharness.reference_solver(m_ref, pts)
    vr = cg.search(pts, lams=[10.0], num_iters=5, sigma_inv=s)
    oc = orc.OracleConjGrad(m_orc, pts)
    vo = oc.search(pts, lams=[10.0], num_iters=5, sigma_inv=s)
    assert np.array_equal(vr, vo) and np.array_equal(cg.S, oc.S) and np.array_equal(cg.res, oc.res)
    assert np.array_equal(cg.w[1], oc.w[1]) and cg.tests == oc.tests


def test_search_weights_mask_vs_reference():
    from oracle import nanowrap_oracle as orc
    from oracle import refharness
    mesh, pts, sig = make_case(n_points=1500, n_geo=4, seed=32, dtype=np.float64)
    m_ref, m_orc = copy.deepcopy(mesh), copy.deepcopy(mesh)
    s = 1.0 / sig.ravel()
    w = s.copy()
    w[::5] = 0
    cg = refharness.reference_solver(m_ref, pts)
    vr = cg.search(pts, lams=[3.0], num_iters=3, sigma_inv=s, weights=w)
    oc = orc.OracleConjGrad(m_orc, pts)
    vo = oc.search(pts, lams=[3.0], num_iters=3, sigma_inv=s, weights=w)
    assert np.array_equal(vr, vo)


def test_curvature_bitwise_vs_reference_including_jitter():
    from ch_shrinkwrap_b200 import synth
    from oracle import nanowrap_oracle as orc
    from oracle import refharness
    m = synth.star_mesh(synth.two_lobed(), 8, scale=1.0)
    nv = int((m._vertices['halfedge'] != -1).sum())
    r = refharness.reference_curvature(m, seed=9)
    o = orc.curvature_grad(m, jitter_u=refharness.libc_uniforms(9, 3 * nv))
    for k in r:
        assert np.array_equal(r[k], o[k], equal_nan=True), k


def test_c_helpers_bitwise_vs_reference():
    from oracle import nanowrap_oracle as orc
    from oracle import refharness
    _, cgu = refharness.load_reference()
    rng = np.random.default_rng(3)
    P, M = 5000, 300
    v_idx = rng.integers(0, M, (P, 3)).astype(np.int32)
    w = rng.random((P, 3)).astype(np.float32)
    fv = rng.standard_normal((P, 3)).astype(np.float32)
    a = np.zeros((M, 3), np.float32)
    b = np.zeros((M, 3), np.float32)
    cgu.c_shrinkwrap_ah_helper(v_idx, w, fv, a)
    orc.ah_scatter(v_idx, w, fv, b)
    assert np.array_equal(a, b)


def test_quality_metrics_and_holepunch_vs_reference():
    from ch_shrinkwrap_b200 import synth
    from oracle import nanowrap_oracle as orc
    from oracle import refharness
    evu = refharness.load_evaluation_utils()
    m = synth.star_mesh(synth.two_lobed(), 5, scale=1.0)
    np.random.seed(3)
    d_ref = evu.points_from_mesh(m, dx_min=12)
    d_orc = orc.points_from_mesh_samples(m, 12)
    np.random.seed(3)
    perm = np.random.choice(np.arange(len(d_orc)), size=len(d_orc), replace=False)
    assert np.array_equal(d_orc[perm], d_ref)                       # same samples, same permutation for the same seed
    rng = np.random.default_rng(1)
    a = rng.standard_normal((4000, 3)) * 100
    b = a[:2500] + rng.standard_normal((2500, 3))
    assert evu.average_squared_distance(a, b) == orc.average_squared_distance(a, b)
    cand = np.arange(len(m._faces), dtype=np.int32)
    assert np.array_equal(refharness.reference_holepunch_pairs(m, cand), orc.holepunch_pairs(m, cand))


def test_search_with_the_wfunc_regulariser_vs_reference():
    """mesh_conj_grad.py:39 -- the one alternative regulariser the reference's search() can run with: bit-exact too."""
    from oracle import nanowrap_oracle as orc
    from oracle import refharness
    mesh, pts, sig = make_case(n_points=2000, n_geo=4, seed=33)
    m_ref, m_orc = copy.deepcopy(mesh), copy.deepcopy(mesh)
    s = (1.0 / sig.ravel()).astype(np.float32)
    cg = refharness.reference_solver(m_ref, pts)
    cg.Lfuncs, cg.Lhfuncs = ["wfunc"], ["wfunc"]
    vr = cg.search(pts, lams=[10.0], num_iters=4, sigma_inv=s)
    oc = orc.OracleConjGrad(m_orc, pts)
    oc.Lfuncs, oc.Lhfuncs = ["wfunc"], ["wfunc"]
    vo = oc.search(pts, lams=[10.0], num_iters=4, sigma_inv=s)
    assert np.array_equal(vr, vo) and np.array_equal(cg.S, oc.S) and cg.tests == oc.tests
    # and the operators the reference cannot run with raise there too (float64 argument read as float32 by the C helper)
    cg2 = refharness.reference_solver(copy.deepcopy(mesh), pts)
    cg2.Lfuncs, cg2.Lhfuncs = ["Lfunc3"], ["Lhfunc3"]
    with pytest.raises(AssertionError):
        cg2.search(pts, lams=[10.0], num_iters=1, sigma_inv=s)

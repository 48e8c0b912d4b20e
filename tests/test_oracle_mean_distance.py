"""The Lipschitz bracket of tests/mean_distance_oracle.py against closed forms, on the CPU."""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import mean_distance_oracle as mo  # noqa: E402


def square(z=0.0, lo=0.0, hi=1.0):
    v = np.array([[lo, lo, z], [hi, lo, z], [hi, hi, z], [lo, hi, z]], np.float32)
    return v, np.array([[0, 1, 2], [0, 2, 3]], np.int32)


def test_subdivision_keeps_the_area_and_covers_the_triangle():
    t = np.array([[[0.0, 0.0, 0.0], [3.0, 0.0, 0.0], [0.5, 2.0, 0.0]]])
    for n in (1, 2, 5):
        s = mo.subdivide(t, n)
        a = 0.5 * np.abs(np.cross(s[:, 1] - s[:, 0], s[:, 2] - s[:, 0])[:, 2])
        assert len(s) == n * n and np.allclose(a, 3.0 / n ** 2)


def test_parallel_squares_and_a_crossing_plane():
    va, fa = square()
    vb, fb = square(0.25, -2.0, 3.0)
    A, mean, rms = mo.mean_distance_bracket(va, fa, vb, fb, n=4)
    assert A == 1.0 and mean[0] <= 0.25 <= mean[1] and rms[0] <= 0.25 <= rms[1]
    _, mean16, _ = mo.mean_distance_bracket(va, fa, vb, fb, n=16)
    assert mean[0] < mean16[0] and mean16[1] < mean[1]                      # a finer subdivision narrows the bracket
    # the plane z = x - 0.5: d = |x - 0.5| / sqrt(2) over the unit square
    vp = np.array([[-8, -8, -8.5], [12, -8, 11.5], [12, 12, 11.5], [-8, 12, -8.5]], np.float32)
    fp = np.array([[0, 1, 2], [0, 2, 3]], np.int32)
    for n in (4, 16):
        _, mean, rms = mo.mean_distance_bracket(va, fa, vp, fp, n=n)
        assert mean[0] <= 1.0 / (4.0 * np.sqrt(2.0)) <= mean[1] and rms[0] <= np.sqrt(1.0 / 24.0) <= rms[1]
    assert mean[1] - mean[0] < 0.1 and rms[1] - rms[0] < 0.1


def test_non_finite_faces_are_left_out():
    va, fa = square()
    va = np.concatenate([va, [[np.nan, 0.0, 0.0]]]).astype(np.float32)
    fa = np.concatenate([fa, [[0, 1, 4]]]).astype(np.int32)
    assert np.allclose(mo.face_areas(va, fa), [0.5, 0.5])

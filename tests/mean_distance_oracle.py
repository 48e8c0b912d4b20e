"""CPU checks for nw_mean_distance_bounds (ch_shrinkwrap_b200/csrc/hausdorff.cu), test infrastructure only: a Lipschitz
bracket of the area-weighted mean and RMS distance from a mesh A to a mesh B, from a uniform barycentric subdivision of A's
finite faces and the brute-force nearest face of surface_oracle.py.

On a sub-triangle of area w with centroid distance delta, every point lies within r of the centroid, r the largest
centroid-to-corner distance (not the circumradius, which a sliver can undercut), and d_B is 1-Lipschitz, so
  integral of d_B   in [w max(0, delta - r),   w (delta + r)],
  integral of d_B^2 in [w max(0, delta - r)^2, w (delta + r)^2]."""
from __future__ import annotations

import numpy as np

import surface_oracle as orc


def finite_faces(vertices, faces):
    v = np.asarray(vertices, np.float32).astype(np.float64)
    f = np.asarray(faces, np.int64)
    return v[f[np.isfinite(v[f]).all((1, 2))]]                                         # (F, 3, 3)


def face_areas(vertices, faces):
    """The area of every finite face, float64."""
    t = finite_faces(vertices, faces)
    return 0.5 * np.sqrt((np.cross(t[:, 1] - t[:, 0], t[:, 2] - t[:, 0]) ** 2).sum(1))


def subdivide(tris, n):
    """The n^2 sub-triangles of the uniform barycentric subdivision of each triangle: (F n^2, 3, 3)."""
    ups = [((i, j), (i + 1, j), (i, j + 1)) for i in range(n) for j in range(n - i)]
    downs = [((i + 1, j), (i + 1, j + 1), (i, j + 1)) for i in range(n) for j in range(n - i - 1)]
    idx = np.array(ups + downs, np.float64) / n                                        # (n^2, 3 corners, (u, v))
    w = np.stack([1.0 - idx[..., 0] - idx[..., 1], idx[..., 0], idx[..., 1]], -1)    # (n^2, 3, 3) barycentric
    return np.einsum('skc,fcd->fskd', w, tris).reshape(-1, 3, 3)


def mean_distance_bracket(vertices_a, faces_a, vertices_b, faces_b, n=8):
    """(area, [mean_lo, mean_hi], [rms_lo, rms_hi]) of A -> B by the Lipschitz bracket above."""
    tris = finite_faces(vertices_a, faces_a)
    area = face_areas(vertices_a, faces_a)
    sub = subdivide(tris, n)
    w = np.repeat(area / n ** 2, n * n)
    g = sub.mean(1)
    r = np.sqrt(((sub - g[:, None]) ** 2).sum(2)).max(1)
    delta = orc.surface_nearest(g, vertices_b, faces_b)[0]
    lo, hi = np.maximum(delta - r, 0.0), delta + r
    A = area.sum()
    return A, ((w * lo).sum() / A, (w * hi).sum() / A), (np.sqrt((w * lo * lo).sum() / A), np.sqrt((w * hi * hi).sum() / A))

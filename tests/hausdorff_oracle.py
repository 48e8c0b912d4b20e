"""CPU checks for nw_hausdorff_bounds (ch_shrinkwrap_b200/csrc/hausdorff.cu), test infrastructure only: dense barycentric
samples of a mesh A measured against a mesh B with the brute-force nearest face of surface_oracle.py, and the rounding
allowance the call states."""
from __future__ import annotations

import numpy as np

import surface_oracle as orc


def barycentric_samples(vertices, faces, n=4):
    """Per finite face: its corners, n - 1 points inside each edge and the interior points of the barycentric grid of step
    1 / n, float64 (duplicates across shared edges are kept)."""
    v = np.asarray(vertices, np.float32).astype(np.float64)
    f = np.asarray(faces, np.int64)
    f = f[np.isfinite(v[f]).all((1, 2))]
    ij = np.array([(i, j) for i in range(n + 1) for j in range(n + 1 - i)], np.float64) / n
    w = np.stack([1.0 - ij[:, 0] - ij[:, 1], ij[:, 0], ij[:, 1]], 1)                  # (S, 3) barycentric weights
    return np.einsum('sk,fkd->fsd', w, v[f]).reshape(-1, 3)


def max_sample_distance(vertices_a, faces_a, vertices_b, faces_b, n=4):
    """The largest exact distance from the dense samples of A to B's closed triangles."""
    d = orc.surface_nearest(barycentric_samples(vertices_a, faces_a, n), vertices_b, faces_b)[0]
    return float(np.nanmax(d))


def rounding_allowance(*vertex_arrays):
    """The eps of nw_hausdorff_bounds: 2^-40 x the sum over the axes of the largest finite |coordinate| (float32)."""
    m = np.zeros(3)
    for v in vertex_arrays:
        a = np.abs(np.asarray(v, np.float32).astype(np.float64))
        a[~np.isfinite(a)] = 0.0
        m = np.maximum(m, a.max(0))
    return float(m.sum()) * 2.0 ** -40

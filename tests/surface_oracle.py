"""CPU restatement of nw_surface_distance (ch_shrinkwrap_b200/csrc/surface.cu), test infrastructure only.

The library's exact point-to-triangle routine restated in numpy, operation for operation in fp64 (the library compiles it
with -fmad=false), so that distances, closest points and faces compare bit for bit; with the region code of the closest
point, which the signed distance (signed_oracle.py) reads.  Plus a brute-force nearest face with the same tie rule.  Not a
reference feature, so it lives beside the tests rather than in the reference oracle (oracle/)."""
from __future__ import annotations

import numpy as np
import scipy.spatial


CORNER, EDGE = 1, 4                      # region codes: 0 interior, CORNER + k corner k, EDGE + k the edge corner k -> k + 1


def dot(u, v):
    return (u[:, 0] * v[:, 0] + u[:, 1] * v[:, 1]) + u[:, 2] * v[:, 2]


def _dist2(p, c):
    d = p - c
    return dot(d, d)


def _closest_on_segment(p, p0, p1, k):
    """(closest point, region code) on the segment p0 -> p1, taken as edge k of a triangle."""
    e = p1 - p0
    ee = dot(e, e)
    with np.errstate(divide='ignore', invalid='ignore'):
        t = np.where(ee > 0.0, dot(p - p0, e) / ee, 0.0)
    t = np.fmin(np.fmax(t, 0.0), 1.0)
    return p0 + t[:, None] * e, np.where(t == 0.0, CORNER + k, np.where(t == 1.0, CORNER + (k + 1) % 3, EDGE + k))


def _closest_on_edges(p, a, b, c):
    """A zero-area triangle is the union of its edges: the closest of ab, bc, ca (the first wins ties)."""
    best, r = _closest_on_segment(p, a, b, 0)
    bd = _dist2(p, best)
    for k, (u, v) in ((1, (b, c)), (2, (c, a))):
        x, rk = _closest_on_segment(p, u, v, k)
        kd = _dist2(p, x)
        m = kd < bd
        best = np.where(m[:, None], x, best)
        bd = np.where(m, kd, bd)
        r = np.where(m, rk, r)
    return best, r


def closest_point_region(p, a, b, c):
    """(closest point, region code) on the closed triangle (a, b, c) to p, row by row, float64 (N,3) arrays: Ericson's
    region test (Real-Time Collision Detection 5.1.5).  Degenerate: ab x ac is exactly zero, or the interior case finds no
    positive barycentric denominator; then the closest of the three edges as segments."""
    ab, ac = b - a, c - a
    degenerate = ((ab[:, 1] * ac[:, 2] - ab[:, 2] * ac[:, 1] == 0.0) & (ab[:, 2] * ac[:, 0] - ab[:, 0] * ac[:, 2] == 0.0)
                  & (ab[:, 0] * ac[:, 1] - ab[:, 1] * ac[:, 0] == 0.0))
    ap, bp, cp = p - a, p - b, p - c
    d1, d2 = dot(ab, ap), dot(ac, ap)
    d3, d4 = dot(ab, bp), dot(ac, bp)
    d5, d6 = dot(ab, cp), dot(ac, cp)
    vc = d1 * d4 - d3 * d2
    vb = d5 * d2 - d1 * d6
    va = d3 * d6 - d5 * d4
    s = va + vb + vc
    with np.errstate(divide='ignore', invalid='ignore'):
        on_ab = a + (d1 / (d1 - d3))[:, None] * ab
        on_ac = a + (d2 / (d2 - d6))[:, None] * ac
        on_bc = b + ((d4 - d3) / ((d4 - d3) + (d5 - d6)))[:, None] * (c - b)
        denom = 1.0 / s
        v, w = vb * denom, vc * denom
        inner = (a + ab * v[:, None]) + ac * w[:, None]
    edges, edges_r = _closest_on_edges(p, a, b, c)
    out, r = np.where((s > 0.0)[:, None], inner, edges), np.where(s > 0.0, 0, edges_r)
    # the regions in reverse order of precedence, so that the first that holds is the one left standing
    for holds, x, code in (((va <= 0.0) & ((d4 - d3) >= 0.0) & ((d5 - d6) >= 0.0), on_bc, EDGE + 1),
                           ((vb <= 0.0) & (d2 >= 0.0) & (d6 <= 0.0), on_ac, EDGE + 2),
                           ((d6 >= 0.0) & (d5 <= d6), c, CORNER + 2),
                           ((vc <= 0.0) & (d1 >= 0.0) & (d3 <= 0.0), on_ab, EDGE + 0),
                           ((d3 >= 0.0) & (d4 <= d3), b, CORNER + 1),
                           ((d1 <= 0.0) & (d2 <= 0.0), a, CORNER + 0)):
        out, r = np.where(holds[:, None], x, out), np.where(holds, code, r)
    return np.where(degenerate[:, None], edges, out), np.where(degenerate, edges_r, r)


def closest_point_triangle(p, a, b, c):
    """The closest point of ``closest_point_region``."""
    return closest_point_region(p, a, b, c)[0]


def surface_nearest(points, vertices, faces, chunk=1 << 21):
    """Brute-force nearest closed triangle per query, nw_surface_distance's contract: (dist float64, face int32 = row of
    `faces`, closest (Q,3) float64).  Exact fp64 ties go to the lowest row; faces with a non-finite corner are skipped; a
    non-finite query gets NaN, -1, NaN.  Points keep their dtype's values (float32 widened exactly).

    Candidates: the distance d_c to the nearest centroid bounds the answer from above (a centroid lies on its triangle), so
    a face can only win if its centroid is within d_c + R of the query, R = the largest corner-to-centroid distance."""
    q = np.asarray(points).astype(np.float64)
    v = np.asarray(vertices, np.float32).astype(np.float64)
    f = np.asarray(faces, np.int64)
    A, B, C = v[f[:, 0]], v[f[:, 1]], v[f[:, 2]]
    fid = np.flatnonzero(np.isfinite(A).all(1) & np.isfinite(B).all(1) & np.isfinite(C).all(1))
    Q = len(q)
    dist = np.full(Q, np.nan)
    face = np.full(Q, -1, np.int32)
    closest = np.full((Q, 3), np.nan)
    qi_ok = np.flatnonzero(np.isfinite(q).all(1))
    if len(fid) == 0 or len(qi_ok) == 0:
        return dist, face, closest
    cent = (A[fid] + B[fid] + C[fid]) / 3.0
    R = max(float(np.sqrt(((X[fid] - cent) ** 2).sum(1)).max()) for X in (A, B, C))
    tree = scipy.spatial.cKDTree(cent)
    dc, _ = tree.query(q[qi_ok], k=1, workers=-1)
    cands = tree.query_ball_point(q[qi_ok], (dc + R) * (1.0 + 1e-7) + 1e-12, workers=-1)
    n = np.array([len(c) for c in cands])
    qi = np.repeat(qi_ok, n)
    fi = fid[np.concatenate([np.asarray(c, np.int64) for c in cands])]
    d2 = np.empty(len(qi))
    cl = np.empty((len(qi), 3))
    for s in range(0, len(qi), chunk):
        e = min(len(qi), s + chunk)
        p, k = q[qi[s:e]], fi[s:e]
        cl[s:e] = closest_point_triangle(p, A[k], B[k], C[k])
        d2[s:e] = _dist2(p, cl[s:e])
    order = np.lexsort((fi, d2, qi))                     # per query: smallest d2, then lowest face row
    first = order[np.r_[True, qi[order][1:] != qi[order][:-1]]]
    dist[qi[first]] = np.sqrt(d2[first])
    face[qi[first]] = fi[first]
    closest[qi[first]] = cl[first]
    return dist, face, closest

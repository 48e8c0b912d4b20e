"""Independent restatement of nw_self_intersections (intersect.cu) in exact rational arithmetic.

The GPU decides every contact from signs of orientation determinants.  This module does not: it converts the float32
coordinates to exact integers (multiples of 2^-149), computes the point where a segment crosses a triangle's plane as an
explicit rational point, and checks that point's barycentric coordinates; in the coplanar case it clips the segment's
parameter interval against the triangle's barycentric constraints.  A conservative fp64 broad phase (bounding boxes, then a
plane-side test with a wide error margin) keeps it fast enough for a few thousand faces, or for the faces near a few
thousand of interest in a large mesh.

The contract (faces f < g, rows of `faces`): no shared vertex index -- the closed triangles share any point; one shared
vertex s -- the edge of either face opposite s meets the other closed triangle; a shared edge uv with opposite corners p, q
-- p, q coplanar with uv and strictly on the same side of it; three shared -- always.  Degenerate faces (collinear corners)
and faces with a non-finite corner are left out and counted."""
from fractions import Fraction

import numpy as np

SCALE = 2 ** 149


class Exact:
    """Vertex coordinates as exact integers (x * 2^149), converted on first use."""

    def __init__(self, vertices):
        self.v = np.asarray(vertices, np.float32)
        self.cache = {}

    def __getitem__(self, i):
        i = int(i)
        p = self.cache.get(i)
        if p is None:
            p = tuple(int(Fraction(float(c)) * SCALE) for c in self.v[i])
            self.cache[i] = p
        return p


def sub(a, b):
    return (a[0] - b[0], a[1] - b[1], a[2] - b[2])


def cross(a, b):
    return (a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0])


def dot(a, b):
    return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]


def barycentric(x, a, n, e1, e2):
    """(u, v) with x = a + u e1 + v e2, for x in the plane of the triangle (normal n = e1 x e2 != 0), as Fractions: Cramer's
    rule in the axis plane where n has its largest component."""
    k = max(range(3), key=lambda j: abs(n[j]))
    i, j = [(1, 2), (2, 0), (0, 1)][k]
    w = [x[m] - a[m] for m in range(3)]
    den = e1[i] * e2[j] - e1[j] * e2[i]
    return Fraction(w[i] * e2[j] - w[j] * e2[i]) / den, Fraction(e1[i] * w[j] - e1[j] * w[i]) / den


def segment_meets_triangle(p, q, a, b, c):
    """The closed segment pq and the closed, non-degenerate triangle abc share a point."""
    e1, e2 = sub(b, a), sub(c, a)
    n = cross(e1, e2)
    sp, sq = dot(n, sub(p, a)), dot(n, sub(q, a))
    if (sp > 0 and sq > 0) or (sp < 0 and sq < 0):
        return False
    if sp != 0 or sq != 0:
        t = Fraction(sp, sp - sq)                                # the crossing point p + t (q - p), t in [0, 1]
        x = [p[m] + t * (q[m] - p[m]) for m in range(3)]
        u, v = barycentric(x, a, n, e1, e2)
        return u >= 0 and v >= 0 and u + v <= 1
    # coplanar: the barycentric coordinates are affine in t; clip [0, 1] by u >= 0, v >= 0, 1 - u - v >= 0
    u0, v0 = barycentric(p, a, n, e1, e2)
    u1, v1 = barycentric(q, a, n, e1, e2)
    lo, hi = Fraction(0), Fraction(1)
    for f0, f1 in ((u0, u1), (v0, v1), (1 - u0 - v0, 1 - u1 - v1)):
        d = f1 - f0                                              # f(t) = f0 + t d >= 0
        if d == 0:
            if f0 < 0:
                return False
        elif d > 0:
            lo = max(lo, -f0 / d)
        else:
            hi = min(hi, -f0 / d)
    return lo <= hi


def pair_intersects(fi, gi, X):
    """The contract for two tested faces given as vertex-index triples."""
    shared = set(fi) & set(gi)
    if len(shared) == 3:
        return True
    P = [X[i] for i in fi]
    Q = [X[i] for i in gi]
    if len(shared) == 2:
        u, v = (X[i] for i in shared)
        p = X[next(i for i in fi if i not in shared)]
        q = X[next(i for i in gi if i not in shared)]
        m = cross(sub(v, u), sub(p, u))
        if dot(m, sub(q, u)) != 0:
            return False
        return dot(m, cross(sub(v, u), sub(q, u))) > 0           # both normals point the same way: q on p's side
    if len(shared) == 1:
        s = next(iter(shared))
        ef = [X[i] for i in fi if i != s]
        eg = [X[i] for i in gi if i != s]
        return segment_meets_triangle(ef[0], ef[1], *Q) or segment_meets_triangle(eg[0], eg[1], *P)
    for k in range(3):
        if segment_meets_triangle(P[k], P[(k + 1) % 3], *Q) or segment_meets_triangle(Q[k], Q[(k + 1) % 3], *P):
            return True
    return False


def _separated(a, b, c, corners):
    """fp64, conservative: True where all three corners (k, 3, 3) lie strictly on one side of the plane of a, b, c (each
    (k, 3) or (3,)), by a margin far above the rounding of the computation."""
    n = np.cross(b - a, c - a)
    nn = np.abs(b - a).sum(-1) * np.abs(c - a).sum(-1)       # bounds |n| and its rounding, cancellation or not
    d = corners - np.asarray(a)[..., None, :]
    s = (d * np.asarray(n)[..., None, :]).sum(-1)
    tol = 1e-9 * np.asarray(nn)[..., None] * np.abs(d).sum(-1).max(-1, keepdims=True)
    return np.all(s > tol, -1) | np.all(s < -tol, -1)


def candidates(vertices, faces, tested, subset=None):
    """Pairs (i, j), i < j, of tested faces whose bounding boxes overlap and that no fp64 plane-side test separates; with
    `subset`, only pairs with at least one face in it."""
    v = np.asarray(vertices, np.float64)
    f = np.asarray(faces, np.int64)
    tri = v[f]
    lo, hi = tri.min(1), tri.max(1)
    idx = np.flatnonzero(tested)
    rows = idx if subset is None else np.intersect1d(np.asarray(subset, np.int64), idx)
    out = []
    for r in rows:
        j = idx[np.all((lo[r] <= hi[idx]) & (hi[r] >= lo[idx]), 1)]
        j = j[j != r]
        j = j[~_separated(tri[r, 0], tri[r, 1], tri[r, 2], tri[j])]
        j = j[~_separated(tri[j, 0], tri[j, 1], tri[j, 2], np.broadcast_to(tri[r], (len(j), 3, 3)))]
        out.append(np.stack([np.minimum(r, j), np.maximum(r, j)], 1))
    if not out:
        return np.zeros((0, 2), np.int64)
    return np.unique(np.concatenate(out), axis=0)


def face_status(vertices, faces):
    """Per face: 0 tested, 1 degenerate (exactly collinear corners), 2 a non-finite corner.  Only faces whose fp64 cross
    product is within a wide margin of zero are decided exactly."""
    v = np.asarray(vertices, np.float32)
    faces = np.asarray(faces, np.int64)
    X = Exact(v)
    st = np.zeros(len(faces), np.int8)
    with np.errstate(invalid='ignore', over='ignore'):
        t = v.astype(np.float64)[faces]
        finite = np.all(np.isfinite(t), (1, 2))
        e1, e2 = t[:, 1] - t[:, 0], t[:, 2] - t[:, 0]
        cr = np.abs(np.cross(e1, e2)).max(1)
        clear = cr > 1e-9 * np.abs(e1).max(1) * np.abs(e2).max(1)
    st[~finite] = 2
    for k in np.flatnonzero(finite & ~clear):
        fr = faces[k]
        if cross(sub(X[fr[1]], X[fr[0]]), sub(X[fr[2]], X[fr[0]])) == (0, 0, 0):
            st[k] = 1
    return st


def self_intersections(vertices, faces, subset=None):
    """(pairs (n, 2) int32 sorted by (f, g), f < g; degenerate count; non-finite count).  `subset`: only pairs with a face
    in it (enough when the rest of the mesh is known to be embedded)."""
    faces = np.asarray(faces, np.int64)
    st = face_status(vertices, faces)
    X = Exact(vertices)
    hits = [(int(i), int(j)) for i, j in candidates(vertices, faces, st == 0, subset)
            if pair_intersects(tuple(faces[i]), tuple(faces[j]), X)]
    pairs = np.array(sorted(hits), np.int32).reshape(-1, 2)
    return pairs, int((st == 1).sum()), int((st == 2).sum())

"""CPU restatement of nw_surface_signed_distance (ch_shrinkwrap_b200/csrc/surface.cu), test infrastructure only.

The region of the winning face by the operations of surface_oracle.closest_point_triangle, the twin table, the vertex ->
face CSR and the defect counts by plain numpy, the vertex pseudonormals with np.arctan2, the sign and the signed volume in
the device's reduction order.  The independent truth is the generalised winding number (solid angles by van Oosterom &
Strackee), brute force over all faces, plus a few small closed test solids."""
from __future__ import annotations

import math

import numpy as np

import surface_oracle as orc

CORNER, EDGE = 1, 4                      # region codes: 0 interior, CORNER + k corner k, EDGE + k the edge corner k -> k + 1


def _cross(u, v):
    return np.stack([u[:, 1] * v[:, 2] - u[:, 2] * v[:, 1], u[:, 2] * v[:, 0] - u[:, 0] * v[:, 2],
                     u[:, 0] * v[:, 1] - u[:, 1] * v[:, 0]], 1)


def _unit_normal(a, b, c):
    cr = _cross(b - a, c - a)
    l2 = orc._dot(cr, cr)
    with np.errstate(divide='ignore', invalid='ignore'):
        n = cr / np.sqrt(l2)[:, None]
    return np.where((l2 > 0.0)[:, None], n, 0.0)


def _segment_region(p, p0, p1, k):
    e = p1 - p0
    ee = orc._dot(e, e)
    with np.errstate(divide='ignore', invalid='ignore'):
        t = np.where(ee > 0.0, orc._dot(p - p0, e) / ee, 0.0)
    t = np.fmin(np.fmax(t, 0.0), 1.0)
    return np.where(t == 0.0, CORNER + k, np.where(t == 1.0, CORNER + (k + 1) % 3, EDGE + k))


def _edges_region(p, a, b, c):
    best = orc._closest_on_segment(p, a, b)
    bd = orc._dist2(p, best)
    r = _segment_region(p, a, b, 0)
    for k, (u, v) in ((1, (b, c)), (2, (c, a))):
        x = orc._closest_on_segment(p, u, v)
        kd = orc._dist2(p, x)
        m = kd < bd
        best = np.where(m[:, None], x, best)
        bd = np.where(m, kd, bd)
        r = np.where(m, _segment_region(p, u, v, k), r)
    return r


def triangle_region(p, a, b, c):
    """(closest point, region code) row by row: closest_point_triangle's precedence of regions, same bits."""
    ab, ac = b - a, c - a
    degenerate = ((ab[:, 1] * ac[:, 2] - ab[:, 2] * ac[:, 1] == 0.0) & (ab[:, 2] * ac[:, 0] - ab[:, 0] * ac[:, 2] == 0.0)
                  & (ab[:, 0] * ac[:, 1] - ab[:, 1] * ac[:, 0] == 0.0))
    ap, bp, cp = p - a, p - b, p - c
    d1, d2 = orc._dot(ab, ap), orc._dot(ac, ap)
    d3, d4 = orc._dot(ab, bp), orc._dot(ac, bp)
    d5, d6 = orc._dot(ab, cp), orc._dot(ac, cp)
    vc = d1 * d4 - d3 * d2
    vb = d5 * d2 - d1 * d6
    va = d3 * d6 - d5 * d4
    s = va + vb + vc
    edges = _edges_region(p, a, b, c)
    r = np.where(s > 0.0, 0, edges)
    r = np.where((va <= 0.0) & ((d4 - d3) >= 0.0) & ((d5 - d6) >= 0.0), EDGE + 1, r)
    r = np.where((vb <= 0.0) & (d2 >= 0.0) & (d6 <= 0.0), EDGE + 2, r)
    r = np.where((d6 >= 0.0) & (d5 <= d6), CORNER + 2, r)
    r = np.where((vc <= 0.0) & (d1 >= 0.0) & (d3 <= 0.0), EDGE + 0, r)
    r = np.where((d3 >= 0.0) & (d4 <= d3), CORNER + 1, r)
    r = np.where((d1 <= 0.0) & (d2 <= 0.0), CORNER + 0, r)
    return orc.closest_point_triangle(p, a, b, c), np.where(degenerate, edges, r)


def tables(faces, M, fans=True):
    """(twin (F,3): the face row across edge k of each row or -1, voff (M+1), vface (3F): incident rows in increasing order,
    defects [boundary edges, edges on > 2 faces, co-directed edge pairs, faces repeating a vertex, vertices with > 1 fan]).
    fans=False skips the per-vertex walk (a Python loop) and reports 0 for the last count."""
    f = np.asarray(faces, np.int64)
    F = len(f)
    u, w = f.ravel(), f[:, [1, 2, 0]].ravel()
    rep = int(((f[:, 0] == f[:, 1]) | (f[:, 1] == f[:, 2]) | (f[:, 2] == f[:, 0])).sum())
    lo, hi = np.minimum(u, w), np.maximum(u, w)
    he = np.flatnonzero(lo != hi)
    key = lo * (1 << 32) + hi
    order = he[np.argsort(key[he], kind='stable')]
    ks = key[order]
    starts = np.flatnonzero(np.r_[True, ks[1:] != ks[:-1]])
    size = np.diff(np.r_[starts, len(ks)])
    twin = np.full(3 * F, -1, np.int64)
    pair = starts[size == 2]
    e0, e1 = order[pair], order[pair + 1]
    same = u[e0] == u[e1]
    twin[e0[~same]], twin[e1[~same]] = e1[~same] // 3, e0[~same] // 3
    cnt = np.bincount(u, minlength=M)
    voff = np.r_[0, np.cumsum(cnt)]
    vface = (np.sort(u * (1 << 32) + np.arange(3 * F) // 3) & 0xffffffff).astype(np.int64)
    n_fans = 0
    for v in np.flatnonzero(cnt) if fans else ():
        n, f0 = cnt[v], vface[voff[v]]
        g, length = f0, 0
        while True:
            k = np.flatnonzero(f[g] == v)
            if len(k) == 0:
                length = n
                break
            length += 1
            g = twin[3 * g + (k[0] + 2) % 3]
            if g < 0:
                length = n
                break
            if g == f0 or length > n:
                break
        n_fans += int(length < n)
    return twin.reshape(F, 3), voff, vface, [int((size == 1).sum()), int((size > 2).sum()), int(same.sum()), rep, n_fans]


def pseudonormals(vertices, faces, voff, vface):
    """(M,3) sum over each vertex's faces in increasing row order of corner angle x unit normal (np.arctan2)."""
    v = np.asarray(vertices, np.float32).astype(np.float64)
    f = np.asarray(faces, np.int64)
    M = len(voff) - 1
    cnt = np.diff(voff)
    own = np.repeat(np.arange(M), cnt)              # vertex of each CSR entry
    rows = vface
    k = np.argmax(f[rows] == own[:, None], 1)
    x = [v[f[rows, j]] for j in range(3)]
    nf = _unit_normal(*x)
    pick = lambda j: np.stack(x, 1)[np.arange(len(rows)), (k + j) % 3]
    p, a, b = pick(0), pick(1), pick(2)
    uu, ww = a - p, b - p
    uw = _cross(uu, ww)
    th = np.arctan2(np.sqrt(orc._dot(uw, uw)), orc._dot(uu, ww))
    contrib = th[:, None] * nf
    N = np.zeros((M, 3))
    for j in range(int(cnt.max(initial=0))):         # in the device's order: entry j of every vertex that has one
        has = np.flatnonzero(cnt > j)
        N[has] = N[has] + contrib[voff[has] + j]
    return N


def volume_terms(vertices, faces):
    """dot(a - o, (b - o) x (c - o)) / 6 per face, o the float32 centre of the bounding box of the vertices the faces use."""
    v32 = np.asarray(vertices, np.float32)
    f = np.asarray(faces, np.int64)
    used = v32[np.unique(f)]
    used = used[np.isfinite(used).all(1)]
    o = ((used.min(0) + used.max(0)) * np.float32(0.5)).astype(np.float64)
    v = v32.astype(np.float64)
    a, b, c = v[f[:, 0]] - o, v[f[:, 1]] - o, v[f[:, 2]] - o
    return orc._dot(a, _cross(b, c)) / 6.0


def fixed_order_sum(terms, blocks=256, threads=256):
    """The device's reduction: thread t of block b sums entries b*threads + t + k*threads*blocks in increasing k, then a tree
    per block and a tree over the blocks."""
    n = blocks * threads
    t = np.zeros(-(-max(len(terms), 1) // n) * n)
    t[:len(terms)] = terms
    t = t.reshape(-1, n)
    s = np.zeros(n)
    for row in t:
        s = s + row
    s = s.reshape(blocks, threads)
    o = threads // 2
    while o:
        s[:, :o] = s[:, :o] + s[:, o:2 * o]
        o //= 2
    p = s[:, 0].copy()
    o = blocks // 2
    while o:
        p[:o] = p[:o] + p[o:2 * o]
        o //= 2
    return float(p[0])


def signed_distance(points, vertices, faces):
    """nw_surface_signed_distance's contract: (sdist, face, closest, volume |V|, margin, region).  margin = |s| / (|q - c| |N|),
    how far the side is from undecidable in relative terms (NaN where d == 0 or the query is non-finite)."""
    q = np.asarray(points).astype(np.float64)
    v32 = np.asarray(vertices, np.float32)
    f = np.asarray(faces, np.int64)
    twin, voff, vface, _ = tables(f, len(v32), fans=False)
    N_v = pseudonormals(v32, f, voff, vface)
    V = fixed_order_sum(volume_terms(v32, f))
    d, face, closest = orc.surface_nearest(q, v32, f)
    ok = np.flatnonzero(face >= 0)
    v = v32.astype(np.float64)
    fr = f[face[ok]]
    x = [v[fr[:, j]] for j in range(3)]
    c, r = triangle_region(q[ok], *x)
    N = _cross(x[1] - x[0], x[2] - x[0])
    corner = (r >= CORNER) & (r < EDGE)
    N[corner] = N_v[fr[corner, r[corner] - CORNER]]
    edge = np.flatnonzero(r >= EDGE)
    if len(edge):
        fi = face[ok][edge].astype(np.int64)
        g = twin[fi, r[edge] - EDGE]
        nf = _unit_normal(*[xx[edge] for xx in x])
        ng = np.zeros_like(nf)
        gg = np.maximum(g, 0)
        ng_all = _unit_normal(v[f[gg, 0]], v[f[gg, 1]], v[f[gg, 2]])
        ng[g >= 0] = ng_all[g >= 0]
        lower = (fi < g)[:, None]
        N[edge] = np.where(lower, nf, ng) + np.where(lower, ng, nf)
    qc = q[ok] - c
    s = orc._dot(qc, N)
    sd = np.full(len(q), np.nan)
    sd[ok] = np.where(d[ok] == 0.0, 0.0, np.where(s == 0.0, np.nan, np.where((s > 0.0) == (V > 0.0), d[ok], -d[ok])))
    margin = np.full(len(q), np.nan)
    with np.errstate(divide='ignore', invalid='ignore'):
        margin[ok] = np.abs(s) / (np.sqrt(orc._dot(qc, qc)) * np.sqrt(orc._dot(N, N)))
    region = np.full(len(q), -1)
    region[ok] = r
    return sd, face, closest, abs(V), margin, region


def face_normal_side(points, vertices, faces, face):
    """The naive side: q - c against the winning face's own normal (what the pseudonormal replaces), oriented by V."""
    q = np.asarray(points).astype(np.float64)
    v32 = np.asarray(vertices, np.float32)
    v = v32.astype(np.float64)
    f = np.asarray(faces, np.int64)[face]
    x = [v[f[:, j]] for j in range(3)]
    c, _ = triangle_region(q, *x)
    V = math.fsum(volume_terms(v32, faces))
    return np.sign(orc._dot(q - c, _cross(x[1] - x[0], x[2] - x[0]))) * np.sign(V)


def winding_number(points, vertices, faces, chunk=1 << 22):
    """Generalised winding number: sum of the faces' signed solid angles / 4 pi (van Oosterom & Strackee 1983)."""
    q = np.asarray(points, np.float64)
    v = np.asarray(vertices, np.float32).astype(np.float64)
    f = np.asarray(faces, np.int64)
    A, B, C = v[f[:, 0]], v[f[:, 1]], v[f[:, 2]]
    out = np.zeros(len(q))
    step = max(1, chunk // max(len(f), 1))
    for s in range(0, len(q), step):
        p = q[s:s + step, None, :]
        a, b, c = A[None] - p, B[None] - p, C[None] - p
        la, lb, lc = (np.sqrt((x * x).sum(-1)) for x in (a, b, c))
        det = (a * np.cross(b, c)).sum(-1)
        den = la * lb * lc + (a * b).sum(-1) * lc + (b * c).sum(-1) * la + (c * a).sum(-1) * lb
        out[s:s + step] = (2.0 * np.arctan2(det, den)).sum(1) / (4.0 * np.pi)
    return out


# ---- closed test solids (outward winding) ------------------------------------------------------------------------------
def tetrahedron(size=10.0):
    v = np.array([[1, 1, 1], [1, -1, -1], [-1, 1, -1], [-1, -1, 1]], np.float64) * size
    f = np.array([[0, 1, 2], [0, 3, 1], [0, 2, 3], [1, 3, 2]], np.int32)
    return v.astype(np.float32), f


def _outward(v, f):
    """Flip every face whose normal points towards the centroid of the solid (convex solids only)."""
    v64 = v.astype(np.float64)
    ctr = v64.mean(0)
    a, b, c = v64[f[:, 0]], v64[f[:, 1]], v64[f[:, 2]]
    flip = orc._dot(_cross(b - a, c - a), (a + b + c) / 3.0 - ctr) < 0.0
    f = f.copy()
    f[flip] = f[flip][:, [0, 2, 1]]
    return f


def prism(length=10.0):
    """A thin triangular prism: its cross-section has a 11 degree corner, so two of its long edges are sharp."""
    tri = np.array([[0.0, 0.0], [5.0, 0.5], [5.0, -0.5]])
    v = np.concatenate([np.c_[tri, np.zeros(3)], np.c_[tri, np.full(3, length)]]).astype(np.float32)
    f = np.array([[0, 1, 2], [3, 4, 5], [0, 1, 4], [0, 4, 3], [1, 2, 5], [1, 5, 4], [2, 0, 3], [2, 3, 5]], np.int32)
    return v, _outward(v, f)


def voxel_solid(cells):
    """Surface of a union of unit cubes (integer cell corners), each exposed unit square split into two triangles."""
    cells = set(map(tuple, cells))
    quads = []
    for (x, y, z) in cells:
        for ax in range(3):
            for sgn in (-1, 1):
                nb = [x, y, z]
                nb[ax] += sgn
                if tuple(nb) in cells:
                    continue
                o = np.array([x, y, z], np.float64)
                o[ax] += 1.0 if sgn > 0 else 0.0
                u, w = np.eye(3)[(ax + 1) % 3], np.eye(3)[(ax + 2) % 3]
                quad = [o, o + u, o + u + w, o + w]                 # counter-clockwise seen from +axis
                if sgn < 0:
                    quad = quad[::-1]
                quads.append(quad)
    pts = np.array(quads).reshape(-1, 3)
    uniq, inv = np.unique(pts, axis=0, return_inverse=True)
    q = inv.reshape(-1, 4)
    f = np.concatenate([q[:, [0, 1, 2]], q[:, [0, 2, 3]]]).astype(np.int32)
    return (uniq * 10.0).astype(np.float32), f


def cube():
    return voxel_solid([(0, 0, 0)])


def l_polycube():
    """Five cubes: a row of three along x and one on the first along y and along z (concave edges, a concave corner where
    three of them meet, saddle vertices)."""
    return voxel_solid([(0, 0, 0), (1, 0, 0), (0, 1, 0), (0, 0, 1), (2, 0, 0)])


def torus(R=30.0, r=10.0, nu=24, nv=12):
    a, b = np.meshgrid(np.arange(nu), np.arange(nv), indexing='ij')
    t, p = 2 * np.pi * a / nu, 2 * np.pi * b / nv
    v = np.stack([(R + r * np.cos(p)) * np.cos(t), (R + r * np.cos(p)) * np.sin(t), r * np.sin(p)], -1).reshape(-1, 3)
    idx = lambda i, j: (i % nu) * nv + (j % nv)
    i, j = a.ravel(), b.ravel()
    f = np.concatenate([np.stack([idx(i, j), idx(i + 1, j), idx(i + 1, j + 1)], 1),
                        np.stack([idx(i, j), idx(i + 1, j + 1), idx(i, j + 1)], 1)]).astype(np.int32)
    return v.astype(np.float32), f


def sphere(n=6, radius=20.0):
    from ch_shrinkwrap_b200 import minimesh
    v, f = minimesh.geodesic_sphere(n)
    return (v * radius).astype(np.float32), f


def feature_queries(vertices, faces, n_per=12, scale=0.08, seed=0):
    """Queries clustered around every corner and edge midpoint of the mesh, both sides, at up to `scale` x the mean edge."""
    rng = np.random.default_rng(seed)
    v = np.asarray(vertices, np.float64)
    f = np.asarray(faces, np.int64)
    e = np.concatenate([f[:, [0, 1]], f[:, [1, 2]], f[:, [2, 0]]])
    e = np.unique(np.sort(e, 1), axis=0)
    mid = 0.5 * (v[e[:, 0]] + v[e[:, 1]])
    h = float(np.sqrt(((v[e[:, 0]] - v[e[:, 1]]) ** 2).sum(1)).mean()) * scale
    centres = np.repeat(np.concatenate([v, mid]), n_per, 0)
    off = rng.normal(0.0, 1.0, centres.shape)
    off *= (h * rng.uniform(0.05, 1.0, len(off)) / np.sqrt((off * off).sum(1)))[:, None]
    return centres + off

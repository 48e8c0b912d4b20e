// surface.cu -- exact distance from query points to the handle's triangle mesh (nw_surface_distance).
//
// The fit's nearest-face search measures distances to face CENTROIDS (mesh_conj_grad.py:451-454); this file measures the
// Euclidean distance to the closed triangles.  It walks the same octree of Hilbert cells (tree.cu: kids, parent_g,
// leaf_of_slot, the frames of the node boxes), but against a second array of boxes, h->tboxes, whose intervals cover the
// three CORNERS of every face below the node instead of its centroid.  Those intervals are re-measured at the start of
// every call from the current positions, so they are never stale; h->boxes, cent, the seeds and the iteration graph are
// only read.
//
// Exactness: every candidate face's distance is evaluated in fp64 (corners widened exactly from float32, queries in
// float32 widened exactly or in float64) by one fixed sequence of operations, Ericson's closest-point region test
// (Real-Time Collision Detection, 5.1.5).  This file is compiled with -fmad=false so that the compiler performs exactly the
// written operations: tests/surface_oracle.py (closest_point_region) restates them in numpy and gets the same bits.
// Ties of the fp64 squared distance go to the lowest face index.  The box test only prunes: its float32 lower bound is
// made conservative by the rounding slack of the call (below), so it can never discard the true minimum.
//
// nw_surface_signed_distance runs the same search, then k_surface_sign re-runs the region test on the winning face with
// closest_on_triangle<true>, which also names the feature the closest point lies on (same bits of the point), and takes the
// side of q - c against the angle-weighted pseudonormal of that feature (face, edge or vertex; Baerentzen & Aanaes 2005),
// oriented by the sign of the mesh's signed volume.  Its edge and vertex tables are built once per topology
// (signed_tables), lazily, so nw_set_topology* does no extra work.
//
// The slack and the triangle-bounded boxes are built by nw_surface_boxes, which nw_self_intersections (intersect.cu) calls
// too: its broad phase walks the same boxes with a face instead of a query.  Distances and inside/outside answers assume an
// embedded mesh; nw_self_intersections is the check for faces that cross or touch.
#include <cfloat>
#include <cmath>
#include <cstdio>
#include <cub/cub.cuh>
#include "common.cuh"

namespace {

// ---- rounding slack of the call (common.cuh: call_slack) -----------------------------------------------------------
// per-axis max |coordinate| over the finite values, as the bits of non-negative floats (which order like unsigned ints)
__device__ __forceinline__ float abs_up(float v) { return fabsf(v); }
__device__ __forceinline__ float abs_up(double v) { return __double2float_ru(fabs(v)); }
template <typename T>
__global__ void __launch_bounds__(256) k_absmax3(const T *__restrict__ x, const T *__restrict__ y, const T *__restrict__ z, int64_t n,
                                                 int64_t stride, unsigned *__restrict__ out3) {
    float m[3] = {0.f, 0.f, 0.f};
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const float v[3] = {abs_up(x[i * stride]), abs_up(y[i * stride]), abs_up(z[i * stride])};
        for (int k = 0; k < 3; ++k) if (v[k] <= FLT_MAX) m[k] = fmaxf(m[k], v[k]);
    }
    for (int k = 0; k < 3; ++k) {
        const unsigned r = __reduce_max_sync(0xffffffffu, __float_as_uint(m[k]));
        if ((threadIdx.x & 31) == 0 && r) atomicMax(out3 + k, r);
    }
}

// ---- triangle-bounded boxes ------------------------------------------------------------------------------------------
// frames and search links of h->boxes, intervals empty
__global__ void k_tbox_init(const Box *__restrict__ boxes, int n, Box *__restrict__ tb) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const Box s = boxes[j];
    Box t;
    t.a = s.a;
    t.b = make_float4(s.b.x, s.b.y, NW_EMPTY_LO, NW_EMPTY_LO);
    t.c = make_float4(s.c.x, s.c.y, s.c.z, NW_EMPTY_HI);
    t.d = make_float4(NW_EMPTY_HI, NW_EMPTY_HI, s.d.z, NW_EMPTY_LO);
    tb[j] = t;
}

// k_extents (tree.cu) with the three corners of each face in place of its centroid: every face projects its corners onto the
// frame of every ancestor (common.cuh: nw_merge_extents).  A face with a non-finite corner contributes nothing (the query
// kernel skips it too).
__global__ void __launch_bounds__(256) k_tri_extents(const int4 *__restrict__ sfaces, const float4 *__restrict__ pos, int F,
                                                     const int *__restrict__ leaf_of_slot, int leaf0, int leaf_level,
                                                     const int *__restrict__ parent_g, Box *__restrict__ boxes) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = i < F;
    float4 v[3] = {make_float4(0.f, 0.f, 0.f, 0.f), make_float4(0.f, 0.f, 0.f, 0.f), make_float4(0.f, 0.f, 0.f, 0.f)};
    bool finite = live;
    if (live) {
        const int4 sf = sfaces[i];
        v[0] = pos[sf.x]; v[1] = pos[sf.y]; v[2] = pos[sf.z];
        for (int k = 0; k < 3; ++k) finite = finite && fabsf(v[k].x) <= FLT_MAX && fabsf(v[k].y) <= FLT_MAX && fabsf(v[k].z) <= FLT_MAX;
    }
    int node = live ? leaf0 + leaf_of_slot[i] : 0;
    for (int l = leaf_level; l >= 1; --l) {
        nw_merge_extents(boxes, node, live, finite, [&](const Box *b, float (&lo)[3], float (&hi)[3]) {
            const float4 ba = b->a, bb = b->b, bc = b->c;
            project_frame(ba, bb, bc, v[0].x, v[0].y, v[0].z, lo[0], lo[1], lo[2]);
            hi[0] = lo[0]; hi[1] = lo[1]; hi[2] = lo[2];
            for (int c = 1; c < 3; ++c) {
                float p[3];
                project_frame(ba, bb, bc, v[c].x, v[c].y, v[c].z, p[0], p[1], p[2]);
                for (int k = 0; k < 3; ++k) { lo[k] = fminf(lo[k], p[k]); hi[k] = fmaxf(hi[k], p[k]); }
            }
        });
        if (live) node = parent_g[node] & 0x7fffffff;
    }
}

// ordered-int -> float, widened by the slack of the call (k_box_decode's rule)
__global__ void k_tbox_decode(Box *__restrict__ tb, int first, int count, const unsigned *__restrict__ bits6) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    nw_decode_box(&tb[first + i], call_slack(bits6));
}

// ---- exact point-to-triangle distance (fp64, fixed operation order; restated in tests/surface_oracle.py) -------------------
struct D3 { double x, y, z; };
__device__ __forceinline__ D3 d3(const float4 v) { return D3{(double)v.x, (double)v.y, (double)v.z}; }
__device__ __forceinline__ D3 sub(const D3 a, const D3 b) { return D3{a.x - b.x, a.y - b.y, a.z - b.z}; }
__device__ __forceinline__ double dot(const D3 a, const D3 b) { return (a.x * b.x + a.y * b.y) + a.z * b.z; }
__device__ __forceinline__ D3 axpy(const D3 a, const double t, const D3 e) { return D3{a.x + t * e.x, a.y + t * e.y, a.z + t * e.z}; }
__device__ __forceinline__ double dist2(const D3 p, const D3 c) { const D3 d = sub(p, c); return dot(d, d); }

// R: also name the feature the closest point lies on (nw_surface_signed_distance), in r.  Region codes: 0 the interior,
// 1 + k corner k, 4 + k the edge from corner k to corner k + 1 (mod 3).  The operations, and so the points, do not depend on R.
#define NW_REGION_CORNER(k) (1 + (k))
#define NW_REGION_EDGE(k) (4 + (k))
// the segment p0 -> p1 as edge k of a triangle
template <bool R>
__device__ __forceinline__ D3 closest_on_segment(const D3 p, const D3 p0, const D3 p1, const int k, int &r) {
    const D3 e = sub(p1, p0);
    const double ee = dot(e, e);
    double t = ee > 0.0 ? dot(sub(p, p0), e) / ee : 0.0;
    t = fmin(fmax(t, 0.0), 1.0);
    if (R) r = t == 0.0 ? NW_REGION_CORNER(k) : t == 1.0 ? NW_REGION_CORNER((k + 1) % 3) : NW_REGION_EDGE(k);
    return axpy(p0, t, e);
}
// a zero-area triangle is the union of its three edges: the closest of them, in the order ab, bc, ca (first wins ties)
template <bool R>
__device__ __noinline__ D3 closest_on_edges(const D3 p, const D3 a, const D3 b, const D3 c, int &r) {
    int rk;
    D3 best = closest_on_segment<R>(p, a, b, 0, r);
    double bd = dist2(p, best);
    D3 k = closest_on_segment<R>(p, b, c, 1, rk);
    double kd = dist2(p, k);
    if (kd < bd) { best = k; bd = kd; if (R) r = rk; }
    k = closest_on_segment<R>(p, c, a, 2, rk);
    kd = dist2(p, k);
    if (kd < bd) { best = k; if (R) r = rk; }
    return best;
}
// Ericson's region test.  Degenerate: the cross product ab x ac is exactly zero, or (rounding of a nearly degenerate
// triangle) the interior case finds no positive barycentric denominator.
template <bool R>
__device__ __forceinline__ D3 closest_on_triangle(const D3 p, const D3 a, const D3 b, const D3 c, int &r) {
    const D3 ab = sub(b, a), ac = sub(c, a);
    if (ab.y * ac.z - ab.z * ac.y == 0.0 && ab.z * ac.x - ab.x * ac.z == 0.0 && ab.x * ac.y - ab.y * ac.x == 0.0)
        return closest_on_edges<R>(p, a, b, c, r);
    const D3 ap = sub(p, a);
    const double d1 = dot(ab, ap), d2 = dot(ac, ap);
    if (d1 <= 0.0 && d2 <= 0.0) { r = NW_REGION_CORNER(0); return a; }
    const D3 bp = sub(p, b);
    const double d3 = dot(ab, bp), d4 = dot(ac, bp);
    if (d3 >= 0.0 && d4 <= d3) { r = NW_REGION_CORNER(1); return b; }
    const double vc = d1 * d4 - d3 * d2;
    if (vc <= 0.0 && d1 >= 0.0 && d3 <= 0.0) { r = NW_REGION_EDGE(0); return axpy(a, d1 / (d1 - d3), ab); }
    const D3 cp = sub(p, c);
    const double d5 = dot(ab, cp), d6 = dot(ac, cp);
    if (d6 >= 0.0 && d5 <= d6) { r = NW_REGION_CORNER(2); return c; }
    const double vb = d5 * d2 - d1 * d6;
    if (vb <= 0.0 && d2 >= 0.0 && d6 <= 0.0) { r = NW_REGION_EDGE(2); return axpy(a, d2 / (d2 - d6), ac); }
    const double va = d3 * d6 - d5 * d4;
    if (va <= 0.0 && (d4 - d3) >= 0.0 && (d5 - d6) >= 0.0) {
        r = NW_REGION_EDGE(1);
        return axpy(b, (d4 - d3) / ((d4 - d3) + (d5 - d6)), sub(c, b));
    }
    const double s = va + vb + vc;
    if (!(s > 0.0)) return closest_on_edges<R>(p, a, b, c, r);
    const double denom = 1.0 / s;
    const double v = vb * denom, w = vc * denom;
    r = 0;
    return D3{(a.x + ab.x * v) + ac.x * w, (a.y + ab.y * v) + ac.y * w, (a.z + ab.z * v) + ac.z * w};
}
__device__ __forceinline__ D3 closest_on_triangle(const D3 p, const D3 a, const D3 b, const D3 c) {
    int r;
    return closest_on_triangle<false>(p, a, b, c, r);
}

// the operations of the degenerate test above: cross(b - a, c - a) of a face in row order
__device__ __forceinline__ D3 cross(const D3 u, const D3 v) { return D3{u.y * v.z - u.z * v.y, u.z * v.x - u.x * v.z, u.x * v.y - u.y * v.x}; }
// unit normal cr / |cr|; a zero-area face has none and contributes zero
__device__ __forceinline__ D3 unit_normal(const D3 a, const D3 b, const D3 c) {
    const D3 cr = cross(sub(b, a), sub(c, a));
    const double l2 = dot(cr, cr);
    if (!(l2 > 0.0)) return D3{0.0, 0.0, 0.0};
    const double l = sqrt(l2);
    return D3{cr.x / l, cr.y / l, cr.z / l};
}

__device__ __forceinline__ bool finite4(const float4 v) { return fabsf(v.x) <= FLT_MAX && fabsf(v.y) <= FLT_MAX && fabsf(v.z) <= FLT_MAX; }

// ---- the walk ------------------------------------------------------------------------------------------------------
struct SurfaceArgs {
    int64_t Q;
    const void *qx, *qy, *qz;           // query coordinates (float or double): element i at q?[i * stride]
    int64_t stride;
    const int *perm;                    // resident points: sorted position -> caller's index (NULL: the identity)
    const int *seed;                    // resident points: nearest-centroid slot of the last sweep, or -1 (NULL: none)
    const Box *tb;
    const int *parent;
    const int2 *kids;
    const int *leaf_of_slot;
    const int4 *sfaces;
    const float4 *posq;
    int leaf0, leaf_level, n_nodes, F;
    double *dist;                       // caller order; always written
    int *face;                          // or NULL
    double *closest;                    // or NULL
};

// One query per thread, stackless: first child and next sibling come from the tables the fit's search uses (tree.cu).
struct SurfaceWalk {
    const SurfaceArgs &a;
    float x, y, z;                      // float32 rounding of the query: the box tests use it
    float eq;                           // how far the float32 rounding can lie from the query (0 for float32 queries)
    D3 p;                               // the query, exactly
    double d2 = DBL_MAX * 2.0;          // best squared distance (+inf: none yet)
    float ub = FLT_MAX * 2.0f;          // d2 rounded up, times the 1.1e-5 the float32 frames owe to orthonormality
    int face = 0x7fffffff, slot = -1;

    __device__ __forceinline__ SurfaceWalk(const SurfaceArgs &a_) : a(a_) {}
    __device__ __forceinline__ void offer(double v, int f, int s) {
        if (v < d2 || (v == d2 && f < face)) { d2 = v; face = f; slot = s; ub = __fmul_ru(__double2float_ru(v), 1.000011f); }
    }
    // lower bound of the squared distance from the query to anything in the node (sweep.cu: Traversal::test_node, with the
    // gaps shrunk by eq), compared with the best so far; `link` = the node's first child | last-child bit
    __device__ __forceinline__ bool open(int node, int &link) const {
        NW_ASSERT(node >= 0 && node < a.n_nodes);
        const Box *bp = &a.tb[node];
        const float4 ba = __ldg(&bp->a), bb = __ldg(&bp->b), bd = __ldg(&bp->d);
        link = __float_as_int(bd.z);
        const float pn = fmaf(ba.x, x, fmaf(ba.z, y, bb.x * z));
        const float p1 = fmaf(ba.y, x, fmaf(ba.w, y, bb.y * z));
        const float g0 = fmaxf(fmaxf(bb.z - pn, pn - bd.x) - eq, 0.f), g1 = fmaxf(fmaxf(bb.w - p1, p1 - bd.y) - eq, 0.f);
        const float s01 = __fmaf_rd(g1, g1, __fmul_rd(g0, g0));
        if (!(s01 <= ub)) return false;
        const float4 bc = __ldg(&bp->c);
        const float p2 = fmaf(bc.x, x, fmaf(bc.y, y, bc.z * z));
        const float g2 = fmaxf(fmaxf(bd.w - p2, p2 - bc.w) - eq, 0.f);
        return __fmaf_rd(g2, g2, s01) <= ub;
    }
    __device__ __forceinline__ void leaf(int node) {
        NW_ASSERT(node >= a.leaf0 && node < a.n_nodes);
        const int2 k = __ldg(&a.kids[node]);
        NW_ASSERT(k.x >= 0 && k.y >= 0 && k.x + k.y <= a.F);
        for (int s = k.x; s < k.x + k.y; ++s) {
            const int4 sf = __ldg(&a.sfaces[s]);
            const float4 va = __ldg(&a.posq[sf.x]), vb = __ldg(&a.posq[sf.y]), vc = __ldg(&a.posq[sf.z]);
            if (!(finite4(va) && finite4(vb) && finite4(vc))) continue;
            offer(dist2(p, closest_on_triangle(p, d3(va), d3(vb), d3(vc))), sf.w, s);
        }
    }
    __device__ __forceinline__ void subtree(int I) {
        int node = I;
        while (true) {
            int link;
            if (open(node, link)) {
                if (node >= a.leaf0) leaf(node);
                else { node = link & 0x7fffffff; continue; }
            }
            while (true) {
                if (node == I) return;
                if (link >= 0) { ++node; break; }
                link = __ldg(&a.parent[node]);
                node = link & 0x7fffffff;
            }
        }
    }
    // greedy descent to a first leaf for a query without a seed (sweep.cu: node_score)
    __device__ __forceinline__ int greedy_leaf() const {
        int node = 0;
        while (node < a.leaf0) {
            const int2 k = __ldg(&a.kids[node]);
            int pick = k.x;
            float bl = FLT_MAX * 2.0f;
            for (int ch = k.x; ch < k.x + k.y; ++ch) {
                const Box *bp = &a.tb[ch];
                const float4 ba = __ldg(&bp->a), bb = __ldg(&bp->b), bc = __ldg(&bp->c), bd = __ldg(&bp->d);
                float pn, p1, p2;
                project_frame(ba, bb, bc, x, y, z, pn, p1, p2);
                const float g0 = fmaxf(fmaxf(bb.z - pn, pn - bd.x), 0.f), g1 = fmaxf(fmaxf(bb.w - p1, p1 - bd.y), 0.f),
                            g2 = fmaxf(fmaxf(bd.w - p2, p2 - bc.w), 0.f);
                const float c0 = pn - 0.5f * (bb.z + bd.x), c1 = p1 - 0.5f * (bb.w + bd.y), c2 = p2 - 0.5f * (bd.w + bc.w);
                const float l = (g0 * g0 + g1 * g1 + g2 * g2) + 1e-4f * (c0 * c0 + c1 * c1 + c2 * c2);
                if (l < bl) { bl = l; pick = ch; }
            }
            node = pick;
        }
        return node;
    }
    // the leaf first, then at every level the sibling subtrees of the path to the root
    __device__ __forceinline__ void from_leaf(int node) {
        leaf(node);
        for (int level = a.leaf_level; level >= 1; --level) {
            const int p = __ldg(&a.parent[node]) & 0x7fffffff;
            const int2 k = __ldg(&a.kids[p]);
            for (int sib = k.x; sib < k.x + k.y; ++sib)
                if (sib != node) subtree(sib);
            node = p;
        }
    }
};

__device__ __forceinline__ float rn_f32(float v) { return v; }
__device__ __forceinline__ float rn_f32(double v) { return __double2float_rn(v); }

template <typename T>
__global__ void __launch_bounds__(128) k_surface_nearest(const __grid_constant__ SurfaceArgs a) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= a.Q) return;
    const T qx = ((const T *)a.qx)[i * a.stride], qy = ((const T *)a.qy)[i * a.stride], qz = ((const T *)a.qz)[i * a.stride];
    const int64_t o = a.perm ? (int64_t)a.perm[i] : i;
    SurfaceWalk w(a);
    w.p = D3{(double)qx, (double)qy, (double)qz};
    w.x = rn_f32(qx); w.y = rn_f32(qy); w.z = rn_f32(qz);
    // |n . (q - q32)| <= |q - q32|_1 <= half an ulp per coordinate <= L1(q32) 2^-24: shrink every gap by twice that
    w.eq = sizeof(T) == 8 ? fmaf(fabsf(w.x) + fabsf(w.y) + fabsf(w.z), 1.1920928955078125e-7f, FLT_MIN) : 0.f;
    if (fabs(w.p.x) <= DBL_MAX && fabs(w.p.y) <= DBL_MAX && fabs(w.p.z) <= DBL_MAX) {
        const int s = a.seed ? __ldg(&a.seed[i]) : -1;
        w.from_leaf(s >= 0 && s < a.F ? a.leaf0 + __ldg(&a.leaf_of_slot[s]) : w.greedy_leaf());
    }
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    D3 c = D3{nan, nan, nan};
    if (w.slot >= 0) {
        const int4 sf = __ldg(&a.sfaces[w.slot]);
        c = closest_on_triangle(w.p, d3(__ldg(&a.posq[sf.x])), d3(__ldg(&a.posq[sf.y])), d3(__ldg(&a.posq[sf.z])));
    }
    a.dist[o] = w.slot >= 0 ? sqrt(w.d2) : nan;
    if (a.face) a.face[o] = w.slot >= 0 ? w.face : -1;
    if (a.closest) { a.closest[3 * o] = c.x; a.closest[3 * o + 1] = c.y; a.closest[3 * o + 2] = c.z; }
}

// ---- summary: max, mean and RMS of the distances, in a fixed order ------------------------------------------------------
// Thread t of block b takes the entries b*256 + t + k*256*G in increasing k, then fixed trees; the result does not depend on
// scheduling.  Non-finite distances (non-finite queries, or a mesh without one finite face) are left out.
#define NW_SUM_BLOCKS 256
__global__ void __launch_bounds__(256) k_dist_partials(const double *__restrict__ d, int64_t n, double *__restrict__ part) {
    __shared__ double sh[4][256];
    double mx = 0.0, s = 0.0, s2 = 0.0, cnt = 0.0;
    for (int64_t i = blockIdx.x * 256 + threadIdx.x; i < n; i += 256 * (int64_t)gridDim.x) {
        const double v = d[i];
        if (v <= DBL_MAX) { mx = fmax(mx, v); s += v; s2 += v * v; cnt += 1.0; }
    }
    sh[0][threadIdx.x] = mx; sh[1][threadIdx.x] = s; sh[2][threadIdx.x] = s2; sh[3][threadIdx.x] = cnt;
    __syncthreads();
    for (int o = 128; o; o >>= 1) {
        if (threadIdx.x < o) {
            sh[0][threadIdx.x] = fmax(sh[0][threadIdx.x], sh[0][threadIdx.x + o]);
            for (int k = 1; k < 4; ++k) sh[k][threadIdx.x] += sh[k][threadIdx.x + o];
        }
        __syncthreads();
    }
    if (threadIdx.x < 4) part[4 * blockIdx.x + threadIdx.x] = sh[threadIdx.x][0];
}
__global__ void __launch_bounds__(256) k_dist_summary(const double *__restrict__ part, double *__restrict__ out3) {
    __shared__ double sh[4][NW_SUM_BLOCKS];
    for (int k = 0; k < 4; ++k) sh[k][threadIdx.x] = part[4 * threadIdx.x + k];
    __syncthreads();
    for (int o = NW_SUM_BLOCKS / 2; o; o >>= 1) {
        if (threadIdx.x < o) {
            sh[0][threadIdx.x] = fmax(sh[0][threadIdx.x], sh[0][threadIdx.x + o]);
            for (int k = 1; k < 4; ++k) sh[k][threadIdx.x] += sh[k][threadIdx.x + o];
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const double n = sh[3][0], nan = __longlong_as_double(0x7ff8000000000000LL);
        out3[0] = n > 0.0 ? sh[0][0] : nan;
        out3[1] = n > 0.0 ? sh[1][0] / n : nan;
        out3[2] = n > 0.0 ? sqrt(sh[2][0] / n) : nan;
    }
}

// ---- signed distance: edge and vertex tables of a topology (built once per nw_set_topology*) ---------------------------
// defects: [0] boundary edges, [1] edges on more than two faces, [2] edges whose two faces traverse them the same way,
// [3] faces that repeat a vertex, [4] vertices whose faces form more than one fan
// half-edge e = 3 f + k runs from corner k of face row f to corner k + 1; its key is the undirected edge (min, max)
__global__ void k_halfedge_keys(const int *__restrict__ faces, int F, unsigned long long *__restrict__ key, int *__restrict__ val,
                                int *__restrict__ defects) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= 3 * F) return;
    const int f = e / 3, k = e - 3 * f;
    const int u = faces[e], w = faces[3 * f + (k + 1) % 3];
    key[e] = ((unsigned long long)(unsigned)min(u, w) << 32) | (unsigned)max(u, w);
    val[e] = e;
    if (k == 0 && (faces[e] == faces[e + 1] || faces[e + 1] == faces[e + 2] || faces[e + 2] == faces[e])) atomicAdd(defects + 3, 1);
}
// one thread per run of equal keys: a closed, consistently oriented edge is exactly two half-edges running opposite ways
__global__ void k_edge_runs(const unsigned long long *__restrict__ key, const int *__restrict__ val, const int *__restrict__ faces, int n,
                            int *__restrict__ twin, int *__restrict__ defects) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n || (j > 0 && key[j - 1] == key[j])) return;
    const unsigned long long k = key[j];
    if ((unsigned)(k >> 32) == (unsigned)k) return;             // an edge from a vertex to itself: its face is counted in [3]
    int m = 1;
    while (j + m < n && key[j + m] == k) ++m;
    if (m == 1) { atomicAdd(defects, 1); return; }
    if (m > 2) { atomicAdd(defects + 1, 1); return; }
    const int e0 = val[j], e1 = val[j + 1];
    if (faces[e0] == faces[e1]) { atomicAdd(defects + 2, 1); return; }   // both start at the same end
    twin[e0] = e1 / 3;
    twin[e1] = e0 / 3;
}
// (vertex, face row) of every corner, and the number of corners per vertex
__global__ void k_corner_keys(const int *__restrict__ faces, int n, unsigned long long *__restrict__ key, int *__restrict__ cnt) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    key[e] = ((unsigned long long)(unsigned)faces[e] << 32) | (unsigned)(e / 3);
    atomicAdd(cnt + faces[e], 1);
}
__global__ void k_low_words(const unsigned long long *__restrict__ key, int n, int *__restrict__ out) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < n) out[j] = (int)(unsigned)key[j];
}
// Walk the faces around each vertex through the twin table: from face f, across the edge that arrives at v (corner k - 1 ->
// k), to the next face.  A manifold vertex comes back to its first face after visiting all of them.  Two solids that touch
// at one vertex pass every edge test, but their shared vertex closes a fan early.  An open fan is left to the edge counts.
__global__ void k_vertex_fans(const int *__restrict__ faces, const int *__restrict__ twin, const int *__restrict__ voff,
                              const int *__restrict__ vface, int M, int *__restrict__ defects) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= M) return;
    const int n = voff[v + 1] - voff[v];
    if (n == 0) return;
    const int f0 = vface[voff[v]];
    int f = f0, len = 0;
    do {
        const int k = faces[3 * f] == v ? 0 : faces[3 * f + 1] == v ? 1 : faces[3 * f + 2] == v ? 2 : -1;
        if (k < 0) return;
        ++len;
        f = twin[3 * f + (k + 2) % 3];
        if (f < 0) return;
    } while (f != f0 && len <= n);
    if (len < n) atomicAdd(defects + 4, 1);
}

// ---- signed distance, every call: pseudonormals, volume, sign ----------------------------------------------------------
// N_v = sum over the incident faces in increasing row order of theta_f n_f, theta_f the corner angle at v between the edges
// to the next and the one after in the face's corner order; also the bounding box of the vertices the faces use
__global__ void __launch_bounds__(256) k_vertex_pseudonormals(const int *__restrict__ faces, const float4 *__restrict__ pos,
                                                              const int *__restrict__ voff, const int *__restrict__ vface, int M,
                                                              double *__restrict__ nv, unsigned *__restrict__ bbox6) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= M) return;
    const int b = voff[v], e = voff[v + 1];
    D3 n = D3{0.0, 0.0, 0.0};
    for (int j = b; j < e; ++j) {
        const int f = vface[j];
        const int c[3] = {faces[3 * f], faces[3 * f + 1], faces[3 * f + 2]};
        const int k = c[0] == v ? 0 : c[1] == v ? 1 : 2;
        const D3 x[3] = {d3(pos[c[0]]), d3(pos[c[1]]), d3(pos[c[2]])};
        const D3 nf = unit_normal(x[0], x[1], x[2]);
        const D3 u = sub(x[(k + 1) % 3], x[k]), w = sub(x[(k + 2) % 3], x[k]);
        const D3 uw = cross(u, w);
        const double th = atan2(sqrt(dot(uw, uw)), dot(u, w));
        n = D3{n.x + th * nf.x, n.y + th * nf.y, n.z + th * nf.z};
    }
    nv[3 * (size_t)v] = n.x; nv[3 * (size_t)v + 1] = n.y; nv[3 * (size_t)v + 2] = n.z;
    const float4 p = pos[v];
    if (e > b && finite4(p)) {
        atomicMin(bbox6, f2u(p.x)); atomicMin(bbox6 + 1, f2u(p.y)); atomicMin(bbox6 + 2, f2u(p.z));
        atomicMax(bbox6 + 3, f2u(p.x)); atomicMax(bbox6 + 4, f2u(p.y)); atomicMax(bbox6 + 5, f2u(p.z));
    }
}
__device__ __forceinline__ float u2f(unsigned u) { return ord2f(u2ord(u)); }
// V = sum_f dot(a - o, cross(b - o, c - o)) / 6, o the float32 centre of that bounding box; the order of k_dist_partials
__global__ void __launch_bounds__(256) k_volume_partials(const int *__restrict__ faces, const float4 *__restrict__ pos, int F,
                                                         const unsigned *__restrict__ bbox6, double *__restrict__ part) {
    __shared__ double sh[256];
    const D3 o = D3{(double)((u2f(bbox6[0]) + u2f(bbox6[3])) * 0.5f), (double)((u2f(bbox6[1]) + u2f(bbox6[4])) * 0.5f),
                    (double)((u2f(bbox6[2]) + u2f(bbox6[5])) * 0.5f)};
    double s = 0.0;
    for (int64_t f = blockIdx.x * 256 + threadIdx.x; f < F; f += 256 * (int64_t)gridDim.x) {
        const D3 a = sub(d3(pos[faces[3 * f]]), o), b = sub(d3(pos[faces[3 * f + 1]]), o), c = sub(d3(pos[faces[3 * f + 2]]), o);
        s += dot(a, cross(b, c)) / 6.0;
    }
    sh[threadIdx.x] = s;
    __syncthreads();
    for (int k = 128; k; k >>= 1) {
        if (threadIdx.x < k) sh[threadIdx.x] += sh[threadIdx.x + k];
        __syncthreads();
    }
    if (threadIdx.x == 0) part[blockIdx.x] = sh[0];
}
__global__ void __launch_bounds__(256) k_volume_fold(const double *__restrict__ part, double *__restrict__ vol) {
    __shared__ double sh[NW_SUM_BLOCKS];
    sh[threadIdx.x] = part[threadIdx.x];
    __syncthreads();
    for (int k = NW_SUM_BLOCKS / 2; k; k >>= 1) {
        if (threadIdx.x < k) sh[threadIdx.x] += sh[threadIdx.x + k];
        __syncthreads();
    }
    if (threadIdx.x == 0) *vol = sh[0];
}

struct SignArgs {
    int64_t Q;
    const void *qx, *qy, *qz;           // the queries of k_surface_nearest
    int64_t stride;
    const int *perm;
    const int *faces, *twin;            // face rows, (F,3); twin table, 3F
    const float4 *posq;
    const double *nv;                   // vertex pseudonormals, 3M
    const double *vol;                  // the signed volume
    const int *face;                    // k_surface_nearest's face rows (caller order)
    double *dist;                       // in: its distances; out: the signed distances (caller order)
};

// The winning face's region test again (the same bits of c), the pseudonormal of that feature, and the side of q - c.
template <typename T>
__global__ void __launch_bounds__(128) k_surface_sign(const __grid_constant__ SignArgs a) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= a.Q) return;
    const int64_t o = a.perm ? (int64_t)a.perm[i] : i;
    const int f = a.face[o];
    const double d = a.dist[o];
    if (f < 0 || d == 0.0) return;                              // NaN (non-finite query) or 0 stay as they are
    const T qx = ((const T *)a.qx)[i * a.stride], qy = ((const T *)a.qy)[i * a.stride], qz = ((const T *)a.qz)[i * a.stride];
    const D3 p = D3{(double)qx, (double)qy, (double)qz};
    const int cv[3] = {a.faces[3 * f], a.faces[3 * f + 1], a.faces[3 * f + 2]};
    const D3 x[3] = {d3(a.posq[cv[0]]), d3(a.posq[cv[1]]), d3(a.posq[cv[2]])};
    int r;
    const D3 c = closest_on_triangle<true>(p, x[0], x[1], x[2], r);
    D3 N;
    if (r == 0) {
        N = cross(sub(x[1], x[0]), sub(x[2], x[0]));
    } else if (r < NW_REGION_EDGE(0)) {
        const int v = cv[r - NW_REGION_CORNER(0)];
        N = D3{a.nv[3 * (size_t)v], a.nv[3 * (size_t)v + 1], a.nv[3 * (size_t)v + 2]};
    } else {
        const int k = r - NW_REGION_EDGE(0), g = a.twin[3 * f + k];
        const D3 nf = unit_normal(x[0], x[1], x[2]);
        D3 ng = D3{0.0, 0.0, 0.0};
        if (g >= 0) ng = unit_normal(d3(a.posq[a.faces[3 * g]]), d3(a.posq[a.faces[3 * g + 1]]), d3(a.posq[a.faces[3 * g + 2]]));
        const D3 lo = f < g ? nf : ng, hi = f < g ? ng : nf;
        N = D3{lo.x + hi.x, lo.y + hi.y, lo.z + hi.z};
    }
    const double s = dot(sub(p, c), N);
    a.dist[o] = s == 0.0 ? __longlong_as_double(0x7ff8000000000000LL) : (s > 0.0) == (*a.vol > 0.0) ? d : -d;
}

}  // namespace

// the handle holds a mesh: the rule of every call that measures the mesh itself (this file, intersect.cu)
int nw_mesh_check(nw_ctx *h, const std::string &w) {
    NW_ARG(h->M > 0 && h->F > 0 && h->tl.n_levels > 1, w + ": no topology (call nw_set_topology first)");
    NW_ARG(!h->points_mode, w + ": the handle holds point targets (nw_set_point_targets), not a mesh");
    return NW_OK;
}

// arguments shared by both entry points
static int surface_check(nw_ctx *h, const char *who, const void *q, int64_t Q) {
    const std::string w(who);
    NW_CHECK(nw_mesh_check(h, w));
    if (q) NW_ARG(Q >= 0 && Q < 2147483647LL, w + ": Q must be in [0, 2^31)");
    else NW_ARG(Q == h->P && (h->px != nullptr || h->P == 0),
                w + ": q == NULL measures the resident points; Q must equal their number (nw_set_points)");
    return NW_OK;
}

// The slack of the call, then the triangle-bounded boxes at the current positions.  Q == 0: the vertices' slack alone
// (nw_self_intersections has no queries).
int nw_surface_boxes(nw_ctx *h, const void *qx, const void *qy, const void *qz, int64_t Q, int64_t stride, bool f64) {
    cudaStream_t s = h->stream;
    const int B = 256;
    const TreeLevels &tl = h->tl;
    const int leaf_level = tl.n_levels - 1, leaf0 = tl.off[leaf_level], total = leaf0 + tl.count[leaf_level];
    NW_CHECK(nw_alloc(h, &h->surf_bits, (size_t)8));
    NW_CUDA(cudaMemsetAsync(h->surf_bits, 0, sizeof(unsigned) * 6, s));
    const float *pq = (const float *)h->posq;      // x, y, z of vertex v at pq[4 v + 0..2]
    k_absmax3<float><<<std::min(nw_grid(h->M, B), 148 * 4), B, 0, s>>>(pq, pq + 1, pq + 2, h->M, 4, h->surf_bits);
    NW_LAUNCH_CHECK();
    if (Q > 0) {
        if (f64) k_absmax3<double><<<std::min(nw_grid(Q, B), 148 * 4), B, 0, s>>>((const double *)qx, (const double *)qy,
                                                                                  (const double *)qz, Q, stride, h->surf_bits + 3);
        else k_absmax3<float><<<std::min(nw_grid(Q, B), 148 * 4), B, 0, s>>>((const float *)qx, (const float *)qy, (const float *)qz,
                                                                            Q, stride, h->surf_bits + 3);
        NW_LAUNCH_CHECK();
    }
    NW_CHECK(nw_alloc(h, &h->tboxes, (size_t)total));
    k_tbox_init<<<nw_grid(total, B), B, 0, s>>>(h->boxes, total, h->tboxes);
    NW_LAUNCH_CHECK();
    k_tri_extents<<<nw_grid(h->F, B), B, 0, s>>>(h->sfaces, h->posq, h->F, h->leaf_of_slot, leaf0, leaf_level, h->parent_g, h->tboxes);
    NW_LAUNCH_CHECK();
    k_tbox_decode<<<nw_grid(total - tl.off[1], B), B, 0, s>>>(h->tboxes, tl.off[1], total - tl.off[1], h->surf_bits);
    NW_LAUNCH_CHECK();
    return NW_OK;
}

// the queries, the slack of the call, the triangle-bounded boxes and k_surface_nearest: h->surf_dist (and surf_face /
// surf_closest when asked for) in the caller's order
static int surface_walk(nw_ctx *h, const void *q, int q_is_f64, int64_t Q, bool want_face, bool want_closest, SurfaceArgs &a,
                        bool &f64) {
    cudaStream_t s = h->stream;
    const TreeLevels &tl = h->tl;
    const int leaf_level = tl.n_levels - 1, leaf0 = tl.off[leaf_level], total = leaf0 + tl.count[leaf_level];

    // queries: the resident points (sorted SoA, results scattered to the caller's order through perm) or a copy of the caller's
    f64 = q ? q_is_f64 != 0 : h->px64 != nullptr;
    a.Q = Q;
    if (q) {
        const size_t bytes = (f64 ? 8 : 4) * 3 * (size_t)Q;
        NW_CHECK(nw_alloc(h, &h->surf_q, std::max<size_t>(bytes, 8)));
        NW_CHECK(nw_h2d(h, h->surf_q, q, bytes));
        const size_t el = f64 ? 8 : 4;
        a.qx = h->surf_q; a.qy = h->surf_q + el; a.qz = h->surf_q + 2 * el; a.stride = 3;
        a.perm = nullptr; a.seed = nullptr;
    } else {
        if (f64) { a.qx = h->px64; a.qy = h->py64; a.qz = h->pz64; }
        else { a.qx = h->px; a.qy = h->py; a.qz = h->pz; }
        a.stride = 1;
        a.perm = h->perm; a.seed = h->slot;
    }

    NW_CHECK(nw_surface_boxes(h, a.qx, a.qy, a.qz, Q, a.stride, f64));

    // the search
    const size_t nq = (size_t)std::max<int64_t>(Q, 1);
    NW_CHECK(nw_alloc(h, &h->surf_dist, nq));
    if (want_face) NW_CHECK(nw_alloc(h, &h->surf_face, nq));
    if (want_closest) NW_CHECK(nw_alloc(h, &h->surf_closest, 3 * nq));
    a.tb = h->tboxes; a.parent = h->parent_g; a.kids = h->kids; a.leaf_of_slot = h->leaf_of_slot; a.sfaces = h->sfaces; a.posq = h->posq;
    a.leaf0 = leaf0; a.leaf_level = leaf_level; a.n_nodes = total; a.F = h->F;
    a.dist = h->surf_dist; a.face = want_face ? h->surf_face : nullptr; a.closest = want_closest ? h->surf_closest : nullptr;
    if (Q > 0) {
        if (f64) k_surface_nearest<double><<<nw_grid(Q, 128), 128, 0, s>>>(a);
        else k_surface_nearest<float><<<nw_grid(Q, 128), 128, 0, s>>>(a);
        NW_LAUNCH_CHECK();
    }
    return NW_OK;
}

extern "C" int nw_surface_distance(nw_ctx *h, const void *q, int q_is_f64, int64_t Q, double *dist, int32_t *face, double *closest,
                                   double summary[3]) {
    if (!h) return NW_ERR_ARG;
    NW_CHECK(surface_check(h, "nw_surface_distance", q, Q));
    NW_CUDA(cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    SurfaceArgs a;
    bool f64;
    NW_CHECK(surface_walk(h, q, q_is_f64, Q, face != nullptr, closest != nullptr, a, f64));
    if (summary) {
        NW_CHECK(nw_alloc(h, &h->surf_part, (size_t)4 * NW_SUM_BLOCKS + 4));
        k_dist_partials<<<NW_SUM_BLOCKS, 256, 0, s>>>(h->surf_dist, Q, h->surf_part);
        NW_LAUNCH_CHECK();
        k_dist_summary<<<1, NW_SUM_BLOCKS, 0, s>>>(h->surf_part, h->surf_part + 4 * NW_SUM_BLOCKS);
        NW_LAUNCH_CHECK();
        NW_CUDA(cudaMemcpyAsync(summary, h->surf_part + 4 * NW_SUM_BLOCKS, sizeof(double) * 3, cudaMemcpyDeviceToHost, s));
    }
    if (Q > 0) {
        if (dist) NW_CUDA(cudaMemcpyAsync(dist, h->surf_dist, sizeof(double) * Q, cudaMemcpyDeviceToHost, s));
        if (face) NW_CUDA(cudaMemcpyAsync(face, h->surf_face, sizeof(int32_t) * Q, cudaMemcpyDeviceToHost, s));
        if (closest) NW_CUDA(cudaMemcpyAsync(closest, h->surf_closest, sizeof(double) * 3 * Q, cudaMemcpyDeviceToHost, s));
    }
    NW_CUDA(cudaStreamSynchronize(s));
    return NW_OK;
}

// The twin table, the vertex -> face CSR and the defect counts of the current topology; rebuilt only when topo_gen moved.
static int signed_tables(nw_ctx *h) {
    if (h->sgn_gen == h->topo_gen) return NW_OK;
    cudaStream_t s = h->stream;
    const int M = h->M, F = h->F, n = 3 * F, B = 256;
    NW_CHECK(nw_alloc(h, &h->sgn_twin, (size_t)n)); NW_CHECK(nw_alloc(h, &h->sgn_vface, (size_t)n));
    NW_CHECK(nw_alloc(h, &h->sgn_voff, (size_t)M + 1));
    NW_CHECK(nw_alloc(h, &h->sgn_k0, (size_t)n)); NW_CHECK(nw_alloc(h, &h->sgn_k1, (size_t)n));
    NW_CHECK(nw_alloc(h, &h->sgn_i0, (size_t)n)); NW_CHECK(nw_alloc(h, &h->sgn_i1, (size_t)n));
    NW_CHECK(nw_alloc(h, &h->sgn_cnt, (size_t)M + 1 + 5));
    int *defects = h->sgn_cnt + M + 1;
    NW_CUDA(cudaMemsetAsync(h->sgn_cnt, 0, sizeof(int) * ((size_t)M + 1 + 5), s));
    NW_CUDA(cudaMemsetAsync(h->sgn_twin, 0xff, sizeof(int) * (size_t)n, s));
    // edges: half-edges sorted by their undirected key, one thread per run
    k_halfedge_keys<<<nw_grid(n, B), B, 0, s>>>(h->faces, F, h->sgn_k0, h->sgn_i0, defects);
    NW_LAUNCH_CHECK();
    size_t tmp = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, tmp, h->sgn_k0, h->sgn_k1, h->sgn_i0, h->sgn_i1, n, 0, 64, s);
    if (tmp > h->cub_tmp_bytes) { NW_CHECK(nw_alloc(h, (char **)&h->cub_tmp, tmp)); h->cub_tmp_bytes = tmp; }
    NW_CUDA(cub::DeviceRadixSort::SortPairs(h->cub_tmp, tmp, h->sgn_k0, h->sgn_k1, h->sgn_i0, h->sgn_i1, n, 0, 64, s));
    k_edge_runs<<<nw_grid(n, B), B, 0, s>>>(h->sgn_k1, h->sgn_i1, h->faces, n, h->sgn_twin, defects);
    NW_LAUNCH_CHECK();
    // vertex -> incident face rows: (vertex, row) keys sorted, counts scanned into offsets
    k_corner_keys<<<nw_grid(n, B), B, 0, s>>>(h->faces, n, h->sgn_k0, h->sgn_cnt);
    NW_LAUNCH_CHECK();
    tmp = 0;
    cub::DeviceRadixSort::SortKeys(nullptr, tmp, h->sgn_k0, h->sgn_k1, n, 0, 64, s);
    if (tmp > h->cub_tmp_bytes) { NW_CHECK(nw_alloc(h, (char **)&h->cub_tmp, tmp)); h->cub_tmp_bytes = tmp; }
    NW_CUDA(cub::DeviceRadixSort::SortKeys(h->cub_tmp, tmp, h->sgn_k0, h->sgn_k1, n, 0, 64, s));
    k_low_words<<<nw_grid(n, B), B, 0, s>>>(h->sgn_k1, n, h->sgn_vface);
    NW_LAUNCH_CHECK();
    tmp = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tmp, h->sgn_cnt, h->sgn_voff, M + 1, s);
    if (tmp > h->cub_tmp_bytes) { NW_CHECK(nw_alloc(h, (char **)&h->cub_tmp, tmp)); h->cub_tmp_bytes = tmp; }
    NW_CUDA(cub::DeviceScan::ExclusiveSum(h->cub_tmp, tmp, h->sgn_cnt, h->sgn_voff, M + 1, s));
    k_vertex_fans<<<nw_grid(M, B), B, 0, s>>>(h->faces, h->sgn_twin, h->sgn_voff, h->sgn_vface, M, defects);
    NW_LAUNCH_CHECK();
    h->launches += 3;
    NW_CUDA(cudaMemcpyAsync(h->sgn_defects, defects, sizeof(h->sgn_defects), cudaMemcpyDeviceToHost, s));
    NW_CUDA(cudaStreamSynchronize(s));
    h->sgn_gen = h->topo_gen;
    return NW_OK;
}

extern "C" int nw_surface_signed_distance(nw_ctx *h, const void *q, int q_is_f64, int64_t Q, double *sdist, int32_t *face,
                                          double *closest, double *volume) {
    if (!h) return NW_ERR_ARG;
    NW_CHECK(surface_check(h, "nw_surface_signed_distance", q, Q));
    NW_CUDA(cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    const int M = h->M, F = h->F, B = 256;
    NW_CHECK(signed_tables(h));
    const int *dc = h->sgn_defects;
    if (dc[0] || dc[1] || dc[2] || dc[3] || dc[4]) {
        char msg[512];
        snprintf(msg, sizeof(msg),
                 "nw_surface_signed_distance: the mesh does not bound a solid (it must be closed, edge-manifold and consistently "
                 "oriented): %d boundary edges, %d edges on more than two faces, %d edges whose two faces traverse them the same "
                 "way, %d faces that repeat a vertex, %d vertices whose faces form more than one fan",
                 dc[0], dc[1], dc[2], dc[3], dc[4]);
        h->err = msg;
        return NW_ERR_ARG;
    }
    // at the current positions: vertex pseudonormals, then the signed volume about the centre of the vertices' bounding box
    NW_CHECK(nw_alloc(h, &h->sgn_nv, (size_t)3 * M));
    NW_CHECK(nw_alloc(h, &h->sgn_bbox, (size_t)6));
    NW_CHECK(nw_alloc(h, &h->sgn_vpart, (size_t)NW_SUM_BLOCKS + 1));
    NW_CUDA(cudaMemsetAsync(h->sgn_bbox, 0xff, sizeof(unsigned) * 3, s));
    NW_CUDA(cudaMemsetAsync(h->sgn_bbox + 3, 0, sizeof(unsigned) * 3, s));
    k_vertex_pseudonormals<<<nw_grid(M, B), B, 0, s>>>(h->faces, h->posq, h->sgn_voff, h->sgn_vface, M, h->sgn_nv, h->sgn_bbox);
    NW_LAUNCH_CHECK();
    k_volume_partials<<<NW_SUM_BLOCKS, 256, 0, s>>>(h->faces, h->posq, F, h->sgn_bbox, h->sgn_vpart);
    NW_LAUNCH_CHECK();
    k_volume_fold<<<1, NW_SUM_BLOCKS, 0, s>>>(h->sgn_vpart, h->sgn_vpart + NW_SUM_BLOCKS);
    NW_LAUNCH_CHECK();
    double V = 0.0;
    NW_CUDA(cudaMemcpyAsync(&V, h->sgn_vpart + NW_SUM_BLOCKS, sizeof(double), cudaMemcpyDeviceToHost, s));
    NW_CUDA(cudaStreamSynchronize(s));
    if (!(std::isfinite(V) && V != 0.0)) {
        char msg[256];
        snprintf(msg, sizeof(msg), "nw_surface_signed_distance: the signed volume of the mesh is %g (a non-finite corner, or a "
                 "surface that encloses nothing): inside and outside are undefined", V);
        h->err = msg;
        return NW_ERR_ARG;
    }
    if (volume) *volume = std::fabs(V);
    if (Q == 0) return NW_OK;

    SurfaceArgs a;
    bool f64;
    NW_CHECK(surface_walk(h, q, q_is_f64, Q, true, closest != nullptr, a, f64));
    SignArgs g;
    g.Q = Q; g.qx = a.qx; g.qy = a.qy; g.qz = a.qz; g.stride = a.stride; g.perm = a.perm;
    g.faces = h->faces; g.twin = h->sgn_twin; g.posq = h->posq; g.nv = h->sgn_nv; g.vol = h->sgn_vpart + NW_SUM_BLOCKS;
    g.face = h->surf_face; g.dist = h->surf_dist;
    if (f64) k_surface_sign<double><<<nw_grid(Q, 128), 128, 0, s>>>(g);
    else k_surface_sign<float><<<nw_grid(Q, 128), 128, 0, s>>>(g);
    NW_LAUNCH_CHECK();
    if (sdist) NW_CUDA(cudaMemcpyAsync(sdist, h->surf_dist, sizeof(double) * Q, cudaMemcpyDeviceToHost, s));
    if (face) NW_CUDA(cudaMemcpyAsync(face, h->surf_face, sizeof(int32_t) * Q, cudaMemcpyDeviceToHost, s));
    if (closest) NW_CUDA(cudaMemcpyAsync(closest, h->surf_closest, sizeof(double) * 3 * Q, cudaMemcpyDeviceToHost, s));
    NW_CUDA(cudaStreamSynchronize(s));
    return NW_OK;
}

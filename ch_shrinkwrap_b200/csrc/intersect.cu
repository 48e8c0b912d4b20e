// intersect.cu -- exact self-intersections of the handle's triangle mesh (nw_self_intersections).
//
// The signed distance and the enclosed volume (surface.cu) mean something only on an EMBEDDED mesh: no two faces cross or
// touch except along the edges and vertices they share.  The topology checks of nw_surface_signed_distance cannot see a fold
// (a vertex pushed through the opposite sheet of a thin region, an edge folded over); this call lists the faces that do.
//
// Contract.  Faces f < g (rows of mesh.faces) intersect when their closed triangles share a point their shared vertex
// INDICES do not explain: none shared -- any common point; one shared vertex s -- the edge of either face opposite s meets
// the other closed face (every common point other than s makes such a contact); a shared edge uv with opposite corners p, q
// -- p and q coplanar with uv and strictly on the same side of line uv (a fold-over); three shared -- always.  Degenerate
// faces (collinear corners, exactly: all three axis projections have zero area) and faces with a non-finite corner are not
// tested, only counted.
//
// Broad phase (k_self_pairs): one thread per sorted face slot walks the triangle-bounded boxes of nw_surface_boxes (the
// octree of the fit's search, intervals over face corners, surface.cu) with the stackless walk nw_walk_subtree.  A node
// is opened when its (widened) intervals overlap those of the face's three corners projected onto its frame with the
// operations of k_tri_extents, widened by the same slack: a common point projects into both, so the test only prunes.
// Each pair is visited once, by its lower slot: a node whose slots all lie at or below the thread's own (node slot ranges are
// contiguous) is skipped without a box test.  In a leaf, the float32 bounding boxes of the two triangles (exact: min and max
// round nothing) must overlap; such a pair is a candidate.
//
// Narrow phase: one primitive, the closed segment-versus-triangle test, built on the signs of orient3d / orient2d of the
// float32 corners.  Each sign is decided by an fp64 filter with Shewchuk's forward error bounds (float32 inputs keep every
// difference, product and bound of it in the normal fp64 range, so the bounds hold; the file is compiled -fmad=false so the
// operations are the written ones) and, when the filter cannot decide, exactly with fixed-width integers (exact_orient3d).
// So the list is exact, and invariant under winding reversal, face-row permutation and scaling by powers of two; it is sorted
// by (f, g) and does not depend on scheduling.  tests/intersect_oracle.py restates the contract independently, with rational
// intersection points instead of orientation signs.
#include <cfloat>
#include <cstdio>
#include <cub/cub.cuh>
#include "common.cuh"

namespace {

typedef unsigned long long u64;

// ---- exact stage: fixed-width integers ---------------------------------------------------------------------------------
// A finite float32 is an integer multiple of 2^-149 below 2^128, so times 2^149 it is an integer below 2^277; a coordinate
// difference (below 2^278) fits five 64-bit limbs as a two's complement number, a product of three differences (below
// 2^834) fits 14 limbs, and so does the six-term determinant (below 2^837) with its sign.
#define NW_XD 5
#define NW_XP 14

__device__ __forceinline__ void fixed_negate(u64 *w, int n) {
    u64 c = 1;
    for (int k = 0; k < n; ++k) { const u64 t = ~w[k] + c; c = (c && t == 0) ? 1 : 0; w[k] = t; }
}
// x * 2^149 as a two's complement integer
__device__ __forceinline__ void fixed_from_float(const float x, u64 (&w)[NW_XD]) {
    const unsigned b = __float_as_uint(x), e = (b >> 23) & 0xffu;
    const u64 m = (u64)((b & 0x7fffffu) | (e ? 0x800000u : 0u));
    const int sh = e ? (int)e - 1 : 0, q = sh >> 6, r = sh & 63;
    for (int k = 0; k < NW_XD; ++k) w[k] = 0;
    w[q] = m << r;
    if (r > 40) w[q + 1] = m >> (64 - r);
    if (b >> 31) fixed_negate(w, NW_XD);
}
// o = |a| * |b| (schoolbook; a * b + o + carry < 2^128 at every step, so the high word never overflows)
template <int NA, int NB>
__device__ __forceinline__ void fixed_mul(const u64 (&a)[NA], const u64 (&b)[NB], u64 (&o)[NA + NB]) {
    for (int k = 0; k < NA + NB; ++k) o[k] = 0;
#pragma unroll 1
    for (int i = 0; i < NA; ++i) {
        u64 carry = 0;
        for (int j = 0; j < NB; ++j) {
            const u64 lo = a[i] * b[j];
            u64 hi = __umul64hi(a[i], b[j]);
            u64 t = o[i + j] + lo;
            hi += t < lo;
            t += carry;
            hi += t < carry;
            o[i + j] = t;
            carry = hi;
        }
        o[i + NB] = carry;
    }
}

// Sign of det[a - d; b - d; c - d], exactly.  Out of line so that its arrays stay off the walk's registers.
__device__ __noinline__ int exact_orient3d(float ax, float ay, float az, float bx, float by, float bz, float cx, float cy, float cz,
                                           float dx, float dy, float dz) {
    const float p[3][3] = {{ax, ay, az}, {bx, by, bz}, {cx, cy, cz}}, q[3] = {dx, dy, dz};
    u64 mag[3][3][NW_XD];                       // |p[i][k] - q[k]|
    bool neg[3][3];
#pragma unroll 1
    for (int k = 0; k < 3; ++k) {
        u64 d[NW_XD];
        fixed_from_float(q[k], d);
        for (int i = 0; i < 3; ++i) {
            u64 v[NW_XD];
            fixed_from_float(p[i][k], v);
            u64 br = 0;
            for (int l = 0; l < NW_XD; ++l) {
                const u64 t = v[l] - d[l], t2 = t - br;
                br = (v[l] < d[l] || t < br) ? 1 : 0;
                mag[i][k][l] = t2;
            }
            neg[i][k] = mag[i][k][NW_XD - 1] >> 63;
            if (neg[i][k]) fixed_negate(mag[i][k], NW_XD);
        }
    }
    // the six terms of the determinant: sign(sigma) * prod_i (p[i] - q)[sigma(i)]
    const int perm[6][3] = {{0, 1, 2}, {1, 2, 0}, {2, 0, 1}, {0, 2, 1}, {2, 1, 0}, {1, 0, 2}};
    u64 acc[NW_XP];
    for (int l = 0; l < NW_XP; ++l) acc[l] = 0;
#pragma unroll 1
    for (int t = 0; t < 6; ++t) {
        u64 p2[2 * NW_XD], p3[3 * NW_XD];
        fixed_mul<NW_XD, NW_XD>(mag[0][perm[t][0]], mag[1][perm[t][1]], p2);
        fixed_mul<2 * NW_XD, NW_XD>(p2, mag[2][perm[t][2]], p3);
        const bool minus = (t >= 3) != (neg[0][perm[t][0]] != (neg[1][perm[t][1]] != neg[2][perm[t][2]]));
        u64 c = 0;
        for (int l = 0; l < NW_XP; ++l) {
            if (minus) {
                const u64 d = acc[l] - p3[l], d2 = d - c;
                c = (acc[l] < p3[l] || d < c) ? 1 : 0;
                acc[l] = d2;
            } else {
                const u64 s = acc[l] + p3[l], s2 = s + c;
                c = (s < p3[l] || s2 < c) ? 1 : 0;
                acc[l] = s2;
            }
        }
    }
    if (acc[NW_XP - 1] >> 63) return -1;
    for (int l = 0; l < NW_XP; ++l) if (acc[l]) return 1;
    return 0;
}

// ---- predicates: fp64 filter (Shewchuk 1997, the A bounds), then the exact stage ------------------------------------------
#define NW_EPS 1.1102230246251565e-16          // 2^-53
// The predicates are out of line (each carries a call of the exact stage, which would otherwise inflate the register count of
// every caller) and return sign + 1, plus 4 when the exact stage decided.
// sign of det[a - d; b - d; c - d] (Shewchuk's orient3d)
__device__ __noinline__ int orient3d_code(const float4 a, const float4 b, const float4 c, const float4 d) {
    const double adx = (double)a.x - (double)d.x, bdx = (double)b.x - (double)d.x, cdx = (double)c.x - (double)d.x;
    const double ady = (double)a.y - (double)d.y, bdy = (double)b.y - (double)d.y, cdy = (double)c.y - (double)d.y;
    const double adz = (double)a.z - (double)d.z, bdz = (double)b.z - (double)d.z, cdz = (double)c.z - (double)d.z;
    const double bdxcdy = bdx * cdy, cdxbdy = cdx * bdy, cdxady = cdx * ady, adxcdy = adx * cdy, adxbdy = adx * bdy, bdxady = bdx * ady;
    const double det = adz * (bdxcdy - cdxbdy) + bdz * (cdxady - adxcdy) + cdz * (adxbdy - bdxady);
    const double perm = (fabs(bdxcdy) + fabs(cdxbdy)) * fabs(adz) + (fabs(cdxady) + fabs(adxcdy)) * fabs(bdz) +
                        (fabs(adxbdy) + fabs(bdxady)) * fabs(cdz);
    // products of nonzero differences never round to zero in this range: a zero permanent is an exactly zero determinant
    if (perm == 0.0) return 1;
    const double bound = (7.0 + 56.0 * NW_EPS) * NW_EPS * perm;
    if (det > bound) return 2;
    if (-det > bound) return 0;
    return 5 + exact_orient3d(a.x, a.y, a.z, b.x, b.y, b.z, c.x, c.y, c.z, d.x, d.y, d.z);
}
// sign of (a - c) x (b - c) (Shewchuk's orient2d)
__device__ __noinline__ int orient2d_code(const float2 a, const float2 b, const float2 c) {
    const double l = ((double)a.x - (double)c.x) * ((double)b.y - (double)c.y);
    const double r = ((double)a.y - (double)c.y) * ((double)b.x - (double)c.x);
    const double det = l - r, sum = fabs(l) + fabs(r);
    if (sum == 0.0) return 1;
    const double bound = (3.0 + 16.0 * NW_EPS) * NW_EPS * sum;
    if (det > bound) return 2;
    if (-det > bound) return 0;
    // det[(a, 0) - (c, 1); (b, 0) - (c, 1); (c, 0) - (c, 1)] = -orient2d(a, b, c)
    return 5 - exact_orient3d(a.x, a.y, 0.f, b.x, b.y, 0.f, c.x, c.y, 0.f, c.x, c.y, 1.f);
}

// the signs; n counts the evaluations the filter left to the exact stage
__device__ __forceinline__ int orient3d(const float4 a, const float4 b, const float4 c, const float4 d, u64 &n) {
    const int r = orient3d_code(a, b, c, d);
    n += r >> 2;
    return (r & 3) - 1;
}
__device__ __forceinline__ int orient2d(const float2 a, const float2 b, const float2 c, u64 &n) {
    const int r = orient2d_code(a, b, c);
    n += r >> 2;
    return (r & 3) - 1;
}

// axis plane k: 0 drops z, 1 drops y, 2 drops x
__device__ __forceinline__ float2 drop(const float4 p, int k) {
    return k == 0 ? make_float2(p.x, p.y) : k == 1 ? make_float2(p.x, p.z) : make_float2(p.y, p.z);
}
// the first axis plane in which the triangle has non-zero area (3: none, the triangle is degenerate)
__device__ __forceinline__ int flat_axis(const float4 a, const float4 b, const float4 c, u64 &n) {
    for (int k = 0; k < 3; ++k)
        if (orient2d(drop(a, k), drop(b, k), drop(c, k), n) != 0) return k;
    return 3;
}

// ---- closed 2-D tests (coplanar case) --------------------------------------------------------------------------------
// r, collinear with the segment pq, lies on it
__device__ __forceinline__ bool on_segment(const float2 p, const float2 q, const float2 r) {
    return fminf(p.x, q.x) <= r.x && r.x <= fmaxf(p.x, q.x) && fminf(p.y, q.y) <= r.y && r.y <= fmaxf(p.y, q.y);
}
__device__ __forceinline__ bool segments_meet(const float2 p, const float2 q, const float2 a, const float2 b, u64 &n) {
    const int d1 = orient2d(p, q, a, n), d2 = orient2d(p, q, b, n), d3 = orient2d(a, b, p, n), d4 = orient2d(a, b, q, n);
    if (d1 * d2 < 0 && d3 * d4 < 0) return true;
    return (d1 == 0 && on_segment(p, q, a)) || (d2 == 0 && on_segment(p, q, b)) || (d3 == 0 && on_segment(a, b, p)) ||
           (d4 == 0 && on_segment(a, b, q));
}
// r in the closed triangle abc of orientation o != 0
__device__ __forceinline__ bool in_triangle(const float2 a, const float2 b, const float2 c, int o, const float2 r, u64 &n) {
    return orient2d(a, b, r, n) * o >= 0 && orient2d(b, c, r, n) * o >= 0 && orient2d(c, a, r, n) * o >= 0;
}

// ---- the primitive: closed segment pq against the closed, non-degenerate triangle t ------------------------------------
// op, oq: orient3d(t, p) and orient3d(t, q)
__device__ __forceinline__ bool segment_meets_triangle(const float4 p, const float4 q, int op, int oq, const float4 (&t)[3], u64 &n) {
    if (op * oq > 0) return false;
    if (op == 0 && oq == 0) {
        const int k = flat_axis(t[0], t[1], t[2], n);
        const float2 a = drop(t[0], k), b = drop(t[1], k), c = drop(t[2], k), p2 = drop(p, k), q2 = drop(q, k);
        const int o = orient2d(a, b, c, n);
        return in_triangle(a, b, c, o, p2, n) || in_triangle(a, b, c, o, q2, n) || segments_meet(p2, q2, a, b, n) ||
               segments_meet(p2, q2, b, c, n) || segments_meet(p2, q2, c, a, n);
    }
    // the line pq crosses the plane inside the segment: it meets the closed triangle iff it passes no edge on the far side
    const int s0 = orient3d(p, q, t[0], t[1], n), s1 = orient3d(p, q, t[1], t[2], n), s2 = orient3d(p, q, t[2], t[0], n);
    return !((s0 > 0 || s1 > 0 || s2 > 0) && (s0 < 0 || s1 < 0 || s2 < 0));
}

// element k of a 3-array by selects (a run-time index would put the array in local memory)
template <typename T>
__device__ __forceinline__ T pick(const T (&v)[3], int k) { return k == 0 ? v[0] : k == 1 ? v[1] : v[2]; }

__device__ __forceinline__ bool pair_meets(const int (&fi)[3], const float4 (&x)[3], const int (&gi)[3], const float4 (&y)[3], u64 &n) {
    int in_g[3], shared = 0;                      // corner k of f is corner in_g[k] of g, or -1
    for (int k = 0; k < 3; ++k) {
        in_g[k] = fi[k] == gi[0] ? 0 : fi[k] == gi[1] ? 1 : fi[k] == gi[2] ? 2 : -1;
        shared += in_g[k] >= 0;
    }
    if (shared == 3) return true;
    if (shared == 2) {
        // the shared edge uv and the opposite corners p of f, q of g: a coplanar fold-over
        const int kp = in_g[0] < 0 ? 0 : in_g[1] < 0 ? 1 : 2;
        const int iu = pick(in_g, (kp + 1) % 3), iv = pick(in_g, (kp + 2) % 3);
        const float4 u = pick(y, iu), v = pick(y, iv), p = pick(x, kp), q = pick(y, 3 - iu - iv);
        if (orient3d(u, v, p, q, n) != 0) return false;
        const int k = flat_axis(u, v, p, n);
        return orient2d(drop(u, k), drop(v, k), drop(p, k), n) * orient2d(drop(u, k), drop(v, k), drop(q, k), n) > 0;
    }
    if (shared == 1) {
        // the edge of each face opposite the shared vertex against the other face
        const int ks = in_g[0] >= 0 ? 0 : in_g[1] >= 0 ? 1 : 2, ls = pick(in_g, ks);
        const float4 p = pick(x, (ks + 1) % 3), q = pick(x, (ks + 2) % 3), r = pick(y, (ls + 1) % 3), s = pick(y, (ls + 2) % 3);
        if (segment_meets_triangle(p, q, orient3d(y[0], y[1], y[2], p, n), orient3d(y[0], y[1], y[2], q, n), y, n)) return true;
        return segment_meets_triangle(r, s, orient3d(x[0], x[1], x[2], r, n), orient3d(x[0], x[1], x[2], s, n), x, n);
    }
    // no shared vertex: plane-side rejection both ways, then the six edges
    int sx[3], sy[3];
    for (int k = 0; k < 3; ++k) sx[k] = orient3d(y[0], y[1], y[2], x[k], n);
    if ((sx[0] > 0 && sx[1] > 0 && sx[2] > 0) || (sx[0] < 0 && sx[1] < 0 && sx[2] < 0)) return false;
    for (int k = 0; k < 3; ++k) sy[k] = orient3d(x[0], x[1], x[2], y[k], n);
    if ((sy[0] > 0 && sy[1] > 0 && sy[2] > 0) || (sy[0] < 0 && sy[1] < 0 && sy[2] < 0)) return false;
    for (int k = 0; k < 3; ++k) {
        const int l = (k + 1) % 3;
        if (segment_meets_triangle(x[k], x[l], sx[k], sx[l], y, n)) return true;
        if (segment_meets_triangle(y[k], y[l], sy[k], sy[l], x, n)) return true;
    }
    return false;
}
// The pair test of the contract for the faces of two sorted slots, out of line so that the walk keeps few registers:
// (exact-stage calls << 1) | the faces intersect.  Arguments by value: an array argument would live in local memory.
__device__ __noinline__ u64 faces_meet(const int4 *__restrict__ sfaces, const float4 *__restrict__ pos, int sf_, int sg_) {
    const int4 f = __ldg(&sfaces[sf_]), g = __ldg(&sfaces[sg_]);
    const int fi[3] = {f.x, f.y, f.z}, gi[3] = {g.x, g.y, g.z};
    const float4 x[3] = {__ldg(&pos[f.x]), __ldg(&pos[f.y]), __ldg(&pos[f.z])}, y[3] = {__ldg(&pos[g.x]), __ldg(&pos[g.y]), __ldg(&pos[g.z])};
    u64 n = 0;
    const bool hit = pair_meets(fi, x, gi, y, n);
    return (n << 1) | (hit ? 1u : 0u);
}

__device__ __forceinline__ bool finite4(const float4 v) { return fabsf(v.x) <= FLT_MAX && fabsf(v.y) <= FLT_MAX && fabsf(v.z) <= FLT_MAX; }

// ---- per slot: which faces are tested, and the last slot of every node -----------------------------------------------
// flag: 0 tested, 1 degenerate, 2 a non-finite corner.  cnt: [2] exact-stage calls, [3] degenerate, [4] non-finite faces.
// A node's slots are contiguous: the slot that ends a leaf ends it, and every ancestor of which the path is the last child.
__global__ void __launch_bounds__(256) k_self_prep(const int4 *__restrict__ sfaces, const float4 *__restrict__ pos, int F,
                                                   const int *__restrict__ leaf_of_slot, int leaf0, const int *__restrict__ parent_g,
                                                   const int2 *__restrict__ kids, uint8_t *__restrict__ flag, int *__restrict__ last,
                                                   u64 *__restrict__ cnt) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= F) return;
    const int4 sf = sfaces[i];
    const float4 a = pos[sf.x], b = pos[sf.y], c = pos[sf.z];
    u64 n = 0;
    uint8_t fl = 0;
    if (!(finite4(a) && finite4(b) && finite4(c))) { fl = 2; atomicAdd(cnt + 4, 1ull); }
    else if (flat_axis(a, b, c, n) == 3) { fl = 1; atomicAdd(cnt + 3, 1ull); }
    if (n) atomicAdd(cnt + 2, n);
    flag[i] = fl;
    int node = leaf0 + leaf_of_slot[i];
    int2 k = kids[node];
    if (i != k.x + k.y - 1) return;
    last[node] = i;
    while (node != 0) {
        const int p = nw_link_node(parent_g[node]);
        k = kids[p];
        if (k.x + k.y - 1 != node) break;
        last[p] = i;
        node = p;
    }
}

// ---- the walk ----------------------------------------------------------------------------------------------------------
struct SelfArgs {
    OctreeView oct;                     // over h->tboxes
    const int *last;
    const int4 *sfaces;
    const float4 *pos;
    const uint8_t *flag;
    const unsigned *bits;               // the slack of the call (nw_surface_boxes)
    u64 *keys;                          // (f << 32) | g, f < g
    u64 cap;
    u64 *cnt;                           // [0] pairs found, [1] candidates, [2] exact-stage calls
};

struct SelfWalk {
    const SelfArgs &a;
    int i;                              // own slot
    int face;                           // own face row
    float4 x[3];
    float lo[3], hi[3];                 // own float32 bounding box
    float w;                            // the slack of the call
    u64 cand = 0, n = 0;

    __device__ __forceinline__ SelfWalk(const SelfArgs &a_) : a(a_) {}
    __device__ __forceinline__ bool tick() const { return false; }
    // the node's intervals overlap those of the face's corners on its frame, each side widened by the slack
    __device__ __forceinline__ bool open(int node, int &link) const {
        const Box *bp = &a.oct.boxes[node];
        const float4 bd = __ldg(&bp->d);
        link = __float_as_int(bd.z);
        if (__ldg(&a.last[node]) <= i) return false;
        const float4 ba = __ldg(&bp->a), bb = __ldg(&bp->b), bc = __ldg(&bp->c);
        float l[3], h[3];
        project_frame(ba, bb, bc, x[0].x, x[0].y, x[0].z, l[0], l[1], l[2]);
        h[0] = l[0]; h[1] = l[1]; h[2] = l[2];
        for (int c = 1; c < 3; ++c) {
            float p[3];
            project_frame(ba, bb, bc, x[c].x, x[c].y, x[c].z, p[0], p[1], p[2]);
            for (int k = 0; k < 3; ++k) { l[k] = fminf(l[k], p[k]); h[k] = fmaxf(h[k], p[k]); }
        }
        return l[0] - w <= bd.x && h[0] + w >= bb.z && l[1] - w <= bd.y && h[1] + w >= bb.w && l[2] - w <= bc.w && h[2] + w >= bd.w;
    }
    __device__ __forceinline__ void leaf(int node) {
        NW_ASSERT(node >= a.oct.leaf0 && node < a.oct.n_nodes);
        const int2 k = __ldg(&a.oct.kids[node]);
        NW_ASSERT(k.x >= 0 && k.y >= 0 && k.x + k.y <= a.oct.n_slots);
        for (int s = max(k.x, i + 1); s < k.x + k.y; ++s) {
            if (__ldg(&a.flag[s])) continue;
            const int4 sf = __ldg(&a.sfaces[s]);
            const float4 y[3] = {__ldg(&a.pos[sf.x]), __ldg(&a.pos[sf.y]), __ldg(&a.pos[sf.z])};
            if (fminf(y[0].x, fminf(y[1].x, y[2].x)) > hi[0] || fmaxf(y[0].x, fmaxf(y[1].x, y[2].x)) < lo[0] ||
                fminf(y[0].y, fminf(y[1].y, y[2].y)) > hi[1] || fmaxf(y[0].y, fmaxf(y[1].y, y[2].y)) < lo[1] ||
                fminf(y[0].z, fminf(y[1].z, y[2].z)) > hi[2] || fmaxf(y[0].z, fmaxf(y[1].z, y[2].z)) < lo[2])
                continue;
            ++cand;
            const u64 r = faces_meet(a.sfaces, a.pos, i, s);
            n += r >> 1;
            if (!(r & 1)) continue;
            const u64 j = atomicAdd(a.cnt, 1ull);
            if (j < a.cap) a.keys[j] = ((u64)(unsigned)min(face, sf.w) << 32) | (unsigned)max(face, sf.w);
        }
    }
    // the root's children in turn (the root has no box: the intervals are measured from level 1 down)
    __device__ __forceinline__ void walk() {
        const int2 k = __ldg(&a.oct.kids[0]);
        for (int c = k.x; c < k.x + k.y; ++c) nw_walk_subtree(*this, a.oct, c);
    }
};

__global__ void __launch_bounds__(128) k_self_pairs(const __grid_constant__ SelfArgs a) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.oct.n_slots || __ldg(&a.flag[i])) return;
    SelfWalk w(a);
    w.i = i;
    const int4 sf = __ldg(&a.sfaces[i]);
    w.face = sf.w;
    w.x[0] = __ldg(&a.pos[sf.x]); w.x[1] = __ldg(&a.pos[sf.y]); w.x[2] = __ldg(&a.pos[sf.z]);
    w.lo[0] = fminf(w.x[0].x, fminf(w.x[1].x, w.x[2].x)); w.hi[0] = fmaxf(w.x[0].x, fmaxf(w.x[1].x, w.x[2].x));
    w.lo[1] = fminf(w.x[0].y, fminf(w.x[1].y, w.x[2].y)); w.hi[1] = fmaxf(w.x[0].y, fmaxf(w.x[1].y, w.x[2].y));
    w.lo[2] = fminf(w.x[0].z, fminf(w.x[1].z, w.x[2].z)); w.hi[2] = fmaxf(w.x[0].z, fmaxf(w.x[1].z, w.x[2].z));
    w.w = call_slack(a.bits);
    w.walk();
    if (w.cand) atomicAdd(a.cnt + 1, w.cand);
    if (w.n) atomicAdd(a.cnt + 2, w.n);
}

// sorted keys -> (f, g) rows
__global__ void k_pair_rows(const u64 *__restrict__ key, int64_t n, int2 *__restrict__ out) {
    const int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (j < n) out[j] = make_int2((int)(key[j] >> 32), (int)(unsigned)key[j]);
}

}  // namespace

extern "C" int nw_self_intersections(nw_ctx *h, int32_t *pairs, int64_t capacity, int64_t *n_pairs, int64_t stats[4]) {
    if (!h) return NW_ERR_ARG;
    NW_CHECK(nw_mesh_check(h, "nw_self_intersections"));
    NW_ARG(n_pairs != nullptr, "nw_self_intersections: n_pairs must not be NULL");
    NW_ARG(capacity >= 0 && (pairs != nullptr || capacity == 0), "nw_self_intersections: pairs may be NULL only with capacity 0");
    NW_CUDA(cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    const int F = h->F;

    NW_CHECK(nw_surface_boxes(h, nullptr, nullptr, nullptr, 0, 1, false));
    SelfArgs a;
    a.oct = nw_octree_view(h, h->tboxes);
    NW_CHECK(nw_alloc(h, &h->sx_flag, (size_t)F));
    NW_CHECK(nw_alloc(h, &h->sx_last, (size_t)a.oct.n_nodes));
    NW_CHECK(nw_alloc(h, &h->sx_cnt, (size_t)5));
    NW_CUDA(cudaMemsetAsync(h->sx_cnt, 0, sizeof(u64) * 5, s));
    k_self_prep<<<nw_grid(F, 256), 256, 0, s>>>(h->sfaces, h->posq, F, h->leaf_of_slot, a.oct.leaf0, h->parent_g, h->kids, h->sx_flag,
                                                h->sx_last, h->sx_cnt);
    NW_LAUNCH_CHECK();

    // pairs into a grow-only buffer; one more pass when it was too small (the set found is the same every time)
    if (!h->sx_keys) NW_CHECK(nw_alloc(h, &h->sx_keys, (size_t)65536));
    a.last = h->sx_last; a.sfaces = h->sfaces; a.pos = h->posq; a.flag = h->sx_flag; a.bits = h->surf_bits;
    a.keys = h->sx_keys; a.cap = h->caps[(void *)&h->sx_keys] / sizeof(u64); a.cnt = h->sx_cnt;
    k_self_pairs<<<nw_grid(F, 128), 128, 0, s>>>(a);
    NW_LAUNCH_CHECK();
    u64 cnt[5];
    NW_CUDA(cudaMemcpyAsync(cnt, h->sx_cnt, sizeof(cnt), cudaMemcpyDeviceToHost, s));
    NW_CUDA(cudaStreamSynchronize(s));
    if (cnt[0] > a.cap) {
        NW_CHECK(nw_alloc(h, &h->sx_keys, (size_t)cnt[0]));
        a.keys = h->sx_keys; a.cap = h->caps[(void *)&h->sx_keys] / sizeof(u64);
        NW_CUDA(cudaMemsetAsync(h->sx_cnt, 0, sizeof(u64) * 3, s));
        k_self_pairs<<<nw_grid(F, 128), 128, 0, s>>>(a);
        NW_LAUNCH_CHECK();
        NW_CUDA(cudaMemcpyAsync(cnt, h->sx_cnt, sizeof(u64) * 3, cudaMemcpyDeviceToHost, s));
        NW_CUDA(cudaStreamSynchronize(s));
        NW_ARG(cnt[0] <= a.cap, "nw_self_intersections: the pair count changed between two passes");
    }
    const int64_t n = (int64_t)cnt[0], out = std::min(n, capacity);
    if (out > 0) {
        NW_CHECK(nw_alloc(h, &h->sx_sorted, (size_t)n));
        NW_CHECK(nw_alloc(h, &h->sx_pairs, (size_t)out));
        size_t tmp = 0;
        cub::DeviceRadixSort::SortKeys(nullptr, tmp, h->sx_keys, h->sx_sorted, (int)n, 0, 64, s);
        if (tmp > h->cub_tmp_bytes) { NW_CHECK(nw_alloc(h, (char **)&h->cub_tmp, tmp)); h->cub_tmp_bytes = tmp; }
        NW_CUDA(cub::DeviceRadixSort::SortKeys(h->cub_tmp, tmp, h->sx_keys, h->sx_sorted, (int)n, 0, 64, s));
        h->launches += 1;
        k_pair_rows<<<nw_grid(out, 256), 256, 0, s>>>(h->sx_sorted, out, h->sx_pairs);
        NW_LAUNCH_CHECK();
        NW_CUDA(cudaMemcpyAsync(pairs, h->sx_pairs, sizeof(int2) * (size_t)out, cudaMemcpyDeviceToHost, s));
        NW_CUDA(cudaStreamSynchronize(s));
    }
    *n_pairs = n;
    if (stats) { stats[0] = (int64_t)cnt[1]; stats[1] = (int64_t)cnt[2]; stats[2] = (int64_t)cnt[3]; stats[3] = (int64_t)cnt[4]; }
    return NW_OK;
}

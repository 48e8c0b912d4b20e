// hausdorff.cu -- certified bounds of the one-sided Hausdorff distance (nw_hausdorff_bounds) and of the area-weighted mean
// and RMS distances (nw_mean_distance_bounds) from a mesh A passed in to the handle's mesh B.
//
// h(A -> B) = max over the points p of A's closed triangles of d_B(p).  A branch and bound over A's triangles, one level at
// a time on the device: level 0 walks the vertices A's finite faces use (k_surface_nearest<double>, surface.cu, unseeded);
// every level then bounds max d_B over each live triangle (an entry) from its corners, retires the entries whose bound is
// within tol of the largest distance found so far, L, and splits the others at their edge midpoints, which are the next
// level's queries, seeded at the slot of an endpoint's nearest face.  The bound of an entry is the smaller of
//   convexity:  d_B <= d(., t) for one face t of B, and d(., t) is convex, so max over T of d_B <= max_k d(c_k, t); the
//               candidates t are the corners' nearest faces and the face that gave the parent its bound (so a child's bound
//               is never above its parent's), each at most 3 evaluations of the region test (closest.cuh);
//   Lipschitz:  d_B is 1-Lipschitz, so max over T of d_B <= min_k (d_k + max_j |c_j - c_k|),
// rounded up, plus the rounding allowance eps of the call (hb_eps; DESIGN.md section 4 derives it).  L only grows, so a
// retired bound stays within the final L + tol.  The order of the queries and entries comes from scans, the maxima from
// 64-bit atomics on the bits of non-negative doubles (exact, so order-free) and the witness from a lowest-index rule:
// the result is the same bits on every call.  This file is compiled with -fmad=false like surface.cu, so the region test
// performs the same operations in both.  Nothing the fit reads is written; tboxes and surf_bits are nw_surface_boxes'.
//
// nw_mean_distance_bounds runs the same set-up (hb_start), level loop, splits and seeded walks (hb_levels) with its own bound
// step: k_mb_bound brackets the integrals of d_B and d_B^2 over every entry, and fixed-order sums give each level's bracket.
#include <cfloat>
#include <cmath>
#include <cstring>
#include <string>
#include <cub/cub.cuh>
#include "common.cuh"
#include "closest.cuh"

namespace {

// ---- certified one-sided Hausdorff bounds (nw_hausdorff_bounds): branch and bound over the triangles of a mesh A -----------
// Level 0 walks A's used vertices; every level bounds max d_B over each live triangle (entry), retires the entries whose bound
// is within tol of the best distance found, and splits the others at their edge midpoints, which are the next level's queries.
#define NW_HB_MAX_LEVELS 64
struct HbEntry {
    D3 c[3];                            // corners
    double d[3];                        // their distances to B (where q[k] < 0)
    int f[3];                           // their nearest face rows of B (where q[k] < 0)
    int q[3];                           // corner k is query q[k] of this level, whose walk gives d and f; -1: known; q[0] = -2: a
                                        // level-0 face with a non-finite corner (never bounded)
    int inh;                            // the face row of B that gave the parent its convexity bound (-1: none)
    int aface;                          // the face row of A the entry lies in
};
struct HbState {
    unsigned long long lmax;            // the largest distance of this level's queries, as bits (non-negative doubles order like them)
    int larg;                           // the lowest query index that attains it
    int bad, nonfinite, b_finite;       // A's faces with an index out of range, with a non-finite corner; B has a finite face
    double L;                           // the largest distance so far (-1: none yet) and its witness: point, face of A, face of B
    double w[3];
    int wa, wb;
    unsigned long long uret, ulive;     // bits of the largest bound of the retired entries, of this level's surviving entries
};
__device__ __forceinline__ double bits2d(unsigned long long u) { return __longlong_as_double((long long)u); }
__device__ __forceinline__ unsigned long long d2bits(double v) { return (unsigned long long)__double_as_longlong(v); }

// A's faces: out-of-range and non-finite ones counted; each vertex of a finite face learns the lowest such face row
__global__ void k_hb_faces(const int *__restrict__ faces, const float *__restrict__ pos, int F, int M, int *__restrict__ vface,
                           HbState *__restrict__ st) {
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= F) return;
    const int v[3] = {faces[3 * f], faces[3 * f + 1], faces[3 * f + 2]};
    if (v[0] < 0 || v[0] >= M || v[1] < 0 || v[1] >= M || v[2] < 0 || v[2] >= M) { atomicAdd(&st->bad, 1); return; }
    for (int k = 0; k < 3; ++k)
        if (!(fabsf(pos[3 * v[k]]) <= FLT_MAX && fabsf(pos[3 * v[k] + 1]) <= FLT_MAX && fabsf(pos[3 * v[k] + 2]) <= FLT_MAX)) {
            atomicAdd(&st->nonfinite, 1);
            return;
        }
    for (int k = 0; k < 3; ++k) atomicMin(vface + v[k], f);
}
// does the handle's mesh have a finite face; its face row -> slot table
__global__ void k_hb_mesh_b(const int4 *__restrict__ sfaces, const float4 *__restrict__ posq, int F, int *__restrict__ slot,
                            HbState *__restrict__ st) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= F) return;
    const int4 sf = sfaces[s];
    slot[sf.w] = s;
    if (finite4(posq[sf.x]) && finite4(posq[sf.y]) && finite4(posq[sf.z])) st->b_finite = 1;
}
__global__ void k_hb_used(const int *__restrict__ vface, int M, int F, int *__restrict__ flag) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v <= M) flag[v] = v < M && vface[v] < F;
}
// level 0: the used vertices as queries, in vertex order, and one entry per face of A
__global__ void k_hb_vertices(const float *__restrict__ pos, const int *__restrict__ vface, const int *__restrict__ flag,
                              const int *__restrict__ idx, int M, double *__restrict__ q, int *__restrict__ qa) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= M || !flag[v]) return;
    const int i = idx[v];
    q[3 * i] = pos[3 * v]; q[3 * i + 1] = pos[3 * v + 1]; q[3 * i + 2] = pos[3 * v + 2];
    qa[i] = vface[v];
}
__global__ void k_hb_level0(const int *__restrict__ faces, const float *__restrict__ pos, const int *__restrict__ idx, int F,
                            HbEntry *__restrict__ e) {
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= F) return;
    HbEntry x;
    bool live = true;
    for (int k = 0; k < 3; ++k) {
        const int v = faces[3 * f + k];
        x.c[k] = D3{(double)pos[3 * v], (double)pos[3 * v + 1], (double)pos[3 * v + 2]};
        x.d[k] = 0.0; x.f[k] = -1;
        x.q[k] = idx[v];
        live = live && fabs(x.c[k].x) <= DBL_MAX && fabs(x.c[k].y) <= DBL_MAX && fabs(x.c[k].z) <= DBL_MAX;
    }
    if (!live) x.q[0] = -2;
    x.inh = -1; x.aface = f;
    e[f] = x;
}

// the largest distance of the level, then the lowest query that attains it, then the running maximum and its witness
// (strictly larger only: ties go to the earliest level)
__global__ void __launch_bounds__(256) k_hb_level_max(const double *__restrict__ qd, int n, HbState *__restrict__ st) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long b = i < n ? d2bits(qd[i]) : 0ull;
    for (int o = 16; o; o >>= 1) b = max(b, __shfl_xor_sync(0xffffffffu, b, o));
    if ((threadIdx.x & 31) == 0 && b) atomicMax(&st->lmax, b);
}
__global__ void __launch_bounds__(256) k_hb_level_arg(const double *__restrict__ qd, int n, HbState *__restrict__ st) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && d2bits(qd[i]) == st->lmax) atomicMin(&st->larg, i);
}
__global__ void k_hb_take(const double *__restrict__ q, const int *__restrict__ qf, const int *__restrict__ qa, HbState *__restrict__ st) {
    const double m = bits2d(st->lmax);
    if (m > st->L) {
        const int i = st->larg;
        st->L = m;
        st->w[0] = q[3 * i]; st->w[1] = q[3 * i + 1]; st->w[2] = q[3 * i + 2];
        st->wa = qa[i]; st->wb = qf[i];
    }
    st->lmax = 0ull; st->larg = 0x7fffffff; st->ulive = 0ull;
}

// distance from p to face row t of B: the operations of k_surface_nearest
__device__ __noinline__ double hb_face_dist(const D3 p, const int *__restrict__ faces, const float4 *__restrict__ posq, int t) {
    const D3 a = d3(posq[faces[3 * t]]), b = d3(posq[faces[3 * t + 1]]), c = d3(posq[faces[3 * t + 2]]);
    return sqrt(dist2(p, closest_on_triangle(p, a, b, c)));
}
// |u - v| rounded up
__device__ __forceinline__ double hb_len_ru(const D3 u, const D3 v) {
    const double x = fmax(__dsub_ru(u.x, v.x), __dsub_ru(v.x, u.x)), y = fmax(__dsub_ru(u.y, v.y), __dsub_ru(v.y, u.y)),
                 z = fmax(__dsub_ru(u.z, v.z), __dsub_ru(v.z, u.z));
    return __dsqrt_ru(__dadd_ru(__dadd_ru(__dmul_ru(x, x), __dmul_ru(y, y)), __dmul_ru(z, z)));
}
// the rounding allowance of the call: 2^-40 x the L1 bound of A's used vertices and B's vertices (k_absmax3's bits)
__device__ __forceinline__ double hb_eps(const unsigned *__restrict__ bits6) {
    double l1 = 0.0;
    for (int k = 0; k < 3; ++k) l1 = __dadd_ru(l1, (double)fmaxf(__uint_as_float(bits6[k]), __uint_as_float(bits6[3 + k])));
    return l1 * 0x1p-40;
}

// Upper bound of max d_B over each entry: the smaller of the convexity bound (one face t of B: max over the corners of
// d(c, t); candidates the corners' nearest faces and the parent's) and the Lipschitz bound (min over corners of d_i + the
// farthest corner), rounded up, plus the allowance.  Retired (ub <= L + tol) or flagged for the split.
__global__ void __launch_bounds__(128) k_hb_bound(HbEntry *__restrict__ e, int n, const double *__restrict__ qd, const int *__restrict__ qf,
                                                  const int *__restrict__ faces, const float4 *__restrict__ posq, int FB,
                                                  const unsigned *__restrict__ bits6, double tol, HbState *__restrict__ st,
                                                  int *__restrict__ flag) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i > n) return;
    if (i == n) { flag[n] = 0; return; }
    HbEntry x = e[i];
    if (x.q[0] == -2) { flag[i] = 0; return; }
    for (int k = 0; k < 3; ++k)
        if (x.q[k] >= 0) { x.d[k] = qd[x.q[k]]; x.f[k] = qf[x.q[k]]; x.q[k] = -1; }
    const int cand[4] = {x.f[0], x.f[1], x.f[2], x.inh};
    double conv = DBL_MAX * 2.0;
    int best = -1;
#pragma unroll 1
    for (int j = 0; j < 4; ++j) {
        const int t = cand[j];
        if (t < 0 || (j > 0 && t == cand[0]) || (j > 1 && t == cand[1]) || (j > 2 && t == cand[2])) continue;
        NW_ASSERT(t < FB);
        double m = 0.0;
#pragma unroll 1
        for (int k = 0; k < 3; ++k) m = fmax(m, x.f[k] == t ? x.d[k] : hb_face_dist(x.c[k], faces, posq, t));
        if (m < conv || (m == conv && t < best)) { conv = m; best = t; }
    }
    double lip = DBL_MAX * 2.0;
    for (int k = 0; k < 3; ++k)
        lip = fmin(lip, __dadd_ru(x.d[k], fmax(hb_len_ru(x.c[(k + 1) % 3], x.c[k]), hb_len_ru(x.c[(k + 2) % 3], x.c[k]))));
    const double ub = __dadd_ru(fmin(conv, lip), hb_eps(bits6));
    const bool split = ub > __dadd_rd(st->L, tol);
    atomicMax(split ? &st->ulive : &st->uret, d2bits(ub));
    x.inh = best;
    e[i] = x;
    flag[i] = split;
}

// the four children of every flagged entry (corner children first, then the middle one) and its three edge midpoints as
// the next level's queries, each seeded at the slot of an endpoint's nearest face
__device__ __forceinline__ D3 hb_mid(const D3 a, const D3 b) { return D3{(a.x + b.x) * 0.5, (a.y + b.y) * 0.5, (a.z + b.z) * 0.5}; }
__global__ void k_hb_split(const HbEntry *__restrict__ e, int n, const int *__restrict__ flag, const int *__restrict__ idx,
                           const int *__restrict__ slot, HbEntry *__restrict__ out, double *__restrict__ q, int *__restrict__ qs,
                           int *__restrict__ qa) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || !flag[i]) return;
    const HbEntry x = e[i];
    const int p = idx[i];
    const D3 m[3] = {hb_mid(x.c[0], x.c[1]), hb_mid(x.c[1], x.c[2]), hb_mid(x.c[2], x.c[0])};   // edge k: corner k -> k + 1
    for (int k = 0; k < 3; ++k) {
        const int j = 3 * p + k;
        q[3 * j] = m[k].x; q[3 * j + 1] = m[k].y; q[3 * j + 2] = m[k].z;
        qs[j] = slot[x.f[k]];
        qa[j] = x.aface;
    }
    for (int k = 0; k < 4; ++k) {
        HbEntry c;
        c.inh = x.inh; c.aface = x.aface;
        for (int r = 0; r < 3; ++r) {
            // corner r of child k < 3: corner k itself (r == k), else the midpoint of the edge between corner k and corner r;
            // child 3 has the three midpoints
            const int a = k, b = r;
            if (k < 3 && r == k) { c.c[r] = x.c[k]; c.d[r] = x.d[k]; c.f[r] = x.f[k]; c.q[r] = -1; continue; }
            const int edge = k == 3 ? r : ((b == (a + 1) % 3) ? a : b);        // edge a -> a + 1 or b -> b + 1 = a
            c.c[r] = m[edge]; c.d[r] = 0.0; c.f[r] = -1; c.q[r] = 3 * p + edge;
        }
        out[4 * p + k] = c;
    }
}

// ---- certified area-weighted mean and RMS distances (nw_mean_distance_bounds): the same entries, levels and walks ---------
// Every entry T (a subtriangle of level l of the face aface of A) has the weight |T0| 4^-l, |T0| its face's area; each level
// brackets the integrals of d_B and d_B^2 over every entry (k_mb_bound) and reduces them in a fixed order (k_mb_sum,
// k_mb_level).  DESIGN.md section 4 derives the bounds and the allowance.
#define NW_MB_BLOCKS 256
struct MbState {
    double area[3];                     // |A| (nearest), a lower and an upper bound of it
    double best[4];                     // the best bracket so far: [lo, hi] of the integral of d_B, then of d_B^2
    double ret[4];                      // the same totals over the retired entries
    double br[4];                       // the best bracket as [mean_lo, mean_hi, rms_lo, rms_hi] (mb_brackets)
    double rms_lo;                      // the best lower bound of the RMS so far (never decreases)
    int zero, converged;                // faces of A whose fp64 area is 0; both gaps <= tol
    unsigned long long cand;            // candidate faces evaluated by the support-plane stage
};

// |T0| of every finite face of A: {nearest, lower, upper}.  The cross product is formed at the corner whose two edges have
// the smallest product of lengths l l', and the rounding error of the area is below 2^-48 l l' (DESIGN.md section 4).
__global__ void k_mb_area(const int *__restrict__ faces, const float *__restrict__ pos, int F, double4 *__restrict__ area,
                          MbState *__restrict__ st) {
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= F) return;
    D3 c[3];
    bool live = true;
    for (int k = 0; k < 3; ++k) {
        const int v = faces[3 * f + k];
        c[k] = D3{(double)pos[3 * v], (double)pos[3 * v + 1], (double)pos[3 * v + 2]};
        live = live && fabs(c[k].x) <= DBL_MAX && fabs(c[k].y) <= DBL_MAX && fabs(c[k].z) <= DBL_MAX;
    }
    if (!live) { area[f] = make_double4(0.0, 0.0, 0.0, 0.0); return; }
    const double l[3] = {hb_len_ru(c[1], c[0]), hb_len_ru(c[2], c[1]), hb_len_ru(c[0], c[2])};   // edge k: corner k -> k + 1
    int k = 0;
    double ll = __dmul_ru(l[2], l[0]);
    for (int j = 1; j < 3; ++j) {
        const double t = __dmul_ru(l[j - 1], l[j]);
        if (t < ll) { ll = t; k = j; }
    }
    const D3 u = sub(c[(k + 1) % 3], c[k]), v = sub(c[(k + 2) % 3], c[k]);
    const D3 cr = D3{u.y * v.z - u.z * v.y, u.z * v.x - u.x * v.z, u.x * v.y - u.y * v.x};
    const double a = 0.5 * sqrt(dot(cr, cr)), err = __dmul_ru(ll, 0x1p-48);
    if (a == 0.0) atomicAdd(&st->zero, 1);
    area[f] = make_double4(a, fmax(__dsub_rd(a, err), 0.0), __dadd_ru(a, err), 0.0);
}

// sum of x and y rounded to nearest (0), down (1) or up (2)
__device__ __forceinline__ double mb_add(double x, double y, int mode) {
    return mode == 1 ? __dadd_rd(x, y) : mode == 2 ? __dadd_ru(x, y) : x + y;
}
__device__ __forceinline__ double4 mb_add4(double4 x, double4 y, int4 m) {
    return make_double4(mb_add(x.x, y.x, m.x), mb_add(x.y, y.y, m.y), mb_add(x.z, y.z, m.z), mb_add(x.w, y.w, m.w));
}
// Fixed-order column sums of v[0..n) (only the rows with flag[i] == 0 when flag is given), each column rounded by its mode:
// NW_MB_BLOCKS blocks of 256 threads, thread t of block b adds rows b 256 + t, + NW_MB_BLOCKS 256, ... in turn, then a tree
// in shared memory; part[b] is the block's sum.  k_mb_level (or k_mb_total) adds the blocks with the same tree.
__device__ __forceinline__ double4 mb_tree(double4 x, int4 m) {
    __shared__ double4 sh[256];
    sh[threadIdx.x] = x;
    __syncthreads();
    for (int o = 128; o; o >>= 1) {
        if (threadIdx.x < o) sh[threadIdx.x] = mb_add4(sh[threadIdx.x], sh[threadIdx.x + o], m);
        __syncthreads();
    }
    return sh[0];
}
__global__ void __launch_bounds__(256) k_mb_sum(const double4 *__restrict__ v, int n, const int *__restrict__ flag, int4 m,
                                                double4 *__restrict__ part) {
    double4 s = make_double4(0.0, 0.0, 0.0, 0.0);
    for (int64_t i = blockIdx.x * 256 + threadIdx.x; i < n; i += NW_MB_BLOCKS * 256)
        if (!flag || !flag[i]) s = mb_add4(s, v[i], m);
    s = mb_tree(s, m);
    if (threadIdx.x == 0) part[blockIdx.x] = s;
}
// |A| and its bounds from the per-face areas' block sums
__global__ void __launch_bounds__(256) k_mb_total(const double4 *__restrict__ part, MbState *__restrict__ st) {
    const double4 s = mb_tree(part[threadIdx.x], make_int4(0, 1, 2, 0));
    if (threadIdx.x == 0) { st->area[0] = s.x; st->area[1] = s.y; st->area[2] = s.z; }
}

// [mean_lo, mean_hi, rms_lo, rms_hi] from the integral brackets and the area bounds, rounded outward
__device__ __forceinline__ void mb_brackets(const double best[4], const double area[3], double out[4]) {
    out[0] = __ddiv_rd(best[0], area[2]); out[1] = __ddiv_ru(best[1], area[1]);
    out[2] = __dsqrt_rd(__ddiv_rd(best[2], area[2])); out[3] = __dsqrt_ru(__ddiv_ru(best[3], area[1]));
}
// One level's totals: the retired sums so far plus this level's entries give a valid bracket; the best bracket keeps the
// largest lower and the smallest upper totals.  Then the entries this level retires join the retired sums.
__global__ void __launch_bounds__(256) k_mb_level(const double4 *__restrict__ part, double tol, MbState *__restrict__ st) {
    const int4 m = make_int4(1, 2, 1, 2);
    const double4 all = mb_tree(part[threadIdx.x], m);
    __syncthreads();
    const double4 ret = mb_tree(part[NW_MB_BLOCKS + threadIdx.x], m);
    if (threadIdx.x) return;
    const double lv[4] = {__dadd_rd(st->ret[0], all.x), __dadd_ru(st->ret[1], all.y), __dadd_rd(st->ret[2], all.z),
                          __dadd_ru(st->ret[3], all.w)};
    st->best[0] = fmax(st->best[0], lv[0]); st->best[1] = fmin(st->best[1], lv[1]);
    st->best[2] = fmax(st->best[2], lv[2]); st->best[3] = fmin(st->best[3], lv[3]);
    st->ret[0] = __dadd_rd(st->ret[0], ret.x); st->ret[1] = __dadd_ru(st->ret[1], ret.y);
    st->ret[2] = __dadd_rd(st->ret[2], ret.z); st->ret[3] = __dadd_ru(st->ret[3], ret.w);
    double *b = st->br;
    mb_brackets(st->best, st->area, b);
    st->rms_lo = fmax(st->rms_lo, b[2]);
    st->converged = b[1] - b[0] <= tol && b[3] - b[2] <= tol;
}

// The support-plane lower bound (stage 3): every face g of B that is nearest somewhere on T lies within U of T (U the upper
// bound of d_B over T), so the faces whose boxes pass the test below are a complete candidate set, and on T
//   d_B(x) >= m(x) = min over them of sigma_g . (x - v) for the corner v of g that maximises sigma_g . v  (|sigma_g| <= 1),
// a concave piecewise linear function, at least its linear interpolant of m(c_k).  The node test is SelfWalk's (intersect.cu)
// with T's corners, widened by U; the leaf test compares float32 face boxes with T's fp64 box widened by U.
struct MbWalk {
    OctreeView oct;                     // over h->tboxes
    const int4 *__restrict__ sfaces;
    const float4 *__restrict__ posq;
    D3 c[3];                            // T's corners
    D3 g;                               // their mean
    float4 x[3];                        // the corners in float32, for the node test
    double lo[3], hi[3];                // T's box widened by U (rounded outward)
    float w;                            // the node test's widening: U and twice the slack of the call
    double eps;                         // the rounding allowance of the call
    double m[3] = {DBL_MAX * 2.0, DBL_MAX * 2.0, DBL_MAX * 2.0};
    double up1 = DBL_MAX * 2.0, up2 = DBL_MAX * 2.0;   // the convexity bounds of k_mb_bound over these faces (sums over the corners)
    unsigned long long cand = 0;

    __device__ __forceinline__ bool tick() const { return false; }
    __device__ __forceinline__ bool open(int node, int &link) const {
        const Box *bp = &oct.boxes[node];
        const float4 bd = __ldg(&bp->d);
        link = __float_as_int(bd.z);
        const float4 ba = __ldg(&bp->a), bb = __ldg(&bp->b), bc = __ldg(&bp->c);
        float l[3], h[3];
        project_frame(ba, bb, bc, x[0].x, x[0].y, x[0].z, l[0], l[1], l[2]);
        h[0] = l[0]; h[1] = l[1]; h[2] = l[2];
        for (int k = 1; k < 3; ++k) {
            float p[3];
            project_frame(ba, bb, bc, x[k].x, x[k].y, x[k].z, p[0], p[1], p[2]);
            for (int j = 0; j < 3; ++j) { l[j] = fminf(l[j], p[j]); h[j] = fmaxf(h[j], p[j]); }
        }
        return l[0] - w <= bd.x && h[0] + w >= bb.z && l[1] - w <= bd.y && h[1] + w >= bb.w && l[2] - w <= bc.w && h[2] + w >= bd.w;
    }
    __device__ __forceinline__ void leaf(int node) {
        NW_ASSERT(node >= oct.leaf0 && node < oct.n_nodes);
        const int2 k = __ldg(&oct.kids[node]);
        NW_ASSERT(k.x >= 0 && k.y >= 0 && k.x + k.y <= oct.n_slots);
#pragma unroll 1
        for (int s = k.x; s < k.x + k.y; ++s) {
            const int4 sf = __ldg(&sfaces[s]);
            const float4 y[3] = {__ldg(&posq[sf.x]), __ldg(&posq[sf.y]), __ldg(&posq[sf.z])};
            if (!(finite4(y[0]) && finite4(y[1]) && finite4(y[2]))) continue;
            if (fminf(y[0].x, fminf(y[1].x, y[2].x)) > hi[0] || fmaxf(y[0].x, fmaxf(y[1].x, y[2].x)) < lo[0] ||
                fminf(y[0].y, fminf(y[1].y, y[2].y)) > hi[1] || fmaxf(y[0].y, fmaxf(y[1].y, y[2].y)) < lo[1] ||
                fminf(y[0].z, fminf(y[1].z, y[2].z)) > hi[2] || fmaxf(y[0].z, fmaxf(y[1].z, y[2].z)) < lo[2])
                continue;
            ++cand;
            const D3 v[3] = {d3(y[0]), d3(y[1]), d3(y[2])};
            double s1 = 0.0, s2 = 0.0;
            for (int j = 0; j < 3; ++j) {
                const double du = __dadd_ru(sqrt(dist2(c[j], closest_on_triangle(c[j], v[0], v[1], v[2]))), eps);
                s1 = __dadd_ru(s1, du); s2 = __dadd_ru(s2, __dmul_ru(du, du));
            }
            up1 = fmin(up1, s1); up2 = fmin(up2, s2);
            // sigma: the unit direction from g's closest point to the centroid, shrunk so that |sigma| <= 1 survives rounding;
            // 0 for a face within eps of the centroid
            const D3 u = sub(g, closest_on_triangle(g, v[0], v[1], v[2]));
            const double len = sqrt(dot(u, u));
            if (!(len > eps)) { for (int j = 0; j < 3; ++j) m[j] = fmin(m[j], 0.0); continue; }
            const double sc = (1.0 - 0x1p-40) / len;
            const D3 sg = D3{u.x * sc, u.y * sc, u.z * sc};
            // m_k = min over the corners v of g of sigma . (c_k - v), rounded down
            for (int j = 0; j < 3; ++j)
                for (int r = 0; r < 3; ++r) {
                    const double tx = sg.x >= 0.0 ? __dmul_rd(sg.x, __dsub_rd(c[j].x, v[r].x)) : __dmul_rd(sg.x, __dsub_ru(c[j].x, v[r].x));
                    const double ty = sg.y >= 0.0 ? __dmul_rd(sg.y, __dsub_rd(c[j].y, v[r].y)) : __dmul_rd(sg.y, __dsub_ru(c[j].y, v[r].y));
                    const double tz = sg.z >= 0.0 ? __dmul_rd(sg.z, __dsub_rd(c[j].z, v[r].z)) : __dmul_rd(sg.z, __dsub_ru(c[j].z, v[r].z));
                    m[j] = fmin(m[j], __dadd_rd(__dadd_rd(tx, ty), tz));
                }
        }
    }
    __device__ __forceinline__ void walk() {
        const int2 k = __ldg(&oct.kids[0]);
        for (int c = k.x; c < k.x + k.y; ++c) nw_walk_subtree(*this, oct, c);
    }
};

// Bounds of the integrals of d_B and d_B^2 over each entry, weights in [w_lo, w_hi] = [lower, upper] bound of |T0| x 4^-l,
// every corner distance widened by eps (DESIGN.md section 4):
//   upper (convexity): d(., t) and d(., t)^2 are convex for one face t of B, so the integral is at most w_hi x the mean over
//     the corners; the candidates t are k_hb_bound's.  U, k_hb_bound's bound of max d_B over T, is kept for the lower bounds;
//   lower, cheap: d_B^2 - |x|^2 is concave, so the integral of d_B^2 is at least w_lo (mean d_k^2 - s/12), s the sum of the
//     squared edge lengths; d_B <= U on T, so the integral of d_B is at least that over U;
//   sharp (only for entries the first two leave unresolved): MbWalk's m_k give w_lo max(0, mean m_k) and, when every
//     m_k >= 0, w_lo (sum m_k^2 + sum_{i<j} m_i m_j) / 6; else (integral of d_B)^2 / w_hi.  The convexity bound is also
//     taken over every face MbWalk finds, which settles T when it lies on a face of B.
// An entry is retired (flag 0) when its gaps are at most tol w and w max(tol^2, 2 tol rms_lo), or when w_lo = 0.
__global__ void __launch_bounds__(128) k_mb_bound(HbEntry *__restrict__ e, int n, int level, const double *__restrict__ qd,
                                                  const int *__restrict__ qf, const int *__restrict__ faces, const float4 *__restrict__ posq,
                                                  int FB, const double4 *__restrict__ area, const __grid_constant__ OctreeView oct,
                                                  const int4 *__restrict__ sfaces, const unsigned *__restrict__ bits6, double tol,
                                                  MbState *__restrict__ st, double4 *__restrict__ val, int *__restrict__ flag) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i > n) return;
    if (i == n) { flag[n] = 0; return; }
    HbEntry x = e[i];
    const double4 a = x.q[0] == -2 ? make_double4(0.0, 0.0, 0.0, 0.0) : area[x.aface];
    if (!(a.z > 0.0)) { val[i] = make_double4(0.0, 0.0, 0.0, 0.0); flag[i] = 0; return; }
    for (int k = 0; k < 3; ++k)
        if (x.q[k] >= 0) { x.d[k] = qd[x.q[k]]; x.f[k] = qf[x.q[k]]; x.q[k] = -1; }
    const double eps = hb_eps(bits6), sc = ldexp(1.0, -2 * level);
    const double w = a.x * sc, wlo = __dmul_rd(a.y, sc), whi = __dmul_ru(a.z, sc);
    // upper bounds
    const int cand[4] = {x.f[0], x.f[1], x.f[2], x.inh};
    double conv = DBL_MAX * 2.0, up1 = DBL_MAX * 2.0, up2 = DBL_MAX * 2.0;
    int best = -1;
#pragma unroll 1
    for (int j = 0; j < 4; ++j) {
        const int t = cand[j];
        if (t < 0 || (j > 0 && t == cand[0]) || (j > 1 && t == cand[1]) || (j > 2 && t == cand[2])) continue;
        NW_ASSERT(t < FB);
        double mx = 0.0, s1 = 0.0, s2 = 0.0;
#pragma unroll 1
        for (int k = 0; k < 3; ++k) {
            const double d = x.f[k] == t ? x.d[k] : hb_face_dist(x.c[k], faces, posq, t), du = __dadd_ru(d, eps);
            mx = fmax(mx, d); s1 = __dadd_ru(s1, du); s2 = __dadd_ru(s2, __dmul_ru(du, du));
        }
        if (mx < conv || (mx == conv && t < best)) { conv = mx; best = t; }
        up1 = fmin(up1, s1); up2 = fmin(up2, s2);
    }
    double lip = DBL_MAX * 2.0, s = 0.0;
    for (int k = 0; k < 3; ++k) {
        const double l1 = hb_len_ru(x.c[(k + 1) % 3], x.c[k]), l2 = hb_len_ru(x.c[(k + 2) % 3], x.c[k]), le = __dadd_ru(l1, eps);
        lip = fmin(lip, __dadd_ru(x.d[k], fmax(l1, l2)));
        s = __dadd_ru(s, __dmul_ru(le, le));
    }
    const double U = __dadd_ru(fmin(conv, lip), eps);
    double hi1 = __dmul_ru(whi, __ddiv_ru(up1, 3.0)), hi2 = __dmul_ru(whi, __ddiv_ru(up2, 3.0));
    // cheap lower bounds
    double sq = 0.0;
    for (int k = 0; k < 3; ++k) { const double dl = fmax(__dsub_rd(x.d[k], eps), 0.0); sq = __dadd_rd(sq, __dmul_rd(dl, dl)); }
    double lo2 = __dmul_rd(wlo, fmax(__dsub_rd(__ddiv_rd(sq, 3.0), __ddiv_ru(s, 12.0)), 0.0));
    double lo1 = U > 0.0 ? __ddiv_rd(lo2, U) : 0.0;
    const double rl = st->rms_lo, g2 = fmax(tol * tol, 2.0 * tol * rl);
    bool done = hi1 - lo1 <= tol * w && hi2 - lo2 <= w * g2;
    unsigned long long cnt = 0;
    if (!done) {
        MbWalk mw;
        mw.oct = oct; mw.sfaces = sfaces; mw.posq = posq; mw.eps = eps;
        const double r = __dadd_ru(U, eps);
        for (int k = 0; k < 3; ++k) {
            mw.c[k] = x.c[k];
            mw.x[k] = make_float4((float)x.c[k].x, (float)x.c[k].y, (float)x.c[k].z, 0.f);
        }
        mw.g = D3{(x.c[0].x + x.c[1].x + x.c[2].x) / 3.0, (x.c[0].y + x.c[1].y + x.c[2].y) / 3.0, (x.c[0].z + x.c[1].z + x.c[2].z) / 3.0};
        mw.lo[0] = __dsub_rd(fmin(fmin(x.c[0].x, x.c[1].x), x.c[2].x), r); mw.hi[0] = __dadd_ru(fmax(fmax(x.c[0].x, x.c[1].x), x.c[2].x), r);
        mw.lo[1] = __dsub_rd(fmin(fmin(x.c[0].y, x.c[1].y), x.c[2].y), r); mw.hi[1] = __dadd_ru(fmax(fmax(x.c[0].y, x.c[1].y), x.c[2].y), r);
        mw.lo[2] = __dsub_rd(fmin(fmin(x.c[0].z, x.c[1].z), x.c[2].z), r); mw.hi[2] = __dadd_ru(fmax(fmax(x.c[0].z, x.c[1].z), x.c[2].z), r);
        mw.w = __fadd_ru(__double2float_ru(r), 2.0f * call_slack(bits6));
        mw.walk();
        cnt = mw.cand;
        hi1 = fmin(hi1, __dmul_ru(whi, __ddiv_ru(mw.up1, 3.0))); hi2 = fmin(hi2, __dmul_ru(whi, __ddiv_ru(mw.up2, 3.0)));
        if (mw.cand) {
            double mk[3], sm = 0.0;
            bool pos = true;
            for (int k = 0; k < 3; ++k) { mk[k] = __dsub_rd(mw.m[k], eps); sm = __dadd_rd(sm, mk[k]); pos = pos && mk[k] >= 0.0; }
            const double l1 = __dmul_rd(wlo, fmax(__ddiv_rd(sm, 3.0), 0.0));
            double l2 = whi > 0.0 ? __ddiv_rd(__dmul_rd(l1, l1), whi) : 0.0;
            if (pos) {
                const double q = __dadd_rd(__dadd_rd(__dadd_rd(__dmul_rd(mk[0], mk[0]), __dmul_rd(mk[1], mk[1])), __dmul_rd(mk[2], mk[2])),
                                           __dadd_rd(__dadd_rd(__dmul_rd(mk[0], mk[1]), __dmul_rd(mk[1], mk[2])), __dmul_rd(mk[2], mk[0])));
                l2 = fmax(l2, __dmul_rd(wlo, __ddiv_rd(q, 6.0)));
            }
            lo1 = fmax(lo1, l1); lo2 = fmax(lo2, l2);
        }
        lo2 = fmax(lo2, whi > 0.0 ? __ddiv_rd(__dmul_rd(lo1, lo1), whi) : 0.0);
        done = hi1 - lo1 <= tol * w && hi2 - lo2 <= w * g2;
    }
    if (cnt) atomicAdd(&st->cand, cnt);
    x.inh = best;
    e[i] = x;
    val[i] = make_double4(lo1, hi1, lo2, hi2);
    flag[i] = !(done || wlo == 0.0);
}

}  // namespace

// exclusive scan of h->hb_flag[0..n] (the last flag 0) into h->hb_idx: hb_idx[n] = the number of flags set
static int hb_scan(nw_ctx *h, int n) {
    cudaStream_t s = h->stream;
    size_t tmp = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tmp, h->hb_flag, h->hb_idx, n + 1, s);
    if (tmp > h->cub_tmp_bytes) { NW_CHECK(nw_alloc(h, (char **)&h->cub_tmp, tmp)); h->cub_tmp_bytes = tmp; }
    NW_CUDA(cub::DeviceScan::ExclusiveSum(h->cub_tmp, tmp, h->hb_flag, h->hb_idx, n + 1, s));
    h->launches += 1;
    return NW_OK;
}

// nq point queries h->hb_q against the handle's mesh (seeded from h->hb_qs unless it is level 0), then the running maximum
static int hb_walk(nw_ctx *h, int nq, bool seeded) {
    cudaStream_t s = h->stream;
    HbState *st = (HbState *)h->hb_st;
    NW_CHECK(nw_surface_walk_f64(h, h->hb_q, nq, seeded ? h->hb_qs : nullptr, h->hb_qd, h->hb_qf));
    k_hb_level_max<<<nw_grid(nq, 256), 256, 0, s>>>(h->hb_qd, nq, st);
    NW_LAUNCH_CHECK();
    k_hb_level_arg<<<nw_grid(nq, 256), 256, 0, s>>>(h->hb_qd, nq, st);
    NW_LAUNCH_CHECK();
    k_hb_take<<<1, 1, 0, s>>>(h->hb_q, h->hb_qf, h->hb_qa, st);
    NW_LAUNCH_CHECK();
    return NW_OK;
}

static int hb_queries(nw_ctx *h, size_t nq) {
    NW_CHECK(nw_alloc(h, &h->hb_q, 3 * nq)); NW_CHECK(nw_alloc(h, &h->hb_qd, nq)); NW_CHECK(nw_alloc(h, &h->hb_qf, nq));
    NW_CHECK(nw_alloc(h, &h->hb_qs, nq)); NW_CHECK(nw_alloc(h, &h->hb_qa, nq));
    return NW_OK;
}

// Shared by both calls: A on the device, its faces checked and its used vertices found; B's face row -> slot table; the
// level-0 walks of the used vertices (unseeded) after the slack of the call, and one entry per face.  Sets nu, the used
// vertices, and hs, the state after the checks.
static int hb_start(nw_ctx *h, const std::string &w, const float *pos, int M, const int32_t *faces, int F, double tol,
                    int64_t max_queries, HbState &hs, int &nu) {
    NW_CHECK(nw_mesh_check(h, w));
    NW_ARG(pos != nullptr && faces != nullptr && M > 0 && F > 0, w + ": the mesh passed in has no vertices or no faces");
    NW_ARG(F <= 0x7fffffff / 3 && M <= 0x7fffffff / 3, w + ": the mesh passed in is too large (3 M and 3 F must fit int32)");
    NW_ARG(tol >= 0.0 && tol <= DBL_MAX, w + ": tol must be finite and >= 0");
    NW_CUDA(cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    const int B = 256;

    NW_CHECK(nw_alloc(h, &h->hb_st, sizeof(HbState)));
    HbState *st = (HbState *)h->hb_st;
    memset(&hs, 0, sizeof(hs));
    hs.larg = 0x7fffffff; hs.L = -1.0;
    NW_CUDA(cudaMemcpyAsync(st, &hs, sizeof(hs), cudaMemcpyHostToDevice, s));
    NW_CHECK(nw_alloc(h, &h->hb_pos, (size_t)3 * M)); NW_CHECK(nw_alloc(h, &h->hb_faces, (size_t)3 * F));
    NW_CHECK(nw_h2d(h, h->hb_pos, pos, sizeof(float) * 3 * (size_t)M));
    NW_CHECK(nw_h2d(h, h->hb_faces, faces, sizeof(int32_t) * 3 * (size_t)F));
    NW_CHECK(nw_alloc(h, &h->hb_vface, (size_t)M));
    NW_CUDA(cudaMemsetAsync(h->hb_vface, 0x7f, sizeof(int) * (size_t)M, s));
    k_hb_faces<<<nw_grid(F, B), B, 0, s>>>(h->hb_faces, h->hb_pos, F, M, h->hb_vface, st);
    NW_LAUNCH_CHECK();
    NW_CHECK(nw_alloc(h, &h->hb_slot, (size_t)h->F));
    k_hb_mesh_b<<<nw_grid(h->F, B), B, 0, s>>>(h->sfaces, h->posq, h->F, h->hb_slot, st);
    NW_LAUNCH_CHECK();
    NW_CHECK(nw_alloc(h, &h->hb_flag, (size_t)std::max(M, F) + 1)); NW_CHECK(nw_alloc(h, &h->hb_idx, (size_t)std::max(M, F) + 1));
    k_hb_used<<<nw_grid(M + 1, B), B, 0, s>>>(h->hb_vface, M, F, h->hb_flag);
    NW_LAUNCH_CHECK();
    NW_CHECK(hb_scan(h, M));
    nu = 0;
    NW_CUDA(cudaMemcpyAsync(&hs, st, sizeof(hs), cudaMemcpyDeviceToHost, s));
    NW_CUDA(cudaMemcpyAsync(&nu, h->hb_idx + M, sizeof(int), cudaMemcpyDeviceToHost, s));
    NW_CUDA(cudaStreamSynchronize(s));
    NW_ARG(hs.bad == 0, w + ": a face index of the mesh passed in is outside [0, M)");
    NW_ARG(hs.nonfinite < F, w + ": the mesh passed in has no face with finite corners");
    NW_ARG(hs.b_finite != 0, w + ": the handle's mesh has no face with finite corners");
    NW_ARG(max_queries >= nu, w + ": max_queries must be at least the number of vertices the finite faces use (" + std::to_string(nu) + ")");

    NW_CHECK(hb_queries(h, (size_t)nu));
    k_hb_vertices<<<nw_grid(M, B), B, 0, s>>>(h->hb_pos, h->hb_vface, h->hb_flag, h->hb_idx, M, h->hb_q, h->hb_qa);
    NW_LAUNCH_CHECK();
    NW_CHECK(nw_surface_boxes(h, h->hb_q, h->hb_q + 1, h->hb_q + 2, nu, 3, true));
    NW_CHECK(nw_alloc(h, &h->hb_ent[0], sizeof(HbEntry) * (size_t)F));
    k_hb_level0<<<nw_grid(F, B), B, 0, s>>>(h->hb_faces, h->hb_pos, h->hb_idx, F, (HbEntry *)h->hb_ent[0]);
    NW_LAUNCH_CHECK();
    return hb_walk(h, nu, false);
}

// Shared by both calls: bound, retire, split, one level at a time, until bound(n, level, stop) sets stop, nothing survives
// (done), or the next level would take the point walks past max_queries.  bound() bounds the n entries of
// h->hb_ent[cur] and sets h->hb_flag[0..n] (1: split; hb_flag[n] = 0).
template <typename Bound>
static int hb_levels(nw_ctx *h, int F, int64_t nu, int64_t bounded0, int64_t max_queries, Bound bound, int &levels,
                     int64_t &walks, int64_t &bounded, bool &done) {
    cudaStream_t s = h->stream;
    int n = F, cur = 0;
    levels = 0; walks = nu; bounded = bounded0; done = false;
    while (true) {
        ++levels;
        NW_CHECK(nw_alloc(h, &h->hb_flag, (size_t)n + 1)); NW_CHECK(nw_alloc(h, &h->hb_idx, (size_t)n + 1));
        bool stop = false;
        NW_CHECK(bound(cur, n, levels - 1, stop));
        if (stop) { done = true; break; }
        NW_CHECK(hb_scan(h, n));
        int S = 0;
        NW_CUDA(cudaMemcpyAsync(&S, h->hb_idx + n, sizeof(int), cudaMemcpyDeviceToHost, s));
        NW_CUDA(cudaStreamSynchronize(s));
        if (S == 0) { done = true; break; }
        if (levels >= NW_HB_MAX_LEVELS || walks + 3 * (int64_t)S > max_queries || 4 * (int64_t)S > 0x7fffffff - 1) break;
        const int nxt = cur ^ 1;
        NW_CHECK(nw_alloc(h, &h->hb_ent[nxt], sizeof(HbEntry) * 4 * (size_t)S));
        NW_CHECK(hb_queries(h, 3 * (size_t)S));
        k_hb_split<<<nw_grid(n, 256), 256, 0, s>>>((const HbEntry *)h->hb_ent[cur], n, h->hb_flag, h->hb_idx, h->hb_slot,
                                                   (HbEntry *)h->hb_ent[nxt], h->hb_q, h->hb_qs, h->hb_qa);
        NW_LAUNCH_CHECK();
        NW_CHECK(hb_walk(h, 3 * S, true));
        walks += 3 * (int64_t)S;
        n = 4 * S;
        bounded += n;
        cur = nxt;
    }
    return NW_OK;
}

extern "C" int nw_hausdorff_bounds(nw_ctx *h, const float *pos, int M, const int32_t *faces, int F, double tol, int64_t max_queries,
                                   double bounds[2], double witness[3], int32_t witness_faces[2], int64_t stats[5]) {
    if (!h) return NW_ERR_ARG;
    HbState hs;
    int nu = 0;
    NW_CHECK(hb_start(h, "nw_hausdorff_bounds", pos, M, faces, F, tol, max_queries, hs, nu));
    cudaStream_t s = h->stream;
    HbState *st = (HbState *)h->hb_st;

    // bound, retire, split: the retired entries are those whose bound is within tol of the running maximum
    int levels = 0;
    int64_t walks = 0, bounded = 0;
    bool converged = false;
    NW_CHECK(hb_levels(h, F, nu, F - hs.nonfinite, max_queries, [&](int cur, int n, int, bool &) {
        k_hb_bound<<<nw_grid((int64_t)n + 1, 128), 128, 0, s>>>((HbEntry *)h->hb_ent[cur], n, h->hb_qd, h->hb_qf, h->faces, h->posq, h->F,
                                                              h->surf_bits, tol, st, h->hb_flag);
        NW_LAUNCH_CHECK();
        return NW_OK;
    }, levels, walks, bounded, converged));
    NW_CUDA(cudaMemcpyAsync(&hs, st, sizeof(hs), cudaMemcpyDeviceToHost, s));
    NW_CUDA(cudaStreamSynchronize(s));
    double uret, ulive;
    memcpy(&uret, &hs.uret, sizeof(double));
    memcpy(&ulive, &hs.ulive, sizeof(double));
    if (bounds) { bounds[0] = hs.L; bounds[1] = std::max(std::max(hs.L, uret), converged ? 0.0 : ulive); }
    if (witness) { witness[0] = hs.w[0]; witness[1] = hs.w[1]; witness[2] = hs.w[2]; }
    if (witness_faces) { witness_faces[0] = hs.wa; witness_faces[1] = hs.wb; }
    if (stats) { stats[0] = levels; stats[1] = bounded; stats[2] = walks; stats[3] = hs.nonfinite; stats[4] = converged; }
    return NW_OK;
}

extern "C" int nw_mean_distance_bounds(nw_ctx *h, const float *pos, int M, const int32_t *faces, int F, double tol, int64_t max_queries,
                                       double out[5], int64_t stats[7]) {
    if (!h) return NW_ERR_ARG;
    const std::string w("nw_mean_distance_bounds");
    HbState hs;
    int nu = 0;
    NW_CHECK(hb_start(h, w, pos, M, faces, F, tol, max_queries, hs, nu));
    cudaStream_t s = h->stream;

    // |T0| of every face and |A|
    NW_CHECK(nw_alloc(h, &h->mb_st, sizeof(MbState)));
    MbState *st = (MbState *)h->mb_st, ms;
    memset(&ms, 0, sizeof(ms));
    ms.best[1] = ms.best[3] = DBL_MAX * 2.0;
    NW_CUDA(cudaMemcpyAsync(st, &ms, sizeof(ms), cudaMemcpyHostToDevice, s));
    NW_CHECK(nw_alloc(h, &h->mb_area, (size_t)4 * F));
    NW_CHECK(nw_alloc(h, &h->mb_part, (size_t)8 * NW_MB_BLOCKS));
    double4 *area = (double4 *)h->mb_area, *part = (double4 *)h->mb_part;
    k_mb_area<<<nw_grid(F, 256), 256, 0, s>>>(h->hb_faces, h->hb_pos, F, area, st);
    NW_LAUNCH_CHECK();
    k_mb_sum<<<NW_MB_BLOCKS, 256, 0, s>>>(area, F, nullptr, make_int4(0, 1, 2, 0), part);
    NW_LAUNCH_CHECK();
    k_mb_total<<<1, 256, 0, s>>>(part, st);
    NW_LAUNCH_CHECK();
    NW_CUDA(cudaMemcpyAsync(&ms, st, sizeof(ms), cudaMemcpyDeviceToHost, s));
    NW_CUDA(cudaStreamSynchronize(s));
    NW_ARG(ms.area[0] > 0.0, w + ": the finite faces of the mesh passed in have zero total area");

    // bound each level; stop as soon as the best bracket is within tol, else retire and split
    const OctreeView oct = nw_octree_view(h, h->tboxes);
    int levels = 0;
    int64_t walks = 0, bounded = 0;
    bool done = false;                  // everything retired; converged is decided by the gaps alone
    NW_CHECK(hb_levels(h, F, nu, F - hs.nonfinite, max_queries, [&](int cur, int n, int level, bool &stop) {
        NW_CHECK(nw_alloc(h, &h->mb_val, (size_t)4 * n));
        double4 *val = (double4 *)h->mb_val;
        k_mb_bound<<<nw_grid((int64_t)n + 1, 128), 128, 0, s>>>((HbEntry *)h->hb_ent[cur], n, level, h->hb_qd, h->hb_qf, h->faces, h->posq,
                                                              h->F, area, oct, h->sfaces, h->surf_bits, tol, st, val, h->hb_flag);
        NW_LAUNCH_CHECK();
        const int4 m = make_int4(1, 2, 1, 2);
        k_mb_sum<<<NW_MB_BLOCKS, 256, 0, s>>>(val, n, nullptr, m, part);
        NW_LAUNCH_CHECK();
        k_mb_sum<<<NW_MB_BLOCKS, 256, 0, s>>>(val, n, h->hb_flag, m, part + NW_MB_BLOCKS);
        NW_LAUNCH_CHECK();
        k_mb_level<<<1, 256, 0, s>>>(part, tol, st);
        NW_LAUNCH_CHECK();
        int conv = 0;
        NW_CUDA(cudaMemcpyAsync(&conv, &st->converged, sizeof(int), cudaMemcpyDeviceToHost, s));
        NW_CUDA(cudaStreamSynchronize(s));
        stop = conv != 0;
        return NW_OK;
    }, levels, walks, bounded, done));
    NW_CUDA(cudaMemcpyAsync(&ms, st, sizeof(ms), cudaMemcpyDeviceToHost, s));
    NW_CUDA(cudaStreamSynchronize(s));
    if (out) { out[0] = ms.area[0]; for (int k = 0; k < 4; ++k) out[1 + k] = ms.br[k]; }
    if (stats) {
        stats[0] = levels; stats[1] = bounded; stats[2] = walks; stats[3] = (int64_t)ms.cand; stats[4] = hs.nonfinite; stats[5] = ms.zero;
        stats[6] = ms.converged;
    }
    return NW_OK;
}

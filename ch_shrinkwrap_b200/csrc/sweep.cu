// sweep.cu -- the per-point kernels of the hot loop.
//
//   k_sweep1 : exact nearest face centroid (fp64 compare, octree of Hilbert cells) -> inverse-distance
//              weights -> A f -> weighted, distance-de-weighted residual   (mesh_conj_grad.py:222-253, 433-516, 518-551)
//   k_adjoint: deterministic scatter of AH res and AH 1 (exact fixed-point sums; the per-face sums of a warp are formed
//              on the tensor cores); without the influence channel it is Ahfunc     (mesh_conj_grad.py:553-588)
//   k_sweep2 : A applied to all search directions at once + Gram sums Hc, Gc, c0 in fp64, without
//              materialising AS                                       (conj_grad.py:189-203)
//   k_apply_A: the single-operator form behind Afunc.
//
// Determinism: the adjoint accumulates in 64-bit fixed point (integer atomics are order-independent,
// float atomics are not); the Gram sums use a fixed thread->point assignment and a fixed two-stage tree.
#include <cub/cub.cuh>
#include <cfloat>
#include <cstring>
#include <type_traits>
#include "common.cuh"

namespace {

// ---- exact-arithmetic helpers (never contracted into FMAs) ---------------------------------------
__device__ __forceinline__ float sq_rd(float g) { return __fmul_rd(g, g); }

struct QueryF32 {
    float x, y, z;
    __device__ __forceinline__ float fx() const { return x; }
    __device__ __forceinline__ float fy() const { return y; }
    __device__ __forceinline__ float fz() const { return z; }
    __device__ __forceinline__ float lb_box(const float4 lo, const float4 hi) const {
        float gx = fmaxf(fmaxf(__fsub_rd(lo.x, x), __fsub_rd(x, hi.x)), 0.f);
        float gy = fmaxf(fmaxf(__fsub_rd(lo.y, y), __fsub_rd(y, hi.y)), 0.f);
        float gz = fmaxf(fmaxf(__fsub_rd(lo.z, z), __fsub_rd(z, hi.z)), 0.f);
        return __fadd_rd(__fadd_rd(sq_rd(gx), sq_rd(gy)), sq_rd(gz));
    }
    // scipy sqeuclidean_distance_double on float32->float64 promoted inputs: ((dx^2)+dy^2)+dz^2
    __device__ __forceinline__ double d2(const float4 c) const {
        double dx = (double)x - (double)c.x, dy = (double)y - (double)c.y, dz = (double)z - (double)c.z;
        return __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
    }
    // the same against a float64 target (points mode, nw_set_point_targets)
    __device__ __forceinline__ double d2(const double *c) const {
        double dx = (double)x - c[0], dy = (double)y - c[1], dz = (double)z - c[2];
        return __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
    }
};

struct QueryF64 {
    double x, y, z;
    float xl, xh, yl, yh, zl, zh;   // float32 enclosure of the float64 coordinates
    __device__ __forceinline__ float fx() const { return xl; }
    __device__ __forceinline__ float fy() const { return yl; }
    __device__ __forceinline__ float fz() const { return zl; }
    __device__ __forceinline__ void set(double px, double py, double pz) {
        x = px; y = py; z = pz;
        xl = __double2float_rd(px); xh = __double2float_ru(px);
        yl = __double2float_rd(py); yh = __double2float_ru(py);
        zl = __double2float_rd(pz); zh = __double2float_ru(pz);
    }
    __device__ __forceinline__ float lb_box(const float4 lo, const float4 hi) const {
        float gx = fmaxf(fmaxf(__fsub_rd(lo.x, xh), __fsub_rd(xl, hi.x)), 0.f);
        float gy = fmaxf(fmaxf(__fsub_rd(lo.y, yh), __fsub_rd(yl, hi.y)), 0.f);
        float gz = fmaxf(fmaxf(__fsub_rd(lo.z, zh), __fsub_rd(zl, hi.z)), 0.f);
        return __fadd_rd(__fadd_rd(sq_rd(gx), sq_rd(gy)), sq_rd(gz));
    }
    __device__ __forceinline__ double d2(const float4 c) const {
        double dx = x - (double)c.x, dy = y - (double)c.y, dz = z - (double)c.z;
        return __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
    }
    __device__ __forceinline__ double d2(const double *c) const {
        double dx = x - c[0], dy = y - c[1], dz = z - c[2];
        return __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
    }
};

// float32 box that certainly contains the float64 value a float32 was rounded from (one ulp either side)
__device__ __forceinline__ float4 ulp_below(const float4 c) { return make_float4(nextafterf(c.x, -FLT_MAX), nextafterf(c.y, -FLT_MAX), nextafterf(c.z, -FLT_MAX), c.w); }
__device__ __forceinline__ float4 ulp_above(const float4 c) { return make_float4(nextafterf(c.x, FLT_MAX), nextafterf(c.y, FLT_MAX), nextafterf(c.z, FLT_MAX), c.w); }


struct Nearest {
    double d2;
    float ub;      // d2 rounded up to float: prune bound for the float32 lower bounds
    int slot, face;
    // no candidate yet: +inf, so that the first offer wins
    static __device__ __forceinline__ Nearest none() {
        Nearest n;
        n.d2 = DBL_MAX * 2.0; n.ub = FLT_MAX * 2.0f; n.slot = -1; n.face = 0x7fffffff;
        return n;
    }
    __device__ __forceinline__ void offer(double v, int s, int f) {
        // strict minimum; exact fp64 ties -> lowest face index (contract of SURVEY 7.3)
        // ub carries the relative 1.1e-5 that the box tests owe to the float32 orthonormality of the node frames (it used to
        // be a multiply by 0.99999 in every node test); a larger bound only ever prunes less
        if (v < d2 || (v == d2 && f < face)) { d2 = v; slot = s; face = f; ub = __fmul_ru(__double2float_ru(v), 1.000011f); }
    }
};

// Conservative lower bound of the squared distance from the query to anything inside a node: the sum over the three
// box axes of (interval gap)^2.  Projections are float32, so every interval is widened by an absolute slack (>= 4x the worst-case rounding error of
// both the query's and the members' evaluation, DESIGN.md "exactness") and the squares by a relative 1e-5 (axes are
// orthonormal only to float32 accuracy).  A node is skipped only if this bound exceeds the best exact fp64 distance,
// so skipping can never change the answer.
// (The walk itself uses the two-stage form of this test, Traversal::open.  Each 128-bit load of a node quarter also
// costs two moves of the warp-uniform node address into the vector registers it is about to overwrite; an opaque per-thread
// copy of the address does not change that allocation at 32 registers, and 256-bit loads do not pay either: DESIGN.md.)
template <typename Q>
__device__ __forceinline__ float node_lb(const Q &q, const Box *__restrict__ bp) {
    const float4 a = __ldg(&bp->a), b = __ldg(&bp->b), c = __ldg(&bp->c), d = __ldg(&bp->d);
    const float x = q.fx(), y = q.fy(), z = q.fz();
    const float pn = fmaf(a.x, x, fmaf(a.z, y, b.x * z));
    const float p1 = fmaf(a.y, x, fmaf(a.w, y, b.y * z));
    const float p2 = fmaf(c.x, x, fmaf(c.y, y, c.z * z));      // t2 = n x t1
    // the stored intervals are already widened by the rounding slack (k_box_decode)
    const float g0 = fmaxf(fmaxf(b.z - pn, pn - d.x), 0.f);
    const float g1 = fmaxf(fmaxf(b.w - p1, p1 - d.y), 0.f);
    const float g2 = fmaxf(fmaxf(d.w - p2, p2 - c.w), 0.f);
    const float lb = __fadd_rd(__fadd_rd(__fmul_rd(g0, g0), __fmul_rd(g1, g1)), __fmul_rd(g2, g2));
    return __fmul_rd(lb, 0.99999f);
}

// Stackless search of the octree of occupied Hilbert cells (tree.cu, common.cuh: nw_walk_subtree).  All state is scalar
// and held BY VALUE so that it stays in registers (a per-thread stack array, or references to the caller's query, made the
// compiler spill the whole object to local memory and reload it inside every node test).
// The tree fields are those of an OctreeView over h->boxes (make_args copies them from nw_octree_view), interleaved with
// the centroid search's own: k_sweep1 reads this struct from its parameters, and holding an OctreeView instead reorders
// those loads and the kernel's register assignment.
struct TreeView {
    const float4 *__restrict__ cent;
    const double *__restrict__ cent64;  // NULL, or (points mode, float64 targets) the exact coordinates per slot: cent[] only prunes
    const Box *__restrict__ boxes;
    const int *__restrict__ parent;
    const int2 *__restrict__ kids;
    const int *__restrict__ leaf_of_slot;
    const unsigned *__restrict__ fcells;   // grid cell (x | y << 10 | z << 20) each sorted centroid was keyed into at upload
    float3 grid_lo;                        // the 1024^3 grid of those keys: g = (p - grid_lo) * grid_inv
    float grid_inv, grid_cellw;            // cells per nm, nm per cell (0 when the mesh has no extent)
    int leaf0, leaf_level;
    int n_nodes, n_slots;
};

//
// PACKET = true: the 32 queries of a warp (Hilbert-sorted neighbours, so their searches overlap almost completely) walk
// the tree TOGETHER: one shared cursor, a node is entered if ANY lane cannot prune it, every lane keeps its own best
// and prunes with its own bound.  Each lane still sees every node it could not prune itself, so the result per lane is
// exactly that of a private search; what changes is that the warp never diverges (node data are warp-uniform
// broadcast loads) and pays for the union of the lanes' node sets instead of 32 interleaved private walks.
// All 32 lanes must call the methods; lanes past the end of the array are constructed with active_ = false, which
// gives them a bound no node can satisfy (no branch on `active` inside the walk).
template <typename Q, bool PACKET = false, bool COUNT = true, bool T64 = false>
struct Traversal {
    Q q;
    Nearest best;
    bool active;
    int lead = 0;                  // packet mode: lane whose query steers the greedy descent of top_down()
    __device__ __forceinline__ bool any(bool p) const { if constexpr (PACKET) return __any_sync(0xffffffffu, p); else return p; }
    __device__ __forceinline__ bool all(bool p) const { if constexpr (PACKET) return __all_sync(0xffffffffu, p); else return p; }
    // packet mode: one lane's query as the packet's centre and the largest distance of any lane's query from it.  A box
    // at distance D from the centre is at least D - pk_r from every lane, so ONE evaluation settles a node for the
    // whole packet -- which lets the lanes test DIFFERENT nodes in the same step (all siblings of a level at once).
    float pk_r = 0.f;
    int pk_lane = 0;
    __device__ __forceinline__ QueryF32 packet_centre() const {
        QueryF32 c;
        c.x = __shfl_sync(0xffffffffu, q.fx(), pk_lane); c.y = __shfl_sync(0xffffffffu, q.fy(), pk_lane); c.z = __shfl_sync(0xffffffffu, q.fz(), pk_lane);
        return c;
    }
    TreeView tv;
    float eps;
    unsigned n_tests = 0, n_leaves = 0, n_exact = 0;
    unsigned budget = 0xffffffffu;   // seeds only: stop refining after this many node tests (the result is then approximate)
    // COUNT = false (the production sweep): no statistics, no budget -- three registers and three instructions per step
    __device__ __forceinline__ bool tick() { if constexpr (COUNT) return ++n_tests > budget; else return false; }
    // Cell clearance.  A level-k node holds exactly the centroids keyed into one aligned cube of 2^(10-k) grid cells.
    // Once everything under the level-k ancestor of the seed has been searched, and that cube is the one the query
    // lies in, every other centroid was keyed OUTSIDE the cube; it has since moved at most `escape` cells (L-infinity,
    // k_refit_centroids), so it is at least (distance from the query to the cube's walls - escape) away.  If that
    // exceeds the best distance the climb can stop: the levels above cannot hold anything closer.
    // (the query's grid coordinates are recomputed where needed: three registers less in the inner loop)
    float escape;                    // < 0: no early-out (no grid, or the query lies outside it)
    __device__ __forceinline__ float grid(float v, float lo) const { return (v - lo) * tv.grid_inv; }

    __device__ __forceinline__ Traversal(const Q &q_, const Nearest &b_, const TreeView &tv_, float eps_, float escape_, bool active_ = true)
        : q(q_), best(b_), active(active_), tv(tv_), eps(eps_), escape(escape_) {
        if (!active) best.ub = -1.f;                                           // every bound is >= 0
        const float gx = grid(q.fx(), tv.grid_lo.x), gy = grid(q.fy(), tv.grid_lo.y), gz = grid(q.fz(), tv.grid_lo.z);
        if (!(gx >= 0.f && gx < 1024.f && gy >= 0.f && gy < 1024.f && gz >= 0.f && gz < 1024.f && tv.grid_inv > 0.f && escape < 1024.f)) escape = -1.f;
    }
    __device__ __forceinline__ void set_packet_centre(int lane) {
        pk_lane = lane;
        const QueryF32 pk_c = packet_centre();
        const float dx = q.fx() - pk_c.x, dy = q.fy() - pk_c.y, dz = q.fz() - pk_c.z;
        // rounded up, plus the float32 rounding of a float64 query (eps is 8 ulp of the coordinates)
        float r = active ? __fadd_ru(__fsqrt_ru(__fadd_ru(__fadd_ru(__fmul_ru(dx, dx), __fmul_ru(dy, dy)), __fmul_ru(dz, dz))), eps) : 0.f;
        if (!(r >= 0.f)) r = __int_as_float(0x7f800000);                       // NaN query: the prefilter never prunes
        pk_r = __uint_as_float(__reduce_max_sync(0xffffffffu, __float_as_uint(r)));
    }
    // deepest level whose cube around `cell` also contains the query
    __device__ __forceinline__ int shared_levels(unsigned cell) const {
        if (escape < 0.f) return 0;
        const float gx = grid(q.fx(), tv.grid_lo.x), gy = grid(q.fy(), tv.grid_lo.y), gz = grid(q.fz(), tv.grid_lo.z);
        const unsigned d = cell ^ ((unsigned)gx | ((unsigned)gy << 10) | ((unsigned)gz << 20));
        const unsigned m = (d | (d >> 10) | (d >> 20)) & 1023u;       // highest differing bit over the three axes
        return m ? __clz(m) - 22 : 10;
    }
    // true if nothing outside the query's level-`level` cube can beat the current best
    __device__ __forceinline__ bool cube_clear(int level) const {
        const int s = 10 - level;
        const float w = (float)(1u << s);
        const float gx = grid(q.fx(), tv.grid_lo.x), gy = grid(q.fy(), tv.grid_lo.y), gz = grid(q.fz(), tv.grid_lo.z);
        const float fx = gx - (float)(((unsigned)gx >> s) << s), fy = gy - (float)(((unsigned)gy >> s) << s),
                    fz = gz - (float)(((unsigned)gz >> s) << s);
        const float cl = fminf(fminf(fminf(fx, w - fx), fminf(fy, w - fy)), fminf(fz, w - fz));
        // slack: rounding of g for the query and for the centroids (a few ulp of 1024 each), of the coordinates (eps)
        const float m = (cl - escape - 1e-3f) * tv.grid_cellw - 2.f * eps;
        return m > 0.f && __fmul_rd(__fmul_rd(m, m), 0.99999f) > best.ub;
    }

    __device__ __forceinline__ void leaf(int node) {
        NW_ASSERT(node >= tv.leaf0 && node < tv.n_nodes);
        const int2 k = __ldg(&tv.kids[node]);
        NW_ASSERT(k.x >= 0 && k.y >= 0 && k.x + k.y <= tv.n_slots);
        if constexpr (COUNT) ++n_leaves;
        for (int s = k.x; s < k.x + k.y; ++s) {
            const float4 c = __ldg(&tv.cent[s]);
            if constexpr (T64) {             // points mode with float64 targets: the float32 copy (widened by an ulp) only prunes
                if (q.lb_box(ulp_below(c), ulp_above(c)) <= best.ub) { if constexpr (COUNT) ++n_exact; best.offer(q.d2(tv.cent64 + 3 * (size_t)s), s, __float_as_int(c.w)); }
            } else if (q.lb_box(c, c) <= best.ub) { if constexpr (COUNT) ++n_exact; best.offer(q.d2(c), s, __float_as_int(c.w)); }
        }
    }
    // The node test of the walk (nw_walk_subtree; children in Hilbert order: with a seed the bound is already (nearly)
    // exact, so nearest-first ordering would buy nothing): node_lb() in two stages.  Normal axis + first tangent axis need
    // three of the node's four 16-byte quarters; if that partial sum (a lower bound of the full one: the third square only
    // adds) already rules the node out for every lane, the fourth quarter is never loaded and the third axis never
    // evaluated.  Otherwise the full bound is formed from the same partial sum: the same nodes are opened as with a
    // one-stage test.
    __device__ __forceinline__ bool open(int node, int &link) {
        const Box *__restrict__ bp = &tv.boxes[node];
        const float4 a = __ldg(&bp->a), b = __ldg(&bp->b), d = __ldg(&bp->d);
        const float x = q.fx(), y = q.fy(), z = q.fz();
        link = __float_as_int(d.z);
        // (pn, p1) = (n, t1) . q ; same operations and association as node_lb
        const float pn = fmaf(a.x, x, fmaf(a.z, y, b.x * z));
        const float p1 = fmaf(a.y, x, fmaf(a.w, y, b.y * z));
        const float g0 = fmaxf(fmaxf(b.z - pn, pn - d.x), 0.f), g1 = fmaxf(fmaxf(b.w - p1, p1 - d.y), 0.f);
        const float s01 = __fmaf_rd(g1, g1, __fmul_rd(g0, g0));            // <= g0^2 + g1^2
        if (!any(s01 <= best.ub)) return false;                     // (best.ub already holds the frames' 1e-5, Nearest::offer)
        const float4 c = __ldg(&bp->c);
        const float p2 = fmaf(c.x, x, fmaf(c.y, y, c.z * z));
        const float g2 = fmaxf(fmaxf(d.w - p2, p2 - c.w), 0.f);
        return any(__fmaf_rd(g2, g2, s01) <= best.ub);
    }
    // Packet prefilter for the climb: all (<= 8) siblings of a level are bounded in ONE step -- lane j evaluates sibling j
    // against the packet centre, which settles it for every lane (set_packet_centre).  Survivors are then searched with
    // every lane's own, tighter bound (nw_walk_subtree).  Measured at C3: using the same prefilter for the children inside
    // the subtree walk (survivor masks per level in registers) cut the steps from 82 to 65 per point but cost 16 registers
    // and ran 8 % slower; relying on the packet bound ALONE is hopeless (warps that straddle a jump of the Hilbert curve
    // have a large radius: 80-190 ms instead of 3).
    __device__ __forceinline__ float packet_reach() const {
        float ubm = active ? best.ub : 0.f;
        if (!(ubm >= 0.f)) ubm = __int_as_float(0x7f800000);
        return __fadd_ru(__fsqrt_ru(__uint_as_float(__reduce_max_sync(0xffffffffu, __float_as_uint(ubm)))), pk_r);
    }
    // mask of the nodes [c0, c0 + n) that the packet cannot prune; `skip` is left out
    __device__ __forceinline__ unsigned family_mask(int c0, int n, int skip) {
        const float reach = packet_reach();
        const QueryF32 pk_c = packet_centre();
        const int j = (int)(threadIdx.x & 31);
        bool hit = false;
        if (j < n && c0 + j != skip) hit = !(__fsqrt_rd(node_lb(pk_c, &tv.boxes[c0 + j])) > reach);
        if constexpr (COUNT) ++n_tests;
        return __ballot_sync(0xffffffffu, hit);
    }
    // climb from a leaf (one of whose centroids was keyed into `cell`): at every level only the sibling subtrees are searched
    __device__ __forceinline__ void from_leaf(int node, unsigned cell) {
        leaf(node);
        const int shared = shared_levels(cell);
        for (int level = tv.leaf_level; level >= 1; --level) {
            if (all(!active || (level <= shared && cube_clear(level)))) return;
            const int p = nw_link_node(__ldg(&tv.parent[node]));
            const int2 k = __ldg(&tv.kids[p]);
            if constexpr (PACKET) {
                unsigned todo = family_mask(k.x, k.y, node) & 0xffu;           // an octree node has <= 8 children
                while (todo) { const int j = __ffs(todo) - 1; todo &= todo - 1; nw_walk_subtree(*this, tv, k.x + j); }
            } else {
                for (int sib = k.x; sib < k.x + k.y; ++sib)
                    if (sib != node) nw_walk_subtree(*this, tv, sib);
            }
            node = p;
        }
    }
    // warm query: start at the seed's leaf
    __device__ __forceinline__ void from_seed(int seed_slot) { from_leaf(tv.leaf0 + __ldg(&tv.leaf_of_slot[seed_slot]), __ldg(&tv.fcells[seed_slot])); }
    // cold query: greedy descent (always into the child with the smallest bound) to get a first candidate, then the
    // exact search from the leaf it reached
    __device__ __forceinline__ int greedy_leaf() {
        int node = 0;
        while (node < tv.leaf0) {
            const int2 k = __ldg(&tv.kids[node]);
            float bl = FLT_MAX * 2.0f;
            for (int ch = k.x; ch < k.x + k.y; ++ch) {
                float l = node_score(&tv.boxes[ch], q.fx(), q.fy(), q.fz());
                if constexpr (PACKET) l = __shfl_sync(0xffffffffu, l, lead);
                if constexpr (COUNT) ++n_tests;
                if (l < bl) { bl = l; node = ch; }
            }
        }
        return node;
    }
    __device__ __forceinline__ void top_down() {
        const int node = greedy_leaf();
        from_leaf(node, __ldg(&tv.fcells[__ldg(&tv.kids[node]).x]));
    }
};

__device__ __forceinline__ double pow2d(int e) { return __longlong_as_double((long long)(1023 + e) << 52); }

__device__ __forceinline__ long long to_fixed(float v, double scale) { return __double2ll_rn((double)v * scale); }
__device__ __forceinline__ void red_fixed(unsigned long long *p, float v, double scale) {
    atomicAdd(p, (unsigned long long)to_fixed(v, scale));
}

// ---- deterministic adjoint scatter (a6): exact segmented sums of a warp on the tensor cores ------------------------
// Every term w_j*r_c is a float32 product converted to 64-bit fixed point (|term| < 2^39 by the shift rule, k_shift_final),
// so the result is an exact integer sum: independent of scheduling and of the number of GPUs.  The 32 points of a warp hit
// ~8-10 distinct faces; their per-face sums used to be taken with MATCH + 18 REDUX per distinct face (the ADU pipe was 87 %
// busy, ncu r02_ncu_full_c3_apply_AH_summary.csv).  Now a warp forms them as ONE small integer matrix product
//      C[group][byte column] = G[group][lane] * V[lane][byte column]        (IMMA.16832.U8.U8, s32 accumulators)
// G is the 0/1 membership matrix of the lanes' faces (built in registers from MATCH + a ballot), V holds each lane's twelve
// biased 40-bit terms as five bytes each plus a column of ones (the group sizes): a byte column sums to <= 32*255, the
// columns are recombined with shifts -- exact two's-complement arithmetic modulo 2^64 -- and one RED.64 per (face corner,
// component) leaves the warp.  V goes through shared memory once: every lane stores its 64-byte row, and
// ldmatrix.m16n16.trans.b8 (LDSM.8.MT1616, new on sm_100a) hands the bytes back transposed as the B fragments.
// Column order: the C fragment gives thread (g = lane/4, t = lane%4) the columns 8 nt + 2 t + {0, 1} of rows g and g + 8,
// so component t (x, y, z, influence) keeps its 16-byte stream [corner 0: b0..b4 | corner 1: b0..b4 | corner 2: b0..b4 | 1]
// in exactly those columns and every thread recombines whole values without a shuffle.
#define NW_ADJ_ROW 80      // bytes per lane row in shared memory: 64 used + 16 of padding (conflict-free 16-byte accesses)
struct AdjWarpSmem {
    unsigned char tile[32 * NW_ADJ_ROW];
    int4 sf[32];            // corner ids of the face of every group (written by the group's first lane)
    unsigned gid[8];        // group id of every lane, one byte each
};

__device__ __forceinline__ unsigned adj_eq4(unsigned x, unsigned r4) {     // bytes of x, r4 below 0x20: 0x01 where they are equal
    return (~((x ^ r4) + 0x7f7f7f7fu) >> 7) & 0x01010101u;
}
__device__ __forceinline__ void adj_imma(int (&c)[4], unsigned a0, unsigned a1, unsigned a2, unsigned a3, unsigned b0, unsigned b1) {
    asm volatile("mma.sync.aligned.m16n8k32.row.col.s32.u8.u8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+r"(c[0]), "+r"(c[1]), "+r"(c[2]), "+r"(c[3]) : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
// term -> biased 40-bit fixed point: rn(v * 2^shift) + 2^39, low word and high byte (v * 2^shift is exact in float32)
__device__ __forceinline__ void adj_fixed(float v, float scale, unsigned bias, unsigned &lo, unsigned &hi) {
    const long long f = __float2ll_rn(__fmul_rn(v, scale));
    lo = (unsigned)f;
    hi = (unsigned)(f >> 32) + bias;
}

// One point per lane: key (sorted face slot; any negative value for an inactive lane, whose weights and residual must be zero), the face's
// corner ids, the three weights and the residual.  INFL: component 3 accumulates the weights themselves (AH applied to ones).
template <bool INFL>
__device__ __forceinline__ void warp_adjoint_scatter(AdjWarpSmem &sm, bool active, int key, const int4 *__restrict__ sfaces,
                                                     const float (&uw)[3], float r_x, float r_y, float r_z, float scale,
                                                     float scale_i, unsigned long long *__restrict__ acc, int n_vertices, int n_faces) {
    NW_ASSERT(!active || (key >= 0 && key < n_faces));
    const int lane = threadIdx.x & 31;
    // ---- this lane's row of V ----
    unsigned S[4][4];                      // [component][word of its 16-byte stream]
    {
        // an inactive lane comes with zero weights and residual: without the bias and the one its whole row is zero
        const unsigned bias = active ? 0x80u : 0u, bias_one = active ? 0x180u : 0u;
        const float rr[3] = {r_x, r_y, r_z};
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            if (t == 3 && !INFL) { S[3][0] = S[3][1] = S[3][2] = S[3][3] = 0u; continue; }
            unsigned lo[3], hi[3];
#pragma unroll
            for (int q = 0; q < 3; ++q) {
                // (byte 1 of the last high word: the column of ones)
                if (t < 3) adj_fixed(__fmul_rn(uw[q], rr[t]), scale, q == 2 ? bias_one : bias, lo[q], hi[q]);
                else adj_fixed(uw[q], scale_i, q == 2 ? bias_one : bias, lo[q], hi[q]);
            }
            S[t][0] = lo[0];
            S[t][1] = __byte_perm(hi[0], lo[1], 0x6540);           // c0.b4 c1.b0 c1.b1 c1.b2
            S[t][2] = __byte_perm(__byte_perm(lo[1], hi[1], 0x0043), lo[2], 0x5410);   // c1.b3 c1.b4 c2.b0 c2.b1
            S[t][3] = __byte_perm(lo[2], hi[2], 0x5432);           // c2.b2 c2.b3 c2.b4 1
        }
    }
    {
        uint4 *row = reinterpret_cast<uint4 *>(sm.tile + lane * NW_ADJ_ROW);
#pragma unroll
        for (int j = 0; j < 4; ++j) {      // 16-byte chunk j = n-tiles 2j, 2j+1: {S0,S1 | S2,S3} halves of stream word j
            uint4 v;
            v.x = __byte_perm(S[0][j], S[1][j], 0x5410); v.y = __byte_perm(S[2][j], S[3][j], 0x5410);
            v.z = __byte_perm(S[0][j], S[1][j], 0x7632); v.w = __byte_perm(S[2][j], S[3][j], 0x7632);
            row[j] = v;
        }
    }
    // ---- groups: lanes with the same face ----
    const unsigned grp = __match_any_sync(0xffffffffu, key);
    const int leader = __ffs(grp) - 1;
    const unsigned leaders = __ballot_sync(0xffffffffu, lane == leader);
    const int gid = __popc(leaders & ((1u << leader) - 1u));
    const int ngroups = __popc(leaders);
    reinterpret_cast<unsigned char *>(sm.gid)[lane] = (unsigned char)gid;
    // the corner ids of a group's face: one gather per group, needed only by the epilogue -- its latency (the second of the
    // dependent chain slot -> face) hides behind the product
    int4 sf = make_int4(0, 0, 0, 0);
    NW_ASSERT(gid >= 0 && gid < 32 && ngroups >= 1 && ngroups <= 32);
    if (lane == leader && active) sf = __ldg(&sfaces[key]);
    __syncwarp();
    const int g = lane >> 2, t = lane & 3;
    const unsigned gw0 = sm.gid[t], gw1 = sm.gid[4 + t];         // group ids of lanes 4t..4t+3 and 16+4t..16+4t+3
    const unsigned addr = (unsigned)__cvta_generic_to_shared(sm.tile + lane * NW_ADJ_ROW);
    // B fragments of n-tiles 2j, 2j+1: rows 0-15 come from the addresses of lanes 0-15, rows 16-31 from lanes 16-31
    auto load_b = [&](int j, unsigned (&b)[2][2]) {
        asm volatile("ldmatrix.sync.aligned.m16n16.x2.trans.shared.b8 {%0,%1,%2,%3}, [%4];"
                     : "=r"(b[0][0]), "=r"(b[1][0]), "=r"(b[0][1]), "=r"(b[1][1]) : "r"(addr + 16 * j));
    };
    // stream byte k of a component sits in n-tile k / 2, accumulator register 2 half + k % 2
    auto emit = [&](int q, int half, int ng, const int4 &f, unsigned s0, unsigned s1, unsigned s2, unsigned s3, unsigned s4) {
        const int vid = q == 0 ? f.x : q == 1 ? f.y : f.z;
        NW_ASSERT(vid >= 0 && vid < n_vertices);
        const unsigned long long v = (unsigned long long)(s0 + (s1 << 8) + (s2 << 16)) + ((unsigned long long)s3 << 24) +
                                     ((unsigned long long)(s4 - ((unsigned)ng << 7)) << 32);      // minus ng * 2^39
        atomicAdd(acc + 4 * (size_t)vid + t, v);
    };
    for (int m0 = 0; m0 < ngroups; m0 += 16) {                    // warp-uniform; a second pass only with > 16 distinct faces
        const unsigned r0 = (unsigned)(m0 + g) * 0x01010101u, r1 = (unsigned)(m0 + g + 8) * 0x01010101u;
        const unsigned a0 = adj_eq4(gw0, r0), a1 = adj_eq4(gw0, r1), a2 = adj_eq4(gw1, r0), a3 = adj_eq4(gw1, r1);
        // two phases of four n-tiles each keep 16 accumulators live instead of 32: first the upper half of the streams
        // (corner 2 and the group sizes), then the lower half (corners 0 and 1; corner 1 ends in n-tile 4, kept)
        int c4[4], ng[2];
        {
            unsigned b23[2][2], b67[2][2];
            load_b(2, b23); load_b(3, b67);
            int c5[4] = {0, 0, 0, 0}, c6[4] = {0, 0, 0, 0}, c7[4] = {0, 0, 0, 0};
            c4[0] = c4[1] = c4[2] = c4[3] = 0;
            adj_imma(c7, a0, a1, a2, a3, b67[1][0], b67[1][1]);
            adj_imma(c6, a0, a1, a2, a3, b67[0][0], b67[0][1]);
            adj_imma(c5, a0, a1, a2, a3, b23[1][0], b23[1][1]);
            adj_imma(c4, a0, a1, a2, a3, b23[0][0], b23[0][1]);
            ng[0] = c7[1]; ng[1] = c7[3];                         // stream byte 15: the group size (0: no such group)
            if (m0 == 0) {                                        // the corner ids are needed only from here on
                if (lane == leader) sm.sf[gid] = sf;
                __syncwarp();
            }
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                if (ng[half] == 0 || (t == 3 && !INFL)) continue;
                const int4 f = sm.sf[m0 + g + 8 * half];
                emit(2, half, ng[half], f, c5[2 * half], c5[2 * half + 1], c6[2 * half], c6[2 * half + 1], c7[2 * half]);   // bytes 10..14
            }
        }
        {
            unsigned b01[2][2], b23[2][2];
            load_b(0, b01); load_b(1, b23);
            int c0[4] = {0, 0, 0, 0}, c1[4] = {0, 0, 0, 0}, c2[4] = {0, 0, 0, 0}, c3[4] = {0, 0, 0, 0};
            adj_imma(c0, a0, a1, a2, a3, b01[0][0], b01[0][1]);
            adj_imma(c1, a0, a1, a2, a3, b01[1][0], b01[1][1]);
            adj_imma(c2, a0, a1, a2, a3, b23[0][0], b23[0][1]);
            adj_imma(c3, a0, a1, a2, a3, b23[1][0], b23[1][1]);
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                if (ng[half] == 0 || (t == 3 && !INFL)) continue;
                const int4 f = sm.sf[m0 + g + 8 * half];
                emit(0, half, ng[half], f, c0[2 * half], c0[2 * half + 1], c1[2 * half], c1[2 * half + 1], c2[2 * half]);   // bytes 0..4
                emit(1, half, ng[half], f, c2[2 * half + 1], c3[2 * half], c3[2 * half + 1], c4[2 * half], c4[2 * half + 1]);   // bytes 5..9
            }
        }
    }
}


struct Sweep1Args {
    int64_t P;
    const float *px, *py, *pz;
    const double *px64, *py64, *pz64;
    const float *sx, *sy, *sz;     // sigma_inv arrays or NULL
    const float *wx, *wy, *wz;     // weight arrays (may alias sigma_inv) or NULL
    float sinv_scalar, wmean;
    int *slot;
    float *w0, *w1, *w2, *rx, *ry, *rz;
    const int *order;              // block schedule (see build_block_order) or NULL
    const float4 *posq;
    const int4 *sfaces;
    TreeView tv;
    int F;
    unsigned long long *acc;
    SolverState *st;
};

template <bool F64, bool STATS, bool T64>
__device__ __noinline__ Nearest find_nearest(const Sweep1Args &a, int64_t i, bool active, float x, float y, float z,
                                             double xd, double yd, double zd, Nearest best, int block_seed = -1) {
    const float eps = (fabsf(x) + fabsf(y) + fabsf(z) + a.st->coord_l1) * 9.5367431640625e-7f;   // 2^-20 * L1 magnitude
    typename std::conditional<F64, QueryF64, QueryF32>::type q;
    if constexpr (F64) q.set(xd, yd, zd);
    else { q.x = x; q.y = y; q.z = z; }
    Traversal<decltype(q), true, STATS, T64> tr(q, best, a.tv, eps, a.st->cell_escape, active);
    int seed = active ? a.slot[i] : -1;
    const unsigned alive = __ballot_sync(0xffffffffu, active);
    if (alive) {                                             // warp-uniform
        // The packet climbs from ONE leaf.  Lanes with a seed of their own first take its exact distance as their
        // bound; lanes without (first iteration after an upload: k_seed_leaders / k_seed_from_feet may have covered
        // only some) borrow the packet's.  If no lane has one, the first lane's query picks a leaf by greedy descent.
        const unsigned warm = __ballot_sync(0xffffffffu, active && seed >= 0);
        int start;
        if (warm) start = __shfl_sync(0xffffffffu, seed, __ffs(warm) - 1);
        else if (block_seed >= 0) start = block_seed;        // cold start: the block's first point carries the root search's result
        else {
            tr.lead = __ffs(alive) - 1;
            start = __ldg(&a.tv.kids[tr.greedy_leaf()]).x;
        }
        if (active && tr.best.slot < 0) {
            if (seed < 0) seed = start;
            const float4 c = __ldg(&a.tv.cent[seed]);
            tr.best.offer(T64 ? tr.q.d2(a.tv.cent64 + 3 * (size_t)seed) : tr.q.d2(c), seed, __float_as_int(c.w));
        }
        tr.set_packet_centre(__ffs(alive) - 1);
        tr.from_seed(start);
    }
    // traversal statistics (one atomic per warp and counter)
    if constexpr (STATS) {
    const unsigned t = __reduce_add_sync(0xffffffffu, active ? tr.n_tests : 0u), l = __reduce_add_sync(0xffffffffu, active ? tr.n_leaves : 0u),
                   e = __reduce_add_sync(0xffffffffu, tr.n_exact), m = __reduce_max_sync(0xffffffffu, tr.n_tests);
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(&a.st->trav[0], (unsigned long long)t); atomicAdd(&a.st->trav[1], (unsigned long long)l);
        atomicAdd(&a.st->trav[2], (unsigned long long)e); atomicMax(&a.st->trav[3], (unsigned long long)m);
    }
    }
    return tr.best;
}

// Cold-start pre-pass: the first point of every 32 (= lane 0 of each warp of k_sweep1) gets an APPROXIMATE nearest
// face from a root search that stops refining after a fixed number of node tests (a seed only has to be close, the
// exact search happens in k_sweep1; bounding the effort removes the long tail of near-equidistant queries).
template <bool F64>
__global__ void __launch_bounds__(128) k_seed_leaders(const __grid_constant__ Sweep1Args a, int stride, unsigned budget) {
    // ONE search per warp, on lane 0: 32 private walks in one warp diverge at every node, and a diverged warp pays the L2
    // latency of every lane's node in turn (measured at C3: 2.5 ms for 78 k searches, one warp's serial chain); with one
    // search per warp the latency is hidden by the other 63 warps of the SM
    if (threadIdx.x & 31) return;
    const int64_t t = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t i = t * stride;
    if (i >= a.P || a.slot[i] >= 0) return;
    Nearest best = Nearest::none();
    const float x = a.px[i], y = a.py[i], z = a.pz[i];
    const float eps = (fabsf(x) + fabsf(y) + fabsf(z) + a.st->coord_l1) * 9.5367431640625e-7f;
    typename std::conditional<F64, QueryF64, QueryF32>::type q;
    if constexpr (F64) q.set(a.px64[i], a.py64[i], a.pz64[i]);
    else { q.x = x; q.y = y; q.z = z; }
    Traversal<decltype(q)> tr(q, best, a.tv, eps, a.st->cell_escape);
    tr.budget = budget;
    tr.top_down();
    a.slot[i] = tr.best.slot;     // >= 0: the first descent always reaches a leaf before the budget can run out
}

// Foot points A f of the previous block (the point on the OLD surface each localisation was attached to).  After a
// remesh the new surface is close to the old one, and a query that lies ON the surface is cheap (its search ball is
// tiny), so the face nearest to the old foot point is an excellent, individually computed seed for the real query.
__global__ void __launch_bounds__(256) k_save_feet(int64_t P, const int *__restrict__ slot, const int4 *__restrict__ sfaces,
                                                   const float4 *__restrict__ posq, const float *__restrict__ w0,
                                                   const float *__restrict__ w1, const float *__restrict__ w2,
                                                   float *__restrict__ fx, float *__restrict__ fy, float *__restrict__ fz) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= P) return;
    const int sl = slot[i];
    if (sl < 0) { fx[i] = fy[i] = fz[i] = __int_as_float(0x7fc00000); return; }
    const int4 sf = sfaces[sl];
    const float4 a = posq[sf.x], b = posq[sf.y], c = posq[sf.z];
    const float u0 = w0[i], u1 = w1[i], u2 = w2[i];
    fx[i] = a.x * u0 + b.x * u1 + c.x * u2; fy[i] = a.y * u0 + b.y * u1 + c.y * u2; fz[i] = a.z * u0 + b.z * u1 + c.z * u2;
}

__device__ __forceinline__ unsigned spread10s(unsigned v) {
    v &= 0x3ffu;
    v = (v | v << 16) & 0x30000ffu;
    v = (v | v << 8) & 0x300f00fu;
    v = (v | v << 4) & 0x30c30c3u;
    v = (v | v << 2) & 0x9249249u;
    return v;
}

// The faces are sorted by the Hilbert key of their centroid, so the face nearest to a point ON the surface is found
// (approximately) by a binary search of the point's own key -- no box tests at all; a short bounded local search from
// there polishes the seed.
__global__ void __launch_bounds__(128) k_seed_from_feet(const __grid_constant__ Sweep1Args a, const float *__restrict__ fx,
                                                        const float *__restrict__ fy, const float *__restrict__ fz,
                                                        const unsigned *__restrict__ fkeys, const int *__restrict__ fkey_tab,
                                                        float3 klo, float kinv, unsigned budget) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= a.P || a.slot[i] >= 0) return;
    const float x = fx[i], y = fy[i], z = fz[i];
    if (!(x == x && y == y && z == z)) return;          // no foot point: k_sweep1 borrows a neighbour's seed
    unsigned qx = (unsigned)fminf(fmaxf((x - klo.x) * kinv, 0.f), 1023.f);
    unsigned qy = (unsigned)fminf(fmaxf((y - klo.y) * kinv, 0.f), 1023.f);
    unsigned qz = (unsigned)fminf(fmaxf((z - klo.z) * kinv, 0.f), 1023.f);
    hilbert_axes_to_transpose(qx, qy, qz, 10);
    const unsigned key = (spread10s(qx) << 2) | (spread10s(qy) << 1) | spread10s(qz);
    int lo = __ldg(&fkey_tab[key >> 15]), hi = __ldg(&fkey_tab[(key >> 15) + 1]);   // lower_bound, bracketed by the prefix table (tree.cu: k_key_table)
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(&fkeys[mid]) < key) lo = mid + 1; else hi = mid;
    }
    Nearest best = Nearest::none();
    const float eps = (fabsf(x) + fabsf(y) + fabsf(z) + a.st->coord_l1) * 9.5367431640625e-7f;
    QueryF32 q;
    q.x = x; q.y = y; q.z = z;
    Traversal<QueryF32> tr(q, best, a.tv, eps, a.st->cell_escape);
    const int s1 = min(lo, a.F - 1), s0 = max(s1 - 1, 0);
    { const float4 c = a.tv.cent[s0]; tr.best.offer(q.d2(c), s0, __float_as_int(c.w)); }
    { const float4 c = a.tv.cent[s1]; tr.best.offer(q.d2(c), s1, __float_as_int(c.w)); }
    tr.budget = budget;
    tr.from_seed(tr.best.slot);
    a.slot[i] = tr.best.slot;
}

// MODE 0: nearest face + weights only (what calc_w triggers);  MODE 1: + residual + adjoint scatter
// 16 blocks of 128 per SM: 32 registers, 64 warps per SM (12 blocks with float64 points).  Measured at C3 (warm sweep, ms): 56 regs
// 3.23, 48 regs 3.08, 40 regs 3.00 before the global-id tables; after them 48 regs 2.47, 40 regs 2.51, 32 regs 2.33 -- the packet
// walk is a dependent chain, occupancy hides it
template <bool F64, int MODE, bool STATS, bool T64 = false>
__global__ void __launch_bounds__(128, F64 ? 12 : 16) k_sweep1(const __grid_constant__ Sweep1Args a) {
    if (MODE == 1 && a.st->stop) return;

    // schedule entry: block of points | quarter << 28.  quarter 0: all 32 lanes of every warp are points; 1..4: only lanes
    // [8 (quarter - 1), 8 quarter) are, the other 24 idle (k_cold_order); negative: nothing to do
    const int entry = a.order ? __ldg(&a.order[blockIdx.x]) : (int)blockIdx.x;
    if (entry < 0) return;
    const int quarter = entry >> 28;
    const int64_t i = (entry & 0x0fffffff) * (int64_t)blockDim.x + threadIdx.x;
    const bool active = i < a.P && (quarter == 0 || (int)((threadIdx.x >> 3) & 3u) == quarter - 1);
    float x = 0.f, y = 0.f, z = 0.f;
    double xd = 0.0, yd = 0.0, zd = 0.0;
    if (active) {
        x = a.px[i]; y = a.py[i]; z = a.pz[i];
        xd = x; yd = y; zd = z;
        if (F64) { xd = a.px64[i]; yd = a.py64[i]; zd = a.pz64[i]; }
    }
    Nearest best = Nearest::none();
    // cold start: only the first point of every block of 128 was searched from the root (k_seed_leaders); the warps that
    // do not hold it climb from its face too (it may already have been replaced by that point's final answer: just as good)
    const int64_t i0 = (entry & 0x0fffffff) * (int64_t)blockDim.x;
    const int block_seed = i0 < a.P ? a.slot[i0] : -1;
    best = find_nearest<F64, STATS, T64>(a, i, active, x, y, z, xd, yd, zd, best, block_seed);
    if (active && best.slot < 0) {      // non-finite query: nothing compares; flag it (the reference asserts on NaN) and stay in bounds
        a.st->nan_flag = 1;
        best.slot = 0;
    }
    float u0 = 0.f, u1 = 0.f, u2 = 0.f, r_x = 0.f, r_y = 0.f, r_z = 0.f;
    int4 sf = make_int4(0, 0, 0, 0);
    if (active) {
    a.slot[i] = best.slot;
    sf = a.sfaces[best.slot];
    const float4 v0 = __ldg(&a.posq[sf.x]), v1 = __ldg(&a.posq[sf.y]), v2 = __ldg(&a.posq[sf.z]);
    // corner distances, mesh_conj_grad.py:491-495 (float32 points: all float32; float64 points: float64 then stored float32)
    float d0, d1, d2;
    if (F64) {
        double ax = (double)v0.x - xd, ay = (double)v0.y - yd, az = (double)v0.z - zd;
        d0 = (float)sqrt(__dadd_rn(__dadd_rn(__dmul_rn(ax, ax), __dmul_rn(ay, ay)), __dmul_rn(az, az)));
        ax = (double)v1.x - xd; ay = (double)v1.y - yd; az = (double)v1.z - zd;
        d1 = (float)sqrt(__dadd_rn(__dadd_rn(__dmul_rn(ax, ax), __dmul_rn(ay, ay)), __dmul_rn(az, az)));
        ax = (double)v2.x - xd; ay = (double)v2.y - yd; az = (double)v2.z - zd;
        d2 = (float)sqrt(__dadd_rn(__dadd_rn(__dmul_rn(ax, ax), __dmul_rn(ay, ay)), __dmul_rn(az, az)));
    } else {
        float ax = __fsub_rn(v0.x, x), ay = __fsub_rn(v0.y, y), az = __fsub_rn(v0.z, z);
        d0 = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(ax, ax), __fmul_rn(ay, ay)), __fmul_rn(az, az)));
        ax = __fsub_rn(v1.x, x); ay = __fsub_rn(v1.y, y); az = __fsub_rn(v1.z, z);
        d1 = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(ax, ax), __fmul_rn(ay, ay)), __fmul_rn(az, az)));
        ax = __fsub_rn(v2.x, x); ay = __fsub_rn(v2.y, y); az = __fsub_rn(v2.z, z);
        d2 = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(ax, ax), __fmul_rn(ay, ay)), __fmul_rn(az, az)));
    }
    // w = 1/max(d,1e-6); w /= w.sum(1)      (:503,510)
    u0 = __fdiv_rn(1.0f, fmaxf(d0, 1e-6f)); u1 = __fdiv_rn(1.0f, fmaxf(d1, 1e-6f)); u2 = __fdiv_rn(1.0f, fmaxf(d2, 1e-6f));
    const float us = __fadd_rn(__fadd_rn(u0, u1), u2);
    u0 = __fdiv_rn(u0, us); u1 = __fdiv_rn(u1, us); u2 = __fdiv_rn(u2, us);
    a.w0[i] = u0; a.w1[i] = u1; a.w2[i] = u2;
    if (MODE == 1) {
    // A f  (:544-545)
    const float afx = __fadd_rn(__fadd_rn(__fmul_rn(v0.x, u0), __fmul_rn(v1.x, u1)), __fmul_rn(v2.x, u2));
    const float afy = __fadd_rn(__fadd_rn(__fmul_rn(v0.y, u0), __fmul_rn(v1.y, u1)), __fmul_rn(v2.y, u2));
    const float afz = __fadd_rn(__fadd_rn(__fmul_rn(v0.z, u0), __fmul_rn(v1.z, u1)), __fmul_rn(v2.z, u2));
    // res = Wn (p - A f) / (D sigma_inv / 2 + 1)      (:222,231,248)
    float s_x = a.sinv_scalar, s_y = a.sinv_scalar, s_z = a.sinv_scalar;
    if (a.sx) { s_x = a.sx[i]; s_y = a.sy[i]; s_z = a.sz[i]; }
    float wnx, wny, wnz;
    if (a.wx) {
        wnx = __fdiv_rn(a.wx == a.sx ? s_x : a.wx[i], a.wmean);
        wny = __fdiv_rn(a.wy == a.sy ? s_y : a.wy[i], a.wmean);
        wnz = __fdiv_rn(a.wz == a.sz ? s_z : a.wz[i], a.wmean);
    } else wnx = wny = wnz = a.sinv_scalar;
    const double D = sqrt(best.d2);
    if (F64) {
        r_x = (float)((double)wnx * (xd - (double)afx)); r_y = (float)((double)wny * (yd - (double)afy)); r_z = (float)((double)wnz * (zd - (double)afz));
    } else {
        r_x = __fmul_rn(wnx, __fsub_rn(x, afx)); r_y = __fmul_rn(wny, __fsub_rn(y, afy)); r_z = __fmul_rn(wnz, __fsub_rn(z, afz));
    }
    r_x = (float)((double)r_x * (1.0 / (D * (double)s_x / 2.0 + 1.0)));
    r_y = (float)((double)r_y * (1.0 / (D * (double)s_y / 2.0 + 1.0)));
    r_z = (float)((double)r_z * (1.0 / (D * (double)s_z / 2.0 + 1.0)));
    a.rx[i] = r_x; a.ry[i] = r_y; a.rz[i] = r_z;
    if (!(fabsf(r_x) <= FLT_MAX && fabsf(r_y) <= FLT_MAX && fabsf(r_z) <= FLT_MAX)) a.st->nan_flag = 1;
    }
    }
}

// ---- single-operator forms ------------------------------------------------------------------------
// y_p = sum_j w_pj x[v_pj]   (Afunc, mesh_conj_grad.py:539-545); x packed float4 per vertex
__global__ void __launch_bounds__(256) k_apply_A(int64_t P, const int *__restrict__ slot, const int4 *__restrict__ sfaces,
                                                 const float *__restrict__ w0, const float *__restrict__ w1, const float *__restrict__ w2,
                                                 const float4 *__restrict__ xq, float *__restrict__ yx, float *__restrict__ yy, float *__restrict__ yz) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= P) return;
    const int4 sf = __ldg(&sfaces[slot[i]]);
    const float u0 = w0[i], u1 = w1[i], u2 = w2[i];
    const float4 a = __ldg(&xq[sf.x]), b = __ldg(&xq[sf.y]), c = __ldg(&xq[sf.z]);
    yx[i] = __fadd_rn(__fadd_rn(__fmul_rn(a.x, u0), __fmul_rn(b.x, u1)), __fmul_rn(c.x, u2));
    yy[i] = __fadd_rn(__fadd_rn(__fmul_rn(a.y, u0), __fmul_rn(b.y, u1)), __fmul_rn(c.y, u2));
    yz[i] = __fadd_rn(__fadd_rn(__fmul_rn(a.z, u0), __fmul_rn(b.z, u1)), __fmul_rn(c.z, u2));
}

// out_v += sum w_pj r_p  (Ahfunc, conj_grad_utils.c:123-167) into the fixed-point accumulators; INFL: channel 3 += sum w_pj
// (AH applied to ones) in the same pass -- the form the CG iteration runs right after k_sweep1.  st != NULL: the shifts are
// the device-side ones of this iteration (k_shift_final) and a raised stop flag makes the kernel a no-op.
#define NW_ADJ_TILES 2      // points per thread: the loads of all of them are in flight before the first one is processed
template <bool INFL>
__global__ void __launch_bounds__(256, 4) k_adjoint(int64_t P, const int *__restrict__ slot, const int4 *__restrict__ sfaces,
                                                 const float *__restrict__ w0, const float *__restrict__ w1, const float *__restrict__ w2,
                                                 const float *__restrict__ rx, const float *__restrict__ ry, const float *__restrict__ rz,
                                                 unsigned long long *__restrict__ acc, const SolverState *__restrict__ st, int shift, int shift_i,
                                                 int n_vertices, int n_faces) {
    __shared__ __align__(16) AdjWarpSmem sm[8];
    int sl[NW_ADJ_TILES];
    float uw[NW_ADJ_TILES][3], r[NW_ADJ_TILES][3];
    bool active[NW_ADJ_TILES];
#pragma unroll
    for (int k = 0; k < NW_ADJ_TILES; ++k) {
        const int64_t i = ((int64_t)blockIdx.x * NW_ADJ_TILES + k) * blockDim.x + threadIdx.x;
        active[k] = i < P;
        sl[k] = -1;
        uw[k][0] = uw[k][1] = uw[k][2] = r[k][0] = r[k][1] = r[k][2] = 0.f;
        if (active[k]) {
            uw[k][0] = w0[i]; uw[k][1] = w1[i]; uw[k][2] = w2[i];
            r[k][0] = rx[i]; r[k][1] = ry[i]; r[k][2] = rz[i];
            sl[k] = slot[i];
        }
    }
    if (st) {                          // all three loads in flight together with the points', then the branch
        const int stop = st->stop, s0 = st->acc_shift, s1 = st->infl_shift;
        if (stop) return;
        shift = s0; shift_i = s1;
    }
    const float scale = (float)pow2d(shift), scale_i = (float)pow2d(shift_i);
#pragma unroll
    for (int k = 0; k < NW_ADJ_TILES; ++k) {
        if (k) __syncwarp();           // the warp's shared-memory tile is reused
        warp_adjoint_scatter<INFL>(sm[threadIdx.x >> 5], active[k], sl[k], sfaces, uw[k], r[k][0], r[k][1], r[k][2], scale, scale_i, acc, n_vertices, n_faces);
    }
}

// influence_v += sum w_pj  (AH applied to ones, channel 3 of the accumulators)
__global__ void __launch_bounds__(256) k_apply_infl(int64_t P, const int *__restrict__ slot, const int4 *__restrict__ sfaces,
                                                    const float *__restrict__ w0, const float *__restrict__ w1, const float *__restrict__ w2,
                                                    unsigned long long *__restrict__ acc, const SolverState *__restrict__ st) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= P) return;
    const int4 sf = __ldg(&sfaces[slot[i]]);
    const double sci = pow2d(st->infl_shift);
    red_fixed(acc + 4 * (size_t)sf.x + 3, w0[i], sci);
    red_fixed(acc + 4 * (size_t)sf.y + 3, w1[i], sci);
    red_fixed(acc + 4 * (size_t)sf.z + 3, w2[i], sci);
}

// ---- Gram pass -------------------------------------------------------------------------------------
#define NW_NSUM 11   // hc00 hc01 hc11 hc02 hc12 hc22 gc0 gc1 gc2 c0 res2

__global__ void __launch_bounds__(256, 1) k_sweep2(int64_t P, const int *__restrict__ slot, const int4 *__restrict__ sfaces,
                                                const float *__restrict__ w0, const float *__restrict__ w1, const float *__restrict__ w2,
                                                const float *__restrict__ rx, const float *__restrict__ ry, const float *__restrict__ rz,
                                                const float4 *__restrict__ Sq,
                                                const uint8_t *__restrict__ pmask, const SolverState *__restrict__ st,
                                                double *__restrict__ partials) {
    if (st->stop) return;
    const bool three = st->n_search == 3;
    double acc[NW_NSUM];
#pragma unroll
    for (int k = 0; k < NW_NSUM; ++k) acc[k] = 0.0;
    const int64_t base = (int64_t)blockIdx.x * (blockDim.x * NW_S2_PTS) + threadIdx.x;
    int sl[NW_S2_PTS];
    float u[NW_S2_PTS][3], r[NW_S2_PTS][3];
    unsigned m[NW_S2_PTS];
    int4 sf[NW_S2_PTS];
#pragma unroll
    for (int j = 0; j < NW_S2_PTS; ++j) {
        const int64_t i = base + (int64_t)j * blockDim.x;
        const bool ok = i < P;
        sl[j] = ok ? slot[i] : -1;
        u[j][0] = ok ? w0[i] : 0.f; u[j][1] = ok ? w1[i] : 0.f; u[j][2] = ok ? w2[i] : 0.f;
        r[j][0] = ok ? rx[i] : 0.f; r[j][1] = ok ? ry[i] : 0.f; r[j][2] = ok ? rz[i] : 0.f;
        m[j] = ok ? (pmask ? pmask[i] : 7u) : 0u;
    }
#pragma unroll
    for (int j = 0; j < NW_S2_PTS; ++j) sf[j] = sl[j] >= 0 ? __ldg(&sfaces[sl[j]]) : make_int4(0, 0, 0, 0);
#pragma unroll
    for (int j = 0; j < NW_S2_PTS; ++j) {
        if (sl[j] < 0) continue;
        const float4 *pa = Sq + 3 * (size_t)sf[j].x, *pb = Sq + 3 * (size_t)sf[j].y, *pc = Sq + 3 * (size_t)sf[j].z;
        float as[3][3];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            if (k == 2 && !three) { as[2][0] = as[2][1] = as[2][2] = 0.f; break; }
            const float4 a = __ldg(pa + k), b = __ldg(pb + k), c = __ldg(pc + k);
            as[k][0] = __fadd_rn(__fadd_rn(__fmul_rn(a.x, u[j][0]), __fmul_rn(b.x, u[j][1])), __fmul_rn(c.x, u[j][2]));
            as[k][1] = __fadd_rn(__fadd_rn(__fmul_rn(a.y, u[j][0]), __fmul_rn(b.y, u[j][1])), __fmul_rn(c.y, u[j][2]));
            as[k][2] = __fadd_rn(__fadd_rn(__fmul_rn(a.z, u[j][0]), __fmul_rn(b.z, u[j][1])), __fmul_rn(c.z, u[j][2]));
        }
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const double rr = (double)r[j][c];
            acc[10] += rr * rr;
            if (m[j] & (1u << c)) {     // res[mask], AS[mask]  (mesh_conj_grad.py:274, conj_grad.py:198)
                const double a0 = as[0][c], a1 = as[1][c], a2 = as[2][c];
                acc[0] += a0 * a0; acc[1] += a0 * a1; acc[2] += a1 * a1;
                acc[3] += a0 * a2; acc[4] += a1 * a2; acc[5] += a2 * a2;
                acc[6] += a0 * rr; acc[7] += a1 * rr; acc[8] += a2 * rr;
                acc[9] += rr * rr;
            }
        }
    }
    __shared__ double sh[8][NW_NSUM];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < NW_NSUM; ++k) {
        double v = acc[k];
        for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0) sh[wid][k] = v;
    }
    __syncthreads();
    if (threadIdx.x < NW_NSUM) {
        double v = 0.0;
        for (int k = 0; k < 8; ++k) v += sh[k][threadIdx.x];
        partials[(size_t)blockIdx.x * NW_NSUM + threadIdx.x] = v;
    }
}

// fold the per-CTA partials in a fixed order into the solver state: one CTA per quantity, thread t sums partials t, t+256, ...
// of it, then a fixed shared-memory tree -- deterministic for a given P.  (One CTA looping over the quantities took 52 us at
// C3: eleven dependent rounds of strided loads and barriers.)
__global__ void __launch_bounds__(256) k_fold_partials(const double *__restrict__ partials, int n_blocks, SolverState *st) {
    if (st->stop) return;
    __shared__ double sh[256];
    const int k = blockIdx.x;
    double v = 0.0;
    for (int b = threadIdx.x; b < n_blocks; b += 256) v += partials[(size_t)b * NW_NSUM + k];
    sh[threadIdx.x] = v;
    __syncthreads();
    for (int o = 128; o; o >>= 1) {
        if (threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const double t = sh[0];
        if (k < 6) st->hc[k] = t;
        else if (k < 9) st->gc[k - 6] = t;
        else if (k == 9) st->c0 = t;
        else st->res2 = t;
    }
}

// ---- host<->device order conversion -------------------------------------------------------------
__global__ void k_gather_sorted3(const float *__restrict__ src, const int *__restrict__ perm, int64_t P,
                                 float *__restrict__ ox, float *__restrict__ oy, float *__restrict__ oz) {
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= P) return;
    int64_t s = perm[i];
    ox[i] = src[3 * s]; oy[i] = src[3 * s + 1]; oz[i] = src[3 * s + 2];
}
__global__ void k_scatter_caller3(const float *__restrict__ ix, const float *__restrict__ iy, const float *__restrict__ iz,
                                  const int *__restrict__ perm, int64_t P, float *__restrict__ dst) {
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= P) return;
    int64_t s = perm[i];
    dst[3 * s] = ix[i]; dst[3 * s + 1] = iy[i]; dst[3 * s + 2] = iz[i];
}
__global__ void k_scatter_vidx(const int *__restrict__ slot, const int4 *__restrict__ sfaces, const int *__restrict__ perm,
                               int64_t P, int *__restrict__ v_idx, int *__restrict__ face) {
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= P) return;
    int64_t s = perm[i];
    int4 sf = sfaces[slot[i]];
    if (v_idx) { v_idx[3 * s] = sf.x; v_idx[3 * s + 1] = sf.y; v_idx[3 * s + 2] = sf.z; }
    if (face) face[s] = sf.w;
}
template <bool F64>
__global__ void k_scatter_dist(const int *__restrict__ slot, const float4 *__restrict__ cent, const double *__restrict__ cent64,
                               const int *__restrict__ perm, int64_t P,
                               const float *__restrict__ px, const float *__restrict__ py, const float *__restrict__ pz,
                               const double *__restrict__ px64, const double *__restrict__ py64, const double *__restrict__ pz64,
                               double *__restrict__ dist) {
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= P) return;
    const int s = slot[i];
    const float4 c = cent[s];
    double d2;
    if (F64) { QueryF64 q; q.set(px64[i], py64[i], pz64[i]); d2 = cent64 ? q.d2(cent64 + 3 * (size_t)s) : q.d2(c); }
    else { QueryF32 q{px[i], py[i], pz[i]}; d2 = cent64 ? q.d2(cent64 + 3 * (size_t)s) : q.d2(c); }
    dist[perm[i]] = sqrt(d2);
}
__global__ void k_pack3(const float *__restrict__ src, int M, float4 *__restrict__ dst) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < M) dst[i] = make_float4(src[3 * i], src[3 * i + 1], src[3 * i + 2], 0.f);
}
// fixed point -> float32 (one rounding), optionally clearing the accumulator
__global__ void k_acc_to_float3(unsigned long long *__restrict__ acc, int M, int shift, float *__restrict__ out, int clear) {
    int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= M) return;
    const float inv = (float)pow2d(-shift);
    for (int c = 0; c < 3; ++c) {
        out[3 * v + c] = __ll2float_rn((long long)acc[4 * (size_t)v + c]) * inv;
        if (clear) acc[4 * (size_t)v + c] = 0ull;
    }
}

}  // namespace

// ---- launchers ------------------------------------------------------------------------------------
static Sweep1Args make_args(nw_ctx *h) {
    Sweep1Args a;
    a.P = h->P;
    a.px = h->px; a.py = h->py; a.pz = h->pz;
    a.px64 = h->px64; a.py64 = h->py64; a.pz64 = h->pz64;
    a.sx = h->sx; a.sy = h->sy; a.sz = h->sz;
    if (h->weights_mode == 2) { a.wx = h->wx; a.wy = h->wy; a.wz = h->wz; }
    else if (h->weights_mode == 1) { a.wx = h->sx; a.wy = h->sy; a.wz = h->sz; }
    else { a.wx = a.wy = a.wz = nullptr; }
    a.sinv_scalar = h->sinv_scalar; a.wmean = h->wmean;
    a.slot = h->slot;
    a.w0 = h->w0; a.w1 = h->w1; a.w2 = h->w2; a.rx = h->rx; a.ry = h->ry; a.rz = h->rz;
    a.posq = h->posq; a.sfaces = h->sfaces; a.F = h->F;
    const OctreeView o = nw_octree_view(h, h->boxes);
    a.tv.cent = h->cent; a.tv.cent64 = h->points_mode ? h->cent64 : nullptr; a.tv.boxes = o.boxes; a.tv.parent = o.parent; a.tv.kids = o.kids;
    a.tv.leaf_of_slot = o.leaf_of_slot; a.tv.leaf0 = o.leaf0; a.tv.leaf_level = o.leaf_level; a.tv.n_nodes = o.n_nodes; a.tv.n_slots = o.n_slots;
    a.tv.fcells = h->fcells; a.tv.grid_lo = make_float3(h->key_lo[0], h->key_lo[1], h->key_lo[2]); a.tv.grid_inv = h->key_inv;
    a.tv.grid_cellw = h->key_inv > 0.f ? 1.f / h->key_inv : 0.f;
    a.acc = h->acc; a.st = h->st;
    a.order = nullptr;
    return a;
}

int nw_save_feet(nw_ctx *h) {
    // called by nw_set_topology BEFORE the old mesh is overwritten
    if (h->P == 0 || !h->weights_valid || !h->sfaces || !h->posq || !h->slot) { h->feet_valid = false; return NW_OK; }
    NW_CHECK(nw_alloc(h, &h->fx, (size_t)h->P)); NW_CHECK(nw_alloc(h, &h->fy, (size_t)h->P)); NW_CHECK(nw_alloc(h, &h->fz, (size_t)h->P));
    k_save_feet<<<nw_grid(h->P, 256), 256, 0, h->stream>>>(h->P, h->slot, h->sfaces, h->posq, h->w0, h->w1, h->w2, h->fx, h->fy, h->fz);
    NW_LAUNCH_CHECK();
    h->feet_valid = true;
    return NW_OK;
}

int nw_launch_seed_leaders(nw_ctx *h) {
    if (h->P == 0 || !h->seeds_cold) return NW_OK;
    const int B = 128;
    Sweep1Args a = make_args(h);
    if (h->feet_valid) {
        // foot points of the previous block exist: on-surface queries, individually good seeds (measured: the cold
        // iteration costs 8.3 ms instead of 27 ms at C3).  On the very first block the localisations themselves are
        // too far from the surface for this lookup to pay off (measured slower than the 1-in-32 root search below).
        k_seed_from_feet<<<nw_grid(h->P, B), B, 0, h->stream>>>(a, h->fx, h->fy, h->fz, h->fkeys, h->fkey_tab,
                                                                make_float3(h->key_lo[0], h->key_lo[1], h->key_lo[2]), h->key_inv,
                                                                0u);   // measured (again with the packet search, also with feet 30 nm off the new surface): polishing the looked-up seed (budgets 12..48) does not make k_sweep1 any faster
        NW_LAUNCH_CHECK();
        h->seeds_cold = false;
        return NW_OK;
    }
    // (measured at C3 and rejected: root searches for one point in 1024 only, then the exact packet search for every 32nd
    // point seeded by them -- the sweep gains 0.8 ms from exact seeds, but packets of points that lie 32 apart cost 6 ms)
    // one bounded root search per block of k_sweep1 (128 points, Hilbert neighbours): measured at C3, seeds + first sweep in
    // ms -- every 32nd point, budget 512: 3.4 + 5.6; 256: 2.5 + 5.7; 128: 1.8 + 6.3; 64: 0.9 + 42 (seeds too poor)
    const unsigned budget = 256;
    const int stride = 128;
    const int GL = nw_grid(((h->P + stride - 1) / stride) * 32, B);
    if (h->px64) k_seed_leaders<true><<<GL, B, 0, h->stream>>>(a, stride, budget);
    else k_seed_leaders<false><<<GL, B, 0, h->stream>>>(a, stride, budget);
    NW_LAUNCH_CHECK();
    h->seeds_cold = false;
    h->leaders_fresh = true;
    return NW_OK;
}

// Longest-first block schedule.  A query deep inside a lobe is (nearly) equidistant to a whole region of the surface and
// its packet needs 10^4 steps where the average one needs 10^2; such packets are neighbours in the sorted order, so in
// index order they all start in the middle of the launch and the last of them finishes long after every other SM has
// gone idle (measured in the first iteration of a fit at C3: SMs active 47 % of the launch).  The distance from a query to
// its seed is known before the sweep and is a good proxy for that cost: blocks are launched in descending order of it.
// Rebuilt whenever the seeds are (new points or new topology); the order never affects results.
__global__ void __launch_bounds__(128) k_block_cost(int64_t P, const float *__restrict__ px, const float *__restrict__ py,
                                                    const float *__restrict__ pz, const int *__restrict__ slot,
                                                    const float4 *__restrict__ cent, unsigned *__restrict__ key, int *__restrict__ idx) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    float d2 = 0.f;
    if (i < P) {
        const int s = slot[i];
        if (s >= 0) {
            const float4 c = __ldg(&cent[s]);
            const float dx = px[i] - c.x, dy = py[i] - c.y, dz = pz[i] - c.z;
            d2 = dx * dx + dy * dy + dz * dz;
            if (!(d2 >= 0.f)) d2 = 0.f;
        }
    }
    __shared__ unsigned sh[4];
    const unsigned m = __reduce_max_sync(0xffffffffu, __float_as_uint(d2));       // non-negative floats order like their bits
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) { key[blockIdx.x] = max(max(sh[0], sh[1]), max(sh[2], sh[3])); idx[blockIdx.x] = blockIdx.x; }
}

// Schedule of the FIRST sweep of a fit.  There the seeds are borrowed (one root search per 32 points), and a packet of
// background localisations deep inside the object -- 32 queries, each nearly equidistant to a large piece of the surface
// in a different direction -- walks the union of 32 huge candidate sets: measured at C3, one such packet ran 16 k steps
// (16.7 M cycles) while the average SM was busy for 9.9 M.  The costliest blocks are therefore split FOUR ways: each of the
// four entries runs the same 128 points with only 8 of every 32 lanes active, so a packet covers 8 queries, its walk
// shrinks accordingly and four times as many warps share the work.  Every point is still searched exactly once, by the
// same exact search.  Layout: 4 entries for each of the first `n_far` blocks of the longest-first order, then the rest.
__global__ void k_cold_order(const int *__restrict__ order, int G, int n_far, int *__restrict__ out) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= G) return;
    const int b = order[k];
    if (k < n_far) { for (int q = 0; q < 4; ++q) out[4 * k + q] = b | ((q + 1) << 28); }
    else out[4 * n_far + (k - n_far)] = b;
}

static int build_block_order(nw_ctx *h, int G) {
    NW_CHECK(nw_alloc(h, &h->blk_key, (size_t)G)); NW_CHECK(nw_alloc(h, &h->blk_key2, (size_t)G));
    NW_CHECK(nw_alloc(h, &h->blk_idx, (size_t)G)); NW_CHECK(nw_alloc(h, &h->blk_order, (size_t)G));
    k_block_cost<<<G, 128, 0, h->stream>>>(h->P, h->px, h->py, h->pz, h->slot, h->cent, h->blk_key, h->blk_idx);
    NW_LAUNCH_CHECK();
    size_t tmp = 0;
    cub::DeviceRadixSort::SortPairsDescending(nullptr, tmp, h->blk_key, h->blk_key2, h->blk_idx, h->blk_order, G, 0, 32, h->stream);
    if (tmp > h->cub_tmp_bytes) { NW_CHECK(nw_alloc(h, (char **)&h->cub_tmp, tmp)); h->cub_tmp_bytes = tmp; }
    NW_CUDA(cub::DeviceRadixSort::SortPairsDescending(h->cub_tmp, tmp, h->blk_key, h->blk_key2, h->blk_idx, h->blk_order, G, 0, 32, h->stream));
    h->launches += 2;
    h->order_stale = false;
    h->cold_grid = 0;
    if (h->leaders_fresh && G >= 64 && G < (1 << 26)) {
        // how many: measured at C3 (78 k blocks), first sweep in ms for the costliest 1/4 .. 1/1024 of the blocks split --
        // 11.6, 8.8, 7.1, 6.5, 6.0, 5.8, 5.7, 5.6, 5.5 (9.5 unsplit): the pathological packets are a handful, and every
        // other block that is split pays for 24 idle lanes per warp
        const int n_far = std::min(G, std::max(32, G / 512));
        NW_CHECK(nw_alloc(h, &h->blk_order_cold, (size_t)G + 3 * (size_t)n_far));
        k_cold_order<<<nw_grid(G, 256), 256, 0, h->stream>>>(h->blk_order, G, n_far, h->blk_order_cold);
        NW_LAUNCH_CHECK();
        h->cold_grid = G + 3 * n_far;
    }
    return NW_OK;
}

int nw_launch_sweep1(nw_ctx *h, bool scatter) {
    if (h->P == 0) return NW_OK;
    const int B = 128;
    const int G = nw_grid(h->P, B);
    NW_CHECK(nw_launch_seed_leaders(h));
    if (h->order_stale) NW_CHECK(build_block_order(h, G));
    Sweep1Args a = make_args(h);
    a.order = h->blk_order;
    int G1 = G;
    if (h->leaders_fresh && h->cold_grid > 0) { a.order = h->blk_order_cold; G1 = h->cold_grid; }
    h->leaders_fresh = false;                       // only the very first sweep after the root searches is scheduled this way
    // traversal statistics (nw_get_traversal_stats) are collected only when asked for: nw_set_profile(h, 3)
    const bool stats = (h->profile & 2) != 0;
    if (a.tv.cent64) {
        // points mode with float64 targets (nw_set_point_targets): only the nearest-target query exists, no statistics
        NW_ARG(!scatter, "sweep1: float64 point targets support nearest-point queries only");
        if (h->px64) k_sweep1<true, 0, false, true><<<G1, B, 0, h->stream>>>(a); else k_sweep1<false, 0, false, true><<<G1, B, 0, h->stream>>>(a);
    } else if (h->px64) {
        if (stats) { if (scatter) k_sweep1<true, 1, true><<<G1, B, 0, h->stream>>>(a); else k_sweep1<true, 0, true><<<G1, B, 0, h->stream>>>(a); }
        else { if (scatter) k_sweep1<true, 1, false><<<G1, B, 0, h->stream>>>(a); else k_sweep1<true, 0, false><<<G1, B, 0, h->stream>>>(a); }
    } else {
        if (stats) { if (scatter) k_sweep1<false, 1, true><<<G1, B, 0, h->stream>>>(a); else k_sweep1<false, 0, true><<<G1, B, 0, h->stream>>>(a); }
        else { if (scatter) k_sweep1<false, 1, false><<<G1, B, 0, h->stream>>>(a); else k_sweep1<false, 0, false><<<G1, B, 0, h->stream>>>(a); }
    }
    NW_LAUNCH_CHECK();
    return NW_OK;
}

// AH res and AH 1 of the iteration: the scatter that follows k_sweep1 (stage "adjoint")
int nw_launch_adjoint(nw_ctx *h) {
    if (h->P == 0) return NW_OK;
    k_adjoint<true><<<nw_grid(h->P, 256 * NW_ADJ_TILES), 256, 0, h->stream>>>(h->P, h->slot, h->sfaces, h->w0, h->w1, h->w2, h->rx, h->ry, h->rz,
                                                                h->acc, h->st, 0, 0, h->M, h->F);
    NW_LAUNCH_CHECK();
    return NW_OK;
}

int nw_launch_sweep2(nw_ctx *h) {
    const int B = 256;
    const int G = h->n_partials;
    k_sweep2<<<G, B, 0, h->stream>>>(h->P, h->slot, h->sfaces, h->w0, h->w1, h->w2, h->rx, h->ry, h->rz, h->Sq,
                                      h->has_mask ? h->pmask : nullptr, h->st, h->partials);
    NW_LAUNCH_CHECK();
    k_fold_partials<<<NW_NSUM, 256, 0, h->stream>>>(h->partials, G, h->st);
    NW_LAUNCH_CHECK();
    return NW_OK;
}

int nw_launch_influence(nw_ctx *h) {
    if (h->P == 0) return NW_OK;
    k_apply_infl<<<nw_grid(h->P, 256), 256, 0, h->stream>>>(h->P, h->slot, h->sfaces, h->w0, h->w1, h->w2, h->acc, h->st);
    NW_LAUNCH_CHECK();
    return NW_OK;
}

static int ensure_scratchP(nw_ctx *h) {
    if (h->scratchP_elems < 6 * h->P || !h->scratchP) {
        NW_CHECK(nw_alloc(h, &h->scratchP, (size_t)6 * h->P + 8));
        h->scratchP_elems = 6 * h->P;
    }
    return NW_OK;
}

static int require_weights(nw_ctx *h, const char *who) {
    NW_ARG(h->M > 0 && h->px, "points and topology must be set first");
    if (!h->weights_valid) {
        h->err = std::string(who) + ": weights not computed (call nw_compute_weights or nw_search first)";
        return NW_ERR_ARG;
    }
    return NW_OK;
}

extern "C" int nw_compute_weights(nw_ctx *h) {
    if (!h) return NW_ERR_ARG;
    NW_ARG(h->M > 0 && (h->px || h->P == 0), "nw_compute_weights: points and topology must be set first");
    NW_CUDA(cudaSetDevice(h->device));
    {
        SolverState z;
        memset(&z, 0, sizeof(z));
        for (int a = 0; a < 3; ++a) { z.bbox[a] = 0x7fffffff; z.bbox[3 + a] = (int)0x80000000; }
        NW_CUDA(cudaMemcpyAsync(h->st, &z, sizeof(SolverState), cudaMemcpyHostToDevice, h->stream));
    }
    NW_CHECK(nw_set_acc_shifts(h));             // first: it refreshes the coordinate bound the refit folds into the boxes
    NW_CHECK(nw_tree_refit(h));
    NW_CHECK(nw_launch_sweep1(h, false));
    NW_CUDA(cudaStreamSynchronize(h->stream));
    h->weights_valid = true;
    return NW_OK;
}

extern "C" int nw_get_weights(nw_ctx *h, int32_t *v_idx, float *w, double *dist, int32_t *face) {
    if (!h) return NW_ERR_ARG;
    NW_CHECK(require_weights(h, "nw_get_weights"));
    NW_CUDA(cudaSetDevice(h->device));
    const int64_t P = h->P;
    if (P == 0) return NW_OK;
    const int B = 256;
    NW_CHECK(ensure_scratchP(h));
    cudaStream_t s = h->stream;
    if (v_idx || face) {
        int *dv = (int *)h->scratchP, *df = dv + 3 * P;
        k_scatter_vidx<<<nw_grid(P, B), B, 0, s>>>(h->slot, h->sfaces, h->perm, P, v_idx ? dv : nullptr, face ? df : nullptr);
        NW_LAUNCH_CHECK();
        if (v_idx) NW_CUDA(cudaMemcpyAsync(v_idx, dv, sizeof(int) * 3 * P, cudaMemcpyDeviceToHost, s));
        if (face) NW_CUDA(cudaMemcpyAsync(face, df, sizeof(int) * P, cudaMemcpyDeviceToHost, s));
        NW_CUDA(cudaStreamSynchronize(s));
    }
    if (w) {
        k_scatter_caller3<<<nw_grid(P, B), B, 0, s>>>(h->w0, h->w1, h->w2, h->perm, P, h->scratchP);
        NW_LAUNCH_CHECK();
        NW_CUDA(cudaMemcpyAsync(w, h->scratchP, sizeof(float) * 3 * P, cudaMemcpyDeviceToHost, s));
        NW_CUDA(cudaStreamSynchronize(s));
    }
    if (dist) {
        double *dd = (double *)h->scratchP;
        if (h->px64) k_scatter_dist<true><<<nw_grid(P, B), B, 0, s>>>(h->slot, h->cent, h->points_mode ? h->cent64 : nullptr, h->perm, P, h->px, h->py, h->pz, h->px64, h->py64, h->pz64, dd);
        else k_scatter_dist<false><<<nw_grid(P, B), B, 0, s>>>(h->slot, h->cent, h->points_mode ? h->cent64 : nullptr, h->perm, P, h->px, h->py, h->pz, nullptr, nullptr, nullptr, dd);
        NW_LAUNCH_CHECK();
        NW_CUDA(cudaMemcpyAsync(dist, dd, sizeof(double) * P, cudaMemcpyDeviceToHost, s));
        NW_CUDA(cudaStreamSynchronize(s));
    }
    return NW_OK;
}

extern "C" int nw_apply_A(nw_ctx *h, const float *x, float *y) {
    if (!h) return NW_ERR_ARG;
    NW_CHECK(require_weights(h, "nw_apply_A"));
    NW_CUDA(cudaSetDevice(h->device));
    const int64_t P = h->P;
    if (P == 0) return NW_OK;
    const int B = 256;
    cudaStream_t s = h->stream;
    NW_CHECK(ensure_scratchP(h));
    float4 *xq = nullptr;
    NW_CHECK(nw_alloc(h, &xq, (size_t)h->M));
    NW_CUDA(cudaMemcpyAsync(h->scratchM, x, sizeof(float) * 3 * h->M, cudaMemcpyHostToDevice, s));
    k_pack3<<<nw_grid(h->M, B), B, 0, s>>>(h->scratchM, h->M, xq);
    NW_LAUNCH_CHECK();
    float *yx = h->scratchP, *yy = yx + P, *yz = yy + P, *out = yz + P;
    k_apply_A<<<nw_grid(P, B), B, 0, s>>>(P, h->slot, h->sfaces, h->w0, h->w1, h->w2, xq, yx, yy, yz);
    NW_LAUNCH_CHECK();
    k_scatter_caller3<<<nw_grid(P, B), B, 0, s>>>(yx, yy, yz, h->perm, P, out);
    NW_LAUNCH_CHECK();
    NW_CUDA(cudaMemcpyAsync(y, out, sizeof(float) * 3 * P, cudaMemcpyDeviceToHost, s));
    NW_CUDA(cudaStreamSynchronize(s));
    nw_free(&xq);
    return NW_OK;
}

int nw_apply_AH_device(nw_ctx *h, const float *rx, const float *ry, const float *rz, double bound, float *out3M) {
    // shift from an a-priori bound on |w r| summed over every rank's points
    const int B = 256;
    cudaStream_t s = h->stream;
    // (the same rule as k_shift_final: the sum over all ranks stays below 2^61 and every term below 2^38)
    double tot = bound * (double)std::max<int64_t>(h->P_global, 1);
    int e = 0, et = 0;
    frexp(tot > 0 ? tot : 1.0, &e);
    frexp(bound > 0 ? bound : 1.0, &et);
    int shift = std::max(-100, std::min(40, std::min(61 - e, 38 - et)));
    NW_CUDA(cudaMemsetAsync(h->acc, 0, sizeof(unsigned long long) * 4 * h->M, s));
    if (h->P) {
        k_adjoint<false><<<nw_grid(h->P, B * NW_ADJ_TILES), B, 0, s>>>(h->P, h->slot, h->sfaces, h->w0, h->w1, h->w2, rx, ry, rz, h->acc, nullptr, shift, 0, h->M, h->F);
        NW_LAUNCH_CHECK();
    }
    NW_CHECK(nw_allreduce_acc(h));
    k_acc_to_float3<<<nw_grid(h->M, B), B, 0, s>>>(h->acc, h->M, shift, out3M, 1);
    NW_LAUNCH_CHECK();
    return NW_OK;
}

__global__ void k_absmax(const float *__restrict__ v, int64_t n, float *out) {
    float m = 0.f;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        float a = fabsf(v[i]);
        if (!(a <= FLT_MAX)) a = FLT_MAX;
        m = fmaxf(m, a);
    }
    for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) atomicMax((int *)out, __float_as_int(m));
}

int nw_comm_allreduce_host_doubles(nw_ctx *h, double *vals, int n);

extern "C" int nw_apply_AH(nw_ctx *h, const float *r, float *y) {
    if (!h) return NW_ERR_ARG;
    NW_CHECK(require_weights(h, "nw_apply_AH"));
    NW_CUDA(cudaSetDevice(h->device));
    const int64_t P = h->P;
    const int B = 256;
    cudaStream_t s = h->stream;
    NW_CHECK(ensure_scratchP(h));
    float *in = h->scratchP, *rx = in + 3 * P, *ry = rx + P, *rz = ry + P;
    float *d_max = nullptr;
    NW_CHECK(nw_alloc(h, &d_max, 1));
    NW_CUDA(cudaMemsetAsync(d_max, 0, sizeof(float), s));
    if (P) {
        NW_CUDA(cudaMemcpyAsync(in, r, sizeof(float) * 3 * P, cudaMemcpyHostToDevice, s));
        k_gather_sorted3<<<nw_grid(P, B), B, 0, s>>>(in, h->perm, P, rx, ry, rz);
        NW_LAUNCH_CHECK();
        k_absmax<<<std::min(nw_grid(3 * P, B), 592), B, 0, s>>>(in, 3 * P, d_max);
        NW_LAUNCH_CHECK();
    }
    float mx = 0.f;
    NW_CUDA(cudaMemcpyAsync(&mx, d_max, sizeof(float), cudaMemcpyDeviceToHost, s));
    NW_CUDA(cudaStreamSynchronize(s));
    nw_free(&d_max);
    double bound = mx;
    if (h->nranks > 1) {
        std::vector<double> slots(h->nranks, 0.0);
        slots[h->rank] = bound;
        NW_CHECK(nw_comm_allreduce_host_doubles(h, slots.data(), h->nranks));
        for (double v : slots) bound = std::max(bound, v);
    }
    NW_CHECK(nw_apply_AH_device(h, rx, ry, rz, bound, h->scratchM));
    NW_CUDA(cudaMemcpyAsync(y, h->scratchM, sizeof(float) * 3 * h->M, cudaMemcpyDeviceToHost, s));
    NW_CUDA(cudaStreamSynchronize(s));
    return NW_OK;
}

extern "C" int nw_get_res(nw_ctx *h, float *res) {
    if (!h) return NW_ERR_ARG;
    NW_ARG(h->px || h->P == 0, "nw_get_res: no points");
    NW_CUDA(cudaSetDevice(h->device));
    const int64_t P = h->P;
    if (P == 0) return NW_OK;
    NW_CHECK(ensure_scratchP(h));
    k_scatter_caller3<<<nw_grid(P, 256), 256, 0, h->stream>>>(h->rx, h->ry, h->rz, h->perm, P, h->scratchP);
    NW_LAUNCH_CHECK();
    NW_CUDA(cudaMemcpyAsync(res, h->scratchP, sizeof(float) * 3 * P, cudaMemcpyDeviceToHost, h->stream));
    NW_CUDA(cudaStreamSynchronize(h->stream));
    return NW_OK;
}

// ---- measurement hook (benchhook.cu) ---------------------------------------------------------------
int nw_bench_launch(nw_ctx *h, const char *name) {
    const int B = 256;
    const int64_t P = h->P;
    cudaStream_t s = h->stream;
    std::string n(name);
    if (n == "apply_A") {
        NW_CHECK(ensure_scratchP(h));
        float *yx = h->scratchP, *yy = yx + P, *yz = yy + P;
        k_apply_A<<<nw_grid(P, B), B, 0, s>>>(P, h->slot, h->sfaces, h->w0, h->w1, h->w2, h->posq, yx, yy, yz);
    } else if (n == "apply_AH") {
        k_adjoint<false><<<nw_grid(P, B * NW_ADJ_TILES), B, 0, s>>>(P, h->slot, h->sfaces, h->w0, h->w1, h->w2, h->rx, h->ry, h->rz, h->acc, nullptr, 20, 0, h->M, h->F);
    } else if (n == "adjoint") {
        return nw_launch_adjoint(h);
    } else if (n == "sweep1") {
        return nw_launch_sweep1(h, true);
    } else if (n == "nn_weights") {
        return nw_launch_sweep1(h, false);
    } else if (n == "sweep2") {
        return nw_launch_sweep2(h);
    } else if (n == "mesh_prior") {
        return nw_launch_mesh_prior(h, true);
    } else if (n == "refit") {
        return nw_tree_refit(h);
    } else if (n == "allreduce_acc") {
        return nw_allreduce_acc(h);              // N > 1: the per-iteration collective alone, all ranks in lockstep
    } else {
        h->err = "nw_bench_kernel: unknown kernel name " + n;
        return NW_ERR_ARG;
    }
    NW_LAUNCH_CHECK();
    return NW_OK;
}

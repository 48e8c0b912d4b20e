// hausdorff.cu -- certified bounds of the one-sided Hausdorff distance from a mesh A passed in to the handle's mesh B
// (nw_hausdorff_bounds).
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

extern "C" int nw_hausdorff_bounds(nw_ctx *h, const float *pos, int M, const int32_t *faces, int F, double tol, int64_t max_queries,
                                   double bounds[2], double witness[3], int32_t witness_faces[2], int64_t stats[5]) {
    if (!h) return NW_ERR_ARG;
    const std::string w("nw_hausdorff_bounds");
    NW_CHECK(nw_mesh_check(h, w));
    NW_ARG(pos != nullptr && faces != nullptr && M > 0 && F > 0, w + ": the mesh passed in has no vertices or no faces");
    NW_ARG(F <= 0x7fffffff / 3 && M <= 0x7fffffff / 3, w + ": the mesh passed in is too large (3 M and 3 F must fit int32)");
    NW_ARG(tol >= 0.0 && tol <= DBL_MAX, w + ": tol must be finite and >= 0");
    NW_CUDA(cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    const int B = 256;

    // A on the device; its faces checked, its used vertices found; B's face row -> slot table
    NW_CHECK(nw_alloc(h, &h->hb_st, sizeof(HbState)));
    HbState *st = (HbState *)h->hb_st;
    HbState hs;
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
    int nu = 0;
    NW_CUDA(cudaMemcpyAsync(&hs, st, sizeof(hs), cudaMemcpyDeviceToHost, s));
    NW_CUDA(cudaMemcpyAsync(&nu, h->hb_idx + M, sizeof(int), cudaMemcpyDeviceToHost, s));
    NW_CUDA(cudaStreamSynchronize(s));
    NW_ARG(hs.bad == 0, w + ": a face index of the mesh passed in is outside [0, M)");
    NW_ARG(hs.nonfinite < F, w + ": the mesh passed in has no face with finite corners");
    NW_ARG(hs.b_finite != 0, w + ": the handle's mesh has no face with finite corners");
    NW_ARG(max_queries >= nu, w + ": max_queries must be at least the number of vertices the finite faces use (" + std::to_string(nu) + ")");

    // level 0: the used vertices, unseeded; the slack of the call from them and B's vertices; one entry per face
    NW_CHECK(hb_queries(h, (size_t)nu));
    k_hb_vertices<<<nw_grid(M, B), B, 0, s>>>(h->hb_pos, h->hb_vface, h->hb_flag, h->hb_idx, M, h->hb_q, h->hb_qa);
    NW_LAUNCH_CHECK();
    NW_CHECK(nw_surface_boxes(h, h->hb_q, h->hb_q + 1, h->hb_q + 2, nu, 3, true));
    NW_CHECK(nw_alloc(h, &h->hb_ent[0], sizeof(HbEntry) * (size_t)F));
    k_hb_level0<<<nw_grid(F, B), B, 0, s>>>(h->hb_faces, h->hb_pos, h->hb_idx, F, (HbEntry *)h->hb_ent[0]);
    NW_LAUNCH_CHECK();
    NW_CHECK(hb_walk(h, nu, false));

    // bound, retire, split: one level at a time, until nothing survives or the next level would pass the budget
    int n = F, cur = 0, levels = 0;
    int64_t walks = nu, bounded = F - hs.nonfinite;
    bool converged = false;
    while (true) {
        ++levels;
        NW_CHECK(nw_alloc(h, &h->hb_flag, (size_t)n + 1)); NW_CHECK(nw_alloc(h, &h->hb_idx, (size_t)n + 1));
        k_hb_bound<<<nw_grid((int64_t)n + 1, 128), 128, 0, s>>>((HbEntry *)h->hb_ent[cur], n, h->hb_qd, h->hb_qf, h->faces, h->posq, h->F,
                                                              h->surf_bits, tol, st, h->hb_flag);
        NW_LAUNCH_CHECK();
        NW_CHECK(hb_scan(h, n));
        int S = 0;
        NW_CUDA(cudaMemcpyAsync(&S, h->hb_idx + n, sizeof(int), cudaMemcpyDeviceToHost, s));
        NW_CUDA(cudaStreamSynchronize(s));
        if (S == 0) { converged = true; break; }
        if (levels >= NW_HB_MAX_LEVELS || walks + 3 * (int64_t)S > max_queries || 4 * (int64_t)S > 0x7fffffff - 1) break;
        const int nxt = cur ^ 1;
        NW_CHECK(nw_alloc(h, &h->hb_ent[nxt], sizeof(HbEntry) * 4 * (size_t)S));
        NW_CHECK(hb_queries(h, 3 * (size_t)S));
        k_hb_split<<<nw_grid(n, B), B, 0, s>>>((const HbEntry *)h->hb_ent[cur], n, h->hb_flag, h->hb_idx, h->hb_slot,
                                               (HbEntry *)h->hb_ent[nxt], h->hb_q, h->hb_qs, h->hb_qa);
        NW_LAUNCH_CHECK();
        NW_CHECK(hb_walk(h, 3 * S, true));
        walks += 3 * (int64_t)S;
        n = 4 * S;
        bounded += n;
        cur = nxt;
    }
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

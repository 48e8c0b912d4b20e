// common.cuh -- handle layout, error plumbing and small device helpers shared by all kernels.
#pragma once
#include <cuda_runtime.h>
#include <cfloat>
#include <stdint.h>
#include <string>
#include <unordered_map>
#include <vector>
#include "../../include/nanowrap.h"

#define NW_MAX_LEVELS 12
#define NW_MAX_ITERS 4096
#define NW_S2_PTS 4      // k_sweep2: points per thread (their dependent load chains slot -> face -> S overlap); sizes its partials
#define NW_N_STAGES 11   // refit, shift, sweep1, allreduce_acc, mesh_prior, sweep2, allreduce_scalars, solve_update, seed_leaders,
                         // topology_build (device side of nw_set_topology*: feet, unpack, Hilbert sort, tables, frames), adjoint

// Node bound = ORIENTED box: a surface patch is thin along its normal and tilted against the coordinate axes, so an
// axis-aligned box is mostly empty space.  Axes n (patch normal), t1 = tangent_of(n), t2 = n x t1; one interval per axis.
// It only ever prunes: the answer never depends on how tight it is.  (A spherical shell fitted to each node, which
// removes the sagitta of large curved patches, was implemented and measured at C3: -4 % node tests, +15 % per test.)
// -DNW_BOUNDS_CHECK (NW_EXTRA_FLAGS=-DNW_BOUNDS_CHECK python -m ch_shrinkwrap_b200.build -f): device-side assertions on every
// index the search and the adjoint scatter form -- node ids, slots, vertex ids, shared-memory rows.  compute-sanitizer is
// closed on the GPU pool this was developed on; the -m gpu suite run against that build is the memory-safety evidence
// (profiles/).
#ifdef NW_BOUNDS_CHECK
#include <cassert>
#define NW_ASSERT(c) assert(c)
#else
#define NW_ASSERT(c) ((void)0)
#endif

struct Box {
    float4 a;   // n.x t1.x | n.y t1.y            the search decides most nodes from a, b, d alone (normal + first tangent axis,
    float4 b;   // n.z t1.z | n-min t1-min        sweep.cu: test_node) and loads c only for the rest; the two axes are interleaved
    float4 c;   // t2.x t2.y t2.z | t2-max        so that each (n, t1) pair is an aligned register pair (packed FFMA2 experiment)
    float4 d;   // n-max t1-max | first child (leaf: first slot) | (node is a last child) << 31, as int bits | t2-min
    __host__ __device__ __forceinline__ float3 normal() const { return make_float3(a.x, a.z, b.x); }
    __host__ __device__ __forceinline__ float3 tan1() const { return make_float3(a.y, a.w, b.y); }
    __host__ __device__ __forceinline__ float3 tan2() const { return make_float3(c.x, c.y, c.z); }
    // interval ends: axis 0 = normal, 1 = t1, 2 = t2
    __host__ __device__ __forceinline__ float *lo(int k) { return k == 0 ? &b.z : k == 1 ? &b.w : &d.w; }
    __host__ __device__ __forceinline__ float *hi(int k) { return k == 0 ? &d.x : k == 1 ? &d.y : &c.w; }
    __host__ __device__ __forceinline__ float lo(int k) const { return k == 0 ? b.z : k == 1 ? b.w : d.w; }
    __host__ __device__ __forceinline__ float hi(int k) const { return k == 0 ? d.x : k == 1 ? d.y : c.w; }
};              // 64 B

// Ordered-int encoding of floats: f2ord orders like the floats as signed ints, f2u as unsigned ints, so interval ends can be
// merged with integer atomics and REDUX.  The box intervals hold f2ord bits while they are being measured.
__device__ __forceinline__ int f2ord(float f) { int i = __float_as_int(f); return i >= 0 ? i : i ^ 0x7fffffff; }
__device__ __forceinline__ float ord2f(int i) { return __int_as_float(i >= 0 ? i : i ^ 0x7fffffff); }
__device__ __forceinline__ unsigned f2u(float f) { return (unsigned)f2ord(f) ^ 0x80000000u; }
__device__ __forceinline__ int u2ord(unsigned u) { return (int)(u ^ 0x80000000u); }
#define NW_EMPTY_LO __int_as_float(f2ord(FLT_MAX))      // ordered-int encodings of an empty interval
#define NW_EMPTY_HI __int_as_float(f2ord(-FLT_MAX))

// One level of an extents pass (tree.cu: k_extents, surface.cu: k_tri_extents): a live lane's member, projected onto the
// frame of boxes[node] by project(box, lo, hi), spans [lo, hi] per axis; finite == false contributes nothing.  Lanes that
// share the node are reduced with REDUX first, then the run's first lane applies one ordered-int atomic min/max per quantity.
template <typename Project>
__device__ __forceinline__ void nw_merge_extents(Box *boxes, int node, bool live, bool finite, Project project) {
    // lanes that share the node: the slots are sorted by key, so equal nodes are runs of consecutive lanes -- run heads
    // from one shuffle and a ballot (match_any costs several times more)
    const unsigned lane = threadIdx.x & 31;
    const int prev = __shfl_up_sync(0xffffffffu, node, 1);
    const unsigned heads = __ballot_sync(0xffffffffu, lane == 0 || prev != node || !live);
    const unsigned upto = 0xffffffffu >> (31 - lane);                           // lanes 0..lane
    const int first = 31 - __clz(heads & upto);
    const unsigned above = heads & ~upto;
    const unsigned grp = (above ? ((1u << (__ffs(above) - 1)) - 1u) : 0xffffffffu) & ~((1u << first) - 1u);
    Box *b = &boxes[node];
    float lo[3] = {0.f, 0.f, 0.f}, hi[3] = {0.f, 0.f, 0.f};
    if (live) project(b, lo, hi);
    unsigned mn[3], mx[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        mn[k] = __reduce_min_sync(grp, finite ? f2u(lo[k]) : 0xffffffffu);
        mx[k] = __reduce_max_sync(grp, finite ? f2u(hi[k]) : 0u);
    }
    if (live && lane == (unsigned)first && mn[0] <= mx[0]) {
        // the upper levels are hit by thousands of warps and all but the first few change nothing: look first
        // (an L2 read; a stale value only costs a redundant atomic, the atomics themselves are monotone)
        const float4 cb = __ldcg(&b->b), cd = __ldcg(&b->d);
        const float ch2 = __ldcg(&b->c.w);
        if (u2ord(mn[0]) < __float_as_int(cb.z)) atomicMin((int *)&b->b.z, u2ord(mn[0]));
        if (u2ord(mx[0]) > __float_as_int(cd.x)) atomicMax((int *)&b->d.x, u2ord(mx[0]));
        if (u2ord(mn[1]) < __float_as_int(cb.w)) atomicMin((int *)&b->b.w, u2ord(mn[1]));
        if (u2ord(mx[1]) > __float_as_int(cd.y)) atomicMax((int *)&b->d.y, u2ord(mx[1]));
        if (u2ord(mn[2]) < __float_as_int(cd.w)) atomicMin((int *)&b->d.w, u2ord(mn[2]));
        if (u2ord(mx[2]) > __float_as_int(ch2)) atomicMax((int *)&b->c.w, u2ord(mx[2]));
    }
}

// the merged ordered-int intervals of a box -> floats, each end moved out by w (field by field: a loop over Box::lo(k) /
// hi(k) compiles to six scalar loads and stores instead of 128- and 64-bit ones)
__device__ __forceinline__ void nw_decode_box(Box *b, float w) {
    b->b.z = ord2f(__float_as_int(b->b.z)) - w; b->d.x = ord2f(__float_as_int(b->d.x)) + w;
    b->b.w = ord2f(__float_as_int(b->b.w)) - w; b->d.y = ord2f(__float_as_int(b->d.y)) + w;
    b->d.w = ord2f(__float_as_int(b->d.w)) - w; b->c.w = ord2f(__float_as_int(b->c.w)) + w;
}

// projection onto a node frame as the box stores it (t2 = c.xyz): the operations of the search's node test (sweep.cu)
__device__ __forceinline__ void project_frame(const float4 a, const float4 b, const float4 c, float x, float y, float z, float &pn,
                                              float &p1, float &p2) {
    pn = fmaf(a.x, x, fmaf(a.z, y, b.x * z));
    p1 = fmaf(a.y, x, fmaf(a.w, y, b.y * z));
    p2 = fmaf(c.x, x, fmaf(c.y, y, c.z * z));
}

// The slack of the triangle-bounded boxes (surface.cu: nw_surface_boxes): 2^-19 x the L1 bound of everything that is
// projected (the vertices, bits 0..2, and the queries, bits 3..5; zero without queries) -- the rule of tree.cu's k_box_decode,
// whose coord_l1 covers the fit's vertices and points only.  Queries given explicitly can lie much farther out than either.
__device__ __forceinline__ float call_slack(const unsigned *__restrict__ bits6) {
    float l1 = 0.f;
    for (int k = 0; k < 3; ++k) l1 += fmaxf(__uint_as_float(bits6[k]), __uint_as_float(bits6[3 + k]));
    return l1 * 1.9073486328125e-6f;
}

// orthonormal completion of a unit vector (Duff et al. 2017, branchless): returns t1; t2 = n x t1 everywhere.
// Used identically when boxes are built and when they are tested.
__host__ __device__ __forceinline__ float3 nw_tangent_of(const float nx, const float ny, const float nz) {
    const float sg = copysignf(1.0f, nz);
    const float a = -1.0f / (sg + nz);
    const float b = nx * ny * a;
    return make_float3(1.0f + sg * nx * nx * a, sg * b, -sg * nx);
}
struct TreeLevels {
    int n_levels;                 // level 0 = root, n_levels-1 = leaf level
    int count[NW_MAX_LEVELS];     // nodes per level
    int off[NW_MAX_LEVELS];       // global id of the first node of the level: levels are stored back to back, root = 0
};

// Scalars produced and consumed on the device inside one search() call.
struct SolverState {
    double c[4];                  // step coefficients of the current iteration
    double hw[6];                 // S^T S  (00,01,11,02,12,22)
    double gw[3];                 // -S^T prefs64
    double hc[6], gc[3], c0, res2;
    double last_tests[3];
    int n_tests;                  // how many of last_tests are valid (<=3), newest last
    int n_done;
    int stop;                     // stop rule fired: remaining kernels become no-ops
    int nan_flag;
    int n_search;                 // 2 on the first iteration of a call, 3 afterwards (last_step)
    int reg_mode;                 // regulariser L = LH: 0 = "I" (the reference's default, mesh_conj_grad.py:38), 1 = "wfunc" (:725-736)
    double tst[3], prefs32_2, prefs64_2;   // S0.S1, |S0|^2, |S1|^2 (test statistic); |prefs|^2 as float32 values / as float64 values
    int acc_shift;                // fixed-point fraction bits of the adjoint accumulators
    int infl_shift;               // ditto for the AH*1 accumulator
    int bbox[6];                  // ordered-int bounding box of the vertices (k_shift_partial -> k_shift_final)
    float coord_l1;               // bound on |x|+|y|+|z| over vertices and points (rounding slack of the box tests)
    float lam;
    float cell_escape;            // grid units: how far any centroid has left the 1024^3 cell it was keyed into at upload (k_refit_centroids)
    unsigned long long trav[4];   // traversal statistics: node tests, leaf visits, exact fp64 evaluations, max node tests of one point
};

struct nw_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    std::string err;
    int64_t launches = 0;
    std::unordered_map<void *, size_t> caps;     // capacity (bytes) of the buffer each pointer variable currently owns

    // ---- points (Hilbert-sorted SoA) ----
    int64_t P = 0;
    int64_t P_global = 0;
    float *px = nullptr, *py = nullptr, *pz = nullptr;
    double *px64 = nullptr, *py64 = nullptr, *pz64 = nullptr;    // only when float64 points were given
    float *sx = nullptr, *sy = nullptr, *sz = nullptr;           // sigma_inv (NULL -> scalar)
    float *wx = nullptr, *wy = nullptr, *wz = nullptr;           // weights when distinct from sigma_inv
    float sinv_scalar = 1.f;
    int reg_mode = 0;            // nw_set_regulariser
    int weights_mode = 0;        // 0: scalar weight = sinv_scalar; 1: weights = sigma_inv array; 2: own array
    float wmean = 1.f;           // mean of the weight array over all ranks (float32 like numpy)
    int has_mask = 0;            // some weight <= 0
    uint8_t *pmask = nullptr;    // 3 bits per point when has_mask
    int *perm = nullptr;         // sorted position -> caller's index
    int *slot = nullptr;         // nearest sorted-centroid slot per point (-1 = none yet)
    float *w0 = nullptr, *w1 = nullptr, *w2 = nullptr;
    float *rx = nullptr, *ry = nullptr, *rz = nullptr;
    float bbox_pts[6] = {0, 0, 0, 0, 0, 0};
    double wn_max = 1.0;
    bool weights_valid = false;

    // ---- mesh ----
    int M = 0, F = 0;
    float4 *posq = nullptr, *nrmq = nullptr;     // xyz + pad: one LDG.128 per gather
    int *faces = nullptr;                        // (F,3) as uploaded
    int *nbrT = nullptr;                         // neighbour table, k-major: nbrT[k*M + v]
    int *valence = nullptr;
    uint8_t *valid = nullptr;
    int *stage_nbr = nullptr, *stage_hev = nullptr;   // upload staging (reused across blocks)
    int *tb_small = nullptr, *tb_i0 = nullptr, *tb_i1 = nullptr;   // tree-build temporaries (reused across blocks)
    unsigned *tb_u0 = nullptr, *tb_u1 = nullptr, *tb_u2 = nullptr;
    // ---- search hierarchy over the face centroids (tree.cu) ----
    int4 *sfaces = nullptr;                      // per sorted slot: corner ids + face id
    float4 *cent = nullptr;                      // per sorted slot: centroid xyz + face id bits
    Box *boxes = nullptr;                        // per global node id (levels back to back, root = 0; see tree.cu)
    int *parent_g = nullptr; int2 *kids = nullptr;   // per global node id: parent | (the parent is a last child) << 31; first child / slot, count
    int *leaf_of_slot = nullptr;                 // per sorted slot: its leaf, numbered within the leaf level
    float *node_f = nullptr;                     // 5 floats per node: normal sums, then sphere-fit moments (upload time)
    TreeLevels tl;
    bool seeds_cold = true;                      // no nearest-face seeds yet for this topology
    float *fx = nullptr, *fy = nullptr, *fz = nullptr;   // foot points on the previous block's surface (seeds after a remesh)
    bool feet_valid = false;
    unsigned *fkeys = nullptr;                   // sorted Hilbert keys of the face centroids at upload time
    int *fkey_tab = nullptr;                     // lower_bound(fkeys, b << 15) for b = 0 .. 2^15: first step of the foot-point lookup
    float key_lo[3] = {0, 0, 0}, key_inv = 0.f;  // quantisation used for those keys
    unsigned *fcells = nullptr;                  // per sorted slot: grid cell of the centroid at upload time, x | y << 10 | z << 20
    bool points_mode = false;                    // the "faces" are raw target points (nw_set_point_targets): centroid = the point itself
    double *cent64 = nullptr;                    // points mode with float64 targets: exact coordinates per sorted slot (3 doubles)
    // ---- nw_surface_distance (surface.cu): only that call reads or writes these ----
    Box *tboxes = nullptr;                       // per global node id: the frames and links of `boxes`, intervals over face CORNERS
    char *surf_q = nullptr;                      // copy of explicit queries
    unsigned *surf_bits = nullptr;               // per-axis max |coordinate| of vertices and queries (rounding slack of the call)
    double *surf_dist = nullptr, *surf_closest = nullptr, *surf_part = nullptr;
    int *surf_face = nullptr;
    // nw_surface_signed_distance: edge and vertex tables of one topology (built on the first signed call), then per call the
    // vertex pseudonormals and the signed volume
    int64_t topo_gen = 0;                        // bumped by every nw_set_topology* and nw_set_point_targets (epoch moves more often)
    int64_t sgn_gen = -1;                        // the topo_gen the tables below describe
    int sgn_defects[5] = {0, 0, 0, 0, 0};        // boundary edges, edges on > 2 faces, co-directed edge pairs, faces repeating a
                                                 // vertex, vertices whose faces form more than one fan
    int *sgn_twin = nullptr;                     // 3F: the face across edge k (corner k -> k+1) of each face row, or -1
    int *sgn_voff = nullptr, *sgn_vface = nullptr;   // vertex -> incident face rows in increasing order (CSR: M+1, 3F)
    unsigned long long *sgn_k0 = nullptr, *sgn_k1 = nullptr;   // 3F sort keys
    int *sgn_i0 = nullptr, *sgn_i1 = nullptr;    // 3F sort values
    int *sgn_cnt = nullptr;                      // M+1 per-vertex counts, then the 5 defect counts
    double *sgn_nv = nullptr;                    // 3M: angle-weighted vertex pseudonormals at the current positions
    double *sgn_vpart = nullptr;                 // signed-volume partials, then the volume
    unsigned *sgn_bbox = nullptr;                // ordered-uint min xyz, max xyz of the vertices the faces use
    // ---- nw_self_intersections (intersect.cu): only that call (and tboxes / surf_bits, see above) touches these ----
    uint8_t *sx_flag = nullptr;                  // per sorted slot: 0 tested, 1 degenerate, 2 a non-finite corner
    int *sx_last = nullptr;                      // per global node id: its last slot
    unsigned long long *sx_keys = nullptr, *sx_sorted = nullptr;   // (f << 32) | g of every pair found, then sorted
    unsigned long long *sx_cnt = nullptr;        // pairs found, then the 4 statistics of nw_self_intersections
    int2 *sx_pairs = nullptr;                    // the sorted pairs as (f, g)
    // ---- solver vectors ----
    unsigned long long *acc = nullptr;           // (M,4) int64 fixed point: AH res xyz, AH 1
    float4 *Sq = nullptr;                        // search directions, interleaved: S_k of vertex v at Sq[3v + k] (48 B per vertex)
    double *fdef = nullptr;                      // (M,3)
    double *partials = nullptr;                  // per-CTA partial sums
    int n_partials = 0;
    SolverState *st = nullptr;                   // device
    double *hist = nullptr;                      // device: 5 x NW_MAX_ITERS (tests, ress, prefs, cpred, wpred)
    void *cub_tmp = nullptr;
    size_t cub_tmp_bytes = 0;
    float *scratchM = nullptr;                   // 3M floats
    float *scratchP = nullptr;                   // 3P floats
    int64_t scratchP_elems = 0;

    // ---- curvature (device copies are kept after a call so the kernel can be re-timed) ----
    float *curvK = nullptr;
    int curvM = 0;
    void *cvV = nullptr, *cvF = nullptr, *cvH = nullptr;
    float *cvOut = nullptr;
    double *cvJ = nullptr;
    int *cvOff = nullptr;
    float cv_dN = 0.1f, cv_kc = 1.f, cv_kg = 0.f, cv_c0 = 0.f;
    unsigned long long cv_seed = 0;

    // ---- measurement: CUDA events on the handle's stream ----
    int profile = 0;                             // 1: per-stage events inside nw_search
    std::vector<cudaEvent_t> ev_pool;
    std::vector<int> ev_stage;                   // stage id of interval [2k, 2k+1]
    size_t ev_used = 0;
    double stage_ms[NW_N_STAGES] = {0};
    std::vector<int> trace_stage; std::vector<float> trace_ms;   // the intervals of the last nw_search call, in launch order
    int64_t stage_launches[NW_N_STAGES] = {0};
    cudaEvent_t ev_search0 = nullptr, ev_search1 = nullptr;
    // nw_set_points temporaries, grow-only like everything else (a fit uploads its points once, a session many times)
    char *sp_pts = nullptr; unsigned long long *sp_k0 = nullptr, *sp_k1 = nullptr; int *sp_idx = nullptr; float *sp_tmp3 = nullptr;
    char *pin_host = nullptr; size_t pin_bytes = 0; bool pin_fresh = false;   // pinned read-back staging (nw_get_positions_strided)
    // k_sweep1 block schedule: blocks in descending order of their largest seed distance (sweep.cu: build_block_order)
    int *blk_order = nullptr, *blk_idx = nullptr; unsigned *blk_key = nullptr, *blk_key2 = nullptr; bool order_stale = true;
    int *blk_order_cold = nullptr; int cold_grid = 0;   // schedule of the first sweep of a fit: its costliest blocks run as quarter-packets
    bool leaders_fresh = false;                  // the seeds are the 1-in-32 root searches of a cold start, nothing has swept yet
    struct nw_uploader *uploader = nullptr;       // xfer.cu: pinned staging lanes for large host->device copies
    cudaEvent_t ev_seg0 = nullptr, ev_seg1 = nullptr;   // topology_build segments (profiling only)
    double last_search_ms = 0.0;
    // one captured CG iteration, instantiated once per (points, topology) epoch and replayed by every nw_search call on it
    cudaGraphExec_t iter_graph = nullptr;
    int64_t iter_graph_epoch = -1; int iter_graph_last_step = -1;
    int64_t epoch = 0;                           // bumped by everything that can move a device buffer or change a launch shape

    // ---- comm ----
    void *nccl = nullptr;                        // ncclComm_t
    int rank = 0, nranks = 1;
    int comm_status = 0;                         // error latched inside a collective sequence (nw_comm_agree)
};

#define NW_CUDA(call)                                                                      \
    do {                                                                                   \
        cudaError_t e_ = (call);                                                           \
        if (e_ != cudaSuccess) {                                                           \
            h->err = std::string(#call) + ": " + cudaGetErrorString(e_);                   \
            return NW_ERR_CUDA;                                                            \
        }                                                                                  \
    } while (0)

#define NW_CHECK(expr)                                                                     \
    do {                                                                                   \
        int r_ = (expr);                                                                   \
        if (r_ != NW_OK) return r_;                                                        \
    } while (0)

#define NW_ARG(cond, msg)                                                                  \
    do {                                                                                   \
        if (!(cond)) {                                                                     \
            h->err = msg;                                                                  \
            return NW_ERR_ARG;                                                             \
        }                                                                                  \
    } while (0)

// Grow-only allocation: a buffer is reused when it is already large enough (cudaFree synchronises the device and
// re-mapping hundreds of MB per remesh block costs far more than the block's kernels).
template <typename T>
static inline int nw_alloc(nw_ctx *h, T **p, size_t n) {
    const size_t bytes = n * sizeof(T);
    size_t cap = bytes;
    if (*p) {
        auto it = h->caps.find((void *)p);
        if (it != h->caps.end() && it->second >= bytes && bytes > 0) return NW_OK;
        // growing an existing array: a remesh changes M and F a little every block, so leave headroom instead of
        // paying cudaFree + cudaMalloc (measured: 0.14 ms per MB, and stalls of hundreds of ms) on every upload
        cap = bytes + bytes / 4;
        cudaFree(*p);
        *p = nullptr;
    }
    h->caps.erase((void *)p);
    if (n == 0) return NW_OK;
    NW_CUDA(cudaMalloc((void **)p, cap));
    h->caps[(void *)p] = cap;
    return NW_OK;
}
template <typename T>
static inline void nw_free(T **p) {
    if (*p) { cudaFree(*p); *p = nullptr; }
}

int nw_h2d(nw_ctx *h, void *dst, const void *src, size_t bytes);   // xfer.cu
int nw_h2d_strided32(nw_ctx *h, void *dst, const void *src, size_t bytes, size_t stride);
struct nw_h2d_job { void *dst; const void *src; size_t bytes, stride; };    // stride 4 = plain copy, else one int32 per `stride` source bytes
int nw_h2d_many(nw_ctx *h, const nw_h2d_job *jobs, int n_jobs);               // xfer.cu: one thread team for several arrays
void nw_uploader_destroy(nw_ctx *h);
int nw_fetch_positions_async(nw_ctx *h);                            // tree.cu

static inline int nw_grid(int64_t n, int block) { return (int)((n + block - 1) / block); }

#define NW_LAUNCH_CHECK()                                                                  \
    do {                                                                                   \
        h->launches++;                                                                     \
        cudaError_t e_ = cudaGetLastError();                                               \
        if (e_ != cudaSuccess) {                                                           \
            h->err = std::string("kernel launch: ") + cudaGetErrorString(e_);              \
            return NW_ERR_CUDA;                                                            \
        }                                                                                  \
    } while (0)

// 3-D Hilbert index (Skilling's transpose algorithm): unlike Morton order, every contiguous key range is a connected,
// compact blob, so fixed-size chunks of the sorted order make tight tree nodes and coherent warps.
template <typename U>
__host__ __device__ __forceinline__ void hilbert_axes_to_transpose(U &x, U &y, U &z, int bits) {
    U X[3] = {x, y, z};
    const U M = (U)1 << (bits - 1);
    for (U Q = M; Q > 1; Q >>= 1) {
        const U P = Q - 1;
        for (int i = 0; i < 3; ++i) {
            if (X[i] & Q) X[0] ^= P;
            else { const U t = (X[0] ^ X[i]) & P; X[0] ^= t; X[i] ^= t; }
        }
    }
    X[1] ^= X[0]; X[2] ^= X[1];
    U t = 0;
    for (U Q = M; Q > 1; Q >>= 1) if (X[2] & Q) t ^= Q - 1;
    x = X[0] ^ t; y = X[1] ^ t; z = X[2] ^ t;
}

// ---- internal entry points implemented across translation units -------------------------------
int nw_tree_build(nw_ctx *h);                 // after topology upload: Hilbert sort of faces, octree tables, frames
int nw_tree_refit(nw_ctx *h);                 // every iteration: centroids + boxes at the current f
int nw_launch_sweep1(nw_ctx *h, bool scatter);
int nw_launch_adjoint(nw_ctx *h);
int nw_launch_seed_leaders(nw_ctx *h);
int nw_save_feet(nw_ctx *h);
int nw_launch_sweep2(nw_ctx *h);
int nw_launch_mesh_prior(nw_ctx *h, bool write_dirs);
int nw_launch_solve_update(nw_ctx *h);
int nw_allreduce_acc(nw_ctx *h);
int nw_upload_replicated(nw_ctx *h, void *dst, const void *src, size_t bytes, size_t stride = 4);   // comm.cu
int nw_check_replicated(nw_ctx *h, const long long *vals, int n, const char *what);
int nw_allreduce_scalars(nw_ctx *h);
int nw_comm_agree(nw_ctx *h);
int nw_set_acc_shifts(nw_ctx *h);
int nw_curvature_relaunch(nw_ctx *h);
int nw_mesh_check(nw_ctx *h, const std::string &who);   // surface.cu: a mesh topology is loaded (not point targets)
// surface.cu: h->surf_bits (the slack of the call: the vertices, and Q queries q?[i * stride] when Q > 0) and h->tboxes (the
// triangle-bounded boxes at the current positions)
int nw_surface_boxes(nw_ctx *h, const void *qx, const void *qy, const void *qz, int64_t Q, int64_t stride, bool f64);

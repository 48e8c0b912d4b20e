// tree.cu -- mesh upload and the nearest-face search hierarchy over the face centroids.
//
// The reference finds each point's nearest face centroid with a host kd-tree rebuilt every iteration
// (mesh_conj_grad.py:443-454).  Here the faces are sorted ONCE per remesh block by the 3-D Hilbert key of
// their centroid (topology is fixed inside a block) and the hierarchy is the octree of occupied Hilbert cells
// (see the block comment further down); every iteration only re-evaluates the centroids at the current f and
// re-measures each node's oriented box.
#include <cub/cub.cuh>
#include <cfloat>
#include "common.cuh"
#include <thread>
#include <vector>

namespace {

// centroid exactly as numpy evaluates fv[faces].mean(1) in float32: ((a+b)+c)/3
__device__ __forceinline__ float3 centroid_f32(const float4 a, const float4 b, const float4 c) {
    float3 r;
    r.x = __fdiv_rn(__fadd_rn(__fadd_rn(a.x, b.x), c.x), 3.0f);
    r.y = __fdiv_rn(__fadd_rn(__fadd_rn(a.y, b.y), c.y), 3.0f);
    r.z = __fdiv_rn(__fadd_rn(__fadd_rn(a.z, b.z), c.z), 3.0f);
    return r;
}

__global__ void k_pack_vec3(const float *__restrict__ src, int M, float4 *__restrict__ dst) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < M) dst[i] = make_float4(src[3 * i], src[3 * i + 1], src[3 * i + 2], 0.f);
}

__global__ void k_unpack_vec3(const float4 *__restrict__ src, int M, float *__restrict__ dst) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < M) { float4 v = src[i]; dst[3 * i] = v.x; dst[3 * i + 1] = v.y; dst[3 * i + 2] = v.z; }
}

// (M,20) row-major -> k-major + valence (entries are -1 terminated, mesh_conj_grad.py:50-54).  With he_vertex the
// table holds half-edge indices and is mapped to neighbour vertices here (halfedges['vertex'][neighbors], :50).
__global__ void k_transpose_nbr(const int *__restrict__ nbr, const int *__restrict__ he_vertex, int n_he, int M,
                                int *__restrict__ nbrT, int *__restrict__ valence) {
    int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= M) return;
    int n = 0;
    bool open = true;
    for (int k = 0; k < NW_NEIGHBORSIZE; ++k) {
        int t = nbr[(size_t)v * NW_NEIGHBORSIZE + k];
        if (t >= 0 && he_vertex) t = (t < n_he) ? he_vertex[t] : -1;
        if (t < 0 || t >= M) open = false;
        if (open) ++n;
        nbrT[(size_t)k * M + v] = open ? t : -1;
    }
    valence[v] = n;
}

// vertex_t records (membrane_mesh_utils.h:57-65, 120 B) -> position / normal float4, valid flag, neighbour table
__global__ void k_unpack_vertex_records(const int *__restrict__ rec, int M, const int *__restrict__ he_vertex, int n_he,
                                        float4 *__restrict__ posq, float4 *__restrict__ nrmq, uint8_t *__restrict__ valid,
                                        int *__restrict__ nbrT, int *__restrict__ valence) {
    int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= M) return;
    const int *r = rec + (size_t)v * 30;            // 30 four-byte fields
    posq[v] = make_float4(__int_as_float(r[0]), __int_as_float(r[1]), __int_as_float(r[2]), 0.f);
    nrmq[v] = make_float4(__int_as_float(r[3]), __int_as_float(r[4]), __int_as_float(r[5]), 0.f);
    valid[v] = r[6] != -1;                          // halfedge != -1 (mesh_conj_grad.py:44)
    int n = 0;
    bool open = true;
    for (int k = 0; k < NW_NEIGHBORSIZE; ++k) {
        int t = r[8 + k];
        if (t >= 0) t = (t < n_he) ? he_vertex[t] : -1;
        if (t < 0 || t >= M) open = false;
        if (open) ++n;
        nbrT[(size_t)k * M + v] = open ? t : -1;
    }
    valence[v] = n;
}

// `points`: the "faces" are single target points (nw_set_point_targets): the centroid IS the point, no arithmetic
__device__ __forceinline__ float3 centroid_of(bool points, const float4 a, const float4 b, const float4 c) {
    return points ? make_float3(a.x, a.y, a.z) : centroid_f32(a, b, c);
}

__global__ void k_face_bbox(const int *__restrict__ faces, const float4 *__restrict__ pos, int F, int *__restrict__ out6, bool points) {
    float lo[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, hi[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
    for (int f = blockIdx.x * blockDim.x + threadIdx.x; f < F; f += gridDim.x * blockDim.x) {
        float3 c = centroid_of(points, pos[faces[3 * f]], pos[faces[3 * f + 1]], pos[faces[3 * f + 2]]);
        float v[3] = {c.x, c.y, c.z};
        for (int a = 0; a < 3; ++a) if (v[a] == v[a]) { lo[a] = fminf(lo[a], v[a]); hi[a] = fmaxf(hi[a], v[a]); }
    }
    for (int a = 0; a < 3; ++a)
        for (int o = 16; o; o >>= 1) {
            lo[a] = fminf(lo[a], __shfl_xor_sync(0xffffffffu, lo[a], o));
            hi[a] = fmaxf(hi[a], __shfl_xor_sync(0xffffffffu, hi[a], o));
        }
    if ((threadIdx.x & 31) == 0)
        for (int a = 0; a < 3; ++a) {
            int l = __float_as_int(lo[a]); l = l >= 0 ? l : l ^ 0x7fffffff;
            int u = __float_as_int(hi[a]); u = u >= 0 ? u : u ^ 0x7fffffff;
            atomicMin(out6 + a, l);
            atomicMax(out6 + 3 + a, u);
        }
}

__device__ __forceinline__ unsigned spread10(unsigned v) {
    v &= 0x3ffu;
    v = (v | v << 16) & 0x30000ffu;
    v = (v | v << 8) & 0x300f00fu;
    v = (v | v << 4) & 0x30c30c3u;
    v = (v | v << 2) & 0x9249249u;
    return v;
}

__global__ void k_face_keys(const int *__restrict__ faces, const float4 *__restrict__ pos, int F, float3 lo, float inv,
                            unsigned *__restrict__ keys, int *__restrict__ idx, unsigned *__restrict__ cells, bool points) {
    int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= F) return;
    float3 c = centroid_of(points, pos[faces[3 * f]], pos[faces[3 * f + 1]], pos[faces[3 * f + 2]]);
    unsigned qx = (unsigned)fminf(fmaxf((c.x - lo.x) * inv, 0.f), 1023.f);
    unsigned qy = (unsigned)fminf(fmaxf((c.y - lo.y) * inv, 0.f), 1023.f);
    unsigned qz = (unsigned)fminf(fmaxf((c.z - lo.z) * inv, 0.f), 1023.f);
    cells[f] = qx | (qy << 10) | (qz << 20);
    hilbert_axes_to_transpose(qx, qy, qz, 10);
    keys[f] = (spread10(qx) << 2) | (spread10(qy) << 1) | spread10(qz);
    idx[f] = f;
}

__global__ void k_sorted_faces(const int *__restrict__ faces, const int *__restrict__ order, int F, int4 *__restrict__ sfaces,
                               const unsigned *__restrict__ cells, unsigned *__restrict__ fcells) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= F) return;
    int f = order[i];
    sfaces[i] = make_int4(faces[3 * f], faces[3 * f + 1], faces[3 * f + 2], f);
    fcells[i] = cells[f];
}

__device__ __forceinline__ void project3(const float3 n, const float4 c, float &pn, float &p1, float &p2) {
    const float3 t1 = nw_tangent_of(n.x, n.y, n.z);
    const float3 t2 = make_float3(n.y * t1.z - n.z * t1.y, n.z * t1.x - n.x * t1.z, n.x * t1.y - n.y * t1.x);
    pn = fmaf(n.x, c.x, fmaf(n.y, c.y, n.z * c.z));
    p1 = fmaf(t1.x, c.x, fmaf(t1.y, c.y, t1.z * c.z));
    p2 = fmaf(t2.x, c.x, fmaf(t2.y, c.y, t2.z * c.z));
}

// ======================================================================================================================
// The hierarchy is the OCTREE OF OCCUPIED HILBERT CELLS: a level-k node is the set of centroids that share the first 3k
// bits of their (sorted) Hilbert key, i.e. one cube of the 2^k grid -- always a compact piece of surface.  (Cutting the
// sorted order into fixed-size chunks instead mixes pieces that are consecutive on the curve but far apart in space:
// measured boxes of 1/120 of the surface spanned half the object.)  Because the keys are sorted every node is a
// contiguous range of slots and its children are a contiguous range of nodes one level down.  Nodes have ONE numbering,
// the global id: the levels are stored back to back (root = 0, TreeLevels::off), and within a level nodes are in key
// order.  Three tables per node, all in global ids, are what the search and the refit walk:
//   kids[g]     = {first child, number of children}; for a leaf {first slot, number of centroids}
//   parent_g[g] = parent | (the PARENT is the last child of ITS parent) << 31, so that popping a level is one load
//                 (the root's entry: 0 | 1 << 31)
//   Box::d.z    = kids[g].x | (this node is a last child) << 31, as int bits: what a search step needs next, whether the
//                 node is pruned (next sibling or pop) or opened (first child), arrives with the box it has just loaded
// leaf_of_slot numbers the leaves within the leaf level (the leaf of slot s is leaf0 + leaf_of_slot[s]).
// ======================================================================================================================

// histogram of the level at which consecutive keys first differ (-> number of nodes of every level)
__global__ void k_level_histogram(const unsigned *__restrict__ keys, int F, int *__restrict__ hist) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    int lvl = 0;
    if (i < F && i > 0) {
        const unsigned x = keys[i] ^ keys[i - 1];
        if (x) lvl = (29 - (31 - __clz(x))) / 3 + 1;   // first level whose prefix differs from the predecessor's, 1..10
    }
    // one atomic per warp and level instead of one per face (11 hot addresses)
    for (int k = 1; k <= 10; ++k) {
        const unsigned m = __ballot_sync(0xffffffffu, lvl == k);
        if (m && (threadIdx.x & 31) == 0) atomicAdd(&hist[k], __popc(m));
    }
}

__global__ void k_level_flags(const unsigned *__restrict__ keys, int F, int shift, int *__restrict__ flag) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= F) return;
    flag[i] = (i == 0) ? 1 : (shift >= 32 ? 0 : ((keys[i] >> shift) != (keys[i - 1] >> shift)));
}

// slot i is the last slot of its level-`lvl` node
__device__ __forceinline__ bool ends_node(const unsigned *__restrict__ keys, int F, int lvl, int i) {
    return i == F - 1 || ((keys[i] ^ keys[i + 1]) >> (30 - 3 * lvl)) != 0;
}

// The tables of the level-`lvl` nodes, written once the level below them is numbered.  id_up / start_up: number within
// level `lvl` (inclusive scan of its flags, 1-based) of every slot / first slot of every node; id / start: the same for
// level `lvl` + 1, whose `start` is recorded here for the next call.  id == nullptr: level `lvl` is the leaf level, its
// children are the slots, and leaf_of_slot is written.  lvl < 0: only the root's start.
__global__ void k_level_tables(const unsigned *__restrict__ keys, int F, int lvl, int off_up, const int *__restrict__ id_up,
                               const int *__restrict__ start_up, int off, const int *__restrict__ id, int *__restrict__ start,
                               int *__restrict__ parent_g, int2 *__restrict__ kids, Box *__restrict__ boxes,
                               int *__restrict__ leaf_of_slot) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= F) return;
    if (!id) leaf_of_slot[i] = id_up[i] - 1;
    else if (i == 0 || id[i - 1] != id[i]) start[id[i] - 1] = i;
    if (lvl < 0 || !ends_node(keys, F, lvl, i)) return;
    // slot i ends node p: its children are the nodes (slots) from the one of its first slot to the one of slot i
    const int p = off_up + id_up[i] - 1, s0 = start_up[id_up[i] - 1];
    const int c0 = id ? off + id[s0] - 1 : s0, c1 = id ? off + id[i] - 1 : i;
    const unsigned last = (lvl == 0 || ends_node(keys, F, lvl - 1, i)) ? 0x80000000u : 0u;    // p ends where its parent does
    kids[p] = make_int2(c0, c1 - c0 + 1);
    boxes[p].d.z = __int_as_float((int)((unsigned)c0 | last));
    if (id) for (int c = c0; c <= c1; ++c) parent_g[c] = (int)((unsigned)p | last);
    if (lvl == 0) parent_g[0] = (int)0x80000000u;
}

// centroids at the current f, in sorted order
// Also measures how far (L-infinity, grid units, evaluated with the operations of k_face_keys) any centroid now lies
// outside the grid cell it was keyed into at upload: the slack of the cell-clearance early-out of the search (sweep.cu).
__global__ void k_refit_centroids(const int4 *__restrict__ sfaces, const float4 *__restrict__ pos, int F, float4 *__restrict__ cent,
                                  const unsigned *__restrict__ fcells, float3 lo, float inv, SolverState *st, bool points) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    float esc = 0.f;
    if (i < F) {
        const int4 sf = sfaces[i];
        const float3 cc = centroid_of(points, pos[sf.x], pos[sf.y], pos[sf.z]);
        cent[i] = make_float4(cc.x, cc.y, cc.z, __int_as_float(sf.w));
        const unsigned cell = fcells[i];
        const float gx = (cc.x - lo.x) * inv, gy = (cc.y - lo.y) * inv, gz = (cc.z - lo.z) * inv;
        const float cx = (float)(cell & 1023u), cy = (float)((cell >> 10) & 1023u), cz = (float)(cell >> 20);
        // the last cell of an axis also holds everything that was clamped into it
        esc = fmaxf(fmaxf(fmaxf(cx - gx, cx == 1023.f ? 0.f : gx - (cx + 1.f)), fmaxf(cy - gy, cy == 1023.f ? 0.f : gy - (cy + 1.f))),
                    fmaxf(fmaxf(cz - gz, cz == 1023.f ? 0.f : gz - (cz + 1.f)), 0.f));
        if (!(esc >= 0.f)) esc = __int_as_float(0x7f800000);      // NaN positions: no early-outs
    }
    const unsigned m = __reduce_max_sync(0xffffffffu, __float_as_uint(esc));    // non-negative floats order like their bits
    if ((threadIdx.x & 31) == 0 && m) atomicMax((unsigned *)&st->cell_escape, m);
}

// build pass A: area-weighted face normals summed into every ancestor -> node frames.  Bottom-up: every face adds its
// normal to its leaf (float atomics: the frames only prune, their last bits do not matter), then every level sums its
// children.  (The first version summed every face into all of its ancestors with MATCH + 96 shuffles per level: 183 us per
// build at C3 against ~40 now.)
__global__ void __launch_bounds__(256) k_leaf_normals(const int4 *__restrict__ sfaces, const float4 *__restrict__ pos, int F,
                                                      const int *__restrict__ leaf_of_slot, int leaf0, float *__restrict__ nsum) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= F) return;
    const int4 sf = sfaces[i];
    const float4 a = pos[sf.x], b = pos[sf.y], d = pos[sf.z];
    const float ux = b.x - a.x, uy = b.y - a.y, uz = b.z - a.z, vx = d.x - a.x, vy = d.y - a.y, vz = d.z - a.z;
    float3 fn = make_float3(uy * vz - uz * vy, uz * vx - ux * vz, ux * vy - uy * vx);
    if (!(fabsf(fn.x) <= FLT_MAX && fabsf(fn.y) <= FLT_MAX && fabsf(fn.z) <= FLT_MAX)) return;
    float *dst = nsum + 3 * (size_t)(leaf0 + leaf_of_slot[i]);
    atomicAdd(dst, fn.x); atomicAdd(dst + 1, fn.y); atomicAdd(dst + 2, fn.z);
}
__global__ void __launch_bounds__(256) k_up_normals(float *__restrict__ nsum, const int2 *__restrict__ kids, int first, int count) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= count) return;
    const int2 k = kids[first + j];
    float sx = 0.f, sy = 0.f, sz = 0.f;
    for (int c = k.x; c < k.x + k.y; ++c) {
        const float *s = nsum + 3 * (size_t)c;
        sx += s[0]; sy += s[1]; sz += s[2];
    }
    float *d = nsum + 3 * (size_t)(first + j);
    d[0] = sx; d[1] = sy; d[2] = sz;
}

// lower_bound of every 15-bit key prefix in the sorted face keys: k_seed_from_feet starts its binary search from this table
// (1 load + ~5 steps instead of 20 dependent steps through a 4 MB array)
__global__ void k_key_table(const unsigned *__restrict__ fkeys, int F, int *__restrict__ tab) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b > 32768) return;
    const unsigned long long key = (unsigned long long)b << 15;
    int lo = 0, hi = F;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if ((unsigned long long)fkeys[mid] < key) lo = mid + 1; else hi = mid;
    }
    tab[b] = lo;
}

// frames from the normal sums; intervals empty
__global__ void k_node_frames(Box *__restrict__ boxes, const float *__restrict__ nsum, int first, int count) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= count) return;
    const float *s = nsum + 3 * (size_t)(first + j);
    float3 n = make_float3(s[0], s[1], s[2]);
    const float nn = sqrtf(n.x * n.x + n.y * n.y + n.z * n.z);
    n = (nn > 1e-20f && nn <= FLT_MAX) ? make_float3(n.x / nn, n.y / nn, n.z / nn) : make_float3(0.f, 0.f, 1.f);
    Box *b = &boxes[first + j];
    const float3 t1 = nw_tangent_of(n.x, n.y, n.z);
    b->a = make_float4(n.x, t1.x, n.y, t1.y);
    b->b = make_float4(n.z, t1.z, NW_EMPTY_LO, NW_EMPTY_LO);
    // t2 = n x t1, exactly as project3 forms it
    b->c = make_float4(n.y * t1.z - n.z * t1.y, n.z * t1.x - n.x * t1.z, n.x * t1.y - n.y * t1.x, NW_EMPTY_HI);
    b->d.x = NW_EMPTY_HI; b->d.y = NW_EMPTY_HI; b->d.w = NW_EMPTY_LO;      // d.z: the search's link, written by k_level_tables
}

// every iteration: intervals back to "empty" (frames are kept for the whole block)
__global__ void k_reset_extents(Box *__restrict__ boxes, int first, int count) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= count) return;
    Box *b = &boxes[first + j];
    b->b.z = NW_EMPTY_LO; b->b.w = NW_EMPTY_LO; b->d.w = NW_EMPTY_LO; b->d.x = NW_EMPTY_HI; b->d.y = NW_EMPTY_HI; b->c.w = NW_EMPTY_HI;
}

// every iteration: each centroid projects onto the frame of every ancestor (common.cuh: nw_merge_extents)
__global__ void __launch_bounds__(256) k_extents(const float4 *__restrict__ cent, int F, const int *__restrict__ leaf_of_slot,
                                                 int leaf0, int leaf_level, const int *__restrict__ parent_g, Box *__restrict__ boxes) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = i < F;
    const float4 c = live ? cent[i] : make_float4(0.f, 0.f, 0.f, 0.f);
    const bool finite = live && (c.x == c.x) && (c.y == c.y) && (c.z == c.z);
    int node = live ? leaf0 + leaf_of_slot[i] : 0;
    for (int l = leaf_level; l >= 1; --l) {
        nw_merge_extents(boxes, node, live, finite, [&](const Box *b, float (&lo)[3], float (&hi)[3]) {
            const float4 ba = b->a;
            project3(make_float3(ba.x, ba.z, b->b.x), c, lo[0], lo[1], lo[2]);
            hi[0] = lo[0]; hi[1] = lo[1]; hi[2] = lo[2];
        });
        if (live) node = parent_g[node] & 0x7fffffff;
    }
}
// ordered-int -> float for the extents written by k_extents.  The intervals are widened by the rounding slack of the
// box test (2^-19 x the coordinate bound: >= 4x the worst-case error of the query's and the members' float32
// projections, see node_lb), so the test itself needs no per-axis subtraction.
__global__ void k_box_decode(Box *__restrict__ boxes, int first, int count, const SolverState *__restrict__ st) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    nw_decode_box(&boxes[first + i], st->coord_l1 * 1.9073486328125e-6f);
}

#define NW_NMOM 3        // floats per node of the build scratch (area-weighted normal sum)

inline float ordered_to_float(int v) {
    v = v >= 0 ? v : v ^ 0x7fffffff;
    float f;
    memcpy(&f, &v, 4);
    return f;
}

}  // namespace

static int set_topology_impl(nw_ctx *h, const float *pos, const float *nrm, const int32_t *faces, const int32_t *nbr,
                             const int32_t *he_vertex, int n_he, const uint8_t *valid, int M, int F, int he_stride = 4);

extern "C" int nw_set_topology(nw_ctx *h, const float *pos, const float *nrm, const int32_t *faces,
                               const int32_t *nbr, const uint8_t *valid, int M, int F) {
    return set_topology_impl(h, pos, nrm, faces, nbr, nullptr, 0, valid, M, F);
}

extern "C" int nw_set_topology_halfedge(nw_ctx *h, const float *pos, const float *nrm, const int32_t *faces,
                                        const int32_t *nbr_halfedge, const int32_t *he_vertex, int n_halfedges,
                                        const uint8_t *valid, int M, int F) {
    if (h && !(he_vertex && n_halfedges > 0)) { h->err = "nw_set_topology_halfedge: missing half-edge table"; return NW_ERR_ARG; }
    return set_topology_impl(h, pos, nrm, faces, nbr_halfedge, he_vertex, n_halfedges, valid, M, F);
}

extern "C" int nw_set_topology_records(nw_ctx *h, const void *vertex_records, const int32_t *faces, const int32_t *he_vertex,
                                       int he_stride_bytes, int n_halfedges, int M, int F) {
    if (h && !(vertex_records && he_vertex && n_halfedges > 0)) { h->err = "nw_set_topology_records: NULL array"; return NW_ERR_ARG; }
    if (h && !(he_stride_bytes >= 4 && he_stride_bytes % 4 == 0)) { h->err = "nw_set_topology_records: he_stride_bytes must be a multiple of 4"; return NW_ERR_ARG; }
    return set_topology_impl(h, (const float *)vertex_records, nullptr, faces, nullptr, he_vertex, n_halfedges, nullptr, M, F, he_stride_bytes);
}

// profiling: device time of the compute segments of an upload (the host->device copies between them are not counted)
static int seg_begin(nw_ctx *h) {
    if (!(h->profile & 1)) return NW_OK;
    if (!h->ev_seg0) { NW_CUDA(cudaEventCreate(&h->ev_seg0)); NW_CUDA(cudaEventCreate(&h->ev_seg1)); }
    NW_CUDA(cudaEventRecord(h->ev_seg0, h->stream));
    h->stage_launches[9] -= h->launches;
    return NW_OK;
}
static int seg_end(nw_ctx *h) {
    if (!(h->profile & 1)) return NW_OK;
    NW_CUDA(cudaEventRecord(h->ev_seg1, h->stream));
    NW_CUDA(cudaEventSynchronize(h->ev_seg1));
    float ms = 0.f;
    NW_CUDA(cudaEventElapsedTime(&ms, h->ev_seg0, h->ev_seg1));
    h->stage_ms[9] += ms;
    h->stage_launches[9] += h->launches;
    return NW_OK;
}

// nrm == NULL && nbr == NULL: `pos` points at M raw vertex_t records
static int set_topology_impl(nw_ctx *h, const float *pos, const float *nrm, const int32_t *faces, const int32_t *nbr,
                             const int32_t *he_vertex, int n_he, const uint8_t *valid, int M, int F, int he_stride) {
    if (!h) return NW_ERR_ARG;
    NW_ARG(M > 0 && F > 0, "nw_set_topology: empty mesh");
    const bool records = (nrm == nullptr && nbr == nullptr);
    NW_ARG(pos && faces && (records || (nrm && nbr)), "nw_set_topology: NULL array");
    NW_CUDA(cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    const int B = 256;
    {   // N > 1: a collective call; rank 0's arrays are the ones every rank ends up with
        const long long shape[7] = {M, F, n_he, records, valid != nullptr, he_vertex != nullptr, he_stride};
        NW_CHECK(nw_check_replicated(h, shape, 7, "nw_set_topology: mesh shape"));
    }
    NW_CHECK(seg_begin(h));
    NW_CHECK(nw_save_feet(h));       // seeds for the next block, taken from the mesh that is about to be replaced
    NW_CHECK(seg_end(h));
    h->M = M; h->F = F;
    h->epoch++;
    h->topo_gen++;
    h->weights_valid = false;
    h->pin_fresh = false;
    h->points_mode = false;
    nw_free(&h->cent64);
    NW_CHECK(nw_alloc(h, &h->posq, (size_t)M)); NW_CHECK(nw_alloc(h, &h->nrmq, (size_t)M));
    NW_CHECK(nw_alloc(h, &h->faces, (size_t)3 * F));
    NW_CHECK(nw_alloc(h, &h->nbrT, (size_t)NW_NEIGHBORSIZE * M)); NW_CHECK(nw_alloc(h, &h->valence, (size_t)M));
    NW_CHECK(nw_alloc(h, &h->valid, (size_t)M));
    NW_CHECK(nw_alloc(h, &h->acc, (size_t)4 * M));
    NW_CHECK(nw_alloc(h, &h->Sq, (size_t)3 * M));
    NW_CHECK(nw_alloc(h, &h->fdef, (size_t)3 * M));
    NW_CHECK(nw_alloc(h, &h->scratchM, (size_t)3 * M));
    NW_CHECK(nw_alloc(h, &h->sfaces, (size_t)F)); NW_CHECK(nw_alloc(h, &h->cent, (size_t)F));

    // staging buffers are members so that they are reused from block to block (grow-only)
    if (he_vertex) NW_CHECK(nw_alloc(h, &h->stage_hev, (size_t)n_he));
    if (records && he_vertex && h->nranks <= 1) {
        // single rank, raw records: the three arrays go up as ONE batch (xfer.cu: nw_h2d_many)
        NW_CHECK(nw_alloc(h, &h->stage_nbr, (size_t)30 * M));
        const nw_h2d_job jobs[3] = {{h->stage_hev, he_vertex, sizeof(int) * (size_t)n_he, (size_t)he_stride},
                                    {h->faces, faces, sizeof(int) * 3 * (size_t)F, 4},
                                    {h->stage_nbr, pos, (size_t)120 * M, 4}};
        NW_CHECK(nw_h2d_many(h, jobs, 3));
        NW_CHECK(seg_begin(h));
        k_unpack_vertex_records<<<nw_grid(M, B), B, 0, s>>>(h->stage_nbr, M, h->stage_hev, n_he, h->posq, h->nrmq, h->valid, h->nbrT, h->valence);
        h->launches += 1;
        NW_CHECK(seg_end(h));
    } else {
    if (he_vertex) NW_CHECK(nw_upload_replicated(h, h->stage_hev, he_vertex, sizeof(int) * (size_t)n_he, (size_t)he_stride));
    NW_CHECK(nw_upload_replicated(h, h->faces, faces, sizeof(int) * 3 * (size_t)F));
    if (records) {
        NW_CHECK(nw_alloc(h, &h->stage_nbr, (size_t)30 * M));
        NW_CHECK(nw_upload_replicated(h, h->stage_nbr, pos, (size_t)120 * M));
        NW_CHECK(seg_begin(h));
        k_unpack_vertex_records<<<nw_grid(M, B), B, 0, s>>>(h->stage_nbr, M, h->stage_hev, n_he, h->posq, h->nrmq, h->valid, h->nbrT, h->valence);
        h->launches += 1;
        NW_CHECK(seg_end(h));
    } else {
        NW_CHECK(nw_alloc(h, &h->stage_nbr, (size_t)NW_NEIGHBORSIZE * M));
        NW_CHECK(nw_upload_replicated(h, h->scratchM, pos, sizeof(float) * 3 * (size_t)M));
        NW_CHECK(seg_begin(h));
        k_pack_vec3<<<nw_grid(M, B), B, 0, s>>>(h->scratchM, M, h->posq);
        h->launches += 1;
        NW_CHECK(seg_end(h));
        NW_CUDA(cudaStreamSynchronize(s));
        NW_CHECK(nw_upload_replicated(h, h->scratchM, nrm, sizeof(float) * 3 * (size_t)M));
        NW_CHECK(seg_begin(h));
        k_pack_vec3<<<nw_grid(M, B), B, 0, s>>>(h->scratchM, M, h->nrmq);
        h->launches += 1;
        NW_CHECK(seg_end(h));
        NW_CHECK(nw_upload_replicated(h, h->stage_nbr, nbr, sizeof(int) * NW_NEIGHBORSIZE * (size_t)M));
        NW_CHECK(seg_begin(h));
        k_transpose_nbr<<<nw_grid(M, B), B, 0, s>>>(h->stage_nbr, he_vertex ? h->stage_hev : nullptr, n_he, M, h->nbrT, h->valence);
        h->launches += 1;
        NW_CHECK(seg_end(h));
        if (valid) NW_CHECK(nw_upload_replicated(h, h->valid, valid, (size_t)M));
        else NW_CUDA(cudaMemsetAsync(h->valid, 1, M, s));
    }
    }
    NW_CUDA(cudaStreamSynchronize(s));
    NW_CHECK(seg_begin(h));
    NW_CUDA(cudaMemsetAsync(h->acc, 0, sizeof(unsigned long long) * 4 * M, s));
    NW_CUDA(cudaMemsetAsync(h->Sq, 0, sizeof(float4) * 3 * M, s));
    // nearest-face slots refer to the previous block's sort order
    if (h->slot && h->P) NW_CUDA(cudaMemsetAsync(h->slot, 0xff, sizeof(int) * h->P, s));
    h->seeds_cold = true;
    h->order_stale = true;
    NW_CHECK(nw_tree_build(h));
    NW_CHECK(seg_end(h));
    return nw_comm_agree(h);        // N > 1: a rank whose upload failed makes EVERY rank return an error (no one is left waiting)
}

static int scan_inclusive(nw_ctx *h, const int *in, int *out, int n) {
    size_t tmp = 0;
    cub::DeviceScan::InclusiveSum(nullptr, tmp, in, out, n, h->stream);
    if (tmp > h->cub_tmp_bytes) { NW_CHECK(nw_alloc(h, (char **)&h->cub_tmp, tmp)); h->cub_tmp_bytes = tmp; }
    NW_CUDA(cub::DeviceScan::InclusiveSum(h->cub_tmp, tmp, in, out, n, h->stream));
    h->launches += 2;
    return NW_OK;
}

static int extents_pass(nw_ctx *h) {
    cudaStream_t s = h->stream;
    const int B = 256;
    const TreeLevels &tl = h->tl;
    const int first = tl.off[1], count = tl.off[tl.n_levels - 1] + tl.count[tl.n_levels - 1] - first;
    k_reset_extents<<<nw_grid(count, B), B, 0, s>>>(h->boxes, first, count);
    NW_LAUNCH_CHECK();
    k_extents<<<nw_grid(h->F, B), B, 0, s>>>(h->cent, h->F, h->leaf_of_slot, tl.off[tl.n_levels - 1], tl.n_levels - 1, h->parent_g,
                                             h->boxes);
    NW_LAUNCH_CHECK();
    k_box_decode<<<nw_grid(count, B), B, 0, s>>>(h->boxes, first, count, h->st);
    NW_LAUNCH_CHECK();
    return NW_OK;
}

static void launch_refit_centroids(nw_ctx *h) {
    cudaMemsetAsync(&h->st->cell_escape, 0, sizeof(float), h->stream);
    k_refit_centroids<<<nw_grid(h->F, 256), 256, 0, h->stream>>>(h->sfaces, h->posq, h->F, h->cent, h->fcells,
                                                                 make_float3(h->key_lo[0], h->key_lo[1], h->key_lo[2]), h->key_inv, h->st,
                                                                 h->points_mode);
}

int nw_tree_refit(nw_ctx *h) {
    launch_refit_centroids(h);
    NW_LAUNCH_CHECK();
    return extents_pass(h);
}

int nw_tree_build(nw_ctx *h) {
    cudaStream_t s = h->stream;
    const int B = 256, F = h->F;
    // build temporaries are members: reused from block to block (cudaFree synchronises and is slow)
    int *&d_bbox = h->tb_small, *&idx = h->tb_i0, *&order = h->tb_i1;
    unsigned *&keys = h->tb_u0, *&keys2 = h->tb_u1;
    NW_CHECK(nw_alloc(h, &d_bbox, 16));
    int init[6] = {0x7fffffff, 0x7fffffff, 0x7fffffff, (int)0x80000000, (int)0x80000000, (int)0x80000000};
    NW_CUDA(cudaMemcpyAsync(d_bbox, init, sizeof(init), cudaMemcpyHostToDevice, s));
    k_face_bbox<<<std::min(nw_grid(F, B), 148 * 4), B, 0, s>>>(h->faces, h->posq, F, d_bbox, h->points_mode);
    int bb[6];
    NW_CUDA(cudaMemcpyAsync(bb, d_bbox, sizeof(bb), cudaMemcpyDeviceToHost, s));
    NW_CUDA(cudaStreamSynchronize(s));
    float lo[3], hi[3];
    for (int a = 0; a < 3; ++a) { lo[a] = ordered_to_float(bb[a]); hi[a] = ordered_to_float(bb[3 + a]); }
    float ext = fmaxf(fmaxf(hi[0] - lo[0], hi[1] - lo[1]), hi[2] - lo[2]);
    float inv = (ext > 0.f && ext < FLT_MAX) ? 1023.f / ext : 0.f;
    NW_CHECK(nw_alloc(h, &keys, (size_t)F)); NW_CHECK(nw_alloc(h, &keys2, (size_t)F));
    NW_CHECK(nw_alloc(h, &idx, (size_t)F)); NW_CHECK(nw_alloc(h, &order, (size_t)F));
    unsigned *&cells = h->tb_u2;
    NW_CHECK(nw_alloc(h, &cells, (size_t)F)); NW_CHECK(nw_alloc(h, &h->fcells, (size_t)F));
    k_face_keys<<<nw_grid(F, B), B, 0, s>>>(h->faces, h->posq, F, make_float3(lo[0], lo[1], lo[2]), inv, keys, idx, cells, h->points_mode);
    size_t tmp = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, tmp, keys, keys2, idx, order, F, 0, 30, s);
    if (tmp > h->cub_tmp_bytes) { NW_CHECK(nw_alloc(h, (char **)&h->cub_tmp, tmp)); h->cub_tmp_bytes = tmp; }
    NW_CUDA(cub::DeviceRadixSort::SortPairs(h->cub_tmp, tmp, keys, keys2, idx, order, F, 0, 30, s));
    NW_CHECK(nw_alloc(h, &h->fkeys, (size_t)F));
    NW_CUDA(cudaMemcpyAsync(h->fkeys, keys2, sizeof(unsigned) * F, cudaMemcpyDeviceToDevice, s));
    NW_CHECK(nw_alloc(h, &h->fkey_tab, (size_t)32769));
    k_key_table<<<nw_grid(32769, B), B, 0, s>>>(h->fkeys, F, h->fkey_tab);
    h->key_lo[0] = lo[0]; h->key_lo[1] = lo[1]; h->key_lo[2] = lo[2]; h->key_inv = inv;
    k_sorted_faces<<<nw_grid(F, B), B, 0, s>>>(h->faces, order, F, h->sfaces, cells, h->fcells);
    h->launches += 7;

    // ---- level sizes: nodes of level k = distinct 3k-bit key prefixes; leaf level = deepest with >= 4 centroids per node
    int *hist = d_bbox;                                   // 16 ints
    NW_CUDA(cudaMemsetAsync(hist, 0, sizeof(int) * 16, s));
    k_level_histogram<<<nw_grid(F, B), B, 0, s>>>(h->fkeys, F, hist);
    int hh[16];
    NW_CUDA(cudaMemcpyAsync(hh, hist, sizeof(hh), cudaMemcpyDeviceToHost, s));
    NW_CUDA(cudaStreamSynchronize(s));
    int cnt[11];
    cnt[0] = 1;
    for (int k = 1; k <= 10; ++k) cnt[k] = cnt[k - 1] + hh[k];
    int kL = 1;
    const double occ = 3.0;                               // mean centroids per leaf cell, at least (measured at C3 with the packet search, blocks 0/1/2 of a fit: 1 -> 17.4/2.45/2.27 ms, 1.5 -> 13.6/2.27/2.19, 3 -> 12.1/2.27/2.09, 6 -> 12.3/2.58/2.45, 12 -> 13.4/2.59/2.43)
    for (int k = 1; k <= 10; ++k) if ((double)F / cnt[k] >= occ) kL = k;
    TreeLevels &tl = h->tl;
    tl.n_levels = kL + 1;
    int off = 0;
    for (int k = 0; k <= kL; ++k) {
        tl.count[k] = cnt[k]; tl.off[k] = off;
        off += cnt[k];
    }
    const int total = off;
    // the node count follows the shape of the mesh: the leaf level can change from one block to the next, which changes
    // the total 4-fold, and re-allocating stalls the upload (measured: 3 ms to 480 ms).  There are <= F/1.5 leaf cells
    // and, for a surface, a third of that above them (0.9 F in all; 1.33 F if the levels only double), so 1.5 F nodes is
    // a size that depends on the topology alone.
    const size_t room = std::max((size_t)total + total / 4, (size_t)F + F / 2) + 64;
    NW_CHECK(nw_alloc(h, &h->boxes, room)); NW_CHECK(nw_alloc(h, &h->parent_g, room)); NW_CHECK(nw_alloc(h, &h->kids, room));
    NW_CHECK(nw_alloc(h, &h->leaf_of_slot, (size_t)F));
    NW_CHECK(nw_alloc(h, &h->node_f, (size_t)NW_NMOM * room));
    // ---- tables: level k is numbered (flags, scan), then the level above it is linked to it; the leaf level last
    // reuse the sort buffers (F ints each; cells is no longer needed once k_sorted_faces has run)
    int *flag = idx, *id_cur = order, *id_prev = (int *)keys, *start_cur = (int *)keys2, *start_prev = (int *)cells;
    for (int k = 0; k <= kL; ++k) {
        k_level_flags<<<nw_grid(F, B), B, 0, s>>>(h->fkeys, F, 30 - 3 * k, flag);
        NW_LAUNCH_CHECK();
        NW_CHECK(scan_inclusive(h, flag, id_cur, F));
        k_level_tables<<<nw_grid(F, B), B, 0, s>>>(h->fkeys, F, k - 1, k ? tl.off[k - 1] : 0, id_prev, start_prev, tl.off[k], id_cur,
                                                   start_cur, h->parent_g, h->kids, h->boxes, h->leaf_of_slot);
        NW_LAUNCH_CHECK();
        std::swap(id_cur, id_prev);
        std::swap(start_cur, start_prev);
    }
    k_level_tables<<<nw_grid(F, B), B, 0, s>>>(h->fkeys, F, kL, tl.off[kL], id_prev, start_prev, 0, nullptr, nullptr, h->parent_g,
                                               h->kids, h->boxes, h->leaf_of_slot);
    NW_LAUNCH_CHECK();
    // ---- frames (fixed for the block), then the first extents
    launch_refit_centroids(h);
    NW_LAUNCH_CHECK();
    NW_CUDA(cudaMemsetAsync(h->node_f, 0, sizeof(float) * NW_NMOM * total, s));
    k_leaf_normals<<<nw_grid(F, B), B, 0, s>>>(h->sfaces, h->posq, F, h->leaf_of_slot, tl.off[kL], h->node_f);
    NW_LAUNCH_CHECK();
    for (int k = kL - 1; k >= 0; --k) {
        k_up_normals<<<nw_grid(tl.count[k], B), B, 0, s>>>(h->node_f, h->kids, tl.off[k], tl.count[k]);
        NW_LAUNCH_CHECK();
    }
    k_node_frames<<<nw_grid(total, B), B, 0, s>>>(h->boxes, h->node_f, 0, total);
    NW_LAUNCH_CHECK();
    NW_CHECK(extents_pass(h));
    return NW_OK;
}

// ---- a raw point set as the search target (quality metrics, hole-punch candidate search) -----------------------------
namespace {
template <typename T>
__global__ void k_targets_unpack(const T *__restrict__ xyz, int N, float4 *__restrict__ posq, int *__restrict__ faces) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    posq[i] = make_float4((float)xyz[3 * (size_t)i], (float)xyz[3 * (size_t)i + 1], (float)xyz[3 * (size_t)i + 2], 0.f);
    faces[3 * (size_t)i] = faces[3 * (size_t)i + 1] = faces[3 * (size_t)i + 2] = i;
}
// float64 targets in sorted-slot order, for the exact distance evaluation (the float32 copies only prune)
__global__ void k_targets_sorted64(const double *__restrict__ xyz, const int4 *__restrict__ sfaces, int N, double *__restrict__ cent64) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= N) return;
    const size_t i = (size_t)sfaces[s].w;
    cent64[3 * (size_t)s] = xyz[3 * i]; cent64[3 * (size_t)s + 1] = xyz[3 * i + 1]; cent64[3 * (size_t)s + 2] = xyz[3 * i + 2];
}
}  // namespace

// The search hierarchy over N arbitrary points instead of face centroids: what scipy.spatial.cKDTree(points) is to the
// reference's quality metrics (evaluation_utils.py:172-180) and hole-punch candidate search (_membrane_mesh.pyx:882-883).
// Queries go through nw_set_points + nw_compute_weights + nw_get_weights(dist, face): `face` is then the index of the
// nearest target point and `dist` its float64 distance, exactly as cKDTree.query(k=1) returns them (float64 targets are
// compared in float64; their float32 roundings only prune).
extern "C" int nw_set_point_targets(nw_ctx *h, const void *xyz, int is_f64, int64_t N) {
    if (!h) return NW_ERR_ARG;
    NW_ARG(xyz && N > 0 && N < 2147483647LL / 3, "nw_set_point_targets: need 1 <= N < 2^31 / 3 points");
    NW_ARG(h->nranks == 1, "nw_set_point_targets: single-rank handles only");
    NW_CUDA(cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    const int n = (int)N, B = 256;
    h->M = n; h->F = n;
    h->epoch++;
    h->topo_gen++;
    h->weights_valid = false; h->pin_fresh = false; h->feet_valid = false;
    h->points_mode = true;
    NW_CHECK(nw_alloc(h, &h->posq, (size_t)n)); NW_CHECK(nw_alloc(h, &h->nrmq, (size_t)n));
    NW_CHECK(nw_alloc(h, &h->faces, (size_t)3 * n));
    NW_CHECK(nw_alloc(h, &h->nbrT, (size_t)NW_NEIGHBORSIZE * n)); NW_CHECK(nw_alloc(h, &h->valence, (size_t)n));
    NW_CHECK(nw_alloc(h, &h->valid, (size_t)n));
    NW_CHECK(nw_alloc(h, &h->acc, (size_t)4 * n)); NW_CHECK(nw_alloc(h, &h->Sq, (size_t)3 * n));
    NW_CHECK(nw_alloc(h, &h->fdef, (size_t)3 * n)); NW_CHECK(nw_alloc(h, &h->scratchM, (size_t)3 * n));
    NW_CHECK(nw_alloc(h, &h->sfaces, (size_t)n)); NW_CHECK(nw_alloc(h, &h->cent, (size_t)n));
    const size_t raw = (is_f64 ? 8 : 4) * 3 * (size_t)n;
    NW_CHECK(nw_alloc(h, &h->sp_pts, raw));                      // staging shared with nw_set_points (queries come later)
    NW_CHECK(nw_h2d(h, h->sp_pts, xyz, raw));
    if (is_f64) k_targets_unpack<double><<<nw_grid(n, B), B, 0, s>>>((const double *)h->sp_pts, n, h->posq, h->faces);
    else k_targets_unpack<float><<<nw_grid(n, B), B, 0, s>>>((const float *)h->sp_pts, n, h->posq, h->faces);
    NW_LAUNCH_CHECK();
    NW_CUDA(cudaMemsetAsync(h->nrmq, 0, sizeof(float4) * n, s));
    NW_CUDA(cudaMemsetAsync(h->valence, 0, sizeof(int) * n, s));
    NW_CUDA(cudaMemsetAsync(h->valid, 1, n, s));
    NW_CUDA(cudaMemsetAsync(h->acc, 0, sizeof(unsigned long long) * 4 * n, s));
    NW_CUDA(cudaMemsetAsync(h->Sq, 0, sizeof(float4) * 3 * n, s));
    if (h->slot && h->P) NW_CUDA(cudaMemsetAsync(h->slot, 0xff, sizeof(int) * h->P, s));
    h->seeds_cold = true;
    h->order_stale = true;
    NW_CHECK(nw_tree_build(h));
    if (is_f64) {
        NW_CHECK(nw_alloc(h, &h->cent64, (size_t)3 * n));
        k_targets_sorted64<<<nw_grid(n, B), B, 0, s>>>((const double *)h->sp_pts, h->sfaces, n, h->cent64);
        NW_LAUNCH_CHECK();
    } else nw_free(&h->cent64);
    NW_CUDA(cudaStreamSynchronize(s));
    return NW_OK;
}

extern "C" int nw_set_positions(nw_ctx *h, const float *pos) {
    if (!h) return NW_ERR_ARG;
    NW_ARG(h->M > 0, "nw_set_positions: no topology");
    NW_CUDA(cudaSetDevice(h->device));
    NW_CUDA(cudaMemcpyAsync(h->scratchM, pos, sizeof(float) * 3 * h->M, cudaMemcpyHostToDevice, h->stream));
    k_pack_vec3<<<nw_grid(h->M, 256), 256, 0, h->stream>>>(h->scratchM, h->M, h->posq);
    NW_LAUNCH_CHECK();
    NW_CUDA(cudaStreamSynchronize(h->stream));
    h->weights_valid = false;
    h->pin_fresh = false;
    return NW_OK;
}

// Current positions (and the valid flags) into the handle's pinned staging buffer.  nw_search enqueues this behind its last
// iteration, so the two getters below usually find the copy already there (pin_fresh) and only do host work.
int nw_fetch_positions_async(nw_ctx *h) {
    const size_t M = (size_t)h->M, need = M * 12 + M;
    if (h->pin_bytes < need) {
        if (h->pin_host) cudaFreeHost(h->pin_host);
        h->pin_host = nullptr; h->pin_bytes = 0;
        NW_CUDA(cudaHostAlloc((void **)&h->pin_host, need + need / 4, cudaHostAllocDefault));
        h->pin_bytes = need + need / 4;
    }
    k_unpack_vec3<<<nw_grid(h->M, 256), 256, 0, h->stream>>>(h->posq, h->M, h->scratchM);
    NW_LAUNCH_CHECK();
    NW_CUDA(cudaMemcpyAsync(h->pin_host, h->scratchM, M * 12, cudaMemcpyDeviceToHost, h->stream));
    NW_CUDA(cudaMemcpyAsync(h->pin_host + M * 12, h->valid, M, cudaMemcpyDeviceToHost, h->stream));
    return NW_OK;
}
static int positions_on_host(nw_ctx *h) {
    if (h->pin_fresh) return NW_OK;
    NW_CHECK(nw_fetch_positions_async(h));
    NW_CUDA(cudaStreamSynchronize(h->stream));
    h->pin_fresh = true;
    return NW_OK;
}

// f written straight into the host mesh's records: position of vertex i (3 x float32) at dst + i * stride_bytes; with
// only_valid rows whose halfedge is -1 keep their bytes (mesh_conj_grad.py:289 without a strided numpy assignment)
extern "C" int nw_get_positions_strided(nw_ctx *h, void *dst, int stride_bytes, int only_valid) {
    if (!h) return NW_ERR_ARG;
    NW_ARG(h->M > 0, "nw_get_positions_strided: no topology");
    NW_ARG(dst && stride_bytes >= 12, "nw_get_positions_strided: bad destination");
    NW_CUDA(cudaSetDevice(h->device));
    NW_CHECK(positions_on_host(h));
    const size_t M = (size_t)h->M;
    const char *src = h->pin_host;
    const unsigned char *ok = (const unsigned char *)h->pin_host + M * 12;
    char *d = (char *)dst;
    // every row is its own cache line of the destination: latency bound on one thread (5 ms for 0.5 M rows), so split it
    auto rows = [=](size_t a, size_t b) {
        for (size_t i = a; i < b; ++i)
            if (!only_valid || ok[i]) memcpy(d + i * (size_t)stride_bytes, src + i * 12, 12);
    };
    const size_t nt = M < 65536 ? 1 : std::min<size_t>(8, std::max(1u, std::thread::hardware_concurrency() / 2));
    std::vector<std::thread> th;
    for (size_t t = 1; t < nt; ++t) th.emplace_back(rows, M * t / nt, M * (t + 1) / nt);
    rows(0, M / nt);
    for (auto &t : th) t.join();
    return NW_OK;
}

extern "C" int nw_get_positions(nw_ctx *h, float *pos) {
    if (!h) return NW_ERR_ARG;
    NW_ARG(h->M > 0, "nw_get_positions: no topology");
    NW_CUDA(cudaSetDevice(h->device));
    NW_CHECK(positions_on_host(h));
    memcpy(pos, h->pin_host, (size_t)h->M * 12);
    return NW_OK;
}

/* nanowrap.h -- C ABI of libnanowrap.so, the B200 (sm_100a) implementation of ch_shrinkwrap's
 * NanoWrap conjugate-gradient shrinkwrap hot path.
 *
 * Plain C: opaque handle, caller-owned host buffers, int return codes (0 = ok), no torch / numpy
 * types.  One caller per handle; two handles may live in one process.  Every entry point names the
 * reference interface it replaces (paths relative to the reference repository, file:line).
 *
 * Host arrays use the reference's layouts: vectors over vertices are raveled C-order
 * [v0x,v0y,v0z,v1x,...] (mesh_conj_grad.py:594-595), per-point arrays are (P,3) row-major in the
 * CALLER'S point order (the library keeps its own Hilbert-sorted copy internally).
 */
#ifndef NANOWRAP_H_
#define NANOWRAP_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NW_NEIGHBORSIZE 20 /* membrane_mesh_utils.h:29 */

/* return codes */
#define NW_OK 0
#define NW_ERR_CUDA 1      /* CUDA runtime / launch failure (nw_last_error has the text)        */
#define NW_ERR_ARG 2       /* bad argument / call order  -> RuntimeError / ValueError in the shim */
#define NW_ERR_NAN 3       /* non-finite value detected  -> AssertionError in the shim; mirrors
                              the reference's `assert(not np.any(np.isnan(...)))`, mesh_conj_grad.py:514,548,580 */
#define NW_ERR_COMM 4      /* NCCL failure or libnccl.so.2 not loadable                           */

typedef struct nw_ctx nw_ctx;

/* ---- lifetime ------------------------------------------------------------------------------- */
int nw_version(void);
/* One handle = one GPU, one stream.  Replaces the per-block object construction at
 * _membrane_mesh.pyx:1510 (ShrinkwrapMeshConjGrad.__init__, mesh_conj_grad.py:33-65). */
int nw_create(int device, nw_ctx **out);
void nw_destroy(nw_ctx *h);
const char *nw_last_error(nw_ctx *h);

/* ---- multi-GPU: points sharded, mesh replicated (SURVEY 8e); one process per GPU -------------- */
int nw_comm_unique_id(char id[128]);                         /* rank 0 calls, bytes are broadcast by the host */
int nw_comm_init(nw_ctx *h, int rank, int nranks, const char id[128]);

/* ---- points: once per fit --------------------------------------------------------------------
 * Replaces the `points` setter and the sigma / weights preparation:
 * mesh_conj_grad.py:127-130,156-164 and _membrane_mesh.pyx:1460-1473.
 *  pts            (P,3) float32 (pts_is_f64 = 0) or float64 (= 1); with float64 input the nearest-
 *                 face search runs on the float64 values, everything else on their float32 rounding.
 *  sigma_inv      (P,3) float32 or NULL -> sigma_inv_scalar is used (note the reference passes a
 *                 scalar sigma through un-inverted, _membrane_mesh.pyx:1460-1461).
 *  weights        (P,3) float32 or NULL.  NULL: weights = sigma_inv (mesh_conj_grad.py:156-158).
 *                 Array weights are normalised by their mean over ALL ranks' points (:162) and define
 *                 mask = weights > 0 (:161); a scalar weight is used as is (weights_scalar, used when
 *                 weights == NULL and sigma_inv == NULL).
 *  P              points in this rank's shard. */
int nw_set_points(nw_ctx *h, const void *pts, int pts_is_f64, int64_t P, const float *sigma_inv,
                  float sigma_inv_scalar, const float *weights);

/* ---- topology: once per remesh block ------------------------------------------------------------
 * Replaces the attribute caching in ShrinkwrapMeshConjGrad.__init__ (mesh_conj_grad.py:44-54) and the
 * live reads in _ncc (:777-816).
 *  pos, nrm  (M,3) float32: mesh._vertices['position'], mesh.vertex_normals (normals are per block)
 *  faces     (F,3) int32  : mesh.faces; nearest-face results index its rows (:488)
 *  nbr       (M,20) int32 : neighbour VERTEX ids, -1 terminated (:50-54)
 *  valid     (M) uint8 or NULL: mesh._vertices['halfedge'] != -1 (:44); NULL = all valid
 * With a communicator of more than one rank (nw_comm_init) the three nw_set_topology* calls are COLLECTIVE: every rank
 * calls with the same mesh, rank 0's arrays are uploaded and broadcast to the others (ncclBroadcast), and a rank whose
 * M, F, half-edge count or optional-array pattern differs from rank 0's gets NW_ERR_ARG. */
int nw_set_topology(nw_ctx *h, const float *pos, const float *nrm, const int32_t *faces,
                    const int32_t *nbr, const uint8_t *valid, int M, int F);
/* Same, but the neighbour table holds HALF-EDGE indices exactly as mesh._vertices['neighbors'] stores them and
 * he_vertex = mesh._halfedges['vertex'] (n_halfedges int32); the library performs the lookup of
 * mesh_conj_grad.py:50-52 on the device instead of a 20M-element numpy gather per block on the host. */
int nw_set_topology_halfedge(nw_ctx *h, const float *pos, const float *nrm, const int32_t *faces,
                             const int32_t *nbr_halfedge, const int32_t *he_vertex, int n_halfedges,
                             const uint8_t *valid, int M, int F);
/* Same from the raw records: vertex_records = mesh._vertices as it lies in memory (M x vertex_t, 120 B each,
 * membrane_mesh_utils.h:57-65: position, normal, halfedge, valence, neighbors[20], component, locally_manifold).
 * One contiguous upload, no host-side packing; position / normal / valid / neighbours are unpacked on the device.
 * he_vertex points at the first 'vertex' entry and he_stride_bytes is the distance between entries: 4 for a packed
 * int32 array, 28 (halfedge_t, membrane_mesh_utils.h:31-39) when it points into mesh._halfedges as it lies in memory. */
int nw_set_topology_records(nw_ctx *h, const void *vertex_records, const int32_t *faces, const int32_t *he_vertex,
                            int he_stride_bytes, int n_halfedges, int M, int F);
int nw_set_positions(nw_ctx *h, const float *pos);           /* overwrite f (3M) */
int nw_get_positions(nw_ctx *h, float *pos);                 /* read f (3M)      */
/* f written straight into the host mesh: vertex i's (x, y, z) float32 at dst + i * stride_bytes (dst =
 * &mesh._vertices['position'][0], stride 120 for vertex_t records); only_valid != 0 leaves the rows with
 * halfedge == -1 untouched: mesh._vertices['position'][mask] = f[mask] (mesh_conj_grad.py:289) */
int nw_get_positions_strided(nw_ctx *h, void *dst, int stride_bytes, int only_valid);

/* ---- the hot loop -------------------------------------------------------------------------------
 * Replaces ShrinkwrapMeshConjGrad.search (mesh_conj_grad.py:150-292) with Lfuncs = ["I"]
 * (:38), i.e. one regulariser lam^2 |f - ncc(f)|^2, plus subsearch (conj_grad.py:183-229).
 *  prev_tests/n_prev : tail (<=3) of the caller's `tests` history for the stop rule (:1009-1016)
 *  pos_out (3M)      : f after the last iteration (what search() returns)
 *  tests, ress, prefs, cpred, wpred : per-iteration histories (:269-274), num_iters doubles each
 *  n_done            : iterations actually run (stop rule may end early) */
int nw_search(nw_ctx *h, float lam, int num_iters, int last_step, const double *prev_tests,
              int n_prev, float *pos_out, double *tests, double *ress, double *prefs,
              double *cpred, double *wpred, int *n_done);

/* Regulariser of the next nw_search calls: the reference reads Lfuncs / Lhfuncs from the solver object
 * (mesh_conj_grad.py:36-39,257-258; conj_grad.py:191-200).  mode 0 = ["I"], ["I"] (its setting); mode 1 = ["wfunc"],
 * ["wfunc"] (:39, :725-736).  The remaining 1-ring operators below cannot regularise a fit in the reference either (its
 * search() passes them a float64 array that the C helpers read as float32), so they stay stand-alone operators. */
int nw_set_regulariser(nw_ctx *h, int mode);

/* ---- operators (the reference's public methods on the solver object) --------------------------- */
/* nearest face + weights at the current f: _compute_weight_matrix4, mesh_conj_grad.py:433-516 */
int nw_compute_weights(nw_ctx *h);
/* read back (any pointer may be NULL): v_idx (P,3) int32, w (P,3) float32, dist (P) float64 = dmean
 * (self.d is dmean repeated x3, :483), face (P) int32 = row of mesh.faces */
int nw_get_weights(nw_ctx *h, int32_t *v_idx, float *w, double *dist, int32_t *face);
/* Afunc, mesh_conj_grad.py:518-551: y(3P) = A x(3M) with the current weights */
int nw_apply_A(nw_ctx *h, const float *x, float *y);
/* Ahfunc, mesh_conj_grad.py:553-588 -> conj_grad_utils.c:123-167: y(3M) = AH r(3P) */
int nw_apply_AH(nw_ctx *h, const float *r, float *y);
/* point_influence, _membrane_mesh.pyx:1625-1634: |AH 1| per vertex (M) */
int nw_point_influence(nw_ctx *h, float *pi);
/* _ncc, mesh_conj_grad.py:770-820: f_def (M,3) float64 at the current f and weights */
int nw_ncc(nw_ctx *h, double *fdef);
/* residual of the last iteration (3P), search directions S (3M,3) row-major as self.S (:286) */
int nw_get_res(nw_ctx *h, float *res);
int nw_get_S(nw_ctx *h, float *S);

/* ---- secondary 1-ring regularisers (selectable Lfuncs, mesh_conj_grad.py:590-736) ------------------
 * Same semantics as conj_grad_utils.c: out (3M) is ACCUMULATED INTO (in place +=), f and ref are 3M.
 * Use the neighbour table given to nw_set_topology. */
int nw_l_func(nw_ctx *h, const float *f, float *out);                      /* conj_grad_utils.c:249-306 */
int nw_lh_func(nw_ctx *h, const float *f, float *out);                     /* :308-368 */
int nw_lw_func(nw_ctx *h, const float *f, const float *ref, float *out);   /* :370-497 */
int nw_lhw_func(nw_ctx *h, const float *f, const float *ref, float *out);  /* :585-710 */
int nw_vertex_area_weights(nw_ctx *h, const float *ref, float *out);       /* :500-582 */

/* ---- curvature ------------------------------------------------------------------------------------
 * Replaces c_curvature_grad (membrane_mesh_utils.c:915-1250; Cython binding _membrane_mesh.pyx:50-70,
 * 323-347).  Same buffer list and record layouts (membrane_mesh_utils.h:31-65: vertex_t 120 B,
 * face_t 24 B, halfedge_t 28 B); the array lengths are added because the buffers are copied to the GPU.
 * Outputs are overwritten in place; rows of deleted vertices follow membrane_mesh_utils.c:962-973.
 *  jitter_u : the uniform [0,1) draws the reference takes from rand() (3 per valid vertex, in vertex
 *             order, :1017).  NULL -> the library draws them from a counter-based generator seeded with
 *             jitter_seed (the reference's rand() stream is not reproducible either, SURVEY B.11).
 * skip_prob (Monte-Carlo vertex skipping, :962) must be 0 -- the only value the reference passes. */
int nw_curvature_grad(nw_ctx *h, const void *vertices, const void *faces, const void *halfedges,
                      int n_vertices, int n_faces, int n_halfedges, float dN, float skip_prob,
                      float *k_0, float *k_1, float *e_0, float *e_1, float *H, float *K, float *dH,
                      float *dK, float *E, float *pE, float *dE_neighbors, float kc, float kg,
                      float c0, float *dEdN, const double *jitter_u, uint64_t jitter_seed);
/* neck criterion, _membrane_mesh.pyx:1212-1213: indices with K < low or K > high from the last
 * nw_curvature_grad call; returns the count in *n (idx may be NULL to query the count) */
int nw_neck_candidates(nw_ctx *h, float low, float high, int32_t *idx, int *n);

/* ---- either side of the solver (SURVEY 8f): quality metrics and the hole-punch candidate search ---------
 * A raw point set as the search target, replacing scipy.spatial.cKDTree(points) at evaluation_utils.py:172-173
 * (average_squared_distance) and _membrane_mesh.pyx:882 (_holepunch_find_candidate_faces).  xyz: (N,3) float32
 * (is_f64 = 0) or float64 (= 1).  Afterwards nw_set_points(queries) + nw_compute_weights + nw_get_weights(NULL,
 * NULL, dist, face) give, per query, the float64 distance to and the index of its nearest target point exactly as
 * cKDTree.query(k=1) does (float64 compare; ties -> lowest index).  Replaces any topology set on the handle. */
int nw_set_point_targets(nw_ctx *h, const void *xyz, int is_f64, int64_t N);
/* points_from_mesh, evaluation_utils.py:35-145: every triangle sampled on a dx_min grid in its own plane.  pos (M,3)
 * float32 = mesh._vertices['position'], faces (F,3) int32 = mesh.faces.  Call with out = NULL to get the number of
 * samples in *n_out, then with out (n,3) float64 and capacity >= n.  Samples come in the reference's generation order
 * and are bit-identical to its `d` array; the random permutation / subsampling of :137 stays with the caller. */
int nw_points_from_mesh(nw_ctx *h, const float *pos, const int32_t *faces, int M, int F, double dx_min, double *out,
                        int64_t capacity, int64_t *n_out);
/* c_holepunch_pair_candidate_faces, membrane_mesh_utils.c:1301-1379 (binding _membrane_mesh.pyx:890-896): same
 * arguments plus the array lengths; pairs[i] = index into candidates of the opposing face nearest to candidates[i] in
 * the mean-normal plane, or -1.  pairs is overwritten (the reference expects it initialised to -1 by the caller). */
int nw_holepunch_pair_candidate_faces(nw_ctx *h, const void *vertices, const void *faces, const void *halfedges,
                                      int n_vertices, int n_faces, int n_halfedges, const int32_t *candidates,
                                      int n_candidates, int32_t *pairs);

/* ---- exact point-to-surface distance (not part of the reference surface) ---------------------------------------
 * Exact distance from each query to the handle's current triangle mesh (the topology of the last nw_set_topology*, at the
 * current f -- after nw_search, the fitted surface).  q == NULL: the handle's own points (this rank's shard, caller order of
 * nw_set_points; Q must equal their number).  Otherwise q is (Q,3) float32 (q_is_f64 = 0) or float64 (= 1).  Per query, in
 * the caller's order: dist (Q) float64 Euclidean distance to the nearest closed triangle, face (Q) int32 its row of
 * mesh.faces (exact fp64 ties -> lowest row), closest (Q,3) float64 the closest point on it.  summary = {max, mean, RMS} of
 * dist from a fixed-order reduction on the device (bit-identical from call to call).  Faces with a non-finite corner are
 * skipped; a non-finite query gets dist = NaN, face = -1 and is left out of summary.  Any output may be NULL.  Changes
 * nothing that nw_search reads.  NW_ERR_ARG in points mode (nw_set_point_targets).  No collectives: each rank of a
 * multi-rank handle measures its own shard. */
int nw_surface_distance(nw_ctx *h, const void *q, int q_is_f64, int64_t Q, double *dist, int32_t *face, double *closest,
                        double summary[3]);
/* Signed distance to a closed mesh: the nearest-triangle search of nw_surface_distance (same queries, same face and closest,
 * |sdist| = its dist), with sdist < 0 inside and > 0 outside.  The side is that of q - closest against the angle-weighted
 * pseudonormal (Baerentzen & Aanaes 2005) of the feature the closest point lies on (face interior, edge, or vertex), times
 * the sign of the mesh's signed volume, so it does not depend on the winding.  sdist = 0 on the surface; NaN where the side
 * is undecidable (q - closest orthogonal to the pseudonormal) and for a non-finite query (face = -1).  volume = the enclosed
 * volume |V| (fixed-order fp64 reduction).  The mesh must be closed, edge-manifold and consistently oriented (every edge on
 * exactly two faces that traverse it in opposite directions, no face repeating a vertex, one fan of faces per vertex) and
 * enclose a finite, non-zero volume; otherwise NW_ERR_ARG with the defect counts in nw_last_error.  A mesh whose components
 * are oriented against each other is not supported: one global orientation decides inside.  Q == 0 with q != NULL checks
 * the mesh and returns the volume only.  Any output may be NULL.  NW_ERR_ARG in points mode; no collectives. */
int nw_surface_signed_distance(nw_ctx *h, const void *q, int q_is_f64, int64_t Q, double *sdist, int32_t *face,
                               double *closest, double *volume);
/* Self-intersections of the handle's current mesh (the topology of the last nw_set_topology*, at the current f -- after
 * nw_search, the fitted surface).  Faces f < g (rows of mesh.faces) are reported when their closed triangles share a point
 * that their shared vertex indices do not explain: with none shared, any common point (touching counts); with one shared
 * vertex s, the edge of either face opposite s meets the other closed face; with a shared edge, the opposite corners are
 * coplanar with it and strictly on the same side (a fold-over); with three, always.  Degenerate faces (exactly collinear
 * corners, a repeated vertex included) and faces with a non-finite corner are not tested.  Exact (every decision is the sign
 * of orient3d / orient2d of the float32 positions), sorted by (f, g), independent of scheduling.  *n_pairs = the number of
 * pairs; the first min(n, capacity) go to pairs (capacity x 2 int32); pairs may be NULL with capacity 0 (count only).
 * stats (or NULL) = {candidate pairs that passed the box test, predicate evaluations the fp64 filter left to the exact
 * stage, degenerate faces, faces with a non-finite corner}.  The signed distance and the enclosed volume assume no such
 * pair.  Changes nothing that nw_search reads.  NW_ERR_ARG in points mode or without a topology; no collectives. */
int nw_self_intersections(nw_ctx *h, int32_t *pairs, int64_t capacity, int64_t *n_pairs, int64_t stats[4]);

/* ---- measurement hooks (bench.py / profiling; not part of the reference surface) ------------------ */
/* device-resident single-kernel launches on the handle's stream, for CUDA-event timing */
int nw_bench_kernel(nw_ctx *h, const char *name, int reps, float *ms_per_launch);
/* forget every nearest-face seed (the previous sweep's faces and the foot points kept across topology uploads), so that the
 * next sweep starts cold like the first sweep of a fit; results never depend on the seeds, only the time does */
int nw_reset_seeds(nw_ctx *h);
int nw_sync(nw_ctx *h);
/* CUDA-event timing on the handle's stream: on & 1 brackets every stage of every iteration inside
 * nw_search and the device-side segments of nw_set_topology*.  nw_get_profile returns accumulated ms and kernel
 * launches per stage (11 stages: refit, shift, sweep1, allreduce_acc, mesh_prior, sweep2, allreduce_scalars,
 * solve_update, seed_leaders, topology_build = foot points + record unpack + Hilbert sort + octree tables + frames of
 * every upload, host->device copies excluded, adjoint; the arrays must hold 16 entries) and the event-timed duration of
 * the last nw_search call (first kernel to last kernel).  on & 2: traversal statistics (below).  on & 4: an NVTX range
 * named after the stage around every stage of nw_search (for ncu --nvtx / nsys; no-ops without an attached tool). */
int nw_set_profile(nw_ctx *h, int on);
int nw_get_profile(nw_ctx *h, double *stage_ms, int64_t *stage_launches, double *search_ms);
/* the stage intervals of the last profiled nw_search call in launch order: stage[k] (index into the list above), ms[k];
 * at most cap entries are written, *n = how many there are */
int nw_get_stage_trace(nw_ctx *h, int32_t *stage, float *ms, int cap, int *n);
/* nearest-face traversal statistics (collected only while nw_set_profile(h, on) has on & 2; the counting variant of the
 * kernel is slower) accumulated since the last nw_search / nw_ncc / nw_bench_kernel state reset:
 * node bound tests, leaf visits, exact fp64 distance evaluations, largest node-test count of a single point */
int nw_get_traversal_stats(nw_ctx *h, uint64_t out[4]);
/* diagnosis: boxes of one level of the centroid pyramid (16 floats per node, layout of csrc/common.cuh: Box) */
int nw_debug_tree(nw_ctx *h, int level, float *boxes16, int *counts, int *n_levels);
/* kernels launched by this handle since creation (for bench.py's gpu_launches) */
int64_t nw_launch_count(nw_ctx *h);

#ifdef __cplusplus
}
#endif
#endif /* NANOWRAP_H_ */

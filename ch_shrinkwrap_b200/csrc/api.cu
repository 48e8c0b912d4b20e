// api.cu -- handle lifetime and the search() driver: all kernels of all iterations are enqueued on
// one stream without host round trips; the stop rule, NaN guard and histories live on the device and
// are read back once at the end (the reference's loop is mesh_conj_grad.py:218-290).
#include <nvtx3/nvToolsExt.h>
#include <cmath>
#include <cstring>
#include "common.cuh"

int nw_launch_solve_update(nw_ctx *h, int iter_index, int last_step);
int nw_launch_influence(nw_ctx *h);

extern "C" int nw_version(void) { return 100; }

extern "C" int nw_create(int device, nw_ctx **out) {
    if (!out) return NW_ERR_ARG;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || device < 0 || device >= n) return NW_ERR_CUDA;
    nw_ctx *h = new nw_ctx();
    h->device = device;
    if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess) {
        delete h;
        return NW_ERR_CUDA;
    }
    if (cudaMalloc((void **)&h->st, sizeof(SolverState)) != cudaSuccess ||
        cudaMalloc((void **)&h->hist, sizeof(double) * 5 * NW_MAX_ITERS) != cudaSuccess) {
        delete h;
        return NW_ERR_CUDA;
    }
    cudaMemset(h->st, 0, sizeof(SolverState));
    h->tl.n_levels = 0;
    *out = h;
    return NW_OK;
}

int nw_comm_destroy(nw_ctx *h);

extern "C" void nw_destroy(nw_ctx *h) {
    if (!h) return;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    if (h->iter_graph) { cudaGraphExecDestroy(h->iter_graph); h->iter_graph = nullptr; }
    nw_comm_destroy(h);
    nw_free(&h->px); nw_free(&h->py); nw_free(&h->pz);
    nw_free(&h->px64); nw_free(&h->py64); nw_free(&h->pz64);
    nw_free(&h->sx); nw_free(&h->sy); nw_free(&h->sz);
    nw_free(&h->wx); nw_free(&h->wy); nw_free(&h->wz);
    nw_free(&h->pmask); nw_free(&h->perm); nw_free(&h->slot); nw_free(&h->fx); nw_free(&h->fy); nw_free(&h->fz); nw_free(&h->fkeys); nw_free(&h->fkey_tab);
    nw_free(&h->w0); nw_free(&h->w1); nw_free(&h->w2);
    nw_free(&h->rx); nw_free(&h->ry); nw_free(&h->rz);
    nw_free(&h->posq); nw_free(&h->nrmq); nw_free(&h->faces); nw_free(&h->nbrT); nw_free(&h->valence); nw_free(&h->valid); nw_free(&h->stage_nbr); nw_free(&h->stage_hev); nw_free(&h->tb_small); nw_free(&h->tb_i0); nw_free(&h->tb_i1); nw_free(&h->tb_u0); nw_free(&h->tb_u1); nw_free(&h->tb_u2); nw_free(&h->fcells); nw_free(&h->cent64); nw_free(&h->parent_g); nw_free(&h->kids);
    nw_free(&h->sfaces); nw_free(&h->cent); nw_free(&h->boxes); nw_free(&h->leaf_of_slot); nw_free(&h->node_f);
    nw_free(&h->tboxes); nw_free(&h->surf_q); nw_free(&h->surf_bits); nw_free(&h->surf_dist); nw_free(&h->surf_closest);
    nw_free(&h->surf_part); nw_free(&h->surf_face);
    nw_free(&h->sgn_twin); nw_free(&h->sgn_voff); nw_free(&h->sgn_vface); nw_free(&h->sgn_k0); nw_free(&h->sgn_k1);
    nw_free(&h->sgn_i0); nw_free(&h->sgn_i1); nw_free(&h->sgn_cnt); nw_free(&h->sgn_nv); nw_free(&h->sgn_vpart); nw_free(&h->sgn_bbox);
    nw_free(&h->sx_flag); nw_free(&h->sx_last); nw_free(&h->sx_keys); nw_free(&h->sx_sorted); nw_free(&h->sx_cnt); nw_free(&h->sx_pairs);
    nw_free(&h->hb_pos); nw_free(&h->hb_faces); nw_free(&h->hb_vface); nw_free(&h->hb_flag); nw_free(&h->hb_idx); nw_free(&h->hb_slot);
    nw_free(&h->hb_ent[0]); nw_free(&h->hb_ent[1]); nw_free(&h->hb_q); nw_free(&h->hb_qd); nw_free(&h->hb_qf); nw_free(&h->hb_qs);
    nw_free(&h->hb_qa); nw_free(&h->hb_st);
    nw_free(&h->mb_area); nw_free(&h->mb_val); nw_free(&h->mb_part); nw_free(&h->mb_st);
    nw_free(&h->acc); nw_free(&h->Sq); nw_free(&h->fdef);
    nw_free(&h->partials); nw_free(&h->st); nw_free(&h->hist);
    nw_free((char **)&h->cub_tmp); nw_free(&h->scratchM); nw_free(&h->scratchP);
    nw_free((char **)&h->cvV); nw_free((char **)&h->cvF); nw_free((char **)&h->cvH); nw_free(&h->cvOut); nw_free(&h->cvJ); nw_free(&h->cvOff);
    nw_free(&h->sp_pts); nw_free(&h->sp_k0); nw_free(&h->sp_k1); nw_free(&h->sp_idx); nw_free(&h->sp_tmp3);
    nw_free(&h->blk_order); nw_free(&h->blk_order_cold); nw_free(&h->blk_idx); nw_free(&h->blk_key); nw_free(&h->blk_key2);
    nw_uploader_destroy(h);
    if (h->pin_host) cudaFreeHost(h->pin_host);
    for (cudaEvent_t e : h->ev_pool) cudaEventDestroy(e);
    if (h->ev_search0) { cudaEventDestroy(h->ev_search0); cudaEventDestroy(h->ev_search1); }
    if (h->ev_seg0) { cudaEventDestroy(h->ev_seg0); cudaEventDestroy(h->ev_seg1); }
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
}

extern "C" const char *nw_last_error(nw_ctx *h) { return h ? h->err.c_str() : "null handle"; }
extern "C" int64_t nw_launch_count(nw_ctx *h) { return h ? h->launches : 0; }
extern "C" int nw_sync(nw_ctx *h) {
    if (!h) return NW_ERR_ARG;
    NW_CUDA(cudaSetDevice(h->device));
    NW_CUDA(cudaStreamSynchronize(h->stream));
    return NW_OK;
}

static int ensure_partials(nw_ctx *h) {
    // layout: [sweep2 partials: n_partials x 16] [mesh partials: ceil(M/256) x 16] [64 doubles of comm staging]
    const int want = std::max(1, nw_grid(h->P, 256 * NW_S2_PTS));
    const size_t need = (size_t)want * 16 + (size_t)nw_grid(h->M, 256) * 16 + 64;
    NW_CHECK(nw_alloc(h, &h->partials, need));
    h->n_partials = want;
    return NW_OK;
}

static int upload_state(nw_ctx *h, const SolverState &s0) {
    SolverState s = s0;
    for (int a = 0; a < 3; ++a) { s.bbox[a] = 0x7fffffff; s.bbox[3 + a] = (int)0x80000000; }
    NW_CUDA(cudaMemcpyAsync(h->st, &s, sizeof(SolverState), cudaMemcpyHostToDevice, h->stream));
    return NW_OK;
}

// per-stage NVTX ranges (profile bit 4: `ncu --nvtx --nvtx-include "sweep1/"` then selects a stage; without an attached tool
// the header-only NVTX calls are no-ops) and per-stage CUDA events (profile bit 1)
static const char *const kStageName[NW_N_STAGES] = {"refit", "shift", "sweep1", "allreduce_acc", "mesh_prior", "sweep2",
                                                    "allreduce_scalars", "solve_update", "seed_leaders", "topology_build", "adjoint"};
static int stage_begin(nw_ctx *h, int stage) {
    if (h->profile & 4) nvtxRangePushA(kStageName[stage]);
    if (!(h->profile & 1)) return NW_OK;
    if (h->ev_used + 2 > h->ev_pool.size()) {
        for (int k = 0; k < 64; ++k) { cudaEvent_t e; NW_CUDA(cudaEventCreate(&e)); h->ev_pool.push_back(e); }
    }
    h->ev_stage.push_back(stage);
    NW_CUDA(cudaEventRecord(h->ev_pool[h->ev_used++], h->stream));
    h->stage_launches[stage] -= h->launches;
    return NW_OK;
}
static int stage_end(nw_ctx *h, int stage) {
    if (h->profile & 4) nvtxRangePop();
    if (!(h->profile & 1)) return NW_OK;
    NW_CUDA(cudaEventRecord(h->ev_pool[h->ev_used++], h->stream));
    h->stage_launches[stage] += h->launches;
    return NW_OK;
}
#define NW_STAGE(id, call) do { NW_CHECK(stage_begin(h, id)); NW_CHECK(call); NW_CHECK(stage_end(h, id)); } while (0)

// one full iteration, enqueued asynchronously
static int enqueue_iteration(nw_ctx *h, int it, int last_step) {
    NW_STAGE(1, nw_set_acc_shifts(h));             // vertex bbox -> fixed-point scales, rounding slack of the box tests
    NW_STAGE(0, nw_tree_refit(h));                 // centroids + boxes at the current f  (:443)
    if (h->seeds_cold) NW_STAGE(8, nw_launch_seed_leaders(h));   // first iteration after a topology upload only
    NW_STAGE(2, nw_launch_sweep1(h, true));        // NN, weights, A f, residual  (:222-253)
    NW_STAGE(10, nw_launch_adjoint(h));            // AH res, AH 1: exact fixed-point scatter
    if (h->nranks > 1) NW_STAGE(3, nw_allreduce_acc(h));   // N>1: vertex-gradient allreduce
    NW_STAGE(4, nw_launch_mesh_prior(h, true));    // S0, ncc, prefs, S1, S^T S  (:224,253-258)
    NW_STAGE(5, nw_launch_sweep2(h));              // A S_k and Gram sums  (conj_grad.py:197-203)
    if (h->nranks > 1) NW_STAGE(6, nw_allreduce_scalars(h));   // N>1: CG scalars
    NW_STAGE(7, nw_launch_solve_update(h, it, last_step));
    return NW_OK;
}

// Forget every nearest-face seed (previous sweep's slots and the foot points kept across topology uploads): the next sweep
// starts as the first sweep of a fit does.  For measurements that must include the cold start; results never depend on seeds.
extern "C" int nw_reset_seeds(nw_ctx *h) {
    if (!h) return NW_ERR_ARG;
    NW_CUDA(cudaSetDevice(h->device));
    if (h->slot && h->P) NW_CUDA(cudaMemsetAsync(h->slot, 0xff, sizeof(int) * h->P, h->stream));
    h->seeds_cold = true;
    h->feet_valid = false;
    h->order_stale = true;
    h->weights_valid = false;
    return NW_OK;
}

extern "C" int nw_set_profile(nw_ctx *h, int on) {
    if (!h) return NW_ERR_ARG;
    if (on != h->profile) h->epoch++;            // the traversal-statistics variant of k_sweep1 is a different launch
    h->profile = on;
    for (int k = 0; k < NW_N_STAGES; ++k) { h->stage_ms[k] = 0.0; h->stage_launches[k] = 0; }
    return NW_OK;
}
extern "C" int nw_get_traversal_stats(nw_ctx *h, uint64_t out[4]) {
    if (!h || !out) return NW_ERR_ARG;
    SolverState r;
    NW_CUDA(cudaMemcpy(&r, h->st, sizeof(SolverState), cudaMemcpyDeviceToHost));
    for (int k = 0; k < 4; ++k) out[k] = r.trav[k];
    return NW_OK;
}
// diagnosis: copy the boxes of one tree level (16 floats each) and the level sizes
extern "C" int nw_debug_tree(nw_ctx *h, int level, float *boxes16, int *counts, int *n_levels) {
    if (!h) return NW_ERR_ARG;
    NW_ARG(h->boxes && h->tl.n_levels > 0, "nw_debug_tree: no tree");
    if (n_levels) *n_levels = h->tl.n_levels;
    if (counts) for (int l = 0; l < h->tl.n_levels; ++l) counts[l] = h->tl.count[l];
    if (boxes16 && level >= 0 && level < h->tl.n_levels)
        NW_CUDA(cudaMemcpy(boxes16, h->boxes + h->tl.off[level], sizeof(Box) * h->tl.count[level], cudaMemcpyDeviceToHost));
    return NW_OK;
}
// the stage intervals of the last profiled nw_search call in launch order (stage id, ms); *n = how many there are
extern "C" int nw_get_stage_trace(nw_ctx *h, int32_t *stage, float *ms, int cap, int *n) {
    if (!h || !n) return NW_ERR_ARG;
    *n = (int)h->trace_stage.size();
    for (int k = 0; k < *n && k < cap; ++k) { if (stage) stage[k] = h->trace_stage[k]; if (ms) ms[k] = h->trace_ms[k]; }
    return NW_OK;
}
extern "C" int nw_get_profile(nw_ctx *h, double *stage_ms, int64_t *stage_launches, double *search_ms) {
    if (!h) return NW_ERR_ARG;
    for (int k = 0; k < NW_N_STAGES; ++k) {
        if (stage_ms) stage_ms[k] = h->stage_ms[k];
        if (stage_launches) stage_launches[k] = h->stage_launches[k];
    }
    if (search_ms) *search_ms = h->last_search_ms;
    return NW_OK;
}

extern "C" int nw_search(nw_ctx *h, float lam, int num_iters, int last_step, const double *prev_tests, int n_prev,
                         float *pos_out, double *tests, double *ress, double *prefs, double *cpred, double *wpred,
                         int *n_done) {
    if (!h) return NW_ERR_ARG;
    NW_ARG(h->M > 0, "nw_search: no topology (call nw_set_topology first)");
    NW_ARG(h->px != nullptr || h->P == 0, "nw_search: no points (call nw_set_points first)");
    NW_ARG(num_iters >= 0 && num_iters <= NW_MAX_ITERS, "nw_search: num_iters out of range");
    NW_ARG(n_prev >= 0 && (n_prev == 0 || prev_tests), "nw_search: bad prev_tests");
    NW_CUDA(cudaSetDevice(h->device));
    NW_CHECK(ensure_partials(h));
    SolverState s;
    memset(&s, 0, sizeof(s));
    s.lam = lam;
    s.reg_mode = h->reg_mode;
    s.n_search = 2;
    int np = n_prev > 3 ? 3 : n_prev;
    for (int k = 0; k < np; ++k) s.last_tests[k] = prev_tests[n_prev - np + k];
    s.n_tests = np;
    if (np == 3 && s.last_tests[2] < s.last_tests[1] && s.last_tests[1] < s.last_tests[0] && s.last_tests[0] < 1e-6) s.stop = 2;
    NW_CHECK(upload_state(h, s));
    // S is freshly zeroed on every search() call (mesh_conj_grad.py:207)
    NW_CUDA(cudaMemsetAsync(h->Sq, 0, sizeof(float4) * 3 * h->M, h->stream));
    NW_CUDA(cudaMemsetAsync(h->acc, 0, sizeof(unsigned long long) * 4 * h->M, h->stream));
    if (!h->ev_search0) { NW_CUDA(cudaEventCreate(&h->ev_search0)); NW_CUDA(cudaEventCreate(&h->ev_search1)); }
    h->ev_used = 0;
    h->ev_stage.clear();
    NW_CUDA(cudaEventRecord(h->ev_search0, h->stream));
    if (!s.stop) {
        int it = 0;
        // the first iteration runs eagerly: it may seed, build the launch schedule and touch allocations
        if (num_iters > 0) { NW_CHECK(enqueue_iteration(h, 0, last_step)); it = 1; }
        // every further iteration is the same ~15 launches with the same arguments: capture one, replay it.  For small
        // fits the iteration is launch-bound (C1: 0.25 ms of launches around microseconds of work).  Not under profiling
        // (per-stage events).  With a communicator the two ncclAllReduce calls of the iteration are captured with it
        // (NCCL supports stream capture; the eager first iteration has already run both collectives once, so nothing is
        // allocated or connected inside the capture).  The instantiated graph is kept for as long as the points and the
        // topology stay (h->epoch): a fit calls nw_search once per block, and repeated calls on one block (continue /
        // finishing iterations) replay the same executable.
        if (!h->profile && num_iters - it >= 2) {
            if (h->iter_graph && (h->iter_graph_epoch != h->epoch || h->iter_graph_last_step != last_step)) {
                cudaGraphExecDestroy(h->iter_graph);
                h->iter_graph = nullptr;
            }
            const int64_t l0 = h->launches;
            static int64_t per_iter_launches = 15;
            if (!h->iter_graph) {
                cudaGraph_t graph = nullptr;
                bool ok = cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal) == cudaSuccess;
                int rc = NW_OK;
                if (ok) {
                    rc = enqueue_iteration(h, it, last_step);
                    ok = cudaStreamEndCapture(h->stream, &graph) == cudaSuccess && rc == NW_OK && graph != nullptr;
                }
                per_iter_launches = h->launches - l0;
                h->launches = l0;                                    // nothing has run yet
                if (ok) ok = cudaGraphInstantiate(&h->iter_graph, graph, 0) == cudaSuccess;
                if (graph) cudaGraphDestroy(graph);
                if (ok) { h->iter_graph_epoch = h->epoch; h->iter_graph_last_step = last_step; }
                else {
                    h->iter_graph = nullptr;
                    cudaGetLastError();                              // capture refused: the loop below runs the iterations eagerly
                    if (rc != NW_OK) return rc;
                }
            }
            if (h->iter_graph) {
                for (; it < num_iters; ++it) {
                    NW_CUDA(cudaGraphLaunch(h->iter_graph, h->stream));
                    h->launches += per_iter_launches;
                }
            }
        }
        for (; it < num_iters; ++it) NW_CHECK(enqueue_iteration(h, it, last_step));
    }
    NW_CUDA(cudaEventRecord(h->ev_search1, h->stream));
    h->pin_fresh = false;
    NW_CHECK(nw_fetch_positions_async(h));          // the caller wants the result on the host next: no second round trip
    SolverState r;
    NW_CUDA(cudaMemcpyAsync(&r, h->st, sizeof(SolverState), cudaMemcpyDeviceToHost, h->stream));
    NW_CUDA(cudaStreamSynchronize(h->stream));
    {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, h->ev_search0, h->ev_search1);
        h->last_search_ms = ms;
        h->trace_stage.clear(); h->trace_ms.clear();
        for (size_t k = 0; k + 1 < h->ev_used; k += 2) {
            float t = 0.f;
            cudaEventElapsedTime(&t, h->ev_pool[k], h->ev_pool[k + 1]);
            h->stage_ms[h->ev_stage[k / 2]] += t;
            h->trace_stage.push_back(h->ev_stage[k / 2]); h->trace_ms.push_back(t);
        }
    }
    if (n_done) *n_done = r.n_done;
    if (r.n_done > 0) {
        h->weights_valid = true;
        double *dst[5] = {tests, ress, prefs, cpred, wpred};
        for (int k = 0; k < 5; ++k)
            if (dst[k]) NW_CUDA(cudaMemcpy(dst[k], h->hist + (size_t)k * NW_MAX_ITERS, sizeof(double) * r.n_done, cudaMemcpyDeviceToHost));
    }
    h->pin_fresh = true;
    if (pos_out) NW_CHECK(nw_get_positions(h, pos_out));
    if (r.nan_flag == 2) { h->err = "nw_search: singular subspace matrix (numpy.linalg.LinAlgError in the reference)"; return NW_ERR_NAN; }
    if (r.nan_flag) { h->err = "nw_search: non-finite value in residual / search directions / update"; return NW_ERR_NAN; }
    return NW_OK;
}

// Which operator regularises the fit: L = LH = "I" (0; the reference's setting, mesh_conj_grad.py:38) or "wfunc" (1; :39,
// :725-736: the prior residual weighted by 1/sqrt(sum of squared edge lengths + 1) of the current mesh).  These are the two
// settings of Lfuncs / Lhfuncs the reference's search() can actually run with (DESIGN.md section 7).
extern "C" int nw_set_regulariser(nw_ctx *h, int mode) {
    if (!h) return NW_ERR_ARG;
    NW_ARG(mode == 0 || mode == 1, "nw_set_regulariser: mode must be 0 (I) or 1 (wfunc)");
    h->reg_mode = mode;                          // read from the device state by the kernels: no new graph needed
    return NW_OK;
}

extern "C" int nw_ncc(nw_ctx *h, double *fdef) {
    if (!h) return NW_ERR_ARG;
    NW_ARG(h->M > 0 && h->weights_valid, "nw_ncc: weights not computed");
    NW_CUDA(cudaSetDevice(h->device));
    SolverState s;
    memset(&s, 0, sizeof(s));
    s.n_search = 2;
    NW_CHECK(upload_state(h, s));
    NW_CHECK(nw_set_acc_shifts(h));
    NW_CUDA(cudaMemsetAsync(h->acc, 0, sizeof(unsigned long long) * 4 * h->M, h->stream));
    NW_CHECK(nw_launch_influence(h));
    NW_CHECK(nw_allreduce_acc(h));
    NW_CHECK(nw_launch_mesh_prior(h, false));
    NW_CUDA(cudaMemsetAsync(h->acc, 0, sizeof(unsigned long long) * 4 * h->M, h->stream));
    NW_CUDA(cudaMemcpyAsync(fdef, h->fdef, sizeof(double) * 3 * h->M, cudaMemcpyDeviceToHost, h->stream));
    NW_CUDA(cudaStreamSynchronize(h->stream));
    return NW_OK;
}

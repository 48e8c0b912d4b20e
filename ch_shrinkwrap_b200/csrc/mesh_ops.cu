// mesh_ops.cu -- the per-vertex side of one CG iteration.
//
//   k_shift      : bounding box of f -> fixed-point scale of the adjoint accumulators
//   k_mesh_prior : accumulators -> S0 and point influence; 1-ring curvature prior f_def = ncc(f)
//                  (mesh_conj_grad.py:770-820); prefs = f - f_def; S1 = -prefs (:257-258); partial
//                  sums of S^T S and -S^T prefs (conj_grad.py:209-213)
//   k_solve      : (Hc + lam^2 Hw) c = Gc + lam^2 Gw (conj_grad.py:208-219), test statistic and stop
//                  rule (mesh_conj_grad.py:262-271,1009-1016), histories
//   k_update     : f <- f + S c, S2 <- step (conj_grad.py:227, mesh_conj_grad.py:281-288)
#include <cfloat>
#include <cmath>
#include "common.cuh"

namespace {

__device__ __forceinline__ double pow2d(int e) { return __longlong_as_double((long long)(1023 + e) << 52); }

// bounding box of the vertices: block reduction + ordered-int atomics into st->bbox (reset by k_shift_final)
__global__ void __launch_bounds__(256) k_shift_partial(const float4 *__restrict__ pos, int M, SolverState *st) {
    if (st->stop) return;
    float lo[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, hi[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < M; i += gridDim.x * blockDim.x) {
        const float4 v = pos[i];
        const float c[3] = {v.x, v.y, v.z};
        for (int a = 0; a < 3; ++a) if (c[a] == c[a]) { lo[a] = fminf(lo[a], c[a]); hi[a] = fmaxf(hi[a], c[a]); }
    }
    __shared__ float slo[3][8], shi[3][8];
    for (int a = 0; a < 3; ++a)
        for (int o = 16; o; o >>= 1) {
            lo[a] = fminf(lo[a], __shfl_xor_sync(0xffffffffu, lo[a], o));
            hi[a] = fmaxf(hi[a], __shfl_xor_sync(0xffffffffu, hi[a], o));
        }
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (lane == 0) for (int a = 0; a < 3; ++a) { slo[a][wid] = lo[a]; shi[a][wid] = hi[a]; }
    __syncthreads();
    if (threadIdx.x < 3) {
        const int a = threadIdx.x;
        float l = slo[a][0], u = shi[a][0];
        for (int k = 1; k < 8; ++k) { l = fminf(l, slo[a][k]); u = fmaxf(u, shi[a][k]); }
        if (l <= u) { atomicMin(&st->bbox[a], f2ord(l)); atomicMax(&st->bbox[3 + a], f2ord(u)); }
    }
}

// combine with the (static) bbox of the points -> fixed-point scales and the coordinate bound of the box tests
__global__ void k_shift_final(float plo_x, float plo_y, float plo_z, float phi_x, float phi_y, float phi_z, double wn_max,
                              double p_global, SolverState *st) {
    if (st->stop || threadIdx.x != 0) return;
    const float plo[3] = {plo_x, plo_y, plo_z}, phi[3] = {phi_x, phi_y, phi_z};
    double ext = 0.0;
    float l1 = 0.f;
    for (int a = 0; a < 3; ++a) {
        const float l = fminf(plo[a], ord2f(st->bbox[a])), u = fmaxf(phi[a], ord2f(st->bbox[3 + a]));
        ext = fmax(ext, (double)u - (double)l);
        l1 += fmaxf(fabsf(l), fabsf(u));
        st->bbox[a] = 0x7fffffff; st->bbox[3 + a] = (int)0x80000000;      // ready for the next iteration
    }
    st->coord_l1 = l1;
    // |w_j res_c| <= Wn_max * extent ; a vertex sums at most P_global of them.  Two conditions on the scale 2^shift: the sum
    // over all ranks stays below 2^61, and every single term below 2^38 (the warp scatter carries terms as five bytes,
    // sweep.cu: warp_adjoint_scatter)
    const double term = fmax(wn_max * ext, 1e-30);
    int e, et;
    frexp(term * fmax(p_global, 1.0), &e);
    frexp(term, &et);
    st->acc_shift = max(-100, min(60, min(61 - e, 38 - et)));
    frexp(fmax(p_global, 1.0), &e);
    st->infl_shift = min(61 - e, 37);             // weights are <= 1
}

#define NW_MSUM 14  // hw00 hw01 hw11 hw02 hw12 hw22 gw0 gw1 gw2 | s0.s1 s0.s0 s1.s1 | sum prefs32^2 | sum prefs64^2

template <bool WRITE_DIRS>
__global__ void __launch_bounds__(256, 3) k_mesh_prior(int M, unsigned long long *__restrict__ acc, SolverState *__restrict__ st,
                                                    const float4 *__restrict__ posq, const float4 *__restrict__ nrmq,
                                                    const int *__restrict__ nbrT, const int *__restrict__ valence,
                                                    float4 *__restrict__ Sq,
                                                    double *__restrict__ fdef_out, float *__restrict__ pi_out,
                                                    double *__restrict__ partials) {
    if (st->stop) return;
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    double sums[NW_MSUM];
#pragma unroll
    for (int k = 0; k < NW_MSUM; ++k) sums[k] = 0.0;
    if (v < M) {
        // ---- adjoint accumulators -> S0, point influence -------------------------------------------
        const float inv = (float)pow2d(-st->acc_shift), invi = (float)pow2d(-st->infl_shift);
        ulonglong2 a01 = *reinterpret_cast<ulonglong2 *>(acc + 4 * (size_t)v);
        ulonglong2 a23 = *reinterpret_cast<ulonglong2 *>(acc + 4 * (size_t)v + 2);
        const float s0x = __ll2float_rn((long long)a01.x) * inv, s0y = __ll2float_rn((long long)a01.y) * inv,
                    s0z = __ll2float_rn((long long)a23.x) * inv;
        const float sw = __ll2float_rn((long long)a23.y) * invi;
        if (WRITE_DIRS) {
            *reinterpret_cast<ulonglong2 *>(acc + 4 * (size_t)v) = make_ulonglong2(0ull, 0ull);
            *reinterpret_cast<ulonglong2 *>(acc + 4 * (size_t)v + 2) = make_ulonglong2(0ull, 0ull);
        }
        // |AH 1| with identical components: sqrt(s^2+s^2+s^2) in float32 (_membrane_mesh.pyx:1633-1634)
        const float sq = __fmul_rn(sw, sw);
        const float pi = __fsqrt_rn(__fadd_rn(__fadd_rn(sq, sq), sq));
        if (pi_out) pi_out[v] = pi;
        // ---- ncc: mesh_conj_grad.py:777-818 --------------------------------------------------------
        const float4 p = posq[v], N = nrmq[v];
        const int ms = valence[v];
        const bool reg = st->reg_mode == 1;
        float ring2 = 0.f;
        double fx = p.x, fy = p.y, fz = p.z;     // ms == 0 -> f_def = vertex (:818)
        if (ms > 0) {
            int nb[NW_NEIGHBORSIZE];
            float cx = 0.f, cy = 0.f, cz = 0.f;
#pragma unroll
            for (int k = 0; k < NW_NEIGHBORSIZE; ++k) {
                nb[k] = (k < ms) ? nbrT[(size_t)k * M + v] : -1;
                if (k < ms) {
                    const float4 q = __ldg(&posq[nb[k]]);
                    cx = __fadd_rn(cx, q.x); cy = __fadd_rn(cy, q.y); cz = __fadd_rn(cz, q.z);   // float32 sum (:782)
                    if (reg) {          // vertex_area_weights on the current f (conj_grad_utils.c:500-528): sum of squared edge lengths
                        float dd = __fsub_rn(q.x, p.x), d2 = __fmul_rn(dd, dd);
                        dd = __fsub_rn(q.y, p.y); d2 = __fadd_rn(d2, __fmul_rn(dd, dd));
                        dd = __fsub_rn(q.z, p.z); d2 = __fadd_rn(d2, __fmul_rn(dd, dd));
                        ring2 = __fadd_rn(ring2, d2);
                    }
                }
            }
            const double dms = (double)ms;
            const double vcx = (double)cx / dms, vcy = (double)cy / dms, vcz = (double)cz / dms;
            // alpha_k, summed in numpy's pairwise order for 20 contiguous doubles
            double r8[8];
            double tail = 0.0;
#pragma unroll
            for (int k = 0; k < NW_NEIGHBORSIZE; ++k) {
                double ak = 0.0;
                if (k < ms) {
                    const float4 q = __ldg(&posq[nb[k]]), nn = __ldg(&nrmq[nb[k]]);
                    const double cnx = (double)q.x - vcx, cny = (double)q.y - vcy, cnz = (double)q.z - vcz;       // :785
                    const double num = __dadd_rn(__dadd_rn(__dmul_rn(cnx, (double)nn.x), __dmul_rn(cny, (double)nn.y)),
                                                 __dmul_rn(cnz, (double)nn.z));
                    const float ndn = __fadd_rn(__fadd_rn(__fmul_rn(nn.x, N.x), __fmul_rn(nn.y, N.y)), __fmul_rn(nn.z, N.z));   // :796
                    const float den = __fsqrt_rn(__fmul_rn(2.0f, __fadd_rn(fmaxf(ndn, 0.f), 1.0f)));                               // :797
                    ak = num / (double)den;
                }
                if (k < 8) r8[k] = ak;
                else if (k < 16) r8[k - 8] = __dadd_rn(r8[k - 8], ak);
                else {
                    if (k == 16)
                        tail = __dadd_rn(__dadd_rn(__dadd_rn(r8[0], r8[1]), __dadd_rn(r8[2], r8[3])),
                                         __dadd_rn(__dadd_rn(r8[4], r8[5]), __dadd_rn(r8[6], r8[7])));
                    tail = __dadd_rn(tail, ak);
                }
            }
            double alpha = tail / dms;                                                   // :800
            alpha = alpha * (double)fminf(__fmul_rn(pi, pi), 1.0f);                      // :814
            fx = __dadd_rn(vcx, __dmul_rn(alpha, (double)N.x));                          // :816
            fy = __dadd_rn(vcy, __dmul_rn(alpha, (double)N.y));
            fz = __dadd_rn(vcz, __dmul_rn(alpha, (double)N.z));
        }
        if (fdef_out) { fdef_out[3 * (size_t)v] = fx; fdef_out[3 * (size_t)v + 1] = fy; fdef_out[3 * (size_t)v + 2] = fz; }
        if (WRITE_DIRS) {
            // prefs = L(f - f_def) (float64 in subsearch, float32 in search); S1 = -LH(prefs); LS_k = L(S_k)
            //   L = "I"     (mesh_conj_grad.py:38):     prefs = f - f_def,        S1 = -prefs32,        LS_k = S_k
            //   L = "wfunc" (:725-736, w = area weight): prefs = (f - f_def) w,    S1 = -(prefs32 w),    LS_k = S_k w
            // (the other 1-ring operators cannot be the regulariser of a fit in the reference either: search() hands them
            // the float64 array f - f_def and the C helpers read it as float32, conj_grad_utils.c:283 -- they raise
            // AssertionError on the NaNs that produces; DESIGN.md section 7)
            float wv = 1.0f;
            if (reg) wv = (ms > 0 && ring2 > 0.f) ? (float)(1.0 / (double)__fsqrt_rn(__fadd_rn(ring2, 1.0f))) : 0.f;   // conj_grad_utils.c:530-540
            double pr[3] = {(double)p.x - fx, (double)p.y - fy, (double)p.z - fz};
            if (reg) { pr[0] = __dmul_rn(pr[0], (double)wv); pr[1] = __dmul_rn(pr[1], (double)wv); pr[2] = __dmul_rn(pr[2], (double)wv); }
            const float p32[3] = {(float)pr[0], (float)pr[1], (float)pr[2]};
            float s1x = -p32[0], s1y = -p32[1], s1z = -p32[2];
            if (reg) { s1x = -__fmul_rn(p32[0], wv); s1y = -__fmul_rn(p32[1], wv); s1z = -__fmul_rn(p32[2], wv); }
            Sq[3 * (size_t)v] = make_float4(s0x, s0y, s0z, 0.f);
            Sq[3 * (size_t)v + 1] = make_float4(s1x, s1y, s1z, 0.f);
            if (!(fabsf(s0x) <= FLT_MAX && fabsf(s0y) <= FLT_MAX && fabsf(s0z) <= FLT_MAX &&
                  fabsf(s1x) <= FLT_MAX && fabsf(s1y) <= FLT_MAX && fabsf(s1z) <= FLT_MAX)) st->nan_flag = 1;
            const float4 s2 = Sq[3 * (size_t)v + 2];
            const float S0[3] = {s0x, s0y, s0z}, S1[3] = {s1x, s1y, s1z}, S2[3] = {s2.x, s2.y, s2.z};
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                // LS_k: float32 products like wfunc's f * w
                const double a0 = reg ? (double)__fmul_rn(S0[c], wv) : (double)S0[c], a1 = reg ? (double)__fmul_rn(S1[c], wv) : (double)S1[c],
                             a2 = reg ? (double)__fmul_rn(S2[c], wv) : (double)S2[c];
                sums[0] += a0 * a0; sums[1] += a0 * a1; sums[2] += a1 * a1;
                sums[3] += a0 * a2; sums[4] += a1 * a2; sums[5] += a2 * a2;
                sums[6] -= a0 * pr[c]; sums[7] -= a1 * pr[c]; sums[8] -= a2 * pr[c];
                sums[9] += (double)S0[c] * (double)S1[c]; sums[10] += (double)S0[c] * (double)S0[c]; sums[11] += (double)S1[c] * (double)S1[c];
                sums[12] += (double)p32[c] * (double)p32[c];
                sums[13] += pr[c] * pr[c];
            }
        }
    }
    if (!WRITE_DIRS) return;
    __shared__ double sh[8][NW_MSUM];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < NW_MSUM; ++k) {
        double x = sums[k];
        for (int o = 16; o; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
        if (lane == 0) sh[wid][k] = x;
    }
    __syncthreads();
    if (threadIdx.x < NW_MSUM) {
        double x = 0.0;
        for (int k = 0; k < 8; ++k) x += sh[k][threadIdx.x];
        partials[(size_t)blockIdx.x * NW_MSUM + threadIdx.x] = x;
    }
}

// fold the mesh partials: one CTA per quantity, fixed order (thread t sums partials t, t+256, ...; then a fixed tree)
__global__ void __launch_bounds__(256) k_fold_mesh(const double *__restrict__ mesh_partials, int n_mesh_blocks, SolverState *st) {
    if (st->stop) return;
    __shared__ double sh[256];
    const int k = blockIdx.x;
    double v = 0.0;
    for (int b = threadIdx.x; b < n_mesh_blocks; b += 256) v += mesh_partials[(size_t)b * NW_MSUM + k];
    sh[threadIdx.x] = v;
    __syncthreads();
    for (int o = 128; o; o >>= 1) {
        if (threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const double t = sh[0];
        if (k < 6) st->hw[k] = t;
        else if (k < 9) st->gw[k - 6] = t;
        else if (k < 12) st->tst[k - 9] = t;
        else if (k == 12) st->prefs32_2 = t;
        else st->prefs64_2 = t;
    }
}

// one thread: solve, log, stop rule
__global__ void k_solve(SolverState *st, double *__restrict__ hist, int iter_index) {
    if (st->stop || threadIdx.x != 0) return;
    iter_index = st->n_done;          // == the host's loop index (n_done starts at 0 in nw_search and is bumped below); reading
                                      // it here leaves the launch without per-iteration arguments, so it can be replayed from a graph
    const int n = st->n_search;
    const double l2 = (double)st->lam * (double)st->lam;
    // symmetric index map (i<=j): 00->0 01->1 11->2 02->3 12->4 22->5
    const int map[3][3] = {{0, 1, 3}, {1, 2, 4}, {3, 4, 5}};
    double Hc[3][3], Hw[3][3], H[3][4];
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) { Hc[i][j] = st->hc[map[i][j]]; Hw[i][j] = st->hw[map[i][j]]; }
    for (int i = 0; i < n; ++i) {
        for (int j = 0; j < n; ++j) H[i][j] = Hc[i][j] + l2 * Hw[i][j];
        H[i][3] = st->gc[i] + l2 * st->gw[i];
    }
    // Gaussian elimination with partial pivoting (np.linalg.solve -> LAPACK gesv)
    double c[3] = {0.0, 0.0, 0.0};
    bool singular = false;
    for (int k = 0; k < n; ++k) {
        int piv = k;
        for (int i = k + 1; i < n; ++i) if (fabs(H[i][k]) > fabs(H[piv][k])) piv = i;
        if (H[piv][k] == 0.0 || !(fabs(H[piv][k]) <= DBL_MAX)) { singular = true; break; }
        if (piv != k) for (int j = 0; j < 4; ++j) { double t = H[k][j]; H[k][j] = H[piv][j]; H[piv][j] = t; }
        for (int i = k + 1; i < n; ++i) {
            const double m = H[i][k] / H[k][k];
            for (int j = k; j < n; ++j) H[i][j] -= m * H[k][j];
            H[i][3] -= m * H[k][3];
        }
    }
    if (!singular)
        for (int i = n - 1; i >= 0; --i) {
            double s = H[i][3];
            for (int j = i + 1; j < n; ++j) s -= H[i][j] * c[j];
            c[i] = s / H[i][i];
        }
    if (singular) st->nan_flag = 2;   // numpy raises LinAlgError("Singular matrix")
    for (int i = 0; i < 3; ++i) { st->c[i] = (i < n) ? c[i] : 0.0; if (!(fabs(st->c[i]) <= DBL_MAX)) st->nan_flag = 1; }
    // diagnostics: cpred uses the *regularised* matrix because H aliases Hc (conj_grad.py:208,223; SURVEY B.3)
    double cHc = 0.0, cGc = 0.0, cHwc = 0.0, cGw = 0.0;
    for (int i = 0; i < n; ++i) {
        for (int j = 0; j < n; ++j) { cHc += c[i] * (Hc[i][j] + l2 * Hw[i][j]) * c[j]; cHwc += c[i] * Hw[i][j] * c[j]; }
        cGc += c[i] * (st->gc[i] + l2 * st->gw[i]);
        cGw += c[i] * st->gw[i];
    }
    const double prefs2 = st->prefs32_2;   // |prefs|^2 of the float32 prefs array (history, mesh_conj_grad.py:271)
    // mesh_conj_grad.py:262-265.  The reference forms the ratio from float32 sums and subtracts it from 1 in float32, so
    // its statistic moves in steps of 2^-24 near convergence, and the stop rule ("strictly decreasing three times",
    // :1009-1016) sees those steps.  Here the ratio comes from float64 sums (more accurate than the reference's own) and
    // is rounded to float32 ONCE, then subtracted in float32: the history and the rule work on the same kind of number as
    // the reference's, and what the caller gets back (float32 in self.tests) is exactly what the device compared.
    const float ratio32 = (float)fabs(st->tst[0] / (sqrt(st->tst[1]) * sqrt(st->tst[2])));
    const double test = (double)(1.0f - ratio32);
    hist[0 * NW_MAX_ITERS + iter_index] = test;
    hist[1 * NW_MAX_ITERS + iter_index] = sqrt(st->res2);
    hist[2 * NW_MAX_ITERS + iter_index] = sqrt(prefs2);
    hist[3 * NW_MAX_ITERS + iter_index] = st->c0 + cHc - cGc;
    hist[4 * NW_MAX_ITERS + iter_index] = st->prefs64_2 + cHwc - cGw;      // wpreds[0], conj_grad.py:192,224
    // histories for the stop rule (:1009-1016): evaluated at the top of the NEXT iteration
    if (st->n_tests < 3) st->last_tests[st->n_tests++] = test;
    else { st->last_tests[0] = st->last_tests[1]; st->last_tests[1] = st->last_tests[2]; st->last_tests[2] = test; }
    st->n_done += 1;
    if (st->n_tests == 3) {
        const double a = st->last_tests[0], b = st->last_tests[1], cc = st->last_tests[2];
        if (cc < b && b < a && a < 1e-6) st->stop = 1;
    }
}

__global__ void __launch_bounds__(256) k_update(int M, SolverState *__restrict__ st, float4 *__restrict__ posq,
                                                float4 *__restrict__ Sq, int last_step, int is_final_launch) {
    // runs for the iteration that k_solve just completed, including the one that set `stop`
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (st->nan_flag == 2) return;
    if (st->stop > 1) return;
    if (v < M) {
        const double c0 = st->c[0], c1 = st->c[1], c2 = st->c[2];
        const float4 p = posq[v], a = Sq[3 * (size_t)v], b = Sq[3 * (size_t)v + 1], d = Sq[3 * (size_t)v + 2];
        const double nx = (double)p.x + (((double)a.x * c0 + (double)b.x * c1) + (double)d.x * c2);
        const double ny = (double)p.y + (((double)a.y * c0 + (double)b.y * c1) + (double)d.y * c2);
        const double nz = (double)p.z + (((double)a.z * c0 + (double)b.z * c1) + (double)d.z * c2);
        if (last_step) Sq[3 * (size_t)v + 2] = make_float4((float)(nx - (double)p.x), (float)(ny - (double)p.y), (float)(nz - (double)p.z), 0.f);
        const float4 q = make_float4((float)nx, (float)ny, (float)nz, 0.f);
        if (!(fabsf(q.x) <= FLT_MAX && fabsf(q.y) <= FLT_MAX && fabsf(q.z) <= FLT_MAX)) st->nan_flag = 1;
        posq[v] = q;
    }
}

// after k_update of an iteration: bump n_search, latch `stop` so later launches are no-ops
__global__ void k_advance(SolverState *st, int last_step) {
    if (st->stop > 1) return;
    if (st->stop == 1) { st->stop = 2; return; }
    if (last_step) st->n_search = 3;
}

__global__ void k_fill(float *p, int64_t n, float v) {
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}
__global__ void k_norm3(const float *__restrict__ in, int M, float *__restrict__ out) {
    int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= M) return;
    float a = in[3 * v], b = in[3 * v + 1], c = in[3 * v + 2];
    out[v] = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(a, a), __fmul_rn(b, b)), __fmul_rn(c, c)));
}
__global__ void k_S_rows(const float4 *__restrict__ Sq, int M, float *__restrict__ out) {
    int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= M) return;
    const float4 a = Sq[3 * (size_t)v], b = Sq[3 * (size_t)v + 1], c = Sq[3 * (size_t)v + 2];
    float *o = out + 9 * (size_t)v;   // rows 3v..3v+2 of the (3M,3) matrix
    o[0] = a.x; o[1] = b.x; o[2] = c.x;
    o[3] = a.y; o[4] = b.y; o[5] = c.y;
    o[6] = a.z; o[7] = b.z; o[8] = c.z;
}

}  // namespace

int nw_apply_AH_device(nw_ctx *h, const float *rx, const float *ry, const float *rz, double bound, float *out3M);

int nw_set_acc_shifts(nw_ctx *h) {
    k_shift_partial<<<std::min(nw_grid(h->M, 256), 148 * 4), 256, 0, h->stream>>>(h->posq, h->M, h->st);
    NW_LAUNCH_CHECK();
    k_shift_final<<<1, 32, 0, h->stream>>>(h->bbox_pts[0], h->bbox_pts[1], h->bbox_pts[2], h->bbox_pts[3], h->bbox_pts[4],
                                            h->bbox_pts[5], h->wn_max, (double)std::max<int64_t>(h->P_global, 1), h->st);
    NW_LAUNCH_CHECK();
    return NW_OK;
}

static int mesh_blocks(nw_ctx *h) { return nw_grid(h->M, 256); }

int nw_launch_mesh_prior(nw_ctx *h, bool write_dirs) {
    const int G = mesh_blocks(h);
    if (write_dirs)
        k_mesh_prior<true><<<G, 256, 0, h->stream>>>(h->M, h->acc, h->st, h->posq, h->nrmq, h->nbrT, h->valence, h->Sq,
                                                     nullptr, nullptr, h->partials + (size_t)h->n_partials * 16);
    else
        k_mesh_prior<false><<<G, 256, 0, h->stream>>>(h->M, h->acc, h->st, h->posq, h->nrmq, h->nbrT, h->valence, h->Sq,
                                                      h->fdef, h->scratchM, nullptr);
    NW_LAUNCH_CHECK();
    return NW_OK;
}

int nw_launch_solve_update(nw_ctx *h, int iter_index, int last_step) {
    k_fold_mesh<<<NW_MSUM, 256, 0, h->stream>>>(h->partials + (size_t)h->n_partials * 16, mesh_blocks(h), h->st);
    NW_LAUNCH_CHECK();
    k_solve<<<1, 32, 0, h->stream>>>(h->st, h->hist, iter_index);
    NW_LAUNCH_CHECK();
    k_update<<<mesh_blocks(h), 256, 0, h->stream>>>(h->M, h->st, h->posq, h->Sq, last_step, 0);
    NW_LAUNCH_CHECK();
    k_advance<<<1, 1, 0, h->stream>>>(h->st, last_step);
    NW_LAUNCH_CHECK();
    return NW_OK;
}

extern "C" int nw_point_influence(nw_ctx *h, float *pi) {
    if (!h) return NW_ERR_ARG;
    NW_ARG(h->M > 0 && h->weights_valid, "nw_point_influence: weights not computed");
    NW_CUDA(cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    const int64_t P = h->P;
    float *ones = nullptr;
    NW_CHECK(nw_alloc(h, &ones, (size_t)std::max<int64_t>(P, 1)));
    if (P) { k_fill<<<nw_grid(P, 256), 256, 0, s>>>(ones, P, 1.0f); NW_LAUNCH_CHECK(); }
    float *tmp = nullptr;
    NW_CHECK(nw_alloc(h, &tmp, (size_t)3 * h->M));
    NW_CHECK(nw_apply_AH_device(h, ones, ones, ones, 1.0, tmp));
    k_norm3<<<nw_grid(h->M, 256), 256, 0, s>>>(tmp, h->M, h->scratchM);
    NW_LAUNCH_CHECK();
    NW_CUDA(cudaMemcpyAsync(pi, h->scratchM, sizeof(float) * h->M, cudaMemcpyDeviceToHost, s));
    NW_CUDA(cudaStreamSynchronize(s));
    nw_free(&ones); nw_free(&tmp);
    return NW_OK;
}

extern "C" int nw_get_S(nw_ctx *h, float *S) {
    if (!h) return NW_ERR_ARG;
    NW_ARG(h->M > 0, "nw_get_S: no topology");
    NW_CUDA(cudaSetDevice(h->device));
    float *tmp = nullptr;
    NW_CHECK(nw_alloc(h, &tmp, (size_t)9 * h->M));
    k_S_rows<<<nw_grid(h->M, 256), 256, 0, h->stream>>>(h->Sq, h->M, tmp);
    NW_LAUNCH_CHECK();
    NW_CUDA(cudaMemcpyAsync(S, tmp, sizeof(float) * 9 * h->M, cudaMemcpyDeviceToHost, h->stream));
    NW_CUDA(cudaStreamSynchronize(h->stream));
    nw_free(&tmp);
    return NW_OK;
}

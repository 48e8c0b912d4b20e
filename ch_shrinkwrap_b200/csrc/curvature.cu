// curvature.cu -- per-vertex Taubin curvature tensor, principal curvatures / directions, mean and
// Gaussian curvature, displaced-surface curvatures, Canham-Helfrich energy and its gradient from the
// 1-ring.  Replaces the serial loop of c_curvature_grad (membrane_mesh_utils.c:915-1250): one thread
// per vertex, fp64 locals exactly where the reference has them.
//
// THIS FILE IS COMPILED WITH -fmad=false: every +,-,*,/ and sqrt below is a single IEEE operation in
// the reference's order, so k0,k1,e0,e1,H,K,E reproduce the reference bit for bit; atan2/sin/cos/exp
// (dH, dK, pE, dEdN) are within the CUDA math library's 1-2 ulp.
#include <cub/cub.cuh>
#include <cmath>
#include <cstddef>
#include <cstring>
#include <thread>
#include <vector>
#include "common.cuh"

namespace {

struct HeRec { int vertex, face, twin, next, prev; float length; int component; };                 // 28 B
struct FaceRec { int halfedge; float normal[3]; float area; int component; };                      // 24 B
struct VertRec { float position[3]; float normal[3]; int halfedge, valence; int neighbors[NW_NEIGHBORSIZE];
                 int component, locally_manifold; };                                               // 120 B
static_assert(sizeof(HeRec) == 28 && sizeof(FaceRec) == 24 && sizeof(VertRec) == 120, "record layouts");

#define TINY 1e-15
struct d3 { double x, y, z; };

__device__ __forceinline__ double nrm(const d3 a) { double n = 0.0; n += a.x * a.x; n += a.y * a.y; n += a.z * a.z; return sqrt(n); }
__device__ __forceinline__ float nrmf(const float *a) { float n = 0.0f; n += a[0] * a[0]; n += a[1] * a[1]; n += a[2] * a[2]; return sqrtf(n); }
__device__ __forceinline__ double sdiv(double x, double y) { return (fabs(y) < TINY) ? 0.0 : x / y; }
__device__ __forceinline__ d3 fsub(const float *a, const float *b) {
    d3 r = {(double)a[0] - (double)b[0], (double)a[1] - (double)b[1], (double)a[2] - (double)b[2]};
    return r;
}
__device__ __forceinline__ double fdot(const float *a, const d3 b) {
    double c = 0.0; c += (double)a[0] * b.x; c += (double)a[1] * b.y; c += (double)a[2] * b.z; return c;
}
__device__ __forceinline__ double chord(double c) { double q = c * c; return (q > 1.0) ? sqrt(2.0) : sqrt(2.0 - 2.0 * sqrt(1.0 - q)); }

__device__ __forceinline__ void projector(const float *v, double coef, double *m) {
    const double a = (double)v[0], b = (double)v[1], c = (double)v[2];
    const float ab = (float)(-1.0 * coef * a * b), ac = (float)(-1.0 * coef * a * c), bc = (float)(-1.0 * coef * b * c);
    m[0] = 1.0 - coef * a * a; m[1] = ab; m[2] = ac;
    m[3] = ab; m[4] = 1.0 - coef * b * b; m[5] = bc;
    m[6] = ac; m[7] = bc; m[8] = 1.0 - coef * c * c;
}

__device__ __forceinline__ void mm3(const double *a, const double *b, double *c) {
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            double s = 0.0;
#pragma unroll
            for (int k = 0; k < 3; ++k) s += a[3 * i + k] * b[3 * k + j];
            c[3 * i + j] = s;
        }
}

__device__ void tensor_eig(const double *Mv, const float *N, double *l1, double *l2, double *v1, double *v2) {
    float dm[3] = {1.0f - N[0], 0.0f - N[1], 0.0f - N[2]};
    float dp[3] = {1.0f + N[0], 0.0f + N[1], 0.0f + N[2]};
    const float nm = nrmf(dm), np_ = nrmf(dp);
    float W[3];
    if (nm > np_) { W[0] = dm[0] / nm; W[1] = dm[1] / nm; W[2] = dm[2] / nm; }
    else { W[0] = dp[0] / np_; W[1] = dp[1] / np_; W[2] = dp[2] / np_; }
    double Q[9], QT[9], QM[9], B[9];
    projector(W, 2.0, Q);
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) QT[3 * j + i] = Q[3 * i + j];
    mm3(Q, Mv, QM);
    mm3(QM, QT, B);
    const double tau = sdiv(B[8] - B[4], 2.0 * B[5]);
    const double t = ((tau < 0) ? -1 : 1) / (fabs(tau) + sqrt(1 + tau * tau));
    const double a = B[4] - t * B[5], b = B[8] + t * B[5];
    const double cs = 1.0 / sqrt(1 + t * t), sn = t * cs;
    const double p[3] = {cs * QT[1] - sn * QT[2], cs * QT[4] - sn * QT[5], cs * QT[7] - sn * QT[8]};
    const double q[3] = {sn * QT[1] + cs * QT[2], sn * QT[4] + cs * QT[5], sn * QT[7] + cs * QT[8]};
    if (a > b) { *l1 = a; *l2 = b; for (int i = 0; i < 3; ++i) { v1[i] = p[i]; v2[i] = q[i]; } }
    else { *l1 = b; *l2 = a; for (int i = 0; i < 3; ++i) { v2[i] = p[i]; v1[i] = q[i]; } }
}

__device__ void pinv2(const double *A, double *Ai) {
    const double a = A[0], b = A[1], c = A[2], d = A[3];
    const double a2 = a * a, b2 = b * b, c2 = c * c, d2 = d * d;
    const double ab2 = a2 + b2, cd2 = c2 + d2, diff = ab2 - cd2, cross = 2 * (a * c + b * d);
    const double th = 0.5 * atan2(2 * (a * b + c * d), a2 + c2 - b2 - d2), ph = 0.5 * atan2(cross, diff);
    const double ct = cos(th), cp = cos(ph), st = sin(th), sp = sin(ph);
    const double ctcp = ct * cp, ctsp = ct * sp, stcp = st * cp, stsp = st * sp;
    const int sg0 = ((ctcp * a + ctsp * c + stcp * b + stsp * d) < 0) ? -1 : 1;
    const int sg1 = ((stsp * a - stcp * c - ctsp * b + ctcp * d) < 0) ? -1 : 1;
    const double ss = ab2 + cd2, sd = sqrt(diff * diff + cross * cross);
    const double s0 = sqrt((ss + sd) / 2.0), rem = ss - sd, s1 = (rem > 0) ? sqrt(rem / 2.0) : 0.0;
    const double thr = (1e-8) * 0.5 * sqrt(5.0) * s0;
    const double i0 = (s0 < thr) ? 0.0 : (1.0 / s0), i1 = (s1 < thr) ? 0.0 : (1.0 / s1);
    const double u = sg0 * i0, v = sg1 * i1;
    Ai[0] = ctcp * u + stsp * v; Ai[1] = ctsp * u - stcp * v;
    Ai[2] = stcp * u - ctsp * v; Ai[3] = stsp * u + ctcp * v;
}

// splitmix64 -> uniform [0,1) with 31 random bits, like rand()/(RAND_MAX+1)
__device__ __forceinline__ double hash_uniform(unsigned long long seed, unsigned long long ctr) {
    unsigned long long z = seed + 0x9e3779b97f4a7c15ULL * (ctr + 1);
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ULL;
    z = (z ^ (z >> 27)) * 0x94d049bb133111ebULL;
    z ^= z >> 31;
    return (double)(z >> 33) / 2147483648.0;
}

__global__ void k_valid_flags(const VertRec *__restrict__ V, int M, int *__restrict__ flag) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < M) flag[i] = V[i].halfedge != -1;
}

struct CurvOut { float *k0, *k1, *e0, *e1, *H, *K, *dH, *dK, *E, *pE, *dEnb, *dEdN; int *n_deleted; };

#define NW_CURV_BLOCK 128
// 4 blocks per SM = 128 registers, 16 warps per SM: measured at C3 0.285 ms (3 blocks, 152 registers) -> 0.242 ms; 5 blocks (96 registers, spills) 0.248 ms
__global__ void __launch_bounds__(NW_CURV_BLOCK, 4) k_curvature(const VertRec *__restrict__ V, const FaceRec *__restrict__ F,
                                                   const HeRec *__restrict__ HE, int M, float dN, float kc, float kg, float c0,
                                                   const double *__restrict__ jitter_u, const int *__restrict__ jitter_off,
                                                   unsigned long long seed, CurvOut o) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= M) return;
    const VertRec *cv = &V[i];
    if (cv->halfedge == -1) {                        // membrane_mesh_utils.c:962-973 (k0,k1,e0,e1 untouched: the copy-out skips these rows)
        atomicAdd(o.n_deleted, 1);
        o.H[i] = o.K[i] = o.dH[i] = o.dK[i] = o.dEnb[i] = o.E[i] = o.pE[i] = 0.0f;
        o.dEdN[3 * i] = o.dEdN[3 * i + 1] = o.dEdN[3 * i + 2] = 0.0f;
        return;
    }
    const double kcd = (double)kc, kgd = (double)kg, c0d = (double)c0, dNd = (double)dN;
    float vi[3] = {cv->position[0], cv->position[1], cv->position[2]};
    float Ni[3] = {cv->normal[0], cv->normal[1], cv->normal[2]};
    int nbh[NW_NEIGHBORSIZE];
    float cen[3] = {0.f, 0.f, 0.f};
    double r_sum = 0.0, jw = 10000000000000000.0;
    int n = 0;
    // pass 1 (:986-1009)
    while (n < NW_NEIGHBORSIZE) {
        const int hn = cv->neighbors[n];
        if (hn == -1) break;
        nbh[n] = hn;
        const float *vj = V[HE[hn].vertex].position;
        for (int a = 0; a < 3; ++a) cen[a] += vj[a];
        const double len = nrm(fsub(vj, vi));
        if (len > TINY) r_sum += 1.0 / len;
        if (len < jw) jw = len;                      // unconditional in the reference (:1002-1005)
        ++n;
    }
    for (int a = 0; a < 3; ++a) cen[a] /= n;
    for (int a = 0; a < 3; ++a) {                     // :1016-1017
        const double u = jitter_u ? jitter_u[3 * (size_t)jitter_off[i] + a] : hash_uniform(seed, 3ull * i + a);
        cen[a] = (float)((double)cen[a] + jw * (u - 0.5));
    }
    float dir[3] = {cen[0] - vi[0], cen[1] - vi[1], cen[2] - vi[2]};
    const float dir_n = nrmf(dir);
    for (int a = 0; a < 3; ++a) dir[a] = (dir_n > 0.0f) ? dir[a] / dir_n : 0.0f;
    const d3 sh = {(double)dir[0] * dNd, (double)dir[1] * dNd, (double)dir[2] * dNd};
    const d3 vsh = {(double)vi[0] - sh.x, (double)vi[1] - sh.y, (double)vi[2] - sh.z};
    double P[9], Mv[9];
    projector(Ni, 1.0, P);
    for (int a = 0; a < 9; ++a) Mv[a] = 0.0;
    double areas = 0.0, dareas = 0.0;
    float dEnb = 0.0f;
    d3 e_hat = {0, 0, 0}, e1_hat = {0, 0, 0};
    // pass 2 (:1046-1122)
    for (int j = 0; j < n; ++j) {
        const HeRec h = HE[nbh[j]];
        const VertRec *nv = &V[h.vertex];
        const float vj[3] = {nv->position[0], nv->position[1], nv->position[2]};
        const float Nj[3] = {nv->normal[0], nv->normal[1], nv->normal[2]};
        const d3 e = fsub(vj, vi);
        const d3 e1 = {e.x - sh.x, e.y - sh.y, e.z - sh.z};
        const double len = nrm(e), len1 = nrm(e1);
        if (len > TINY) { e_hat.x = e.x / len; e_hat.y = e.y / len; e_hat.z = e.z / len; }
        if (len1 > TINY) { e1_hat.x = e1.x / len1; e1_hat.y = e1.y / len1; e1_hat.z = e1.z / len1; }
        const d3 me = {e.x * -1.0, e.y * -1.0, e.z * -1.0};
        const d3 T = {P[0] * me.x + P[1] * me.y + P[2] * me.z, P[3] * me.x + P[4] * me.y + P[5] * me.z,
                      P[6] * me.x + P[7] * me.y + P[8] * me.z};
        const double Tn = nrm(T);
        double Tij[3] = {0, 0, 0};
        if (Tn > TINY) { Tij[0] = T.x / Tn; Tij[1] = T.y / Tn; Tij[2] = T.z / Tn; }
        const double ci = chord(fdot(Ni, e_hat));
        const double cj = chord(fdot(Nj, e_hat));
        const double cj1 = chord(fdot(Nj, e1_hat));
        const double kj = sdiv(2.0 * cj, len), kj1 = sdiv(2.0 * cj1, len1);
        const double w = sdiv(sdiv(1.0, len), r_sum);
        const double k = sdiv(2.0 * ((fdot(Ni, me) < 0) ? -1 : 1) * ci, len);
        const double Aj = (double)F[h.face].area;
        const float *vnp = V[HE[h.next].vertex].position;
        const d3 en = {(double)vnp[0] - vsh.x, (double)vnp[1] - vsh.y, (double)vnp[2] - vsh.z};
        const d3 cr = {e1.y * en.z - e1.z * en.y, e1.z * en.x - e1.x * en.z, e1.x * en.y - e1.y * en.x};
        const double dAj = 0.5 * nrm(cr);
        dareas += dAj;
        areas += Aj;
        const double t0 = 2.0 * kj - c0d, t1 = 2.0 * kj1 - c0d;
        dEnb += ((float)(Aj * w * 0.5 * kcd * (t0 * t0) - dAj * w * 0.5 * kcd * (t1 * t1))) / dN;   // :1115
        const double wk = w * k;
#pragma unroll
        for (int r = 0; r < 3; ++r)
#pragma unroll
            for (int c = 0; c < 3; ++c) Mv[3 * r + c] += (Tij[r] * Tij[c]) * wk;
    }
    o.dEnb[i] = dEnb;
    double l1, l2, v1[3], v2[3];
    tensor_eig(Mv, Ni, &l1, &l2, v1, v2);
    float k0f, k1f;
    if (isnan(l1)) {                                  // :1129-1139
        k0f = k1f = 0.0f;
        for (int a = 0; a < 3; ++a) v1[a] = v2[a] = 0.0;
    } else {
        k0f = (float)(3.0 * l1 - l2);
        k1f = (float)(3.0 * l2 - l1);
    }
    o.k0[i] = k0f; o.k1[i] = k1f;
    for (int a = 0; a < 3; ++a) { o.e0[3 * i + a] = (float)v1[a]; o.e1[3 * i + a] = (float)v2[a]; }
    const float Hf = (float)(0.5 * (double)(k0f + k1f));    // :1151
    const float Kf = k0f * k1f;                               // :1152
    o.H[i] = Hf; o.K[i] = Kf;
    // pass 3 (:1161-1192)
    double a00 = 0.0, a01 = 0.0, a10 = 0.0, a11 = 0.0;
    double Ar[2 * NW_NEIGHBORSIZE], br[NW_NEIGHBORSIZE];
    for (int j = 0; j < n; ++j) {
        const d3 e = fsub(V[HE[nbh[j]].vertex].position, vi);
        const double p = e.x * v1[0] + e.y * v1[1] + e.z * v1[2];
        const double q = e.x * v2[0] + e.y * v2[1] + e.z * v2[2];
        Ar[2 * j] = p * p; Ar[2 * j + 1] = q * q;
        br[j] = Ar[2 * j] * (double)k0f + Ar[2 * j + 1] * (double)k1f - dNd;
    }
    for (int j = 0; j < n; ++j) {
        a00 += Ar[2 * j] * Ar[2 * j]; a01 += Ar[2 * j] * Ar[2 * j + 1];
        a10 += Ar[2 * j + 1] * Ar[2 * j]; a11 += Ar[2 * j + 1] * Ar[2 * j + 1];
    }
    double AtA[4] = {a00, a01, a10, a11}, Ai[4], kp0 = 0.0, kp1 = 0.0;
    pinv2(AtA, Ai);
    for (int j = 0; j < n; ++j) {
        double r0 = 0.0, r1 = 0.0;
        r0 += Ai[0] * Ar[2 * j]; r0 += Ai[1] * Ar[2 * j + 1];
        r1 += Ai[2] * Ar[2 * j]; r1 += Ai[3] * Ar[2 * j + 1];
        kp0 += r0 * br[j]; kp1 += r1 * br[j];
    }
    const float dHf = (float)(0.5 * (kp0 + kp1)), dKf = (float)(kp0 * kp1);
    o.dH[i] = dHf; o.dK[i] = dKf;
    const double th = 2.0 * (double)Hf - c0d;
    const float Ef = (float)(areas * ((0.5 * kcd * (th * th) + kgd * (double)Kf)));        // :1195
    const float pEf = (float)exp(-(1.0 / 0.0257) * (double)Ef);                            // :1197
    o.E[i] = Ef; o.pE[i] = pEf;
    const double td = 2.0 * (double)dHf - c0d;
    const double dE_H = dareas * ((0.5 * kcd * (td * td) + kgd * (double)dKf));
    const double dsum = ((double)Ef - dE_H) / dNd + (double)dEnb;
    const double lim = 0.5 * (double)dir_n;
    const double cl = (dsum > lim) ? lim : ((dsum < -lim) ? -lim : dsum);
    const float g = (float)(-1.0 * (double)((float)cl) * (1.0 - (double)pEf));              // :1213
    for (int a = 0; a < 3; ++a) o.dEdN[3 * i + a] = g * dir[a];
}

__global__ void k_neck_flags(const float *__restrict__ K, int M, float low, float high, int *__restrict__ flag) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < M) flag[i] = (K[i] < low) || (K[i] > high);
}
__global__ void k_compact(const int *__restrict__ flag, const int *__restrict__ off, int M, int *__restrict__ out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < M && flag[i]) out[off[i]] = i;
}

}  // namespace

static int exclusive_scan(nw_ctx *h, const int *in, int *out, int n) {
    size_t tmp = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tmp, in, out, n, h->stream);
    if (tmp > h->cub_tmp_bytes) { NW_CHECK(nw_alloc(h, (char **)&h->cub_tmp, tmp)); h->cub_tmp_bytes = tmp; }
    NW_CUDA(cub::DeviceScan::ExclusiveSum(h->cub_tmp, tmp, in, out, n, h->stream));
    h->launches += 2;
    return NW_OK;
}

static void curv_outputs(nw_ctx *h, CurvOut &co, size_t *offs) {
    const size_t M = (size_t)h->curvM;
    size_t o_ = 0;
    for (int k = 0; k < 12; ++k) { offs[k] = o_; o_ += (k < 9 ? 1 : 3) * M; }
    float *out = h->cvOut;
    co.k0 = out + offs[0]; co.k1 = out + offs[1]; co.H = out + offs[2]; co.K = out + offs[3]; co.dH = out + offs[4];
    co.dK = out + offs[5]; co.E = out + offs[6]; co.pE = out + offs[7]; co.dEnb = out + offs[8];
    co.e0 = out + offs[9]; co.e1 = out + offs[10]; co.dEdN = out + offs[11];
    co.n_deleted = (int *)(out + 18 * M);              // one counter behind the 18 M floats: comes back with the same copy
}

int nw_curvature_relaunch(nw_ctx *h) {
    NW_ARG(h->cvV && h->curvM > 0, "curvature: call nw_curvature_grad first");
    CurvOut co;
    size_t offs[12];
    curv_outputs(h, co, offs);
    k_curvature<<<nw_grid(h->curvM, NW_CURV_BLOCK), NW_CURV_BLOCK, 0, h->stream>>>((const VertRec *)h->cvV, (const FaceRec *)h->cvF, (const HeRec *)h->cvH,
                                                                h->curvM, h->cv_dN, h->cv_kc, h->cv_kg, h->cv_c0, h->cvJ, h->cvOff,
                                                                h->cv_seed, co);
    NW_LAUNCH_CHECK();
    return NW_OK;
}

// rows [a, b) of one output array: plain copy, or (masked) only the rows of live vertices
static void copy_rows(float *dst, const float *src, size_t a, size_t b, int width, const char *vertex_records) {
    if (!vertex_records) { memcpy(dst + a * width, src + a * width, (b - a) * width * sizeof(float)); return; }
    for (size_t i = a; i < b; ++i) {
        int he;
        memcpy(&he, vertex_records + i * sizeof(VertRec) + offsetof(VertRec, halfedge), sizeof(int));
        if (he != -1) memcpy(dst + i * width, src + i * width, width * sizeof(float));
    }
}

extern "C" int nw_curvature_grad(nw_ctx *h, const void *vertices, const void *faces, const void *halfedges, int n_vertices,
                                 int n_faces, int n_halfedges, float dN, float skip_prob, float *k_0, float *k_1, float *e_0,
                                 float *e_1, float *H, float *K, float *dH, float *dK, float *E, float *pE, float *dE_neighbors,
                                 float kc, float kg, float c0, float *dEdN, const double *jitter_u, uint64_t jitter_seed) {
    if (!h) return NW_ERR_ARG;
    NW_ARG(vertices && faces && halfedges && n_vertices > 0 && n_faces > 0 && n_halfedges > 0, "nw_curvature_grad: empty mesh");
    NW_ARG(skip_prob == 0.0f, "nw_curvature_grad: skip_prob must be 0 (the only value the reference passes)");
    NW_ARG(k_0 && k_1 && e_0 && e_1 && H && K && dH && dK && E && pE && dE_neighbors && dEdN, "nw_curvature_grad: NULL output");
    NW_CUDA(cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    const int M = n_vertices;
    int *flag = nullptr;
    // device copies are grow-only members: remove_necks calls this once per remesh block (_membrane_mesh.pyx:1212)
    NW_CHECK(nw_alloc(h, (VertRec **)&h->cvV, (size_t)M)); NW_CHECK(nw_alloc(h, (FaceRec **)&h->cvF, (size_t)n_faces));
    NW_CHECK(nw_alloc(h, (HeRec **)&h->cvH, (size_t)n_halfedges)); NW_CHECK(nw_alloc(h, &h->cvOut, (size_t)18 * M + 4));
    nw_free(&h->cvJ); nw_free(&h->cvOff);
    h->curvM = M; h->cv_dN = dN; h->cv_kc = kc; h->cv_kg = kg; h->cv_c0 = c0; h->cv_seed = (unsigned long long)jitter_seed;
    // the three record arrays go up through the pinned multi-lane path (xfer.cu), back to back on the handle's stream
    const nw_h2d_job up[3] = {{h->cvV, vertices, sizeof(VertRec) * (size_t)M, 4}, {h->cvF, faces, sizeof(FaceRec) * (size_t)n_faces, 4},
                              {h->cvH, halfedges, sizeof(HeRec) * (size_t)n_halfedges, 4}};
    NW_CHECK(nw_h2d_many(h, up, 3));
    CurvOut co;
    size_t offs[12];
    curv_outputs(h, co, offs);
    NW_CUDA(cudaMemsetAsync(co.n_deleted, 0, sizeof(int), s));
    if (jitter_u) {
        NW_CHECK(nw_alloc(h, &flag, (size_t)M)); NW_CHECK(nw_alloc(h, &h->cvOff, (size_t)M));
        k_valid_flags<<<nw_grid(M, 256), 256, 0, s>>>((const VertRec *)h->cvV, M, flag);
        h->launches++;
        int rc = exclusive_scan(h, flag, h->cvOff, M);
        int last_off = 0, last_flag = 0;
        if (rc == NW_OK) {
            cudaMemcpyAsync(&last_off, h->cvOff + M - 1, sizeof(int), cudaMemcpyDeviceToHost, s);
            cudaMemcpyAsync(&last_flag, flag + M - 1, sizeof(int), cudaMemcpyDeviceToHost, s);
            cudaStreamSynchronize(s);
        }
        nw_free(&flag);
        NW_CHECK(rc);
        const size_t nj = 3 * (size_t)(last_off + last_flag);
        NW_CHECK(nw_alloc(h, &h->cvJ, nj + 1));
        NW_CUDA(cudaMemcpyAsync(h->cvJ, jitter_u, sizeof(double) * nj, cudaMemcpyHostToDevice, s));
    }
    NW_CHECK(nw_curvature_relaunch(h));
    // ONE device->host copy of all 18 M output floats (+ the deleted-row counter) into the handle's pinned buffer, then
    // a threaded scatter into the caller's twelve arrays.  k0, k1, e0, e1 of deleted vertices keep the caller's values
    // (the reference leaves them untouched, membrane_mesh_utils.c:962-973): those four arrays are copied row by row,
    // skipping rows whose record has halfedge == -1, only when the kernel met such a row at all.
    const size_t out_bytes = sizeof(float) * 18 * (size_t)M + sizeof(int);
    if (h->pin_bytes < out_bytes) {
        if (h->pin_host) cudaFreeHost(h->pin_host);
        h->pin_host = nullptr; h->pin_bytes = 0;
        NW_CUDA(cudaHostAlloc((void **)&h->pin_host, out_bytes + out_bytes / 4, cudaHostAllocDefault));
        h->pin_bytes = out_bytes + out_bytes / 4;
    }
    h->pin_fresh = false;                       // the buffer no longer holds the positions
    NW_CUDA(cudaMemcpyAsync(h->pin_host, h->cvOut, out_bytes, cudaMemcpyDeviceToHost, s));
    NW_CUDA(cudaStreamSynchronize(s));
    const float *src = (const float *)h->pin_host;
    int n_deleted = 0;
    memcpy(&n_deleted, src + 18 * (size_t)M, sizeof(int));
    float *host_out[12] = {k_0, k_1, H, K, dH, dK, E, pE, dE_neighbors, e_0, e_1, dEdN};
    const char *recs = n_deleted > 0 ? (const char *)vertices : nullptr;
    auto part = [&](size_t a, size_t b) {
        for (int k = 0; k < 12; ++k) {
            const bool keep_deleted = (k == 0 || k == 1 || k == 9 || k == 10);
            copy_rows(host_out[k], src + offs[k], a, b, k < 9 ? 1 : 3, keep_deleted ? recs : nullptr);
        }
    };
    const size_t nt = (size_t)M < 65536 ? 1 : std::min<size_t>(8, std::max(1u, std::thread::hardware_concurrency() / 2));
    std::vector<std::thread> th;
    for (size_t t = 1; t < nt; ++t) th.emplace_back(part, (size_t)M * t / nt, (size_t)M * (t + 1) / nt);
    part(0, (size_t)M / nt);
    for (auto &t : th) t.join();
    h->curvK = co.K;       // stays on the device for the neck criterion
    return NW_OK;
}

extern "C" int nw_neck_candidates(nw_ctx *h, float low, float high, int32_t *idx, int *n) {
    if (!h) return NW_ERR_ARG;
    NW_ARG(h->curvK && h->curvM > 0, "nw_neck_candidates: call nw_curvature_grad first");
    NW_ARG(n != nullptr, "nw_neck_candidates: n is NULL");
    NW_CUDA(cudaSetDevice(h->device));
    const int M = h->curvM;
    int *flag = nullptr, *off = nullptr, *out = nullptr;
    NW_CHECK(nw_alloc(h, &flag, (size_t)M)); NW_CHECK(nw_alloc(h, &off, (size_t)M)); NW_CHECK(nw_alloc(h, &out, (size_t)M));
    k_neck_flags<<<nw_grid(M, 256), 256, 0, h->stream>>>(h->curvK, M, low, high, flag);
    NW_LAUNCH_CHECK();
    int rc = exclusive_scan(h, flag, off, M);
    if (rc == NW_OK) {
        k_compact<<<nw_grid(M, 256), 256, 0, h->stream>>>(flag, off, M, out);
        h->launches++;
        int lo = 0, lf = 0;
        cudaMemcpyAsync(&lo, off + M - 1, sizeof(int), cudaMemcpyDeviceToHost, h->stream);
        cudaMemcpyAsync(&lf, flag + M - 1, sizeof(int), cudaMemcpyDeviceToHost, h->stream);
        cudaStreamSynchronize(h->stream);
        *n = lo + lf;
        if (idx && *n > 0) cudaMemcpy(idx, out, sizeof(int) * (*n), cudaMemcpyDeviceToHost);
    }
    nw_free(&flag); nw_free(&off); nw_free(&out);
    return rc;
}

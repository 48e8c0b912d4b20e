// closest.cuh -- the exact point-to-triangle routine of surface.cu (nw_surface_distance) and hausdorff.cu
// (nw_hausdorff_bounds): fp64, one fixed sequence of operations.  Both files are compiled with -fmad=false, so the operations
// are exactly the written ones and tests/surface_oracle.py (closest_point_region) restates them bit for bit.
#pragma once
#include <cfloat>
#include <cuda_runtime.h>

namespace {

// ---- exact point-to-triangle distance (fp64, fixed operation order; restated in tests/surface_oracle.py) -------------------
struct D3 { double x, y, z; };
__device__ __forceinline__ D3 d3(const float4 v) { return D3{(double)v.x, (double)v.y, (double)v.z}; }
__device__ __forceinline__ D3 sub(const D3 a, const D3 b) { return D3{a.x - b.x, a.y - b.y, a.z - b.z}; }
__device__ __forceinline__ double dot(const D3 a, const D3 b) { return (a.x * b.x + a.y * b.y) + a.z * b.z; }
__device__ __forceinline__ D3 axpy(const D3 a, const double t, const D3 e) { return D3{a.x + t * e.x, a.y + t * e.y, a.z + t * e.z}; }
__device__ __forceinline__ double dist2(const D3 p, const D3 c) { const D3 d = sub(p, c); return dot(d, d); }

// R: also name the feature the closest point lies on (nw_surface_signed_distance), in r.  Region codes: 0 the interior,
// 1 + k corner k, 4 + k the edge from corner k to corner k + 1 (mod 3).  The operations, and so the points, do not depend on R.
#define NW_REGION_CORNER(k) (1 + (k))
#define NW_REGION_EDGE(k) (4 + (k))
// the segment p0 -> p1 as edge k of a triangle
template <bool R>
__device__ __forceinline__ D3 closest_on_segment(const D3 p, const D3 p0, const D3 p1, const int k, int &r) {
    const D3 e = sub(p1, p0);
    const double ee = dot(e, e);
    double t = ee > 0.0 ? dot(sub(p, p0), e) / ee : 0.0;
    t = fmin(fmax(t, 0.0), 1.0);
    if (R) r = t == 0.0 ? NW_REGION_CORNER(k) : t == 1.0 ? NW_REGION_CORNER((k + 1) % 3) : NW_REGION_EDGE(k);
    return axpy(p0, t, e);
}
// a zero-area triangle is the union of its three edges: the closest of them, in the order ab, bc, ca (first wins ties)
template <bool R>
__device__ __noinline__ D3 closest_on_edges(const D3 p, const D3 a, const D3 b, const D3 c, int &r) {
    int rk;
    D3 best = closest_on_segment<R>(p, a, b, 0, r);
    double bd = dist2(p, best);
    D3 k = closest_on_segment<R>(p, b, c, 1, rk);
    double kd = dist2(p, k);
    if (kd < bd) { best = k; bd = kd; if (R) r = rk; }
    k = closest_on_segment<R>(p, c, a, 2, rk);
    kd = dist2(p, k);
    if (kd < bd) { best = k; if (R) r = rk; }
    return best;
}
// Ericson's region test.  Degenerate: the cross product ab x ac is exactly zero, or (rounding of a nearly degenerate
// triangle) the interior case finds no positive barycentric denominator.
template <bool R>
__device__ __forceinline__ D3 closest_on_triangle(const D3 p, const D3 a, const D3 b, const D3 c, int &r) {
    const D3 ab = sub(b, a), ac = sub(c, a);
    if (ab.y * ac.z - ab.z * ac.y == 0.0 && ab.z * ac.x - ab.x * ac.z == 0.0 && ab.x * ac.y - ab.y * ac.x == 0.0)
        return closest_on_edges<R>(p, a, b, c, r);
    const D3 ap = sub(p, a);
    const double d1 = dot(ab, ap), d2 = dot(ac, ap);
    if (d1 <= 0.0 && d2 <= 0.0) { r = NW_REGION_CORNER(0); return a; }
    const D3 bp = sub(p, b);
    const double d3 = dot(ab, bp), d4 = dot(ac, bp);
    if (d3 >= 0.0 && d4 <= d3) { r = NW_REGION_CORNER(1); return b; }
    const double vc = d1 * d4 - d3 * d2;
    if (vc <= 0.0 && d1 >= 0.0 && d3 <= 0.0) { r = NW_REGION_EDGE(0); return axpy(a, d1 / (d1 - d3), ab); }
    const D3 cp = sub(p, c);
    const double d5 = dot(ab, cp), d6 = dot(ac, cp);
    if (d6 >= 0.0 && d5 <= d6) { r = NW_REGION_CORNER(2); return c; }
    const double vb = d5 * d2 - d1 * d6;
    if (vb <= 0.0 && d2 >= 0.0 && d6 <= 0.0) { r = NW_REGION_EDGE(2); return axpy(a, d2 / (d2 - d6), ac); }
    const double va = d3 * d6 - d5 * d4;
    if (va <= 0.0 && (d4 - d3) >= 0.0 && (d5 - d6) >= 0.0) {
        r = NW_REGION_EDGE(1);
        return axpy(b, (d4 - d3) / ((d4 - d3) + (d5 - d6)), sub(c, b));
    }
    const double s = va + vb + vc;
    if (!(s > 0.0)) return closest_on_edges<R>(p, a, b, c, r);
    const double denom = 1.0 / s;
    const double v = vb * denom, w = vc * denom;
    r = 0;
    return D3{(a.x + ab.x * v) + ac.x * w, (a.y + ab.y * v) + ac.y * w, (a.z + ab.z * v) + ac.z * w};
}
__device__ __forceinline__ D3 closest_on_triangle(const D3 p, const D3 a, const D3 b, const D3 c) {
    int r;
    return closest_on_triangle<false>(p, a, b, c, r);
}

__device__ __forceinline__ bool finite4(const float4 v) { return fabsf(v.x) <= FLT_MAX && fabsf(v.y) <= FLT_MAX && fabsf(v.z) <= FLT_MAX; }

}  // namespace

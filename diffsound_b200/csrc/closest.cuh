// Closest point of a triangle to a query point, in fp64 from fp32 corners: the vertex / edge / face region analysis of
// Ericson, Real-Time Collision Detection 5.1.5.  Shared by the triangle-mesh SDF (sdf.cu: its gradient) and the modal
// gains (gains.cu: strike points put on the boundary of a tet mesh).  Explicit round-to-nearest intrinsics (no
// contraction into FMA), so every caller evaluates bit-identical values.
#pragma once
#include <cuda_runtime.h>

namespace ds {

__device__ __forceinline__ double dsub(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ double dadd(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double dmul(double a, double b) { return __dmul_rn(a, b); }

struct D3 {
    double x, y, z;
};
__device__ __forceinline__ D3 d3(float4 v) { return {(double)v.x, (double)v.y, (double)v.z}; }
__device__ __forceinline__ D3 sub3(D3 a, D3 b) { return {dsub(a.x, b.x), dsub(a.y, b.y), dsub(a.z, b.z)}; }
__device__ __forceinline__ double dot3(D3 a, D3 b) { return dadd(dadd(dmul(a.x, b.x), dmul(a.y, b.y)), dmul(a.z, b.z)); }
__device__ __forceinline__ D3 axpy3(D3 a, double t, D3 d) { return {dadd(a.x, dmul(t, d.x)), dadd(a.y, dmul(t, d.y)), dadd(a.z, dmul(t, d.z))}; }
__device__ __forceinline__ double dist2(D3 p, D3 q) { const D3 d = sub3(p, q); return dot3(d, d); }

// closest point of the segment [a, b] to p and its parameter t (c = a + t (b - a))
__device__ __forceinline__ D3 seg_closest(D3 p, D3 a, D3 b, double& t) {
    const D3 ab = sub3(b, a);
    const double l2 = dot3(ab, ab);
    t = l2 > 0.0 ? dot3(sub3(p, a), ab) / l2 : 0.0;
    t = fmin(fmax(t, 0.0), 1.0);
    return axpy3(a, t, ab);
}

// closest point of the union of the three edges, the first of (ab, bc, ca) on ties, with its weights on (a, b, c)
__device__ __forceinline__ D3 edges_closest(D3 p, D3 a, D3 b, D3 c, double (&w)[3]) {
    double t0, t1, t2;
    const D3 c0 = seg_closest(p, a, b, t0), c1 = seg_closest(p, b, c, t1), c2 = seg_closest(p, c, a, t2);
    const double e0 = dist2(p, c0), e1 = dist2(p, c1), e2 = dist2(p, c2);
    if (e0 <= e1 && e0 <= e2) { w[0] = 1.0 - t0; w[1] = t0; w[2] = 0.0; return c0; }
    if (e1 <= e2) { w[0] = 0.0; w[1] = 1.0 - t1; w[2] = t1; return c1; }
    w[0] = t2; w[1] = 0.0; w[2] = 1.0 - t2;
    return c2;
}

// closest point of triangle (A, B, C) to p and its barycentric weights w on (A, B, C); A.w != 0 marks a degenerate face
// (the union of its three edges).  The region is read off the weights: one nonzero weight is a vertex, two an edge,
// three the face.  sdf.cu's tri_d2 follows the same branches, so dist2(p, c) is the value it returns.
__device__ __forceinline__ D3 tri_closest(D3 p, float4 A4, float4 B4, float4 C4, double (&w)[3]) {
    const D3 a = d3(A4), b = d3(B4), c = d3(C4);
    if (A4.w != 0.f) return edges_closest(p, a, b, c, w);
    w[0] = w[1] = w[2] = 0.0;
    const D3 ab = sub3(b, a), ac = sub3(c, a), ap = sub3(p, a);
    const double d1 = dot3(ab, ap), d2 = dot3(ac, ap);
    if (d1 <= 0.0 && d2 <= 0.0) { w[0] = 1.0; return a; }
    const D3 bp = sub3(p, b);
    const double d3_ = dot3(ab, bp), d4 = dot3(ac, bp);
    if (d3_ >= 0.0 && d4 <= d3_) { w[1] = 1.0; return b; }
    const double vc = dsub(dmul(d1, d4), dmul(d3_, d2));
    if (vc <= 0.0 && d1 >= 0.0 && d3_ <= 0.0) {
        const double t = d1 / dsub(d1, d3_);
        w[0] = 1.0 - t; w[1] = t;
        return axpy3(a, t, ab);
    }
    const D3 cp = sub3(p, c);
    const double d5 = dot3(ab, cp), d6 = dot3(ac, cp);
    if (d6 >= 0.0 && d5 <= d6) { w[2] = 1.0; return c; }
    const double vb = dsub(dmul(d5, d2), dmul(d1, d6));
    if (vb <= 0.0 && d2 >= 0.0 && d6 <= 0.0) {
        const double t = d2 / dsub(d2, d6);
        w[0] = 1.0 - t; w[2] = t;
        return axpy3(a, t, ac);
    }
    const double va = dsub(dmul(d3_, d6), dmul(d5, d4));
    const double e43 = dsub(d4, d3_), e56 = dsub(d5, d6);
    if (va <= 0.0 && e43 >= 0.0 && e56 >= 0.0) {
        const double t = e43 / dadd(e43, e56);
        w[1] = 1.0 - t; w[2] = t;
        return axpy3(b, t, sub3(c, b));
    }
    const double den = dadd(dadd(va, vb), vc);
    if (!(den > 0.0)) return edges_closest(p, a, b, c, w);
    const double v = vb / den, ww = vc / den;
    w[0] = 1.0 - v - ww; w[1] = v; w[2] = ww;
    return axpy3(axpy3(a, v, ab), ww, ac);
}

}  // namespace ds

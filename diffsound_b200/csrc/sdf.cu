// Signed distance from query points to a triangle mesh: the open3d RaycastingScene sampling of apply_sdf(path) in the
// reference (src/dmtet/geometry/dmtet_thickness.py:301-314; SURVEY.md section 8f-4).
//
// Contract (include/diffsound_sm100.h, ds_mesh_sdf):
//   * |sdf(p)| = Euclidean distance from p to the closest point of the triangle set: closest point on each triangle by the
//     vertex / edge / face region analysis (Ericson, Real-Time Collision Detection 5.1.5), evaluated in fp64 from the fp32
//     inputs, rounded once to fp32.  Degenerate faces (zero cross product) are the union of their three edges.
//   * sign: positive inside, negative outside, by the parity of ray crossings (face orientation does not matter), majority
//     of three fixed rays that are not axis-aligned.  Ray / triangle: the watertight test of Woop, Benthin & Wald
//     (JCGT 2(1), 2013) in fp32 with a per-edge fp64 recomputation when an edge function is exactly 0; a crossing through
//     an edge or a vertex is assigned to exactly one triangle of a closed mesh by a top-left rule on the projected edge
//     direction, taken in the triangle's counter-clockwise order so that the choice does not depend on face orientation.
//     Degenerate faces and faces seen edge-on never count.  A point at distance 0 gives +0.
//
// BVH mode: Morton codes of the triangle centroids (k_bbox / k_morton_codes of precond32.cu), CUB radix sort, binary
// radix tree (Karras, HPG 2012; equal codes ordered by index), boxes refit bottom-up with per-node arrival counters.
// Each internal node stores the boxes of its two children.  Node boxes are padded by 2^-16 of the largest coordinate
// magnitude of mesh and queries: that margin exceeds the fp32 rounding of the ray test's sheared coordinates and the fp64
// rounding of the distances, so a box is never pruned while it holds a triangle the brute-force loop would count
// (nearest: pruned only when its squared box distance is strictly greater than the best; rays: conservative slab test
// of Ize 2013, t_max scaled by 1 + 2 gamma_3).  The minimum and the crossing counts then do not depend on the hierarchy
// or on the visit order, and BVH and brute-force outputs are bitwise equal.  Queries run in Morton order of the points.
// Per-triangle arithmetic uses explicit round-to-nearest intrinsics (no contraction into FMA), so both kernels evaluate
// bit-identical per-triangle values.
//
// Gradient (ds_mesh_sdf_nearest, ds_mesh_sdf_backward): the query kernels, instantiated to record the nearest face (the
// lowest original index among faces at exactly the minimum, in both modes; ds_mesh_sdf runs the non-recording
// instantiations, whose code is unchanged).  k_sdf_backward recomputes the closest point c = sum b_k v_k of that face by
// the region analysis of tri_d2 and gives d sdf / d p = s u, d sdf / d v_k = -s b_k u (u = (p - c) / |p - c|; the
// envelope theorem, so one formula for the face, edge and vertex regions).  The corner terms are reduced onto the
// vertices in a fixed order (stable radix sort of the 3P corner vertex ids, fp64 sums per run): bitwise reproducible.
//
// Winding number (ds_mesh_winding_number, ds_mesh_sdf_winding): w(p) = sum of the faces' oriented solid angles / 4 pi
// (Jacobson, Kavan & Sorkine-Hornung 2013), each face's exact term 2 atan2(num, den) (Van Oosterom & Strackee) in fp64
// from its sorted corners, times the orientation of the sort (C.w of the gathered triangle, k_sdf_gather<true>).  Brute
// force: every face in face order.  BVH (Barill, Dickson, Schmidt, Levin & Jacobson 2018): a radix tree built as for
// ds_mesh_sdf but from the centroids of the sorted corners (k_sdf_centroids<true>), so that the tree, and the order of
// every sum over it, do not depend on how the faces are written (flipped faces give exactly -w, re-indexed or unshared
// vertices the same bits, in both modes); k_sdf_wn_moments forms each node's moments bottom-up (child 0 + child 1,
// fp64), and k_sdf_winding_bvh replaces a subtree far from the point by its far-field expansion (WN_BETA).
// ds_mesh_sdf_winding writes +1 / -1 (|w| >= 1/2 in fp64) to sdf_out and runs the
// query kernels instantiated WIND: the same nearest-face search, the sign taken from sdf_out instead of the rays.
#include "common.cuh"
#include "../../include/diffsound_sm100.h"
#include "kernels.cuh"
#include "closest.cuh"
#include <cub/cub.cuh>
#include <cfloat>
#include <climits>

namespace ds {

namespace {

constexpr int SDF_BLOCK = 64;      // query threads per CTA (the traversal stacks live in shared memory)
constexpr int SDF_STACK = 64;      // > depth of a radix tree over 30-bit codes + 32-bit indices
constexpr int SDF_TILE = 256;      // triangles per shared-memory tile of the brute-force kernel

// three fixed ray directions, none axis-aligned, no two components equal in magnitude
__constant__ float c_ray_dir[3][3] = {{0.3090f, 0.5878f, 0.7470f}, {-0.8024f, 0.2590f, 0.5375f}, {0.4531f, -0.8127f, -0.3664f}};

// internal node: b[0..5] = lo xyz, hi xyz of child 0, b[6..11] of child 1; child >= 0 internal node, < 0 leaf ~index
struct __align__(16) BvhNode {
    float b[12];
    int child[2];
    int pad[2];
};

// squared distance from p to the segment [a, b] (a point when a == b)
__device__ __forceinline__ double seg_d2(D3 p, D3 a, D3 b) {
    const D3 ab = sub3(b, a);
    const double l2 = dot3(ab, ab);
    double t = l2 > 0.0 ? dot3(sub3(p, a), ab) / l2 : 0.0;
    t = fmin(fmax(t, 0.0), 1.0);
    return dist2(p, axpy3(a, t, ab));
}

// squared distance from p to triangle (A, B, C); A.w != 0 marks a degenerate face (its three edges)
__device__ __forceinline__ double tri_d2(D3 p, float4 A4, float4 B4, float4 C4) {
    const D3 a = d3(A4), b = d3(B4), c = d3(C4);
    if (A4.w != 0.f) return fmin(fmin(seg_d2(p, a, b), seg_d2(p, b, c)), seg_d2(p, c, a));
    const D3 ab = sub3(b, a), ac = sub3(c, a), ap = sub3(p, a);
    const double d1 = dot3(ab, ap), d2 = dot3(ac, ap);
    if (d1 <= 0.0 && d2 <= 0.0) return dist2(p, a);
    const D3 bp = sub3(p, b);
    const double d3_ = dot3(ab, bp), d4 = dot3(ac, bp);
    if (d3_ >= 0.0 && d4 <= d3_) return dist2(p, b);
    const double vc = dsub(dmul(d1, d4), dmul(d3_, d2));
    if (vc <= 0.0 && d1 >= 0.0 && d3_ <= 0.0) return dist2(p, axpy3(a, d1 / dsub(d1, d3_), ab));
    const D3 cp = sub3(p, c);
    const double d5 = dot3(ab, cp), d6 = dot3(ac, cp);
    if (d6 >= 0.0 && d5 <= d6) return dist2(p, c);
    const double vb = dsub(dmul(d5, d2), dmul(d1, d6));
    if (vb <= 0.0 && d2 >= 0.0 && d6 <= 0.0) return dist2(p, axpy3(a, d2 / dsub(d2, d6), ac));
    const double va = dsub(dmul(d3_, d6), dmul(d5, d4));
    const double e43 = dsub(d4, d3_), e56 = dsub(d5, d6);
    if (va <= 0.0 && e43 >= 0.0 && e56 >= 0.0) return dist2(p, axpy3(b, e43 / dadd(e43, e56), sub3(c, b)));
    const double den = dadd(dadd(va, vb), vc);
    if (!(den > 0.0)) return fmin(fmin(seg_d2(p, a, b), seg_d2(p, b, c)), seg_d2(p, c, a));   // cancellation on a sliver
    const double v = vb / den, w = vc / den;
    return dist2(p, axpy3(axpy3(a, v, ab), w, ac));
}

// ray from o along c_ray_dir[r], in the sheared frame of Woop et al.: kz = dominant axis, S = shear
struct Ray {
    float o[3];
    float Sx, Sy, Sz;
    float inv[3];
    int kx, ky, kz;
};
__device__ __forceinline__ float sel3(float4 v, int k) { return k == 0 ? v.x : (k == 1 ? v.y : v.z); }
__device__ __forceinline__ float sel3(const float* v, int k) { return k == 0 ? v[0] : (k == 1 ? v[1] : v[2]); }

__device__ __forceinline__ Ray make_ray(float px, float py, float pz, int r) {
    Ray R;
    R.o[0] = px; R.o[1] = py; R.o[2] = pz;
    const float dx = c_ray_dir[r][0], dy = c_ray_dir[r][1], dz = c_ray_dir[r][2];
    const float ax = fabsf(dx), ay = fabsf(dy), az = fabsf(dz);
    R.kz = (ax >= ay && ax >= az) ? 0 : (ay >= az ? 1 : 2);
    R.kx = R.kz == 2 ? 0 : R.kz + 1;
    R.ky = R.kx == 2 ? 0 : R.kx + 1;
    const float d[3] = {dx, dy, dz};
    const float dkz = sel3(d, R.kz);
    R.Sx = sel3(d, R.kx) / dkz;
    R.Sy = sel3(d, R.ky) / dkz;
    R.Sz = 1.0f / dkz;
    R.inv[0] = 1.0f / dx; R.inv[1] = 1.0f / dy; R.inv[2] = 1.0f / dz;
    return R;
}

struct P2 {
    float x, y, z;
};
__device__ __forceinline__ P2 shear(const Ray& R, float4 V) {
    const float vx = __fsub_rn(sel3(V, R.kx), sel3(R.o, R.kx));
    const float vy = __fsub_rn(sel3(V, R.ky), sel3(R.o, R.ky));
    const float vz = __fsub_rn(sel3(V, R.kz), sel3(R.o, R.kz));
    return {__fsub_rn(vx, __fmul_rn(R.Sx, vz)), __fsub_rn(vy, __fmul_rn(R.Sy, vz)), __fmul_rn(R.Sz, vz)};
}
// 2-D edge function of the directed edge P -> Q at the origin (twice the signed area of O, P, Q); fp64 when the fp32
// value is exactly 0.  A shared edge gets exactly negated values in its two triangles.
__device__ __forceinline__ double edge_fn(P2 P, P2 Q) {
    const float e = __fsub_rn(__fmul_rn(P.x, Q.y), __fmul_rn(P.y, Q.x));
    if (e != 0.0f) return (double)e;
    return dsub(dmul((double)P.x, (double)Q.y), dmul((double)P.y, (double)Q.x));
}
// a zero edge function counts as inside only for edges whose counter-clockwise direction is "top-left"
__device__ __forceinline__ bool top_left(P2 P, P2 Q, bool ccw) {
    const float dx = ccw ? __fsub_rn(Q.x, P.x) : __fsub_rn(P.x, Q.x);
    const float dy = ccw ? __fsub_rn(Q.y, P.y) : __fsub_rn(P.y, Q.y);
    return dy > 0.0f || (dy == 0.0f && dx < 0.0f);
}

// 1 when the ray crosses triangle (A, B, C) at t > 0
__device__ __forceinline__ int ray_hit(const Ray& R, float4 A4, float4 B4, float4 C4) {
    if (A4.w != 0.f) return 0;
    const P2 A = shear(R, A4), B = shear(R, B4), C = shear(R, C4);
    const double e0 = edge_fn(B, C), e1 = edge_fn(C, A), e2 = edge_fn(A, B);
    if ((e0 < 0.0 || e1 < 0.0 || e2 < 0.0) && (e0 > 0.0 || e1 > 0.0 || e2 > 0.0)) return 0;
    const double det = dadd(dadd(e0, e1), e2);
    if (det == 0.0) return 0;
    const bool ccw = det > 0.0;
    if (e0 == 0.0 && !top_left(B, C, ccw)) return 0;
    if (e1 == 0.0 && !top_left(C, A, ccw)) return 0;
    if (e2 == 0.0 && !top_left(A, B, ccw)) return 0;
    const double T = dadd(dadd(dmul(e0, (double)A.z), dmul(e1, (double)B.z)), dmul(e2, (double)C.z));
    return (ccw ? T > 0.0 : T < 0.0) ? 1 : 0;
}

__device__ __forceinline__ double box_d2(double px, double py, double pz, const float* lo, const float* hi) {
    const double dx = fmax(fmax((double)lo[0] - px, px - (double)hi[0]), 0.0);
    const double dy = fmax(fmax((double)lo[1] - py, py - (double)hi[1]), 0.0);
    const double dz = fmax(fmax((double)lo[2] - pz, pz - (double)hi[2]), 0.0);
    return dx * dx + dy * dy + dz * dz;
}
__device__ __forceinline__ bool ray_box(const Ray& R, const float* lo, const float* hi) {
    constexpr float gamma3 = 3.0f * FLT_EPSILON * 0.5f / (1.0f - 3.0f * FLT_EPSILON * 0.5f);
    float tn = -FLT_MAX, tf = FLT_MAX;
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        const float t0 = (lo[d] - R.o[d]) * R.inv[d], t1 = (hi[d] - R.o[d]) * R.inv[d];
        tn = fmaxf(tn, fminf(t0, t1));
        tf = fminf(tf, fmaxf(t0, t1));
    }
    tf *= 1.0f + 2.0f * gamma3;
    return tn <= tf && tf >= 0.0f;
}

__device__ __forceinline__ void load_node(const BvhNode* nodes, int n, float (&b)[12], int& c0, int& c1) {
    const float4* q = reinterpret_cast<const float4*>(nodes + n);
    const float4 v0 = __ldg(q), v1 = __ldg(q + 1), v2 = __ldg(q + 2);
    const int4 v3 = __ldg(reinterpret_cast<const int4*>(q + 3));
    b[0] = v0.x; b[1] = v0.y; b[2] = v0.z; b[3] = v0.w; b[4] = v1.x; b[5] = v1.y;
    b[6] = v1.z; b[7] = v1.w; b[8] = v2.x; b[9] = v2.y; b[10] = v2.z; b[11] = v2.w;
    c0 = v3.x;
    c1 = v3.y;
}

// ---- validation ------------------------------------------------------------------------------------------------
// bad[0] = first face with an index outside [0, V), bad[1] = first non-finite vertex, bad[2] = first non-finite point,
// bad[3] = first point whose nearest-face id (when given) is outside [0, F)
__global__ void k_sdf_validate(const float* __restrict__ verts, int64_t V, const int64_t* __restrict__ faces, int64_t F,
                               const float* __restrict__ pts, int64_t P, const int32_t* __restrict__ nearest,
                               unsigned long long* __restrict__ bad) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    if (nearest)
        for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < P; i += stride)
            if (nearest[i] < 0 || nearest[i] >= F) atomicMin(&bad[3], (unsigned long long)i);
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < 3 * F; i += stride) {
        const int64_t v = faces[i];
        if (v < 0 || v >= V) atomicMin(&bad[0], (unsigned long long)(i / 3));
    }
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < 3 * V; i += stride)
        if (!isfinite(verts[i])) atomicMin(&bad[1], (unsigned long long)(i / 3));
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < 3 * P; i += stride)
        if (!isfinite(pts[i])) atomicMin(&bad[2], (unsigned long long)(i / 3));
}

// ---- build -----------------------------------------------------------------------------------------------------
// corners of face f, sorted, with their vertex ids; v[0].w = 1 for a zero cross product.  Returns the orientation of the
// sorted corners relative to the face as written: +1 (even permutation) or -1 (odd)
__device__ __forceinline__ float sorted_face(const float* __restrict__ verts, const int64_t* __restrict__ faces, int64_t f,
                                            float4 (&v)[3], int64_t (&id)[3]) {
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        id[k] = faces[3 * f + k];
        v[k] = make_float4(verts[3 * id[k]], verts[3 * id[k] + 1], verts[3 * id[k] + 2], 0.f);
    }
    // corners in lexicographic order: the per-triangle arithmetic then does not depend on how the face was written
    // (orientation, first corner), so flipped or re-indexed meshes give bitwise equal results
    bool odd = false;
    auto cswap = [&](int i, int j) {
        const float4 a = v[i], b = v[j];
        const bool less = b.x < a.x || (b.x == a.x && (b.y < a.y || (b.y == a.y && b.z < a.z)));
        if (less) {
            v[i] = b; v[j] = a;
            const int64_t t = id[i]; id[i] = id[j]; id[j] = t;
            odd = !odd;
        }
    };
    cswap(0, 1);
    cswap(1, 2);
    cswap(0, 1);
    const D3 a = d3(v[0]), ab = sub3(d3(v[1]), a), ac = sub3(d3(v[2]), a);
    const double nx = dsub(dmul(ab.y, ac.z), dmul(ab.z, ac.y));
    const double ny = dsub(dmul(ab.z, ac.x), dmul(ab.x, ac.z));
    const double nz = dsub(dmul(ab.x, ac.y), dmul(ab.y, ac.x));
    v[0].w = (nx == 0.0 && ny == 0.0 && nz == 0.0) ? 1.f : 0.f;
    return odd ? -1.f : 1.f;
}

// cent[3 f ..] = centroid of face f in fp32, its corners summed in the order written.  SORTED: summed in lexicographic
// order instead (sorted_face), so the centroids, and with them the Morton order and the tree, do not depend on the face's
// orientation or first corner: the winding number's far-field sums are then bitwise odd under flipping every face
template <bool SORTED>
__global__ void k_sdf_centroids(const float* __restrict__ verts, const int64_t* __restrict__ faces, int64_t F,
                                float* __restrict__ cent) {
    const int64_t f = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (f >= F) return;
    if (SORTED) {
        float4 v[3];
        int64_t id[3];
        sorted_face(verts, faces, f, v, id);
        cent[3 * f] = (v[0].x + v[1].x + v[2].x) * (1.0f / 3.0f);
        cent[3 * f + 1] = (v[0].y + v[1].y + v[2].y) * (1.0f / 3.0f);
        cent[3 * f + 2] = (v[0].z + v[1].z + v[2].z) * (1.0f / 3.0f);
        return;
    }
    const int64_t a = faces[3 * f], b = faces[3 * f + 1], c = faces[3 * f + 2];
#pragma unroll
    for (int d = 0; d < 3; ++d) cent[3 * f + d] = (verts[3 * a + d] + verts[3 * b + d] + verts[3 * c + d]) * (1.0f / 3.0f);
}

// tri[3 i .. 3 i + 2] = corners of face order[i] (identity when order is NULL), sorted; A.w = 1 for a zero cross product,
// B.w = the bits of the original face index (read only by the face-recording BVH query, which loads B whole anyway);
// ORIENT: C.w = +1 / -1, the orientation of the sorted corners relative to the face as written (for the winding number)
template <bool ORIENT>
__global__ void k_sdf_gather(const float* __restrict__ verts, const int64_t* __restrict__ faces,
                             const uint32_t* __restrict__ order, int64_t F, float4* __restrict__ tri) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= F) return;
    const int64_t f = order ? (int64_t)order[i] : i;
    float4 v[3];
    int64_t id[3];
    const float o = sorted_face(verts, faces, f, v, id);
    if (ORIENT) v[2].w = o;
    v[1].w = __int_as_float((int)f);
    tri[3 * i] = v[0];
    tri[3 * i + 1] = v[1];
    tri[3 * i + 2] = v[2];
}

__device__ __forceinline__ int delta(const uint32_t* __restrict__ codes, int n, int i, int j) {
    if (j < 0 || j >= n) return -1;
    const uint32_t a = codes[i], b = codes[j];
    return a != b ? __clz(a ^ b) : 32 + __clz((uint32_t)(i ^ j));
}

// internal node i of the radix tree over n sorted codes (Karras 2012, algorithm 2); parent[] over node ids
// (internal j -> j, leaf k -> n - 1 + k), parent[0] = -1
__global__ void k_sdf_karras(const uint32_t* __restrict__ codes, int n, BvhNode* __restrict__ nodes, int* __restrict__ parent) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n - 1) return;
    const int d = delta(codes, n, i, i + 1) - delta(codes, n, i, i - 1) >= 0 ? 1 : -1;
    const int dmin = delta(codes, n, i, i - d);
    int lmax = 2;
    while (delta(codes, n, i, i + lmax * d) > dmin) lmax *= 2;
    int l = 0;
    for (int t = lmax / 2; t >= 1; t /= 2)
        if (delta(codes, n, i, i + (l + t) * d) > dmin) l += t;
    const int j = i + l * d;
    const int dnode = delta(codes, n, i, j);
    int s = 0, t = l;
    do {
        t = (t + 1) >> 1;
        if (delta(codes, n, i, i + (s + t) * d) > dnode) s += t;
    } while (t > 1);
    const int gamma = i + s * d + min(d, 0);
    const int left = min(i, j) == gamma ? ~gamma : gamma;
    const int right = max(i, j) == gamma + 1 ? ~(gamma + 1) : gamma + 1;
    nodes[i].child[0] = left;
    nodes[i].child[1] = right;
    parent[left < 0 ? n - 1 + ~left : left] = i;
    parent[right < 0 ? n - 1 + ~right : right] = i;
    if (i == 0) parent[0] = -1;
}

// bottom-up box refit: one thread per leaf; the second thread to reach a node continues with the union of its children
__global__ void k_sdf_refit(const float4* __restrict__ tri, int n, BvhNode* nodes, const int* __restrict__ parent,
                            int* __restrict__ arrived, const uint32_t* __restrict__ mm_v, const uint32_t* __restrict__ mm_p) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    float S = FLT_MIN;
#pragma unroll
    for (int d = 0; d < 6; ++d) S = fmaxf(S, fmaxf(fabsf(key_to_float(mm_v[d])), fabsf(key_to_float(mm_p[d]))));
    const float pad = S * (1.0f / 65536.0f);
    const float4 A = tri[3 * k], B = tri[3 * k + 1], C = tri[3 * k + 2];
    float lo[3] = {fminf(fminf(A.x, B.x), C.x), fminf(fminf(A.y, B.y), C.y), fminf(fminf(A.z, B.z), C.z)};
    float hi[3] = {fmaxf(fmaxf(A.x, B.x), C.x), fmaxf(fmaxf(A.y, B.y), C.y), fmaxf(fmaxf(A.z, B.z), C.z)};
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        lo[d] = __fsub_rd(lo[d], pad);
        hi[d] = __fadd_ru(hi[d], pad);
    }
    int enc = ~k;
    int p = parent[n - 1 + k];
    while (p >= 0) {
        const int slot = nodes[p].child[0] == enc ? 0 : 1;
        volatile float* b = nodes[p].b;
#pragma unroll
        for (int d = 0; d < 3; ++d) {
            b[6 * slot + d] = lo[d];
            b[6 * slot + 3 + d] = hi[d];
        }
        __threadfence();
        if (atomicAdd(&arrived[p], 1) == 0) return;
        __threadfence();
#pragma unroll
        for (int d = 0; d < 3; ++d) {
            lo[d] = fminf(b[d], b[6 + d]);
            hi[d] = fmaxf(b[3 + d], b[9 + d]);
        }
        enc = p;
        p = parent[p];
    }
}

// ---- queries ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ float signed_out(double best, int votes) {
    const float d = (float)sqrt(best);
    return d == 0.0f ? 0.0f : (votes >= 2 ? d : -d);
}

// REC: also write the nearest face to face_out, as an original face index (B.w of the Morton-ordered triangle, see
// k_sdf_gather); of several faces at exactly the same squared distance, the one with the lowest original index.  Boxes at a
// distance equal to the current best are visited, so every face reaching the final minimum is evaluated.
// WIND: no rays; out[q] holds +1 / -1 on entry (inside / outside by the winding number, k_sdf_winding_*) and the sign
// is taken from it.  The nearest-face search is the same code in every instantiation.
template <bool REC, bool WIND = false>
__global__ void __launch_bounds__(SDF_BLOCK)
k_sdf_query_bvh(const float4* __restrict__ tri, const BvhNode* __restrict__ nodes, int F, const float* __restrict__ pts,
                const uint32_t* __restrict__ order, int64_t P, float* __restrict__ out, int32_t* __restrict__ face_out) {
    __shared__ int s_node[SDF_STACK][SDF_BLOCK];
    __shared__ float s_d2[SDF_STACK][SDF_BLOCK];
    const int64_t i = blockIdx.x * (int64_t)SDF_BLOCK + threadIdx.x;
    if (i >= P) return;
    const int tid = threadIdx.x;
    const int64_t q = order[i];
    const float px = pts[3 * q], py = pts[3 * q + 1], pz = pts[3 * q + 2];
    const D3 p = {(double)px, (double)py, (double)pz};
    float b[12];
    int c[2];
    // nearest triangle
    double best = INFINITY;
    int bestf = INT_MAX;
    if (F == 1) {
        best = tri_d2(p, tri[0], tri[1], tri[2]);
        bestf = 0;
    } else {
        int sp = 0, node = 0;
        for (;;) {
            load_node(nodes, node, b, c[0], c[1]);
            double bd[2] = {box_d2(p.x, p.y, p.z, b, b + 3), box_d2(p.x, p.y, p.z, b + 6, b + 9)};
            bool go[2] = {bd[0] <= best, bd[1] <= best};
#pragma unroll
            for (int s = 0; s < 2; ++s)
                if (go[s] && c[s] < 0) {
                    const int t = ~c[s];
                    const float4 B = tri[3 * t + 1];
                    const double d2 = tri_d2(p, tri[3 * t], B, tri[3 * t + 2]);
                    if (REC) {
                        const int f = __float_as_int(B.w);
                        if (d2 < best || (d2 == best && f < bestf)) {
                            best = d2;
                            bestf = f;
                        }
                    } else {
                        best = fmin(best, d2);
                    }
                    go[s] = false;
                }
            if (go[0] && go[1]) {
                const bool r_first = bd[1] < bd[0];      // nearer child first, the other one on the stack
                s_node[sp][tid] = r_first ? c[0] : c[1];
                s_d2[sp][tid] = __double2float_rd(r_first ? bd[0] : bd[1]);
                ++sp;
                node = r_first ? c[1] : c[0];
                continue;
            }
            if (go[0] || go[1]) {
                node = go[0] ? c[0] : c[1];
                continue;
            }
            node = -1;
            while (sp > 0) {
                --sp;
                if ((double)s_d2[sp][tid] <= best) {
                    node = s_node[sp][tid];
                    break;
                }
            }
            if (node < 0) break;
        }
    }
    // crossing parity of the three rays
    int votes = 0;
    if constexpr (WIND) votes = out[q] > 0.f ? 2 : 0;
    else
#pragma unroll 1
    for (int r = 0; r < 3; ++r) {
        const Ray R = make_ray(px, py, pz, r);
        int cnt = 0;
        if (F == 1) {
            cnt = ray_hit(R, tri[0], tri[1], tri[2]);
        } else {
            int sp = 0, node = 0;
            for (;;) {
                load_node(nodes, node, b, c[0], c[1]);
                bool go[2] = {ray_box(R, b, b + 3), ray_box(R, b + 6, b + 9)};
#pragma unroll
                for (int s = 0; s < 2; ++s)
                    if (go[s] && c[s] < 0) {
                        const int t = ~c[s];
                        cnt += ray_hit(R, tri[3 * t], tri[3 * t + 1], tri[3 * t + 2]);
                        go[s] = false;
                    }
                if (go[0] && go[1]) {
                    s_node[sp++][tid] = c[1];
                    node = c[0];
                } else if (go[0] || go[1]) {
                    node = go[0] ? c[0] : c[1];
                } else if (sp > 0) {
                    node = s_node[--sp][tid];
                } else {
                    break;
                }
            }
        }
        votes += cnt & 1;
    }
    out[q] = signed_out(best, votes);
    if (REC) face_out[q] = bestf;
}

// every point against every triangle (shared-memory tiles of SDF_TILE triangles): the reference for the BVH path.
// REC: also write the nearest face (the first in index order at the minimum); WIND: as k_sdf_query_bvh
template <bool REC, bool WIND = false>
__global__ void __launch_bounds__(SDF_BLOCK)
k_sdf_query_brute(const float4* __restrict__ tri, int F, const float* __restrict__ pts, int64_t P, float* __restrict__ out,
                  int32_t* __restrict__ face_out) {
    __shared__ float4 s_tri[3 * SDF_TILE];
    const int64_t i = blockIdx.x * (int64_t)SDF_BLOCK + threadIdx.x;
    const bool valid = i < P;
    const float px = valid ? pts[3 * i] : 0.f, py = valid ? pts[3 * i + 1] : 0.f, pz = valid ? pts[3 * i + 2] : 0.f;
    const D3 p = {(double)px, (double)py, (double)pz};
    const Ray R0 = make_ray(px, py, pz, 0), R1 = make_ray(px, py, pz, 1), R2 = make_ray(px, py, pz, 2);
    double best = INFINITY;
    int bestf = 0;
    int c0 = 0, c1 = 0, c2 = 0;
    for (int base = 0; base < F; base += SDF_TILE) {
        const int nt = min(SDF_TILE, F - base);
        __syncthreads();
        for (int k = threadIdx.x; k < 3 * nt; k += SDF_BLOCK) s_tri[k] = tri[3 * (int64_t)base + k];
        __syncthreads();
        if (!valid) continue;
#pragma unroll 1
        for (int t = 0; t < nt; ++t) {
            const float4 A = s_tri[3 * t], B = s_tri[3 * t + 1], C = s_tri[3 * t + 2];
            if (REC) {
                const double d2 = tri_d2(p, A, B, C);
                if (d2 < best) {
                    best = d2;
                    bestf = base + t;
                }
            } else {
                best = fmin(best, tri_d2(p, A, B, C));
            }
            if constexpr (!WIND) {
                c0 += ray_hit(R0, A, B, C);
                c1 += ray_hit(R1, A, B, C);
                c2 += ray_hit(R2, A, B, C);
            }
        }
    }
    if constexpr (WIND) c0 = c1 = valid && out[i] > 0.f ? 1 : 0;
    if (valid) out[i] = signed_out(best, (c0 & 1) + (c1 & 1) + (c2 & 1));
    if (REC && valid) face_out[i] = bestf;
}

// ---- generalised winding number ----------------------------------------------------------------------------------
// Far-field acceptance: a subtree whose corners all lie within r of its centroid c is replaced by its expansion when
// |q - c| > WN_BETA r.  The expansion goes through the first moment m (below).  Barill et al. use beta = 2; at 3 the BVH
// mode's max |w - exact| measured 0.024 on the test meshes (tested bar 0.05) and 0.019 on the icospheres of
// scripts/bench_winding.py.  This is a measurement, not a bound: the truncation error of a node grows with the face area
// inside its radius, which is unbounded (many stacked or crumpled layers).
constexpr double WN_BETA = 3.0;
constexpr double WN_INV_4PI = 0.079577471545947667884;      // 1 / (4 pi)

// Moments of an internal node's subtree (indexed like BvhNode), fp64: c = area-weighted centroid of the face centroids,
// r = radius around c bounding every corner, n = sum of the oriented area vectors a_f, m[3 i + j] = sum a_f,i (c_f - c)_j
// (Barill et al. 2018's second-order term), area = sum |a_f|
struct __align__(16) WnNode {
    double c[3], r;
    double n[3], area;
    double m[9], pad;
};

// solid angle of the oriented triangle (A, B, C) seen from p (Van Oosterom & Strackee 1983): 2 atan2(num, den) of the
// sorted corners, times their orientation C.w; 0 for a degenerate face
__device__ __forceinline__ double solid_angle(D3 p, float4 A4, float4 B4, float4 C4) {
    if (A4.w != 0.f) return 0.0;
    const D3 a = sub3(d3(A4), p), b = sub3(d3(B4), p), c = sub3(d3(C4), p);
    const double la = sqrt(dot3(a, a)), lb = sqrt(dot3(b, b)), lc = sqrt(dot3(c, c));
    const D3 bxc = {dsub(dmul(b.y, c.z), dmul(b.z, c.y)), dsub(dmul(b.z, c.x), dmul(b.x, c.z)), dsub(dmul(b.x, c.y), dmul(b.y, c.x))};
    const double num = dot3(a, bxc);
    const double den = dadd(dadd(dadd(dmul(dmul(la, lb), lc), dmul(dot3(a, b), lc)), dmul(dot3(a, c), lb)), dmul(dot3(b, c), la));
    return dmul((double)C4.w, 2.0 * atan2(num, den));
}

// moments of one face (m = 0: the face's centroid is the expansion centre)
__device__ __forceinline__ WnNode leaf_moments(float4 A4, float4 B4, float4 C4) {
    WnNode L;
    const D3 a = d3(A4), b = d3(B4), c = d3(C4);
    const double third = 1.0 / 3.0;
    const D3 g = {dmul(dadd(dadd(a.x, b.x), c.x), third), dmul(dadd(dadd(a.y, b.y), c.y), third),
                  dmul(dadd(dadd(a.z, b.z), c.z), third)};
    const D3 ab = sub3(b, a), ac = sub3(c, a);
    D3 n = {dsub(dmul(ab.y, ac.z), dmul(ab.z, ac.y)), dsub(dmul(ab.z, ac.x), dmul(ab.x, ac.z)), dsub(dmul(ab.x, ac.y), dmul(ab.y, ac.x))};
    const double s = A4.w != 0.f ? 0.0 : 0.5 * (double)C4.w;
    n = {dmul(s, n.x), dmul(s, n.y), dmul(s, n.z)};
    L.c[0] = g.x; L.c[1] = g.y; L.c[2] = g.z;
    L.r = sqrt(fmax(fmax(dist2(a, g), dist2(b, g)), dist2(c, g)));
    L.n[0] = n.x; L.n[1] = n.y; L.n[2] = n.z;
    L.area = sqrt(dot3(n, n));
#pragma unroll
    for (int k = 0; k < 9; ++k) L.m[k] = 0.0;
    L.pad = 0.0;
    return L;
}

// moments of child s of a node: a leaf's from its triangle, an internal node's as stored (read through L2: written by
// another thread of the same launch)
__device__ __forceinline__ WnNode child_moments(const float4* __restrict__ tri, const WnNode* mom, int ch) {
    if (ch < 0) {
        const int t = ~ch;
        return leaf_moments(tri[3 * t], tri[3 * t + 1], tri[3 * t + 2]);
    }
    WnNode M;
    const double2* src = reinterpret_cast<const double2*>(mom + ch);
    double2* dst = reinterpret_cast<double2*>(&M);
#pragma unroll
    for (int k = 0; k < 9; ++k) dst[k] = __ldcg(src + k);
    return M;
}

// bottom-up moments, one thread per leaf; the second thread to reach a node forms it as child 0 + child 1 (so the
// result does not depend on which thread arrives last):
//   area = A0 + A1, c = (A0 c0 + A1 c1) / area (the midpoint when area == 0), n = n0 + n1,
//   m = (m0 + n0 (c0 - c)^T) + (m1 + n1 (c1 - c)^T), r = max(|c0 - c| + r0, |c1 - c| + r1)
__global__ void k_sdf_wn_moments(const float4* __restrict__ tri, int n, const BvhNode* __restrict__ nodes,
                                 const int* __restrict__ parent, int* __restrict__ arrived, WnNode* mom) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    int p = parent[n - 1 + k];
    while (p >= 0) {
        __threadfence();
        if (atomicAdd(&arrived[p], 1) == 0) return;
        __threadfence();
        const WnNode X = child_moments(tri, mom, nodes[p].child[0]);
        const WnNode Y = child_moments(tri, mom, nodes[p].child[1]);
        WnNode Z;
        Z.area = dadd(X.area, Y.area);
        const double wx = Z.area > 0.0 ? X.area / Z.area : 0.5, wy = Z.area > 0.0 ? Y.area / Z.area : 0.5;
        double dx[3], dy[3];
#pragma unroll
        for (int d = 0; d < 3; ++d) {
            Z.c[d] = dadd(dmul(wx, X.c[d]), dmul(wy, Y.c[d]));
            Z.n[d] = dadd(X.n[d], Y.n[d]);
            dx[d] = dsub(X.c[d], Z.c[d]);
            dy[d] = dsub(Y.c[d], Z.c[d]);
        }
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
            for (int j = 0; j < 3; ++j)
                Z.m[3 * i + j] = dadd(dadd(X.m[3 * i + j], dmul(X.n[i], dx[j])), dadd(Y.m[3 * i + j], dmul(Y.n[i], dy[j])));
        const double ex = sqrt(dadd(dadd(dmul(dx[0], dx[0]), dmul(dx[1], dx[1])), dmul(dx[2], dx[2])));
        const double ey = sqrt(dadd(dadd(dmul(dy[0], dy[0]), dmul(dy[1], dy[1])), dmul(dy[2], dy[2])));
        Z.r = fmax(dadd(ex, X.r), dadd(ey, Y.r));
        Z.pad = 0.0;
        double2* dst = reinterpret_cast<double2*>(mom + p);
        const double2* src = reinterpret_cast<const double2*>(&Z);
#pragma unroll
        for (int t = 0; t < 9; ++t) __stcg(dst + t, src[t]);
        p = parent[p];
    }
}

// far-field solid angle of node `node` seen from p when |p - c| > WN_BETA r (returns true and adds it to acc): with
// x = c - p, sum_f a_f . G(c_f) for G(y) = (y - p) / |y - p|^3 to first order around c,
//   n . x / |x|^3 + tr(m) / |x|^3 - 3 x^T m x / |x|^5
__device__ __forceinline__ bool far_field(const WnNode* __restrict__ mom, int node, D3 p, double& acc) {
    const double2* q = reinterpret_cast<const double2*>(mom + node);
    const double2 c01 = __ldg(q), c2r = __ldg(q + 1);
    const D3 x = {dsub(c01.x, p.x), dsub(c01.y, p.y), dsub(c2r.x, p.z)};
    const double d2 = dot3(x, x);
    if (!(d2 > WN_BETA * WN_BETA * c2r.y * c2r.y)) return false;
    const double2 n01 = __ldg(q + 2), n2a = __ldg(q + 3), m01 = __ldg(q + 4), m23 = __ldg(q + 5), m45 = __ldg(q + 6),
                  m67 = __ldg(q + 7), m8p = __ldg(q + 8);
    const D3 nv = {n01.x, n01.y, n2a.x};
    const double m[9] = {m01.x, m01.y, m23.x, m23.y, m45.x, m45.y, m67.x, m67.y, m8p.x};
    const double d = sqrt(d2);
    const double i3 = 1.0 / dmul(d2, d), i5 = i3 / d2;
    const double mx0 = dadd(dadd(dmul(m[0], x.x), dmul(m[1], x.y)), dmul(m[2], x.z));
    const double mx1 = dadd(dadd(dmul(m[3], x.x), dmul(m[4], x.y)), dmul(m[5], x.z));
    const double mx2 = dadd(dadd(dmul(m[6], x.x), dmul(m[7], x.y)), dmul(m[8], x.z));
    const double xmx = dadd(dadd(dmul(x.x, mx0), dmul(x.y, mx1)), dmul(x.z, mx2));
    const double nx = dadd(dadd(dmul(nv.x, x.x), dmul(nv.y, x.y)), dmul(nv.z, x.z));
    const double tr = dadd(dadd(m[0], m[4]), m[8]);
    acc = dadd(acc, dsub(dmul(dadd(nx, tr), i3), dmul(3.0, dmul(xmx, i5))));
    return true;
}

// generalised winding number, BVH mode: one thread per point in Morton order; the tree fixes the visit order (child 0
// before child 1), so the sum is bitwise reproducible.  SIGN: out[q] = +1 where |w| >= 1/2 (decided in fp64), else -1;
// otherwise out[q] = w rounded to fp32
template <bool SIGN>
__global__ void __launch_bounds__(SDF_BLOCK)
k_sdf_winding_bvh(const float4* __restrict__ tri, const BvhNode* __restrict__ nodes, const WnNode* __restrict__ mom, int F,
                  const float* __restrict__ pts, const uint32_t* __restrict__ order, int64_t P, float* __restrict__ out) {
    __shared__ int s_node[SDF_STACK][SDF_BLOCK];
    const int64_t i = blockIdx.x * (int64_t)SDF_BLOCK + threadIdx.x;
    if (i >= P) return;
    const int tid = threadIdx.x;
    const int64_t q = order[i];
    const D3 p = {(double)pts[3 * q], (double)pts[3 * q + 1], (double)pts[3 * q + 2]};
    double acc = 0.0;
    if (F == 1) {
        acc = solid_angle(p, tri[0], tri[1], tri[2]);
    } else if (!far_field(mom, 0, p, acc)) {
        int sp = 0, node = 0;
        for (;;) {
            const int2 c = __ldg(reinterpret_cast<const int2*>(&nodes[node].child[0]));
            bool go[2] = {false, false};
#pragma unroll
            for (int s = 0; s < 2; ++s) {
                const int ch = s == 0 ? c.x : c.y;
                if (ch < 0) {
                    const int t = ~ch;
                    acc = dadd(acc, solid_angle(p, tri[3 * t], tri[3 * t + 1], tri[3 * t + 2]));
                } else {
                    go[s] = !far_field(mom, ch, p, acc);
                }
            }
            if (go[0] && go[1]) {
                s_node[sp++][tid] = c.y;
                node = c.x;
            } else if (go[0] || go[1]) {
                node = go[0] ? c.x : c.y;
            } else if (sp > 0) {
                node = s_node[--sp][tid];
            } else {
                break;
            }
        }
    }
    const double w = dmul(acc, WN_INV_4PI);
    out[q] = SIGN ? (fabs(w) >= 0.5 ? 1.f : -1.f) : (float)w;
}

// generalised winding number, exact: every face in face order (shared-memory tiles), fp64 sum; the reference for the
// BVH mode.  SIGN as k_sdf_winding_bvh
template <bool SIGN>
__global__ void __launch_bounds__(SDF_BLOCK)
k_sdf_winding_brute(const float4* __restrict__ tri, int F, const float* __restrict__ pts, int64_t P, float* __restrict__ out) {
    __shared__ float4 s_tri[3 * SDF_TILE];
    const int64_t i = blockIdx.x * (int64_t)SDF_BLOCK + threadIdx.x;
    const bool valid = i < P;
    const D3 p = {valid ? (double)pts[3 * i] : 0.0, valid ? (double)pts[3 * i + 1] : 0.0, valid ? (double)pts[3 * i + 2] : 0.0};
    double acc = 0.0;
    for (int base = 0; base < F; base += SDF_TILE) {
        const int nt = min(SDF_TILE, F - base);
        __syncthreads();
        for (int k = threadIdx.x; k < 3 * nt; k += SDF_BLOCK) s_tri[k] = tri[3 * (int64_t)base + k];
        __syncthreads();
        if (!valid) continue;
#pragma unroll 1
        for (int t = 0; t < nt; ++t) acc = dadd(acc, solid_angle(p, s_tri[3 * t], s_tri[3 * t + 1], s_tri[3 * t + 2]));
    }
    if (!valid) return;
    const double w = dmul(acc, WN_INV_4PI);
    out[i] = SIGN ? (fabs(w) >= 0.5 ? 1.f : -1.f) : (float)w;
}

__global__ void k_sdf_init(uint32_t* __restrict__ mm, unsigned long long* __restrict__ bad) {
    const int t = threadIdx.x;
    if (t < 24) mm[t] = (t % 8) < 3 ? 0xffffffffu : 0u;
    if (t < 4) bad[t] = ULLONG_MAX;
}

// ---- backward --------------------------------------------------------------------------------------------------
// One thread per point: closest point c of the point's nearest face (tri_closest on the sorted corners, as the forward
// evaluated it), u = (p - c) / |p - c|, s = sign of sdf.  d sdf / d p = s u; d sdf / d v_k = -s b_k u for the corners
// of the face.  gpt[p] = g s u (fp32, NULL: not written); coef[p] = -g s u (fp64) and w[3 p + k] = b_k, vid[3 p + k] =
// vertex id of corner k, for the reduction onto the vertices (coef NULL: not written).  sdf == 0 or |p - c| == 0: 0.
__global__ void k_sdf_backward(const float* __restrict__ verts, const int64_t* __restrict__ faces,
                               const float* __restrict__ pts, int64_t P, const int32_t* __restrict__ nearest,
                               const float* __restrict__ sdf, const float* __restrict__ g, float* __restrict__ gpt,
                               double* __restrict__ coef, double* __restrict__ w, uint64_t* __restrict__ vid,
                               uint32_t* __restrict__ entry) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= P) return;
    float4 v[3];
    int64_t id[3];
    sorted_face(verts, faces, nearest[i], v, id);
    const D3 p = {(double)pts[3 * i], (double)pts[3 * i + 1], (double)pts[3 * i + 2]};
    double b[3];
    const D3 c = tri_closest(p, v[0], v[1], v[2], b);
    const D3 r = sub3(p, c);
    const double d = sqrt(dot3(r, r));
    const float s = sdf[i];
    double gs = 0.0;
    if (s != 0.0f && d > 0.0) gs = (s > 0.0f ? (double)g[i] : -(double)g[i]) / d;
    const D3 gu = {dmul(gs, r.x), dmul(gs, r.y), dmul(gs, r.z)};
    if (gpt) {
        gpt[3 * i] = (float)gu.x;
        gpt[3 * i + 1] = (float)gu.y;
        gpt[3 * i + 2] = (float)gu.z;
    }
    if (coef) {
        coef[3 * i] = -gu.x;
        coef[3 * i + 1] = -gu.y;
        coef[3 * i + 2] = -gu.z;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            w[3 * i + k] = b[k];
            vid[3 * i + k] = (uint64_t)id[k];
            entry[3 * i + k] = (uint32_t)(3 * i + k);
        }
    }
}

// grad_verts: one thread per run of equal vertex ids in the sorted (vertex id, entry) list; the run's entries are in
// ascending (point, corner) order (stable sort), summed in fp64, rounded once.  Vertices without entries stay 0.
__global__ void k_sdf_vert_reduce(const uint64_t* __restrict__ key, const uint32_t* __restrict__ ent, int64_t n,
                                  const double* __restrict__ coef, const double* __restrict__ w, float* __restrict__ gv) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n || (i > 0 && key[i - 1] == key[i])) return;
    const uint64_t k = key[i];
    double sx = 0.0, sy = 0.0, sz = 0.0;
    for (int64_t j = i; j < n && key[j] == k; ++j) {
        const uint32_t e = ent[j];
        const double b = w[e];
        const int64_t q = e / 3;
        sx = dadd(sx, dmul(b, coef[3 * q]));
        sy = dadd(sy, dmul(b, coef[3 * q + 1]));
        sz = dadd(sz, dmul(b, coef[3 * q + 2]));
    }
    gv[3 * k] = (float)sx;
    gv[3 * k + 1] = (float)sy;
    gv[3 * k + 2] = (float)sz;
}

inline unsigned nblk(int64_t n, int b) { return (unsigned)ceil_div(n > 0 ? n : 1, b); }

}  // namespace

}  // namespace ds

using namespace ds;

namespace {

// the V / F / P checks and the limits every entry point shares
int check_sizes(const char* fn, const ds_workspace* ws, const float* tri_verts, int64_t V, const int64_t* faces, int64_t F,
                int64_t P) {
    DS_REQUIRE(ws && tri_verts && faces, "%s: null argument", fn);
    DS_REQUIRE(V > 0 && F > 0, "%s: empty mesh (V = %lld, F = %lld)", fn, (long long)V, (long long)F);
    DS_REQUIRE(P >= 0, "%s: negative point count", fn);
    DS_REQUIRE(F < ((int64_t)1 << 30) && P < ((int64_t)1 << 31) - SDF_BLOCK && V < ((int64_t)1 << 40),
               "%s: too many faces or points", fn);
    return DS_OK;
}

// face indices in [0, V), finite coordinates and (nearest != NULL) nearest-face ids in [0, F): one synchronisation
int validate(const char* fn, cudaStream_t st, unsigned long long* bad, const float* tri_verts, int64_t V,
             const int64_t* faces, int64_t F, const float* points, int64_t P, const int32_t* nearest) {
    k_sdf_validate<<<296, 256, 0, st>>>(tri_verts, V, faces, F, points, P, nearest, bad);
    DS_LAUNCH_CHECK();
    unsigned long long bh[4];
    DS_CUDA(cudaMemcpyAsync(bh, bad, sizeof(bh), cudaMemcpyDeviceToHost, st));
    DS_CUDA(cudaStreamSynchronize(st));
    DS_REQUIRE(bh[0] == ULLONG_MAX, "%s: face %llu has a vertex index outside [0, %lld)", fn, bh[0], (long long)V);
    DS_REQUIRE(bh[1] == ULLONG_MAX, "%s: vertex %llu has a non-finite coordinate", fn, bh[1]);
    DS_REQUIRE(bh[2] == ULLONG_MAX, "%s: query point %llu has a non-finite coordinate", fn, bh[2]);
    DS_REQUIRE(bh[3] == ULLONG_MAX, "%s: point %llu has nearest face outside [0, %lld)", fn, bh[3], (long long)F);
    return DS_OK;
}

// what mesh_sdf_impl computes: the signed distance with the ray-parity sign, the signed distance with the winding-number
// sign, or the winding number alone (into sdf_out)
enum SdfJob { SDF_PARITY, SDF_WINDING, SDF_WINDING_NUMBER };

// the query kernel of a job: face_out == NULL runs the non-recording instantiations
template <bool WIND>
void launch_query(bool bvh, cudaStream_t st, const float4* tri, const BvhNode* nodes, int F, const float* points,
                  const uint32_t* porder, int64_t P, float* sdf_out, int32_t* face_out) {
    if (bvh && face_out)
        k_sdf_query_bvh<true, WIND><<<nblk(P, SDF_BLOCK), SDF_BLOCK, 0, st>>>(tri, nodes, F, points, porder, P, sdf_out, face_out);
    else if (bvh)
        k_sdf_query_bvh<false, WIND><<<nblk(P, SDF_BLOCK), SDF_BLOCK, 0, st>>>(tri, nodes, F, points, porder, P, sdf_out, nullptr);
    else if (face_out)
        k_sdf_query_brute<true, WIND><<<nblk(P, SDF_BLOCK), SDF_BLOCK, 0, st>>>(tri, F, points, P, sdf_out, face_out);
    else
        k_sdf_query_brute<false, WIND><<<nblk(P, SDF_BLOCK), SDF_BLOCK, 0, st>>>(tri, F, points, P, sdf_out, nullptr);
}

// ds_mesh_sdf, ds_mesh_sdf_nearest, ds_mesh_sdf_winding and ds_mesh_winding_number
int mesh_sdf_impl(const char* fn, ds_workspace* ws, const float* tri_verts, int64_t V, const int64_t* faces, int64_t F,
                  const float* points, int64_t P, int mode, float* sdf_out, int32_t* face_out, bool want_face,
                  SdfJob job, void* stream) {
    DS_TRY(check_sizes(fn, ws, tri_verts, V, faces, F, P));
    DS_REQUIRE(mode == 0 || mode == 1, "%s: unknown mode %d (0 = BVH, 1 = brute force)", fn, mode);
    if (P == 0) return DS_OK;
    DS_REQUIRE(points && sdf_out && (face_out || !want_face), "%s: null argument", fn);
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t nmax = std::max(F, P);
    size_t sort_tmp = 0;
    DS_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, sort_tmp, (uint32_t*)nullptr, (uint32_t*)nullptr, (uint32_t*)nullptr,
                                            (uint32_t*)nullptr, (int)nmax, 0, 30, st));
    const size_t need = (size_t)F * (12 + 16 + 48 + 64 + 12 + (job == SDF_PARITY ? 0 : sizeof(WnNode))) + (size_t)P * 16 +
                        sort_tmp + (1 << 16);
    DS_TRY(ws->arena.reserve(need, st));
    Arena& a = ws->arena;
    uint32_t* mm = a.take<uint32_t>(24);
    unsigned long long* bad = a.take<unsigned long long>(4);
    float4* tri = a.take<float4>(3 * F);
    DS_REQUIRE(mm && bad && tri, "%s: workspace arena exhausted", fn);
    k_sdf_init<<<1, 32, 0, st>>>(mm, bad);
    DS_LAUNCH_CHECK();
    DS_TRY(validate(fn, st, bad, tri_verts, V, faces, F, points, P, nullptr));

    if (mode == 1) {
        {
            ProfScope prof(PROF_SDF_BUILD, st);
            if (job == SDF_PARITY)
                k_sdf_gather<false><<<nblk(F, 256), 256, 0, st>>>(tri_verts, faces, nullptr, F, tri);
            else
                k_sdf_gather<true><<<nblk(F, 256), 256, 0, st>>>(tri_verts, faces, nullptr, F, tri);
            DS_LAUNCH_CHECK();
        }
        if (job != SDF_PARITY) {
            ProfScope prof(PROF_SDF_WINDING, st);
            if (job == SDF_WINDING)
                k_sdf_winding_brute<true><<<nblk(P, SDF_BLOCK), SDF_BLOCK, 0, st>>>(tri, (int)F, points, P, sdf_out);
            else
                k_sdf_winding_brute<false><<<nblk(P, SDF_BLOCK), SDF_BLOCK, 0, st>>>(tri, (int)F, points, P, sdf_out);
            DS_LAUNCH_CHECK();
            if (job == SDF_WINDING_NUMBER) return DS_OK;
        }
        ProfScope prof(PROF_SDF_QUERY, st);
        if (job == SDF_WINDING)
            launch_query<true>(false, st, tri, nullptr, (int)F, points, nullptr, P, sdf_out, face_out);
        else
            launch_query<false>(false, st, tri, nullptr, (int)F, points, nullptr, P, sdf_out, face_out);
        DS_LAUNCH_CHECK();
        return DS_OK;
    }

    float* cent = a.take<float>(3 * F);
    uint32_t* codes = a.take<uint32_t>(nmax);
    uint32_t* codes2 = a.take<uint32_t>(nmax);
    uint32_t* iota = a.take<uint32_t>(nmax);
    uint32_t* order = a.take<uint32_t>(F);
    uint32_t* porder = a.take<uint32_t>(P);
    BvhNode* nodes = a.take<BvhNode>(F);
    int* parent = a.take<int>(2 * F);
    int* arrived = a.take<int>(F);
    void* scratch = a.take<char>(sort_tmp + 16);
    WnNode* mom = job == SDF_PARITY ? nullptr : a.take<WnNode>(F);
    DS_REQUIRE(cent && codes && codes2 && iota && order && porder && nodes && parent && arrived && scratch &&
               (mom || job == SDF_PARITY), "%s: workspace arena exhausted", fn);
    uint32_t *mm_v = mm, *mm_c = mm + 8, *mm_p = mm + 16;
    {
    ProfScope prof(PROF_SDF_BUILD, st);
    // triangles in Morton order of their centroids
    if (job == SDF_PARITY)
        k_sdf_centroids<false><<<nblk(F, 256), 256, 0, st>>>(tri_verts, faces, F, cent);
    else
        k_sdf_centroids<true><<<nblk(F, 256), 256, 0, st>>>(tri_verts, faces, F, cent);
    DS_LAUNCH_CHECK();
    k_bbox<<<148, 256, 0, st>>>(cent, F, mm_c);
    DS_LAUNCH_CHECK();
    k_bbox<<<148, 256, 0, st>>>(tri_verts, V, mm_v);
    DS_LAUNCH_CHECK();
    k_bbox<<<148, 256, 0, st>>>(points, P, mm_p);
    DS_LAUNCH_CHECK();
    k_morton_codes<<<nblk(F, 256), 256, 0, st>>>(cent, F, mm_c, codes, iota);
    DS_LAUNCH_CHECK();
    DS_CUDA(cub::DeviceRadixSort::SortPairs(scratch, sort_tmp, codes, codes2, iota, order, (int)F, 0, 30, st));
    count_launch();
    if (job == SDF_PARITY)
        k_sdf_gather<false><<<nblk(F, 256), 256, 0, st>>>(tri_verts, faces, order, F, tri);
    else
        k_sdf_gather<true><<<nblk(F, 256), 256, 0, st>>>(tri_verts, faces, order, F, tri);
    DS_LAUNCH_CHECK();
    if (F > 1) {
        DS_CUDA(cudaMemsetAsync(arrived, 0, (size_t)F * sizeof(int), st));
        k_sdf_karras<<<nblk(F - 1, 256), 256, 0, st>>>(codes2, (int)F, nodes, parent);
        DS_LAUNCH_CHECK();
        k_sdf_refit<<<nblk(F, 256), 256, 0, st>>>(tri, (int)F, nodes, parent, arrived, mm_v, mm_p);
        DS_LAUNCH_CHECK();
    }
    }
    // queries in Morton order of the points (for the winding jobs the point order is part of the winding stage)
    auto point_order = [&]() -> int {
        k_morton_codes<<<nblk(P, 256), 256, 0, st>>>(points, P, mm_p, codes, iota);
        DS_LAUNCH_CHECK();
        DS_CUDA(cub::DeviceRadixSort::SortPairs(scratch, sort_tmp, codes, codes2, iota, porder, (int)P, 0, 30, st));
        count_launch();
        return DS_OK;
    };
    if (job != SDF_PARITY) {
        ProfScope prof(PROF_SDF_WINDING, st);
        if (F > 1) {
            DS_CUDA(cudaMemsetAsync(arrived, 0, (size_t)F * sizeof(int), st));
            k_sdf_wn_moments<<<nblk(F, 256), 256, 0, st>>>(tri, (int)F, nodes, parent, arrived, mom);
            DS_LAUNCH_CHECK();
        }
        DS_TRY(point_order());
        if (job == SDF_WINDING)
            k_sdf_winding_bvh<true><<<nblk(P, SDF_BLOCK), SDF_BLOCK, 0, st>>>(tri, nodes, mom, (int)F, points, porder, P, sdf_out);
        else
            k_sdf_winding_bvh<false><<<nblk(P, SDF_BLOCK), SDF_BLOCK, 0, st>>>(tri, nodes, mom, (int)F, points, porder, P, sdf_out);
        DS_LAUNCH_CHECK();
        if (job == SDF_WINDING_NUMBER) return DS_OK;
    }
    ProfScope prof(PROF_SDF_QUERY, st);
    if (job == SDF_PARITY) {
        DS_TRY(point_order());
        launch_query<false>(true, st, tri, nodes, (int)F, points, porder, P, sdf_out, face_out);
    } else {
        launch_query<true>(true, st, tri, nodes, (int)F, points, porder, P, sdf_out, face_out);
    }
    DS_LAUNCH_CHECK();
    return DS_OK;
}

}  // namespace

extern "C" int ds_mesh_sdf(ds_workspace* ws, const float* tri_verts, int64_t V, const int64_t* faces, int64_t F,
                           const float* points, int64_t P, int mode, float* sdf_out, void* stream) {
    return mesh_sdf_impl("ds_mesh_sdf", ws, tri_verts, V, faces, F, points, P, mode, sdf_out, nullptr, false, SDF_PARITY,
                         stream);
}

extern "C" int ds_mesh_sdf_nearest(ds_workspace* ws, const float* tri_verts, int64_t V, const int64_t* faces, int64_t F,
                                   const float* points, int64_t P, int mode, float* sdf_out, int32_t* face_out,
                                   void* stream) {
    return mesh_sdf_impl("ds_mesh_sdf_nearest", ws, tri_verts, V, faces, F, points, P, mode, sdf_out, face_out, true,
                         SDF_PARITY, stream);
}

extern "C" int ds_mesh_winding_number(ds_workspace* ws, const float* tri_verts, int64_t V, const int64_t* faces, int64_t F,
                                      const float* points, int64_t P, int mode, float* w_out, void* stream) {
    return mesh_sdf_impl("ds_mesh_winding_number", ws, tri_verts, V, faces, F, points, P, mode, w_out, nullptr, false,
                         SDF_WINDING_NUMBER, stream);
}

extern "C" int ds_mesh_sdf_winding(ds_workspace* ws, const float* tri_verts, int64_t V, const int64_t* faces, int64_t F,
                                   const float* points, int64_t P, int mode, float* sdf_out, int32_t* face_out,
                                   void* stream) {
    return mesh_sdf_impl("ds_mesh_sdf_winding", ws, tri_verts, V, faces, F, points, P, mode, sdf_out, face_out, false,
                         SDF_WINDING, stream);
}

extern "C" int ds_mesh_sdf_backward(ds_workspace* ws, const float* tri_verts, int64_t V, const int64_t* faces, int64_t F,
                                    const float* points, int64_t P, const int32_t* face, const float* sdf,
                                    const float* grad_sdf, float* grad_verts, float* grad_points, void* stream) {
    const char* fn = "ds_mesh_sdf_backward";
    DS_TRY(check_sizes(fn, ws, tri_verts, V, faces, F, P));
    DS_REQUIRE(3 * P < ((int64_t)1 << 31), "%s: too many faces or points", fn);
    cudaStream_t st = (cudaStream_t)stream;
    if (grad_verts) DS_CUDA(cudaMemsetAsync(grad_verts, 0, (size_t)V * 3 * sizeof(float), st));
    if (P == 0) return DS_OK;
    DS_REQUIRE(points && face && sdf && grad_sdf, "%s: null argument", fn);
    int vbits = 1;
    while (vbits < 64 && ((uint64_t)(V - 1) >> vbits) != 0) ++vbits;
    const int64_t E = 3 * P;
    size_t sort_tmp = 0;
    DS_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, sort_tmp, (uint64_t*)nullptr, (uint64_t*)nullptr, (uint32_t*)nullptr,
                                            (uint32_t*)nullptr, (int)E, 0, vbits, st));
    const size_t need = (size_t)E * (8 + 8 + 16 + 8) + sort_tmp + (1 << 16);
    DS_TRY(ws->arena.reserve(need, st));
    Arena& a = ws->arena;
    unsigned long long* bad = a.take<unsigned long long>(4);
    uint32_t* mm = a.take<uint32_t>(24);
    DS_REQUIRE(bad && mm, "%s: workspace arena exhausted", fn);
    k_sdf_init<<<1, 32, 0, st>>>(mm, bad);
    DS_LAUNCH_CHECK();
    DS_TRY(validate(fn, st, bad, tri_verts, V, faces, F, points, P, face));
    if (!grad_verts && !grad_points) return DS_OK;
    double* coef = nullptr;
    double* w = nullptr;
    uint64_t *vid = nullptr, *vid2 = nullptr;
    uint32_t *ent = nullptr, *ent2 = nullptr;
    void* scratch = nullptr;
    if (grad_verts) {
        coef = a.take<double>(E);
        w = a.take<double>(E);
        vid = a.take<uint64_t>(E);
        vid2 = a.take<uint64_t>(E);
        ent = a.take<uint32_t>(E);
        ent2 = a.take<uint32_t>(E);
        scratch = a.take<char>(sort_tmp + 16);
        DS_REQUIRE(coef && w && vid && vid2 && ent && ent2 && scratch, "%s: workspace arena exhausted", fn);
    }
    k_sdf_backward<<<nblk(P, 256), 256, 0, st>>>(tri_verts, faces, points, P, face, sdf, grad_sdf, grad_points, coef, w,
                                                 vid, ent);
    DS_LAUNCH_CHECK();
    if (!grad_verts) return DS_OK;
    // stable sort by vertex id: each vertex's entries stay in ascending (point, corner) order
    DS_CUDA(cub::DeviceRadixSort::SortPairs(scratch, sort_tmp, vid, vid2, ent, ent2, (int)E, 0, vbits, st));
    count_launch();
    k_sdf_vert_reduce<<<nblk(E, 256), 256, 0, st>>>(vid2, ent2, E, coef, w, grad_verts);
    DS_LAUNCH_CHECK();
    return DS_OK;
}

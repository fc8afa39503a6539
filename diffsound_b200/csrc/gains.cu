// Modal gains: where a struck surface point excites each mode.  With mass-normalised mode shapes (U^T M U = I) a unit
// impulse at surface point x in direction d excites mode m with gain g_m(x, d) = d . u_m(x), u_m(x) the P1 / P2
// interpolation of column m of U at x.  Nothing in the reference computes this: its audio paths take mode amplitudes
// from learned parameters or ones.
//
// ds_tet_boundary_count / _fill: the triangles that belong to exactly one tet.  The 4 T face triples (corner ids sorted
// ascending) are ordered by three stable LSD radix-sort passes (largest id, middle id, smallest id; the multi-pass
// scheme of ds_unique_rows3 in mesh.cu) carrying the face index 4 t + f, then a face is on the boundary when neither
// neighbour in that order holds the same triple.  The output is in ascending triple order, so it does not depend on the
// tet order or the rotation of corners within a tet, and no atomic decides it.  Each face is written (a, b, c) from its
// sorted triple, swapped to (a, c, b) when the opposite corner s lies on the side of (b - a) x (c - a) (fp64 determinant
// of the fp32 corners), so its normal points out of the owning tet.
//
// ds_modal_gains / _backward: one warp per point, lanes across modes.  U is row-major, so the three rows of a node are
// contiguous and each row read is one coalesced load; the sums run in fp64 in a fixed order (local node, then
// component) and are rounded once.  The point is first put on its boundary face by the closest-point region analysis
// of closest.cuh (shared with sdf.cu); the owning tet's barycentrics are the face weights with 0 at the opposite
// corner.  The backward reduces over modes with a fixed xor-shuffle tree: no atomics, bitwise reproducible.
#include "common.cuh"
#include "../../include/diffsound_sm100.h"
#include "closest.cuh"
#include "tet_faces.cuh"
#include <cub/cub.cuh>
#include <climits>

namespace ds {

namespace {

constexpr int GAINS_WARPS = 8;     // points per CTA (one warp each)

// corner ids of face f (opposite corner f) of tet t, sorted ascending
__device__ __forceinline__ void face_triple(const int32_t* __restrict__ tets, int npe, int order, int64_t i, uint32_t (&v)[3]) {
    const int64_t t = i >> 2;
    const int f = (int)(i & 3);
    int q = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j)
        if (j != f) v[q++] = (uint32_t)tets[t * npe + corner_local(order, j)];
    uint32_t s;
    if (v[0] > v[1]) { s = v[0]; v[0] = v[1]; v[1] = s; }
    if (v[1] > v[2]) { s = v[1]; v[1] = v[2]; v[2] = s; }
    if (v[0] > v[1]) { s = v[0]; v[0] = v[1]; v[1] = s; }
}

__device__ __forceinline__ D3 node3(const float* __restrict__ verts, int64_t n) {
    return {(double)verts[3 * n], (double)verts[3 * n + 1], (double)verts[3 * n + 2]};
}
__device__ __forceinline__ D3 cross3(D3 a, D3 b) {
    return {dsub(dmul(a.y, b.z), dmul(a.z, b.y)), dsub(dmul(a.z, b.x), dmul(a.x, b.z)), dsub(dmul(a.x, b.y), dmul(a.y, b.x))};
}

// bad[0]: smallest (tet * npe + slot) with a node id outside [0, n); bad[1]: smallest node with a non-finite coordinate
__global__ void k_gb_validate(const float* __restrict__ verts, int64_t n, const int32_t* __restrict__ tets, int64_t TN,
                              unsigned long long* __restrict__ bad) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < TN || i < n; i += (int64_t)gridDim.x * blockDim.x) {
        if (i < TN && (tets[i] < 0 || tets[i] >= n)) atomicMin(&bad[0], (unsigned long long)i);
        if (i < n && !(isfinite(verts[3 * i]) && isfinite(verts[3 * i + 1]) && isfinite(verts[3 * i + 2])))
            atomicMin(&bad[1], (unsigned long long)i);
    }
}

// keys[i] = component `comp` of the sorted triple of face idx[i] (idx == nullptr: face i, and iota[i] = i)
__global__ void k_gb_keys(const int32_t* __restrict__ tets, int npe, int order, int64_t N, int comp,
                          const uint32_t* __restrict__ idx, uint32_t* __restrict__ keys, uint32_t* __restrict__ iota) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= N) return;
    uint32_t v[3];
    face_triple(tets, npe, order, idx ? (int64_t)idx[i] : i, v);
    keys[i] = v[comp];
    if (iota) iota[i] = (uint32_t)i;
}

// flag[i] = 1 when the triple at sorted position i occurs once; a triple in three or more tets marks bad[2]
__global__ void k_gb_flags(const int32_t* __restrict__ tets, int npe, int order, int64_t N, const uint32_t* __restrict__ idx,
                           int32_t* __restrict__ flag, unsigned long long* __restrict__ bad) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= N) return;
    uint32_t v[3], u[3];
    face_triple(tets, npe, order, idx[i], v);
    bool prev = false, next = false;
    if (i > 0) {
        face_triple(tets, npe, order, idx[i - 1], u);
        prev = u[0] == v[0] && u[1] == v[1] && u[2] == v[2];
    }
    if (i + 1 < N) {
        face_triple(tets, npe, order, idx[i + 1], u);
        next = u[0] == v[0] && u[1] == v[1] && u[2] == v[2];
    }
    flag[i] = !prev && !next;
    if (prev && next) atomicMin(&bad[2], (unsigned long long)(idx[i] >> 2));
}

__global__ void k_gb_fill(const float* __restrict__ verts, const int32_t* __restrict__ tets, int npe, int order, int64_t N,
                          const uint32_t* __restrict__ idx, const int32_t* __restrict__ flag, const int32_t* __restrict__ pos,
                          int32_t* __restrict__ faces, int32_t* __restrict__ owner, int32_t* __restrict__ local) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= N || !flag[i]) return;
    const int64_t fi = idx[i], t = fi >> 2;
    const int f = (int)(fi & 3);
    uint32_t v[3];
    face_triple(tets, npe, order, fi, v);
    const D3 a = node3(verts, v[0]);
    const D3 s = node3(verts, tets[t * npe + corner_local(order, f)]);
    const double det = dot3(cross3(sub3(node3(verts, v[1]), a), sub3(node3(verts, v[2]), a)), sub3(s, a));
    const int64_t o = pos[i];
    faces[3 * o] = (int32_t)v[0];
    faces[3 * o + 1] = (int32_t)(det > 0.0 ? v[2] : v[1]);
    faces[3 * o + 2] = (int32_t)(det > 0.0 ? v[1] : v[2]);
    owner[o] = (int32_t)t;
    local[o] = f;
}

struct GainsArgs {
    const float* verts;
    const int32_t* tets;
    int order, k;
    const int32_t *bfaces, *owner, *local;
    const float* pts;
    const int32_t* face;
    const float* dirs;       // nullptr: the outward unit normal of the face
    int64_t P, ldu;
    const double* U;
    float* gains;            // forward [P x k]
    float* closest;          // forward [P x 3]
    const float* up;         // backward: upstream gradient [P x k]
    float* gpt;              // backward [P x 3]
    float* gdir;             // backward [P x 3], nullptr when the directions were not given
};

// bad[0]: face id outside [0, F); bad[1]: non-finite point; bad[2]: non-finite direction; bad[3]: a boundary record that
// does not name a face of its owning tet with node ids in [0, n) (each the smallest point index)
__global__ void k_gains_validate(GainsArgs g, int64_t F, int64_t T, int64_t n, unsigned long long* __restrict__ bad) {
    const int npe = g.order == 1 ? 4 : 10;
    for (int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; p < g.P; p += (int64_t)gridDim.x * blockDim.x) {
        if (!(isfinite(g.pts[3 * p]) && isfinite(g.pts[3 * p + 1]) && isfinite(g.pts[3 * p + 2])))
            atomicMin(&bad[1], (unsigned long long)p);
        if (g.dirs && !(isfinite(g.dirs[3 * p]) && isfinite(g.dirs[3 * p + 1]) && isfinite(g.dirs[3 * p + 2])))
            atomicMin(&bad[2], (unsigned long long)p);
        const int32_t f = g.face[p];
        if (f < 0 || f >= F) { atomicMin(&bad[0], (unsigned long long)p); continue; }
        const int32_t t = g.owner[f], lf = g.local[f];
        bool ok = t >= 0 && t < T && lf >= 0 && lf < 4;
        if (ok) {
            for (int a = 0; a < npe; ++a) ok = ok && g.tets[(int64_t)t * npe + a] >= 0 && g.tets[(int64_t)t * npe + a] < n;
            int hit = 0;
            for (int j = 0; j < 4; ++j) {
                if (j == lf) continue;
                const int32_t c = g.tets[(int64_t)t * npe + corner_local(g.order, j)];
                hit += (c == g.bfaces[3 * f]) + (c == g.bfaces[3 * f + 1]) + (c == g.bfaces[3 * f + 2]);
            }
            ok = ok && hit == 3;
        }
        if (!ok) atomicMin(&bad[3], (unsigned long long)p);
    }
}

// everything of a point but the mode sums: node ids, shape functions N_a at the closest point, the direction and, for
// the backward, the physical gradients of N_a and the closest-point Jacobian (face: I - n n^T, edge: t t^T, vertex: 0)
template <int NPE>
struct PointGeom {
    int64_t node[NPE];
    double N[NPE];
    double dN[NPE][3];
    double d[3];
    D3 c, n, tan;
    int region;              // nonzero face weights: 3 face, 2 edge, 1 vertex
};

template <int NPE, bool GRAD>
__device__ __forceinline__ void point_geom(const GainsArgs& g, int64_t p, PointGeom<NPE>& G) {
    constexpr int order = NPE == 4 ? 1 : 2;
    const int32_t f = g.face[p];
    const int64_t t = g.owner[f];
    const int lf = g.local[f];
    const int32_t fid[3] = {g.bfaces[3 * f], g.bfaces[3 * f + 1], g.bfaces[3 * f + 2]};
    const D3 A = node3(g.verts, fid[0]), B = node3(g.verts, fid[1]), C = node3(g.verts, fid[2]);
    D3 nrm = cross3(sub3(B, A), sub3(C, A));
    const double nn = sqrt(dot3(nrm, nrm));
    const float4 A4 = {g.verts[3 * fid[0]], g.verts[3 * fid[0] + 1], g.verts[3 * fid[0] + 2], nn > 0.0 ? 0.f : 1.f};
    const float4 B4 = {g.verts[3 * fid[1]], g.verts[3 * fid[1] + 1], g.verts[3 * fid[1] + 2], 0.f};
    const float4 C4 = {g.verts[3 * fid[2]], g.verts[3 * fid[2] + 1], g.verts[3 * fid[2] + 2], 0.f};
    const D3 q = {(double)g.pts[3 * p], (double)g.pts[3 * p + 1], (double)g.pts[3 * p + 2]};
    double w[3];
    G.c = tri_closest(q, A4, B4, C4, w);
    G.n = nn > 0.0 ? D3{nrm.x / nn, nrm.y / nn, nrm.z / nn} : D3{0.0, 0.0, 0.0};
    G.region = (w[0] != 0.0) + (w[1] != 0.0) + (w[2] != 0.0);
    int64_t cn[4];
    double L[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        cn[j] = g.tets[t * NPE + corner_local(order, j)];
        L[j] = j == lf ? 0.0 : (cn[j] == fid[0] ? w[0] : (cn[j] == fid[1] ? w[1] : w[2]));
    }
#pragma unroll
    for (int a = 0; a < NPE; ++a) {
        G.node[a] = g.tets[t * NPE + a];
        if (order == 1) {
            G.N[a] = L[a];
        } else {
            const int l = c_p2_l[a], m = c_p2_m[a];
            G.N[a] = l == m ? dmul(L[l], dsub(dmul(2.0, L[l]), 1.0)) : dmul(4.0, dmul(L[l], L[m]));
        }
    }
    if (g.dirs) {
        G.d[0] = g.dirs[3 * p]; G.d[1] = g.dirs[3 * p + 1]; G.d[2] = g.dirs[3 * p + 2];
    } else {
        G.d[0] = G.n.x; G.d[1] = G.n.y; G.d[2] = G.n.z;
    }
    if (!GRAD) return;
    // grad L_j = rows of J^-1 (J = [X1 - X0, X2 - X0, X3 - X0]) for j = 1..3, grad L_0 = -(their sum)
    const D3 X0 = node3(g.verts, cn[0]);
    const D3 e1 = sub3(node3(g.verts, cn[1]), X0), e2 = sub3(node3(g.verts, cn[2]), X0), e3 = sub3(node3(g.verts, cn[3]), X0);
    const D3 r1 = cross3(e2, e3), r2 = cross3(e3, e1), r3 = cross3(e1, e2);
    const double det = dot3(e1, r1);
    const double inv = det != 0.0 ? 1.0 / det : 0.0;
    double gL[4][3] = {{0, 0, 0}, {r1.x * inv, r1.y * inv, r1.z * inv}, {r2.x * inv, r2.y * inv, r2.z * inv},
                       {r3.x * inv, r3.y * inv, r3.z * inv}};
#pragma unroll
    for (int c = 0; c < 3; ++c) gL[0][c] = -(gL[1][c] + gL[2][c] + gL[3][c]);
#pragma unroll
    for (int a = 0; a < NPE; ++a) {
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            if (order == 1) {
                G.dN[a][c] = gL[a][c];
            } else {
                const int l = c_p2_l[a], m = c_p2_m[a];
                G.dN[a][c] = l == m ? (4.0 * L[l] - 1.0) * gL[l][c] : 4.0 * (L[m] * gL[l][c] + L[l] * gL[m][c]);
            }
        }
    }
    G.tan = {0.0, 0.0, 0.0};
    if (G.region == 2) {
        const D3 P0 = w[0] != 0.0 ? A : B, P1 = w[2] != 0.0 ? C : B;
        const D3 e = sub3(P1, P0);
        const double l = sqrt(dot3(e, e));
        if (l > 0.0) G.tan = {e.x / l, e.y / l, e.z / l};
    }
}

template <int NPE>
__global__ void __launch_bounds__(32 * GAINS_WARPS, 2) k_modal_gains(const GainsArgs g) {
    const int lane = threadIdx.x & 31;
    const int64_t p = (int64_t)blockIdx.x * GAINS_WARPS + (threadIdx.x >> 5);
    if (p >= g.P) return;
    PointGeom<NPE> G;
    point_geom<NPE, false>(g, p, G);
#pragma unroll 1
    for (int m = lane; m < g.k; m += 32) {
        double acc = 0.0;
#pragma unroll
        for (int a = 0; a < NPE; ++a) {
            const double* row = g.U + 3 * G.node[a] * g.ldu + m;
            const double du = dadd(dadd(dmul(G.d[0], __ldg(row)), dmul(G.d[1], __ldg(row + g.ldu))),
                                   dmul(G.d[2], __ldg(row + 2 * g.ldu)));
            acc = dadd(acc, dmul(G.N[a], du));
        }
        g.gains[p * g.k + m] = (float)acc;
    }
    if (lane == 0) {
        g.closest[3 * p] = (float)G.c.x;
        g.closest[3 * p + 1] = (float)G.c.y;
        g.closest[3 * p + 2] = (float)G.c.z;
    }
}

template <int NPE>
__global__ void __launch_bounds__(32 * GAINS_WARPS, 2) k_modal_gains_bwd(const GainsArgs g) {
    const int lane = threadIdx.x & 31;
    const int64_t p = (int64_t)blockIdx.x * GAINS_WARPS + (threadIdx.x >> 5);
    if (p >= g.P) return;
    PointGeom<NPE> G;
    point_geom<NPE, true>(g, p, G);
    double sa[NPE], tc[3] = {0.0, 0.0, 0.0};
#pragma unroll
    for (int a = 0; a < NPE; ++a) sa[a] = 0.0;
#pragma unroll 1
    for (int m = lane; m < g.k; m += 32) {
        const double u = (double)g.up[p * g.k + m];
#pragma unroll
        for (int a = 0; a < NPE; ++a) {
            const double* row = g.U + 3 * G.node[a] * g.ldu + m;
            const double x = __ldg(row), y = __ldg(row + g.ldu), z = __ldg(row + 2 * g.ldu);
            sa[a] = dadd(sa[a], dmul(u, dadd(dadd(dmul(G.d[0], x), dmul(G.d[1], y)), dmul(G.d[2], z))));
            const double un = dmul(u, G.N[a]);
            tc[0] = dadd(tc[0], dmul(un, x));
            tc[1] = dadd(tc[1], dmul(un, y));
            tc[2] = dadd(tc[2], dmul(un, z));
        }
    }
#pragma unroll
    for (int a = 0; a < NPE; ++a) sa[a] = warp_sum(sa[a]);
#pragma unroll
    for (int c = 0; c < 3; ++c) tc[c] = warp_sum(tc[c]);
    if (lane != 0) return;
    D3 v = {0.0, 0.0, 0.0};
#pragma unroll
    for (int a = 0; a < NPE; ++a) v = {dadd(v.x, dmul(sa[a], G.dN[a][0])), dadd(v.y, dmul(sa[a], G.dN[a][1])),
                                        dadd(v.z, dmul(sa[a], G.dN[a][2]))};
    if (G.region == 3) {
        v = axpy3(v, -dot3(G.n, v), G.n);
    } else if (G.region == 2) {
        const double s = dot3(G.tan, v);
        v = {s * G.tan.x, s * G.tan.y, s * G.tan.z};
    } else {
        v = {0.0, 0.0, 0.0};
    }
    g.gpt[3 * p] = (float)v.x;
    g.gpt[3 * p + 1] = (float)v.y;
    g.gpt[3 * p + 2] = (float)v.z;
    if (g.gdir) {
        g.gdir[3 * p] = (float)tc[0];
        g.gdir[3 * p + 1] = (float)tc[1];
        g.gdir[3 * p + 2] = (float)tc[2];
    }
}

__global__ void k_bad_init(unsigned long long* bad) {
    if (threadIdx.x < 4) bad[threadIdx.x] = ULLONG_MAX;
}

inline unsigned nblk(int64_t n, int b) { return (unsigned)ceil_div(n > 0 ? n : 1, b); }

int check_mesh(const char* fn, const ds_workspace* ws, const float* verts, int64_t n_nodes, const int32_t* tets, int64_t T,
               int order) {
    DS_REQUIRE(ws && verts && tets, "%s: null argument", fn);
    DS_REQUIRE(order == 1 || order == 2, "%s: order %d is not 1 or 2", fn, order);
    DS_REQUIRE(n_nodes > 0 && T > 0, "%s: empty mesh (%lld nodes, %lld tets)", fn, (long long)n_nodes, (long long)T);
    DS_REQUIRE(n_nodes < ((int64_t)1 << 31) && T < ((int64_t)1 << 29), "%s: too many nodes or tets", fn);
    return DS_OK;
}

// ds_modal_gains and its backward: argument checks, one validation pass (one synchronisation), the launch
int gains_impl(const char* fn, ds_workspace* ws, const float* verts, int64_t n_nodes, const int32_t* tets, int64_t T,
               int order, const int32_t* bfaces, const int32_t* bowner, const int32_t* blocal, int64_t F,
               const float* points, const int32_t* face, const float* dirs, int64_t P, const double* U, int64_t ldu,
               int k, GainsArgs& g, bool backward, void* stream) {
    DS_TRY(check_mesh(fn, ws, verts, n_nodes, tets, T, order));
    DS_REQUIRE(bfaces && bowner && blocal, "%s: null boundary array", fn);
    DS_REQUIRE(F > 0 && F < ((int64_t)1 << 31), "%s: boundary face count %lld out of range", fn, (long long)F);
    DS_REQUIRE(k >= 1 && ldu >= k, "%s: bad mode block (k = %d, ldu = %lld)", fn, k, (long long)ldu);
    DS_REQUIRE(P >= 0 && P < ((int64_t)1 << 40), "%s: point count %lld out of range", fn, (long long)P);
    if (P == 0) return DS_OK;
    DS_REQUIRE(points && face && U, "%s: null argument", fn);
    DS_REQUIRE(backward ? (g.up && g.gpt) : (g.gains && g.closest), "%s: null output", fn);
    cudaStream_t st = (cudaStream_t)stream;
    g.verts = verts; g.tets = tets; g.order = order; g.k = k;
    g.bfaces = bfaces; g.owner = bowner; g.local = blocal;
    g.pts = points; g.face = face; g.dirs = dirs; g.P = P; g.U = U; g.ldu = ldu;
    DS_TRY(ws->arena.reserve(4096, st));
    unsigned long long* bad = ws->arena.take<unsigned long long>(4);
    DS_REQUIRE(bad, "%s: workspace arena exhausted", fn);
    k_bad_init<<<1, 32, 0, st>>>(bad);
    DS_LAUNCH_CHECK();
    k_gains_validate<<<std::min<int64_t>(nblk(P, 256), 1184), 256, 0, st>>>(g, F, T, n_nodes, bad);
    DS_LAUNCH_CHECK();
    unsigned long long bh[4];
    DS_CUDA(cudaMemcpyAsync(bh, bad, sizeof(bh), cudaMemcpyDeviceToHost, st));
    DS_CUDA(cudaStreamSynchronize(st));
    DS_REQUIRE(bh[0] == ULLONG_MAX, "%s: point %llu has boundary face id outside [0, %lld)", fn, bh[0], (long long)F);
    DS_REQUIRE(bh[1] == ULLONG_MAX, "%s: point %llu has a non-finite coordinate", fn, bh[1]);
    DS_REQUIRE(bh[2] == ULLONG_MAX, "%s: direction %llu has a non-finite coordinate", fn, bh[2]);
    DS_REQUIRE(bh[3] == ULLONG_MAX, "%s: the boundary face of point %llu is not a face of its owning tet", fn, bh[3]);
    ProfScope prof(PROF_GAINS, st);
    const unsigned blocks = nblk(P, GAINS_WARPS);
    if (backward) {
        if (order == 1) k_modal_gains_bwd<4><<<blocks, 32 * GAINS_WARPS, 0, st>>>(g);
        else k_modal_gains_bwd<10><<<blocks, 32 * GAINS_WARPS, 0, st>>>(g);
    } else {
        if (order == 1) k_modal_gains<4><<<blocks, 32 * GAINS_WARPS, 0, st>>>(g);
        else k_modal_gains<10><<<blocks, 32 * GAINS_WARPS, 0, st>>>(g);
    }
    DS_LAUNCH_CHECK();
    prof_account(PROF_GAINS, (double)P * (order == 1 ? 4 : 10) * 3 * k * 8, (double)P * (order == 1 ? 4 : 10) * 3 * k * 2);
    return DS_OK;
}

}  // namespace

}  // namespace ds

using namespace ds;

extern "C" int ds_tet_boundary_count(ds_workspace* ws, const float* verts, int64_t n_nodes, const int32_t* tets, int64_t T,
                                     int order, int64_t* n_faces_host, void* stream) {
    const char* fn = "ds_tet_boundary_count";
    DS_TRY(check_mesh(fn, ws, verts, n_nodes, tets, T, order));
    DS_REQUIRE(n_faces_host, "%s: null argument", fn);
    cudaStream_t st = (cudaStream_t)stream;
    ProfScope prof(PROF_GAINS, st);
    const int npe = order == 1 ? 4 : 10;
    const int64_t N = 4 * T;
    int bits = 1;
    while (bits < 32 && ((uint64_t)(n_nodes - 1) >> bits) != 0) ++bits;
    size_t tmp_sort = 0, tmp_scan = 0;
    DS_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp_sort, (uint32_t*)nullptr, (uint32_t*)nullptr, (uint32_t*)nullptr,
                                            (uint32_t*)nullptr, (int)N, 0, bits, st));
    DS_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp_scan, (int32_t*)nullptr, (int32_t*)nullptr, (int)N, st));
    const size_t tmp = std::max(tmp_sort, tmp_scan);
    DS_TRY(ws->arena.reserve(6 * ((size_t)N * 4 + 512) + tmp + 4096, st));
    Arena& a = ws->arena;
    unsigned long long* bad = a.take<unsigned long long>(4);
    uint32_t* k0 = a.take<uint32_t>(N);
    uint32_t* k1 = a.take<uint32_t>(N);
    uint32_t* v0 = a.take<uint32_t>(N);
    uint32_t* v1 = a.take<uint32_t>(N);
    int32_t* flag = a.take<int32_t>(N);
    int32_t* pos = a.take<int32_t>(N);
    void* scratch = a.take<char>(tmp);
    DS_REQUIRE(bad && k0 && k1 && v0 && v1 && flag && pos && scratch, "%s: workspace arena exhausted", fn);
    k_bad_init<<<1, 32, 0, st>>>(bad);
    DS_LAUNCH_CHECK();
    k_gb_validate<<<1184, 256, 0, st>>>(verts, n_nodes, tets, T * npe, bad);
    DS_LAUNCH_CHECK();
    unsigned long long bh[4];
    DS_CUDA(cudaMemcpyAsync(bh, bad, sizeof(bh), cudaMemcpyDeviceToHost, st));
    DS_CUDA(cudaStreamSynchronize(st));
    DS_REQUIRE(bh[0] == ULLONG_MAX, "%s: tet %llu has a node id outside [0, %lld)", fn, bh[0] / npe, (long long)n_nodes);
    DS_REQUIRE(bh[1] == ULLONG_MAX, "%s: node %llu has a non-finite coordinate", fn, bh[1]);
    // stable LSD passes: largest, middle, then smallest corner id -> faces in ascending sorted-triple order
    const unsigned blocks = nblk(N, 256);
    uint32_t *vin = v0, *vout = v1;
    for (int pass = 0; pass < 3; ++pass) {
        k_gb_keys<<<blocks, 256, 0, st>>>(tets, npe, order, N, 2 - pass, pass == 0 ? nullptr : vin, k0,
                                          pass == 0 ? vin : nullptr);
        DS_LAUNCH_CHECK();
        size_t t = tmp;
        DS_CUDA(cub::DeviceRadixSort::SortPairs(scratch, t, k0, k1, vin, vout, (int)N, 0, bits, st));
        count_launch();
        uint32_t* s = vin; vin = vout; vout = s;
    }
    k_gb_flags<<<blocks, 256, 0, st>>>(tets, npe, order, N, vin, flag, bad);
    DS_LAUNCH_CHECK();
    size_t t = tmp;
    DS_CUDA(cub::DeviceScan::ExclusiveSum(scratch, t, flag, pos, (int)N, st));
    count_launch();
    int32_t last[2] = {0, 0};
    DS_CUDA(cudaMemcpyAsync(&last[0], pos + N - 1, 4, cudaMemcpyDeviceToHost, st));
    DS_CUDA(cudaMemcpyAsync(&last[1], flag + N - 1, 4, cudaMemcpyDeviceToHost, st));
    DS_CUDA(cudaMemcpyAsync(bh, bad, sizeof(bh), cudaMemcpyDeviceToHost, st));
    DS_CUDA(cudaStreamSynchronize(st));
    DS_REQUIRE(bh[2] == ULLONG_MAX, "%s: a face of tet %llu is shared by more than two tets (non-conforming mesh)", fn, bh[2]);
    ws->gb_ptr[0] = vin; ws->gb_ptr[1] = flag; ws->gb_ptr[2] = pos;
    ws->gb_ptr[3] = (void*)tets;
    ws->gb_ptr[4] = (void*)verts;
    ws->gb_val[0] = N; ws->gb_val[1] = order; ws->gb_val[2] = last[0] + last[1];
    *n_faces_host = last[0] + last[1];
    return DS_OK;
}

extern "C" int ds_tet_boundary_fill(ds_workspace* ws, int32_t* faces_out, int32_t* owner_out, int32_t* local_out, void* stream) {
    DS_REQUIRE(ws && ws->gb_ptr[0], "ds_tet_boundary_fill: call ds_tet_boundary_count first");
    DS_REQUIRE(faces_out && owner_out && local_out, "ds_tet_boundary_fill: null output");
    cudaStream_t st = (cudaStream_t)stream;
    ProfScope prof(PROF_GAINS, st);
    const int64_t N = ws->gb_val[0];
    const int order = (int)ws->gb_val[1];
    k_gb_fill<<<nblk(N, 256), 256, 0, st>>>((const float*)ws->gb_ptr[4], (const int32_t*)ws->gb_ptr[3],
                                            order == 1 ? 4 : 10, order, N, (const uint32_t*)ws->gb_ptr[0],
                                            (const int32_t*)ws->gb_ptr[1], (const int32_t*)ws->gb_ptr[2], faces_out,
                                            owner_out, local_out);
    DS_LAUNCH_CHECK();
    ws->gb_ptr[0] = nullptr;
    return DS_OK;
}

extern "C" int ds_modal_gains(ds_workspace* ws, const float* verts, int64_t n_nodes, const int32_t* tets, int64_t T, int order,
                              const int32_t* bfaces, const int32_t* bowner, const int32_t* blocal, int64_t F,
                              const float* points, const int32_t* face, const float* dirs, int64_t P, const double* U,
                              int64_t ldu, int k, float* gains_out, float* closest_out, void* stream) {
    GainsArgs g = {};
    g.gains = gains_out;
    g.closest = closest_out;
    return gains_impl("ds_modal_gains", ws, verts, n_nodes, tets, T, order, bfaces, bowner, blocal, F, points, face, dirs,
                      P, U, ldu, k, g, false, stream);
}

extern "C" int ds_modal_gains_backward(ds_workspace* ws, const float* verts, int64_t n_nodes, const int32_t* tets, int64_t T,
                                       int order, const int32_t* bfaces, const int32_t* bowner, const int32_t* blocal,
                                       int64_t F, const float* points, const int32_t* face, const float* dirs, int64_t P,
                                       const double* U, int64_t ldu, int k, const float* grad_gains, float* grad_points,
                                       float* grad_dirs, void* stream) {
    GainsArgs g = {};
    g.up = grad_gains;
    g.gpt = grad_points;
    g.gdir = dirs ? grad_dirs : nullptr;
    return gains_impl("ds_modal_gains_backward", ws, verts, n_nodes, tets, T, order, bfaces, bowner, blocal, F, points,
                      face, dirs, P, U, ldu, k, g, true, stream);
}

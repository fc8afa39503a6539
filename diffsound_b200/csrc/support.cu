// Elastic supports: a Winkler (spring-bed) foundation on chosen boundary faces.  Nothing in the reference corresponds: it
// solves every object free-free.
//
// Support face f (a boundary face, given by its owning tet and the local index of the opposite corner, as ds_tet_boundary
// returns them) carries normal and tangential stiffnesses per unit area k_n, k_t (N/m^3); its traction is
// -(k_n n n^T + k_t (I - n n^T)) u, which adds to K
//
//     K_s,f[a, b] = int_f N_a N_b dA  S_f,   S_f = (k_n - k_t) n n^T + k_t I,
//
// N_a the face's P1 (3-node) or P2 (6-node) shape functions.  The face is affine from its three corners (as every tet is
// in assemble.cu), so int_f N_a N_b dA = A tab_ab / den exactly, with the P1 table (2, 1) / 12 and the P2 table (corner-corner
// 6 / -1, corner-opposite mid-edge -4, corner-adjacent mid-edge 0, mid-mid 32 / 16) / 180.  With the area vector
// a = 1/2 (p1 - p0) x (p2 - p0), A n n^T = a a^T / |a| and A = |a|.  M does not change.
//
// ds_support_km adds K_s into Kval in place (after the assembly, before ds_fix_nodes_km).  Every node pair of a face is a
// node pair of its owning tet, so every block exists in the pattern.  One thread per node row of the support
// incidence (node -> (face, face-local node) in ascending face order): it walks its faces in that order and adds each
// face's 3x3 block into the row's slots (the element -> slot map when the pattern has one, else a binary search of the
// row's bcol).  Each slot is written by one thread, its contributions summed in fp64 in ascending face order: no atomics,
// bitwise reproducible, and since block (i, j) and block (j, i) receive the same values in the same order, a bitwise
// symmetric K stays so.
//
// ds_support_grad / ds_support_energies: one warp per support face, lanes across modes.  Per mode the face's nodal
// displacements give the symmetric W = sum_ab tab_ab u_a u_b^T, and u^T K_s,f u = ((k_n - k_t) a^T W a / |a| +
// k_t |a| tr W) / den.  The gradient kernel reduces g_i W_i over the modes with a fixed xor-shuffle tree, then forms
// d/dk_n, d/dk_t and d/d(corner positions) through a(p0, p1, p2); a second pass sums the per-face corner gradients onto
// the nodes through the same incidence, in ascending face order.  No atomics anywhere.
#include "common.cuh"
#include "../../include/diffsound_sm100.h"
#include "closest.cuh"
#include "tet_faces.cuh"

namespace ds {

namespace {

constexpr int SUP_WARPS = 8;       // support faces per CTA of the per-face kernels (one warp each)

// face mass table in units of A / den: P1 (den 12) and P2 (den 180, face-local order: 3 corners, then the 3 mid-edge
// nodes of face_local_nodes)
__device__ __forceinline__ double face_mass(int order, int lnA, int lnB, int a, int b) {
    if (order == 1) return a == b ? 2.0 : 1.0;
    const bool ca = a < 3, cb = b < 3;
    if (ca && cb) return a == b ? 6.0 : -1.0;
    if (!ca && !cb) return a == b ? 32.0 : 16.0;
    // corner (tet-local lnC, corner index l == m) and mid-edge node (l, m): 0 when the corner is an end of the edge
    const int lc = ca ? c_p2_l[lnA] : c_p2_l[lnB];
    const int le = ca ? lnB : lnA;
    return (c_p2_l[le] == lc || c_p2_m[le] == lc) ? 0.0 : -4.0;
}

struct FaceGeom {
    int nf;                 // 3 or 6 nodes
    int ln[6];              // tet-local node ids
    int64_t node[6];        // global node ids
    D3 p[3];                // corner positions
    D3 a;                   // area vector 1/2 (p1 - p0) x (p2 - p0)
    double area;            // |a|
};

__device__ __forceinline__ D3 cross3s(D3 u, D3 v) {
    return {dsub(dmul(u.y, v.z), dmul(u.z, v.y)), dsub(dmul(u.z, v.x), dmul(u.x, v.z)), dsub(dmul(u.x, v.y), dmul(u.y, v.x))};
}

__device__ __forceinline__ void face_geom(const float* __restrict__ verts, const int32_t* __restrict__ tets, int order,
                                          int32_t t, int lf, FaceGeom& G) {
    const int npe = order == 1 ? 4 : 10;
    G.nf = face_local_nodes(order, lf, G.ln);
#pragma unroll
    for (int q = 0; q < 6; ++q) G.node[q] = q < G.nf ? (int64_t)tets[(int64_t)t * npe + G.ln[q]] : 0;
#pragma unroll
    for (int q = 0; q < 3; ++q)
        G.p[q] = {(double)verts[3 * G.node[q]], (double)verts[3 * G.node[q] + 1], (double)verts[3 * G.node[q] + 2]};
    const D3 c = cross3s(sub3(G.p[1], G.p[0]), sub3(G.p[2], G.p[0]));
    G.a = {dmul(0.5, c.x), dmul(0.5, c.y), dmul(0.5, c.z)};
    G.area = sqrt(dot3(G.a, G.a));
}

// the face's S_f |a| / den, bitwise symmetric: S[c][d] and S[d][c] are one value
__device__ __forceinline__ void face_stiffness(const FaceGeom& G, double kn, double kt, int order, double (&S)[3][3]) {
    const double den = order == 1 ? 12.0 : 180.0;
    const double an = G.area > 0.0 ? dsub(kn, kt) / G.area : 0.0;
    const double av[3] = {G.a.x, G.a.y, G.a.z};
#pragma unroll
    for (int c = 0; c < 3; ++c)
#pragma unroll
        for (int d = c; d < 3; ++d) {
            double v = dmul(an, dmul(av[c], av[d]));
            if (c == d) v = dadd(v, dmul(kt, G.area));
            S[c][d] = S[d][c] = v / den;
        }
}

__global__ void __launch_bounds__(128) k_support_km(const float* __restrict__ verts, const int32_t* __restrict__ tets, int order,
                                                    const int32_t* __restrict__ owner, const int32_t* __restrict__ local,
                                                    const double* __restrict__ kn, const double* __restrict__ kt,
                                                    const int32_t* __restrict__ inc_node, const int32_t* __restrict__ inc_ptr,
                                                    const int32_t* __restrict__ inc, int64_t R,
                                                    const int32_t* __restrict__ brow, const int32_t* __restrict__ bcol,
                                                    const int32_t* __restrict__ slot, double* __restrict__ Kval) {
    const int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (r >= R) return;
    const int npe = order == 1 ? 4 : 10;
    const int64_t i = inc_node[r];
    const int64_t b0 = brow[i];
    const int deg = (int)(brow[i + 1] - b0);
    double* krow = Kval + 9 * b0;
#pragma unroll 1
    for (int e = inc_ptr[r]; e < inc_ptr[r + 1]; ++e) {
        const int32_t s = inc[e] >> 3;
        const int a = inc[e] & 7;
        const int32_t t = owner[s];
        FaceGeom G;
        face_geom(verts, tets, order, t, local[s], G);
        double S[3][3];
        face_stiffness(G, kn[s], kt[s], order, S);
#pragma unroll 1
        for (int b = 0; b < G.nf; ++b) {
            const double m = face_mass(order, G.ln[a], G.ln[b], a, b);
            if (m == 0.0) continue;
            int p;
            if (slot) {
                p = (int)(slot[((int64_t)t * npe + G.ln[a]) * npe + G.ln[b]] - b0);
            } else {                            // bcol is ascending within the row
                const int32_t j = (int32_t)G.node[b];
                int lo = 0, hi = deg - 1;
                while (lo < hi) {
                    const int mid = (lo + hi) >> 1;
                    if (bcol[b0 + mid] < j) lo = mid + 1; else hi = mid;
                }
                p = lo;
            }
            double* k = krow + 3 * p;
#pragma unroll
            for (int c = 0; c < 3; ++c)
#pragma unroll
                for (int d = 0; d < 3; ++d) {
                    double* x = k + (int64_t)c * 3 * deg + d;
                    *x = dadd(*x, dmul(m, S[c][d]));
                }
        }
    }
}

// per face and mode: W = sum_ab tab_ab u_a u_b^T, the 6 entries (xx, yy, zz, yz, xz, xy)
__device__ __forceinline__ void face_w(const FaceGeom& G, int order, const double* __restrict__ U, int64_t ldu, int m,
                                       double (&W)[6]) {
    double u[6][3];
#pragma unroll
    for (int q = 0; q < 6; ++q)
#pragma unroll
        for (int c = 0; c < 3; ++c) u[q][c] = q < G.nf ? __ldg(U + (3 * G.node[q] + c) * ldu + m) : 0.0;
#pragma unroll
    for (int q = 0; q < 6; ++q) W[q] = 0.0;
#pragma unroll
    for (int a = 0; a < 6; ++a) {
        if (a >= G.nf) break;
        double v[3] = {0.0, 0.0, 0.0};
#pragma unroll
        for (int b = 0; b < 6; ++b) {
            if (b >= G.nf) break;
            const double t = face_mass(order, G.ln[a], G.ln[b], a, b);
#pragma unroll
            for (int c = 0; c < 3; ++c) v[c] = dadd(v[c], dmul(t, u[b][c]));
        }
        W[0] = dadd(W[0], dmul(u[a][0], v[0]));
        W[1] = dadd(W[1], dmul(u[a][1], v[1]));
        W[2] = dadd(W[2], dmul(u[a][2], v[2]));
        W[3] = dadd(W[3], dmul(u[a][1], v[2]));
        W[4] = dadd(W[4], dmul(u[a][0], v[2]));
        W[5] = dadd(W[5], dmul(u[a][0], v[1]));
    }
}

// a^T W a and W a for the symmetric W of face_w
__device__ __forceinline__ D3 w_apply(const double (&W)[6], D3 a) {
    return {dadd(dadd(dmul(W[0], a.x), dmul(W[5], a.y)), dmul(W[4], a.z)),
            dadd(dadd(dmul(W[5], a.x), dmul(W[1], a.y)), dmul(W[3], a.z)),
            dadd(dadd(dmul(W[4], a.x), dmul(W[3], a.y)), dmul(W[2], a.z))};
}

// ENERGY: out[s * k + m] = u_m^T K_s,f u_m.  Otherwise the gradient of sum_m g_m u_m^T K_s,f u_m to (k_n, k_t) -> gk[2 s],
// and to the face's three corner positions -> gface[9 s + 3 q + c]
template <bool ENERGY>
__global__ void __launch_bounds__(32 * SUP_WARPS) k_support_face(const float* __restrict__ verts,
                                                                 const int32_t* __restrict__ tets, int order,
                                                                 const int32_t* __restrict__ owner,
                                                                 const int32_t* __restrict__ local, int64_t S,
                                                                 const double* __restrict__ kn, const double* __restrict__ kt,
                                                                 const double* __restrict__ U, int64_t ldu, int k,
                                                                 const double* __restrict__ g, double* __restrict__ out,
                                                                 double* __restrict__ gk, double* __restrict__ gface) {
    const int lane = threadIdx.x & 31;
    const int64_t s = (int64_t)blockIdx.x * SUP_WARPS + (threadIdx.x >> 5);
    if (s >= S) return;
    FaceGeom G;
    face_geom(verts, tets, order, owner[s], local[s], G);
    const double den = order == 1 ? 12.0 : 180.0;
    const double ka = kn[s], kb = kt[s];
    const double inv = G.area > 0.0 ? 1.0 / G.area : 0.0;
    double Wg[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
#pragma unroll 1
    for (int m = lane; m < k; m += 32) {
        double W[6];
        face_w(G, order, U, ldu, m, W);
        if (ENERGY) {
            const double awa = dot3(G.a, w_apply(W, G.a));
            const double tr = dadd(dadd(W[0], W[1]), W[2]);
            out[s * k + m] = dadd(dmul(dmul(dsub(ka, kb), awa), inv), dmul(dmul(kb, G.area), tr)) / den;
        } else {
            const double gm = g[m];
#pragma unroll
            for (int q = 0; q < 6; ++q) Wg[q] = dadd(Wg[q], dmul(gm, W[q]));
        }
    }
    if (ENERGY) return;
#pragma unroll
    for (int q = 0; q < 6; ++q) Wg[q] = warp_sum(Wg[q]);
    if (lane != 0) return;
    const D3 Wa = w_apply(Wg, G.a);
    const double awa = dot3(G.a, Wa);
    const double tr = dadd(dadd(Wg[0], Wg[1]), Wg[2]);
    // h(a) = (k_n - k_t) a^T W a / |a| + k_t |a| tr W;  dh/dk_n, dh/dk_t, dh/da
    gk[2 * s] = dmul(awa, inv) / den;
    gk[2 * s + 1] = dsub(dmul(G.area, tr), dmul(awa, inv)) / den;
    const double c1 = dmul(2.0 * dsub(ka, kb), inv);
    const double c2 = dsub(dmul(kb, dmul(tr, inv)), dmul(dsub(ka, kb), dmul(awa, dmul(inv, dmul(inv, inv)))));
    const D3 H = {dadd(dmul(c1, Wa.x), dmul(c2, G.a.x)) / den, dadd(dmul(c1, Wa.y), dmul(c2, G.a.y)) / den,
                  dadd(dmul(c1, Wa.z), dmul(c2, G.a.z)) / den};
    // a = 1/2 e1 x e2 (e1 = p1 - p0, e2 = p2 - p0): dh/dp1 = 1/2 e2 x H, dh/dp2 = 1/2 H x e1, dh/dp0 = -(their sum)
    const D3 e1 = sub3(G.p[1], G.p[0]), e2 = sub3(G.p[2], G.p[0]);
    const D3 g1 = cross3s(e2, H), g2 = cross3s(H, e1);
    const double gp[3][3] = {{-0.5 * dadd(g1.x, g2.x), -0.5 * dadd(g1.y, g2.y), -0.5 * dadd(g1.z, g2.z)},
                             {0.5 * g1.x, 0.5 * g1.y, 0.5 * g1.z},
                             {0.5 * g2.x, 0.5 * g2.y, 0.5 * g2.z}};
#pragma unroll
    for (int q = 0; q < 3; ++q)
#pragma unroll
        for (int c = 0; c < 3; ++c) gface[9 * s + 3 * q + c] = gp[q][c];
}

// grad[node] = sum over the node's support faces (ascending) of the face's corner gradient; one thread per incidence row
__global__ void k_support_gather(const int32_t* __restrict__ inc_node, const int32_t* __restrict__ inc_ptr,
                                 const int32_t* __restrict__ inc, int64_t R, const double* __restrict__ gface,
                                 double* __restrict__ grad) {
    const int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (r >= R) return;
    double v[3] = {0.0, 0.0, 0.0};
    for (int e = inc_ptr[r]; e < inc_ptr[r + 1]; ++e) {
        const int a = inc[e] & 7;
        if (a >= 3) continue;                   // mid-edge nodes: the face geometry does not depend on them
        const double* x = gface + 9 * (int64_t)(inc[e] >> 3) + 3 * a;
#pragma unroll
        for (int c = 0; c < 3; ++c) v[c] = dadd(v[c], x[c]);
    }
    const int64_t i = inc_node[r];
#pragma unroll
    for (int c = 0; c < 3; ++c) grad[3 * i + c] = v[c];
}

int check_faces(const char* fn, const float* verts, const int32_t* tets, int64_t T, int order, int64_t n_nodes,
                const int32_t* owner, const int32_t* local, int64_t S, const double* kn, const double* kt) {
    DS_REQUIRE(verts && tets && owner && local && kn && kt, "%s: null argument", fn);
    DS_REQUIRE(order == 1 || order == 2, "%s: order %d is not 1 or 2", fn, order);
    DS_REQUIRE(n_nodes > 0 && T > 0 && n_nodes < ((int64_t)1 << 31) && T < ((int64_t)1 << 29),
               "%s: bad mesh sizes (%lld nodes, %lld tets)", fn, (long long)n_nodes, (long long)T);
    DS_REQUIRE(S > 0 && S < ((int64_t)1 << 28), "%s: support face count %lld out of range", fn, (long long)S);
    return DS_OK;
}

int check_incidence(const char* fn, const int32_t* inc_node, const int32_t* inc_ptr, const int32_t* inc, int64_t R,
                    int64_t S) {
    DS_REQUIRE(inc_node && inc_ptr && inc, "%s: null incidence", fn);
    DS_REQUIRE(R > 0 && R <= 6 * S, "%s: incidence row count %lld out of range for %lld faces", fn, (long long)R,
               (long long)S);
    return DS_OK;
}

}  // namespace

}  // namespace ds

using namespace ds;

extern "C" int ds_support_km(const float* verts, const int32_t* tets, int64_t T, int order, int64_t n_nodes,
                             const int32_t* owner, const int32_t* local, int64_t S, const double* kn, const double* kt,
                             const int32_t* inc_node, const int32_t* inc_ptr, const int32_t* inc, int64_t R,
                             const int32_t* brow, const int32_t* bcol, const int32_t* slot, int64_t nnzb, double* Kval,
                             void* stream) {
    const char* fn = "ds_support_km";
    DS_TRY(check_faces(fn, verts, tets, T, order, n_nodes, owner, local, S, kn, kt));
    DS_TRY(check_incidence(fn, inc_node, inc_ptr, inc, R, S));
    DS_REQUIRE(brow && bcol && Kval, "%s: null pattern or Kval", fn);
    DS_REQUIRE(nnzb >= n_nodes, "%s: bad pattern (n_nodes=%lld, nnzb=%lld)", fn, (long long)n_nodes, (long long)nnzb);
    cudaStream_t st = (cudaStream_t)stream;
    ProfScope prof(PROF_SUPPORT, st);
    const int nf = order == 1 ? 3 : 6;
    prof_account(PROF_SUPPORT, (double)S * nf * nf * 9 * 16, (double)S * nf * nf * 9 * 2);
    k_support_km<<<(unsigned)ceil_div(R, 128), 128, 0, st>>>(verts, tets, order, owner, local, kn, kt, inc_node, inc_ptr, inc,
                                                              R, brow, bcol, slot, Kval);
    DS_LAUNCH_CHECK();
    return DS_OK;
}

extern "C" int ds_support_grad(const float* verts, const int32_t* tets, int64_t T, int order, int64_t n_nodes,
                               const int32_t* owner, const int32_t* local, int64_t S, const double* kn, const double* kt,
                               const double* U, int64_t ldu, int k, const double* g, const int32_t* inc_node,
                               const int32_t* inc_ptr, const int32_t* inc, int64_t R, double* face_scratch,
                               double* grad_k, double* grad_verts, void* stream) {
    const char* fn = "ds_support_grad";
    DS_TRY(check_faces(fn, verts, tets, T, order, n_nodes, owner, local, S, kn, kt));
    DS_REQUIRE(U && g && grad_k && face_scratch, "%s: null argument", fn);
    DS_REQUIRE(k >= 1 && ldu >= k, "%s: bad mode block (k = %d, ldu = %lld)", fn, k, (long long)ldu);
    if (grad_verts) DS_TRY(check_incidence(fn, inc_node, inc_ptr, inc, R, S));
    cudaStream_t st = (cudaStream_t)stream;
    ProfScope prof(PROF_SUPPORT, st);
    const int nf = order == 1 ? 3 : 6;
    prof_account(PROF_SUPPORT, (double)S * k * nf * 3 * 8, (double)S * k * nf * (nf + 3) * 6);
    k_support_face<false><<<(unsigned)ceil_div(S, SUP_WARPS), 32 * SUP_WARPS, 0, st>>>(
        verts, tets, order, owner, local, S, kn, kt, U, ldu, k, g, nullptr, grad_k, face_scratch);
    DS_LAUNCH_CHECK();
    if (grad_verts) {
        DS_CUDA(cudaMemsetAsync(grad_verts, 0, sizeof(double) * 3 * n_nodes, st));
        k_support_gather<<<(unsigned)ceil_div(R, 128), 128, 0, st>>>(inc_node, inc_ptr, inc, R, face_scratch, grad_verts);
        DS_LAUNCH_CHECK();
    }
    return DS_OK;
}

extern "C" int ds_support_energies(const float* verts, const int32_t* tets, int64_t T, int order, int64_t n_nodes,
                                   const int32_t* owner, const int32_t* local, int64_t S, const double* kn, const double* kt,
                                   const double* U, int64_t ldu, int k, double* out, void* stream) {
    const char* fn = "ds_support_energies";
    DS_TRY(check_faces(fn, verts, tets, T, order, n_nodes, owner, local, S, kn, kt));
    DS_REQUIRE(U && out, "%s: null argument", fn);
    DS_REQUIRE(k >= 1 && ldu >= k, "%s: bad mode block (k = %d, ldu = %lld)", fn, k, (long long)ldu);
    cudaStream_t st = (cudaStream_t)stream;
    ProfScope prof(PROF_SUPPORT, st);
    const int nf = order == 1 ? 3 : 6;
    prof_account(PROF_SUPPORT, (double)S * k * (nf * 3 + 1) * 8, (double)S * k * nf * (nf + 3) * 6);
    k_support_face<true><<<(unsigned)ceil_div(S, SUP_WARPS), 32 * SUP_WARPS, 0, st>>>(
        verts, tets, order, owner, local, S, kn, kt, U, ldu, k, nullptr, out, nullptr, nullptr);
    DS_LAUNCH_CHECK();
    return DS_OK;
}

// Eigenvalue derivatives: d(lambda)/d(vertices) and the material quadratic forms.
//
// Reference behaviour replaced (file:line under /root/reference/src):
//   diffelastic/diff_model.py:390-399  get_vals(): lambda + diag(U^T K U) - lambda diag(U^T M U), whose
//       autograd backward walks sparse-mm -> coalesce -> bmm -> torch.inverse -> vertices;
//   diffelastic/diff_model.py:314-328, 371-388 + deform.py:70-87, 149-165  the fp32 matrix-free
//       K(theta) U (gather -> F -> P -> scatter-add) behind get_undamped_freqs().
//
// Shape gradient.  For weights g_i the scalar E = sum_i g_i (u_i^T K u_i - lam_i u_i^T M u_i) splits per
// element.  With W = U_e diag(g) U_e^T (the weighted Gram of the element's rows of U, DMMA) and the
// same contraction table as assembly,
//     Q_lm = sum_ab ctab[a][b][l][m] W_ab              (3x3, 16 of them)
//     e(G) = sum_lm mu tr(Q_lm) G_l.G_m + mu G_m^T Q_lm G_l + lam G_l^T Q_lm G_m
//     E_K  = |det A| e(G),     E_M = -|det6V| sum_ab mtab[a][b] tr(W'_ab),  W' weighted by g_i lam_i
// e is a quadratic form in the 4x3 matrix G = dL/dxi A^-1, so dE/dG is linear in G and the chain
// rule to the four corner positions is closed form.  One warp per element; per-corner results go to
// tet_grad and are summed per node by a gather kernel (deterministic, no atomics).
//
// Material forms.  lane = mode.  Linear tets have a constant displacement gradient F; for quadratic
// tets F is linear in the barycentric coordinates, F(L) = sum_m L_m F_m with F_m its value at corner
// m, so the exact integral of a quadratic form phi is |det A|/120 (phi(sum_m F_m) + sum_m phi(F_m)).
//
// Material fields.  The same element forms per (tet, mode) give d lambda_i / d(mu_t, lam_t, rho_t) and the element
// energies (k_material_field); the shape gradient reads (mu_t, lam_t, rho_t) per element (k_eigval_grad_shape<_, MAT_LAME>).
//
// Elasticity-tensor fields (Voigt convention of csrc/assemble.cu, C_t packed as 21 upper-triangle entries).  With
// C_{ckdl} the rank-4 form of C_t, e(G) = sum_{p,m} Q_pm[c][d] C_{ckdl} G_p[k] G_m[l], and by the major symmetry of C
//     de/dG_p[j] = 2 sum_m sum_{c,d,k} Q_pm[c][d] C_{cjdk} G_m[k]                (k_eigval_grad_shape<_, MAT_TENSOR>).
// d lambda_i / dC_t is the strain Gram E_t,i = int_t eps_V(u_i) eps_V(u_i)^T dV, integrated exactly like the material
// forms (k_elasticity_field); lambda_i = sum_t <C_t, E_t,i> because the strain energy is quadratic in eps.
#include "common.cuh"
#include "../../include/diffsound_sm100.h"
#include "kernels.cuh"
#include <cub/cub.cuh>
#include <type_traits>

namespace ds {

__device__ __forceinline__ void dmma884(double& d0, double& d1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(d0), "+d"(d1)
                 : "d"(a), "d"(b));
}

// nodes whose shape function depends on barycentric coordinate l (quadratic tet, reference local order)
__device__ __constant__ int c_L2[4][4] = {{0, 1, 5, 6}, {2, 1, 3, 7}, {4, 3, 5, 8}, {9, 6, 7, 8}};

struct TetGeom {
    double G[4][3];   // rows of dL/dxi A^-1
    double detK;      // |det A| (A from fp32 differences, as mesh.py:90-98)
    double detM;      // |6V| from fp64 corner coordinates (diff_model.py:272-289)
    double sgnM;      // sign of the signed 6V
    double dD[4][3];  // d(6V signed)/d(corner)
};

template <bool WITH_DD>
__device__ __forceinline__ void tet_geometry(const float* __restrict__ verts, const int32_t c[4], TetGeom& g) {
    float v[4][3];
#pragma unroll
    for (int p = 0; p < 4; ++p) {
        v[p][0] = __ldg(verts + 3 * (int64_t)c[p] + 0);
        v[p][1] = __ldg(verts + 3 * (int64_t)c[p] + 1);
        v[p][2] = __ldg(verts + 3 * (int64_t)c[p] + 2);
    }
    double A[3][3];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        A[r][0] = (double)__fsub_rn(v[0][r], v[3][r]);
        A[r][1] = (double)__fsub_rn(v[1][r], v[3][r]);
        A[r][2] = (double)__fsub_rn(v[2][r], v[3][r]);
    }
    double c00 = A[1][1] * A[2][2] - A[1][2] * A[2][1];
    double c01 = A[1][2] * A[2][0] - A[1][0] * A[2][2];
    double c02 = A[1][0] * A[2][1] - A[1][1] * A[2][0];
    double det = A[0][0] * c00 + A[0][1] * c01 + A[0][2] * c02;
    double id = 1.0 / det;
    g.G[0][0] = c00 * id;
    g.G[0][1] = (A[0][2] * A[2][1] - A[0][1] * A[2][2]) * id;
    g.G[0][2] = (A[0][1] * A[1][2] - A[0][2] * A[1][1]) * id;
    g.G[1][0] = c01 * id;
    g.G[1][1] = (A[0][0] * A[2][2] - A[0][2] * A[2][0]) * id;
    g.G[1][2] = (A[0][2] * A[1][0] - A[0][0] * A[1][2]) * id;
    g.G[2][0] = c02 * id;
    g.G[2][1] = (A[0][1] * A[2][0] - A[0][0] * A[2][1]) * id;
    g.G[2][2] = (A[0][0] * A[1][1] - A[0][1] * A[1][0]) * id;
#pragma unroll
    for (int d = 0; d < 3; ++d) g.G[3][d] = -(g.G[0][d] + g.G[1][d] + g.G[2][d]);
    g.detK = fabs(det);
    double e1[3], e2[3], e3[3];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        e1[r] = (double)v[1][r] - (double)v[0][r];
        e2[r] = (double)v[2][r] - (double)v[0][r];
        e3[r] = (double)v[3][r] - (double)v[0][r];
    }
    double n1[3] = {e2[1] * e3[2] - e2[2] * e3[1], e2[2] * e3[0] - e2[0] * e3[2], e2[0] * e3[1] - e2[1] * e3[0]};
    double D = e1[0] * n1[0] + e1[1] * n1[1] + e1[2] * n1[2];
    g.detM = fabs(D);
    g.sgnM = D < 0.0 ? -1.0 : 1.0;
    if (WITH_DD) {
        double n2[3] = {e3[1] * e1[2] - e3[2] * e1[1], e3[2] * e1[0] - e3[0] * e1[2], e3[0] * e1[1] - e3[1] * e1[0]};
        double n3[3] = {e1[1] * e2[2] - e1[2] * e2[1], e1[2] * e2[0] - e1[0] * e2[2], e1[0] * e2[1] - e1[1] * e2[0]};
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            g.dD[1][r] = n1[r];
            g.dD[2][r] = n2[r];
            g.dD[3][r] = n3[r];
            g.dD[0][r] = -(n1[r] + n2[r] + n3[r]);
        }
    }
}

__device__ __forceinline__ void load_corners(const int32_t* __restrict__ t, int order, int32_t c[4]) {
    if (order == 1) {
        c[0] = __ldg(t + 0); c[1] = __ldg(t + 1); c[2] = __ldg(t + 2); c[3] = __ldg(t + 3);
    } else {
        c[0] = __ldg(t + 0); c[1] = __ldg(t + 2); c[2] = __ldg(t + 4); c[3] = __ldg(t + 9);
    }
}

// ---------------------------------------------------------------------------
// shape gradient
// ---------------------------------------------------------------------------
constexpr int GS_WARPS = 4;
constexpr int GS_WLD = 33;   // leading dimension of the per-warp W tile in shared memory

template <int ORDER>
struct GradSmem {
    static constexpr int NPE = ORDER == 1 ? 4 : 10;
    static constexpr int ROWS = 3 * NPE;                 // 12 | 30
    static constexpr int RT = (ROWS + 7) / 8;            // 2 | 4 row tiles
    static constexpr int RP = RT * 8;                    // padded rows 16 | 32
    double ctab[NPE * NPE * 16];
    double mhat[RP * RP];                                // (mtab (x) I3), zero padded
    double W[GS_WARPS][RP * GS_WLD];
    double Q[GS_WARPS][192];                             // 144 Q entries, 12 dE/dG, 12 G (at 160), 12 dD (at 172)
};

// tensor fields: one packed elasticity tensor per warp in addition
template <int ORDER>
struct GradSmemTensor : GradSmem<ORDER> {
    double C[GS_WARPS][24];
};

template <int ORDER, int MODE>
using GradSmemOf = std::conditional_t<MODE == MAT_TENSOR, GradSmemTensor<ORDER>, GradSmem<ORDER>>;

// Per-tet material of the field variants (ds_eigval_grad_shape_field, ds_eigval_grad_shape_tensor); unused by the
// scalar instantiation.
struct GradField {
    const double* __restrict__ mu;
    const double* __restrict__ lam;
    const float* __restrict__ rho;
    const double* __restrict__ C;   // [T][21]
};

// MAT_LAME: mu, lam of element e from the field; MAT_TENSOR: its elasticity tensor.  Both: mtab_g the unit-density table
// (promoted fp32) and the mass part of the element scaled by rho_e.
template <int ORDER, int MODE>
__global__ void __launch_bounds__(GS_WARPS * 32)
k_eigval_grad_shape(const float* __restrict__ verts, const int32_t* __restrict__ tets, int64_t T, double mu_s,
                    double lam_s, GradField f, const double* __restrict__ ctab_g, const double* __restrict__ mtab_g,
                    const double* __restrict__ U, int64_t ldu, int k, const double* __restrict__ lamv,
                    const double* __restrict__ gv, double* __restrict__ tet_grad) {
    using SM = GradSmemOf<ORDER, MODE>;
    constexpr bool FIELD = MODE != MAT_SCALAR;
    constexpr int NPE = SM::NPE, ROWS = SM::ROWS, RT = SM::RT, RP = SM::RP;
    constexpr int NL = ORDER == 1 ? 1 : 4;
    constexpr int NTILE = RT * (RT + 1) / 2;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    SM& sm = *reinterpret_cast<SM*>(smem_raw);
    double* s_w = reinterpret_cast<double*>(smem_raw + sizeof(SM));   // [2][kpad]: g, g*lam
    const int kpad = (k + 15) & ~15;
    for (int t = threadIdx.x; t < NPE * NPE * 16; t += blockDim.x) sm.ctab[t] = ctab_g[t];
    for (int t = threadIdx.x; t < RP * RP; t += blockDim.x) {
        int r = t / RP, c = t - r * RP;
        sm.mhat[t] = (r < ROWS && c < ROWS && (r % 3) == (c % 3)) ? mtab_g[(r / 3) * NPE + (c / 3)] : 0.0;
    }
    for (int t = threadIdx.x; t < kpad; t += blockDim.x) {
        double g = t < k ? gv[t] : 0.0;
        s_w[t] = g;
        s_w[kpad + t] = t < k ? g * lamv[t] : 0.0;
    }
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int mm = lane >> 2, kk = lane & 3;
    double* Ws = sm.W[warp];
    double* Qs = sm.Q[warp];
    const int64_t wstride = (int64_t)gridDim.x * GS_WARPS;
    for (int64_t e = (int64_t)blockIdx.x * GS_WARPS + warp; e < T; e += wstride) {
        const int32_t* tp = tets + e * NPE;
        const double mu = MODE == MAT_LAME ? __ldg(f.mu + e) : mu_s;
        const double lam = MODE == MAT_LAME ? __ldg(f.lam + e) : lam_s;
        if constexpr (MODE == MAT_TENSOR) {
            if (lane < 21) sm.C[warp][lane] = __ldg(f.C + e * 21 + lane);
        }
        int32_t cn[4];
        load_corners(tp, ORDER, cn);
        TetGeom geo;
        tet_geometry<true>(verts, cn, geo);
        if (lane < 12) {   // lane-indexed reads of G and dD go through shared memory (no local-memory arrays)
            const int p = lane / 3, j = lane - 3 * p;
            double gv_ = 0.0, dv_ = 0.0;
#pragma unroll
            for (int pp = 0; pp < 4; ++pp)
#pragma unroll
                for (int jj = 0; jj < 3; ++jj)
                    if (pp == p && jj == j) { gv_ = geo.G[pp][jj]; dv_ = geo.dD[pp][jj]; }
            Qs[160 + lane] = gv_;
            Qs[172 + lane] = dv_;
        }
        const double* Gs = Qs + 160;
        // ---- weighted Grams of the element rows of U on the FP64 tensor pipe
        const double* rowp[RT];
#pragma unroll
        for (int ti = 0; ti < RT; ++ti) {
            int r = 8 * ti + mm;
            rowp[ti] = nullptr;
            if (r < ROWS) {
                int64_t node = __ldg(tp + r / 3);
                rowp[ti] = U + (3 * node + (r % 3)) * ldu;
            }
        }
        double accK[NTILE][2], accM[NTILE][2];
#pragma unroll
        for (int t = 0; t < NTILE; ++t) accK[t][0] = accK[t][1] = accM[t][0] = accM[t][1] = 0.0;
        for (int k0 = 0; k0 < kpad; k0 += 16) {
            const int kb = k0 + 4 * kk;   // this lane's four consecutive modes
            double u[RT][4];
#pragma unroll
            for (int ti = 0; ti < RT; ++ti) {
#pragma unroll
                for (int j = 0; j < 4; ++j) u[ti][j] = (rowp[ti] && kb + j < k) ? __ldg(rowp[ti] + kb + j) : 0.0;
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                double wk = s_w[kb + j], wm = s_w[kpad + kb + j];
                double bK[RT], bM[RT];
#pragma unroll
                for (int ti = 0; ti < RT; ++ti) {
                    bK[ti] = u[ti][j] * wk;
                    bM[ti] = u[ti][j] * wm;
                }
                int t = 0;
#pragma unroll
                for (int ti = 0; ti < RT; ++ti)
#pragma unroll
                    for (int tj = ti; tj < RT; ++tj, ++t) {
                        dmma884(accK[t][0], accK[t][1], u[ti][j], bK[tj]);
                        dmma884(accM[t][0], accM[t][1], u[ti][j], bM[tj]);
                    }
            }
        }
        double s_mass = 0.0;
        {
            int t = 0;
#pragma unroll
            for (int ti = 0; ti < RT; ++ti)
#pragma unroll
                for (int tj = ti; tj < RT; ++tj, ++t) {
                    int r = 8 * ti + mm, c = 8 * tj + 2 * kk;
                    Ws[r * GS_WLD + c] = accK[t][0];
                    Ws[r * GS_WLD + c + 1] = accK[t][1];
                    if (ti != tj) {
                        Ws[c * GS_WLD + r] = accK[t][0];
                        Ws[(c + 1) * GS_WLD + r] = accK[t][1];
                    }
                    double f = ti == tj ? 1.0 : 2.0;
                    s_mass += f * (sm.mhat[r * RP + c] * accM[t][0] + sm.mhat[r * RP + c + 1] * accM[t][1]);
                }
        }
        s_mass = warp_sum(s_mass);
        if (FIELD) s_mass *= (double)__ldg(f.rho + e);
        __syncwarp();
        // ---- Q_lm = sum_ab ctab[a][b][l][m] W_ab
        for (int o = lane; o < 144; o += 32) {
            int lmi = o / 9, cd = o - lmi * 9;
            int l = lmi >> 2, m = lmi & 3, c = cd / 3, d = cd - 3 * c;
            double acc = 0.0;
#pragma unroll
            for (int ai = 0; ai < NL; ++ai) {
                int a = ORDER == 1 ? l : c_L2[l][ai];
#pragma unroll
                for (int bi = 0; bi < NL; ++bi) {
                    int b = ORDER == 1 ? m : c_L2[m][bi];
                    acc = fma(sm.ctab[((a * NPE + b) * 4 + l) * 4 + m], Ws[(3 * a + c) * GS_WLD + 3 * b + d], acc);
                }
            }
            Qs[o] = acc;
        }
        __syncwarp();
        // ---- dE/dG (lanes 0..11 = (p, j)) and e = 1/2 G : dE/dG
        double dG = 0.0;
        if constexpr (MODE == MAT_TENSOR) {
            if (lane < 12) {
                const int p = lane / 3, j = lane - 3 * p;
                const double* Cs = sm.C[warp];
                double Cj[3][3][3];     // C_{cjdk} of this lane's j
#pragma unroll
                for (int c = 0; c < 3; ++c)
#pragma unroll
                    for (int d = 0; d < 3; ++d)
#pragma unroll
                        for (int k = 0; k < 3; ++k) Cj[c][d][k] = Cs[voigt_packed(voigt(c, j), voigt(d, k))];
#pragma unroll
                for (int m = 0; m < 4; ++m) {
                    const double* Qpm = Qs + (p * 4 + m) * 9;
                    double s = 0.0;
#pragma unroll
                    for (int c = 0; c < 3; ++c)
#pragma unroll
                        for (int d = 0; d < 3; ++d)
                            s = fma(Qpm[3 * c + d],
                                    fma(Cj[c][d][0], geo.G[m][0], fma(Cj[c][d][1], geo.G[m][1], Cj[c][d][2] * geo.G[m][2])), s);
                    dG = fma(2.0, s, dG);
                }
            }
        } else if (lane < 12) {
            int p = lane / 3, j = lane - 3 * p;
#pragma unroll
            for (int m = 0; m < 4; ++m) {
                const double* Qpm = Qs + (p * 4 + m) * 9;
                const double* Qmp = Qs + (m * 4 + p) * 9;
                double tpm = Qpm[0] + Qpm[4] + Qpm[8];
                double s1 = Qmp[j * 3 + 0] * geo.G[m][0] + Qmp[j * 3 + 1] * geo.G[m][1] + Qmp[j * 3 + 2] * geo.G[m][2];
                double s2 = Qpm[j * 3 + 0] * geo.G[m][0] + Qpm[j * 3 + 1] * geo.G[m][1] + Qpm[j * 3 + 2] * geo.G[m][2];
                dG += 2.0 * mu * (tpm * Gs[3 * m + j] + s1) + 2.0 * lam * s2;
            }
        }
        double ee = 0.0;
        if (lane < 12) {
            int p = lane / 3, j = lane - 3 * p;
            ee = 0.5 * Gs[lane] * dG;
            Qs[144 + lane] = dG;
        }
        ee = warp_sum(ee);
        __syncwarp();
        // ---- chain rule to the four corners (lanes 0..11 = (corner p, coordinate r))
        if (lane < 12) {
            int p = lane / 3, r = lane - 3 * p;
            double B[3][3];   // B[l][d] = dG_l[d] - dG_3[d]
#pragma unroll
            for (int l = 0; l < 3; ++l)
#pragma unroll
                for (int d = 0; d < 3; ++d) B[l][d] = Qs[144 + 3 * l + d] - Qs[144 + 9 + d];
            // Abar[r][q] = detK * ( e Ai[q][r] - (Ai B^T Ai)[q][r] ),  Ai[q][:] = G[q][:]
            double val = 0.0;
#pragma unroll
            for (int q = 0; q < 3; ++q) {
                double t = 0.0;
#pragma unroll
                for (int i = 0; i < 3; ++i) {
                    double bt = B[0][i] * Gs[r] + B[1][i] * Gs[3 + r] + B[2][i] * Gs[6 + r];   // (B^T Ai)[i][r]
                    t += geo.G[q][i] * bt;
                }
                double aq = geo.detK * (ee * Gs[3 * q + r] - t);
                if (p == q) val += aq;
                if (p == 3) val -= aq;
            }
            val -= s_mass * geo.sgnM * Qs[172 + lane];
            tet_grad[e * 12 + lane] = val;
        }
        __syncwarp();
    }
}

// grad_verts[node] = sum over incident (tet, corner) of tet_grad, cast to fp32
__global__ void k_node_gather(const int32_t* __restrict__ inc_ptr, const int32_t* __restrict__ inc,
                              const double* __restrict__ tet_grad, int64_t n_nodes, float* __restrict__ grad_verts) {
    int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= 3 * n_nodes) return;
    int64_t node = t / 3;
    int r = (int)(t - 3 * node);
    double s = 0.0;
    for (int q = inc_ptr[node]; q < inc_ptr[node + 1]; ++q) s += tet_grad[(int64_t)inc[q] * 3 + r];
    grad_verts[t] = (float)s;
}

__global__ void k_corner_keys(const int32_t* __restrict__ tets, int64_t T, int npe, int order,
                              uint32_t* __restrict__ keys, uint32_t* __restrict__ vals) {
    int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (q >= 4 * T) return;
    int64_t e = q >> 2;
    int p = (int)(q & 3);
    int loc = order == 1 ? p : (p == 3 ? 9 : 2 * p);
    keys[q] = (uint32_t)tets[e * npe + loc];
    vals[q] = (uint32_t)q;
}

__global__ void k_inc_ptr(const uint32_t* __restrict__ keys, int64_t nq, int64_t n_nodes, int32_t* __restrict__ inc_ptr) {
    int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (q >= nq) return;
    int64_t cur = keys[q];
    int64_t prev = q == 0 ? -1 : (int64_t)keys[q - 1];
    for (int64_t r = prev + 1; r <= cur; ++r) inc_ptr[r] = (int32_t)q;
    if (q == nq - 1)
        for (int64_t r = cur + 1; r <= n_nodes; ++r) inc_ptr[r] = (int32_t)nq;
}

// ---------------------------------------------------------------------------
// material quadratic forms
// ---------------------------------------------------------------------------
constexpr int QF_WARPS = 4;
constexpr int QF_MAX_CTAS = 148 * 4;

__device__ __forceinline__ void phi_pair(const double F[3][3], double& pmu, double& plam) {
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) s = fma(F[i][j], F[i][j] + F[j][i], s);
    double tr = F[0][0] + F[1][1] + F[2][2];
    pmu = s;
    plam = tr * tr;
}

template <int ORDER>
__global__ void __launch_bounds__(QF_WARPS * 32)
k_quadforms(const float* __restrict__ verts, const int32_t* __restrict__ tets, int64_t T,
            const double* __restrict__ mtab_g, double wsum, const double* __restrict__ U, int64_t ldu, int k,
            double* __restrict__ partial) {
    constexpr int NPE = ORDER == 1 ? 4 : 10;
    __shared__ double s_mtab[NPE * NPE];
    for (int t = threadIdx.x; t < NPE * NPE; t += blockDim.x) s_mtab[t] = mtab_g[t];
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t gw = (int64_t)blockIdx.x * QF_WARPS + warp;
    const int64_t wstride = (int64_t)gridDim.x * QF_WARPS;
    const int kpad = (k + 31) & ~31;
    for (int i0 = 0; i0 < kpad; i0 += 32) {
        const int i = i0 + lane;
        const bool on = i < k;
        double q_mu = 0.0, q_la = 0.0, q_m = 0.0;
        for (int64_t e = gw; e < T; e += wstride) {
            const int32_t* tp = tets + e * NPE;
            int32_t cn[4];
            load_corners(tp, ORDER, cn);
            TetGeom geo;
            tet_geometry<false>(verts, cn, geo);
            double u[NPE][3];
#pragma unroll
            for (int a = 0; a < NPE; ++a) {
                int64_t node = __ldg(tp + a);
#pragma unroll
                for (int c = 0; c < 3; ++c) u[a][c] = on ? __ldg(U + (3 * node + c) * ldu + i) : 0.0;
            }
            // mass form
            double ms = 0.0;
#pragma unroll
            for (int a = 0; a < NPE; ++a) {
                double ta[3] = {0.0, 0.0, 0.0};
#pragma unroll
                for (int b = a + 1; b < NPE; ++b) {
                    double mab = s_mtab[a * NPE + b];
                    ta[0] = fma(mab, u[b][0], ta[0]);
                    ta[1] = fma(mab, u[b][1], ta[1]);
                    ta[2] = fma(mab, u[b][2], ta[2]);
                }
                double maa = s_mtab[a * NPE + a];
#pragma unroll
                for (int c = 0; c < 3; ++c) ms = fma(u[a][c], fma(maa, u[a][c], 2.0 * ta[c]), ms);
            }
            q_m = fma(geo.detM, ms, q_m);
            if (ORDER == 1) {
                double F[3][3];
#pragma unroll
                for (int r = 0; r < 3; ++r)
#pragma unroll
                    for (int j = 0; j < 3; ++j)
                        F[r][j] = u[0][r] * geo.G[0][j] + u[1][r] * geo.G[1][j] + u[2][r] * geo.G[2][j] +
                                  u[3][r] * geo.G[3][j];
                double pm, pl;
                phi_pair(F, pm, pl);
                q_mu = fma(geo.detK * wsum, pm, q_mu);
                q_la = fma(geo.detK * wsum, pl, q_la);
            } else {
                // corner / edge nodes in the reference local order
                constexpr int CORNER[4] = {0, 2, 4, 9};
                constexpr int EDGE[4][4] = {{-1, 1, 5, 6}, {1, -1, 3, 7}, {5, 3, -1, 8}, {6, 7, 8, -1}};
                double S[3][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}};
                double smu = 0.0, sla = 0.0;
#pragma unroll
                for (int m = 0; m < 4; ++m) {
                    double F[3][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}};
#pragma unroll
                    for (int l = 0; l < 4; ++l) {
                        double h[3];
#pragma unroll
                        for (int r = 0; r < 3; ++r)
                            h[r] = (l == m) ? 3.0 * u[CORNER[l]][r] : 4.0 * u[EDGE[l][m] < 0 ? 0 : EDGE[l][m]][r] - u[CORNER[l]][r];
#pragma unroll
                        for (int r = 0; r < 3; ++r)
#pragma unroll
                            for (int j = 0; j < 3; ++j) F[r][j] = fma(h[r], geo.G[l][j], F[r][j]);
                    }
                    double pm, pl;
                    phi_pair(F, pm, pl);
                    smu += pm;
                    sla += pl;
#pragma unroll
                    for (int r = 0; r < 3; ++r)
#pragma unroll
                        for (int j = 0; j < 3; ++j) S[r][j] += F[r][j];
                }
                double pm, pl;
                phi_pair(S, pm, pl);
                const double w = geo.detK * (1.0 / 120.0);
                q_mu = fma(w, smu + pm, q_mu);
                q_la = fma(w, sla + pl, q_la);
            }
        }
        if (on) {
            double* out = partial + gw * 3 * (int64_t)k;
            out[i] = q_mu;
            out[k + i] = q_la;
            out[2 * k + i] = q_m;
        }
    }
}

__global__ void k_quadform_reduce(const double* __restrict__ partial, int nparts, int width, double* __restrict__ out) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= width) return;
    double s = 0.0;
    for (int p = 0; p < nparts; ++p) s += partial[(size_t)p * width + t];
    out[t] = s;
}

// ---------------------------------------------------------------------------
// material-field gradient and element energies
// ---------------------------------------------------------------------------
// One warp per tet, lane = mode (chunks of 32 modes), the element forms of k_quadforms per (tet, mode):
//     q_mu = u^T K_mu,t u,  q_lam = u^T K_lam,t u,  q_m = u^T Mhat_t u  (Mhat_t: unit-density mass of tet t).
// GRAD:   out[t] = (sum_i g_i q_mu, sum_i g_i q_lam, -sum_i g_i lam_i q_m), summed over the lanes by a fixed xor-shuffle
//         tree -- no atomics, so two runs are bitwise equal.
// ENERGY: strain[t, i] = mu_t q_mu + lam_t q_lam, kinetic[t, i] = u^T M_t u with the mass table entries rounded as the
//         field assembly rounds them (float32(m_ab) * float32(rho_t)).
constexpr int MF_WARPS = 4;

// u^T Mhat u of one element (the mass form of k_quadforms) with the table entries rounded as the field assembly rounds
// them, float32(m_ab) * float32(rho), when SCALED
template <int NPE, bool SCALED>
__device__ __forceinline__ double elem_mass_form(const float* s_m32, float rho, const double (&u)[NPE][3]) {
    double ms = 0.0;
#pragma unroll
    for (int a = 0; a < NPE; ++a) {
        double ta[3] = {0.0, 0.0, 0.0};
#pragma unroll
        for (int b = a + 1; b < NPE; ++b) {
            const double mab = SCALED ? (double)__fmul_rn(s_m32[a * NPE + b], rho) : (double)s_m32[a * NPE + b];
            ta[0] = fma(mab, u[b][0], ta[0]);
            ta[1] = fma(mab, u[b][1], ta[1]);
            ta[2] = fma(mab, u[b][2], ta[2]);
        }
        const double maa = SCALED ? (double)__fmul_rn(s_m32[a * NPE + a], rho) : (double)s_m32[a * NPE + a];
#pragma unroll
        for (int c = 0; c < 3; ++c) ms = fma(u[a][c], fma(maa, u[a][c], 2.0 * ta[c]), ms);
    }
    return ms;
}

// displacement gradient F[r][j] = du_r / dx_j of a quadratic tet at corner m (F is linear in the barycentric coordinates)
__device__ __forceinline__ void p2_corner_grad(const double (&u)[10][3], const TetGeom& geo, int m, double (&F)[3][3]) {
    constexpr int CORNER[4] = {0, 2, 4, 9};
    constexpr int EDGE[4][4] = {{-1, 1, 5, 6}, {1, -1, 3, 7}, {5, 3, -1, 8}, {6, 7, 8, -1}};
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int j = 0; j < 3; ++j) F[r][j] = 0.0;
#pragma unroll
    for (int l = 0; l < 4; ++l) {
        double h[3];
#pragma unroll
        for (int r = 0; r < 3; ++r)
            h[r] = (l == m) ? 3.0 * u[CORNER[l]][r] : 4.0 * u[EDGE[l][m] < 0 ? 0 : EDGE[l][m]][r] - u[CORNER[l]][r];
#pragma unroll
        for (int r = 0; r < 3; ++r)
#pragma unroll
            for (int j = 0; j < 3; ++j) F[r][j] = fma(h[r], geo.G[l][j], F[r][j]);
    }
}

template <int ORDER, bool ENERGY>
__global__ void __launch_bounds__(MF_WARPS * 32)
k_material_field(const float* __restrict__ verts, const int32_t* __restrict__ tets, int64_t T, const float* __restrict__ m32,
                 double wsum, const double* __restrict__ U, int64_t ldu, int k, const double* __restrict__ lamv,
                 const double* __restrict__ gv, const double* __restrict__ mu_t, const double* __restrict__ lam_t,
                 const float* __restrict__ rho_t, double* __restrict__ out, double* __restrict__ out2) {
    constexpr int NPE = ORDER == 1 ? 4 : 10;
    __shared__ float s_m32[NPE * NPE];
    for (int t = threadIdx.x; t < NPE * NPE; t += blockDim.x) s_m32[t] = m32[t];
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t wstride = (int64_t)gridDim.x * MF_WARPS;
    const int kpad = (k + 31) & ~31;
    for (int64_t e = (int64_t)blockIdx.x * MF_WARPS + warp; e < T; e += wstride) {
        const int32_t* tp = tets + e * NPE;
        int32_t cn[4];
        load_corners(tp, ORDER, cn);
        TetGeom geo;
        tet_geometry<false>(verts, cn, geo);
        const float rho = ENERGY ? __ldg(rho_t + e) : 1.0f;
        double a_mu = 0.0, a_la = 0.0, a_m = 0.0;
        for (int i0 = 0; i0 < kpad; i0 += 32) {
            const int i = i0 + lane;
            const bool on = i < k;
            double u[NPE][3];
#pragma unroll
            for (int a = 0; a < NPE; ++a) {
                const int64_t node = __ldg(tp + a);
#pragma unroll
                for (int c = 0; c < 3; ++c) u[a][c] = on ? __ldg(U + (3 * node + c) * ldu + i) : 0.0;
            }
            // mass form, as k_quadforms
            const double q_m = geo.detM * elem_mass_form<NPE, ENERGY>(s_m32, rho, u);
            double q_mu, q_la;
            if constexpr (ORDER == 1) {
                double F[3][3];
#pragma unroll
                for (int r = 0; r < 3; ++r)
#pragma unroll
                    for (int j = 0; j < 3; ++j)
                        F[r][j] = u[0][r] * geo.G[0][j] + u[1][r] * geo.G[1][j] + u[2][r] * geo.G[2][j] +
                                  u[3][r] * geo.G[3][j];
                double pm, pl;
                phi_pair(F, pm, pl);
                q_mu = geo.detK * wsum * pm;
                q_la = geo.detK * wsum * pl;
            } else {
                double S[3][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}};
                double smu = 0.0, sla = 0.0;
#pragma unroll
                for (int m = 0; m < 4; ++m) {
                    double F[3][3];
                    p2_corner_grad(u, geo, m, F);
                    double pm, pl;
                    phi_pair(F, pm, pl);
                    smu += pm;
                    sla += pl;
#pragma unroll
                    for (int r = 0; r < 3; ++r)
#pragma unroll
                        for (int j = 0; j < 3; ++j) S[r][j] += F[r][j];
                }
                double pm, pl;
                phi_pair(S, pm, pl);
                const double w = geo.detK * (1.0 / 120.0);
                q_mu = w * (smu + pm);
                q_la = w * (sla + pl);
            }
            if (ENERGY) {
                if (on) {
                    __stcs(out + e * k + i, fma(__ldg(mu_t + e), q_mu, __ldg(lam_t + e) * q_la));
                    __stcs(out2 + e * k + i, q_m);
                }
            } else if (on) {
                const double g = __ldg(gv + i);
                a_mu = fma(g, q_mu, a_mu);
                a_la = fma(g, q_la, a_la);
                a_m = fma(-g * __ldg(lamv + i), q_m, a_m);
            }
        }
        if (!ENERGY) {
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) {
                a_mu += __shfl_xor_sync(0xffffffffu, a_mu, off);
                a_la += __shfl_xor_sync(0xffffffffu, a_la, off);
                a_m += __shfl_xor_sync(0xffffffffu, a_m, off);
            }
            if (lane == 0) {
                out[3 * e + 0] = a_mu;
                out[3 * e + 1] = a_la;
                out[3 * e + 2] = a_m;
            }
        }
    }
}

// ---------------------------------------------------------------------------
// elasticity-tensor gradient and element energies
// ---------------------------------------------------------------------------
// The sibling of k_material_field for tensor fields: one warp per tet, lane = mode (chunks of 32 modes).  Per (tet, mode)
// the strain Gram E = int_t eps_V eps_V^T dV (21 packed entries): |det A| wsum phi(F) for linear tets, the vertex rule
// |det A| / 120 (phi(sum_m F_m) + sum_m phi(F_m)) for quadratic ones, phi(F) = eps_V(F) eps_V(F)^T.
// GRAD:   outC[t] = sum_i g_i E_t,i (21 entries), out2[t] = -sum_i g_i lam_i q_m, summed over the lanes by a fixed
//         xor-shuffle tree -- no atomics, bitwise reproducible.
// ENERGY: outC[t, i] = <C_t, E_t,i> (strain), out2[t, i] = u^T M_t u (kinetic, mass entries float32(m_ab) * float32(rho_t)).

// e += phi(F): the packed upper triangle of eps_V eps_V^T, eps_V = (F00, F11, F22, F12 + F21, F02 + F20, F01 + F10)
__device__ __forceinline__ void add_strain_gram(const double (&F)[3][3], double (&e)[21]) {
    const double v[6] = {F[0][0], F[1][1], F[2][2], F[1][2] + F[2][1], F[0][2] + F[2][0], F[0][1] + F[1][0]};
#pragma unroll
    for (int I = 0; I < 6; ++I)
#pragma unroll
        for (int J = I; J < 6; ++J) e[voigt_packed(I, J)] = fma(v[I], v[J], e[voigt_packed(I, J)]);
}

template <int ORDER, bool ENERGY>
__global__ void __launch_bounds__(MF_WARPS * 32)
k_elasticity_field(const float* __restrict__ verts, const int32_t* __restrict__ tets, int64_t T, const float* __restrict__ m32,
                   double wsum, const double* __restrict__ U, int64_t ldu, int k, const double* __restrict__ lamv,
                   const double* __restrict__ gv, const double* __restrict__ C21, const float* __restrict__ rho_t,
                   double* __restrict__ outC, double* __restrict__ out2) {
    constexpr int NPE = ORDER == 1 ? 4 : 10;
    __shared__ float s_m32[NPE * NPE];
    for (int t = threadIdx.x; t < NPE * NPE; t += blockDim.x) s_m32[t] = m32[t];
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t wstride = (int64_t)gridDim.x * MF_WARPS;
    const int kpad = (k + 31) & ~31;
    for (int64_t e = (int64_t)blockIdx.x * MF_WARPS + warp; e < T; e += wstride) {
        const int32_t* tp = tets + e * NPE;
        int32_t cn[4];
        load_corners(tp, ORDER, cn);
        TetGeom geo;
        tet_geometry<false>(verts, cn, geo);
        const float rho = ENERGY ? __ldg(rho_t + e) : 1.0f;
        double Cw[21];          // ENERGY: C_t with the off-diagonal entries doubled, so that <C, E> = sum_p Cw[p] E[p]
        if (ENERGY) {
#pragma unroll
            for (int I = 0; I < 6; ++I)
#pragma unroll
                for (int J = I; J < 6; ++J) {
                    const int p = voigt_packed(I, J);
                    Cw[p] = (I == J ? 1.0 : 2.0) * __ldg(C21 + e * 21 + p);
                }
        }
        double acc[21], a_m = 0.0;
#pragma unroll
        for (int p = 0; p < 21; ++p) acc[p] = 0.0;
        for (int i0 = 0; i0 < kpad; i0 += 32) {
            const int i = i0 + lane;
            const bool on = i < k;
            double u[NPE][3];
#pragma unroll
            for (int a = 0; a < NPE; ++a) {
                const int64_t node = __ldg(tp + a);
#pragma unroll
                for (int c = 0; c < 3; ++c) u[a][c] = on ? __ldg(U + (3 * node + c) * ldu + i) : 0.0;
            }
            const double q_m = geo.detM * elem_mass_form<NPE, ENERGY>(s_m32, rho, u);
            double E[21];
#pragma unroll
            for (int p = 0; p < 21; ++p) E[p] = 0.0;
            double w;
            if constexpr (ORDER == 1) {
                double F[3][3];
#pragma unroll
                for (int r = 0; r < 3; ++r)
#pragma unroll
                    for (int j = 0; j < 3; ++j)
                        F[r][j] = u[0][r] * geo.G[0][j] + u[1][r] * geo.G[1][j] + u[2][r] * geo.G[2][j] +
                                  u[3][r] * geo.G[3][j];
                add_strain_gram(F, E);
                w = geo.detK * wsum;
            } else {
                double S[3][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}};
#pragma unroll
                for (int m = 0; m < 4; ++m) {
                    double F[3][3];
                    p2_corner_grad(u, geo, m, F);
                    add_strain_gram(F, E);
#pragma unroll
                    for (int r = 0; r < 3; ++r)
#pragma unroll
                        for (int j = 0; j < 3; ++j) S[r][j] += F[r][j];
                }
                add_strain_gram(S, E);
                w = geo.detK * (1.0 / 120.0);
            }
            if (ENERGY) {
                if (on) {
                    double en = 0.0;
#pragma unroll
                    for (int p = 0; p < 21; ++p) en = fma(Cw[p], E[p], en);
                    __stcs(outC + e * k + i, w * en);
                    __stcs(out2 + e * k + i, q_m);
                }
            } else if (on) {
                const double gw = __ldg(gv + i) * w;
#pragma unroll
                for (int p = 0; p < 21; ++p) acc[p] = fma(gw, E[p], acc[p]);
                a_m = fma(-__ldg(gv + i) * __ldg(lamv + i), q_m, a_m);
            }
        }
        if (!ENERGY) {
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) {
#pragma unroll
                for (int p = 0; p < 21; ++p) acc[p] += __shfl_xor_sync(0xffffffffu, acc[p], off);
                a_m += __shfl_xor_sync(0xffffffffu, a_m, off);
            }
            if (lane == 0) {
#pragma unroll
                for (int p = 0; p < 21; ++p) outC[21 * e + p] = acc[p];
                out2[e] = a_m;
            }
        }
    }
}

static int qf_ctas(int64_t T) {
    int64_t c = ceil_div(T, QF_WARPS * 8);
    if (c < 1) c = 1;
    return (int)(c < QF_MAX_CTAS ? c : QF_MAX_CTAS);
}

}  // namespace ds

using namespace ds;

extern "C" int ds_corner_incidence(ds_workspace* ws, const int32_t* tets, int64_t T, int npe, int order,
                                   int64_t n_nodes, int32_t* inc_ptr, int32_t* inc, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    DS_REQUIRE(ws && tets && inc_ptr && inc, "ds_corner_incidence: null argument");
    DS_REQUIRE((order == 1 && npe == 4) || (order == 2 && npe == 10), "ds_corner_incidence: order/npe mismatch");
    DS_REQUIRE(T > 0 && n_nodes > 0 && 4 * T < (int64_t)2147483647, "ds_corner_incidence: bad sizes");
    int64_t nq = 4 * T;
    ProfScope prof(PROF_PATTERN, stream);
    int end_bit = 1;
    while (end_bit < 32 && ((int64_t)1 << end_bit) < n_nodes) ++end_bit;
    size_t tmp = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, tmp, (uint32_t*)nullptr, (uint32_t*)nullptr, (uint32_t*)nullptr,
                                    (uint32_t*)nullptr, (int)nq, 0, end_bit, stream);
    DS_TRY(ws->arena.reserve((size_t)nq * 12 + tmp + 8 * 256, stream));
    uint32_t* keys_in = ws->arena.take<uint32_t>(nq);
    uint32_t* keys_out = ws->arena.take<uint32_t>(nq);
    uint32_t* vals_in = ws->arena.take<uint32_t>(nq);
    void* cub_tmp = ws->arena.take<char>(tmp);
    DS_REQUIRE(cub_tmp != nullptr, "ds_corner_incidence: arena too small");
    unsigned blocks = (unsigned)ceil_div(nq, 256);
    k_corner_keys<<<blocks, 256, 0, stream>>>(tets, T, npe, order, keys_in, vals_in);
    DS_LAUNCH_CHECK();
    DS_CUDA(cub::DeviceRadixSort::SortPairs(cub_tmp, tmp, keys_in, keys_out, vals_in, (uint32_t*)inc, (int)nq, 0,
                                            end_bit, stream));
    k_inc_ptr<<<blocks, 256, 0, stream>>>(keys_out, nq, n_nodes, inc_ptr);
    DS_LAUNCH_CHECK();
    return DS_OK;
}

template <int MODE>
static int grad_shape(const float* verts, const int32_t* tets, int64_t T, int order, int64_t n_nodes, double mu,
                      double lam_lame, const GradField& f, const double* ctab, const double* mtab, const double* U,
                      int64_t ldu, int k, const double* lam, const double* g, const int32_t* inc_ptr, const int32_t* inc,
                      double* tet_grad, float* grad_verts, cudaStream_t stream) {
    const int kpad = (k + 15) & ~15;
    ProfScope prof(PROF_GRAD, stream);
    {   // SURVEY 8d: n k 8 (U once) + T npe 4 + nodes 12 + nodes 24; flops: per tet and mode the quadratic forms of the 4 corner
        // derivatives, ~ 2 (3 npe)^2 x 12 / 4 (counted from the kernel's DMMA tiles in DESIGN.md)
        const int npe_ = order == 1 ? 4 : 10;
        prof_account(PROF_GRAD, (double)n_nodes * 3.0 * k * 8.0 + (double)T * npe_ * 4.0 + (double)n_nodes * 36.0 +
                     (MODE == MAT_LAME ? (double)T * 20.0 : MODE == MAT_TENSOR ? (double)T * (21.0 * 8.0 + 4.0) : 0.0), 0.0);
    }
    int64_t ctas64 = ceil_div(T, GS_WARPS);
    int ctas = (int)(ctas64 < 148 * 8 ? ctas64 : 148 * 8);
    if (order == 1) {
        size_t smem = sizeof(GradSmemOf<1, MODE>) + 2 * kpad * sizeof(double);
        DS_CUDA(cudaFuncSetAttribute(k_eigval_grad_shape<1, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k_eigval_grad_shape<1, MODE><<<ctas, GS_WARPS * 32, smem, stream>>>(verts, tets, T, mu, lam_lame, f, ctab, mtab, U, ldu,
                                                                             k, lam, g, tet_grad);
    } else {
        size_t smem = sizeof(GradSmemOf<2, MODE>) + 2 * kpad * sizeof(double);
        DS_CUDA(cudaFuncSetAttribute(k_eigval_grad_shape<2, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k_eigval_grad_shape<2, MODE><<<ctas, GS_WARPS * 32, smem, stream>>>(verts, tets, T, mu, lam_lame, f, ctab, mtab, U, ldu,
                                                                             k, lam, g, tet_grad);
    }
    DS_LAUNCH_CHECK();
    k_node_gather<<<(unsigned)ceil_div(3 * n_nodes, 256), 256, 0, stream>>>(inc_ptr, inc, tet_grad, n_nodes, grad_verts);
    DS_LAUNCH_CHECK();
    return DS_OK;
}

extern "C" int ds_eigval_grad_shape(const float* verts, const int32_t* tets, int64_t T, int order, int64_t n_nodes,
                                    double mu, double lam_lame, const double* ctab, const double* mtab,
                                    const double* U, int64_t ldu, int k, const double* lam, const double* g,
                                    const int32_t* inc_ptr, const int32_t* inc, double* tet_grad,
                                    float* grad_verts, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    DS_REQUIRE(order == 1 || order == 2, "ds_eigval_grad_shape: order must be 1 or 2 (got %d)", order);
    DS_REQUIRE(verts && tets && ctab && mtab && U && lam && g && inc_ptr && inc && tet_grad && grad_verts,
               "ds_eigval_grad_shape: null argument");
    DS_REQUIRE(T > 0 && n_nodes > 0 && k > 0 && k <= 1024 && ldu >= k, "ds_eigval_grad_shape: bad sizes");
    return grad_shape<MAT_SCALAR>(verts, tets, T, order, n_nodes, mu, lam_lame, GradField{}, ctab, mtab, U, ldu, k, lam, g, inc_ptr,
                             inc, tet_grad, grad_verts, (cudaStream_t)stream_);
}

extern "C" int ds_eigval_grad_shape_field(const float* verts, const int32_t* tets, int64_t T, int order, int64_t n_nodes,
                                          const double* mu_t, const double* lam_t, const float* rho_t, const double* ctab,
                                          const double* mtab1, const double* U, int64_t ldu, int k, const double* lam,
                                          const double* g, const int32_t* inc_ptr, const int32_t* inc, double* tet_grad,
                                          float* grad_verts, void* stream_) {
    DS_REQUIRE(order == 1 || order == 2, "ds_eigval_grad_shape_field: order must be 1 or 2 (got %d)", order);
    DS_REQUIRE(verts && tets && mu_t && lam_t && rho_t && ctab && mtab1 && U && lam && g && inc_ptr && inc && tet_grad &&
               grad_verts, "ds_eigval_grad_shape_field: null argument");
    DS_REQUIRE(T > 0 && n_nodes > 0 && k > 0 && k <= 1024 && ldu >= k, "ds_eigval_grad_shape_field: bad sizes");
    return grad_shape<MAT_LAME>(verts, tets, T, order, n_nodes, 0.0, 0.0, GradField{mu_t, lam_t, rho_t, nullptr}, ctab, mtab1, U, ldu, k, lam,
                            g, inc_ptr, inc, tet_grad, grad_verts, (cudaStream_t)stream_);
}

template <bool ENERGY>
static int material_field(const float* verts, const int32_t* tets, int64_t T, int order, const float* m32,
                          double wsum, const double* U, int64_t ldu, int k, const double* lam, const double* g,
                          const double* mu_t, const double* lam_t, const float* rho_t, double* out, double* out2,
                          cudaStream_t stream) {
    ProfScope prof(PROF_MATERIAL_FIELD, stream);
    {   // U rows of every tet (re-read per tet: L2), geometry, per-tet material / outputs
        const int npe = order == 1 ? 4 : 10;
        prof_account(PROF_MATERIAL_FIELD, (double)T * (npe * 3.0 * k * 8.0 + npe * 4.0 + 48.0) +
                     (ENERGY ? (double)T * (20.0 + 16.0 * k) : (double)T * 24.0), 0.0);
    }
    const int64_t ctas64 = ceil_div(T, MF_WARPS);
    const unsigned ctas = (unsigned)(ctas64 < 148 * 16 ? ctas64 : 148 * 16);
    if (order == 1)
        k_material_field<1, ENERGY><<<ctas, MF_WARPS * 32, 0, stream>>>(verts, tets, T, m32, wsum, U, ldu, k, lam, g, mu_t, lam_t,
                                                                        rho_t, out, out2);
    else
        k_material_field<2, ENERGY><<<ctas, MF_WARPS * 32, 0, stream>>>(verts, tets, T, m32, wsum, U, ldu, k, lam, g, mu_t, lam_t,
                                                                        rho_t, out, out2);
    DS_LAUNCH_CHECK();
    return DS_OK;
}

extern "C" int ds_material_field_grad(const float* verts, const int32_t* tets, int64_t T, int order, const float* m32,
                                      double wsum, const double* U, int64_t ldu, int k, const double* lam, const double* g,
                                      double* out, void* stream_) {
    DS_REQUIRE(order == 1 || order == 2, "ds_material_field_grad: order must be 1 or 2 (got %d)", order);
    DS_REQUIRE(verts && tets && m32 && U && lam && g && out, "ds_material_field_grad: null argument");
    DS_REQUIRE(T > 0 && k > 0 && ldu >= k, "ds_material_field_grad: bad sizes");
    return material_field<false>(verts, tets, T, order, m32, wsum, U, ldu, k, lam, g, nullptr,
                                 nullptr, nullptr, out, nullptr, (cudaStream_t)stream_);
}

extern "C" int ds_element_energies(const float* verts, const int32_t* tets, int64_t T, int order, const float* m32,
                                   double wsum, const double* U, int64_t ldu, int k, const double* mu_t, const double* lam_t,
                                   const float* rho_t, double* strain, double* kinetic, void* stream_) {
    DS_REQUIRE(order == 1 || order == 2, "ds_element_energies: order must be 1 or 2 (got %d)", order);
    DS_REQUIRE(verts && tets && m32 && U && mu_t && lam_t && rho_t && strain && kinetic, "ds_element_energies: null argument");
    DS_REQUIRE(T > 0 && k > 0 && ldu >= k, "ds_element_energies: bad sizes");
    return material_field<true>(verts, tets, T, order, m32, wsum, U, ldu, k, nullptr, nullptr, mu_t,
                                lam_t, rho_t, strain, kinetic, (cudaStream_t)stream_);
}

template <bool ENERGY>
static int elasticity_field(const float* verts, const int32_t* tets, int64_t T, int order, const float* m32, double wsum,
                            const double* U, int64_t ldu, int k, const double* lam, const double* g, const double* C21,
                            const float* rho_t, double* outC, double* out2, cudaStream_t stream) {
    ProfScope prof(PROF_MATERIAL_FIELD, stream);
    {   // U rows of every tet (re-read per tet: L2), geometry, per-tet tensor / outputs
        const int npe = order == 1 ? 4 : 10;
        prof_account(PROF_MATERIAL_FIELD, (double)T * (npe * 3.0 * k * 8.0 + npe * 4.0 + 48.0) +
                     (ENERGY ? (double)T * (21.0 * 8.0 + 4.0 + 16.0 * k) : (double)T * 22.0 * 8.0), 0.0);
    }
    const int64_t ctas64 = ceil_div(T, MF_WARPS);
    const unsigned ctas = (unsigned)(ctas64 < 148 * 16 ? ctas64 : 148 * 16);
    if (order == 1)
        k_elasticity_field<1, ENERGY><<<ctas, MF_WARPS * 32, 0, stream>>>(verts, tets, T, m32, wsum, U, ldu, k, lam, g, C21,
                                                                          rho_t, outC, out2);
    else
        k_elasticity_field<2, ENERGY><<<ctas, MF_WARPS * 32, 0, stream>>>(verts, tets, T, m32, wsum, U, ldu, k, lam, g, C21,
                                                                          rho_t, outC, out2);
    DS_LAUNCH_CHECK();
    return DS_OK;
}

extern "C" int ds_eigval_grad_shape_tensor(const float* verts, const int32_t* tets, int64_t T, int order, int64_t n_nodes,
                                           const double* C21, const float* rho_t, const double* ctab, const double* mtab1,
                                           const double* U, int64_t ldu, int k, const double* lam, const double* g,
                                           const int32_t* inc_ptr, const int32_t* inc, double* tet_grad, float* grad_verts,
                                           void* stream_) {
    DS_REQUIRE(order == 1 || order == 2, "ds_eigval_grad_shape_tensor: order must be 1 or 2 (got %d)", order);
    DS_REQUIRE(verts && tets && C21 && rho_t && ctab && mtab1 && U && lam && g && inc_ptr && inc && tet_grad && grad_verts,
               "ds_eigval_grad_shape_tensor: null argument");
    DS_REQUIRE(T > 0 && n_nodes > 0 && k > 0 && k <= 1024 && ldu >= k, "ds_eigval_grad_shape_tensor: bad sizes");
    return grad_shape<MAT_TENSOR>(verts, tets, T, order, n_nodes, 0.0, 0.0, GradField{nullptr, nullptr, rho_t, C21}, ctab, mtab1,
                                  U, ldu, k, lam, g, inc_ptr, inc, tet_grad, grad_verts, (cudaStream_t)stream_);
}

extern "C" int ds_elasticity_field_grad(const float* verts, const int32_t* tets, int64_t T, int order, const float* m32,
                                        double wsum, const double* U, int64_t ldu, int k, const double* lam, const double* g,
                                        double* outC, double* out_rho, void* stream_) {
    DS_REQUIRE(order == 1 || order == 2, "ds_elasticity_field_grad: order must be 1 or 2 (got %d)", order);
    DS_REQUIRE(verts && tets && m32 && U && lam && g && outC && out_rho, "ds_elasticity_field_grad: null argument");
    DS_REQUIRE(T > 0 && k > 0 && ldu >= k, "ds_elasticity_field_grad: bad sizes");
    return elasticity_field<false>(verts, tets, T, order, m32, wsum, U, ldu, k, lam, g, nullptr, nullptr, outC, out_rho,
                                   (cudaStream_t)stream_);
}

extern "C" int ds_element_energies_tensor(const float* verts, const int32_t* tets, int64_t T, int order, const float* m32,
                                          double wsum, const double* U, int64_t ldu, int k, const double* C21,
                                          const float* rho_t, double* strain, double* kinetic, void* stream_) {
    DS_REQUIRE(order == 1 || order == 2, "ds_element_energies_tensor: order must be 1 or 2 (got %d)", order);
    DS_REQUIRE(verts && tets && m32 && U && C21 && rho_t && strain && kinetic, "ds_element_energies_tensor: null argument");
    DS_REQUIRE(T > 0 && k > 0 && ldu >= k, "ds_element_energies_tensor: bad sizes");
    return elasticity_field<true>(verts, tets, T, order, m32, wsum, U, ldu, k, nullptr, nullptr, C21, rho_t, strain, kinetic,
                                  (cudaStream_t)stream_);
}

extern "C" int64_t ds_quadform_scratch_elems(int k) { return (int64_t)QF_MAX_CTAS * QF_WARPS * 3 * k; }

extern "C" int ds_eigval_quadforms_material(const float* verts, const int32_t* tets, int64_t T, int order,
                                            const double* mtab, double wsum, const double* U, int64_t ldu, int k,
                                            double* partial, double* out, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    DS_REQUIRE(order == 1 || order == 2, "ds_eigval_quadforms_material: order must be 1 or 2 (got %d)", order);
    DS_REQUIRE(verts && tets && mtab && U && partial && out, "ds_eigval_quadforms_material: null argument");
    DS_REQUIRE(T > 0 && k > 0 && ldu >= k, "ds_eigval_quadforms_material: bad sizes");
    int ctas = qf_ctas(T);
    ProfScope prof(PROF_QUADFORM, stream);
    if (order == 1)
        k_quadforms<1><<<ctas, QF_WARPS * 32, 0, stream>>>(verts, tets, T, mtab, wsum, U, ldu, k, partial);
    else
        k_quadforms<2><<<ctas, QF_WARPS * 32, 0, stream>>>(verts, tets, T, mtab, wsum, U, ldu, k, partial);
    DS_LAUNCH_CHECK();
    k_quadform_reduce<<<(3 * k + 127) / 128, 128, 0, stream>>>(partial, ctas * QF_WARPS, 3 * k, out);
    DS_LAUNCH_CHECK();
    return DS_OK;
}

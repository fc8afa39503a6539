// Fused stiffness + mass assembly into the fixed block-CSR pattern.
//
// Reference behaviour replaced (file:line under /root/reference/src):
//   diffelastic/diff_model.py:184-220  update_stiff_matrix  (batched A^T B A + COO coalesce)
//   diffelastic/diff_model.py:222-312  update_mass_matrix   (900 strided writes + coalesce)
//   diffelastic/deform.py:35-68,136-147  grad_x N and w_g |det A| tables (T*G*npe*3 fp32)
//   cuda/massMatrixDouble.cu:3-78       compute_mass_matrix_kernel (1 thread / tet, COO)
//
// Design: geometry is affine per tet (mesh.py:69-99 uses the corner nodes only), so
//   grad_x N_a(g) = sum_l dN_a/dL_l(g) G_l,   G = dL/dxi A^-1   (4x3 per tet)
// and the Gauss sum collapses into a constant table
//   ctab[a][b][l][m] = sum_g w_g dN_a/dL_l(g) dN_b/dL_m(g)
// built on the host from the reference's own fp32 rule.  Then per element block
//   S_ab = sum_{l,m} ctab[a][b][l][m] G_l G_m^T
//   K_ab[c][d] = |det A| ( mu (delta_cd tr S_ab + S_ab[d][c]) + lam S_ab[c][d] )
//   M_ab = mtab[a][b] |det6V| I3.
// Owner-computes: the warp that owns node row i sums all element contributions of its blocks
// (i, bcol[brow[i]+p]) in ascending element order, the work split evenly over its lanes (k_assemble_rows).
// Material fields (MODE = MAT_LAME): mu, lam and the mass table entry come from tet e's own (mu_e, lam_e, rho_e) with the
// scalar kernels' operation order, so a constant field reproduces the homogeneous K and M bit for bit.
// Elasticity-tensor fields (MODE = MAT_TENSOR): tet e's own 6x6 Voigt matrix C_e (order 11, 22, 33, 23, 13, 12, engineering
// shear strains, sigma_V = C eps_V) in the global frame, packed as its 21-entry upper triangle row by row, and
//   K_ab[c][d] = |det A| sum_{k,l} C_{ckdl} S_ab[k][l]      (C_{ckdl}: the rank-4 form of C_e).
// An isotropic C = lam 11^T + mu diag(2, 2, 2, 1, 1, 1) gives the Lame expression above (in another summation order).
#include "common.cuh"
#include "../../include/diffsound_sm100.h"
#include <algorithm>

namespace ds {

constexpr int GEOM_STRIDE = 14;  // G[4][3], detK, detM

__device__ __constant__ int c_sup2[10][2] = {{0, 0}, {0, 1}, {1, 1}, {1, 2}, {2, 2},
                                             {2, 0}, {0, 3}, {1, 3}, {2, 3}, {3, 3}};
__device__ __constant__ int c_nsup2[10] = {1, 2, 1, 2, 1, 2, 2, 2, 2, 1};

__device__ __forceinline__ void corner_ids(const int32_t* t, int order, int32_t c[4]) {
    if (order == 1) {
        c[0] = t[0]; c[1] = t[1]; c[2] = t[2]; c[3] = t[3];
    } else {
        c[0] = t[0]; c[1] = t[2]; c[2] = t[4]; c[3] = t[9];
    }
}

// One thread per tet.  A is built from fp32 differences exactly as mesh.py:90-98;
// inverse and determinant are then taken in fp64 (more accurate than the
// reference's fp32 torch.inverse / torch.det; SURVEY.md section 7 item 2).
__global__ void k_tet_geometry(const float* __restrict__ verts, const int32_t* __restrict__ tets, int64_t T,
                               int npe, int order, double* __restrict__ geom) {
    int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (e >= T) return;
    int32_t c[4];
    corner_ids(tets + e * npe, order, c);
    float v[4][3];
#pragma unroll
    for (int p = 0; p < 4; ++p) {
        v[p][0] = verts[3 * (int64_t)c[p] + 0];
        v[p][1] = verts[3 * (int64_t)c[p] + 1];
        v[p][2] = verts[3 * (int64_t)c[p] + 2];
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
    double Ai[3][3];
    Ai[0][0] = c00 * id;
    Ai[0][1] = (A[0][2] * A[2][1] - A[0][1] * A[2][2]) * id;
    Ai[0][2] = (A[0][1] * A[1][2] - A[0][2] * A[1][1]) * id;
    Ai[1][0] = c01 * id;
    Ai[1][1] = (A[0][0] * A[2][2] - A[0][2] * A[2][0]) * id;
    Ai[1][2] = (A[0][2] * A[1][0] - A[0][0] * A[1][2]) * id;
    Ai[2][0] = c02 * id;
    Ai[2][1] = (A[0][1] * A[2][0] - A[0][0] * A[2][1]) * id;
    Ai[2][2] = (A[0][0] * A[1][1] - A[0][1] * A[1][0]) * id;
    double* g = geom + e * GEOM_STRIDE;
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        g[0 + d] = Ai[0][d];
        g[3 + d] = Ai[1][d];
        g[6 + d] = Ai[2][d];
        g[9 + d] = -(Ai[0][d] + Ai[1][d] + Ai[2][d]);
    }
    g[12] = fabs(det);
    // |6V| from fp64 corner coordinates, same expansion as diff_model.py:272-289
    // (no FMA contraction so that it rounds like the CPU reference).
    double x[4], y[4], z[4];
#pragma unroll
    for (int p = 0; p < 4; ++p) {
        x[p] = (double)v[p][0];
        y[p] = (double)v[p][1];
        z[p] = (double)v[p][2];
    }
    double x10 = __dsub_rn(x[1], x[0]), y10 = __dsub_rn(y[1], y[0]), z10 = __dsub_rn(z[1], z[0]);
    double x20 = __dsub_rn(x[2], x[0]), y20 = __dsub_rn(y[2], y[0]), z20 = __dsub_rn(z[2], z[0]);
    double x30 = __dsub_rn(x[3], x[0]), y30 = __dsub_rn(y[3], y[0]), z30 = __dsub_rn(z[3], z[0]);
    double t1 = __dmul_rn(x10, __dsub_rn(__dmul_rn(y20, z30), __dmul_rn(y30, z20)));
    double t2 = __dmul_rn(y10, __dsub_rn(__dmul_rn(z20, x30), __dmul_rn(z30, x20)));
    double t3 = __dmul_rn(z10, __dsub_rn(__dmul_rn(x20, y30), __dmul_rn(x30, y20)));
    g[13] = fabs(__dadd_rn(__dadd_rn(t1, t2), t3));
}

// Per-tet material of the field variants (ds_assemble_km_field, ds_assemble_km_tensor): Lame parameters (fp64) or the
// packed elasticity tensor (fp64 [T][21]), the density (fp32) of tet e, and the fp32 unit-density mass table.  The scalar
// kernels are the MAT_SCALAR instantiations and never read it.
struct FieldArgs {
    const double* __restrict__ mu;
    const double* __restrict__ lam;
    const float* __restrict__ rho;
    const float* __restrict__ m32;
    const double* __restrict__ C;
};

// mass table entry of one element: s_mtab holds double(float32(m_ab) * float32(rho)) for one material, double(m_ab) for a
// field, whose entry is then rounded exactly as mass_density_table rounds the scalar density: a constant field gives
// the homogeneous M bit for bit
template <bool FIELD>
__device__ __forceinline__ double mass_entry(double tab, float rho_e) {
    return FIELD ? (double)__fmul_rn((float)tab, rho_e) : tab;
}

template <bool FIELD>
__device__ __forceinline__ void stage_mtab(double* s_mtab, const double* __restrict__ mtab_g, const FieldArgs& f, int n) {
    for (int t = threadIdx.x; t < n; t += blockDim.x) s_mtab[t] = FIELD ? (double)f.m32[t] : mtab_g[t];
}

// one element contribution (tet e, local nodes a, b) added to a 3x3 accumulator and the mass scalar
template <int ORDER, int MODE>
__device__ __forceinline__ void add_contribution(int pair, const double* __restrict__ geom, const double* s_ctab,
                                                 const double* s_mtab, double mu_s, double lam_s, const FieldArgs& f,
                                                 double (&acc)[3][3], double& macc) {
    constexpr int NPE = ORDER == 1 ? 4 : 10;
    constexpr int NPE2 = NPE * NPE;
    constexpr bool FIELD = MODE != MAT_SCALAR;
    const int e = pair / NPE2;
    const int ab = pair - e * NPE2;
    const double mu = MODE == MAT_LAME ? __ldg(f.mu + e) : mu_s;
    const double lam = MODE == MAT_LAME ? __ldg(f.lam + e) : lam_s;
    const int a = ab / NPE, b = ab - a * NPE;
    const double* g = geom + (int64_t)e * GEOM_STRIDE;
    double S[3][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}};
    int na, nb, la[2], lb[2];
    if (ORDER == 1) {
        na = nb = 1;
        la[0] = a; lb[0] = b; la[1] = lb[1] = 0;
    } else {
        na = c_nsup2[a]; nb = c_nsup2[b];
        la[0] = c_sup2[a][0]; la[1] = c_sup2[a][1];
        lb[0] = c_sup2[b][0]; lb[1] = c_sup2[b][1];
    }
    const double* ct = s_ctab + ab * 16;
    for (int li = 0; li < na; ++li) {
        const int l = la[li];
        const double gl0 = g[3 * l], gl1 = g[3 * l + 1], gl2 = g[3 * l + 2];
        for (int mi = 0; mi < nb; ++mi) {
            const int m = lb[mi];
            const double c = ct[l * 4 + m];
            const double gm0 = g[3 * m], gm1 = g[3 * m + 1], gm2 = g[3 * m + 2];
            const double a0 = c * gl0, a1 = c * gl1, a2 = c * gl2;
            S[0][0] += a0 * gm0; S[0][1] += a0 * gm1; S[0][2] += a0 * gm2;
            S[1][0] += a1 * gm0; S[1][1] += a1 * gm1; S[1][2] += a1 * gm2;
            S[2][0] += a2 * gm0; S[2][1] += a2 * gm1; S[2][2] += a2 * gm2;
        }
    }
    const double detK = g[12], detM = g[13];
    if constexpr (MODE == MAT_TENSOR) {
        const double* __restrict__ Ce = f.C + (int64_t)e * 21;
        double Cv[21];
#pragma unroll
        for (int t = 0; t < 21; ++t) Cv[t] = __ldg(Ce + t);
#pragma unroll
        for (int c = 0; c < 3; ++c)
#pragma unroll
            for (int d = 0; d < 3; ++d) {
                double v = 0.0;
#pragma unroll
                for (int k = 0; k < 3; ++k)
#pragma unroll
                    for (int l = 0; l < 3; ++l) v = fma(Cv[voigt_packed(voigt(c, k), voigt(d, l))], S[k][l], v);
                acc[c][d] += detK * v;
            }
    } else {
        const double tr = mu * (S[0][0] + S[1][1] + S[2][2]);
#pragma unroll
        for (int c = 0; c < 3; ++c)
#pragma unroll
            for (int d = 0; d < 3; ++d) {
                double v = mu * S[d][c] + lam * S[c][d];
                if (c == d) v += tr;
                acc[c][d] += detK * v;
            }
    }
    macc += mass_entry<FIELD>(s_mtab[ab], FIELD ? __ldg(f.rho + e) : 0.0f) * detM;
}

// Owner-computes with BALANCED lanes.  A warp owns one node row; the element contributions of all its block slots
// form one contiguous, slot-sorted run [Q0, Q1) of the contributor list (1 .. 24+ per slot: the diagonal slot of a
// corner node collects every tet around it, most slots one or two).  The run is cut into 32 equal chunks, one per
// lane; a lane sums its chunk slot by slot in list order.  A slot that lies inside one chunk is written directly;
// a slot that is cut by chunk borders leaves partial sums in shared memory (at most a head and a tail partial per
// lane), which the lane holding the slot's first contribution adds up in lane order -- a fixed order, no atomics.
// (The lane-per-slot version spent 7x the instructions of a balanced warp waiting for the longest slot.)
constexpr int AS_WARPS = 4;

template <int ORDER, int MODE>
__global__ void __launch_bounds__(32 * AS_WARPS)
k_assemble_rows(const double* __restrict__ geom, const double* __restrict__ ctab_g,
                const double* __restrict__ mtab_g, const int32_t* __restrict__ brow,
                const int32_t* __restrict__ contrib_ptr, const int32_t* __restrict__ contrib,
                int64_t n_nodes, double mu, double lam, FieldArgs f, double* __restrict__ Kval, double* __restrict__ Mblk) {
    constexpr int NPE = ORDER == 1 ? 4 : 10;
    constexpr int NPE2 = NPE * NPE;
    __shared__ double s_ctab[NPE2 * 16];
    __shared__ double s_mtab[NPE2];
    __shared__ double s_part[AS_WARPS][32][2][10];     // [lane][head / tail][9 stiffness entries + mass]
    __shared__ int s_head[AS_WARPS][32];               // slot of the lane's head partial, -1: none
    for (int t = threadIdx.x; t < NPE2 * 16; t += blockDim.x) s_ctab[t] = ctab_g[t];
    stage_mtab<MODE != MAT_SCALAR>(s_mtab, mtab_g, f, NPE2);
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double (*part)[2][10] = s_part[warp];
    int* head = s_head[warp];
    for (int64_t row = (int64_t)blockIdx.x * AS_WARPS + warp; row < n_nodes; row += (int64_t)gridDim.x * AS_WARPS) {
        const int b0 = brow[row];
        const int deg = brow[row + 1] - b0;
        const int Q0 = contrib_ptr[b0], Q1 = contrib_ptr[b0 + deg];
        const int chunk = (Q1 - Q0 + 31) >> 5;
        const int qa = min(Q0 + lane * chunk, Q1), qb = min(qa + chunk, Q1);
        double* krow = Kval + 9 * (int64_t)b0;
        const int rs = 3 * deg;
        auto write_slot = [&](int s, const double (&acc)[3][3], double macc) {
            double* out = krow + 3 * (s - b0);
#pragma unroll
            for (int c = 0; c < 3; ++c)
#pragma unroll
                for (int d = 0; d < 3; ++d) out[c * rs + d] = acc[c][d];
            Mblk[s] = macc;
        };
        int head_slot = -1, tail_slot = -1;
        if (qa < qb) {
            // slot of the first contribution: last s in [b0, b0 + deg) with contrib_ptr[s] <= qa
            int lo = b0, hi = b0 + deg - 1;
            while (lo < hi) {
                const int mid = (lo + hi + 1) >> 1;
                if (contrib_ptr[mid] <= qa) lo = mid; else hi = mid - 1;
            }
            int cur = lo;
            int s_begin = contrib_ptr[cur], s_end = contrib_ptr[cur + 1];
            double acc[3][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}};
            double macc = 0.0;
            for (int q = qa; q < qb; ++q) {
                if (q == s_end) {                    // slot `cur` ended inside this chunk
                    if (s_begin >= qa) {
                        write_slot(cur, acc, macc);
                    } else {                         // it began in an earlier lane: head partial
                        head_slot = cur;
#pragma unroll
                        for (int c = 0; c < 3; ++c)
#pragma unroll
                            for (int d = 0; d < 3; ++d) part[lane][0][3 * c + d] = acc[c][d];
                        part[lane][0][9] = macc;
                    }
#pragma unroll
                    for (int c = 0; c < 3; ++c)
#pragma unroll
                        for (int d = 0; d < 3; ++d) acc[c][d] = 0.0;
                    macc = 0.0;
                    ++cur;
                    s_begin = s_end;
                    s_end = contrib_ptr[cur + 1];
                }
                add_contribution<ORDER, MODE>(contrib[q], geom, s_ctab, s_mtab, mu, lam, f, acc, macc);
            }
            // the slot in progress at the end of the chunk
            const bool began_here = s_begin >= qa, ends_here = s_end == qb;
            if (began_here && ends_here) {
                write_slot(cur, acc, macc);
            } else {
                const int side = began_here ? 1 : 0;      // began here and continues: tail partial (this lane owns the slot)
                if (side) tail_slot = cur; else head_slot = cur;
#pragma unroll
                for (int c = 0; c < 3; ++c)
#pragma unroll
                    for (int d = 0; d < 3; ++d) part[lane][side][3 * c + d] = acc[c][d];
                part[lane][side][9] = macc;
            }
        }
        head[lane] = head_slot;
        __syncwarp();
        if (tail_slot >= 0) {                        // owner: own tail + the head partials of the following lanes
            double acc[3][3];
#pragma unroll
            for (int c = 0; c < 3; ++c)
#pragma unroll
                for (int d = 0; d < 3; ++d) acc[c][d] = part[lane][1][3 * c + d];
            double macc = part[lane][1][9];
            for (int l2 = lane + 1; l2 < 32 && head[l2] == tail_slot; ++l2) {
#pragma unroll
                for (int c = 0; c < 3; ++c)
#pragma unroll
                    for (int d = 0; d < 3; ++d) acc[c][d] += part[l2][0][3 * c + d];
                macc += part[l2][0][9];
            }
            write_slot(tail_slot, acc, macc);
        }
        __syncwarp();                                // partials are free for the next row
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Round 2: tet-sequential rows (quadratic tets).  The balanced kernel above pays per CONTRIBUTION: it decodes (tet, a, b),
// fetches ~14 scattered 8-byte geometry values that differ from lane to lane (one L1 wavefront per distinct tet and
// instruction: L1 data pipe 68 %) and scatters 9 doubles per slot.  Here a warp still owns one node row i, but walks the
// tets AROUND node i one after the other (they are the contributors of the row's diagonal slot, ascending).  For tet e
// with i = local node a, lane (b, c) = (lane / 3, lane % 3) produces row c of the 3x3 block (a, b): every geometry load is
// one broadcast address per warp, the block lands at slot[e, a, b] - brow[i] of a shared-memory image of the row
// (11 doubles per slot: 9 stiffness entries + the mass scalar + padding; lanes of one tet hit distinct slots, tets are strictly
// ordered, so the sums are deterministic and need no atomics), and the finished row leaves as three contiguous runs of
// 3 deg doubles (the reference's scalar-CSR value order) + deg mass scalars: fully coalesced streaming stores.
// `slot` is the element -> pattern-slot map ds_pattern_fill already produces (4 B per (tet, a, b)).
// ---------------------------------------------------------------------------------------------------------------
constexpr int AT_WARPS = 8;
constexpr int AT_SLOT = 11;                       // doubles per slot of the row image: 9 + 1 + one of padding (an odd pitch
                                                  // spreads the 64-bit accesses over all bank pairs; 10 gave 5-way conflicts)

template <int MODE>
__global__ void __launch_bounds__(32 * AT_WARPS)
k_assemble_rows_tets2(const double* __restrict__ geom, const double* __restrict__ ctab_g, const double* __restrict__ mtab_g,
                      const int32_t* __restrict__ brow, const int32_t* __restrict__ bcol,
                      const int32_t* __restrict__ contrib_ptr, const int32_t* __restrict__ contrib,
                      const int32_t* __restrict__ slot, int64_t n_nodes, int cap, double mu_s, double lam_s, FieldArgs f,
                      double* __restrict__ Kval, double* __restrict__ Mblk) {
    constexpr int NPE = 10, NPE2 = 100;
    constexpr bool FIELD = MODE != MAT_SCALAR;
    extern __shared__ __align__(16) double s_dyn[];
    double* s_ct4 = s_dyn;                        // [a][b][li][mi]: the <= 2 x 2 support products of ctab, zero where absent
    double* s_mtab = s_ct4 + NPE2 * 4;            // [a][b]
    double* s_acc = s_mtab + NPE2;                // [AT_WARPS][cap][AT_SLOT]
    for (int t = threadIdx.x; t < NPE2 * 4; t += blockDim.x) {
        const int ab = t >> 2, li = (t >> 1) & 1, mi = t & 1;
        const int a = ab / NPE, b = ab - a * NPE;
        const bool ok = li < c_nsup2[a] && mi < c_nsup2[b];
        s_ct4[t] = ok ? ctab_g[ab * 16 + c_sup2[a][li] * 4 + c_sup2[b][mi]] : 0.0;
    }
    stage_mtab<FIELD>(s_mtab, mtab_g, f, NPE2);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double* acc = s_acc + (size_t)warp * cap * AT_SLOT;
    for (int t = lane; t < cap * AT_SLOT; t += 32) acc[t] = 0.0;
    __syncthreads();
    const int b = lane / 3, c = lane - 3 * b;     // lanes 30, 31 idle in the tet loop
    const bool lane_on = lane < 3 * NPE;
    const int bb = lane_on ? b : 0;
    const int mb0 = 3 * c_sup2[bb][0], mb1 = 3 * c_sup2[bb][1];
    for (int64_t row = (int64_t)blockIdx.x * AT_WARPS + warp; row < n_nodes; row += (int64_t)gridDim.x * AT_WARPS) {
        const int b0 = brow[row];
        const int deg = brow[row + 1] - b0;
        if (deg <= 0) continue;
        if (deg > cap) asm volatile("trap;");     // the caller's max_deg is wrong: fail loudly rather than overrun the row image
        // diagonal slot: bcol is ascending inside a row
        int lo = b0, hi = b0 + deg - 1;
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (__ldg(bcol + mid) < (int32_t)row) lo = mid + 1; else hi = mid;
        }
        const int q0 = contrib_ptr[lo], q1 = contrib_ptr[lo + 1];
        int pair = q0 < q1 ? __ldg(contrib + q0) : 0;
        int pair_next = q0 + 1 < q1 ? __ldg(contrib + q0 + 1) : 0;
        for (int q = q0; q < q1; ++q) {
            const int pair_next2 = q + 2 < q1 ? __ldg(contrib + q + 2) : 0;      // two entries ahead: an L2 round trip is longer than a step
            const int e = pair / NPE2;
            const int a = (pair - e * NPE2) / NPE;                       // the entry is (e, a, a)
            const double* __restrict__ g = geom + (int64_t)e * GEOM_STRIDE;
            const double mu = MODE == MAT_LAME ? __ldg(f.mu + e) : mu_s;      // warp-uniform: broadcast loads
            const double lam = MODE == MAT_LAME ? __ldg(f.lam + e) : lam_s;
            const float rho = FIELD ? __ldg(f.rho + e) : 0.0f;
            const int la0 = 3 * c_sup2[a][0], la1 = 3 * c_sup2[a][1];    // warp-uniform
            const int so = lane_on ? __ldg(slot + (int64_t)e * NPE2 + a * NPE + bb) - b0 : 0;
            const double2 ct01 = *reinterpret_cast<const double2*>(s_ct4 + (a * NPE + bb) * 4);       // (l0,m0) (l0,m1)
            const double2 ct23 = *reinterpret_cast<const double2*>(s_ct4 + (a * NPE + bb) * 4 + 2);   // (l1,m0) (l1,m1)
            double gl0[3], gl1[3], gm0[3], gm1[3];
#pragma unroll
            for (int d = 0; d < 3; ++d) {
                gl0[d] = __ldg(g + la0 + d);
                gl1[d] = __ldg(g + la1 + d);
                gm0[d] = __ldg(g + mb0 + d);
                gm1[d] = __ldg(g + mb1 + d);
            }
            const double detK = __ldg(g + 12), detM = __ldg(g + 13);
            // w_l = sum_m ct[l][m] G_m;  S = sum_l G_l w_l^T
            double w0[3], w1[3];
#pragma unroll
            for (int d = 0; d < 3; ++d) {
                w0[d] = fma(ct01.x, gm0[d], ct01.y * gm1[d]);
                w1[d] = fma(ct23.x, gm0[d], ct23.y * gm1[d]);
            }
            const double glc0 = c == 0 ? gl0[0] : (c == 1 ? gl0[1] : gl0[2]);
            const double glc1 = c == 0 ? gl1[0] : (c == 1 ? gl1[1] : gl1[2]);
            const double wc0 = c == 0 ? w0[0] : (c == 1 ? w0[1] : w0[2]);
            const double wc1 = c == 0 ? w1[0] : (c == 1 ? w1[1] : w1[2]);
            if constexpr (MODE == MAT_TENSOR) {
                // row c of the block: v[d] = sum_{k,l} C_{ckdl} S[k][l] with all nine S[k][l] = sum_li G_li[k] w_li[l];
                // C is warp-uniform (broadcast loads), lane c picks its three Voigt rows voigt(c, k)
                const double* __restrict__ Ce = f.C + (int64_t)e * 21;
                double Cv[21];
#pragma unroll
                for (int t = 0; t < 21; ++t) Cv[t] = __ldg(Ce + t);
                if (lane_on) {
                    double* out = acc + so * AT_SLOT + 3 * c;
                    double v[3] = {0.0, 0.0, 0.0};
#pragma unroll
                    for (int k = 0; k < 3; ++k) {
                        const int r0 = voigt(0, k), r1 = voigt(1, k), r2 = voigt(2, k);
#pragma unroll
                        for (int l = 0; l < 3; ++l) {
                            const double Skl = fma(gl0[k], w0[l], gl1[k] * w1[l]);
#pragma unroll
                            for (int d = 0; d < 3; ++d) {
                                const int J = voigt(d, l);
                                const double ck = c == 0 ? Cv[voigt_packed(r0, J)]
                                                         : (c == 1 ? Cv[voigt_packed(r1, J)] : Cv[voigt_packed(r2, J)]);
                                v[d] = fma(ck, Skl, v[d]);
                            }
                        }
                    }
                    out[0] += detK * v[0];
                    out[1] += detK * v[1];
                    out[2] += detK * v[2];
                    if (c == 0) acc[so * AT_SLOT + 9] += mass_entry<FIELD>(s_mtab[a * NPE + bb], rho) * detM;
                }
            } else {
                const double tr = mu * (fma(gl0[0], w0[0], fma(gl0[1], w0[1], gl0[2] * w0[2])) +
                                        fma(gl1[0], w1[0], fma(gl1[1], w1[1], gl1[2] * w1[2])));
                if (lane_on) {
                    double* out = acc + so * AT_SLOT + 3 * c;
                    double v[3];
#pragma unroll
                    for (int d = 0; d < 3; ++d) {
                        const double Scd = fma(glc0, w0[d], glc1 * w1[d]);          // S[c][d]
                        const double Sdc = fma(gl0[d], wc0, gl1[d] * wc1);          // S[d][c]
                        v[d] = fma(mu, Sdc, lam * Scd);
                    }
                    out[0] += detK * (c == 0 ? v[0] + tr : v[0]);
                    out[1] += detK * (c == 1 ? v[1] + tr : v[1]);
                    out[2] += detK * (c == 2 ? v[2] + tr : v[2]);
                    if (c == 0) acc[so * AT_SLOT + 9] += mass_entry<FIELD>(s_mtab[a * NPE + bb], rho) * detM;
                }
            }
            __syncwarp();
            pair = pair_next;
            pair_next = pair_next2;
        }
        // the finished row: three runs of 3 deg stiffness values, deg mass scalars; the image is cleared on the way out
        double* krow = Kval + 9 * (int64_t)b0;
        const int rs = 3 * deg;
#pragma unroll
        for (int cc = 0; cc < 3; ++cc)
            for (int t = lane; t < rs; t += 32) {
                const int s = t / 3, d = t - 3 * s;
                __stcs(krow + cc * rs + t, acc[s * AT_SLOT + 3 * cc + d]);
            }
        for (int s = lane; s < deg; s += 32) __stcs(Mblk + b0 + s, acc[s * AT_SLOT + 9]);
        __syncwarp();
        for (int t = lane; t < deg * AT_SLOT; t += 32) acc[t] = 0.0;
        __syncwarp();
    }
}

__global__ void k_mass_expand(const int32_t* __restrict__ brow, int64_t n_nodes, const double* __restrict__ Mblk,
                              double* __restrict__ Mval) {
    int lane = threadIdx.x & 31;
    int64_t row = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    if (row >= n_nodes) return;
    int64_t b0 = brow[row];
    int64_t deg = brow[row + 1] - b0;
    for (int64_t t = lane; t < 9 * deg; t += 32) {
        int c = (int)(t / (3 * deg));
        int64_t r = t - c * 3 * deg;
        int64_t p = r / 3;
        int d = (int)(r - 3 * p);
        Mval[9 * b0 + t] = (c == d) ? Mblk[b0 + p] : 0.0;
    }
}

// Legacy COO export, one thread per output triple (coalesced writes; the
// reference kernel writes msize^2 strided entries per thread).
__global__ void k_mass_coo(const double* __restrict__ vertices, const int32_t* __restrict__ tets, int64_t T,
                           int order, int vnum, const double* __restrict__ m, double d,
                           double* __restrict__ values, int32_t* __restrict__ rows, int32_t* __restrict__ cols) {
    int msize = 3 * vnum;
    int64_t msz2 = (int64_t)msize * msize;
    int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (idx >= T * msz2) return;
    int64_t e = idx / msz2;
    int r = (int)(idx - e * msz2);
    int i = r / msize, j = r - i * msize;
    const int32_t* t = tets + e * vnum;
    int32_t c[4];
    if (order == 1) { c[0] = t[0]; c[1] = t[1]; c[2] = t[2]; c[3] = t[3]; }
    else if (order == 2) { c[0] = t[0]; c[1] = t[2]; c[2] = t[4]; c[3] = t[9]; }
    else { c[0] = t[0]; c[1] = t[3]; c[2] = t[6]; c[3] = t[16]; }
    double x[4], y[4], z[4];
#pragma unroll
    for (int p = 0; p < 4; ++p) {
        x[p] = vertices[3 * (int64_t)c[p]];
        y[p] = vertices[3 * (int64_t)c[p] + 1];
        z[p] = vertices[3 * (int64_t)c[p] + 2];
    }
    double V = ((x[1] - x[0]) * ((y[2] - y[0]) * (z[3] - z[0]) - (y[3] - y[0]) * (z[2] - z[0])) +
                (y[1] - y[0]) * ((x[3] - x[0]) * (z[2] - z[0]) - (x[2] - x[0]) * (z[3] - z[0])) +
                (z[1] - z[0]) * ((x[2] - x[0]) * (y[3] - y[0]) - (x[3] - x[0]) * (y[2] - y[0]))) / 6;
    V = fabs(V) * 6;
    values[idx] = m[r] * d * V;
    rows[idx] = t[i / 3] * 3 + i % 3;
    cols[idx] = t[j / 3] * 3 + j % 3;
}

}  // namespace ds

using namespace ds;

static void assemble_account(int64_t T, int npe, int64_t n_nodes, int64_t nnzb, int mode) {
    prof_account(PROF_ASSEMBLE, 2.0 * 9.0 * (double)nnzb * 8.0 + (double)T * npe * 4.0 + (double)n_nodes * 12.0 + (double)T * npe * npe * 4.0 +
                 (mode == MAT_LAME ? (double)T * 20.0 : mode == MAT_TENSOR ? (double)T * (21.0 * 8.0 + 4.0) : 0.0), 0.0);
}

template <int MODE>
static int assemble_rows(const float* verts, const int32_t* tets, int64_t T, int order, int64_t n_nodes, double mu,
                         double lam, const FieldArgs& f, const double* ctab, const double* mtab, const int32_t* brow,
                         const int32_t* contrib_ptr, const int32_t* contrib, int64_t nnzb, double* geom, double* Kval,
                         double* Mblk, cudaStream_t stream) {
    int npe = order == 1 ? 4 : 10;
    ProfScope prof(PROF_ASSEMBLE, stream);
    assemble_account(T, npe, n_nodes, nnzb, MODE);
    k_tet_geometry<<<(unsigned)ceil_div(T, 128), 128, 0, stream>>>(verts, tets, T, npe, order, geom);
    DS_LAUNCH_CHECK();
    // grid-stride over rows: the per-order tables are staged into shared memory once per CTA
    unsigned blocks = (unsigned)std::min<int64_t>(ceil_div(n_nodes, AS_WARPS), 148 * 12);
    if (order == 1)
        k_assemble_rows<1, MODE><<<blocks, 32 * AS_WARPS, 0, stream>>>(geom, ctab, mtab, brow, contrib_ptr, contrib, n_nodes,
                                                                        mu, lam, f, Kval, Mblk);
    else
        k_assemble_rows<2, MODE><<<blocks, 32 * AS_WARPS, 0, stream>>>(geom, ctab, mtab, brow, contrib_ptr, contrib, n_nodes,
                                                                        mu, lam, f, Kval, Mblk);
    DS_LAUNCH_CHECK();
    return DS_OK;
}

template <int MODE>
static int assemble_tets(const float* verts, const int32_t* tets, int64_t T, int order, int64_t n_nodes, double mu,
                         double lam, const FieldArgs& f, const double* ctab, const double* mtab, const int32_t* brow,
                         const int32_t* bcol, const int32_t* contrib_ptr, const int32_t* contrib, const int32_t* slot,
                         int max_deg, int64_t nnzb, double* geom, double* Kval, double* Mblk, cudaStream_t stream) {
    const int npe = 10;
    ProfScope prof(PROF_ASSEMBLE, stream);
    assemble_account(T, npe, n_nodes, nnzb, MODE);
    k_tet_geometry<<<(unsigned)ceil_div(T, 128), 128, 0, stream>>>(verts, tets, T, npe, order, geom);
    DS_LAUNCH_CHECK();
    const int cap = (max_deg + 3) & ~3;
    const size_t smem = (size_t)(100 * 4 + 100 + (size_t)AT_WARPS * cap * AT_SLOT) * sizeof(double);
    DS_CUDA(cudaFuncSetAttribute(k_assemble_rows_tets2<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 1;
    DS_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_assemble_rows_tets2<MODE>, 32 * AT_WARPS, smem));
    int dev = 0, sms = 148;
    DS_CUDA(cudaGetDevice(&dev));
    DS_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const unsigned blocks = (unsigned)std::min<int64_t>(ceil_div(n_nodes, AT_WARPS), (int64_t)sms * std::max(per_sm, 1));
    k_assemble_rows_tets2<MODE><<<blocks, 32 * AT_WARPS, smem, stream>>>(geom, ctab, mtab, brow, bcol, contrib_ptr, contrib,
                                                                          slot, n_nodes, cap, mu, lam, f, Kval, Mblk);
    DS_LAUNCH_CHECK();
    return DS_OK;
}

extern "C" int ds_assemble_km(const float* verts, const int32_t* tets, int64_t T, int order, int64_t n_nodes,
                              double mu, double lam, const double* ctab, const double* mtab,
                              const int32_t* brow, const int32_t* bcol, const int32_t* contrib_ptr,
                              const int32_t* contrib, int64_t nnzb, double* geom, double* Kval, double* Mblk,
                              void* stream_) {
    (void)bcol;
    DS_REQUIRE(order == 1 || order == 2, "ds_assemble_km: order must be 1 or 2 (got %d)", order);
    DS_REQUIRE(verts && tets && ctab && mtab && brow && contrib_ptr && contrib && geom && Kval && Mblk,
               "ds_assemble_km: null argument");
    DS_REQUIRE(T > 0 && n_nodes > 0, "ds_assemble_km: empty mesh");
    return assemble_rows<MAT_SCALAR>(verts, tets, T, order, n_nodes, mu, lam, FieldArgs{}, ctab, mtab, brow, contrib_ptr, contrib,
                                nnzb, geom, Kval, Mblk, (cudaStream_t)stream_);
}

extern "C" int ds_assemble_km_field(const float* verts, const int32_t* tets, int64_t T, int order, int64_t n_nodes,
                                    const double* mu_t, const double* lam_t, const float* rho_t, const double* ctab,
                                    const float* m32, const int32_t* brow, const int32_t* bcol, const int32_t* contrib_ptr,
                                    const int32_t* contrib, int64_t nnzb, double* geom, double* Kval, double* Mblk,
                                    void* stream_) {
    (void)bcol;
    DS_REQUIRE(order == 1 || order == 2, "ds_assemble_km_field: order must be 1 or 2 (got %d)", order);
    DS_REQUIRE(verts && tets && mu_t && lam_t && rho_t && ctab && m32 && brow && contrib_ptr && contrib && geom && Kval && Mblk,
               "ds_assemble_km_field: null argument");
    DS_REQUIRE(T > 0 && n_nodes > 0, "ds_assemble_km_field: empty mesh");
    return assemble_rows<MAT_LAME>(verts, tets, T, order, n_nodes, 0.0, 0.0, FieldArgs{mu_t, lam_t, rho_t, m32, nullptr}, ctab, nullptr,
                               brow, contrib_ptr, contrib, nnzb, geom, Kval, Mblk, (cudaStream_t)stream_);
}

// Same result as ds_assemble_km for quadratic tets through the tet-sequential row kernel (k_assemble_rows_tets2);
// slot: the element -> pattern-slot map of ds_pattern_fill; max_deg: the longest block row (sizes the row image).
extern "C" int ds_assemble_km_tets(const float* verts, const int32_t* tets, int64_t T, int order, int64_t n_nodes,
                                   double mu, double lam, const double* ctab, const double* mtab,
                                   const int32_t* brow, const int32_t* bcol, const int32_t* contrib_ptr,
                                   const int32_t* contrib, const int32_t* slot, int max_deg, int64_t nnzb, double* geom,
                                   double* Kval, double* Mblk, void* stream_) {
    DS_REQUIRE(order == 2, "ds_assemble_km_tets: quadratic tets only (order 1 goes through ds_assemble_km)");
    DS_REQUIRE(verts && tets && ctab && mtab && brow && bcol && contrib_ptr && contrib && slot && geom && Kval && Mblk,
               "ds_assemble_km_tets: null argument");
    DS_REQUIRE(T > 0 && n_nodes > 0, "ds_assemble_km_tets: empty mesh");
    DS_REQUIRE(max_deg >= 1 && max_deg <= 256, "ds_assemble_km_tets: max_deg=%d must be in [1, 256] (longer rows: ds_assemble_km)",
               max_deg);
    return assemble_tets<MAT_SCALAR>(verts, tets, T, order, n_nodes, mu, lam, FieldArgs{}, ctab, mtab, brow, bcol, contrib_ptr,
                                contrib, slot, max_deg, nnzb, geom, Kval, Mblk, (cudaStream_t)stream_);
}

extern "C" int ds_assemble_km_tets_field(const float* verts, const int32_t* tets, int64_t T, int order, int64_t n_nodes,
                                         const double* mu_t, const double* lam_t, const float* rho_t, const double* ctab,
                                         const float* m32, const int32_t* brow, const int32_t* bcol,
                                         const int32_t* contrib_ptr, const int32_t* contrib, const int32_t* slot, int max_deg,
                                         int64_t nnzb, double* geom, double* Kval, double* Mblk, void* stream_) {
    DS_REQUIRE(order == 2, "ds_assemble_km_tets_field: quadratic tets only (order 1 goes through ds_assemble_km_field)");
    DS_REQUIRE(verts && tets && mu_t && lam_t && rho_t && ctab && m32 && brow && bcol && contrib_ptr && contrib && slot && geom &&
               Kval && Mblk, "ds_assemble_km_tets_field: null argument");
    DS_REQUIRE(T > 0 && n_nodes > 0, "ds_assemble_km_tets_field: empty mesh");
    DS_REQUIRE(max_deg >= 1 && max_deg <= 256,
               "ds_assemble_km_tets_field: max_deg=%d must be in [1, 256] (longer rows: ds_assemble_km_field)", max_deg);
    return assemble_tets<MAT_LAME>(verts, tets, T, order, n_nodes, 0.0, 0.0, FieldArgs{mu_t, lam_t, rho_t, m32, nullptr}, ctab, nullptr,
                               brow, bcol, contrib_ptr, contrib, slot, max_deg, nnzb, geom, Kval, Mblk, (cudaStream_t)stream_);
}

extern "C" int ds_assemble_km_tensor(const float* verts, const int32_t* tets, int64_t T, int order, int64_t n_nodes,
                                     const double* C21, const float* rho_t, const double* ctab, const float* m32,
                                     const int32_t* brow, const int32_t* bcol, const int32_t* contrib_ptr,
                                     const int32_t* contrib, int64_t nnzb, double* geom, double* Kval, double* Mblk,
                                     void* stream_) {
    (void)bcol;
    DS_REQUIRE(order == 1 || order == 2, "ds_assemble_km_tensor: order must be 1 or 2 (got %d)", order);
    DS_REQUIRE(verts && tets && C21 && rho_t && ctab && m32 && brow && contrib_ptr && contrib && geom && Kval && Mblk,
               "ds_assemble_km_tensor: null argument");
    DS_REQUIRE(T > 0 && n_nodes > 0, "ds_assemble_km_tensor: empty mesh");
    return assemble_rows<MAT_TENSOR>(verts, tets, T, order, n_nodes, 0.0, 0.0, FieldArgs{nullptr, nullptr, rho_t, m32, C21},
                                     ctab, nullptr, brow, contrib_ptr, contrib, nnzb, geom, Kval, Mblk, (cudaStream_t)stream_);
}

extern "C" int ds_assemble_km_tets_tensor(const float* verts, const int32_t* tets, int64_t T, int order, int64_t n_nodes,
                                          const double* C21, const float* rho_t, const double* ctab, const float* m32,
                                          const int32_t* brow, const int32_t* bcol, const int32_t* contrib_ptr,
                                          const int32_t* contrib, const int32_t* slot, int max_deg, int64_t nnzb,
                                          double* geom, double* Kval, double* Mblk, void* stream_) {
    DS_REQUIRE(order == 2, "ds_assemble_km_tets_tensor: quadratic tets only (order 1 goes through ds_assemble_km_tensor)");
    DS_REQUIRE(verts && tets && C21 && rho_t && ctab && m32 && brow && bcol && contrib_ptr && contrib && slot && geom && Kval &&
               Mblk, "ds_assemble_km_tets_tensor: null argument");
    DS_REQUIRE(T > 0 && n_nodes > 0, "ds_assemble_km_tets_tensor: empty mesh");
    DS_REQUIRE(max_deg >= 1 && max_deg <= 256,
               "ds_assemble_km_tets_tensor: max_deg=%d must be in [1, 256] (longer rows: ds_assemble_km_tensor)", max_deg);
    return assemble_tets<MAT_TENSOR>(verts, tets, T, order, n_nodes, 0.0, 0.0, FieldArgs{nullptr, nullptr, rho_t, m32, C21},
                                     ctab, nullptr, brow, bcol, contrib_ptr, contrib, slot, max_deg, nnzb, geom, Kval, Mblk,
                                     (cudaStream_t)stream_);
}

extern "C" int ds_mass_expand(const int32_t* brow, int64_t n_nodes, int64_t nnzb, const double* Mblk,
                              double* Mval, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    (void)nnzb;
    DS_REQUIRE(brow && Mblk && Mval, "ds_mass_expand: null argument");
    k_mass_expand<<<(unsigned)ceil_div(n_nodes * 32, 256), 256, 0, stream>>>(brow, n_nodes, Mblk, Mval);
    DS_LAUNCH_CHECK();
    return DS_OK;
}

extern "C" int ds_assemble_mass_coo(const double* vertices, const int32_t* tets, int64_t T, int order,
                                    const double* element_mm, double density, double* values, int32_t* rows,
                                    int32_t* cols, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    DS_REQUIRE(order >= 1 && order <= 3, "ds_assemble_mass_coo: order must be 1, 2 or 3 (got %d)", order);
    DS_REQUIRE(vertices && tets && element_mm && values && rows && cols, "ds_assemble_mass_coo: null argument");
    if (T == 0) return DS_OK;
    int vnum = order == 1 ? 4 : (order == 2 ? 10 : 20);
    int64_t total = T * 9 * vnum * vnum;
    k_mass_coo<<<(unsigned)ceil_div(total, 256), 256, 0, stream>>>(vertices, tets, T, order, vnum, element_mm,
                                                                  density, values, rows, cols);
    DS_LAUNCH_CHECK();
    return DS_OK;
}

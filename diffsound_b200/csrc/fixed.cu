// Clamped nodes: homogeneous Dirichlet conditions on whole nodes (all three displacement components fixed to zero).
// Nothing in the reference corresponds: it solves every object free-free.
//
// ds_fix_nodes_km constrains K and M in place on their block pattern.  Every off-diagonal block (i, j) with fixed[i] or
// fixed[j] becomes zero (its 9 K entries and its M scalar); diagonal blocks stay as assembled, so M stays SPD and the
// block-Jacobi D^-1 K of a fixed row is the identity.  The fixed dofs then decouple: K = diag(K_ff, K_cc), M likewise.
// A block vector whose fixed rows are exactly zero stays so under K and M, and every product, Gram matrix and residual
// of such vectors equals the one of the reduced problem on the free dofs.  The eigensolver (lobpcg.cu) keeps X, W and P
// in that subspace with the masking launches below, so the spurious pairs of the kept diagonal blocks never enter.
//
// One warp per node row, lanes over its blocks; each block is written by exactly one lane: no atomics, deterministic.
#include "common.cuh"
#include "../../include/diffsound_sm100.h"
#include "kernels.cuh"

namespace ds {

// Kval is in the scalar-CSR order of the reference: node row i is three scalar rows of 3 deg(i) entries each, so entry
// (c, d) of block p of row i sits at 9 brow[i] + 3 deg c + 3 p + d.
__global__ void __launch_bounds__(256) k_fix_nodes_km(const int32_t* __restrict__ brow, const int32_t* __restrict__ bcol,
                                                      int64_t n_nodes, const uint8_t* __restrict__ fixed,
                                                      double* __restrict__ Kval, double* __restrict__ Mblk) {
    const int64_t i = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (i >= n_nodes) return;
    const int64_t b0 = brow[i];
    const int deg = (int)(brow[i + 1] - b0);
    const bool fi = fixed[i] != 0;
    for (int p = lane; p < deg; p += 32) {
        const int32_t j = bcol[b0 + p];
        if (j == (int32_t)i || !(fi || fixed[j])) continue;
        if (Mblk) Mblk[b0 + p] = 0.0;
        double* k = Kval + 9 * b0 + 3 * p;
#pragma unroll
        for (int c = 0; c < 3; ++c)
#pragma unroll
            for (int d = 0; d < 3; ++d) k[(int64_t)c * 3 * deg + d] = 0.0;
    }
}

// V[3 i + q, c] = 0 for the nodes i of a row numbering with fixed[perm ? perm[i] : i] (q < 3, c < w); one thread per
// (node, column), so the writes of a fixed node are coalesced across its columns
template <typename T>
__global__ void __launch_bounds__(256) k_mask_fixed_rows(const uint8_t* __restrict__ fixed, const int32_t* __restrict__ perm,
                                                         int64_t n_nodes, T* __restrict__ V, int64_t ld, int w) {
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= n_nodes * w) return;
    const int64_t i = t / w;
    const int c = (int)(t - i * w);
    if (!fixed[perm ? perm[i] : i]) return;
#pragma unroll
    for (int q = 0; q < 3; ++q) V[(3 * i + q) * ld + c] = T(0);
}

template <typename T>
static int mask_rows(const uint8_t* fixed, const int32_t* perm, int64_t n_nodes, T* V, int64_t ld, int w, cudaStream_t st) {
    ProfScope prof(PROF_FIXED, st);
    k_mask_fixed_rows<T><<<(unsigned)ceil_div(n_nodes * w, 256), 256, 0, st>>>(fixed, perm, n_nodes, V, ld, w);
    DS_LAUNCH_CHECK();
    return DS_OK;
}

int mask_fixed_rows_f64(const uint8_t* fixed, const int32_t* perm, int64_t n_nodes, double* V, int64_t ld, int w,
                        cudaStream_t st) {
    return mask_rows(fixed, perm, n_nodes, V, ld, w, st);
}

int mask_fixed_rows_f32(const uint8_t* fixed, const int32_t* perm, int64_t n_nodes, float* V, int64_t ld, int w,
                        cudaStream_t st) {
    return mask_rows(fixed, perm, n_nodes, V, ld, w, st);
}

}  // namespace ds

using namespace ds;

extern "C" int ds_fix_nodes_km(const int32_t* brow, const int32_t* bcol, int64_t n_nodes, int64_t nnzb, const uint8_t* fixed,
                               double* Kval, double* Mblk, void* stream) {
    DS_REQUIRE(brow && bcol && fixed && Kval, "ds_fix_nodes_km: null argument");
    DS_REQUIRE(n_nodes > 0 && nnzb >= n_nodes, "ds_fix_nodes_km: bad sizes (n_nodes=%lld, nnzb=%lld)", (long long)n_nodes,
               (long long)nnzb);
    cudaStream_t st = (cudaStream_t)stream;
    ProfScope prof(PROF_FIXED, st);
    prof_account(PROF_FIXED, (double)nnzb * 4 + (double)n_nodes * 9, 0.0);
    k_fix_nodes_km<<<(unsigned)ceil_div(n_nodes * 32, 256), 256, 0, st>>>(brow, bcol, n_nodes, fixed, Kval, Mblk);
    DS_LAUNCH_CHECK();
    return DS_OK;
}

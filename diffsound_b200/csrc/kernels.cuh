// Internal (C++) entry points shared between translation units of the library.
#pragma once
#include "common.cuh"

namespace ds {

// spmm.cu
int spmm_km(const int32_t* brow, const int32_t* bcol, int64_t n_nodes, const double* Kval, const double* Mblk,
            double shift, const double* X, int64_t ldx, int ncols, double alpha, double beta, const double* Y0,
            int64_t ldy0, double* Y, int64_t ldy, cudaStream_t stream);
int spmm_dual(const int32_t* brow, const int32_t* bcol, int64_t n_nodes, const double* Kval, const double* Mblk,
              const double* X, int64_t ldx, int ncols, double* YK, int64_t ldyk, double* YM, int64_t ldym,
              cudaStream_t stream, const int32_t* order = nullptr, const int32_t* chunk_row = nullptr, int nchunks = 0);
// K Z, M Z for an fp32 block Z in a level's own (Morton) numbering; see k_spmm_dual_z32
int spmm_dual_z32(const int32_t* brow, const int32_t* browP, const int32_t* bcolP, const int32_t* perm,
                  const int32_t* chunk_row, int nchunks, int64_t n_nodes, const double* Kval, const double* Mblk,
                  const float* Z, int ncols, double* YK, int64_t ldyk, double* YM, int64_t ldym, cudaStream_t stream,
                  int64_t nnzb = 0);
int spmm32_chunk_count(int64_t n_nodes);

// precond32.cu -- FP32 preconditioner pieces
struct ColIdx {
    short v[128];
};
enum { S32_MODE_PLAIN = 0, S32_MODE_RESID = 1, S32_MODE_CHEB = 2 };
// Out = A X | R - A X | X + ab (X - Zprev) + cc invD (R - A X) on 48-byte block records; ncols in {16,32,48,64}
int spmm32(int mode, const int32_t* brow, const void* rec, int64_t n_nodes, int ncols, const float* X, const float* R,
           const float* invD, const float* Zprev, float* Out, float ab, float cc, int prof_cls, cudaStream_t st,
           const int32_t* chunk_row = nullptr);
// row chunks of the SpMM grid (one contiguous chunk per CTA, balanced by blocks + rows); chunk_row: >= 1024 ints
int spmm32_chunks(const int32_t* brow, int64_t n_nodes, int32_t* chunk_row, cudaStream_t st);
int pack_k32(const int32_t* brow, const int32_t* bcol, int64_t n_nodes, const double* Kval, const double* Mblk,
             double shift, void* rec, float* invD, cudaStream_t st, const uint32_t* colmap = nullptr,
             int64_t row_offset = 0, const int32_t* perm = nullptr, const int32_t* inv = nullptr,
             const int32_t* brow_out = nullptr);
int jacobi32(const float* invD, const float* R, int64_t n_nodes, int ncols, float cc, float* Out, cudaStream_t st);   // timed as PROF_JACOBI
// perm_* / inv_*: node renumberings of the levels' private (Morton) orderings, NULL = identity
int restrict32(const int32_t* rptr, const int32_t* rlist, int64_t n_coarse, const float* res, int ncols, float* rc,
               cudaStream_t st, const int32_t* perm_c = nullptr, const int32_t* inv_f = nullptr);
int prolong_add32(const int32_t* par, int64_t n_fine, const float* zc, int ncols, float* z, cudaStream_t st,
                  const int32_t* perm_f = nullptr, const int32_t* inv_c = nullptr);
int prolong64(const int32_t* par, int64_t n_fine, const double* xc, int64_t ldc, int w, double* x, int64_t ldx,
              cudaStream_t st);
int inject64(const int32_t* rptr, const int32_t* rlist, int64_t n_coarse, const double* x, int64_t ldx, int w,
             double* xc, int64_t ldc, cudaStream_t st);
int gather_cols_f32(const double* src, int64_t lds, const ColIdx& idx, int count, int width, int64_t n, float* dst,
                    cudaStream_t st, const int32_t* perm = nullptr);
int widen_f32(const float* src, int width, int64_t n, double* dst, int64_t ldd, cudaStream_t st,
              const int32_t* perm = nullptr);
int colnorm2_f32(const float* V, int w, int64_t n, double* partial, int ctas, cudaStream_t st);
// fixed.cu: V[3 i + q, :w] = 0 for the nodes i of a row numbering with fixed[perm ? perm[i] : i] (timed as PROF_FIXED)
int mask_fixed_rows_f64(const uint8_t* fixed, const int32_t* perm, int64_t n_nodes, double* V, int64_t ld, int w,
                        cudaStream_t st);
int mask_fixed_rows_f32(const uint8_t* fixed, const int32_t* perm, int64_t n_nodes, float* V, int64_t ld, int w,
                        cudaStream_t st);
int fill_random_f32(float* V, int64_t count, uint64_t seed, cudaStream_t st);

// Morton codes of points (also used by the triangle-mesh BVH of sdf.cu).  ordered_key maps a float to a uint32 whose
// unsigned order is the float order (atomicMin / atomicMax on keys give float bounds); key_to_float inverts it.
__device__ __forceinline__ uint32_t ordered_key(float f) {
    const uint32_t u = __float_as_uint(f + 0.0f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float key_to_float(uint32_t k) {
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}
// mm[0..2] = min key per axis, mm[3..5] = max key per axis of coords [n x 3] (mm initialised to 0xffffffff / 0 by the
// caller; any grid, grid-stride loop)
__global__ void k_bbox(const float* __restrict__ coords, int64_t n, uint32_t* __restrict__ mm);
// codes[i] = 30-bit Morton code of point i inside the box mm, iota[i] = i
__global__ void k_morton_codes(const float* __restrict__ coords, int64_t n, const uint32_t* __restrict__ mm,
                               uint32_t* __restrict__ codes, uint32_t* __restrict__ iota);

// one level of the FP32 preconditioner: records + block-Jacobi inverse + spectral bound of invD A
struct Level32 {
    const int32_t* brow = nullptr;           // row pointers in the level's own numbering
    const int32_t *perm = nullptr, *inv = nullptr;   // own row -> matrix row and back (NULL: identity)
    bool want_bcolP = false;                 // set before setup(): also keep the column ids in the level's numbering
    const int32_t* bcolP = nullptr;          // [nnzb] column ids in the level's numbering, rows in the level's order
    int64_t n_nodes = 0, nnzb = 0;
    unsigned char* rec = nullptr;
    float* invD = nullptr;
    int32_t* chunk_row = nullptr;
    unsigned* gbar = nullptr;                // [0] grid-barrier counter, [1] error flag of the persistent Chebyshev kernel
    bool persistent = false;                 // cooperative launches available
    double lmax = 0.0;
    int prof_cls = PROF_CHEB;
    int64_t launches = 0, cols = 0;          // SpMM launches and the sum of their column counts
    static size_t bytes(int64_t n_nodes, int64_t nnzb);
    int setup(Arena& a, const int32_t* brow, const int32_t* bcol, int64_t n_nodes, int64_t nnzb, const double* Kval,
              const double* Mblk, double shift, const float* coords, cudaStream_t st);
    // z = p(invD A) invD r, `degree` Chebyshev steps on [lmax/ratio, lmax]; from_zero: z0 = 0, else z0 = *zc.
    // zc / zp ping-pong; the result is in *zc on return.
    int cheb(const float* r, int ncols, int degree, double ratio, bool from_zero, float** zc, float** zp,
             cudaStream_t st);
};

// dense.cu
int64_t gram_scratch_elems(int p, int q);
int gram_f64(const double* A, int64_t lda, int p, const double* B, int64_t ldb, int q, int64_t n, double* G,
             int64_t ldg, double* partial, cudaStream_t stream);
// gram_sym.cu: GK = S^T KS, GM = S^T MS (upper-triangle 8x8 tiles over the active tile columns), one pass
int64_t gram_sym2_scratch_elems(int num_sms);
int gram_sym2(const double* S, const double* KS, const double* MS, int64_t ld, int64_t n, const int* tiles, int ntiles,
              double* GK, double* GM, int64_t ldg, double* partial, int num_sms, cudaStream_t stream);
// Y = beta Y + alpha A C
int block_gemm_f64(const double* A, int64_t lda, int p, const double* C, int64_t ldc, int q, int64_t n, double alpha,
                   double beta, double* Y, int64_t ldy, cudaStream_t stream);
// fused Rayleigh-Ritz update of the three wide buffers: Y[:, :m] = A[:, :prow] C1, Y[:, 2m:2m+q2] = A[:, m:prow] C2
int rr_update_f64(const double* const A[3], int64_t lda, int prow, int m, const double* C1, const double* C2, int q2,
                  int64_t ldc, int64_t n, double* const Y[3], int64_t ldy, cudaStream_t stream);
// rr.cu: strips of the Gram pair that involve the new W, small-matrix recurrences for the rest, leaner basis update
int64_t gram_strip_scratch_elems(int num_sms);
int gram_strip(const double* KW, const double* MW, int64_t ldw, int wa, const double* S, int64_t lds, int ncol, int64_t n,
               double* GsK, double* GsM, int64_t ldg, double* partial, int num_sms, cudaStream_t stream);
int gram_algebra(const double* GK, const double* GM, double* GKn, double* GMn, int64_t ldg, const double* C, int64_t ldc,
                 const double* theta, int m, double* scratch, cudaStream_t stream);
int64_t gram_algebra_scratch_elems();
int gram_insert(double* GK, double* GM, int64_t ldg, const double* GsK, const double* GsM, int64_t lds, int m, int wa,
                cudaStream_t stream);
int sym_upper(double* GK, double* GM, int64_t ldg, int N, cudaStream_t stream);
int rr_update2_f64(const double* const A[3], int64_t lda, int m, int wa, int use_p, const double* C, int64_t ldc, int64_t n,
                   double* const Y[3], int64_t ldy, cudaStream_t stream);
// idx_host (may be NULL = identity): slot of compact index i inside the ldg x ldg Gram storage;
// only the upper triangle of the storage is read; rows of C are written at the mapped slots.
// sigma < 0 selects an automatic shift |sigma| * mean(diag(scaled GK)).
int64_t eigh_scratch_elems(int N);
int eigh_generalized_f64(const double* GK, const double* GM, int N, int64_t ldg, const int* idx_host, double sigma,
                         double* theta, double* C, int64_t ldc, double* scratch, int* info, cudaStream_t stream);

}  // namespace ds

/*
 * libdiffsound_sm100.so -- C-ABI of the B200-native modal-analysis hot path.
 *
 * This is the drop-in boundary.  The reference's only native plugin is the
 * torch extension `diffFEM` (src/cuda_module.py:7-41) exporting one op,
 * `assemble_mass_matrix` (src/cuda/massMatrixDouble.h:14-15, bind.cu:11); the
 * rest of the path is torch-eager + SciPy inside src/diffelastic, src/lobpcg
 * and src/ddsp.  Each entry point below names the reference code it replaces.
 *
 * Conventions (all functions):
 *   - return 0 on success, <0 on error; message via ds_last_error() (thread-local)
 *   - every pointer is a DEVICE pointer owned by the caller (torch) unless the
 *     parameter is documented as "host"; nothing is allocated except inside an
 *     explicit ds_workspace
 *   - work is enqueued on `stream` (a cudaStream_t passed as void*); calls are
 *     asynchronous unless documented as synchronising
 *   - callable from any host thread (autograd runs backward on its own thread);
 *     the caller has made the right device current
 *   - dense block vectors are ROW-MAJOR (n x ncols) with a leading dimension ld
 */
#ifndef DIFFSOUND_SM100_H
#define DIFFSOUND_SM100_H

#include <stdint.h>

/* The library is built with -fvisibility=hidden: only the C-ABI declared here is exported. */
#if defined(__GNUC__)
#pragma GCC visibility push(default)
#endif
#ifdef __cplusplus
extern "C" {
#endif

typedef struct ds_workspace ds_workspace;

/* ---- library ------------------------------------------------------------ */
int ds_version(void);
const char* ds_last_error(void);
/* scratch arena; replaces the implicit temporaries torch allocates inside
 * coalesce()/sparse.mm on the reference path (diff_model.py:217-220).  One workspace may be used from several
 * streams of ONE host thread (a call on another stream than the previous one is ordered behind it with an event);
 * concurrent host threads need a workspace each. */
int ds_workspace_create(ds_workspace** ws);
int ds_workspace_destroy(ds_workspace* ws);
int64_t ds_workspace_bytes(const ds_workspace* ws);

/* ---- sparsity pattern (integer, bit-exact) --------------------------------
 * Replaces the pattern that `sparse_coo_tensor(...).coalesce()` derives by
 * sort-and-reduce on every batch (diff_model.py:214-220, 305-312; SURVEY A.3).
 * tets: int32 [T*npe] node ids (npe = 4 or 10).  The pattern is the node-level
 * block CSR (brow/bcol, dense 3x3 blocks); ds_pattern_expand_csr emits the
 * scalar CSR (crow, col int64) that equals the reference's coalesced indices.
 * ds_pattern_count synchronises the stream (it returns nnzb to the host). */
int ds_pattern_count(ds_workspace* ws, const int32_t* tets, int64_t T, int npe,
                     int64_t n_nodes, int64_t* nnzb_host, void* stream);
/* contrib_ptr[nnzb+1], contrib[T*npe*npe]: for every block slot the element
 * entries e*npe*npe + a*npe + b that sum into it (ascending); slot (optional,
 * may be NULL) is the inverse map [T*npe*npe] -> block slot. */
int ds_pattern_fill(ds_workspace* ws, int64_t n_nodes, int32_t* brow, int32_t* bcol,
                    int32_t* contrib_ptr, int32_t* contrib, int32_t* slot, void* stream);
int ds_pattern_expand_csr(const int32_t* brow, const int32_t* bcol, int64_t n_nodes,
                          int64_t nnzb, int64_t* crow, int64_t* col, void* stream);

/* ---- assembly --------------------------------------------------------------
 * Fused K and M assembly straight into the fixed pattern; replaces
 * DiffSoundObj.update_stiff_matrix + update_mass_matrix (diff_model.py:184-312),
 * Deform.precompute_* (deform.py:35-68, 136-147) and the dead-code kernel
 * compute_mass_matrix_kernel (src/cuda/massMatrixDouble.cu:3-78).
 * verts: fp32 [n_nodes*3]; order 1|2; ctab: fp64 [npe*npe*16] = sum_g w_g
 * dN_a/dL_l dN_b/dL_m from the reference's fp32 Gauss rule; mtab: fp64
 * [npe*npe] = double(float(m_ab)*float(rho)) (diff_model.py:299-303).
 * Kval: fp64 [9*nnzb] in the reference's scalar-CSR (row, col) order.
 * Mblk: fp64 [nnzb], M = Mblk (x) I3 (the expanded reference values come from
 * ds_mass_expand).  geom: fp64 scratch [T*14].  Owner-computes: the warp that owns
 * a node row sums the contributors of its block slots in ascending order, the
 * work split evenly over its lanes -- no atomics, deterministic. */
int ds_assemble_km(const float* verts, const int32_t* tets, int64_t T, int order,
                   int64_t n_nodes, double mu, double lam, const double* ctab,
                   const double* mtab, const int32_t* brow, const int32_t* bcol,
                   const int32_t* contrib_ptr, const int32_t* contrib, int64_t nnzb,
                   double* geom, double* Kval, double* Mblk, void* stream);
/* Same result for quadratic tets (order 2) through the tet-sequential row kernel: a warp owns a node row and walks the
 * tets around that node in ascending order, every geometry load is one broadcast address per warp, the row is summed in a
 * shared-memory image and leaves as coalesced streaming stores (csrc/assemble.cu, k_assemble_rows_tets2).  Replaces the
 * same reference lines as ds_assemble_km.  slot: int32 [T*npe*npe], the element -> pattern-slot map ds_pattern_fill
 * writes when asked to; max_deg: the longest block row of the pattern, 1..256 (longer rows: use ds_assemble_km). */
int ds_assemble_km_tets(const float* verts, const int32_t* tets, int64_t T, int order, int64_t n_nodes,
                        double mu, double lam, const double* ctab, const double* mtab,
                        const int32_t* brow, const int32_t* bcol, const int32_t* contrib_ptr,
                        const int32_t* contrib, const int32_t* slot, int max_deg, int64_t nnzb, double* geom,
                        double* Kval, double* Mblk, void* stream);
int ds_mass_expand(const int32_t* brow, int64_t n_nodes, int64_t nnzb, const double* Mblk,
                   double* Mval, void* stream);
/* Legacy twin of the reference export `assemble_mass_matrix` (massMatrixDouble.cu:138-158):
 * COO triples, msize*msize per tet, same layout/dtypes (vertices fp64 flat, tets int32 flat,
 * element_mm fp64 flat msize*msize). */
int ds_assemble_mass_coo(const double* vertices, const int32_t* tets, int64_t T, int order,
                         const double* element_mm, double density, double* values,
                         int32_t* rows, int32_t* cols, void* stream);

/* ---- sparse x dense block --------------------------------------------------
 * Replaces torch sparse COO `K @ U`, `M @ U` (diff_model.py:395-397, 385;
 * _linalg_utils.py:27-39).  Y = alpha*(K + shift*M) X + beta*Y0 on the block
 * pattern; any of Kval / Mblk may be NULL (treated as zero).  ncols multiple of
 * 16, <= 128.  X must not alias Y. */
int ds_spmm_km(const int32_t* brow, const int32_t* bcol, int64_t n_nodes,
               const double* Kval, const double* Mblk, double shift,
               const double* X, int64_t ldx, int ncols,
               double alpha, double beta, const double* Y0, int64_t ldy0,
               double* Y, int64_t ldy, void* stream);
/* YK = K X and YM = M X in one pass over X (both needed by LOBPCG). */
int ds_spmm_k_and_m(const int32_t* brow, const int32_t* bcol, int64_t n_nodes,
                    const double* Kval, const double* Mblk, const double* X, int64_t ldx,
                    int ncols, double* YK, int64_t ldyk, double* YM, int64_t ldym, void* stream);

/* ---- dense tall-skinny pieces of Rayleigh-Ritz ------------------------------
 * Replace torch.matmul / qform / linalg.cholesky / linalg.eigh calls in
 * src/lobpcg/_lobpcg.py:433-525 and _linalg_utils.py:63-96. */
/* G[p x q] (row-major, ldg) = A^T B, A (n x p, lda), B (n x q, ldb); FP64 DMMA,
 * split over row chunks, deterministic two-pass reduction.  partial: scratch
 * fp64 [ds_gram_scratch_elems(p,q)]. */
int64_t ds_gram_scratch_elems(int p, int q);
int ds_gram_f64(const double* A, int64_t lda, int p, const double* B, int64_t ldb, int q,
                int64_t n, double* G, int64_t ldg, double* partial, void* stream);
/* Fused Rayleigh-Ritz Gram pair in one pass over S, KS, MS (n x ld row-major, ld multiple of 8,
 * <= 144): GK = S^T KS, GM = S^T MS restricted to the 8-column tiles listed in tiles_host
 * (ascending, host int[ntiles]); only tiles with row-tile <= column-tile (upper triangle) of the
 * ldg-strided outputs are written.  partial: fp64 [ds_gram_sym2_scratch_elems()]. */
int64_t ds_gram_sym2_scratch_elems(void);
int ds_gram_sym2_f64(const double* S, const double* KS, const double* MS, int64_t ld, int64_t n,
                     const int* tiles_host, int ntiles, double* GK, double* GM, int64_t ldg,
                     double* partial, void* stream);
/* Y (n x q) = beta*Y + A (n x p) C (p x q, row-major ldc) */
int ds_block_gemm_f64(const double* A, int64_t lda, int p, const double* C, int64_t ldc, int q,
                      int64_t n, double beta, double* Y, int64_t ldy, void* stream);
/* Fused Rayleigh-Ritz update of a LOBPCG step (_lobpcg.py:463-466, X = S Z and the new P block), for the
 * three wide buffers A in {S, KS, MS} (n x lda, columns [X | W | P], m columns each) in one launch:
 *   A_out[:, 0:m] = A[:, 0:prow] C1 (prow x m);   A_out[:, 2m:2m+q2] = A[:, m:prow] C2 ((prow-m) x q2).
 * m in {16, 32, 48}; q2 in {0, 16, 32, 48}; prow a multiple of 4 in [m, 144]; C1, C2 row-major, ldc. */
int ds_rr_update_f64(const double* S, const double* KS, const double* MS, int64_t lda, int prow, int m,
                     const double* C1, const double* C2, int q2, int64_t ldc, int64_t n, double* S_out,
                     double* KS_out, double* MS_out, int64_t ldy, void* stream);
/* Generalised symmetric eigenproblem GK c = theta GM c, N <= 144: Cholesky of GM and of
 * GK + sigma*GM (one CTA), one-sided Jacobi on a thread-block cluster of 8 CTAs (rows in registers,
 * row exchange through distributed shared memory), back substitution (one CTA).
 * theta ascending [N], C [N x N] row-major (columns = GM-orthonormal vectors).
 * scratch: fp64 [ds_eigh_scratch_elems(N)].  info (device int[2]): {0 ok | failing pivot index+1
 * (+1000 when the failure is in GK + sigma*GM), sweeps used}. */
int64_t ds_eigh_scratch_elems(int N);
int ds_eigh_generalized_f64(const double* GK, const double* GM, int N, int64_t ldg, double sigma,
                            double* theta, double* C, int64_t ldc, double* scratch, int* info,
                            void* stream);

/* ---- eigensolver -----------------------------------------------------------
 * Lowest `nev` eigenpairs of K u = lambda M u; replaces eigen_decomposition_arpack
 * (diff_model.py:335-369: scipy eigsh shift-invert on the CPU) and is the engine
 * behind the lobpcg / lobpcg_func API mirror (src/lobpcg/_lobpcg.py:8-212).
 * X: fp64 [n x m] row-major start block on entry (m >= nev, multiple of 16),
 * M-orthonormal Ritz vectors on exit; lambda_out [m]; resid_out [m] relative
 * residuals; stats_host (host int64[12]) = {iterations, converged, spmm_count, status,
 * fine-level FP32 SpMM launches, sum over those launches of the column count,
 * coarse-level launches, sum of their column counts, iterations of the nested coarse eigen-solve,
 * its status, round(1e9 * lmax) of the fine level's Chebyshev interval (the estimate of the largest eigenvalue of invD K,
 * safety factor included), the same for the coarse level (0 without one)}.
 * Preconditioner (FP32, see ds_spmm32): `cheb_degree` steps of block-Jacobi Chebyshev on
 * K + sigma*M, or, when `coarse` is given (quadratic meshes), a two-level p-multigrid V-cycle:
 * `smooth_steps` Chebyshev-Jacobi steps on [lmax/smooth_ratio, lmax] before and after a
 * `coarse_degree`-step Chebyshev solve on the P1 operator.
 * Synchronises the stream. */
typedef struct ds_lobpcg_opts {
    int nev;            /* number of pairs that must converge (lowest nev) */
    int maxit;
    int cheb_degree;
    double tol;         /* ||K x - lam M x|| / (lam ||M x||) */
    double sigma;       /* shift for the preconditioner / RR (<=0: automatic) */
    double cheb_ratio;  /* lmax / lmin of the Chebyshev interval */
    int n_rigid;        /* leading columns that hold (near-)null-space vectors; -1: detect */
    int verbose;
    int smooth_steps;   /* two-level only: Chebyshev-Jacobi steps per smoothing leg (default 3) */
    int coarse_degree;  /* two-level only: Chebyshev steps of the coarse solve */
    double smooth_ratio;/* lmax / lmin of the smoother interval (default 8) */
    double coarse_ratio;/* lmax / lmin of the coarse Chebyshev interval */
    int nested;         /* two-level only (needs coarse->Mblk): solve the P1 eigenproblem first and start
                           the P2 iteration from its prolonged Ritz vectors (nested iteration) */
    double nested_tol;  /* residual tolerance of that coarse solve (default 3e-2) */
    int nested_degree;  /* Chebyshev degree of the coarse solve's one-level preconditioner (0: automatic) */
    const float* coords;/* device fp32 [n_nodes x 3] node coordinates or NULL.  When given, the FP32 preconditioner
                           stores its operator renumbered along a Morton curve through the nodes (a private
                           numbering: locality for the gathered rows of the SpMM); results are unaffected */
    const double* locked;/* device fp64 [n x n_locked] (ld = n_locked) or NULL: M-orthonormal eigenvectors already
                           converged by earlier calls.  The iteration is kept M-orthogonal to them (hard locking /
                           deflation), so this call returns the NEXT lowest pairs: how DiffSoundObj solves
                           mode_num + 6 > 44 pairs (geometry_train.py:147 asks for 64) in batches of one block */
    int n_locked;       /* columns of `locked`, a multiple of 16, <= 192 (pad with zero columns) */
    int precond_fp64;   /* != 0: the preconditioner is a block-Jacobi Chebyshev polynomial of degree cheb_degree on K evaluated in
                           FP64 (one level, no coarse correction).  Robust fall-back for meshes with sliver elements
                           (marching-tets output), where a residual's stiff components exceed its smooth part by more than
                           the 2^24 an FP32 cycle resolves.  0 (default): the FP32 cycle */
    int ortho_w;        /* != 0: M-orthogonalise the new search block W against X in FP64 before K W / M W are formed
                           (round-1 behaviour; lobpcg/_lobpcg.py 'ortho').  0 (default): W is the fp32 preconditioner
                           output as is and K W, M W are formed from it directly (k_spmm_dual_z32) */
} ds_lobpcg_opts;
/* Coarse level of the two-level preconditioner: the P1 operator on the corner nodes of a quadratic
 * mesh (pattern + values from ds_pattern_* / ds_assemble_km at order 1 on ds_pmg_coarse_fill's
 * output) and the transfer tables.  All device pointers. */
typedef struct ds_pmg_level {
    const int32_t* brow;      /* [n_nodes+1] */
    const int32_t* bcol;      /* [nnzb] */
    int64_t n_nodes;          /* coarse (corner) nodes */
    int64_t nnzb;
    const double* Kval;       /* [9*nnzb] */
    const double* Mblk;       /* [nnzb] or NULL (only used with sigma > 0) */
    const int32_t* parents;   /* [2*n_fine_nodes]: fine node i = 0.5 (coarse parents[2i] + parents[2i+1]) */
    const int32_t* rptr;      /* [n_nodes+1]  transpose (gather) lists of the prolongation */
    const int32_t* rlist;     /* [2*n_fine_nodes] */
    const float* coords;      /* fp32 [n_nodes x 3] coarse node coordinates or NULL (see ds_lobpcg_opts.coords) */
} ds_pmg_level;
int ds_lobpcg(ds_workspace* ws, const int32_t* brow, const int32_t* bcol, int64_t n_nodes,
              const double* Kval, const double* Mblk, const ds_pmg_level* coarse /* may be NULL */,
              double* X, int m, const ds_lobpcg_opts* opts, double* lambda_out, double* resid_out,
              int64_t* stats_host, void* stream);

/* ---- mesh promotion: node numbering -----------------------------------------------------------
 * Replaces torch.unique(vertices, dim=0, return_inverse=True) + scatter(min) in
 * TetMesh.remove_duplicate_vertices (diffelastic/mesh.py:162-179), called by to_high_order
 * (mesh.py:101-160) on the V + 6T candidate nodes and by import_from_file (mesh.py:196).
 * rows: device fp32 [N x 3].  count: sorts and returns the number of distinct rows (one stream sync);
 * fill: inverse[N] (int64, id of every input row = rank of its coordinates in ascending (x, y, z)
 * order) and first[n_unique] (int64, smallest input index of every group).  -0.0 == +0.0. */
int ds_unique_rows3_count(ds_workspace* ws, const float* rows, int64_t N, int64_t* n_unique_host, void* stream);
int ds_unique_rows3_fill(ds_workspace* ws, int64_t* inverse, int64_t* first, void* stream);

/* ---- FP32 preconditioner pieces (exported for tests and for callers that build their own cycle) ---
 * No reference counterpart: the reference factorises K - sigma M with SuperLU on the CPU
 * (diff_model.py:356-358).  rec: ds_k32_record_bytes(nnzb) bytes, 16-byte aligned, one 48-byte
 * record {k00..k22 (fp32), bcol, 8 bytes of padding} per block of K + shift*M; invD: fp32 [9*n_nodes] inverses of the
 * diagonal blocks.  ds_spmm32 modes: 0: Out = A X; 1: Out = R - A X; 2 (one Chebyshev step):
 * Out = X + ab (X - Zprev) + cc invD (R - A X), Zprev may alias Out, X must not.  Dense blocks are
 * fp32 row-major [3*n_nodes x ncols] with ld = ncols in {16, 32, 48, 64}. */
int64_t ds_k32_record_bytes(int64_t nnzb);
int ds_k32_pack(const int32_t* brow, const int32_t* bcol, int64_t n_nodes, int64_t nnzb,
                const double* Kval, const double* Mblk, double shift, void* rec, float* invD,
                void* stream);
int ds_spmm32(int mode, const int32_t* brow, const void* rec, int64_t n_nodes, int ncols,
              const float* X, const float* R, const float* invD, const float* Zprev, float* Out,
              double ab, double cc, const int32_t* chunk_row, void* stream);
/* Row chunks of the SpMM grid: one 1024-thread CTA per SM sweeps a contiguous chunk of node rows so that
 * the gathered rows of X stay in that SM's L1; chunk_row[ds_spmm32_chunk_count(n_nodes) + 1] (device)
 * holds the first row of every chunk, balanced by blocks + rows.  ds_spmm32 accepts chunk_row = NULL and
 * then builds the chunks into a stream-ordered temporary on every call. */
int ds_spmm32_chunk_count(int64_t n_nodes);
/* z = p(invD A) invD R: `degree` block-Jacobi Chebyshev steps on [lmax / ratio, lmax] from a zero initial guess (the
 * coarse solve of the V-cycle and the one-level preconditioner of the nested eigen-solve).  persistent != 0: all
 * steps in ONE cooperative launch, one CTA per SM, the block records of each CTA's row chunk held in shared memory
 * and the steps separated by a grid barrier (levels whose records fit on chip); 0: one SpMM launch per step.
 * Za, Zb: fp32 ping-pong buffers [3*n_nodes x ncols]; *which_host = 0 / 1: result in Za / Zb.  Synchronises. */
int ds_cheb32_solve(const int32_t* brow, const void* rec, const float* invD, int64_t n_nodes, int64_t nnzb,
                    const float* R, int ncols, int degree, double lmax, double ratio, int persistent,
                    float* Za, float* Zb, int* which_host, void* stream);
int ds_spmm32_chunks(const int32_t* brow, int64_t n_nodes, int32_t* chunk_row, void* stream);

/* Row-partitioned SpMM for one large mesh on several GPUs of a node (SURVEY.md section 8e): rank r owns
 * a contiguous slab of node rows; the records of its slab carry column ids packed as
 * owner << 28 | index inside the owner's slab (colmap), and the kernel gathers the dense block through
 * Xparts_host[world] -- device pointers, valid in THIS process, of every rank's slab (the peers' come
 * from ds_peer_open; loads cross NVLink).  No collective: the caller orders the ranks (barrier) between
 * a step that writes a slab and the step that gathers it.  Replaces the all-gather + torch.sparse.mm a
 * torch implementation of the reference's K @ U would need. */
int ds_k32_pack_slab(const int32_t* brow_win, const int32_t* bcol_slab, int64_t n_local,
                     int64_t nnzb_local, int64_t row0, const double* Kval_slab,
                     const double* Mblk_slab, double shift, const uint32_t* colmap, void* rec,
                     float* invD, void* stream);
int ds_spmm32_rowpart(int mode, const int32_t* brow_local, const void* rec, int64_t n_local, int ncols,
                      const float* const* Xparts_host, int world, int rank, const float* R,
                      const float* invD, const float* Zprev, float* Out, double ab, double cc,
                      void* stream);
/* peer-visible device memory (cudaMalloc + 64-byte CUDA IPC handle) */
int ds_peer_alloc(int64_t bytes, void** ptr, unsigned char* handle64);
int ds_peer_open(const unsigned char* handle64, void** ptr);
int ds_peer_close(void* ptr);
int ds_peer_free(void* ptr);
/* Quadratic -> linear coarsening (integer work).  tets: int32 [T*10] in the reference's local
 * order (mesh.py:139-154: corners at 0,2,4,9).  cid[n_nodes]: coarse id of each corner node
 * (ascending fine id) or -1; ds_pmg_coarse_count synchronises and returns n_coarse.
 * ds_pmg_coarse_fill writes ctets [T*4], cverts fp32 [n_coarse*3], parents [2*n_nodes] (8-byte
 * aligned), rptr [n_coarse+1], rlist [2*n_nodes]. */
int ds_pmg_coarse_count(ds_workspace* ws, const int32_t* tets, int64_t T, int64_t n_nodes,
                        int32_t* cid, int64_t* n_coarse_host, void* stream);
int ds_pmg_coarse_fill(ds_workspace* ws, const float* verts, const int32_t* tets, int64_t T,
                       int64_t n_nodes, const int32_t* cid, int64_t n_coarse, int32_t* ctets,
                       float* cverts, int32_t* parents, int32_t* rptr, int32_t* rlist, void* stream);
/* rc = P^T res, z += P zc on fp32 blocks [3*nodes x ncols] (ncols multiple of 4) */
int ds_pmg_restrict32(const int32_t* rptr, const int32_t* rlist, int64_t n_coarse, const float* res,
                      int ncols, float* rc, void* stream);
int ds_pmg_prolong_add32(const int32_t* parents, int64_t n_fine, const float* zc, int ncols,
                         float* z, void* stream);

/* ---- eigenvalue derivative --------------------------------------------------
 * Shape: grad_verts += d/dx sum_i g_i (u_i^T K u_i - lam_i u_i^T M u_i); replaces
 * autograd through get_vals (diff_model.py:390-399 -> coalesce/bmm/inverse graph).
 * ctab/mtab: the assembly tables (ds_assemble_km).
 * U fp64 [3*n_nodes x ldu] (k columns used), lam/g fp64 [k]; tet_grad scratch
 * fp64 [T*12]; inc_ptr/inc: node -> (tet*4+corner) incidence (ds_corner_incidence);
 * grad_verts fp32 [n_nodes*3] (overwritten). */
int ds_corner_incidence(ds_workspace* ws, const int32_t* tets, int64_t T, int npe, int order,
                        int64_t n_nodes, int32_t* inc_ptr, int32_t* inc, void* stream);
int ds_eigval_grad_shape(const float* verts, const int32_t* tets, int64_t T, int order,
                         int64_t n_nodes, double mu, double lam_lame, const double* ctab,
                         const double* mtab,
                         const double* U, int64_t ldu, int k, const double* lam, const double* g,
                         const int32_t* inc_ptr, const int32_t* inc, double* tet_grad,
                         float* grad_verts, void* stream);
/* Material: q_mu[i] = u_i^T K(mu=1,lam=0) u_i, q_lam[i] = u_i^T K(0,1) u_i,
 * q_m[i] = u_i^T M u_i; replaces the matrix-free stiff_func path
 * (diff_model.py:314-328, 371-388; deform.py:70-87, 149-165).  wsum = sum of the
 * reference's fp32 Gauss weights (used by linear tets only).  out fp64 [3*k];
 * partial scratch fp64 [ds_quadform_scratch_elems(k)]. */
int64_t ds_quadform_scratch_elems(int k);
int ds_eigval_quadforms_material(const float* verts, const int32_t* tets, int64_t T, int order,
                                 const double* mtab, double wsum, const double* U, int64_t ldu, int k,
                                 double* partial, double* out, void* stream);

/* ---- modal synthesis --------------------------------------------------------
 * y[b,t] = sum_m a[b,m] exp(-d[m] (t+1)/sr) sin(2 pi f[m] (t+1)/sr); replaces the
 * cumsum/exp/sin/sum chain of oscillator.py:297-304 (and :128-138, :160-171).
 * amp fp32 [B*k]; damp, freq fp32 [k] (shared over the batch) ; y fp32 [B*T].
 * Backward: gy [B*T] -> gamp [B*k], gdamp [k], gfreq [k]. */
int64_t ds_synth_scratch_elems(int64_t B, int k, int64_t T);
int ds_modal_synth_fwd(const float* amp, const float* damp, const float* freq, int64_t B, int k,
                       int64_t T, double sr, float* y, float* scratch, void* stream);
int ds_modal_synth_bwd(const float* amp, const float* damp, const float* freq, const float* gy,
                       int64_t B, int k, int64_t T, double sr, float* gamp, float* gdamp,
                       float* gfreq, float* scratch, void* stream);
/* Causal force FIR on the rendered audio, replacing F.conv1d(signal, flipped force, groups=audio_num,
 * padding=F-1)[..., :T] of the oscillators (ddsp/oscillator.py:305-309, 139-141, 172-174, 239-241).
 * x, out: fp32 [B x T]; force: fp32 [B x F] in natural (un-flipped) order, F <= 2048.
 * reverse = 0: out[b,t] = sum_i force[b,i] x[b,t-i];  reverse = 1 (adjoint, the backward pass w.r.t. x):
 * out[b,t] = sum_i force[b,i] x[b,t+i]. */
int ds_force_fir(const float* x, const float* force, int64_t B, int64_t T, int F, int reverse, float* out,
                 void* stream);

/* ---- filtered noise (the noise branch of GTDampedOscillator) ---------------------------------
 * Replaces FilteredNoise.forward (ddsp/filtered_noise.py:20-67: irfft of a zero-phase response, roll,
 * Hann window, FFT convolution with uniform noise frames, overlap-add by conv_transpose1d), added to
 * the modal signal as `noise * noise_rate` (ddsp/oscillator.py:226,243; material_real_train.py:118).
 * coeff: fp32 [B x F x C] raw coefficient_bank parameters (the modified sigmoid is applied inside);
 * noise: fp32 [B x F x L] uniform(-1, 1) frames drawn by the caller (the reference draws them with
 * torch.rand on the host generator); y: fp32 [B x T], F * L >= T.  C = filter_coeff_length <= 129,
 * L = frame_length <= 256.  Backward: gy [B x T] -> gcoeff [B x F x C]. */
int ds_filtered_noise_fwd(const float* coeff, const float* noise, int64_t B, int F, int C, int L, int64_t T,
                          double gain, float* y, void* stream);
int ds_filtered_noise_bwd(const float* coeff, const float* noise, const float* gy, int64_t B, int F, int C, int L,
                          int64_t T, double gain, float* gcoeff, void* stream);

/* ---- multi-scale spectral loss (one scale per call) ------------------------------------------
 * Replaces SSSLoss (ddsp/mss_loss.py:70-121) on torchaudio.transforms.Spectrogram(n_fft, hop): periodic Hann
 * window of n_fft, center = True / reflect padding, power 2, one-sided; frames = 1 + T / hop.
 * ds_stft_power: S fp32 [B x (n_fft/2+1) x frames] (SSSLoss.spec / log_spec).
 * ds_mss_loss_fwd: mode 0 = 'l1_loss' (alpha * weighted L1 of log2(S + eps) + weighted L1 of S, DC bin dropped,
 * mss_loss.py:55-66,101-106), mode 1 = 'rmse_loss' (mss_loss.py:116-119).  x_pred, x_true: fp32 [B x T];
 * scratch: fp32 [ds_mss_scratch_elems], 8-byte aligned; loss: one double on the device.
 * ds_mss_loss_bwd: d(upstream * loss)/d x_pred into gx [B x T] (accumulate != 0: added to gx); `loss` is the
 * forward result (needed by the RMSE chain rule).  No spectrogram is materialised by the loss calls. */
int ds_stft_frames(int64_t T, int hop);
int ds_stft_power(const float* x, int64_t B, int64_t T, int n_fft, int hop, float* S, void* stream);
int64_t ds_mss_scratch_elems(int64_t B, int64_t T, int n_fft, int hop);
int ds_mss_loss_fwd(const float* x_pred, const float* x_true, int64_t B, int64_t T, int n_fft, int hop, int mode,
                    double alpha, double eps, float* scratch, double* loss, void* stream);
int ds_mss_loss_bwd(const float* x_pred, const float* x_true, int64_t B, int64_t T, int n_fft, int hop, int mode,
                    double alpha, double eps, const double* loss, double upstream, float* scratch, float* gx,
                    int accumulate, void* stream);

/* ---- pieces of a row-partitioned LOBPCG step (csrc/slab.cu; host driver diffsound_b200/parallel/rowpart_lobpcg.py) -------
 * One large mesh on several GPUs (SURVEY.md section 8e): rank r owns a contiguous slab of node rows.  These are the kernels
 * of the single-GPU driver (ds_lobpcg) as stand-alone calls on a slab; the exchanges between them (all-reduce of Gram strips,
 * residual sums and partial coarse residuals, all-gather of the new fp32 search block) are NCCL collectives issued by the host.
 * ds_lobpcg_residual: R = KX - MX diag(lam) (n x m) and sums[2m] = column sums of R^2 | MX^2; partial: 296 * 2m doubles.
 * ds_gather_cols_f32: dst (n x width, fp32) = src[:, cols_host[0..count)] (zero padded); ds_widen_f32: fp32 -> fp64 block.
 * ds_jacobi32: Out = cc invD R (first Chebyshev step from zero).  ds_spmm_dual_z32: YK = K Z, YM = M Z for the rows of a
 * slab (brow local, bcolP = column ids as ROW INDICES OF Z, chunk_row from ds_spmm32_chunks) with Z an fp32 block (ld = ncols).
 * ds_pmg_restrict32_range: rc = 0.5 sum of the gather lists restricted to the fine nodes [fine_lo, fine_hi) (res_local holds
 * exactly those rows): a partial coarse residual, summed over ranks by the caller.  ds_pmg_prolong64: x_i = 0.5 (xc[p0] + xc[p1]).
 * ds_gram_insert_f64 / ds_sym_upper_f64: rows and columns [m, 2m) of the Gram pair from the strips / mirror the upper triangle.
 * ds_eigh_generalized_idx_f64: ds_eigh_generalized_f64 on the slots idx_host[0..N) of the ldg x ldg Gram storage. */
int ds_lobpcg_residual(const double* KX, const double* MX, int64_t ld, int m, int64_t n, const double* lam, double* R, int64_t ldr,
                       double* sums, double* partial, void* stream);
int ds_gather_cols_f32(const double* src, int64_t lds, const int* cols_host, int count, int width, int64_t n, float* dst, void* stream);
int ds_widen_f32(const float* src, int width, int64_t n, double* dst, int64_t ldd, void* stream);
int ds_jacobi32(const float* invD, const float* R, int64_t n_nodes, int ncols, double cc, float* Out, void* stream);
int ds_spmm_dual_z32(const int32_t* brow, const int32_t* bcolP, int64_t n_rows, int64_t nnzb, const int32_t* chunk_row,
                     const double* Kval, const double* Mblk, const float* Z, int ncols, double* YK, int64_t ldyk, double* YM,
                     int64_t ldym, void* stream);
int ds_pmg_restrict32_range(const int32_t* rptr, const int32_t* rlist, int64_t n_coarse, const float* res_local, int ncols,
                            int64_t fine_lo, int64_t fine_hi, float* rc, void* stream);
int ds_pmg_prolong64(const int32_t* parents, int64_t n_fine, const double* xc, int64_t ldc, int w, double* x, int64_t ldx, void* stream);
int ds_gram_insert_f64(double* GK, double* GM, int64_t ldg, const double* GsK, const double* GsM, int64_t lds, int m, int wa, void* stream);
int ds_sym_upper_f64(double* GK, double* GM, int64_t ldg, int N, void* stream);
int ds_eigh_generalized_idx_f64(const double* GK, const double* GM, int N, int64_t ldg, const int* idx_host, double sigma,
                                double* theta, double* C, int64_t ldc, double* scratch, int* info, void* stream);

/* ---- marching tetrahedra -> tet mesh of a hollow shell, compaction, largest connected component ----------------
 * Replaces DMTet.__call__ and DMTetGeometry.get_largest_connected_component (src/dmtet/geometry/dmtet_thickness.py:99-200,
 * :254-285; the same code in dmtet_interpolate.py:115-205,265-296 and dmtet_geometry.py:115-267,411-443): torch.unique
 * sorts + mask gathers + a GPU -> CPU round trip through scipy.sparse.csgraph.connected_components.  Output order and
 * numbering are the reference's bit for bit (they define the sparsity pattern downstream); see csrc/mtet.cu.
 * sdf: fp32 [n_verts]; tets: int64 [F x 4]; a vertex is inside the shell when 0 < sdf <= (float)thickness.
 * ds_mtet_count -> counts_host[7] = {valid tets, unique edges, crossing edges, one-tet tets, three-tet tets, inner tets,
 * surface triangles}; ds_mtet_fill -> interp_v int64 [crossing x 2] (end points a < b of every crossing edge, ascending;
 * edge e becomes vertex n_verts + e), tets_out int64 [(one + 3 three + inner) x 4] over ids in [0, n_verts + crossing),
 * faces_out int64 [triangles x 3] over edge-vertex ids (may be NULL).
 * ds_compact_ids_*: ascending unique values of ids[M] (all in [0, R)) and each id's rank among them
 * (torch.unique(return_inverse=True) of dmtet_thickness.py:195-199).
 * ds_tet_components_*: labels int32 [n_verts] = smallest vertex id of the vertex's component; counts_host[3] = {components,
 * vertices, tets of the largest component (ties: the component with the smallest vertex id, the one SciPy labels
 * first)}; fill -> kept_verts int64 [vertices] (old ids, ascending), tets_out int64 [tets x 4] renumbered, order kept. */
int ds_mtet_count(ds_workspace* ws, const float* sdf, double thickness, const int64_t* tets, int64_t F, int64_t n_verts,
                  int64_t* counts_host, void* stream);
int ds_mtet_fill(ds_workspace* ws, const int64_t* tets, int64_t* interp_v, int64_t* tets_out, int64_t* faces_out, void* stream);
int ds_compact_ids_count(ds_workspace* ws, const int64_t* ids, int64_t M, int64_t R, int64_t* n_unique_host, void* stream);
int ds_compact_ids_fill(ds_workspace* ws, const int64_t* ids, int64_t* unique_out, int64_t* inverse_out, void* stream);
int ds_tet_components_count(ds_workspace* ws, const int64_t* tets, int64_t T, int64_t n_verts, int32_t* labels,
                            int64_t* counts_host, void* stream);
int ds_tet_components_fill(ds_workspace* ws, const int64_t* tets, int64_t* kept_verts, int64_t* tets_out, void* stream);

/* ---- signed distance from points to a triangle mesh ---------------------------------------------------------------
 * Replaces the open3d RaycastingScene sampling of DMTetGeometry.apply_sdf(path) (src/dmtet/geometry/dmtet_thickness.py:
 * 301-314, whose compute_signed_distance is negated there): sdf_out[i] = +d inside, -d outside, with d the fp64 distance
 * from points[i] to the closest point of the triangle set rounded once to fp32 (degenerate faces count as their edges;
 * a point on the surface gives +0), inside = odd number of crossings for at least two of three fixed rays (watertight
 * ray / triangle test, face orientation does not matter).  The mesh is used in its own coordinates.
 * tri_verts fp32 [V x 3], faces int64 [F x 3], points fp32 [P x 3], sdf_out fp32 [P]; see csrc/sdf.cu.
 * mode 0 = BVH, 1 = brute force (test reference; both give bitwise equal outputs).  Synchronises once: face indices
 * outside [0, V) and non-finite coordinates return DS_ERR_ARG with a message, never a fault; so do V == 0, F == 0, a
 * null pointer and an unknown mode.  P == 0 returns 0 without doing any work. */
int ds_mesh_sdf(ds_workspace* ws, const float* tri_verts, int64_t V, const int64_t* faces, int64_t F, const float* points,
                int64_t P, int mode, float* sdf_out, void* stream);
/* ds_mesh_sdf, and face_out int32 [P] = the face nearest to each point (an index into faces; of several faces at exactly
 * the same fp64 squared distance, the lowest index, in both modes, so BVH and brute force give bitwise equal ids).
 * sdf_out is bitwise equal to ds_mesh_sdf's.  Same checks and synchronisation as ds_mesh_sdf. */
int ds_mesh_sdf_nearest(ds_workspace* ws, const float* tri_verts, int64_t V, const int64_t* faces, int64_t F,
                        const float* points, int64_t P, int mode, float* sdf_out, int32_t* face_out, void* stream);
/* Gradient of ds_mesh_sdf: with c = sum_k b_k v_k the closest point of face[i] to points[i] (the forward's region
 * analysis; degenerate faces: the nearest edge), u = (p - c) / |p - c| and s = sign(sdf[i]):
 *   grad_points[i] = grad_sdf[i] s u;   grad_verts[v] = sum over points i and corners k of face[i] with vertex id v of
 *   -grad_sdf[i] s b_k u.
 * Zero where sdf[i] == 0 or |p - c| == 0.  fp64 throughout, rounded once to fp32; grad_verts is summed in ascending
 * (point, corner) order without atomics, so the result is bitwise reproducible.  face int32 [P] and sdf fp32 [P] as
 * ds_mesh_sdf_nearest returned them, grad_sdf fp32 [P], grad_verts fp32 [V x 3], grad_points fp32 [P x 3]; either output
 * may be NULL.  Synchronises once: the checks of ds_mesh_sdf, and a nearest-face id outside [0, F) returns DS_ERR_ARG. */
int ds_mesh_sdf_backward(ds_workspace* ws, const float* tri_verts, int64_t V, const int64_t* faces, int64_t F,
                         const float* points, int64_t P, const int32_t* face, const float* sdf, const float* grad_sdf,
                         float* grad_verts, float* grad_points, void* stream);
/* Generalised winding number w(p) = sum over faces of the oriented solid angle / 4 pi (Jacobson, Kavan & Sorkine-Hornung
 * 2013): 1 inside and 0 outside a closed surface whose faces are consistently oriented with outward normals (-1 / 0 when
 * they all point inward), 2 where two such surfaces overlap, and a smooth value between across holes.  Degenerate faces
 * contribute 0.  w_out fp32 [P].  mode 1 = exact: the fp64 sum over all faces in face order (Van Oosterom-Strackee solid
 * angles), rounded once.  mode 0 = BVH over the faces (a radix tree on the centroids of the sorted corners), with subtrees
 * far from the point replaced by their far-field expansion (Barill et al. 2018, through the first moment, acceptance
 * |p - centroid| > 3 x the subtree's radius).  Its error is measured, not bounded: at most 0.024 on the test meshes, whose
 * bar is 0.05; it grows with the face area packed inside a subtree (many stacked or crumpled layers).  Both modes are
 * bitwise reproducible; flipping every face gives exactly -w, and neither the first corner written nor vertex sharing
 * changes the result.  Same checks and synchronisation as ds_mesh_sdf. */
int ds_mesh_winding_number(ds_workspace* ws, const float* tri_verts, int64_t V, const int64_t* faces, int64_t F,
                           const float* points, int64_t P, int mode, float* w_out, void* stream);
/* ds_mesh_sdf with the sign of the winding number: inside (+) where |w| >= 1/2 (decided in fp64 from the w of
 * ds_mesh_winding_number in the same mode), so the overlap of a self-intersecting surface stays inside and holes do not
 * streak the sign.  Needs consistently oriented faces (either way round); for inconsistently oriented meshes the ray
 * parity of ds_mesh_sdf is the right rule.  |sdf_out| and face_out are bitwise those of ds_mesh_sdf_nearest (same
 * search, tie rule and ids), a point at distance 0 gives +0.  face_out int32 [P] may be NULL.  Same checks and
 * synchronisation as ds_mesh_sdf. */
int ds_mesh_sdf_winding(ds_workspace* ws, const float* tri_verts, int64_t V, const int64_t* faces, int64_t F,
                        const float* points, int64_t P, int mode, float* sdf_out, int32_t* face_out, void* stream);

/* ---- device-side timing per kernel class ---------------------------------------
 * Replaces the reference's opt-in torch.profiler hook of lobpcg (src/lobpcg/_lobpcg.py:357-369)
 * and the TICK/TOCK macros (src/include/macro.h:31-44): CUDA events around every launch site,
 * accumulated per class ("spmm", "cheb_step", "gram", ...).  Off by default.  ds_prof_read
 * synchronises on the recorded events. */
int ds_prof_enable(int on);
/* create n timing events up front (event creation inside a timed region can stall on a driver allocation) */
int ds_prof_reserve(int n);
/* time only the classes whose bit (1 << class index, see ds_prof_class_name) is set; 0 turns timing off */
int ds_prof_enable_classes(uint32_t mask);
int ds_prof_reset(void);
int ds_prof_num_classes(void);
/* kernels launched by this library in this process so far (cub and memcpy/memset excluded) */
int64_t ds_launch_count(void);
const char* ds_prof_class_name(int cls);
int ds_prof_read(int cls, double* ms, int64_t* count);
/* algorithmic bytes and flops accounted by the launch sites of the class while it was being timed */
int ds_prof_read_work(int cls, double* bytes, double* flops);

/* ---- Rayleigh-Ritz pieces of the round-2 LOBPCG step (csrc/rr.cu; replaces the full Gram products and the basis
 * update of lobpcg/_lobpcg.py:433-525).  All blocks fp64 row-major, 16-byte aligned, even leading dimensions.
 * ds_gram_strip_f64:  GsK[wa x ncol] = KW^T S, GsM = MW^T S (KW, MW: n x wa, wa in {16,32,48}; S: n x ncol <= 144).
 * ds_rr_update2_f64:  for A in {S, KS, MS} (n x 3m, columns [X | W | P]):  P' = A[:, m:m+wa] C[m:m+wa, :m]
 *                     (+ A[:, 2m:3m] C[2m:3m, :m] when use_p);  A_out[:, 2m:3m] = P';  A_out[:, :m] = P' + A[:, :m] C[:m, :m].
 * ds_gram_algebra_f64: Gram pair of [X' | . | P'] from the Gram pair G of [X | W | P] (full symmetric, ldg x ldg),
 *                     the coefficient matrix C (rows = slots, columns = rank) and the Ritz values theta.
 * ds_fp64_peak: register-resident FP64 throughput of this device, mode 0 = DFMA, 1 = DMMA m8n8k4 (TFLOP/s). */
int64_t ds_gram_strip_scratch_elems(void);
int ds_gram_strip_f64(const double* KW, const double* MW, int64_t ldw, int wa, const double* S, int64_t lds, int ncol,
                      int64_t n, double* GsK, double* GsM, int64_t ldg, double* partial, void* stream);
int ds_rr_update2_f64(const double* S, const double* KS, const double* MS, int64_t lda, int m, int wa, int use_p,
                      const double* C, int64_t ldc, int64_t n, double* S_out, double* KS_out, double* MS_out, int64_t ldy,
                      void* stream);
int64_t ds_gram_algebra_scratch_elems(void);
int ds_gram_algebra_f64(const double* GK, const double* GM, double* GKn, double* GMn, int64_t ldg, const double* C,
                        int64_t ldc, const double* theta, int m, double* scratch, void* stream);
int ds_fp64_peak(int mode, int iters, int ctas_per_sm, double* scratch, double* tflops_host, void* stream);

#ifdef __cplusplus
}
#endif
#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#endif /* DIFFSOUND_SM100_H */

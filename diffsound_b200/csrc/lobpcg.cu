// Device-resident LOBPCG for K u = lambda M u (lowest pairs), FP64.
//
// Reference behaviour replaced: DiffSoundObj.eigen_decomposition_arpack
// (/root/reference/src/diffelastic/diff_model.py:335-369 -- scipy eigsh shift-invert on
// the CPU after a device->host copy of K and M) and the LOBPCG worker behind
// lobpcg / lobpcg_func (/root/reference/src/lobpcg/_lobpcg.py:214-679).  The iteration
// is the classical [X, W, P] scheme with soft locking:
//   R = K X - M X diag(lam);  W = T R (active columns only), M-orthogonalised against X;
//   Rayleigh-Ritz on span[X, W, P];  X, P updated from the Ritz vectors.
// T ~ K^-1 is evaluated in FP32 (csrc/precond32.cu): either `cheb_degree` steps of
// block-Jacobi-scaled Chebyshev iteration on K (+ sigma M), or -- when the caller supplies the
// P1 operator of a quadratic mesh (ds_pmg_level) -- a symmetric two-level V-cycle: Chebyshev
// smoothing on the P2 operator around a Chebyshev solve on the 15x smaller P1 operator.  Either
// way T is a fixed SPD polynomial in the SpMM kernel, so the eigen-solve is a stream of SpMM
// (HBM-bound) + DMMA Gram/GEMM kernels + one single-CTA Jacobi per step.
//
// Clamped nodes (ds_lobpcg_opts.fixed, csrc/fixed.cu): K and M arrive constrained, and the rows of the fixed nodes are
// zeroed in the start block (after the nested start's prolongation) and in every preconditioner output, one masking
// launch each.  X, W and P then stay exactly zero there, so the iteration is the one of the reduced problem.
//
// Storage: three wide row-major buffers S, KS, MS of n x 3m (columns [X | W | P]) plus a
// ping-pong copy, so the Ritz update is one tall-skinny GEMM per buffer.
#include "common.cuh"
#include "../../include/diffsound_sm100.h"
#include "kernels.cuh"
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <vector>

namespace ds {

// R = KX - MX * lam  (n x m, leading dims given); per-CTA partial sums of R^2 and MX^2 per column.
__global__ void k_residual(const double* __restrict__ KX, const double* __restrict__ MX, int64_t ld, int m, int64_t n,
                           const double* __restrict__ lam, double* __restrict__ R, int64_t ldr,
                           double* __restrict__ partial) {
    extern __shared__ double sh[];   // [rows_per_pass][2m]
    const int rpp = blockDim.x / m;  // rows per pass
    const int c = threadIdx.x % m, rr = threadIdx.x / m;
    double l = lam[c];
    double s_r = 0.0, s_m = 0.0;
    if (rr < rpp) {
        for (int64_t row = (int64_t)blockIdx.x * rpp + rr; row < n; row += (int64_t)gridDim.x * rpp) {
            double kx = KX[row * ld + c], mx = MX[row * ld + c];
            double r = kx - l * mx;
            R[row * ldr + c] = r;
            s_r = fma(r, r, s_r);
            s_m = fma(mx, mx, s_m);
        }
        sh[(rr * 2 + 0) * m + c] = s_r;
        sh[(rr * 2 + 1) * m + c] = s_m;
    }
    __syncthreads();
    if (threadIdx.x < 2 * m) {
        int which = threadIdx.x / m, cc = threadIdx.x % m;
        double s = 0.0;
        for (int r2 = 0; r2 < rpp; ++r2) s += sh[(r2 * 2 + which) * m + cc];
        partial[(size_t)blockIdx.x * 2 * m + threadIdx.x] = s;
    }
}

// out[t] = sum over the per-CTA partials of column t: one WARP per column (lane l adds partials l, l + 32, ... in order, the
// 32 lane sums meet in a fixed butterfly: deterministic).  One thread per column took 30 us for 296 partials -- a
// latency-bound chain that ran 34 times per modal solve.
__global__ void __launch_bounds__(256) k_colsum_reduce(const double* __restrict__ partial, int nparts, int width,
                                                       double* __restrict__ out) {
    const int t = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (t >= width) return;
    double s = 0.0;
    for (int p = lane; p < nparts; p += 32) s += partial[(size_t)p * width + t];
    s = warp_sum(s);
    if (lane == 0) out[t] = s;
}
static inline unsigned colsum_blocks(int width) { return (unsigned)((width * 32 + 255) / 256); }

// per-column sum of squares of a block (n x w, ld)
__global__ void k_colnorm2(const double* __restrict__ V, int64_t ld, int w, int64_t n, double* __restrict__ partial) {
    extern __shared__ double sh[];
    const int rpp = blockDim.x / w;
    const int c = threadIdx.x % w, rr = threadIdx.x / w;
    double s = 0.0;
    if (rr < rpp) {
        for (int64_t row = (int64_t)blockIdx.x * rpp + rr; row < n; row += (int64_t)gridDim.x * rpp) {
            double v = V[row * ld + c];
            s = fma(v, v, s);
        }
        sh[rr * w + c] = s;
    }
    __syncthreads();
    if (threadIdx.x < w) {
        double t = 0.0;
        for (int r2 = 0; r2 < rpp; ++r2) t += sh[r2 * w + threadIdx.x];
        partial[(size_t)blockIdx.x * w + threadIdx.x] = t;
    }
}

// partial[cta][s] = sum over rows of R[row, idx[s]] * W[row, s]  (s < count): r_j^T T r_j, the preconditioned (energy) norm
// of the residual of active column idx[s], whose search direction W[:, s] = T r_j has just been computed
__global__ void k_coldot_rw(const double* __restrict__ R, int64_t ldr, const __grid_constant__ ColIdx idx, int count,
                            const double* __restrict__ W, int64_t ldw, int64_t n, double* __restrict__ partial) {
    extern __shared__ double sh[];
    const int w = count, rpp = blockDim.x / w;
    const int c = threadIdx.x % w, rr = threadIdx.x / w;
    double s = 0.0;
    if (rr < rpp) {
        const int rc = idx.v[c];
        for (int64_t row = (int64_t)blockIdx.x * rpp + rr; row < n; row += (int64_t)gridDim.x * rpp)
            s = fma(R[row * ldr + rc], W[row * ldw + c], s);
        sh[rr * w + c] = s;
    }
    __syncthreads();
    if (threadIdx.x < w) {
        double t = 0.0;
        for (int r2 = 0; r2 < rpp; ++r2) t += sh[r2 * w + threadIdx.x];
        partial[(size_t)blockIdx.x * w + threadIdx.x] = t;
    }
}

// dst[:, s] = src[:, idx[s]] for s < count, zero for count <= s < width
__global__ void k_gather_cols(const double* __restrict__ src, int64_t lds, const __grid_constant__ ColIdx idx,
                              int count, int width, int64_t n, double* __restrict__ dst, int64_t ldd) {
    int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= n * width) return;
    int64_t row = t / width;
    int s = (int)(t - row * width);
    dst[row * ldd + s] = s < count ? src[row * lds + idx.v[s]] : 0.0;
}

__global__ void k_fill_random(double* __restrict__ V, int64_t count, uint64_t seed) {
    int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= count) return;
    uint64_t z = seed + 0x9E3779B97F4A7C15ull * (uint64_t)(t + 1);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    z ^= z >> 31;
    V[t] = (double)(z >> 11) * (2.0 / 9007199254740992.0) - 1.0;
}

// ---- FP64 fall-back preconditioner (ds_lobpcg_opts.precond_fp64): block-Jacobi Chebyshev on K in double precision.
// The FP32 cycle loses the smooth part of a residual whose stiff components are >= 1e7 times larger (sliver elements of
// marching-tets meshes: r = K x - lam M x amplifies the rounding noise of x along modes with lam_stiff / lam ~ 1e10);
// the same polynomial in FP64 does not.  One SpMM (k_spmm) + one update kernel per step.
__global__ void k_invd64(const int32_t* __restrict__ brow, const int32_t* __restrict__ bcol, int64_t n_nodes,
                         const double* __restrict__ Kval, double* __restrict__ invD) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n_nodes) return;
    const int64_t b0 = brow[i];
    const int deg = (int)(brow[i + 1] - b0);
    int p = 0;
    while (p < deg && bcol[b0 + p] != (int32_t)i) ++p;
    double k[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
    if (p < deg)
        for (int c = 0; c < 3; ++c)
            for (int d = 0; d < 3; ++d) k[3 * c + d] = Kval[9 * b0 + (int64_t)c * 3 * deg + 3 * p + d];
    const double c00 = k[4] * k[8] - k[5] * k[7], c01 = k[5] * k[6] - k[3] * k[8], c02 = k[3] * k[7] - k[4] * k[6];
    const double id = 1.0 / (k[0] * c00 + k[1] * c01 + k[2] * c02);
    double* o = invD + 9 * i;
    o[0] = c00 * id; o[1] = (k[2] * k[7] - k[1] * k[8]) * id; o[2] = (k[1] * k[5] - k[2] * k[4]) * id;
    o[3] = c01 * id; o[4] = (k[0] * k[8] - k[2] * k[6]) * id; o[5] = (k[2] * k[3] - k[0] * k[5]) * id;
    o[6] = c02 * id; o[7] = (k[1] * k[6] - k[0] * k[7]) * id; o[8] = (k[0] * k[4] - k[1] * k[3]) * id;
}

// Znew = Z + ab (Z - Zp) + cc invD Res   (per node: 3 rows x w columns; Zp may alias Znew; Z == NULL: Znew = cc invD Res)
__global__ void k_cheb64_update(const double* __restrict__ invD, const double* __restrict__ Res, int64_t ldr,
                                const double* __restrict__ Z, const double* Zp, double* Znew, int64_t ldz, int64_t n_nodes,
                                int w, double ab, double cc) {
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= n_nodes * w) return;
    const int64_t i = t / w;
    const int c = (int)(t - i * w);
    const double* d = invD + 9 * i;
    const double r0 = Res[(3 * i) * ldr + c], r1 = Res[(3 * i + 1) * ldr + c], r2 = Res[(3 * i + 2) * ldr + c];
#pragma unroll
    for (int q = 0; q < 3; ++q) {
        const double dr = d[3 * q] * r0 + d[3 * q + 1] * r1 + d[3 * q + 2] * r2;
        const int64_t o = (3 * i + q) * ldz + c;
        double v = cc * dr;
        if (Z) { const double z = Z[o]; v += z + ab * (z - Zp[o]); }
        Znew[o] = v;
    }
}

__global__ void k_gather_cols64(const double* __restrict__ src, int64_t lds, const __grid_constant__ ColIdx idx, int count,
                                int width, int64_t n, double* __restrict__ dst) {
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= n * width) return;
    const int64_t row = t / width;
    const int s = (int)(t - row * width);
    dst[t] = s < count ? src[row * lds + idx.v[s]] : 0.0;
}

struct Driver {
    ds_workspace* ws;
    cudaStream_t st;
    const int32_t *brow, *bcol;
    int64_t n_nodes, n;
    const double *Kval, *Mblk;
    int m;
    ds_lobpcg_opts o;

    const ds_pmg_level* cl = nullptr;   // optional coarse (P1) level
    int fine_prof_cls = PROF_CHEB;      // timing class of this driver's own level (the nested coarse solve reports as coarse)
    Level32 fine, coarse;
    float *R32, *Za, *Zb, *RC32, *ZCa, *ZCb;
    double *Xc = nullptr, *lamc = nullptr, *resc = nullptr;    // nested coarse eigen-solve
    double *invD64 = nullptr, *R64 = nullptr, *Z64a = nullptr, *Z64b = nullptr, *RES64 = nullptr;   // FP64 preconditioner
    const double* Q = nullptr;   // locked (already converged, M-orthonormal) eigenvectors, n x nq, ld = nq
    int nq = 0;
    double* MQ = nullptr;        // M Q
    int64_t nested_iters = 0, nested_status = 0;
    double child_lmax = 0.0;     // spectral-radius estimate of the nested solve's fine level = this solve's coarse level

    int ld;                      // 3m
    double *S[2], *KS[2], *MS[2];
    double *R;
    double *GK, *GM, *Cm, *theta, *eig_scratch, *gram_partial, *gram_partial2, *norm_partial, *norms, *lam_d, *lmax_samples = nullptr;
    double *GKn = nullptr, *GMn = nullptr, *GsK = nullptr, *GsM = nullptr, *strip_partial = nullptr, *alg_scratch = nullptr;   // Gram recurrences (rr.cu)
    int* info_d;
    int cur = 0;
    int64_t spmm_count = 0;
    int norm_ctas = 296;

    int alloc() {
        ld = 3 * m;
        size_t blk = (size_t)n * m;
        size_t need = 0;
        auto add = [&](size_t elems) { need += ((elems * 8 + 255) & ~size_t(255)) + 256; };
        for (int i = 0; i < 6; ++i) add(3 * blk);
        add(blk);
        const int64_t nnzb = nnzb_of(brow, n_nodes);
        if (nnzb < 0) return DS_ERR_CUDA;
        need += Level32::bytes(n_nodes, nnzb);
        for (int i = 0; i < 3; ++i) add(blk / 2 + 64);
        int64_t nnzb_c = 0;
        if (cl) {
            nnzb_c = cl->nnzb;
            need += Level32::bytes(cl->n_nodes, nnzb_c);
            for (int i = 0; i < 3; ++i) add((size_t)3 * cl->n_nodes * m / 2 + 64);
            if (o.nested && cl->Mblk) { add((size_t)3 * cl->n_nodes * m); add(128); add(128); }
        }
        add(144 * 144); add(144 * 144); add(144 * 144); add(144); add((size_t)eigh_scratch_elems(144));
        add((size_t)gram_scratch_elems(64, 64)); add((size_t)norm_ctas * 2 * 128); add(2 * 128); add(128);
        add((size_t)gram_sym2_scratch_elems(ws->num_sms));
        add(64); add(128);
        for (int i = 0; i < 4; ++i) add(144 * 144);
        add((size_t)gram_strip_scratch_elems(ws->num_sms));
        add((size_t)gram_algebra_scratch_elems());
        if (nq) add((size_t)n * nq);
        if (o.precond_fp64) { add((size_t)n_nodes * 9); for (int i = 0; i < 4; ++i) add(blk); }
        DS_TRY(ws->arena.reserve(need, st));
        Arena& a = ws->arena;
        for (int i = 0; i < 2; ++i) {
            S[i] = a.take<double>(3 * blk);
            KS[i] = a.take<double>(3 * blk);
            MS[i] = a.take<double>(3 * blk);
        }
        R = a.take<double>(blk);
        R32 = a.take<float>(blk); Za = a.take<float>(blk); Zb = a.take<float>(blk);
        RC32 = ZCa = ZCb = nullptr;
        if (cl) {
            const size_t cb = (size_t)3 * cl->n_nodes * m;
            RC32 = a.take<float>(cb); ZCa = a.take<float>(cb); ZCb = a.take<float>(cb);
            if (o.nested && cl->Mblk) {
                Xc = a.take<double>(cb); lamc = a.take<double>(128); resc = a.take<double>(128);
            }
        }
        GK = a.take<double>(144 * 144); GM = a.take<double>(144 * 144); Cm = a.take<double>(144 * 144);
        theta = a.take<double>(144); eig_scratch = a.take<double>((size_t)eigh_scratch_elems(144));
        gram_partial = a.take<double>((size_t)gram_scratch_elems(64, 64));
        gram_partial2 = a.take<double>((size_t)gram_sym2_scratch_elems(ws->num_sms));
        norm_partial = a.take<double>((size_t)norm_ctas * 2 * 128);
        norms = a.take<double>(2 * 128);
        lam_d = a.take<double>(128);
        info_d = a.take<int>(16);
        lmax_samples = a.take<double>(2 * (LMAX_STEPS0 / 4) * LMAX_W);
        GKn = a.take<double>(144 * 144); GMn = a.take<double>(144 * 144);
        GsK = a.take<double>(144 * 144); GsM = a.take<double>(144 * 144);
        strip_partial = a.take<double>((size_t)gram_strip_scratch_elems(ws->num_sms));
        alg_scratch = a.take<double>((size_t)gram_algebra_scratch_elems());
        if (nq) MQ = a.take<double>((size_t)n * nq);
        if (o.precond_fp64) {
            invD64 = a.take<double>((size_t)n_nodes * 9);
            R64 = a.take<double>(blk); Z64a = a.take<double>(blk); Z64b = a.take<double>(blk); RES64 = a.take<double>(blk);
            DS_REQUIRE(RES64 != nullptr, "lobpcg: workspace arena exhausted");
        }
        DS_REQUIRE(info_d != nullptr && strip_partial != nullptr && alg_scratch != nullptr && (!nq || MQ), "lobpcg: workspace arena exhausted");
        // Never multiply uninitialised memory by zero coefficients: k_gram_strip reads ALL 3m columns of S (unused W / P
        // slots included; their products land in Gram entries that the small-matrix recurrences later multiply by zero
        // rows of C), so S starts finite.  KS / MS are only ever read at slots that were written (k_residual: X;
        // k_rr_update2: X, W[:wa], P when in use; k_gram_sym2: active tiles), so they need no 1.9 GB of memsets each.
        for (int i = 0; i < 2; ++i) DS_CUDA(cudaMemsetAsync(S[i], 0, 3 * blk * 8, st));
        // FP32 copies of the operators (records + block-Jacobi inverses)
        fine.want_bcolP = true;       // K W / M W are formed from the fp32 preconditioner output (k_spmm_dual_z32)
        DS_TRY(fine.setup(a, brow, bcol, n_nodes, nnzb, Kval, Mblk, o.sigma > 0.0 ? o.sigma : 0.0, o.coords, st));
        fine.prof_cls = fine_prof_cls;
        if (cl) {
            DS_TRY(coarse.setup(a, cl->brow, cl->bcol, cl->n_nodes, nnzb_c, cl->Kval, cl->Mblk,
                                o.sigma > 0.0 ? o.sigma : 0.0, cl->coords, st));
            coarse.prof_cls = PROF_COARSE;
        }
        return DS_OK;
    }

    static int64_t nnzb_of(const int32_t* brow, int64_t n_nodes) {
        int32_t v = 0;
        if (cudaMemcpy(&v, brow + n_nodes, sizeof(int32_t), cudaMemcpyDeviceToHost) != cudaSuccess) {
            set_error("ds_lobpcg: cannot read brow[n_nodes]");
            return -1;
        }
        return v;
    }

    // V (n x w, ld = ldv) <- V - Q (MQ^T V): keeps the iteration M-orthogonal to the locked eigenvectors
    int project_locked(double* V, int64_t ldv, int w) {
        for (int c0 = 0; c0 < nq; c0 += 48) {
            const int wc = std::min(48, nq - c0);
            DS_TRY(gram_f64(MQ + c0, nq, wc, V, ldv, w, n, GK, 144, gram_partial, st));
            DS_TRY(block_gemm_f64(Q + c0, nq, wc, GK, 144, w, n, -1.0, 1.0, V, ldv, st));
        }
        return DS_OK;
    }

    double* Xb(int w) { return S[w]; }
    double* Wb(int w) { return S[w] + m; }
    double* Pb(int w) { return S[w] + 2 * m; }

    // G[off_a.., off_b..] (144-ld storage) = A^T B over blocks of width <= 48 (gram limit 64)
    int gram_block(const double* A, int wa, const double* B, int wb, double* G, int ra, int cb) {
        if (wa == 0 || wb == 0) return DS_OK;
        return gram_f64(A, ld, wa, B, ld, wb, n, G + (size_t)ra * 144 + cb, 144, gram_partial, st);
    }

    int colnorms(const double* V, int64_t ldv, int w, std::vector<double>& out) {
        int threads = (1024 / w) * w;
        size_t sm = (size_t)(threads / w) * w * sizeof(double);
        k_colnorm2<<<norm_ctas, threads, sm, st>>>(V, ldv, w, n, norm_partial);
        DS_LAUNCH_CHECK();
        k_colsum_reduce<<<colsum_blocks(w), 256, 0, st>>>(norm_partial, norm_ctas, w, norms);
        DS_LAUNCH_CHECK();
        out.resize(w);
        DS_CUDA(cudaMemcpyAsync(out.data(), norms, w * sizeof(double), cudaMemcpyDeviceToHost, st));
        DS_CUDA(cudaStreamSynchronize(st));
        return DS_OK;
    }

    // largest eigenvalue of invD A by power iteration on invD A itself (16 fp32 columns; the un-shifted iteration
    // reaches 0.95 lmax in 12 steps where I + invD A needs 16-20, scripts/proto_pmg.py).
    // e_k = max over columns of ||A^(k+1) x|| / ||A^k x|| increases monotonically towards lmax for the SPD pencil.
    // It is sampled after 4, 8, 12, ... steps.  Accepted: a sample that moved by less than 1 % (x 1.1), or -- the usual
    // case, 12 steps -- Aitken's extrapolation of the last three samples when it is consistent (between e_k and
    // 1.5 e_k), which bounds the limit of the geometric tail instead of trusting a fixed step count (ADVICE r1: a
    // Chebyshev interval that ends below lmax amplifies the top of the spectrum).  Cap: 40 steps.
    // Two halves: lmax_enqueue launches the first 12 steps and their three samples on any stream with NO host
    // synchronisation (the samples stay on the device), lmax_finish reads them back, applies the acceptance rule in the
    // order the samples were taken (the result is the one a step-by-step host loop would have stopped at) and only
    // continues step by step in the rare case that neither rule fired.
    static constexpr int LMAX_W = 16, LMAX_STEPS0 = 12;
    int lmax_norms(const float* v, int64_t nl, double* out_dev, cudaStream_t s) {
        DS_TRY(colnorm2_f32(v, LMAX_W, nl, norm_partial, norm_ctas, s));
        k_colsum_reduce<<<colsum_blocks(LMAX_W), 256, 0, s>>>(norm_partial, norm_ctas, LMAX_W, out_dev);
        DS_LAUNCH_CHECK();
        return DS_OK;
    }
    int lmax_step(Level32& L, float*& a, float*& b, float* zero_r, cudaStream_t s) {
        // b = a + (-1) (a - 0) + (-1) invD (0 - A a) = invD A a     (Zprev = R = the zero block)
        DS_TRY(spmm32(S32_MODE_CHEB, L.brow, L.rec, L.n_nodes, LMAX_W, a, zero_r, L.invD, zero_r, b, -1.f, -1.f, L.prof_cls,
                      s, L.chunk_row));
        std::swap(a, b);
        L.launches++;
        L.cols += LMAX_W;
        return DS_OK;
    }
    // samples_dev: [2 * LMAX_STEPS0 / 4][LMAX_W] doubles; uses norm_partial (one estimate in flight per driver)
    int lmax_enqueue(Level32& L, float* a, float* b, float* zero_r, double* samples_dev, cudaStream_t s) {
        const int64_t nl = 3 * L.n_nodes;
        DS_CUDA(cudaMemsetAsync(zero_r, 0, sizeof(float) * nl * LMAX_W, s));
        DS_TRY(fill_random_f32(a, nl * LMAX_W, 0x1234567ull, s));
        for (int it = 0; it < LMAX_STEPS0; ++it) {
            const bool sample = (it & 3) == 3;
            if (sample) DS_TRY(lmax_norms(a, nl, samples_dev + (size_t)(2 * (it / 4)) * LMAX_W, s));
            DS_TRY(lmax_step(L, a, b, zero_r, s));
            if (sample) DS_TRY(lmax_norms(a, nl, samples_dev + (size_t)(2 * (it / 4) + 1) * LMAX_W, s));
        }
        return DS_OK;
    }
    int lmax_finish(Level32& L, float* a, float* b, float* zero_r, const double* samples_dev, cudaStream_t s) {
        constexpr int NS = LMAX_STEPS0 / 4;
        const int64_t nl = 3 * L.n_nodes;
        double h[2 * NS * LMAX_W];
        DS_CUDA(cudaMemcpyAsync(h, samples_dev, sizeof(h), cudaMemcpyDeviceToHost, s));
        DS_CUDA(cudaStreamSynchronize(s));
        double best = 0.0, e1 = 0.0, e2 = 0.0;
        bool done = false;
        auto accept = [&](double e3) {          // the acceptance rule after one more sample
            best = e3;
            if (e2 > 0.0 && e3 <= 1.01 * e2) return true;
            if (e1 > 0.0) {
                const double d1 = e2 - e1, d2 = e3 - e2;
                if (d1 > d2 && d2 > 0.0) {
                    const double lim = e3 + d2 * d2 / (d1 - d2);          // Aitken: e3 + d2 q / (1 - q), q = d2 / d1
                    if (lim <= 1.5 * e3) { best = std::max(e3, lim / 1.1 * 1.05); return true; }
                }
            }
            e1 = e2;
            e2 = e3;
            return false;
        };
        for (int k = 0; k < NS && !done; ++k) {
            double e3 = 0.0;
            for (int c = 0; c < LMAX_W; ++c)
                e3 = std::max(e3, std::sqrt(h[(2 * k + 1) * LMAX_W + c] / h[(2 * k) * LMAX_W + c]));
            done = accept(e3);
        }
        // LMAX_STEPS0 is even: after the enqueued steps the iterate is back in `a`
        std::vector<double> n0(LMAX_W), n1(LMAX_W);
        auto norms_sync = [&](const float* v, std::vector<double>& out) -> int {
            DS_TRY(lmax_norms(v, nl, norms, s));
            DS_CUDA(cudaMemcpyAsync(out.data(), norms, LMAX_W * sizeof(double), cudaMemcpyDeviceToHost, s));
            DS_CUDA(cudaStreamSynchronize(s));
            return DS_OK;
        };
        for (int it = LMAX_STEPS0; it < 40 && !done; ++it) {
            const bool sample = (it & 3) == 3;
            if (sample) DS_TRY(norms_sync(a, n0));
            DS_TRY(lmax_step(L, a, b, zero_r, s));
            if (sample) {
                DS_TRY(norms_sync(a, n1));
                double e3 = 0.0;
                for (int c = 0; c < LMAX_W; ++c) e3 = std::max(e3, std::sqrt(n1[c] / n0[c]));
                done = accept(e3);
            }
        }
        L.lmax = 1.1 * best;
        return DS_OK;
    }
    int estimate_lmax(Level32& L, float* a, float* b, float* zero_r) {
        DS_TRY(lmax_enqueue(L, a, b, zero_r, lmax_samples, st));
        return lmax_finish(L, a, b, zero_r, lmax_samples, st);
    }

    // W32 = T R32 (w columns): Chebyshev polynomial (one level) or the two-level V-cycle
    int apply_precond(int w, float** out) {
        float* zc = Za;
        float* zp = Zb;
        if (!cl) {
            DS_TRY(fine.cheb(R32, w, o.cheb_degree, o.cheb_ratio > 1.0 ? o.cheb_ratio : 30.0, true, &zc, &zp, st));
            *out = zc;
            return DS_OK;
        }
        const int nu = o.smooth_steps > 0 ? o.smooth_steps : 3;
        const double sr = o.smooth_ratio > 1.0 ? o.smooth_ratio : 8.0;
        DS_TRY(fine.cheb(R32, w, nu, sr, true, &zc, &zp, st));                               // pre-smooth from zero
        DS_TRY(spmm32(S32_MODE_RESID, fine.brow, fine.rec, n_nodes, w, zc, R32, nullptr, nullptr, zp, 0.f, 0.f,
                      PROF_CHEB, st, fine.chunk_row));                                                       // zp = r - A z
        fine.launches++; fine.cols += w;
        DS_TRY(restrict32(cl->rptr, cl->rlist, cl->n_nodes, zp, w, RC32, st, coarse.perm, fine.inv));
        float* cc = ZCa;
        float* cp = ZCb;
        DS_TRY(coarse.cheb(RC32, w, o.coarse_degree, o.coarse_ratio > 1.0 ? o.coarse_ratio : 30.0, true, &cc, &cp, st));
        DS_TRY(prolong_add32(cl->parents, n_nodes, cc, w, zc, st, fine.perm, coarse.inv));
        DS_TRY(fine.cheb(R32, w, nu, sr, false, &zc, &zp, st));                              // post-smooth
        *out = zc;
        return DS_OK;
    }

    // Wout (n x w, ld) = p(invD K) invD R64: `degree` Chebyshev steps on [lmax / ratio, lmax] in FP64, from zero
    int apply_precond64(int w, int degree, double ratio, double lmax, double* Wout, int64_t ldw) {
        ProfScope prof(PROF_CHEB, st);
        const double lmin = lmax / ratio, theta = 0.5 * (lmax + lmin), delta = 0.5 * (lmax - lmin), sig = theta / delta;
        double rho = 1.0 / sig;
        const unsigned blocks = (unsigned)ceil_div(n_nodes * w, 256);
        double *zc = Z64a, *zp = Z64b;
        k_cheb64_update<<<blocks, 256, 0, st>>>(invD64, R64, w, nullptr, nullptr, zc, w, n_nodes, w, 0.0, 1.0 / theta);
        DS_LAUNCH_CHECK();
        DS_CUDA(cudaMemsetAsync(zp, 0, sizeof(double) * (size_t)n * w, st));
        for (int k = 1; k < degree; ++k) {
            const double rho_new = 1.0 / (2.0 * sig - rho);
            // RES = R - K zc
            DS_TRY(spmm_km(brow, bcol, n_nodes, Kval, nullptr, 0.0, zc, w, w, -1.0, 1.0, R64, w, RES64, w, st));
            spmm_count++;
            k_cheb64_update<<<blocks, 256, 0, st>>>(invD64, RES64, w, zc, zp, zp, w, n_nodes, w, rho_new * rho, 2.0 * rho_new / delta);
            DS_LAUNCH_CHECK();
            std::swap(zc, zp);
            rho = rho_new;
        }
        DS_CUDA(cudaMemcpy2DAsync(Wout, ldw * 8, zc, (size_t)w * 8, (size_t)w * 8, n, cudaMemcpyDeviceToDevice, st));
        return DS_OK;
    }

    int run(double* X, double* lambda_out, double* resid_out, int64_t* stats);

    // Nested iteration: lowest pairs of the P1 problem (same driver, one-level Chebyshev preconditioner,
    // loose tolerance), prolonged into the P2 start block.  The coarse start block is the injection of X
    // (its first columns are the analytic rigid-body modes, which P reproduces exactly).
    int nested_start(double* X) {
        if (!ws->child) {
            ws->child = new ds_workspace();
            ws->child->num_sms = ws->num_sms;
        }
        DS_TRY(inject64(cl->rptr, cl->rlist, cl->n_nodes, X, m, m, Xc, m, st));
        Driver dc;
        dc.ws = ws->child;
        dc.st = st;
        dc.brow = cl->brow; dc.bcol = cl->bcol;
        dc.n_nodes = cl->n_nodes; dc.n = 3 * cl->n_nodes;
        dc.Kval = cl->Kval; dc.Mblk = cl->Mblk;
        dc.m = m;
        dc.fine_prof_cls = PROF_COARSE;
        dc.o = o;
        dc.o.nested = 0;
        dc.o.locked = nullptr;
        dc.o.n_locked = 0;
        dc.o.coords = cl->coords;
        dc.o.fixed = cl->fixed;
        dc.o.tol = o.nested_tol > 0.0 ? o.nested_tol : 3e-2;
        dc.o.maxit = 40;
        const int deg = o.nested_degree > 0
                            ? o.nested_degree
                            : (int)std::min(48.0, std::max(24.0, std::round(std::cbrt((double)dc.n) / 1.2)));   // floor: thin shells; 1.2: one nested iteration fewer than 1.5 at n_c = 107 811 (r2t tuning)
        dc.o.cheb_degree = deg;
        dc.o.cheb_ratio = 0.4 * deg * deg;
        int64_t cstats[12] = {0};
        DS_TRY(dc.run(Xc, lamc, resc, cstats));
        nested_iters = cstats[0];
        child_lmax = dc.fine.lmax;
        nested_status = cstats[3];
        spmm_count += cstats[2];
        coarse.launches += cstats[4];           // the nested solve's SpMMs are coarse-level work
        coarse.cols += cstats[5];
        DS_TRY(prolong64(cl->parents, n_nodes, Xc, m, m, X, m, st));
        return DS_OK;
    }
};

}  // namespace ds

namespace ds {

int Driver::run(double* X, double* lambda_out, double* resid_out, int64_t* stats) {
    const int nev = o.nev;
    int nr = o.n_rigid < 0 ? 0 : o.n_rigid;
    DS_TRY(alloc());
    if (o.precond_fp64) {
        k_invd64<<<(unsigned)ceil_div(n_nodes, 256), 256, 0, st>>>(brow, bcol, n_nodes, Kval, invD64);
        DS_LAUNCH_CHECK();
    }
    if (Xc && !nq) DS_TRY(nested_start(X));
    // Spectral radii of the Chebyshev intervals: 12 SpMM launches and three samples per level without a host
    // synchronisation in between.  The P1 operator of the coarse level is the nested solve's fine level (same records, same
    // start vector), so its estimate is taken over.  (Running the fine-level estimate on a side stream next to the nested
    // solve was measured and dropped: full-SM SpMM CTAs cannot share an SM with the nested solve's cooperative kernels, the
    // two streams only delay each other's launches -- no gain, and one 100 ms stall in four runs.)
    DS_TRY(estimate_lmax(fine, Za, Zb, R32));
    if (cl) {
        if (child_lmax > 0.0) coarse.lmax = child_lmax;
        else DS_TRY(estimate_lmax(coarse, ZCa, ZCb, RC32));
    }
    if (o.verbose)
        fprintf(stderr, "[ds_lobpcg] n=%lld m=%d nev=%d lmax(invD K)=%.4f %s deg=%d coarse: n=%lld lmax=%.4f deg=%d nu=%d\n",
                (long long)n, m, nev, fine.lmax / 1.1, cl ? "two-level" : "chebyshev", o.cheb_degree,
                (long long)(cl ? 3 * cl->n_nodes : 0), coarse.lmax / 1.1, o.coarse_degree, o.smooth_steps);

    // ---- initial Rayleigh-Ritz on X
    cur = 0;
    DS_CUDA(cudaMemcpy2DAsync(Xb(0), ld * 8, X, m * 8, m * 8, n, cudaMemcpyDeviceToDevice, st));
    if (o.fixed) DS_TRY(mask_fixed_rows_f64(o.fixed, nullptr, n_nodes, Xb(0), ld, m, st));
    if (nq) {
        for (int c0 = 0; c0 < nq; c0 += 64) {
            const int wc = std::min(64, nq - c0);
            DS_TRY(spmm_km(brow, bcol, n_nodes, nullptr, Mblk, 1.0, Q + c0, nq, wc, 1.0, 0.0, nullptr, 0, MQ + c0, nq, st));
        }
        spmm_count += 1;
        DS_TRY(project_locked(Xb(0), ld, m));
        DS_TRY(project_locked(Xb(0), ld, m));      // twice: the start block may be far from M-orthogonal to Q
    }
    DS_TRY(spmm_dual(brow, bcol, n_nodes, Kval, Mblk, Xb(0), ld, m, KS[0], ld, MS[0], ld, st, fine.perm, fine.chunk_row,
                     spmm32_chunk_count(n_nodes)));
    spmm_count += 2;
    // Small generalised eigen-solve on the slots in play.  full = true: both Gram matrices are recomputed over
    // [X | W | P] in one pass (k_gram_sym2) -- the initial step, every REFRESH-th step and the fallback when the small
    // Cholesky fails; otherwise GK / GM hold the recurrences of rr.cu plus the strips of the new W.
    auto eig = [&](const std::vector<int>& slots) -> int {
        DS_CUDA(cudaMemsetAsync(Cm, 0, sizeof(double) * 144 * 144, st));
        return eigh_generalized_f64(GK, GM, (int)slots.size(), 144, slots.data(), -1e-6, theta, Cm, 144, eig_scratch, info_d, st);
    };
    auto full_gram = [&](int w, int nw, bool withP) -> int {
        DS_CUDA(cudaMemsetAsync(GK, 0, sizeof(double) * 144 * 144, st));
        DS_CUDA(cudaMemsetAsync(GM, 0, sizeof(double) * 144 * 144, st));
        int tiles[18], nt = 0;
        for (int t = 0; t < m / 8; ++t) tiles[nt++] = t;
        for (int t = 0; t < (nw + 7) / 8; ++t) tiles[nt++] = m / 8 + t;
        if (withP) for (int t = 0; t < m / 8; ++t) tiles[nt++] = 2 * m / 8 + t;
        DS_TRY(gram_sym2(S[w], KS[w], MS[w], ld, n, tiles, nt, GK, GM, 144, gram_partial2, ws->num_sms, st));
        return sym_upper(GK, GM, 144, 3 * m, st);
    };
    std::vector<int> slots;
    for (int j = 0; j < m; ++j) slots.push_back(j);
    DS_TRY(full_gram(0, 0, false));
    DS_TRY(eig(slots));
    int info_h[2] = {0, 0};
    DS_CUDA(cudaMemcpyAsync(info_h, info_d, sizeof(info_h), cudaMemcpyDeviceToHost, st));
    DS_CUDA(cudaStreamSynchronize(st));
    if (info_h[0] != 0) {
        set_error("ds_lobpcg: initial block is not M-independent (Cholesky pivot %d)", info_h[0]);
        return DS_ERR_NUMERIC;
    }
    // X <- X C etc. into buffer 1
    DS_TRY(block_gemm_f64(S[0], ld, m, Cm, 144, m, n, 1.0, 0.0, S[1], ld, st));
    DS_TRY(block_gemm_f64(KS[0], ld, m, Cm, 144, m, n, 1.0, 0.0, KS[1], ld, st));
    DS_TRY(block_gemm_f64(MS[0], ld, m, Cm, 144, m, n, 1.0, 0.0, MS[1], ld, st));
    cur = 1;
    DS_CUDA(cudaMemcpyAsync(lam_d, theta, m * sizeof(double), cudaMemcpyDeviceToDevice, st));
    // Gram pair of [X' | - | -]: diag(theta), I  (C has no W / P rows yet: the recurrence reduces to exactly that)
    DS_TRY(gram_algebra(GK, GM, GKn, GMn, 144, Cm, 144, theta, m, alg_scratch, st));
    std::swap(GK, GKn);
    std::swap(GM, GMn);

    std::vector<double> lam(m), hn(2 * m), rel(m, 1.0);
    std::vector<int> act;
    bool haveP = false;                // the P slots of buffer `cur` hold the previous step's directions (slot j <-> X column j)
    int it = 0, nconv = 0, status = 1, since_refresh = 0;
    int REFRESH = 8;
    if (const char* e = getenv("DS_LOBPCG_REFRESH")) REFRESH = atoi(e);              // diagnostics only
    if (const char* e = getenv("DS_LOBPCG_ORTHO_W")) o.ortho_w = atoi(e);
    if (const char* e = getenv("DS_LOBPCG_VERBOSE")) o.verbose = atoi(e);
    const bool z32 = fine.bcolP != nullptr && nq == 0 && !o.ortho_w && !o.precond_fp64;   // W = fp32 preconditioner output, unmodified
    const int res_threads = (1024 / m) * m;
    const size_t res_smem = (size_t)(res_threads / m) * 2 * m * sizeof(double);
    for (it = 0; it <= o.maxit; ++it) {
        // ---- residual and convergence
        { ProfScope prof(PROF_RESIDUAL, st);
        k_residual<<<norm_ctas, res_threads, res_smem, st>>>(KS[cur], MS[cur], ld, m, n, lam_d, R, m, norm_partial);
        DS_LAUNCH_CHECK();
        k_colsum_reduce<<<colsum_blocks(2 * m), 256, 0, st>>>(norm_partial, norm_ctas, 2 * m, norms);
        DS_LAUNCH_CHECK(); }
        DS_CUDA(cudaMemcpyAsync(hn.data(), norms, 2 * m * sizeof(double), cudaMemcpyDeviceToHost, st));
        DS_CUDA(cudaMemcpyAsync(lam.data(), lam_d, m * sizeof(double), cudaMemcpyDeviceToHost, st));
        DS_CUDA(cudaStreamSynchronize(st));
        if (o.n_rigid < 0) {   // automatic: leading eigenvalues that are numerically zero next to the block's largest
            const double big = std::fabs(lam[m - 1]);
            nr = 0;
            while (nr < m - 1 && std::fabs(lam[nr]) < 1e-9 * big) ++nr;
        }
        double lref = std::fabs(lam[std::min(nr, m - 1)]);
        act.clear();
        nconv = 0;
        for (int j = 0; j < m; ++j) {
            double rn = std::sqrt(hn[j]), mn = std::sqrt(hn[m + j]);
            double scale = (j < nr ? lref : std::fabs(lam[j])) * mn;
            rel[j] = scale > 0 ? rn / scale : rn;
            bool conv = rel[j] < o.tol;
            if (!conv) act.push_back(j);
            if (j < nev && conv) nconv++;
        }
        if (o.verbose) {
            double worst = 0;
            for (int j = nr; j < nev; ++j) worst = std::max(worst, rel[j]);
            fprintf(stderr, "[ds_lobpcg] it %3d  conv %d/%d  active %d  max rel res %.3e  lam[%d]=%.6e\n", it, nconv, nev,
                    (int)act.size(), worst, nr, lam[std::min(nr, m - 1)]);
        }
        if (nconv >= nev) { status = 0; break; }
        if (it == o.maxit) break;
        const int na = (int)act.size();
        const int wpad = (na + 15) & ~15;
        ColIdx ci;
        for (int s = 0; s < 128; ++s) ci.v[s] = (short)(s < na ? act[s] : 0);
        // ---- W = T(R[:, act])
        float* Zres = nullptr;
        if (o.precond_fp64) {
            k_gather_cols64<<<(unsigned)ceil_div(n * wpad, 256), 256, 0, st>>>(R, m, ci, na, wpad, n, R64);
            DS_LAUNCH_CHECK();
            const int deg64 = o.cheb_degree > 0 ? o.cheb_degree : 16;
            DS_TRY(apply_precond64(wpad, deg64, o.cheb_ratio > 1.0 ? o.cheb_ratio : 0.4 * deg64 * deg64, 1.25 * fine.lmax / 1.1,
                                   Wb(cur), ld));
            if (o.fixed) DS_TRY(mask_fixed_rows_f64(o.fixed, nullptr, n_nodes, Wb(cur), ld, wpad, st));
        } else {
            DS_TRY(gather_cols_f32(R, m, ci, na, wpad, n, R32, st, fine.perm));
            DS_TRY(apply_precond(wpad, &Zres));
            // Zres is in the preconditioner's numbering (read as is by k_spmm_dual_z32): mask it through the permutation
            if (o.fixed) DS_TRY(mask_fixed_rows_f32(o.fixed, fine.perm, n_nodes, Zres, wpad, wpad, st));
            DS_TRY(widen_f32(Zres, wpad, n, Wb(cur), ld, st, fine.perm));
        }
        if (o.verbose && !o.precond_fp64) {          // diagnostics: energy norm of the residuals, r_j^T T r_j / lambda_j
            const int threads = (1024 / na) * na;
            k_coldot_rw<<<norm_ctas, threads, (size_t)(threads / na) * na * sizeof(double), st>>>(R, m, ci, na, Wb(cur), ld, n, norm_partial);
            DS_LAUNCH_CHECK();
            k_colsum_reduce<<<colsum_blocks(na), 256, 0, st>>>(norm_partial, norm_ctas, na, norms);
            DS_LAUNCH_CHECK();
            std::vector<double> en(na);
            DS_CUDA(cudaMemcpyAsync(en.data(), norms, na * sizeof(double), cudaMemcpyDeviceToHost, st));
            DS_CUDA(cudaStreamSynchronize(st));
            double worst = 0.0, worst_rel = 0.0;
            for (int s2 = 0; s2 < na; ++s2) {
                const int j = act[s2];
                if (j < nr || j >= nev) continue;
                const double e = en[s2] / std::fabs(lam[j]);
                if (e > worst) { worst = e; worst_rel = rel[j]; }
            }
            fprintf(stderr, "[ds_lobpcg]        max energy residual r^T T r / lam = %.3e (its 2-norm rel res %.3e)\n", worst, worst_rel);
        }
        if (z32) {
            // K W, M W straight from the fp32 block in the preconditioner's numbering: W is used as it comes out of T
            // (the Rayleigh-Ritz step does not need W M-orthogonal to X; near convergence T R is M-orthogonal to X to
            // O(residual) anyway), so no FP64 copy is gathered
            DS_TRY(spmm_dual_z32(brow, fine.brow, fine.bcolP, fine.perm, fine.chunk_row, spmm32_chunk_count(n_nodes), n_nodes,
                                 Kval, Mblk, Zres, wpad, KS[cur] + m, ld, MS[cur] + m, ld, st, fine.nnzb));
        } else {
            if (nq) DS_TRY(project_locked(Wb(cur), ld, wpad));
            // ---- W <- W - X (MX^T W)
            DS_TRY(gram_f64(MS[cur], ld, m, Wb(cur), ld, wpad, n, GsK, 144, gram_partial, st));
            DS_TRY(block_gemm_f64(Xb(cur), ld, m, GsK, 144, wpad, n, -1.0, 1.0, Wb(cur), ld, st));
            DS_TRY(spmm_dual(brow, bcol, n_nodes, Kval, Mblk, Wb(cur), ld, wpad, KS[cur] + m, ld, MS[cur] + m, ld, st, fine.perm,
                             fine.chunk_row, spmm32_chunk_count(n_nodes)));
        }
        spmm_count += 2;
        // ---- Gram pair of [X | W | P]: the strips of the new W on top of the recurrences, or everything afresh
        bool useP = haveP;
        bool fresh = since_refresh >= REFRESH;
        if (fresh) {
            DS_TRY(full_gram(cur, wpad, haveP));
            since_refresh = 0;
        } else {
            DS_TRY(gram_strip(KS[cur] + m, MS[cur] + m, ld, wpad, S[cur], ld, ld, n, GsK, GsM, 144, strip_partial, ws->num_sms, st));
            DS_TRY(gram_insert(GK, GM, 144, GsK, GsM, 144, m, wpad, st));
        }
        // ---- Rayleigh-Ritz on [X, W(na), P(columns that are still active)]
        for (int attempt = 0; attempt < 3; ++attempt) {
            slots.clear();
            for (int j = 0; j < m; ++j) slots.push_back(j);
            for (int s = 0; s < na; ++s) slots.push_back(m + s);
            if (useP) for (int j : act) slots.push_back(2 * m + j);
            DS_TRY(eig(slots));
            DS_CUDA(cudaMemcpyAsync(info_h, info_d, sizeof(info_h), cudaMemcpyDeviceToHost, st));
            DS_CUDA(cudaStreamSynchronize(st));
            if (o.verbose) fprintf(stderr, "[ds_lobpcg]        small eigen-solve: N = %d, %d Jacobi sweeps\n", (int)slots.size(), info_h[1]);
            if (info_h[0] == 0) break;
            if (o.verbose) fprintf(stderr, "[ds_lobpcg] it %d: RR Cholesky failed (info %d, attempt %d)\n", it, info_h[0], attempt);
            if (!fresh) {                      // first suspect: drift of the Gram recurrences
                DS_TRY(full_gram(cur, wpad, haveP));
                fresh = true;
                since_refresh = 0;
                continue;
            }
            if (!useP) {
                set_error("ds_lobpcg: Rayleigh-Ritz breakdown at iteration %d (info %d)", it, info_h[0]);
                return DS_ERR_NUMERIC;
            }
            useP = false;                      // then: P nearly dependent on [X, W] -- restart without it
        }
        if (info_h[0] != 0) {
            set_error("ds_lobpcg: Rayleigh-Ritz breakdown at iteration %d (info %d)", it, info_h[0]);
            return DS_ERR_NUMERIC;
        }
        // ---- update: P' = [W P] C[m:, :m] into the P slots, X' = X C[:m, :m] + P' into the X slots (all three buffers)
        int nxt = cur ^ 1;
        {
            const double* Ain[3] = {S[cur], KS[cur], MS[cur]};
            double* Yout[3] = {S[nxt], KS[nxt], MS[nxt]};
            DS_TRY(rr_update2_f64(Ain, ld, m, wpad, useP ? 1 : 0, Cm, 144, n, Yout, ld, st));
        }
        // ---- Gram pair of [X' | - | P'] from the small matrices (rows of C at unused slots are zero)
        DS_TRY(gram_algebra(GK, GM, GKn, GMn, 144, Cm, 144, theta, m, alg_scratch, st));
        std::swap(GK, GKn);
        std::swap(GM, GMn);
        haveP = true;
        since_refresh++;
        DS_CUDA(cudaMemcpyAsync(lam_d, theta, m * sizeof(double), cudaMemcpyDeviceToDevice, st));
        cur = nxt;
    }
    // ---- results
    DS_CUDA(cudaMemcpy2DAsync(X, m * 8, Xb(cur), ld * 8, m * 8, n, cudaMemcpyDeviceToDevice, st));
    DS_CUDA(cudaMemcpyAsync(lambda_out, lam_d, m * sizeof(double), cudaMemcpyDeviceToDevice, st));
    DS_CUDA(cudaMemcpyAsync(resid_out, rel.data(), m * sizeof(double), cudaMemcpyHostToDevice, st));
    unsigned gb_f[2] = {0, 0}, gb_c[2] = {0, 0};      // [1]: grid-barrier timeout flag of the persistent Chebyshev kernel
    DS_CUDA(cudaMemcpyAsync(gb_f, fine.gbar, sizeof(gb_f), cudaMemcpyDeviceToHost, st));
    if (cl) DS_CUDA(cudaMemcpyAsync(gb_c, coarse.gbar, sizeof(gb_c), cudaMemcpyDeviceToHost, st));
    DS_CUDA(cudaStreamSynchronize(st));
    if (gb_f[1] || gb_c[1]) {
        set_error("ds_lobpcg: grid barrier of the persistent Chebyshev kernel timed out (device shared with other work?)");
        return DS_ERR_CUDA;
    }
    stats[0] = it;
    stats[1] = nconv;
    stats[3] = status;
    stats[2] = spmm_count + fine.launches + coarse.launches;
    stats[4] = fine.launches;
    stats[5] = fine.cols;
    stats[6] = coarse.launches;
    stats[7] = coarse.cols;
    stats[8] = nested_iters;
    stats[9] = nested_status;
    // spectral-radius estimates lmax(invD K) of the fine and the coarse level, as round(1e9 * estimate): a caller that runs
    // its own cycle on the same operator (the row-slab driver's replicated coarse level) takes them over
    stats[10] = (int64_t)std::llround(1e9 * fine.lmax);
    stats[11] = (int64_t)std::llround(1e9 * coarse.lmax);
    return DS_OK;
}

}  // namespace ds

using namespace ds;

// R = KX - MX diag(lam) and the column sums of R^2 and MX^2 (sums[2m], device) over the rows given: the residual step of
// the iteration as a stand-alone call (row-partitioned driver: the sums are all-reduced over the ranks)
extern "C" int ds_lobpcg_residual(const double* KX, const double* MX, int64_t ld, int m, int64_t n, const double* lam, double* R,
                                  int64_t ldr, double* sums, double* partial, void* stream) {
    DS_REQUIRE(KX && MX && lam && R && sums && partial && m > 0 && m <= 64 && n > 0, "ds_lobpcg_residual: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    ProfScope prof(PROF_RESIDUAL, st);
    const int ctas = 296, threads = (1024 / m) * m;
    k_residual<<<ctas, threads, (size_t)(threads / m) * 2 * m * sizeof(double), st>>>(KX, MX, ld, m, n, lam, R, ldr, partial);
    DS_LAUNCH_CHECK();
    k_colsum_reduce<<<colsum_blocks(2 * m), 256, 0, st>>>(partial, ctas, 2 * m, sums);
    DS_LAUNCH_CHECK();
    return DS_OK;
}

extern "C" int ds_lobpcg(ds_workspace* ws, const int32_t* brow, const int32_t* bcol, int64_t n_nodes,
                         const double* Kval, const double* Mblk, const ds_pmg_level* coarse, double* X, int m,
                         const ds_lobpcg_opts* opts, double* lambda_out, double* resid_out, int64_t* stats_host,
                         void* stream) {
    DS_REQUIRE(ws && brow && bcol && Kval && Mblk && X && opts && lambda_out && resid_out && stats_host,
               "ds_lobpcg: null argument");
    DS_REQUIRE(m >= 16 && m % 16 == 0 && m <= 48, "ds_lobpcg: block size m=%d must be 16, 32 or 48", m);
    DS_REQUIRE(opts->nev >= 1 && opts->nev <= m, "ds_lobpcg: nev=%d must be in [1, m=%d]", opts->nev, m);
    DS_REQUIRE(3 * n_nodes >= 3 * (int64_t)m, "ds_lobpcg: matrix too small for block size (n=%lld, 3m=%d)",
               (long long)(3 * n_nodes), 3 * m);
    DS_REQUIRE(opts->cheb_degree >= 1 && opts->maxit >= 1 && opts->tol > 0, "ds_lobpcg: bad options");
    DS_REQUIRE(opts->n_rigid >= -1 && opts->n_rigid <= opts->nev, "ds_lobpcg: bad n_rigid");
    DS_REQUIRE(!opts->fixed || opts->n_rigid == 0, "ds_lobpcg: clamped nodes leave no rigid modes: n_rigid must be 0");
    if (coarse) {
        DS_REQUIRE(coarse->brow && coarse->bcol && coarse->Kval && coarse->parents && coarse->rptr && coarse->rlist &&
                       coarse->n_nodes > 0 && coarse->nnzb > 0,
                   "ds_lobpcg: incomplete coarse level");
        DS_REQUIRE(opts->coarse_degree >= 1, "ds_lobpcg: coarse_degree must be >= 1 with a coarse level");
    }
    Driver d;
    d.cl = coarse;
    d.ws = ws;
    d.st = (cudaStream_t)stream;
    d.brow = brow; d.bcol = bcol;
    d.n_nodes = n_nodes; d.n = 3 * n_nodes;
    d.Kval = Kval; d.Mblk = Mblk;
    d.m = m;
    d.o = *opts;
    if (opts->locked) {
        DS_REQUIRE(opts->n_locked > 0 && opts->n_locked % 16 == 0 && opts->n_locked <= 192,
                   "ds_lobpcg: n_locked=%d must be a positive multiple of 16, <= 192", opts->n_locked);
        DS_REQUIRE((uintptr_t)opts->locked % 16 == 0, "ds_lobpcg: locked block must be 16-byte aligned");
        d.Q = opts->locked;
        d.nq = opts->n_locked;
    }
    return d.run(X, lambda_out, resid_out, stats_host);
}

// Generalised symmetric eigenproblem GK c = theta GM c of the Rayleigh-Ritz step, N <= 144, FP64.
//
// Reference behaviour replaced: torch.linalg.cholesky / torch.linalg.eigh on the projected problem
// (/root/reference/src/lobpcg/_lobpcg.py:507-525, _linalg_utils.py:87-96).
//
// Method (implicit Cholesky / one-sided Jacobi, high relative accuracy for the small eigenvalues):
//   D = diag(GM)^-1/2;  L L^T = D GM D;  R R^T = D (GK + sigma GM) D;  Y = L^-1 R;
//   one-sided Jacobi orthogonalises the ROWS of Y:  Q^T Y,  |row_j|^2 = theta_j + sigma;
//   c_j = D R^-T row_j.
// Four kernels (round 2: the factorisations and the triangular solves no longer sit on one CTA -- 0.40 + 0.12 ms of a
// 1.2 ms solve were spent there with 147 SMs idle):
//   k_eigh_chol    (two CTAs)     gather / scale; CTA 0 factorises D GM D, CTA 1 D (GK + sigma GM) D, concurrently
//   k_eigh_solve   (ten CTAs)     Y = L^-1 R, one warp per column (columns are independent), Y -> global scratch
//   k_eigh_jacobi  (cluster of 8) the Jacobi sweeps.  One WARP per pair of rows, rows in registers
//                                 (5 elements per lane); pairs follow the odd-even transposition
//                                 ordering on a line of positions, so per step exactly one row per warp
//                                 moves to the neighbouring warp -- through a mailbox in the RECEIVER's
//                                 shared memory, written with st.shared::cluster (DSMEM) when the
//                                 neighbour sits in another CTA of the cluster, and one
//                                 barrier.cluster per step.  One SM's FP64 pipe and shared-memory
//                                 bandwidth were the limit of the single-CTA version (4.3 ms at N = 144).
//   k_eigh_finish  (nine CTAs)    eigenvalues, ascending rank; c_j = D R^-T row_j, one warp per row (rows are independent).
// Measured and dropped (round 2): blocks of two rows per line position / four rows per warp with pairs of independent
// rotations interleaved (half the mailbox hand-overs): 2.16 ms against 1.78 ms at N = 144 on a dense test pencil.  A
// rotation is ~1000 cycles of dependent FP64 latency (5-stage warp sum, sqrt, divide, rsqrt); the hand-over is only
// ~150 of the ~1150 cycles of a step, and N - 1 sequential rotation rounds per sweep are the floor of any ordering.
#include "common.cuh"
#include "../../include/diffsound_sm100.h"
#include "kernels.cuh"
#include "ptx.cuh"

namespace ds {

constexpr int EIG_MAXN = 144;
constexpr int EIG_THREADS = 1024;                 // prepare / finish
constexpr int JC_CL = 8;                          // CTAs per cluster
constexpr int JC_GPC = EIG_MAXN / 2 / JC_CL;      // 9 row pairs (warps) per CTA
constexpr int JC_THREADS = JC_GPC * 32;           // 288
constexpr int JC_E = 5;                           // row elements per lane: 5 * 32 = 160 >= 144
constexpr int JC_LD = 32 * JC_E;                  // row pitch of Y in global scratch
constexpr int JC_SLOT = JC_LD + 8;                // mailbox slot: elements + |row|^2 at [JC_LD]
static_assert(JC_GPC * JC_CL * 2 == EIG_MAXN, "line positions must tile the cluster");

// scratch layout (doubles): L [N*N] | R [N*N] | Y [(N+1) * JC_LD] | scale [N] | 1/diag(L) [N] | 1/diag(R) [N] |
// meta [8]: sigma, fail, code of CTA 0, code of CTA 1 | R^T [N*N]
__host__ __device__ inline size_t eig_off_Rt(int N) { return (size_t)N * N; }
__host__ __device__ inline size_t eig_off_Y(int N) { return 2 * (size_t)N * N; }
__host__ __device__ inline size_t eig_off_scale(int N) { return eig_off_Y(N) + (size_t)(N + 1) * JC_LD; }
__host__ __device__ inline size_t eig_off_invL(int N) { return eig_off_scale(N) + N; }
__host__ __device__ inline size_t eig_off_invR(int N) { return eig_off_invL(N) + N; }
__host__ __device__ inline size_t eig_off_meta(int N) { return eig_off_invR(N) + N; }
__host__ __device__ inline size_t eig_off_RT(int N) { return eig_off_meta(N) + 8; }      // R^T (row k = column k of R)
int64_t eigh_scratch_elems(int N) { return (int64_t)eig_off_RT(N) + (int64_t)N * N; }

constexpr int EIG_NB = 16;                        // block size of the blocked factorisations / substitutions

// in-place Cholesky (lower) of the N x N matrix in shared memory (row stride ld), right-looking with
// EIG_NB-wide panels: the diagonal block is factorised by warp 0 alone (warp-synchronous), the panel
// below it by one thread per row, the trailing update by the whole CTA -- 3 CTA barriers per panel
// instead of 3 per column.  returns 0 or failing column + 1 (same value in every thread).
__device__ int chol_lower(double* S, int N, int ld, int* s_flag) {
    const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31;
    for (int kb = 0; kb < N; kb += EIG_NB) {
        const int nb = min(EIG_NB, N - kb);
        double* D = S + (size_t)kb * ld + kb;        // diagonal block, D[i * ld + j]
        if (tid < 32) {
            // lane i holds row i of the block in registers; column k is broadcast by shuffles
            double a[EIG_NB];
#pragma unroll
            for (int j = 0; j < EIG_NB; ++j) a[j] = (lane < nb && j <= lane && j < nb) ? D[lane * ld + j] : 0.0;
            int fail = 0;
#pragma unroll
            for (int k = 0; k < EIG_NB; ++k) {
                if (k < nb) {                                       // warp-uniform
                    const double d = __shfl_sync(0xffffffffu, a[k], k);
                    if (!(d > 0.0)) { if (!fail) fail = kb + k + 1; }
                    const double sq = sqrt(d > 0.0 ? d : 1.0), rd = 1.0 / sq;
                    if (lane == k) a[k] = sq;
                    else if (lane > k) a[k] *= rd;
                    const double lik = a[k];
#pragma unroll
                    for (int j = k + 1; j < EIG_NB; ++j) {
                        const double ljk = __shfl_sync(0xffffffffu, a[k], j);
                        if (j < nb && lane >= j) a[j] -= lik * ljk;
                    }
                }
            }
            if (fail) { if (lane == 0) *s_flag = fail; }
            else if (lane < nb) {
#pragma unroll
                for (int j = 0; j < EIG_NB; ++j)
                    if (j <= lane && j < nb) D[lane * ld + j] = a[j];
            }
        }
        __syncthreads();
        if (*s_flag) return *s_flag;
        const int r = N - kb - nb;                   // rows below the panel
        if (r > 0) {
            // panel: x L_d^T = a for every row below (forward substitution, one thread per row)
            if (tid < r) {
                double* ap = S + (size_t)(kb + nb + tid) * ld + kb;
                double a[EIG_NB];
#pragma unroll
                for (int k = 0; k < EIG_NB; ++k) a[k] = k < nb ? ap[k] : 0.0;
#pragma unroll
                for (int k = 0; k < EIG_NB; ++k) {
                    if (k < nb) {
                        double v = a[k];
#pragma unroll
                        for (int q = 0; q < EIG_NB; ++q)
                            if (q < k) v -= a[q] * D[k * ld + q];
                        a[k] = v / D[k * ld + k];
                        ap[k] = a[k];
                    }
                }
            }
            __syncthreads();
            // trailing update S[i][j] -= sum_k S[i][kb+k] S[j][kb+k], i >= j in the trailing block
            for (int t = tid; t < r * r; t += nt) {
                const int i = t / r, j = t - i * r;
                if (j <= i) {
                    const double* pi = S + (size_t)(kb + nb + i) * ld + kb;
                    const double* pj = S + (size_t)(kb + nb + j) * ld + kb;
                    double v = 0.0;
                    for (int k = 0; k < nb; ++k) v = fma(pi[k], pj[k], v);
                    S[(size_t)(kb + nb + i) * ld + kb + nb + j] -= v;
                }
            }
            __syncthreads();
        }
    }
    return 0;
}

struct EigIdx {
    short v[EIG_MAXN];
};

// upper-triangle read through the slot map: entry (i, j) of the compact problem
__device__ __forceinline__ double g_up(const double* __restrict__ G, int64_t ldg, const EigIdx& ix, int i, int j) {
    int a = ix.v[i], b = ix.v[j];
    return a <= b ? G[(int64_t)a * ldg + b] : G[(int64_t)b * ldg + a];
}

// blockIdx.x = 0: L = chol(D GM D);  1: R = chol(D (GK + sigma GM) D).  Factors go to global scratch row-major with
// their reciprocal diagonals; failure codes to meta[2 + blockIdx.x] (0 = ok, else failing column + 1).
__global__ void __launch_bounds__(EIG_THREADS)
k_eigh_chol(const double* __restrict__ GK, const double* __restrict__ GM, int N, int64_t ldg,
            const __grid_constant__ EigIdx ix, double sigma_in, double* __restrict__ scratch) {
    extern __shared__ __align__(16) double S[];  // [N][ld]
    const int ld = N + 2;
    double* s_scale = S + (size_t)N * ld;        // [N]
    int* s_flag = reinterpret_cast<int*>(s_scale + N);
    const int tid = threadIdx.x, nt = blockDim.x, which = blockIdx.x;
    double* out = scratch + (which == 0 ? 0 : eig_off_Rt(N));
    double* inv = scratch + (which == 0 ? eig_off_invL(N) : eig_off_invR(N));
    double* meta = scratch + eig_off_meta(N);
    if (tid == 0) s_flag[0] = 0;
    for (int i = tid; i < N; i += nt) {
        double d = g_up(GM, ldg, ix, i, i);
        s_scale[i] = d > 0.0 ? rsqrt(d) : 1.0;
    }
    __syncthreads();
    double sigma = sigma_in;
    if (which == 1 && sigma_in < 0.0) {          // automatic shift = |sigma| * mean diagonal of the scaled GK
        double tr = 0.0;
        for (int i = 0; i < N; ++i) tr += fabs(g_up(GK, ldg, ix, i, i)) * s_scale[i] * s_scale[i];
        sigma = -sigma_in * tr / N;
    }
    for (int t = tid; t < N * N; t += nt) {
        int i = t / N, j = t % N;
        double v = 0.0;
        if (j <= i) v = which == 0 ? g_up(GM, ldg, ix, i, j) : g_up(GK, ldg, ix, i, j) + sigma * g_up(GM, ldg, ix, i, j);
        S[i * ld + j] = v * s_scale[i] * s_scale[j];
    }
    __syncthreads();
    const int bad = chol_lower(S, N, ld, s_flag);
    if (tid == 0) meta[2 + which] = (double)bad;
    if (bad) return;
    for (int t = tid; t < N * N; t += nt) {
        int i = t / N, j = t % N;
        out[t] = (j <= i) ? S[i * ld + j] : 0.0;
    }
    if (which == 1) {
        double* RT = scratch + eig_off_RT(N);
        for (int t = tid; t < N * N; t += nt) {
            int k = t / N, q = t % N;            // RT[k][q] = R[q][k]
            RT[t] = (k <= q) ? S[q * ld + k] : 0.0;
        }
    }
    for (int i = tid; i < N; i += nt) inv[i] = 1.0 / S[i * ld + i];
    if (which == 0) for (int i = tid; i < N; i += nt) scratch[eig_off_scale(N) + i] = s_scale[i];
    if (which == 1 && tid == 0) meta[0] = sigma;
}

constexpr int ES_WARPS = 16;                     // columns (solve) / rows (finish) per CTA

// Y = L^-1 R, column by column: warp w of CTA c owns column j = 16 c + w; lane l keeps y_k for k = l (mod 32).
// Also merges the failure codes of k_eigh_chol into info / meta[1] and zero-pads Y to JC_LD columns, Np rows.
__global__ void __launch_bounds__(ES_WARPS * 32)
k_eigh_solve(int N, double* __restrict__ scratch, int* __restrict__ info) {
    const double* __restrict__ L = scratch;
    const double* __restrict__ R = scratch + eig_off_Rt(N);
    const double* __restrict__ invL = scratch + eig_off_invL(N);
    double* __restrict__ Yg = scratch + eig_off_Y(N);
    double* meta = scratch + eig_off_meta(N);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int c0 = (int)meta[2], c1 = (int)meta[3];
    if (c0 || c1) {
        if (blockIdx.x == 0 && threadIdx.x == 0) { info[0] = c0 ? c0 : 1000 + c1; info[1] = 0; meta[1] = 1.0; }
        return;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) meta[1] = 0.0;
    const int Np = (N + 1) & ~1;
    const int j = blockIdx.x * ES_WARPS + warp;
    if (j >= JC_LD) return;
    if (j >= N) {                                // padding column
        for (int i = lane; i < Np; i += 32) Yg[(size_t)i * JC_LD + j] = 0.0;
        return;
    }
    double y[JC_E];
#pragma unroll
    for (int t = 0; t < JC_E; ++t) y[t] = 0.0;
    // The substitution is a chain of N - j warp reductions; the row of L, the R entry and the reciprocal pivot of step i do not
    // depend on it, so they are fetched two steps ahead (an L2 round trip is longer than one reduction).
    double l0[JC_E], l1[JC_E], l2[JC_E], r0 = 0.0, r1 = 0.0, r2 = 0.0, d0 = 0.0, d1 = 0.0, d2 = 0.0;
    auto load_row = [&](int i, double (&l)[JC_E], double& r, double& d) {
        if (i < N) {
            const double* Li = L + (size_t)i * N;
#pragma unroll
            for (int t = 0; t < JC_E; ++t) { const int k = lane + 32 * t; l[t] = k < i ? __ldg(Li + k) : 0.0; }
            r = __ldg(R + (size_t)i * N + j);
            d = __ldg(invL + i);
        }
    };
    load_row(j, l0, r0, d0);
    load_row(j + 1, l1, r1, d1);
#pragma unroll
    for (int ti = 0; ti < JC_E; ++ti) {          // i = 32 ti + ii: the register that receives y_i is static
        for (int ii = 0; ii < 32; ++ii) {
            const int i = 32 * ti + ii;
            if (i < j || i >= N) continue;       // warp-uniform
            load_row(i + 2, l2, r2, d2);
            double s = 0.0;
#pragma unroll
            for (int t = 0; t < JC_E; ++t) {
                const int k = lane + 32 * t;
                if (k >= j && k < i) s = fma(l0[t], y[t], s);
            }
            s = warp_sum(s);
            const double yi = (r0 - s) * d0;
            if (lane == ii) y[ti] = yi;
#pragma unroll
            for (int t = 0; t < JC_E; ++t) { l0[t] = l1[t]; l1[t] = l2[t]; }
            r0 = r1; r1 = r2; d0 = d1; d1 = d2;
        }
    }
#pragma unroll
    for (int t = 0; t < JC_E; ++t) {
        const int i = lane + 32 * t;
        if (i < Np) Yg[(size_t)i * JC_LD + j] = (i >= j && i < N) ? y[t] : 0.0;
    }
}

// ---- cluster primitives ----------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;\n" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;\n" ::: "memory");
}
// address of `p` (a shared-memory pointer of this CTA's layout) inside CTA `rank` of the cluster
__device__ __forceinline__ uint32_t map_to_cta(const void* p, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;\n" : "=r"(r) : "r"(smem_u32(p)), "r"(rank));
    return r;
}
__device__ __forceinline__ void st_cluster_f64(uint32_t addr, double v) {
    asm volatile("st.shared::cluster.f64 [%0], %1;\n" ::"r"(addr), "d"(v) : "memory");
}
__device__ __forceinline__ void st_cluster_u32(uint32_t addr, uint32_t v) {
    asm volatile("st.shared::cluster.u32 [%0], %1;\n" ::"r"(addr), "r"(v) : "memory");
}
// mailbox hand-shake between neighbouring warps of the cluster: the row travels as asynchronous DSMEM stores that
// complete transaction bytes on an mbarrier in the RECEIVER's shared memory (st.async ... complete_tx); the
// receiver arms the barrier with the expected byte count and waits on its phase -- no fences, no cluster barrier
__device__ __forceinline__ void st_async_f64(uint32_t addr, double v, uint32_t mbar) {
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b64 [%0], %1, [%2];\n" ::"r"(addr),
                 "l"(__double_as_longlong(v)), "r"(mbar)
                 : "memory");
}
__device__ __forceinline__ uint32_t ld_cluster_u32(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared::cluster.u32 %0, [%1];\n" : "=r"(v) : "r"(addr) : "memory");
    return v;
}

__global__ void __cluster_dims__(JC_CL, 1, 1) __launch_bounds__(JC_THREADS)
k_eigh_jacobi(int N, double* __restrict__ scratch, int* __restrict__ info) {
    __shared__ __align__(16) double slotO[JC_GPC][JC_SLOT];   // odd steps: position 2g+2 arriving at group g
    __shared__ __align__(16) double slotE[JC_GPC][JC_SLOT];   // even steps: position 2g arriving at group g
    __shared__ __align__(16) double park[JC_SLOT];            // position 0 rests here during odd steps
    __shared__ uint32_t s_again;                              // used in CTA 0 of the cluster
    __shared__ __align__(8) uint64_t barO[JC_GPC], barE[JC_GPC];   // transaction barriers of slotO / slotE
    double* Yg = scratch + eig_off_Y(N);
    if (scratch[eig_off_meta(N) + 1] != 0.0) return;          // factorisation failed (every CTA sees the same flag)
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t rank = cluster_ctarank();
    const int g = (int)rank * JC_GPC + warp;                  // this warp's pair of line positions: 2g, 2g+1
    const int Np = (N + 1) & ~1, G = Np / 2;
    const bool active = g < G;
    const double tol2 = 1.44e-32 * (double)N;                 // (1.2e-16 sqrt(N))^2
    // A sweep in which every rotated cosine was below 3.2e-9 is the last one: a rotation zeroes its own pair and disturbs the
    // inner product of another pair (i, k) by cos(i, j) cos(j, k), so whatever the <= N - 1 rotations of row i leave behind is
    // below N * 1e-17 <= 1.44e-15, the threshold itself.  Without this test every solve paid one more full sweep that only
    // confirmed that nothing is left to rotate (1 of ~10 at N = 132).  The rotation's tangent must be below 3.2e-9 as
    // well: two rows of nearly equal norm (a cluster of theta + sigma, e.g. every value of a pencil whose shift dominates)
    // turn by a large angle at a tiny cosine, which carries the other pairs' inner products over instead of shrinking them
    // (N = 144, spectrum [-1e-5, 1] at sigma = 1e5: stopping on the cosine alone left theta_min wrong by 1.3e-6).
    const double big2 = 1e-17;
    int big = 0;

    double ra[JC_E], rb[JC_E];                                // even configuration: ra = position 2g, rb = 2g+1
    double na = 0.0, nb = 0.0;
#pragma unroll
    for (int i = 0; i < JC_E; ++i) {
        ra[i] = active ? Yg[(size_t)(2 * g) * JC_LD + lane + 32 * i] : 0.0;
        rb[i] = active ? Yg[(size_t)(2 * g + 1) * JC_LD + lane + 32 * i] : 0.0;
    }
    // receivers of this warp's outgoing rows
    const uint32_t dstO = g >= 1 ? map_to_cta(&slotO[(g - 1) % JC_GPC][0], (uint32_t)((g - 1) / JC_GPC)) : 0u;
    const uint32_t dstE = g + 1 < G ? map_to_cta(&slotE[(g + 1) % JC_GPC][0], (uint32_t)((g + 1) / JC_GPC)) : 0u;
    const uint32_t again_addr = map_to_cta(&s_again, 0u);
    const uint32_t fdstO = g >= 1 ? map_to_cta(&barO[(g - 1) % JC_GPC], (uint32_t)((g - 1) / JC_GPC)) : 0u;
    const uint32_t fdstE = g + 1 < G ? map_to_cta(&barE[(g + 1) % JC_GPC], (uint32_t)((g + 1) / JC_GPC)) : 0u;
    if (lane == 0) {
        mbar_init(&barO[warp], 1);
        mbar_init(&barE[warp], 1);
        fence_barrier_init();
    }
    uint32_t phO = 0u, phE = 0u;                              // parity of the next phase of this warp's barriers
    constexpr uint32_t ROW_BYTES = (JC_LD + 1) * 8u;          // elements + |row|^2

    // rotate x (|x|^2 = nx) against y; returns 1 if a rotation was applied (all lanes of the warp call it)
    auto rotate = [&](bool enable, double (&x)[JC_E], double& nx, double (&y)[JC_E], double& ny) -> int {
        double g0 = 0.0, g1 = 0.0;
#pragma unroll
        for (int i = 0; i < JC_E; ++i) {
            if (i & 1) g1 = fma(x[i], y[i], g1);
            else g0 = fma(x[i], y[i], g0);
        }
        const double ga = warp_sum(g0 + g1);
        if (!(enable && ga * ga > tol2 * nx * ny)) return 0;
        // tan(theta) = 2 ga / (d + sign(d) sqrt(d^2 + 4 ga^2)),  d = ny - nx
        const double d = ny - nx;
        const double h = sqrt(fma(d, d, 4.0 * ga * ga));
        const double t = 2.0 * ga / (d + (d >= 0.0 ? h : -h));
        big |= ga * ga > big2 * nx * ny || t * t > big2;
        const double c = rsqrt(fma(t, t, 1.0)), sn = c * t;
#pragma unroll
        for (int i = 0; i < JC_E; ++i) {
            const double xv = x[i], yv = y[i];
            x[i] = fma(c, xv, -sn * yv);
            y[i] = fma(sn, xv, c * yv);
        }
        nx -= t * ga;
        ny += t * ga;
        return 1;
    };
    // Rows travel between neighbouring warps without a cluster-wide barrier.  A mailbox is never overwritten
    // early: the sender's next store into it is ordered after a row it receives from that same neighbour, which the
    // neighbour sends only after it has emptied the mailbox.
    auto send = [&](uint32_t dst, uint32_t bar, const double (&x)[JC_E], double nx) {
#pragma unroll
        for (int i = 0; i < JC_E; ++i) st_async_f64(dst + (uint32_t)(lane + 32 * i) * 8u, x[i], bar);
        if (lane == 0) st_async_f64(dst + (uint32_t)JC_LD * 8u, nx, bar);
    };
    auto wait_row = [&](uint64_t* bar, uint32_t& parity) {
        if (lane == 0) mbar_expect_tx(bar, ROW_BYTES);
        mbar_wait(bar, parity);
        parity ^= 1u;
    };
    auto recv = [&](const double* src, double (&x)[JC_E], double& nx) {
#pragma unroll
        for (int i = 0; i < JC_E; ++i) x[i] = src[lane + 32 * i];
        nx = src[JC_LD];
    };

    int sweep = 0;
    for (; sweep < 24; ++sweep) {
        if (rank == 0 && tid == 0) s_again = 0u;
        {   // refresh the norms (they are updated by -+ t*gamma inside a sweep)
            double qa = 0.0, qb = 0.0;
#pragma unroll
            for (int i = 0; i < JC_E; ++i) { qa = fma(ra[i], ra[i], qa); qb = fma(rb[i], rb[i], qb); }
            na = warp_sum(qa);
            nb = warp_sum(qb);
        }
        cluster_sync_all();
        int rotated = 0;
        for (int step = 0; step < Np; step += 2) {
            // even step: positions (2g, 2g+1) = (ra, rb); afterwards the rows trade places:
            // position 2g is in rb, position 2g+1 in ra
            rotated |= rotate(active, ra, na, rb, nb);
            // odd step: position 2g (rb) goes to the left neighbour; position 2g+2 arrives in rb
            if (active) {
                if (g == 0) {
#pragma unroll
                    for (int i = 0; i < JC_E; ++i) park[lane + 32 * i] = rb[i];
                    if (lane == 0) park[JC_LD] = nb;
                    __syncwarp();
                } else {
                    send(dstO, fdstO, rb, nb);
                }
                if (g < G - 1) {
                    wait_row(&barO[warp], phO);
                    recv(&slotO[warp][0], rb, nb);
                } else {                                       // beyond the end of the line: a zero row
#pragma unroll
                    for (int i = 0; i < JC_E; ++i) rb[i] = 0.0;
                    nb = 0.0;
                }
            }
            rotated |= rotate(active && g < G - 1, ra, na, rb, nb);           // positions (2g+1, 2g+2)
            // trade places: position 2g+1 is now in rb, position 2g+2 in ra -- except for the last group,
            // which keeps its row at position 2g+1
            if (active && g == G - 1) {
#pragma unroll
                for (int i = 0; i < JC_E; ++i) { const double tv = ra[i]; ra[i] = rb[i]; rb[i] = tv; }
                const double tv = na; na = nb; nb = tv;
            }
            // next even step: position 2g+2 (ra) goes to the right neighbour; position 2g arrives in ra
            if (active) {
                if (g + 1 < G) send(dstE, fdstE, ra, na);
                if (g == 0) {
                    recv(park, ra, na);
                } else {
                    wait_row(&barE[warp], phE);
                    recv(&slotE[warp][0], ra, na);
                }
            }
        }
        (void)rotated;
        if (big && lane == 0) st_cluster_u32(again_addr, 1u);   // `big` is warp-uniform (gamma and the norms are)
        cluster_sync_all();
        const uint32_t again = ld_cluster_u32(again_addr);
        cluster_sync_all();                                    // everybody has read the flag before it is reset
        big = 0;
        if (!again) break;                                     // nothing rotated, or only cosines below 3.2e-9: converged
    }
    if (active) {
#pragma unroll
        for (int i = 0; i < JC_E; ++i) {
            Yg[(size_t)(2 * g) * JC_LD + lane + 32 * i] = ra[i];
            Yg[(size_t)(2 * g + 1) * JC_LD + lane + 32 * i] = rb[i];
        }
    }
    if (rank == 0 && tid == 0) info[1] = sweep + 1;
    cluster_sync_all();                                        // no CTA leaves while DSMEM traffic may be pending
}

// Eigenvalues = |row|^2 - sigma, ascending rank (every CTA recomputes the 144 norms: cheap), then for the rows of this
// CTA (one warp each)  c_j = D R^-T row_j:  x R = y_j by back substitution, lane l keeps x_k for k = l (mod 32).
__global__ void __launch_bounds__(ES_WARPS * 32)
k_eigh_finish(int N, const __grid_constant__ EigIdx ix, double* __restrict__ theta, double* __restrict__ C, int64_t ldc,
              const double* __restrict__ scratch, int* __restrict__ info) {
    __shared__ double s_theta[EIG_MAXN + 2];
    __shared__ int s_rank[EIG_MAXN + 2];
    __shared__ int s_hole;
    const int tid = threadIdx.x, nt = blockDim.x, warp = tid >> 5, lane = tid & 31;
    const double* __restrict__ RT = scratch + eig_off_RT(N);
    const double* __restrict__ invR = scratch + eig_off_invR(N);
    const double* __restrict__ Yg = scratch + eig_off_Y(N);
    const double* __restrict__ scale = scratch + eig_off_scale(N);
    const double* meta = scratch + eig_off_meta(N);
    if (meta[1] != 0.0) return;                  // info was set by k_eigh_solve
    const double sigma = meta[0];
    const int Np = (N + 1) & ~1;
    // norms of all line positions; an odd N leaves exactly one zero row somewhere on the line
    for (int p = warp; p < Np; p += nt / 32) {
        double v = 0.0;
        for (int e = lane; e < N; e += 32) { const double a = Yg[(size_t)p * JC_LD + e]; v = fma(a, a, v); }
        v = warp_sum(v);
        if (lane == 0) s_theta[p] = v;
    }
    __syncthreads();
    if (tid == 0) {
        int ph = Np;
        if (Np > N)
            for (int p = 0; p < Np; ++p)
                if (s_theta[p] == 0.0) { ph = p; break; }
        s_hole = ph;
    }
    __syncthreads();
    const int ph = s_hole;
    // compact: row j of the problem sits at line position j + (j >= ph)
    double mine = 0.0;
    if (tid < N) mine = s_theta[tid + (tid >= ph ? 1 : 0)] - sigma;
    __syncthreads();
    if (tid < N) s_theta[tid] = mine;
    __syncthreads();
    for (int j = tid; j < N; j += nt) {
        const double tj = s_theta[j];
        int rk = 0;
        for (int i = 0; i < N; ++i) {
            const double ti = s_theta[i];
            rk += (ti < tj) || (ti == tj && i < j);
        }
        s_rank[j] = rk;
        if (blockIdx.x == 0) theta[rk] = tj;
    }
    __syncthreads();
    const int j = blockIdx.x * ES_WARPS + warp;
    if (j < N) {
        const double* yrow = Yg + (size_t)(j + (j >= ph ? 1 : 0)) * JC_LD;
        double x[JC_E];
#pragma unroll
        for (int t = 0; t < JC_E; ++t) { const int k = lane + 32 * t; x[t] = k < N ? yrow[k] : 0.0; }
        // x_k = (y_k - sum_{q > k} x_q R[q][k]) / R[k][k], k = N-1 .. 0; at step k the lanes hold final x_q for q > k.
        // Row k of R^T and the reciprocal pivot are fetched two steps ahead of the reduction chain.
        double c0[JC_E], c1[JC_E], c2[JC_E], p0 = 0.0, p1 = 0.0, p2 = 0.0;
        auto load_row = [&](int k, double (&c)[JC_E], double& pv) {
            if (k >= 0) {
#pragma unroll
                for (int t = 0; t < JC_E; ++t) { const int q = lane + 32 * t; c[t] = (q > k && q < N) ? __ldg(RT + (size_t)k * N + q) : 0.0; }
                pv = __ldg(invR + k);
            }
        };
        load_row(N - 1, c0, p0);
        load_row(N - 2, c1, p1);
#pragma unroll
        for (int tk = JC_E - 1; tk >= 0; --tk) {     // k = 32 tk + kk: the register that holds x_k is static
            for (int kk = 31; kk >= 0; --kk) {
                const int k = 32 * tk + kk;
                if (k >= N) continue;                // warp-uniform
                load_row(k - 2, c2, p2);
                double s = 0.0;
#pragma unroll
                for (int t = 0; t < JC_E; ++t) s = fma(x[t], c0[t], s);      // c0 is zero outside q in (k, N)
                s = warp_sum(s);
                if (lane == kk) x[tk] = (x[tk] - s) * p0;
#pragma unroll
                for (int t = 0; t < JC_E; ++t) { c0[t] = c1[t]; c1[t] = c2[t]; }
                p0 = p1; p1 = p2;
            }
        }
        const int col = s_rank[j];
#pragma unroll
        for (int t = 0; t < JC_E; ++t) {
            const int k = lane + 32 * t;
            if (k < N) C[(int64_t)ix.v[k] * ldc + col] = x[t] * scale[k];
        }
    }
    if (blockIdx.x == 0 && tid == 0) info[0] = 0;
}

int eigh_generalized_f64(const double* GK, const double* GM, int N, int64_t ldg, const int* idx_host, double sigma,
                         double* theta, double* C, int64_t ldc, double* scratch, int* info, cudaStream_t stream) {
    DS_REQUIRE(N >= 2 && N <= EIG_MAXN, "eigh_generalized: N=%d must be in [2,%d]", N, EIG_MAXN);
    DS_REQUIRE(GK && GM && theta && C && scratch && info, "eigh_generalized: null argument");
    ProfScope prof(PROF_EIGH, stream);
    EigIdx ix;
    for (int i = 0; i < EIG_MAXN; ++i) ix.v[i] = (short)(i < N ? (idx_host ? idx_host[i] : i) : 0);
    const size_t smem = ((size_t)N * (N + 2) + 2 * N + 2) * sizeof(double) + (N + 4) * sizeof(int);
    static bool attr = false;
    if (!attr) {
        const int mx = (int)(((size_t)EIG_MAXN * (EIG_MAXN + 2) + 2 * EIG_MAXN + 2) * sizeof(double) + (EIG_MAXN + 4) * sizeof(int));
        DS_CUDA(cudaFuncSetAttribute(k_eigh_chol, cudaFuncAttributeMaxDynamicSharedMemorySize, mx));
        attr = true;
    }
    k_eigh_chol<<<2, EIG_THREADS, smem, stream>>>(GK, GM, N, ldg, ix, sigma, scratch);
    DS_LAUNCH_CHECK();
    k_eigh_solve<<<JC_LD / ES_WARPS, ES_WARPS * 32, 0, stream>>>(N, scratch, info);
    DS_LAUNCH_CHECK();
    k_eigh_jacobi<<<JC_CL, JC_THREADS, 0, stream>>>(N, scratch, info);
    DS_LAUNCH_CHECK();
    k_eigh_finish<<<(N + ES_WARPS - 1) / ES_WARPS, ES_WARPS * 32, 0, stream>>>(N, ix, theta, C, ldc, scratch, info);
    DS_LAUNCH_CHECK();
    return DS_OK;
}

}  // namespace ds

using namespace ds;

extern "C" int64_t ds_eigh_scratch_elems(int N) { return eigh_scratch_elems(N); }

extern "C" int ds_eigh_generalized_f64(const double* GK, const double* GM, int N, int64_t ldg, double sigma,
                                       double* theta, double* C, int64_t ldc, double* scratch, int* info,
                                       void* stream) {
    return eigh_generalized_f64(GK, GM, N, ldg, nullptr, sigma, theta, C, ldc, scratch, info, (cudaStream_t)stream);
}

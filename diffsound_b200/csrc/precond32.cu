// FP32 preconditioner kernels of the eigensolver: block-CSR SpMM on 48-byte block records with an
// L1-resident gather, fused with the Chebyshev / residual epilogue.
//
// Reference behaviour replaced: none one-to-one -- the reference factorises K - sigma M on the CPU
// (SciPy SuperLU inside eigsh, /root/reference/src/diffelastic/diff_model.py:356-358) and its own
// LOBPCG takes an optional dense/callable preconditioner `iK` (src/lobpcg/_lobpcg.py:453,475).
// Here the preconditioner T ~ K^-1 is a fixed polynomial / V-cycle in the SpMM below, evaluated in
// FP32 (LOBPCG only needs an approximate SPD operator; the eigenpairs themselves stay FP64).
//
// Layout: one record per 3x3 block, 12 x 4 bytes = {k00 k01 k02 k10 | k11 k12 k20 k21 | k22 bcol - -}
// (three aligned 128-bit loads; the 8 bytes of padding cost 20 % more record bytes but halve the L1
// wavefronts of the record loads against unaligned 40-byte records read as five 64-bit words),
// in block-CSR order of the level's own node numbering (a Morton curve through the node coordinates
// when the caller supplies them: consecutive rows then gather overlapping sets of X rows).  Dense
// blocks are row-major fp32 (n x c), c in {16, 32, 48, 64}; the 3 rows of a node are contiguous
// (3c floats), so a gathered neighbour is one 192..768-byte run.
//
// Mapping (k_spmm32v): one 1024-thread CTA per SM sweeps a contiguous chunk of node rows; a warp owns
// one node row at a time (rows are handed out through a shared-memory ticket, so long and short
// rows balance and the ~32 rows in flight are neighbours); LPR lanes cover the c columns (CPT
// columns each, 64/128-bit loads), the 32/LPR lane groups walk alternate blocks of the row and are
// combined by a butterfly at the end.  Lane groups 0..2 then apply the epilogue for component 0..2
// of the node.  The gathered X rows live in the SM's L1 (no shared memory is used, all 256 KB are
// L1); records, R and Zprev are streamed once with L1::no_allocate behind bulk L2 prefetches.
#include "common.cuh"
#include "../../include/diffsound_sm100.h"
#include "kernels.cuh"
#include "ptx.cuh"
#include <algorithm>
#include <utility>
#include <cstring>
#include <cub/cub.cuh>

namespace ds {

constexpr int S32_REC_BYTES = 48;           // 9 fp32 values + column id + 8 bytes of padding: three aligned 128-bit loads
constexpr int S32_REC_WORDS = S32_REC_BYTES / 4;

enum { S32_PLAIN = S32_MODE_PLAIN, S32_RESID = S32_MODE_RESID, S32_CHEB = S32_MODE_CHEB };

template <int VEC> struct VecT;
template <> struct VecT<2> { using type = float2; };
template <> struct VecT<4> { using type = float4; };

template <int VEC>
__device__ __forceinline__ void ld_vec(const float* p, float* out) {
    if constexpr (VEC == 4) {
        float4 v = __ldg(reinterpret_cast<const float4*>(p));
        out[0] = v.x; out[1] = v.y; out[2] = v.z; out[3] = v.w;
    } else {
        float2 v = __ldg(reinterpret_cast<const float2*>(p));
        out[0] = v.x; out[1] = v.y;
    }
}
// plain (coherent) load: for buffers the same kernel also writes (Zprev may alias Out)
template <int VEC>
__device__ __forceinline__ void ld_vec_plain(const float* p, float* out) {
    if constexpr (VEC == 4) {
        float4 v = *reinterpret_cast<const float4*>(p);
        out[0] = v.x; out[1] = v.y; out[2] = v.z; out[3] = v.w;
    } else {
        float2 v = *reinterpret_cast<const float2*>(p);
        out[0] = v.x; out[1] = v.y;
    }
}
template <int VEC>
__device__ __forceinline__ void st_vec(float* p, const float* v) {
    if constexpr (VEC == 4) *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
    else *reinterpret_cast<float2*>(p) = make_float2(v[0], v[1]);
}

// Column ownership of lane l (of LPR) inside a C = LPR * CPT wide row: 128-bit chunk [4l, 4l+4) and, for
// CPT = 6 / 8, a second 64- / 128-bit chunk behind the first 4*LPR columns -- so that the LPR lanes of a
// group always touch CONTIGUOUS bytes (a lane owning CPT contiguous columns makes every load
// instruction of the group hit all sectors of the row: 3x sector over-fetch measured at c = 48).
template <int LPR, int CPT>
__device__ __forceinline__ void ld_row(const float* row, int l, float* out) {
    ld_vec<4>(row + 4 * l, out);
    if constexpr (CPT == 6) ld_vec<2>(row + 4 * LPR + 2 * l, out + 4);
    if constexpr (CPT == 8) ld_vec<4>(row + 4 * LPR + 4 * l, out + 4);
}
template <int LPR, int CPT>
__device__ __forceinline__ void ld_row_plain(const float* row, int l, float* out) {
    ld_vec_plain<4>(row + 4 * l, out);
    if constexpr (CPT == 6) ld_vec_plain<2>(row + 4 * LPR + 2 * l, out + 4);
    if constexpr (CPT == 8) ld_vec_plain<4>(row + 4 * LPR + 4 * l, out + 4);
}
template <int LPR, int CPT>
__device__ __forceinline__ void st_row(float* row, int l, const float* v) {
    st_vec<4>(row + 4 * l, v);
    if constexpr (CPT == 6) st_vec<2>(row + 4 * LPR + 2 * l, v + 4);
    if constexpr (CPT == 8) st_vec<4>(row + 4 * LPR + 4 * l, v + 4);
}

// Row-partitioned operation (one slab of node rows per GPU): the column id of a record is packed as
// owner << 28 | node index inside the owner's slab, and the gathered block is addressed through a
// table of per-rank base pointers -- the peers' slabs are mapped into this process (CUDA IPC) and read
// over NVLink by plain loads.
struct PeerTable {
    const float* p[8];
};
template <bool PEER, int C>
__device__ __forceinline__ const float* node_rows(const float* __restrict__ X, const PeerTable& tab, uint32_t j) {
    if constexpr (PEER) return tab.p[j >> 28] + (int64_t)(j & 0x0fffffffu) * (3 * C);
    else return X + (int64_t)(int)j * (3 * C);
}

// ---------------------------------------------------------------------------------------------
// v2: L1-resident gather.  One 1024-thread CTA per SM sweeps a CONTIGUOUS chunk of node rows (chunks
// balanced by blocks + rows), its 32 warps taking consecutive rows through a shared-memory ticket, so
// the X rows gathered by the ~32 rows in flight overlap heavily and are served by the SM's L1
// (no shared-memory staging: the whole 256 KB stays L1).  Everything that is read once -- block
// records, R, Zprev -- is loaded with L1::no_allocate so it does not evict the gathered rows, and
// is pulled into L2 64 rows ahead by bulk prefetches (cp.async.bulk.prefetch.L2), which takes the
// DRAM latency off the warps.  The 3x3 block FMAs are packed (FFMA2: fma.rn.f32x2 with the K entry
// broadcast), halving the dominant instruction count.
// ---------------------------------------------------------------------------------------------
constexpr int S32V_THREADS = 1024;
constexpr int S32V_PF = 64;                  // rows of look-ahead of the L2 prefetch

typedef unsigned long long u64;

__device__ __forceinline__ uint4 ldg_na_u4(const uint4* p) {
    uint4 v;
    asm("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
    return v;
}
__device__ __forceinline__ uint32_t ldg_na_u32(const uint32_t* p) {
    uint32_t v;
    asm("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ void ldg_v2u64(const float* p, u64& a, u64& b) {
    asm("ld.global.nc.v2.u64 {%0,%1}, [%2];" : "=l"(a), "=l"(b) : "l"(p));
}
__device__ __forceinline__ u64 ldg_u64(const float* p) {
    u64 a;
    asm("ld.global.nc.u64 %0, [%1];" : "=l"(a) : "l"(p));
    return a;
}
__device__ __forceinline__ void prefetch_l2_bulk(const void* p, uint32_t bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes) : "memory");
}
__device__ __forceinline__ void prefetch_l1(const void* p) {
    asm volatile("prefetch.global.L1 [%0];" ::"l"(p));
}
__device__ __forceinline__ void prefetch_l2(const void* p) {
    asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
}
__device__ __forceinline__ void ffma2(u64& acc, float k, u64 x) {
    u64 kk;
    asm("mov.b64 %0, {%1, %1};" : "=l"(kk) : "f"(k));
    asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc) : "l"(kk), "l"(x));
}
__device__ __forceinline__ u64 fadd2(u64 a, u64 b) {
    u64 r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ void unpack2(u64 v, float& a, float& b) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v));
}

// the lane's CPT columns of one fp32 row as CPT/2 packed pairs (same ownership as ld_row)
template <int LPR, int CPT>
__device__ __forceinline__ void ld_row2(const float* row, int l, u64* out) {
    ldg_v2u64(row + 4 * l, out[0], out[1]);
    if constexpr (CPT == 6) out[2] = ldg_u64(row + 4 * LPR + 2 * l);
    if constexpr (CPT == 8) ldg_v2u64(row + 4 * LPR + 4 * l, out[2], out[3]);
}
// streamed-once variants (R: read-only; Zprev: may alias Out)
template <int LPR, int CPT>
__device__ __forceinline__ void ld_row_stream(const float* row, int l, float* out) {
    asm("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
        : "=f"(out[0]), "=f"(out[1]), "=f"(out[2]), "=f"(out[3]) : "l"(row + 4 * l));
    if constexpr (CPT == 6)
        asm("ld.global.nc.L1::no_allocate.v2.f32 {%0,%1}, [%2];" : "=f"(out[4]), "=f"(out[5]) : "l"(row + 4 * LPR + 2 * l));
    if constexpr (CPT == 8)
        asm("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
            : "=f"(out[4]), "=f"(out[5]), "=f"(out[6]), "=f"(out[7]) : "l"(row + 4 * LPR + 4 * l));
}
template <int LPR, int CPT>
__device__ __forceinline__ void ld_row_stream_plain(const float* row, int l, float* out) {
    asm volatile("ld.global.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(out[0]), "=f"(out[1]), "=f"(out[2]), "=f"(out[3]) : "l"(row + 4 * l) : "memory");
    if constexpr (CPT == 6)
        asm volatile("ld.global.L1::no_allocate.v2.f32 {%0,%1}, [%2];"
                     : "=f"(out[4]), "=f"(out[5]) : "l"(row + 4 * LPR + 2 * l) : "memory");
    if constexpr (CPT == 8)
        asm volatile("ld.global.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                     : "=f"(out[4]), "=f"(out[5]), "=f"(out[6]), "=f"(out[7]) : "l"(row + 4 * LPR + 4 * l) : "memory");
}
template <int LPR, int CPT>
__device__ __forceinline__ void st_row_stream(float* row, int l, const float* v) {
    asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(row + 4 * l), "f"(v[0]), "f"(v[1]), "f"(v[2]),
                 "f"(v[3]) : "memory");
    if constexpr (CPT == 6)
        asm volatile("st.global.L1::no_allocate.v2.f32 [%0], {%1,%2};" ::"l"(row + 4 * LPR + 2 * l), "f"(v[4]), "f"(v[5])
                     : "memory");
    if constexpr (CPT == 8)
        asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(row + 4 * LPR + 4 * l), "f"(v[4]),
                     "f"(v[5]), "f"(v[6]), "f"(v[7]) : "memory");
}

// acc[c][:] += K[c][:] . X[3j..3j+2][cols of this lane] for one block record read from global
template <int LPR, int CPT, bool PEER>
__device__ __forceinline__ void block_fma_v(const uint4* __restrict__ r, uint32_t ja, const float* __restrict__ X,
                                            const PeerTable& tab, int l, u64 (&acc)[3][CPT / 2]) {
    constexpr int C = LPR * CPT, NP = CPT / 2;
    const float* xr = node_rows<PEER, C>(X, tab, ja);
    const uint4 a2 = ldg_na_u4(r + 2), a0 = ldg_na_u4(r), a1 = ldg_na_u4(r + 1);
    u64 x[3][NP];
#pragma unroll
    for (int d = 0; d < 3; ++d) ld_row2<LPR, CPT>(xr + d * C, l, x[d]);
    const float k[9] = {__uint_as_float(a0.x), __uint_as_float(a0.y), __uint_as_float(a0.z),
                        __uint_as_float(a0.w), __uint_as_float(a1.x), __uint_as_float(a1.y),
                        __uint_as_float(a1.z), __uint_as_float(a1.w), __uint_as_float(a2.x)};
#pragma unroll
    for (int c = 0; c < 3; ++c)
#pragma unroll
        for (int d = 0; d < 3; ++d)
#pragma unroll
            for (int t = 0; t < NP; ++t) ffma2(acc[c][t], k[3 * c + d], x[d][t]);
}

template <int LPR, int CPT, bool PEER>
__device__ __forceinline__ void block_fma2_v(const uint4* __restrict__ ra, const uint4* __restrict__ rb, uint32_t ja,
                                             uint32_t jb, const float* __restrict__ X, const PeerTable& tab, int l,
                                             u64 (&acc)[3][CPT / 2]) {
    constexpr int C = LPR * CPT, NP = CPT / 2;
    // the column ids arrive from the previous iteration (software pipelining): the X loads go out together with the
    // loads of the K values instead of one L2 round trip behind them
    const float* xa = node_rows<PEER, C>(X, tab, ja);
    const float* xb = node_rows<PEER, C>(X, tab, jb);
    const uint4 a2 = ldg_na_u4(ra + 2), b2 = ldg_na_u4(rb + 2);
    const uint4 a0 = ldg_na_u4(ra), a1 = ldg_na_u4(ra + 1);
    const uint4 b0 = ldg_na_u4(rb), b1 = ldg_na_u4(rb + 1);
    u64 x[3][NP], y[3][NP];
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        ld_row2<LPR, CPT>(xa + d * C, l, x[d]);
        ld_row2<LPR, CPT>(xb + d * C, l, y[d]);
    }
    {
        const float k[9] = {__uint_as_float(a0.x), __uint_as_float(a0.y), __uint_as_float(a0.z),
                            __uint_as_float(a0.w), __uint_as_float(a1.x), __uint_as_float(a1.y),
                            __uint_as_float(a1.z), __uint_as_float(a1.w), __uint_as_float(a2.x)};
#pragma unroll
        for (int c = 0; c < 3; ++c)
#pragma unroll
            for (int d = 0; d < 3; ++d)
#pragma unroll
                for (int t = 0; t < NP; ++t) ffma2(acc[c][t], k[3 * c + d], x[d][t]);
    }
    {
        const float k[9] = {__uint_as_float(b0.x), __uint_as_float(b0.y), __uint_as_float(b0.z),
                            __uint_as_float(b0.w), __uint_as_float(b1.x), __uint_as_float(b1.y),
                            __uint_as_float(b1.z), __uint_as_float(b1.w), __uint_as_float(b2.x)};
#pragma unroll
        for (int c = 0; c < 3; ++c)
#pragma unroll
            for (int d = 0; d < 3; ++d)
#pragma unroll
                for (int t = 0; t < NP; ++t) ffma2(acc[c][t], k[3 * c + d], y[d][t]);
    }
}

template <int LPR, int CPT, int MODE, bool PEER>
__global__ void __launch_bounds__(S32V_THREADS, 1)
k_spmm32v(const int32_t* __restrict__ brow, const uint4* __restrict__ rec, const int32_t* __restrict__ chunk_row,
          const float* __restrict__ X, const float* __restrict__ R, const float* __restrict__ invD,
          const float* Zprev, float* Out, float ab, float cc, int prefetch, const __grid_constant__ PeerTable tab) {
    constexpr int C = LPR * CPT;
    constexpr int NG = 32 / LPR;
    constexpr int NP = CPT / 2;
    __shared__ int s_ticket;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane / LPR, l = lane % LPR;
    const int r_lo = chunk_row[blockIdx.x], r_hi = chunk_row[blockIdx.x + 1];
    if (tid == 0) s_ticket = 0;

    // pull what row r streams exactly once into L2 (lane 0 of the calling warp)
    auto prefetch_row = [&](int r) {
        const int64_t b0 = brow[r], b1 = brow[r + 1];
        if (b1 > b0) {
            prefetch_l2_bulk(reinterpret_cast<const unsigned char*>(rec) + b0 * S32_REC_BYTES,
                             (uint32_t)((b1 - b0) * S32_REC_BYTES));
        }
        const int64_t ob = (int64_t)3 * r * C;
        if (MODE != S32_PLAIN) prefetch_l2_bulk(R + ob, 3 * C * 4);
        if (MODE == S32_CHEB) {
            prefetch_l2_bulk(Zprev + ob, 3 * C * 4);
            prefetch_l2(invD + 9 * (int64_t)r);
        }
        if ((r & 15) == 0) prefetch_l2(brow + min(r + 2 * S32V_PF, r_hi));      // the row pointers themselves
    };
    if (lane == 0 && prefetch) {
        if (r_lo + warp < r_hi) prefetch_row(r_lo + warp);
        if (r_lo + 32 + warp < r_hi) prefetch_row(r_lo + 32 + warp);
    }
    __syncthreads();

    for (;;) {
        int rr = 0;
        if (lane == 0) rr = atomicAdd(&s_ticket, 1);
        rr = __shfl_sync(0xffffffffu, rr, 0);
        const int row = r_lo + rr;
        if (row >= r_hi) break;
        if (lane == 0 && prefetch && row + S32V_PF < r_hi) prefetch_row(row + S32V_PF);
        const int rb0 = brow[row], rb1 = brow[row + 1];
        u64 acc[3][NP];
#pragma unroll
        for (int c = 0; c < 3; ++c)
#pragma unroll
            for (int t = 0; t < NP; ++t) acc[c][t] = 0ull;
        int p = rb0 + g;
        const uint32_t* colw = reinterpret_cast<const uint32_t*>(rec) + 9;         // word 9 of a record = column id
        uint32_t ja = p < rb1 ? ldg_na_u32(colw + (int64_t)S32_REC_WORDS * p) : 0u;
        uint32_t jb = p + NG < rb1 ? ldg_na_u32(colw + (int64_t)S32_REC_WORDS * (p + NG)) : 0u;
        for (; p + NG < rb1; p += 2 * NG) {
            const uint32_t jan = p + 2 * NG < rb1 ? ldg_na_u32(colw + (int64_t)S32_REC_WORDS * (p + 2 * NG)) : 0u;
            const uint32_t jbn = p + 3 * NG < rb1 ? ldg_na_u32(colw + (int64_t)S32_REC_WORDS * (p + 3 * NG)) : 0u;
            block_fma2_v<LPR, CPT, PEER>(rec + (int64_t)3 * p, rec + (int64_t)3 * (p + NG), ja, jb, X, tab, l, acc);
            ja = jan;
            jb = jbn;
        }
        if (p < rb1) block_fma_v<LPR, CPT, PEER>(rec + (int64_t)3 * p, ja, X, tab, l, acc);
#pragma unroll
        for (int off = LPR; off < 32; off <<= 1)
#pragma unroll
            for (int c = 0; c < 3; ++c)
#pragma unroll
                for (int t = 0; t < NP; ++t) acc[c][t] = fadd2(acc[c][t], __shfl_xor_sync(0xffffffffu, acc[c][t], off));
        if (g < 3) {
            const int64_t o = ((int64_t)3 * row + g) * C;          // output row of this lane group
            float a[3][CPT];
#pragma unroll
            for (int c = 0; c < 3; ++c)
#pragma unroll
                for (int t = 0; t < NP; ++t) unpack2(acc[c][t], a[c][2 * t], a[c][2 * t + 1]);
            float v[CPT];
            if (MODE == S32_PLAIN) {
#pragma unroll
                for (int t = 0; t < CPT; ++t) v[t] = g == 0 ? a[0][t] : (g == 1 ? a[1][t] : a[2][t]);
            } else if (MODE == S32_RESID) {
                float rv[CPT];
                ld_row_stream<LPR, CPT>(R + o, l, rv);
#pragma unroll
                for (int t = 0; t < CPT; ++t) v[t] = rv[t] - (g == 0 ? a[0][t] : (g == 1 ? a[1][t] : a[2][t]));
            } else {
                const float d0 = __ldg(invD + 9 * (int64_t)row + 3 * g), d1 = __ldg(invD + 9 * (int64_t)row + 3 * g + 1),
                            d2 = __ldg(invD + 9 * (int64_t)row + 3 * g + 2);
                float r0v[CPT], r1v[CPT], r2v[CPT], z[CPT], zp[CPT];
                const int64_t ob = (int64_t)3 * row * C;
                ld_row_stream<LPR, CPT>(R + ob, l, r0v);
                ld_row_stream<LPR, CPT>(R + ob + C, l, r1v);
                ld_row_stream<LPR, CPT>(R + ob + 2 * C, l, r2v);
                ld_row<LPR, CPT>(X + o, l, z);
                ld_row_stream_plain<LPR, CPT>(Zprev + o, l, zp);
#pragma unroll
                for (int t = 0; t < CPT; ++t) {
                    const float dr = d0 * (r0v[t] - a[0][t]) + d1 * (r1v[t] - a[1][t]) + d2 * (r2v[t] - a[2][t]);
                    v[t] = z[t] + ab * (z[t] - zp[t]) + cc * dr;
                }
            }
            st_row_stream<LPR, CPT>(Out + o, l, v);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Persistent Chebyshev solve for a level that fits on chip (the P1 coarse operator: ~25 MB of records):
// ALL `degree` steps of z = p(invD A) invD r run in ONE cooperative launch, one 1024-thread CTA per SM.
// Every CTA copies the block records of its row chunk into shared memory once (~170 KB) and reuses them
// in every step; the steps are separated by a grid barrier (one atomic per CTA on a global counter + an
// acquire fence that also drops the stale L1 lines of the iterate).  Per step the only traffic left is the
// gather of the iterate from L2.  Replaces `degree` launches of k_spmm32v whose time at this size (~40 us
// each) was launch + dependent-latency, not bandwidth.
// ---------------------------------------------------------------------------------------------
constexpr int CHP_MAX_DEGREE = 64;
struct ChebCoef {
    float cc0;                       // z_1 = cc0 invD r
    float ab[CHP_MAX_DEGREE];        // step k = 1 .. degree-1
    float cc[CHP_MAX_DEGREE];
    int degree;
};

__device__ __forceinline__ unsigned ld_acquire_gpu_u32(const unsigned* p) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
// coherent (L1-cacheable within a step, invalidated by the fence of the grid barrier) loads of the iterate
__device__ __forceinline__ void ld_v2u64_coh(const float* p, u64& a, u64& b) {
    asm volatile("ld.global.v2.u64 {%0,%1}, [%2];" : "=l"(a), "=l"(b) : "l"(p) : "memory");
}
__device__ __forceinline__ u64 ld_u64_coh(const float* p) {
    u64 a;
    asm volatile("ld.global.u64 %0, [%1];" : "=l"(a) : "l"(p) : "memory");
    return a;
}
template <int LPR, int CPT>
__device__ __forceinline__ void ld_row2_coh(const float* row, int l, u64* out) {
    ld_v2u64_coh(row + 4 * l, out[0], out[1]);
    if constexpr (CPT == 6) out[2] = ld_u64_coh(row + 4 * LPR + 2 * l);
    if constexpr (CPT == 8) ld_v2u64_coh(row + 4 * LPR + 4 * l, out[2], out[3]);
}

// all CTAs of the (cooperative) grid; `target` = barriers passed so far * gridDim.x.  A CTA that waits longer
// than ~1 s raises *err and leaves (the results are then garbage, but the device does not hang).
__device__ __forceinline__ void grid_barrier(unsigned* ctr, unsigned target, int* err, int* ticket) {
    __syncthreads();                 // every warp of this CTA has left the row loop of the step
    if (threadIdx.x == 0) {
        *ticket = 0;                 // only now may the row ticket be rewound
        __threadfence();             // release: this CTA's rows of the new iterate (cumulative over the bar.sync)
        atomicAdd(ctr, 1u);
        const long long t0 = clock64();
        while (ld_acquire_gpu_u32(ctr) < target) {
            if (*(volatile int*)err || clock64() - t0 > (2ll << 30)) { *err = 1; break; }
        }
        __threadfence();             // acquire; the gpu-scope fence also invalidates this SM's L1 (CCTL.IVALL), so the
                                     // stale lines of the buffer that now holds the new iterate are dropped
    }
    __syncthreads();
}

template <int LPR, int CPT>
__global__ void __launch_bounds__(S32V_THREADS, 1)
k_cheb32_persistent(const int32_t* __restrict__ brow, const uint4* __restrict__ rec, const int32_t* __restrict__ chunk_row,
                    const float* __restrict__ R, const float* __restrict__ invD, float* Za, float* Zb,
                    const __grid_constant__ ChebCoef coef, int smem_records, unsigned* gbar, int* err) {
    constexpr int C = LPR * CPT;
    constexpr int NG = 32 / LPR;
    constexpr int NP = CPT / 2;
    extern __shared__ __align__(16) uint4 srec[];           // records of this chunk (first smem_records of them)
    __shared__ int s_ticket;
    const int tid = threadIdx.x, lane = tid & 31;
    const int g = lane / LPR, l = lane % LPR;
    const int r_lo = chunk_row[blockIdx.x], r_hi = chunk_row[blockIdx.x + 1];
    const int rec_lo = brow[r_lo], rec_hi = brow[r_hi];
    const int n_s = min(rec_hi - rec_lo, smem_records);
    for (int i = tid; i < 3 * n_s; i += S32V_THREADS) srec[i] = __ldg(rec + (int64_t)3 * rec_lo + i);
    const int s_hi = rec_lo + n_s;                           // records [rec_lo, s_hi) are in shared memory
    // ---- step 0: z_1 = cc0 invD r on the own rows -> Za
    for (int idx = tid; idx < (r_hi - r_lo) * (C / 4); idx += S32V_THREADS) {
        const int row = r_lo + idx / (C / 4), q = idx % (C / 4);
        const float4 r0 = __ldg(reinterpret_cast<const float4*>(R + (int64_t)3 * row * C) + q);
        const float4 r1 = __ldg(reinterpret_cast<const float4*>(R + ((int64_t)3 * row + 1) * C) + q);
        const float4 r2 = __ldg(reinterpret_cast<const float4*>(R + ((int64_t)3 * row + 2) * C) + q);
        const float* d = invD + 9 * (int64_t)row;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const float d0 = coef.cc0 * __ldg(d + 3 * c), d1 = coef.cc0 * __ldg(d + 3 * c + 1), d2 = coef.cc0 * __ldg(d + 3 * c + 2);
            float4 v;
            v.x = d0 * r0.x + d1 * r1.x + d2 * r2.x;
            v.y = d0 * r0.y + d1 * r1.y + d2 * r2.y;
            v.z = d0 * r0.z + d1 * r1.z + d2 * r2.z;
            v.w = d0 * r0.w + d1 * r1.w + d2 * r2.w;
            reinterpret_cast<float4*>(Za + ((int64_t)3 * row + c) * C)[q] = v;
        }
    }
    float* X = Za;      // z_k
    float* Zp = Zb;     // z_{k-1}, overwritten by z_{k+1}
    unsigned passed = 0;
    for (int k = 1; k < coef.degree; ++k) {
        grid_barrier(gbar, (++passed) * gridDim.x, err, &s_ticket);
        const float ab = coef.ab[k], cc = coef.cc[k];
        const bool have_prev = k > 1;                        // z_0 = 0
        for (;;) {
            int rr = 0;
            if (lane == 0) rr = atomicAdd(&s_ticket, 1);
            rr = __shfl_sync(0xffffffffu, rr, 0);
            const int row = r_lo + rr;
            if (row >= r_hi) break;
            const int rb0 = brow[row], rb1 = brow[row + 1];
            u64 acc[3][NP];
#pragma unroll
            for (int c = 0; c < 3; ++c)
#pragma unroll
                for (int t = 0; t < NP; ++t) acc[c][t] = 0ull;
            for (int p = rb0 + g; p < rb1; p += NG) {
                uint4 a0, a1, a2;
                if (p < s_hi) {
                    const uint4* rp = srec + 3 * (p - rec_lo);
                    a0 = rp[0]; a1 = rp[1]; a2 = rp[2];
                } else {
                    const uint4* rp = rec + (int64_t)3 * p;
                    a0 = ldg_na_u4(rp); a1 = ldg_na_u4(rp + 1); a2 = ldg_na_u4(rp + 2);
                }
                const float* xr = X + (int64_t)(int)a2.y * (3 * C);
                u64 x[3][NP];
#pragma unroll
                for (int d = 0; d < 3; ++d) ld_row2_coh<LPR, CPT>(xr + d * C, l, x[d]);
                const float kv[9] = {__uint_as_float(a0.x), __uint_as_float(a0.y), __uint_as_float(a0.z),
                                     __uint_as_float(a0.w), __uint_as_float(a1.x), __uint_as_float(a1.y),
                                     __uint_as_float(a1.z), __uint_as_float(a1.w), __uint_as_float(a2.x)};
#pragma unroll
                for (int c = 0; c < 3; ++c)
#pragma unroll
                    for (int d = 0; d < 3; ++d)
#pragma unroll
                        for (int t = 0; t < NP; ++t) ffma2(acc[c][t], kv[3 * c + d], x[d][t]);
            }
#pragma unroll
            for (int off = LPR; off < 32; off <<= 1)
#pragma unroll
                for (int c = 0; c < 3; ++c)
#pragma unroll
                    for (int t = 0; t < NP; ++t) acc[c][t] = fadd2(acc[c][t], __shfl_xor_sync(0xffffffffu, acc[c][t], off));
            if (g < 3) {
                const int64_t o = ((int64_t)3 * row + g) * C;
                float a[3][CPT];
#pragma unroll
                for (int c = 0; c < 3; ++c)
#pragma unroll
                    for (int t = 0; t < NP; ++t) unpack2(acc[c][t], a[c][2 * t], a[c][2 * t + 1]);
                const float d0 = __ldg(invD + 9 * (int64_t)row + 3 * g), d1 = __ldg(invD + 9 * (int64_t)row + 3 * g + 1),
                            d2 = __ldg(invD + 9 * (int64_t)row + 3 * g + 2);
                float r0v[CPT], r1v[CPT], r2v[CPT], z[CPT], zp[CPT], v[CPT];
                const int64_t ob = (int64_t)3 * row * C;
                ld_row<LPR, CPT>(R + ob, l, r0v);
                ld_row<LPR, CPT>(R + ob + C, l, r1v);
                ld_row<LPR, CPT>(R + ob + 2 * C, l, r2v);
                ld_row_plain<LPR, CPT>(X + o, l, z);
                if (have_prev) ld_row_plain<LPR, CPT>(Zp + o, l, zp);
#pragma unroll
                for (int t = 0; t < CPT; ++t) {
                    const float dr = d0 * (r0v[t] - a[0][t]) + d1 * (r1v[t] - a[1][t]) + d2 * (r2v[t] - a[2][t]);
                    v[t] = z[t] + ab * (z[t] - (have_prev ? zp[t] : 0.f)) + cc * dr;
                }
                st_row<LPR, CPT>(Zp + o, l, v);
            }
        }
        float* tsw = X; X = Zp; Zp = tsw;
    }
}

// chunk_row[c] = first row of chunk c: chunks of equal weight w(r) = brow[r] + 15 r (blocks + per-row overhead)
__global__ void k_chunk_rows(const int32_t* __restrict__ brow, int n_nodes, int nchunks, int32_t* __restrict__ chunk_row) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c > nchunks) return;
    if (c == nchunks) { chunk_row[c] = n_nodes; return; }
    const int64_t total = (int64_t)(brow[n_nodes] - brow[0]) + 15 * (int64_t)n_nodes;
    const int64_t target = total * c / nchunks;
    int lo = 0, hi = n_nodes;                    // first r with w(r) >= target
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if ((int64_t)(brow[mid] - brow[0]) + 15 * (int64_t)mid < target) lo = mid + 1; else hi = mid;
    }
    chunk_row[c] = lo;
}

// records + block-Jacobi inverse from the FP64 matrix: one warp per node row of the OPERATOR's numbering.
// perm (optional): operator row r is matrix row perm[r] and column j becomes inv[j] (Morton renumbering inside
// the preconditioner; brow_out then holds the row pointers of the permuted rows).  colmap (optional, slabs):
// record column id = colmap[global column]; row_offset: global id of local row 0.
__global__ void __launch_bounds__(256)
k_pack_k32(const int32_t* __restrict__ brow, const int32_t* __restrict__ bcol, int64_t n_nodes,
           const double* __restrict__ Kval, const double* __restrict__ Mblk, double shift,
           uint32_t* __restrict__ rec, float* __restrict__ invD, const uint32_t* __restrict__ colmap,
           int64_t row_offset, const int32_t* __restrict__ perm, const int32_t* __restrict__ inv,
           const int32_t* __restrict__ brow_out) {
    const int lane = threadIdx.x & 31;
    const int64_t row = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    if (row >= n_nodes) return;
    const int64_t src = perm ? (int64_t)perm[row] : row;
    const int64_t b0 = brow[src] - brow[0];      // a slab passes a window of the global brow
    const int deg = (int)(brow[src + 1] - brow[src]);
    const int64_t o0 = perm ? (int64_t)brow_out[row] : b0;
    const double* kb = Kval + 9 * b0;
    const int64_t rs = 3 * (int64_t)deg;
    for (int p = lane; p < deg; p += 32) {
        const int32_t j = bcol[b0 + p];
        double k[9];
#pragma unroll
        for (int c = 0; c < 3; ++c)
#pragma unroll
            for (int d = 0; d < 3; ++d) k[3 * c + d] = kb[c * rs + 3 * p + d];
        if (Mblk != nullptr && shift != 0.0) {
            const double m = shift * Mblk[b0 + p];
            k[0] += m; k[4] += m; k[8] += m;
        }
        uint4* o = reinterpret_cast<uint4*>(rec + (o0 + p) * S32_REC_WORDS);
        o[0] = make_uint4(__float_as_uint((float)k[0]), __float_as_uint((float)k[1]), __float_as_uint((float)k[2]),
                          __float_as_uint((float)k[3]));
        o[1] = make_uint4(__float_as_uint((float)k[4]), __float_as_uint((float)k[5]), __float_as_uint((float)k[6]),
                          __float_as_uint((float)k[7]));
        o[2] = make_uint4(__float_as_uint((float)k[8]), colmap ? colmap[j] : (inv ? (uint32_t)inv[j] : (uint32_t)j), 0u, 0u);
        if (j == src + row_offset) {
            const double c00 = k[4] * k[8] - k[5] * k[7];
            const double c01 = k[5] * k[6] - k[3] * k[8];
            const double c02 = k[3] * k[7] - k[4] * k[6];
            const double id = 1.0 / (k[0] * c00 + k[1] * c01 + k[2] * c02);
            float* iv = invD + 9 * row;
            iv[0] = (float)(c00 * id);
            iv[1] = (float)((k[2] * k[7] - k[1] * k[8]) * id);
            iv[2] = (float)((k[1] * k[5] - k[2] * k[4]) * id);
            iv[3] = (float)(c01 * id);
            iv[4] = (float)((k[0] * k[8] - k[2] * k[6]) * id);
            iv[5] = (float)((k[2] * k[3] - k[0] * k[5]) * id);
            iv[6] = (float)(c02 * id);
            iv[7] = (float)((k[1] * k[6] - k[0] * k[7]) * id);
            iv[8] = (float)((k[0] * k[4] - k[1] * k[3]) * id);
        }
    }
}

// ---- Morton renumbering of the operator's rows (locality of the gathered X rows) ------------------
// mm[0..2] = min key per axis, mm[3..5] = max key per axis (initialised to 0xffffffff / 0 by the caller)
__global__ void k_bbox(const float* __restrict__ coords, int64_t n, uint32_t* __restrict__ mm) {
    uint32_t lo[3] = {0xffffffffu, 0xffffffffu, 0xffffffffu}, hi[3] = {0u, 0u, 0u};
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
#pragma unroll
        for (int d = 0; d < 3; ++d) {
            const uint32_t k = ordered_key(coords[3 * i + d]);
            lo[d] = min(lo[d], k);
            hi[d] = max(hi[d], k);
        }
#pragma unroll
    for (int d = 0; d < 3; ++d) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            lo[d] = min(lo[d], __shfl_xor_sync(0xffffffffu, lo[d], o));
            hi[d] = max(hi[d], __shfl_xor_sync(0xffffffffu, hi[d], o));
        }
        if ((threadIdx.x & 31) == 0) {
            atomicMin(&mm[d], lo[d]);
            atomicMax(&mm[3 + d], hi[d]);
        }
    }
}
__device__ __forceinline__ uint32_t spread3(uint32_t v) {     // 10 bits -> every third bit
    v = (v | (v << 16)) & 0x030000ffu;
    v = (v | (v << 8)) & 0x0300f00fu;
    v = (v | (v << 4)) & 0x030c30c3u;
    v = (v | (v << 2)) & 0x09249249u;
    return v;
}
__global__ void k_morton_codes(const float* __restrict__ coords, int64_t n, const uint32_t* __restrict__ mm,
                               uint32_t* __restrict__ codes, uint32_t* __restrict__ iota) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t code = 0;
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        const float lo = key_to_float(mm[d]), hi = key_to_float(mm[3 + d]);
        const float ext = hi - lo;
        float t = ext > 0.f ? (coords[3 * i + d] - lo) / ext : 0.f;
        t = fminf(fmaxf(t, 0.f), 1.f);
        code |= spread3((uint32_t)(t * 1023.f)) << (2 - d);
    }
    codes[i] = code;
    iota[i] = (uint32_t)i;
}
__global__ void k_invert_perm(const int32_t* __restrict__ perm, int64_t n, int32_t* __restrict__ inv) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) inv[perm[i]] = (int32_t)i;
}
// out[r] = deg(perm[r]), out[n] = 0: the input of the exclusive scan that gives the row pointers of the renumbered level
// (a device-wide CUB scan; the single-CTA scan it replaces took 0.37 ms on the 274 625 rows of the bench mesh)
__global__ void __launch_bounds__(256) k_perm_deg(const int32_t* __restrict__ brow, const int32_t* __restrict__ perm,
                                                  int n, int32_t* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i > n) return;
    int v = 0;
    if (i < n) { const int s = perm[i]; v = brow[s + 1] - brow[s]; }
    out[i] = v;
}

// Out = cc * invD R   (first Chebyshev step from a zero initial guess); one thread per (node, 4 columns)
__global__ void k_jacobi32(const float* __restrict__ invD, const float* __restrict__ R, int64_t n_nodes, int c4,
                           float cc, float* __restrict__ Out) {
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= n_nodes * c4) return;
    const int64_t row = t / c4;
    const int q = (int)(t - row * c4);
    const int C = 4 * c4;
    const float4 r0 = __ldg(reinterpret_cast<const float4*>(R + 3 * row * C) + q);
    const float4 r1 = __ldg(reinterpret_cast<const float4*>(R + (3 * row + 1) * C) + q);
    const float4 r2 = __ldg(reinterpret_cast<const float4*>(R + (3 * row + 2) * C) + q);
    const float* d = invD + 9 * row;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const float d0 = cc * d[3 * c], d1 = cc * d[3 * c + 1], d2 = cc * d[3 * c + 2];
        float4 v;
        v.x = d0 * r0.x + d1 * r1.x + d2 * r2.x;
        v.y = d0 * r0.y + d1 * r1.y + d2 * r2.y;
        v.z = d0 * r0.z + d1 * r1.z + d2 * r2.z;
        v.w = d0 * r0.w + d1 * r1.w + d2 * r2.w;
        reinterpret_cast<float4*>(Out + (3 * row + c) * C)[q] = v;
    }
}

// dst32[:, s] = (float) src64[:, idx[s]] for s < count, 0 for count <= s < width; with perm, dof row 3 r + c of
// dst is dof row 3 perm[r] + c of src (the preconditioner's own node numbering).  One thread per (row, 4 columns).
__global__ void k_gather_cols_f32(const double* __restrict__ src, int64_t lds, const __grid_constant__ ColIdx idx,
                                  int count, int width, int64_t n, float* __restrict__ dst,
                                  const int32_t* __restrict__ perm) {
    const int w4 = width >> 2;
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= n * w4) return;
    const int64_t row = t / w4;
    const int s = (int)(t - row * w4) * 4;
    int64_t srow = row;
    if (perm) { const int64_t node = row / 3; srow = 3 * (int64_t)perm[node] + (row - 3 * node); }
    const double* sp = src + srow * lds;
    float4 v;
    v.x = s + 0 < count ? (float)__ldg(sp + idx.v[s + 0]) : 0.f;
    v.y = s + 1 < count ? (float)__ldg(sp + idx.v[s + 1]) : 0.f;
    v.z = s + 2 < count ? (float)__ldg(sp + idx.v[s + 2]) : 0.f;
    v.w = s + 3 < count ? (float)__ldg(sp + idx.v[s + 3]) : 0.f;
    reinterpret_cast<float4*>(dst + row * width)[s >> 2] = v;
}

// dst64[:, :width] (ld) = (double) src32 (n x width); with perm, dof row 3 perm[r] + c of dst from row 3 r + c of src.
// One thread per (row, 4 columns); dst rows must be 16-byte aligned (even ld, aligned base).
__global__ void k_widen_f32(const float* __restrict__ src, int width, int64_t n, double* __restrict__ dst, int64_t ldd,
                            const int32_t* __restrict__ perm) {
    const int w4 = width >> 2;
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= n * w4) return;
    const int64_t row = t / w4;
    const int q = (int)(t - row * w4);
    int64_t drow = row;
    if (perm) { const int64_t node = row / 3; drow = 3 * (int64_t)perm[node] + (row - 3 * node); }
    const float4 v = __ldg(reinterpret_cast<const float4*>(src + row * width) + q);
    double2* dp = reinterpret_cast<double2*>(dst + drow * ldd + 4 * q);
    dp[0] = make_double2((double)v.x, (double)v.y);
    dp[1] = make_double2((double)v.z, (double)v.w);
}

// per-column sum of squares of an fp32 block (n x w), fp64 accumulation; partial[cta][w]
__global__ void k_colnorm2_f32(const float* __restrict__ V, int w, int64_t n, double* __restrict__ partial) {
    extern __shared__ double sh[];
    const int rpp = blockDim.x / w;
    const int c = threadIdx.x % w, rr = threadIdx.x / w;
    double s = 0.0;
    if (rr < rpp) {
        for (int64_t row = (int64_t)blockIdx.x * rpp + rr; row < n; row += (int64_t)gridDim.x * rpp) {
            const double v = (double)V[row * w + c];
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

// ---- two-level transfer operators (nodes; 3 components x c columns per node) -------------------
// rc[I] = 0.5 * sum_{t in rptr[I]..rptr[I+1]} res[rlist[t]]      (P^T, gather form, fixed order)
// perm_c / inv_f (optional): coarse row I of rc is coarse node perm_c[I]; fine node f lives at row inv_f[f] of res
__global__ void k_restrict32(const int32_t* __restrict__ rptr, const int32_t* __restrict__ rlist, int64_t n_coarse,
                             const float* __restrict__ res, int c4x3, float* __restrict__ rc,
                             const int32_t* __restrict__ perm_c, const int32_t* __restrict__ inv_f) {
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= n_coarse * c4x3) return;
    const int64_t I = t / c4x3;
    const int q = (int)(t - I * c4x3);
    const int64_t Is = perm_c ? (int64_t)perm_c[I] : I;
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    const int e = rptr[Is + 1];
    for (int u = rptr[Is]; u < e; ++u) {
        const int f = inv_f ? inv_f[rlist[u]] : rlist[u];
        const float4 v = __ldg(reinterpret_cast<const float4*>(res) + (int64_t)f * c4x3 + q);
        s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
    }
    s.x *= 0.5f; s.y *= 0.5f; s.z *= 0.5f; s.w *= 0.5f;
    reinterpret_cast<float4*>(rc)[t] = s;
}

// z[i] += 0.5 * (zc[par[2i]] + zc[par[2i+1]])                  (P)
// perm_f / inv_c (optional): row i of z is fine node perm_f[i]; coarse node c lives at row inv_c[c] of zc
__global__ void k_prolong_add32(const int32_t* __restrict__ par, int64_t n_fine, const float* __restrict__ zc, int c4x3,
                                float* __restrict__ z, const int32_t* __restrict__ perm_f,
                                const int32_t* __restrict__ inv_c) {
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= n_fine * c4x3) return;
    const int64_t i = t / c4x3;
    const int q = (int)(t - i * c4x3);
    int2 pp = __ldg(reinterpret_cast<const int2*>(par) + (perm_f ? (int64_t)perm_f[i] : i));
    if (inv_c) { pp.x = inv_c[pp.x]; pp.y = inv_c[pp.y]; }
    const float4 a = __ldg(reinterpret_cast<const float4*>(zc) + (int64_t)pp.x * c4x3 + q);
    const float4 b = __ldg(reinterpret_cast<const float4*>(zc) + (int64_t)pp.y * c4x3 + q);
    float4 v = reinterpret_cast<float4*>(z)[t];
    v.x += 0.5f * (a.x + b.x); v.y += 0.5f * (a.y + b.y); v.z += 0.5f * (a.z + b.z); v.w += 0.5f * (a.w + b.w);
    reinterpret_cast<float4*>(z)[t] = v;
}

// fp64 variant used to prolong a coarse eigenvector block into the fine start block
__global__ void k_prolong64(const int32_t* __restrict__ par, int64_t n_fine, const double* __restrict__ xc, int64_t ldc,
                            int w, double* __restrict__ x, int64_t ldx) {
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= n_fine * 3 * w) return;
    const int64_t i = t / (3 * w);
    const int r = (int)(t - i * 3 * w);
    const int c = r / w, s = r - c * w;
    const int2 pp = __ldg(reinterpret_cast<const int2*>(par) + i);
    x[(3 * i + c) * ldx + s] = 0.5 * (xc[(3 * (int64_t)pp.x + c) * ldc + s] + xc[(3 * (int64_t)pp.y + c) * ldc + s]);
}

// xc[3I + c][:] = x[3 f(I) + c][:], f(I) = the fine (corner) node of coarse node I: the one entry that
// appears twice in I's gather list (a corner is its own parent twice)
__global__ void k_inject64(const int32_t* __restrict__ rptr, const int32_t* __restrict__ rlist, int64_t n_coarse,
                           const double* __restrict__ x, int64_t ldx, int w, double* __restrict__ xc, int64_t ldc) {
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= n_coarse * 3 * w) return;
    const int64_t I = t / (3 * w);
    const int r = (int)(t - I * 3 * w);
    const int c = r / w, s = r - c * w;
    int64_t f = -1;
    for (int u = rptr[I]; u + 1 < rptr[I + 1]; ++u)
        if (rlist[u] == rlist[u + 1]) { f = rlist[u]; break; }
    xc[(3 * I + c) * ldc + s] = f >= 0 ? x[(3 * f + c) * ldx + s] : 0.0;
}

int inject64(const int32_t* rptr, const int32_t* rlist, int64_t n_coarse, const double* x, int64_t ldx, int w,
             double* xc, int64_t ldc, cudaStream_t st) {
    ProfScope prof(PROF_TRANSFER, st);
    k_inject64<<<(unsigned)ceil_div(n_coarse * 3 * w, 256), 256, 0, st>>>(rptr, rlist, n_coarse, x, ldx, w, xc, ldc);
    DS_LAUNCH_CHECK();
    return DS_OK;
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
static int s32v_grid(int64_t n_nodes) {
    static int sms = 0;
    if (!sms) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    }
    const int64_t want = ceil_div(n_nodes, 32);
    return (int)(want < sms ? want : sms);
}

int spmm32_chunk_count(int64_t n_nodes) { return s32v_grid(n_nodes); }

int spmm32_chunks(const int32_t* brow, int64_t n_nodes, int32_t* chunk_row, cudaStream_t st) {
    const int nchunks = s32v_grid(n_nodes);
    k_chunk_rows<<<ceil_div(nchunks + 1, 128), 128, 0, st>>>(brow, (int)n_nodes, nchunks, chunk_row);
    DS_LAUNCH_CHECK();
    return DS_OK;
}

template <int LPR, int CPT, bool PEER>
static int launch_spmm32(int mode, const int32_t* brow, const void* rec, int64_t n_nodes, const int32_t* chunk_row,
                         const float* X, const float* R, const float* invD, const float* Zprev, float* Out, float ab,
                         float cc, const PeerTable& tab, cudaStream_t st) {
    DS_REQUIRE(chunk_row != nullptr, "spmm32: missing row chunks");
    const int grid = s32v_grid(n_nodes);
    auto go = [&](auto kern) -> int {
        static bool carved = false;          // per instantiation: all of the SM's 256 KB as L1
        if (!carved) {
            DS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxL1));
            carved = true;
        }
        // a level whose records and four dense blocks fit in half of the 126 MB L2 stays resident between the
        // launches of a Chebyshev sequence: the look-ahead prefetch would only add latency to every row
        const int prefetch = (n_nodes * (int64_t)(30 * S32_REC_BYTES + 48 * LPR * CPT)) > ((int64_t)60 << 20);
        kern<<<grid, S32V_THREADS, 0, st>>>(brow, reinterpret_cast<const uint4*>(rec), chunk_row, X, R, invD, Zprev, Out,
                                            ab, cc, prefetch, tab);
        DS_LAUNCH_CHECK();
        return DS_OK;
    };
    switch (mode) {
        case S32_PLAIN: return go(k_spmm32v<LPR, CPT, S32_PLAIN, PEER>);
        case S32_RESID: return go(k_spmm32v<LPR, CPT, S32_RESID, PEER>);
        default: return go(k_spmm32v<LPR, CPT, S32_CHEB, PEER>);
    }
}

template <bool PEER>
static int dispatch_spmm32(int mode, const int32_t* brow, const void* rec, int64_t n_nodes, const int32_t* chunk_row,
                           int ncols, const float* X, const float* R, const float* invD, const float* Zprev, float* Out,
                           float ab, float cc, const PeerTable& tab, cudaStream_t st) {
    switch (ncols) {
        case 16: return launch_spmm32<4, 4, PEER>(mode, brow, rec, n_nodes, chunk_row, X, R, invD, Zprev, Out, ab, cc, tab, st);
        case 32: return launch_spmm32<8, 4, PEER>(mode, brow, rec, n_nodes, chunk_row, X, R, invD, Zprev, Out, ab, cc, tab, st);
        case 48: return launch_spmm32<8, 6, PEER>(mode, brow, rec, n_nodes, chunk_row, X, R, invD, Zprev, Out, ab, cc, tab, st);
        case 64: return launch_spmm32<8, 8, PEER>(mode, brow, rec, n_nodes, chunk_row, X, R, invD, Zprev, Out, ab, cc, tab, st);
        default: set_error("spmm32: ncols=%d must be 16, 32, 48 or 64", ncols); return DS_ERR_ARG;
    }
}

// chunk_row: s32v_grid(n_nodes) + 1 row offsets from spmm32_chunks (NULL: built into a stream-ordered temporary)
// Stream-ordered temporaries come from the device's default memory pool; its release threshold is 0 by default, so every
// synchronisation hands the pool back to the driver and the next cudaMallocAsync pays a full allocation.  Keep the pool.
static void keep_async_pool() {
    static thread_local int done_for = -1;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev == done_for) return;
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
        uint64_t keep = UINT64_MAX;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
    done_for = dev;
}

struct ChunkTmp {
    int32_t* p = nullptr;
    cudaStream_t st;
    int get(const int32_t* brow, int64_t n_nodes, const int32_t* given, cudaStream_t s, const int32_t** out) {
        st = s;
        if (given) { *out = given; return DS_OK; }
        keep_async_pool();
        DS_CUDA(cudaMallocAsync(&p, sizeof(int32_t) * (s32v_grid(n_nodes) + 1), s));
        DS_TRY(spmm32_chunks(brow, n_nodes, p, s));
        *out = p;
        return DS_OK;
    }
    ~ChunkTmp() { if (p) cudaFreeAsync(p, st); }
};

int spmm32(int mode, const int32_t* brow, const void* rec, int64_t n_nodes, int ncols, const float* X, const float* R,
           const float* invD, const float* Zprev, float* Out, float ab, float cc, int prof_cls, cudaStream_t st,
           const int32_t* chunk_row) {
    DS_REQUIRE(brow && rec && X && Out, "spmm32: null argument");
    DS_REQUIRE(X != Out, "spmm32: the gathered block must not alias the output");
    DS_REQUIRE(mode == S32_PLAIN || R, "spmm32: this mode needs R");
    DS_REQUIRE(mode != S32_CHEB || (invD && Zprev), "spmm32: Chebyshev mode needs invD and Zprev");
    ChunkTmp tmp;
    const int32_t* chunks = nullptr;
    DS_TRY(tmp.get(brow, n_nodes, chunk_row, st, &chunks));
    ProfScope prof(prof_cls, st);
    PeerTable none = {};
    return dispatch_spmm32<false>(mode, brow, rec, n_nodes, chunks, ncols, X, R, invD, Zprev, Out, ab, cc, none, st);
}

// row-partitioned: Xparts[r] = base of rank r's slab of the gathered block (device pointers valid in this
// process); X_own = this rank's slab (Xparts[rank]); all other arrays are local slabs
int spmm32_rowpart(int mode, const int32_t* brow, const void* rec, int64_t n_local, int ncols, const float* const* Xparts,
                   int world, int rank, const float* R, const float* invD, const float* Zprev, float* Out, float ab,
                   float cc, cudaStream_t st) {
    DS_REQUIRE(brow && rec && Xparts && Out, "spmm32_rowpart: null argument");
    DS_REQUIRE(world >= 1 && world <= 8 && rank >= 0 && rank < world, "spmm32_rowpart: world=%d rank=%d (max 8 ranks)", world, rank);
    DS_REQUIRE(mode == S32_PLAIN || R, "spmm32_rowpart: this mode needs R");
    DS_REQUIRE(mode != S32_CHEB || (invD && Zprev), "spmm32_rowpart: Chebyshev mode needs invD and Zprev");
    PeerTable tab = {};
    for (int r = 0; r < world; ++r) {
        DS_REQUIRE(Xparts[r] != nullptr, "spmm32_rowpart: missing slab pointer of rank %d", r);
        tab.p[r] = Xparts[r];
    }
    DS_REQUIRE(tab.p[rank] != Out, "spmm32_rowpart: the gathered block must not alias the output");
    ChunkTmp tmp;
    const int32_t* chunks = nullptr;
    DS_TRY(tmp.get(brow, n_local, nullptr, st, &chunks));
    ProfScope prof(PROF_CHEB, st);
    return dispatch_spmm32<true>(mode, brow, rec, n_local, chunks, ncols, tab.p[rank], R, invD, Zprev, Out, ab, cc, tab, st);
}

int pack_k32(const int32_t* brow, const int32_t* bcol, int64_t n_nodes, const double* Kval, const double* Mblk,
             double shift, void* rec, float* invD, cudaStream_t st, const uint32_t* colmap, int64_t row_offset,
             const int32_t* perm, const int32_t* inv, const int32_t* brow_out) {
    DS_REQUIRE(brow && bcol && Kval && rec && invD, "pack_k32: null argument");
    DS_REQUIRE(((uintptr_t)rec & 15) == 0, "pack_k32: records must be 16-byte aligned");
    DS_REQUIRE(!perm || (inv && brow_out && !colmap), "pack_k32: a row permutation needs inv and brow_out (and no colmap)");
    ProfScope prof(PROF_COPY, st);
    k_pack_k32<<<(unsigned)ceil_div(n_nodes * 32, 256), 256, 0, st>>>(brow, bcol, n_nodes, Kval, Mblk, shift,
                                                                      reinterpret_cast<uint32_t*>(rec), invD, colmap,
                                                                      row_offset, perm, inv, brow_out);
    DS_LAUNCH_CHECK();
    return DS_OK;
}

int jacobi32(const float* invD, const float* R, int64_t n_nodes, int ncols, float cc, float* Out, cudaStream_t st) {
    ProfScope prof(PROF_JACOBI, st);      // not an SpMM launch: kept out of the classes the roofline is computed from
    const int c4 = ncols / 4;
    k_jacobi32<<<(unsigned)ceil_div(n_nodes * c4, 256), 256, 0, st>>>(invD, R, n_nodes, c4, cc, Out);
    DS_LAUNCH_CHECK();
    return DS_OK;
}

int restrict32(const int32_t* rptr, const int32_t* rlist, int64_t n_coarse, const float* res, int ncols, float* rc,
               cudaStream_t st, const int32_t* perm_c, const int32_t* inv_f) {
    ProfScope prof(PROF_TRANSFER, st);
    const int q = 3 * ncols / 4;
    k_restrict32<<<(unsigned)ceil_div(n_coarse * q, 256), 256, 0, st>>>(rptr, rlist, n_coarse, res, q, rc, perm_c, inv_f);
    DS_LAUNCH_CHECK();
    return DS_OK;
}

int prolong_add32(const int32_t* par, int64_t n_fine, const float* zc, int ncols, float* z, cudaStream_t st,
                  const int32_t* perm_f, const int32_t* inv_c) {
    ProfScope prof(PROF_TRANSFER, st);
    const int q = 3 * ncols / 4;
    k_prolong_add32<<<(unsigned)ceil_div(n_fine * q, 256), 256, 0, st>>>(par, n_fine, zc, q, z, perm_f, inv_c);
    DS_LAUNCH_CHECK();
    return DS_OK;
}

int prolong64(const int32_t* par, int64_t n_fine, const double* xc, int64_t ldc, int w, double* x, int64_t ldx,
              cudaStream_t st) {
    ProfScope prof(PROF_TRANSFER, st);
    k_prolong64<<<(unsigned)ceil_div(n_fine * 3 * w, 256), 256, 0, st>>>(par, n_fine, xc, ldc, w, x, ldx);
    DS_LAUNCH_CHECK();
    return DS_OK;
}

int gather_cols_f32(const double* src, int64_t lds, const ColIdx& idx, int count, int width, int64_t n, float* dst,
                    cudaStream_t st, const int32_t* perm) {
    ProfScope prof(PROF_COPY, st);
    DS_REQUIRE(width % 4 == 0, "gather_cols_f32: width must be a multiple of 4");
    k_gather_cols_f32<<<(unsigned)ceil_div(n * (width / 4), 256), 256, 0, st>>>(src, lds, idx, count, width, n, dst, perm);
    DS_LAUNCH_CHECK();
    return DS_OK;
}

int widen_f32(const float* src, int width, int64_t n, double* dst, int64_t ldd, cudaStream_t st, const int32_t* perm) {
    ProfScope prof(PROF_COPY, st);
    DS_REQUIRE(width % 4 == 0 && ldd % 2 == 0 && ((uintptr_t)dst & 15) == 0, "widen_f32: width % 4, even ld and 16-byte aligned dst");
    k_widen_f32<<<(unsigned)ceil_div(n * (width / 4), 256), 256, 0, st>>>(src, width, n, dst, ldd, perm);
    DS_LAUNCH_CHECK();
    return DS_OK;
}

__global__ void k_fill_random_f32(float* __restrict__ V, int64_t count, uint64_t seed) {
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= count) return;
    uint64_t z = seed + 0x9E3779B97F4A7C15ull * (uint64_t)(t + 1);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    z ^= z >> 31;
    V[t] = (float)((double)(z >> 11) * (2.0 / 9007199254740992.0) - 1.0);
}

int fill_random_f32(float* V, int64_t count, uint64_t seed, cudaStream_t st) {
    k_fill_random_f32<<<(unsigned)ceil_div(count, 256), 256, 0, st>>>(V, count, seed);
    DS_LAUNCH_CHECK();
    return DS_OK;
}

int colnorm2_f32(const float* V, int w, int64_t n, double* partial, int ctas, cudaStream_t st) {
    const int threads = (1024 / w) * w;
    const size_t sm = (size_t)(threads / w) * w * sizeof(double);
    k_colnorm2_f32<<<ctas, threads, sm, st>>>(V, w, n, partial);
    DS_LAUNCH_CHECK();
    return DS_OK;
}

// ---- Level32 -----------------------------------------------------------------------------------
static size_t morton_sort_temp(int64_t n_nodes) {
    size_t t = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, t, (uint32_t*)nullptr, (uint32_t*)nullptr, (uint32_t*)nullptr,
                                    (uint32_t*)nullptr, (int)n_nodes, 0, 30);
    size_t u = 0;           // the scan of the permuted row lengths reuses the same scratch
    cub::DeviceScan::ExclusiveSum(nullptr, u, (int32_t*)nullptr, (int32_t*)nullptr, (int)n_nodes + 1);
    return std::max(t, u);
}

// bcolP[browP[r] + p] = inv[bcol[brow[perm[r]] + p]]: the level's column ids as a plain int32 array (the FP64 SpMM on
// fp32 iterates reads 4 bytes per block instead of fishing them out of the 48-byte records)
__global__ void __launch_bounds__(256)
k_perm_bcol(const int32_t* __restrict__ brow, const int32_t* __restrict__ bcol, const int32_t* __restrict__ browP,
            const int32_t* __restrict__ perm, const int32_t* __restrict__ inv, int64_t n_nodes, int32_t* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t r = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    if (r >= n_nodes) return;
    const int64_t src = perm ? (int64_t)perm[r] : r;
    const int64_t b0 = brow[src], o0 = browP[r];
    const int deg = (int)(brow[src + 1] - b0);
    for (int p = lane; p < deg; p += 32) {
        const int32_t j = bcol[b0 + p];
        out[o0 + p] = inv ? inv[j] : j;
    }
}

size_t Level32::bytes(int64_t n_nodes, int64_t nnzb) {
    auto al = [](size_t b) { return ((b + 255) & ~size_t(255)) + 256; };
    return al((size_t)nnzb * sizeof(int32_t)) + al((size_t)nnzb * S32_REC_BYTES + 64) + al((size_t)n_nodes * 9 * sizeof(float)) + al(1024 * sizeof(int32_t)) +
           6 * al((size_t)(n_nodes + 1) * sizeof(int32_t)) + al(morton_sort_temp(n_nodes)) + 2 * al(64);
}

// coords (optional, fp32 [n_nodes x 3]): the operator is stored with its rows and columns renumbered along a
// Morton curve through the node coordinates, so that consecutive rows gather overlapping sets of X rows (served by
// the SM's L1 in k_spmm32v).  The numbering is private to the level: perm / inv translate at its boundary
// (gather_cols_f32, widen_f32, restrict32, prolong_add32).
int Level32::setup(Arena& a, const int32_t* brow_, const int32_t* bcol, int64_t n_nodes_, int64_t nnzb_,
                   const double* Kval, const double* Mblk, double shift, const float* coords, cudaStream_t st) {
    n_nodes = n_nodes_;
    nnzb = nnzb_;
    rec = a.take<unsigned char>((size_t)nnzb * S32_REC_BYTES + 64);
    invD = a.take<float>((size_t)n_nodes * 9);
    chunk_row = a.take<int32_t>(1024);
    gbar = a.take<unsigned>(16);
    DS_REQUIRE(rec && invD && chunk_row && gbar, "Level32: workspace arena exhausted");
    DS_CUDA(cudaMemsetAsync(gbar, 0, 16 * sizeof(unsigned), st));
    {
        int dev = 0, coop = 0;
        DS_CUDA(cudaGetDevice(&dev));
        DS_CUDA(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev));
        persistent = coop != 0;
    }
    DS_REQUIRE(s32v_grid(n_nodes) < 1024, "Level32: more than 1023 SMs");
    DS_CUDA(cudaMemsetAsync(rec + (size_t)nnzb * S32_REC_BYTES, 0, 64, st));    // bulk prefetches read up to 8 bytes past the end
    perm = inv = nullptr;
    brow = brow_;
    if (coords) {
        ProfScope prof(PROF_COPY, st);
        int32_t* perm_w = a.take<int32_t>(n_nodes + 1);
        int32_t* inv_w = a.take<int32_t>(n_nodes + 1);
        int32_t* brow_w = a.take<int32_t>(n_nodes + 1);
        uint32_t* codes = a.take<uint32_t>(n_nodes + 1);
        uint32_t* codes2 = a.take<uint32_t>(n_nodes + 1);
        uint32_t* iota = a.take<uint32_t>(n_nodes + 1);
        size_t tmp = morton_sort_temp(n_nodes);
        void* scratch = a.take<char>(tmp);
        uint32_t* mm = a.take<uint32_t>(8);
        DS_REQUIRE(scratch && mm, "Level32: workspace arena exhausted");
        DS_CUDA(cudaMemsetAsync(mm, 0xff, 3 * sizeof(uint32_t), st));
        DS_CUDA(cudaMemsetAsync(mm + 3, 0, 3 * sizeof(uint32_t), st));
        k_bbox<<<148, 256, 0, st>>>(coords, n_nodes, mm);
        DS_LAUNCH_CHECK();
        const unsigned blocks = (unsigned)ceil_div(n_nodes, 256);
        k_morton_codes<<<blocks, 256, 0, st>>>(coords, n_nodes, mm, codes, iota);
        DS_LAUNCH_CHECK();
        DS_CUDA(cub::DeviceRadixSort::SortPairs(scratch, tmp, codes, codes2, iota, reinterpret_cast<uint32_t*>(perm_w),
                                                (int)n_nodes, 0, 30, st));
        count_launch();
        k_invert_perm<<<blocks, 256, 0, st>>>(perm_w, n_nodes, inv_w);
        DS_LAUNCH_CHECK();
        k_perm_deg<<<(unsigned)ceil_div(n_nodes + 1, 256), 256, 0, st>>>(brow_, perm_w, (int)n_nodes, brow_w);
        DS_LAUNCH_CHECK();
        DS_CUDA(cub::DeviceScan::ExclusiveSum(scratch, tmp, brow_w, brow_w, (int)n_nodes + 1, st));
        count_launch();
        perm = perm_w;
        inv = inv_w;
        brow = brow_w;
    }
    DS_TRY(pack_k32(brow_, bcol, n_nodes, Kval, Mblk, shift, rec, invD, st, nullptr, 0, perm, inv, perm ? brow : nullptr));
    bcolP = nullptr;
    if (want_bcolP) {
        int32_t* bp = a.take<int32_t>((size_t)nnzb);
        DS_REQUIRE(bp, "Level32: workspace arena exhausted");
        ProfScope prof(PROF_COPY, st);
        k_perm_bcol<<<(unsigned)ceil_div(n_nodes * 32, 256), 256, 0, st>>>(brow_, bcol, brow, perm, inv, n_nodes, bp);
        DS_LAUNCH_CHECK();
        bcolP = bp;
    }
    return spmm32_chunks(brow, n_nodes, chunk_row, st);
}

// z = p(invD A) invD r by `degree` Chebyshev steps on [lmax/ratio, lmax].
//   from_zero: z0 = 0 (first step is a pure Jacobi scaling); else z0 = contents of *zc.
// zc / zp: ping-pong buffers; on return *zc holds the result.
template <int LPR, int CPT>
static int launch_cheb_persistent(const Level32& L, const float* r, const ChebCoef& coef, float* Za, float* Zb,
                                  int smem_records, size_t smem_bytes, cudaStream_t st) {
    auto kern = k_cheb32_persistent<LPR, CPT>;
    static bool attr = false;
    if (!attr) {
        DS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
        attr = true;
    }
    const int32_t* brow = L.brow;
    const uint4* rec = reinterpret_cast<const uint4*>(L.rec);
    const int32_t* chunk_row = L.chunk_row;
    const float* invD = L.invD;
    unsigned* gbar = L.gbar;
    int* err = reinterpret_cast<int*>(L.gbar + 1);
    void* args[] = {(void*)&brow, (void*)&rec, (void*)&chunk_row, (void*)&r, (void*)&invD, (void*)&Za, (void*)&Zb,
                    (void*)&coef, (void*)&smem_records, (void*)&gbar, (void*)&err};
    DS_CUDA(cudaMemsetAsync(L.gbar, 0, sizeof(unsigned), st));
    const cudaError_t e = cudaLaunchCooperativeKernel((const void*)kern, dim3(spmm32_chunk_count(L.n_nodes)),
                                                      dim3(S32V_THREADS), args, smem_bytes, st);
    if (e != cudaSuccess) {          // e.g. the device cannot co-schedule the grid right now: the caller steps instead
        cudaGetLastError();
        return 1;
    }
    count_launch();
    return DS_OK;
}

int Level32::cheb(const float* r, int ncols, int degree, double ratio, bool from_zero, float** zc, float** zp,
                  cudaStream_t st) {
    const double lmin = lmax / ratio;
    const double theta = 0.5 * (lmax + lmin), delta = 0.5 * (lmax - lmin), sig = theta / delta;
    double rho = 1.0 / sig;
    int k = 0;
    // a level whose records fit into the SMs' shared memory runs all its steps in one cooperative launch
    const int nchunks = spmm32_chunk_count(n_nodes);
    const size_t avg_rec_bytes = (size_t)nnzb * S32_REC_BYTES / (size_t)nchunks;
    if (from_zero && persistent && degree >= 3 && degree <= CHP_MAX_DEGREE && nchunks >= 8 && avg_rec_bytes <= 190 * 1024 &&
        (ncols == 16 || ncols == 32 || ncols == 48)) {
        ChebCoef coef;
        coef.cc0 = (float)(1.0 / theta);
        coef.degree = degree;
        for (k = 1; k < degree; ++k) {
            const double rho_new = 1.0 / (2.0 * sig - rho);
            coef.ab[k] = (float)(rho_new * rho);
            coef.cc[k] = (float)(2.0 * rho_new / delta);
            rho = rho_new;
        }
        // shared memory: the average chunk + 12 % (chunks are balanced by blocks + rows); a longer chunk reads its
        // tail from global memory
        size_t smem_bytes = std::min<size_t>(avg_rec_bytes + avg_rec_bytes / 8 + 4096, 216 * 1024);
        smem_bytes &= ~size_t(15);
        const int smem_records = (int)(smem_bytes / S32_REC_BYTES);
        int rc;
        {
            ProfScope prof(prof_cls, st);
            switch (ncols) {
                case 16: rc = launch_cheb_persistent<4, 4>(*this, r, coef, *zc, *zp, smem_records, smem_bytes, st); break;
                case 32: rc = launch_cheb_persistent<8, 4>(*this, r, coef, *zc, *zp, smem_records, smem_bytes, st); break;
                default: rc = launch_cheb_persistent<8, 6>(*this, r, coef, *zc, *zp, smem_records, smem_bytes, st); break;
            }
        }
        if (rc < 0) return rc;
        if (rc == DS_OK) {
            if ((degree - 1) & 1) std::swap(*zc, *zp);      // z_1 in zc; every further step swaps the roles
            launches += degree - 1;
            cols += (int64_t)(degree - 1) * ncols;
            return DS_OK;
        }
        persistent = false;          // cooperative launch refused: one launch per step from now on
        rho = 1.0 / sig;
    }
    if (from_zero) {
        DS_TRY(jacobi32(invD, r, n_nodes, ncols, (float)(1.0 / theta), *zc, st));
    } else {
        DS_TRY(spmm32(S32_CHEB, brow, rec, n_nodes, ncols, *zc, r, invD, *zc, *zp, 0.f, (float)(1.0 / theta), prof_cls,
                      st, chunk_row));
        std::swap(*zc, *zp);
        ++launches;
        cols += ncols;
    }
    for (k = 1; k < degree; ++k) {
        const double rho_new = 1.0 / (2.0 * sig - rho);
        const float ab = (float)(rho_new * rho);
        const float cc = (float)(2.0 * rho_new / delta);
        // z_{k+1} = z_k + ab (z_k - z_{k-1}) + cc invD (r - A z_k); for k == 1 from zero, z_0 = 0
        if (k == 1 && from_zero) DS_CUDA(cudaMemsetAsync(*zp, 0, sizeof(float) * 3 * (size_t)n_nodes * ncols, st));
        DS_TRY(spmm32(S32_CHEB, brow, rec, n_nodes, ncols, *zc, r, invD, *zp, *zp, ab, cc, prof_cls, st, chunk_row));
        std::swap(*zc, *zp);
        rho = rho_new;
        ++launches;
        cols += ncols;
    }
    return DS_OK;
}

}  // namespace ds

using namespace ds;

extern "C" int64_t ds_k32_record_bytes(int64_t nnzb) { return nnzb * S32_REC_BYTES + 64; }

extern "C" int ds_k32_pack(const int32_t* brow, const int32_t* bcol, int64_t n_nodes, int64_t nnzb, const double* Kval,
                           const double* Mblk, double shift, void* rec, float* invD, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    DS_REQUIRE(rec, "ds_k32_pack: null argument");
    DS_CUDA(cudaMemsetAsync(reinterpret_cast<unsigned char*>(rec) + nnzb * S32_REC_BYTES, 0, 64, st));
    return pack_k32(brow, bcol, n_nodes, Kval, Mblk, shift, rec, invD, st);
}

extern "C" int ds_spmm32(int mode, const int32_t* brow, const void* rec, int64_t n_nodes, int ncols, const float* X,
                         const float* R, const float* invD, const float* Zprev, float* Out, double ab, double cc,
                         const int32_t* chunk_row, void* stream) {
    DS_REQUIRE(mode >= 0 && mode <= 2, "ds_spmm32: mode must be 0 (A X), 1 (R - A X) or 2 (Chebyshev step)");
    return spmm32(mode, brow, rec, n_nodes, ncols, X, R, invD, Zprev, Out, (float)ab, (float)cc, PROF_CHEB,
                  (cudaStream_t)stream, chunk_row);
}

extern "C" int ds_spmm32_chunk_count(int64_t n_nodes) { return s32v_grid(n_nodes); }

/* z = p(invD A) invD R by `degree` Chebyshev steps on [lmax / ratio, lmax] from a zero initial guess (the coarse solve
 * and the one-level preconditioner of the eigensolver).  persistent != 0: all steps in one cooperative launch with the
 * records in shared memory (levels that fit); 0: one k_spmm32v launch per step.  Za, Zb: ping-pong buffers
 * [3*n_nodes x ncols]; *which_host = 0 / 1: the result is in Za / Zb. */
extern "C" int ds_cheb32_solve(const int32_t* brow, const void* rec, const float* invD, int64_t n_nodes, int64_t nnzb,
                               const float* R, int ncols, int degree, double lmax, double ratio, int persistent,
                               float* Za, float* Zb, int* which_host, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    DS_REQUIRE(brow && rec && invD && R && Za && Zb && which_host && degree >= 1 && lmax > 0 && ratio > 1,
               "ds_cheb32_solve: bad argument");
    Level32 L;
    L.brow = brow;
    L.n_nodes = n_nodes;
    L.nnzb = nnzb;
    L.rec = const_cast<unsigned char*>(reinterpret_cast<const unsigned char*>(rec));
    L.invD = const_cast<float*>(invD);
    L.lmax = lmax;
    int32_t* tmp = nullptr;
    keep_async_pool();
    DS_CUDA(cudaMallocAsync(&tmp, sizeof(int32_t) * (1024 + 16), st));
    L.chunk_row = tmp;
    L.gbar = reinterpret_cast<unsigned*>(tmp + 1024);
    DS_CUDA(cudaMemsetAsync(L.gbar, 0, 16 * sizeof(unsigned), st));
    L.persistent = persistent != 0;
    int rc = spmm32_chunks(brow, n_nodes, L.chunk_row, st);
    float *zc = Za, *zp = Zb;
    if (rc == DS_OK) rc = L.cheb(R, ncols, degree, ratio, true, &zc, &zp, st);
    unsigned flags[2] = {0, 0};
    if (rc == DS_OK && cudaMemcpyAsync(flags, L.gbar, sizeof(flags), cudaMemcpyDeviceToHost, st) != cudaSuccess) rc = DS_ERR_CUDA;
    cudaFreeAsync(tmp, st);
    DS_CUDA(cudaStreamSynchronize(st));
    DS_TRY(rc);
    DS_REQUIRE(flags[1] == 0, "ds_cheb32_solve: grid barrier timed out");
    *which_host = zc == Za ? 0 : 1;
    return DS_OK;
}

extern "C" int ds_spmm32_chunks(const int32_t* brow, int64_t n_nodes, int32_t* chunk_row, void* stream) {
    DS_REQUIRE(brow && chunk_row && n_nodes > 0, "ds_spmm32_chunks: bad argument");
    return spmm32_chunks(brow, n_nodes, chunk_row, (cudaStream_t)stream);
}

/* slab variant: brow_win = &brow[row0] (n_local + 1 entries of the GLOBAL row pointer), bcol / Kval / Mblk start
 * at the slab's first block; colmap[n_global_nodes] packs owner << 28 | index inside the owner's slab */
extern "C" int ds_k32_pack_slab(const int32_t* brow_win, const int32_t* bcol_slab, int64_t n_local, int64_t nnzb_local,
                                int64_t row0, const double* Kval_slab, const double* Mblk_slab, double shift,
                                const uint32_t* colmap, void* rec, float* invD, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    DS_REQUIRE(rec && colmap, "ds_k32_pack_slab: null argument");
    DS_CUDA(cudaMemsetAsync(reinterpret_cast<unsigned char*>(rec) + nnzb_local * S32_REC_BYTES, 0, 64, st));
    return pack_k32(brow_win, bcol_slab, n_local, Kval_slab, Mblk_slab, shift, rec, invD, st, colmap, row0);
}

extern "C" int ds_spmm32_rowpart(int mode, const int32_t* brow_local, const void* rec, int64_t n_local, int ncols,
                                 const float* const* Xparts_host, int world, int rank, const float* R, const float* invD,
                                 const float* Zprev, float* Out, double ab, double cc, void* stream) {
    DS_REQUIRE(mode >= 0 && mode <= 2, "ds_spmm32_rowpart: mode must be 0, 1 or 2");
    return spmm32_rowpart(mode, brow_local, rec, n_local, ncols, Xparts_host, world, rank, R, invD, Zprev, Out, (float)ab,
                          (float)cc, (cudaStream_t)stream);
}

/* peer-visible device memory: cudaMalloc + CUDA IPC handle (64 bytes) for the other ranks of the node */
extern "C" int ds_peer_alloc(int64_t bytes, void** ptr, unsigned char* handle64) {
    DS_REQUIRE(bytes > 0 && ptr && handle64, "ds_peer_alloc: bad argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    DS_CUDA(cudaMalloc(ptr, (size_t)bytes));
    cudaIpcMemHandle_t h;
    DS_CUDA(cudaIpcGetMemHandle(&h, *ptr));
    memcpy(handle64, &h, 64);
    return DS_OK;
}
extern "C" int ds_peer_open(const unsigned char* handle64, void** ptr) {
    DS_REQUIRE(handle64 && ptr, "ds_peer_open: bad argument");
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, 64);
    DS_CUDA(cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return DS_OK;
}
extern "C" int ds_peer_close(void* ptr) {
    if (ptr) DS_CUDA(cudaIpcCloseMemHandle(ptr));
    return DS_OK;
}
extern "C" int ds_peer_free(void* ptr) {
    if (ptr) DS_CUDA(cudaFree(ptr));
    return DS_OK;
}

extern "C" int ds_pmg_restrict32(const int32_t* rptr, const int32_t* rlist, int64_t n_coarse, const float* res,
                                 int ncols, float* rc, void* stream) {
    DS_REQUIRE(rptr && rlist && res && rc && ncols % 4 == 0, "ds_pmg_restrict32: bad argument");
    return restrict32(rptr, rlist, n_coarse, res, ncols, rc, (cudaStream_t)stream);
}

extern "C" int ds_pmg_prolong_add32(const int32_t* parents, int64_t n_fine, const float* zc, int ncols, float* z,
                                    void* stream) {
    DS_REQUIRE(parents && zc && z && ncols % 4 == 0, "ds_pmg_prolong_add32: bad argument");
    return prolong_add32(parents, n_fine, zc, ncols, z, (cudaStream_t)stream);
}

// Shared helpers for libdiffsound_sm100.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstdarg>

#define DS_OK 0
#define DS_ERR_CUDA -1
#define DS_ERR_ARG -2
#define DS_ERR_NOMEM -3
#define DS_ERR_NUMERIC -4

namespace ds {

void set_error(const char* fmt, ...);
void count_launch();

inline int check_cuda(cudaError_t e, const char* what, const char* file, int line) {
    if (e == cudaSuccess) return DS_OK;
    set_error("%s failed at %s:%d: %s", what, file, line, cudaGetErrorString(e));
    return DS_ERR_CUDA;
}

#define DS_CUDA(call)                                                          \
    do {                                                                       \
        int _rc = ::ds::check_cuda((call), #call, __FILE__, __LINE__);         \
        if (_rc != DS_OK) return _rc;                                          \
    } while (0)

// every kernel launch of the library is followed by this: error check + launch counter
#define DS_LAUNCH_CHECK()                                                      \
    do {                                                                       \
        ::ds::count_launch();                                                  \
        DS_CUDA(cudaGetLastError());                                           \
    } while (0)

#define DS_REQUIRE(cond, ...)                                                  \
    do {                                                                       \
        if (!(cond)) {                                                         \
            ::ds::set_error(__VA_ARGS__);                                      \
            return DS_ERR_ARG;                                                 \
        }                                                                      \
    } while (0)

#define DS_TRY(expr)                                                           \
    do {                                                                       \
        int _rc = (expr);                                                      \
        if (_rc != DS_OK) return _rc;                                          \
    } while (0)

inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

// Growable device scratch arena owned by a ds_workspace (the only allocation
// the library performs; everything else is caller-owned torch memory).
struct Arena {
    char* base = nullptr;
    size_t cap = 0;
    size_t used = 0;
    // stream of the previous reserve(): a call on a different stream is ordered behind everything queued there (one event),
    // so two torch streams of one host thread cannot race on the scratch.  (Concurrent host threads need one workspace each.)
    cudaStream_t last_stream = nullptr;
    bool have_stream = false;
    cudaEvent_t order_ev = nullptr;
    int reserve(size_t bytes, cudaStream_t s);
    void reset() { used = 0; }
    template <typename T>
    T* take(size_t count) {
        size_t off = (used + 255) & ~size_t(255);
        size_t need = off + count * sizeof(T);
        if (need > cap) return nullptr;
        used = need;
        return reinterpret_cast<T*>(base + off);
    }
    void release();
};

// Per-kernel-class device timing (CUDA events on the launch stream), off by default.
// bench.py turns it on to attribute the step to kernels without a profiler attached.
enum ProfClass {
    PROF_PATTERN = 0, PROF_GEOMETRY, PROF_ASSEMBLE, PROF_SPMM, PROF_CHEB, PROF_GRAM, PROF_GEMM, PROF_EIGH,
    PROF_RESIDUAL, PROF_COPY, PROF_GRAD, PROF_QUADFORM, PROF_SYNTH, PROF_OTHER, PROF_COARSE, PROF_TRANSFER, PROF_JACOBI,
    PROF_SDF_BUILD, PROF_SDF_QUERY, PROF_SDF_WINDING, PROF_NCLASS
};
bool prof_enabled(int cls);
void prof_begin(int cls, cudaStream_t s);
void prof_end(int cls, cudaStream_t s);
// algorithmic bytes / flops of a launch, accumulated per class while that class is being timed (bench.py: roofline_all)
void prof_account(int cls, double bytes, double flops);
struct ProfScope {
    int cls; cudaStream_t s; bool on;
    ProfScope(int c, cudaStream_t st) : cls(c), s(st), on(prof_enabled(c)) { if (on) prof_begin(cls, s); }
    ~ProfScope() { if (on) prof_end(cls, s); }
};

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

}  // namespace ds

struct ds_workspace {
    ds::Arena arena;
    // pattern-build state carried between ds_pattern_count and ds_pattern_fill
    uint64_t* sorted_keys = nullptr;
    uint32_t* sorted_vals = nullptr;
    uint32_t* slot_of_sorted = nullptr;
    int64_t n_pairs = 0;
    int64_t nnzb = 0;
    int num_sms = 0;
    ds_workspace* child = nullptr;   // arena of the nested coarse eigen-solve (created on first use)
    // state carried between the *_count and *_fill halves of the marching-tets / compaction / component calls (mtet.cu)
    void* mt_ptr[16] = {};
    int64_t mt_val[16] = {};
};

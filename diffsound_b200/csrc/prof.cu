// Optional per-kernel-class timing with CUDA events (see common.cuh: ProfScope).
// There is no nsys in the build image; this is how bench.py attributes a modal solve to its
// kernels on the device clock without a profiler attached.  Off by default (zero overhead: one
// branch per launch site).
#include "common.cuh"
#include "../../include/diffsound_sm100.h"
#include <atomic>
#include <mutex>
#include <vector>

namespace ds {

struct ProfState {
    bool on = false;
    uint32_t mask = 0xffffffffu;      // classes being timed while `on`
    std::mutex mu;
    struct Rec { cudaEvent_t a, b; int cls; };
    std::vector<Rec> pending;
    std::vector<cudaEvent_t> pool;
    cudaEvent_t open_ev[PROF_NCLASS] = {};
    double ms[PROF_NCLASS] = {};
    int64_t count[PROF_NCLASS] = {};
    double bytes[PROF_NCLASS] = {};
    double flops[PROF_NCLASS] = {};
};
static ProfState g_prof;

bool prof_enabled(int cls) { return g_prof.on && ((g_prof.mask >> cls) & 1u); }

static std::atomic<int64_t> g_launches{0};
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

static cudaEvent_t take_event() {
    if (!g_prof.pool.empty()) {
        cudaEvent_t e = g_prof.pool.back();
        g_prof.pool.pop_back();
        return e;
    }
    cudaEvent_t e;
    cudaEventCreate(&e);
    return e;
}

void prof_begin(int cls, cudaStream_t s) {
    std::lock_guard<std::mutex> lk(g_prof.mu);
    cudaEvent_t e = take_event();
    cudaEventRecord(e, s);
    g_prof.open_ev[cls] = e;
}

void prof_end(int cls, cudaStream_t s) {
    std::lock_guard<std::mutex> lk(g_prof.mu);
    cudaEvent_t e = take_event();
    cudaEventRecord(e, s);
    g_prof.pending.push_back({g_prof.open_ev[cls], e, cls});
}

void prof_account(int cls, double bytes, double flops) {
    if (!prof_enabled(cls)) return;
    std::lock_guard<std::mutex> lk(g_prof.mu);
    g_prof.bytes[cls] += bytes;
    g_prof.flops[cls] += flops;
}

static void drain() {
    for (auto& r : g_prof.pending) {
        float t = 0.f;
        if (cudaEventSynchronize(r.b) == cudaSuccess && cudaEventElapsedTime(&t, r.a, r.b) == cudaSuccess) {
            g_prof.ms[r.cls] += t;
            g_prof.count[r.cls] += 1;
        }
        g_prof.pool.push_back(r.a);
        g_prof.pool.push_back(r.b);
    }
    g_prof.pending.clear();
}

static const char* kNames[PROF_NCLASS] = {"pattern", "geometry", "assemble", "spmm", "cheb_step", "gram", "block_gemm",
                                          "eigh", "residual", "copy", "grad_shape", "quadforms", "synth", "other",
                                          "coarse_step", "transfer", "jacobi_scale", "sdf_build", "sdf_query",
                                          "sdf_winding"};

}  // namespace ds

using namespace ds;

extern "C" int ds_prof_enable(int on) {
    std::lock_guard<std::mutex> lk(g_prof.mu);
    g_prof.on = on != 0;
    g_prof.mask = 0xffffffffu;
    return DS_OK;
}

extern "C" int ds_prof_enable_classes(uint32_t mask) {
    std::lock_guard<std::mutex> lk(g_prof.mu);
    g_prof.on = mask != 0;
    g_prof.mask = mask;
    return DS_OK;
}

extern "C" int ds_prof_reset(void) {
    std::lock_guard<std::mutex> lk(g_prof.mu);
    drain();
    for (int c = 0; c < PROF_NCLASS; ++c) { g_prof.ms[c] = 0.0; g_prof.count[c] = 0; g_prof.bytes[c] = 0.0; g_prof.flops[c] = 0.0; }
    return DS_OK;
}

// Create `n` events up front.  cudaEventCreate inside a timed region is not free: when the driver's event pool runs out it
// allocates, which waits for the device -- one 100-220 ms step among 88 ms steps, always the step in which the ~128th event
// of the process was created (bench.py reserves before its timed regions).
extern "C" int ds_prof_reserve(int n) {
    std::lock_guard<std::mutex> lk(g_prof.mu);
    while ((int)g_prof.pool.size() < n) {
        cudaEvent_t e;
        DS_CUDA(cudaEventCreate(&e));
        g_prof.pool.push_back(e);
    }
    return DS_OK;
}

extern "C" int64_t ds_launch_count(void) { return g_launches.load(); }

extern "C" int ds_prof_num_classes(void) { return PROF_NCLASS; }

extern "C" const char* ds_prof_class_name(int cls) { return (cls >= 0 && cls < PROF_NCLASS) ? kNames[cls] : ""; }

extern "C" int ds_prof_read(int cls, double* ms, int64_t* count) {
    DS_REQUIRE(cls >= 0 && cls < PROF_NCLASS && ms && count, "ds_prof_read: bad argument");
    std::lock_guard<std::mutex> lk(g_prof.mu);
    drain();
    *ms = g_prof.ms[cls];
    *count = g_prof.count[cls];
    return DS_OK;
}

extern "C" int ds_prof_read_work(int cls, double* bytes, double* flops) {
    DS_REQUIRE(cls >= 0 && cls < PROF_NCLASS && bytes && flops, "ds_prof_read_work: bad argument");
    std::lock_guard<std::mutex> lk(g_prof.mu);
    *bytes = g_prof.bytes[cls];
    *flops = g_prof.flops[cls];
    return DS_OK;
}

// lmcma_internal.cuh — what the translation units of liblmcma_b200.so share: error helpers, the two handle types and the
// launch helpers that cross a file boundary.  The create-time tuning knobs and the launch plan: lmcma_plan.hpp.
//   lmcma_capi.cu        library / device queries, the optimiser entry points, the launchers, CUDA graphs
//   lmcma_plan.cpp       the launch plan of an optimiser handle: kernel builds, block sizes, grids, shared memory
//   lmcma_capi_map.cu    cost map handles, distance transform, the cost evaluator (k_cost, k_edt, k_brick)
//   lmcma_capi_state.cu  state getters / setters, the host-side pieces of the reference API
#pragma once
#include <cuda_runtime.h>
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <mutex>
#include <string>
#include <utility>
#include <vector>
#include "../../include/lmcma_b200.h"
#include "lmcma_host.hpp"
#include "lmcma_plan.hpp"
#include "lmcma_common.cuh"

namespace lmcma_capi {
using namespace lmcma;

extern thread_local std::string g_err;     // lmcma_capi.cu
extern std::atomic<long long> g_launches;
extern thread_local long long* g_capture_launches;   // while this thread captures a graph: its count of the kernels captured

inline int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

#define CU(call)                                                                                    \
    do {                                                                                            \
        cudaError_t e__ = (call);                                                                   \
        if (e__ != cudaSuccess)                                                                     \
            return fail(LMCMA_B200_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
    } while (0)
#define ARG(cond, msg)                                                   \
    do {                                                                 \
        if (!(cond)) return fail(LMCMA_B200_ERR_ARG, "%s (%s)", msg, #cond); \
    } while (0)

template <class T>
inline int dmalloc(T** p, size_t count) {
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(p), std::max<size_t>(count, 1) * sizeof(T));
    if (e != cudaSuccess) return fail(LMCMA_B200_ERR_NOMEM, "cudaMalloc(%zu bytes): %s", count * sizeof(T), cudaGetErrorString(e));
    e = cudaMemset(*p, 0, std::max<size_t>(count, 1) * sizeof(T));
    // the memset is asynchronous on the legacy stream, which the library's non-blocking streams do not wait for: without
    // this wait it can land AFTER a copy / kernel that one of those streams issues into the new buffer
    if (e == cudaSuccess) e = cudaStreamSynchronize(cudaStreamLegacy);
    if (e != cudaSuccess) return fail(LMCMA_B200_ERR_CUDA, "cudaMemset: %s", cudaGetErrorString(e));
    return 0;
}
#define DM(ptr, count)                              \
    do {                                            \
        int rc__ = dmalloc(&(ptr), (count));        \
        if (rc__) return rc__;                      \
    } while (0)

// Every kernel of the library is launched here.  Dynamic shared memory above 48 KiB is opted into; pdl makes the kernel a
// programmatic dependent of the kernel enqueued just before it on `st`.  The launch is counted in g_launches, or, while
// this thread captures a graph, in the graph's own count, which each replay adds (lmcma_capi.cu: capture / replay).
template <class... P, class... A>
int launch(void (*kern)(P...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, bool pdl, A&&... args) {
    if (smem > 48 * 1024) CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaLaunchAttribute attr;
    attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr.val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cfg.attrs = &attr; cfg.numAttrs = pdl ? 1 : 0;
    CU(cudaLaunchKernelEx(&cfg, kern, std::forward<A>(args)...));
    if (g_capture_launches) ++*g_capture_launches;
    else g_launches++;
    return 0;
}

// an instantiated CUDA graph and the number of kernels it holds (what one replay adds to lmcma_b200_launch_count)
struct Graph {
    cudaGraphExec_t exec = nullptr;
    int launches = 0;
};


struct DeviceProps {
    int sm_count = 0;
    size_t l2 = 0, smem_optin = 0, persist_max = 0;
    int cc = 0;
    bool ok = false;
    int cosched = -1;     // probe_coschedule: -1 not probed yet, 0 branches of a forked graph are serialised here, 1 they run concurrently
};
extern DeviceProps g_props[64];           // lmcma_capi.cu
inline int query_props(int device, DeviceProps** out) {
    ARG(device >= 0 && device < 64, "device ordinal out of range");
    DeviceProps& p = g_props[device];
    if (!p.ok) {
        cudaDeviceProp dp;
        CU(cudaGetDeviceProperties(&dp, device));
        p.sm_count = dp.multiProcessorCount;
        p.l2 = dp.l2CacheSize;
        p.smem_optin = dp.sharedMemPerBlockOptin;
        p.persist_max = dp.persistingL2CacheMaxSize;
        p.cc = dp.major * 10 + dp.minor;
        if (dp.major < 10) return fail(LMCMA_B200_ERR_CUDA, "device %d is sm_%d%d; this library is built for sm_100a only", device, dp.major, dp.minor);
        p.ok = true;
    }
    *out = &p;
    return 0;
}

}  // namespace lmcma_capi

// =================================================================================================
// handles (global namespace: the opaque types of include/lmcma_b200.h)
// =================================================================================================
struct lmcma_b200_map {
    int device = 0;
    lmcma_capi::Tuning tune;
    lmcma::MapDev dev{};
    int storage = 0;
    float c_min = 0.5f, scale = 1.f;
    size_t cells = 0, stored = 0;   // logical cells / stored elements (bricked, padded)
    float* d_g32 = nullptr;
    unsigned char* d_q8 = nullptr;
    float* d_lut = nullptr;
    bool persist = false;
    cudaStream_t stream = nullptr;   // private stream for the stand-alone evaluate calls
    // staging for the host-buffer evaluate path
    float* d_X = nullptr; size_t d_X_cap = 0;
    float* d_f = nullptr; int* d_nc = nullptr; int* d_ns = nullptr; size_t d_out_cap = 0;
    std::mutex host_path;            // lmcma_b200_cost_evaluate / cost_trace share the staging buffers and the private stream
};

struct lmcma_b200_opt {
    lmcma_b200_config cfg{};
    lmcma_capi::Tuning tune;
    lmcma::OptDev d{};
    lmcma_capi::DeviceProps* props = nullptr;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    // host mirrors
    std::vector<double> weights;       // mu
    std::vector<float> lo_f, hi_f;
    float* d_lo = nullptr; float* d_hi = nullptr; float* d_w = nullptr;
    // rng
    lmcma::HansenStream hansen{1};
    std::vector<float> z_host;         // staging for HANSEN
    bool needs_sample = false, pending_z = false;
    // reference one-at-a-time protocol
    int sample_idx = 0;
    std::vector<float> x_cache; bool x_cache_valid = false;
    std::vector<float> f_host;
    // attached cost
    lmcma_b200_map* map = nullptr;
    lmcma_b200_objective obj{};
    float* d_ends = nullptr;
    // graph
    lmcma_capi::Graph graph;                  // one fused generation (lmcma_b200_run)
    lmcma_capi::Graph graph_multi;            // Tuning::graph_unroll generations in one graph (lmcma_b200_run of many generations)
    cudaStream_t graph_built_for = nullptr;
    lmcma_capi::Graph tell_graph;             // tell_all of one query: H2D fitness -> k_rank -> k_sample, k_update on a side branch
    cudaStream_t tell_graph_for = nullptr;
    bool tell_graph_failed = false;
    // speculative update (k_update.cuh, UpdateArgs::phase): every tell_all graph ends with the fitness-independent part of the
    // NEXT generation's update (into d_spec, beside the sampler's tail and the candidates' trip across PCIe); the next tell_all
    // resumes from it (tell_graph_resume) unless anything else touched the optimiser's state in between
    lmcma_capi::Graph tell_graph_resume;
    float* d_spec = nullptr; size_t spec_stride = 0;
    bool spec_valid = false;
    bool tell_graph_spec = false;             // the tell graphs were captured with the speculative pass (host mirror on)
    float* f_pinned = nullptr;                // the graph's copy source (the caller's fitness array is copied here first)
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    bool have_run_timing = false;
    lmcma_capi::LaunchPlan plan;       // every kernel configuration, chosen at create (lmcma_plan.hpp)
    float* d_Lf = nullptr;             // lower Cholesky factor of the smoothness prior (n x ns FP32) or null
    bool mirror_dirty = true;          // the sequence-ordered pair mirror must be rebuilt (k_pack_pairs) before sampling
    lmcma::CostShape cost_shape;
    // fused generation with k_update on a side branch, concurrent with k_cost / k_rank (k_update.cuh): plan.overlap, until
    // something at run time rules it out (no side stream, the co-scheduling probe, a failed forked capture, check_lost)
    bool overlap = false;
    cudaStream_t side_stream = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    float* x_mirror = nullptr;        // page-locked, mapped host mirror of X (lmcma_b200_ask_all_view); OptDev::Xh is its device alias
    bool mirror_on = false, mirror_suppressed = false, xh_fresh = false;
    int* err_host = nullptr;          // page-locked, mapped: OptDev::err (a kernel of the overlapped generation gave up on its partner)
};


namespace lmcma_capi {
// ---- defined in lmcma_capi_map.cu ----
int launch_cost(const MapDev& mp, const CostArgs& a, int rows, int B, CostShape shape, bool trace, cudaStream_t st);
CostShape pick_cost_shape(int W, const float* start, const float* goal, int dims, const Tuning& tune);
int apply_l2_window(lmcma_b200_map* m, cudaStream_t st);
int check_obj(const lmcma_b200_map* m, const lmcma_b200_objective* obj);
void register_mirror(const void* host, size_t bytes, const float* dev, long long ld, int device);
void unregister_mirror(const void* host);
// ---- defined in lmcma_capi.cu ----
int check_lost(lmcma_b200_opt* o);

// dense <-> pitched copies
inline int d2h_rows(void* dst, const void* src, size_t rows, size_t width_bytes, size_t src_pitch_bytes, cudaStream_t st) {
    if (width_bytes == src_pitch_bytes) CU(cudaMemcpyAsync(dst, src, rows * width_bytes, cudaMemcpyDeviceToHost, st));   // dense: one 1-D copy
    else CU(cudaMemcpy2DAsync(dst, width_bytes, src, src_pitch_bytes, width_bytes, rows, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return 0;
}
inline int h2d_rows(void* dst, const void* src, size_t rows, size_t width_bytes, size_t dst_pitch_bytes, cudaStream_t st) {
    if (width_bytes == dst_pitch_bytes) CU(cudaMemcpyAsync(dst, src, rows * width_bytes, cudaMemcpyHostToDevice, st));
    else CU(cudaMemcpy2DAsync(dst, dst_pitch_bytes, src, width_bytes, width_bytes, rows, cudaMemcpyHostToDevice, st));
    CU(cudaStreamSynchronize(st));
    return 0;
}

}  // namespace lmcma_capi

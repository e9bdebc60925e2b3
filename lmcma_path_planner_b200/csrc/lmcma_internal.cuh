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

// The device buffers of a handle.  alloc fills a member slot of the handle (zeroed, as dmalloc), freeing what the slot
// held before, and records the slot; free_all releases every recorded slot, so a buffer cannot be left off a list at destroy.
struct DeviceBuffers {
    std::vector<void**> slots;
    template <class T>
    int alloc(T** slot, size_t count) {
        void** s = reinterpret_cast<void**>(slot);
        if (std::find(slots.begin(), slots.end(), s) == slots.end()) slots.push_back(s);
        if (*s) cudaFree(*s);
        *s = nullptr;
        return dmalloc(slot, count);
    }
    void free_all() {
        for (void** s : slots) { if (*s) cudaFree(*s); *s = nullptr; }
        slots.clear();
    }
};
// a device buffer of the handle `owner` into its member `slot`
#define DM(owner, slot, count)                                  \
    do {                                                        \
        int rc__ = (owner)->buffers.alloc(&(slot), (count));    \
        if (rc__) return rc__;                                  \
    } while (0)
// returns the code of an int-returning call that failed
#define TRY(call)                   \
    do {                            \
        int rc__ = (call);          \
        if (rc__) return rc__;      \
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

// the forked graphs of one query's tell (lmcma_capi.cu: ensure_tell_graph): the whole update, and the one that resumes from
// the rows a speculative pass left in d_spec
struct TellGraphs {
    Graph whole, resume;
    cudaStream_t built_for = nullptr;
    bool spec = false;                 // the graphs end with the speculative pass (tell_all with the host mirror on)
    bool failed = false;               // could not be built here: this tell takes the stream-ordered path for good
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
    lmcma_capi::DeviceBuffers buffers;   // every device buffer below but d_update (lmcma_b200_map_destroy frees them all)
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
    // built by lmcma_b200_map_create_from_occupancy (with this clamp): the storage encodes the occupancy, and
    // lmcma_b200_map_update_occupancy may edit it
    bool from_occupancy = false;
    float clamp = 0.f;
    // grow-only scratch of lmcma_b200_map_update_occupancy (stream-ordered on `stream`: growing it never synchronises the device)
    char* d_update = nullptr; size_t d_update_cap = 0;
    std::mutex host_path;            // lmcma_b200_cost_evaluate / cost_trace / map_update_occupancy share the staging buffers
                                     // and the private stream
};

struct lmcma_b200_opt {
    lmcma_b200_config cfg{};
    lmcma_capi::Tuning tune;
    lmcma::OptDev d{};
    lmcma_capi::DeviceBuffers buffers;    // every device buffer of the handle, d and the d_* members (DM)
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
    // The host's view of the device state: spec_valid, x_cache_valid, xh_fresh, sample_idx and mirror_dirty.  Entry points
    // change it through the transitions below (new_population, rows_written, state_written, pairs_written); besides those,
    // only the code that consumes a flag writes it: ensure_mirror, tell_all's replay, ask_all_view, ask_one / tell_one,
    // check_lost and the graph drop.
    // reference one-at-a-time protocol
    int sample_idx = 0;
    std::vector<float> x_cache; bool x_cache_valid = false;
    std::vector<float> f_host;
    // attached cost.  map: the map of a single-map handle, maps[0] of a multi-map one (lmcma_b200_attach_cost_maps), whose
    // dims, storage and device every map shares.  A multi-map handle (maps.size() > 1) keeps the MapDev table of its maps
    // (d_maps) and the map index of every instance (d_map_of, B ints, allocated at the first such attach and kept for the
    // handle's lifetime); cost_args_for hands both to k_cost
    lmcma_b200_map* map = nullptr;
    std::vector<lmcma_b200_map*> maps;
    lmcma::MapDev* d_maps = nullptr; size_t d_maps_cap = 0;
    int* d_map_of = nullptr;
    lmcma_b200_objective obj{};
    float* d_ends = nullptr;
    float* d_rescore = nullptr;        // B costs of best_x on the attached map (lmcma_b200_rescore_best)
    char* d_reset = nullptr;           // lmcma_b200_reset_instances stages its ResetArgs arrays here (reset_layout), from the first call on
    // graph
    lmcma_capi::Graph graph;                  // one fused generation (lmcma_b200_run)
    lmcma_capi::Graph graph_multi;            // Tuning::graph_unroll generations in one graph (lmcma_b200_run of many generations)
    cudaStream_t graph_built_for = nullptr;
    lmcma_capi::TellGraphs tell_host, tell_dev;  // the forked tell graphs of tell_all and of tell_all_dev (ensure_tell_graph)
    // lmcma_b200_tell_all_dev recorded generations into a caller's stream capture.  Their replays advance the state without
    // this library seeing them, so from then on no host-side record of the population is trusted (ask_all_view copies,
    // ask_one reloads) and a state setter rebuilds the pair mirror at once instead of at the next library launch
    bool caller_graphs = false;
    // speculative update (k_update.cuh, UpdateArgs::phase): with the host mirror on, every tell_all graph ends with the
    // fitness-independent part of the NEXT generation's update (into d_spec, beside the sampler's tail and the candidates' trip
    // across PCIe); the next tell_all resumes from it (tell_host.resume) unless anything else touched the state in between
    // (state_written)
    float* d_spec = nullptr; size_t spec_stride = 0;
    bool spec_valid = false;
    float* f_pinned = nullptr;                // the graph's copy source (the caller's fitness array is copied here first)
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    bool have_run_timing = false;
    lmcma_capi::LaunchPlan plan;       // every kernel configuration, chosen at create (lmcma_plan.hpp)
    float* d_Lf = nullptr;             // lower Cholesky factor of the smoothness prior (n x ns FP32) or null
    bool mirror_dirty = true;          // the sequence-ordered pair mirror must be rebuilt (k_pack_pairs) before sampling (pairs_written)
    lmcma::CostShape cost_shape;
    // fused generation with k_update on a side branch, concurrent with k_cost / k_rank (k_update.cuh): plan.overlap, until
    // something at run time rules it out (no side stream, the co-scheduling probe, a failed forked capture, check_lost)
    bool overlap = false;
    cudaStream_t side_stream = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    float* x_mirror = nullptr;        // page-locked, mapped host mirror of X (lmcma_b200_ask_all_view); OptDev::Xh is its device alias
    bool xh_fresh = false;            // x_mirror holds the population (the last sampler wrote it, or ask_all_view copied it)
    int* err_host = nullptr;          // page-locked, mapped: OptDev::err (a kernel of the overlapped generation gave up on its partner)
};


namespace lmcma_capi {
// ---- defined in lmcma_capi_map.cu ----
int launch_cost(const MapDev& mp, const CostArgs& a, int rows, int B, CostShape shape, bool trace, cudaStream_t st);
CostShape pick_cost_shape(int W, const float* start, const float* goal, int dims, const Tuning& tune);
int apply_l2_window(lmcma_b200_map* m, cudaStream_t st);
int check_obj(const lmcma_b200_map* m, const lmcma_b200_objective* obj);
void pack_ends(const lmcma_b200_endpoints* ends, int count, float* out);
void register_mirror(const void* host, size_t bytes, const float* dev, long long ld, int device);
void unregister_mirror(const void* host);
// ---- defined in lmcma_capi.cu ----
int check_lost(lmcma_b200_opt* o);

// ---- the transitions of the host's view of the device state ----
// The optimiser state was written by something other than the forked tell: whatever tell_all's speculative pass left in
// d_spec is stale.  Every entry point that writes the state calls it once its checks have passed.
inline void state_written(lmcma_b200_opt* o) { o->spec_valid = false; }
// d.X was written: ask_one's cache no longer holds it, nor does the host mirror unless the sampler that wrote d.X wrote the
// mirror too (mirror)
inline void rows_written(lmcma_b200_opt* o, bool mirror) {
    o->x_cache_valid = false;
    o->xh_fresh = mirror && o->x_mirror;
}
// A sampler has been enqueued or replayed (mirror: it wrote the host mirror): rows_written, and the one-at-a-time protocol
// starts at the first row.  A sampler that redraws some instances only (lmcma_b200_reset_instances) leaves the mirror fresh
// only if it was fresh before: it passes mirror && xh_fresh.
inline void new_population(lmcma_b200_opt* o, bool mirror) {
    rows_written(o, mirror);
    o->sample_idx = 0;
}
// The direction pairs (V, P, Nj, Lj, t, vec) were written from the host: the pair mirror is rebuilt before the next
// library sampler, or at once on a handle whose generations replay in a caller's graph (caller_graphs), because the next
// sampler to read it may be such a replay.  Defined in lmcma_capi.cu.
int pairs_written(lmcma_b200_opt* o);

// ---- the ERR_STATE preconditions several entry points share (`who`: the entry point, for the message) ----
inline int need_population(const lmcma_b200_opt* o, const char* who) {
    return o->needs_sample ? fail(LMCMA_B200_ERR_STATE, "%s: no population yet (rng INJECT: inject_z first)", who) : 0;
}
inline int need_unsplit(const lmcma_b200_opt* o, const char* who) {
    return o->d.pop_count != o->d.lambda
               ? fail(LMCMA_B200_ERR_STATE, "%s: not supported on a split-population handle (it takes the mg_* entry points)", who) : 0;
}
inline int need_philox(const lmcma_b200_opt* o, const char* who) {
    return o->cfg.rng != LMCMA_B200_RNG_PHILOX ? fail(LMCMA_B200_ERR_STATE, "%s needs the PHILOX rng", who) : 0;
}
// an attached cost: o->map, and with it the device end points d_ends (attach_body)
inline int need_cost(const lmcma_b200_opt* o, const char* who) {
    return o->map ? 0 : fail(LMCMA_B200_ERR_STATE, "%s: no cost attached (lmcma_b200_attach_cost)", who);
}
inline int need_batch_of_one(const lmcma_b200_opt* o, const char* who) {
    return o->d.B != 1 ? fail(LMCMA_B200_ERR_STATE, "%s needs batch == 1", who) : 0;
}

// The B Scalars of the handle through the host, in order on o->stream; both return when their copies are done.
// read_scalars calls f(b, const Scalars&) for every instance b; write_scalars lets f(b, Scalars&) edit a copy of every
// instance's Scalars and writes the copies back.
template <class F>
int read_scalars(lmcma_b200_opt* o, F&& f) {
    std::vector<Scalars> sc(o->d.B);
    CU(cudaMemcpyAsync(sc.data(), o->d.sc, sc.size() * sizeof(Scalars), cudaMemcpyDeviceToHost, o->stream));
    CU(cudaStreamSynchronize(o->stream));
    for (int b = 0; b < o->d.B; ++b) f(b, sc[b]);
    return 0;
}
template <class F>
int write_scalars(lmcma_b200_opt* o, F&& f) {
    std::vector<Scalars> sc(o->d.B);
    TRY(read_scalars(o, [&](int b, const Scalars& s) { sc[b] = s; f(b, sc[b]); }));
    CU(cudaMemcpyAsync(o->d.sc, sc.data(), sc.size() * sizeof(Scalars), cudaMemcpyHostToDevice, o->stream));
    CU(cudaStreamSynchronize(o->stream));
    return 0;
}

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

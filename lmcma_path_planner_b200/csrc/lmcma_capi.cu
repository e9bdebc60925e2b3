// lmcma_capi.cu — the C ABI declared in include/lmcma_b200.h: library / device queries, the optimiser entry points, the
// launchers of the sampler / rank / update kernels (their configuration: the handle's plan, lmcma_plan.cpp), the
// per-generation CUDA graphs, the split-population stages.
// No CPU fallback: every compute entry point needs a CUDA device.  Cost map + evaluator: lmcma_capi_map.cu; state
// access + host-side reference pieces: lmcma_capi_state.cu; shared declarations: lmcma_internal.cuh.
#include "lmcma_internal.cuh"
#include "k_rank.cuh"
#include "k_sample.cuh"
#include "k_update.cuh"
#include "k_prior.cuh"
#include "k_gram.cuh"
#include "k_reset.cuh"

using namespace lmcma;
using namespace lmcma_capi;

namespace lmcma_capi {
thread_local std::string g_err;
std::atomic<long long> g_launches{0};
thread_local long long* g_capture_launches = nullptr;
DeviceProps g_props[64];
}  // namespace lmcma_capi
namespace lmcma {
// error reporting for the other translation units of the library (lmcma_ingest.cpp)
int set_error(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    lmcma_capi::g_err = buf;
    return code;
}
}  // namespace lmcma

namespace {
// the three sampler families; block, grid and shared memory of every launch: o->plan.sample
template <int NV>
int launch_sample_t(lmcma_b200_opt* o, const OptDev& d, bool pdl, cudaStream_t st) {
    const auto& s = o->plan.sample;
    return launch(k_sample<NV, narrow_rb(NV), narrow_maxt(NV), narrow_spec(NV)>, dim3(s.ctas, d.B), s.threads, s.smem, st, pdl,
                  d, s.kc, s.stages);
}
template <int RBW>
int launch_sample_wide_t(lmcma_b200_opt* o, const OptDev& d, bool pdl, cudaStream_t st, int progressive) {
    const auto& s = o->plan.sample;
    return launch(k_sample_wide<RBW, wide_maxt(RBW)>, dim3(s.ctas, d.B), s.threads, s.smem, st, pdl, d, s.kc, s.stages, s.R, s.CW,
                  s.qpw, progressive);
}
template <int QW, int RL>
int launch_sample_rows_t(lmcma_b200_opt* o, const OptDev& d, bool pdl, cudaStream_t st) {
    const auto& s = o->plan.sample;
    return launch(k_sample_rows<QW, RL>, dim3(s.ctas, d.B), s.threads, s.smem, st, pdl, d, s.kc, s.stages, s.region);
}
int launch_sample_rows(lmcma_b200_opt* o, const OptDev& d, bool pdl, cudaStream_t st) {
    const bool two = o->plan.sample.rl == 2;
    switch (o->plan.sample.qw) {
        case 4: return two ? launch_sample_rows_t<4, 2>(o, d, pdl, st) : launch_sample_rows_t<4, 1>(o, d, pdl, st);
        case 7: return two ? launch_sample_rows_t<7, 2>(o, d, pdl, st) : launch_sample_rows_t<7, 1>(o, d, pdl, st);
        default: return two ? launch_sample_rows_t<8, 2>(o, d, pdl, st) : launch_sample_rows_t<8, 1>(o, d, pdl, st);
    }
}

int launch_sample_wide(lmcma_b200_opt* o, const OptDev& d, bool pdl, cudaStream_t st, int progressive) {
    return o->plan.sample.RBW == 2 ? launch_sample_wide_t<2>(o, d, pdl, st, progressive) : launch_sample_wide_t<4>(o, d, pdl, st, progressive);
}

// the sequence-ordered (v, pc) mirror k_sample streams from is maintained by k_update; after create or a state
// setter it is rebuilt from the slot-indexed arrays
int ensure_mirror(lmcma_b200_opt* o, cudaStream_t st) {
    if (!o->mirror_dirty) return 0;
    int rc = launch(k_pack_pairs, dim3(o->d.m, o->d.B), 128, 0, st, false, o->d);
    if (rc) return rc;
    o->mirror_dirty = false;
    return 0;
}

// mirror: write the host mirror of X too (if any, lmcma_b200_ask_all_view): the host-buffer protocol does; the fused
// generations (lmcma_b200_run), the device-resident tell and the split-population stages keep the candidates on the device
// pdl: launched as a programmatic dependent of the kernel enqueued just before it on `st` (k_update)
// progressive: that k_update was launched with UpdateArgs::progressive (only meaningful with pdl)
// only: OptDev::only, the instances to draw (the plain launch of lmcma_b200_reset_instances), or null for all of them
int launch_sample(lmcma_b200_opt* o, cudaStream_t st, bool mirror, bool pdl = false, bool progressive = false, int progressive_mode = 1,
                  const int* only = nullptr) {
    if (o->mirror_dirty) { int rc = ensure_mirror(o, st); if (rc) return rc; pdl = false; }
    OptDev d = o->d;
    d.only = only;
    if (o->d_Lf) {   // smoothness prior: z <- L z for the whole population before computeAz (lmcma.cpp:216-217)
        int rc = 0;
        if (o->cfg.rng == LMCMA_B200_RNG_PHILOX) rc = launch(k_gauss, dim3((d.ns / 4 + 127) / 128 * d.pop_count, 1, d.B), 128, 0, st, false, d);
        // every row: an instance k_gauss skipped still holds this generation's deviates in Z, so its Zc comes out unchanged
        const int rows = d.B * d.pop_count;
        if (!rc) rc = launch(k_prior, dim3((d.ns + 63) / 64 * ((rows + 63) / 64)), 256, 0, st, false, d.Z, o->d_Lf, d.Zc, rows, d.n, d.ns);
        if (rc) return rc;
        pdl = false;
    }
    if (!mirror) d.Xh = nullptr;
    if (o->plan.sample.kind == Sampler::ROWS) return launch_sample_rows(o, d, pdl, st);
    if (o->plan.sample.kind == Sampler::WIDE)
        return launch_sample_wide(o, d, pdl, st, (pdl && progressive && o->plan.progressive) ? progressive_mode : 0);
    switch (o->plan.sample.nv) {
        case 1: return launch_sample_t<1>(o, d, pdl, st);
        case 2: return launch_sample_t<2>(o, d, pdl, st);
        case 4: return launch_sample_t<4>(o, d, pdl, st);
        case 8: return launch_sample_t<8>(o, d, pdl, st);
        case 12: return launch_sample_t<12>(o, d, pdl, st);
        case 16: return launch_sample_t<16>(o, d, pdl, st);
    }
    return fail(LMCMA_B200_ERR_ARG, "unsupported n for k_sample (nv=%d)", o->plan.sample.nv);
}

// ranks + recombination partial sums (k_rank.cuh); RANK_PACK is the split-population stage
// pdl: launched as a programmatic dependent of the kernel enqueued just before it on `st` (k_cost)
int launch_rank(lmcma_b200_opt* o, const float* f_all, int mode, float* payload, cudaStream_t st, bool pdl = false) {
    const auto& r = o->plan.rank;
    if (r.tile_sorted) {                                          // lambda > 4096, unsplit: sort the fitness tiles first (k_rank.cuh)
        int rc = launch(k_rank_tiles, dim3((o->d.lambda + TELL_FTILE - 1) / TELL_FTILE, o->d.B), 1024, 0, st, pdl, o->d, f_all);
        if (rc) return rc;
        pdl = false;                                              // k_rank itself follows in stream order
    }
    return launch(k_rank<1024>, dim3(r.slices, o->d.B), r.threads, r.smem, st, pdl, o->d, f_all, mode, payload);
}

template <int NVB, int RMAX, bool SMEM, bool OVERLAP = false, int WARPS = UPD_WARPS>
int launch_update_t(lmcma_b200_opt* o, const UpdateArgs& a, bool pdl, cudaStream_t st) {
    return launch(k_update<NVB, RMAX, SMEM, OVERLAP, WARPS>, o->d.B, 32 * WARPS, o->plan.update.smem, st, pdl, o->d, a);
}

// the serial part of update() (k_update.cuh).  pdl: launched as a programmatic dependent of the kernel enqueued just
// before it on `st` (k_rank), so that its prologue overlaps that kernel
int launch_update(lmcma_b200_opt* o, const UpdateArgs& a, bool pdl, cudaStream_t st) {
    const auto& u = o->plan.update;
    if (u.gram) {
        int rc = u.nvb == 4 ? launch_update_t<4, -1, false>(o, a, pdl, st) : launch_update_t<16, -1, false>(o, a, pdl, st);
        if (rc) return rc;
        const OptDev& d = o->d;
        const int tiles = (d.m + GRAM_TILE - 1) / GRAM_TILE;
        if ((rc = launch(k_gram, dim3(tiles, tiles, d.B * GRAM_KS), 256, 0, st, false, d))) return rc;
        const auto& c = o->plan.coef;
        auto coef = c.elems == 5 ? k_coef<5> : (c.elems == 10 ? k_coef<10> : (c.elems == 12 ? k_coef<12> : k_coef<16>));
        if ((rc = launch(coef, d.B, c.threads, c.smem, st, false, d))) return rc;
        return launch(k_combine, dim3((d.ns / 4 + 127) / 128, (d.m + COMBINE_ROWS - 1) / COMBINE_ROWS, d.B), 128, 0, st, false, d);
    }
    if (u.nvb == 4) {
        if (a.overlap) {                                         // the overlapped generation (ensure_graph): register sweep only
            if (u.rmax == 3) return launch_update_t<4, 3, true, true>(o, a, pdl, st);
            if (u.rmax == 5) return launch_update_t<4, 5, true, true>(o, a, pdl, st);
            return fail(LMCMA_B200_ERR_STATE, "overlapped generation without the register sweep");
        }
        if (u.warps == 8) {                                      // batched instances: two CTAs of 8 warps per SM (plan_launch)
            if (u.rmax == 3) return launch_update_t<4, 3, true, false, 8>(o, a, pdl, st);
            if (u.rmax == 5) return launch_update_t<4, 5, true, false, 8>(o, a, pdl, st);
        }
        if (u.rmax == 3) return launch_update_t<4, 3, true>(o, a, pdl, st);
        if (u.rmax == 5) return launch_update_t<4, 5, true>(o, a, pdl, st);
        return u.rows_in_smem ? launch_update_t<4, 0, true>(o, a, pdl, st) : launch_update_t<4, 0, false>(o, a, pdl, st);
    }
    return u.rows_in_smem ? launch_update_t<16, 0, true>(o, a, pdl, st) : launch_update_t<16, 0, false>(o, a, pdl, st);
}

UpdateArgs update_args_local(lmcma_b200_opt* o) {
    UpdateArgs a;
    memset(&a, 0, sizeof(a));
    a.f_all = o->d.fit;
    a.slices = o->d.partial; a.n_slices = o->d.RS; a.slice_stride = o->d.ns; a.inst_stride = (long long)o->d.RS * o->d.ns;
    a.spec = o->d_spec; a.spec_stride = (long long)o->spec_stride;
    a.dbg = o->d.dbg ? o->d.dbg + TL_UPD : nullptr;
    return a;
}

// the k_cost arguments of the attached cost (callers have checked need_cost)
CostArgs cost_args_for(const lmcma_b200_opt* o) {
    CostArgs a;
    memset(&a, 0, sizeof(a));
    a.W = o->obj.waypoints; a.w_len = o->obj.w_len; a.w_clr = o->obj.w_clr; a.w_col = o->obj.w_col;
    a.X = o->d.X; a.ld = o->d.ns; a.inst_rows = o->d.pop_count;
    a.ends = o->d_ends; a.ends_per_instance = 1;
    a.f = o->d.fit; a.f_stride = o->d.lambda; a.f_offset = o->d.pop_offset;
    a.ncoll = o->d.ncoll; a.nsamp = o->d.nsamp;
    if (o->maps.size() > 1) { a.maps = o->d_maps; a.map_of = o->d_map_of; a.map_count = (int)o->maps.size(); }
    return a;
}

// every launch of the attached cost (the generations, rescore_best, profile_kernels): the map passed by value gives the
// build's dims and storage; with several maps k_cost reads each instance's map from the table in `a` (cost_args_for)
int launch_attached_cost(lmcma_b200_opt* o, const CostArgs& a, int rows, cudaStream_t st) {
    return launch_cost(o->map->dev, a, rows, o->d.B, o->cost_shape, false, st);
}

// the L2 persistence window of the attached map on `st`.  An access-policy window covers one address range: a handle on
// several maps sets none
int attached_l2_window(lmcma_b200_opt* o, cudaStream_t st) {
    return o->maps.size() > 1 ? 0 : apply_l2_window(o->map, st);
}

// lmcma_b200_rescore_best: best_f <- the cost of best_x on the map as it is now, for every instance that has been evaluated
// (canonicalised as k_update canonicalises a fitness before it compares it with best_f)
__global__ void k_set_best_f(Scalars* sc, const float* f, int B) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b < B && sc[b].counteval > 0) sc[b].best_f = (double)canon_fitness(f[b]);
}

// generate / stage deviates on the host for HANSEN mode, then sample
int host_rng_and_sample(lmcma_b200_opt* o, cudaStream_t st, bool mirror, bool progressive = false) {
    if (o->cfg.rng == LMCMA_B200_RNG_HANSEN) {
        const size_t rows = (size_t)o->d.pop_count;
        o->z_host.assign(rows * o->d.ns, 0.f);
        // the reference draws row by row, N deviates per offspring (lmcma.cpp:303-305, 212-215)
        for (size_t r = 0; r < rows; ++r)
            for (int k = 0; k < o->d.n; ++k) o->z_host[r * o->d.ns + k] = (float)o->hansen.gauss();
        CU(cudaMemcpyAsync(o->d.Z, o->z_host.data(), o->z_host.size() * sizeof(float), cudaMemcpyHostToDevice, st));
        CU(cudaStreamSynchronize(st));   // z_host is pageable and reused
    }
    return launch_sample(o, st, mirror, o->cfg.rng != LMCMA_B200_RNG_HANSEN, progressive);
}

// lmcma_b200_reset_instances(_dev): k_reset, then the sampler for the flagged instances only, a plain launch (the
// generation's PDL and hand-over pair a sampler with the k_update before it).  mirror: the sampler writes the flagged rows
// of the host mirror.  No graph is dropped: the captured ones read the state, the end points and the flags through pointers.
int enqueue_reset(lmcma_b200_opt* o, cudaStream_t st, ResetArgs a, bool mirror) {
    a.sigma_default = o->cfg.sigma0;
    a.d_ends = o->d_ends;
    state_written(o);                                            // the speculative pass saw the retired instances
    int rc = launch(k_reset, o->d.B, 256, 0, st, false, o->d, a);
    if (!rc) rc = launch_sample(o, st, mirror, false, false, 1, a.flags);
    if (rc) return rc;
    new_population(o, mirror && o->xh_fresh);                    // the other instances keep their rows
    return 0;
}

// where a generation's fitness comes from: k_cost on the attached map, a copy from f_pinned, or d.fit as it is
enum class Fit { COST, FROM_HOST, IN_PLACE };

int launch_own_cost(lmcma_b200_opt* o, cudaStream_t st) {
    return launch_attached_cost(o, cost_args_for(o), o->d.pop_count, st);
}

// One generation in stream order (fit: COST or IN_PLACE): [k_cost ->] k_rank -> k_update -> [HANSEN deviates ->] the
// sampler, or without the sampler (sample = false).  k_rank is a programmatic dependent of k_cost only.
int enqueue_linear(lmcma_b200_opt* o, cudaStream_t st, Fit fit, bool mirror, bool sample = true) {
    int rc;
    if (fit == Fit::COST && (rc = launch_own_cost(o, st))) return rc;
    if ((rc = launch_rank(o, o->d.fit, RANK_PLAIN, nullptr, st, fit == Fit::COST))) return rc;
    // device RNG: k_sample follows k_update directly and can take its outputs as they become final
    const bool prog = o->plan.progressive && o->cfg.rng == LMCMA_B200_RNG_PHILOX && !o->mirror_dirty;
    UpdateArgs ua = update_args_local(o);
    ua.progressive = prog ? 1 : 0;
    if ((rc = launch_update(o, ua, true, st))) return rc;
    return sample ? host_rng_and_sample(o, st, mirror, prog) : 0;
}

// the two branches of a forked graph: the side stream starts behind `st`, and `st` ends behind the side stream
int fork_side(lmcma_b200_opt* o, cudaStream_t st) {
    CU(cudaEventRecord(o->ev_fork, st));
    CU(cudaStreamWaitEvent(o->side_stream, o->ev_fork, 0));
    return 0;
}
int join_side(lmcma_b200_opt* o, cudaStream_t st) {
    CU(cudaEventRecord(o->ev_join, o->side_stream));
    CU(cudaStreamWaitEvent(st, o->ev_join, 0));
    return 0;
}

// One overlapped generation (DESIGN.md 4.3) for a graph.  Side branch: k_update [-> the speculative pass of the next one
// (spec)]; main branch: [the fitness from f_pinned ->] k_gate -> [k_cost ->] k_rank -> the sampler; joined at the end.
// phase: k_update's UpdateArgs::phase (0: the whole update; 2: resume from the rows the last speculative pass left)
int enqueue_forked(lmcma_b200_opt* o, cudaStream_t st, Fit fit, bool mirror, int phase = 0, bool spec = false) {
    const OptDev& d = o->d;
    UpdateArgs ua = update_args_local(o);
    ua.progressive = 1;                                          // the overlapped generation is a progressive one (plan_launch)
    ua.overlap = 1;
    ua.phase = phase;
    int rc;
    if ((rc = fork_side(o, st)) || (rc = launch_update(o, ua, false, o->side_stream))) return rc;
    if (spec) { UpdateArgs us = ua; us.phase = 1; us.dbg = nullptr; if ((rc = launch_update(o, us, false, o->side_stream))) return rc; }
    if (fit == Fit::FROM_HOST) CU(cudaMemcpyAsync(d.fit, o->f_pinned, (size_t)d.B * d.lambda * sizeof(float), cudaMemcpyHostToDevice, st));
    if ((rc = launch(k_gate, (d.B + 31) / 32, 32, 0, st, false, d))) return rc;   // until k_update has reset the flags and holds its SM
    if (fit == Fit::COST && (rc = launch_own_cost(o, st))) return rc;
    // the sampler is released when k_rank starts: the pairs it needs first are final (resume: at once; else as the sweep goes)
    if ((rc = launch_rank(o, d.fit, RANK_PLAIN | RANK_KEEP_FLAGS, nullptr, st, fit == Fit::COST))) return rc;
    if ((rc = launch_sample(o, st, mirror, true, true, 2))) return rc;
    return join_side(o, st);
}

// update() + sample() after the fitness of a generation is in d.fit.  INJECT without the next deviates stops after the
// update: inject_z samples
int generation_tail(lmcma_b200_opt* o, cudaStream_t st, bool mirror) {
    const bool sample = o->cfg.rng != LMCMA_B200_RNG_INJECT || o->pending_z;
    state_written(o);                                            // a whole update
    int rc = enqueue_linear(o, st, Fit::IN_PLACE, mirror, sample);
    if (rc) return rc;
    if (!sample) o->needs_sample = true;
    o->pending_z = false;
    new_population(o, sample && mirror);
    return 0;
}

// ---- CUDA graphs: built by capture(), replayed by replay(), freed by drop_fused_graphs / drop_tell_graphs ----
void drop(Graph& g) {
    if (g.exec) cudaGraphExecDestroy(g.exec);
    g = Graph{};
}
void drop_fused_graphs(lmcma_b200_opt* o) {
    drop(o->graph);
    drop(o->graph_multi);
}
// the tell graphs, and with them what their speculative pass left behind
void drop_tell_graphs(lmcma_b200_opt* o, TellGraphs& tg) {
    drop(tg.whole);
    drop(tg.resume);
    tg.built_for = nullptr;
    o->spec_valid = false;
}
void drop_tell_graphs(lmcma_b200_opt* o) {
    drop_tell_graphs(o, o->tell_host);
    drop_tell_graphs(o, o->tell_dev);
}

// while it lives, this thread's kernel launches are counted in *count instead of g_launches
struct CountLaunchesIn {
    explicit CountLaunchesIn(long long* count) { g_capture_launches = count; }
    ~CountLaunchesIn() { g_capture_launches = nullptr; }
};

// Records what body() enqueues on `st` (and on the streams it forks from `st`) into *g, which is empty.  Capture enqueues
// nothing: the kernels the body launches are counted in g->launches, and each replay adds them to g_launches.
template <class Body>
int capture(cudaStream_t st, Body&& body, Graph* g) {
    cudaGraph_t graph = nullptr;
    long long launches = 0;
    CountLaunchesIn counted(&launches);
    CU(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
    int rc = body();
    cudaError_t e = cudaStreamEndCapture(st, &graph);
    if (!rc && e == cudaSuccess) e = cudaGraphInstantiate(&g->exec, graph, 0);
    if (graph) cudaGraphDestroy(graph);
    if (!rc && e != cudaSuccess) rc = fail(LMCMA_B200_ERR_CUDA, "graph capture / instantiate failed: %s", cudaGetErrorString(e));
    if (rc) g->exec = nullptr;
    else g->launches = (int)launches;
    return rc;
}

int replay(const Graph& g, cudaStream_t st) {
    CU(cudaGraphLaunch(g.exec, st));
    g_launches += g.launches;
    return 0;
}

// The device-side entry points (tell_all_dev, reset_instances_dev) enqueue through here: enqueue(captured) on o->stream,
// captured when o->stream is in the caller's stream capture.  Then enqueue must replay or build no library graph and
// allocate or synchronise nothing; its kernels are counted by nobody (they run when the caller replays the graph), and
// the handle has caller_graphs from then on.
template <class Enqueue>
int enqueue_dev(lmcma_b200_opt* o, Enqueue&& enqueue) {
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    CU(cudaStreamIsCapturing(o->stream, &cs));
    if (cs == cudaStreamCaptureStatusNone) return enqueue(false);
    long long uncounted = 0;
    CountLaunchesIn counted(&uncounted);
    const int rc = enqueue(true);
    o->caller_graphs = true;
    return rc;
}

// LMCMA_B200_DBG: the device timeline (TimelineSlot) on stderr, in ns after its earliest stamp ("-": not stamped), then
// cleared, so that each print shows only what ran since the last one
int print_timeline(lmcma_b200_opt* o) {
    long long h[TL_SLOTS];
    CU(cudaMemcpyAsync(h, o->d.dbg, sizeof(h), cudaMemcpyDeviceToHost, o->stream));
    CU(cudaStreamSynchronize(o->stream));
    const long long* u = h + TL_UPD;
    long long t0 = 0;
    for (int i = 0; i < TL_SLOTS; ++i)
        if (h[i] && i != TL_UPD + TL_UPD_FIRST_STALE && i != TL_UPD + TL_UPD_LIVE && (!t0 || h[i] < t0)) t0 = h[i];
    auto at = [&](long long t) { t ? fprintf(stderr, "%lld", t - t0) : fprintf(stderr, "-"); };
    auto named = [&](const char* section, const long long* base, std::initializer_list<std::pair<const char*, int>> slots) {
        fprintf(stderr, "  %s:", section);
        for (const auto& s : slots) { fprintf(stderr, " %s=", s.first); at(base[s.second]); }
        fprintf(stderr, "\n");
    };
    auto series = [&](const char* name, const long long* t, int count) {
        fprintf(stderr, "    %s:", name);
        for (int i = 0; i < count; ++i) { fprintf(stderr, " "); at(t[i]); }
        fprintf(stderr, "\n");
    };
    fprintf(stderr, "device timeline (ns after the earliest stamp)\n");
    named("k_update", u, {{"start", TL_UPD_START}, {"bookkeeping", TL_UPD_BOOKKEEPING}, {"prologue", TL_UPD_PROLOGUE},
                          {"rows_final", TL_UPD_ROWS_FINAL}, {"ranks_seen", TL_UPD_RANKS_SEEN}, {"post_rank", TL_UPD_POST},
                          {"mean", TL_UPD_MEAN}, {"step_size", TL_UPD_STEP_SIZE}, {"best_copied", TL_UPD_BEST_COPIED},
                          {"newest_row", TL_UPD_NEWEST}, {"tail", TL_UPD_TAIL}, {"end", TL_UPD_END}});
    fprintf(stderr, "    first_stale=%lld live=%lld\n", u[TL_UPD_FIRST_STALE], u[TL_UPD_LIVE]);
    series("chain blocks", u + TL_UPD_CHAIN, TL_UPD_CHAIN_STAMPS);
    series("rows", u + TL_UPD_ROWS, TL_UPD_ROW_STAMPS);
    named("k_rank CTA 0", h, {{"start", TL_RANK_START}, {"ranked", TL_RANK_RANKED}, {"compacted", TL_RANK_COMPACTED},
                              {"gathered", TL_RANK_GATHERED}, {"stored", TL_RANK_STORED}, {"last_slice", TL_RANK_LAST_SLICE}});
    named("k_sample_wide CTA 0", h, {{"start", TL_SMP_START}, {"flags", TL_SMP_FLAGS}, {"scalars", TL_SMP_SCALARS}, {"z", TL_SMP_Z},
                                     {"first_pairs", TL_SMP_FIRST_PAIRS}, {"dots", TL_SMP_DOTS}, {"exchanged", TL_SMP_EXCHANGED},
                                     {"loop_done", TL_SMP_LOOP_DONE}, {"end", TL_SMP_END}});
    series("chunks", h + TL_SMP_CHUNK, TL_SMP_CHUNKS);
    CU(cudaMemsetAsync(o->d.dbg, 0, sizeof(h), o->stream));
    return 0;
}

// Do the two branches of a forked CUDA graph really run concurrently on this device, in this process?  (Not under a
// profiler / sanitizer that serialises kernels, not when someone else holds the SMs.)  Probed once per device with two
// one-thread kernels that shake hands within 5 ms; the second of two launches counts (the first pays module loading).
int probe_coschedule(lmcma_b200_opt* o) {
    if (o->props->cosched >= 0) return o->props->cosched;
    int result = 0;
    int* d = nullptr;
    Graph probe;
    cudaStream_t st = o->own_stream;
    if (cudaMalloc(&d, 4 * sizeof(int)) != cudaSuccess) { cudaGetLastError(); return 0; }
    bool ok = capture(st, [&] {
        int rc = fork_side(o, st);
        if (!rc) rc = launch(k_probe, 1, 1, 0, o->side_stream, false, d, d + 2, 0, 5000000ll);
        if (!rc) rc = launch(k_probe, 1, 1, 0, st, false, d, d + 2, 1, 5000000ll);
        return rc ? rc : join_side(o, st);
    }, &probe) == 0;
    for (int attempt = 0; attempt < 2 && ok; ++attempt) {
        int h[4] = {0, 0, 0, 0};
        ok = cudaMemcpyAsync(d, h, sizeof(h), cudaMemcpyHostToDevice, st) == cudaSuccess && replay(probe, st) == 0 &&
             cudaMemcpyAsync(h, d, sizeof(h), cudaMemcpyDeviceToHost, st) == cudaSuccess && cudaStreamSynchronize(st) == cudaSuccess;
        result = ok && h[2] == 1 && h[3] == 1;
    }
    drop(probe);
    cudaFree(d);
    cudaGetLastError();
    o->props->cosched = result;
    return result;
}

// A kernel of the overlapped generation gave up waiting for its partner (OptDev::err): report it ONCE, and keep the
// handle usable on the linear PDL graph from here on.  The generation in flight is void: the optimiser state must be
// restored by the caller (set_* from a checkpoint) or the handle recreated.
}  // namespace
int lmcma_capi::check_lost(lmcma_b200_opt* o) {
    if (!o->err_host || *reinterpret_cast<volatile int*>(o->err_host) == 0) return 0;
    const int code = *reinterpret_cast<volatile int*>(o->err_host);
    *reinterpret_cast<volatile int*>(o->err_host) = 0;
    o->overlap = false;
    o->props->cosched = 0;
    drop_fused_graphs(o);
    drop_tell_graphs(o);
    o->mirror_dirty = true;
    return fail(LMCMA_B200_ERR_CUDA, "overlapped generation lost co-scheduling (%s): the branches of the CUDA graph did not run "
                "concurrently (profiler / sanitizer / SMs held elsewhere).  This handle now uses the linear graph; the generation in "
                "flight is void - restore the state or recreate the handle (LMCMA_B200_OVERLAP=0 avoids the overlapped graph)",
                code == LOST_UPDATE_WAITING_FOR_RANK ? "k_update timed out waiting for k_rank" : "k_sample timed out waiting for k_update");
}
int lmcma_capi::pairs_written(lmcma_b200_opt* o) {
    o->mirror_dirty = true;
    if (!o->caller_graphs) return 0;                             // the next library sampler rebuilds it (ensure_mirror)
    int rc = ensure_mirror(o, o->stream);
    if (rc) return rc;
    CU(cudaStreamSynchronize(o->stream));
    return 0;
}
namespace {

// the fused graphs for o->stream, and the pair mirror their samplers read (a state setter since the last run made it dirty)
int ensure_graph(lmcma_b200_opt* o) {
    cudaStream_t st = o->stream;
    int rc = ensure_mirror(o, st);
    if (rc || (o->graph.exec && o->graph_built_for == st)) return rc;
    drop_fused_graphs(o);
    // `reps` generations in ONE graph: between two graph launches the device idles for the launch latency of the next one
    // (~5 us of a 52 us generation); inside a graph a generation follows the previous one as a plain dependency
    auto body = [&](int reps) -> int {
        int rc2 = 0;
        for (int g = 0; g < reps && !rc2; ++g)
            rc2 = o->overlap ? enqueue_forked(o, st, Fit::COST, false) : enqueue_linear(o, st, Fit::COST, false);
        return rc2;
    };
    rc = capture(st, [&] { return body(1); }, &o->graph);
    if (!rc && o->tune.graph_unroll > 1 && capture(st, [&] { return body(o->tune.graph_unroll); }, &o->graph_multi) != 0)
        cudaGetLastError();                                      // optional: the single one still works
    if (rc && o->overlap) {
        // the forked graph could not be built here (capture / instantiation of the side branch): fall back to the linear one
        cudaGetLastError();
        drop_fused_graphs(o);
        o->overlap = false;
        return ensure_graph(o);
    }
    if (rc) return rc;
    o->graph_built_for = st;
    return 0;
}

// Does this tell replay a forked graph?  One query with the overlapped generation, unless its graphs could not be built here
bool forked_tell(const lmcma_b200_opt* o, const TellGraphs& tg) { return o->overlap && !tg.failed && o->tune.tell_overlap != 0; }

// The tell of one query as a forked graph (see lmcma_b200_tell_all).  dev: the graph of lmcma_b200_tell_all_dev, which
// finds the fitness in d.fit already (no H2D node) and never writes the host mirror.  On failure the caller takes the
// stream-ordered path.
int ensure_tell_graph(lmcma_b200_opt* o, bool dev) {
    TellGraphs& tg = dev ? o->tell_dev : o->tell_host;
    cudaStream_t st = o->stream;
    int rc = ensure_mirror(o, st);
    if (rc || (tg.whole.exec && tg.built_for == st)) return rc;
    drop_tell_graphs(o, tg);
    const OptDev& d = o->d;
    if (!dev && !o->f_pinned && cudaHostAlloc(&o->f_pinned, (size_t)d.B * d.lambda * sizeof(float), cudaHostAllocDefault) != cudaSuccess) {
        cudaGetLastError(); o->f_pinned = nullptr; tg.failed = true; return 0;
    }
    // the speculative pass pays only where something hides it: with the host mirror on, the candidates' trip across PCIe
    // (35 us behind the sampler).  Without the mirror tell_all returns when the sampler is done, and a 25 us kernel behind
    // k_update would be the longer branch of the graph (measured: tell_all 57 -> 69 us).  tell_all_dev: not even when it
    // is left running beside the caller's cost (DESIGN.md 4.4)
    tg.spec = !dev && o->d_spec != nullptr && o->x_mirror != nullptr;
    const Fit fit = dev ? Fit::IN_PLACE : Fit::FROM_HOST;
    rc = capture(st, [&] { return enqueue_forked(o, st, fit, !dev, 0, tg.spec); }, &tg.whole);
    if (!rc && tg.spec) rc = capture(st, [&] { return enqueue_forked(o, st, fit, !dev, 2, tg.spec); }, &tg.resume);
    if (rc) {
        cudaGetLastError();
        drop_tell_graphs(o, tg);
        tg.failed = true;
        return 0;
    }
    tg.built_for = st;
    return 0;
}

}  // namespace

extern "C" {

int lmcma_b200_abi_version(void) { return LMCMA_B200_ABI_VERSION; }
const char* lmcma_b200_last_error(void) { return g_err.c_str(); }
int64_t lmcma_b200_launch_count(void) { return g_launches.load(); }

int lmcma_b200_device_count(int* count_out) {
    ARG(count_out, "null output");
    CU(cudaGetDeviceCount(count_out));
    return 0;
}
int lmcma_b200_device_info(int device, int* sm_count, int64_t* l2_bytes, int64_t* hbm_bytes, int* cc) {
    cudaDeviceProp dp;
    CU(cudaGetDeviceProperties(&dp, device));
    if (sm_count) *sm_count = dp.multiProcessorCount;
    if (l2_bytes) *l2_bytes = dp.l2CacheSize;
    if (hbm_bytes) *hbm_bytes = (int64_t)dp.totalGlobalMem;
    if (cc) *cc = dp.major * 10 + dp.minor;
    return 0;
}

// =================================================================================================
// optimiser
// =================================================================================================
int lmcma_b200_create(const lmcma_b200_config* cfg, const double* x0, const double* lo, const double* hi,
                      lmcma_b200_opt** out) {
    return lmcma_b200_create_with_prior(cfg, x0, lo, hi, nullptr, out);
}

static int create_body(lmcma_b200_opt* o, DeviceProps* props, const lmcma_b200_config* cfg, const double* x0, const double* lo,
                       const double* hi, const double* covariance);

int lmcma_b200_create_with_prior(const lmcma_b200_config* cfg, const double* x0, const double* lo, const double* hi,
                                 const double* covariance, lmcma_b200_opt** out) {
    ARG(cfg && out, "null pointer");
    ARG(cfg->n >= 1, "n must be >= 1");
    ARG(cfg->batch >= 1, "batch must be >= 1");
    ARG(cfg->rng >= 0 && cfg->rng <= 2, "unknown rng mode");
    ARG(cfg->sigma0 > 0.0, "sigma0 must be > 0");
    ARG(x0 || cfg->rng == LMCMA_B200_RNG_HANSEN, "x0 == NULL needs the HANSEN rng (uniform start, lmcma.cpp:161-163)");
    ARG(cfg->rng != LMCMA_B200_RNG_HANSEN || cfg->batch == 1, "HANSEN rng is a single serial stream: batch must be 1");
    DeviceProps* props;
    int rc = query_props(cfg->device, &props);
    if (rc) return rc;
    CU(cudaSetDevice(cfg->device));

    lmcma_b200_opt* o = new lmcma_b200_opt();
    rc = create_body(o, props, cfg, x0, lo, hi, covariance);   // any failure inside: everything allocated so far is released here
    if (rc) { const std::string keep = g_err; lmcma_b200_destroy(o); g_err = keep; return rc; }
    *out = o;
    return 0;
}

static int create_body(lmcma_b200_opt* o, DeviceProps* props, const lmcma_b200_config* cfg, const double* x0, const double* lo,
                       const double* hi, const double* covariance) {
    int rc = 0;
    o->tune = Tuning::from_env();
    o->cfg = *cfg;
    o->props = props;
    OptDev& d = o->d;
    d.n = cfg->n;
    d.ns = (cfg->n + 3) & ~3;
    d.lambda = cfg->lambda < 1 ? 4 + int(3 * std::log((double)cfg->n)) : cfg->lambda;   // lmcma.cpp:134-135
    d.mu = d.lambda / 2;                                                                  // lmcma.cpp:136
    d.m = cfg->m < 1 ? d.lambda : cfg->m;                                                 // lmcma.cpp:266
    d.B = cfg->batch;
    if (d.lambda < 2 || d.mu < 1 || d.m < 2) { return fail(LMCMA_B200_ERR_ARG, "need lambda >= 2 and m >= 2"); }
    d.pop_offset = cfg->pop_count < 1 ? 0 : cfg->pop_offset;
    d.pop_count = cfg->pop_count < 1 ? d.lambda : cfg->pop_count;
    if (d.pop_offset < 0 || d.pop_offset + d.pop_count > d.lambda) { return fail(LMCMA_B200_ERR_ARG, "population slice out of range"); }
    if (cfg->rng == LMCMA_B200_RNG_HANSEN && d.pop_count != d.lambda) { return fail(LMCMA_B200_ERR_ARG, "HANSEN rng cannot be split"); }
    std::string why;
    const PlanInput in{d.n, d.lambda, d.m, d.B, d.pop_count, cfg->rng, covariance != nullptr};
    if (!plan_launch(in, DeviceLimits{props->sm_count, props->smem_optin}, o->tune, &o->plan, &why)) return fail(LMCMA_B200_ERR_ARG, "%s", why.c_str());
    d.RS = o->plan.rank.slices;
    d.rank_ftile = o->plan.rank.ftile;
    d.rng_mode = cfg->rng;
    d.record_z = cfg->record_z;
    d.seed = (unsigned long long)cfg->seed;
    o->hansen.reseed(cfg->seed);

    // constants (lmcma.cpp:144-156, 238, 268-272)
    o->weights.resize(d.mu);
    double sw = 0;
    for (int i = 0; i < d.mu; ++i) { o->weights[i] = std::log(double(d.mu) + 0.5) - std::log(double(1 + i)); sw += o->weights[i]; }
    double mueff = 0;
    for (int i = 0; i < d.mu; ++i) { o->weights[i] /= sw; mueff += o->weights[i] * o->weights[i]; }
    d.mueff = 1.0 / mueff;
    d.c1 = 1.0 / (10 * std::log((double)(d.n + 1)));
    d.cc = 1.0 / d.m;
    d.cs = 0.3; d.target = 0.25;
    d.K = 1 / std::sqrt(1 - d.c1);
    d.M = std::sqrt(1 - d.c1);
    d.pc_coef = std::sqrt(d.cc * (2 - d.cc) * d.mueff);

    CU(cudaStreamCreateWithFlags(&o->own_stream, cudaStreamNonBlocking));
    o->stream = o->own_stream;
    CU(cudaEventCreate(&o->ev0));
    CU(cudaEventCreate(&o->ev1));

    const size_t B = d.B, ns = d.ns, lam = d.lambda, pc = d.pop_count, m = d.m;
    DM(o, d.X, B * pc * ns);
    DM(o, d.D, B * pc * ns);
    if (cfg->rng != LMCMA_B200_RNG_PHILOX || cfg->record_z || covariance) DM(o, d.Z, B * pc * ns);
    if (covariance) {   // CMABase::init factors the prior once (cholesky, lmcma.cpp:165-169)
        std::vector<double> Ld((size_t)d.n * d.n);
        if (!cholesky_lower(covariance, d.n, Ld.data())) { return fail(LMCMA_B200_ERR_ARG, "covariance prior is not symmetric positive definite"); }
        std::vector<float> Lf((size_t)d.n * ns, 0.f);
        for (int i = 0; i < d.n; ++i)
            for (int k = 0; k <= i; ++k) Lf[(size_t)i * ns + k] = (float)Ld[(size_t)i * d.n + k];
        DM(o, o->d_Lf, (size_t)d.n * ns);
        CU(cudaMemcpy(o->d_Lf, Lf.data(), Lf.size() * sizeof(float), cudaMemcpyHostToDevice));
        d.Lf = o->d_Lf;
        DM(o, d.Zc, B * pc * ns);
    }
    DM(o, d.fit, B * lam); DM(o, d.fit_sorted, B * lam); DM(o, d.prev_fit, B * lam);
    DM(o, d.rank, B * lam); DM(o, d.arindex, B * lam);
    if (o->plan.rank.tile_sorted) {
        DM(o, d.prev_sorted, B * lam); DM(o, d.tile_sorted, B * lam); DM(o, d.tile_pos, B * lam);
    }
    DM(o, d.ncoll, B * pc); DM(o, d.nsamp, B * pc);
    DM(o, d.xmean, B * ns); DM(o, d.pc, B * ns);
    DM(o, d.V, B * m * ns); DM(o, d.P, B * m * ns);
    DM(o, d.Nj, B * m); DM(o, d.Lj, B * m); DM(o, d.Njf, B * m); DM(o, d.Njs, B * m);
    DM(o, d.VPs, B * m * 2 * ns);
    DM(o, d.t, B * m); DM(o, d.vec, B * m);
    DM(o, d.sc, B); DM(o, d.best_x, B * ns); DM(o, d.S_count, B); DM(o, d.done_count, B); DM(o, d.progress, B * progress_len(m)); DM(o, d.rank_ticket, B); DM(o, d.resident, B);
    if (o->tune.dbg) DM(o, d.dbg, TL_SLOTS);
    DM(o, d.partial, B * d.RS * ns);

    std::vector<float> wf(o->weights.begin(), o->weights.end());
    DM(o, o->d_w, d.mu);
    CU(cudaMemcpy(o->d_w, wf.data(), d.mu * sizeof(float), cudaMemcpyHostToDevice));
    d.w = o->d_w;
    if (lo) {   // padded to the row stride so that the kernels clamp whole float4 columns
        o->lo_f.assign(d.ns, -std::numeric_limits<float>::max());
        for (int k = 0; k < d.n; ++k) o->lo_f[k] = (float)lo[k];
        DM(o, o->d_lo, d.ns);
        CU(cudaMemcpy(o->d_lo, o->lo_f.data(), d.ns * sizeof(float), cudaMemcpyHostToDevice));
        d.lo = o->d_lo;
    }
    if (hi) {
        o->hi_f.assign(d.ns, std::numeric_limits<float>::max());
        for (int k = 0; k < d.n; ++k) o->hi_f[k] = (float)hi[k];
        DM(o, o->d_hi, d.ns);
        CU(cudaMemcpy(o->d_hi, o->hi_f.data(), d.ns * sizeof(float), cudaMemcpyHostToDevice));
        d.hi = o->d_hi;
    }
    // initial mean (lmcma.cpp:158-163)
    std::vector<double> xm(B * ns, 0.0);
    for (size_t b = 0; b < B; ++b)
        for (int k = 0; k < d.n; ++k) xm[b * ns + k] = x0 ? x0[b * d.n + k] : o->hansen.uniform();
    CU(cudaMemcpy(d.xmean, xm.data(), xm.size() * sizeof(double), cudaMemcpyHostToDevice));
    rc = write_scalars(o, [&](int, Scalars& s) {
        memset(&s, 0, sizeof(s));
        s.sigma = cfg->sigma0; s.s = 0.0; s.best_f = std::numeric_limits<double>::max();
    });
    if (rc) return rc;

    o->overlap = o->plan.overlap;
    if (o->overlap) {
        cudaError_t e2 = cudaStreamCreateWithFlags(&o->side_stream, cudaStreamNonBlocking);
        if (e2 == cudaSuccess) e2 = cudaEventCreateWithFlags(&o->ev_fork, cudaEventDisableTiming);
        if (e2 == cudaSuccess) e2 = cudaEventCreateWithFlags(&o->ev_join, cudaEventDisableTiming);
        if (e2 == cudaSuccess) e2 = cudaHostAlloc(&o->err_host, sizeof(int), cudaHostAllocMapped);
        if (e2 == cudaSuccess) { *o->err_host = 0; e2 = cudaHostGetDevicePointer(&d.err, o->err_host, 0); }
        if (e2 != cudaSuccess) { cudaGetLastError(); o->overlap = false; d.err = nullptr; }
        // the overlapped generation needs the two branches of a forked graph to run CONCURRENTLY: enabled only where a probe
        // has seen that happen (LMCMA_B200_OVERLAP=2 skips the probe)
        if (o->overlap && o->tune.overlap != 2 && probe_coschedule(o) != 1) o->overlap = false;
        if (o->overlap && o->tune.tell_spec != 0) {              // scratch of the speculative update (best effort)
            o->spec_stride = (spec_floats(m, d.ns) + 3) & ~(size_t)3;
            if (o->buffers.alloc(&o->d_spec, B * o->spec_stride)) { cudaGetLastError(); o->d_spec = nullptr; }
            else cudaMemset(o->d_spec, 0xff, B * o->spec_stride * sizeof(float));   // generation -1: matches nothing
        }
    }
    if (o->plan.update.gram) {
        DM(o, d.G, B * GRAM_KS * m * m);
        DM(o, d.Cf, B * m * m);
        DM(o, d.gram_hdr, B);
    }
    o->f_host.assign(B * lam, 0.f);
    // first population (LMCMA::init -> sample(), lmcma.cpp:298)
    if (cfg->rng == LMCMA_B200_RNG_INJECT) o->needs_sample = true;
    else {
        rc = host_rng_and_sample(o, o->stream, true);
        if (!rc) { cudaError_t e = cudaStreamSynchronize(o->stream); if (e != cudaSuccess) rc = fail(LMCMA_B200_ERR_CUDA, "first sample: %s", cudaGetErrorString(e)); }
        if (rc) return rc;
        new_population(o, true);
    }
    return 0;
}

int lmcma_b200_destroy(lmcma_b200_opt* o) {
    if (!o) return 0;
    cudaSetDevice(o->cfg.device);
    if (o->stream) cudaStreamSynchronize(o->stream);
    o->buffers.free_all();
    drop_fused_graphs(o);
    drop_tell_graphs(o);
    if (o->f_pinned) cudaFreeHost(o->f_pinned);
    if (o->err_host) cudaFreeHost(o->err_host);
    if (o->x_mirror) { unregister_mirror(o->x_mirror); cudaFreeHost(o->x_mirror); }
    if (o->ev0) cudaEventDestroy(o->ev0);
    if (o->ev1) cudaEventDestroy(o->ev1);
    if (o->own_stream) cudaStreamDestroy(o->own_stream);
    if (o->side_stream) cudaStreamDestroy(o->side_stream);
    if (o->ev_fork) cudaEventDestroy(o->ev_fork);
    if (o->ev_join) cudaEventDestroy(o->ev_join);
    delete o;
    return 0;
}

int lmcma_b200_set_stream(lmcma_b200_opt* o, void* cuda_stream) {
    ARG(o, "null handle");
    CU(cudaStreamSynchronize(o->stream));
    o->stream = cuda_stream ? (cudaStream_t)cuda_stream : o->own_stream;
    return 0;
}

int lmcma_b200_shape(const lmcma_b200_opt* o, int32_t* out8) {
    ARG(o && out8, "null pointer");
    const OptDev& d = o->d;
    out8[0] = d.n; out8[1] = d.lambda; out8[2] = d.mu; out8[3] = d.m; out8[4] = d.B;
    out8[5] = d.pop_offset; out8[6] = d.pop_count; out8[7] = d.ns;
    return 0;
}

int lmcma_b200_inject_z(lmcma_b200_opt* o, const float* Z) {
    ARG(o && Z, "null pointer");
    if (o->cfg.rng != LMCMA_B200_RNG_INJECT) return fail(LMCMA_B200_ERR_STATE, "inject_z needs rng == INJECT");
    CU(cudaSetDevice(o->cfg.device));
    const OptDev& d = o->d;
    int rc = h2d_rows(d.Z, Z, (size_t)d.B * d.pop_count, d.n * sizeof(float), d.ns * sizeof(float), o->stream);
    if (rc) return rc;
    if (o->needs_sample) {
        o->needs_sample = false;
        rc = launch_sample(o, o->stream, true);
        if (rc) return rc;
        new_population(o, true);
        CU(cudaStreamSynchronize(o->stream));
    } else {
        o->pending_z = true;
    }
    return 0;
}

int lmcma_b200_resample(lmcma_b200_opt* o) {
    ARG(o, "null handle");
    TRY(need_population(o, "resample"));
    if (o->cfg.rng == LMCMA_B200_RNG_HANSEN) return fail(LMCMA_B200_ERR_STATE, "resample would advance the serial HANSEN stream");
    CU(cudaSetDevice(o->cfg.device));
    int rc = launch_sample(o, o->stream, true);
    if (rc) return rc;
    new_population(o, true);
    CU(cudaStreamSynchronize(o->stream));
    return 0;
}

int lmcma_b200_ask_all(lmcma_b200_opt* o, float* X) {
    ARG(o && X, "null pointer");
    TRY(need_population(o, "ask_all"));
    CU(cudaSetDevice(o->cfg.device));
    const OptDev& d = o->d;
    int rc = d2h_rows(X, d.X, (size_t)d.B * d.pop_count, d.n * sizeof(float), d.ns * sizeof(float), o->stream);
    return rc ? rc : check_lost(o);
}

int lmcma_b200_ask_all_view(lmcma_b200_opt* o, const float** X_view, int64_t* ld_out) {
    ARG(o && X_view, "null pointer");
    TRY(need_population(o, "ask_all_view"));
    CU(cudaSetDevice(o->cfg.device));
    OptDev& d = o->d;
    const size_t floats = (size_t)d.B * d.pop_count * d.ns;
    if (!o->x_mirror) {
        CU(cudaStreamSynchronize(o->stream));
        CU(cudaHostAlloc(&o->x_mirror, floats * sizeof(float), cudaHostAllocMapped));
        cudaError_t e = cudaHostGetDevicePointer(&d.Xh, o->x_mirror, 0);
        if (e != cudaSuccess) { cudaFreeHost(o->x_mirror); o->x_mirror = nullptr; d.Xh = nullptr; return fail(LMCMA_B200_ERR_CUDA, "cudaHostGetDevicePointer: %s", cudaGetErrorString(e)); }
        register_mirror(o->x_mirror, floats * sizeof(float), d.X, d.ns, o->cfg.device);
        // the captured graphs carry the old kernel parameters (OptDev by value): rebuild them on next use
        drop_tell_graphs(o);
    }
    // first use / after a fused run, a state setter or a tell_all_dev (or, once the caller has recorded generations: every
    // time): one ordinary copy
    if (!o->xh_fresh || o->caller_graphs) {
        CU(cudaMemcpyAsync(o->x_mirror, d.X, floats * sizeof(float), cudaMemcpyDeviceToHost, o->stream));
        o->xh_fresh = true;
    }
    CU(cudaStreamSynchronize(o->stream));
    *X_view = o->x_mirror;
    if (ld_out) *ld_out = d.ns;
    return check_lost(o);
}

int lmcma_b200_tell_all(lmcma_b200_opt* o, const float* f) {
    ARG(o && f, "null pointer");
    TRY(need_population(o, "tell_all"));
    TRY(need_unsplit(o, "tell_all"));
    CU(cudaSetDevice(o->cfg.device));
    const OptDev& d = o->d;
    int rc;
    if (forked_tell(o, o->tell_host)) {
        // One query (the conditions of the overlapped generation, DESIGN.md 4.3): everything in update() that does not
        // depend on this generation's fitness — slot bookkeeping, the sweep over every pending row but the newest — runs on
        // a side branch while the fitness crosses PCIe and k_rank runs; k_update then waits for k_rank's tickets and
        // k_sample follows its hand-over flags.  Same kernels and arithmetic as the fused generation (bit-identical to the
        // serial order), replayed as one CUDA graph: launched kernel by kernel, the fork / join costs more host time than
        // the overlap saves.
        if ((rc = ensure_tell_graph(o, false)) == 0 && o->tell_host.whole.exec) {
            memcpy(o->f_pinned, f, (size_t)d.B * d.lambda * sizeof(float));
            const bool resume = o->spec_valid && o->tell_host.resume.exec;   // the last tell left the next update's rows behind
            if ((rc = replay(resume ? o->tell_host.resume : o->tell_host.whole, o->stream))) return rc;
            o->spec_valid = o->tell_host.spec;                    // ... and so does this one
            new_population(o, true);
            CU(cudaStreamSynchronize(o->stream));
            return check_lost(o);
        }
        if (rc) return rc;
    }
    CU(cudaMemcpyAsync(d.fit, f, (size_t)d.B * d.lambda * sizeof(float), cudaMemcpyHostToDevice, o->stream));
    if ((rc = generation_tail(o, o->stream, true))) return rc;
    CU(cudaStreamSynchronize(o->stream));
    return 0;
}

int lmcma_b200_device_buffers(lmcma_b200_opt* o, const float** X_dev, int64_t* ld_out, float** f_dev) {
    ARG(o && X_dev && ld_out && f_dev, "null pointer");
    *X_dev = o->d.X;
    *ld_out = o->d.ns;
    *f_dev = o->d.fit;
    return 0;
}

int lmcma_b200_tell_all_dev(lmcma_b200_opt* o) {
    ARG(o, "null handle");
    TRY(need_philox(o, "tell_all_dev"));                         // HANSEN / INJECT: tell_all
    TRY(need_unsplit(o, "tell_all_dev"));
    CU(cudaSetDevice(o->cfg.device));
    return enqueue_dev(o, [&](bool captured) {
        // in the caller's capture, the linear generation (same bits as the forked one) keeps kernels that spin on a partner
        // out of a graph the library does not control
        if (!captured && forked_tell(o, o->tell_dev)) {
            // one query: the forked graph of tell_all without the fitness copy (and without the speculative pass, DESIGN.md 4.4)
            int rc = ensure_tell_graph(o, true);
            if (rc) return rc;
            if (o->tell_dev.whole.exec) {
                rc = replay(o->tell_dev.whole, o->stream);
                state_written(o);
                new_population(o, false);
                return rc;
            }
        }
        return generation_tail(o, o->stream, false);
    });
}

// what lmcma_b200_reset_instances(_dev) refuses with ERR_STATE: HANSEN / INJECT draw their deviates on the host, a split
// population's best and slots live on several handles, and end points need the device end points of an attached cost
static int reset_refused(const lmcma_b200_opt* o, bool ends) {
    TRY(need_philox(o, "reset_instances"));
    TRY(need_unsplit(o, "reset_instances"));
    return ends ? need_cost(o, "reset_instances with end points") : 0;
}

// o->d_reset: sigma0 (B doubles), x0 (B x n doubles), ends (B x 6 floats), flags (B ints), each at a 16-byte boundary
struct ResetLayout { size_t sigma0, x0, ends, flags, bytes; };
static ResetLayout reset_layout(const OptDev& d) {
    auto up = [](size_t v) { return (v + 15) & ~(size_t)15; };
    ResetLayout l;
    l.sigma0 = 0;
    l.x0 = up(l.sigma0 + (size_t)d.B * sizeof(double));
    l.ends = up(l.x0 + (size_t)d.B * d.n * sizeof(double));
    l.flags = up(l.ends + (size_t)d.B * 6 * sizeof(float));
    l.bytes = l.flags + (size_t)d.B * sizeof(int);
    return l;
}

int lmcma_b200_reset_instances(lmcma_b200_opt* o, int32_t count, const int32_t* idx, const double* x0, const double* sigma0,
                               const lmcma_b200_endpoints* ends) {
    ARG(o, "null handle");
    int rc = reset_refused(o, ends != nullptr);
    if (rc) return rc;
    ARG(count >= 0, "count must be >= 0");
    if (count == 0) return 0;
    ARG(idx && x0, "null pointer");
    const OptDev& d = o->d;
    const int n = d.n;
    std::vector<int> flags(d.B, 0);
    int lo = d.B, hi = -1;                                       // the rows the call touches: [lo, hi]
    for (int i = 0; i < count; ++i) {
        ARG(idx[i] >= 0 && idx[i] < d.B, "instance index out of range");
        ARG(flags[idx[i]] == 0, "instance index repeated");
        flags[idx[i]] = 1;
        lo = std::min(lo, idx[i]);
        hi = std::max(hi, idx[i]);
        ARG(!sigma0 || (std::isfinite(sigma0[i]) && sigma0[i] > 0.0), "sigma0 must be finite and > 0");
        for (int k = 0; k < n; ++k) ARG(std::isfinite(x0[(size_t)i * n + k]), "x0 must be finite");
    }
    CU(cudaSetDevice(o->cfg.device));
    const ResetLayout l = reset_layout(d);
    if (!o->d_reset) DM(o, o->d_reset, l.bytes);
    // only rows [lo, hi] of x0, sigma0 and the end points cross PCIe; the flags of every instance do
    const size_t rows = (size_t)(hi - lo + 1);
    std::vector<double> xs(rows * n), ss(rows, o->cfg.sigma0);
    std::vector<float> es(ends ? rows * 6 : 0);
    for (int i = 0; i < count; ++i) {
        const size_t r = (size_t)(idx[i] - lo);
        std::copy(x0 + (size_t)i * n, x0 + (size_t)(i + 1) * n, xs.begin() + r * n);
        if (sigma0) ss[r] = sigma0[i];
        if (ends) pack_ends(ends + i, 1, &es[r * 6]);
    }
    ResetArgs a;
    memset(&a, 0, sizeof(a));
    a.flags = reinterpret_cast<const int*>(o->d_reset + l.flags);
    a.x0 = reinterpret_cast<const double*>(o->d_reset + l.x0);
    a.sigma0 = reinterpret_cast<const double*>(o->d_reset + l.sigma0);
    a.ends = ends ? reinterpret_cast<const float*>(o->d_reset + l.ends) : nullptr;
    cudaStream_t st = o->stream;
    CU(cudaMemcpyAsync(o->d_reset + l.flags, flags.data(), flags.size() * sizeof(int), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(o->d_reset + l.x0 + (size_t)lo * n * sizeof(double), xs.data(), xs.size() * sizeof(double), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(o->d_reset + l.sigma0 + (size_t)lo * sizeof(double), ss.data(), ss.size() * sizeof(double), cudaMemcpyHostToDevice, st));
    if (ends) CU(cudaMemcpyAsync(o->d_reset + l.ends + (size_t)lo * 6 * sizeof(float), es.data(), es.size() * sizeof(float), cudaMemcpyHostToDevice, st));
    if ((rc = enqueue_reset(o, st, a, true))) return rc;
    CU(cudaStreamSynchronize(st));                               // the staging vectors are pageable
    return check_lost(o);
}

int lmcma_b200_reset_instances_dev(lmcma_b200_opt* o, const int32_t* flags_dev, const double* x0_dev, const double* sigma0_dev,
                                   const float* ends_dev, float* best_x_out_dev, double* best_f_out_dev) {
    ARG(o, "null handle");
    int rc = reset_refused(o, ends_dev != nullptr);
    if (rc) return rc;
    ARG(flags_dev && x0_dev, "null pointer");
    CU(cudaSetDevice(o->cfg.device));
    ResetArgs a;
    memset(&a, 0, sizeof(a));
    a.flags = flags_dev; a.x0 = x0_dev; a.sigma0 = sigma0_dev; a.ends = ends_dev;
    a.best_x_out = best_x_out_dev; a.best_f_out = best_f_out_dev;
    return enqueue_dev(o, [&](bool) { return enqueue_reset(o, o->stream, a, false); });
}

int lmcma_b200_ask_one(lmcma_b200_opt* o, double* params, int32_t n) {
    ARG(o && params, "null pointer");
    ARG(n == o->d.n, "N mismatch");
    TRY(need_batch_of_one(o, "ask_one"));
    TRY(need_unsplit(o, "ask_one"));
    if (!o->x_cache_valid || o->caller_graphs) {                  // a replay of the caller's graph may have moved on
        o->x_cache.resize((size_t)o->d.lambda * o->d.n);
        int rc = lmcma_b200_ask_all(o, o->x_cache.data());
        if (rc) return rc;
        o->x_cache_valid = true;
    }
    for (int k = 0; k < n; ++k) params[k] = (double)o->x_cache[(size_t)o->sample_idx * n + k];
    return 0;
}

int lmcma_b200_tell_one(lmcma_b200_opt* o, const double* feedbacks, int32_t num) {
    ARG(o && (feedbacks || num == 0) && num >= 0, "null pointer");
    TRY(need_batch_of_one(o, "tell_one"));
    TRY(need_unsplit(o, "tell_one"));
    double f = 0.0;                                    // lmcma.cpp:186-188
    for (int i = 0; i < num; ++i) f += feedbacks[i];
    // the device ranks FP32 values: keep huge penalties finite and ordered instead of letting them round to +-inf
    const double fmax = (double)std::numeric_limits<float>::max();
    o->f_host[o->sample_idx] = (float)(f > fmax ? fmax : (f < -fmax ? -fmax : f));
    if (++o->sample_idx % o->d.lambda == 0) {          // lmcma.cpp:199-204
        o->sample_idx = 0;
        return lmcma_b200_tell_all(o, o->f_host.data());
    }
    return 0;
}

int lmcma_b200_is_done(lmcma_b200_opt* o, int32_t* done) {
    ARG(o && done, "null pointer");
    CU(cudaSetDevice(o->cfg.device));
    return read_scalars(o, [&](int b, const Scalars& s) { done[b] = s.sigma < 1e-20 ? 1 : 0; });   // lmcma.cpp:426-429
}

// what attach_cost and attach_cost_maps share once their arguments are checked: the objective, the end points, the cost's
// launch shape, and the graphs that launched the previous cost.  The end points are on the device before o->map is set
// (need_cost: an attached cost has them)
static int attach_body(lmcma_b200_opt* o, lmcma_b200_map* map, const lmcma_b200_objective* obj, const lmcma_b200_endpoints* ends) {
    CU(cudaSetDevice(o->cfg.device));
    std::vector<float> e6((size_t)o->d.B * 6);
    pack_ends(ends, o->d.B, e6.data());
    if (!o->d_ends) DM(o, o->d_ends, (size_t)o->d.B * 6);
    CU(cudaMemcpy(o->d_ends, e6.data(), e6.size() * sizeof(float), cudaMemcpyHostToDevice));
    o->map = map; o->obj = *obj;
    o->cost_shape = pick_cost_shape(obj->waypoints, ends[0].start, ends[0].goal, map->dev.dims, o->tune);
    drop_fused_graphs(o);
    return 0;
}

int lmcma_b200_attach_cost(lmcma_b200_opt* o, lmcma_b200_map* map, const lmcma_b200_objective* obj,
                           const lmcma_b200_endpoints* ends) {
    ARG(o && ends, "null pointer");
    int rc = check_obj(map, obj);
    if (rc) return rc;
    ARG(map->device == o->cfg.device, "map and optimiser live on different devices");
    ARG(map->dev.dims * obj->waypoints == o->d.n, "n != dims * waypoints");
    o->maps.assign(1, map);
    return attach_body(o, map, obj, ends);
}

int lmcma_b200_attach_cost_maps(lmcma_b200_opt* o, int32_t map_count, lmcma_b200_map* const* maps, const int32_t* map_of,
                                const lmcma_b200_objective* obj, const lmcma_b200_endpoints* ends) {
    ARG(o && maps && map_of && obj && ends, "null pointer");
    TRY(need_unsplit(o, "attach_cost_maps"));                    // a split population takes one map: attach_cost
    ARG(map_count >= 1, "map_count must be >= 1");
    for (int k = 0; k < map_count; ++k) {
        ARG(maps[k], "null map");
        ARG(maps[k]->device == o->cfg.device, "map and optimiser live on different devices");
        ARG(maps[k]->dev.dims == maps[0]->dev.dims && maps[k]->storage == maps[0]->storage, "maps of different dims or storage");
    }
    int rc = check_obj(maps[0], obj);
    if (rc) return rc;
    ARG(maps[0]->dev.dims * obj->waypoints == o->d.n, "n != dims * waypoints");
    for (int b = 0; b < o->d.B; ++b) ARG(map_of[b] >= 0 && map_of[b] < map_count, "map_of entry outside [0, map_count)");
    if (map_count == 1) {                                        // a single-map handle, as attach_cost makes it
        o->maps.assign(1, maps[0]);
        return attach_body(o, maps[0], obj, ends);
    }
    CU(cudaSetDevice(o->cfg.device));
    // the table: MapDev is written by the map builds only (an occupancy update rewrites the storage it points to), so the
    // copy stays current for as long as the maps live
    std::vector<MapDev> table((size_t)map_count);
    for (int k = 0; k < map_count; ++k) table[k] = maps[k]->dev;
    if (o->d_maps_cap < (size_t)map_count) {
        o->d_maps_cap = 0;
        DM(o, o->d_maps, (size_t)map_count);
        o->d_maps_cap = (size_t)map_count;
    }
    if (!o->d_map_of) DM(o, o->d_map_of, (size_t)o->d.B);
    CU(cudaMemcpyAsync(o->d_maps, table.data(), table.size() * sizeof(MapDev), cudaMemcpyHostToDevice, o->stream));
    CU(cudaMemcpyAsync(o->d_map_of, map_of, (size_t)o->d.B * sizeof(int), cudaMemcpyHostToDevice, o->stream));
    CU(cudaStreamSynchronize(o->stream));
    o->maps.assign(maps, maps + map_count);
    return attach_body(o, maps[0], obj, ends);
}

int lmcma_b200_instance_maps_dev(lmcma_b200_opt* o, int32_t** map_of_dev) {
    ARG(o && map_of_dev, "null pointer");
    if (o->maps.size() < 2) return fail(LMCMA_B200_ERR_STATE, "instance_maps_dev: the handle is not attached to several maps (attach_cost_maps)");
    *map_of_dev = o->d_map_of;
    return 0;
}

int lmcma_b200_run(lmcma_b200_opt* o, int32_t generations) {
    ARG(o && generations >= 0, "bad argument");
    TRY(need_cost(o, "run"));
    TRY(need_population(o, "run"));
    TRY(need_unsplit(o, "run"));
    if (o->cfg.rng == LMCMA_B200_RNG_INJECT && generations > 1)
        return fail(LMCMA_B200_ERR_STATE, "INJECT rng: run one generation per injected Z");
    CU(cudaSetDevice(o->cfg.device));
    state_written(o);
    int rc = attached_l2_window(o, o->stream);
    if (rc) return rc;
    if (o->cfg.rng == LMCMA_B200_RNG_PHILOX) {
        if ((rc = ensure_graph(o))) return rc;
        CU(cudaEventRecord(o->ev0, o->stream));                  // after the (host-side) graph build: last_run_ms is device time
        const int unroll = o->graph_multi.exec ? o->tune.graph_unroll : 0;
        for (int g = 0; g < generations;) {
            const bool multi = unroll > 1 && generations - g >= unroll;
            if ((rc = replay(multi ? o->graph_multi : o->graph, o->stream))) return rc;
            g += multi ? unroll : 1;
        }
        if (generations > 0) new_population(o, false);           // the graph's sampler does not write the host mirror
    } else {
        CU(cudaEventRecord(o->ev0, o->stream));
        for (int g = 0; g < generations; ++g)
            if ((rc = launch_own_cost(o, o->stream)) || (rc = generation_tail(o, o->stream, true))) return rc;
    }
    CU(cudaEventRecord(o->ev1, o->stream));
    o->have_run_timing = true;
    return 0;
}

int lmcma_b200_sync(lmcma_b200_opt* o) {
    ARG(o, "null handle");
    CU(cudaSetDevice(o->cfg.device));
    CU(cudaStreamSynchronize(o->stream));
    { int lost = check_lost(o); if (lost) return lost; }
    return o->d.dbg ? print_timeline(o) : 0;
}

int lmcma_b200_last_run_ms(lmcma_b200_opt* o, float* ms) {
    ARG(o && ms, "null pointer");
    if (!o->have_run_timing) return fail(LMCMA_B200_ERR_STATE, "no run yet");
    CU(cudaEventSynchronize(o->ev1));
    CU(cudaEventElapsedTime(ms, o->ev0, o->ev1));
    return 0;
}

int lmcma_b200_profile_kernels(lmcma_b200_opt* o, int32_t generations, float* ms4) {
    ARG(o && ms4 && generations >= 1, "bad argument");
    TRY(need_cost(o, "profile_kernels"));
    TRY(need_philox(o, "profile_kernels"));
    CU(cudaSetDevice(o->cfg.device));
    const CostArgs ca = cost_args_for(o);
    cudaStream_t st = o->stream;
    std::vector<cudaEvent_t> ev((size_t)generations * 5);
    for (auto& e : ev) CU(cudaEventCreate(&e));
    state_written(o);
    int rc = 0;
    for (int g = 0; g < generations && !rc; ++g) {
        cudaEvent_t* e = &ev[(size_t)g * 5];
        cudaEventRecord(e[0], st);
        rc = launch_attached_cost(o, ca, o->d.pop_count, st);
        cudaEventRecord(e[1], st);
        if (!rc) rc = launch_rank(o, o->d.fit, RANK_PLAIN, nullptr, st);
        cudaEventRecord(e[2], st);
        if (!rc) rc = launch_update(o, update_args_local(o), false, st);   // serialised here so that the events separate the kernels
        cudaEventRecord(e[3], st);
        if (!rc) rc = launch_sample(o, st, true);
        cudaEventRecord(e[4], st);
    }
    new_population(o, true);
    cudaError_t se = cudaStreamSynchronize(st);
    if (!rc && se != cudaSuccess) rc = fail(LMCMA_B200_ERR_CUDA, "profile run: %s", cudaGetErrorString(se));
    if (!rc && o->d.dbg) rc = print_timeline(o);
    if (!rc && o->d.dbg && o->maps.size() > 1)
        fprintf(stderr, "k_cost timeline: skipped, a handle on several maps has no TRACE build of k_cost\n");
    else if (!rc && o->d.dbg) {     // and the per-CTA timeline of k_cost (phase stamps): one extra launch of its TRACE build
        const size_t ctas = (size_t)o->d.pop_count * o->d.B;
        long long* dbg = nullptr;
        if (cudaMalloc(&dbg, ctas * 8 * sizeof(long long)) == cudaSuccess) {
            std::vector<long long> h(ctas * 8);
            cudaMemsetAsync(dbg, 0, h.size() * sizeof(long long), st);
            CostArgs cd = ca; cd.dbg = dbg; cd.cells = nullptr; cd.max_cells = 0;
            launch_cost(o->map->dev, cd, o->d.pop_count, o->d.B, o->cost_shape, true, st);   // the TRACE build carries the stamps (no cells requested)
            cudaMemcpyAsync(h.data(), dbg, h.size() * sizeof(long long), cudaMemcpyDeviceToHost, st);
            cudaStreamSynchronize(st);
            long long t0 = h[0];
            for (size_t c = 0; c < ctas; ++c) t0 = std::min(t0, h[c * 8]);
            static const char* nm[] = {"start", "x loaded", "phase 1 done", "loop done", "end samples done", "end"};
            fprintf(stderr, "k_cost timeline over %zu CTAs (ns since the first CTA start; min / median / max):", ctas);
            for (int k = 0; k < 6; ++k) {
                std::vector<long long> v(ctas);
                for (size_t c = 0; c < ctas; ++c) v[c] = h[c * 8 + k] - t0;
                std::sort(v.begin(), v.end());
                fprintf(stderr, " %s=%lld/%lld/%lld", nm[k], v[0], v[ctas / 2], v[ctas - 1]);
            }
            // per-CTA durations of the phases
            static const char* dn[] = {"x load", "phase 1", "loop", "end samples", "reduce"};
            fprintf(stderr, " | per-CTA phase durations (median):");
            for (int k = 0; k < 5; ++k) {
                std::vector<long long> v(ctas);
                for (size_t c = 0; c < ctas; ++c) v[c] = h[c * 8 + k + 1] - h[c * 8 + k];
                std::sort(v.begin(), v.end());
                fprintf(stderr, " %s=%lld", dn[k], v[ctas / 2]);
            }
            fprintf(stderr, "\n");
            cudaFree(dbg);
        }
    }
    for (int k = 0; k < 4; ++k) ms4[k] = 0.f;
    if (!rc)
        for (int g = 0; g < generations; ++g)
            for (int k = 0; k < 4; ++k) {
                float ms = 0.f;
                cudaEventElapsedTime(&ms, ev[(size_t)g * 5 + k], ev[(size_t)g * 5 + k + 1]);
                ms4[k] += ms / generations;
            }
    for (auto& e : ev) cudaEventDestroy(e);
    return rc;
}

int lmcma_b200_best(lmcma_b200_opt* o, float* x_best, float* f_best) {
    ARG(o, "null handle");
    CU(cudaSetDevice(o->cfg.device));
    const OptDev& d = o->d;
    if (x_best) {
        int rc = d2h_rows(x_best, d.best_x, d.B, d.n * sizeof(float), d.ns * sizeof(float), o->stream);
        if (rc) return rc;
    }
    return f_best ? read_scalars(o, [&](int b, const Scalars& s) { f_best[b] = (float)s.best_f; }) : 0;
}

int lmcma_b200_rescore_best(lmcma_b200_opt* o) {
    ARG(o, "null handle");
    TRY(need_cost(o, "rescore_best"));
    TRY(need_unsplit(o, "rescore_best"));                        // best_x may hold a peer's row
    CU(cudaSetDevice(o->cfg.device));
    const OptDev& d = o->d;
    if (!o->d_rescore) DM(o, o->d_rescore, (size_t)d.B);
    state_written(o);                                            // like the state setters: tell_all's speculative pass saw the old best
    CostArgs ca = cost_args_for(o);
    ca.X = d.best_x; ca.inst_rows = 1;                           // one row per instance, the instance's own end points
    ca.f = o->d_rescore; ca.f_stride = 1; ca.f_offset = 0; ca.ncoll = nullptr; ca.nsamp = nullptr;
    int rc = attached_l2_window(o, o->stream);
    if (rc) return rc;
    if ((rc = launch_attached_cost(o, ca, 1, o->stream))) return rc;   // each instance's best_x on its own map
    if ((rc = launch(k_set_best_f, (unsigned)((d.B + 127) / 128), 128, 0, o->stream, false, d.sc, (const float*)o->d_rescore, d.B))) return rc;
    CU(cudaStreamSynchronize(o->stream));
    return 0;
}

// ---- split-population mode ---------------------------------------------------------------------
int lmcma_b200_mg_payload_floats(lmcma_b200_opt* o, int32_t* floats_out) {
    ARG(o && floats_out, "null pointer");
    *floats_out = o->d.ns + 4;
    return 0;
}

int lmcma_b200_mg_evaluate(lmcma_b200_opt* o, float* f_local_dev, void* stream) {
    ARG(o && f_local_dev, "null pointer");
    TRY(need_batch_of_one(o, "mg_evaluate"));
    TRY(need_population(o, "mg_evaluate"));
    TRY(need_cost(o, "mg_evaluate"));
    CU(cudaSetDevice(o->cfg.device));
    CostArgs ca = cost_args_for(o);
    ca.f = f_local_dev; ca.f_stride = o->d.pop_count; ca.f_offset = 0;
    cudaStream_t st = stream ? (cudaStream_t)stream : o->stream;
    int rc = apply_l2_window(o->map, st);
    if (rc) return rc;
    return launch_cost(o->map->dev, ca, o->d.pop_count, o->d.B, o->cost_shape, false, st);
}

int lmcma_b200_mg_rank(lmcma_b200_opt* o, const float* f_all_dev, float* payload_dev, void* stream) {
    ARG(o && f_all_dev && payload_dev, "null pointer");
    TRY(need_batch_of_one(o, "mg_rank"));
    CU(cudaSetDevice(o->cfg.device));
    cudaStream_t st = stream ? (cudaStream_t)stream : o->stream;
    // keep the gathered fitness: k_update needs it for prev_fit / best tracking
    CU(cudaMemcpyAsync(o->d.fit, f_all_dev, (size_t)o->d.lambda * sizeof(float), cudaMemcpyDeviceToDevice, st));
    return launch_rank(o, o->d.fit, RANK_PACK, payload_dev, st);
}

int lmcma_b200_mg_update(lmcma_b200_opt* o, const float* payload_all_dev, int32_t world, void* stream) {
    ARG(o && payload_all_dev && world >= 1, "bad argument");
    TRY(need_philox(o, "mg_update"));
    CU(cudaSetDevice(o->cfg.device));
    cudaStream_t st = stream ? (cudaStream_t)stream : o->stream;
    const long long pf = o->d.ns + 4;
    UpdateArgs a;
    memset(&a, 0, sizeof(a));
    a.f_all = o->d.fit; a.slices = payload_all_dev; a.n_slices = world;
    a.slice_stride = (long long)o->d.B * pf; a.inst_stride = pf; a.payload_mode = 1;
    state_written(o);
    int rc = launch_update(o, a, false, st);
    if (!rc) rc = launch_sample(o, st, false, true);
    new_population(o, false);
    return rc;
}

}  // extern "C"

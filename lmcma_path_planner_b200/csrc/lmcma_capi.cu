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

// pdl: launched as a programmatic dependent of the kernel enqueued just before it on `st` (k_update)
// progressive: that k_update was launched with UpdateArgs::progressive (only meaningful with pdl)
int launch_sample(lmcma_b200_opt* o, cudaStream_t st, bool pdl = false, bool progressive = false, int progressive_mode = 1) {
    if (o->mirror_dirty) { int rc = ensure_mirror(o, st); if (rc) return rc; pdl = false; }
    if (o->d_Lf) {   // smoothness prior: z <- L z for the whole population before computeAz (lmcma.cpp:216-217)
        const OptDev& d = o->d;
        int rc = 0;
        if (o->cfg.rng == LMCMA_B200_RNG_PHILOX) rc = launch(k_gauss, dim3((d.ns / 4 + 127) / 128, d.pop_count, d.B), 128, 0, st, false, d);
        const int rows = d.B * d.pop_count;
        if (!rc) rc = launch(k_prior, dim3((d.ns + 63) / 64, (rows + 63) / 64), 256, 0, st, false, d.Z, o->d_Lf, d.Zc, rows, d.n, d.ns);
        if (rc) return rc;
        pdl = false;
    }
    // the host mirror of X (lmcma_b200_ask_all_view) is written by the samplers of the host-buffer protocol only: the fused
    // on-device generations (lmcma_b200_run) and the split-population stages keep the candidates on the device
    OptDev d = o->d;
    if (!o->mirror_on || o->mirror_suppressed) d.Xh = nullptr;
    o->xh_fresh = d.Xh != nullptr;
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
    if (a.phase == 0) o->spec_valid = false;                        // a whole update: whatever the speculative pass left is stale
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

int cost_args_for(lmcma_b200_opt* o, CostArgs* a) {
    if (!o->map) return fail(LMCMA_B200_ERR_STATE, "no cost attached (call lmcma_b200_attach_cost)");
    memset(a, 0, sizeof(*a));
    a->W = o->obj.waypoints; a->w_len = o->obj.w_len; a->w_clr = o->obj.w_clr; a->w_col = o->obj.w_col;
    a->X = o->d.X; a->ld = o->d.ns; a->inst_rows = o->d.pop_count;
    a->ends = o->d_ends; a->ends_per_instance = 1;
    a->f = o->d.fit; a->f_stride = o->d.lambda; a->f_offset = o->d.pop_offset;
    a->ncoll = o->d.ncoll; a->nsamp = o->d.nsamp;
    return 0;
}

// generate / stage deviates on the host for HANSEN mode, then sample
int host_rng_and_sample(lmcma_b200_opt* o, cudaStream_t st, bool progressive = false) {
    if (o->cfg.rng == LMCMA_B200_RNG_HANSEN) {
        const size_t rows = (size_t)o->d.pop_count;
        o->z_host.assign(rows * o->d.ns, 0.f);
        // the reference draws row by row, N deviates per offspring (lmcma.cpp:303-305, 212-215)
        for (size_t r = 0; r < rows; ++r)
            for (int k = 0; k < o->d.n; ++k) o->z_host[r * o->d.ns + k] = (float)o->hansen.gauss();
        CU(cudaMemcpyAsync(o->d.Z, o->z_host.data(), o->z_host.size() * sizeof(float), cudaMemcpyHostToDevice, st));
        CU(cudaStreamSynchronize(st));   // z_host is pageable and reused
    }
    return launch_sample(o, st, o->cfg.rng != LMCMA_B200_RNG_HANSEN, progressive);
}

// update() + sample() after the fitness of a generation is in d.fit
int generation_tail(lmcma_b200_opt* o, cudaStream_t st) {
    int rc;
    if ((rc = launch_rank(o, o->d.fit, RANK_PLAIN, nullptr, st))) return rc;
    // device RNG: k_sample follows k_update directly and can take its outputs as they become final
    const bool prog = o->plan.progressive && o->cfg.rng == LMCMA_B200_RNG_PHILOX && !o->mirror_dirty;
    UpdateArgs ua = update_args_local(o);
    ua.progressive = prog ? 1 : 0;
    if ((rc = launch_update(o, ua, true, st))) return rc;
    o->x_cache_valid = false;
    o->sample_idx = 0;
    if (o->cfg.rng == LMCMA_B200_RNG_INJECT && !o->pending_z) { o->needs_sample = true; return 0; }
    o->pending_z = false;
    return host_rng_and_sample(o, st, prog);
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
void drop_tell_graphs(lmcma_b200_opt* o) {
    drop(o->tell_graph);
    drop(o->tell_graph_resume);
    o->spec_valid = false;
}

// Records what body() enqueues on `st` (and on the streams it forks from `st`) into *g, which is empty.  Capture enqueues
// nothing: the kernels the body launches are counted in g->launches, and each replay adds them to g_launches.
template <class Body>
int capture(cudaStream_t st, Body&& body, Graph* g) {
    cudaGraph_t graph = nullptr;
    long long launches = 0;
    CU(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
    g_capture_launches = &launches;
    int rc = body();
    g_capture_launches = nullptr;
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
        bool ok2 = cudaEventRecord(o->ev_fork, st) == cudaSuccess && cudaStreamWaitEvent(o->side_stream, o->ev_fork, 0) == cudaSuccess;
        if (ok2) ok2 = launch(k_probe, 1, 1, 0, o->side_stream, false, d, d + 2, 0, 5000000ll) == 0 && cudaEventRecord(o->ev_join, o->side_stream) == cudaSuccess;
        if (ok2) ok2 = launch(k_probe, 1, 1, 0, st, false, d, d + 2, 1, 5000000ll) == 0 && cudaStreamWaitEvent(st, o->ev_join, 0) == cudaSuccess;
        return ok2 ? 0 : LMCMA_B200_ERR_CUDA;
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
    o->tell_graph_failed = true;
    o->mirror_dirty = true;
    return fail(LMCMA_B200_ERR_CUDA, "overlapped generation lost co-scheduling (%s): the branches of the CUDA graph did not run "
                "concurrently (profiler / sanitizer / SMs held elsewhere).  This handle now uses the linear graph; the generation in "
                "flight is void - restore the state or recreate the handle (LMCMA_B200_OVERLAP=0 avoids the overlapped graph)",
                code == LOST_UPDATE_WAITING_FOR_RANK ? "k_update timed out waiting for k_rank" : "k_sample timed out waiting for k_update");
}
namespace {

int ensure_graph(lmcma_b200_opt* o) {
    if (o->graph.exec && o->graph_built_for == o->stream) return 0;
    drop_fused_graphs(o);
    CostArgs ca;
    int rc = cost_args_for(o, &ca);
    if (rc) return rc;
    cudaStream_t st = o->stream;
    if ((rc = ensure_mirror(o, st))) return rc;
    // `reps` generations in ONE graph: between two graph launches the device idles for the launch latency of the next one
    // (~5 us of a 52 us generation); inside a graph a generation follows the previous one as a plain dependency
    auto body = [&](int reps) -> int {
        UpdateArgs ua = update_args_local(o);
        ua.progressive = o->plan.progressive ? 1 : 0;            // ensure_mirror above: the mirror is clean
        int rc2 = 0;
        for (int g = 0; g < reps && !rc2; ++g) {
            if (o->overlap) {
                // side branch: k_update starts with the generation; main branch: k_gate (waits until k_update holds its SM) ->
                // k_cost -> k_rank -> k_sample (released by k_rank, follows k_update's flags); join before the generation ends
                ua.overlap = 1;
                if (cudaEventRecord(o->ev_fork, st) != cudaSuccess || cudaStreamWaitEvent(o->side_stream, o->ev_fork, 0) != cudaSuccess) rc2 = fail(LMCMA_B200_ERR_CUDA, "graph fork failed");
                if (!rc2) rc2 = launch_update(o, ua, false, o->side_stream);
                if (!rc2 && cudaEventRecord(o->ev_join, o->side_stream) != cudaSuccess) rc2 = fail(LMCMA_B200_ERR_CUDA, "graph join record failed");
                if (!rc2) rc2 = launch(k_gate, (o->d.B + 31) / 32, 32, 0, st, false, o->d);
                if (!rc2) rc2 = launch_cost(o->map->dev, ca, o->d.pop_count, o->d.B, o->cost_shape, false, st);
                if (!rc2) rc2 = launch_rank(o, o->d.fit, RANK_PLAIN | RANK_KEEP_FLAGS, nullptr, st, true);
                if (!rc2) rc2 = launch_sample(o, st, true, true, 2);
                if (!rc2 && cudaStreamWaitEvent(st, o->ev_join, 0) != cudaSuccess) rc2 = fail(LMCMA_B200_ERR_CUDA, "graph join failed");
            } else {
                rc2 = launch_cost(o->map->dev, ca, o->d.pop_count, o->d.B, o->cost_shape, false, st);
                if (!rc2) rc2 = launch_rank(o, o->d.fit, RANK_PLAIN, nullptr, st, true);
                if (!rc2) rc2 = launch_update(o, ua, true, st);
                if (!rc2) rc2 = launch_sample(o, st, true, o->plan.progressive);
            }
        }
        return rc2;
    };
    o->mirror_suppressed = true;                                 // fused generations keep the candidates on the device
    rc = capture(st, [&] { return body(1); }, &o->graph);
    if (!rc && o->tune.graph_unroll > 1 && capture(st, [&] { return body(o->tune.graph_unroll); }, &o->graph_multi) != 0)
        cudaGetLastError();                                      // optional: the single one still works
    o->mirror_suppressed = false;
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

// tell_all of one query as a forked graph (see lmcma_b200_tell_all); on failure the caller takes the stream-ordered path
int ensure_tell_graph(lmcma_b200_opt* o) {
    if (o->tell_graph.exec && o->tell_graph_for == o->stream) return ensure_mirror(o, o->stream);
    drop_tell_graphs(o);
    cudaStream_t st = o->stream;
    const OptDev& d = o->d;
    int rc = ensure_mirror(o, st);
    if (rc) return rc;
    if (!o->f_pinned && cudaHostAlloc(&o->f_pinned, (size_t)d.B * d.lambda * sizeof(float), cudaHostAllocDefault) != cudaSuccess) {
        cudaGetLastError(); o->f_pinned = nullptr; o->tell_graph_failed = true; return 0;
    }
    // the speculative pass pays only where something hides it: with the host mirror on, the candidates' trip across PCIe
    // (35 us behind the sampler).  Without the mirror tell_all returns when the sampler is done, and a 25 us kernel behind
    // k_update would be the longer branch of the graph (measured: tell_all 57 -> 69 us)
    const bool spec = o->d_spec != nullptr && o->mirror_on && !o->mirror_suppressed;
    o->tell_graph_spec = spec;
    // resume = 0: the whole update; resume = 1: k_update picks up the rows the last graph's speculative pass left.  With the
    // scratch both graphs END with that pass for the next generation, on the side branch behind k_update
    auto body = [&](int resume) -> int {
        UpdateArgs ua = update_args_local(o);
        ua.progressive = 1;
        ua.overlap = 1;
        ua.phase = resume ? 2 : 0;
        const bool valid_before = o->spec_valid;
        bool ok = cudaEventRecord(o->ev_fork, st) == cudaSuccess && cudaStreamWaitEvent(o->side_stream, o->ev_fork, 0) == cudaSuccess;
        if (ok) ok = launch_update(o, ua, false, o->side_stream) == 0;
        if (ok && spec) { UpdateArgs us = ua; us.phase = 1; us.dbg = nullptr; ok = launch_update(o, us, false, o->side_stream) == 0; }
        o->spec_valid = valid_before;                            // capture enqueues nothing
        if (ok) ok = cudaEventRecord(o->ev_join, o->side_stream) == cudaSuccess;
        if (ok) ok = cudaMemcpyAsync(d.fit, o->f_pinned, (size_t)d.B * d.lambda * sizeof(float), cudaMemcpyHostToDevice, st) == cudaSuccess;
        if (ok) ok = launch(k_gate, (d.B + 31) / 32, 32, 0, st, false, d) == 0;   // k_update has reset the flags and holds its SM
        // the sampler is released when k_rank starts: the pairs it needs first are final (resume: at once; else as the sweep goes)
        if (ok) ok = launch_rank(o, d.fit, RANK_PLAIN | RANK_KEEP_FLAGS, nullptr, st, false) == 0;
        if (ok) ok = launch_sample(o, st, true, true, 2) == 0;
        if (ok) ok = cudaStreamWaitEvent(st, o->ev_join, 0) == cudaSuccess;
        return ok ? 0 : LMCMA_B200_ERR_CUDA;
    };
    rc = capture(st, [&] { return body(0); }, &o->tell_graph);
    if (!rc && spec) rc = capture(st, [&] { return body(1); }, &o->tell_graph_resume);
    if (rc) {
        cudaGetLastError();
        drop_tell_graphs(o);
        o->tell_graph_failed = true;
        return 0;
    }
    o->tell_graph_for = st;
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
    DM(d.X, B * pc * ns);
    DM(d.D, B * pc * ns);
    if (cfg->rng != LMCMA_B200_RNG_PHILOX || cfg->record_z || covariance) DM(d.Z, B * pc * ns);
    if (covariance) {   // CMABase::init factors the prior once (cholesky, lmcma.cpp:165-169)
        std::vector<double> Ld((size_t)d.n * d.n);
        if (!cholesky_lower(covariance, d.n, Ld.data())) { return fail(LMCMA_B200_ERR_ARG, "covariance prior is not symmetric positive definite"); }
        std::vector<float> Lf((size_t)d.n * ns, 0.f);
        for (int i = 0; i < d.n; ++i)
            for (int k = 0; k <= i; ++k) Lf[(size_t)i * ns + k] = (float)Ld[(size_t)i * d.n + k];
        DM(o->d_Lf, (size_t)d.n * ns);
        CU(cudaMemcpy(o->d_Lf, Lf.data(), Lf.size() * sizeof(float), cudaMemcpyHostToDevice));
        d.Lf = o->d_Lf;
        DM(d.Zc, B * pc * ns);
    }
    DM(d.fit, B * lam); DM(d.fit_sorted, B * lam); DM(d.prev_fit, B * lam);
    DM(d.rank, B * lam); DM(d.arindex, B * lam);
    if (o->plan.rank.tile_sorted) {
        DM(d.prev_sorted, B * lam); DM(d.tile_sorted, B * lam); DM(d.tile_pos, B * lam);
    }
    DM(d.ncoll, B * pc); DM(d.nsamp, B * pc);
    DM(d.xmean, B * ns); DM(d.pc, B * ns);
    DM(d.V, B * m * ns); DM(d.P, B * m * ns);
    DM(d.Nj, B * m); DM(d.Lj, B * m); DM(d.Njf, B * m); DM(d.Njs, B * m);
    DM(d.VPs, B * m * 2 * ns);
    DM(d.t, B * m); DM(d.vec, B * m);
    DM(d.sc, B); DM(d.best_x, B * ns); DM(d.S_count, B); DM(d.done_count, B); DM(d.progress, B * progress_len(m)); DM(d.rank_ticket, B); DM(d.resident, B);
    if (o->tune.dbg) DM(d.dbg, TL_SLOTS);
    DM(d.partial, B * d.RS * ns);

    std::vector<float> wf(o->weights.begin(), o->weights.end());
    DM(o->d_w, d.mu);
    CU(cudaMemcpy(o->d_w, wf.data(), d.mu * sizeof(float), cudaMemcpyHostToDevice));
    d.w = o->d_w;
    if (lo) {   // padded to the row stride so that the kernels clamp whole float4 columns
        o->lo_f.assign(d.ns, -std::numeric_limits<float>::max());
        for (int k = 0; k < d.n; ++k) o->lo_f[k] = (float)lo[k];
        DM(o->d_lo, d.ns);
        CU(cudaMemcpy(o->d_lo, o->lo_f.data(), d.ns * sizeof(float), cudaMemcpyHostToDevice));
        d.lo = o->d_lo;
    }
    if (hi) {
        o->hi_f.assign(d.ns, std::numeric_limits<float>::max());
        for (int k = 0; k < d.n; ++k) o->hi_f[k] = (float)hi[k];
        DM(o->d_hi, d.ns);
        CU(cudaMemcpy(o->d_hi, o->hi_f.data(), d.ns * sizeof(float), cudaMemcpyHostToDevice));
        d.hi = o->d_hi;
    }
    // initial mean (lmcma.cpp:158-163)
    std::vector<double> xm(B * ns, 0.0);
    for (size_t b = 0; b < B; ++b)
        for (int k = 0; k < d.n; ++k) xm[b * ns + k] = x0 ? x0[b * d.n + k] : o->hansen.uniform();
    CU(cudaMemcpy(d.xmean, xm.data(), xm.size() * sizeof(double), cudaMemcpyHostToDevice));
    std::vector<Scalars> sc(B);
    for (auto& s : sc) {
        memset(&s, 0, sizeof(s));
        s.sigma = cfg->sigma0; s.s = 0.0; s.best_f = std::numeric_limits<double>::max();
    }
    CU(cudaMemcpy(d.sc, sc.data(), B * sizeof(Scalars), cudaMemcpyHostToDevice));

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
            if (cudaMalloc(&o->d_spec, B * o->spec_stride * sizeof(float)) != cudaSuccess) { cudaGetLastError(); o->d_spec = nullptr; }
            else cudaMemset(o->d_spec, 0xff, B * o->spec_stride * sizeof(float));   // generation -1: matches nothing
        }
    }
    if (o->plan.update.gram) {
        DM(d.G, B * GRAM_KS * m * m);
        DM(d.Cf, B * m * m);
        DM(d.gram_hdr, B);
    }
    o->f_host.assign(B * lam, 0.f);
    // first population (LMCMA::init -> sample(), lmcma.cpp:298)
    if (cfg->rng == LMCMA_B200_RNG_INJECT) o->needs_sample = true;
    else {
        rc = host_rng_and_sample(o, o->stream);
        if (!rc) { cudaError_t e = cudaStreamSynchronize(o->stream); if (e != cudaSuccess) rc = fail(LMCMA_B200_ERR_CUDA, "first sample: %s", cudaGetErrorString(e)); }
        if (rc) return rc;
    }
    return 0;
}

int lmcma_b200_destroy(lmcma_b200_opt* o) {
    if (!o) return 0;
    cudaSetDevice(o->cfg.device);
    if (o->stream) cudaStreamSynchronize(o->stream);
    OptDev& d = o->d;
    void* ptrs[] = {d.prev_sorted, d.tile_sorted, d.tile_pos, d.X, d.D, d.Z, d.Zc, o->d_Lf, d.fit, d.fit_sorted, d.prev_fit, d.rank, d.arindex, d.ncoll, d.nsamp, d.xmean, d.pc, d.V, d.P,
                    d.Nj, d.Lj, d.Njf, d.Njs, d.VPs, d.dbg, d.G, d.Cf, d.gram_hdr, d.t, d.vec, d.sc, d.best_x, d.S_count, d.done_count, d.progress, d.rank_ticket, d.resident, d.partial, o->d_lo, o->d_hi, o->d_w, o->d_ends};
    for (void* p : ptrs) cudaFree(p);
    drop_fused_graphs(o);
    drop_tell_graphs(o);
    cudaFree(o->d_spec);
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
        rc = launch_sample(o, o->stream);
        if (rc) return rc;
        CU(cudaStreamSynchronize(o->stream));
    } else {
        o->pending_z = true;
    }
    return 0;
}

int lmcma_b200_resample(lmcma_b200_opt* o) {
    ARG(o, "null handle");
    if (o->needs_sample) return fail(LMCMA_B200_ERR_STATE, "no deviates yet: inject_z first");
    if (o->cfg.rng == LMCMA_B200_RNG_HANSEN) return fail(LMCMA_B200_ERR_STATE, "resample would advance the serial HANSEN stream");
    CU(cudaSetDevice(o->cfg.device));
    int rc = launch_sample(o, o->stream);
    if (rc) return rc;
    CU(cudaStreamSynchronize(o->stream));
    o->x_cache_valid = false;
    return 0;
}

int lmcma_b200_ask_all(lmcma_b200_opt* o, float* X) {
    ARG(o && X, "null pointer");
    if (o->needs_sample) return fail(LMCMA_B200_ERR_STATE, "no population yet: inject_z first");
    CU(cudaSetDevice(o->cfg.device));
    const OptDev& d = o->d;
    int rc = d2h_rows(X, d.X, (size_t)d.B * d.pop_count, d.n * sizeof(float), d.ns * sizeof(float), o->stream);
    return rc ? rc : check_lost(o);
}

int lmcma_b200_ask_all_view(lmcma_b200_opt* o, const float** X_view, int64_t* ld_out) {
    ARG(o && X_view, "null pointer");
    if (o->needs_sample) return fail(LMCMA_B200_ERR_STATE, "no population yet: inject_z first");
    CU(cudaSetDevice(o->cfg.device));
    OptDev& d = o->d;
    const size_t floats = (size_t)d.B * d.pop_count * d.ns;
    if (!o->x_mirror) {
        CU(cudaStreamSynchronize(o->stream));
        CU(cudaHostAlloc(&o->x_mirror, floats * sizeof(float), cudaHostAllocMapped));
        cudaError_t e = cudaHostGetDevicePointer(&d.Xh, o->x_mirror, 0);
        if (e != cudaSuccess) { cudaFreeHost(o->x_mirror); o->x_mirror = nullptr; d.Xh = nullptr; return fail(LMCMA_B200_ERR_CUDA, "cudaHostGetDevicePointer: %s", cudaGetErrorString(e)); }
        o->mirror_on = true;
        o->xh_fresh = false;
        register_mirror(o->x_mirror, floats * sizeof(float), d.X, d.ns, o->cfg.device);
        // the captured graphs carry the old kernel parameters (OptDev by value): rebuild them on next use
        drop_tell_graphs(o);
    }
    if (!o->xh_fresh) {                                  // first use / after a fused run or a state setter: one ordinary copy
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
    if (o->needs_sample) return fail(LMCMA_B200_ERR_STATE, "no population yet: inject_z first");
    if (o->d.pop_count != o->d.lambda) return fail(LMCMA_B200_ERR_STATE, "split-population handles use the mg_* entry points");
    CU(cudaSetDevice(o->cfg.device));
    const OptDev& d = o->d;
    int rc;
    if (o->overlap && !o->tell_graph_failed && o->tune.tell_overlap != 0) {
        // One query (the conditions of the overlapped generation, DESIGN.md 4.3): everything in update() that does not
        // depend on this generation's fitness — slot bookkeeping, the sweep over every pending row but the newest — runs on
        // a side branch while the fitness crosses PCIe and k_rank runs; k_update then waits for k_rank's tickets and
        // k_sample follows its hand-over flags.  Same kernels and arithmetic as the fused generation (bit-identical to the
        // serial order), replayed as one CUDA graph: launched kernel by kernel, the fork / join costs more host time than
        // the overlap saves.
        if ((rc = ensure_tell_graph(o)) == 0 && o->tell_graph.exec) {
            memcpy(o->f_pinned, f, (size_t)d.B * d.lambda * sizeof(float));
            const bool resume = o->spec_valid && o->tell_graph_resume.exec;   // the last tell_all graph left the next update's rows behind
            if ((rc = replay(resume ? o->tell_graph_resume : o->tell_graph, o->stream))) return rc;
            o->spec_valid = o->tell_graph_spec;                   // ... and so does this one
            o->xh_fresh = o->mirror_on;                          // the captured sampler writes the host mirror when it is on
            o->x_cache_valid = false;
            o->sample_idx = 0;
            o->pending_z = false;
            CU(cudaStreamSynchronize(o->stream));
            return check_lost(o);
        }
        if (rc) return rc;
    }
    CU(cudaMemcpyAsync(d.fit, f, (size_t)d.B * d.lambda * sizeof(float), cudaMemcpyHostToDevice, o->stream));
    rc = generation_tail(o, o->stream);
    if (rc) return rc;
    CU(cudaStreamSynchronize(o->stream));
    return 0;
}

int lmcma_b200_ask_one(lmcma_b200_opt* o, double* params, int32_t n) {
    ARG(o && params, "null pointer");
    ARG(n == o->d.n, "N mismatch");
    if (o->d.B != 1 || o->d.pop_count != o->d.lambda) return fail(LMCMA_B200_ERR_STATE, "ask_one needs batch == 1 and an unsplit population");
    if (!o->x_cache_valid) {
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
    if (o->d.B != 1 || o->d.pop_count != o->d.lambda) return fail(LMCMA_B200_ERR_STATE, "tell_one needs batch == 1 and an unsplit population");
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
    std::vector<Scalars> sc(o->d.B);
    CU(cudaMemcpyAsync(sc.data(), o->d.sc, sc.size() * sizeof(Scalars), cudaMemcpyDeviceToHost, o->stream));
    CU(cudaStreamSynchronize(o->stream));
    for (int b = 0; b < o->d.B; ++b) done[b] = sc[b].sigma < 1e-20 ? 1 : 0;   // lmcma.cpp:426-429
    return 0;
}

int lmcma_b200_attach_cost(lmcma_b200_opt* o, lmcma_b200_map* map, const lmcma_b200_objective* obj,
                           const lmcma_b200_endpoints* ends) {
    ARG(o && ends, "null pointer");
    int rc = check_obj(map, obj);
    if (rc) return rc;
    ARG(map->device == o->cfg.device, "map and optimiser live on different devices");
    ARG(map->dev.dims * obj->waypoints == o->d.n, "n != dims * waypoints");
    CU(cudaSetDevice(o->cfg.device));
    o->map = map; o->obj = *obj;
    std::vector<float> e6((size_t)o->d.B * 6);
    for (int b = 0; b < o->d.B; ++b)
        for (int c = 0; c < 3; ++c) { e6[b * 6 + c] = ends[b].start[c]; e6[b * 6 + 3 + c] = ends[b].goal[c]; }
    if (!o->d_ends) DM(o->d_ends, (size_t)o->d.B * 6);
    CU(cudaMemcpy(o->d_ends, e6.data(), e6.size() * sizeof(float), cudaMemcpyHostToDevice));
    o->cost_shape = pick_cost_shape(obj->waypoints, ends[0].start, ends[0].goal, map->dev.dims, o->tune);
    drop_fused_graphs(o);
    return 0;
}

int lmcma_b200_run(lmcma_b200_opt* o, int32_t generations) {
    ARG(o && generations >= 0, "bad argument");
    if (!o->map) return fail(LMCMA_B200_ERR_STATE, "no cost attached");
    if (o->needs_sample) return fail(LMCMA_B200_ERR_STATE, "no population yet: inject_z first");
    if (o->d.pop_count != o->d.lambda) return fail(LMCMA_B200_ERR_STATE, "split-population handles use the mg_* entry points");
    CU(cudaSetDevice(o->cfg.device));
    int rc = apply_l2_window(o->map, o->stream);
    if (rc) return rc;
    o->spec_valid = false;                                       // the fused generations advance the state past what tell_all's speculative pass saw
    if (o->cfg.rng == LMCMA_B200_RNG_PHILOX) {
        if ((rc = ensure_graph(o))) return rc;
        if ((rc = ensure_mirror(o, o->stream))) return rc;       // a state setter since the last run: the graph's sampler reads the mirror
        CU(cudaEventRecord(o->ev0, o->stream));                  // after the (host-side) graph build: last_run_ms is device time
        const int unroll = o->graph_multi.exec ? o->tune.graph_unroll : 0;
        for (int g = 0; g < generations;) {
            const bool multi = unroll > 1 && generations - g >= unroll;
            if ((rc = replay(multi ? o->graph_multi : o->graph, o->stream))) return rc;
            g += multi ? unroll : 1;
        }
    } else {
        if (o->cfg.rng == LMCMA_B200_RNG_INJECT && generations > 1)
            return fail(LMCMA_B200_ERR_STATE, "INJECT rng: run one generation per injected Z");
        CostArgs ca;
        if ((rc = cost_args_for(o, &ca))) return rc;
        CU(cudaEventRecord(o->ev0, o->stream));
        for (int g = 0; g < generations; ++g) {
            if ((rc = launch_cost(o->map->dev, ca, o->d.pop_count, o->d.B, o->cost_shape, false, o->stream))) return rc;
            if ((rc = generation_tail(o, o->stream))) return rc;
        }
    }
    CU(cudaEventRecord(o->ev1, o->stream));
    o->have_run_timing = true;
    o->x_cache_valid = false;
    if (o->cfg.rng == LMCMA_B200_RNG_PHILOX) o->xh_fresh = false;    // the graph's sampler does not write the host mirror
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
    if (!o->map) return fail(LMCMA_B200_ERR_STATE, "no cost attached");
    if (o->cfg.rng != LMCMA_B200_RNG_PHILOX) return fail(LMCMA_B200_ERR_STATE, "profile_kernels needs the PHILOX rng");
    CU(cudaSetDevice(o->cfg.device));
    CostArgs ca;
    int rc = cost_args_for(o, &ca);
    if (rc) return rc;
    cudaStream_t st = o->stream;
    std::vector<cudaEvent_t> ev((size_t)generations * 5);
    for (auto& e : ev) CU(cudaEventCreate(&e));
    for (int g = 0; g < generations && !rc; ++g) {
        cudaEvent_t* e = &ev[(size_t)g * 5];
        cudaEventRecord(e[0], st);
        rc = launch_cost(o->map->dev, ca, o->d.pop_count, o->d.B, o->cost_shape, false, st);
        cudaEventRecord(e[1], st);
        if (!rc) rc = launch_rank(o, o->d.fit, RANK_PLAIN, nullptr, st);
        cudaEventRecord(e[2], st);
        if (!rc) rc = launch_update(o, update_args_local(o), false, st);   // serialised here so that the events separate the kernels
        cudaEventRecord(e[3], st);
        if (!rc) rc = launch_sample(o, st);
        cudaEventRecord(e[4], st);
    }
    cudaError_t se = cudaStreamSynchronize(st);
    if (!rc && se != cudaSuccess) rc = fail(LMCMA_B200_ERR_CUDA, "profile run: %s", cudaGetErrorString(se));
    if (!rc && o->d.dbg) rc = print_timeline(o);
    if (!rc && o->d.dbg) {     // and the per-CTA timeline of k_cost (phase stamps): one extra launch of its TRACE build
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
    o->x_cache_valid = false;
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
    if (f_best) {
        std::vector<Scalars> sc(d.B);
        CU(cudaMemcpyAsync(sc.data(), d.sc, sc.size() * sizeof(Scalars), cudaMemcpyDeviceToHost, o->stream));
        CU(cudaStreamSynchronize(o->stream));
        for (int b = 0; b < d.B; ++b) f_best[b] = (float)sc[b].best_f;
    }
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
    if (o->d.B != 1) return fail(LMCMA_B200_ERR_STATE, "split-population mode needs batch == 1");
    if (o->needs_sample) return fail(LMCMA_B200_ERR_STATE, "no population yet");
    CU(cudaSetDevice(o->cfg.device));
    CostArgs ca;
    int rc = cost_args_for(o, &ca);
    if (rc) return rc;
    ca.f = f_local_dev; ca.f_stride = o->d.pop_count; ca.f_offset = 0;
    cudaStream_t st = stream ? (cudaStream_t)stream : o->stream;
    if ((rc = apply_l2_window(o->map, st))) return rc;
    return launch_cost(o->map->dev, ca, o->d.pop_count, o->d.B, o->cost_shape, false, st);
}

int lmcma_b200_mg_rank(lmcma_b200_opt* o, const float* f_all_dev, float* payload_dev, void* stream) {
    ARG(o && f_all_dev && payload_dev, "null pointer");
    if (o->d.B != 1) return fail(LMCMA_B200_ERR_STATE, "split-population mode needs batch == 1");
    CU(cudaSetDevice(o->cfg.device));
    cudaStream_t st = stream ? (cudaStream_t)stream : o->stream;
    // keep the gathered fitness: k_update needs it for prev_fit / best tracking
    CU(cudaMemcpyAsync(o->d.fit, f_all_dev, (size_t)o->d.lambda * sizeof(float), cudaMemcpyDeviceToDevice, st));
    return launch_rank(o, o->d.fit, RANK_PACK, payload_dev, st);
}

int lmcma_b200_mg_update(lmcma_b200_opt* o, const float* payload_all_dev, int32_t world, void* stream) {
    ARG(o && payload_all_dev && world >= 1, "bad argument");
    if (o->cfg.rng != LMCMA_B200_RNG_PHILOX) return fail(LMCMA_B200_ERR_STATE, "split-population mode needs the PHILOX rng");   // before anything is launched
    CU(cudaSetDevice(o->cfg.device));
    cudaStream_t st = stream ? (cudaStream_t)stream : o->stream;
    const long long pf = o->d.ns + 4;
    UpdateArgs a;
    memset(&a, 0, sizeof(a));
    a.f_all = o->d.fit; a.slices = payload_all_dev; a.n_slices = world;
    a.slice_stride = (long long)o->d.B * pf; a.inst_stride = pf; a.payload_mode = 1;
    int rc = launch_update(o, a, false, st);
    if (rc) return rc;
    o->x_cache_valid = false;
    o->mirror_suppressed = true;
    rc = launch_sample(o, st, true);
    o->mirror_suppressed = false;
    return rc;
}

}  // extern "C"

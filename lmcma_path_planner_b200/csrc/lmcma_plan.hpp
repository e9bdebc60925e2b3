// lmcma_plan.hpp — the launch plan of an optimiser handle: which sampler, update, k_rank and k_coef build it runs and with
// what block size, grid and shared memory, chosen once at create from the shape, the rng, the prior, the LMCMA_B200_*
// knobs and two device limits.  Plain integer arithmetic in plain C++ (no CUDA header), so the choice can be checked
// without a GPU.  Also the constants both the plan and the kernels use, defined here once.
#pragma once
#include <cstddef>
#include <cstdint>
#include <cstdlib>
#include <string>

namespace lmcma {

constexpr int SAMPLE_G = 8;   // direction pairs per group: their dots are independent, reduced together
constexpr int SAMPLE_MAX_STAGES = 8;

constexpr int TELL_FTILE = 4096;       // fitness values staged per shared-memory tile
constexpr int TELL_MAX_ROWS = 256;     // rows per slice upper bound (rows_per = max(32, ceil(pop/256)))

constexpr int UPD_WARPS = 16;
constexpr int UPD_GROUPS = UPD_WARPS / 4;   // 128-thread groups of the mean phase
constexpr int UPD_BLK = 8;            // factors per block of the newest row's chain (k_update: newest_row)

// the narrow sampler k_sample<NV, RB, MAXT, SPEC> of NV float4 columns per lane: rows per warp, CTA size bound, and
// whether full groups of 8 pairs run without per-pair predicates
constexpr int narrow_rb(int nv) { return nv <= 2 ? 4 : (nv <= 4 ? 2 : 1); }
constexpr int narrow_maxt(int nv) { return nv >= 12 ? 256 : 512; }
constexpr bool narrow_spec(int nv) { return nv == 4; }
// the wide sampler k_sample_wide<RBW, MAXT> of RBW rows per warp: CTA size bound
constexpr int wide_maxt(int rbw) { return rbw == 2 ? 1024 : 512; }

}  // namespace lmcma

namespace lmcma_capi {

inline int env_int(const char* name, int dflt) {
    const char* v = getenv(name);
    return v && *v ? atoi(v) : dflt;
}

// Every LMCMA_B200_* environment knob, read ONCE when a handle (map or optimiser) is created and kept on the handle:
// nothing on a launch path calls getenv.  The defaults are the product; each switch is a serial-order reference of the
// bit-identity tests, a test seam, an operational override or a diagnostic (INTEGRATION.md section 5 lists them all).
struct Tuning {
    int cost_minb = 0 /* 0 = by launch size */, cost_tpt = 0, cost_cb = 0, zerocopy = 1;
    int sample_rows = 0;    // 1: k_sample_rows also for one large population (else only where it pays: many rows)
    int update_gram = 0, progressive = 1, overlap = 1, tell_overlap = 1;
    int tell_spec = 1;      // tell_all: speculative update of the next generation at the end of the graph (LMCMA_B200_TELL_SPEC=0: off)
    int graph_unroll = 8;   // fused generations per CUDA graph for runs of at least that many (LMCMA_B200_GRAPH_UNROLL, 1 = off)
    int update_warps = 0;   // k_update CTA size: 0 = by batch size, 8 / 16 forced (LMCMA_B200_UPDATE_WARPS)
    int dbg = 0;            // device timelines, printed by lmcma_b200_sync and profile_kernels (LMCMA_B200_DBG set)
    static Tuning from_env() {
        Tuning t;
        t.cost_minb = env_int("LMCMA_B200_COST_MINB", t.cost_minb);
        t.cost_tpt = env_int("LMCMA_B200_COST_TPT", 0);
        t.cost_cb = env_int("LMCMA_B200_COST_CB", 0);
        t.zerocopy = env_int("LMCMA_B200_ZEROCOPY", 1);
        t.sample_rows = env_int("LMCMA_B200_SAMPLE_ROWS", 0);
        t.update_gram = env_int("LMCMA_B200_UPDATE_GRAM", 0);
        t.progressive = env_int("LMCMA_B200_PROGRESSIVE", 1);
        t.overlap = env_int("LMCMA_B200_OVERLAP", 1);
        t.tell_overlap = env_int("LMCMA_B200_TELL_OVERLAP", 1);
        t.tell_spec = env_int("LMCMA_B200_TELL_SPEC", 1);
        t.update_warps = env_int("LMCMA_B200_UPDATE_WARPS", 0);
        t.graph_unroll = env_int("LMCMA_B200_GRAPH_UNROLL", 8);
        if (t.graph_unroll < 1 || t.graph_unroll > 64) t.graph_unroll = 1;
        t.dbg = getenv("LMCMA_B200_DBG") ? 1 : 0;
        return t;
    }
};

// the shape of a handle, with lambda and m already defaulted (lmcma.cpp:134-136, 266)
struct PlanInput {
    int n = 0, lambda = 0, m = 0, batch = 1, pop_count = 0;
    int rng = 0;              // LMCMA_B200_RNG_*
    bool has_prior = false;   // a covariance prior (lmcma_b200_create_with_prior)
};

struct DeviceLimits {
    int sm_count = 0;
    size_t smem_optin = 0;    // dynamic shared memory one block may opt into
};

enum class Sampler : int { NARROW = 0, WIDE = 1, ROWS = 2 };   // the values of LMCMA_B200_LAUNCH_SAMPLER

// Every launch configuration of a handle.  The launchers and LMCMA_B200_I32_LAUNCH read it; nothing re-derives it.
// A family's own fields are 0 when the handle runs another family.
struct LaunchPlan {
    struct {
        Sampler kind = Sampler::NARROW;
        int threads = 0, ctas = 0;        // block size; CTAs per instance (grid = ctas x batch)
        size_t smem = 0;
        int kc = 0, stages = 0;           // pairs per stage, stages in flight
        int nv = 0;                       // float4 columns per lane of the narrow sampler (set for every family)
        int R = 0, CW = 0, qpw = 0, RBW = 0;   // wide: row groups per CTA, column-warps per row, float4 columns per warp, rows per warp
        int qw = 0, rl = 0, region = 0;   // rows: float4 columns per warp, rows per lane, floats of the staging region
    } sample;
    struct {
        int threads = 0, ftile = 0, slices = 0;   // grid = slices x batch
        size_t smem = 0;
        bool tile_sorted = false;                 // k_rank_tiles sorts the fitness tiles first (lambda > TELL_FTILE, unsplit)
    } rank;
    struct {
        int nvb = 0, rmax = 0, warps = 0;         // k_update<nvb, rmax, rows_in_smem, OVERLAP, WARPS>; rmax 0: no register sweep
        bool rows_in_smem = false, gram = false;  // gram: Gram-matrix recompute (k_gram.cuh) instead of the sweep
        size_t smem = 0;
    } update;
    struct {
        int elems = 0, threads = 0;               // k_coef<elems> (gram only)
        size_t smem = 0;
    } coef;
    bool progressive = false;   // k_update -> k_sample hand-over inside the fused generation (k_update.cuh)
    bool overlap = false;       // eligible for the overlapped generation; the handle may still turn it off at run time
};

// Chooses the plan of a handle; false with the reason in *err for a shape no build can run.
bool plan_launch(const PlanInput& in, const DeviceLimits& dev, const Tuning& tune, LaunchPlan* plan, std::string* err);

// The LMCMA_B200_LAUNCH_FIELDS values of LMCMA_B200_I32_LAUNCH for a plan (OVERLAP: the plan's eligibility).
void launch_fields(const LaunchPlan& plan, int32_t* v);

}  // namespace lmcma_capi

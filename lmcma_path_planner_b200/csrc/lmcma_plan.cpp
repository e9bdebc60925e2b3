// lmcma_plan.cpp — plan_launch: the launch configuration of an optimiser handle (lmcma_plan.hpp).  Part of
// liblmcma_b200.so; plain C++.
#include "lmcma_plan.hpp"
#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include "../../include/lmcma_b200.h"

namespace lmcma_capi {
using namespace lmcma;

namespace {
bool refuse(std::string* err, const char* fmt, ...) {
    char buf[256];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    *err = buf;
    return false;
}
}  // namespace

bool plan_launch(const PlanInput& in, const DeviceLimits& dev, const Tuning& tune, LaunchPlan* plan, std::string* err) {
    LaunchPlan p;
    const int ns = (in.n + 3) & ~3, nq = ns / 4, m = in.m, B = in.batch, pop = in.pop_count;

    // ---- k_rank.  Row slices of k_tell's phase A: 32 rows per slice, at most 256 slices
    auto& r = p.rank;
    const int rows_per = std::max(32, (pop + 255) / 256);
    if (rows_per > TELL_MAX_ROWS) return refuse(err, "population too large (max %d rows per handle)", 256 * TELL_MAX_ROWS);
    r.slices = (pop + rows_per - 1) / rows_per;
    r.tile_sorted = in.lambda > TELL_FTILE && pop == in.lambda;
    // small populations (lambda <= 256) take CTAs of 256 threads and tiles of lambda values — the choice depends on
    // lambda alone, so that a batched instance and the same instance run alone sum their partial sums in the same order
    r.threads = in.lambda <= 256 ? 256 : 1024;
    r.ftile = in.lambda <= 256 ? ((in.lambda + 3) & ~3) : TELL_FTILE;
    r.smem = (size_t)2 * r.ftile * 4 + (size_t)3 * TELL_MAX_ROWS * 4 + (size_t)7 * 128 * 16;

    // ---- sampler
    auto& s = p.sample;
    const int need = (nq + 31) / 32;
    static const int nvs[] = {1, 2, 4, 8, 12, 16};
    for (int v : nvs)
        if (v >= need) { s.nv = v; break; }
    if (!s.nv) return refuse(err, "n = %d too large (max 2048)", in.n);
    const int rb = narrow_rb(s.nv);
    // as many warps per CTA as keeps >= ~1 CTA per SM
    int threads = narrow_maxt(s.nv);
    while (threads > 64) {
        const int rows_per_cta = (threads / 32) * rb;
        const long long ctas = (long long)((pop + rows_per_cta - 1) / rows_per_cta) * B;
        if (ctas * 4 >= (long long)dev.sm_count * 3) break;   // bigger tiles re-read the pairs less often
        threads >>= 1;
    }
    s.threads = threads;
    s.ctas = (pop + (threads / 32) * rb - 1) / ((threads / 32) * rb);
    const size_t pair_bytes = (size_t)2 * ns * sizeof(float);
    // pairs per stage: one group of 8 when it fits (else 4 / 2 / 1); as many stages as the live pairs need, within
    // 160 KB, so that for the common shapes every pair is requested up front and nothing is re-issued
    const size_t budget = (size_t)160 * 1024;
    int kc = (int)(budget / 2 / pair_bytes);
    kc = kc >= 8 ? 8 : (kc >= 4 ? 4 : (kc >= 2 ? 2 : 1));
    // long rows (C4: 12 KB per pair): two stages of a FULL group of 8 still fit one SM (192 KB), and a 4-pair stage runs the
    // 8-wide group code half empty
    if (kc == 4 && 2 * 8 * pair_bytes + 24 * 1024 <= dev.smem_optin) kc = 8;
    s.kc = kc;
    const int max_chunks = (m + kc - 1) / kc;
    s.stages = (int)std::max<size_t>(2, std::min<size_t>(std::min(max_chunks, SAMPLE_MAX_STAGES), budget / (kc * pair_bytes)));   // >= 2 even beyond the budget
    s.smem = (size_t)s.stages * kc * pair_bytes + SAMPLE_MAX_STAGES * 8 + (size_t)(2 * m + 16) * sizeof(float);
    // one large population: split every row over CW column-warps (k_sample_wide) for occupancy
    if (pop >= 256 && nq > 32) {
        s.kind = Sampler::WIDE;
        s.CW = (nq + 31) / 32;
        s.qpw = (nq + s.CW - 1) / s.CW;
        // rows per warp: 2 (4 for very large populations); row-groups per CTA so that the grid still covers the SMs
        s.RBW = pop >= 1024 ? 4 : 2;
        int R = std::max(1, std::min(15, wide_maxt(s.RBW) / 32 / s.CW));
        while (R > 1 && (long long)((pop + R * s.RBW - 1) / (R * s.RBW)) * B * 4 < (long long)dev.sm_count * 3) R >>= 1;
        s.R = R;
        s.smem += (size_t)s.stages * ((kc + SAMPLE_G - 1) / SAMPLE_G) * s.R * s.CW * s.RBW * SAMPLE_G * sizeof(float);
        s.threads = 32 * s.R * s.CW;
        s.ctas = (pop + s.R * s.RBW - 1) / (s.R * s.RBW);
    }
    if (s.smem > dev.smem_optin) return refuse(err, "k_sample needs %zu B shared memory", s.smem);
    // many rows (batched queries, or one very large population): rows on lanes, column slices on warps (k_sample_rows)
    const long long total_rows = (long long)B * pop;
    // one population: from lambda = 8192 on it beats the wide sampler even though the progressive hand-over / overlapped
    // generation (wide sampler only) is given up (fused generation 0.271 -> 0.253 ms at 8192, 1.71 -> 1.41 ms at 65536)
    const bool many = total_rows >= 4096 && pop >= 32 &&
                      (B > 1 || tune.sample_rows == 1 || (pop >= 8192 && pop == in.lambda));
    if (many && nq <= 128 && m <= 256 && !in.has_prior) {
        const int NW = 16;
        const int qper = (nq + NW - 1) / NW;
        const int qw = qper <= 4 ? 4 : (qper <= 7 ? 7 : 8);
        // two rows per lane when an instance has them and the grid still fills the SMs
        const int rl = (pop >= 64 && total_rows / 64 >= 2LL * dev.sm_count) ? 2 : 1;
        const int rows = 32 * rl, kc2 = 8;
        const int chunks = (m + kc2 - 1) / kc2;
        const size_t stage_bytes = (size_t)kc2 * pair_bytes;
        const size_t fixed2 = SAMPLE_MAX_STAGES * 8 + (size_t)((m + kc2 + 3) & ~3) * 4 + (size_t)chunks * kc2 * rows * 4 + (size_t)NW * kc2 * rows * 4;
        const size_t tile_bytes = (size_t)rows * (ns + 4) * 4;
        if (fixed2 + std::max(2 * stage_bytes, tile_bytes) + 1024 <= dev.smem_optin) {
            const size_t room = dev.smem_optin - 1024 - fixed2;
            int stages = (int)std::min<size_t>(std::min(chunks, SAMPLE_MAX_STAGES), room / stage_bytes);
            stages = std::max(stages, 2);
            const size_t region = std::max((size_t)stages * stage_bytes, tile_bytes);
            const int nv = s.nv;
            s = {};
            s.kind = Sampler::ROWS;
            s.nv = nv;
            s.qw = qw; s.rl = rl; s.kc = kc2; s.stages = stages; s.region = (int)(region / 4);
            s.smem = region + fixed2;
            s.threads = 512;
            s.ctas = (pop + 32 * rl - 1) / (32 * rl);
        }
    }

    // ---- k_update
    auto& u = p.update;
    if (nq > 512) return refuse(err, "n = %d too large (max 2048)", in.n);
    u.nvb = nq <= 128 ? 4 : 16;
    const size_t fixed = (((size_t)m * 36 + 8 + 127) & ~(size_t)127) + (size_t)2048 * (UPD_GROUPS - 1);
    // + the block Gram entries, and the stages of the newest row's multi-warp chain (k_update.cuh: chain_part)
    const size_t rows = (size_t)m * ns * sizeof(float) + (size_t)m * (UPD_BLK + 1) * sizeof(float) +
                        (u.nvb == 4 ? (size_t)(2 * 4 * UPD_BLK * 32 + 16) * sizeof(float) + 16 : 0);
    const size_t ubudget = dev.smem_optin - 2048;            // static shared + slack
    u.rows_in_smem = fixed + rows <= ubudget;
    u.smem = fixed + (u.rows_in_smem ? rows : 0);
    if (u.smem > ubudget) return refuse(err, "k_update needs %zu B shared memory (m = %d too large)", u.smem, m);
    // rows that fit neither the registers nor the shared memory of one SM: Gram-matrix recompute (k_gram.cuh)
    const size_t coef_smem = (size_t)2 * m * (m | 1) * sizeof(double) + (size_t)2 * m * sizeof(double);
    u.gram = (!u.rows_in_smem || tune.update_gram) && m <= 128 && coef_smem <= ubudget;
    if (u.gram) {
        u.rows_in_smem = false; u.smem = fixed;
        // k_coef elements per lane: ceil(m / 8), rounded up to a compiled build (m <= 128); 8 lanes per basis row
        p.coef.elems = m <= 40 ? 5 : (m <= 80 ? 10 : (m <= 96 ? 12 : 16));
        p.coef.threads = std::min(1024, (8 * m + 31) & ~31);
        p.coef.smem = coef_smem;
    }
    // pending rows in registers when they fit: m <= 8 warps x RMAX rows of <= 128 float4 columns
    u.warps = UPD_WARPS;
    if (u.nvb == 4 && u.rows_in_smem && !u.gram) {
        // batched instances (more than one wave of one-CTA-per-SM launches: two 8-warp CTAs per SM take ~1.3x the time of one
        // 16-warp CTA, so a second wave is what they beat) whose rows fit 8 warps x 5: CTAs of 8 warps, two per
        // SM — the sweep of one instance is a chain of dependent steps that leaves its SM two thirds idle (k_update.cuh)
        const bool two_per_sm = 2 * u.smem + 4096 <= dev.smem_optin && m <= 8 * 5;
        if (tune.update_warps == 8 ? two_per_sm : (tune.update_warps == 0 && two_per_sm && B > dev.sm_count)) u.warps = 8;
        if (m <= u.warps * 3) u.rmax = 3;
        else if (m <= u.warps * 5) u.rmax = 5;
    }

    // one query with a wide sampler and the register sweep: k_sample consumes the direction pairs while k_update's sweep
    // is still producing them (k_update.cuh / k_sample.cuh "progressive")
    p.progressive = B == 1 && s.kind == Sampler::WIDE && u.rmax > 0 && !u.gram && !in.has_prior && s.kc == 8 &&
                    s.stages >= (m + s.kc - 1) / s.kc && in.rng == LMCMA_B200_RNG_PHILOX && tune.progressive != 0;
    p.overlap = p.progressive && tune.overlap != 0;
    *plan = p;
    return true;
}

void launch_fields(const LaunchPlan& p, int32_t* v) {
    const auto& s = p.sample;
    v[LMCMA_B200_LAUNCH_SAMPLER] = (int)s.kind;
    v[LMCMA_B200_LAUNCH_SMP_NV] = s.nv;
    v[LMCMA_B200_LAUNCH_SMP_SPEC] = 1;
    v[LMCMA_B200_LAUNCH_SMP_THREADS] = s.threads;
    v[LMCMA_B200_LAUNCH_SMP_RBW] = s.RBW;
    v[LMCMA_B200_LAUNCH_SMP_CW] = s.CW;
    v[LMCMA_B200_LAUNCH_SMP_R] = s.R;
    v[LMCMA_B200_LAUNCH_SMP_ROWS_QW] = s.qw;
    v[LMCMA_B200_LAUNCH_SMP_ROWS_RL] = s.rl;
    v[LMCMA_B200_LAUNCH_SMP_KC] = s.kc;
    v[LMCMA_B200_LAUNCH_SMP_STAGES] = s.stages;
    v[LMCMA_B200_LAUNCH_UPD_NVB] = p.update.nvb;
    v[LMCMA_B200_LAUNCH_UPD_RMAX] = p.update.rmax;
    v[LMCMA_B200_LAUNCH_UPD_ROWS_IN_SMEM] = p.update.rows_in_smem ? 1 : 0;
    v[LMCMA_B200_LAUNCH_UPD_GRAM] = p.update.gram ? 1 : 0;
    v[LMCMA_B200_LAUNCH_UPD_WARPS] = p.update.warps;
    v[LMCMA_B200_LAUNCH_UPD_SWEEP_WARPS] = p.update.warps;
    v[LMCMA_B200_LAUNCH_COEF_ELEMS] = p.coef.elems;
    v[LMCMA_B200_LAUNCH_RANK_THREADS] = p.rank.threads;
    v[LMCMA_B200_LAUNCH_RANK_FTILE] = p.rank.ftile;
    v[LMCMA_B200_LAUNCH_RANK_TILE_SORTED] = p.rank.tile_sorted ? 1 : 0;
    v[LMCMA_B200_LAUNCH_PROGRESSIVE] = p.progressive ? 1 : 0;
    v[LMCMA_B200_LAUNCH_OVERLAP] = p.overlap ? 1 : 0;
}

}  // namespace lmcma_capi

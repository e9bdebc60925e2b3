// k_update.cuh — the serial part of LMCMA::update (lmcma.cpp:316-424): mean, evolution path, slot
// bookkeeping, recomputation of the inverse-direction vectors (invAz, lmcma.cpp:449-463), population-success
// step size, best-so-far.  One CTA of 16 warps per optimiser instance.
//
// A single query is latency-bound (one generation moves a few MB), so this kernel is organised around
// its dependency chain:
//  * it is launched with programmatic dependent launch: everything that does not need this generation's
//    ranks — slot bookkeeping, the 1-D bulk async copies that bring the direction rows into shared memory,
//    their norms, the best-so-far arg-min — runs while k_rank is still ranking; griddep_wait() sits in front
//    of the first read of k_rank's partial sums;
//  * the triangular recompute runs factor-major (step j applies factor j to every pending row i > j: same
//    per-row operation order as the reference's row-major loops, lmcma.cpp:375-390).  All ~live^2/2 row-steps
//    run on this one SM, where shared-memory bandwidth is the scarce resource, so the pending rows are held in
//    REGISTERS by the warp that owns them and only finished rows pass through shared memory;
//  * progressive hand-over (UpdateArgs::progressive): the outputs are published with release stores as they become
//    final and the sampler, released early, consumes the direction pairs while the sweep is still producing them;
//  * overlapped generation (template parameter OVERLAP, one query): only the mean / step size / new evolution path
//    and the NEWEST row depend on this generation's fitness, so the kernel runs on a side branch of the CUDA graph
//    beside k_cost and k_rank — bookkeeping and the sweep over all older rows first, then a wait for k_rank's tickets,
//    then the rest.  Same operations in the same order as the serial launch order, bit for bit (DESIGN.md 4.2, 4.3).
#pragma once
#include "lmcma_common.cuh"
#include "lmcma_plan.hpp"
#include <type_traits>

namespace lmcma {

constexpr int UPD_THREADS = 32 * UPD_WARPS;

struct UpdateArgs {
    const float* f_all;        // B x lambda fitness of this generation (global candidate order)
    const float* slices;       // n_slices partial sums of w (x - xmean) per instance
    int n_slices;
    long long slice_stride, inst_stride;
    int payload_mode;          // slices are all-gather payloads (S rides in the 2 floats after ns)
    long long* dbg;            // optional: OptDev::dbg + TL_UPD, the TL_UPD_* timeline slots (LMCMA_B200_DBG); null in normal runs
    int overlap;               // fused single-query generation: this kernel runs on a side branch of the graph, CONCURRENTLY
                               // with k_cost and k_rank.  Everything that does not depend on this generation's fitness —
                               // bookkeeping, and the sweep over every pending row but the newest — comes first; then it
                               // waits for k_rank's tickets, forms the mean / new evolution path and finishes the newest
                               // row.  Implies `progressive` (k_sample is released by k_rank and follows the flags)
    int phase;                 // overlapped tell_all only (lmcma_b200_tell_all): 0 = the whole update; 1 = SPECULATIVE part of the NEXT
                               // generation's update, run right after this generation's (beside the sampler's last chunk and the
                               // candidates' trip across PCIe): bookkeeping, the sweep over every pending row but the newest and the
                               // block Gram entries — none of which depends on a fitness — with every global store switched off;
                               // the final rows, their |v|^2 and Lj / K and the Gram entries go to `spec`.  2 = the next tell_all
                               // resumes from `spec`: no sweep, the rows are committed to V / the mirror and published at once.
                               // Same arithmetic on the same inputs: bit-identical to phase 0
    float* spec;               // phase 1 / 2 scratch of one instance x spec_stride floats (layout: spec_* below)
    long long spec_stride;
    int progressive;           // publish OptDev::progress flags as the outputs become final: k_sample (launched as a
                               // programmatic dependent) consumes the pairs while the sweep is still producing them
};

// layout of UpdateArgs::spec (floats): [0] the generation (itr) the rows were computed for, [4 ..) Lj / K per position,
// |v|^2 per position, block Gram entries (m x UPD_BLK), rows (m x ns, 16-byte aligned)
__host__ __device__ __forceinline__ size_t spec_lj_off() { return 4; }
__host__ __device__ __forceinline__ size_t spec_nv_off(int m) { return 4 + (size_t)((m + 3) & ~3); }
__host__ __device__ __forceinline__ size_t spec_gs_off(int m) { return 4 + 2 * (size_t)((m + 3) & ~3); }
__host__ __device__ __forceinline__ size_t spec_rows_off(int m) { return spec_gs_off(m) + (size_t)m * UPD_BLK; }
__host__ __device__ __forceinline__ size_t spec_floats(int m, int ns) { return spec_rows_off(m) + (size_t)m * ns; }

#define UPD_STAMP(k) do { if (a.dbg && threadIdx.x == 0) a.dbg[k] = gtime(); } while (0)

template <bool SMEM> __device__ __forceinline__ float4 ld_row4(const float4* p) { return SMEM ? *p : __ldcg(p); }

// NVB  = float4 column slots per lane (ns <= 128 * NVB)
// RMAX = pending rows a warp can hold in registers (m <= WARPS * RMAX); 0 = streaming sweep (rows stay in
//        shared memory, or in HBM/L2 when SMEM is false); -1 = no sweep here: the recompute is done by the Gram-matrix
//        kernels (k_gram.cuh) for shapes whose rows fit neither registers nor shared memory; this kernel then only
//        hands them {first_stale, live}
// WARPS = warps per CTA: 16 (one CTA per SM), or 8 with two CTAs per SM for BATCHED instances — one instance's sweep is a
//        chain of dependent steps that leaves its SM two thirds idle (issue-active 32 %), two of them interleave.  Every
//        floating-point result is the same for both sizes (same per-row operation order, same summation tree in the mean
//        phase), so a batched instance stays bit-identical to the same instance run alone
template <int NVB, int RMAX, bool SMEM, bool OVERLAP, int WARPS = UPD_WARPS>
__global__ void __launch_bounds__(32 * WARPS, WARPS == UPD_WARPS ? 1 : 2) k_update(OptDev o, UpdateArgs a) {
    static_assert(WARPS == 16 || WARPS == 8, "CTA sizes the mean phase's summation tree is written for");
    static_assert(!OVERLAP || WARPS == UPD_WARPS, "the overlapped generation is a single-instance path");
    static_assert(RMAX <= 0 || NVB <= WARPS, "the newest row's chain takes NVB warps");
    static_assert(!OVERLAP || (RMAX > 0 && SMEM), "the overlapped generation uses the register sweep");
    static_assert(!OVERLAP || NVB + 2 <= WARPS, "the overlapped generation's tail: chain warps, best-so-far warps, one step-size warp");
    static_assert(RMAX <= 0 || SMEM, "the register sweep publishes finished rows through shared memory");
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int m = o.m, ns = o.ns, nq = ns >> 2;
    float* lj_s = reinterpret_cast<float*>(smem_raw);             // m: Lj / K in sequence order
    float* nv_s = lj_s + m;                                       // m: |v|^2 of the recomputed rows
    int* order = reinterpret_cast<int*>(nv_s + m);                // m: slot order
    int* stamp = order + m;                                       // m: generation stamp per SLOT
    float* ljslot = reinterpret_cast<float*>(stamp + m);          // m: Lj by slot (prefetched)
    unsigned long long* rowbar = reinterpret_cast<unsigned long long*>(smem_raw + (((size_t)m * 20 + 7) & ~(size_t)7));   // m mbarriers: row i is final
    unsigned long long* scalbar = rowbar + m;                      // m mbarriers: |v_i|^2 and Lj_i / K are published
    float4* red4 = reinterpret_cast<float4*>(smem_raw + (((size_t)m * 36 + 8 + 127) & ~(size_t)127));                      // 128 float4 scratch
    float* rows_s = reinterpret_cast<float*>(red4 + 128 * (UPD_GROUPS - 1));   // (the same layout for every WARPS)                                                                  // m x ns (SMEM)
    float* Gs = rows_s + (size_t)m * ns;                           // register sweep: m x UPD_BLK, Gs[k][r] = v_k . v_(j0 + r), j0 = k rounded down to its block, r < k - j0
    // register sweep: lane-partial dot products of the newest row's chain, 2 stages x NVB warps x UPD_BLK rows x 32 lanes, + NVB norms
    float* chain_part = reinterpret_cast<float*>((reinterpret_cast<size_t>(Gs + (size_t)m * (UPD_BLK + 1)) + 15) & ~(size_t)15);
    __shared__ unsigned long long sh_key;
    __shared__ int sh_dry;
    __shared__ __align__(8) unsigned long long sh_bar;
    __shared__ float am_v[UPD_WARPS];
    __shared__ int am_i[UPD_WARPS];
    const int b = blockIdx.x;
    const int tid = threadIdx.x, nthr = 32 * WARPS;
    const int lane = tid & 31, warp = tid >> 5, nwarps = WARPS;
    Scalars* scp = o.sc + b;
    int* tg = o.t + (size_t)b * m;
    int* vg = o.vec + (size_t)b * m;
    double* Njd = o.Nj + (size_t)b * m;
    double* Ljd = o.Lj + (size_t)b * m;
    float* Njf = o.Njf + (size_t)b * m;
    float* Vb = o.V + (size_t)b * m * ns;
    float* Pb = o.P + (size_t)b * m * ns;
    float* VPb = o.VPs + (size_t)b * m * 2 * ns;                   // sequence-ordered mirror for k_sample
    float* Njsb = o.Njs + (size_t)b * m;
    const float* fa = a.f_all + (size_t)b * o.lambda;

    // classic: k_sample may be scheduled right away; it waits for this grid to complete before reading anything.
    // progressive: it is released after this kernel's own wait (k_rank has reset the hand-over flags by then)
    if (!a.progressive) griddep_launch_dependents();
    int* flags = progress_flags(o.progress, m, b);
    const Scalars sc0 = *scp;
    float* const spec = OVERLAP && a.spec ? a.spec + (size_t)b * a.spec_stride : nullptr;
    int phase = OVERLAP ? a.phase : 0;
    // resume only from rows that were computed for THIS generation (the host invalidates after a state setter; this is the
    // belt to those braces): otherwise the whole update
    if (phase == 2 && (!spec || reinterpret_cast<const int*>(spec)[0] != sc0.itr)) phase = 0;
    if (phase == 1 && !spec) return;
    if (OVERLAP && phase != 1) {
        // the previous generation's sampler has completed (graph order): reset its flags, then tell k_gate that this CTA
        // holds its SM (k_cost is released only then and fills the other SMs)
        for (int i = tid; i < progress_len(m); i += nthr) flags[i] = 0;
        __syncthreads();
        if (tid == 0) { __threadfence(); st_release_gpu(o.resident + b, 1); }
    }
    UPD_STAMP(TL_UPD_START);
    // =============================== prologue: independent of k_rank ===============================
    for (int i = tid; i < m; i += nthr) { order[i] = tg[i]; stamp[i] = vg[i]; ljslot[i] = (float)Ljd[i]; mbar_init(&rowbar[i], 1); mbar_init(&scalbar[i], 1); }
    if (tid == 0) { sh_key = ~0ull; if (SMEM) mbar_init(&sh_bar, 1); }
    fence_barrier_init();
    __syncthreads();

    // ---- slot bookkeeping (lmcma.cpp:331-364): data-independent integer logic on shared-memory copies ----
    const int itr = sc0.itr;
    const double sigma_old = sc0.sigma;
    int first_stale = 0;
    if (itr < m) {
        if (tid == 0) order[itr] = itr;
    } else {
        // first minimal gap between adjacent generation stamps: key = (gap, j) lexicographic minimum
        if (warp == 0) {
            unsigned long long key = ~0ull;
            for (int j = lane; j < m - 1; j += 32) {
                const unsigned gap = (unsigned)(stamp[order[j + 1]] - stamp[order[j]]);
                const unsigned long long k2 = ((unsigned long long)gap << 32) | (unsigned)j;
                key = k2 < key ? k2 : key;
            }
#pragma unroll
            for (int ofs = 16; ofs > 0; ofs >>= 1) {
                const unsigned long long k2 = __shfl_xor_sync(0xffffffffu, key, ofs);
                key = k2 < key ? k2 : key;
            }
            if (lane == 0) sh_key = key;
        }
        __syncthreads();
        const unsigned long long key = sh_key;
        first_stale = (int)(unsigned)key + 1;
        if ((int)(key >> 32) >= m /* maxsteps = nvectors, lmcma.cpp:267 */) first_stale = 0;
        if (first_stale != m - 1) {                                  // rotate the recycled slot to the end
            const int recycled = order[first_stale];
            int* tmp = reinterpret_cast<int*>(nv_s);                  // nv_s is not in use yet
            for (int j = first_stale + tid; j < m - 1; j += nthr) tmp[j] = order[j + 1];
            __syncthreads();
            for (int j = first_stale + tid; j < m - 1; j += nthr) order[j] = tmp[j];
            if (tid == 0) order[m - 1] = recycled;
        }
    }
    __syncthreads();
    const int live = min(itr + 1, m);
    const int slot_new = order[live - 1];
    if (OVERLAP && tid == 0 && phase != 1) {                       // what the sampler needs to start on the finished pairs
        scp->itr = itr + 1; scp->live = live;
        st_release_gpu(flag_early(flags, m), 1);
    }
    if (first_stale == 1) first_stale = 0;                           // lmcma.cpp:373-374
    UPD_STAMP(TL_UPD_BOOKKEEPING);

    // ---- direction rows -> shared memory by 1-D bulk async copies issued by the lanes of warp 0: final rows
    //      (i < first_stale) come from V, pending rows start as their pc_j (lmcma.cpp:376-378); the newest
    //      pending row is this generation's pc, formed below ----
    if (SMEM && warp == 0) {
        const unsigned row_bytes = (unsigned)(ns * sizeof(float));
        if (lane == 0 && live > 1) mbar_expect_tx(&sh_bar, row_bytes * (unsigned)(live - 1));
        __syncwarp();
        for (int i = lane; i + 1 < live; i += 32) {
            // phase 2: every row but the newest is final already (the speculative pass of the last tell_all left them in `spec`)
            const float* src = phase == 2 ? spec + spec_rows_off(m) + (size_t)i * ns : (i < first_stale ? Vb : Pb) + (size_t)order[i] * ns;
            bulk_g2s(rows_s + (size_t)i * ns, src, row_bytes, &sh_bar);
        }
    }
    auto row_ptr = [&](int i) -> float* { return SMEM ? rows_s + (size_t)i * ns : Vb + (size_t)order[i] * ns; };
    const float invK = (float)(1.0 / o.K);
    for (int i = tid; i < m; i += nthr) {
        const int slot = order[i];
        if (phase != 1) {                                            // the speculative pass leaves the optimiser's state alone
            tg[i] = slot;
            vg[i] = (i == slot_new) ? itr : stamp[i];               // stamp is per SLOT
        }
        lj_s[i] = (i < live) ? ljslot[slot] * invK : 0.f;           // rows >= first_stale are recomputed below
        if (phase == 2 && i >= first_stale && i + 1 < live) {        // ... or were, by the speculative pass
            lj_s[i] = spec[spec_lj_off() + i];
            nv_s[i] = spec[spec_nv_off(m) + i];
        }
    }

    // ---- best-so-far: first occurrence of the minimum in evaluation order; strict improvement, or the very first
    //      evaluation (lmcma.cpp:192-198).  The fitness is k_cost's output (block-collective) ----
    // warps w0 .. w0 + nw - 1 take part (the whole CTA: barrier 0; otherwise named barrier 2 while the others are busy elsewhere)
    auto best_so_far = [&](const int w0, const int nw) {
    const int nt = 32 * nw, t = tid - 32 * w0;
    {
        float bf = __int_as_float(0x7f800000); int bi = 0x7fffffff;
        for (int j0 = 0; j0 < o.lambda; j0 += 4 * nt) {              // 4 loads in flight per thread
            float v[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) { const int j = j0 + u * nt + t; v[u] = (j < o.lambda) ? canon_fitness(__ldcg(fa + j)) : __int_as_float(0x7f800000); }
#pragma unroll
            for (int u = 0; u < 4; ++u) { const int j = j0 + u * nt + t; if (j < o.lambda && (v[u] < bf || (v[u] == bf && j < bi))) { bf = v[u]; bi = j; } }
        }
#pragma unroll
        for (int ofs = 16; ofs > 0; ofs >>= 1) {
            const float v2 = __shfl_xor_sync(0xffffffffu, bf, ofs); const int i2 = __shfl_xor_sync(0xffffffffu, bi, ofs);
            if (v2 < bf || (v2 == bf && i2 < bi)) { bf = v2; bi = i2; }
        }
        if (lane == 0) { am_v[warp] = bf; am_i[warp] = bi; }
    }
    if (nw == nwarps) __syncthreads(); else named_bar_sync(2, nt);
    {
        float bf = am_v[w0]; int bi = am_i[w0];
        for (int w2 = w0 + 1; w2 < w0 + nw; ++w2) if (am_v[w2] < bf || (am_v[w2] == bf && am_i[w2] < bi)) { bf = am_v[w2]; bi = am_i[w2]; }
        if (bi == 0x7fffffff) bi = 0;
        const bool take = ((double)bf < sc0.best_f) || (sc0.counteval == 0);
        const bool local = bi >= o.pop_offset && bi < o.pop_offset + o.pop_count;
        if (take && local && warp == w0 + nw - 1) {
            const float4* src = reinterpret_cast<const float4*>(o.X + ((size_t)b * o.pop_count + (bi - o.pop_offset)) * ns);
            float4* dst = reinterpret_cast<float4*>(o.best_x + (size_t)b * ns);
            for (int q = lane; q < nq; q += 32) dst[q] = src[q];
        }
        if (take && t == 0) { scp->best_f = (double)bf; scp->best_local = local ? 1 : 0; }
    }
    };
    if (RMAX < 0) {
        if (tid == 0) o.gram_hdr[b] = make_int2(first_stale, live);
    } else if (!SMEM) {                                              // rows stay in HBM/L2: pending rows start as pc_j
        for (int i = first_stale + warp; i + 1 < live; i += nwarps) {
            const float4* src = reinterpret_cast<const float4*>(Pb + (size_t)order[i] * ns);
            float4* dst = reinterpret_cast<float4*>(row_ptr(i));
            for (int q = lane; q < nq; q += 32) dst[q] = __ldcg(src + q);
        }
        __threadfence();
    } else if (live > 1) {
        mbar_wait(&sh_bar, 0);
    }
    if (OVERLAP) __syncthreads(); else best_so_far(0, nwarps);             // overlap: k_cost is still running
    UPD_STAMP(TL_UPD_PROLOGUE);

    // =============================== needs k_rank's partial sums ===============================
    // ---- population-success step size (lmcma.cpp:393-419), counters (lmcma.cpp:189, 423): needs only k_rank's pair
    //      count (one thread) ----
    unsigned long long S_early = 0;                                  // overlap: k_rank's pair count, taken when the ranks are in
    auto step_size_and_counters = [&]() {
        unsigned long long S = S_early;
        if (a.payload_mode) {
            for (int k = 0; k < a.n_slices; ++k) {
                const float* pay = a.slices + (size_t)k * a.slice_stride + (size_t)b * a.inst_stride + ns;
                S += ((unsigned long long)__float_as_uint(__ldcg(pay + 1)) << 32) | __float_as_uint(__ldcg(pay));
            }
        } else {
            if (!OVERLAP) S = atomicExch(o.S_count + b, 0ull);
        }
        if (itr > 0) {
            const double lam = (double)o.lambda;
            const unsigned long long L = (unsigned long long)o.lambda;
            const unsigned long long sum_cur = L * (L - 1ull) / 2ull + S;       // ranks of this generation in the merged order
            const unsigned long long sum_prev = L * (2ull * L - 1ull) - sum_cur;
            const double mean_cur = (double)sum_cur / lam, mean_prev = (double)sum_prev / lam;
            const double success = (mean_prev - mean_cur) / lam;
            const double snew = (1.0 - o.cs) * sc0.s + o.cs * (success - o.target);
            scp->s = snew;
            scp->sigma = sigma_old * exp(snew);
        }
        scp->itr = itr + 1;
        scp->live = live;
        scp->counteval = sc0.counteval + o.lambda;
    };
    // ---- one float4 column of the mean / evolution path / new pc_j (lmcma.cpp:316-329, 365-366); d = sum_i w_i (x_i - xmean) ----
    auto finish_column = [&](const int q, const float (&d)[4], const double2 xm01, const double2 xm23, const float4 pc4, const bool dry) {
        const double coef = o.pc_coef / sigma_old;                   // sqrt(cc (2 - cc) mueff) / sigma
        double* xm = o.xmean + (size_t)b * ns;
        float* pc = o.pc + (size_t)b * ns;
        float* pnew = Pb + (size_t)slot_new * ns;
        float* rnew = row_ptr(live - 1);
        const double xo[4] = {xm01.x, xm01.y, xm23.x, xm23.y};
        const float po[4] = {pc4.x, pc4.y, pc4.z, pc4.w};
        double xn[4]; float pn[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const double shift = (double)d[c];                       // new mean - old mean = sum_i w_i (x_i - xmean)
            xn[c] = xo[c] + shift;
            pn[c] = (float)__fma_rn(1.0 - o.cc, (double)po[c], __dmul_rn(coef, shift));   // explicit: the same bits wherever this is inlined
        }
        if (dry) return;                                             // pre-execution pass (see the overlapped tail): no side effects
        reinterpret_cast<double2*>(xm)[2 * q] = make_double2(xn[0], xn[1]);
        reinterpret_cast<double2*>(xm)[2 * q + 1] = make_double2(xn[2], xn[3]);
        const float4 p4 = make_float4(pn[0], pn[1], pn[2], pn[3]);
        reinterpret_cast<float4*>(pc)[q] = p4;
        reinterpret_cast<float4*>(pnew)[q] = p4;
        reinterpret_cast<float4*>(rnew)[q] = p4;
    };
    // prev_fit (lmcma.cpp:420-421) and the sorted fitness the next generation's k_rank searches (k_rank.cuh): k_rank has finished
    // reading the previous generation's values; nothing of this generation's update reads these
    auto copy_fitness = [&]() {
        for (int j = tid; j < o.lambda; j += nthr) {
            const float f = canon_fitness(__ldcg(fa + j));
            const float fs = o.prev_sorted ? __ldcg(o.fit_sorted + (size_t)b * o.lambda + j) : 0.f;
            o.prev_fit[(size_t)b * o.lambda + j] = f;
            if (o.prev_sorted) o.prev_sorted[(size_t)b * o.lambda + j] = fs;
        }
    };
    auto post_rank = [&](const bool dry) {                           // block-collective; dry: same instructions, no side effects
    if (!dry) UPD_STAMP(TL_UPD_POST);
    // overlap: the pair count is fetched here and used beside the chain, so its round trip hides behind the slice loads
    if (OVERLAP && tid == nthr - 1 && !dry && !a.payload_mode) S_early = atomicExch(o.S_count + b, 0ull);
    if (tid == 0 && !dry) o.rank_ticket[b] = 0u;                             // k_rank's CTAs of this generation have all drawn one
    // ---- population-success step size (lmcma.cpp:393-419), counters (lmcma.cpp:189, 423): needs only k_rank's pair
    //      count, so it goes first (the progressive hand-over publishes the scalars before the sweep).  The overlapped generation
    //      does it beside the newest row's chain and copies the fitness at its end, so that the mean's column sums wait for
    //      neither ----
    if (!OVERLAP) {
        if (tid == nthr - 1 && !dry) step_size_and_counters();
        if (!dry) copy_fitness();
    }

    // ---- mean, evolution path, new pc_j (lmcma.cpp:316-329, 365-366): 128 float4 columns x 2 slice groups, up to
    //      8 slice loads in flight per thread; fixed summation order -> deterministic ----
    {
        const double* xm = o.xmean + (size_t)b * ns;
        const float* pc = o.pc + (size_t)b * ns;
        // UPD_GROUPS (4) VIRTUAL groups of 128 threads share the slices out (group g sums slices g, g + 4, ...); a CTA of 16
        // warps has one hardware group per virtual group, a CTA of 8 warps runs two virtual groups per hardware group one after
        // the other: the summation tree is the same
        constexpr int HG = WARPS / 4, VPH = UPD_GROUPS / HG;         // hardware groups, virtual groups per hardware group
        const int tq = tid & 127, h = tid >> 7;
        for (int q0 = 0; q0 < nq; q0 += 128) {
            const int q = q0 + tq;
            float4 accv[VPH];
            double2 xm01 = make_double2(0.0, 0.0), xm23 = xm01;
            float4 pc4 = make_float4(0.f, 0.f, 0.f, 0.f);
            if (q < nq && h == 0) {
                xm01 = reinterpret_cast<const double2*>(xm)[2 * q]; xm23 = reinterpret_cast<const double2*>(xm)[2 * q + 1];
                pc4 = reinterpret_cast<const float4*>(pc)[q];
            }
#pragma unroll
            for (int vi = 0; vi < VPH; ++vi) {
                const int g = h + vi * HG;
                float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
                if (q < nq) {
                    const float4* sp = reinterpret_cast<const float4*>(a.slices + (size_t)b * a.inst_stride) + q;
                    const size_t sstride4 = (size_t)a.slice_stride >> 2;
                    int k = g;
                    for (; k + 7 * UPD_GROUPS < a.n_slices; k += 8 * UPD_GROUPS) {   // 8 loads in flight
                        float4 v[8];
#pragma unroll
                        for (int u = 0; u < 8; ++u) v[u] = __ldcg(sp + (size_t)(k + UPD_GROUPS * u) * sstride4);
#pragma unroll
                        for (int u = 0; u < 8; ++u) { acc.x += v[u].x; acc.y += v[u].y; acc.z += v[u].z; acc.w += v[u].w; }
                    }
                    for (; k < a.n_slices; k += UPD_GROUPS) { const float4 v = __ldcg(sp + (size_t)k * sstride4); acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w; }
                }
                accv[vi] = acc;
                if (g > 0) red4[(g - 1) * 128 + tq] = acc;
            }
            __syncthreads();
            if (h == 0 && q < nq) {
                float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                for (int g2 = 0; g2 + 1 < UPD_GROUPS; ++g2) { const float4 u4 = red4[g2 * 128 + tq]; t.x += u4.x; t.y += u4.y; t.z += u4.z; t.w += u4.w; }
                const float d[4] = {accv[0].x + t.x, accv[0].y + t.y, accv[0].z + t.z, accv[0].w + t.w};
                finish_column(q, d, xm01, xm23, pc4, dry);
            }
            __syncthreads();
        }
    }
    if (!SMEM) __threadfence();
    __syncthreads();
    if (!dry) UPD_STAMP(TL_UPD_MEAN);
    if (a.progressive && !dry) {
        // scalars and mean are final; so are the pairs in front of the first stale position (untouched this generation;
        // overlap mode has published those before its sweep)
        if (!OVERLAP) for (int i = tid; i < first_stale; i += nthr) st_release_gpu(flag_pair(flags, i), 1);
        if (tid == 0 && !OVERLAP) st_release_gpu(flag_mean(flags), 1);   // overlap: with the step size, beside the chain
    }
    };
    if (!OVERLAP) {
        griddep_wait();
        if (a.progressive) griddep_launch_dependents();
        post_rank(false);
    } else {
        if (phase != 1) for (int i = tid; i < first_stale; i += nthr) st_release_gpu(flag_pair(flags, i), 1);   // untouched pairs: final already
    }

    // ---- recompute v from the first stale position (lmcma.cpp:373-390) ----
    // Closed forms of lmcma.cpp:386-389 with t = sqrt(1 + c1/(1-c1) |v|^2), rewritten without cancellation:
    //   Nj = (sqrt(1-c1)/|v|^2)(t - 1)            = sqrt(1-c1) * r / (t + 1)
    //   Lj = (1/(sqrt(1-c1)|v|^2))(1 - 1/t)       = r / (sqrt(1-c1) * t * (t + 1)),   r = c1/(1-c1)
    // (identical in exact arithmetic; finite where the reference divides 0/0 for a zero vector).
    //
    // Factor-major sweep: step j applies factor j, x <- K x - Lj_j (v_j . x) v_j, to every pending row i > j.
    //  * pending rows are held as y = x / K^j (all pending rows have had the same number of factors applied),
    //    which turns the update into y <- y - (Lj_j / K)(v_j . y) v_j: one FMA per element; a row is multiplied
    //    by K^i once, when it becomes final;
    //  * |v_i|^2 (which Lj_i needs) is a real reduction over the finished row, as in the reference (lmcma.cpp:383-384) —
    //    a scalar recurrence |y'|^2 = |y|^2 - 2 e d + e^2 |v_j|^2 cancels catastrophically once the evolution paths
    //    are nearly collinear with the stored directions — but it is taken AFTER the row has been handed over:
    //    the consumers need Lj_i only after their own dot products, so it is off the chain;
    //  * a row is owned by one warp for the whole sweep; when its last factor has been applied the owner
    //    publishes it (row, |v|^2, Lj/K, then an mbarrier arrive by every lane) and the other warps pick it up
    //    as factor i with a blocking mbarrier wait: no block-wide barrier and no spinning warps competing
    //    with the owner of the next row for issue slots.
    const double Kd = o.K;
    const float r_f = (float)(o.c1 / (1.0 - o.c1)), a_f = (float)o.M;
    auto publish_scalars = [&](int i, float nv) {                   // lane 0: |v_i|^2 and Lj_i / K
        const float t = sqrtf(fmaf(r_f, nv, 1.0f));
        nv_s[i] = nv;
        lj_s[i] = __fdividef(r_f, a_f * t * (t + 1.0f)) * invK;
    };
    auto pair_final = [&](int i, float nv) {                        // one thread: pair i of the mirror and Njs[i] are final
        Njsb[i] = (float)nj_form(nj_ratio(o), o.M, nv).nj;
        st_release_gpu(flag_pair(flags, i), 1);
    };

    if (RMAX < 0) {
        // the Gram-matrix kernels take it from here (they also write Nj / Lj)
    } else if (RMAX > 0) {
        // ---------------- register sweep: warp w owns rows first_stale + w + r * WARPS ----------------
        constexpr int R = RMAX > 0 ? RMAX : 1;
        constexpr int rstride = WARPS;
        // The newest row (this generation's evolution path) is not part of the sweep: it takes its factors a BLOCK at a time
        // (newest_row below).  In the overlapped generation it does not even exist yet when the sweep starts.
        const int hi = live - 1;
        const int base = phase != 2 ? first_stale + warp : hi;      // phase 2: no sweep
        float4 y[R][NVB];
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int i = base + r * rstride;
            const bool on = i < hi;
#pragma unroll
            for (int it = 0; it < NVB; ++it) {
                const int q = lane + 32 * it;
                y[r][it] = (on && q < nq) ? reinterpret_cast<const float4*>(rows_s + (size_t)i * ns)[q] : make_float4(0.f, 0.f, 0.f, 0.f);
                if (on && q < nq && phase != 1) reinterpret_cast<float4*>(VPb + ((size_t)i * 2 + 1) * ns)[q] = y[r][it];   // pc_i at its (new) position
            }
        }
        // y[0 .. n-1] are my pending rows in index order, y[0] the next one to become final (row `next`): when it does, the
        // others move down one place, so that a step costs what the rows still pending cost (the SM is issue-bound here)
        int n = 0;
#pragma unroll
        for (int r = 0; r < R; ++r) n += (base + r * rstride < hi) ? 1 : 0;
        int next = base;
        auto retire_first = [&]() {
#pragma unroll
            for (int r = 0; r + 1 < R; ++r) {
#pragma unroll
                for (int it = 0; it < NVB; ++it) y[r][it] = y[r + 1][it];
            }
            --n; next += rstride;
        };
        // Block Gram entries of a final row k (in registers, x) against the earlier rows of its block of UPD_BLK: what lets the
        // newest row take a whole block of factors at once.  Warp-collective; rows j0 .. k-1 are final in shared memory.
        auto gram_entries = [&](const float4 (&x)[NVB], const int k) {
            const int j0 = k & ~(UPD_BLK - 1), nbk = k - j0;
            if (nbk == 0) return;
            float gd[UPD_BLK - 1];
#pragma unroll
            for (int r = 0; r < UPD_BLK - 1; ++r) {
                gd[r] = 0.f;
                if (r < nbk) {
                    const float4* vr = reinterpret_cast<const float4*>(rows_s + (size_t)(j0 + r) * ns);
                    float2 d0 = make_float2(0.f, 0.f), d1 = d0;
#pragma unroll
                    for (int it = 0; it < NVB; ++it) {
                        const int q = lane + 32 * it;
                        const float4 v = (q < nq) ? vr[q] : make_float4(0.f, 0.f, 0.f, 0.f);
                        d0 = ffma2(lo2(v), lo2(x[it]), d0); d1 = ffma2(hi2(v), hi2(x[it]), d1);
                    }
                    gd[r] = (d0.x + d0.y) + (d1.x + d1.y);
                }
            }
#pragma unroll
            for (int ofs = 16; ofs > 0; ofs >>= 1) {
#pragma unroll
                for (int r = 0; r < UPD_BLK - 1; ++r) gd[r] += __shfl_xor_sync(0xffffffffu, gd[r], ofs);
            }
            if (lane == 0) {
#pragma unroll
                for (int r = 0; r < UPD_BLK - 1; ++r) if (r < nbk) Gs[k * UPD_BLK + r] = gd[r];
            }
        };
        auto gram_row = [&](const int k) {                           // row k is final in shared memory
            float4 x[NVB];
#pragma unroll
            for (int it = 0; it < NVB; ++it) {
                const int q = lane + 32 * it;
                x[it] = (q < nq) ? reinterpret_cast<const float4*>(rows_s + (size_t)k * ns)[q] : make_float4(0.f, 0.f, 0.f, 0.f);
            }
            gram_entries(x, k);
        };
        auto publish = [&](const float4 (&row)[NVB], int i, double kp) {   // warp-collective: y_i K^i is the final v_i
            const float kf = (float)kp;
            float4* srow = reinterpret_cast<float4*>(rows_s + (size_t)i * ns);
            float4* dst = reinterpret_cast<float4*>(Vb + (size_t)order[i] * ns);
            float4* dst2 = reinterpret_cast<float4*>(VPb + (size_t)i * 2 * ns);
            float4 x[NVB];
#pragma unroll
            for (int it = 0; it < NVB; ++it) {
                const int q = lane + 32 * it;
                const float2 k2 = make_float2(kf, kf), l = fmul2(lo2(row[it]), k2), h = fmul2(hi2(row[it]), k2);
                x[it] = make_float4(l.x, l.y, h.x, h.y);
                if (q < nq) srow[q] = x[it];
            }
            __syncwarp();                                            // orders the lanes' stores before lane 0's release
            if (lane == 0) mbar_arrive(&rowbar[i]);                  // ONE arrive: 32 arrives on one mbarrier serialise (~27 cycles each)
            if (a.dbg && lane == 0 && i < TL_UPD_ROW_STAMPS) a.dbg[TL_UPD_ROWS + i] = gtime();
            float2 nn = make_float2(0.f, 0.f);                       // |v_i|^2: after the hand-over, off the chain
#pragma unroll
            for (int it = 0; it < NVB; ++it) { nn = ffma2(lo2(x[it]), lo2(x[it]), nn); nn = ffma2(hi2(x[it]), hi2(x[it]), nn); }
            const float nv = warp_sum(nn.x + nn.y);
            if (lane == 0) {
                publish_scalars(i, nv);
                mbar_arrive(&scalbar[i]);
            }
            // the copy to HBM goes after the arrive: a release has to wait for every earlier store of the thread, and
            // a store to HBM takes an L2 round trip that the next step of the sweep must not sit behind
#pragma unroll
            for (int it = 0; it < NVB; ++it) {
                const int q = lane + 32 * it;
                if (q < nq && phase != 1) { dst[q] = x[it]; dst2[q] = x[it]; }
            }
            if (a.progressive && phase != 1) {
                __syncwarp();
                if (lane == 0) pair_final(i, nv);
            }
        };
        // ---- the newest row: this generation's evolution path through the factors 0 .. live-2 (lmcma.cpp:375-382), a block of
        //      UPD_BLK factors at a time.  With y the row at the start of a block j0 .. j0+nb-1 (held as x / K^j like the sweep's
        //      rows) and g_k = v_k . y, the dot products the factors would see one after the other are
        //          d_k = g_k - sum_{i < k} e_i (v_k . v_i),   e_k = (Lj_k / K) d_k,
        //      a recurrence on scalars over the block's Gram entries (gram_entries above: they do not depend on this generation's
        //      fitness), and the block leaves y - sum_k e_k v_k: nb independent dot products, ONE batched reduction and nb
        //      multiply-adds per element instead of nb dependent dot-reduce-update steps.
        //      The chain is on the critical path of the single-query generation (nothing else runs on this SM by then), so it is
        //      spread over NVB warps: warp w owns float4 column lane + 32 w of the row, the lane-partial dot products of the NVB
        //      warps meet in shared memory (one named barrier per block, double-buffered), and every warp runs the same
        //      reduction and scalar recurrence on the same numbers in the same order, so all of them hold the same e_k.  One
        //      warp walking 4 columns per lane took 1.2 us per block (2.4 K cycles of dependent loads and multiply-adds).
        //      Collective over warps 0 .. NVB-1. ----
        auto newest_row = [&](const bool dry, const unsigned need) {
            const int q = lane + 32 * warp;
            const bool has = q < nq;
            const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
            const float4 pc4 = has ? reinterpret_cast<const float4*>(rows_s + (size_t)(live - 1) * ns)[q] : zero4;
            float4 yn = pc4;
            double kn = 1.0;
            for (int j = 0; j + 1 < live; ++j) kn *= Kd;             // the same product the sweep forms step by step
            const int rr = lane >> 2, qq = lane & 3;                 // lanes 4 rr .. 4 rr + 3 look after row j0 + rr of the block
            float* norm_part = chain_part + 2 * NVB * UPD_BLK * 32;  // behind the two dot-product stages: NVB norms, 2 verdicts of the dry pass
            int buf = 0;
#pragma unroll 1
            for (int j0 = 0; j0 + 1 < live; j0 += UPD_BLK, buf ^= 1) {
                const int nb = min(UPD_BLK, live - 1 - j0);
                float* pw = chain_part + (size_t)((buf * NVB + warp) * UPD_BLK) * 32;
                float4 v[UPD_BLK];
#pragma unroll
                for (int r = 0; r < UPD_BLK; ++r) {                  // my column's share of g_r (an absent row gives 0)
                    v[r] = (has && r < nb) ? reinterpret_cast<const float4*>(rows_s + (size_t)(j0 + r) * ns)[q] : zero4;
                    float2 d = fmul2(lo2(v[r]), lo2(yn));
                    d = ffma2(hi2(v[r]), hi2(yn), d);
                    pw[r * 32 + lane] = d.x + d.y;
                }
                // what the recurrence needs besides g: my row's Gram entries against the earlier rows of the block and its Lj / K
                float gi[UPD_BLK];
                {
                    const float4* gp = reinterpret_cast<const float4*>(Gs + (size_t)(j0 + min(rr, nb - 1)) * UPD_BLK);
                    const float4 g0 = gp[0], g1 = gp[1];
                    const float gg[UPD_BLK] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
#pragma unroll
                    for (int i = 0; i < UPD_BLK; ++i) gi[i] = (rr > i && rr < nb) ? gg[i] : 0.f;
                }
                const float ljm = (rr < nb) ? lj_s[j0 + rr] : 0.f;
                // dry pass: one thread looks for k_rank's tickets; its verdict crosses the barrier, so that every chain warp
                // leaves the loop in the same block
                if (dry && tid == 0) norm_part[4 + buf] = (*reinterpret_cast<const volatile int*>(o.rank_ticket + b) == (int)need) ? 1.f : 0.f;
                named_bar_sync(3, 32 * NVB);
                if (dry && norm_part[4 + buf] != 0.f) break;
                float gs;                                            // g of my row: 8 lanes' partials per quarter and warp, then the 4 quarters
                {
                    float sw[NVB];
#pragma unroll
                    for (int w = 0; w < NVB; ++w) {
                        const float4* pp = reinterpret_cast<const float4*>(chain_part + (size_t)((buf * NVB + w) * UPD_BLK + rr) * 32 + qq * 8);
                        const float4 p0 = pp[0], p1 = pp[1];
                        sw[w] = ((p0.x + p0.y) + (p0.z + p0.w)) + ((p1.x + p1.y) + (p1.z + p1.w));
                    }
                    gs = sw[0];
#pragma unroll
                    for (int w = 1; w < NVB; ++w) gs += sw[w];
                }
                gs += __shfl_xor_sync(0xffffffffu, gs, 1);
                gs += __shfl_xor_sync(0xffffffffu, gs, 2);
                // the scalar recurrence: e_i is final on the lanes of row i once e_0 .. e_(i-1) have been taken off (rows past the
                // block's end have Lj = 0: their e is 0)
                float acc = 0.f, em = 0.f;
#pragma unroll
                for (int i = 0; i < UPD_BLK; ++i) {
                    const float ei = __shfl_sync(0xffffffffu, ljm * (gs - acc), 4 * i);
                    if (rr == i) em = ei;
                    acc = fmaf(ei, gi[i], acc);
                }
#pragma unroll
                for (int r = 0; r < UPD_BLK; ++r) {                  // y <- y - e_r v_r, in the order of the factors
                    const float er = __shfl_sync(0xffffffffu, em, 4 * r);
                    const float2 me = make_float2(-er, -er);
                    const float2 l = ffma2(me, lo2(v[r]), lo2(yn)), h = ffma2(me, hi2(v[r]), hi2(yn));
                    yn = make_float4(l.x, l.y, h.x, h.y);
                }
                if (a.dbg && tid == 0 && OVERLAP && !dry) a.dbg[TL_UPD_CHAIN + (j0 >> 3)] = gtime();
            }
            // pc at its position in the mirror (after the chain: nothing in it should queue behind these stores)
            if (has && !dry) reinterpret_cast<float4*>(VPb + ((size_t)(live - 1) * 2 + 1) * ns)[q] = pc4;
            if (OVERLAP) { if (a.dbg && tid == 0 && !dry) a.dbg[TL_UPD_BEST_COPIED] = gtime(); __syncthreads(); }   // the other warps have copied the best-so-far candidate out of X
            // ---- publish: y K^(live-1) is the final v of the newest pair (what publish() does for a row held by one warp) ----
            const int i = live - 1;
            const float kf = (float)kn;
            const float2 k2 = make_float2(kf, kf), xl = fmul2(lo2(yn), k2), xh = fmul2(hi2(yn), k2);
            const float4 x = make_float4(xl.x, xl.y, xh.x, xh.y);
            if (has && !dry) reinterpret_cast<float4*>(rows_s + (size_t)i * ns)[q] = x;
            float2 nn = fmul2(lo2(x), lo2(x));
            nn = ffma2(hi2(x), hi2(x), nn);
            const float nw = warp_sum(nn.x + nn.y);
            if (lane == 0) norm_part[warp] = nw;
            if (has && !dry) {
                reinterpret_cast<float4*>(Vb + (size_t)order[i] * ns)[q] = x;
                reinterpret_cast<float4*>(VPb + (size_t)i * 2 * ns)[q] = x;
            }
            named_bar_sync(3, 32 * NVB);                              // every chain warp's stores come before thread 0's release
            if (tid == 0 && !dry) {
                float nv = norm_part[0];
#pragma unroll
                for (int w = 1; w < NVB; ++w) nv += norm_part[w];
                mbar_arrive(&rowbar[i]);
                if (a.dbg && i < TL_UPD_ROW_STAMPS) a.dbg[TL_UPD_ROWS + i] = gtime();
                publish_scalars(i, nv);
                mbar_arrive(&scalbar[i]);
                if (a.progressive) pair_final(i, nv);
            }
        };
        if (first_stale == 0 && warp == 0 && hi > 0 && phase != 2) { publish(y[0], 0, 1.0); retire_first(); }   // row 0 has no factors (v_0 = pc_0)
        double kp = 1.0;                                             // K^(j+1) inside step j
        for (int j = 0; j + 1 < hi; ++j) {
            kp *= Kd;
            if (n == 0) break;                                       // all my rows are final
            if (j >= first_stale) mbar_wait(&rowbar[j], 0);
            const float4* vj = reinterpret_cast<const float4*>(rows_s + (size_t)j * ns);
            float4 a4[NVB];
#pragma unroll
            for (int it = 0; it < NVB; ++it) {
                const int q = lane + 32 * it;
                a4[it] = (q < nq) ? vj[q] : make_float4(0.f, 0.f, 0.f, 0.f);
            }
            // the row that becomes final in this step goes first and alone: the next step waits for it
            if (next == j + 1) {
                float2 dd = make_float2(0.f, 0.f);
#pragma unroll
                for (int it = 0; it < NVB; ++it) { dd = ffma2(lo2(a4[it]), lo2(y[0][it]), dd); dd = ffma2(hi2(a4[it]), hi2(y[0][it]), dd); }
                const float d = warp_sum(dd.x + dd.y);
                if (j >= first_stale) mbar_wait(&scalbar[j], 0);   // Lj_j / K, |v_j|^2: published right after the row (long done)
                const float e = lj_s[j] * d;
                const float2 me = make_float2(-e, -e);
#pragma unroll
                for (int it = 0; it < NVB; ++it) {
                    const float2 l = ffma2(me, lo2(a4[it]), lo2(y[0][it])), h = ffma2(me, hi2(a4[it]), hi2(y[0][it]));
                    y[0][it] = make_float4(l.x, l.y, h.x, h.y);
                }
                publish(y[0], j + 1, kp);
                retire_first();
            }
            // my other pending rows: one straight-line block per count, so that the dot-product chains and the 5 shuffle
            // rounds of the rows interleave (a branch per row would serialise their latencies)
            auto others = [&](auto nc) {
                constexpr int N = decltype(nc)::value;
                float d[N];
#pragma unroll
                for (int r = 0; r < N; ++r) {
                    float2 d0 = make_float2(0.f, 0.f), d1 = d0;
#pragma unroll
                    for (int it = 0; it < NVB; ++it) { d0 = ffma2(lo2(a4[it]), lo2(y[r][it]), d0); d1 = ffma2(hi2(a4[it]), hi2(y[r][it]), d1); }
                    d[r] = (d0.x + d0.y) + (d1.x + d1.y);
                }
#pragma unroll
                for (int ofs = 16; ofs > 0; ofs >>= 1) {
#pragma unroll
                    for (int r = 0; r < N; ++r) d[r] += __shfl_xor_sync(0xffffffffu, d[r], ofs);
                }
                if (j >= first_stale) mbar_wait(&scalbar[j], 0);
                const float ljk = lj_s[j];
#pragma unroll
                for (int r = 0; r < N; ++r) {
                    const float e = ljk * d[r];
                    const float2 me = make_float2(-e, -e);
#pragma unroll
                    for (int it = 0; it < NVB; ++it) {
                        const float2 l = ffma2(me, lo2(a4[it]), lo2(y[r][it])), h = ffma2(me, hi2(a4[it]), hi2(y[r][it]));
                        y[r][it] = make_float4(l.x, l.y, h.x, h.y);
                    }
                }
            };
            switch (n) {
                case 0: break;
                case 1: others(std::integral_constant<int, 1>()); break;
                case 2: others(std::integral_constant<int, (R >= 2 ? 2 : 1)>()); break;
                case 3: others(std::integral_constant<int, (R >= 3 ? 3 : 1)>()); break;
                case 4: others(std::integral_constant<int, (R >= 4 ? 4 : 1)>()); break;
                default: others(std::integral_constant<int, (R >= 5 ? 5 : 1)>()); break;
            }
        }
        if (phase == 2) {
            // ---- resume: the rows are in shared memory (bulk copies from `spec`, waited for above); commit the recomputed ones to
            //      V and the mirror and publish them, a warp per row — what publish() did step by step in the sweep ----
            for (int i = tid; i < m * UPD_BLK; i += nthr) Gs[i] = spec[spec_gs_off(m) + i];
            for (int i = first_stale + warp; i < hi; i += WARPS) {
                const float4* srow = reinterpret_cast<const float4*>(rows_s + (size_t)i * ns);
                const float4* prow = reinterpret_cast<const float4*>(Pb + (size_t)order[i] * ns);
                float4* dst = reinterpret_cast<float4*>(Vb + (size_t)order[i] * ns);
                float4* dst2 = reinterpret_cast<float4*>(VPb + (size_t)i * 2 * ns);
                for (int q = lane; q < nq; q += 32) { const float4 x = srow[q]; dst[q] = x; dst2[q] = x; dst2[nq + q] = __ldcg(prow + q); }
                __syncwarp();
                if (lane == 0) pair_final(i, nv_s[i]);
            }
        }
        // every older row is final
        __syncthreads();
        UPD_STAMP(TL_UPD_ROWS_FINAL);
        if (phase != 2) for (int k = 1 + warp; k < hi; k += WARPS) gram_row(k);  // block Gram entries for the newest row's chain
        if (phase == 1) {
            // ---- speculative pass: leave the rows, their scalars and the Gram entries for the next tell_all and stop here ----
            __syncthreads();
            for (int i = tid; i < m * UPD_BLK; i += nthr) spec[spec_gs_off(m) + i] = Gs[i];
            for (int i = tid; i < hi; i += nthr) { spec[spec_lj_off() + i] = lj_s[i]; spec[spec_nv_off(m) + i] = nv_s[i]; }
            const float4* s4 = reinterpret_cast<const float4*>(rows_s);
            float4* d4 = reinterpret_cast<float4*>(spec + spec_rows_off(m));
            for (int i = tid; i < hi * nq; i += nthr) d4[i] = s4[i];
            if (tid == 0) reinterpret_cast<int*>(spec)[0] = itr;
            return;
        }
        if (OVERLAP) {
            // ---------------- overlap: the part that needs this generation's ranks ----------------
            // Everything from here to the sampler's last chunk is the critical path of the single-query generation, and it is
            // code this SM has not executed yet: its instruction lines come from L2 (from HBM after an L2 flush) one miss after
            // the other - the first block of the newest row's chain took 4.7 us against 0.65 us for each of the following ones.
            // The sweep, however, is normally done well before k_rank is (the fused generation: ~10 us), so while the ranks
            // are not there yet the SAME instructions are run once with their side effects switched off (`dry`: loads, arithmetic,
            // barriers, no global store, no flag): the real pass then finds them in the instruction cache.  One code path for
            // both passes (a loop, not two inlined copies).  No dry pass when the ranks are already there (tell_all, where the
            // sweep is the longer branch).
            const unsigned need = (unsigned)o.RS;                    // k_rank: one ticket per CTA after its last store (k_rank.cuh)
            // steps: 0 the chain, dry; 1 mean / step size / path, dry; 2 the same for real (after the ranks); 3 the chain for real.
            // A dry step starts only while tickets are missing, and the dry chain gives up between two blocks once they are all there.
#pragma unroll 1
            for (int step = 0; step < 4; ++step) {
                const bool dry = step < 2;
                if (dry) {
                    if (tid == 32) sh_dry = *reinterpret_cast<const volatile int*>(o.rank_ticket + b) != (int)need ? 1 : 0;
                    __syncthreads();
                    if (!sh_dry) { step = 1; continue; }
                } else if (step == 2) {
                    if (tid == 32) {
                        // plain polling by one thread (this wait is on the critical path); the fence is the acquire for the ranks /
                        // partial sums behind the tickets
                        const long long t0 = gtime();
                        for (long long spin = 0; *reinterpret_cast<const volatile int*>(o.rank_ticket + b) != (int)need; ++spin)
                            if ((spin & 255) == 255 && gtime() - t0 > LOST_TIMEOUT_NS) {   // k_rank never ran beside this kernel: tell the
                                report_lost(o.err, LOST_UPDATE_WAITING_FOR_RANK);          // host and carry on (this generation is void)
                                break;
                            }
                        __threadfence();
                    }
                    __syncthreads();
                    UPD_STAMP(TL_UPD_RANKS_SEEN);
                }
                if (step == 1 || step == 2) {
                    post_rank(dry);                                  // mean, step size, the new evolution path -> rows_s[live - 1]
                } else if (warp >= NVB) {
                    // while warps 0 .. NVB-1 run the newest row's chain, the last warp forms the step size and counters and releases
                    // them with the mean (the sampler reads sigma behind that flag), and the others track the best-so-far candidate
                    // (it reads X, which the sampler overwrites only after the newest pair has been published)
                    if (warp == nwarps - 1) {
                        if (tid == nthr - 1 && !dry) {                // the thread that took the pair count in post_rank
                            step_size_and_counters();
                            if (a.progressive) st_release_gpu(flag_mean(flags), 1);
                            if (a.dbg) a.dbg[TL_UPD_STEP_SIZE] = gtime();
                        }
                    } else if (!dry) {
                        best_so_far(NVB, nwarps - NVB - 1);
                    }
                    __syncthreads();
                } else {
                    newest_row(dry, need);
                    if (!dry) UPD_STAMP(TL_UPD_NEWEST);
                }
            }
        } else {
            __syncthreads();
            if (warp < NVB) newest_row(false, 0u);
        }
    } else {
        // ---------------- streaming sweep: pending rows stay in shared memory (or HBM/L2) ----------------
        const int pend = live - first_stale;
        const int act_warps = min(nwarps, pend);
        for (int i = first_stale + warp; i < live; i += nwarps) {    // pc_i at its (new) position in the mirror
            const float4* src = reinterpret_cast<const float4*>(row_ptr(i));
            float4* dst2 = reinterpret_cast<float4*>(VPb + ((size_t)i * 2 + 1) * ns);
            for (int q = lane; q < nq; q += 32) dst2[q] = ld_row4<SMEM>(src + q);
        }
        auto publish = [&](int i, double kp) {                       // warp-collective: y_i K^i is the final v_i
            const float kf = (float)kp;
            float4* row = reinterpret_cast<float4*>(row_ptr(i));
            float4* dst = reinterpret_cast<float4*>(Vb + (size_t)order[i] * ns);
            float4* dst2 = reinterpret_cast<float4*>(VPb + (size_t)i * 2 * ns);
            float nn = 0.f;
            for (int q = lane; q < nq; q += 32) {
                float4 x = ld_row4<SMEM>(row + q);
                x.x *= kf; x.y *= kf; x.z *= kf; x.w *= kf;
                row[q] = x;
                nn += fmaf(x.x, x.x, x.y * x.y) + fmaf(x.z, x.z, x.w * x.w);
            }
            nn = warp_sum(nn);
            if (lane == 0) publish_scalars(i, nn);
            if (!SMEM) __threadfence();
            __syncwarp();                                            // orders the lanes' stores before lane 0's release
            if (lane == 0) mbar_arrive(&rowbar[i]);
            for (int q = lane; q < nq; q += 32) {                    // copies to HBM after the release (see the register sweep)
                const float4 x = ld_row4<SMEM>(row + q);
                if (SMEM) dst[q] = x;
                dst2[q] = x;
            }
        };
        if (warp < act_warps) {
            int i0 = first_stale + warp;                             // my first row that is not final yet
            if (first_stale == 0 && warp == 0) publish(0, 1.0);      // row 0 has no factors (v_0 = pc_0)
            double kp = 1.0;                                         // K^(j+1) inside step j
            for (int j = 0; j + 1 < live; ++j) {
                kp *= Kd;
                while (i0 <= j) i0 += act_warps;
                if (i0 >= live) break;
                if (j >= first_stale) mbar_wait(&rowbar[j], 0);
                const float4* vj = reinterpret_cast<const float4*>(row_ptr(j));
                const float ljk = lj_s[j];
                for (int i = i0; i < live; i += act_warps) {
                    float4* vi = reinterpret_cast<float4*>(row_ptr(i));
                    float d0 = 0.f, d1 = 0.f;
                    for (int q = lane; q < nq; q += 32) {
                        const float4 av = ld_row4<SMEM>(vj + q), c = ld_row4<SMEM>(vi + q);
                        d0 = fmaf(av.x, c.x, d0); d1 = fmaf(av.y, c.y, d1);
                        d0 = fmaf(av.z, c.z, d0); d1 = fmaf(av.w, c.w, d1);
                    }
                    const float d = warp_sum(d0 + d1);
                    const float e = ljk * d;
                    for (int q = lane; q < nq; q += 32) {
                        const float4 av = ld_row4<SMEM>(vj + q);
                        float4 c = ld_row4<SMEM>(vi + q);
                        c.x = fmaf(-e, av.x, c.x); c.y = fmaf(-e, av.y, c.y);
                        c.z = fmaf(-e, av.z, c.z); c.w = fmaf(-e, av.w, c.w);
                        vi[q] = c;
                    }
                    if (i == j + 1) publish(i, kp);
                }
            }
        }
    }
    __syncthreads();
    UPD_STAMP(TL_UPD_TAIL);
    if (OVERLAP) copy_fitness();                                     // (post_rank leaves it to the end in this build)
    if (a.dbg && threadIdx.x == 0) { a.dbg[TL_UPD_FIRST_STALE] = first_stale; a.dbg[TL_UPD_LIVE] = live; }
    for (int i = first_stale + tid; i < live && RMAX >= 0; i += nthr) {   // FP64 scalar state of the recomputed rows
        const int slot = order[i];
        const double r = nj_ratio(o), am = o.M;
        const NjForm f = nj_form(r, am, (double)nv_s[i]);
        const double nj = f.nj, lj = r / (am * f.t * (f.t + 1.0));
        Njd[slot] = nj; Ljd[slot] = lj; Njf[slot] = (float)nj; Njsb[i] = (float)nj;
    }
    UPD_STAMP(TL_UPD_END);
}

// overlapped generation: k_cost must not be released before every k_update CTA holds its SM (a full SM: 512 threads x 128
// registers), otherwise k_cost's single wave takes every SM and k_update starts when k_cost ends.  One thread per instance.
__global__ void k_gate(OptDev o) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= o.B) return;
    // bounded: if k_update is not resident after 20 ms it is not going to run beside this branch (serialised launch); letting
    // k_cost go is always correct - the gate only keeps one SM free for k_update
    const long long t0 = gtime();
    for (long long spin = 0; ld_acquire_gpu(o.resident + b) == 0; ++spin) {
        __nanosleep(64);
        if ((spin & 63) == 63 && gtime() - t0 > 20000000ll) break;
    }
    o.resident[b] = 0;
}

// Co-scheduling probe (lmcma_capi.cu: probe_coschedule): two one-thread kernels on the two branches of a forked graph
// shake hands through flags[side] / flags[1 - side] within `budget_ns`; ok[side] = 1 when the partner showed up.  Run once
// per device before the overlapped generation is enabled: under a profiler or sanitizer that serialises kernels (or with
// the SMs held by someone else) the branches do not run concurrently and the handle keeps the linear PDL graph.
__global__ void k_probe(int* flags, int* ok, int side, long long budget_ns) {
    st_release_gpu(flags + side, 1);
    const long long t0 = gtime();
    int seen = 0;
    while (!(seen = ld_acquire_gpu(flags + 1 - side)) && gtime() - t0 < budget_ns) __nanosleep(100);
    ok[side] = seen ? 1 : 0;
}

// rebuild the sequence-ordered mirror from the slot-indexed state (after create / a state setter): grid = (m, B)
__global__ void __launch_bounds__(128) k_pack_pairs(OptDev o) {
    const int i = blockIdx.x, b = blockIdx.y, nq = o.ns >> 2;
    const int slot = o.t[(size_t)b * o.m + i];
    const float4* v = reinterpret_cast<const float4*>(o.V + ((size_t)b * o.m + slot) * o.ns);
    const float4* p = reinterpret_cast<const float4*>(o.P + ((size_t)b * o.m + slot) * o.ns);
    float4* dv = reinterpret_cast<float4*>(o.VPs + ((size_t)b * o.m + i) * 2 * o.ns);
    float4* dp = dv + nq;
    for (int q = threadIdx.x; q < nq; q += blockDim.x) { dv[q] = v[q]; dp[q] = p[q]; }
    if (threadIdx.x == 0) o.Njs[(size_t)b * o.m + i] = o.Njf[(size_t)b * o.m + slot];
}

}  // namespace lmcma

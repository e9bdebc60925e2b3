// k_cost.cuh — batched trajectory cost kernel.
#pragma once
#include "lmcma_common.cuh"

namespace lmcma {

// ------------------------------------------------------------------------------------------------
// k_cost — batched trajectory cost (DESIGN.md "cost model"; the reference's per-state pieces are
// ValidityChecker::isValid/clearance planner.cpp:591-631, ClearanceObjective::stateCost :655-669,
// weights :677-690).  One CTA per trajectory.
// Phase 1: one thread per segment: record {A, B-A, 1/K, len/K, first sample} into shared memory, block scan of the
//   sample counts.
// Phase 2: the flattened sample sequence is cut into 32-sample blocks, consecutive samples on consecutive lanes: they
//   are <= 1 cell apart, and the map is stored in 128-byte bricks (lmcma_layout.hpp), so one warp load touches a
//   handful of lines instead of 32 (the L1 wavefront rate, not DRAM, bounds a row-major gather).
//   2a — per-block records {bit mask of the segment ends inside the block, first segment}, written by the segment
//   threads (a segment names itself first segment of the blocks that start inside it and sets its end bit); a lane's
//   segment is then first + popc(mask below the lane): no per-lane search, no warp reduction, and no dependency
//   between blocks in the loop.  Trajectories longer than the record stage (CostArgs::cb blocks) take several rounds.
//   2b — the loop, a contiguous run of blocks per warp (drawing chunks from a shared counter was measured slower:
//   the draw costs more than the imbalance it removes).  Every sample is accumulated with the INTERIOR trapezoid weight len/K and counted as a potential collision;
//   phase 2c then takes back half a weight at k = 0 and k = K of every segment and the doubly counted joint (k = K of
//   every segment but the last) — that keeps weights, end-point tests and K itself out of the loop.  The loop is
//   software-pipelined: three block loads are in flight while the oldest one is accumulated (the kernel is bound by
//   the load-to-use latency and the L1 line rate, not by DRAM).
//   2c — the end samples, one thread per segment, after the loop: their lines were just touched (L1 / L2 hits), and
//   warps that finish the loop early do this instead of waiting at the barrier.
//   Trajectories whose waypoints all lie inside the map (always, for candidates clamped by the optimiser's box
//   bounds) take a loop without bounds tests; others take the CHECK variant (out of the map = collision).
// Phase 3: block reduction.
// The index path (t = k * (1/K); q = A + t*d; rint; bounds test) uses explicitly rounded FP32
// mul/add so that no FMA contraction can change a cell index relative to the CPU oracle.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int substeps_of(float linf) {
    if (linf >= 1.0f) return linf <= (float)KMAX_SUBSTEPS ? (int)ceilf(linf) : KMAX_SUBSTEPS;
    return 1;   // also NaN
}

constexpr int COST_MAX_WARPS = 8;
#ifndef COST_DEPTH
#define COST_DEPTH 3
#endif

// what a map load returns before it is turned into the sign-tagged reciprocal clearance
template <int STORAGE> struct RawCell { typedef float type; };
template <> struct RawCell<1> { typedef unsigned char type; };

template <int DIMS, int STORAGE, bool TRACE, int MINB = 7, bool MULTI = false>
// 8 warps per CTA, 7 CTAs per SM: 32 registers per thread, every trajectory of a 1024-wide population resident at once.
// MINB = 6 (LMCMA_B200_COST_MINB=6: 40 registers, no local-memory spill, 1.17 waves at lambda = 1024) is compiled
// beside it; measured slower on the single C2 query (33.9 vs 31.0 us, profiles/r1g_minb_compare.txt), kept for the
// many-wave batched shapes.
// MULTI (lmcma_b200_attach_cost_maps; DESIGN.md 4.7): the map of instance b is a.maps[a.map_of[b]], loaded by every CTA
// (one uniform address) instead of `mp0`, whose fields the single-map builds read from the parameter bank.  An index
// outside [0, a.map_count) gives the trajectory f = +inf, ncoll = nsamp = 0: the CTA stores that and returns before any
// barrier, without reading the table.
__global__ void __launch_bounds__(COST_MAX_WARPS * 32, MINB) k_cost(MapDev mp0, CostArgs a) {
    typedef typename RawCell<STORAGE>::type raw_t;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int W = a.W, NSEG = W + 1;
    // segment s: rec[2s] = 2-D {Ax, Ay, dx, dy} / 3-D {Ax, Ay, Az, dx};  rec[2s+1] = 2-D {invK, len/K, first sample, -} / 3-D {dy, dz, invK, len/K}
    float4* rec = reinterpret_cast<float4*>(smem_raw);
    uint2* blkrec = reinterpret_cast<uint2*>(rec + 2 * NSEG);    // a.cb per-block records {segment-end mask, first segment}
    int* segC = reinterpret_cast<int*>(blkrec + a.cb);           // 3-D first sample (NSEG entries, unused in 2-D)
    int* off = segC + NSEG;                                      // NSEG + 1 exclusive sample offsets
    float* lut = reinterpret_cast<float*>(off + NSEG + 1);       // 256 (U8 only)
    float* xs = reinterpret_cast<float*>((reinterpret_cast<size_t>(lut + (STORAGE == 1 ? 256 : 0)) + 15) & ~(size_t)15);   // the candidate row
    __shared__ float red_f[3][COST_MAX_WARPS];
    __shared__ int red_i[COST_MAX_WARPS];
    __shared__ int warp_tot[COST_MAX_WARPS];

    griddep_launch_dependents();          // k_rank may become resident as this grid drains; it waits for completion
    const int row = blockIdx.x, b = blockIdx.y;
    int mi = 0;
    if (MULTI) {
        mi = a.map_of[b];
        if ((unsigned)mi >= (unsigned)a.map_count) {              // the whole CTA leaves here: no barrier has been reached
            if (threadIdx.x == 0) {
                a.f[(size_t)b * a.f_stride + a.f_offset + row] = __int_as_float(0x7f800000);
                if (a.ncoll) a.ncoll[(size_t)b * a.inst_rows + row] = 0;
                if (a.nsamp) a.nsamp[(size_t)b * a.inst_rows + row] = 0;
            }
            return;
        }
    }
    const MapDev mp = MULTI ? a.maps[mi] : mp0;
#define COST_STAMP(k) do { if (TRACE && a.dbg && (threadIdx.x & 31) == 0) { const long long t__ = gtime(); if ((k) == 0 || (k) == 1 || (k) == 2) { if (threadIdx.x == 0) a.dbg[((size_t)blockIdx.y * gridDim.x + blockIdx.x) * 8 + (k)] = t__; } else atomicMax(reinterpret_cast<unsigned long long*>(a.dbg + ((size_t)blockIdx.y * gridDim.x + blockIdx.x) * 8 + (k)), (unsigned long long)t__); } } while (0)
    COST_STAMP(0);
    const int tid = threadIdx.x, nthr = blockDim.x, lane = tid & 31, warp = tid >> 5, nwarps = nthr >> 5;
    const float* x = a.X + ((size_t)b * a.inst_rows + row) * a.ld;
    // xs holds the whole poly-line per dimension: xs[c * (W + 2) + i], i = 0 start, 1..W the candidate's waypoints, W + 1 goal
    const int WS = W + 2;
    if (tid == 0) {
#pragma unroll
        for (int c = 0; c < DIMS; ++c) {                         // constant indices: ends0 is read from the parameter bank
            xs[c * WS] = a.ends_per_instance ? a.ends[(size_t)b * 6 + c] : a.ends0[c];
            xs[c * WS + W + 1] = a.ends_per_instance ? a.ends[(size_t)b * 6 + 3 + c] : a.ends0[3 + c];
        }
    }
    if (STORAGE == 1) for (int i = tid; i < 256; i += nthr) lut[i] = mp.lut[i];
    // first round of block records (phase 2a), zeroed ahead of the barrier below: two records per 16-byte store (a.cb is even;
    // the .y halves are written after the next barrier)
    for (int lb = tid; lb < (a.cb >> 1); lb += nthr) reinterpret_cast<uint4*>(blkrec)[lb] = make_uint4(0u, 0u, 0u, 0u);
    // the candidate row, read ONCE and coalesced (it may live in pinned host memory: lmcma_b200_cost_evaluate hands a
    // page-locked caller buffer to the kernel directly, and the row then crosses PCIe while other CTAs compute)
    {
        const int nflt = DIMS * W;
        if ((reinterpret_cast<size_t>(x) & 15) == 0 && (W & 3) == 0) {   // a float4 never straddles two dimensions
            for (int i = tid; i < (nflt >> 2); i += nthr) {
                const float4 v = reinterpret_cast<const float4*>(x)[i];
                const int e = i << 2, c = (e >= W ? 1 : 0) + (DIMS == 3 && e >= 2 * W ? 1 : 0);
                float* dst = xs + c * WS + 1 + (e - c * W);
                dst[0] = v.x; dst[1] = v.y; dst[2] = v.z; dst[3] = v.w;
            }
        } else {
#pragma unroll
            for (int c = 0; c < DIMS; ++c)
                for (int i = tid; i < W; i += nthr) xs[c * WS + 1 + i] = x[c * W + i];
        }
    }
    __syncthreads();                                             // xs (and the lut)
    COST_STAMP(1);

    const unsigned nxm1 = (unsigned)(mp.nx - 1), nym1 = (unsigned)(mp.ny - 1), nzm1 = (unsigned)(mp.nz - 1);
    const float fx1 = (float)(mp.nx - 1), fy1 = (float)(mp.ny - 1), fz1 = (float)(mp.nz - 1);
    const unsigned py = mp.py, pz = mp.pz;                       // brick pitches (lmcma_layout.hpp), formed on the host
    const float ng_coll = -mp.g_coll;
    const float* __restrict__ g32 = mp.g32;
    const unsigned char* __restrict__ q8 = mp.q8;
    const int last = NSEG - 1;

    // sample k * invK of a segment -> cell; returns false outside the map.  Round-half-even conversion == (int)rintf(q);
    // it saturates for huge |q| (-> fails the unsigned test); explicitly rounded mul / add (see the header)
    auto cell_of = [&](float tk, float ax, float ay, float az, float dx, float dy, float dz, int& ix, int& iy, int& iz) {
        ix = __float2int_rn(__fadd_rn(ax, __fmul_rn(tk, dx)));
        iy = __float2int_rn(__fadd_rn(ay, __fmul_rn(tk, dy)));
        bool inb = ((unsigned)ix <= nxm1) && ((unsigned)iy <= nym1);
        iz = 0;
        if (DIMS == 3) {
            iz = __float2int_rn(__fadd_rn(az, __fmul_rn(tk, dz)));
            inb = inb && ((unsigned)iz <= nzm1);
        }
        return inb;
    };
    auto load_raw = [&](unsigned adr) -> raw_t {
        if (STORAGE == 0) return (raw_t)__ldg(g32 + adr);
        return (raw_t)__ldg(q8 + adr);
    };
    auto value_of = [&](raw_t r) -> float { return STORAGE == 0 ? (float)r : lut[(int)r]; };   // lut is read after a barrier

    // ---- phase 1: per-segment records, sub-step counts, lengths, end samples; block scan of the sample counts ----
    const int spt = a.spt;                                       // consecutive segments per thread, ceil(NSEG / nthr): formed by the launcher
    const int s_begin = min(NSEG, tid * spt), s_end = min(NSEG, s_begin + spt);
    float len_acc = 0.f; int my_cnt = 0;
    bool safe = true;                                            // every waypoint of my segments inside the map
    const raw_t idle = (raw_t)(STORAGE == 1 ? 1 : 0);             // a free cell
    for (int s = s_begin; s < s_end; ++s) {
        float A[3], D[3]; float linf = 0.f, l2 = 0.f; bool bad = false;
        A[2] = 0.f; D[2] = 0.f;
#pragma unroll
        for (int c = 0; c < DIMS; ++c) {
            A[c] = xs[c * WS + s];
            const float Bc = xs[c * WS + s + 1];
            const float hi_c = c == 0 ? fx1 : (c == 1 ? fy1 : fz1);
            safe = safe && (A[c] >= 0.f) && (A[c] <= hi_c) && (Bc >= 0.f) && (Bc <= hi_c);
            D[c] = __fsub_rn(Bc, A[c]);
            const float ad = fabsf(D[c]);
            bad |= (ad != ad);
            if (ad > linf) linf = ad;
            l2 = fmaf(D[c], D[c], l2);
        }
        if (bad) linf = __int_as_float(0x7fc00000);
        const int K = substeps_of(linf);
        const float invK = __frcp_rn((float)K);                  // == 1.0f / (float)K, IEEE round-to-nearest
        const float len = sqrtf(l2);
        len_acc += len;
        // A segment with a non-finite end point has no sample inside the map (NaN / inf coordinates fail the
        // oracle's bounds test for every k): encode that as a finite far-away anchor so that the sample loop
        // can use integer conversion + unsigned bounds tests (NaN would convert to 0).
        bool finite = true;
#pragma unroll
        for (int c = 0; c < DIMS; ++c) finite = finite && (fabsf(A[c]) < 3.0e38f) && (fabsf(D[c]) < 3.0e38f);
        if (!finite) {
#pragma unroll
            for (int c = 0; c < DIMS; ++c) { A[c] = -1.0e9f; D[c] = 0.f; }
        }
        const float scale = len * invK;
        if (DIMS == 2) { rec[2 * s] = make_float4(A[0], A[1], D[0], D[1]); rec[2 * s + 1] = make_float4(invK, scale, 0.f, 0.f); }
        else { rec[2 * s] = make_float4(A[0], A[1], A[2], D[0]); rec[2 * s + 1] = make_float4(D[1], D[2], invK, scale); }
        off[s + 1] = K + 1;                                      // samples of this segment (rewritten below)
        my_cnt += K + 1;
    }
    int incl = my_cnt;                                           // block-wide exclusive scan of my_cnt
#pragma unroll
    for (int o2 = 1; o2 < 32; o2 <<= 1) {
        const int nb = __shfl_up_sync(0xffffffffu, incl, o2);
        if (lane >= o2) incl += nb;
    }
    if (lane == 31) warp_tot[warp] = incl;
    const bool all_safe = __syncthreads_and(safe ? 1 : 0) != 0;
    // the warps' totals: one load and two integer warp reductions (REDUX.SUM) instead of a dependent loop over shared memory
    const int wt = lane < nwarps ? warp_tot[lane] : 0;
    const int T = __reduce_add_sync(0xffffffffu, wt);
    int base = incl - my_cnt + __reduce_add_sync(0xffffffffu, lane < warp ? wt : 0);
    if (tid == 0) off[0] = 0;
    const int nblk0 = min(a.cb, (int)((unsigned)(T + 31) >> 5));    // blocks of the first round
    for (int s = s_begin; s < s_end; ++s) {
        if (DIMS == 2) rec[2 * s + 1].z = __int_as_float(base); else segC[s] = base;   // first sample of the segment
        const int f0 = base;
        base += off[s + 1]; off[s + 1] = base;
        // phase 2a of the first round, from the registers at hand (no second pass over off[], no extra barrier): segment s
        // covers samples [f0, base): it is the first segment of every block that starts inside it, and its last sample
        // sets one end bit
        for (int blk = (f0 + 31) >> 5; blk < nblk0 && (blk << 5) < base; ++blk) blkrec[blk].y = (unsigned)s;
        const int e = base - 1;
        if ((e >> 5) < nblk0) atomicOr(&blkrec[e >> 5].x, 1u << (e & 31));
    }
    __syncthreads();
    COST_STAMP(2);

    // ---- phase 2 ----
    const int nblk = (int)((unsigned)(T + 31) >> 5);
    const unsigned below = (1u << lane) - 1u;
    float clr_acc = 0.f; int coll = 0;
    // one 32-sample block: address + load issue.  bp = the block's record, tl = this lane's sample index (TAIL: clamped
    // to the last sample).  TAIL = the trajectory's last block, where the lanes past the last sample contribute nothing.
    // CHECK = bounds tests (a sample outside the map is a collision)
    auto fetch = [&](const uint2* bp, const int tl, const bool TAIL, const bool dead, const bool CHECK, raw_t& raw, float& wgt, bool& outside) {
        const uint2 br = *bp;
        const unsigned bel = TAIL ? ((1u << (tl & 31)) - 1u) : below;
        const int s = (int)br.y + __popc(br.x & bel);             // segment ends before this lane's sample
        const float4 ra = rec[2 * s];
        const float4 rb = rec[2 * s + 1];
        float invK, scale, ax = ra.x, ay = ra.y, az = 0.f, dx, dy, dz = 0.f; int cur;
        if (DIMS == 2) { invK = rb.x; scale = rb.y; cur = __float_as_int(rb.z); dx = ra.z; dy = ra.w; }
        else { dx = ra.w; dy = rb.x; dz = rb.y; invK = rb.z; scale = rb.w; az = ra.z; cur = segC[s]; }
        const int k = tl - cur;
        int ix, iy, iz;
        const bool inb = cell_of(__fmul_rn((float)k, invK), ax, ay, az, dx, dy, dz, ix, iy, iz);
        unsigned adr = brick_offset_p<DIMS, STORAGE>((unsigned)ix, (unsigned)iy, (unsigned)iz, py, pz);
        if (CHECK) adr = inb ? adr : 0u;
        raw = load_raw(adr);
        outside = CHECK && !inb;
        wgt = scale;
        if (TAIL && dead) { raw = idle; outside = false; wgt = 0.f; }
        if (TRACE) {
            if (!dead && (long long)tl < a.max_cells) a.cells[tl] = inb ? ((long long)iz * mp.ny + iy) * mp.nx + ix : -1;
        }
    };
    // |g| x weight into the clearance sum; a collision is the sign bit of g (obstacle cells and out-of-map samples
    // are negative, never -0)
    auto accumulate = [&](raw_t raw, float wgt, bool outside, const bool CHECK) {
        float g = value_of(raw);
        if (CHECK) g = outside ? ng_coll : g;
        clr_acc = fmaf(fabsf(g), wgt, clr_acc);
        coll += (int)(__float_as_uint(g) >> 31);
    };
    // blocks in flight per warp while the oldest is accumulated (COST_DEPTH, 3 unless the build says otherwise)
    constexpr int DEPTH = COST_DEPTH;
    raw_t pq[DEPTH]; float wq[DEPTH]; bool oq[DEPTH];
#pragma unroll
    for (int u = 0; u < DEPTH; ++u) { pq[u] = idle; wq[u] = 0.f; oq[u] = false; }
    // blocks [lb0, lb1) of the round that starts at block c0; the pipeline keeps running across calls
    auto run = [&](const int c0, const int lb0, const int lb1, const bool CHECK) {
        const bool has_tail = (c0 + lb1 == nblk);                 // the trajectory's last block may be partial
        const uint2* bp = blkrec + lb0;
        const uint2* const bp_full = blkrec + (has_tail ? lb1 - 1 : lb1);
        int tl = ((c0 + lb0) << 5) + lane;
#pragma unroll 1
        for (; bp + (DEPTH - 1) < bp_full; bp += DEPTH, tl += 32 * DEPTH) {   // DEPTH blocks in flight, the oldest is accumulated
#pragma unroll
            for (int u = 0; u < DEPTH; ++u) {
                raw_t r; float v; bool q;
                fetch(bp + u, tl + 32 * u, false, false, CHECK, r, v, q); accumulate(pq[u], wq[u], oq[u], CHECK); pq[u] = r; wq[u] = v; oq[u] = q;
            }
        }
#pragma unroll 1
        for (; bp < bp_full; ++bp, tl += 32) {
            raw_t r; float v; bool q;
            fetch(bp, tl, false, false, CHECK, r, v, q); accumulate(pq[0], wq[0], oq[0], CHECK);
#pragma unroll
            for (int u = 0; u + 1 < DEPTH; ++u) { pq[u] = pq[u + 1]; wq[u] = wq[u + 1]; oq[u] = oq[u + 1]; }
            pq[DEPTH - 1] = r; wq[DEPTH - 1] = v; oq[DEPTH - 1] = q;
        }
        if (has_tail) {
            raw_t r; float v; bool q;
            fetch(bp, min(tl, T - 1), true, tl >= T, CHECK, r, v, q); accumulate(pq[0], wq[0], oq[0], CHECK);
#pragma unroll
            for (int u = 0; u + 1 < DEPTH; ++u) { pq[u] = pq[u + 1]; wq[u] = wq[u + 1]; oq[u] = oq[u + 1]; }
            pq[DEPTH - 1] = r; wq[DEPTH - 1] = v; oq[DEPTH - 1] = q;
        }
    };
    for (int c0 = 0; c0 < nblk; c0 += a.cb) {
        const int nb = min(a.cb, nblk - c0);
        // 2a: block records of this round.  Segment s covers samples [off[s], off[s+1]): it is the first segment of
        // every block that starts inside it, and its last sample sets one end bit
        if (c0 > 0) {                                             // the first round's records were written in phase 1
            for (int lb = tid; lb < nb; lb += nthr) blkrec[lb].x = 0u;
            __syncthreads();
            const int r_lo = c0 << 5, r_hi = (c0 + nb) << 5;      // samples of this round
            for (int sg = s_begin; sg < s_end; ++sg) {
                const int f0 = off[sg], f1 = off[sg + 1];
                for (int blk = max((f0 + 31) >> 5, c0); blk < c0 + nb && (blk << 5) < f1; ++blk) blkrec[blk - c0].y = (unsigned)sg;
                const int e = f1 - 1;
                if (e >= r_lo && e < r_hi) atomicOr(&blkrec[(e >> 5) - c0].x, 1u << (e & 31));
            }
            __syncthreads();
        }
        // 2b: a contiguous run of blocks per warp
        // (the usual CTA has 1 / 2 / 4 / 8 warps: a shift instead of two integer divisions per warp and round)
        const bool pow2 = (nwarps & (nwarps - 1)) == 0;
        const int lg = 31 - __clz(nwarps);
        const int lb0 = pow2 ? (int)(((unsigned)warp * (unsigned)nb) >> lg) : (int)(((unsigned)warp * (unsigned)nb) / (unsigned)nwarps);
        const int lb1 = pow2 ? (int)(((unsigned)(warp + 1) * (unsigned)nb) >> lg) : (int)(((unsigned)(warp + 1) * (unsigned)nb) / (unsigned)nwarps);
        if (lb0 < lb1) { if (all_safe) run(c0, lb0, lb1, false); else run(c0, lb0, lb1, true); }
        if (c0 + a.cb < nblk) __syncthreads();                    // the stage is rebuilt
    }
#pragma unroll
    for (int u = 0; u < DEPTH; ++u) { if (all_safe) accumulate(pq[u], wq[u], oq[u], false); else accumulate(pq[u], wq[u], oq[u], true); }

    COST_STAMP(3);                                               // (max over warps) sample loop done
    // ---- 2c: the end samples (k = 0 and k = K) of my segments, by the same arithmetic as the sample loop ----
    float corr_clr = 0.f; int corr_coll = 0;
    for (int sg = s_begin; sg < s_end; ++sg) {
        const float4 ra = rec[2 * sg];
        const float4 rb = rec[2 * sg + 1];
        float invK, scale, ax = ra.x, ay = ra.y, az = 0.f, dx, dy, dz = 0.f;
        if (DIMS == 2) { invK = rb.x; scale = rb.y; dx = ra.z; dy = ra.w; }
        else { dx = ra.w; dy = rb.x; dz = rb.y; invK = rb.z; scale = rb.w; az = ra.z; }
        const int K = off[sg + 1] - off[sg] - 1;
        int ix, iy, iz;
        const bool in0 = cell_of(__fmul_rn(0.f, invK), ax, ay, az, dx, dy, dz, ix, iy, iz);
        const raw_t e0 = load_raw(in0 ? brick_offset_p<DIMS, STORAGE>((unsigned)ix, (unsigned)iy, (unsigned)iz, py, pz) : 0u);
        const bool inK = cell_of(__fmul_rn((float)K, invK), ax, ay, az, dx, dy, dz, ix, iy, iz);
        const raw_t eK = load_raw(inK ? brick_offset_p<DIMS, STORAGE>((unsigned)ix, (unsigned)iy, (unsigned)iz, py, pz) : 0u);
        const float g0 = in0 ? value_of(e0) : ng_coll, gK = inK ? value_of(eK) : ng_coll;
        corr_clr = fmaf(0.5f * scale, fabsf(g0) + fabsf(gK), corr_clr);
        corr_coll += (sg != last && gK < 0.f) ? 1 : 0;
    }

    COST_STAMP(4);                                               // (max over warps) end samples done
    // ---- phase 3: block reduction ----
    len_acc = warp_sum(len_acc);
    clr_acc = warp_sum(clr_acc);
    corr_clr = warp_sum(corr_clr);
    coll = warp_sum_i(coll - corr_coll);
    if (lane == 0) { red_f[0][warp] = len_acc; red_f[1][warp] = clr_acc; red_f[2][warp] = corr_clr; red_i[warp] = coll; }
    __syncthreads();
    if (tid == 0) {
        float L = 0.f, C = 0.f, Cc = 0.f; int NC = 0;
        for (int w2 = 0; w2 < nwarps; ++w2) { L += red_f[0][w2]; C += red_f[1][w2]; Cc += red_f[2][w2]; NC += red_i[w2]; }
        const float f = fmaf(a.w_col, (float)NC, fmaf(a.w_clr, C - Cc, a.w_len * L));
        a.f[(size_t)b * a.f_stride + a.f_offset + row] = f;
        if (a.ncoll) a.ncoll[(size_t)b * a.inst_rows + row] = NC;
        if (a.nsamp) a.nsamp[(size_t)b * a.inst_rows + row] = T;
    }
    COST_STAMP(5);
#undef COST_STAMP
}

}  // namespace lmcma

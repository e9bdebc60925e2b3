// k_rank.cuh — ranking + recombination partial sums of LMCMA::update (lmcma.cpp:315-326, 393-411).
//
// grid = (RS, B): RS row slices per optimiser instance.  Every CTA computes the ranks of its slice's
// candidates by counting (myqsort/compare, lmcma.cpp:84-104: stable ascending order, ties keep the lower id,
// -0 == +0, NaN last) together with the pair count S of the merged 2*lambda ranking of the step-size rule,
// and the slice's weighted partial sum of d = x - xmean (OptDev::D).  k_update (k_update.cuh) folds the partials.
// Split-population mode (RANK_PACK): the last CTA of an instance to finish — fence + atomic ticket, no CTA
// ever waits on another — folds the partials into the all-gather payload.
// Every CTA also adds one ticket to OptDev::rank_ticket after its last store: the overlapped generation's k_update is not
// a stream successor of this grid and waits for RS tickets (RANK_KEEP_FLAGS: the hand-over flags are then k_update's to
// reset, and the dependent grid is the sampler).
#pragma once
#include "lmcma_common.cuh"
#include "lmcma_plan.hpp"

namespace lmcma {

enum { RANK_PLAIN = 0, RANK_PACK = 1, RANK_KEEP_FLAGS = 2 };   // bit 1: the hand-over flags belong to a concurrently running k_update

// ------------------------------------------------------------------------------------------------
// Large unsplit populations (lambda > TELL_FTILE): counting costs lambda^2 compares (1.4 ms at lambda = 65536, half of
// the generation).  k_rank_tiles sorts every TELL_FTILE-candidate tile of the fitness by (value, id) — the reference's
// order: ascending, ties keep the lower id, -0 == +0, NaN as +inf — and k_rank then takes a candidate's rank as the sum
// over the tiles of a binary search: tiles in front of its own count "<=", tiles behind it "<", its own tile contributes
// its position in the sorted tile.  Exactly the rank the counting pass produces; the pair count of the step-size rule
// becomes a binary search in the previous generation's sorted fitness.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long rank_key(float f, unsigned id) {
    f = canon_fitness(f) + 0.0f;                                  // NaN -> +inf, -0 -> +0
    unsigned u = __float_as_uint(f);
    u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);              // order-preserving map of the float onto unsigned
    return ((unsigned long long)u << 32) | id;
}
// grid = (tiles, B), 1024 threads: bitonic sort of one tile in shared memory (32 KB of 64-bit keys)
__global__ void __launch_bounds__(1024) k_rank_tiles(OptDev o, const float* __restrict__ f_all) {
    __shared__ unsigned long long key[TELL_FTILE];
    griddep_wait();                                               // the fitness is the predecessor's output
    griddep_launch_dependents();
    const int b = blockIdx.y, base = blockIdx.x * TELL_FTILE, cnt = min(TELL_FTILE, o.lambda - base);
    const float* cur = f_all + (size_t)b * o.lambda + base;
    for (int j = threadIdx.x; j < TELL_FTILE; j += blockDim.x) key[j] = j < cnt ? rank_key(cur[j], (unsigned)j) : ~0ull;
    __syncthreads();
    for (int k = 2; k <= TELL_FTILE; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int t = threadIdx.x; t < TELL_FTILE / 2; t += blockDim.x) {
                const int lo = ((t & ~(j - 1)) << 1) | (t & (j - 1)), hi = lo | j;    // pair (lo, hi = lo + j)
                const bool up = (lo & k) == 0;
                const unsigned long long a = key[lo], c = key[hi];
                if ((a > c) == up) { key[lo] = c; key[hi] = a; }
            }
            __syncthreads();
        }
    float* ts = o.tile_sorted + (size_t)b * o.lambda + base;
    int* tp = o.tile_pos + (size_t)b * o.lambda + base;
    for (int j = threadIdx.x; j < cnt; j += blockDim.x) {
        const unsigned long long kk = key[j];
        unsigned u = (unsigned)(kk >> 32);
        u = (u & 0x80000000u) ? (u & 0x7fffffffu) : ~u;
        ts[j] = __uint_as_float(u);
        tp[(unsigned)kk] = j;
    }
}
// number of entries of the ascending array a[0, cnt) that are < v (STRICT) or <= v
template <bool STRICT>
__device__ __forceinline__ int count_below(const float* a, int cnt, float v) {
    int lo = 0, hi = cnt;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        const float x = a[mid];
        if (STRICT ? (x < v) : (x <= v)) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// ------------------------------------------------------------------------------------------------
// ranks + partial sums of one slice
// ------------------------------------------------------------------------------------------------
// What a CTA can do BEFORE the fitness exists (k_rank is resident while k_cost drains): stage the previous generation's
// fitness (written by the last generation's k_update) when one tile holds it, and pull the slice's rows of d = x - xmean
// towards L2 — after an L2 flush both would otherwise be HBM round trips between the ranks and the partial sums.
__device__ __forceinline__ void tell_prologue(const OptDev& o, int b, int rs, unsigned char* smem_raw) {
    const int tid = threadIdx.x, nthr = blockDim.x, lambda = o.lambda;
    if (lambda <= TELL_FTILE) {
        float* prev_s = reinterpret_cast<float*>(smem_raw) + o.rank_ftile;
        const float* prev = (o.tile_sorted ? o.prev_sorted : o.prev_fit) + (size_t)b * lambda;
        const int cnt4 = (lambda + 3) & ~3;
        for (int j = tid; j < cnt4; j += nthr) prev_s[j] = j < lambda ? prev[j] : __int_as_float(0x7f800000);
    }
    if (o.B == 1) {                                                   // one query: latency; a batch is throughput-bound and only mu of its rows are read
        const int rows_per = (o.pop_count + o.RS - 1) / o.RS;
        const int r0 = rs * rows_per, r1 = min(o.pop_count, r0 + rows_per);
        const char* d0 = reinterpret_cast<const char*>(o.D + (size_t)r0 * o.ns);
        const int bytes = (r1 - r0) * o.ns * (int)sizeof(float);     // a slice: at most TELL_MAX_ROWS rows
        for (int ofs = tid * 128; ofs < bytes; ofs += nthr * 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(d0 + ofs));
    }
}

__device__ __forceinline__ void tell_phase_a(const OptDev& o, const float* __restrict__ f_all, int b, int rs,
                                             unsigned char* smem_raw, const bool prev_staged) {
    const int tid = threadIdx.x, nthr = blockDim.x, lane = tid & 31;
    const int lambda = o.lambda;
    const int rows_per = (o.pop_count + o.RS - 1) / o.RS;
    const int r0 = rs * rows_per, r1 = min(o.pop_count, r0 + rows_per), nrows = max(0, r1 - r0);

    // the staging tiles hold TELL_FTILE values, or just lambda (rounded up to 4) for small populations: a batch of small
    // instances is then not limited to four CTAs per SM by 32 KB tiles it does not use (OptDev::rank_ftile, set at create)
    const int ftile = o.rank_ftile;
    float* cur_s = reinterpret_cast<float*>(smem_raw);               // ftile
    float* prev_s = cur_s + ftile;                                   // ftile
    int* rk_s = reinterpret_cast<int*>(prev_s + ftile);              // TELL_MAX_ROWS ranks of the slice's rows
    int* sel_row = rk_s + TELL_MAX_ROWS;                             // compacted selected rows (rank < mu)
    float* sel_w = reinterpret_cast<float*>(sel_row + TELL_MAX_ROWS);
    float4* red = reinterpret_cast<float4*>(sel_w + TELL_MAX_ROWS);  // 7 x 128 cross-group reduction
    __shared__ int sh_nsel;
    __shared__ unsigned long long sh_S;

#define RNK_STAMP(k) do { if (o.dbg && threadIdx.x == 0 && blockIdx.x == 0 && b == 0) o.dbg[k] = gtime(); } while (0)
    RNK_STAMP(TL_RANK_START);
    const bool sorted = o.tile_sorted != nullptr;                    // sorted-tile mode (k_rank_tiles ran just before this grid)
    const float* cur = f_all + (size_t)b * lambda;
    const float* cur_stage = sorted ? o.tile_sorted + (size_t)b * lambda : cur;
    const float* prev = (sorted ? o.prev_sorted : o.prev_fit) + (size_t)b * lambda;
    if (tid == 0) sh_S = 0ull;

    // threads per row: a power of two <= 32 so that a row's partial counts fold with warp shuffles
    int tpr = 32;
    while (tpr > 1 && (nthr / tpr) < nrows) tpr >>= 1;
    const int rows_par = nthr / tpr, sub = tid % tpr, grp = tid / tpr;

    const int npass = (nrows + rows_par - 1) / rows_par;
    // counts for (up to) npass rows per thread group are kept in registers across the fitness tiles when
    // npass == 1 (the common shape); otherwise the tiles are re-staged per pass (lambda > 4096 only).
    for (int pass = 0; pass < npass; ++pass) {
        const int il = r0 + pass * rows_par + grp;                   // local row
        const bool valid = (pass * rows_par + grp) < nrows;
        const int i = o.pop_offset + il;                             // global candidate id
        const float ki = valid ? canon_fitness(cur[i]) : 0.f;
        int c_lt = 0; unsigned long long p_lt = 0;
        for (int base = 0; base < lambda; base += TELL_FTILE) {
            const int cnt = min(TELL_FTILE, lambda - base), cnt4 = (cnt + 3) & ~3;
            __syncthreads();                                         // previous tile fully consumed
            for (int j = tid; j < cnt4; j += nthr) {
                const bool in = j < cnt;
                cur_s[j] = in ? canon_fitness(cur_stage[base + j]) : __int_as_float(0x7f800000);
                if (!prev_staged) prev_s[j] = in ? prev[base + j] : __int_as_float(0x7f800000);   // else: tell_prologue
            }
            __syncthreads();
            if (valid && sorted) {
                // both staged tiles are ascending: binary searches, the tiles shared out over the row's tpr threads
                const int tile = base / TELL_FTILE;
                if ((tile % tpr) == sub) {
                    const int own = i / TELL_FTILE;
                    c_lt += tile < own ? count_below<false>(cur_s, cnt, ki)
                                       : (tile > own ? count_below<true>(cur_s, cnt, ki) : o.tile_pos[(size_t)b * lambda + i]);
                    p_lt += (unsigned long long)count_below<true>(prev_s, cnt, ki);
                }
            } else if (valid) {
                int pl = 0;
                for (int j = sub * 4; j < cnt4; j += tpr * 4) {
                    const float4 kj = *reinterpret_cast<const float4*>(cur_s + j);
                    const float4 pj = *reinterpret_cast<const float4*>(prev_s + j);
                    const int jg = base + j;
                    // ties keep the lower id first: j < i counts on "<=", j >= i on "<" (j == i compares equal)
                    if (jg + 3 < i) {
                        c_lt += (kj.x <= ki) + (kj.y <= ki) + (kj.z <= ki) + (kj.w <= ki);
                    } else if (jg >= i) {
                        c_lt += (kj.x < ki) + (kj.y < ki) + (kj.z < ki) + (kj.w < ki);
                    } else {
                        c_lt += (kj.x < ki) || (kj.x == ki && jg < i);
                        c_lt += (kj.y < ki) || (kj.y == ki && jg + 1 < i);
                        c_lt += (kj.z < ki) || (kj.z == ki && jg + 2 < i);
                        c_lt += (kj.w < ki) || (kj.w == ki && jg + 3 < i);
                    }
                    pl += (pj.x < ki) + (pj.y < ki) + (pj.z < ki) + (pj.w < ki);
                }
                p_lt += (unsigned long long)pl;
            }
        }
        // fold over the tpr lanes of the row (groups are aligned inside a warp)
        unsigned plo = (unsigned)p_lt, phi = (unsigned)(p_lt >> 32);
        for (int ofs = tpr >> 1; ofs > 0; ofs >>= 1) {
            c_lt += __shfl_xor_sync(0xffffffffu, c_lt, ofs);
            const unsigned l2 = __shfl_xor_sync(0xffffffffu, plo, ofs), h2 = __shfl_xor_sync(0xffffffffu, phi, ofs);
            const unsigned long long a = (((unsigned long long)phi << 32) | plo) + (((unsigned long long)h2 << 32) | l2);
            plo = (unsigned)a; phi = (unsigned)(a >> 32);
        }
        if (valid && sub == 0) {
            o.rank[(size_t)b * lambda + i] = c_lt;
            o.arindex[(size_t)b * lambda + c_lt] = i;
            o.fit_sorted[(size_t)b * lambda + c_lt] = ki;
            rk_s[pass * rows_par + grp] = c_lt;
            atomicAdd(&sh_S, ((unsigned long long)phi << 32) | plo);   // integer: order-independent
        }
    }
    __syncthreads();
    RNK_STAMP(TL_RANK_RANKED);
    if (tid == 0 && sh_S) atomicAdd(o.S_count + b, sh_S);

    // ---- compact the selected rows (rank < mu) in row order: deterministic summation order ----
    if (tid < 32) {
        int nsel = 0;
        for (int basei = 0; basei < nrows; basei += 32) {
            const int r = basei + lane;
            const int rk = (r < nrows) ? rk_s[r] : o.mu;
            const bool s = rk < o.mu;
            const unsigned bal = __ballot_sync(0xffffffffu, s);
            if (s) {
                const int pos = nsel + __popc(bal & ((1u << lane) - 1u));
                sel_row[pos] = r0 + r;
                sel_w[pos] = o.w[rk];
            }
            nsel += __popc(bal);
        }
        if (lane == 0) sh_nsel = nsel;
    }
    __syncthreads();
    RNK_STAMP(TL_RANK_COMPACTED);
    const int nsel = sh_nsel;

    // ---- weighted partial sums of d = x - xmean: 128 float4 columns x (nthr/128) row groups ----
    const int nq = o.ns >> 2, ngrp = nthr >> 7, tq = tid & 127, g = tid >> 7;
    float* part = o.partial + ((size_t)b * o.RS + rs) * o.ns;
    for (int q0 = 0; q0 < nq; q0 += 128) {
        const int q = q0 + tq;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        if (q < nq) {
            for (int k = g; k < nsel; k += 4 * ngrp) {               // up to 4 rows in flight per thread
                float w[4]; float4 x[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int kk = k + u * ngrp;
                    const bool on = kk < nsel;
                    w[u] = on ? sel_w[kk] : 0.f;
                    x[u] = on ? reinterpret_cast<const float4*>(o.D + ((size_t)b * o.pop_count + sel_row[kk]) * o.ns)[q] : make_float4(0.f, 0.f, 0.f, 0.f);
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    acc.x = fmaf(w[u], x[u].x, acc.x);
                    acc.y = fmaf(w[u], x[u].y, acc.y);
                    acc.z = fmaf(w[u], x[u].z, acc.z);
                    acc.w = fmaf(w[u], x[u].w, acc.w);
                }
            }
        }
        RNK_STAMP(TL_RANK_GATHERED);
        if (g > 0) red[(g - 1) * 128 + tq] = acc;
        __syncthreads();
        if (g == 0 && q < nq) {
            for (int gg = 0; gg + 1 < ngrp; ++gg) { const float4 t = red[gg * 128 + tq]; acc.x += t.x; acc.y += t.y; acc.z += t.z; acc.w += t.w; }
            reinterpret_cast<float4*>(part)[q] = acc;
        }
        __syncthreads();
    }
    RNK_STAMP(TL_RANK_STORED);
#undef RNK_STAMP
}

// A_PACK tail (split mode): fold the RS local partials and the local S count into the all-gather payload
__device__ __forceinline__ void tell_pack_payload(const OptDev& o, float* __restrict__ payload, int b) {
    float* pay = payload + (size_t)b * (o.ns + 4);
    for (int e = threadIdx.x; e < o.ns; e += blockDim.x) {
        float acc = 0.f;
        for (int rs = 0; rs < o.RS; ++rs) acc += __ldcg(o.partial + ((size_t)b * o.RS + rs) * o.ns + e);
        pay[e] = acc;
    }
    if (threadIdx.x == 0) {
        const unsigned long long S = atomicExch(o.S_count + b, 0ull);
        pay[o.ns] = __uint_as_float((unsigned)S);
        pay[o.ns + 1] = __uint_as_float((unsigned)(S >> 32));
        pay[o.ns + 2] = 0.f; pay[o.ns + 3] = 0.f;
    }
}


template <int MAXT>
__global__ void __launch_bounds__(MAXT, 2) k_rank(OptDev o, const float* __restrict__ f_all, int mode, float* __restrict__ payload) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ int sh_last;
    // Launched as a programmatic dependent of k_cost inside the fused generation.  The trigger for k_update comes AFTER
    // this kernel's own wait: k_update's prologue reads the fitness, so it may only start once k_cost has completed
    // (its prologue does not depend on THIS kernel, see k_update.cuh).
    const bool prev_staged = o.lambda <= TELL_FTILE;              // one tile, one pass: staged once, ahead of the wait
    tell_prologue(o, blockIdx.y, blockIdx.x, smem_raw);
    griddep_wait();
    // The dependent is released here, as soon as the fitness is there.  In the overlapped generation and tell_all
    // (RANK_KEEP_FLAGS) it is k_sample, which then works through the pairs k_update has already finished while this grid
    // ranks (its CTAs share SMs with this grid: the ranks arrive ~1 us later, the sampler is done 8 us earlier)
    griddep_launch_dependents();
    const int b = blockIdx.y;
    // the hand-over flags of this generation's k_update -> k_sample (both start after this grid has completed)
    if (blockIdx.x == 0 && !(mode & RANK_KEEP_FLAGS)) for (int i = threadIdx.x; i < progress_len(o.m); i += blockDim.x) progress_flags(o.progress, o.m, b)[i] = 0;
    tell_phase_a(o, f_all, b, blockIdx.x, smem_raw, prev_staged);
    // one ticket per CTA once its ranks / partial sums are stored: the overlapped generation's k_update (not a stream
    // successor of this grid) waits for RS of them; every k_update resets the counter
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        atomicAdd(o.rank_ticket + b, 1u);
        if (o.dbg && b == 0 && blockIdx.x == gridDim.x - 1) o.dbg[TL_RANK_LAST_SLICE] = gtime();
    }
    if (!(mode & RANK_PACK)) return;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned ticket = atomicAdd(o.done_count + b, 1u);
        sh_last = (ticket == (unsigned)(gridDim.x - 1)) ? 1 : 0;
        if (sh_last) o.done_count[b] = 0u;
    }
    __syncthreads();
    if (!sh_last) return;
    __threadfence();
    tell_pack_payload(o, payload, b);
}

}  // namespace lmcma

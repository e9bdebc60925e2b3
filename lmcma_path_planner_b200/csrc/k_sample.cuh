// k_sample.cuh — offspring sampling kernel.
#pragma once
#include "lmcma_common.cuh"
#include "lmcma_plan.hpp"

namespace lmcma {

// Sum v[g] over the 32 lanes for 8 values with 9 shuffles instead of 40: three exchange-and-halve stages
// (each lane gives away the half of the values it will not own), then two butterfly stages.  On return
// every lane holds the total of value p = lane >> 2 & 7, i.e. value g lives on lanes 4g .. 4g+3.
__device__ __forceinline__ float reduce_scatter8(const float (&v)[SAMPLE_G], int lane) {
    const bool h16 = lane & 16, h8 = lane & 8, h4 = lane & 4;
    float a[4], b[2];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const float send = h16 ? v[k] : v[k + 4], keep = h16 ? v[k + 4] : v[k];
        a[k] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
    }
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        const float send = h8 ? a[k] : a[k + 2], keep = h8 ? a[k + 2] : a[k];
        b[k] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
    }
    const float send = h4 ? b[0] : b[1], keep = h4 ? b[1] : b[0];
    float c = keep + __shfl_xor_sync(0xffffffffu, send, 4);
    c += __shfl_xor_sync(0xffffffffu, c, 2);
    c += __shfl_xor_sync(0xffffffffu, c, 1);
    return c;
}

// ------------------------------------------------------------------------------------------------
// k_sample — LMCMA::sample + computeAz + applyBoundaries (lmcma.cpp:301-311, 431-447, 220-230) for
// all offspring at once.  One CTA per tile of (blockDim/32)*RB offspring rows of one instance; the
// live (v_j, pc_j) pairs are streamed through shared memory in sequence order by 1-D bulk async
// copies (double-buffered, mbarrier-tracked); each warp keeps RB rows of z and Az in registers,
// lanes own float4 column slots (lane + 32*i).
//
// Pairs are processed in groups of 8.  All dots are against the ORIGINAL z (lmcma.cpp:441-443), so the
// 8*RB dot products of a group are independent FMA chains and are summed over the lanes with one
// reduce-scatter.  The ordered recurrence Az <- M*Az + d_j*pc_j (lmcma.cpp:444-445) is unrolled over a
// group as  Az <- M^8 * (Az + sum_g (d_g * M^-(g+1)) * pc_g): the same value in exact arithmetic, one
// FMA per element and pair instead of a multiply and an FMA.
// ------------------------------------------------------------------------------------------------

// The deviate v of float4 column q of local row `row` of instance b, whose offset in Z / Zc is roff: the prior's L z
// (k_prior has formed it), the generator's (recorded into Z when Z is kept), or the injected Z.
__device__ __forceinline__ void sample_deviate4(const OptDev& o, int b, int row, size_t roff, int q, int itr, int epoch, float4& v) {
    if (o.Zc) {
        v = reinterpret_cast<const float4*>(o.Zc + roff)[q];
    } else if (o.rng_mode == 0) {
        philox_deviate4(o, b, row, q, itr, epoch, v);
        if (o.Z) reinterpret_cast<float4*>(o.Z + roff)[q] = v;
    } else {
        v = reinterpret_cast<const float4*>(o.Z + roff)[q];
    }
}

// The stage ring of the samplers: `nstages` stages of kc pairs {v, pc} (2 ns floats each) in shared memory, one mbarrier
// per stage.  Thread 0 initialises it.
__device__ __forceinline__ void init_stages(unsigned long long* bars, int nstages) {
    for (int s2 = 0; s2 < nstages; ++s2) mbar_init(&bars[s2], 1);
    fence_barrier_init();
}
// One thread: chunk c of the first npairs pairs of the sequence-ordered mirror vps, pairs [c kc, min((c + 1) kc, npairs)),
// into stage c % nstages.  The pairs of a chunk are one contiguous block of the mirror: ONE bulk async copy.
__device__ __forceinline__ void request_stage(float* stage_base, size_t stage_floats, unsigned long long* bars, int nstages,
                                              const float* vps, int ns, int kc, int c, int npairs) {
    const int st = c % nstages;
    const int k0 = c * kc, cnt = min(kc, npairs - k0);
    const unsigned bytes = (unsigned)(cnt * 2 * ns * sizeof(float));
    mbar_expect_tx(&bars[st], bytes);
    bulk_g2s(stage_base + st * stage_floats, vps + (size_t)k0 * 2 * ns, bytes, &bars[st]);
}

// Element c of a float4 column of a candidate that starts at element e: x = xmean + sigma * Az in FP64, clamp lo then hi
// (lmcma.cpp:307-310, 222-229); a padding element (e + c >= n) gets 0.  Gives the candidate (FP32) and its offset from the
// mean d = x - xmean, formed in FP64 and rounded once (see OptDev::D).
__device__ __forceinline__ void finish_element(double mean, double sigma, float az, float lo, float hi, int e, int c, int n,
                                               float& x, float& d) {
    double x64 = mean + sigma * (double)az;
    float xf = (float)x64;
    if (xf < lo) { xf = lo; x64 = (double)lo; }    // max(x, lo) then min(x, hi), lmcma.cpp:222-229
    if (xf > hi) { xf = hi; x64 = (double)hi; }
    const bool pad = e + c >= n;
    x = pad ? 0.f : xf;
    d = pad ? 0.f : (float)(x64 - mean);
}

// The candidate's float4 column q; lo / hi are padded to ns with -FLT_MAX / +FLT_MAX.  Writes the candidate and d.
__device__ __forceinline__ void sample_finish(const OptDev& o, const double* __restrict__ xm, double sigma, float4 az, int q,
                                              float* __restrict__ xrow, float* __restrict__ drow, float* __restrict__ hrow = nullptr) {
    const double2 m01 = reinterpret_cast<const double2*>(xm)[2 * q];
    const double2 m23 = reinterpret_cast<const double2*>(xm)[2 * q + 1];
    float4 lo4 = make_float4(-3.4e38f, -3.4e38f, -3.4e38f, -3.4e38f), hi4 = make_float4(3.4e38f, 3.4e38f, 3.4e38f, 3.4e38f);
    if (o.lo) lo4 = reinterpret_cast<const float4*>(o.lo)[q];
    if (o.hi) hi4 = reinterpret_cast<const float4*>(o.hi)[q];
    const double mm[4] = {m01.x, m01.y, m23.x, m23.y};
    const float aa[4] = {az.x, az.y, az.z, az.w}, ll[4] = {lo4.x, lo4.y, lo4.z, lo4.w}, hh[4] = {hi4.x, hi4.y, hi4.z, hi4.w};
    float xx[4], dd[4];
    const int e = q * 4;
#pragma unroll
    for (int c = 0; c < 4; ++c) finish_element(mm[c], sigma, aa[c], ll[c], hh[c], e, c, o.n, xx[c], dd[c]);
    reinterpret_cast<float4*>(xrow)[q] = make_float4(xx[0], xx[1], xx[2], xx[3]);
    reinterpret_cast<float4*>(drow)[q] = make_float4(dd[0], dd[1], dd[2], dd[3]);
    if (hrow) __stcs(reinterpret_cast<float4*>(hrow) + q, make_float4(xx[0], xx[1], xx[2], xx[3]));   // host mirror (OptDev::Xh)
}

// SPEC: full groups of 8 pairs run a copy of the two group loops without the per-pair `g < gcnt` predicates
template <int NV, int RB, int MAXT, bool SPEC = false>
__global__ void __launch_bounds__(MAXT) k_sample(OptDev o, int kc /* pairs per stage, multiple of 8 */, int nstages) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int b = blockIdx.y;
    if (o.only && o.only[b] == 0) return;                     // an instance the reset leaves alone (OptDev::only)
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const int ns = o.ns, nq = ns >> 2;
    float* stage_base = reinterpret_cast<float*>(smem_raw);
    const size_t stage_floats = (size_t)kc * 2 * ns;
    unsigned long long* bars = reinterpret_cast<unsigned long long*>(stage_base + (size_t)nstages * stage_floats);
    float* nj_s = reinterpret_cast<float*>(bars + SAMPLE_MAX_STAGES);   // Nj of the live pairs, in sequence order (padded to 8)
    if (threadIdx.x == 0) init_stages(bars, nstages);
    // launched as a programmatic dependent of k_update: resident early, but every input is k_update's output
    griddep_wait();
    const Scalars sc = o.sc[b];
    const int live = sc.live;
    const int nchunks = (live + kc - 1) / kc;
    const float* vps = o.VPs + (size_t)b * o.m * 2 * ns;
    auto issue = [&](int c) { request_stage(stage_base, stage_floats, bars, nstages, vps, ns, kc, c, live); };   // thread 0
    if (threadIdx.x == 0)
        for (int c = 0; c < nchunks && c < nstages; ++c) issue(c);
    const int live8 = (live + SAMPLE_G - 1) & ~(SAMPLE_G - 1);
    for (int k = threadIdx.x; k < live8; k += blockDim.x) nj_s[k] = (k < live) ? o.Njs[(size_t)b * o.m + k] : 0.f;
    // (nj_s is first read after the __syncthreads below)

    // ---- load / generate z for this warp's RB rows ----
    const int row0 = (blockIdx.x * nwarps + warp) * RB;       // local row index
    float4 z[RB][NV], az[RB][NV];
#pragma unroll
    for (int r = 0; r < RB; ++r) {
        const int row = row0 + r;
        const bool rv = row < o.pop_count;
        const size_t roff = ((size_t)b * o.pop_count + (rv ? row : 0)) * ns;
#pragma unroll
        for (int i = 0; i < NV; ++i) {
            const int q = lane + 32 * i;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (rv && q < nq) sample_deviate4(o, b, row, roff, q, sc.itr, sc.epoch, v);
            z[r][i] = v;
            az[r][i] = v;
        }
    }

    // per-lane constants of the unrolled recurrence: this lane owns pair p = (lane >> 2) & 7 of every group
    const float Mf = (float)o.M, Minv = 1.0f / Mf;
    float M8 = 1.0f;                                           // M^8
#pragma unroll
    for (int c = 0; c < SAMPLE_G; ++c) M8 *= Mf;
    const int p_lane = (lane >> 2) & 7;
    float minv_lane = Minv;                                    // M^-(p+1)
    for (int c = 0; c < p_lane; ++c) minv_lane *= Minv;

    __syncthreads();                          // nj_s
    for (int c = 0; c < nchunks; ++c) {
        const int st = c % nstages;
        mbar_wait(&bars[st], (unsigned)((c / nstages) & 1));
        const float* sb = stage_base + st * stage_floats;
        const int k0 = c * kc, cnt = min(kc, live - k0);
        for (int k = 0; k < cnt; k += SAMPLE_G) {
            const int gcnt = min(SAMPLE_G, cnt - k);           // pairs in this group (warp-uniform)
            // ---- 8*RB dot products against the original z ----
            float d[RB][SAMPLE_G];
#pragma unroll
            for (int r = 0; r < RB; ++r)
#pragma unroll
                for (int g = 0; g < SAMPLE_G; ++g) d[r][g] = 0.f;
            auto dots = [&](auto full_c) {
                constexpr bool FULL = decltype(full_c)::value;
#pragma unroll
                for (int i = 0; i < NV; ++i) {
                    const int q = lane + 32 * i;
                    if (q < nq) {
#pragma unroll
                        for (int g = 0; g < SAMPLE_G; ++g) {
                            if (FULL || g < gcnt) {
                                const float4 v = reinterpret_cast<const float4*>(sb + (size_t)(2 * (k + g)) * ns)[q];
#pragma unroll
                                for (int r = 0; r < RB; ++r) {
                                    d[r][g] = fmaf(v.x, z[r][i].x, d[r][g]);
                                    d[r][g] = fmaf(v.y, z[r][i].y, d[r][g]);
                                    d[r][g] = fmaf(v.z, z[r][i].z, d[r][g]);
                                    d[r][g] = fmaf(v.w, z[r][i].w, d[r][g]);
                                }
                            }
                        }
                    }
                }
            };
            if (SPEC && gcnt == SAMPLE_G) dots(std::true_type()); else dots(std::false_type());
            // ---- lane-sum, scale: c_g = Nj_g * (v_g . z) * M^-(g+1); broadcast to every lane ----
            const float scale_lane = (p_lane < gcnt) ? nj_s[k0 + k + p_lane] * minv_lane : 0.f;
            float w[RB][SAMPLE_G];
#pragma unroll
            for (int r = 0; r < RB; ++r) {
                const float tot = reduce_scatter8(d[r], lane) * scale_lane;
#pragma unroll
                for (int g = 0; g < SAMPLE_G; ++g) w[r][g] = __shfl_sync(0xffffffffu, tot, 4 * g);
            }
            // ---- Az <- M^gcnt * (Az + sum_g c_g * pc_g) ----
            float mg = M8;
            if (gcnt < SAMPLE_G) { mg = 1.0f; for (int c2 = 0; c2 < gcnt; ++c2) mg *= Mf; }
            auto recur = [&](auto full_c) {
                constexpr bool FULL = decltype(full_c)::value;
#pragma unroll
                for (int i = 0; i < NV; ++i) {
                    const int q = lane + 32 * i;
                    if (q < nq) {
#pragma unroll
                        for (int g = 0; g < SAMPLE_G; ++g) {
                            if (FULL || g < gcnt) {
                                const float4 p = reinterpret_cast<const float4*>(sb + (size_t)(2 * (k + g) + 1) * ns)[q];
#pragma unroll
                                for (int r = 0; r < RB; ++r) {
                                    az[r][i].x = fmaf(w[r][g], p.x, az[r][i].x);
                                    az[r][i].y = fmaf(w[r][g], p.y, az[r][i].y);
                                    az[r][i].z = fmaf(w[r][g], p.z, az[r][i].z);
                                    az[r][i].w = fmaf(w[r][g], p.w, az[r][i].w);
                                }
                            }
                        }
#pragma unroll
                        for (int r = 0; r < RB; ++r) { az[r][i].x *= mg; az[r][i].y *= mg; az[r][i].z *= mg; az[r][i].w *= mg; }
                    }
                }
            };
            if (SPEC && gcnt == SAMPLE_G) recur(std::true_type()); else recur(std::false_type());
        }
        if (c + nstages < nchunks) {
            __syncthreads();                  // every warp is done with stage st
            if (threadIdx.x == 0) issue(c + nstages);
        }
    }

    // ---- x = xmean + sigma * Az, clamp lo then hi (lmcma.cpp:307-310, 222-229) ----
    const double* xm = o.xmean + (size_t)b * ns;
#pragma unroll
    for (int r = 0; r < RB; ++r) {
        const int row = row0 + r;
        if (row >= o.pop_count) continue;
        float* xrow = o.X + ((size_t)b * o.pop_count + row) * ns;
        float* drow = o.D + ((size_t)b * o.pop_count + row) * ns;
        float* hrow = o.Xh ? o.Xh + ((size_t)b * o.pop_count + row) * ns : nullptr;
#pragma unroll
        for (int i = 0; i < NV; ++i) {
            const int q = lane + 32 * i;
            if (q < nq) sample_finish(o, xm, sc.sigma, az[r][i], q, xrow, drow, hrow);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// k_sample_wide — the same computation for ONE large population (lambda in the hundreds and up), where a
// warp per offspring row leaves the SMs almost empty (lambda / 2 warps over 592 warp schedulers) and every
// dependent FMA / shared-memory load latency is exposed.  Here a row is split over CW warps (each lane owns one
// float4 column), a warp carries RBW rows for its columns (each pair element read from shared memory serves RBW
// rows: shared-memory bandwidth is the scarce resource), a CTA holds R row-groups x CW column-warps, and the
// 8 partial dot products of a group are exchanged through shared memory with one named barrier per row-group
// and group.  4x..16x more resident warps per SM than the warp-per-row kernel.
// grid = (ceil(pop_count / (R * RBW)), B), block = 32 * R * CW.
// ------------------------------------------------------------------------------------------------
//
// progressive != 0 (one query, fused generation): the kernel is released while k_update is still in its triangular
// sweep and consumes the pairs as k_update publishes them (OptDev::progress, gpu-scope release / acquire), one chunk
// per round, so that only the last chunk's work is left when the sweep ends.  Requires one stage per chunk.
template <int RBW, int MAXT>
__global__ void __launch_bounds__(MAXT) k_sample_wide(OptDev o, int kc, int nstages, int R, int CW, int qpw /* float4 columns per warp */,
                                                       int progressive) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int b = blockIdx.y;
    if (o.only && o.only[b] == 0) return;                       // an instance the reset leaves alone (OptDev::only)
#define SMP_STAMP(k) do { if (o.dbg && threadIdx.x == 0 && blockIdx.x == 0 && blockIdx.y == 0) o.dbg[k] = gtime(); } while (0)
    SMP_STAMP(TL_SMP_START);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int rl = warp / CW, cw = warp - rl * CW;              // row-group within the CTA, column-warp within the row
    const int ns = o.ns, nq = ns >> 2;
    float* stage_base = reinterpret_cast<float*>(smem_raw);
    const size_t stage_floats = (size_t)kc * 2 * ns;
    unsigned long long* bars = reinterpret_cast<unsigned long long*>(stage_base + (size_t)nstages * stage_floats);
    float* nj_s = reinterpret_cast<float*>(bars + SAMPLE_MAX_STAGES);   // Nj * M^-(g+1) of the live pairs (padded to 8)
    float* dpart = nj_s + o.m + SAMPLE_G;                               // (groups per round) x R x CW x RBW x 8 partial dot products
    if (threadIdx.x == 0) init_stages(bars, nstages);
    int* flags = progress_flags(o.progress, o.m, b);
    // bounded spin on a hand-over flag; if it never comes (a launch that did not pair this kernel with a publishing
    // k_update) fall back to waiting for the whole predecessor grid, after which everything is final anyway
    // progressive == 2 (overlapped generation): k_update is NOT a stream predecessor (it runs on a side branch of the graph,
    // concurrently with k_cost / k_rank), so there is no grid to fall back to: spin long, then fail loudly
    auto wait_flag = [&](const int* f) {
        if (progressive == 2) {
            const long long t0 = gtime();
            for (long long spin = 0;; ++spin) {
                if (ld_acquire_gpu(f) != 0) return;
                __nanosleep(32);
                if ((spin & 1023) == 1023 && (already_lost(o.err) || gtime() - t0 > LOST_TIMEOUT_NS)) break;
            }
            report_lost(o.err, LOST_SAMPLE_WAITING_FOR_UPDATE);   // the host sees it at its next sync; results of this generation are void
            return;
        }
        for (long long spin = 0; spin < (1ll << 22); ++spin) {
            if (ld_acquire_gpu(f) != 0) return;
            __nanosleep(32);
        }
        griddep_wait();
    };
    if (!progressive) {
        griddep_wait();                        // every input is k_update's output
    } else {
        if (threadIdx.x == 0) wait_flag(progressive == 2 ? flag_early(flags, o.m) : flag_mean(flags));   // (early) scalars
        __syncthreads();
    }
    SMP_STAMP(TL_SMP_FLAGS);
    const float* vps = o.VPs + (size_t)b * o.m * 2 * ns;
    // chunks of the first m pairs, not of the live ones, so that the first chunks are requested before the scalar state has
    // even been read (rows beyond `live` are never used)
    auto issue = [&](int c) { request_stage(stage_base, stage_floats, bars, nstages, vps, ns, kc, c, o.m); };   // thread 0
    const int max_chunks = (o.m + kc - 1) / kc;
    if (threadIdx.x == 0 && !progressive)
        for (int c = 0; c < max_chunks && c < nstages; ++c) issue(c);
    const Scalars sc = o.sc[b];
    const int live = sc.live;
    const int nchunks = (live + kc - 1) / kc;
    SMP_STAMP(TL_SMP_SCALARS);
    const float Mf = (float)o.M, Minv = 1.0f / Mf;
    // the groups of 8 start at chunk boundaries: with kc < 8 (rows longer than ~1600) pair k is element (k mod kc) of its
    // group, and the last group reads up to 7 entries past its last live pair (zeros: they scale dots of zero pairs)
    if (!progressive) {
        const int gmask = min(kc, SAMPLE_G) - 1;                    // kc is 1, 2, 4 or 8
        for (int k = threadIdx.x; k < live + SAMPLE_G - 1; k += blockDim.x) {
            float sc8 = Minv;                                       // M^-((k mod min(kc, 8)) + 1)
            for (int c = 0; c < (k & gmask); ++c) sc8 *= Minv;
            nj_s[k] = (k < live) ? o.Njs[(size_t)b * o.m + k] * sc8 : 0.f;
        }
    }
    // progressive (warp 0, all lanes): chunk c = pairs [c kc, c kc + cnt) — poll their flags, stage Nj, request the copy
    int next_issue = 0;                                         // warp 0: chunks [0, next_issue) have been requested
    auto chunk_ready = [&](int c) -> bool {
        const int k0 = c * kc, cnt = min(kc, live - k0);
        int f = 1;
        if (lane < cnt) f = ld_acquire_gpu(flag_pair(flags, k0) + lane);
        return __all_sync(0xffffffffu, f != 0);
    };
    auto request_chunk = [&](int c) {                           // flags are set
        const int k0 = c * kc, cnt = min(kc, live - k0);
        if (lane < SAMPLE_G && lane < ((cnt + SAMPLE_G - 1) & ~(SAMPLE_G - 1))) {
            float sc8 = Minv;
            for (int c2 = 0; c2 < (lane & 7); ++c2) sc8 *= Minv;
            nj_s[k0 + lane] = (lane < cnt) ? o.Njs[(size_t)b * o.m + k0 + lane] * sc8 : 0.f;
        }
        __syncwarp();
        if (lane == 0) {
            fence_proxy_async_all();                            // the rows were written through the generic proxy (by k_update)
            request_stage(stage_base, stage_floats, bars, nstages, vps, ns, kc, c, live);
        }
    };
    auto provide_chunk = [&](int c) {                           // warp 0: make sure chunk c is on its way, then run ahead
        while (next_issue <= c) {
            bool ok = false;
            if (progressive == 2) {
                const long long t0 = gtime();
                for (long long spin = 0; !ok; ++spin) {
                    ok = chunk_ready(next_issue);
                    if (ok) break;
                    __nanosleep(32);
                    if ((spin & 1023) == 1023) {                 // lane 0 decides for the warp
                        const int giveup = (already_lost(o.err) || gtime() - t0 > LOST_TIMEOUT_NS) ? 1 : 0;
                        if (__shfl_sync(0xffffffffu, giveup, 0)) break;
                    }
                }
                if (!ok && lane == 0) report_lost(o.err, LOST_SAMPLE_WAITING_FOR_UPDATE);   // carry on (the chunk is requested as is)
            } else {
                for (long long spin = 0; spin < (1ll << 22) && !ok; ++spin) { ok = chunk_ready(next_issue); if (!ok) __nanosleep(32); }
                if (!ok) griddep_wait();                        // see wait_flag
            }
            request_chunk(next_issue++);
        }
        while (next_issue < nchunks && chunk_ready(next_issue)) request_chunk(next_issue++);
    };
    float M8 = 1.0f;
#pragma unroll
    for (int c = 0; c < SAMPLE_G; ++c) M8 *= Mf;

    // ---- z of this lane's float4 column, RBW rows ----
    const int row0 = (blockIdx.x * R + rl) * RBW;
    const int q = cw * qpw + lane;
    const bool qon = lane < qpw && q < nq;
    const int qs = qon ? q : 0;                                 // idle lanes read column 0 and contribute z = 0
    float4 z[RBW], az[RBW];
#pragma unroll
    for (int r = 0; r < RBW; ++r) {
        const int row = row0 + r;
        const bool on = qon && row < o.pop_count;
        const size_t roff = ((size_t)b * o.pop_count + (row < o.pop_count ? row : 0)) * ns;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (on) sample_deviate4(o, b, row, roff, q, sc.itr, sc.epoch, v);
        z[r] = v; az[r] = v;
    }
    SMP_STAMP(TL_SMP_Z);
    __syncthreads();                                            // nj_s
    // The chunks are consumed in rounds of up to `nstages` resident chunks.  Within a round every dot product comes
    // first (all against the ORIGINAL z: no ordering between pairs), the partial sums are exchanged ONCE, then the
    // ordered recurrence runs over the round's pairs: one named barrier per round instead of one per group.
    const int gpc = (kc + SAMPLE_G - 1) / SAMPLE_G;             // groups per chunk
    const int round = progressive ? 1 : nstages;                // chunks per round
    for (int c0 = 0; c0 < nchunks; c0 += round) {
        const int c1 = min(nchunks, c0 + round);
        float* dp0 = dpart + (size_t)rl * CW * RBW * SAMPLE_G;
        const size_t grp_stride = (size_t)R * CW * RBW * SAMPLE_G;
        // progressive: no block-wide barrier between rounds, so the exchange buffer alternates (a warp can be one
        // round ahead of its row-group, never two: the named barrier below)
        const int grp0 = progressive ? (c0 & 1) * gpc : 0;
        int grp = grp0;
        for (int c = c0; c < c1; ++c) {
            const int st = c % nstages;
            if (progressive && warp == 0) provide_chunk(c);
            mbar_wait(&bars[st], (unsigned)((c / nstages) & 1));
            if (c == 0) SMP_STAMP(TL_SMP_FIRST_PAIRS);
            if (c < TL_SMP_CHUNKS) SMP_STAMP(TL_SMP_CHUNK + c);
            const float* sb = stage_base + st * stage_floats;
            const int cnt = min(kc, live - c * kc);
            for (int k = 0; k < cnt; k += SAMPLE_G, ++grp) {
                const int gcnt = min(SAMPLE_G, cnt - k);       // pairs in this group (CTA-uniform)
                float d[RBW][SAMPLE_G];
#pragma unroll
                for (int g = 0; g < SAMPLE_G; ++g) {
                    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (g < gcnt) v = reinterpret_cast<const float4*>(sb + (size_t)(2 * (k + g)) * ns)[qs];
#pragma unroll
                    for (int r = 0; r < RBW; ++r) d[r][g] = fmaf(v.x, z[r].x, fmaf(v.y, z[r].y, fmaf(v.z, z[r].z, v.w * z[r].w)));
                }
                float* dp = dp0 + grp * grp_stride;
#pragma unroll
                for (int r = 0; r < RBW; ++r) {
                    const float part = reduce_scatter8(d[r], lane);   // pair (lane >> 2) & 7, summed over this warp's columns
                    if ((lane & 3) == 0) dp[(cw * RBW + r) * SAMPLE_G + (lane >> 2)] = part;
                }
            }
        }
        SMP_STAMP(TL_SMP_DOTS);
        if (CW > 1) named_bar_sync(1 + rl, CW * 32);            // the CW warps of this row-group (ids 1..15: R <= 15)
        else __syncwarp();
        SMP_STAMP(TL_SMP_EXCHANGED);
        grp = grp0;
        for (int c = c0; c < c1; ++c) {
            const int st = c % nstages;
            const float* sb = stage_base + st * stage_floats;
            const int k0 = c * kc, cnt = min(kc, live - k0);
            for (int k = 0; k < cnt; k += SAMPLE_G, ++grp) {
                const int gcnt = min(SAMPLE_G, cnt - k);
                const float* dp = dp0 + grp * grp_stride;
                float tot = 0.f;                                // lane = r * 8 + g: c_g of row r
                if (lane < RBW * SAMPLE_G) {
                    const int r = lane >> 3, g = lane & 7;
                    for (int w2 = 0; w2 < CW; ++w2) tot += dp[(w2 * RBW + r) * SAMPLE_G + g];
                    tot *= nj_s[k0 + k + g];                    // c_g = Nj_g (v_g . z) M^-(g+1); 0 beyond gcnt
                }
                float4 acc[RBW];
#pragma unroll
                for (int r = 0; r < RBW; ++r) acc[r] = az[r];
#pragma unroll
                for (int g = 0; g < SAMPLE_G; ++g) {
                    float4 p = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (g < gcnt) p = reinterpret_cast<const float4*>(sb + (size_t)(2 * (k + g) + 1) * ns)[qs];
#pragma unroll
                    for (int r = 0; r < RBW; ++r) {
                        const float w = __shfl_sync(0xffffffffu, tot, r * SAMPLE_G + g);
                        acc[r].x = fmaf(w, p.x, acc[r].x); acc[r].y = fmaf(w, p.y, acc[r].y);
                        acc[r].z = fmaf(w, p.z, acc[r].z); acc[r].w = fmaf(w, p.w, acc[r].w);
                    }
                }
                float mg = M8;
                if (gcnt < SAMPLE_G) { mg = 1.0f; for (int c2 = 0; c2 < gcnt; ++c2) mg *= Mf; }
#pragma unroll
                for (int r = 0; r < RBW; ++r) az[r] = make_float4(acc[r].x * mg, acc[r].y * mg, acc[r].z * mg, acc[r].w * mg);
            }
        }
        if (c1 < nchunks && !progressive) {                     // next round: every warp is done with all stages
            __syncthreads();
            if (threadIdx.x == 0)
                for (int c = c1; c < max_chunks && c < c1 + nstages; ++c) issue(c);
        }
    }
    SMP_STAMP(TL_SMP_LOOP_DONE);
    double sigma = sc.sigma;
    if (progressive == 2) {                                     // step size and mean arrive after k_rank, late in k_update
        if (threadIdx.x == 0) wait_flag(flag_mean(flags));
        __syncthreads();
        sigma = __ldcg(&o.sc[b].sigma);
    }
#pragma unroll
    for (int r = 0; r < RBW; ++r) {
        const int row = row0 + r;
        if (qon && row < o.pop_count) {
            const size_t roff2 = ((size_t)b * o.pop_count + row) * ns;
            sample_finish(o, o.xmean + (size_t)b * ns, sigma, az[r], q, o.X + roff2, o.D + roff2, o.Xh ? o.Xh + roff2 : nullptr);
        }
    }
    if (progressive) griddep_wait();                            // stream order: this grid ends after k_update has
    SMP_STAMP(TL_SMP_END);
#undef SMP_STAMP
}

}  // namespace lmcma

namespace lmcma {

// ------------------------------------------------------------------------------------------------
// k_sample_rows — the same computation laid out for MANY rows (batched queries: B x lambda in the hundreds of thousands;
// one very large population), where the two kernels above spend more issue slots on cross-lane reductions than on
// multiply-adds (one 32-lane reduction per dot product: ~2x the FMA work of the wide kernel).
//
//   * a LANE owns RL offspring rows, a WARP owns a slice of QW float4 columns: a dot product v_j . z is accumulated by
//     the lane itself over its warp's slice — no shuffle at all — and the NW partial sums per (row, pair) are added once
//     per chunk through shared memory;
//   * every element of a direction pair is read by a warp as ONE broadcast shared-memory load (all lanes, same
//     address) that feeds RL rows x 4 elements: 2 * RL packed multiply-adds (fma.rn.f32x2) per 16-byte load, so the
//     inner loops are bound by the FP32 pipe, not by shared-memory bandwidth or issue slots;
//   * two passes over the pairs instead of one interleaved pass: all dots are against the ORIGINAL z (lmcma.cpp:441-443),
//     so pass 1 forms every coefficient c_j = Nj_j (v_j . z) M^(L-1-j) and pass 2 the closed form of the recurrence
//     Az <- M Az + d_j pc_j (lmcma.cpp:444-445):  Az = M^L z + sum_j c_j pc_j  (same value in exact arithmetic; z is dead
//     after pass 1, Az is born there: half the registers of the interleaved form);
//   * the finished tile is transposed through shared memory so that x = xmean + sigma Az (FP64), the clamp and the two
//     (three with the host mirror) row stores are coalesced.
// grid = (ceil(pop_count / (32 RL)), B), block = 32 NW; all pairs resident in shared memory when they fit (C2 / C3 / C5
// shapes: 128 KB), otherwise streamed twice through a ring of stages.
// ------------------------------------------------------------------------------------------------
template <int QW, int RL>
__global__ void __launch_bounds__(512, 1) k_sample_rows(OptDev o, int kc, int nstages, int region_floats /* >= stages, >= transposition tile */) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int b = blockIdx.y;
    if (o.only && o.only[b] == 0) return;                     // an instance the reset leaves alone (OptDev::only)
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5, nthr = blockDim.x;
    const int ns = o.ns, nq = ns >> 2, m = o.m;
    constexpr int ROWS = 32 * RL;
    const size_t stage_floats = (size_t)kc * 2 * ns;
    float* stage_base = reinterpret_cast<float*>(smem_raw);                        // nstages x kc x {v, pc} x ns
    unsigned long long* bars = reinterpret_cast<unsigned long long*>(stage_base + (size_t)region_floats);
    float* scale_s = reinterpret_cast<float*>(bars + SAMPLE_MAX_STAGES);           // m (padded to kc): Nj_j M^(L-1-j)
    float* coef_s = scale_s + ((m + kc + 3) & ~3);                                  // (m padded) x ROWS: c_j per row
    float* part_s = coef_s + (size_t)((m + kc - 1) / kc) * kc * ROWS;              // nwarps x kc x ROWS partial dots
    if (threadIdx.x == 0) init_stages(bars, nstages);
    griddep_wait();                           // launched as a programmatic dependent of k_update: every input is its output
    const Scalars sc = o.sc[b];
    const int live = sc.live;
    const int nchunks = (live + kc - 1) / kc;
    const float* vps = o.VPs + (size_t)b * m * 2 * ns;
    auto issue = [&](int c) { request_stage(stage_base, stage_floats, bars, nstages, vps, ns, kc, c, live); };   // thread 0
    if (threadIdx.x == 0)
        for (int c = 0; c < nchunks && c < nstages; ++c) issue(c);
    // Nj_j M^(L-1-j): the powers by repeated multiplication from the newest pair down (one warp, fixed order)
    const float Mf = (float)o.M;
    if (warp == 0) {
        const int lpad = nchunks * kc;
        for (int j0 = 0; j0 < lpad; j0 += 32) {
            const int j = j0 + lane;
            float pw = 1.0f;
            for (int e = 0; e < live - 1 - j; ++e) pw *= Mf;
            if (j < lpad) scale_s[j] = j < live ? o.Njs[(size_t)b * m + j] * pw : 0.f;
        }
    }
    float mL = 1.0f;
    for (int e = 0; e < live; ++e) mL *= Mf;

    // ---- z of my rows, my warp's column slice ----
    const int qper = (nq + nwarps - 1) / nwarps;                    // <= QW
    const int q0 = warp * qper;
    const int row0 = blockIdx.x * ROWS;
    float4 acc[RL][QW];                                             // z in pass 1, Az in pass 2
#pragma unroll
    for (int r = 0; r < RL; ++r) {
        const int row = row0 + r * 32 + lane;
        const bool rv = row < o.pop_count;
        const size_t roff = ((size_t)b * o.pop_count + (rv ? row : 0)) * ns;
#pragma unroll
        for (int i = 0; i < QW; ++i) {
            const int q = q0 + i;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (rv && i < qper && q < nq) sample_deviate4(o, b, row, roff, q, sc.itr, sc.epoch, v);
            acc[r][i] = v;
        }
    }
    __syncthreads();                                                // scale_s

    // ---- pass 1: c_j for every live pair ----
    for (int c = 0; c < nchunks; ++c) {
        const int st = c % nstages;
        mbar_wait(&bars[st], (unsigned)((c / nstages) & 1));
        const float* sb = stage_base + st * stage_floats;
        const int k0 = c * kc, cnt = min(kc, live - k0);
        for (int g = 0; g < cnt; ++g) {
            const float4* vrow = reinterpret_cast<const float4*>(sb + (size_t)(2 * g) * ns) + q0;
            float2 d[RL];
#pragma unroll
            for (int r = 0; r < RL; ++r) d[r] = make_float2(0.f, 0.f);
#pragma unroll
            for (int i = 0; i < QW; ++i) {
                if (i < qper && q0 + i < nq) {
                    const float4 v = vrow[i];                       // broadcast: every lane reads the same 16 bytes
#pragma unroll
                    for (int r = 0; r < RL; ++r) {
                        d[r] = ffma2(lo2(v), lo2(acc[r][i]), d[r]);
                        d[r] = ffma2(hi2(v), hi2(acc[r][i]), d[r]);
                    }
                }
            }
#pragma unroll
            for (int r = 0; r < RL; ++r) part_s[((size_t)warp * kc + g) * ROWS + r * 32 + lane] = d[r].x + d[r].y;
        }
        __syncthreads();                                            // all partials of the chunk; every warp is done with its stage
        for (int e = threadIdx.x; e < cnt * ROWS; e += nthr) {       // (pair, row): add the nwarps partials in warp order
            const int g = e / ROWS, rr = e - g * ROWS;
            float s = 0.f;
            for (int w2 = 0; w2 < nwarps; ++w2) s += part_s[((size_t)w2 * kc + g) * ROWS + rr];
            coef_s[(size_t)(k0 + g) * ROWS + rr] = s * scale_s[k0 + g];
        }
        if (threadIdx.x == 0 && c + nstages < nchunks) issue(c + nstages);     // ring: only when the pairs do not all fit
        __syncthreads();                                            // part_s is free again; coef_s rows of this chunk are visible
    }
    // Az = M^L z + ...
#pragma unroll
    for (int r = 0; r < RL; ++r)
#pragma unroll
        for (int i = 0; i < QW; ++i) acc[r][i] = make_float4(acc[r][i].x * mL, acc[r][i].y * mL, acc[r][i].z * mL, acc[r][i].w * mL);

    // ---- pass 2: Az += sum_j c_j pc_j ----
    const bool resident = nchunks <= nstages;                       // the chunks of pass 1 are still in their stages
    if (!resident) {
        __syncthreads();
        if (threadIdx.x == 0)
            for (int c = 0; c < nchunks && c < nstages; ++c) issue(c);
    }
    for (int c = 0; c < nchunks; ++c) {
        const int st = c % nstages;
        if (!resident) mbar_wait(&bars[st], (unsigned)((((nchunks - 1 - st) / nstages + 1) + c / nstages) & 1));
        const float* sb = stage_base + st * stage_floats;
        const int k0 = c * kc, cnt = min(kc, live - k0);
        for (int g = 0; g < cnt; ++g) {
            const float4* prow = reinterpret_cast<const float4*>(sb + (size_t)(2 * g + 1) * ns) + q0;
            float2 w[RL];
#pragma unroll
            for (int r = 0; r < RL; ++r) { const float cw = coef_s[(size_t)(k0 + g) * ROWS + r * 32 + lane]; w[r] = make_float2(cw, cw); }
#pragma unroll
            for (int i = 0; i < QW; ++i) {
                if (i < qper && q0 + i < nq) {
                    const float4 p = prow[i];
#pragma unroll
                    for (int r = 0; r < RL; ++r) {
                        const float2 l = ffma2(w[r], lo2(p), lo2(acc[r][i])), h = ffma2(w[r], hi2(p), hi2(acc[r][i]));
                        acc[r][i] = make_float4(l.x, l.y, h.x, h.y);
                    }
                }
            }
        }
        if (!resident && c + nstages < nchunks) {
            __syncthreads();
            if (threadIdx.x == 0) issue(c + nstages);
        }
    }

    // ---- transpose through shared memory (the stages are free), then the coalesced finish ----
    __syncthreads();
    const int tstride = ns + 4;                                     // rows 16 bytes apart modulo 128: conflict-free 16-byte stores
    float* tile = stage_base;
#pragma unroll
    for (int r = 0; r < RL; ++r)
#pragma unroll
        for (int i = 0; i < QW; ++i)
            if (i < qper && q0 + i < nq) reinterpret_cast<float4*>(tile + (size_t)(r * 32 + lane) * tstride)[q0 + i] = acc[r][i];
    __syncthreads();
    // a thread keeps ONE float4 column and walks down the rows: mean, bounds and the padding mask of the column are loaded
    // once, consecutive threads still store consecutive 16 bytes of a row
    const double* xm = o.xmean + (size_t)b * ns;
    const int rstep = nthr / nq, q = threadIdx.x % nq, r_first = threadIdx.x / nq;     // nq <= 128 <= nthr
    if (r_first < rstep) {
        const double2 m01 = reinterpret_cast<const double2*>(xm)[2 * q], m23 = reinterpret_cast<const double2*>(xm)[2 * q + 1];
        const double mm[4] = {m01.x, m01.y, m23.x, m23.y};
        float4 lo4 = make_float4(-3.4e38f, -3.4e38f, -3.4e38f, -3.4e38f), hi4 = make_float4(3.4e38f, 3.4e38f, 3.4e38f, 3.4e38f);
        if (o.lo) lo4 = reinterpret_cast<const float4*>(o.lo)[q];
        if (o.hi) hi4 = reinterpret_cast<const float4*>(o.hi)[q];
        const float ll[4] = {lo4.x, lo4.y, lo4.z, lo4.w}, hh[4] = {hi4.x, hi4.y, hi4.z, hi4.w};
        const int npad = max(0, q * 4 + 4 - o.n);                    // trailing padding lanes of this column (0 except in the last one)
        const double sigma = sc.sigma;
        for (int rr = r_first; rr < ROWS && row0 + rr < o.pop_count; rr += rstep) {
            const float4 az = reinterpret_cast<const float4*>(tile + (size_t)rr * tstride)[q];
            const float aa[4] = {az.x, az.y, az.z, az.w};
            float xx[4], dd[4];
#pragma unroll
            for (int c = 0; c < 4; ++c) finish_element(mm[c], sigma, aa[c], ll[c], hh[c], 0, c, 4 - npad, xx[c], dd[c]);   // column-relative padding
            const size_t roff = ((size_t)b * o.pop_count + row0 + rr) * ns;
            reinterpret_cast<float4*>(o.X + roff)[q] = make_float4(xx[0], xx[1], xx[2], xx[3]);
            reinterpret_cast<float4*>(o.D + roff)[q] = make_float4(dd[0], dd[1], dd[2], dd[3]);
            if (o.Xh) __stcs(reinterpret_cast<float4*>(o.Xh + roff) + q, make_float4(xx[0], xx[1], xx[2], xx[3]));
        }
    }
}

}  // namespace lmcma

// lmcma_common.cuh — device-side structs and helpers shared by the hand-written sm_100a kernels of the
// LM-CMA trajectory-optimisation hot path (k_cost.cuh, k_tell.cuh, k_sample.cuh).
//
// One generation = k_cost -> k_rank -> k_update -> k_sample, all on one stream and
// replayed from a CUDA graph (lmcma_capi.cu).  Everything is batched over B independent optimiser
// instances (gridDim.y or gridDim.x = B).  FP32 on CUDA cores for the bulk data, FP64 for the
// handful of per-instance scalars whose closed forms cancel (sigma, s, Nj, Lj, xmean).
//
// Reference lines each kernel stands in for are cited at the kernel.  Row stride `ns` is n rounded
// up to a multiple of 4 floats so that every row is 16-byte aligned (float4 / bulk-copy granularity);
// the padding lanes are kept at exactly 0.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "lmcma_layout.hpp"

namespace lmcma {

constexpr int KMAX_SUBSTEPS = 65536;   // cap on sub-steps per segment (DESIGN.md, cost model)

struct Scalars {          // per-instance scalar state
    double sigma;         // LMCMA::sigma
    double s;             // LMCMA::s
    double best_f;        // CMABase::BestF
    long long counteval;  // CMABase::counteval
    int itr;              // CMABase::itr
    int live;             // LMCMA::iterator_sz
    int best_local;       // 1 if best_x holds the row that achieved best_f (split mode: may live on a peer)
    int pad;
};

struct OptDev {
    int n, ns, lambda, mu, m, B;
    int pop_offset, pop_count;     // rows of lambda owned by this handle
    int rng_mode, record_z;
    unsigned long long seed;
    // population
    float* X;          // B x pop_count x ns
    float* Xh;         // null, or the device alias of the handle's page-locked host mirror of X (same layout): the sampler
                       // writes every candidate row there as well (posted PCIe writes that overlap the sampling), so the
                       // host-buffer protocol needs no D2H copy of the population after the generation (lmcma_b200_ask_all_view)
    float* Z;          // B x pop_count x ns (INJECT / record_z) or null
    float* Zc;         // B x pop_count x ns  L z (smoothness prior, k_prior.cuh) or null: what computeAz sees
    const float* Lf;   // n x ns lower Cholesky factor of the prior (FP32) or null
    float* D;          // B x pop_count x ns  x - xmean, formed in FP64 and rounded once: FP32 X cannot resolve a step
                       //                     below ulp(x) (sigma / |x| < 6e-8), the recombination must not depend on it
    float* fit;        // B x lambda   fitness as evaluated / told (all rows, global order)
    float* fit_sorted; // B x lambda
    float* prev_fit;   // B x lambda   previous generation (any order)
    // large unsplit populations (lambda > 4096, k_rank.cuh "sorted tiles"): ranks by binary search instead of counting
    float* prev_sorted;   // B x lambda   previous generation, ascending (= its fit_sorted), or null
    float* tile_sorted;   // B x lambda   this generation's fitness, each 4096-candidate tile sorted ascending, or null
    int* tile_pos;        // B x lambda   position of candidate i inside its sorted tile
    int* rank;         // B x lambda   (only [pop_offset, +pop_count) written in split mode)
    int* arindex;      // B x lambda
    int* ncoll;        // B x pop_count
    int* nsamp;        // B x pop_count
    // distribution state
    double* xmean;     // B x ns
    float* pc;         // B x ns
    float* V;          // B x m x ns   (slot-indexed)
    float* P;          // B x m x ns
    double* Nj;        // B x m
    double* Lj;        // B x m
    float* Njf;        // B x m   FP32 copies, slot-indexed
    // sequence-ordered mirror read by k_sample: pair i of the sequence is {v, pc} = VPs[(b*m + i)*2 + {0,1}][ns], so a
    // chunk of consecutive pairs is ONE contiguous block (one bulk async copy instead of one per row)
    float* VPs;        // B x m x 2 x ns
    float* Njs;        // B x m   Nj in sequence order
    // Gram-matrix recompute (k_gram.cuh), allocated only for shapes that take it
    double* G;         // B x m x m
    double* Cf;        // B x m x m
    int2* gram_hdr;    // B : {first_stale, live} handed from k_update to k_gram / k_coef / k_combine
    // progressive hand-over k_update -> k_sample inside one generation (see k_update.cuh).  Reset by k_rank (by k_update
    // itself in the overlapped generation).
    int* progress;     // B x (m + 2): slots named by progress_len, progress_flags and flag_* below
    unsigned* rank_ticket;   // B : one ticket per k_rank CTA after its last store; k_update waits for RS of them in the overlapped generation
    int* resident;     // B : k_update (overlapped generation) holds its SM; k_gate releases k_cost
    int* t;            // B x m   slot order, oldest -> newest
    int* vec;          // B x m   generation stamp per slot
    Scalars* sc;       // B
    float* best_x;     // B x ns
    const float* lo;   // n or null
    const float* hi;   // n or null
    const float* w;    // mu recombination weights
    float* partial;    // B x RS x ns weighted partial sums of (x - xmean)
    int RS;
    int rank_ftile;    // fitness values k_rank stages per shared-memory tile: TELL_FTILE, or lambda rounded up to 4 for small populations
    unsigned long long* S_count;   // B : #{(i,j): prev_j < cur_i}
    unsigned* done_count;          // B : tickets of k_rank (split-population payload packing)
    double c1, cc, cs, target, K, M, mueff;
    double pc_coef;    // sqrt(cc (2 - cc) mueff), lmcma.cpp:328
    long long* dbg;    // optional device timeline of TL_SLOTS stamps (LMCMA_B200_DBG, see TimelineSlot); null in normal runs
    int* err;          // host-visible (mapped, page-locked) error word of the handle: a kernel of the overlapped generation
                       // that gives up waiting for its concurrently running partner writes a code here and carries on
                       // (never __trap: that would poison the whole CUDA context); the host checks it at every sync
};

// The hand-over flags OptDev::progress of instance b: progress_len(m) = m + 2 ints, [0] scalars and mean are final
// (flag_mean), [1 + i] pair i of the sequence-ordered mirror and Njs[i] are final (flag_pair), [m + 1] the early scalars
// (itr, live) of the overlapped generation are final (flag_early).
__host__ __device__ __forceinline__ int progress_len(int m) { return m + 2; }
__device__ __forceinline__ int* progress_flags(int* progress, int m, int b) { return progress + (size_t)b * progress_len(m); }
__device__ __forceinline__ int* flag_mean(int* flags) { return flags; }
__device__ __forceinline__ int* flag_pair(int* flags, int i) { return flags + 1 + i; }
__device__ __forceinline__ int* flag_early(int* flags, int m) { return flags + m + 1; }

// The slots of the device timeline OptDev::dbg (LMCMA_B200_DBG): globaltimer stamps taken by one thread of instance 0,
// printed and cleared by print_timeline (lmcma_capi.cu).  k_rank and k_sample_wide stamp [0, TL_UPD) through
// OptDev::dbg; k_update stamps through UpdateArgs::dbg = OptDev::dbg + TL_UPD, so the TL_UPD_* slots count from there.
enum TimelineSlot : int {
    // k_rank, CTA 0: start, ranks stored, selected rows compacted, partial sums gathered / stored; the last CTA's ticket
    TL_RANK_START = 16, TL_RANK_RANKED, TL_RANK_COMPACTED, TL_RANK_GATHERED, TL_RANK_STORED, TL_RANK_LAST_SLICE,
    // k_sample_wide, CTA 0: start, flags / griddep, scalars read, z ready, first pairs, loop done, end; chunk c < 8
    // arrived; last round's dots done and exchanged
    TL_SMP_START = 32, TL_SMP_FLAGS, TL_SMP_SCALARS, TL_SMP_Z, TL_SMP_FIRST_PAIRS, TL_SMP_LOOP_DONE, TL_SMP_END,
    TL_SMP_CHUNK, TL_SMP_CHUNKS = 8, TL_SMP_DOTS = TL_SMP_CHUNK + TL_SMP_CHUNKS, TL_SMP_EXCHANGED,
    TL_UPD = 64,
    // k_update, relative to TL_UPD: start, bookkeeping, prologue, post-rank start, mean, tail start, end, every older row
    // final, ranks seen, newest row done (overlapped build)
    TL_UPD_START = 0, TL_UPD_BOOKKEEPING, TL_UPD_PROLOGUE, TL_UPD_POST, TL_UPD_MEAN, TL_UPD_TAIL, TL_UPD_END,
    TL_UPD_ROWS_FINAL, TL_UPD_RANKS_SEEN, TL_UPD_NEWEST,
    TL_UPD_FIRST_STALE = 10, TL_UPD_LIVE = 11,          // values, not stamps
    TL_UPD_BEST_COPIED = 18,                            // overlapped build: the best-so-far candidate is copied out of X
    TL_UPD_STEP_SIZE = 22,                              // overlapped build: step size released (progress[0])
    TL_UPD_ROWS = 24, TL_UPD_ROW_STAMPS = 40,           // row i < 40 published
    TL_UPD_CHAIN = 64, TL_UPD_CHAIN_STAMPS = 10,        // overlapped build: block j0 / UPD_BLK of the newest row's chain (m <= 80)
    TL_SLOTS = TL_UPD + TL_UPD_CHAIN + TL_UPD_CHAIN_STAMPS
};

// codes written to OptDev::err
enum { LOST_UPDATE_WAITING_FOR_RANK = 2, LOST_SAMPLE_WAITING_FOR_UPDATE = 3 };
constexpr long long LOST_TIMEOUT_NS = 2000000000ll;      // 2 s: far beyond any scheduling jitter of a co-resident partner

struct MapDev {
    int dims, nx, ny, nz;
    unsigned nbx, nby;         // bricks per row / per column (lmcma_layout.hpp)
    unsigned py, pz;           // brick_pitch_y / brick_pitch_z of the layout (constant-bank operands of the sample loop)
    int storage;               // 0 = F32 sign-tagged reciprocal clearance, 1 = U8 quantised distance
    const float* g32;
    const unsigned char* q8;
    const float* lut;          // 256 sign-tagged reciprocal clearances (U8)
    float g_coll;              // 1 / c_min
};

struct CostArgs {
    int W;
    float w_len, w_clr, w_col;
    const float* X;            // candidates
    long long ld;              // row stride (floats)
    long long inst_rows;       // rows per instance (gridDim.x)
    const float* ends;         // per instance: start[3], goal[3]   (stride 6 floats); used when ends_per_instance != 0
    int ends_per_instance;     // 1: ends[b] (device array of the attached optimiser), 0: ends0 for every instance
    float ends0[6];            // start[3], goal[3] BY VALUE for the stand-alone evaluate calls: no device buffer shared
                               // between callers / streams (two queries evaluated on one map from two streams cannot race)
    float* f;                  // outputs, indexed [b * f_stride + f_offset + row]
    long long f_stride;
    int f_offset;
    int* ncoll;                // indexed [b * inst_rows + row] (nullable)
    int* nsamp;
    long long* cells;          // trace mode (nullable)
    long long max_cells;
    int cb;                    // capacity of the per-block record stage (32-sample blocks), set by the launcher
    int spt;                   // segments per thread = ceil((W + 1) / threads per trajectory), set by the launcher
    long long* dbg;            // optional (LMCMA_B200_DBG, profile_kernels): 8 globaltimer stamps per CTA, [cta * 8 + k]
};

struct CostShape { int tpt = 128, cb = 256, minb = 0; };   // launch shape of k_cost: threads per trajectory, block-record capacity, CTAs per SM of the build to launch (0 = chosen by the launch size)

// ------------------------------------------------------------------------------------------------
// small device helpers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ int warp_sum_i(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
// Packed FP32 (Blackwell FFMA2 / FMUL2: two IEEE fp32 operations per lane per issue slot, each component rounded
// exactly like the scalar instruction).  The FMA-bound inner loops are issue-slot bound, so this halves their cost.
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
    unsigned long long r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r)
        : "l"(*reinterpret_cast<const unsigned long long*>(&a)), "l"(*reinterpret_cast<const unsigned long long*>(&b)),
          "l"(*reinterpret_cast<const unsigned long long*>(&c)));
    return *reinterpret_cast<float2*>(&r);
}
__device__ __forceinline__ float2 fmul2(float2 a, float2 b) {
    unsigned long long r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r)
        : "l"(*reinterpret_cast<const unsigned long long*>(&a)), "l"(*reinterpret_cast<const unsigned long long*>(&b)));
    return *reinterpret_cast<float2*>(&r);
}
__device__ __forceinline__ float2 lo2(const float4& v) { return make_float2(v.x, v.y); }
__device__ __forceinline__ float2 hi2(const float4& v) { return make_float2(v.z, v.w); }

__device__ __forceinline__ float canon_fitness(float f) { return (f != f) ? __int_as_float(0x7f800000) : f; }

// mbarrier + 1-D bulk async copy (TMA engine, SASS UBLKCP) wrappers
__device__ __forceinline__ unsigned smem_u32(const void* p) { return static_cast<unsigned>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void mbar_init(void* bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(void* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(void* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(void* bar, unsigned parity) {
    unsigned ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n" : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(void* bar, unsigned parity) {
    while (!mbar_try_wait(bar, parity)) {}
}
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, unsigned bytes, void* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// gpu-scope release / acquire on a flag in global memory, and the generic -> async proxy fence a bulk async copy of
// data published that way needs
__device__ __forceinline__ void st_release_gpu(int* p, int v) { asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
__device__ __forceinline__ int ld_acquire_gpu(const int* p) {
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
// cta-scope release / acquire on a flag in shared memory (no membar: a fence would wait for the thread's global stores)
__device__ __forceinline__ void st_release_cta_shared(int* p, int v) { asm volatile("st.release.cta.shared::cta.s32 [%0], %1;" ::"r"(smem_u32(p)), "r"(v) : "memory"); }
__device__ __forceinline__ int ld_acquire_cta_shared(const int* p) {
    int v;
    asm volatile("ld.acquire.cta.shared::cta.s32 %0, [%1];" : "=r"(v) : "r"(smem_u32(p)) : "memory");
    return v;
}
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }

__device__ __forceinline__ long long gtime() {
    long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}

// overlapped generation: the partner kernel did not show up in time (branches of the graph were serialised: profiler,
// sanitizer, SMs held by another process).  Record it for the host and let the caller continue without waiting.
__device__ __forceinline__ void report_lost(int* err, int code) {
    if (err) { *reinterpret_cast<volatile int*>(err) = code; __threadfence_system(); }
}
__device__ __forceinline__ bool already_lost(const int* err) { return err && *reinterpret_cast<const volatile int*>(err) != 0; }

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// programmatic dependent launch (PDL): a kernel launched with the programmatic-stream-serialization attribute may
// start while its predecessor is still running; it must not touch the predecessor's outputs before
// griddep_wait() (which returns once the predecessor grid has completed and its writes are visible).  Both are
// no-ops for a normally launched kernel.
__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void griddep_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// Philox4x32-10 (Salmon et al. 2011): counter-based, so any rank can regenerate any offspring row.
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const unsigned hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const unsigned hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += 0x9E3779B9u;
        k.y += 0xBB67AE85u;
    }
    return c;
}
__device__ __forceinline__ float4 philox_normal4(unsigned q, unsigned row, unsigned gen, unsigned inst, unsigned long long seed) {
    const uint4 r = philox4x32_10(make_uint4(q, row, gen, inst), make_uint2((unsigned)seed, (unsigned)(seed >> 32)));
    const float s = 2.3283064365386963e-10f;   // 2^-32
    const float u0 = r.x * s + 1.1641532182693481e-10f, u1 = r.y * s + 1.1641532182693481e-10f;
    const float u2 = r.z * s + 1.1641532182693481e-10f, u3 = r.w * s + 1.1641532182693481e-10f;
    // throughput mode only (parity runs inject z): hardware log2 / sin / cos, abs. error ~1e-6
    const float ra = sqrtf(-1.3862943611198906f * __log2f(u0)), rb = sqrtf(-1.3862943611198906f * __log2f(u2));
    float s0, c0, s1, c1;
    __sincosf(6.283185307179586f * u1, &s0, &c0);
    __sincosf(6.283185307179586f * u3, &s1, &c1);
    return make_float4(ra * c0, ra * s0, rb * c1, rb * s1);
}
// The generator's deviates v of float4 column q of local row `row` of instance b in generation itr, padding lanes zeroed:
// what the samplers draw (sample_deviate4, k_sample.cuh) and k_gauss materialises for the prior, so that a prior run and
// a plain run see the same raw deviates.
__device__ __forceinline__ void philox_deviate4(const OptDev& o, int b, int row, int q, int itr, float4& v) {
    v = philox_normal4((unsigned)q, (unsigned)(o.pop_offset + row), (unsigned)itr, (unsigned)b, o.seed);
    const int e = q * 4;
    if (e + 1 >= o.n) v.y = 0.f;
    if (e + 2 >= o.n) v.z = 0.f;
    if (e + 3 >= o.n) v.w = 0.f;
}

// Nj from |v|^2 in FP64 (lmcma.cpp:386-387, cancellation-free form: see the sweep in k_update.cuh): with r = nj_ratio(o),
// t = sqrt(1 + r |v|^2) and Nj = M r / (t + 1).  t comes back too: k_update's closed form of Lj is built on it.  Every
// store of Nj (k_update's hand-over and epilogue, k_coef) goes through here, so that all of them round alike.
__device__ __forceinline__ double nj_ratio(const OptDev& o) { return o.c1 / (1.0 - o.c1); }
struct NjForm { double t, nj; };
__device__ __forceinline__ NjForm nj_form(double r, double M, double nv) {
    const double t = sqrt(1.0 + r * nv);
    return {t, M * r / (t + 1.0)};
}

}  // namespace lmcma

// k_reset.cuh — restart chosen instances of a live batch in place (lmcma_b200_reset_instances): each flagged instance gets
// exactly the state lmcma_b200_create leaves (LMCMA::init, lmcma.cpp:233-299) for a new start and step size, with its
// deviate stream moved on by one epoch; the masked sampler launch that follows draws its first population.
#pragma once
#include "lmcma_common.cuh"
#include "k_gram.cuh"

namespace lmcma {

struct ResetArgs {
    const int* flags;          // B: non-zero = reset this instance
    const double* x0;          // B x n dense: the new mean (rows of unflagged instances are not read)
    const double* sigma0;      // B or null (sigma_default)
    double sigma_default;
    const float* ends;         // B x 6 {start xyz, goal xyz} or null (keep the instance's end points)
    float* d_ends;             // the handle's end points (B x 6), written from `ends`
    float* best_x_out;         // B x n or null: the retiring instance's best_x, flagged rows only
    double* best_f_out;        // B or null: its best_f as stored
};

template <class T>
__device__ __forceinline__ void reset_zero(T* p, size_t count) {
    for (size_t i = threadIdx.x; i < count; i += blockDim.x) p[i] = T(0);
}
// count floats at a 16-byte aligned address, count a multiple of 4 (rows of ns floats)
__device__ __forceinline__ void reset_zero4(float* p, size_t count) {
    float4* p4 = reinterpret_cast<float4*>(p);
    for (size_t i = threadIdx.x; i < count / 4; i += blockDim.x) p4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
}

// grid = B, one CTA per instance; the CTAs of unflagged instances exit.  Per-generation scratch that the kernels
// initialise before they read it (S_count, rank_ticket, resident, progress, done_count, partial, tile_*, gram_hdr, D)
// is left alone, and so are X, Z and Zc, which the masked sampler rewrites for the flagged instances.
__global__ void __launch_bounds__(256) k_reset(OptDev o, ResetArgs a) {
    const int b = blockIdx.x;
    if (a.flags[b] == 0) return;
    const int n = o.n, ns = o.ns, m = o.m, lam = o.lambda, pc = o.pop_count;
    if (a.best_x_out)
        for (int k = threadIdx.x; k < n; k += blockDim.x) a.best_x_out[(size_t)b * n + k] = o.best_x[(size_t)b * ns + k];
    const Scalars old = o.sc[b];
    __syncthreads();                                             // every read of the retiring instance is done
    if (threadIdx.x == 0) {
        if (a.best_f_out) a.best_f_out[b] = old.best_f;
        Scalars s;
        s.sigma = a.sigma0 ? a.sigma0[b] : a.sigma_default;
        s.s = 0.0;
        s.best_f = 1.7976931348623157e308;                         // DBL_MAX, as create
        s.counteval = 0;
        s.itr = 0; s.live = 0; s.best_local = 0;
        s.epoch = old.epoch + 1;                                 // a fresh deviate stream from itr = 0
        o.sc[b] = s;
    }
    if (a.ends && threadIdx.x < 6) a.d_ends[(size_t)b * 6 + threadIdx.x] = a.ends[(size_t)b * 6 + threadIdx.x];
    for (int k = threadIdx.x; k < ns; k += blockDim.x) o.xmean[(size_t)b * ns + k] = k < n ? a.x0[(size_t)b * n + k] : 0.0;
    reset_zero4(o.pc + (size_t)b * ns, ns);
    reset_zero4(o.best_x + (size_t)b * ns, ns);
    reset_zero4(o.V + (size_t)b * m * ns, (size_t)m * ns);
    reset_zero4(o.P + (size_t)b * m * ns, (size_t)m * ns);
    reset_zero4(o.VPs + (size_t)b * m * 2 * ns, (size_t)m * 2 * ns);   // the pair mirror of live = 0: no mirror_dirty
    reset_zero(o.Nj + (size_t)b * m, m);
    reset_zero(o.Lj + (size_t)b * m, m);
    reset_zero(o.Njf + (size_t)b * m, m);
    reset_zero(o.Njs + (size_t)b * m, m);
    reset_zero(o.t + (size_t)b * m, m);
    reset_zero(o.vec + (size_t)b * m, m);
    reset_zero(o.fit + (size_t)b * lam, lam);
    reset_zero(o.fit_sorted + (size_t)b * lam, lam);
    reset_zero(o.prev_fit + (size_t)b * lam, lam);
    reset_zero(o.rank + (size_t)b * lam, lam);
    reset_zero(o.arindex + (size_t)b * lam, lam);
    if (o.prev_sorted) reset_zero(o.prev_sorted + (size_t)b * lam, lam);
    reset_zero(o.ncoll + (size_t)b * pc, pc);
    reset_zero(o.nsamp + (size_t)b * pc, pc);
    if (o.G) reset_zero(o.G + (size_t)b * GRAM_KS * m * m, (size_t)GRAM_KS * m * m);
    if (o.Cf) reset_zero(o.Cf + (size_t)b * m * m, (size_t)m * m);
}

}  // namespace lmcma

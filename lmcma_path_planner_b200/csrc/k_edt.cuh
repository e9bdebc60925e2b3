// k_edt.cuh — occupancy grid -> exact Euclidean distance field on the device (SURVEY.md section 8f.1): the step in
// front of the hot path that the reference does with a two-pass 8SSEDT on a fixed 100 x 100 grid (planner.cpp:
// 403-490) or with dynamicEDT3D (planner.cpp:81-87, 305-307).  Separable, exact in integer arithmetic:
//   pass x   per line, distance to the nearest obstacle along x (two warp-level scans, coalesced)
//   pass y,z per line, lower envelope of the parabolas (u - i)^2 + G(i) (Meijster, Roerdink & Hesselink 2000),
//            one thread per line, lines laid out so that the threads of a warp touch consecutive addresses
// then dist = sqrt(d2) (FP64 sqrt, rounded once to FP32 — what scipy's exact EDT gives), optional clamp, and the
// conversion to the bricked map storage k_cost reads (k_brick) without a host round trip.
#pragma once
#include <cfloat>
#include "lmcma_common.cuh"

namespace lmcma {

// Squared distances are unsigned 32-bit: the largest one an accepted grid holds (axes <= 32767 cells) is 3 * 32766^2 =
// 3 220 832 268, past INT_MAX but below EDT_NONE, the "no obstacle" sentinel.  Envelope arithmetic is 64-bit.
constexpr unsigned EDT_NONE = 0xffffffffu;   // no obstacle on this line / in this grid: above any real squared distance
constexpr int EDT_FAR = 1 << 29;             // obstacle index of "none" in pass x's scans: farther than any real index
constexpr float EDT_EMPTY = FLT_MAX;         // distance where the grid holds no obstacle at all, unless clamped

// ---- pass x: one warp per line of nx cells (lines = ny * nz), d2[x] = (distance to the nearest obstacle along x)^2
__global__ void __launch_bounds__(256) k_edt_x(const unsigned char* __restrict__ occ, unsigned* __restrict__ d2, int nx, long long nlines) {
    const int lane = threadIdx.x & 31;
    const long long line = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (line >= nlines) return;
    const unsigned char* src = occ + line * nx;
    unsigned* dst = d2 + line * nx;
    // forward: index of the last obstacle at or before x (max-scan), chunk by chunk with a carry
    int carry = -EDT_FAR;
    for (int x0 = 0; x0 < nx; x0 += 32) {
        const int x = x0 + lane;
        int v = (x < nx && src[x]) ? x : -EDT_FAR;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int u = __shfl_up_sync(0xffffffffu, v, o); if (lane >= o) v = max(v, u); }
        v = max(v, carry);
        carry = __shfl_sync(0xffffffffu, v, 31);
        if (x < nx) dst[x] = (v <= -EDT_FAR) ? EDT_FAR : x - v;        // plain distance for now
    }
    // backward: index of the first obstacle at or after x (min-scan from the right)
    carry = EDT_FAR;
    for (int x0 = ((nx - 1) / 32) * 32; x0 >= 0; x0 -= 32) {
        const int x = x0 + lane;
        int v = (x < nx && src[x]) ? x : EDT_FAR;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int u = __shfl_down_sync(0xffffffffu, v, o); if (lane + o < 32) v = min(v, u); }
        v = min(v, carry);
        carry = __shfl_sync(0xffffffffu, v, 0);
        if (x < nx) {
            const int fwd = (int)dst[x], bwd = (v >= EDT_FAR) ? EDT_FAR : v - x;
            const int d = min(fwd, bwd);
            dst[x] = d >= 32768 ? EDT_NONE : (unsigned)(d * d);       // lines longer than 32767 cells are refused at the ABI
        }
    }
}

// ---- pass along an axis of length m with element stride `stride`: lines are enumerated by (inner, outer) with
//      address = outer * outer_stride + inner, inner < n_inner consecutive in memory (coalesced across threads).
//      s / t / gh: scratch of m entries per line, laid out [position][line] for the same reason.
__global__ void __launch_bounds__(128) k_edt_axis(unsigned* __restrict__ d2, int m, long long stride, int n_inner, long long n_outer,
                                                  long long outer_stride, int* __restrict__ s, int* __restrict__ t, unsigned* __restrict__ gh) {
    const long long line = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long nlines = (long long)n_inner * n_outer;
    if (line >= nlines) return;
    const long long inner = line % n_inner, outer = line / n_inner;
    unsigned* base = d2 + outer * outer_stride + inner;
    auto S = [&](int q) -> int& { return s[(long long)q * nlines + line]; };
    auto T = [&](int q) -> int& { return t[(long long)q * nlines + line]; };
    auto G = [&](int q) -> unsigned& { return gh[(long long)q * nlines + line]; };
    // lower envelope: hull point q is the parabola centred at S(q) with height G(q), dominant from T(q) on
    int q = 0;
    S(0) = 0; T(0) = 0; G(0) = base[0];
    for (int u = 1; u < m; ++u) {
        const long long gu = base[(long long)u * stride];
        while (q >= 0) {
            const long long tq = T(q), sq = S(q), gq = G(q);
            const long long f_old = (tq - sq) * (tq - sq) + gq, f_new = (tq - u) * (tq - u) + gu;
            if (f_old > f_new) --q; else break;
        }
        if (q < 0) { q = 0; S(0) = u; T(0) = 0; G(0) = (unsigned)gu; }
        else {
            const long long sq = S(q), gq = G(q);
            // Sep(i, u) = (u^2 - i^2 + G(u) - G(i)) div (2 (u - i)), floor division (numerator may be negative)
            const long long num = (long long)u * u - sq * sq + gu - gq, den = 2 * ((long long)u - sq);
            long long sep = num / den;
            if ((num % den != 0) && ((num < 0) != (den < 0))) --sep;
            const long long w = 1 + sep;
            if (w < m) { ++q; S(q) = u; T(q) = (int)max(w, 0LL); G(q) = (unsigned)gu; }
        }
    }
    for (int u = m - 1; u >= 0; --u) {
        const long long sq = S(q), gq = G(q);
        const long long d = ((long long)u - sq) * ((long long)u - sq) + gq;
        base[(long long)u * stride] = d >= (long long)EDT_NONE ? EDT_NONE : (unsigned)d;
        if (u == T(q)) --q;
    }
}

// ---- d2 -> distance in cells (FP32), optional clamp; no obstacle anywhere -> clamp (or EDT_EMPTY = FLT_MAX when unclamped)
__global__ void __launch_bounds__(256) k_edt_finish(const unsigned* __restrict__ d2, float* __restrict__ dist, long long cells, float clamp) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= cells) return;
    const unsigned v = d2[i];
    float d = v == EDT_NONE ? EDT_EMPTY : (float)sqrt((double)v);
    if (clamp > 0.f) d = fminf(d, clamp);
    dist[i] = d;
}

// ---- row-major distance field -> the bricked storage of the cost map (lmcma_layout.hpp):
//      F32: sign-tagged reciprocal clearance (negative on obstacles); U8: quantised distance
template <int DIMS, int STORAGE>
__global__ void __launch_bounds__(256) k_brick(const float* __restrict__ dist, float* __restrict__ g32, unsigned char* __restrict__ q8,
                                               int nx, int ny, int nz, unsigned nbx, unsigned nby, float c_min, float u8_scale) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long cells = (long long)nx * ny * nz;
    if (i >= cells) return;
    const unsigned x = (unsigned)(i % nx), y = (unsigned)((i / nx) % ny), z = (unsigned)(i / ((long long)nx * ny));
    const float e = dist[i];
    const unsigned o = brick_offset<DIMS, STORAGE>(x, y, z, nbx, nby);
    if (STORAGE == 0) {
        g32[o] = (e > 0.f) ? 1.0f / fmaxf(e, c_min) : -1.0f / c_min;
    } else {
        int v = 0;
        if (e > 0.f) { v = (int)floorf(e / u8_scale); v = min(255, max(1, v)); }
        q8[o] = (unsigned char)v;
    }
}

}  // namespace lmcma

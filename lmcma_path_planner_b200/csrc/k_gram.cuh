// k_gram.cuh — the recompute of the inverse-direction vectors (lmcma.cpp:373-390, 449-463) for shapes whose
// direction rows fit neither the registers nor the shared memory of one SM (C4: m = 77 rows of n = 1500).
// The factor-major sweep of k_update.cuh would then stream every row-step through L2 from a single SM
// (~1 ms).  Every vector of the sweep is a linear combination of the L basis rows
//     b_i = v_i (i < first_stale, unchanged)   |   b_i = pc_i (i >= first_stale, to be recomputed),
// so the whole recurrence can be carried out on L-vectors of coefficients once the Gram matrix G = B B^T is known:
//     v_j . x  =  coef(v_j)^T G coef(x).
//   k_gram     G in FP64 from the FP32 rows, many CTAs (the only pass over the long rows besides the last one)
//   k_coef     the recurrence x <- K x - Lj_j (v_j . x) v_j on coefficient vectors, FP64, one CTA per instance,
//              same factor order as the reference; |v_j|^2 = c_j^T G c_j, Nj / Lj closed forms
//   k_combine  v_i = sum_k C[i][k] b_k for the recomputed rows, FP64 accumulation, many CTAs; also refreshes the
//              sequence-ordered mirror k_sample streams from
// All cancellation (|pc| ~ 10^3 collapsing to |v| ~ 10 once the paths are collinear) happens in FP64 here, so this
// path is also the more accurate one.
#pragma once
#include "lmcma_common.cuh"

namespace lmcma {

constexpr int GRAM_TILE = 16;
constexpr int GRAM_KC = 64;        // columns staged per step
constexpr int GRAM_KS = 8;         // column slices of a tile pair, one CTA each; OptDev::G holds the GRAM_KS partial matrices of an
                                   // instance, k_coef adds them in slice order (no atomics: every rank of a split population
                                   // must form the same bits)

__device__ __forceinline__ const float* basis_row(const OptDev& o, int b, int i, int first_stale) {
    const int slot = o.t[(size_t)b * o.m + i];
    return (i < first_stale ? o.V : o.P) + ((size_t)b * o.m + slot) * o.ns;
}

// grid = (tiles_a, tiles_b, B * GRAM_KS) with tiles_b >= tiles_a used (upper triangle incl. diagonal), 256 threads = 16 x 16 dots
__global__ void __launch_bounds__(256) k_gram(OptDev o) {
    __shared__ float As[GRAM_TILE][GRAM_KC + 1];
    __shared__ float Bs[GRAM_TILE][GRAM_KC + 1];
    const int b = blockIdx.z / GRAM_KS, ks = blockIdx.z - b * GRAM_KS, ta = blockIdx.x, tb = blockIdx.y;
    if (tb < ta) return;
    const int2 hdr = o.gram_hdr[b];
    const int first_stale = hdr.x, live = hdr.y;
    const int a0 = ta * GRAM_TILE, b0 = tb * GRAM_TILE;
    if (a0 >= live || b0 >= live) return;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;       // G[a0 + ty][b0 + tx]
    const int lr = threadIdx.x >> 4, lc = (threadIdx.x & 15) * 4; // loader: 16 rows x 16 float4
    const float* arow = (a0 + lr < live) ? basis_row(o, b, a0 + lr, first_stale) : nullptr;
    const float* brow = (b0 + lr < live) ? basis_row(o, b, b0 + lr, first_stale) : nullptr;
    double acc0 = 0.0, acc1 = 0.0;
    const int steps = (o.ns + GRAM_KC - 1) / GRAM_KC, per = (steps + GRAM_KS - 1) / GRAM_KS;   // this slice: steps [ks per, (ks + 1) per)
    const int c_end = min(o.ns, (ks + 1) * per * GRAM_KC);
    for (int c0 = ks * per * GRAM_KC; c0 < c_end; c0 += GRAM_KC) {
        float4 av = make_float4(0.f, 0.f, 0.f, 0.f), bv = av;
        if (arow && c0 + lc < o.ns) av = *reinterpret_cast<const float4*>(arow + c0 + lc);
        if (brow && c0 + lc < o.ns) bv = *reinterpret_cast<const float4*>(brow + c0 + lc);
        __syncthreads();
        As[lr][lc] = av.x; As[lr][lc + 1] = av.y; As[lr][lc + 2] = av.z; As[lr][lc + 3] = av.w;
        Bs[lr][lc] = bv.x; Bs[lr][lc + 1] = bv.y; Bs[lr][lc + 2] = bv.z; Bs[lr][lc + 3] = bv.w;
        __syncthreads();
#pragma unroll 8
        for (int c = 0; c < GRAM_KC; c += 2) {
            acc0 = fma((double)As[ty][c], (double)Bs[tx][c], acc0);
            acc1 = fma((double)As[ty][c + 1], (double)Bs[tx][c + 1], acc1);
        }
    }
    const int ia = a0 + ty, ib = b0 + tx;
    if (ia < live && ib < live) {
        double* G = o.G + ((size_t)b * GRAM_KS + ks) * o.m * o.m;
        const double g = acc0 + acc1;
        G[(size_t)ia * o.m + ib] = g;
        G[(size_t)ib * o.m + ia] = g;
    }
}

// one CTA per instance, 8 lanes per basis row.  Row i of C = coefficients of the current x_i; row i of U = G coef(x_i),
// carried along with every update (x <- K x - e v_j  =>  U_i <- K U_i - e U_j), so that when a row becomes final its
// W = G coef(v) is already there and v_j . x_i = coef(v_j) . U_i needs no pass over G: ONE phase and ONE barrier per factor.
// What paces it is the dependent chain of a factor (loads, FMA chain, shuffle rounds, update, the finished row's |v|^2,
// sqrt and divide, barrier: ~2500 cycles, ncu: half of the warp samples wait at the barrier), not the FP64 pipe (64 FMAs
// per clock and SM, tools/micro/dfma.cu); the instructions per factor are kept minimal:
//  * a pending row is held as y = x / K^j (every pending row has had the same j factors), which turns both updates into
//    ONE fused multiply-add per element, y <- y - (Lj_j / K)(v_j . y) v_j, and drops the K c_i[i] term; a row is scaled back
//    by K^i when it becomes final;
//  * only the support is touched: coef(v_j) and coef(x_i) live on {0 .. j} (and i); U_i is a full row.
// A pending row lives in the REGISTERS of its 8 lanes (lane `sub` holds the elements k = sub + 8 t, t < TMAX, of both
// vectors, loops unrolled with block-uniform bounds); only final rows are in shared memory (U, C as L x LP doubles, read
// as broadcasts by every pending row).  Earlier versions: all rows in shared memory with W_j = G c_j and |v_j|^2
// recomputed in two more block-wide phases per factor (126 us for C4's 77 rows); registers without the scaling and the
// support bounds (122 us, 5 FP64 instructions per element and factor over the padded row).
template <int TMAX>
__global__ void __launch_bounds__(64 * TMAX) k_coef(OptDev o) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int b = blockIdx.x, tid = threadIdx.x, nthr = blockDim.x;
    const int m = o.m;
    const int2 hdr = o.gram_hdr[b];
    const int first_stale = hdr.x, L = hdr.y;
    const int LP = m | 1;
    double* Us = reinterpret_cast<double*>(smem_raw);             // [L][LP]: final rows only
    double* Cs = Us + (size_t)m * LP;                             // [L][LP]: recomputed final rows only
    double* lj_s = Cs + (size_t)m * LP;                           // [L]: Lj / K
    double* nv_s = lj_s + m;                                      // [L]
    const double* G = o.G + (size_t)b * GRAM_KS * m * m;
    const int* order = o.t + (size_t)b * m;
    const int sub = tid & 7, i = tid >> 3;                        // this thread's row (8 aligned lanes of one warp per row)
    const bool row_on = i < L;
    const double Kd = o.K, invK = 1.0 / o.K, r = nj_ratio(o), am = o.M;
    double c[TMAX], u[TMAX];
#pragma unroll
    for (int t = 0; t < TMAX; ++t) {
        const int k = sub + 8 * t;
        double g = 0.0;
        if (row_on && k < L) {
#pragma unroll
            for (int ks = 0; ks < GRAM_KS; ++ks) g += G[((size_t)ks * m + i) * m + k];   // the column slices of k_gram, in slice order
        }
        u[t] = g;                                                 // coef(x_i) = e_i: U_i = row i of G
        c[t] = (row_on && k == i) ? 1.0 : 0.0;
        if (row_on && i < first_stale && k < L) Us[i * LP + k] = g;   // unchanged rows: W_i = row i of G, coef = e_i
    }
    for (int j = tid; j < L; j += nthr) lj_s[j] = (j < first_stale) ? o.Lj[(size_t)b * m + order[j]] * invK : 0.0;
    auto oct_sum = [&](double v) {
        v += __shfl_xor_sync(0xffffffffu, v, 1);
        v += __shfl_xor_sync(0xffffffffu, v, 2);
        v += __shfl_xor_sync(0xffffffffu, v, 4);
        return v;
    };
    // a row that has had all its factors applied is scaled back (kp = K^i) and goes to shared memory; |v|^2 = c . U,
    // Lj (cancellation-free form of lmcma.cpp:388-389).  Warp-collective (shuffles); `mine` is uniform over a row's 8 lanes
    auto finish = [&](bool mine, double kp) {
        double s0 = 0.0;
        if (mine) {
#pragma unroll
            for (int t = 0; t < TMAX; ++t) {
                const int k = sub + 8 * t;
                const double cv = c[t] * kp, uv = u[t] * kp;
                if (k < L) { Cs[i * LP + k] = cv; Us[i * LP + k] = uv; }
                if (8 * t <= i) s0 = fma(cv, uv, s0);              // c is 0 beyond the row's support {0 .. i}
            }
        }
        s0 = oct_sum(s0);
        if (mine && sub == 0) {
            const double nv = s0 > 0.0 ? s0 : 0.0;
            const double t2 = sqrt(1.0 + r * nv);
            nv_s[i] = nv;
            lj_s[i] = r / (am * t2 * (t2 + 1.0)) * invK;
        }
    };
    if (first_stale == 0) finish(i == 0, 1.0);                    // v_0 = pc_0
    __syncthreads();
    double kp = 1.0;                                              // K^(j+1) inside step j
    // a warp carries 4 consecutive rows: once its last row is final (or all of them are unchanged rows in front of the first
    // stale position) it has nothing left but the barrier — without this every warp issued the shuffles and predicated
    // bodies of every factor, and the one SM of this kernel is short of issue slots (ncu: 184 warp instructions per warp and
    // factor, the samples waiting at the barrier)
    const int warp_last_row = min(L - 1, (tid >> 5) * 4 + 3);
    const bool warp_recomputes = (tid >> 5) * 4 < L && warp_last_row >= first_stale;
    for (int j = 0; j + 1 < L; ++j) {
        kp *= Kd;
        if (!warp_recomputes || warp_last_row <= j) { __syncthreads(); continue; }   // warp-uniform
        // factor j on every pending row i > j: x <- K x - Lj_j (v_j . x) v_j (lmcma.cpp:455-461), on y = x / K^j
        const bool fresh = j >= first_stale;                      // v_j was recomputed in this sweep (else coef(v_j) = e_j)
        const bool on = row_on && i > j && i >= first_stale;
        const double* cj = Cs + j * LP;
        const double* wj = Us + j * LP;
        double cv[TMAX];
        double d = 0.0;
        if (on) {
#pragma unroll
            for (int t = 0; t < TMAX; ++t) {
                if (8 * t <= j) {                                  // block-uniform: the support of coef(v_j) is {0 .. j}
                    const int k = sub + 8 * t;
                    cv[t] = fresh ? ((k <= j) ? cj[k] : 0.0) : ((k == j) ? 1.0 : 0.0);
                    d = fma(cv[t], u[t], d);
                }
            }
        }
        const double e = -lj_s[j] * oct_sum(d);
        if (on) {
#pragma unroll
            for (int t = 0; t < TMAX; ++t) {
                const int k = sub + 8 * t;
                if (8 * t <= j) c[t] = fma(e, cv[t], c[t]);
                if (k < L) u[t] = fma(e, wj[k], u[t]);             // the whole row: W_i[k], k > i, updates the rows behind i
            }
        }
        if (((j + 1) >> 2) == (tid >> 5)) finish(on && i == j + 1, kp);   // row j + 1 is final now (the warp that carries it)
        __syncthreads();
    }
    // ---- outputs: coefficients of the recomputed rows, Nj / Lj (lmcma.cpp:386-389) by slot and by position ----
    double* Cf = o.Cf + (size_t)b * m * m;
    for (int e = tid; e < L * L; e += nthr) { const int i2 = e / L, k = e - i2 * L; if (i2 >= first_stale) Cf[(size_t)i2 * m + k] = (k <= i2) ? Cs[i2 * LP + k] : 0.0; }
    for (int i2 = first_stale + tid; i2 < L; i2 += nthr) {
        const int slot = order[i2];
        const double nj = nj_form(r, am, nv_s[i2]).nj;
        o.Nj[(size_t)b * m + slot] = nj; o.Lj[(size_t)b * m + slot] = lj_s[i2] * Kd;
        o.Njf[(size_t)b * m + slot] = (float)nj; o.Njs[(size_t)b * m + i2] = (float)nj;
    }
}

// v_i = sum_{k <= i} C[i][k] b_k for the recomputed rows: grid = (ceil(nq / 128), ceil(m / COMBINE_ROWS), B), 128 threads,
// each thread one float4 column of COMBINE_ROWS rows; writes V (slot-indexed) and both halves of the mirror.  Bound by the
// walk over the basis rows (one CTA reads rows 0 .. kmax of its column slab in turn), not by the FP64 accumulation: 2 rows
// per CTA (117 CTAs for C4) measured 41 us against 28 us for 8 rows per CTA (30 CTAs).
constexpr int COMBINE_ROWS = 8;
__global__ void __launch_bounds__(128) k_combine(OptDev o) {
    __shared__ double cs[COMBINE_ROWS][128];                        // coefficients of this CTA's rows (m <= 128)
    __shared__ const float* rowp[128];                              // basis row pointers (one dependent load chain, not L)
    const int b = blockIdx.z, nq = o.ns >> 2, q = blockIdx.x * 128 + threadIdx.x;
    const int2 hdr = o.gram_hdr[b];
    const int first_stale = hdr.x, L = hdr.y;
    const int i0 = first_stale + blockIdx.y * COMBINE_ROWS;
    if (i0 >= L) return;
    const int rows = min(COMBINE_ROWS, L - i0), kmax = i0 + rows - 1;
    const double* Cf = o.Cf + (size_t)b * o.m * o.m;
    for (int e = threadIdx.x; e < COMBINE_ROWS * 128; e += 128) { const int r2 = e >> 7, k = e & 127; cs[r2][k] = (r2 < rows && k <= i0 + r2) ? Cf[(size_t)(i0 + r2) * o.m + k] : 0.0; }
    if (threadIdx.x <= kmax) rowp[threadIdx.x] = basis_row(o, b, threadIdx.x, first_stale);
    __syncthreads();
    if (q >= nq) return;
    double acc[COMBINE_ROWS][4];
#pragma unroll
    for (int r2 = 0; r2 < COMBINE_ROWS; ++r2) { acc[r2][0] = acc[r2][1] = acc[r2][2] = acc[r2][3] = 0.0; }
    for (int k0 = 0; k0 <= kmax; k0 += 4) {                         // 4 independent row loads in flight
        float4 bk[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) bk[u] = (k0 + u <= kmax) ? __ldg(reinterpret_cast<const float4*>(rowp[k0 + u]) + q) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const double x = bk[u].x, y = bk[u].y, z = bk[u].z, w = bk[u].w;
            const int k = min(k0 + u, 127);
#pragma unroll
            for (int r2 = 0; r2 < COMBINE_ROWS; ++r2) {
                const double c = cs[r2][k];                         // 0 beyond a row's support
                acc[r2][0] = fma(c, x, acc[r2][0]); acc[r2][1] = fma(c, y, acc[r2][1]);
                acc[r2][2] = fma(c, z, acc[r2][2]); acc[r2][3] = fma(c, w, acc[r2][3]);
            }
        }
    }
    for (int r2 = 0; r2 < rows; ++r2) {
        const int i = i0 + r2, slot = o.t[(size_t)b * o.m + i];
        const float4 v = make_float4((float)acc[r2][0], (float)acc[r2][1], (float)acc[r2][2], (float)acc[r2][3]);
        // V[slot] is not a basis row of any CTA (pending rows are read from P), so it can be written in place
        reinterpret_cast<float4*>(o.V + ((size_t)b * o.m + slot) * o.ns)[q] = v;
        float4* mir = reinterpret_cast<float4*>(o.VPs + ((size_t)b * o.m + i) * 2 * o.ns);
        mir[q] = v;
        mir[nq + q] = reinterpret_cast<const float4*>(o.P + ((size_t)b * o.m + slot) * o.ns)[q];
    }
}

}  // namespace lmcma

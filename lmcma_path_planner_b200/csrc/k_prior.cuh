// k_prior.cuh — the smoothness-prior sampling path of CMABase::sampleStandardNormal (lmcma.cpp:212-218): with a
// covariance prior every deviate vector becomes z <- L z, L = lower Cholesky factor of the prior
// (cholesky + applyCovL, lmcma.cpp:844-864), before computeAz.  For the whole population that is the one dense
// contraction of the path: Zc[rows x n] = Z[rows x n] * L^T.  FP32 on CUDA cores (the deviates feed the 1e-5
// parity contract; TF32 would not), tiled 64 x 64 with 4 x 4 register blocks, skipping the zero upper triangle.
#pragma once
#include "lmcma_common.cuh"

namespace lmcma {

// Z <- N(0,1), the samplers' deviates (philox_deviate4): grid = (ceil(nq / 128) x pop_count, 1, B), the column tile
// fastest.  The rows share grid x with the column tiles, in the order a (tiles, rows) grid would launch them: pop_count
// reaches 65 536, past the 65 535 that y and z take.  With OptDev::only, the instances it does not flag keep their Z.
__global__ void __launch_bounds__(128) k_gauss(OptDev o) {
    const int nq = o.ns >> 2, tiles = (nq + 127) >> 7;
    const int row = blockIdx.x / tiles, q = (blockIdx.x - row * tiles) * 128 + threadIdx.x, b = blockIdx.z;
    if (q >= nq || (o.only && o.only[b] == 0)) return;
    const int itr = o.sc[b].itr, epoch = o.sc[b].epoch;
    float4 v;
    philox_deviate4(o, b, row, q, itr, epoch, v);
    reinterpret_cast<float4*>(o.Z + ((size_t)b * o.pop_count + row) * o.ns)[q] = v;
}

// Zc[r][i] = sum_{k <= i} L[i][k] Z[r][k];  L: n x ns row-major FP32 (zero above the diagonal and in the padding)
// grid = ceil(ns / 64) x ceil(rows / 64) blocks on x, the column tile fastest (the order of a (columns, rows) grid, which
// keeps the long last column tiles apart), 256 threads: rows = B x pop_count can pass the 65 535 x 64 that y would take
__global__ void __launch_bounds__(256) k_prior(const float* __restrict__ Z, const float* __restrict__ Lf, float* __restrict__ Zc,
                                               int rows, int n, int ns) {
    __shared__ float zs[16][64 + 4];      // [k][r]
    __shared__ float ls[16][64 + 4];      // [k][i]
    const int tiles = (ns + 63) >> 6, rt = blockIdx.x / tiles;
    const int r0 = rt * 64, i0 = (blockIdx.x - rt * tiles) * 64;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;          // 16 x 16 threads, 4 x 4 outputs each
    float acc[4][4];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[a][c] = 0.f;
    const int kend = min(n, i0 + 64);                                // columns k > i contribute nothing
    const int lr = threadIdx.x >> 2, lk = (threadIdx.x & 3) * 4;     // loader: 64 rows x 4 float4 of k
    for (int k0 = 0; k0 < kend; k0 += 16) {
        float4 zv = make_float4(0.f, 0.f, 0.f, 0.f), lv = zv;
        if (r0 + lr < rows && k0 + lk < ns) zv = *reinterpret_cast<const float4*>(Z + (size_t)(r0 + lr) * ns + k0 + lk);
        if (i0 + lr < n && k0 + lk < ns) lv = *reinterpret_cast<const float4*>(Lf + (size_t)(i0 + lr) * ns + k0 + lk);
        __syncthreads();
        zs[lk][lr] = zv.x; zs[lk + 1][lr] = zv.y; zs[lk + 2][lr] = zv.z; zs[lk + 3][lr] = zv.w;
        ls[lk][lr] = lv.x; ls[lk + 1][lr] = lv.y; ls[lk + 2][lr] = lv.z; ls[lk + 3][lr] = lv.w;
        __syncthreads();
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            const float4 zr = *reinterpret_cast<const float4*>(&zs[k][ty * 4]);
            const float4 li = *reinterpret_cast<const float4*>(&ls[k][tx * 4]);
            const float zz[4] = {zr.x, zr.y, zr.z, zr.w}, ll[4] = {li.x, li.y, li.z, li.w};
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int c = 0; c < 4; ++c) acc[a][c] = fmaf(zz[a], ll[c], acc[a][c]);
        }
    }
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        const int r = r0 + ty * 4 + a, i = i0 + tx * 4;
        if (r < rows && i < ns) {
            float4 out = make_float4(acc[a][0], acc[a][1], acc[a][2], acc[a][3]);
            if (i + 1 >= n) out.y = 0.f;
            if (i + 2 >= n) out.z = 0.f;
            if (i + 3 >= n) out.w = 0.f;
            if (i >= n) out.x = 0.f;
            *reinterpret_cast<float4*>(Zc + (size_t)r * ns + i) = out;
        }
    }
}

}  // namespace lmcma

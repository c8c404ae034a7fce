// Skinny products that are really reductions: HBM-bound, one pass over the tall operand.
//
// The generic FFMA GEMM (gemm_simt.cu) tiles 64 x 64 outputs; products with a handful of outputs per
// row (critic head N = 1, policy head N = nb_action, position features K = 2) leave 60 of its 64
// columns idle and ran at 150-470 us per launch at T*M = 65 536 rows (ncu launch list, config c4) for
// 100 MB of traffic (~16 us of HBM time).  These kernels read the tall operand once, coalesced:
//   rowdot    Y[r]      = X[r,:] . w + b                           (critic.3 forward, N = 1)
//   tn_small  dW[n,k]  += sum_r dY[r,n] X[r,k],  N <= 8            (head .3 weight gradients)
//   tn_tiny   dW[n,k]  += sum_r dY[r,n] X[r,k],  N * K <= 32       (map_pos.0 weight gradient, K = 2)
// All exact fp32 (FFMA), accumulation order differs from the reference's (tolerance 1e-3, see tests).
#include <stdlib.h>

#include "common.cuh"

namespace marlc {

// one warp per row, 128-bit loads when the row is 16-byte aligned
__global__ void __launch_bounds__(256) rowdot_kernel(const float* __restrict__ X, long ldx, const float* __restrict__ w,
                                                     const float* __restrict__ bias, float* __restrict__ Y, long ldy,
                                                     int R, int K, int accumulate) {
    const int lane = threadIdx.x & 31;
    const int warps = (gridDim.x * blockDim.x) >> 5;
    const bool vec = ((K & 3) == 0) && ((ldx & 3) == 0) && (((uintptr_t)X & 15) == 0) && (((uintptr_t)w & 15) == 0);
    for (int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < R; r += warps) {
        const float* x = X + (long)r * ldx;
        float s = 0.f;
        if (vec) {
            for (int k = lane * 4; k < K; k += 128) {
                const float4 a = *reinterpret_cast<const float4*>(x + k);
                const float4 b = __ldg(reinterpret_cast<const float4*>(w + k));
                s = fmaf(a.x, b.x, s); s = fmaf(a.y, b.y, s); s = fmaf(a.z, b.z, s); s = fmaf(a.w, b.w, s);
            }
        } else {
            for (int k = lane; k < K; k += 32) s = fmaf(x[k], __ldg(w + k), s);
        }
        s = warp_sum(s);
        if (lane == 0) {
            if (bias) s += bias[0];
            float* y = Y + (long)r * ldy;
            *y = accumulate ? *y + s : s;
        }
    }
}

int rowdot(const float* X, long ldx, const float* w, const float* bias, float* Y, long ldy, int R, int K, int accumulate,
           cudaStream_t s) {
    if (R <= 0) return 0;
    const int blocks = min((R + 7) / 8, 4 * MARLC_SMS);
    rowdot_kernel<<<blocks, 256, 0, s>>>(X, ldx, w, bias, Y, ldy, R, K, accumulate);
    MARLC_LAUNCH_CHECK();
    return 0;
}

// dW[n,k] += sum_r dY[r,n] X[r,k] for N <= 8: block = 32 columns x 8 row lanes; every thread walks its
// rows (coalesced 128-byte reads of X, broadcast reads of the dY row), partial sums of the 8 row lanes
// meet in shared memory, one atomicAdd per output per block.
template <int N>
__global__ void __launch_bounds__(256) tn_small_kernel(const float* __restrict__ dY, long lddy,
                                                       const float* __restrict__ X, long ldx, float* __restrict__ dW,
                                                       long lddw, int R, int K, int rows_per_block) {
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int k = blockIdx.x * 32 + tx;
    const int r0 = blockIdx.y * rows_per_block, r1 = min(R, r0 + rows_per_block);
    float acc[N];
#pragma unroll
    for (int n = 0; n < N; ++n) acc[n] = 0.f;
    if (k < K) {
#pragma unroll 4
        for (int r = r0 + ty; r < r1; r += 8) {
            const float x = X[(long)r * ldx + k];
            const float* d = dY + (long)r * lddy;
#pragma unroll
            for (int n = 0; n < N; ++n) acc[n] = fmaf(__ldg(d + n), x, acc[n]);
        }
    }
    __shared__ float red[8][N][33];
#pragma unroll
    for (int n = 0; n < N; ++n) red[ty][n][tx] = acc[n];
    __syncthreads();
    for (int e = threadIdx.x; e < N * 32; e += 256) {
        const int n = e >> 5, c = e & 31;
        if (blockIdx.x * 32 + c >= K) continue;
        float s = 0.f;
#pragma unroll
        for (int j = 0; j < 8; ++j) s += red[j][n][c];
        atomicAdd(dW + (long)n * lddw + blockIdx.x * 32 + c, s);
    }
}

// N * K <= 32 outputs: every thread keeps all of them, rows grid-strided; warp shuffle + one atomicAdd
// per output per warp.
__global__ void __launch_bounds__(256) tn_tiny_kernel(const float* __restrict__ dY, long lddy, const float* __restrict__ X,
                                                      long ldx, float* __restrict__ dW, long lddw, int R, int N, int K) {
    float acc[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) acc[i] = 0.f;
    const int stride = gridDim.x * blockDim.x;
    for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < R; r += stride) {
        const float* d = dY + (long)r * lddy;
        const float* x = X + (long)r * ldx;
        float xv[32];
#pragma unroll
        for (int k = 0; k < 32; ++k) xv[k] = k < K ? x[k] : 0.f;
#pragma unroll
        for (int i = 0; i < 32; ++i) {
            // i = n * K + k without a division: walk n and k together
            if (i < N * K) {
                const int n = i / K, k = i - n * K;
                acc[i] = fmaf(d[n], xv[k], acc[i]);
            }
        }
    }
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int i = 0; i < 32; ++i) {
        if (i < N * K) {
            const float s = warp_sum(acc[i]);
            if (lane == 0 && s != 0.f) { const int n = i / K, k = i - n * K; atomicAdd(dW + (long)n * lddw + k, s); }
        }
    }
}

// Returns 1 if the shape is not one of the skinny cases (caller falls back to the generic GEMM).
int tn_skinny(const float* dY, long lddy, const float* X, long ldx, float* dW, long lddw, int R, int N, int K,
              int accumulate, cudaStream_t s, bool* done) {
    *done = false;
    if (R <= 0 || N <= 0 || K <= 0) return 0;
    const bool tiny = N * K <= 32 && K <= 32;
    const bool small = N <= 8;
    if (!tiny && !small) return 0;
    if (!accumulate) {
        if (lddw == K) MARLC_CUDA(cudaMemsetAsync(dW, 0, sizeof(float) * (size_t)N * K, s));
        else MARLC_CUDA(cudaMemset2DAsync(dW, sizeof(float) * lddw, 0, sizeof(float) * K, N, s));
    }
    if (tiny) {
        const int blocks = max(1, min((R + 255) / 256, 2 * MARLC_SMS));
        tn_tiny_kernel<<<blocks, 256, 0, s>>>(dY, lddy, X, ldx, dW, lddw, R, N, K);
        MARLC_LAUNCH_CHECK();
        *done = true;
        return 0;
    }
    const int kb = (K + 31) / 32;
    int rb = max(1, min((R + 63) / 64, (4 * MARLC_SMS + kb - 1) / kb));  // >= 64 rows per block, ~4 blocks per SM
    const int rows_per_block = ((R + rb - 1) / rb + 7) / 8 * 8;
    rb = (R + rows_per_block - 1) / rows_per_block;
    const dim3 grid(kb, rb);
#define TN_SMALL(NV) case NV: tn_small_kernel<NV><<<grid, 256, 0, s>>>(dY, lddy, X, ldx, dW, lddw, R, K, rows_per_block); break;
    switch (N) {
        TN_SMALL(1) TN_SMALL(2) TN_SMALL(3) TN_SMALL(4) TN_SMALL(5) TN_SMALL(6) TN_SMALL(7) TN_SMALL(8)
    }
#undef TN_SMALL
    MARLC_LAUNCH_CHECK();
    *done = true;
    return 0;
}

}  // namespace marlc

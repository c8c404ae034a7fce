// Layer-wise backward of the feature extractor, batched over ALL T*M windows of the episode.
//
// The per-window fused backward (cnn.cu::cnn_bwd_kernel) spends its time in FFMA loops for the
// conv input gradient.  Here every conv product is a tensor-core GEMM over all windows instead:
//     dCol_l = dY_l . W_l              [P*npos_l, cout_l] x [cout_l, cin_l*9]     (input gradient)
//     dW_l  += dY_l^T . col_l          reduction over P*npos_l rows                (weight gradient)
// and the only SIMT work left is element-wise per window (one warp per window, this file):
//   * col2im gather of dCol_{l+1} -> dA_l (or the rows of dU for the top layer),
//   * GroupNorm + SiLU backward -> dY_l (row layout for the GEMMs) and the per-window
//     dgamma / dbeta partials,
//   * im2col of the recomputed activation A_l -> col_{l+1} (operand of dW_{l+1}).
#include <stdlib.h>

#include <algorithm>

#include "common.cuh"
#include "kernels.cuh"

namespace marlc {

constexpr float GN_EPS2 = 1e-5f;

struct CnnBwdLayerKernelArgs {
    CnnBwdLayerArgs a;
    int total, npos, npn, per_warp;  // per_warp: floats of smem per warp (3 * total rounded + staged dCol block)
    FastDiv d_npos, d_ho, d_co, d_kk, d_hon;  // index decompositions without runtime division
};

// MARLC_CNNBWD_DIV=1 selects the runtime-division instantiation (A/B timing only).
static bool cnn_bwd_use_div() {
    const char* e = getenv("MARLC_CNNBWD_DIV");
    return e && e[0] == '1';
}
#define MARLC_DIV(n, fd, d) (FAST ? (fd).div(n) : (n) / (d))

template <bool FAST>
__global__ void __launch_bounds__(256) cnn_bwd_layer_kernel(const CnnBwdLayerKernelArgs ka) {
    extern __shared__ float sm[];
    const CnnBwdLayerArgs& a = ka.a;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpc = blockDim.x >> 5;
    const int p = blockIdx.x * wpc + warp;
    const int total = ka.total, npos = ka.npos, ho = a.ho, co_n = a.cout;
    float* cta_acc = sm + (size_t)wpc * ka.per_warp;  // [3][cout]: dgamma, dbeta, dbias of this CTA's windows
    const bool fold = a.d_gn_w != nullptr;
    if (fold) {
        for (int i = threadIdx.x; i < 3 * co_n; i += blockDim.x) cta_acc[i] = 0.f;
        __syncthreads();
    }
    if (p < a.P) {
    float* xh = sm + (size_t)warp * ka.per_warp;  // y, then xhat
    float* dz = xh + total;                       // dA, then dz, then dy
    float* act = dz + total;                      // SiLU(GN(y))
    // ---- 1. load y and the incoming gradient dA_l
    const float* yg = a.Y + (long)p * total;
    if (a.dOut) {
        const float* go = a.dOut + (long)p * a.lddo;
        for (int e = lane; e < total; e += 32) { xh[e] = yg[e]; dz[e] = go[e]; }
    } else {
        // col2im: dA[c, iy, ix] = sum over taps (ky,kx) with (iy+1-ky, ix+1-kx) even and in range.
        // The window's dCol block (npn x cout*9 floats, contiguous) is first staged in shared memory
        // with coalesced 128-bit loads, all in flight together: gathering the taps straight from
        // global memory serialised ~9 dependent L2 round trips per element.
        const int hon = a.ho_next, npn = ka.npn, kk = co_n * 9;
        float* dc = xh + 3 * ((total + 3) & ~3);  // 16-byte aligned: per_warp and the rounded sizes are multiples of 4
        {
            const float* src = a.dColNext + (long)p * npn * kk;
            const int n = npn * kk;
            if ((n & 3) == 0 && ((reinterpret_cast<uintptr_t>(src) & 15) == 0)) {
                const float4* s4 = reinterpret_cast<const float4*>(src);
                float4* d4 = reinterpret_cast<float4*>(dc);
#pragma unroll 4
                for (int i = lane; i < (n >> 2); i += 32) d4[i] = __ldg(s4 + i);
            } else {
                for (int i = lane; i < n; i += 32) dc[i] = __ldg(src + i);
            }
        }
        for (int e = lane; e < total; e += 32) xh[e] = yg[e];
        __syncwarp();
        for (int e = lane; e < total; e += 32) {
            const int c = MARLC_DIV(e, ka.d_npos, npos), pos = e - c * npos, iy = MARLC_DIV(pos, ka.d_ho, ho),
                      ix = pos - iy * ho;
            float acc = 0.f;
#pragma unroll
            for (int ky = 0; ky < 3; ++ky) {
                const int ty = iy + 1 - ky;
                if (ty < 0 || (ty & 1) || (ty >> 1) >= hon) continue;
#pragma unroll
                for (int kx = 0; kx < 3; ++kx) {
                    const int tx = ix + 1 - kx;
                    if (tx < 0 || (tx & 1) || (tx >> 1) >= hon) continue;
                    acc += dc[((ty >> 1) * hon + (tx >> 1)) * kk + c * 9 + ky * 3 + kx];
                }
            }
            dz[e] = acc;
        }
    }
    __syncwarp();
    // ---- 2. GroupNorm + SiLU backward, group by group (a group's channels are contiguous)
    const int G = a.groups, cpg = co_n / G, ng = cpg * npos;
    const float inv = 1.0f / (float)ng;
    for (int g = 0; g < G; ++g) {
        float* xg = xh + g * ng;
        float* dg = dz + g * ng;
        float* ag = act + g * ng;
        float s = 0.f;
        for (int e = lane; e < ng; e += 32) s += xg[e];
        const float mean = warp_sum(s) * inv;
        float v = 0.f;
        for (int e = lane; e < ng; e += 32) { const float d = xg[e] - mean; v += d * d; }
        const float rstd = 1.0f / sqrtf(warp_sum(v) * inv + GN_EPS2);
        float s1 = 0.f, s2 = 0.f;
        for (int e = lane; e < ng; e += 32) {
            const int c = g * cpg + MARLC_DIV(e, ka.d_npos, npos);
            const float gam = a.gn_w[c];
            const float x = (xg[e] - mean) * rstd, z = x * gam + a.gn_b[c];
            const float sg = sigmoidf_(z);
            ag[e] = z * sg;
            const float d = dg[e] * (sg * (1.f + z * (1.f - sg)));
            xg[e] = x;
            dg[e] = d;
            s1 += d * gam;
            s2 += d * gam * x;
        }
        s1 = warp_sum(s1) * inv;
        s2 = warp_sum(s2) * inv;
        __syncwarp();
        // per-channel partials for dgamma / dbeta (lanes over the group's channels)
        for (int cc = lane; cc < cpg; cc += 32) {
            float t1 = 0.f, t2 = 0.f;
            for (int q = 0; q < npos; ++q) { const float d = dg[cc * npos + q]; t1 += d * xg[cc * npos + q]; t2 += d; }
            if (fold) {
                atomicAdd(&cta_acc[g * cpg + cc], t1);
                atomicAdd(&cta_acc[co_n + g * cpg + cc], t2);
            } else {
                float* gp = a.gnpart + (long)p * 2 * co_n;
                gp[g * cpg + cc] = t1;
                gp[co_n + g * cpg + cc] = t2;
            }
        }
        __syncwarp();
        for (int e = lane; e < ng; e += 32) {
            const int c = g * cpg + MARLC_DIV(e, ka.d_npos, npos);
            dg[e] = rstd * (dg[e] * a.gn_w[c] - s1 - xg[e] * s2);
        }
        if (fold) {  // conv bias gradient: sum of dY over the positions of each channel
            __syncwarp();
            for (int cc = lane; cc < cpg; cc += 32) {
                float t3 = 0.f;
                for (int q = 0; q < npos; ++q) t3 += dg[cc * npos + q];
                atomicAdd(&cta_acc[2 * co_n + g * cpg + cc], t3);
            }
        }
    }
    __syncwarp();
    // ---- 3. dY rows [pos][co] (GEMM layout), coalesced
    {
        float* dyg = a.dY + (long)p * total;
        for (int e = lane; e < total; e += 32) {
            const int pos = MARLC_DIV(e, ka.d_co, co_n), c = e - pos * co_n;
            dyg[e] = dz[c * npos + pos];
        }
    }
    // ---- 4. im2col of A_l for the weight gradient of layer l+1
    if (a.colNext) {
        const int hon = a.ho_next, npn = ka.npn, kk = co_n * 9;
        float* cg = a.colNext + (long)p * npn * kk;
        for (int e = lane; e < npn * kk; e += 32) {
            const int o = MARLC_DIV(e, ka.d_kk, kk), r = e - o * kk, c = r / 9, q = r - c * 9, ky = q / 3, kx = q - ky * 3;
            const int oy = MARLC_DIV(o, ka.d_hon, hon);
            const int iy = 2 * oy - 1 + ky, ix = 2 * (o - oy * hon) - 1 + kx;
            cg[e] = (iy >= 0 && iy < ho && ix >= 0 && ix < ho) ? act[c * npos + iy * ho + ix] : 0.f;
        }
    }
    }  // p < P
    if (fold) {
        __syncthreads();
        for (int i = threadIdx.x; i < co_n; i += blockDim.x) {
            atomicAdd(a.d_gn_w + i, cta_acc[i]);
            atomicAdd(a.d_gn_b + i, cta_acc[co_n + i]);
            atomicAdd(a.d_conv_b + i, cta_acc[2 * co_n + i]);
        }
    }
}

int cnn_bwd_layer(const CnnBwdLayerArgs& a, cudaStream_t s) {
    if (a.P <= 0) return 0;
    CnnBwdLayerKernelArgs ka;
    ka.a = a;
    ka.npos = a.ho * a.ho;
    ka.total = a.cout * ka.npos;
    ka.npn = a.ho_next * a.ho_next;
    ka.per_warp = 3 * ((ka.total + 3) & ~3) + (a.dOut ? 0 : ((ka.npn * a.cout * 9 + 3) & ~3));
    int wpc = 8;
    while (wpc > 1 && (size_t)wpc * ka.per_warp * sizeof(float) > 160 * 1024) wpc >>= 1;
    MARLC_CHECK((a.d_gn_w != nullptr) == (a.d_gn_b != nullptr) && (a.d_gn_w != nullptr) == (a.d_conv_b != nullptr) &&
                    (a.d_gn_w != nullptr || a.gnpart != nullptr),
                "cnn_bwd_layer: give either gnpart or all three accumulation targets");
    const size_t smem = ((size_t)wpc * ka.per_warp + 3 * a.cout) * sizeof(float);
    MARLC_CHECK(smem <= 200 * 1024, "cnn_bwd_layer: layer too large for shared memory (%zu B)", smem);
    ka.d_npos = FastDiv((unsigned)ka.npos);
    ka.d_ho = FastDiv((unsigned)a.ho);
    ka.d_co = FastDiv((unsigned)a.cout);
    ka.d_kk = FastDiv((unsigned)(a.cout * 9));
    ka.d_hon = FastDiv((unsigned)std::max(a.ho_next, 1));
    // FastDiv exactness: the largest dividends are total (/ npos, / cout) and npn * kk (/ kk)
    const long nmax = std::max((long)ka.total, (long)ka.npn * a.cout * 9);
    const bool fast = FastDiv::exact_up_to(nmax, std::max(std::max(ka.npos, a.cout * 9), 1)) && !cnn_bwd_use_div();
    static size_t attr = 0;
    if (smem > 48 * 1024 && smem > attr) {
        MARLC_CUDA(cudaFuncSetAttribute(cnn_bwd_layer_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        MARLC_CUDA(cudaFuncSetAttribute(cnn_bwd_layer_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr = smem;
    }
    if (fast) cnn_bwd_layer_kernel<true><<<(a.P + wpc - 1) / wpc, wpc * 32, smem, s>>>(ka);
    else cnn_bwd_layer_kernel<false><<<(a.P + wpc - 1) / wpc, wpc * 32, smem, s>>>(ka);
    MARLC_LAUNCH_CHECK();
    return 0;
}

// im2col of the input windows (operand of the first layer's weight gradient):
// col[(p*npos + o), ci*9 + ky*3 + kx] = window_p[ci, 2oy-1+ky, 2ox-1+kx] (0 outside the window)
// Rows are padded with zeros to kkp = round_up(cin*9, 4) floats so that the matrix is a TMA-addressable
// (16-byte row pitch) operand of the tensor-core weight-gradient GEMM: the 27-float rows of an RGB
// first layer otherwise sent that product to the FFMA kernel (470 us at 65 536 windows).
template <bool FAST, bool PATCH>
__global__ void __launch_bounds__(256) cnn_im2col_input_kernel(const CnnWindows win, float* __restrict__ col, int P,
                                                               int cin, int ho, FastDiv d_kk, FastDiv d_ho) {
    const int lane = threadIdx.x & 31;
    const int p = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (p >= P) return;
    long chan;
    int row;
    const float* src = cnn_window<PATCH>(win, p, chan, row);
    const int f = win.f, kk = cin * 9, kkp = (kk + 3) & ~3, npos = ho * ho;
    float* cg = col + (long)p * npos * kkp;
    for (int e = lane; e < npos * kkp; e += 32) {
        const int o = MARLC_DIV(e, d_kk, kkp), r = e - o * kkp, c = r / 9, q = r - c * 9, ky = q / 3, kx = q - ky * 3;
        const int oy = MARLC_DIV(o, d_ho, ho);
        const int iy = 2 * oy - 1 + ky, ix = 2 * (o - oy * ho) - 1 + kx;
        cg[e] = (r < kk && iy >= 0 && iy < f && ix >= 0 && ix < f) ? __ldg(src + c * chan + (long)iy * row + ix) : 0.f;
    }
}

int cnn_im2col_input(const CnnWindows& win, float* col, int P, int cin, int ho, cudaStream_t s) {
    if (P <= 0) return 0;
    const int kkp = (cin * 9 + 3) & ~3;
    const FastDiv d_kk((unsigned)kkp), d_ho((unsigned)ho);
    const bool fast = FastDiv::exact_up_to((long long)ho * ho * kkp, kkp) && !cnn_bwd_use_div();
    const unsigned grid = (P * 32 + 255) / 256;
    if (win.patch) {
        if (fast) cnn_im2col_input_kernel<true, true><<<grid, 256, 0, s>>>(win, col, P, cin, ho, d_kk, d_ho);
        else cnn_im2col_input_kernel<false, true><<<grid, 256, 0, s>>>(win, col, P, cin, ho, d_kk, d_ho);
    } else {
        if (fast) cnn_im2col_input_kernel<true, false><<<grid, 256, 0, s>>>(win, col, P, cin, ho, d_kk, d_ho);
        else cnn_im2col_input_kernel<false, false><<<grid, 256, 0, s>>>(win, col, P, cin, ho, d_kk, d_ho);
    }
    MARLC_LAUNCH_CHECK();
    return 0;
}

}  // namespace marlc

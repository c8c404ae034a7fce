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

// FAST = false: runtime divisions, for sizes where FastDiv is not exact.
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
    const bool fast = FastDiv::exact_up_to(nmax, std::max(std::max(ka.npos, a.cout * 9), 1));
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
    const bool fast = FastDiv::exact_up_to((long long)ho * ho * kkp, kkp);
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

// Image gradient (marlc_episode_image_grad): for conv 3x3, stride 2, padding 1 and the window gather,
//     d_img[b,c,y,x] = sum over windows (t,a) of image b that cover (y,x), in (t,a) order,
//                      sum over taps (ky,kx) with 2*oy-1+ky = y-py, 2*ox-1+kx = x-px, and co,
//                      dY0[t,a,b][oy,ox][co] * W0[co,c,ky,kx].
// One CTA per (image, 32x16 pixel tile), 2 pixels per thread (16x2 pixels per warp in each 16x16 half), the sums
// in registers: no atomics, no intermediate in global memory, and every pixel adds its windows in the same
// order on every call.  The image's windows are tested against the tile IG_THREADS at a time; each chunk's
// overlapping windows are compacted in order into shared memory and consumed before the next chunk is tested,
// so the list never overflows whatever the number of windows per image.  The dY0 blocks of the listed windows
// are staged in shared memory `batch` windows at a time with all loads in flight (read one after the other
// from global memory, each tap waited a full memory latency).  A pixel at window row ly gets 1 tap row (ly
// even: ky = 1) or 2 (ly odd: ky = 2, and ky = 0 unless oy = (ly+1)/2 falls off the last output row), the same
// for columns: the taps are found without division.
constexpr int IG_TW = 32, IG_TH = 16;  // pixel tile: columns, rows
constexpr int IG_THREADS = 256;
constexpr int IG_PX = 2;   // pixels per thread
constexpr int IG_CB = 4;   // input channels per accumulation pass (W_0 rows padded to a multiple of 4)
constexpr int IG_STAGE_BYTES = 24 * 1024;  // dY0 staging budget per CTA
// 3 CTAs per SM: the register budget (80) at which the two pixels' accumulators and taps fit without spills

__global__ void __launch_bounds__(IG_THREADS, 3) cnn_image_grad_kernel(const ImageGradArgs a, FastDiv d_na,
                                                                     FastDiv d_cin, FastDiv d_blk4, int cinp,
                                                                     int batch) {
    extern __shared__ float4 sm4[];
    const int co_n = a.cout, ci_n = a.cin, f = a.f, ho = a.ho, M = a.Na * a.B, n_win = a.T * a.Na;
    const int wsz = co_n * cinp;     // floats per tap of W_0
    const int blk = ho * ho * co_n;  // floats of one window's dY0 block (a multiple of 4)
    float* sw = reinterpret_cast<float*>(sm4);  // W_0 as [tap][cout][cinp], zero in the padded channels
    float* sdy = sw + 9 * wsz;                  // dY0 blocks of `batch` listed windows
    __shared__ int list_p[IG_THREADS], list_y[IG_THREADS], list_x[IG_THREADS];
    __shared__ int warp_n[IG_THREADS / 32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int b = blockIdx.z, y0 = blockIdx.y * IG_TH, x0 = blockIdx.x * IG_TW;
    for (int i = tid; i < 9 * wsz; i += IG_THREADS) sw[i] = 0.f;
    __syncthreads();
    for (int j = tid; j < co_n * ci_n * 9; j += IG_THREADS) {  // source index (co*cin + c)*9 + tap
        const int q = j / 9, tap = j - q * 9, co = d_cin.div(q), c = q - co * ci_n;
        sw[tap * wsz + co * cinp + c] = __ldg(a.w0 + j);
    }
    int py[IG_PX], px[IG_PX];
#pragma unroll
    for (int k = 0; k < IG_PX; ++k) {
        py[k] = y0 + (tid >> 4);
        px[k] = x0 + (tid & 15) + 16 * k;
    }
    const long plane = (long)a.H * a.W;
    float* out = a.d_img + (long)b * a.C * plane;
    const float4* dy4 = reinterpret_cast<const float4*>(a.dY0);
    const int blk4 = blk >> 2;
    for (int c0 = 0; c0 < ci_n; c0 += IG_CB) {
        float acc[IG_PX][IG_CB];
#pragma unroll
        for (int k = 0; k < IG_PX; ++k)
#pragma unroll
            for (int u = 0; u < IG_CB; ++u) acc[k][u] = 0.f;
        for (int w0 = 0; w0 < n_win; w0 += IG_THREADS) {
            // 1. this chunk's windows overlapping the tile, compacted in (t, a) order
            const int w = w0 + tid;
            int p = 0, wy = 0, wx = 0;
            bool hit = false;
            if (w < n_win) {
                const int t = d_na.div(w), ag = w - t * a.Na;
                p = t * M + ag * a.B + b;
                wy = a.pos_hist[2 * (long)p];
                wx = a.pos_hist[2 * (long)p + 1];
                hit = wy < y0 + IG_TH && wy + f > y0 && wx < x0 + IG_TW && wx + f > x0;
            }
            const unsigned bal = __ballot_sync(0xffffffffu, hit);
            __syncthreads();  // the previous chunk's list is consumed
            if (lane == 0) warp_n[warp] = __popc(bal);
            __syncthreads();
            int off = 0, n = 0;
#pragma unroll
            for (int k = 0; k < IG_THREADS / 32; ++k) {
                const int v = warp_n[k];
                off += k < warp ? v : 0;
                n += v;
            }
            if (hit) {
                const int slot = off + __popc(bal & ((1u << lane) - 1u));
                list_p[slot] = p;
                list_y[slot] = wy;
                list_x[slot] = wx;
            }
            for (int i0 = 0; i0 < n; i0 += batch) {
                const int nb = min(batch, n - i0);
                __syncthreads();  // the list is written / the previous batch is consumed
                // 2. stage the batch's dY0 blocks
                float4* s4 = reinterpret_cast<float4*>(sdy);
#pragma unroll 4
                for (int e = tid; e < nb * blk4; e += IG_THREADS) {
                    const int jw = d_blk4.div(e);
                    s4[e] = __ldg(dy4 + (long)list_p[i0 + jw] * blk4 + (e - jw * blk4));
                }
                __syncthreads();
                // 3. the transposed convolution of each staged window at this thread's pixels
                for (int jw = 0; jw < nb; ++jw) {
                    const int wyj = list_y[i0 + jw], wxj = list_x[i0 + jw];
                    const float* g = sdy + jw * blk;
#pragma unroll
                    for (int k = 0; k < IG_PX; ++k) {
                        const int ly = py[k] - wyj, lx = px[k] - wxj;
                        if ((unsigned)ly >= (unsigned)f || (unsigned)lx >= (unsigned)f) continue;
#pragma unroll
                        for (int iy = 0; iy < 2; ++iy) {
                            int ky, oy;
                            if (ly & 1) {
                                ky = iy ? 0 : 2;
                                oy = iy ? (ly + 1) >> 1 : (ly - 1) >> 1;
                                if (oy >= ho) continue;
                            } else {
                                if (iy) continue;
                                ky = 1;
                                oy = ly >> 1;
                            }
#pragma unroll
                            for (int ix = 0; ix < 2; ++ix) {
                                int kx, ox;
                                if (lx & 1) {
                                    kx = ix ? 0 : 2;
                                    ox = ix ? (lx + 1) >> 1 : (lx - 1) >> 1;
                                    if (ox >= ho) continue;
                                } else {
                                    if (ix) continue;
                                    kx = 1;
                                    ox = lx >> 1;
                                }
                                const float4* gp = reinterpret_cast<const float4*>(g + (oy * ho + ox) * co_n);
                                const float4* wp = reinterpret_cast<const float4*>(sw + (ky * 3 + kx) * wsz + c0);
                                const int wstride = cinp >> 2;
                                for (int q = 0; q < (co_n >> 2); ++q) {
                                    const float4 gv = gp[q];
                                    const float gs[4] = {gv.x, gv.y, gv.z, gv.w};
#pragma unroll
                                    for (int u = 0; u < 4; ++u) {
                                        const float4 wv = wp[(4 * q + u) * wstride];
                                        acc[k][0] += gs[u] * wv.x;
                                        acc[k][1] += gs[u] * wv.y;
                                        acc[k][2] += gs[u] * wv.z;
                                        acc[k][3] += gs[u] * wv.w;
                                    }
                                }
                            }
                        }
                    }
                }
            }
        }
#pragma unroll
        for (int k = 0; k < IG_PX; ++k)
            if (py[k] < a.H && px[k] < a.W)
#pragma unroll
                for (int u = 0; u < IG_CB; ++u)
                    if (c0 + u < ci_n) out[(c0 + u) * plane + (long)py[k] * a.W + px[k]] = acc[k][u];
    }
#pragma unroll
    for (int k = 0; k < IG_PX; ++k)  // channels the network does not read (MnistCnn on a 3-channel batch)
        if (py[k] < a.H && px[k] < a.W)
            for (int c = ci_n; c < a.C; ++c) out[c * plane + (long)py[k] * a.W + px[k]] = 0.f;
}

int cnn_image_grad(const ImageGradArgs& a, cudaStream_t s) {
    MARLC_CHECK(a.dY0 && a.w0 && a.pos_hist && a.d_img, "image_grad: null pointer");
    MARLC_CHECK(a.cin >= 1 && a.cin <= a.C && a.cout >= 1 && a.ho == (a.f - 1) / 2 + 1, "image_grad: bad CNN shape");
    // dY0 rows are read as float4: every feature extractor of the package has a multiple of 4 first-layer channels
    MARLC_CHECK((a.cout & 3) == 0 && (reinterpret_cast<uintptr_t>(a.dY0) & 15) == 0,
                "image_grad: the first conv layer needs a multiple of 4 output channels (has %d)", a.cout);
    const unsigned tx = (a.W + IG_TW - 1) / IG_TW, ty = (a.H + IG_TH - 1) / IG_TH;
    MARLC_CHECK(ty <= 65535 && a.B <= 65535, "image_grad: image batch %d x %d rows too large for the grid", a.B, a.H);
    const long n_win = (long)a.T * a.Na;
    MARLC_CHECK(n_win < (1L << 31) && FastDiv::exact_up_to(n_win, a.Na), "image_grad: %ld windows per image", n_win);
    const int cinp = (a.cin + IG_CB - 1) / IG_CB * IG_CB;
    const int blk = a.ho * a.ho * a.cout;
    const int batch = std::max(1, std::min(IG_THREADS, IG_STAGE_BYTES / (blk * (int)sizeof(float))));
    MARLC_CHECK(FastDiv::exact_up_to((long long)batch * blk / 4, blk / 4) &&
                    FastDiv::exact_up_to((long long)a.cout * a.cin * 9, a.cin),
                "image_grad: window block of %d floats too large", blk);
    const size_t smem = ((size_t)9 * a.cout * cinp + (size_t)batch * blk) * sizeof(float);
    MARLC_CHECK(smem <= 200 * 1024, "image_grad: first-layer shapes too large for shared memory (%zu B)", smem);
    static size_t attr = 0;
    if (smem > 48 * 1024 && smem > attr) {
        MARLC_CUDA(cudaFuncSetAttribute(cnn_image_grad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr = smem;
    }
    const dim3 grid(tx, ty, (unsigned)a.B);
    cnn_image_grad_kernel<<<grid, IG_THREADS, smem, s>>>(a, FastDiv((unsigned)a.Na), FastDiv((unsigned)a.cin),
                                                         FastDiv((unsigned)(blk / 4)), cinp, batch);
    MARLC_LAUNCH_CHECK();
    return 0;
}

// W_0 [cout][cin][3][3] -> shared [tap][cout][cinp], zero in the padded channels (nt threads)
__device__ __forceinline__ void stage_w0(float* sw, const float* w0, int co_n, int ci_n, int cinp, FastDiv d_cin,
                                         int nt) {
    const int wsz = co_n * cinp;
    for (int i = threadIdx.x; i < 9 * wsz; i += nt) sw[i] = 0.f;
    __syncthreads();
    for (int j = threadIdx.x; j < co_n * ci_n * 9; j += nt) {  // source index (co*cin + c)*9 + tap
        const int q = j / 9, tap = j - q * 9, co = d_cin.div(q), c = q - co * ci_n;
        sw[tap * wsz + co * cinp + c] = __ldg(w0 + j);
    }
}

// Input channels c0 .. c0+3 of the first conv layer's input gradient at pixel (ly, lx) of one window
// (0 <= ly, lx < f): acc[u] += sum over the pixel's taps, in (ky, kx) order, and over co of
// g[(oy*ho + ox)*cout + co] * W0[co, c0+u, ky, kx].  g: the window's dY0 block; sw: W_0 as stage_w0 left it.
// The tap walk of cnn_image_grad_kernel, which keeps it inline: as a call there it costs a spill at the image
// kernel's 80-register budget.
__device__ __forceinline__ void conv0_pixel_grad(const float* g, const float* sw, int ly, int lx, int ho, int co_n,
                                                 int cinp, int c0, float (&acc)[IG_CB]) {
    const int wsz = co_n * cinp;
#pragma unroll
    for (int iy = 0; iy < 2; ++iy) {
        int ky, oy;
        if (ly & 1) {
            ky = iy ? 0 : 2;
            oy = iy ? (ly + 1) >> 1 : (ly - 1) >> 1;
            if (oy >= ho) continue;
        } else {
            if (iy) continue;
            ky = 1;
            oy = ly >> 1;
        }
#pragma unroll
        for (int ix = 0; ix < 2; ++ix) {
            int kx, ox;
            if (lx & 1) {
                kx = ix ? 0 : 2;
                ox = ix ? (lx + 1) >> 1 : (lx - 1) >> 1;
                if (ox >= ho) continue;
            } else {
                if (ix) continue;
                kx = 1;
                ox = lx >> 1;
            }
            const float4* gp = reinterpret_cast<const float4*>(g + (oy * ho + ox) * co_n);
            const float4* wp = reinterpret_cast<const float4*>(sw + (ky * 3 + kx) * wsz + c0);
            const int wstride = cinp >> 2;
            for (int q = 0; q < (co_n >> 2); ++q) {
                const float4 gv = gp[q];
                const float gs[4] = {gv.x, gv.y, gv.z, gv.w};
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const float4 wv = wp[(4 * q + u) * wstride];
                    acc[0] += gs[u] * wv.x;
                    acc[1] += gs[u] * wv.y;
                    acc[2] += gs[u] * wv.z;
                    acc[3] += gs[u] * wv.w;
                }
            }
        }
    }
}

// Gradient on the caller's windows of one stand-alone step (marlc_model_step_input_grad): the first conv
// layer's input gradient, window by window,
//     d_patch[p,c,ly,lx] = sum over taps (ky,kx) with 2*oy-1+ky = ly, 2*ox-1+kx = lx, and co,
//                          dY0[p][oy,ox][co] * W0[co,c,ky,kx],
// and 0 in the channels c >= cin the network does not read.  No gather: the windows are the caller's.  Each
// output element has one owner thread, which sums its taps in a fixed order (conv0_pixel_grad): no atomics.
// One CTA per `batch` consecutive windows: W_0 staged once, then the windows' dY0 blocks (one contiguous
// range) with all loads in flight, then one thread per (window, pixel), consecutive threads on consecutive
// pixels of a channel plane (coalesced stores).
constexpr int PG_THREADS = 256;
constexpr int PG_MAX_BATCH = 8;            // windows per CTA: 8 x 144 pixels at f = 12
constexpr int PG_STAGE_BYTES = 24 * 1024;  // dY0 staging budget per CTA

__global__ void __launch_bounds__(PG_THREADS) cnn_patch_grad_kernel(const PatchGradArgs a, FastDiv d_cin, FastDiv d_ff,
                                                                    FastDiv d_f, int cinp, int batch) {
    extern __shared__ float4 sm4[];
    const int co_n = a.cout, ci_n = a.cin, f = a.f, ff = f * f, ho = a.ho;
    const int blk = ho * ho * co_n;
    float* sw = reinterpret_cast<float*>(sm4);
    float* sdy = sw + 9 * co_n * cinp;
    const int p0 = blockIdx.x * batch, nb = min(batch, a.M - p0);
    stage_w0(sw, a.w0, co_n, ci_n, cinp, d_cin, PG_THREADS);
    {
        const float4* src = reinterpret_cast<const float4*>(a.dY0) + (long)p0 * (blk >> 2);
        float4* s4 = reinterpret_cast<float4*>(sdy);
#pragma unroll 4
        for (int e = threadIdx.x; e < nb * (blk >> 2); e += PG_THREADS) s4[e] = __ldg(src + e);
    }
    __syncthreads();
    for (int it = threadIdx.x; it < nb * ff; it += PG_THREADS) {
        const int jw = d_ff.div(it), q = it - jw * ff, ly = d_f.div(q), lx = q - ly * f;
        const float* g = sdy + jw * blk;
        float* out = a.d_patch + (long)(p0 + jw) * a.C * ff + q;
        for (int c0 = 0; c0 < ci_n; c0 += IG_CB) {
            float acc[IG_CB] = {0.f, 0.f, 0.f, 0.f};
            conv0_pixel_grad(g, sw, ly, lx, ho, co_n, cinp, c0, acc);
#pragma unroll
            for (int u = 0; u < IG_CB; ++u)
                if (c0 + u < ci_n) out[(c0 + u) * ff] = acc[u];
        }
        for (int c = ci_n; c < a.C; ++c) out[c * ff] = 0.f;  // MnistCnn on 3-channel windows
    }
}

int cnn_patch_grad(const PatchGradArgs& a, cudaStream_t s) {
    MARLC_CHECK(a.dY0 && a.w0 && a.d_patch, "patch_grad: null pointer");
    MARLC_CHECK(a.cin >= 1 && a.cin <= a.C && a.cout >= 1 && a.f >= 1 && a.ho == (a.f - 1) / 2 + 1,
                "patch_grad: bad CNN shape");
    MARLC_CHECK((a.cout & 3) == 0 && (reinterpret_cast<uintptr_t>(a.dY0) & 15) == 0,
                "patch_grad: the first conv layer needs a multiple of 4 output channels (has %d)", a.cout);
    if (a.M <= 0) return 0;
    const int cinp = (a.cin + IG_CB - 1) / IG_CB * IG_CB;
    const int blk = a.ho * a.ho * a.cout, ff = a.f * a.f;
    const int batch = std::max(1, std::min(PG_MAX_BATCH, PG_STAGE_BYTES / (blk * (int)sizeof(float))));
    MARLC_CHECK(FastDiv::exact_up_to((long long)batch * ff, ff) && FastDiv::exact_up_to(ff, a.f) &&
                    FastDiv::exact_up_to((long long)a.cout * a.cin * 9, a.cin),
                "patch_grad: window of %d x %d too large", a.f, a.f);
    const size_t smem = ((size_t)9 * a.cout * cinp + (size_t)batch * blk) * sizeof(float);
    MARLC_CHECK(smem <= 200 * 1024, "patch_grad: first-layer shapes too large for shared memory (%zu B)", smem);
    static size_t attr = 0;
    if (smem > 48 * 1024 && smem > attr) {
        MARLC_CUDA(cudaFuncSetAttribute(cnn_patch_grad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr = smem;
    }
    const unsigned grid = (unsigned)((a.M + batch - 1) / batch);
    cnn_patch_grad_kernel<<<grid, PG_THREADS, smem, s>>>(a, FastDiv((unsigned)a.cin), FastDiv((unsigned)ff),
                                                          FastDiv((unsigned)a.f), cinp, batch);
    MARLC_LAUNCH_CHECK();
    return 0;
}

}  // namespace marlc

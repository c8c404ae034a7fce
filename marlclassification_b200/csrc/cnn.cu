// Per-agent feature extractor (networks/vision.py:23-77): k x [conv3x3 s2 p1 ->
// GroupNorm(eps 1e-5) -> SiLU] -> flatten, fused with the window gather.
// One CTA per window; every activation stays in shared memory; only the
// pre-norm conv outputs are saved (for backward) and the final features are
// written straight into the LSTM input matrix u_t (no concat kernel).
#include "cnn_device.cuh"
#include "kernels.cuh"

namespace marlc {

__global__ void __launch_bounds__(256) cnn_fwd_kernel(const CnnFwdArgs a) {
    extern __shared__ float sm[];
    cnn_fwd_block(a, blockIdx.x, sm);
}

int cnn_fwd(const CnnDesc& d, const float* img, const int* pos, const float* patch, int B, int H, int W, int M,
            float* const* y_save, float* out, long ldo, cudaStream_t s) {
    if (M <= 0) return 0;
    CnnFwdArgs a;
    a.d = d; a.img = img; a.pos = pos; a.patch = patch; a.out = out; a.ldo = ldo;
    a.B = B; a.H = H; a.W = W; a.M = M;
    cnn_fwd_plan(d, &a.padsz, &a.ysz, &a.wbuf);
    for (int l = 0; l < MAX_CNN_LAYERS; ++l) a.y_save[l] = (y_save && l < d.L) ? y_save[l] : nullptr;
    size_t smem = cnn_fwd_smem_bytes(a);
    MARLC_CHECK(smem <= 200 * 1024, "cnn_fwd: window too large for shared memory (%zu B)", smem);
    static size_t attr = 0;
    if (smem > 48 * 1024 && smem > attr) {
        MARLC_CUDA(cudaFuncSetAttribute(cnn_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr = smem;
    }
    cnn_fwd_kernel<<<M, 256, smem, s>>>(a);
    MARLC_LAUNCH_CHECK();
    return 0;
}

// ---------------------------------------------------------------------------
// Transposed copies of the conv weights, wT_l[(ci*9 + tap)][co] (output channel contiguous), used
// by the register-tiled forward block: a thread computing 4 consecutive output channels reads the
// 4 weights of a tap with one 128-bit load, and a whole layer is one contiguous bulk copy.
// Refreshed once per forward (the parameters may have been updated by the optimiser).
// ---------------------------------------------------------------------------
struct CnnTransposeArgs { const float* w[MAX_CNN_LAYERS]; float* wT[MAX_CNN_LAYERS]; int co[MAX_CNN_LAYERS], wrow[MAX_CNN_LAYERS]; int L; };
__global__ void __launch_bounds__(256) cnn_transpose_kernel(const CnnTransposeArgs a) {
    for (int l = 0; l < a.L; ++l) {
        const int n = a.co[l] * a.wrow[l];
        for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < n; e += gridDim.x * blockDim.x) {
            const int k = e / a.co[l], c = e - k * a.co[l];  // coalesced writes
            a.wT[l][e] = __ldg(a.w[l] + (long)c * a.wrow[l] + k);
        }
    }
}
int cnn_weights_transpose(const CnnDesc& d, float* const* wT, cudaStream_t s) {
    CnnTransposeArgs a;
    a.L = d.L;
    int mx = 0;
    for (int l = 0; l < d.L; ++l) {
        a.w[l] = d.w[l]; a.wT[l] = wT[l]; a.co[l] = d.cout[l]; a.wrow[l] = d.cin[l] * 9;
        mx = max(mx, d.cout[l] * d.cin[l] * 9);
    }
    cnn_transpose_kernel<<<max(1, min(148, (mx + 255) / 256)), 256, 0, s>>>(a);
    MARLC_LAUNCH_CHECK();
    return 0;
}

// ---------------------------------------------------------------------------
// Backward.  One CTA per window p (p = t*M + m).  Re-gathers the input window,
// rebuilds the activations from the saved pre-norm outputs, then walks the
// layers backwards.  It does NOT reduce weight gradients itself: it emits, per
// layer, the conv-output gradient rows dY [P*npos, cout] and the im2col rows
// [P*npos, cin*9] so that dW = dY^T col is one large GEMM over all T*M windows
// (reduction dim T*M*npos), plus per-window GroupNorm partials.
// ---------------------------------------------------------------------------
struct CnnBwdArgs {
    CnnDesc d;
    CnnWindows win;
    const float* y_save[MAX_CNN_LAYERS];
    const float* dOut;
    long lddo;
    CnnBwdBuffers buf;
    int offA[MAX_CNN_LAYERS], offY[MAX_CNN_LAYERS], offStat[MAX_CNN_LAYERS];
    int offD0, offD1, offW, wbuf;
    int P, p0;
};

template <bool PATCH>
__global__ void __launch_bounds__(256) cnn_bwd_kernel(const CnnBwdArgs a) {
    extern __shared__ float sm[];
    const CnnDesc& d = a.d;
    const int p = a.p0 + blockIdx.x;
    const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5, nwarps = nt >> 5;
    const int f = d.f, ff = f * f;

    // ---- A_0: the input window
    {
        long chan;
        int row;
        const float* src = cnn_window<PATCH>(a.win, p, chan, row);
        float* A0 = sm + a.offA[0];
        for (int e = tid; e < d.cin[0] * ff; e += nt) {
            const int c = e / ff, i = (e / f) % f, j = e % f;
            A0[e] = __ldg(src + c * chan + (long)i * row + j);
        }
    }
    // ---- Y_l, group statistics, A_{l+1} = SiLU(GN(Y_l))
    for (int l = 0; l < d.L; ++l) {
        const int co_n = d.cout[l], npos = d.hout[l] * d.hout[l], total = co_n * npos;
        float* Y = sm + a.offY[l];
        const float* ys = a.y_save[l] + (long)p * total;
        for (int e = tid; e < total; e += nt) Y[e] = ys[e];
        __syncthreads();
        const int G = d.groups[l], cpg = co_n / G, ng = cpg * npos;
        const float inv = 1.0f / (float)ng;
        float* stat = sm + a.offStat[l];  // [G][2] mean, rstd
        for (int g = warp; g < G; g += nwarps) {
            const float* base = Y + g * ng;
            float s = 0.f;
            for (int e = lane; e < ng; e += 32) s += base[e];
            const float mean = warp_sum(s) * inv;
            float v = 0.f;
            for (int e = lane; e < ng; e += 32) { float dd = base[e] - mean; v += dd * dd; }
            const float rstd = 1.0f / sqrtf(warp_sum(v) * inv + GN_EPS);
            if (lane == 0) { stat[2 * g] = mean; stat[2 * g + 1] = rstd; }
            if (l + 1 < d.L) {
                float* An = sm + a.offA[l + 1] + g * ng;
                for (int e = lane; e < ng; e += 32) {
                    const int c = g * cpg + e / npos;
                    An[e] = siluf_((base[e] - mean) * rstd * d.gn_w[l][c] + d.gn_b[l][c]);
                }
            }
        }
    }
    float* Dcur = sm + a.offD0;
    float* Dprev = sm + a.offD1;
    {
        const float* go = a.dOut + (long)p * a.lddo;
        for (int e = tid; e < d.out_size; e += nt) Dcur[e] = go[e];
    }
    __syncthreads();

    for (int l = d.L - 1; l >= 0; --l) {
        const int ci_n = d.cin[l], co_n = d.cout[l], hi = d.hin[l], ho = d.hout[l];
        const int npos = ho * ho, total = co_n * npos;
        const int G = d.groups[l], cpg = co_n / G, ng = cpg * npos;
        float* Y = sm + a.offY[l];
        const float* stat = sm + a.offStat[l];
        const float* A = sm + a.offA[l];
        // 1. xhat (kept in Y) and dz = dA * silu'(z) (kept in Dcur)
        for (int e = tid; e < total; e += nt) {
            const int c = e / npos, g = c / cpg;
            const float xh = (Y[e] - stat[2 * g]) * stat[2 * g + 1];
            Y[e] = xh;
            Dcur[e] *= silu_grad_(xh * d.gn_w[l][c] + d.gn_b[l][c]);
        }
        __syncthreads();
        // 1b. per-channel partials for dgamma / dbeta (one warp per channel)
        {
            float* gp = a.buf.gnpart[l] + (long)p * 2 * co_n;
            for (int c = warp; c < co_n; c += nwarps) {
                float s1 = 0.f, s2 = 0.f;
                for (int e = lane; e < npos; e += 32) {
                    const float dz = Dcur[c * npos + e];
                    s1 += dz * Y[c * npos + e];
                    s2 += dz;
                }
                s1 = warp_sum(s1); s2 = warp_sum(s2);
                if (lane == 0) { gp[c] = s1; gp[co_n + c] = s2; }
            }
        }
        // 2a. group sums for the normalisation backward
        float* gs = Dprev;  // Dprev is free here; [G][2]
        for (int g = warp; g < G; g += nwarps) {
            float s1 = 0.f, s2 = 0.f;
            for (int e = lane; e < ng; e += 32) {
                const int c = g * cpg + e / npos;
                const float t = Dcur[g * ng + e] * d.gn_w[l][c];
                s1 += t;
                s2 += t * Y[g * ng + e];
            }
            s1 = warp_sum(s1); s2 = warp_sum(s2);
            if (lane == 0) { gs[2 * g] = s1 / (float)ng; gs[2 * g + 1] = s2 / (float)ng; }
        }
        __syncthreads();
        // 2b. dy (conv-output gradient), in place
        for (int e = tid; e < total; e += nt) {
            const int c = e / npos, g = c / cpg;
            Dcur[e] = stat[2 * g + 1] * (Dcur[e] * d.gn_w[l][c] - gs[2 * g] - Y[e] * gs[2 * g + 1]);
        }
        __syncthreads();
        // 3. emit dY rows [pos][co] and im2col rows [pos][ci*9 + ky*3 + kx]
        {
            float* dYg = a.buf.dY[l] + (long)p * npos * co_n;
            for (int e = tid; e < total; e += nt) {
                const int pos = e / co_n, co = e % co_n;
                dYg[e] = Dcur[co * npos + pos];
            }
            const int kk = ci_n * 9;
            float* colg = a.buf.col[l] + (long)p * npos * kk;
            for (int e = tid; e < npos * kk; e += nt) {
                const int pos = e / kk, r = e % kk, ci = r / 9, ky = (r % 9) / 3, kx = r % 3;
                const int iy = 2 * (pos / ho) - 1 + ky, ix = 2 * (pos % ho) - 1 + kx;
                colg[e] = (iy >= 0 && iy < hi && ix >= 0 && ix < hi) ? A[ci * hi * hi + iy * hi + ix] : 0.f;
            }
        }
        // 4. input gradient dA_l (not needed for the image itself); weights staged in smem chunks
        if (l > 0) {
            const float* __restrict__ w = d.w[l];
            const int tin = ci_n * hi * hi, wrow = ci_n * 9, P = cnn_wpitch(wrow);
            const int cc = min(co_n, a.wbuf / P);
            float* ws = sm + a.offW;
            for (int co0 = 0; co0 < co_n; co0 += cc) {
                const int ncur = min(cc, co_n - co0);
                __syncthreads();
                stage_rows(ws, w + (long)co0 * wrow, ncur, wrow, P);
                __syncthreads();
                for (int e = tid; e < tin; e += nt) {
                    const int ci = e / (hi * hi), iy = (e / hi) % hi, ix = e % hi;
                    float acc = co0 == 0 ? 0.f : Dprev[e];
#pragma unroll
                    for (int ky = 0; ky < 3; ++ky) {
                        const int ty = iy + 1 - ky;
                        if (ty < 0 || (ty & 1)) continue;
                        const int oy = ty >> 1;
                        if (oy >= ho) continue;
#pragma unroll
                        for (int kx = 0; kx < 3; ++kx) {
                            const int tx = ix + 1 - kx;
                            if (tx < 0 || (tx & 1)) continue;
                            const int ox = tx >> 1;
                            if (ox >= ho) continue;
                            const float* wp = ws + ci * 9 + ky * 3 + kx;
                            const float* dp = Dcur + (long)co0 * npos + oy * ho + ox;
                            float a0 = 0.f, a1 = 0.f;
                            int cq = 0;
                            for (; cq + 1 < ncur; cq += 2) {
                                a0 = fmaf(dp[cq * npos], wp[cq * P], a0);
                                a1 = fmaf(dp[(cq + 1) * npos], wp[(cq + 1) * P], a1);
                            }
                            if (cq < ncur) a0 = fmaf(dp[cq * npos], wp[cq * P], a0);
                            acc += a0 + a1;
                        }
                    }
                    Dprev[e] = acc;
                }
            }
        }
        __syncthreads();
        float* t = Dcur; Dcur = Dprev; Dprev = t;
    }
}

int cnn_bwd(const CnnDesc& d, const CnnWindows& win, int p0, int P, const float* const* y_save, const float* dOut,
            long lddo, const CnnBwdBuffers& buf, cudaStream_t s) {
    if (P <= 0) return 0;
    CnnBwdArgs a;
    a.p0 = p0;
    a.d = d; a.win = win; a.dOut = dOut; a.lddo = lddo; a.buf = buf;
    a.P = P;
    int off = 0, mx = 0;
    for (int l = 0; l < d.L; ++l) {
        a.y_save[l] = y_save[l];
        a.offA[l] = off; off += d.cin[l] * d.hin[l] * d.hin[l];
        a.offY[l] = off; off += d.cout[l] * d.hout[l] * d.hout[l];
        a.offStat[l] = off; off += 2 * d.groups[l];
        mx = max(mx, max(d.cin[l] * d.hin[l] * d.hin[l], d.cout[l] * d.hout[l] * d.hout[l]));
        mx = max(mx, 2 * d.groups[l]);
    }
    a.offD0 = off; off += mx;
    a.offD1 = off; off += mx;
    {
        int wmax = 0;
        for (int l = 1; l < d.L; ++l) wmax = max(wmax, d.cout[l] * cnn_wpitch(d.cin[l] * 9));
        a.wbuf = min(wmax, 24 * 1024);
        a.offW = off; off += a.wbuf;
    }
    size_t smem = sizeof(float) * (size_t)off;
    MARLC_CHECK(smem <= 200 * 1024, "cnn_bwd: window too large for shared memory (%zu B)", smem);
    static size_t attr_b = 0;
    if (smem > 48 * 1024 && smem > attr_b) {
        MARLC_CUDA(cudaFuncSetAttribute(cnn_bwd_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        MARLC_CUDA(cudaFuncSetAttribute(cnn_bwd_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_b = smem;
    }
    if (win.patch) cnn_bwd_kernel<true><<<P, 256, smem, s>>>(a);
    else cnn_bwd_kernel<false><<<P, 256, smem, s>>>(a);
    MARLC_LAUNCH_CHECK();
    return 0;
}

}  // namespace marlc

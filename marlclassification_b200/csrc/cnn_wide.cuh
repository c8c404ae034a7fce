// Wide gather + CNN forward: NW windows per pass, weights stationary in shared memory.
//
// The per-window block (cnn_device.cuh) is the right shape for the reference's batch sizes (128
// windows = one CTA per SM, latency-bound).  At the sharded-batch configurations (M = 512 .. 4096
// windows per step) it re-stages 95 KB of weights per window (390 MB of L2 -> SMEM traffic per step
// at M = 4096) and runs one window's three-layer dependency chain per SM at a time: 265 us per
// step at M = 4096, i.e. 4 TFLOP/s of fp32 (ncu launch list, round 2).  Here a CTA
//   * loads all conv weights (transposed [cin*9][cout]), biases and GroupNorm affines ONCE and
//     then loops over batches of NW = 8 windows (persistent, grid <= #SM);
//   * keeps activations as [channel][y][x][window] (window fastest, zero border): a thread owns 4
//     output channels x 8 windows at one output position, so a tap costs three 128-bit shared
//     loads (8 inputs, 4 weights) for 32 FMAs -- 10x fewer shared-memory bytes per FMA than one
//     window at a time -- and the lanes of a warp read distinct banks or broadcast;
//   * splits the input channels of the narrow late layers over `ks` thread groups (partial
//     planes, summed when the pre-norm outputs are saved for backward);
//   * computes GroupNorm statistics two-pass (as the reference), a lane owning 4 windows of an
//     element (128-bit shared accesses, branch-free loops, channel / scatter indices from a table);
//   * prefetches the next batch's windows with cp.async as soon as layer 0 has consumed the
//     current ones.
// Same arithmetic as cnn_fwd_block_t (fp32 FFMA, fast SiLU); summation order differs (parity tests
// hold both to the oracle).  vision.py:23-57.
#pragma once
#include "cnn_device.cuh"

namespace marlc {

// Windows per pass.  4 (twice the CTAs while 8 leave SMs idle) measured slower at 512 and 1024 windows (476 vs
// 438 us, 795 vs 745 us per 16 steps): a pass is bound by the latency of its phases, not by its FMA count.
constexpr int CW_NW = 8;
constexpr int CW_THREADS = 256;  // = the chain kernels' CTA (step_pre hosts this role); 512 threads as a separate launch
                                 // measured no faster per batch and cost a fork / join per step
constexpr int CW_MAX_KS = 8;

struct CnnWidePlan {
    int ok;                          // 0: shapes not supported (caller uses the per-window block)
    int w_off[MAX_CNN_LAYERS];       // floats: transposed weights of layer l
    int p_off[MAX_CNN_LAYERS];       // bias | gamma | beta (3 * cout)
    int lut_off[MAX_CNN_LAYERS];     // per output element e = c * npos + pos: (c << 16) | position in the next layer's input
    int in_off[MAX_CNN_LAYERS];      // zero-bordered input of layer l: [cin][hin+2][hin+2][NW]
    int y_off;                       // pre-norm outputs, up to CW_MAX_KS partial planes of [cout][npos][NW]
    int st_off;                      // GroupNorm: cross-warp partial sums [warps][NW]
    int ks[MAX_CNN_LAYERS];          // input-channel slices of layer l
    int smem_floats;
};

// have_wT: the engine keeps transposed conv weights (d.wT, one buffer per layer; with the chain kernels).  A flag
// rather than a test of d.wT[0], which is only set at bind, so that an engine's plan can be queried before.
inline CnnWidePlan cnn_wide_plan(const CnnDesc& d, bool have_img, bool have_wT) {
    constexpr int nw = CW_NW;
    CnnWidePlan p;
    memset(&p, 0, sizeof(p));
    if (!have_img || !have_wT) return p;
    int off = 0;
    for (int l = 0; l < d.L; ++l) {
        if ((d.cout[l] & 3) || d.groups[l] > 32 || d.cout[l] % d.groups[l]) return p;
        p.w_off[l] = off;
        off += d.cout[l] * d.cin[l] * 9;
    }
    for (int l = 0; l < d.L; ++l) { p.p_off[l] = off; off += 3 * d.cout[l]; }
    for (int l = 0; l < d.L; ++l) {
        if (d.cout[l] >= 32768 || d.cout[l] * (d.hout[l] + 2) * (d.hout[l] + 2) >= 65536) return p;  // packed in 16 + 16 bits
        p.lut_off[l] = off;
        off += d.cout[l] * d.hout[l] * d.hout[l];
    }
    off = (off + 3) & ~3;
    for (int l = 0; l < d.L; ++l) {
        p.in_off[l] = off;
        off += d.cin[l] * (d.hin[l] + 2) * (d.hin[l] + 2) * nw;
    }
    // input-channel slices: as many as there are idle threads, within what is left of shared memory for the
    // partial planes (224 KB budget: one CTA per SM owns practically all of its shared memory)
    const int st_floats = (CW_THREADS / 32) * nw;
    const int ybudget = 224 * 256 - off - st_floats;
    int ymax = 0;
    for (int l = 0; l < d.L; ++l) {
        const int items = d.hout[l] * d.hout[l] * (d.cout[l] >> 2);
        const int plane = d.cout[l] * d.hout[l] * d.hout[l] * nw;
        if (plane > ybudget) return p;
        int ks = 1;
        while (ks < CW_MAX_KS && items * (ks + 1) <= CW_THREADS && ks + 1 <= d.cin[l] && (ks + 1) * plane <= ybudget) ++ks;
        const int cpk = (d.cin[l] + ks - 1) / ks;
        ks = (d.cin[l] + cpk - 1) / cpk;  // drop slices that would be empty
        p.ks[l] = ks;
        ymax = max(ymax, ks * plane);
    }
    p.y_off = off;
    off += ymax;
    p.st_off = off;
    off += st_floats;
    p.smem_floats = off;
    p.ok = (size_t)off * sizeof(float) <= 224 * 1024;
    return p;
}

__device__ __forceinline__ int cw_div(int n, float rcp) { return __float2int_rz(((float)n + 0.5f) * rcp); }  // n < 2^16

// Request the interior of layer 0's input for the windows of a batch (4-byte cp.async: rows of f floats are
// contiguous in the image, the destination is window-interleaved).  One thread per (window, channel, row):
// the window's corner and image index come from shared memory (`win`: {py, px, image} per window, loaded by
// cw_load_windows one phase earlier), the f copies of a row need no index arithmetic.  (First version: one
// element per thread iteration with three divisions, a modulo and two dependent global loads of the
// position each -- 4.8 M warp instructions per launch at 4096 windows and ~5000 exposed cycles per batch.)
template <int NW>
__device__ __forceinline__ void cw_load_windows(const CnnFwdArgs& a, int* win, int batch) {
    const int m = batch * NW + (int)threadIdx.x;
    if (threadIdx.x < NW && m < a.M) {
        win[threadIdx.x * 4 + 0] = a.pos[2 * m];
        win[threadIdx.x * 4 + 1] = a.pos[2 * m + 1];
        win[threadIdx.x * 4 + 2] = m % a.B;
    }
}
template <int NW>
__device__ __forceinline__ void cw_issue_gather(const CnnFwdArgs& a, float* in0, const int* win, int batch) {
    const CnnDesc& d = a.d;
    const int f = d.f, c0 = d.cin[0], hp = f + 2, ff = f * f;
    const int nvalid = min(NW, a.M - batch * NW);
    const int per_w = c0 * ff;
    const float r_per = 1.0f / (float)per_w, r_ff = 1.0f / (float)ff, r_f = 1.0f / (float)f;
    const uint32_t dst0 = (uint32_t)__cvta_generic_to_shared(in0);
    // one 4-byte request per thread iteration, the lanes of a warp walk ALONG the rows of a window (f contiguous
    // floats each), so a warp-wide request touches 32 / f + 1 cache lines.  (Round 2 trace: the earlier mapping,
    // one thread per row issuing its f requests, made every warp-wide request touch 32 lines -- ~5000 cycles of
    // load/store-unit time per batch of 8 windows, the largest single item of the batch.)
    for (int q = threadIdx.x; q < nvalid * per_w; q += CW_THREADS) {
        const int w = cw_div(q, r_per), r = q - w * per_w, c = cw_div(r, r_ff), r2 = r - c * ff;
        const int i = cw_div(r2, r_f), j = r2 - i * f;
        const int py = win[w * 4], px = win[w * 4 + 1], b = win[w * 4 + 2];
        const float* src = a.img + ((long)(b * d.img_c + c) * a.H + py + i) * a.W + px + j;
        const uint32_t dst = dst0 + 4u * (uint32_t)(((c * hp + i + 1) * hp + 1 + j) * NW + w);
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(src) : "memory");
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
}

// CTA `cta` of `n_cta` cooperating CTAs; all CW_THREADS threads must call.
template <int NW>
__device__ __forceinline__ void cnn_fwd_wide_t(const CnnFwdArgs& a, const CnnWidePlan& pl, const int cta, const int n_cta,
                                               float* sm) {
    const CnnDesc& d = a.d;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nbatch = (a.M + NW - 1) / NW;
    if (cta >= nbatch) return;
#ifdef MARLC_CNN_TRACE  // timeline of CTA 0 (cycles since entry): setup, then per batch / layer: conv, pass A, B, C
    __shared__ long long cw_tr[48];
    const long long cw_t0 = clock64();
    int cw_i = 0;
#define CW_TRACE() do { if (cta == 0 && tid == 0 && cw_i < 48) cw_tr[cw_i] = clock64() - cw_t0; ++cw_i; } while (0)
#else
#define CW_TRACE() do { } while (0)
#endif
    // ---- once per CTA: zero the activation buffers (their borders stay zero), stage weights + affines
    __shared__ __align__(8) uint64_t wbar[MAX_CNN_LAYERS];  // one per layer: layer 0 (1.7 KB at RESISC45) must not wait for layer 2 (73 KB)
    __shared__ int s_win[2][NW * 4];  // {py, px, image} of the current / next batch's windows
    // (everything up to pdl_wait() reads launch constants only -- weights, biases, affines -- so under a programmatic
    //  dependent launch it overlaps the previous kernel of the step chain; the window corners come from that kernel)
    if (tid == 0) {
        for (int l = 0; l < d.L; ++l)
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"((uint32_t)__cvta_generic_to_shared(&wbar[l])));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        // weights: ONE bulk copy per layer (the copy engine moves them while the threads go on), completion on wbar
        for (int l = 0; l < d.L; ++l) {
            const uint32_t bar = (uint32_t)__cvta_generic_to_shared(&wbar[l]);
            const uint32_t bytes = (uint32_t)(d.cout[l] * d.cin[l] * 9 * 4);
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                             (uint32_t)__cvta_generic_to_shared(sm + pl.w_off[l])), "l"(d.wT[l]), "r"(bytes), "r"(bar) : "memory");
        }
    }
    {
        float4* z = reinterpret_cast<float4*>(sm + pl.in_off[0]);
        const int n4 = (pl.y_off - pl.in_off[0]) >> 2;
        for (int i = tid; i < n4; i += CW_THREADS) z[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    for (int l = 0; l < d.L; ++l) {
        float* pp = sm + pl.p_off[l];
        for (int i = tid; i < d.cout[l]; i += CW_THREADS) {
            pp[i] = d.b[l][i];
            pp[d.cout[l] + i] = d.gn_w[l][i];
            pp[2 * d.cout[l] + i] = d.gn_b[l][i];
        }
    }
    for (int l = 0; l < d.L; ++l) {  // element -> (channel, slot in the next layer's zero-bordered input)
        int* lut = reinterpret_cast<int*>(sm + pl.lut_off[l]);
        const int ho = d.hout[l], npos = ho * ho, hop = ho + 2, total = d.cout[l] * npos;
        const bool last = (l + 1 == d.L);
        for (int e = tid; e < total; e += CW_THREADS) {
            const int c = e / npos, pos = e - c * npos, oy = pos / ho, ox = pos - oy * ho;
            lut[e] = (c << 16) | (last ? 0 : (c * hop + oy + 1) * hop + ox + 1);
        }
    }
    pdl_wait();
    cw_load_windows<NW>(a, s_win[0], cta);
    __syncthreads();  // the gather below reads s_win and writes into the zeroed buffer; wbar is initialised for all
    cw_issue_gather<NW>(a, sm + pl.in_off[0], s_win[0], cta);
    CW_TRACE();  // 0: zeroed, gather + weight staging issued
    float* ybuf = sm + pl.y_off;
    float* s_red = sm + pl.st_off;  // cross-warp partial sums of the GroupNorm statistics [warps][NW]

    int wbuf = 0;
    for (int batch = cta; batch < nbatch; batch += n_cta, wbuf ^= 1) {
        const int m0 = batch * NW, nvalid = min(NW, a.M - m0);
        if (batch + n_cta < nbatch) cw_load_windows<NW>(a, s_win[wbuf ^ 1], batch + n_cta);  // visible after layer 0's barrier
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncthreads();  // windows of this batch (and, first time, the affines) are in shared memory
        CW_TRACE();  // batch start: inputs ready
        for (int l = 0; l < d.L; ++l) {
            const int ci_n = d.cin[l], co_n = d.cout[l], hi = d.hin[l], ho = d.hout[l];
            const int hp = hi + 2, npos = ho * ho, total = co_n * npos, ncg = co_n >> 2;
            const int G = d.groups[l], cpg = co_n / G, ng = cpg * npos;
            const bool last = (l + 1 == d.L);
            const float* in = sm + pl.in_off[l];
            const float* wl = sm + pl.w_off[l];
            const float* prm = sm + pl.p_off[l];
            const int ks = pl.ks[l], cpk = (ci_n + ks - 1) / ks, items = npos * ncg;
            if (batch == cta) {  // first batch: this layer's weights must have landed
                const uint32_t bar = (uint32_t)__cvta_generic_to_shared(&wbar[l]);
                uint32_t done;
                do {
                    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                                 : "=r"(done) : "r"(bar) : "memory");
                } while (!done);
            }
            // ---- convolution: work item = (input-channel slice, output position, group of 4 output channels)
            {
                const float r_items = 1.0f / (float)items, r_ncg = 1.0f / (float)ncg, r_ho = 1.0f / (float)ho;
                for (int wk = tid; wk < items * ks; wk += CW_THREADS) {
                    const int kslice = cw_div(wk, r_items), item = wk - kslice * items;
                    const int pos = cw_div(item, r_ncg), c4 = (item - pos * ncg) << 2;
                    const int oy = cw_div(pos, r_ho), ox = pos - oy * ho;
                    const int ci0 = kslice * cpk, ci1 = min(ci_n, ci0 + cpk);
                    float acc[4][NW];
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const float bj = kslice == 0 ? prm[c4 + j] : 0.f;
#pragma unroll
                        for (int w = 0; w < NW; ++w) acc[j][w] = bj;
                    }
                    const float* x = in + ((ci0 * hp + 2 * oy) * hp + 2 * ox) * NW;
                    const float* wq = wl + (ci0 * 9) * co_n + c4;
                    for (int ci = ci0; ci < ci1; ++ci, x += hp * hp * NW, wq += 9 * co_n) {
#pragma unroll
                        for (int ky = 0; ky < 3; ++ky)
#pragma unroll
                            for (int kx = 0; kx < 3; ++kx) {
                                float xv[NW];
#pragma unroll
                                for (int h4 = 0; h4 < NW / 4; ++h4) {
                                    const float4 xq = *reinterpret_cast<const float4*>(x + (ky * hp + kx) * NW + 4 * h4);
                                    xv[4 * h4] = xq.x; xv[4 * h4 + 1] = xq.y; xv[4 * h4 + 2] = xq.z; xv[4 * h4 + 3] = xq.w;
                                }
                                const float4 w4 = *reinterpret_cast<const float4*>(wq + (ky * 3 + kx) * co_n);
                                const float wv[4] = {w4.x, w4.y, w4.z, w4.w};
#pragma unroll
                                for (int j = 0; j < 4; ++j)
#pragma unroll
                                    for (int w = 0; w < NW; ++w) acc[j][w] = fmaf(wv[j], xv[w], acc[j][w]);
                            }
                    }
                    float* y = ybuf + (kslice * total + c4 * npos + pos) * NW;
#pragma unroll
                    for (int j = 0; j < 4; ++j)
#pragma unroll
                        for (int h4 = 0; h4 < NW / 4; ++h4)
                            *reinterpret_cast<float4*>(y + j * npos * NW + 4 * h4) =
                                make_float4(acc[j][4 * h4], acc[j][4 * h4 + 1], acc[j][4 * h4 + 2], acc[j][4 * h4 + 3]);
                }
            }
            __syncthreads();
            CW_TRACE();  // conv done
            if (l == 0 && batch + n_cta < nbatch)  // layer 0's input buffer is free: prefetch the next batch's windows
                cw_issue_gather<NW>(a, sm + pl.in_off[0], s_win[wbuf ^ 1], batch + n_cta);
            // ---- GroupNorm + SiLU.  Warps are bound to groups (nwarps / G warps share a group when G < nwarps,
            //      their partial sums meet in shared memory).  A lane owns FOUR windows of an element (one 128-bit
            //      shared access; lane = (32 / WV elements) x (WV = NW / 4 window vectors)), U elements in flight,
            //      and the loops are branch-free (clamped indices, predicated stores): the first version -- one
            //      window per lane, per-element index divisions, `if (e < n_el)` bodies that serialised the 4
            //      elements of an iteration -- took 24 000 of a batch's 44 000 cycles (in-kernel trace, round 2).
            //      Two-pass statistics as the reference; the per-element channel / scatter index comes from a
            //      table built once per CTA.
            {
#ifdef CW_NO_YSAVE
                float* ysave = nullptr;
#else
                float* ysave = a.y_save[l];
#endif
                const float* gam = prm + co_n;
                const float* bet = prm + 2 * co_n;
                const int* lut = reinterpret_cast<const int*>(sm + pl.lut_off[l]);
                constexpr int WV = NW / 4;    // 128-bit window vectors per element
                constexpr int EPW = 32 / WV;  // elements a warp covers per step
                constexpr int U = 4;          // element slots in flight per lane
                const int wh = lane % WV, es = lane / WV;
                constexpr int nwarps = CW_THREADS / 32;
                const bool shared_groups = G < nwarps && nwarps % G == 0;
                const int wpg = shared_groups ? nwarps / G : 1;
                const int estep = EPW * wpg;
                const float inv = 1.0f / (float)ng;
                float* nxt = last ? nullptr : sm + pl.in_off[l + 1];
                bool wok[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) wok[j] = 4 * wh + j < nvalid;
                auto ld4 = [](const float* p) { return *reinterpret_cast<const float4*>(p); };
                auto group_sum = [&](float4 v, int g) -> float4 {  // over the lanes' elements, then over the group's warps
#pragma unroll
                    for (int o = WV; o < 32; o <<= 1) {
                        v.x += __shfl_xor_sync(0xffffffffu, v.x, o); v.y += __shfl_xor_sync(0xffffffffu, v.y, o);
                        v.z += __shfl_xor_sync(0xffffffffu, v.z, o); v.w += __shfl_xor_sync(0xffffffffu, v.w, o);
                    }
                    if (shared_groups) {
                        if (es == 0) *reinterpret_cast<float4*>(s_red + warp * NW + 4 * wh) = v;
                        __syncthreads();
                        v = make_float4(0.f, 0.f, 0.f, 0.f);
                        for (int i = 0; i < wpg; ++i) {
                            const float4 t = ld4(s_red + (g * wpg + i) * NW + 4 * wh);
                            v.x += t.x; v.y += t.y; v.z += t.z; v.w += t.w;
                        }
                        __syncthreads();
                    }
                    return v;
                };
                for (int g0 = 0; g0 < G; g0 += (shared_groups ? G : nwarps)) {
                    const int g = shared_groups ? warp / wpg : g0 + warp;
                    const int sub = shared_groups ? warp % wpg : 0;
                    const int el0 = sub * EPW + es;
                    const int n_el = (g < G) ? ng : 0;  // inactive warps run empty loops (they still meet the barriers)
                    const int gbase = (g < G ? g : 0) * ng;
                    float* yg = ybuf + gbase * NW + 4 * wh;
                    float* ys = ysave ? ysave + (long)(m0 + 4 * wh) * total + gbase : nullptr;
                    // pass 1: sum the input-channel slices (kept in plane 0), save for backward, accumulate the sum
                    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 1
                    for (int el = el0; el < n_el; el += U * estep) {
                        float4 x[U];
                        int e[U];
#pragma unroll
                        for (int u = 0; u < U; ++u) {
                            e[u] = el + u * estep < n_el ? el + u * estep : el;  // idle slots re-read the lane's own first element
                            x[u] = ld4(yg + e[u] * NW);
                        }
                        for (int p = 1; p < ks; ++p)
#pragma unroll
                            for (int u = 0; u < U; ++u) {
                                const float4 t = ld4(yg + (p * total + e[u]) * NW);
                                x[u].x += t.x; x[u].y += t.y; x[u].z += t.z; x[u].w += t.w;
                            }
#pragma unroll
                        for (int u = 0; u < U; ++u) {
                            const bool ok = el + u * estep < n_el;
                            if (ks > 1 && ok) *reinterpret_cast<float4*>(yg + e[u] * NW) = x[u];
                            if (ys) {
                                if (ok && wok[0]) ys[e[u]] = x[u].x;
                                if (ok && wok[1]) ys[(long)total + e[u]] = x[u].y;
                                if (ok && wok[2]) ys[2 * (long)total + e[u]] = x[u].z;
                                if (ok && wok[3]) ys[3 * (long)total + e[u]] = x[u].w;
                            }
                            if (ok) { s.x += x[u].x; s.y += x[u].y; s.z += x[u].z; s.w += x[u].w; }
                        }
                    }
                    s = group_sum(s, g);
                    const float4 mean = make_float4(s.x * inv, s.y * inv, s.z * inv, s.w * inv);
                    CW_TRACE();  // pass 1 done
                    // pass 2: centred second moment
                    float4 q = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 1
                    for (int el = el0; el < n_el; el += U * estep) {
                        float4 x[U];
#pragma unroll
                        for (int u = 0; u < U; ++u) x[u] = ld4(yg + (el + u * estep < n_el ? el + u * estep : el) * NW);
#pragma unroll
                        for (int u = 0; u < U; ++u) {
                            if (el + u * estep < n_el) {
                                const float dx = x[u].x - mean.x, dy = x[u].y - mean.y, dz = x[u].z - mean.z, dw = x[u].w - mean.w;
                                q.x = fmaf(dx, dx, q.x); q.y = fmaf(dy, dy, q.y); q.z = fmaf(dz, dz, q.z); q.w = fmaf(dw, dw, q.w);
                            }
                        }
                    }
                    q = group_sum(q, g);
                    const float4 rstd = make_float4(1.0f / sqrtf(q.x * inv + GN_EPS), 1.0f / sqrtf(q.y * inv + GN_EPS),
                                                    1.0f / sqrtf(q.z * inv + GN_EPS), 1.0f / sqrtf(q.w * inv + GN_EPS));
                    CW_TRACE();  // pass 2 done
                    // pass 3: normalise, SiLU, hand over (next layer's zero-bordered input, or the output rows)
                    float* orow = a.out + (long)(m0 + 4 * wh) * a.ldo + gbase;
                    float* orow_lo = a.out_lo ? a.out_lo + (long)(m0 + 4 * wh) * a.ldo + gbase : nullptr;
#pragma unroll 1
                    for (int el = el0; el < n_el; el += U * estep) {
                        float4 x[U];
                        int e[U], lu[U];
#pragma unroll
                        for (int u = 0; u < U; ++u) {
                            e[u] = el + u * estep < n_el ? el + u * estep : el;  // idle slots re-read the lane's own first element
                            x[u] = ld4(yg + e[u] * NW);
                            lu[u] = lut[gbase + e[u]];
                        }
                        float ga[U], be[U];
#pragma unroll
                        for (int u = 0; u < U; ++u) { ga[u] = gam[lu[u] >> 16]; be[u] = bet[lu[u] >> 16]; }
#pragma unroll
                        for (int u = 0; u < U; ++u) {
                            const bool ok = el + u * estep < n_el;
                            const float z0 = (x[u].x - mean.x) * rstd.x * ga[u] + be[u];
                            const float z1 = (x[u].y - mean.y) * rstd.y * ga[u] + be[u];
                            const float z2 = (x[u].z - mean.z) * rstd.z * ga[u] + be[u];
                            const float z3 = (x[u].w - mean.w) * rstd.w * ga[u] + be[u];
                            const float4 o = make_float4(__fdividef(z0, 1.0f + __expf(-z0)), __fdividef(z1, 1.0f + __expf(-z1)),
                                                         __fdividef(z2, 1.0f + __expf(-z2)), __fdividef(z3, 1.0f + __expf(-z3)));  // SiLU
                            if (!last) {
                                if (ok) *reinterpret_cast<float4*>(nxt + (lu[u] & 0xffff) * NW + 4 * wh) = o;
                            } else {
                                const long ld = a.ldo;
                                if (ok && wok[0]) orow[e[u]] = o.x;
                                if (ok && wok[1]) orow[ld + e[u]] = o.y;
                                if (ok && wok[2]) orow[2 * ld + e[u]] = o.z;
                                if (ok && wok[3]) orow[3 * ld + e[u]] = o.w;
                                if (orow_lo) {
                                    if (ok && wok[0]) orow_lo[e[u]] = tf32_lo(o.x);
                                    if (ok && wok[1]) orow_lo[ld + e[u]] = tf32_lo(o.y);
                                    if (ok && wok[2]) orow_lo[2 * ld + e[u]] = tf32_lo(o.z);
                                    if (ok && wok[3]) orow_lo[3 * ld + e[u]] = tf32_lo(o.w);
                                }
                            }
                        }
                    }
                }
            }
            __syncthreads();
            CW_TRACE();  // GroupNorm + SiLU done
        }
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
#ifdef MARLC_CNN_TRACE
    if (cta == 0 && tid == 0) {
        printf("cnn wide trace:");
        for (int i = 0; i < cw_i && i < 48; ++i) printf(" %lld", cw_tr[i]);
        printf(" | end %lld\n", clock64() - cw_t0);
    }
#endif
}

// All CW_THREADS threads of CTA `cta` (of `n_cta` cooperating CTAs) must call.
__device__ __forceinline__ void cnn_fwd_wide(const CnnFwdArgs& a, const CnnWidePlan& pl, const int cta, const int n_cta,
                                             float* sm) {
    cnn_fwd_wide_t<CW_NW>(a, pl, cta, n_cta, sm);
}

}  // namespace marlc

// Fused per-step chain kernels -- see chain.cuh.  All arithmetic fp32 (FFMA); the
// GEMM-heavy parts of a step (LSTM gates, policy/encoder block-0, dX) stay on the
// tensor cores (gemm_tc.cu); these kernels glue the small row-local pieces together
// so a rollout step is 4 launches forward and 3 backward instead of 17 + 13.
#include <initializer_list>

#include <stdlib.h>

#include "chain.cuh"
#include "cnn_wide.cuh"

namespace marlc {

constexpr int RB = 4;          // rows per CTA in the row-block roles
constexpr int CT = 256;        // threads per CTA
constexpr int WT_K = 16;       // k-extent of the staged weight tile
constexpr int WT_P = WT_K + 1; // pitch (conflict-free column reads)
constexpr float LN_EPS_C = 1e-5f;

// ---------------------------------------------------------------------------------
// row-block building blocks (every thread of the CTA must call them)
// ---------------------------------------------------------------------------------

// ys[r][n] = sum_k xT[k][r] * W[n][k] + bias[n]     (nn.Linear on RB rows)
__device__ void rb_linear(const float* xT, const float* __restrict__ W, const float* __restrict__ bias, float* ys,
                          int ldy, int N, int K, float* wt) {
    const int tid = threadIdx.x;
    const bool vec = ((K & 3) == 0) && (((uintptr_t)W & 15) == 0);
    for (int n0 = 0; n0 < N; n0 += CT) {
        float acc[RB];
#pragma unroll
        for (int r = 0; r < RB; ++r) acc[r] = 0.f;
        const int n = n0 + tid;
        for (int k0 = 0; k0 < K; k0 += WT_K) {
            if (vec) {
#pragma unroll
                for (int i = 0; i < (CT * WT_K / 4) / CT; ++i) {
                    const int idx = tid + i * CT, row = idx >> 2, c4 = idx & 3, k = k0 + 4 * c4;
                    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (n0 + row < N && k < K) v = __ldg(reinterpret_cast<const float4*>(W + (long)(n0 + row) * K + k));
                    float* d = wt + row * WT_P + 4 * c4;
                    d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
                }
            } else {
                for (int idx = tid; idx < CT * WT_K; idx += CT) {
                    const int row = idx / WT_K, kk = idx % WT_K;
                    wt[row * WT_P + kk] = (n0 + row < N && k0 + kk < K) ? __ldg(W + (long)(n0 + row) * K + k0 + kk) : 0.f;
                }
            }
            __syncthreads();
            if (n < N) {
                const int kmax = min(WT_K, K - k0);
                const float* wrow = wt + tid * WT_P;
                for (int kk = 0; kk < kmax; ++kk) {
                    const float w = wrow[kk];
                    const float4 x = *reinterpret_cast<const float4*>(xT + (k0 + kk) * RB);
                    acc[0] = fmaf(w, x.x, acc[0]); acc[1] = fmaf(w, x.y, acc[1]);
                    acc[2] = fmaf(w, x.z, acc[2]); acc[3] = fmaf(w, x.w, acc[3]);
                }
            }
            __syncthreads();
        }
        if (n < N) {
            const float b = bias ? bias[n] : 0.f;
#pragma unroll
            for (int r = 0; r < RB; ++r) ys[r * ldy + n] = acc[r] + b;
        }
    }
    __syncthreads();
}

// dx[r][k] = sum_n dyT[n][r] * W[n][k]   (input gradient; W rows are read coalesced)
// out: smem [RB][ldo] (+ optional add), nothing global
__device__ void rb_dx(const float* dyT, const float* __restrict__ W, float* out, int ldo, int N, int K) {
    for (int k = threadIdx.x; k < K; k += CT) {
        float acc[RB];
#pragma unroll
        for (int r = 0; r < RB; ++r) acc[r] = 0.f;
        for (int n = 0; n < N; ++n) {
            const float w = __ldg(W + (long)n * K + k);
            const float4 d = *reinterpret_cast<const float4*>(dyT + n * RB);
            acc[0] = fmaf(w, d.x, acc[0]); acc[1] = fmaf(w, d.y, acc[1]);
            acc[2] = fmaf(w, d.z, acc[2]); acc[3] = fmaf(w, d.w, acc[3]);
        }
#pragma unroll
        for (int r = 0; r < RB; ++r) out[r * ldo + k] = acc[r];
    }
    __syncthreads();
}


// ---- shared-memory resident weights -------------------------------------------------
// The whole weight matrix of a small layer is copied once into shared memory (coalesced
// 128-bit global loads, all independent) so the inner loops never wait on L2.
__device__ __forceinline__ void stage_w(float* dst, const float* __restrict__ W, int N, int K, int P) {
    stage_rows(dst, W, N, K, P);
}
__host__ __device__ inline int odd_pitch(int K) { return K | 1; }

// Asynchronous variant for matrices that are only walked column-wise (rb_dx_s: pitch == K needs no
// padding): 16-byte cp.async requests are issued and the thread moves on; stage_wait() + a
// __syncthreads() make the data visible.  Lets the copy overlap the first phases of a kernel.
__device__ __forceinline__ bool stage_w_async(float* dst, const float* __restrict__ W, int N, int K) {
    if (((K & 3) != 0) || ((reinterpret_cast<uintptr_t>(W) & 15) != 0)) { stage_rows(dst, W, N, K, K); return false; }
    const int tot4 = (N * K) >> 2;
    const uint32_t d0 = (uint32_t)__cvta_generic_to_shared(dst);
    for (int i = threadIdx.x; i < tot4; i += CT)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d0 + 16u * i), "l"(W + 4 * (long)i) : "memory");
    asm volatile("cp.async.commit_group;" ::: "memory");
    return true;
}
__device__ __forceinline__ void stage_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

// rb_linear with W resident in smem (row pitch P odd => conflict-free column walk)
__device__ void rb_linear_s(const float* xT, const float* Ws, int P, const float* __restrict__ bias, float* ys, int ldy,
                            int N, int K) {
    for (int n = threadIdx.x; n < N; n += CT) {
        const float* w = Ws + n * P;
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll 4
        for (int k = 0; k < K; ++k) {
            const float wv = w[k];
            const float4 x = *reinterpret_cast<const float4*>(xT + k * RB);
            a0 = fmaf(wv, x.x, a0); a1 = fmaf(wv, x.y, a1); a2 = fmaf(wv, x.z, a2); a3 = fmaf(wv, x.w, a3);
        }
        const float b = bias ? bias[n] : 0.f;
        ys[n] = a0 + b; ys[ldy + n] = a1 + b; ys[2 * ldy + n] = a2 + b; ys[3 * ldy + n] = a3 + b;
    }
    __syncthreads();
}

// rb_dx with W resident in smem
__device__ void rb_dx_s(const float* dyT, const float* Ws, int P, float* out, int ldo, int N, int K) {
    for (int k = threadIdx.x; k < K; k += CT) {
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll 4
        for (int n = 0; n < N; ++n) {
            const float wv = Ws[n * P + k];
            const float4 d = *reinterpret_cast<const float4*>(dyT + n * RB);
            a0 = fmaf(wv, d.x, a0); a1 = fmaf(wv, d.y, a1); a2 = fmaf(wv, d.z, a2); a3 = fmaf(wv, d.w, a3);
        }
        out[k] = a0; out[ldo + k] = a1; out[2 * ldo + k] = a2; out[3 * ldo + k] = a3;
    }
    __syncthreads();
}

// LayerNorm + SiLU on RB rows held in smem ys[r][n]; warp r handles row r.
//   pre_g : optional global copy of the pre-norm values (saved for backward)
//   s_g   : optional global output          sT: optional smem output, transposed [n][RB]
__device__ void rb_ln_silu(const float* ys, int ldy, int N, const float* __restrict__ gamma,
                           const float* __restrict__ beta, int rows_valid, long row0, float* pre_g, long ld_pre,
                           float* s_g, long ld_s, float* sT, float* s_lo = nullptr) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp < RB) {
        const int r = warp;
        if (r < rows_valid) {
            const float* y = ys + r * ldy;
            const float inv = 1.0f / (float)N;
            float s = 0.f;
            for (int n = lane; n < N; n += 32) s += y[n];
            const float mean = warp_sum(s) * inv;
            float v = 0.f;
            for (int n = lane; n < N; n += 32) { const float d = y[n] - mean; v += d * d; }
            const float rstd = 1.0f / sqrtf(warp_sum(v) * inv + LN_EPS_C);
            for (int n = lane; n < N; n += 32) {
                const float yv = y[n];
                if (pre_g) pre_g[(row0 + r) * ld_pre + n] = yv;
                const float o = siluf_((yv - mean) * rstd * gamma[n] + beta[n]);
                if (s_g) s_g[(row0 + r) * ld_s + n] = o;
                if (s_lo) s_lo[(row0 + r) * ld_s + n] = tf32_lo(o);
                if (sT) sT[n * RB + r] = o;
            }
        } else if (sT) {
            for (int n = lane; n < N; n += 32) sT[n * RB + r] = 0.f;
        }
    }
    __syncthreads();
}

// Backward of LayerNorm + SiLU on RB rows.
//   ds   [RB][ld] smem: incoming gradient w.r.t. the block output (DESTROYED: becomes dz)
//   ypre [RB][ld] smem: saved pre-norm values                      (DESTROYED: becomes xhat)
//   dy   [RB][ld] smem out; dyT [N][RB] smem out (optional); dy_g global out (optional)
//   dgamma / dbeta / dbias: global accumulators (atomicAdd of the RB-row partial sums)
__device__ void rb_ln_silu_bwd(float* ds, float* ypre, int ld, int N, const float* __restrict__ gamma,
                               const float* __restrict__ beta, int rows_valid, long row0, float* dy, float* dyT,
                               float* dy_g, long ld_dyg, float* dgamma, float* dbeta, float* dbias) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp < RB) {
        const int r = warp;
        float* y = ypre + r * ld;
        float* g = ds + r * ld;
        if (r < rows_valid) {
            const float inv = 1.0f / (float)N;
            float s = 0.f;
            for (int n = lane; n < N; n += 32) s += y[n];
            const float mean = warp_sum(s) * inv;
            float v = 0.f;
            for (int n = lane; n < N; n += 32) { const float d = y[n] - mean; v += d * d; }
            const float rstd = 1.0f / sqrtf(warp_sum(v) * inv + LN_EPS_C);
            float c1 = 0.f, c2 = 0.f;
            for (int n = lane; n < N; n += 32) {
                const float xh = (y[n] - mean) * rstd;
                const float dz = g[n] * silu_grad_(xh * gamma[n] + beta[n]);
                const float dxh = dz * gamma[n];
                c1 += dxh;
                c2 += dxh * xh;
                y[n] = xh;
                g[n] = dz;
            }
            c1 = warp_sum(c1) * inv;
            c2 = warp_sum(c2) * inv;
            for (int n = lane; n < N; n += 32) {
                const float o = rstd * (g[n] * gamma[n] - c1 - y[n] * c2);
                dy[r * ld + n] = o;
                if (dyT) dyT[n * RB + r] = o;
                if (dy_g) dy_g[(row0 + r) * ld_dyg + n] = o;
            }
        } else {
            for (int n = lane; n < N; n += 32) {
                y[n] = 0.f; g[n] = 0.f; dy[r * ld + n] = 0.f;
                if (dyT) dyT[n * RB + r] = 0.f;
            }
        }
    }
    __syncthreads();
    for (int n = threadIdx.x; n < N; n += CT) {
        float a = 0.f, b = 0.f, c = 0.f;
#pragma unroll
        for (int r = 0; r < RB; ++r) {
            a += ds[r * ld + n] * ypre[r * ld + n];
            b += ds[r * ld + n];
            c += dy[r * ld + n];
        }
        if (dgamma) atomicAdd(dgamma + n, a);
        if (dbeta) atomicAdd(dbeta + n, b);
        if (dbias) atomicAdd(dbias + n, c);
    }
    __syncthreads();
}

// (sum over the other agents of the same image) / (Na - 1): message.py:5-17 and its adjoint
__device__ __forceinline__ float other_agents_mean(const float* __restrict__ x, int m, int j, int Na, int Nb, int n) {
    if (Na <= 1) return 0.f;
    const int b = m % Nb;
    const float* base = x + (long)b * n + j;
    const long stride = (long)Nb * n;
    float s = 0.f;
    int a = 0;
    for (; a + 8 <= Na; a += 8) {  // 8 loads in flight, then the adds
        float v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = base[(a + i) * stride];
        s += ((v[0] + v[1]) + (v[2] + v[3])) + ((v[4] + v[5]) + (v[6] + v[7]));
    }
    for (; a < Na; ++a) s += base[a * stride];
    return (s - x[(long)m * n + j]) / (float)(Na - 1);
}

struct ChainSmem {
    float *bufA, *bufB, *bufC, *bufT, *wt, *wres;
    __device__ ChainSmem(float* sm, int maxw) {
        bufA = sm; bufB = bufA + RB * maxw; bufC = bufB + RB * maxw; bufT = bufC + RB * maxw; wt = bufT + RB * maxw;
        wres = wt + CT * WT_P;
    }
};
static size_t chain_smem_bytes(int maxw) { return sizeof(float) * ((size_t)4 * RB * maxw + (size_t)CT * WT_P); }
constexpr size_t CHAIN_SMEM_LIMIT = 200 * 1024;
// floats of staged weights for two matrices, or 0 if they do not fit next to the row buffers
static int staged_floats(int maxw, int n1, int p1, int n2, int p2) {
    const size_t w = (size_t)n1 * p1 + (size_t)n2 * p2;
    return (chain_smem_bytes(maxw) + sizeof(float) * w <= CHAIN_SMEM_LIMIT) ? (int)w : 0;
}
// Weights are staged whenever they fit: resident in shared memory they make ONE row block fast (no L2 round trips
// inside its dependent chain), at 80-190 KB per CTA (one CTA = 4 rows per SM at a time).  Wider layers read them
// through L1/L2.
static int maxw_of(std::initializer_list<int> v) {
    int m = 4;
    for (int x : v) m = max(m, x);
    return (m + 3) & ~3;
}
ChainStage step_pre_stage(int n_m, int n1, int n2, int nd) {
    const int maxw = maxw_of({n_m, n1, n2, nd});
    return {maxw, staged_floats(maxw, n1, odd_pitch(n_m), n2, odd_pitch(n1))};
}
ChainStage step_post_stage(int n1, int n2) {
    const int maxw = maxw_of({n1, n2});
    return {maxw, staged_floats(maxw, n2, odd_pitch(n1), 0, 0)};
}
ChainStage bwd_pre_stage(int n_m, int n1, int nb) {
    const int maxw = maxw_of({n_m, n1, nb});
    return {maxw, staged_floats(maxw, n_m, n1, n1, nb)};
}
ChainStage bwd_post_stage(int n_m, int n1, int n2) {
    const int maxw = maxw_of({n_m, n1, n2});
    return {maxw, staged_floats(maxw, n2, n1, n1, n_m)};
}

// ---------------------------------------------------------------------------------
// forward "pre": CNN role (blocks [0,M)) | decoder + position-feature role
// ---------------------------------------------------------------------------------
// Many windows per step (sharded-batch configurations): grid = feature-extractor CTAs (first, so they are
// scheduled first) + decoder CTAs, all persistent.
//   cnn_blocks: wide feature extractor (cnn_wide.cuh), each CTA loops over batches of CW_NW windows;
//   dec_blocks: PERSISTENT row-block CTAs: weights and LayerNorm affines are staged once per CTA, then the CTA
//               walks row blocks rb = i, i + dec_blocks, ...  (At 4096 rows a step had 1024 CTAs that each
//               re-staged 82 KB of decoder weights for 4 rows: 81 us per step, ncu launch list round 2.)
struct StepPreWideArgs { StepPreArgs a; int maxw; int staged; int cnn_blocks; int dec_blocks; int trig; CnnWidePlan wide; };

__global__ void __launch_bounds__(CT, 1) step_pre_wide_kernel(const StepPreWideArgs ka) {
    extern __shared__ __align__(16) float sm[];
    const StepPreArgs& a = ka.a;
    if (ka.trig) pdl_trigger();  // step chain: the LSTM GEMM's CTAs may set up while this kernel runs (common.cuh)
    if ((int)blockIdx.x < ka.cnn_blocks) {
        cnn_fwd_wide(a.cnn, ka.wide, blockIdx.x, ka.cnn_blocks, sm);
        return;
    }
    const int db = (int)blockIdx.x - ka.cnn_blocks;
    const int nrb = (a.M + RB - 1) / RB;
    const int n_m = a.d0.n_in, n1 = a.d0.n_out, n2 = a.d3.n_out;
    ChainSmem S(sm, ka.maxw);
    const int P0 = odd_pitch(n_m), P3 = odd_pitch(n1);
    float* W0s = S.wres;
    float* W3s = W0s + n1 * P0;
    const int tid = threadIdx.x;
    const bool fast = ka.staged && RB * n_m <= CT && n1 <= CT && n2 <= CT && 2 * (n1 + n2) <= CT * WT_P;
    float* sG0 = S.wt;  // fast path: LayerNorm affines parked in the (otherwise unused) weight-tile scratch
    float* sB0 = sG0 + n1;
    float* sG3 = sB0 + n1;
    float* sB3 = sG3 + n2;
    const int mr = tid / n_m, mj = tid - mr * n_m;  // fast path: (row, column) of the collected message this thread owns
    auto load_mean = [&](int rb) -> float {
        const int row0 = rb * RB;
        return (tid < RB * n_m && rb < nrb && row0 + mr < a.M) ? other_agents_mean(a.msg_in, row0 + mr, mj, a.Na, a.Nb, n_m) : 0.f;
    };
    // ---- once per CTA: the launch constants (affines, synchronously staged weights) first -- under a programmatic
    //      dependent launch this part overlaps the previous kernel of the step chain -- then, after pdl_wait(), the
    //      first row block's message mean (produced by that kernel)
    if (fast) {
        float g0 = 0.f, b0 = 0.f, g3 = 0.f, b3 = 0.f;
        if (tid < n1) { g0 = a.d0.g[tid]; b0 = a.d0.be[tid]; }
        if (tid < n2) { g3 = a.d3.g[tid]; b3 = a.d3.be[tid]; }
        stage_w(W0s, a.d0.W, n1, n_m, P0);
        stage_w(W3s, a.d3.W, n2, n1, P3);
        if (tid < n1) { sG0[tid] = g0; sB0[tid] = b0; }
        if (tid < n2) { sG3[tid] = g3; sB3[tid] = b3; }
    } else if (ka.staged) {
        stage_w(W0s, a.d0.W, n1, n_m, P0);
        stage_w(W3s, a.d3.W, n2, n1, P3);
    }
    pdl_wait();
    float mv = fast ? load_mean(db) : 0.f;
    for (int rb = db; rb < nrb; rb += ka.dec_blocks) {
        const int row0 = rb * RB;
        const int rows_valid = min(RB, a.M - row0);
        if (fast) {
            if (tid < RB * n_m) {
                if (mr < rows_valid) a.coll[(long)(row0 + mr) * n_m + mj] = mv;
                S.bufT[mj * RB + mr] = mv;
            }
            __syncthreads();
            mv = load_mean(rb + ka.dec_blocks);  // next row block's operand, in flight under this block's chain
            rb_linear_s(S.bufT, W0s, P0, a.d0.b, S.bufA, ka.maxw, n1, n_m);
            rb_ln_silu(S.bufA, ka.maxw, n1, sG0, sB0, rows_valid, row0, a.dec_y1, n1, a.dec_s1, n1, S.bufT);
            rb_linear_s(S.bufT, W3s, P3, a.d3.b, S.bufA, ka.maxw, n2, n1);
            rb_ln_silu(S.bufA, ka.maxw, n2, sG3, sB3, rows_valid, row0, a.dec_y2, n2, a.U + a.F, a.ldu, nullptr,
                       a.U_lo ? a.U_lo + a.F : nullptr);
        } else {
            // collected message (mean of the other agents)                      message.py:5-17
            for (int e = tid; e < RB * n_m; e += CT) {
                const int r = e / n_m, j = e % n_m;
                float v = 0.f;
                if (r < rows_valid) {
                    v = other_agents_mean(a.msg_in, row0 + r, j, a.Na, a.Nb, n_m);
                    a.coll[(long)(row0 + r) * n_m + j] = v;
                }
                S.bufT[j * RB + r] = v;
            }
            __syncthreads();
            // decoder block 0 and block 3                                        message.py:36-49
            if (ka.staged) rb_linear_s(S.bufT, W0s, P0, a.d0.b, S.bufA, ka.maxw, n1, n_m);
            else rb_linear(S.bufT, a.d0.W, a.d0.b, S.bufA, ka.maxw, n1, n_m, S.wt);
            rb_ln_silu(S.bufA, ka.maxw, n1, a.d0.g, a.d0.be, rows_valid, row0, a.dec_y1, n1, a.dec_s1, n1, S.bufT);
            if (ka.staged) rb_linear_s(S.bufT, W3s, P3, a.d3.b, S.bufA, ka.maxw, n2, n1);
            else rb_linear(S.bufT, a.d3.W, a.d3.b, S.bufA, ka.maxw, n2, n1, S.wt);
            rb_ln_silu(S.bufA, ka.maxw, n2, a.d3.g, a.d3.be, rows_valid, row0, a.dec_y2, n2, a.U + a.F, a.ldu, nullptr,
                       a.U_lo ? a.U_lo + a.F : nullptr);
        }
        // position features                                                  state.py:7-17
        {
            const int warp = tid >> 5, lane = tid & 31, nd = a.pos.n_out;
            if (warp < rows_valid) {
                const long m = row0 + warp;
                const float p0 = a.npos[2 * m], p1 = a.npos[2 * m + 1];
                const float inv = 1.0f / (float)nd;
                float sum = 0.f;
                for (int j = lane; j < nd; j += 32) {
                    const float y = fmaf(p1, a.pos.W[2 * j + 1], p0 * a.pos.W[2 * j]) + a.pos.b[j];
                    a.pos_y[m * nd + j] = y;
                    S.bufB[warp * ka.maxw + j] = y;
                    sum += y;
                }
                const float mean = warp_sum(sum) * inv;
                float v = 0.f;
                for (int j = lane; j < nd; j += 32) { const float d = S.bufB[warp * ka.maxw + j] - mean; v += d * d; }
                const float rstd = 1.0f / sqrtf(warp_sum(v) * inv + LN_EPS_C);
                float* o = a.U + m * a.ldu + a.F + n2;
                float* ol = a.U_lo ? a.U_lo + m * a.ldu + a.F + n2 : nullptr;
                for (int j = lane; j < nd; j += 32) {
                    const float v2 = siluf_((S.bufB[warp * ka.maxw + j] - mean) * rstd * a.pos.g[j] + a.pos.be[j]);
                    o[j] = v2;
                    if (ol) ol[j] = tf32_lo(v2);
                }
            }
        }
        __syncthreads();  // the row buffers are reused by the next row block
    }
}

// CTAs of a persistent row-block role: every row block gets its own CTA while that fits in `waves` waves of the
// machine (the latency-bound regime: nothing to amortise), more rows make the CTAs loop
static int persistent_blocks(int nrb, size_t smem_bytes, int waves = 1) {
    const int per_sm = (int)max((size_t)1, min((size_t)8, (size_t)(220 * 1024) / max(smem_bytes, (size_t)1)));
    return max(1, min(nrb, MARLC_SMS * per_sm * waves));
}

static int step_pre_small(const StepPreArgs& a, cudaStream_t s);

constexpr int CNN_WIDE_MIN = 256;
StepPrePlan step_pre_plan(const CnnDesc& d, bool have_img, bool have_wT, int M, CnnWidePlan* wide) {
    // feature extractor: one CTA per window while a step has few windows (latency-bound, every SM gets one:
    // step_pre_kernel); from CNN_WIDE_MIN windows on, persistent CTAs with stationary weights, CW_NW windows
    // per pass, next to persistent decoder CTAs (step_pre_wide_kernel)
    CnnWidePlan w;
    memset(&w, 0, sizeof(w));
    if (M >= CNN_WIDE_MIN) w = cnn_wide_plan(d, have_img, have_wT);
    if (wide) *wide = w;
    StepPrePlan p;
    p.nw = w.ok ? CW_NW : 1;
    p.cnn_blocks = w.ok ? min((M + CW_NW - 1) / CW_NW, MARLC_SMS) : 0;
    return p;
}

int step_pre(const StepPreArgs& a, cudaStream_t s) {
    if (a.M <= 0) return 0;
    static_assert(CW_THREADS == CT, "the wide feature extractor runs inside the chain kernel's CTA shape");
    StepPreWideArgs ka;
    // (the chain path keeps transposed conv weights: engine.cu allocates them whenever the chains are on)
    const StepPrePlan pl = step_pre_plan(a.cnn.d, a.cnn.img != nullptr && a.cnn.patch == nullptr, true, a.M, &ka.wide);
    if (!ka.wide.ok) return step_pre_small(a, s);
    ka.a = a;
    const ChainStage st = step_pre_stage(a.d0.n_in, a.d0.n_out, a.d3.n_out, a.pos.n_out);
    ka.maxw = st.maxw;
    const int wfl = st.wfl;
    ka.staged = wfl > 0;
    ka.cnn_blocks = pl.cnn_blocks;
    const size_t smem = max(chain_smem_bytes(ka.maxw) + sizeof(float) * (size_t)wfl, sizeof(float) * (size_t)ka.wide.smem_floats);
    MARLC_CHECK(smem <= 226 * 1024, "step_pre: shared memory %zu B too large", smem);
    static size_t attr = 0;
    if (smem > 48 * 1024 && smem > attr) {
        MARLC_CUDA(cudaFuncSetAttribute(step_pre_wide_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr = smem;
    }
    // (the launch's shared memory is the larger role's: one CTA per SM, so the decoder CTAs share the SMs with the
    //  feature extractor's in time; one wave of them)
    ka.dec_blocks = persistent_blocks((a.M + RB - 1) / RB, smem);
    const int grid = ka.cnn_blocks + ka.dec_blocks;
    ka.trig = pdl_trigger_early();
    MARLC_CUDA(launch_pdl(step_pre_wide_kernel, dim3(grid), dim3(CT), smem, s, ka));
    MARLC_LAUNCH_CHECK();
    return 0;
}

struct StepPreKernelArgs { StepPreArgs a; int maxw; int staged; int trig; };

__global__ void __launch_bounds__(CT) step_pre_kernel(const StepPreKernelArgs ka) {
    extern __shared__ __align__(16) float sm[];
    const StepPreArgs& a = ka.a;
    if (ka.trig) pdl_trigger();  // step chain: the LSTM GEMM's CTAs may set up while this kernel runs (common.cuh)
    if ((int)blockIdx.x < a.M) {
        cnn_fwd_block(a.cnn, blockIdx.x, sm);  // (waits for the previous kernel before it reads the window position)
        return;
    }
    const int row0 = ((int)blockIdx.x - a.M) * RB;
    const int rows_valid = min(RB, a.M - row0);
    const int n_m = a.d0.n_in, n1 = a.d0.n_out, n2 = a.d3.n_out;
    ChainSmem S(sm, ka.maxw);
    const int P0 = odd_pitch(n_m), P3 = odd_pitch(n1);
    float* W0s = S.wres;
    float* W3s = W0s + n1 * P0;
    if (ka.staged && RB * n_m <= CT && n1 <= CT && n2 <= CT && 2 * (n1 + n2) <= CT * WT_P) {
        // every global operand requested up front, grouped ahead of any use (see bwd_pre): the message
        // mean and the LayerNorm affines first, then the (synchronously staged) weights
        float* sG0 = S.wt;
        float* sB0 = sG0 + n1;
        float* sG3 = sB0 + n1;
        float* sB3 = sG3 + n2;
        const int tid = threadIdx.x;
        float mv = 0.f;
        const int r = tid / n_m, j = tid - r * n_m;
        pdl_wait();  // the messages come from the previous kernel of the step chain
        if (tid < RB * n_m && r < rows_valid) mv = other_agents_mean(a.msg_in, row0 + r, j, a.Na, a.Nb, n_m);
        float g0 = 0.f, b0 = 0.f, g3 = 0.f, b3 = 0.f;
        if (tid < n1) { g0 = a.d0.g[tid]; b0 = a.d0.be[tid]; }
        if (tid < n2) { g3 = a.d3.g[tid]; b3 = a.d3.be[tid]; }
        stage_w(W0s, a.d0.W, n1, n_m, P0);
        stage_w(W3s, a.d3.W, n2, n1, P3);
        if (tid < n1) { sG0[tid] = g0; sB0[tid] = b0; }
        if (tid < n2) { sG3[tid] = g3; sB3[tid] = b3; }
        if (tid < RB * n_m) {
            if (r < rows_valid) a.coll[(long)(row0 + r) * n_m + j] = mv;
            S.bufT[j * RB + r] = mv;
        }
        __syncthreads();
        rb_linear_s(S.bufT, W0s, P0, a.d0.b, S.bufA, ka.maxw, n1, n_m);
        rb_ln_silu(S.bufA, ka.maxw, n1, sG0, sB0, rows_valid, row0, a.dec_y1, n1, a.dec_s1, n1, S.bufT);
        rb_linear_s(S.bufT, W3s, P3, a.d3.b, S.bufA, ka.maxw, n2, n1);
        rb_ln_silu(S.bufA, ka.maxw, n2, sG3, sB3, rows_valid, row0, a.dec_y2, n2, a.U + a.F, a.ldu, nullptr,
                   a.U_lo ? a.U_lo + a.F : nullptr);
    } else {
    if (ka.staged) { stage_w(W0s, a.d0.W, n1, n_m, P0); stage_w(W3s, a.d3.W, n2, n1, P3); }
    pdl_wait();
    // collected message (mean of the other agents)                      message.py:5-17
    for (int e = threadIdx.x; e < RB * n_m; e += CT) {
        const int r = e / n_m, j = e % n_m;
        float v = 0.f;
        if (r < rows_valid) {
            v = other_agents_mean(a.msg_in, row0 + r, j, a.Na, a.Nb, n_m);
            a.coll[(long)(row0 + r) * n_m + j] = v;
        }
        S.bufT[j * RB + r] = v;
    }
    __syncthreads();
    // decoder block 0 and block 3                                        message.py:36-49
    if (ka.staged) rb_linear_s(S.bufT, W0s, P0, a.d0.b, S.bufA, ka.maxw, n1, n_m);
    else rb_linear(S.bufT, a.d0.W, a.d0.b, S.bufA, ka.maxw, n1, n_m, S.wt);
    rb_ln_silu(S.bufA, ka.maxw, n1, a.d0.g, a.d0.be, rows_valid, row0, a.dec_y1, n1, a.dec_s1, n1, S.bufT);
    if (ka.staged) rb_linear_s(S.bufT, W3s, P3, a.d3.b, S.bufA, ka.maxw, n2, n1);
    else rb_linear(S.bufT, a.d3.W, a.d3.b, S.bufA, ka.maxw, n2, n1, S.wt);
    rb_ln_silu(S.bufA, ka.maxw, n2, a.d3.g, a.d3.be, rows_valid, row0, a.dec_y2, n2, a.U + a.F, a.ldu, nullptr,
               a.U_lo ? a.U_lo + a.F : nullptr);
    }
    // position features                                                  state.py:7-17
    {
        const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nd = a.pos.n_out;
        if (warp < rows_valid) {
            const long m = row0 + warp;
            const float p0 = a.npos[2 * m], p1 = a.npos[2 * m + 1];
            const float inv = 1.0f / (float)nd;
            float s = 0.f;
            for (int j = lane; j < nd; j += 32) {
                const float y = fmaf(p1, a.pos.W[2 * j + 1], p0 * a.pos.W[2 * j]) + a.pos.b[j];
                a.pos_y[m * nd + j] = y;
                S.bufB[warp * ka.maxw + j] = y;
                s += y;
            }
            const float mean = warp_sum(s) * inv;
            float v = 0.f;
            for (int j = lane; j < nd; j += 32) { const float d = S.bufB[warp * ka.maxw + j] - mean; v += d * d; }
            const float rstd = 1.0f / sqrtf(warp_sum(v) * inv + LN_EPS_C);
            float* o = a.U + m * a.ldu + a.F + n2;
            float* ol = a.U_lo ? a.U_lo + m * a.ldu + a.F + n2 : nullptr;
            for (int j = lane; j < nd; j += 32) {
                const float v2 = siluf_((S.bufB[warp * ka.maxw + j] - mean) * rstd * a.pos.g[j] + a.pos.be[j]);
                o[j] = v2;
                if (ol) ol[j] = tf32_lo(v2);
            }
        }
    }
}

static int step_pre_small(const StepPreArgs& a, cudaStream_t s) {
    if (a.M <= 0) return 0;
    StepPreKernelArgs ka;
    ka.a = a;
    const ChainStage st = step_pre_stage(a.d0.n_in, a.d0.n_out, a.d3.n_out, a.pos.n_out);
    ka.maxw = st.maxw;
    const int wfl = st.wfl;
    ka.staged = wfl > 0;
    const size_t smem = max(chain_smem_bytes(ka.maxw) + sizeof(float) * (size_t)wfl, cnn_fwd_smem_bytes(a.cnn));
    MARLC_CHECK(smem <= 200 * 1024, "step_pre: shared memory %zu B too large", smem);
    static size_t attr = 0;
    if (smem > 48 * 1024 && smem > attr) {
        MARLC_CUDA(cudaFuncSetAttribute(step_pre_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr = smem;
    }
    const int grid = a.M + (a.M + RB - 1) / RB;
    ka.trig = pdl_trigger_early();
    MARLC_CUDA(launch_pdl(step_pre_kernel, dim3(grid), dim3(CT), smem, s, ka));
    MARLC_LAUNCH_CHECK();
    return 0;
}

// ---------------------------------------------------------------------------------
// forward "post": policy tail + sampling + transition (warp per row) | encoder tail (row blocks)
// ---------------------------------------------------------------------------------
constexpr int MAX_ACT = 16;

// One warp per row.  Every global operand of the row (pre-norm activations, LayerNorm affine, the
// nb_action rows of the final Linear) is requested up front into registers, so the row pays ONE
// exposed memory round trip instead of one per pass (measured: the serial version spent 40 % of
// its samples waiting on these loads).  NCOL = ceil(nl / 32) columns per lane, <= 16.
template <int NCOL>
__device__ __forceinline__ void policy_logits_regs(const StepPostArgs& a, const int m, float* logit) {
    const PolicyActArgs& p = a.act;
    const int lane = threadIdx.x & 31, nl = p.nl;
    const float* y = a.pol_y1 + (long)m * nl;
    float yv[NCOL], gv[NCOL], bv[NCOL];
#pragma unroll
    for (int i = 0; i < NCOL; ++i) {
        const int k = lane + 32 * i;
        const bool ok = k < nl;
        yv[i] = ok ? y[k] : 0.f;
        gv[i] = ok ? a.pol_g[k] : 0.f;
        bv[i] = ok ? a.pol_be[k] : 0.f;
    }
    const float inv = 1.0f / (float)nl;
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < NCOL; ++i) s += yv[i];
    const float mean = warp_sum(s) * inv;
    float v = 0.f;
#pragma unroll
    for (int i = 0; i < NCOL; ++i)
        if (lane + 32 * i < nl) { const float d = yv[i] - mean; v += d * d; }
    const float rstd = 1.0f / sqrtf(warp_sum(v) * inv + LN_EPS_C);
    float* s1 = const_cast<float*>(p.s1) + (long)m * nl;
#pragma unroll
    for (int i = 0; i < NCOL; ++i) {
        const int k = lane + 32 * i;
        yv[i] = (k < nl) ? siluf_((yv[i] - mean) * rstd * gv[i] + bv[i]) : 0.f;
        if (k < nl) s1[k] = yv[i];  // saved for the batched weight gradient of policy.3
    }
    for (int j0 = 0; j0 < p.nA; j0 += 4) {  // four rows of W3 in flight at a time
        float d[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) {
            if (j0 + jj < p.nA) {
                const float* w = p.W3 + (long)(j0 + jj) * nl;
#pragma unroll
                for (int i = 0; i < NCOL; ++i)
                    if (lane + 32 * i < nl) d[jj] = fmaf(yv[i], __ldg(w + lane + 32 * i), d[jj]);
            }
        }
#pragma unroll
        for (int jj = 0; jj < 4; ++jj)
            if (j0 + jj < p.nA) logit[j0 + jj] = warp_sum(d[jj]) + p.b3[j0 + jj];
    }
}

__device__ void policy_tail_row(const StepPostArgs& a, const int m, float* srow /* smem [nl] */) {
    const PolicyActArgs& p = a.act;
    const int lane = threadIdx.x & 31, nl = p.nl;
    float logit[MAX_ACT];
    if (nl <= 128) policy_logits_regs<4>(a, m, logit);
    else if (nl <= 256) policy_logits_regs<8>(a, m, logit);
    else if (nl <= 384) policy_logits_regs<12>(a, m, logit);
    else if (nl <= 512) policy_logits_regs<16>(a, m, logit);
    else {
        const float* y = a.pol_y1 + (long)m * nl;
        const float inv = 1.0f / (float)nl;
        float s = 0.f;
        for (int k = lane; k < nl; k += 32) s += y[k];
        const float mean = warp_sum(s) * inv;
        float v = 0.f;
        for (int k = lane; k < nl; k += 32) { const float d = y[k] - mean; v += d * d; }
        const float rstd = 1.0f / sqrtf(warp_sum(v) * inv + LN_EPS_C);
        float* s1 = const_cast<float*>(p.s1) + (long)m * nl;
        for (int k = lane; k < nl; k += 32) {
            const float o = siluf_((y[k] - mean) * rstd * a.pol_g[k] + a.pol_be[k]);
            s1[k] = o;      // saved for the batched weight gradient of policy.3
            srow[k] = o;
        }
        __syncwarp();
#pragma unroll 1
        for (int j = 0; j < p.nA; ++j) {
            const float* w = p.W3 + (long)j * nl;
            float d = 0.f;
            for (int k = lane; k < nl; k += 32) d = fmaf(srow[k], w[k], d);
            logit[j] = warp_sum(d) + p.b3[j];
        }
    }
    float mx = -INFINITY;
    for (int j = 0; j < p.nA; ++j) mx = fmaxf(mx, logit[j]);
    float den = 0.f;
    for (int j = 0; j < p.nA; ++j) { logit[j] = expf(logit[j] - mx); den += logit[j]; }
    const float invd = 1.0f / den;
    int act;
    if (p.act_in) act = (int)p.act_in[m];
    else {
        const uint64_t episode = p.rng_state[1];
        const Philox ph(p.rng_state[0]);
        const uint4 r = ph((uint64_t)p.t * (uint64_t)p.M + (uint64_t)m, (episode << 8) | 7);
        const float u = u01(r.x);
        float cdf = 0.f;
        act = p.nA - 1;
        for (int j = 0; j < p.nA; ++j) {
            cdf += logit[j] * invd;
            if (u < cdf) { act = j; break; }
        }
    }
    if (lane == 0) {
        float pa = 0.f;
        for (int j = 0; j < p.nA; ++j) {
            const float pr = logit[j] * invd;
            p.probs[(long)m * p.nA + j] = pr;
            if (j == act) pa = pr;
        }
        p.logp[m] = logf(pa);
        p.act_out[m] = act;
        int py = p.pos_in[2 * m], px = p.pos_in[2 * m + 1];
        if (act >= 0 && act < p.nA) {
            const int ny = py + p.moves[2 * act], nx = px + p.moves[2 * act + 1];
            if ((ny >= 0) & (ny + p.f < p.H) & (nx >= 0) & (nx + p.f < p.W)) { py = ny; px = nx; }
        }
        p.pos_out[2 * m] = py; p.pos_out[2 * m + 1] = px;
        p.step_pos[2 * (long)m] = py; p.step_pos[2 * (long)m + 1] = px;
        p.npos_out[2 * m] = (float)py / (float)p.H;
        p.npos_out[2 * m + 1] = (float)px / (float)p.W;
    }
}

struct StepPostKernelArgs { StepPostArgs a; int maxw; int pol_blocks; int staged; int trig; };

__global__ void __launch_bounds__(CT) step_post_kernel(const StepPostKernelArgs ka) {
    extern __shared__ __align__(16) float sm[];
    const StepPostArgs& a = ka.a;
    if (ka.trig) pdl_trigger();  // step chain: the next step's "pre" kernel may set up (stage its weights) while this one runs
    if ((int)blockIdx.x < ka.pol_blocks) {
        const int warp = threadIdx.x >> 5;
        const int m = blockIdx.x * (CT / 32) + warp;
        pdl_wait();  // pol_y1 comes from the block-0 GEMMs
        if (m < a.M) policy_tail_row(a, m, sm + warp * a.act.nl);
        return;
    }
    const int row0 = ((int)blockIdx.x - ka.pol_blocks) * RB;
    const int rows_valid = min(RB, a.M - row0);
    const int n1 = a.e3.n_in, n2 = a.e3.n_out;
    ChainSmem S(sm, ka.maxw);
    const int P3 = odd_pitch(n1);
    if (ka.staged && RB * n1 <= 2 * CT && n1 <= CT && n2 <= CT && 2 * (n1 + n2) <= CT * WT_P) {
        // every global operand requested up front, grouped ahead of any use (see bwd_pre)
        float* sG1 = S.wt;
        float* sB1 = sG1 + n1;
        float* sG3 = sB1 + n1;
        float* sB3 = sG3 + n2;
        const int tid = threadIdx.x;
        float y1v[2] = {0.f, 0.f};
        int r1[2], k1[2];
#pragma unroll
        for (int i = 0; i < 2; ++i) { const int e = tid + i * CT; r1[i] = e / n1; k1[i] = e - r1[i] * n1; }
        pdl_wait();  // enc_y1 comes from the block-0 GEMMs
#pragma unroll
        for (int i = 0; i < 2; ++i)
            if (r1[i] < rows_valid) y1v[i] = a.enc_y1[(long)(row0 + r1[i]) * n1 + k1[i]];
        float g1 = 0.f, b1 = 0.f, g3 = 0.f, b3 = 0.f;
        if (tid < n1) { g1 = a.enc_g[tid]; b1 = a.enc_be[tid]; }
        if (tid < n2) { g3 = a.e3.g[tid]; b3 = a.e3.be[tid]; }
        stage_w(S.wres, a.e3.W, n2, n1, P3);
        if (tid < n1) { sG1[tid] = g1; sB1[tid] = b1; }
        if (tid < n2) { sG3[tid] = g3; sB3[tid] = b3; }
#pragma unroll
        for (int i = 0; i < 2; ++i)
            if (r1[i] < RB) S.bufA[r1[i] * ka.maxw + k1[i]] = y1v[i];
        __syncthreads();
        rb_ln_silu(S.bufA, ka.maxw, n1, sG1, sB1, rows_valid, row0, nullptr, 0, a.enc_s1, n1, S.bufT);
        rb_linear_s(S.bufT, S.wres, P3, a.e3.b, S.bufA, ka.maxw, n2, n1);
        rb_ln_silu(S.bufA, ka.maxw, n2, sG3, sB3, rows_valid, row0, a.enc_y2, n2, a.msg_out, n2, nullptr);
        return;
    }
    if (ka.staged) stage_w(S.wres, a.e3.W, n2, n1, P3);
    pdl_wait();
    for (int e = threadIdx.x; e < RB * n1; e += CT) {
        const int r = e / n1, k = e % n1;
        S.bufA[r * ka.maxw + k] = r < rows_valid ? a.enc_y1[(long)(row0 + r) * n1 + k] : 0.f;
    }
    __syncthreads();
    rb_ln_silu(S.bufA, ka.maxw, n1, a.enc_g, a.enc_be, rows_valid, row0, nullptr, 0, a.enc_s1, n1, S.bufT);
    if (ka.staged) rb_linear_s(S.bufT, S.wres, P3, a.e3.b, S.bufA, ka.maxw, n2, n1);
    else rb_linear(S.bufT, a.e3.W, a.e3.b, S.bufA, ka.maxw, n2, n1, S.wt);
    rb_ln_silu(S.bufA, ka.maxw, n2, a.e3.g, a.e3.be, rows_valid, row0, a.enc_y2, n2, a.msg_out, n2, nullptr);
}

int step_post(const StepPostArgs& a, cudaStream_t s) {
    if (a.M <= 0) return 0;
    MARLC_CHECK(a.act.nA <= MAX_ACT, "step_post: nb_action=%d > %d", a.act.nA, MAX_ACT);
    StepPostKernelArgs ka;
    ka.a = a;
    const ChainStage st = step_post_stage(a.e3.n_in, a.e3.n_out);
    ka.maxw = st.maxw;
    ka.pol_blocks = (a.M + CT / 32 - 1) / (CT / 32);
    const int wfl = st.wfl;
    ka.staged = wfl > 0;
    const size_t smem = max(chain_smem_bytes(ka.maxw) + sizeof(float) * (size_t)wfl, sizeof(float) * (size_t)(CT / 32) * a.act.nl);
    MARLC_CHECK(smem <= 200 * 1024, "step_post: shared memory %zu B too large", smem);
    static size_t attr = 0;
    if (smem > 48 * 1024 && smem > attr) {
        MARLC_CUDA(cudaFuncSetAttribute(step_post_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr = smem;
    }
    const int grid = ka.pol_blocks + (a.M + RB - 1) / RB;
    ka.trig = pdl_trigger_early();
    MARLC_CUDA(launch_pdl(step_post_kernel, dim3(grid), dim3(CT), smem, s, ka));
    MARLC_LAUNCH_CHECK();
    return 0;
}

// ---------------------------------------------------------------------------------
// backward "pre" (step t): adjoint message mean -> encoder backward -> dh += ... -> both LSTM cells
// ---------------------------------------------------------------------------------

// Point-wise LSTM backward for RB rows of one cell (recurrent.py:30).  Columns are strided over the
// threads, the RB rows are unrolled so their ~9 loads each are all in flight together.
__device__ __forceinline__ void cell_bwd_rows(const int row0, const int rows_valid, const int n,
                                              const float* __restrict__ gates, const float* __restrict__ dh_heads,
                                              const float* __restrict__ dh_carry, const float* __restrict__ dc_next,
                                              const float* __restrict__ c_prev, const float* __restrict__ c_new,
                                              const float* dhx, const int ldx, float* __restrict__ dgates,
                                              float* __restrict__ dgates_lo, float* __restrict__ dc_prev) {
    for (int j = threadIdx.x; j < n; j += CT) {
        float gi[RB], gf[RB], gg[RB], go[RB], dh[RB], dcn[RB], cp[RB], cn[RB];
#pragma unroll
        for (int r = 0; r < RB; ++r) {
            if (r < rows_valid) {
                const long m = row0 + r, idx = m * n + j;
                const float* g = gates + m * 4 * n;
                gi[r] = g[j]; gf[r] = g[n + j]; gg[r] = g[2 * n + j]; go[r] = g[3 * n + j];
                dh[r] = dh_heads[idx] + (dh_carry ? dh_carry[idx] : 0.f);
                dcn[r] = dc_next ? dc_next[idx] : 0.f;
                cp[r] = c_prev[idx]; cn[r] = c_new[idx];
            }
        }
#pragma unroll
        for (int r = 0; r < RB; ++r) {
            if (r < rows_valid) {
                const long m = row0 + r, idx = m * n + j;
                const float dhv = dh[r] + (dhx ? dhx[r * ldx + j] : 0.f);
                const float tc = tanhf(cn[r]);
                const float dc = dcn[r] + dhv * go[r] * (1.f - tc * tc);
                float* dg = dgates + m * 4 * n;
                const float d_i = dc * gg[r] * gi[r] * (1.f - gi[r]);
                const float d_f = dc * cp[r] * gf[r] * (1.f - gf[r]);
                const float d_g = dc * gi[r] * (1.f - gg[r] * gg[r]);
                const float d_o = dhv * tc * go[r] * (1.f - go[r]);
                dg[j] = d_i; dg[n + j] = d_f; dg[2 * n + j] = d_g; dg[3 * n + j] = d_o;
                if (dgates_lo) {
                    float* dl = dgates_lo + m * 4 * n;
                    dl[j] = tf32_lo(d_i); dl[n + j] = tf32_lo(d_f); dl[2 * n + j] = tf32_lo(d_g); dl[3 * n + j] = tf32_lo(d_o);
                }
                dc_prev[idx] = dc * gf[r];
            }
        }
    }
}

// The same cell backward split in two, for n <= CT (one column j = threadIdx.x per thread): the loads
// are issued at kernel entry for BOTH cells, so their global-memory latency overlaps the encoder
// chain instead of being exposed twice (in-kernel trace of the serial version: 4000 cycles for the
// action cell at entry and 5700 for the belief cell at the end, of 31 000).
// (no arithmetic in the load phase: an add right after two loads would make the in-order thread wait
// for them before it can issue the next loads)
struct CellIn { float gi[RB], gf[RB], gg[RB], go[RB], dh[RB], dhc[RB], dcn[RB], cp[RB], cn[RB]; };
__device__ __forceinline__ void cell_bwd_load(CellIn& c, const int row0, const int rows_valid, const int n,
                                              const float* __restrict__ gates, const float* __restrict__ dh_heads,
                                              const float* __restrict__ dh_carry, const float* __restrict__ dc_next,
                                              const float* __restrict__ c_prev, const float* __restrict__ c_new) {
    const int j = threadIdx.x;
#pragma unroll
    for (int r = 0; r < RB; ++r) {
        c.gi[r] = c.gf[r] = c.gg[r] = c.go[r] = c.dh[r] = c.dhc[r] = c.dcn[r] = c.cp[r] = c.cn[r] = 0.f;
        if (j < n && r < rows_valid) {
            const long m = row0 + r, idx = m * n + j;
            const float* g = gates + m * 4 * n;
            c.gi[r] = g[j]; c.gf[r] = g[n + j]; c.gg[r] = g[2 * n + j]; c.go[r] = g[3 * n + j];
            c.dh[r] = dh_heads[idx];
            if (dh_carry) c.dhc[r] = dh_carry[idx];
            if (dc_next) c.dcn[r] = dc_next[idx];
            c.cp[r] = c_prev[idx]; c.cn[r] = c_new[idx];
        }
    }
}
__device__ __forceinline__ void cell_bwd_compute(const CellIn& c, const int row0, const int rows_valid, const int n,
                                                 const float* dhx, const int ldx, float* __restrict__ dgates,
                                                 float* __restrict__ dgates_lo, float* __restrict__ dc_prev) {
    const int j = threadIdx.x;
    if (j >= n) return;
#pragma unroll
    for (int r = 0; r < RB; ++r) {
        if (r < rows_valid) {
            const long m = row0 + r, idx = m * n + j;
            const float dhv = c.dh[r] + c.dhc[r] + (dhx ? dhx[r * ldx + j] : 0.f);
            const float tc = tanhf(c.cn[r]);
            const float dc = c.dcn[r] + dhv * c.go[r] * (1.f - tc * tc);
            float* dg = dgates + m * 4 * n;
            const float d_i = dc * c.gg[r] * c.gi[r] * (1.f - c.gi[r]);
            const float d_f = dc * c.cp[r] * c.gf[r] * (1.f - c.gf[r]);
            const float d_g = dc * c.gi[r] * (1.f - c.gg[r] * c.gg[r]);
            const float d_o = dhv * tc * c.go[r] * (1.f - c.go[r]);
            dg[j] = d_i; dg[n + j] = d_f; dg[2 * n + j] = d_g; dg[3 * n + j] = d_o;
            if (dgates_lo) {
                float* dl = dgates_lo + m * 4 * n;
                dl[j] = tf32_lo(d_i); dl[n + j] = tf32_lo(d_f); dl[2 * n + j] = tf32_lo(d_g); dl[3 * n + j] = tf32_lo(d_o);
            }
            dc_prev[idx] = dc * c.gf[r];
        }
    }
}

struct BwdPreKernelArgs { BwdPreArgs a; int maxw; int staged;  int trig; };

#ifdef MARLC_CHAIN_TRACE  // timeline of CTA 0 (cycles since entry), printed by thread 0
#define CHAIN_TRACE_DECL() __shared__ long long ch_tr[24]; const long long ch_t0 = clock64(); int ch_i = 0
#define CHAIN_TRACE() do { if (blockIdx.x == 0 && threadIdx.x == 0 && ch_i < 24) ch_tr[ch_i] = clock64() - ch_t0; ++ch_i; } while (0)
#define CHAIN_TRACE_PRINT(name) do { if (blockIdx.x == 0 && threadIdx.x == 0) { printf("%s trace:", name); \
    for (int i_ = 0; i_ < ch_i && i_ < 24; ++i_) printf(" %lld", ch_tr[i_]); printf(" | end %lld\n", clock64() - ch_t0); } } while (0)
#else
#define CHAIN_TRACE_DECL() do { } while (0)
#define CHAIN_TRACE() do { } while (0)
#define CHAIN_TRACE_PRINT(name) do { } while (0)
#endif

__global__ void __launch_bounds__(CT) bwd_pre_kernel(const BwdPreKernelArgs ka) {
    extern __shared__ __align__(16) float sm[];
    const BwdPreArgs& a = ka.a;
    const int row0 = blockIdx.x * RB, rows_valid = min(RB, a.M - row0), mw = ka.maxw;
    ChainSmem S(sm, mw);
    const int n_m = a.n_m, n1 = a.e0.n_out, nb = a.n[0];
    float* dhx = S.bufC;  // [RB][mw] encoder contribution to dh (belief cell only)
    float* W3s = S.wres;             // encode_msg.3 weight [n_m][n1]
    float* W0s = W3s + n_m * n1;     // encode_msg.0 weight [n1][nb]
    const bool enc = a.dcoll != nullptr || a.dmsg != nullptr;
    CHAIN_TRACE_DECL();
    if (ka.trig) pdl_trigger();  // sweep chain: the input-gradient GEMM's CTAs may set up while this kernel runs (common.cuh)
    pdl_wait();     // at entry: the operand loads must be queued AHEAD of the weight copies (see below)
    // ---- fast path: every global operand of the CTA is requested up front (cell inputs and encoder
    //      activations to registers, LayerNorm affines to shared memory), and only THEN the 164 KB of
    //      weights (cp.async): the load/store unit is in order, and with the weight copies queued
    //      first the ~95 operand loads per thread took 9200 cycles just to issue (in-kernel trace).
    const bool fast = ka.staged && a.n[0] <= CT && a.n[1] <= CT && RB * n_m <= CT && RB * n1 <= 2 * CT &&
                      2 * (n_m + n1) + RB * mw <= CT * WT_P;
    if (!fast && enc && ka.staged) {  // asynchronous: overlaps the action cell and the first encoder phases
        stage_w_async(W3s, a.e3.W, n_m, n1);
        stage_w_async(W0s, a.e0.W, n1, nb);
    }
    CHAIN_TRACE();  // 0
    if (fast) {
        float* sG3 = S.wt;            // encode_msg.4 affine
        float* sB3 = sG3 + n_m;
        float* sG0 = sB3 + n_m;       // encode_msg.1 affine
        float* sB0 = sG0 + n1;
        float* Y1S = sB0 + n1;        // [RB][mw] pre-norm activations of block 0
        CellIn ca, cb;
        cell_bwd_load(ca, row0, rows_valid, a.n[1], a.gates[1], a.dh_heads[1], a.dh_carry[1], a.dc_next[1], a.c_prev[1], a.c_new[1]);
        cell_bwd_load(cb, row0, rows_valid, a.n[0], a.gates[0], a.dh_heads[0], a.dh_carry[0], a.dc_next[0], a.c_prev[0], a.c_new[0]);
        float meanv = 0.f, y2v = 0.f, y1v[2] = {0.f, 0.f};
        const int tid = threadIdx.x;
        if (enc) {
            if (tid < RB * n_m) {
                const int r = tid / n_m, j = tid - r * n_m;
                if (r < rows_valid) {
                    meanv = a.dmsg ? a.dmsg[(long)(row0 + r) * n_m + j]
                                   : other_agents_mean(a.dcoll, row0 + r, j, a.Na, a.Nb, n_m);
                    y2v = a.enc_y2[(long)(row0 + r) * n_m + j];
                }
            }
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const int e = tid + i * CT;
                if (e < RB * n1) {
                    const int r = e / n1, k = e - r * n1;
                    if (r < rows_valid) y1v[i] = a.enc_y1[(long)(row0 + r) * n1 + k];
                }
            }
            if (tid < n_m) { sG3[tid] = a.e3.g[tid]; sB3[tid] = a.e3.be[tid]; }
            if (tid < n1) { sG0[tid] = a.e0.g[tid]; sB0[tid] = a.e0.be[tid]; }
            stage_w_async(W3s, a.e3.W, n_m, n1);
            stage_w_async(W0s, a.e0.W, n1, nb);
        }
        CHAIN_TRACE();  // loads issued
#ifdef MARLC_CHAIN_TRACE
        if (ca.gi[0] == 1234.5f) printf("x");
        CHAIN_TRACE();  // first cell operand arrived
        if (cb.cn[RB - 1] == 1234.5f) printf("x");
        CHAIN_TRACE();  // last cell operand arrived
        if (y1v[1] == 1234.5f || meanv == 1234.5f) printf("x");
        CHAIN_TRACE();  // encoder operands arrived
#endif
        cell_bwd_compute(ca, row0, rows_valid, a.n[1], nullptr, 0, a.dgates[1], a.dgates_lo[1], a.dc_prev[1]);
        CHAIN_TRACE();  // 1: loads issued + action cell
        if (enc) {
            if (tid < RB * n_m) {
                const int r = tid / n_m, j = tid - r * n_m;
                S.bufA[r * mw + j] = meanv;
                S.bufB[r * mw + j] = y2v;
            }
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const int e = tid + i * CT;
                if (e < RB * n1) { const int r = e / n1, k = e - r * n1; Y1S[r * mw + k] = y1v[i]; }
            }
            __syncthreads();
            CHAIN_TRACE();  // 2: operands in shared memory
            rb_ln_silu_bwd(S.bufA, S.bufB, mw, n_m, sG3, sB3, rows_valid, row0, dhx, S.bufT, a.d_enc_y2, n_m,
                           a.e3.dg, a.e3.dbe, a.e3.db);
            CHAIN_TRACE();  // 3: LN backward (block 3)
            stage_wait_all();
            __syncthreads();
            CHAIN_TRACE();  // 4: weights landed
            rb_dx_s(S.bufT, W3s, n1, S.bufA, mw, n_m, n1);  // ds1 [RB][2n_m]
            CHAIN_TRACE();  // 5: dx through W3
            rb_ln_silu_bwd(S.bufA, Y1S, mw, n1, sG0, sB0, rows_valid, row0, dhx, S.bufT, a.d_enc_y1, n1,
                           a.e0.dg, a.e0.dbe, a.e0.db);
            CHAIN_TRACE();  // 6: LN backward (block 0)
            rb_dx_s(S.bufT, W0s, nb, dhx, mw, n1, nb);      // dh contribution [RB][n_b]
            CHAIN_TRACE();  // 7: dx through W0
        }
        cell_bwd_compute(cb, row0, rows_valid, a.n[0], enc ? dhx : nullptr, mw, a.dgates[0], a.dgates_lo[0], a.dc_prev[0]);
        CHAIN_TRACE();  // 8: belief cell
        CHAIN_TRACE_PRINT("bwd_pre");
        return;
    }
    // the action cell does not depend on the encoder chain: do it while the weights stream in
    cell_bwd_rows(row0, rows_valid, a.n[1], a.gates[1], a.dh_heads[1], a.dh_carry[1], a.dc_next[1], a.c_prev[1],
                  a.c_new[1], nullptr, 0, a.dgates[1], a.dgates_lo[1], a.dc_prev[1]);
    CHAIN_TRACE();  // 1: action cell
    if (enc) {
        // gradient of the message produced at step t = adjoint mean of dcoll(t+1) (or dmsg); encoder block 3 backward
        for (int e = threadIdx.x; e < RB * n_m; e += CT) {
            const int r = e / n_m, j = e % n_m;
            const bool ok = r < rows_valid;
            S.bufA[r * mw + j] = !ok ? 0.f
                                 : a.dmsg ? a.dmsg[(long)(row0 + r) * n_m + j]
                                          : other_agents_mean(a.dcoll, row0 + r, j, a.Na, a.Nb, n_m);
            S.bufB[r * mw + j] = ok ? a.enc_y2[(long)(row0 + r) * n_m + j] : 0.f;
        }
        __syncthreads();
        CHAIN_TRACE();  // 2: adjoint mean + y2 loaded
        rb_ln_silu_bwd(S.bufA, S.bufB, mw, n_m, a.e3.g, a.e3.be, rows_valid, row0, dhx, S.bufT, a.d_enc_y2, n_m,
                       a.e3.dg, a.e3.dbe, a.e3.db);
        CHAIN_TRACE();  // 3: LN backward (block 3)
        if (ka.staged) { stage_wait_all(); __syncthreads(); }
        CHAIN_TRACE();  // 4: weights landed
        if (ka.staged) rb_dx_s(S.bufT, W3s, n1, S.bufA, mw, n_m, n1);  // ds1 [RB][2n_m]
        else rb_dx(S.bufT, a.e3.W, S.bufA, mw, n_m, n1);
        CHAIN_TRACE();  // 5: dx through W3
        for (int e = threadIdx.x; e < RB * n1; e += CT) {
            const int r = e / n1, k = e % n1;
            S.bufB[r * mw + k] = r < rows_valid ? a.enc_y1[(long)(row0 + r) * n1 + k] : 0.f;
        }
        __syncthreads();
        rb_ln_silu_bwd(S.bufA, S.bufB, mw, n1, a.e0.g, a.e0.be, rows_valid, row0, dhx, S.bufT, a.d_enc_y1, n1,
                       a.e0.dg, a.e0.dbe, a.e0.db);
        CHAIN_TRACE();  // 6: y1 load + LN backward (block 0)
        if (ka.staged) rb_dx_s(S.bufT, W0s, nb, dhx, mw, n1, nb);      // dh contribution [RB][n_b]
        else rb_dx(S.bufT, a.e0.W, dhx, mw, n1, nb);
        CHAIN_TRACE();  // 7: dx through W0
    }
    cell_bwd_rows(row0, rows_valid, a.n[0], a.gates[0], a.dh_heads[0], a.dh_carry[0], a.dc_next[0], a.c_prev[0],
                  a.c_new[0], enc ? dhx : nullptr, mw, a.dgates[0], a.dgates_lo[0], a.dc_prev[0]);
    CHAIN_TRACE();  // 8: belief cell
    CHAIN_TRACE_PRINT("bwd_pre");
}

int bwd_pre(const BwdPreArgs& a, cudaStream_t s) {
    if (a.M <= 0) return 0;
    BwdPreKernelArgs ka;
    ka.a = a;
    const ChainStage st = bwd_pre_stage(a.n_m, a.e0.n_out, a.n[0]);
    ka.maxw = st.maxw;
    const int wfl = st.wfl;
    ka.staged = wfl > 0;
    const size_t smem = chain_smem_bytes(ka.maxw) + sizeof(float) * (size_t)wfl;
    MARLC_CHECK(smem <= 200 * 1024, "bwd_pre: shared memory %zu B too large", smem);
    static size_t attr = 0;
    if (smem > 48 * 1024 && smem > attr) {
        MARLC_CUDA(cudaFuncSetAttribute(bwd_pre_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr = smem;
    }
    ka.trig = pdl_trigger_early();
    MARLC_CUDA(launch_pdl(bwd_pre_kernel, dim3((a.M + RB - 1) / RB), dim3(CT), smem, s, ka));
    MARLC_LAUNCH_CHECK();
    return 0;
}

// ---------------------------------------------------------------------------------
// backward "post" (step t): decoder backward from du_t -> dcoll
// ---------------------------------------------------------------------------------
struct BwdPostKernelArgs { BwdPostArgs a; int maxw; int staged; int trig; };

__global__ void __launch_bounds__(CT) bwd_post_kernel(const BwdPostKernelArgs ka) {
    extern __shared__ __align__(16) float sm[];
    const BwdPostArgs& a = ka.a;
    const int row0 = blockIdx.x * RB, rows_valid = min(RB, a.M - row0), mw = ka.maxw;
    ChainSmem S(sm, mw);
    const int n_m = a.n_m, n1 = a.d0.n_out, n2 = a.n_m_o;
    float* W3s = S.wres;           // decode_msg.3 weight [n2][n1]
    float* W0s = W3s + n2 * n1;    // decode_msg.0 weight [n1][n_m]
    if (ka.trig) pdl_trigger();  // sweep chain: the next step's bwd_pre may become resident while this kernel runs
    pdl_wait();     // at entry, as in bwd_pre
    // ---- fast path (as in bwd_pre): every global operand is requested up front, loads grouped ahead of
    //      any use, LayerNorm affines and the block-0 activations parked in the unused tile scratch
    const bool fast = ka.staged && RB * n2 <= 2 * CT && RB * n1 <= 2 * CT && n1 <= CT && n2 <= CT &&
                      2 * (n1 + n2) + RB * mw <= CT * WT_P;
    if (fast) {
        float* sG3 = S.wt;
        float* sB3 = sG3 + n2;
        float* sG0 = sB3 + n2;
        float* sB0 = sG0 + n1;
        float* Y1S = sB0 + n1;  // [RB][mw]
        const int tid = threadIdx.x;
        float du[2] = {0.f, 0.f}, y2v[2] = {0.f, 0.f}, y1v[2] = {0.f, 0.f};
        int r2[2], j2[2], r1[2], k1[2];
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const int e = tid + i * CT;
            r2[i] = e / n2; j2[i] = e - r2[i] * n2;
            r1[i] = e / n1; k1[i] = e - r1[i] * n1;
        }
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            if (r2[i] < rows_valid) {
                du[i] = a.dU[(long)(row0 + r2[i]) * a.ldu + a.F + j2[i]];
                y2v[i] = a.dec_y2[(long)(row0 + r2[i]) * n2 + j2[i]];
            }
            if (r1[i] < rows_valid) y1v[i] = a.dec_y1[(long)(row0 + r1[i]) * n1 + k1[i]];
        }
        float g3 = 0.f, b3 = 0.f, g0 = 0.f, b0 = 0.f;
        if (tid < n2) { g3 = a.d3.g[tid]; b3 = a.d3.be[tid]; }
        if (tid < n1) { g0 = a.d0.g[tid]; b0 = a.d0.be[tid]; }
        stage_w_async(W3s, a.d3.W, n2, n1);
        if (a.dcoll) stage_w_async(W0s, a.d0.W, n1, n_m);
        if (tid < n2) { sG3[tid] = g3; sB3[tid] = b3; }
        if (tid < n1) { sG0[tid] = g0; sB0[tid] = b0; }
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            if (r2[i] < RB) { S.bufA[r2[i] * mw + j2[i]] = du[i]; S.bufB[r2[i] * mw + j2[i]] = y2v[i]; }
            if (r1[i] < RB) Y1S[r1[i] * mw + k1[i]] = y1v[i];
        }
        __syncthreads();
        rb_ln_silu_bwd(S.bufA, S.bufB, mw, n2, sG3, sB3, rows_valid, row0, S.bufC, S.bufT, a.d_dec_y2, n2, a.d3.dg,
                       a.d3.dbe, a.d3.db);
        stage_wait_all();
        __syncthreads();
        rb_dx_s(S.bufT, W3s, n1, S.bufA, mw, n2, n1);
        rb_ln_silu_bwd(S.bufA, Y1S, mw, n1, sG0, sB0, rows_valid, row0, S.bufC, S.bufT, a.d_dec_y1, n1, a.d0.dg,
                       a.d0.dbe, a.d0.db);
        if (a.dcoll) {
            rb_dx_s(S.bufT, W0s, n_m, S.bufA, mw, n1, n_m);
            for (int e = tid; e < rows_valid * n_m; e += CT) {
                const int r = e / n_m, j = e % n_m;
                a.dcoll[(long)(row0 + r) * n_m + j] = S.bufA[r * mw + j];
            }
        }
        return;
    }
    if (ka.staged) { stage_w_async(W3s, a.d3.W, n2, n1); if (a.dcoll) stage_w_async(W0s, a.d0.W, n1, n_m); }
    for (int e = threadIdx.x; e < RB * n2; e += CT) {
        const int r = e / n2, j = e % n2;
        const bool ok = r < rows_valid;
        S.bufA[r * mw + j] = ok ? a.dU[(long)(row0 + r) * a.ldu + a.F + j] : 0.f;
        S.bufB[r * mw + j] = ok ? a.dec_y2[(long)(row0 + r) * n2 + j] : 0.f;
    }
    __syncthreads();
    rb_ln_silu_bwd(S.bufA, S.bufB, mw, n2, a.d3.g, a.d3.be, rows_valid, row0, S.bufC, S.bufT, a.d_dec_y2, n2, a.d3.dg,
                   a.d3.dbe, a.d3.db);
    if (ka.staged) { stage_wait_all(); __syncthreads(); }
    if (ka.staged) rb_dx_s(S.bufT, W3s, n1, S.bufA, mw, n2, n1);
    else rb_dx(S.bufT, a.d3.W, S.bufA, mw, n2, n1);
    for (int e = threadIdx.x; e < RB * n1; e += CT) {
        const int r = e / n1, k = e % n1;
        S.bufB[r * mw + k] = r < rows_valid ? a.dec_y1[(long)(row0 + r) * n1 + k] : 0.f;
    }
    __syncthreads();
    rb_ln_silu_bwd(S.bufA, S.bufB, mw, n1, a.d0.g, a.d0.be, rows_valid, row0, S.bufC, S.bufT, a.d_dec_y1, n1, a.d0.dg,
                   a.d0.dbe, a.d0.db);
    if (a.dcoll) {
        if (ka.staged) rb_dx_s(S.bufT, W0s, n_m, S.bufA, mw, n1, n_m);
        else rb_dx(S.bufT, a.d0.W, S.bufA, mw, n1, n_m);
        for (int e = threadIdx.x; e < rows_valid * n_m; e += CT) {
            const int r = e / n_m, j = e % n_m;
            a.dcoll[(long)(row0 + r) * n_m + j] = S.bufA[r * mw + j];
        }
    }
}

int bwd_post(const BwdPostArgs& a, cudaStream_t s) {
    if (a.M <= 0) return 0;
    BwdPostKernelArgs ka;
    ka.a = a;
    const ChainStage st = bwd_post_stage(a.n_m, a.d0.n_out, a.n_m_o);
    ka.maxw = st.maxw;
    const int wfl = st.wfl;
    ka.staged = wfl > 0;
    const size_t smem = chain_smem_bytes(ka.maxw) + sizeof(float) * (size_t)wfl;
    MARLC_CHECK(smem <= 200 * 1024, "bwd_post: shared memory %zu B too large", smem);
    static size_t attr = 0;
    if (smem > 48 * 1024 && smem > attr) {
        MARLC_CUDA(cudaFuncSetAttribute(bwd_post_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr = smem;
    }
    ka.trig = pdl_trigger_early();
    MARLC_CUDA(launch_pdl(bwd_post_kernel, dim3((a.M + RB - 1) / RB), dim3(CT), smem, s, ka));
    MARLC_LAUNCH_CHECK();
    return 0;
}

}  // namespace marlc

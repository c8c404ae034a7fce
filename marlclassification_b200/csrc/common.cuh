// Shared device helpers and internal launcher declarations for libmarlc.
// sm_100a only (B200).  No torch types anywhere in this library.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#define MARLC_SMS 148

namespace marlc {
// low-order part of a float for the error-compensated 3xTF32 product: x - trunc_tf32(x) (exact in fp32)
__device__ __forceinline__ float tf32_lo(float x) { return x - __uint_as_float(__float_as_uint(x) & 0xFFFFE000u); }


// ---- error plumbing (C-ABI returns int, message via marlc_last_error) -----
void set_error(const char* fmt, ...);
#define MARLC_FAIL(...)            \
    do {                           \
        marlc::set_error(__VA_ARGS__); \
        return 1;                  \
    } while (0)
#define MARLC_CHECK(cond, ...)     \
    do {                           \
        if (!(cond)) MARLC_FAIL(__VA_ARGS__); \
    } while (0)
#define MARLC_CUDA(expr)                                                         \
    do {                                                                         \
        cudaError_t e__ = (expr);                                                \
        if (e__ != cudaSuccess)                                                  \
            MARLC_FAIL("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
    } while (0)
extern int g_launch_count;  // kernels launched through this library (bench accounting)
extern long g_simt_gemm_launches, g_tc_gemm_launches;  // per GEMM back end (marlc_gemm_launch_count)
#define MARLC_LAUNCH_CHECK()             \
    do {                                 \
        ++marlc::g_launch_count;         \
        MARLC_CUDA(cudaGetLastError());  \
    } while (0)
#define MARLC_TRY(expr)        \
    do {                       \
        int r__ = (expr);      \
        if (r__) return r__;   \
    } while (0)

// ---- programmatic dependent launch (PDL) ---------------------------------------
// The per-step kernels of the rollout and of the BPTT sweep form one dependent chain per stream
// (episode.py:70-78: step t+1 needs step t), ~1.9 us of launch / drain latency per edge.  A kernel launched
// with the programmatic-stream-serialization attribute may become resident while its predecessor is still
// running: its CTAs run their prologue (barrier init, TMEM allocation, descriptor prefetch, constant staging)
// and block in pdl_wait() until the predecessor has completed and its writes are visible.  Contract for every
// kernel launched through launch_pdl(): NOTHING but launch-constant memory (parameters, tensor maps, weights
// of the current iteration) is read, and no global memory is written, before pdl_wait(); pdl_trigger() at
// entry lets the NEXT kernel of the chain do the same.  g_pdl is set by the engine (PdlScope) only around
// launches whose predecessor in the stream is a kernel of the same chain; everywhere else the launch is an
// ordinary one and pdl_wait() returns immediately.  MARLC_PDL=0 switches the attribute off (to bisect a suspected ordering race).
extern thread_local int g_pdl, g_pdl_trig;
struct PdlScope {  // on: the launches inside are programmatic dependents; trig: they trigger THEIR dependents at entry
    int prev, prev_trig;
    explicit PdlScope(int on, int trig = 0) : prev(g_pdl), prev_trig(g_pdl_trig) { g_pdl = on; g_pdl_trig = trig; }
    ~PdlScope() { g_pdl = prev; g_pdl_trig = prev_trig; }
};
bool pdl_enabled();
// Which edges, and where the trigger sits, is measured, not derived (profiles/README.md, round 2: 512 rows per step):
//   * forward: step_pre, block-0 GEMMs and step_post as dependents with the trigger at kernel entry: -52 us per
//     16 steps; the LSTM pair as a dependent: +15 us (left an ordinary launch);
//   * BPTT sweep: an entry trigger makes every edge slower (+44 us for bwd_pre alone: the next kernel's CTAs pile
//     onto the SMs the running kernel leaves free and start unevenly); without an explicit trigger (dependents
//     launch when the last CTA exits, skipping only the drain) the three edges gain 26 us.
// So every PdlScope of the engine makes its launches dependents except the LSTM pair's, and only the forward chain's
// scopes set the entry trigger.
int pdl_trigger_early(); // value for the kernels' `trig` argument (from the enclosing PdlScope)
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
// Launch `kern(arg)`; with g_pdl set (and PDL enabled) as a programmatic dependent of the previous kernel in `s`.
// cluster_x > 1 adds a cluster dimension along x.
template <typename KP, typename A>
inline cudaError_t launch_pdl(void (*kern)(KP), dim3 grid, dim3 block, size_t smem, cudaStream_t s, const A& arg,
                              int cluster_x = 1) {
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cudaLaunchAttribute at[2];
    int n = 0;
    if (cluster_x > 1) {
        at[n].id = cudaLaunchAttributeClusterDimension;
        at[n].val.clusterDim.x = (unsigned)cluster_x; at[n].val.clusterDim.y = 1; at[n].val.clusterDim.z = 1;
        ++n;
    }
    if (g_pdl && pdl_enabled()) {
        at[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at[n].val.programmaticStreamSerializationAllowed = 1;
        ++n;
    }
    cfg.attrs = n ? at : nullptr; cfg.numAttrs = (unsigned)n;
    return cudaLaunchKernelEx(&cfg, kern, arg);
}

// ---- math ------------------------------------------------------------------
__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + expf(-x)); }
__device__ __forceinline__ float siluf_(float x) { return x * sigmoidf_(x); }
// d/dz [z * sigmoid(z)]
__device__ __forceinline__ float silu_grad_(float z) {
    float s = sigmoidf_(z);
    return s * (1.0f + z * (1.0f - s));
}

// Division by a launch-constant d as one multiply-high: q = (n * ceil(2^32 / d)) >> 32, exact for
// 0 <= n and n * d < 2^32 (callers check their largest n on the host).  Runtime `/` costs ~20
// instructions; index decompositions (e -> channel, row, column) are often most of an
// element-wise kernel's issue slots.
struct FastDiv {
    unsigned d, m;
    FastDiv() : d(1), m(0) {}
    __host__ explicit FastDiv(unsigned d_) : d(d_), m(d_ > 1 ? (unsigned)((0x100000000ull + d_ - 1) / d_) : 0u) {}
    __host__ __device__ __forceinline__ static unsigned mulhi(unsigned a, unsigned b) {
#ifdef __CUDA_ARCH__
        return __umulhi(a, b);
#else
        return (unsigned)(((unsigned long long)a * b) >> 32);  // host twin, used by marlc_selftest_fastdiv
#endif
    }
    __host__ __device__ __forceinline__ int div(int n) const { return d > 1 ? (int)mulhi((unsigned)n, m) : n; }
    __host__ __device__ __forceinline__ int div_nz(int n) const { return (int)mulhi((unsigned)n, m); }  // d >= 2 only
    // largest dividend bound the launchers check: exact for every 0 <= n with n * d < 2^32
    __host__ static bool exact_up_to(long long n_max, long long d_) { return n_max * d_ < 0x100000000ll; }
};

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ---- Philox4x32-10 (counter-based RNG; own implementation) ------------------
struct Philox {
    uint32_t k0, k1;
    __device__ Philox(uint64_t seed) : k0((uint32_t)seed), k1((uint32_t)(seed >> 32)) {}
    __device__ uint4 operator()(uint64_t ctr, uint64_t stream) const {
        uint32_t c0 = (uint32_t)ctr, c1 = (uint32_t)(ctr >> 32), c2 = (uint32_t)stream, c3 = (uint32_t)(stream >> 32);
        uint32_t a = k0, b = k1;
#pragma unroll
        for (int r = 0; r < 10; ++r) {
            uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
            uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
            uint32_t n0 = hi1 ^ c1 ^ a, n1 = lo1, n2 = hi0 ^ c3 ^ b, n3 = lo0;
            c0 = n0; c1 = n1; c2 = n2; c3 = n3;
            a += 0x9E3779B9u; b += 0xBB67AE85u;
        }
        return make_uint4(c0, c1, c2, c3);
    }
};
// uniform in [0,1) with 24 bits
__device__ __forceinline__ float u01(uint32_t x) { return (float)(x >> 8) * (1.0f / 16777216.0f); }


// ---- cooperative global -> shared copy of a dense row-major matrix into padded rows -----------
// src: nrows x rowlen contiguous floats; dst row pitch `pitch`.  Loads are issued in batches of
// 8 independent 128-bit requests per thread before any store, so the copy costs a few L2 round
// trips instead of one per element (the loop is latency-bound otherwise).
__device__ __forceinline__ void stage_rows(float* dst, const float* __restrict__ src, int nrows, int rowlen, int pitch) {
    const int tid = threadIdx.x, nt = blockDim.x;
    const int total = nrows * rowlen;
    if (((rowlen & 3) == 0) && ((reinterpret_cast<uintptr_t>(src) & 15) == 0)) {
        constexpr int U = 8;
        for (int base = tid * 4; base < total; base += nt * 4 * U) {
            float4 v[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int i = base + u * nt * 4;
                if (i < total) v[u] = __ldg(reinterpret_cast<const float4*>(src + i));
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int i = base + u * nt * 4;
                if (i < total) {
                    const int n = i / rowlen, k = i - n * rowlen;
                    float* d = dst + n * pitch + k;
                    d[0] = v[u].x; d[1] = v[u].y; d[2] = v[u].z; d[3] = v[u].w;
                }
            }
        }
    } else {
        constexpr int U = 8;
        for (int base = tid; base < total; base += nt * U) {
            float v[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int i = base + u * nt;
                if (i < total) v[u] = __ldg(src + i);
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int i = base + u * nt;
                if (i < total) {
                    const int n = i / rowlen, k = i - n * rowlen;
                    dst[n * pitch + k] = v[u];
                }
            }
        }
    }
}

// ---- generic fp32 GEMM (SIMT), gemm_simt.cu ----------------------------------
// C[m,n] (+)= sum_k A(m,k) B(k,n) [+ sum_k2 A2(m,k2) B2(k2,n)] + bias[n] + bias2[n]
// A(m,k) = A[m*sam + k*sak]; B(k,n) = B[k*sbk + n*sbn]; C[m*ldc + n].
struct GemmProblem {
    const float* A; long sam, sak;
    const float* B; long sbk, sbn;
    const float* A2; long sam2, sak2;
    const float* B2; long sbk2, sbn2;
    const float* bias; const float* bias2;
    float* C; long ldc;
    int M, N, K, K2;
    int accumulate;  // 1: C += result
};
struct GemmGroup {
    GemmProblem p[4];
    int count;
};
int gemm_group(const GemmGroup& g, cudaStream_t s);
// Y[M,N] = X[M,K] W[N,K]^T (+ bias)       (nn.Linear forward)
int gemm_nt(const float* X, long ldx, const float* W, long ldw, const float* bias, float* Y, long ldy, int M, int N,
            int K, int accumulate, cudaStream_t s);
// dX[M,K] (+)= dY[M,N] W[N,K]              (input gradient)
int gemm_nn(const float* dY, long lddy, const float* W, long ldw, float* dX, long lddx, int M, int N, int K,
            int accumulate, cudaStream_t s);
// dW[N,K] (+)= dY[R,N]^T X[R,K]            (weight gradient, reduction over rows)
// ---- skinny.cu: products with a handful of outputs per row (HBM-bound reductions)
int rowdot(const float* X, long ldx, const float* w, const float* bias, float* Y, long ldy, int R, int K, int accumulate,
           cudaStream_t s);
int tn_skinny(const float* dY, long lddy, const float* X, long ldx, float* dW, long lddw, int R, int N, int K,
              int accumulate, cudaStream_t s, bool* done);
int gemm_tn(const float* dY, long lddy, const float* X, long ldx, float* dW, long lddw, int R, int N, int K,
            int accumulate, cudaStream_t s);

// ---- row-wise kernels, rowwise.cu --------------------------------------------
int ln_silu_fwd(const float* Y, long ldy, const float* gamma, const float* beta, float* S, long lds, int R, int N,
                cudaStream_t s);
// dY = d(LN->SiLU)/dY * dS ; accumulates dgamma/dbeta/dbias (column sums) atomically
int ln_silu_bwd_fused(const float* dS, long ldds, const float* dOut, int No, const float* W3, const float* Y, long ldy,
                      const float* gamma, const float* beta, float* dY, long lddy, float* dgamma, float* dbeta,
                      float* dbias, int R, int N, cudaStream_t s);
int ln_silu_bwd(const float* dS, long ldds, const float* Y, long ldy, const float* gamma, const float* beta, float* dY,
                long lddy, float* dgamma, float* dbeta, float* dbias, int R, int N, cudaStream_t s);
int colsum_add(const float* X, long ldx, float* out, int R, int N, cudaStream_t s);
int colsum_add2(const float* X, long ldx, float* out, float* out2, int R, int N, cudaStream_t s);
int msg_mean(const float* msg, float* coll, int Na, int Nb, int n, cudaStream_t s);  // also its own adjoint
int pos_features_fwd(const float* npos, const float* W, const float* b, const float* gamma, const float* beta,
                     float* y_pre, float* out, long ldo, int R, int nd, cudaStream_t s);
int lstm_cell_fwd(float* gates /*[M,4n] pre -> post activations*/, const float* c_prev, float* c_new, float* h_new,
                  int M, int n, cudaStream_t s);
int lstm_cell_bwd(const float* dh, const float* dh2 /*nullable, added*/, const float* dc_next, const float* gates,
                  const float* c_prev, const float* c_new, float* dgates, float* dc_prev, int M, int n, cudaStream_t s);
int add_inplace(float* dst, const float* src, long n, cudaStream_t s);

}  // namespace marlc

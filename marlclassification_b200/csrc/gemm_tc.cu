// Tensor-core GEMMs for sm_100a: TMA (cp.async.bulk.tensor) -> 128B-swizzled
// shared memory -> tcgen05.mma kind::tf32 (fp32 operands read directly, fp32
// accumulators in TMEM) -> tcgen05.ld epilogue.  Hand-written PTX; no CUTLASS.
//
//   D[M,N] (+)= sum_k A(m,k) B(n,k)  [+ second operand pair]  (+ bias)
//
// Operand majors (both supported for A and B, so no transposed copies exist):
//   K-major : memory [rows = M or N][K contiguous]      (nn.Linear forward: X, W)
//   MN-major: memory [K rows][M or N contiguous]        (dX = dY.W: B = W;  dW = dY^T.X: both)
//
// CTA = 192 threads: warp 0 = TMA producer, warp 1 = MMA issuer (+ TMEM alloc),
// warps 2..5 = epilogue (one TMEM lane quarter each).  Tile 128 x BN x 32, STAGES-deep
// mbarrier ring.  Epilogues: plain store / accumulate / split-K atomic add, and the
// fused LSTM cell (gates i,f,g,o of one hidden unit live in the same CTA tile).
#include <cuda.h>
#include <stdlib.h>

#include "common.cuh"
#include "tc.cuh"

namespace marlc {

constexpr int BM = 128;
constexpr int BK = 32;  // floats = 128 bytes = one swizzle row
constexpr int UMMA_K = 8;
constexpr int TC_THREADS = 192;
constexpr int TC_THREADS_X3 = 320;  // + 4 warps that only split operands (the splitter is throughput-bound)
constexpr int TC_SPLITTERS = TC_THREADS_X3 - 64;
#define TC_SPLIT_GROUPS(stages) (((stages) % 2 == 0) ? 2 : 1)  // operand-splitter groups (see tc_gemm_body)
constexpr int TC_MAX_CHAIN = 4096;  // longest K range one CTA accumulates in TMEM when split-K is allowed

// ---------------------------------------------------------------------------------
// host: tensor maps
// ---------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn get_encode() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)p;
    }
    return fn;
}

// 3-D map over [slabs][rows][inner] fp32, box = [1][box_rows][32], 128B swizzle, zero OOB fill
// mn_major operands use the 32B-atom variant of the 128B swizzle: the only shared-memory
// layout tcgen05 accepts for MN-major TF32 (UMMA layout type SWIZZLE_128B_BASE32B)
static int make_map(CUtensorMap* m, const float* ptr, long inner, long rows, long slabs, long ld, long slab_stride,
                    int box_rows, bool mn_major = false, int box_slabs = 1) {
    EncodeTiledFn enc = get_encode();
    MARLC_CHECK(enc, "cuTensorMapEncodeTiled not available");
    cuuint64_t dims[3] = {(cuuint64_t)inner, (cuuint64_t)rows, (cuuint64_t)slabs};
    cuuint64_t strides[2] = {(cuuint64_t)ld * 4, (cuuint64_t)(slabs > 1 ? slab_stride : rows * ld) * 4};
    cuuint32_t box[3] = {32, (cuuint32_t)box_rows, (cuuint32_t)box_slabs};
    cuuint32_t es[3] = {1, 1, 1};
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, (void*)ptr, dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE,
                     mn_major ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B,
                     CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    MARLC_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed (%d): ptr=%p inner=%ld rows=%ld ld=%ld box_rows=%d",
                (int)r, (const void*)ptr, inner, rows, ld, box_rows);
    return 0;
}

// 2-D map over C[M][N] (row stride ldc) for the epilogue's TMA store / reduce-add: box 32 cols x 32 rows
// (one TMEM lane quarter x one 128-byte swizzle row); out-of-range rows / columns are clipped by TMA
static int make_map_c(CUtensorMap* m, float* C, long M, long N, long ldc) {
    EncodeTiledFn enc = get_encode();
    MARLC_CHECK(enc, "cuTensorMapEncodeTiled not available");
    cuuint64_t dims[2] = {(cuuint64_t)N, (cuuint64_t)M};
    cuuint64_t strides[1] = {(cuuint64_t)ldc * 4};
    cuuint32_t box[2] = {32, 32};
    cuuint32_t es[2] = {1, 1};
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)C, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    MARLC_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled (C) failed (%d): ptr=%p M=%ld N=%ld ldc=%ld", (int)r, (void*)C, M, N, ldc);
    return 0;
}

bool tc_operand_ok(const TcOperand& o) {
    return o.ptr && (((uintptr_t)o.ptr & 15) == 0) && (o.ld % 4 == 0) && (o.slab_stride % 4 == 0);
}

// ---------------------------------------------------------------------------------
// device: PTX wrappers
// ---------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    const uint32_t addr = smem_u32(bar);
    uint32_t done;
    do {
        asm volatile(
            "{\n\t"
            ".reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t"
            "}"
            : "=r"(done)
            : "r"(addr), "r"(parity)
            : "memory");
    } while (!done);
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(smem_u32(dst)), "l"((uint64_t)map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
        : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

#define TMEM_LD8(addr, r)                                                                             \
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"            \
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), \
                   "=r"(r[7])                                                                         \
                 : "r"(addr))
#define TMEM_LD32(addr, r)                                                                                  \
    asm volatile(                                                                                          \
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "                                                          \
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"                                          \
        "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"                         \
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),  \
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]),         \
          "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]),       \
          "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]),       \
          "=r"(r[29]), "=r"(r[30]), "=r"(r[31])                                                            \
        : "r"(addr))
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// MUFU-based activations for the tensor-core epilogue (abs error ~1e-7, far below TF32's).  The cell epilogue is bound
// by instruction throughput (in-kernel trace, round 2: ~1 750 cycles of a scheduler per 8 hidden units x 32 rows), so
// the two special-function operations are issued directly (ex2 / rcp, flush-to-zero forms: __expf and __fdividef each
// wrap theirs in range fix-ups) and the scale of the exponent is folded into the bias add:
//   sigmoid(a + b) = rcp(1 + ex2(a * -log2(e) + b * -log2(e))),   tanh(x) = 2 * sigmoid(2x) - 1.
constexpr float NEG_LOG2E = -1.4426950408889634f;
__device__ __forceinline__ float ex2_ftz(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float rcp_ftz(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
// t = x * -log2(e) for sigmoid(x), x * -2 log2(e) for tanh(x)
__device__ __forceinline__ float sigmoid_of_scaled(float t) { return rcp_ftz(1.0f + ex2_ftz(t)); }
__device__ __forceinline__ float tanh_of_scaled(float t) { return fmaf(2.0f, rcp_ftz(1.0f + ex2_ftz(t)), -1.0f); }
__device__ __forceinline__ float fast_tanh(float x) { return tanh_of_scaled(2.0f * NEG_LOG2E * x); }

// smem matrix descriptor (cute::UMMA::SmemDescriptor bit layout).
// layout_type: 2 = SWIZZLE_128B (K-major tiles), 1 = SWIZZLE_128B_BASE32B (MN-major TF32 tiles)
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout_type) {
    return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) |
           ((uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32) | (1ull << 46) | ((uint64_t)layout_type << 61);
}

// ---------------------------------------------------------------------------------
// kernel
// ---------------------------------------------------------------------------------
enum { EPI_STORE = 0, EPI_LSTM = 1 };

struct TcKernelParams {
    CUtensorMap a1, b1, a2, b2;  // second pair unused when nk2 == 0
    // 3xTF32 with PRE-SPLIT operands: low-order parts kept in global memory by the producer of the
    // tensor (weights: refreshed once per forward; activations: written next to the value) and
    // fetched by TMA into the lo ring, so no CTA has to split them (at small M every CTA of a
    // launch would otherwise re-split the same A tiles)
    CUtensorMap a1l, b1l, a2l, b2l;
    CUtensorMap cmap;            // EPI_STORE: C as [M rows][N cols], box 32 x 32, 128B swizzle (TMA store / reduce)
    int c_tma;                   // 1: cmap is valid (C 16-byte aligned, ldc % 4 == 0)
    int ksplit;                  // EPI_LSTM: 2 = a pair of CTAs (cluster of 2 along x) splits K; the odd CTA ships its
                                 // partial accumulators into the even CTA's shared memory (DSMEM) before the cell
    int a_lo_g, b_lo_g;          // 1: the lo part of A / B comes from global memory
    int nk1, nk2;                // K blocks of each pair
    int slab_a1, slab_b1, slab_a2, slab_b2;
    int M, N;
    // EPI_STORE
    float* C;
    long ldc;
    const float* bias;
    const float* bias2;
    int accumulate, splits;
    // EPI_LSTM (N = 4*n; tile = HU hidden units x 4 gates)
    const float* c_prev;
    float* c_new;
    float* h_new;
    float* h_new_lo;  // optional: lo part of h_new for the next consumer's pre-split A operand
    float* gates;
    int n_hidden;
};
constexpr int TC_MAX_GROUP = 3;
struct TcKernelGroup {  // up to 3 independent problems in one launch; blockIdx.z -> (problem, K split)
    TcKernelParams p[TC_MAX_GROUP];
    int zofs[TC_MAX_GROUP + 1];
    int count;
    int trig;  // 1: griddepcontrol.launch_dependents at entry (common.cuh)
};

// KS = number of 32-float K sub-blocks per pipeline stage.  The single-thread producer / MMA loops
// pay ~0.15-0.2 us of barrier round trip per stage whatever the ring depth (measured: depth 2..10
// makes no difference), so latency-bound launches use fat stages (KS = 2 or 4) and a 2-deep ring.
template <int BN, int STAGES, bool X3 = false, int KS = 1>
struct TcSmem {
    static constexpr int A_SUB = BM * BK * 4;
    static constexpr int B_SUB = BN * BK * 4;
    static constexpr int A_BYTES = KS * A_SUB;
    static constexpr int B_BYTES = KS * B_SUB;
    // X3 (error-compensated 3xTF32): every stage also holds the low-order tiles A_lo, B_lo
    static constexpr int BYTES = STAGES * (A_BYTES + B_BYTES) * (X3 ? 2 : 1) + 1024;
};


// The body is instantiated once per problem slot so that every access to the kernel parameters
// (in particular the TMA descriptors) uses a compile-time offset: indexing the parameter block
// with a runtime problem index costs ~2 us per launch on B200 (measured).
//
// X3 = error-compensated "3xTF32": tcgen05 kind::tf32 truncates each fp32 operand to 10 mantissa
// bits.  The 4 epilogue warps, idle during the main loop, split every landed stage into
// hi = trunc(x) (what the tensor core sees of the original tile) and lo = x - hi (written to a
// mirror tile with the same swizzled layout), and the MMA warp issues A.B + A_lo.B + A.B_lo:
// products keep ~21 mantissa bits, i.e. fp32-class accuracy at 1/3 of the TF32 MMA rate.
template <int BN, bool A_MN, bool B_MN, int EPI, int STAGES, int PI, bool X3, int KS>
__device__ __forceinline__ void tc_gemm_body(const TcKernelGroup& pp, const int split) {
    using S = TcSmem<BN, STAGES, X3, KS>;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    constexpr int stages = STAGES;  // (a runtime ring depth of 2..8 made no measurable difference)
    uint8_t* sA = smem;
    uint8_t* sB = smem + stages * S::A_BYTES;
    constexpr int LO_OFF = stages * (S::A_BYTES + S::B_BYTES);  // lo tiles mirror the hi ring at this offset
    __shared__ __align__(8) uint64_t full_bar[STAGES];
    __shared__ __align__(8) uint64_t empty_bar[STAGES];
    __shared__ __align__(8) uint64_t split_bar[STAGES];
    __shared__ __align__(8) uint64_t tmem_full_bar;
    __shared__ uint32_t tmem_base_smem;
    __shared__ float s_bias[8][BN];  // per epilogue warp (2..9): bias (+ bias2) of this tile's columns

    const TcKernelParams& p = pp.p[PI];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#ifdef MARLC_TC_TRACE  // in-kernel timeline of CTA (0,0,0): cycles since entry at each pipeline event
    __shared__ long long trace[12];
    const bool tr = blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0;
    const long long t_entry = clock64();
#define TC_TRACE(i) do { if (tr) trace[i] = clock64() - t_entry; } while (0)
#else
#define TC_TRACE(i) do { } while (0)
#endif
    const int m0 = blockIdx.y * BM;
    const int ksp = (EPI == EPI_LSTM && p.ksplit > 1) ? p.ksplit : 1;
    const int n_tile = ksp > 1 ? blockIdx.x / ksp : blockIdx.x;
    const int kslice = ksp > 1 ? blockIdx.x % ksp : 0;  // = rank in the cluster of ksp CTAs
    if (m0 >= p.M || n_tile * BN >= p.N) return;  // grid is sized for the largest problem of the group
    // K-block range of this CTA (split-K over the concatenated list of both pairs)
    const int nkb = p.nk1 + p.nk2;
    int kb_begin = 0, kb_end = nkb;
    if (EPI == EPI_STORE && p.splits > 1) {
        const int per = (nkb + p.splits - 1) / p.splits;
        kb_begin = split * per;
        kb_end = min(nkb, kb_begin + per);
    }
    if (ksp > 1) {
        const int per = (nkb + ksp - 1) / ksp;
        kb_begin = kslice * per;
        kb_end = min(nkb, kb_begin + per);
    }
    const int my_kb = max(0, kb_end - kb_begin);
    constexpr int TMEM_COLS = BN < 32 ? 32 : BN;

    if (warp == 0 && lane == 0) {  // descriptor fetch overlaps barrier init / TMEM allocation
        auto pf = [](const CUtensorMap* m) { asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)m) : "memory"); };
        pf(&p.a1); pf(&p.b1);
        if (p.nk2 > 0) { pf(&p.a2); pf(&p.b2); }
        if (X3 && p.a_lo_g) { pf(&p.a1l); if (p.nk2 > 0) pf(&p.a2l); }
        if (X3 && p.b_lo_g) { pf(&p.b1l); if (p.nk2 > 0) pf(&p.b2l); }
        if (EPI == EPI_STORE && p.c_tma) pf(&p.cmap);
    }
    if (threadIdx.x == 32) {
        for (int s = 0; s < stages; ++s) {
            mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1);
            mbar_init(&split_bar[s], TC_SPLITTERS / TC_SPLIT_GROUPS(STAGES));  // one splitter group per slot
        }
        mbar_init(&tmem_full_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_smem)),
                     "r"(TMEM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_smem;
    // Everything above touched only the kernel parameters and this CTA's shared memory / TMEM.  From here on the
    // operands, c_prev and C are read / written: wait for the predecessor kernel (no-op for ordinary launches).
    pdl_wait();
    if (threadIdx.x == 0) TC_TRACE(0);  // setup done (barriers, TMEM)
    // K split over a CTA pair: the odd CTA will write into the even CTA's shared memory (DSMEM).  A CTA of a
    // cluster may only be written once it has STARTED executing: every thread arrives on the cluster barrier now
    // (non-blocking) and waits for this phase right before the first remote store / before the final barrier
    // (compute-sanitizer racecheck: "block that might not have entered yet", round 2).
    if (ksp > 1) asm volatile("barrier.cluster.arrive.release;" ::: "memory");

    if (warp == 0) {
        // ============================ TMA producer ============================
        if (lane == 0) {
            // loop-invariant parameters in registers (a single thread issues every copy of the CTA: constant-
            // bank reads and their dependent branches inside this loop delayed the first stage by ~500 cycles)
            int q_nk1 = p.nk1, q_alo = X3 ? p.a_lo_g : 0, q_blo = X3 ? p.b_lo_g : 0;
            int q_za1 = p.slab_a1, q_za2 = p.slab_a2, q_zb1 = p.slab_b1, q_zb2 = p.slab_b2, q_nh = p.n_hidden;
            asm volatile("" : "+r"(q_nk1), "+r"(q_alo), "+r"(q_blo), "+r"(q_za1), "+r"(q_za2), "+r"(q_zb1), "+r"(q_zb2), "+r"(q_nh));
            const uint32_t tx_bytes = S::A_BYTES + S::B_BYTES + (q_alo ? S::A_BYTES : 0) + (q_blo ? S::B_BYTES : 0);
            (void)q_nh;
            for (int i = 0; i < my_kb; ++i) {
                const int s = i % stages, ph = (i / stages) & 1;
                mbar_wait(&empty_bar[s], ph ^ 1);
                mbar_expect_tx(&full_bar[s], tx_bytes);
                const int kb = kb_begin + i;
                const bool second = kb >= q_nk1;
                const int za = second ? q_za2 : q_za1, zb = second ? q_zb2 : q_zb1;
                const int nlo = X3 ? 2 : 1;
                for (int hl = 0; hl < nlo; ++hl) {  // hl == 1: the pre-split lo tiles (when provided)
                if (hl == 1 && !q_alo && !q_blo) break;
                const CUtensorMap* ma = hl ? (second ? &p.a2l : &p.a1l) : (second ? &p.a2 : &p.a1);
                const CUtensorMap* mb = hl ? (second ? &p.b2l : &p.b1l) : (second ? &p.b2 : &p.b1);
                const bool do_a = hl == 0 || q_alo, do_b = hl == 0 || q_blo;
#pragma unroll
                for (int sub = 0; sub < KS; ++sub) {  // sub-blocks past the end of K are zero-filled by TMA
                    const int k0 = ((second ? kb - q_nk1 : kb) * KS + sub) * BK;
                    uint8_t* a_dst = sA + s * S::A_BYTES + sub * S::A_SUB + hl * LO_OFF;
                    uint8_t* b_dst = sB + s * S::B_BYTES + sub * S::B_SUB + hl * LO_OFF;
                    if (do_a) {
                        if (!A_MN) tma_load_3d(a_dst, ma, &full_bar[s], k0, m0, za);
                        else
                            for (int j = 0; j < BM / 32; ++j) tma_load_3d(a_dst + j * 4096, ma, &full_bar[s], m0 + 32 * j, k0, za);
                    }
                    if (!do_b) continue;
                    if (EPI == EPI_LSTM) {
                        // gather the 4 gate row-blocks of HU hidden units: rows g*n + j0 .. +HU
                        // one box {32 floats of K, HU units, 4 gates} of the [gate][unit][K] weight view
                        constexpr int HU = BN / 4;
                        tma_load_3d(b_dst, mb, &full_bar[s], k0, n_tile * HU, 0);
                    } else if (!B_MN) {
                        tma_load_3d(b_dst, mb, &full_bar[s], k0, n_tile * BN, zb);
                    } else {
                        for (int j = 0; j < BN / 32; ++j)
                            tma_load_3d(b_dst + j * 4096, mb, &full_bar[s], n_tile * BN + 32 * j, k0, zb);
                    }
                }
                }
                if (i == 0) TC_TRACE(1);  // first stage's TMA issued
            }
        }
    } else if (warp == 1) {
        // ============================ MMA issuer ============================
        if (lane == 0) {
            const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((A_MN ? 1u : 0u) << 15) |
                                   ((B_MN ? 1u : 0u) << 16) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
            int wait_split = (X3 && !(p.a_lo_g && p.b_lo_g)) ? 1 : 0;
            asm volatile("" : "+r"(wait_split));
            for (int i = 0; i < my_kb; ++i) {
                const int s = i % stages, ph = (i / stages) & 1;
                mbar_wait(wait_split ? &split_bar[s] : &full_bar[s], ph);
                tc_fence_after();
                if (i == 0) TC_TRACE(2);  // first stage landed (and split)
#pragma unroll
                for (int sub = 0; sub < KS; ++sub) {
                const uint32_t a_addr = smem_u32(sA + s * S::A_BYTES + sub * S::A_SUB);
                const uint32_t b_addr = smem_u32(sB + s * S::B_BYTES + sub * S::B_SUB);
#pragma unroll
                for (int k = 0; k < BK / UMMA_K; ++k) {
                    // K-major : advance 32 B inside the swizzled 128 B row; SBO = 1024 (8 rows x 128 B)
                    // MN-major: 8 k-rows (1024 B) per MMA = two 4-row swizzle atoms, SBO = 512 between
                    //           them; LBO = 4096 between the 32-float MN groups (one TMA box each)
                    const uint64_t ad = A_MN ? make_desc(a_addr + k * 1024, 4096, 512, 1) : make_desc(a_addr + k * 32, 16, 1024, 2);
                    const uint64_t bd = B_MN ? make_desc(b_addr + k * 1024, 4096, 512, 1) : make_desc(b_addr + k * 32, 16, 1024, 2);
                    umma_tf32(tmem_base, ad, bd, idesc, (i > 0 || k > 0 || sub > 0) ? 1u : 0u);
                    if (X3) {  // descriptors of the lo tiles: same layout, start address + LO_OFF
                        const uint64_t lo = (uint64_t)((LO_OFF >> 4) & 0x3FFF);
                        umma_tf32(tmem_base, ad + lo, bd, idesc, 1u);
                        umma_tf32(tmem_base, ad, bd + lo, idesc, 1u);
                    }
                }
                }
                umma_commit(&empty_bar[s]);  // frees the smem slot once these MMAs retire
            }
            umma_commit(&tmem_full_bar);
            TC_TRACE(3);  // last MMA issued
        }
    } else {
        // ============================ epilogue (warps 2..5) ============================
        const int q = warp & 3;  // TMEM lane quarter this warp may touch
        const int m = m0 + 32 * q + lane;
        // Everything the epilogue needs from global memory is requested BEFORE the main loop ends:
        // the tile's bias values go to shared memory (one copy per warp, so a __syncwarp suffices) and
        // the LSTM cell's c_prev to registers.  Loading them after the accumulator wait cost one
        // exposed L2 round trip per 8-column chunk (~2 us of a 4.7 us launch, in-kernel trace).
        // EIGHT epilogue warps for wide LSTM tiles when the four splitter warps have nothing to split (both operands
        // arrive pre-split) and the tile is not K-split over a CTA pair: warps 6..9 sit on the same TMEM lane quarters as
        // warps 4, 5, 2, 3 (quarter = warp % 4) and take the upper half of the tile's hidden units.  The activations
        // of 8 units take ~1 750 cycles for a warp that runs alone on its scheduler (dependent MUFU chains: in-kernel
        // trace, round 2) -- 14 000 of the 22 500-cycle epilogue of a 128 x 256 tile; two warps per scheduler overlap them.
        constexpr int HU_E = BN / 4;
        const bool epi8 = EPI == EPI_LSTM && X3 && HU_E >= 32 && ksp == 1 && p.a_lo_g && p.b_lo_g;
        const bool epi_warp = warp < 6 || epi8;
        const int jb_begin = (epi8 && warp >= 6) ? HU_E / 2 : 0;
        const int jb_end = epi8 ? (warp >= 6 ? HU_E : HU_E / 2) : HU_E;
        float cp_pref[8];
        if (epi_warp) {
            float* sb = s_bias[warp - 2];
            if (EPI == EPI_STORE) {
                const bool first_split0 = (p.splits <= 1) || (split == 0);
                for (int j = lane; j < BN; j += 32) {
                    const int n = n_tile * BN + j;
                    float b = 0.f;
                    if (first_split0 && n < p.N) {
                        if (p.bias) b += __ldg(p.bias + n);
                        if (p.bias2) b += __ldg(p.bias2 + n);
                    }
                    sb[j] = b;
                }
            } else {
                constexpr int HU = BN / 4;
                const int n = p.n_hidden, j0 = n_tile * HU;
                for (int j = lane; j < BN; j += 32) {
                    const int g = j / HU, col = g * n + j0 + (j - g * HU);
                    // pre-scaled for the activation the gate goes through (i, f, o: sigmoid; g: tanh), see sigmoid_of_scaled
                    sb[j] = (__ldg(p.bias + col) + __ldg(p.bias2 + col)) * (g == 2 ? 2.0f * NEG_LOG2E : NEG_LOG2E);
                }
                if (m < p.M) {
                    const long off = (long)m * n + j0 + jb_begin;
                    const float4 c0 = *reinterpret_cast<const float4*>(p.c_prev + off);
                    const float4 c1 = *reinterpret_cast<const float4*>(p.c_prev + off + 4);
                    cp_pref[0] = c0.x; cp_pref[1] = c0.y; cp_pref[2] = c0.z; cp_pref[3] = c0.w;
                    cp_pref[4] = c1.x; cp_pref[5] = c1.y; cp_pref[6] = c1.z; cp_pref[7] = c1.w;
                }
            }
            __syncwarp();
        }
        if (X3) {
            // ---- operand splitter: lo = x - trunc_tf32(x) for every landed stage
            // two groups of 4 warps take alternate K blocks, so one group's barrier wake-up / proxy
            // fence / arrive latency overlaps the other group's copy loop
            // (EVEN ring depth only: a group then meets the same slots on every round.  With an odd depth the two
            //  groups alternate on a slot and each sees only every other phase of its full barrier; a parity wait
            //  is unambiguous only against the immediately preceding phase, so a group that arrived while the
            //  round it SKIPPED was still in flight -- TMA copies complete out of order -- took "parity differs"
            //  for "my round has landed", split stale data and arrived on the other group's split barrier: phases
            //  slipped, then a hang or `unspecified launch failure`.  Seen with the 3-stage 128-wide MN/MN variant
            //  next to other streams' kernels, never under the serialising sanitizer.  Odd depths use ONE group.)
            constexpr int NGRP = TC_SPLIT_GROUPS(STAGES);
            constexpr int GRP = TC_SPLITTERS / NGRP;
            const int t = (threadIdx.x - 64) % GRP, grp = (threadIdx.x - 64) / GRP;
            const bool split_a = !p.a_lo_g, split_b = !p.b_lo_g;
            for (int i = grp; (split_a || split_b) && i < my_kb; i += NGRP) {
                const int s = i % stages, ph = (i / stages) & 1;
                mbar_wait(&full_bar[s], ph);
                float4* a_hi = reinterpret_cast<float4*>(sA + s * S::A_BYTES);
                float4* b_hi = reinterpret_cast<float4*>(sB + s * S::B_BYTES);
                float4* a_lo = reinterpret_cast<float4*>(sA + s * S::A_BYTES + LO_OFF);
                float4* b_lo = reinterpret_cast<float4*>(sB + s * S::B_BYTES + LO_OFF);
                auto lo_of = [](float x) { return x - __uint_as_float(__float_as_uint(x) & 0xFFFFE000u); };
#pragma unroll 4
                for (int v = t; split_a && v < S::A_BYTES / 16; v += GRP) {
                    const float4 x = a_hi[v];
                    a_lo[v] = make_float4(lo_of(x.x), lo_of(x.y), lo_of(x.z), lo_of(x.w));
                }
#pragma unroll 4
                for (int v = t; split_b && v < S::B_BYTES / 16; v += GRP) {
                    const float4 x = b_hi[v];
                    b_lo[v] = make_float4(lo_of(x.x), lo_of(x.y), lo_of(x.z), lo_of(x.w));
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes -> visible to UMMA
                asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&split_bar[s])) : "memory");
            }
        }
        if (epi_warp) {  // warps 2..5 own the four TMEM lane quarters (wide LSTM tiles: + warps 6..9, see above)
        // Epilogue parameters are pulled into registers NOW (and made opaque to the compiler, which
        // would otherwise re-read them from the constant bank inside the store loop: the SASS had four
        // dependent LDCU -> compare -> branch chains per row, ~250 cycles per iteration in the trace).
        int e_M = p.M, e_N = p.N, e_mode = p.splits > 1 ? 2 : (p.accumulate ? 1 : 0);
        long e_ldc = p.ldc;
        float* e_C = p.C;
        asm volatile("" : "+r"(e_M), "+r"(e_N), "+r"(e_mode), "+l"(e_ldc), "+l"(e_C));
        mbar_wait(&tmem_full_bar, 0);
        tc_fence_after();
        if (warp == 2 && lane == 0) TC_TRACE(4);  // accumulators complete
        const uint32_t trow = tmem_base + ((uint32_t)(32 * q) << 16);
        if (EPI == EPI_STORE) {
            // Accumulator tile -> shared memory (row per lane) -> global memory with ROW-coalesced 128-bit
            // accesses.  Writing straight from the TMEM registers makes every store instruction touch 32
            // different rows (one 16-byte piece each): the in-kernel trace showed 3700 cycles for a
            // 128 x 64 tile, ~40 % of a small launch.  The pipeline ring is dead by now (every MMA has
            // retired), so the staging tile reuses it.
            constexpr int PITCH = BN + 4;  // 16-byte aligned rows, conflict-free for 128-bit accesses
            static_assert(EPI != EPI_STORE || 4 * 32 * PITCH * 4 <= S::BYTES - 1024, "epilogue staging tile does not fit in the ring");
            float* stg = reinterpret_cast<float*>(smem) + q * 32 * PITCH;
            const int nbase = n_tile * BN;
            const bool vec = ((e_ldc & 3) == 0) && (((uintptr_t)e_C & 15) == 0);
            if (p.c_tma) {
                // TMA epilogue: the warp's 32 x BN accumulator slab goes to shared memory as BN/32 boxes of
                // 32 rows x 128 bytes in the 128B-swizzled layout (conflict-free 128-bit stores: 16-byte
                // chunk c of row r lands at chunk c ^ (r & 7)), and ONE elected lane hands each box to the
                // TMA unit: a plain tensor store, or an f32 reduce-add when the launch accumulates into C
                // or is one of several K splits.  Row / column tails are clipped by the TMA unit.  The
                // per-row store loop below (kept for unaligned C) costs ~230 cycles per row per warp with
                // one warp per scheduler (in-kernel trace): 3700-4200 cycles for a 128 x 64 tile.
                constexpr int BOXES = BN / 32;
                const uint32_t box0 = smem_u32(smem) + (uint32_t)(q * BOXES) * 4096u;
#pragma unroll 1
                for (int c0 = 0; c0 < BN; c0 += 32) {
                    uint32_t r[32];
                    if (my_kb > 0) { TMEM_LD32(trow + c0, r); tmem_ld_wait(); }
                    else {
#pragma unroll
                        for (int j = 0; j < 32; ++j) r[j] = 0u;
                    }
                    const float* sb = s_bias[warp - 2] + c0;
                    const uint32_t rowb = box0 + (uint32_t)(c0 >> 5) * 4096u + (uint32_t)lane * 128u;
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        const uint32_t dst = rowb + (uint32_t)(((j >> 2) ^ (lane & 7)) << 4);
                        asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(dst),
                                     "f"(__uint_as_float(r[j]) + sb[j]), "f"(__uint_as_float(r[j + 1]) + sb[j + 1]),
                                     "f"(__uint_as_float(r[j + 2]) + sb[j + 2]), "f"(__uint_as_float(r[j + 3]) + sb[j + 3])
                                     : "memory");
                    }
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes -> TMA reads
                __syncwarp();
                if (warp == 2 && lane == 0) TC_TRACE(6);
                if (lane == 0 && m0 + 32 * q < e_M) {
#pragma unroll 1
                    for (int b = 0; b < BOXES; ++b) {
                        const int cn = nbase + 32 * b;
                        if (cn >= e_N) break;
                        const uint32_t src = box0 + (uint32_t)b * 4096u;
                        if (e_mode == 0)
                            asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                                             (uint64_t)&p.cmap), "r"(src), "r"(cn), "r"(m0 + 32 * q) : "memory");
                        else
                            asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                                             (uint64_t)&p.cmap), "r"(src), "r"(cn), "r"(m0 + 32 * q) : "memory");
                    }
                    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");  // smem must outlive the reads
                }
            } else {
            const uint32_t stg_s = smem_u32(stg);  // explicit shared-space accesses (generic ones are slower)
#pragma unroll 1
            for (int c0 = 0; c0 < BN; c0 += 32) {
                uint32_t r[32];
                if (my_kb > 0) { TMEM_LD32(trow + c0, r); tmem_ld_wait(); }
                else {
#pragma unroll
                    for (int j = 0; j < 32; ++j) r[j] = 0u;
                }
                const float* sb = s_bias[warp - 2] + c0;
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                    const float4 v = make_float4(__uint_as_float(r[j]) + sb[j], __uint_as_float(r[j + 1]) + sb[j + 1],
                                                 __uint_as_float(r[j + 2]) + sb[j + 2], __uint_as_float(r[j + 3]) + sb[j + 3]);
                    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(stg_s + (uint32_t)(lane * PITCH + c0 + j) * 4),
                                 "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
                }
            }
            __syncwarp();
            constexpr int LPR = BN / 4;    // lanes per row (one float4 each)
            constexpr int RPI = 32 / LPR;  // rows per warp-wide instruction
            const int rr = lane / LPR, c4 = (lane % LPR) * 4;
            const int n = nbase + c4;
            const bool full4 = vec && n + 4 <= e_N;
            if (n < e_N) {
#pragma unroll 1  // executed once per launch: keep the loop body short
                for (int r0 = 0; r0 < 32; r0 += RPI) {
                    const int row = r0 + rr, mrow = m0 + 32 * q + row;
                    if (mrow >= e_M) break;  // rows grow with r0
                    float4 v;
                    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                                 : "r"(stg_s + (uint32_t)(row * PITCH + c4) * 4));
                    float* crow = e_C + (long)mrow * e_ldc + n;
#ifdef MARLC_TC_NOSTORE
                    if (v.x == 123.456f) crow[0] = v.y;
                    continue;
#endif
#ifdef MARLC_TC_TRACE
                    if (warp == 2 && lane == 0 && r0 == RPI * 2) TC_TRACE(7);
#endif
                    if (full4) {
                        if (e_mode == 2) {
                            atomicAdd(reinterpret_cast<float4*>(crow), v);
                        } else {
                            if (e_mode == 1) {
                                const float4 o = *reinterpret_cast<const float4*>(crow);
                                v.x += o.x; v.y += o.y; v.z += o.z; v.w += o.w;
                            }
                            *reinterpret_cast<float4*>(crow) = v;
                        }
                    } else {
                        const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            if (n + j >= e_N) break;
                            if (e_mode == 2) atomicAdd(crow + j, vv[j]);
                            else crow[j] = e_mode == 1 ? crow[j] + vv[j] : vv[j];
                        }
                    }
                }
            }
            }  // !c_tma
        } else {
            // fused LSTM cell (recurrent.py:30): columns [g*HU + j] hold gate g of hidden unit j0 + j
            constexpr int HU = BN / 4;
            const int n = p.n_hidden, j0 = n_tile * HU;
            // K split over a CTA pair: each SM streams only half of the A tile (the main loop is bound by
            // per-SM TMA ingest).  The odd CTA writes its partial gate sums into the even CTA's shared
            // memory (distributed shared memory), one cluster barrier, the even CTA adds them.
            constexpr int PPITCH = BN + 4;
            float* part = reinterpret_cast<float*>(smem + (S::BYTES - 1024));  // [BM][PPITCH], after the ring
            if (ksp > 1) asm volatile("barrier.cluster.wait.acquire;" ::: "memory");  // the partner CTA has entered
            if (ksp > 1 && kslice != 0) {
                uint32_t remote;
                asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(smem_u32(part)), "r"(0));
                const uint32_t rrow = remote + (uint32_t)((32 * q + lane) * PPITCH) * 4u;
#pragma unroll 1
                for (int c0 = 0; c0 < BN; c0 += 8) {
                    uint32_t r[8];
                    if (my_kb > 0) { TMEM_LD8(trow + c0, r); tmem_ld_wait(); }
                    else {
#pragma unroll
                        for (int j = 0; j < 8; ++j) r[j] = 0u;
                    }
                    asm volatile("st.shared::cluster.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(rrow + (uint32_t)c0 * 4u), "r"(r[0]),
                                 "r"(r[1]), "r"(r[2]), "r"(r[3]) : "memory");
                    asm volatile("st.shared::cluster.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(rrow + (uint32_t)c0 * 4u + 16u), "r"(r[4]),
                                 "r"(r[5]), "r"(r[6]), "r"(r[7]) : "memory");
                }
            }
            if (ksp > 1) {
                asm volatile("barrier.cluster.arrive.release;" ::: "memory");
                asm volatile("barrier.cluster.wait.acquire;" ::: "memory");
            }
            const float* prow = part + (32 * q + lane) * PPITCH;
            // The seven outputs of the cell (4 activated gates, c, h, low-order part of h) are row-major arrays in
            // global memory while TMEM hands every lane ONE ROW of the tile: stored straight from the registers, each
            // 128-bit store instruction touched 32 rows (32 half-sector requests), and the epilogue took 7 300 cycles
            // of a 27 000-cycle launch at 512 rows -- the same with 4 or 8 warps sharing it, i.e. bound by the
            // requests, not by the arithmetic (in-kernel trace, round 2).  Now a chunk of CH hidden units is staged in
            // the (dead) pipeline ring, row per lane, and leaves with the lanes running ALONG the rows: 4 x CH bytes
            // contiguous per row and array.  (K-split pairs keep the direct stores: their tile is 8 units wide.)
            constexpr int RINGF = (S::BYTES - 1024) / 4;  // floats of the ring
            constexpr int NEW = (X3 && HU >= 32) ? 8 : 4;  // epilogue warps that may stage at once (see epi8)
            constexpr int CH_FIT = NEW * 7 * 32 * (32 + 4) <= RINGF ? 32 : (NEW * 7 * 32 * (16 + 4) <= RINGF ? 16 : 8);
            constexpr int CH = HU / (NEW / 4) < CH_FIT ? HU / (NEW / 4) : CH_FIT;  // hidden units per staged chunk
            constexpr int SP = CH + 4;             // staging row pitch: conflict-free 128-bit row-per-lane writes
            constexpr int LPR = CH / 4, RPI = 32 / LPR;  // lanes per row / rows per store instruction on the way out
            static_assert(EPI != EPI_LSTM || NEW * 7 * 32 * SP * 4 <= S::BYTES - 1024, "cell staging does not fit in the ring");
            const bool staged = ksp == 1;
            float* stg = reinterpret_cast<float*>(smem) + (warp - 2) * (7 * 32 * SP);  // [7 arrays][32 rows][SP] of this warp
            if (ksp == 1 || kslice == 0) {
#pragma unroll 1
            for (int jb = jb_begin; jb < jb_end; jb += 8) {
                uint32_t ri[8], rf[8], rg[8], ro[8];
                TMEM_LD8(trow + 0 * HU + jb, ri);
                TMEM_LD8(trow + 1 * HU + jb, rf);
                TMEM_LD8(trow + 2 * HU + jb, rg);
                TMEM_LD8(trow + 3 * HU + jb, ro);
                tmem_ld_wait();
#ifdef MARLC_TC_TRACE
                if (warp == 2 && lane == 0 && jb == 0) TC_TRACE(6);  // first chunk's accumulators in registers
#endif
                if (ksp > 1) {  // add the partner's half of K
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        ri[j] = __float_as_uint(__uint_as_float(ri[j]) + prow[0 * HU + jb + j]);
                        rf[j] = __float_as_uint(__uint_as_float(rf[j]) + prow[1 * HU + jb + j]);
                        rg[j] = __float_as_uint(__uint_as_float(rg[j]) + prow[2 * HU + jb + j]);
                        ro[j] = __float_as_uint(__uint_as_float(ro[j]) + prow[3 * HU + jb + j]);
                    }
                }
                const bool row_ok = m < p.M;
                if (row_ok || staged) {  // (staged: lanes past the last row compute on zero-filled operands, store nothing)
                    const long off = (long)m * n + j0 + jb;
                    // c_prev of this chunk was requested one chunk ago (the first one before the main loop ended);
                    // the next chunk's request goes out now, ahead of this chunk's activations
                    float cp[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) cp[j] = row_ok ? cp_pref[j] : 0.f;
                    if (row_ok && jb + 8 < jb_end) {
                        const float4 cp0 = *reinterpret_cast<const float4*>(p.c_prev + off + 8);
                        const float4 cp1 = *reinterpret_cast<const float4*>(p.c_prev + off + 12);
                        cp_pref[0] = cp0.x; cp_pref[1] = cp0.y; cp_pref[2] = cp0.z; cp_pref[3] = cp0.w;
                        cp_pref[4] = cp1.x; cp_pref[5] = cp1.y; cp_pref[6] = cp1.z; cp_pref[7] = cp1.w;
                    }
                    const float* sb = s_bias[warp - 2];
                    float gi[8], gf[8], gc[8], go[8], cn[8], hn[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        gi[j] = sigmoid_of_scaled(fmaf(__uint_as_float(ri[j]), NEG_LOG2E, sb[0 * HU + jb + j]));
                        gf[j] = sigmoid_of_scaled(fmaf(__uint_as_float(rf[j]), NEG_LOG2E, sb[1 * HU + jb + j]));
                        gc[j] = tanh_of_scaled(fmaf(__uint_as_float(rg[j]), 2.0f * NEG_LOG2E, sb[2 * HU + jb + j]));
                        go[j] = sigmoid_of_scaled(fmaf(__uint_as_float(ro[j]), NEG_LOG2E, sb[3 * HU + jb + j]));
                        cn[j] = gf[j] * cp[j] + gi[j] * gc[j];
                        hn[j] = go[j] * fast_tanh(cn[j]);
                    }
                    auto st8 = [](float* dst, const float* v) {
                        *reinterpret_cast<float4*>(dst) = make_float4(v[0], v[1], v[2], v[3]);
                        *reinterpret_cast<float4*>(dst + 4) = make_float4(v[4], v[5], v[6], v[7]);
                    };
                    float hl[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) hl[j] = hn[j] - __uint_as_float(__float_as_uint(hn[j]) & 0xFFFFE000u);
#ifdef MARLC_TC_TRACE
                    if (warp == 2 && lane == 0 && jb == 0) TC_TRACE(7);  // first chunk's activations done
#endif
                    if (staged) {
                        float* srow = stg + lane * SP + (jb % CH);
                        st8(srow, gi); st8(srow + 32 * SP, gf); st8(srow + 2 * 32 * SP, gc); st8(srow + 3 * 32 * SP, go);
                        st8(srow + 4 * 32 * SP, cn); st8(srow + 5 * 32 * SP, hn); st8(srow + 6 * 32 * SP, hl);
                    } else {
                        float* g_row = p.gates + (long)m * 4 * n + j0 + jb;
                        st8(g_row, gi); st8(g_row + n, gf); st8(g_row + 2 * n, gc); st8(g_row + 3 * n, go);
                        st8(p.c_new + off, cn);
                        st8(p.h_new + off, hn);
                        if (p.h_new_lo) st8(p.h_new_lo + off, hl);
                    }
                }
#ifdef MARLC_TC_TRACE
                if (warp == 2 && lane == 0 && jb == 0) TC_TRACE(8);  // first chunk staged
                if (warp == 2 && lane == 0 && jb == 8) TC_TRACE(10);  // second chunk staged
#endif
                if (staged && (jb + 8) % CH == 0) {  // a chunk of CH units is complete: out, lanes along the rows
                    __syncwarp();
                    const int jc = jb + 8 - CH, rr = lane / LPR, c4 = (lane % LPR) * 4;
#pragma unroll 1
                    for (int a = 0; a < 7; ++a) {
                        float* base;
                        long ld = n;
                        if (a < 4) { base = p.gates + a * n + j0 + jc; ld = 4L * n; }
                        else if (a == 4) base = p.c_new + j0 + jc;
                        else if (a == 5) base = p.h_new + j0 + jc;
                        else { if (!p.h_new_lo) break; base = p.h_new_lo + j0 + jc; }
                        const float* sa = stg + a * 32 * SP;
#pragma unroll
                        for (int r0 = 0; r0 < 32; r0 += RPI) {
                            const int row = r0 + rr, mrow = m0 + 32 * q + row;
                            if (mrow < p.M)
                                *reinterpret_cast<float4*>(base + (long)mrow * ld + c4) =
                                    *reinterpret_cast<const float4*>(sa + row * SP + c4);
                        }
                    }
                    __syncwarp();  // the next chunk overwrites the staging rows
#ifdef MARLC_TC_TRACE
                    if (warp == 2 && lane == 0 && jb + 8 == CH) TC_TRACE(9);  // first staged chunk written out
#endif
                }
            }
            }  // receiving / only CTA
        }
        }  // warp < 6
    }
    if (ksp > 1 && !(warp >= 2 && warp < 6)) {  // every thread of the pair takes part in the cluster barriers
        asm volatile("barrier.cluster.wait.acquire;" ::: "memory");  // phase 1 ("entered"), see above
        asm volatile("barrier.cluster.arrive.release;" ::: "memory");
        asm volatile("barrier.cluster.wait.acquire;" ::: "memory");
    }
    if (warp == 2 && lane == 0) TC_TRACE(5);  // epilogue of warp 2 done
    tc_fence_before();
    __syncthreads();
#ifdef MARLC_TC_TRACE
    if (tr && threadIdx.x == 0)
        printf("tc trace BN=%d X3=%d KS=%d EPI=%d kb=%d: setup %lld | tma0 %lld | full0 %lld | mma_issued %lld | acc_done %lld | epi_done %lld | end %lld\n",
               BN, (int)X3, KS, EPI, my_kb, trace[0], trace[1], trace[2], trace[3], trace[4], trace[5], clock64() - t_entry);
    if (tr && threadIdx.x == 0 && EPI == EPI_STORE) printf("   staged at %lld, third store iteration at %lld\n", trace[6], trace[7]);
    if (tr && threadIdx.x == 0 && EPI == EPI_LSTM)
        printf("   cell: first 8 units loaded %lld | activated %lld | staged %lld | second 8 staged %lld | first chunk written out %lld\n",
               trace[6], trace[7], trace[8], trace[10], trace[9]);
#endif
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS));
    }
}

template <int BN, bool A_MN, bool B_MN, int EPI, int STAGES, bool X3, int KS>
__global__ void __launch_bounds__(X3 ? TC_THREADS_X3 : TC_THREADS, 1) tc_gemm_kernel(const __grid_constant__ TcKernelGroup pp) {
    if (pp.trig) pdl_trigger();  // the next kernel of a dependent chain may start its prologue (common.cuh)
    const int z = blockIdx.z;
    if (pp.count >= 3 && z >= pp.zofs[2]) tc_gemm_body<BN, A_MN, B_MN, EPI, STAGES, 2, X3, KS>(pp, z - pp.zofs[2]);
    else if (pp.count >= 2 && z >= pp.zofs[1]) tc_gemm_body<BN, A_MN, B_MN, EPI, STAGES, 1, X3, KS>(pp, z - pp.zofs[1]);
    else tc_gemm_body<BN, A_MN, B_MN, EPI, STAGES, 0, X3, KS>(pp, z);
}

// ---------------------------------------------------------------------------------
// host launchers
// ---------------------------------------------------------------------------------
static int operand_map(CUtensorMap* m, const TcOperand& o, int mn_extent, int k_extent, int box_rows_kmajor) {
    // K-major: [mn_extent rows][k_extent inner];  MN-major: [k_extent rows][mn_extent inner]
    if (!o.mn_major) return make_map(m, o.ptr, k_extent, mn_extent, o.slabs, o.ld, o.slab_stride, box_rows_kmajor);
    return make_map(m, o.ptr, mn_extent, k_extent, o.slabs, o.ld, o.slab_stride, 32, true);
}

template <int BN, bool A_MN, bool B_MN, bool X3, int KS>
static int launch_store(TcKernelGroup& kp, int gx, int gy, int gz, int max_kb, cudaStream_t s) {
    (void)max_kb;
    // KS == 1: <= 96 KB per CTA, two CTAs per SM (epilogue / main loop overlap); fat stages: 2-deep ring
    constexpr int STAGES = KS > 1 ? 2 : (BN >= 128 ? 3 : 4);
    using S = TcSmem<BN, STAGES, X3, KS>;
    static_assert(S::BYTES <= 227 * 1024, "tile configuration exceeds shared memory");
    auto kern = tc_gemm_kernel<BN, A_MN, B_MN, EPI_STORE, STAGES, X3, KS>;
    static bool attr_done = false;
    if (!attr_done) {
        MARLC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, S::BYTES));
        attr_done = true;
    }
    kp.trig = pdl_trigger_early();
    MARLC_CUDA(launch_pdl(kern, dim3(gx, gy, gz), dim3(X3 ? TC_THREADS_X3 : TC_THREADS), S::BYTES, s, kp));
    ++g_tc_gemm_launches;
    MARLC_LAUNCH_CHECK();
    return 0;
}

// Tile width for a launch of `count` problems: narrow tiles keep small launches spread over the SMs,
// 128-wide tiles halve the operand bytes per flop once there is a wave of CTAs anyway.  K splits count as
// CTAs (weight gradients: few output tiles, reductions of 10^4..10^6 rows cut into TC_MAX_CHAIN chains).
// The per-step input-gradient group (du | dh | dh^) is bound by the chip-wide L2 -> SM throughput: every tile
// re-streams its K range, so 128-wide tiles (split-K restores the CTA count) move a third fewer bytes.  Measured
// per 16 steps: 512 rows 320 -> 238 us, 1024 rows 590 -> 418 us, 128 rows 180 -> 181 us (kept at 64 there).
constexpr int TC_DX128_MIN_CTAS = 16;
// Weight gradients (MN-major x MN-major, reductions of 10^4.. rows cut into chains) stay at 128 wide.  128 x 256
// tiles would read A once per 256 output columns instead of once per 128 (dW_ih at 65 536 rows: 1.58 -> 1.31 GB per
// cell), but MEASURED SLOWER (backward at c4: 8.14 vs 7.99 ms): the 96 KB stages leave room for a 2-deep ring only.
// (The 128-wide MN/MN variant once exposed a phase-aliasing bug of the operand splitter with odd ring depths --
//  fixed in tc_gemm_body, see the comment there.)
static int pick_bn(const TcGemmArgs* args, int count) {
    int max_n = 0;
    long ctas128 = 0;
    for (int i = 0; i < count; ++i) {
        const TcGemmArgs& a = args[i];
        max_n = max(max_n, a.N);
        long chains = a.allow_split ? max(1L, ((long)a.K + a.K2 + TC_MAX_CHAIN - 1) / TC_MAX_CHAIN) : 1L;
        // weight gradients: split-K (>= 4 K blocks of 32 per split) restores the CTA count of wide tiles
        // (measured per iteration with / without: 512 rows per step 2415 vs 2515 us, 1024 rows 4002 vs 4068, 128 rows 1563 vs 1576)
        if (a.allow_split == 1 && a.A.mn_major && a.B.mn_major) chains = max(chains, ((long)a.K + a.K2) / 128);
        ctas128 += (long)((a.M + BM - 1) / BM) * ((a.N + 127) / 128) * chains;
    }
    if (max_n <= 32) return 32;
    const bool dx_group = !args[0].A.mn_major && args[0].B.mn_major && count > 1;  // per-step input-gradient group
    if (max_n <= 64 || ctas128 < (dx_group ? TC_DX128_MIN_CTAS : MARLC_SMS / 2)) return 64;
    return 128;
}

// Up to TC_MAX_GROUP problems with the same operand majors in ONE launch.
int tc_gemm_group(const TcGemmArgs* args, int count, cudaStream_t s) {
    MARLC_CHECK(count >= 1 && count <= TC_MAX_GROUP, "tc_gemm_group: count=%d", count);
    const int BN = pick_bn(args, count);
    TcKernelGroup kp;
    memset(&kp, 0, sizeof(kp));
    kp.count = count;
    int gx = 0, gy = 0, ctas = 0, min_k = 1 << 30;
    int pdl_ok = g_pdl;
    for (int i = 0; i < count; ++i) {
        const TcGemmArgs& a = args[i];
        ctas += ((a.M + BM - 1) / BM) * ((a.N + BN - 1) / BN);
        min_k = min(min_k, a.K + a.K2);
    }
    // fat stages (2 x 32 floats of K per barrier round trip) for latency-bound launches
    const int KS = (ctas < MARLC_SMS && BN <= 64 && min_k >= 128) ? 2 : 1;
    const int BKS = BK * KS;
    for (int i = 0; i < count; ++i) {
        const TcGemmArgs& a = args[i];
        MARLC_CHECK(tc_operand_ok(a.A) && tc_operand_ok(a.B), "tc_gemm: operand not TMA-addressable");
        MARLC_CHECK(a.K > 0 && a.M > 0 && a.N > 0, "tc_gemm: empty problem");
        MARLC_CHECK(a.A.mn_major == args[0].A.mn_major && a.B.mn_major == args[0].B.mn_major,
                    "tc_gemm_group: all problems must share operand majors");
        const bool pair2 = a.K2 > 0;
        if (pair2) {
            MARLC_CHECK(tc_operand_ok(a.A2) && tc_operand_ok(a.B2), "tc_gemm: second operand pair not TMA-addressable");
            MARLC_CHECK(a.A2.mn_major == a.A.mn_major && a.B2.mn_major == a.B.mn_major, "tc_gemm: operand pairs must share majors");
        }
        TcKernelParams& p = kp.p[i];
        MARLC_TRY(operand_map(&p.a1, a.A, a.M, a.K, BM));
        MARLC_TRY(operand_map(&p.b1, a.B, a.N, a.K, BN));
        p.nk1 = (a.K + BKS - 1) / BKS;
        p.slab_a1 = a.A.slab; p.slab_b1 = a.B.slab;
        p.a_lo_g = (a.x3 && a.A.lo && (!pair2 || a.A2.lo)) ? 1 : 0;
        p.b_lo_g = (a.x3 && a.B.lo && (!pair2 || a.B2.lo)) ? 1 : 0;
        if (p.a_lo_g) { TcOperand o = a.A; o.ptr = a.A.lo; MARLC_TRY(operand_map(&p.a1l, o, a.M, a.K, BM)); }
        if (p.b_lo_g) { TcOperand o = a.B; o.ptr = a.B.lo; MARLC_TRY(operand_map(&p.b1l, o, a.N, a.K, BN)); }
        if (pair2) {
            MARLC_TRY(operand_map(&p.a2, a.A2, a.M, a.K2, BM));
            MARLC_TRY(operand_map(&p.b2, a.B2, a.N, a.K2, BN));
            p.nk2 = (a.K2 + BKS - 1) / BKS;
            p.slab_a2 = a.A2.slab; p.slab_b2 = a.B2.slab;
            if (p.a_lo_g) { TcOperand o = a.A2; o.ptr = a.A2.lo; MARLC_TRY(operand_map(&p.a2l, o, a.M, a.K2, BM)); }
            if (p.b_lo_g) { TcOperand o = a.B2; o.ptr = a.B2.lo; MARLC_TRY(operand_map(&p.b2l, o, a.N, a.K2, BN)); }
        }
        p.M = a.M; p.N = a.N; p.C = a.C; p.ldc = a.ldc; p.bias = a.bias; p.bias2 = a.bias2;
        p.accumulate = a.accumulate;
        p.c_tma = ((a.ldc & 3) == 0 && ((uintptr_t)a.C & 15) == 0) ? 1 : 0;
        if (p.c_tma) MARLC_TRY(make_map_c(&p.cmap, a.C, a.M, a.N, a.ldc));
        const int mt = (a.M + BM - 1) / BM, nt = (a.N + BN - 1) / BN, nkb = p.nk1 + p.nk2;
        int splits = 1;
        if (a.allow_split && ctas < MARLC_SMS) {
            // allow_split == 2: latency-bound per-step launch, split down to ONE stage per CTA
            // one wave: the ring leaves room for ONE CTA per SM, so more than 148 CTAs run as two waves
            // (in-kernel trace: 5.3 us per CTA, 13.4 us for the 190-CTA dX group)
            splits = min(a.allow_split >= 2 ? nkb : max(1, nkb * KS / 4), max(1, MARLC_SMS / ctas));
            splits = min(splits, nkb);
        }
        if (a.allow_split) {
            // Long reductions (weight gradients: K = T*M rows, up to millions for the conv layers): the
            // tensor core adds into its fp32 TMEM accumulator with truncation, a bias that grows with the
            // length of the chain (measured on dW_ih: 2.5e-5 rel. at K = 2048, 6.3e-4 at K = 65536).  Chains are
            // therefore capped at TC_MAX_CHAIN elements of K per CTA; the partial sums meet in the epilogue's
            // f32 reduce-add (round-to-nearest in L2).  Those launches are throughput-bound: extra waves are free.
            const int chain_blocks = max(1, TC_MAX_CHAIN / BKS);
            splits = max(splits, (nkb + chain_blocks - 1) / chain_blocks);
            // every split must own at least one K block
            while (splits > 1 && ((nkb + splits - 1) / splits) * (splits - 1) >= nkb) --splits;
        }
        p.splits = splits;
        if (splits > 1 && !a.accumulate && !a.c_zeroed) {
            pdl_ok = 0;  // the predecessor in the stream is a memset now: ordinary launch
            if (a.ldc == a.N) MARLC_CUDA(cudaMemsetAsync(a.C, 0, sizeof(float) * (size_t)a.M * a.N, s));
            else MARLC_CUDA(cudaMemset2DAsync(a.C, sizeof(float) * a.ldc, 0, sizeof(float) * a.N, a.M, s));
        }
        kp.zofs[i + 1] = kp.zofs[i] + splits;
        gx = max(gx, nt);
        gy = max(gy, mt);
    }
    const int gz = kp.zofs[count];
    PdlScope pdl_scope(pdl_ok, g_pdl_trig);
    int max_kb = 1;
    for (int i = 0; i < count; ++i) {
        const int nkb = kp.p[i].nk1 + kp.p[i].nk2;
        max_kb = max(max_kb, (nkb + kp.p[i].splits - 1) / kp.p[i].splits);
    }
    const bool amn = args[0].A.mn_major, bmn = args[0].B.mn_major;
    const bool x3 = args[0].x3 != 0;
#define DISPATCH3(BNv, X, KSv)                                                                   \
    if (amn) {                                                                                   \
        if (bmn) return launch_store<BNv, true, true, X, KSv>(kp, gx, gy, gz, max_kb, s);        \
        return launch_store<BNv, true, false, X, KSv>(kp, gx, gy, gz, max_kb, s);                \
    } else {                                                                                     \
        if (bmn) return launch_store<BNv, false, true, X, KSv>(kp, gx, gy, gz, max_kb, s);       \
        return launch_store<BNv, false, false, X, KSv>(kp, gx, gy, gz, max_kb, s);               \
    }
#define DISPATCH(BNv, KSv)            \
    if (x3) { DISPATCH3(BNv, true, KSv) } \
    else { DISPATCH3(BNv, false, KSv) }
    if (BN == 32) { if (KS == 2) { DISPATCH(32, 2) } DISPATCH(32, 1) }
    if (BN == 64) { if (KS == 2) { DISPATCH(64, 2) } DISPATCH(64, 1) }
    DISPATCH(128, 1)
#undef DISPATCH
#undef DISPATCH3
}

int tc_gemm(const TcGemmArgs& a, cudaStream_t s) { return tc_gemm_group(&a, 1, s); }

template <int BN, bool X3, int KS>
static int launch_lstm(TcKernelGroup& kp, int gx, int gy, int nkb, cudaStream_t s) {
    (void)nkb;
    constexpr int STAGES = BN >= 256 ? (X3 ? 2 : 4) : (KS > 1 ? 2 : (BN >= 128 ? 3 : 4));  // KS == 1: 3 x 32 KB, two CTAs per SM
    using S = TcSmem<BN, STAGES, X3, KS>;
    static_assert(S::BYTES <= 227 * 1024, "tile configuration exceeds shared memory");
    auto kern = tc_gemm_kernel<BN, false, false, EPI_LSTM, STAGES, X3, KS>;
    static bool attr_done = false;
    if (!attr_done) {
        MARLC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, S::BYTES));
        attr_done = true;
    }
    const int ksp = kp.p[0].ksplit > 1 ? kp.p[0].ksplit : 1;  // a K-split pair runs as a cluster of ksp CTAs
    const size_t smem_bytes = S::BYTES + (ksp > 1 ? (size_t)BM * (BN + 4) * 4 : 0);
    MARLC_CHECK(smem_bytes <= 227 * 1024, "tc_lstm_pair: K-split staging does not fit in shared memory");
    static size_t attr_sz = 0;
    if (smem_bytes > attr_sz) {
        MARLC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes));
        attr_sz = smem_bytes;
    }
    kp.trig = pdl_trigger_early();
    MARLC_CUDA(launch_pdl(kern, dim3(gx * ksp, gy, 2), dim3(X3 ? TC_THREADS_X3 : TC_THREADS), smem_bytes, s, kp, ksp));
    ++g_tc_gemm_launches;
    MARLC_LAUNCH_CHECK();
    return 0;
}

bool tc_lstm_shapes_ok(int Kin, int n) { return Kin % 4 == 0 && n % 8 == 0 && n >= 8; }

bool tc_lstm_supported(const TcLstmArgs& a) {
    return tc_operand_ok(a.U) && tc_operand_ok(a.Hprev) && (((uintptr_t)a.Wih | (uintptr_t)a.Whh) & 15) == 0 &&
           tc_lstm_shapes_ok(a.Kin, a.n) && (((uintptr_t)a.c_prev | (uintptr_t)a.c_new | (uintptr_t)a.h_new |
           (uintptr_t)a.gates) & 15) == 0;
}

TcLstmPlan tc_lstm_plan(int M, int n0, int n1, bool x3) {
    // hidden units per CTA: small tiles when M is small (more CTAs), 32 when rows are plentiful
    const int mt = (M + BM - 1) / BM;
    int HU = mt >= 8 ? 32 : (mt >= 2 ? 16 : 8);
    // 128 x 256 tiles (64 hidden units x 4 gates) once they still fill the machine: a kind::tf32 MMA reads its
    // operands from shared memory at 128 B/clk for a 128 x 128 tile (the whole shared-memory bandwidth of the
    // SM, before the TMA writes and the 3xTF32 low-order tiles), 96 B/clk for 128 x 256 -- and the tile streams
    // 25 % fewer operand bytes per flop
    // (measured, 16 steps at n = 256: M = 2048 -> 796 us with 64 units per tile vs 858 with 32; M = 1024 -> 673 vs 439)
    if (n0 % 64 == 0 && n1 % 64 == 0 && 2 * mt * (n0 / 64) >= 120) HU = 64;
    while (HU > 8 && (n0 % HU != 0 || n1 % HU != 0)) HU >>= 1;
    // few CTAs (small M): fat stages, KS sub-blocks of 32 floats per barrier round trip
    const bool fat = HU <= 16 && 2 * mt * (n0 / HU) <= MARLC_SMS;
    const int KSv = !fat ? 1 : (x3 ? 2 : (HU == 8 ? 4 : 2));
    // (A-tile TMA multicast across the n/HU CTAs of one M tile was measured: no gain at M=128 - 14.4 vs 14.1 us -
    // and slightly slower at M=4096: what binds is the bytes ARRIVING in each SM, not the requests its TMA engine
    // issues.  Removed.)
    // K split over CTA pairs (DSMEM reduction): halves the bytes each SM streams; used when the launch is
    // small enough that twice the CTAs still fit in one wave
    const int ksplit = (fat && HU == 8 && 2 * 2 * mt * (n0 / HU) <= MARLC_SMS) ? 2 : 1;
    TcLstmPlan p;
    p.hu = HU; p.bn = 4 * HU; p.fat = fat ? 1 : 0; p.ks = KSv; p.ksplit = ksplit;
    p.tail_rows = M - (mt - 1) * BM;
    return p;
}

int tc_lstm_pair(const TcLstmArgs& c0, const TcLstmArgs& c1, cudaStream_t s) {
    MARLC_CHECK(tc_lstm_supported(c0) && tc_lstm_supported(c1), "tc_lstm_pair: unsupported shapes / alignment");
    MARLC_CHECK(c0.M == c1.M, "tc_lstm_pair: row counts differ");
    const int mt = (c0.M + BM - 1) / BM;
    const TcLstmPlan pl = tc_lstm_plan(c0.M, c0.n, c1.n, c0.x3 != 0);
    const int HU = pl.hu, KSv = pl.ks, ksplit = pl.ksplit;
    const bool fat = pl.fat != 0;
    MARLC_CHECK(c0.n % HU == 0 && c1.n % HU == 0, "tc_lstm_pair: hidden size not a multiple of %d", HU);
    TcKernelGroup kp;
    memset(&kp, 0, sizeof(kp));
    kp.count = 2;
    kp.zofs[0] = 0; kp.zofs[1] = 1; kp.zofs[2] = 2;
    const int BKS = BK * KSv;
    const TcLstmArgs* cs[2] = {&c0, &c1};
    int gx = 0;
    for (int k = 0; k < 2; ++k) {
        const TcLstmArgs& c = *cs[k];
        TcKernelParams& p = kp.p[k];
        p.ksplit = ksplit;
        MARLC_TRY(make_map(&p.a1, c.U.ptr, c.Kin, c.M, c.U.slabs, c.U.ld, c.U.slab_stride, BM));
        // weights viewed as [gate][unit][K]: ONE box of HU units x 4 gates per K sub-block (the producer
        // thread is issue-bound: 4 separate gate boxes per sub-block made 20 TMA instructions per stage)
        MARLC_TRY(make_map(&p.b1, c.Wih, c.Kin, c.n, 4, c.Kin, (long)c.n * c.Kin, HU, false, 4));
        MARLC_TRY(make_map(&p.a2, c.Hprev.ptr, c.n, c.M, c.Hprev.slabs, c.Hprev.ld, c.Hprev.slab_stride, BM));
        MARLC_TRY(make_map(&p.b2, c.Whh, c.n, c.n, 4, c.n, (long)c.n * c.n, HU, false, 4));
        p.nk1 = (c.Kin + BKS - 1) / BKS;
        p.nk2 = (c.n + BKS - 1) / BKS;
        p.a_lo_g = (c.x3 && c.U.lo && c.Hprev.lo) ? 1 : 0;
        p.b_lo_g = (c.x3 && c.Wih_lo && c.Whh_lo) ? 1 : 0;
        if (p.a_lo_g) {
            MARLC_TRY(make_map(&p.a1l, c.U.lo, c.Kin, c.M, c.U.slabs, c.U.ld, c.U.slab_stride, BM));
            MARLC_TRY(make_map(&p.a2l, c.Hprev.lo, c.n, c.M, c.Hprev.slabs, c.Hprev.ld, c.Hprev.slab_stride, BM));
        }
        if (p.b_lo_g) {
            MARLC_TRY(make_map(&p.b1l, c.Wih_lo, c.Kin, c.n, 4, c.Kin, (long)c.n * c.Kin, HU, false, 4));
            MARLC_TRY(make_map(&p.b2l, c.Whh_lo, c.n, c.n, 4, c.n, (long)c.n * c.n, HU, false, 4));
        }
        p.h_new_lo = c.h_new_lo;
        p.slab_a1 = c.U.slab; p.slab_a2 = c.Hprev.slab;
        p.M = c.M; p.N = 4 * c.n;
        p.bias = c.bih; p.bias2 = c.bhh;
        p.c_prev = c.c_prev; p.c_new = c.c_new; p.h_new = c.h_new; p.gates = c.gates;
        p.n_hidden = c.n;
        p.splits = 1;
        gx = max(gx, c.n / HU);
    }
    MARLC_CHECK(c0.n == c1.n, "tc_lstm_pair: the two cells must have the same hidden size (got %d, %d)", c0.n, c1.n);
    const int nkb = kp.p[0].nk1 + kp.p[0].nk2;
    if (fat) {  // latency-bound (few CTAs): fat stages
        if (c0.x3) {
            if (HU == 8) return launch_lstm<32, true, 2>(kp, gx, mt, nkb, s);
            return launch_lstm<64, true, 2>(kp, gx, mt, nkb, s);
        }
        if (HU == 8) return launch_lstm<32, false, 4>(kp, gx, mt, nkb, s);
        return launch_lstm<64, false, 2>(kp, gx, mt, nkb, s);
    }
    if (c0.x3) {
        if (HU == 8) return launch_lstm<32, true, 1>(kp, gx, mt, nkb, s);
        if (HU == 16) return launch_lstm<64, true, 1>(kp, gx, mt, nkb, s);
        if (HU == 32) return launch_lstm<128, true, 1>(kp, gx, mt, nkb, s);
        return launch_lstm<256, true, 1>(kp, gx, mt, nkb, s);
    }
    if (HU == 8) return launch_lstm<32, false, 1>(kp, gx, mt, nkb, s);
    if (HU == 16) return launch_lstm<64, false, 1>(kp, gx, mt, nkb, s);
    if (HU == 32) return launch_lstm<128, false, 1>(kp, gx, mt, nkb, s);
    return launch_lstm<256, false, 1>(kp, gx, mt, nkb, s);
}

}  // namespace marlc

// Tensor-core (tcgen05 / TMA) GEMM interface, implemented in gemm_tc.cu.
#pragma once
#include <string.h>

#include "common.cuh"

namespace marlc {

// One GEMM operand in global memory.
//   K-major  (mn_major = false): [M or N rows][K contiguous], row stride ld
//   MN-major (mn_major = true) : [K rows][M or N contiguous], row stride ld
// Optionally one slab of a [slabs][rows][ld] stack (time-stacked activations).
struct TcOperand {
    const float* ptr = nullptr;
    const float* lo = nullptr;  // optional pre-split low-order part (x - trunc_tf32(x)), same layout
    long ld = 0;
    bool mn_major = false;
    int slabs = 1;
    long slab_stride = 0;
    int slab = 0;
};
inline TcOperand tc_op(const float* p, long ld, bool mn_major = false) {
    TcOperand o;
    o.ptr = p; o.ld = ld; o.mn_major = mn_major;
    return o;
}
bool tc_operand_ok(const TcOperand& o);

// D[M,N] (+)= sum_k A(m,k) B(n,k) + sum_k2 A2(m,k2) B2(n,k2) + bias[n] + bias2[n]
struct TcGemmArgs {
    TcOperand A, B;
    int K = 0;
    TcOperand A2, B2;
    int K2 = 0;
    float* C = nullptr;
    long ldc = 0;
    int M = 0, N = 0;
    const float* bias = nullptr;
    const float* bias2 = nullptr;
    int accumulate = 0;
    int allow_split = 0;  // 1: split-K (TMA reduce-add epilogue) when the grid would be small; 2: down to one stage per CTA
    int c_zeroed = 0;     // C is known to be zero already: skip the memset a split-K launch needs
    int x3 = 0;           // error-compensated 3xTF32 (fp32-class accuracy)
};
int tc_gemm(const TcGemmArgs& a, cudaStream_t s);
// up to 3 problems with the same operand majors in ONE launch (blockIdx.z selects problem / K split)
int tc_gemm_group(const TcGemmArgs* args, int count, cudaStream_t s);

// One LSTM cell: gates = U Wih^T + Hprev Whh^T + bih + bhh, then the point-wise cell,
// all in one kernel (recurrent.py:30).  gates receives the ACTIVATED i,f,g,o.
struct TcLstmArgs {
    TcOperand U;       // [M, Kin]
    TcOperand Hprev;   // [M, n]
    const float* Wih;  // [4n, Kin]
    const float* Whh;  // [4n, n]
    const float* Wih_lo = nullptr;  // optional pre-split low-order parts of the weights
    const float* Whh_lo = nullptr;
    float* h_new_lo = nullptr;      // optional output: low-order part of h_new
    const float* bih;
    const float* bhh;
    const float* c_prev;  // [M, n]
    float* c_new;
    float* h_new;
    float* gates;  // [M, 4n]
    int M, Kin, n;
    int x3 = 0;
};
// shape part of tc_lstm_supported (the engine's workspace slices are aligned whenever this holds)
bool tc_lstm_shapes_ok(int Kin, int n);
bool tc_lstm_supported(const TcLstmArgs& a);
// The tile configuration tc_lstm_pair launches for M rows and hidden sizes n0 / n1 (host only; also
// what marlc_engine_plan reports): HU hidden units x 4 gates = BN columns per CTA, fat stages of KS
// 32-float K sub-blocks, K split over `ksplit` CTAs (a cluster); `tail_rows` rows in the last 128-row tile.
struct TcLstmPlan { int hu, bn, fat, ks, ksplit, tail_rows; };
TcLstmPlan tc_lstm_plan(int M, int n0, int n1, bool x3);
int tc_lstm_pair(const TcLstmArgs& belief, const TcLstmArgs& action, cudaStream_t s);

}  // namespace marlc

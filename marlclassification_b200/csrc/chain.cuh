// Fused per-step "chain" kernels (chain.cu): the small row-local networks of one
// rollout step collapsed into a few launches, because at the reference's batch
// sizes (M = Na*Nb = 128 rows) the step is bound by launch / dependency latency,
// not by FLOPs or bytes (profiles/: ~1.9 us per dependent graph node on B200).
#pragma once
#include "cnn_device.cuh"
#include "kernels.cuh"

namespace marlc {

// Linear (+ optional LayerNorm affine) parameters; grads used by the backward chains
struct ChainLin {
    const float* W;   // [n_out, n_in]
    const float* b;   // [n_out]
    const float* g;   // LN gamma [n_out] (nullptr: no norm)
    const float* be;  // LN beta
    float* dW;        // gradients (backward chains only; dW itself is done by batched GEMMs)
    float* db;
    float* dg;
    float* dbe;
    int n_in, n_out;
};

// ---- forward, before the LSTM: CNN (one CTA per window) | message mean + decoder + position features
struct StepPreArgs {
    CnnFwdArgs cnn;
    const float* msg_in;  // [Na,Nb,n_m] messages produced at the previous step
    float* coll;          // [M,n_m]   saved
    ChainLin d0, d3;      // decode_msg.{0,1} and .{3,4}
    float* dec_y1;        // [M,2n_m]  pre-norm, saved
    float* dec_s1;        // [M,2n_m]  saved
    float* dec_y2;        // [M,n_m_o] pre-norm, saved
    const float* npos;    // [M,2]
    ChainLin pos;         // map_pos.{0,1}
    float* pos_y;         // [M,n_d] pre-norm, saved
    float* U;             // [M,ldu]: decoder output at column F, position features at F+n_m_o
    float* U_lo = nullptr;  // optional [M,ldu]: tf32_lo(U) (pre-split 3xTF32 operand of the LSTM GEMM)
    long ldu;
    int F, Na, Nb, M;
};
int step_pre(const StepPreArgs& a, cudaStream_t s);

// ---- forward, after the LSTM and the two block-0 GEMMs: policy tail + action | encoder tail
struct StepPostArgs {
    PolicyActArgs act;    // act.s1 is OUTPUT here (pol_s1, saved); input is pol_y1
    const float* pol_y1;  // [M,nl_a] pre-norm
    const float* pol_g;   // policy.1 affine
    const float* pol_be;
    const float* enc_y1;  // [M,2n_m] pre-norm
    const float* enc_g;   // encode_msg.1 affine
    const float* enc_be;
    float* enc_s1;        // [M,2n_m] saved
    ChainLin e3;          // encode_msg.{3,4}
    float* enc_y2;        // [M,n_m] pre-norm, saved
    float* msg_out;       // [M,n_m]
    int M;
};
int step_post(const StepPostArgs& a, cudaStream_t s);

// ---- backward sweep, part 1 (step t): adjoint message mean + encoder backward + dh accumulation
//      + point-wise backward of both LSTM cells
struct BwdPreArgs {
    const float* dcoll;   // [M,n_m] from step t+1's decoder backward (nullptr at t = T-1)
    const float* dmsg = nullptr;  // [M,n_m] gradient of the emitted message itself (a stand-alone step's d msg');
                                  // when set, used instead of the adjoint mean of dcoll
    ChainLin e0, e3;      // encode_msg blocks (with gradient pointers)
    const float* enc_y1;  // saved forward values of step t
    const float* enc_y2;
    float* d_enc_y1;      // [M,2n_m] out (kept for the batched dW)
    float* d_enc_y2;      // [M,n_m]  out
    // LSTM cells: k = 0 belief, 1 action
    const float* dh_carry[2];   // dgates(t+1) Whh          (zero at t = T-1)
    const float* dh_heads[2];   // head gradients at step t
    const float* dc_next[2];
    const float* gates[2];
    const float* c_prev[2];
    const float* c_new[2];
    float* dgates[2];
    float* dgates_lo[2] = {nullptr, nullptr};  // optional tf32_lo(dgates)
    float* dc_prev[2];
    int n[2];
    int Na, Nb, M, n_m;
};
int bwd_pre(const BwdPreArgs& a, cudaStream_t s);

// ---- backward sweep, part 2 (step t): decoder backward from du_t -> dcoll
struct BwdPostArgs {
    const float* dU;      // [M,ldu], decoder slice at column F
    long ldu;
    int F;
    ChainLin d0, d3;
    const float* dec_y1;
    const float* dec_y2;
    float* d_dec_y1;      // [M,2n_m] out (kept for the batched dW)
    float* d_dec_y2;      // [M,n_m_o] out
    float* dcoll;         // [M,n_m] out (nullptr at t = 0: the first message is the constant zero)
    int M, n_m, n_m_o;
};
int bwd_post(const BwdPostArgs& a, cudaStream_t s);

// ---- host-side launch plans: the launchers above and marlc_engine_plan call the same functions
struct CnnWidePlan;
// Feature-extractor role of step_pre for M windows: the wide extractor (cnn_wide.cuh) in cnn_blocks persistent CTAs,
// nw windows per batch, or (cnn_blocks == 0) one CTA per window.  `wide` (optional) receives the wide layout.
struct StepPrePlan { int nw, cnn_blocks; };
StepPrePlan step_pre_plan(const CnnDesc& d, bool have_img, bool have_wT, int M, CnnWidePlan* wide = nullptr);
// Shared memory of one chain launcher: row-buffer width and floats of weights staged per CTA (0: the weights are
// read through L1 / L2).
struct ChainStage { int maxw, wfl; };
ChainStage step_pre_stage(int n_m, int n1, int n2, int nd);
ChainStage step_post_stage(int n1, int n2);
ChainStage bwd_pre_stage(int n_m, int n1, int nb);
ChainStage bwd_post_stage(int n_m, int n1, int n2);

}  // namespace marlc

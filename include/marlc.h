/* libmarlc -- B200 (sm_100a) kernels for the MARLClassification hot path.
 *
 * C ABI: plain pointers and sizes, no torch types.  All pointers are DEVICE
 * pointers unless stated; `stream` is a cudaStream_t passed as void*.  Every
 * function is asynchronous on `stream`, never allocates or synchronises (so it
 * can be captured in a CUDA graph), returns 0 on success and non-zero on a
 * host-side argument / launch error (message via marlc_last_error()).
 *
 * Each entry point names the reference interface it replaces (paths relative to
 * marl_classification/ in Ipsedo/MARLClassification).
 */
#ifndef MARLC_H
#define MARLC_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define MARLC_MAX_ACTIONS 16
#define MARLC_MAX_CNN_LAYERS 6

int marlc_version(void);
const char* marlc_last_error(void);
/* Host-only self-test of the reciprocal division used for index math in the element-wise kernels
 * (no reference counterpart; no GPU needed).  Returns the number of inexact quotients found over
 * divisors 1..d_max and dividends 0, stride, 2*stride, ... up to the launchers' exactness bound. */
long marlc_selftest_fastdiv(int d_max, int stride);

/* ---- Environment operators (core/environment.py) -------------------------- */

/* Environment.observe / __observation, environment.py:47-54,96-126.
 * obs[a,b,c,i,j] = img[b,c,pos[a,b,0]+i,pos[a,b,1]+j]; img f32[B,C,H,W],
 * pos i64[Na,B,2], obs f32[Na,B,C,f,f]. */
int marlc_patch_gather(const float* img, const int64_t* pos, float* obs, int Na, int B, int C, int H, int W, int f,
                       void* stream);
/* Backward of marlc_patch_gather (the adjoint of the window gather): overwrites d_img f32[B,C,H,W], every
 * element, with d_img[b,c,y,x] = sum over a = 0..Na-1 whose window covers (y,x), in that order, of
 * d_obs[a,b,c,y-pos[a,b,0],x-pos[a,b,1]]; d_obs f32[Na,B,C,f,f], pos as for marlc_patch_gather.  Pixels no
 * window covers get 0.  Each pixel sums in fp32 from 0 in agent order: deterministic, the same bits as that
 * sequential loop.  Neither allocates nor synchronises (capturable). */
int marlc_patch_gather_backward(const float* d_obs, const int64_t* pos, float* d_img, int Na, int B, int C, int H,
                                int W, int f, void* stream);

/* Environment.step / __transition, environment.py:56-66,128-150 (+ the
 * normalized_positions property, 74-81).  pos i64[Na*B,2] updated in place;
 * act i64[Na*B] indices into table i64[nA,2]; norm_pos f32[Na*B,2] or NULL;
 * err_flag (int, device, or NULL) is set to 1 if an action index is out of range. */
int marlc_transition(int64_t* pos, const int64_t* act, const int64_t* table, int nA, int M, int f, int H, int W,
                     float* norm_pos, int* err_flag, void* stream);

/* Environment.normalized_positions, environment.py:74-81. */
int marlc_normalized_positions(const int64_t* pos, float* out, int M, int H, int W, void* stream);

/* Input pipeline, device side: what torchvision's ToTensor does on the host in the reference
 * (registry.py:56-57, applied per image by the DataLoader workers of train.py:91-107):
 * uint8 pixels -> fp32 / 255, NCHW.  src is u8[B,H,W,C] (PIL order) when src_hwc != 0, else
 * u8[B,C,H,W]; dst is f32[B,C,H,W].  Bit-identical to ToTensor. */
int marlc_images_u8_to_f32(const uint8_t* src, float* dst, int B, int C, int H, int W, int src_hwc, void* stream);

/* ---- building blocks, exposed for unit parity tests ------------------------ */

/* nn.Linear forward: Y[M,N] = X[M,K] W[N,K]^T + bias (bias may be NULL). */
int marlc_linear(const float* X, const float* W, const float* bias, float* Y, int M, int N, int K, void* stream);
/* Linear -> LayerNorm -> SiLU tail (message.py:26-33 ...): S = SiLU(LN(Y)). */
int marlc_ln_silu(const float* Y, const float* gamma, const float* beta, float* S, int R, int N, void* stream);
/* aggregate_messages, message.py:5-17. msg/out f32[Na,Nb,n]. */
int marlc_msg_mean(const float* msg, float* out, int Na, int Nb, int n, void* stream);

/* tcgen05 TF32 GEMM (TMA-fed, TMEM accumulators): C[M,N] (+)= A B^T (+ A2 B2^T) (+ bias).
 * K-major operand: [M|N rows][K contiguous]; MN-major (a_mn/b_mn != 0): [K rows][M|N
 * contiguous].  Pointers 16-byte aligned, leading dimensions multiples of 4.  This is
 * the kernel behind nn.Linear / nn.LSTMCell forward (recurrent.py:30) and their
 * input / weight gradients.  x3 != 0: error-compensated 3xTF32 (operands split into hi + lo
 * tiles in shared memory, three MMAs per K step): fp32-class accuracy. */
int marlc_tc_gemm(const float* A, int64_t lda, int a_mn, const float* B, int64_t ldb, int b_mn, const float* A2,
                  int64_t lda2, const float* B2, int64_t ldb2, int K2, const float* bias, float* C, int64_t ldc,
                  int M, int N, int K, int accumulate, int allow_split, int x3, void* stream);

/* Both LSTM cells of one step (belief + action, models.py:107-123; nn.LSTMCell,
 * recurrent.py:30) in ONE tcgen05 launch with the cell non-linearities fused into the
 * epilogue.  Arrays of 2 device pointers (HOST arrays): index 0 = belief, 1 = action.
 * u f32[M,Kin]; h_prev/c_prev f32[M,n]; w_ih f32[4n,Kin]; w_hh f32[4n,n]; b_* f32[4n];
 * outputs c_new/h_new f32[M,n], gates f32[M,4n] (activated i,f,g,o, kept for backward).
 * Needs Kin % 4 == 0 and n % 8 == 0. */
int marlc_tc_lstm_pair(const float* u, int M, int Kin, int n, const float* const* h_prev, const float* const* c_prev,
                       const float* const* w_ih, const float* const* w_hh, const float* const* b_ih,
                       const float* const* b_hh, float* const* c_new, float* const* h_new, float* const* gates,
                       int x3, void* stream);

/* Error-compensated 3xTF32 with PRE-SPLIT operands (what the episode engine runs per step): every
 * operand comes with its low-order part lo = x - trunc_tf32(x) in a second array of the same
 * layout, produced by marlc_split_lo (weights, once per forward) or by the kernel that wrote the
 * operand (h_new_lo here).  The tensor core then needs no in-kernel splitting pass. */
int marlc_split_lo(const float* x, float* lo, int64_t n, void* stream);
int marlc_tc_lstm_pair_presplit(const float* u, const float* u_lo, int M, int Kin, int n, const float* const* h_prev,
                                const float* const* h_prev_lo, const float* const* c_prev, const float* const* w_ih,
                                const float* const* w_ih_lo, const float* const* w_hh, const float* const* w_hh_lo,
                                const float* const* b_ih, const float* const* b_hh, float* const* c_new,
                                float* const* h_new, float* const* h_new_lo, float* const* gates, void* stream);

/* _Generic2dCnnModule.forward, vision.py:47-49: k x [conv3x3 s2 p1 -> GroupNorm ->
 * SiLU] -> flatten on N stand-alone windows patch f32[N,img_c,f,f] (the first
 * cin[0] channels are read) -> out f32[N, cout[k-1]*h_k^2].  w/b/gn_w/gn_b are
 * HOST arrays of `layers` device pointers. */
int marlc_cnn_forward(int layers, const int* cin, const int* cout, const int* groups, int f, int img_c,
                      const float* const* w, const float* const* b, const float* const* gn_w,
                      const float* const* gn_b, const float* patch, float* out, int N, void* stream);

/* ---- the episode engine ---------------------------------------------------- */

typedef struct marlc_config {
    /* episode geometry (episode.py:23-30, environment.py:14-21) */
    int na, nb, T, C, H, W, f;
    int n_actions;
    int actions[MARLC_MAX_ACTIONS][2];
    /* feature extractor (vision.py:23-113) */
    int cnn_layers;
    int cnn_cin[MARLC_MAX_CNN_LAYERS], cnn_cout[MARLC_MAX_CNN_LAYERS], cnn_groups[MARLC_MAX_CNN_LAYERS];
    /* widths (models.py:37-76) */
    int n_b, n_a, n_m, n_m_o, n_d, nl_b, nl_a, nb_class;
    float gamma;     /* trainer.py:35 */
    int use_tc;      /* GEMM arithmetic: 0 = exact fp32 FFMA everywhere; 1 = tcgen05 TF32; 2 = tcgen05 3xTF32
                        (error-compensated, fp32-class accuracy) where shapes allow */
    int use_chains;  /* 1: fused per-step chain kernels (4 launches fwd / 3 bwd per step), 0: one kernel per op */
} marlc_config;

typedef struct marlc_engine marlc_engine;

int marlc_engine_create(const marlc_config* cfg, marlc_engine** out);
void marlc_engine_destroy(marlc_engine* e);

/* What the engine's launchers choose for its geometry (per step: M = na*nb rows).  Host only: works on an
 * engine that is created but not bound, and no GPU is needed.  The launchers decide with the same functions. */
typedef struct marlc_plan {
    /* feature-extractor forward */
    int cnn_wide;       /* 1: persistent CTAs with stationary weights, batches of cnn_nw windows; 0: one CTA per window */
    int cnn_nw;         /* windows per batch (1 per window) */
    int cnn_batches;    /* ceil(M / cnn_nw) */
    int cnn_ctas;       /* CTAs of the feature-extractor role */
    int cnn_passes;     /* batches of the busiest CTA: ceil(cnn_batches / cnn_ctas) */
    int cnn_tail;       /* windows in the last batch */
    /* both LSTM cells of a step */
    int lstm_tc;        /* 1: one fused tensor-core launch; 0: FFMA gate GEMMs + point-wise cell (the fields below are 0) */
    int lstm_hu;        /* hidden units per CTA (x 4 gates = lstm_bn output columns) */
    int lstm_bn;
    int lstm_fat;       /* 1: fat pipeline stages (latency-bound launch) */
    int lstm_ks;        /* 32-float K sub-blocks per stage */
    int lstm_ksplit;    /* CTAs that split K (2: cluster pair with a shared-memory reduction) */
    int lstm_tail_rows; /* rows in the last 128-row tile */
    /* backward */
    int sweep_chained;  /* 1: BPTT sweep with the fused chain kernels; 0: one kernel per op */
    /* chain kernels (0 when use_chains == 0): weights staged in shared memory per CTA */
    int staged_step_pre, staged_step_post, staged_bwd_pre, staged_bwd_post;
} marlc_plan;
int marlc_engine_plan(const marlc_engine* e, marlc_plan* out);

/* Flat parameter layout (reference state_dict names, models.py:55-76). */
int marlc_engine_param_count(const marlc_engine* e);
/* name buffer >= 128 bytes; shape has 4 entries (unused = 1); offset in floats. */
int marlc_engine_param_info(const marlc_engine* e, int idx, char* name, int64_t* offset, int* ndim, int64_t* shape);
int64_t marlc_engine_param_floats(const marlc_engine* e); /* size of the flat buffer, floats */

/* Workspace: one caller-allocated, ZERO-INITIALISED device buffer; named views inside it. */
size_t marlc_engine_workspace_bytes(const marlc_engine* e);
int marlc_engine_bind(marlc_engine* e, void* workspace, float* params, float* grads);
int marlc_engine_buffer(const marlc_engine* e, const char* name, size_t* offset, size_t* nbytes);

/* EpisodeSampler.run_episode, episode.py:32-85 (+ agent.py:40-68, models.py:78-138,
 * environment.py:23-68).  img f32[nb,C,H,W].  Injection (all nullable): pos0
 * i64[na,nb,2]; hidden0[k] f32[na,nb,n] for h,c,h^,c^; actions i64[T,na,nb].
 * Results land in the workspace buffers step_preds / step_log_probas /
 * step_values / step_pos (+ everything backward needs). */
int marlc_episode_forward(marlc_engine* e, const float* img, const int64_t* pos0, const float* const* hidden0,
                          const int64_t* actions, void* stream);
/* ModelsWrapper.forward, models.py:78-138: one step of every network on caller
 * tensors: patch f32[na,nb,C,f,f], msg f32[na,nb,n_m], npos f32[na,nb,2],
 * hidden[k] f32[na,nb,n].  Results in workspace slot 0/1: probs, step_values,
 * step_preds (first na*nb rows), msg[1], H[1], Cb[1], Hc[1], Cc[1]. */
int marlc_model_step(marlc_engine* e, const float* patch, const float* msg, const float* npos,
                     const float* const* hidden, void* stream);
/* Re-seed the on-device Philox stream used when nothing is injected. */
int marlc_engine_seed(marlc_engine* e, uint64_t seed, void* stream);

/* Trainer loss block, trainer.py:75-111.  Phase A leaves {sum, sumsq, n} of the
 * advantages in buffer "loss_stats" (3 doubles) for an optional cross-rank
 * all-reduce; phase B writes d_preds / d_logp / d_values and "loss_out"
 * (loss, path, error, actor, critic). targets i64[nb]. */
int marlc_loss_phase_a(marlc_engine* e, const int64_t* targets, void* stream);
int marlc_loss_phase_b(marlc_engine* e, void* stream);

/* loss.backward(), trainer.py:115: BPTT from d_preds / d_logp / d_values (workspace
 * buffers; written by phase B or by the caller) into the flat grads buffer
 * (zeroed first unless accumulate != 0). img must be the forward's batch. */
int marlc_episode_backward(marlc_engine* e, const float* img, int accumulate, void* stream);

/* Gradient on the image batch of the engine's last rollout: overwrites d_img (f32 [nb, C, H, W], every
 * element) with d(whatever the last marlc_episode_backward was seeded with) / d img.  Only the T observations
 * the networks consumed count; pixels no window covers and channels the feature extractor does not read are
 * 0.  Call it after marlc_episode_backward, on the same stream and before the parameters change (the first
 * conv layer's weights are read here).  Deterministic; neither allocates nor synchronises (capturable).
 * Fails when there was no complete episode backward since the last marlc_episode_forward /
 * marlc_model_step, after marlc_model_step_backward, or after a backward cut short by
 * marlc_engine_debug_stop. */
int marlc_episode_image_grad(marlc_engine* e, float* d_img, void* stream);

/* Backward of marlc_model_step on a T = 1 engine (the step-wise API in training).  patch / msg / npos /
 * hidden are the inputs that were given to marlc_model_step; the step is re-run from them first (the
 * workspace is shared by every step-wise call of the geometry).  d_out[8], each nullable (= zero):
 * gradients on probs, values, preds, msg', h', c', h^', c^'.  d_in[5], each nullable (= not wanted):
 * receive the gradients on msg, h, c, h^, c^.  grads: marlc_engine_param_floats floats, overwritten with
 * the parameter gradients (the engine's bound grads buffer is left untouched). */
int marlc_model_step_backward(marlc_engine* e, const float* patch, const float* msg, const float* npos,
                              const float* const* hidden, const float* const* d_out, float* const* d_in,
                              float* grads, void* stream);

/* Gradients on the window and position inputs of the last marlc_model_step_backward (the step-wise API with
 * input gradients): d_patch f32[na,nb,C,f,f] (0 in the channels the feature extractor does not read) and
 * d_npos f32[na,nb,2], each nullable (= not wanted), at least one non-null; both overwritten.  Call it after
 * marlc_model_step_backward, on the same stream and before the parameters change (the first conv layer's and
 * map_pos.0's weights are read here).  Deterministic; neither allocates nor synchronises (capturable).  Fails
 * when there was no complete marlc_model_step_backward since the last marlc_episode_forward / marlc_model_step
 * / marlc_episode_backward, or after a backward cut short by marlc_engine_debug_stop. */
int marlc_model_step_input_grad(marlc_engine* e, float* d_patch, float* d_npos, void* stream);

/* optim.step(), trainer.py:33,116: torch.optim.Adam semantics (no weight decay,
 * no amsgrad) over the flat bucket; g is multiplied by grad_scale first (1/world
 * under data parallelism).  `step` is a device int64 counter, incremented here. */
int marlc_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n, float lr,
                    float beta1, float beta2, float eps, float grad_scale, int64_t* step, void* stream);

/* Profiling aid: make marlc_episode_backward return after the head backward (1) or after the
 * BPTT sweep (2); 0 restores the full backward.  Not for production use. */
int marlc_engine_debug_stop(marlc_engine* e, int phase);

/* Number of kernels the last forward/backward call launched (for bench accounting). */
int marlc_engine_last_launches(const marlc_engine* e);
/* Launch counters of the two GEMM back ends since library load (no reference counterpart): launches of the
 * tcgen05 kernel and of the exact-fp32 FFMA kernel.  Tests use the difference around a call to assert WHICH
 * path a shape took (e.g. hidden_size_linear_action = 758: row pitch not TMA-addressable -> FFMA on purpose). */
long marlc_gemm_launch_count(int ffma);

#ifdef __cplusplus
}
#endif
#endif /* MARLC_H */

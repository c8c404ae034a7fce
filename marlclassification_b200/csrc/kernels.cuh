// Internal launcher declarations for the environment / CNN / loss kernels.
#pragma once
#include "common.cuh"

namespace marlc {

// ---- env.cu -------------------------------------------------------------------
int patch_gather_i64(const float* img, const int64_t* pos, float* obs, int Na, int B, int C, int H, int W, int f,
                     cudaStream_t s);
int patch_gather_i32(const float* img, const int* pos, float* obs, int Na, int B, int C, int H, int W, int f,
                     cudaStream_t s);
int transition_i64(int64_t* pos, const int64_t* act, const int64_t* table, int nA, int M, int f, int H, int W,
                   float* npos, int* err, cudaStream_t s);
int normalized_positions_i64(const int64_t* pos, float* out, int M, int H, int W, cudaStream_t s);
// Adjoint of patch_gather_i64: d_img[b,c,y,x] = sum over a = 0..Na-1 whose window covers (y,x), in that order, of
// d_obs[a,b,c,y-pos_y,x-pos_x]; every element of d_img written.
int patch_gather_backward_i64(const float* d_obs, const int64_t* pos, float* d_img, int Na, int B, int C, int H, int W,
                              int f, cudaStream_t s);

struct EpisodeInitArgs {
    const int64_t* pos0;       // nullable: injected initial positions [M,2]
    const float* hidden0[4];   // nullable each: injected h, c, h^, c^
    const uint64_t* rng_state; // device {seed, episode counter}
    int* pos;                  // out [M,2] int32
    float* npos;               // out [M,2]
    float* hidden[4];          // out
    float* msg0;               // out [M,n_m] zeros
    int width[4];
    int M, n_m, H, W, f;
};
int episode_init(const EpisodeInitArgs& a, cudaStream_t s);
int rng_advance(uint64_t* rng_state, cudaStream_t s);

struct PolicyActArgs {
    const float* s1;     // [M,nl] post LN-SiLU of policy block 0
    const float* W3;     // [nA,nl]
    const float* b3;     // [nA]
    const int64_t* act_in;  // nullable: injected actions [M]
    const uint64_t* rng_state;
    const int* pos_in;   // [M,2]
    float* probs;        // [M,nA]
    float* logp;         // [M]
    int* act_out;        // [M]
    int* pos_out;        // [M,2]
    int64_t* step_pos;   // [M,2] (API output, int64)
    float* npos_out;     // [M,2]
    int moves[32];       // action table, [nA][2]
    int M, nl, nA, t, f, H, W;
};
int policy_act(const PolicyActArgs& a, cudaStream_t s);

// ---- cnn.cu -------------------------------------------------------------------
constexpr int MAX_CNN_LAYERS = 6;
struct CnnDesc {
    int L;
    int cin[MAX_CNN_LAYERS], cout[MAX_CNN_LAYERS], groups[MAX_CNN_LAYERS];
    int hin[MAX_CNN_LAYERS], hout[MAX_CNN_LAYERS];  // square maps
    int f;         // input window
    int img_c;     // channels of the image batch (>= cin[0]; MnistCnn reads channel 0 only)
    int out_size;  // cout[L-1] * hout[L-1]^2
    // parameter pointers
    const float* w[MAX_CNN_LAYERS];
    const float* b[MAX_CNN_LAYERS];
    const float* gn_w[MAX_CNN_LAYERS];
    const float* gn_b[MAX_CNN_LAYERS];
    // optional: conv weights transposed to [cin*9][cout] (output channel contiguous), refreshed by the
    // engine once per forward; enables the register-tiled forward block (cnn_device.cuh)
    const float* wT[MAX_CNN_LAYERS];
};
// Fused gather + CNN forward for M windows.  If `patch` is non-null the windows
// are read from it ([M, img_c, f, f]) instead of gathered from `img` by `pos`.
// y_save[l] (nullable) receives the pre-norm conv outputs for backward.
int cnn_fwd(const CnnDesc& d, const float* img, const int* pos, const float* patch, int B, int H, int W, int M,
            float* const* y_save, float* out, long ldo, cudaStream_t s);

struct CnnBwdBuffers {
    float* dY[MAX_CNN_LAYERS];      // [P*hout^2, cout]  conv-output grads (row = window x output position)
    float* col[MAX_CNN_LAYERS];     // [P*hout^2, cin*9] im2col of the layer input
    float* gnpart[MAX_CNN_LAYERS];  // [P, 2*cout] per-window partial sums for dgamma | dbeta
};
// Where the feature-extractor backward reads its input windows: gathered from the image batch at the
// episode's positions (window p = image (p % M) % B at pos_hist[p]), or, when `patch` is set, the caller's
// [P, img_c, f, f] windows of a stand-alone step (only the first cin[0] channels are read either way).
struct CnnWindows {
    const float* img;
    const int* pos_hist;
    const float* patch;
    int M, B, img_c, H, W, f;
};
// Pixel (c, y, x) of window p is origin[c * chan + y * row + x].
template <bool PATCH>
__device__ __forceinline__ const float* cnn_window(const CnnWindows& w, int p, long& chan, int& row) {
    if (PATCH) {
        chan = (long)w.f * w.f;
        row = w.f;
        return w.patch + (long)p * w.img_c * chan;
    }
    chan = (long)w.H * w.W;
    row = w.W;
    return w.img + (long)((p % w.M) % w.B) * w.img_c * chan + (long)w.pos_hist[2 * (long)p] * w.W +
           w.pos_hist[2 * (long)p + 1];
}
// Backward through the CNN for windows p0 .. p0+P-1 of the T*M stack: reads the input windows,
// recomputes the activations from y_save, writes dY / col / gnpart rows of those windows.  All
// buffer pointers are for window 0.
int cnn_bwd(const CnnDesc& d, const CnnWindows& win, int p0, int P, const float* const* y_save, const float* dOut,
            long lddo, const CnnBwdBuffers& buf, cudaStream_t s);

int cnn_weights_transpose(const CnnDesc& d, float* const* wT, cudaStream_t s);

// ---- cnn_bwd2.cu: layer-wise, batched backward (conv products on the tensor cores) ------------
struct CnnBwdLayerArgs {
    int cout, ho, groups;   // this layer's output is [cout][ho*ho] per window
    int P;                  // number of windows (T*M)
    const float* Y;         // [P, cout*ho*ho] saved pre-norm conv outputs
    const float* gn_w;      // GroupNorm affine
    const float* gn_b;
    const float* dOut;      // top layer: gradient rows [P, lddo] in (c, pos) order; else nullptr
    long lddo;
    const float* dColNext;  // other layers: dCol of layer l+1, [P*ho_next^2, cout*9]
    int ho_next;
    float* dY;              // out [P*ho*ho, cout]
    float* gnpart;          // out [P, 2*cout] per-window GroupNorm affine partials, or nullptr when the
                            // three gradients below are accumulated by the kernel itself
    float* d_gn_w;          // += sum over windows (atomicAdd, one per channel per CTA)
    float* d_gn_b;
    float* d_conv_b;        // += sum over windows and positions of dY
    float* colNext;         // out im2col of this layer's activation for layer l+1 (nullptr for the top layer)
};
int cnn_bwd_layer(const CnnBwdLayerArgs& a, cudaStream_t s);
// The host-side checks of cnn_bwd_layer alone (accumulation targets, shared memory): nothing is launched.
int cnn_bwd_layer_check(const CnnBwdLayerArgs& a);
int cnn_im2col_input(const CnnWindows& win, float* col, int P, int cin, int ho, cudaStream_t s);
// Gradient on the image batch from the first layer's conv-output gradients of all T*M windows: the transposed
// convolution with W_0 fused with the adjoint of the window gather (a pixel sums every window covering it).
struct ImageGradArgs {
    const float* dY0;     // [T*M windows][ho*ho][cout] (cnn_dY0; window p = t*M + a*B + b)
    const float* w0;      // [cout][cin][3][3]
    const int* pos_hist;  // [T][M][2] window corners (row, column) of the observations the networks consumed
    float* d_img;         // out [B][C][H][W], every element written
    int T, Na, B, C, H, W, f, cin, cout, ho;
};
int cnn_image_grad(const ImageGradArgs& a, cudaStream_t s);
// Gradient on the M windows of one stand-alone step from their first-layer conv-output gradients: the
// transposed convolution with W_0, window by window (no gather).
struct PatchGradArgs {
    const float* dY0;  // [M windows][ho*ho][cout] (cnn_dY0 of a T = 1 engine)
    const float* w0;   // [cout][cin][3][3]
    float* d_patch;    // out [M][C][f][f], every element written (0 in the channels c >= cin)
    int M, C, f, cin, cout, ho;
};
int cnn_patch_grad(const PatchGradArgs& a, cudaStream_t s);
// The host-side checks of cnn_patch_grad alone (pointers, shapes, shared memory): nothing is launched.
int cnn_patch_grad_check(const PatchGradArgs& a);

// ---- loss.cu ------------------------------------------------------------------
struct LossArgs {
    const float* preds;   // [T,Na,Nb,Nc]
    const float* logp;    // [T,Na,Nb]
    const float* values;  // [T,Na,Nb]
    const int64_t* targets;  // [Nb]
    float* rewards;       // scratch [T,M]
    float* returns;       // scratch [T,M]
    float* adv;           // scratch [T,M]
    double* stats;        // [16]: 0 sum(adv) 1 sum(adv^2) 2 count | 4 path 5 error 6 critic 7 loss
    float* d_preds;       // out [T,Na,Nb,Nc]
    float* d_logp;        // out [T,M]
    float* d_values;      // out [T,M]
    float* loss_out;      // out [8] floats: loss, path, error, actor, critic
    int T, Na, Nb, Nc;
    float gamma;
};
int loss_phase_a(const LossArgs& a, cudaStream_t s);  // rewards, returns, advantages, local stats
int loss_phase_b(const LossArgs& a, cudaStream_t s);  // standardise, loss parts, gradients
// policy head: dlogits[r,j] = dlogp[r] * (1[j==a_r] - p[r,j]), or, when d_probs is set (gradients on the
// probabilities of a stand-alone step), the softmax backward dlogits[r,j] = p[r,j] (g[r,j] - sum_a p[r,a] g[r,a])
int policy_logit_grad(const float* d_logp, const float* probs, const int* act, float* dlogits, int R, int nA,
                      cudaStream_t s, const float* d_probs = nullptr);

}  // namespace marlc

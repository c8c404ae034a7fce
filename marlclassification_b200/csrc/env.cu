// Environment kernels: patch gather, integer position transition, normalised
// positions, episode initial state, and the fused policy-head -> sample ->
// log-prob -> transition step (reference: core/environment.py, core/agent.py).
#include <stdlib.h>

#include "common.cuh"
#include "kernels.cuh"

namespace marlc {

// ---------------------------------------------------------------------------
// K1 patch gather (environment.py:96-126):
//   obs[a,b,c,i,j] = img[b,c,pos[a,b,0]+i,pos[a,b,1]+j]
// (The first version staged aligned 128-bit row reads through shared memory, one CTA per window:
// 2.4 TB/s at 65 536 windows.  Two block barriers and the index math per window dominated.)
// ---------------------------------------------------------------------------
// One WARP per window, no shared memory, no block barrier: lane-strided over the contiguous
// C*f*f output (perfectly coalesced 128 B stores); each warp-load covers 32 consecutive output
// elements = 32/f source row segments (coalesced within a segment).  All iterations' loads are
// issued before the first store (UNROLL independent requests per lane) so a window costs about
// one memory round trip.  Measured 2.4 -> see profiles/README.md for the achieved GB/s.
// The three divisions per element (e -> c, i, j) were ~60 of the ~75 instructions per element as
// runtime `/`; FastDiv (common.cuh) + 32-bit offsets + a branch-free tail: 88 -> 45 us at 65 536 windows.
template <typename PosT, int UNROLL, bool FAST>
__global__ void __launch_bounds__(256)
patch_gather_kernel(const float* __restrict__ img, const PosT* __restrict__ pos, float* __restrict__ obs, int Na, int B,
                    int C, int H, int W, int f, FastDiv dff, FastDiv df) {
    const int lane = threadIdx.x & 31;
    // consecutive warps take the agents of ONE image (b-major): an image is then read in a burst
    // while its DRAM pages are open / its sectors are in L2, instead of once per agent row
    const int g = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (g >= Na * B) return;
    const int b = g / Na, m = (g - b * Na) * B + b;  // output row m = a*B + b
    const int py = (int)pos[2 * (long)m], px = (int)pos[2 * (long)m + 1];
    const int ff = f * f, total = C * ff;
    const int plane = H * W;  // offsets inside one image fit 32 bits (host-checked)
    const float* src = img + (long)b * C * plane + (py * W + px);
    float* dst = obs + (long)m * total;
    for (int e0 = lane; e0 < total; e0 += 32 * UNROLL) {
        float v[UNROLL];
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
            // tail lanes re-read the last element instead of branching around the load
            const int e = min(e0 + 32 * u, total - 1);
            const int c = FAST ? dff.div_nz(e) : e / ff;
            const int r = e - c * ff;
            const int i = FAST ? df.div_nz(r) : r / f;
            v[u] = __ldg(src + (c * plane + i * W + (r - i * f)));
        }
#pragma unroll
        for (int u = 0; u < UNROLL; ++u)
            if (e0 + 32 * u < total) dst[e0 + 32 * u] = v[u];
    }
}

template <typename PosT>
static int patch_gather_t(const float* img, const PosT* pos, float* obs, int Na, int B, int C, int H, int W, int f,
                          cudaStream_t s) {
    MARLC_CHECK(f >= 1 && f <= H && f <= W, "patch_gather: window f=%d does not fit %dx%d", f, H, W);
    const int M = Na * B;
    if (M <= 0) return 0;
    const int blocks = (M + 7) / 8;  // 8 warps = 8 windows per CTA
    const long ff = (long)f * f, total = (long)C * ff;
    MARLC_CHECK((long)C * H * W < 0x7fffffffl, "patch_gather: one image must hold fewer than 2^31 elements");
    const bool fast = f >= 2 && FastDiv::exact_up_to(total, ff);
    const FastDiv dff((unsigned)max(ff, 2l)), df((unsigned)max(f, 2));
#define MARLC_GATHER_LAUNCH(U, F) \
    patch_gather_kernel<PosT, U, F><<<blocks, 256, 0, s>>>(img, pos, obs, Na, B, C, H, W, f, dff, df)
    if (total <= 32 * 8) { if (fast) MARLC_GATHER_LAUNCH(8, true); else MARLC_GATHER_LAUNCH(8, false); }
    else { if (fast) MARLC_GATHER_LAUNCH(16, true); else MARLC_GATHER_LAUNCH(16, false); }
#undef MARLC_GATHER_LAUNCH
    MARLC_LAUNCH_CHECK();
    return 0;
}
int patch_gather_i64(const float* img, const int64_t* pos, float* obs, int Na, int B, int C, int H, int W, int f,
                     cudaStream_t s) {
    return patch_gather_t<int64_t>(img, pos, obs, Na, B, C, H, W, f, s);
}
int patch_gather_i32(const float* img, const int* pos, float* obs, int Na, int B, int C, int H, int W, int f,
                     cudaStream_t s) {
    return patch_gather_t<int>(img, pos, obs, Na, B, C, H, W, f, s);
}

// K1' adjoint of the patch gather (the backward of Environment.observe):
//   d_img[b,c,y,x] = sum over agents a = 0..Na-1 whose window covers (y,x), in that order, of
//                    d_obs[a,b,c,y-pos[a,b,0],x-pos[a,b,1]]
// One CTA per (image, 32x16 pixel tile); a warp owns 32 consecutive columns of two rows, so every store of
// d_img (mostly zeros: most pixels are under no window) is one 128-byte line.  The image's windows are tested
// against the tile GB_THREADS at a time and each chunk's overlapping windows are compacted in agent order
// (tile_window_list), so the list cannot overflow whatever Na is.  Each pixel
// sums in registers from 0.0f in agent order: no atomics, and the result is the same bits as a sequential fp32
// loop over the agents.
constexpr int GB_TW = 32, GB_TH = 16, GB_THREADS = 256;
constexpr int GB_PX = GB_TH * GB_TW / GB_THREADS;  // pixels (rows) per thread
constexpr int GB_CB = 4;                            // channels per accumulation pass

// The windows of image b that overlap the pixel tile, in agent order.  Each of the NT threads of the CTA brings
// one candidate window (observation row m, corner wy, wx; valid = false past the last agent); those overlapping
// the TH x TW tile at (y0, x0) are written in thread order to list_m / list_y / list_x, and their number is
// returned to every thread.  At most NT candidates per call, so the list cannot overflow.  Starts with a block
// barrier (the previous chunk's list may be read until then); the caller needs one more before it reads the new
// list.  This is phase 1 of cnn_image_grad_kernel (cnn_bwd2.cu), which keeps its own copy: compiled into that
// kernel, the helper costs an 8-byte spill at its 80-register budget.
template <int NT, int TH, int TW>
__device__ __forceinline__ int tile_window_list(bool valid, int m, int wy, int wx, int f, int y0, int x0, int* list_m,
                                                int* list_y, int* list_x, int* warp_n) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const bool hit = valid && wy < y0 + TH && wy + f > y0 && wx < x0 + TW && wx + f > x0;
    const unsigned bal = __ballot_sync(0xffffffffu, hit);
    __syncthreads();  // the previous chunk's list is consumed
    if (lane == 0) warp_n[warp] = __popc(bal);
    __syncthreads();
    int off = 0, n = 0;
#pragma unroll
    for (int k = 0; k < NT / 32; ++k) {
        const int v = warp_n[k];
        off += k < warp ? v : 0;
        n += v;
    }
    if (hit) {
        const int slot = off + __popc(bal & ((1u << lane) - 1u));
        list_m[slot] = m;
        list_y[slot] = wy;
        list_x[slot] = wx;
    }
    return n;
}

__global__ void __launch_bounds__(GB_THREADS) patch_gather_backward_kernel(const float* __restrict__ d_obs,
                                                                           const int64_t* __restrict__ pos,
                                                                           float* __restrict__ d_img, int Na, int B,
                                                                           int C, int H, int W, int f) {
    __shared__ int list_m[GB_THREADS], list_y[GB_THREADS], list_x[GB_THREADS];
    __shared__ int warp_n[GB_THREADS / 32];
    const int tid = threadIdx.x;
    const int b = blockIdx.z, y0 = blockIdx.y * GB_TH, x0 = blockIdx.x * GB_TW;
    const int px = x0 + (tid & 31);
    int py[GB_PX];
#pragma unroll
    for (int k = 0; k < GB_PX; ++k) py[k] = y0 + (tid >> 5) + k * (GB_THREADS / 32);
    const int ff = f * f, plane = H * W;  // offsets inside one image fit 32 bits (host-checked)
    float* out = d_img + (long)b * C * plane;
    for (int c0 = 0; c0 < C; c0 += GB_CB) {
        float acc[GB_PX][GB_CB];
#pragma unroll
        for (int k = 0; k < GB_PX; ++k)
#pragma unroll
            for (int u = 0; u < GB_CB; ++u) acc[k][u] = 0.f;
        for (int a0 = 0; a0 < Na; a0 += GB_THREADS) {
            const int ag = a0 + tid;
            int m = 0, wy = 0, wx = 0;
            if (ag < Na) {
                m = ag * B + b;  // observation row m = a*B + b
                wy = (int)pos[2 * (long)m];
                wx = (int)pos[2 * (long)m + 1];
            }
            const int n = tile_window_list<GB_THREADS, GB_TH, GB_TW>(ag < Na, m, wy, wx, f, y0, x0, list_m, list_y,
                                                                      list_x, warp_n);
            __syncthreads();  // the list is written
            for (int j = 0; j < n; ++j) {
                const int lx = px - list_x[j];
                if ((unsigned)lx >= (unsigned)f) continue;
                const float* src = d_obs + (long)list_m[j] * C * ff + c0 * ff + lx;
#pragma unroll
                for (int k = 0; k < GB_PX; ++k) {
                    const int ly = py[k] - list_y[j];
                    if ((unsigned)ly >= (unsigned)f) continue;
#pragma unroll
                    for (int u = 0; u < GB_CB; ++u)
                        if (c0 + u < C) acc[k][u] += __ldg(src + u * ff + ly * f);
                }
            }
        }
        if (px < W)
#pragma unroll
            for (int k = 0; k < GB_PX; ++k)
                if (py[k] < H)
#pragma unroll
                    for (int u = 0; u < GB_CB; ++u)
                        if (c0 + u < C) out[(c0 + u) * plane + py[k] * W + px] = acc[k][u];
    }
}

int patch_gather_backward_i64(const float* d_obs, const int64_t* pos, float* d_img, int Na, int B, int C, int H, int W,
                              int f, cudaStream_t s) {
    MARLC_CHECK(f >= 1 && f <= H && f <= W, "patch_gather_backward: window f=%d does not fit %dx%d", f, H, W);
    MARLC_CHECK(Na >= 0 && B >= 0 && C >= 1, "patch_gather_backward: bad shape (Na=%d, B=%d, C=%d)", Na, B, C);
    MARLC_CHECK((long)C * H * W < 0x7fffffffl, "patch_gather_backward: one image must hold fewer than 2^31 elements");
    MARLC_CHECK((long)Na * B < 0x7fffffffl, "patch_gather_backward: %d x %d windows", Na, B);
    if (B == 0) return 0;
    const unsigned tx = (W + GB_TW - 1) / GB_TW, ty = (H + GB_TH - 1) / GB_TH;
    MARLC_CHECK(ty <= 65535 && B <= 65535, "patch_gather_backward: image batch %d x %d rows too large for the grid", B,
                H);
    patch_gather_backward_kernel<<<dim3(tx, ty, (unsigned)B), GB_THREADS, 0, s>>>(d_obs, pos, d_img, Na, B, C, H, W, f);
    MARLC_LAUNCH_CHECK();
    return 0;
}

// ---------------------------------------------------------------------------
// K2 transition (environment.py:56-66, 128-150) in pure integer arithmetic:
// the move is applied only if every dim stays inside (0 <= p+m, p+m+f < S).
// Also emits normalised positions float(p)/float(S) (environment.py:74-81).
// ---------------------------------------------------------------------------
__device__ __forceinline__ void apply_move(int& py, int& px, int my, int mx, int f, int H, int W) {
    const int ny = py + my, nx = px + mx;
    const bool ok = (ny >= 0) & (ny + f < H) & (nx >= 0) & (nx + f < W);
    if (ok) { py = ny; px = nx; }
}

__global__ void transition_i64_kernel(int64_t* __restrict__ pos, const int64_t* __restrict__ act,
                                      const int64_t* __restrict__ table, int nA, int M, int f, int H, int W,
                                      float* __restrict__ npos, int* __restrict__ err) {
    const int m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= M) return;
    // one 16-byte load / store per agent for the (y, x) pair, 8-byte for the action and the float2
    longlong2 p = reinterpret_cast<const longlong2*>(pos)[m];
    int py = (int)p.x, px = (int)p.y;
    const int64_t a = act[m];
    if (a < 0 || a >= nA) { if (err) atomicExch(err, 1); }
    else apply_move(py, px, (int)__ldg(table + 2 * a), (int)__ldg(table + 2 * a + 1), f, H, W);
    p.x = py; p.y = px;
    reinterpret_cast<longlong2*>(pos)[m] = p;
    if (npos) reinterpret_cast<float2*>(npos)[m] = make_float2((float)py / (float)H, (float)px / (float)W);
}

int transition_i64(int64_t* pos, const int64_t* act, const int64_t* table, int nA, int M, int f, int H, int W,
                   float* npos, int* err, cudaStream_t s) {
    if (M <= 0) return 0;
    MARLC_CHECK(((uintptr_t)pos & 15) == 0 && ((uintptr_t)npos & 7) == 0, "transition: positions must be 16-byte aligned");
    transition_i64_kernel<<<(M + 255) / 256, 256, 0, s>>>(pos, act, table, nA, M, f, H, W, npos, err);
    MARLC_LAUNCH_CHECK();
    return 0;
}

__global__ void normalized_positions_kernel(const int64_t* __restrict__ pos, float* __restrict__ out, int M, int H, int W) {
    const int m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= M) return;
    out[2 * m] = (float)pos[2 * m] / (float)H;
    out[2 * m + 1] = (float)pos[2 * m + 1] / (float)W;
}
int normalized_positions_i64(const int64_t* pos, float* out, int M, int H, int W, cudaStream_t s) {
    if (M <= 0) return 0;
    normalized_positions_kernel<<<(M + 127) / 128, 128, 0, s>>>(pos, out, M, H, W);
    MARLC_LAUNCH_CHECK();
    return 0;
}

// ---------------------------------------------------------------------------
// Episode initial state.  Either copies injected values or draws them:
// positions ~ U{0..S_d-f-1} (environment.py:33-43), recurrent state ~ N(0,1)
// (models.py:148-159).  Random streams are Philox(seed) with the episode
// counter read from device memory so CUDA-graph replays draw fresh numbers.
// ---------------------------------------------------------------------------
__global__ void episode_init_kernel(EpisodeInitArgs a) {
    const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t episode = a.rng_state ? a.rng_state[1] : 0;
    const Philox ph(a.rng_state ? a.rng_state[0] : 0);
    if (idx < a.M) {
        int py, px;
        if (a.pos0) { py = (int)a.pos0[2 * idx]; px = (int)a.pos0[2 * idx + 1]; }
        else {
            uint4 r = ph((uint64_t)idx, (episode << 8) | 1);
            py = (int)(((uint64_t)r.x * (uint64_t)(a.H - a.f)) >> 32);
            px = (int)(((uint64_t)r.y * (uint64_t)(a.W - a.f)) >> 32);
        }
        a.pos[2 * idx] = py; a.pos[2 * idx + 1] = px;
        a.npos[2 * idx] = (float)py / (float)a.H;
        a.npos[2 * idx + 1] = (float)px / (float)a.W;
    }
    // hidden states: 4 tensors, element idx over max size
    for (int k = 0; k < 4; ++k) {
        const long n = (long)a.M * a.width[k];
        if (idx >= n) continue;
        float v;
        if (a.hidden0[k]) v = a.hidden0[k][idx];
        else {
            uint4 r = ph((uint64_t)idx, (episode << 8) | (2 + k));
            // Box-Muller
            float u1 = fmaxf(u01(r.x), 1.0f / 16777216.0f), u2 = u01(r.y);
            v = sqrtf(-2.0f * logf(u1)) * cospif(2.0f * u2);
        }
        a.hidden[k][idx] = v;
    }
    for (long i = idx; i < (long)a.M * a.n_m; i += (long)gridDim.x * blockDim.x) a.msg0[i] = 0.f;
}

int episode_init(const EpisodeInitArgs& a, cudaStream_t s) {
    long n = a.M;
    for (int k = 0; k < 4; ++k) n = max(n, (long)a.M * a.width[k]);
    episode_init_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(a);
    MARLC_LAUNCH_CHECK();
    return 0;
}

__global__ void rng_advance_kernel(uint64_t* rng_state) { rng_state[1] += 1; }
int rng_advance(uint64_t* rng_state, cudaStream_t s) {
    rng_advance_kernel<<<1, 1, 0, s>>>(rng_state);
    MARLC_LAUNCH_CHECK();
    return 0;
}

// ---------------------------------------------------------------------------
// K7 policy tail (policy.py:15-16 + agent.py:51-61 + environment.py:56-66), one
// warp per row: logits = s1 W3^T + b3 -> softmax -> sample (or injected action)
// -> log p[a] -> integer transition -> next normalised position.
// ---------------------------------------------------------------------------
constexpr int MAX_ACTIONS = 16;

__global__ void policy_act_kernel(PolicyActArgs a) {
    const int lane = threadIdx.x & 31;
    const int m = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (m >= a.M) return;
    const float* x = a.s1 + (long)m * a.nl;
    float logit[MAX_ACTIONS];
#pragma unroll 1
    for (int j = 0; j < a.nA; ++j) {
        const float* w = a.W3 + (long)j * a.nl;
        float s = 0.f;
        for (int k = lane; k < a.nl; k += 32) s = fmaf(x[k], w[k], s);
        logit[j] = warp_sum(s) + a.b3[j];
    }
    float mx = -INFINITY;
    for (int j = 0; j < a.nA; ++j) mx = fmaxf(mx, logit[j]);
    float den = 0.f;
    for (int j = 0; j < a.nA; ++j) { logit[j] = expf(logit[j] - mx); den += logit[j]; }
    const float inv = 1.0f / den;
    int act;
    if (a.act_in) act = (int)a.act_in[m];
    else {
        const uint64_t episode = a.rng_state[1];
        const Philox ph(a.rng_state[0]);
        uint4 r = ph((uint64_t)a.t * (uint64_t)a.M + (uint64_t)m, (episode << 8) | 7);
        const float u = u01(r.x);
        float cdf = 0.f;
        act = a.nA - 1;
        for (int j = 0; j < a.nA; ++j) {
            cdf += logit[j] * inv;
            if (u < cdf) { act = j; break; }
        }
    }
    if (lane == 0) {
        float pa = 0.f;
        for (int j = 0; j < a.nA; ++j) {
            const float p = logit[j] * inv;
            a.probs[(long)m * a.nA + j] = p;
            if (j == act) pa = p;
        }
        a.logp[m] = logf(pa);
        a.act_out[m] = act;
        int py = a.pos_in[2 * m], px = a.pos_in[2 * m + 1];
        if (act >= 0 && act < a.nA) apply_move(py, px, a.moves[2 * act], a.moves[2 * act + 1], a.f, a.H, a.W);
        a.pos_out[2 * m] = py; a.pos_out[2 * m + 1] = px;
        a.step_pos[2 * (long)m] = py; a.step_pos[2 * (long)m + 1] = px;
        a.npos_out[2 * m] = (float)py / (float)a.H;
        a.npos_out[2 * m + 1] = (float)px / (float)a.W;
    }
}

int policy_act(const PolicyActArgs& a, cudaStream_t s) {
    MARLC_CHECK(a.nA <= MAX_ACTIONS, "policy_act: nb_action=%d > %d", a.nA, MAX_ACTIONS);
    if (a.M <= 0) return 0;
    policy_act_kernel<<<(a.M * 32 + 127) / 128, 128, 0, s>>>(a);
    MARLC_LAUNCH_CHECK();
    return 0;
}

}  // namespace marlc

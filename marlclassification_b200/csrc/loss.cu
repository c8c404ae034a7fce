// Fused actor-critic loss, forward + gradients w.r.t. the rollout outputs
// (training/trainer.py:75-111, training/functions.py:7-55).
//
// Phase A: per-agent rewards, vote cross-entropy (+ its gradient), discounted
//          returns, advantages and their LOCAL sums (sum, sum of squares, n).
// [data-parallel: the three sums are all-reduced between the phases so that
//  standardize() (functions.py:54-55) sees the global batch]
// Phase B: standardise, path / critic losses and d/dlogp, d/dvalues.
//
// Gradient routing of the reference (SURVEY 3.2): rewards/returns are only used
// detached; values get gradient from the critic loss only; logits only from the
// vote error; log-probs only from the path loss.
#include "kernels.cuh"

namespace marlc {

// warp per (t, m): reward = (ln Nc - CE(pred[t,m,:], y_b)) / ln Nc
__global__ void reward_kernel(const LossArgs a) {
    const int lane = threadIdx.x & 31;
    const long w = ((long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int M = a.Na * a.Nb;
    if (w >= (long)a.T * M) return;
    const int m = (int)(w % M), b = m % a.Nb;
    const float* x = a.preds + w * a.Nc;
    float mx = -INFINITY;
    for (int c = lane; c < a.Nc; c += 32) mx = fmaxf(mx, x[c]);
    mx = warp_max(mx);
    float s = 0.f;
    for (int c = lane; c < a.Nc; c += 32) s += expf(x[c] - mx);
    s = warp_sum(s);
    if (lane == 0) {
        // labels outside [0, Nc) are flagged by vote_kernel; here they are only kept from reading out of bounds
        const long yb = a.targets[b];
        const float ce = (mx + logf(s)) - x[(yb >= 0 && yb < a.Nc) ? yb : 0];
        const float lnc = logf((float)a.Nc);
        a.rewards[w] = (lnc - ce) / lnc;
    }
}

// warp per (t, b): vote = mean_a pred[t,a,b,:]; error = CE(vote, y_b);
// d loss / d pred[t,a,b,c] = (softmax(vote)_c - 1[c == y_b]) / (Na * Nb)
__global__ void vote_kernel(const LossArgs a) {
    const int lane = threadIdx.x & 31;
    const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (w >= a.T * a.Nb) return;
    const int t = w / a.Nb, b = w % a.Nb;
    const long stride = (long)a.Nb * a.Nc;
    const float* base = a.preds + ((long)t * a.Na * a.Nb + b) * a.Nc;
    const float invNa = 1.0f / (float)a.Na;
    auto vote = [&](int c) {
        float v = 0.f;
        for (int ag = 0; ag < a.Na; ++ag) v += base[ag * stride + c];
        return v * invNa;
    };
    float mx = -INFINITY;
    for (int c = lane; c < a.Nc; c += 32) mx = fmaxf(mx, vote(c));
    mx = warp_max(mx);
    float s = 0.f;
    for (int c = lane; c < a.Nc; c += 32) s += expf(vote(c) - mx);
    s = warp_sum(s);
    // a label outside [0, Nc) (e.g. --nb-class smaller than the dataset's class count) is the reference's
    // device assert in cross_entropy (trainer.py:83-87): counted in stats[7], reported as loss_out[5] and
    // turned into a NaN loss by loss_finalize_kernel; the index is clamped so nothing is read out of bounds
    const long y_raw = a.targets[b];
    const bool y_bad = y_raw < 0 || y_raw >= a.Nc;
    const int y = y_bad ? 0 : (int)y_raw;
    if (y_bad && lane == 0 && t == 0) atomicAdd(&a.stats[7], 1.0);
    const float lse = mx + logf(s);
    const float scale = 1.0f / ((float)a.Na * (float)a.Nb);
    float* dbase = a.d_preds + ((long)t * a.Na * a.Nb + b) * a.Nc;
    for (int c = lane; c < a.Nc; c += 32) {
        const float g = (expf(vote(c) - lse) - (c == y ? 1.f : 0.f)) * scale;
        for (int ag = 0; ag < a.Na; ++ag) dbase[ag * stride + c] = g;
    }
    if (lane == 0) atomicAdd(&a.stats[5], (double)(lse - vote(y)));
}

// thread per m: G_t = r_t + gamma G_{t+1} (== functions.py:35-51), adv = G - V.
// Deliberate departure at gamma = 0: the reference's closed form (flip-cumsum-flip of r gamma^t, divided by gamma^t)
// is 0/0 there from t = 1 on, so its returns, losses and gradients are NaN; this recursion gives G_t = r_t, the
// returns that closed form stands for (tests/test_gpu_update.py pins both)
__global__ void returns_kernel(const LossArgs a) {
    const int M = a.Na * a.Nb;
    const int m = blockIdx.x * blockDim.x + threadIdx.x;
    double s1 = 0.0, s2 = 0.0;
    if (m < M) {
        float G = 0.f;
        // 8 steps of operands in flight before the dependent scan touches them: with one load per iteration (the
        // stores to returns / adv may alias, so the compiler cannot hoist it) every step paid an L2 round trip --
        // 17 us for a 16-step scan (launch list, round 2)
        for (int t1 = a.T; t1 > 0; t1 -= 8) {
            float r[8], v[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const int t = t1 - 1 - k;
                r[k] = t >= 0 ? a.rewards[(long)t * M + m] : 0.f;
                v[k] = t >= 0 ? a.values[(long)t * M + m] : 0.f;
            }
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const int t = t1 - 1 - k;
                if (t >= 0) {
                    const long i = (long)t * M + m;
                    G = fmaf(a.gamma, G, r[k]);
                    a.returns[i] = G;
                    const float ad = G - v[k];
                    a.adv[i] = ad;
                    s1 += ad;
                    s2 += (double)ad * ad;
                }
            }
        }
    }
    s1 = warp_sum_d(s1); s2 = warp_sum_d(s2);
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(&a.stats[0], s1);
        atomicAdd(&a.stats[1], s2);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&a.stats[2], (double)a.T * M);
}

int loss_phase_a(const LossArgs& a, cudaStream_t s) {
    const int M = a.Na * a.Nb;
    MARLC_CUDA(cudaMemsetAsync(a.stats, 0, 16 * sizeof(double), s));
    long warps = (long)a.T * M;
    reward_kernel<<<(unsigned)((warps * 32 + 255) / 256), 256, 0, s>>>(a);
    MARLC_LAUNCH_CHECK();
    vote_kernel<<<(a.T * a.Nb * 32 + 255) / 256, 256, 0, s>>>(a);
    MARLC_LAUNCH_CHECK();
    returns_kernel<<<(M + 127) / 128, 128, 0, s>>>(a);
    MARLC_LAUNCH_CHECK();
    return 0;
}

// thread per (t, m)
__global__ void loss_b_kernel(const LossArgs a) {
    const int M = a.Na * a.Nb;
    const long n_local = (long)a.T * M;
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    double path = 0.0, critic = 0.0;
    if (i < n_local) {
        const double n = a.stats[2];
        const double mean = a.stats[0] / n;
        const double var = (a.stats[1] - n * mean * mean) / (n - 1.0);  // unbiased (torch.std default)
        // one advantage in the whole batch (T * Na * Nb == 1): torch.std of one element is NaN, and so is the
        // reference's loss.  The clamp below used to turn that 0/0 into 0 and return a finite loss; the NaN is
        // kept instead, like the bad-label NaN of loss_finalize_kernel (error and critic stay finite, as there)
        const float stdv = n < 2.0 ? __int_as_float(0x7fc00000) : (float)sqrt(var > 0.0 ? var : 0.0);
        const float nadv = (a.adv[i] - (float)mean) / (stdv + 1e-8f);
        const float invM = 1.0f / (float)M;
        path = (double)(-a.logp[i] * nadv);
        a.d_logp[i] = -nadv * invM;
        const float x = a.values[i] - a.returns[i];
        const float ax = fabsf(x);
        critic = (double)(ax < 1.f ? 0.5f * x * x : ax - 0.5f);  // smooth_l1, beta = 1
        a.d_values[i] = (ax < 1.f ? x : (x > 0.f ? 1.f : -1.f)) * invM;
    }
    path = warp_sum_d(path); critic = warp_sum_d(critic);
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(&a.stats[4], path);
        atomicAdd(&a.stats[6], critic);
    }
}

__global__ void loss_finalize_kernel(const LossArgs a) {
    const double M = (double)a.Na * a.Nb;
    const double path = a.stats[4] / M;                 // path_loss.sum(0).mean()
    const double err_sum_t = a.stats[5] / (double)a.Nb; // sum_t mean_b error
    const double critic = a.stats[6] / M;
    a.loss_out[0] = (float)(path + err_sum_t + critic);  // loss (trainer.py:111)
    a.loss_out[1] = (float)path;
    a.loss_out[2] = (float)(a.stats[5] / ((double)a.T * a.Nb));  // error.mean()
    a.loss_out[3] = (float)(path + err_sum_t);           // actor_loss.sum(0).mean()
    a.loss_out[4] = (float)critic;
    a.loss_out[5] = (float)a.stats[7];  // number of images whose label is outside [0, Nc)
    if (a.stats[7] > 0.0)
        for (int i = 0; i < 5; ++i) a.loss_out[i] = __int_as_float(0x7fc00000);  // NaN: never a silently wrong number
}

int loss_phase_b(const LossArgs& a, cudaStream_t s) {
    const long n = (long)a.T * a.Na * a.Nb;
    loss_b_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(a);
    MARLC_LAUNCH_CHECK();
    loss_finalize_kernel<<<1, 1, 0, s>>>(a);
    MARLC_LAUNCH_CHECK();
    return 0;
}

__global__ void policy_logit_grad_kernel(const float* __restrict__ d_logp, const float* __restrict__ probs,
                                         const int* __restrict__ act, const float* __restrict__ d_probs,
                                         float* __restrict__ dlogits, long R, int nA) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= R * nA) return;
    const long r = i / nA;
    const int j = (int)(i % nA);
    if (d_probs) {  // softmax backward; nA <= MAX_ACTIONS, so each thread forms its row's dot product
        const float* p = probs + r * nA;
        const float* g = d_probs + r * nA;
        float dot = 0.f;
        for (int a = 0; a < nA; ++a) dot = fmaf(p[a], g[a], dot);
        dlogits[i] = p[j] * (g[j] - dot);
        return;
    }
    dlogits[i] = d_logp[r] * ((j == act[r] ? 1.f : 0.f) - probs[i]);
}

int policy_logit_grad(const float* d_logp, const float* probs, const int* act, float* dlogits, int R, int nA,
                      cudaStream_t s, const float* d_probs) {
    long n = (long)R * nA;
    if (n <= 0) return 0;
    policy_logit_grad_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(d_logp, probs, act, d_probs, dlogits, R, nA);
    MARLC_LAUNCH_CHECK();
    return 0;
}

}  // namespace marlc

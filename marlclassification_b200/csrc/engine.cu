// Episode engine: flat parameter layout, workspace carving, and the host-side
// orchestration of one rollout (forward), the fused loss and the BPTT sweep.
// This file is the C ABI of libmarlc (see include/marlc.h).
#include <stdarg.h>
#include <string.h>

#include <algorithm>

#include <string>
#include <vector>

#include <nvtx3/nvToolsExt.h>  // header-only NVTX v3: ranges show up in nsys / ncu --nvtx, cost ~nothing otherwise

#include "../../include/marlc.h"
#include "kernels.cuh"
#include "chain.cuh"
#include "tc.cuh"

namespace marlc {

int g_launch_count = 0;
long g_simt_gemm_launches = 0, g_tc_gemm_launches = 0;
static thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
// programmatic dependent launch: state and the MARLC_PDL switch (common.cuh)
thread_local int g_pdl = 0, g_pdl_trig = 0;
bool pdl_enabled() {
    static const bool on = !(getenv("MARLC_PDL") && atoi(getenv("MARLC_PDL")) == 0);
    return on;
}
int pdl_trigger_early() { return g_pdl_trig; }

struct ParamInfo {
    std::string name;
    int64_t offset;  // floats
    int ndim;
    int64_t shape[4];
    int64_t numel;
};
struct BufInfo {
    std::string name;
    size_t offset, bytes;
};

}  // namespace marlc

using namespace marlc;

// NVTX range over a host-side phase of the engine (SURVEY section 5: tracing).  Ranges mark where the
// launches of a phase are ISSUED (under CUDA-graph capture that is capture time; eager runs and
// `ncu --nvtx --nvtx-include "marlc/..."` attribute kernels to phases with them).
struct NvtxRange {
    explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
};

struct marlc_engine {
    marlc_config cfg;
    int M, TM, F, Kin, L;
    CnnDesc cnn;  // dims; pointers filled at bind
    int cnn_sz[MAX_CNN_LAYERS];  // cout*hout^2
    std::vector<ParamInfo> params;
    int64_t param_floats = 0;
    std::vector<BufInfo> bufs;
    size_t ws_bytes = 0;
    char* ws = nullptr;
    float* P = nullptr;
    float* G = nullptr;
    int last_launches = 0;
    // profiling aid (scripts/phase_times.py).  backward: 1 = stop after the heads, 2 = after the sweep,
    // 21 / 22 = sweep with only bwd_pre / bwd_pre + dX GEMMs per step.  forward: 11 / 12 / 13 = per step
    // only step_pre / + LSTM / + block-0 GEMMs, 14 = whole loop without the batched heads.
    int debug_stop = 0;
    // fork/join plumbing for independent branches (works eagerly and under stream capture)
    cudaStream_t side[2] = {nullptr, nullptr};
    cudaStream_t hp = nullptr;  // highest priority: the latency-bound BPTT sweep
    // Whose first-layer conv-output gradients cnn_dY0 holds: those of the last rollout after a complete
    // marlc_episode_backward (read by marlc_episode_image_grad), those of a stand-alone step after a complete
    // marlc_model_step_backward (read by marlc_model_step_input_grad), or neither: every forward, model step and
    // backward clears it first, and a backward cut short by marlc_engine_debug_stop leaves it cleared.
    enum class Dy0Owner { none, episode, step } dy0_owner = Dy0Owner::none;
    cudaEvent_t ev[64];
    int n_ev = 0, ev_i = 0;
    cudaEvent_t next_event() { cudaEvent_t x = ev[ev_i]; ev_i = (ev_i + 1) % n_ev; return x; }
    // make `to` wait for everything issued so far on `from`
    int chain(cudaStream_t from, cudaStream_t to) {
        cudaEvent_t x = next_event();
        MARLC_CUDA(cudaEventRecord(x, from));
        MARLC_CUDA(cudaStreamWaitEvent(to, x, 0));
        return 0;
    }

    // ---- layout helpers
    void add_param(const std::string& name, std::initializer_list<int64_t> shape) {
        ParamInfo p;
        p.name = "_ModelsWrapper__" + name;
        p.ndim = (int)shape.size();
        p.numel = 1;
        int i = 0;
        for (int k = 0; k < 4; ++k) p.shape[k] = 1;
        for (auto s : shape) { p.shape[i++] = s; p.numel *= s; }
        p.offset = param_floats;
        param_floats += (p.numel + 63) / 64 * 64;  // 256-byte aligned slots (TMA / vector friendly)
        params.push_back(p);
    }
    void add_buf(const std::string& name, size_t bytes) {
        BufInfo b{name, ws_bytes, bytes};
        ws_bytes += (bytes + 255) / 256 * 256;
        bufs.push_back(b);
    }
    const ParamInfo* find_param(const std::string& suffix) const {
        for (auto& p : params)
            if (p.name == "_ModelsWrapper__" + suffix) return &p;
        return nullptr;
    }
    float* prm(const std::string& suffix) const { return P + find_param(suffix)->offset; }
    // ---- pre-split low-order parts for 3xTF32 (see tc.cuh): parameters are split once per forward,
    // activations next to where they are produced.  lo_of(p) is the lo twin of a pointer into the
    // parameter block / H / Hc / U / dgates history, or nullptr (the GEMM then splits in-kernel).
    bool lo_on = false;
    // H_lo / Hc_lo are written by the fused tensor-core LSTM epilogue only; when a step falls back to
    // the FFMA gate GEMMs + point-wise cell (n_a != n_b, shapes TMA cannot address) they are NOT
    // maintained and must not be offered as operands (a stale lo silently degrades 3xTF32 to TF32)
    bool h_lo_ok = false;
    const float* lo_of(const float* p) const {
        if (!lo_on || !p) return nullptr;
        struct R { const float* base; size_t n; const float* lo; };
        const size_t Ms = (size_t)M, T1 = (size_t)cfg.T + 1;
        const R r[] = {{P, (size_t)param_floats, buf("params_lo")},
                       {buf("H"), T1 * Ms * cfg.n_b, buf("H_lo")},
                       {buf("Hc"), T1 * Ms * cfg.n_a, buf("Hc_lo")}
                       };
        for (int i = 0; i < 3; ++i) {
            const R& q = r[i];
            if (i > 0 && !h_lo_ok) break;
            if (q.lo && p >= q.base && p < q.base + q.n) return q.lo + (p - q.base);
        }
        return nullptr;
    }
    TcOperand op(const float* p, long ld, bool mn = false) const {
        TcOperand o = tc_op(p, ld, mn);
        o.lo = lo_of(p);
        return o;
    }
    float* grd(const std::string& suffix) const { return G + find_param(suffix)->offset; }
    template <typename T = float>
    T* buf(const std::string& name) const {
        for (auto& b : bufs)
            if (b.name == name) return reinterpret_cast<T*>(ws + b.offset);
        return nullptr;
    }
};

static const char* CNN_PREFIX = "map_obs._Generic2dCnnModule__layers.";
static const char* LSTM_B = "belief_unit._LSTMCellWrapper__lstm.";
static const char* LSTM_A = "action_unit._LSTMCellWrapper__lstm.";

static void add_block(marlc_engine* e, const std::string& name, int i, int n_in, int n_out, bool norm) {
    e->add_param(name + "." + std::to_string(i) + ".weight", {n_out, n_in});
    e->add_param(name + "." + std::to_string(i) + ".bias", {n_out});
    if (norm) {
        e->add_param(name + "." + std::to_string(i + 1) + ".weight", {n_out});
        e->add_param(name + "." + std::to_string(i + 1) + ".bias", {n_out});
    }
}

extern "C" int marlc_version(void) { return 1; }

// Host-side check of the reciprocal division the element-wise kernels index with (FastDiv,
// common.cuh): for every divisor 1..d_max, every dividend the launchers' bound admits (sampled with
// `stride`, plus the values around each multiple of d near the bound) must divide exactly.
// Returns the number of mismatches; needs no GPU.
extern "C" long marlc_selftest_fastdiv(int d_max, int stride) {
    long bad = 0;
    if (stride < 1) stride = 1;
    for (int d = 1; d <= d_max; ++d) {
        const marlc::FastDiv fd((unsigned)d);
        const long long limit = std::min<long long>(0x7fffffffll, (0x100000000ll - 1) / d);  // n * d < 2^32
        for (long long n = 0; n <= limit; n += stride) bad += fd.div((int)n) != (int)(n / d);
        for (long long q = std::max<long long>(0, limit / d - 2); q <= limit / d; ++q)
            for (long long n = std::max<long long>(0, q * d - 1); n <= std::min(limit, q * d + 1); ++n)
                bad += fd.div((int)n) != (int)(n / d);
        bad += !marlc::FastDiv::exact_up_to(limit, d);
    }
    return bad;
}
extern "C" const char* marlc_last_error(void) { return g_err; }

extern "C" int marlc_engine_create(const marlc_config* c, marlc_engine** out) {
    MARLC_CHECK(c && out, "null argument");
    MARLC_CHECK(c->na >= 1 && c->nb >= 1 && c->T >= 1, "bad episode geometry na=%d nb=%d T=%d", c->na, c->nb, c->T);
    MARLC_CHECK(c->f >= 1 && c->f < c->H && c->f < c->W, "window f=%d does not fit image %dx%d (need f < size)", c->f,
                c->H, c->W);
    MARLC_CHECK(c->n_actions >= 1 && c->n_actions <= MARLC_MAX_ACTIONS, "nb_action=%d out of range", c->n_actions);
    MARLC_CHECK(c->cnn_layers >= 1 && c->cnn_layers <= MARLC_MAX_CNN_LAYERS, "cnn_layers=%d out of range", c->cnn_layers);
    MARLC_CHECK(c->cnn_cin[0] <= c->C, "CNN wants %d input channels, image has %d", c->cnn_cin[0], c->C);
    marlc_engine* e = new marlc_engine();
    e->cfg = *c;
    if (c->na * c->nb < 1) e->cfg.use_chains = 0;
    e->M = c->na * c->nb;
    e->TM = e->M * c->T;
    e->L = c->cnn_layers;
    CnnDesc& d = e->cnn;
    memset(&d, 0, sizeof(d));
    d.L = e->L;
    d.f = c->f;
    d.img_c = c->C;
    int h = c->f;
    for (int l = 0; l < e->L; ++l) {
        d.cin[l] = c->cnn_cin[l];
        d.cout[l] = c->cnn_cout[l];
        d.groups[l] = c->cnn_groups[l];
        if (d.cout[l] % d.groups[l] != 0 || (l > 0 && d.cin[l] != d.cout[l - 1])) {
            delete e;
            MARLC_FAIL("inconsistent CNN description at layer %d", l);
        }
        d.hin[l] = h;
        h = (h - 1) / 2 + 1;  // k=3, s=2, p=1 (vision.py:31-33,41-43)
        d.hout[l] = h;
        e->cnn_sz[l] = d.cout[l] * h * h;
    }
    d.out_size = e->cnn_sz[e->L - 1];
    e->F = d.out_size;
    e->Kin = e->F + c->n_m_o + c->n_d;
    e->lo_on = c->use_tc == 2 && e->cfg.use_chains;

    // ---- parameters, in the reference's registration order (models.py:55-76)
    for (int l = 0; l < e->L; ++l) {
        e->add_param(CNN_PREFIX + std::to_string(3 * l) + ".weight", {d.cout[l], d.cin[l], 3, 3});
        e->add_param(CNN_PREFIX + std::to_string(3 * l) + ".bias", {d.cout[l]});
        e->add_param(CNN_PREFIX + std::to_string(3 * l + 1) + ".weight", {d.cout[l]});
        e->add_param(CNN_PREFIX + std::to_string(3 * l + 1) + ".bias", {d.cout[l]});
    }
    add_block(e, "map_pos", 0, 2, c->n_d, true);
    add_block(e, "encode_msg", 0, c->n_b, 2 * c->n_m, true);
    add_block(e, "encode_msg", 3, 2 * c->n_m, c->n_m, true);
    add_block(e, "decode_msg", 0, c->n_m, 2 * c->n_m, true);
    add_block(e, "decode_msg", 3, 2 * c->n_m, c->n_m_o, true);
    for (int k = 0; k < 2; ++k) {
        const std::string pre = k ? LSTM_A : LSTM_B;
        const int n = k ? c->n_a : c->n_b;
        e->add_param(pre + "weight_ih", {4 * n, e->Kin});
        e->add_param(pre + "weight_hh", {4 * n, n});
        e->add_param(pre + "bias_ih", {4 * n});
        e->add_param(pre + "bias_hh", {4 * n});
    }
    add_block(e, "policy", 0, c->n_a, c->nl_a, true);
    add_block(e, "policy", 3, c->nl_a, c->n_actions, false);
    add_block(e, "critic", 0, c->n_a, c->nl_a, true);
    add_block(e, "critic", 3, c->nl_a, 1, false);
    add_block(e, "predict", 0, c->n_b, c->nl_b, true);
    add_block(e, "predict", 3, c->nl_b, c->nb_class, false);

    // ---- workspace
    const size_t M = e->M, TM = e->TM, T = c->T, F4 = sizeof(float);
    e->add_buf("rng_state", 2 * sizeof(uint64_t));
    e->add_buf("pos_hist", (T + 1) * M * 2 * sizeof(int));
    e->add_buf("npos", (T + 1) * M * 2 * F4);
    e->add_buf("act", TM * sizeof(int));
    e->add_buf("zero_act", M * sizeof(int64_t));  // must stay zero (workspace is zero-initialised by the caller)
    e->add_buf("step_pos", TM * 2 * sizeof(int64_t));
    for (int l = 0; l < e->L; ++l) e->add_buf("cnn_y" + std::to_string(l), TM * e->cnn_sz[l] * F4);
    e->add_buf("U", TM * e->Kin * F4);
    e->add_buf("msg", (T + 1) * M * c->n_m * F4);
    e->add_buf("coll", TM * c->n_m * F4);
    e->add_buf("dec_y1", TM * 2 * c->n_m * F4);
    e->add_buf("dec_s1", TM * 2 * c->n_m * F4);
    e->add_buf("dec_y2", TM * c->n_m_o * F4);
    e->add_buf("pos_y", TM * c->n_d * F4);
    e->add_buf("H", (T + 1) * M * c->n_b * F4);
    e->add_buf("Cb", (T + 1) * M * c->n_b * F4);
    e->add_buf("Hc", (T + 1) * M * c->n_a * F4);
    e->add_buf("Cc", (T + 1) * M * c->n_a * F4);
    e->add_buf("gates_b", TM * 4 * c->n_b * F4);
    e->add_buf("gates_a", TM * 4 * c->n_a * F4);
    e->add_buf("enc_y1", TM * 2 * c->n_m * F4);
    e->add_buf("enc_s1", TM * 2 * c->n_m * F4);
    e->add_buf("enc_y2", TM * c->n_m * F4);
    e->add_buf("pol_y1", TM * c->nl_a * F4);
    e->add_buf("pol_s1", TM * c->nl_a * F4);
    e->add_buf("probs", TM * c->n_actions * F4);
    e->add_buf("cri_y1", TM * c->nl_a * F4);
    e->add_buf("cri_s1", TM * c->nl_a * F4);
    e->add_buf("prd_y1", TM * c->nl_b * F4);
    e->add_buf("prd_s1", TM * c->nl_b * F4);
    e->add_buf("step_preds", TM * c->nb_class * F4);
    e->add_buf("step_log_probas", TM * F4);
    e->add_buf("step_values", TM * F4);
    // loss
    e->add_buf("rewards", TM * F4);
    e->add_buf("returns", TM * F4);
    e->add_buf("adv", TM * F4);
    e->add_buf("loss_stats", 16 * sizeof(double));
    e->add_buf("loss_out", 8 * F4);
    e->add_buf("d_preds", TM * c->nb_class * F4);
    e->add_buf("d_logp", TM * F4);
    e->add_buf("d_values", TM * F4);
    // backward
    const size_t nl_max = (size_t)std::max(c->nl_a, c->nl_b);
    e->add_buf("d_pol_logits", TM * c->n_actions * F4);
    e->add_buf("scratchS", TM * nl_max * F4);
    e->add_buf("scratchY", TM * nl_max * F4);
    e->add_buf("scratchS2", TM * nl_max * F4);  // second pair: the prediction head runs on a side stream
    e->add_buf("scratchY2", TM * nl_max * F4);
    e->add_buf("scratchS3", TM * nl_max * F4);  // third pair: the critic head
    e->add_buf("scratchY3", TM * nl_max * F4);
    e->add_buf("dH_heads", TM * c->n_b * F4);
    e->add_buf("dHc_heads", TM * c->n_a * F4);
    e->add_buf("dgates_b", TM * 4 * c->n_b * F4);
    e->add_buf("dgates_a", TM * 4 * c->n_a * F4);
    e->add_buf("dU", TM * e->Kin * F4);
    e->add_buf("d_enc_y2", TM * c->n_m * F4);
    e->add_buf("d_enc_y1", TM * 2 * c->n_m * F4);
    e->add_buf("d_dec_y2", TM * c->n_m_o * F4);
    e->add_buf("d_dec_y1", TM * 2 * c->n_m * F4);
    e->add_buf("d_pos_y", TM * c->n_d * F4);
    e->add_buf("tmpS", M * 2 * c->n_m * F4);
    e->add_buf("dcoll", M * c->n_m * F4);
    e->add_buf("dmsg", M * c->n_m * F4);
    e->add_buf("dh_hist", TM * c->n_b * F4);   // per-step carries dgates(t) Whh (split-K targets, zeroed once)
    e->add_buf("dhc_hist", TM * c->n_a * F4);
    e->add_buf("dh", M * c->n_b * F4);
    e->add_buf("dc0", M * c->n_b * F4);
    e->add_buf("dc1", M * c->n_b * F4);
    e->add_buf("dhc", M * c->n_a * F4);
    e->add_buf("dcc0", M * c->n_a * F4);
    e->add_buf("dcc1", M * c->n_a * F4);
    if (e->cfg.use_chains)
        for (int l = 0; l < e->L; ++l)  // transposed conv weights for the register-tiled forward block
            e->add_buf("cnn_wT" + std::to_string(l), (size_t)d.cout[l] * d.cin[l] * 9 * F4);
    if (e->lo_on) {
        e->add_buf("params_lo", (size_t)e->param_floats * F4);
        e->add_buf("U_lo", M * e->Kin * F4);  // one step at a time: only the per-step LSTM GEMM reads it
        e->add_buf("H_lo", (T + 1) * M * c->n_b * F4);
        e->add_buf("Hc_lo", (T + 1) * M * c->n_a * F4);
        e->add_buf("dgates_b_lo", M * 4 * c->n_b * F4);  // one step at a time (the dX GEMMs of the sweep)
        e->add_buf("dgates_a_lo", M * 4 * c->n_a * F4);
    }
    for (int l = 0; l < e->L; ++l) {
        const size_t npos = (size_t)d.hout[l] * d.hout[l];
        e->add_buf("cnn_dY" + std::to_string(l), TM * npos * d.cout[l] * F4);
        // (rows padded to a multiple of 4 floats: the 27-float rows of the first layer become a TMA-addressable
        //  operand of the weight-gradient GEMM)
        e->add_buf("cnn_col" + std::to_string(l), TM * npos * (size_t)((d.cin[l] * 9 + 3) & ~3) * F4);
        e->add_buf("cnn_gnpart" + std::to_string(l), TM * 2 * d.cout[l] * F4);
        if (l > 0) e->add_buf("cnn_dcol" + std::to_string(l), TM * npos * d.cin[l] * 9 * F4);
    }
    *out = e;
    return 0;
}

extern "C" void marlc_engine_destroy(marlc_engine* e) {
    if (!e) return;
    for (int i = 0; i < e->n_ev; ++i) cudaEventDestroy(e->ev[i]);
    for (int i = 0; i < 2; ++i)
        if (e->side[i]) cudaStreamDestroy(e->side[i]);
    if (e->hp) cudaStreamDestroy(e->hp);
    delete e;
}
extern "C" int marlc_engine_param_count(const marlc_engine* e) { return (int)e->params.size(); }
extern "C" int64_t marlc_engine_param_floats(const marlc_engine* e) { return e->param_floats; }
extern "C" int marlc_engine_param_info(const marlc_engine* e, int idx, char* name, int64_t* offset, int* ndim,
                                       int64_t* shape) {
    MARLC_CHECK(idx >= 0 && idx < (int)e->params.size(), "param index %d out of range", idx);
    const ParamInfo& p = e->params[idx];
    strncpy(name, p.name.c_str(), 127);
    name[127] = 0;
    *offset = p.offset;
    *ndim = p.ndim;
    for (int k = 0; k < 4; ++k) shape[k] = p.shape[k];
    return 0;
}
extern "C" size_t marlc_engine_workspace_bytes(const marlc_engine* e) { return e->ws_bytes; }
extern "C" int marlc_engine_buffer(const marlc_engine* e, const char* name, size_t* offset, size_t* nbytes) {
    for (auto& b : e->bufs)
        if (b.name == name) {
            *offset = b.offset;
            *nbytes = b.bytes;
            return 0;
        }
    MARLC_FAIL("unknown workspace buffer '%s'", name);
}

extern "C" int marlc_engine_bind(marlc_engine* e, void* workspace, float* params, float* grads) {
    MARLC_CHECK(workspace && params, "bind: null workspace / params");
    MARLC_CHECK(((uintptr_t)workspace & 255) == 0 && ((uintptr_t)params & 255) == 0, "bind: buffers must be 256-byte aligned");
    e->ws = (char*)workspace;
    e->P = params;
    e->G = grads;
    if (e->n_ev == 0) {
        for (int i = 0; i < 2; ++i) MARLC_CUDA(cudaStreamCreateWithFlags(&e->side[i], cudaStreamNonBlocking));
        int least = 0, greatest = 0;
        MARLC_CUDA(cudaDeviceGetStreamPriorityRange(&least, &greatest));
        MARLC_CUDA(cudaStreamCreateWithPriority(&e->hp, cudaStreamNonBlocking, greatest));
        for (int i = 0; i < 64; ++i) {
            MARLC_CUDA(cudaEventCreateWithFlags(&e->ev[i], cudaEventDisableTiming));
            e->n_ev = i + 1;
        }
    }
    for (int l = 0; l < e->L; ++l) {
        e->cnn.w[l] = e->prm(CNN_PREFIX + std::to_string(3 * l) + ".weight");
        e->cnn.b[l] = e->prm(CNN_PREFIX + std::to_string(3 * l) + ".bias");
        e->cnn.gn_w[l] = e->prm(CNN_PREFIX + std::to_string(3 * l + 1) + ".weight");
        e->cnn.gn_b[l] = e->prm(CNN_PREFIX + std::to_string(3 * l + 1) + ".bias");
        e->cnn.wT[l] = e->cfg.use_chains ? e->buf("cnn_wT" + std::to_string(l)) : nullptr;
    }
    return 0;
}

__global__ void seed_kernel(uint64_t* st, uint64_t seed) { st[0] = seed; st[1] = 0; }
extern "C" int marlc_engine_seed(marlc_engine* e, uint64_t seed, void* stream) {
    MARLC_CHECK(e->ws, "engine not bound");
    seed_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(e->buf<uint64_t>("rng_state"), seed);
    MARLC_LAUNCH_CHECK();
    return 0;
}


static inline TcOperand tc_op_lo(const float* p, const float* lo, long ld) {
    TcOperand o = tc_op(p, ld);
    o.lo = lo;
    return o;
}
// tf32_lo of up to three arrays in one launch (parameters, h_0, h^_0)
struct SplitLoArgs { const float* src[3]; float* dst[3]; long n[3]; };
__global__ void __launch_bounds__(256) split_lo_kernel(const SplitLoArgs a) {
    const int k = blockIdx.y;
    const long n4 = a.n[k] >> 2;
    const float4* s4 = reinterpret_cast<const float4*>(a.src[k]);
    float4* d4 = reinterpret_cast<float4*>(a.dst[k]);
    for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n4; i += (long)gridDim.x * blockDim.x) {
        float4 v = s4[i];
        v.x = tf32_lo(v.x); v.y = tf32_lo(v.y); v.z = tf32_lo(v.z); v.w = tf32_lo(v.w);
        d4[i] = v;
    }
    if (blockIdx.x == 0 && threadIdx.x < (a.n[k] & 3)) {  // ragged tail
        const long i = (n4 << 2) + threadIdx.x;
        a.dst[k][i] = tf32_lo(a.src[k][i]);
    }
}
// h0 / hc0: the first step's recurrent inputs (nullptr: skip; only the parameters are refreshed)
static int refresh_lo(marlc_engine* e, const float* h0, const float* hc0, cudaStream_t s) {
    if (e->cfg.use_chains) {  // derived copies of the parameters, once per forward
        float* wT[MAX_CNN_LAYERS];
        for (int l = 0; l < e->L; ++l) wT[l] = const_cast<float*>(e->cnn.wT[l]);
        MARLC_TRY(cnn_weights_transpose(e->cnn, wT, s));
    }
    if (!e->lo_on) return 0;
    SplitLoArgs a;
    a.src[0] = e->P; a.dst[0] = e->buf("params_lo"); a.n[0] = e->param_floats;  // slots are multiples of 64 floats
    // (slot 0 of the histories: always refreshed, whether or not the LSTM launch ends up consuming it)
    a.src[1] = h0; a.dst[1] = h0 ? e->buf("H_lo") + (h0 - e->buf("H")) : nullptr; a.n[1] = h0 ? (long)e->M * e->cfg.n_b : 0;
    a.src[2] = hc0; a.dst[2] = hc0 ? e->buf("Hc_lo") + (hc0 - e->buf("Hc")) : nullptr; a.n[2] = hc0 ? (long)e->M * e->cfg.n_a : 0;
    split_lo_kernel<<<dim3(296, 3), 256, 0, s>>>(a);
    MARLC_LAUNCH_CHECK();
    return 0;
}

// ---- GEMM dispatch: tcgen05 TF32 when enabled and TMA-addressable, else exact fp32 FFMA ----------
static inline int x3_of(const marlc_engine* e) { return e->cfg.use_tc == 2 ? 1 : 0; }

// ---- launch decisions that depend on the geometry only (the launchers and marlc_engine_plan share them)
// both LSTM cells in one tensor-core launch (tc_lstm_pair) rather than FFMA gate GEMMs + point-wise cells
static bool lstm_on_tc(const marlc_engine* e) {
    const marlc_config& c = e->cfg;
    return c.use_tc && c.n_a == c.n_b && tc_lstm_shapes_ok(e->Kin, c.n_b);
}
// Fused chain kernels for the sweep while a step has fewer than 4096 rows (latency-bound: 3 launches per step).
// From 4096 rows per step on (config 4 on ONE GPU) the one-kernel-per-op sweep with its products on the
// tensor cores wins: the chains run 4 rows per CTA, one CTA per SM.  Measured (sweep of 16 steps): 4096 rows
// 2.72 vs 3.01 ms, 2048 rows 2.91 vs 2.48 ms -- hence the threshold.
constexpr int SWEEP_UNFUSED_MIN_M = 4096;
static bool sweep_chained(const marlc_engine* e) { return e->cfg.use_chains && e->M < SWEEP_UNFUSED_MIN_M; }

extern "C" int marlc_engine_plan(const marlc_engine* e, marlc_plan* out) {
    MARLC_CHECK(e && out, "plan: null argument");
    const marlc_config& c = e->cfg;
    const int M = e->M;
    marlc_plan p;
    memset(&p, 0, sizeof(p));
    // feature extractor of the episode forward: step_pre with the chains, else cnn_fwd (one CTA per window)
    const StepPrePlan sp = c.use_chains ? step_pre_plan(e->cnn, true, true, M) : StepPrePlan{1, 0};
    p.cnn_wide = sp.cnn_blocks > 0;
    p.cnn_nw = sp.nw;
    p.cnn_batches = (M + sp.nw - 1) / sp.nw;
    p.cnn_ctas = p.cnn_wide ? sp.cnn_blocks : M;
    p.cnn_passes = (p.cnn_batches + p.cnn_ctas - 1) / p.cnn_ctas;
    p.cnn_tail = M - (p.cnn_batches - 1) * sp.nw;
    if (lstm_on_tc(e)) {
        const TcLstmPlan lp = tc_lstm_plan(M, c.n_b, c.n_a, x3_of(e) != 0);
        p.lstm_tc = 1;
        p.lstm_hu = lp.hu; p.lstm_bn = lp.bn; p.lstm_fat = lp.fat; p.lstm_ks = lp.ks; p.lstm_ksplit = lp.ksplit;
        p.lstm_tail_rows = lp.tail_rows;
    }
    p.sweep_chained = sweep_chained(e);
    if (c.use_chains) {
        p.staged_step_pre = step_pre_stage(c.n_m, 2 * c.n_m, c.n_m_o, c.n_d).wfl > 0;
        p.staged_step_post = step_post_stage(2 * c.n_m, c.n_m).wfl > 0;
    }
    if (p.sweep_chained) {
        p.staged_bwd_pre = bwd_pre_stage(c.n_m, 2 * c.n_m, c.n_b).wfl > 0;
        p.staged_bwd_post = bwd_post_stage(c.n_m, 2 * c.n_m, c.n_m_o).wfl > 0;
    }
    *out = p;
    return 0;
}
static bool tc_worth(int m_out, int n_out, int k_red) { return n_out >= 16 && k_red >= 32 && m_out >= 1; }

// Y[M,N] = X[M,K] W[N,K]^T + bias
static int G_nt(const marlc_engine* e, const float* X, long ldx, const float* W, long ldw, const float* bias, float* Y,
                long ldy, int M, int N, int K, int accumulate, cudaStream_t s) {
    if (e->cfg.use_tc && tc_worth(M, N, K)) {
        TcGemmArgs a;
        a.A = tc_op(X, ldx); a.B = tc_op(W, ldw); a.K = K;
        a.C = Y; a.ldc = ldy; a.M = M; a.N = N; a.bias = bias; a.accumulate = accumulate;
        a.x3 = x3_of(e);
        if (tc_operand_ok(a.A) && tc_operand_ok(a.B)) return tc_gemm(a, s);
    }
    return gemm_nt(X, ldx, W, ldw, bias, Y, ldy, M, N, K, accumulate, s);
}
// GEMM arithmetic of a backward product: tensor cores where the shape allows (use_tc), error-compensated 3xTF32
// there (x3); everything else on the exact-fp32 FFMA kernels
struct GemmMode { int use_tc, x3; };
static inline GemmMode gemm_mode(const marlc_engine* e) { return {e->cfg.use_tc, x3_of(e)}; }

// dX[M,K] (+)= dY[M,N] W[N,K]   (reduction over N; W is the MN-major B operand)
static int G_nn(GemmMode m, const float* dY, long lddy, const float* W, long ldw, float* dX, long lddx, int M, int N,
                int K, int accumulate, cudaStream_t s) {
    if (m.use_tc && tc_worth(M, K, N)) {
        TcGemmArgs a;
        a.A = tc_op(dY, lddy); a.B = tc_op(W, ldw, true); a.K = N;
        a.C = dX; a.ldc = lddx; a.M = M; a.N = K; a.accumulate = accumulate;
        a.x3 = m.x3;
        a.allow_split = accumulate ? 0 : 1;
        if (tc_operand_ok(a.A) && tc_operand_ok(a.B)) return tc_gemm(a, s);
    }
    return gemm_nn(dY, lddy, W, ldw, dX, lddx, M, N, K, accumulate, s);
}
static int G_nn(const marlc_engine* e, const float* dY, long lddy, const float* W, long ldw, float* dX, long lddx, int M,
                int N, int K, int accumulate, cudaStream_t s) {
    return G_nn(gemm_mode(e), dY, lddy, W, ldw, dX, lddx, M, N, K, accumulate, s);
}
// dW[N,K] += dY[R,N]^T X[R,K]   (reduction over rows R; both operands MN-major)
static int G_tn(GemmMode m, const float* dY, long lddy, const float* X, long ldx, float* dW, long lddw, int R, int N,
                int K, cudaStream_t s) {
    if (m.use_tc && N > 8 && tc_worth(N, K, R) && K >= 16) {  // N <= 8: one-pass reduction (skinny.cu)
        TcGemmArgs a;
        a.A = tc_op(dY, lddy, true); a.B = tc_op(X, ldx, true); a.K = R;
        a.C = dW; a.ldc = lddw; a.M = N; a.N = K; a.accumulate = 1;
        a.x3 = m.x3;
        a.allow_split = 1;
        if (tc_operand_ok(a.A) && tc_operand_ok(a.B)) return tc_gemm(a, s);
    }
    return gemm_tn(dY, lddy, X, ldx, dW, lddw, R, N, K, 1, s);
}
static int G_tn(const marlc_engine* e, const float* dY, long lddy, const float* X, long ldx, float* dW, long lddw, int R,
                int N, int K, cudaStream_t s) {
    return G_tn(gemm_mode(e), dY, lddy, X, ldx, dW, lddw, R, N, K, s);
}

// Layer-wise backward of the feature extractor over P windows (kernels of cnn_bwd2.cu), shared by the episode /
// step backward and marlc_cnn_backward.  Every conv product is a GEMM: input gradient dCol_l = dY_l W_l, weight
// gradient dW_l += dY_l^T col_l.  The serial chain on s0 is only layer kernel -> input-gradient GEMM -> next layer
// kernel; the im2col of the input windows (s1) is independent of it, and the weight-gradient GEMMs wait at the end
// and fan out over s0 / s1 / sL (through `done`; nullptr when the three are one stream).  GroupNorm-affine and
// conv-bias gradients are accumulated inside the layer kernel, so d_b / d_gn_w / d_gn_b must all be set.  A null
// d_w[l] skips layer l's weight-gradient GEMM and the im2col that feeds it (col[l] is not touched).
struct CnnBwdLayers {
    const CnnDesc* d;   // shapes and parameters
    CnnWindows win;     // the input windows (operand of the first layer's weight gradient)
    int P;              // windows
    const float* ysave[MAX_CNN_LAYERS];  // [P, cout*ho^2] pre-norm conv outputs, (c, pos) order
    const float* dOut;  // [P, lddo] gradient on the flattened output, (c, pos) order
    long lddo;
    float* dY[MAX_CNN_LAYERS];    // [P*ho^2, cout]
    float* col[MAX_CNN_LAYERS];   // [P*ho^2, pitch]: pitch round_up(cin*9, 4) for layer 0, cin*9 above
    float* dcol[MAX_CNN_LAYERS];  // l > 0: [P*ho^2, cin*9]
    float* d_w[MAX_CNN_LAYERS];   // accumulated into; nullable
    float* d_b[MAX_CNN_LAYERS];   // accumulated into
    float* d_gn_w[MAX_CNN_LAYERS];
    float* d_gn_b[MAX_CNN_LAYERS];
};
static int cnn_backward_layers(GemmMode m, const CnnBwdLayers& a, cudaStream_t s0, cudaStream_t s1, cudaStream_t sL,
                               cudaEvent_t done) {
    const CnnDesc& d = *a.d;
    if (a.d_w[0]) MARLC_TRY(cnn_im2col_input(a.win, a.col[0], a.P, d.cin[0], d.hout[0], s1));
    for (int l = d.L - 1; l >= 0; --l) {
        CnnBwdLayerArgs la;
        memset(&la, 0, sizeof(la));
        la.cout = d.cout[l]; la.ho = d.hout[l]; la.groups = d.groups[l]; la.P = a.P;
        la.Y = a.ysave[l]; la.gn_w = d.gn_w[l]; la.gn_b = d.gn_b[l];
        const bool top = (l == d.L - 1);
        la.dOut = top ? a.dOut : nullptr; la.lddo = a.lddo;
        la.dColNext = top ? nullptr : a.dcol[l + 1];
        la.ho_next = top ? 1 : d.hout[l + 1];
        la.dY = a.dY[l]; la.gnpart = nullptr;
        la.d_gn_w = a.d_gn_w[l]; la.d_gn_b = a.d_gn_b[l]; la.d_conv_b = a.d_b[l];
        la.colNext = (top || !a.d_w[l + 1]) ? nullptr : a.col[l + 1];
        MARLC_TRY(cnn_bwd_layer(la, s0));
        if (l > 0) {
            const int npos = d.hout[l] * d.hout[l], kk = d.cin[l] * 9;
            MARLC_TRY(G_nn(m, a.dY[l], d.cout[l], d.w[l], kk, a.dcol[l], kk, a.P * npos, d.cout[l], kk, 0, s0));
        }
    }
    if (done) {
        MARLC_CUDA(cudaEventRecord(done, s0));
        if (s1 != s0) MARLC_CUDA(cudaStreamWaitEvent(s1, done, 0));
        if (sL != s0) MARLC_CUDA(cudaStreamWaitEvent(sL, done, 0));
    }
    // layer 0 reads the im2col of the input windows, produced on s1: it stays on s1
    const cudaStream_t fan[3] = {s0, s1, sL};
    for (int l = d.L - 1, i = 0; l >= 0; --l, ++i) {
        if (!a.d_w[l]) continue;
        const int npos = d.hout[l] * d.hout[l], kk = d.cin[l] * 9, co = d.cout[l];
        const int pitch = l == 0 ? (kk + 3) & ~3 : kk;  // the batched im2col pads the input layer's rows
        MARLC_TRY(G_tn(m, a.dY[l], co, a.col[l], pitch, a.d_w[l], kk, a.P * npos, co, kk, l == 0 ? s1 : fan[(i & 1) ? 2 : 0]));
    }
    return 0;
}


// several dW[N,K] += dY[R,N]^T X[R,K] products in one grouped tensor-core launch (<= 3), falling back to
// one launch each when any of them is not TMA-addressable / worth a tensor-core tile
struct TnProblem { const float* dY; long lddy; const float* X; long ldx; float* dW; long lddw; int R, N, K; };
static int G_tn_group(const marlc_engine* e, const TnProblem* p, int count, cudaStream_t s) {
    bool ok = e->cfg.use_tc != 0 && count <= 3;
    TcGemmArgs g[3];
    for (int i = 0; ok && i < count; ++i) {
        TcGemmArgs& a = g[i];
        a.A = tc_op(p[i].dY, p[i].lddy, true); a.B = tc_op(p[i].X, p[i].ldx, true); a.K = p[i].R;
        a.C = p[i].dW; a.ldc = p[i].lddw; a.M = p[i].N; a.N = p[i].K; a.accumulate = 1;
        a.x3 = x3_of(e); a.allow_split = 1;
        ok = tc_worth(p[i].N, p[i].K, p[i].R) && p[i].K >= 16 && tc_operand_ok(a.A) && tc_operand_ok(a.B);
    }
    if (ok) return tc_gemm_group(g, count, s);
    for (int i = 0; i < count; ++i)
        MARLC_TRY(G_tn(e, p[i].dY, p[i].lddy, p[i].X, p[i].ldx, p[i].dW, p[i].lddw, p[i].R, p[i].N, p[i].K, s));
    return 0;
}

static ChainLin chain_lin(const marlc_engine* e, const std::string& name, int i, int n_in, int n_out, bool norm) {
    const std::string a = name + "." + std::to_string(i), b = name + "." + std::to_string(i + 1);
    ChainLin c;
    c.W = e->prm(a + ".weight"); c.b = e->prm(a + ".bias");
    c.g = norm ? e->prm(b + ".weight") : nullptr; c.be = norm ? e->prm(b + ".bias") : nullptr;
    c.dW = e->G ? e->grd(a + ".weight") : nullptr; c.db = e->G ? e->grd(a + ".bias") : nullptr;
    c.dg = (norm && e->G) ? e->grd(b + ".weight") : nullptr; c.dbe = (norm && e->G) ? e->grd(b + ".bias") : nullptr;
    c.n_in = n_in; c.n_out = n_out;
    return c;
}

// Linear -> LN -> SiLU block forward on R rows (message.py:26-33 etc.)
static int block_fwd(marlc_engine* e, const std::string& name, int i, const float* X, long ldx, int R, int n_in,
                     int n_out, float* y_pre, float* S, long lds, cudaStream_t s) {
    const std::string a = name + "." + std::to_string(i), b = name + "." + std::to_string(i + 1);
    MARLC_TRY(G_nt(e, X, ldx, e->prm(a + ".weight"), n_in, e->prm(a + ".bias"), y_pre, n_out, R, n_out, n_in, 0, s));
    MARLC_TRY(ln_silu_fwd(y_pre, n_out, e->prm(b + ".weight"), e->prm(b + ".bias"), S, lds, R, n_out, s));
    return 0;
}

// One step of every network for all M rows (models.py:78-138) up to the policy
// block-0 activations.  Slot t of the workspace receives everything backward needs.
// Inputs are explicit so that the same code serves the fused episode (workspace
// slots) and the stand-alone ModelsWrapper.forward (caller tensors).
static int step_networks(marlc_engine* e, int t, const float* img, const int* pos, const float* patch,
                         const float* msg_in, const float* npos_in, const float* h_in, const float* c_in,
                         const float* hc_in, const float* cc_in, cudaStream_t s, int pdl = 0) {
    // pdl (common.cuh, programmatic dependent launch): 0 = ordinary launches (stand-alone step), 1 = every launch but
    // the first is a programmatic dependent of its predecessor, 2 = the first one too (its predecessor in `s` is the
    // previous step's last kernel)
    const marlc_config& c = e->cfg;
    const int M = e->M, Kin = e->Kin, F = e->F;
    const int pdl_rest = pdl >= 1;
    float* Ut = e->buf("U") + (size_t)t * M * Kin;
    float* H = e->buf("H");
    float* Cb = e->buf("Cb");
    float* Hc = e->buf("Hc");
    float* Cc = e->buf("Cc");
    if (c.use_chains) {
        // fused "pre" launch: CNN | message mean + decoder + position features  (models.py:92-101)
        StepPreArgs pa;
        memset(&pa, 0, sizeof(pa));
        pa.cnn.d = e->cnn; pa.cnn.img = img; pa.cnn.pos = pos; pa.cnn.patch = patch; pa.cnn.out = Ut; pa.cnn.ldo = Kin;
        pa.cnn.out_lo = pa.U_lo = e->lo_on ? e->buf("U_lo") : nullptr;
        pa.cnn.B = c.nb; pa.cnn.H = c.H; pa.cnn.W = c.W; pa.cnn.M = M;
        cnn_fwd_plan(e->cnn, &pa.cnn.padsz, &pa.cnn.ysz, &pa.cnn.wbuf);
        for (int l = 0; l < e->L; ++l) pa.cnn.y_save[l] = e->buf("cnn_y" + std::to_string(l)) + (size_t)t * M * e->cnn_sz[l];
        pa.msg_in = msg_in;
        pa.coll = e->buf("coll") + (size_t)t * M * c.n_m;
        pa.d0 = chain_lin(e, "decode_msg", 0, c.n_m, 2 * c.n_m, true);
        pa.d3 = chain_lin(e, "decode_msg", 3, 2 * c.n_m, c.n_m_o, true);
        pa.dec_y1 = e->buf("dec_y1") + (size_t)t * M * 2 * c.n_m;
        pa.dec_s1 = e->buf("dec_s1") + (size_t)t * M * 2 * c.n_m;
        pa.dec_y2 = e->buf("dec_y2") + (size_t)t * M * c.n_m_o;
        pa.npos = npos_in;
        pa.pos = chain_lin(e, "map_pos", 0, 2, c.n_d, true);
        pa.pos_y = e->buf("pos_y") + (size_t)t * M * c.n_d;
        pa.U = Ut; pa.ldu = Kin; pa.F = F; pa.Na = c.na; pa.Nb = c.nb; pa.M = M;
        {
            PdlScope pdl_first(pdl >= 2, pdl >= 1);
            MARLC_TRY(step_pre(pa, s));
        }
        if (e->debug_stop == 11) return 0;
    } else {
        // b_t: gather + CNN straight into u_t[:, 0:F]                (models.py:92-94)
        float* ysave[MAX_CNN_LAYERS];
        for (int l = 0; l < e->L; ++l) ysave[l] = e->buf("cnn_y" + std::to_string(l)) + (size_t)t * M * e->cnn_sz[l];
        MARLC_TRY(cnn_fwd(e->cnn, img, pos, patch, c.nb, c.H, c.W, M, ysave, Ut, Kin, s));
        // d_bar_t: message mean + decoder into u_t[:, F:F+n_m_o]     (models.py:97-98)
        float* coll = e->buf("coll") + (size_t)t * M * c.n_m;
        MARLC_TRY(msg_mean(msg_in, coll, c.na, c.nb, c.n_m, s));
        float* dec_s1 = e->buf("dec_s1") + (size_t)t * M * 2 * c.n_m;
        MARLC_TRY(block_fwd(e, "decode_msg", 0, coll, c.n_m, M, c.n_m, 2 * c.n_m,
                            e->buf("dec_y1") + (size_t)t * M * 2 * c.n_m, dec_s1, 2 * c.n_m, s));
        MARLC_TRY(block_fwd(e, "decode_msg", 3, dec_s1, 2 * c.n_m, M, 2 * c.n_m, c.n_m_o,
                            e->buf("dec_y2") + (size_t)t * M * c.n_m_o, Ut + F, Kin, s));
        // lambda_t into u_t[:, F+n_m_o:]                             (models.py:101)
        MARLC_TRY(pos_features_fwd(npos_in, e->prm("map_pos.0.weight"), e->prm("map_pos.0.bias"),
                                   e->prm("map_pos.1.weight"), e->prm("map_pos.1.bias"),
                                   e->buf("pos_y") + (size_t)t * M * c.n_d, Ut + F + c.n_m_o, Kin, M, c.n_d, s));
    }
    // both LSTM cells share u_t                                   (models.py:107-123)
    float* gb = e->buf("gates_b") + (size_t)t * M * 4 * c.n_b;
    float* ga = e->buf("gates_a") + (size_t)t * M * 4 * c.n_a;
    bool fused = false;
    if (lstm_on_tc(e)) {
        TcLstmArgs la[2];
        for (int k = 0; k < 2; ++k) {
            const std::string pre = k ? LSTM_A : LSTM_B;
            const int n = k ? c.n_a : c.n_b;
            TcLstmArgs& a = la[k];
            a.U = tc_op(Ut, Kin);
            a.Hprev = tc_op(k ? hc_in : h_in, n);
            a.Wih = e->prm(pre + "weight_ih"); a.Whh = e->prm(pre + "weight_hh");
            a.bih = e->prm(pre + "bias_ih"); a.bhh = e->prm(pre + "bias_hh");
            a.c_prev = k ? cc_in : c_in;
            a.c_new = (k ? Cc : Cb) + (size_t)(t + 1) * M * n;
            a.h_new = (k ? Hc : H) + (size_t)(t + 1) * M * n;
            a.gates = k ? ga : gb;
            a.M = M; a.Kin = Kin; a.n = n;
            a.x3 = x3_of(e);
        }
        fused = tc_lstm_supported(la[0]) && tc_lstm_supported(la[1]);
        e->h_lo_ok = fused && e->lo_on;  // decided BEFORE the lo twins below are looked up
        if (fused) {
            for (int k = 0; k < 2; ++k) {  // pre-split low-order operands (3xTF32 without an in-kernel split)
                TcLstmArgs& a = la[k];
                a.U.lo = e->lo_on ? e->buf("U_lo") : nullptr;
                a.Hprev.lo = e->lo_of(a.Hprev.ptr);
                a.Wih_lo = e->lo_of(a.Wih); a.Whh_lo = e->lo_of(a.Whh);
                a.h_new_lo = const_cast<float*>(e->lo_of(a.h_new));
            }
            PdlScope pdl_lstm(0, pdl_rest);  // an ordinary launch: as a dependent it was slower (common.cuh)
            MARLC_TRY(tc_lstm_pair(la[0], la[1], s));
        }
    }
    if (!fused) e->h_lo_ok = false;
    if (!fused) {
        GemmGroup gg;
        memset(&gg, 0, sizeof(gg));
        gg.count = 2;
        for (int k = 0; k < 2; ++k) {
            const std::string pre = k ? LSTM_A : LSTM_B;
            const int n = k ? c.n_a : c.n_b;
            GemmProblem& p = gg.p[k];
            p.A = Ut; p.sam = Kin; p.sak = 1;
            p.B = e->prm(pre + "weight_ih"); p.sbk = 1; p.sbn = Kin;
            p.A2 = k ? hc_in : h_in; p.sam2 = n; p.sak2 = 1;
            p.B2 = e->prm(pre + "weight_hh"); p.sbk2 = 1; p.sbn2 = n;
            p.bias = e->prm(pre + "bias_ih"); p.bias2 = e->prm(pre + "bias_hh");
            p.C = k ? ga : gb; p.ldc = 4 * n;
            p.M = M; p.N = 4 * n; p.K = Kin; p.K2 = n;
        }
        MARLC_TRY(gemm_group(gg, s));
        MARLC_TRY(lstm_cell_fwd(gb, c_in, Cb + (size_t)(t + 1) * M * c.n_b, H + (size_t)(t + 1) * M * c.n_b, M, c.n_b, s));
        MARLC_TRY(lstm_cell_fwd(ga, cc_in, Cc + (size_t)(t + 1) * M * c.n_a, Hc + (size_t)(t + 1) * M * c.n_a, M, c.n_a, s));
    }
    if (e->debug_stop == 12) return 0;
    if (c.use_chains) {
        // block-0 GEMMs of the encoder and the policy (tensor cores, ONE grouped launch), tails fused in step_act()
        const float* enc_x = H + (size_t)(t + 1) * M * c.n_b;
        const float* pol_x = Hc + (size_t)(t + 1) * M * c.n_a;
        float* enc_y1 = e->buf("enc_y1") + (size_t)t * M * 2 * c.n_m;
        float* pol_y1 = e->buf("pol_y1") + (size_t)t * M * c.nl_a;
        bool grouped = false;
        if (c.use_tc && tc_worth(M, 2 * c.n_m, c.n_b) && tc_worth(M, c.nl_a, c.n_a)) {
            TcGemmArgs g[2];
            g[0].A = e->op(enc_x, c.n_b); g[0].B = e->op(e->prm("encode_msg.0.weight"), c.n_b); g[0].K = c.n_b;
            g[0].C = enc_y1; g[0].ldc = 2 * c.n_m; g[0].M = M; g[0].N = 2 * c.n_m; g[0].bias = e->prm("encode_msg.0.bias");
            g[1].A = e->op(pol_x, c.n_a); g[1].B = e->op(e->prm("policy.0.weight"), c.n_a); g[1].K = c.n_a;
            g[1].C = pol_y1; g[1].ldc = c.nl_a; g[1].M = M; g[1].N = c.nl_a; g[1].bias = e->prm("policy.0.bias");
            g[0].x3 = g[1].x3 = x3_of(e);
            // 8 CTAs would each stream the whole K (the loop is bound by per-SM ingest): split K down to one
            // stage per CTA; the outputs are zeroed once per episode, the first split adds the bias and the
            // epilogue is a TMA reduce-add
            g[0].allow_split = g[1].allow_split = 2;
            g[0].c_zeroed = g[1].c_zeroed = 1;
            if (tc_operand_ok(g[0].A) && tc_operand_ok(g[0].B) && tc_operand_ok(g[1].A) && tc_operand_ok(g[1].B)) {
                PdlScope pdl_g0(pdl_rest, pdl_rest);
                MARLC_TRY(tc_gemm_group(g, 2, s));
                grouped = true;
            }
        }
        if (!grouped) {
            MARLC_TRY(G_nt(e, enc_x, c.n_b, e->prm("encode_msg.0.weight"), c.n_b, e->prm("encode_msg.0.bias"), enc_y1,
                           2 * c.n_m, M, 2 * c.n_m, c.n_b, 0, s));
            MARLC_TRY(G_nt(e, pol_x, c.n_a, e->prm("policy.0.weight"), c.n_a, e->prm("policy.0.bias"), pol_y1, c.nl_a, M,
                           c.nl_a, c.n_a, 0, s));
        }
        return 0;
    }
    // message for the next step                                   (models.py:114-116)
    float* enc_s1 = e->buf("enc_s1") + (size_t)t * M * 2 * c.n_m;
    MARLC_TRY(block_fwd(e, "encode_msg", 0, H + (size_t)(t + 1) * M * c.n_b, c.n_b, M, c.n_b, 2 * c.n_m,
                        e->buf("enc_y1") + (size_t)t * M * 2 * c.n_m, enc_s1, 2 * c.n_m, s));
    MARLC_TRY(block_fwd(e, "encode_msg", 3, enc_s1, 2 * c.n_m, M, 2 * c.n_m, c.n_m,
                        e->buf("enc_y2") + (size_t)t * M * c.n_m, e->buf("msg") + (size_t)(t + 1) * M * c.n_m, c.n_m, s));
    // policy block 0                                              (models.py:126-128)
    MARLC_TRY(block_fwd(e, "policy", 0, Hc + (size_t)(t + 1) * M * c.n_a, c.n_a, M, c.n_a, c.nl_a,
                        e->buf("pol_y1") + (size_t)t * M * c.nl_a, e->buf("pol_s1") + (size_t)t * M * c.nl_a, c.nl_a, s));
    return 0;
}

// policy tail -> action -> transition  (policy.py:15-16, agent.py:51-61, environment.py:56-66)
static int step_act(marlc_engine* e, int t, const int64_t* act_in, cudaStream_t s) {
    const marlc_config& c = e->cfg;
    const int M = e->M;
    int* pos_hist = e->buf<int>("pos_hist");
    PolicyActArgs pa;
    memset(&pa, 0, sizeof(pa));
    pa.s1 = e->buf("pol_s1") + (size_t)t * M * c.nl_a;
    pa.W3 = e->prm("policy.3.weight");
    pa.b3 = e->prm("policy.3.bias");
    pa.act_in = act_in;
    pa.rng_state = e->buf<uint64_t>("rng_state");
    pa.pos_in = pos_hist + (size_t)t * M * 2;
    pa.probs = e->buf("probs") + (size_t)t * M * c.n_actions;
    pa.logp = e->buf("step_log_probas") + (size_t)t * M;
    pa.act_out = e->buf<int>("act") + (size_t)t * M;
    pa.pos_out = pos_hist + (size_t)(t + 1) * M * 2;
    pa.step_pos = e->buf<int64_t>("step_pos") + (size_t)t * M * 2;
    pa.npos_out = e->buf("npos") + (size_t)(t + 1) * M * 2;
    for (int j = 0; j < c.n_actions; ++j) { pa.moves[2 * j] = c.actions[j][0]; pa.moves[2 * j + 1] = c.actions[j][1]; }
    pa.M = M; pa.nl = c.nl_a; pa.nA = c.n_actions; pa.t = t; pa.f = c.f; pa.H = c.H; pa.W = c.W;
    if (c.use_chains) {
        // fused "post" launch: policy LN/SiLU + logits + softmax + sample + transition | encoder tail
        StepPostArgs sp;
        memset(&sp, 0, sizeof(sp));
        sp.act = pa;
        sp.pol_y1 = e->buf("pol_y1") + (size_t)t * M * c.nl_a;
        sp.pol_g = e->prm("policy.1.weight"); sp.pol_be = e->prm("policy.1.bias");
        sp.enc_y1 = e->buf("enc_y1") + (size_t)t * M * 2 * c.n_m;
        sp.enc_g = e->prm("encode_msg.1.weight"); sp.enc_be = e->prm("encode_msg.1.bias");
        sp.enc_s1 = e->buf("enc_s1") + (size_t)t * M * 2 * c.n_m;
        sp.e3 = chain_lin(e, "encode_msg", 3, 2 * c.n_m, c.n_m, true);
        sp.enc_y2 = e->buf("enc_y2") + (size_t)t * M * c.n_m;
        sp.msg_out = e->buf("msg") + (size_t)(t + 1) * M * c.n_m;
        sp.M = M;
        return step_post(sp, s);
    }
    return policy_act(pa, s);
}

// critic and prediction heads on R rows starting at state slot 1 (models.py:131-134)
static int value_pred_heads(marlc_engine* e, int R, cudaStream_t s) {
    const marlc_config& c = e->cfg;
    const int M = e->M;
    cudaStream_t sc = c.use_chains ? e->side[0] : s;  // critic head concurrently with the prediction head
    if (c.use_chains) MARLC_TRY(e->chain(s, sc));
    MARLC_TRY(block_fwd(e, "critic", 0, e->buf("Hc") + (size_t)M * c.n_a, c.n_a, R, c.n_a, c.nl_a, e->buf("cri_y1"),
                        e->buf("cri_s1"), c.nl_a, sc));
    MARLC_TRY(gemm_nt(e->buf("cri_s1"), c.nl_a, e->prm("critic.3.weight"), c.nl_a, e->prm("critic.3.bias"),
                      e->buf("step_values"), 1, R, 1, c.nl_a, 0, sc));
    MARLC_TRY(block_fwd(e, "predict", 0, e->buf("H") + (size_t)M * c.n_b, c.n_b, R, c.n_b, c.nl_b, e->buf("prd_y1"),
                        e->buf("prd_s1"), c.nl_b, s));
    MARLC_TRY(G_nt(e, e->buf("prd_s1"), c.nl_b, e->prm("predict.3.weight"), c.nl_b, e->prm("predict.3.bias"),
                   e->buf("step_preds"), c.nb_class, R, c.nb_class, c.nl_b, 0, s));
    if (c.use_chains) MARLC_TRY(e->chain(sc, s));
    return 0;
}

extern "C" int marlc_episode_forward(marlc_engine* e, const float* img, const int64_t* pos0,
                                     const float* const* hidden0, const int64_t* actions, void* stream) {
    MARLC_CHECK(e && e->ws, "engine not bound");
    MARLC_CHECK(img, "null image batch");
    NvtxRange nvtx_fwd("marlc/forward");
    e->dy0_owner = marlc_engine::Dy0Owner::none;
    cudaStream_t s = (cudaStream_t)stream;
    const marlc_config& c = e->cfg;
    const int M = e->M, T = c.T;
    const int start = g_launch_count;

    int* pos_hist = e->buf<int>("pos_hist");
    float* npos = e->buf("npos");
    float* msg = e->buf("msg");
    float* H = e->buf("H");
    float* Cb = e->buf("Cb");
    float* Hc = e->buf("Hc");
    float* Cc = e->buf("Cc");
    uint64_t* rng = e->buf<uint64_t>("rng_state");

    EpisodeInitArgs ia;
    ia.pos0 = pos0;
    for (int k = 0; k < 4; ++k) ia.hidden0[k] = hidden0 ? hidden0[k] : nullptr;
    ia.rng_state = rng;
    ia.pos = pos_hist;
    ia.npos = npos;
    ia.hidden[0] = H; ia.hidden[1] = Cb; ia.hidden[2] = Hc; ia.hidden[3] = Cc;
    ia.msg0 = msg;
    ia.width[0] = ia.width[1] = c.n_b;
    ia.width[2] = ia.width[3] = c.n_a;
    ia.M = M; ia.n_m = c.n_m; ia.H = c.H; ia.W = c.W; ia.f = c.f;
    MARLC_TRY(episode_init(ia, s));
    MARLC_TRY(refresh_lo(e, H, Hc, s));
    if (c.use_chains && c.use_tc) {  // split-K targets of the per-step block-0 GEMMs
        MARLC_CUDA(cudaMemsetAsync(e->buf("enc_y1"), 0, sizeof(float) * (size_t)e->TM * 2 * c.n_m, s));
        MARLC_CUDA(cudaMemsetAsync(e->buf("pol_y1"), 0, sizeof(float) * (size_t)e->TM * c.nl_a, s));
    }

    for (int t = 0; t < T; ++t) {
        NvtxRange nvtx_step("marlc/forward/step");
        // the step chain pre -> LSTM -> block-0 GEMMs -> post -> pre(t+1) ... runs as programmatic dependent launches
        MARLC_TRY(step_networks(e, t, img, pos_hist + (size_t)t * M * 2, nullptr, msg + (size_t)t * M * c.n_m,
                                npos + (size_t)t * M * 2, H + (size_t)t * M * c.n_b, Cb + (size_t)t * M * c.n_b,
                                Hc + (size_t)t * M * c.n_a, Cc + (size_t)t * M * c.n_a, s, t > 0 ? 2 : 1));
        if (e->debug_stop >= 11 && e->debug_stop <= 13) continue;  // profiling: skip the tail
        PdlScope pdl_post(c.use_chains, c.use_chains);
        MARLC_TRY(step_act(e, t, actions ? actions + (size_t)t * M : nullptr, s));
    }
    if (e->debug_stop >= 11 && e->debug_stop <= 14) { e->last_launches = g_launch_count - start; return 0; }
    // critic and prediction heads do not feed back into the trajectory: batch them
    // over all T steps (R = T*M rows)
    NvtxRange nvtx_heads("marlc/forward/batched_heads");
    MARLC_TRY(value_pred_heads(e, e->TM, s));
    MARLC_TRY(rng_advance(rng, s));
    e->last_launches = g_launch_count - start;
    return 0;
}

// ModelsWrapper.forward, models.py:78-138: one step on caller-provided tensors.
// Outputs land in workspace slot 0/1: probs[0:M], step_values[0:M], step_preds[0:M],
// msg[1], H[1], Cb[1], Hc[1], Cc[1].
static int model_step_fwd(marlc_engine* e, const float* patch, const float* msg, const float* npos,
                          const float* const* hidden, cudaStream_t s) {
    e->dy0_owner = marlc_engine::Dy0Owner::none;
    MARLC_TRY(refresh_lo(e, nullptr, nullptr, s));
    if (e->cfg.use_chains && e->cfg.use_tc) {
        MARLC_CUDA(cudaMemsetAsync(e->buf("enc_y1"), 0, sizeof(float) * (size_t)e->M * 2 * e->cfg.n_m, s));
        MARLC_CUDA(cudaMemsetAsync(e->buf("pol_y1"), 0, sizeof(float) * (size_t)e->M * e->cfg.nl_a, s));
    }
    MARLC_TRY(step_networks(e, 0, nullptr, nullptr, patch, msg, npos, hidden[0], hidden[1], hidden[2], hidden[3], s));
    // the tail also needs an action to form log p[a]; use the all-zero index buffer
    // (only probs are read back by ModelsWrapper.forward)
    MARLC_TRY(step_act(e, 0, e->buf<int64_t>("zero_act"), s));
    MARLC_TRY(value_pred_heads(e, e->M, s));
    return 0;
}
extern "C" int marlc_model_step(marlc_engine* e, const float* patch, const float* msg, const float* npos,
                                const float* const* hidden, void* stream) {
    MARLC_CHECK(e && e->ws, "engine not bound");
    MARLC_CHECK(patch && msg && npos && hidden && hidden[0] && hidden[1] && hidden[2] && hidden[3],
                "model_step: null input");
    const int start = g_launch_count;
    MARLC_TRY(model_step_fwd(e, patch, msg, npos, hidden, (cudaStream_t)stream));
    e->last_launches = g_launch_count - start;
    return 0;
}

static LossArgs loss_args(marlc_engine* e, const int64_t* targets) {
    LossArgs a;
    a.preds = e->buf("step_preds");
    a.logp = e->buf("step_log_probas");
    a.values = e->buf("step_values");
    a.targets = targets;
    a.rewards = e->buf("rewards");
    a.returns = e->buf("returns");
    a.adv = e->buf("adv");
    a.stats = e->buf<double>("loss_stats");
    a.d_preds = e->buf("d_preds");
    a.d_logp = e->buf("d_logp");
    a.d_values = e->buf("d_values");
    a.loss_out = e->buf("loss_out");
    a.T = e->cfg.T; a.Na = e->cfg.na; a.Nb = e->cfg.nb; a.Nc = e->cfg.nb_class;
    a.gamma = e->cfg.gamma;
    return a;
}

extern "C" int marlc_loss_phase_a(marlc_engine* e, const int64_t* targets, void* stream) {
    MARLC_CHECK(e && e->ws && targets, "loss: engine not bound / null targets");
    NvtxRange nvtx_loss("marlc/loss/phase_a");
    const int start = g_launch_count;
    MARLC_TRY(loss_phase_a(loss_args(e, targets), (cudaStream_t)stream));
    e->last_launches = g_launch_count - start;
    return 0;
}
extern "C" int marlc_loss_phase_b(marlc_engine* e, void* stream) {
    MARLC_CHECK(e && e->ws, "loss: engine not bound");
    NvtxRange nvtx_loss("marlc/loss/phase_b");
    const int start = g_launch_count;
    MARLC_TRY(loss_phase_b(loss_args(e, nullptr), (cudaStream_t)stream));
    e->last_launches = g_launch_count - start;
    return 0;
}

// Backward of a Linear->LN->SiLU block given dS; leaves dY (pre-norm grad) in dY
// and accumulates dgamma/dbeta/dbias.  Weight grads are done by the caller (batched).
static int block_bwd_norm(marlc_engine* e, const std::string& name, int i, const float* dS, long ldds,
                          const float* y_pre, int R, int n_out, float* dY, cudaStream_t s) {
    const std::string a = name + "." + std::to_string(i), b = name + "." + std::to_string(i + 1);
    return ln_silu_bwd(dS, ldds, y_pre, n_out, e->prm(b + ".weight"), e->prm(b + ".bias"), dY, n_out,
                       e->grd(b + ".weight"), e->grd(b + ".bias"), e->grd(a + ".bias"), R, n_out, s);
}

// Head backward, batched over all T*M rows: final Linear (N outputs) <- Linear->LN->SiLU <- state
static int head_bwd(marlc_engine* e, const std::string& name, const float* dOut, int N, const float* s1,
                    const float* y1, const float* state, int n_state, int nl, float* dState, int accumulate_state,
                    cudaStream_t s, int scratch = 0) {
    const int TM = e->TM;
    float* S = e->buf(scratch ? "scratchS2" : "scratchS");
    float* Y = e->buf(scratch ? "scratchY2" : "scratchY");
    MARLC_TRY(colsum_add(dOut, N, e->grd(name + ".3.bias"), TM, N, s));
    MARLC_TRY(G_tn(e, dOut, N, s1, nl, e->grd(name + ".3.weight"), nl, TM, N, nl, s));
    MARLC_TRY(G_nn(e, dOut, N, e->prm(name + ".3.weight"), nl, S, nl, TM, N, nl, 0, s));
    MARLC_TRY(block_bwd_norm(e, name, 0, S, nl, y1, TM, nl, Y, s));
    MARLC_TRY(G_tn(e, Y, nl, state, n_state, e->grd(name + ".0.weight"), n_state, TM, nl, n_state, s));
    MARLC_TRY(G_nn(e, Y, nl, e->prm(name + ".0.weight"), n_state, dState, n_state, TM, nl, n_state, accumulate_state, s));
    return 0;
}

// The same head backward split in two: the part the BPTT sweep waits for (the gradient that flows
// back into the recurrent state) and the parameter gradients, which nothing downstream consumes and
// which therefore run on a side stream underneath the sweep.
//   head_bwd_state: dS = dOut W3 ; dY = LN/SiLU backward(dS)     (also LN affine + block-0 bias grads)
//   head_bwd_params: db3 += colsum(dOut) ; dW3 += dOut^T s1 ; dW0 += dY^T state
static int head_bwd_state(marlc_engine* e, const std::string& name, const float* dOut, int N, const float* y1, int nl,
                          float* S, float* Y, cudaStream_t s) {
    if (N <= 64 && nl <= 1024 && (size_t)(N + 3) * nl * sizeof(float) <= 160 * 1024)  // fused: dS never materialised
        return ln_silu_bwd_fused(nullptr, 0, dOut, N, e->prm(name + ".3.weight"), y1, nl, e->prm(name + ".1.weight"),
                                 e->prm(name + ".1.bias"), Y, nl, e->grd(name + ".1.weight"), e->grd(name + ".1.bias"),
                                 e->grd(name + ".0.bias"), e->TM, nl, s);
    MARLC_TRY(G_nn(e, dOut, N, e->prm(name + ".3.weight"), nl, S, nl, e->TM, N, nl, 0, s));
    return block_bwd_norm(e, name, 0, S, nl, y1, e->TM, nl, Y, s);
}
static int head_bwd_params(marlc_engine* e, const std::string& name, const float* dOut, int N, const float* s1,
                           const float* Y, const float* state, int n_state, int nl, cudaStream_t s) {
    const int TM = e->TM;
    MARLC_TRY(colsum_add(dOut, N, e->grd(name + ".3.bias"), TM, N, s));
    MARLC_TRY(G_tn(e, dOut, N, s1, nl, e->grd(name + ".3.weight"), nl, TM, N, nl, s));
    return G_tn(e, Y, nl, state, n_state, e->grd(name + ".0.weight"), n_state, TM, nl, n_state, s);
}

// The two ends of the BPTT sweep when it serves one stand-alone step (marlc_model_step_backward, T = 1) instead
// of an episode.  Outer end: gradients arriving on the step's outputs, each nullable (= zero), in the order
// probs, values, preds, msg', h', c', h^', c^'.  Inner end: gradients leaving through its inputs msg, h, c, h^,
// c^, each nullable (= not wanted).  The feature-extractor backward reads the caller's windows.
struct StepEnds {
    const float* patch;
    const float* const* d_out;
    float* const* d_in;
};

// se == nullptr: the episode's BPTT (marlc_episode_backward); otherwise one step with the ends above
static int episode_backward(marlc_engine* e, const float* img, int accumulate, const StepEnds* se, cudaStream_t s) {
    MARLC_CHECK(e && e->ws && e->G, "backward: engine not bound (need a grads buffer)");
    NvtxRange nvtx_bwd("marlc/backward");
    const marlc_config& c = e->cfg;
    const int M = e->M, T = c.T, TM = e->TM, Kin = e->Kin, F = e->F;
    const int start = g_launch_count;
    e->dy0_owner = marlc_engine::Dy0Owner::none;  // until this backward runs to its end
    const float* d_probs = se ? se->d_out[0] : nullptr;
    const float* d_msg_out = se ? se->d_out[3] : nullptr;  // seeds the encoder backward of the last step
    const bool want_dh0 = se && (se->d_in[1] || se->d_in[3]);  // input gradients of step 0's recurrent states
    const bool want_dmsg0 = se && se->d_in[0];                 // ... and of its message
    if (!accumulate) MARLC_CUDA(cudaMemsetAsync(e->G, 0, sizeof(float) * (size_t)e->param_floats, s));

    float* H = e->buf("H");
    float* Cb = e->buf("Cb");
    float* Hc = e->buf("Hc");
    float* Cc = e->buf("Cc");
    float* dU = e->buf("dU");

    // ---- heads, batched over T*M rows (their gradients do not depend on the sweep)
    // (prediction head on a side stream, policy + critic heads on the main one)
    {
    NvtxRange nvtx_heads("marlc/backward/heads");
    if (c.use_chains) {
        // three heads on three streams up to dY; the policy and critic heads share their input h^, so
        // their state gradients are ONE dual-pair GEMM: dh^ = dY_pol W0_pol + dY_cri W0_cri
        cudaStream_t sp = e->side[0], sc = e->side[1];
        float *Yp = e->buf("scratchY"), *Yq = e->buf("scratchY2"), *Yc = e->buf("scratchY3");
        MARLC_TRY(e->chain(s, sp));
        MARLC_TRY(e->chain(s, sc));
        MARLC_TRY(head_bwd_state(e, "predict", e->buf("d_preds"), c.nb_class, e->buf("prd_y1"), c.nl_b,
                                 e->buf("scratchS2"), Yq, sp));
        MARLC_TRY(G_nn(e, Yq, c.nl_b, e->prm("predict.0.weight"), c.n_b, e->buf("dH_heads"), c.n_b, TM, c.nl_b, c.n_b, 0, sp));
        MARLC_TRY(head_bwd_state(e, "critic", e->buf("d_values"), 1, e->buf("cri_y1"), c.nl_a, e->buf("scratchS3"), Yc, sc));
        MARLC_TRY(policy_logit_grad(e->buf("d_logp"), e->buf("probs"), e->buf<int>("act"), e->buf("d_pol_logits"), TM,
                                    c.n_actions, s, d_probs));
        MARLC_TRY(head_bwd_state(e, "policy", e->buf("d_pol_logits"), c.n_actions, e->buf("pol_y1"), c.nl_a,
                                 e->buf("scratchS"), Yp, s));
        MARLC_TRY(e->chain(sc, s));
        bool dual = false;
        if (c.use_tc && tc_worth(TM, c.n_a, c.nl_a)) {
            TcGemmArgs a;
            a.A = tc_op(Yp, c.nl_a); a.B = e->op(e->prm("policy.0.weight"), c.n_a, true); a.K = c.nl_a;
            a.A2 = tc_op(Yc, c.nl_a); a.B2 = e->op(e->prm("critic.0.weight"), c.n_a, true); a.K2 = c.nl_a;
            a.C = e->buf("dHc_heads"); a.ldc = c.n_a; a.M = TM; a.N = c.n_a; a.x3 = x3_of(e); a.allow_split = 1;
            if (tc_operand_ok(a.A) && tc_operand_ok(a.B) && tc_operand_ok(a.A2) && tc_operand_ok(a.B2)) {
                MARLC_TRY(tc_gemm(a, s));
                dual = true;
            }
        }
        if (!dual) {
            MARLC_TRY(G_nn(e, Yp, c.nl_a, e->prm("policy.0.weight"), c.n_a, e->buf("dHc_heads"), c.n_a, TM, c.nl_a, c.n_a, 0, s));
            MARLC_TRY(G_nn(e, Yc, c.nl_a, e->prm("critic.0.weight"), c.n_a, e->buf("dHc_heads"), c.n_a, TM, c.nl_a, c.n_a, 1, s));
        }
        MARLC_TRY(e->chain(sp, s));  // the sweep needs dH_heads
        // parameter gradients of the heads: side streams, underneath the sweep (joined at the end)
        MARLC_TRY(head_bwd_params(e, "predict", e->buf("d_preds"), c.nb_class, e->buf("prd_s1"), Yq,
                                  H + (size_t)M * c.n_b, c.n_b, c.nl_b, sp));
        MARLC_TRY(e->chain(s, sc));  // dY_pol is produced on the main stream
        MARLC_TRY(head_bwd_params(e, "policy", e->buf("d_pol_logits"), c.n_actions, e->buf("pol_s1"), Yp,
                                  Hc + (size_t)M * c.n_a, c.n_a, c.nl_a, sc));
        MARLC_TRY(head_bwd_params(e, "critic", e->buf("d_values"), 1, e->buf("cri_s1"), Yc, Hc + (size_t)M * c.n_a,
                                  c.n_a, c.nl_a, sc));
    } else {
        MARLC_TRY(head_bwd(e, "predict", e->buf("d_preds"), c.nb_class, e->buf("prd_s1"), e->buf("prd_y1"),
                           H + (size_t)M * c.n_b, c.n_b, c.nl_b, e->buf("dH_heads"), 0, s, 1));
        MARLC_TRY(policy_logit_grad(e->buf("d_logp"), e->buf("probs"), e->buf<int>("act"), e->buf("d_pol_logits"), TM,
                                    c.n_actions, s, d_probs));
        MARLC_TRY(head_bwd(e, "policy", e->buf("d_pol_logits"), c.n_actions, e->buf("pol_s1"), e->buf("pol_y1"),
                           Hc + (size_t)M * c.n_a, c.n_a, c.nl_a, e->buf("dHc_heads"), 0, s));
        MARLC_TRY(head_bwd(e, "critic", e->buf("d_values"), 1, e->buf("cri_s1"), e->buf("cri_y1"), Hc + (size_t)M * c.n_a,
                           c.n_a, c.nl_a, e->buf("dHc_heads"), 1, s));
    }

    }  // heads
    auto join_sides = [&]() -> int {  // early (profiling) exits must not leave forked work unjoined
        if (!c.use_chains) return 0;
        MARLC_TRY(e->chain(e->side[0], s));
        MARLC_TRY(e->chain(e->side[1], s));
        return 0;
    };
    if (e->debug_stop == 1) { MARLC_TRY(join_sides()); e->last_launches = g_launch_count - start; return 0; }
    // ---- weight gradients of steps [t0, t1), batched over their (t1-t0)*M rows (the reduction
    //      dimension).  Three independent branches on three streams: LSTM (sL) | encoder / decoder /
    //      position features (s1) | feature extractor (s0).  With the fused chains they run once the
    //      sweep (high-priority stream) is done.  Overlapping them with the sweep in chunks of time steps
    //      was measured at C2: 2 and 4 chunks take the same time (the overlapped launches delay the sweep
    //      as much as they save), 8 are slower.
    const bool par = c.use_chains != 0;
    auto batched = [&](int t0, int t1, cudaStream_t sL, cudaStream_t s1, cudaStream_t s0) -> int {
        NvtxRange nvtx_batched("marlc/backward/batched_grads");
        const size_t r0 = (size_t)t0 * M;       // first row of the chunk
        const int R = (t1 - t0) * M;            // rows in the chunk
        if (R <= 0) return 0;
        {
            const float* dgb = e->buf("dgates_b") + r0 * 4 * c.n_b;
            const float* dga = e->buf("dgates_a") + r0 * 4 * c.n_a;
            const float* Ur = e->buf("U") + r0 * Kin;
            const std::string pb = LSTM_B, pa = LSTM_A;
            const TnProblem ih[2] = {{dgb, 4L * c.n_b, Ur, Kin, e->grd(pb + "weight_ih"), Kin, R, 4 * c.n_b, Kin},
                                     {dga, 4L * c.n_a, Ur, Kin, e->grd(pa + "weight_ih"), Kin, R, 4 * c.n_a, Kin}};
            const TnProblem hh[2] = {{dgb, 4L * c.n_b, H + r0 * c.n_b, c.n_b, e->grd(pb + "weight_hh"), c.n_b, R, 4 * c.n_b, c.n_b},
                                     {dga, 4L * c.n_a, Hc + r0 * c.n_a, c.n_a, e->grd(pa + "weight_hh"), c.n_a, R, 4 * c.n_a, c.n_a}};
            MARLC_TRY(G_tn_group(e, ih, 2, sL));
            MARLC_TRY(G_tn_group(e, hh, 2, sL));
            MARLC_TRY(colsum_add2(dgb, 4 * c.n_b, e->grd(pb + "bias_ih"), e->grd(pb + "bias_hh"), R, 4 * c.n_b, sL));
            MARLC_TRY(colsum_add2(dga, 4 * c.n_a, e->grd(pa + "bias_ih"), e->grd(pa + "bias_hh"), R, 4 * c.n_a, sL));
        }
        {
            const int Re = (std::min(t1, d_msg_out ? T : T - 1) - t0) * M;  // an episode's last message is never consumed
            const TnProblem enc[2] = {
                {e->buf("d_enc_y2") + r0 * c.n_m, c.n_m, e->buf("enc_s1") + r0 * 2 * c.n_m, 2L * c.n_m,
                 e->grd("encode_msg.3.weight"), 2L * c.n_m, Re, c.n_m, 2 * c.n_m},
                {e->buf("d_enc_y1") + r0 * 2 * c.n_m, 2L * c.n_m, H + (r0 + M) * c.n_b, c.n_b,
                 e->grd("encode_msg.0.weight"), c.n_b, Re, 2 * c.n_m, c.n_b}};
            if (Re > 0) MARLC_TRY(G_tn_group(e, enc, 2, s1));
            const TnProblem dec[2] = {
                {e->buf("d_dec_y2") + r0 * c.n_m_o, c.n_m_o, e->buf("dec_s1") + r0 * 2 * c.n_m, 2L * c.n_m,
                 e->grd("decode_msg.3.weight"), 2L * c.n_m, R, c.n_m_o, 2 * c.n_m},
                {e->buf("d_dec_y1") + r0 * 2 * c.n_m, 2L * c.n_m, e->buf("coll") + r0 * c.n_m, c.n_m,
                 e->grd("decode_msg.0.weight"), c.n_m, R, 2 * c.n_m, c.n_m}};
            MARLC_TRY(G_tn_group(e, dec, 2, s1));
        }
        // position features (state.py:13-17)
        MARLC_TRY(block_bwd_norm(e, "map_pos", 0, dU + r0 * Kin + F + c.n_m_o, Kin, e->buf("pos_y") + r0 * c.n_d, R, c.n_d,
                                 e->buf("d_pos_y") + r0 * c.n_d, s1));
        MARLC_TRY(G_tn(e, e->buf("d_pos_y") + r0 * c.n_d, c.n_d, e->buf("npos") + r0 * 2, 2, e->grd("map_pos.0.weight"), 2,
                       R, c.n_d, 2, s1));
        // feature extractor: layer-wise, batched over the chunk's windows (cnn_backward_layers); every conv product
        // (input gradient dCol_l = dY_l W_l, weight gradient dW_l = dY_l^T col_l) is a tensor-core GEMM
        const CnnDesc& d = e->cnn;
        CnnWindows win{img, e->buf<int>("pos_hist") + r0 * 2, se ? se->patch : nullptr, M, c.nb, c.C, c.H, c.W, c.f};
        if (win.patch) win.patch += r0 * c.C * c.f * c.f;
        if (!par) {  // unfused reference path: one whole-episode call of the per-window kernel
            const float* ysave[MAX_CNN_LAYERS];
            CnnBwdBuffers bb;
            for (int l = 0; l < e->L; ++l) {
                ysave[l] = e->buf("cnn_y" + std::to_string(l));
                bb.dY[l] = e->buf("cnn_dY" + std::to_string(l));
                bb.col[l] = e->buf("cnn_col" + std::to_string(l));
                bb.gnpart[l] = e->buf("cnn_gnpart" + std::to_string(l));
            }
            MARLC_TRY(cnn_bwd(e->cnn, win, 0, TM, ysave, dU, Kin, bb, s0));
            for (int l = 0; l < e->L; ++l) {
                const int npos = d.hout[l] * d.hout[l], kk = d.cin[l] * 9, co = d.cout[l];
                const std::string cw = CNN_PREFIX + std::to_string(3 * l), gn = CNN_PREFIX + std::to_string(3 * l + 1);
                MARLC_TRY(G_tn(e, bb.dY[l], co, bb.col[l], kk, e->grd(cw + ".weight"), kk, R * npos, co, kk, s0));
                MARLC_TRY(colsum_add(bb.dY[l], co, e->grd(cw + ".bias"), R * npos, co, s0));
                MARLC_TRY(colsum_add(bb.gnpart[l], 2 * co, e->grd(gn + ".weight"), R, co, s0));
                MARLC_TRY(colsum_add(bb.gnpart[l] + co, 2 * co, e->grd(gn + ".bias"), R, co, s0));
            }
            return 0;
        }
        CnnBwdLayers cb;
        memset(&cb, 0, sizeof(cb));
        cb.d = &d; cb.win = win; cb.P = R;
        cb.dOut = dU + r0 * Kin; cb.lddo = Kin;
        for (int l = 0; l < e->L; ++l) {
            const size_t npos = (size_t)d.hout[l] * d.hout[l];
            const std::string cw = CNN_PREFIX + std::to_string(3 * l), gn = CNN_PREFIX + std::to_string(3 * l + 1);
            cb.ysave[l] = e->buf("cnn_y" + std::to_string(l)) + r0 * e->cnn_sz[l];
            cb.dY[l] = e->buf("cnn_dY" + std::to_string(l)) + r0 * npos * d.cout[l];
            cb.col[l] = e->buf("cnn_col" + std::to_string(l)) + r0 * npos * (size_t)((d.cin[l] * 9 + 3) & ~3);
            if (l > 0) cb.dcol[l] = e->buf("cnn_dcol" + std::to_string(l)) + r0 * npos * d.cin[l] * 9;
            cb.d_w[l] = e->grd(cw + ".weight"); cb.d_b[l] = e->grd(cw + ".bias");
            cb.d_gn_w[l] = e->grd(gn + ".weight"); cb.d_gn_b[l] = e->grd(gn + ".bias");
        }
        return cnn_backward_layers(gemm_mode(e), cb, s0, s1, sL, e->next_event());
    };
    // ---- BPTT sweep
    NvtxRange nvtx_sweep("marlc/backward/sweep");
    float* dh = e->buf("dh");
    float* dhc = e->buf("dhc");
    float* dc[2] = {e->buf("dc0"), e->buf("dc1")};
    float* dcc[2] = {e->buf("dcc0"), e->buf("dcc1")};
    float* dmsg = e->buf("dmsg");
    float* tmpS = e->buf("tmpS");
    // carries into the last step: zero for an episode, d h' / d c' / d h^' / d c^' for a stand-alone step
    auto seed = [&](float* dst, int k, int n) -> int {
        const float* src = se ? se->d_out[k] : nullptr;
        if (src) MARLC_CUDA(cudaMemcpyAsync(dst, src, sizeof(float) * (size_t)M * n, cudaMemcpyDeviceToDevice, s));
        else MARLC_CUDA(cudaMemsetAsync(dst, 0, sizeof(float) * (size_t)M * n, s));
        return 0;
    };
    MARLC_TRY(seed(dh, 4, c.n_b));
    MARLC_TRY(seed(dhc, 6, c.n_a));
    MARLC_TRY(seed(dc[0], 5, c.n_b));
    MARLC_TRY(seed(dcc[0], 7, c.n_a));
    int cur = 0;
    const bool chain_sweep = sweep_chained(e);  // fused chain kernels, or one kernel per op from 4096 rows on
    if (chain_sweep) {
        float* dcoll = e->buf("dcoll");
        float* dh_hist = e->buf("dh_hist");
        float* dhc_hist = e->buf("dhc_hist");
        // split-K (atomicAdd) targets of the whole sweep are zeroed once, not once per step
        MARLC_CUDA(cudaMemsetAsync(dU, 0, sizeof(float) * (size_t)TM * Kin, s));
        MARLC_CUDA(cudaMemsetAsync(dh_hist, 0, sizeof(float) * (size_t)TM * c.n_b, s));
        MARLC_CUDA(cudaMemsetAsync(dhc_hist, 0, sizeof(float) * (size_t)TM * c.n_a, s));
        // the sweep moves to the high-priority stream; the caller's stream becomes the LSTM branch
        const bool profiling_stop = e->debug_stop == 2 || e->debug_stop == 21 || e->debug_stop == 22;
        cudaStream_t sw = e->hp, s0 = e->side[0], s1 = e->side[1];
        MARLC_TRY(e->chain(s, sw));
        for (int t = T - 1; t >= 0; --t) {
            float* dgb = e->buf("dgates_b") + (size_t)t * M * 4 * c.n_b;
            float* dga = e->buf("dgates_a") + (size_t)t * M * 4 * c.n_a;
            float* dgb_lo = e->lo_on ? e->buf("dgates_b_lo") : nullptr;
            float* dga_lo = e->lo_on ? e->buf("dgates_a_lo") : nullptr;
            // fused: adjoint mean + encoder backward + dh accumulation + both LSTM cells' point-wise backward
            BwdPreArgs bp;
            memset(&bp, 0, sizeof(bp));
            bp.dcoll = (t < T - 1) ? dcoll : nullptr;  // an episode's last message is never consumed
            bp.dmsg = (t == T - 1) ? d_msg_out : nullptr;
            bp.e0 = chain_lin(e, "encode_msg", 0, c.n_b, 2 * c.n_m, true);
            bp.e3 = chain_lin(e, "encode_msg", 3, 2 * c.n_m, c.n_m, true);
            bp.enc_y1 = e->buf("enc_y1") + (size_t)t * M * 2 * c.n_m;
            bp.enc_y2 = e->buf("enc_y2") + (size_t)t * M * c.n_m;
            bp.d_enc_y1 = e->buf("d_enc_y1") + (size_t)t * M * 2 * c.n_m;
            bp.d_enc_y2 = e->buf("d_enc_y2") + (size_t)t * M * c.n_m;
            bp.dh_carry[0] = (t < T - 1) ? dh_hist + (size_t)(t + 1) * M * c.n_b : se ? dh : nullptr;
            bp.dh_carry[1] = (t < T - 1) ? dhc_hist + (size_t)(t + 1) * M * c.n_a : se ? dhc : nullptr;
            bp.dh_heads[0] = e->buf("dH_heads") + (size_t)t * M * c.n_b;
            bp.dh_heads[1] = e->buf("dHc_heads") + (size_t)t * M * c.n_a;
            bp.dc_next[0] = (t < T - 1 || se) ? dc[cur] : nullptr;
            bp.dc_next[1] = (t < T - 1 || se) ? dcc[cur] : nullptr;
            bp.gates[0] = e->buf("gates_b") + (size_t)t * M * 4 * c.n_b;
            bp.gates[1] = e->buf("gates_a") + (size_t)t * M * 4 * c.n_a;
            bp.c_prev[0] = Cb + (size_t)t * M * c.n_b;
            bp.c_prev[1] = Cc + (size_t)t * M * c.n_a;
            bp.c_new[0] = Cb + (size_t)(t + 1) * M * c.n_b;
            bp.c_new[1] = Cc + (size_t)(t + 1) * M * c.n_a;
            bp.dgates[0] = dgb; bp.dgates[1] = dga;
            bp.dgates_lo[0] = dgb_lo; bp.dgates_lo[1] = dga_lo;
            bp.dc_prev[0] = dc[cur ^ 1]; bp.dc_prev[1] = dcc[cur ^ 1];
            bp.n[0] = c.n_b; bp.n[1] = c.n_a;
            bp.Na = c.na; bp.Nb = c.nb; bp.M = M; bp.n_m = c.n_m;
            {
                PdlScope pdl(t < T - 1);  // predecessor in `sw`: bwd_post of step t+1 (an event wait at t = T-1)
                MARLC_TRY(bwd_pre(bp, sw));
            }
            cur ^= 1;
            if (e->debug_stop == 21) continue;
            // input gradients: du = dg_b Wih_b + dg_a Wih_a ; dh = dg_b Whh_b ; dh^ = dg_a Whh_a  (ONE grouped launch)
            float* dUt = dU + (size_t)t * M * Kin;
            float* dh_t = dh_hist + (size_t)t * M * c.n_b;
            float* dhc_t = dhc_hist + (size_t)t * M * c.n_a;
            bool tc_dx = false;
            if (c.use_tc && c.n_a >= 16 && c.n_b >= 16) {
                TcGemmArgs g[3];
                g[0].A = tc_op_lo(dgb, dgb_lo, 4 * c.n_b); g[0].B = e->op(e->prm(std::string(LSTM_B) + "weight_ih"), Kin, true); g[0].K = 4 * c.n_b;
                g[0].A2 = tc_op_lo(dga, dga_lo, 4 * c.n_a); g[0].B2 = e->op(e->prm(std::string(LSTM_A) + "weight_ih"), Kin, true); g[0].K2 = 4 * c.n_a;
                g[0].C = dUt; g[0].ldc = Kin; g[0].M = M; g[0].N = Kin;
                g[1].A = tc_op_lo(dgb, dgb_lo, 4 * c.n_b); g[1].B = e->op(e->prm(std::string(LSTM_B) + "weight_hh"), c.n_b, true); g[1].K = 4 * c.n_b;
                g[1].C = dh_t; g[1].ldc = c.n_b; g[1].M = M; g[1].N = c.n_b;
                g[2].A = tc_op_lo(dga, dga_lo, 4 * c.n_a); g[2].B = e->op(e->prm(std::string(LSTM_A) + "weight_hh"), c.n_a, true); g[2].K = 4 * c.n_a;
                g[2].C = dhc_t; g[2].ldc = c.n_a; g[2].M = M; g[2].N = c.n_a;
                bool ok = true;
                for (int q = 0; q < 3; ++q) {
                    g[q].allow_split = 1; g[q].c_zeroed = 1; g[q].x3 = x3_of(e);
                    ok = ok && tc_operand_ok(g[q].A) && tc_operand_ok(g[q].B);
                }
                ok = ok && tc_operand_ok(g[0].A2) && tc_operand_ok(g[0].B2);
                if (ok) {
                    PdlScope pdl(1);
                    MARLC_TRY(tc_gemm_group(g, t > 0 || want_dh0 ? 3 : 1, sw));  // at t == 0 only a step's caller consumes dh / dh^
                    tc_dx = true;
                }
            }
            if (!tc_dx) {
                GemmGroup gg;
                memset(&gg, 0, sizeof(gg));
                gg.count = 3;
                {
                    GemmProblem& p = gg.p[0];
                    p.A = dgb; p.sam = 4 * c.n_b; p.sak = 1;
                    p.B = e->prm(std::string(LSTM_B) + "weight_ih"); p.sbk = Kin; p.sbn = 1;
                    p.A2 = dga; p.sam2 = 4 * c.n_a; p.sak2 = 1;
                    p.B2 = e->prm(std::string(LSTM_A) + "weight_ih"); p.sbk2 = Kin; p.sbn2 = 1;
                    p.C = dUt; p.ldc = Kin;
                    p.M = M; p.N = Kin; p.K = 4 * c.n_b; p.K2 = 4 * c.n_a;
                }
                {
                    GemmProblem& p = gg.p[1];
                    p.A = dgb; p.sam = 4 * c.n_b; p.sak = 1;
                    p.B = e->prm(std::string(LSTM_B) + "weight_hh"); p.sbk = c.n_b; p.sbn = 1;
                    p.C = dh_t; p.ldc = c.n_b;
                    p.M = M; p.N = c.n_b; p.K = 4 * c.n_b;
                }
                {
                    GemmProblem& p = gg.p[2];
                    p.A = dga; p.sam = 4 * c.n_a; p.sak = 1;
                    p.B = e->prm(std::string(LSTM_A) + "weight_hh"); p.sbk = c.n_a; p.sbn = 1;
                    p.C = dhc_t; p.ldc = c.n_a;
                    p.M = M; p.N = c.n_a; p.K = 4 * c.n_a;
                }
                MARLC_TRY(gemm_group(gg, sw));
            }
            // fused decoder backward (models.py:97-98) -> dcoll for step t-1
            if (e->debug_stop == 22) continue;
            BwdPostArgs bq;
            memset(&bq, 0, sizeof(bq));
            bq.dU = dUt; bq.ldu = Kin; bq.F = F;
            bq.d0 = chain_lin(e, "decode_msg", 0, c.n_m, 2 * c.n_m, true);
            bq.d3 = chain_lin(e, "decode_msg", 3, 2 * c.n_m, c.n_m_o, true);
            bq.dec_y1 = e->buf("dec_y1") + (size_t)t * M * 2 * c.n_m;
            bq.dec_y2 = e->buf("dec_y2") + (size_t)t * M * c.n_m_o;
            bq.d_dec_y1 = e->buf("d_dec_y1") + (size_t)t * M * 2 * c.n_m;
            bq.d_dec_y2 = e->buf("d_dec_y2") + (size_t)t * M * c.n_m_o;
            bq.dcoll = (t > 0 || want_dmsg0) ? dcoll : nullptr;
            bq.M = M; bq.n_m = c.n_m; bq.n_m_o = c.n_m_o;
            {
                PdlScope pdl(1);
                MARLC_TRY(bwd_post(bq, sw));
            }
        }
        if (!profiling_stop) {  // every step's gradients are final
            cudaEvent_t done = e->next_event();
            MARLC_CUDA(cudaEventRecord(done, sw));
            MARLC_CUDA(cudaStreamWaitEvent(s, done, 0));
            MARLC_CUDA(cudaStreamWaitEvent(s0, done, 0));
            MARLC_CUDA(cudaStreamWaitEvent(s1, done, 0));
            MARLC_TRY(batched(0, T, s, s1, s0));
        }
        MARLC_TRY(e->chain(sw, s));
    } else
    for (int t = T - 1; t >= 0; --t) {
        if (t < T - 1 || d_msg_out) {
            // message produced at step t was consumed at t+1 (or has a gradient of its own): encoder backward
            // (models.py:114-116)
            float* dy2 = e->buf("d_enc_y2") + (size_t)t * M * c.n_m;
            float* dy1 = e->buf("d_enc_y1") + (size_t)t * M * 2 * c.n_m;
            MARLC_TRY(block_bwd_norm(e, "encode_msg", 3, t < T - 1 ? dmsg : d_msg_out, c.n_m,
                                     e->buf("enc_y2") + (size_t)t * M * c.n_m, M, c.n_m, dy2, s));
            MARLC_TRY(G_nn(e, dy2, c.n_m, e->prm("encode_msg.3.weight"), 2 * c.n_m, tmpS, 2 * c.n_m, M, c.n_m,
                              2 * c.n_m, 0, s));
            MARLC_TRY(block_bwd_norm(e, "encode_msg", 0, tmpS, 2 * c.n_m,
                                     e->buf("enc_y1") + (size_t)t * M * 2 * c.n_m, M, 2 * c.n_m, dy1, s));
            MARLC_TRY(G_nn(e, dy1, 2 * c.n_m, e->prm("encode_msg.0.weight"), c.n_b, dh, c.n_b, M, 2 * c.n_m, c.n_b, 1, s));
        }
        float* dgb = e->buf("dgates_b") + (size_t)t * M * 4 * c.n_b;
        float* dga = e->buf("dgates_a") + (size_t)t * M * 4 * c.n_a;
        MARLC_TRY(lstm_cell_bwd(dh, e->buf("dH_heads") + (size_t)t * M * c.n_b, dc[cur],
                                e->buf("gates_b") + (size_t)t * M * 4 * c.n_b, Cb + (size_t)t * M * c.n_b,
                                Cb + (size_t)(t + 1) * M * c.n_b, dgb, dc[cur ^ 1], M, c.n_b, s));
        MARLC_TRY(lstm_cell_bwd(dhc, e->buf("dHc_heads") + (size_t)t * M * c.n_a, dcc[cur],
                                e->buf("gates_a") + (size_t)t * M * 4 * c.n_a, Cc + (size_t)t * M * c.n_a,
                                Cc + (size_t)(t + 1) * M * c.n_a, dga, dcc[cur ^ 1], M, c.n_a, s));
        cur ^= 1;
        // input gradients: du = dg_b Wih_b + dg_a Wih_a ; dh = dg_b Whh_b ; dh^ = dg_a Whh_a
        float* dUt = dU + (size_t)t * M * Kin;
        bool tc_dx = false;
        if (c.use_tc) {
            TcGemmArgs a;
            a.A = tc_op(dgb, 4 * c.n_b); a.B = tc_op(e->prm(std::string(LSTM_B) + "weight_ih"), Kin, true); a.K = 4 * c.n_b;
            a.A2 = tc_op(dga, 4 * c.n_a); a.B2 = tc_op(e->prm(std::string(LSTM_A) + "weight_ih"), Kin, true); a.K2 = 4 * c.n_a;
            a.C = dUt; a.ldc = Kin; a.M = M; a.N = Kin; a.allow_split = 1;
            TcGemmArgs b;
            b.A = tc_op(dgb, 4 * c.n_b); b.B = tc_op(e->prm(std::string(LSTM_B) + "weight_hh"), c.n_b, true); b.K = 4 * c.n_b;
            b.C = dh; b.ldc = c.n_b; b.M = M; b.N = c.n_b; b.allow_split = 1;
            TcGemmArgs d;
            d.A = tc_op(dga, 4 * c.n_a); d.B = tc_op(e->prm(std::string(LSTM_A) + "weight_hh"), c.n_a, true); d.K = 4 * c.n_a;
            d.C = dhc; d.ldc = c.n_a; d.M = M; d.N = c.n_a; d.allow_split = 1;
            a.x3 = b.x3 = d.x3 = x3_of(e);
            if (tc_operand_ok(a.A) && tc_operand_ok(a.B) && tc_operand_ok(a.A2) && tc_operand_ok(a.B2) &&
                tc_operand_ok(b.B) && tc_operand_ok(d.B) && c.n_a >= 16 && c.n_b >= 16) {
                MARLC_TRY(tc_gemm(a, s));
                MARLC_TRY(tc_gemm(b, s));
                MARLC_TRY(tc_gemm(d, s));
                tc_dx = true;
            }
        }
        if (!tc_dx) {
        GemmGroup gg;
        memset(&gg, 0, sizeof(gg));
        gg.count = 3;
        {
            GemmProblem& p = gg.p[0];
            p.A = dgb; p.sam = 4 * c.n_b; p.sak = 1;
            p.B = e->prm(std::string(LSTM_B) + "weight_ih"); p.sbk = Kin; p.sbn = 1;
            p.A2 = dga; p.sam2 = 4 * c.n_a; p.sak2 = 1;
            p.B2 = e->prm(std::string(LSTM_A) + "weight_ih"); p.sbk2 = Kin; p.sbn2 = 1;
            p.C = dUt; p.ldc = Kin;
            p.M = M; p.N = Kin; p.K = 4 * c.n_b; p.K2 = 4 * c.n_a;
        }
        {
            GemmProblem& p = gg.p[1];
            p.A = dgb; p.sam = 4 * c.n_b; p.sak = 1;
            p.B = e->prm(std::string(LSTM_B) + "weight_hh"); p.sbk = c.n_b; p.sbn = 1;
            p.C = dh; p.ldc = c.n_b;
            p.M = M; p.N = c.n_b; p.K = 4 * c.n_b;
        }
        {
            GemmProblem& p = gg.p[2];
            p.A = dga; p.sam = 4 * c.n_a; p.sak = 1;
            p.B = e->prm(std::string(LSTM_A) + "weight_hh"); p.sbk = c.n_a; p.sbn = 1;
            p.C = dhc; p.ldc = c.n_a;
            p.M = M; p.N = c.n_a; p.K = 4 * c.n_a;
        }
        MARLC_TRY(gemm_group(gg, s));
        }
        // decoder backward (models.py:97-98); at t == 0 the input message is the constant zero
        float* ddy2 = e->buf("d_dec_y2") + (size_t)t * M * c.n_m_o;
        float* ddy1 = e->buf("d_dec_y1") + (size_t)t * M * 2 * c.n_m;
        MARLC_TRY(block_bwd_norm(e, "decode_msg", 3, dUt + F, Kin, e->buf("dec_y2") + (size_t)t * M * c.n_m_o, M,
                                 c.n_m_o, ddy2, s));
        MARLC_TRY(G_nn(e, ddy2, c.n_m_o, e->prm("decode_msg.3.weight"), 2 * c.n_m, tmpS, 2 * c.n_m, M, c.n_m_o,
                          2 * c.n_m, 0, s));
        MARLC_TRY(block_bwd_norm(e, "decode_msg", 0, tmpS, 2 * c.n_m, e->buf("dec_y1") + (size_t)t * M * 2 * c.n_m, M,
                                 2 * c.n_m, ddy1, s));
        if (t > 0 || want_dmsg0) {
            MARLC_TRY(G_nn(e, ddy1, 2 * c.n_m, e->prm("decode_msg.0.weight"), c.n_m, e->buf("dcoll"), c.n_m, M,
                              2 * c.n_m, c.n_m, 0, s));
            if (t > 0) MARLC_TRY(msg_mean(e->buf("dcoll"), dmsg, c.na, c.nb, c.n_m, s));  // symmetric operator = own adjoint
        }
    }
    if (se) {  // inner end: the gradients that leave through the step's inputs
        auto emit = [&](int k, const float* src, int n) -> int {
            if (se->d_in[k])
                MARLC_CUDA(cudaMemcpyAsync(se->d_in[k], src, sizeof(float) * (size_t)M * n, cudaMemcpyDeviceToDevice, s));
            return 0;
        };
        MARLC_TRY(emit(1, chain_sweep ? e->buf("dh_hist") : dh, c.n_b));
        MARLC_TRY(emit(2, dc[cur], c.n_b));
        MARLC_TRY(emit(3, chain_sweep ? e->buf("dhc_hist") : dhc, c.n_a));
        MARLC_TRY(emit(4, dcc[cur], c.n_a));
        // d msg = adjoint message mean of the decoder's input gradient (zero with one agent, message.py:12-17)
        if (want_dmsg0) MARLC_TRY(msg_mean(e->buf("dcoll"), se->d_in[0], c.na, c.nb, c.n_m, s));
    }

    if (e->debug_stop == 2 || e->debug_stop == 21 || e->debug_stop == 22) {
        MARLC_TRY(join_sides());
        e->last_launches = g_launch_count - start;
        return 0;
    }
    if (!par) MARLC_TRY(batched(0, T, s, s, s));
    if (par && !chain_sweep) {  // unfused sweep, batched gradients on the three streams as in the chain path
        MARLC_TRY(e->chain(s, e->side[0]));
        MARLC_TRY(e->chain(s, e->side[1]));
        MARLC_TRY(batched(0, T, s, e->side[1], e->side[0]));
    }
    if (par) MARLC_TRY(join_sides());  // dY0 included: the caller's stream is ordered after every side-stream launch
    e->dy0_owner = se ? marlc_engine::Dy0Owner::step : marlc_engine::Dy0Owner::episode;
    e->last_launches = g_launch_count - start;
    return 0;
}

extern "C" int marlc_episode_backward(marlc_engine* e, const float* img, int accumulate, void* stream) {
    MARLC_CHECK(img, "null image batch");
    return episode_backward(e, img, accumulate, nullptr, (cudaStream_t)stream);
}

// The backward of marlc_model_step.  Every step-wise call of one geometry shares this T = 1 engine's workspace,
// so the activations of the forward being differentiated are gone by now: the step is re-run from its inputs
// first.  Split-K reduce-adds are unordered, so the recomputed activations may differ from the forward's in the
// last bits.  The inputs are then copied into slot 0 of the state histories, where every read of step 0's
// inputs in the sweep finds them (weight_hh gradients, c_prev, position-feature weight gradient).
extern "C" int marlc_model_step_backward(marlc_engine* e, const float* patch, const float* msg, const float* npos,
                                         const float* const* hidden, const float* const* d_out, float* const* d_in,
                                         float* grads, void* stream) {
    MARLC_CHECK(e && e->ws, "engine not bound");
    MARLC_CHECK(e->cfg.T == 1, "model_step_backward: needs a T = 1 engine (T = %d)", e->cfg.T);
    MARLC_CHECK(patch && msg && npos && hidden && hidden[0] && hidden[1] && hidden[2] && hidden[3],
                "model_step_backward: null input");
    MARLC_CHECK(d_out && d_in && grads, "model_step_backward: null gradient array / buffer");
    NvtxRange nvtx_step_bwd("marlc/model_step_backward");
    cudaStream_t s = (cudaStream_t)stream;
    const marlc_config& c = e->cfg;
    const size_t M = e->M;
    const int start = g_launch_count;
    MARLC_TRY(model_step_fwd(e, patch, msg, npos, hidden, s));
    const struct { float* dst; const float* src; size_t n; } in[6] = {
        {e->buf("H"), hidden[0], M * c.n_b}, {e->buf("Cb"), hidden[1], M * c.n_b},
        {e->buf("Hc"), hidden[2], M * c.n_a}, {e->buf("Cc"), hidden[3], M * c.n_a},
        {e->buf("msg"), msg, M * c.n_m}, {e->buf("npos"), npos, M * 2}};
    for (const auto& x : in)
        MARLC_CUDA(cudaMemcpyAsync(x.dst, x.src, sizeof(float) * x.n, cudaMemcpyDeviceToDevice, s));
    // the heads' seeds: d values / d preds as given (zero when absent); d probs replaces d log p (kept zero)
    const struct { float* dst; const float* src; size_t n; } head[3] = {
        {e->buf("d_values"), d_out[1], M}, {e->buf("d_preds"), d_out[2], M * c.nb_class}, {e->buf("d_logp"), nullptr, M}};
    for (const auto& x : head) {
        if (x.src) MARLC_CUDA(cudaMemcpyAsync(x.dst, x.src, sizeof(float) * x.n, cudaMemcpyDeviceToDevice, s));
        else MARLC_CUDA(cudaMemsetAsync(x.dst, 0, sizeof(float) * x.n, s));
    }
    // the parameter gradients go to the caller's buffer for the duration of the call
    struct GradBase {
        marlc_engine* e;
        float* saved;
        ~GradBase() { e->G = saved; }
    } base{e, e->G};
    e->G = grads;
    const StepEnds se{patch, d_out, d_in};
    MARLC_TRY(episode_backward(e, nullptr, 0, &se, s));
    e->last_launches = g_launch_count - start;
    return 0;
}

// d img of the last rollout from cnn_dY0 (see include/marlc.h).  The first conv layer's weights are read as they
// are now: call it before the parameters change.
extern "C" int marlc_episode_image_grad(marlc_engine* e, float* d_img, void* stream) {
    MARLC_CHECK(e && e->ws, "engine not bound");
    MARLC_CHECK(d_img, "episode_image_grad: null output");
    MARLC_CHECK(e->dy0_owner == marlc_engine::Dy0Owner::episode,
                "episode_image_grad: no complete marlc_episode_backward of the engine's last rollout (none since the "
                "last forward / model step, a step-wise backward, or a backward cut short by marlc_engine_debug_stop)");
    const marlc_config& c = e->cfg;
    ImageGradArgs a;
    a.dY0 = e->buf("cnn_dY0");
    a.w0 = e->cnn.w[0];
    a.pos_hist = e->buf<int>("pos_hist");
    a.d_img = d_img;
    a.T = c.T; a.Na = c.na; a.B = c.nb; a.C = c.C; a.H = c.H; a.W = c.W; a.f = c.f;
    a.cin = e->cnn.cin[0]; a.cout = e->cnn.cout[0]; a.ho = e->cnn.hout[0];
    NvtxRange nvtx("marlc/image_grad");
    return cnn_image_grad(a, (cudaStream_t)stream);
}

// d patch / d npos of the last marlc_model_step_backward from cnn_dY0 / d_pos_y (see include/marlc.h).  The
// first conv layer's and map_pos.0's weights are read as they are now: call it before the parameters change.
extern "C" int marlc_model_step_input_grad(marlc_engine* e, float* d_patch, float* d_npos, void* stream) {
    MARLC_CHECK(e, "model_step_input_grad: null engine");
    MARLC_CHECK(d_patch || d_npos, "model_step_input_grad: both outputs are null");
    MARLC_CHECK(e->ws, "engine not bound");
    MARLC_CHECK(e->dy0_owner == marlc_engine::Dy0Owner::step,
                "model_step_input_grad: no complete marlc_model_step_backward since the last forward / model step / "
                "episode backward (or a backward cut short by marlc_engine_debug_stop)");
    const marlc_config& c = e->cfg;
    cudaStream_t s = (cudaStream_t)stream;
    NvtxRange nvtx("marlc/model_step_input_grad");
    if (d_patch) {
        PatchGradArgs a;
        a.dY0 = e->buf("cnn_dY0");
        a.w0 = e->cnn.w[0];
        a.d_patch = d_patch;
        a.M = e->M; a.C = c.C; a.f = c.f;
        a.cin = e->cnn.cin[0]; a.cout = e->cnn.cout[0]; a.ho = e->cnn.hout[0];
        MARLC_TRY(cnn_patch_grad(a, s));
    }
    // map_pos.0 is Linear(2, n_d): d npos[M,2] = d_pos_y[M,n_d] . W[n_d,2] (pitch 2: the FFMA back end)
    if (d_npos)
        MARLC_TRY(G_nn(e, e->buf("d_pos_y"), c.n_d, e->prm("map_pos.0.weight"), 2, d_npos, 2, e->M, c.n_d, 2, 0, s));
    return 0;
}

extern "C" int marlc_engine_last_launches(const marlc_engine* e) { return e->last_launches; }
extern "C" long marlc_gemm_launch_count(int ffma) { return ffma ? marlc::g_simt_gemm_launches : marlc::g_tc_gemm_launches; }

// ---- standalone operators ----------------------------------------------------
extern "C" int marlc_patch_gather(const float* img, const int64_t* pos, float* obs, int Na, int B, int C, int H, int W,
                                  int f, void* stream) {
    MARLC_CHECK(img && pos && obs, "patch_gather: null pointer");
    return patch_gather_i64(img, pos, obs, Na, B, C, H, W, f, (cudaStream_t)stream);
}
extern "C" int marlc_patch_gather_backward(const float* d_obs, const int64_t* pos, float* d_img, int Na, int B, int C,
                                           int H, int W, int f, void* stream) {
    MARLC_CHECK(d_obs && pos && d_img, "patch_gather_backward: null pointer");
    return patch_gather_backward_i64(d_obs, pos, d_img, Na, B, C, H, W, f, (cudaStream_t)stream);
}
extern "C" int marlc_transition(int64_t* pos, const int64_t* act, const int64_t* table, int nA, int M, int f, int H,
                                int W, float* norm_pos, int* err_flag, void* stream) {
    MARLC_CHECK(pos && act && table, "transition: null pointer");
    return transition_i64(pos, act, table, nA, M, f, H, W, norm_pos, err_flag, (cudaStream_t)stream);
}
extern "C" int marlc_normalized_positions(const int64_t* pos, float* out, int M, int H, int W, void* stream) {
    MARLC_CHECK(pos && out, "normalized_positions: null pointer");
    return normalized_positions_i64(pos, out, M, H, W, (cudaStream_t)stream);
}
extern "C" int marlc_linear(const float* X, const float* W, const float* bias, float* Y, int M, int N, int K,
                            void* stream) {
    return gemm_nt(X, K, W, K, bias, Y, N, M, N, K, 0, (cudaStream_t)stream);
}
extern "C" int marlc_ln_silu(const float* Y, const float* gamma, const float* beta, float* S, int R, int N,
                             void* stream) {
    return ln_silu_fwd(Y, N, gamma, beta, S, N, R, N, (cudaStream_t)stream);
}
extern "C" int marlc_msg_mean(const float* msg, float* out, int Na, int Nb, int n, void* stream) {
    return msg_mean(msg, out, Na, Nb, n, (cudaStream_t)stream);
}

// Description of a stand-alone feature extractor (no engine) from the caller's host arrays; the shapes are checked
static int standalone_cnn_desc(CnnDesc& d, const char* who, int layers, const int* cin, const int* cout,
                               const int* groups, int f, int img_c, const float* const* w, const float* const* b,
                               const float* const* gn_w, const float* const* gn_b) {
    MARLC_CHECK(layers >= 1 && layers <= MAX_CNN_LAYERS, "%s: %d layers unsupported", who, layers);
    MARLC_CHECK(cin && cout && groups && w && b && gn_w && gn_b, "%s: null pointer", who);
    memset(&d, 0, sizeof(d));
    d.L = layers; d.f = f; d.img_c = img_c;
    int h = f;
    for (int l = 0; l < layers; ++l) {
        MARLC_CHECK(cin[l] >= 1 && cout[l] >= 1 && groups[l] >= 1 && cout[l] % groups[l] == 0 &&
                        (l == 0 || cin[l] == cout[l - 1]),
                    "%s: bad shape of layer %d (cin %d, cout %d, groups %d)", who, l, cin[l], cout[l], groups[l]);
        d.cin[l] = cin[l]; d.cout[l] = cout[l]; d.groups[l] = groups[l];
        d.hin[l] = h; h = (h - 1) / 2 + 1; d.hout[l] = h;
        d.w[l] = w[l]; d.b[l] = b[l]; d.gn_w[l] = gn_w[l]; d.gn_b[l] = gn_b[l];
    }
    MARLC_CHECK(f >= 1 && img_c >= cin[0], "%s: window %d x %d with %d channels, the first layer reads %d", who, f, f,
                img_c, cin[0]);
    d.out_size = d.cout[layers - 1] * h * h;
    return 0;
}

// _Generic2dCnnModule.forward, vision.py:47-49 on N stand-alone windows [N, img_c, f, f]
extern "C" int marlc_cnn_forward_save(int layers, const int* cin, const int* cout, const int* groups, int f, int img_c,
                                      const float* const* w, const float* const* b, const float* const* gn_w,
                                      const float* const* gn_b, const float* patch, float* const* y_save, float* out,
                                      int N, void* stream) {
    CnnDesc d;
    MARLC_TRY(standalone_cnn_desc(d, "cnn_forward", layers, cin, cout, groups, f, img_c, w, b, gn_w, gn_b));
    MARLC_CHECK(patch && out, "cnn_forward: null pointer");
    return cnn_fwd(d, nullptr, nullptr, patch, 1, f, f, N, y_save, out, d.out_size, (cudaStream_t)stream);
}
extern "C" int marlc_cnn_forward(int layers, const int* cin, const int* cout, const int* groups, int f, int img_c,
                                 const float* const* w, const float* const* b, const float* const* gn_w,
                                 const float* const* gn_b, const float* patch, float* out, int N, void* stream) {
    return marlc_cnn_forward_save(layers, cin, cout, groups, f, img_c, w, b, gn_w, gn_b, patch, nullptr, out, N, stream);
}

// Workspace of marlc_cnn_backward: 256-byte aligned sections, per layer dY [N*ho^2, cout], dCol (l > 0)
// [N*ho^2, cin*9], with parameter gradients the im2col rows col [N*ho^2, pitch] (pitch round_up(cin*9, 4) for the
// first layer, cin*9 above), and 3 x cout floats of accumulation targets for the conv-bias / GroupNorm-affine
// gradients the caller did not ask for (the layer kernel always accumulates them).
struct CnnBwdWorkspace {
    size_t dY[MAX_CNN_LAYERS], dcol[MAX_CNN_LAYERS], col[MAX_CNN_LAYERS], scratch[MAX_CNN_LAYERS];
    size_t bytes;
};
static CnnBwdWorkspace cnn_bwd_workspace(const CnnDesc& d, long N, bool param_grads) {
    CnnBwdWorkspace ws;
    memset(&ws, 0, sizeof(ws));
    auto take = [&](size_t floats) {
        const size_t at = ws.bytes;
        ws.bytes += (floats * sizeof(float) + 255) / 256 * 256;
        return at;
    };
    for (int l = 0; l < d.L; ++l) {
        const size_t rows = (size_t)N * d.hout[l] * d.hout[l], kk = (size_t)d.cin[l] * 9;
        ws.dY[l] = take(rows * d.cout[l]);
        if (l > 0) ws.dcol[l] = take(rows * kk);
        if (param_grads) ws.col[l] = take(rows * (l == 0 ? (kk + 3) & ~(size_t)3 : kk));
        ws.scratch[l] = take(3 * (size_t)d.cout[l]);
    }
    return ws;
}

extern "C" size_t marlc_cnn_backward_workspace_bytes(int layers, const int* cin, const int* cout, int f, int N,
                                                     int want_param_grads) {
    // 0 = bad argument: a valid request always includes the scratch targets
    if (!(layers >= 1 && layers <= MAX_CNN_LAYERS && cin && cout && f >= 1 && N >= 0)) {
        set_error("cnn_backward_workspace_bytes: bad argument (layers %d, f %d, N %d)", layers, f, N);
        return 0;
    }
    CnnDesc d;
    memset(&d, 0, sizeof(d));
    d.L = layers;
    for (int l = 0, h = f; l < layers; ++l) {
        if (cin[l] < 1 || cout[l] < 1) {
            set_error("cnn_backward_workspace_bytes: bad shape of layer %d (cin %d, cout %d)", l, cin[l], cout[l]);
            return 0;
        }
        d.cin[l] = cin[l]; d.cout[l] = cout[l];
        h = (h - 1) / 2 + 1; d.hout[l] = h;
    }
    return cnn_bwd_workspace(d, N, want_param_grads != 0).bytes;
}

// Backward of marlc_cnn_forward_save on the caller's windows: the layer-wise path of the episode backward
// (cnn_backward_layers) on one stream, in 3xTF32 on the tensor cores where operands are TMA-addressable, then the
// first layer's transposed convolution into d_patch (see include/marlc.h).
extern "C" int marlc_cnn_backward(int layers, const int* cin, const int* cout, const int* groups, int f, int img_c,
                                  const float* const* w, const float* const* b, const float* const* gn_w,
                                  const float* const* gn_b, const float* patch, const float* const* y_save,
                                  const float* d_out, int N, void* workspace, size_t workspace_bytes, float* d_patch,
                                  float* const* d_w, float* const* d_b, float* const* d_gn_w,
                                  float* const* d_gn_b, void* stream) {
    CnnDesc d;
    MARLC_TRY(standalone_cnn_desc(d, "cnn_backward", layers, cin, cout, groups, f, img_c, w, b, gn_w, gn_b));
    MARLC_CHECK(N >= 0 && (long)N * d.hout[0] * d.hout[0] <= INT32_MAX, "cnn_backward: %d windows unsupported", N);
    MARLC_CHECK(y_save && workspace, "cnn_backward: null pointer");
    if (N == 0) return 0;
    MARLC_CHECK(patch && d_out, "cnn_backward: null pointer");
    bool param_grads = false;
    for (int l = 0; l < layers; ++l) {
        MARLC_CHECK(w[l] && b[l] && gn_w[l] && gn_b[l] && y_save[l], "cnn_backward: null pointer (layer %d)", l);
        param_grads = param_grads || (d_w && d_w[l]);
    }
    const CnnBwdWorkspace ws = cnn_bwd_workspace(d, N, param_grads);
    MARLC_CHECK((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "cnn_backward: workspace not 256-byte aligned");
    MARLC_CHECK(workspace_bytes >= ws.bytes,
                "cnn_backward: workspace of %zu bytes, need %zu (marlc_cnn_backward_workspace_bytes with "
                "want_param_grads = %d)", workspace_bytes, ws.bytes, param_grads ? 1 : 0);
    char* base = static_cast<char*>(workspace);
    CnnBwdLayers cb;
    memset(&cb, 0, sizeof(cb));
    cb.d = &d; cb.win = CnnWindows{nullptr, nullptr, patch, N, 1, img_c, f, f, f}; cb.P = N;
    cb.dOut = d_out; cb.lddo = d.out_size;
    for (int l = 0; l < layers; ++l) {
        float* scratch = reinterpret_cast<float*>(base + ws.scratch[l]);
        cb.ysave[l] = y_save[l];
        cb.dY[l] = reinterpret_cast<float*>(base + ws.dY[l]);
        cb.dcol[l] = l > 0 ? reinterpret_cast<float*>(base + ws.dcol[l]) : nullptr;
        cb.col[l] = param_grads ? reinterpret_cast<float*>(base + ws.col[l]) : nullptr;
        cb.d_w[l] = d_w ? d_w[l] : nullptr;
        cb.d_b[l] = (d_b && d_b[l]) ? d_b[l] : scratch + 2 * d.cout[l];
        cb.d_gn_w[l] = (d_gn_w && d_gn_w[l]) ? d_gn_w[l] : scratch;
        cb.d_gn_b[l] = (d_gn_b && d_gn_b[l]) ? d_gn_b[l] : scratch + d.cout[l];
    }
    // every launcher's host-side checks before the first launch
    for (int l = layers - 1; l >= 0; --l) {
        CnnBwdLayerArgs la;
        memset(&la, 0, sizeof(la));
        la.cout = d.cout[l]; la.ho = d.hout[l]; la.P = N;
        la.dOut = l == layers - 1 ? d_out : nullptr;
        la.ho_next = l == layers - 1 ? 1 : d.hout[l + 1];
        la.d_gn_w = cb.d_gn_w[l]; la.d_gn_b = cb.d_gn_b[l]; la.d_conv_b = cb.d_b[l];
        MARLC_TRY(cnn_bwd_layer_check(la));
    }
    PatchGradArgs pg;
    pg.dY0 = cb.dY[0]; pg.w0 = d.w[0]; pg.d_patch = d_patch;
    pg.M = N; pg.C = img_c; pg.f = f; pg.cin = d.cin[0]; pg.cout = d.cout[0]; pg.ho = d.hout[0];
    if (d_patch) MARLC_TRY(cnn_patch_grad_check(pg));
    cudaStream_t s = (cudaStream_t)stream;
    NvtxRange nvtx("marlc/cnn_backward");
    MARLC_TRY(cnn_backward_layers(GemmMode{1, 1}, cb, s, s, s, nullptr));
    if (d_patch) MARLC_TRY(cnn_patch_grad(pg, s));
    return 0;
}

// Tensor-core GEMM, exposed for unit tests: C[M,N] (+)= A.B^T (+ A2.B2^T) (+ bias).
// a_mn / b_mn select MN-major operands ([K rows][M|N contiguous]) instead of K-major.
extern "C" int marlc_tc_gemm(const float* A, int64_t lda, int a_mn, const float* B, int64_t ldb, int b_mn,
                             const float* A2, int64_t lda2, const float* B2, int64_t ldb2, int K2, const float* bias,
                             float* C, int64_t ldc, int M, int N, int K, int accumulate, int allow_split, int x3, void* stream) {
    TcGemmArgs a;
    a.x3 = x3;
    a.A = tc_op(A, lda, a_mn != 0); a.B = tc_op(B, ldb, b_mn != 0); a.K = K;
    if (K2 > 0) { a.A2 = tc_op(A2, lda2, a_mn != 0); a.B2 = tc_op(B2, ldb2, b_mn != 0); a.K2 = K2; }
    a.C = C; a.ldc = ldc; a.M = M; a.N = N; a.bias = bias; a.accumulate = accumulate; a.allow_split = allow_split;
    return tc_gemm(a, (cudaStream_t)stream);
}

// The fused LSTM pair kernel on caller tensors (unit tests / bench roofline): both cells of
// models.py:107-123 in ONE launch.  u f32[M,Kin]; for k in {belief, action}: h_prev/c_prev
// f32[M,n], w_ih f32[4n,Kin], w_hh f32[4n,n], b_ih/b_hh f32[4n] -> c_new/h_new f32[M,n],
// gates f32[M,4n] (activated i,f,g,o).
extern "C" int marlc_tc_lstm_pair(const float* u, int M, int Kin, int n, const float* const* h_prev,
                                  const float* const* c_prev, const float* const* w_ih, const float* const* w_hh,
                                  const float* const* b_ih, const float* const* b_hh, float* const* c_new,
                                  float* const* h_new, float* const* gates, int x3, void* stream) {
    TcLstmArgs la[2];
    for (int k = 0; k < 2; ++k) {
        TcLstmArgs& a = la[k];
        a.U = tc_op(u, Kin); a.Hprev = tc_op(h_prev[k], n);
        a.Wih = w_ih[k]; a.Whh = w_hh[k]; a.bih = b_ih[k]; a.bhh = b_hh[k];
        a.c_prev = c_prev[k]; a.c_new = c_new[k]; a.h_new = h_new[k]; a.gates = gates[k];
        a.M = M; a.Kin = Kin; a.n = n; a.x3 = x3;
    }
    return tc_lstm_pair(la[0], la[1], (cudaStream_t)stream);
}

extern "C" int marlc_split_lo(const float* x, float* lo, int64_t n, void* stream) {
    MARLC_CHECK(x && lo && n >= 0, "split_lo: bad argument");
    if (n == 0) return 0;
    SplitLoArgs a;
    memset(&a, 0, sizeof(a));
    a.src[0] = x; a.dst[0] = lo; a.n[0] = n;
    MARLC_CHECK((((uintptr_t)x | (uintptr_t)lo) & 15) == 0, "split_lo: buffers must be 16-byte aligned");
    split_lo_kernel<<<dim3((unsigned)std::max<int64_t>(1, std::min<int64_t>(296, (n / 4 + 255) / 256)), 1), 256, 0, (cudaStream_t)stream>>>(a);
    MARLC_LAUNCH_CHECK();
    return 0;
}

extern "C" int marlc_tc_lstm_pair_presplit(const float* u, const float* u_lo, int M, int Kin, int n,
                                           const float* const* h_prev, const float* const* h_prev_lo,
                                           const float* const* c_prev, const float* const* w_ih,
                                           const float* const* w_ih_lo, const float* const* w_hh,
                                           const float* const* w_hh_lo, const float* const* b_ih,
                                           const float* const* b_hh, float* const* c_new, float* const* h_new,
                                           float* const* h_new_lo, float* const* gates, void* stream) {
    TcLstmArgs la[2];
    for (int k = 0; k < 2; ++k) {
        TcLstmArgs& a = la[k];
        a.U = tc_op(u, Kin); a.U.lo = u_lo;
        a.Hprev = tc_op(h_prev[k], n); a.Hprev.lo = h_prev_lo[k];
        a.Wih = w_ih[k]; a.Whh = w_hh[k]; a.Wih_lo = w_ih_lo[k]; a.Whh_lo = w_hh_lo[k];
        a.bih = b_ih[k]; a.bhh = b_hh[k];
        a.c_prev = c_prev[k]; a.c_new = c_new[k]; a.h_new = h_new[k]; a.h_new_lo = h_new_lo ? h_new_lo[k] : nullptr;
        a.gates = gates[k];
        a.M = M; a.Kin = Kin; a.n = n; a.x3 = 1;
    }
    return tc_lstm_pair(la[0], la[1], (cudaStream_t)stream);
}

// Profiling aid (scripts/phase_times.py): truncate marlc_episode_backward after a phase.
extern "C" int marlc_engine_debug_stop(marlc_engine* e, int phase) { e->debug_stop = phase; return 0; }

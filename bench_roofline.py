"""Roofline micro-measurements used by bench.py (and runnable alone).

Each kernel is launched through the C ABI on the current stream, `reps` times
back to back after warm-up, bracketed by CUDA events; achieved = ALGORITHMIC
bytes / flops per launch (SURVEY section 8d, restated in DESIGN.md) / mean
launch time.  Peaks come from MEASURED_PEAKS.json (driver-written); the TF32
tensor peak is measured live with cuBLAS (torch.matmul, allow_tf32) because the
file only holds the bf16 figure.
"""
from __future__ import annotations

import ctypes as ct
import json
import os

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
FALLBACK = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}
MARLC_SMS = 148


def peaks() -> tuple[dict, str]:
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            return json.load(fh), "measured (MEASURED_PEAKS.json)"
    return dict(FALLBACK), "fallback (B200_PROFILING.md)"


def _time(fn, reps: int, warm: int = 5, graph: bool = True) -> float:
    """Seconds per launch.  The `reps` launches are captured in ONE CUDA graph and replayed, so
    the figure is device time of back-to-back launches (as inside the graphed train step), not
    host launch overhead (each eager call also encodes TMA descriptors on the host)."""
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        for _ in range(warm):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    runner = None
    if graph:
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for _ in range(reps):
                fn()
        runner = g.replay
        runner()
        torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    if runner is not None:
        runner()
    else:
        for _ in range(reps):
            fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1e-3 / reps


def tf32_cublas_peak(dev) -> float:
    """TFLOP/s of torch.matmul fp32 with TF32 allowed, 8192^3, best of 5 (burst)."""
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        n = 8192
        a = torch.randn(n, n, device=dev)
        b = torch.randn(n, n, device=dev)
        best = min(_time(lambda: torch.matmul(a, b), 3, 2, graph=False) for _ in range(5))
        return 2 * n**3 / best / 1e12
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old


def lstm_pair(M: int, Kin: int, n: int, dev, reps: int = 200, x3: int = 1) -> dict:
    """The fused LSTM kernel (both cells, gate GEMMs on tcgen05 + cell epilogue)."""
    from marlclassification_b200 import _lib

    L = _lib.lib()
    g = torch.Generator(device=dev).manual_seed(0)
    rnd = lambda *s: torch.randn(*s, device=dev, generator=g)  # noqa: E731
    u = rnd(M, Kin)
    hp, cp = [rnd(M, n), rnd(M, n)], [rnd(M, n), rnd(M, n)]
    wih, whh = [rnd(4 * n, Kin) * 0.05, rnd(4 * n, Kin) * 0.05], [rnd(4 * n, n) * 0.05, rnd(4 * n, n) * 0.05]
    bih, bhh = [rnd(4 * n), rnd(4 * n)], [rnd(4 * n), rnd(4 * n)]
    cn, hn = [torch.empty(M, n, device=dev) for _ in range(2)], [torch.empty(M, n, device=dev) for _ in range(2)]
    gates = [torch.empty(M, 4 * n, device=dev) for _ in range(2)]
    arr = lambda ts: (ct.c_void_p * 2)(*[t.data_ptr() for t in ts])  # noqa: E731
    args = (u.data_ptr(), M, Kin, n, arr(hp), arr(cp), arr(wih), arr(whh), arr(bih), arr(bhh), arr(cn), arr(hn), arr(gates), x3)

    def run():
        _lib.check(L.marlc_tc_lstm_pair(*args, _lib.stream_ptr(dev)))

    if x3:
        # what the episode engine launches per step: operands pre-split (weights once per forward,
        # activations by their producer), so the kernel only streams tiles and issues 3 MMAs per K step
        def lo_of(t):
            out = torch.empty_like(t)
            _lib.check(L.marlc_split_lo(t.data_ptr(), out.data_ptr(), t.numel(), _lib.stream_ptr(dev)))
            return out

        u_lo, hp_lo, wih_lo, whh_lo = lo_of(u), [lo_of(t) for t in hp], [lo_of(t) for t in wih], [lo_of(t) for t in whh]
        hn_lo = [torch.empty(M, n, device=dev) for _ in range(2)]
        pargs = (u.data_ptr(), u_lo.data_ptr(), M, Kin, n, arr(hp), arr(hp_lo), arr(cp), arr(wih), arr(wih_lo), arr(whh),
                 arr(whh_lo), arr(bih), arr(bhh), arr(cn), arr(hn), arr(hn_lo), arr(gates))

        def run():  # noqa: F811
            _lib.check(L.marlc_tc_lstm_pair_presplit(*pargs, _lib.stream_ptr(dev)))

    t = _time(run, reps)
    flops = 2.0 * M * (Kin + n) * 4 * n * 2  # both cells (SURVEY 8d: lstm = 2(K_in+n)4n per row per cell)
    bytes_min = 4.0 * (M * Kin + 2 * M * n * 2 + 2 * 4 * n * (Kin + n) + 2 * M * 6 * n)
    return {"kernel": "tc_gemm_kernel<EPI_LSTM> (fused LSTM pair)", "shape": {"M": M, "K_in": Kin, "n": n},
            "us_per_launch": t * 1e6, "flops_per_launch": flops, "tflops": flops / t / 1e12,
            "min_bytes_per_launch": bytes_min}


def gather(na: int, nb: int, C: int, H: int, W: int, f: int, dev, reps: int = 200) -> dict:
    """K1 patch gather through Environment.observe's entry point."""
    from marlclassification_b200 import _lib

    L = _lib.lib()
    g = torch.Generator(device=dev).manual_seed(0)
    img = torch.rand(nb, C, H, W, device=dev, generator=g)
    pos = torch.stack([torch.randint(H - f, (na, nb), device=dev, generator=g),
                       torch.randint(W - f, (na, nb), device=dev, generator=g)], -1).contiguous()
    obs = torch.empty(na, nb, C, f, f, device=dev)

    def run():
        _lib.check(L.marlc_patch_gather(img.data_ptr(), pos.data_ptr(), obs.data_ptr(), na, nb, C, H, W, f,
                                        _lib.stream_ptr(dev)))

    t = _time(run, reps)
    M = na * nb
    bytes_alg = 2.0 * M * C * f * f * 4 + M * 16  # read each needed pixel once + write patch + read pos (SURVEY 8d)
    return {"kernel": "patch_gather_kernel", "shape": {"windows": M, "C": C, "f": f, "image": [H, W]},
            "us_per_launch": t * 1e6, "bytes_per_launch": bytes_alg, "gbs": bytes_alg / t / 1e9}


def transition(M: int, H: int, W: int, f: int, dev, reps: int = 100) -> dict:
    """K2 integer transition through Environment.step's entry point."""
    from marlclassification_b200 import _lib

    L = _lib.lib()
    g = torch.Generator(device=dev).manual_seed(0)
    pos = torch.stack([torch.randint(H - f, (M,), device=dev, generator=g), torch.randint(W - f, (M,), device=dev, generator=g)], -1).contiguous()
    act = torch.randint(4, (M,), device=dev, generator=g)
    table = torch.tensor([[1, 0], [-1, 0], [0, 1], [0, -1]], device=dev)
    npos = torch.empty(M, 2, device=dev)
    err = torch.zeros(1, dtype=torch.int32, device=dev)

    def run():
        _lib.check(L.marlc_transition(pos.data_ptr(), act.data_ptr(), table.data_ptr(), 4, M, f, H, W, npos.data_ptr(),
                                      err.data_ptr(), _lib.stream_ptr(dev)))

    t = _time(run, reps)
    bytes_alg = 48.0 * M  # read pos 16 + action 8, write pos 16 + normalised pos 8 (SURVEY 8d)
    return {"kernel": "transition_i64_kernel", "shape": {"agents": M}, "us_per_launch": t * 1e6,
            "bytes_per_launch": bytes_alg, "gbs": bytes_alg / t / 1e9}


def to_tensor_u8(B: int, C: int, H: int, W: int, dev, reps: int = 50) -> dict:
    """Device-side ToTensor (u8[B,H,W,C] -> f32[B,C,H,W] / 255), the input pipeline's kernel."""
    from marlclassification_b200.input_pipeline import images_u8_to_f32

    g = torch.Generator(device=dev).manual_seed(0)
    src = torch.randint(0, 256, (B, H, W, C), device=dev, generator=g, dtype=torch.uint8)
    out = torch.empty(B, C, H, W, device=dev)
    t = _time(lambda: images_u8_to_f32(src, out, hwc=True), reps)
    bytes_alg = 5.0 * B * C * H * W  # 1 byte read + 4 bytes written per element (DESIGN section 4)
    return {"kernel": "images_u8_to_f32 (HWC)", "shape": {"images": B, "C": C, "image": [H, W]},
            "us_per_launch": t * 1e6, "bytes_per_launch": bytes_alg, "gbs": bytes_alg / t / 1e9}


def weight_grad_gemm(R: int, N: int, K: int, dev, reps: int = 20, x3: int = 1) -> dict:
    """The batched weight-gradient product dW[N,K] += dY[R,N]^T X[R,K] (reduction over the R = T*M rows of an
    iteration; both operands MN-major, split-K chains of 4096 rows, f32 reduce-add epilogue): the launch the
    engine issues per LSTM cell for weight_ih (N = 4n, K = K_in)."""
    from marlclassification_b200 import _lib

    L = _lib.lib()
    g = torch.Generator(device=dev).manual_seed(0)
    dY = torch.randn(R, N, device=dev, generator=g)
    X = torch.randn(R, K, device=dev, generator=g)
    dW = torch.zeros(N, K, device=dev)

    def run():
        _lib.check(L.marlc_tc_gemm(dY.data_ptr(), N, 1, X.data_ptr(), K, 1, None, 0, None, 0, 0, None, dW.data_ptr(), K,
                                   N, K, R, 1, 1, x3, _lib.stream_ptr(dev)))

    t = _time(run, reps)
    flops = 2.0 * R * N * K
    return {"kernel": "tc_gemm_kernel<128, MN-major A, MN-major B, EPI_STORE> (batched weight gradient)",
            "shape": {"R": R, "N": N, "K": K}, "us_per_launch": t * 1e6, "flops_per_launch": flops,
            "tflops": flops / t / 1e12, "min_bytes_per_launch": 4.0 * (R * N + R * K + N * K)}


def step_pre_wide(model, w: dict, nb: int, dev, reps: int = 20) -> dict:
    """The per-step 'pre' launch of the episode at this batch (gather + feature extractor | message mean +
    decoder + position features), timed through the engine's profiling stop (forward with only that launch
    per step).  fp32 FFMA: reported against the CUDA-core peak, 148 SMs x 128 lanes x 2 flop x max clock."""
    from marlclassification_b200.config import ModelConfig  # noqa: F401
    from marlclassification_b200.engine import get_engine

    img = torch.rand(nb, w["C"], w["H"], w["W"], device=dev)
    eng = get_engine(model, na=w["na"], nb=nb, T=w["T"], C=w["C"], H=w["H"], W=w["W"], actions=w["actions"], gamma=0.99)

    def run():
        eng._L.marlc_engine_debug_stop(eng._h, 11)
        eng.forward(img)
        eng._L.marlc_engine_debug_stop(eng._h, 0)

    t = _time(run, reps) / w["T"]  # T launches per forward (+ two small init launches)
    M = w["na"] * nb
    spec = model.feature_extractor.cnn_spec
    f, layers = spec[0], spec[1]
    h, flops_win = f, 0.0
    for ci, co in layers:
        h = (h - 1) // 2 + 1
        flops_win += 2.0 * co * h * h * ci * 9
    d = model.dims
    flops = M * (flops_win + 2.0 * (d["n_m"] * 2 * d["n_m"] + 2 * d["n_m"] * d["n_m_o"]))
    return {"kernel": "step_pre_wide_kernel" if M >= 256 else "step_pre_kernel", "shape": {"windows": M},
            "us_per_launch": t * 1e6, "flops_per_launch": flops, "tflops": flops / t / 1e12}


def step_post(model, w: dict, nb: int, dev, reps: int = 10) -> dict:
    """The per-step 'post' launch (policy LayerNorm/SiLU + logits + softmax + sample + transition | encoder tail),
    timed as the difference of two truncated forwards (with / without it).  Row-local, reads and writes each
    activation once: HBM-bound nominally, latency-bound in practice (4 rows per CTA)."""
    from marlclassification_b200.engine import get_engine

    img = torch.rand(nb, w["C"], w["H"], w["W"], device=dev)
    eng = get_engine(model, na=w["na"], nb=nb, T=w["T"], C=w["C"], H=w["H"], W=w["W"], actions=w["actions"], gamma=0.99)

    def run(stop):
        def f():
            eng._L.marlc_engine_debug_stop(eng._h, stop)
            eng.forward(img)
            eng._L.marlc_engine_debug_stop(eng._h, 0)
        return f

    t = (_time(run(14), reps) - _time(run(13), reps)) / w["T"]
    d = model.dims
    M = w["na"] * nb
    bytes_row = 4.0 * (2 * d["nl_a"] + 2 * 2 * d["n_m"] + 2 * d["n_m"] + d["nb_action"]) + 48
    return {"kernel": "step_post_kernel", "shape": {"rows": M}, "us_per_launch": t * 1e6,
            "bytes_per_launch": bytes_row * M, "gbs": bytes_row * M / t / 1e9}


def roofline_for(model, w: dict, nb: int, dev) -> dict:
    """The `roofline` object of bench.py's JSON line.  Main entry = the fused LSTM pair at the workload's row count
    (one of three tensor-bound kernel families with 9-12 % of the iteration each at c4, the largest tensor kernel
    at the batch-8 configurations; profiles/r2/launches_*_summary.txt), measured live here; `others` holds the rest of the top of the launch list (weight-gradient GEMM, the fp32-FFMA
    `pre` launch) and the saturating micro-benchmarks of the HBM-bound kernels."""
    pk, src = peaks()
    d = model.dims
    M = w["na"] * nb
    TM = M * w["T"]
    Kin = model.feature_extractor.out_size + d["n_m_o"] + d["n_d"]
    tf32_peak = tf32_cublas_peak(dev)
    half_bf16 = 0.5 * float(pk.get("bf16_tflops", FALLBACK["bf16_tflops"]))
    x3 = 1 if getattr(model, "precision", "tf32x3") == "tf32x3" else 0
    prec = "tf32x3 (3 MMAs per K step; achieved counts ALGORITHMIC flops once)" if x3 else "tf32"
    lstm = lstm_pair(M, Kin, d["n_b"], dev, x3=x3, reps=50 if M > 1024 else 200)
    dw = weight_grad_gemm(TM, 4 * d["n_b"], Kin, dev, reps=10 if TM > 16384 else 50, x3=x3)
    pre = step_pre_wide(model, w, nb, dev)
    post = step_post(model, w, nb, dev)
    g_small = gather(w["na"], nb, w["C"], w["H"], w["W"], w["f"], dev)
    g_big = gather(256, 256, w["C"], w["H"], w["W"], w["f"], dev, reps=50)  # 65536 windows: saturating
    tr_big = transition(1 << 24, w["H"], w["W"], w["f"], dev, reps=20)
    n_img = max(1, (1 << 28) // (w["C"] * w["H"] * w["W"]))  # 268 M elements: 1.3 GB moved, far beyond L2
    tt_big = to_tensor_u8(n_img, w["C"], w["H"], w["W"], dev, reps=20)
    traffic, ncu_lstm = None, None
    tpath = os.path.join(ROOT, "profiles", "r2", "ncu_lstm_pair_m4096.json")
    if os.path.exists(tpath):
        with open(tpath) as fh:
            cap = json.load(fh)["captures"]
        best = cap.get("tile 128x256 (HU=64, default from M>=1793 at n=256)", {})
        try:
            traffic = (float(best["dram__bytes_read.sum"][0]) + float(best["dram__bytes_write.sum"][0])) * 1e6
            ncu_lstm = {"tensor_pipe_active_pct": float(best["sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active"][0]),
                        "tensor_pipe_active_pct_of_elapsed": float(best["sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_elapsed"][0]),
                        "l2_to_sm_read_mbytes": float(best["l1tex__m_xbar2l1tex_read_bytes.sum"][0]),
                        "source": "profiles/r2/ncu_lstm_pair_m4096.json (ncu --set full, one launch at M=4096)"}
        except Exception:
            pass
    ffma_peak = MARLC_SMS * 128 * 2 * float(pk.get("sm_max_mhz", 1965.0)) * 1e6 / 1e12

    def tensor_entry(r, name, extra=None):
        e = {"kernel": name, "bound": "tensor", "achieved": r["tflops"], "peak": tf32_peak, "unit": "TFLOP/s",
             "frac": r["tflops"] / tf32_peak, "frac_of_half_bf16_peak": r["tflops"] / half_bf16,
             "launch_us": r["us_per_launch"], "flops_per_launch": r["flops_per_launch"], "shape": r["shape"]}
        if extra:
            e.update(extra)
        return e

    lstm_e = tensor_entry(lstm, lstm["kernel"] + f" @ M={M}", {"ncu": ncu_lstm} if (ncu_lstm and M == 4096) else None)
    dw_e = tensor_entry(dw, dw["kernel"] + f" @ R=T*M={TM}")
    big = M >= 1024
    main = dict(lstm_e)
    main.update({
        "traffic": traffic if M == 4096 else None,
        "peak_source": "cuBLAS TF32 8192^3 measured in this run (MEASURED_PEAKS.json holds bf16 only: "
                       f"{pk.get('bf16_tflops')} TFLOP/s burst, {src}; frac_of_half_bf16_peak uses half of it)",
        "precision": prec,
        "time_share": ("the tensor-bound kernels take 9-12 % of the iteration each in the ncu launch list of this workload "
                       "(profiles/r2/launches_c4_nb256_summary.txt: weight-gradient GEMMs 12.1 %, input-gradient GEMMs 12.0 %, "
                       "fused LSTM pair 9.4 % -- list taken before the LSTM epilogue changes of the last commits); the main entry is "
                       "the LSTM pair (the one captured with ncu --set full), the "
                       "weight-gradient GEMM is listed under others; the largest share overall is step_pre_wide_kernel "
                       "(15 %, fp32 FFMA: under others against the CUDA-core peak)" if big else
                       "largest tensor-kernel share at the batch-8 configurations (profiles/r2/launches_c2_summary.txt)"),
        "others": [
            dw_e,
            {"kernel": pre["kernel"] + " (gather + CNN | decoder + position features)", "bound": "fp32-ffma",
             "achieved": pre["tflops"], "peak": ffma_peak, "unit": "TFLOP/s", "frac": pre["tflops"] / ffma_peak,
             "launch_us": pre["us_per_launch"], "flops_per_launch": pre["flops_per_launch"], "shape": pre["shape"],
             "peak_source": "CUDA-core fp32: 148 SMs x 128 lanes x 2 flop x sm_max_mhz (no measured figure in MEASURED_PEAKS.json)"},
            {"kernel": "step_post_kernel @ workload (policy tail + sample + transition | encoder tail)", "bound": "hbm",
             "achieved": post["gbs"], "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": post["gbs"] / pk["hbm_gbs"],
             "launch_us": post["us_per_launch"], "bytes_per_launch": post["bytes_per_launch"],
             "note": "row-local chain, 4 rows per CTA: latency-bound, not bandwidth-bound"},
            {"kernel": "patch_gather_kernel @ workload", "bound": "hbm", "achieved": g_small["gbs"],
             "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": g_small["gbs"] / pk["hbm_gbs"],
             "launch_us": g_small["us_per_launch"], "bytes_per_launch": g_small["bytes_per_launch"]},
            {"kernel": "patch_gather_kernel @ 65536 windows (saturating)", "bound": "hbm", "achieved": g_big["gbs"],
             "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": g_big["gbs"] / pk["hbm_gbs"],
             "launch_us": g_big["us_per_launch"], "bytes_per_launch": g_big["bytes_per_launch"]},
            {"kernel": "transition_i64_kernel @ 16.8 M agents (saturating)", "bound": "hbm", "achieved": tr_big["gbs"],
             "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": tr_big["gbs"] / pk["hbm_gbs"],
             "launch_us": tr_big["us_per_launch"], "bytes_per_launch": tr_big["bytes_per_launch"]},
            {"kernel": f"images_u8_to_f32 @ {n_img} images (saturating)", "bound": "hbm", "achieved": tt_big["gbs"],
             "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": tt_big["gbs"] / pk["hbm_gbs"],
             "launch_us": tt_big["us_per_launch"], "bytes_per_launch": tt_big["bytes_per_launch"]},
        ],
    })
    return main


if __name__ == "__main__":
    dev = torch.device("cuda", 0)
    pk, src = peaks()
    print("peaks:", pk.get("hbm_gbs"), pk.get("bf16_tflops"), src)
    print("tf32 cuBLAS peak TFLOP/s:", tf32_cublas_peak(dev))
    x3 = int(os.environ.get("X3", "1"))
    for M in (128, 1024, 4096, 16384):
        print(json.dumps(lstm_pair(M, 368, 256, dev, reps=50, x3=x3)))
    for na, nb in ((16, 8), (64, 64), (256, 256)):
        print(json.dumps(gather(na, nb, 3, 256, 256, 12, dev, reps=50)))
    print(json.dumps(gather(256, 64, 3, 600, 600, 24, dev, reps=50)))
    for M in (128, 1 << 20, 1 << 24):
        print(json.dumps(transition(M, 256, 256, 12, dev, reps=20)))
    print(json.dumps(to_tensor_u8(8, 3, 256, 256, dev)))
    print(json.dumps(to_tensor_u8(1365, 3, 256, 256, dev, reps=20)))

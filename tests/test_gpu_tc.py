"""tcgen05 / TMA TF32 GEMM kernel (csrc/gemm_tc.cu) against torch fp64, every
operand-major combination, ragged edges, split-K, dual operand pairs; and the
TF32 engine mode (fused LSTM-cell epilogue, tensor-core dX / dW) against the
fixtures recorded from the reference.

Default tensor-core mode = error-compensated 3xTF32 ("tf32x3"): held to the
north-star fp32 bound, 1e-3 (measured ~1e-5).  Plain TF32 ("tf32", inputs
truncated to 10 mantissa bits) has the stated looser bound: forward outputs
rel-L2 <= 5e-3, per-parameter gradients <= 2e-2.  Inputs exactly representable
in TF32 must reproduce fp32 to 1e-5 in either mode.
"""
import pytest
import torch

from tests.conftest import GOLDEN_NAMES, load_golden, rel_l2

pytestmark = pytest.mark.gpu
DEV = "cuda"
TF32_FWD_TOL = 5e-3
TF32_GRAD_TOL = 2e-2
X3_TOL = 1e-3  # the north-star fp32 bound: the default tensor-core mode (3xTF32) must meet it
# per-row bounds of the fused LSTM pair (tests.test_gpu_regimes.row_err), about 10x the worst over all shapes measured
# on one B200 (1000 W power limit): tf32 6.2e-4, tf32x3 4.3e-6, presplit 4.3e-6
LSTM_ROW_TOL = {"tf32": 6e-3, "tf32x3": 4e-5, "presplit": 4e-5}


def tf32_round(x):
    """Keep 10 mantissa bits (exactly representable TF32 values)."""
    return (x.view(torch.int32) & ~0x1FFF).view(torch.float32)


def run_tc(A, B, a_mn, b_mn, M, N, K, bias=None, A2=None, B2=None, K2=0, C0=None, accumulate=0, allow_split=0, x3=0):
    from marlclassification_b200 import _lib

    C = torch.zeros(M, N, device=DEV) if C0 is None else C0.clone()
    _lib.check(_lib.lib().marlc_tc_gemm(
        A.data_ptr(), A.stride(0), a_mn, B.data_ptr(), B.stride(0), b_mn,
        None if A2 is None else A2.data_ptr(), 0 if A2 is None else A2.stride(0),
        None if B2 is None else B2.data_ptr(), 0 if B2 is None else B2.stride(0), K2,
        None if bias is None else bias.data_ptr(), C.data_ptr(), C.stride(0), M, N, K, accumulate, allow_split, x3,
        _lib.stream_ptr()))
    torch.cuda.synchronize()
    return C


@pytest.mark.parametrize("a_mn,b_mn", [(0, 0), (0, 1), (1, 0), (1, 1)])
@pytest.mark.parametrize("M,N,K", [(128, 128, 64), (128, 64, 32), (200, 96, 160), (128, 1024, 368), (64, 32, 2048),
                                   (300, 40, 72), (2048, 384, 256)])
def test_tc_gemm_exact_on_tf32_inputs(a_mn, b_mn, M, N, K):
    g = torch.Generator(device=DEV).manual_seed(M + N + K + 2 * a_mn + b_mn)
    # logical A [M,K], B [N,K]
    A = tf32_round(torch.randn(M, K, device=DEV, generator=g))
    B = tf32_round(torch.randn(N, K, device=DEV, generator=g))
    Am = A.t().contiguous() if a_mn else A  # MN-major storage: [K rows][M contiguous]
    Bm = B.t().contiguous() if b_mn else B
    if (Am.stride(0) % 4) or (Bm.stride(0) % 4):
        pytest.skip("leading dimension not a multiple of 4 floats (TMA stride rule)")
    bias = torch.randn(N, device=DEV, generator=g)
    C = run_tc(Am, Bm, a_mn, b_mn, M, N, K, bias=bias)
    ref = A.double() @ B.double().t() + bias.double()
    assert rel_l2(C.cpu(), ref.cpu()) < 1e-5


@pytest.mark.parametrize("a_mn,b_mn", [(0, 0), (0, 1), (1, 1)])
def test_tc_gemm_tf32_error_bound(a_mn, b_mn):
    M, N, K = 256, 192, 512
    g = torch.Generator(device=DEV).manual_seed(7)
    A, B = torch.randn(M, K, device=DEV, generator=g), torch.randn(N, K, device=DEV, generator=g)
    Am = A.t().contiguous() if a_mn else A
    Bm = B.t().contiguous() if b_mn else B
    C = run_tc(Am, Bm, a_mn, b_mn, M, N, K)
    err = rel_l2(C.cpu(), (A.double() @ B.double().t()).cpu())
    print(f"tf32 rel-L2 error, K={K}: {err:.2e}")
    assert err < 2e-3


@pytest.mark.parametrize("a_mn,b_mn", [(0, 0), (0, 1), (1, 0), (1, 1)])
@pytest.mark.parametrize("M,N,K", [(128, 128, 256), (200, 96, 160), (128, 1024, 368), (2048, 384, 256)])
def test_tc_gemm_x3_fp32_class_accuracy(a_mn, b_mn, M, N, K):
    """Error-compensated 3xTF32: arbitrary fp32 inputs, result within fp32 rounding of fp64."""
    g = torch.Generator(device=DEV).manual_seed(M + N + K + 2 * a_mn + b_mn)
    A, B = torch.randn(M, K, device=DEV, generator=g), torch.randn(N, K, device=DEV, generator=g)
    Am = A.t().contiguous() if a_mn else A
    Bm = B.t().contiguous() if b_mn else B
    C = run_tc(Am, Bm, a_mn, b_mn, M, N, K, x3=1)
    err = rel_l2(C.cpu(), (A.double() @ B.double().t()).cpu())
    assert err < 5e-6, err


def test_tc_gemm_x3_split_k_dual_pair():
    M, N, K, K2 = 128, 368, 1024, 1024
    g = torch.Generator(device=DEV).manual_seed(12)
    A, A2 = torch.randn(M, K, device=DEV, generator=g), torch.randn(M, K2, device=DEV, generator=g)
    W, W2 = torch.randn(K, N, device=DEV, generator=g), torch.randn(K2, N, device=DEV, generator=g)
    ref = A.double() @ W.double() + A2.double() @ W2.double()
    C = run_tc(A, W, 0, 1, M, N, K, A2=A2, B2=W2, K2=K2, allow_split=1, x3=1)
    assert rel_l2(C.cpu(), ref.cpu()) < 5e-6


def test_tc_gemm_split_k_dual_pair_accumulate():
    M, N, K, K2 = 128, 368, 1024, 1024
    g = torch.Generator(device=DEV).manual_seed(11)
    A = tf32_round(torch.randn(M, K, device=DEV, generator=g))
    A2 = tf32_round(torch.randn(M, K2, device=DEV, generator=g))
    W = tf32_round(torch.randn(K, N, device=DEV, generator=g))    # MN-major B: [K rows][N contiguous]
    W2 = tf32_round(torch.randn(K2, N, device=DEV, generator=g))
    ref = A.double() @ W.double() + A2.double() @ W2.double()
    C = run_tc(A, W, 0, 1, M, N, K, A2=A2, B2=W2, K2=K2, allow_split=1)
    assert rel_l2(C.cpu(), ref.cpu()) < 1e-5
    C0 = torch.randn(M, N, device=DEV, generator=g)
    C = run_tc(A, W, 0, 1, M, N, K, A2=A2, B2=W2, K2=K2, C0=C0, accumulate=1, allow_split=1)
    assert rel_l2(C.cpu(), (ref + C0.double()).cpu()) < 1e-5
    C = run_tc(A, W, 0, 1, M, N, K, C0=C0, accumulate=1, allow_split=0)
    assert rel_l2(C.cpu(), (A.double() @ W.double() + C0.double()).cpu()) < 1e-5


def test_tc_gemm_strided_views():
    """Operands / outputs that are column slices of wider buffers (u_t slices)."""
    M, N, K = 128, 96, 128
    g = torch.Generator(device=DEV).manual_seed(3)
    Abig = tf32_round(torch.randn(M, 368, device=DEV, generator=g))
    B = tf32_round(torch.randn(N, K, device=DEV, generator=g))
    Cbig = torch.zeros(M, 368, device=DEV)
    A = Abig[:, 64:64 + K]
    Cv = Cbig[:, 256:256 + N]
    from marlclassification_b200 import _lib

    _lib.check(_lib.lib().marlc_tc_gemm(A.data_ptr(), 368, 0, B.data_ptr(), K, 0, None, 0, None, 0, 0, None,
                                        Cv.data_ptr(), 368, M, N, K, 0, 0, 0, _lib.stream_ptr()))
    torch.cuda.synchronize()
    assert rel_l2(Cv.cpu(), (A.double() @ B.double().t()).cpu()) < 1e-5
    assert Cbig[:, :256].abs().max().item() == 0 and Cbig[:, 256 + N:].abs().max().item() == 0


@pytest.mark.parametrize("precision", ["tf32", "tf32x3"])
@pytest.mark.parametrize("name", ["mnist_ckpt", "resisc_small", "aid_small"])
def test_tf32_engine_vs_reference(name, precision):
    from tests.test_gpu_parity import run_fixture

    fx = load_golden(name)
    model, marl, env, sampler, inject = run_fixture(fx, use_tc=True)
    model.precision = precision
    img = fx["img"].to(DEV)
    eng = sampler.engine_for(img)
    eng.forward(img, **inject)
    assert torch.equal(eng.step_pos.cpu(), fx["step_pos"])  # positions stay bit-exact in every mode
    e = [rel_l2(eng.step_preds.cpu(), fx["step_preds"]), rel_l2(eng.step_log_probas.cpu(), fx["step_log_probas"]),
         rel_l2(eng.step_values.cpu(), fx["step_values"])]
    loss_out = eng.loss(fx["targets"].to(DEV)).cpu()
    eng.backward()
    model.attach_grads()
    worst = max(rel_l2(p.grad.cpu(), fx["grads"][k]) for k, p in model.named_parameters() if fx["grads"][k].norm() > 0)
    print(f"{name} {precision}: preds/logp/values rel-L2 = {e[0]:.1e}/{e[1]:.1e}/{e[2]:.1e}, worst grad = {worst:.1e}")
    # 3xTF32 is held here to what it actually delivers (fp32-class: measured <= 6e-6 forward, <= 4e-5 on the
    # worst parameter gradient), far inside the 1e-3 north-star bound, so that a path that silently loses
    # its low-order correction (TF32-class error, ~1e-4..1e-3) fails instead of hiding under the bound
    fwd_tol, grad_tol = (TF32_FWD_TOL, TF32_GRAD_TOL) if precision == "tf32" else (3e-5, 2e-4)
    assert fwd_tol <= X3_TOL or precision == "tf32"
    assert max(e) < fwd_tol
    assert abs(loss_out[0].item() - fx["logged"]["loss"]) <= fwd_tol * abs(fx["logged"]["loss"])
    assert worst < grad_tol


def test_tf32_full_c2_vs_fp32_mode():
    """RESISC45 shape (README nets): the TF32 mode against our own exact-fp32 mode."""
    from marlclassification_b200.config import ModelConfig
    from marlclassification_b200.core import EpisodeSampler
    from tests.test_gpu_parity import FULL

    spec = FULL["c2_resisc45"]
    na, nb, T = spec["na"], spec["nb"], spec["T"]
    torch.manual_seed(0)
    model, marl, env = ModelConfig(**spec["mc"]).build_marl(na)
    model.to(DEV)
    g = torch.Generator().manual_seed(5)
    img = torch.rand(nb, 3, 256, 256, generator=g).to(DEV)
    y = torch.randint(45, (nb,), generator=g).to(DEV)
    pos0 = torch.stack([torch.randint(244, (na, nb), generator=g), torch.randint(244, (na, nb), generator=g)], -1).to(DEV)
    hidden0 = [torch.randn(na, nb, 256, generator=g).to(DEV) for _ in range(4)]
    actions = torch.randint(4, (T, na, nb), generator=g).to(DEV)
    res = {}
    for use_tc in (False, True, "tf32"):
        model.use_tc = bool(use_tc)
        model.precision = "tf32" if use_tc == "tf32" else "tf32x3"
        sampler = EpisodeSampler(marl, env, T, gamma=0.99)
        eng = sampler.engine_for(img)
        eng.forward(img, pos0, hidden0, actions)
        loss = eng.loss(y).clone()
        eng.backward()
        res[use_tc] = (eng.step_preds.clone(), eng.step_values.clone(), loss, model.flat_grads.clone(),
                       eng.step_pos.clone())
    for key, ftol, gtol in ((True, X3_TOL, X3_TOL), ("tf32", TF32_FWD_TOL, TF32_GRAD_TOL)):
        assert torch.equal(res[key][4], res[False][4])
        ep, ev = rel_l2(res[key][0].cpu(), res[False][0].cpu()), rel_l2(res[key][1].cpu(), res[False][1].cpu())
        eg = rel_l2(res[key][3].cpu(), res[False][3].cpu())
        print(f"c2 {'tf32x3' if key is True else key} vs fp32: preds {ep:.1e}, values {ev:.1e}, flat grads {eg:.1e}")
        assert ep < ftol and ev < ftol and eg < gtol


# ---- fused LSTM pair (recurrent.py:7-35: both cells share u_t) as one tensor-core launch ----------
def _lstm_ref64(u, h, c, wih, whh, bih, bhh):
    g = u.double() @ wih.double().t() + bih.double() + h.double() @ whh.double().t() + bhh.double()
    i, f, gg, o = g.chunk(4, dim=1)
    i, f, gg, o = torch.sigmoid(i), torch.sigmoid(f), torch.tanh(gg), torch.sigmoid(o)
    cn = f * c.double() + i * gg
    return torch.cat([i, f, gg, o], 1), cn, o * torch.tanh(cn)


# (600: 16 hidden units per CTA, not fat; 1000: 32 units, 128-wide tile with a 3-stage ring; 1793: the fewest rows
#  with 64 units at n = 256; 4097: 64 units, one row in the last tile; 1027 at n = 64: 32 units)
@pytest.mark.parametrize("M,Kin,n", [(128, 368, 256), (96, 96, 64), (4096, 368, 256), (20, 624, 256), (130, 100, 32), (512, 368, 256),
                                     (600, 368, 256), (1000, 368, 256), (1793, 368, 256), (4097, 368, 256), (1027, 96, 64)])
@pytest.mark.parametrize("mode", ["tf32", "tf32x3", "presplit"])
def test_tc_lstm_pair_vs_fp64(M, Kin, n, mode):
    import ctypes as ct

    from marlclassification_b200 import _lib
    from tests.test_gpu_regimes import row_err

    L = _lib.lib()
    g = torch.Generator(device=DEV).manual_seed(M + Kin + n)
    rnd = lambda *s: torch.randn(*s, device=DEV, generator=g)  # noqa: E731
    u = rnd(M, Kin)
    hp, cp = [rnd(M, n), rnd(M, n)], [rnd(M, n), rnd(M, n)]
    wih, whh = [rnd(4 * n, Kin) * 0.05 for _ in range(2)], [rnd(4 * n, n) * 0.05 for _ in range(2)]
    bih, bhh = [rnd(4 * n) * 0.1 for _ in range(2)], [rnd(4 * n) * 0.1 for _ in range(2)]
    cn = [torch.zeros(M, n, device=DEV) for _ in range(2)]
    hn = [torch.zeros(M, n, device=DEV) for _ in range(2)]
    hn_lo = [torch.zeros(M, n, device=DEV) for _ in range(2)]
    gates = [torch.zeros(M, 4 * n, device=DEV) for _ in range(2)]
    arr = lambda ts: (ct.c_void_p * 2)(*[t.data_ptr() for t in ts])  # noqa: E731
    if mode == "presplit":
        def lo_of(t):
            out = torch.empty_like(t)
            _lib.check(L.marlc_split_lo(t.data_ptr(), out.data_ptr(), t.numel(), _lib.stream_ptr()))
            return out

        # the split is exact: hi + lo == x bit for bit, hi has at most 10 mantissa bits
        lo = lo_of(u)
        assert torch.equal((u - lo) + lo, u) and torch.equal(tf32_round(u - lo), u - lo)
        hp_lo, wih_lo, whh_lo = [lo_of(t) for t in hp], [lo_of(t) for t in wih], [lo_of(t) for t in whh]  # keep alive
        _lib.check(L.marlc_tc_lstm_pair_presplit(
            u.data_ptr(), lo.data_ptr(), M, Kin, n, arr(hp), arr(hp_lo), arr(cp), arr(wih), arr(wih_lo), arr(whh),
            arr(whh_lo), arr(bih), arr(bhh), arr(cn), arr(hn), arr(hn_lo), arr(gates), _lib.stream_ptr()))
    else:
        _lib.check(L.marlc_tc_lstm_pair(u.data_ptr(), M, Kin, n, arr(hp), arr(cp), arr(wih), arr(whh), arr(bih), arr(bhh),
                                        arr(cn), arr(hn), arr(gates), 1 if mode == "tf32x3" else 0, _lib.stream_ptr()))
    torch.cuda.synchronize()
    tol = 5e-3 if mode == "tf32" else 2e-5
    row_tol = LSTM_ROW_TOL[mode]
    tail = M - (M - 1) // 128 * 128  # rows in the last 128-row tile
    worst = 0.0
    for k in range(2):
        g_ref, c_ref, h_ref = _lstm_ref64(u, hp[k], cp[k], wih[k], whh[k], bih[k], bhh[k])
        for out, ref in ((gates[k], g_ref), (cn[k], c_ref), (hn[k], h_ref)):
            assert rel_l2(out.double().cpu(), ref.cpu()) < tol
            e, row = row_err(out, ref)  # a wrong row (a tile's ragged edge) is not diluted by the others
            worst = max(worst, e)
            assert e < row_tol, (k, row, e)
        if mode == "presplit":  # the kernel also emits the low-order part of h for the next step's operand
            hi = tf32_round(hn[k])
            assert torch.equal(hn_lo[k], hn[k] - hi)
            assert torch.equal(hn_lo[k][-tail:], hn[k][-tail:] - hi[-tail:]) and hn[k][-tail:].abs().min() > 0
    print(f"M={M} n={n} {mode}: worst per-row error {worst:.1e}")


# ---- round-2 regressions ---------------------------------------------------------------------------------
def test_tc_gemm_long_reduction_keeps_fp32_class_accuracy():
    """Weight-gradient shape: both operands MN-major, reduction over 65 536 rows.  The tensor core adds into
    its TMEM accumulator with truncation; without the 4096-element chain cap (TC_MAX_CHAIN, partial sums meeting
    in the f32 reduce-add epilogue) this product was 6e-4 off -- the 3xTF32 path must stay fp32-class."""
    R, N, K = 65536, 256, 368
    g = torch.Generator(device=DEV).manual_seed(11)
    dY = torch.randn(R, N, device=DEV, generator=g)
    X = torch.randn(R, K, device=DEV, generator=g)
    C = run_tc(dY, X, 1, 1, N, K, R, allow_split=1, x3=1)
    ref = dY.double().t() @ X.double()
    err = rel_l2(C.cpu(), ref.cpu())
    print(f"dW[{N}x{K}] over {R} rows, 3xTF32: rel-L2 {err:.1e}")
    assert err < 1e-4


@pytest.mark.timeout(180)
def test_tc_gemm_in_kernel_split_under_stream_concurrency():
    """3-stage ring + in-kernel operand split (3xTF32 without pre-split twins), several launches in flight on
    different streams next to an unrelated memory-bound kernel: the configuration in which the operand splitter's
    barrier phases slipped (hang / unspecified launch failure) before round 2's fix.  Results must also be right."""
    from marlclassification_b200 import _lib

    L = _lib.lib()
    R, N, K = 16384, 384, 256  # dW = dY^T X: 128-wide MN/MN tiles (3-stage ring), split-K chains
    M2, N2, K2 = 4096, 368, 1024  # dX-like: K-major A, MN-major B, 128-wide (3-stage ring)
    g = torch.Generator(device=DEV).manual_seed(5)
    dY, X = torch.randn(R, N, device=DEV, generator=g), torch.randn(R, K, device=DEV, generator=g)
    A2, B2 = torch.randn(M2, K2, device=DEV, generator=g), torch.randn(K2, N2, device=DEV, generator=g)
    ref1 = (dY.double().t() @ X.double()).cpu()
    ref2 = (A2.double() @ B2.double()).cpu()
    streams = [torch.cuda.Stream() for _ in range(3)]
    filler = torch.empty(64 << 20, device=DEV)
    outs1 = [torch.zeros(N, K, device=DEV) for _ in range(3)]
    outs2 = [torch.zeros(M2, N2, device=DEV) for _ in range(3)]
    torch.cuda.synchronize()
    for it in range(20):
        for i, st in enumerate(streams):
            with torch.cuda.stream(st):
                _lib.check(L.marlc_tc_gemm(dY.data_ptr(), N, 1, X.data_ptr(), K, 1, None, 0, None, 0, 0, None,
                                           outs1[i].data_ptr(), K, N, K, R, 0, 1, 1, st.cuda_stream))
                filler.add_(1.0)
                _lib.check(L.marlc_tc_gemm(A2.data_ptr(), K2, 0, B2.data_ptr(), N2, 1, None, 0, None, 0, 0, None,
                                           outs2[i].data_ptr(), N2, M2, N2, K2, 0, 0, 1, st.cuda_stream))
    torch.cuda.synchronize()
    for o in outs1:
        assert rel_l2(o.cpu(), ref1) < 1e-4
    for o in outs2:
        assert rel_l2(o.cpu(), ref2) < 1e-4

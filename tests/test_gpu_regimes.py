"""Every kernel variant the episode engine's dispatch can select, held to an fp64 oracle row by row.

The engine picks kernels by M = na * nb, the rows of one step (the thresholds are in ``marlc_engine_plan``,
include/marlc.h): per-window or wide feature extractor (batches of 8 windows, persistent CTAs), the LSTM
pair's tile (HU hidden units per CTA, fat stages, K split), the chained or unfused BPTT sweep, and the
4-row blocks of the chain kernels.  The cases below choose M so that each variant runs with a ragged edge:
a last wide batch of fewer than 8 windows, a last 128-row tile of a few rows, a last row block of
fewer than 4 rows.  A kernel that is wrong only there is diluted by thousands of right rows in a
whole-tensor norm, so the forward is compared per row (``row_err``) and the backward through probes
that put a gradient on a few rows only.

* ``test_plan_table`` (CPU): the plan of every case equals the table, and the cases cover every variant.
* ``test_forward_rows``: per step, every row of u_t, h/c/h^/c^, the message, the logits, log-probs and
  values against the fp64 oracle; positions bit-exact.
* ``test_backward_probes``: d_preds / d_logp / d_values nonzero on the tail rows, on one row, or the real
  loss; per-parameter gradients against the oracle's fp64 vector-Jacobian product.
"""
import ctypes as ct
import functools

import pytest
import torch

from oracle import marl_oracle as O
from tests.conftest import oracle_config, rel_l2
from tests.test_gpu_configs import C2_NET, MOVES1, MOVES3, _graphed_iteration, _mc

DEV = "cuda"
MNIST_NET = _mc("mnist", 6, 64, 16, 24, 8, 96, 96, 10, MOVES1)  # n = 64, channel 0 of 3
AID_NET = _mc("aid", 24, 256, 64, 96, 16, 320, 320, 30, MOVES3)  # 388 KB of conv weights: never wide

# Expected plan columns, computed from the launchers' code:
#   cnn  = None (one CTA per window) or (batches of 8 windows, CTAs, passes, windows in the last batch)
#   lstm = (HU, fat, K split, rows in the last 128-row tile)    sweep = 1 chained / 0 unfused
# HU: 8 for one 128-row tile, 16 from 2 tiles, 32 from 8, 64 once 2 * tiles * (n / 64) >= 120 (M >= 1793 at
# n = 256); fat while HU <= 16 and 2 * tiles * (n / HU) <= 148; K split for HU = 8 when twice the CTAs fit.
CASES = {
    "93": dict(net=C2_NET, na=3, nb=31, T=5, H=256, W=256, cnn=None, lstm=(8, 1, 2, 93), sweep=1),
    "255": dict(net=C2_NET, na=5, nb=51, T=3, H=256, W=256, cnn=None, lstm=(16, 1, 1, 127), sweep=1),
    "259": dict(net=C2_NET, na=7, nb=37, T=3, H=256, W=256, cnn=(33, 33, 1, 3), lstm=(16, 1, 1, 3), sweep=1),
    "300": dict(net=C2_NET, na=1, nb=300, T=3, H=256, W=256, cnn=(38, 38, 1, 4), lstm=(16, 1, 1, 44), sweep=1),
    "605": dict(net=C2_NET, na=11, nb=55, T=3, H=256, W=256, cnn=(76, 76, 1, 5), lstm=(16, 0, 1, 93), sweep=1),
    "1190": dict(net=C2_NET, na=14, nb=85, T=3, H=200, W=256, cnn=(149, 148, 2, 6), lstm=(32, 0, 1, 38), sweep=1),
    "1795": dict(net=C2_NET, na=5, nb=359, T=3, H=256, W=256, cnn=(225, 148, 2, 3), lstm=(64, 0, 1, 3), sweep=1),
    "4098": dict(net=C2_NET, na=6, nb=683, T=3, H=256, W=256, cnn=(513, 148, 4, 2), lstm=(64, 0, 1, 2), sweep=0),
    "387": dict(net=MNIST_NET, na=3, nb=129, T=4, H=28, W=28, cnn=(49, 49, 1, 3), lstm=(16, 1, 1, 3), sweep=1),
    "1027": dict(net=MNIST_NET, na=13, nb=79, T=3, H=28, W=28, cnn=(129, 129, 1, 3), lstm=(32, 0, 1, 3), sweep=1),
    "261": dict(net=AID_NET, na=3, nb=87, T=3, H=200, W=200, cnn=None, lstm=(16, 1, 1, 5), sweep=1),
}
# rows in the last 4-row block of the chain kernels (M % 4; 0 = full), per the table of the cases above
M_MOD_4 = {"93": 1, "255": 3, "259": 3, "300": 0, "605": 1, "1190": 2, "1795": 3, "4098": 2, "387": 3, "1027": 3,
           "261": 1}

# Bounds on the worst per-row error (forward) and on the worst per-parameter rel-L2 (probes): about 10x the worst
# value over all cases measured on one B200 (1000 W power limit), never above the north-star 1e-3.
# measured, tf32x3:  u 3.1e-6, h 6.7e-6, c 6.6e-6, h^ 6.7e-6, c^ 7.0e-6, msg 8.0e-6, preds 7.8e-6, logp 8.7e-6,
#                    values 2.3e-5 (values are a 384-term dot product on each row: the largest relative error)
FWD_BOUND = {"u": 3e-5, "h": 7e-5, "c": 7e-5, "h_caret": 7e-5, "c_caret": 7e-5, "msg": 8e-5, "preds": 8e-5,
             "logp": 9e-5, "values": 2.5e-4}
# measured, exact fp32 (use_tc=False): u 4.4e-7, h 4.8e-7, c 4.7e-7, h^ 4.8e-7, c^ 4.7e-7, msg 1.0e-6, preds 8.9e-7,
#                    logp 9.1e-7, values 3.1e-6
FWD_BOUND_FP32 = {"u": 5e-6, "h": 5e-6, "c": 5e-6, "h_caret": 5e-6, "c_caret": 5e-6, "msg": 1e-5, "preds": 1e-5,
                  "logp": 1e-5, "values": 3e-5}
# measured, tf32x3: tail 2.7e-5, one row 2.1e-5, full loss 5.2e-5
PROBE_BOUND = {"tail": 3e-4, "row": 2e-4, "full": 5e-4}


def _mplan(key):
    c = CASES[key]
    p = dict(sweep_chained=c["sweep"], staged_step_pre=1, staged_step_post=1, staged_bwd_pre=c["sweep"],
             staged_bwd_post=c["sweep"], lstm_tc=1)
    if c["cnn"] is None:
        M = c["na"] * c["nb"]
        p.update(cnn_wide=0, cnn_nw=1, cnn_batches=M, cnn_ctas=M, cnn_passes=1, cnn_tail=1)
    else:
        b, ctas, passes, tail = c["cnn"]
        p.update(cnn_wide=1, cnn_nw=8, cnn_batches=b, cnn_ctas=ctas, cnn_passes=passes, cnn_tail=tail)
    hu, fat, ksplit, tail_rows = c["lstm"]
    p.update(lstm_hu=hu, lstm_bn=4 * hu, lstm_fat=fat, lstm_ks=2 if fat else 1, lstm_ksplit=ksplit,
             lstm_tail_rows=tail_rows)
    return p


def _config(key, use_tc=True):
    from marlclassification_b200.config import ModelConfig
    from marlclassification_b200.engine import build_config

    c = CASES[key]
    model = ModelConfig(**c["net"]).build_networks()
    model.use_tc = use_tc
    return build_config(model, na=c["na"], nb=c["nb"], T=c["T"], C=3, H=c["H"], W=c["W"], actions=c["net"]["actions"],
                        gamma=0.99)


def _plans():
    """{case: marlc_engine_plan} of engines created (never bound) for every case: host only."""
    from marlclassification_b200.engine import engine_plan

    return {key: engine_plan(_config(key)) for key in CASES}


def test_plan_table():
    plans = _plans()
    for key, c in CASES.items():
        got, want = plans[key], _mplan(key)
        diff = {k: (got[k], v) for k, v in want.items() if got[k] != v}
        assert not diff, f"case {key}: (plan, table) {diff} -- the case no longer lands in its regime"
        assert (c["na"] * c["nb"]) % 4 == M_MOD_4[key]
    # coverage: every LSTM launch variant of the default mode at n = 256, every feature-extractor / sweep variant
    n256 = [plans[k] for k, c in CASES.items() if c["net"]["hidden_size_belief"] == 256]
    lstm = {(p["lstm_hu"], p["lstm_fat"], p["lstm_ksplit"]) for p in n256}
    assert {(8, 1, 2), (16, 1, 1), (16, 0, 1), (32, 0, 1), (64, 0, 1)} <= lstm, lstm
    ps = list(plans.values())
    assert any(not p["cnn_wide"] for p in ps)
    assert any(p["cnn_wide"] and p["cnn_tail"] < p["cnn_nw"] for p in ps)
    assert any(p["cnn_wide"] and p["cnn_passes"] > 1 and p["cnn_tail"] < p["cnn_nw"] for p in ps)
    assert {p["sweep_chained"] for p in ps} == {0, 1}
    assert any(not p["sweep_chained"] and p["lstm_tail_rows"] < 128 for p in ps)
    assert {(c["na"] * c["nb"]) % 4 for c in CASES.values()} == {0, 1, 2, 3}


# ---------------------------------------------------------------------------------------------------------------
# GPU: the engine against the fp64 oracle
# ---------------------------------------------------------------------------------------------------------------
def row_err(a, b):
    """max_r ||a_r - b_r|| / max(||b_r||, rms_r ||b_r||) over the rows of [R, ...] tensors, and the worst row.
    The floor (root mean square of the row norms) keeps rows near zero from dominating."""
    a = a.detach().double().cpu().reshape(a.shape[0], -1)
    b = b.detach().double().cpu().reshape(b.shape[0], -1)
    nb = b.norm(dim=1)
    den = torch.maximum(nb, nb.pow(2).mean().sqrt()).clamp_min(1e-300)
    e = (a - b).norm(dim=1) / den
    i = int(e.argmax())
    return float(e[i]), i


@functools.lru_cache(maxsize=1)
def _case(key):
    """Inputs, fp32 parameters and oracle-sampled actions of a case, and the fp64 oracle rollout (one graph,
    kept for the probes' vector-Jacobian products)."""
    c = CASES[key]
    ocfg = oracle_config(c["net"])
    params = O.init_params(ocfg, seed=7)
    na, nb, T, H, W, f = c["na"], c["nb"], c["T"], c["H"], c["W"], ocfg.f
    g = torch.Generator().manual_seed(1000 + na * nb)
    img = torch.rand(nb, 3, H, W, generator=g)
    y = torch.randint(ocfg.nb_class, (nb,), generator=g)
    pos0 = torch.stack([torch.randint(H - f, (na, nb), generator=g), torch.randint(W - f, (na, nb), generator=g)], -1)
    pos0[0, 0] = torch.tensor([0, 0])  # the extreme corners
    pos0[-1, -1] = torch.tensor([H - f - 1, W - f - 1])
    hidden0 = [torch.randn(na, nb, n, generator=g) for n in (ocfg.n_b, ocfg.n_b, ocfg.n_a, ocfg.n_a)]
    actions = O.rollout(params, ocfg, img, pos0, hidden0, None, T, generator=g).actions
    p64 = {k: v.double().requires_grad_(True) for k, v in params.items()}
    ro = O.rollout(p64, ocfg, img.double(), pos0, [h.double() for h in hidden0], actions, T, record=True)
    return dict(ocfg=ocfg, params=params, img=img, y=y, pos0=pos0, hidden0=hidden0, actions=actions, p64=p64, ro=ro)


def _engine(key, use_tc=True):
    from marlclassification_b200.config import ModelConfig
    from marlclassification_b200.core import EpisodeSampler

    c, d = CASES[key], _case(key)
    model, marl, env = ModelConfig(**c["net"]).build_marl(c["na"])
    model.use_tc = use_tc
    model.load_state_dict(d["params"])
    model.to(DEV)
    assert model.use_chains and (not use_tc or model.precision == "tf32x3")
    sampler = EpisodeSampler(marl, env, c["T"], gamma=0.99)
    imgd = d["img"].to(DEV)
    eng = sampler.engine_for(imgd)
    inject = (d["pos0"].to(DEV), [h.to(DEV) for h in d["hidden0"]], d["actions"].to(DEV))
    return model, eng, imgd, inject


def _u_rows(eng, T, M):
    """The engine's LSTM input buffer "U" as [T, M, row pitch] (pitch from the buffer's size)."""
    from marlclassification_b200 import _lib

    off, nbytes = ct.c_size_t(), ct.c_size_t()
    _lib.check(eng._L.marlc_engine_buffer(eng._h, b"U", ct.byref(off), ct.byref(nbytes)))
    pitch = nbytes.value // (4 * T * M)
    return eng.view("U", torch.float32, (T, M, pitch))


def _forward_errors(key, eng):
    """Worst per-row error of every per-step quantity: {name: (error, step, row)}."""
    c, ro = CASES[key], _case(key)["ro"]
    T, M = c["T"], c["na"] * c["nb"]
    U = _u_rows(eng, T, M)
    state = {"h": eng.H_state, "c": eng.C_state, "h_caret": eng.Hc_state, "c_caret": eng.Cc_state, "msg": eng.msg}
    worst = {}

    def put(name, t, a, b):
        e, r = row_err(a, b)
        if e >= worst.get(name, (-1.0,))[0]:
            worst[name] = (e, t, r)

    for t in range(T):
        st = ro.steps[t]
        kin = st["u"].shape[1]
        assert U.shape[2] >= kin
        put("u", t, U[t, :, :kin], st["u"])
        for name, buf in state.items():
            put(name, t, buf[t + 1].reshape(M, -1), st[name].reshape(M, -1))
        put("preds", t, eng.step_preds[t].reshape(M, -1), ro.step_preds[t].reshape(M, -1))
        put("logp", t, eng.step_log_probas[t].reshape(M, 1), ro.step_log_probas[t].reshape(M, 1))
        put("values", t, eng.step_values[t].reshape(M, 1), ro.step_values[t].reshape(M, 1))
    return worst


def _check_forward(key, eng, bound, label):
    ro = _case(key)["ro"]
    assert torch.equal(eng.step_pos.cpu(), ro.step_pos)  # bit-exact in every mode
    worst = _forward_errors(key, eng)
    print(f"\ncase {key} {label}: " + ", ".join(f"{k} {e:.1e} (t={t}, row {r})" for k, (e, t, r) in worst.items()))
    bad = {k: v for k, v in worst.items() if not v[0] < bound[k]}
    assert not bad, f"case {key} {label}: per-row error over the bound: {bad}"


@pytest.mark.gpu
@pytest.mark.parametrize("key", list(CASES))
def test_forward_rows(key):
    model, eng, imgd, inject = _engine(key)
    print(f"\ncase {key} plan: {eng.plan()}")
    assert eng.plan() == {**eng.plan(), **_mplan(key)}
    eng.forward(imgd, *inject)
    torch.cuda.synchronize()
    _check_forward(key, eng, FWD_BOUND, "tf32x3")


@pytest.mark.gpu
@pytest.mark.parametrize("key", ["259", "1190"])
def test_forward_rows_exact_fp32(key):
    """The exact-FFMA kernels (use_tc=False) at ragged M."""
    model, eng, imgd, inject = _engine(key, use_tc=False)
    assert eng.plan()["lstm_tc"] == 0
    eng.forward(imgd, *inject)
    torch.cuda.synchronize()
    _check_forward(key, eng, FWD_BOUND_FP32, "fp32")


def _probe_rows(key, plan):
    """Rows of the last partial 128-row tile and of the last wide batch (the tail probe)."""
    c = CASES[key]
    M = c["na"] * c["nb"]
    first = min(M - plan["lstm_tail_rows"], (plan["cnn_batches"] - 1) * plan["cnn_nw"])
    return torch.arange(first, M)


def _grad_errors(model, ref, label):
    """Per-parameter rel-L2 of the engine's gradients against the oracle's; exact zeros must stay zero."""
    worst, name = 0.0, None
    for k, p in model.named_parameters():
        r = ref[k]
        if r is None or r.norm() == 0:
            assert p.grad.abs().max().item() < 1e-7, (label, k)
            continue
        e = rel_l2(p.grad.cpu(), r)
        if e >= worst:
            worst, name = e, k
    return worst, name


def _oracle_vjp(d, dP, dL, dV):
    ro, p64 = d["ro"], d["p64"]
    out = (ro.step_preds * dP).sum() + (ro.step_log_probas * dL).sum() + (ro.step_values * dV).sum()
    names = list(p64)
    gs = torch.autograd.grad(out, [p64[k] for k in names], retain_graph=True, allow_unused=True)
    return dict(zip(names, gs))


@pytest.mark.gpu
@pytest.mark.parametrize("key", list(CASES))
def test_backward_probes(key):
    c, d = CASES[key], _case(key)
    T, na, nb = c["T"], c["na"], c["nb"]
    M = na * nb
    model, eng, imgd, inject = _engine(key)
    plan = eng.plan()
    nc = eng.step_preds.shape[-1]
    g = torch.Generator().manual_seed(M)
    results = {}
    probes = {"tail": _probe_rows(key, plan), "row": torch.tensor([M // 2])}
    for probe, rows in probes.items():
        mask = torch.zeros(M, dtype=torch.float64)
        mask[rows] = 1.0
        dP = torch.randn(T, M, nc, generator=g, dtype=torch.float64) * mask[None, :, None]
        dL = torch.randn(T, M, generator=g, dtype=torch.float64) * mask[None, :]
        dV = torch.randn(T, M, generator=g, dtype=torch.float64) * mask[None, :]
        ref = _oracle_vjp(d, dP.view(T, na, nb, nc), dL.view(T, na, nb), dV.view(T, na, nb))
        eng.forward(imgd, *inject)
        eng.d_preds.copy_(dP.view(T, na, nb, nc).float())
        eng.d_logp.copy_(dL.view(T, na, nb).float())
        eng.d_values.copy_(dV.view(T, na, nb).float())
        eng.backward(imgd)
        torch.cuda.synchronize()
        model.attach_grads()
        results[probe] = _grad_errors(model, ref, probe) + (len(rows),)
    # the real loss (trainer.py:75-111) through the engine's fused loss
    parts = O.a2c_loss(d["ro"].step_preds, d["ro"].step_log_probas, d["ro"].step_values, d["y"], 0.99)
    names = list(d["p64"])
    ref = dict(zip(names, torch.autograd.grad(parts.loss, [d["p64"][k] for k in names], retain_graph=True,
                                              allow_unused=True)))
    eng.forward(imgd, *inject)
    eng.loss(d["y"].to(DEV))
    eng.backward(imgd)
    torch.cuda.synchronize()
    model.attach_grads()
    results["full"] = _grad_errors(model, ref, "full") + (M,)
    print(f"\ncase {key} probes: " + ", ".join(f"{p} ({n} rows) {e:.1e} [{k}]" for p, (e, k, n) in results.items()))
    bad = {p: v for p, v in results.items() if not v[0] < PROBE_BOUND[p]}
    assert not bad, f"case {key}: worst per-parameter gradient over the bound: {bad}"


@pytest.mark.gpu
def test_graphed_iteration_rows():
    """Case 1190 with rollout, loss and BPTT captured in one CUDA graph and replayed."""
    key = "1190"
    d = _case(key)
    model, eng, imgd, inject = _engine(key)
    _graphed_iteration(eng, imgd, d["y"].to(DEV), *inject)
    _check_forward(key, eng, FWD_BOUND, "graph replay")
    parts = O.a2c_loss(d["ro"].step_preds, d["ro"].step_log_probas, d["ro"].step_values, d["y"], 0.99)
    names = list(d["p64"])
    ref = dict(zip(names, torch.autograd.grad(parts.loss, [d["p64"][k] for k in names], retain_graph=True,
                                              allow_unused=True)))
    model.attach_grads()
    worst, name = _grad_errors(model, ref, "graph")
    print(f"case {key} graph replay: worst per-parameter gradient {worst:.1e} [{name}]")
    assert worst < PROBE_BOUND["full"]

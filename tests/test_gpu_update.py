"""The end of the training step held to fp64 references element by element: the fused actor-critic loss
(csrc/loss.cu), its data-parallel split around the advantage-statistics exchange, the fused Adam (csrc/optim.cu)
and a few steps of the graphed single-GPU ``Trainer``.

The loss reads nothing of the rollout but ``step_preds``, ``step_log_probas`` and ``step_values``, so it is driven
here with synthetic inputs written into the engine's workspace: its launch geometry (8-step batches of the returns
scan, warp loops over the classes, 128- and 256-thread blocks) is exercised at its edges without the rollout.

Errors are measured per element in units of eps32 = 2^-23 of a mixed scale: ``ulps = |got - ref| / (eps32 * (S +
|ref|))``, where S is the natural scale of the quantity (see ``_loss_reference``).  A bound of K ulps is the bound
``|got - ref| <= K eps32 S + K eps32 |ref|``; every K below is under 8388 (1e-3 relative).

* CPU: the case table covers every edge; the fp64 Adam is torch.optim.Adam; the reference's returns, its NaN at one
  advantage and at gamma = 0 (where the engine departs from it on purpose, see ``_engine_returns``).
* ``test_loss_elements``: rewards, returns, advantages, d_preds, d_logp, d_values and the five logged loss values
  against the fp64 oracle with autograd gradients, for five input families per case.
* ``test_loss_graph_replay``: the loss captured in a CUDA graph, replayed over poisoned outputs == eager.
* ``test_sharded_advantage_statistics``: phase A per shard, summed statistics, phase B per shard == full batch.
* ``test_one_advantage_is_nan``: T * Na * Nb == 1 gives the reference's NaN; the Trainer refuses such a batch.
* ``test_adam_*``: the fused Adam through the C ABI against an fp64 Adam: sizes around the vector loop's one-pass
  boundary and the real flat buckets, misaligned views, grad_scale, 2000-step runs, CUDA-graph replay.
* ``test_single_gpu_graph_steps_follow_oracle``: the whole-iteration graph of the single-GPU Trainer follows the
  oracle's fp64 optimisation steps.
"""
import contextlib
import math
from unittest import mock

import numpy as np
import pytest
import torch

from oracle import marl_oracle as O
from tests.conftest import load_golden, oracle_config, rel_l2
from tests.nets import C1_NET, C2_NET, MOVES1, SHIPPED_AID_NET, model_config, oracle_case

DEV = "cuda"
EPS32 = 2.0 ** -23
NAN = float("nan")


def _net(nc):
    """An MNIST-shaped net (f = 6, n = 64) with ``nc`` classes: the loss only sees its class count."""
    return model_config("mnist", 6, 64, 16, 24, 8, 96, 96, nc, MOVES1)


# T: the returns scan walks 8 steps at a time (T % 8 != 0 with T > 8 leaves a partial last batch); Nc: the reward and
# vote warps loop over classes 32 at a time; M = Na * Nb: the returns scan runs 128-thread blocks (M = 129 is one past
# a block), M = 4096 is config 4's shard; Na = 1 has no agent mean, Nb = 1 one image.
LOSS_CASES = {
    "T1_M129": dict(T=1, na=3, nb=43, nc=2, gamma=0.99),
    "T7_na1": dict(T=7, na=1, nb=5, nc=31, gamma=1.0),
    "T8_na16": dict(T=8, na=16, nb=4, nc=32, gamma=0.99),
    "T9_nb1": dict(T=9, na=4, nb=1, nc=33, gamma=0.0),
    "T16_M4096": dict(T=16, na=16, nb=256, nc=45, gamma=0.99),
    "T17": dict(T=17, na=2, nb=7, nc=64, gamma=1.0),
    "T33_M129": dict(T=33, na=1, nb=129, nc=97, gamma=0.99),
    "T35": dict(T=35, na=5, nb=3, nc=65, gamma=0.0),
}
FAMILIES = ("realistic", "large", "smoothl1", "identical", "labels")
SHARDS = [("T8_na16", 2), ("T8_na16", 4), ("T16_M4096", 2), ("T16_M4096", 4)]

# Bounds in ulps (see the module docstring): about 10x the worst over all cases and families, measured on one B200
# (1000 W power limit).  Measured: rewards 0.9, returns 0.85, adv 0.88, d_preds 28, d_logp 23, d_values 29 (d_preds:
# large logits; d_logp / d_values: smooth-L1 boundary at gamma = 0.99 over 33 steps, where |V - G| = 1 cancels
# against |G|), loss 0.47, path 0.61, error 0.33, actor 0.25, critic 1.1; the sharded runs stay below these
LOSS_BOUND = {"rewards": 16, "returns": 16, "adv": 16, "d_preds": 300, "d_logp": 250, "d_values": 300,
              "loss": 16, "path": 16, "error": 16, "actor": 16, "critic": 16}
PARTS = ("loss", "path", "error", "actor", "critic")


# ---------------------------------------------------------------------------------------------------------------
# fp64 references
# ---------------------------------------------------------------------------------------------------------------
def _returns_recursion(r, gamma):
    """G_t = r_t + gamma G_{t+1} over the leading axis, in the dtype of ``r``."""
    out = torch.empty_like(r)
    acc = torch.zeros_like(r[0])
    for t in range(r.shape[0] - 1, -1, -1):
        acc = r[t] + gamma * acc
        out[t] = acc
    return out


@contextlib.contextmanager
def _engine_returns(gamma):
    """The returns the engine is held to.  For gamma > 0 the oracle's, unchanged.  At gamma = 0 the engine departs
    from the reference on purpose (loss.cu, returns_kernel): the reference's closed form is 0/0 there from t = 1 on
    (NaN returns, losses and gradients, pinned by ``test_reference_returns_are_nan_at_gamma_0``), while the engine
    computes the recursion's G_t = r_t.  There, and only there, the oracle runs with ``_returns_recursion`` for its
    returns; everything else in its loss is its own."""
    if gamma != 0:
        yield
        return
    with mock.patch.object(O, "discounted_returns", _returns_recursion):
        yield


def _loss_inputs(key, family):
    """fp32 preds [T,Na,Nb,Nc], log-probs, values [T,Na,Nb] and int64 targets [Nb] of one input family."""
    c = LOSS_CASES[key]
    T, na, nb, nc = c["T"], c["na"], c["nb"], c["nc"]
    g = torch.Generator().manual_seed(17 * T + 1000 * nc + 7 * na * nb + FAMILIES.index(family))
    y = torch.randint(nc, (nb,), generator=g)
    if family == "labels":  # only the extreme classes
        y = torch.where(torch.arange(nb) % 2 == 0, nc - 1, 0)
    if family == "large":  # |x| up to 100: exp(x) overflows fp32 from x = 88.7 without the max subtraction
        preds = (torch.rand(T, na, nb, nc, generator=g) * 2 - 1) * 100
    else:  # logits at a scale of 1 to 3
        preds = torch.randn(T, na, nb, nc, generator=g) * (1 + 2 * torch.rand(T, na, nb, 1, generator=g))
    if family == "identical":
        preds = preds[:, :1].expand(T, na, nb, nc).contiguous()
    logp = torch.rand(T, na, nb, generator=g).clamp_min(1e-4).log()
    values = torch.randn(T, na, nb, generator=g)
    if family == "smoothl1":  # |V - G| = 1 -+ 1e-3: both branches of smooth_l1 on known elements
        with _engine_returns(c["gamma"]):
            ret = O.discounted_returns(O.classification_rewards(preds.double(), y), c["gamma"])
        sign = torch.randint(2, (T, na, nb), generator=g).double() * 2 - 1
        side = torch.randint(2, (T, na, nb), generator=g).double() * 2 - 1
        values = (ret + sign * (1 + side * 1e-3)).float()
    return preds, logp, values, y


def _loss_reference(preds, logp, values, y, gamma, adv_stats=None):
    """The oracle's loss in fp64 on the fp32 inputs, its gradients with respect to the three inputs, and the scale
    S of every quantity (at gamma = 0 with the engine's returns, see ``_engine_returns``):
    rewards   (2 max_c |x_c| + ln Nc) / ln Nc        (the cross-entropy's cancellation)
    returns   sum_k gamma^k (|r_{t+k}| + S_r(t+k))     adv: S_G + |V|
    d_preds   1 / (Na Nb)                             d_logp, d_values: 1 / M
    path      sum |logp nadv| / M                     error: mean_{t,b} (|lse| + |vote_y|)
    critic    itself                                  loss / actor: their terms' scales added."""
    T, na, nb, nc = preds.shape
    P, L, V = (t.double().requires_grad_(True) for t in (preds, logp, values))
    with _engine_returns(gamma):
        parts = O.a2c_loss(P, L, V, y, gamma, adv_stats)
        dP, dL, dV = torch.autograd.grad(parts.loss, (P, L, V))
        P, L, V = P.detach(), L.detach(), V.detach()
        rew = O.classification_rewards(P, y)
        ret = O.discounted_returns(rew, gamma)
    adv = ret - V
    lnc = math.log(nc)
    s_rew = (2 * P.abs().amax(-1) + lnc) / lnc
    s_ret = _returns_recursion(rew.abs() + s_rew, gamma)
    if adv_stats is None:
        adv_stats = (adv.mean(), adv.std())
    nadv = (adv - adv_stats[0]) / (adv_stats[1] + 1e-8)
    M = na * nb
    vote = P.mean(1)  # [T, nb, nc]
    lse = vote.logsumexp(-1)
    vy = vote.gather(-1, y.view(1, nb, 1).expand(T, nb, 1)).squeeze(-1)
    s_path = float((L * nadv).abs().sum() / M)
    s_err = float((lse.abs() + vy.abs()).mean())
    s_crit = float(parts.critic.detach())
    ref = dict(rewards=rew, returns=ret, adv=adv, d_preds=dP, d_logp=dL, d_values=dV,
               **{k: getattr(parts, k).detach() for k in PARTS})
    one = torch.ones(())
    scale = dict(rewards=s_rew, returns=s_ret, adv=s_ret + V.abs(), d_preds=one / M, d_logp=one / M,
                 d_values=one / M, loss=one * (s_path + T * s_err + s_crit), path=one * s_path, error=one * s_err,
                 actor=one * (s_path + T * s_err), critic=one * s_crit)
    return ref, scale


def _ulps(got, ref, scale, floor=0.0):
    """(worst |got - ref| / (eps32 (S + |ref|) + floor), flat index of the worst element); NaN counts as inf."""
    got = got.detach().double().cpu()
    ref = ref.detach().double()
    q = (got - ref).abs() / (EPS32 * (scale + ref.abs()) + floor)
    q = torch.nan_to_num(q.reshape(-1), nan=math.inf)
    i = int(q.argmax())
    return float(q[i]), i


# ---------------------------------------------------------------------------------------------------------------
# CPU checks
# ---------------------------------------------------------------------------------------------------------------
def test_loss_case_table_covers_the_edges():
    cs = list(LOSS_CASES.values())
    Ts = {c["T"] for c in cs}
    assert {1, 7, 8, 9, 16, 17} <= Ts and max(Ts) >= 33
    assert any(c["T"] > 8 and c["T"] % 8 for c in cs)  # a partial last batch of the returns scan after a full one
    ncs = {c["nc"] for c in cs}
    assert {2, 31, 32, 33, 45, 64} <= ncs and max(ncs) >= 65
    assert any(c["na"] == 1 for c in cs) and any(c["na"] >= 16 for c in cs)
    assert any(c["nb"] == 1 for c in cs)
    Ms = {c["na"] * c["nb"] for c in cs}
    assert 129 in Ms and 4096 in Ms
    assert {c["gamma"] for c in cs} == {0.99, 1.0, 0.0}
    for key, k in SHARDS:
        assert LOSS_CASES[key]["nb"] % k == 0
    assert any(LOSS_CASES[key]["nb"] // k == 1 for key, k in SHARDS)  # a shard of one image
    assert {k for _, k in SHARDS} == {2, 4}


def test_returns_reference_is_the_recursion():
    """For gamma > 0 the oracle's closed form (functions.py:35-51) is the recursion G_t = r_t + gamma G_{t+1} the
    engine computes."""
    r = torch.randn(35, 3, 4, dtype=torch.float64, generator=torch.Generator().manual_seed(0))
    for gamma in (0.5, 0.99, 1.0):
        assert torch.allclose(O.discounted_returns(r, gamma), _returns_recursion(r, gamma), rtol=1e-12, atol=1e-12)


def test_reference_returns_are_nan_at_gamma_0():
    """The reference at gamma = 0: its closed form divides 0 by 0 from t = 1 on, so its returns there, and its loss,
    critic loss and gradients, are NaN (only t = 0 and the vote error survive).  The engine departs from it on
    purpose there (loss.cu, returns_kernel): its returns are the rewards, the recursion's value."""
    g = torch.Generator().manual_seed(3)
    r = torch.randn(9, 4, 1, dtype=torch.float64, generator=g)
    ret = O.discounted_returns(r, 0.0)
    assert torch.equal(ret[0], r[0]) and torch.isnan(ret[1:]).all()
    assert torch.equal(_returns_recursion(r, 0.0), r)
    preds = torch.randn(9, 4, 1, 33, dtype=torch.float64, generator=g)
    logp, values = -torch.rand(9, 4, 1, dtype=torch.float64, generator=g), torch.randn(9, 4, 1, dtype=torch.float64)
    parts = O.a2c_loss(preds, logp, values, torch.tensor([32]), 0.0)
    assert all(math.isnan(float(getattr(parts, k))) for k in ("loss", "path", "actor", "critic"))
    assert math.isfinite(float(parts.error))
    assert any(c["gamma"] == 0 and c["T"] > 1 for c in LOSS_CASES.values())  # the departure is exercised on the GPU


@pytest.mark.filterwarnings(r"ignore:std\(\)")
def test_reference_loss_is_nan_for_one_advantage():
    """torch.std of one element is NaN: the reference's loss (and its path / actor parts) are NaN when
    T * Na * Nb == 1, while the vote error and the critic loss stay finite."""
    g = torch.Generator().manual_seed(1)
    preds, logp, values = torch.randn(1, 1, 1, 10, generator=g), -torch.rand(1, 1, 1, generator=g), torch.randn(1, 1, 1)
    parts = O.a2c_loss(preds.double(), logp.double(), values.double(), torch.tensor([3]), 0.99)
    assert all(math.isnan(float(getattr(parts, k))) for k in ("loss", "path", "actor"))
    assert math.isfinite(float(parts.error)) and math.isfinite(float(parts.critic))


def _adam_reference(p, m, v, g, t, lr, b1, b2, eps, grad_scale):
    """One step of torch.optim.Adam (no weight decay, not amsgrad) in the dtype of its inputs; ``t`` counts this
    step: step_size = lr / (1 - b1^t), denom = sqrt(v) / sqrt(1 - b2^t) + eps."""
    g = g * grad_scale
    m = b1 * m + (1 - b1) * g
    v = b2 * v + (1 - b2) * g * g
    denom = v.sqrt() / math.sqrt(1 - b2 ** t) + eps
    return p - (lr / (1 - b1 ** t)) * (m / denom), m, v


def _adam_grads(n, steps, seed):
    """[steps, n] fp32 gradients mixing N(0, 1), exact zeros, ~1e-20 and ~1e3."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(steps, n, generator=g)
    kind = torch.randint(4, (steps, n), generator=g)
    x = torch.where(kind == 1, torch.zeros(()), x)
    x = torch.where(kind == 2, x * 1e-20, x)
    return torch.where(kind == 3, x * 1e3, x)


def test_adam_reference_is_torch_adam():
    n, lr = 1000, 3e-3
    grads = _adam_grads(n, 60, 5).double()
    p0 = torch.randn(n, dtype=torch.float64, generator=torch.Generator().manual_seed(6))
    for b1, b2, eps, scale in ((0.9, 0.999, 1e-8, 1.0), (0.8, 0.99, 1e-6, 0.125)):
        ref = p0.clone().requires_grad_(True)
        opt = torch.optim.Adam([ref], lr=lr, betas=(b1, b2), eps=eps, foreach=False)
        p, m, v = p0.clone(), torch.zeros(n, dtype=torch.float64), torch.zeros(n, dtype=torch.float64)
        sm = torch.zeros(n, dtype=torch.float64)  # the same average of |g|: the scale m cancels against
        for t in range(1, grads.shape[0] + 1):
            ref.grad = grads[t - 1] * scale
            opt.step()
            p, m, v = _adam_reference(p, m, v, grads[t - 1], t, lr, b1, b2, eps, scale)
            sm = b1 * sm + (1 - b1) * (grads[t - 1] * scale).abs()
        st = opt.state[ref]
        assert ((p - ref.detach()).abs() <= 1e-13 * (lr + p.abs())).all()
        assert ((m - st["exp_avg"]).abs() <= 1e-13 * sm).all()
        assert ((v - st["exp_avg_sq"]).abs() <= 1e-13 * v).all()


ADAM_ONE_PASS = 148 * 8 * 256 * 4  # floats one pass of the vector loop covers (blocks capped at 148 * 8): 1 212 416
# ONE_PASS + {-1, 0, 3} end the vector loop exactly at or before one pass (at + 3 only the scalar tail follows);
# ONE_PASS + 1027 gives 256 float4 of a second vector pass and a 3-element tail, as do the real flat buckets
ADAM_NETS = {"c2": C2_NET, "shipped_aid": SHIPPED_AID_NET}


def _bucket_floats(mc):
    from marlclassification_b200.config import ModelConfig

    return ModelConfig(**mc).build_networks()._layout()[1]


def test_adam_sizes_cross_the_one_pass_boundary():
    """The flat buckets of the c2 and shipped AID nets take more than one pass of the vector loop."""
    sizes = {k: _bucket_floats(mc) for k, mc in ADAM_NETS.items()}
    print(f"flat buckets: {sizes}; one pass = {ADAM_ONE_PASS}")
    assert all(s > ADAM_ONE_PASS + 3 for s in sizes.values()), sizes


# ---------------------------------------------------------------------------------------------------------------
# GPU: the fused loss
# ---------------------------------------------------------------------------------------------------------------
_MODELS = {}


def _model(nc):
    from marlclassification_b200.config import ModelConfig

    if nc not in _MODELS:
        model = ModelConfig(**_net(nc)).build_networks()
        model.to(DEV)
        _MODELS[nc] = model
    return _MODELS[nc]


def _engine(key, nb=None, T=None, na=None):
    from marlclassification_b200.engine import EpisodeEngine

    c = LOSS_CASES[key] if key is not None else {}
    nc = c.get("nc", 10)
    return EpisodeEngine(_model(nc), na=na or c["na"], nb=nb or c["nb"], T=T or c["T"], C=3, H=12, W=12,
                         actions=MOVES1, gamma=c.get("gamma", 0.99))


def _outputs(eng):
    T, na, nb = eng.T, eng.na, eng.nb
    f32 = torch.float32
    return dict(rewards=eng.view("rewards", f32, (T, na, nb)), returns=eng.view("returns", f32, (T, na, nb)),
                adv=eng.view("adv", f32, (T, na, nb)), d_preds=eng.d_preds, d_logp=eng.d_logp, d_values=eng.d_values)


def _write_inputs(eng, preds, logp, values):
    eng.step_preds.copy_(preds)
    eng.step_log_probas.copy_(logp)
    eng.step_values.copy_(values)
    for t in _outputs(eng).values():  # whatever the loss fails to write stays NaN
        t.fill_(NAN)


def _loss_errors(out, loss_out, ref, scale):
    """{quantity: (ulps, flat index)} of one run."""
    err = {k: _ulps(out[k], ref[k], scale[k]) for k in ("rewards", "returns", "adv", "d_preds", "d_logp", "d_values")}
    for i, k in enumerate(PARTS):
        err[k] = _ulps(loss_out[i], ref[k], scale[k])
    return err


@pytest.mark.gpu
@pytest.mark.parametrize("key", list(LOSS_CASES))
def test_loss_elements(key):
    c = LOSS_CASES[key]
    eng = _engine(key)
    worst = {}
    for family in FAMILIES:
        preds, logp, values, y = _loss_inputs(key, family)
        ref, scale = _loss_reference(preds, logp, values, y, c["gamma"])
        _write_inputs(eng, preds.to(DEV), logp.to(DEV), values.to(DEV))
        loss_out = eng.loss(y.to(DEV)).clone()
        torch.cuda.synchronize()
        assert loss_out[5].item() == 0
        if family == "smoothl1":  # both branches of smooth_l1 were taken, on known elements
            x = (values.double() - ref["returns"]).abs()
            assert (x < 1 - 5e-4).any() and (x > 1 + 5e-4).any()
        errs = _loss_errors(_outputs(eng), loss_out.cpu(), ref, scale)
        for k, (e, i) in errs.items():
            if e >= worst.get(k, (-1.0,))[0]:
                worst[k] = (e, family, i)
    print(f"\nloss {key}: " + ", ".join(f"{k} {e:.2g} ({f}@{i})" for k, (e, f, i) in worst.items()))
    bad = {k: v for k, v in worst.items() if not v[0] <= LOSS_BOUND[k]}
    assert not bad, f"case {key}: ulps over the bound: {bad}"


@pytest.mark.gpu
@pytest.mark.parametrize("key", ["T9_nb1", "T33_M129"])
def test_loss_graph_replay(key):
    """The loss captured in a CUDA graph and replayed twice over NaN-poisoned outputs equals the eager loss bit for
    bit."""
    eng = _engine(key)
    preds, logp, values, y = _loss_inputs(key, "realistic")
    yd = y.to(DEV)
    _write_inputs(eng, preds.to(DEV), logp.to(DEV), values.to(DEV))
    eager_out = eng.loss(yd).clone()
    eager = {k: t.clone() for k, t in _outputs(eng).items()}
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        eng.loss(yd)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        eng.loss(yd)
    for _ in range(2):
        for t in _outputs(eng).values():
            t.fill_(NAN)
        eng.loss_out.fill_(NAN)
        graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(eng.loss_out[:6], eager_out[:6])
    for k, t in _outputs(eng).items():
        assert torch.equal(t, eager[k]), k


@pytest.mark.gpu
@pytest.mark.parametrize("key,k", SHARDS)
def test_sharded_advantage_statistics(key, k):
    """The data-parallel protocol on one GPU: phase A on each of k shards, the sum of their loss_stats[:3] (what
    DataParallelContext.all_reduce_stats computes) written into every shard, phase B; the shard gradients
    concatenated and scaled by 1/k (the trainer's grad_scale) are the full batch's."""
    c = LOSS_CASES[key]
    T, na, nb = c["T"], c["na"], c["nb"]
    per = nb // k
    preds, logp, values, y = _loss_inputs(key, "realistic")
    ref, scale = _loss_reference(preds, logp, values, y, c["gamma"])
    raw = ref["adv"]
    stats = (raw.mean(), raw.std())
    engs = [_engine(key, nb=per) for _ in range(k)]
    sl = [slice(s * per, (s + 1) * per) for s in range(k)]
    for e, s in zip(engs, sl):
        _write_inputs(e, preds[:, :, s].to(DEV), logp[:, :, s].to(DEV), values[:, :, s].to(DEV))
        e.loss_phase_a(y[s].to(DEV))
    total = torch.stack([e.loss_stats[:3] for e in engs]).sum(0)
    for e in engs:
        e.loss_stats[:3].copy_(total)
        e.loss_phase_b()
    torch.cuda.synchronize()
    worst = {}
    for name in ("d_preds", "d_logp", "d_values"):
        got = torch.cat([getattr(e, name).cpu() for e in engs], dim=2) / k
        worst[name] = _ulps(got, ref[name], scale[name])
    for name in ("rewards", "returns", "adv"):
        got = torch.cat([_outputs(e)[name].cpu() for e in engs], dim=2)
        worst[name] = _ulps(got, ref[name], scale[name])
    for s, e in zip(sl, engs):
        sref, sscale = _loss_reference(preds[:, :, s], logp[:, :, s], values[:, :, s], y[s], c["gamma"], stats)
        out = e.loss_out.cpu()
        for i, name in enumerate(PARTS):
            w = _ulps(out[i], sref[name], sscale[name])
            if w[0] >= worst.get(name, (-1.0,))[0]:
                worst[name] = w
    print(f"\nshards {key} k={k}: " + ", ".join(f"{n} {e:.2g}" for n, (e, _) in worst.items()))
    bad = {n: v for n, v in worst.items() if not v[0] <= LOSS_BOUND[n]}
    assert not bad, f"{key} k={k}: ulps over the bound: {bad}"


@pytest.mark.gpu
@pytest.mark.filterwarnings(r"ignore:std\(\)")
def test_one_advantage_is_nan():
    """T * Na * Nb == 1: the engine's loss, path and actor loss and d_logp are NaN, as the reference's are; the
    vote error, the critic loss, d_preds and d_values stay finite and right.  The Trainer refuses such a batch
    before it updates anything."""
    from marlclassification_b200.config import ModelConfig
    from marlclassification_b200.core import EpisodeSampler
    from marlclassification_b200.training import Trainer

    eng = _engine(None, na=1, nb=1, T=1)
    g = torch.Generator().manual_seed(2)
    preds, logp, values = torch.randn(1, 1, 1, 10, generator=g), -torch.rand(1, 1, 1, generator=g), torch.randn(1, 1, 1)
    y = torch.tensor([9])
    ref, scale = _loss_reference(preds, logp, values, y, 0.99)
    _write_inputs(eng, preds.to(DEV), logp.to(DEV), values.to(DEV))
    out = eng.loss(y.to(DEV)).cpu()
    for i, name in enumerate(PARTS):
        assert math.isnan(out[i]) == math.isnan(ref[name]), name
    assert torch.isnan(ref["d_logp"]).all() and torch.isnan(eng.d_logp).all()
    for name in ("error", "critic"):
        assert _ulps(out[PARTS.index(name)], ref[name], scale[name])[0] <= LOSS_BOUND[name]
    for name in ("rewards", "returns", "adv", "d_preds", "d_values"):
        assert _ulps(_outputs(eng)[name], ref[name], scale[name])[0] <= LOSS_BOUND[name], name

    model, marl, env = ModelConfig(**_net(10)).build_marl(1)
    model.to(DEV)
    trainer = Trainer(model, 10, 1e-3, 0.99)
    before = model.flat_params.clone()
    with pytest.raises(RuntimeError, match="single advantage"):
        trainer.train_step(torch.rand(1, 3, 28, 28, device=DEV), y.to(DEV), EpisodeSampler(marl, env, 1))
    assert torch.equal(model.flat_params, before)


# ---------------------------------------------------------------------------------------------------------------
# GPU: the fused Adam
# ---------------------------------------------------------------------------------------------------------------
LR = 1e-3
B1, B2, ADAM_EPS = 0.9, 0.999, 1e-8
# what the kernel receives through the C ABI's float parameters: the fp64 reference runs with the same betas
B1_32, B2_32, EPS_32 = (float(np.float32(x)) for x in (B1, B2, ADAM_EPS))
# about 10x the worst ulps measured on one B200 (1000 W power limit), over every size, alignment and grad_scale:
# m 0.7, v 2.3, p 4.1
ADAM_BOUND = {"m": 8, "v": 24, "p": 40}
ADAM_LONG_BOUND = 3  # ulps of p per step taken, over the checkpoints of the long run; measured 0.26 (2.6 ulps at step
# 10, 218 at step 2000)
ADAM_SIZES = [1, 2, 3, 4, 5, 4095, ADAM_ONE_PASS - 1, ADAM_ONE_PASS, ADAM_ONE_PASS + 3, ADAM_ONE_PASS + 1027, "c2",
              "shipped_aid"]
DENORM = 2.0 ** -149  # one ulp below the normal range: v of a ~1e-20 gradient is subnormal in fp32


def _adam_step(p, g, m, v, step, scale):
    from marlclassification_b200 import _lib

    _lib.check(_lib.lib().marlc_adam_step(p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), p.numel(), LR, B1,
                                          B2, ADAM_EPS, scale, step.data_ptr(), _lib.stream_ptr(p.device)))


def _at_offset(x, off):
    """A view of a copy of ``x`` at ``off`` floats into its device buffer (off = 1..3: not 16-byte aligned)."""
    buf = torch.empty(x.numel() + 4, dtype=torch.float32, device=DEV)
    view = buf[off: off + x.numel()]
    view.copy_(x)
    return view


@pytest.mark.gpu
@pytest.mark.parametrize("n", ADAM_SIZES)
def test_adam_steps(n):
    """exp_avg, exp_avg_sq and the parameters after steps 1-3 of the fused Adam against the fp64 Adam, element by
    element, for 16-byte aligned buffers and views that force the scalar path, at grad_scale 1 and 1/8."""
    if isinstance(n, str):
        n = _bucket_floats(ADAM_NETS[n])
    big = n > 2 * ADAM_ONE_PASS
    offsets = [(0, 0, 0, 0), (3, 3, 3, 3)] if big else [(0, 0, 0, 0), (1, 1, 1, 1), (2, 2, 2, 2), (3, 3, 3, 3),
                                                         (0, 2, 0, 0)]
    grads = _adam_grads(n, 3, n)
    p0 = torch.randn(n, generator=torch.Generator().manual_seed(n + 1))
    worst = {}
    for scale in (1.0, 0.125):
        for offs in offsets:
            p, m, v = (_at_offset(x, o) for x, o in zip((p0, torch.zeros(n), torch.zeros(n)), (offs[0], offs[2], offs[3])))
            g = _at_offset(torch.zeros(n), offs[1])
            step = torch.zeros(1, dtype=torch.int64, device=DEV)
            rp, rm, rv = p0.double(), torch.zeros(n, dtype=torch.float64), torch.zeros(n, dtype=torch.float64)
            sm = torch.zeros(n, dtype=torch.float64)  # the scale of exp_avg: the same average of |g|
            for t in range(1, 4):
                g.copy_(grads[t - 1])
                _adam_step(p, g, m, v, step, scale)
                gd = grads[t - 1].double()
                rp, rm, rv = _adam_reference(rp, rm, rv, gd, t, LR, B1_32, B2_32, EPS_32, scale)
                sm = B1_32 * sm + (1 - B1_32) * gd.abs() * scale
                errs = {"m": _ulps(m, rm, sm, DENORM), "v": _ulps(v, rv, 0.0, DENORM), "p": _ulps(p, rp, LR)}
                for k, (e, i) in errs.items():
                    if e >= worst.get(k, (-1.0,))[0]:
                        worst[k] = (e, t, scale, offs, i)
            assert step.item() == 3
    print(f"\nadam n={n}: " + ", ".join(f"{k} {w[0]:.1f} (step {w[1]}, scale {w[2]}, offsets {w[3]}, i {w[4]})"
                                         for k, w in worst.items()))
    bad = {k: w for k, w in worst.items() if not w[0] <= ADAM_BOUND[k]}
    assert not bad, f"n={n}: ulps over the bound: {bad}"


@pytest.mark.gpu
@pytest.mark.parametrize("n,off", [(4099, 0), (4099, 1)])
def test_adam_long_run(n, off):
    """2000 steps on fresh gradients every step: the parameters after steps 10, 100, 1000 and 2000 stay within a
    cumulative bound |dp| <= steps * K * eps32 (lr + |p|), and the device step counter counts them."""
    steps = 2000
    grads = _adam_grads(n, steps, 99).to(DEV)
    p0 = torch.randn(n, generator=torch.Generator().manual_seed(3))
    p, m, v = (_at_offset(x, off) for x in (p0, torch.zeros(n), torch.zeros(n)))
    g = _at_offset(torch.zeros(n), off)
    step = torch.zeros(1, dtype=torch.int64, device=DEV)
    rp, rm, rv = p0.double(), torch.zeros(n, dtype=torch.float64), torch.zeros(n, dtype=torch.float64)
    cpu = grads.double().cpu()
    seen = []
    for t in range(1, steps + 1):
        g.copy_(grads[t - 1])
        _adam_step(p, g, m, v, step, 0.125)
        rp, rm, rv = _adam_reference(rp, rm, rv, cpu[t - 1], t, LR, B1_32, B2_32, EPS_32, 0.125)
        if t in (10, 100, 1000, 2000):
            assert step.item() == t
            e, i = _ulps(p, rp, LR)
            seen.append((t, e, e / t, i))
    print(f"\nadam long run n={n} off={off}: " + ", ".join(f"step {t}: {e:.1f} ulps ({r:.2f} per step)"
                                                         for t, e, r, _ in seen))
    assert max(r for _, _, r, _ in seen) <= ADAM_LONG_BOUND, seen


@pytest.mark.gpu
@pytest.mark.parametrize("n,off", [(ADAM_ONE_PASS + 3, 0), (4095, 1)])
def test_adam_graph_replay(n, off):
    """K steps captured in one CUDA graph and replayed twice == 2K eager steps, bit for bit (step counter too)."""
    K = 5
    p0 = torch.randn(n, generator=torch.Generator().manual_seed(4))
    grad = _adam_grads(n, 1, 8)[0]
    runs = []
    for graphed in (False, True):
        p, m, v, g = (_at_offset(x, off) for x in (p0, torch.zeros(n), torch.zeros(n), grad))
        step = torch.zeros(1, dtype=torch.int64, device=DEV)
        if graphed:
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                for _ in range(K):
                    _adam_step(p, g, m, v, step, 0.125)
            graph.replay()
            graph.replay()
        else:
            for _ in range(2 * K):
                _adam_step(p, g, m, v, step, 0.125)
        torch.cuda.synchronize()
        runs.append((p.clone(), m.clone(), v.clone(), step.clone()))
    assert runs[1][3].item() == 2 * K
    for a, b in zip(*runs):
        assert torch.equal(a, b)


# ---------------------------------------------------------------------------------------------------------------
# GPU: the single-GPU Trainer's whole-iteration graph against the oracle's optimisation steps
# ---------------------------------------------------------------------------------------------------------------
TRAJ_STEPS = 8
# about 10x the worst measured on one B200 (1000 W power limit): loss parts 1.6e-7,
# per-tensor update 2.2e-5, parameters 1.2e-7
TRAJ_BOUND = {"loss": 2e-6, "update": 3e-4, "params": 2e-6}


def _trajectory_case(name):
    if name == "conftest_odd":
        fx = load_golden(name)
        return (fx["model_config"], fx["na"], fx["T"], fx["gamma"], fx["state_dict"], fx["img"], fx["targets"],
                fx["pos0"], fx["hidden0"], fx["actions"])
    spec = dict(mc=C1_NET, na=3, nb=32, T=5, C=3, H=28, W=28)  # BASELINE config 1
    ocfg, params, img, y, pos0, hidden0, actions = oracle_case(spec)
    return spec["mc"], spec["na"], spec["T"], 0.99, params, img, y, pos0, hidden0, actions


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["conftest_odd", "c1_mnist"])
def test_single_gpu_graph_steps_follow_oracle(name):
    from marlclassification_b200.config import ModelConfig
    from marlclassification_b200.core import EpisodeSampler
    from marlclassification_b200.training import Trainer

    mc, na, T, gamma, state, img, y, pos0, hidden0, actions = _trajectory_case(name)
    model, marl, env = ModelConfig(**mc).build_marl(na)
    model.load_state_dict(state)
    model.to(DEV)
    assert model.use_tc and model.precision == "tf32x3"
    sampler = EpisodeSampler(marl, env, T, gamma=gamma)
    trainer = Trainer(model, mc["nb_class"], LR, gamma, cuda_graph=True)
    inject = dict(pos0=pos0.to(DEV), hidden0=[h.to(DEV) for h in hidden0], actions=actions.to(DEV))
    imgd, yd = img.to(DEV), y.to(DEV)
    outs = [trainer.train_step(imgd, yd, sampler, **inject)[:5].clone() for _ in range(TRAJ_STEPS)]
    torch.cuda.synchronize()
    step = next(iter(trainer._Trainer__steps.values()))
    assert step._graphs[True] is not None and len(step._graphs[True]) == 1, "no whole-iteration graph was captured"

    parts = []
    new, _ = O.train_steps({k: v.double() for k, v in state.items()}, oracle_config(mc), img.double(), y, pos0,
                           [h.double() for h in hidden0], actions, T, gamma, LR, TRAJ_STEPS, parts_out=parts)
    got = torch.stack(outs).double().cpu()
    ref = torch.tensor(parts, dtype=torch.float64)
    # each step's five values, relative to the largest of them
    e_loss = float(((got - ref).abs() / ref.abs().amax(1, keepdim=True)).max())
    worst, worst_k = 0.0, ""
    params = {k: p.detach().cpu() for k, p in model.named_parameters()}
    for k, p0 in state.items():
        upd_ref = new[k] - p0.double()
        if upd_ref.norm() == 0:
            continue
        err = rel_l2(params[k].double() - p0.double(), upd_ref)
        if err > worst:
            worst, worst_k = err, k
    flat = lambda d: torch.cat([d[k].double().flatten() for k in state])  # noqa: E731
    e_params = rel_l2(flat(params), flat(new))
    print(f"\ntrajectory {name}: loss parts {e_loss:.2e}, worst per-tensor update rel-L2 {worst:.2e} "
          f"({worst_k.split('__')[-1]}), params rel-L2 {e_params:.2e}; oracle loss {ref[0, 0]:.4f} -> {ref[-1, 0]:.4f}")
    assert e_loss < TRAJ_BOUND["loss"]
    assert worst < TRAJ_BOUND["update"], (worst_k, worst)
    assert e_params < TRAJ_BOUND["params"]

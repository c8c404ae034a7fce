"""The step-wise API in training: ``model.differentiable_steps = True`` gives ``ModelsWrapper.forward`` /
``MultiAgent.act`` a backward (``marlc_model_step_backward``).

* One step against the fp64 oracle: random gradients on all eight outputs; per-parameter gradients (rel-L2) and
  the input gradients d msg, d h, d c, d h^, d c^ per row (``row_err``) against ``torch.autograd.grad`` of
  ``O.step_forward`` in fp64.  Geometries: the odd-sized fixture, the c2 net at M = 128 and single-step versions
  of the regime cases of ``test_gpu_regimes.py``.
* Isolation probes: the gradient on one output at a time, then on one row only.
* Episodes composed from ``act`` / ``env.step``: the loss of the stacked outputs, backpropagated, against the
  reference's recorded gradients and against ``run_episode``.
* Accumulation, the flat gradient bucket, the guards, and that the fused episode is unchanged.
"""
import pytest
import torch

from oracle import marl_oracle as O
from tests.conftest import GOLDEN_NAMES, load_golden, oracle_config, rel_l2
from tests.test_gpu_configs import C2_NET, CONFIGS
from tests.test_gpu_regimes import CASES, row_err

DEV = "cuda"
OUTS = ("probs", "values", "preds", "msg", "h", "c", "h_caret", "c_caret")
INS = ("msg", "h", "c", "h_caret", "c_caret")

# geometries of one step: (net, na, nb)
_ODD = load_golden("conftest_odd")
STEPS = {"conftest_odd": (_ODD["model_config"], _ODD["na"], _ODD["nb"]), "c2_m128": (C2_NET, 16, 8)}
STEPS.update({key: (CASES[key]["net"], CASES[key]["na"], CASES[key]["nb"]) for key in
              ("93", "259", "1795", "4098", "261", "300")})
# (geometry, mode): tf32x3 everywhere, exact fp32 on two, the unfused kernels (use_chains = False) on one
MODES = [(k, "tf32x3") for k in STEPS] + [("conftest_odd", "fp32"), ("259", "fp32"), ("93", "unfused")]

# Bounds: about 10x the worst error measured on one NVIDIA B200 (1000 W power limit), never above 1e-3.
# measured, tf32x3:  parameters 2.5e-5 (case 4098, first conv layer), inputs per row msg 2.3e-5, h 7.9e-6, c 3.5e-6,
#                    h^ 7.7e-6, c^ 2.3e-6
# measured, fp32:    parameters 4.6e-6, inputs per row 1.2e-6
# measured, unfused: parameters 3.7e-6, inputs per row 2.8e-6
BOUND = {"tf32x3": {"param": 3e-4, "input": 3e-4}, "fp32": {"param": 5e-5, "input": 2e-5},
         "unfused": {"param": 5e-5, "input": 3e-5}}
PROBE_BOUND = 7e-5  # measured 6.7e-6 (case 259, gradient on probs only)
TOL = 1e-3  # the bar of test_gpu_parity.py against the reference's recorded gradients (measured at most 1.8e-5)
RUN_EPISODE_BOUND = 2e-5  # against run_episode + the same loss: measured at most 1.7e-6


def _model(mc, na, mode, params):
    from marlclassification_b200.config import ModelConfig

    model, marl, env = ModelConfig(**mc).build_marl(na)
    model.use_tc = mode != "fp32"
    model.use_chains = mode != "unfused"
    model.load_state_dict(params)
    model.to(DEV)
    model.differentiable_steps = True
    return model, marl, env


def _inputs(ocfg, na, nb, seed):
    g = torch.Generator().manual_seed(seed)
    C = 3
    patch = torch.rand(na, nb, C, ocfg.f, ocfg.f, generator=g)
    msg = torch.randn(na, nb, ocfg.n_m, generator=g)
    npos = torch.rand(na, nb, 2, generator=g) * 2 - 1
    hid = [torch.randn(na, nb, n, generator=g) for n in (ocfg.n_b, ocfg.n_b, ocfg.n_a, ocfg.n_a)]
    return patch, msg, npos, hid


def _oracle(params, ocfg, patch, msg, npos, hid, d_out):
    """fp64 gradients of sum_k <out_k, d_out_k> w.r.t. every parameter and msg, h, c, h^, c^."""
    p64 = {k: v.double().requires_grad_(True) for k, v in params.items()}
    ins = [x.double().requires_grad_(True) for x in (msg, *hid)]
    probs, values, preds, new_msg, new_hid = O.step_forward(p64, ocfg, patch.double(), ins[0], npos.double(),
                                                            tuple(ins[1:]))
    outs = (probs, values, preds, new_msg, *new_hid)
    total = sum((o * g.double()).sum() for o, g in zip(outs, d_out) if g is not None)
    names = list(p64)
    gs = torch.autograd.grad(total, [p64[k] for k in names] + ins, allow_unused=True)
    zero = lambda x, g: torch.zeros_like(x) if g is None else g  # noqa: E731
    return dict(zip(names, gs[:len(names)])), [zero(x, g) for x, g in zip(ins, gs[len(names):])]


def _engine_step(model, patch, msg, npos, hid, d_out):
    from marlclassification_b200.networks.models import RecurrentOutput

    ins = [x.to(DEV).requires_grad_(True) for x in (msg, *hid)]
    model.zero_grad(set_to_none=True)
    out, rec = model(patch.to(DEV), ins[0], npos.to(DEV), RecurrentOutput(*ins[1:]))
    outs = (out.actions_probabilities, out.values, out.predictions, out.messages, rec.h, rec.c, rec.h_caret,
            rec.c_caret)
    pairs = [(o, g.to(DEV)) for o, g in zip(outs, d_out) if g is not None]
    torch.autograd.backward([o for o, _ in pairs], [g for _, g in pairs])
    torch.cuda.synchronize()
    return ins


def _compare(model, ins, ref_p, ref_in, na, nb, label):
    """(worst per-parameter rel-L2, its name), {input: worst per-row error}; exact zeros must stay (near) zero."""
    worst, wname = 0.0, None
    for k, p in model.named_parameters():
        r = ref_p[k]
        if r is None or r.norm() == 0:
            assert p.grad is None or p.grad.abs().max().item() < 1e-7, (label, k)
            continue
        e = rel_l2(p.grad.cpu(), r)
        if e >= worst:
            worst, wname = e, k
    errs = {}
    for name, x, r in zip(INS, ins, ref_in):
        got = torch.zeros_like(x) if x.grad is None else x.grad
        if r.norm() == 0:
            assert got.abs().max().item() < 1e-7, (label, name)
            errs[name] = 0.0
            continue
        errs[name] = row_err(got.reshape(na * nb, -1), r.reshape(na * nb, -1))[0]
    return worst, wname, errs


def _d_out(ocfg, na, nb, seed, only=None, row=None):
    g = torch.Generator().manual_seed(seed)
    shapes = [(na, nb, len(ocfg.actions)), (na, nb), (na, nb, ocfg.nb_class), (na, nb, ocfg.n_m),
              (na, nb, ocfg.n_b), (na, nb, ocfg.n_b), (na, nb, ocfg.n_a), (na, nb, ocfg.n_a)]
    d = [torch.randn(*s, generator=g) for s in shapes]
    if only is not None:
        d = [x if i == only else None for i, x in enumerate(d)]
    if row is not None:
        mask = torch.zeros(na * nb)
        mask[row] = 1.0
        d = [None if x is None else x * mask.view(na, nb, *([1] * (x.dim() - 2))) for x in d]
    return d


@pytest.mark.gpu
@pytest.mark.parametrize("key,mode", MODES)
def test_step_grad_vs_fp64(key, mode):
    mc, na, nb = STEPS[key]
    ocfg = oracle_config(mc)
    params = O.init_params(ocfg, seed=7)
    model, _, _ = _model(mc, na, mode, params)
    patch, msg, npos, hid = _inputs(ocfg, na, nb, seed=na * nb)
    d_out = _d_out(ocfg, na, nb, seed=1)
    ref_p, ref_in = _oracle(params, ocfg, patch, msg, npos, hid, d_out)
    ins = _engine_step(model, patch, msg, npos, hid, d_out)
    worst, wname, errs = _compare(model, ins, ref_p, ref_in, na, nb, key)
    print(f"\nstep {key} {mode}: worst parameter {worst:.1e} [{wname}], inputs per row "
          + ", ".join(f"{k} {v:.1e}" for k, v in errs.items()))
    assert worst < BOUND[mode]["param"], (wname, worst)
    bad = {k: v for k, v in errs.items() if not v < BOUND[mode]["input"]}
    assert not bad, bad


@pytest.mark.gpu
@pytest.mark.parametrize("key,mode", [("conftest_odd", "tf32x3"), ("259", "tf32x3"), ("4098", "tf32x3"),
                                      ("93", "unfused")])
def test_isolation_probes(key, mode):
    """One output at a time (a seed or an emitted input gradient that is not wired shows up alone), then one row.
    Chained sweep (conftest_odd, 259), unfused sweep from 4096 rows (4098) and the one-kernel-per-op path
    (use_chains = False): each wires the seeds and the emitted input gradients its own way."""
    mc, na, nb = STEPS[key]
    ocfg = oracle_config(mc)
    params = O.init_params(ocfg, seed=7)
    model, _, _ = _model(mc, na, mode, params)
    patch, msg, npos, hid = _inputs(ocfg, na, nb, seed=3)
    probes = {OUTS[k]: dict(only=k) for k in range(8)}
    probes["row"] = dict(row=(na * nb) // 2 + 1)
    worst = {}
    for name, kw in probes.items():
        d_out = _d_out(ocfg, na, nb, seed=11, **kw)
        ref_p, ref_in = _oracle(params, ocfg, patch, msg, npos, hid, d_out)
        ins = _engine_step(model, patch, msg, npos, hid, d_out)
        wp, wname, errs = _compare(model, ins, ref_p, ref_in, na, nb, f"{key}/{name}")
        worst[name] = max([wp, *errs.values()])
    print(f"\nprobes {key} {mode}: " + ", ".join(f"{k} {v:.1e}" for k, v in worst.items()))
    bad = {k: v for k, v in worst.items() if not v < PROBE_BOUND}
    assert not bad, bad


def _stepwise_episode(fx, model, marl, env, hidden_scale=1.0):
    """test_stepwise_api_matches_fused_episode's loop (episode.py:70-78) with grad on: stacked outputs."""
    import torch as th

    img = fx["img"].to(DEV)
    draws = {"randint": [fx["pos0"][..., 0].to(DEV), fx["pos0"][..., 1].to(DEV)],
             "randn": [h.to(DEV) * hidden_scale for h in fx["hidden0"]],
             "multinomial": [a.reshape(-1, 1).to(DEV) for a in fx["actions"]]}
    orig = (th.randint, th.randn, th.multinomial)
    th.randint = lambda *a, **k: draws["randint"].pop(0)
    th.randn = lambda *a, **k: draws["randn"].pop(0)
    th.multinomial = lambda *a, **k: draws["multinomial"].pop(0)
    try:
        obs = env.reset(img, fx["na"])
        marl.reset(fx["nb"])
        preds, logps, vals = [], [], []
        for _ in range(fx["T"]):
            out = marl.act(obs, env.normalized_positions)
            obs = env.step(out.actions)
            preds.append(out.predictions)
            logps.append(out.actions_log_probs)
            vals.append(out.values)
    finally:
        th.randint, th.randn, th.multinomial = orig
    return torch.stack(preds), torch.stack(logps), torch.stack(vals)


def _fixture_model(fx, use_tc):
    from marlclassification_b200.config import ModelConfig

    model, marl, env = ModelConfig(**fx["model_config"]).build_marl(fx["na"])
    model.use_tc = use_tc
    model.load_state_dict(fx["state_dict"])
    model.to(DEV)
    model.differentiable_steps = True
    return model, marl, env


def _episode_grads(fx, model, marl, env, hidden_scale=1.0):
    preds, logps, vals = _stepwise_episode(fx, model, marl, env, hidden_scale)
    O.a2c_loss(preds, logps, vals, fx["targets"].to(DEV), fx["gamma"]).loss.backward()
    torch.cuda.synchronize()
    return {k: p.grad.detach().clone() for k, p in model.named_parameters()}


@pytest.mark.gpu
@pytest.mark.parametrize("use_tc", [True, False], ids=["tf32x3", "fp32"])
@pytest.mark.parametrize("name", GOLDEN_NAMES)
def test_stepwise_episode_matches_reference(name, use_tc):
    from marlclassification_b200.core import EpisodeSampler

    fx = load_golden(name)
    model, marl, env = _fixture_model(fx, use_tc)
    model.zero_grad(set_to_none=True)
    grads = _episode_grads(fx, model, marl, env)
    worst = 0.0
    for k, g in grads.items():
        ref = fx["grads"][k]
        if ref.norm() == 0:
            assert g.abs().max().item() < 1e-7, k
            continue
        err = rel_l2(g.cpu(), ref)
        worst = max(worst, err)
        assert err < TOL, (k, err)
    # the same loss through the fused episode (run_episode: one autograd node with the episode's BPTT)
    sampler = EpisodeSampler(marl, env, fx["T"], gamma=fx["gamma"])
    inject = dict(pos0=fx["pos0"].to(DEV), hidden0=[h.to(DEV) for h in fx["hidden0"]], actions=fx["actions"].to(DEV))
    model.zero_grad(set_to_none=True)
    out = sampler.run_episode(fx["img"].to(DEV), **inject)
    O.a2c_loss(out.step_preds, out.step_log_probas, out.step_values, fx["targets"].to(DEV), fx["gamma"]).loss.backward()
    fused_worst = 0.0
    for k, p in model.named_parameters():
        if grads[k].norm() > 0:
            fused_worst = max(fused_worst, rel_l2(grads[k].cpu(), p.grad.cpu()))
    print(f"\n{name} {'tf32x3' if use_tc else 'fp32'}: worst vs reference {worst:.1e}, vs run_episode {fused_worst:.1e}")
    assert fused_worst < RUN_EPISODE_BOUND


@pytest.mark.gpu
def test_accumulation_and_bucket():
    fx = load_golden("resisc_small")
    model, marl, env = _fixture_model(fx, True)
    model.zero_grad(set_to_none=True)
    g1 = _episode_grads(fx, model, marl, env)
    model.zero_grad(set_to_none=True)
    g2 = _episode_grads(fx, model, marl, env, hidden_scale=0.5)
    # both graphs built first: the second episode overwrites the step engine's workspace before either backward
    model.zero_grad(set_to_none=True)
    losses = []
    for scale in (1.0, 0.5):
        preds, logps, vals = _stepwise_episode(fx, model, marl, env, scale)
        losses.append(O.a2c_loss(preds, logps, vals, fx["targets"].to(DEV), fx["gamma"]).loss)
    for loss in losses:
        loss.backward()
    torch.cuda.synchronize()
    flat = model.flat_grads
    lo, hi = flat.data_ptr(), flat.data_ptr() + 4 * flat.numel()
    for k, p in model.named_parameters():
        want = g1[k] + g2[k]
        assert rel_l2(p.grad.cpu(), want.cpu()) < 1e-5, k
        # param.grad is the parameter's slot of the flat bucket the fused Adam reads
        assert lo <= p.grad.data_ptr() < hi, k
    # after zero_grad (plain, then set_to_none) the bucket restarts from zero
    for set_to_none in (False, True):
        model.zero_grad(set_to_none=set_to_none)
        got = _episode_grads(fx, model, marl, env)
        for k, p in model.named_parameters():
            assert lo <= p.grad.data_ptr() < hi, k
            assert rel_l2(got[k].cpu(), g1[k].cpu()) < 1e-5, k
        flat_view = {k: flat[(p.data.data_ptr() - model.flat_params.data_ptr()) // 4:][:p.numel()].view(p.shape)
                     for k, p in model.named_parameters()}
        for k, p in model.named_parameters():
            assert torch.equal(flat_view[k], p.grad), k
    # a run_episode backward after zero_grad(set_to_none=True) leaves param.grad outside the bucket; a step-wise
    # backward that follows moves it into the bucket and adds to it
    from marlclassification_b200.core import EpisodeSampler

    model.zero_grad(set_to_none=True)
    sampler = EpisodeSampler(marl, env, fx["T"], gamma=fx["gamma"])
    inject = dict(pos0=fx["pos0"].to(DEV), hidden0=[h.to(DEV) for h in fx["hidden0"]], actions=fx["actions"].to(DEV))
    out = sampler.run_episode(fx["img"].to(DEV), **inject)
    O.a2c_loss(out.step_preds, out.step_log_probas, out.step_values, fx["targets"].to(DEV), fx["gamma"]).loss.backward()
    g_ep = {k: p.grad.detach().clone() for k, p in model.named_parameters()}
    got = _episode_grads(fx, model, marl, env)
    for k, p in model.named_parameters():
        assert lo <= p.grad.data_ptr() < hi, k
        assert rel_l2(got[k].cpu(), (g_ep[k] + g1[k]).cpu()) < 1e-5, k


def _one_step(model, fx, requires=()):
    from marlclassification_b200.networks.models import RecurrentOutput

    na, nb = fx["na"], fx["nb"]
    ocfg = oracle_config(fx["model_config"])
    patch, msg, npos, hid = _inputs(ocfg, na, nb, seed=5)
    patch, npos = patch.to(DEV), npos.to(DEV)
    if "img_patch" in requires:
        patch.requires_grad_(True)
    if "norm_pos" in requires:
        npos.requires_grad_(True)
    return model(patch, msg.to(DEV), npos, RecurrentOutput(*[h.to(DEV) for h in hid]))


@pytest.mark.gpu
def test_guards():
    from marlclassification_b200.training.optim import FlatAdam

    fx = load_golden("conftest_odd")
    model, _, _ = _fixture_model(fx, True)
    # an in-place parameter update between forward and backward
    out, rec = _one_step(model, fx)
    with torch.no_grad():
        next(model.parameters()).add_(1e-3)
    with pytest.raises(RuntimeError, match="parameter was updated"):
        (out.predictions.sum() + rec.h.sum()).backward()
    # the fused Adam writes through a raw pointer
    out, rec = _one_step(model, fx)
    FlatAdam(model, 1e-3).step()
    with pytest.raises(RuntimeError, match="parameter was updated"):
        out.values.sum().backward()
    # an in-place torch write to the flat buffer every parameter views
    out, rec = _one_step(model, fx)
    with torch.no_grad():
        model.flat_params.mul_(1.0)
    with pytest.raises(RuntimeError, match="parameter was updated"):
        out.values.sum().backward()
    # inputs that get no gradient
    for name in ("img_patch", "norm_pos"):
        with pytest.raises(RuntimeError, match=name):
            _one_step(model, fx, requires=(name,))
    # under no_grad the switch changes nothing
    with torch.no_grad():
        on = _one_step(model, fx)
        model.differentiable_steps = False
        off = _one_step(model, fx)
    flat = lambda r: [r[0].actions_probabilities, r[0].values, r[0].predictions, r[0].messages,  # noqa: E731
                      r[1].h, r[1].c, r[1].h_caret, r[1].c_caret]
    for a, b in zip(flat(on), flat(off)):
        assert a.grad_fn is None and torch.equal(a, b)


@pytest.mark.gpu
def test_guard_sees_graphed_train_step():
    """Trainer.train_step replays its fused Adam from a CUDA graph, without calling FlatAdam.step(): a step-wise
    backward across such a replay must refuse as well."""
    from marlclassification_b200.core import EpisodeSampler
    from marlclassification_b200.training import Trainer

    fx = load_golden("resisc_small")
    model, marl, env = _fixture_model(fx, True)
    trainer = Trainer(model, fx["model_config"]["nb_class"], 1e-3, fx["gamma"])
    sampler = EpisodeSampler(marl, env, fx["T"], gamma=fx["gamma"])
    img, y = fx["img"].to(DEV), fx["targets"].to(DEV)
    for _ in range(3):  # two eager iterations, then the iteration is captured (and replayed)
        trainer.train_step(img, y, sampler)
    out, rec = _one_step(model, fx)
    trainer.train_step(img, y, sampler)  # replay only
    torch.cuda.synchronize()
    with pytest.raises(RuntimeError, match="parameter was updated"):
        out.values.sum().backward()


# Kernel launches of one eager iteration of the fused episode, forward and backward, as the parent of this
# feature launched them: the step-wise backward reuses the episode's sweep, which must launch exactly as before.
# Recorded on a B200 by running the body of this test at commit f9ad6b8 (the parent, before the step-wise backward)
# and again with the step-wise backward in place: both printed these counts.  Re-check with
# `pytest -m gpu -s tests/test_gpu_stepwise_grad.py -k launch_counts` (the body needs nothing newer than f9ad6b8).
LAUNCHES = {"c2_resisc45": (74, 80), "c4_shard256": (74, 250)}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(LAUNCHES))
def test_fused_episode_launch_counts(name):
    from marlclassification_b200.config import ModelConfig
    from marlclassification_b200.core import EpisodeSampler

    spec = CONFIGS[name]
    ocfg = oracle_config(spec["mc"])
    model, marl, env = ModelConfig(**spec["mc"]).build_marl(spec["na"])
    model.load_state_dict(O.init_params(ocfg, seed=7))
    model.to(DEV)
    g = torch.Generator().manual_seed(0)
    img = torch.rand(spec["nb"], spec["C"], spec["H"], spec["W"], generator=g).to(DEV)
    y = torch.randint(ocfg.nb_class, (spec["nb"],), generator=g).to(DEV)
    eng = EpisodeSampler(marl, env, spec["T"], gamma=0.99).engine_for(img)
    eng.forward(img)
    eng.loss(y)
    eng.backward(img)
    torch.cuda.synchronize()
    got = (eng.launches["forward"], eng.launches["backward"])
    print(f"\n{name}: launches forward / backward {got}")
    assert got == LAUNCHES[name]

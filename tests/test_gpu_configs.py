"""Every BASELINE.json configuration through the DEFAULT product path -- tf32x3 tensor-core mode,
fused chains, the whole iteration replayed as a CUDA graph -- against the live CPU oracle on
identical injected draws (SURVEY 8c/8d; VERDICT r1 items 2 and 3).

Bars (north_star): positions bit-exact; logits / log-probs / values / loss and every per-parameter
gradient within 1e-3 norm-wise.  Also here: EvalStep's vote (trainer.py:164-196) against the
reference's recorded outputs, and the device-side ConfusionMeter against vectors of the reference's
own meter (metrics.py:25-108, tests/test_metrics.py:6-37).
"""
import os

import pytest
import torch

from oracle import marl_oracle as O
from tests.conftest import GOLDEN_DIR, load_golden, rel_l2
from tests.nets import C2_NET, MOVES1, MOVES3  # noqa: F401  (re-exported to the other GPU test modules)
from tests.nets import model_config as _mc
from tests.nets import oracle_case as _oracle_case

pytestmark = pytest.mark.gpu

TOL = 1e-3
DEV = "cuda"

CONFIGS = {
    # BASELINE.json configs 1-3 (README.md:39-43 hyper-parameters)
    "c1_mnist": dict(mc=_mc("mnist", 6, 64, 16, 24, 8, 96, 96, 10, MOVES1), na=3, nb=32, T=5, C=3, H=28, W=28),
    "c2_resisc45": dict(mc=C2_NET, na=16, nb=8, T=16, C=3, H=256, W=256),
    "c3_aid": dict(mc=_mc("aid", 24, 256, 64, 96, 16, 320, 320, 30, MOVES3), na=16, nb=8, T=16, C=3, H=600, W=600),
    # config 4: RESISC45 net, global batch 256 -> per-GPU shards of 256 (1 GPU, M=4096 rows) and 32 (8 GPUs, M=512)
    "c4_shard32": dict(mc=C2_NET, na=16, nb=32, T=16, C=3, H=256, W=256),
    "c4_shard256": dict(mc=C2_NET, na=16, nb=256, T=16, C=3, H=256, W=256),
    # the wide feature extractor (>= 256 windows per step) on the other CNN shapes: MNIST (1 input channel out of 3,
    # f = 6, 2 layers) takes it; AID (392 KB of conv weights: not eligible) must fall back to one CTA per window
    "c1_mnist_b128": dict(mc=_mc("mnist", 6, 64, 16, 24, 8, 96, 96, 10, MOVES1), na=3, nb=128, T=5, C=3, H=28, W=28),
    "c3_aid_b16": dict(mc=_mc("aid", 24, 256, 64, 96, 16, 320, 320, 30, MOVES3), na=16, nb=16, T=4, C=3, H=200, W=200),
    # config 5: agent sweep, 32 steps
    "c5_na32": dict(mc=C2_NET, na=32, nb=8, T=32, C=3, H=256, W=256),
    "c5_na256": dict(mc=C2_NET, na=256, nb=8, T=32, C=3, H=256, W=256),
    # the reference's shipped trained shape sets (resources/trained_models/{resisc45,aid}/marl.json): 5 actions
    # incl. stay; resisc45 has hidden_size_linear_action = 758 (row stride not a multiple of 16 bytes)
    "shipped_resisc45": dict(mc=_mc("resisc45", 12, 512, 64, 96, 16, 768, 758, 45, MOVES1 + [[0, 0]]),
                             na=16, nb=8, T=16, C=3, H=256, W=256),
    "shipped_aid": dict(mc=_mc("aid", 24, 768, 128, 192, 16, 1024, 1024, 30, MOVES3 + [[0, 0]]),
                        na=16, nb=8, T=16, C=3, H=600, W=600),
}


def _graphed_iteration(eng, img, y, pos0, hidden0, actions):
    """rollout -> loss -> BPTT captured in ONE CUDA graph (static injected draws) and replayed."""
    def body():
        eng.forward(img, pos0, hidden0, actions)
        eng.loss(y)
        eng.backward(img)

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        body()
        body()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        body()
    # poison what the replay must rewrite, then replay twice (replays are idempotent under injection)
    eng.step_preds.fill_(float("nan"))
    eng.model.flat_grads.fill_(float("nan"))
    graph.replay()
    graph.replay()
    torch.cuda.synchronize()


@pytest.mark.parametrize("name", list(CONFIGS))
def test_default_graph_path_vs_oracle(name):
    from marlclassification_b200.config import ModelConfig
    from marlclassification_b200.core import EpisodeSampler

    spec = CONFIGS[name]
    ocfg, params, img, y, pos0, hidden0, actions = _oracle_case(spec)
    ro, parts, grads = O.loss_and_grads(params, ocfg, img, y, pos0, hidden0, actions, spec["T"], 0.99)

    model, marl, env = ModelConfig(**spec["mc"]).build_marl(spec["na"])
    model.load_state_dict(params)
    model.to(DEV)
    assert model.use_tc and model.precision == "tf32x3" and model.use_chains  # the defaults bench.py times
    sampler = EpisodeSampler(marl, env, spec["T"], gamma=0.99)
    imgd, yd = img.to(DEV), y.to(DEV)
    eng = sampler.engine_for(imgd)
    from marlclassification_b200 import _lib

    ffma0, tc0 = _lib.lib().marlc_gemm_launch_count(1), _lib.lib().marlc_gemm_launch_count(0)
    _graphed_iteration(eng, imgd, yd, pos0.to(DEV), [h.to(DEV) for h in hidden0], actions.to(DEV))
    ffma = (_lib.lib().marlc_gemm_launch_count(1) - ffma0) // 3  # 2 eager passes + 1 capture issue the launches
    tc = (_lib.lib().marlc_gemm_launch_count(0) - tc0) // 3
    # WHICH GEMM back end ran: the tensor cores carry the iteration; the exact-fp32 FFMA kernel is left with the
    # products whose operands TMA cannot address (row pitch not a multiple of 16 bytes).  README-shaped nets: only the
    # prediction head's final-layer weight gradient (pitch nb_class = 45 / 30 / 10).  The shipped RESISC45 shape set
    # (hidden_size_linear_action = 758): additionally, ON PURPOSE, the input / weight gradients of policy.0 and
    # critic.0 and the first conv layer... every other product of that model stays on the tensor cores.
    print(f"{name}: GEMM launches per iteration: tcgen05 {tc}, FFMA {ffma}")
    assert tc >= 3 * spec["T"], (tc, ffma)
    if name == "shipped_resisc45":
        assert 4 <= ffma <= 12, ffma
    else:
        assert ffma <= 3, ffma

    assert torch.equal(eng.step_pos.cpu(), ro.step_pos)  # bit-exact
    e_fwd = [rel_l2(eng.step_preds.cpu(), ro.step_preds), rel_l2(eng.step_log_probas.cpu(), ro.step_log_probas),
             rel_l2(eng.step_values.cpu(), ro.step_values)]
    loss = eng.loss_out.cpu()
    e_loss = abs(loss[0].item() - parts.loss.item()) / abs(parts.loss.item())
    model.attach_grads()
    ours = {k: p.grad.cpu() for k, p in model.named_parameters()}
    e_grad = {}
    for k in ours:
        if grads[k].norm() == 0:
            continue
        if grads[k].numel() == 1:
            # a one-element gradient (critic.3.bias = sum of d loss / d V over all T*M rows) is a single heavily
            # cancelling sum: at shipped_resisc45 |sum| = 0.14 against sum|terms| = 16, so the 1.4e-5 forward
            # error of V shows up 100x larger in it (the fp32 oracle itself is 6e-6 off its fp64 twin there).
            # Norm-wise parity for it is measured over the Linear it belongs to: [weight, bias] jointly.
            wk = k.replace(".bias", ".weight")
            e_grad[k] = rel_l2(torch.cat([ours[wk].flatten(), ours[k].flatten()]),
                               torch.cat([grads[wk].flatten(), grads[k].flatten()]))
        else:
            e_grad[k] = rel_l2(ours[k], grads[k])
    worst = max(e_grad, key=e_grad.get)
    print(f"{name}: preds/logp/values {e_fwd[0]:.1e}/{e_fwd[1]:.1e}/{e_fwd[2]:.1e}  loss {e_loss:.1e}  "
          f"worst grad {e_grad[worst]:.1e} ({worst.split('__')[-1]})")
    assert max(e_fwd) < TOL and e_loss < TOL
    assert e_grad[worst] < TOL, (worst, e_grad[worst])


# ---- a21 / f4: EvalStep (trainer.py:164-196) ---------------------------------------------------------
@pytest.mark.parametrize("name", ["mnist_ckpt", "resisc_small", "aid_small"])
def test_eval_step_vote_matches_reference(name):
    """The forward-only graph path: vote = mean over agents of the last step's predictions
    (trainer.py:180), against the outputs recorded from the reference on the same draws."""
    from marlclassification_b200.training import Trainer
    from tests.test_gpu_parity import run_fixture

    fx = load_golden(name)
    model, marl, env, sampler, inject = run_fixture(fx, use_tc=True)
    trainer = Trainer(model, fx["model_config"]["nb_class"], 1e-4, fx["gamma"])
    ref_vote = fx["step_preds"][-1].mean(dim=0)
    img = fx["img"].to(DEV)
    for i in range(5):  # 2 eager calls, capture, 2 replays
        vote = trainer.eval_step(img, sampler, **inject).clone()
        torch.cuda.synchronize()
        assert rel_l2(vote.cpu(), ref_vote) < TOL, i
        assert torch.equal(vote.argmax(dim=1).cpu(), ref_vote.argmax(dim=1))
    eng = sampler.engine_for(img, gamma=fx["gamma"])
    assert torch.equal(eng.step_pos.cpu(), fx["step_pos"])
    # the un-injected graph (device draws) still works beside the injected one
    free = trainer.eval_step(img, sampler).clone()
    assert free.shape == ref_vote.shape and torch.isfinite(free).all()


def test_eval_epoch_confusion_matches_oracle_votes():
    """Trainer.eval_epoch end to end on device draws: its ConfusionMeter must equal the matrix built
    from the votes the engine actually produced (argmax of step_preds[-1].mean(0))."""
    from marlclassification_b200.training import Trainer
    from tests.test_gpu_parity import run_fixture

    fx = load_golden("mnist_ckpt")
    model, marl, env, sampler, _ = run_fixture(fx, use_tc=True)
    nc = fx["model_config"]["nb_class"]
    trainer = Trainer(model, nc, 1e-4, fx["gamma"])
    g = torch.Generator().manual_seed(3)
    nb = fx["img"].shape[0]
    batches = [(torch.rand(nb, *fx["img"].shape[1:], generator=g), torch.randint(nc, (nb,), generator=g)) for _ in range(6)]
    seen = []
    orig = trainer.eval_step

    def spy(x, s, **kw):
        v = orig(x, s, **kw)
        seen.append(v.clone())
        return v

    trainer.eval_step = spy
    meter = trainer.eval_epoch(batches, 0, sampler)
    cm_ref, prec_ref, rec_ref = O.confusion_matrix([(v.cpu(), y) for v, (_, y) in zip(seen, batches)], nc, None)
    assert torch.equal(meter.conf_mat().cpu(), cm_ref)
    assert torch.allclose(meter.precision().cpu(), prec_ref) and torch.allclose(meter.recall().cpu(), rec_ref)


# ---- f2: device-side ConfusionMeter / LossMeter against the reference's meter -----------------------------
def test_confusion_meter_on_device_matches_reference_vectors():
    from marlclassification_b200.metrics import ConfusionMeter, LossMeter

    fx = torch.load(os.path.join(GOLDEN_DIR, "metrics.pt"), weights_only=False)
    for case in fx["cases"]:
        meter = ConfusionMeter(case["nb_class"], case["window"])
        for i, (proba, y) in enumerate(case["batches"]):
            meter.add(proba.to(DEV), y.to(DEV))
            cm = meter.conf_mat()
            assert cm.is_cuda and cm.dtype == torch.int64
            assert torch.equal(cm.cpu(), case["conf_mat"][i].to(torch.int64)), (case["nb_class"], i)
            assert torch.allclose(meter.precision().cpu(), case["precision"][i])
            assert torch.allclose(meter.recall().cpu(), case["recall"][i])
            pr = meter.mean_precision_recall().cpu()
            assert torch.allclose(pr, torch.stack((case["precision"][i].mean(), case["recall"][i].mean())))
    one = fx["identity_one_error"]  # /root/reference/tests/test_metrics.py:6-29
    meter = ConfusionMeter(one["nb_class"], None)
    meter.add(one["y_pred"].to(DEV), torch.arange(one["nb_class"], device=DEV))
    cm = meter.conf_mat().cpu()
    assert cm[0, 0] == 0 and cm[0, 1] == 1 and (torch.diag(cm)[1:] == 1).all() and cm.sum() == one["nb_class"]
    assert torch.equal(cm, one["conf_mat"])
    lm = LossMeter(fx["loss_meter"]["window"])
    for v, m in zip(fx["loss_meter"]["values"], fx["loss_meter"]["means"]):
        lm.add(v)
        assert abs(lm.loss() - m) < 1e-12


# ---- API guards (ADVICE r1; VERDICT r1 item 8) -------------------------------------------------------------
def test_stepwise_api_backward_raises_clear_error():
    """models.py:78-138 / agent.py:40-68 are differentiable in the reference; here the step-wise API is
    forward-only and must say so when a backward reaches it (not torch's generic 'does not require grad')."""
    from marlclassification_b200.networks.models import RecurrentOutput
    from tests.test_gpu_parity import build

    fx = load_golden("conftest_odd")
    cfg, model, marl, env = build(fx, use_tc=True)
    model.load_state_dict(fx["state_dict"])
    model.to(DEV)
    hid = RecurrentOutput(*[h.to(DEV) for h in fx["hidden0"]])
    msg = model.zero_first_message(fx["na"], fx["nb"])
    npos = torch.rand(fx["na"], fx["nb"], 2, device=DEV)
    out, rec = model(fx["obs"][0].to(DEV), msg, npos, hid)
    assert out.predictions.requires_grad
    with pytest.raises(RuntimeError, match="forward-only"):
        (out.predictions.sum() + rec.h.sum()).backward()
    with torch.no_grad():  # inference usage is unaffected
        out2, _ = model(fx["obs"][0].to(DEV), msg, npos, hid)
    assert not out2.predictions.requires_grad and torch.equal(out2.predictions, out.predictions.detach())


def test_autograd_node_refuses_stale_workspace():
    """loss.backward() of an episode whose activations were overwritten by a later rollout must raise."""
    from tests.test_gpu_parity import run_fixture

    fx = load_golden("conftest_odd")
    model, marl, env, sampler, inject = run_fixture(fx, use_tc=True)
    img, y = fx["img"].to(DEV), fx["targets"].to(DEV)
    first = sampler.run_episode(img, **inject)
    with torch.no_grad():
        sampler.run_episode(img)  # e.g. an eval / visualisation episode on the same geometry
    loss = O.a2c_loss(first.step_preds, first.step_log_probas, first.step_values, y, fx["gamma"]).loss
    with pytest.raises(RuntimeError, match="overwritten by a later rollout"):
        loss.backward()
    # the supported order works and matches the reference's gradients
    for p in model.parameters():
        p.grad = None
    again = sampler.run_episode(img, **inject)
    O.a2c_loss(again.step_preds, again.step_log_probas, again.step_values, y, fx["gamma"]).loss.backward()
    for k, p in model.named_parameters():
        if fx["grads"][k].norm() > 0:
            assert rel_l2(p.grad.cpu(), fx["grads"][k]) < TOL, k


def test_out_of_range_label_is_flagged_not_read_out_of_bounds():
    """cross_entropy raises a device assert for a label >= nb_class (trainer.py:83-87); the fused loss
    reports the count in loss_out[5], returns NaN losses and never indexes out of bounds."""
    from tests.test_gpu_parity import run_fixture

    fx = load_golden("conftest_odd")
    model, marl, env, sampler, inject = run_fixture(fx, use_tc=True)
    img = fx["img"].to(DEV)
    eng = sampler.engine_for(img)
    eng.forward(img, **inject)
    good = eng.loss(fx["targets"].to(DEV)).cpu()
    assert good[5].item() == 0 and torch.isfinite(good[:5]).all()
    bad_y = fx["targets"].clone()
    bad_y[0] = fx["model_config"]["nb_class"]  # one past the end
    bad_y[1] = -3
    bad = eng.loss(bad_y.to(DEV)).cpu()
    assert bad[5].item() == 2 and torch.isnan(bad[:5]).all()


def test_engine_seed_differs_by_rank_and_geometry(monkeypatch):
    from tests.test_gpu_parity import run_fixture

    fx = load_golden("conftest_odd")
    model, marl, env, sampler, _ = run_fixture(fx, use_tc=True)
    torch.manual_seed(1234)
    img = fx["img"].to(DEV)
    eng = sampler.engine_for(img)
    s0 = eng._default_seed()
    monkeypatch.setenv("RANK", "1")
    s1 = eng._default_seed()
    eng2 = sampler.engine_for(img[:5])  # ragged last batch: another engine of the same process
    monkeypatch.setenv("RANK", "0")
    assert len({s0, s1, eng2._default_seed()}) == 3
    assert s0 == eng._default_seed()  # deterministic under torch.manual_seed

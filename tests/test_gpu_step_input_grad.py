"""Gradients on the inputs of the step-wise API: ``Environment.observe()`` carries a backward to the image batch
(``marlc_patch_gather_backward``), and with ``model.differentiable_step_inputs`` the step-wise backward gives
``img_patch`` / ``norm_pos`` their gradients (``marlc_model_step_input_grad``).  A hand-written episode loop over an
image that requires grad then fills ``img.grad``, as the reference's autograd does.

* CPU: both entry points are exported and declared; host-side argument errors.
* The gather adjoint: bit for bit against a sequential fp32 loop over the agents, against ``torch.autograd.grad``
  of the oracle's gather in fp64, deterministic, and the same from a CUDA graph.
* One step: d img_patch per window and d norm_pos per row against ``torch.autograd.grad`` of ``O.step_forward``
  in fp64 (the geometries and modes of ``test_gpu_stepwise_grad.py``), and cotangent probes on one output.
* Whole step-wise episodes of the five golden fixtures: ``img.grad`` against the fp64 oracle and against
  ``run_episode``; parameter gradients unchanged by the switch; a frozen model.
* Guards of ``marlc_model_step_input_grad`` and of the switch.
"""
import ctypes as C

import pytest
import torch

from marlclassification_b200 import _lib
from oracle import marl_oracle as O
from tests.conftest import GOLDEN_NAMES, load_golden, oracle_config, rel_l2
from tests.test_gpu_image_grad import check_zeros, cin0, covered, engine_grad, img_errors, oracle_grad
from tests.test_gpu_regimes import row_err
from tests.test_gpu_stepwise_grad import MODES, OUTS, STEPS, _d_out, _fixture_model, _inputs, _model

DEV = "cuda"

# Bounds: about 10x the worst error measured on one NVIDIA B200 (1000 W power limit), never above 1e-3.
# One step against the fp64 oracle: every geometry and mode passed at the 1e-3 ceiling on the B200; the per-mode worst
# errors were not recorded, so the bounds stay there (the probes below, on three of the same geometries, measured
# at most 2.5e-5).
BOUND = {"tf32x3": {"patch": 1e-3, "npos": 1e-3}, "fp32": {"patch": 1e-3, "npos": 1e-3},
         "unfused": {"patch": 1e-3, "npos": 1e-3}}
# measured 2.5e-5 (case 259, d norm_pos, gradient on msg' only); d img_patch at most 8.1e-6
PROBE_BOUND = 2.5e-4
# whole step-wise episodes, img.grad against the fp64 oracle: measured rel-L2 4.8e-6, per-pixel 5.4e-6 (aid_small)
EPISODE_BOUND = {"rel": 5e-5, "pix": 6e-5}
# ... and against run_episode + the same loss: measured rel-L2 4.8e-7, per-pixel 9.9e-7
RUN_EPISODE_BOUND = {"rel": 5e-6, "pix": 1e-5}
PARAM_BOUND = 1e-5  # parameter gradients of the same loop with and without the switch

# gather geometries (Na, B, C, H, W, f)
GATHER = {
    "one_agent": (1, 3, 3, 20, 20, 6),
    # 24 agents on 16 x 16: every pixel under many windows, windows on every border
    "dense": (24, 3, 3, 16, 16, 6),
    # 257 agents: two chunks of the per-tile window list, the second one ragged (1 window)
    "two_chunks": (257, 2, 1, 28, 28, 6),
    # non-square image (several pixel tiles each way), odd window
    "non_square": (5, 3, 3, 37, 70, 7),
    "grey_odd": (6, 2, 1, 13, 13, 5),
}


# ---------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------
def test_symbols_exported_and_declared():
    lib = _lib.lib()
    for name in ("marlc_patch_gather_backward", "marlc_model_step_input_grad"):
        assert hasattr(lib, name)
        assert name in _lib.exported_symbols()


def _unbound_engine():
    from marlclassification_b200.config import ModelConfig
    from marlclassification_b200.engine import build_config

    fx = load_golden("conftest_odd")
    model = ModelConfig(**fx["model_config"]).build_networks()
    f = fx["model_config"]["window_size"]
    cfg = build_config(model, na=2, nb=3, T=1, C=1, H=f + 1, W=f + 1, actions=fx["model_config"]["actions"],
                       gamma=1.0)
    h = C.c_void_p()
    _lib.check(_lib.lib().marlc_engine_create(C.byref(cfg), C.byref(h)))
    return h


def test_host_argument_errors():
    L = _lib.lib()
    dummy = C.c_void_p(256)  # never dereferenced: every call below fails its host-side checks first
    for args in ((None, dummy, dummy), (dummy, None, dummy), (dummy, dummy, None)):
        assert L.marlc_patch_gather_backward(*args, 2, 3, 1, 16, 16, 6, None) != 0
        assert b"null pointer" in L.marlc_last_error()
    assert L.marlc_patch_gather_backward(dummy, dummy, dummy, 2, 3, 1, 16, 16, 17, None) != 0
    assert b"does not fit" in L.marlc_last_error()
    assert L.marlc_model_step_input_grad(None, dummy, dummy, None) != 0
    assert b"null engine" in L.marlc_last_error()
    h = _unbound_engine()
    try:
        assert L.marlc_model_step_input_grad(h, dummy, dummy, None) != 0
        assert b"not bound" in L.marlc_last_error()
        assert L.marlc_model_step_input_grad(h, dummy, None, None) != 0
        assert b"not bound" in L.marlc_last_error()
        assert L.marlc_model_step_input_grad(h, None, None, None) != 0
        assert b"both outputs are null" in L.marlc_last_error()
    finally:
        L.marlc_engine_destroy(h)


# ---------------------------------------------------------------------------------------------------------------
# GPU: the gather adjoint
# ---------------------------------------------------------------------------------------------------------------
def _gather_case(key, seed=0):
    na, B, Cc, H, W, f = GATHER[key]
    g = torch.Generator().manual_seed(seed)
    # corners anywhere the gather accepts (0 .. S - f), the four extreme ones included
    pos = torch.stack([torch.randint(H - f + 1, (na, B), generator=g), torch.randint(W - f + 1, (na, B), generator=g)],
                      -1)
    extremes = [(0, 0), (H - f, W - f), (0, W - f), (H - f, 0)]
    for i, (y, x) in enumerate(extremes[:na]):
        pos[i, 0] = torch.tensor([y, x])
    if na > 5:
        pos[5, :] = pos[0, :]  # coincident agents
    d_obs = torch.randn(na, B, Cc, f, f, generator=g)
    return pos, d_obs, (B, Cc, H, W), f


def _sequential(pos, d_obs, shape, f):
    """The definition, in fp32 on the CPU: a zero image, then d_obs[a, b] added for a = 0 .. Na-1 in order."""
    z = torch.zeros(shape, dtype=torch.float32)
    for a in range(pos.shape[0]):
        for b in range(shape[0]):
            y, x = int(pos[a, b, 0]), int(pos[a, b, 1])
            z[b, :, y:y + f, x:x + f] += d_obs[a, b]
    return z


def _gather_backward(d_obs, pos, out, f):
    na, B = pos.shape[:2]
    _, Cc, H, W = out.shape
    _lib.check(_lib.lib().marlc_patch_gather_backward(d_obs.data_ptr(), pos.data_ptr(), out.data_ptr(), na, B, Cc, H,
                                                      W, f, _lib.stream_ptr(out.device)))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("key", list(GATHER))
def test_gather_adjoint_bit_exact(key):
    pos, d_obs, shape, f = _gather_case(key)
    want = _sequential(pos, d_obs, shape, f)
    pos_d, d_obs_d = pos.to(DEV), d_obs.to(DEV)
    out = torch.full(shape, float("nan"), device=DEV)  # every element must be written
    got = _gather_backward(d_obs_d, pos_d, out, f).cpu()
    assert torch.equal(got, want)
    # the oracle's gather, differentiated in fp64
    img = torch.rand(shape, dtype=torch.float64).requires_grad_(True)
    ref = torch.autograd.grad((O.observation(img, pos, f) * d_obs.double()).sum(), img)[0]
    assert (got.double() - ref).abs().max().item() <= 1e-5 * ref.abs().max().item()
    # through Environment.observe: reset() / step() observations carry the backward
    from marlclassification_b200.core import Environment

    env = Environment([[1, 0], [-1, 0], [0, 1], [0, -1]], f)
    x = torch.rand(shape, device=DEV).requires_grad_(True)
    orig = torch.randint
    draws = [pos_d[..., 0].contiguous(), pos_d[..., 1].contiguous()]
    torch.randint = lambda *a, **k: draws.pop(0)
    try:
        obs = env.reset(x, pos.shape[0])
    finally:
        torch.randint = orig
    assert torch.equal(env.positions.cpu(), pos)
    obs.backward(d_obs_d)
    assert torch.equal(x.grad.cpu(), want)
    with torch.no_grad():
        assert env.observe().grad_fn is None


@pytest.mark.gpu
def test_gather_adjoint_deterministic_and_graph():
    pos, d_obs, shape, f = _gather_case("dense", seed=3)
    pos, d_obs = pos.to(DEV), d_obs.to(DEV)
    a = _gather_backward(d_obs, pos, torch.empty(shape, device=DEV), f)
    b = _gather_backward(d_obs, pos, torch.empty(shape, device=DEV), f)
    torch.cuda.synchronize()
    assert torch.equal(a, b)
    out = torch.empty(shape, device=DEV)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        _gather_backward(d_obs, pos, out, f)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        _gather_backward(d_obs, pos, out, f)
    out.fill_(float("nan"))
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, a)


@pytest.mark.gpu
def test_step_observation_keeps_its_positions():
    """A step's observation is differentiated at the positions it was gathered from, not the environment's current
    ones: step() binds a new position tensor."""
    from marlclassification_b200.core import Environment

    pos, d_obs, shape, f = _gather_case("non_square", seed=5)
    torch.manual_seed(0)
    env = Environment([[1, 0], [-1, 0], [0, 1], [0, -1]], f)
    x = torch.rand(shape, device=DEV).requires_grad_(True)
    obs0 = env.reset(x, pos.shape[0])
    p0 = env.positions.clone()
    obs1 = env.step(torch.zeros(pos.shape[:2], dtype=torch.int64, device=DEV))
    p1 = env.positions.clone()
    assert not torch.equal(p0, p1)
    (obs0 * d_obs.to(DEV)).sum().backward(retain_graph=True)
    assert torch.equal(x.grad.cpu(), _sequential(p0.cpu(), d_obs, shape, f))
    x.grad = None
    (obs1 * d_obs.to(DEV)).sum().backward()
    assert torch.equal(x.grad.cpu(), _sequential(p1.cpu(), d_obs, shape, f))


# ---------------------------------------------------------------------------------------------------------------
# GPU: one step
# ---------------------------------------------------------------------------------------------------------------
def _oracle_inputs(params, ocfg, patch, msg, npos, hid, d_out):
    """fp64 gradients of sum_k <out_k, d_out_k> w.r.t. img_patch and norm_pos."""
    p64 = {k: v.double() for k, v in params.items()}
    x, q = patch.double().requires_grad_(True), npos.double().requires_grad_(True)
    probs, values, preds, new_msg, new_hid = O.step_forward(p64, ocfg, x, msg.double(), q,
                                                            tuple(h.double() for h in hid))
    outs = (probs, values, preds, new_msg, *new_hid)
    total = sum((o * g.double()).sum() for o, g in zip(outs, d_out) if g is not None)
    return torch.autograd.grad(total, [x, q])


def _engine_inputs(model, patch, msg, npos, hid, d_out):
    from marlclassification_b200.networks.models import RecurrentOutput

    x, q = patch.to(DEV).requires_grad_(True), npos.to(DEV).requires_grad_(True)
    model.zero_grad(set_to_none=True)
    out, rec = model(x, msg.to(DEV), q, RecurrentOutput(*[h.to(DEV) for h in hid]))
    outs = (out.actions_probabilities, out.values, out.predictions, out.messages, rec.h, rec.c, rec.h_caret,
            rec.c_caret)
    pairs = [(o, g.to(DEV)) for o, g in zip(outs, d_out) if g is not None]
    torch.autograd.backward([o for o, _ in pairs], [g for _, g in pairs])
    torch.cuda.synchronize()
    return x.grad, q.grad


def _input_errors(got, ref, na, nb, cin):
    d_patch, d_npos = got
    assert torch.count_nonzero(d_patch[:, :, cin:]) == 0, "channels the network does not read must be zero"
    return (row_err(d_patch.reshape(na * nb, -1), ref[0].reshape(na * nb, -1))[0],
            row_err(d_npos.reshape(na * nb, -1), ref[1].reshape(na * nb, -1))[0])


@pytest.mark.gpu
@pytest.mark.parametrize("key,mode", MODES)
def test_step_input_grad_vs_fp64(key, mode):
    mc, na, nb = STEPS[key]
    ocfg = oracle_config(mc)
    params = O.init_params(ocfg, seed=7)
    model, _, _ = _model(mc, na, mode, params)
    model.differentiable_step_inputs = True
    patch, msg, npos, hid = _inputs(ocfg, na, nb, seed=na * nb)  # 3-channel windows: MnistCnn reads channel 0
    d_out = _d_out(ocfg, na, nb, seed=1)
    ref = _oracle_inputs(params, ocfg, patch, msg, npos, hid, d_out)
    got = _engine_inputs(model, patch, msg, npos, hid, d_out)
    e_patch, e_npos = _input_errors(got, ref, na, nb, cin0(model))
    print(f"\nstep {key} {mode}: d img_patch per window {e_patch:.1e}, d norm_pos per row {e_npos:.1e}")
    assert e_patch < BOUND[mode]["patch"] and e_npos < BOUND[mode]["npos"], (e_patch, e_npos)


@pytest.mark.gpu
@pytest.mark.parametrize("key,mode", [("conftest_odd", "tf32x3"), ("259", "tf32x3"), ("93", "unfused")])
def test_step_input_grad_probes(key, mode):
    """The gradient on one output only: a path from that output to the windows or the positions that is not wired
    shows up alone."""
    mc, na, nb = STEPS[key]
    ocfg = oracle_config(mc)
    params = O.init_params(ocfg, seed=7)
    model, _, _ = _model(mc, na, mode, params)
    model.differentiable_step_inputs = True
    patch, msg, npos, hid = _inputs(ocfg, na, nb, seed=3)
    worst = {}
    for k in (2, 1, 0, 3, 4):  # preds, values, probs, msg', h'
        d_out = _d_out(ocfg, na, nb, seed=11, only=k)
        ref = _oracle_inputs(params, ocfg, patch, msg, npos, hid, d_out)
        got = _engine_inputs(model, patch, msg, npos, hid, d_out)
        worst[OUTS[k]] = _input_errors(got, ref, na, nb, cin0(model))
    print(f"\nprobes {key} {mode}: " + ", ".join(f"{k} {p:.1e}/{q:.1e}" for k, (p, q) in worst.items()))
    bad = {k: v for k, v in worst.items() if not max(v) < PROBE_BOUND}
    assert not bad, bad


# ---------------------------------------------------------------------------------------------------------------
# GPU: whole step-wise episodes to the image
# ---------------------------------------------------------------------------------------------------------------
def _stepwise_loop(fx, marl, env, img):
    """The reference's episode loop (episode.py:70-78) written out, with the fixture's draws injected."""
    draws = {"randint": [fx["pos0"][..., 0].to(DEV), fx["pos0"][..., 1].to(DEV)],
             "randn": [h.to(DEV) for h in fx["hidden0"]],
             "multinomial": [a.reshape(-1, 1).to(DEV) for a in fx["actions"]]}
    orig = (torch.randint, torch.randn, torch.multinomial)
    torch.randint = lambda *a, **k: draws["randint"].pop(0)
    torch.randn = lambda *a, **k: draws["randn"].pop(0)
    torch.multinomial = lambda *a, **k: draws["multinomial"].pop(0)
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
        torch.randint, torch.randn, torch.multinomial = orig
    loss = O.a2c_loss(torch.stack(preds), torch.stack(logps), torch.stack(vals), fx["targets"].to(DEV), fx["gamma"])
    loss.loss.backward()
    torch.cuda.synchronize()


def _fixture_dict(fx):
    return dict(mc=fx["model_config"], ocfg=oracle_config(fx["model_config"]), params=fx["state_dict"],
                img=fx["img"], y=fx["targets"], pos0=fx["pos0"], hidden0=fx["hidden0"], actions=fx["actions"],
                T=fx["T"], gamma=fx["gamma"], na=fx["na"])


@pytest.mark.gpu
@pytest.mark.parametrize("name", GOLDEN_NAMES)
def test_stepwise_episode_image_grad(name):
    from marlclassification_b200.core import EpisodeSampler

    fx = load_golden(name)
    d = _fixture_dict(fx)
    model, marl, env = _fixture_model(fx, True)
    # parameter gradients of the loop without input gradients
    model.zero_grad(set_to_none=True)
    _stepwise_loop(fx, marl, env, fx["img"].to(DEV))
    plain = {k: p.grad.detach().clone() for k, p in model.named_parameters()}
    # the same loop over an image that requires grad
    model.differentiable_step_inputs = True
    model.zero_grad(set_to_none=True)
    x = fx["img"].to(DEV).requires_grad_(True)
    _stepwise_loop(fx, marl, env, x)
    for k, p in model.named_parameters():
        if plain[k].norm() == 0:
            assert p.grad.abs().max().item() < 1e-7, k
            continue
        assert rel_l2(p.grad.cpu(), plain[k].cpu()) <= PARAM_BOUND, k
    ref, ro = oracle_grad(d)
    rel, pix = img_errors(x.grad, ref)
    check_zeros(x.grad, covered(fx["pos0"], ro.step_pos, fx["T"], d["ocfg"].f, fx["img"].shape), cin0(model))
    # run_episode on the same draws
    fused, _, _ = engine_grad(d, model=model, sampler=EpisodeSampler(marl, env, fx["T"], gamma=fx["gamma"]))
    rel_f, pix_f = img_errors(x.grad, fused)
    print(f"\n{name}: step-wise img.grad vs fp64 rel-L2 {rel:.1e}, per-pixel {pix:.1e}; vs run_episode rel-L2 "
          f"{rel_f:.1e}, per-pixel {pix_f:.1e}")
    assert rel < EPISODE_BOUND["rel"] and pix < EPISODE_BOUND["pix"], (rel, pix)
    assert rel_f < RUN_EPISODE_BOUND["rel"] and pix_f < RUN_EPISODE_BOUND["pix"], (rel_f, pix_f)


@pytest.mark.gpu
def test_stepwise_episode_frozen_model():
    """Attribution on a frozen model through the step-wise API: img.grad is filled, every param.grad stays."""
    fx = load_golden("resisc_small")
    d = _fixture_dict(fx)
    model, marl, env = _fixture_model(fx, True)
    model.differentiable_step_inputs = True
    model.requires_grad_(False)
    model.ensure_flat()
    model.attach_grads()
    model.flat_grads.normal_()
    before = {k: p.grad.clone() for k, p in model.named_parameters()}
    flat = model.flat_grads.clone()
    x = fx["img"].to(DEV).requires_grad_(True)
    _stepwise_loop(fx, marl, env, x)
    ref, _ = oracle_grad(d)
    rel, pix = img_errors(x.grad, ref)
    assert rel < EPISODE_BOUND["rel"] and pix < EPISODE_BOUND["pix"], (rel, pix)
    for k, p in model.named_parameters():
        assert torch.equal(p.grad, before[k]), k
    assert torch.equal(model.flat_grads, flat)


# ---------------------------------------------------------------------------------------------------------------
# GPU: guards
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_guards():
    from marlclassification_b200.networks.models import RecurrentOutput

    fx = load_golden("conftest_odd")
    model, marl, env = _fixture_model(fx, True)
    ocfg = oracle_config(fx["model_config"])
    na, nb = fx["na"], fx["nb"]
    patch, msg, npos, hid = _inputs(ocfg, na, nb, seed=5)
    patch, msg, npos, hid = patch.to(DEV), msg.to(DEV), npos.to(DEV), [h.to(DEV) for h in hid]

    def step(requires=True):
        x = patch.clone().requires_grad_(requires)
        out, rec = model(x, msg, npos, RecurrentOutput(*hid))
        return x, out, rec

    # the switch is off: the forward refuses inputs that require grad, and names the switch
    for name in ("img_patch", "norm_pos"):
        with pytest.raises(RuntimeError, match="differentiable_step_inputs"):
            model(patch.requires_grad_(name == "img_patch"), msg, npos.requires_grad_(name == "norm_pos"),
                  RecurrentOutput(*hid))
        patch.requires_grad_(False)
        npos.requires_grad_(False)
    # ... and so does a step-wise loop over an image that requires grad
    with pytest.raises(RuntimeError, match="differentiable_step_inputs"):
        _stepwise_loop(fx, marl, env, fx["img"].to(DEV).requires_grad_(True))
    model.differentiable_step_inputs = True
    with torch.no_grad():
        step(requires=False)
    eng = next(e for e in model._engines.values() if e.T == 1)
    d_patch, d_npos = torch.empty_like(patch), torch.empty_like(npos)
    with pytest.raises(RuntimeError, match="model_step_input_grad"):
        eng.step_input_grad(d_patch, d_npos)  # a model step, no step backward
    x, out, rec = step()
    out.predictions.sum().backward()
    eng.step_input_grad(d_patch, None)
    assert torch.equal(d_patch, x.grad)
    with torch.no_grad():
        step(requires=False)
    with pytest.raises(RuntimeError, match="model_step_input_grad"):
        eng.step_input_grad(d_patch, None)  # a later model step
    x, out, rec = step()
    out.values.sum().backward()
    eng.step_input_grad(None, d_npos)
    # an episode backward on the same engine (its T = 1 geometry: (f + 1) x (f + 1) images)
    img = torch.rand(nb, patch.shape[2], ocfg.f + 1, ocfg.f + 1, device=DEV)
    eng.forward(img)
    eng.loss(fx["targets"].to(DEV))
    eng.backward(img)
    eng.image_grad()
    with pytest.raises(RuntimeError, match="model_step_input_grad"):
        eng.step_input_grad(d_patch, d_npos)
    # a step backward cut short by marlc_engine_debug_stop: its autograd backward fails, and so does a later call
    x, out, rec = step()
    try:
        eng._L.marlc_engine_debug_stop(eng._h, 2)
        with pytest.raises(RuntimeError, match="model_step_input_grad"):
            out.predictions.sum().backward()
        with pytest.raises(RuntimeError, match="model_step_input_grad"):
            eng.step_input_grad(d_patch, d_npos)
    finally:
        eng._L.marlc_engine_debug_stop(eng._h, 0)
    x, out, rec = step()
    out.predictions.sum().backward()
    eng.step_input_grad(d_patch, d_npos)
    with pytest.raises(RuntimeError, match="episode_image_grad"):
        eng.image_grad()  # cnn_dY0 now holds a step's gradients
    with pytest.raises(RuntimeError, match="step_input_grad"):
        eng.step_input_grad(torch.empty(1, device=DEV), None)

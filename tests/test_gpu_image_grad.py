"""Gradients on the image batch of an episode: ``run_episode`` with ``img.requires_grad`` (``EpisodeEngine.image_grad``,
``marlc_episode_image_grad``), held to ``torch.autograd.grad`` of the fp64 oracle with respect to the image.

* CPU: the oracle's closed-form gather (``observation``) has the same image gradient as the reference's own
  ``masked_select`` algorithm (``observation_masked``), so the oracle is a valid reference for it.
* The five golden fixtures through the reference's loss; geometries of ``test_gpu_regimes.py`` and three more (an
  odd window, dense overlap on a small image, more than 4096 windows per image); the exact-fp32, unfused and
  chunked-gradient modes; cotangent probes; determinism; guards; a CUDA graph; a frozen model.

Metrics, per image b: rel-L2, and the per-pixel max |a - r| / max |r| so that one wrong pixel or tile edge is not
diluted.  Pixels outside every window the networks consumed, and channels the feature extractor does not read,
must be exactly zero.
"""
import pytest
import torch

from oracle import marl_oracle as O
from tests.conftest import GOLDEN_NAMES, load_golden, oracle_config, rel_l2
from tests.test_gpu_configs import MOVES1, _mc
from tests.test_gpu_regimes import CASES

DEV = "cuda"

# Bounds: about 10x the worst error measured on one NVIDIA B200 (1000 W power limit), never above 1e-3.
# measured, tf32x3 (fixtures, geometries, unfused, chunked, probes): rel-L2 2.3e-5, per-pixel 3.4e-5 (case 4098)
# measured, exact fp32 (use_tc=False): rel-L2 1.5e-6, per-pixel 1.7e-6
BOUND = {"rel": 2.5e-4, "pix": 4e-4}
BOUND_FP32 = {"rel": 2e-5, "pix": 2e-5}
PARAM_TOL = 1e-3  # the bar of test_gpu_parity.py against the reference's recorded parameter gradients

# geometries beyond the regime cases: (net, na, nb, T, C, H, W)
EXTRA = {
    # f = 9: the window's last row and column take the ky = 2 tap only (an even window drops ky = 0 there)
    "odd_window": (_mc("resisc45", 9, 64, 16, 24, 8, 96, 96, 45, MOVES1), 4, 6, 5, 3, 40, 40),
    # 24 agents on 16 x 16 MNIST images with f = 6: every pixel under many windows, windows on every border
    "dense": (_mc("mnist", 6, 64, 16, 24, 8, 96, 96, 10, MOVES1), 24, 3, 4, 3, 16, 16),
    # 257 agents x 16 steps = 4112 windows per image: 17 chunks of the per-tile window list, the last one ragged
    "many_windows": (_mc("mnist", 6, 64, 16, 24, 8, 96, 96, 10, MOVES1), 257, 2, 16, 1, 28, 28),
}
GEOMETRIES = {k: (CASES[k]["net"], CASES[k]["na"], CASES[k]["nb"], CASES[k]["T"], 3, CASES[k]["H"], CASES[k]["W"])
              for k in ("93", "300", "1190", "4098", "387", "261")}
GEOMETRIES.update(EXTRA)


# ---------------------------------------------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------------------------------------------
def img_errors(got, ref):
    """(worst per-image rel-L2, worst per-image max |a - r| / max |r|); an image whose reference is zero must be
    exactly zero."""
    got, ref = got.detach().double().cpu(), ref.detach().double().cpu()
    rel = pix = 0.0
    for b in range(ref.shape[0]):
        a, r = got[b], ref[b]
        top = r.abs().max().item()
        if top == 0:
            assert torch.count_nonzero(a) == 0, f"image {b}: reference is zero, engine is not"
            continue
        rel = max(rel, rel_l2(a, r))
        pix = max(pix, (a - r).abs().max().item() / top)
    return rel, pix


def covered(pos0, step_pos, T, f, shape):
    """[B, H, W] bool: pixels inside a window observed at some t < T (corners pos0, step_pos[:T-1])."""
    B, _, H, W = shape
    mask = torch.zeros(B, H, W, dtype=torch.bool)
    corners = [pos0.cpu()] + [step_pos[t].cpu() for t in range(T - 1)]
    for pos in corners:
        for a in range(pos.shape[0]):
            for b in range(B):
                y, x = int(pos[a, b, 0]), int(pos[a, b, 1])
                mask[b, y:y + f, x:x + f] = True
    return mask


def check_zeros(grad, cover, cin):
    """Exact zeros outside the union of windows and in channels >= cin."""
    g = grad.detach().cpu()
    assert torch.count_nonzero(g[:, cin:]) == 0, "channels the network does not read must be zero"
    outside = ~cover[:, None].expand(-1, g.shape[1], -1, -1)
    assert torch.count_nonzero(g[outside]) == 0, "pixels outside every window must be zero"


def inputs(mc, na, nb, T, C, H, W, seed):
    """Image, targets, corners (extreme ones included), initial state, oracle-sampled actions and fp32 params."""
    ocfg = oracle_config(mc)
    params = O.init_params(ocfg, seed=7)
    f = ocfg.f
    g = torch.Generator().manual_seed(seed)
    img = torch.rand(nb, C, H, W, generator=g)
    y = torch.randint(ocfg.nb_class, (nb,), generator=g)
    pos0 = torch.stack([torch.randint(H - f, (na, nb), generator=g), torch.randint(W - f, (na, nb), generator=g)], -1)
    pos0[0, 0] = torch.tensor([0, 0])
    pos0[-1, -1] = torch.tensor([H - f - 1, W - f - 1])
    if na > 2:
        pos0[1, :] = pos0[0, :]  # coincident agents
        pos0[2, 0] = torch.tensor([0, W - f - 1])
    hidden0 = [torch.randn(na, nb, n, generator=g) for n in (ocfg.n_b, ocfg.n_b, ocfg.n_a, ocfg.n_a)]
    actions = O.rollout(params, ocfg, img, pos0, hidden0, None, T, generator=g).actions
    return dict(mc=mc, ocfg=ocfg, params=params, img=img, y=y, pos0=pos0, hidden0=hidden0, actions=actions, T=T,
                gamma=0.99, na=na)


def oracle_grad(d, cot=None):
    """fp64 d loss / d img through the oracle rollout: the reference's loss, or sum <outputs, cot>."""
    p64 = {k: v.double() for k, v in d["params"].items()}
    x = d["img"].double().requires_grad_(True)
    ro = O.rollout(p64, d["ocfg"], x, d["pos0"], [h.double() for h in d["hidden0"]], d["actions"], d["T"])
    if cot is None:
        loss = O.a2c_loss(ro.step_preds, ro.step_log_probas, ro.step_values, d["y"], d["gamma"]).loss
    else:
        loss = sum((o * c).sum() for o, c in zip((ro.step_preds, ro.step_log_probas, ro.step_values), cot))
    return torch.autograd.grad(loss, x)[0], ro


def build(d, mode="tf32x3"):
    from marlclassification_b200.config import ModelConfig
    from marlclassification_b200.core import EpisodeSampler

    model, marl, env = ModelConfig(**d["mc"]).build_marl(d["na"])
    model.use_tc = mode != "fp32"
    model.use_chains = mode != "unfused"
    model.load_state_dict(d["params"])
    model.to(DEV)
    return model, EpisodeSampler(marl, env, d["T"], gamma=d["gamma"])


def engine_grad(d, mode="tf32x3", cot=None, model=None, sampler=None):
    """img.grad after run_episode + (reference loss | sum <outputs, cot>) + backward()."""
    if model is None:
        model, sampler = build(d, mode)
    x = d["img"].to(DEV).requires_grad_(True)
    out = sampler.run_episode(x, pos0=d["pos0"].to(DEV), hidden0=[h.to(DEV) for h in d["hidden0"]],
                              actions=d["actions"].to(DEV))
    if cot is None:
        loss = O.a2c_loss(out.step_preds, out.step_log_probas, out.step_values, d["y"].to(DEV), d["gamma"]).loss
    else:
        outs = (out.step_preds, out.step_log_probas, out.step_values)
        loss = sum((o * c.to(DEV).float()).sum() for o, c in zip(outs, cot))
    loss.backward()
    torch.cuda.synchronize()
    return x.grad, out, model


def cin0(model):
    return model.feature_extractor.cnn_spec[1][0][0]


@pytest.fixture(scope="module")
def geometry_cache():
    return {}


def geometry(key, cache):
    if key not in cache:
        mc, na, nb, T, C, H, W = GEOMETRIES[key]
        d = inputs(mc, na, nb, T, C, H, W, seed=2000 + na * nb)
        ref, ro = oracle_grad(d)
        cache.clear()  # one geometry at a time: the fp64 graphs of the large cases are big
        cache[key] = (d, ref, ro)
    return cache[key]


# ---------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------
def test_oracle_gather_adjoint_matches_reference_algorithm():
    """observation (closed form) and observation_masked (environment.py:96-126) give the same fp64 image
    gradient: random corners, windows on every border, coincident agents."""
    g = torch.Generator().manual_seed(5)
    for (na, B, C, H, W, f) in [(6, 3, 3, 20, 17, 6), (9, 2, 1, 13, 13, 5), (4, 2, 3, 28, 28, 12)]:
        pos = torch.stack([torch.randint(H - f + 1, (na, B), generator=g), torch.randint(W - f + 1, (na, B), generator=g)], -1)
        pos[0, 0] = torch.tensor([0, 0])
        pos[1, 0] = torch.tensor([H - f, W - f])
        pos[2, :] = torch.tensor([0, W - f])
        pos[3, :] = pos[2, :]  # coincident agents
        img = torch.rand(B, C, H, W, generator=g, dtype=torch.float64)
        cot = torch.randn(na, B, C, f, f, generator=g, dtype=torch.float64)
        grads = []
        for gather in (O.observation, O.observation_masked):
            x = img.clone().requires_grad_(True)
            grads.append(torch.autograd.grad((gather(x, pos, f) * cot).sum(), x)[0])
        assert torch.equal(O.observation(img, pos, f), O.observation_masked(img, pos, f))
        assert torch.allclose(grads[0], grads[1], rtol=0, atol=1e-12), (na, B, C, H, W, f)


# ---------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", GOLDEN_NAMES)
def test_fixture_image_grad(name):
    fx = load_golden(name)
    d = dict(mc=fx["model_config"], ocfg=oracle_config(fx["model_config"]), params=fx["state_dict"], img=fx["img"],
             y=fx["targets"], pos0=fx["pos0"], hidden0=fx["hidden0"], actions=fx["actions"], T=fx["T"],
             gamma=fx["gamma"], na=fx["na"])
    ref, ro = oracle_grad(d)
    got, out, model = engine_grad(d)
    rel, pix = img_errors(got, ref)
    print(f"\n{name}: image gradient rel-L2 {rel:.1e}, per-pixel {pix:.1e}")
    assert rel < BOUND["rel"] and pix < BOUND["pix"], (rel, pix)
    cover = covered(fx["pos0"], out.step_pos, fx["T"], d["ocfg"].f, fx["img"].shape)
    check_zeros(got, cover, cin0(model))
    if name == "mnist_ckpt":
        assert fx["img"].shape[1] == 3 and torch.count_nonzero(got[:, 1:]) == 0
    for k, p in model.named_parameters():
        r = fx["grads"][k]
        if r.norm() == 0:
            assert p.grad.abs().max().item() < 1e-7, k
            continue
        assert rel_l2(p.grad.cpu(), r) < PARAM_TOL, k


@pytest.mark.gpu
@pytest.mark.parametrize("key", list(GEOMETRIES))
def test_geometry_image_grad(key, geometry_cache):
    d, ref, ro = geometry(key, geometry_cache)
    got, out, model = engine_grad(d)
    assert torch.equal(out.step_pos.cpu(), ro.step_pos)
    rel, pix = img_errors(got, ref)
    print(f"\n{key}: image gradient rel-L2 {rel:.1e}, per-pixel {pix:.1e}")
    assert rel < BOUND["rel"] and pix < BOUND["pix"], (rel, pix)
    check_zeros(got, covered(d["pos0"], ro.step_pos, d["T"], d["ocfg"].f, d["img"].shape), cin0(model))


@pytest.mark.gpu
@pytest.mark.parametrize("key,mode", [("93", "fp32"), ("dense", "fp32"), ("93", "unfused"), ("odd_window", "unfused")])
def test_modes_image_grad(key, mode, geometry_cache):
    d, ref, _ = geometry(key, geometry_cache)
    got, _, _ = engine_grad(d, mode=mode)
    rel, pix = img_errors(got, ref)
    print(f"\n{key} {mode}: image gradient rel-L2 {rel:.1e}, per-pixel {pix:.1e}")
    bound = BOUND_FP32 if mode == "fp32" else BOUND
    assert rel < bound["rel"] and pix < bound["pix"], (rel, pix)


@pytest.mark.gpu
@pytest.mark.parametrize("key", ["93", "dense"])
def test_probes_image_grad(key, geometry_cache):
    """Cotangents on one image's predictions, on one step, on one row (t, a, b)."""
    d, _, _ = geometry(key, geometry_cache)
    T, na, nb = d["T"], d["na"], d["img"].shape[0]
    nc = d["ocfg"].nb_class
    g = torch.Generator().manual_seed(17)
    full = [torch.randn(T, na, nb, nc, generator=g, dtype=torch.float64),
            torch.randn(T, na, nb, generator=g, dtype=torch.float64),
            torch.randn(T, na, nb, generator=g, dtype=torch.float64)]
    model, sampler = build(d)
    worst = {}
    b1 = nb // 2
    for probe in ("image", "step", "row"):
        if probe == "image":  # predictions of image b1 only
            m = torch.zeros(T, na, nb, dtype=torch.float64)
            m[:, :, b1] = 1
            cot = [full[0] * m[..., None], torch.zeros_like(full[1]), torch.zeros_like(full[2])]
        elif probe == "step":
            m = torch.zeros(T, na, nb, dtype=torch.float64)
            m[T // 2] = 1
            cot = [full[0] * m[..., None], full[1] * m, full[2] * m]
        else:
            m = torch.zeros(T, na, nb, dtype=torch.float64)
            m[T - 1, na - 1, b1] = 1
            cot = [full[0] * m[..., None], full[1] * m, full[2] * m]
        ref, _ = oracle_grad(d, cot)
        got, _, _ = engine_grad(d, cot=cot, model=model, sampler=sampler)
        worst[probe] = img_errors(got, ref)
        if probe == "image":
            others = [b for b in range(nb) if b != b1]
            assert torch.count_nonzero(got[others]) == 0, "a cotangent on one image reached another"
    print(f"\n{key} probes: " + ", ".join(f"{p} rel-L2 {r:.1e} per-pixel {q:.1e}" for p, (r, q) in worst.items()))
    for p, (r, q) in worst.items():
        assert r < BOUND["rel"] and q < BOUND["pix"], (p, r, q)


def _engine_after_loss(d, model, sampler):
    x = d["img"].to(DEV)
    eng = sampler.engine_for(x)
    inject = (d["pos0"].to(DEV), [h.to(DEV) for h in d["hidden0"]], d["actions"].to(DEV))
    return eng, x, inject


@pytest.mark.gpu
def test_deterministic_and_graph(geometry_cache):
    """Two image_grad calls after one backward give the same bits; forward, loss, backward and image_grad captured
    in one CUDA graph and replayed give the eager result (up to the backward's unordered split-K reduce-adds)."""
    d, ref, _ = geometry("dense", geometry_cache)
    model, sampler = build(d)
    eng, x, inject = _engine_after_loss(d, model, sampler)
    y = d["y"].to(DEV)
    eng.forward(x, *inject)
    eng.loss(y)
    eng.backward(x)
    a = eng.image_grad().clone()
    b = eng.image_grad()
    torch.cuda.synchronize()
    assert torch.equal(a, b)
    # the engine's fused loss is the reference's loss
    rel, pix = img_errors(a, ref)
    assert rel < BOUND["rel"] and pix < BOUND["pix"], (rel, pix)

    out = torch.empty_like(x)

    def body():
        eng.forward(x, *inject)
        eng.loss(y)
        eng.backward(x)
        eng.image_grad(out)

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
    out.fill_(float("nan"))
    graph.replay()
    graph.replay()
    torch.cuda.synchronize()
    assert rel_l2(out, a) < 1e-5
    rel, pix = img_errors(out, ref)
    assert rel < BOUND["rel"] and pix < BOUND["pix"], (rel, pix)


@pytest.mark.gpu
def test_guards(geometry_cache):
    from marlclassification_b200.networks.models import RecurrentOutput

    d, _, _ = geometry("dense", geometry_cache)
    model, sampler = build(d)
    eng, x, inject = _engine_after_loss(d, model, sampler)
    y = d["y"].to(DEV)
    with pytest.raises(RuntimeError, match="episode_image_grad"):
        eng.image_grad()  # no backward yet
    eng.forward(x, *inject)
    eng.loss(y)
    eng.backward(x)
    eng.image_grad()
    eng.forward(x, *inject)
    with pytest.raises(RuntimeError, match="episode_image_grad"):
        eng.image_grad()  # a new rollout since the backward
    eng.loss(y)
    try:
        eng._L.marlc_engine_debug_stop(eng._h, 2)
        eng.backward(x)
        with pytest.raises(RuntimeError, match="episode_image_grad"):
            eng.image_grad()  # backward cut short after the sweep
    finally:
        eng._L.marlc_engine_debug_stop(eng._h, 0)
    eng.backward(x)
    eng.image_grad()
    # a step-wise backward on the T = 1 engine of the step-wise API
    model.differentiable_steps = True
    ocfg, na, nb = d["ocfg"], d["na"], d["img"].shape[0]
    g = torch.Generator().manual_seed(3)
    patch = torch.rand(na, nb, x.shape[1], ocfg.f, ocfg.f, generator=g).to(DEV)
    msg = torch.randn(na, nb, ocfg.n_m, generator=g).to(DEV)
    npos = torch.rand(na, nb, 2, generator=g).to(DEV)
    hid = RecurrentOutput(*[torch.randn(na, nb, n, generator=g).to(DEV)
                            for n in (ocfg.n_b, ocfg.n_b, ocfg.n_a, ocfg.n_a)])
    o, _ = model(patch, msg, npos, hid)
    o.predictions.sum().backward()
    steps = [e for e in model._engines.values() if e.T == 1]
    assert steps
    with pytest.raises(RuntimeError, match="episode_image_grad"):
        steps[0].image_grad()
    with pytest.raises(RuntimeError, match="image_grad"):
        eng.image_grad(torch.empty(1, device=DEV))


@pytest.mark.gpu
def test_frozen_model(geometry_cache):
    """Attribution on a frozen model: img.grad is filled, every param.grad stays as it was."""
    d, ref, _ = geometry("93", geometry_cache)
    model, sampler = build(d)
    model.requires_grad_(False)
    sampler.engine_for(d["img"].to(DEV))  # the engine makes every param.grad a view of model.flat_grads
    model.flat_grads.normal_()
    before = {k: p.grad.clone() for k, p in model.named_parameters()}
    flat = model.flat_grads.clone()
    got, out, _ = engine_grad(d, model=model, sampler=sampler)
    assert out.step_preds.grad_fn is not None
    rel, pix = img_errors(got, ref)
    assert rel < BOUND["rel"] and pix < BOUND["pix"], (rel, pix)
    for k, p in model.named_parameters():
        assert torch.equal(p.grad, before[k]), k
    assert torch.equal(model.flat_grads, flat)
    # run_episode_get_last_step carries the image gradient as well
    x = d["img"].to(DEV).requires_grad_(True)
    last = sampler.run_episode_get_last_step(x, pos0=d["pos0"].to(DEV), hidden0=[h.to(DEV) for h in d["hidden0"]],
                                             actions=d["actions"].to(DEV))
    last.prediction.sum().backward()
    assert x.grad is not None and torch.count_nonzero(x.grad) > 0

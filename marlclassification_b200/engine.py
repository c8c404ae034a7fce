"""Python face of the CUDA episode engine (csrc/engine.cu through the C ABI).

``EpisodeEngine`` owns one workspace for a fixed episode geometry
(na, nb, T, C, H, W) of a given ``ModelsWrapper`` and exposes

* ``forward``  -- the whole T-step rollout (episode.py:32-85),
* ``loss``     -- the fused actor-critic loss and its gradients (trainer.py:75-111),
* ``backward`` -- hand-written BPTT into the model's flat gradient buffer,
* ``image_grad`` -- the gradient that backward leaves on the image batch,

plus ``rollout_autograd`` which wraps forward/backward in ONE autograd node so
the reference's own loss code (``loss.backward()``) works unchanged.
"""
from __future__ import annotations

import ctypes as ct
from typing import Optional, Sequence

import torch as th

from . import _lib
from ._lib import MarlcConfig


def build_config(model, *, na: int, nb: int, T: int, C: int, H: int, W: int, actions, gamma: float) -> MarlcConfig:
    f, layers, groups, _first_only = model.feature_extractor.cnn_spec
    d = model.dims
    if len(actions) != d["nb_action"]:
        raise RuntimeError(f"environment has {len(actions)} actions, policy head has {d['nb_action']}")
    if len(actions) > _lib.MAX_ACTIONS or len(layers) > _lib.MAX_CNN_LAYERS:
        raise RuntimeError("too many actions / CNN layers for the engine")
    cfg = MarlcConfig()
    cfg.na, cfg.nb, cfg.T, cfg.C, cfg.H, cfg.W, cfg.f = na, nb, T, C, H, W, f
    cfg.n_actions = len(actions)
    for i, mv in enumerate(actions):
        if len(mv) != 2:
            raise RuntimeError("only 2-D moves are supported (state_dim == 2)")
        cfg.actions[i][0], cfg.actions[i][1] = int(mv[0]), int(mv[1])
    cfg.cnn_layers = len(layers)
    for i, ((ci, co), g) in enumerate(zip(layers, groups)):
        cfg.cnn_cin[i], cfg.cnn_cout[i], cfg.cnn_groups[i] = ci, co, g
    cfg.n_b, cfg.n_a, cfg.n_m, cfg.n_m_o, cfg.n_d = d["n_b"], d["n_a"], d["n_m"], d["n_m_o"], d["n_d"]
    cfg.nl_b, cfg.nl_a, cfg.nb_class = d["nl_b"], d["nl_a"], d["nb_class"]
    cfg.gamma = float(gamma)
    # GEMM arithmetic: "fp32" exact FFMA | "tf32" tcgen05 | "tf32x3" tcgen05, error-compensated
    prec = getattr(model, "precision", "tf32x3") if getattr(model, "use_tc", True) else "fp32"
    cfg.use_tc = {"fp32": 0, "tf32": 1, "tf32x3": 2}[prec]
    cfg.use_chains = 1 if getattr(model, "use_chains", True) else 0
    return cfg


class EpisodeEngine:
    """One bound engine = (model, geometry).  All device memory is allocated here,
    once; forward/loss/backward never allocate (CUDA-graph capturable)."""

    def __init__(self, model, *, na: int, nb: int, T: int, C: int, H: int, W: int, actions, gamma: float = 0.99,
                 seed: Optional[int] = None) -> None:
        model.ensure_flat()
        self.model = model
        self.device = model.device
        self.na, self.nb, self.T, self.C, self.H, self.W = na, nb, T, C, H, W
        self.actions = [list(a) for a in actions]
        self.gamma = gamma
        self.cfg = build_config(model, na=na, nb=nb, T=T, C=C, H=H, W=W, actions=actions, gamma=gamma)
        self._L = _lib.lib()
        self._h = C_void_p()
        _lib.check(self._L.marlc_engine_create(ct.byref(self.cfg), ct.byref(self._h)))
        nbytes = self._L.marlc_engine_workspace_bytes(self._h)
        with th.cuda.device(self.device):
            self.workspace = th.zeros(nbytes, dtype=th.uint8, device=self.device)
        self._params, self._grads = model.flat_params, model.flat_grads
        _lib.check(self._L.marlc_engine_bind(self._h, self.workspace.data_ptr(), self._params.data_ptr(),
                                             self._grads.data_ptr()))
        d = model.dims
        M, nc = na * nb, d["nb_class"]
        f32, i64, i32, f64 = th.float32, th.int64, th.int32, th.float64
        self.step_preds = self.view("step_preds", f32, (T, na, nb, nc))
        self.step_log_probas = self.view("step_log_probas", f32, (T, na, nb))
        self.step_values = self.view("step_values", f32, (T, na, nb))
        self.step_pos = self.view("step_pos", i64, (T, na, nb, 2))
        self.probs = self.view("probs", f32, (T, na, nb, len(actions)))
        self.actions_taken = self.view("act", i32, (T, na, nb))
        self.d_preds = self.view("d_preds", f32, (T, na, nb, nc))
        self.d_logp = self.view("d_logp", f32, (T, na, nb))
        self.d_values = self.view("d_values", f32, (T, na, nb))
        self.loss_out = self.view("loss_out", f32, (8,))
        self.loss_stats = self.view("loss_stats", f64, (16,))
        self.H_state = self.view("H", f32, (T + 1, na, nb, d["n_b"]))
        self.C_state = self.view("Cb", f32, (T + 1, na, nb, d["n_b"]))
        self.Hc_state = self.view("Hc", f32, (T + 1, na, nb, d["n_a"]))
        self.Cc_state = self.view("Cc", f32, (T + 1, na, nb, d["n_a"]))
        self.msg = self.view("msg", f32, (T + 1, na, nb, d["n_m"]))
        self.seed(seed if seed is not None else self._default_seed())
        self.launches = {"forward": 0, "loss": 0, "backward": 0}
        # bumped by every forward(): an autograd node built on one rollout refuses to run its backward
        # once another rollout has overwritten the workspace (H, C, U, probs, actions, positions)
        self.generation = 0

    def _default_seed(self) -> int:
        """torch's seed mixed with the process rank and the engine's geometry: data-parallel ranks that all
        called ``torch.manual_seed(s)`` (the usual practice) must not draw identical initial positions /
        states / action uniforms for the same local slot, and two engines of one process (main batch and
        ragged last batch) must not replay the same Philox stream."""
        import os
        import zlib

        rank = int(os.environ.get("RANK", "0"))
        geo = zlib.crc32(repr((self.na, self.nb, self.T, self.C, self.H, self.W)).encode())
        mixed = int(th.initial_seed()) ^ (rank * 0x9E3779B97F4A7C15) ^ (geo * 0xC2B2AE3D27D4EB4F)
        return mixed & 0x7FFFFFFFFFFFFFFF

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                self._L.marlc_engine_destroy(self._h)
                self._h = None
        except Exception:
            pass

    # ---- workspace views ----------------------------------------------------------
    def view(self, name: str, dtype: th.dtype, shape: Sequence[int]) -> th.Tensor:
        off, nb = ct.c_size_t(), ct.c_size_t()
        _lib.check(self._L.marlc_engine_buffer(self._h, name.encode(), ct.byref(off), ct.byref(nb)))
        n = 1
        for s in shape:
            n *= s
        item = th.empty((), dtype=dtype).element_size()
        assert n * item <= nb.value, (name, shape, nb.value)
        return self.workspace[off.value: off.value + n * item].view(dtype).view(*shape)

    def _stream(self) -> int:
        return th.cuda.current_stream(self.device).cuda_stream

    def _check_model(self) -> None:
        if self.model.flat_params.data_ptr() != self._params.data_ptr():
            raise RuntimeError("model parameters were re-allocated after the engine was built; rebuild the engine")

    def plan(self) -> dict:
        """What the launchers choose for this geometry (``marlc_plan``, include/marlc.h)."""
        plan = _lib.MarlcPlan()
        _lib.check(self._L.marlc_engine_plan(self._h, ct.byref(plan)))
        return plan.as_dict()

    def seed(self, seed: int) -> None:
        _lib.check(self._L.marlc_engine_seed(self._h, ct.c_uint64(seed), self._stream()))

    # ---- the three calls ------------------------------------------------------------
    def forward(self, img: th.Tensor, pos0: Optional[th.Tensor] = None,
                hidden0: Optional[Sequence[th.Tensor]] = None, actions: Optional[th.Tensor] = None) -> None:
        """Rollout.  ``img`` f32 [nb,C,H,W] CUDA.  Optional injection of the three
        random sites of the reference: initial positions (environment.py:33-43),
        initial recurrent state (models.py:148-159), per-step actions (agent.py:53)."""
        self._check_model()
        img = _lib.require_cuda(img, "run_episode(img_batch)", th.float32)
        if tuple(img.shape) != (self.nb, self.C, self.H, self.W):
            raise RuntimeError(f"image batch {tuple(img.shape)} != engine geometry {(self.nb, self.C, self.H, self.W)}")
        keep = [img]
        p0 = None
        if pos0 is not None:
            pos0 = _lib.require_cuda(pos0, "pos0", th.int64)
            assert tuple(pos0.shape) == (self.na, self.nb, 2)
            p0 = pos0.data_ptr()
            keep.append(pos0)
        hid = None
        if hidden0 is not None:
            hs = [_lib.require_cuda(h, "hidden0", th.float32) for h in hidden0]
            d = self.model.dims
            for h, n in zip(hs, (d["n_b"], d["n_b"], d["n_a"], d["n_a"])):
                assert tuple(h.shape) == (self.na, self.nb, n), (tuple(h.shape), n)
            hid = (ct.c_void_p * 4)(*[h.data_ptr() for h in hs])
            keep += hs
        act = None
        if actions is not None:
            actions = _lib.require_cuda(actions, "actions", th.int64)
            assert tuple(actions.shape) == (self.T, self.na, self.nb)
            act = actions.data_ptr()
            keep.append(actions)
        self._last_img = img
        self._keep = keep
        self.generation += 1
        _lib.check(self._L.marlc_episode_forward(self._h, img.data_ptr(), p0, hid, act, self._stream()))
        self.launches["forward"] = self._L.marlc_engine_last_launches(self._h)

    def loss_phase_a(self, targets: th.Tensor) -> None:
        targets = _lib.require_cuda(targets, "targets", th.int64)
        assert tuple(targets.shape) == (self.nb,)
        self._targets = targets
        _lib.check(self._L.marlc_loss_phase_a(self._h, targets.data_ptr(), self._stream()))
        self.launches["loss"] = self._L.marlc_engine_last_launches(self._h)

    def loss_phase_b(self) -> None:
        _lib.check(self._L.marlc_loss_phase_b(self._h, self._stream()))
        self.launches["loss"] += self._L.marlc_engine_last_launches(self._h)

    def loss(self, targets: th.Tensor) -> th.Tensor:
        """Fused loss + gradients w.r.t. the rollout outputs.  Returns the device
        tensor [loss, path, error, actor, critic, ...] (no host sync)."""
        self.loss_phase_a(targets)
        self.loss_phase_b()
        return self.loss_out

    def backward(self, img: Optional[th.Tensor] = None, accumulate: bool = False) -> None:
        """BPTT from d_preds / d_logp / d_values into ``model.flat_grads``."""
        self._check_model()
        img = self._last_img if img is None else _lib.require_cuda(img, "img", th.float32)
        _lib.check(self._L.marlc_episode_backward(self._h, img.data_ptr(), 1 if accumulate else 0, self._stream()))
        self.launches["backward"] = self._L.marlc_engine_last_launches(self._h)

    def image_grad(self, out: Optional[th.Tensor] = None) -> th.Tensor:
        """d(what the last ``backward`` was seeded with) / d img, f32 [nb, C, H, W] (``marlc_episode_image_grad``),
        written into ``out`` when given.  Call it after ``backward`` of the last rollout and before the parameters
        change; raises when that backward is missing."""
        shape = (self.nb, self.C, self.H, self.W)
        if out is None:
            out = th.empty(shape, dtype=th.float32, device=self.device)
        elif (tuple(out.shape) != shape or out.dtype != th.float32 or out.device != th.device(self.device)
              or not out.is_contiguous()):
            raise RuntimeError(f"image_grad(out): need a contiguous float32 {shape} tensor on {self.device}")
        _lib.check(self._L.marlc_episode_image_grad(self._h, out.data_ptr(), self._stream()))
        return out

    def model_step(self, patch, msg, npos, hidden) -> None:
        hid = (ct.c_void_p * 4)(*[h.data_ptr() for h in hidden])
        self._keep = [patch, msg, npos, *hidden]
        self.generation += 1
        _lib.check(self._L.marlc_model_step(self._h, patch.data_ptr(), msg.data_ptr(), npos.data_ptr(), hid,
                                            self._stream()))

    def model_step_backward(self, patch, msg, npos, hidden, d_out, d_in, grads) -> None:
        """``marlc_model_step_backward``: re-runs the step from its inputs, then backpropagates ``d_out``
        (8 tensors or None) into ``d_in`` (5 tensors or None) and the flat ``grads`` buffer."""
        self._check_model()
        ptrs = lambda ts: (ct.c_void_p * len(ts))(*[_lib.ptr(t) for t in ts])  # noqa: E731
        self._keep = [patch, msg, npos, *hidden, *d_out, *d_in, grads]
        self.generation += 1
        _lib.check(self._L.marlc_model_step_backward(self._h, patch.data_ptr(), msg.data_ptr(), npos.data_ptr(),
                                                     ptrs(hidden), ptrs(d_out), ptrs(d_in), grads.data_ptr(),
                                                     self._stream()))
        self.launches["backward"] = self._L.marlc_engine_last_launches(self._h)

    def step_input_grad(self, d_patch: Optional[th.Tensor], d_npos: Optional[th.Tensor]) -> None:
        """``marlc_model_step_input_grad``: the gradients the last ``model_step_backward`` leaves on its windows
        (``d_patch`` f32 [na, nb, C, f, f]) and normalised positions (``d_npos`` f32 [na, nb, 2]), each None when
        not wanted.  Call it right after ``model_step_backward`` and before the parameters change."""
        f = self.cfg.f
        for t, shape in ((d_patch, (self.na, self.nb, self.C, f, f)), (d_npos, (self.na, self.nb, 2))):
            if t is not None and (tuple(t.shape) != shape or t.dtype != th.float32 or not t.is_contiguous()
                                  or t.device != th.device(self.device)):
                raise RuntimeError(f"step_input_grad: need a contiguous float32 {shape} tensor on {self.device}")
        _lib.check(self._L.marlc_model_step_input_grad(self._h, _lib.ptr(d_patch), _lib.ptr(d_npos), self._stream()))


def C_void_p():
    return ct.c_void_p()


def engine_plan(cfg: MarlcConfig) -> dict:
    """``marlc_plan`` of an engine created for ``cfg`` and never bound: no device memory, no GPU needed."""
    L = _lib.lib()
    h = ct.c_void_p()
    _lib.check(L.marlc_engine_create(ct.byref(cfg), ct.byref(h)))
    try:
        plan = _lib.MarlcPlan()
        _lib.check(L.marlc_engine_plan(h, ct.byref(plan)))
        return plan.as_dict()
    finally:
        L.marlc_engine_destroy(h)


def get_engine(model, *, na, nb, T, C, H, W, actions, gamma=0.99) -> EpisodeEngine:
    """Engines are cached on the model per geometry (workspaces are reused across iterations)."""
    model.ensure_flat()
    key = (na, nb, T, C, H, W, tuple(tuple(a) for a in actions), float(gamma), bool(getattr(model, "use_tc", True)), getattr(model, "precision", "tf32x3"),
           bool(getattr(model, "use_chains", True)))
    eng = model._engines.get(key)
    if eng is None:
        eng = EpisodeEngine(model, na=na, nb=nb, T=T, C=C, H=H, W=W, actions=actions, gamma=gamma)
        model._engines[key] = eng
    return eng


class _RolloutFn(th.autograd.Function):
    """The whole episode as ONE autograd node: forward = fused rollout, backward =
    hand-written BPTT.  Parameter gradients are returned to autograd as clones
    of the flat-bucket views so ``loss.backward()`` accumulates them normally; the
    image gradient, when the image requires grad, comes from ``image_grad``."""

    @staticmethod
    def forward(ctx, engine: EpisodeEngine, img, pos0, hidden0, actions, *params):
        engine.forward(img, pos0, hidden0, actions)
        ctx.engine = engine
        ctx.generation = engine.generation
        ctx.img = img
        ctx.n_params = len(params)
        ctx.mark_non_differentiable(engine.step_pos)
        return engine.step_preds.clone(), engine.step_log_probas.clone(), engine.step_values.clone(), engine.step_pos.clone()

    @staticmethod
    def backward(ctx, g_preds, g_logp, g_values, _g_pos):
        eng: EpisodeEngine = ctx.engine
        if eng.generation != ctx.generation:
            raise RuntimeError(
                "run_episode(): the engine's workspace was overwritten by a later rollout of the same geometry "
                "(another run_episode / eval / visualisation call) before loss.backward() of this one; the "
                "activations BPTT needs are gone.  Call backward() before the next episode on this sampler "
                "(gradient accumulation: backward each episode in turn).")
        eng.d_preds.copy_(g_preds) if g_preds is not None else eng.d_preds.zero_()
        eng.d_logp.copy_(g_logp) if g_logp is not None else eng.d_logp.zero_()
        eng.d_values.copy_(g_values) if g_values is not None else eng.d_values.zero_()
        # BPTT into a scratch use of the flat bucket: save + restore what was there
        saved = eng.model.flat_grads.clone()
        eng.backward(ctx.img, accumulate=False)
        d_img = eng.image_grad() if ctx.needs_input_grad[1] else None
        grads = []
        for i, p in enumerate(eng.model.parameters()):
            if not ctx.needs_input_grad[5 + i]:
                grads.append(None)
                continue
            off = (p.data.data_ptr() - eng.model.flat_params.data_ptr()) // 4
            grads.append(eng.model.flat_grads[off: off + p.numel()].view(p.shape).clone())
        eng.model.flat_grads.copy_(saved)
        return (None, d_img, None, None, None, *grads)


def rollout_autograd(engine: EpisodeEngine, img, pos0=None, hidden0=None, actions=None):
    params = list(engine.model.parameters())
    return _RolloutFn.apply(engine, img, pos0, hidden0, actions, *params)


# ---- stand-alone module forwards ------------------------------------------------------
class _ForwardOnly(th.autograd.Function):
    """The step-wise API (ModelsWrapper.forward / MultiAgent.act) computes through the engine, which keeps
    no per-call autograd graph.  In grad mode its outputs are routed through this node so that a
    ``backward()`` reaching them fails with a clear message instead of silently training nothing (the
    reference's models.py:78-138 / agent.py:40-68 are differentiable; here training goes through
    ``EpisodeSampler.run_episode`` -- one autograd node with the hand-written BPTT -- or ``Trainer``)."""

    @staticmethod
    def forward(ctx, anchor, *outs):
        return tuple(o.view_as(o) for o in outs)

    @staticmethod
    def backward(ctx, *grads):
        raise RuntimeError(
            "ModelsWrapper.forward / MultiAgent.act are forward-only in this build: gradients flow through "
            "EpisodeSampler.run_episode(...) (whole episode = one autograd node with hand-written BPTT) or "
            "Trainer.train_step; wrap step-wise inference in torch.no_grad().  Set "
            "model.differentiable_steps = True to backpropagate through the step-wise API instead.")


def _step_outputs(eng: EpisodeEngine):
    """probs, values, preds, msg', h', c', h^', c^' of the last marlc_model_step, copied out of the workspace."""
    return (eng.probs[0].clone(), eng.step_values[0].clone(), eng.step_preds[0].clone(), eng.msg[1].clone(),
            eng.H_state[1].clone(), eng.C_state[1].clone(), eng.Hc_state[1].clone(), eng.Cc_state[1].clone())


class _StepFn(th.autograd.Function):
    """ModelsWrapper.forward as one autograd node (``model.differentiable_steps``).  Forward = marlc_model_step;
    backward = marlc_model_step_backward, which re-runs the step from the saved inputs (the next step-wise call
    of the geometry overwrites the workspace, so nothing but the inputs is kept) and then runs the engine's
    BPTT at T = 1 with the output gradients as its outer end.  Parameter gradients land in a fresh flat buffer
    per call, handed to autograd as one view per parameter.  With ``model.differentiable_step_inputs`` the
    windows and positions may require grad too: their gradients come from ``marlc_model_step_input_grad``."""

    @staticmethod
    def forward(ctx, eng: EpisodeEngine, model, patch, msg, npos, h, c, hc, cc, *params):
        eng.model_step(patch, msg, npos, [h, c, hc, cc])
        ctx.eng, ctx.model, ctx.params = eng, model, params
        ctx.param_generation = model.param_generation
        ctx.save_for_backward(patch, msg, npos, h, c, hc, cc)
        ctx.set_materialize_grads(False)  # an output nothing depends on passes nullptr: no seed, no copy
        return _step_outputs(eng)

    @staticmethod
    def backward(ctx, *d_out):
        eng: EpisodeEngine = ctx.eng
        model = ctx.model
        if model.param_generation != ctx.param_generation:
            raise RuntimeError(
                "ModelsWrapper.forward: a parameter was updated (optimizer step or in-place write) between this "
                "step's forward and its backward; the step's gradients would be those of different weights.  "
                "Call backward() before updating the parameters.")
        patch, msg, npos, h, c, hc, cc = ctx.saved_tensors
        d_out = [None if g is None else g.float().contiguous() for g in d_out]
        need = ctx.needs_input_grad
        d_in = [th.empty_like(x) if need[i] else None for i, x in ((3, msg), (5, h), (6, c), (7, hc), (8, cc))]
        flat = model.flat_params
        grads = th.empty_like(flat)
        eng.model_step_backward(patch, msg, npos, (h, c, hc, cc), d_out, d_in, grads)
        d_patch = th.empty_like(patch) if need[2] else None
        d_npos = th.empty_like(npos) if need[4] else None
        if need[2] or need[4]:
            eng.step_input_grad(d_patch, d_npos)
        # autograd adds each parameter gradient into param.grad in place: make sure param.grad is the parameter's
        # slot of model.flat_grads, so the bucket the fused Adam reads and param.grad stay one tensor.  After
        # zero_grad(set_to_none=True) param.grad is None: the slot starts from zero.  A gradient held outside
        # the bucket (e.g. the one a run_episode backward left after set_to_none) moves into the slot.
        base, bucket = flat.data_ptr(), model.flat_grads
        out = []
        for i, p in enumerate(ctx.params):
            if not need[9 + i]:
                out.append(None)
                continue
            off = (p.data.data_ptr() - base) // 4
            if p.grad is None or p.grad.untyped_storage().data_ptr() != bucket.untyped_storage().data_ptr():
                slot = bucket[off: off + p.numel()].view(p.shape)
                if p.grad is None:
                    slot.zero_()
                else:
                    slot.copy_(p.grad)
                p.grad = slot
            out.append(grads[off: off + p.numel()].view(p.shape))
        return (None, None, d_patch, d_in[0], d_npos, *d_in[1:], *out)


def model_step(model, img_patch, msg_t, norm_pos, hidden):
    """ModelsWrapper.forward (models.py:78-138) through the engine, slot 0."""
    from .networks.models import ModelOutput, RecurrentOutput

    patch = _lib.require_cuda(img_patch, "img_patch", th.float32)
    na, nb, Cc, f, f2 = patch.shape
    msg = _lib.require_cuda(msg_t, "msg_t", th.float32)
    npos = _lib.require_cuda(norm_pos, "norm_pos", th.float32)
    hid = [_lib.require_cuda(t, "recurrent_hidden", th.float32)
           for t in (hidden.h, hidden.c, hidden.h_caret, hidden.c_caret)]
    d = model.dims
    if f != model.feature_extractor.cnn_spec[0] or f2 != f:
        raise RuntimeError(f"img_patch window {f}x{f2} != model window {model.feature_extractor.cnn_spec[0]}")
    eng = get_engine(model, na=na, nb=nb, T=1, C=Cc, H=f + 1, W=f + 1, actions=[[0, 0]] * d["nb_action"], gamma=1.0)
    if th.is_grad_enabled() and getattr(model, "differentiable_steps", False):
        if not getattr(model, "differentiable_step_inputs", False):
            for t, name in ((img_patch, "img_patch"), (norm_pos, "norm_pos")):
                if t.requires_grad:
                    raise RuntimeError(f"ModelsWrapper.forward: {name} requires grad, but the step-wise backward "
                                       f"computes no gradient for it; pass {name}.detach(), or set "
                                       "model.differentiable_step_inputs = True to backpropagate into it")
        o = _StepFn.apply(eng, model, patch, msg, npos, *hid, *model.parameters())
        return ModelOutput(*o[:4]), RecurrentOutput(*o[4:])
    eng.model_step(patch, msg, npos, hid)
    o = _step_outputs(eng)
    out, rec = ModelOutput(*o[:4]), RecurrentOutput(*o[4:])
    if th.is_grad_enabled():
        anchor = next((p for p in model.parameters() if p.requires_grad), None)
        if anchor is not None:  # same values; a backward() through them raises (see _ForwardOnly)
            o = _ForwardOnly.apply(anchor, out.actions_probabilities, out.values, out.predictions, out.messages,
                                   rec.h, rec.c, rec.h_caret, rec.c_caret)
            out = ModelOutput(*o[:4])
            rec = RecurrentOutput(*o[4:])
    return out, rec


def cnn_forward(module, o_t: th.Tensor) -> th.Tensor:
    """_Generic2dCnnModule.forward (vision.py:47-49) on [N,C,f,f] windows."""
    x = _lib.require_cuda(o_t, "o_t", th.float32)
    f, layers, groups, _ = module.cnn_spec
    n, c_img = x.shape[0], x.shape[1]
    if x.shape[2] != f or x.shape[3] != f or c_img < layers[0][0]:
        raise RuntimeError(f"CNN expects [N,>={layers[0][0]},{f},{f}], got {tuple(x.shape)}")
    L = len(layers)
    seq = [m for m in module.modules() if isinstance(m, (th.nn.Conv2d, th.nn.GroupNorm))]
    convs, norms = seq[0::2], seq[1::2]
    arr = lambda vals: (ct.c_int * L)(*vals)  # noqa: E731
    parr = lambda ts: (ct.c_void_p * L)(*[t.data_ptr() for t in ts])  # noqa: E731
    w = [m.weight.detach().contiguous() for m in convs]
    b = [m.bias.detach().contiguous() for m in convs]
    gw = [m.weight.detach().contiguous() for m in norms]
    gb = [m.bias.detach().contiguous() for m in norms]
    for t in w + b + gw + gb:
        _lib.require_cuda(t, "CNN parameter", th.float32)
    out = th.empty(n, module.out_size, dtype=th.float32, device=x.device)
    _lib.check(_lib.lib().marlc_cnn_forward(
        L, arr([ci for ci, _ in layers]), arr([co for _, co in layers]), arr(groups), f, c_img,
        parr(w), parr(b), parr(gw), parr(gb), x.data_ptr(), out.data_ptr(), n, _lib.stream_ptr(x.device)))
    return out

"""ModelsWrapper: every agent network behind the reference's interface
(reference: networks/models.py).

All parameters live in ONE flat fp32 device buffer (``flat_params``) laid out by
the CUDA engine (256-byte aligned slots); each ``nn.Parameter`` is a view into
it with the reference's shape, so ``state_dict`` round-trips with reference
checkpoints while the kernels (and a single NCCL all-reduce) see one bucket.
Gradients live in a parallel flat buffer (``flat_grads``) that the backward
kernels write directly; ``param.grad`` are views into it.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import torch as th
from torch import nn

from .. import _lib
from .blocks import (
    Critic, LSTMCellWrapper, MessageReceiver, MessageSender, Policy, Prediction, StateToFeatures, init_layers,
)
from .vision import VisionCnnModule, _Generic2dCnnModule


@dataclass
class ModelOutput:
    actions_probabilities: th.Tensor
    values: th.Tensor
    predictions: th.Tensor
    messages: th.Tensor


@dataclass
class RecurrentOutput:
    h: th.Tensor
    c: th.Tensor
    h_caret: th.Tensor
    c_caret: th.Tensor


class ModelsWrapper(nn.Module):
    """Same constructor, attributes and ``state_dict`` keys as the reference
    (models.py:31-76); compute goes through libmarlc."""

    def __init__(
        self,
        ft_extractor: VisionCnnModule,
        n_b: int,
        n_a: int,
        n_m: int,
        n_m_o: int,
        n_d: int,
        d: int,
        nb_action: int,
        nb_class: int,
        hidden_size_belief: int,
        hidden_size_action: int,
    ) -> None:
        super().__init__()
        if d != 2:
            raise RuntimeError(f"state_dim={d}: only 2-D images are supported by the B200 hot path")
        if not isinstance(ft_extractor, _Generic2dCnnModule):
            raise RuntimeError(
                "the CUDA engine supports the conv3x3-s2/GroupNorm/SiLU feature extractors "
                "(MnistCnn, Resisc45Cnn, AidCnn, WorldStratCnn, SkinCancerCnn); got " + type(ft_extractor).__name__
            )
        self.__n_b, self.__n_a, self.__n_m = n_b, n_a, n_m
        self.__dims = dict(n_b=n_b, n_a=n_a, n_m=n_m, n_m_o=n_m_o, n_d=n_d, nb_action=nb_action,
                           nb_class=nb_class, nl_b=hidden_size_belief, nl_a=hidden_size_action)

        self.__map_obs = ft_extractor
        self.__map_pos = StateToFeatures(d, n_d)
        self.__encode_msg = MessageSender(n_b, n_m, n_m * 2)
        self.__decode_msg = MessageReceiver(n_m, n_m_o, n_m * 2)
        k_in = ft_extractor.out_size + n_d + n_m_o
        self.__belief_unit = LSTMCellWrapper(k_in, n_b)
        self.__action_unit = LSTMCellWrapper(k_in, n_a)
        self.__policy = Policy(nb_action, n_a, hidden_size_action)
        self.__critic = Critic(n_a, hidden_size_action)
        self.__predict = Prediction(n_b, nb_class, hidden_size_belief)
        self.__nb_class = nb_class

        self.apply(init_layers)

        self._flat_params: th.Tensor | None = None
        self._flat_grads: th.Tensor | None = None
        self._engines: dict = {}
        self.use_tc = True  # tensor-core GEMMs where shapes allow; False = exact fp32 FFMA everywhere
        self.precision = "tf32x3"  # "tf32x3" (error-compensated, fp32-class) | "tf32" (fastest, ~1e-3)
        self.use_chains = True  # fused per-step chain kernels; False = one kernel per op (debug / comparison)
        # True: forward() / MultiAgent.act in grad mode carry a backward (engine.model_step); False: they are
        # forward-only and a backward() reaching them raises
        self.differentiable_steps = False
        # True (with differentiable_steps): the step-wise backward also gives gradients to img_patch / norm_pos that
        # require grad (pixel attribution, input optimisation with a hand-written loop); False: such inputs raise
        self.differentiable_step_inputs = False
        self._param_updates = 0  # parameter writes torch cannot see (the fused Adam): see param_generation

    # ---- reference surface ------------------------------------------------------
    @property
    def nb_class(self) -> int:
        return self.__nb_class

    @property
    def device(self) -> th.device:
        return next(self.parameters()).device

    def random_first_state(self, nb_agents: int, batch_size: int) -> RecurrentOutput:
        """h, c, h^, c^ ~ N(0,1), drawn in that order (models.py:148-159)."""
        def draw(size: int) -> th.Tensor:
            return th.randn(nb_agents, batch_size, size, device=self.device)

        return RecurrentOutput(h=draw(self.__n_b), c=draw(self.__n_b), h_caret=draw(self.__n_a), c_caret=draw(self.__n_a))

    def zero_first_message(self, nb_agents: int, batch_size: int) -> th.Tensor:
        return th.zeros(nb_agents, batch_size, self.__n_m, device=self.device)

    def forward(
        self, img_patch: th.Tensor, msg_t: th.Tensor, norm_pos: th.Tensor, recurrent_hidden: RecurrentOutput
    ) -> tuple[ModelOutput, RecurrentOutput]:
        """One step of every network (models.py:78-138) on CUDA.  With ``differentiable_steps`` set, the
        outputs carry a backward to every parameter, ``msg_t`` and ``recurrent_hidden``, and, with
        ``differentiable_step_inputs`` set as well, to ``img_patch`` / ``norm_pos``; otherwise this is
        forward-only and training goes through EpisodeSampler.run_episode, whose outputs carry the hand-written
        BPTT backward."""
        from ..engine import model_step

        return model_step(self, img_patch, msg_t, norm_pos, recurrent_hidden)

    # ---- engine plumbing --------------------------------------------------------
    @property
    def dims(self) -> dict:
        return dict(self.__dims)

    @property
    def param_generation(self) -> int:
        """Changes whenever a parameter is written: in place through torch, on a parameter or on the flat buffer
        they all view (version counters), or by the fused Adam (``note_param_update``).  A step-wise backward
        refuses to run across such a write."""
        flat = self._flat_params._version if self._flat_params is not None else 0
        return self._param_updates + flat + sum(p._version for p in self.parameters())

    def note_param_update(self) -> None:
        """Record a parameter write that bypasses torch (a kernel writing ``flat_params`` through its pointer)."""
        self._param_updates += 1

    @property
    def feature_extractor(self) -> _Generic2dCnnModule:
        return self.__map_obs

    @property
    def flat_params(self) -> th.Tensor:
        self.ensure_flat()
        return self._flat_params

    @property
    def flat_grads(self) -> th.Tensor:
        self.ensure_flat()
        return self._flat_grads

    def _layout(self):
        """Ask the engine for the flat layout (names, offsets, shapes)."""
        from ..engine import build_config

        f = self.__map_obs.cnn_spec[0]
        cfg = build_config(self, na=1, nb=1, T=1, C=max(1, self.__map_obs.cnn_spec[1][0][0]), H=f + 1, W=f + 1,
                           actions=[[0, 0]] * self.__dims["nb_action"], gamma=1.0)
        L = _lib.lib()
        handle = C.c_void_p()
        _lib.check(L.marlc_engine_create(C.byref(cfg), C.byref(handle)))
        try:
            out = []
            name = C.create_string_buffer(128)
            off, ndim, shape = C.c_int64(), C.c_int(), (C.c_int64 * 4)()
            for i in range(L.marlc_engine_param_count(handle)):
                _lib.check(L.marlc_engine_param_info(handle, i, name, C.byref(off), C.byref(ndim), shape))
                out.append((name.value.decode(), off.value, tuple(shape[k] for k in range(ndim.value))))
            return out, L.marlc_engine_param_floats(handle)
        finally:
            L.marlc_engine_destroy(handle)

    def ensure_flat(self) -> None:
        """(Re)pack the parameters into the flat device buffer if needed."""
        if self._flat_params is not None:
            return
        params = dict(self.named_parameters())
        dev = next(iter(params.values())).device
        if dev.type != "cuda":
            raise RuntimeError("ModelsWrapper must be on a CUDA device (no CPU path): call .to('cuda')")
        layout, total = self._layout()
        if {n for n, _, _ in layout} != set(params):
            raise RuntimeError("engine / module parameter names differ: " + str(set(params) ^ {n for n, _, _ in layout}))
        flat = th.zeros(total, dtype=th.float32, device=dev)
        grads = th.zeros(total, dtype=th.float32, device=dev)
        with th.no_grad():
            for name, off, shape in layout:
                p = params[name]
                if tuple(p.shape) != shape:
                    raise RuntimeError(f"{name}: module shape {tuple(p.shape)} != engine shape {shape}")
                n = p.numel()
                flat[off:off + n].view(shape).copy_(p.data.to(dev, th.float32))
                p.data = flat[off:off + n].view(shape)
                p.grad = grads[off:off + n].view(shape)
        self._flat_params, self._flat_grads = flat, grads
        self._engines.clear()
        from ..engine import register_flat_owner

        register_flat_owner(self.__map_obs, self)  # a stand-alone feature-extractor backward fills this bucket too

    def attach_grads(self) -> None:
        """Point every ``param.grad`` at its slot of the flat bucket (after
        ``zero_grad(set_to_none=True)`` or a fused backward)."""
        self.ensure_flat()
        base = self._flat_params.data_ptr()
        for p in self.parameters():
            if p.grad is None or p.grad.untyped_storage().data_ptr() != self._flat_grads.untyped_storage().data_ptr():
                off = (p.data.data_ptr() - base) // 4
                p.grad = self._flat_grads[off: off + p.numel()].view(p.shape)

    def _apply(self, fn, recurse=True):  # .to() / .cuda() re-create parameter storage: re-pack lazily
        out = super()._apply(fn, recurse)
        self._flat_params = None
        self._flat_grads = None
        self._engines.clear()
        return out

    def load_state_dict(self, state_dict, strict: bool = True, assign: bool = False):
        out = super().load_state_dict(state_dict, strict=strict, assign=False)
        return out

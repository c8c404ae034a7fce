"""Environment: image batch, integer agent positions, action semantics
(reference: core/environment.py).  Same constructor / methods / properties;
observation and transition run as CUDA kernels (csrc/env.cu)."""
from __future__ import annotations

import torch as th

from .. import _lib


def _gather(img: th.Tensor, pos: th.Tensor, f: int) -> th.Tensor:
    na, nb = pos.shape[0], pos.shape[1]
    _, c, h, w = img.shape
    obs = th.empty(na, nb, c, f, f, dtype=th.float32, device=img.device)
    _lib.check(_lib.lib().marlc_patch_gather(img.data_ptr(), pos.data_ptr(), obs.data_ptr(), na, nb, c, h, w, f,
                                             _lib.stream_ptr(img.device)))
    return obs


class _ObserveFn(th.autograd.Function):
    """Environment.observe as an autograd node: forward = marlc_patch_gather, backward = its adjoint
    marlc_patch_gather_backward (a pixel sums the gradients of the windows covering it, in agent order).  The
    positions of the call are saved: ``step`` binds a new tensor, so they stay those of this observation."""

    @staticmethod
    def forward(ctx, img, pos, f):
        ctx.save_for_backward(pos)
        ctx.f, ctx.img_shape = f, img.shape
        return _gather(img, pos, f)

    @staticmethod
    def backward(ctx, d_obs):
        (pos,) = ctx.saved_tensors
        d_obs = d_obs.float().contiguous()
        na, nb = pos.shape[0], pos.shape[1]
        _, c, h, w = ctx.img_shape
        d_img = th.empty(ctx.img_shape, dtype=th.float32, device=d_obs.device)
        _lib.check(_lib.lib().marlc_patch_gather_backward(d_obs.data_ptr(), pos.data_ptr(), d_img.data_ptr(), na, nb,
                                                          c, h, w, ctx.f, _lib.stream_ptr(d_obs.device)))
        return d_img, None, None


class Environment:
    def __init__(self, actions: list[list[int]], window_size: int) -> None:
        self.__actions = actions
        self.__window_size = window_size
        self.__img_batch: th.Tensor | None = None
        self.__img_sizes: list[int] = []
        self.__pos = th.empty(0)
        self.__actions_table = th.empty(0)
        self.__err: th.Tensor | None = None

    # ---- reference surface (environment.py:23-93) ---------------------------------
    def reset(self, img_batch: th.Tensor, nb_agents: int) -> th.Tensor:
        """Place the agents uniformly at random (one ``th.randint`` per spatial
        dim, dim 0 first -- environment.py:33-43) and return o_0."""
        img = _lib.require_cuda(img_batch, "Environment.reset(img_batch)", th.float32)
        if img.dim() != 4:
            raise RuntimeError(f"only 2-D images [B,C,H,W] are supported (state_dim == 2), got {tuple(img.shape)}")
        device, batch_size = img.device, img.size(0)
        sizes = list(img.shape[2:])
        if self.__window_size >= min(sizes):
            raise RuntimeError(f"window f={self.__window_size} does not fit image {sizes}")
        self.__img_batch, self.__img_sizes = img, sizes
        if self.__actions_table.device != device or self.__actions_table.numel() == 0:
            self.__actions_table = th.tensor(self.__actions, dtype=th.long, device=device)
            self.__err = th.zeros(1, dtype=th.int32, device=device)
        self.__pos = th.stack(
            [th.randint(s - self.__window_size, (nb_agents, batch_size), device=device) for s in sizes], dim=-1
        ).contiguous()
        return self.observe()

    def observe(self) -> th.Tensor:
        """The agents' windows [Na, B, C, f, f].  When the image batch requires grad (in grad mode) they carry
        a backward to it, as the reference's masked_select does (environment.py:96-126)."""
        assert self.__img_batch is not None, "reset() must be called before observe()"
        img, pos, f = self.__img_batch, self.__pos, self.__window_size
        if th.is_grad_enabled() and img.requires_grad:
            return _ObserveFn.apply(img, pos, f)
        return _gather(img, pos, f)

    def step(self, action_indices: th.Tensor) -> th.Tensor:
        """Apply the chosen actions (integer rule of environment.py:128-150: a
        move leaving the image on ANY dim is rejected) and return the new observations."""
        assert self.__img_batch is not None, "reset() must be called before step()"
        act = _lib.require_cuda(action_indices, "Environment.step(action_indices)", th.int64)
        pos = self.__pos
        if act.shape != pos.shape[:2]:
            raise RuntimeError(f"action_indices {tuple(act.shape)} != (Na, Nb) {tuple(pos.shape[:2])}")
        new_pos = pos.clone()  # the reference rebinds positions each step; keep earlier handles valid
        h, w = self.__img_sizes
        _lib.check(_lib.lib().marlc_transition(new_pos.data_ptr(), act.data_ptr(), self.__actions_table.data_ptr(),
                                               len(self.__actions), act.numel(), self.__window_size, h, w, None,
                                               self.__err.data_ptr(), _lib.stream_ptr(pos.device)))
        self.__pos = new_pos
        return self.observe()

    def check_errors(self) -> None:
        """Synchronising check of the device-side flag (action index out of range)."""
        if self.__err is not None and int(self.__err.item()) != 0:
            self.__err.zero_()
            raise RuntimeError("Environment.step: action index out of range")

    @property
    def positions(self) -> th.Tensor:
        return self.__pos

    @property
    def normalized_positions(self) -> th.Tensor:
        pos = self.__pos
        h, w = self.__img_sizes
        out = th.empty(*pos.shape, dtype=th.float32, device=pos.device)
        _lib.check(_lib.lib().marlc_normalized_positions(pos.data_ptr(), out.data_ptr(), pos.shape[0] * pos.shape[1],
                                                         h, w, _lib.stream_ptr(pos.device)))
        return out

    @property
    def window_size(self) -> int:
        return self.__window_size

    @property
    def actions(self) -> list[list[int]]:
        return self.__actions

    @property
    def nb_actions(self) -> int:
        return len(self.__actions)

    # ---- used by the fused episode path ----------------------------------------------
    def _adopt(self, img_batch: th.Tensor, positions: th.Tensor) -> None:
        """Make the environment reflect the end state of a fused episode."""
        self.__img_batch = img_batch
        self.__img_sizes = list(img_batch.shape[2:])
        self.__pos = positions
        if self.__actions_table.device != img_batch.device or self.__actions_table.numel() == 0:
            self.__actions_table = th.tensor(self.__actions, dtype=th.long, device=img_batch.device)
            self.__err = th.zeros(1, dtype=th.int32, device=img_batch.device)

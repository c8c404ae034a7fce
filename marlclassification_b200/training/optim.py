"""Fused Adam over the model's flat parameter bucket (csrc/optim.cu)."""
from __future__ import annotations

import torch as th

from .. import _lib


class FlatAdam:
    """torch.optim.Adam semantics (lr, betas, eps; no weight decay) in ONE kernel
    over ``model.flat_params`` / ``model.flat_grads``; step counter on the device."""

    def __init__(self, model, lr: float, betas=(0.9, 0.999), eps: float = 1e-8) -> None:
        model.ensure_flat()
        self.model = model
        self.lr, self.betas, self.eps = float(lr), (float(betas[0]), float(betas[1])), float(eps)
        flat = model.flat_params
        self.exp_avg = th.zeros_like(flat)
        self.exp_avg_sq = th.zeros_like(flat)
        self.step_count = th.zeros(1, dtype=th.int64, device=flat.device)
        self._params = flat

    def zero_grad(self, set_to_none: bool = False) -> None:
        self.model.flat_grads.zero_()

    def step(self, grad_scale: float = 1.0) -> None:
        m = self.model
        if m.flat_params.data_ptr() != self._params.data_ptr():
            raise RuntimeError("model parameters were re-allocated after the optimizer was built")
        _lib.check(_lib.lib().marlc_adam_step(
            m.flat_params.data_ptr(), m.flat_grads.data_ptr(), self.exp_avg.data_ptr(), self.exp_avg_sq.data_ptr(),
            m.flat_params.numel(), self.lr, self.betas[0], self.betas[1], self.eps, float(grad_scale),
            self.step_count.data_ptr(), _lib.stream_ptr(m.flat_params.device)))
        m.note_param_update()

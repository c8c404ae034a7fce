"""Small networks of the agents (reference: networks/message.py, state.py,
recurrent.py, policy.py, prediction.py, init.py).  These classes are parameter
containers with the reference's module structure, so ``state_dict`` keys match;
the arithmetic runs in the CUDA engine (csrc/)."""
from __future__ import annotations

import math

import torch as th
from torch import nn


def _lin_norm_act(n_in: int, n_out: int) -> list[nn.Module]:
    return [nn.Linear(n_in, n_out), nn.LayerNorm(n_out), nn.SiLU()]


class MessageSender(nn.Sequential):
    """m: R^n -> R^n_m (message.py:20-33)."""

    def __init__(self, n: int, n_m: int, hidden_size: int) -> None:
        super().__init__(*_lin_norm_act(n, hidden_size), *_lin_norm_act(hidden_size, n_m))


class MessageReceiver(nn.Sequential):
    """d: R^n_m -> R^n (message.py:36-49)."""

    def __init__(self, n_m: int, n: int, hidden_size: int) -> None:
        super().__init__(*_lin_norm_act(n_m, hidden_size), *_lin_norm_act(hidden_size, n))


class StateToFeatures(nn.Sequential):
    """lambda: R^d -> R^n_d (state.py:7-17)."""

    def __init__(self, d: int, n_d: int) -> None:
        super().__init__(*_lin_norm_act(d, n_d))


class LSTMCellWrapper(nn.Module):
    """Holds an nn.LSTMCell (recurrent.py:7-18); gates i,f,g,o."""

    def __init__(self, input_size: int, n: int) -> None:
        super().__init__()
        self.__lstm = nn.LSTMCell(input_size, n)

    @property
    def cell(self) -> nn.LSTMCell:
        return self.__lstm


class Policy(nn.Sequential):
    """pi (policy.py:4-17)."""

    def __init__(self, nb_action: int, n: int, hidden_size: int) -> None:
        super().__init__(*_lin_norm_act(n, hidden_size), nn.Linear(hidden_size, nb_action), nn.Softmax(dim=-1))


class Critic(nn.Sequential):
    """V (policy.py:20-28)."""

    def __init__(self, n: int, hidden_size: int) -> None:
        super().__init__(*_lin_norm_act(n, hidden_size), nn.Linear(hidden_size, 1), nn.Flatten(-2, -1))


class Prediction(nn.Sequential):
    """q: R^n -> R^nb_class (prediction.py:4-15)."""

    def __init__(self, n: int, nb_class: int, hidden_size: int) -> None:
        super().__init__(*_lin_norm_act(n, hidden_size), nn.Linear(hidden_size, nb_class))


def init_layers(m: nn.Module) -> None:
    """Same initial distribution as the reference (init.py:6-29): orthogonal
    weights with gain sqrt(2), zero biases, unit/zero norm affines."""
    gain = math.sqrt(2.0)
    if isinstance(m, (nn.Linear, nn.Conv2d, nn.Conv3d)):
        nn.init.orthogonal_(m.weight, gain=gain)
        if m.bias is not None:
            nn.init.zeros_(m.bias)
    elif isinstance(m, nn.LSTMCell):
        nn.init.orthogonal_(m.weight_hh, gain=gain)
        nn.init.orthogonal_(m.weight_ih, gain=gain)
        if m.bias:
            nn.init.zeros_(m.bias_hh)
            nn.init.zeros_(m.bias_ih)
    elif isinstance(m, (nn.LayerNorm, nn.GroupNorm)):
        if getattr(m, "elementwise_affine", getattr(m, "affine", False)):
            nn.init.ones_(m.weight)
            nn.init.zeros_(m.bias)


def _msg_mean(msg: th.Tensor) -> th.Tensor:
    from .. import _lib

    out = th.empty_like(msg)
    na, nb, n = msg.shape
    _lib.check(_lib.lib().marlc_msg_mean(msg.data_ptr(), out.data_ptr(), na, nb, n, _lib.stream_ptr(msg.device)))
    return out


class _MsgMeanFn(th.autograd.Function):
    """The mean of the other agents' messages is a symmetric linear map over the agents (out_a = (S - m_a) /
    (Na - 1)), so it is its own adjoint: the backward is the same kernel on the incoming gradient (exactly 0 for
    Na = 1)."""

    @staticmethod
    def forward(ctx, msg):
        return _msg_mean(msg)

    @staticmethod
    def backward(ctx, grad):
        return _MsgMeanFn.apply(grad.float().contiguous())


def aggregate_messages(messages: th.Tensor) -> th.Tensor:
    """Mean of the OTHER agents' messages (message.py:5-17), CUDA kernel
    csrc/rowwise.cu::msg_mean_kernel (warp-shuffle reduction over agents); differentiable in ``messages``."""
    from .. import _lib

    msg = _lib.require_cuda(messages, "aggregate_messages", th.float32)
    if th.is_grad_enabled() and msg.requires_grad:
        return _MsgMeanFn.apply(msg)
    return _msg_mean(msg)

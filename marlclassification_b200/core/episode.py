"""EpisodeSampler: the T-step rollout (reference: core/episode.py).

``run_episode`` executes the whole episode inside the CUDA engine (one host
call: gather -> CNN -> messages -> LSTMs -> heads -> sample -> transition, T
times) and returns tensors that carry the hand-written BPTT backward as a single
autograd node, so the reference's loss code and ``loss.backward()`` work as is: the
gradients reach the parameters and, when it requires grad, the image batch.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional, Sequence

import torch as th

from ..engine import EpisodeEngine, get_engine, rollout_autograd
from ..networks.models import RecurrentOutput
from .agent import MultiAgent
from .environment import Environment


@dataclass
class EpisodeOutput:
    prediction: th.Tensor
    actions_log_probs: th.Tensor


@dataclass
class EpisodeDetailedOutput:
    step_preds: th.Tensor  # [T, Na, Nb, Nc]
    step_log_probas: th.Tensor  # [T, Na, Nb]
    step_values: th.Tensor  # [T, Na, Nb]
    step_pos: th.Tensor  # [T, Na, Nb, 2] int64, positions AFTER each move


class EpisodeSampler:
    def __init__(self, agents: MultiAgent, env: Environment, nb_step: int, gamma: float = 0.99) -> None:
        self.__agents = agents
        self.__env = env
        self.__nb_step = nb_step
        self.__gamma = gamma

    def engine_for(self, img_batch: th.Tensor, gamma: Optional[float] = None) -> EpisodeEngine:
        nb, c, h, w = img_batch.shape
        return get_engine(self.__agents.model, na=len(self.__agents), nb=nb, T=self.__nb_step, C=c, H=h, W=w,
                          actions=self.__env.actions, gamma=self.__gamma if gamma is None else gamma)

    def __episode_impl(self, img_batch, pos0, hidden0, actions) -> EpisodeDetailedOutput:
        device = self.__agents.device
        if device.type != "cuda":
            raise RuntimeError("the model must live on a CUDA device (no CPU path)")
        img = img_batch.to(device=device, dtype=th.float32).contiguous()  # episode.py:34
        if img.dim() != 4:
            raise RuntimeError(f"only 2-D images [B,C,H,W] are supported, got {tuple(img.shape)}")
        eng = self.engine_for(img)
        # the autograd node is built for the parameters or for the image (attribution on a frozen model); the
        # conversion above is differentiable, so the image gradient reaches img_batch itself
        if th.is_grad_enabled() and (img.requires_grad or any(p.requires_grad for p in eng.model.parameters())):
            preds, logp, values, pos = rollout_autograd(eng, img, pos0, hidden0, actions)
        else:
            eng.forward(img, pos0, hidden0, actions)
            preds, logp, values, pos = (eng.step_preds.clone(), eng.step_log_probas.clone(),
                                        eng.step_values.clone(), eng.step_pos.clone())
        # leave env / agents in the state the reference's loop would
        self.__env._adopt(img, pos[-1])
        T = self.__nb_step
        self.__agents._adopt(
            RecurrentOutput(eng.H_state[T].clone(), eng.C_state[T].clone(), eng.Hc_state[T].clone(),
                            eng.Cc_state[T].clone()),
            eng.msg[T].clone(),
        )
        return EpisodeDetailedOutput(preds, logp, values, pos)

    def run_episode(self, img_batch: th.Tensor, *, pos0: Optional[th.Tensor] = None,
                    hidden0: Optional[Sequence[th.Tensor]] = None,
                    actions: Optional[th.Tensor] = None) -> EpisodeDetailedOutput:
        """episode.py:84-85.  The keyword-only arguments inject the reference's three
        random sites (initial positions, initial recurrent state, sampled actions)
        for parity testing; by default everything is drawn on the device."""
        return self.__episode_impl(img_batch, pos0, hidden0, actions)

    def run_episode_get_last_step(self, img_batch: th.Tensor, **inject) -> EpisodeOutput:
        out = self.__episode_impl(img_batch, inject.get("pos0"), inject.get("hidden0"), inject.get("actions"))
        return EpisodeOutput(prediction=out.step_preds[-1], actions_log_probs=out.step_log_probas[-1])

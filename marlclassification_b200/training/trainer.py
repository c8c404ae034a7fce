"""Actor-critic training loop (reference: training/trainer.py).

Same constructor / ``train_epoch`` / ``eval_epoch`` / ``curr_step`` surface.  One
iteration is: fused rollout -> fused loss (+ gradients w.r.t. the rollout
outputs) -> hand-written BPTT into the flat gradient bucket -> (data-parallel:
one NCCL all-reduce of the bucket) -> Adam.  The five logged scalars come back
in ONE small device->host copy instead of the reference's 5+ ``.item()`` syncs.
"""
from __future__ import annotations

from typing import Callable, Dict, Optional

import torch as th
from tqdm import tqdm

from ..core import EpisodeSampler
from ..input_pipeline import DevicePrefetcher
from ..metrics import ConfusionMeter, LossMeter
from ..networks import ModelsWrapper
from ..parallel import DataParallelContext
from .optim import FlatAdam
from .step import EvalStep, TrainStep

MetricLogger = Callable[[int, Dict[str, float]], None]


class Trainer:
    def __init__(
        self,
        model: ModelsWrapper,
        nb_class: int,
        learning_rate: float,
        gamma: float,
        metric_logger: Optional[MetricLogger] = None,
        log_interval: int = 100,
        meter_window_size: int = 64,
        *,
        dp: Optional[DataParallelContext] = None,
        cuda_graph: bool = True,
    ) -> None:
        self.__model = model
        model.ensure_flat()
        self.__optim = FlatAdam(model, lr=learning_rate)  # th.optim.Adam semantics, trainer.py:33
        self.__cuda_graph = cuda_graph
        self.__steps: dict = {}
        self.__eval_steps: dict = {}
        self.__nb_class = nb_class
        self.__gamma = gamma
        self.__metric_logger = metric_logger
        self.__log_interval = log_interval
        self.__curr_step = 0
        self.__dp = dp if dp is not None else DataParallelContext()
        self.__conf_meter = ConfusionMeter(nb_class, window_size=meter_window_size)
        self.__path_loss_meter = LossMeter(window_size=meter_window_size)
        self.__error_meter = LossMeter(window_size=meter_window_size)
        self.__actor_loss_meter = LossMeter(window_size=meter_window_size)
        self.__critic_loss_meter = LossMeter(window_size=meter_window_size)

    @property
    def curr_step(self) -> int:
        return self.__curr_step

    def train_step(self, x: th.Tensor, y: th.Tensor, episode_sampler: EpisodeSampler, **inject) -> th.Tensor:
        """One optimisation step (trainer.py:66-116): rollout, loss, backward, Adam.
        Returns the device tensor [loss, path, error, actor, critic] without
        synchronising.  ``x`` / ``y`` may be host (pinned) or device tensors, or ``x`` a
        StagedBatch produced by :meth:`prefetch` (then ``y`` is ignored)."""
        eng = episode_sampler.engine_for(x, gamma=self.__gamma)
        if eng.T * eng.na * eng.nb * self.__dp.world_size < 2:
            # the fused loss would be NaN (the standard deviation of one advantage, as in the reference) and its
            # NaN gradients would reach every parameter through Adam: refuse before anything is updated
            raise RuntimeError("the batch holds a single advantage (nb_step * nb_agents * images == 1), whose "
                               "standard deviation is undefined: use more steps, agents or images per batch")
        step = self.__steps.get(id(eng))
        if step is None:
            step = TrainStep(eng, self.__optim, self.__dp, use_graph=self.__cuda_graph)
            self.__steps[id(eng)] = step
        return step(x, y, **inject)

    def eval_step(self, x, episode_sampler: EpisodeSampler, **inject) -> th.Tensor:
        """Forward-only episode; returns the [Nb, Nc] agent-mean prediction of the last step
        (static device buffer, overwritten by the next call).  ``x``: tensor or StagedBatch.
        ``pos0`` / ``hidden0`` / ``actions`` inject the reference's random draws (parity tests)."""
        eng = episode_sampler.engine_for(x, gamma=self.__gamma)
        step = self.__eval_steps.get(id(eng))
        if step is None:
            step = EvalStep(eng, use_graph=self.__cuda_graph)
            self.__eval_steps[id(eng)] = step
        with th.no_grad():
            return step(x, **inject)

    def prefetch(self, batches, *, hwc: bool = True) -> DevicePrefetcher:
        """Wrap an iterable of host ``(images, labels)`` batches (fp32 NCHW as the reference's
        DataLoader yields them, or raw uint8) so that the copy of batch i+1 overlaps step i."""
        return DevicePrefetcher(batches, self.__model.device, hwc=hwc)

    def train_epoch(self, dataloader, epoch_index: int, episode_sampler: EpisodeSampler) -> None:
        self.__model.train()
        tqdm_bar = tqdm(self.prefetch(dataloader))
        for staged in tqdm_bar:
            loss_out = self.train_step(staged, None, episode_sampler)
            eng = episode_sampler.engine_for(staged, gamma=self.__gamma)
            y_train = self.__steps[id(eng)].static_y.clone()
            # meters: ONE packed device->host read per iteration (the five loss scalars + mean
            # precision / recall of the running confusion matrix) instead of the reference's 7+ syncs
            self.__conf_meter.add(eng.step_preds[-1].mean(dim=0), y_train)
            packed = th.cat((loss_out[:6], self.__conf_meter.mean_precision_recall().to(loss_out.dtype)))
            loss_item, path_item, error_item, actor_item, critic_item, bad_labels, *prec_rec = packed.tolist()
            if bad_labels > 0:  # the reference's cross_entropy raises a device assert here (trainer.py:83-87)
                raise RuntimeError(f"{int(bad_labels)} label(s) of the batch are outside [0, {self.__nb_class}): "
                                   "nb_class is smaller than the dataset's number of classes")
            self.__path_loss_meter.add(path_item)
            self.__error_meter.add(error_item)
            self.__actor_loss_meter.add(actor_item)
            self.__critic_loss_meter.add(critic_item)
            if self.__metric_logger is not None and self.__curr_step % self.__log_interval == 0:
                self.__metric_logger(
                    self.__curr_step,
                    {"error": error_item, "path_loss": path_item, "loss": loss_item,
                     "train_prec": prec_rec[0], "train_rec": prec_rec[1]},
                )
            tqdm_bar.set_description(
                f"Epoch {epoch_index} - Train, train_prec = {prec_rec[0]:.3f}, train_rec = {prec_rec[1]:.3f}, "
                f"error = {self.__error_meter.loss():.4f}, path = {self.__path_loss_meter.loss():.4f}, "
                f"actor = {self.__actor_loss_meter.loss():.4f}, critic = {self.__critic_loss_meter.loss():.4f}"
            )
            self.__curr_step += 1

    def eval_epoch(self, dataloader, epoch_index: int, episode_sampler: EpisodeSampler) -> ConfusionMeter:
        self.__model.eval()
        conf_meter = ConfusionMeter(self.__nb_class, None)
        with th.no_grad():
            tqdm_bar = tqdm(self.prefetch(dataloader))
            for staged in tqdm_bar:
                vote = self.eval_step(staged, episode_sampler)  # mean over agents, trainer.py:180
                eng = episode_sampler.engine_for(staged, gamma=self.__gamma)
                conf_meter.add(vote, self.__eval_steps[id(eng)].static_y.clone())
                pr = conf_meter.mean_precision_recall().tolist()
                tqdm_bar.set_description(
                    f"Epoch {epoch_index} - Eval, eval_prec = {pr[0]:.4f}, eval_rec = {pr[1]:.4f}"
                )
        return conf_meter

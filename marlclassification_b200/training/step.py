"""One optimisation step for a fixed episode geometry, replayed as CUDA graphs.

The step is   rollout -> loss phase A -> [all-reduce 3 doubles] -> loss phase B
-> BPTT -> [all-reduce flat grads] -> fused Adam.   Everything between the
collectives is one captured graph (the engine never allocates or synchronises),
so a 16-step episode costs a handful of host calls instead of ~10^4 launches.
"""
from __future__ import annotations

from typing import Optional

import torch as th

from ..engine import EpisodeEngine
from ..input_pipeline import StagedBatch
from ..parallel import DataParallelContext
from .optim import FlatAdam


class TrainStep:
    def __init__(self, engine: EpisodeEngine, optim: FlatAdam, dp: Optional[DataParallelContext] = None,
                 use_graph: bool = True) -> None:
        self.engine, self.optim = engine, optim
        self.dp = dp if dp is not None else DataParallelContext()
        self.use_graph = use_graph
        dev = engine.device
        self.static_img = th.zeros(engine.nb, engine.C, engine.H, engine.W, dtype=th.float32, device=dev)
        self.static_y = th.zeros(engine.nb, dtype=th.int64, device=dev)
        # one set of graphs per mode: drawn on the device (False) / injected draws in static buffers (True)
        self._graphs: dict = {False: None, True: None}
        self._warm = {False: 0, True: 0}
        self._inj: Optional[dict] = None  # static pos0 / hidden0 / actions (parity runs through the graph path)
        # Data parallel: three graphs with the two NCCL all-reduces issued eagerly between them.  One graph with the
        # collectives captured inside it was measured on 2 B200 (config c4, 128 images per GPU): 8.03 ms per
        # iteration against 7.93 ms for three graphs, and it hung in tests/test_gpu_dp.py, so it was removed.
        # Reported by bench.py: the collectives are never part of a captured graph.
        self.nccl_in_graph = False

    # ---- the segments between collectives -----------------------------------------
    def _seg_forward(self, injected: bool = False) -> None:
        if injected:
            self.engine.forward(self.static_img, self._inj["pos0"], self._inj["hidden0"], self._inj["actions"])
        else:
            self.engine.forward(self.static_img)
        self.engine.loss_phase_a(self.static_y)

    def _seg_backward(self) -> None:
        self.engine.loss_phase_b()
        self.engine.backward(self.static_img)

    def _seg_update(self) -> None:
        self.optim.step(1.0 / self.dp.world_size)

    def _segments(self, injected: bool = False):
        fwd = lambda: self._seg_forward(injected)  # noqa: E731
        if self.dp.enabled:
            return [fwd, self._seg_backward, self._seg_update]
        return [lambda: (fwd(), self._seg_backward(), self._seg_update())]

    def _capture(self, injected: bool) -> None:
        """Single GPU: ONE CUDA graph for the whole iteration.  Data parallel: the segments between the two
        NCCL all-reduces (3 doubles of advantage statistics, the flat gradient bucket) are one graph each."""
        graphs = []
        for seg in self._segments(injected):
            g = th.cuda.CUDAGraph()
            with th.cuda.graph(g):
                seg()
            graphs.append(g)
        self._graphs[injected] = graphs

    @property
    def launches_per_step(self) -> int:
        l = self.engine.launches
        return l["forward"] + l["loss"] + l["backward"] + 2  # + Adam (2 kernels)

    def run_static(self, injected: bool = False) -> th.Tensor:
        """Run one step on whatever is in static_img / static_y (and, when ``injected``, in the static
        draw buffers).  Two eager steps, then the step is captured and replayed."""
        eng, dp = self.engine, self.dp
        if self.use_graph and self._graphs[injected] is None and self._warm[injected] >= 2:
            self._capture(injected)
        if self._graphs[injected] is not None:
            segs = [g.replay for g in self._graphs[injected]]
        else:
            segs = self._segments(injected)
            self._warm[injected] += 1
        if dp.enabled:
            segs[0]()
            dp.all_reduce_stats(eng.loss_stats)
            segs[1]()
            dp.all_reduce_grads_sum(eng.model.flat_grads)
            segs[2]()
        else:
            segs[0]()
        if self._graphs[injected] is not None:
            # a replay runs the fused Adam without calling FlatAdam.step(): record the parameter write here, so a
            # step-wise backward across it refuses to run (ModelsWrapper.param_generation)
            eng.model.note_param_update()
        return eng.loss_out

    def __call__(self, img: th.Tensor, y: th.Tensor, **inject) -> th.Tensor:
        """img / y may live on the host (pinned -> async H2D) or on the device, or be a
        StagedBatch from the DevicePrefetcher (copy already in flight on the copy stream)."""
        if isinstance(img, StagedBatch):
            img.deliver(self.static_img, self.static_y)
            return self.run_static()
        self.static_img.copy_(img, non_blocking=True)
        self.static_y.copy_(y, non_blocking=True)
        if inject.get("pos0") is not None or inject.get("hidden0") is not None or inject.get("actions") is not None:
            self._stage_injection(inject)
            return self.run_static(injected=True)
        return self.run_static()

    def _stage_injection(self, inject) -> None:
        """Parity path: the three random sites of the reference (initial positions, initial recurrent
        state, per-step actions) are copied into STATIC buffers, so the injected step runs through the
        same capture / replay machinery as the production step (all three must be given)."""
        if any(inject.get(k) is None for k in ("pos0", "hidden0", "actions")):
            raise RuntimeError("injected train step: pos0, hidden0 and actions must all be given")
        if self._inj is None:
            self._inj = {"pos0": th.empty_like(inject["pos0"], device=self.engine.device).contiguous(),
                         "hidden0": [th.empty_like(h, device=self.engine.device).contiguous() for h in inject["hidden0"]],
                         "actions": th.empty_like(inject["actions"], device=self.engine.device).contiguous()}
        self._inj["pos0"].copy_(inject["pos0"], non_blocking=True)
        for dst, src in zip(self._inj["hidden0"], inject["hidden0"]):
            dst.copy_(src, non_blocking=True)
        self._inj["actions"].copy_(inject["actions"], non_blocking=True)


class EvalStep:
    """Forward-only rollout for a fixed geometry (trainer.py:164-196: ``no_grad`` episode, vote =
    mean over agents of the last step's predictions), replayed as one CUDA graph."""

    def __init__(self, engine: EpisodeEngine, use_graph: bool = True) -> None:
        self.engine, self.use_graph = engine, use_graph
        dev = engine.device
        self.static_img = th.zeros(engine.nb, engine.C, engine.H, engine.W, dtype=th.float32, device=dev)
        self.static_y = th.zeros(engine.nb, dtype=th.int64, device=dev)
        self.vote = th.zeros(engine.nb, engine.step_preds.shape[-1], dtype=th.float32, device=dev)
        self._graph: dict = {False: None, True: None}
        self._warm = {False: 0, True: 0}
        self._inj: Optional[dict] = None

    def _body(self, injected: bool = False) -> None:
        if injected:
            self.engine.forward(self.static_img, self._inj["pos0"], self._inj["hidden0"], self._inj["actions"])
        else:
            self.engine.forward(self.static_img)
        th.mean(self.engine.step_preds[-1], dim=0, out=self.vote)  # prediction.mean(0), trainer.py:180

    def run_static(self, injected: bool = False) -> th.Tensor:
        if self.use_graph and self._graph[injected] is None and self._warm[injected] >= 2:
            g = th.cuda.CUDAGraph()
            with th.cuda.graph(g):
                self._body(injected)
            self._graph[injected] = g
        if self._graph[injected] is not None:
            self._graph[injected].replay()
        else:
            self._body(injected)
            self._warm[injected] += 1
        return self.vote

    def __call__(self, img, **inject) -> th.Tensor:
        """Returns the [Nb, Nc] vote (a static buffer: clone it to keep it across calls).  ``pos0`` /
        ``hidden0`` / ``actions`` inject the reference's random draws (static buffers, same graph path)."""
        if isinstance(img, StagedBatch):
            img.deliver(self.static_img, self.static_y)
        else:
            self.static_img.copy_(img, non_blocking=True)
        if any(inject.get(k) is not None for k in ("pos0", "hidden0", "actions")):
            TrainStep._stage_injection(self, inject)
            return self.run_static(injected=True)
        return self.run_static()

#!/usr/bin/env python
"""Benchmark of the hot path: one train iteration of the multi-agent episode
(rollout + actor-critic loss + BPTT + Adam) on synthetic images.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c4] [--impl ours|reference]

Prints ONE JSON line (rank 0).  Metric = image-episodes/s (BASELINE.json);
agent-steps/s = image-episodes/s * Na * T is reported beside it.

Default workload = BASELINE config 4: RESISC45 shape, GLOBAL batch 256 sharded over the N GPUs (strong
scaling: 256 / 128 / 64 / 32 images per GPU at N = 1 / 2 / 4 / 8; N = 1 is also the largest single-GPU
configuration, M = 4096 rows per step).  The reference's own batch-8 configuration (c2) is timed in the same
run at N = 1 and reported under ``secondary``.

* ``value``      inputs resident in HBM (pool of batches larger than L2, cycled),
                 timed with CUDA events around each step, max over ranks.
* ``e2e``        same step through the public API (Trainer.train_step) from PINNED
                 HOST buffers: H2D of the batch + labels and D2H of the loss scalars
                 inside the timed region, every step.
* ``roofline``   the dominant kernel, timed alone with CUDA events (see DESIGN.md).
* ``cpu_baseline`` the CPU oracle port (reference algorithm incl. its mask +
                 masked_select gather) on this box's host cores, bounded sample.
* ``--impl reference``: the CPU port alone, all host threads, same metric/config.
* ``--dump-outputs DIR``: after the timed steps of the headline workload, write what its last step
                 computed as float32 ``DIR/<name>.npy`` (rank 0): ``losses`` [loss, path, error, actor,
                 critic] (what Trainer.train_step returns), ``params`` and ``param_grads`` (every
                 parameter after the Adam update / the gradient it applied, concatenated in the order
                 of model.parameters()), and the rollout's ``step_preds``, ``step_log_probas``,
                 ``step_values`` and ``step_pos``.  The inputs, weights and draws are seeded, so two
                 builds run with the same arguments can be compared output for output.  Two runs of one
                 build agree on ``step_pos`` exactly and on the rest to ~1e-6 relative L2, not bit for
                 bit (c4, 20 steps, one B200 at its 1000 W power limit).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

README_ACTIONS = [[1, 0], [-1, 0], [0, 1], [0, -1]]
WORKLOADS = {
    # README.md:39-43 hyper-parameters (SURVEY section 8d)
    "c1": dict(desc="MNIST-shape 28x28, 3 agents, 5 steps, f=6, batch 32", ft="mnist", f=6, n_b=64, n_a=64, n_m=16,
               n_m_o=24, n_d=8, nl=96, nc=10, na=3, T=5, C=3, H=28, W=28, B=32, actions=README_ACTIONS),
    "c2": dict(desc="NWPU-RESISC45-shape 256x256 RGB, 16 agents, 16 steps, f=12, nb-class 45, batch 8", ft="resisc45",
               f=12, n_b=256, n_a=256, n_m=64, n_m_o=96, n_d=16, nl=384, nc=45, na=16, T=16, C=3, H=256, W=256, B=8,
               actions=README_ACTIONS),
    "c3": dict(desc="AID-shape 600x600 RGB, 16 agents, 16 steps, f=24, nb-class 30, batch 8", ft="aid", f=24, n_b=256,
               n_a=256, n_m=64, n_m_o=96, n_d=16, nl=320, nc=30, na=16, T=16, C=3, H=600, W=600, B=8,
               actions=[[3, 0], [-3, 0], [0, 3], [0, -3]]),
}
WORKLOADS["c4"] = dict(WORKLOADS["c2"], desc="RESISC45-shape 256x256 RGB, 16 agents, 16 steps, f=12, nb-class 45, GLOBAL batch 256 "
                       "sharded over the GPUs (strong scaling)", B=256, strong=True)
for _na in (16, 32, 64, 128, 256):
    WORKLOADS[f"c5_na{_na}"] = dict(WORKLOADS["c2"], desc=f"agent sweep: {_na} agents, 32 steps, 256x256, batch 8",
                                    na=_na, T=32)


def model_config(w: dict) -> dict:
    return dict(ft_extr_str=w["ft"], window_size=w["f"], hidden_size_belief=w["n_b"], hidden_size_action=w["n_a"],
                hidden_size_msg=w["n_m"], hidden_size_msg_output=w["n_m_o"], hidden_size_state=w["n_d"], state_dim=2,
                actions=w["actions"], nb_class=w["nc"], hidden_size_linear_belief=w["nl"],
                hidden_size_linear_action=w["nl"])


# ------------------------------------------------------------------------------------
# clocks sampling (B200_PROFILING.md "clocks DURING the timed region")
# ------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int) -> None:
        self.rows: list[list[str]] = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(index)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self) -> None:
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict | None:
        if self.proc is None:
            return None
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        if not sm:
            return None
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------
# CPU port (oracle) timing: cpu_baseline and --impl reference
# ------------------------------------------------------------------------------------
def cpu_port_iteration_fn(w: dict, nb: int, threads: int, device: str = "cpu"):
    """Returns a closure running ONE train iteration of the reference algorithm on
    the CPU (oracle port: rollout with the reference's mask+masked_select gather,
    loss, autograd backward, Adam).  ``device="cuda"`` runs the same eager-PyTorch
    port on the GPU (the reference's ``--cuda`` mode; SURVEY.md 8(d) like-for-like line)."""
    from oracle import marl_oracle as O

    torch.set_num_threads(threads)
    ocfg = O.OracleConfig(ft_extr=w["ft"], f=w["f"], n_b=w["n_b"], n_a=w["n_a"], n_m=w["n_m"], n_m_o=w["n_m_o"],
                          n_d=w["n_d"], nb_class=w["nc"], nl_b=w["nl"], nl_a=w["nl"], actions=w["actions"])
    params = {k: v.to(device).requires_grad_(True) for k, v in O.init_params(ocfg, seed=0).items()}
    opt = torch.optim.Adam(list(params.values()), lr=1e-4)
    g = torch.Generator().manual_seed(1234)
    img = torch.rand(nb, w["C"], w["H"], w["W"], generator=g).to(device)
    y = torch.randint(w["nc"], (nb,), generator=g).to(device)
    na, T = w["na"], w["T"]

    def one_iteration() -> float:
        pos0 = torch.stack([torch.randint(w["H"] - w["f"], (na, nb), device=device),
                            torch.randint(w["W"] - w["f"], (na, nb), device=device)], -1)
        hidden0 = [torch.randn(na, nb, n, device=device) for n in (ocfg.n_b, ocfg.n_b, ocfg.n_a, ocfg.n_a)]
        ro = O.rollout(params, ocfg, img, pos0, hidden0, None, T, faithful_gather=True)
        parts = O.a2c_loss(ro.step_preds, ro.step_log_probas, ro.step_values, y, 0.99)
        opt.zero_grad()
        parts.loss.backward()
        opt.step()
        return float(parts.loss.detach())

    return one_iteration


def time_cpu_port(w: dict, nb: int, budget_s: float, max_iters: int, warmup: int = 1, device: str = "cpu",
                  exact_iters: bool = False):
    """Seconds per iteration of the port at batch `nb`.  ``exact_iters``: run exactly `max_iters` timed
    iterations (the --impl reference arm: the requested step count is never shortened)."""
    threads = os.cpu_count() or 1
    fn = cpu_port_iteration_fn(w, nb, threads, device)  # float(loss) at the end of fn synchronises
    t0 = time.perf_counter()
    for _ in range(warmup):
        fn()
    t_first = (time.perf_counter() - t0) / max(1, warmup)
    iters = max_iters if exact_iters else max(1, min(max_iters, int(budget_s / max(t_first, 1e-6))))
    t0 = time.perf_counter()
    for _ in range(iters):
        fn()
    dt = (time.perf_counter() - t0) / iters
    return dt, iters, threads


def cpu_sample_batch(w: dict, steps: int, budget_s: float) -> int:
    """Images per CPU iteration: the workload's batch when `steps` iterations of it fit the budget, else a
    bounded sample of its images (episodes of different images are independent: image-episodes/s of the
    port does not depend on the batch beyond threading efficiency).  ~0.25 s per image-episode at the
    RESISC45 shape on 16 cores (measured, round 1)."""
    per_image = 0.25 * (w["H"] * w["W"]) / (256 * 256) * (w["na"] * w["T"]) / 256.0
    nb = w["B"]
    while nb > 1 and nb * per_image * max(1, steps) > budget_s:
        nb //= 2
    return max(1, nb)


# ------------------------------------------------------------------------------------
def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--workload", default="c4", choices=sorted(WORKLOADS))
    ap.add_argument("--no-secondary", action="store_true", help="skip the c2 (batch 8) secondary measurement at N=1")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--fp32", action="store_true", help="exact-fp32 FFMA GEMMs instead of the tensor cores")
    ap.add_argument("--precision", default="tf32x3", choices=["tf32x3", "tf32"],
                    help="tensor-core arithmetic: error-compensated 3xTF32 (default, fp32-class parity) or plain TF32")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-roofline", action="store_true", help="skip the micro-benchmarks (profiling runs)")
    ap.add_argument("--cpu-budget", type=float, default=15.0, help="seconds of CPU work for cpu_baseline")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU arm (--impl ours)")
    args.warmup = max(3, args.warmup)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    w = WORKLOADS[args.workload]
    strong = bool(w.get("strong"))
    nb = w["B"] // world if strong else w["B"]
    global_batch = nb * world
    # `config` describes the WORKLOAD and is identical in both arms (the driver compares them); everything
    # that describes how one arm ran it lives in `run`
    cfg_out = {"workload": f"{args.workload}: {w['desc']}", "agents": w["na"], "steps_per_episode": w["T"],
               "window": w["f"], "image": [w["C"], w["H"], w["W"]], "classes": w["nc"],
               "global_batch": w["B"] * (1 if strong else world), "parallelism": f"dp{world}",
               "l2": "inputs cycle through a pool of distinct batches larger than L2 (GPU arm; see run.l2)"}

    if args.impl == "reference":
        if rank != 0:
            return
        warm = min(args.warmup, 1)
        nb_cpu = cpu_sample_batch(w, args.steps + warm, budget_s=170.0)
        dt, iters, threads = time_cpu_port(w, nb_cpu, budget_s=170.0, max_iters=args.steps, warmup=warm, exact_iters=True)
        val = nb_cpu / dt
        sample = (f"{iters} full train iterations (rollout+loss+backward+Adam) of the reference algorithm on "
                  f"{nb_cpu} of the workload's {w['B']} images per iteration, after {warm} warm-up")
        line = {"impl": "reference", "metric": "image_episodes_per_sec", "value": val, "unit": "image-episodes/s",
                "agent_steps_per_sec": val * w["na"] * w["T"], "n_gpus": args.gpus, "steps": iters,
                "steps_requested": args.steps, "warmup": warm, "ms_per_step": dt * 1e3, "higher_is_better": True,
                "scaling": "strong" if strong else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": cfg_out,
                "run": {"arm": "cpu", "batch_per_iteration": nb_cpu, "threads": threads},
                "cpu_baseline": {"value": val, "unit": "image-episodes/s", "cores": threads, "kind": "port",
                                 "sample": sample},
                "e2e": {"value": val, "unit": "image-episodes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        if torch.cuda.is_available():  # the same eager-PyTorch port on the GPU: the like-for-like line (SURVEY 8d)
            try:
                dtg, itg, _ = time_cpu_port(w, nb_cpu, budget_s=8.0, max_iters=20, warmup=2, device="cuda:0")
                line["cpu_baseline"]["eager_gpu_port"] = {
                    "value": nb_cpu / dtg, "unit": "image-episodes/s",
                    "sample": f"{itg} iterations of the same port with device=cuda (eager PyTorch, ~10^4 launches/iteration), "
                              f"batch {nb_cpu}"}
            except Exception as exc:
                line["cpu_baseline"]["eager_gpu_port"] = {"error": repr(exc)[:200]}
        print(json.dumps(line))
        return

    # ---------------- ours ----------------
    import torch.distributed as dist

    from marlclassification_b200.parallel import DataParallelContext

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    dp = DataParallelContext()

    clocks = ClockSampler(local_rank) if rank == 0 else None
    res = measure(w, nb, args, dp, dev, world, rank, args.steps, args.warmup,
                  dump_dir=args.dump_outputs if rank == 0 else None)
    clk = clocks.stop() if clocks else None
    global_batch = nb * world
    if rank == 0:
        val = global_batch / (res["step_ms"] * 1e-3)
        line = {"metric": "image_episodes_per_sec", "value": val, "unit": "image-episodes/s",
                "agent_steps_per_sec": val * w["na"] * w["T"], "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": res["step_ms"], "higher_is_better": True,
                "scaling": "strong" if strong else "weak", "vs_baseline": None,
                "dtype": "f32" if args.fp32 else args.precision, "data": "synthetic", "config": cfg_out,
                "run": {"arm": "gpu", "batch_per_gpu": nb, "rows_per_step_per_gpu": nb * w["na"], "l2": res["l2"],
                        "cuda_graph": not args.no_graph, "nccl_in_graph": res["nccl_in_graph"]},
                "e2e": e2e_block(res, global_batch),
                "eval": {"value": global_batch / (res["eval_ms"] * 1e-3), "unit": "image-episodes/s",
                         "ms_per_step": res["eval_ms"],
                         "what": "forward-only episode + agent-mean vote (Trainer.eval_step), inputs in HBM"},
                "gpu_launches": res["launches"] * args.steps, "gpu_launches_per_step": res["launches"], "clocks": clk}
        if not args.no_roofline:
            try:
                from bench_roofline import roofline_for

                line["roofline"] = roofline_for(res["model"], w, nb, dev)
            except Exception as exc:  # keep the headline even if the micro-benchmark breaks
                line["roofline"] = {"error": repr(exc)}
    del res
    torch.cuda.empty_cache()
    if world == 1 and not args.no_secondary and args.workload != "c2":
        # the reference's own configuration (README hyper-parameters, batch 8: 128 rows per step, latency-bound)
        w2 = WORKLOADS["c2"]
        r2 = measure(w2, w2["B"], args, dp, dev, world, rank, args.steps, args.warmup)
        v2 = w2["B"] / (r2["step_ms"] * 1e-3)
        line["secondary"] = {"c2": {"workload": f"c2: {w2['desc']}", "value": v2, "unit": "image-episodes/s",
                                    "agent_steps_per_sec": v2 * w2["na"] * w2["T"], "ms_per_step": r2["step_ms"],
                                    "e2e": e2e_block(r2, w2["B"]),
                                    "eval": {"value": w2["B"] / (r2["eval_ms"] * 1e-3), "ms_per_step": r2["eval_ms"]},
                                    "gpu_launches_per_step": r2["launches"]}}
        del r2
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            nb_cpu = min(w["B"], 8)  # bounded sample: the reference's own batch size out of the workload's images
            dt, iters, threads = time_cpu_port(w, nb_cpu, budget_s=args.cpu_budget, max_iters=20)
            line["cpu_baseline"] = {"value": nb_cpu / dt, "unit": "image-episodes/s", "cores": threads, "kind": "port",
                                    "sample": f"{iters} full train iterations of the reference algorithm (CPU oracle port) on "
                                              f"{nb_cpu} of the workload's {w['B']} images per iteration, after 1 warm-up"}
            try:  # the same eager-PyTorch port on the GPU itself (the reference's --cuda mode)
                dtg, itg, _ = time_cpu_port(w, nb_cpu, budget_s=5.0, max_iters=20, warmup=2, device=str(dev))
                line["cpu_baseline"]["eager_gpu_port"] = {"value": nb_cpu / dtg, "unit": "image-episodes/s",
                                                          "sample": f"{itg} iterations of the oracle port run with "
                                                                    f"device=cuda (eager PyTorch, ~10^4 launches/iteration), batch {nb_cpu}"}
            except Exception as exc:
                line["cpu_baseline"]["eager_gpu_port"] = {"error": repr(exc)[:200]}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def e2e_block(res: dict, global_batch: int) -> dict:
    return {"value": global_batch / (res["e2e_ms"] * 1e-3), "unit": "image-episodes/s", "ms_per_step": res["e2e_ms"],
            "h2d_bytes_per_step": res["batch_bytes"] + res["nb"] * 8, "d2h_bytes_per_step": 20,
            "input": "pinned host f32[B,C,H,W] + i64[B] labels, copied one batch ahead on a copy stream",
            "u8_input": {"value": global_batch / (res["e2e_u8_ms"] * 1e-3), "ms_per_step": res["e2e_u8_ms"],
                         "h2d_bytes_per_step": res["batch_bytes"] // 4 + res["nb"] * 8,
                         "input": "pinned host u8[B,H,W,C] (decoded image bytes), ToTensor on the device"}}


DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir: str, loss_out: torch.Tensor, model, eng) -> None:
    """Write one train step's outputs (names in the module docstring) as float32 DIR/<name>.npy."""
    import numpy as np

    flat_p, flat_g = model.flat_params, model.flat_grads
    spans = [((p.data_ptr() - flat_p.data_ptr()) // 4, p.numel()) for p in model.parameters()]
    arrays = {"losses": loss_out[:5],
              "params": torch.cat([flat_p[o:o + n] for o, n in spans]),
              "param_grads": torch.cat([flat_g[o:o + n] for o, n in spans]),
              "step_preds": eng.step_preds, "step_log_probas": eng.step_log_probas, "step_values": eng.step_values,
              "step_pos": eng.step_pos}
    arrays = {k: v.detach().to("cpu", torch.float32).numpy() for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes of outputs exceed the {DUMP_MAX_BYTES}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, f"{k}.npy"), a)


def measure(w: dict, nb: int, args, dp, dev, world: int, rank: int, steps: int, warmup: int,
            dump_dir: str | None = None) -> dict:
    """Time one workload at `nb` images per GPU: device-resident `value`, `e2e` from pinned host batches
    (fp32 and uint8), forward-only `eval`.  Every figure is the max over ranks.  `dump_dir`: write the
    outputs of the last step of the `value` window there (see dump_outputs)."""
    import torch.distributed as dist

    from marlclassification_b200.config import ModelConfig
    from marlclassification_b200.core import EpisodeSampler
    from marlclassification_b200.training import Trainer

    torch.manual_seed(0)
    model, marl, env = ModelConfig(**model_config(w)).build_marl(w["na"])
    model.use_tc = not args.fp32
    model.precision = args.precision
    model.to(dev)
    dp.broadcast_params(model.flat_params)
    sampler = EpisodeSampler(marl, env, w["T"], gamma=0.99)
    trainer = Trainer(model, w["nc"], 1e-4, 0.99, dp=dp, cuda_graph=not args.no_graph)

    # synthetic data: a pool of distinct batches larger than L2 (126 MB), cycled
    g = torch.Generator().manual_seed(1234 + rank)
    batch_bytes = nb * w["C"] * w["H"] * w["W"] * 4
    pool_n = max(4, min(64, int(160e6 // batch_bytes) + 1))
    host_pool = [torch.rand(nb, w["C"], w["H"], w["W"], generator=g).pin_memory() for _ in range(pool_n)]
    host_y = [torch.randint(w["nc"], (nb,), generator=g).pin_memory() for _ in range(pool_n)]
    dev_pool = [t.to(dev) for t in host_pool]
    dev_y = [t.to(dev) for t in host_y]
    l2 = (f"inputs cycle through a pool of {pool_n} distinct batches = {pool_n * batch_bytes / 1e6:.0f} MB"
          + (" (> 126 MB L2)" if pool_n * batch_bytes > 126e6 else " (< L2: pool capped at 64 batches)"))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def run(pool, ys, n):
        """Time `n` steps with CUDA events on the current stream; returns (device ms, wall ms, the
        last step's loss tensor)."""
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
        t_wall = time.perf_counter()
        for i in range(n):
            evs[i][0].record()
            out = trainer.train_step(pool[i % len(pool)], ys[i % len(pool)], sampler)
            evs[i][1].record()
        torch.cuda.synchronize()
        wall = (time.perf_counter() - t_wall) * 1e3
        return sum(a.elapsed_time(b) for a, b in evs), wall, out

    def run_eval(pool, n):
        """Forward-only episodes (Trainer.eval_step, the eval_epoch path), inputs resident."""
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_wall = time.perf_counter()
        a.record()
        for i in range(n):
            trainer.eval_step(pool[i % len(pool)], sampler)
        b.record()
        torch.cuda.synchronize()
        return max(a.elapsed_time(b), (time.perf_counter() - t_wall) * 1e3) / n

    def run_e2e(pool, ys, n):
        """The public API end to end: Trainer.prefetch (copy stream, one batch ahead) feeding
        Trainer.train_step from PINNED HOST batches, the step's five loss scalars read back every
        step.  Every step's H2D copy and D2H read happen inside the timed region."""
        batches = [(pool[i % len(pool)], ys[i % len(pool)]) for i in range(n)]
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_wall = time.perf_counter()
        a.record()
        for staged in trainer.prefetch(batches):
            out = trainer.train_step(staged, None, sampler)
            scal = out[:5].to("cpu", non_blocking=False)  # D2H of the step's result (implies a sync)
            assert scal.numel() == 5
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b), (time.perf_counter() - t_wall) * 1e3

    # warm-up (also captures the CUDA graphs: 2 eager steps, then capture)
    run(dev_pool, dev_y, max(3, warmup))
    barrier()
    dev_ms, wall_ms, loss_out = run(dev_pool, dev_y, steps)
    barrier()
    if dump_dir:
        dump_outputs(dump_dir, loss_out, model, sampler.engine_for(dev_pool[0], gamma=0.99))
    # the step stream is saturated only if the host keeps ahead; report the slower of
    # device-event time and wall time so host-bound runs are not flattered
    step_ms = max(dev_ms, wall_ms) / steps
    # e2e: pinned host inputs (fp32 NCHW, what the reference's DataLoader yields), loss read back
    run_e2e(host_pool, host_y, 3)
    barrier()
    e2e_dev_ms, e2e_wall_ms = run_e2e(host_pool, host_y, steps)
    barrier()
    e2e_ms = max(e2e_dev_ms, e2e_wall_ms) / steps
    # same, from uint8 HWC host batches (decoded images before ToTensor): 4x fewer PCIe bytes,
    # converted on the device by marlc_images_u8_to_f32
    u8_pool = [(t.permute(0, 2, 3, 1) * 255).round().to(torch.uint8).contiguous().pin_memory() for t in host_pool]
    run_e2e(u8_pool, host_y, 3)
    barrier()
    u8_dev_ms, u8_wall_ms = run_e2e(u8_pool, host_y, steps)
    barrier()
    e2e_u8_ms = max(u8_dev_ms, u8_wall_ms) / steps
    run_eval(dev_pool, 4)
    barrier()
    eval_ms = run_eval(dev_pool, steps)
    barrier()

    t = torch.tensor([step_ms, e2e_ms, e2e_u8_ms, eval_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    step_ms, e2e_ms, e2e_u8_ms, eval_ms = t.tolist()
    eng = sampler.engine_for(dev_pool[0], gamma=0.99)
    launches = eng.launches["forward"] + eng.launches["loss"] + eng.launches["backward"] + 2
    step_objs = list(trainer._Trainer__steps.values())
    return {"step_ms": step_ms, "e2e_ms": e2e_ms, "e2e_u8_ms": e2e_u8_ms, "eval_ms": eval_ms, "launches": launches,
            "batch_bytes": batch_bytes, "nb": nb, "l2": l2, "model": model,
            "nccl_in_graph": bool(step_objs and step_objs[0].nccl_in_graph)}


if __name__ == "__main__":
    main()

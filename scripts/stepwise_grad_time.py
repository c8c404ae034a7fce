"""Cost of training through the step-wise API (model.differentiable_steps = True) against the fused episode.

One training iteration each way, on the same model and batch:
  * step API:  T x (MultiAgent.act, Environment.step), the A2C loss of the stacked outputs (oracle formula, torch
    ops), loss.backward() (one marlc_model_step_backward per step), fused Adam;
  * fused:     Trainer.train_step (rollout, fused loss, BPTT, Adam; one CUDA graph).
Wall time per iteration from a host clock around work that ends in a device synchronise, after warm-up.
Prints one JSON line with the card's name and power limit.

    python scripts/stepwise_grad_time.py [--workloads c1 c2] [--iters 20] [--warmup 3]
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from bench import WORKLOADS, model_config  # noqa: E402
from marlclassification_b200.config import ModelConfig  # noqa: E402
from marlclassification_b200.core import EpisodeSampler  # noqa: E402
from marlclassification_b200.training import Trainer  # noqa: E402
from marlclassification_b200.training.optim import FlatAdam  # noqa: E402
from oracle import marl_oracle as O  # noqa: E402


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    name, _, limit = q.stdout.strip().splitlines()[0].partition(",") if q.returncode == 0 else ("?", "", "?")
    return {"gpu": name.strip() or torch.cuda.get_device_name(0), "power_limit": limit.strip()}


def timed(fn, iters: int, warmup: int) -> float:
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(iters):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / iters * 1e3


def measure(wl: str, iters: int, warmup: int) -> dict:
    w = WORKLOADS[wl]
    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    model, marl, env = ModelConfig(**model_config(w)).build_marl(w["na"])
    model.to(dev)
    img = torch.rand(w["B"], w["C"], w["H"], w["W"], device=dev)
    y = torch.randint(w["nc"], (w["B"],), device=dev)

    model.differentiable_steps = True
    opt = FlatAdam(model, 1e-4)

    def stepwise():
        obs = env.reset(img, w["na"])
        marl.reset(w["B"])
        preds, logps, vals = [], [], []
        for _ in range(w["T"]):
            out = marl.act(obs, env.normalized_positions)
            obs = env.step(out.actions)
            preds.append(out.predictions)
            logps.append(out.actions_log_probs)
            vals.append(out.values)
        opt.zero_grad()
        O.a2c_loss(torch.stack(preds), torch.stack(logps), torch.stack(vals), y, 0.99).loss.backward()
        opt.step()

    ms_step = timed(stepwise, iters, warmup)
    model.differentiable_steps = False
    trainer = Trainer(model, w["nc"], 1e-4, 0.99)
    sampler = EpisodeSampler(marl, env, w["T"], gamma=0.99)
    ms_fused = timed(lambda: trainer.train_step(img, y, sampler), iters, warmup)
    return {"workload": wl, "desc": w["desc"], "stepwise_ms": round(ms_step, 3), "train_step_ms": round(ms_fused, 3),
            "ratio": round(ms_step / ms_fused, 2)}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", nargs="+", default=["c1", "c2"])
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    res = {**card(), "results": [measure(wl, args.iters, args.warmup) for wl in args.workloads]}
    print(json.dumps(res))


if __name__ == "__main__":
    main()

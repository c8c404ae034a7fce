"""Time of the image gradient (EpisodeEngine.image_grad, marlc_episode_image_grad) against the episode backward.

At each workload's per-GPU geometry: one rollout, the fused loss and the episode backward, then
  * image_grad: CUDA events around --reps back-to-back calls, after --warmup calls;
  * backward:   CUDA events around --bwd-reps episode backwards, after one warm-up.
The algorithmic bytes are the first layer's conv-output gradients read (T*M windows x ho^2 x cout floats) plus the
image gradient written (nb x C x H x W floats); the achieved rate is divided by the data-sheet 7.7 TB/s of one B200.
When those bytes fit the 126 MB L2 the repeated calls are served from it ("l2_resident"), so the rate is not an
HBM rate.  Prints one JSON line with the card's name and power limit, read in the same run.

    python scripts/image_grad_time.py [--workloads c2 c4] [--reps 300] [--warmup 20] [--bwd-reps 20]
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from bench import WORKLOADS, model_config  # noqa: E402
from marlclassification_b200.config import ModelConfig  # noqa: E402
from marlclassification_b200.core import EpisodeSampler  # noqa: E402
from scripts.stepwise_grad_time import card  # noqa: E402

HBM_BYTES_PER_S = 7.7e12  # NVIDIA HGX B200 data sheet, one GPU
L2_BYTES = 126e6


def events_ms(fn, reps: int) -> float:
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(reps):
        fn()
    end.record()
    torch.cuda.synchronize()
    return start.elapsed_time(end) / reps


def measure(wl: str, reps: int, warmup: int, bwd_reps: int) -> dict:
    w = WORKLOADS[wl]
    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    model, marl, env = ModelConfig(**model_config(w)).build_marl(w["na"])
    model.to(dev)
    img = torch.rand(w["B"], w["C"], w["H"], w["W"], device=dev)
    y = torch.randint(w["nc"], (w["B"],), device=dev)
    eng = EpisodeSampler(marl, env, w["T"], gamma=0.99).engine_for(img)
    eng.forward(img)
    eng.loss(y)
    eng.backward(img)
    out = torch.empty_like(img)
    for _ in range(warmup):
        eng.image_grad(out)
    ms_img = events_ms(lambda: eng.image_grad(out), reps)
    ms_bwd = events_ms(lambda: eng.backward(img), bwd_reps)
    f, layers, _, _ = model.feature_extractor.cnn_spec
    ho, cout = (f - 1) // 2 + 1, layers[0][1]
    nbytes = 4 * (w["T"] * w["na"] * w["B"] * ho * ho * cout + w["B"] * w["C"] * w["H"] * w["W"])
    return {"workload": wl, "geometry": dict(na=w["na"], nb=w["B"], T=w["T"], C=w["C"], H=w["H"], W=w["W"], f=f),
            "windows_per_image": w["T"] * w["na"], "image_grad_us": round(ms_img * 1e3, 2),
            "bytes": nbytes, "l2_resident": nbytes < L2_BYTES,
            "hbm_fraction": round(nbytes / (ms_img * 1e-3) / HBM_BYTES_PER_S, 3),
            "episode_backward_ms": round(ms_bwd, 3), "ratio_to_backward": round(ms_img / ms_bwd, 4)}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", nargs="+", default=["c2", "c4"])
    ap.add_argument("--reps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--bwd-reps", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    res = {**card(), "results": [measure(wl, args.reps, args.warmup, args.bwd_reps) for wl in args.workloads]}
    print(json.dumps(res))


if __name__ == "__main__":
    main()

"""Cost of the input gradients of the step-wise API (Environment.observe's backward, model.differentiable_step_inputs).

At each workload's per-GPU geometry:
  * marlc_patch_gather_backward: CUDA events around --reps back-to-back calls on random d_obs / positions, after
    --warmup calls.  Algorithmic bytes: d_obs and the positions read, d_img written (nb x C x H x W floats, mostly
    zeros); the rate is divided by the data-sheet 7.7 TB/s of one B200.  The repeated calls are served from L2 when
    those bytes fit its 126 MB ("l2_resident"), so the rate is then not an HBM rate;
  * marlc_model_step_input_grad (d img_patch and d norm_pos) after one marlc_model_step_backward at M = na * nb,
    and that step backward itself (CUDA events, --bwd-reps calls);
  * one step-wise episode (T x (MultiAgent.act, Environment.step), the A2C loss, backward()) over an image that
    requires grad, against the same episode over a plain image: host clock around work that ends in a device
    synchronise, after warm-up.
Prints one JSON line with the card's name and power limit, read in the same run.

    python scripts/step_input_grad_time.py [--workloads c2 c4] [--reps 300] [--warmup 20] [--bwd-reps 20]
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from bench import WORKLOADS, model_config  # noqa: E402
from marlclassification_b200 import _lib  # noqa: E402
from marlclassification_b200.config import ModelConfig  # noqa: E402
from marlclassification_b200.networks.models import RecurrentOutput  # noqa: E402
from oracle import marl_oracle as O  # noqa: E402
from scripts.image_grad_time import HBM_BYTES_PER_S, L2_BYTES, events_ms  # noqa: E402
from scripts.stepwise_grad_time import card, timed  # noqa: E402


def measure(wl: str, reps: int, warmup: int, bwd_reps: int, episodes: int) -> dict:
    w = WORKLOADS[wl]
    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    na, nb, C, H, W, f = w["na"], w["B"], w["C"], w["H"], w["W"], w["f"]
    model, marl, env = ModelConfig(**model_config(w)).build_marl(na)
    model.to(dev)
    model.differentiable_steps = True
    stream = _lib.stream_ptr(dev)

    # ---- the gather adjoint
    d_obs = torch.randn(na, nb, C, f, f, device=dev)
    pos = torch.stack([torch.randint(H - f, (na, nb), device=dev), torch.randint(W - f, (na, nb), device=dev)], -1)
    d_img = torch.empty(nb, C, H, W, device=dev)

    def gather_bwd():
        _lib.check(_lib.lib().marlc_patch_gather_backward(d_obs.data_ptr(), pos.data_ptr(), d_img.data_ptr(), na, nb,
                                                          C, H, W, f, stream))

    for _ in range(warmup):
        gather_bwd()
    ms_gather = events_ms(gather_bwd, reps)
    g_read = 4 * d_obs.numel() + 8 * pos.numel()
    g_bytes = g_read + 4 * d_img.numel()

    # ---- the step's input gradients, after one step backward
    dims = model.dims
    patch = torch.rand(na, nb, C, f, f, device=dev)
    msg = torch.randn(na, nb, dims["n_m"], device=dev)
    npos = torch.rand(na, nb, 2, device=dev)
    hid = [torch.randn(na, nb, n, device=dev) for n in (dims["n_b"], dims["n_b"], dims["n_a"], dims["n_a"])]
    with torch.no_grad():
        model(patch, msg, npos, RecurrentOutput(*hid))
    eng = next(e for e in model._engines.values() if e.T == 1)
    d_out = [torch.randn(na, nb, n, device=dev) for n in (dims["nb_action"],)] + [torch.randn(na, nb, device=dev)] + \
        [torch.randn(na, nb, n, device=dev) for n in (dims["nb_class"], dims["n_m"], dims["n_b"], dims["n_b"],
                                                      dims["n_a"], dims["n_a"])]
    grads = torch.empty_like(model.flat_params)

    def step_bwd():
        eng.model_step_backward(patch, msg, npos, hid, d_out, [None] * 5, grads)

    d_patch, d_npos = torch.empty_like(patch), torch.empty_like(npos)
    step_bwd()
    for _ in range(warmup):
        eng.step_input_grad(d_patch, d_npos)
    ms_input = events_ms(lambda: eng.step_input_grad(d_patch, d_npos), reps)
    step_bwd()
    ms_step_bwd = events_ms(step_bwd, bwd_reps)

    # ---- one step-wise episode, with and without the image gradient
    img = torch.rand(nb, C, H, W, device=dev)
    y = torch.randint(w["nc"], (nb,), device=dev)

    def episode(x):
        obs = env.reset(x, na)
        marl.reset(nb)
        preds, logps, vals = [], [], []
        for _ in range(w["T"]):
            out = marl.act(obs, env.normalized_positions)
            obs = env.step(out.actions)
            preds.append(out.predictions)
            logps.append(out.actions_log_probs)
            vals.append(out.values)
        model.zero_grad(set_to_none=False)
        O.a2c_loss(torch.stack(preds), torch.stack(logps), torch.stack(vals), y, 0.99).loss.backward()

    model.differentiable_step_inputs = False
    ms_plain = timed(lambda: episode(img), episodes, 2)
    model.differentiable_step_inputs = True
    x = img.clone().requires_grad_(True)

    def with_grad():
        x.grad = None
        episode(x)

    ms_img = timed(with_grad, episodes, 2)
    return {"workload": wl, "geometry": dict(na=na, nb=nb, C=C, H=H, W=W, f=f, T=w["T"]),
            "patch_gather_backward_us": round(ms_gather * 1e3, 2), "gather_bytes_read": g_read,
            "gather_bytes": g_bytes, "l2_resident": g_bytes < L2_BYTES,
            "gather_hbm_fraction": round(g_bytes / (ms_gather * 1e-3) / HBM_BYTES_PER_S, 3),
            "step_input_grad_us": round(ms_input * 1e3, 2), "model_step_backward_ms": round(ms_step_bwd, 3),
            "input_grad_ratio_to_step_backward": round(ms_input / ms_step_bwd, 4),
            "episode_plain_ms": round(ms_plain, 3), "episode_image_grad_ms": round(ms_img, 3),
            "episode_ratio": round(ms_img / ms_plain, 3)}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", nargs="+", default=["c2", "c4"])
    ap.add_argument("--reps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--bwd-reps", type=int, default=20)
    ap.add_argument("--episodes", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    res = {**card(), "results": [measure(wl, args.reps, args.warmup, args.bwd_reps, args.episodes)
                                 for wl in args.workloads]}
    print(json.dumps(res))


if __name__ == "__main__":
    main()

"""Cost of training the stand-alone feature extractor (VisionCnnModule.forward in grad mode + backward:
marlc_cnn_forward_save / marlc_cnn_backward) beside eager torch modules (Conv2d / GroupNorm / SiLU, cuDNN) holding
the same weights, on the same GPU.

For Resisc45Cnn at f = 12 and AidCnn at f = 24, at --windows windows each: one step is forward, a random-cotangent
backward into the windows and every parameter.  Host clock around --iters steps that end in a device synchronise,
after --warmup steps; the gradients of both sides are compared norm-wise so the two time the same work.  The
result is reported, not a gate.  Prints one JSON line with the card's name and power limit, read in the same run.

    python scripts/cnn_grad_time.py [--windows 4096 65536] [--iters 20] [--warmup 5]
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from marlclassification_b200.networks import vision  # noqa: E402
from marlclassification_b200.networks.blocks import init_layers  # noqa: E402
from scripts.stepwise_grad_time import card, timed  # noqa: E402

NETS = {"resisc45_f12": ("Resisc45Cnn", 12), "aid_f24": ("AidCnn", 24)}


def torch_twin(m) -> torch.nn.Sequential:
    """Eager torch modules with the weights of the feature extractor m."""
    convs = [c for c in m.modules() if isinstance(c, torch.nn.Conv2d)]
    norms = [g for g in m.modules() if isinstance(g, torch.nn.GroupNorm)]
    mods = []
    for c, g in zip(convs, norms):
        mods += [torch.nn.Conv2d(c.in_channels, c.out_channels, 3, 2, 1), torch.nn.GroupNorm(g.num_groups, g.num_channels),
                 torch.nn.SiLU()]
    twin = torch.nn.Sequential(*mods, torch.nn.Flatten(1)).to(next(m.parameters()).device)
    with torch.no_grad():
        for a, b in zip(twin.parameters(), m.parameters()):
            a.copy_(b)
    return twin


def measure(name: str, n: int, iters: int, warmup: int) -> dict:
    cls, f = NETS[name]
    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    m = getattr(vision, cls)(f)
    m.apply(init_layers)
    m.to(dev)
    twin = torch_twin(m)
    x = torch.rand(n, 3, f, f, device=dev, requires_grad=True)
    d_out = torch.randn(n, m.out_size, device=dev)

    def step(module):
        def fn():
            x.grad = None
            module.zero_grad(set_to_none=True)
            module(x).backward(d_out)
        return fn

    ours, eager = step(m), step(twin)
    ours()
    g_ours = [x.grad.clone()] + [p.grad.clone() for p in m.parameters()]
    eager()
    g_eager = [x.grad.clone()] + [p.grad.clone() for p in twin.parameters()]
    diff = max(((a - b).norm() / b.norm().clamp_min(1e-30)).item() for a, b in zip(g_ours, g_eager))
    t_ours = timed(ours, iters, warmup)
    t_eager = timed(eager, iters, warmup)
    t_ours2 = timed(ours, iters, 0)  # alternated: a drift of the card shows as a difference between the two runs
    return {"net": name, "windows": n, "cnn_fwd_bwd_ms": round(min(t_ours, t_ours2), 3),
            "cnn_fwd_bwd_ms_runs": [round(t_ours, 3), round(t_ours2, 3)], "torch_eager_ms": round(t_eager, 3),
            "ratio_to_eager": round(min(t_ours, t_ours2) / t_eager, 3), "max_grad_rel_diff": float(f"{diff:.2e}")}


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--windows", type=int, nargs="+", default=[4096, 65536])
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("cnn_grad_time.py: needs a CUDA device")
    results = [measure(name, n, args.iters, args.warmup) for name in NETS for n in args.windows]
    print(json.dumps({**card(), "results": results}))


if __name__ == "__main__":
    main()

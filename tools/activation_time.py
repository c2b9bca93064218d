"""Sampling throughput of the config-2 model (image-conditional RayNetwork + SetTransformer L6, C = 384, I = 64, 8 heads,
GaussianReparam, ConvNeXt-T conditioner, seeded random weights) with each MLP activation the engine supports: the
normalised Gaussian (the reference configurations'), the raw Gaussian and ReLU (the SetTransformer default).
Usage: python tools/activation_time.py [--activations gaussian,gaussian_raw,relu] [--clouds 64] [--points 2048]
                                       [--steps 64] [--reps 3]

Per activation: one warm-up call of Diffusion.sample_stochastic on the batch (captures the sampler's CUDA graph), then
--reps calls timed with CUDA events; ms per call (best) and clouds/s.  Then one profiled denoiser evaluation lists the
engine's kernel classes (launches, ms).  The card name and its power limit are read in the same run.  Writes nothing into
the tree.
"""
from __future__ import annotations

import argparse
import functools
import json
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

from chamfer_time import _events_ms, card_info  # noqa: E402
from width_time import CFG2  # noqa: E402


def build(activation: str, device):
    import gecco_b200 as G
    from gecco_b200.models import ConvNeXtExtractor, GaussianActivation, RayNetwork, SetTransformer
    from gecco_b200.reparam import GaussianReparam

    act = torch.nn.ReLU if activation == "relu" else functools.partial(GaussianActivation,
                                                                         normalized=activation == "gaussian")
    torch.manual_seed(0)
    rp = GaussianReparam(torch.tensor(CFG2["mean"]), torch.tensor(CFG2["sigma"]))
    st = SetTransformer(n_layers=6, num_inducers=64, feature_dim=384, t_embed_dim=1, num_heads=8, activation=act)
    net = RayNetwork(backbone=st, reparam=rp, context_dims=(96, 192, 384))
    model = G.Diffusion(backbone=G.EDMPrecond(model=net), conditioner=ConvNeXtExtractor(pretrained=False), reparam=rp,
                        loss=G.EDMLoss(schedule=G.LogUniformSchedule(max=CFG2["sigma_max"])))
    return model.to(device).eval()


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--activations", default="gaussian,gaussian_raw,relu")
    ap.add_argument("--clouds", type=int, default=64)
    ap.add_argument("--points", type=int, default=2048)
    ap.add_argument("--steps", type=int, default=64)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("activation_time.py measures on the GPU; no CUDA device is visible")

    import gecco_b200 as G
    from gecco_b200 import engine as E

    dev = torch.device("cuda:0")
    B, N = args.clouds, args.points
    card = card_info()
    print(json.dumps({"card": card}))
    rows = []
    for activation in args.activations.split(","):
        model = build(activation, dev)
        K = torch.tensor(CFG2["K"]).expand(B, 3, 3).contiguous().to(dev)
        img = torch.rand(B, 3, CFG2["image"], CFG2["image"], generator=torch.Generator().manual_seed(1)).to(dev)
        ctx = G.Context3d(image=img, K=K)
        rng = torch.Generator(dev).manual_seed(42)
        call = lambda: model.sample_stochastic((B, N, 3), ctx, rng=rng, num_steps=args.steps)
        with torch.no_grad():
            out = call()
            assert torch.isfinite(out).all(), activation
            ms = _events_ms(call, args.reps)
            # kernel classes of one evaluation (profiling runs eagerly, outside the timed calls)
            x = torch.randn(B, N, 3, device=dev)
            sig = torch.full((B,), 2.0, device=dev)
            model(x, sig, ctx)
            torch.cuda.synchronize()
            E.profile_start()
            model(x, sig, ctx)
            classes = {p["name"]: (p["launches"], round(p["ms"], 3)) for p in E.profile_stop()}
        best = min(ms)
        row = dict(activation=activation, clouds=B, points=N, steps=args.steps, ms_per_call=ms,
                   clouds_per_s=B / (best * 1e-3), classes_one_eval=classes)
        rows.append(row)
        print(json.dumps(row))
        del model
        torch.cuda.empty_cache()
    print(f"{card}")
    print("| activation | ms per call (best of {}) | clouds/s |".format(args.reps))
    print("|---|---|---|")
    for r in rows:
        print(f"| {r['activation']} | {min(r['ms_per_call']):.0f} | {r['clouds_per_s']:.2f} |")


if __name__ == "__main__":
    main()

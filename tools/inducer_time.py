"""Sampling throughput of the config-2 model (image-conditional RayNetwork + SetTransformer L6, C = 384, 8 heads,
GaussianReparam, ConvNeXt-T conditioner, seeded random weights) at several inducer counts.
Usage: python tools/inducer_time.py [--inducers 64,128,192,256] [--clouds 64] [--points 2048] [--steps 64] [--reps 2]

Per count I: one warm-up call of Diffusion.sample_stochastic on the batch (captures the sampler's CUDA graph), then
--reps calls timed with CUDA events; clouds/s, the dense FLOPs of one network evaluation per cloud
(training.flops_per_cloud(points, inducers=I)), the achieved rate over the 2 * steps - 1 evaluations of a call, and its
share of the B200 data-sheet dense BF16 rate (2250 TFLOP/s at 1000 W).  Then one profiled denoiser evaluation per count
lists the engine's kernel classes (launches, ms).  The card name and its power limit are read in the same run.  Writes
nothing into the tree.
"""
from __future__ import annotations

import argparse
import json
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

from chamfer_time import _events_ms, card_info  # noqa: E402
from width_time import CFG2, DATASHEET_BF16_TFLOPS  # noqa: E402


def build(inducers: int, device):
    import gecco_b200 as G
    from gecco_b200.models import ConvNeXtExtractor, GaussianActivation, RayNetwork, SetTransformer
    from gecco_b200.reparam import GaussianReparam

    torch.manual_seed(0)
    rp = GaussianReparam(torch.tensor(CFG2["mean"]), torch.tensor(CFG2["sigma"]))
    st = SetTransformer(n_layers=6, num_inducers=inducers, feature_dim=384, t_embed_dim=1, num_heads=8,
                        activation=GaussianActivation)
    net = RayNetwork(backbone=st, reparam=rp, context_dims=(96, 192, 384))
    model = G.Diffusion(backbone=G.EDMPrecond(model=net), conditioner=ConvNeXtExtractor(pretrained=False), reparam=rp,
                        loss=G.EDMLoss(schedule=G.LogUniformSchedule(max=CFG2["sigma_max"])))
    return model.to(device).eval()


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--inducers", default="64,128,192,256")
    ap.add_argument("--clouds", type=int, default=64)
    ap.add_argument("--points", type=int, default=2048)
    ap.add_argument("--steps", type=int, default=64)
    ap.add_argument("--reps", type=int, default=2)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("inducer_time.py measures on the GPU; no CUDA device is visible")

    import gecco_b200 as G
    from gecco_b200 import engine as E
    from gecco_b200.training import flops_per_cloud

    dev = torch.device("cuda:0")
    B, N = args.clouds, args.points
    print(json.dumps({"card": card_info()}))
    rows = []
    for inducers in [int(i) for i in args.inducers.split(",")]:
        model = build(inducers, dev)
        K = torch.tensor(CFG2["K"]).expand(B, 3, 3).contiguous().to(dev)
        img = torch.rand(B, 3, CFG2["image"], CFG2["image"], generator=torch.Generator().manual_seed(1)).to(dev)
        ctx = G.Context3d(image=img, K=K)
        rng = torch.Generator(dev).manual_seed(42)
        call = lambda: model.sample_stochastic((B, N, 3), ctx, rng=rng, num_steps=args.steps)
        with torch.no_grad():
            out = call()
            assert torch.isfinite(out).all(), inducers
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
        fpc = flops_per_cloud(N, inducers=inducers)
        evals = 2 * args.steps - 1
        tflops = B * evals * fpc / (best * 1e-3) / 1e12
        row = dict(inducers=inducers, clouds=B, points=N, steps=args.steps, ms_per_call=ms, clouds_per_s=B / (best * 1e-3),
                   flops_per_cloud_eval=fpc, tflops=tflops, datasheet_bf16_share=tflops / DATASHEET_BF16_TFLOPS,
                   classes_one_eval=classes)
        rows.append(row)
        print(json.dumps(row))
        del model
        torch.cuda.empty_cache()
    print("| I | ms per call | clouds/s | GFLOP per cloud per evaluation | TFLOP/s | share of 2250 TFLOP/s |")
    print("|---|---|---|---|---|---|")
    for r in rows:
        print(f"| {r['inducers']} | {min(r['ms_per_call']):.0f} | {r['clouds_per_s']:.2f} | "
              f"{r['flops_per_cloud_eval'] / 1e9:.1f} | {r['tflops']:.0f} | {r['datasheet_bf16_share']:.3f} |")


if __name__ == "__main__":
    main()

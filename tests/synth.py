"""Deterministic synthetic weights / inputs shared by oracle/make_golden.py, the tests, smoke() and bench.py.

The golden fixtures under tests/golden/ store only the recipe (seeds, shapes, config) and the reference
OUTPUTS; weights and inputs are regenerated from seeds with the CPU torch generator, so full-width
(C=384, 6 layer) goldens stay a few hundred KB.  Nothing here touches the reference or the CUDA library.
"""
from __future__ import annotations

import math
from typing import Dict, Sequence

import torch

# Reference hyper-parameters (SURVEY.md §3.1): cfg/shapenet_airplane_unconditional.py:27-56,
# cfg/taskonomy_conditional.py:29-69.
FEATURE_DIM = 384
NUM_INDUCERS = 64
NUM_HEADS = 8
N_LAYERS = 6
CONTEXT_DIMS = (96, 192, 384)

UNCOND_REPARAM = dict(mean=[0.0, 0.01, 0.05], sigma=[0.11, 0.04, 0.17])  # GaussianReparam, σmax 165
SHAPENET_VOL_REPARAM = dict(mean=[0.0, 0.0, 1.0], sigma=[0.15, 0.15, 0.15])  # SURVEY §8d config 2
UVL_REPARAM = dict(mean=[0.0, 0.0, 1.38], sigma=[0.56, 0.60, 0.49])  # cfg/taskonomy_conditional.py, σmax 180
K_SHAPENET = [[1.0859, 0.0, 0.4964], [0.0, 1.0859, 0.4964], [0.0, 0.0, 1.0]]
K_TASKONOMY = [[1.2, 0.0, 0.5], [0.0, 1.2, 0.5], [0.0, 0.0, 1.0]]


def gen(seed: int) -> torch.Generator:
    return torch.Generator(device="cpu").manual_seed(seed)


def _scale_for(name: str, shape: Sequence[int]) -> tuple[float, float]:
    """(std, offset) of the synthetic value of parameter `name`."""
    leaf = name.rsplit(".", 1)[-1]
    if name.endswith("alpha"):
        return 0.15, 1.2
    if name.endswith("inducers"):
        return 1.0, 0.0
    # AdaGN (models/normalization.py:26-34): scale = Linear(t), bias = Linear(t); zero-init in the reference,
    # randomised here so that the t-conditioning is actually exercised (SURVEY.md §4).
    if ".scale." in name or name.endswith("norm.scale") or "_norm.scale." in name:
        return (0.3, 0.0) if leaf == "weight" else (0.1, 1.0)
    if any(k in name for k in ("broadcast_norm.bias.", "mlp_norm.bias.", "norm_1.bias.", "norm_2.bias.")):
        return (0.3, 0.0) if leaf == "weight" else (0.1, 0.0)
    if leaf in ("weight", "in_proj_weight") and len(shape) == 2:
        std = 1.0 / math.sqrt(shape[1])
        if name.endswith("unpool.out_proj.weight") or name.endswith("mlp.2.weight"):
            std *= 0.5  # residual branches (the reference scales them by 0.1 at init, set_transformer.py:150-153)
        return std, 0.0
    return 0.1, 0.0  # biases


def synth_state_dict(shapes: Dict[str, Sequence[int]], seed: int) -> Dict[str, torch.Tensor]:
    """fp32 tensors for every entry of `shapes` (iterated in sorted key order) from one CPU generator."""
    g = gen(seed)
    out = {}
    for name in sorted(shapes):
        shape = tuple(shapes[name])
        std, off = _scale_for(name, shape)
        out[name] = torch.randn(shape, generator=g, dtype=torch.float32) * std + off
    return out


def network_shapes(kind: str, n_layers: int = N_LAYERS, c: int = FEATURE_DIM, heads: int = NUM_HEADS,
                   inducers: int = NUM_INDUCERS, hidden: int | None = None,
                   context_dims: Sequence[int] = CONTEXT_DIMS, do_norm: bool = True) -> Dict[str, tuple]:
    """Names and shapes of the learnable tensors of the denoiser in the reference state_dict schema
    (SURVEY.md §8b; prefix `backbone.model.`).  kind: "uncond" (LinearLift) or "cond" (RayNetwork).
    do_norm=False is LinearLift(do_norm=False): the head is a bare Linear, `lower.*` instead of `lower.1.*`."""
    hidden = hidden or 2 * c
    p = "backbone.model."
    s: Dict[str, tuple] = {}
    if kind == "uncond":
        s[p + "lift.weight"], s[p + "lift.bias"] = (c, 3), (c,)
        lower = p + ("lower.1." if do_norm else "lower.")
        s[lower + "weight"], s[lower + "bias"] = (3, c), (3,)
        st = p + "inner."
    else:
        s[p + "xyz_embed.weight"], s[p + "xyz_embed.bias"] = (c, 3), (c,)
        s[p + "img_feature_proj.1.weight"], s[p + "img_feature_proj.1.bias"] = (c, sum(context_dims)), (c,)
        s[p + "output_proj.1.weight"], s[p + "output_proj.1.bias"] = (3, c), (3,)
        st = p + "backbone."
    for l in range(n_layers):
        q = f"{st}layers.{l}."
        for norm in ("broadcast_norm.", "mlp_norm.", "broadcast.norm_1.", "broadcast.norm_2."):
            for half in ("scale.", "bias."):
                s[q + norm + half + "weight"], s[q + norm + half + "bias"] = (c, 1), (c,)
        s[q + "broadcast.pool.inducers"] = (1, heads, inducers, c // heads)
        s[q + "broadcast.pool.kv_proj.weight"] = (2 * c, c)
        s[q + "broadcast.pool.out_proj.weight"] = (c, c)
        for m in ("broadcast.mlp.", "mlp."):
            s[q + m + "0.weight"], s[q + m + "0.bias"] = (hidden, c), (hidden,)
            s[q + m + "1.alpha"] = ()
            s[q + m + "2.weight"], s[q + m + "2.bias"] = (c, hidden), (c,)
        s[q + "broadcast.unpool.in_proj_weight"], s[q + "broadcast.unpool.in_proj_bias"] = (3 * c, c), (3 * c,)
        s[q + "broadcast.unpool.out_proj.weight"], s[q + "broadcast.unpool.out_proj.bias"] = (c, c), (c,)
    return s


def reparam_buffers(reparam: str, mean, sigma) -> Dict[str, torch.Tensor]:
    """Top-level and network-level copies of the reparam buffers (reparam.py:54-55,90-91; models/ray.py:47)."""
    m, s = torch.as_tensor(mean, dtype=torch.float32).clone(), torch.as_tensor(sigma, dtype=torch.float32).clone()
    if reparam == "gaussian":
        return {"reparam.mean": m, "reparam.sigma": s}
    if reparam == "uvl":
        return {"reparam.uvl_mean": m, "reparam.uvl_std": s}
    return {}


def full_state_dict(kind: str, reparam: str, mean, sigma, seed: int, **kw) -> Dict[str, torch.Tensor]:
    sd = synth_state_dict(network_shapes(kind, **kw), seed)
    bufs = reparam_buffers(reparam, mean, sigma)
    sd.update(bufs)
    if kind == "cond":  # RayNetwork keeps its own reference to the same reparam module (models/ray.py:47)
        sd.update({"backbone.model." + k: v.clone() for k, v in bufs.items()})
    return sd


def tame(sd: Dict[str, torch.Tensor], out_scale: float) -> Dict[str, torch.Tensor]:
    """The "tame" recipe: the same synthetic weights with the output head (`lower.1`, `lower` without the LayerNorm, or
    `output_proj.1`) scaled by
    `out_scale`.  With the raw recipe the Lipschitz constant of F is far above 1 and the 64-step sampler amplifies any
    perturbation (the unmodified reference drifts by 10-35 % under its own bf16 autocast); scaled to ~1 the
    probability-flow map contracts and full trajectories can be held to a tight tolerance."""
    out = dict(sd)
    for k, v in sd.items():
        if ".lower.1." in k or ".output_proj.1." in k or k.endswith((".lower.weight", ".lower.bias")):
            out[k] = v * out_scale
    return out


def noisy_input(batch: int, points: int, sigma: torch.Tensor, data_seed: int, noise_seed: int) -> torch.Tensor:
    """What the denoiser sees in the sampler and in the training loss (diffusion.py:139-140, 325): diffusion-space data of
    unit variance plus sigma * noise, so that c_in(sigma) * x has unit variance at every noise level."""
    x0 = torch.randn(batch, points, 3, generator=gen(data_seed))
    n = torch.randn(batch, points, 3, generator=gen(noise_seed))
    return x0 + sigma.reshape(-1, 1, 1) * n


def synth_features(batch: int, sizes: Sequence[int], seed: int, dims: Sequence[int] = CONTEXT_DIMS):
    """Synthetic feature pyramid (what ConvNeXtExtractor would return, models/feature_pyramid.py:62-73): NCHW fp32."""
    g = gen(seed)
    return [torch.randn(batch, c, s, s, generator=g, dtype=torch.float32) for c, s in zip(dims, sizes)]


def camera(batch: int, K) -> torch.Tensor:
    return torch.tensor(K, dtype=torch.float32).expand(batch, 3, 3).contiguous()

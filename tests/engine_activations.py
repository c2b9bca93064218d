"""MLP activations other than the normalised Gaussian, for the engine tests (test_engine_activations_*.py).  Every MLP of a
model uses one activation: "gaussian" (GaussianActivation(), the production recipe), "gaussian_raw"
(GaussianActivation(normalized=False)) or "relu" (nn.ReLU, the default of SetTransformer / MLP).

The synthetic weights are tests/synth.py's recipe without the MLPs' `1.alpha` for ReLU (and that recipe itself, bit for
bit, for the Gaussians).  The float64 oracle (oracle/gecco_oracle.py) restates the reference's normalised-Gaussian MLP;
`oracle_activation` runs it with another activation by restating its `mlp` (models/mlp.py:5-39 with
models/activation.py:17-24 or nn.ReLU) for the duration.  Models are built with the reference constructor keywords.
Nothing here imports the CUDA library at import time."""
from __future__ import annotations

import contextlib
import functools
from dataclasses import dataclass
from typing import Dict

import torch
import torch.nn.functional as F

from oracle import gecco_oracle as O
from tests import synth
from tests.engine_inducers import InducerConfig

ACTIVATIONS = ["relu", "gaussian_raw"]
CODES = {"gaussian": 1, "gaussian_raw": 2, "relu": 3}  # GECCO_ACT_*


def activation_module(name: str):
    """The `activation=` constructor argument of SetTransformer for `name`."""
    from gecco_b200.models import GaussianActivation

    if name == "relu":
        return torch.nn.ReLU
    return functools.partial(GaussianActivation, normalized=name == "gaussian")


# ------------------------------------------------------------------------------------------------ synthetic weights
def network_shapes(kind: str, activation: str = "gaussian", **kw) -> Dict[str, tuple]:
    """synth.network_shapes, without the MLPs' `1.alpha` when the activation is ReLU (nn.ReLU has no parameter)."""
    shapes = synth.network_shapes(kind, **kw)
    if activation == "relu":
        shapes = {k: v for k, v in shapes.items() if not k.endswith("mlp.1.alpha")}
    return shapes


def full_state_dict(kind: str, reparam: str, mean, sigma, seed: int, activation: str = "gaussian",
                    **kw) -> Dict[str, torch.Tensor]:
    """synth.full_state_dict over `network_shapes(kind, activation)`; at the Gaussians it is synth.full_state_dict."""
    sd = synth.synth_state_dict(network_shapes(kind, activation, **kw), seed)
    bufs = synth.reparam_buffers(reparam, mean, sigma)
    sd.update(bufs)
    if kind == "cond":  # RayNetwork keeps its own reference to the same reparam module (models/ray.py:47)
        sd.update({"backbone.model." + k: v.clone() for k, v in bufs.items()})
    return sd


# ------------------------------------------------------------------------------------------------ oracle
def activation(name: str, sd: dict, pre: str, h: torch.Tensor) -> torch.Tensor:
    """The MLP activation `name` on the first projection's output; `pre` + "1.alpha" is read for the Gaussians."""
    if name == "gaussian":
        return O.gaussian_act(h, sd[pre + "1.alpha"])
    if name == "gaussian_raw":  # models/activation.py:17-24 with normalized=False
        return (-(h**2) / (2 * sd[pre + "1.alpha"] ** 2)).exp()
    if name == "relu":
        return F.relu(h)
    raise ValueError(f"unknown activation {name!r}")


def mlp(sd: dict, pre: str, x: torch.Tensor, name: str) -> torch.Tensor:
    """gecco_oracle.mlp (models/mlp.py:5-39, depth 1) with the activation `name`."""
    h = F.linear(x, sd[pre + "0.weight"], sd[pre + "0.bias"])
    return F.linear(activation(name, sd, pre, h), sd[pre + "2.weight"], sd[pre + "2.bias"])


@contextlib.contextmanager
def oracle_activation(name: str):
    """Every oracle function called inside the block (denoise, the samplers, set_transformer, ...) uses MLPs with the
    activation `name`: the oracle's layers look `mlp` up in their module at call time, so it is replaced by `mlp` above
    for the block and restored afterwards.  At "gaussian" the oracle runs as it is."""
    if name == "gaussian":
        yield
        return
    saved = O.mlp
    O.mlp = lambda sd, pre, x: mlp(sd, pre, x, name)
    try:
        yield
    finally:
        O.mlp = saved


@dataclass(frozen=True)
class ActivationConfig(InducerConfig):
    activation: str = "gaussian"

    def state_dict(self, seed: int = 1234) -> dict:
        return full_state_dict(self.kind, self.reparam, self.stats["mean"], self.stats["sigma"], seed, self.activation,
                               c=self.width, n_layers=self.layers, heads=self.heads, inducers=self.inducers,
                               hidden=self.blowup * self.width, context_dims=self.context_dims, do_norm=self.do_norm)


def set_transformer(cfg: ActivationConfig):
    from gecco_b200.models import SetTransformer

    return SetTransformer(n_layers=cfg.layers, num_inducers=cfg.inducers, feature_dim=cfg.width, t_embed_dim=1,
                          num_heads=cfg.heads, mlp_blowup=cfg.blowup, activation=activation_module(cfg.activation))


def build(cfg: ActivationConfig, device, features=None, state_dict=None, weight_seed: int | None = 1234, st=None):
    """The model of `cfg` under LinearLift or RayNetwork, EDMPrecond, EDMLoss with `state_dict`, else the synthetic weights
    of `weight_seed`; `st` replaces the SetTransformer (e.g. a default-constructed one)."""
    import gecco_b200 as G
    from gecco_b200.models import LinearLift, RayNetwork
    from gecco_b200.reparam import GaussianReparam, UVLReparam

    from tests.models_b200 import FixedConditioner

    st = set_transformer(cfg) if st is None else st
    m = torch.tensor(cfg.stats["mean"], dtype=torch.float32)
    s = torch.tensor(cfg.stats["sigma"], dtype=torch.float32)
    rp = GaussianReparam(m, s) if cfg.reparam == "gaussian" else UVLReparam(m, s)
    if cfg.kind == "uncond":
        net, cond = LinearLift(inner=st, feature_dim=cfg.width, do_norm=cfg.do_norm), G.IdleConditioner()
    else:
        net = RayNetwork(backbone=st, reparam=rp, context_dims=list(cfg.context_dims))
        cond = FixedConditioner(None if features is None else [f.to(device) for f in features])
    model = G.Diffusion(backbone=G.EDMPrecond(model=net, sigma_data=cfg.sigma_data), conditioner=cond, reparam=rp,
                        loss=G.EDMLoss(schedule=G.LogUniformSchedule(max=cfg.sigma_max), sigma_data=cfg.sigma_data))
    if state_dict is None and weight_seed is not None:
        state_dict = cfg.state_dict(weight_seed)
    if state_dict is not None:
        model.load_state_dict(state_dict)
    return model.to(device).eval()


def activation_config(activation: str, kind: str = "uncond", reparam: str = "gaussian", width: int = synth.FEATURE_DIM,
                      heads: int = synth.NUM_HEADS, inducers: int = synth.NUM_INDUCERS, blowup: int = 2) -> ActivationConfig:
    return ActivationConfig(f"{activation}_{kind}_{reparam}_c{width}_h{heads}_i{inducers}_b{blowup}", kind=kind,
                            reparam=reparam, heads=heads, width=width, inducers=inducers, blowup=blowup,
                            activation=activation)


def _rows(act: str) -> list:
    return [
        activation_config(act),                                    # production shape: AdaGN in the GEMM, mlp_pair, chain
        activation_config(act, "cond", "gaussian"),
        activation_config(act, "cond", "uvl"),
        activation_config(act, width=256, heads=8),                # fallback kernels (no chain, fused MLP without AdaGN)
        activation_config(act, width=768, heads=12),
        activation_config(act, inducers=128),                      # separate inducer-side launches
        activation_config(act, blowup=3),                          # two-GEMM MLP
    ]


CONFIGS = [c for act in ACTIVATIONS for c in _rows(act)]
BY_NAME = {c.name: c for c in CONFIGS}
PROD = {act: activation_config(act) for act in ACTIVATIONS}

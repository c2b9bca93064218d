"""Inducer counts other than the production 64, for the engine tests (test_engine_inducers_*.py).  The engine takes whole
blocks of 64 inducers up to 256; the tcgen05 attention cores and the inducer cluster kernel stay 64-only, so every row
here runs the mma.sync attention cores and the separate inducer-side launches.  Weights come from tests/synth.py
(`network_shapes` takes the count as `inducers`) and models are built with the reference constructor keywords; at 64
inducers `build` and `state_dict` reproduce tests/models_b200.py and the production recipe exactly
(test_engine_inducers_cpu.py).  Nothing here imports the CUDA library at import time."""
from __future__ import annotations

from dataclasses import dataclass

import torch

from tests import synth
from tests.engine_widths import WidthConfig

COUNTS = [128, 192, 256]
# whole 64-inducer blocks beyond 256, or half blocks: no kernels
REFUSED = [32, 96, 320]


@dataclass(frozen=True)
class InducerConfig(WidthConfig):
    inducers: int = synth.NUM_INDUCERS

    def state_dict(self, seed: int = 1234) -> dict:
        return synth.full_state_dict(self.kind, self.reparam, self.stats["mean"], self.stats["sigma"], seed, c=self.width,
                                     n_layers=self.layers, heads=self.heads, inducers=self.inducers,
                                     hidden=self.blowup * self.width, context_dims=self.context_dims, do_norm=self.do_norm)


def set_transformer(cfg: InducerConfig):
    from gecco_b200.models import GaussianActivation, SetTransformer

    return SetTransformer(n_layers=cfg.layers, num_inducers=cfg.inducers, feature_dim=cfg.width, t_embed_dim=1,
                          num_heads=cfg.heads, mlp_blowup=cfg.blowup, activation=GaussianActivation)


def build(cfg: InducerConfig, device, features=None, state_dict=None, weight_seed: int | None = 1234):
    """The model of `cfg` (SetTransformer(num_inducers=cfg.inducers, feature_dim=cfg.width, ...) under LinearLift or
    RayNetwork, EDMPrecond, EDMLoss) with `state_dict`, else the synthetic weights of `weight_seed`; conditional models
    read the fixed pyramid `features`."""
    import gecco_b200 as G
    from gecco_b200.models import LinearLift, RayNetwork
    from gecco_b200.reparam import GaussianReparam, UVLReparam

    from tests.models_b200 import FixedConditioner

    st = set_transformer(cfg)
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


def inducer_config(kind: str, reparam: str, inducers: int, width: int = synth.FEATURE_DIM,
                   heads: int = synth.NUM_HEADS) -> InducerConfig:
    return InducerConfig(f"{kind}_{reparam}_i{inducers}_c{width}_h{heads}", kind=kind, reparam=reparam, heads=heads,
                         width=width, inducers=inducers)


# every count at the production width for the unconditional and the conditional Gaussian and UVL models, plus head dims
# 32 (C = 256, 8 heads) and 64 (C = 768, 12 heads)
CONFIGS = [inducer_config(kind, rp, i) for kind, rp in (("uncond", "gaussian"), ("cond", "gaussian"), ("cond", "uvl"))
           for i in COUNTS]
CONFIGS += [inducer_config("uncond", "gaussian", 128, 256, 8), inducer_config("cond", "gaussian", 256, 768, 12)]
BY_NAME = {c.name: c for c in CONFIGS}

"""Feature widths other than the production 384, for the engine tests (test_engine_widths_*.py).  With the reference's 32
AdaGN groups a width C has C / 32-channel groups; the engine takes every C whose group width divides the 192-column GEMM
epilogue panel.  Weights come from tests/synth.py (`network_shapes` takes the width as `c`) and models are built with the
reference constructor keywords, as tests/models_b200.py does at 384; `build` and `state_dict` reproduce those two exactly at
C = 384 (test_engine_widths_cpu.py).  Nothing here imports the CUDA library at import time."""
from __future__ import annotations

from dataclasses import dataclass

import torch

from tests import synth
from tests.engine_configs import Config

# (feature_dim, num_heads): head dims 32 / 32 / 64 / 64 / 64
WIDTHS = [(128, 4), (256, 8), (512, 8), (768, 12), (1024, 16)]
# widths whose AdaGN groups (20 and 28 channels) do not divide the panel
REFUSED = [(640, 10), (896, 14)]


@dataclass(frozen=True)
class WidthConfig(Config):
    width: int = synth.FEATURE_DIM

    def state_dict(self, seed: int = 1234) -> dict:
        return synth.full_state_dict(self.kind, self.reparam, self.stats["mean"], self.stats["sigma"], seed, c=self.width,
                                     n_layers=self.layers, heads=self.heads, hidden=self.blowup * self.width,
                                     context_dims=self.context_dims, do_norm=self.do_norm)


def build(cfg: WidthConfig, device, features=None, state_dict=None, weight_seed: int | None = 1234):
    """The model of `cfg` (SetTransformer(feature_dim=cfg.width, ...) under LinearLift or RayNetwork, EDMPrecond, EDMLoss)
    with `state_dict`, else the synthetic weights of `weight_seed`; conditional models read the fixed pyramid `features`."""
    import gecco_b200 as G
    from gecco_b200.models import GaussianActivation, LinearLift, RayNetwork, SetTransformer
    from gecco_b200.reparam import GaussianReparam, UVLReparam

    from tests.models_b200 import FixedConditioner

    st = SetTransformer(n_layers=cfg.layers, num_inducers=synth.NUM_INDUCERS, feature_dim=cfg.width, t_embed_dim=1,
                        num_heads=cfg.heads, mlp_blowup=cfg.blowup, activation=GaussianActivation)
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


def width_config(kind: str, reparam: str, width: int, heads: int) -> WidthConfig:
    return WidthConfig(f"{kind}_{reparam}_c{width}_h{heads}", kind=kind, reparam=reparam, heads=heads, width=width)


# every width for the unconditional model and the conditional Gaussian and UVL models
CONFIGS = [width_config(kind, rp, c, h) for kind, rp in (("uncond", "gaussian"), ("cond", "gaussian"), ("cond", "uvl"))
           for c, h in WIDTHS]
BY_NAME = {c.name: c for c in CONFIGS}

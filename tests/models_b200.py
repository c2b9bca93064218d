"""Builds gecco_b200 models (reference constructor surface) with the synthetic weights of tests/synth.py."""
from __future__ import annotations

import torch

from tests import synth


class FixedConditioner(torch.nn.Module):
    """Returns a fixed synthetic pyramid in place of ConvNeXtExtractor (the conditioner is upstream of the hot path)."""

    def __init__(self, features):
        super().__init__()
        self.features = features

    def forward(self, raw_ctx):
        from gecco_b200.structs import FeaturePyramidContext

        return FeaturePyramidContext(features=self.features, K=raw_ctx.K)


class FreshConditioner(torch.nn.Module):
    """Returns NEW tensors (clones) on every call, like a real CNN: the engine must not reuse a packed pyramid keyed on
    recycled addresses (ADVICE r1: feature cache)."""

    def __init__(self, features):
        super().__init__()
        self.features = features

    def forward(self, raw_ctx):
        from gecco_b200.structs import FeaturePyramidContext

        return FeaturePyramidContext(features=[f.clone() for f in self.features], K=raw_ctx.K)


def build(kind: str, reparam: str, mean, sigma, sigma_max: float, weight_seed: int | None, device, features=None,
          n_layers: int = synth.N_LAYERS, convnext_seed: int | None = None, state_dict=None, num_heads: int = synth.NUM_HEADS,
          mlp_blowup: int = 2, do_norm: bool = True, sigma_data: float = 1.0, context_dims=synth.CONTEXT_DIMS):
    """The reference constructor keywords `num_heads`, `mlp_blowup` (SetTransformer), `do_norm` (LinearLift),
    `sigma_data` (EDMPrecond and EDMLoss) and `context_dims` (RayNetwork) default to the production configuration."""
    import gecco_b200 as G
    from gecco_b200.models import GaussianActivation, LinearLift, RayNetwork, SetTransformer
    from gecco_b200.reparam import GaussianReparam, UVLReparam

    st = SetTransformer(n_layers=n_layers, num_inducers=synth.NUM_INDUCERS, feature_dim=synth.FEATURE_DIM, t_embed_dim=1,
                        num_heads=num_heads, mlp_blowup=mlp_blowup, activation=GaussianActivation)
    m, s = torch.tensor(mean, dtype=torch.float32), torch.tensor(sigma, dtype=torch.float32)
    rp = GaussianReparam(m, s) if reparam == "gaussian" else UVLReparam(m, s)
    if kind == "uncond":
        net, cond = LinearLift(inner=st, feature_dim=synth.FEATURE_DIM, do_norm=do_norm), G.IdleConditioner()
    else:
        net = RayNetwork(backbone=st, reparam=rp, context_dims=list(context_dims))
        if convnext_seed is not None:
            # the reference's own conditioner (models/feature_pyramid.py:28-73), random init from the global CPU generator
            from gecco_b200.models import ConvNeXtExtractor

            torch.manual_seed(convnext_seed)
            cond = ConvNeXtExtractor(n_stages=3, model="tiny", pretrained=False)
        else:
            cond = FixedConditioner(None if features is None else [f.to(device) for f in features])
    model = G.Diffusion(backbone=G.EDMPrecond(model=net, sigma_data=sigma_data), conditioner=cond, reparam=rp,
                        loss=G.EDMLoss(schedule=G.LogUniformSchedule(max=sigma_max), sigma_data=sigma_data))
    if state_dict is not None:
        model.load_state_dict(state_dict, strict=convnext_seed is None)
    elif weight_seed is not None:
        sd = synth.full_state_dict(kind, reparam, mean, sigma, weight_seed, n_layers=n_layers, heads=num_heads,
                                   hidden=mlp_blowup * synth.FEATURE_DIM, context_dims=context_dims, do_norm=do_norm)
        model.load_state_dict(sd, strict=convnext_seed is None)
    return model.to(device).eval()

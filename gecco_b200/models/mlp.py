"""Per-point MLP parameter container (reference: gecco_torch/models/mlp.py:5-39).

Linear -> activation -> [Linear -> activation] x (depth-1) -> Linear as an nn.Sequential, so the state_dict keys
are `0.weight, 0.bias, 1.alpha, 2.weight, 2.bias` for depth 1.  Inside the denoiser engine the point-side MLP runs as
tcgen05 GEMMs with the activation, bias and residual in their epilogues (depth 1, with GaussianActivation in either
form or nn.ReLU, the reference's default; every MLP of a model uses the same one); the stand-alone `forward` below runs
the same GEMM kernel per Linear for any depth.  Other activation modules are refused by the engine.
"""
from typing import Callable

import torch
import torch.nn as nn


class MLP(nn.Sequential):
    def __init__(self, in_features: int, out_features: int, width_size: int, depth: int = 1,
                 activation: Callable = nn.ReLU):
        mods = [nn.Linear(in_features, width_size), activation()]
        for _ in range(depth - 1):
            mods += [nn.Linear(width_size, width_size), activation()]
        mods.append(nn.Linear(width_size, out_features))
        super().__init__(*mods)
        self.depth = depth

    @torch.no_grad()
    def forward(self, x):
        """[..., in_features] -> [..., out_features]; every Linear is one `gecco_gemm` launch.  GaussianActivation (either
        form) and nn.ReLU are fused into the epilogue of the projection in front of them; any other activation module
        runs as its own torch forward on the fp32 projection output."""
        from . import _native

        lead = x.shape[:-1]
        x3 = x.reshape(1, -1, x.shape[-1]) if x.ndim != 3 else x
        out = _native.mlp_forward(self, x3)
        return out.reshape(*lead, out.shape[-1])

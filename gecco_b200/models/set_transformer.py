"""Inducer-point SetTransformer: parameter containers with the reference's module tree
(gecco_torch/models/set_transformer.py:14-216), so `state_dict()` keys and random initialisation match.

Inside a denoiser (`LinearLift` / `RayNetwork` / `EDMPrecond` / `Diffusion`) the computation does not run module by
module: `gecco_b200.engine.Engine` walks this tree once, packs the weights and runs the whole stack fused in the CUDA
engine (csrc/engine.cu).  Every module here ALSO has the reference's stand-alone `forward` (same arguments and return
conventions), executed with the same C-ABI kernels through `models/_native.py`: tcgen05 GEMMs with fused bias /
activation / residual epilogues, the two attention cores and the AdaGN kernels.  No torch math, no CPU path.
`activation` (every MLP of the model): nn.ReLU (the reference's default), GaussianActivation (normalised, the reference
configurations' choice) or GaussianActivation(normalized=False), e.g. `functools.partial(GaussianActivation,
normalized=False)`; the engine refuses any other module.
"""
from __future__ import annotations

import torch
from torch import Tensor, nn

from . import _native
from .mlp import MLP
from .normalization import AdaGN


class AttentionPool(nn.Module):
    """points -> inducers cross-attention with learned queries (set_transformer.py:14-65)."""

    def __init__(self, feature_dim: int, num_heads: int, num_inducers: int):
        super().__init__()
        assert feature_dim % num_heads == 0, (feature_dim, num_heads)
        self.num_heads = num_heads
        self.feature_dim = feature_dim
        self.dims_per_head = feature_dim // num_heads
        self.inducers = nn.Parameter(torch.randn(1, num_heads, num_inducers, self.dims_per_head))
        self.kv_proj = nn.Linear(feature_dim, 2 * feature_dim, bias=False)
        self.out_proj = nn.Linear(feature_dim, feature_dim, bias=False)

    @torch.no_grad()
    def forward(self, kv: Tensor) -> Tensor:
        """[B, N, C] -> [B, num_inducers, C] (set_transformer.py:47-65)."""
        return _native.attention_pool_forward(self, kv)


class Broadcast(nn.Module):
    """pool -> AdaGN -> MLP -> AdaGN on the inducers, then inducers -> points attention (set_transformer.py:68-117).
    `unpool` is an nn.MultiheadAttention so that its parameter names and initialisation are the reference's."""

    def __init__(self, feature_dim: int, num_inducers: int, t_embed_dim: int, num_heads: int = 8, mlp_blowup: int = 2,
                 activation: nn.Module = nn.ReLU):
        super().__init__()
        self.pool = AttentionPool(feature_dim, num_heads, num_inducers)
        self.norm_1 = AdaGN(feature_dim, t_embed_dim)
        self.mlp = MLP(feature_dim, feature_dim, mlp_blowup * feature_dim, activation=activation)
        self.norm_2 = AdaGN(feature_dim, t_embed_dim)
        self.unpool = nn.MultiheadAttention(feature_dim, num_heads, batch_first=True)

    @torch.no_grad()
    def forward(self, x: Tensor, t_embed: Tensor, return_h: bool = False, h: Tensor | None = None):
        """(attn, h | None) like the reference (set_transformer.py:92-117); a given `h` skips the inducer side."""
        return self._forward(x, t_embed, return_h, h, None)

    def _forward(self, x, t_embed, return_h, h, residual):
        if h is None:
            h = self.pool(x)
            h = self.norm_1(h, t_embed)
            h = self.mlp(h)
            h = self.norm_2(h, t_embed)
        attn = _native.unpool_forward(self.unpool, x, h, residual)  # (+ residual in the out-projection epilogue)
        return attn, (h if return_h else None)


class BroadcastingLayer(nn.Module):
    """Pre-norm residual block: x += Broadcast(AdaGN(x)); x += MLP(AdaGN(x)) (set_transformer.py:120-168)."""

    def __init__(self, feature_dim: int, num_inducers: int, embed_dim: int, num_heads: int = 8, mlp_blowup: int = 2,
                 activation: nn.Module = nn.ReLU):
        super().__init__()
        self.broadcast_norm = AdaGN(feature_dim, embed_dim)
        self.broadcast = Broadcast(feature_dim, num_inducers, embed_dim, num_heads, mlp_blowup=mlp_blowup,
                                   activation=activation)
        self.mlp_norm = AdaGN(feature_dim, embed_dim)
        self.mlp = MLP(feature_dim, feature_dim, mlp_blowup * feature_dim, activation=activation)
        with torch.no_grad():  # residual branches start small (:150-153)
            self.broadcast.unpool.out_proj.weight.mul_(0.1)
            self.mlp[-1].weight.mul_(0.1)

    @torch.no_grad()
    def forward(self, x: Tensor, t_embed: Tensor, return_h: bool = False, h: Tensor | None = None):
        """x += Broadcast(AdaGN(x)); x += MLP(AdaGN(x)) (set_transformer.py:155-168); both residual adds run in the
        epilogue of the projection that produces the branch."""
        y = self.broadcast_norm(x, t_embed)
        x, h = self.broadcast._forward(y, t_embed, return_h, h, x)
        y = self.mlp_norm(x, t_embed)
        x = _native.mlp_forward(self.mlp, y, residual=x)
        return x, h


class SetTransformer(nn.Module):
    def __init__(self, n_layers: int, feature_dim: int, num_inducers: int, t_embed_dim: int, **kwargs):
        super().__init__()
        self.layers = nn.ModuleList(
            [BroadcastingLayer(feature_dim=feature_dim, num_inducers=num_inducers, embed_dim=t_embed_dim, **kwargs)
             for _ in range(n_layers)])
        self.feature_dim = feature_dim

    @torch.no_grad()
    def forward(self, features: Tensor, t_embed: Tensor, return_h: bool = False, hs: list | None = None):
        """(features, [h per layer] | None), consuming cached inducer states `hs` when given (set_transformer.py:198-216)."""
        if hs is None:
            hs = [None] * len(self.layers)
        stored_h = []
        for layer, h in zip(self.layers, hs):
            features, h = layer(features, t_embed, return_h=return_h, h=h)
            stored_h.append(h)
        return (features, stored_h) if return_h else (features, None)

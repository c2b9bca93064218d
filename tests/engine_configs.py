"""Network configurations other than the production one, for the engine tests (test_engine_configs_*.py): each row sets
the reference constructor keywords that send the engine down a different set of kernels (head dim 32 / 64 -> the
mma.sync attention kernels and the non-chain inducer side; hidden != 768 -> two-GEMM MLP; LinearLift(do_norm=False)
-> the head without a norm; sigma_data != 1; other feature pyramids -> other lookup channel splits).  Only weights,
inputs and the oracle side live here; nothing imports the CUDA library."""
from __future__ import annotations

from dataclasses import dataclass

import torch

from oracle import gecco_oracle as O
from tests import synth


@dataclass(frozen=True)
class Config:
    name: str
    kind: str = "uncond"
    reparam: str = "gaussian"
    heads: int = synth.NUM_HEADS
    blowup: int = 2
    do_norm: bool = True
    sigma_data: float = 1.0
    context_dims: tuple = synth.CONTEXT_DIMS
    layers: int = 2

    @property
    def stats(self):
        if self.reparam == "uvl":
            return synth.UVL_REPARAM
        return synth.UNCOND_REPARAM if self.kind == "uncond" else synth.SHAPENET_VOL_REPARAM

    @property
    def sigma_max(self) -> float:
        return 180.0 if self.reparam == "uvl" else 165.0

    @property
    def K(self):
        return synth.K_TASKONOMY if self.reparam == "uvl" else synth.K_SHAPENET

    def build_kw(self) -> dict:
        """Keywords of tests.models_b200.build."""
        return dict(n_layers=self.layers, num_heads=self.heads, mlp_blowup=self.blowup, do_norm=self.do_norm,
                    sigma_data=self.sigma_data, context_dims=self.context_dims)

    def oracle(self) -> O.OracleConfig:
        return O.OracleConfig(kind=self.kind, n_layers=self.layers, num_heads=self.heads, reparam=self.reparam,
                              sigma_data=self.sigma_data, sigma_max=self.sigma_max)

    def state_dict(self, seed: int = 1234) -> dict:
        return synth.full_state_dict(self.kind, self.reparam, self.stats["mean"], self.stats["sigma"], seed, n_layers=self.layers,
                                     heads=self.heads, hidden=self.blowup * synth.FEATURE_DIM, context_dims=self.context_dims,
                                     do_norm=self.do_norm)

    def features(self, clouds: int, seed: int = 21):
        """A synthetic pyramid, one level per entry of context_dims, halving in size from 34 x 34."""
        sizes = [max(34 >> l, 3) for l in range(len(self.context_dims))]
        return synth.synth_features(clouds, sizes, seed, dims=self.context_dims)


# The matrix of the engine-configuration tests.  Rows 1-9 in order; "prod" is the production configuration the shape sweep
# runs at.
CONFIGS = [
    Config("heads12", heads=12),
    Config("heads6", heads=6),
    Config("blowup1", blowup=1),
    Config("blowup4", blowup=4),
    Config("no_norm", do_norm=False),
    Config("sigma_data0.5", sigma_data=0.5),
    Config("cond_heads12_blowup3", kind="cond", heads=12, blowup=3, context_dims=(128,)),
    Config("cond_uvl_heads6_4levels", kind="cond", reparam="uvl", heads=6, sigma_data=0.5, context_dims=(64, 64, 128, 768)),
    Config("heads12_blowup1_no_norm_6layers", heads=12, blowup=1, do_norm=False, sigma_data=0.5, layers=6),
]
BY_NAME = {c.name: c for c in CONFIGS}
PROD = Config("prod")
PROD_COND6 = Config("prod_cond_6layers", kind="cond", layers=6)

SIGMAS = (0.3, 2.0, 40.0)


def sigmas(clouds: int) -> torch.Tensor:
    """Per-cloud noise levels cycling through SIGMAS."""
    return torch.tensor([SIGMAS[b % len(SIGMAS)] for b in range(clouds)], dtype=torch.float32)


def precond(sigma: torch.Tensor, sigma_data: float):
    """(c_skip, c_out) of EDMPrecond (diffusion.py:37-62), float64, shaped [B, 1, 1]."""
    s = sigma.reshape(-1, 1, 1).double()
    sd2 = sigma_data**2
    return sd2 / (s**2 + sd2), s * sigma_data / (s**2 + sd2).sqrt()


def raw_output(D: torch.Tensor, x: torch.Tensor, sigma: torch.Tensor, sigma_data: float) -> torch.Tensor:
    """The network output F = (D - c_skip x) / c_out, float64."""
    c_skip, c_out = precond(sigma.to(D.device), sigma_data)
    return (D.double() - c_skip * x.to(D.device).double()) / c_out


def rms(t: torch.Tensor) -> float:
    return t.double().pow(2).mean().sqrt().item()

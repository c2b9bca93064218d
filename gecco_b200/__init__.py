"""gecco_b200 — B200 (sm_100a) implementation of gecco-torch's reverse-diffusion sampling path.

Same module / call surface as `gecco_torch` for that path (Diffusion, EDMPrecond, SetTransformer, LinearLift,
RayNetwork, reparam schemes, Context3d), plus the 1-NNA / MMD / COV sample-quality metrics over a GPU Chamfer distance
(`metrics`); the work runs in hand-written CUDA kernels behind the C ABI declared in
include/gecco_b200.h (libgecco_b200.so, built by `python -m gecco_b200.build`).  No CPU fallback.
"""
from . import metrics, models, reparam
from .config import load_config
from .diffusion import Diffusion, EDMLoss, EDMPrecond, IdleConditioner, LogUniformSchedule
from .metrics import chamfer_distance, chamfer_matrix, metrics_from_distances, sample_metrics
from .structs import Context3d, Example

__all__ = ["metrics", "models", "reparam", "load_config", "Diffusion", "EDMLoss", "EDMPrecond", "IdleConditioner",
           "LogUniformSchedule", "Context3d", "Example", "chamfer_distance", "chamfer_matrix", "metrics_from_distances",
           "sample_metrics"]

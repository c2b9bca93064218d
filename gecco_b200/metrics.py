"""Sample-quality metrics: Chamfer distance (CD) on the GPU and the 1-NNA / MMD / COV numbers built on it.

These are the numbers reported for GECCO and its peers (PointFlow, LION); gecco-jax computes them in ``metrics.py`` /
``benchmark.py``.  The definitions follow PointFlow's ``compute_all_metrics``:

- ``CD(X, Y) = mean_{x in X} min_{y in Y} |x - y|^2 + mean_{y in Y} min_{x in X} |x - y|^2`` -- squared Euclidean
  distances, means (not sums); X and Y may have different point counts.
- ``MMD-CD = mean_{r in S_r} min_{g in S_g} CD(g, r)``.
- ``COV-CD = |{argmin_{r in S_r} CD(g, r) : g in S_g}| / |S_r|``.
- ``1-NNA-CD``: over the union ``[S_g; S_r]`` every cloud's nearest neighbour other than itself; the fraction of clouds whose
  nearest neighbour comes from their own set.  Perfect generation gives 0.5, a generator whose samples are all told apart
  from the reference gives 1.0.
- Ties: every argmin takes the lowest index; for 1-NNA the index in the concatenation ``[S_g; S_r]`` (PointFlow leaves this
  to ``topk``).
- No normalisation: clouds are compared as given, in data space, which is what the samplers return.  Centring or scaling
  the clouds (PointFlow normalises per shape or globally depending on the table) is the caller's choice.

The distance matrices come from the ``gecco_chamfer`` kernel (``csrc/chamfer.cu``): one block per cloud pair, both
directions in one pass, fp32 arithmetic on clouds translated to the first cloud's bounding-box centre, bitwise
deterministic.  CPU tensors are refused (there is no CPU path); ``metrics_from_distances`` is plain torch on the small
``[M, M]`` matrices and takes CPU or GPU tensors.
"""
from __future__ import annotations

import ctypes as C
import math

import torch
from torch import Tensor

from . import _abi
from .ops import _lib_for, _stream


def _clouds(t: Tensor, name: str) -> Tensor:
    """[M, N, 3] CUDA tensor -> contiguous fp32 on the same device; non-finite points raise ValueError naming the clouds
    (the kernel's minima would skip a NaN and return a finite, wrong distance)."""
    if not isinstance(t, Tensor):
        raise TypeError(f"{name}: expected a tensor, got {type(t).__name__}")
    if t.dim() != 3 or t.shape[-1] != 3:
        raise ValueError(f"{name}: expected clouds of shape [M, N, 3], got {tuple(t.shape)}")
    if t.shape[1] < 1:
        raise ValueError(f"{name}: clouds need at least one point")
    if not t.is_floating_point():
        raise TypeError(f"{name}: expected floating-point points, got {t.dtype}")
    bad = (~torch.isfinite(t)).flatten(1).any(1).nonzero().flatten().tolist()
    if bad:
        shown = ", ".join(map(str, bad[:10])) + (", ..." if len(bad) > 10 else "")
        raise ValueError(f"{name}: {len(bad)} cloud(s) with non-finite points (indices {shown})")
    if not t.is_cuda:
        raise _abi.GeccoError(f"{name}: gecco_b200 metrics need CUDA tensors (there is no CPU path)")
    return t.to(torch.float32).contiguous()


def _launch(a: Tensor, b: Tensor | None, mode: int, out: Tensor) -> None:
    lib = _lib_for(a)
    args = _abi.ChamferArgs()
    args.a, args.ma, args.na = a.data_ptr(), a.shape[0], a.shape[1]
    if b is not None:
        args.b, args.mb, args.nb = b.data_ptr(), b.shape[0], b.shape[1]
    args.mode = mode
    args.out = out.data_ptr()
    _abi.check(lib.gecco_chamfer(C.byref(args), _stream(a)))


def chamfer_distance(x: Tensor, y: Tensor) -> Tensor:
    """Paired Chamfer distance: ``out[i] = CD(x[i], y[i])``, fp32 ``[B]``.  x: ``[B, Nx, 3]``, y: ``[B, Ny, 3]``."""
    a, b = _clouds(x, "x"), _clouds(y, "y")
    if a.shape[0] != b.shape[0] or a.device != b.device:
        raise ValueError(f"chamfer_distance: x and y need the same number of clouds on one device, got {tuple(x.shape)} "
                         f"on {x.device} and {tuple(y.shape)} on {y.device}")
    out = torch.empty(a.shape[0], device=a.device, dtype=torch.float32)
    _launch(a, b, _abi.CHAMFER_PAIRED, out)
    return out


def chamfer_matrix(a: Tensor, b: Tensor | None = None) -> Tensor:
    """All-pairs Chamfer distances, fp32 ``[Ma, Mb]`` with ``out[i, j] = CD(a[i], b[j])``.  a: ``[Ma, Na, 3]``,
    b: ``[Mb, Nb, 3]``.  ``b=None`` gives the self matrix of ``a``: each pair computed once, exactly symmetric, diagonal
    exactly 0."""
    ta = _clouds(a, "a")
    if b is None:
        out = torch.empty(ta.shape[0], ta.shape[0], device=ta.device, dtype=torch.float32)
        _launch(ta, None, _abi.CHAMFER_SELF, out)
        return out
    tb = _clouds(b, "b")
    if ta.device != tb.device:
        raise ValueError(f"chamfer_matrix: a is on {ta.device}, b on {tb.device}")
    out = torch.empty(ta.shape[0], tb.shape[0], device=ta.device, dtype=torch.float32)
    _launch(ta, tb, _abi.CHAMFER_ALL, out)
    return out


def metrics_from_distances(d_gg: Tensor, d_rr: Tensor, d_gr: Tensor) -> dict:
    """1-NNA, MMD and COV (all over CD) from the three distance matrices: ``d_gg [Mg, Mg]`` among the generated clouds,
    ``d_rr [Mr, Mr]`` among the reference clouds, ``d_gr [Mg, Mr]`` between them.  Definitions and tie rule: module
    docstring.  Works on CPU or GPU tensors (a reduction over small matrices, not a hot path).  Returns Python floats
    ``dict(one_nna=, mmd=, cov=)``."""
    mg, mr = d_gr.shape
    if tuple(d_gg.shape) != (mg, mg) or tuple(d_rr.shape) != (mr, mr):
        raise ValueError(f"metrics_from_distances: shapes {tuple(d_gg.shape)}, {tuple(d_rr.shape)}, {tuple(d_gr.shape)} do "
                         "not fit [Mg, Mg], [Mr, Mr], [Mg, Mr]")
    if mg < 1 or mr < 1 or mg + mr < 2:
        raise ValueError("metrics_from_distances: needs at least one generated and one reference cloud")
    d_gr = d_gr.to(torch.float64)
    # MMD: closest generated cloud of every reference cloud; the sum is correctly rounded (order-free)
    mmd = math.fsum(d_gr.min(dim=0).values.cpu().tolist()) / mr
    # COV: reference clouds that are the nearest (lowest index on ties: torch.argmin) of some generated cloud
    cov = torch.unique(d_gr.argmin(dim=1)).numel() / mr
    # 1-NNA over [S_g; S_r], the cloud itself excluded
    full = torch.cat([torch.cat([d_gg.to(torch.float64), d_gr], 1), torch.cat([d_gr.t(), d_rr.to(torch.float64)], 1)], 0)
    full.fill_diagonal_(math.inf)
    nn = full.argmin(dim=1)
    own = torch.arange(mg + mr, device=full.device) < mg
    one_nna = int(((nn < mg) == own).sum()) / (mg + mr)
    return dict(one_nna=one_nna, mmd=mmd, cov=cov)


def sample_metrics(samples: Tensor, reference: Tensor) -> dict:
    """1-NNA, MMD and COV over CD of generated clouds ``samples [Mg, N, 3]`` against ``reference [Mr, N', 3]`` (float64
    sampler output is cast to fp32 on the device).  Three ``gecco_chamfer`` launches (``S_g x S_g`` and ``S_r x S_r`` as
    self matrices, ``S_g x S_r``), then :func:`metrics_from_distances`."""
    d_gg = chamfer_matrix(samples)
    d_rr = chamfer_matrix(reference)
    d_gr = chamfer_matrix(samples, reference)
    return metrics_from_distances(d_gg, d_rr, d_gr)


__all__ = ["chamfer_distance", "chamfer_matrix", "metrics_from_distances", "sample_metrics"]

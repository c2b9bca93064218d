"""Sample-quality metrics: Chamfer distance (CD) and earth mover's distance (EMD) on the GPU, and the 1-NNA / MMD / COV
numbers built on either.

These are the numbers reported for GECCO and its peers (PointFlow, LION); gecco-jax computes them in ``metrics.py`` /
``benchmark.py``.  The definitions follow PointFlow's ``compute_all_metrics``:

- ``CD(X, Y) = mean_{x in X} min_{y in Y} |x - y|^2 + mean_{y in Y} min_{x in X} |x - y|^2`` -- squared Euclidean
  distances, means (not sums); X and Y may have different point counts.
- ``MMD-CD = mean_{r in S_r} min_{g in S_g} CD(g, r)``.
- ``COV-CD = |{argmin_{r in S_r} CD(g, r) : g in S_g}| / |S_r|``.
- ``1-NNA-CD``: over the union ``[S_g; S_r]`` every cloud's nearest neighbour other than itself; the fraction of clouds whose
  nearest neighbour comes from their own set.  Perfect generation gives 0.5, a generator whose samples are all told apart
  from the reference gives 1.0.
- ``EMD(X, Y)``: the approximate matching of Fan et al. 2017 (``approxmatch`` / ``match_cost`` in PSGN and PointFlow's
  ``StructuralLosses``) divided by N, as PointFlow's ``emd_approx``.  With ``d2[k,l] = |x_k - y_l|^2``, ``dist = sqrt(d2)``,
  ``remL = remR = 1``, ``cost = 0``, for ``j = 7, 6, ..., 0, -1, -2`` and ``e = exp(level * d2)``, ``level = -4^j`` (0 for
  ``j = -2``)::

      ratioL[k] = remL[k] / (1e-9 + sum_l e[k,l] remR[l])
      sumr[l]   = remR[l] sum_k e[k,l] ratioL[k]
      ratioR[l] = min(remR[l] / (sumr[l] + 1e-9), 1) remR[l];   remR[l] = max(0, remR[l] - sumr[l])
      w[k,l]    = e[k,l] ratioL[k] ratioR[l];   remL[k] = max(0, remL[k] - sum_l w[k,l]);   cost += sum w dist
      EMD(X, Y) = cost / N

  It is the literature's number, not the optimal transport cost: it lies above the exact assignment.  X and Y need the
  same point count (at most 4096).  Rows are normalised before columns, so ``EMD(X, Y) != EMD(Y, X)``, and the
  orientation of every matrix is PointFlow's.  PointFlow computes ``M_rs[r, s] = EMD(ref_r, sample_s)`` and the full
  ordered self matrices ``M_rr``, ``M_ss`` (``M[i, j] = EMD(first_i, second_j)``).  MMD / COV take ``M_rs.T``.  1-NNA
  (its ``knn``) takes the nearest neighbour DOWN EACH COLUMN of ``[[M_rr, M_rs], [M_rs.T, M_ss]]``: cloud c is judged by
  ``EMD(other, c)`` within its own set and by ``EMD(ref, sample)`` across the sets.  :func:`metrics_from_distances` takes
  the minimum along rows, so :func:`sample_metrics` passes it ``M_ss.T``, ``M_rr.T`` and ``M_rs.T``.  ``EMD(X, X)`` is
  small but not 0; the self matrix of :func:`emd_matrix` writes its diagonal as 0 (the metrics exclude it).  The levels
  are absolute, so EMD depends on the units of the clouds, like CD.
- ``MMD-EMD``, ``COV-EMD``, ``1-NNA-EMD``: the definitions above with EMD in place of CD.
- Ties: every argmin takes the lowest index; for 1-NNA the index in the concatenation ``[S_g; S_r]`` (PointFlow leaves this
  to ``topk``).
- No normalisation: clouds are compared as given, in data space, which is what the samplers return.  Centring or scaling
  the clouds (PointFlow normalises per shape or globally depending on the table) is the caller's choice.

The CD matrices come from the ``gecco_chamfer`` kernel (``csrc/chamfer.cu``): one block per cloud pair, both
directions in one pass, fp32 arithmetic on clouds translated to the first cloud's bounding-box centre, bitwise
deterministic.  The EMD matrices come from ``gecco_emd`` (``csrc/emd.cu``): one block per cloud pair, fp32, the match
matrix never stored, bitwise deterministic.  CPU tensors are refused (there is no CPU path); ``metrics_from_distances``
is plain torch on the small ``[M, M]`` matrices and takes CPU or GPU tensors.
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


EMD_MAX_POINTS = 4096


def _launch(fn: str, a: Tensor, b: Tensor | None, mode: int, out: Tensor) -> None:
    """Runs the C function ``fn`` (``gecco_chamfer`` or ``gecco_emd``: same arguments) on a's device and stream."""
    lib = _lib_for(a)
    args = _abi.ChamferArgs()
    args.a, args.ma, args.na = a.data_ptr(), a.shape[0], a.shape[1]
    if b is not None:
        args.b, args.mb, args.nb = b.data_ptr(), b.shape[0], b.shape[1]
    args.mode = mode
    args.out = out.data_ptr()
    _abi.check(getattr(lib, fn)(C.byref(args), _stream(a)))


def chamfer_distance(x: Tensor, y: Tensor) -> Tensor:
    """Paired Chamfer distance: ``out[i] = CD(x[i], y[i])``, fp32 ``[B]``.  x: ``[B, Nx, 3]``, y: ``[B, Ny, 3]``."""
    a, b = _clouds(x, "x"), _clouds(y, "y")
    if a.shape[0] != b.shape[0] or a.device != b.device:
        raise ValueError(f"chamfer_distance: x and y need the same number of clouds on one device, got {tuple(x.shape)} "
                         f"on {x.device} and {tuple(y.shape)} on {y.device}")
    out = torch.empty(a.shape[0], device=a.device, dtype=torch.float32)
    _launch("gecco_chamfer", a, b, _abi.CHAMFER_PAIRED, out)
    return out


def chamfer_matrix(a: Tensor, b: Tensor | None = None) -> Tensor:
    """All-pairs Chamfer distances, fp32 ``[Ma, Mb]`` with ``out[i, j] = CD(a[i], b[j])``.  a: ``[Ma, Na, 3]``,
    b: ``[Mb, Nb, 3]``.  ``b=None`` gives the self matrix of ``a``: each pair computed once, exactly symmetric, diagonal
    exactly 0."""
    ta = _clouds(a, "a")
    if b is None:
        out = torch.empty(ta.shape[0], ta.shape[0], device=ta.device, dtype=torch.float32)
        _launch("gecco_chamfer", ta, None, _abi.CHAMFER_SELF, out)
        return out
    tb = _clouds(b, "b")
    if ta.device != tb.device:
        raise ValueError(f"chamfer_matrix: a is on {ta.device}, b on {tb.device}")
    out = torch.empty(ta.shape[0], tb.shape[0], device=ta.device, dtype=torch.float32)
    _launch("gecco_chamfer", ta, tb, _abi.CHAMFER_ALL, out)
    return out


def _emd_points(fn: str, *clouds: tuple[Tensor, str]) -> None:
    """EMD's limits on the point counts, checked on the shapes (before :func:`_clouds`, so CPU tensors get them too):
    equal counts, as PointFlow's ``emd_approx`` asserts, and at most ``EMD_MAX_POINTS``."""
    counts = [(name, t.shape[1]) for t, name in clouds if isinstance(t, Tensor) and t.dim() == 3]
    if len({n for _, n in counts}) > 1:
        raise ValueError(f"{fn}: EMD needs clouds with equal point counts, got " +
                         " and ".join(f"{n} ({name})" for name, n in counts))
    for name, n in counts:
        if n > EMD_MAX_POINTS:
            raise ValueError(f"{fn}: {name}: EMD takes clouds of at most {EMD_MAX_POINTS} points, got {n}")


def emd_distance(x: Tensor, y: Tensor) -> Tensor:
    """Paired approximate EMD: ``out[i] = EMD(x[i], y[i])``, fp32 ``[B]``.  x, y: ``[B, N, 3]`` with the same N (at most
    4096).  Definition and orientation: module docstring."""
    _emd_points("emd_distance", (x, "x"), (y, "y"))
    a, b = _clouds(x, "x"), _clouds(y, "y")
    if a.shape[0] != b.shape[0] or a.device != b.device:
        raise ValueError(f"emd_distance: x and y need the same number of clouds on one device, got {tuple(x.shape)} "
                         f"on {x.device} and {tuple(y.shape)} on {y.device}")
    out = torch.empty(a.shape[0], device=a.device, dtype=torch.float32)
    _launch("gecco_emd", a, b, _abi.CHAMFER_PAIRED, out)
    return out


def emd_matrix(a: Tensor, b: Tensor | None = None) -> Tensor:
    """All-pairs approximate EMD, fp32 ``[Ma, Mb]`` with ``out[i, j] = EMD(a[i], b[j])`` (not symmetric).
    a: ``[Ma, N, 3]``, b: ``[Mb, N, 3]``, the same N (at most 4096).  ``b=None`` gives the self matrix of ``a``: every
    ordered pair ``i != j``, bitwise equal to ``emd_matrix(a, a)`` there; the diagonal is not computed and is exactly 0."""
    _emd_points("emd_matrix", (a, "a"), (b, "b"))
    ta = _clouds(a, "a")
    if b is None:
        out = torch.empty(ta.shape[0], ta.shape[0], device=ta.device, dtype=torch.float32)
        _launch("gecco_emd", ta, None, _abi.CHAMFER_SELF, out)
        return out
    tb = _clouds(b, "b")
    if ta.device != tb.device:
        raise ValueError(f"emd_matrix: a is on {ta.device}, b on {tb.device}")
    out = torch.empty(ta.shape[0], tb.shape[0], device=ta.device, dtype=torch.float32)
    _launch("gecco_emd", ta, tb, _abi.CHAMFER_ALL, out)
    return out


def metrics_from_distances(d_gg: Tensor, d_rr: Tensor, d_gr: Tensor) -> dict:
    """1-NNA, MMD and COV from the three distance matrices (CD or EMD): ``d_gg [Mg, Mg]`` among the generated clouds,
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


def sample_metrics(samples: Tensor, reference: Tensor, distance: str = "cd") -> dict:
    """1-NNA, MMD and COV of generated clouds ``samples [Mg, N, 3]`` against ``reference [Mr, N', 3]`` (float64 sampler
    output is cast to fp32 on the device), over ``distance``:

    - ``"cd"``: three ``gecco_chamfer`` launches (``S_g x S_g`` and ``S_r x S_r`` as self matrices, ``S_g x S_r``);
    - ``"emd"``: three ``gecco_emd`` launches in PointFlow's orientation (module docstring): ``emd_matrix(samples).T``,
      ``emd_matrix(reference).T`` and ``emd_matrix(reference, samples).T``; N' must equal N (at most 4096).

    then :func:`metrics_from_distances`."""
    if distance == "cd":
        d_gg = chamfer_matrix(samples)
        d_rr = chamfer_matrix(reference)
        d_gr = chamfer_matrix(samples, reference)
    elif distance == "emd":
        _emd_points("sample_metrics", (samples, "samples"), (reference, "reference"))
        # transposed: metrics_from_distances looks along rows, PointFlow's knn down the columns of the ordered matrices
        d_gg = emd_matrix(samples).t()
        d_rr = emd_matrix(reference).t()
        d_gr = emd_matrix(reference, samples).t()
    else:
        raise ValueError(f"sample_metrics: distance must be 'cd' or 'emd', got {distance!r}")
    return metrics_from_distances(d_gg, d_rr, d_gr)


__all__ = ["chamfer_distance", "chamfer_matrix", "emd_distance", "emd_matrix", "metrics_from_distances", "sample_metrics"]

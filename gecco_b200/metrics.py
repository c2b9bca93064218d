"""Sample-quality metrics: Chamfer distance (CD), approximate and exact earth mover's distance (EMD, EMD*) on the GPU,
and the 1-NNA / MMD / COV numbers built on any of them; per-point nearest neighbours and the per-cloud F-score / paired
CD of conditional reconstructions; the exact optimal matching of paired clouds.

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
- ``EMD*(X, Y) = min over permutations s of (1/N) sum_i |x_i - y_s(i)|``: the exact earth mover's distance, the optimal
  assignment between clouds of the same N points (at most 4096), with the Euclidean distance (not its square) as the
  cost.  It is what gecco-jax's ``metrics.py`` computes with scipy's ``linear_sum_assignment``.  EMD* is symmetric,
  ``EMD*(X, X) = 0``, and ``EMD* <= EMD`` pair by pair (the approximate matching is one transport plan).  The
  ``gecco_emd_exact`` kernel finds it by a forward auction with epsilon scaling down to ``eps = 2^-20 D``, D the
  bounding-box diagonal of the pair, and certifies it: the reported value is the cost of the permutation found (rounded
  up), and the final prices give a dual bound ``lower`` (rounded down) with ``lower <= OPT <= emd`` on the fp32 costs and
  ``emd - lower <= 2^-20 D`` up to the rounding of the bids.  Against the exact distances the bounds widen by
  ``6 * 2^-24 D`` (``include/gecco_b200.h``).  Ties: equal bids go to the lowest point of the first cloud, equal values
  to the lowest point of the second; results are bitwise deterministic.  ``MMD-EMD*``, ``COV-EMD*`` and ``1-NNA-EMD*``
  are the definitions above with EMD* in place of CD; its matrices are symmetric, so they have no orientation to choose.
- Ties: every argmin takes the lowest index; for 1-NNA the index in the concatenation ``[S_g; S_r]`` (PointFlow leaves this
  to ``topk``).
- No normalisation: clouds are compared as given, in data space, which is what the samplers return.  Centring or scaling
  the clouds (PointFlow normalises per shape or globally depending on the table) is the caller's choice.

Conditional outputs (single-view reconstruction, inpainting, upsampling) each have their own ground-truth cloud and are
scored per sample, as in Tatarchenko et al. 2019 ("What do single-view 3D reconstruction networks learn?"):

- :func:`nearest_neighbours` gives, for every point of ``x`` and of ``y``, the index of its nearest point in the other
  cloud of the pair and the squared distance to it.  Ties go to the lowest index, as everywhere in this module.
- With ``d_xy`` the squared distances from the prediction to the target and ``d_yx`` those back, and a threshold ``tau``
  (a distance, in the units of the clouds): ``precision(tau) = mean_i [d_xy[i] < tau^2]``,
  ``recall(tau) = mean_j [d_yx[j] < tau^2]`` (strict, compared in float64), ``F(tau) = 2 P R / (P + R)`` and
  ``F = 0`` when ``P + R = 0``.
- ``reconstruction_metrics(...)["cd"]`` is the CD defined above, the same number :func:`chamfer_distance` computes, with
  different arithmetic: the distance to every chosen neighbour is recomputed in fp32 difference form and the means are
  taken in float64, where ``gecco_chamfer`` sums the fp32 expansion's minima; the tests hold the two to 1e-4
  relative.  ``gecco_nearest`` has no point cap below 2^24 per cloud, where ``gecco_chamfer``
  refuses pairs whose clouds both exceed 32768 points.

The CD matrices come from the ``gecco_chamfer`` kernel (``csrc/chamfer.cu``): one block per cloud pair, both
directions in one pass, fp32 arithmetic on clouds translated to the first cloud's bounding-box centre, bitwise
deterministic.  The EMD matrices come from ``gecco_emd`` (``csrc/emd.cu``): one block per cloud pair, fp32, the match
matrix never stored, bitwise deterministic.  The exact EMD comes from ``gecco_emd_exact`` (``csrc/emd_exact.cu``): one
block per cloud pair, the costs recomputed on the fly, bitwise deterministic.  The nearest neighbours come from
``gecco_nearest`` (``csrc/nearest.cu``): many blocks per pair, both directions in one pass, merged with 64-bit integer
minima, bitwise deterministic; its error bound is stated in ``include/gecco_b200.h``.  CPU tensors are refused (there is
no CPU path); ``metrics_from_distances`` is plain torch on the small ``[M, M]`` matrices and takes CPU or GPU tensors.
"""
from __future__ import annotations

import ctypes as C
import math
import numbers
from typing import NamedTuple, Sequence

import numpy as np
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


class OptimalMatching(NamedTuple):
    """Result of :func:`optimal_matching`: the exact EMD (fp32 ``[B]``, the cost of the permutation found, rounded up),
    its certified lower bound (fp32 ``[B]``, rounded down) and the permutation (int64 ``[B, N]``, ``idx[b, i]`` the
    point of ``y[b]`` matched to ``x[b, i]``)."""
    emd: Tensor
    lower: Tensor
    idx: Tensor


def _launch_exact(a: Tensor, b: Tensor | None, mode: int, out: Tensor, lower: Tensor | None = None,
                  match: Tensor | None = None) -> None:
    """Runs ``gecco_emd_exact``; a pair whose auction did not finish (NaN in ``out``) raises GeccoError naming it."""
    lib = _lib_for(a)
    args = _abi.EmdExactArgs()
    args.a, args.ma, args.na = a.data_ptr(), a.shape[0], a.shape[1]
    if b is not None:
        args.b, args.mb, args.nb = b.data_ptr(), b.shape[0], b.shape[1]
    args.mode = mode
    args.out = out.data_ptr()
    args.lower = lower.data_ptr() if lower is not None else None
    args.match = match.data_ptr() if match is not None else None
    _abi.check(lib.gecco_emd_exact(C.byref(args), _stream(a)))
    bad = torch.isnan(out).nonzero().tolist()
    if bad:
        shown = ", ".join(str(tuple(p)) if len(p) > 1 else str(p[0]) for p in bad[:10]) + (", ..." if len(bad) > 10 else "")
        raise _abi.GeccoError(f"gecco_emd_exact: the auction did not finish for {len(bad)} cloud pair(s): {shown}")


def optimal_matching(x: Tensor, y: Tensor) -> OptimalMatching:
    """Paired exact EMD with its certificate and permutation: ``emd[b] = EMD*(x[b], y[b])``, ``lower[b]`` the dual
    bound, ``idx[b]`` the optimal permutation found.  x, y: ``[B, N, 3]`` with the same N (at most 4096) on one CUDA
    device (float64 sampler output is cast to fp32 on the device).  Definition, certificate and tie rule: module
    docstring."""
    for t, name in ((x, "x"), (y, "y")):
        if not isinstance(t, Tensor):
            raise TypeError(f"{name}: expected a tensor, got {type(t).__name__}")
    if x.dim() == 3 and y.dim() == 3 and (x.shape[0] != y.shape[0] or x.device != y.device):
        raise ValueError(f"optimal_matching: x and y need the same number of clouds on one device, got {tuple(x.shape)} "
                         f"on {x.device} and {tuple(y.shape)} on {y.device}")
    _emd_points("optimal_matching", (x, "x"), (y, "y"))
    a, b = _clouds(x, "x"), _clouds(y, "y")
    dev, m, n = a.device, a.shape[0], a.shape[1]
    out = OptimalMatching(torch.empty(m, device=dev, dtype=torch.float32), torch.empty(m, device=dev, dtype=torch.float32),
                          torch.empty(m, n, device=dev, dtype=torch.int32))
    _launch_exact(a, b, _abi.CHAMFER_PAIRED, out.emd, out.lower, out.idx)
    return out._replace(idx=out.idx.long())


def emd_exact_matrix(a: Tensor, b: Tensor | None = None) -> Tensor:
    """All-pairs exact EMD, fp32 ``[Ma, Mb]`` with ``out[i, j] = EMD*(a[i], b[j])`` (the upper value of the
    certificate).  a: ``[Ma, N, 3]``, b: ``[Mb, N, 3]``, the same N (at most 4096).  ``b=None`` gives the self matrix of
    ``a``: each pair computed once, exactly symmetric, diagonal exactly 0."""
    _emd_points("emd_exact_matrix", (a, "a"), (b, "b"))
    ta = _clouds(a, "a")
    if b is None:
        out = torch.empty(ta.shape[0], ta.shape[0], device=ta.device, dtype=torch.float32)
        _launch_exact(ta, None, _abi.CHAMFER_SELF, out)
        return out
    tb = _clouds(b, "b")
    if ta.device != tb.device:
        raise ValueError(f"emd_exact_matrix: a is on {ta.device}, b on {tb.device}")
    out = torch.empty(ta.shape[0], tb.shape[0], device=ta.device, dtype=torch.float32)
    _launch_exact(ta, tb, _abi.CHAMFER_ALL, out)
    return out


NEAREST_MAX_POINTS = 1 << 24


class NearestNeighbours(NamedTuple):
    """Result of :func:`nearest_neighbours`: squared fp32 distances and int64 indices, ``[B, Nx]`` / ``[B, Ny]``."""
    dist_xy: Tensor
    idx_xy: Tensor
    dist_yx: Tensor
    idx_yx: Tensor


def nearest_neighbours(x: Tensor, y: Tensor) -> NearestNeighbours:
    """Nearest neighbours within each cloud pair, both directions: ``idx_xy[b, i] = argmin_j |x[b, i] - y[b, j]|^2``
    (lowest j on ties) and ``dist_xy[b, i]`` the squared distance to it; ``idx_yx`` / ``dist_yx`` from y to x.
    x: ``[B, Nx, 3]``, y: ``[B, Ny, 3]`` on one CUDA device, 1 to 2^24 points per cloud (float64 sampler output is cast
    to fp32 on the device).  Distances are fp32, recomputed in difference form for the chosen neighbour; the bound on
    how far they can lie above the exact minimum is stated in ``include/gecco_b200.h``."""
    for t, name in ((x, "x"), (y, "y")):
        if not isinstance(t, Tensor):
            raise TypeError(f"{name}: expected a tensor, got {type(t).__name__}")
    if x.dim() == 3 and y.dim() == 3 and (x.shape[0] != y.shape[0] or x.device != y.device):
        raise ValueError(f"nearest_neighbours: x and y need the same number of clouds on one device, got {tuple(x.shape)} "
                         f"on {x.device} and {tuple(y.shape)} on {y.device}")
    for t, name in ((x, "x"), (y, "y")):
        if t.dim() == 3 and t.shape[1] > NEAREST_MAX_POINTS:
            raise ValueError(f"nearest_neighbours: {name}: at most {NEAREST_MAX_POINTS} points per cloud, got {t.shape[1]}")
    a, b = _clouds(x, "x"), _clouds(y, "y")
    clouds, nx, ny = a.shape[0], a.shape[1], b.shape[1]
    lib = _lib_for(a)
    dev = a.device
    f32, i32 = torch.float32, torch.int32
    out = NearestNeighbours(torch.empty(clouds, nx, device=dev, dtype=f32), torch.empty(clouds, nx, device=dev, dtype=i32),
                            torch.empty(clouds, ny, device=dev, dtype=f32), torch.empty(clouds, ny, device=dev, dtype=i32))
    nbytes = lib.gecco_nearest_scratch_bytes(clouds, nx, ny)
    scratch = torch.empty((nbytes + 7) // 8, device=dev, dtype=torch.int64)
    args = _abi.NearestArgs()
    args.x, args.y = a.data_ptr(), b.data_ptr()
    args.clouds, args.nx, args.ny = clouds, nx, ny
    args.dist_xy, args.idx_xy = out.dist_xy.data_ptr(), out.idx_xy.data_ptr()
    args.dist_yx, args.idx_yx = out.dist_yx.data_ptr(), out.idx_yx.data_ptr()
    args.scratch, args.scratch_bytes = scratch.data_ptr(), nbytes
    _abi.check(lib.gecco_nearest(C.byref(args), _stream(a)))
    return out._replace(idx_xy=out.idx_xy.long(), idx_yx=out.idx_yx.long())


def _thresholds(thresholds) -> list[float]:
    """A non-empty sequence (or 1-D tensor / numpy array) of positive finite numbers (distances, in the units of the
    clouds) -> floats."""
    if isinstance(thresholds, (Tensor, np.ndarray)):  # 1-D arrays, e.g. np.linspace(0.005, 0.02, 4)
        thresholds = thresholds.tolist() if thresholds.ndim == 1 else None
    if not isinstance(thresholds, Sequence) or isinstance(thresholds, (str, bytes)) or len(thresholds) == 0:
        raise ValueError(f"reconstruction_metrics: thresholds must be a non-empty sequence of distances, got {thresholds!r}")
    out = []
    for t in thresholds:
        if isinstance(t, bool) or not isinstance(t, numbers.Real) or not math.isfinite(t) or t <= 0:
            raise ValueError(f"reconstruction_metrics: thresholds must be positive finite numbers, got {t!r}")
        out.append(float(t))
    return out


def reconstruction_metrics(pred: Tensor, target: Tensor, thresholds: Sequence[float]) -> dict:
    """Per-cloud scores of conditional outputs against their own ground truth: pred ``[B, Np, 3]``, target
    ``[B, Nt, 3]``, thresholds: distances tau in the units of the clouds (no default: the module does not normalise
    clouds).  Returns float64 tensors ``cd [B]`` (mean of ``dist_xy`` plus mean of ``dist_yx``) and ``precision``,
    ``recall``, ``fscore [B, T]`` (definitions: module docstring).  Averages over a test set, or the best of several
    samples per input, are the caller's to take."""
    th = _thresholds(thresholds)
    nn = nearest_neighbours(pred, target)
    d_xy, d_yx = nn.dist_xy.double(), nn.dist_yx.double()
    tau2 = torch.tensor([t * t for t in th], dtype=torch.float64, device=d_xy.device)
    precision = (d_xy[:, :, None] < tau2).sum(1).double() / d_xy.shape[1]
    recall = (d_yx[:, :, None] < tau2).sum(1).double() / d_yx.shape[1]
    s = precision + recall
    fscore = torch.where(s > 0, 2 * precision * recall / torch.where(s > 0, s, 1.0), 0.0)
    return dict(cd=d_xy.mean(1) + d_yx.mean(1), precision=precision, recall=recall, fscore=fscore)


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
      ``emd_matrix(reference).T`` and ``emd_matrix(reference, samples).T``; N' must equal N (at most 4096);
    - ``"emd_exact"``: three ``gecco_emd_exact`` launches, ``emd_exact_matrix(samples)``, ``emd_exact_matrix(reference)``
      and ``emd_exact_matrix(samples, reference)``; N' must equal N (at most 4096).  EMD* is symmetric, so unlike
      ``"emd"`` there is no orientation to choose;

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
    elif distance == "emd_exact":
        _emd_points("sample_metrics", (samples, "samples"), (reference, "reference"))
        d_gg = emd_exact_matrix(samples)
        d_rr = emd_exact_matrix(reference)
        d_gr = emd_exact_matrix(samples, reference)
    else:
        raise ValueError(f"sample_metrics: distance must be 'cd', 'emd' or 'emd_exact', got {distance!r}")
    return metrics_from_distances(d_gg, d_rr, d_gr)


__all__ = ["chamfer_distance", "chamfer_matrix", "emd_distance", "emd_matrix", "metrics_from_distances", "sample_metrics",
           "NearestNeighbours", "nearest_neighbours", "reconstruction_metrics", "OptimalMatching", "optimal_matching",
           "emd_exact_matrix"]

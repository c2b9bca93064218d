"""Reference restatements of the approximate earth mover's distance of gecco_b200/metrics.py, written independently of it.

The definition (Fan et al. 2017 ``approxmatch`` / ``match_cost``, divided by N as PointFlow's ``emd_approx``): for clouds
X = {x_k}, Y = {y_l} of N points, ``d2[k,l] = |x_k - y_l|^2``, ``dist = sqrt(d2)``, ``remL = remR = 1``, ``cost = 0``::

    for j = 7, 6, ..., 0, -1, -2:       level = -4**j (0 for j = -2),  e[k,l] = exp(level * d2[k,l])
        ratioL[k] = remL[k] / (1e-9 + sum_l e[k,l] * remR[l])
        sumr[l]   = remR[l] * sum_k e[k,l] * ratioL[k]
        ratioR[l] = min(remR[l] / (sumr[l] + 1e-9), 1) * remR[l]
        remR[l]   = max(0, remR[l] - sumr[l])
        w[k,l]    = e[k,l] * ratioL[k] * ratioR[l]
        remL[k]   = max(0, remL[k] - sum_l w[k,l])
        cost     += sum_{k,l} w[k,l] * dist[k,l]
    EMD(X, Y) = cost / N

- ``emd_matrix_f64``: the three passes per level exactly as written (not the fused schedule of the kernel), float64 torch
  on the input's device, vectorised over a chunk of cloud pairs.
- ``approxmatch_loops``: explicit per-element loops in numpy, one accumulator per row or column, for tiny N only: an
  independent check of the vectorised restatement.
"""
from __future__ import annotations

import math

import numpy as np
import torch

LEVELS = [-(4.0 ** j) for j in range(7, -2, -1)] + [0.0]


def _approxmatch(x: torch.Tensor, y: torch.Tensor) -> tuple[torch.Tensor, torch.Tensor]:
    """x, y ``[c, N, 3]`` float64 -> (cost / N, transported mass) per pair, ``[c]`` each."""
    d2 = (x[:, :, None, :] - y[:, None, :, :]).pow(2).sum(-1)  # [c, N, N]
    dist = d2.sqrt()
    c, n = x.shape[:2]
    rem_l = torch.ones(c, n, dtype=x.dtype, device=x.device)
    rem_r = torch.ones(c, n, dtype=x.dtype, device=x.device)
    cost = torch.zeros(c, dtype=x.dtype, device=x.device)
    mass = torch.zeros(c, dtype=x.dtype, device=x.device)
    for level in LEVELS:
        e = torch.exp(level * d2)
        ratio_l = rem_l / (1e-9 + (e * rem_r[:, None, :]).sum(2))
        sumr = rem_r * (e * ratio_l[:, :, None]).sum(1)
        ratio_r = torch.clamp(rem_r / (sumr + 1e-9), max=1.0) * rem_r
        rem_r = (rem_r - sumr).clamp_min(0.0)
        w = e * ratio_l[:, :, None] * ratio_r[:, None, :]
        rem_l = (rem_l - w.sum(2)).clamp_min(0.0)
        cost = cost + (w * dist).sum((1, 2))
        mass = mass + w.sum((1, 2))
    return cost / n, mass


def emd_matrix_f64(a: torch.Tensor, b: torch.Tensor | None = None, return_mass: bool = False,
                   chunk_elems: int = 1 << 24):
    """``out[i, j] = EMD(a[i], b[j])`` for a ``[Ma, N, 3]``, b ``[Mb, N, 3]``, float64 on a's device.  b=None: the ordered
    self matrix of a with the diagonal set to 0 (as the kernel's self mode).  return_mass: also the transported mass
    ``sum_{k,l} w`` of every pair (at most N)."""
    self_mode = b is None
    a = a.to(torch.float64)
    b = a if b is None else b.to(device=a.device, dtype=torch.float64)
    ma, n = a.shape[:2]
    mb = b.shape[0]
    if b.shape[1] != n:
        raise ValueError(f"emd_matrix_f64: equal point counts needed, got {n} and {b.shape[1]}")
    out = torch.zeros(ma, mb, dtype=torch.float64, device=a.device)
    mass = torch.zeros(ma, mb, dtype=torch.float64, device=a.device)
    pairs = [(i, j) for i in range(ma) for j in range(mb) if not (self_mode and i == j)]
    step = max(1, chunk_elems // (n * n))
    for p0 in range(0, len(pairs), step):
        ii = torch.tensor([p[0] for p in pairs[p0:p0 + step]], device=a.device)
        jj = torch.tensor([p[1] for p in pairs[p0:p0 + step]], device=a.device)
        cost, moved = _approxmatch(a[ii], b[jj])
        out[ii, jj] = cost
        mass[ii, jj] = moved
    return (out, mass) if return_mass else out


def approxmatch_loops(x: np.ndarray, y: np.ndarray) -> float:
    """EMD(x, y) for x, y ``[N, 3]`` by explicit loops over the definition (tiny N only)."""
    x = np.asarray(x, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64)
    n = len(x)
    assert len(y) == n
    d2 = [[sum((x[k][c] - y[l][c]) ** 2 for c in range(3)) for l in range(n)] for k in range(n)]
    dist = [[math.sqrt(d2[k][l]) for l in range(n)] for k in range(n)]
    rem_l = [1.0] * n
    rem_r = [1.0] * n
    cost = 0.0
    for level in LEVELS:
        e = [[math.exp(level * d2[k][l]) for l in range(n)] for k in range(n)]
        ratio_l = []
        for k in range(n):
            s = 0.0
            for l in range(n):
                s += e[k][l] * rem_r[l]
            ratio_l.append(rem_l[k] / (1e-9 + s))
        ratio_r = []
        for l in range(n):
            s = 0.0
            for k in range(n):
                s += e[k][l] * ratio_l[k]
            sumr = rem_r[l] * s
            ratio_r.append(min(rem_r[l] / (sumr + 1e-9), 1.0) * rem_r[l])
            rem_r[l] = max(0.0, rem_r[l] - sumr)
        for k in range(n):
            s = 0.0
            for l in range(n):
                w = e[k][l] * ratio_l[k] * ratio_r[l]
                s += w
                cost += w * dist[k][l]
            rem_l[k] = max(0.0, rem_l[k] - s)
    return cost / n


def pointflow_knn_one_nna(m_rr: np.ndarray, m_rs: np.ndarray, m_ss: np.ndarray) -> float:
    """PointFlow's ``knn(M_rr, M_rs, M_ss, 1)`` accuracy restated column by column, for ordered (non-symmetric) matrices
    ``M[i, j] = d(first_i, second_j)``: ``M = [[M_rr, M_rs], [M_rs.T, M_ss]]`` with the reference clouds first (label 1),
    the diagonal excluded, and the nearest neighbour of cloud c the row of the smallest entry of COLUMN c (``topk(1, 0)``;
    lowest row on ties)."""
    m_rr, m_rs, m_ss = (np.asarray(m, dtype=np.float64) for m in (m_rr, m_rs, m_ss))
    n0, n1 = m_rs.shape
    label = [1] * n0 + [0] * n1
    m = np.block([[m_rr, m_rs], [m_rs.T, m_ss]])
    correct = 0
    for c in range(n0 + n1):
        best, nearest = math.inf, -1
        for r in range(n0 + n1):
            if r != c and m[r, c] < best:
                best, nearest = m[r, c], r
        correct += label[nearest] == label[c]
    return correct / (n0 + n1)

"""Reference restatement of the sample-quality metrics (gecco_b200/metrics.py), written independently of it.

- ``chamfer_matrix_f64``: Chamfer distance in float64 torch from the direct ``(x - y)^2`` (no expansion, no centring),
  chunked so that the ``[chunk, Na, Nb]`` difference tensor stays small.
- ``knn_one_nna`` / ``lgan_mmd_cov``: numpy restatements of PointFlow's ``knn`` (k = 1) and ``lgan_mmd_cov``
  (``metrics/evaluation_metrics.py``), with the tie rule pinned to the lowest index (``np.argmin``) and the union taken
  in the order ``[S_g; S_r]``.
"""
from __future__ import annotations

import math

import numpy as np
import torch


def chamfer_matrix_f64(a: torch.Tensor, b: torch.Tensor | None = None, chunk_elems: int = 1 << 25) -> torch.Tensor:
    """``out[i, j] = mean_x min_y |x - y|^2 + mean_y min_x |x - y|^2`` for a ``[Ma, Na, 3]``, b ``[Mb, Nb, 3]`` (b=None: a
    against itself), float64 on a's device."""
    a = a.to(torch.float64)
    b = a if b is None else b.to(device=a.device, dtype=torch.float64)
    ma, na = a.shape[:2]
    mb, nb = b.shape[:2]
    out = torch.empty(ma, mb, dtype=torch.float64, device=a.device)
    step = max(1, chunk_elems // (na * nb * 3))
    for i in range(ma):
        x = a[i]
        for j0 in range(0, mb, step):
            y = b[j0:j0 + step]                                        # [c, Nb, 3]
            d = (x[None, :, None, :] - y[:, None, :, :]).pow(2).sum(-1)  # [c, Na, Nb]
            out[i, j0:j0 + step] = d.min(2).values.mean(1) + d.min(1).values.mean(1)
    return out


def lgan_mmd_cov(d_gr: np.ndarray) -> tuple[float, float]:
    """PointFlow ``lgan_mmd_cov`` on ``d_gr [Mg, Mr]``: (MMD, COV)."""
    d = np.asarray(d_gr, dtype=np.float64)
    mg, mr = d.shape
    nearest_ref = np.argmin(d, axis=1)     # for every generated cloud (lowest index on ties)
    closest_gen = np.min(d, axis=0)        # for every reference cloud
    mmd = math.fsum(closest_gen.tolist()) / mr
    cov = len(set(nearest_ref.tolist())) / mr
    return mmd, cov


def knn_one_nna(d_gg: np.ndarray, d_rr: np.ndarray, d_gr: np.ndarray) -> float:
    """PointFlow ``knn(..., k=1)`` accuracy: 1-NN classifier over the union ``[S_g; S_r]``, leave-one-out."""
    d_gg, d_rr, d_gr = (np.asarray(m, dtype=np.float64) for m in (d_gg, d_rr, d_gr))
    mg, mr = d_gr.shape
    label = np.concatenate([np.ones(mg), np.zeros(mr)])
    m = np.block([[d_gg, d_gr], [d_gr.T, d_rr]])
    m = m + np.diag(np.full(mg + mr, np.inf))
    idx = np.argmin(m, axis=1)
    pred = label[idx]
    return float(np.sum(pred == label)) / (mg + mr)


def metrics(d_gg, d_rr, d_gr) -> dict:
    mmd, cov = lgan_mmd_cov(d_gr)
    return dict(one_nna=knn_one_nna(d_gg, d_rr, d_gr), mmd=mmd, cov=cov)

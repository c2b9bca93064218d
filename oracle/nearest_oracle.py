"""Reference restatement of the per-point reconstruction metrics (gecco_b200/metrics.py: nearest_neighbours,
reconstruction_metrics), written independently of them.

- ``nearest_f64``: nearest neighbours of paired clouds in float64 torch from the direct ``(x - y)^2`` (no expansion, no
  centring), chunked over rows so that it runs at 16384 x 65536 points on a GPU.  ``torch.argmin`` / ``topk`` take the
  lowest index on ties.
- ``fscore_np``: precision / recall / F-score at thresholds tau (Tatarchenko et al. 2019) in numpy, F = 0 where P + R = 0.
"""
from __future__ import annotations

import numpy as np
import torch


def nearest_f64(x: torch.Tensor, y: torch.Tensor, chunk_elems: int = 1 << 25, second: bool = False):
    """x ``[B, Nx, 3]``, y ``[B, Ny, 3]`` -> ``(d_xy, i_xy, d_yx, i_yx)``: float64 squared distances and int64 indices,
    on x's device.  ``second=True`` appends the float64 distances to the second nearest point of each direction
    (``inf`` where the other cloud has one point)."""
    x = x.to(torch.float64)
    y = y.to(device=x.device, dtype=torch.float64)
    bsz, nx, ny = x.shape[0], x.shape[1], y.shape[1]
    dev = x.device
    d_xy = torch.empty(bsz, nx, dtype=torch.float64, device=dev)
    s_xy = torch.full((bsz, nx), float("inf"), dtype=torch.float64, device=dev)
    i_xy = torch.empty(bsz, nx, dtype=torch.int64, device=dev)
    d_yx = torch.full((bsz, ny), float("inf"), dtype=torch.float64, device=dev)
    s_yx = torch.full((bsz, ny), float("inf"), dtype=torch.float64, device=dev)
    i_yx = torch.zeros(bsz, ny, dtype=torch.int64, device=dev)
    step = max(1, chunk_elems // (ny * 3))
    for b in range(bsz):
        for i0 in range(0, nx, step):
            d = (x[b, i0:i0 + step, None, :] - y[b, None, :, :]).pow(2).sum(-1)  # [c, Ny]
            k = min(2, ny)
            v, i = d.topk(k, dim=1, largest=False, sorted=True)
            d_xy[b, i0:i0 + step], i_xy[b, i0:i0 + step] = v[:, 0], d.argmin(1)
            if k == 2:
                s_xy[b, i0:i0 + step] = v[:, 1]
            # y -> x: merge the chunk's column minima into the running ones; chunks come in row order, so a strict "<"
            # keeps the lower row on ties
            kc = min(2, d.shape[0])
            cv = d.topk(kc, dim=0, largest=False, sorted=True).values
            cmin, carg = cv[0], d.argmin(0) + i0
            old = d_yx[b].clone()
            better = cmin < old
            s_yx[b] = torch.where(better, torch.minimum(old, cv[1] if kc == 2 else torch.full_like(old, float("inf"))),
                                  torch.minimum(s_yx[b], cmin))
            d_yx[b] = torch.where(better, cmin, old)
            i_yx[b] = torch.where(better, carg, i_yx[b])
    out = (d_xy, i_xy, d_yx, i_yx)
    return out + (s_xy, s_yx) if second else out


def fscore_np(d_xy, d_yx, thresholds) -> tuple[np.ndarray, np.ndarray, np.ndarray]:
    """Precision, recall and F-score ``[B, T]`` from squared distances ``d_xy [B, Nx]`` (prediction -> target) and
    ``d_yx [B, Ny]`` (target -> prediction): ``P = mean(d_xy < tau^2)``, ``R = mean(d_yx < tau^2)``,
    ``F = 2PR / (P + R)``, 0 where ``P + R = 0``."""
    d_xy = np.atleast_2d(np.asarray(d_xy, dtype=np.float64))
    d_yx = np.atleast_2d(np.asarray(d_yx, dtype=np.float64))
    p = np.empty((d_xy.shape[0], len(thresholds)))
    r = np.empty_like(p)
    f = np.zeros_like(p)
    for t, tau in enumerate(thresholds):
        t2 = float(tau) * float(tau)
        p[:, t] = np.count_nonzero(d_xy < t2, axis=1) / d_xy.shape[1]
        r[:, t] = np.count_nonzero(d_yx < t2, axis=1) / d_yx.shape[1]
    for b in range(p.shape[0]):
        for t in range(p.shape[1]):
            if p[b, t] + r[b, t] > 0:
                f[b, t] = 2 * p[b, t] * r[b, t] / (p[b, t] + r[b, t])
    return p, r, f

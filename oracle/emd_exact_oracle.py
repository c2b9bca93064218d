"""Reference for the exact earth mover's distance of gecco_b200/metrics.py, written independently of the kernel.

For clouds X, Y of the same N points: ``EMD*(X, Y) = min over permutations s of (1/N) sum_i |x_i - y_s(i)|``, with the
Euclidean distance (not its square) as the cost.  Everything here is float64 on the CPU.

- ``lsa``: scipy's ``cdist`` and ``linear_sum_assignment`` per pair, returning the cost and the assignment; this is how
  gecco-jax's ``metrics.py`` computes EMD.
- ``emd_exact_matrix_f64``: ``lsa`` over all pairs (or the self matrix, each pair once, diagonal 0).
- ``brute_force``: the minimum over all N! permutations, for N <= 7: an independent check of ``lsa``.
"""
from __future__ import annotations

import itertools

import numpy as np
import torch
from scipy.optimize import linear_sum_assignment
from scipy.spatial.distance import cdist


def _np(t) -> np.ndarray:
    return t.detach().to("cpu", torch.float64).numpy() if isinstance(t, torch.Tensor) else np.asarray(t, np.float64)


def lsa(x, y) -> tuple[float, np.ndarray]:
    """EMD*(x, y) of one pair ([N, 3] each) and the optimal assignment ``sigma`` (int64 [N], ``sigma[i]`` the point of y
    matched to x[i])."""
    x, y = _np(x), _np(y)
    if x.shape != y.shape or x.ndim != 2 or x.shape[1] != 3:
        raise ValueError(f"lsa: expected two [N, 3] clouds of one size, got {x.shape} and {y.shape}")
    c = cdist(x, y)
    rows, cols = linear_sum_assignment(c)
    sigma = np.empty(x.shape[0], np.int64)
    sigma[rows] = cols
    return float(c[rows, cols].sum() / x.shape[0]), sigma


def lsa_batch(x, y) -> tuple[np.ndarray, np.ndarray]:
    """Paired: costs [B] and assignments [B, N] of x[b] against y[b]."""
    x, y = _np(x), _np(y)
    res = [lsa(x[b], y[b]) for b in range(x.shape[0])]
    return np.array([r[0] for r in res]), np.stack([r[1] for r in res])


def emd_exact_matrix_f64(a, b=None) -> np.ndarray:
    """``out[i, j] = EMD*(a[i], b[j])``; ``b=None``: the self matrix of a, each pair once, exactly symmetric, diagonal 0."""
    a = _np(a)
    if b is None:
        m = a.shape[0]
        out = np.zeros((m, m))
        for i in range(m):
            for j in range(i + 1, m):
                out[i, j] = out[j, i] = lsa(a[i], a[j])[0]
        return out
    b = _np(b)
    return np.array([[lsa(a[i], b[j])[0] for j in range(b.shape[0])] for i in range(a.shape[0])])


def brute_force(x, y) -> tuple[float, tuple[int, ...]]:
    """EMD*(x, y) by trying every permutation (N <= 7), and the first permutation (in lexicographic order) reaching it."""
    x, y = _np(x), _np(y)
    n = x.shape[0]
    if n > 7:
        raise ValueError(f"brute_force: at most 7 points, got {n}")
    c = np.sqrt(((x[:, None, :] - y[None, :, :]) ** 2).sum(-1))
    best, arg = np.inf, None
    for perm in itertools.permutations(range(n)):
        s = sum(c[i, perm[i]] for i in range(n))
        if s < best:
            best, arg = s, perm
    return best / n, arg

"""CPU checks of the approximate earth mover's distance: the float64 oracle (oracle/emd_oracle.py) against its explicit-loop
restatement, properties of the definition (single points, permutations, transported mass, a lower bound from the exact
assignment, orientation), PointFlow's 1-NNA orientation on ordered matrices, and the input checks of the GPU entry
points."""
import numpy as np
import pytest
import torch
from scipy.optimize import linear_sum_assignment
from scipy.spatial.distance import cdist

from gecco_b200 import _abi
from gecco_b200.metrics import emd_distance, emd_matrix, metrics_from_distances, sample_metrics
from oracle import emd_oracle as EO
from oracle import metrics_oracle as MO


def _pair(seed, n, scale=1.0, shift=0.2):
    g = torch.Generator().manual_seed(seed)
    a = torch.randn(1, n, 3, generator=g, dtype=torch.float64) * scale
    b = torch.randn(1, n, 3, generator=g, dtype=torch.float64) * scale * 0.8 + shift
    return a, b


@pytest.mark.parametrize("n", [2, 3, 7, 16, 40])
def test_oracle_matches_explicit_loops(n):
    g = torch.Generator().manual_seed(n)
    a = torch.randn(3, n, 3, generator=g, dtype=torch.float64)
    b = torch.randn(2, n, 3, generator=g, dtype=torch.float64) * 0.7 + 0.3
    m = EO.emd_matrix_f64(a, b, chunk_elems=2 * n * n)  # small chunks exercise the chunk loop
    for i in range(3):
        for j in range(2):
            assert m[i, j].item() == pytest.approx(EO.approxmatch_loops(a[i].numpy(), b[j].numpy()), rel=1e-12)
    s = EO.emd_matrix_f64(a)
    assert torch.all(s.diagonal() == 0)
    assert s[0, 1].item() == pytest.approx(EO.approxmatch_loops(a[0].numpy(), a[1].numpy()), rel=1e-12)


def test_single_point_is_the_distance():
    g = torch.Generator().manual_seed(3)
    a = torch.randn(4, 1, 3, generator=g, dtype=torch.float64)
    b = torch.randn(5, 1, 3, generator=g, dtype=torch.float64) * 2
    m = EO.emd_matrix_f64(a, b)
    want = (a[:, None, 0, :] - b[None, :, 0, :]).norm(dim=-1)
    assert torch.allclose(m, want, rtol=1e-8, atol=0)


def test_permutations_change_nothing():
    a, b = _pair(4, 48)
    base = EO.emd_matrix_f64(a, b).item()
    g = torch.Generator().manual_seed(5)
    pa, pb = torch.randperm(48, generator=g), torch.randperm(48, generator=g)
    assert EO.emd_matrix_f64(a[:, pa], b).item() == pytest.approx(base, rel=1e-12)
    assert EO.emd_matrix_f64(a, b[:, pb]).item() == pytest.approx(base, rel=1e-12)


@pytest.mark.parametrize("seed,n,scale,shift", [(0, 64, 1.0, 0.2), (1, 200, 1.0, 0.2), (2, 256, 0.05, 0.0),
                                                (3, 96, 0.5, 10.0)])
def test_mass_and_lower_bound_from_the_exact_assignment(seed, n, scale, shift):
    a, b = _pair(seed, n, scale, shift)
    emd, mass = EO.emd_matrix_f64(a, b, return_mass=True)
    emd, mass = emd.item(), mass.item()
    assert abs(mass - n) < 1e-6, mass - n
    d = cdist(a[0].numpy(), b[0].numpy())
    rows, cols = linear_sum_assignment(d)
    exact = d[rows, cols].sum()
    # w is a partial plan (row and column sums <= 1); completing it moves N - mass more at most the diameter each, and no
    # complete plan costs less than the optimal assignment
    assert emd * n >= exact - (n - mass) * d.max() - 1e-9 * exact
    assert emd * n > exact  # the approximate matching is not optimal on these clouds


def test_orientation_matters():
    # rows are normalised before columns: EMD(a, b) != EMD(b, a); the GPU orientation tests rely on pairs like this one
    a, b = _pair(0, 64)
    ab, ba = EO.emd_matrix_f64(a, b).item(), EO.emd_matrix_f64(b, a).item()
    assert abs(ab - ba) / ab > 1e-3, (ab, ba)


def _one_nna(m_ss, m_rr, m_rs, transpose_self):
    """1-NNA of metrics_from_distances on PointFlow's ordered matrices, the self blocks transposed (as sample_metrics
    passes them for EMD) or not."""
    t = (lambda m: m.t()) if transpose_self else (lambda m: m)
    return metrics_from_distances(t(m_ss), t(m_rr), m_rs.t())["one_nna"]


def test_pointflow_knn_restatement():
    # symmetric matrices: the column-wise restatement agrees with the row-wise one of the CD metrics
    rng = np.random.default_rng(0)
    pts = rng.normal(size=(17, 4))
    full = ((pts[:, None] - pts[None]) ** 2).sum(-1)
    d_gg, d_rr, d_gr = full[:9, :9], full[9:, 9:], full[:9, 9:]
    assert EO.pointflow_knn_one_nna(d_rr, d_gr.T, d_gg) == MO.knn_one_nna(d_gg, d_rr, d_gr)
    # ordered matrices: only the transposed self blocks give PointFlow's number
    differs = 0
    for seed in range(6):
        rng = np.random.default_rng(seed)
        m_ss, m_rr, m_rs = rng.random((10, 10)), rng.random((8, 8)), rng.random((8, 10))
        want = EO.pointflow_knn_one_nna(m_rr, m_rs, m_ss)
        args = [torch.from_numpy(m) for m in (m_ss, m_rr, m_rs)]
        assert _one_nna(*args, transpose_self=True) == want
        differs += _one_nna(*args, transpose_self=False) != want
    assert differs >= 3


def test_emd_one_nna_orientation_on_near_tie_sets():
    # identically distributed sets: nearest-neighbour decisions are close, and EMD(a, b) != EMD(b, a) decides some of them
    differs = 0
    for seed in range(4):
        g = torch.Generator().manual_seed(seed)
        gen = torch.randn(12, 32, 3, generator=g, dtype=torch.float64)
        ref = torch.randn(12, 32, 3, generator=g, dtype=torch.float64)
        m_ss, m_rr, m_rs = EO.emd_matrix_f64(gen), EO.emd_matrix_f64(ref), EO.emd_matrix_f64(ref, gen)
        want = EO.pointflow_knn_one_nna(m_rr.numpy(), m_rs.numpy(), m_ss.numpy())
        assert _one_nna(m_ss, m_rr, m_rs, transpose_self=True) == want
        differs += _one_nna(m_ss, m_rr, m_rs, transpose_self=False) != want
    assert differs >= 2


def test_gpu_entry_points_check_their_input():
    x = torch.randn(3, 16, 3, dtype=torch.float64)
    with pytest.raises(_abi.GeccoError):
        emd_matrix(x)
    with pytest.raises(_abi.GeccoError):
        emd_matrix(x.float(), x.float())
    with pytest.raises(_abi.GeccoError):
        emd_distance(x, x)
    bad = x.clone()
    bad[1, 3, 2] = float("nan")
    bad[2, 0, 0] = float("inf")
    with pytest.raises(ValueError, match=r"2 cloud\(s\) with non-finite points \(indices 1, 2\)"):
        emd_matrix(bad)
    with pytest.raises(ValueError, match=r"indices 1, 2"):
        emd_distance(bad, x)
    with pytest.raises(ValueError, match="equal point counts"):
        emd_matrix(x, torch.randn(2, 17, 3))
    with pytest.raises(ValueError, match="equal point counts"):
        emd_distance(x, torch.randn(3, 15, 3))
    with pytest.raises(ValueError, match="equal point counts"):
        sample_metrics(x, torch.randn(2, 17, 3), distance="emd")
    with pytest.raises(ValueError, match="at most 4096"):
        emd_matrix(torch.zeros(1, 4097, 3))
    with pytest.raises(ValueError, match="at most 4096"):
        emd_distance(torch.zeros(2, 4097, 3), torch.zeros(2, 4097, 3))
    with pytest.raises(ValueError, match="distance must be"):
        sample_metrics(x, x, distance="l2")

"""CPU checks of the sample-quality metrics: the float64 Chamfer oracle against brute force and a k-d tree, the metric
reductions of gecco_b200.metrics against the independent numpy restatement (ties included), hand-made cases with known
answers, and the input checks of the GPU entry points."""
import numpy as np
import pytest
import torch
from scipy.spatial import cKDTree

from gecco_b200 import _abi
from gecco_b200.metrics import chamfer_distance, chamfer_matrix, metrics_from_distances
from oracle import metrics_oracle as MO


def _brute_cd(x: np.ndarray, y: np.ndarray) -> float:
    d = ((x[:, None, :] - y[None, :, :]) ** 2).sum(-1)
    return d.min(1).mean() + d.min(0).mean()


def _kdtree_cd(x: np.ndarray, y: np.ndarray) -> float:
    dxy, _ = cKDTree(y).query(x, k=1)
    dyx, _ = cKDTree(x).query(y, k=1)
    return (dxy ** 2).mean() + (dyx ** 2).mean()


def test_oracle_chamfer_matches_brute_force_and_kdtree():
    g = torch.Generator().manual_seed(0)
    a = torch.randn(3, 37, 3, generator=g, dtype=torch.float64)
    b = torch.randn(4, 53, 3, generator=g, dtype=torch.float64) * 1.5 + 0.3
    m = MO.chamfer_matrix_f64(a, b, chunk_elems=4000)  # small chunks exercise the chunk loop
    for i in range(3):
        for j in range(4):
            x, y = a[i].numpy(), b[j].numpy()
            assert m[i, j].item() == pytest.approx(_brute_cd(x, y), rel=1e-12)
            assert m[i, j].item() == pytest.approx(_kdtree_cd(x, y), rel=1e-9)
    s = MO.chamfer_matrix_f64(a)
    assert torch.equal(s, s.t()) and torch.all(s.diagonal() == 0)


def _random_case(seed, mg, mr, ties):
    rng = np.random.default_rng(seed)
    pts = rng.normal(size=(mg + mr, 4))
    full = ((pts[:, None] - pts[None]) ** 2).sum(-1)
    if ties:  # quantise so that equal distances are common
        full = np.round(full * 2) / 2
    d_gg, d_rr, d_gr = full[:mg, :mg].copy(), full[mg:, mg:].copy(), full[:mg, mg:].copy()
    np.fill_diagonal(d_gg, 0.0)
    np.fill_diagonal(d_rr, 0.0)
    return d_gg, d_rr, d_gr


@pytest.mark.parametrize("seed,mg,mr,ties", [(0, 7, 9, False), (1, 16, 16, False), (2, 12, 10, True), (3, 30, 25, True),
                                             (4, 1, 5, False), (5, 6, 1, True)])
def test_metrics_from_distances_matches_oracle(seed, mg, mr, ties):
    d_gg, d_rr, d_gr = _random_case(seed, mg, mr, ties)
    ref = MO.metrics(d_gg, d_rr, d_gr)
    for dt in (torch.float64, torch.float32):
        got = metrics_from_distances(*(torch.from_numpy(m).to(dt) for m in (d_gg, d_rr, d_gr)))
        ref_dt = MO.metrics(*(torch.from_numpy(m).to(dt).double().numpy() for m in (d_gg, d_rr, d_gr)))
        assert got == ref_dt, (got, ref_dt)
    assert metrics_from_distances(*(torch.from_numpy(m) for m in (d_gg, d_rr, d_gr))) == ref


def test_ties_take_the_lowest_index():
    # every generated cloud is equally close to references 1 and 2 -> all pick 1; COV = 1/3
    d_gr = torch.tensor([[5.0, 1.0, 1.0], [4.0, 1.0, 1.0]])
    d_gg = torch.tensor([[0.0, 9.0], [9.0, 0.0]])
    d_rr = torch.tensor([[0.0, 9.0, 9.0], [9.0, 0.0, 9.0], [9.0, 9.0, 0.0]])
    out = metrics_from_distances(d_gg, d_rr, d_gr)
    assert out["cov"] == pytest.approx(1 / 3) and out["cov"] == MO.metrics(d_gg, d_rr, d_gr)["cov"]
    # 1-NNA tie across the sets: generated cloud 0 is at 1.0 from generated cloud 1 and from reference 0; in [S_g; S_r]
    # order the generated one (index 1) wins
    d_gg = torch.tensor([[0.0, 1.0], [1.0, 0.0]])
    d_gr = torch.tensor([[1.0, 7.0], [8.0, 8.0]])
    d_rr = torch.tensor([[0.0, 8.0], [8.0, 0.0]])
    nn_same = metrics_from_distances(d_gg, d_rr, d_gr)["one_nna"]
    assert nn_same == MO.knn_one_nna(d_gg.numpy(), d_rr.numpy(), d_gr.numpy())
    # cloud 0 -> g1 (tie, lowest index), g1 -> g0, r0 -> g0 (1.0), r1 -> g0 / g1 / r0 all 7 / 8 / 8 -> g0: 2 of 4 correct
    assert nn_same == 0.5


def test_separated_sets_known_answers():
    # generated clouds around x = 0, reference clouds around x = 100: every nearest neighbour is in the own set
    g = torch.Generator().manual_seed(1)
    gen = torch.randn(5, 20, 3, generator=g, dtype=torch.float64)
    ref = torch.randn(4, 24, 3, generator=g, dtype=torch.float64)
    ref[..., 0] += 100.0
    d_gg, d_rr, d_gr = MO.chamfer_matrix_f64(gen), MO.chamfer_matrix_f64(ref), MO.chamfer_matrix_f64(gen, ref)
    out = metrics_from_distances(d_gg, d_rr, d_gr)
    assert out["one_nna"] == 1.0
    # COV by hand: nearest reference of each generated cloud
    picked = {int(torch.argmin(d_gr[i])) for i in range(5)}
    assert out["cov"] == len(picked) / 4
    # identical sets: every cloud's nearest other cloud is its copy in the other set -> 1-NNA 0, COV 1, MMD 0
    same = metrics_from_distances(d_gg, d_gg, d_gg)
    assert same == dict(one_nna=0.0, mmd=0.0, cov=1.0)


def test_metrics_from_distances_checks_shapes():
    with pytest.raises(ValueError):
        metrics_from_distances(torch.zeros(3, 3), torch.zeros(2, 2), torch.zeros(3, 3))


def test_gpu_entry_points_refuse_cpu_and_non_finite_input():
    x = torch.randn(3, 16, 3, dtype=torch.float64)
    with pytest.raises(_abi.GeccoError):
        chamfer_matrix(x)
    with pytest.raises(_abi.GeccoError):
        chamfer_matrix(x.float(), x.float())
    with pytest.raises(_abi.GeccoError):
        chamfer_distance(x, x)
    bad = x.clone()
    bad[1, 3, 2] = float("nan")
    bad[2, 0, 0] = float("inf")
    with pytest.raises(ValueError, match=r"2 cloud\(s\) with non-finite points \(indices 1, 2\)"):
        chamfer_matrix(bad)
    with pytest.raises(ValueError, match=r"indices 1, 2"):
        chamfer_matrix(bad, x)
    with pytest.raises(ValueError, match="shape"):
        chamfer_matrix(torch.zeros(2, 5, 2))

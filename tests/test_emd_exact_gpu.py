"""The exact earth mover's distance kernel (csrc/emd_exact.cu) on the GPU: the certified bounds against scipy's assignment
in float64 (oracle/emd_exact_oracle.py) within the cost-rounding term stated in include/gecco_b200.h, the permutation,
point counts from 1 to 4096, ties and lattices, bitwise agreement of the three modes and of repeated runs, the bound
from gecco_emd, the set metrics, and float64 and sampler output fed straight in."""
import numpy as np
import pytest
import torch

from oracle import emd_exact_oracle as XO
from oracle import metrics_oracle as MO

pytestmark = pytest.mark.gpu

U = 2.0 ** -24


def _clouds(seed, m, n, scale=1.0, offset=(0.0, 0.0, 0.0)):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(m, n, 3, generator=g) * scale + torch.tensor(offset)


def _diag(x, y):
    """D per pair: the diagonal of the bounding box of both clouds, float64 [B]."""
    both = torch.cat([x, y], 1).double()
    return (both.amax(1) - both.amin(1)).norm(dim=-1).cpu()


def _tol(x, y):
    """The header's cost-rounding term 6 * 2^-24 D per pair."""
    return 6 * U * _diag(x, y)


def _check(x, y, got=None):
    """Bounds, gap, permutation and its cost against the float64 assignment; returns (oracle costs, got)."""
    from gecco_b200.metrics import optimal_matching

    got = optimal_matching(x, y) if got is None else got
    assert got.emd.dtype == torch.float32 and got.lower.dtype == torch.float32 and got.idx.dtype == torch.int64
    assert got.idx.shape == x.shape[:2]
    want, _ = XO.lsa_batch(x, y)
    want = torch.from_numpy(want)
    up, lo = got.emd.double().cpu(), got.lower.double().cpu()
    tol, eps = _tol(x, y), 2.0 ** -20 * _diag(x, y)
    assert (lo - tol <= want).all() and (want <= up + tol).all(), (lo - want, up - want, tol)
    assert (up - lo <= eps + tol).all(), ((up - lo) / eps).max().item()
    idx = got.idx.cpu()
    assert torch.equal(idx.sort(1).values, torch.arange(x.shape[1]).expand_as(idx))  # a permutation
    xd, yd = x.double().cpu(), y.double().cpu()
    cost = (xd - torch.gather(yd, 1, idx[..., None].expand(-1, -1, 3))).norm(dim=-1).mean(1)
    assert ((cost - up).abs() <= tol + up * 2.0 ** -23).all(), (cost - up).abs().max().item()
    nz = want > 0
    assert ((up - want).abs()[nz] <= 1e-4 * want[nz]).all(), ((up - want).abs()[nz] / want[nz]).max().item()
    return want, got


def test_bounds_16_pairs(cuda):
    from gecco_b200.metrics import emd_distance

    x = torch.cat([_clouds(1, 8, 2048), _clouds(2, 4, 2048, 0.05), _clouds(3, 4, 2048, 0.5, (0.0, 0.0, 5.0))]).to(cuda)
    y = torch.cat([_clouds(4, 8, 2048, 0.8, (0.1, 0.0, 0.0)), _clouds(5, 4, 2048, 0.05, (0.01, 0.0, 0.0)),
                   _clouds(6, 4, 2048, 0.6, (0.2, -0.1, 5.0))]).to(cuda)
    want, got = _check(x, y)
    rel = ((got.emd.double().cpu() - want) / want).abs().max().item()
    gap = ((got.emd - got.lower).double().cpu() / want).max().item()
    print(f"exact EMD 16 x 2048: max rel diff to the assignment {rel:.2e}, max certified rel gap {gap:.2e}")
    # the approximate matching is one transport plan: never below the certified lower bound
    approx = emd_distance(x, y)
    assert (approx >= got.lower).all()


@pytest.mark.parametrize("n", [1, 2, 3, 31, 32, 33, 1000, 2047, 2048, 2049, 4096])
def test_sizes(cuda, n):
    x = _clouds(100 + n, 2, n).to(cuda)
    y = _clouds(200 + n, 2, n, 0.9, (0.1, 0.0, 0.0)).to(cuda)
    want, got = _check(x, y)
    if n == 1:  # one point each: the distance itself
        d = (x - y).double().norm(dim=-1)[:, 0].cpu()
        assert torch.allclose(got.emd.double().cpu(), d, rtol=1e-6, atol=0) and (got.idx == 0).all()


def _lattice(k, spacing=0.1):
    ax = torch.arange(k, dtype=torch.float64) * spacing
    return torch.stack(torch.meshgrid(ax, ax, ax, indexing="ij"), -1).reshape(-1, 3)


def test_ties_and_price_wars(cuda):
    from gecco_b200.metrics import optimal_matching

    g = torch.Generator().manual_seed(7)
    # identical clouds, permuted: 0 within eps (exactly 0 once the identity is found)
    x = _clouds(8, 3, 1500).to(cuda)
    y = x[:, torch.randperm(1500, generator=g).to(cuda)]
    got = optimal_matching(x, y)
    eps = 2.0 ** -20 * _diag(x, y)
    assert (got.emd.double().cpu() <= eps).all() and (got.lower.double().cpu() <= 0 + _tol(x, y)).all()
    # a cloud of one repeated point against itself: exactly 0
    p = torch.full((2, 777, 3), 0.25, device=cuda)
    rep = optimal_matching(p, p)
    assert (rep.emd == 0).all() and (rep.lower == 0).all()
    assert torch.equal(rep.idx.sort(1).values, torch.arange(777, device=cuda).expand(2, -1))
    # one repeated point against another: every permutation is optimal, every bid ties
    q = torch.full((1, 48, 3), -0.5, device=cuda)
    tie = optimal_matching(p[:1, :48], q)
    d = torch.tensor(0.75 * 3 ** 0.5, dtype=torch.float64)
    assert abs(tie.emd.double().item() - d.item()) <= 1e-6 and tie.lower.double().item() <= d + 1e-6
    # lattices: many equal costs; a 12^3 grid against itself shifted by half a spacing, and against a permuted copy
    lat = _lattice(12)
    perm = lat[torch.randperm(lat.shape[0], generator=g)]
    shifted = lat[torch.randperm(lat.shape[0], generator=g)] + torch.tensor([0.05, 0.0, 0.0], dtype=torch.float64)
    xs = torch.stack([lat, lat]).float().to(cuda)
    ys = torch.stack([shifted, perm]).float().to(cuda)
    want, got = _check(xs, ys)
    assert got.emd[1].item() <= 2.0 ** -20 * _diag(xs, ys)[1].item()


def test_modes_agree_and_runs_repeat(cuda):
    from gecco_b200.metrics import emd_exact_matrix, optimal_matching

    a = torch.cat([_clouds(20, 4, 700), _clouds(21, 2, 700, 0.3, (0.0, 0.0, 5.0))]).to(cuda)
    b = _clouds(22, 3, 700, 0.8).to(cuda)
    full = emd_exact_matrix(a, a)
    self_m = emd_exact_matrix(a)
    assert torch.equal(self_m, self_m.t()) and (self_m.diagonal() == 0).all()
    iu = torch.triu_indices(6, 6, 1, device=cuda)
    assert torch.equal(self_m[iu[0], iu[1]], full[iu[0], iu[1]])  # a[i] the persons, i < j, in both
    pm = optimal_matching(a[:5], a[1:])
    assert torch.equal(pm.emd, full[torch.arange(5), torch.arange(1, 6)])
    cross = emd_exact_matrix(a, b)
    pb = optimal_matching(a[:3], b)
    assert torch.equal(pb.emd, cross[torch.arange(3), torch.arange(3)])
    # symmetric up to the certified bound: the other orientation is another auction on the same optimum
    other = emd_exact_matrix(b, a).t()
    tol = 2.0 ** -20 * 2 * max(_diag(a[i:i + 1], b[j:j + 1]).item() for i in range(6) for j in range(3))
    assert ((cross - other).abs() <= tol).all()
    # repeated runs: identical bits, indices and lower bounds included
    again = optimal_matching(a[:5], a[1:])
    assert all(torch.equal(u, v) for u, v in zip(pm, again))
    assert torch.equal(emd_exact_matrix(a), self_m) and torch.equal(emd_exact_matrix(a, b), cross)


def test_sample_metrics_emd_exact_matches_oracle(cuda):
    from gecco_b200.metrics import sample_metrics

    g = torch.Generator().manual_seed(0)
    # two slightly different families, so that the nearest-neighbour decisions are clear
    gen = (torch.randn(12, 256, 3, generator=g) * torch.linspace(0.8, 1.2, 12)[:, None, None]).double()
    ref = (torch.randn(12, 256, 3, generator=g) * torch.linspace(0.85, 1.25, 12)[:, None, None] + 0.05).double()
    d_gg = XO.emd_exact_matrix_f64(gen)
    d_rr = XO.emd_exact_matrix_f64(ref)
    d_gr = XO.emd_exact_matrix_f64(gen, ref)
    # every argmin decision has a margin larger than twice the certified bound of an entry (eps_final + tol)
    both = torch.cat([gen, ref]).float()
    lo, hi = both.double().amin((0, 1)), both.double().amax((0, 1))
    bound = (2.0 ** -20 + 6 * U) * (hi - lo).norm().item()
    full = np.block([[d_gg, d_gr], [d_gr.T, d_rr]])
    np.fill_diagonal(full, np.inf)
    for m, axis in ((d_gr, 0), (d_gr, 1), (full, 1)):
        s = np.sort(m, axis=axis)
        margin = (np.take(s, 1, axis=axis) - np.take(s, 0, axis=axis)).min()
        assert margin > 2 * bound, (margin, bound)
    want = MO.metrics(d_gg, d_rr, d_gr)
    got = sample_metrics(gen.to(cuda), ref.to(cuda), distance="emd_exact")
    print("sample_metrics(distance='emd_exact')", got, "oracle", want)
    assert got["one_nna"] == want["one_nna"] and got["cov"] == want["cov"]
    assert abs(got["mmd"] - want["mmd"]) <= bound
    assert sample_metrics(gen.to(cuda), ref.to(cuda)) == sample_metrics(gen.to(cuda), ref.to(cuda), distance="cd")


def test_float64_input(cuda):
    from gecco_b200.metrics import emd_exact_matrix, optimal_matching

    x, y = _clouds(30, 3, 900).to(cuda), _clouds(31, 3, 900, 0.9).to(cuda)
    a, b = optimal_matching(x.double(), y.double()), optimal_matching(x, y)
    assert all(torch.equal(u, v) for u, v in zip(a, b))
    assert torch.equal(emd_exact_matrix(x.double()), emd_exact_matrix(x))
    before = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        c = optimal_matching(x, y)
    finally:
        torch.set_default_dtype(before)
    assert c.emd.dtype == torch.float32 and all(torch.equal(u, v) for u, v in zip(c, b))


def test_conditional_sampler_output_feeds_the_exact_emd(cuda):
    import gecco_b200 as G
    from tests import synth
    from tests.models_b200 import build

    B, N = 2, 384
    feats = synth.synth_features(B, (34, 17, 8), 21)
    rp = synth.SHAPENET_VOL_REPARAM
    sd = synth.tame(synth.full_state_dict("cond", "gaussian", rp["mean"], rp["sigma"], 1234), 0.15)
    model = build("cond", "gaussian", rp["mean"], rp["sigma"], 165.0, None, cuda, feats, state_dict=sd)
    ctx = G.Context3d(image=torch.zeros(B, 3, 8, 8, device=cuda), K=synth.camera(B, synth.K_SHAPENET).to(cuda))
    samples = model.sample_stochastic((B, N, 3), ctx, rng=synth.gen(7), num_steps=4)
    assert samples.dtype == torch.float64 and samples.is_cuda
    g = torch.Generator(device=cuda).manual_seed(3)
    target = samples + 0.01 * torch.randn(samples.shape, device=cuda, dtype=torch.float64, generator=g)
    got = G.optimal_matching(samples, target)
    _check(samples.float(), target.float(), got)
    m = G.sample_metrics(samples, target, distance="emd_exact")
    assert 0.0 <= m["one_nna"] <= 1.0 and 0.0 < m["cov"] <= 1.0 and m["mmd"] >= 0.0

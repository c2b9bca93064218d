"""The nearest-neighbour kernel (csrc/nearest.cu) and the per-cloud reconstruction metrics on the GPU: distances and
indices against the float64 direct oracle (oracle/nearest_oracle.py) within the error bound stated in
include/gecco_b200.h, ties, shapes past the Chamfer kernel's cap, determinism, agreement with gecco_chamfer, the F-score
against its numpy restatement, and sampler output fed straight in."""
import numpy as np
import pytest
import torch

from oracle import nearest_oracle as NO

pytestmark = pytest.mark.gpu

U = 2.0 ** -24


def _clouds(seed, m, n, scale=1.0, offset=(0.0, 0.0, 0.0)):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(m, n, 3, generator=g) * scale + torch.tensor(offset)


def _bound(x, y, d_min):
    """The header's bound B = 2^-13 d* + 72 u R^2 per point; R about the kernel's centre (fp32 bounding-box centre of x)."""
    c = (0.5 * (x.amin(1) + x.amax(1))).double()[:, None, :]
    r2 = torch.maximum((x.double() - c).pow(2).sum(-1).amax(1), (y.double() - c).pow(2).sum(-1).amax(1))
    return 2.0 ** -13 * d_min + 72 * U * r2[:, None]


def _check(x, y, got=None):
    """Both directions against the oracle: reported distances and the float64 distance to every returned index within
    the bound of the minimum, indices exact wherever the second neighbour is more than twice the bound away.  Returns the
    fraction of points whose index equals the oracle's."""
    from gecco_b200.metrics import nearest_neighbours

    got = nearest_neighbours(x, y) if got is None else got
    d_xy, i_xy, d_yx, i_yx, s_xy, s_yx = NO.nearest_f64(x, y, second=True)
    same = []
    for dist, idx, d_ref, i_ref, s_ref, p, q in ((got.dist_xy, got.idx_xy, d_xy, i_xy, s_xy, x, y),
                                                 (got.dist_yx, got.idx_yx, d_yx, i_yx, s_yx, y, x)):
        assert dist.dtype == torch.float32 and idx.dtype == torch.int64 and dist.shape == d_ref.shape
        b = _bound(x, y, d_ref)
        assert ((dist.double() - d_ref).abs() <= b).all(), ((dist.double() - d_ref).abs() / b).max().item()
        assert idx.min() >= 0 and idx.max() < q.shape[1]
        chosen = (p.double() - torch.gather(q.double(), 1, idx[..., None].expand(-1, -1, 3))).pow(2).sum(-1)
        assert (chosen - d_ref <= b).all()
        clear = s_ref - d_ref > 2 * b
        assert torch.equal(idx[clear], i_ref[clear])
        same.append((idx == i_ref).double().mean().item())
    return same


def test_parity_16_pairs(cuda):
    x = torch.cat([_clouds(1, 12, 2048), _clouds(2, 4, 2048, 0.5, (0.0, 0.0, 5.0))]).to(cuda)  # 4 pairs around z = 5
    y = torch.cat([_clouds(3, 12, 2048, 0.8), _clouds(4, 4, 2048, 1.0, (0.2, -0.1, 5.0))]).to(cuda)
    same = _check(x, y)
    print("nearest 16 x 2048 x 2048: index equals the oracle's for", same)
    assert min(same) > 0.99


def test_ties_take_the_lowest_index(cuda):
    from gecco_b200.metrics import nearest_neighbours

    g = torch.Generator().manual_seed(11)
    x = torch.rand(2, 1000, 3, generator=g) * 2 - 1
    y = torch.rand(2, 1500, 3, generator=g) * 2 - 1
    y[:, 500:600] = x[:, 0:100]    # coincident with x points: distance 0 ...
    y[:, 900:1000] = x[:, 0:100]   # ... twice: index 500 + i must win
    y[:, 1200:1300] = y[:, 100:200]  # plain duplicates in y
    x[:, 300:400] = x[:, 0:100]    # duplicates in x: y -> x must take x[i], not x[300 + i]
    x, y = x.to(cuda), y.to(cuda)
    d_xy, i_xy, d_yx, i_yx, s_xy, s_yx = NO.nearest_f64(x, y, second=True)
    # precondition: every other candidate of a coincident point is further than the bound, so only exact ties compete
    far = lambda d2: (d2 > _bound(x, y, torch.zeros_like(d2)) * 2)
    other_x = (x[:, 0:100, None, :].double() - y.double()[:, None, :, :]).pow(2).sum(-1)
    other_x[:, torch.arange(100), torch.arange(100) + 500] = 1.0
    other_x[:, torch.arange(100), torch.arange(100) + 900] = 1.0
    assert far(other_x.amin(2)).all()
    got = nearest_neighbours(x, y)
    ar = torch.arange(100, device=cuda)
    assert torch.equal(got.idx_xy[:, 0:100], (ar + 500).expand(2, -1)) and torch.all(got.dist_xy[:, 0:100] == 0)
    assert torch.equal(got.idx_xy[:, 300:400], (ar + 500).expand(2, -1)) and torch.all(got.dist_xy[:, 300:400] == 0)
    assert torch.equal(got.idx_yx[:, 500:600], ar.expand(2, -1)) and torch.all(got.dist_yx[:, 500:600] == 0)
    assert torch.equal(got.idx_yx[:, 900:1000], ar.expand(2, -1)) and torch.all(got.dist_yx[:, 900:1000] == 0)
    # the duplicated y columns: whichever x point is nearest, it is the same for both copies and never a higher copy
    assert torch.equal(got.idx_yx[:, 1200:1300], got.idx_yx[:, 100:200])
    assert not ((got.idx_xy >= 1200) & (got.idx_xy < 1300)).any()
    assert not ((got.idx_xy >= 900) & (got.idx_xy < 1000)).any()
    _check(x, y, got)


@pytest.mark.parametrize("clouds,nx,ny", [(2, 1, 1), (2, 1, 33), (2, 33, 1), (2, 2047, 33), (2, 3000, 5000),
                                          (2, 2048, 16384), (2, 16384, 65536), (1, 100000, 2048)])
def test_shapes(cuda, clouds, nx, ny):
    x = _clouds(10 + nx, clouds, nx).to(cuda)
    y = _clouds(20 + ny, clouds, ny, 0.9, (0.1, 0.0, 0.0)).to(cuda)
    _check(x, y)


def test_deterministic_and_float64_input(cuda):
    from gecco_b200.metrics import nearest_neighbours

    x, y = _clouds(30, 2, 16384).to(cuda), _clouds(31, 2, 65536, 0.9).to(cuda)
    a, b = nearest_neighbours(x, y), nearest_neighbours(x, y)
    assert all(torch.equal(u, v) for u, v in zip(a, b))
    xs, ys = x[:, :3000], y[:, :5000]
    c, d = nearest_neighbours(xs.double(), ys.double()), nearest_neighbours(xs, ys)
    assert all(torch.equal(u, v) for u, v in zip(c, d))


def test_float64_default_dtype(cuda):
    # the output buffers are fp32 whatever torch's default dtype is (samplers return float64, users may set it)
    from gecco_b200.metrics import nearest_neighbours, reconstruction_metrics

    x, y = _clouds(50, 2, 700).to(cuda), _clouds(51, 2, 900, 0.9).to(cuda)
    want = nearest_neighbours(x, y)
    before = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        got = nearest_neighbours(x, y)
        rec = reconstruction_metrics(x, y, [0.05, 0.1])
    finally:
        torch.set_default_dtype(before)
    assert got.dist_xy.dtype == torch.float32 and got.dist_yx.dtype == torch.float32
    assert all(torch.equal(u, v) for u, v in zip(got, want))
    d_xy, _, d_yx, _ = NO.nearest_f64(x, y)
    assert torch.allclose(rec["cd"], d_xy.mean(1) + d_yx.mean(1), rtol=1e-5, atol=0)
    p, r, f = NO.fscore_np(want.dist_xy.double().cpu().numpy(), want.dist_yx.double().cpu().numpy(), [0.05, 0.1])
    np.testing.assert_array_equal(rec["fscore"].cpu().numpy(), f)
    _check(x, y, got)


def test_cd_agrees_with_chamfer_kernel(cuda):
    from gecco_b200.metrics import chamfer_distance, reconstruction_metrics

    x = torch.cat([_clouds(41, 12, 2048), _clouds(42, 4, 2048, 0.5, (0.0, 0.0, 5.0))]).to(cuda)
    y = torch.cat([_clouds(43, 12, 2048, 0.8), _clouds(44, 4, 2048, 1.0, (0.2, -0.1, 5.0))]).to(cuda)
    cd = reconstruction_metrics(x, y, [0.01])["cd"]
    assert cd.dtype == torch.float64 and cd.shape == (16,)
    ch = chamfer_distance(x, y).double()
    rel = ((cd - ch).abs() / ch).max().item()
    print(f"reconstruction cd against gecco_chamfer: max rel diff {rel:.2e}")
    assert rel < 1e-4
    d_xy, _, d_yx, _ = NO.nearest_f64(x, y)
    ref = d_xy.mean(1) + d_yx.mean(1)
    allowed = _bound(x, y, d_xy).mean(1) + _bound(x, y, d_yx).mean(1)
    assert ((cd - ref).abs() <= allowed).all()


def _grid_pair(seed, n=2048, kept=1900, offset=(0.0, 0.0, 0.0)):
    """Target: a jittered 13^3 grid in the unit cube (2197 points, spacing 1/13, at least 0.057 apart).  Prediction, n
    points: `kept` target points moved by 0.003, 0.007 or 0.014, plus outliers above the cube.  Every nearest-neighbour
    distance then sits well away from the thresholds 0.005, 0.01, 0.02."""
    g = torch.Generator().manual_seed(seed)
    ax = (torch.arange(13, dtype=torch.float64) + 0.5) / 13 - 0.5
    grid = torch.stack(torch.meshgrid(ax, ax, ax, indexing="ij"), -1).reshape(-1, 3)
    target = grid[torch.randperm(grid.shape[0], generator=g)]
    target = target + (torch.rand(target.shape, generator=g, dtype=torch.float64) - 0.5) * 0.02
    step = torch.tensor([0.003, 0.007, 0.014], dtype=torch.float64)[torch.randint(0, 3, (kept,), generator=g)]
    v = torch.randn(kept, 3, generator=g, dtype=torch.float64)
    moved = target[:kept] + v / v.norm(dim=1, keepdim=True) * step[:, None]
    out = torch.rand(n - kept, 3, generator=g, dtype=torch.float64) * torch.tensor([1.0, 1.0, 0.2]) + torch.tensor(
        [-0.5, -0.5, 0.8])
    pred = torch.cat([moved, out])[torch.randperm(n, generator=g)]
    off = torch.tensor(offset, dtype=torch.float64)
    return (pred + off).float(), (target + off).float()


def test_fscore_matches_restatement(cuda):
    from gecco_b200.metrics import reconstruction_metrics

    pairs = [_grid_pair(s, offset=(0.0, 0.0, 5.0) if s == 3 else (0.0, 0.0, 0.0)) for s in range(4)]
    pred = torch.stack([p for p, _ in pairs]).to(cuda)
    target = torch.stack([t for _, t in pairs]).to(cuda)
    taus = [0.005, 0.01, 0.02]
    d_xy, _, d_yx, _ = NO.nearest_f64(pred, target)
    for d in (d_xy, d_yx):  # every decision has a margin larger than the bound
        b = _bound(pred, target, d)
        for tau in taus:
            assert ((d - tau * tau).abs() > b).all(), tau
    got = reconstruction_metrics(pred, target, taus)
    p, r, f = NO.fscore_np(d_xy.cpu().numpy(), d_yx.cpu().numpy(), taus)
    print("precision", got["precision"].tolist(), "recall", got["recall"].tolist())
    assert got["precision"].shape == (4, 3) and got["fscore"].dtype == torch.float64
    np.testing.assert_array_equal(got["precision"].cpu().numpy(), p)
    np.testing.assert_array_equal(got["recall"].cpu().numpy(), r)
    np.testing.assert_array_equal(got["fscore"].cpu().numpy(), f)
    assert (p[:, 0] < p[:, 2]).all() and (r < p).all()  # the thresholds and the outliers matter


def test_conditional_sampler_output_feeds_the_metrics(cuda):
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
    target = samples + 0.005 * torch.randn(samples.shape, device=cuda, dtype=torch.float64, generator=g)
    out = G.reconstruction_metrics(samples, target, [0.01])
    assert torch.isfinite(out["cd"]).all() and (out["cd"] >= 0).all()
    for k in ("precision", "recall", "fscore"):
        assert out[k].shape == (B, 1) and torch.isfinite(out[k]).all()
        assert ((out[k] >= 0) & (out[k] <= 1)).all()

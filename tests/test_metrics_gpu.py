"""The Chamfer kernel (csrc/chamfer.cu) and the sample-quality metrics on the GPU: distances against the float64 direct
oracle (oracle/metrics_oracle.py), shapes and tails, the self / paired modes, determinism, and the metrics end to end."""
import pytest
import torch

from oracle import metrics_oracle as MO

pytestmark = pytest.mark.gpu

REL = 1e-4  # fp32 expansion |x|^2 + |y|^2 - 2 x.y on centred clouds against the float64 direct form, per entry


def _clouds(seed, m, n, scale=1.0, offset=(0.0, 0.0, 0.0)):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(m, n, 3, generator=g) * scale + torch.tensor(offset)


def _sets(seed, mg, mr, n):
    """Clouds with random offsets and scales: distinct enough that every nearest-neighbour decision has a wide margin."""
    g = torch.Generator().manual_seed(seed)

    def draw(m):
        off = torch.rand(m, 1, 3, generator=g, dtype=torch.float64) * 4 - 2
        sc = torch.rand(m, 1, 1, generator=g, dtype=torch.float64) * 0.5 + 0.5
        return torch.randn(m, n, 3, generator=g, dtype=torch.float64) * sc + off

    return draw(mg), draw(mr)


def _check(got, ref):
    rel = ((got.double() - ref).abs() / ref.abs().clamp_min(1e-30)).max().item()
    assert rel < REL, rel
    return rel


@pytest.fixture(scope="module")
def clouds_16x12(cuda):
    a = torch.cat([_clouds(1, 12, 2048), _clouds(2, 4, 2048, 0.5, (0.0, 0.0, 5.0))])  # 4 clouds around z = 5
    b = torch.cat([_clouds(3, 9, 2048, 0.8), _clouds(4, 3, 2048, 1.0, (0.2, -0.1, 5.0))])
    return a.to(cuda), b.to(cuda)


def test_matrix_matches_oracle(clouds_16x12):
    from gecco_b200.metrics import chamfer_matrix

    a, b = clouds_16x12
    got = chamfer_matrix(a, b)
    assert got.shape == (16, 12) and got.dtype == torch.float32
    rel = _check(got, MO.chamfer_matrix_f64(a, b))
    print(f"chamfer_matrix 16 x 12 x 2048: max rel err {rel:.2e}")


def test_far_from_origin(cuda):
    # camera-frame-like clouds: small extent far from the origin (the expanded form would cancel without centring)
    from gecco_b200.metrics import chamfer_matrix

    a = _clouds(5, 3, 2048, 0.05, (0.3, -0.2, 5.0)).to(cuda)
    b = _clouds(6, 2, 2048, 0.05, (0.3, -0.19, 5.01)).to(cuda)
    _check(chamfer_matrix(a, b), MO.chamfer_matrix_f64(a, b))


@pytest.mark.parametrize("na,nb", [(2048, 16384), (16384, 2048), (1, 33), (33, 1), (2047, 33), (1, 1), (3000, 5000),
                                   (65, 2047)])
def test_shapes_and_tails(cuda, na, nb):
    from gecco_b200.metrics import chamfer_distance, chamfer_matrix

    a = _clouds(10 + na, 2, na).to(cuda)
    b = _clouds(20 + nb, 3, nb, 0.9, (0.1, 0.0, 0.0)).to(cuda)
    ref = MO.chamfer_matrix_f64(a, b)
    got = chamfer_matrix(a, b)
    _check(got, ref)
    assert torch.equal(chamfer_distance(a, b[:2]), got.diagonal())


def test_self_and_paired_modes(clouds_16x12):
    from gecco_b200.metrics import chamfer_distance, chamfer_matrix

    a, b = clouds_16x12
    s = chamfer_matrix(a)
    assert torch.equal(s, s.t())
    assert torch.all(s.diagonal() == 0)
    full = chamfer_matrix(a, a)
    iu = torch.triu_indices(16, 16, 1, device=a.device)
    assert torch.equal(s[iu[0], iu[1]], full[iu[0], iu[1]])  # the upper triangle is the same per-pair code
    _check(s[iu[0], iu[1]], MO.chamfer_matrix_f64(a)[iu[0], iu[1]])
    assert torch.equal(chamfer_distance(a[:12], b), chamfer_matrix(a[:12], b).diagonal())
    # float64 input is cast on the device; the result is the one of the fp32 copy
    assert torch.equal(chamfer_matrix(a.double(), b.double()), chamfer_matrix(a, b))
    for m in (1, 2, 3):  # the smallest self matrices (diagonal-only blocks)
        sm = chamfer_matrix(a[:m])
        assert torch.equal(sm, sm.t()) and torch.all(sm.diagonal() == 0)
        assert torch.equal(sm, chamfer_matrix(a[:m], a[:m]).triu(1) + chamfer_matrix(a[:m], a[:m]).triu(1).t())


def test_deterministic(clouds_16x12):
    from gecco_b200.metrics import chamfer_matrix

    a, b = clouds_16x12
    assert torch.equal(chamfer_matrix(a, b), chamfer_matrix(a, b))
    big_a, big_b = _clouds(30, 2, 16384).cuda(), _clouds(31, 2, 9000).cuda()
    assert torch.equal(chamfer_matrix(big_a, big_b), chamfer_matrix(big_a, big_b))


def test_sample_metrics_matches_oracle(cuda):
    from gecco_b200.metrics import sample_metrics

    gen, ref = _sets(0, 16, 16, 1024)
    gen, ref = gen.to(cuda), ref.to(cuda)
    d_gg, d_rr, d_gr = MO.chamfer_matrix_f64(gen), MO.chamfer_matrix_f64(ref), MO.chamfer_matrix_f64(gen, ref)
    # every nearest-neighbour decision (COV: per generated cloud over S_r; 1-NNA: per cloud over the union) is won by more
    # than 10x the per-entry tolerance, so the fp32 matrices must take the same decisions
    full = torch.cat([torch.cat([d_gg, d_gr], 1), torch.cat([d_gr.t(), d_rr], 1)], 0)
    full.fill_diagonal_(float("inf"))
    for m in (d_gr, full):
        s = m.sort(dim=1).values
        assert ((s[:, 1] - s[:, 0]) / s[:, 0]).min().item() > 10 * REL
    want = MO.metrics(d_gg.cpu().numpy(), d_rr.cpu().numpy(), d_gr.cpu().numpy())
    got = sample_metrics(gen, ref)
    print("sample_metrics", got, "oracle", want)
    assert got["one_nna"] == want["one_nna"] and got["cov"] == want["cov"]
    assert got["mmd"] == pytest.approx(want["mmd"], rel=REL)


def test_sampler_output_feeds_the_metrics(cuda):
    from gecco_b200.metrics import sample_metrics
    from tests import synth
    from tests.models_b200 import build

    rp = synth.UNCOND_REPARAM
    sd = synth.tame(synth.full_state_dict("uncond", "gaussian", rp["mean"], rp["sigma"], 1234), 0.15)
    model = build("uncond", "gaussian", rp["mean"], rp["sigma"], 165.0, None, cuda, None, state_dict=sd)
    samples = model.sample_stochastic((4, 256, 3), None, rng=synth.gen(7), num_steps=4)
    assert samples.dtype == torch.float64 and samples.is_cuda
    reference = samples[:3].flip(0).float() + 0.01
    out = sample_metrics(samples, reference)
    assert set(out) == {"one_nna", "mmd", "cov"}
    assert 0.0 <= out["one_nna"] <= 1.0 and 0.0 < out["cov"] <= 1.0 and out["mmd"] >= 0.0

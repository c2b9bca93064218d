"""The approximate EMD kernel (csrc/emd.cu) and the EMD sample-quality metrics on the GPU: distances against the float64
oracle (oracle/emd_oracle.py) in both orientations, point-count tails, the self / paired modes, determinism, and the
metrics end to end in PointFlow's orientation."""
import pytest
import torch

from oracle import emd_oracle as EO
from oracle import metrics_oracle as MO

pytestmark = pytest.mark.gpu

REL = 1e-4  # fp32 kernel (fused schedule, scaled centred coordinates) against the float64 three-pass statement, per entry


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


def test_matrix_matches_oracle_in_both_orientations(clouds_16x12):
    from gecco_b200.metrics import emd_matrix

    a, b = clouds_16x12
    got_ab, got_ba = emd_matrix(a, b), emd_matrix(b, a)
    assert got_ab.shape == (16, 12) and got_ba.shape == (12, 16) and got_ab.dtype == torch.float32
    ref_ab, ref_ba = EO.emd_matrix_f64(a, b), EO.emd_matrix_f64(b, a)
    # the two orientations differ by more than the gate on some pairs, so each is checked against its own oracle
    assert ((ref_ab - ref_ba.t()).abs() / ref_ab).max().item() > 10 * REL
    rel = max(_check(got_ab, ref_ab), _check(got_ba, ref_ba))
    print(f"emd_matrix 16 x 12 x 2048, both orientations: max rel err {rel:.2e}")


def test_small_clouds_far_from_origin(cuda):
    # camera-frame-like clouds: small extent far from the origin, where exp(-16384 d2) needs d2 from coordinate differences
    from gecco_b200.metrics import emd_matrix

    a = _clouds(5, 3, 2048, 0.05, (0.3, -0.2, 5.0)).to(cuda)
    b = _clouds(6, 2, 2048, 0.05, (0.3, -0.19, 5.01)).to(cuda)
    _check(emd_matrix(a, b), EO.emd_matrix_f64(a, b))
    _check(emd_matrix(b, a), EO.emd_matrix_f64(b, a))


@pytest.mark.parametrize("n", [1, 2, 31, 33, 255, 257, 2047, 3000, 4096])
def test_point_count_tails(cuda, n):
    from gecco_b200.metrics import emd_distance, emd_matrix

    a = _clouds(10 + n, 2, n).to(cuda)
    b = _clouds(20 + n, 3, n, 0.9, (0.1, 0.0, 0.0)).to(cuda)
    got = emd_matrix(a, b)
    _check(got, EO.emd_matrix_f64(a, b))
    assert torch.equal(emd_distance(a, b[:2]), got[:, :2].diagonal())
    s = emd_matrix(b)
    full = emd_matrix(b, b)
    off = ~torch.eye(3, dtype=torch.bool, device=cuda)
    assert torch.equal(s[off], full[off]) and torch.all(s.diagonal() == 0)


def test_self_and_paired_modes(clouds_16x12):
    from gecco_b200.metrics import emd_distance, emd_matrix

    a, b = clouds_16x12
    s = emd_matrix(a)
    full = emd_matrix(a, a)
    off = ~torch.eye(16, dtype=torch.bool, device=a.device)
    assert torch.equal(s[off], full[off])  # the same per-pair code, ordered pairs
    assert torch.all(s.diagonal() == 0)
    assert not torch.equal(s, s.t())  # EMD is not symmetric
    _check(s[off], EO.emd_matrix_f64(a)[off])
    assert torch.equal(emd_distance(a[:12], b), emd_matrix(a[:12], b).diagonal())
    for m in (1, 2, 3):  # the smallest self matrices (diagonal-only blocks)
        sm = emd_matrix(a[:m])
        assert torch.all(sm.diagonal() == 0)
        offm = ~torch.eye(m, dtype=torch.bool, device=a.device)
        assert torch.equal(sm[offm], emd_matrix(a[:m], a[:m])[offm])


def test_float64_input_and_determinism(clouds_16x12):
    from gecco_b200.metrics import emd_distance, emd_matrix

    a, b = clouds_16x12
    first = emd_matrix(a, b)
    assert torch.equal(emd_matrix(a.double(), b.double()), first)  # cast on the device: the fp32 copy's result
    assert torch.equal(emd_distance(a[:12].double(), b.double()), emd_distance(a[:12], b))
    for _ in range(2):
        assert torch.equal(emd_matrix(a, b), first)
        assert torch.equal(emd_matrix(a), emd_matrix(a))


def test_sample_metrics_emd_matches_oracle(cuda):
    from gecco_b200.metrics import sample_metrics

    gen, ref = _sets(0, 16, 16, 512)
    gen, ref = gen.to(cuda), ref.to(cuda)
    # PointFlow's ordered matrices: M_rs[r, s] = EMD(ref_r, sample_s), M_ss, M_rr; MMD / COV over M_rs.T, 1-NNA down the
    # columns (row-wise here: the self blocks transposed)
    m_ss, m_rr, m_rs = EO.emd_matrix_f64(gen), EO.emd_matrix_f64(ref), EO.emd_matrix_f64(ref, gen)
    d_gg, d_rr, d_gr = m_ss.t(), m_rr.t(), m_rs.t()
    # every nearest-neighbour decision is won by more than 10x the per-entry tolerance, so the fp32 matrices must take the
    # same decisions
    full = torch.cat([torch.cat([d_gg, d_gr], 1), torch.cat([d_gr.t(), d_rr], 1)], 0)
    full.fill_diagonal_(float("inf"))
    for m in (d_gr, full):
        s = m.sort(dim=1).values
        assert ((s[:, 1] - s[:, 0]) / s[:, 0]).min().item() > 10 * REL
    want = MO.metrics(d_gg.cpu().numpy(), d_rr.cpu().numpy(), d_gr.cpu().numpy())
    assert want["one_nna"] == EO.pointflow_knn_one_nna(m_rr.cpu().numpy(), m_rs.cpu().numpy(), m_ss.cpu().numpy())
    got = sample_metrics(gen, ref, distance="emd")
    print("sample_metrics(distance='emd')", got, "oracle", want)
    assert got["one_nna"] == want["one_nna"] and got["cov"] == want["cov"]
    assert got["mmd"] == pytest.approx(want["mmd"], rel=REL)
    # the default is still CD
    assert sample_metrics(gen, ref) == sample_metrics(gen, ref, distance="cd")


def test_sample_metrics_emd_one_nna_is_pointflows_on_near_tie_sets(cuda):
    # identically distributed sets, where the orientation of the self matrices decides part of the 1-NNA: sample_metrics
    # must give PointFlow's knn restated column by column on the kernel's own matrices
    from gecco_b200.metrics import emd_matrix, metrics_from_distances, sample_metrics

    differs = 0
    for seed in range(3):
        g = torch.Generator().manual_seed(seed)
        gen = torch.randn(24, 256, 3, generator=g).to(cuda)
        ref = torch.randn(24, 256, 3, generator=g).to(cuda)
        m_ss, m_rr, m_rs = emd_matrix(gen), emd_matrix(ref), emd_matrix(ref, gen)
        want = EO.pointflow_knn_one_nna(m_rr.cpu().numpy(), m_rs.cpu().numpy(), m_ss.cpu().numpy())
        mmd, cov = MO.lgan_mmd_cov(m_rs.t().cpu().numpy())
        got = sample_metrics(gen, ref, distance="emd")
        print(f"seed {seed}: sample_metrics {got}, PointFlow knn {want}")
        assert got["one_nna"] == want and got["cov"] == cov
        assert got["mmd"] == pytest.approx(mmd, rel=1e-12)
        differs += metrics_from_distances(m_ss, m_rr, m_rs.t())["one_nna"] != want
    assert differs >= 1  # the untransposed self matrices would have given a different number


def test_sampler_output_feeds_the_emd_metrics(cuda):
    from gecco_b200.metrics import emd_matrix, sample_metrics
    from tests import synth
    from tests.models_b200 import build

    rp = synth.UNCOND_REPARAM
    sd = synth.tame(synth.full_state_dict("uncond", "gaussian", rp["mean"], rp["sigma"], 1234), 0.15)
    model = build("uncond", "gaussian", rp["mean"], rp["sigma"], 165.0, None, cuda, None, state_dict=sd)
    samples = model.sample_stochastic((4, 256, 3), None, rng=synth.gen(7), num_steps=4)
    assert samples.dtype == torch.float64 and samples.is_cuda
    reference = samples[:3].flip(0).float() + 0.01
    out = sample_metrics(samples, reference, distance="emd")
    assert set(out) == {"one_nna", "mmd", "cov"}
    assert 0.0 <= out["one_nna"] <= 1.0 and 0.0 < out["cov"] <= 1.0 and out["mmd"] >= 0.0
    _check(emd_matrix(reference, samples), EO.emd_matrix_f64(reference, samples))

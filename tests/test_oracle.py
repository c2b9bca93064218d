"""Pins the CPU oracle (oracle/gecco_oracle.py) against the golden vectors minted from the UNMODIFIED
reference package by oracle/make_golden.py (the reference ships no tests of its own, SURVEY.md §4)."""
from pathlib import Path

import pytest
import torch

from oracle import gecco_oracle as O
from tests import synth

GOLD = Path(__file__).parent / "golden"
TOL = 2e-5  # fp32 re-association only


def load(name):
    g = torch.load(GOLD / name, weights_only=False)
    r = g["recipe"]
    cfg = O.OracleConfig(kind=r["kind"], reparam=r["reparam"], sigma_max=r["sigma_max"], n_layers=r["n_layers"],
                         num_heads=r["num_heads"])
    sd = synth.full_state_dict(r["kind"], r["reparam"], r["mean"], r["sigma"], r["weight_seed"])
    return g, r, cfg, sd


def rel(a, b):
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-12)).item()


def test_uncond_denoise_cache_sample():
    g, r, cfg, sd = load("uncond.pt")
    x = torch.randn(r["B"], r["N"], 3, generator=synth.gen(r["x_seed"])) * r["x_scale"]
    D, hs = O.denoise(cfg, sd, x, r["noise_sigma"], return_h=True)
    assert rel(D, g["D"]) < TOL
    for h, hg in zip(hs, g["hs_sub"]):
        assert rel(h[:, ::8, ::8], hg) < TOL
    x2 = torch.randn(r["B"], r["N2"], 3, generator=synth.gen(r["x2_seed"])) * r["x_scale"]
    assert rel(O.denoise(cfg, sd, x2, r["noise_sigma"], hs=hs), g["D_cached"]) < TOL
    s = O.sample_stochastic(cfg, sd, r["sample_shape"], rng=synth.gen(r["sample_seed"]), num_steps=r["sample_steps"])
    assert s.dtype == torch.float64
    assert rel(s, g["sample"]) < 1e-4
    assert torch.equal(O.t_steps(64, 165.0, 0.002, 7), g["t_steps"])


def test_cond_gaussian():
    g, r, cfg, sd = load("cond_gaussian.pt")
    feats = synth.synth_features(r["B"], r["feat_sizes"], r["feat_seed"])
    K = synth.camera(r["B"], r["K"])
    x = torch.randn(r["B"], r["N"], 3, generator=synth.gen(r["x_seed"])) * r["x_scale"]
    assert rel(O.denoise(cfg, sd, x, r["noise_sigma"], feats, K), g["D"]) < TOL
    c_in = 1 / (1 + r["noise_sigma"] ** 2).sqrt()
    look = O.extract_image_features(cfg, sd, x * c_in[:, None, None], feats, K)
    assert rel(look[:, ::3], g["lookup_sub"]) < TOL
    s = O.sample_stochastic(cfg, sd, r["sample_shape"], feats, K, rng=synth.gen(r["sample_seed"]), num_steps=r["sample_steps"])
    assert rel(s, g["sample"]) < 1e-4


def test_cond_uvl_cache_upsample_roundtrip():
    g, r, cfg, sd = load("cond_uvl.pt")
    feats = synth.synth_features(r["B"], r["feat_sizes"], r["feat_seed"])
    K = synth.camera(r["B"], r["K"])
    x = torch.randn(r["B"], r["N"], 3, generator=synth.gen(r["x_seed"])) * r["x_scale"]
    D, hs = O.denoise(cfg, sd, x, r["noise_sigma"], feats, K, return_h=True)
    assert rel(D, g["D"]) < TOL
    for h, hg in zip(hs, g["hs_sub"]):
        assert rel(h[:, ::8, ::8], hg) < TOL
    c_in = 1 / (1 + r["noise_sigma"] ** 2).sqrt()
    look = O.extract_image_features(cfg, sd, x * c_in[:, None, None], feats, K)
    assert rel(look[:, ::3], g["lookup_sub"]) < TOL
    x2 = torch.randn(r["B"], r["N2"], 3, generator=synth.gen(r["x2_seed"])) * r["x_scale"]
    assert rel(O.denoise(cfg, sd, x2, r["noise_sigma"], feats, K, hs=hs), g["D_cached"]) < TOL
    diff = torch.randn(r["B"], 64, 3, generator=synth.gen(r["rt_seed"]))
    data = O.diffusion_to_data(cfg, sd, diff, K)
    assert rel(data, g["rt_data"]) < TOL
    assert rel(O.data_to_diffusion(cfg, sd, data, K), g["rt_back"]) < 1e-4
    # samples are compared in diffusion space: data space goes through exp() of the depth coordinate.  With random-init UVL
    # weights the sampler trajectories amplify fp32 rounding: on a CPU like the one that minted the goldens the oracle
    # matches them bit for bit, but another thread count or vector ISA (1 thread, AVX2, SSE) moves the 5-step sample by up
    # to 5e-3 (max) and the upsampled cloud by up to 4e-2 (rms), where a wrong noise draw moves it by 1.2 (rms).  The short
    # trajectory (2 steps from sigma 2, oracle/make_golden.py) amplifies nothing (<= 1e-4 on every CPU) and is held tight.
    to_diff = lambda d: O.data_to_diffusion(cfg, sd, d, K.double())
    s2 = O.sample_stochastic(cfg, sd, (2, 160, 3), feats, K, rng=synth.gen(5), num_steps=2, sigma_max=2.0)
    assert rel(to_diff(s2), to_diff(g["sample2"])) < 2e-4
    s = O.sample_stochastic(cfg, sd, r["sample_shape"], feats, K, rng=synth.gen(r["sample_seed"]), num_steps=r["sample_steps"])
    assert rel(to_diff(s), to_diff(g["sample"])) < 2e-2
    seed_cloud = O.diffusion_to_data(cfg, sd, torch.randn(r["B"], r["ups_n_seed"], 3, generator=synth.gen(r["ups_seed_cloud_seed"])), K)
    u = O.upsample(cfg, sd, seed_cloud, n_new=r["ups_n_new"], features=feats, K=K, seed=r["ups_seed"],
                   num_substeps=r["ups_substeps"], num_steps=r["ups_steps"])
    u_ref = to_diff(g["upsample"])
    assert (to_diff(u) - u_ref).pow(2).mean().sqrt() < 0.15 * u_ref.pow(2).mean().sqrt()


def test_upsample_argument_check():
    g, r, cfg, sd = load("uncond.pt")
    with pytest.raises(ValueError):  # diffusion.py:398-401
        O.upsample(cfg, sd, torch.zeros(1, 8, 3))


@pytest.mark.parametrize("name", ["bench_uncond", "bench_cond_gaussian"])
def test_bench_shape_goldens(name):
    """The oracle against the reference at the benchmarked shape (B = 4, N = 2048): denoiser output, inducer states and
    the EDM loss value; the conditional case rebuilds the reference's ConvNeXtExtractor pyramid from its seed."""
    g = torch.load(GOLD / (name + ".pt"), weights_only=False)
    r = g["recipe"]
    cfg = O.OracleConfig(kind=r["kind"], reparam=r["reparam"], sigma_max=r["sigma_max"])
    sd = synth.full_state_dict(r["kind"], r["reparam"], r["mean"], r["sigma"], r["weight_seed"])
    B, N = r["B"], r["N"]
    feats = K = None
    if r["kind"] == "cond":
        import torchvision.models as tvm

        torch.manual_seed(r["convnext_seed"])
        net = tvm.convnext_tiny(weights=None).eval()
        for m in net.modules():
            if isinstance(m, tvm.convnext.CNBlock):
                m.stochastic_depth = torch.nn.Identity()
        x = torch.rand(B, 3, r["image"], r["image"], generator=synth.gen(r["image_seed"]))
        feats = []
        with torch.no_grad():
            for i in range(0, 6, 2):  # (downsampling, processing) pairs, first three stages (models/feature_pyramid.py:44-52)
                x = net.features[i + 1](net.features[i](x))
                feats.append(x)
        for f, sub in zip(feats, g["pyramid_sub"]):
            assert rel(f[:, ::8, ::3, ::3], sub) < TOL
        K = synth.camera(B, r["K"])
    x = synth.noisy_input(B, N, r["noise_sigma"], r["x_seed"], r["x_noise_seed"])
    with torch.no_grad():
        D, hs = O.denoise(cfg, sd, x, r["noise_sigma"], feats, K, return_h=True)
    assert rel(D, g["D"]) < 5e-5
    for h, hg in zip(hs, g["hs_sub"]):
        assert rel(h[:, ::8, ::8], hg) < 5e-5
    # EDM loss (diffusion.py:118-143) on the reference's draws
    ex = O.diffusion_to_data(cfg, sd, torch.randn(B, N, 3, generator=synth.gen(r["ex_seed"])), K)
    torch.manual_seed(r["loss_seed"])
    u = torch.rand(B)
    noise = torch.randn_like(ex)
    assert torch.equal(u, g["loss_u"])
    with torch.no_grad():
        loss = O.edm_loss(cfg, sd, ex, u, noise, feats, K)
    assert abs(loss.item() - g["loss"].item()) < 1e-4 * abs(g["loss"].item())

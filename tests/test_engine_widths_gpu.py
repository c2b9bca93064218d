"""The denoiser engine at feature widths other than 384 (tests/engine_widths.py) against the float64 oracle on the device,
at the gates of test_engine_configs_gpu.py (F and D rel rms <= 1.5e-2 and rel max <= 8e-2 per cloud, inducer states rel
rms <= 1.5e-2), plus the GEMM statistics epilogue at every AdaGN group width it is instantiated for."""
import math

import pytest
import torch

from oracle import gecco_oracle as O
from tests import synth
from tests.engine_widths import BY_NAME, CONFIGS, REFUSED, build, width_config
from tests.test_engine_configs_gpu import _oracle, _x, check, check_h

pytestmark = pytest.mark.gpu


def _model(cfg, cuda, clouds: int, state_dict=None):
    """(model, context, oracle features, oracle K) for `clouds` clouds of width configuration `cfg`."""
    import gecco_b200 as G

    feats = cfg.features(clouds) if cfg.kind == "cond" else None
    model = build(cfg, cuda, feats, state_dict=state_dict)
    ctx = K = None
    if cfg.kind == "cond":
        K = synth.camera(clouds, cfg.K)
        ctx = G.Context3d(image=torch.zeros(clouds, 3, 8, 8, device=cuda), K=K.to(cuda))
    return model, ctx, feats, K


# ------------------------------------------------------------------------------------------------ a. GEMM epilogue
# (clouds, rows_per_cloud, valid_rows, n_out, k): the engine's residual-stream producers have n_out = C = 32 w; 480 rows leave
# a partial 128-row tile, n_out 512 a partial 192-column panel; the last shape fits the CTA-pair kernel, which keeps
# 12-channel statistics only, so the single-CTA kernel takes the other widths.
SHAPES = [(3, 256, 200, None, 256), (3, 160, 150, None, 136), (2, 1024, 1000, 768, 384)]


@pytest.mark.parametrize("shape", SHAPES, ids=["tiles", "partial_tile", "pair_shape"])
@pytest.mark.parametrize("w", [4, 8, 12, 16, 24, 32])
def test_gemm_statistics_width(cuda, w, shape):
    from gecco_b200 import ops

    B, Np, N, n_out, K = shape
    C = n_out or 32 * w
    if C % w:
        pytest.skip("n_out not a multiple of the width")
    g = torch.Generator(device="cpu").manual_seed(w + Np)
    a = torch.randn(B * Np, K, generator=g).to(cuda).bfloat16()
    wt = (torch.randn(C, K, generator=g) / math.sqrt(K)).to(cuda).bfloat16()
    bias = torch.randn(C, generator=g).to(cuda)
    res = torch.randn(B * Np, C, generator=g).to(cuda)
    x = res.clone()
    stats = torch.zeros(B, C // w, 2, dtype=torch.float64, device=cuda)
    ops.gemm(a, wt, bias=bias, res=x, out_f32=x, stats=stats, stat_gs=w, rows_per_cloud=Np, valid_rows=N)
    torch.cuda.synchronize()
    ref = a.float() @ wt.float().t() + bias + res
    xv = x.view(B, Np, C)
    assert (xv[:, :N] - ref.view(B, Np, C)[:, :N]).abs().max().item() < 2e-3
    # float64 sums per (cloud, group) of what the kernel wrote, over the valid rows only
    v = xv[:, :N].double().reshape(B, N, C // w, w)
    s1, s2 = v.sum(dim=(1, 3)), (v * v).sum(dim=(1, 3))
    scale = (v * v).sum(dim=(1, 3)).sqrt() * math.sqrt(N * w)  # bound of the fp32 partial-sum rounding
    assert ((stats[..., 0] - s1).abs() <= 1e-5 * scale + 1e-9).all(), (stats[..., 0] - s1).abs().max()
    assert ((stats[..., 1] - s2).abs() <= 1e-5 * s2 + 1e-9).all(), (stats[..., 1] - s2).abs().max()


def test_gemm_statistics_width_refused(cuda):
    from gecco_b200 import ops

    a = torch.zeros(256, 64, device=cuda, dtype=torch.bfloat16)
    wt = torch.zeros(640, 64, device=cuda, dtype=torch.bfloat16)
    stats = torch.zeros(1, 32, 2, dtype=torch.float64, device=cuda)
    with pytest.raises(ValueError, match="stat_gs"):
        ops.gemm(a, wt, out_f32=True, stats=stats, stat_gs=20)


# ------------------------------------------------------------------------------------------------ b. denoise
@pytest.mark.parametrize("cfg", CONFIGS, ids=lambda c: c.name)
def test_denoise_width(cuda, cfg):
    """Full evaluation with do_cache=True: D against the oracle, and one [clouds, 64, C] inducer state per layer."""
    clouds, points = 2, 1000
    model, ctx, feats, K = _model(cfg, cuda, clouds)
    x, sig = _x(clouds, points)
    with torch.no_grad():
        D, hs = model(x.to(cuda), sig.to(cuda), ctx, do_cache=True)
    assert len(hs) == cfg.layers and all(tuple(h.shape) == (clouds, synth.NUM_INDUCERS, cfg.width) for h in hs)
    D_ref, hs_ref = _oracle(cfg, cuda, x, sig, feats, K)
    check(D, D_ref, x.to(cuda), sig.to(cuda), cfg.sigma_data, f"{cfg.name} {clouds}x{points} D")
    check_h(hs, hs_ref, f"{cfg.name} h")


@pytest.mark.parametrize("name", ["uncond_gaussian_c512_h8", "cond_uvl_c256_h8"])
def test_inducer_cache_width(cuda, name):
    """The states of do_cache=True, then the evaluation from that cache at another point count (3 x 300: Np = 384)."""
    cfg = BY_NAME[name]
    clouds = 3
    model, ctx, feats, K = _model(cfg, cuda, clouds)
    x, sig = _x(clouds, 700)
    with torch.no_grad():
        _, hs = model(x.to(cuda), sig.to(cuda), ctx, do_cache=True)
    _, hs_ref = _oracle(cfg, cuda, x, sig, feats, K)
    check_h(hs, hs_ref, f"{name} h")
    x2, _ = _x(clouds, 300, seed=81)
    with torch.no_grad():
        Dc = model(x2.to(cuda), sig.to(cuda), ctx, cache=hs)
    Dc_ref, _ = _oracle(cfg, cuda, x2, sig, feats, K, hs=hs_ref)
    check(Dc, Dc_ref, x2.to(cuda), sig.to(cuda), cfg.sigma_data, f"{name} cached")


# ------------------------------------------------------------------------------------------------ c. samplers at C = 512
def _tame(cfg, cuda, clouds):
    sd = synth.tame(cfg.state_dict(), 0.15)
    model, ctx, feats, K = _model(cfg, cuda, clouds, state_dict=sd)
    return model, ctx, feats, K, sd


def _rel(a, b):
    a, b = a.cpu().double(), b.cpu().double()
    return (a - b).pow(2).mean().sqrt().item() / b.pow(2).mean().sqrt().item()


def test_sample_stochastic_512(cuda):
    cfg = BY_NAME["cond_gaussian_c512_h8"]
    B, shape = 2, (2, 160, 3)
    model, ctx, feats, K, sd = _tame(cfg, cuda, B)
    s = model.sample_stochastic(shape, ctx, rng=synth.gen(5), num_steps=2)
    o = O.sample_stochastic(cfg.oracle(), sd, shape, feats, K, rng=synth.gen(5), num_steps=2)
    assert torch.isfinite(s).all()
    e = _rel(s, o)
    print(f"C=512 2-step stochastic sample rel rms vs oracle {e:.2e}")
    assert e <= 2e-2


def test_sample_ode_512(cuda):
    cfg = BY_NAME["cond_gaussian_c512_h8"]
    B, N, steps = 2, 300, 8
    model, ctx, feats, K, sd = _tame(cfg, cuda, B)
    got = model.sample_ode((B, N, 3), ctx, rng=synth.gen(3), num_steps=steps)
    ref = O.sample_stochastic(cfg.oracle(), sd, (B, N, 3), feats, K, rng=synth.gen(3), num_steps=steps, S_churn=0.0)
    to_diff = lambda d: O.data_to_diffusion(cfg.oracle(), sd, d.cpu().double(), None)
    e = _rel(to_diff(got), to_diff(ref))
    print(f"C=512 ODE sample rel rms (diffusion space) {e:.2e}")
    assert e < 1e-2


def test_sample_inpaint_512(cuda):
    cfg = BY_NAME["uncond_gaussian_c512_h8"]
    B, N, M, steps = 2, 200, 184, 4
    model, _, _, _, sd = _tame(cfg, cuda, B)
    oc = cfg.oracle()
    known = O.diffusion_to_data(oc, sd, torch.randn(B, N, 3, generator=synth.gen(5)), None)
    got = model.sample_inpaint(known.to(cuda), M, None, rng=synth.gen(6), num_substeps=2, num_steps=steps, S_churn=0.5)
    ref = O.sample_inpaint(oc, sd, known, M, rng=synth.gen(6), num_substeps=2, num_steps=steps, S_churn=0.5)
    to_diff = lambda d: O.data_to_diffusion(oc, sd, d.cpu().double(), None)
    e = _rel(to_diff(got), to_diff(ref))
    print(f"C=512 inpaint rel rms (diffusion space) {e:.2e}")
    assert got.shape == (B, M, 3) and e < 1e-2


def test_upsample_512(cuda):
    """Upsampling at a small sigma_max (contractive): the upsampling step's KV cache holds [layers][clouds * 64, 2 C]."""
    cfg = BY_NAME["cond_uvl_c512_h8"]
    B = 2
    model, ctx, feats, K = _model(cfg, cuda, B)
    sd = cfg.state_dict()
    oc = cfg.oracle()
    seed_cloud = O.diffusion_to_data(oc, sd, torch.randn(B, 128, 3, generator=synth.gen(35)), K)
    us = model.upsample(seed_cloud.to(cuda), n_new=200, context=ctx, num_substeps=3, num_steps=3, sigma_max=0.05,
                        rng=synth.gen(9))
    uo = O.upsample(oc, sd, seed_cloud, n_new=200, features=feats, K=K, seed=9, num_substeps=3, num_steps=3, sigma_max=0.05)
    assert torch.isfinite(us).all()
    to_diff = lambda d: O.data_to_diffusion(oc, sd, d.cpu().double(), K.double())
    e = _rel(to_diff(us), to_diff(uo))
    print(f"C=512 small-sigma upsample rel rms vs oracle {e:.2e}")
    assert e <= 1e-2


# ------------------------------------------------------------------------------------------------ d. train, then sample
def test_train_then_sample_256(cuda):
    """A 256-wide model trained by Trainer (eager) for a few steps is then sampled by the engine, against the oracle's
    sampler on the trained weights."""
    from gecco_b200.training import Trainer

    cfg = width_config("uncond", "gaussian", 256, 8)
    B = 2
    model, _, _, _, sd = _tame(cfg, cuda, B)
    before = {k: v.clone() for k, v in model.state_dict().items()}
    tr = Trainer(model, lr=5e-5, graph=False)
    ex = O.diffusion_to_data(cfg.oracle(), sd, torch.randn(B, 512, 3, generator=synth.gen(52)), None).float().to(cuda)
    losses = [tr.step((ex, None)).item() for _ in range(3)]
    assert all(math.isfinite(l) for l in losses)
    trained = {k: v.detach().cpu() for k, v in model.state_dict().items() if k in sd}
    assert any(not torch.equal(trained[k], before[k].cpu()) for k in trained)
    model.eval()
    shape = (B, 160, 3)
    s = model.sample_stochastic(shape, None, rng=synth.gen(5), num_steps=2)
    o = O.sample_stochastic(cfg.oracle(), trained, shape, None, None, rng=synth.gen(5), num_steps=2)
    assert torch.isfinite(s).all()
    e = _rel(s, o)
    print(f"C=256 losses {losses}, 2-step sample of the trained model rel rms vs oracle {e:.2e}")
    assert e <= 2e-2


# ------------------------------------------------------------------------------------------------ e. refusals
@pytest.mark.parametrize("width,heads", REFUSED)
def test_refused_width(cuda, width, heads):
    """Widths whose AdaGN groups do not divide the epilogue panel are refused at the first call with a message naming
    feature_dim; a valid model still runs afterwards."""
    import gecco_b200 as G
    from gecco_b200._abi import GeccoError
    from gecco_b200.models import GaussianActivation, LinearLift, SetTransformer
    from gecco_b200.reparam import GaussianReparam

    st = SetTransformer(n_layers=1, num_inducers=synth.NUM_INDUCERS, feature_dim=width, t_embed_dim=1, num_heads=heads,
                        activation=GaussianActivation)
    model = G.Diffusion(backbone=G.EDMPrecond(model=LinearLift(inner=st, feature_dim=width)), conditioner=G.IdleConditioner(),
                        reparam=GaussianReparam(torch.zeros(3), torch.ones(3)),
                        loss=G.EDMLoss(schedule=G.LogUniformSchedule(max=165.0))).to(cuda).eval()
    with pytest.raises((GeccoError, ValueError), match="feature_dim"):
        with torch.no_grad():
            model(torch.randn(1, 100, 3, device=cuda), torch.ones(1, device=cuda), None)
    cfg = BY_NAME["uncond_gaussian_c512_h8"]
    good, _, _, _ = _model(cfg, cuda, 1)
    xs, sig = _x(1, 300)
    with torch.no_grad():
        D = good(xs.to(cuda), sig.to(cuda), None)
    D_ref, _ = _oracle(cfg, cuda, xs, sig, None, None)
    check(D, D_ref, xs.to(cuda), sig.to(cuda), cfg.sigma_data, "valid model after a refusal")

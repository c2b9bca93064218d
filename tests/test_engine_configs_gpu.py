"""The denoiser engine end to end at every network configuration it accepts (tests/engine_configs.py) and at batch shapes
on either side of its path switches, against the float64 oracle on the device (same fp32 weights and inputs).

Gates (those of test_denoiser_gpu.check_F, in units of the raw network output F, per cloud; clouds with c_out < 0.01 are
skipped): rel rms <= 1.5e-2 and rel max <= 8e-2 of F, the same on D; inducer states rel rms <= 1.5e-2.  The oracle's own
float32 / float64 disagreement at these configurations is below 1e-4 (test_engine_configs_cpu.py).
"""
import time

import pytest
import torch

from oracle import gecco_oracle as O
from tests import synth
from tests.engine_configs import BY_NAME, CONFIGS, PROD, PROD_COND6, Config, precond, raw_output, rms, sigmas
from tests.models_b200 import build

pytestmark = pytest.mark.gpu

F_RMS, F_MAX, H_RMS = 1.5e-2, 8e-2, 1.5e-2


def _model(cfg: Config, cuda, clouds: int, state_dict=None):
    """(model, context, oracle features, oracle K) for `clouds` clouds of configuration `cfg`."""
    import gecco_b200 as G

    feats = cfg.features(clouds) if cfg.kind == "cond" else None
    model = build(cfg.kind, cfg.reparam, cfg.stats["mean"], cfg.stats["sigma"], cfg.sigma_max,
                  None if state_dict is not None else 1234, cuda, feats, state_dict=state_dict, **cfg.build_kw())
    ctx = K = None
    if cfg.kind == "cond":
        K = synth.camera(clouds, cfg.K)
        ctx = G.Context3d(image=torch.zeros(clouds, 3, 8, 8, device=cuda), K=K.to(cuda))
    return model, ctx, feats, K


def _oracle(cfg: Config, cuda, x, sig, feats, K, clouds=None, hs=None):
    """float64 oracle on the device for the clouds `clouds` (all when None): (D, inducer states)."""
    idx = torch.arange(x.shape[0]) if clouds is None else torch.tensor(clouds)
    sd = {k: v.to(cuda, torch.float64) for k, v in cfg.state_dict().items()}
    f = None if feats is None else [t[idx].to(cuda, torch.float64) for t in feats]
    k = None if K is None else K[idx].to(cuda, torch.float64)
    h = None if hs is None else [t[idx.to(t.device)] for t in hs]
    return O.denoise(cfg.oracle(), sd, x[idx].to(cuda, torch.float64), sig[idx].to(cuda, torch.float64), f, k, hs=h, return_h=True)


def check(D, D_ref, x, sig, sigma_data, what, clouds=None):
    """Per-cloud gates on F and on D; D, x, sig hold every cloud, D_ref the clouds listed in `clouds` (all when None)."""
    idx = list(range(D.shape[0])) if clouds is None else list(clouds)
    assert torch.isfinite(D).all(), what
    x, sig = x[idx], sig[idx]
    D = D[idx].double()
    D_ref = D_ref.to(D.device).double()
    F_got, F_ref = raw_output(D, x, sig, sigma_data), raw_output(D_ref, x, sig, sigma_data)
    _, c_out = precond(sig, sigma_data)
    worst = (0.0, 0.0)
    for j, b in enumerate(idx):
        if c_out[j].item() < 0.01:
            continue
        for name, got, ref in (("F", F_got[j], F_ref[j]), ("D", D[j], D_ref[j])):
            e = got - ref
            r, mx = rms(e) / rms(ref), e.abs().max().item() / ref.abs().max().item()
            if name == "F":
                worst = (max(worst[0], r), max(worst[1], mx))
            assert r <= F_RMS and mx <= F_MAX, (what, name, b, sig[j].item(), r, mx)
    print(f"{what}: worst rel rms {worst[0]:.2e}, rel max {worst[1]:.2e} of F")
    return worst


def check_h(hs, hs_ref, what, clouds=None):
    for l, (h, hr) in enumerate(zip(hs, hs_ref)):
        h = h if clouds is None else h[list(clouds)]
        e = rms(h.double() - hr.to(h.device)) / rms(hr)
        assert e <= H_RMS, (what, l, e)


def _x(clouds, points, seed=71):
    sig = sigmas(clouds)
    return synth.noisy_input(clouds, points, sig, seed, seed + 1), sig


# ------------------------------------------------------------------------------------------------ a. configuration matrix
# production batch shape, a ragged one (both normalise the AdaGN inputs inside the GEMMs: m >= 2048, Np % 256 == 0) and
# one small enough for the per-cloud weight fold (m = 768), whose workspace is sized by the MLP width
@pytest.mark.parametrize("clouds,points", [(4, 2048), (3, 1000), (2, 300)])
@pytest.mark.parametrize("cfg", CONFIGS, ids=lambda c: c.name)
def test_config_matrix(cuda, cfg, clouds, points):
    """Full evaluation with do_cache=True, then the cached evaluation at another point count from each side's own cache."""
    t0 = time.perf_counter()
    model, ctx, feats, K = _model(cfg, cuda, clouds)
    x, sig = _x(clouds, points)
    with torch.no_grad():
        D, hs = model(x.to(cuda), sig.to(cuda), ctx, do_cache=True)
    assert len(hs) == cfg.layers
    D_ref, hs_ref = _oracle(cfg, cuda, x, sig, feats, K)
    check(D, D_ref, x.to(cuda), sig.to(cuda), cfg.sigma_data, f"{cfg.name} {clouds}x{points} D")
    check_h(hs, hs_ref, f"{cfg.name} {clouds}x{points} h")
    x2, _ = _x(clouds, 450, seed=81)
    with torch.no_grad():
        Dc = model(x2.to(cuda), sig.to(cuda), ctx, cache=hs)
    Dc_ref, _ = _oracle(cfg, cuda, x2, sig, feats, K, hs=hs_ref)
    check(Dc, Dc_ref, x2.to(cuda), sig.to(cuda), cfg.sigma_data, f"{cfg.name} {clouds}x450 cached")
    print(f"{cfg.name} {clouds}x{points}: {time.perf_counter() - t0:.1f} s")


# ------------------------------------------------------------------------------------------------ b. shape sweep
SHAPES = [
    # ragged tails, including clouds smaller than one 64-key tile
    (1, 1), (1, 2), (1, 63), (1, 64), (1, 65), (2, 127), (2, 129), (3, 255), (3, 257),
    # AdaGN fold path (m = 3072 is large enough, but Np = 384 is not a multiple of 256) vs A-operand AdaGN (Np = 1024),
    # with and without a ragged tail
    (8, 300), (8, 1000), (8, 1024),
    # pool key splits: > 4 merged by pool_combine_kernel (<= 36 clouds), <= 4 merged in the chain (>= 37); more clouds
    # than SMs
    (16, 2048), (36, 2048), (37, 2048), (149, 512),
    (1, 16384),
]


def _subset(clouds):
    """The clouds the oracle checks: all of a small batch, else the first, one in the middle and the last."""
    return None if clouds <= 4 else (0, clouds // 2, clouds - 1)


@pytest.mark.parametrize("cfg,clouds,points", [(PROD, b, n) for b, n in SHAPES] + [(PROD_COND6, 2, 2049)],
                         ids=lambda v: v.name if isinstance(v, Config) else str(v))
def test_shape_sweep(cuda, cfg, clouds, points):
    model, ctx, feats, K = _model(cfg, cuda, clouds)
    x, sig = _x(clouds, points, seed=91)
    with torch.no_grad():
        D, hs = model(x.to(cuda), sig.to(cuda), ctx, do_cache=True)
    sub = _subset(clouds)
    D_ref, hs_ref = _oracle(cfg, cuda, x, sig, feats, K, clouds=sub)
    check(D, D_ref, x.to(cuda), sig.to(cuda), cfg.sigma_data, f"{cfg.name} {clouds}x{points}", clouds=sub)
    check_h(hs, hs_ref, f"{cfg.name} {clouds}x{points} h", clouds=sub)


# ------------------------------------------------------------------------------------------------ c. sampler / upsampling
@pytest.mark.parametrize("name", ["heads12", "no_norm", "sigma_data0.5", "cond_uvl_heads6_4levels"])
def test_sampler(cuda, name):
    """Two stochastic steps (gecco_sample: fused Euler / Heun head modes with the configuration's sigma_data) against
    the oracle's sampler on the same CPU generator, with the tame head so that the map contracts."""
    cfg = BY_NAME[name]
    B, shape = 2, (2, 160, 3)
    sd = synth.tame(cfg.state_dict(), 0.15)
    model, ctx, feats, K = _model(cfg, cuda, B, state_dict=sd)
    # (UVL: sigma_max lowered so that exp() of the ray-length coordinate stays finite after one giant step, as in
    # test_denoiser_gpu.test_cond_uvl)
    kw = dict(sigma_max=2.0) if cfg.reparam == "uvl" else {}
    s = model.sample_stochastic(shape, ctx, rng=synth.gen(5), num_steps=2, **kw).cpu()
    o = O.sample_stochastic(cfg.oracle(), sd, shape, feats, K, rng=synth.gen(5), num_steps=2, **kw)
    assert torch.isfinite(s).all() and torch.isfinite(o).all()
    if cfg.reparam == "uvl":
        to_diff = lambda d: O.data_to_diffusion(cfg.oracle(), sd, d.double(), K.double())
        s, o = to_diff(s), to_diff(o)
    e = rms(s - o) / rms(o)
    print(f"{name} 2-step sample rel rms vs oracle {e:.2e}")
    assert e <= 2e-2


def test_upsample_cond_uvl_heads6(cuda):
    """Upsampling at a small sigma_max (contractive, see test_denoiser_gpu.test_cond_uvl): the cached evaluations read
    the key / value projections of the per-noise-level inducer cache, here with the inducer side as separate launches."""
    cfg = BY_NAME["cond_uvl_heads6_4levels"]
    B = 2
    model, ctx, feats, K = _model(cfg, cuda, B)
    sd = cfg.state_dict()
    oc = cfg.oracle()
    seed_cloud = O.diffusion_to_data(oc, sd, torch.randn(B, 128, 3, generator=synth.gen(35)), K)
    us = model.upsample(seed_cloud.to(cuda), n_new=200, context=ctx, num_substeps=3, num_steps=3, sigma_max=0.05,
                        rng=synth.gen(9))
    uo = O.upsample(oc, sd, seed_cloud, n_new=200, features=feats, K=K, seed=9, num_substeps=3, num_steps=3, sigma_max=0.05)
    assert torch.isfinite(us).all() and torch.isfinite(uo).all()
    to_diff = lambda d: O.data_to_diffusion(oc, sd, d.cpu().double(), K.double())
    e = rms(to_diff(us) - to_diff(uo)) / rms(to_diff(uo))
    print(f"cond_uvl_heads6_4levels small-sigma upsample rel rms vs oracle {e:.2e}")
    assert e <= 1e-2


# ------------------------------------------------------------------------------------------------ d. training path
@pytest.fixture()
def _exact():
    old = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


@pytest.mark.parametrize("name", ["heads12", "blowup1", "no_norm"])
def test_training_path(cuda, monkeypatch, _exact, name):
    """Train-mode forward against the oracle, then the EDM loss and every parameter gradient against float64 autograd
    through the oracle's loss on the same draws (gates of test_training_gpu.test_loss_and_gradients_match_reference)."""
    cfg = BY_NAME[name]
    B, N = 2, 1000
    model, ctx, feats, K = _model(cfg, cuda, B)
    model.train()
    x, sig = _x(B, N, seed=101)
    D = model(x.to(cuda), sig.to(cuda), ctx)
    assert D.requires_grad
    D_ref, _ = _oracle(cfg, cuda, x, sig, feats, K)
    check(D.detach(), D_ref, x.to(cuda), sig.to(cuda), cfg.sigma_data, f"{name} train-mode forward")

    ex = model.reparam.diffusion_to_data(torch.randn(B, N, 3, generator=synth.gen(52)).to(cuda), ctx)
    u = torch.rand(B, generator=synth.gen(53))
    noise = torch.randn(B, N, 3, generator=synth.gen(54))
    monkeypatch.setattr(torch, "rand", lambda n, device=None, **kw: u.to(device))
    monkeypatch.setattr(torch, "randn_like", lambda t, **kw: noise.to(t.device, t.dtype))
    model.zero_grad(set_to_none=True)
    loss = model.training_step((ex, ctx), 0)
    loss.backward()
    monkeypatch.undo()

    sd = {k: v.to(cuda, torch.float64) for k, v in cfg.state_dict().items()}
    params = dict(model.named_parameters())
    for k in params:
        sd[k].requires_grad_(True)
    loss_ref = O.edm_loss(cfg.oracle(), sd, ex.double(), u.to(cuda, torch.float64), noise.to(cuda, torch.float64))
    loss_ref.backward()
    rel = abs(loss.item() - loss_ref.item()) / abs(loss_ref.item())
    print(f"{name}: loss {loss.item():.6g} vs float64 oracle {loss_ref.item():.6g} (rel {rel:.2e})")
    assert rel < 1e-2
    got = {k: p.grad for k, p in params.items() if p.grad is not None}
    assert set(got) == set(params)
    ref = {k: sd[k].grad for k in params}
    total = sum(g.double().pow(2).sum().item() for g in got.values()) ** 0.5
    total_ref = sum(g.pow(2).sum().item() for g in ref.values()) ** 0.5
    print(f"{name}: total gradient norm {total:.6g} vs float64 oracle {total_ref:.6g}")
    assert abs(total - total_ref) <= 3e-2 * total_ref
    worst_norm, worst_cos, worst_key = 0.0, 1.0, None
    for k, g in got.items():
        n_ref = ref[k].norm().item()
        if n_ref < 1e-3 * total_ref:  # negligible gradients are compared on the absolute scale of the step
            assert g.double().norm().item() < 2e-3 * total_ref, k
            continue
        e_norm = abs(g.double().norm().item() - n_ref) / max(n_ref, 1e-2 * total_ref)
        if e_norm > worst_norm:
            worst_norm, worst_key = e_norm, k
        a, b = g.double().flatten(), ref[k].flatten()
        if b.numel() >= 16:
            worst_cos = min(worst_cos, (a @ b / (a.norm() * b.norm())).item())
    print(f"{name}: worst per-parameter norm error {worst_norm:.3e} ({worst_key}), worst direction cosine {worst_cos:.5f}")
    assert worst_norm < 5e-2 and worst_cos > 0.97


# ------------------------------------------------------------------------------------------------ e. refusals
@pytest.mark.parametrize("kw,knob", [(dict(num_heads=4), "head dim"), (dict(num_inducers=32), "inducers")])
def test_refused_configurations(cuda, kw, knob):
    """Configurations without kernels are refused with a message naming the knob at the first call; the process then
    still runs a valid model."""
    import gecco_b200 as G
    from gecco_b200._abi import GeccoError
    from gecco_b200.models import GaussianActivation, LinearLift, SetTransformer
    from gecco_b200.reparam import GaussianReparam

    st_kw = dict(n_layers=1, num_inducers=synth.NUM_INDUCERS, feature_dim=synth.FEATURE_DIM, t_embed_dim=1,
                 num_heads=synth.NUM_HEADS, activation=GaussianActivation)
    st_kw.update(kw)
    net = LinearLift(inner=SetTransformer(**st_kw), feature_dim=synth.FEATURE_DIM)
    model = G.Diffusion(backbone=G.EDMPrecond(model=net), conditioner=G.IdleConditioner(),
                        reparam=GaussianReparam(torch.zeros(3), torch.ones(3)),
                        loss=G.EDMLoss(schedule=G.LogUniformSchedule(max=165.0))).to(cuda).eval()
    x = torch.randn(1, 100, 3, device=cuda)
    with pytest.raises((GeccoError, ValueError), match=knob):
        with torch.no_grad():
            model(x, torch.ones(1, device=cuda), None)
    cfg = PROD
    good, _, _, _ = _model(cfg, cuda, 1)
    xs, sig = _x(1, 300)
    with torch.no_grad():
        D = good(xs.to(cuda), sig.to(cuda), None)
    D_ref, _ = _oracle(cfg, cuda, xs, sig, None, None)
    check(D, D_ref, xs.to(cuda), sig.to(cuda), cfg.sigma_data, "valid model after a refusal")

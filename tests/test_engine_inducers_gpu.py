"""The attention cores and the denoiser engine at 128, 192 and 256 inducers (tests/engine_inducers.py) against float64
references on the device, at the gates of test_engine_configs_gpu.py (F and D rel rms <= 1.5e-2 and rel max <= 8e-2 per
cloud, inducer states rel rms <= 1.5e-2), plus the mma.sync attention cores at every count and head dim, the samplers,
the stand-alone module forwards, a trained model and the refused counts."""
import math

import pytest
import torch
import torch.nn.functional as F

from oracle import gecco_oracle as O
from tests import synth
from tests.engine_configs import rms
from tests.engine_inducers import BY_NAME, CONFIGS, REFUSED, build, inducer_config, set_transformer
from tests.test_engine_configs_gpu import _oracle, _x, check, check_h

pytestmark = pytest.mark.gpu

QS = math.log2(math.e)  # the exp -> exp2 change of base the kernels expect folded into the queries


def _model(cfg, cuda, clouds: int, state_dict=None):
    """(model, context, oracle features, oracle K) for `clouds` clouds of inducer configuration `cfg`."""
    import gecco_b200 as G

    feats = cfg.features(clouds) if cfg.kind == "cond" else None
    model = build(cfg, cuda, feats, state_dict=state_dict)
    ctx = K = None
    if cfg.kind == "cond":
        K = synth.camera(clouds, cfg.K)
        ctx = G.Context3d(image=torch.zeros(clouds, 3, 8, 8, device=cuda), K=K.to(cuda))
    return model, ctx, feats, K


def _rel(a, b):
    a, b = a.cpu().double(), b.cpu().double()
    return (a - b).pow(2).mean().sqrt().item() / b.pow(2).mean().sqrt().item()


# ------------------------------------------------------------------------------------------------ a. attention cores
def _heads(D):
    return 4 if D == 48 else 6  # C = 192, 192, 384: never the 8 x 48 shape of the tcgen05 cores


@pytest.mark.parametrize("D", [32, 48, 64])
@pytest.mark.parametrize("I", [64, 128, 192, 256])
def test_pool_attention_inducers(cuda, monkeypatch, I, D):
    """The mma.sync pool core (one CTA per 64 inducers of each key split, then the combine kernel) against float64
    softmax(Q K^T) V on the same bf16 operands, with ragged clouds (1, 65, 1000 keys, padding rows holding finite keys
    and values that must be masked) and one or eight key splits."""
    from gecco_b200 import ops

    monkeypatch.setenv("GECCO_POOL_TC", "0")
    H = _heads(D)
    C, B = H * D, 2
    g = synth.gen(I + D)
    ind = torch.randn(1, H, I, D, generator=g)
    qs = (ind[0] * (D**-0.5 * QS)).to(cuda).bfloat16().contiguous()
    qr = (qs.double().cpu() / (D**-0.5 * QS))[None]
    for N in (1, 65, 1000):
        Np = (N + 127) // 128 * 128
        kv = torch.full((B, Np, 2 * C), 3.0)
        kv[:, :N] = torch.randn(B, N, 2 * C, generator=g)
        kvd = kv.to(cuda).bfloat16().reshape(B * Np, 2 * C)
        kvr = kvd.double().cpu().view(B, Np, 2 * C)[:, :N]
        k = kvr[..., :C].reshape(B, N, H, D).transpose(1, 2)
        v = kvr[..., C:].reshape(B, N, H, D).transpose(1, 2)
        ref = F.scaled_dot_product_attention(qr.expand(B, -1, -1, -1), k, v).transpose(1, 2).reshape(B, I, C)
        for splits in (1, 8):
            out = ops.pool_attention(kvd, qs, clouds=B, rows_per_cloud=Np, valid_rows=N, heads=H, head_dim=D, k_off=0,
                                     v_off=C, splits=splits)
            assert out.shape == (B * I, C)
            err = (out.double().cpu().view(B, I, C) - ref).abs().max().item()
            assert err < 2e-2, (I, D, N, splits, err)


@pytest.mark.parametrize("D", [32, 48, 64])
@pytest.mark.parametrize("I", [64, 128, 192, 256])
def test_unpool_attention_inducers(cuda, I, D):
    """The mma.sync unpool core (online softmax over 64-key chunks) against float64 softmax(Q K^T) V on the same bf16
    operands.  In the second case the keys grow along the inducers, so the running maximum moves at every chunk."""
    from gecco_b200 import ops

    H = _heads(D)
    C = H * D
    g = synth.gen(3 * I + D)
    for B, Np, growing in ((2, 256, False), (3, 128, True)):
        q = torch.randn(B * Np, C, generator=g)
        khv = torch.randn(B, I, 2 * C, generator=g)
        if growing:
            khv[..., :C] *= (1.0 + torch.arange(I) / 32.0)[None, :, None]
        qd = (q * (D**-0.5 * QS)).to(cuda).bfloat16()
        kd = khv.reshape(B * I, 2 * C).to(cuda).bfloat16()
        out = ops.unpool_attention(qd, kd, clouds=B, rows_per_cloud=Np, heads=H, head_dim=D, v_off=C, inducers=I,
                                   tensor_cores=False)
        qr = (qd.double().cpu() / (D**-0.5 * QS)).view(B, Np, H, D).transpose(1, 2)
        kr = kd.double().cpu().view(B, I, 2 * C)
        k = kr[..., :C].reshape(B, I, H, D).transpose(1, 2)
        v = kr[..., C:].reshape(B, I, H, D).transpose(1, 2)
        ref = F.scaled_dot_product_attention(qr, k, v).transpose(1, 2).reshape(B * Np, C)
        err = (out.double().cpu() - ref).abs().max().item()
        assert err < 3e-2, (I, D, B, Np, growing, err)


# ------------------------------------------------------------------------------------------------ b. denoise
@pytest.mark.parametrize("clouds,points", [(4, 2048), (3, 1000), (2, 300)])
@pytest.mark.parametrize("cfg", CONFIGS, ids=lambda c: c.name)
def test_denoise_inducers(cuda, cfg, clouds, points):
    """Full evaluation with do_cache=True (one [clouds, I, C] inducer state per layer), then the cached evaluation at
    another point count from each side's own cache."""
    model, ctx, feats, K = _model(cfg, cuda, clouds)
    x, sig = _x(clouds, points)
    with torch.no_grad():
        D, hs = model(x.to(cuda), sig.to(cuda), ctx, do_cache=True)
    assert len(hs) == cfg.layers and all(tuple(h.shape) == (clouds, cfg.inducers, cfg.width) for h in hs)
    D_ref, hs_ref = _oracle(cfg, cuda, x, sig, feats, K)
    check(D, D_ref, x.to(cuda), sig.to(cuda), cfg.sigma_data, f"{cfg.name} {clouds}x{points} D")
    check_h(hs, hs_ref, f"{cfg.name} {clouds}x{points} h")
    x2, _ = _x(clouds, 450, seed=81)
    with torch.no_grad():
        Dc = model(x2.to(cuda), sig.to(cuda), ctx, cache=hs)
    Dc_ref, _ = _oracle(cfg, cuda, x2, sig, feats, K, hs=hs_ref)
    check(Dc, Dc_ref, x2.to(cuda), sig.to(cuda), cfg.sigma_data, f"{cfg.name} {clouds}x450 cached")


# ------------------------------------------------------------------------------------------------ c. shape sweep at 256
# ragged tails down to one point, many key splits merged by pool_combine_kernel (16 clouds), few (37), one long cloud
SHAPES = [(1, 1), (1, 65), (2, 129), (16, 2048), (37, 2048), (1, 16384)]


@pytest.mark.parametrize("clouds,points", SHAPES, ids=str)
def test_shape_sweep_256(cuda, clouds, points):
    cfg = BY_NAME["uncond_gaussian_i256_c384_h8"]
    model, ctx, feats, K = _model(cfg, cuda, clouds)
    x, sig = _x(clouds, points, seed=91)
    with torch.no_grad():
        D, hs = model(x.to(cuda), sig.to(cuda), ctx, do_cache=True)
    sub = None if clouds <= 4 else (0, clouds // 2, clouds - 1)
    D_ref, hs_ref = _oracle(cfg, cuda, x, sig, feats, K, clouds=sub)
    check(D, D_ref, x.to(cuda), sig.to(cuda), cfg.sigma_data, f"{cfg.name} {clouds}x{points}", clouds=sub)
    check_h(hs, hs_ref, f"{cfg.name} {clouds}x{points} h", clouds=sub)


# ------------------------------------------------------------------------------------------------ d. samplers at 128
def _tame(cfg, cuda, clouds):
    sd = synth.tame(cfg.state_dict(), 0.15)
    model, ctx, feats, K = _model(cfg, cuda, clouds, state_dict=sd)
    return model, ctx, feats, K, sd


def test_sample_stochastic_128(cuda):
    """Two stochastic steps against the oracle's sampler; the same call again replays the cached graph and reproduces the
    first result bit for bit."""
    from gecco_b200.engine import engine_for

    cfg = BY_NAME["cond_gaussian_i128_c384_h8"]
    B, shape = 2, (2, 160, 3)
    model, ctx, feats, K, sd = _tame(cfg, cuda, B)
    s = model.sample_stochastic(shape, ctx, rng=synth.gen(5), num_steps=2)
    o = O.sample_stochastic(cfg.oracle(), sd, shape, feats, K, rng=synth.gen(5), num_steps=2)
    assert torch.isfinite(s).all()
    e = _rel(s, o)
    print(f"I=128 2-step stochastic sample rel rms vs oracle {e:.2e}")
    assert e <= 2e-2
    eng = engine_for(*model._network())
    assert eng.graph_status() in (1, 2)
    s2 = model.sample_stochastic(shape, ctx, rng=synth.gen(5), num_steps=2)
    assert eng.graph_status() == 2 and torch.equal(s, s2)


def test_sample_ode_128(cuda):
    cfg = BY_NAME["cond_gaussian_i128_c384_h8"]
    B, N, steps = 2, 300, 8
    model, ctx, feats, K, sd = _tame(cfg, cuda, B)
    got = model.sample_ode((B, N, 3), ctx, rng=synth.gen(3), num_steps=steps)
    ref = O.sample_stochastic(cfg.oracle(), sd, (B, N, 3), feats, K, rng=synth.gen(3), num_steps=steps, S_churn=0.0)
    to_diff = lambda d: O.data_to_diffusion(cfg.oracle(), sd, d.cpu().double(), None)
    e = _rel(to_diff(got), to_diff(ref))
    print(f"I=128 ODE sample rel rms (diffusion space) {e:.2e}")
    assert e < 1e-2


def test_sample_inpaint_128(cuda):
    cfg = BY_NAME["uncond_gaussian_i128_c384_h8"]
    B, N, M, steps = 2, 200, 184, 4
    model, _, _, _, sd = _tame(cfg, cuda, B)
    oc = cfg.oracle()
    known = O.diffusion_to_data(oc, sd, torch.randn(B, N, 3, generator=synth.gen(5)), None)
    got = model.sample_inpaint(known.to(cuda), M, None, rng=synth.gen(6), num_substeps=2, num_steps=steps, S_churn=0.5)
    ref = O.sample_inpaint(oc, sd, known, M, rng=synth.gen(6), num_substeps=2, num_steps=steps, S_churn=0.5)
    to_diff = lambda d: O.data_to_diffusion(oc, sd, d.cpu().double(), None)
    e = _rel(to_diff(got), to_diff(ref))
    print(f"I=128 inpaint rel rms (diffusion space) {e:.2e}")
    assert got.shape == (B, M, 3) and e < 1e-2


def test_upsample_128(cuda):
    """Upsampling at a small sigma_max (contractive): the upsampling step's KV cache holds [layers][clouds * I, 2 C]."""
    cfg = BY_NAME["cond_uvl_i128_c384_h8"]
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
    print(f"I=128 small-sigma upsample rel rms vs oracle {e:.2e}")
    assert e <= 1e-2


# ------------------------------------------------------------------------------------------------ e. module forwards
def test_module_forwards_128(cuda):
    """Stand-alone AttentionPool, Broadcast (with and without h) and SetTransformer (with and without hs) forwards at
    128 inducers against the float64 oracle on the same weights."""
    cfg = inducer_config("uncond", "gaussian", 128)
    oc = cfg.oracle()
    pre = oc.st_prefix
    sd = cfg.state_dict()
    st = set_transformer(cfg)
    st.load_state_dict({k[len(pre):]: v for k, v in sd.items() if k.startswith(pre)})
    st = st.to(cuda).eval()
    sd64 = {k: v.to(cuda, torch.float64) for k, v in sd.items()}
    B, C, H = 2, cfg.width, cfg.heads
    x = torch.randn(B, 1000, C, generator=synth.gen(41)).to(cuda)
    x2 = torch.randn(B, 300, C, generator=synth.gen(42)).to(cuda)
    t = (torch.randn(B, 1, 1, generator=synth.gen(43)) * 0.5).to(cuda)
    xd, x2d, td = x.double(), x2.double(), t.double()
    lp = pre + "layers.0."
    bc = st.layers[0].broadcast
    errs = {}

    pooled = bc.pool(x)
    assert pooled.shape == (B, cfg.inducers, C)
    errs["pool"] = _rel(pooled, O.attention_pool(sd64, lp + "broadcast.pool.", xd, H))

    h_ref = O.attention_pool(sd64, lp + "broadcast.pool.", xd, H)
    h_ref = O.adagn(sd64, lp + "broadcast.norm_1.", h_ref, td)
    h_ref = O.mlp(sd64, lp + "broadcast.mlp.", h_ref)
    h_ref = O.adagn(sd64, lp + "broadcast.norm_2.", h_ref, td)
    attn, h = bc(x, t, return_h=True)
    errs["broadcast"] = _rel(attn, O.mha_unpool(sd64, lp + "broadcast.unpool.", xd, h_ref, H))
    errs["broadcast_h"] = _rel(h, h_ref)
    attn2, none = bc(x2, t, return_h=False, h=h_ref.float())
    assert none is None and attn2.shape == x2.shape
    errs["broadcast_given_h"] = _rel(attn2, O.mha_unpool(sd64, lp + "broadcast.unpool.", x2d, h_ref, H))

    f, hs = st(x, t, return_h=True)
    f_ref, hs_ref = O.set_transformer(oc, sd64, xd, td)
    assert len(hs) == cfg.layers and all(tuple(a.shape) == (B, cfg.inducers, C) for a in hs)
    errs["st"] = _rel(f, f_ref)
    for l, (a, b) in enumerate(zip(hs, hs_ref)):
        errs[f"st_h{l}"] = _rel(a, b)
    f2, none = st(x2, t, return_h=False, hs=[a.float() for a in hs_ref])
    assert none is None
    errs["st_given_hs"] = _rel(f2, O.set_transformer(oc, sd64, x2d, td, hs=hs_ref)[0])
    print({k: f"{v:.2e}" for k, v in errs.items()})
    bad = {k: v for k, v in errs.items() if v > 1.5e-2}
    assert not bad, bad


# ------------------------------------------------------------------------------------------------ f. train, then sample
def test_train_then_sample_128(cuda):
    """A 128-inducer model trained by Trainer (eager) for a few steps is then sampled by the engine, against the oracle's
    sampler on the trained weights."""
    from gecco_b200.training import Trainer

    cfg = inducer_config("uncond", "gaussian", 128)
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
    print(f"I=128 losses {losses}, 2-step sample of the trained model rel rms vs oracle {e:.2e}")
    assert e <= 2e-2


# ------------------------------------------------------------------------------------------------ g. refusals
@pytest.mark.parametrize("inducers", REFUSED)
def test_refused_inducers(cuda, inducers):
    """Counts that are not whole 64-inducer blocks up to 256 are refused at the first call with a message naming the
    inducers; a valid model still runs afterwards."""
    from gecco_b200._abi import GeccoError

    cfg = inducer_config("uncond", "gaussian", inducers)
    model = build(cfg, cuda)
    with pytest.raises((GeccoError, ValueError), match="inducers"):
        with torch.no_grad():
            model(torch.randn(1, 100, 3, device=cuda), torch.ones(1, device=cuda), None)
    good = BY_NAME["uncond_gaussian_i128_c384_h8"]
    model, _, _, _ = _model(good, cuda, 1)
    xs, sig = _x(1, 300)
    with torch.no_grad():
        D = model(xs.to(cuda), sig.to(cuda), None)
    D_ref, _ = _oracle(good, cuda, xs, sig, None, None)
    check(D, D_ref, xs.to(cuda), sig.to(cuda), good.sigma_data, "valid model after a refusal")

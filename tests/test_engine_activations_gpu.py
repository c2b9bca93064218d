"""The ReLU and raw-Gaussian MLP activations on the device (tests/engine_activations.py): every kernel that applies the
activation in an epilogue against fp32 torch on the same bf16 operands, then the denoiser engine against the float64
oracle at the gates of test_engine_configs_gpu.py (F and D rel rms <= 1.5e-2 and rel max <= 8e-2 per cloud, inducer
states rel rms <= 1.5e-2), at each MLP launch site, in the samplers, the stand-alone module forwards, a default-constructed
(ReLU) model trained and then sampled, and the refused activations."""
import math

import pytest
import torch

from oracle import gecco_oracle as O
from tests import synth
from tests import engine_activations as A
from tests.engine_activations import ACTIVATIONS, CONFIGS, PROD, activation_config, build, oracle_activation, set_transformer
from tests.test_engine_configs_gpu import _oracle as _oracle_gaussian
from tests.test_engine_configs_gpu import _x, check, check_h

pytestmark = pytest.mark.gpu

CODE = {"gaussian_raw": 2, "relu": 3}  # GECCO_ACT_*


def _act(name, z, alpha):
    return torch.exp(-z * z / (2 * alpha * alpha)) if name == "gaussian_raw" else torch.relu(z)


def _oracle(cfg, *args, **kw):
    """test_engine_configs_gpu._oracle (float64 denoise) with the MLPs of `cfg`'s activation."""
    with oracle_activation(cfg.activation):
        return _oracle_gaussian(cfg, *args, **kw)


def _rel(a, b):
    a, b = a.cpu().double(), b.cpu().double()
    return (a - b).pow(2).mean().sqrt().item() / b.pow(2).mean().sqrt().item()


def _model(cfg, cuda, clouds: int, state_dict=None):
    import gecco_b200 as G

    feats = cfg.features(clouds) if cfg.kind == "cond" else None
    model = build(cfg, cuda, feats, state_dict=state_dict)
    ctx = K = None
    if cfg.kind == "cond":
        K = synth.camera(clouds, cfg.K)
        ctx = G.Context3d(image=torch.zeros(clouds, 3, 8, 8, device=cuda), K=K.to(cuda))
    return model, ctx, feats, K


# ------------------------------------------------------------------------------------------------ a. op level
@pytest.mark.parametrize("path", ["single_cta", "pair_generic", "pair_fast"])
@pytest.mark.parametrize("act", ACTIVATIONS)
def test_gemm_activation(cuda, act, path):
    """bias + activation -> bf16 (+ fp32 on the generic kernels) on each epilogue, against fp32 torch; ReLU with a positive
    bias makes the padding rows non-zero before the masking, which must leave them exactly 0."""
    from gecco_b200 import ops

    clouds, Np, N, K, n_out, alpha = 4, 512, 300, 384, 768, 1.3
    g = synth.gen(17)
    a = torch.randn(clouds, Np, K, generator=g)
    a[:, N:] = 0
    a = a.reshape(clouds * Np, K).to(cuda).bfloat16()
    w = (torch.randn(n_out, K, generator=g) / math.sqrt(K)).to(cuda).bfloat16()
    bias = (0.5 + 0.3 * torch.randn(n_out, generator=g)).to(cuda)
    out32 = None if path == "pair_fast" else torch.full((clouds * Np, n_out), 7.0, device=cuda)
    out16 = torch.full((clouds * Np, n_out), 7.0, device=cuda, dtype=torch.bfloat16)
    try:
        ops.set_option("gemm_pairs", 0 if path == "single_cta" else 1)
        ops.set_option("fast_epilogue", 1 if path == "pair_fast" else 0)
        ops.gemm(a, w, bias=bias, act=CODE[act], act_alpha=alpha, out_f32=out32, out_bf16=out16, rows_per_cloud=Np,
                 valid_rows=N)
    finally:
        ops.set_option("gemm_pairs", 1)
        ops.set_option("fast_epilogue", 1)
    torch.cuda.synchronize()
    ref = _act(act, a.float() @ w.float().t() + bias, alpha).view(clouds, Np, n_out)
    o16 = out16.view(clouds, Np, n_out)
    assert (o16[:, :N].float() - ref[:, :N]).abs().max().item() < 2e-2 * ref.abs().max().item()
    assert o16[:, N:].abs().max().item() == 0.0
    if out32 is not None:
        o32 = out32.view(clouds, Np, n_out)
        assert (o32[:, :N] - ref[:, :N]).abs().max().item() < 1e-3 * ref.abs().max().item() + 1e-4
        assert o32[:, N:].abs().max().item() == 0.0
        assert torch.equal(o32.bfloat16(), o16)


def _mlp_operands(g, cuda, clouds, Np, N, C=384, hidden=768):
    xf = torch.randn(clouds * Np, C, generator=g) * 1.5 + 0.3
    xf.view(clouds, Np, C)[:, N:] = 0
    w1 = (torch.randn(hidden, C, generator=g) / math.sqrt(C)).to(cuda).bfloat16()
    b1 = (0.2 + 0.3 * torch.randn(hidden, generator=g)).to(cuda)
    w2 = (torch.randn(C, hidden, generator=g) / math.sqrt(hidden)).to(cuda).bfloat16()
    b2 = torch.randn(C, generator=g).to(cuda)
    return xf.to(cuda), w1, b1, w2, b2


@pytest.mark.parametrize("anorm", [False, True], ids=["mlp_fused", "mlp_pair"])
@pytest.mark.parametrize("act", ACTIVATIONS)
def test_mlp_activation(cuda, act, anorm):
    """gecco_mlp on the fused kernel (no AdaGN) and the CTA-pair kernel (AdaGN on the A operand) against torch and against
    the same product as two gecco_gemm launches (the hidden tensor through HBM): outputs to bf16 rounding of the hidden,
    statistics to 1e-5 relative, padding rows exactly 0."""
    from gecco_b200 import ops

    C, hidden, alpha = 384, 768, 1.3
    clouds, Np, N = 3, 2048, 2000
    g = synth.gen(23 + anorm)
    xf, w1, b1, w2, b2 = _mlp_operands(g, cuda, clouds, Np, N)
    xb = xf.bfloat16()
    an = None
    if anorm:
        t = torch.randn(clouds, generator=g).to(cuda)
        sw, sb, bw, bb = [(torch.randn(C, generator=g) * k + o).to(cuda) for k, o in ((0.5, 0), (0.3, 1), (0.5, 0), (0.3, 0))]
        an = dict(stats=ops.group_stats(xf, Np, N, 12), t=t, scale_w=sw, scale_b=sb, bias_w=bw, bias_b=bb, groups=32)
    outs = {}
    for how in ("fused", "two_gemm"):
        x = xf.clone()
        xo = torch.full((clouds * Np, C), 7.0, device=cuda, dtype=torch.bfloat16)
        st = torch.zeros(clouds, C // 12, 2, dtype=torch.float64, device=cuda)
        if how == "fused":
            ops.mlp(xb, w1, b1, alpha, w2, b2, x, out_f32=x, out_bf16=xo, stats=st, rows_per_cloud=Np, valid_rows=N, anorm=an,
                    act=CODE[act])
        else:
            _, h = ops.gemm(xb, w1, bias=b1, act=CODE[act], act_alpha=alpha, out_bf16=True, rows_per_cloud=Np, valid_rows=N,
                            anorm=an)
            ops.gemm(h, w2, bias=b2, res=x, out_f32=x, out_bf16=xo, stats=st, rows_per_cloud=Np, valid_rows=N)
        outs[how] = (x, xo, st)
    torch.cuda.synchronize()
    (x1, xo1, st1), (x2, xo2, st2) = outs["fused"], outs["two_gemm"]
    a_in = xb.float()
    if anorm:
        from tests.test_mlp_fused_gpu import _adagn_ref

        a_in = _adagn_ref(xb.float(), None, an["t"], an["scale_w"], an["scale_b"], an["bias_w"], an["bias_b"], clouds, Np,
                          N).bfloat16().float()
    h = _act(act, a_in @ w1.float().t() + b1, alpha).bfloat16().float()
    ref = (xf + h @ w2.float().t() + b2).view(clouds, Np, C)[:, :N]
    for x, xo, st in outs.values():
        xv = x.view(clouds, Np, C)
        assert _rel(xv[:, :N] - xf.view(clouds, Np, C)[:, :N], ref - xf.view(clouds, Np, C)[:, :N]) < 6e-3
        assert x.view(clouds, Np, C)[:, N:].abs().max().item() == 0.0
        assert xo.view(clouds, Np, C)[:, N:].abs().max().item() == 0.0
        assert torch.equal(xo.view(clouds, Np, C)[:, :N], xv[:, :N].bfloat16())
    assert (x1 - x2).abs().max().item() < 5e-3 * x2.abs().max().item()
    assert torch.allclose(st1, st2, rtol=1e-5, atol=1e-2), (st1 - st2).abs().max()
    for x, _, st in outs.values():
        v = x.view(clouds, Np, C)[:, :N].double().reshape(clouds, N, C // 12, 12)
        assert torch.allclose(st[:, :, 0], v.sum(dim=(1, 3)), rtol=1e-6, atol=1e-2)
        assert torch.allclose(st[:, :, 1], (v * v).sum(dim=(1, 3)), rtol=1e-6, atol=1e-2)


@pytest.mark.parametrize("act", ACTIVATIONS)
def test_inducer_chain_activation(cuda, act):
    """The cluster kernel with the activation against an fp32 torch restatement on the same bf16 operands."""
    from gecco_b200 import ops
    from tests.test_chain_gpu import C, NI, _adagn, _bf, _weights

    clouds, alpha = 5, 1.3
    w, g = _weights(40)
    w["b0"] = w["b0"] + 0.3
    pooled = torch.randn(clouds * NI, C, generator=g) * 1.5 + 0.2
    t = torch.randn(clouds, generator=g)
    bf = torch.bfloat16
    d = lambda x, dt=None: x.to(cuda, dtype=dt) if dt else x.to(cuda)
    h3, khv, _, cache = ops.inducer_chain(
        d(pooled, bf), d(w["pool_out"], bf), [d(x) for x in w["n1"]], d(w["mlp0"], bf), d(w["b0"]), alpha, d(w["mlp2"], bf),
        d(w["b2"]), [d(x) for x in w["n2"]], d(w["kv"], bf), d(w["bkv"]), d(t), act=CODE[act])
    torch.cuda.synchronize()
    h = _bf(pooled) @ w["pool_out"].t()
    hn = _bf(_adagn(h, t, w["n1"], clouds))
    hh = _bf(_act(act, hn @ w["mlp0"].t() + w["b0"], alpha))
    h3_ref = _adagn(hh @ w["mlp2"].t() + w["b2"], t, w["n2"], clouds)
    khv_ref = _bf(h3_ref) @ w["kv"].t() + w["bkv"]
    assert _rel(cache, h3_ref) < 1e-2 and _rel(h3.float(), h3_ref) < 1.2e-2 and _rel(khv.float(), khv_ref) < 1.5e-2


# ------------------------------------------------------------------------------------------------ b. denoise
@pytest.mark.parametrize("clouds,points", [(4, 2048), (3, 1000), (2, 300)])
@pytest.mark.parametrize("cfg", CONFIGS, ids=lambda c: c.name)
def test_denoise_activation(cuda, cfg, clouds, points):
    """Full evaluation with do_cache=True, then the cached evaluation at another point count, against the oracle."""
    model, ctx, feats, K = _model(cfg, cuda, clouds)
    x, sig = _x(clouds, points)
    with torch.no_grad():
        D, hs = model(x.to(cuda), sig.to(cuda), ctx, do_cache=True)
    D_ref, hs_ref = _oracle(cfg, cuda, x, sig, feats, K)
    check(D, D_ref, x.to(cuda), sig.to(cuda), cfg.sigma_data, f"{cfg.name} {clouds}x{points} D")
    check_h(hs, hs_ref, f"{cfg.name} {clouds}x{points} h")
    x2, _ = _x(clouds, 450, seed=81)
    with torch.no_grad():
        Dc = model(x2.to(cuda), sig.to(cuda), ctx, cache=hs)
    Dc_ref, _ = _oracle(cfg, cuda, x2, sig, feats, K, hs=hs_ref)
    check(Dc, Dc_ref, x2.to(cuda), sig.to(cuda), cfg.sigma_data, f"{cfg.name} {clouds}x450 cached")


@pytest.mark.parametrize("option", ["mlp_pair", "chain", "anorm"])
def test_launch_sites_relu(cuda, option):
    """The ReLU production denoise with one fused path switched off: the two-GEMM AdaGN MLP, the separate inducer-side
    launches (and the separate key / value projection of the cached evaluation), the fold path."""
    from gecco_b200 import ops

    cfg = PROD["relu"]
    clouds, points = 4, 2048
    model, ctx, feats, K = _model(cfg, cuda, clouds)
    x, sig = _x(clouds, points)
    x2, _ = _x(clouds, 450, seed=81)
    try:
        ops.set_option(option, 0)
        with torch.no_grad():
            D, hs = model(x.to(cuda), sig.to(cuda), ctx, do_cache=True)
            Dc = model(x2.to(cuda), sig.to(cuda), ctx, cache=hs)
    finally:
        ops.set_option(option, 1)
    D_ref, hs_ref = _oracle(cfg, cuda, x, sig, feats, K)
    check(D, D_ref, x.to(cuda), sig.to(cuda), cfg.sigma_data, f"{option}=0 D")
    check_h(hs, hs_ref, f"{option}=0 h")
    Dc_ref, _ = _oracle(cfg, cuda, x2, sig, feats, K, hs=hs_ref)
    check(Dc, Dc_ref, x2.to(cuda), sig.to(cuda), cfg.sigma_data, f"{option}=0 cached")


# ------------------------------------------------------------------------------------------------ c. samplers (ReLU)
def _tame(cfg, cuda, clouds):
    sd = synth.tame(cfg.state_dict(), 0.15)
    model, ctx, feats, K = _model(cfg, cuda, clouds, state_dict=sd)
    return model, ctx, feats, K, sd


def test_sample_stochastic_relu(cuda):
    """Two stochastic steps against the oracle's sampler; the same call again replays the cached graph bit for bit."""
    from gecco_b200.engine import engine_for

    cfg = PROD["relu"]
    B, shape = 2, (2, 2048, 3)
    model, ctx, feats, K, sd = _tame(cfg, cuda, B)
    s = model.sample_stochastic(shape, ctx, rng=synth.gen(5), num_steps=2)
    with oracle_activation("relu"):
        o = O.sample_stochastic(cfg.oracle(), sd, shape, feats, K, rng=synth.gen(5), num_steps=2)
    assert torch.isfinite(s).all()
    e = _rel(s, o)
    print(f"ReLU 2-step stochastic sample rel rms vs oracle {e:.2e}")
    assert e <= 2e-2
    eng = engine_for(*model._network())
    assert eng.graph_status() in (1, 2)
    s2 = model.sample_stochastic(shape, ctx, rng=synth.gen(5), num_steps=2)
    assert eng.graph_status() == 2 and torch.equal(s, s2)


def test_sample_ode_relu(cuda):
    cfg = PROD["relu"]
    B, N, steps = 2, 300, 8
    model, ctx, feats, K, sd = _tame(cfg, cuda, B)
    got = model.sample_ode((B, N, 3), ctx, rng=synth.gen(3), num_steps=steps)
    with oracle_activation("relu"):
        ref = O.sample_stochastic(cfg.oracle(), sd, (B, N, 3), feats, K, rng=synth.gen(3), num_steps=steps, S_churn=0.0)
    to_diff = lambda d: O.data_to_diffusion(cfg.oracle(), sd, d.cpu().double(), None)
    e = _rel(to_diff(got), to_diff(ref))
    print(f"ReLU ODE sample rel rms (diffusion space) {e:.2e}")
    assert e < 1e-2


def test_sample_inpaint_relu(cuda):
    cfg = PROD["relu"]
    B, N, M, steps = 2, 200, 184, 4
    model, _, _, _, sd = _tame(cfg, cuda, B)
    oc = cfg.oracle()
    known = O.diffusion_to_data(oc, sd, torch.randn(B, N, 3, generator=synth.gen(5)), None)
    got = model.sample_inpaint(known.to(cuda), M, None, rng=synth.gen(6), num_substeps=2, num_steps=steps, S_churn=0.5)
    with oracle_activation("relu"):
        ref = O.sample_inpaint(oc, sd, known, M, rng=synth.gen(6), num_substeps=2, num_steps=steps, S_churn=0.5)
    to_diff = lambda d: O.data_to_diffusion(oc, sd, d.cpu().double(), None)
    e = _rel(to_diff(got), to_diff(ref))
    print(f"ReLU inpaint rel rms (diffusion space) {e:.2e}")
    assert got.shape == (B, M, 3) and e < 1e-2


def test_upsample_relu(cuda):
    """Upsampling at a small sigma_max (contractive), the cached inducer evaluations through the same launch sites."""
    cfg = activation_config("relu", "cond", "uvl")
    B = 2
    model, ctx, feats, K = _model(cfg, cuda, B)
    sd = cfg.state_dict()
    oc = cfg.oracle()
    seed_cloud = O.diffusion_to_data(oc, sd, torch.randn(B, 128, 3, generator=synth.gen(35)), K)
    us = model.upsample(seed_cloud.to(cuda), n_new=200, context=ctx, num_substeps=3, num_steps=3, sigma_max=0.05,
                        rng=synth.gen(9))
    with oracle_activation("relu"):
        uo = O.upsample(oc, sd, seed_cloud, n_new=200, features=feats, K=K, seed=9, num_substeps=3, num_steps=3, sigma_max=0.05)
    assert torch.isfinite(us).all()
    to_diff = lambda d: O.data_to_diffusion(oc, sd, d.cpu().double(), K.double())
    e = _rel(to_diff(us), to_diff(uo))
    print(f"ReLU small-sigma upsample rel rms vs oracle {e:.2e}")
    assert e <= 1e-2


# ------------------------------------------------------------------------------------------------ d. module forwards
def test_module_forwards_relu(cuda):
    """Stand-alone MLP, Broadcast and SetTransformer forwards with ReLU against the float64 oracle on the same weights."""
    cfg = PROD["relu"]
    oc = cfg.oracle()
    pre = oc.st_prefix
    sd = cfg.state_dict()
    st = set_transformer(cfg)
    st.load_state_dict({k[len(pre):]: v for k, v in sd.items() if k.startswith(pre)})
    st = st.to(cuda).eval()
    sd64 = {k: v.to(cuda, torch.float64) for k, v in sd.items()}
    B, C, H = 2, cfg.width, cfg.heads
    x = torch.randn(B, 1000, C, generator=synth.gen(41)).to(cuda)
    t = (torch.randn(B, 1, 1, generator=synth.gen(43)) * 0.5).to(cuda)
    xd, td = x.double(), t.double()
    lp = pre + "layers.0."
    errs = {"mlp": _rel(st.layers[0].mlp(x), A.mlp(sd64, lp + "mlp.", xd, "relu"))}
    h_ref = O.attention_pool(sd64, lp + "broadcast.pool.", xd, H)
    h_ref = O.adagn(sd64, lp + "broadcast.norm_1.", h_ref, td)
    h_ref = A.mlp(sd64, lp + "broadcast.mlp.", h_ref, "relu")
    h_ref = O.adagn(sd64, lp + "broadcast.norm_2.", h_ref, td)
    attn, h = st.layers[0].broadcast(x, t, return_h=True)
    errs["broadcast"] = _rel(attn, O.mha_unpool(sd64, lp + "broadcast.unpool.", xd, h_ref, H))
    errs["broadcast_h"] = _rel(h, h_ref)
    f, hs = st(x, t, return_h=True)
    with oracle_activation("relu"):
        f_ref, hs_ref = O.set_transformer(oc, sd64, xd, td)
    errs["st"] = _rel(f, f_ref)
    for l, (a, b) in enumerate(zip(hs, hs_ref)):
        errs[f"st_h{l}"] = _rel(a, b)
    print({k: f"{v:.2e}" for k, v in errs.items()})
    bad = {k: v for k, v in errs.items() if v > 1.5e-2}
    assert not bad, bad


# ------------------------------------------------------------------------------------------------ e. train, then sample
def test_train_then_sample_default_relu(cuda):
    """A default-constructed SetTransformer (ReLU MLPs) trained by Trainer (eager) for three steps, then sampled by the
    engine, against the oracle's sampler on the trained weights."""
    from gecco_b200.models import SetTransformer
    from gecco_b200.training import Trainer

    cfg = PROD["relu"]
    B = 2
    st = SetTransformer(n_layers=cfg.layers, feature_dim=cfg.width, num_inducers=cfg.inducers, t_embed_dim=1)
    sd = synth.tame(cfg.state_dict(), 0.15)
    model = build(cfg, cuda, state_dict=sd, st=st)
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
    with oracle_activation("relu"):
        o = O.sample_stochastic(cfg.oracle(), trained, shape, None, None, rng=synth.gen(5), num_steps=2)
    assert torch.isfinite(s).all()
    e = _rel(s, o)
    print(f"ReLU losses {losses}, 2-step sample of the trained model rel rms vs oracle {e:.2e}")
    assert e <= 2e-2


# ------------------------------------------------------------------------------------------------ f. refusals
@pytest.mark.parametrize("kind", ["GELU", "mixed"])
def test_refused_activation(cuda, kind):
    """nn.GELU, and a model whose MLPs mix activations, are refused at the first call with a message naming the
    activation; a valid model still runs afterwards."""
    from gecco_b200.models import GaussianActivation, SetTransformer

    cfg = PROD["relu"]
    if kind == "GELU":
        st = SetTransformer(n_layers=cfg.layers, feature_dim=cfg.width, num_inducers=cfg.inducers, t_embed_dim=1,
                            activation=torch.nn.GELU)
        model = build(cfg, cuda, st=st)
    else:
        model = build(cfg, cuda)
        model.backbone.model.inner.layers[1].broadcast.mlp[1] = GaussianActivation().to(cuda)
    with pytest.raises(ValueError, match="GELU" if kind == "GELU" else "same activation"):
        with torch.no_grad():
            model(torch.randn(1, 100, 3, device=cuda), torch.ones(1, device=cuda), None)
    model, _, _, _ = _model(cfg, cuda, 1)
    xs, sig = _x(1, 300)
    with torch.no_grad():
        D = model(xs.to(cuda), sig.to(cuda), None)
    D_ref, _ = _oracle(cfg, cuda, xs, sig, None, None)
    check(D, D_ref, xs.to(cuda), sig.to(cuda), cfg.sigma_data, "valid model after a refusal")

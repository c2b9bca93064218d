"""The oracle is well-conditioned at every configuration of tests/engine_configs.py: in float32 it agrees with itself in
float64 to 1e-4 relative rms of the raw network output F, so the float64 oracle is a sharp reference for the bf16 engine
(whose gates are 1.5e-2, test_engine_configs_gpu.py).  Also pins the synthetic-weight plumbing those tests rely on."""
import pytest
import torch

from oracle import gecco_oracle as O
from tests import synth
from tests.engine_configs import CONFIGS, raw_output, rms


def _inputs(cfg, clouds, points, dtype):
    sd = {k: v.to(dtype) for k, v in cfg.state_dict().items()}
    sig = torch.tensor([0.3, 40.0])[:clouds]
    x = synth.noisy_input(clouds, points, sig, 61, 62)
    feats = K = None
    if cfg.kind == "cond":
        feats = [f.to(dtype) for f in cfg.features(clouds)]
        K = synth.camera(clouds, cfg.K).to(dtype)
    return sd, x, sig, feats, K


@pytest.mark.parametrize("cfg", CONFIGS, ids=lambda c: c.name)
def test_oracle_float32_matches_float64(cfg):
    B, N = 2, 200
    out = {}
    for dt in (torch.float32, torch.float64):
        sd, x, sig, feats, K = _inputs(cfg, B, N, dt)
        D, hs = O.denoise(cfg.oracle(), sd, x.to(dt), sig.to(dt), feats, K, return_h=True)
        assert D.dtype == dt and len(hs) == cfg.layers
        out[dt] = raw_output(D, x, sig, cfg.sigma_data), hs
    (F32, h32), (F64, h64) = out[torch.float32], out[torch.float64]
    assert torch.isfinite(F64).all()
    for b in range(B):
        e = rms(F32[b] - F64[b]) / rms(F64[b])
        print(f"{cfg.name}[{b}] sigma={sig[b].item():g}: float32 vs float64 rel rms {e:.2e}")
        assert e <= 1e-4, (cfg.name, b, e)
    for l, (a, b) in enumerate(zip(h32, h64)):
        assert rms(a.double() - b) <= 1e-4 * rms(b), (cfg.name, l)


@pytest.mark.parametrize("cfg", CONFIGS, ids=lambda c: c.name)
def test_state_dict_matches_module(cfg):
    """The synthetic state dict of a configuration has exactly the parameter names and shapes of the module that the
    reference constructor keywords build (tests.models_b200.build)."""
    from tests.models_b200 import build

    model = build(cfg.kind, cfg.reparam, cfg.stats["mean"], cfg.stats["sigma"], cfg.sigma_max, None, "cpu", **cfg.build_kw())
    want = {k: tuple(v.shape) for k, v in model.state_dict().items()}
    got = {k: tuple(v.shape) for k, v in cfg.state_dict().items()}
    assert want == got
    assert model.backbone.sigma_data == cfg.sigma_data and model.loss.sigma_data == cfg.sigma_data


def test_default_recipe_unchanged():
    """do_norm=True is the default recipe: same keys, same generator draws (the goldens are regenerated from it)."""
    base = synth.full_state_dict("uncond", "gaussian", [0.0] * 3, [1.0] * 3, 7, n_layers=1)
    again = synth.full_state_dict("uncond", "gaussian", [0.0] * 3, [1.0] * 3, 7, n_layers=1, do_norm=True)
    assert base.keys() == again.keys() and all(torch.equal(base[k], again[k]) for k in base)
    assert "backbone.model.lower.1.weight" in base
    bare = synth.full_state_dict("uncond", "gaussian", [0.0] * 3, [1.0] * 3, 7, n_layers=1, do_norm=False)
    assert set(bare) ^ set(base) == {"backbone.model.lower.weight", "backbone.model.lower.bias",
                                     "backbone.model.lower.1.weight", "backbone.model.lower.1.bias"}
    tamed = synth.tame(bare, 0.5)
    assert torch.equal(tamed["backbone.model.lower.weight"], 0.5 * bare["backbone.model.lower.weight"])


def test_oracle_head_without_norm():
    """`lower.weight` in the state dict selects the bare Linear head (models/linear_lift.py, do_norm=False)."""
    sd = synth.full_state_dict("uncond", "gaussian", [0.0] * 3, [1.0] * 3, 3, n_layers=1, do_norm=False)
    oc = O.OracleConfig(kind="uncond", n_layers=1, reparam="gaussian")
    x = torch.randn(1, 50, 3, generator=synth.gen(4))
    t = torch.full((1, 1, 1), 0.1)
    F_got, _ = O.network(oc, sd, x, t, None, None)
    p = oc.net_prefix
    y = torch.nn.functional.linear(x, sd[p + "lift.weight"], sd[p + "lift.bias"])
    y, _ = O.set_transformer(oc, sd, y, t)
    assert torch.allclose(F_got, torch.nn.functional.linear(y, sd[p + "lower.weight"], sd[p + "lower.bias"]))

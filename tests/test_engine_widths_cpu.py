"""The test helpers at feature widths other than 384 (tests/engine_widths.py): at 384 they reproduce the production recipe
and model of tests/synth.py and tests/models_b200.py bit for bit, the synthetic state dict matches the module the
constructor builds at every width, and the float64 oracle (which reads every width from the state dict) runs and agrees
with itself in float32 at every width."""
import pytest
import torch

from oracle import gecco_oracle as O
from tests import synth
from tests.engine_configs import Config, raw_output, rms
from tests.engine_widths import CONFIGS, WIDTHS, WidthConfig, build, width_config


@pytest.mark.parametrize("kind,reparam", [("uncond", "gaussian"), ("cond", "gaussian"), ("cond", "uvl")])
def test_width_recipe_at_384_is_the_production_recipe(kind, reparam):
    base = Config("base", kind=kind, reparam=reparam).state_dict()
    again = WidthConfig("again", kind=kind, reparam=reparam, width=synth.FEATURE_DIM).state_dict()
    assert list(base) == list(again) and all(torch.equal(base[k], again[k]) for k in base)


@pytest.mark.parametrize("kind,reparam", [("uncond", "gaussian"), ("cond", "uvl")])
def test_width_model_at_384_is_the_production_model(kind, reparam):
    from tests import models_b200

    cfg = WidthConfig("w384", kind=kind, reparam=reparam, width=synth.FEATURE_DIM)
    base = models_b200.build(kind, reparam, cfg.stats["mean"], cfg.stats["sigma"], cfg.sigma_max, 1234, "cpu",
                             **cfg.build_kw()).state_dict()
    again = build(cfg, "cpu").state_dict()
    assert list(base) == list(again) and all(torch.equal(base[k], again[k]) for k in base)


@pytest.mark.parametrize("cfg", CONFIGS, ids=lambda c: c.name)
def test_state_dict_matches_module(cfg):
    model = build(cfg, "cpu", weight_seed=None)
    want = {k: tuple(v.shape) for k, v in model.state_dict().items()}
    got = {k: tuple(v.shape) for k, v in cfg.state_dict().items()}
    assert want == got
    assert got[[k for k in got if k.endswith("layers.0.mlp.0.weight")][0]] == (2 * cfg.width, cfg.width)


@pytest.mark.parametrize("cfg", CONFIGS, ids=lambda c: c.name)
def test_oracle_runs_at_width(cfg):
    """float32 against float64 on the same inputs: D has the input's shape, the inducer states are [clouds, 64, C], and the
    two precisions agree to 1e-4 of F, so the float64 oracle is a sharp reference for the bf16 engine at this width."""
    B, N = 2, 150
    sig = torch.tensor([0.3, 40.0])
    x = synth.noisy_input(B, N, sig, 61, 62)
    out = {}
    for dt in (torch.float32, torch.float64):
        sd = {k: v.to(dt) for k, v in cfg.state_dict().items()}
        feats = K = None
        if cfg.kind == "cond":
            feats = [f.to(dt) for f in cfg.features(B)]
            K = synth.camera(B, cfg.K).to(dt)
        D, hs = O.denoise(cfg.oracle(), sd, x.to(dt), sig.to(dt), feats, K, return_h=True)
        assert D.shape == (B, N, 3) and len(hs) == cfg.layers
        assert all(tuple(h.shape) == (B, synth.NUM_INDUCERS, cfg.width) for h in hs)
        out[dt] = raw_output(D, x, sig, cfg.sigma_data)
    F32, F64 = out[torch.float32], out[torch.float64]
    assert torch.isfinite(F64).all()
    for b in range(B):
        assert rms(F32[b] - F64[b]) <= 1e-4 * rms(F64[b]), (cfg.name, b)


def test_widths_cover_every_supported_group_width():
    assert sorted([c // 32 for c, _ in WIDTHS] + [synth.FEATURE_DIM // 32]) == [4, 8, 12, 16, 24, 32]
    assert width_config("uncond", "gaussian", 512, 8).state_dict()["backbone.model.lift.weight"].shape == (512, 3)

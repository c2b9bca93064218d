"""The test helpers at inducer counts other than 64 (tests/engine_inducers.py): at 64 they reproduce the production
recipe and model of tests/synth.py and tests/models_b200.py bit for bit, the synthetic state dict matches the module the
constructor builds at every row, and the float64 oracle (which reads the inducers from the state dict) runs and agrees
with itself in float32 at every row."""
import pytest
import torch

from oracle import gecco_oracle as O
from tests import synth
from tests.engine_configs import Config, raw_output, rms
from tests.engine_inducers import CONFIGS, COUNTS, REFUSED, InducerConfig, build, inducer_config


@pytest.mark.parametrize("kind,reparam", [("uncond", "gaussian"), ("cond", "gaussian"), ("cond", "uvl")])
def test_inducer_recipe_at_64_is_the_production_recipe(kind, reparam):
    base = Config("base", kind=kind, reparam=reparam).state_dict()
    again = InducerConfig("again", kind=kind, reparam=reparam, inducers=synth.NUM_INDUCERS).state_dict()
    assert list(base) == list(again) and all(torch.equal(base[k], again[k]) for k in base)


@pytest.mark.parametrize("kind,reparam", [("uncond", "gaussian"), ("cond", "uvl")])
def test_inducer_model_at_64_is_the_production_model(kind, reparam):
    from tests import models_b200

    cfg = InducerConfig("i64", kind=kind, reparam=reparam, inducers=synth.NUM_INDUCERS)
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
    key = [k for k in got if k.endswith("layers.0.broadcast.pool.inducers")][0]
    assert got[key] == (1, cfg.heads, cfg.inducers, cfg.width // cfg.heads)


@pytest.mark.parametrize("cfg", CONFIGS, ids=lambda c: c.name)
def test_oracle_runs_at_inducer_count(cfg):
    """float32 against float64 on the same inputs: D has the input's shape, the inducer states are [clouds, I, C], and
    the two precisions agree to 1e-4 of F, so the float64 oracle is a sharp reference for the bf16 engine at this count."""
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
        assert all(tuple(h.shape) == (B, cfg.inducers, cfg.width) for h in hs)
        out[dt] = raw_output(D, x, sig, cfg.sigma_data)
    F32, F64 = out[torch.float32], out[torch.float64]
    assert torch.isfinite(F64).all()
    for b in range(B):
        assert rms(F32[b] - F64[b]) <= 1e-4 * rms(F64[b]), (cfg.name, b)


def test_rows_cover_every_count_and_head_dim():
    assert sorted({c.inducers for c in CONFIGS}) == COUNTS
    assert sorted({c.width // c.heads for c in CONFIGS}) == [32, 48, 64]
    assert not set(REFUSED) & set(COUNTS + [synth.NUM_INDUCERS])
    sd = inducer_config("uncond", "gaussian", 192).state_dict()
    assert sd["backbone.model.inner.layers.0.broadcast.pool.inducers"].shape == (1, 8, 192, 48)

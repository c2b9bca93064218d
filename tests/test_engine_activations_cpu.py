"""The MLP activations on the host side (tests/engine_activations.py): the engine description maps each module to its
GECCO_ACT_* code and refuses other or mixed activations, the synthetic recipe matches a default-constructed (ReLU) model and
is synth.py's at the Gaussian, and the float64 oracle applies the three formulas and is left as it was after each block."""
import pytest
import torch

from oracle import gecco_oracle as O
from tests import synth
from tests import engine_activations as A
from tests.engine_activations import ACTIVATIONS, CODES, CONFIGS, activation_config, build, oracle_activation
from tests.engine_configs import Config, raw_output, rms


def _net(model):
    return model.backbone.model


@pytest.mark.parametrize("act", ["gaussian", "gaussian_raw", "relu"])
def test_describe_maps_activation(act):
    from gecco_b200 import _abi
    from gecco_b200.engine import Engine

    cfg = activation_config(act)
    net = _net(build(cfg, "cpu"))  # the engine holds its network weakly
    d, _, layer_t = Engine(net)._describe()
    assert d.mlp_act == CODES[act]
    alphas = [layer_t[l * _abi.LW_COUNT + i] for l in range(cfg.layers) for i in (13, 30)]  # GECCO_LW_{BMLP,MLP}_ALPHA
    if act == "relu":
        assert all(a is None for a in alphas)
    else:
        assert all(isinstance(a, torch.Tensor) and a.shape == () for a in alphas)
    assert all(t is not None for i, t in enumerate(layer_t) if i % _abi.LW_COUNT not in (13, 30))


@pytest.mark.parametrize("module", ["GELU", "SiLU"])
def test_describe_refuses_other_activations(module):
    from gecco_b200.engine import Engine
    from gecco_b200.models import SetTransformer

    cfg = activation_config("relu")
    st = SetTransformer(n_layers=2, feature_dim=384, num_inducers=64, t_embed_dim=1, activation=getattr(torch.nn, module))
    net = _net(build(cfg, "cpu", st=st, weight_seed=None))
    with pytest.raises(ValueError, match=module) as e:
        Engine(net)._describe()
    assert "ReLU" in str(e.value) and "GaussianActivation" in str(e.value)


def test_describe_refuses_mixed_activations():
    from gecco_b200.engine import Engine
    from gecco_b200.models import GaussianActivation

    model = build(activation_config("relu"), "cpu")
    _net(model).inner.layers[1].mlp[1] = GaussianActivation()
    with pytest.raises(ValueError, match="same activation") as e:
        Engine(_net(model))._describe()
    assert "ReLU" in str(e.value) and "GaussianActivation" in str(e.value)


def test_default_model_is_relu_and_matches_recipe():
    """SetTransformer without `activation=` has ReLU MLPs; its state_dict keys and shapes are the ReLU recipe's."""
    from gecco_b200.models import SetTransformer

    cfg = activation_config("relu")
    st = SetTransformer(n_layers=cfg.layers, feature_dim=cfg.width, num_inducers=cfg.inducers, t_embed_dim=1)
    assert all(isinstance(l.mlp[1], torch.nn.ReLU) and isinstance(l.broadcast.mlp[1], torch.nn.ReLU) for l in st.layers)
    model = build(cfg, "cpu", st=st, weight_seed=None)
    want = {k: tuple(v.shape) for k, v in model.state_dict().items()}
    got = {k: tuple(v.shape) for k, v in cfg.state_dict().items()}
    assert want == got
    assert not any(k.endswith("alpha") for k in got)
    build(cfg, "cpu", st=st)  # the recipe loads into it


@pytest.mark.parametrize("kind", ["uncond", "cond"])
def test_gaussian_recipe_and_oracle_unchanged(kind):
    """At the Gaussians the synthetic weights are synth.py's recipe bit for bit, and the restated MLP at "gaussian" is the
    oracle's own mlp exactly."""
    base = Config("base", kind=kind).state_dict()
    for act in ("gaussian", "gaussian_raw"):
        again = activation_config(act, kind).state_dict()
        assert list(base) == list(again) and all(torch.equal(base[k], again[k]) for k in base)
    relu = activation_config("relu", kind).state_dict()
    assert sorted(relu) == sorted(k for k in base if not k.endswith("mlp.1.alpha"))
    sd = {k: v.double() for k, v in base.items()}
    pre = [k for k in sd if k.endswith("layers.0.mlp.0.weight")][0][: -len("0.weight")]
    x = torch.randn(2, 50, 384, generator=synth.gen(3), dtype=torch.float64)
    with oracle_activation("gaussian"):
        assert torch.equal(O.mlp(sd, pre, x), A.mlp(sd, pre, x, "gaussian"))


def test_oracle_activation_formulas():
    z = torch.linspace(-4, 4, 801, dtype=torch.float64)
    alpha = torch.tensor(1.3, dtype=torch.float64)
    sd = {"p.1.alpha": alpha}
    g = torch.exp(-z * z / (2 * alpha * alpha))
    assert torch.allclose(A.activation("gaussian", sd, "p.", z), (g - 0.7) / 0.28, rtol=0, atol=1e-15)
    assert torch.allclose(A.activation("gaussian_raw", sd, "p.", z), g, rtol=0, atol=1e-15)
    assert torch.equal(A.activation("relu", {}, "p.", z), torch.clamp(z, min=0))
    with pytest.raises(ValueError):
        A.activation("gelu", sd, "p.", z)


def test_oracle_activation_restores_the_oracle():
    """The oracle's mlp is the restated one inside the block only, also when the block raises."""
    original = O.mlp
    sd = {"p.0.weight": torch.eye(3, dtype=torch.float64), "p.0.bias": torch.full((3,), -1.0, dtype=torch.float64),
          "p.2.weight": torch.eye(3, dtype=torch.float64), "p.2.bias": torch.zeros(3, dtype=torch.float64)}
    x = torch.tensor([[0.5, 1.5, 3.0]], dtype=torch.float64)
    with pytest.raises(RuntimeError):
        with oracle_activation("relu"):
            assert O.mlp is not original
            assert torch.equal(O.mlp(sd, "p.", x), torch.tensor([[0.0, 0.5, 2.0]], dtype=torch.float64))
            raise RuntimeError("inside the block")
    assert O.mlp is original


@pytest.mark.parametrize("act", ACTIVATIONS)
def test_oracle_runs_with_activation(act):
    """float32 against float64 on the same inputs at the production shape: the two agree to 1e-4 of F, so the float64
    oracle is a sharp reference for the bf16 engine with this activation, and its output differs from the Gaussian model's."""
    cfg = activation_config(act)
    B, N = 2, 150
    sig = torch.tensor([0.3, 40.0])
    x = synth.noisy_input(B, N, sig, 61, 62)
    out = {}
    for dt in (torch.float32, torch.float64):
        sd = {k: v.to(dt) for k, v in cfg.state_dict().items()}
        with oracle_activation(act):
            D, hs = O.denoise(cfg.oracle(), sd, x.to(dt), sig.to(dt), None, None, return_h=True)
        out[dt] = raw_output(D, x, sig, cfg.sigma_data)
    F32, F64 = out[torch.float32], out[torch.float64]
    assert torch.isfinite(F64).all()
    for b in range(B):
        assert rms(F32[b] - F64[b]) <= 1e-4 * rms(F64[b]), (cfg.name, b)
    gauss = activation_config("gaussian")
    sd = {k: v.double() for k, v in cfg.state_dict().items()}
    D_g, _ = O.denoise(gauss.oracle(), sd if act != "relu" else {k: v.double() for k, v in gauss.state_dict().items()},
                       x.double(), sig.double(), None, None, return_h=True)
    assert rms(raw_output(D_g, x, sig, 1.0) - F64) > 1e-2 * rms(F64)


def test_rows_cover_every_path():
    assert {c.activation for c in CONFIGS} == set(ACTIVATIONS)
    for act in ACTIVATIONS:
        rows = [c for c in CONFIGS if c.activation == act]
        assert {(c.kind, c.reparam) for c in rows} == {("uncond", "gaussian"), ("cond", "gaussian"), ("cond", "uvl")}
        assert {c.width for c in rows} == {256, 384, 768} and {c.inducers for c in rows} == {64, 128}
        assert {c.blowup for c in rows} == {2, 3}

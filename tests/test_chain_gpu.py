"""The inducer side of a Broadcast layer as one cluster kernel (gecco_inducer_chain) against an fp32 torch restatement of
set_transformer.py:106-112 on the same bf16-rounded operands, and against the separate-launch path of the engine."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

C, HID, NI, NH, HD = 384, 768, 64, 8, 48


def _gen(seed):
    return torch.Generator(device="cpu").manual_seed(seed)


def _bf(x):
    return x.to(torch.bfloat16).float()


def _adagn(h, t, nw, clouds):
    # models/normalization.py:36-44 on [B, I, C]
    x = h.view(clouds, NI, C)
    normed = F.group_norm(x.transpose(1, 2), 32, eps=1e-5).transpose(1, 2)
    scale = t[:, None] * nw[0][None] + nw[1][None]
    bias = t[:, None] * nw[2][None] + nw[3][None]
    return (scale[:, None] * normed + bias[:, None]).reshape(clouds * NI, C)


def _reference(pooled, w, t, clouds, alpha):
    h = _bf(pooled) @ w["pool_out"].t()
    hn = _bf(_adagn(h, t, w["n1"], clouds))
    z = hn @ w["mlp0"].t() + w["b0"]
    hh = _bf((torch.exp(-z * z / (2 * alpha * alpha)) - 0.7) / 0.28)
    h2 = hh @ w["mlp2"].t() + w["b2"]
    h3 = _adagn(h2, t, w["n2"], clouds)
    khv = _bf(h3) @ w["kv"].t() + w["bkv"]
    return h3, khv


def _weights(seed):
    g = _gen(seed)
    r = lambda *s, k=1.0: torch.randn(*s, generator=g) * k
    w = {
        "pool_out": _bf(r(C, C, k=C**-0.5)), "mlp0": _bf(r(HID, C, k=C**-0.5)), "mlp2": _bf(r(C, HID, k=HID**-0.5)),
        "kv": _bf(r(2 * C, C, k=C**-0.5)),
        "b0": r(HID, k=0.3), "b2": r(C, k=0.3), "bkv": r(2 * C, k=0.3),
        "n1": [r(C, k=0.5), 1 + r(C, k=0.3), r(C, k=0.5), r(C, k=0.3)],
        "n2": [r(C, k=0.5), 1 + r(C, k=0.3), r(C, k=0.5), r(C, k=0.3)],
    }
    return w, g


@pytest.mark.parametrize("clouds", [1, 2, 5, 64])
def test_inducer_chain_matches_torch(cuda, clouds):
    from gecco_b200 import ops

    w, g = _weights(10 + clouds)
    alpha = 1.3
    pooled = torch.randn(clouds * NI, C, generator=g) * 1.5 + 0.2
    t = torch.randn(clouds, generator=g)
    bf = torch.bfloat16
    d = lambda x, dt=None: x.to(cuda, dtype=dt) if dt else x.to(cuda)
    h3, khv, vt, cache = ops.inducer_chain(
        d(pooled, bf), d(w["pool_out"], bf), [d(x) for x in w["n1"]], d(w["mlp0"], bf), d(w["b0"]), alpha, d(w["mlp2"], bf),
        d(w["b2"]), [d(x) for x in w["n2"]], d(w["kv"], bf), d(w["bkv"]), d(t))
    torch.cuda.synchronize()
    h3_ref, khv_ref = _reference(pooled, w, t, clouds, alpha)
    rms = lambda x: x.pow(2).mean().sqrt().item()
    e_cache = rms(cache.cpu() - h3_ref) / rms(h3_ref)
    e_h3 = rms(h3.float().cpu() - h3_ref) / rms(h3_ref)
    e_kv = rms(khv.float().cpu() - khv_ref) / rms(khv_ref)
    assert e_cache < 1e-2 and e_h3 < 1.2e-2 and e_kv < 1.5e-2, (e_cache, e_h3, e_kv)
    # V transposed per cloud: vt[cloud][c][i] = khv[cloud*64 + i][C + c], bit for bit
    v = khv.view(clouds, NI, 2 * C)[:, :, C:]
    assert torch.equal(vt, v.transpose(1, 2).contiguous())
    assert torch.equal(cache.to(bf), h3)


@pytest.mark.parametrize("clouds,N,splits", [(2, 2048, 3), (3, 500, 2)])
def test_inducer_chain_merges_key_splits(cuda, clouds, N, splits):
    """The chain's first step merges the key-split partials of the pool core: same result as gecco_pool_attention's own
    merge followed by the chain."""
    from gecco_b200 import _abi, ops
    import ctypes as Ct

    w, g = _weights(31)
    Np = (N + 127) // 128 * 128
    bf = torch.bfloat16
    kv = torch.zeros(clouds, Np, 2 * C)
    kv[:, :N] = torch.randn(clouds, N, 2 * C, generator=g)
    kv = kv.reshape(clouds * Np, 2 * C).to(cuda, dtype=bf)
    qi = (torch.randn(NH, NI, HD, generator=g) * 0.3).to(cuda, dtype=bf)
    t = torch.randn(clouds, generator=g).to(cuda)
    pooled = ops.pool_attention(kv, qi, clouds=clouds, rows_per_cloud=Np, valid_rows=N, heads=NH, head_dim=HD, k_off=0, v_off=C,
                                splits=splits)
    d = lambda x, dt=None: x.to(cuda, dtype=dt) if dt else x.to(cuda)
    args = (d(w["pool_out"], bf), [d(x) for x in w["n1"]], d(w["mlp0"], bf), d(w["b0"]), 1.1, d(w["mlp2"], bf), d(w["b2"]),
            [d(x) for x in w["n2"]], d(w["kv"], bf), d(w["bkv"]), t)
    ref = ops.inducer_chain(pooled, *args)
    # the same with the merge inside the chain: run the pool core and leave the partials
    partial, used = ops.pool_attention_partial(kv, qi, clouds=clouds, rows_per_cloud=Np, valid_rows=N, heads=NH, head_dim=HD,
                                               k_off=0, v_off=C, splits=splits)
    scratch = torch.zeros_like(pooled) if used > 1 else pooled
    got = ops.inducer_chain(scratch, *args, partial=partial, splits=used)
    torch.cuda.synchronize()
    if used > 1:
        assert torch.equal(scratch, pooled)
    for a, b in zip(got[:3], ref[:3]):
        assert torch.equal(a, b)


def test_engine_chain_matches_separate_launches(cuda):
    """One denoiser evaluation with the chain kernel against the same evaluation with the "chain" option off."""
    from gecco_b200 import ops
    from tests import synth
    from tests.models_b200 import build as build_model

    B, N = 3, 700
    model = build_model("uncond", "gaussian", [0.0, 0.0, 0.0], [1.0, 1.0, 1.0], 80.0, 77, cuda, None)
    x = (torch.randn(B, N, 3, generator=synth.gen(5)) * 1.5).to(cuda)
    sig = torch.tensor([0.1, 1.0, 30.0], device=cuda)
    try:
        ops.set_option("chain", 0)
        d0, c0 = model(x, sig, None, do_cache=True)
        ops.set_option("chain", 1)
        d1, c1 = model(x, sig, None, do_cache=True)
    finally:
        ops.set_option("chain", 1)
    torch.cuda.synchronize()
    rms = lambda v: v.float().pow(2).mean().sqrt().item()
    assert rms(d1 - d0) < 1e-2 * rms(d0), rms(d1 - d0) / rms(d0)
    for a, b in zip(c0, c1):
        assert rms(a - b) < 1e-2 * rms(a)
    # cached evaluation (first_stage = 3 of the chain) against the separate key / value projection
    try:
        ops.set_option("chain", 0)
        e0 = model(x, sig, None, cache=c0)
        ops.set_option("chain", 1)
        e1 = model(x, sig, None, cache=c0)
    finally:
        ops.set_option("chain", 1)
    assert rms(e1 - e0) < 1e-3 * rms(e0), rms(e1 - e0) / rms(e0)

"""CPU oracle for the gecco-torch reverse-diffusion sampling path.  TEST INFRASTRUCTURE ONLY.

A functional (state_dict in, tensors out) restatement of the reference algorithm in plain fp32
torch, written from the reference sources and checked against golden vectors produced by the
UNMODIFIED reference package (oracle/make_golden.py -> tests/golden/*.pt, tests/test_oracle.py).
Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import
this module; nothing under gecco_b200/ does.

Parity pinning: the reference ships no tests or golden vectors of its own (SURVEY.md §4), so the
oracle is pinned against outputs of the reference itself run in the build container through the
import stubs in oracle/stubs/ (kornia's projection arithmetic is restated there: "parity unpinned"
at that third-party boundary only, see oracle/stubs/kornia/geometry/camera/perspective.py).

All citations are relative to /root/reference/gecco-torch/src/gecco_torch/.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import Optional, Sequence

import torch
import torch.nn.functional as F
from torch import Tensor


@dataclass
class OracleConfig:
    """Hyper-parameters that are not recoverable from tensor shapes alone."""

    kind: str = "uncond"  # "uncond": LinearLift (models/linear_lift.py), "cond": RayNetwork (models/ray.py)
    n_layers: int = 6
    num_heads: int = 8
    reparam: str = "none"  # "none" | "gaussian" | "uvl"   (reparam.py)
    logit_scale: float = 1.1
    sigma_data: float = 1.0
    sigma_max: float = 165.0
    net_prefix: str = "backbone.model."
    sampler: dict = field(
        default_factory=lambda: dict(num_steps=64, sigma_min=0.002, rho=7, S_churn=0.5, S_min=0, S_max=float("inf"), S_noise=1)
    )

    @property
    def st_prefix(self) -> str:
        return self.net_prefix + ("inner." if self.kind == "uncond" else "backbone.")


# --------------------------------------------------------------------------------------------
# kornia restatement (see oracle/stubs/kornia/... for provenance)
def project_points(p: Tensor, K: Tensor) -> Tensor:
    eps = 1e-8
    z = p[..., -1:]
    scale = torch.where(z.abs() > eps, 1.0 / (z + eps), torch.ones_like(z))
    xy = scale * p[..., :-1]
    u = xy[..., 0] * K[..., 0, 0] + K[..., 0, 2]
    v = xy[..., 1] * K[..., 1, 1] + K[..., 1, 2]
    return torch.stack([u, v], dim=-1)


def unproject_points(uv: Tensor, depth: Tensor, K: Tensor) -> Tensor:
    x = (uv[..., 0] - K[..., 0, 2]) / K[..., 0, 0]
    y = (uv[..., 1] - K[..., 1, 2]) / K[..., 1, 1]
    xyz = F.normalize(torch.stack([x, y, torch.ones_like(x)], dim=-1), dim=-1, p=2.0)
    return xyz * depth


# --------------------------------------------------------------------------------------------
# reparam.py
def diffusion_to_data(cfg: OracleConfig, sd: dict, diff: Tensor, K: Optional[Tensor]) -> Tensor:
    if cfg.reparam == "none":  # reparam.py:31-40
        return diff
    if cfg.reparam == "gaussian":  # reparam.py:62-64
        return diff * sd["reparam.sigma"].to(diff) + sd["reparam.mean"].to(diff)
    # UVLReparam.diffusion_to_data, reparam.py:191-201 (uvl_to_hwd :166-184, hwd_to_xyz :131-137)
    uvl = diff * sd["reparam.uvl_std"].to(diff) + sd["reparam.uvl_mean"].to(diff)
    u, v, l = uvl.unbind(-1)
    r01 = lambda r: (torch.tanh(r) * cfg.logit_scale + 1.0) / 2
    hw = torch.stack([r01(u), r01(v)], dim=-1)
    d = torch.exp(l).unsqueeze(-1)
    return unproject_points(hw, d, K.unsqueeze(1).to(diff))


def data_to_diffusion(cfg: OracleConfig, sd: dict, data: Tensor, K: Optional[Tensor]) -> Tensor:
    if cfg.reparam == "none":
        return data
    if cfg.reparam == "gaussian":  # reparam.py:58-60
        return (data - sd["reparam.mean"].to(data)) / sd["reparam.sigma"].to(data)
    # UVLReparam.data_to_diffusion, reparam.py:178-189 (xyz_to_hwd :122-129, hwd_to_uvl :139-159)
    hw = project_points(data, K.unsqueeze(1).to(data))
    d = torch.linalg.norm(data, dim=-1, keepdim=True)
    real = lambda s: torch.arctanh((2 * s - 1.0) / cfg.logit_scale)
    uvl = torch.stack([real(hw[..., 0]), real(hw[..., 1]), torch.log(d[..., 0])], dim=-1)
    return (uvl - sd["reparam.uvl_mean"].to(data)) / sd["reparam.uvl_std"].to(data)


# --------------------------------------------------------------------------------------------
# models/normalization.py:36-44 — GroupNorm over (points x channels-in-group), then t-conditioned affine
def adagn(sd: dict, pre: str, x: Tensor, t: Tensor, groups: int = 32) -> Tensor:
    normed = F.group_norm(x.transpose(1, 2), groups, eps=1e-5).transpose(1, 2)
    scale = F.linear(t, sd[pre + "scale.weight"], sd[pre + "scale.bias"])  # [B,1,C]
    bias = F.linear(t, sd[pre + "bias.weight"], sd[pre + "bias.bias"])
    return scale * normed + bias


# models/mlp.py:5-39 with models/activation.py:17-24 (depth 1)
def gaussian_act(x: Tensor, alpha: Tensor) -> Tensor:
    return ((-(x**2) / (2 * alpha**2)).exp() - 0.7) / 0.28


def mlp(sd: dict, pre: str, x: Tensor) -> Tensor:
    h = F.linear(x, sd[pre + "0.weight"], sd[pre + "0.bias"])
    h = gaussian_act(h, sd[pre + "1.alpha"])
    return F.linear(h, sd[pre + "2.weight"], sd[pre + "2.bias"])


# models/set_transformer.py:47-65
def attention_pool(sd: dict, pre: str, y: Tensor, heads: int) -> Tensor:
    B, N, C = y.shape
    d = C // heads
    kv = F.linear(y, sd[pre + "kv_proj.weight"])  # columns: (t h d)
    k = kv[..., :C].reshape(B, N, heads, d).transpose(1, 2)
    v = kv[..., C:].reshape(B, N, heads, d).transpose(1, 2)
    q = sd[pre + "inducers"].expand(B, -1, -1, -1)
    attn = F.scaled_dot_product_attention(q, k, v)  # [B,h,I,d]
    attn = attn.transpose(1, 2).reshape(B, -1, C)
    return F.linear(attn, sd[pre + "out_proj.weight"])


# nn.MultiheadAttention(batch_first=True)(query=y, key=h, value=h), models/set_transformer.py:90,112
def mha_unpool(sd: dict, pre: str, y: Tensor, h: Tensor, heads: int) -> Tensor:
    B, N, C = y.shape
    I = h.shape[1]
    d = C // heads
    wq, wk, wv = sd[pre + "in_proj_weight"].chunk(3)
    bq, bk, bv = sd[pre + "in_proj_bias"].chunk(3)
    q = F.linear(y, wq, bq).reshape(B, N, heads, d).transpose(1, 2)
    k = F.linear(h, wk, bk).reshape(B, I, heads, d).transpose(1, 2)
    v = F.linear(h, wv, bv).reshape(B, I, heads, d).transpose(1, 2)
    a = F.scaled_dot_product_attention(q, k, v)
    a = a.transpose(1, 2).reshape(B, N, C)
    return F.linear(a, sd[pre + "out_proj.weight"], sd[pre + "out_proj.bias"])


# models/set_transformer.py:92-117 (Broadcast) and :155-168 (BroadcastingLayer)
def broadcasting_layer(sd: dict, pre: str, x: Tensor, t: Tensor, heads: int, h: Optional[Tensor] = None):
    y = adagn(sd, pre + "broadcast_norm.", x, t)
    if h is None:
        h = attention_pool(sd, pre + "broadcast.pool.", y, heads)
        h = adagn(sd, pre + "broadcast.norm_1.", h, t)
        h = mlp(sd, pre + "broadcast.mlp.", h)
        h = adagn(sd, pre + "broadcast.norm_2.", h, t)
    x = x + mha_unpool(sd, pre + "broadcast.unpool.", y, h, heads)
    y = adagn(sd, pre + "mlp_norm.", x, t)
    x = x + mlp(sd, pre + "mlp.", y)
    return x, h


# models/set_transformer.py:198-216
def set_transformer(cfg: OracleConfig, sd: dict, x: Tensor, t: Tensor, hs: Optional[Sequence[Tensor]] = None):
    out_h = []
    for l in range(cfg.n_layers):
        x, h = broadcasting_layer(sd, f"{cfg.st_prefix}layers.{l}.", x, t, cfg.num_heads, None if hs is None else hs[l])
        out_h.append(h)
    return x, out_h


# models/ray.py:64-87
def extract_image_features(cfg: OracleConfig, sd: dict, geometry_diffusion: Tensor, features: Sequence[Tensor], K: Tensor) -> Tensor:
    geometry_data = diffusion_to_data(cfg, sd, geometry_diffusion, K)
    hw = project_points(geometry_data, K.unsqueeze(1))[..., :2]
    grid = hw.unsqueeze(2) * 2 - 1  # [B,N,1,2]
    looks = []
    for f in features:
        look = F.grid_sample(f, grid, align_corners=False)  # [B,C,N,1]
        looks.append(look[..., 0].transpose(1, 2))
    return torch.cat(looks, dim=-1)


def group_norm_bnc(x: Tensor, groups: int) -> Tensor:  # models/ray.py:20-30
    return F.group_norm(x.transpose(1, 2), groups, eps=1e-5).transpose(1, 2)


# models/ray.py:89-120 / models/linear_lift.py:33-46
def network(cfg: OracleConfig, sd: dict, geometry: Tensor, t: Tensor, features, K, hs=None):
    p = cfg.net_prefix
    if cfg.kind == "uncond":
        x = F.linear(geometry, sd[p + "lift.weight"], sd[p + "lift.bias"])
        x, out_h = set_transformer(cfg, sd, x, t, hs)
        if p + "lower.weight" in sd:  # LinearLift(do_norm=False): a bare Linear head (models/linear_lift.py:26-29)
            return F.linear(x, sd[p + "lower.weight"], sd[p + "lower.bias"]), out_h
        x = F.layer_norm(x, (x.shape[-1],), eps=1e-5)
        return F.linear(x, sd[p + "lower.1.weight"], sd[p + "lower.1.bias"]), out_h
    xyz = F.linear(geometry, sd[p + "xyz_embed.weight"], sd[p + "xyz_embed.bias"])
    # the network's own copy of the reparam buffers (models/ray.py:47) has the same values
    img_raw = extract_image_features(cfg, sd, geometry, features, K)
    img = F.linear(group_norm_bnc(img_raw, 16), sd[p + "img_feature_proj.1.weight"], sd[p + "img_feature_proj.1.bias"])
    x, out_h = set_transformer(cfg, sd, xyz + img, t, hs)
    out = F.linear(group_norm_bnc(x, 16), sd[p + "output_proj.1.weight"], sd[p + "output_proj.1.bias"])
    return out, out_h


# diffusion.py:37-62 (EDMPrecond.forward) behind Diffusion.forward (:233-247)
def denoise(cfg: OracleConfig, sd: dict, x: Tensor, sigma: Tensor, features=None, K=None, hs=None, return_h=False):
    sigma = sigma.reshape(-1, 1, 1)
    sd2 = cfg.sigma_data**2
    c_skip = sd2 / (sigma**2 + sd2)
    c_out = sigma * cfg.sigma_data / (sigma**2 + sd2).sqrt()
    c_in = 1 / (sd2 + sigma**2).sqrt()
    c_noise = sigma.log() / 4
    F_x, out_h = network(cfg, sd, c_in * x, c_noise, features, K, hs)
    D = c_skip * x + c_out * F_x
    return (D, out_h) if return_h else D


# diffusion.py:253-269
def t_steps(num_steps: int, sigma_max: float, sigma_min: float, rho: float) -> Tensor:
    i = torch.arange(num_steps, dtype=torch.float64)
    t = (sigma_max ** (1 / rho) + i / (num_steps - 1) * (sigma_min ** (1 / rho) - sigma_max ** (1 / rho))) ** rho
    return torch.cat([t, torch.zeros_like(t[:1])])


# diffusion.py:271-352
@torch.no_grad()
def sample_stochastic(cfg: OracleConfig, sd: dict, shape, features=None, K=None, rng: torch.Generator | None = None, **kw):
    k = {**cfg.sampler, "sigma_max": cfg.sigma_max, **kw}
    n, S_churn, S_min, S_max, S_noise = k["num_steps"], k["S_churn"], k["S_min"], k["S_max"], k["S_noise"]
    if rng is None:
        rng = torch.Generator("cpu").manual_seed(42)
    B = shape[0]
    latents = torch.randn(shape, generator=rng, dtype=torch.float32)
    ts = t_steps(n, k["sigma_max"], k["sigma_min"], k["rho"])
    x_next = latents.to(torch.float64) * ts[0]
    for i, (t_cur, t_next) in enumerate(zip(ts[:-1], ts[1:])):
        x_cur = x_next
        gamma = min(S_churn / n, math.sqrt(2.0) - 1) if S_min <= t_cur <= S_max else 0
        t_hat = t_cur + gamma * t_cur
        noise = torch.randn(x_cur.shape, generator=rng, dtype=torch.float32)
        x_hat = x_cur + (t_hat**2 - t_cur**2).sqrt() * S_noise * noise
        den = denoise(cfg, sd, x_hat.float(), t_hat.repeat(B).float(), features, K).to(torch.float64)
        d_cur = (x_hat - den) / t_hat
        x_next = x_hat + (t_next - t_hat) * d_cur
        if i < n - 1:
            den = denoise(cfg, sd, x_next.float(), t_next.repeat(B).float(), features, K).to(torch.float64)
            d_prime = (x_next - den) / t_next
            x_next = x_hat + (t_next - t_hat) * (0.5 * d_cur + 0.5 * d_prime)
    return diffusion_to_data(cfg, sd, x_next, K)


@torch.no_grad()
def sample_stochastic_device(cfg: OracleConfig, sd: dict, shape, features=None, K=None, device="cuda", seed: int = 42, **kw):
    """`sample_stochastic` with state, noise and sigma on `device` (bench.py's PyTorch-eager-on-GPU arm): the same loop,
    draws from a generator of that device."""
    k = {**cfg.sampler, "sigma_max": cfg.sigma_max, **kw}
    n, S_churn, S_min, S_max, S_noise = k["num_steps"], k["S_churn"], k["S_min"], k["S_max"], k["S_noise"]
    rng = torch.Generator(device).manual_seed(seed)
    B = shape[0]
    latents = torch.randn(shape, generator=rng, dtype=torch.float32, device=device)
    ts = t_steps(n, k["sigma_max"], k["sigma_min"], k["rho"]).tolist()
    x_next = latents.to(torch.float64) * ts[0]
    for i, (t_cur, t_next) in enumerate(zip(ts[:-1], ts[1:])):
        x_cur = x_next
        gamma = min(S_churn / n, math.sqrt(2.0) - 1) if S_min <= t_cur <= S_max else 0
        t_hat = t_cur + gamma * t_cur
        noise = torch.randn(x_cur.shape, generator=rng, dtype=torch.float32, device=device)
        x_hat = x_cur + math.sqrt(t_hat**2 - t_cur**2) * S_noise * noise
        sig = torch.full((B,), t_hat, device=device, dtype=torch.float32)
        den = denoise(cfg, sd, x_hat.float(), sig, features, K).to(torch.float64)
        d_cur = (x_hat - den) / t_hat
        x_next = x_hat + (t_next - t_hat) * d_cur
        if i < n - 1:
            sig = torch.full((B,), t_next, device=device, dtype=torch.float32)
            den = denoise(cfg, sd, x_next.float(), sig, features, K).to(torch.float64)
            d_prime = (x_next - den) / t_next
            x_next = x_hat + (t_next - t_hat) * (0.5 * d_cur + 0.5 * d_prime)
    return diffusion_to_data(cfg, sd, x_next, K)


# diffusion.py:354-470
@torch.no_grad()
def upsample(cfg: OracleConfig, sd: dict, data: Tensor, n_new: int | None = None, new_latents: Tensor | None = None,
             features=None, K=None, seed: int | None = 42, num_substeps: int = 5, **kw):
    k = {**cfg.sampler, "sigma_max": cfg.sigma_max, **kw}
    n, S_churn, S_min, S_max, S_noise = k["num_steps"], k["S_churn"], k["S_min"], k["S_max"], k["S_noise"]
    rng = torch.Generator("cpu")
    if seed is not None:
        rng.manual_seed(seed)
    randn = lambda shape: torch.randn(tuple(shape), generator=rng, dtype=torch.float32)
    if (new_latents is None) == (n_new is None):
        raise ValueError("Either new_latents or n_new must be specified, but not both.")
    if new_latents is None:
        new_latents = randn((data.shape[0], n_new, data.shape[2]))
    data = data_to_diffusion(cfg, sd, data, K)
    ts = t_steps(n, k["sigma_max"], k["sigma_min"], k["rho"])
    B = data.shape[0]
    x_next = new_latents.to(torch.float64) * ts[0]
    for i, (t_cur, t_next) in enumerate(zip(ts[:-1], ts[1:])):
        data_ctx = data + randn(data.shape) * t_cur
        _, cache = denoise(cfg, sd, data_ctx.float(), t_cur.float().expand(B), features, K, return_h=True)
        for u in range(num_substeps):
            x_cur = x_next
            gamma = min(S_churn / n, math.sqrt(2) - 1) if S_min <= t_cur <= S_max else 0
            t_hat = t_cur + gamma * t_cur
            x_hat = x_cur + (t_hat**2 - t_cur**2).sqrt() * S_noise * randn(x_cur.shape)
            den = denoise(cfg, sd, x_hat.float(), t_hat.float().expand(B), features, K, hs=cache).to(torch.float64)
            d_cur = (x_hat - den) / t_hat
            x_next = x_hat + (t_next - t_hat) * d_cur
            if i < n - 1:
                den = denoise(cfg, sd, x_next.float(), t_next.float().expand(B), features, K, hs=cache).to(torch.float64)
                d_prime = (x_next - den) / t_next
                x_next = x_hat + (t_next - t_hat) * (0.5 * d_cur + 0.5 * d_prime)
            if u < num_substeps - 1 and i < n - 1:
                x_next = x_next + (t_cur**2 - t_next**2).sqrt() * randn(x_next.shape)
    return diffusion_to_data(cfg, sd, x_next, K)


# gecco-jax models/stochastic.py:101-231 (`_sample_inpaint`), restated with the EDM schedule sigma(t) = t of gecco-torch and
# torch draws in the order: initial noise; per sub-step known-point noise, churn noise, re-noise.  gecco-jax cannot run in
# the build container (no jax / equinox / diffrax), so this restatement is NOT pinned by reference outputs.
@torch.no_grad()
def sample_inpaint(cfg: OracleConfig, sd: dict, known: Tensor, m_to_inpaint: int, features=None, K=None,
                   rng: torch.Generator | None = None, num_substeps: int = 1, **kw):
    k = {**cfg.sampler, "sigma_max": cfg.sigma_max, "S_churn": 0.0, **kw}
    n, S_churn, S_noise = k["num_steps"], k["S_churn"], k["S_noise"]
    if rng is None:
        rng = torch.Generator("cpu").manual_seed(42)
    randn = lambda shape: torch.randn(tuple(shape), generator=rng, dtype=torch.float32)
    known_diff = data_to_diffusion(cfg, sd, known, K).float()
    B, N = known_diff.shape[:2]
    M = m_to_inpaint
    ts = t_steps(n, k["sigma_max"], k["sigma_min"], k["rho"]).tolist()
    gamma = min(S_churn / n, math.sqrt(2.0) - 1)
    x = torch.cat([torch.zeros(B, M, 3), known_diff], dim=1).to(torch.float64)
    x = x + (randn(x.shape) * ts[0]).to(torch.float64)
    for i in range(n):
        s_cur, s_next = ts[i], ts[i + 1]
        s_hat = s_cur * (1 + gamma)
        for j in range(num_substeps):
            x[:, M:] = (known_diff + randn(known_diff.shape) * s_cur).to(torch.float64)
            x_hat = x + (math.sqrt(s_hat**2 - s_cur**2) * S_noise * randn(x.shape)).to(torch.float64)
            sig = torch.full((B,), s_hat, dtype=torch.float32)
            d_cur = (x_hat - denoise(cfg, sd, x_hat.float(), sig, features, K).to(torch.float64)) / s_hat
            x_next = x_hat + (s_next - s_hat) * d_cur
            if i < n - 1:
                sig = torch.full((B,), s_next, dtype=torch.float32)
                d_prime = (x_next - denoise(cfg, sd, x_next.float(), sig, features, K).to(torch.float64)) / s_next
                x_next = x_hat + (s_next - s_hat) * (0.5 * d_cur + 0.5 * d_prime)
            x = x_next
            if j < num_substeps - 1:
                x = x + (math.sqrt(max(s_cur**2 - s_next**2, 0.0)) * randn(x.shape)).to(torch.float64)
    return diffusion_to_data(cfg, sd, x, K)[:, :M]


# diffusion.py:87-143 — LogUniformSchedule (low-discrepancy) + EDMLoss on given draws u ~ U[0,1)^B, noise ~ N(0,1)
def edm_loss(cfg: OracleConfig, sd: dict, examples: Tensor, u: Tensor, noise: Tensor, features=None, K=None,
             sigma_min: float = 0.002, loss_scale: float = 100.0) -> Tensor:
    ex_diff = data_to_diffusion(cfg, sd, examples, K)
    n = examples.shape[0]
    div = 1 / n
    uu = div * u + div * torch.arange(n, device=u.device)  # :105-108
    lo, hi = math.log(sigma_min), math.log(cfg.sigma_max)
    sigma = (uu * (hi - lo) + lo).exp().reshape(-1, 1, 1)  # :110-113
    weight = (sigma**2 + cfg.sigma_data**2) / ((sigma * cfg.sigma_data) ** 2)  # :138
    D = denoise(cfg, sd, ex_diff + noise * sigma, sigma, features, K)
    return (loss_scale * weight * (D - ex_diff) ** 2).mean()  # :141-142


# gecco-jax models/diffusion.py:444-541 (`evaluate_logp`) with `trace_jac_estimator` (:175-193) and `_dx_dt` (:309-332),
# restated with the EDM schedule sigma(t) = t, scale = 1 of gecco-torch: Heun's method (diffrax `Heun` under `StepTo`, no
# FSAL: the derivative is re-evaluated at the start of every step) over the reversed noise levels from sigma_min to
# sigma_max on the pair (x, accumulated divergence); divergence = mean over the Rademacher probes `noise`
# [S, B, N, 3] of eps . grad_x(f(x) . eps).  The log-abs-det of data -> diffusion follows `ReparamDiagonalBlockJacrev`
# (models/reparam.py:27-48): per-point 3 x 3 Jacobians by reverse mode, slogdet, summed per cloud.  gecco-jax cannot run in
# the build container, so this restatement is NOT pinned by reference outputs; tests/test_oracle.py checks it against the
# closed-form likelihood of a linear denoiser instead.
def log_likelihood(cfg: OracleConfig, sd: dict, data: Tensor, noise: Tensor, features=None, K=None, denoise_fn=None, **kw):
    k = {**cfg.sampler, "sigma_max": cfg.sigma_max, **kw}
    ts = t_steps(k["num_steps"], k["sigma_max"], k["sigma_min"], k["rho"])[:-1].flip(0).tolist()
    if denoise_fn is None:
        denoise_fn = lambda x, sig: denoise(cfg, sd, x, sig, features, K)
    B = data.shape[0]
    d_in = data.detach().clone().float().requires_grad_(True)
    x0 = data_to_diffusion(cfg, sd, d_in, K)
    if cfg.reparam == "none":
        ladj = torch.zeros(B, dtype=torch.float64)
    else:
        rows = [torch.autograd.grad(x0[..., i].sum(), d_in, retain_graph=True)[0] for i in range(3)]
        ladj = torch.linalg.slogdet(torch.stack(rows, dim=-2).double())[1].sum(dim=1)

    def f_and_div(x: Tensor, t: float):
        xin = x.float().detach().requires_grad_(True)
        f = (xin - denoise_fn(xin, torch.full((B,), t, dtype=torch.float32))) / t
        div = torch.zeros(B, dtype=torch.float64)
        for s in range(noise.shape[0]):
            g = torch.autograd.grad((f * noise[s]).sum(), xin, retain_graph=True)[0]
            div += (g * noise[s]).double().flatten(1).sum(1)
        return f.detach().double(), div / noise.shape[0]

    x = x0.detach().double()
    delta = torch.zeros(B, dtype=torch.float64)
    for i in range(len(ts) - 1):
        dt = ts[i + 1] - ts[i]
        f0, d0 = f_and_div(x, ts[i])
        f1, d1 = f_and_div(x + dt * f0, ts[i + 1])
        x = x + 0.5 * dt * (f0 + f1)
        delta = delta + 0.5 * dt * (d0 + d1)
    smax = ts[-1]
    prior = (-0.5 * (x / smax) ** 2 - math.log(smax) - 0.5 * math.log(2 * math.pi)).flatten(1).sum(1)
    return dict(logp=prior + delta + ladj, prior_logp=prior, delta_jacobian=delta, delta_reparam=ladj, latent=x)

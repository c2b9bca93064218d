"""Op-level parity of the CUDA kernels against plain fp32 torch restatements of the reference ops."""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def _gen(seed):
    return torch.Generator(device="cpu").manual_seed(seed)


def test_group_stats_and_adagn(cuda):
    from gecco_b200 import ops

    B, N, Np, C = 3, 200, 256, 384
    g = _gen(1)
    x = torch.zeros(B, Np, C)
    x[:, :N] = torch.randn(B, N, C, generator=g) * 2 + 0.5
    t = torch.randn(B, 1, generator=g)
    sw, sb, bw, bb = (torch.randn(C, 1, generator=g), torch.randn(C, generator=g), torch.randn(C, 1, generator=g),
                      torch.randn(C, generator=g))
    xd = x.to(cuda).reshape(B * Np, C)
    stats = ops.group_stats(xd, Np, N, 12)
    o32, o16 = ops.adagn(xd, stats, 12, t.to(cuda), sw.to(cuda), sb.to(cuda), bw.to(cuda), bb.to(cuda),
                         rows_per_cloud=Np, valid_rows=N, groups=32, out_bf16=True, out_f32=True)
    torch.cuda.synchronize()
    xv = x[:, :N]
    normed = F.group_norm(xv.transpose(1, 2), 32, eps=1e-5).transpose(1, 2)
    scale = t @ sw.t() + sb
    bias = t @ bw.t() + bb
    ref = scale[:, None] * normed + bias[:, None]
    got = o32.view(B, Np, C)[:, :N].cpu()
    assert (got - ref).abs().max().item() < 2e-4
    assert o32.view(B, Np, C)[:, N:].abs().max().item() == 0.0
    assert (o16.view(B, Np, C)[:, :N].float().cpu() - ref).abs().max().item() < 0.1
    # GroupNorm(16) from the same 12-channel statistics (24-channel groups)
    o32b, _ = ops.adagn(xd, stats, 12, t.to(cuda), sw.to(cuda), sb.to(cuda), bw.to(cuda), bb.to(cuda),
                        rows_per_cloud=Np, valid_rows=N, groups=16, out_f32=True)
    normed16 = F.group_norm(xv.transpose(1, 2), 16, eps=1e-5).transpose(1, 2)
    ref16 = scale[:, None] * normed16 + bias[:, None]
    assert (o32b.view(B, Np, C)[:, :N].cpu() - ref16).abs().max().item() < 2e-4


def test_lift(cuda):
    from gecco_b200 import ops

    B, N, Np, C = 2, 100, 128, 384
    g = _gen(2)
    xin = torch.randn(B, N, 3, generator=g)
    w, b = torch.randn(C, 3, generator=g), torch.randn(C, generator=g)
    sigma = torch.tensor([0.3, 20.0])
    stats = torch.zeros(B, C // 12, 2, dtype=torch.float64, device=cuda)
    x = ops.lift(xin.to(cuda), w.to(cuda), b.to(cuda), rows_per_cloud=Np, sigma=sigma.to(cuda), stats=stats)
    torch.cuda.synchronize()
    c_in = 1 / (1 + sigma**2).sqrt()
    ref = F.linear(xin * c_in[:, None, None], w, b)
    got = x.view(B, Np, C)[:, :N].cpu()
    assert (got - ref).abs().max().item() < 1e-5
    v = ref.view(B, N, C // 12, 12).double()
    assert torch.allclose(stats[..., 0].cpu(), v.sum(dim=(1, 3)), rtol=1e-5, atol=1e-3)
    assert torch.allclose(stats[..., 1].cpu(), (v * v).sum(dim=(1, 3)), rtol=1e-5, atol=1e-3)


@pytest.mark.parametrize("norm", [0, 1, 2])
def test_head_modes(cuda, norm):
    """Head (no norm: LinearLift(do_norm=False); LayerNorm; GroupNorm) and its EDM modes, at sigma_data 1 and 0.5."""
    from gecco_b200 import ops

    B, N, Np, C = 2, 150, 256, 384
    g = _gen(3)
    x = torch.zeros(B, Np, C)
    x[:, :N] = torch.randn(B, N, C, generator=g) * 1.5 + 0.2
    w, b = torch.randn(3, C, generator=g) / math.sqrt(C), torch.randn(3, generator=g)
    xin = torch.randn(B, N, 3, generator=g)
    sigma = torch.tensor([0.7, 3.0])
    xd = x.to(cuda).reshape(B * Np, C)
    stats = ops.group_stats(xd, Np, N, 12)
    if norm == 0:
        nx = x[:, :N]
    elif norm == 1:
        nx = F.layer_norm(x[:, :N], (C,), eps=1e-5)
    else:
        nx = F.group_norm(x[:, :N].transpose(1, 2), 16, eps=1e-5).transpose(1, 2)
    Fref = F.linear(nx, w, b)
    kw = dict(clouds=B, rows_per_cloud=Np, valid_rows=N, norm=norm, groups=16, stats=stats)
    Fg = ops.head(xd, w.to(cuda), b.to(cuda), mode=0, **kw)
    assert (Fg.cpu() - Fref).abs().max().item() < 2e-4
    for sd in (1.0, 0.5):
        c_skip = lambda s: sd**2 / (s**2 + sd**2)
        c_out = lambda s: s * sd / (s**2 + sd**2) ** 0.5
        s = sigma[:, None, None]
        Dref = c_skip(s) * xin + c_out(s) * Fref
        Dg = ops.head(xd, w.to(cuda), b.to(cuda), mode=1, xin=xin.to(cuda), sigma=sigma.to(cuda), sigma_data=sd, **kw)
        assert (Dg.cpu() - Dref).abs().max().item() < 3e-4, sd
        # Euler then Heun with a shared sigma (sampler use)
        sig1 = torch.tensor([2.5], device=cuda)
        s1 = 2.5
        t_hat, t_next, churn = 2.5, 1.7, 0.3
        x_hat = torch.randn(B, N, 3, generator=g, dtype=torch.float64)
        xin_e = x_hat.float()
        noise = torch.randn(B, N, 3, generator=g)
        D1 = (c_skip(s1) * xin_e + c_out(s1) * Fref).double()
        d_cur = (x_hat - D1) / t_hat
        x_next = x_hat + (t_next - t_hat) * d_cur
        xh, xn, dc = x_hat.to(cuda).clone(), torch.empty_like(x_hat, device=cuda), torch.empty_like(x_hat, device=cuda)
        xin_next = torch.empty(B, N, 3, device=cuda)
        ops.head(xd, w.to(cuda), b.to(cuda), mode=2, xin=xin_e.to(cuda), sigma=sig1, sigma_stride=0, sigma_data=sd, x_hat=xh,
                 x_next=xn, d_cur=dc, xin_next=xin_next, t_hat=t_hat, t_next=t_next, **kw)
        assert (xn.cpu() - x_next).abs().max().item() < 1e-3, sd
        assert (xin_next.cpu() - x_next.float()).abs().max().item() < 1e-3, sd
        # Heun: evaluate "at x_next" with the same features (only the arithmetic is under test)
        s2 = 1.7
        sig2 = torch.tensor([s2], device=cuda)
        xin_h = xn.float()
        D2 = (c_skip(s2) * xin_h.cpu() + c_out(s2) * Fref).double()
        d_prime = (xn.cpu() - D2) / t_next
        x_new = x_hat + (t_next - t_hat) * (0.5 * dc.cpu() + 0.5 * d_prime) + churn * noise.double()
        ops.head(xd, w.to(cuda), b.to(cuda), mode=3, xin=xin_h, sigma=sig2, sigma_stride=0, sigma_data=sd, x_hat=xh, x_next=xn,
                 d_cur=dc, xin_next=xin_next, noise_next=noise.to(cuda), t_hat=t_hat, t_next=t_next, churn_next=churn, **kw)
        assert (xh.cpu() - x_new).abs().max().item() < 1e-3, sd


def _proj(p, K):
    z = p[..., -1:]
    sc = torch.where(z.abs() > 1e-8, 1.0 / (z + 1e-8), torch.ones_like(z))
    xy = sc * p[..., :-1]
    return torch.stack([xy[..., 0] * K[..., 0, 0] + K[..., 0, 2], xy[..., 1] * K[..., 1, 1] + K[..., 1, 2]], -1)


@pytest.mark.parametrize("kind", ["gaussian", "uvl"])
def test_lookup(cuda, kind):
    from gecco_b200 import ops

    B, N, Np = 2, 333, 384
    g = _gen(4)
    dims, sizes = (96, 192, 384), (34, 17, 8)
    feats = [torch.randn(B, c, s, s, generator=g) for c, s in zip(dims, sizes)]
    K = torch.tensor([[1.0859, 0, 0.4964], [0, 1.0859, 0.4964], [0, 0, 1]]).expand(B, 3, 3).contiguous()
    xin = torch.randn(B, N, 3, generator=g) * 3
    sigma = torch.tensor([0.5, 4.0])
    c_in = 1 / (1 + sigma**2).sqrt()
    geo = xin * c_in[:, None, None]
    if kind == "gaussian":
        mean, sig = [0.0, 0.0, 1.0], [0.15, 0.15, 0.15]
        data = geo * torch.tensor(sig) + torch.tensor(mean)
    else:
        mean, sig = [0.0, 0.0, 1.38], [0.56, 0.60, 0.49]
        uvl = geo * torch.tensor(sig) + torch.tensor(mean)
        r01 = lambda r: (torch.tanh(r) * 1.1 + 1.0) / 2
        hw = torch.stack([r01(uvl[..., 0]), r01(uvl[..., 1])], -1)
        d = torch.exp(uvl[..., 2:])
        Ku = K.unsqueeze(1)
        xy = torch.stack([(hw[..., 0] - Ku[..., 0, 2]) / Ku[..., 0, 0], (hw[..., 1] - Ku[..., 1, 2]) / Ku[..., 1, 1],
                          torch.ones_like(hw[..., 0])], -1)
        data = F.normalize(xy, dim=-1) * d
    uv = _proj(data, K.unsqueeze(1))
    grid = uv.unsqueeze(2) * 2 - 1
    # reference on the bf16-rounded maps (the kernel gathers from bf16 channels-last maps)
    ref = torch.cat([F.grid_sample(f.bfloat16().float(), grid, align_corners=False)[..., 0].transpose(1, 2) for f in feats], -1)
    levels = [ops.pack_features(f.to(cuda)) for f in feats]
    for f, l in zip(feats, levels):
        assert torch.equal(l.cpu(), f.permute(0, 2, 3, 1).bfloat16())
    stats = torch.zeros(B, 16, 2, dtype=torch.float64, device=cuda)
    o32, o16 = ops.lookup(xin.to(cuda), levels, K.to(cuda), reparam_kind=ops.REPARAM_KIND[kind], mean=mean, sigma_r=sig,
                          sigma=sigma.to(cuda), rows_per_cloud=Np, out_bf16=True, out_f32=True, stats=stats)
    torch.cuda.synchronize()
    got = o32.view(B, Np, -1)[:, :N].cpu()
    err = (got - ref).abs()
    # a point within float rounding of a pixel boundary may pick the neighbouring cell: compare robustly
    assert err.max().item() < 5e-2 and (err > 1e-3).float().mean().item() < 1e-3, (err.max(), (err > 1e-3).float().mean())
    assert (o16.view(B, Np, -1)[:, :N].float().cpu() - got).abs().max().item() < 0.05
    v = got.view(B, N, 16, 42).double()
    assert torch.allclose(stats[..., 0].cpu(), v.sum(dim=(1, 3)), rtol=1e-4, atol=1e-2)
    assert torch.allclose(stats[..., 1].cpu(), (v * v).sum(dim=(1, 3)), rtol=1e-4, atol=1e-2)
    # fold GroupNorm(16) + Linear and compare against the explicit path
    W = torch.randn(384, 672, generator=g) / math.sqrt(672)
    bia = torch.randn(384, generator=g)
    wb, bb = ops.fold_group_norm(W.to(cuda), bia.to(cuda), stats, float(N * 42), 16)
    refp = F.linear(F.group_norm(got.transpose(1, 2), 16, eps=1e-5).transpose(1, 2), W, bia)
    folded = torch.einsum("bnc,boc->bno", got, wb.view(B, 384, 672).float().cpu()) + bb.cpu()[:, None]
    assert (folded - refp).abs().max().item() < 5e-2


@pytest.mark.parametrize("sizes,N,slices", [((34, 17, 8), 333, None), ((34, 17, 8), 2048, "2"), ((34, 17, 8), 700, "4"),
                                            ((34, 17, 8), 257, "12"), ((64, 32, 16), 1000, "12"), ((9, 5, 3), 64, "1")])
def test_lookup_staged_matches_global_gather(cuda, monkeypatch, sizes, N, slices):
    """The shared-memory staged lookup (production path, bf16 output only) against the global-gather kernel: same
    taps, same fp32 blend order -> bit-identical rows; statistics agree to fp32 summation order."""
    from gecco_b200 import ops

    B, Np = 3, (N + 127) // 128 * 128
    g = _gen(11)
    dims = (96, 192, 384)
    levels = [ops.pack_features(torch.randn(B, c, s, s, generator=g).to(cuda)) for c, s in zip(dims, sizes)]
    K = torch.tensor([[1.0859, 0, 0.4964], [0, 1.0859, 0.4964], [0, 0, 1]]).expand(B, 3, 3).contiguous().to(cuda)
    xin = (torch.randn(B, N, 3, generator=g) * 2).to(cuda)
    xin[0, :5] = float("nan")  # non-finite coordinates gather zeros (grid_sample padding)
    sigma = torch.tensor([0.5, 4.0, 80.0]).to(cuda)
    kw = dict(reparam_kind=1, mean=[0.0, 0.0, 1.0], sigma_r=[0.15] * 3, sigma=sigma, rows_per_cloud=Np)

    def run():
        stats = torch.zeros(B, 16, 2, dtype=torch.float64, device=cuda)
        out = torch.full((B * Np, 672), 7.0, device=cuda, dtype=torch.bfloat16)
        ops.lookup(xin, levels, K, out_bf16=out, stats=stats, **kw)
        torch.cuda.synchronize()
        return out.view(B, Np, 672), stats

    monkeypatch.setenv("GECCO_LOOKUP_SLICES", "0")
    ref, ref_stats = run()
    if slices is None:
        monkeypatch.delenv("GECCO_LOOKUP_SLICES")
    else:
        monkeypatch.setenv("GECCO_LOOKUP_SLICES", slices)
    got, stats = run()
    assert torch.equal(got[:, :N].view(torch.int16), ref[:, :N].view(torch.int16))
    assert torch.equal(got[:, N:], ref[:, N:])  # padding rows untouched by both
    assert got[0, :5].abs().max().item() == 0.0
    assert torch.allclose(stats, ref_stats, rtol=1e-4, atol=1e-2)


@pytest.mark.parametrize("sizes,slices", [((34, 17, 8), None), ((34, 17, 8), "4"), ((64, 32, 16), None)])
def test_lookup_bench_shape_vs_grid_sample(cuda, monkeypatch, sizes, slices):
    """The production lookup at the BENCHMARKED shape (2048 points per cloud; 137^2 pyramid -> staged kernel with S = 2
    channel slices, 256^2 pyramid -> the kernel the engine picks there) directly against torch's F.grid_sample on the
    same bf16-rounded maps (ray.py:64-87), not against another kernel of this repo."""
    from gecco_b200 import ops

    B, N = 4, 2048
    g = _gen(21)
    dims = (96, 192, 384)
    feats = [torch.randn(B, c, s, s, generator=g) for c, s in zip(dims, sizes)]
    K = torch.tensor([[1.0859, 0, 0.4964], [0, 1.0859, 0.4964], [0, 0, 1]]).expand(B, 3, 3).contiguous()
    xin = torch.randn(B, N, 3, generator=g) * 2
    sigma = torch.tensor([0.002, 0.5, 4.0, 165.0])
    mean, sig = [0.0, 0.0, 1.0], [0.15, 0.15, 0.15]
    geo = xin / (1 + sigma**2).sqrt()[:, None, None]
    uv = _proj(geo * torch.tensor(sig) + torch.tensor(mean), K.unsqueeze(1))
    grid = (uv.unsqueeze(2) * 2 - 1).to(cuda)
    ref = torch.cat([F.grid_sample(f.bfloat16().float().to(cuda), grid, align_corners=False)[..., 0].transpose(1, 2) for f in feats], -1)
    levels = [ops.pack_features(f.to(cuda)) for f in feats]
    if slices is not None:
        monkeypatch.setenv("GECCO_LOOKUP_SLICES", slices)
    stats = torch.zeros(B, 16, 2, dtype=torch.float64, device=cuda)
    _, o16 = ops.lookup(xin.to(cuda), levels, K.to(cuda), reparam_kind=1, mean=mean, sigma_r=sig, sigma=sigma.to(cuda),
                        rows_per_cloud=N, out_bf16=True, stats=stats)
    torch.cuda.synchronize()
    got = o16.view(B, N, -1).float()
    err = (got - ref).abs()
    # bf16 output rounding (2^-9 relative) plus the rare point within float rounding of a pixel boundary
    tol = 1e-2 * ref.abs().clamp_min(1.0)
    assert (err > tol).float().mean().item() < 1e-3 and err.max().item() < 0.1, (err.max().item(), (err > tol).float().mean().item())
    v = ref.view(B, N, 16, 42).double()
    assert torch.allclose(stats[..., 0], v.sum(dim=(1, 3)), rtol=2e-3, atol=2.0)
    assert torch.allclose(stats[..., 1], (v * v).sum(dim=(1, 3)), rtol=2e-3, atol=2.0)


@pytest.mark.parametrize("kind,dtype", [("gaussian", torch.float32), ("uvl", torch.float32), ("uvl", torch.float64)])
def test_reparam_roundtrip(cuda, kind, dtype):
    from gecco_b200 import ops

    B, N = 2, 500
    g = _gen(5)
    diff = torch.randn(B, N, 3, generator=g, dtype=dtype)
    K = torch.tensor([[1.2, 0, 0.5], [0, 1.2, 0.5], [0, 0, 1]]).expand(B, 3, 3).contiguous()
    mean, sig = ([0.0, 0.01, 0.05], [0.11, 0.04, 0.17]) if kind == "gaussian" else ([0.0, 0.0, 1.38], [0.56, 0.60, 0.49])
    k = ops.REPARAM_KIND[kind]
    data = ops.reparam(diff.to(cuda), k, True, mean, sig, 1.1, K.to(cuda))
    back = ops.reparam(data, k, False, mean, sig, 1.1, K.to(cuda))
    tol = 1e-3 if dtype == torch.float32 else 1e-6
    assert (back.cpu() - diff).abs().max().item() < tol
    if kind == "gaussian":
        assert (data.cpu() - (diff * torch.tensor(sig, dtype=dtype) + torch.tensor(mean, dtype=dtype))).abs().max() < 1e-6


def _pool_case(cuda, B, N, splits, H, D, dtype=torch.float32):
    from gecco_b200 import ops

    I = 64
    C = H * D
    Np = (N + 127) // 128 * 128
    g = _gen(6)
    kv = torch.full((B, Np, 3 * C), 3.0)
    kv[:, :N] = torch.randn(B, N, 3 * C, generator=g)
    if splits < 0:
        # keys growing along the cloud: the running maximum of the scores jumps by hundreds between tiles (the
        # single-pass softmax of the tcgen05 kernel must fall back to moving its reference first)
        splits = 1
        kv[:, :N, :C] *= (1.0 + torch.arange(N) / 16.0)[None, :, None]
    ind = torch.randn(1, H, I, D, generator=g)
    kvd = kv.to(cuda).bfloat16().reshape(B * Np, 3 * C)
    qs = (ind[0] * (D**-0.5 * math.log2(math.e))).to(cuda).bfloat16().contiguous()
    out = ops.pool_attention(kvd, qs, clouds=B, rows_per_cloud=Np, valid_rows=N, heads=H, head_dim=D, k_off=0, v_off=C,
                             splits=splits)
    torch.cuda.synchronize()
    kvr = kvd.to(dtype).cpu().view(B, Np, 3 * C)[:, :N]
    k = kvr[..., :C].reshape(B, N, H, D).transpose(1, 2)
    v = kvr[..., C:2 * C].reshape(B, N, H, D).transpose(1, 2)
    # queries as the kernel sees them (bf16-rounded after the scale fold): with logits in the hundreds the rounding of
    # the queries alone moves the softmax
    qr = (qs.to(dtype).cpu() / (D**-0.5 * math.log2(math.e)))[None]
    ref = F.scaled_dot_product_attention(qr.expand(B, -1, -1, -1), k, v).transpose(1, 2).reshape(B, I, C)
    return (out.to(dtype).cpu().view(B, I, C) - ref).abs().max().item()


@pytest.mark.parametrize("tensor_cores,B,N,splits", [(False, 2, 2048, 1), (False, 2, 2048, 4), (False, 2, 300, 2),
                                                     (True, 2, 2048, 1), (True, 2, 2048, 4), (True, 2, 300, 2),
                                                     (True, 3, 1000, 3), (True, 80, 640, 1), (True, 1, 128, 1),
                                                     (True, 2, 1024, -1), (False, 2, 1024, -1)])
def test_pool_attention(cuda, monkeypatch, tensor_cores, B, N, splits):
    """mma.sync kernel and tcgen05 / TMEM kernel (key splits + combine, ragged last tile, several items per warpgroup)
    against torch SDPA.  Padding rows hold finite non-zero keys / values that must be masked out."""
    monkeypatch.setenv("GECCO_POOL_TC", "1" if tensor_cores else "0")
    err = _pool_case(cuda, B, N, splits, 8, 48)
    assert err < 2e-2, err


@pytest.mark.parametrize("B,N,splits", [(2, 2048, 1), (2, 2048, 4), (2, 300, 1), (2, 300, 4), (3, 1000, 3), (2, 1024, -1)])
@pytest.mark.parametrize("H,D", [(12, 32), (6, 64)])
def test_pool_attention_head_dims(cuda, B, N, splits, H, D):
    """The mma.sync pool kernels of head dim 32 and 64 (num_heads 12 / 6 at feature_dim 384), which the tcgen05 kernel
    refuses, against float64 SDPA on the same bf16 operands."""
    err = _pool_case(cuda, B, N, splits, H, D, dtype=torch.float64)
    assert err < 2e-2, err


def _unpool_case(cuda, B, Np, H, D, tensor_cores, dtype=torch.float32):
    from gecco_b200 import ops

    I = 64
    C = H * D
    g = _gen(7)
    q = torch.randn(B * Np, C, generator=g)
    khv = torch.randn(B * I, 2 * C, generator=g)
    qd = (q * (D**-0.5 * math.log2(math.e))).to(cuda).bfloat16()
    kd = khv.to(cuda).bfloat16()
    out = ops.unpool_attention(qd, kd, clouds=B, rows_per_cloud=Np, heads=H, head_dim=D, v_off=C, tensor_cores=tensor_cores)
    torch.cuda.synchronize()
    qr = (qd.to(dtype).cpu() / (D**-0.5 * math.log2(math.e)) ).view(B, Np, H, D).transpose(1, 2)
    kr = kd.to(dtype).cpu().view(B, I, 2 * C)
    k = kr[..., :C].reshape(B, I, H, D).transpose(1, 2)
    v = kr[..., C:].reshape(B, I, H, D).transpose(1, 2)
    ref = F.scaled_dot_product_attention(qr, k, v).transpose(1, 2).reshape(B * Np, C)
    return (out.to(dtype).cpu() - ref).abs().max().item()


@pytest.mark.parametrize("tensor_cores,B,Np", [(False, 2, 256), (True, 2, 256), (True, 5, 128), (True, 70, 384)])
def test_unpool_attention(cuda, tensor_cores, B, Np):
    """mma.sync kernel and tcgen05 / TMEM kernel (several tiles per CTA, CTAs spanning two clouds) against torch SDPA."""
    err = _unpool_case(cuda, B, Np, 8, 48, tensor_cores)
    assert err < 3e-2, err


@pytest.mark.parametrize("B,Np", [(2, 256), (5, 128), (3, 384)])
@pytest.mark.parametrize("H,D", [(12, 32), (6, 64)])
def test_unpool_attention_head_dims(cuda, B, Np, H, D):
    """The mma.sync unpool kernels of head dim 32 and 64 (offered the tcgen05 scratch, which they must not take) against
    float64 SDPA on the same bf16 operands."""
    err = _unpool_case(cuda, B, Np, H, D, True, dtype=torch.float64)
    assert err < 3e-2, err


def test_reparam_leading_dims(cuda):
    """The reference's reparams accept any leading dimensions ([..., 3]); the kernel sees them flattened."""
    from gecco_b200.reparam import GaussianReparam, UVLReparam
    import gecco_b200 as G

    g = _gen(31)
    gr = GaussianReparam(torch.tensor([0.0, 0.1, 1.0]), torch.tensor([0.2, 0.3, 0.4])).to(cuda)
    for shape in [(3,), (7, 3), (2, 5, 3), (2, 3, 4, 3)]:
        x = torch.randn(*shape, generator=g).to(cuda)
        d = gr.diffusion_to_data(x, None)
        assert d.shape == x.shape and torch.allclose(d, x * gr.sigma + gr.mean, atol=1e-6)
        assert torch.allclose(gr.data_to_diffusion(d, None), x, atol=1e-5)
    ur = UVLReparam(torch.tensor([0.0, 0.0, 1.38]), torch.tensor([0.56, 0.60, 0.49])).to(cuda)
    K = torch.tensor([[1.2, 0, 0.5], [0, 1.2, 0.5], [0, 0, 1]]).expand(2, 3, 3).contiguous().to(cuda)
    ctx = G.Context3d(image=torch.zeros(2, 3, 4, 4, device=cuda), K=K)
    x = torch.randn(2, 3, 4, 3, generator=g).to(cuda)
    d = ur.diffusion_to_data(x, ctx)
    assert d.shape == x.shape and torch.allclose(ur.diffusion_to_data(x.reshape(2, 12, 3), ctx).view(2, 3, 4, 3), d)
    assert torch.allclose(ur.data_to_diffusion(d, ctx), x, atol=1e-4)

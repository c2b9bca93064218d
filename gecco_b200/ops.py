"""Op-level Python entry points over the C ABI (one function per exported kernel family).

Torch is used for memory, streams and dtype plumbing only; every computation below runs in
the hand-written sm_100a kernels of libgecco_b200.so.
"""
from __future__ import annotations

import ctypes as C

import torch
from torch import Tensor

from . import _abi


def _stream(t: Tensor) -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


def _ptr(t: Tensor | None) -> C.c_void_p:
    return C.c_void_p(0 if t is None else t.data_ptr())


def _lib_for(t: Tensor):
    if not t.is_cuda:
        raise _abi.GeccoError("gecco_b200 ops need CUDA tensors (there is no CPU path)")
    return _abi.init(t.device.index if t.device.index is not None else torch.cuda.current_device())


def _round_up(x: int, m: int) -> int:
    return (x + m - 1) // m * m


def gemm(
    a: Tensor,
    w: Tensor,
    *,
    bias: Tensor | None = None,
    bias_stride: int = 0,
    act_alpha: float | None = None,
    res: Tensor | None = None,
    out_f32: Tensor | bool | None = None,
    out_bf16: Tensor | bool | None = None,
    stats: Tensor | None = None,
    rows_per_cloud: int | None = None,
    valid_rows: int | None = None,
    w_rows_per_cloud: int = 0,
    n_out: int | None = None,
    geom: Tensor | None = None,
    sigma: Tensor | None = None,
    sigma_stride: int = 0,
    wx: Tensor | None = None,
    sigma_data: float = 1.0,
    anorm: dict | None = None,
):
    """out = epilogue(a @ w.T) on the tcgen05 tensor cores; see gecco_gemm in include/gecco_b200.h.
    anorm = dict(stats f64 [clouds, K/stat_gs, 2], t fp32 [clouds], scale_w, scale_b, bias_w, bias_b, groups, stat_gs=12,
    eps=1e-5): `a` is the un-normalised bf16 tensor and AdaGN is applied to it inside the kernel."""
    assert a.dtype == torch.bfloat16
    lib = _lib_for(a)
    assert w.dtype == torch.bfloat16
    assert a.dim() == 2 and w.dim() == 2 and a.stride(1) == 1 and w.stride(1) == 1
    m, k = a.shape
    if n_out is None:
        n_out = w.shape[0]
    if rows_per_cloud is None:
        rows_per_cloud = _round_up(m, 32)
        valid_rows = m
    if valid_rows is None:
        valid_rows = rows_per_cloud
    if out_f32 is True:
        out_f32 = torch.empty((m, n_out), device=a.device, dtype=torch.float32)
    if out_bf16 is True:
        out_bf16 = torch.empty((m, n_out), device=a.device, dtype=torch.bfloat16)
    if out_f32 is False:
        out_f32 = None
    if out_bf16 is False:
        out_bf16 = None
    args = _abi.GemmArgs()
    args.a, args.lda = a.data_ptr(), a.stride(0)
    if anorm is not None:
        n = args.anorm
        n.stats, n.stat_gs, n.groups, n.eps = anorm["stats"].data_ptr(), anorm.get("stat_gs", STAT_GS), anorm["groups"], anorm.get("eps", 1e-5)
        n.t, n.t_stride = anorm["t"].data_ptr(), 1
        n.scale_w, n.scale_b = anorm["scale_w"].data_ptr(), anorm["scale_b"].data_ptr()
        n.bias_w, n.bias_b = anorm["bias_w"].data_ptr(), anorm["bias_b"].data_ptr()
    args.w, args.ldw = w.data_ptr(), w.stride(0)
    args.m, args.n_out, args.k = m, n_out, k
    args.rows_per_cloud, args.valid_rows, args.w_rows_per_cloud = rows_per_cloud, valid_rows, w_rows_per_cloud
    args.bias = 0 if bias is None else bias.data_ptr()
    args.bias_stride = bias_stride
    args.act = 0 if act_alpha is None else 1
    args.act_alpha = 1.0 if act_alpha is None else float(act_alpha)
    if res is not None:
        assert res.dtype == torch.float32 and res.stride(1) == 1
        args.res, args.ldr = res.data_ptr(), res.stride(0)
    if out_f32 is not None:
        assert out_f32.dtype == torch.float32 and out_f32.stride(1) == 1
        args.out_f32, args.ldo32 = out_f32.data_ptr(), out_f32.stride(0)
    if out_bf16 is not None:
        assert out_bf16.dtype == torch.bfloat16 and out_bf16.stride(1) == 1
        args.out_bf16, args.ldo16 = out_bf16.data_ptr(), out_bf16.stride(0)
    if stats is not None:
        assert stats.dtype == torch.float64 and stats.is_contiguous()
        args.stats = stats.data_ptr()
    if geom is not None:
        assert geom.dtype == torch.float32 and geom.is_contiguous()
        assert sigma is not None and wx is not None and sigma.dtype == torch.float32 and wx.dtype == torch.float32
        args.geom, args.sigma, args.sigma_stride, args.wx = geom.data_ptr(), sigma.data_ptr(), sigma_stride, wx.data_ptr()
        args.sigma_data = sigma_data
    _abi.check(lib.gecco_gemm(C.byref(args), _stream(a)))
    return out_f32, out_bf16


def gemm_anorm_supported(m: int, rows_per_cloud: int, n_out: int, k: int) -> bool:
    return bool(_abi.load().gecco_gemm_anorm_supported(m, rows_per_cloud, n_out, k))


def set_option(name: str, value: int) -> None:
    """gecco_set_option: "gemm_pairs", "graphs", "anorm", "chain", "mlp_pair", "fast_epilogue", "epi_skip" (see
    include/gecco_b200.h)."""
    _abi.check(_abi.load().gecco_set_option(name.encode(), C.c_int(int(value))))


def mlp(a: Tensor, w1: Tensor, b1: Tensor, act_alpha: float, w2: Tensor, b2: Tensor, res: Tensor, *,
        out_f32: Tensor | None = None, out_bf16: Tensor | bool | None = None, stats: Tensor | None = None,
        rows_per_cloud: int | None = None, valid_rows: int | None = None, w1_rows_per_cloud: int = 0,
        b1_stride: int = 0, anorm: dict | None = None):
    """out = res + w2 @ g(w1_cloud @ a + b1_cloud) + b2 with the hidden activation kept on chip; see gecco_mlp in
    include/gecco_b200.h (models/set_transformer.py:165-166)."""
    lib = _lib_for(a)
    assert a.dtype == torch.bfloat16 and w1.dtype == torch.bfloat16 and w2.dtype == torch.bfloat16
    assert a.dim() == 2 and a.stride(1) == 1 and w1.stride(1) == 1 and w2.stride(1) == 1
    assert b1.dtype == torch.float32 and b2.dtype == torch.float32 and res.dtype == torch.float32 and res.stride(1) == 1
    m, c = a.shape
    hidden = w2.shape[1]
    if rows_per_cloud is None:
        rows_per_cloud, valid_rows = m, m
    if valid_rows is None:
        valid_rows = rows_per_cloud
    if out_f32 is None:
        out_f32 = torch.empty((m, c), device=a.device, dtype=torch.float32)
    if out_bf16 is True:
        out_bf16 = torch.empty((m, c), device=a.device, dtype=torch.bfloat16)
    if out_bf16 is False:
        out_bf16 = None
    args = _abi.MlpArgs()
    args.a, args.lda = a.data_ptr(), a.stride(0)
    args.w1, args.ldw1, args.w1_rows_per_cloud = w1.data_ptr(), w1.stride(0), w1_rows_per_cloud
    args.b1, args.b1_stride = b1.data_ptr(), b1_stride
    args.act_alpha = float(act_alpha)
    args.w2, args.ldw2 = w2.data_ptr(), w2.stride(0)
    args.b2 = b2.data_ptr()
    args.m, args.c, args.hidden = m, c, hidden
    args.rows_per_cloud, args.valid_rows = rows_per_cloud, valid_rows
    args.res, args.ldr = res.data_ptr(), res.stride(0)
    assert out_f32.dtype == torch.float32 and out_f32.stride(1) == 1
    args.out_f32, args.ldo32 = out_f32.data_ptr(), out_f32.stride(0)
    if out_bf16 is not None:
        assert out_bf16.dtype == torch.bfloat16 and out_bf16.stride(1) == 1
        args.out_bf16, args.ldo16 = out_bf16.data_ptr(), out_bf16.stride(0)
    if stats is not None:
        assert stats.dtype == torch.float64 and stats.is_contiguous()
        args.stats = stats.data_ptr()
    scratch = None
    if anorm is not None:  # AdaGN on the A operand: the CTA-pair kernel with the hidden tile parked in an L2-resident scratch
        n = args.anorm
        n.stats, n.stat_gs, n.groups, n.eps = anorm["stats"].data_ptr(), anorm.get("stat_gs", STAT_GS), anorm["groups"], anorm.get("eps", 1e-5)
        n.t, n.t_stride = anorm["t"].data_ptr(), 1
        n.scale_w, n.scale_b = anorm["scale_w"].data_ptr(), anorm["scale_b"].data_ptr()
        n.bias_w, n.bias_b = anorm["bias_w"].data_ptr(), anorm["bias_b"].data_ptr()
        sms = torch.cuda.get_device_properties(a.device).multi_processor_count
        scratch = torch.empty((min(m, 128 * sms), hidden), device=a.device, dtype=torch.bfloat16)
        args.scratch = scratch.data_ptr()
    _abi.check(lib.gecco_mlp(C.byref(args), _stream(a)))
    return out_f32, out_bf16


def gaussian_activation(x: Tensor, alpha: float, normalized: bool = True) -> Tensor:
    """GaussianActivation.forward as a stand-alone kernel (gecco_gaussian_activation)."""
    lib = _lib_for(x)
    xf = x.detach().to(torch.float32).contiguous()
    out = torch.empty_like(xf)
    _abi.check(lib.gecco_gaussian_activation(_ptr(xf), _ptr(out), C.c_int64(xf.numel()), C.c_float(float(alpha)),
                                             C.c_int32(1 if normalized else 0), _stream(xf)))
    return out.to(x.dtype)


STAT_GS = 12  # channel granularity of the AdaGN statistics kept by the GEMM epilogue (C / 32 for C = 384)


def group_stats(x: Tensor, rows_per_cloud: int, valid_rows: int, group_size: int, stats: Tensor | None = None) -> Tensor:
    """stats[cloud, group, {sum, sumsq}] (float64) over the valid rows of each cloud; x is [clouds*rows_per_cloud, C]."""
    lib = _lib_for(x)
    assert x.dtype == torch.float32 and x.dim() == 2 and x.stride(1) == 1
    clouds = x.shape[0] // rows_per_cloud
    c = x.shape[1]
    if stats is None:
        stats = torch.zeros((clouds, c // group_size, 2), device=x.device, dtype=torch.float64)
    _abi.check(lib.gecco_group_stats(_ptr(x), C.c_int64(x.stride(0)), clouds, rows_per_cloud, valid_rows, c, group_size,
                                     _ptr(stats), _stream(x)))
    return stats


def adagn(x: Tensor, stats: Tensor, stat_gs: int, t: Tensor, scale_w: Tensor, scale_b: Tensor, bias_w: Tensor,
          bias_b: Tensor, *, rows_per_cloud: int, valid_rows: int, groups: int = 32, eps: float = 1e-5,
          out_bf16: Tensor | bool | None = None, out_f32: Tensor | bool | None = None, t_stride: int | None = None):
    lib = _lib_for(x)
    assert x.dtype == torch.float32 and x.dim() == 2 and x.stride(1) == 1
    rows, c = x.shape
    clouds = rows // rows_per_cloud
    ctx_dim = scale_w.shape[1] if scale_w.dim() == 2 else 1
    if out_bf16 is True:
        out_bf16 = torch.empty((rows, c), device=x.device, dtype=torch.bfloat16)
    if out_f32 is True:
        out_f32 = torch.empty((rows, c), device=x.device, dtype=torch.float32)
    if out_bf16 is False:
        out_bf16 = None
    if out_f32 is False:
        out_f32 = None
    a = _abi.AdaGNArgs()
    a.x, a.ldx = x.data_ptr(), x.stride(0)
    a.stats, a.stat_gs = stats.data_ptr(), stat_gs
    a.t, a.t_stride, a.ctx_dim = t.data_ptr(), (ctx_dim if t_stride is None else t_stride), ctx_dim
    a.scale_w, a.scale_b, a.bias_w, a.bias_b = scale_w.data_ptr(), scale_b.data_ptr(), bias_w.data_ptr(), bias_b.data_ptr()
    a.clouds, a.rows_per_cloud, a.valid_rows, a.c, a.groups = clouds, rows_per_cloud, valid_rows, c, groups
    a.eps = eps
    if out_bf16 is not None:
        a.out_bf16, a.ldo16 = out_bf16.data_ptr(), out_bf16.stride(0)
    if out_f32 is not None:
        a.out_f32, a.ldo32 = out_f32.data_ptr(), out_f32.stride(0)
    _abi.check(lib.gecco_adagn(C.byref(a), _stream(x)))
    return out_f32, out_bf16


def fold_adagn(w: Tensor, bias: Tensor | None, stats: Tensor, t: Tensor, scale_w: Tensor, scale_b: Tensor, bias_w: Tensor,
               bias_b: Tensor, *, clouds: int, valid_rows: int, groups: int = 32, stat_gs: int = STAT_GS, eps: float = 1e-5):
    """AdaGN + Linear folded per cloud: returns (w_folded bf16 [clouds, n_out, C], bias_folded fp32 [clouds, n_out])."""
    lib = _lib_for(w)
    assert w.dtype == torch.float32 and w.stride(1) == 1 and stats.dtype == torch.float64
    n_out, c = w.shape
    wf = torch.empty((clouds, n_out, c), device=w.device, dtype=torch.bfloat16)
    bf = torch.empty((clouds, n_out), device=w.device, dtype=torch.float32)
    a = _abi.FoldAdaGNArgs()
    a.w, a.ldw = w.data_ptr(), w.stride(0)
    a.bias = 0 if bias is None else bias.data_ptr()
    a.n_out, a.c = n_out, c
    a.stats, a.stat_gs, a.groups, a.valid_rows, a.eps = stats.data_ptr(), stat_gs, groups, valid_rows, eps
    a.t, a.t_stride, a.ctx_dim = t.data_ptr(), 1, 1
    a.scale_w, a.scale_b, a.bias_w, a.bias_b = scale_w.data_ptr(), scale_b.data_ptr(), bias_w.data_ptr(), bias_b.data_ptr()
    a.clouds = clouds
    a.w_folded_bf16, a.ldwf, a.wf_cloud_stride = wf.data_ptr(), c, n_out * c
    a.bias_folded, a.bias_stride = bf.data_ptr(), n_out
    _abi.check(lib.gecco_fold_adagn(C.byref(a), _stream(w)))
    return wf, bf


def lift(xin: Tensor, w: Tensor, b: Tensor, *, rows_per_cloud: int, sigma: Tensor | None = None, sigma_stride: int = 1,
         sigma_data: float = 1.0, stats: Tensor | None = None, stat_gs: int = STAT_GS, out: Tensor | None = None,
         out_bf16: Tensor | None = None) -> Tensor:
    lib = _lib_for(xin)
    assert xin.dtype == torch.float32 and xin.is_contiguous() and xin.shape[-1] == 3
    clouds, n = xin.shape[0], xin.shape[1]
    c = w.shape[0]
    if out is None:
        out = torch.empty((clouds * rows_per_cloud, c), device=xin.device, dtype=torch.float32)
    a = _abi.LiftArgs()
    a.xin = xin.data_ptr()
    a.sigma, a.sigma_stride, a.sigma_data = (0 if sigma is None else sigma.data_ptr()), sigma_stride, sigma_data
    a.w, a.b = w.data_ptr(), b.data_ptr()
    a.clouds, a.rows_per_cloud, a.valid_rows, a.c = clouds, rows_per_cloud, n, c
    a.x, a.ldx = out.data_ptr(), out.stride(0)
    if out_bf16 is not None:
        a.x_bf16, a.ldxb = out_bf16.data_ptr(), out_bf16.stride(0)
    a.stats, a.stat_gs = (0 if stats is None else stats.data_ptr()), stat_gs
    _abi.check(lib.gecco_lift(C.byref(a), _stream(xin)))
    return out


def head(x: Tensor, w_out: Tensor, b_out: Tensor, *, clouds: int, rows_per_cloud: int, valid_rows: int, norm: int,
         groups: int = 16, stats: Tensor | None = None, stat_gs: int = STAT_GS, eps: float = 1e-5,
         xin: Tensor | None = None, sigma: Tensor | None = None, sigma_stride: int = 1, sigma_data: float = 1.0,
         mode: int = 0, out: Tensor | None = None, x_hat: Tensor | None = None, x_next: Tensor | None = None,
         d_cur: Tensor | None = None, xin_next: Tensor | None = None, noise_next: Tensor | None = None,
         t_hat: float = 0.0, t_next: float = 0.0, churn_next: float = 0.0):
    lib = _lib_for(x)
    assert x.dtype == torch.float32 and x.stride(1) == 1
    if mode in (0, 1) and out is None:
        out = torch.empty((clouds, valid_rows, 3), device=x.device, dtype=torch.float32)
    a = _abi.HeadArgs()
    a.x, a.ldx = x.data_ptr(), x.stride(0)
    a.clouds, a.rows_per_cloud, a.valid_rows, a.c = clouds, rows_per_cloud, valid_rows, x.shape[1]
    a.norm, a.groups, a.stats, a.stat_gs, a.eps = norm, groups, (0 if stats is None else stats.data_ptr()), stat_gs, eps
    a.w_out, a.b_out = w_out.data_ptr(), b_out.data_ptr()
    a.xin = 0 if xin is None else xin.data_ptr()
    a.sigma, a.sigma_stride, a.sigma_data = (0 if sigma is None else sigma.data_ptr()), sigma_stride, sigma_data
    a.mode = mode
    a.out_f32 = 0 if out is None else out.data_ptr()
    a.x_hat = 0 if x_hat is None else x_hat.data_ptr()
    a.x_next = 0 if x_next is None else x_next.data_ptr()
    a.d_cur = 0 if d_cur is None else d_cur.data_ptr()
    a.xin_next = 0 if xin_next is None else xin_next.data_ptr()
    a.noise_next = 0 if noise_next is None else noise_next.data_ptr()
    a.t_hat, a.t_next, a.churn_next = t_hat, t_next, churn_next
    _abi.check(lib.gecco_head(C.byref(a), _stream(x)))
    return out


REPARAM_KIND = {"none": 0, "gaussian": 1, "uvl": 2}


def reparam(x: Tensor, kind: int, to_data: bool, mean=None, sigma=None, logit_scale: float = 1.1, K: Tensor | None = None) -> Tensor:
    """reparam.py data_to_diffusion / diffusion_to_data on [..., 3] float32 or float64 (the reference accepts any leading
    dimensions: GaussianReparam broadcasts, UVLReparam needs [B, ..., 3] with one camera per leading index)."""
    lib = _lib_for(x)
    assert x.dtype in (torch.float32, torch.float64) and x.shape[-1] == 3
    shape = x.shape
    if x.dim() == 1:
        x = x.view(1, 1, 3)
    elif x.dim() == 2:
        x = x.unsqueeze(0) if K is None else x.unsqueeze(1)
    elif x.dim() > 3:
        x = x.reshape(shape[0], -1, 3)
    x = x.contiguous()
    out = torch.empty_like(x)
    mean_a = (C.c_float * 3)(*(mean if mean is not None else (0.0, 0.0, 0.0)))
    sig_a = (C.c_float * 3)(*(sigma if sigma is not None else (1.0, 1.0, 1.0)))
    if K is not None:
        K = K.to(torch.float32).contiguous()
    clouds, pts = x.shape[0], x.shape[1]
    _abi.check(lib.gecco_reparam(_ptr(x), _ptr(out), int(x.dtype == torch.float64), kind, int(to_data), mean_a, sig_a,
                                 C.c_float(logit_scale), _ptr(K), clouds, pts, _stream(x)))
    return out.view(shape)


def pack_features(f: Tensor, out: Tensor | None = None) -> Tensor:
    """fp32 NCHW feature map -> bf16 NHWC (the layout gecco_lookup gathers from); `out` reuses an existing buffer."""
    lib = _lib_for(f)
    f = f.to(torch.float32).contiguous()
    b, c, h, w = f.shape
    if out is None or tuple(out.shape) != (b, h, w, c) or out.device != f.device or out.dtype != torch.bfloat16:
        out = torch.empty((b, h, w, c), device=f.device, dtype=torch.bfloat16)
    _abi.check(lib.gecco_pack_features(_ptr(f), _ptr(out), b, c, h, w, _stream(f)))
    return out


def lookup(xin: Tensor, levels: list[Tensor], K: Tensor, *, reparam_kind: int, mean=None, sigma_r=None,
           logit_scale: float = 1.1, sigma: Tensor | None = None, sigma_stride: int = 1, sigma_data: float = 1.0,
           rows_per_cloud: int | None = None, out_bf16: Tensor | bool | None = None, out_f32: Tensor | bool | None = None,
           stats: Tensor | None = None, stat_groups: int = 16):
    """levels: bf16 NHWC maps [B, H, W, C]; returns ([B*rows_per_cloud, sum C] fp32, bf16)."""
    lib = _lib_for(xin)
    assert xin.dtype == torch.float32 and xin.is_contiguous()
    clouds, pts = xin.shape[0], xin.shape[1]
    if rows_per_cloud is None:
        rows_per_cloud = pts
    ctot = sum(l.shape[-1] for l in levels)
    if out_bf16 is True:
        out_bf16 = torch.zeros((clouds * rows_per_cloud, ctot), device=xin.device, dtype=torch.bfloat16)
    if out_f32 is True:
        out_f32 = torch.zeros((clouds * rows_per_cloud, ctot), device=xin.device, dtype=torch.float32)
    if out_bf16 is False:
        out_bf16 = None
    if out_f32 is False:
        out_f32 = None
    a = _abi.LookupArgs()
    a.xin = xin.data_ptr()
    a.sigma, a.sigma_stride, a.sigma_data = (0 if sigma is None else sigma.data_ptr()), sigma_stride, sigma_data
    a.reparam = reparam_kind
    for j in range(3):
        a.mean[j] = 0.0 if mean is None else float(mean[j])
        a.sigma_r[j] = 1.0 if sigma_r is None else float(sigma_r[j])
    a.logit_scale = logit_scale
    K = K.to(torch.float32).contiguous()
    a.K = K.data_ptr()
    a.n_levels = len(levels)
    for i, l in enumerate(levels):
        assert l.dtype == torch.bfloat16 and l.is_contiguous() and l.shape[0] == clouds
        a.level_ptr[i] = l.data_ptr()
        a.level_h[i], a.level_w[i], a.level_c[i] = l.shape[1], l.shape[2], l.shape[3]
    a.clouds, a.points, a.rows_per_cloud = clouds, pts, rows_per_cloud
    if out_bf16 is not None:
        a.out_bf16, a.ldo16 = out_bf16.data_ptr(), out_bf16.stride(0)
    if out_f32 is not None:
        a.out_f32, a.ldo32 = out_f32.data_ptr(), out_f32.stride(0)
    if stats is not None:
        a.stats, a.stat_groups = stats.data_ptr(), stat_groups
    _abi.check(lib.gecco_lookup(C.byref(a), _stream(xin)))
    return out_f32, out_bf16


def fold_group_norm(w: Tensor, bias: Tensor, stats: Tensor, count: float, groups: int, eps: float = 1e-5):
    """GroupNorm(groups, affine=False) -> Linear folded into per-cloud bf16 weights and fp32 biases."""
    lib = _lib_for(w)
    c_out, c_in = w.shape
    clouds = stats.shape[0]
    wb = torch.empty((clouds * c_out, c_in), device=w.device, dtype=torch.bfloat16)
    bb = torch.empty((clouds, c_out), device=w.device, dtype=torch.float32)
    _abi.check(lib.gecco_fold_group_norm(_ptr(w), _ptr(bias), _ptr(stats), C.c_double(count), C.c_float(eps), groups,
                                         c_in, c_out, clouds, _ptr(wb), C.c_int64(c_in), _ptr(bb), _stream(w)))
    return wb, bb


def pool_attention(kv: Tensor, q_inducers: Tensor, *, clouds: int, rows_per_cloud: int, valid_rows: int, heads: int,
                   head_dim: int, k_off: int, v_off: int, splits: int = 1, out: Tensor | None = None) -> Tensor:
    lib = _lib_for(kv)
    assert kv.dtype == torch.bfloat16 and q_inducers.dtype == torch.bfloat16 and q_inducers.is_contiguous()
    inducers = q_inducers.shape[1]
    partial = torch.empty((clouds * heads * splits * inducers * (head_dim + 2),), device=kv.device, dtype=torch.float32)
    if out is None:
        out = torch.empty((clouds * inducers, heads * head_dim), device=kv.device, dtype=torch.bfloat16)
    a = _abi.PoolArgs()
    a.kv, a.ld, a.k_off, a.v_off = kv.data_ptr(), kv.stride(0), k_off, v_off
    a.clouds, a.rows_per_cloud, a.valid_rows = clouds, rows_per_cloud, valid_rows
    a.heads, a.head_dim, a.inducers = heads, head_dim, inducers
    a.q_inducers = q_inducers.data_ptr()
    a.splits, a.partial = splits, partial.data_ptr()
    a.out_bf16, a.ldo = out.data_ptr(), out.stride(0)
    _abi.check(lib.gecco_pool_attention(C.byref(a), _stream(kv)))
    return out


def pool_attention_partial(kv: Tensor, q_inducers: Tensor, *, clouds: int, rows_per_cloud: int, valid_rows: int, heads: int,
                           head_dim: int, k_off: int, v_off: int, splits: int = 1):
    """Pool attention core without the merge of the key splits (gecco_pool_attention_partial).  Returns (partial fp32
    scratch, splits_used) when splits_used > 1, else (pooled bf16, 1)."""
    lib = _lib_for(kv)
    inducers = q_inducers.shape[1]
    partial = torch.empty((clouds * heads * splits * inducers * (head_dim + 2),), device=kv.device, dtype=torch.float32)
    out = torch.empty((clouds * inducers, heads * head_dim), device=kv.device, dtype=torch.bfloat16)
    a = _abi.PoolArgs()
    a.kv, a.ld, a.k_off, a.v_off = kv.data_ptr(), kv.stride(0), k_off, v_off
    a.clouds, a.rows_per_cloud, a.valid_rows = clouds, rows_per_cloud, valid_rows
    a.heads, a.head_dim, a.inducers = heads, head_dim, inducers
    a.q_inducers = q_inducers.data_ptr()
    a.splits, a.partial = splits, partial.data_ptr()
    a.out_bf16, a.ldo = out.data_ptr(), out.stride(0)
    used = C.c_int32(1)
    _abi.check(lib.gecco_pool_attention_partial(C.byref(a), C.byref(used), _stream(kv)))
    return (partial, used.value) if used.value > 1 else (out, 1)


def inducer_chain(pooled: Tensor, w_pool_out: Tensor, norm1: list[Tensor], w_mlp0: Tensor, b_mlp0: Tensor, act_alpha: float,
                  w_mlp2: Tensor, b_mlp2: Tensor, norm2: list[Tensor], w_kv: Tensor, b_kv: Tensor, t: Tensor, *,
                  partial: Tensor | None = None, splits: int = 1, eps: float = 1e-5, want_cache: bool = True, first_stage: int = 0):
    """Inducer side of one Broadcast layer in one launch (gecco_inducer_chain).  pooled: bf16 [clouds*64, C] (input when
    splits <= 1, scratch otherwise); weights bf16 [n_out, k]; norm1 / norm2: [scale.weight, scale.bias, bias.weight,
    bias.bias] fp32 [C]; t: fp32 [clouds].  Returns (h3 bf16 [clouds*64, C], khv bf16 [clouds*64, 2C], vt bf16 [clouds, C, 64],
    cache fp32 [clouds*64, C] or None).  first_stage = 3: `pooled` is taken as h3 (bf16 cached inducer states)."""
    lib = _lib_for(pooled)
    m, c = pooled.shape
    clouds = m // 64
    hid = w_mlp0.shape[0]
    dev = pooled.device
    bf = torch.bfloat16
    for w in (pooled, w_pool_out, w_mlp0, w_mlp2, w_kv):
        assert w.dtype == bf and w.is_contiguous()
    hn = torch.empty((m, c), device=dev, dtype=bf)
    hh = torch.empty((m, hid), device=dev, dtype=bf)
    h3 = pooled if first_stage == 3 else torch.empty((m, c), device=dev, dtype=bf)
    khv = torch.empty((m, 2 * c), device=dev, dtype=bf)
    vt = torch.empty((clouds, c, 64), device=dev, dtype=bf)
    cache = torch.empty((m, c), device=dev, dtype=torch.float32) if (want_cache and first_stage == 0) else None
    a = _abi.ChainArgs()
    a.clouds, a.inducers, a.c, a.hidden, a.heads, a.groups = clouds, 64, c, hid, 8, 32
    a.first_stage = first_stage
    a.partial, a.splits = _ptr(partial), splits
    a.pooled = pooled.data_ptr()
    a.w_pool_out, a.w_mlp0, a.w_mlp2, a.w_kv = w_pool_out.data_ptr(), w_mlp0.data_ptr(), w_mlp2.data_ptr(), w_kv.data_ptr()
    a.b_mlp0, a.b_mlp2, a.b_kv = b_mlp0.data_ptr(), b_mlp2.data_ptr(), b_kv.data_ptr()
    a.act_alpha = act_alpha
    for n, ws in enumerate((norm1, norm2)):
        for i in range(4):
            assert ws[i].dtype == torch.float32 and ws[i].is_contiguous()
            a.norm[n][i] = ws[i].data_ptr()
    a.t, a.t_stride, a.eps = t.data_ptr(), t.stride(0) if t.dim() > 0 else 0, eps
    a.hn, a.hh, a.h3, a.khv, a.vt = hn.data_ptr(), hh.data_ptr(), h3.data_ptr(), khv.data_ptr(), vt.data_ptr()
    a.cache_out = _ptr(cache)
    _abi.check(lib.gecco_inducer_chain(C.byref(a), _stream(pooled)))
    return h3, khv, vt, cache


def unpool_attention(q: Tensor, khv: Tensor, *, clouds: int, rows_per_cloud: int, heads: int, head_dim: int, v_off: int,
                     inducers: int = 64, out: Tensor | None = None, tensor_cores: bool = True) -> Tensor:
    """Attention core of the unpool MultiheadAttention; with tensor_cores the tcgen05 / TMEM kernel is used where it
    applies (8 heads of 48 channels, rows_per_cloud % 128 == 0), see gecco_unpool_attention."""
    lib = _lib_for(q)
    assert q.dtype == torch.bfloat16 and khv.dtype == torch.bfloat16
    if out is None:
        out = torch.empty((clouds * rows_per_cloud, heads * head_dim), device=q.device, dtype=torch.bfloat16)
    a = _abi.UnpoolArgs()
    a.q, a.ldq = q.data_ptr(), q.stride(0)
    a.kv, a.ldkv, a.v_off = khv.data_ptr(), khv.stride(0), v_off
    a.clouds, a.rows_per_cloud = clouds, rows_per_cloud
    a.heads, a.head_dim, a.inducers = heads, head_dim, inducers
    a.out_bf16, a.ldo = out.data_ptr(), out.stride(0)
    if tensor_cores:
        vt = torch.empty((clouds, heads * head_dim, inducers), device=q.device, dtype=torch.bfloat16)
        a.vt_scratch = vt.data_ptr()
    _abi.check(lib.gecco_unpool_attention(C.byref(a), _stream(q)))
    return out


def adam_ema_step(p: Tensor, g: Tensor, m: Tensor, v: Tensor, ema: Tensor | None, step: int, *, lr: float = 1e-4,
                  betas: tuple[float, float] = (0.9, 0.999), eps: float = 1e-8, grad_scale: float = 1.0,
                  ema_decay: float = 0.999) -> None:
    """One fused Adam + weight-EMA update over flat fp32 buffers, in place (gecco_adam_ema_step; the reference's
    torch.optim.Adam defaults, diffusion.py:207-208, and ema.py:187-194)."""
    lib = _lib_for(p)
    for t in (p, g, m, v) + ((ema,) if ema is not None else ()):
        assert t.dtype == torch.float32 and t.is_contiguous() and t.numel() == p.numel() and t.device == p.device
    _abi.check(lib.gecco_adam_ema_step(_ptr(p), _ptr(g), _ptr(m), _ptr(v), _ptr(ema), p.numel(), int(step), float(lr), float(betas[0]),
                                       float(betas[1]), float(eps), float(grad_scale), float(ema_decay), _stream(p)))


# ---------------------------------------------------------------------------------------------------------------------
# training-path element-wise kernels (csrc/train_ops.cu)
def _f32c(t: Tensor) -> Tensor:
    assert t.dtype == torch.float32 and t.is_contiguous(), "fp32 contiguous tensor expected"
    return t


def train_gauss_act_fwd(x: Tensor, alpha: Tensor, normalized: bool = True) -> Tensor:
    lib = _lib_for(x)
    y = torch.empty_like(_f32c(x))
    _abi.check(lib.gecco_train_gauss_act_fwd(_ptr(x), _ptr(_f32c(alpha)), _ptr(y), x.numel(), int(normalized), _stream(x)))
    return y


def train_gauss_act_bwd(x: Tensor, dy: Tensor, alpha: Tensor, normalized: bool = True) -> tuple[Tensor, Tensor]:
    lib = _lib_for(x)
    dx = torch.empty_like(_f32c(x))
    parts = torch.empty((max(1, int(lib.gecco_train_gauss_act_bwd_parts(x.numel()))),), device=x.device, dtype=torch.float32)
    _abi.check(lib.gecco_train_gauss_act_bwd(_ptr(x), _ptr(_f32c(dy)), _ptr(_f32c(alpha)), _ptr(dx), _ptr(parts), x.numel(),
                                             int(normalized), _stream(x)))
    return dx, parts.sum() if x.numel() else parts.sum() * 0


def train_affine(u: Tensor, w: Tensor | None, p: Tensor, q: Tensor | None, r: Tensor) -> Tensor:
    """out[b,n,c] = p[b,c] u + (q[b,c] w) + r[b,c] for u (and w) [B, N, C]; p, q, r [B, C]."""
    lib = _lib_for(u)
    B, N, Cc = u.shape
    out = torch.empty_like(_f32c(u))
    _abi.check(lib.gecco_train_affine(_ptr(u), _ptr(None if w is None else _f32c(w)), _ptr(_f32c(p)),
                                      _ptr(None if q is None else _f32c(q)), _ptr(_f32c(r)), _ptr(out), B, N, Cc, _stream(u)))
    return out


def train_colsum2(dy: Tensor, x: Tensor) -> Tensor:
    """[B, C, 2]: sum over the rows of dy and of dy * x."""
    lib = _lib_for(x)
    B, N, Cc = x.shape
    parts = int(lib.gecco_train_colsum2_parts(N, Cc))
    out = torch.empty((B, max(parts, 1), Cc, 2), device=x.device, dtype=torch.float32)
    _abi.check(lib.gecco_train_colsum2(_ptr(_f32c(dy)), _ptr(_f32c(x)), _ptr(out), B, N, Cc, _stream(x)))
    return out.sum(dim=1)

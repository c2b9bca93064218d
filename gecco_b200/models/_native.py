"""Module-level execution of the SetTransformer pieces over the C-ABI kernels (`ops.*`).

The denoiser engine (`engine.py` / `csrc/engine.cu`) runs the whole stack with its own fusions; these helpers back the
stand-alone `forward`s of `MLP`, `AttentionPool`, `Broadcast`, `BroadcastingLayer` and `SetTransformer`
(reference call surface, set_transformer.py:47-216) with the SAME kernels: tcgen05 GEMMs with fused bias / activation /
residual epilogues and the two attention cores.  Torch only pads, reshapes and converts dtypes here.
"""
from __future__ import annotations

import math

import torch
from torch import Tensor

from .. import _abi, ops

ROW_TILE = 128  # rows per cloud are padded to the row tile of the tcgen05 kernels
SUPPORTED_INDUCERS = (64, 128, 192, 256)  # whole 64-row blocks of the attention cores
_LOG2E = 1.4426950408889634


def pad_rows(x: Tensor) -> tuple[Tensor, int, int]:
    """[B, N, C] (any float dtype) -> bf16 [B * Np, C] with zero rows N..Np, plus (N, Np)."""
    assert x.ndim == 3, "expected [batch, points, channels]"
    B, N, C = x.shape
    Np = (N + ROW_TILE - 1) // ROW_TILE * ROW_TILE
    xb = torch.zeros((B, Np, C), device=x.device, dtype=torch.bfloat16)
    xb[:, :N] = x.detach()
    return xb.view(B * Np, C), N, Np


def pad_rows_f32(x: Tensor, Np: int) -> Tensor:
    B, N, C = x.shape
    xf = torch.zeros((B, Np, C), device=x.device, dtype=torch.float32)
    xf[:, :N] = x.detach()
    return xf.view(B * Np, C)


def bf16(w: Tensor, scale: float = 1.0) -> Tensor:
    w = w.detach()
    return (w * scale if scale != 1.0 else w).to(torch.bfloat16).contiguous()


def f32(b: Tensor | None, scale: float = 1.0) -> Tensor | None:
    if b is None:
        return None
    b = b.detach().to(torch.float32)
    return (b * scale if scale != 1.0 else b).contiguous()


def linear(a: Tensor, weight: Tensor, bias: Tensor | None, *, rows_per_cloud: int, valid_rows: int, act_alpha: float | None = None,
           act: int | None = None, res: Tensor | None = None, want_f32: bool = False, want_bf16: bool = False,
           w_scale: float = 1.0):
    """a: bf16 [M, K]; returns (fp32 | None, bf16 | None) of epilogue(a @ weight.T + bias) (gecco_gemm)."""
    return ops.gemm(a, bf16(weight, w_scale), bias=f32(bias, w_scale), act_alpha=act_alpha, act=act, res=res,
                    out_f32=want_f32 or None, out_bf16=want_bf16 or None, rows_per_cloud=rows_per_cloud, valid_rows=valid_rows)


def epilogue_activation(act) -> tuple[int, float | None] | None:
    """(GECCO_ACT_* code, alpha) of an activation module the GEMM epilogue applies (the two GaussianActivation forms and
    nn.ReLU), else None."""
    from .activation import GaussianActivation

    if isinstance(act, GaussianActivation):
        return (_abi.ACT_GAUSSIAN if act.normalized else _abi.ACT_GAUSSIAN_RAW), float(act.alpha)
    if isinstance(act, torch.nn.ReLU):
        return _abi.ACT_RELU, None
    return None


def mlp_forward(mlp, x: Tensor, residual: Tensor | None = None) -> Tensor:
    """MLP.forward (mlp.py:5-39) on [B, N, C_in]; `residual` ([B, N, C_out]) is added in the last epilogue."""
    B, N, _ = x.shape
    a, N, Np = pad_rows(x)
    mods = list(mlp)
    lin, rest = mods[0], mods[1:]
    h16 = None
    while rest:
        act, nxt, rest = rest[0], rest[1], rest[2:]
        fused = epilogue_activation(act)
        if fused is not None:
            # activation fused into the epilogue of the projection that feeds it
            _, h16 = linear(a if h16 is None else h16, lin.weight, lin.bias, rows_per_cloud=Np, valid_rows=N,
                            act=fused[0], act_alpha=fused[1], want_bf16=True)
        else:
            z, _ = linear(a if h16 is None else h16, lin.weight, lin.bias, rows_per_cloud=Np, valid_rows=N, want_f32=True)
            h16 = act(z).to(torch.bfloat16)  # any other activation module runs on the fp32 projection output
        lin = nxt
    res = None if residual is None else pad_rows_f32(residual, Np)
    out, _ = linear(h16 if h16 is not None else a, lin.weight, lin.bias, rows_per_cloud=Np, valid_rows=N, res=res, want_f32=True)
    return out.view(B, Np, -1)[:, :N].to(x.dtype)


def attention_pool_forward(pool, kv: Tensor) -> Tensor:
    """AttentionPool.forward (set_transformer.py:47-65): kv_proj GEMM -> split-key attention core -> out_proj GEMM."""
    B, N, C = kv.shape
    H, d = pool.num_heads, pool.dims_per_head
    I = pool.inducers.shape[2]
    a, N, Np = pad_rows(kv)
    _, kvp = linear(a, pool.kv_proj.weight, None, rows_per_cloud=Np, valid_rows=N, want_bf16=True)  # [B*Np, 2C]: (t h d)
    q = bf16(pool.inducers[0], _LOG2E / math.sqrt(d))  # [H, I, d], softmax scale and exp -> exp2 folded in
    pooled = ops.pool_attention(kvp, q, clouds=B, rows_per_cloud=Np, valid_rows=N, heads=H, head_dim=d, k_off=0, v_off=C)
    out, _ = linear(pooled, pool.out_proj.weight, None, rows_per_cloud=I, valid_rows=I, want_f32=True)
    return out.view(B, I, C).to(kv.dtype)


def unpool_forward(mha, x: Tensor, h: Tensor, residual: Tensor | None = None) -> Tensor:
    """nn.MultiheadAttention(batch_first)(query=x, key=h, value=h) (set_transformer.py:90,112): in-projections, attention
    core over the inducers, out-projection (+ residual)."""
    B, N, C = x.shape
    H = mha.num_heads
    d = C // H
    I = h.shape[1]
    if I not in SUPPORTED_INDUCERS:
        raise ValueError(f"gecco_b200: the unpool attention kernels support 64, 128, 192 or 256 inducers, got {I}")
    a, N, Np = pad_rows(x)
    w, b = mha.in_proj_weight, mha.in_proj_bias
    qs = _LOG2E / math.sqrt(d)
    _, q = linear(a, w[:C], None if b is None else b[:C], rows_per_cloud=Np, valid_rows=N, want_bf16=True, w_scale=qs)
    h16 = h.detach().to(torch.bfloat16).reshape(B * I, C).contiguous()
    _, khv = linear(h16, w[C:], None if b is None else b[C:], rows_per_cloud=I, valid_rows=I, want_bf16=True)  # [B*I, 2C]
    y = ops.unpool_attention(q, khv, clouds=B, rows_per_cloud=Np, heads=H, head_dim=d, v_off=C, inducers=I)
    res = None if residual is None else pad_rows_f32(residual, Np)
    out, _ = linear(y, mha.out_proj.weight, mha.out_proj.bias, rows_per_cloud=Np, valid_rows=N, res=res, want_f32=True)
    return out.view(B, Np, C)[:, :N].to(x.dtype)

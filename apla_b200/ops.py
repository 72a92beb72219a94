"""Tensor-level wrappers over the C ABI (include/apla_b200.h).  Device memory comes from torch tensors, all
arithmetic happens in libapla_b200.so on torch's current stream.  Every wrapper validates dtype / device /
contiguity and raises; nothing here falls back to PyTorch math."""
from __future__ import annotations

from typing import Optional, Tuple

import torch

from ._lib import LIB, ptr, require_device, stream

BF16, F32 = torch.bfloat16, torch.float32


def _chk(t: torch.Tensor, dtype, name: str, dim: Optional[int] = None):
    if not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor")
    if t.dtype != dtype:
        raise RuntimeError(f"{name} must be {dtype}, got {t.dtype}")
    if dim is not None and t.dim() != dim:
        raise RuntimeError(f"{name} must be {dim}-D, got shape {tuple(t.shape)}")
    if t.stride(-1) != 1:
        raise RuntimeError(f"{name} must be contiguous along the last dimension")


def _ld(t: torch.Tensor) -> int:
    return t.stride(0) if t.dim() == 2 else t.shape[-1]


def gemm_bias(a, w, bias=None, out=None):
    """out[M,N] = a[M,K] @ w[N,K]^T + bias (bf16)."""
    require_device()
    _chk(a, BF16, "a", 2); _chk(w, BF16, "w", 2)
    M, K = a.shape; N = w.shape[0]
    if out is None:
        out = torch.empty(M, N, device=a.device, dtype=BF16)
    LIB.call("apla_gemm_bias_fwd", ptr(a), _ld(a), ptr(w), _ld(w), ptr(bias), ptr(out), _ld(out), M, N, K, stream())
    return out


def gemm_bias_gelu(a, w, bias=None, h=None, g=None):
    require_device()
    _chk(a, BF16, "a", 2); _chk(w, BF16, "w", 2)
    M, K = a.shape; N = w.shape[0]
    if h is None:
        h = torch.empty(M, N, device=a.device, dtype=BF16)
    if g is None:
        g = torch.empty(M, N, device=a.device, dtype=BF16)
    assert _ld(h) == _ld(g)
    LIB.call("apla_gemm_bias_gelu_fwd", ptr(a), _ld(a), ptr(w), _ld(w), ptr(bias), ptr(h), ptr(g), _ld(h), M, N, K,
             stream())
    return h, g


def gemm_bias_ls_residual(a, w, bias, gamma, resid, out=None):
    """out_f32 = resid_f32 + gamma * (a @ w^T + bias); out may alias resid."""
    require_device()
    _chk(a, BF16, "a", 2); _chk(w, BF16, "w", 2); _chk(resid, F32, "resid", 2)
    M, K = a.shape; N = w.shape[0]
    if out is None:
        out = torch.empty(M, N, device=a.device, dtype=F32)
    assert _ld(out) == _ld(resid)
    LIB.call("apla_gemm_bias_ls_residual_fwd", ptr(a), _ld(a), ptr(w), _ld(w), ptr(bias), ptr(gamma), ptr(resid),
             ptr(out), _ld(out), M, N, K, stream())
    return out


def gemm_bias_ls_residual_ln(a, w, bias, gamma, resid, ln_w, ln_b, eps: float, out=None, ln_out=None, one_launch: int = -1):
    """out_f32 = resid + gamma * (a @ w^T + bias) and ln_out_bf16 = LayerNorm(out_f32); one_launch=1 asks for the single
    fused launch (widths 384 / 768 / 1024), 0 for the two kernels, -1 for the library default.  -> (out, ln_out)."""
    require_device()
    _chk(a, BF16, "a", 2); _chk(w, BF16, "w", 2); _chk(resid, F32, "resid", 2)
    _chk(ln_w, F32, "ln_w", 1); _chk(ln_b, F32, "ln_b", 1)
    M, K = a.shape; N = w.shape[0]
    if out is None:
        out = torch.empty(M, N, device=a.device, dtype=F32)
    if ln_out is None:
        ln_out = torch.empty(M, N, device=a.device, dtype=BF16)
    assert _ld(out) == _ld(resid)
    LIB.call("apla_gemm_bias_ls_residual_ln_fwd", ptr(a), _ld(a), ptr(w), _ld(w), ptr(bias), ptr(gamma), ptr(resid),
             ptr(out), _ld(out), ptr(ln_w), ptr(ln_b), ptr(ln_out), _ld(ln_out), float(eps), M, N, K, int(one_launch), stream())
    return out, ln_out


def gemm_dgrad(dy, wt, out=None):
    """dx[M,Kin] = dy[M,Nout] @ wt[Kin,Nout]^T with wt the pre-transposed frozen weight."""
    require_device()
    _chk(dy, BF16, "dy", 2); _chk(wt, BF16, "wt", 2)
    M, Nout = dy.shape; Kin = wt.shape[0]
    if out is None:
        out = torch.empty(M, Kin, device=dy.device, dtype=BF16)
    LIB.call("apla_gemm_dgrad", ptr(dy), _ld(dy), ptr(wt), _ld(wt), ptr(out), _ld(out), M, Kin, Nout, stream())
    return out


def gemm_bias_gelu_dgelu(a, w, bias=None, d=None, g=None):
    """g_bf16 = gelu(a @ w^T + bias), d_f16 = gelu'(a @ w^T + bias): fc1 forward that saves the derivative."""
    require_device()
    _chk(a, BF16, "a", 2); _chk(w, BF16, "w", 2)
    M, K = a.shape; N = w.shape[0]
    if d is None:
        d = torch.empty(M, N, device=a.device, dtype=torch.float16)
    if g is None:
        g = torch.empty(M, N, device=a.device, dtype=BF16)
    _chk(d, torch.float16, "d", 2); _chk(g, BF16, "g", 2)
    assert _ld(d) == _ld(g)
    LIB.call("apla_gemm_bias_gelu_dgelu_fwd", ptr(a), _ld(a), ptr(w), _ld(w), ptr(bias), ptr(d), ptr(g), _ld(d), M, N, K,
             stream())
    return d, g


def gemm_dgrad_mul(dy, wt, mul, out=None):
    """dH_bf16 = (dy @ wt^T) * mul_f16."""
    require_device()
    _chk(dy, BF16, "dy", 2); _chk(wt, BF16, "wt", 2); _chk(mul, torch.float16, "mul", 2)
    M, Nout = dy.shape; Kin = wt.shape[0]
    if out is None:
        out = torch.empty(M, Kin, device=dy.device, dtype=BF16)
    assert _ld(out) == _ld(mul)
    LIB.call("apla_gemm_dgrad_mul", ptr(dy), _ld(dy), ptr(wt), _ld(wt), ptr(mul), ptr(out), _ld(out), M, Kin, Nout,
             stream())
    return out


def gemm_dgrad_delta(dy, wt, o, out=None, delta=None):
    """dO[M,D] = dy @ wt^T and delta[M, D/64] = per-head rowsum(dO * o): projection dgrad + attention-backward delta."""
    require_device()
    _chk(dy, BF16, "dy", 2); _chk(wt, BF16, "wt", 2); _chk(o, BF16, "o", 2)
    M, Nout = dy.shape; D = wt.shape[0]
    if D % 64 != 0 or tuple(o.shape) != (M, D):
        raise RuntimeError(f"o must be [{M},{D}] with D a multiple of 64, got {tuple(o.shape)}")
    if out is None:
        out = torch.empty(M, D, device=dy.device, dtype=BF16)
    if delta is None:
        delta = torch.empty(M, D // 64, device=dy.device, dtype=F32)
    assert _ld(out) == _ld(o) and delta.is_contiguous()
    LIB.call("apla_gemm_dgrad_delta", ptr(dy), _ld(dy), ptr(wt), _ld(wt), ptr(o), ptr(out), _ld(out), ptr(delta), M, D,
             Nout, stream())
    return out, delta


def gemm_dgrad_gelu_bwd(dy, wt, h, out=None):
    require_device()
    _chk(dy, BF16, "dy", 2); _chk(wt, BF16, "wt", 2); _chk(h, BF16, "h", 2)
    M, Nout = dy.shape; Kin = wt.shape[0]
    if out is None:
        out = torch.empty(M, Kin, device=dy.device, dtype=BF16)
    assert _ld(out) == _ld(h)
    LIB.call("apla_gemm_dgrad_gelu_bwd", ptr(dy), _ld(dy), ptr(wt), _ld(wt), ptr(h), ptr(out), _ld(out), M, Kin, Nout,
             stream())
    return out


def proj_wgrad(dysub, x, dw1, r: int, rowmap=None):
    """dw1_f32[r, Din] += dysub[T, n_pad]^T @ x[T, Din] (dw1 zero-initialised by the caller)."""
    require_device()
    _chk(dysub, BF16, "dysub", 2); _chk(x, BF16, "x", 2); _chk(dw1, F32, "dw1", 2)
    T, n_pad = dysub.shape
    LIB.call("apla_proj_wgrad_gather", ptr(dysub), _ld(dysub), ptr(x), _ld(x), ptr(rowmap), ptr(dw1), _ld(dw1), T,
             x.shape[1], n_pad, r, stream())
    return dw1


def colsum(dy, db, n: int, rowmap=None):
    require_device()
    _chk(dy, BF16, "dy", 2); _chk(db, F32, "db")
    LIB.call("apla_colsum", ptr(dy), _ld(dy), dy.shape[0], n, ptr(rowmap), ptr(db), stream())
    return db


def layernorm_fwd(x, w, b, eps: float, out=None):
    require_device()
    _chk(x, F32, "x", 2)
    rows, D = x.shape
    if out is None:
        out = torch.empty(rows, D, device=x.device, dtype=BF16)
    LIB.call("apla_layernorm_fwd", ptr(x), _ld(x), ptr(w), ptr(b), ptr(out), _ld(out), rows, D, eps, stream())
    return out


def layernorm_bwd(dy, x, w, eps: float, dres=None, dx=None, dxb=None, gamma=None, sub=None, idx=None, r: int = 0):
    """dx = dres + LN'(dy); optional dxb = bf16(gamma*dx); optional sub = gathered bf16 columns."""
    require_device()
    _chk(dy, BF16, "dy", 2); _chk(x, F32, "x", 2)
    rows, D = x.shape
    if dx is None:
        dx = torch.empty(rows, D, device=x.device, dtype=F32)
    r_pad = sub.shape[1] if sub is not None else 0
    LIB.call("apla_layernorm_bwd", ptr(dy), _ld(dy), ptr(x), _ld(x), ptr(w), ptr(dres),
             _ld(dres) if dres is not None else D, ptr(dx), _ld(dx), ptr(dxb), _ld(dxb) if dxb is not None else D,
             ptr(gamma), ptr(sub), _ld(sub) if sub is not None else 0, ptr(idx), r, r_pad, rows, D, eps, stream())
    return dx


def ls_cast(x, gamma=None, out=None):
    """out_bf16 = gamma * x_f32 (gamma None = plain down-cast)."""
    require_device()
    _chk(x, F32, "x", 2)
    rows, D = x.shape
    if out is None:
        out = torch.empty(rows, D, device=x.device, dtype=BF16)
    LIB.call("apla_ls_cast", ptr(x), _ld(x), ptr(gamma), ptr(out), _ld(out), rows, D, stream())
    return out


def gather_cols(dy, idx, r: int, r_pad: int, out=None):
    require_device()
    _chk(dy, BF16, "dy", 2)
    if out is None:
        out = torch.empty(dy.shape[0], r_pad, device=dy.device, dtype=BF16)
    LIB.call("apla_gather_cols", ptr(dy), _ld(dy), ptr(out), _ld(out), ptr(idx), r, r_pad, dy.shape[0], stream())
    return out


def attn_fwd(qkv, H: int, scale: float, num_seqs: int, max_seqlen: int, cu_seqlens=None, out=None, lse=None):
    require_device()
    _chk(qkv, BF16, "qkv", 2)
    T = qkv.shape[0]
    assert qkv.shape[1] == 3 * H * 64 and qkv.is_contiguous()
    if out is None:
        out = torch.empty(T, H * 64, device=qkv.device, dtype=BF16)
    if lse is None:
        lse = torch.empty(T, H, device=qkv.device, dtype=F32)
    LIB.call("apla_attn_fwd", ptr(qkv), ptr(out), ptr(lse), ptr(cu_seqlens), num_seqs, max_seqlen, T, H, scale, stream())
    return out, lse


def attn_bwd(qkv, out, dout, lse, H: int, scale: float, num_seqs: int, max_seqlen: int, cu_seqlens=None, dqkv=None,
             delta=None):
    require_device()
    _chk(qkv, BF16, "qkv", 2); _chk(dout, BF16, "dout", 2); _chk(lse, F32, "lse", 2)
    T = qkv.shape[0]
    assert dout.is_contiguous() and qkv.is_contiguous()
    if out is None:      # delta precomputed by gemm_dgrad_delta
        if delta is None:
            raise RuntimeError("attn_bwd: out=None needs the precomputed delta")
    else:
        _chk(out, BF16, "out", 2)
        assert out.is_contiguous()
    if dqkv is None:
        dqkv = torch.empty_like(qkv)
    if delta is None:
        delta = torch.empty(T, H, device=qkv.device, dtype=F32)
    LIB.call("apla_attn_bwd", ptr(qkv), ptr(out), ptr(dout), ptr(lse), ptr(delta), ptr(dqkv), ptr(cu_seqlens),
             num_seqs, max_seqlen, T, H, scale, stream())
    return dqkv


def attn_cls_fwd(qkv, H: int, scale: float, B: int, N: int, out=None, lse=None):
    """Row b*N of the attention output / lse only (the CLS query of each of the B sequences of N tokens)."""
    require_device()
    _chk(qkv, BF16, "qkv", 2)
    T = qkv.shape[0]
    assert T == B * N and qkv.shape[1] == 3 * H * 64 and qkv.is_contiguous()
    if out is None:
        out = torch.zeros(T, H * 64, device=qkv.device, dtype=BF16)
    if lse is None:
        lse = torch.zeros(T, H, device=qkv.device, dtype=F32)
    LIB.call("apla_attn_cls_fwd", ptr(qkv), ptr(out), ptr(lse), B, N, H, scale, stream())
    return out, lse


def attn_cls_bwd(qkv, out, dout, lse, H: int, scale: float, B: int, N: int, dqkv=None):
    """dqkv for a dout that is non-zero on the CLS rows only (rows b*N of out / dout / lse are read)."""
    require_device()
    _chk(qkv, BF16, "qkv", 2); _chk(out, BF16, "out", 2); _chk(dout, BF16, "dout", 2); _chk(lse, F32, "lse", 2)
    assert qkv.shape[0] == B * N and qkv.is_contiguous() and out.is_contiguous() and dout.is_contiguous()
    if dqkv is None:
        dqkv = torch.empty_like(qkv)
    LIB.call("apla_attn_cls_bwd", ptr(qkv), ptr(out), ptr(dout), ptr(lse), ptr(dqkv), B, N, H, scale, stream())
    return dqkv


def attn_probs(qkv, lse, H: int, scale: float, B: int, N: int, q_rows: Optional[int] = None, out=None):
    """fp32 [B, H, q_rows, N] attention probabilities of the first q_rows (default N) queries of each of the B dense
    sequences, from the qkv and lse of the forward (`attn_fwd`, or `attn_cls_fwd` for q_rows = 1)."""
    require_device()
    _chk(qkv, BF16, "qkv", 2); _chk(lse, F32, "lse", 2)
    q_rows = N if q_rows is None else int(q_rows)
    if qkv.shape != (B * N, 3 * H * 64) or not qkv.is_contiguous():
        raise RuntimeError(f"qkv must be contiguous [{B * N}, {3 * H * 64}], got {tuple(qkv.shape)}")
    if lse.shape != (B * N, H) or not lse.is_contiguous():
        raise RuntimeError(f"lse must be contiguous [{B * N}, {H}], got {tuple(lse.shape)}")
    if out is None:
        out = torch.empty(B, H, q_rows, N, device=qkv.device, dtype=F32)
    else:
        _chk(out, F32, "out")
        if out.numel() < B * H * q_rows * N or not out.is_contiguous():
            raise RuntimeError(f"out must be contiguous with at least {B * H * q_rows * N} elements")
    LIB.call("apla_attn_probs", ptr(qkv), ptr(lse), ptr(out), B, N, H, q_rows, scale, stream())
    return out


def gemm_bias_ls_accumulate(a, w, bias, gamma, out):
    """out_f32 += gamma * (a @ w^T + bias), in place (TMA reduce-add epilogue)."""
    require_device()
    _chk(a, BF16, "a", 2); _chk(w, BF16, "w", 2); _chk(out, F32, "out", 2)
    M, K = a.shape; N = w.shape[0]
    LIB.call("apla_gemm_bias_ls_accumulate", ptr(a), _ld(a), ptr(w), _ld(w), ptr(bias), ptr(gamma), ptr(out), _ld(out),
             M, N, K, stream())
    return out

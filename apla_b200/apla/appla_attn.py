"""`APLA_Attention`: drop-in for the reference module of the same name (src/apla/appla_attn.py:10-83).

Same constructor signature, attributes, parameter / buffer names and random-number consumption (the index
permutation is drawn from the global CPU generator BEFORE the qkv Linear is initialised, appla_attn.py:26,37), so
reference checkpoints and `inds` interchange.  The arithmetic of `forward` and of its autograd backward runs in
libapla_b200.so:

    qkv GEMM (tcgen05)  ->  fused softmax attention (saves log-sum-exp only)  ->  ONE dense projection GEMM over a
    full-layout bf16 copy of the weight (replaces the two F.linear + torch.empty + two index uploads + two scatter_
    of appla_attn.py:64-79)

    backward: input gradients through proj / attention / qkv when the input requires grad, weight gradient ONLY for
    the trainable rows:  dW1 = dY[:, idx]^T . X ,  db1 = sum_t dY[t, idx]   (what autograd derives from scatter_).

There is no PyTorch fallback: on a non-CUDA input or without the library a RuntimeError is raised.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from .. import ops
from .._lib import LIB, ptr, require_device, stream

_VERBOSE = False


def print_ddp(msg: str) -> None:
    """Rank-0 print of the reference (src/utils/dist_utills.py:34-39); silent unless apla.appla_attn._VERBOSE."""
    if not _VERBOSE:
        return
    if torch.distributed.is_available() and torch.distributed.is_initialized() and torch.distributed.get_rank() != 0:
        return
    print(msg)


def _pad64(n: int) -> int:
    return (n + 63) // 64 * 64


class _AplaAttentionFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, w1, b1, mod, cu_seqlens, seqlens, want_attn=False):
        ws = mod._working_set(x.device)
        shape = x.shape
        C = shape[-1]
        xb = x.reshape(-1, C).to(torch.bfloat16).contiguous()
        T = xb.shape[0]
        if cu_seqlens is None:
            num_seqs, max_len = (shape[0], shape[1]) if x.dim() == 3 else (1, T)
        else:
            num_seqs, max_len = len(seqlens), max(seqlens)
        qkv = ops.gemm_bias(xb, ws["wqkv"], ws["bqkv"])
        ao, lse = ops.attn_fwd(qkv, mod.num_heads, float(mod.scale), num_seqs, max_len, cu_seqlens=cu_seqlens)
        y = ops.gemm_bias(ao, ws["wproj"], ws["bproj"])
        if want_attn:                # the probabilities of this very forward, from its qkv and lse (dense input only)
            attn = ops.attn_probs(qkv, lse, mod.num_heads, float(mod.scale), num_seqs, max_len)
            ctx.mark_non_differentiable(attn)
        ctx.mod, ctx.ws = mod, ws
        ctx.geom = (num_seqs, max_len, cu_seqlens)
        ctx.x_dtype, ctx.x_shape = x.dtype, shape
        ctx.save_for_backward(qkv, ao, lse)
        y = y.view(shape).to(x.dtype)
        return (y, attn) if want_attn else y

    @staticmethod
    def backward(ctx, dy, *_):
        mod, ws = ctx.mod, ctx.ws
        qkv, ao, lse = ctx.saved_tensors
        num_seqs, max_len, cu = ctx.geom
        C = ctx.x_shape[-1]
        r = mod.partial_size
        dyb = dy.reshape(-1, C).to(torch.bfloat16).contiguous()
        dw1 = db1 = dx = None
        if ctx.needs_input_grad[1] or ctx.needs_input_grad[2]:
            dw1 = torch.zeros(r, C, device=dy.device, dtype=torch.float32)
            db1 = torch.zeros(r, device=dy.device, dtype=torch.float32)
            if ws["rowmap"] is not None:                # partial_size == dim: dense dY, rows permuted in the epilogue
                ops.proj_wgrad(dyb, ao, dw1, r, rowmap=ws["rowmap"])
                ops.colsum(dyb, db1, C, rowmap=ws["rowmap"])
            else:
                sub = ops.gather_cols(dyb, ws["idx"], r, _pad64(r))
                ops.proj_wgrad(sub, ao, dw1, r)
                ops.colsum(sub, db1, r)
        if ctx.needs_input_grad[0]:
            d_ao, delta = ops.gemm_dgrad_delta(dyb, ws["wprojT"], ao)
            dqkv = ops.attn_bwd(qkv, None, d_ao, lse, mod.num_heads, float(mod.scale), num_seqs, max_len,
                                cu_seqlens=cu, delta=delta)
            dx = ops.gemm_dgrad(dqkv, ws["wqkvT"]).view(ctx.x_shape).to(ctx.x_dtype)
        return dx, dw1, db1, None, None, None, None


class APLA_Attention(nn.Module):
    # set by `apla_b200.apla.attention_probabilities(model)`: forward then also returns the [B,H,N,N] probabilities
    _attention_probs = False

    def __init__(self, config, dim, indices=None, num_heads=8, qkv_bias=False, qk_scale=None, attn_drop=0.,
                 proj_drop=0.):
        super().__init__()
        if dim % num_heads != 0 or dim // num_heads != 64:
            raise ValueError(f"apla_b200 kernels are built for head_dim 64 (dim={dim}, num_heads={num_heads})")
        self.num_heads = num_heads
        self.scale = qk_scale or (dim // num_heads) ** -0.5
        self.partial_size = config.partial_size
        self.dim = dim

        # indices: given, or one permutation drawn at construction from the global CPU generator
        if indices is not None:
            self.indices = indices
            print_ddp("APLA_Attention init: Using provided indices")
        else:
            self.indices = torch.randperm(self.dim)
            print_ddp("APLA_Attention init: Sampled a set of random indices")
        self.register_buffer("inds", self.indices)
        self.trainable_inds = self.indices[:self.partial_size]
        self.freezed_inds = self.indices[self.partial_size:]

        self.qkv = nn.Linear(dim, dim * 3, bias=qkv_bias)          # frozen
        for p in self.qkv.parameters():
            p.requires_grad = False

        r = self.partial_size
        self.proj_weight1 = nn.Parameter(torch.empty(r, dim), requires_grad=True)
        self.proj_weight2 = nn.Parameter(torch.empty(dim - r, dim), requires_grad=False)
        self.proj_bias1 = nn.Parameter(torch.empty(r), requires_grad=True)
        self.proj_bias2 = nn.Parameter(torch.empty(dim - r), requires_grad=False)

        self.attn_drop = nn.Dropout(attn_drop)
        self.proj_drop = nn.Dropout(proj_drop)
        self._ws = None
        self._ws_key = None
        self._ws_train_key = None

    # ---- bf16 working copies of the (mostly frozen) weights ------------------------------------------------------
    @staticmethod
    def _tkey(t):
        return (t.data_ptr(), t._version, t.device)

    def refresh_working_set(self):
        """Drop the cached bf16 working copies; the next forward rebuilds them from the parameters.

        The cache is keyed on (data_ptr, _version, device) of every source tensor, which sees optimiser steps, `copy_`,
        `load_state_dict` and `.to()`.  It does NOT see a write that bypasses autograd's version counter: `p.data.add_()`,
        an optimiser that steps on `.data`, or an external kernel writing through the raw pointer.  After such a write
        call this (or `torch.autograd.graph.increment_version(p)`, which is what `SSLMetaArch.update_teacher` does after
        its fused EMA kernel)."""
        self._ws = None
        self._ws_key = None
        self._ws_train_key = None

    def _working_set(self, device):
        """Dense bf16 copies consumed by the kernels.  Frozen tensors are converted once; the trainable rows are
        scattered into the dense projection copies again whenever proj_weight1 / proj_bias1 changed (see
        `refresh_working_set` for the one kind of write this cannot notice)."""
        frozen_key = (self._tkey(self.qkv.weight), self._tkey(self.proj_weight2), self._tkey(self.proj_bias2),
                      None if self.qkv.bias is None else self._tkey(self.qkv.bias))
        r, D = self.partial_size, self.dim
        if self._ws is None or self._ws_key != frozen_key:
            with torch.no_grad():
                # like the reference, the split follows the constructor-time `indices` attribute (appla_attn.py:33-34),
                # not the `inds` buffer a checkpoint may have overwritten
                inds = torch.as_tensor(self.indices).to(device=device, dtype=torch.long)
                wq = self.qkv.weight.detach().to(device=device, dtype=torch.bfloat16).contiguous()
                bq = (self.qkv.bias.detach().to(device=device, dtype=torch.float32).contiguous()
                      if self.qkv.bias is not None else torch.zeros(3 * D, device=device))
                wfull = torch.zeros(D, D, device=device, dtype=torch.bfloat16)
                bfull = torch.zeros(D, device=device, dtype=torch.float32)
                if r < D:
                    wfull[inds[r:]] = self.proj_weight2.detach().to(device=device, dtype=torch.bfloat16)
                    bfull[inds[r:]] = self.proj_bias2.detach().to(device=device, dtype=torch.float32)
                rowmap = None
                if r > 128:
                    rowmap = torch.full((D,), -1, dtype=torch.int32, device=device)
                    rowmap[inds[:r]] = torch.arange(r, dtype=torch.int32, device=device)
                self._ws = dict(wqkv=wq, wqkvT=wq.t().contiguous(), bqkv=bq, wproj=wfull, wprojT=wfull.t().contiguous(),
                                bproj=bfull, idx=inds[:r].to(torch.int32).contiguous(), rowmap=rowmap)
            self._ws_key = frozen_key
            self._ws_train_key = None
        train_key = (self._tkey(self.proj_weight1), self._tkey(self.proj_bias1))
        if self._ws_train_key != train_key:
            ws = self._ws
            w1 = self.proj_weight1.detach()
            b1 = self.proj_bias1.detach()
            if w1.dtype != torch.float32 or not w1.is_contiguous() or b1.dtype != torch.float32:
                raise RuntimeError("proj_weight1 / proj_bias1 must be contiguous fp32 CUDA parameters")
            LIB.call("apla_proj_refresh", ptr(w1), ptr(b1), ptr(ws["idx"]), ptr(ws["wproj"]), ptr(ws["wprojT"]),
                     ptr(ws["bproj"]), 1, r, D, 0, 0, stream())
            self._ws_train_key = train_key
        return self._ws

    def _run(self, x, cu_seqlens=None, seqlens=None, want_attn=False):
        if not x.is_cuda:
            raise RuntimeError("apla_b200.APLA_Attention runs on CUDA (sm_100a) only; there is no CPU fallback")
        require_device()
        if self.training and (self.attn_drop.p > 0 or self.proj_drop.p > 0):
            raise RuntimeError("fused APLA attention supports dropout p=0 only (all shipped reference configs use 0)")
        if self.proj_weight1.device != x.device:
            raise RuntimeError("module parameters and input are on different devices")
        return _AplaAttentionFn.apply(x, self.proj_weight1, self.proj_bias1, self, cu_seqlens, seqlens, want_attn)

    def forward(self, x):
        """x [B,N,C] -> (out [B,N,C], attn).  The reference returns the [B,H,N,N] probabilities, which the fused
        kernel does not materialise: `attn` is None (its only consumers are visualisation paths, vit.py:282-287), unless
        the module is inside `apla_b200.apla.attention_probabilities(...)`.  There `attn` is the fp32 [B,H,N,N] softmax
        of this call (contiguous, rebuilt by one extra kernel from the forward's own qkv and log-sum-exp) with no
        autograd history: no gradient flows through it.  `out` and the gradients come from the same launches as without
        it (the extra kernel only reads qkv and lse)."""
        if not self._attention_probs:
            return self._run(x), None
        if x.dim() != 3:
            raise RuntimeError(f"attention probabilities need a dense [B, N, C] input, got shape {tuple(x.shape)}")
        return self._run(x, want_attn=True)

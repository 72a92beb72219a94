"""`FusedAplaBlock` / `fuse_apla_blocks`: the whole transformer block around an APLA attention as ONE autograd node.

`APLA_Attention` (appla_attn.py) replaces the reference's attention module only; the block around it
(`Block.forward` src/utils/transformers/vit.py:279-288: LayerNorm, LayerScale, residual adds, `Mlp` :162-168 with exact
GELU; `NestedTensorBlock` src/self_supervised/dinov2/layers/block.py:244-288 for lists of crops) would still run as
~10 ATen kernels per direction, keep every LayerNorm / fc1 / GELU output for autograd and compute nothing in bf16
tensor-core GEMMs unless the caller wraps it in autocast.  `fuse_apla_blocks(model)` swaps each block whose attention
is an `APLA_Attention` for a `FusedAplaBlock` that holds the SAME sub-modules under the SAME names (state-dict keys and
checkpoints unchanged) and runs forward and backward through the kernels the step engine uses:

  (two native calls per block and step: `apla_block_fwd`, `apla_block_bwd`, csrc/block.cu; when autograd would record
  nothing -- under torch.no_grad(), or with neither the input nor proj_weight1 / proj_bias1 requiring grad -- the forward
  is `apla_block_fwd_infer` instead: same output bit for bit, no saved tensors, no GELU derivative written)
  forward   LN1 -> qkv GEMM -> fused attention (saves log-sum-exp) -> proj GEMM (+bias, xLayerScale, +residual, fp32)
            -> LN2 -> fc1 GEMM (+bias, GELU, saves gelu' in fp16) -> fc2 GEMM (+bias, xLayerScale, +residual, fp32)
  backward  LayerScale+cast -> fc2 dgrad x gelu' -> fc1 dgrad -> LN2' (+residual grad, xLayerScale, APLA column gather)
            -> weight gradient of the r trainable projection rows -> proj dgrad (+attention delta) -> attention'
            -> qkv dgrad -> LN1' (+residual grad)

Saved per block: the two fp32 residual checkpoints, qkv, the attention output, log-sum-exp and gelu' -- no LayerNorm
output, no [B,H,N,N] probabilities, no fc1 pre- or post-activation.  Gradients flow to EVERY token of the input (dense
prediction heads, SSL patch losses) and to `proj_weight1` / `proj_bias1`; nothing is computed for frozen tensors.
Accepts `[B,N,D]` tensors (vit.py Block) and lists of `[b_i,N_i,D]` crops, which are packed and attended
block-diagonally (dinov2 NestedTensorBlock.forward_nested; get_attn_bias_and_cat block.py:191-217).

The residual stream is fp32 inside the node whatever the input dtype (what autocast keeps in fp32, SURVEY.md 8a); the
output has the input's dtype.  CUDA (sm_100a) only, no fallback.  Dropout must be off (all shipped reference configs run
it at 0).  Stochastic depth (drop path, vit.py drop_path / timm `drop_path1` / `drop_path2`) runs on `[B,N,D]` tensors:
in training mode the block calls its own drop-path modules on a ones tensor for the per-image branch scales, so it
draws exactly the masks the unfused block draws, and the native calls scale each image's branch output by them
(`apla_block_fwd_scaled` / `apla_block_bwd_scaled`).  Lists of crops with a nonzero drop-path rate are refused.
"""
from __future__ import annotations

import contextlib
import ctypes
import os
import weakref
from typing import List, Optional, Sequence

import torch
import torch.nn as nn

from .. import ops
from .._lib import LIB, BlockWeights, ptr, require_device, stream
from .appla_attn import APLA_Attention, _pad64


_CHAIN = os.environ.get("APLA_BLOCK_CHAIN", "1") != "0"      # hand bf16(gamma2 * dx) from block to block in backward


def _fwd_setup(blk, x, cu_seqlens, seqlens):
    """Native weights, fp32 input rows, geometry and the buffers both forwards write:
    -> (nat, x_in, T, num_seqs, max_len, (x_mid, x_out, qkv, ao, lse, ln_tmp, gelu_tmp))."""
    at = blk.attn
    nat = blk._native(x.device)
    D, H, Hd = at.dim, at.num_heads, blk.mlp.fc1.out_features
    x_in = x.reshape(-1, D).to(torch.float32).contiguous()
    T = x_in.shape[0]
    if cu_seqlens is None:
        num_seqs, max_len = (x.shape[0], x.shape[1]) if x.dim() == 3 else (1, T)
    else:
        num_seqs, max_len = len(seqlens), max(seqlens)
    dev, bf, f32 = x.device, torch.bfloat16, torch.float32
    bufs = (torch.empty(T, D, device=dev, dtype=f32), torch.empty(T, D, device=dev, dtype=f32),
            torch.empty(T, 3 * D, device=dev, dtype=bf), torch.empty(T, D, device=dev, dtype=bf),
            torch.empty(T, H, device=dev, dtype=f32), torch.empty(T, D, device=dev, dtype=bf),
            torch.empty(T, Hd, device=dev, dtype=bf))
    return nat, x_in, T, num_seqs, max_len, bufs


class _AplaBlockFn(torch.autograd.Function):
    """One native call per direction (`apla_block_fwd` / `apla_block_bwd`, csrc/block.cu): 7 + up to 13 kernel launches
    with no Python between them."""

    @staticmethod
    def forward(ctx, x, w1, b1, blk, cu_seqlens, seqlens, scales):
        nat, x_in, T, num_seqs, max_len, (x_mid, x_out, qkv, ao, lse, ln_tmp, gelu_tmp) = _fwd_setup(blk, x, cu_seqlens,
                                                                                                    seqlens)
        dgelu = torch.empty(T, blk.mlp.fc1.out_features, device=x.device, dtype=torch.float16)
        args = (ctypes.addressof(nat), ptr(x_in), ptr(x_mid), ptr(x_out), ptr(ln_tmp), ptr(qkv), ptr(ao), ptr(lse),
                ptr(dgelu), ptr(gelu_tmp), ptr(cu_seqlens), num_seqs, max_len, T)
        if scales is None:
            LIB.call("apla_block_fwd", *args, stream())
        else:
            LIB.call("apla_block_fwd_scaled", *args, ptr(scales), T // x.shape[0], stream())
        ctx.blk, ctx.nat, ctx.refs = blk, nat, blk._nat_refs      # the struct points into these tensors
        blk._dyb_stash = None                                     # (see backward: nothing survives from the last step)
        ctx.geom = (num_seqs, max_len, cu_seqlens)
        ctx.x_dtype, ctx.x_shape = x.dtype, x.shape
        ctx.save_for_backward(x_in, x_mid, qkv, ao, lse, dgelu, scales)
        return x_out.view(x.shape).to(x.dtype)

    @staticmethod
    def backward(ctx, dy):
        blk, nat = ctx.blk, ctx.nat
        at = blk.attn
        x_in, x_mid, qkv, ao, lse, dgelu, scales = ctx.saved_tensors
        num_seqs, max_len, cu = ctx.geom
        D, H, Hd, r = at.dim, at.num_heads, blk.mlp.fc1.out_features, at.partial_size
        want_w = ctx.needs_input_grad[1] or ctx.needs_input_grad[2]
        want_x = ctx.needs_input_grad[0]
        dx_out = dy.reshape(-1, D).to(torch.float32).contiguous()
        T = dx_out.shape[0]
        dev, bf, f32 = dy.device, torch.bfloat16, torch.float32
        dx_mid = torch.empty(T, D, device=dev, dtype=f32)        # the input gradient lands in the same buffer
        # Chained blocks (fuse_apla_blocks links each fused block to the one in front of it): the first thing a block's
        # backward needs is bf16(gamma2 * dy), a 6-byte-per-element pass over the gradient the block behind it has just
        # written.  That block writes it from its last LayerNorm backward instead and leaves it here -- accepted only if
        # `dy` IS that gradient, untouched: same storage, same version counter (autograd accumulating a second consumer's
        # gradient into it, in place or not, changes one of the two).
        # With drop path, a block needs bf16(s1 * gamma2 * dy), whose per-image scale s1 the block behind it cannot know:
        # it forms that itself (a row-scaled cast), and the block behind writes no hand-over for it.
        stash, blk._dyb_stash = getattr(blk, "_dyb_stash", None), None
        dyb_ready = int(scales is None and stash is not None and stash[0] == dx_out.data_ptr()
                        and stash[1] == dx_out._version and stash[2] == T and stash[3].device == dev)
        dyb = stash[3] if dyb_ready else torch.empty(T, D, device=dev, dtype=bf)
        front = blk._front_ref() if getattr(blk, "_front_ref", None) is not None else None
        chain = bool(want_x and front is not None and _CHAIN and front.attn.dim == D and not front._drop_path_active())
        dyb_front = torch.empty(T, D, device=dev, dtype=bf) if chain else None
        g_front = front._mlp_working_set(dev)["g2"] if chain else None
        dh = torch.empty(T, Hd, device=dev, dtype=bf)
        dln = torch.empty(T, D, device=dev, dtype=bf)
        dsub = torch.empty(T, nat.r_pad, device=dev, dtype=bf) if (want_w and not nat.rowmap) else None
        d_ao = delta = dqkv = dw1 = db1 = None
        if want_x:
            d_ao = torch.empty(T, D, device=dev, dtype=bf)
            delta = torch.empty(T, H, device=dev, dtype=f32)
            dqkv = torch.empty(T, 3 * D, device=dev, dtype=bf)
        if want_w:
            dw1 = torch.empty(r, D, device=dev, dtype=f32)       # zeroed by the library
            db1 = torch.empty(r, device=dev, dtype=f32)
        args = (ctypes.addressof(nat), ptr(dx_out), ptr(x_in), ptr(x_mid), ptr(qkv), ptr(ao), ptr(lse), ptr(dgelu),
                ptr(dx_mid), ptr(dx_mid) if want_x else None, ptr(dyb), ptr(dh), ptr(dln), ptr(dsub), ptr(d_ao), ptr(delta),
                ptr(dqkv), ptr(dw1), ptr(db1), ptr(cu), num_seqs, max_len, T, dyb_ready, ptr(dyb_front), ptr(g_front))
        if scales is None:
            LIB.call("apla_block_bwd", *args, stream())
        else:
            LIB.call("apla_block_bwd_scaled", *args, ptr(scales), T // ctx.x_shape[0], stream())
        dx = dx_mid.view(ctx.x_shape).to(ctx.x_dtype) if want_x else None
        if chain and dx.data_ptr() == dx_mid.data_ptr():
            front._dyb_stash = (dx_mid.data_ptr(), dx._version, T, dyb_front)
        return dx, dw1, db1, None, None, None, None


def _gamma_of(ls) -> Optional[torch.Tensor]:
    """LayerScale's per-channel vector (vit.py:236-244; dinov2/layers/layer_scale.py:15-27), None for nn.Identity."""
    if ls is None or isinstance(ls, nn.Identity):
        return None
    g = getattr(ls, "gamma", None)
    if g is None:
        raise TypeError(f"cannot fuse a block whose ls module is {type(ls).__name__} (expected LayerScale or Identity)")
    return g


def _drop_rate(mod) -> float:
    if mod is None or isinstance(mod, nn.Identity):
        return 0.0
    return float(getattr(mod, "drop_prob", None) or getattr(mod, "p", 0.0) or 0.0)


class FusedAplaBlock(nn.Module):
    """Holds the wrapped block's sub-modules under their own names; only `forward` is replaced."""

    # set by `attention_probabilities(model)`: forward(x, return_attention=True) returns the attention probabilities
    _attention_probs = False

    def __init__(self, block: nn.Module):
        super().__init__()
        if not isinstance(block.attn, APLA_Attention):
            raise TypeError("FusedAplaBlock needs a block whose .attn is an apla_b200 APLA_Attention "
                            "(run build_apla / replace_attn_with_apla first)")
        fc1, fc2 = block.mlp.fc1, block.mlp.fc2
        act = getattr(block.mlp, "act", None)
        if act is not None and not (isinstance(act, nn.GELU) and getattr(act, "approximate", "none") == "none"):
            raise TypeError("the fused MLP implements exact (erf) GELU only (vit.py:153)")
        if fc1.in_features % 64 or fc1.out_features % 64 or fc2.out_features != fc1.in_features:
            raise ValueError("fused block needs embed and hidden sizes that are multiples of 64")
        for name, child in block.named_children():       # norm1, attn, ls1, drop_path*, norm2, mlp, ls2 -- same keys
            self.add_module(name, child)
        for opt in ("ls1", "ls2"):
            if not hasattr(self, opt):
                self.add_module(opt, nn.Identity())
        self.sample_drop_ratio = float(getattr(block, "sample_drop_ratio", 0.0) or 0.0)
        self._ms = None
        self._ms_key = None

    # ---- bf16 working copies of the frozen MLP / norm / LayerScale tensors -----------------------------------------
    def refresh_working_set(self):
        """Drop the cached copies of this block's frozen MLP / norm / LayerScale tensors and of its attention
        (`APLA_Attention.refresh_working_set` explains when that is needed)."""
        self._ms = None
        self._ms_key = None
        if hasattr(self.attn, "refresh_working_set"):
            self.attn.refresh_working_set()

    def _mlp_working_set(self, device):
        tk = APLA_Attention._tkey
        g1, g2 = _gamma_of(self.ls1), _gamma_of(self.ls2)
        srcs = [self.mlp.fc1.weight, self.mlp.fc1.bias, self.mlp.fc2.weight, self.mlp.fc2.bias, self.norm1.weight,
                self.norm1.bias, self.norm2.weight, self.norm2.bias, g1, g2]
        key = tuple(None if t is None else tk(t) for t in srcs)
        if self._ms is None or self._ms_key != key:
            bf, f32 = torch.bfloat16, torch.float32

            def dev(t, dt):
                return None if t is None else t.detach().to(device=device, dtype=dt).contiguous()

            with torch.no_grad():
                w1, w2 = dev(self.mlp.fc1.weight, bf), dev(self.mlp.fc2.weight, bf)
                zeros = lambda n: torch.zeros(n, device=device, dtype=f32)          # noqa: E731
                self._ms = dict(
                    wfc1=w1, wfc1T=w1.t().contiguous(), wfc2=w2, wfc2T=w2.t().contiguous(),
                    bfc1=dev(self.mlp.fc1.bias, f32) if self.mlp.fc1.bias is not None else zeros(w1.shape[0]),
                    bfc2=dev(self.mlp.fc2.bias, f32) if self.mlp.fc2.bias is not None else zeros(w2.shape[0]),
                    ln1w=dev(self.norm1.weight, f32), ln1b=dev(self.norm1.bias, f32),
                    ln2w=dev(self.norm2.weight, f32), ln2b=dev(self.norm2.bias, f32), g1=dev(g1, f32), g2=dev(g2, f32))
            self._ms_key = key
        return self._ms

    def _native(self, device) -> BlockWeights:
        """The `apla_block_weights` struct over the two working sets (rebuilt only when one of them was)."""
        at = self.attn
        ws = at._working_set(device)          # also re-scatters proj_weight1 / proj_bias1 when they changed
        ms = self._mlp_working_set(device)
        key = (id(ws), id(ms))
        if getattr(self, "_nat_key", None) != key:
            r = at.partial_size
            fields = dict(ws)
            fields.update(ms)
            nat = BlockWeights()
            for name in ("wqkv", "wqkvT", "wproj", "wprojT", "wfc1", "wfc1T", "wfc2", "wfc2T", "bqkv", "bproj", "bfc1",
                         "bfc2", "ln1w", "ln1b", "ln2w", "ln2b", "g1", "g2", "rowmap"):
                setattr(nat, name, ptr(fields[name]))
            nat.idx = ptr(ws["idx"]) if ws["rowmap"] is None else None
            nat.D, nat.H, nat.hidden, nat.r, nat.r_pad = at.dim, at.num_heads, self.mlp.fc1.out_features, r, _pad64(r)
            nat.eps1, nat.eps2, nat.scale = float(self.norm1.eps), float(self.norm2.eps), float(at.scale)
            self._nat, self._nat_key, self._nat_refs = nat, key, (ws, ms)
        return self._nat

    def _drop_path_modules(self):
        """The (attention, MLP) branch's drop-path module: timm's / DINOv2's `drop_path1` / `drop_path2`, else the one
        `drop_path` the reference's Block calls for both branches (vit.py); None where the block has none."""
        one = getattr(self, "drop_path", None)
        return getattr(self, "drop_path1", one), getattr(self, "drop_path2", one)

    def _drop_path_active(self) -> bool:
        return self.training and any(_drop_rate(m) > 0 for m in self._drop_path_modules())

    def _branch_scales(self, x) -> Optional[torch.Tensor]:
        """fp32 [2, B] per-image scales of the attention (row 0) and MLP (row 1) branch, or None when nothing is drawn
        (eval mode, rate 0, nn.Identity).  Each comes from the branch's own drop-path module applied to ones(B, 1, 1) in
        the dtype of the reference's branch output, attention branch first: the CUDA generator advances exactly as in the
        unfused block, so the same seed gives the same masks whatever the DropPath implementation."""
        if not self._drop_path_active():
            return None
        # dtypes of the branch outputs the reference drops: attn(norm1(x)) has x's dtype, the MLP's Linear output
        # autocast's when it is on; LayerScale's gamma promotes either
        g1, g2 = _gamma_of(self.ls1), _gamma_of(self.ls2)
        dt_attn = x.dtype if g1 is None else torch.promote_types(x.dtype, g1.dtype)
        dt_mlp = torch.get_autocast_dtype("cuda") if torch.is_autocast_enabled("cuda") else torch.promote_types(x.dtype,
                                                                                                                 dt_attn)
        dt_mlp = dt_mlp if g2 is None else torch.promote_types(dt_mlp, g2.dtype)
        B = x.shape[0]
        rows = []
        for mod, dt in zip(self._drop_path_modules(), (dt_attn, dt_mlp)):
            ones = torch.ones(B, 1, 1, device=x.device, dtype=dt)
            rows.append((mod(ones) if _drop_rate(mod) > 0 else ones).reshape(B).to(torch.float32))
        return torch.stack(rows)

    def _check(self, x, crops: bool = False):
        if self.training:
            at = self.attn
            drops = {"attn.attn_drop": at.attn_drop.p, "attn.proj_drop": at.proj_drop.p,
                     "mlp.drop": _drop_rate(getattr(self.mlp, "drop", None))}
            bad = [f"{k}={p}" for k, p in drops.items() if p > 0]
            if bad:
                raise RuntimeError(f"fused APLA block supports dropout rate 0 only (got {', '.join(bad)}; all shipped "
                                   "reference configs use 0)")
            if self.sample_drop_ratio > 0.1:
                raise RuntimeError(f"fused APLA block: sample_drop_ratio={self.sample_drop_ratio} > 0.1 selects DINOv2's "
                                   "batch-subset stochastic depth, which is not supported (per-image drop path is)")
            if crops and self._drop_path_active():
                raise RuntimeError("fused APLA block: drop path on a list of crops (DINOv2's batch-subset stochastic depth "
                                   "of forward_nested) is not supported; drop path runs on dense [B, N, D] input only")
            if self.attn.dim % 128 and self._drop_path_active():
                raise RuntimeError(f"fused APLA block: drop path needs an embedding width that is a multiple of 128 (the "
                                   f"row-scaled LayerNorm backward), got {self.attn.dim}; set the drop-path rate to 0")
        if not x.is_cuda:
            raise RuntimeError("apla_b200.FusedAplaBlock runs on CUDA (sm_100a) only; there is no CPU fallback")
        require_device()
        for p in (self.norm1.weight, self.norm2.weight, self.mlp.fc1.weight, self.mlp.fc2.weight):
            if p.requires_grad:
                raise RuntimeError("fused APLA block computes weight gradients for proj_weight1 / proj_bias1 only; "
                                   "norm / MLP parameters must be frozen (build_apla's freeze policy)")

    def _run_fused(self, x, cu=None, seqlens=None, scales=None):
        at = self.attn
        if not torch.is_grad_enabled() or not (x.requires_grad or at.proj_weight1.requires_grad
                                                or at.proj_bias1.requires_grad):
            return self._run_infer(x, cu, seqlens, scales)      # autograd would record nothing: keep nothing for backward
        return _AplaBlockFn.apply(x, at.proj_weight1, at.proj_bias1, self, cu, seqlens, scales)

    def _run_infer(self, x, cu, seqlens, scales=None):
        """`apla_block_fwd_infer`: the forward of _AplaBlockFn, bit for bit, without its saved tensors (lse is scratch,
        fc1 writes no GELU derivative).  x_out is a buffer of its own: x_in may be the caller's tensor.  A training-mode
        block drops branches here too (`scales`), as the reference's Block does under torch.no_grad()."""
        nat, x_in, T, num_seqs, max_len, (x_mid, x_out, qkv, ao, lse, ln_tmp, gelu_tmp) = _fwd_setup(self, x, cu, seqlens)
        args = (ctypes.addressof(nat), ptr(x_in), ptr(x_mid), ptr(x_out), ptr(ln_tmp), ptr(qkv), ptr(ao), ptr(lse),
                ptr(gelu_tmp), ptr(cu), num_seqs, max_len, T)
        if scales is None:
            LIB.call("apla_block_fwd_infer", *args, stream())
        else:
            LIB.call("apla_block_fwd_infer_scaled", *args, ptr(scales), T // x.shape[0], stream())
        return x_out.view(x.shape).to(x.dtype)

    def _attention(self, x):
        """The reference Block's `return_attention=True` result (vit.py:282-283): LayerNorm 1, the qkv GEMM, the attention
        forward for its log-sum-exp, then the fp32 [B,H,N,N] probabilities; the rest of the block is not run."""
        at = self.attn
        B, N, D = x.shape
        ws, ms = at._working_set(x.device), self._mlp_working_set(x.device)
        x_in = x.detach().reshape(-1, D).to(torch.float32).contiguous()
        ln = ops.layernorm_fwd(x_in, ms["ln1w"], ms["ln1b"], float(self.norm1.eps))
        qkv = ops.gemm_bias(ln, ws["wqkv"], ws["bqkv"])
        _, lse = ops.attn_fwd(qkv, at.num_heads, float(at.scale), B, N)
        return ops.attn_probs(qkv, lse, at.num_heads, float(at.scale), B, N)

    def forward(self, x_or_x_list, return_attention: bool = False, return_intermediate: bool = False):
        """`[B,N,D]` -> `[B,N,D]` (vit.py:279-288) or list of `[b_i,N_i,D]` -> list (dinov2 block.py:274-288).
        Inside `attention_probabilities(model)`, `forward(x, return_attention=True)` on a `[B,N,D]` tensor returns the
        fp32 [B,H,N,N] attention probabilities of the block (no autograd history), as the reference Block does."""
        if return_intermediate or (return_attention and not self._attention_probs):
            raise RuntimeError("the fused block does not materialise the [B,H,N,N] attention probabilities "
                               "(vit.py:282-287 visualisation paths) unless it runs inside "
                               "apla_b200.apla.attention_probabilities(model); return_intermediate is not supported")
        if return_attention:
            if not isinstance(x_or_x_list, torch.Tensor) or x_or_x_list.dim() != 3:
                raise RuntimeError("attention probabilities need a dense [B, N, D] tensor, not a list of crops")
            self._check(x_or_x_list)
            return self._attention(x_or_x_list)
        if isinstance(x_or_x_list, torch.Tensor):
            self._check(x_or_x_list)
            return self._run_fused(x_or_x_list, scales=self._branch_scales(x_or_x_list))
        xs: Sequence[torch.Tensor] = list(x_or_x_list)
        if not xs:
            raise AssertionError("empty crop list")
        self._check(xs[0], crops=True)
        D = xs[0].shape[-1]
        seqlens: List[int] = []
        for t in xs:
            seqlens += [t.shape[1]] * t.shape[0]
        # The crops a previous fused block returned are consecutive views of ITS packed output: take that tensor instead of
        # copying them together again (one 240 MB torch.cat per block and direction at the C4 shape: 4 ms of a 149 ms step)
        packed = x_or_x_list.packed_if_untouched() if isinstance(x_or_x_list, PackedCropList) else None
        if packed is None:
            packed = torch.cat([t.reshape(1, -1, D) for t in xs], dim=1)                 # [1, sum b_i*N_i, D]
        out = self._run_fused(packed, _cu_seqlens(tuple(seqlens), packed.device), seqlens)
        sizes = [t.shape[0] * t.shape[1] for t in xs]
        return PackedCropList([o.reshape(t.shape) for o, t in zip(out.split(sizes, dim=1), xs)], out)


class PackedCropList(list):
    """The list of crop tensors a fused block returns (what dinov2's NestedTensorBlock returns, block.py:274-288) that also
    remembers the packed `[1, T, D]` tensor its elements are views of.  The next fused block takes that tensor -- with its
    autograd history -- instead of concatenating the views again, as long as the list is handed on unchanged."""

    def __init__(self, views, packed):
        super().__init__(views)
        self._views = tuple(views)
        self._packed = packed

    def packed_if_untouched(self) -> Optional[torch.Tensor]:
        if len(self) != len(self._views) or any(a is not b for a, b in zip(self, self._views)):
            return None
        return self._packed


@contextlib.contextmanager
def attention_probabilities(model: nn.Module):
    """Within the block, every `APLA_Attention` of `model` returns `(out, attn)` with `attn` the fp32 [B,H,N,N]
    attention probabilities (dense inputs; no autograd history), and every `FusedAplaBlock` answers
    `forward(x, return_attention=True)` with them, as the reference's modules do (appla_attn.py:83, vit.py:282-287).
    The previous settings are restored on exit, also on an exception and when blocks nest.  Outside it nothing
    changes: the probabilities are never computed."""
    mods = [m for m in model.modules() if isinstance(m, (APLA_Attention, FusedAplaBlock))]
    saved = [m.__dict__.get("_attention_probs") for m in mods]
    try:
        for m in mods:
            m._attention_probs = True
        yield model
    finally:
        for m, v in zip(mods, saved):
            if v is None:
                m.__dict__.pop("_attention_probs", None)
            else:
                m._attention_probs = v


_CU_CACHE = {}


def _cu_seqlens(seqlens: tuple, device) -> torch.Tensor:
    """int32 prefix sums of the sequence lengths on `device`, cached: the crop geometry repeats every block and step."""
    key = (seqlens, str(device))
    cu = _CU_CACHE.get(key)
    if cu is None:
        if len(_CU_CACHE) > 64:
            _CU_CACHE.clear()
        host = torch.zeros(len(seqlens) + 1, dtype=torch.int32)
        host[1:] = torch.tensor(seqlens, dtype=torch.int32).cumsum(0)
        cu = _CU_CACHE[key] = host.to(device)
    return cu


def fuse_apla_blocks(model: nn.Module) -> nn.Module:
    """Swap every block of `model.blocks` (a backbone, or a Classifier's `.backbone`) that carries an `APLA_Attention`
    for a `FusedAplaBlock` in place.  Parameters, buffers and state-dict keys are untouched.  Returns `model`."""
    bb = model if hasattr(model, "blocks") else getattr(model, "backbone", None)
    if bb is None or not hasattr(bb, "blocks"):
        raise AttributeError("model exposes no .blocks (SURVEY.md 8b: what the host model must expose)")
    n = 0
    for i, blk in enumerate(bb.blocks):
        if isinstance(blk, FusedAplaBlock):
            continue
        if isinstance(getattr(blk, "attn", None), APLA_Attention):
            bb.blocks[i] = FusedAplaBlock(blk)
            n += 1
    # each fused block learns which fused block is in front of it (a weak reference outside the module tree: state-dict
    # keys and `.modules()` stay as they were); see _AplaBlockFn.backward
    prev = None
    for blk in bb.blocks:
        if isinstance(blk, FusedAplaBlock):
            object.__setattr__(blk, "_front_ref", weakref.ref(prev) if prev is not None else None)
            prev = blk
        else:
            prev = None
    if n == 0 and not any(isinstance(b, FusedAplaBlock) for b in bb.blocks):
        raise RuntimeError("no block carries an APLA_Attention: call build_apla(config, model, attn_class) first "
                           "(multi-GPU partial_size='full' keeps the stock attention and cannot be fused)")
    return model

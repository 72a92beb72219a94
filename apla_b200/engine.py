"""`FineTuneEngine`: host side of the native step engine (csrc/engine.cu).

Takes a classifier built the reference way (`Classifier`: backbone ViT with APLA attention + `fc` head,
src/defaults/models.py:24-92; here usually `hostvit.HostClassifier`), lays its tensors out for the B200 and runs
`Trainer.global_step` (src/defaults/trainer.py:106-138) -- forward, the criterion (CrossEntropy, or BCE-with-logits for
multi-label tasks), backward restricted to the APLA rows and the head, data-parallel gradient mean,
clip_grad_norm_(1.0), AdamW -- as native kernel launches.

PyTorch's role here is plumbing only: device allocation (torch tensors own every buffer), the one-time conversion
of frozen fp32 weights into bf16 [out,in] / [in,out] copies, stream handles and torch.distributed/NCCL for the
gradient all-reduce.  All step arithmetic is in libapla_b200.so; nothing falls back to torch ops.

Memory layout in HBM (T = B*N tokens, D embed, L blocks), sized for B=64 ViT-B/14 (~5 GB of 180 GB):
  xs        fp32 [2L+1, T, D]   residual-stream checkpoints (block input / after attention / ... / final)
  qkv[l]    bf16 [T, 3D]  ao[l] bf16 [T, D]  lse[l] fp32 [T, H]  hpre[l] fp16 [T, 4D] (gelu' of the fc1 pre-activation)   saved for backward
  ln_out, gelu_out, dx, dxb, dO, dqkv, dsub, delta                                         transients, reused
  params / grads / exp_avg / exp_avg_sq   fp32 arenas [W1 x L | fc.weight | b1 x L | fc.bias]  (one all-reduce)
  drop_path fp32 [L, 2, B]  stochastic-depth scales of the attention / MLP branch per image (only with a rate > 0)
  infer_*   evaluation workspace of predict / embed / evaluate (eval_batch_size images, allocated on first use): two fp32
            [T_eval, D] residual buffers and one block's transients -- no checkpoints, nothing kept for backward
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Tuple

import os

import torch
import torch.nn as nn

from ._lib import LIB, ptr, require_device, stream
from .apla.apla_block import _drop_rate as _rate

BF16, F32 = torch.bfloat16, torch.float32


def _pad64(n: int) -> int:
    return (n + 63) // 64 * 64


def criterion_code(criterion) -> int:
    """The engine's "criterion" option for the loss a reference trainer built (`DefaultWrapper`, wrappers.py:310-320):
    None or a default nn.CrossEntropyLoss -> 0, an nn.BCEWithLogitsLoss with reduction="mean" and neither weight nor
    pos_weight -> 1.  Anything else is refused with a ValueError, so that a step never trains another objective."""
    supported = ("supported: None or nn.CrossEntropyLoss() (multi-class), nn.BCEWithLogitsLoss() (multi-label), both "
                 "with default arguments")
    if criterion is None:
        return 0
    if type(criterion) is nn.CrossEntropyLoss:
        if criterion.label_smoothing > 0:
            raise ValueError(f"CrossEntropyLoss(label_smoothing={criterion.label_smoothing}) is not supported: pass "
                             "smoothed fp32 [n, C] targets to step() instead (what timm's Mixup / label smoothing yields); "
                             + supported)
        if criterion.reduction != "mean" or criterion.weight is not None or criterion.ignore_index != -100:
            raise ValueError(f"CrossEntropyLoss(reduction={criterion.reduction!r}, weight="
                             f"{'set' if criterion.weight is not None else None}, ignore_index={criterion.ignore_index}) "
                             "is not supported; " + supported)
        return 0
    if type(criterion) is nn.BCEWithLogitsLoss:
        if criterion.reduction != "mean" or criterion.weight is not None or criterion.pos_weight is not None:
            raise ValueError(f"BCEWithLogitsLoss(reduction={criterion.reduction!r}, weight="
                             f"{'set' if criterion.weight is not None else None}, pos_weight="
                             f"{'set' if criterion.pos_weight is not None else None}) is not supported; " + supported)
        return 1
    raise ValueError(f"criterion {type(criterion).__name__} is not supported; " + supported)


def drop_path_rates(model) -> List[Tuple[float, float]]:
    """The stochastic-depth rates (p_attn, p_mlp) of every block of `model.backbone`: `blk.drop_path.drop_prob` for both
    branches (the reference's Block, vit.py), or timm's `drop_path1` / `drop_path2`; nn.Identity is rate 0.  The engine
    draws the masks itself (one per image, branch and step).  Raises ValueError for what it cannot honour: dropout
    anywhere (`attn.attn_drop`, `attn.proj_drop`, `mlp.drop`, `backbone.pos_drop` -- it would need RNG inside the kernels),
    DropPath(scale_by_keep=False), DINOv2's batch-subset stochastic depth (sample_drop_ratio > 0.1) and rates >= 1."""
    bb = model.backbone

    def no_dropout(name, mod):
        p = _rate(mod)
        if p > 0:
            raise ValueError(f"{name} has dropout rate {p}: the step engine cannot honour dropout (--dr / --adr); set it to "
                             "0 (stochastic depth, drop_path_rate / --dpr, is supported)")

    no_dropout("backbone.pos_drop", getattr(bb, "pos_drop", None))
    rates = []
    for l, blk in enumerate(bb.blocks):
        pre = f"backbone.blocks.{l}."
        no_dropout(pre + "attn.attn_drop", getattr(blk.attn, "attn_drop", None))
        no_dropout(pre + "attn.proj_drop", getattr(blk.attn, "proj_drop", None))
        for name in ("drop", "drop1", "drop2"):
            no_dropout(pre + "mlp." + name, getattr(blk.mlp, name, None))
        if float(getattr(blk, "sample_drop_ratio", 0.0) or 0.0) > 0.1:
            raise ValueError(f"{pre[:-1]}: sample_drop_ratio > 0.1 selects DINOv2's batch-subset stochastic depth, which "
                             "the step engine cannot honour")
        if hasattr(blk, "drop_path1") or hasattr(blk, "drop_path2"):
            mods = (getattr(blk, "drop_path1", None), getattr(blk, "drop_path2", None))
        else:
            mods = (getattr(blk, "drop_path", None),) * 2
        for m in mods:
            if getattr(m, "scale_by_keep", True) is False:
                raise ValueError(f"{pre[:-1]}: DropPath(scale_by_keep=False) is not supported; the engine scales the kept "
                                 "samples by 1 / keep as the reference's drop_path does")
        pair = (_rate(mods[0]), _rate(mods[1]))
        if not all(0.0 <= p < 1.0 for p in pair):
            raise ValueError(f"{pre[:-1]}: drop-path rates {pair} outside [0, 1)")
        rates.append(pair)
    return rates


def interpolate_pos_table(pos_embed: torch.Tensor, npatch: int) -> torch.Tensor:
    """Bicubic resize of a [1, 1+n0, D] position table to an npatch grid (vit.py:421-437); done ONCE at engine
    construction because pos_embed is frozen (the reference recomputes it every forward, SURVEY.md K21)."""
    n0 = pos_embed.shape[1] - 1
    if npatch == n0:
        return pos_embed[0]
    D = pos_embed.shape[-1]
    s = int(math.sqrt(n0))
    grid = pos_embed[:, 1:].reshape(1, s, s, D).permute(0, 3, 1, 2)
    grid = nn.functional.interpolate(grid, scale_factor=math.sqrt(npatch / n0), mode="bicubic", align_corners=False,
                                     recompute_scale_factor=False)
    return torch.cat((pos_embed[:, :1], grid.permute(0, 2, 3, 1).reshape(1, -1, D)), dim=1)[0]


class FineTuneEngine:
    def __init__(self, model: nn.Module, batch_size: int, img_size: int, device="cuda", lr: float = 3e-5,
                 weight_decay: float = 1e-5, clip: float = 1.0, betas=(0.9, 0.999), adam_eps: float = 1e-8,
                 process_group=None, cls_only_last_block: bool = True, use_graph: bool = True,
                 eval_batch_size: Optional[int] = None, criterion=None):
        # the trainer's loss (`criterion=self.criterion`): 0 = cross-entropy, 1 = BCE-with-logits (multi-label)
        self.criterion = criterion_code(criterion)
        # stochastic depth per block and branch (the reference's --dpr); models with dropout are refused here
        self.drop_path = drop_path_rates(model)
        require_device()
        # Only norm(x)[:, 0] of the last block reaches the head (vit.py:417-419): its projection, LayerNorm 2, MLP and
        # their input gradients run on the CLS rows only.  False = every token (identical results, for A/B checks).
        self.cls_only_last_block = 2 if cls_only_last_block is True else int(cls_only_last_block)   # 1: tail only
        self.device = torch.device(device)
        self.model = model
        self.lr, self.wd, self.clip, self.betas, self.adam_eps = lr, weight_decay, clip, betas, adam_eps
        self.pg = process_group
        self.world = torch.distributed.get_world_size(process_group) if self._dist_on() else 1
        self.step_count = 0
        # One CUDA graph per (images, labels) buffer pair replays the step's ~200 launches (single GPU only: with a
        # process group the all-reduce runs on a side stream between two backward ranges).  lr and Adam's bias
        # corrections reach the captured AdamW kernel through a 3-float device buffer refreshed before every replay.
        # With a process group the step is three graphs (forward + upper backward | lower backward | optimiser) with the
        # two gradient all-reduces launched eagerly between them on the side stream: capturing the NCCL collectives
        # themselves hung on this stack (torch 2.11 / NCCL 2.28), and they are two launches anyway.
        self.use_graph = bool(use_graph)
        self._graphs: Dict[tuple, object] = {}
        self._graph_seen: Dict[tuple, int] = {}
        self._keep: List[torch.Tensor] = []          # every device buffer the engine points at
        self._handle = None
        self.buffers: Dict[tuple, Optional[torch.Tensor]] = {}
        # predict / embed / evaluate run up to this many images per native call over a workspace of their own, allocated
        # on first use (about 5 MB per image at ViT-B/14, 518 px, against about 78 MB for the training step)
        self.eval_batch_size = int(eval_batch_size) if eval_batch_size is not None else int(batch_size)
        if self.eval_batch_size < 1:
            raise ValueError("eval_batch_size must be >= 1")
        self._infer_ws: Optional[Dict[str, torch.Tensor]] = None
        # the drop-path masks of every training forward come from this generator, on the host; seeded per rank so that
        # ranks drop different images, as the reference's per-process RNG does
        rank = torch.distributed.get_rank(process_group) if self._dist_on() else 0
        self._dp_gen = torch.Generator().manual_seed((torch.initial_seed() + 1_000_003 * rank) % 2 ** 63)
        self._dp_dev: Optional[torch.Tensor] = None
        # CPU fp32 [L, 2, n]: the scales (0 or 1 / keep) the last training forward applied; None when every rate is 0
        self.last_drop_path_scales: Optional[torch.Tensor] = None
        self._build(model, batch_size, img_size)

    # ------------------------------------------------------------------------------------------------------------
    def _dist_on(self) -> bool:
        return torch.distributed.is_available() and torch.distributed.is_initialized()

    def _dev(self, t: torch.Tensor, dtype) -> torch.Tensor:
        out = t.detach().to(device=self.device, dtype=dtype).contiguous()
        self._keep.append(out)
        return out

    def _new(self, *shape, dtype=BF16, zero=False) -> torch.Tensor:
        t = (torch.zeros if zero else torch.empty)(*shape, dtype=dtype, device=self.device)
        self._keep.append(t)
        return t

    def _set(self, name: str, t: Optional[torch.Tensor], block: int = -1):
        LIB.call("apla_engine_set_ptr", self._handle, name.encode(), block, ptr(t))
        self.buffers[(name, block)] = t       # what the native engine points at, by name (block -1: global)

    def _build(self, model, B, img):
        bb = model.backbone
        conv = bb.patch_embed.proj
        patch = conv.kernel_size[0]
        D = bb.cls_token.shape[-1]
        L = len(bb.blocks)
        P = (img // patch) ** 2
        N = P + 1
        T = B * N
        blk0 = bb.blocks[0]
        H = blk0.attn.num_heads
        hidden = blk0.mlp.fc1.out_features
        C = model.fc.out_features
        kpad = (3 * patch * patch + 63) // 64 * 64
        self.stock_proj = hasattr(blk0.attn, "proj")            # multi-GPU 'full': stock attention, proj trainable
        r = D if self.stock_proj else int(blk0.attn.partial_size)
        full_rows = 1 if r > 128 else 0
        r_pad = _pad64(r)
        self.shape = dict(B=B, N=N, D=D, H=H, L=L, hidden=hidden, C=C, P=P, patch=patch, img=img, kpad=kpad, r=r,
                          r_pad=r_pad, full_rows=full_rows, T=T)
        eps = float(blk0.norm1.eps)
        scale = float(blk0.attn.scale)
        self._handle = LIB.load().apla_engine_create(B, N, D, H, L, hidden, C, patch, img, kpad, r, r_pad, full_rows,
                                                     eps, scale)
        if not self._handle:
            raise RuntimeError("apla_engine_create failed: " + LIB.last_error())
        LIB.call("apla_engine_set_option", self._handle, b"cls_only_last_block", int(self.cls_only_last_block))
        LIB.call("apla_engine_set_option", self._handle, b"criterion", self.criterion)
        # measured: no gain on C2 (7.94 vs 7.98 ms), +0.4 % on C3 -- the step runs into the power cap, not into idle SMs;
        # kept as an option (APLA_SIDE_WGRAD=1), off by default
        self.side_wgrad = os.environ.get("APLA_SIDE_WGRAD", "0") != "0"

        # ---- embedding ----
        wpe = torch.zeros(D, kpad, dtype=F32)
        wpe[:, :3 * patch * patch] = conv.weight.detach().float().reshape(D, -1).cpu()
        self._set("wpe", self._dev(wpe, BF16))
        self._set("bpe", self._dev(conv.bias if conv.bias is not None else torch.zeros(D), F32))
        self._set("cls", self._dev(bb.cls_token.reshape(D), F32))
        self._set("pos", self._dev(interpolate_pos_table(bb.pos_embed.detach().float().cpu(), P), F32))
        self._set("patches", self._new(B * P, kpad))
        self._set("pe_out", self._new(B * P, D))

        # ---- trainable arena ----
        n = LIB.load().apla_engine_arena_size(self._handle)
        self.n_arena = int(n)
        self.params = self._new(n, dtype=F32, zero=True)
        # data parallel: the gradient arena lives in symmetric (peer-mapped) memory and is reduced by the library's own
        # kernel (apla_grad_arena_allreduce), which -- unlike an NCCL call -- is captured in the step's CUDA graph
        self._peer = None
        if self.world > 1:
            from .dp import make_peer_arena
            self._peer = make_peer_arena(n, self.device, self.pg)
            # every rank must take the same path: if symmetric memory failed anywhere, all ranks use NCCL
            ok = torch.tensor([1 if self._peer is not None else 0], device=self.device)
            torch.distributed.all_reduce(ok, op=torch.distributed.ReduceOp.MIN, group=self.pg)
            if int(ok.item()) == 0:
                self._peer = None
        if self._peer is not None:
            self.grads = self._peer.grads()
            self._keep.append(self._peer.buf)
        else:
            self.grads = self._new(n, dtype=F32, zero=True)
        self.exp_avg = self._new(n, dtype=F32, zero=True)
        self.exp_avg_sq = self._new(n, dtype=F32, zero=True)
        self.sumsq = self._new(600, dtype=F32, zero=True)      # APLA_SUMSQ_FLOATS: [0] = result, rest scratch
        o_w1, o_fcw = 0, L * r * D
        o_b1 = o_fcw + C * D
        o_fcb = o_b1 + L * r
        self.offsets = dict(w1=o_w1, fcw=o_fcw, b1=o_b1, fcb=o_fcb, n=o_fcb + C)
        assert self.offsets["n"] == n
        self.slices: Dict[str, slice] = {}     # parameter name -> slice of the arena
        self.shapes: Dict[str, tuple] = {}

        idx_all = torch.zeros(L, r, dtype=torch.int32)
        rowmap_all = torch.full((L, D), -1, dtype=torch.int32)
        # dense projection copies of all blocks back to back: refreshed by ONE kernel after every optimiser step
        self._wproj_all = self._new(L, D, D)
        self._wprojT_all = self._new(L, D, D)
        self._bproj_all = self._new(L, D, dtype=F32)
        # ---- blocks ----
        for l, blk in enumerate(bb.blocks):
            at = blk.attn
            pre = f"backbone.blocks.{l}."
            if self.stock_proj:
                inds = torch.arange(D)
                w_full = at.proj.weight.detach().float().cpu()
                b_full = at.proj.bias.detach().float().cpu()
                w1, b1 = w_full, b_full
                names = (pre + "attn.proj.weight", pre + "attn.proj.bias")
            else:
                inds = torch.as_tensor(at.indices).long().cpu()
                w1 = at.proj_weight1.detach().float().cpu()
                b1 = at.proj_bias1.detach().float().cpu()
                w_full = torch.zeros(D, D)
                b_full = torch.zeros(D)
                w_full[inds[:r]] = w1
                b_full[inds[:r]] = b1
                if r < D:
                    w_full[inds[r:]] = at.proj_weight2.detach().float().cpu()
                    b_full[inds[r:]] = at.proj_bias2.detach().float().cpu()
                names = (pre + "attn.proj_weight1", pre + "attn.proj_bias1")
            idx_all[l] = inds[:r].to(torch.int32)
            rowmap_all[l, inds[:r]] = torch.arange(r, dtype=torch.int32)
            self.slices[names[0]] = slice(o_w1 + l * r * D, o_w1 + (l + 1) * r * D)
            self.shapes[names[0]] = (r, D)
            self.slices[names[1]] = slice(o_b1 + l * r, o_b1 + (l + 1) * r)
            self.shapes[names[1]] = (r,)
            self.params[self.slices[names[0]]] = w1.reshape(-1).to(self.device)
            self.params[self.slices[names[1]]] = b1.to(self.device)

            def lin(mod):
                w = mod.weight.detach().float()
                b = mod.bias.detach().float() if mod.bias is not None else torch.zeros(w.shape[0])
                return self._dev(w, BF16), self._dev(w.t(), BF16), self._dev(b, F32)

            self._wproj_all[l].copy_(w_full.to(self.device))
            self._wprojT_all[l].copy_(w_full.t().to(self.device))
            self._bproj_all[l].copy_(b_full.to(self.device))
            wqkv, wqkvT, bqkv = lin(at.qkv)
            wfc1, wfc1T, bfc1 = lin(blk.mlp.fc1)
            wfc2, wfc2T, bfc2 = lin(blk.mlp.fc2)
            for k, v in dict(wqkv=wqkv, wqkvT=wqkvT, bqkv=bqkv, wfc1=wfc1, wfc1T=wfc1T, bfc1=bfc1, wfc2=wfc2,
                             wfc2T=wfc2T, bfc2=bfc2, wproj=self._wproj_all[l], wprojT=self._wprojT_all[l],
                             bproj=self._bproj_all[l], ln1w=self._dev(blk.norm1.weight, F32),
                             ln1b=self._dev(blk.norm1.bias, F32), ln2w=self._dev(blk.norm2.weight, F32),
                             ln2b=self._dev(blk.norm2.bias, F32)).items():
                self._set(k, v, l)
            g1 = getattr(blk.ls1, "gamma", None)
            g2 = getattr(blk.ls2, "gamma", None)
            self._set("g1", self._dev(g1, F32) if g1 is not None else None, l)
            self._set("g2", self._dev(g2, F32) if g2 is not None else None, l)
            self._set("qkv", self._new(T, 3 * D), l)
            self._set("ao", self._new(T, D, zero=True), l)   # last block: only its CLS rows are ever written
            self._set("hpre", self._new(T, hidden, dtype=torch.float16), l)
            self._set("lse", self._new(T, H, dtype=F32), l)

        # ---- head ----
        self.slices["fc.weight"] = slice(o_fcw, o_fcw + C * D)
        self.shapes["fc.weight"] = (C, D)
        self.slices["fc.bias"] = slice(o_fcb, o_fcb + C)
        self.shapes["fc.bias"] = (C,)
        self.params[self.slices["fc.weight"]] = model.fc.weight.detach().float().reshape(-1).to(self.device)
        self.params[self.slices["fc.bias"]] = model.fc.bias.detach().float().to(self.device)
        self._set("lnfw", self._dev(bb.norm.weight, F32))
        self._set("lnfb", self._dev(bb.norm.bias, F32))

        # ---- globals ----
        self.xs = self._new(2 * L + 1, T, D, dtype=F32)
        self.logits = self._new(B, C, dtype=F32)
        self.loss = self._new(1, dtype=F32, zero=True)
        self.idx = self._dev(idx_all, torch.int32)
        for name, t in dict(xs=self.xs, ln_out=self._new(T, D), gelu_out=self._new(T, hidden),
                            dx=self._new(T, D, dtype=F32), dxb=self._new(T, D), dO=self._new(T, D),
                            dqkv=self._new(T, 3 * D), delta=self._new(T, H, dtype=F32),
                            cls_ln=self._new(B, D), logits=self.logits, dlogits=self._new(B, C, dtype=F32),
                            loss=self.loss, dcls=self._new(B, D), params=self.params, grads=self.grads,
                            exp_avg=self.exp_avg, exp_avg_sq=self.exp_avg_sq, idx=self.idx, sumsq=self.sumsq).items():
            self._set(name, t)
        if full_rows:
            self._set("rowmap", self._dev(rowmap_all, torch.int32))
        else:
            self._set("dsub", self._new(2 if self.side_wgrad else 1, T, r_pad))
        # weight / bias gradients of a block on the engine's side stream beside the projection dgrad, the attention
        # backward and the qkv dgrad (csrc/engine.cu, Engine::side_wgrad) when APLA_SIDE_WGRAD=1
        LIB.call("apla_engine_set_option", self._handle, b"side_wgrad", (1 if full_rows else 2) if self.side_wgrad else 0)
        self._hyper_dev = self._new(3, dtype=F32, zero=True)
        if self.use_graph:
            self._set("hyper", self._hyper_dev)
        if any(p > 0 for pair in self.drop_path for p in pair):
            self._dp_keep = 1.0 - torch.tensor(self.drop_path, dtype=torch.float64)     # [L, 2]
            self._dp_dev = self._new(L, 2, B, dtype=F32)
            self._dp_dev.fill_(1.0)
            self._set("drop_path", self._dp_dev)
        self.images_dev = self._new(B, 3, img, img, dtype=F32)
        self.labels_dev = self._new(B, dtype=torch.int64)
        self._ar_stream = torch.cuda.Stream(device=self.device) if self.world > 1 else None
        torch.cuda.synchronize(self.device)

    def __del__(self):
        try:
            if self._handle:
                LIB.load().apla_engine_destroy(self._handle)
                self._handle = None
        except Exception:
            pass

    # ------------------------------------------------------------------------------------------------------------
    def trainable_names(self) -> List[str]:
        """Same order as the reference's named_parameters() filter (I5/I7 of SURVEY.md 4.2)."""
        L = self.shape["L"]
        w, b = ("attn.proj.weight", "attn.proj.bias") if self.stock_proj else ("attn.proj_weight1", "attn.proj_bias1")
        out = []
        for l in range(L):
            out += [f"backbone.blocks.{l}.{w}", f"backbone.blocks.{l}.{b}"]
        return out + ["fc.weight", "fc.bias"]

    def named_grads(self) -> Dict[str, torch.Tensor]:
        return {k: self.grads[self.slices[k]].view(self.shapes[k]) for k in self.trainable_names()}

    def named_params(self) -> Dict[str, torch.Tensor]:
        return {k: self.params[self.slices[k]].view(self.shapes[k]) for k in self.trainable_names()}

    def sync_to_model(self):
        """Write the arena's fp32 parameters back into the nn.Module (state_dict / checkpoint compatibility)."""
        sd = dict(self.model.named_parameters())
        with torch.no_grad():
            for k, v in self.named_params().items():
                sd[k].copy_(v.to(sd[k].device))

    # ---- checkpoint interchange with the reference (apla_b200/checkpoint.py, SURVEY.md 8f row f4) ---------------
    def _named_shapes(self):
        return [(k, self.shapes[k]) for k in self.trainable_names()]

    def state_dict(self):
        """The Classifier's CPU state dict with the engine's current trainable tensors written back
        (what bases.py:455-458 saves under 'state_dict')."""
        from .checkpoint import model_to_cpu_state
        torch.cuda.current_stream().synchronize()
        self.sync_to_model()
        return model_to_cpu_state(self.model)

    def optimizer_state_dict(self) -> dict:
        """`torch.optim.AdamW.state_dict()` of the reference's optimiser (two groups of wrappers.py:205-221) holding
        the engine's moments and step count."""
        from .checkpoint import optimizer_state_dict
        torch.cuda.current_stream().synchronize()
        m = {k: self.exp_avg[self.slices[k]] for k in self.trainable_names()}
        v = {k: self.exp_avg_sq[self.slices[k]] for k in self.trainable_names()}
        return optimizer_state_dict(self._named_shapes(), m, v, self.step_count, lr=self.lr, betas=self.betas,
                                    eps=self.adam_eps, weight_decay=self.wd)

    def load_state_dict(self, sd):
        """Take the TRAINABLE tensors of a reference state dict into the arena and refresh the dense projection copies.
        Frozen tensors are laid out (bf16, both orientations) when the engine is built, so they are only checked: a
        state dict whose APLA indices differ from the ones this engine was built with is refused."""
        bb = self.model.backbone
        for l, blk in enumerate(bb.blocks):
            k = f"backbone.blocks.{l}.attn.inds"
            if k in sd and hasattr(blk.attn, "inds") and not torch.equal(sd[k].cpu().long(), blk.attn.inds.cpu().long()):
                raise RuntimeError(f"{k} differs from the indices this engine was built with; load the checkpoint into "
                                   "the model (load_from_pretrained) before constructing the engine")
        missing = [k for k in self.trainable_names() if k not in sd]
        if missing:
            raise KeyError(f"state dict lacks trainable tensors: {missing[:4]}{' ...' if len(missing) > 4 else ''}")
        for k in self.trainable_names():
            t = sd[k]
            if tuple(t.shape) != tuple(self.shapes[k]):
                raise RuntimeError(f"{k}: checkpoint shape {tuple(t.shape)}, engine {tuple(self.shapes[k])}")
            self.params[self.slices[k]] = t.detach().to(self.device, F32).reshape(-1)
        self._refresh_proj()
        self.sync_to_model()

    def _refresh_proj(self):
        s = self.shape
        o = self.offsets
        LIB.call("apla_proj_refresh", self.params[o["w1"]:].data_ptr(), self.params[o["b1"]:].data_ptr(), ptr(self.idx),
                 ptr(self._wproj_all), ptr(self._wprojT_all), ptr(self._bproj_all), s["L"], s["r"], s["D"],
                 s["r"] * s["D"], s["r"], stream())

    def load_optimizer_state_dict(self, opt_sd: dict):
        """Adam moments, step count and hyper-parameters from a reference optimiser state dict (bases.py:423-428)."""
        from .checkpoint import split_optimizer_state
        m, v, step, hyper = split_optimizer_state(opt_sd, self._named_shapes())
        for k in self.trainable_names():
            self.exp_avg[self.slices[k]] = m[k].to(self.device).reshape(-1)
            self.exp_avg_sq[self.slices[k]] = v[k].to(self.device).reshape(-1)
        self.step_count = step
        changed = (hyper["betas"] != tuple(self.betas) or hyper["eps"] != self.adam_eps
                   or hyper["weight_decay"] != self.wd)
        self.lr, self.betas, self.adam_eps, self.wd = hyper["lr"], hyper["betas"], hyper["eps"], hyper["weight_decay"]
        if changed:
            self.reset_graphs()         # captured graphs bake everything except lr and the step count

    def save_session(self, path: str, *, iters: Optional[int] = None, epoch: int = 0, parameters=None,
                     best_val_target=None, original_state=None) -> str:
        """Write `<path>` in the reference's session format (bases.py:448-468).  Data parallel: rank 0 writes (every
        rank holds the same parameters and moments), then all ranks meet, as the reference does (`if self.is_rank0`
        ... `synchronize()`, bases.py:453,467)."""
        from .checkpoint import save_session
        dist_on = self._dist_on() and self.world > 1
        if not dist_on or torch.distributed.get_rank(self.pg) == 0:
            save_session(path, state_dict=self.state_dict(), optimizer=self.optimizer_state_dict(),
                         iters=self.step_count if iters is None else iters, epoch=epoch, parameters=parameters,
                         best_val_target=best_val_target, original_state=original_state)
        if dist_on:
            torch.distributed.barrier(self.pg)
        return path

    def load_session(self, path: str, restore_only_model: bool = False) -> dict:
        """bases.py:405-433: model tensors, then (unless restore_only_model) iters / epoch / optimiser state.
        Returns the checkpoint dict (iters, epoch, parameters, ... for the caller's bookkeeping)."""
        from .checkpoint import load_session_file
        ckpt = load_session_file(path)
        self.load_state_dict(ckpt["state_dict"])
        if not restore_only_model:
            self.load_optimizer_state_dict(ckpt["optimizer"])
        torch.cuda.current_stream().synchronize()
        return ckpt

    # ------------------------------------------------------------------------------------------------------------
    def _check_inputs(self, images, labels, on_device: bool = True) -> int:
        """-> n, the number of images of a training batch: fp32 images [n, 3, S, S] with 1 <= n <= batch_size, and labels
        either int64 class indices [n] or fp32 class probabilities [n, C] (what F.cross_entropy takes: a DataLoader's
        partial last batch, AdvancedAugCollate's mixup / cutmix / label-smoothed targets).  A BCE-with-logits engine takes
        fp32 multi-label targets [n, C] only."""
        B, img, C = self.shape["B"], self.shape["img"], self.shape["C"]
        where = "CUDA " if on_device else ""
        if (images.dim() != 4 or tuple(images.shape[1:]) != (3, img, img) or images.dtype != F32
                or (on_device and not images.is_cuda)):
            raise RuntimeError(f"images must be a {where}fp32 tensor of shape [n, 3, {img}, {img}] with 1 <= n <= {B}, "
                               f"got {images.dtype} {tuple(images.shape)}")
        n = int(images.shape[0])
        if not 1 <= n <= B:
            raise RuntimeError(f"a step takes 1 to batch_size={B} images, got {n}")
        if labels is None:
            return n
        if on_device and not labels.is_cuda:
            raise RuntimeError("labels must be a CUDA tensor")
        if self.criterion == 1:
            if labels.dtype != F32 or tuple(labels.shape) != (n, C):
                raise RuntimeError(f"a BCE-with-logits engine takes fp32 multi-label targets of shape [{n}, {C}], got "
                                   f"{labels.dtype} {tuple(labels.shape)}")
            return n
        if labels.dtype == torch.int64:
            if tuple(labels.shape) != (n,):
                raise RuntimeError(f"int64 labels must have shape [{n}] (one class index per image), got {tuple(labels.shape)}")
        elif labels.dtype == F32:
            if tuple(labels.shape) != (n, C):
                raise RuntimeError(f"fp32 targets must have shape [{n}, {C}] (class probabilities per image), got "
                                   f"{tuple(labels.shape)}")
        else:
            raise RuntimeError(f"labels must be int64 [n] class indices or fp32 [n, C] class probabilities, got {labels.dtype}")
        return n

    def _launch_forward(self, images: torch.Tensor, labels: Optional[torch.Tensor], n: int):
        # CrossEntropyLoss(mean) over the local batch of n images (wrappers.py:314), BCEWithLogitsLoss(mean) over its n*C
        # elements; DDP later averages over ranks.  The full hard-label batch keeps its original entry point; a partial
        # batch or fp32 targets take the n-row one.
        inv = 1.0 / n if self.criterion == 0 else 1.0 / (n * self.shape["C"])
        if n == self.shape["B"] and (labels is None or labels.dtype == torch.int64):
            LIB.call("apla_engine_forward", self._handle, ptr(images), ptr(labels), inv, inv, stream())
            return
        soft = labels is not None and labels.dtype == F32
        LIB.call("apla_engine_forward_n", self._handle, ptr(images), n, None if soft else ptr(labels),
                 ptr(labels) if soft else None, inv, inv, stream())

    def _draw_drop_path(self, n: int) -> torch.Tensor:
        """-> CPU fp32 [L, 2, n] stochastic-depth scales: image b keeps branch (l, j) with probability keep = 1 - p[l][j]
        (an independent draw per image, branch and call, as vit.py's drop_path) and is then scaled by 1 / keep."""
        keep = self._dp_keep[:, :, None]
        u = torch.rand(self.shape["L"], 2, n, generator=self._dp_gen, dtype=torch.float64)
        return ((u < keep).double() / keep).float()

    def _push_drop_path(self, n: int):
        """New masks for the training forward about to run -> the device buffer (stream-ordered, like _push_hyper)."""
        scales = self._draw_drop_path(n)
        self.last_drop_path_scales = scales
        full = torch.ones(self.shape["L"], 2, self.shape["B"], dtype=F32)
        full[:, :, :n] = scales
        # a fresh pageable tensor: its bytes are staged at call time (see _push_hyper)
        self._dp_dev.copy_(full, non_blocking=True)

    def forward(self, images: torch.Tensor, labels: Optional[torch.Tensor] = None) -> torch.Tensor:
        """images fp32 [n,3,S,S] (1 <= n <= B) on the engine's device -> logits fp32 [n,C], a view of the first n rows of
        `self.logits` (and loss / dlogits when labels are given: int64 [n] class indices or fp32 [n, C] probabilities;
        on a BCE-with-logits engine fp32 [n, C] multi-label targets, with the mean over the n*C elements).
        The next backward() runs over the same n images.  With drop path (a model built with drop_path_rate > 0) this is
        the training forward: it draws new masks (`last_drop_path_scales`); `predict` is the evaluation forward."""
        n = self._check_inputs(images, labels)
        images = images.contiguous()
        labels = labels.contiguous() if labels is not None else None
        if self._dp_dev is not None:
            self._push_drop_path(n)
        self._launch_forward(images, labels, n)
        return self.logits if n == self.shape["B"] else self.logits[:n]

    def backward(self):
        L = self.shape["L"]
        if self.world == 1:
            LIB.call("apla_engine_backward", self._handle, L - 1, 0, stream())
            return
        # data parallel: reduce the upper blocks' gradients (plus fc.weight, contiguous with them in the arena) on a
        # side stream while the lower blocks are still in backward (chunk plan: apla_b200/dp.py)
        from .dp import ArenaLayout, allreduce_arena
        lay = ArenaLayout(L=L, r=self.shape["r"], D=self.shape["D"], C=self.shape["C"])
        half = lay.split_block()
        cur = torch.cuda.current_stream()

        def reduce(which):
            if self._peer is not None:
                # few CTAs while the lower backward shares the GPU, more for the exposed tail
                self._peer.all_reduce_chunks(lay, which, ctas=32 if which == "early" else 96)
            else:
                allreduce_arena(self.grads, lay, group=self.pg, which=which)

        LIB.call("apla_engine_backward", self._handle, L - 1, half, stream())
        ev = torch.cuda.Event()
        ev.record(cur)
        with torch.cuda.stream(self._ar_stream):
            self._ar_stream.wait_event(ev)
            reduce("early")
        if half > 0:
            LIB.call("apla_engine_backward", self._handle, half - 1, 0, stream())
        ev2 = torch.cuda.Event()
        ev2.record(cur)
        with torch.cuda.stream(self._ar_stream):
            self._ar_stream.wait_event(ev2)
            reduce("late")
        cur.wait_stream(self._ar_stream)

    def reset_graphs(self):
        """Drop the captured CUDA graphs (they bake weight_decay, clip, betas and adam_eps -- everything except lr and the
        step count, which travel through the device-side hyper buffer); the next steps re-capture."""
        self._graphs.clear()
        self._graph_seen.clear()
        self._graph_keep = []

    def _push_hyper(self):
        """lr and the bias corrections of the step about to run -> device (stream-ordered, before the AdamW kernel)."""
        t = self.step_count
        # a fresh PAGEABLE tensor: the runtime stages its bytes at call time, so the host may prepare the next step's
        # values while this copy is still queued (a reused pinned buffer would be read when the copy executes)
        self._hyper_dev.copy_(torch.tensor([self.lr, 1.0 - self.betas[0] ** t, (1.0 - self.betas[1] ** t) ** 0.5],
                                           dtype=F32), non_blocking=True)

    def optim_step(self):
        self.step_count += 1
        if self.use_graph:
            self._push_hyper()
        LIB.call("apla_engine_optim", self._handle, 1.0 / self.world, float(self.clip or 0.0), self.lr, self.wd,
                 self.betas[0], self.betas[1], self.adam_eps, self.step_count, stream())

    def step(self, images: torch.Tensor, labels: torch.Tensor) -> torch.Tensor:
        """One Trainer.global_step on device-resident inputs -- fp32 images [n, 3, S, S] with 1 <= n <= batch_size, int64
        labels [n] or fp32 targets [n, C] -- with the mean loss over the n images; returns the (device) loss scalar.  On a
        BCE-with-logits engine the labels are fp32 multi-label targets [n, C] and the loss is the mean over n*C elements."""
        if not self.use_graph:
            self.forward(images, labels)
            self.backward()
            self.optim_step()
            return self.loss
        # graph path: a buffer pair is run eagerly the first time it is seen, captured on its second step (same launch
        # sequence, nothing executes during capture) and replayed from then on
        if not images.is_contiguous():
            images = images.contiguous()      # (a fresh buffer every call: stays on the eager path)
        if not labels.is_contiguous():
            labels = labels.contiguous()
        # the row count (images.shape) and the label kind (dtype / shape) are baked into a captured step: a partial batch
        # gets a graph of its own, captured on its second sighting like any buffer pair
        key = (images.data_ptr(), labels.data_ptr(), tuple(images.shape), labels.dtype, tuple(labels.shape))
        g = self._graphs.get(key)
        if g is None:
            seen = self._graph_seen.get(key, 0)
            self._graph_seen[key] = seen + 1
            if seen == 0 or len(self._graphs) >= 4:
                self.forward(images, labels)
                self.backward()
                self.optim_step()
                return self.loss
            n = self._check_inputs(images, labels)
            torch.cuda.current_stream().synchronize()
            L = self.shape["L"]

            def capture(fn):
                gr = torch.cuda.CUDAGraph()
                # captured on a high-priority stream: the kernel nodes inherit it, so the main chain's CTAs are placed
                # before those of the lowest-priority side branch (weight gradients) whenever both are pending
                if getattr(self, "_cap_stream", None) is None:
                    self._cap_stream = torch.cuda.Stream(device=self.device, priority=-1)
                with torch.cuda.graph(gr, stream=self._cap_stream, capture_error_mode="thread_local"):
                    fn()
                return gr

            def optim():
                LIB.call("apla_engine_optim", self._handle, 1.0 / self.world, float(self.clip or 0.0), self.lr, self.wd,
                         self.betas[0], self.betas[1], self.adam_eps, 1, stream())

            if self.world == 1:
                def whole():
                    self._launch_forward(images, labels, n)
                    LIB.call("apla_engine_backward", self._handle, L - 1, 0, stream())
                    optim()
                g = (capture(whole),)
            elif self._peer is not None:
                # data parallel with the native all-reduce: ONE graph; the early slice's reduction is forked onto the
                # side stream inside the capture and joins before the optimiser
                def whole_dp():
                    self._launch_forward(images, labels, n)
                    self.backward()
                    optim()
                g = (capture(whole_dp),)
            else:
                from .dp import ArenaLayout
                half = ArenaLayout(L=L, r=self.shape["r"], D=self.shape["D"], C=self.shape["C"]).split_block()

                def upper():
                    self._launch_forward(images, labels, n)
                    LIB.call("apla_engine_backward", self._handle, L - 1, half, stream())

                def lower():
                    LIB.call("apla_engine_backward", self._handle, half - 1, 0, stream())
                g = (capture(upper), capture(lower) if half > 0 else None, capture(optim))
            self._graphs[key] = g
            self._graph_keep = getattr(self, "_graph_keep", []) + [(images, labels)]   # keep the buffers alive
        self.step_count += 1
        self._push_hyper()
        if self._dp_dev is not None:
            # drawn outside any capture: the graphs read the buffer, every replay gets new masks
            self._push_drop_path(int(images.shape[0]))
        if self.world == 1 or self._peer is not None:
            g[0].replay()
            return self.loss
        from .dp import ArenaLayout, allreduce_arena
        lay = ArenaLayout(L=self.shape["L"], r=self.shape["r"], D=self.shape["D"], C=self.shape["C"])
        cur = torch.cuda.current_stream()
        g[0].replay()
        ev = torch.cuda.Event()
        ev.record(cur)
        with torch.cuda.stream(self._ar_stream):
            self._ar_stream.wait_event(ev)
            allreduce_arena(self.grads, lay, group=self.pg, which="early")
        if g[1] is not None:
            g[1].replay()
        ev2 = torch.cuda.Event()
        ev2.record(cur)
        with torch.cuda.stream(self._ar_stream):
            self._ar_stream.wait_event(ev2)
            allreduce_arena(self.grads, lay, group=self.pg, which="late")
        cur.wait_stream(self._ar_stream)
        g[2].replay()
        return self.loss

    def step_from_host(self, images_pinned: torch.Tensor, labels_pinned: torch.Tensor, lag: bool = True):
        """The end-to-end call: pinned host batch -> H2D -> step -> loss read back to the host.

        The batch is copied on a side stream into one of two device slots (so the copy of step k overlaps the compute
        of step k-1) and the loss comes back through a pinned buffer.  With `lag=True` (default) the call returns the
        loss of the PREVIOUS step (None on the first call) so that the host never waits for the step it just enqueued
        -- the same one-step-late logging the reference does every `log_every` (src/defaults/trainer.py:145-151);
        `lag=False` synchronises and returns this step's loss.  `drain()` returns the last pending loss.

        A batch may hold 1 <= n <= batch_size images (a loader's partial last batch) and int64 [n] labels or fp32 [n, C]
        targets (on a BCE-with-logits engine: fp32 [n, C] multi-label targets only): it is copied into the first n rows of
        the slot, and the first fp32-target batch allocates a pair of fp32 [B, C] target slots."""
        n = self._check_inputs(images_pinned, labels_pinned, on_device=False)
        if not hasattr(self, "_e2e"):
            B, img = self.shape["B"], self.shape["img"]
            self._e2e = dict(
                copy_stream=torch.cuda.Stream(device=self.device),
                img=[self.images_dev, self._new(B, 3, img, img, dtype=F32)],
                lab=[self.labels_dev, self._new(B, dtype=torch.int64)],
                copied=[torch.cuda.Event(), torch.cuda.Event()],
                done=[torch.cuda.Event(), torch.cuda.Event()],
                loss_host=[torch.zeros(1, dtype=F32).pin_memory(), torch.zeros(1, dtype=F32).pin_memory()],
                pending=[False, False], slot=0)
        st = self._e2e
        slot = st["slot"]
        st["slot"] = slot ^ 1
        cur = torch.cuda.current_stream()
        if labels_pinned.dtype == F32 and "tgt" not in st:
            # allocated on the compute stream that reads them, like the other slots
            B, C = self.shape["B"], self.shape["C"]
            st["tgt"] = [self._new(B, C, dtype=F32), self._new(B, C, dtype=F32)]
        img_dev = st["img"][slot][:n]
        lab_dev = (st["tgt"] if labels_pinned.dtype == F32 else st["lab"])[slot][:n]
        with torch.cuda.stream(st["copy_stream"]):
            if st["pending"][slot]:
                st["copy_stream"].wait_event(st["done"][slot])      # the step that last read this slot has finished
            img_dev.copy_(images_pinned, non_blocking=True)
            lab_dev.copy_(labels_pinned, non_blocking=True)
            st["copied"][slot].record()
        cur.wait_event(st["copied"][slot])
        self.step(img_dev, lab_dev)
        st["loss_host"][slot].copy_(self.loss, non_blocking=True)
        st["done"][slot].record(cur)
        st["pending"][slot] = True
        if lag:
            # this step is enqueued; only now wait for the previous one, so the GPU always has a step queued
            prev = slot ^ 1
            prev_loss = None
            if st["pending"][prev]:
                st["done"][prev].synchronize()
                prev_loss = float(st["loss_host"][prev][0])
                st["pending"][prev] = False
            return prev_loss
        st["done"][slot].synchronize()
        st["pending"][slot] = False
        return float(st["loss_host"][slot][0])

    def drain(self):
        """Wait for the last enqueued step_from_host() and return its loss (None if nothing is pending)."""
        st = getattr(self, "_e2e", None)
        if st is None:
            return None
        last = st["slot"] ^ 1
        if not st["pending"][last]:
            return None
        st["done"][last].synchronize()
        st["pending"][last] = False
        return float(st["loss_host"][last][0])

    # ---- evaluation (Trainer.evaluate / test, src/defaults/trainer.py:162-345) ----------------------------------------
    def _infer_workspace(self) -> Dict[str, torch.Tensor]:
        if self._infer_ws is None:
            s, cap = self.shape, self.eval_batch_size
            T, P, D = cap * s["N"], cap * s["P"], s["D"]
            ws = dict(infer_x=torch.empty(2, T, D, dtype=F32, device=self.device),
                      infer_ln=torch.empty(T, D, dtype=BF16, device=self.device),
                      infer_qkv=torch.empty(T, 3 * D, dtype=BF16, device=self.device),
                      infer_ao=torch.empty(T, D, dtype=BF16, device=self.device),
                      infer_lse=torch.empty(T, s["H"], dtype=F32, device=self.device),
                      infer_gelu=torch.empty(T, s["hidden"], dtype=BF16, device=self.device),
                      infer_patches=torch.empty(P, s["kpad"], dtype=BF16, device=self.device),
                      infer_pe_out=torch.empty(P, D, dtype=BF16, device=self.device),
                      infer_cls_ln=torch.empty(cap, D, dtype=BF16, device=self.device))
            for name, t in ws.items():
                self._set(name, t)
            LIB.call("apla_engine_set_option", self._handle, b"infer_batch", cap)
            self._infer_ws = ws
        return self._infer_ws

    def _check_eval_images(self, images: torch.Tensor):
        img = self.shape["img"]
        if images.dim() != 4 or tuple(images.shape[1:]) != (3, img, img) or images.shape[0] < 1:
            raise RuntimeError(f"images must be [n >= 1, 3, {img}, {img}], got {tuple(images.shape)}")
        if images.dtype != F32:
            raise RuntimeError("images must be fp32")

    def _infer(self, images: torch.Tensor, want_emb: bool):
        """-> (logits fp32 [n, C], bf16 embedding [n, D] or None), chunk by chunk of eval_batch_size images."""
        self._check_eval_images(images)
        self._infer_workspace()
        n = images.shape[0]
        logits = torch.empty(n, self.shape["C"], dtype=F32, device=self.device)
        emb = torch.empty(n, self.shape["D"], dtype=BF16, device=self.device) if want_emb else None
        for i in range(0, n, self.eval_batch_size):
            chunk = images[i:i + self.eval_batch_size].to(self.device, non_blocking=True).contiguous()
            LIB.call("apla_engine_infer", self._handle, ptr(chunk), chunk.shape[0], ptr(logits[i:]),
                     ptr(emb[i:]) if emb is not None else None, stream())
        return logits, emb

    @torch.no_grad()
    def predict(self, images: torch.Tensor) -> torch.Tensor:
        """Classifier.forward (models.py:81-92) with the engine's current weights: fp32 images [n, 3, S, S] (device or
        host, any n >= 1) -> a new fp32 logits tensor [n, C].  Runs in chunks of `eval_batch_size`; the training
        buffers, and so the captured step graphs, are left as they are."""
        return self._infer(images, want_emb=False)[0]

    @torch.no_grad()
    def embed(self, images: torch.Tensor) -> torch.Tensor:
        """Classifier.forward(x, return_embedding=True)'s embedding (models.py:88-92), the input of the reference's kNN
        evaluation (trainer.py:347-455): the final-norm CLS row the head reads, [n, D], as fp32 values of its bf16."""
        return self._infer(images, want_emb=True)[1].float()

    @torch.no_grad()
    def cls_attention(self, images: torch.Tensor) -> torch.Tensor:
        """The last block's attention of the CLS query over all N tokens, `get_last_selfattention(x)[:, :, 0, :]`
        (vit.py:439-485), with the engine's current weights: fp32 images [n, 3, S, S] (device or host, any n >= 1) -> a new
        fp32 tensor [n, H, N] whose rows sum to 1.  Runs like `predict` (chunks of `eval_batch_size` over the same
        workspace, training buffers and captured graphs untouched) and stops after the last block's attention.  For full
        [N, N] maps or other blocks, `sync_to_model()` and use `apla_b200.apla.attention_probabilities` on the model."""
        self._check_eval_images(images)
        self._infer_workspace()
        n, s = images.shape[0], self.shape
        probs = torch.empty(n, s["H"], s["N"], dtype=F32, device=self.device)
        for i in range(0, n, self.eval_batch_size):
            chunk = images[i:i + self.eval_batch_size].to(self.device, non_blocking=True).contiguous()
            LIB.call("apla_engine_cls_attention", self._handle, ptr(chunk), chunk.shape[0], ptr(probs[i:]), stream())
        return probs

    @torch.no_grad()
    def evaluate(self, batches) -> Dict[str, float]:
        """Mean cross-entropy and top-1 accuracy over an iterable of (images, labels) batches on the device or on the host
        (host batches are copied with non_blocking=True; pinned memory makes that asynchronous).  The sums stay on the
        device until the end; with a process group they are all-reduced once, so every rank returns the same numbers.
        -> {"loss": mean CE, "top1": fraction of correct argmax, "n": number of images}.

        On a BCE-with-logits engine the labels are fp32 multi-label targets [n, C], summed in double on the device
        -> {"loss": mean BCE over the n*C elements, "label_acc": fraction of elements with (logit > 0) == (target >= 0.5),
        "n": number of images}.  For ranking metrics (ROC-AUC, mAP) take `predict`'s logits."""
        bce = self.criterion == 1
        C = self.shape["C"]
        acc = torch.zeros(2, dtype=torch.float64 if bce else F32, device=self.device)
        n = 0
        for images, labels in batches:
            labels = labels.to(self.device, non_blocking=True).contiguous()
            if bce:
                if labels.dtype != F32 or tuple(labels.shape) != (images.shape[0], C):
                    raise RuntimeError(f"targets must be fp32 [n, {C}] matching the images, got {labels.dtype} "
                                       f"{tuple(labels.shape)}")
            elif labels.dtype != torch.int64 or labels.dim() != 1 or labels.shape[0] != images.shape[0]:
                raise RuntimeError("labels must be int64 [n] matching the images")
            logits = self.predict(images)
            LIB.call("apla_eval_accumulate_bce" if bce else "apla_eval_accumulate", ptr(logits), ptr(labels),
                     logits.shape[0], logits.shape[1], ptr(acc), stream())
            n += int(labels.shape[0])
        tot = torch.cat([acc.double(), torch.tensor([float(n)], dtype=torch.float64, device=self.device)])
        if self._dist_on() and self.world > 1:
            if torch.distributed.get_backend(self.pg) == "gloo":
                tot = tot.cpu()
            torch.distributed.all_reduce(tot, group=self.pg)
        loss_sum, hits, count = tot.tolist()
        if count == 0:
            raise ValueError("evaluate() got no batches")
        if bce:
            return {"loss": loss_sum / (count * C), "label_acc": hits / (count * C), "n": int(count)}
        return {"loss": loss_sum / count, "top1": hits / count, "n": int(count)}

    def grad_norm(self) -> torch.Tensor:
        """sqrt of the sum of squares the last optim_step clipped with (after the 1/world scaling)."""
        return self.sumsq[:1].sqrt()

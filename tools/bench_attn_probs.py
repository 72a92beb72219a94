#!/usr/bin/env python
"""Attention probabilities on one B200: what `apla_attn_probs` (csrc/attention_probs.cu) costs, and the user-level paths
built on it.

  kernel        probs_f32[B, H, q_rows, N] from the forward's qkv / lse at C2 (ViT-B/14, 64 x 257 tokens, 12 heads) with
                every query row ("full") and with the CLS row only ("cls"), at C5 (2 x 1370 tokens) and at ViT-L/14
                (64 x 257 tokens, 16 heads); CUDA events over many launches.  Written GB/s against the byte floor (the
                output bytes at the 6.5 TB/s HBM copy rate measured in SURVEY.md, computed, not measured) and, alternated
                with it, torch eager `((q @ k^T) * scale).softmax(-1)` in fp32 on the same qkv.  The full outputs (180-270 MB)
                are larger than the 126 MB L2.
  engine        C2 (224 px) `FineTuneEngine.cls_attention` images/s next to `predict` at the same eval_batch_size (64)
  module        last self-attention of 64 C2 images through fused blocks (`attention_probabilities` +
                `blocks[-1](x, return_attention=True)`) under torch.no_grad

Prints one JSON line per measurement, each with the GPU's name and power limit read in the same run."""
import argparse
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from bench_infer import INFO, c2_model, emit, gpu_info, timed    # noqa: E402
from apla_b200 import ops                                        # noqa: E402
from apla_b200._lib import require_device                        # noqa: E402
from apla_b200.apla import attention_probabilities, fuse_apla_blocks   # noqa: E402
from apla_b200.engine import FineTuneEngine                      # noqa: E402

HBM_COPY_GBPS = 6541.5          # SURVEY.md: measured HBM copy rate of this card type (used as the floor, not re-measured)


def bench_kernel(iters, warmup, rounds):
    for tag, B, N, H, full in (("c2_full", 64, 257, 12, True), ("c2_cls", 64, 257, 12, False),
                               ("c5_full", 2, 1370, 12, True), ("vitl_full", 64, 257, 16, True)):
        q_rows = N if full else 1
        g = torch.Generator(device="cuda").manual_seed(0)
        qkv = torch.randn(B * N, 3 * H * 64, device="cuda", generator=g).bfloat16()
        scale = 0.125
        _, lse = ops.attn_fwd(qkv, H, scale, B, N)
        out = torch.empty(B, H, q_rows, N, device="cuda")
        written = out.numel() * 4
        floor_us = written / HBM_COPY_GBPS / 1e3

        def kernel():
            ops.attn_probs(qkv, lse, H, scale, B, N, q_rows=q_rows, out=out)

        def eager():
            t = qkv.float().view(B, N, 3, H, 64).permute(2, 0, 3, 1, 4)
            return ((t[0][:, :, :q_rows] @ t[1].transpose(-2, -1)) * scale).softmax(-1)

        ref = eager()
        kernel()
        torch.cuda.synchronize()
        err = float((out - ref).norm() / ref.norm())
        del ref
        for r in range(rounds):
            for impl, fn in (("apla_attn_probs", kernel), ("torch_eager_fp32", eager)):
                ms = timed(fn, iters, warmup)
                emit(what="attn_probs_kernel", shape=tag, B=B, N=N, H=H, q_rows=q_rows, impl=impl, round=r, us=ms * 1e3,
                     written_mb=written / 1e6, written_gb_per_s=written / ms / 1e6, floor_us=floor_us,
                     fraction_of_floor=floor_us / (ms * 1e3), rel_err_vs_eager=err, iters=iters)
        del qkv, lse, out
        torch.cuda.empty_cache()


def bench_engine(n_images, iters, warmup, rounds):
    images = torch.randn(n_images, 3, 224, 224, generator=torch.Generator().manual_seed(1234)).cuda()
    eng = FineTuneEngine(c2_model(), batch_size=64, img_size=224, eval_batch_size=64)
    for r in range(rounds):
        for path, fn in (("predict", lambda: eng.predict(images)), ("cls_attention", lambda: eng.cls_attention(images))):
            ms = timed(fn, iters, warmup)
            emit(what="engine_eval", path=path, eval_batch_size=64, images=n_images, round=r, ms=ms,
                 images_per_s=n_images / ms * 1e3)
    return eng


def bench_module(eng, iters, warmup, rounds):
    model = eng.model
    fuse_apla_blocks(model)
    eng.sync_to_model()
    model.cuda().eval()
    bb = model.backbone
    images = torch.randn(64, 3, 224, 224, generator=torch.Generator().manual_seed(7)).cuda()

    def last_attention():
        with torch.no_grad(), attention_probabilities(model):
            x = bb.tokens(images)
            for blk in bb.blocks[:-1]:
                x = blk(x)
            return bb.blocks[-1](x, return_attention=True)

    def forward():
        with torch.no_grad():
            return model(images)

    for r in range(rounds):
        for path, fn in (("last_self_attention", last_attention), ("model_forward_no_grad", forward)):
            ms = timed(fn, iters, warmup)
            emit(what="module_fused", path=path, images=64, round=r, ms=ms, images_per_s=64 / ms * 1e3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--images", type=int, default=1024, help="C2 images per timed engine pass")
    ap.add_argument("--parts", default="kernel,engine,module")
    a = ap.parse_args()
    require_device()
    INFO.update(gpu_info())
    parts = a.parts.split(",")
    if "kernel" in parts:
        bench_kernel(a.iters, a.warmup, a.rounds)
    if "engine" in parts or "module" in parts:
        eng = bench_engine(a.images, max(1, a.iters // 10), a.warmup, a.rounds)
        if "module" in parts:
            bench_module(eng, max(1, a.iters // 10), a.warmup, a.rounds)


if __name__ == "__main__":
    main()

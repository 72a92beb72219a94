#!/usr/bin/env python
"""Stochastic depth in the fused blocks on one B200: the module path of a user who keeps the reference's trainer
(fuse_apla_blocks + fuse_patch_embed + cache_pos_encoding, fwd + CE + bwd + clip + torch AdamW) at bench.py's C2
workload (ViT-B/14, 224 px, 257 tokens, partial_size 8, 555 classes, batch 64), alternated round by round:

  rate 0            the model built with drop_path_rate 0: today's calls, nothing drawn
  rate 0.1          drop_path_rate 0.1 (linspace over the 12 blocks): masks drawn by the blocks' DropPath modules, the
                    row-scaled native calls, and no gradient hand-over into a block that drops (it casts for itself)
  rate 0, no chain  rate 0 with the block-to-block hand-over off (APLA_BLOCK_CHAIN=0): what the hand-over saves, i.e. the
                    most the lost hand-overs under drop path can cost

Every line carries the GPU's name, power limit and maximum SM clock read in the same run; the lines are printed and
written to --out."""
import argparse
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import apla_b200.apla.apla_block as AB                                  # noqa: E402
from apla_b200._lib import require_device                               # noqa: E402
from apla_b200.apla import cache_pos_encoding, fuse_apla_blocks, fuse_patch_embed  # noqa: E402
from apla_b200.config import AplaConfig                                 # noqa: E402
from apla_b200.hostvit import build_classifier                          # noqa: E402
from tools.bench_engine_batches import B, IMG, C, INFO, OUT, emit, gpu_info, timed  # noqa: E402
from tools.bench_module_paths import groups                             # noqa: E402


def stepper(rate):
    model = build_classifier("vit_base", img_size=518, patch_size=14, n_classes=C, apla_config=AplaConfig(8), seed=0,
                             drop_path_rate=rate)
    model = cache_pos_encoding(fuse_patch_embed(fuse_apla_blocks(model))).cuda().train()
    opt = torch.optim.AdamW(groups(model), lr=3e-5, weight_decay=1e-5)
    params = [p for p in model.parameters() if p.requires_grad]
    g = torch.Generator().manual_seed(1234)
    images = torch.randn(B, 3, IMG, IMG, generator=g).cuda()
    labels = torch.randint(0, C, (B,), generator=g).cuda()

    def step():
        opt.zero_grad(set_to_none=True)
        loss = torch.nn.functional.cross_entropy(model(images), labels)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(params, 1.0)
        opt.step()

    return step


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=250, help="steps per timed window (~2.4 s at C2)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles",
                                                  "bench_block_drop_path.jsonl"))
    a = ap.parse_args()
    require_device()
    INFO.update(gpu_info())
    steps = {0.0: stepper(0.0), 0.1: stepper(0.1)}
    configs = [("rate 0", 0.0, True), ("rate 0.1", 0.1, True), ("rate 0, no chain", 0.0, False)]
    for r in range(a.rounds):
        for name, rate, chain in configs:
            AB._CHAIN = chain
            ms = timed(steps[rate], a.iters, a.warmup)
            emit(what="module_path_step", config=name, drop_path_rate=rate, chain=chain, n=B, round=r, ms_per_step=ms,
                 images_per_s=B / ms * 1e3, iters=a.iters, timing="CUDA events around eager steps")
    AB._CHAIN = True
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write("\n".join(OUT) + "\n")


if __name__ == "__main__":
    main()

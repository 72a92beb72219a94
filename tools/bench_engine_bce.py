#!/usr/bin/env python
"""Multi-label (BCE-with-logits) training steps on one B200, at bench.py's C2 workload (ViT-B/14, 224 px, 257 tokens,
partial_size 8, 555 outputs, batch_size 64).

  step         a graph-replayed step of a cross-entropy engine on int64 labels against one of a BCE-with-logits engine
               (criterion=nn.BCEWithLogitsLoss()) on multi-hot fp32 [64, 555] targets, alternated round by round in one
               process
  head_kernel  bce_kernel against ce_kernel at (64, 555) and (1024, 1000): CUDA events over graph replays of 200
               back-to-back launches, alternated (the operands sit in L2, as they do inside the step)

Every line carries the GPU's name, power limit and maximum SM clock read in the same run; the lines are printed and
written to --out."""
import argparse
import os
import sys

import torch
import torch.nn as nn

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from apla_b200._lib import LIB, ptr, require_device, stream      # noqa: E402
from tools.bench_engine_batches import (B, IMG, C, INFO, OUT, batch, c2_engine, emit, gpu_info,  # noqa: E402
                                        timed)


def bench_step(iters, warmup, rounds):
    engines = {"cross_entropy": c2_engine(), "bce_with_logits": c2_engine(criterion=nn.BCEWithLogitsLoss())}
    images, labels = batch(B, 30)
    g = torch.Generator().manual_seed(31)
    targets = (torch.rand(B, C, generator=g) < 0.05).float().cuda()          # multi-hot, about 28 labels per image
    inputs = {"cross_entropy": (images, labels), "bce_with_logits": (images, targets)}
    for r in range(rounds):
        for crit, eng in engines.items():
            ms = timed(lambda: eng.step(*inputs[crit]), iters, warmup)
            emit(what="step", criterion=crit, labels=str(inputs[crit][1].dtype), n=B, round=r, ms_per_step=ms,
                 images_per_s=B / ms * 1e3, iters=iters, graphs=len(eng._graphs))


def bench_head_kernel(rounds, launches=200, replays=20):
    for rows, classes in ((64, 555), (1024, 1000)):
        g = torch.Generator(device="cuda").manual_seed(0)
        z = torch.randn(rows, classes, device="cuda", generator=g) * 3
        y = torch.randint(0, classes, (rows,), device="cuda", generator=g)
        t = (torch.rand(rows, classes, device="cuda", generator=g) < 0.05).float()
        dl = torch.empty_like(z)
        loss = torch.zeros(1, device="cuda")

        def ce():
            LIB.call("apla_cross_entropy", ptr(z), ptr(y), ptr(dl), ptr(loss), rows, classes, 1.0, 1.0, stream())

        def bce():
            LIB.call("apla_bce_with_logits", ptr(z), ptr(t), ptr(dl), ptr(loss), rows, classes, 1.0, 1.0, stream())

        def graph_of(fn):
            # `launches` launches captured in one CUDA graph: the replay times the kernel back to back, not the host's
            # ctypes call rate (about 8 us per call, longer than either kernel at these shapes)
            fn()
            torch.cuda.synchronize()
            gr = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gr):
                for _ in range(launches):
                    fn()
            return gr

        graphs = {"ce_kernel": graph_of(ce), "bce_kernel": graph_of(bce)}
        for r in range(rounds):
            for kernel, reads in (("ce_kernel", 4 + 8 / classes), ("bce_kernel", 8)):
                ms = timed(graphs[kernel].replay, replays, 2) / launches
                byts = rows * classes * (reads + 4)          # logits (+ targets) read, dlogits written
                emit(what="head_kernel", kernel=kernel, rows=rows, classes=classes, round=r, us=ms * 1e3,
                     gb_per_s=byts / ms / 1e6, launches=launches * replays, timing="CUDA graph of back-to-back launches")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50, help="steps per timed window")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--parts", default="step,head_kernel")
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles",
                                                  "bench_engine_bce.jsonl"))
    a = ap.parse_args()
    require_device()
    INFO.update(gpu_info())
    parts = a.parts.split(",")
    if "step" in parts:
        bench_step(a.iters, a.warmup, a.rounds)
        torch.cuda.empty_cache()
    if "head_kernel" in parts:
        bench_head_kernel(a.rounds)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write("\n".join(OUT) + "\n")


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""Training steps on partial batches and on probability targets on one B200, at bench.py's C2 workload (ViT-B/14, 224 px,
257 tokens, partial_size 8, 555 classes, batch_size 64).

  entry        the full 64-image hard-label step launched through apla_engine_forward and through
               apla_engine_forward_n(n_img = 64), eager, alternated round by round in one process
  partial      per-step time of n = 64 / 32 / 1 images, eager and replayed from the step's CUDA graph
  soft         a graph-replayed step with int64 labels against one with fp32 [64, 555] mixup targets, alternated
  ce_kernel    ce_soft_kernel against ce_kernel at (64, 555) and (1024, 1000): CUDA events over graph replays of 200
               back-to-back launches, alternated (the operands sit in L2, as they do inside the step)

Every line carries the GPU's name and power limit read in the same run; the lines are printed and written to --out."""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from apla_b200._lib import LIB, ptr, require_device, stream      # noqa: E402
from apla_b200.config import AplaConfig                           # noqa: E402
from apla_b200.engine import FineTuneEngine                       # noqa: E402
from apla_b200.hostvit import build_classifier                    # noqa: E402


def gpu_info():
    info = dict(gpu=torch.cuda.get_device_name(0))
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [s.strip() for s in q.split(",")]
    except Exception as e:                     # the measurement stands; the line says what could not be read
        info["power_limit"] = f"unread ({type(e).__name__})"
    return info


INFO = {}
OUT = []


def emit(**kw):
    line = json.dumps(dict(kw, **INFO))
    OUT.append(line)
    print(line, flush=True)


def timed(fn, iters, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


B, IMG, C = 64, 224, 555


def c2_engine(**kw):
    model = build_classifier("vit_base", img_size=518, patch_size=14, n_classes=C, apla_config=AplaConfig(8), seed=0)
    return FineTuneEngine(model, batch_size=B, img_size=IMG, **kw)


def batch(n, seed, soft=False):
    g = torch.Generator().manual_seed(seed)
    images = torch.randn(n, 3, IMG, IMG, generator=g).cuda()
    labels = torch.randint(0, C, (n,), generator=g)
    if not soft:
        return images, labels.cuda()
    lam, eps = 0.7, 0.1
    a = torch.full((n, C), eps / C).scatter_(1, labels[:, None], 1 - eps + eps / C)
    b = torch.full((n, C), eps / C).scatter_(1, labels.flip(0)[:, None], 1 - eps + eps / C)
    return images, (lam * a + (1 - lam) * b).float().cuda()


def bench_entry(eng, iters, warmup, rounds):
    images, labels = batch(B, 1)
    L = eng.shape["L"]

    def tail():
        LIB.call("apla_engine_backward", eng._handle, L - 1, 0, stream())
        eng.optim_step()

    def old():
        LIB.call("apla_engine_forward", eng._handle, ptr(images), ptr(labels), 1.0 / B, 1.0 / B, stream())
        tail()

    def new():
        LIB.call("apla_engine_forward_n", eng._handle, ptr(images), B, ptr(labels), None, 1.0 / B, 1.0 / B, stream())
        tail()

    for r in range(rounds):
        for entry, fn in (("apla_engine_forward", old), ("apla_engine_forward_n", new)):
            ms = timed(fn, iters, warmup)
            emit(what="entry", entry=entry, n=B, round=r, ms_per_step=ms, images_per_s=B / ms * 1e3, iters=iters)


def bench_partial(eng, iters, warmup, rounds):
    for n in (B, 32, 1):
        images, labels = batch(n, 10 + n)

        def eager():
            eng.forward(images, labels)
            eng.backward()
            eng.optim_step()

        def graph():
            eng.step(images, labels)

        for r in range(rounds):
            for mode, fn in (("eager", eager), ("graph", graph)):
                ms = timed(fn, iters, warmup)
                emit(what="partial", n=n, mode=mode, round=r, ms_per_step=ms, images_per_s=n / ms * 1e3, iters=iters)
    emit(what="partial", graphs_captured=len(eng._graphs))


def bench_soft(eng, iters, warmup, rounds):
    eng.reset_graphs()                                  # (the partial part filled the cap of 4 graphs)
    hard = batch(B, 20)
    soft = batch(B, 20, soft=True)
    for r in range(rounds):
        for kind, (images, labels) in (("int64_labels", hard), ("fp32_targets", soft)):
            ms = timed(lambda: eng.step(images, labels), iters, warmup)
            emit(what="soft", labels=kind, n=B, round=r, ms_per_step=ms, images_per_s=B / ms * 1e3, iters=iters)


def bench_ce(rounds, launches=200, replays=20):
    for rows, classes in ((64, 555), (1024, 1000)):
        g = torch.Generator(device="cuda").manual_seed(0)
        z = torch.randn(rows, classes, device="cuda", generator=g) * 3
        y = torch.randint(0, classes, (rows,), device="cuda", generator=g)
        t = torch.softmax(torch.randn(rows, classes, device="cuda", generator=g), -1)
        dl = torch.empty_like(z)
        loss = torch.zeros(1, device="cuda")

        def hard():
            LIB.call("apla_cross_entropy", ptr(z), ptr(y), ptr(dl), ptr(loss), rows, classes, 1.0, 1.0, stream())

        def soft():
            LIB.call("apla_cross_entropy_soft", ptr(z), ptr(t), ptr(dl), ptr(loss), rows, classes, 1.0, 1.0, stream())

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

        graphs = {"ce_kernel": graph_of(hard), "ce_soft_kernel": graph_of(soft)}
        for r in range(rounds):
            for kernel, reads in (("ce_kernel", 4 + 8 / classes), ("ce_soft_kernel", 8)):
                ms = timed(graphs[kernel].replay, replays, 2) / launches
                byts = rows * classes * (reads + 4)          # logits (+ targets) read, dlogits written
                emit(what="ce_kernel", kernel=kernel, rows=rows, classes=classes, round=r, us=ms * 1e3,
                     gb_per_s=byts / ms / 1e6, launches=launches * replays, timing="CUDA graph of back-to-back launches")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50, help="steps per timed window")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--parts", default="entry,partial,soft,ce")
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles",
                                                  "bench_engine_batches.jsonl"))
    a = ap.parse_args()
    require_device()
    INFO.update(gpu_info())
    parts = a.parts.split(",")
    if {"entry", "partial", "soft"} & set(parts):
        eng = c2_engine()
        if "entry" in parts:
            bench_entry(eng, a.iters, a.warmup, a.rounds)
        if "partial" in parts:
            bench_partial(eng, a.iters, a.warmup, a.rounds)
        if "soft" in parts:
            bench_soft(eng, a.iters, a.warmup, a.rounds)
        del eng
        torch.cuda.empty_cache()
    if "ce" in parts:
        bench_ce(a.rounds)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write("\n".join(OUT) + "\n")


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""Stochastic depth (drop path) in the step engine on one B200, at bench.py's C2 workload (ViT-B/14, 224 px, 257 tokens,
partial_size 8, 555 classes, batch_size 64).

  step     a graph-replayed step of an engine over a rate-0 model against one over the same model built with
           drop_path_rate 0.1 (new masks drawn on the host and copied before every replay), alternated round by round
  kernels  at C2 shapes (64 x 257 token rows, D = 768): the row-scaled residual GEMM (EPI_RESID_SCALED) against the
           unscaled one (EPI_RESID) for the projection (K = 768) and fc2 (K = 3072), and the row-scaled LayerNorm
           backward against the unscaled one; CUDA events over graph replays of back-to-back launches, alternated

Every line carries the GPU's name, power limit and maximum SM clock read in the same run; the lines are printed and
written to --out."""
import argparse
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from apla_b200._lib import LIB, ptr, require_device, stream      # noqa: E402
from apla_b200.config import AplaConfig                           # noqa: E402
from apla_b200.engine import FineTuneEngine                       # noqa: E402
from apla_b200.hostvit import build_classifier                    # noqa: E402
from tools.bench_engine_batches import B, IMG, C, INFO, OUT, batch, emit, gpu_info, timed  # noqa: E402

N, D = 257, 768


def bench_step(iters, warmup, rounds):
    engines = {}
    for rate in (0.0, 0.1):
        model = build_classifier("vit_base", img_size=518, patch_size=14, n_classes=C, apla_config=AplaConfig(8),
                                 seed=0, drop_path_rate=rate)
        engines[rate] = FineTuneEngine(model, batch_size=B, img_size=IMG)
    images, labels = batch(B, 40)
    for r in range(rounds):
        for rate, eng in engines.items():
            ms = timed(lambda: eng.step(images, labels), iters, warmup)
            emit(what="step", drop_path_rate=rate, n=B, round=r, ms_per_step=ms, images_per_s=B / ms * 1e3,
                 iters=iters, graphs=len(eng._graphs))


def graph_of(fn, launches):
    # back-to-back launches in one CUDA graph: the replay times the kernels, not the host's ctypes call rate
    fn()
    torch.cuda.synchronize()
    gr = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gr):
        for _ in range(launches):
            fn()
    return gr


def bench_kernels(rounds, launches=50, replays=10):
    T = B * N
    g = torch.Generator(device="cuda").manual_seed(0)
    scale = ((torch.rand(B, device="cuda", generator=g) < 0.9).float() / 0.9)
    resid = torch.randn(T, D, device="cuda", generator=g)
    out = torch.empty(T, D, device="cuda")
    bias, gamma = torch.randn(D, device="cuda", generator=g), torch.ones(D, device="cuda")
    for K, layer in ((D, "proj"), (4 * D, "fc2")):
        A = torch.randn(T, K, device="cuda", generator=g).to(torch.bfloat16)
        W = (torch.randn(D, K, device="cuda", generator=g) * 0.02).to(torch.bfloat16)

        def plain():
            LIB.call("apla_gemm_bias_ls_residual_fwd", ptr(A), K, ptr(W), K, ptr(bias), ptr(gamma), ptr(resid), ptr(out),
                     D, T, D, K, stream())

        def scaled():
            LIB.call("apla_gemm_bias_ls_residual_scaled_fwd", ptr(A), K, ptr(W), K, ptr(bias), ptr(gamma), ptr(resid),
                     ptr(scale), N, ptr(out), D, T, D, K, stream())

        graphs = {"EPI_RESID": graph_of(plain, launches), "EPI_RESID_SCALED": graph_of(scaled, launches)}
        for r in range(rounds):
            for epi, gr in graphs.items():
                ms = timed(gr.replay, replays, 2) / launches
                emit(what="residual_gemm", layer=layer, epilogue=epi, M=T, N=D, K=K, round=r, us=ms * 1e3,
                     tflops=2.0 * T * D * K / ms / 1e9, timing="CUDA graph of back-to-back launches")
    dy = torch.randn(T, D, device="cuda", generator=g).to(torch.bfloat16)
    x = torch.randn(T, D, device="cuda", generator=g)
    dx = torch.zeros(T, D, device="cuda")
    dxb = torch.empty(T, D, device="cuda", dtype=torch.bfloat16)
    sub = torch.empty(T, 64, device="cuda", dtype=torch.bfloat16)
    idx = torch.arange(8, device="cuda", dtype=torch.int32)
    w = torch.ones(D, device="cuda")
    args = lambda: [ptr(dy), D, ptr(x), D, ptr(w), ptr(dx), D, ptr(dx), D, ptr(dxb), D, ptr(gamma), ptr(sub), 64,  # noqa: E731
                    ptr(idx), 8, 64]
    graphs = {"ln_bwd_kernel": graph_of(lambda: LIB.call("apla_layernorm_bwd", *args(), T, D, 1e-6, stream()), launches),
              "ln_bwd_scaled_kernel": graph_of(lambda: LIB.call("apla_layernorm_bwd_scaled", *args(), ptr(scale), N, T,
                                                                D, 1e-6, stream()), launches)}
    for r in range(rounds):
        for kernel, gr in graphs.items():
            ms = timed(gr.replay, replays, 2) / launches
            byts = T * D * (4 + 2 + 4 + 4 + 2) + T * 64 * 2   # x, dy, dres read; dx, dxb, sub written
            emit(what="layernorm_bwd", kernel=kernel, rows=T, D=D, round=r, us=ms * 1e3, gb_per_s=byts / ms / 1e6,
                 timing="CUDA graph of back-to-back launches")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50, help="steps per timed window")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--parts", default="step,kernels")
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles",
                                                  "bench_engine_drop_path.jsonl"))
    a = ap.parse_args()
    require_device()
    INFO.update(gpu_info())
    parts = a.parts.split(",")
    if "step" in parts:
        bench_step(a.iters, a.warmup, a.rounds)
        torch.cuda.empty_cache()
    if "kernels" in parts:
        bench_kernels(a.rounds)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write("\n".join(OUT) + "\n")


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""Forward-only evaluation on one B200: what the forward that keeps no backward state costs and saves.

  fc1_kernel     the fc1 GEMM with the forward-only epilogue (EPI_BIAS_GELU_G: gelu(h) only) against the training one
                 (EPI_BIAS_GELU_D: gelu(h) and gelu'(h)), at the C2 shape (ViT-B/14, 64 x 257 tokens) and the C4 teacher
                 shape (ViT-L/14, 128 x 257 tokens); CUDA events over operand sets that rotate through more than the
                 126 MB of L2, the two epilogues alternated
  c2_eval        ViT-B/14 224 px (bench.py's workload) images/s and peak memory of: FineTuneEngine.predict at
                 eval_batch_size 64 / 256 / 1024; engine.forward at the training batch 64; the module path
                 (sync_to_model, then the model with fused blocks under torch.no_grad) with the training block sequence
                 ("before") and with the forward-only one ("after"), alternated
  c4_teacher     the C4 teacher's 24 ViT-L/14 blocks over 128 global 224-px crops under torch.no_grad, training block
                 sequence against forward-only, alternated over the same input

Prints one JSON line per measurement, each with the GPU's name and power limit read in the same run."""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from apla_b200._lib import LIB, ptr, require_device, stream      # noqa: E402
from apla_b200.apla import apla_block as AB                       # noqa: E402
from apla_b200.apla import cache_pos_encoding, fuse_apla_blocks, fuse_patch_embed    # noqa: E402
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


def emit(**kw):
    print(json.dumps(dict(kw, **INFO)), flush=True)


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


def bench_fc1(iters, warmup, rounds):
    for tag, M, N, K in (("c2", 16448, 3072, 768), ("c4_teacher", 32896, 4096, 1024)):
        g = torch.Generator(device="cuda").manual_seed(0)
        out_bytes = M * N * 2
        nsets = max(2, -(-3 * 126 * 2 ** 20 // (M * K * 2 + 2 * out_bytes)) + 1)   # > 3x L2 per rotation
        A = [torch.randn(M, K, device="cuda", generator=g).bfloat16() for _ in range(nsets)]
        W = (torch.randn(N, K, device="cuda", generator=g) * K ** -0.5).bfloat16()
        bias = torch.randn(N, device="cuda", generator=g)
        G = [torch.empty(M, N, device="cuda", dtype=torch.bfloat16) for _ in range(nsets)]
        Dg = [torch.empty(M, N, device="cuda", dtype=torch.float16) for _ in range(nsets)]
        it = [0]

        def both():
            i = it[0] % nsets
            it[0] += 1
            LIB.call("apla_gemm_bias_gelu_dgelu_fwd", ptr(A[i]), K, ptr(W), K, ptr(bias), ptr(Dg[i]), ptr(G[i]), N, M, N, K,
                     stream())

        def g_only():
            i = it[0] % nsets
            it[0] += 1
            LIB.call("apla_gemm_bias_gelu_only_fwd", ptr(A[i]), K, ptr(W), K, ptr(bias), ptr(G[i]), N, M, N, K, stream())

        flops = 2.0 * M * N * K
        for r in range(rounds):
            for epi, fn, nout in (("EPI_BIAS_GELU_D", both, 2), ("EPI_BIAS_GELU_G", g_only, 1)):
                ms = timed(fn, iters, warmup)
                byts = M * K * 2 + N * K * 2 + nout * out_bytes
                emit(what="fc1_kernel", shape=tag, M=M, N=N, K=K, epilogue=epi, round=r, us=ms * 1e3,
                     tflops=flops / ms / 1e9, min_bytes_gb_per_s=byts / ms / 1e6, operand_sets=nsets, iters=iters)
        del A, G, Dg
        torch.cuda.empty_cache()


def c2_model():
    return build_classifier("vit_base", img_size=518, patch_size=14, n_classes=555, apla_config=AplaConfig(8), seed=0)


def training_sequence(self, x, cu, seqlens):
    """FusedAplaBlock's forward before the forward-only path: the training Function, which writes lse and gelu'."""
    at = self.attn
    return AB._AplaBlockFn.apply(x, at.proj_weight1, at.proj_bias1, self, cu, seqlens)


def bench_c2(n_images, iters, warmup, rounds):
    g = torch.Generator().manual_seed(1234)
    images = torch.randn(n_images, 3, 224, 224, generator=g).cuda()

    def report(path, fn, batch, **extra):
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        ms = timed(fn, iters, warmup)
        emit(what="c2_eval", path=path, batch=batch, images=n_images, ms=ms, images_per_s=n_images / ms * 1e3,
             peak_mem_gb=torch.cuda.max_memory_allocated() / 1e9,
             above_start_gb=(torch.cuda.max_memory_allocated() - base) / 1e9, **extra)

    for eb in (64, 256, 1024):
        torch.cuda.synchronize()
        before = torch.cuda.memory_allocated()
        eng = FineTuneEngine(c2_model(), batch_size=64, img_size=224, eval_batch_size=eb)
        engine_gb = (torch.cuda.memory_allocated() - before) / 1e9
        report("predict", lambda: eng.predict(images), eb, engine_gb=engine_gb)
        if eb == 64:
            chunks = images.split(64)

            def fwd():
                for c in chunks:
                    eng.forward(c)
            report("engine_forward", fwd, 64, engine_gb=engine_gb)
            model = eng.model
            cache_pos_encoding(fuse_patch_embed(fuse_apla_blocks(model)))
            eng.sync_to_model()
            model.cuda().eval()

            def module():
                with torch.no_grad():
                    for c in chunks:
                        model(c)
            fwd_only = AB.FusedAplaBlock._run_infer
            for r in range(rounds):
                AB.FusedAplaBlock._run_infer = training_sequence
                report("module_no_grad_before", module, 64, round=r)
                AB.FusedAplaBlock._run_infer = fwd_only
                report("module_no_grad_after", module, 64, round=r)
            del model
        del eng
        torch.cuda.empty_cache()


def bench_c4_teacher(images_n, iters, warmup, rounds):
    m = build_classifier("vit_large", apla_config=AplaConfig(1024), img_size=518, patch_size=14, n_classes=8, seed=0)
    fuse_apla_blocks(m.cuda())
    blocks = m.backbone.blocks
    glob = torch.randn(2 * images_n, 257, 1024, device="cuda", generator=torch.Generator(device="cuda").manual_seed(0))

    def teacher():
        with torch.no_grad():
            t = glob
            for blk in blocks:
                t = blk(t)
        return t

    fwd_only = AB.FusedAplaBlock._run_infer
    outs = {}
    for r in range(rounds):
        for path, impl in (("training_sequence", training_sequence), ("forward_only", fwd_only)):
            AB.FusedAplaBlock._run_infer = impl
            torch.cuda.synchronize()
            base = torch.cuda.memory_allocated()
            torch.cuda.reset_peak_memory_stats()
            ms = timed(teacher, iters, warmup)
            outs[path] = teacher()
            emit(what="c4_teacher", path=path, round=r, crops=2 * images_n, tokens=2 * images_n * 257, blocks=len(blocks),
                 ms=ms, peak_above_start_gb=(torch.cuda.max_memory_allocated() - base) / 1e9)
    AB.FusedAplaBlock._run_infer = fwd_only
    emit(what="c4_teacher", check="outputs_bitwise_equal", value=bool(torch.equal(outs["training_sequence"],
                                                                                  outs["forward_only"])))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--images", type=int, default=1024, help="C2 images per timed pass")
    ap.add_argument("--c4-images", type=int, default=64, help="C4 images (2 global crops each)")
    ap.add_argument("--parts", default="fc1,c2,c4")
    a = ap.parse_args()
    require_device()
    INFO.update(gpu_info())
    parts = a.parts.split(",")
    if "fc1" in parts:
        bench_fc1(a.iters * 5, a.warmup, a.rounds)
    if "c2" in parts:
        bench_c2(a.images, a.iters, a.warmup, a.rounds)
    if "c4" in parts:
        bench_c4_teacher(a.c4_images, a.iters, a.warmup, a.rounds)


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""bench.py -- the APLA fine-tune step on B200 (BASELINE.json configs[1]: ViT-B/14, partial_size=8, 224 px,
555 classes, batch 64 per GPU, bf16 compute, synthetic data, seeded random-init weights of that architecture).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path
    python bench.py --impl reference [--gpus N] ...                # the reference algorithm on the host CPU cores
    python bench.py --dump-outputs DIR                             # also write the last timed step's outputs

One step = Trainer.global_step (src/defaults/trainer.py:106-138): forward, CrossEntropy, backward (weight
gradients only for the APLA projection rows + head), data-parallel gradient mean, clip_grad_norm_(1.0), AdamW.
Prints ONE JSON line (rank 0).  `value` = whole-job images/s with the batch resident in HBM; `e2e` = the same
through the public API from pinned host buffers (H2D of the batch and D2H of the loss inside the timed region).
Every timed leg runs exactly --steps steps; the >= 2.5 s sustained leg runs only with --sustained.

Weights, APLA indices and batches are seeded, so the same arguments give the same inputs on every run and
`--dump-outputs` of two builds can be compared array for array.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "ViT-B/14 APLA fine-tune images/sec/GPU at 1/2/4/8 B200; % bf16 tensor roofline"
WORKLOAD = dict(arch="vit_base", img=224, table_img=518, patch=14, n_classes=555, partial_size=8, batch_per_gpu=64)
# --workload: the default is the configuration the metric is quoted on (BASELINE.json configs[1] = C2); the others are
# the remaining single-box shapes of SURVEY.md App. A through the SAME engine (reported in DESIGN.md, not the bench line
# the driver reads).  c5 / vitl end in the classifier head: the mmseg decoder and the DINOv2 SSL heads are out of scope.
WORKLOADS = {
    "c2": WORKLOAD,
    "c3": dict(WORKLOAD, partial_size=768),
    "c5": dict(WORKLOAD, img=518, partial_size=768, batch_per_gpu=2),
    "vitl": dict(WORKLOAD, arch="vit_large", partial_size=128),
    # BASELINE.json configs[3]: ViT-L/14 DINOv2 self-supervised APLA adaptation, ISIC2019-shape multi-crop batch (64 images
    # per GPU -> 128 global 224-px + 512 local 98-px crops), shared DINO / iBOT head with 65 536 prototypes, every
    # projection row trainable (the shipped multi-GPU config is partial_size "full", SURVEY.md 3.4); module-level path
    "c4": dict(arch="vit_large", img=224, local_img=98, table_img=518, patch=14, n_classes=65536, partial_size=1024,
               batch_per_gpu=64, n_local=8, head_hidden=2048, head_bottleneck=256),
}
GFLOP_PER_IMAGE_C4 = 1534.0          # SURVEY.md 8d: student 2 x 343.6 + 8 x 63.4, teacher fwd 2 x 162.0, DINO head ~16


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(tflops_burst=d["bf16_tflops"], tflops_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    hbm_gbs=d["hbm_gbs"], source="measured")
    return dict(tflops_burst=1590.0, tflops_sustained=1400.0, hbm_gbs=6650.0, source="fallback")


class ClockSampler:
    """Samples SM clock / throttle reasons of one GPU during the timed region (NVML, else nvidia-smi)."""

    def __init__(self, index):
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop = threading.Event()
        self._thread = None
        self._nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nvml = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self._nvml = None

    def _loop(self):
        nv = self._nvml
        names = {}
        if nv is not None:
            for k in dir(nv):
                if k.startswith("nvmlClocksEventReason") or k.startswith("nvmlClocksThrottleReason"):
                    v = getattr(nv, k)
                    if isinstance(v, int) and v not in (0,):
                        names.setdefault(v, k.replace("nvmlClocksEventReason", "").replace("nvmlClocksThrottleReason", ""))
        while not self._stop.is_set():
            try:
                if nv is not None:
                    self.samples.append(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM))
                    try:
                        mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self._h)
                    except Exception:
                        mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
                    for bit, nm in names.items():
                        if mask & bit and bit & (bit - 1) == 0:
                            self.reasons.add(nm)
                else:
                    out = subprocess.run(["nvidia-smi", f"--id={self.index}",
                                          "--query-gpu=clocks.sm,clocks.max.sm,clocks_event_reasons.active",
                                          "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5)
                    f = [x.strip() for x in out.stdout.strip().split(",")]
                    self.samples.append(int(f[0]))
                    self.max_mhz = int(f[1])
                    self.reasons.add(f[2])
            except Exception:
                pass
            self._stop.wait(0.02)

    def start(self):
        self._thread = threading.Thread(target=self._loop, daemon=True)
        self._thread.start()

    def stop(self):
        self._stop.set()
        if self._thread:
            self._thread.join(timeout=2)
        s = sorted(self.samples)
        rs = sorted(r for r in self.reasons if r and r.lower() not in ("none", "gpuidle", "applicationsclockssetting"))
        return dict(sm_mhz=(s[len(s) // 2] if s else None), sm_max_mhz=self.max_mhz, reasons=rs, samples=len(s))


def describe_workload(w):
    if "n_local" in w:
        return (f"ViT-L/14 DINOv2 self-supervised APLA adaptation step (student + EMA teacher, DINO + iBOT + KoLeo, shared "
                f"head with {w['n_classes']} prototypes), multi-crop: 2 x {w['img']}px + {w['n_local']} x {w['local_img']}px "
                f"crops per image, partial_size={w['partial_size']} (every projection row), AdamW lr 3e-5 clip 3.0")
    return (f"{'ViT-L' if w['arch'] == 'vit_large' else 'ViT-B'}/14 dinov2-arch (518-px pos table, LayerScale, qkv bias) APLA "
            f"partial_size={w['partial_size']} supervised fine-tune step, {w['img']}px, 555 classes, AdamW lr 3e-5 wd 1e-5 "
            "clip 1.0")


def make_config(w, B, world):
    """The `config` object of the JSON line -- built the same way by the GPU arm and by the reference (CPU) arm."""
    return dict(workload=describe_workload(w), global_batch=B * world, batch_per_gpu=B,
                tokens_per_image=(w["img"] // w["patch"]) ** 2 + 1, parallelism=f"dp{world}",
                l2="per-step working set (saved activations of every block, several GB) >> 126 MB L2: no flush needed",
                **{k: v for k, v in w.items() if k != "batch_per_gpu"})


def synthetic_batch(batch, img, n_classes, seed=1234, rank=0):
    import torch
    g = torch.Generator().manual_seed(seed + rank)
    return torch.randn(batch, 3, img, img, generator=g), torch.randint(0, n_classes, (batch,), generator=g)


DUMP_MAX_BYTES = 64_000_000


def host_outputs(named):
    """{name: tensor} -> float32 CPU copies, taken right after the timed leg (later legs keep updating the state)."""
    return {k: v.detach().float().cpu() for k, v in named.items()}


def dump_outputs(path, arrays):
    """Write {name: float32 CPU tensor} as <path>/<name>.npy.  When they hold more than DUMP_MAX_BYTES in all, every
    array is replaced by a fixed, seeded sample of its flattened elements (a share proportional to its size; the same
    positions on every run and every build), so that the dump stays within the limit."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    total = sum(t.numel() for t in arrays.values())
    budget = (DUMP_MAX_BYTES - 4096 * len(arrays)) // 4          # values, leaving room for the .npy headers
    for name, t in arrays.items():
        if total > budget:
            keep = max(1, t.numel() * budget // total)
            pick = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:keep].sort().values
            t = t.flatten()[pick]
        np.save(os.path.join(path, name + ".npy"), t.numpy())


# ----------------------------------------------------------------------------------------------------------------
# CPU arm: the reference algorithm (oracle port) on the host cores
# ----------------------------------------------------------------------------------------------------------------
def cpu_reference_steps(steps, warmup, batch, w=WORKLOAD):
    """Times oracle.fine_tune_step (fp32 restatement of the reference step) on `batch` images of the workload."""
    import torch
    from oracle import apla_oracle as O
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    base = {"vit_large": O.VIT_L14, "vit_small": O.VIT_S16}.get(w["arch"], O.VIT_B14)
    cfg = O.VitCfg(**base, n_classes=w["n_classes"], partial_size=w["partial_size"])
    sd = O.build_state(cfg, seed=0)
    images, labels = O.synthetic_batch(batch, w["img"], w["n_classes"])
    st = O.AdamWState()
    ts = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        O.fine_tune_step(sd, cfg, images, labels, st)
        ts.append(time.perf_counter() - t0)
    ts = ts[warmup:]
    sec = sum(ts) / len(ts)
    return dict(value=batch / sec, unit="images/s", cores=threads, kind="port",
                sample=f"oracle/apla_oracle.py fine_tune_step, {w['arch']}/{w['patch']} r={w['partial_size']} {w['img']}px fp32, "
                       f"batch {batch}, "
                       f"{len(ts)} steps after {warmup} warm-up, {sec * 1e3:.0f} ms/step"), sec


C1 = dict(arch="vit_small", img=224, table_img=224, patch=16, n_classes=555, partial_size=32, batch_per_gpu=8)


def run_reference(args):
    """The reference arm: the reference's algorithm (oracle port, `kind: "port"` -- /root/reference is a script tree that
    cannot be installed and does not exist on the GPU box) on the host cores, on OUR arm's metric / unit / config.  Each
    step is a bounded sample of the workload (8 images of the per-GPU batch); --steps / --warmup are honoured as given.
    Under torchrun only rank 0 works."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warmup = max(1, args.steps), max(0, args.warmup)
    w = WORKLOADS[args.workload]
    if "n_local" in w:
        print(json.dumps(dict(impl="reference", unavailable="the C4 self-supervised step has no CPU arm: its oracle "
                              "(oracle/ssl_oracle.py) is a parity checker for tiny shapes; ViT-L/14 x 640 crops x 65 536 "
                              "prototypes does not fit a bounded CPU sample")))
        return
    B = args.batch or w["batch_per_gpu"]
    sample = min(8, B)
    cb, sec = cpu_reference_steps(steps, warmup, batch=sample, w=w)
    line = dict(metric=METRIC, value=cb["value"], unit="images/s", n_gpus=args.gpus, steps=steps, warmup=warmup,
                ms_per_step=sec * 1e3, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32",
                data="synthetic", impl="reference", config=make_config(w, B, args.gpus),
                cpu_baseline=cb,
                e2e=dict(value=cb["value"], unit="images/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------------------------
def dominant_traffic(workload, B):
    """DRAM bytes (read + write) per launch of the dominant kernel: NOT measurable inside this process (it needs ncu's
    dram__bytes counters), so it is read from the committed summary of the round's `ncu --set full` capture of this same
    command (profiles/dominant_traffic.json: bytes per launch shape, weighted here by the step's launch counts), or null."""
    p = os.path.join(ROOT, "profiles", "dominant_traffic.json")
    if not os.path.exists(p) or workload not in ("c2", "c3") or B != 64:
        return None, None
    with open(p) as f:
        d = json.load(f)
    b = d["bytes_per_launch"]
    return (12 * b["qkv_fwd"] + 12 * b["fc1_dgrad"] + 11 * b["qkv_dgrad"]) / 35, d.get("source")


def time_dominant_kernel(eng, torch, rounds=3):
    """CUDA-event timing (torch's current stream = the launching stream) of the kernel with the largest share of the
    step, gemm2_kernel<256, EPI_BIAS> (21.6 % in profiles/launches_r1d_summary.txt): the plain 2-CTA tcgen05 GEMM that
    runs qkv forward [T,768]x[768,2304], fc1 dgrad [T,3072]x[3072,768] and qkv dgrad [T,2304]x[2304,768] -- timed
    on exactly those shapes in the step's 12 / 12 / 11 proportion, rotating over 4 operand sets so they come from
    HBM / L2 like in the step.  Also times the fc1 + GELU epilogue kernel (the single most expensive launch)."""
    from apla_b200 import ops
    sh = eng.shape
    T, D, Hd, L = sh["T"], sh["D"], sh["hidden"], sh["L"]
    bf = torch.bfloat16

    def mats(n, k):
        return [(torch.randn(n, k, device="cuda") * 0.02).to(bf) for _ in range(4)]
    x_d = [torch.randn(T, D, device="cuda").to(bf) for _ in range(2)]
    x_h = [torch.randn(T, Hd, device="cuda").to(bf) for _ in range(2)]
    x_q = [torch.randn(T, 3 * D, device="cuda").to(bf) for _ in range(2)]
    w_qkv, w_fc1t, w_qkvt = mats(3 * D, D), mats(D, Hd), mats(D, 3 * D)
    o_q = [torch.empty(T, 3 * D, device="cuda", dtype=bf) for _ in range(2)]
    o_d = [torch.empty(T, D, device="cuda", dtype=bf) for _ in range(2)]
    bias = torch.zeros(3 * D, device="cuda")
    plan = []      # (callable, flops) in the step's proportion
    for i in range(L):
        plan.append((lambda i=i: ops.gemm_bias(x_d[i % 2], w_qkv[i % 4], bias, out=o_q[i % 2]), 2.0 * T * 3 * D * D))
        plan.append((lambda i=i: ops.gemm_dgrad(x_h[i % 2], w_fc1t[i % 4], out=o_d[i % 2]), 2.0 * T * D * Hd))
        if i:
            plan.append((lambda i=i: ops.gemm_dgrad(x_q[i % 2], w_qkvt[i % 4], out=o_d[i % 2]), 2.0 * T * D * 3 * D))
    for fn, _ in plan:
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(rounds):
        for fn, _ in plan:
            fn()
    b.record()
    torch.cuda.synchronize()
    sec = a.elapsed_time(b) * 1e-3 / (rounds * len(plan))
    flops = sum(f for _, f in plan) / len(plan)
    dom = dict(kernel="g2::gemm2_kernel<256, EPI_BIAS> (qkv fwd / fc1 dgrad / qkv dgrad, 12:12:11)", launches=len(plan),
               us_per_launch=sec * 1e6, flops_per_launch=flops, tflops=flops / sec / 1e12)
    # the fc1 + GELU + saved-derivative epilogue kernel
    ws = mats(Hd, D)
    hs = [torch.empty(T, Hd, device="cuda", dtype=torch.float16) for _ in range(2)]
    gs = [torch.empty(T, Hd, device="cuda", dtype=bf) for _ in range(2)]
    b1 = torch.zeros(Hd, device="cuda")
    for i in range(4):
        ops.gemm_bias_gelu_dgelu(x_d[i % 2], ws[i], b1, d=hs[i % 2], g=gs[i % 2])
    torch.cuda.synchronize()
    a.record()
    for i in range(24):
        ops.gemm_bias_gelu_dgelu(x_d[i % 2], ws[i % 4], b1, d=hs[i % 2], g=gs[i % 2])
    b.record()
    torch.cuda.synchronize()
    sec1 = a.elapsed_time(b) * 1e-3 / 24
    fc1 = dict(kernel="g2::gemm2_kernel<256, EPI_BIAS_GELU_D> (Mlp.fc1 + GELU + saved GELU', 16448x3072x768)",
               us_per_launch=sec1 * 1e6, tflops=2.0 * T * D * Hd / sec1 / 1e12)
    return dom, fc1


def _dist_setup():
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device (B200); there is no CPU fallback for the product path")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return world, rank, local


def _timer(world):
    """-> timed(fn, steps, warmup): ms per step, CUDA events bracketed by barrier + synchronize, MAX over ranks."""
    import torch
    import torch.distributed as dist

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            fn()
        b.record()
        barrier()
        ms = torch.tensor([a.elapsed_time(b)], device="cuda")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()) / steps
    return timed


def _params_identical(eng, world):
    """Data-parallel self-check: after the timed steps every rank must hold bit-identical parameters and Adam moments
    (same initial state, same all-reduced gradients, same deterministic optimiser kernel)."""
    import torch
    import torch.distributed as dist
    if world == 1:
        return None
    torch.cuda.synchronize()
    sig = torch.stack([eng.params.double().sum(), eng.params.double().abs().sum(), eng.exp_avg.double().sum(),
                       eng.exp_avg_sq.double().sum(), eng.params[:: max(1, eng.n_arena // 4096)].double().pow(2).sum()])
    all_sig = [torch.empty_like(sig) for _ in range(world)]
    dist.all_gather(all_sig, sig)
    return bool(all(torch.equal(all_sig[0], t) for t in all_sig))


def run_gpu(args):
    import torch
    import torch.distributed as dist
    from apla_b200._lib import LIB
    from apla_b200.config import AplaConfig
    from apla_b200.engine import FineTuneEngine
    from apla_b200.flops import flops_per_image
    from apla_b200.hostvit import ARCHS, build_classifier

    world, rank, local = _dist_setup()
    if args.gpus != world:
        raise RuntimeError(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch N>1 through torch.distributed.run")
    w = WORKLOADS[args.workload]
    B = args.batch or w["batch_per_gpu"]
    timed = _timer(world)

    def build_engine(wl):
        # identical weights and APLA indices on every rank: same seed, same constructor order (SURVEY.md 8e)
        model = build_classifier(wl["arch"], img_size=wl["table_img"], patch_size=wl["patch"], n_classes=wl["n_classes"],
                                 apla_config=AplaConfig(wl["partial_size"]), seed=0)
        return FineTuneEngine(model, batch_size=B, img_size=wl["img"], device=f"cuda:{local}")

    eng = build_engine(w)
    images, labels = synthetic_batch(B, w["img"], w["n_classes"], rank=rank)
    images_pin, labels_pin = images.pin_memory(), labels.pin_memory()
    images_dev, labels_dev = images.cuda(), labels.cuda()

    sampler = ClockSampler(local) if rank == 0 else None
    n0 = LIB.load().apla_launch_count()
    eng.step(images_dev, labels_dev)
    launches_per_step = int(LIB.load().apla_launch_count() - n0)
    if sampler:
        sampler.start()
    # (the engine runs a buffer pair eagerly once, captures its CUDA graph on the second step and replays from the third:
    #  at least two untimed steps here, four for the two input slots of the end-to-end path)
    ms_step = timed(lambda: eng.step(images_dev, labels_dev), args.steps, max(2, args.warmup - 1))
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        # what the caller of eng.step() holds after the last timed step: loss, logits, trainable parameters and their
        # (clipped, rank-averaged) gradients
        outputs = host_outputs(dict(loss=eng.loss.reshape(1), logits=eng.logits,
                                    **{"param." + k: v for k, v in eng.named_params().items()},
                                    **{"grad." + k: v for k, v in eng.named_grads().items()}))
    ms_e2e = timed(lambda: eng.step_from_host(images_pin, labels_pin), args.steps, max(4, args.warmup // 2))
    loss = eng.drain()
    if loss is None:
        loss = float(eng.loss.item())
    # sustained leg: the driver's 20 steps are a 0.16 s burst at boost clocks; the same step for >= 2.5 s (power-capped)
    sus_sampler = ClockSampler(local) if rank == 0 else None
    n_sus = max(args.steps, int(2500.0 / ms_step) + 1) if args.sustained else 0
    ms_sus = None
    if n_sus:
        if sus_sampler:
            sus_sampler.start()
        ms_sus = timed(lambda: eng.step(images_dev, labels_dev), n_sus, 0)
        sus_clocks = sus_sampler.stop() if sus_sampler else None
    dp_ok = _params_identical(eng, world)

    # BASELINE.json configs[2] (partial_size = 768, a 30 MB gradient arena) through the same engine at this N: the
    # multi-GPU configuration the baseline names; `value` above stays on configs[1] so that N = 1 is the headline metric
    c3 = None
    if args.workload == "c2" and not args.no_c3:
        w3 = WORKLOADS["c3"]
        eng3 = build_engine(w3)
        ms3 = timed(lambda: eng3.step(images_dev, labels_dev), args.steps, max(3, args.warmup - 1))
        c3 = dict(workload=describe_workload(w3), value=B * world / (ms3 * 1e-3), unit="images/s", per_gpu=B / (ms3 * 1e-3),
                  ms_per_step=ms3, n_gpus=world, global_batch=B * world, grad_arena_bytes=eng3.n_arena * 4,
                  params_identical_across_ranks=_params_identical(eng3, world))
        del eng3

    if rank == 0:
        peaks = load_peaks()
        a = ARCHS[w["arch"]]
        f_fwd, f_bwd = flops_per_image(a.embed_dim, a.depth, w["patch"], w["img"], w["partial_size"], w["n_classes"])
        flops_step_ref = (f_fwd + f_bwd) * B                      # the reference's dense algorithm (SURVEY App. B)
        e_fwd, e_bwd = flops_per_image(a.embed_dim, a.depth, w["patch"], w["img"], w["partial_size"], w["n_classes"],
                                       cls_only_last_block=int(eng.cls_only_last_block))
        flops_step = (e_fwd + e_bwd) * B                          # what this engine executes (last block: CLS rows)
        achieved = flops_step / (ms_step * 1e-3) / 1e12
        dom, fc1 = time_dominant_kernel(eng, torch)
        traffic, traffic_src = dominant_traffic(args.workload, B)
        step = dict(scope="whole step (all kernels); EXECUTED algorithmic FLOPs: SURVEY.md App. B minus the "
                          "last block's per-token work on non-CLS tokens, which the engine proves dead "
                          "and does not run (DESIGN.md section 5)",
                    achieved=achieved, peak=peaks["tflops_sustained"], unit="TFLOP/s",
                    frac=achieved / peaks["tflops_sustained"], frac_of_burst=achieved / peaks["tflops_burst"],
                    note="`achieved` is the (burst) timed region of --steps; sustained_* is the same step run for >= 2.5 s",
                    flops_per_step=flops_step, flops_per_step_reference_dense=flops_step_ref,
                    frac_reference_dense_flops=flops_step_ref / (ms_step * 1e-3) / 1e12 / peaks["tflops_sustained"])
        if ms_sus is not None:
            sus = flops_step / (ms_sus * 1e-3) / 1e12
            step.update(sustained_steps=n_sus, sustained_ms_per_step=ms_sus,
                        sustained_images_per_s=B * world / (ms_sus * 1e-3), sustained_achieved=sus,
                        sustained_frac=sus / peaks["tflops_sustained"],
                        sustained_frac_reference_dense_flops=flops_step_ref / (ms_sus * 1e-3) / 1e12
                        / peaks["tflops_sustained"], sustained_clocks=sus_clocks)
        line = dict(
            metric=METRIC, value=B * world / (ms_step * 1e-3), unit="images/s", n_gpus=world, steps=args.steps,
            warmup=args.warmup, ms_per_step=ms_step, higher_is_better=True, scaling="weak", vs_baseline=None,
            dtype="bf16", data="synthetic", per_gpu=B / (ms_step * 1e-3), loss=loss,
            config=make_config(w, B, world),
            # dominant kernel (largest share of the step), algorithmic FLOPs 2*M*N*K per launch / live CUDA-event time;
            # peak = measured burst cuBLAS bf16 (kernel timed alone); `step` = the whole step against the sustained peak
            roofline=dict(bound="tensor", kernel=dom["kernel"], achieved=dom["tflops"], peak=peaks["tflops_burst"],
                          unit="TFLOP/s", frac=dom["tflops"] / peaks["tflops_burst"],
                          peak_source=f"{peaks['source']} MEASURED_PEAKS.json bf16_tflops (burst)",
                          us_per_launch=dom["us_per_launch"], flops_per_launch=dom["flops_per_launch"],
                          launches_timed=dom["launches"], traffic=traffic,
                          traffic_note=(f"dram read+write bytes per launch; not a live counter: {traffic_src}"
                                        if traffic is not None else "no ncu capture for this shape"),
                          fc1_gelu_kernel=dict(**fc1, frac=fc1["tflops"] / peaks["tflops_burst"]), step=step),
            e2e=dict(value=B * world / (ms_e2e * 1e-3), unit="images/s", ms_per_step=ms_e2e,
                     h2d_bytes_per_step=images_pin.numel() * 4 + labels_pin.numel() * 8, d2h_bytes_per_step=4),
            gpu_launches=launches_per_step * args.steps, gpu_launches_per_step=launches_per_step, clocks=clocks)
        if dp_ok is not None:
            line["dp_check"] = dict(params_identical_across_ranks=dp_ok)
        if c3 is not None:
            line["c3"] = c3
        if world == 1 and not args.no_cpu:
            cb, _ = cpu_reference_steps(steps=3, warmup=1, batch=min(8, w["batch_per_gpu"]), w=w)
            line["cpu_baseline"] = cb
            if args.workload == "c2":
                # BASELINE.json configs[0] / BASELINE.md section 3: the reference path on C1 exactly (ViT-S/16, r = 32, batch 8)
                c1, _ = cpu_reference_steps(steps=6, warmup=2, batch=8, w=C1)
                line["cpu_baseline_c1"] = c1
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ----------------------------------------------------------------------------------------------------------------
# C4: the DINOv2 self-supervised APLA adaptation step (module-level path: SSLMetaArch + DINOHead + loss classes)
# ----------------------------------------------------------------------------------------------------------------
def ssl_batch(B, w, seed=1234, mask_prob=0.5, ratio=(0.1, 0.5)):
    """Synthetic stand-in for `collate_data_and_cast` (src/self_supervised/dinov2/dinov2_utils.py:21-62): every other
    global crop is masked at a ratio drawn uniformly from `ratio` (uniform random positions instead of the block-wise
    generator)."""
    import torch
    g = torch.Generator().manual_seed(seed)
    P = (w["img"] // w["patch"]) ** 2
    glob = torch.randn(2 * B, 3, w["img"], w["img"], generator=g)
    loc = torch.randn(w["n_local"] * B, 3, w["local_img"], w["local_img"], generator=g)
    masks = torch.zeros(2 * B, P, dtype=torch.bool)
    for i in range(2 * B):
        if float(torch.rand(1, generator=g)) < mask_prob:
            n = int(P * (ratio[0] + (ratio[1] - ratio[0]) * float(torch.rand(1, generator=g))))
            masks[i, torch.randperm(P, generator=g)[:n]] = True
    idx = masks.flatten().nonzero().flatten()
    mw = (1 / masks.sum(-1).clamp(min=1.0)).unsqueeze(-1).expand_as(masks)[masks]
    return {"collated_global_crops": glob, "collated_local_crops": loc, "collated_masks": masks,
            "mask_indices_list": idx, "masks_weight": mw, "upperbound": int(idx.shape[0]),
            "n_masked_patches": torch.full((1,), idx.shape[0], dtype=torch.long)}


def run_ssl(args):
    """One step = Dinov2Trainer.global_step (src/self_supervised/dinov2/trainer.py:106-162): teacher forward, student
    forward over the packed multi-crop batch, DINO + iBOT + KoLeo objective, backward (projection rows + head), gradient
    mean over ranks (DDP, as the reference wraps the student), clip, AdamW, teacher EMA; the two centre statistics are
    all-reduced asynchronously inside the loss classes (dino_clstoken_loss.py:85, ibot_patch_loss.py:132)."""
    import contextlib
    import io
    import torch
    import torch.distributed as dist
    from apla_b200._lib import LIB
    from apla_b200.config import AplaConfig
    from apla_b200.dinov2 import DINOHead
    from apla_b200.hostdino import SSLMetaArch, build_dino_backbone
    from apla_b200.hostvit import ARCHS

    world, rank, local = _dist_setup()
    if args.gpus != world:
        raise RuntimeError(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch N>1 through torch.distributed.run")
    w = WORKLOADS["c4"]
    B = args.batch or w["batch_per_gpu"]
    dev = f"cuda:{local}"
    timed = _timer(world)
    torch.manual_seed(0)
    cfg = AplaConfig(w["partial_size"])
    with contextlib.redirect_stdout(io.StringIO()):
        student = build_dino_backbone(w["arch"], img_size=w["table_img"], patch_size=w["patch"], apla_config=cfg)
        inds = [b.attn.inds.clone() for b in student.blocks]
        teacher = build_dino_backbone(w["arch"], img_size=w["table_img"], patch_size=w["patch"], apla_config=cfg,
                                      indices=inds)
    teacher.load_state_dict(student.state_dict())                     # models.py:138
    D = ARCHS[w["arch"]].embed_dim
    sh = DINOHead(D, w["n_classes"], nlayers=3, hidden_dim=w["head_hidden"], bottleneck_dim=w["head_bottleneck"])
    th = DINOHead(D, w["n_classes"], nlayers=3, hidden_dim=w["head_hidden"], bottleneck_dim=w["head_bottleneck"])
    th.load_state_dict(sh.state_dict())
    model = SSLMetaArch(student, teacher, sh, th, w["n_classes"], n_local_crops=w["n_local"],
                        fused_objective=not args.per_term_losses).to(dev)
    trainable = [p for p in model.student.parameters() if p.requires_grad]
    opt = torch.optim.AdamW(trainable, lr=3e-5, weight_decay=1e-5)
    batch_host = ssl_batch(B, w, seed=1234 + rank)
    batch_pin = {k: (v.pin_memory() if torch.is_tensor(v) else v) for k, v in batch_host.items()}
    batch_dev = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in batch_host.items()}
    flat = peer = None
    if world > 1:
        # the reference wraps the student in DDP (dinov2/wrappers.py:76-77); here the trainable gradients are reduced as
        # ONE flat buffer after backward (mean) -- by the library's own NVLink all-reduce kernel over symmetric memory
        # (apla_grad_arena_allreduce; 49 M parameters = 195 MB), NCCL if symmetric memory is unavailable
        from apla_b200.dp import make_peer_arena
        n_flat = sum(p.numel() for p in trainable)
        peer = make_peer_arena(n_flat, dev)
        ok = torch.tensor([1 if peer is not None else 0], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if int(ok.item()) == 0:
            peer = None
        flat = peer.grads() if peer is not None else torch.zeros(n_flat, device=dev)

    def step(batch):
        opt.zero_grad(set_to_none=True)
        loss, _ = model(batch, teacher_temp=0.04)
        loss.backward()
        if world > 1:
            torch.cat([p.grad.reshape(-1) for p in trainable], out=flat)
            if peer is not None:
                peer.all_reduce(0, flat.numel(), 0, ctas=64)
            else:
                dist.all_reduce(flat)
            flat.mul_(1.0 / world)
            o = 0
            for p in trainable:
                p.grad.copy_(flat[o:o + p.numel()].view_as(p.grad))
                o += p.numel()
        torch.nn.utils.clip_grad_norm_(trainable, 3.0)
        opt.step()
        model.update_teacher(0.994)
        return loss

    def step_e2e():
        b = {k: (v.to(dev, non_blocking=True) if torch.is_tensor(v) else v) for k, v in batch_pin.items()}
        return float(step(b))                                         # loss read back to the host every step

    last = {}

    def timed_step():
        last["loss"] = step(batch_dev).detach()

    sampler = ClockSampler(local) if rank == 0 else None
    step(batch_dev)
    n0 = LIB.load().apla_launch_count()
    step(batch_dev)
    launches_per_step = int(LIB.load().apla_launch_count() - n0)
    if sampler:
        sampler.start()
    ms_step = timed(timed_step, args.steps, max(1, args.warmup - 2))
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        # what the caller of the step holds after the last timed step: the loss, the student's trainable parameters
        # after AdamW and their clipped gradients
        named = [(n, p) for n, p in model.student.named_parameters() if p.requires_grad]
        outputs = host_outputs(dict(loss=last["loss"].reshape(1), **{"param." + n: p for n, p in named},
                                    **{"grad." + n: p.grad for n, p in named}))
    ms_e2e = timed(step_e2e, args.steps, 1)
    loss = float(step(batch_dev))
    if rank == 0:
        peaks = load_peaks()
        achieved = GFLOP_PER_IMAGE_C4 * 1e9 * B / (ms_step * 1e-3) / 1e12
        h2d = sum(v.numel() * v.element_size() for v in batch_pin.values() if torch.is_tensor(v))
        ssl_kernels = None
        p = os.path.join(ROOT, "profiles", "ssl_kernels_r2.jsonl")
        if os.path.exists(p):
            with open(p) as f:
                rows = [json.loads(x) for x in f if x.strip().startswith("{") and "kernel" in x]
            ssl_kernels = {r["kernel"]: dict(us=r["us"], gbs=r["gbs"], frac_of_hbm_peak=r["frac_of_hbm_peak"]) for r in rows}
        line = dict(
            metric=METRIC + " -- configs[3]: ViT-L/14 DINOv2 SSL APLA adaptation images/sec", value=B * world / (ms_step * 1e-3),
            unit="images/s", n_gpus=world, steps=args.steps, warmup=args.warmup, ms_per_step=ms_step,
            higher_is_better=True, scaling="weak", vs_baseline=None, dtype="bf16", data="synthetic",
            per_gpu=B / (ms_step * 1e-3), loss=loss, config=make_config(w, B, world),
            roofline=dict(bound="tensor", kernel="whole step (block path GEMMs / attention + DINO head GEMMs + HBM-bound "
                                                 "objective kernels)", achieved=achieved, peak=peaks["tflops_sustained"],
                          unit="TFLOP/s", frac=achieved / peaks["tflops_sustained"],
                          frac_of_burst=achieved / peaks["tflops_burst"],
                          peak_source=f"{peaks['source']} MEASURED_PEAKS.json bf16_tflops_sustained",
                          flops_per_image=GFLOP_PER_IMAGE_C4 * 1e9, traffic=None,
                          hbm_bound_kernels=ssl_kernels,
                          hbm_bound_kernels_note="isolated CUDA-event timings of the objective's row kernels at these shapes "
                                                 "(tools/bench_ssl_kernels.py, profiles/ssl_kernels_r2.jsonl) against "
                                                 "the measured HBM copy peak"),
            e2e=dict(value=B * world / (ms_e2e * 1e-3), unit="images/s", ms_per_step=ms_e2e, h2d_bytes_per_step=h2d,
                     d2h_bytes_per_step=4),
            objective="per-term loss classes" if args.per_term_losses else "fused head + apla_ssl_objective",
            grad_allreduce=("native apla_grad_arena_allreduce" if peer is not None else "nccl") if world > 1 else None,
            masked_patches=int(batch_host["mask_indices_list"].shape[0]),
            trainable_params=sum(p.numel() for p in trainable), peak_hbm_gb=round(torch.cuda.max_memory_allocated() / 1e9, 1),
            gpu_launches=launches_per_step * args.steps, gpu_launches_per_step=launches_per_step, clocks=clocks)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps of every timed leg")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch override (default: the workload's 64)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS),
                    help="c2 = BASELINE.json configs[1] (the metric's configuration, default); c3 / c5 / vitl: other shapes "
                         "through the engine; c4 = configs[3], the DINOv2 self-supervised step (module-level path)")
    ap.add_argument("--no-c3", action="store_true", help="skip the nested configs[2] (partial_size 768) leg of the c2 line")
    ap.add_argument("--sustained", action="store_true",
                    help="add a leg that runs the step for >= 2.5 s, however many steps that takes (roofline.step.sustained_*)")
    ap.add_argument("--no-sustained", dest="sustained", action="store_false", help="no sustained leg (the default)")
    ap.add_argument("--per-term-losses", action="store_true",
                    help="c4: the reference's call structure (one loss-class call per term) instead of the fused objective")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed (loss, logits, trainable "
                         "parameters and gradients) as DIR/<name>.npy, float32, at most 64 MB in all (larger outputs: "
                         "a fixed, seeded sample)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of this project's CUDA path; --impl reference has none")
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "c4":
        run_ssl(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()

"""Forward-only evaluation on the B200: `FineTuneEngine.predict / embed / evaluate` (csrc/engine.cu `apla_engine_infer`),
the no-grad path of `FusedAplaBlock` (`apla_block_fwd_infer`) and the fc1 epilogue that writes gelu(h) only, against
 (a) the training forward on the same weights and inputs (bitwise where the launch sequence is the same),
 (b) the golden vectors of the unmodified reference and the fp32 CPU oracle (relative error <= 1e-2)."""
import pytest
import torch
import torch.nn.functional as F

from helpers import build_case, rel, synthetic_batch

pytestmark = pytest.mark.gpu


def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")


def _engine(model, batch, img, **kw):
    _need_gpu()
    from apla_b200.engine import FineTuneEngine
    return FineTuneEngine(model, batch_size=batch, img_size=img, **kw)


def _tiny_oracle():
    from oracle import apla_oracle as O
    cfg = O.VitCfg(embed_dim=128, depth=2, num_heads=2, patch_size=14, img_size=56, n_classes=10, partial_size=16)
    sd = O.build_state(cfg, seed=0)
    O.perturb_state(sd)
    return O, cfg, sd


@pytest.mark.parametrize("mode", [0, 1, 2])
@pytest.mark.parametrize("name", ["tiny_r16", "c1_vits16_r32", "c2_vitb14_r8"])
def test_predict_equals_training_forward(name, mode):
    model, meta, arr = build_case(name)
    m = meta["meta"]
    eng = _engine(model, m["batch"], m["img"], cls_only_last_block=mode)
    images, labels = synthetic_batch(m["batch"], m["img"], m["n_classes"])
    images = images.cuda()
    eng.forward(images, labels.cuda())
    want = eng.logits.clone()
    got = eng.predict(images)
    torch.cuda.synchronize()
    assert got.dtype == torch.float32 and got.shape == want.shape and got.data_ptr() != eng.logits.data_ptr()
    assert torch.equal(got, want)
    assert rel(got, arr["s0/logits"]) <= 1e-2, rel(got, arr["s0/logits"])


def test_predict_partial_and_chunked_batches():
    """Capacity 8: 3 images (one partial chunk), 8 (one full chunk) and 19 (8 + 8 + 3) against the rows of one
    19-image training forward, and against the live oracle."""
    O, cfg, sd = _tiny_oracle()
    model, _, _ = build_case("tiny_r16")
    eng = _engine(model, 19, 56, eval_batch_size=8)
    images, labels = synthetic_batch(19, 56, 10, seed=77)
    eng.forward(images.cuda(), labels.cuda())
    full = eng.logits.clone()
    ref = O.forward_logits(sd, cfg, images)
    for n in (3, 8, 19):
        got = eng.predict(images[:n].cuda())
        assert got.shape == (n, 10)
        assert rel(got, full[:n]) <= 2e-3, (n, rel(got, full[:n]))
        assert rel(got, ref[:n]) <= 1e-2, (n, rel(got, ref[:n]))
    # host-resident images take the same path chunk by chunk
    assert torch.equal(eng.predict(images[:19].pin_memory()), eng.predict(images[:19].cuda()))


def test_embed_is_the_final_norm_cls_row():
    O, cfg, sd = _tiny_oracle()
    model, _, _ = build_case("tiny_r16")
    eng = _engine(model, 4, 56, eval_batch_size=3)
    images, _ = synthetic_batch(5, 56, 10, seed=31)
    emb = eng.embed(images.cuda())
    logits = eng.predict(images.cuda())
    torch.cuda.synchronize()
    assert emb.shape == (5, 128) and emb.dtype == torch.float32
    assert torch.equal(emb, emb.bfloat16().float())                   # fp32 values of the bf16 the head reads
    want = O.forward_tokens(sd, cfg, images)[:, 0]
    assert rel(emb, want) <= 1e-2, rel(emb, want)
    p = eng.named_params()
    head = emb.double() @ p["fc.weight"].double().t() + p["fc.bias"].double()
    assert rel(head, logits) <= 1e-5, rel(head, logits)


def test_evaluate_matches_cross_entropy_and_argmax():
    model, _, _ = build_case("tiny_r16")
    eng = _engine(model, 4, 56)
    images, labels = synthetic_batch(11, 56, 10, seed=5)
    logits = eng.predict(images.cuda()).double().cpu()
    want_loss = float(F.cross_entropy(logits, labels))
    want_top1 = float((logits.argmax(1) == labels).double().mean())
    sizes = [(0, 4), (4, 8), (8, 11)]                                 # the last batch is partial
    dev = [(images[a:b].cuda(), labels[a:b].cuda()) for a, b in sizes]
    host = [(images[a:b].pin_memory(), labels[a:b].pin_memory()) for a, b in sizes]
    for batches in (dev, host):
        out = eng.evaluate(iter(batches))
        assert out["n"] == 11
        assert abs(out["loss"] - want_loss) <= 1e-5 * abs(want_loss), (out, want_loss)
        assert abs(out["top1"] - want_top1) <= 1e-5 * max(want_top1, 1e-12) + 1e-12, (out, want_top1)
    # a batch where every prediction is right, and one where the first of two equal maxima decides
    C = 10
    lg = torch.zeros(3, C, device="cuda")
    lg[0, 7] = 5.0
    lg[1, 2] = lg[1, 5] = 3.0
    lg[2, 0] = 1.0
    acc = torch.zeros(2, device="cuda")
    from apla_b200._lib import LIB, ptr, stream
    lab = torch.tensor([7, 5, 0], device="cuda")
    LIB.call("apla_eval_accumulate", ptr(lg), ptr(lab), 3, C, ptr(acc), stream())
    torch.cuda.synchronize()
    assert float(acc[1]) == 2.0                                       # row 1: argmax is 2 (first maximum), label 5
    assert abs(float(acc[0]) - float(F.cross_entropy(lg, lab, reduction="sum"))) <= 1e-5 * float(acc[0])


def test_predict_leaves_the_training_state_alone():
    model, meta, _ = build_case("tiny_r16")
    eng = _engine(model, 4, 56, eval_batch_size=3)
    images, labels = synthetic_batch(4, 56, 10)
    images, labels = images.cuda(), labels.cuda()
    eng.step(images, labels)                 # eager
    eng.step(images, labels)                 # captured, replayed
    torch.cuda.synchronize()
    assert len(eng._graphs) == 1
    bufs = list(eng._keep) + [eng.params, eng.grads, eng.exp_avg, eng.exp_avg_sq, eng.logits, eng.loss, eng.xs]
    # bytes, not values: rows the step never writes (the last block's non-CLS rows of hpre, ...) may hold NaN patterns
    snap = [t.view(torch.uint8).clone() for t in bufs]
    other, _ = synthetic_batch(7, 56, 10, seed=3)
    eng.predict(other.cuda())
    eng.embed(other.cuda())
    torch.cuda.synchronize()
    for i, (t, s) in enumerate(zip(bufs, snap)):
        assert torch.equal(t.view(torch.uint8), s), f"training buffer {i} {tuple(t.shape)} {t.dtype} changed"
    p = eng.params.clone()
    eng.step(images, labels)                 # replay of the graph captured before predict
    torch.cuda.synchronize()
    assert len(eng._graphs) == 1
    assert torch.isfinite(eng.loss).all() and float((eng.params - p).norm()) > 0
    # and predict follows the new weights (chunks of 3 + 1 images against one forward of 4)
    eng.forward(images, labels)
    assert rel(eng.predict(images), eng.logits) <= 2e-3


def _peak_of(fn):
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    out = fn()
    torch.cuda.synchronize()
    return out, torch.cuda.max_memory_allocated() - base


@pytest.mark.parametrize("name,l,B,N", [("tiny_r16", 1, 3, 257), ("c5_vitb14_518_r768", 3, 1, 1370)])
def test_no_grad_fused_block_dense(name, l, B, N):
    _need_gpu()
    from apla_b200.apla import fuse_apla_blocks
    model, _, _ = build_case(name)
    fuse_apla_blocks(model.cuda())
    blk = model.backbone.blocks[l]
    D, Hd = blk.attn.dim, blk.mlp.fc1.out_features
    x = torch.randn(B, N, D, generator=torch.Generator().manual_seed(3)).cuda()
    xg = x.clone().requires_grad_(True)
    blk(xg)                                                           # warm the weight caches
    with torch.no_grad():
        blk(x)
    y_grad, peak_grad = _peak_of(lambda: blk(xg))
    assert y_grad.grad_fn is not None
    with torch.no_grad():
        y, peak = _peak_of(lambda: blk(x))
    assert y.grad_fn is None and torch.equal(y, y_grad.detach())
    assert peak_grad - peak >= B * N * Hd * 2, (peak_grad, peak)
    # grad enabled but nothing requires grad: the same forward-only path
    at = blk.attn
    at.proj_weight1.requires_grad_(False)
    at.proj_bias1.requires_grad_(False)
    try:
        y2 = blk(x)
        assert y2.grad_fn is None and torch.equal(y2, y)
    finally:
        at.proj_weight1.requires_grad_(True)
        at.proj_bias1.requires_grad_(True)


def test_no_grad_fused_block_packed_crops():
    _need_gpu()
    from apla_b200.apla import fuse_apla_blocks
    model, _, _ = build_case("tiny_r16")
    fuse_apla_blocks(model.cuda())
    b0, b1 = model.backbone.blocks[0], model.backbone.blocks[1]
    g = torch.Generator().manual_seed(8)
    crops = [torch.randn(2, 257, 128, generator=g).cuda(), torch.randn(4, 50, 128, generator=g).cuda()]
    want = b1(b0([c.clone().requires_grad_(True) for c in crops]))
    with torch.no_grad():
        mid = b0(crops)                          # a PackedCropList handed on to the next block without repacking
        got = b1(mid)
    assert [o.shape for o in got] == [c.shape for c in crops]
    for a, b in zip(got, want):
        assert a.grad_fn is None and torch.equal(a, b.detach())


def test_teacher_backbone_output_unchanged():
    """The DINOv2 teacher runs under torch.no_grad(): its fused blocks take the forward-only path and must give exactly
    what the training forward gives (global crops as a list: packed, block-diagonal)."""
    _need_gpu()
    from apla_b200.config import AplaConfig
    from apla_b200.hostdino import build_dino_backbone
    from apla_b200.hostvit import VitArch
    torch.manual_seed(2)
    teacher = build_dino_backbone(VitArch(128, 2, 2), img_size=56, patch_size=14, apla_config=AplaConfig(16)).cuda()
    g = torch.Generator().manual_seed(9)
    x = torch.randn(4, 3, 56, 56, generator=g).cuda()
    crops = [torch.randn(2, 3, 56, 56, generator=g).cuda(), torch.randn(3, 3, 42, 42, generator=g).cuda()]
    with torch.enable_grad():
        want = teacher(x, is_training=True)
        want_l = teacher(crops, [None, None], is_training=True)
    with torch.no_grad():
        got = teacher(x, is_training=True)
        got_l = teacher(crops, [None, None], is_training=True)
    assert want["x_norm_clstoken"].grad_fn is not None and got["x_norm_clstoken"].grad_fn is None
    for k in ("x_norm_clstoken", "x_norm_patchtokens", "x_prenorm"):
        assert torch.equal(got[k], want[k].detach()), k
        for a, b in zip(got_l, want_l):
            assert torch.equal(a[k], b[k].detach()), k


@pytest.mark.parametrize("M,N,K", [(16448, 3072, 768), (32896, 4096, 1024), (1000, 3072, 768)])
def test_gelu_only_epilogue_is_bitwise_the_training_g(M, N, K):
    _need_gpu()
    from apla_b200._lib import LIB, ptr, require_device, stream
    require_device()
    g = torch.Generator(device="cuda").manual_seed(M)
    A = torch.randn(M, K, device="cuda", generator=g).bfloat16()
    W = (torch.randn(N, K, device="cuda", generator=g) * K ** -0.5).bfloat16()
    bias = torch.randn(N, device="cuda", generator=g) * 0.5
    d = torch.empty(M, N, device="cuda", dtype=torch.float16)
    g_train = torch.empty(M, N, device="cuda", dtype=torch.bfloat16)
    g_only = torch.full((M, N), float("nan"), device="cuda", dtype=torch.bfloat16)
    LIB.call("apla_gemm_bias_gelu_dgelu_fwd", ptr(A), K, ptr(W), K, ptr(bias), ptr(d), ptr(g_train), N, M, N, K, stream())
    LIB.call("apla_gemm_bias_gelu_only_fwd", ptr(A), K, ptr(W), K, ptr(bias), ptr(g_only), N, M, N, K, stream())
    torch.cuda.synchronize()
    assert torch.equal(g_only.view(torch.int16), g_train.view(torch.int16))
    h = A[:64].float() @ W.float().t() + bias                        # and it is gelu(h)
    assert rel(g_only[:64], F.gelu(h)) <= 1e-2

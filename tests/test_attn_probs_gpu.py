"""Attention probabilities on the B200: the tcgen05 kernel `apla_attn_probs` (csrc/attention_probs.cu), the opt-in
`(out, attn)` of `APLA_Attention` and `FusedAplaBlock.forward(x, return_attention=True)` under
`apla_b200.apla.attention_probabilities`, and `FineTuneEngine.cls_attention`, against fp32 torch restatements of the
reference softmax (appla_attn.py:56-60) and the oracle.
Bars (BASELINE.json north_star): relative error <= 1e-2 and cosine >= 0.999 per tensor, rows summing to 1 within 1e-2."""
import types

import pytest
import torch
import torch.nn.functional as F

from helpers import build_case, cosine, rel, synthetic_batch

pytestmark = pytest.mark.gpu

CANARY = 12345.0


def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")


def _probs_ref(qkv, B, N, H, scale):
    """fp32 [B,H,N,N] softmax of appla_attn.py:56-60 on the bf16 qkv, and v [B,H,N,64]."""
    t = qkv.float().reshape(B, N, 3, H, 64).permute(2, 0, 3, 1, 4)
    return ((t[0] @ t[1].transpose(-2, -1)) * scale).softmax(-1), t[2]


def _check(p, ref):
    assert rel(p, ref) <= 1e-2, rel(p, ref)
    assert cosine(p, ref) >= 0.999, cosine(p, ref)
    err = float((p.double().sum(-1) - 1).abs().max())
    assert err <= 1e-2, err


def _run_into_canary_buffer(ops, qkv, lse, H, scale, B, N, q_rows):
    n = B * H * q_rows * N
    buf = torch.full((n + 4096,), float("nan"), device="cuda")
    buf[n:] = CANARY
    ops.attn_probs(qkv, lse, H, scale, B, N, q_rows=q_rows, out=buf)
    torch.cuda.synchronize()
    p = buf[:n].view(B, H, q_rows, N)
    assert not torch.isnan(p).any(), "a probability was left unwritten"
    assert bool((buf[n:] == CANARY).all()), "the kernel wrote past [B, H, q_rows, N]"
    return p


@pytest.mark.parametrize("q_rows", ["N", 1])
@pytest.mark.parametrize("B,N,H", [(2, 257, 12), (30, 257, 12), (3, 197, 6), (1, 1370, 12), (4, 50, 16), (5, 17, 2),
                                   (2, 272, 2), (2, 129, 2)])
def test_kernel_matches_the_fp32_softmax(B, N, H, q_rows):
    _need_gpu()
    from apla_b200 import ops
    q_rows = N if q_rows == "N" else q_rows
    g = torch.Generator(device="cuda").manual_seed(B * N + H)
    qkv = torch.randn(B * N, 3 * H * 64, device="cuda", generator=g).bfloat16()
    scale = 64 ** -0.5
    out, lse = ops.attn_fwd(qkv, H, scale, B, N)
    p = _run_into_canary_buffer(ops, qkv, lse, H, scale, B, N, q_rows)
    ref, v = _probs_ref(qkv, B, N, H, scale)
    _check(p, ref[:, :, :q_rows])
    # probs . V against the forward's own output
    pv = (p @ v).transpose(1, 2).reshape(B, q_rows, H * 64)
    o = out.float().view(B, N, H * 64)[:, :q_rows]
    assert rel(pv, o) <= 1e-2, rel(pv, o)


@pytest.mark.parametrize("B,N,H", [(3, 257, 12), (2, 1370, 2), (4, 50, 4)])
def test_kernel_cls_row_from_the_cls_forward(B, N, H):
    """q_rows = 1 on the lse of the CLS-only forward, which writes rows b*N only: no other row of lse is read."""
    _need_gpu()
    from apla_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(B + N + H)
    qkv = torch.randn(B * N, 3 * H * 64, device="cuda", generator=g).bfloat16()
    lse = torch.full((B * N, H), float("nan"), device="cuda")
    _, lse = ops.attn_cls_fwd(qkv, H, 0.125, B, N, lse=lse)
    p = _run_into_canary_buffer(ops, qkv, lse, H, 0.125, B, N, 1)
    ref, _ = _probs_ref(qkv, B, N, H, 0.125)
    _check(p, ref[:, :, :1])


def _attention_module(r, dim, heads, seed):
    from apla_b200.apla import APLA_Attention
    from apla_b200.config import AplaConfig
    torch.manual_seed(seed)
    mod = APLA_Attention(AplaConfig(r), dim, num_heads=heads, qkv_bias=True)
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for p in mod.parameters():
            p.copy_(torch.randn(p.shape, generator=g) * (0.05 if p.dim() == 2 else 0.1))
    return mod.cuda()


@pytest.mark.parametrize("B,N,dim,heads,r", [(3, 257, 128, 2, 16), (2, 197, 384, 6, 32)])
def test_apla_attention_returns_probabilities_inside_the_context(B, N, dim, heads, r):
    _need_gpu()
    from apla_b200.apla import attention_probabilities
    from oracle import apla_oracle as O
    mod = _attention_module(r, dim, heads, seed=B * N)
    g = torch.Generator(device="cuda").manual_seed(5)
    x = torch.randn(B, N, dim, device="cuda", generator=g)
    dy = torch.randn(B, N, dim, device="cuda", generator=g)

    def run(ctx):
        xg = x.clone().requires_grad_(True)
        mod.zero_grad(set_to_none=True)
        if ctx:
            with attention_probabilities(mod):
                out, attn = mod(xg)
        else:
            out, attn = mod(xg)
        out.backward(dy)
        return out.detach(), attn, xg.grad, mod.proj_weight1.grad.clone(), mod.proj_bias1.grad.clone()

    base = run(False)
    got = run(True)
    assert base[1] is None
    assert torch.equal(got[0], base[0]) and torch.equal(got[2], base[2])           # out, x.grad: bit for bit
    # the weight and bias gradients sum partials with fp32 atomics (apla_proj_wgrad_gather, apla_colsum): their last
    # bits vary from call to call with or without the context
    for a, b in zip(got[3:], base[3:]):
        assert rel(a, b) <= 1e-5, rel(a, b)
    attn = got[1]
    assert attn.dtype == torch.float32 and attn.shape == (B, heads, N, N) and attn.is_contiguous()
    assert not attn.requires_grad and attn.grad_fn is None
    qkv = F.linear(x, mod.qkv.weight.float(), mod.qkv.bias.float())
    _check(attn, O.softmax_attention(qkv, B, N, heads, float(mod.scale))[1])
    # None again after the block, also when it was left through an exception
    assert mod(x)[1] is None
    with pytest.raises(ValueError):
        with attention_probabilities(mod):
            raise ValueError("leave the block")
    assert mod(x)[1] is None


def _oracle_last_attention(model, images):
    """fp32 oracle (oracle/apla_oracle.py) of the last block's attention probabilities [B,H,N,N] on the model's weights."""
    from oracle import apla_oracle as O
    bb = model.backbone
    L, H = len(bb.blocks), bb.blocks[0].attn.num_heads
    sd = {k: v.detach().cpu().float() if v.is_floating_point() else v.detach().cpu() for k, v in model.state_dict().items()}
    cfg = types.SimpleNamespace(patch_size=bb.patch_embed.patch_size)
    x = O.embed(sd, cfg, images.cpu())
    eps = float(bb.blocks[0].norm1.eps)
    for i in range(L - 1):
        x = O.block_forward(sd, f"backbone.blocks.{i}.", x, H, eps)
    b = f"backbone.blocks.{L - 1}."
    h = F.layer_norm(x, (x.shape[-1],), sd[b + "norm1.weight"], sd[b + "norm1.bias"], eps)
    qkv = F.linear(h, sd[b + "attn.qkv.weight"], sd.get(b + "attn.qkv.bias"))
    return O.softmax_attention(qkv, x.shape[0], x.shape[1], H, (x.shape[-1] // H) ** -0.5)[1]


def _module_last_attention(model, images):
    """get_last_selfattention through the un-fused module path: the blocks, then norm1 + attention of the last one."""
    from apla_b200.apla import attention_probabilities
    bb = model.backbone
    with torch.no_grad(), attention_probabilities(model):
        x = bb.tokens(images.cuda())
        for blk in bb.blocks[:-1]:
            x = blk(x)
        return bb.blocks[-1].attn(bb.blocks[-1].norm1(x))[1]


@pytest.mark.parametrize("name", ["tiny_r16", "c1_vits16_r32", "c2_vitb14_r8"])
def test_last_self_attention_of_a_whole_model(name):
    _need_gpu()
    from apla_b200.apla import attention_probabilities, fuse_apla_blocks
    model, meta, _ = build_case(name)
    m = meta["meta"]
    model = model.cuda()
    images, _ = synthetic_batch(2, m["img"], m["n_classes"], seed=21)
    want = _oracle_last_attention(model, images)
    got = _module_last_attention(model, images)
    _check(got, want)
    fuse_apla_blocks(model)
    bb = model.backbone
    with torch.no_grad(), attention_probabilities(model):
        x = bb.tokens(images.cuda())
        for blk in bb.blocks[:-1]:
            x = blk(x)
        fused = bb.blocks[-1](x, return_attention=True)
        with pytest.raises(RuntimeError, match="list"):
            bb.blocks[-1]([x], return_attention=True)
        with pytest.raises(RuntimeError, match="return_intermediate"):
            bb.blocks[-1](x, return_intermediate=True)
    assert fused.dtype == torch.float32 and fused.shape == want.shape
    _check(fused, want)
    with pytest.raises(RuntimeError, match="attention_probabilities"):
        bb.blocks[-1](x, return_attention=True)


def _engine(model, batch, img, **kw):
    _need_gpu()
    from apla_b200.engine import FineTuneEngine
    return FineTuneEngine(model, batch_size=batch, img_size=img, **kw)


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_engine_cls_attention_matches_the_module_path(mode):
    model, meta, _ = build_case("c1_vits16_r32")
    m = meta["meta"]
    eng = _engine(model, 4, m["img"], cls_only_last_block=mode, eval_batch_size=3)
    images, labels = synthetic_batch(5, m["img"], m["n_classes"], seed=13)
    eng.step(images[:4].cuda(), labels[:4].cuda())          # weights that differ from the initial ones
    eng.sync_to_model()
    want = _module_last_attention(model.cuda(), images)[:, :, 0, :]
    H, N = want.shape[1], want.shape[2]
    for n in (1, 5):                                         # one image; 3 + 2 in two chunks
        got = eng.cls_attention(images[:n].cuda())
        assert got.dtype == torch.float32 and got.shape == (n, H, N)
        _check(got, want[:n])
    assert torch.equal(eng.cls_attention(images.pin_memory()), eng.cls_attention(images.cuda()))


def test_cls_attention_leaves_the_training_state_alone():
    from apla_b200._lib import LIB
    model, _, _ = build_case("tiny_r16")
    eng = _engine(model, 4, 56, eval_batch_size=3)
    images, labels = synthetic_batch(4, 56, 10)
    images, labels = images.cuda(), labels.cuda()

    def eager_step_launches():
        torch.cuda.synchronize()
        n0 = LIB.load().apla_launch_count()
        eng.forward(images, labels)
        eng.backward()
        eng.optim_step()
        torch.cuda.synchronize()
        return int(LIB.load().apla_launch_count() - n0)

    before = eager_step_launches()
    eng.step(images, labels)                 # eager (first sight of this buffer pair)
    eng.step(images, labels)                 # captured, replayed
    torch.cuda.synchronize()
    assert len(eng._graphs) == 1
    bufs = list(eng._keep) + [eng.params, eng.grads, eng.exp_avg, eng.exp_avg_sq, eng.logits, eng.loss, eng.xs]
    snap = [t.view(torch.uint8).clone() for t in bufs]
    other, _ = synthetic_batch(7, 56, 10, seed=3)
    probs = eng.cls_attention(other.cuda())
    torch.cuda.synchronize()
    assert probs.shape == (7, 2, 17)
    for i, (t, s) in enumerate(zip(bufs, snap)):
        assert torch.equal(t.view(torch.uint8), s), f"training buffer {i} {tuple(t.shape)} {t.dtype} changed"
    p = eng.params.clone()
    eng.step(images, labels)                 # replay of the graph captured before cls_attention
    torch.cuda.synchronize()
    assert len(eng._graphs) == 1
    assert torch.isfinite(eng.loss).all() and float((eng.params - p).norm()) > 0
    assert eager_step_launches() == before

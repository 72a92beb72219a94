"""Stochastic depth (drop path) in the fused blocks on the B200: the row-scaled LayerScale cast against torch, and
`FusedAplaBlock` in training mode against the same unfused block under the same seed -- the masks come from the block's
own drop-path modules, so they are the unfused block's bit for bit and the CUDA generator ends in the same state.
Bars (BASELINE.json north_star): relative error <= 1e-2, gradient cosine >= 0.999."""
import types

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from helpers import cosine, perturb_module, rel, synthetic_batch

pytestmark = pytest.mark.gpu


def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")


class TimmDropPath(nn.Module):
    """timm.layers.DropPath: a bernoulli_ mask in the input's dtype, optionally not rescaled."""

    def __init__(self, drop_prob, scale_by_keep=True):
        super().__init__()
        self.drop_prob, self.scale_by_keep = drop_prob, scale_by_keep

    def forward(self, x):
        if self.drop_prob == 0.0 or not self.training:
            return x
        keep = 1.0 - self.drop_prob
        mask = x.new_empty((x.shape[0],) + (1,) * (x.ndim - 1)).bernoulli_(keep)
        if keep > 0.0 and self.scale_by_keep:
            mask.div_(keep)
        return x * mask


def _timm_forward(self, x):
    """timm's Block.forward: one drop-path module per branch."""
    y = self.attn(self.norm1(x))
    y = y[0] if isinstance(y, tuple) else y
    x = x + self.drop_path1(self.ls1(y))
    return x + self.drop_path2(self.ls2(self.mlp(self.norm2(x))))


def _set_drop_path(model, rate, kind):
    """Every block gets drop-path rate `rate`: the reference's one DropPath ("ref"), or timm's drop_path1 / drop_path2
    ("timm", "timm_nokeep" = scale_by_keep=False)."""
    from apla_b200.hostvit import DropPath
    for blk in model.backbone.blocks:
        if kind == "ref":
            blk.drop_path = DropPath(rate)
        else:
            del blk.drop_path
            blk.drop_path1 = TimmDropPath(rate, kind == "timm")
            blk.drop_path2 = TimmDropPath(rate, kind == "timm")
            blk.forward = types.MethodType(_timm_forward, blk)
    return model


def _pair(arch=None, img=56, patch=14, rate=0.0, kind="ref", r=16):
    """Two identical models on the GPU in train mode, the second with fused blocks."""
    from apla_b200.apla import fuse_apla_blocks
    from apla_b200.config import AplaConfig
    from apla_b200.hostvit import VitArch, build_classifier
    models = []
    for _ in range(2):
        m = build_classifier(arch or VitArch(128, 2, 2), img_size=img, patch_size=patch, n_classes=10,
                             apla_config=AplaConfig(r), seed=0)
        perturb_module(m)                            # LayerScale vectors away from 1, biases away from 0
        models.append(_set_drop_path(m, rate, kind).cuda().train())
    fuse_apla_blocks(models[1])
    return models


def _record_masks(model):
    """Keep-or-drop per image of every drop-path call, in call order (the fused block calls its modules on ones)."""
    from apla_b200.hostvit import DropPath
    rec = []

    def hook(mod, inp, out):
        rec.append((out.detach().reshape(out.shape[0], -1) != 0).any(1).cpu())

    for m in model.modules():
        if isinstance(m, (DropPath, TimmDropPath)):
            m.register_forward_hook(hook)
    return rec


# ---- the kernel ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,N,D", [(4, 257, 768), (3, 197, 384), (5, 1, 128)])
def test_scaled_ls_cast_matches_torch(B, N, D):
    """bf16(s[t / N] * gamma * x) against torch, bit for bit (same fp32 products in the same order); all-ones scales give
    apla_ls_cast's bits.  The output is NaN-prefilled with a canary tail."""
    _need_gpu()
    from apla_b200._lib import LIB, ptr, stream
    g = torch.Generator().manual_seed(B * N + D)
    rows = B * N
    x = torch.randn(rows, D, generator=g).cuda()
    gamma = (1 + 0.1 * torch.randn(D, generator=g)).cuda()
    keep = 0.7
    s = ((torch.rand(B, generator=g) < keep).float() / keep)
    s[0] = 0.0
    s = s.cuda()

    def run(scale, gm):
        buf = torch.full((rows * D + 64,), float("nan"), device="cuda", dtype=torch.bfloat16)
        buf[rows * D:] = 7.0
        if scale is None:
            LIB.call("apla_ls_cast", ptr(x), D, ptr(gm), ptr(buf), D, rows, D, stream())
        else:
            LIB.call("apla_ls_cast_scaled", ptr(x), D, ptr(gm), ptr(buf), D, ptr(scale), N, rows, D, stream())
        torch.cuda.synchronize()
        assert (buf[rows * D:] == 7.0).all()
        return buf[:rows * D].view(rows, D)

    for gm in (gamma, None):
        got = run(s, gm)
        xg = x * gm if gm is not None else x
        want = (xg * s.repeat_interleave(N)[:, None]).to(torch.bfloat16)
        assert torch.equal(got, want)
        assert (got.view(B, N, D)[0] == 0).all()
        assert torch.equal(run(torch.ones(B, device="cuda"), gm), run(None, gm))


# ---- one block ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["ref", "timm", "timm_nokeep"])
@pytest.mark.parametrize("rate", [0.1, 0.5])
def test_fused_block_drop_path_matches_unfused(rate, kind):
    """One block in train mode under torch.manual_seed(k): output, input gradient, proj_weight1 / proj_bias1 gradients,
    the masks drawn and the CUDA generator state afterwards, against the unfused block."""
    _need_gpu()
    ref_m, fus_m = _pair(rate=rate, kind=kind)
    l = 1
    blocks = (ref_m.backbone.blocks[l], fus_m.backbone.blocks[l])
    masks = [_record_masks(ref_m), _record_masks(fus_m)]
    B, N, D = 6, 50, 128
    dropped = 0
    for k in range(3):
        g = torch.Generator().manual_seed(100 + k)
        x_cpu, dy_cpu = torch.randn(B, N, D, generator=g), torch.randn(B, N, D, generator=g)
        res = []
        for blk in blocks:
            for p in blk.parameters():
                p.grad = None
            torch.manual_seed(k)
            x = x_cpu.cuda().requires_grad_(True)
            out = blk(x)
            out.backward(dy_cpu.cuda())
            torch.cuda.synchronize()
            res.append((out.detach(), x.grad, blk.attn.proj_weight1.grad, blk.attn.proj_bias1.grad,
                        torch.cuda.get_rng_state()))
        (o_r, dx_r, w_r, b_r, st_r), (o_f, dx_f, w_f, b_f, st_f) = res
        assert torch.equal(st_r, st_f), "the fused block advanced the generator differently"
        assert rel(o_f, o_r) <= 1e-2, rel(o_f, o_r)
        assert rel(dx_f, dx_r) <= 1e-2 and cosine(dx_f, dx_r) >= 0.999, rel(dx_f, dx_r)
        assert rel(w_f, w_r) <= 1e-2, rel(w_f, w_r)
        if w_r.abs().sum() > 0:                      # (zero when every image dropped the attention branch)
            assert cosine(w_f, w_r) >= 0.999, cosine(w_f, w_r)
        assert rel(b_f, b_r) <= 1e-2, rel(b_f, b_r)
    assert len(masks[0]) == len(masks[1]) == 6
    for a, b in zip(*masks):
        assert torch.equal(a, b)
        dropped += int((~a).sum())
    if rate == 0.5:
        assert dropped > 0


class FixedDropPath(nn.Module):
    """A drop-path module with fixed masks, one per call in turn (2 / keep = 2 for kept images)."""

    def __init__(self, masks):
        super().__init__()
        self.drop_prob, self.masks, self.calls = 0.5, masks, 0

    def forward(self, x):
        m = self.masks[self.calls % len(self.masks)]
        self.calls += 1
        return x * (2.0 * m).to(device=x.device, dtype=x.dtype).view(-1, *([1] * (x.ndim - 1)))


def test_dropped_images_pass_through_exactly():
    """Image 0 drops both branches: its output is its input and its input gradient the output gradient, bit for bit.
    The other images (one branch dropped, or none) match the unfused block."""
    _need_gpu()
    ref_m, fus_m = _pair()
    s_attn, s_mlp = torch.tensor([0.0, 1.0, 0.0, 1.0]), torch.tensor([0.0, 0.0, 1.0, 1.0])
    B, N, D = 4, 65, 128
    g = torch.Generator().manual_seed(3)
    x_cpu, dy_cpu = torch.randn(B, N, D, generator=g), torch.randn(B, N, D, generator=g)
    res = []
    for m in (ref_m, fus_m):
        blk = m.backbone.blocks[1]
        blk.drop_path = FixedDropPath([s_attn, s_mlp])
        x = x_cpu.cuda().requires_grad_(True)
        out = blk(x)
        out.backward(dy_cpu.cuda())
        torch.cuda.synchronize()
        res.append((out.detach(), x.grad))
    (o_r, dx_r), (o_f, dx_f) = res
    assert torch.equal(o_f[0], x_cpu[0].cuda()) and torch.equal(dx_f[0], dy_cpu[0].cuda())
    assert rel(o_f, o_r) <= 1e-2 and rel(dx_f, dx_r) <= 1e-2 and cosine(dx_f, dx_r) >= 0.999


def _log_calls(monkeypatch):
    """Record the name of every native call the Python layer makes."""
    from apla_b200._lib import LIB
    names, real_call = [], LIB.call
    monkeypatch.setattr(LIB, "call", lambda name, *a: (names.append(name), real_call(name, *a))[1])
    return names


def test_no_grad_training_forward_drops_like_the_reference(monkeypatch):
    """Under torch.no_grad() a training-mode block still drops (the forward-only native call with scales)."""
    _need_gpu()
    ref_m, fus_m = _pair(rate=0.5)
    masks = [_record_masks(ref_m), _record_masks(fus_m)]
    x = torch.randn(6, 50, 128, generator=torch.Generator().manual_seed(4)).cuda()
    outs, states = [], []
    names = _log_calls(monkeypatch)
    for m in (ref_m, fus_m):
        torch.manual_seed(9)
        with torch.no_grad():
            outs.append(m.backbone.blocks[1](x))
        states.append(torch.cuda.get_rng_state())
    assert "apla_block_fwd_infer_scaled" in names
    assert torch.equal(states[0], states[1])
    assert all(torch.equal(a, b) for a, b in zip(*masks)) and len(masks[1]) == 2
    assert rel(outs[1], outs[0]) <= 1e-2, rel(outs[1], outs[0])


# ---- whole models -------------------------------------------------------------------------------------------------
MODELS = {
    "tiny": (None, 56, 14, 4),
    "c1": ("vit_small", 224, 16, 4),              # 197 tokens
    "c2": ("vit_base", 224, 14, 4),               # 257 tokens
}


@pytest.mark.parametrize("chain", [True, False])
@pytest.mark.parametrize("name", list(MODELS))
def test_model_of_fused_blocks_trains_like_unfused(name, chain):
    """A classifier built with drop path, every block fused, three steps of torch AdamW against the unfused model under
    the same seeds: logits and loss per step, the first step's proj_weight1 / proj_bias1 gradients of every block, the
    masks, the generator state and the parameters afterwards.  With and
    without the block-to-block gradient hand-over (APLA_BLOCK_CHAIN)."""
    _need_gpu()
    import apla_b200.apla.apla_block as AB
    arch, img, patch, B = MODELS[name]
    ref_m, fus_m = _pair(arch, img, patch)
    for m in (ref_m, fus_m):
        from apla_b200.hostvit import DropPath
        L = len(m.backbone.blocks)
        for l, blk in enumerate(m.backbone.blocks):     # the reference's linspace(0, 0.3, depth)
            rate = 0.3 * l / (L - 1)
            blk.drop_path = DropPath(rate) if rate > 0 else nn.Identity()
    masks = [_record_masks(ref_m), _record_masks(fus_m)]
    p0 = {n: p.detach().clone() for n, p in ref_m.named_parameters() if p.requires_grad}
    opts = [torch.optim.AdamW([p for p in m.parameters() if p.requires_grad], lr=1e-4) for m in (ref_m, fus_m)]
    AB._CHAIN = chain
    try:
        for step in range(3):
            images, labels = synthetic_batch(B, img, 10, seed=200 + step)
            res = []
            for m, opt in zip((ref_m, fus_m), opts):
                torch.manual_seed(1000 + step)
                logits = m(images.cuda())
                loss = F.cross_entropy(logits, labels.cuda())
                opt.zero_grad()
                loss.backward()
                grads = [torch.cat([getattr(b.attn, n).grad.flatten() for b in m.backbone.blocks])
                         for n in ("proj_weight1", "proj_bias1")]
                opt.step()
                torch.cuda.synchronize()
                res.append((logits.detach(), float(loss.detach()), torch.cuda.get_rng_state(), grads))
            assert torch.equal(res[0][2], res[1][2]), step
            if step == 0:                                # same parameters: every block's trainable-row gradients
                for want, got in zip(res[0][3], res[1][3]):
                    assert rel(got, want) <= 1e-2 and cosine(got, want) >= 0.999, (rel(got, want), cosine(got, want))
            assert rel(res[1][0], res[0][0]) <= 1e-2, (step, rel(res[1][0], res[0][0]))
            assert abs(res[1][1] - res[0][1]) <= 1e-2 * abs(res[0][1])
    finally:
        AB._CHAIN = True
    assert len(masks[0]) == len(masks[1]) > 0
    assert all(torch.equal(a, b) for a, b in zip(*masks))
    pr, pf = dict(ref_m.named_parameters()), dict(fus_m.named_parameters())
    got = torch.cat([pf[n].detach().flatten() for n in p0])
    want = torch.cat([pr[n].detach().flatten() for n in p0])
    init = torch.cat([p0[n].flatten() for n in p0])
    assert rel(got, want) <= 1e-2, rel(got, want)
    assert cosine(got - init, want - init) >= 0.95, cosine(got - init, want - init)


# ---- what does not change -----------------------------------------------------------------------------------------
def test_rate_zero_and_eval_issue_todays_calls_and_draw_nothing(monkeypatch):
    """At rate 0 (train) and in eval mode (rate 0.3) the fused model makes the unscaled native calls -- the same
    launches, bit-identical outputs and gradients -- and leaves the generator untouched.  With drop path the backward
    costs one launch per block whose block behind it can no longer hand over its gradient; lists still raise."""
    _need_gpu()
    from apla_b200._lib import LIB
    from apla_b200.apla import fuse_apla_blocks
    from apla_b200.config import AplaConfig
    from apla_b200.hostvit import VitArch, build_classifier
    dll = LIB.load()
    models = {}
    for rate in (0.0, 0.3):
        m = build_classifier(VitArch(128, 3, 2), img_size=56, patch_size=14, n_classes=10, apla_config=AplaConfig(16),
                             seed=0, drop_path_rate=rate)
        perturb_module(m)
        models[rate] = fuse_apla_blocks(m.cuda())
    images, labels = synthetic_batch(4, 56, 10, seed=5)
    images, labels = images.cuda(), labels.cuda()
    log = _log_calls(monkeypatch)

    def run(m, train):
        m.train(train)
        for p in m.parameters():
            p.grad = None
        del log[:]
        state = torch.cuda.get_rng_state()
        n0 = dll.apla_launch_count()
        logits = m(images)
        n1 = dll.apla_launch_count()
        F.cross_entropy(logits, labels).backward()
        torch.cuda.synchronize()
        n2 = dll.apla_launch_count()
        grads = [p.grad.clone() for p in m.parameters() if p.requires_grad]
        return logits.detach(), grads, (n1 - n0, n2 - n1), list(log), torch.equal(state, torch.cuda.get_rng_state())

    for m in models.values():                        # first calls build the working sets (one scatter per block)
        run(m, False)
    base = run(models[0.0], True)
    for got in (run(models[0.3], False), run(models[0.0], False)):
        assert got[2] == base[2] and got[4] and base[4]
        assert not any(n.endswith("_scaled") for n in got[3] + base[3])
        assert torch.equal(got[0], base[0])
        for a, b in zip(got[1], base[1]):
            assert rel(a, b) < 1e-5                  # (weight gradients: fp32 atomics of the split-K kernel)
    # rates linspace(0, 0.3, 3) = (0, 0.15, 0.3): block 1 draws, so block 2 hands it nothing and it casts for itself;
    # block 0 (rate 0) still receives block 1's hand-over
    dp = run(models[0.3], True)
    assert dp[2] == (base[2][0], base[2][1] + 1), (dp[2], base[2])
    assert "apla_block_fwd_scaled" in dp[3] and "apla_block_bwd_scaled" in dp[3] and not dp[4]
    with pytest.raises(RuntimeError, match="list of crops"):
        models[0.3].backbone.blocks[1]([torch.randn(2, 17, 128, device="cuda")])

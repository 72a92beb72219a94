"""Stochastic depth (drop path) without a GPU: the argument checks of the two row-scaled C entries and the engine's
"drop_path" buffer name; `drop_path_rates`, which reads the reference's per-block rates and refuses what the engine
cannot honour before touching a device; and the host ViT's `drop_path_rate`, which changes no weight and, in train mode,
computes x + s * ls(branch) with one scale per image."""
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from apla_b200._lib import LIB
from apla_b200.hostvit import DropPath, HostViT, VitArch


def _refused(rc, what):
    assert rc == 1, (what, rc)
    msg = LIB.load().apla_last_error()
    assert msg, what
    return msg.decode()


def test_scaled_entries_refuse_bad_arguments_without_a_gpu():
    dll = LIB.load()
    fake = 256                                        # a non-NULL address that is never dereferenced

    def gemm(ptrs, rps=1, M=64, N=128, K=64):
        A, W, resid, scale, out = ptrs
        return dll.apla_gemm_bias_ls_residual_scaled_fwd(A, K, W, K, fake, fake, resid, scale, rps, out, N, M, N, K, None)

    def lnb(ptrs, rps=1, rows=8, D=128):
        dy, x, w, dx, dxb, scale = ptrs
        return dll.apla_layernorm_bwd_scaled(dy, D, x, D, w, None, 0, dx, D, dxb, D, fake, None, 0, None, 0, 0, scale,
                                             rps, rows, D, 1e-6, None)

    for i in range(5):
        ptrs = [fake] * 5
        ptrs[i] = None
        assert "null" in _refused(gemm(ptrs), f"gemm pointer {i} NULL")
    for i in range(6):
        ptrs = [fake] * 6
        ptrs[i] = None
        assert "null" in _refused(lnb(ptrs), f"layernorm pointer {i} NULL")
    for M, N, K in ((0, 128, 64), (64, 0, 64), (64, 128, 0), (-1, 128, 64)):
        assert "empty" in _refused(gemm([fake] * 5, M=M, N=N, K=K), (M, N, K))
    for rows, D in ((0, 128), (8, 0), (-3, 128)):
        assert "empty" in _refused(lnb([fake] * 6, rows=rows, D=D), (rows, D))
    for rps in (0, -1):
        assert "rows_per_scale" in _refused(gemm([fake] * 5, rps=rps), f"gemm rps={rps}")
        assert "rows_per_scale" in _refused(lnb([fake] * 6, rps=rps), f"layernorm rps={rps}")
    # the row-scaled LayerNorm backward has no generic-width form
    assert "multiple of 128" in _refused(lnb([fake] * 6, D=64), "D=64")


def test_drop_path_is_an_engine_buffer():
    dll = LIB.load()
    fake = 256
    e = dll.apla_engine_create(4, 17, 128, 2, 2, 512, 10, 14, 56, 640, 16, 64, 0, 1e-6, 0.125)
    assert e
    try:
        assert dll.apla_engine_set_ptr(e, b"drop_path", -1, fake) == 0
        assert dll.apla_engine_set_ptr(e, b"drop_path", -1, None) == 0
        assert "unknown" in _refused(dll.apla_engine_set_ptr(e, b"drop_paths", -1, fake), "misspelt name")
        # optional: an engine without it still stops at the step's own unset buffers
        assert "not set" in _refused(dll.apla_engine_forward(e, fake, fake, 1.0, 1.0, None), "forward")
    finally:
        dll.apla_engine_destroy(e)


def _classifier(rate=0.0, depth=4):
    from apla_b200.config import AplaConfig
    from apla_b200.hostvit import build_classifier
    return build_classifier(VitArch(128, depth, 2), img_size=56, patch_size=14, n_classes=10,
                            apla_config=AplaConfig(16), seed=0, drop_path_rate=rate)


def test_drop_path_rates_read_the_linspace():
    from apla_b200.engine import drop_path_rates
    rates = drop_path_rates(_classifier(0.2, depth=5))
    want = torch.linspace(0, 0.2, 5).tolist()
    assert [a for a, _ in rates] == pytest.approx(want) and [b for _, b in rates] == pytest.approx(want)
    assert all(a == b for a, b in rates)
    assert drop_path_rates(_classifier(0.0)) == [(0.0, 0.0)] * 4


def test_drop_path_rates_accept_timm_names_and_identity():
    from apla_b200.engine import drop_path_rates
    model = _classifier(0.0, depth=3)

    class TimmDropPath(nn.Module):                   # timm.layers.DropPath's attributes
        def __init__(self, p, scale_by_keep=True):
            super().__init__()
            self.drop_prob, self.scale_by_keep = p, scale_by_keep

    blocks = model.backbone.blocks
    del blocks[0].drop_path
    blocks[0].drop_path1, blocks[0].drop_path2 = TimmDropPath(0.1), nn.Identity()
    blocks[1].drop_path = DropPath(None)             # the reference's DropPath() default
    blocks[2].drop_path = TimmDropPath(0.3)
    assert drop_path_rates(model) == [(0.1, 0.0), (0.0, 0.0), (0.3, 0.3)]


@pytest.mark.parametrize("where,match", [
    ("scale_by_keep", "scale_by_keep=False"),
    ("attn_drop", "attn.attn_drop has dropout rate 0.1"),
    ("proj_drop", "attn.proj_drop has dropout rate 0.1"),
    ("mlp_drop", "mlp.drop has dropout rate 0.1"),
    ("pos_drop", "backbone.pos_drop has dropout rate 0.1"),
    ("sample_drop_ratio", "batch-subset stochastic depth"),
    ("rate_one", "outside"),
])
def test_drop_path_rates_refuse_what_the_engine_cannot_honour(where, match):
    from apla_b200.engine import FineTuneEngine, drop_path_rates
    model = _classifier(0.0, depth=2)
    blk = model.backbone.blocks[1]
    if where == "scale_by_keep":
        blk.drop_path = DropPath(0.1)
        blk.drop_path.scale_by_keep = False
    elif where == "attn_drop":
        blk.attn.attn_drop.p = 0.1
    elif where == "proj_drop":
        blk.attn.proj_drop.p = 0.1
    elif where == "mlp_drop":
        blk.mlp.drop = nn.Dropout(0.1)
    elif where == "pos_drop":
        model.backbone.pos_drop = nn.Dropout(0.1)
    elif where == "sample_drop_ratio":
        blk.sample_drop_ratio = 0.2
    else:
        blk.drop_path = DropPath(1.0)
    with pytest.raises(ValueError, match=match):
        drop_path_rates(model)
    # the engine refuses the model before it looks for a device
    with pytest.raises(ValueError, match=match):
        FineTuneEngine(model, batch_size=4, img_size=56)


def test_host_vit_weights_do_not_depend_on_the_rate():
    def state(rate):
        torch.manual_seed(0)
        return HostViT(VitArch(128, 4, 2), img_size=56, patch_size=14, drop_path_rate=rate).state_dict()

    ref = state(0.0)
    for rate in (0.1, 0.5):
        sd = state(rate)
        assert list(sd) == list(ref)
        assert all(torch.equal(sd[k], ref[k]) for k in ref)
    a, b = _classifier(0.0).state_dict(), _classifier(0.3).state_dict()
    assert list(a) == list(b) and all(torch.equal(a[k], b[k]) for k in a)
    vit = HostViT(VitArch(128, 4, 2), img_size=56, patch_size=14, drop_path_rate=0.3)
    assert isinstance(vit.blocks[0].drop_path, nn.Identity)
    assert [blk.drop_path.drop_prob for blk in vit.blocks[1:]] == pytest.approx([0.1, 0.2, 0.3])


def test_host_vit_train_mode_applies_one_scale_per_image_and_branch():
    """Masks patched to fixed values (each call takes the next [B] scale vector): the host model's train-mode forward
    against an fp32 reference built from F.layer_norm / F.linear / F.gelu with x + s * ls(branch); eval mode is the
    identity, and unpatched train mode draws zeros and 1 / keep only."""
    torch.manual_seed(0)
    B, depth, rate = 5, 3, 0.4
    vit = HostViT(VitArch(128, depth, 2), img_size=56, patch_size=14, drop_path_rate=rate).train()
    with torch.no_grad():
        for blk in vit.blocks:
            blk.ls1.gamma.normal_(1.0, 0.1)
            blk.ls2.gamma.normal_(1.0, 0.1)
    images = torch.randn(B, 3, 56, 56, generator=torch.Generator().manual_seed(1))
    g = torch.Generator().manual_seed(2)
    scales = []
    for blk in vit.blocks:
        keep = 1.0 - (blk.drop_path.drop_prob if isinstance(blk.drop_path, DropPath) else 0.0)
        scales.append([(torch.rand(B, generator=g) < keep).float() / keep for _ in range(2)])
    calls = iter([s for pair in scales[1:] for s in pair])     # block 0 has rate 0: nn.Identity, never called

    def fixed(self, x):
        return x * next(calls).view(-1, 1, 1)

    orig = DropPath.forward
    DropPath.forward = fixed
    try:
        got = vit(images)
    finally:
        DropPath.forward = orig

    def reference():
        x = vit.tokens(images)
        for l, blk in enumerate(vit.blocks):
            D = x.shape[-1]
            s1, s2 = scales[l] if l > 0 else (torch.ones(B), torch.ones(B))
            h = F.layer_norm(x, (D,), blk.norm1.weight, blk.norm1.bias, blk.norm1.eps)
            qkv = F.linear(h, blk.attn.qkv.weight, blk.attn.qkv.bias).view(B, -1, 3, 2, D // 2).permute(2, 0, 3, 1, 4)
            a = torch.softmax((qkv[0] @ qkv[1].transpose(-2, -1)) * blk.attn.scale, -1) @ qkv[2]
            y = F.linear(a.transpose(1, 2).reshape(B, -1, D), blk.attn.proj.weight, blk.attn.proj.bias)
            x = x + s1.view(-1, 1, 1) * (y * blk.ls1.gamma)
            h = F.layer_norm(x, (D,), blk.norm2.weight, blk.norm2.bias, blk.norm2.eps)
            h = F.linear(F.gelu(F.linear(h, blk.mlp.fc1.weight, blk.mlp.fc1.bias)), blk.mlp.fc2.weight, blk.mlp.fc2.bias)
            x = x + s2.view(-1, 1, 1) * (h * blk.ls2.gamma)
        return F.layer_norm(x, (x.shape[-1],), vit.norm.weight, vit.norm.bias, vit.norm.eps)[:, 0]

    with torch.no_grad():
        want = reference()
        assert float((got - want).abs().max()) <= 1e-5 * float(want.abs().max()), float((got - want).abs().max())
        # eval: identity, whatever the rate
        torch.manual_seed(0)
        plain = HostViT(VitArch(128, depth, 2), img_size=56, patch_size=14).eval()
        plain.load_state_dict(vit.state_dict())
        assert torch.equal(vit.eval()(images), plain(images))
        # unpatched train mode: every per-image scale of a DropPath call is 0 or 1 / keep
        x = torch.ones(64, 3, 4)
        out = DropPath(rate).train()(x)
        v = out[:, 0, 0]
        assert bool(((v == 0) | ((v - 1.0 / (1.0 - rate)).abs() < 1e-6)).all()), v
        assert torch.equal(out, out[:, :1, :1].expand_as(out))

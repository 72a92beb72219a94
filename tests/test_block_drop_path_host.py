"""Stochastic depth in the fused blocks without a GPU: the argument checks of the row-scaled block entries and of the
row-scaled LayerScale cast, and what `FusedAplaBlock` still refuses in training mode (dropout, DINOv2's batch-subset
stochastic depth, drop path on lists of crops), raised before any device work."""
import ctypes

import pytest
import torch

from apla_b200._lib import LIB, BlockWeights


def _refused(rc, what):
    assert rc == 1, (what, rc)
    msg = LIB.load().apla_last_error()
    assert msg, what
    return msg.decode()


def _weights():
    fake = 256                                        # a non-NULL address that is never dereferenced
    w = BlockWeights()
    for n in ("wqkv", "wproj", "wfc1", "wfc2", "ln1w", "ln1b", "ln2w", "ln2b", "wfc1T", "wfc2T"):
        setattr(w, n, fake)
    w.D, w.H, w.hidden, w.eps1, w.eps2, w.scale = 128, 2, 512, 1e-6, 1e-6, 0.125
    return w


def test_scaled_block_entries_refuse_bad_arguments_without_a_gpu():
    dll = LIB.load()
    fake = 256
    w = _weights()
    wp = ctypes.addressof(w)

    def fwd(scale, rps, T=16, lse=fake):
        return dll.apla_block_fwd_scaled(wp, fake, fake, fake, fake, fake, fake, lse, fake, fake, None, 2, 8, T, scale,
                                         rps, None)

    def infer(scale, rps, T=16, lse=fake):
        return dll.apla_block_fwd_infer_scaled(wp, fake, fake, fake, fake, fake, fake, lse, fake, None, 2, 8, T, scale,
                                               rps, None)

    def bwd(scale, rps, T=16, dyb_ready=0, db1=fake):
        return dll.apla_block_bwd_scaled(wp, fake, fake, fake, fake, fake, fake, fake, fake, fake, fake, fake, fake, fake,
                                         fake, fake, fake, fake, db1, None, 2, 8, T, dyb_ready, None, None, scale, rps,
                                         None)

    for name, call in (("fwd", fwd), ("infer", infer), ("bwd", bwd)):
        for scale in (None, fake):
            for rps in (0, -8):
                assert "rows_per_scale" in _refused(call(scale, rps), f"{name} rps={rps}")
        # scales: T must be whole images of rows_per_scale rows
        assert "whole number" in _refused(call(fake, 5), f"{name} T=16 rps=5")
        assert "empty" in _refused(call(fake, 8, T=0), f"{name} T=0")
    # NULL scales pass the scale checks whatever rows_per_scale divides: the call stops at the next check instead
    assert "null buffer" in _refused(fwd(None, 5, lse=None), "fwd NULL scales")
    assert "null buffer" in _refused(infer(None, 5, lse=None), "infer NULL scales")
    assert "db1" in _refused(bwd(None, 5, db1=None), "bwd NULL scales")
    assert "null buffer" in _refused(fwd(fake, 8, lse=None), "fwd scales")
    # the row-scaled LayerNorm backward needs D % 128 == 0: refused before any launch (the forwards take any width)
    w192 = _weights()
    w192.D, w192.H = 192, 3
    assert "multiple of 128" in _refused(
        dll.apla_block_bwd_scaled(ctypes.addressof(w192), *([fake] * 17), fake, None, 2, 8, 16, 0, None, None, fake, 8,
                                  None), "bwd scales D=192")
    # a hand-over carries no branch scale: a block with scales forms its own dyb
    assert "dyb_ready" in _refused(bwd(fake, 8, dyb_ready=1), "bwd scales with dyb_ready")
    assert "db1" in _refused(bwd(None, 8, dyb_ready=1, db1=None), "bwd dyb_ready without scales")


def test_scaled_ls_cast_refuses_bad_arguments_without_a_gpu():
    dll = LIB.load()
    fake = 256
    for i in range(3):
        x, out, scale = [fake if j != i else None for j in range(3)]
        assert "null" in _refused(dll.apla_ls_cast_scaled(x, 128, None, out, 128, scale, 4, 8, 128, None), f"NULL {i}")
    for rows, D in ((0, 128), (8, 0), (8, 126)):
        assert "bad shape" in _refused(dll.apla_ls_cast_scaled(fake, 128, None, fake, 128, fake, 4, rows, D, None),
                                       (rows, D))
    for rps in (0, -1):
        assert "rows_per_scale" in _refused(dll.apla_ls_cast_scaled(fake, 128, None, fake, 128, fake, rps, 8, 128, None),
                                            rps)


def _fused(rate=0.2, depth=2):
    from apla_b200.apla import fuse_apla_blocks
    from apla_b200.config import AplaConfig
    from apla_b200.hostvit import VitArch, build_classifier
    model = build_classifier(VitArch(128, depth, 2), img_size=56, patch_size=14, n_classes=10,
                             apla_config=AplaConfig(16), seed=0, drop_path_rate=rate)
    fuse_apla_blocks(model)
    return model.train()


@pytest.mark.parametrize("what,match", [
    ("attn_drop", "dropout"), ("proj_drop", "dropout"), ("mlp_drop", "dropout"),
    ("sample_drop_ratio", "batch-subset"), ("crops", "list of crops"), ("timm_crops", "list of crops")])
def test_fused_block_refusals_come_before_device_work(what, match):
    """Each refusal names what is unsupported and is raised on a CPU tensor, before the CUDA check and before the
    generator is touched."""
    from apla_b200.hostvit import DropPath
    blk = _fused().backbone.blocks[1]                  # linspace(0, 0.2, 2): block 1 has rate 0.2
    x = torch.randn(2, 17, 128)
    arg = x
    if what == "attn_drop":
        blk.attn.attn_drop.p = 0.1
    elif what == "proj_drop":
        blk.attn.proj_drop.p = 0.1
    elif what == "mlp_drop":
        blk.mlp.drop = torch.nn.Dropout(0.1)
    elif what == "sample_drop_ratio":
        blk.sample_drop_ratio = 0.2
    elif what == "crops":
        arg = [x, torch.randn(3, 5, 128)]
    else:                                              # timm names, only the MLP branch drops
        del blk.drop_path
        blk.drop_path1, blk.drop_path2 = torch.nn.Identity(), DropPath(0.1)
        arg = [x]
    state = torch.random.get_rng_state()
    with pytest.raises(RuntimeError, match=match):
        blk(arg)
    assert torch.equal(torch.random.get_rng_state(), state)


def test_fused_block_refuses_drop_path_at_widths_not_a_multiple_of_128():
    """ViT-Ti's 192-wide blocks: drop path in training mode is refused on a CPU tensor, before the CUDA check and before
    any draw; at rate 0 or in eval mode the block gets to its CUDA check."""
    from apla_b200.apla import fuse_apla_blocks
    from apla_b200.config import AplaConfig
    from apla_b200.hostvit import VitArch, build_classifier
    model = build_classifier(VitArch(192, 2, 3), img_size=56, patch_size=14, n_classes=10, apla_config=AplaConfig(16),
                             seed=0, drop_path_rate=0.2)
    fuse_apla_blocks(model).train()
    b0, b1 = model.backbone.blocks
    x = torch.randn(2, 17, 192)
    state = torch.random.get_rng_state()
    with pytest.raises(RuntimeError, match="multiple of 128.*192"):
        b1(x)
    assert torch.equal(torch.random.get_rng_state(), state)
    with pytest.raises(RuntimeError, match="CUDA"):
        b0(x)                                          # rate 0
    model.eval()
    with pytest.raises(RuntimeError, match="CUDA"):
        b1(x)


def test_fused_block_accepts_what_it_now_runs():
    """Drop path on dense input in training mode, a DINOv2 sample_drop_ratio <= 0.1, and crop lists in eval mode or at
    rate 0 pass the checks: on a CPU tensor the block then stops at its CUDA check."""
    model = _fused()
    b0, b1 = model.backbone.blocks
    x = torch.randn(2, 17, 128)
    for blk, arg in ((b1, x), (b0, [x, x[:1]])):                            # rate 0.2 dense; rate 0 crops
        with pytest.raises(RuntimeError, match="CUDA"):
            blk(arg)
    b1.sample_drop_ratio = 0.1
    with pytest.raises(RuntimeError, match="CUDA"):
        b1(x)
    model.eval()
    with pytest.raises(RuntimeError, match="CUDA"):
        b1([x, x[:1]])
    assert not b1._drop_path_active() and b0._drop_path_active() is False
    model.train()
    assert b1._drop_path_active() and not b0._drop_path_active()

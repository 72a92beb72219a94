"""The attention-probability entry points of the C ABI refuse malformed arguments before touching a device (CPU only):
the kernel (`apla_attn_probs`: null pointers, empty shapes, q_rows outside [1, N]) and the engine's CLS attention map
(`apla_engine_cls_attention`: the checks of `apla_engine_infer` plus a null output)."""
from apla_b200._lib import LIB


def _refused(rc, what):
    dll = LIB.load()
    assert rc == 1, (what, rc)
    msg = dll.apla_last_error()
    assert msg, what
    return msg.decode()


def test_attn_probs_refuses_bad_arguments_without_a_gpu():
    dll = LIB.load()
    fake = 256                                        # a non-NULL address that is never dereferenced
    for args, what in (((None, fake, fake), "qkv"), ((fake, None, fake), "lse"), ((fake, fake, None), "probs")):
        assert "null" in _refused(dll.apla_attn_probs(*args, 2, 257, 12, 257, 0.125, None), f"{what}=NULL")
    for B, N, H in ((0, 257, 12), (2, 0, 12), (2, 257, 0), (-1, 257, 12)):
        assert "bad shape" in _refused(dll.apla_attn_probs(fake, fake, fake, B, N, H, 1, 0.125, None), f"{B},{N},{H}")
    for q_rows in (0, -1, 258):
        assert "q_rows" in _refused(dll.apla_attn_probs(fake, fake, fake, 2, 257, 12, q_rows, 0.125, None),
                                    f"q_rows={q_rows}")


def test_engine_cls_attention_refuses_bad_arguments_without_a_gpu():
    dll = LIB.load()
    fake = 256
    assert "null" in _refused(dll.apla_engine_cls_attention(None, fake, 1, fake, None), "engine handle=NULL")
    e = dll.apla_engine_create(4, 17, 128, 2, 2, 512, 10, 14, 56, 640, 16, 64, 0, 1e-6, 0.125)
    assert e
    try:
        assert "null" in _refused(dll.apla_engine_cls_attention(e, None, 1, fake, None), "images=NULL")
        assert "null" in _refused(dll.apla_engine_cls_attention(e, fake, 1, None, None), "probs=NULL")
        assert "workspace" in _refused(dll.apla_engine_cls_attention(e, fake, 1, fake, None), "without workspace")
        assert dll.apla_engine_set_option(e, b"infer_batch", 4) == 0
        for n_img in (0, 5, -3):
            assert "outside" in _refused(dll.apla_engine_cls_attention(e, fake, n_img, fake, None), f"n_img={n_img}")
        for n in ("infer_x", "infer_ln", "infer_qkv", "infer_ao", "infer_lse", "infer_gelu", "infer_patches",
                  "infer_pe_out", "infer_cls_ln"):
            assert dll.apla_engine_set_ptr(e, n.encode(), -1, fake) == 0
        assert "not set" in _refused(dll.apla_engine_cls_attention(e, fake, 2, fake, None), "without weights")
    finally:
        dll.apla_engine_destroy(e)

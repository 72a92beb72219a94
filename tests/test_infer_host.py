"""The evaluation entry points of the C ABI refuse malformed arguments before touching a device (CPU only): the
engine's forward-only call (image count, missing workspace, null buffers), the forward-only block, the fc1 GEMM that
writes gelu(h) only and the evaluation sums."""
import ctypes

from apla_b200._lib import LIB, BlockWeights


def _refused(rc, what):
    dll = LIB.load()
    assert rc == 1, (what, rc)
    msg = dll.apla_last_error()
    assert msg, what
    return msg.decode()


def test_infer_entry_points_refuse_bad_arguments_without_a_gpu():
    dll = LIB.load()
    fake = 256                                        # a non-NULL address that is never dereferenced
    # fc1, forward only: empty problem, null output
    assert "empty" in _refused(dll.apla_gemm_bias_gelu_only_fwd(fake, 64, fake, 64, None, fake, 256, 0, 256, 64, None),
                               "gelu_only M=0")
    assert "null" in _refused(dll.apla_gemm_bias_gelu_only_fwd(fake, 64, fake, 64, None, None, 256, 128, 256, 64, None),
                              "gelu_only g=NULL")
    # evaluation sums
    assert "empty" in _refused(dll.apla_eval_accumulate(fake, fake, 0, 10, fake, None), "eval B=0")
    assert "null" in _refused(dll.apla_eval_accumulate(fake, None, 4, 10, fake, None), "eval labels=NULL")
    assert "null" in _refused(dll.apla_eval_accumulate(fake, fake, 4, 10, None, None), "eval acc=NULL")

    # forward-only block: null weights, empty problem, a missing buffer
    assert "null weights" in _refused(dll.apla_block_fwd_infer(None, fake, fake, fake, fake, fake, fake, fake, fake, None,
                                                               1, 8, 8, None), "block null weights")
    w = BlockWeights()
    for n in ("wqkv", "wproj", "wfc1", "wfc2", "ln1w", "ln1b", "ln2w", "ln2b"):
        setattr(w, n, fake)
    w.D, w.H, w.hidden, w.eps1, w.eps2, w.scale = 128, 2, 512, 1e-6, 1e-6, 0.125
    wp = ctypes.addressof(w)
    assert "empty" in _refused(dll.apla_block_fwd_infer(wp, fake, fake, fake, fake, fake, fake, fake, fake, None, 1, 8, 0,
                                                        None), "block T=0")
    assert "null buffer" in _refused(dll.apla_block_fwd_infer(wp, fake, fake, fake, fake, fake, fake, None, fake, None, 1,
                                                              8, 8, None), "block lse_tmp=NULL")
    assert "alias" in _refused(dll.apla_block_fwd_infer(wp, fake, fake, 512, fake, fake, fake, fake, fake, None, 1, 8, 8,
                                                        None), "block x_mid aliases x_in")

    # engine: no workspace, then n_img outside [1, capacity], then a missing workspace buffer
    e = dll.apla_engine_create(4, 17, 128, 2, 2, 512, 10, 14, 56, 640, 16, 64, 0, 1e-6, 0.125)
    assert e
    try:
        assert "null" in _refused(dll.apla_engine_infer(e, None, 1, fake, None, None), "engine images=NULL")
        assert "null" in _refused(dll.apla_engine_infer(e, fake, 1, None, None, None), "engine logits=NULL")
        assert "workspace" in _refused(dll.apla_engine_infer(e, fake, 1, fake, None, None), "engine without workspace")
        assert dll.apla_engine_set_option(e, b"infer_batch", -1) == 1
        assert dll.apla_engine_set_option(e, b"infer_batch", 4) == 0
        for n_img in (0, 5, -3):
            assert "outside" in _refused(dll.apla_engine_infer(e, fake, n_img, fake, None, None), f"engine n_img={n_img}")
        names = ["infer_x", "infer_ln", "infer_qkv", "infer_ao", "infer_lse", "infer_gelu", "infer_patches",
                 "infer_pe_out", "infer_cls_ln"]
        for n in names[:-1]:
            assert dll.apla_engine_set_ptr(e, n.encode(), -1, fake) == 0
        assert "infer_cls_ln" in _refused(dll.apla_engine_infer(e, fake, 2, fake, None, None), "engine missing cls_ln")
        assert dll.apla_engine_set_ptr(e, b"infer_cls_ln", -1, fake) == 0
        # the weights are still unset: refused before any launch as well
        assert "not set" in _refused(dll.apla_engine_infer(e, fake, 2, fake, None, None), "engine without weights")
    finally:
        dll.apla_engine_destroy(e)

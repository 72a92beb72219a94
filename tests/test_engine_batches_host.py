"""The partial-batch / soft-target entry points of the C ABI refuse malformed arguments before touching a device (CPU
only): apla_engine_forward_n (image count outside [1, B], labels and targets together, null images or handle) and
apla_cross_entropy_soft (empty problem, null buffers)."""
from apla_b200._lib import LIB


def _refused(rc, what):
    dll = LIB.load()
    assert rc == 1, (what, rc)
    msg = dll.apla_last_error()
    assert msg, what
    return msg.decode()


def test_soft_cross_entropy_refuses_bad_arguments_without_a_gpu():
    dll = LIB.load()
    fake = 256                                        # a non-NULL address that is never dereferenced
    for B, C in ((0, 10), (4, 0), (-1, 10)):
        assert "empty" in _refused(dll.apla_cross_entropy_soft(fake, fake, fake, fake, B, C, 1.0, 1.0, None),
                                   f"B={B} C={C}")
    for i in range(4):
        args = [fake] * 4
        args[i] = None
        assert "null" in _refused(dll.apla_cross_entropy_soft(*args, 4, 10, 1.0, 1.0, None), f"pointer {i} NULL")


def test_forward_n_refuses_bad_arguments_without_a_gpu():
    dll = LIB.load()
    fake = 256
    assert "null" in _refused(dll.apla_engine_forward_n(None, fake, 1, fake, None, 1.0, 1.0, None), "null handle")
    e = dll.apla_engine_create(4, 17, 128, 2, 2, 512, 10, 14, 56, 640, 16, 64, 0, 1e-6, 0.125)
    assert e
    try:
        assert "null" in _refused(dll.apla_engine_forward_n(e, None, 2, fake, None, 1.0, 1.0, None), "images=NULL")
        for n_img in (0, 5, -1):
            assert "outside" in _refused(dll.apla_engine_forward_n(e, fake, n_img, fake, None, 1.0, 1.0, None),
                                         f"n_img={n_img}")
        assert "both" in _refused(dll.apla_engine_forward_n(e, fake, 2, fake, fake, 1.0, 1.0, None), "labels and targets")
        # valid arguments, but the engine's buffers are unset: still refused before any launch
        for labels, targets in ((fake, None), (None, fake), (None, None)):
            assert "not set" in _refused(dll.apla_engine_forward_n(e, fake, 4, labels, targets, 1.0, 1.0, None),
                                         "engine without buffers")
    finally:
        dll.apla_engine_destroy(e)

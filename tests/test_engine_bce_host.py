"""Multi-label (BCE-with-logits) training refuses malformed arguments before touching a device (CPU only): the C entries
apla_bce_with_logits and apla_eval_accumulate_bce (null buffers, empty shapes), the engine option "criterion" (values
other than 0 and 1), int64 labels on a criterion-1 engine, and FineTuneEngine's check of the trainer's criterion."""
import pytest
import torch
import torch.nn as nn

from apla_b200._lib import LIB


def _refused(rc, what):
    dll = LIB.load()
    assert rc == 1, (what, rc)
    msg = dll.apla_last_error()
    assert msg, what
    return msg.decode()


def test_bce_entries_refuse_bad_arguments_without_a_gpu():
    dll = LIB.load()
    fake = 256                                        # a non-NULL address that is never dereferenced
    for B, C in ((0, 10), (4, 0), (-1, 10), (4, -1)):
        assert "empty" in _refused(dll.apla_bce_with_logits(fake, fake, fake, fake, B, C, 1.0, 1.0, None), f"B={B} C={C}")
        assert "empty" in _refused(dll.apla_eval_accumulate_bce(fake, fake, B, C, fake, None), f"eval B={B} C={C}")
    for i in range(4):
        args = [fake] * 4
        args[i] = None
        assert "null" in _refused(dll.apla_bce_with_logits(*args, 4, 10, 1.0, 1.0, None), f"pointer {i} NULL")
    for i in range(3):
        args = [fake] * 3
        args[i] = None
        assert "null" in _refused(dll.apla_eval_accumulate_bce(args[0], args[1], 4, 10, args[2], None),
                                  f"eval pointer {i} NULL")


def test_criterion_option_and_int64_labels_refused_without_a_gpu():
    dll = LIB.load()
    fake = 256
    e = dll.apla_engine_create(4, 17, 128, 2, 2, 512, 10, 14, 56, 640, 16, 64, 0, 1e-6, 0.125)
    assert e
    try:
        for v in (-1, 2):
            assert "criterion" in _refused(dll.apla_engine_set_option(e, b"criterion", v), f"criterion={v}")
        assert dll.apla_engine_set_option(e, b"criterion", 0) == 0
        # cross-entropy engine: int64 labels pass the argument checks and stop at the unset buffers
        assert "not set" in _refused(dll.apla_engine_forward(e, fake, fake, 1.0, 1.0, None), "CE labels")
        assert dll.apla_engine_set_option(e, b"criterion", 1) == 0
        # BCE engine: int64 labels are refused before the buffer check, by both entries; fp32 targets are not
        msg = _refused(dll.apla_engine_forward_n(e, fake, 2, fake, None, 1.0, 1.0, None), "forward_n labels")
        assert "criterion 1" in msg and "not set" not in msg, msg
        msg = _refused(dll.apla_engine_forward(e, fake, fake, 1.0, 1.0, None), "forward labels")
        assert "criterion 1" in msg and "not set" not in msg, msg
        assert "not set" in _refused(dll.apla_engine_forward_n(e, fake, 2, None, fake, 1.0, 1.0, None), "BCE targets")
        assert "not set" in _refused(dll.apla_engine_forward(e, fake, None, 1.0, 1.0, None), "logits only")
    finally:
        dll.apla_engine_destroy(e)


def test_criterion_check_accepts_the_reference_losses():
    from apla_b200.engine import criterion_code
    assert criterion_code(None) == 0
    assert criterion_code(nn.CrossEntropyLoss()) == 0
    assert criterion_code(nn.BCEWithLogitsLoss()) == 1


@pytest.mark.parametrize("crit,match", [
    (nn.MSELoss(), "MSELoss is not supported"),
    (nn.BCELoss(), "BCELoss is not supported"),
    (nn.BCEWithLogitsLoss(reduction="sum"), "reduction='sum'"),
    (nn.BCEWithLogitsLoss(pos_weight=torch.ones(3)), "pos_weight=set"),
    (nn.BCEWithLogitsLoss(weight=torch.ones(3)), "'mean', weight=set"),
    (nn.CrossEntropyLoss(label_smoothing=0.1), "smoothed fp32"),
    (nn.CrossEntropyLoss(reduction="none"), "reduction='none'"),
])
def test_criterion_check_refuses_other_losses(crit, match):
    from apla_b200.engine import FineTuneEngine, criterion_code
    with pytest.raises(ValueError, match=match) as info:
        criterion_code(crit)
    assert "supported: None or nn.CrossEntropyLoss()" in str(info.value)
    # the engine refuses it before it looks for a device
    with pytest.raises(ValueError, match=match):
        FineTuneEngine(None, batch_size=4, img_size=56, criterion=crit)

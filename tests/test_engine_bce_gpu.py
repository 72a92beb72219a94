"""Multi-label fine-tuning on the B200: the BCE-with-logits head kernel and its evaluation sums against torch in float64,
and engines built with `criterion=nn.BCEWithLogitsLoss()` against the fp32 CPU oracle with BCEWithLogitsLoss(mean) as the
loss -- single steps on full and partial batches, whole steps eager and from graphs, step_from_host, evaluate.  The
oracle's forward, clip and AdamW are used as they are; only the loss differs.  A cross-entropy engine built from an
explicit nn.CrossEntropyLoss() runs the default engine's launches.
Bars of the steps as in test_engine_gpu.py: logits / loss relative error <= 1e-2, gradient cosine >= 0.999 and relative
error <= 1e-2."""
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from helpers import build_case, cosine, rel, synthetic_batch
from test_engine_batches_gpu import PARTIAL_CASES, _check_against_oracle, _oracle_of, _poison_stale_rows, _small

pytestmark = pytest.mark.gpu

BCE = F.binary_cross_entropy_with_logits


def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from apla_b200._lib import require_device
    require_device()


def _engine(model, batch, img, **kw):
    _need_gpu()
    from apla_b200.engine import FineTuneEngine
    return FineTuneEngine(model, batch_size=batch, img_size=img, **kw)


def _multi_hot(n, C, seed, p=0.3):
    g = torch.Generator().manual_seed(seed)
    return (torch.rand(n, C, generator=g) < p).float()


def _bce_loss_and_grads(O, sd, cfg, images, targets):
    """`O.loss_and_grads` with BCEWithLogitsLoss(mean) in place of the cross-entropy."""
    keys = O.trainable_keys(cfg, sd)
    leaves = {k: sd[k].detach().clone().requires_grad_(True) for k in keys}
    logits = O.forward_logits(dict(sd, **leaves), cfg, images)
    loss = BCE(logits, targets)
    gs = torch.autograd.grad(loss, [leaves[k] for k in keys])
    return O.StepResult(logits.detach(), loss.detach(), dict(zip(keys, gs)))


def _bce_fine_tune_step(O, sd, cfg, images, targets, st):
    """`O.fine_tune_step` (single rank, clip 1.0, AdamW at the engine's defaults) with BCEWithLogitsLoss(mean)."""
    res = _bce_loss_and_grads(O, sd, cfg, images, targets)
    grads = {k: g.clone() for k, g in res.grads.items()}
    res.grad_norm = O.clip_grad_norm_(grads, 1.0)
    O.adamw_step(sd, grads, st)
    res.new_params = {k: sd[k].clone() for k in grads}
    return res


# ---- the kernels --------------------------------------------------------------------------------------------------
def _targets(kind, B, C, g):
    return {
        "multi_hot": lambda: (torch.rand(B, C, generator=g) < 0.3).float(),
        "uniform": lambda: torch.rand(B, C, generator=g),
        "zeros": lambda: torch.zeros(B, C),
        "ones": lambda: torch.ones(B, C),
        "outside_0_1": lambda: torch.rand(B, C, generator=g) * 3.0 - 1.0,     # [-1, 2): torch checks nothing
    }[kind]()


def _logits(kind, B, C, g):
    z = torch.randn(B, C, generator=g) * 3.0
    if kind == "extreme":      # a fifth of the elements (at least one) at +-30, +-100, +-1e4
        pick = torch.randperm(B * C, generator=g)[:max(1, B * C // 5)]
        vals = torch.tensor([30.0, -30.0, 100.0, -100.0, 1e4, -1e4])
        z.view(-1)[pick] = vals[torch.arange(pick.numel()) % vals.numel()]
    return z


def _bce_dev(z, t, grad_scale=1.0, loss_scale=1.0, canary=64):
    """apla_bce_with_logits into a NaN-filled dlogits buffer with a canary tail; -> (dlogits, loss, tail)."""
    from apla_b200._lib import LIB, ptr, stream
    B, C = z.shape
    buf = torch.full((B * C + canary,), float("nan"), device="cuda")
    buf[B * C:] = 12345.0
    loss = torch.zeros(1, device="cuda")
    LIB.call("apla_bce_with_logits", ptr(z), ptr(t), ptr(buf), ptr(loss), B, C, grad_scale, loss_scale, stream())
    torch.cuda.synchronize()
    return buf[:B * C].view(B, C).cpu(), float(loss), buf[B * C:].cpu()


@pytest.mark.parametrize("B,C", [(1, 1), (3, 7), (64, 555), (1024, 1000), (5, 4097)])
def test_bce_kernel_matches_torch(B, C):
    """Sum loss and dlogits (grad_scale 1) against F.binary_cross_entropy_with_logits(reduction="sum") and its autograd
    gradient in float64, for five kinds of target and logits of both ordinary and extreme size: everything finite, the
    buffer's canary tail untouched."""
    _need_gpu()
    g = torch.Generator().manual_seed(B * 7919 + C)
    for zk in ("randn3", "extreme"):
        z = _logits(zk, B, C, g)
        for tk in ("multi_hot", "uniform", "zeros", "ones", "outside_0_1"):
            t = _targets(tk, B, C, g)
            dl, loss, tail = _bce_dev(z.cuda(), t.cuda())
            zd = z.double().requires_grad_(True)
            ref = BCE(zd, t.double(), reduction="sum")
            (gref,) = torch.autograd.grad(ref, zd)
            what = (zk, tk)
            assert torch.isfinite(dl).all() and torch.isfinite(torch.tensor(loss)), what
            assert torch.equal(tail, torch.full_like(tail, 12345.0)), what
            assert abs(loss - float(ref)) <= 1e-5 * abs(float(ref)) + 1e-30, (what, loss, float(ref))
            assert float((dl.double() - gref).abs().max()) <= 1e-6, (what, float((dl.double() - gref).abs().max()))
    # the scales: mean reduction over the B*C elements
    z, t = _logits("randn3", B, C, g), _targets("uniform", B, C, g)
    dl, loss, _ = _bce_dev(z.cuda(), t.cuda(), 1.0 / (B * C), 1.0 / (B * C))
    zd = z.double().requires_grad_(True)
    ref = BCE(zd, t.double())
    (gref,) = torch.autograd.grad(ref, zd)
    assert abs(loss - float(ref)) <= 1e-5 * abs(float(ref)), (loss, float(ref))
    assert rel(dl, gref) <= 1e-5, rel(dl, gref)


def test_bce_eval_kernel_sums_three_batches():
    """Three calls into one double[2]: the loss sum within 1e-6 relative of float64 torch, the count of elements with
    (z > 0) == (t >= 0.5) exact -- including z == 0 (not positive) and t == 0.5 (a positive label)."""
    _need_gpu()
    from apla_b200._lib import LIB, ptr, stream
    g = torch.Generator().manual_seed(5)
    acc = torch.zeros(2, dtype=torch.float64, device="cuda")
    want_l, want_h = 0.0, 0
    for (B, C), zk, tk in (((64, 555), "randn3", "multi_hot"), ((1024, 1000), "extreme", "uniform"),
                           ((5, 4097), "randn3", "outside_0_1")):
        z, t = _logits(zk, B, C, g), _targets(tk, B, C, g)
        z[0, :3] = 0.0
        t[0, 1:4] = 0.5
        zc, tc = z.cuda(), t.cuda()           # held until the kernel has run
        LIB.call("apla_eval_accumulate_bce", ptr(zc), ptr(tc), B, C, ptr(acc), stream())
        torch.cuda.synchronize()
        want_l += float(BCE(z.double(), t.double(), reduction="sum"))
        want_h += int(((z > 0) == (t >= 0.5)).sum())
    got_l, got_h = acc.tolist()
    assert abs(got_l - want_l) <= 1e-6 * abs(want_l), (got_l, want_l)
    assert got_h == float(want_h), (got_h, want_h)


# ---- the engine ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(PARTIAL_CASES))
def test_bce_step_matches_oracle(name, monkeypatch):
    """Multi-hot targets through a BCE engine, at n = batch_size and at a partial n (stale rows NaN-poisoned first), in
    every cls_only_last_block mode of the case: loss, logits[:n] and every trainable gradient against the oracle with
    BCEWithLogitsLoss(mean) on the same n images."""
    _need_gpu()
    factory, B, img, sizes, modes, side = PARTIAL_CASES[name]
    monkeypatch.setenv("APLA_SIDE_WGRAD", side)
    model = factory()
    O, cfg, sd = _oracle_of(model)
    C = cfg.n_classes
    images, _ = synthetic_batch(B, img, C, seed=61)
    targets = _multi_hot(B, C, seed=62)
    full_images, full_targets = synthetic_batch(B, img, C, seed=63)[0].cuda(), _multi_hot(B, C, seed=64).cuda()
    ns = (B, sizes[-1])
    refs = {n: _bce_loss_and_grads(O, sd, cfg, images[:n], targets[:n]) for n in ns}
    for mode in modes:
        eng = _engine(model, B, img, cls_only_last_block=mode, criterion=nn.BCEWithLogitsLoss())
        for n in ns:
            eng.forward(full_images, full_targets)
            eng.backward()
            torch.cuda.synchronize()
            if n < B:
                _poison_stale_rows(eng, n)
            out = eng.forward(images[:n].cuda(), targets[:n].cuda())
            assert out.shape == (n, C)
            eng.backward()
            _check_against_oracle(eng, refs[n], n)
        del eng


@pytest.mark.parametrize("use_graph", [False, True])
def test_bce_whole_steps_match_fine_tune_step(use_graph):
    """Three whole steps on one buffer pair (with graphs: eager, captured, replayed): parameters and both Adam moments
    after every step against the oracle's step with BCEWithLogitsLoss(mean)."""
    _need_gpu()
    B, C = 6, 10
    model = _small(128, 2, 2, 16)
    O, cfg, sd = _oracle_of(model)
    st = O.AdamWState()
    eng = _engine(model, B, 56, use_graph=use_graph, criterion=nn.BCEWithLogitsLoss())
    p0 = {k: v.detach().cpu().clone() for k, v in eng.named_params().items()}
    buf = (torch.empty(B, 3, 56, 56, device="cuda"), torch.empty(B, C, device="cuda"))
    names = eng.trainable_names()
    for k in range(3):
        images = synthetic_batch(B, 56, C, seed=800 + k)[0]
        targets = _multi_hot(B, C, seed=850 + k)
        ref = _bce_fine_tune_step(O, sd, cfg, images, targets, st)
        buf[0].copy_(images)
        buf[1].copy_(targets)
        loss = eng.step(*buf)
        torch.cuda.synchronize()
        assert abs(float(loss) - float(ref.loss)) <= 1e-2 * abs(float(ref.loss)), (k, float(loss), float(ref.loss))
        params = eng.named_params()
        p = torch.cat([params[key].cpu().flatten() for key in names])
        p_ref = torch.cat([ref.new_params[key].flatten() for key in names])
        assert rel(p, p_ref) <= 1e-2, (k, rel(p, p_ref))
        upd_o = torch.cat([(params[key].cpu() - p0[key]).flatten() for key in names])
        upd_r = torch.cat([(ref.new_params[key] - p0[key]).flatten() for key in names])
        assert torch.isfinite(upd_o).all() and cosine(upd_o, upd_r) >= 0.95, (k, cosine(upd_o, upd_r))
        m = torch.cat([eng.exp_avg[eng.slices[key]].cpu() for key in names])
        m_ref = torch.cat([st.exp_avg[key].flatten() for key in names])
        v = torch.cat([eng.exp_avg_sq[eng.slices[key]].cpu() for key in names])
        v_ref = torch.cat([st.exp_avg_sq[key].flatten() for key in names])
        assert rel(m, m_ref) <= 1e-2, (k, rel(m, m_ref))
        assert rel(v, v_ref) <= 1e-2, (k, rel(v, v_ref))
    if use_graph:
        assert len(eng._graphs) == 1


def test_bce_step_from_host_matches_eager_steps():
    """A loader-like sequence of pinned multi-label batches that ends in a partial batch, through step_from_host (two
    device slots with fp32 target slots, graphs from the second sighting) against eager step calls on a second engine."""
    _need_gpu()
    B, C = 6, 10
    batches = []
    for k, size in enumerate([6, 6, 6, 6, 6, 4]):
        images = synthetic_batch(size, 56, C, seed=900 + k)[0]
        batches.append((images.pin_memory(), _multi_hot(size, C, seed=950 + k).pin_memory()))
    host = _engine(_small(128, 2, 2, 16), B, 56, criterion=nn.BCEWithLogitsLoss())
    eager = _engine(_small(128, 2, 2, 16), B, 56, use_graph=False, criterion=nn.BCEWithLogitsLoss())
    got, want = [], []
    for images, targets in batches:
        got.append(host.step_from_host(images, targets, lag=False))
        want.append(float(eager.step(images.cuda(), targets.cuda())))
    torch.cuda.synchronize()
    assert "tgt" in host._e2e and len(host._graphs) >= 1
    for k, (a, b) in enumerate(zip(got, want)):
        assert abs(a - b) <= 1e-4 * abs(b), (k, a, b)
    assert rel(host.params, eager.params) < 1e-5


def test_bce_evaluate_matches_torch_on_predict():
    """evaluate() on a BCE engine over device and host batches (the last one partial): the mean BCE within 1e-5 relative
    of float64 torch on predict's logits, label_acc exactly equal."""
    B, C = 4, 10
    eng = _engine(build_case("tiny_r16")[0], B, 56, criterion=nn.BCEWithLogitsLoss())
    images = synthetic_batch(11, 56, C, seed=5)[0]
    targets = _multi_hot(11, C, seed=6)
    logits = eng.predict(images.cuda()).double().cpu()
    want_loss = float(BCE(logits, targets.double()))
    want_acc = int(((logits > 0) == (targets >= 0.5)).sum()) / (11 * C)
    sizes = [(0, 4), (4, 8), (8, 11)]
    dev = [(images[a:b].cuda(), targets[a:b].cuda()) for a, b in sizes]
    host = [(images[a:b].pin_memory(), targets[a:b].pin_memory()) for a, b in sizes]
    for batches in (dev, host):
        out = eng.evaluate(iter(batches))
        assert out["n"] == 11 and set(out) == {"loss", "label_acc", "n"}
        assert abs(out["loss"] - want_loss) <= 1e-5 * abs(want_loss), (out, want_loss)
        assert out["label_acc"] == want_acc, (out, want_acc)


def test_explicit_cross_entropy_is_the_default_engine():
    """criterion=nn.CrossEntropyLoss() against criterion=None on the C2 batch: the same launches, logits bitwise equal,
    loss and gradients within the default engine's own run-to-run spread (the split-K weight gradient and the loss are
    fp32 atomics, not bitwise reproducible)."""
    _need_gpu()
    from apla_b200._lib import LIB
    model = build_case("c2_vitb14_r8")[0]
    B = 8
    images, labels = synthetic_batch(B, 224, 555, seed=77)
    images, labels = images.cuda(), labels.cuda()

    def run(eng):
        before = LIB.load().apla_launch_count()
        eng.forward(images, labels)
        eng.backward()
        torch.cuda.synchronize()
        return LIB.load().apla_launch_count() - before, eng.logits.clone(), eng.loss.clone(), eng.grads.clone()

    default = _engine(model, B, 224)
    explicit = _engine(model, B, 224, criterion=nn.CrossEntropyLoss())
    d1, e1, d2 = run(default), run(explicit), run(default)
    assert e1[0] == d1[0] == d2[0]
    assert torch.equal(e1[1], d1[1]) and torch.equal(d2[1], d1[1])
    spread = rel(d2[3], d1[3])
    assert rel(e1[3], d1[3]) <= max(4 * spread, 1e-6), (rel(e1[3], d1[3]), spread)
    assert abs(float(e1[2]) - float(d1[2])) <= 1e-6 * abs(float(d1[2]))


def test_bce_engine_refuses_wrong_labels():
    _need_gpu()
    B, C = 4, 10
    eng = _engine(_small(128, 2, 2, 16), B, 56, criterion=nn.BCEWithLogitsLoss())
    images, labels = synthetic_batch(B, 56, C, seed=3)
    images, labels = images.cuda(), labels.cuda()
    targets = _multi_hot(B, C, seed=4).cuda()
    bad = [labels, targets[:3], targets[:, :9], targets.double(), labels.float()]
    for lab in bad:
        for call in (eng.forward, eng.step):
            with pytest.raises(RuntimeError, match="BCE-with-logits engine takes fp32 multi-label targets"):
                call(images, lab)
        with pytest.raises(RuntimeError, match="BCE-with-logits engine takes fp32 multi-label targets"):
            eng.step_from_host(images.cpu(), lab.cpu(), lag=False)
        with pytest.raises(RuntimeError, match="targets must be fp32"):
            eng.evaluate([(images, lab)])
    # a refused batch leaves the engine usable
    eng.step(images, targets)
    torch.cuda.synchronize()
    assert torch.isfinite(eng.params).all() and float(eng.loss) > 0

"""Training steps on batches other than `batch_size` images with hard labels, on the B200: the partial last batch of an
epoch (1 <= n < B images through the engine's n-row launch sequence) and probability targets (mixup / cutmix /
label smoothing, fp32 [n, C]) through the soft-target cross-entropy kernel.  References: the fp32 CPU oracle on the same
n images (`loss_and_grads`, `fine_tune_step`) and torch's F.cross_entropy with probability targets.
Bars as in test_engine_gpu.py: logits / loss relative error <= 1e-2, gradient cosine >= 0.999 and relative error <= 1e-2."""
import pytest
import torch
import torch.nn.functional as F

from helpers import build_case, cosine, perturb_module, rel, synthetic_batch

pytestmark = pytest.mark.gpu


def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")


def _engine(model, batch, img, **kw):
    _need_gpu()
    from apla_b200.engine import FineTuneEngine
    return FineTuneEngine(model, batch_size=batch, img_size=img, **kw)


def _oracle_of(model):
    """-> (oracle module, cfg, fp32 state dict) describing `model` as built (before any engine step)."""
    from oracle import apla_oracle as O
    bb = model.backbone
    blk = bb.blocks[0]
    cfg = O.VitCfg(embed_dim=bb.cls_token.shape[-1], depth=len(bb.blocks), num_heads=blk.attn.num_heads,
                   patch_size=bb.patch_embed.proj.kernel_size[0], n_classes=model.fc.out_features,
                   ln_eps=float(blk.norm1.eps))
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    return O, cfg, sd


def _small(dim, depth, heads, r, seed=0):
    from apla_b200.config import AplaConfig
    from apla_b200.hostvit import VitArch, build_classifier
    model = build_classifier(VitArch(dim, depth, heads), img_size=56, patch_size=14, n_classes=10,
                             apla_config=AplaConfig(r), seed=seed)
    perturb_module(model)
    return model


def _soft_targets(labels, C, seed, smoothing=0.1):
    """timm Mixup-style targets: lam * smooth(onehot(y)) + (1 - lam) * smooth(onehot(y.flip(0)))."""
    g = torch.Generator().manual_seed(seed)
    lam = 0.2 + 0.6 * float(torch.rand(1, generator=g))
    off, on = smoothing / C, 1.0 - smoothing + smoothing / C
    a = torch.full((labels.shape[0], C), off).scatter_(1, labels[:, None], on)
    b = torch.full((labels.shape[0], C), off).scatter_(1, labels.flip(0)[:, None], on)
    return (lam * a + (1.0 - lam) * b).float()


def _check_against_oracle(eng, ref, n):
    torch.cuda.synchronize()
    assert rel(eng.logits[:n], ref.logits) <= 1e-2, rel(eng.logits[:n], ref.logits)
    assert abs(float(eng.loss) - float(ref.loss)) <= 1e-2 * abs(float(ref.loss)), (float(eng.loss), float(ref.loss))
    g = eng.named_grads()
    ours = torch.cat([g[k].flatten().cpu() for k in eng.trainable_names()])
    theirs = torch.cat([ref.grads[k].flatten() for k in eng.trainable_names()])
    assert cosine(ours, theirs) >= 0.999, cosine(ours, theirs)
    assert rel(ours, theirs) <= 1e-2, rel(ours, theirs)


# (model factory, batch_size, img, partial sizes, cls_only_last_block modes, APLA_SIDE_WGRAD)
PARTIAL_CASES = {
    "tiny_r16": (lambda: _small(128, 2, 2, 16), 6, 56, (1, 3, 5), (0, 1, 2), "0"),
    "tiny_r16_side_wgrad": (lambda: _small(128, 3, 2, 16), 6, 56, (1, 3, 5), (2,), "1"),   # two dsub slots, side stream
    "tiny_r192_full_rows": (lambda: _small(256, 2, 4, 192), 5, 56, (1, 3, 4), (0, 1, 2), "0"),   # dense-dY weight grad
    "c1_vits16_r32": (lambda: build_case("c1_vits16_r32")[0], 8, 224, (1, 3, 7), (0, 1, 2), "0"),   # N = 197
    "c2_vitb14_r8": (lambda: build_case("c2_vitb14_r8")[0], 8, 224, (1, 5), (2,), "0"),              # N = 257
}


@pytest.mark.parametrize("name", list(PARTIAL_CASES))
def test_partial_batch_matches_oracle(name, monkeypatch):
    """A full batch first (so that every buffer holds values of other images beyond the partial rows), those rows then
    filled with NaN, then partial batches of n images: loss, logits[:n] and every trainable gradient against the oracle
    on the same n images.  n = 1 runs the backward GEMMs at M = N (197 / 257 rows); odd n gives a weight-gradient K that
    is not a multiple of 64."""
    _need_gpu()
    factory, B, img, sizes, modes, side = PARTIAL_CASES[name]
    monkeypatch.setenv("APLA_SIDE_WGRAD", side)
    model = factory()
    O, cfg, sd = _oracle_of(model)
    images, labels = synthetic_batch(B, img, cfg.n_classes, seed=55)
    full_images, full_labels = synthetic_batch(B, img, cfg.n_classes, seed=56)
    refs = {n: O.loss_and_grads(sd, cfg, images[:n], labels[:n]) for n in sizes}
    for mode in modes:
        eng = _engine(model, B, img, cls_only_last_block=mode)
        assert eng.side_wgrad == (side == "1")
        fi, fl = full_images.cuda(), full_labels.cuda()
        for n in sizes:
            eng.forward(fi, fl)
            eng.backward()
            torch.cuda.synchronize()
            _poison_stale_rows(eng, n)
            out = eng.forward(images[:n].cuda(), labels[:n].cuda())
            assert out.shape == (n, cfg.n_classes) and out.data_ptr() == eng.logits.data_ptr()
            eng.backward()
            _check_against_oracle(eng, refs[n], n)
        del eng


_TOKEN_ROWS = ("qkv", "ao", "hpre", "lse", "ln_out", "gelu_out", "dx", "dxb", "dO", "dqkv", "delta")
_IMAGE_ROWS = ("cls_ln", "dcls", "logits", "dlogits")


def _poison_stale_rows(eng, n):
    """NaN into every row beyond the next step's n images of every training buffer that has one per token, patch or image
    (residual checkpoints, qkv / ao / hpre / lse of every block, the transients, dsub, the head's rows): a kernel that reads
    one of them turns the step's loss, gradients and, through AdamW, parameters into NaN.  The one exception is the last
    block's ao under the CLS-only attention (cls_only_last_block = 2): only its CLS rows are ever written and the weight
    gradient reads the zeros of the others against zero dsub rows, so only the CLS rows of images >= n are poisoned."""
    s, nan = eng.shape, float("nan")
    N, P, L = s["N"], s["P"], s["L"]
    poisoned = set()
    for (name, block), t in eng.buffers.items():
        if t is None or not t.is_floating_point():
            continue
        if name in ("xs", "dsub"):                                  # [2L+1, T, D] / [slots, T, r_pad]
            t[:, n * N:] = nan
        elif name == "ao" and block == L - 1 and eng.cls_only_last_block >= 2:
            t.view(s["B"], N, -1)[n:, 0] = nan
        elif name in _TOKEN_ROWS:
            t[n * N:] = nan
        elif name in ("patches", "pe_out"):
            t[n * P:] = nan
        elif name in _IMAGE_ROWS:
            t[n:] = nan
        else:
            continue
        poisoned.add(name)
    assert {"xs", "qkv", "ao", "hpre", "dx", "dxb", "logits"} <= poisoned, poisoned


@pytest.mark.parametrize("use_graph", [False, True])
def test_full_partial_full_sequence_matches_fine_tune_step(use_graph):
    """full -> partial -> full, three times over the same two buffer pairs (so that with graphs the partial batch is run
    eagerly, captured, then replayed), with stale rows poisoned before each partial step: parameters and Adam moments
    after every step against the oracle's fine_tune_step on the same sequence."""
    _need_gpu()
    B, n = 6, 2
    model = _small(128, 2, 2, 16)
    O, cfg, sd = _oracle_of(model)
    st = O.AdamWState()
    eng = _engine(model, B, 56, use_graph=use_graph)
    p0 = {k: v.detach().cpu().clone() for k, v in eng.named_params().items()}
    buf_full = (torch.empty(B, 3, 56, 56, device="cuda"), torch.empty(B, dtype=torch.int64, device="cuda"))
    buf_part = (torch.empty(n, 3, 56, 56, device="cuda"), torch.empty(n, dtype=torch.int64, device="cuda"))
    for k, size in enumerate([B, n, B, n, B, n, B]):
        images, labels = synthetic_batch(size, 56, 10, seed=700 + k)
        ref = O.fine_tune_step(sd, cfg, images, labels, st)
        buf = buf_full if size == B else buf_part
        buf[0].copy_(images)
        buf[1].copy_(labels)
        if size < B:
            torch.cuda.synchronize()
            _poison_stale_rows(eng, size)
        loss = eng.step(*buf)
        torch.cuda.synchronize()
        assert abs(float(loss) - float(ref.loss)) <= 1e-2 * abs(float(ref.loss)), (k, float(loss), float(ref.loss))
        params = eng.named_params()
        upd_o = torch.cat([(params[key].cpu() - p0[key]).flatten() for key in eng.trainable_names()])
        upd_r = torch.cat([(ref.new_params[key] - p0[key]).flatten() for key in eng.trainable_names()])
        assert torch.isfinite(upd_o).all(), k
        assert cosine(upd_o, upd_r) >= 0.95, (k, cosine(upd_o, upd_r))
        m = torch.cat([eng.exp_avg[eng.slices[key]].cpu() for key in eng.trainable_names()])
        m_ref = torch.cat([st.exp_avg[key].flatten() for key in eng.trainable_names()])
        v = torch.cat([eng.exp_avg_sq[eng.slices[key]].cpu() for key in eng.trainable_names()])
        v_ref = torch.cat([st.exp_avg_sq[key].flatten() for key in eng.trainable_names()])
        assert cosine(m, m_ref) >= 0.999 and rel(m, m_ref) <= 1e-2, (k, cosine(m, m_ref), rel(m, m_ref))
        assert rel(v, v_ref) <= 2e-2, (k, rel(v, v_ref))
    if use_graph:
        assert len(eng._graphs) == 2


def test_forward_n_full_batch_equals_old_entry():
    """apla_engine_forward_n with n_img = B and hard labels issues apla_engine_forward's launches: logits and every residual
    checkpoint bitwise equal; loss and gradients within the step's own run-to-run spread (split-K weight gradient and the
    loss are fp32 atomics, not bitwise reproducible)."""
    _need_gpu()
    from apla_b200._lib import LIB, ptr, stream
    model = build_case("c1_vits16_r32")[0]
    B = 8
    eng = _engine(model, B, 224)
    images, labels = synthetic_batch(B, 224, 555, seed=77)
    images, labels = images.cuda(), labels.cuda()

    def run(new):
        if new:
            LIB.call("apla_engine_forward_n", eng._handle, ptr(images), B, ptr(labels), None, 1.0 / B, 1.0 / B, stream())
        else:
            LIB.call("apla_engine_forward", eng._handle, ptr(images), ptr(labels), 1.0 / B, 1.0 / B, stream())
        eng.backward()
        torch.cuda.synchronize()
        return eng.logits.clone(), eng.xs.clone(), eng.loss.clone(), eng.grads.clone()

    old1, new1, old2 = run(False), run(True), run(False)
    assert torch.equal(new1[0], old1[0]) and torch.equal(new1[1], old1[1])
    assert torch.equal(old2[0], old1[0]) and torch.equal(old2[1], old1[1])
    spread_g = rel(old2[3], old1[3])
    assert rel(new1[3], old1[3]) <= max(4 * spread_g, 1e-6), (rel(new1[3], old1[3]), spread_g)
    assert abs(float(new1[2]) - float(old1[2])) <= 1e-6 * abs(float(old1[2]))


def _ce_soft(logits, targets, grad_scale, loss_scale):
    from apla_b200._lib import LIB, ptr, stream
    B, C = logits.shape
    dl = torch.full_like(logits, float("nan"))
    loss = torch.zeros(1, dtype=torch.float32, device=logits.device)
    LIB.call("apla_cross_entropy_soft", ptr(logits), ptr(targets), ptr(dl), ptr(loss), B, C, grad_scale, loss_scale,
             stream())
    return dl, loss


def _ce_hard(logits, labels, grad_scale, loss_scale):
    from apla_b200._lib import LIB, ptr, stream
    B, C = logits.shape
    dl = torch.full_like(logits, float("nan"))
    loss = torch.zeros(1, dtype=torch.float32, device=logits.device)
    LIB.call("apla_cross_entropy", ptr(logits), ptr(labels), ptr(dl), ptr(loss), B, C, grad_scale, loss_scale, stream())
    return dl, loss


@pytest.mark.parametrize("B,C", [(1, 2), (64, 555), (256, 1000), (7, 10000)])
def test_soft_cross_entropy_kernel_matches_torch(B, C):
    """Loss and autograd gradient of F.cross_entropy(z, t) (mean over rows, in float64) for four kinds of targets; one-hot
    targets give apla_cross_entropy's dlogits bitwise (and its loss bitwise at B = 1)."""
    _need_gpu()
    from apla_b200._lib import require_device
    require_device()
    g = torch.Generator().manual_seed(B * 7919 + C)
    z = (torch.randn(B, C, generator=g) * 3.0).float()
    y = torch.randint(0, C, (B,), generator=g)
    onehot = F.one_hot(y, C).float()
    kinds = {
        "mixup_smoothed": _soft_targets(y, C, seed=B + C),
        "unnormalised": torch.rand(B, C, generator=g) * (2.0 / C) * torch.rand(B, 1, generator=g) * 3.0,
        "zero_rows": torch.zeros(B, C),
        "onehot": onehot,
    }
    if B > 1:     # zero rows among ordinary ones
        kinds["zero_rows"] = kinds["mixup_smoothed"].clone()
        kinds["zero_rows"][::2] = 0.0
    zc = z.cuda()
    for kind, t in kinds.items():
        dl, loss = _ce_soft(zc, t.cuda(), 1.0 / B, 1.0 / B)
        torch.cuda.synchronize()
        zd = z.double().requires_grad_(True)
        ref = F.cross_entropy(zd, t.double())
        (gref,) = torch.autograd.grad(ref, zd)
        assert torch.isfinite(dl).all(), kind
        assert abs(float(loss) - float(ref)) <= 1e-5 * abs(float(ref)) + 1e-7, (kind, float(loss), float(ref))
        assert rel(dl, gref) <= 3e-5, (kind, rel(dl, gref))
        if kind == "zero_rows":
            zero = t.sum(1) == 0
            assert torch.equal(dl.cpu()[zero], torch.zeros_like(dl.cpu()[zero]))
    dl_s, loss_s = _ce_soft(zc, onehot.cuda(), 1.0 / B, 1.0 / B)
    dl_h, loss_h = _ce_hard(zc, y.cuda(), 1.0 / B, 1.0 / B)
    torch.cuda.synchronize()
    assert torch.equal(dl_s, dl_h)
    if B == 1:
        assert torch.equal(loss_s, loss_h)
    else:
        assert abs(float(loss_s) - float(loss_h)) <= 1e-6 * abs(float(loss_h))


@pytest.mark.parametrize("name,n", [("tiny_r16", 6), ("tiny_r16", 3), ("c1_vits16_r32", 8), ("c1_vits16_r32", 5)])
def test_soft_target_step_matches_oracle(name, n):
    """Probability targets through the engine (full and partial batches) against the oracle's F.cross_entropy with the
    same targets."""
    _need_gpu()
    factory, B, img = PARTIAL_CASES[name][:3]
    model = factory()
    O, cfg, sd = _oracle_of(model)
    images, labels = synthetic_batch(n, img, cfg.n_classes, seed=91)
    targets = _soft_targets(labels, cfg.n_classes, seed=92)
    ref = O.loss_and_grads(sd, cfg, images, targets)
    eng = _engine(model, B, img)
    out = eng.forward(images.cuda(), targets.cuda())
    assert out.shape == (n, cfg.n_classes)
    eng.backward()
    _check_against_oracle(eng, ref, n)


def test_step_from_host_loader_sequence_matches_eager_steps():
    """A loader-like sequence of pinned batches -- full and partial, hard labels and mixup targets -- through
    step_from_host (two device slots, graphs captured on second sightings, at most 4 kept) against eager step calls on a
    second engine: same losses, same final parameters."""
    _need_gpu()
    B, C = 6, 10
    sizes = [6, 6, 4] * 3 + [6, 4] * 3
    batches = []
    for k, size in enumerate(sizes):
        images, labels = synthetic_batch(size, 56, C, seed=900 + k)
        if k >= 9:
            labels = _soft_targets(labels, C, seed=950 + k)
        batches.append((images.pin_memory(), labels.pin_memory()))
    host = _engine(_small(128, 2, 2, 16), B, 56)
    eager = _engine(_small(128, 2, 2, 16), B, 56, use_graph=False)
    got, want = [], []
    for images, labels in batches:
        got.append(host.step_from_host(images, labels, lag=False))
        want.append(float(eager.step(images.cuda(), labels.cuda())))
        assert len(host._graphs) <= 4
    torch.cuda.synchronize()
    assert "tgt" in host._e2e
    for k, (a, b) in enumerate(zip(got, want)):
        assert abs(a - b) <= 1e-4 * abs(b), (k, a, b)
    assert rel(host.params, eager.params) < 1e-5
    assert len(host._graphs) == 4


def test_bad_batches_are_refused():
    _need_gpu()
    B, C = 4, 10
    eng = _engine(_small(128, 2, 2, 16), B, 56)
    images, labels = synthetic_batch(B + 1, 56, C, seed=3)
    images, labels = images.cuda(), labels.cuda()
    targets = _soft_targets(labels.cpu(), C, seed=4).cuda()
    bad = [
        (images[:0], labels[:0], "1 to batch_size"),                              # n = 0
        (images, labels, "1 to batch_size"),                                       # n > B
        (images[:3].half(), labels[:3], "fp32"),                                   # image dtype
        (images[:3], labels[:3].int(), "int64"),                                   # label dtype
        (images[:3], targets[:3].double(), "int64"),                               # target dtype
        (images[:3], labels[:2], r"shape \[3\]"),                                 # label rows != image rows
        (images[:3], targets[:4], r"shape \[3, 10\]"),                            # target rows != image rows
        (images[:3], targets[:3, :9], r"shape \[3, 10\]"),                        # target classes != C
    ]
    for im, lab, msg in bad:
        for call in (eng.forward, eng.step):
            with pytest.raises(RuntimeError, match=msg):
                call(im, lab)
        with pytest.raises(RuntimeError, match=msg):
            eng.step_from_host(im.cpu(), lab.cpu(), lag=False)
    # a refused batch leaves the engine usable
    eng.step(images[:3], labels[:3])
    torch.cuda.synchronize()
    assert torch.isfinite(eng.params).all()

"""Stochastic depth (drop path) on the B200: the row-scaled residual GEMM epilogue and LayerNorm backward against their
unscaled forms and torch, and engines over models built with drop_path_rate > 0 against an fp32 reference that applies
the engine's own masks (`last_drop_path_scales`): x_mid = x_in + s[l,0,b] * ls1(attn), x_out = x_mid + s[l,1,b] * ls2(mlp).
The reference is built from the oracle's `embed` / `attention_module`, F.layer_norm / F.linear / F.gelu and its
`clip_grad_norm_` / `adamw_step`.  Bars as in test_engine_gpu.py: logits / loss relative error <= 1e-2, gradient cosine
>= 0.999 and relative error <= 1e-2."""
import pytest
import torch
import torch.nn.functional as F

from helpers import build_case, cosine, rel, synthetic_batch
from test_engine_batches_gpu import PARTIAL_CASES, _check_against_oracle, _oracle_of, _poison_stale_rows, _small

pytestmark = pytest.mark.gpu


def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from apla_b200._lib import require_device
    require_device()


def _engine(model, batch, img, **kw):
    _need_gpu()
    from apla_b200.engine import FineTuneEngine
    return FineTuneEngine(model, batch_size=batch, img_size=img, **kw)


def _with_rate(model, rate):
    """The model with the reference's per-block DropPath(linspace(0, rate, depth)[l]); no weight changes."""
    from apla_b200.hostvit import DropPath
    blocks = model.backbone.blocks
    for blk, p in zip(blocks, torch.linspace(0, rate, len(blocks)).tolist()):
        blk.drop_path = DropPath(p) if p > 0 else torch.nn.Identity()
    return model


def _forward_logits(O, sd, cfg, images, scales):
    """forward_logits with every branch output of image b scaled by scales[l, branch, b]."""
    x = O.embed(sd, cfg, images)
    D = x.shape[-1]
    for l in range(cfg.depth):
        b = f"backbone.blocks.{l}."
        s1, s2 = scales[l, 0].view(-1, 1, 1), scales[l, 1].view(-1, 1, 1)
        y = O.attention_module(sd, b + "attn.", F.layer_norm(x, (D,), sd[b + "norm1.weight"], sd[b + "norm1.bias"],
                                                             cfg.ln_eps), cfg.num_heads)
        if b + "ls1.gamma" in sd:
            y = y * sd[b + "ls1.gamma"]
        x = x + s1 * y
        h = F.layer_norm(x, (D,), sd[b + "norm2.weight"], sd[b + "norm2.bias"], cfg.ln_eps)
        h = F.linear(F.gelu(F.linear(h, sd[b + "mlp.fc1.weight"], sd[b + "mlp.fc1.bias"])), sd[b + "mlp.fc2.weight"],
                     sd[b + "mlp.fc2.bias"])
        if b + "ls2.gamma" in sd:
            h = h * sd[b + "ls2.gamma"]
        x = x + s2 * h
    x = F.layer_norm(x, (D,), sd["backbone.norm.weight"], sd["backbone.norm.bias"], cfg.ln_eps)
    return F.linear(x[:, 0], sd["fc.weight"], sd["fc.bias"])


def _loss_and_grads(O, sd, cfg, images, labels, scales):
    keys = O.trainable_keys(cfg, sd)
    leaves = {k: sd[k].detach().clone().requires_grad_(True) for k in keys}
    logits = _forward_logits(O, dict(sd, **leaves), cfg, images, scales)
    loss = F.cross_entropy(logits, labels)
    gs = torch.autograd.grad(loss, [leaves[k] for k in keys])
    return O.StepResult(logits.detach(), loss.detach(), dict(zip(keys, gs)))


def _check_step(O, sd, cfg, st, eng, ref, p0):
    """clip + AdamW on the reference's gradients against the engine's optimiser step: parameters and the update."""
    grads = {k: g.clone() for k, g in ref.grads.items()}
    O.clip_grad_norm_(grads, 1.0)
    O.adamw_step(sd, grads, st)
    eng.optim_step()
    torch.cuda.synchronize()
    names = eng.trainable_names()
    params = eng.named_params()
    p = torch.cat([params[k].cpu().flatten() for k in names])
    p_ref = torch.cat([sd[k].flatten() for k in names])
    assert rel(p, p_ref) <= 1e-2, rel(p, p_ref)
    upd = p - torch.cat([p0[k].flatten() for k in names])
    upd_ref = p_ref - torch.cat([p0[k].flatten() for k in names])
    assert torch.isfinite(upd).all() and cosine(upd, upd_ref) >= 0.95, cosine(upd, upd_ref)


# ---- the kernels --------------------------------------------------------------------------------------------------
def _scales(n, keep, g):
    return ((torch.rand(n, generator=g) < keep).float() / keep).cuda()


def _filled(rows, cols, canary=64):
    buf = torch.full((rows * cols + canary,), float("nan"), device="cuda")
    buf[rows * cols:] = 12345.0
    return buf


@pytest.mark.parametrize("K", [768, 3072])
@pytest.mark.parametrize("cls_rows", [False, True])
def test_scaled_residual_gemm(K, cls_rows):
    """C2 shapes (N = 257, D = 768; K = 768 the projection, 3072 fc2), over every token row (rows_per_scale = N) or the
    CLS rows only (rows_per_scale = 1, row stride N*D): all-ones scales give the unscaled entry's bits, random {0, 1/keep}
    scales match torch; the output is NaN-prefilled, rows the call does not own stay NaN and the canary tail is intact."""
    _need_gpu()
    from apla_b200._lib import LIB, ptr, stream
    B, N, D = 4, 257, 768
    g = torch.Generator().manual_seed(K + cls_rows)
    A = (torch.randn(B * N, K, generator=g) * 0.5).to(torch.bfloat16).cuda()
    W = (torch.randn(D, K, generator=g) * 0.02).to(torch.bfloat16).cuda()
    bias, gamma = torch.randn(D, generator=g).cuda(), (1 + 0.1 * torch.randn(D, generator=g)).cuda()
    resid = torch.randn(B * N, D, generator=g).cuda()
    M, ld_a, ld, rps = (B, N * K, N * D, 1) if cls_rows else (B * N, K, D, N)
    rows = torch.arange(B, device="cuda") * N if cls_rows else torch.arange(B * N, device="cuda")

    def scaled(s):
        out = _filled(B * N, D)
        LIB.call("apla_gemm_bias_ls_residual_scaled_fwd", ptr(A), ld_a, ptr(W), K, ptr(bias), ptr(gamma), ptr(resid),
                 ptr(s), rps, ptr(out), ld, M, D, K, stream())
        torch.cuda.synchronize()
        assert torch.equal(out[B * N * D:], torch.full_like(out[B * N * D:], 12345.0))
        out = out[:B * N * D].view(B * N, D)
        others = torch.ones(B * N, dtype=torch.bool, device="cuda")
        others[rows] = False
        assert torch.isnan(out[others]).all()
        return out[rows]

    plain = _filled(B * N, D)
    LIB.call("apla_gemm_bias_ls_residual_fwd", ptr(A), ld_a, ptr(W), K, ptr(bias), ptr(gamma), ptr(resid), ptr(plain),
             ld, M, D, K, stream())
    torch.cuda.synchronize()
    assert torch.equal(scaled(torch.ones(B, device="cuda")), plain[:B * N * D].view(B * N, D)[rows])
    for keep in (0.9, 0.5):
        s = _scales(B, keep, g)
        got = scaled(s)
        s_row = s.repeat_interleave(1 if cls_rows else N)
        a_rows = A[rows].float()
        want = resid[rows] + s_row[:, None] * gamma * (a_rows @ W.float().t() + bias)
        err = float((got - want).abs().max())
        assert err <= 1e-3 * float(want.abs().max()), (keep, err)
        dropped = s_row == 0
        assert torch.equal(got[dropped], resid[rows][dropped])       # a dropped image keeps its residual exactly


@pytest.mark.parametrize("D", [384, 768, 1024])
@pytest.mark.parametrize("cls_rows", [False, True])
def test_scaled_layernorm_backward(D, cls_rows):
    """The row-scaled LayerNorm backward with the residual add, LayerScale and APLA gather: all-ones scales give the
    unscaled entry's bits; random {0, 1/keep} scales leave dx as it was and give dxb = bf16(s * gamma * dx) and
    sub = its gathered columns (NaN-prefilled outputs, canary tails)."""
    _need_gpu()
    from apla_b200._lib import LIB, ptr, stream
    B, N, r, r_pad = 3, 257, 24, 64
    g = torch.Generator().manual_seed(D + cls_rows)
    T = B * N
    x = torch.randn(T, D, generator=g).cuda()
    dy = torch.randn(T, D, generator=g).to(torch.bfloat16).cuda()
    dres = torch.randn(T, D, generator=g).cuda()
    w, gamma = (1 + 0.1 * torch.randn(D, generator=g)).cuda(), (1 + 0.1 * torch.randn(D, generator=g)).cuda()
    idx = torch.randperm(D, generator=g)[:r].to(torch.int32).cuda()
    rows, ld, ld_sub, rps = (B, N * D, N * r_pad, 1) if cls_rows else (T, D, r_pad, N)
    sel = torch.arange(B, device="cuda") * N if cls_rows else torch.arange(T, device="cuda")

    def run(s):
        dx, dxb = _filled(T, D), torch.full((T * D + 64,), float("nan"), device="cuda").to(torch.bfloat16)
        sub = torch.full((T * r_pad + 64,), float("nan"), device="cuda").to(torch.bfloat16)
        dxb[T * D:] = 7.0
        sub[T * r_pad:] = 7.0
        args = [ptr(dy), ld, ptr(x), ld, ptr(w), ptr(dres), ld, ptr(dx), ld, ptr(dxb), ld, ptr(gamma), ptr(sub), ld_sub,
                ptr(idx), r, r_pad]
        if s is None:
            LIB.call("apla_layernorm_bwd", *args, rows, D, 1e-6, stream())
        else:
            LIB.call("apla_layernorm_bwd_scaled", *args, ptr(s), rps, rows, D, 1e-6, stream())
        torch.cuda.synchronize()
        assert torch.equal(dx[T * D:], torch.full((64,), 12345.0, device="cuda"))
        assert (dxb[T * D:] == 7.0).all() and (sub[T * r_pad:] == 7.0).all()
        return (dx[:T * D].view(T, D)[sel], dxb[:T * D].view(T, D)[sel], sub[:T * r_pad].view(T, r_pad)[sel])

    plain = run(None)
    ones = run(torch.ones(B, device="cuda"))
    assert all(torch.equal(a, b) for a, b in zip(ones, plain))
    s = _scales(B, 0.5, g)
    dx, dxb, sub = run(s)
    s_row = s.repeat_interleave(1 if cls_rows else N)[:, None]
    assert torch.equal(dx, plain[0])
    want = (plain[0] * gamma) * s_row
    # (bf16 of the same fp32 products: at most one rounding step apart)
    torch.testing.assert_close(dxb.float(), want.to(torch.bfloat16).float(), rtol=2 ** -7, atol=0)
    torch.testing.assert_close(sub[:, :r].float(), want[:, idx.long()].to(torch.bfloat16).float(), rtol=2 ** -7, atol=0)
    assert torch.equal(dxb[s_row.view(-1) == 0], torch.zeros_like(dxb[s_row.view(-1) == 0]))
    assert (sub[:, r:] == 0).all()


# ---- the engine ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rate", [0.1, 0.5])
@pytest.mark.parametrize("name", list(PARTIAL_CASES))
def test_drop_path_step_matches_reference(name, rate, monkeypatch):
    """Every PARTIAL_CASES model (tiny, the side-stream weight gradient, the dense-rows path, C1, C2) built with drop path,
    at n = batch_size and a partial n (stale rows NaN-poisoned first), in every cls_only_last_block mode of the case:
    logits, loss and gradients against the reference with the engine's masks, then clip + AdamW against the reference's."""
    _need_gpu()
    factory, B, img, sizes, modes, side = PARTIAL_CASES[name]
    monkeypatch.setenv("APLA_SIDE_WGRAD", side)
    model = _with_rate(factory(), rate)
    O, cfg, sd0 = _oracle_of(model)
    images, labels = synthetic_batch(B, img, cfg.n_classes, seed=71)
    full_images, full_labels = synthetic_batch(B, img, cfg.n_classes, seed=72)
    for mode in modes:
        eng = _engine(model, B, img, cls_only_last_block=mode)
        sd, st = {k: v.clone() for k, v in sd0.items()}, O.AdamWState()
        for n in (B, sizes[-1]):
            eng.forward(full_images.cuda(), full_labels.cuda())
            eng.backward()
            torch.cuda.synchronize()
            if n < B:
                _poison_stale_rows(eng, n)
            eng.forward(images[:n].cuda(), labels[:n].cuda())
            eng.backward()
            scales = eng.last_drop_path_scales
            assert scales.shape == (cfg.depth, 2, n) and scales.dtype == torch.float32
            ref = _loss_and_grads(O, sd, cfg, images[:n], labels[:n], scales)
            _check_against_oracle(eng, ref, n)
            p0 = {k: v.cpu().clone() for k, v in eng.named_params().items()}
            _check_step(O, sd, cfg, st, eng, ref, p0)
        del eng


def _forced(eng, scales):
    """Make the engine's next draws return `scales` [L, 2, B] (cut to the step's n)."""
    eng._draw_drop_path = lambda n: scales[:, :, :n].clone()


def test_dropped_branches_are_exact():
    """A block whose branches drop every image gets exactly zero proj_weight1 / proj_bias1 gradients; dropping only a
    block's MLP branch leaves x_out == x_mid bit for bit and x_mid as it was with every branch kept."""
    B, img, L = 6, 56, 3
    model = _with_rate(_small(128, L, 2, 16), 0.3)
    eng = _engine(model, B, img)
    images, labels = synthetic_batch(B, img, 10, seed=81)
    images, labels = images.cuda(), labels.cuda()
    ones = torch.ones(L, 2, B)
    _forced(eng, ones)
    eng.forward(images, labels)
    torch.cuda.synchronize()
    xs_keep = eng.xs.clone()
    for l in range(1, L):
        s = ones.clone()
        s[l] = 0.0
        _forced(eng, s)
        eng.forward(images, labels)
        eng.backward()
        torch.cuda.synchronize()
        g = eng.named_grads()
        for key in (f"backbone.blocks.{l}.attn.proj_weight1", f"backbone.blocks.{l}.attn.proj_bias1"):
            assert torch.count_nonzero(g[key]) == 0, key
        assert torch.count_nonzero(g["backbone.blocks.0.attn.proj_weight1"]) > 0
        s = ones.clone()
        s[l, 1] = 0.0
        _forced(eng, s)
        eng.forward(images, labels)
        torch.cuda.synchronize()
        # the last block's per-token tail runs on the CLS rows only (cls_only_last_block = 2): the rest are not written
        own = (lambda t: t.view(B, -1, t.shape[-1])[:, 0]) if l == L - 1 else (lambda t: t)
        assert torch.equal(own(eng.xs[2 * l + 2]), own(eng.xs[2 * l + 1])), l
        assert torch.equal(own(eng.xs[2 * l + 1]), own(xs_keep[2 * l + 1])), l


def test_repeated_steps_eager_and_graph():
    """Four whole steps of a drop-path engine eagerly, again on a second eager engine, and from graphs (eager, captured,
    replayed): the same masks every step (one host generator per engine, seeded alike), new masks every step, and the
    graph engine's parameters within the eager engines' run-to-run spread."""
    B, img = 6, 56
    model = _with_rate(_small(128, 3, 2, 16), 0.5)
    engines = [_engine(model, B, img, use_graph=False), _engine(model, B, img, use_graph=False),
               _engine(model, B, img, use_graph=True)]
    buf = [(torch.empty(B, 3, img, img, device="cuda"), torch.empty(B, dtype=torch.int64, device="cuda"))
           for _ in engines]
    prev = None
    for k in range(4):
        images, labels = synthetic_batch(B, img, 10, seed=90 + k)
        drawn = []
        for eng, (bi, bl) in zip(engines, buf):
            bi.copy_(images)
            bl.copy_(labels)
            eng.step(bi, bl)
            drawn.append(eng.last_drop_path_scales.clone())
        torch.cuda.synchronize()
        assert all(torch.equal(d, drawn[0]) for d in drawn), k
        assert prev is None or not torch.equal(drawn[0], prev), k
        prev = drawn[0]
    assert len(engines[2]._graphs) == 1
    spread = rel(engines[1].params, engines[0].params)
    assert rel(engines[2].params, engines[0].params) <= max(4 * spread, 1e-6), (rel(engines[2].params,
                                                                                    engines[0].params), spread)
    assert abs(float(engines[2].loss) - float(engines[0].loss)) <= 1e-4 * abs(float(engines[0].loss))


def test_rate_zero_is_the_plain_engine():
    """A model whose rates are all 0 sets no drop-path buffer and draws nothing; a drop-path engine whose masks keep every
    image issues the same number of launches and gives bitwise-equal logits (a scale of 1 gives the unscaled bits); the
    loss, an fp32 atomic sum over the rows, agrees to its rounding."""
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
        return LIB.load().apla_launch_count() - before, eng.logits.clone(), eng.loss.clone()

    plain = _engine(model, B, 224)
    assert plain.buffers.get(("drop_path", -1)) is None and plain._dp_dev is None
    a = run(plain)
    assert plain.last_drop_path_scales is None
    dp = _engine(_with_rate(model, 0.1), B, 224)
    _forced(dp, torch.ones(12, 2, B))
    b = run(dp)
    assert a[0] == b[0]
    assert torch.equal(a[1], b[1])
    assert abs(float(a[2]) - float(b[2])) <= 1e-6 * abs(float(a[2]))


def test_predict_ignores_drop_path():
    """predict on a drop-path engine (after training forwards that dropped images) is bitwise equal to predict on a
    rate-0 engine with the same weights."""
    B, img = 6, 56
    base = _small(128, 3, 2, 16)
    plain = _engine(base, B, img)
    dp = _engine(_with_rate(_small(128, 3, 2, 16), 0.5), B, img)
    images, labels = synthetic_batch(B, img, 10, seed=5)
    images, labels = images.cuda(), labels.cuda()
    dp.forward(images, labels)
    assert (dp.last_drop_path_scales == 0).any()
    test = synthetic_batch(9, img, 10, seed=6)[0].cuda()
    assert torch.equal(dp.predict(test), plain.predict(test))
    assert torch.equal(dp.cls_attention(test), plain.cls_attention(test))


def test_refused_model_allocates_nothing():
    _need_gpu()
    model = _small(128, 2, 2, 16)
    model.backbone.blocks[1].attn.proj_drop.p = 0.1
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated()
    with pytest.raises(ValueError, match="cannot honour dropout"):
        _engine(model, 4, 56)
    assert torch.cuda.memory_allocated() == before

"""Integrated gradients through the sNet towers with block 1 factored out of the path integral (csrc/ig.cu,
transmf_ad_b200.interpret.integrated_gradients; DESIGN section 3.10).

Op level: tmf_ig_expand / tmf_ig_combine against float64 on their own inputs, and the combine's independence of the chunking.
Model level: against a plain IG built here from the saliency path (the alpha_k x volumes batched through the model with
autograd to the volumes), completeness on model_ad, every model with sNet towers, and the side-effect rules.  The factored
and plain paths differ by bf16 rounding: the factored one pools the bias-free folded conv1.0 output u' once, the plain one
the biased pre-BatchNorm output at every alpha, so near-tied max-pool winners can differ.  Measured values print with ``-s``.
"""
import copy

import pytest
import torch
import torch.nn.functional as F

from tests import helpers as H
from transmf_ad_b200 import _lib as L
from transmf_ad_b200 import functional as TF
from transmf_ad_b200.interpret import ig_path, integrated_gradients
from transmf_ad_b200.models import mymodel as M

pytestmark = pytest.mark.gpu
DEV = "cuda"
BF16_ULP = 2.0 ** -8                 # relative spacing of bf16 (8 significand bits)
# bounds from the first measurement on a B200, with headroom (measured worst case in brackets)
# factored vs plain IG, worst tower of model_single / model_cnn_ad / model_ad_h4, relative L2 of the voxel maps (0.261), of
# their 4x4x4 block means (0.177) and of the per-sample totals (0.034).  The plain path moves as much on its own when x is
# scaled by 1 + 2^-10 (0.191, 0.144, 0.030): the voxel maps are dominated by max-pool winners that tie at bf16 resolution
PLAIN_REL = {"voxel": 0.35, "coarse": 0.25, "totals": 0.06}
PLAIN_SENS = 2.0                     # ... and at most this times the plain path's own move, + 0.01 (1.41)
DELTA_FRAC = 0.05                    # model_ad_h4, 64 steps: sum |delta| / sum |f(x) - f(0)| (1.9e-2)
CHUNK_REL = 1e-5                     # internal_batch_size = B vs B * n_steps, relative L2 (bitwise equal)


def _expand_inputs(B, dims, C, n, seed):
    g = torch.Generator().manual_seed(seed)
    umax = (torch.randn((B,) + dims + (C,), generator=g) * 2).bfloat16().to(DEV)
    bias = (torch.randn(C, generator=g) * 0.5).to(DEV)
    alpha = (torch.rand(n, generator=g) * 0.99 + 0.01).to(DEV)
    w = (torch.rand(n, generator=g) + 0.1).to(DEV)
    return umax, bias, alpha, w


def _z64(umax, bias, alpha):
    return alpha.double().view(-1, 1, 1, 1, 1, 1) * umax.double().unsqueeze(0) + bias.double()


@pytest.mark.parametrize("slope", [0.0, 0.01])
@pytest.mark.parametrize("dims,C", [((4, 5, 6), 32), ((3, 1, 7), 8)])
def test_expand_against_float64(slope, dims, C):
    umax, bias, alpha, _ = _expand_inputs(2, dims, C, 3, seed=C + len(dims))
    a16, a32 = TF.ig_expand([umax, umax], [bias, bias], alpha, slope)
    z = _z64(umax, bias, alpha)
    ref = torch.where(z > 0, z, z * slope).reshape(a32[0].shape)
    assert torch.equal(a16[0], a32[0].bfloat16())                    # the fp32 twin rounds to the bf16 operand
    assert torch.allclose(a32[0].double(), ref, rtol=2 ** -22, atol=0)  # fmaf, then the slope product: fp32 roundings
    assert ((a16[0].double() - ref).abs() <= BF16_ULP * ref.abs() + 1e-30).all()
    assert torch.equal(a16[0], a16[1]) and torch.equal(a32[0], a32[1])


@pytest.mark.parametrize("slope", [0.0, 0.01])
@pytest.mark.parametrize("dims,C", [((4, 5, 6), 32), ((3, 1, 7), 16)])
def test_combine_against_float64(slope, dims, C):
    B, n = 2, 5
    umax, bias, alpha, w = _expand_inputs(B, dims, C, n, seed=7 + C)
    g = torch.Generator().manual_seed(11)
    grads = torch.randn((n * B,) + dims + (C,), generator=g).to(DEV)
    G0 = torch.randn((B,) + dims + (C,), generator=g).to(DEV)
    G = G0.clone()
    TF.ig_combine([grads], [umax], [bias], alpha, w, [G], slope)
    z = _z64(umax, bias, alpha)
    d = torch.where(z > 0, torch.ones_like(z), torch.full_like(z, slope))
    terms = w.double().view(-1, 1, 1, 1, 1, 1) * grads.double().view((n, B) + dims + (C,)) * d
    ref = G0.double() + terms.sum(0)
    scale = G0.double().abs() + terms.abs().sum(0)
    assert ((G.double() - ref).abs() <= 4 * (n + 1) * 2 ** -24 * scale + 1e-30).all()


def test_combine_is_bitwise_independent_of_the_chunking():
    B, n, dims, C = 2, 9, (3, 5, 7), 32
    umax, bias, alpha, w = _expand_inputs(B, dims, C, n, seed=5)
    grads = torch.randn((n * B,) + dims + (C,), device=DEV)
    out = []
    for cuts in ([0, n], [0, 3, 6, n], list(range(n + 1))):
        G = torch.zeros((B,) + dims + (C,), device=DEV)
        for k0, k1 in zip(cuts[:-1], cuts[1:]):
            TF.ig_combine([grads[k0 * B:k1 * B]], [umax], [bias], alpha[k0:k1], w[k0:k1], [G], 0.01)
        out.append(G)
    assert torch.equal(out[0], out[1]) and torch.equal(out[0], out[2])


# ---------------------------------------------------------------------------------------------------------------
# model level
# ---------------------------------------------------------------------------------------------------------------
def _model(gold):
    model = getattr(M, gold["kind"])(**gold["kwargs"])
    model.load_state_dict(H.case_state(gold), strict=True)
    model = model.to(DEV).eval()
    H.set_head_dropout(model, 0.0)
    return model


def _inputs(gold):
    mri, pet, label = H.case_inputs(gold)
    xs = (mri,) if gold["kind"] == "model_single" else (mri, pet)
    return [x.to(DEV) for x in xs], label.to(DEV)


def _towers(model):
    return [m for m in model.modules() if isinstance(m, M.sNet)]


def _logits(outs):
    return outs[0] if isinstance(outs, (tuple, list)) else outs


def _plain_ig(model, xs, target, n, method, chunk):
    """IG through the saliency path: alpha_k x batched through the model, autograd to the volumes, weighted sum, times x."""
    alpha, w = ig_path(n, method)
    B = xs[0].shape[0]
    acc = [torch.zeros_like(x) for x in xs]
    flags = [(p, p.requires_grad) for p in model.parameters()]
    try:
        for p, _ in flags:
            p.requires_grad_(False)
        for k0 in range(0, n, chunk):
            m = min(chunk, n - k0)
            a = torch.tensor(alpha[k0:k0 + m], dtype=torch.float32, device=DEV).view(-1, 1, 1, 1, 1, 1)
            wk = torch.tensor(w[k0:k0 + m], dtype=torch.float32, device=DEV).view(-1, 1, 1, 1, 1, 1)
            X = [(a * x.unsqueeze(0)).reshape((m * B,) + tuple(x.shape[1:])).requires_grad_(True) for x in xs]
            obj = _logits(model(*X)).gather(1, target.repeat(m).view(-1, 1)).sum()
            for t, g in enumerate(torch.autograd.grad(obj, X)):
                acc[t] += (wk * g.view((m,) + tuple(xs[t].shape))).sum(0)
    finally:
        for p, f in flags:
            p.requires_grad_(f)
    return [x * a for x, a in zip(xs, acc)]


def _rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30))


def _coarse(m):
    """4x4x4 block means: where a winner sits inside its 2x2x2 max-pool window no longer matters."""
    return F.avg_pool3d(m, 4, ceil_mode=True)


@pytest.mark.parametrize("name", ["model_single", "model_cnn_ad", "model_ad_h4"])
def test_factored_ig_against_the_plain_path(name):
    gold = H.load_golden(name)
    model = _model(gold)
    xs, tgt = _inputs(gold)
    B = xs[0].shape[0]
    res = integrated_gradients(model, xs, tgt, n_steps=16, internal_batch_size=8 * B)
    ref = _plain_ig(model, xs, tgt, 16, "gausslegendre", 8)
    # the plain path's own sensitivity: x scaled by 1 + 2^-10 (an exact scaling of the maps in real arithmetic) moves
    # max-pool winners that tie at bf16 resolution, as the factored path's different rounding does
    s = 1 + 2 ** -10
    ref2 = [m / s for m in _plain_ig(model, [x * s for x in xs], tgt, 16, "gausslegendre", 8)]
    for t, (got, want, moved) in enumerate(zip(res.maps, ref, ref2)):
        assert got.shape == want.shape and got.dtype == torch.float32
        r = {"voxel": (_rel(got, want), _rel(moved, want)),
             "coarse": (_rel(_coarse(got), _coarse(want)), _rel(_coarse(moved), _coarse(want))),
             "totals": (_rel(got.sum(dim=(1, 2, 3, 4)), want.sum(dim=(1, 2, 3, 4))),
                        _rel(moved.sum(dim=(1, 2, 3, 4)), want.sum(dim=(1, 2, 3, 4))))}
        print(f"[ig] {name} tower {t}: factored vs plain relative L2 (plain at x vs at (1 + 2^-10) x): " +
              ", ".join(f"{k} {a:.2e} ({b:.2e})" for k, (a, b) in r.items()))
        for k, (a, b) in r.items():
            assert a < PLAIN_REL[k] and a < PLAIN_SENS * b + 0.01, (t, k, a, b)


def test_completeness_on_model_ad():
    gold = H.load_golden("model_ad_h4")
    model = _model(gold)
    xs, tgt = _inputs(gold)
    with torch.no_grad():
        fx = _logits(model(*xs)).gather(1, tgt.view(-1, 1)).view(-1)
        f0 = _logits(model(*[torch.zeros_like(x) for x in xs])).gather(1, tgt.view(-1, 1)).view(-1)
    span = float((fx - f0).abs().sum())
    for n in (8, 16, 32, 64):
        res = integrated_gradients(model, xs, tgt, n_steps=n)
        total = sum(m.double().sum(dim=(1, 2, 3, 4)) for m in res.maps)
        assert torch.allclose(res.delta.double(), total - (fx - f0).double(), rtol=1e-4, atol=1e-4 * span)
        frac = float(res.delta.abs().sum()) / span
        print(f"[ig completeness] {n} steps: sum |delta| / sum |f(x) - f(0)| = {frac:.3e} "
              f"(delta {[round(float(d), 5) for d in res.delta]})")
    assert frac <= DELTA_FRAC


@pytest.mark.parametrize("name", ["model_single", "model_cnn", "model_cnn_ad", "model_ad_h4", "model_transformer",
                                  "model_transformer_res"])
def test_every_model_with_towers(name):
    gold = H.load_golden(name)
    model = _model(gold)
    xs, tgt = _inputs(gold)
    res = integrated_gradients(model, xs, tgt, n_steps=4, method="riemann_middle", internal_batch_size=3)
    assert len(res.maps) == len(_towers(model)) == len(xs)
    for m, x in zip(res.maps, xs):
        assert m.shape == x.shape and m.dtype == torch.float32 and bool(torch.isfinite(m).all())
        assert float(m.abs().sum()) > 0
    assert res.delta.shape == (xs[0].shape[0],) and bool(torch.isfinite(res.delta).all())


def test_determinism_chunking_and_side_effects(monkeypatch):
    gold = H.load_golden("model_ad_h4")
    model = _model(gold)
    model.fc_cls[0].weight.requires_grad_(False)
    xs, tgt = _inputs(gold)
    B, n = xs[0].shape[0], 6
    flags = {k: p.requires_grad for k, p in model.named_parameters()}
    before = {k: v.clone() for k, v in model.state_dict().items()}
    called = []
    real = L.call

    def spy(name, *args, **kw):
        called.append(kw.get("tag") or name)
        return real(name, *args, **kw)

    monkeypatch.setattr(L, "call", spy)
    a = integrated_gradients(model, xs, tgt, n_steps=n, internal_batch_size=B)
    monkeypatch.setattr(L, "call", real)
    b = integrated_gradients(model, xs, tgt, n_steps=n, internal_batch_size=B)
    c = integrated_gradients(model, xs, tgt, n_steps=n, internal_batch_size=B * n)
    for x, y in zip(a.maps + [a.delta], b.maps + [b.delta]):
        assert torch.equal(x, y)
    for x, y in zip(a.maps, c.maps):
        r = _rel(y, x)
        print(f"[ig] internal_batch_size B vs B*n: relative L2 {r:.2e} (bitwise equal: {torch.equal(x, y)})")
        assert r <= CHUNK_REL
    assert all(p.grad is None for p in model.parameters())
    assert flags == {k: p.requires_grad for k, p in model.named_parameters()}
    assert not any(m.training for m in model.modules())
    for k, v in model.state_dict().items():
        assert torch.equal(v, before[k]), k
    assert all(t._ig_src is None for t in _towers(model))
    bad = [s for s in called if "wgrad" in s or s.startswith("tmf_conv1_bwd")]
    assert not bad, bad
    assert called.count("tmf_conv1_dgrad_fused") == 1                # both towers, once for the whole path
    assert called.count("tmf_ig_expand") == n and called.count("tmf_ig_combine") == n


def test_an_error_mid_call_leaves_the_model_usable(monkeypatch):
    gold = H.load_golden("model_cnn_ad")
    model = _model(gold)
    xs, tgt = _inputs(gold)
    B = xs[0].shape[0]
    ref = integrated_gradients(model, xs, tgt, n_steps=4, internal_batch_size=B)
    with torch.no_grad():
        out0 = _logits(model(*xs)).clone()
    real, seen = TF.ig_combine, []

    def failing(*args, **kw):
        seen.append(1)
        if len(seen) == 2:
            raise RuntimeError("injected failure")
        return real(*args, **kw)

    monkeypatch.setattr(TF, "ig_combine", failing)
    with pytest.raises(RuntimeError, match="injected"):
        integrated_gradients(model, xs, tgt, n_steps=4, internal_batch_size=B)
    monkeypatch.setattr(TF, "ig_combine", real)
    assert all(t._ig_src is None for t in _towers(model))
    assert all(p.requires_grad for p in model.parameters())
    with torch.no_grad():
        assert torch.equal(_logits(model(*xs)), out0)
    again = integrated_gradients(model, xs, tgt, n_steps=4, internal_batch_size=B)
    for x, y in zip(ref.maps, again.maps):
        assert torch.equal(x, y)


def test_an_observing_conv3_hook_fires_and_leaves_maps_unchanged():
    gold = H.load_golden("model_ad_h4")
    model = _model(gold)
    xs, tgt = _inputs(gold)
    B = xs[0].shape[0]
    a = integrated_gradients(model, xs, tgt, n_steps=4, internal_batch_size=2 * B)
    seen = []
    hs = [t.conv3.register_forward_hook(lambda m, i, o: seen.append((i[0].shape[0], o.shape[0]))) for t in _towers(model)]
    try:
        b = integrated_gradients(model, xs, tgt, n_steps=4, internal_batch_size=2 * B)
    finally:
        for h in hs:
            h.remove()
    assert len(seen) == 2 * 2 + 2 * 2                 # two chunks and the eval forwards on x and on zeros, two towers each
    assert (2 * B, 2 * B) in seen
    for x, y in zip(a.maps, b.maps):
        r = _rel(y, x)
        print(f"[ig] conv3 hook: relative L2 {r:.2e} (bitwise equal: {torch.equal(x, y)})")
        assert r <= CHUNK_REL


def test_ig_refuses_training_mode_on_the_gpu():
    gold = H.load_golden("model_cnn_ad")
    model = _model(gold).train()
    xs, tgt = _inputs(gold)
    with pytest.raises(ValueError, match="eval"):
        integrated_gradients(model, xs, tgt)
    assert all(t._ig_src is None for t in _towers(model))
    assert copy.deepcopy(model).training

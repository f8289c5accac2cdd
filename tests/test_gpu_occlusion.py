"""Occlusion sensitivity with incremental recomputation (csrc/occlusion.cu, transmf_ad_b200.interpret.occlusion; DESIGN
section 3.11).

Op level: tmf_occ_input and tmf_occ_compose are copies, so they match a torch-indexing restatement bit for bit (outputs inside
NaN guard bands); tmf_occ_map against float64.  Model level: the scores against brute force -- the model's own forward on the
materialised occluded volumes, same windows --, null windows (an all-zero region under baseline 0, where brute force's own
value is the floor), determinism, and the side-effect rules.  The incremental path runs the crops through other conv plans
than the full volumes, so its bf16 roundings differ from brute force's; measured values print with ``-s``.
"""
import copy

import numpy as np
import pytest
import torch

from tests import helpers as H
from transmf_ad_b200 import _lib as L
from transmf_ad_b200 import functional as TF
from transmf_ad_b200.interpret import occlusion
from transmf_ad_b200.models import mymodel as M

pytestmark = pytest.mark.gpu
DEV = "cuda"
# bounds from the first measurement on a B200, with headroom (measured worst case in brackets): max |incremental - brute
# force| over the subjects' max |f(x)|, worst tower of the four cases (5.5e-05, model_ad at 91 x 109 x 91)
SCORE_ERR = 5e-4
# null windows: max |score| over max |f(x)|, either path (incremental 3.9e-06, brute force 0: its occluded volumes run the
# same conv plans as x itself)
NULL_ERR = 1e-4


def _layers():
    return [(ks, pool) for _, _, ks, pool in TF.SNetSpec(128).layers]


def _guarded(shape, dtype, pad=4096):
    """A tensor of ``shape`` inside NaN-filled guard bands: (view, whole buffer, slice of the view)."""
    n = int(np.prod(shape))
    buf = torch.full((n + 2 * pad,), float("nan"), dtype=dtype, device=DEV)
    return buf[pad:pad + n].view(shape), buf, (pad, pad + n)


def _guards_intact(buf, span):
    return bool(torch.isnan(buf[:span[0]].float()).all()) and bool(torch.isnan(buf[span[1]:].float()).all())


def _sl(origin, size):
    return tuple(slice(int(o), int(o) + n) for o, n in zip(origin, size))


# ---------------------------------------------------------------------------------------------------------------
# kernels
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dims,win,st", [((23, 17, 29), (5, 4, 7), (3, 6, 4)), ((35, 38, 33), (8, 8, 8), (8, 5, 11)),
                                         ((16, 16, 16), (16, 3, 1), (1, 13, 2))])
@pytest.mark.parametrize("ng", [1, 2])
def test_occ_input_against_torch_indexing(dims, win, st, ng):
    B = 2
    plan = TF.OccPlan(dims, win, st, _layers())
    xs = [torch.randn((B, 1) + dims, device=DEV) for _ in range(ng)]
    tab = torch.from_numpy(plan.tab[0]).to(DEV)
    m = plan.nwin
    guarded = [_guarded((m * B, 1) + plan.crop[0], torch.float32) for _ in range(ng)]
    L.call("tmf_occ_input", ng, L.ptrs(xs), L.ptr(tab), m, -1.25, L.ptrs([g[0] for g in guarded]), B, *dims, *plan.crop[0])
    for x, (out, buf, span) in zip(xs, guarded):
        assert _guards_intact(buf, span)
        for n in range(m):
            t = plan.tab[0][n]
            ref = x[(slice(None), slice(None)) + _sl(t[:, 0], plan.crop[0])].clone()
            ref[(slice(None), slice(None)) + tuple(slice(int(lo - o), int(hi - o)) for o, lo, hi in t[:, :3])] = -1.25
            assert torch.equal(out[n * B:(n + 1) * B], ref)


def _compose_ref(base, crop, plan, l, n, B):
    t = plan.tab[l][n]
    ref = base[(slice(None),) + _sl(t[:, 0], plan.crop[l])].clone()
    if crop is not None:
        dst = tuple(slice(int(lo - o), int(hi - o)) for o, lo, hi in t[:, :3])
        src = tuple(slice(int(lo - s), int(hi - s)) for lo, hi, s in t[:, 1:])
        ref[(slice(None),) + dst] = crop[n * B:(n + 1) * B][(slice(None),) + src]
    return ref


@pytest.mark.parametrize("C", [32, 64, 128, 256])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
@pytest.mark.parametrize("ng", [1, 2])
def test_occ_compose_against_torch_indexing(C, dtype, ng):
    B = 2
    dims, win, st = (35, 38, 33), (7, 9, 5), (9, 6, 7)      # odd extents; the windows reach every face
    plan = TF.OccPlan(dims, win, st, _layers())
    layers = _layers()
    for l in (1, 2, 5, 7):                                    # unpooled, pooled, full-extent and output compositions
        ks, pool = layers[l - 1]
        prev = plan.out_extent(l - 1, pool)
        m = plan.nwin
        base = [torch.randn((B,) + plan.full[l] + (C,), device=DEV).to(dtype) for _ in range(ng)]
        crop = [torch.randn((m * B,) + prev + (C,), device=DEV).to(dtype) for _ in range(ng)]
        tab = torch.from_numpy(plan.tab[l]).to(DEV)
        for src in (crop, None):
            guarded = [_guarded((m * B,) + plan.crop[l] + (C,), dtype) for _ in range(ng)]
            TF.occ_compose(base, src, tab, m, plan.crop[l], out=[g[0] for g in guarded])
            for g, (out, buf, span) in enumerate(guarded):
                assert _guards_intact(buf, span)
                for n in range(m):
                    ref = _compose_ref(base[g], None if src is None else src[g], plan, l, n, B)
                    assert torch.equal(out[n * B:(n + 1) * B], ref), (l, n, src is None)


@pytest.mark.parametrize("dims,win,st", [((16, 17, 18), (4, 5, 6), (4, 2, 7)), ((23, 19, 21), (7, 3, 5), (5, 3, 9)),
                                         ((91, 109, 91), (16, 16, 16), (16, 16, 16))])
def test_occ_map_against_float64(dims, win, st):
    B = 3
    plan = TF.OccPlan(dims, win, st, _layers())
    scores = [torch.randn((B,) + plan.grid, device=DEV) for _ in range(2)]
    maps = TF.occ_map(scores, plan)
    for s, mp in zip(scores, maps):
        acc = torch.zeros((B,) + dims, dtype=torch.float64, device=DEV)
        cnt = torch.zeros(dims, dtype=torch.float64, device=DEV)
        for i in range(plan.grid[0]):
            for j in range(plan.grid[1]):
                for k in range(plan.grid[2]):
                    sl = _sl((i * st[0], j * st[1], k * st[2]), win)
                    acc[(slice(None),) + sl] += s[:, i, j, k].double().view(B, 1, 1, 1)
                    cnt[sl] += 1
        ref = torch.where(cnt > 0, acc / cnt.clamp_min(1), torch.zeros_like(acc))
        bound = cnt.clamp_min(1) * 2 ** -23 * s.abs().max().double() + 1e-30
        assert mp.shape == (B, 1) + dims and mp.dtype == torch.float32
        assert ((mp[:, 0].double() - ref).abs() <= bound).all()
        assert (mp[:, 0][:, cnt == 0] == 0).all()


# ---------------------------------------------------------------------------------------------------------------
# model level
# ---------------------------------------------------------------------------------------------------------------
def _model(gold):
    model = getattr(M, gold["kind"])(**gold["kwargs"])
    model.load_state_dict(H.case_state(gold), strict=True)
    model = model.to(DEV).eval()
    H.set_head_dropout(model, 0.0)
    return model


def _inputs(gold, zero_planes=0):
    mri, pet, label = H.case_inputs(gold)
    xs = (mri,) if gold["kind"] == "model_single" else (mri, pet)
    xs = [x.to(DEV).clone() for x in xs]
    for x in xs:
        x[:, :, :zero_planes] = 0
    return xs, label.to(DEV)


def _towers(model):
    return [m for m in model.modules() if isinstance(m, M.sNet)]


def _logits(outs):
    return outs[0] if isinstance(outs, (tuple, list)) else outs


def _brute(model, xs, target, window, stride, baseline, chunk):
    """Scores from the model's own forward on materialised occluded volumes, ``chunk`` windows per model call."""
    B, dims = xs[0].shape[0], tuple(xs[0].shape[2:])
    starts = [TF.occ_positions(E, w, s) for E, w, s in zip(dims, window, stride)]
    wins = [(a, b, c) for a in starts[0] for b in starts[1] for c in starts[2]]
    out = []
    with torch.no_grad():
        fx = _logits(model(*xs)).gather(1, target.view(-1, 1)).view(-1)
        for t in range(len(xs)):
            sc = []
            for k0 in range(0, len(wins), chunk):
                part = wins[k0:k0 + chunk]
                vols = []
                for o in part:
                    v = xs[t].clone()
                    v[(slice(None), slice(None)) + _sl(o, window)] = baseline
                    vols.append(v)
                occ = torch.cat(vols)
                X = [occ if u == t else x.repeat(len(part), 1, 1, 1, 1) for u, x in enumerate(xs)]
                f = _logits(model(*X)).gather(1, target.repeat(len(part)).view(-1, 1)).view(len(part), B)
                sc.append(fx.view(1, B) - f)
            out.append(torch.cat(sc).t().reshape((B,) + tuple(len(s) for s in starts)))
    return out, fx


CASES = [("model_single", (8, 8, 8), (8, 8, 8), 0.0), ("model_cnn_ad", (10, 7, 9), (7, 9, 6), 0.5),
         ("model_ad_h4", (8, 8, 8), (6, 7, 9), 0.0), ("model_ad_full_b2", (16, 16, 16), (24, 24, 24), 0.0)]


@pytest.mark.parametrize("name,window,stride,baseline", CASES)
def test_scores_against_brute_force(name, window, stride, baseline):
    gold = H.load_golden(name)
    model = _model(gold)
    xs, tgt = _inputs(gold, zero_planes=window[0])               # the first windows along D are null under baseline 0
    B = xs[0].shape[0]
    res = occlusion(model, xs, tgt, window=window, stride=stride, baseline=baseline, internal_batch_size=8 * B)
    ref, fx = _brute(model, xs, tgt, window, stride, baseline, chunk=8)
    scale = float(fx.abs().max())
    plan = TF.OccPlan(tuple(xs[0].shape[2:]), window, stride, _layers())
    for t, (got, want) in enumerate(zip(res.scores, ref)):
        assert got.shape == want.shape == (B,) + plan.grid and got.dtype == torch.float32
        err = float((got - want).abs().max()) / scale
        rel = float((got - want).norm() / want.norm().clamp_min(1e-30))
        msg = f"[occ] {name} tower {t}: max |inc - brute| / max |f(x)| {err:.2e}, relative L2 {rel:.2e}"
        if baseline == 0.0:
            null = slice(0, 1)                                   # window row i = 0 along D covers only zero planes
            ni, nb = float(got[:, null].abs().max()) / scale, float(want[:, null].abs().max()) / scale
            msg += f"; null windows: incremental {ni:.2e}, brute force {nb:.2e}"
            assert ni <= NULL_ERR and nb <= NULL_ERR
        print(msg)
        assert err <= SCORE_ERR, msg
        mp = res.maps[t]
        assert mp.shape == xs[t].shape and bool(torch.isfinite(mp).all())


def test_maps_apply_the_averaging_rule_to_the_scores():
    gold = H.load_golden("model_cnn_ad")
    model = _model(gold)
    xs, tgt = _inputs(gold)
    res = occlusion(model, xs, tgt, window=(10, 7, 9), stride=(7, 9, 6))
    plan = TF.OccPlan(tuple(xs[0].shape[2:]), (10, 7, 9), (7, 9, 6), _layers())
    for s, mp in zip(res.scores, res.maps):
        assert torch.equal(mp, TF.occ_map([s], plan)[0])


def test_determinism_and_pass_size():
    gold = H.load_golden("model_ad_h4")
    model = _model(gold)
    xs, tgt = _inputs(gold)
    B = xs[0].shape[0]
    a = occlusion(model, xs, tgt, window=8, stride=6, internal_batch_size=B)
    b = occlusion(model, xs, tgt, window=8, stride=6, internal_batch_size=B)
    c = occlusion(model, xs, tgt, window=8, stride=6)
    for x, y in zip(a.maps + a.scores, b.maps + b.scores):
        assert torch.equal(x, y)
    for x, y in zip(a.scores, c.scores):
        print(f"[occ] internal_batch_size B vs None: max |diff| {float((x - y).abs().max()):.2e}")
        assert torch.equal(x, y)


def test_side_effects(monkeypatch):
    gold = H.load_golden("model_ad_h4")
    model = _model(gold)
    model.fc_cls[0].weight.requires_grad_(False)
    xs, tgt = _inputs(gold)
    flags = {k: p.requires_grad for k, p in model.named_parameters()}
    before = {k: v.clone() for k, v in model.state_dict().items()}
    called = []
    real = L.call

    def spy(name, *args, **kw):
        called.append(kw.get("tag") or name)
        return real(name, *args, **kw)

    monkeypatch.setattr(L, "call", spy)
    occlusion(model, xs, tgt, window=12, stride=12, internal_batch_size=4 * xs[0].shape[0])
    monkeypatch.setattr(L, "call", real)
    assert all(p.grad is None for p in model.parameters())
    assert flags == {k: p.requires_grad for k, p in model.named_parameters()}
    assert not any(m.training for m in model.modules())
    for k, v in model.state_dict().items():
        assert torch.equal(v, before[k]), k
    assert all(t._occ_out is None and t._lrp_keep is None for t in _towers(model))
    bad = [s for s in called if "wgrad" in s or "bwd" in s or "dgrad" in s]
    assert not bad, bad
    plan = TF.OccPlan(tuple(xs[0].shape[2:]), (12,) * 3, (12,) * 3, _layers())
    passes = -(-plan.nwin // 4)
    assert called.count("tmf_occ_input") == passes and called.count("tmf_conv1_fwd@occ") == passes
    assert called.count("tmf_occ_map") == 1


def test_an_error_mid_call_leaves_the_model_usable(monkeypatch):
    gold = H.load_golden("model_cnn_ad")
    model = _model(gold)
    xs, tgt = _inputs(gold)
    B = xs[0].shape[0]
    ref = occlusion(model, xs, tgt, window=10, stride=10, internal_batch_size=B)
    with torch.no_grad():
        out0 = _logits(model(*xs)).clone()
    real, seen = TF.occ_towers, []

    def failing(*args, **kw):
        seen.append(1)
        if len(seen) == 2:
            raise RuntimeError("injected failure")
        return real(*args, **kw)

    monkeypatch.setattr(TF, "occ_towers", failing)
    with pytest.raises(RuntimeError, match="injected"):
        occlusion(model, xs, tgt, window=10, stride=10, internal_batch_size=B)
    monkeypatch.setattr(TF, "occ_towers", real)
    assert all(t._occ_out is None and t._lrp_keep is None for t in _towers(model))
    assert all(p.requires_grad for p in model.parameters())
    with torch.no_grad():
        assert torch.equal(_logits(model(*xs)), out0)
    again = occlusion(model, xs, tgt, window=10, stride=10, internal_batch_size=B)
    for x, y in zip(ref.scores + ref.maps, again.scores + again.maps):
        assert torch.equal(x, y)


def test_train_step_after_occlusion_is_bitwise_the_plain_one():
    gold = H.load_golden("model_cnn_ad")
    xs, label = _inputs(gold)

    def step(model):
        model.train()
        outs = model(*xs)
        loss = H.losses(outs if isinstance(outs, tuple) else (outs,), label)[2]
        loss.backward()
        return [p.grad.clone() for p in model.parameters() if p.grad is not None], \
            [b.clone() for b in model.buffers()], loss.detach()

    plain = _model(gold)
    other = copy.deepcopy(plain)
    occlusion(other, xs, label, window=10, stride=12)
    ga, ba, la = step(plain)
    gb, bb, lb = step(other)
    assert torch.equal(la, lb)
    for x, y in zip(ga + ba, gb + bb):
        assert torch.equal(x, y)


def test_occlusion_refuses_training_mode_on_the_gpu():
    gold = H.load_golden("model_cnn_ad")
    model = _model(gold).train()
    xs, tgt = _inputs(gold)
    with pytest.raises(ValueError, match="eval"):
        occlusion(model, xs, tgt, window=8, stride=8)
    assert all(t._occ_out is None for t in _towers(model))

"""Feature ablation over the regions of a mask with incremental recomputation (csrc/ablation.cu,
transmf_ad_b200.interpret.feature_ablation; DESIGN section 3.12).

Op level: tmf_abl_input and tmf_abl_map are copies, so they match a torch-indexing restatement bit for bit (outputs inside NaN
guard bands).  Model level: the scores against brute force -- the model's own forward on the materialised ablated volumes,
same regions --, null regions, agreement with occlusion on a mask that tiles its grid, absent and negative ids,
determinism, and the side-effect rules.  Measured values print with ``-s``.
"""
import copy

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests import helpers as H
from tests.test_gpu_occlusion import NULL_ERR, SCORE_ERR, _guarded, _guards_intact, _inputs, _logits, _model, _towers
from transmf_ad_b200 import _lib as L
from transmf_ad_b200 import functional as TF
from transmf_ad_b200.interpret import feature_ablation, occlusion
from transmf_ad_b200.synthetic import make_atlas

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _layers():
    return [(ks, pool) for _, _, ks, pool in TF.SNetSpec(128).layers]


def _atlas(dims, cells, seed, B=1):
    """make_atlas reaching every face (background: the corners), ids 1 and 2 merged (non-convex), id 2 absent; with B > 1
    every later sample is the first one shifted."""
    m = make_atlas(dims, cells, seed, radius=0.55)
    m[m == 2] = 1
    if B > 1:
        m = torch.cat([m] + [torch.roll(m, shifts=(b, -b), dims=(2, 4)) for b in range(1, B)])
    return m.to(DEV)


# ---------------------------------------------------------------------------------------------------------------
# kernels
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mask_b", [1, 2])
@pytest.mark.parametrize("kinds", [("scalar",), ("vol1",), ("volB",), ("scalar", "volB"), ("vol1", "scalar")])
def test_abl_input_against_torch_indexing(mask_b, kinds):
    B, dims = 2, (23, 17, 29)
    ng = len(kinds)
    mask = _atlas(dims, 7, 5, B=mask_b).to(torch.int32).contiguous()
    Fn = int(mask.max()) + 1
    boxes = TF.abl_boxes(mask, Fn)
    ids = [f for f in range(Fn) if boxes[f, 3] > boxes[f, 0]]
    plan = TF.abl_plan(boxes, ids, dims, _layers())
    xs = [torch.randn((B, 1) + dims, device=DEV) for _ in range(ng)]
    bl = []
    for g, k in enumerate(kinds):
        bl.append(-1.25 - g if k == "scalar" else torch.randn((1 if k == "vol1" else B, 1) + dims, device=DEV))
    tab = torch.from_numpy(plan.tab[0]).to(DEV)
    fid = torch.from_numpy(plan.ids).to(DEV)
    m = plan.n
    guarded = [_guarded((m * B, 1) + plan.crop[0], torch.float32) for _ in range(ng)]
    import ctypes
    vals = (ctypes.c_float * ng)(*[0.0 if torch.is_tensor(b) else b for b in bl])
    per = sum(1 << g for g, b in enumerate(bl) if torch.is_tensor(b) and b.shape[0] > 1)
    L.call("tmf_abl_input", ng, L.ptrs(xs), L.ptr(mask), int(mask_b > 1), L.ptrs([b if torch.is_tensor(b) else None for b in bl]),
           vals, per, L.ptr(tab), L.ptr(fid), m, L.ptrs([g[0] for g in guarded]), B, *dims, *plan.crop[0])
    for x, b, (out, buf, span) in zip(xs, bl, guarded):
        assert _guards_intact(buf, span)
        full = b.expand_as(x) if torch.is_tensor(b) else torch.full_like(x, b)
        for n in range(m):
            t = plan.tab[0][n]
            sl = (slice(None), slice(None)) + tuple(slice(int(o), int(o) + c) for o, c in zip(t[:, 0], plan.crop[0]))
            box = torch.zeros((B, 1) + dims, dtype=torch.bool, device=DEV)
            box[(slice(None), slice(None)) + tuple(slice(int(lo), int(hi)) for lo, hi in t[:, 1:3])] = True
            sel = (mask == int(plan.ids[n])).expand_as(x) & box
            ref = torch.where(sel, full, x)[sl]
            assert torch.equal(out[n * B:(n + 1) * B], ref), (kinds, n)
    # the wrapper launches the same thing
    again = TF.abl_input(xs, mask, bl, tab, fid, m, plan.crop[0])
    for a, (out, _, _) in zip(again, guarded):
        assert torch.equal(a, out)


@pytest.mark.parametrize("mask_b", [1, 3])
@pytest.mark.parametrize("ng", [1, 2])
def test_abl_map_against_a_torch_gather(mask_b, ng):
    B, dims = 3, (35, 38, 33)
    mask = _atlas(dims, 11, 2, B=mask_b).to(torch.int32).contiguous()
    Fn = int(mask.max()) + 1
    scores = [torch.randn((B, Fn), device=DEV) for _ in range(ng)]
    guarded = [_guarded((B, 1) + dims, torch.float32) for _ in range(ng)]
    L.call("tmf_abl_map", ng, L.ptrs(scores), L.ptr(mask), int(mask_b > 1), Fn, L.ptrs([g[0] for g in guarded]), B, *dims)
    for s, (out, buf, span) in zip(scores, guarded):
        assert _guards_intact(buf, span)
        ref = torch.gather(s, 1, mask.expand(B, -1, -1, -1, -1).reshape(B, -1).long()).view((B, 1) + dims)
        assert torch.equal(out, ref)
    assert all(torch.equal(a, g[0]) for a, g in zip(TF.abl_map(scores, mask), guarded))


# ---------------------------------------------------------------------------------------------------------------
# model level
# ---------------------------------------------------------------------------------------------------------------
def _brute(model, xs, target, mask, baselines, joint, chunk=4):
    """Scores (per tower, (B, F)) from the model's own forward on materialised ablated volumes."""
    B = xs[0].shape[0]
    Fn = int(mask.max()) + 1
    ids = [f for f in range(Fn) if bool((mask == f).any())]
    full = [b.expand_as(x) if torch.is_tensor(b) else torch.full_like(x, b) for x, b in zip(xs, baselines)]
    out = []
    with torch.no_grad():
        fx = _logits(model(*xs)).gather(1, target.view(-1, 1)).view(-1)
        for t in range(1 if joint else len(xs)):
            sc = torch.zeros((B, Fn), device=DEV)
            for k0 in range(0, len(ids), chunk):
                part = ids[k0:k0 + chunk]
                X = []
                for u, x in enumerate(xs):
                    if joint or u == t:
                        X.append(torch.cat([torch.where((mask == f).expand_as(x), full[u], x) for f in part]))
                    else:
                        X.append(x.repeat(len(part), 1, 1, 1, 1))
                f = _logits(model(*X)).gather(1, target.repeat(len(part)).view(-1, 1)).view(len(part), B)
                sc[:, part] = (fx.view(1, B) - f).t()
            out.append(sc)
    return (out * len(xs) if joint else out), fx


CASES = [("model_single", 12), ("model_cnn_ad", 10), ("model_ad_h4", 9), ("model_ad_full_b2", 24)]


@pytest.mark.parametrize("joint", [False, True])
@pytest.mark.parametrize("kind", ["scalar", "per_voxel"])
@pytest.mark.parametrize("name,cells", CASES)
def test_scores_against_brute_force(name, cells, kind, joint):
    gold = H.load_golden(name)
    model = _model(gold)
    xs, tgt = _inputs(gold)
    B, dims = xs[0].shape[0], tuple(xs[0].shape[2:])
    mask = _atlas(dims, cells, len(name), B=B if kind == "per_voxel" else 1)
    null = 3                                                            # x already equals the baseline on region 3
    if kind == "scalar":
        baselines = 0.0
        bl = [0.0] * len(xs)
    else:
        bl = [F.avg_pool3d(x, 5, 1, 2, count_include_pad=False).contiguous() for x in xs]   # a blurred copy of the subject
        baselines = tuple(bl)
    for x, b in zip(xs, bl):
        sel = (mask == null).expand_as(x)
        x[sel] = b.expand_as(x)[sel] if torch.is_tensor(b) else b
    res = feature_ablation(model, xs, tgt, mask, baselines, joint=joint, internal_batch_size=4 * B)
    ref, fx = _brute(model, xs, tgt, mask, bl, joint)
    scale = float(fx.abs().max())
    Fn = int(mask.max()) + 1
    for t, (got, want) in enumerate(zip(res.scores, ref)):
        assert got.shape == want.shape == (B, Fn) and got.dtype == torch.float32
        err = float((got - want).abs().max()) / scale
        rel = float((got - want).norm() / want.norm().clamp_min(1e-30))
        ni = float(got[:, null].abs().max()) / scale
        print(f"[abl] {name} {kind} joint={joint} tower {t}: max |inc - brute| / max |f(x)| {err:.2e}, relative L2 "
              f"{rel:.2e}; null region {ni:.2e}")
        assert err <= SCORE_ERR and ni <= NULL_ERR
        assert bool((got[:, 2] == 0).all())                              # id 2 is absent
        mp = res.maps[t]
        assert mp.shape == xs[t].shape and torch.equal(mp, TF.abl_map([got], mask.to(torch.int32).contiguous())[0])
    if joint:
        assert all(torch.equal(s, res.scores[0]) for s in res.scores)


def test_agreement_with_occlusion_on_its_grid():
    gold = H.load_golden("model_ad_h4")
    model = _model(gold)
    xs, tgt = _inputs(gold)
    B, dims = xs[0].shape[0], tuple(xs[0].shape[2:])
    w = (8, 9, 7)
    grid = tuple(len(TF.occ_positions(E, a, a)) for E, a in zip(dims, w))
    mask = torch.full((1, 1) + dims, int(np.prod(grid)), dtype=torch.long, device=DEV)   # voxels no window covers
    for i in range(grid[0]):
        for j in range(grid[1]):
            for k in range(grid[2]):
                mask[0, 0, i * w[0]:(i + 1) * w[0], j * w[1]:(j + 1) * w[1], k * w[2]:(k + 1) * w[2]] = (i * grid[1] + j) * grid[2] + k
    occ = occlusion(model, xs, tgt, window=w, stride=w, baseline=0.5)
    abl = feature_ablation(model, xs, tgt, mask, 0.5)
    with torch.no_grad():
        scale = float(_logits(model(*xs)).gather(1, tgt.view(-1, 1)).abs().max())
    for o, a in zip(occ.scores, abl.scores):
        err = float((o.reshape(B, -1) - a[:, :-1]).abs().max()) / scale
        print(f"[abl] against occlusion(window = stride = {w}): max |diff| / max |f(x)| {err:.2e}")
        assert err <= SCORE_ERR


def test_absent_ids_score_zero_and_launch_nothing(monkeypatch):
    gold = H.load_golden("model_cnn_ad")
    model = _model(gold)
    xs, tgt = _inputs(gold)
    dims = tuple(xs[0].shape[2:])
    mask = torch.zeros((1, 1) + dims, dtype=torch.int16, device=DEV)
    mask[..., 10:20, 5:25, :] = 5
    mask[..., 25:, :, 3:9] = 2
    seen = []
    real = TF.abl_input

    def spy(xs_, mask_, bl_, tab, ids, m, extent):
        seen.extend(ids.tolist())
        return real(xs_, mask_, bl_, tab, ids, m, extent)

    monkeypatch.setattr(TF, "abl_input", spy)
    res = feature_ablation(model, xs, tgt, mask, internal_batch_size=xs[0].shape[0])
    assert sorted(set(seen)) == [0, 2, 5]
    for s in res.scores:
        assert s.shape == (xs[0].shape[0], 6)
        assert bool((s[:, [1, 3, 4]] == 0).all()) and bool((s[:, [0, 2, 5]] != 0).any())


def test_negative_ids_are_refused_before_any_launch(monkeypatch):
    gold = H.load_golden("model_cnn_ad")
    model = _model(gold)
    xs, tgt = _inputs(gold)
    mask = torch.zeros((1, 1) + tuple(xs[0].shape[2:]), dtype=torch.int64, device=DEV)
    mask[..., 3, 4, 5] = -1

    def refuse(name, *args, **kw):
        raise AssertionError(f"{name} launched")

    monkeypatch.setattr(L, "call", refuse)
    with pytest.raises(ValueError, match=">= 0"):
        feature_ablation(model, xs, tgt, mask)
    assert all(t._occ_out is None and t._lrp_keep is None for t in _towers(model))


def test_determinism_and_pass_size():
    gold = H.load_golden("model_ad_h4")
    model = _model(gold)
    xs, tgt = _inputs(gold)
    B, dims = xs[0].shape[0], tuple(xs[0].shape[2:])
    mask = _atlas(dims, 20, 7, B=B)
    bl = (0.25, F.avg_pool3d(xs[1], 3, 1, 1).contiguous())
    for joint in (False, True):
        a = feature_ablation(model, xs, tgt, mask, bl, joint=joint, internal_batch_size=B)
        b = feature_ablation(model, xs, tgt, mask, bl, joint=joint, internal_batch_size=B)
        c = feature_ablation(model, xs, tgt, mask, bl, joint=joint)
        for x, y in zip(a.maps + a.scores, b.maps + b.scores):
            assert torch.equal(x, y)
        for x, y in zip(a.scores + a.maps, c.scores + c.maps):
            print(f"[abl] joint={joint} internal_batch_size B vs None: max |diff| {float((x - y).abs().max()):.2e}")
            assert torch.equal(x, y)


def test_side_effects(monkeypatch):
    gold = H.load_golden("model_ad_h4")
    model = _model(gold)
    model.fc_cls[0].weight.requires_grad_(False)
    xs, tgt = _inputs(gold)
    B, dims = xs[0].shape[0], tuple(xs[0].shape[2:])
    mask = _atlas(dims, 9, 1)
    flags = {k: p.requires_grad for k, p in model.named_parameters()}
    before = {k: v.clone() for k, v in model.state_dict().items()}
    called = []
    real = L.call

    def spy(name, *args, **kw):
        called.append(kw.get("tag") or name)
        return real(name, *args, **kw)

    monkeypatch.setattr(L, "call", spy)
    feature_ablation(model, xs, tgt, mask, internal_batch_size=3 * B)
    monkeypatch.setattr(L, "call", real)
    assert all(p.grad is None for p in model.parameters())
    assert flags == {k: p.requires_grad for k, p in model.named_parameters()}
    assert not any(m.training for m in model.modules())
    for k, v in model.state_dict().items():
        assert torch.equal(v, before[k]), k
    assert all(t._occ_out is None and t._lrp_keep is None for t in _towers(model))
    bad = [s for s in called if "wgrad" in s or "bwd" in s or "dgrad" in s]
    assert not bad, bad
    boxes = TF.abl_boxes(mask, int(mask.max()) + 1)
    passes = sum(-(-len(ids) // 3) for _, ids in TF.abl_classes(boxes, dims))
    assert called.count("tmf_abl_input") == passes and called.count("tmf_conv1_fwd@occ") == passes
    assert called.count("tmf_abl_map") == 1 and "tmf_occ_input" not in called


def test_an_error_mid_call_leaves_the_model_usable(monkeypatch):
    gold = H.load_golden("model_cnn_ad")
    model = _model(gold)
    xs, tgt = _inputs(gold)
    B, dims = xs[0].shape[0], tuple(xs[0].shape[2:])
    mask = _atlas(dims, 9, 4)
    ref = feature_ablation(model, xs, tgt, mask, internal_batch_size=2 * B)
    with torch.no_grad():
        out0 = _logits(model(*xs)).clone()
    real, seen = TF.occ_crops, []

    def failing(*args, **kw):
        seen.append(1)
        if len(seen) == 2:
            raise RuntimeError("injected failure")
        return real(*args, **kw)

    monkeypatch.setattr(TF, "occ_crops", failing)
    with pytest.raises(RuntimeError, match="injected"):
        feature_ablation(model, xs, tgt, mask, internal_batch_size=2 * B)
    monkeypatch.setattr(TF, "occ_crops", real)
    assert all(t._occ_out is None and t._lrp_keep is None for t in _towers(model))
    assert all(p.requires_grad for p in model.parameters())
    with torch.no_grad():
        assert torch.equal(_logits(model(*xs)), out0)
    again = feature_ablation(model, xs, tgt, mask, internal_batch_size=2 * B)
    for x, y in zip(ref.scores + ref.maps, again.scores + again.maps):
        assert torch.equal(x, y)


def test_train_step_after_ablation_is_bitwise_the_plain_one():
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
    feature_ablation(other, xs, label, _atlas(tuple(xs[0].shape[2:]), 9, 6), 0.5, joint=True)
    ga, ba, la = step(plain)
    gb, bb, lb = step(other)
    assert torch.equal(la, lb)
    for x, y in zip(ga + ba, gb + bb):
        assert torch.equal(x, y)

"""Shapley value sampling over the regions of a mask with per-chain state (csrc/shapley.cu,
transmf_ad_b200.interpret.shapley_sampling; DESIGN section 3.13).

Op level: tmf_shap_input and tmf_shap_compose are copies, so they match a torch-indexing restatement bit for bit (outputs
inside NaN guard bands; the written-back state, and the state outside the changed regions untouched), including a chain
state of more than 2^31 elements.  Model level: the scores against brute force -- the model's own forward on the
materialised composite volumes of the same permutations --, the telescoping delta, a one-region mask and absent ids,
bitwise independence of the pass size, the state budget and repeated calls, and the side-effect rules.  Measured values
print with ``-s``.
"""
import copy

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests import helpers as H
from tests.test_gpu_ablation import CASES, _atlas, _layers
from tests.test_gpu_occlusion import _guarded, _guards_intact, _inputs, _logits, _model, _towers
from transmf_ad_b200 import _lib as L
from transmf_ad_b200 import functional as TF
from transmf_ad_b200.interpret import shapley_sampling

pytestmark = pytest.mark.gpu
DEV = "cuda"
# worst |incremental - brute force| score over max |f(x)|, and |delta| over max |f(x)|
SCORE_ERR = 1e-3


# ---------------------------------------------------------------------------------------------------------------
# kernels
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mask_b", [1, 2])
@pytest.mark.parametrize("kinds", [("scalar",), ("vol1",), ("volB",), ("scalar", "volB"), ("vol1", "scalar")])
def test_shap_input_against_torch_indexing(mask_b, kinds):
    B, dims = 2, (23, 17, 29)
    ng = len(kinds)
    mask = _atlas(dims, 7, 5, B=mask_b).to(torch.int32).contiguous()
    Fn = int(mask.max()) + 1
    boxes = TF.abl_boxes(mask, Fn)
    ids = [f for f in range(Fn) if boxes[f, 3] > boxes[f, 0]]
    plan = TF.abl_plan(boxes, ids, dims, _layers())
    g = torch.Generator().manual_seed(mask_b + ng)
    P = 4
    perms = torch.stack([torch.as_tensor(ids)[torch.randperm(len(ids), generator=g)] for _ in range(P)])
    rank = torch.full((P, Fn), 2 ** 31 - 1, dtype=torch.int32)
    for p in range(P):
        rank[p, perms[p]] = torch.arange(len(ids), dtype=torch.int32)
    xs = [torch.randn((B, 1) + dims, device=DEV) for _ in range(ng)]
    bl = [-1.25 - i if k == "scalar" else torch.randn((1 if k == "vol1" else B, 1) + dims, device=DEV)
          for i, k in enumerate(kinds)]
    rows = [(p, k) for p in range(P) for k in range(len(ids)) if (p + k) % 3 == 0]       # (chain, step), any order
    where = {int(f): n for n, f in enumerate(plan.ids)}
    tab = torch.from_numpy(np.stack([plan.tab[0][where[int(perms[p, k])]] for p, k in rows])).to(DEV)
    perm = torch.tensor([p for p, _ in rows], dtype=torch.int32, device=DEV)
    step = torch.tensor([k for _, k in rows], dtype=torch.int32, device=DEV)
    rank_d = rank.to(DEV)
    m = len(rows)
    guarded = [_guarded((m * B, 1) + plan.crop[0], torch.float32) for _ in range(ng)]
    import ctypes
    vals = (ctypes.c_float * ng)(*[0.0 if torch.is_tensor(b) else b for b in bl])
    per = sum(1 << i for i, b in enumerate(bl) if torch.is_tensor(b) and b.shape[0] > 1)
    L.call("tmf_shap_input", ng, L.ptrs(xs), L.ptr(mask), int(mask_b > 1), L.ptrs([b if torch.is_tensor(b) else None for b in bl]),
           vals, per, L.ptr(tab), L.ptr(rank_d), Fn, L.ptr(perm), L.ptr(step), m, L.ptrs([q[0] for q in guarded]), B, *dims,
           *plan.crop[0])
    for x, b, (out, buf, span) in zip(xs, bl, guarded):
        assert _guards_intact(buf, span)
        full = b.expand_as(x) if torch.is_tensor(b) else torch.full_like(x, b)
        for n, (p, k) in enumerate(rows):
            o = tab[n, :, 0].tolist()
            sl = (slice(None), slice(None)) + tuple(slice(a, a + c) for a, c in zip(o, plan.crop[0]))
            keep = (rank_d[p][mask.long()] <= k).expand_as(x)
            assert torch.equal(out[n * B:(n + 1) * B], torch.where(keep, x, full)[sl]), (kinds, p, k)
    again = TF.shap_input(xs, mask, bl, tab, rank_d, perm, step, m, plan.crop[0])
    assert all(torch.equal(a, q[0]) for a, q in zip(again, guarded))


def _compose_case(S, B, dims, C, crop, m, dtype, ng, seed):
    """Random chain states, crops and tables: per row an origin, a changed region inside the crop and a previous-output
    origin at most 2 below it, so that the previous crop (extent crop + 2) covers the region."""
    rng = np.random.default_rng(seed)
    prev = tuple(c + 2 for c in crop)
    tab = np.zeros((m, 3, 4), dtype=np.int32)
    for n in range(m):
        for a in range(3):
            c0 = int(rng.integers(0, dims[a] - crop[a] + 1))
            lo = int(rng.integers(c0, c0 + crop[a]))
            hi = int(rng.integers(lo + 1, c0 + crop[a] + 1))
            tab[n, a] = (c0, lo, hi, lo - int(rng.integers(0, min(lo, 2) + 1)))
    sidx = rng.permutation(S)[:m].astype(np.int32)
    state = [torch.randn((S * B,) + dims + (C,), device=DEV).to(dtype) for _ in range(ng)]
    crops = [torch.randn((m * B,) + prev + (C,), device=DEV).to(dtype) for _ in range(ng)]
    return tab, sidx, state, crops


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
@pytest.mark.parametrize("ng", [1, 2])
def test_shap_compose_against_torch_indexing(dtype, ng):
    S, B, dims, C, crop, m = 7, 2, (11, 13, 9), 24, (5, 6, 4), 5
    tab, sidx, state, crops = _compose_case(S, B, dims, C, crop, m, dtype, ng, seed=ng)
    _check_compose(tab, sidx, state, crops, B, crop, dtype)


def _check_compose(tab, sidx, state, crops, B, crop, dtype):
    m = len(sidx)
    C = state[0].shape[-1]
    before = [s.clone() for s in state]
    guarded = [_guarded((m * B,) + crop + (C,), dtype) for _ in state]
    tab_d, sidx_d = torch.from_numpy(tab).to(DEV), torch.from_numpy(sidx).to(DEV)
    L.call("tmf_shap_compose", len(state), L.ptrs(state), L.ptr(sidx_d), L.ptrs(crops), L.ptr(tab_d), m,
           L.ptrs([q[0] for q in guarded]), B, *state[0].shape[1:4], *crop, *crops[0].shape[1:4], C,
           int(dtype == torch.float32))
    for s, b0, c, (out, buf, span) in zip(state, before, crops, guarded):
        assert _guards_intact(buf, span)
        after = b0.clone()
        for n in range(m):
            t = tab[n]
            rows = slice(int(sidx[n]) * B, (int(sidx[n]) + 1) * B)
            region = tuple(slice(int(t[a, 1]), int(t[a, 2])) for a in range(3))
            src = tuple(slice(int(t[a, 1] - t[a, 3]), int(t[a, 2] - t[a, 3])) for a in range(3))
            after[(rows,) + region] = c[(slice(n * B, (n + 1) * B),) + src]
        assert torch.equal(s, after)                                 # written back inside [lo, hi), untouched elsewhere
        for n in range(m):
            t = tab[n]
            rows = slice(int(sidx[n]) * B, (int(sidx[n]) + 1) * B)
            win = tuple(slice(int(t[a, 0]), int(t[a, 0]) + crop[a]) for a in range(3))
            assert torch.equal(out[n * B:(n + 1) * B], after[(rows,) + win]), n
    return [q[0] for q in guarded]


def test_shap_compose_wrapper_and_a_state_past_2_31_elements():
    S, B, dims, C, crop = 40, 1, (40, 40, 40), 1024, (6, 5, 7)
    assert S * B * np.prod(dims) * C > 2 ** 31
    rng = np.random.default_rng(9)
    tab = np.zeros((3, 3, 4), dtype=np.int32)
    for n in range(3):
        for a in range(3):
            c0 = int(rng.integers(0, dims[a] - crop[a] + 1))
            tab[n, a] = (c0, c0 + 1, c0 + crop[a] - 1, c0)
    sidx = np.array([S - 1, 0, S - 2], dtype=np.int32)                   # the last chains sit past 2^31 elements
    state = [torch.randn((S * B,) + dims + (C,), device=DEV, dtype=torch.bfloat16)]
    crops = [torch.randn((3 * B,) + crop + (C,), device=DEV, dtype=torch.bfloat16)]
    out = _check_compose(tab, sidx, state, crops, B, crop, torch.bfloat16)
    # the wrapper launches the same thing (on fresh copies: the first launch already wrote back)
    st2 = [s.clone() for s in state]
    again = TF.shap_compose(st2, torch.from_numpy(sidx).to(DEV), crops, torch.from_numpy(tab).to(DEV), 3, crop)
    assert torch.equal(again[0], out[0]) and torch.equal(st2[0], state[0])


# ---------------------------------------------------------------------------------------------------------------
# model level
# ---------------------------------------------------------------------------------------------------------------
def _f(model, X, target, reps):
    return _logits(model(*X)).gather(1, target.repeat(reps).view(-1, 1)).view(reps, -1)


def _brute(model, xs, target, mask, baselines, joint, perms, chunk=8):
    """Scores (per tower, (B, F)) and f(start) per block from the model's own forward on the materialised composite volumes
    of every chain of ``perms``."""
    B = xs[0].shape[0]
    Fn = int(mask.max()) + 1
    P, Fp = perms.shape
    full = [b.expand_as(x) if torch.is_tensor(b) else torch.full_like(x, b) for x, b in zip(xs, baselines)]
    out, starts = [], []
    with torch.no_grad():
        for t in range(1 if joint else len(xs)):
            sc = torch.zeros((B, Fn), device=DEV, dtype=torch.float64)
            for p in range(P):
                rank = torch.full((Fn,), Fp, dtype=torch.long, device=DEV)
                rank[perms[p].to(DEV)] = torch.arange(Fp, device=DEV)
                fs = []
                ks = list(range(-1, Fp))
                for k0 in range(0, len(ks), chunk):
                    part = ks[k0:k0 + chunk]
                    X = []
                    for u, x in enumerate(xs):
                        if joint or u == t:
                            X.append(torch.cat([torch.where((rank[mask.long()] <= k).expand_as(x), x, full[u]) for k in part]))
                        else:
                            X.append(x.repeat(len(part), 1, 1, 1, 1))
                    fs.append(_f(model, X, target, len(part)))
                fs = torch.cat(fs).double()
                sc[:, perms[p].to(DEV)] += (fs[1:] - fs[:-1]).t()
                if p == 0:
                    starts.append(fs[0].float())
            out.append((sc / P).float())
    return (out * len(xs) if joint else out), (starts * len(xs) if joint else starts)


@pytest.mark.parametrize("joint", [False, True])
@pytest.mark.parametrize("kind", ["scalar", "per_voxel"])
@pytest.mark.parametrize("name,cells", CASES)
def test_scores_against_brute_force(name, cells, kind, joint):
    gold = H.load_golden(name)
    model = _model(gold)
    xs, tgt = _inputs(gold)
    B, dims = xs[0].shape[0], tuple(xs[0].shape[2:])
    mask = _atlas(dims, cells, len(name), B=B if kind == "per_voxel" else 1)
    if kind == "scalar":
        baselines = 0.0
        bl = [0.0] * len(xs)
    else:
        bl = [F.avg_pool3d(x, 5, 1, 2, count_include_pad=False).contiguous() for x in xs]   # a blurred copy of the subject
        baselines = tuple(bl)
    n = 2 if "full" in name else 3
    torch.manual_seed(len(name) + joint)
    res = shapley_sampling(model, xs, tgt, mask, baselines, joint=joint, n_samples=n, internal_batch_size=4 * B)
    assert res.permutations.shape[0] == n and res.permutations.dtype == torch.int64
    ref, f_start = _brute(model, xs, tgt, mask, bl, joint, res.permutations)
    with torch.no_grad():
        fx = _logits(model(*xs)).gather(1, tgt.view(-1, 1)).view(-1)
    scale = float(fx.abs().max())
    Fn = int(mask.max()) + 1
    for t, (got, want) in enumerate(zip(res.scores, ref)):
        assert got.shape == want.shape == (B, Fn) and got.dtype == torch.float32
        err = float((got - want).abs().max()) / scale
        rel = float((got - want).norm() / want.norm().clamp_min(1e-30))
        d = float(res.delta[t].abs().max()) / scale
        dref = float((want.sum(1) - (fx - f_start[t])).abs().max()) / scale
        print(f"[shap] {name} {kind} joint={joint} tower {t}: max |inc - brute| / max |f(x)| {err:.2e}, relative L2 "
              f"{rel:.2e}; |delta| / max |f(x)| {d:.2e} (brute force {dref:.2e})")
        assert err <= SCORE_ERR and d <= SCORE_ERR
        assert res.delta[t].shape == (B,) and res.delta[t].dtype == torch.float32
        assert bool((got[:, 2] == 0).all())                              # id 2 is absent
        assert torch.equal(res.maps[t], TF.abl_map([got], mask.to(torch.int32).contiguous())[0])
    if joint:
        assert all(torch.equal(s, res.scores[0]) for s in res.scores)


def test_one_region_and_absent_ids():
    gold = H.load_golden("model_ad_h4")
    model = _model(gold)
    xs, tgt = _inputs(gold)
    dims = tuple(xs[0].shape[2:])
    mask = torch.full((1, 1) + dims, 3, dtype=torch.int16, device=DEV)
    res = shapley_sampling(model, xs, tgt, mask, 0.25, n_samples=4)
    assert res.permutations.tolist() == [[3]] * 4
    with torch.no_grad():
        fx = _logits(model(*xs)).gather(1, tgt.view(-1, 1)).view(-1)
        scale = float(fx.abs().max())
        for t, s in enumerate(res.scores):
            X = [torch.full_like(x, 0.25) if u == t else x for u, x in enumerate(xs)]
            want = fx - _logits(model(*X)).gather(1, tgt.view(-1, 1)).view(-1)
            assert s.shape == (xs[0].shape[0], 4) and bool((s[:, :3] == 0).all())
            err = float((s[:, 3] - want).abs().max()) / scale
            print(f"[shap] one region, tower {t}: |score - (f(x) - f(start))| / max |f(x)| {err:.2e}")
            assert err <= SCORE_ERR
    mask[..., 10:20, 5:25, :] = 5
    mask[..., 25:, :, 3:9] = 0
    res = shapley_sampling(model, xs, tgt, mask, n_samples=5)
    assert all(sorted(r) == [0, 3, 5] for r in res.permutations.tolist())
    for s in res.scores:
        assert s.shape == (xs[0].shape[0], 6) and bool((s[:, [1, 2, 4]] == 0).all()) and bool((s[:, [0, 3, 5]] != 0).any())


def test_bits_do_not_depend_on_pass_size_state_budget_or_the_call(monkeypatch):
    gold = H.load_golden("model_ad_h4")
    model = _model(gold)
    xs, tgt = _inputs(gold)
    B, dims = xs[0].shape[0], tuple(xs[0].shape[2:])
    mask = _atlas(dims, 14, 7, B=B)
    bl = (0.25, F.avg_pool3d(xs[1], 3, 1, 1).contiguous())
    for joint in (False, True):
        runs = []
        for ibs, budget in ((B, None), (3 * B, None), (None, None), (None, 1), (None, None)):
            if budget is not None:
                monkeypatch.setattr(TF, "SHAP_STATE_BYTES", budget)            # one permutation per group
            torch.manual_seed(11)
            runs.append(shapley_sampling(model, xs, tgt, mask, bl, joint=joint, n_samples=4, internal_batch_size=ibs))
            monkeypatch.undo()
        for r in runs[1:]:
            assert torch.equal(r.permutations, runs[0].permutations)
            for x, y in zip(runs[0].scores + runs[0].maps + runs[0].delta, r.scores + r.maps + r.delta):
                assert torch.equal(x, y)
        print(f"[shap] joint={joint}: bitwise equal over internal_batch_size B, 3B, None, one permutation per group and a "
              f"repeated call")


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
    res = shapley_sampling(model, xs, tgt, mask, n_samples=3, internal_batch_size=2 * B)
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
    classes = TF.abl_classes(boxes, dims)
    cls_of = {f: c for c, (_, ids) in enumerate(classes) for f in ids}
    passes = len(TF.shap_schedule(res.permutations.numpy(), cls_of, [2] * len(classes)))
    assert called.count("tmf_shap_input") == passes and called.count("tmf_conv1_fwd@occ") == passes
    assert called.count("tmf_shap_compose@out") == passes and called.count("tmf_abl_map") == 1
    assert "tmf_occ_input" not in called and "tmf_abl_input" not in called


def test_an_error_mid_call_leaves_the_model_usable(monkeypatch):
    gold = H.load_golden("model_cnn_ad")
    model = _model(gold)
    xs, tgt = _inputs(gold)
    B, dims = xs[0].shape[0], tuple(xs[0].shape[2:])
    mask = _atlas(dims, 9, 4)
    torch.manual_seed(2)
    ref = shapley_sampling(model, xs, tgt, mask, n_samples=2, internal_batch_size=2 * B)
    with torch.no_grad():
        out0 = _logits(model(*xs)).clone()
    real, seen = TF.shap_crops, []

    def failing(*args, **kw):
        seen.append(1)
        if len(seen) == 2:
            raise RuntimeError("injected failure")
        return real(*args, **kw)

    monkeypatch.setattr(TF, "shap_crops", failing)
    with pytest.raises(RuntimeError, match="injected"):
        shapley_sampling(model, xs, tgt, mask, n_samples=2, internal_batch_size=2 * B)
    monkeypatch.setattr(TF, "shap_crops", real)
    assert all(t._occ_out is None and t._lrp_keep is None for t in _towers(model))
    assert all(p.requires_grad for p in model.parameters())
    with torch.no_grad():
        assert torch.equal(_logits(model(*xs)), out0)
    torch.manual_seed(2)
    again = shapley_sampling(model, xs, tgt, mask, n_samples=2, internal_batch_size=2 * B)
    for x, y in zip(ref.scores + ref.maps + ref.delta, again.scores + again.maps + again.delta):
        assert torch.equal(x, y)


def test_train_step_after_shapley_is_bitwise_the_plain_one():
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
    shapley_sampling(other, xs, label, _atlas(tuple(xs[0].shape[2:]), 9, 6), 0.5, joint=True, n_samples=2)
    ga, ba, la = step(plain)
    gb, bb, lb = step(other)
    assert torch.equal(la, lb)
    for x, y in zip(ga + ba, gb + bb):
        assert torch.equal(x, y)

"""Host-side rules of interpret.feature_ablation (no GPU, no kernel launch): the argument refusals, the box planner
(functional.BoxPlan) against OccPlan on the occlusion grids, the extent classes, and the box planner against a float64
restatement of the folded eval sNet: composing crops exactly as the planner's tables say must reproduce the tower output of
every ablated volume (DESIGN section 3.12)."""
import numpy as np
import pytest
import torch

from tests.test_occlusion_host import _forward, _layer, _layers, _params, _sl
from transmf_ad_b200 import _lib as L
from transmf_ad_b200 import functional as TF
from transmf_ad_b200.interpret import feature_ablation
from transmf_ad_b200.models import mymodel as M
from transmf_ad_b200.models.MiSePyNet import Mnet
from transmf_ad_b200.synthetic import make_atlas


@pytest.fixture
def no_launch(monkeypatch):
    def refuse(name, *args, **kw):
        raise AssertionError(f"{name} launched before the arguments were checked")
    monkeypatch.setattr(L, "call", refuse)


def _model():
    return M.model_CNN_ad(128).eval()


DIMS = (16, 16, 16)


def _inputs(B=2, dims=DIMS):
    return torch.zeros((B, 1) + dims), torch.zeros((B, 1) + dims)


def _mask(B=1, dims=DIMS, dtype=torch.int64):
    return torch.zeros((B, 1) + dims, dtype=dtype)


def _call(model=None, inputs=None, target=0, mask=None, **kw):
    return feature_ablation(_model() if model is None else model, _inputs() if inputs is None else inputs, target,
                            _mask() if mask is None else mask, **kw)


@pytest.mark.parametrize("mask", [_mask(dtype=torch.float32), _mask(dtype=torch.bool), _mask(dtype=torch.float64),
                                  torch.zeros((1, 16, 16, 16), dtype=torch.long), _mask(B=3), _mask(dims=(16, 16, 17)),
                                  torch.zeros((1, 2) + DIMS, dtype=torch.long), _mask().to("meta"), np.zeros((1, 1) + DIMS),
                                  None, 0])
def test_bad_masks_are_refused(mask, no_launch):
    with pytest.raises(ValueError, match="feature_mask"):
        feature_ablation(_model(), _inputs(), 0, mask)


@pytest.mark.parametrize("dtype", [torch.uint8, torch.int8, torch.int16, torch.int32, torch.int64])
@pytest.mark.parametrize("B", [1, 2])
def test_integer_masks_pass_the_mask_checks(dtype, B, no_launch):
    with pytest.raises(ValueError, match="CUDA"):                    # the next refusal: the inputs are on the CPU
        _call(mask=_mask(B=B, dtype=dtype))


@pytest.mark.parametrize("baselines", [float("nan"), float("inf"), -float("inf"), None, True, "0", np.zeros(3),
                                       torch.tensor(0.0), (0.0,), (0.0, 0.0, 0.0), [0.0, float("nan")],
                                       (0.0, torch.zeros((2, 1) + DIMS, dtype=torch.float64)),
                                       (0.0, torch.zeros((3, 1) + DIMS)), (torch.zeros((1, 1, 16, 16, 15)), 0.0),
                                       (torch.zeros((1,) + DIMS), 0.0), (0.0, torch.zeros((1, 1) + DIMS).to("meta")),
                                       torch.zeros((1, 1) + DIMS)])
def test_bad_baselines_are_refused(baselines, no_launch):
    with pytest.raises(ValueError, match="baseline"):
        _call(baselines=baselines)


@pytest.mark.parametrize("baselines", [0.5, -2, (0.0, 1.0), [torch.zeros((1, 1) + DIMS), torch.ones((2, 1) + DIMS)]])
def test_good_baselines_pass_the_baseline_checks(baselines, no_launch):
    with pytest.raises(ValueError, match="CUDA"):
        _call(baselines=baselines)


@pytest.mark.parametrize("ibs", [0, -8, 8.0, False, "64"])
def test_bad_internal_batch_sizes_are_refused(ibs, no_launch):
    with pytest.raises(ValueError, match="internal_batch_size"):
        _call(internal_batch_size=ibs)


@pytest.mark.parametrize("joint", [1, 0, None, "True"])
def test_bad_joint_flags_are_refused(joint, no_launch):
    with pytest.raises(ValueError, match="joint"):
        _call(joint=joint)


def test_training_mode_is_refused(no_launch):
    with pytest.raises(ValueError, match="eval"):
        _call(model=_model().train())
    model = _model()
    model.fc_cls.train()
    with pytest.raises(ValueError, match="eval"):
        _call(model=model)


def test_a_model_without_towers_is_refused(no_launch):
    with pytest.raises(ValueError, match="sNet"):
        _call(model=Mnet().eval())


@pytest.mark.parametrize("inputs", [torch.zeros(2, 1, 16, 16), (torch.zeros(2, 2, 16, 16, 16),) * 2, (), ("mri", "pet"),
                                    (torch.zeros(2, 1, 16, 16, 16),),
                                    (torch.zeros(2, 1, 16, 16, 16), torch.zeros(2, 1, 16, 16, 17)),
                                    (torch.zeros(2, 1, 16, 16, 16),) * 3])
def test_bad_inputs_are_refused(inputs, no_launch):
    with pytest.raises(ValueError, match="inputs"):
        _call(inputs=inputs)


@pytest.mark.parametrize("target", [2.0, "0", torch.zeros(3, dtype=torch.long), torch.zeros(2), torch.zeros(2, 1, dtype=torch.long),
                                    True, None])
def test_bad_targets_are_refused(target, no_launch):
    with pytest.raises(ValueError, match="target"):
        _call(target=target)


def test_cpu_inputs_are_refused(no_launch):
    with pytest.raises(ValueError, match="CUDA"):
        _call()


@pytest.mark.parametrize("where", ["mri_cnn", "pet_cnn.conv1", "mri_cnn.conv2", "pet_cnn.conv3", "mri_cnn.conv4"])
@pytest.mark.parametrize("kind", ["forward", "pre", "backward"])
def test_hooks_on_a_tower_or_its_blocks_are_refused(where, kind, no_launch):
    model = _model()
    mod = model.get_submodule(where)
    if kind == "pre":
        mod.register_forward_pre_hook(lambda m, a: None)
    elif kind == "forward":
        mod.register_forward_hook(lambda m, a, o: None)
    else:
        mod.register_full_backward_hook(lambda m, gi, go: None)
    with pytest.raises(ValueError, match="hook"):
        _call(model=model)


def test_refusals_leave_the_model_as_found(no_launch):
    model = _model()
    model.fc_cls[0].weight.requires_grad_(False)
    flags = [p.requires_grad for p in model.parameters()]
    for kw in ({"baselines": float("nan")}, {"mask": _mask(dtype=torch.float32)}, {}):
        with pytest.raises(ValueError):
            _call(model=model, **kw)
    assert flags == [p.requires_grad for p in model.parameters()]
    towers = [t for t in model.modules() if isinstance(t, M.sNet)]
    assert all(t._occ_out is None and t._lrp_keep is None for t in towers)
    assert not model.training


# ---------------------------------------------------------------------------------------------------------------
# the box planner on the occlusion grids
# ---------------------------------------------------------------------------------------------------------------
def _occlusion_cases():
    """Every (dims, window, stride) for which tests/test_occlusion_host.py builds an OccPlan, drawn the same way."""
    cases = [((16, 17, 18), (4, 5, 6), (4, 2, 7)), ((91, 109, 91), (16, 16, 16), (16, 16, 16))]
    for dims in [(91, 109, 91), (79, 95, 79), (128, 128, 79)]:
        rng = np.random.default_rng(dims[0] + dims[2])
        cases += [(dims, (16, 16, 16), (16, 16, 16)), (dims, (16, 16, 16), (8, 8, 8))]
        w = tuple(int(v) for v in rng.integers(3, 24, 3))
        cases.append((dims, w, tuple(int(v) for v in rng.integers(1, 20, 3))))
    for dims in [(16, 16, 16), (17, 16, 19), (23, 17, 29), (31, 33, 18), (16, 47, 21), (35, 38, 33)]:
        rng = np.random.default_rng(sum(dims))
        for _ in range(4):
            w = tuple(int(rng.integers(1, E + 1)) for E in dims)
            s = tuple(int(rng.integers(1, max(2, E // 2))) for E in dims)
            rng.choice([0.0, 1.5, -2.0])
            cases.append((dims, w, s))
        cases += [(dims, (1, 1, 1), (1, 1, 1)), (dims, dims, (1, 1, 1))]
    return cases


@pytest.mark.parametrize("dims,win,st", _occlusion_cases())
def test_box_planner_reproduces_the_occlusion_tables(dims, win, st):
    occ = TF.OccPlan(dims, win, st, _layers())
    starts = [TF.occ_positions(E, w, s) for E, w, s in zip(dims, win, st)]
    boxes = [((a, a + win[0]), (b, b + win[1]), (c, c + win[2])) for a in starts[0] for b in starts[1] for c in starts[2]]
    plan = TF.BoxPlan(dims, boxes, _layers(), range(len(boxes)))
    assert plan.n == occ.nwin and plan.crop == occ.crop and plan.full == occ.full
    for a, b in zip(plan.tab, occ.tab):
        assert a.dtype == b.dtype == np.int32 and a.shape == b.shape and np.array_equal(a, b)


# ---------------------------------------------------------------------------------------------------------------
# bounding boxes and extent classes
# ---------------------------------------------------------------------------------------------------------------
def _atlas(dims, cells, seed, B=1):
    """The synthetic parcellation plus the cases the planner must take: cells reach every volume face, background 0 (the
    corners) spans the whole volume's box, ids 1 and 2 merge into one non-convex region whose box holds other regions, id
    cells + 2 is one voxel, ids 2 and cells + 1 are absent; with B > 1 every later sample is the first one shifted."""
    m = make_atlas(dims, cells, seed, radius=0.55)
    m[m == 2] = 1
    m[0, 0, dims[0] // 2, dims[1] // 2, dims[2] // 2] = cells + 2
    if B > 1:
        m = torch.cat([m] + [torch.roll(m, shifts=(b, -b), dims=(2, 4)) for b in range(1, B)])
    return m


def test_bounding_boxes_against_numpy():
    dims = (23, 17, 29)
    m = _atlas(dims, 12, 3, B=2)
    F = int(m.max()) + 1
    boxes = TF.abl_boxes(m, F)
    assert boxes.shape == (F, 6)
    a = m.numpy()
    for f in range(F):
        where = np.nonzero((a == f).any(axis=(0, 1)))
        if len(where[0]) == 0:
            assert (boxes[f, 3:] <= boxes[f, :3]).all(), f
            continue
        assert boxes[f].tolist() == [int(w.min()) for w in where] + [int(w.max()) + 1 for w in where], f
    assert boxes[0].tolist() == [0, 0, 0, *dims]                           # background: the whole volume
    assert (boxes[12 + 2, 3:] - boxes[12 + 2, :3] == [2, 1, 2]).all()      # one voxel per sample, shifted by the roll
    faces = [(boxes[1:, a] == 0).any() and (boxes[1:, 3 + a] == E).any() for a, E in enumerate(dims)]
    assert all(faces)                                                      # cells touch every volume face


def test_extent_classes_follow_the_ladder(monkeypatch):
    dims = (91, 109, 91)
    m = _atlas(dims, 96, 0)
    F = int(m.max()) + 1
    boxes = TF.abl_boxes(m, F)
    classes = TF.abl_classes(boxes, dims)
    ids = sorted(f for _, c in classes for f in c)
    assert ids == [f for f in range(F) if boxes[f, 3] > boxes[f, 0]] and 2 not in ids and 97 not in ids and 98 in ids
    for key, c in classes:
        for f in c:
            ext = boxes[f, 3:] - boxes[f, :3]
            for e, k, E in zip(ext, key, dims):
                rungs = [r for r in TF.ABL_LADDER if r < E] + [E]
                assert k == min(r for r in rungs if r >= e)
    assert (tuple(dims), [0]) in [(k, c) for k, c in classes]


@pytest.mark.parametrize("B", [1, 2, 8])
def test_crop_extents_do_not_depend_on_the_pass_size(B):
    """The crop extent picks the conv plan, which decides the bf16 rounding: a feature's extents must be the same however the
    passes are cut.  Each class is planned as one unit, and a pass takes a slice of its boxes."""
    dims = (91, 109, 91)
    m = _atlas(dims, 96, 0)
    boxes = TF.abl_boxes(m, int(m.max()) + 1)
    seen = {}
    for ibs in (B, 4 * B, 32 * B, None):
        for _, ids in TF.abl_classes(boxes, dims):
            plan = TF.abl_plan(boxes, ids, dims, _layers())
            chunk = plan.n if ibs is None else max(1, ibs // B)
            for n0 in range(0, plan.n, chunk):
                for f in plan.ids[n0:n0 + chunk]:
                    assert seen.setdefault(int(f), plan.crop) == plan.crop
    # planning each pass on its own would not give this: at least one feature's extents would change
    _, ids = max(TF.abl_classes(boxes, dims), key=lambda kc: len(kc[1]))
    whole = TF.abl_plan(boxes, ids, dims, _layers()).crop
    assert any(TF.abl_plan(boxes, [f], dims, _layers()).crop != whole for f in ids)


# ---------------------------------------------------------------------------------------------------------------
# the box planner against a float64 restatement of the folded eval sNet
# ---------------------------------------------------------------------------------------------------------------
def _incremental(x, mask, acts, ps, plan, n, baseline):
    """Box n of the plan, composed as the kernels compose it: tmf_abl_input, then per layer the conv on the crop and
    tmf_occ_compose from the recomputed region and the base activation."""
    prev = None
    fid = int(plan.ids[n])
    for l in range(8):
        t = plan.tab[l][n]
        c0, lo, hi, src = t[:, 0], t[:, 1], t[:, 2], t[:, 3]
        size = plan.crop[l]
        if l == 0:
            sl = _sl(x, c0, size)
            a = x[sl].clone()
            inside = torch.zeros(a.shape[2:], dtype=torch.bool)
            inside[tuple(slice(int(lo[i] - c0[i]), int(hi[i] - c0[i])) for i in range(3))] = True
            sel = (mask[sl] == fid) & inside
            sel = sel.expand_as(a)
            b = baseline[sl].expand_as(a) if torch.is_tensor(baseline) else torch.full_like(a, baseline)
            a = torch.where(sel, b, a)
        else:
            a = acts[l][_sl(acts[l], c0, size)].clone()
            dst = tuple(slice(int(lo[i] - c0[i]), int(hi[i] - c0[i])) for i in range(3))
            srcs = tuple(slice(int(lo[i] - src[i]), int(hi[i] - src[i])) for i in range(3))
            assert all(s.stop <= e for s, e in zip(srcs, prev.shape[2:]))
            a[(slice(None), slice(None)) + dst] = prev[(slice(None), slice(None)) + srcs]
        if l == 7:
            return a
        prev = _layer(l, a, ps)


def _check_shape(dims, cells, B, picks_extra, seed):
    rng = np.random.default_rng(seed)
    ps = _params(seed)
    mask = _atlas(dims, cells, seed, B=B if B > 1 else 1)
    x = torch.from_numpy(rng.standard_normal((B, 1) + dims))
    per_voxel = torch.from_numpy(rng.standard_normal((1, 1) + dims)) * 0.5
    acts = _forward(x, ps)
    F = int(mask.max()) + 1
    boxes = TF.abl_boxes(mask, F)
    picks = {0, cells + 2, 1, *picks_extra}                               # background, one voxel, the merged region
    picks |= {int(f) for f in rng.choice(range(3, cells + 1), 2, replace=False)}
    checked = set()
    for _, ids in TF.abl_classes(boxes, dims):
        plan = TF.abl_plan(boxes, ids, dims, _layers())
        assert plan.full[-1] == tuple(acts[-1].shape[2:])
        for n, f in enumerate(plan.ids):
            if int(f) not in picks:
                continue
            checked.add(int(f))
            for baseline in (0.0, per_voxel):
                sel = (mask == int(f)).expand_as(x)
                xa = torch.where(sel, baseline.expand_as(x) if torch.is_tensor(baseline) else torch.zeros_like(x), x)
                want = _forward(xa, ps)[-1]
                got = _incremental(x, mask, acts, ps, plan, n, baseline)
                err = float((got - want).abs().max())
                assert err <= 1e-12 * max(float(want.abs().max()), 1.0), (dims, int(f), err)
    assert checked == {f for f in picks if boxes[f, 3] > boxes[f, 0]} and {0, 1, cells + 2} <= checked


@pytest.mark.parametrize("dims", [(91, 109, 91), (79, 95, 79)])
def test_box_planner_against_the_restatement_at_full_size(dims):
    _check_shape(dims, 96, 1, (), seed=dims[1])


@pytest.mark.parametrize("dims,B", [((16, 16, 16), 1), ((23, 17, 29), 2), ((31, 33, 18), 1), ((35, 38, 33), 2)])
def test_box_planner_against_the_restatement_on_small_odd_shapes(dims, B):
    _check_shape(dims, 9, B, range(12), seed=sum(dims))

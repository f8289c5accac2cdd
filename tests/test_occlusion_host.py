"""Host-side rules of interpret.occlusion (no GPU, no kernel launch): the argument refusals, the window placement and the
voxel-averaging rule of tmf_occ_map, and the crop planner (functional.OccPlan) against a float64 restatement of the folded
eval sNet: composing crops exactly as the planner's tables say must reproduce the tower output of every occluded volume
(DESIGN section 3.11)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from transmf_ad_b200 import _lib as L
from transmf_ad_b200 import functional as TF
from transmf_ad_b200.interpret import occlusion
from transmf_ad_b200.models import mymodel as M
from transmf_ad_b200.models.MiSePyNet import Mnet


@pytest.fixture
def no_launch(monkeypatch):
    def refuse(name, *args, **kw):
        raise AssertionError(f"{name} launched before the arguments were checked")
    monkeypatch.setattr(L, "call", refuse)


def _model():
    return M.model_CNN_ad(128).eval()


def _inputs(B=2, dims=(16, 16, 16)):
    return torch.zeros((B, 1) + dims), torch.zeros((B, 1) + dims)


@pytest.mark.parametrize("kw", [{"window": 0}, {"window": (4, 4)}, {"window": (4, 4, 0)}, {"window": 4.0},
                                {"window": True}, {"stride": 0}, {"stride": -1}, {"stride": (1, 2, 0)}, {"stride": "8"},
                                {"window": (17, 4, 4)}, {"window": (4, 4, 17)}])
def test_bad_windows_and_strides_are_refused(kw, no_launch):
    with pytest.raises(ValueError, match="window|stride"):
        occlusion(_model(), _inputs(), 0, **{"window": 4, "stride": 4, **kw})


@pytest.mark.parametrize("baseline", [float("nan"), float("inf"), -float("inf"), torch.tensor(0.0), torch.zeros(2), None,
                                      True, "0", np.zeros(3)])
def test_bad_baselines_are_refused(baseline, no_launch):
    with pytest.raises(ValueError, match="baseline"):
        occlusion(_model(), _inputs(), 0, window=4, stride=4, baseline=baseline)


@pytest.mark.parametrize("ibs", [0, -8, 8.0, False, "64"])
def test_bad_internal_batch_sizes_are_refused(ibs, no_launch):
    with pytest.raises(ValueError, match="internal_batch_size"):
        occlusion(_model(), _inputs(), 0, window=4, stride=4, internal_batch_size=ibs)


def test_training_mode_is_refused(no_launch):
    with pytest.raises(ValueError, match="eval"):
        occlusion(_model().train(), _inputs(), 0, window=4, stride=4)
    model = _model()
    model.fc_cls.train()
    with pytest.raises(ValueError, match="eval"):
        occlusion(model, _inputs(), 0, window=4, stride=4)


def test_a_model_without_towers_is_refused(no_launch):
    with pytest.raises(ValueError, match="sNet"):
        occlusion(Mnet().eval(), _inputs(), 0, window=4, stride=4)


@pytest.mark.parametrize("inputs", [torch.zeros(2, 1, 16, 16), (torch.zeros(2, 2, 16, 16, 16),) * 2, (), ("mri", "pet"),
                                    (torch.zeros(2, 1, 16, 16, 16),),
                                    (torch.zeros(2, 1, 16, 16, 16), torch.zeros(2, 1, 16, 16, 17)),
                                    (torch.zeros(2, 1, 16, 16, 16),) * 3])
def test_bad_inputs_are_refused(inputs, no_launch):
    with pytest.raises(ValueError, match="inputs"):
        occlusion(_model(), inputs, 0, window=4, stride=4)


@pytest.mark.parametrize("target", [2.0, "0", torch.zeros(3, dtype=torch.long), torch.zeros(2), torch.zeros(2, 1, dtype=torch.long),
                                    True, None])
def test_bad_targets_are_refused(target, no_launch):
    with pytest.raises(ValueError, match="target"):
        occlusion(_model(), _inputs(), target, window=4, stride=4)


def test_cpu_inputs_are_refused(no_launch):
    with pytest.raises(ValueError, match="CUDA"):
        occlusion(_model(), _inputs(), 0, window=4, stride=4)


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
        occlusion(model, _inputs(), 0, window=4, stride=4)


def test_refusals_leave_the_model_as_found(no_launch):
    model = _model()
    model.fc_cls[0].weight.requires_grad_(False)
    flags = [p.requires_grad for p in model.parameters()]
    for kw in ({"window": 0}, {"baseline": float("nan")}, {}):
        with pytest.raises(ValueError):
            occlusion(model, _inputs(), 0, **{"window": 4, "stride": 4, **kw})
    assert flags == [p.requires_grad for p in model.parameters()]
    towers = [t for t in model.modules() if isinstance(t, M.sNet)]
    assert all(t._occ_out is None and t._lrp_keep is None for t in towers)
    assert not model.training


# ---------------------------------------------------------------------------------------------------------------
# window placement and the voxel-averaging rule
# ---------------------------------------------------------------------------------------------------------------
AXES = [(16, 4, 4), (16, 4, 2), (16, 4, 6), (17, 5, 3), (91, 16, 16), (91, 16, 8), (109, 16, 16), (23, 7, 5), (9, 9, 1),
        (9, 9, 4), (10, 3, 7), (79, 8, 8)]


@pytest.mark.parametrize("E,w,s", AXES)
def test_window_placement_matches_captum(E, w, s):
    starts = TF.occ_positions(E, w, s)
    assert starts == [i * s for i in range((E - w) // s + 1)]
    assert starts[-1] + w <= E and starts[-1] + s + w > E


def _kernel_range(c, w, s, n):
    """The per-axis window range tmf_occ_map computes for index c."""
    return ((c - w + s) // s if c >= w else 0), min(n, c // s + 1)


@pytest.mark.parametrize("case", [((16, 17, 18), (4, 5, 6), (4, 2, 7)), ((91, 109, 91), (16, 16, 16), (16, 16, 16)),
                                  ((23, 19, 21), (7, 3, 5), (5, 3, 9)), ((9, 10, 11), (9, 3, 2), (1, 4, 3))])
def test_voxel_averaging_against_a_float64_restatement(case):
    dims, win, st = case
    plan = TF.OccPlan(dims, win, st, [(ks, pool) for _, _, ks, pool in TF.SNetSpec(32).layers]) if min(dims) >= 16 else None
    grid = tuple(len(TF.occ_positions(E, w, s)) for E, w, s in zip(dims, win, st))
    if plan is not None:
        assert plan.grid == grid and plan.nwin == int(np.prod(grid))
    rng = np.random.default_rng(sum(dims))
    scores = rng.standard_normal(grid)
    acc, cnt = np.zeros(dims), np.zeros(dims)
    for i in range(grid[0]):
        for j in range(grid[1]):
            for k in range(grid[2]):
                sl = tuple(slice(a * s, a * s + w) for a, s, w in zip((i, j, k), st, win))
                acc[sl] += scores[i, j, k]
                cnt[sl] += 1
    ref = np.where(cnt > 0, acc / np.maximum(cnt, 1), 0.0)
    assert (cnt == 0).any() or all((E - w) % s == 0 for E, w, s in zip(dims, win, st))
    rng_ax = [[_kernel_range(c, w, s, n) for c in range(E)] for E, w, s, n in zip(dims, win, st, grid)]
    got = np.zeros(dims)
    for x in range(dims[0]):
        for y in range(dims[1]):
            for z in range(dims[2]):
                (a0, a1), (b0, b1), (c0, c1) = rng_ax[0][x], rng_ax[1][y], rng_ax[2][z]
                n = max(a1 - a0, 0) * max(b1 - b0, 0) * max(c1 - c0, 0)
                assert n == cnt[x, y, z]
                got[x, y, z] = scores[a0:a1, b0:b1, c0:c1].sum() / n if n else 0.0
    assert np.allclose(got, ref, rtol=1e-13, atol=1e-13)


# ---------------------------------------------------------------------------------------------------------------
# the planner against a float64 restatement of the folded eval sNet
# ---------------------------------------------------------------------------------------------------------------
CH = [1, 3, 3, 4, 4, 5, 6, 3]                   # few channels: the geometry does not depend on them
SLOPE = 0.01


def _layers():
    return [(ks, pool) for _, _, ks, pool in TF.SNetSpec(32).layers]


def _params(seed):
    g = torch.Generator().manual_seed(seed)
    ps = []
    for l, (ks, _) in enumerate(_layers()):
        w = torch.randn(CH[l + 1], CH[l], ks, ks, ks, generator=g).double() / (CH[l] * ks ** 3) ** 0.5
        ps.append((w, torch.randn(CH[l + 1], generator=g).double() * 0.1))
    return ps


def _layer(l, a, ps):
    ks, pool = _layers()[l]
    z = F.leaky_relu(F.conv3d(a, ps[l][0], ps[l][1], padding=ks // 2), SLOPE)
    if pool == L.POOL_MAX:
        return F.max_pool3d(z, 2)
    return F.avg_pool3d(z, 2) if pool == L.POOL_AVG else z


def _forward(x, ps):
    acts = [x]
    for l in range(7):
        acts.append(_layer(l, acts[-1], ps))
    return acts                                  # layer inputs 0 .. 6, then the tower output


def _sl(t, origin, size):
    return (slice(None), slice(None)) + tuple(slice(int(o), int(o) + n) for o, n in zip(origin, size))


def _incremental(x, acts, ps, plan, n, baseline):
    """Window n of the plan, composed as the kernels compose it: tmf_occ_input, then per layer the conv on the crop and
    tmf_occ_compose from the recomputed region and the base activation."""
    prev = None
    for l in range(8):
        t = plan.tab[l][n]                       # [axis][origin, lo, hi, previous output origin]
        c0, lo, hi, src = t[:, 0], t[:, 1], t[:, 2], t[:, 3]
        size = plan.crop[l]
        if l == 0:
            a = x[_sl(x, c0, size)].clone()
            inside = tuple(slice(int(lo[i] - c0[i]), int(hi[i] - c0[i])) for i in range(3))
            a[(slice(None), slice(None)) + inside] = baseline
        else:
            assert (lo >= c0).all() and (hi <= c0 + np.array(size)).all()
            a = acts[l][_sl(acts[l], c0, size)].clone()
            dst = tuple(slice(int(lo[i] - c0[i]), int(hi[i] - c0[i])) for i in range(3))
            srcs = tuple(slice(int(lo[i] - src[i]), int(hi[i] - src[i])) for i in range(3))
            assert all(s.stop <= e for s, e in zip(srcs, prev.shape[2:]))
            a[(slice(None), slice(None)) + dst] = prev[(slice(None), slice(None)) + srcs]
        if l == 7:
            return a
        prev = _layer(l, a, ps)


def _check_shape(dims, cases, seed):
    rng = np.random.default_rng(seed)
    ps = _params(seed)
    x = torch.from_numpy(rng.standard_normal((1, 1) + dims))
    x[:, :, :dims[0] // 3] = 0                                       # an all-zero slab: null windows with baseline 0
    acts = _forward(x, ps)
    for win, st, baseline in cases:
        plan = TF.OccPlan(dims, win, st, _layers())
        assert plan.full[-1] == tuple(acts[-1].shape[2:])
        for l in range(7):
            assert all(c <= e for c, e in zip(plan.crop[l], plan.full[l]))
        picks = sorted({0, plan.nwin - 1, *rng.integers(0, plan.nwin, 2).tolist()})
        for n in picks:
            i, j, k = np.unravel_index(n, plan.grid)
            xo = x.clone()
            xo[_sl(xo, (i * st[0], j * st[1], k * st[2]), win)] = baseline
            want = _forward(xo, ps)[-1]
            got = _incremental(x, acts, ps, plan, n, baseline)
            scale = float(want.abs().max())
            err = float((got - want).abs().max())
            assert err <= 1e-12 * max(scale, 1.0), (dims, win, st, n, err)


@pytest.mark.parametrize("dims", [(91, 109, 91), (79, 95, 79), (128, 128, 79)])
def test_planner_against_the_restatement_at_full_size(dims):
    rng = np.random.default_rng(dims[0] + dims[2])
    cases = [((16, 16, 16), (16, 16, 16), 0.0), ((16, 16, 16), (8, 8, 8), -0.5)]
    w = tuple(int(v) for v in rng.integers(3, 24, 3))
    cases.append((w, tuple(int(v) for v in rng.integers(1, 20, 3)), 0.25))
    _check_shape(dims, cases, seed=dims[1])


@pytest.mark.parametrize("dims", [(16, 16, 16), (17, 16, 19), (23, 17, 29), (31, 33, 18), (16, 47, 21), (35, 38, 33)])
def test_planner_against_the_restatement_on_small_odd_shapes(dims):
    rng = np.random.default_rng(sum(dims))
    cases = []
    for _ in range(4):
        w = tuple(int(rng.integers(1, E + 1)) for E in dims)
        s = tuple(int(rng.integers(1, max(2, E // 2))) for E in dims)
        cases.append((w, s, float(rng.choice([0.0, 1.5, -2.0]))))
    cases.append(((1, 1, 1), (1, 1, 1), 3.0))
    cases.append((dims, (1, 1, 1), 0.0))                              # one window over the whole volume
    _check_shape(dims, cases, seed=len(dims) + dims[0])

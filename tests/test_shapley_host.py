"""Host-side rules of interpret.shapley_sampling (no GPU, no kernel launch): the argument refusals, the permutations, the
pass schedule, and a float64 restatement of the chains with write-back: composing every step's crops from a chain's own
state, as the planner's tables say, and writing the changed region back must reproduce the tower output of every composite
volume along the chain (DESIGN section 3.13)."""
import numpy as np
import pytest
import torch

from tests.test_ablation_host import _atlas, _inputs, _mask
from tests.test_ablation_host import _model as _abl_model
from tests.test_occlusion_host import _forward, _layer, _layers, _params, _sl
from transmf_ad_b200 import _lib as L
from transmf_ad_b200 import functional as TF
from transmf_ad_b200.interpret import shapley_sampling
from transmf_ad_b200.models import mymodel as M
from transmf_ad_b200.models.MiSePyNet import Mnet
from transmf_ad_b200.synthetic import make_atlas


@pytest.fixture
def no_launch(monkeypatch):
    def refuse(name, *args, **kw):
        raise AssertionError(f"{name} launched before the arguments were checked")
    monkeypatch.setattr(L, "call", refuse)


DIMS = (16, 16, 16)


def _call(model=None, inputs=None, target=0, mask=None, **kw):
    return shapley_sampling(_abl_model() if model is None else model, _inputs() if inputs is None else inputs, target,
                            _mask() if mask is None else mask, **kw)


@pytest.mark.parametrize("n", [0, -1, 2.0, True, "25", None])
def test_bad_sample_counts_are_refused(n, no_launch):
    with pytest.raises(ValueError, match="n_samples"):
        _call(n_samples=n)


@pytest.mark.parametrize("mask", [_mask(dtype=torch.float32), _mask(dtype=torch.bool), _mask(B=3), _mask(dims=(16, 16, 17)),
                                  torch.zeros((1, 16, 16, 16), dtype=torch.long), np.zeros((1, 1) + DIMS), 0])
def test_bad_masks_are_refused(mask, no_launch):
    with pytest.raises(ValueError, match="feature_mask"):
        _call(mask=mask)


@pytest.mark.parametrize("baselines", [float("nan"), None, True, torch.tensor(0.0), (0.0,), (0.0, 0.0, 0.0),
                                       (0.0, torch.zeros((3, 1) + DIMS)), (0.0, torch.zeros((2, 1) + DIMS, dtype=torch.float64))])
def test_bad_baselines_are_refused(baselines, no_launch):
    with pytest.raises(ValueError, match="baseline"):
        _call(baselines=baselines)


@pytest.mark.parametrize("kw,what", [({"internal_batch_size": 0}, "internal_batch_size"),
                                     ({"internal_batch_size": 8.0}, "internal_batch_size"), ({"joint": 1}, "joint"),
                                     ({"joint": None}, "joint"), ({"target": 2.0}, "target"),
                                     ({"target": torch.zeros(3, dtype=torch.long)}, "target"),
                                     ({"inputs": (torch.zeros(2, 1, 16, 16, 16),)}, "inputs"), ({}, "CUDA")])
def test_bad_arguments_are_refused(kw, what, no_launch):
    with pytest.raises(ValueError, match=what):
        _call(**kw)


def test_training_mode_and_models_without_towers_are_refused(no_launch):
    with pytest.raises(ValueError, match="eval"):
        _call(model=_abl_model().train())
    with pytest.raises(ValueError, match="sNet"):
        _call(model=Mnet().eval())


@pytest.mark.parametrize("where", ["mri_cnn", "pet_cnn.conv1", "mri_cnn.conv4"])
@pytest.mark.parametrize("kind", ["forward", "pre", "backward"])
def test_hooks_on_a_tower_or_its_blocks_are_refused(where, kind, no_launch):
    model = _abl_model()
    mod = model.get_submodule(where)
    if kind == "pre":
        mod.register_forward_pre_hook(lambda m, a: None)
    elif kind == "forward":
        mod.register_forward_hook(lambda m, a, o: None)
    else:
        mod.register_full_backward_hook(lambda m, gi, go: None)
    with pytest.raises(ValueError, match="hook"):
        _call(model=model)


def test_refusals_leave_the_model_and_the_generator_as_found(no_launch):
    model = _abl_model()
    model.fc_cls[0].weight.requires_grad_(False)
    flags = [p.requires_grad for p in model.parameters()]
    torch.manual_seed(5)
    state = torch.get_rng_state()
    for kw in ({"n_samples": 0}, {"baselines": float("nan")}, {"mask": _mask(dtype=torch.float32)}, {}):
        with pytest.raises(ValueError):
            _call(model=model, **kw)
    assert flags == [p.requires_grad for p in model.parameters()]
    towers = [t for t in model.modules() if isinstance(t, M.sNet)]
    assert all(t._occ_out is None and t._lrp_keep is None for t in towers)
    assert not model.training
    assert torch.equal(state, torch.get_rng_state())            # no permutation is drawn before the checks pass


# ---------------------------------------------------------------------------------------------------------------
# permutations and the pass schedule
# ---------------------------------------------------------------------------------------------------------------
def test_permutations_are_reproducible_from_the_seed():
    ids = np.array([0, 1, 3, 4, 7, 11, 12], dtype=np.int64)
    torch.manual_seed(3)
    a = TF.shap_permutations(ids, 6)
    torch.manual_seed(3)
    b = TF.shap_permutations(ids, 6)
    torch.manual_seed(3)
    want = torch.stack([torch.as_tensor(ids)[torch.randperm(len(ids))] for _ in range(6)])   # captum's draw
    assert a.dtype == torch.int64 and a.shape == (6, 7) and torch.equal(a, b) and torch.equal(a, want)
    assert all(sorted(r.tolist()) == ids.tolist() for r in a)
    assert not torch.equal(a, TF.shap_permutations(ids, 6))


def _bench_atlas():
    dims = (91, 109, 91)
    m = make_atlas(dims, 96, seed=0)
    boxes = TF.abl_boxes(m, int(m.max()) + 1)
    classes = TF.abl_classes(boxes, dims)
    return {f: c for c, (_, ids) in enumerate(classes) for f in ids}, len(classes)


@pytest.mark.parametrize("cap", [1, 3, 8, 10 ** 9])
@pytest.mark.parametrize("n", [1, 10, 25])
def test_schedule_properties(n, cap):
    cls_of, nc = _bench_atlas()
    torch.manual_seed(0)
    perms = TF.shap_permutations(np.array(sorted(cls_of)), n).numpy()
    passes = TF.shap_schedule(perms, cls_of, [cap] * nc)
    seen = {}
    for c, steps in passes:
        ps = [p for p, _ in steps]
        assert 1 <= len(steps) <= cap and len(set(ps)) == len(ps) and ps == sorted(ps)
        for p, k in steps:
            assert cls_of[int(perms[p, k])] == c
            assert seen.get(p, -1) == k - 1                      # each chain's steps in order
            seen[p] = k
    assert sorted(seen) == list(range(n)) and all(k == perms.shape[1] - 1 for k in seen.values())
    assert sum(len(s) for _, s in passes) == perms.size


@pytest.mark.parametrize("n,lock,greedy", [(10, 457, 409), (25, 647, 437)])
def test_greedy_schedule_beats_lock_step_on_the_bench_atlas(n, lock, greedy):
    cls_of, nc = _bench_atlas()
    torch.manual_seed(0)
    perms = TF.shap_permutations(np.array(sorted(cls_of)), n).numpy()
    assert sum(len({cls_of[int(f)] for f in perms[:, k]}) for k in range(perms.shape[1])) == lock
    assert len(TF.shap_schedule(perms, cls_of, [10 ** 9] * nc)) == greedy


# ---------------------------------------------------------------------------------------------------------------
# the chains with write-back against a float64 restatement of the folded eval sNet
# ---------------------------------------------------------------------------------------------------------------
def _composite(x, mask, baseline, rank, k):
    """The volume after step k of a chain: x where the voxel's region has rank <= k, else the baseline."""
    keep = (rank[mask.long()] <= k).expand_as(x)
    b = baseline.expand_as(x) if torch.is_tensor(baseline) else torch.full_like(x, baseline)
    return torch.where(keep, x, b)


def _step(x, mask, baseline, rank, k, state, plan, n, ps):
    """Step k of a chain adding box n of the plan, as the kernels run it: tmf_shap_input, then per layer the conv on the crop
    and tmf_shap_compose from the recomputed region and the chain state, writing that region back into the state."""
    prev = None
    for l in range(8):
        t = plan.tab[l][n]
        c0, lo, hi, src = t[:, 0], t[:, 1], t[:, 2], t[:, 3]
        size = plan.crop[l]
        if l == 0:
            a = _composite(x, mask, baseline, rank, k)[_sl(x, c0, size)]
        else:
            a = state[l][_sl(state[l], c0, size)].clone()
            dst = tuple(slice(int(lo[i] - c0[i]), int(hi[i] - c0[i])) for i in range(3))
            srcs = tuple(slice(int(lo[i] - src[i]), int(hi[i] - src[i])) for i in range(3))
            new = prev[(slice(None), slice(None)) + srcs]
            a[(slice(None), slice(None)) + dst] = new
            state[l][(slice(None), slice(None)) + tuple(slice(int(lo[i]), int(hi[i])) for i in range(3))] = new
        if l == 7:
            return a
        prev = _layer(l, a, ps)


def _chains(dims, cells, B, mask_b, n_chains, steps, seed, forced=()):
    """Chains of random permutations (the first entries ``forced``) with write-back, every step's composed tower output
    against the float64 forward of the composite volume; returns the largest relative error and the worst telescoping
    defect sum_j phi_j - (f(x) - f(start)) of a linear objective on the tower output."""
    rng = np.random.default_rng(seed)
    ps = _params(seed)
    mask = _atlas(dims, cells, seed, B=mask_b)
    x = torch.from_numpy(rng.standard_normal((B, 1) + dims))
    per_voxel = torch.from_numpy(rng.standard_normal((1, 1) + dims)) * 0.5
    F = int(mask.max()) + 1
    boxes = TF.abl_boxes(mask, F)
    plans = [TF.abl_plan(boxes, ids, dims, _layers()) for _, ids in TF.abl_classes(boxes, dims)]
    where = {int(f): (plan, n) for plan in plans for n, f in enumerate(plan.ids)}
    players = sorted(where)
    out_x = _forward(x, ps)[-1]
    head = torch.from_numpy(rng.standard_normal(out_x.shape[1:]))

    def f(out):
        return (out * head).sum(dim=(1, 2, 3, 4))

    worst, tele = 0.0, 0.0
    for baseline in (0.0, per_voxel):
        start = _forward(baseline.expand_as(x).clone() if torch.is_tensor(baseline) else torch.full_like(x, baseline), ps)
        phi = torch.zeros((B, F), dtype=torch.float64)
        for c in range(n_chains):
            rest = [p for p in rng.permutation(players).tolist() if p not in forced]
            perm = list(forced) + rest
            rank = torch.full((F,), F, dtype=torch.long)
            rank[perm] = torch.arange(len(perm))
            state = {l: start[l].clone() for l in range(1, 8)}
            f_prev = f(start[-1])
            for k in range(min(steps, len(perm))):
                plan, n = where[perm[k]]
                got = _step(x, mask, baseline, rank, k, state, plan, n, ps)
                want = _forward(_composite(x, mask, baseline, rank, k), ps)[-1]
                assert torch.equal(got, state[7])                    # the tower output state is the composed output
                worst = max(worst, float((got - want).abs().max()) / max(float(want.abs().max()), 1.0))
                f_new = f(got)
                phi[:, perm[k]] += f_new - f_prev
                f_prev = f_new
        if steps >= len(players):
            tele = max(tele, float((phi.sum(1) / n_chains - (f(out_x) - f(start[-1]))).abs().max())
                       / max(float(f(out_x).abs().max()), 1.0))
    return worst, tele, players


def test_chains_against_the_restatement_at_full_size():
    dims = (91, 109, 91)
    worst, _, players = _chains(dims, 96, 1, 1, 2, 3, seed=5, forced=(0, 96 + 2))   # background and the one-voxel region
    assert {0, 98} <= set(players)
    assert worst <= 1e-12, worst


@pytest.mark.parametrize("dims,B,mask_b", [((16, 16, 16), 1, 1), ((23, 17, 29), 2, 2), ((31, 33, 18), 2, 1),
                                           ((35, 38, 33), 2, 2)])
def test_whole_chains_against_the_restatement_on_small_odd_shapes(dims, B, mask_b):
    worst, tele, players = _chains(dims, 9, B, mask_b, 3, 10 ** 9, seed=sum(dims))
    assert len(players) >= 9
    assert worst <= 1e-12, worst
    assert tele <= 1e-12, tele                                          # the telescoping identity

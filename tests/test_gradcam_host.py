"""Host-side rules of the segmented sNet run and of grad_cam (no GPU): which block outputs the hooks expose, how the
towers are split, what is refused or warned about, and grad_cam's argument checks."""
import warnings

import pytest
import torch

from transmf_ad_b200.interpret import grad_cam
from transmf_ad_b200.models import mymodel as M
from transmf_ad_b200.models.networks import _tapped_boundaries, sNet, segment_plan


def test_segment_plan():
    assert segment_plan(set()) == [(0, 7)]
    assert segment_plan({3}) == [(0, 7)]                       # the tower output needs no split
    assert segment_plan({2}) == [(0, 5), (5, 7)]
    assert segment_plan({0, 1, 2, 3}) == [(0, 1), (1, 3), (3, 5), (5, 7)]


@pytest.mark.parametrize("block,taps", [("conv1", {0}), ("conv2", {0, 1}), ("conv3", {1, 2}), ("conv4", {2, 3})])
@pytest.mark.parametrize("kind", ["forward", "pre"])
def test_a_block_hook_taps_its_input_and_output(block, taps, kind):
    net = sNet(128)
    blk = getattr(net, block)
    if kind == "forward":
        blk.register_forward_hook(lambda m, i, o: None)
    else:
        blk.register_forward_pre_hook(lambda m, i: None)
    assert _tapped_boundaries([net]) == taps


def test_no_hooks_no_taps_and_tower_hooks_need_no_split():
    a, b = sNet(128), sNet(128)
    assert _tapped_boundaries([a, b]) == set()
    a.register_forward_hook(lambda m, i, o: None)
    b.register_forward_pre_hook(lambda m, i: None)
    assert _tapped_boundaries([a, b]) == set()


def test_taps_are_the_union_over_both_towers():
    a, b = sNet(128), sNet(128)
    a.conv1.register_forward_hook(lambda m, i, o: None)
    b.conv4.register_forward_hook(lambda m, i, o: None)
    assert _tapped_boundaries([a, b]) == {0, 2, 3}


@pytest.mark.parametrize("child", [0, 1, 2, 3])
def test_hook_inside_a_block_warns_once_per_module(child):
    net = sNet(128)
    net.conv2[child].register_forward_hook(lambda m, i, o: None)
    with warnings.catch_warnings(record=True) as rec:
        warnings.simplefilter("always")
        assert _tapped_boundaries([net]) == set()
        _tapped_boundaries([net])
    msgs = [str(w.message) for w in rec if issubclass(w.category, UserWarning)]
    assert len(msgs) == 1 and "conv1, conv2, conv3, conv4" in msgs[0] and "sNet.conv2" in msgs[0]


@pytest.mark.parametrize("register", ["register_full_backward_hook", "register_full_backward_pre_hook"])
def test_backward_hook_on_a_block_is_refused(register):
    net = sNet(128)
    getattr(net.conv3, register)(lambda *a: None)
    with pytest.raises(NotImplementedError, match="register_hook|autograd.grad"):
        _tapped_boundaries([net])


def test_replacing_pre_hook_on_a_block_is_refused():
    net = sNet(128)
    net.conv1.register_forward_pre_hook(lambda m, args: (args[0] * 2,))
    with pytest.raises(NotImplementedError, match="only observe"):
        net(torch.zeros(1, 1, 8, 8, 8))                       # refused before anything is launched


def _small_model_ad():
    return M.model_ad(dim=128, depth=1, heads=4, dim_head=32, mlp_dim=512, dropout=0.0)


@pytest.mark.parametrize("kw,match", [(dict(layer="conv5"), "layer"), (dict(layer="conv3.0"), "layer")])
def test_grad_cam_rejects_bad_layer(kw, match):
    x = torch.zeros(2, 1, 8, 8, 8)
    with pytest.raises(ValueError, match=match):
        grad_cam(_small_model_ad(), (x, x), 0, **kw)


@pytest.mark.parametrize("target", [1.5, torch.tensor([0.0, 1.0]), torch.tensor([[0, 1]]), torch.tensor([0, 1, 1]), "a"])
def test_grad_cam_rejects_bad_target(target):
    from transmf_ad_b200.interpret import _target_index
    with pytest.raises(ValueError, match="target"):
        _target_index(target, 2, "cpu")


def test_grad_cam_target_forms():
    from transmf_ad_b200.interpret import _target_index
    assert _target_index(1, 3, "cpu").tolist() == [1, 1, 1]
    assert _target_index(torch.tensor([0, 1, 0]), 3, "cpu").tolist() == [0, 1, 0]
    assert _target_index(torch.tensor(1), 3, "cpu").tolist() == [1, 1, 1]


def test_grad_cam_rejects_models_without_towers_and_bad_inputs():
    with pytest.raises(ValueError, match="no sNet"):
        grad_cam(torch.nn.Linear(2, 2), (torch.zeros(1, 1, 4, 4, 4),), 0)
    with pytest.raises(ValueError, match="volumes"):
        grad_cam(_small_model_ad(), (torch.zeros(2, 8, 8),), 0)


def test_grad_cam_restores_flags_on_error():
    model = M.model_single(128)
    model.fc[0].weight.requires_grad_(False)
    flags = {k: p.requires_grad for k, p in model.named_parameters()}
    with pytest.raises(Exception):
        grad_cam(model, torch.zeros(1, 1, 8, 8, 8), 0)        # no GPU here: the forward fails
    assert flags == {k: p.requires_grad for k, p in model.named_parameters()}
    assert model.cnn._cam_tap is None and model.cnn._cam_act is None

"""Host-side rules of interpret.lrp (no GPU): argument checks, the refusal of training mode, and which block-1
implementation tmf_lrp_conv1 takes."""
import pytest
import torch

from transmf_ad_b200 import _lib as L
from transmf_ad_b200 import functional as TF
from transmf_ad_b200.interpret import lrp
from transmf_ad_b200.models import mymodel as M


def _model():
    return M.model_CNN_ad(128).eval()


def _inputs(B=2):
    return torch.zeros(B, 1, 8, 8, 8), torch.zeros(B, 1, 8, 8, 8)


@pytest.mark.parametrize("rule", ["z+", "alpha1beta0", "zB", "", None, "EPSILON"])
def test_unknown_rules_are_refused(rule):
    with pytest.raises(ValueError, match="rule"):
        lrp(_model(), _inputs(), 0, rule=rule)


@pytest.mark.parametrize("eps", [-1e-6, float("nan"), float("inf"), "0.1", True, None])
def test_bad_eps_is_refused(eps):
    with pytest.raises(ValueError, match="eps"):
        lrp(_model(), _inputs(), 0, eps=eps)


def test_training_mode_is_refused():
    with pytest.raises(ValueError, match="eval"):
        lrp(_model().train(), _inputs(), 0)


def test_a_model_without_towers_is_refused():
    with pytest.raises(ValueError, match="sNet"):
        lrp(torch.nn.Linear(4, 2).eval(), _inputs(), 0)


@pytest.mark.parametrize("inputs", [torch.zeros(2, 1, 8, 8), (torch.zeros(2, 2, 8, 8, 8),), (), ("mri",)])
def test_bad_inputs_are_refused(inputs):
    with pytest.raises(ValueError, match="inputs"):
        lrp(_model(), inputs, 0)


@pytest.mark.parametrize("target", [1.0, torch.tensor([0.0, 1.0]), torch.tensor([0, 1, 1]), torch.tensor([True, False]),
                                    "1", None])
def test_bad_targets_are_refused(target):
    with pytest.raises(ValueError, match="target"):
        lrp(_model(), _inputs(), target)


def test_refusals_leave_the_model_as_found():
    model = _model()
    model.fc_cls[0].weight.requires_grad_(False) if hasattr(model, "fc_cls") else None
    flags = [p.requires_grad for p in model.parameters()]
    with pytest.raises(ValueError):
        lrp(model, _inputs(), 2.5)
    assert flags == [p.requires_grad for p in model.parameters()]
    assert all(t._lrp_keep is None for t in model.modules() if isinstance(t, M.sNet))


@pytest.mark.parametrize("W,cout,env,expect", [
    (128, 32, "auto", L.CONV_UMMA), (91, 32, "auto", L.CONV_UMMA), (129, 32, "auto", L.CONV_DIRECT),
    (91, 16, "auto", L.CONV_DIRECT), (91, 32, "direct", L.CONV_DIRECT), (91, 32, "umma", L.CONV_UMMA)])
def test_block1_implementation_choice(W, cout, env, expect, monkeypatch):
    monkeypatch.setenv("TMF_CONV_IMPL", env)
    monkeypatch.delenv("TMF_DISABLE_UMMA", raising=False)
    assert TF.lrp_conv1_impl(8, 91, 109, W, cout, ng=2) == expect

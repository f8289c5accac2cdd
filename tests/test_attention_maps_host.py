"""Host-side rules of the attention-probability hooks and of cross_attention (no GPU): which encoders run tapped, what is
refused or warned about, and cross_attention's argument checks."""
import warnings

import pytest
import torch

from transmf_ad_b200 import functional as TF
from transmf_ad_b200.interpret import cross_attention
from transmf_ad_b200.models import mymodel as M
from transmf_ad_b200.models.networks import Transformer, _attend_hooked, _fire_attend_hooks


def _enc(dim=128, heads=4, dim_head=32):
    return Transformer(dim, 1, heads, dim_head, 4 * dim)


def test_an_encoder_is_tapped_only_when_attend_has_forward_hooks():
    enc = _enc()
    att = enc.layers[0][0].fn.attend
    assert not _attend_hooked(att)
    h = att.register_forward_hook(lambda m, a, o: None)
    assert _attend_hooked(att)
    h.remove()
    assert not _attend_hooked(att)
    att.register_forward_pre_hook(lambda m, a: None)
    assert _attend_hooked(att)


@pytest.mark.parametrize("register", ["register_full_backward_hook", "register_full_backward_pre_hook"])
def test_backward_hooks_on_attend_are_refused(register):
    att = _enc().layers[0][0].fn.attend
    getattr(att, register)(lambda *a: None)
    with pytest.raises(NotImplementedError, match="register_hook|autograd.grad"):
        _attend_hooked(att)


def _fire(att):
    dots, attn = torch.zeros(1, 2, 3, 4), torch.full((1, 2, 3, 4), 0.25)
    _fire_attend_hooks(att, dots, attn)
    return dots, attn


def test_hooks_receive_what_module_call_would_give():
    att = _enc().layers[0][0].fn.attend
    seen = []
    att.register_forward_pre_hook(lambda m, args: seen.append(("pre", m, len(args))))
    att.register_forward_pre_hook(lambda m, args, kw: seen.append(("pre_kw", kw)), with_kwargs=True)
    att.register_forward_hook(lambda m, args, out: seen.append(("fwd", args[0].shape, out.shape)))
    att.register_forward_hook(lambda m, args, kw, out: seen.append(("fwd_kw", kw)), with_kwargs=True)
    _fire(att)
    assert seen == [("pre", att, 1), ("pre_kw", {}), ("fwd", (1, 2, 3, 4), (1, 2, 3, 4)), ("fwd_kw", {})]


@pytest.mark.parametrize("kind,exc", [("fwd_replace", NotImplementedError), ("pre_replace", NotImplementedError),
                                      ("fwd_inplace", RuntimeError), ("pre_inplace", RuntimeError)])
def test_replacing_or_modifying_hooks_are_refused(kind, exc):
    att = _enc().layers[0][0].fn.attend
    if kind == "fwd_replace":
        att.register_forward_hook(lambda m, a, o: o * 2)
    elif kind == "pre_replace":
        att.register_forward_pre_hook(lambda m, a: (a[0] + 1,))
    elif kind == "fwd_inplace":
        att.register_forward_hook(lambda m, a, o: (o.mul_(2), None)[1])
    else:
        att.register_forward_pre_hook(lambda m, a: (a[0].add_(1), None)[1])
    with pytest.raises(exc):
        _fire(att)


def _warned(fn):
    with warnings.catch_warnings(record=True) as rec:
        warnings.simplefilter("always")
        fn()
        fn()
    return [str(w.message) for w in rec if issubclass(w.category, UserWarning)]


@pytest.mark.parametrize("path", ["fused", "unfused"])
@pytest.mark.parametrize("child", ["to_q", "to_kv", "to_out.0", "to_out.1", "norm", "ff.net.0", "ff.net.1", "ff.net.2",
                                   "final_norm"])
def test_hooks_on_modules_that_never_run_warn_once(child, path):
    enc = _enc()
    pre_attn, pre_ff = enc.layers[0]
    mod = {"to_q": pre_attn.fn.to_q, "to_kv": pre_attn.fn.to_kv, "to_out.0": pre_attn.fn.to_out[0],
           "to_out.1": pre_attn.fn.to_out[1], "norm": pre_attn.norm, "ff.net.0": pre_ff.fn.net[0],
           "ff.net.1": pre_ff.fn.net[1], "ff.net.2": pre_ff.fn.net[2], "final_norm": enc.norm}[child]
    mod.register_forward_hook(lambda *a: None)
    msgs = _warned(lambda: enc._dead_hook_scan(path == "fused"))
    assert len(msgs) == 1 and "Attention.attend" in msgs[0]


@pytest.mark.parametrize("which", ["prenorm", "attention", "feedforward"])
def test_wrapper_modules_warn_on_the_fused_path_only(which):
    enc = _enc()
    pre_attn, pre_ff = enc.layers[0]
    mod = {"prenorm": pre_attn, "attention": pre_attn.fn, "feedforward": pre_ff.fn}[which]
    mod.register_forward_hook(lambda *a: None)
    assert _warned(lambda: enc._dead_hook_scan(False)) == []
    assert len(_warned(lambda: enc._dead_hook_scan(True))) == 1


def test_active_dropout_runs_on_the_unfused_path():
    enc = Transformer(64, 1, 4, 16, 256, dropout=0.1).train()
    enc.layers[0][1].fn.net[2].register_forward_hook(lambda *a: None)
    assert _warned(lambda: enc._dead_hook_scan(False)) == []
    enc.eval()
    assert len(_warned(lambda: enc._dead_hook_scan(False))) == 1


def test_attend_hooks_do_not_warn():
    enc = _enc()
    enc.layers[0][0].fn.attend.register_forward_hook(lambda *a: None)
    assert _warned(lambda: enc._dead_hook_scan(True)) == []


def test_tap_refuses_a_gradient_that_is_not_its_own():
    tap = TF.AttnTap()
    tap.check(None)                                        # attn received no gradient: nothing to check
    tap.dattn = torch.zeros(2)
    tap.version = tap.dattn._version
    tap.check(tap.dattn)                                   # its own, unmodified
    tap.dattn = torch.zeros(2)
    tap.version = tap.dattn._version
    with pytest.raises(NotImplementedError, match="only be observed"):
        tap.check(torch.zeros(2))
    own = tap.dattn
    own.add_(1)
    tap.dattn = own
    with pytest.raises(NotImplementedError, match="only be observed"):
        tap.check(own)


def _model_ad():
    return M.model_ad(dim=128, depth=1, heads=4, dim_head=32, mlp_dim=512, dropout=0.0)


def test_cross_attention_rejects_models_without_a_fusion_transformer():
    x = torch.zeros(1, 1, 8, 8, 8)
    for model in (M.model_CNN(128), M.model_CNN_ad(128), M.model_single(128), torch.nn.Linear(2, 2)):
        with pytest.raises(ValueError, match="no fusion transformer"):
            cross_attention(model, (x, x))


def test_cross_attention_rejects_bad_inputs_and_targets():
    model = _model_ad()
    with pytest.raises(ValueError, match="inputs"):
        cross_attention(model, torch.zeros(1, 1, 8, 8, 8))
    with pytest.raises(ValueError, match="inputs"):
        cross_attention(model, (torch.zeros(2, 8, 8), torch.zeros(2, 8, 8)))
    from transmf_ad_b200.interpret import _target_index
    with pytest.raises(ValueError, match="cross_attention: target"):
        _target_index(1.5, 2, "cpu", "cross_attention")


@pytest.mark.parametrize("target", [None, 1])
def test_cross_attention_restores_flags_and_removes_its_hooks_on_error(target):
    model = _model_ad()
    model.fc_cls[0].weight.requires_grad_(False)
    flags = {k: p.requires_grad for k, p in model.named_parameters()}
    x = torch.zeros(1, 1, 16, 16, 16)
    with pytest.raises(Exception):
        cross_attention(model, (x, x), target)               # no GPU here: the forward fails
    assert flags == {k: p.requires_grad for k, p in model.named_parameters()}
    assert not any(m._forward_hooks or m._forward_pre_hooks for m in model.modules())

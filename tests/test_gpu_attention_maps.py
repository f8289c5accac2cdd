"""The fusion transformer's attention probabilities exposed to module hooks on ``Attention.attend`` and the cross-modal
attention maps built on them (csrc/attention_mma.cu ``tmf_attn_scores`` / ``tmf_attn_relevance``, csrc/gradcam.cu
``tmf_map_resample``, ``transmf_ad_b200.interpret.cross_attention``; DESIGN section 3.8).

Tolerances are fixed; measured values are printed with ``-s``.
  op level: float64 restatements on the identical fp32 inputs -- dots / dattn relative Frobenius 1e-4, attn max abs 1e-5
    and rows summing to 1 within 1e-5; relevance 1e-6 relative; resampling 1e-5 of the maximum, and bitwise tmf_gradcam's.
  model level: hooked runs are bitwise the unhooked ones; attn against a float64 restatement of the encoder from its actual
    inputs 1e-4 relative, dL/d attn against the restatement backpropagated from the encoder output's actual gradient 1e-3.
"""
import os
import subprocess
import sys

import pytest
import torch
import torch.nn.functional as F

from oracle import restatement as R
from tests import helpers as H
from transmf_ad_b200 import _lib as L
from transmf_ad_b200 import functional as TF
from transmf_ad_b200.interpret import cross_attention
from transmf_ad_b200.models import mymodel as M
from transmf_ad_b200.synthetic import make_labels, make_volumes, procedural_state

pytestmark = pytest.mark.gpu
DEV = "cuda"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-300))


# ---------------------------------------------------------------------------------------------------------------
# op level
# ---------------------------------------------------------------------------------------------------------------
def _operands(B, Nq, Nk, heads, dh, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    inner = heads * dh
    q = torch.randn((B, Nq, inner), device=DEV, generator=g)
    kv = torch.randn((B, Nk, 2 * inner), device=DEV, generator=g)
    dout = torch.randn((B, Nq, inner), device=DEV, generator=g)
    return q, kv, dout


def _split(t, heads):
    B, N, inner = t.shape
    return t.double().cpu().reshape(B, N, heads, inner // heads).permute(0, 2, 1, 3)


def _scores_ref(q, kv, dout, heads):
    dh = q.shape[-1] // heads
    k, v = kv.chunk(2, dim=-1)
    qh, kh, vh, gh = _split(q, heads), _split(k, heads), _split(v, heads), _split(dout, heads)
    dots = qh @ kh.transpose(-1, -2) * dh ** -0.5
    return dots, torch.softmax(dots, -1), gh @ vh.transpose(-1, -2)


def _scores(q, kv, dout, heads):
    B, Nq, inner = q.shape
    out = torch.empty_like(q)
    lse = torch.empty((B, heads, Nq), device=DEV)
    if kv.shape[1] * (inner // heads) <= 256 * 64:
        L.call("tmf_attn_fwd", L.ptr(q), L.ptr(kv), L.ptr(out), L.ptr(lse), B, Nq, kv.shape[1], heads, inner // heads,
               (inner // heads) ** -0.5)
    else:
        # beyond the shared-memory envelope of tmf_attn_fwd's fallback kernels: the float64 log-sum-exp, rounded
        lse = torch.logsumexp(_scores_ref(q, kv, dout, heads)[0], -1).float().to(DEV)
    dots, attn = TF.attn_scores(q, kv, heads, (inner // heads) ** -0.5, lse)
    return dots, attn, TF.attn_scores_grad(dout, kv, heads)


def check_scores(B, Nq, Nk, heads, dh, seed=0):
    q, kv, dout = _operands(B, Nq, Nk, heads, dh, seed)
    dots, attn, dattn = _scores(q, kv, dout, heads)
    rdots, rattn, rdattn = _scores_ref(q, kv, dout, heads)
    e_dots, e_dattn = rel(dots, rdots), rel(dattn, rdattn)
    e_attn = float((attn.double().cpu() - rattn).abs().max())
    e_sum = float((attn.double().sum(-1) - 1).abs().max())
    print(f"scores B={B} Nq={Nq} Nk={Nk} h={heads} dh={dh}: dots {e_dots:.2e} attn {e_attn:.2e} rowsum {e_sum:.2e} "
          f"dattn {e_dattn:.2e}")
    assert dots.shape == attn.shape == dattn.shape == (B, heads, Nq, Nk)
    assert e_dots <= 1e-4 and e_dattn <= 1e-4 and e_attn <= 1e-5 and e_sum <= 1e-5
    again = _scores(q, kv, dout, heads)
    assert all(torch.equal(a, b) for a, b in zip((dots, attn, dattn), again))


@pytest.mark.parametrize("dh", [16, 32, 64])
@pytest.mark.parametrize("Nq,Nk", [(150, 150), (150, 300), (256, 512), (37, 201), (70, 13), (1, 1)])
def test_attn_scores_against_float64(Nq, Nk, dh):
    check_scores(2, Nq, Nk, 4, dh)


@pytest.mark.parametrize("impl", ["0", "1"])
def test_attn_scores_with_lse_of_every_attention_implementation(impl):
    """TMF_ATTN_IMPL is read once per process: each implementation's lse is checked in a process of its own."""
    code = ("import sys; sys.path.insert(0, %r); from tests.test_gpu_attention_maps import check_scores; "
            "check_scores(2, 150, 150, 4, 32); check_scores(2, 150, 300, 4, 32); check_scores(1, 37, 61, 4, 16)" % ROOT)
    env = dict(os.environ, TMF_ATTN_IMPL=impl)
    res = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    print(res.stdout)
    assert res.returncode == 0, res.stderr[-3000:]


def test_attn_scores_refuses_other_head_dims():
    q, kv, dout = _operands(1, 8, 8, 2, 24, 0)
    lse = torch.zeros((1, 2, 8), device=DEV)
    with pytest.raises(RuntimeError, match="dim_head must be 16, 32 or 64"):
        TF.attn_scores(q, kv, 2, 0.2, lse)


@pytest.mark.parametrize("weighted", [False, True])
def test_attn_relevance_against_float64(weighted):
    g = torch.Generator(device=DEV).manual_seed(3)
    B, heads, Nq, Nk = 3, 4, 37, 150
    attn = torch.softmax(torch.randn((B, heads, Nq, Nk), device=DEV, generator=g), -1)
    dattn = torch.randn((B, heads, Nq, Nk), device=DEV, generator=g) if weighted else None
    w = attn.double() if dattn is None else (attn.double() * dattn.double()).clamp_min(0)
    Mref = w.mean(1)
    M, r = TF.attn_relevance(attn, dattn)
    print(f"relevance weighted={weighted}: M {rel(M, Mref):.2e} r {rel(r, Mref.mean(1)):.2e}")
    assert rel(M, Mref) <= 1e-6 and rel(r, Mref.mean(1)) <= 1e-6
    r2 = r.clone()
    TF.attn_relevance(attn, dattn, r2, accumulate=True)
    assert rel(r2, 2 * Mref.mean(1)) <= 1e-6
    M2, r3 = TF.attn_relevance(attn, dattn)
    assert torch.equal(M, M2) and torch.equal(r, r3)


def _resample_ref(lo, size, normalize):
    up = F.interpolate(lo.double().cpu().unsqueeze(1), size=size, mode="trilinear", align_corners=False)
    if normalize:
        mn = up.amin(dim=(1, 2, 3, 4), keepdim=True)
        mx = up.amax(dim=(1, 2, 3, 4), keepdim=True)
        up = (up - mn) / (mx - mn + 1e-7)
    return up


@pytest.mark.parametrize("normalize", [False, True])
@pytest.mark.parametrize("lo_shape,size", [((5, 6, 5), (91, 109, 91)), ((3, 3, 3), (48, 40, 33)), ((4, 5, 6), (4, 5, 6))])
def test_map_resample_against_float64(lo_shape, size, normalize):
    g = torch.Generator(device=DEV).manual_seed(5)
    lo = torch.rand((2, 3) + lo_shape, device=DEV, generator=g)
    outs = TF.map_resample(lo, size, normalize)
    for t in range(2):
        ref = _resample_ref(lo[t], size, normalize)
        err = float((outs[t].double().cpu() - ref).abs().max() / ref.abs().max())
        print(f"resample {lo_shape}->{size} normalize={normalize}: {err:.2e}")
        assert outs[t].shape == (3, 1) + tuple(size) and err <= 1e-5
    if tuple(size) == lo_shape and not normalize:
        assert torch.equal(outs[0][:, 0], lo[0])
    assert all(torch.equal(a, b) for a, b in zip(outs, TF.map_resample(lo, size, normalize)))


@pytest.mark.parametrize("normalize", [False, True])
def test_map_resample_is_gradcams_resampling(normalize):
    g = torch.Generator(device=DEV).manual_seed(7)
    B, C, d, h, w = 3, 64, 5, 6, 5
    A = torch.randn((B, d, h, w, C), device=DEV, generator=g).abs().permute(0, 4, 1, 2, 3)
    G = torch.randn((B, d, h, w, C), device=DEV, generator=g).permute(0, 4, 1, 2, 3)
    lo = TF.gradcam([A], [G], size=None, normalize=False)[0]
    up = TF.gradcam([A], [G], size=(91, 109, 91), normalize=normalize)[0]
    mine = TF.map_resample(lo[:, 0].unsqueeze(0), (91, 109, 91), normalize)[0]
    assert torch.equal(mine, up)


# ---------------------------------------------------------------------------------------------------------------
# model level
# ---------------------------------------------------------------------------------------------------------------
SHAPE = (48, 48, 48)                 # sNet output 3 x 3 x 3: N = 27 tokens per modality
CASES = {
    "model_ad": (M.model_ad, dict(dim=128, depth=2, heads=4, dim_head=32, mlp_dim=512, dropout=0.0), {}),
    "model_ad_unfused_env": (M.model_ad, dict(dim=128, depth=2, heads=4, dim_head=32, mlp_dim=512, dropout=0.0),
                             {"TMF_ENC_FUSED": "0"}),
    "model_ad_dim64": (M.model_ad, dict(dim=64, depth=2, heads=4, dim_head=16, mlp_dim=256, dropout=0.0), {}),
    "model_transformer_res": (M.model_transformer_res, dict(dim=128, depth=2, heads=4, dim_head=32, mlp_dim=512,
                                                            dropout=0.0), {}),
}


def _build(name, monkeypatch, B=2):
    ctor, kw, env = CASES[name]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    model = ctor(**kw)
    state = procedural_state(model.state_dict(), seed=0)
    model.load_state_dict(state)
    model = model.to(DEV)
    H.set_head_dropout(model, 0.0)
    label = make_labels(B)
    mri = make_volumes(B, SHAPE, seed=1, labels=label).to(DEV)
    pet = make_volumes(B, SHAPE, seed=2, labels=label).to(DEV)
    return model, state, kw, (mri, pet), label.to(DEV)


def _encoders(model):
    """(qualified name, Transformer) of every fusion encoder in reference call order: mri_enc then pet_enc, per layer."""
    return [(f"fuse_transformer.layers.{l}.{i}", pair[i]) for l, pair in enumerate(model.fuse_transformer.layers)
            for i in range(2)]


def _loss(outs, label):
    outs = outs if isinstance(outs, tuple) else (outs,)
    loss = F.cross_entropy(outs[0], label)
    for o in outs[1:]:
        loss = loss + F.cross_entropy(o, label)
    return loss


def _run(model, state, inputs, label, train, hooked, reducer_flat=None):
    """One forward + backward; with ``hooked``, observing hooks on every attend and a tensor hook on every attn."""
    model.load_state_dict(state)
    model.train(train)
    model.zero_grad(set_to_none=True)
    seen, handles = [], []
    if hooked:
        for name, enc in _encoders(model):
            att = enc.layers[0][0].fn.attend

            def hook(m, args, attn, name=name):
                seen.append((name, args[0], attn))
                if attn.requires_grad:
                    attn.register_hook(lambda g, name=name: seen.append((name + ".grad", g)))
            handles.append(att.register_forward_hook(hook))
            handles.append(att.register_forward_pre_hook(lambda m, args, name=name: seen.append((name + ".pre", args[0]))))
    torch.manual_seed(0)
    outs = model(*inputs)
    loss = _loss(outs, label)
    loss.backward()
    torch.cuda.synchronize()
    for h in handles:
        h.remove()
    grads = {k: p.grad.clone() for k, p in model.named_parameters() if p.grad is not None}
    bufs = {k: b.clone() for k, b in model.named_buffers()}
    outs = tuple(o.detach().clone() for o in (outs if isinstance(outs, tuple) else (outs,)))
    return outs, loss.detach().clone(), grads, bufs, seen


# dim 64: some sNet layers (16-channel convolutions) are outside the tcgen05 kernels' envelope and run on the direct
# kernels, whose BatchNorm statistics and weight gradients are summed with atomics -- two unhooked runs of the whole model
# already differ there.  The bitwise comparison of that configuration is made on its fusion stack alone (the unfused
# encoder path with dim_head 16), in test_observing_hooks_change_nothing_on_the_dim64_fusion_stack.
REPRODUCIBLE = {"model_ad", "model_ad_unfused_env", "model_transformer_res"}


@pytest.mark.parametrize("train", [True, False])
@pytest.mark.parametrize("name", list(CASES))
def test_observing_hooks_change_nothing_and_fire_in_reference_order(name, train, monkeypatch):
    model, state, kw, inputs, label = _build(name, monkeypatch)
    base = _run(model, state, inputs, label, train, False)
    n0 = L.launch_count()
    plain = _run(model, state, inputs, label, train, False)
    n_plain = L.launch_count() - n0
    n0 = L.launch_count()
    hooked = _run(model, state, inputs, label, train, True)
    n_hooked = L.launch_count() - n0
    differ0 = sorted(k for k in base[2] if not torch.equal(base[2][k], plain[2][k]))
    print(f"{name} train={train}: gradients that differ between two unhooked runs: {differ0}")
    if name in REPRODUCIBLE:
        for run in (plain, hooked):
            for a, b in zip(base[0], run[0]):
                assert torch.equal(a, b)
            assert torch.equal(base[1], run[1])
            differ = [k for k in base[2] if not torch.equal(base[2][k], run[2][k])]
            assert base[2].keys() == run[2].keys() and not differ, (run is plain, differ)
            assert all(torch.equal(base[3][k], run[3][k]) for k in base[3])
    names = [n for n, _ in _encoders(model)]
    seen = hooked[4]
    fwd = [s for s in seen if len(s) == 3]
    pre = [s[0] for s in seen if s[0].endswith(".pre")]
    assert [s[0] for s in fwd] == names and pre == [n + ".pre" for n in names]
    grads = [s for s in seen if s[0].endswith(".grad")]
    assert sorted(s[0] for s in grads) == sorted(n + ".grad" for n in names)
    N = 27
    Nk = 2 * N if name == "model_transformer_res" else N
    for (_, dots, attn), (_, g) in zip(fwd, sorted(grads, key=lambda s: names.index(s[0][:-5]))):
        assert dots.shape == attn.shape == g.shape == (2, kw["heads"], N, Nk)
        assert attn.requires_grad and not dots.requires_grad
    # one scores launch per encoder call in the forward pass, one more in the backward pass
    print(f"{name} train={train}: launches {n_plain} -> {n_hooked}")
    assert n_hooked == n_plain + 2 * len(names)


def _fusion_step(fuser, tokens, wout, hooked):
    seen, handles = [], []
    if hooked:
        for pair in fuser.layers:
            for enc in pair:
                def hook(m, args, attn):
                    seen.append(attn)
                    attn.register_hook(lambda g: seen.append(g))
                handles.append(enc.layers[0][0].fn.attend.register_forward_hook(hook))
    fuser.zero_grad(set_to_none=True)
    tm, tp = (t.detach().clone().requires_grad_(True) for t in tokens)
    n0 = L.launch_count()
    out = fuser(tm, tp)
    (out * wout).sum().backward()
    torch.cuda.synchronize()
    n = L.launch_count() - n0
    for h in handles:
        h.remove()
    grads = {k: p.grad.clone() for k, p in fuser.named_parameters()}
    return out.detach().clone(), tm.grad.clone(), tp.grad.clone(), grads, n, len(seen)


@pytest.mark.parametrize("train", [True, False])
def test_observing_hooks_change_nothing_on_the_dim64_fusion_stack(train):
    from transmf_ad_b200.models.networks import CrossTransformer_MOD_AVG
    torch.manual_seed(0)
    fuser = CrossTransformer_MOD_AVG(64, 2, 4, 16, 256, 0.0).to(DEV).train(train)
    g = torch.Generator(device=DEV).manual_seed(11)
    tokens = [torch.randn((2, 27, 64), device=DEV, generator=g) for _ in range(2)]
    wout = torch.randn((2, 4 * 64), device=DEV, generator=g)
    base = _fusion_step(fuser, tokens, wout, False)
    plain = _fusion_step(fuser, tokens, wout, False)
    hooked = _fusion_step(fuser, tokens, wout, True)
    for run in (plain, hooked):
        assert all(torch.equal(a, b) for a, b in zip(base[:3], run[:3]))
        assert base[3].keys() == run[3].keys() and all(torch.equal(base[3][k], run[3][k]) for k in base[3])
    assert hooked[5] == 8                                  # four encoder calls: attn, then its gradient
    assert hooked[4] == plain[4] + 2 * 4


def test_observing_hooks_leave_the_flat_gradient_buffer_bitwise(monkeypatch):
    from transmf_ad_b200.dp import FlatGradReducer
    model, state, kw, inputs, label = _build("model_ad", monkeypatch)
    red = FlatGradReducer(model=model).install()
    try:
        _run(model, state, inputs, label, True, False)
        flat0 = red.flat.clone()
        _run(model, state, inputs, label, True, True)
        assert torch.equal(flat0, red.flat)
    finally:
        TF.set_grad_slots(None)


def _enc64(sd, pfx, x, ctx, heads, keep):
    """The reference encoder (restatement.transformer_encoder) in float64, keeping its attention probabilities."""
    p = pfx + ".layers.0"
    xn = R.layernorm(sd, p + ".0.norm", x)
    q = F.linear(xn, sd[p + ".0.fn.to_q.weight"])
    k, v = F.linear(ctx, sd[p + ".0.fn.to_kv.weight"]).chunk(2, dim=-1)
    B, n, inner = q.shape
    dh = inner // heads
    sp = lambda t: t.reshape(B, t.shape[1], heads, dh).permute(0, 2, 1, 3)
    attn = torch.softmax(sp(q) @ sp(k).transpose(-1, -2) * dh ** -0.5, -1)
    keep.append(attn)
    out = (attn @ sp(v)).permute(0, 2, 1, 3).reshape(B, n, inner)
    x = F.linear(out, sd[p + ".0.fn.to_out.0.weight"], sd[p + ".0.fn.to_out.0.bias"]) + x
    x = R.feedforward(sd, p + ".1.fn", R.layernorm(sd, p + ".1.norm", x)) + x
    return R.layernorm(sd, pfx + ".norm", x)


@pytest.mark.parametrize("train", [True, False])
@pytest.mark.parametrize("name", list(CASES))
def test_attn_and_its_gradient_against_float64(name, train, monkeypatch):
    model, state, kw, inputs, label = _build(name, monkeypatch)
    model.train(train)
    sd = R.clone_state(state, requires_grad=False, dtype=torch.float64)
    cap, handles = {}, []
    for ename, enc in _encoders(model):
        def pre(m, args, kwargs, ename=ename):
            cap[ename + ".in"] = (args[0].detach().clone(), kwargs["context"].detach().clone())

        def post(m, args, kwargs, out, ename=ename):
            out.register_hook(lambda g: cap.__setitem__(ename + ".dy", g.clone()))

        def att(m, args, attn, ename=ename):
            cap[ename + ".attn"] = attn.detach().clone()
            attn.register_hook(lambda g: cap.__setitem__(ename + ".dattn", g.clone()))
        handles += [enc.register_forward_pre_hook(pre, with_kwargs=True), enc.register_forward_hook(post, with_kwargs=True),
                    enc.layers[0][0].fn.attend.register_forward_hook(att)]
    _loss(model(*inputs), label).backward()
    torch.cuda.synchronize()
    for h in handles:
        h.remove()
    for ename, _ in _encoders(model):
        x, ctx = (t.double().cpu() for t in cap[ename + ".in"])
        keep = []
        _enc64(sd, ename, x, ctx, kw["heads"], keep)
        e_attn = rel(cap[ename + ".attn"], keep[0])
        # backpropagate the captured output gradient through the restated encoder, from attn on; the output includes the
        # caller's outer residual (add_input), as the Transformer's output does
        a64 = keep[0].detach().requires_grad_(True)
        p = ename + ".layers.0"
        xn = R.layernorm(sd, p + ".0.norm", x)
        v = F.linear(ctx, sd[p + ".0.fn.to_kv.weight"]).chunk(2, dim=-1)[1]
        B, n, inner = xn.shape[0], xn.shape[1], kw["heads"] * kw["dim_head"]
        dh = kw["dim_head"]
        out = (a64 @ v.reshape(B, v.shape[1], kw["heads"], dh).permute(0, 2, 1, 3)).permute(0, 2, 1, 3).reshape(B, n, inner)
        h = F.linear(out, sd[p + ".0.fn.to_out.0.weight"], sd[p + ".0.fn.to_out.0.bias"]) + x
        h = R.feedforward(sd, p + ".1.fn", R.layernorm(sd, p + ".1.norm", h)) + h
        y = R.layernorm(sd, ename + ".norm", h) + x
        dattn = torch.autograd.grad(y, a64, cap[ename + ".dy"].double().cpu())[0]
        e_grad = rel(cap[ename + ".dattn"], dattn)
        print(f"{name} train={train} {ename}: attn {e_attn:.2e} dattn {e_grad:.2e}")
        assert e_attn <= 1e-4 and e_grad <= 1e-3


def test_hooks_fire_under_no_grad_without_a_graph(monkeypatch):
    model, state, kw, inputs, label = _build("model_ad", monkeypatch)
    model.eval()
    seen = []
    for _, enc in _encoders(model):
        enc.layers[0][0].fn.attend.register_forward_hook(lambda m, a, attn: seen.append((a[0], attn)), with_kwargs=False)
    with torch.no_grad():
        model(*inputs)
    assert len(seen) == 4 and not any(a.requires_grad or d.requires_grad for d, a in seen)


# ---------------------------------------------------------------------------------------------------------------
# refusals
# ---------------------------------------------------------------------------------------------------------------
def _attend(model):
    return model.fuse_transformer.layers[0][0].layers[0][0].fn.attend


@pytest.mark.parametrize("name", ["model_ad", "model_ad_dim64"])
def test_replacing_and_in_place_hooks_are_refused(name, monkeypatch):
    model, state, kw, inputs, label = _build(name, monkeypatch)
    att = _attend(model)
    for register, fn, exc in [("register_forward_hook", lambda m, a, o: o * 2, NotImplementedError),
                              ("register_forward_pre_hook", lambda m, a: (a[0] * 2,), NotImplementedError),
                              ("register_forward_hook", lambda m, a, o: (o.detach().mul_(1.0), None)[1], RuntimeError),
                              ("register_forward_pre_hook", lambda m, a: (a[0].detach().add_(0.0), None)[1], RuntimeError)]:
        h = getattr(att, register)(fn)
        with pytest.raises(exc):
            model(*inputs)
        h.remove()


@pytest.mark.parametrize("name", ["model_ad", "model_ad_dim64"])
@pytest.mark.parametrize("how", ["replace_grad", "modify_grad", "attn_in_loss"])
def test_gradients_other_than_the_taps_own_are_refused(name, how, monkeypatch):
    model, state, kw, inputs, label = _build(name, monkeypatch)
    model.train()
    kept = []

    def hook(m, a, attn):
        kept.append(attn)
        if how == "replace_grad":
            attn.register_hook(lambda g: g * 2)
        elif how == "modify_grad":
            attn.register_hook(lambda g: (g.mul_(2), None)[1])
    _attend(model).register_forward_hook(hook)
    loss = _loss(model(*inputs), label)
    if how == "attn_in_loss":
        loss = loss + kept[0].sum()
    with pytest.raises(NotImplementedError, match="only be observed"):
        loss.backward()


def test_backward_hook_on_attend_is_refused(monkeypatch):
    model, state, kw, inputs, label = _build("model_ad", monkeypatch)
    _attend(model).register_full_backward_hook(lambda *a: None)
    with pytest.raises(NotImplementedError, match="backward hooks"):
        model(*inputs)


def test_dead_hooks_warn_and_the_model_still_runs(monkeypatch):
    model, state, kw, inputs, label = _build("model_ad", monkeypatch)
    enc = model.fuse_transformer.layers[0][0]
    enc.layers[0][0].fn.to_q.register_forward_hook(lambda *a: None)
    enc.layers[0][1].register_forward_hook(lambda *a: None)        # PreNorm(FeedForward): never runs on the fused path
    with pytest.warns(UserWarning, match="Attention.attend"):
        model(*inputs)


# ---------------------------------------------------------------------------------------------------------------
# cross_attention
# ---------------------------------------------------------------------------------------------------------------
def _xattn_ref(model, name, kw, sd, fm, fp, label, weighted):
    """Float64 restatement of the fusion transformer and the head from the towers' actual outputs; the maps as
    cross_attention defines them."""
    tm, tp = (R._tokens(f.double().cpu()).requires_grad_(weighted) for f in (fm, fp))
    N = tm.shape[1]
    keep = []
    depth = len(model.fuse_transformer.layers)
    m, p = tm, tp
    for l in range(depth):
        if name == "model_transformer_res":
            m = _enc64(sd, f"fuse_transformer.layers.{l}.0", m, torch.cat([m, p], 1), kw["heads"], keep) + m
            p = _enc64(sd, f"fuse_transformer.layers.{l}.1", p, torch.cat([m, p], 1), kw["heads"], keep) + p
        else:
            m = _enc64(sd, f"fuse_transformer.layers.{l}.0", m, p, kw["heads"], keep) + m
            p = _enc64(sd, f"fuse_transformer.layers.{l}.1", p, m, kw["heads"], keep) + p
    if name == "model_transformer_res":
        c = torch.cat([(m + tm).mean(1), (p + tp).mean(1)], dim=1)
        h = F.relu(F.linear(c, sd["fc_cls.0.weight"], sd["fc_cls.0.bias"]))
        h = F.relu(F.linear(h, sd["fc_cls.3.weight"], sd["fc_cls.3.bias"]))
        logits = F.linear(h, sd["fc_cls.6.weight"], sd["fc_cls.6.bias"])
    else:
        cls = torch.cat([m.mean(1), p.mean(1), m.amax(1), p.amax(1)], dim=1)
        logits = R.fc_cls_transformer(sd, "fc_cls", cls, False, 0.0)
    grads = [None] * len(keep)
    if weighted:
        grads = torch.autograd.grad(logits.gather(1, label.cpu().view(-1, 1)).sum(), keep)
    maps = [a.mean(1) if g is None else (a * g).clamp_min(0).mean(1) for a, g in zip(keep, grads)]
    r = [M.mean(1) for M in maps]
    if name == "model_transformer_res":
        tot = sum(r)
        rm, rp = tot[:, :N], tot[:, N:]
    else:
        rp, rm = sum(r[0::2]), sum(r[1::2])
    return [M.detach() for M in maps], rm.detach(), rp.detach()


@pytest.mark.parametrize("weighted", [False, True])
@pytest.mark.parametrize("name", ["model_ad", "model_transformer_res", "model_ad_dim64"])
def test_cross_attention_against_float64(name, weighted, monkeypatch):
    model, state, kw, inputs, label = _build(name, monkeypatch)
    model.eval()
    sd = R.clone_state(state, requires_grad=False, dtype=torch.float64)
    feats = {}
    model.mri_cnn.register_forward_hook(lambda m, a, o: feats.__setitem__("m", o.detach().clone()))
    model.pet_cnn.register_forward_hook(lambda m, a, o: feats.__setitem__("p", o.detach().clone()))
    flags = {k: p.requires_grad for k, p in model.named_parameters()}
    L.TIMER.start()
    res = cross_attention(model, inputs, label if weighted else None, upsample=True, normalize=True)
    tags = set(L.TIMER.stop())
    lo = cross_attention(model, inputs, label if weighted else None, upsample=False, normalize=False)
    maps, rm, rp = _xattn_ref(model, name, kw, sd, feats["m"], feats["p"], label, weighted)
    tol_map, tol_vol = (1e-3, 2e-3) if weighted else (1e-4, 1e-4)
    got = [M for pair in res.maps for M in pair]
    assert len(res.maps) == len(model.fuse_transformer.layers) and len(got) == len(maps)
    for a, b in zip(got, maps):
        assert a.shape == b.shape
        assert rel(a, b) <= tol_map, rel(a, b)
    d, h, w = feats["m"].shape[2:]
    for vol, lo_map, r in ((res.mri, lo.mri, rm), (res.pet, lo.pet, rp)):
        r = r.reshape(-1, d, h, w)
        assert lo_map.shape == (2, 1, d, h, w) and rel(lo_map[:, 0], r) <= tol_map
        ref = _resample_ref(r, SHAPE, True)
        err = float((vol.double().cpu() - ref).abs().max())
        print(f"cross_attention {name} weighted={weighted}: maps {max(rel(a, b) for a, b in zip(got, maps)):.2e} "
              f"volume {err:.2e}")
        assert vol.shape == (2, 1) + SHAPE and err <= tol_vol
    # side effects: no parameter gradient, flags restored, no weight-gradient or sNet backward launch
    assert all(p.grad is None for p in model.parameters())
    assert flags == {k: p.requires_grad for k, p in model.named_parameters()}
    bad = [t for t in tags if "wgrad" in t or "_bwd" in t and ("conv" in t or "bn_" in t) or "dgrad@" in t]
    assert not bad, bad
    if weighted and name != "model_ad_dim64":                        # the fused encoders' chain backward feeds the tap
        assert "tmf_encoder_chain_bwd" in tags and "tmf_attn_scores" in tags
    again = cross_attention(model, inputs, label if weighted else None)
    assert torch.equal(again.mri, res.mri) and torch.equal(again.pet, res.pet)
    assert all(torch.equal(a, b) for pa, pb in zip(again.maps, res.maps) for a, b in zip(pa, pb))


def test_cross_attention_in_train_mode_restores_flags(monkeypatch):
    model, state, kw, inputs, label = _build("model_ad", monkeypatch)
    model.train()
    model.fc_cls[0].weight.requires_grad_(False)
    flags = {k: p.requires_grad for k, p in model.named_parameters()}
    res = cross_attention(model, inputs, 1)
    assert flags == {k: p.requires_grad for k, p in model.named_parameters()}
    assert all(p.grad is None for p in model.parameters())
    assert torch.isfinite(res.mri).all() and torch.isfinite(res.pet).all()


@pytest.mark.parametrize("weighted", [False, True])
def test_cross_attention_full_size(weighted):
    model = M.model_ad(dim=128, depth=3, heads=4, dim_head=32, mlp_dim=512, dropout=0.0)
    model.load_state_dict(procedural_state(model.state_dict(), seed=0))
    model = model.to(DEV).eval()
    B, shape = 8, (91, 109, 91)
    label = make_labels(B)
    mri = make_volumes(B, shape, seed=1, labels=label).to(DEV)
    pet = make_volumes(B, shape, seed=2, labels=label).to(DEV)
    res = cross_attention(model, (mri, pet), label.to(DEV) if weighted else None)
    assert len(res.maps) == 3 and res.maps[0][0].shape == (B, 150, 150)
    for vol in (res.mri, res.pet):
        assert vol.shape == (B, 1) + shape and torch.isfinite(vol).all()
        # (x - min) / (max - min + 1e-7): gradient-weighted relevances are small, so the maximum sits visibly below 1
        assert float(vol.amin()) == 0.0 and 0.5 < float(vol.amax()) <= 1.0
    again = cross_attention(model, (mri, pet), label.to(DEV) if weighted else None)
    assert torch.equal(again.mri, res.mri) and torch.equal(again.pet, res.pet)

"""Block outputs of the sNet towers exposed to module hooks (a segmented run: one autograd node per segment, split at the
exposed block outputs) and Grad-CAM on them (csrc/gradcam.cu, transmf_ad_b200.interpret.grad_cam).

Tolerances are fixed; measured values are printed with ``-s`` (B200, first measurement noted next to each constant).
  op level: the dual-output pass is bitwise the single-output pass for bf16 out / ymax; its fp32 twin rounds to out and
    sits within 1e-6 of the fp32 CPU composition.  tmf_gradcam against a float64 torch restatement: 1e-5 of the maximum.
  model level: hooked runs are bitwise the unhooked ones (the gradient at a boundary is a widened bf16 value, fed to the
    same arithmetic).  Tap activations / gradients and Grad-CAM maps against Oracle-A (oracle/restatement.py with bf16
    rounding): cosine and rel-L2; bounds from the first measurement with headroom.
"""
import copy

import pytest
import torch
import torch.nn.functional as F

from oracle import restatement as R
from tests import helpers as H
from transmf_ad_b200 import _lib as L
from transmf_ad_b200 import functional as TF
from transmf_ad_b200.interpret import grad_cam
from transmf_ad_b200.models import mymodel as M
from transmf_ad_b200.models.networks import BLOCKS

pytestmark = pytest.mark.gpu
DEV = "cuda"
SLOPE = 0.01
TAP_LAYER = {"conv1": "conv1.0", "conv2": "conv2.3", "conv3": "conv3.3", "conv4": "conv4.3"}
ACT_COS, ACT_REL = 0.9999, 0.012            # block activations vs Oracle-A (worst 0.999983 / 0.0058)
GRAD_COS, GRAD_REL = 0.95, 0.45              # gradient at a block output vs Oracle-A (0.976 / 0.22)
CAM_COS, CAM_REL = 0.9, 0.6                  # Grad-CAM (block extent, not normalised) vs Oracle-A (0.953 / 0.306)
NOGRAD_REL = 0.01                            # eval: folded no-grad path vs the grad-enabled path (0.0044)


# ---------------------------------------------------------------------------------------------------------------
# op level: dual-output pass
# ---------------------------------------------------------------------------------------------------------------
def _coef(C, g):
    gamma = torch.randn(C, generator=g)
    gamma[:3] = -gamma[:3].abs()                       # negative BatchNorm scales
    gamma[3] = 0.0                                     # and a zero one
    mean, invstd = torch.randn(C, generator=g) * 0.1, torch.rand(C, generator=g) + 0.5
    scale = gamma * invstd
    shift = torch.randn(C, generator=g) * 0.1 - mean * scale
    return torch.cat([scale, shift, mean, invstd]).float()


def _cpu_fp32(y, coef, pool):
    C = y.shape[-1]
    scale, shift = coef[:C], coef[C:2 * C]
    a = F.leaky_relu(y.float() * scale + shift, SLOPE).permute(0, 4, 1, 2, 3)
    if pool == L.POOL_MAX:
        a = F.max_pool3d(a, 2)
    elif pool == L.POOL_AVG:
        a = F.avg_pool3d(a, 2)
    return a.permute(0, 2, 3, 4, 1).contiguous()


@pytest.mark.parametrize("pool", [L.POOL_MAX, L.POOL_NONE, L.POOL_AVG])
@pytest.mark.parametrize("shape", [(2, 9, 11, 7, 32), (1, 5, 6, 13, 64), (3, 4, 7, 5, 128)])
@pytest.mark.parametrize("ties", [False, True])
def test_dual_output_pass(shape, pool, ties):
    B, D, Hh, W, C = shape
    g = torch.Generator().manual_seed(hash((shape, pool, ties)) % 997)
    ng = 2
    if ties:
        ys = [(torch.randint(-3, 4, shape, generator=g).float() * 0.25).bfloat16() for _ in range(ng)]
    else:
        ys = [torch.randn(shape, generator=g).bfloat16() for _ in range(ng)]
    coefs = [_coef(C, g) for _ in range(ng)]
    yd, cd = [y.to(DEV) for y in ys], [c.to(DEV) for c in coefs]
    oshape = (B, D, Hh, W, C) if pool == L.POOL_NONE else (B, D // 2, Hh // 2, W // 2, C)
    E = lambda dt: [torch.empty(oshape, dtype=dt, device=DEV) for _ in range(ng)]
    ref, out, out32 = E(torch.bfloat16), E(torch.bfloat16), E(torch.float32)
    L.call("tmf_bn_act_pool_fwd", ng, L.ptrs(yd), L.ptrs(cd), L.ptrs(ref), 0, B, D, Hh, W, C, pool, SLOPE)
    L.call("tmf_bn_act_pool_fwd_dual", ng, L.ptrs(yd), L.ptrs(cd), L.ptrs(out), L.ptrs(out32), B, D, Hh, W, C, pool, SLOPE)
    if pool == L.POOL_MAX:
        ref_k, ymax_ref, out_k, out32_k, ymax = E(torch.bfloat16), E(torch.bfloat16), E(torch.bfloat16), E(torch.float32), E(torch.bfloat16)
        L.call("tmf_bn_act_pool_fwd_keepmax", ng, L.ptrs(yd), L.ptrs(cd), L.ptrs(ref_k), L.ptrs(ymax_ref), 0, B, D, Hh, W, C, SLOPE)
        L.call("tmf_bn_act_pool_fwd_keepmax_dual", ng, L.ptrs(yd), L.ptrs(cd), L.ptrs(out_k), L.ptrs(out32_k), L.ptrs(ymax),
               B, D, Hh, W, C, SLOPE)
    torch.cuda.synchronize()
    for t in range(ng):
        cpu = _cpu_fp32(ys[t], coefs[t], pool)
        pairs = [(ref[t], out[t], out32[t])] + ([(ref_k[t], out_k[t], out32_k[t])] if pool == L.POOL_MAX else [])
        for r, o, o32 in pairs:
            assert torch.equal(r.view(torch.int16), o.view(torch.int16))
            assert torch.equal(o32.bfloat16().view(torch.int16), o.view(torch.int16))
            err = float((o32.cpu() - cpu).abs().max() / cpu.abs().max().clamp_min(1e-30))
            assert err <= 1e-6, err
        if pool == L.POOL_MAX:
            assert torch.equal(ymax[t].view(torch.int16), ymax_ref[t].view(torch.int16))


def test_widen_narrow_roundtrip():
    x = torch.randn(2, 3, 5, 7, 32, device=DEV).bfloat16()
    w = torch.empty(x.shape, dtype=torch.float32, device=DEV)
    n = torch.empty_like(x)
    L.call("tmf_widen_bf16", 1, L.ptrs([x]), L.ptrs([w]), x.numel())
    L.call("tmf_narrow_f32", 1, L.ptrs([w]), L.ptrs([n]), x.numel())
    assert torch.equal(w, x.float()) and torch.equal(n.view(torch.int16), x.view(torch.int16))
    f = torch.randn(x.shape, device=DEV)
    L.call("tmf_narrow_f32", 1, L.ptrs([f]), L.ptrs([n]), x.numel())
    assert torch.equal(n.view(torch.int16), f.bfloat16().view(torch.int16))


# ---------------------------------------------------------------------------------------------------------------
# op level: tmf_gradcam
# ---------------------------------------------------------------------------------------------------------------
def _assert_cam_close(cam, ref, what):
    """A map that is zero everywhere (every class-weighted sum negative) must come out zero; otherwise cosine / rel-L2."""
    assert cam.shape == ref.shape
    if float(ref.abs().max()) == 0.0:
        print(f"{what}: zero map")
        assert float(cam.abs().max()) == 0.0
        return
    c, r = H.cosine(cam, ref), H.rel_err(cam, ref)
    print(f"{what}: cos {c:.5f} rel {r:.3g}")
    assert c >= CAM_COS and r <= CAM_REL


def _cam_ref(A, G, size, normalize):
    A, G = A.double().cpu(), G.double().cpu()
    alpha = G.mean(dim=(2, 3, 4), keepdim=True)
    cam = torch.relu((alpha * A).sum(1, keepdim=True))
    if size is not None:
        cam = F.interpolate(cam, size=size, mode="trilinear", align_corners=False)
    if normalize:
        mn = cam.amin(dim=(1, 2, 3, 4), keepdim=True)
        mx = cam.amax(dim=(1, 2, 3, 4), keepdim=True)
        cam = (cam - mn) / (mx - mn + 1e-7)
    return cam


def _cl(B, C, d, h, w, g, neg=False):
    t = torch.randn((B, d, h, w, C), generator=g)
    return t.permute(0, 4, 1, 2, 3).to(DEV)


CAM_CASES = [(2, 32, 45, 54, 45, (91, 109, 91)), (2, 64, 22, 27, 22, (91, 109, 91)), (2, 128, 11, 13, 11, (91, 109, 91)),
             (2, 128, 5, 6, 5, (91, 109, 91)), (1, 32, 7, 9, 5, (15, 19, 11)), (3, 64, 3, 5, 7, (7, 11, 13)),
             (2, 96, 4, 3, 5, (9, 6, 10))]


@pytest.mark.parametrize("case", CAM_CASES)
@pytest.mark.parametrize("upsample", [True, False])
@pytest.mark.parametrize("normalize", [True, False])
def test_gradcam_op_against_float64(case, upsample, normalize):
    B, C, d, h, w, size = case
    g = torch.Generator().manual_seed(hash(case) % 991)
    A = _cl(B, C, d, h, w, g).abs()
    G = _cl(B, C, d, h, w, g) + 0.05
    cam = TF.gradcam([A], [G], size=size if upsample else None, normalize=normalize)[0]
    ref = _cam_ref(A, G, size if upsample else None, normalize)
    assert cam.shape == ref.shape
    err = float((cam.cpu().double() - ref).abs().max() / ref.abs().max().clamp_min(1e-30))
    print(f"[gradcam op] {case} ups={upsample} norm={normalize}: max err / max {err:.3g}")
    assert err <= 1e-5


@pytest.mark.parametrize("normalize", [True, False])
def test_gradcam_op_all_negative_map_is_zero(normalize):
    g = torch.Generator().manual_seed(3)
    A = _cl(2, 64, 6, 7, 5, g).abs() + 0.1
    G = -(_cl(2, 64, 6, 7, 5, g).abs() + 0.1)                # every alpha < 0: every cam value < 0 before the ReLU
    for size in ((13, 15, 11), None):
        cam = TF.gradcam([A], [G], size=size, normalize=normalize)[0]
        assert torch.isfinite(cam).all() and float(cam.abs().max()) == 0.0


def test_gradcam_op_determinism_and_two_towers():
    g = torch.Generator().manual_seed(4)
    As = [_cl(3, 32, 45, 54, 45, g).abs() for _ in range(2)]
    Gs = [_cl(3, 32, 45, 54, 45, g) for _ in range(2)]
    for size in ((91, 109, 91), None):
        both = TF.gradcam(As, Gs, size=size)
        again = TF.gradcam(As, Gs, size=size)
        for t in range(2):
            one = TF.gradcam([As[t]], [Gs[t]], size=size)[0]
            assert torch.equal(both[t], one) and torch.equal(both[t], again[t])


# ---------------------------------------------------------------------------------------------------------------
# model level
# ---------------------------------------------------------------------------------------------------------------
def _model(gold, train):
    model = getattr(M, gold["kind"])(**gold["kwargs"])
    model.load_state_dict(H.case_state(gold), strict=True)
    model = model.to(DEV).train(train)
    H.set_head_dropout(model, 0.0)
    return model


def _inputs(gold):
    mri, pet, label = H.case_inputs(gold)
    return ((mri,) if gold["kind"] == "model_single" else (mri, pet)), label


def _towers(model):
    return [m for m in model.modules() if isinstance(m, M.sNet)]


def _objective(outs, label, train):
    outs = outs if isinstance(outs, tuple) else (outs,)
    if train:
        return H.losses(outs, label)[2]
    return outs[0].gather(1, label.view(-1, 1).to(outs[0].device)).sum()


def _observe(model, which="all"):
    """Observing forward hooks and pre-hooks on every block (and the towers) of `which` towers; returns the call log."""
    log, handles = [], []
    towers = _towers(model)
    for ti, tw in enumerate(towers if which == "all" else towers[:1]):
        for name in BLOCKS:
            blk = getattr(tw, name)
            handles.append(blk.register_forward_pre_hook(lambda m, a, ti=ti, name=name: log.append(("pre", ti, name, a))))
            handles.append(blk.register_forward_hook(lambda m, a, o, ti=ti, name=name: log.append(("fwd", ti, name, a, o))))
        handles.append(tw.register_forward_pre_hook(lambda m, a, ti=ti: log.append(("pre", ti, "tower", a))))
        handles.append(tw.register_forward_hook(lambda m, a, o, ti=ti: log.append(("fwd", ti, "tower", a, o))))
    return log, handles


def _run(model, inputs, label, train, want_x):
    xs = [x.to(DEV).clone().requires_grad_(want_x) for x in inputs]
    outs = model(*xs)
    obj = _objective(outs, label.to(DEV), train)
    obj.backward()
    outs = outs if isinstance(outs, tuple) else (outs,)
    return ([o.detach() for o in outs], obj.detach(), {k: p.grad for k, p in model.named_parameters()},
            {k: v.clone() for k, v in model.state_dict().items()}, [x.grad for x in xs])


@pytest.mark.parametrize("name", ["model_ad_h4", "model_cnn_ad"])
@pytest.mark.parametrize("train", [True, False])
@pytest.mark.parametrize("want_x", [False, True])
@pytest.mark.parametrize("which", ["all", "one"])
def test_observing_hooks_change_nothing(name, train, want_x, which):
    gold = H.load_golden(name)
    inputs, label = _inputs(gold)
    base = _model(gold, train)
    plain = _run(copy.deepcopy(base), inputs, label, train, want_x)
    model = copy.deepcopy(base)
    log, _ = _observe(model, which)
    hooked = _run(model, inputs, label, train, want_x)
    assert len(log) == (2 if which == "all" else 1) * 10
    for a, b in zip(plain[0], hooked[0]):
        assert torch.equal(a, b)
    assert torch.equal(plain[1], hooked[1])
    for k in plain[2]:
        assert (plain[2][k] is None) == (hooked[2][k] is None), k
        assert plain[2][k] is None or torch.equal(plain[2][k], hooked[2][k]), k
    for k in plain[3]:
        assert torch.equal(plain[3][k], hooked[3][k]), k
    for a, b in zip(plain[4], hooked[4]):
        assert (a is None and b is None) or torch.equal(a, b)


EXTENTS = {"conv1": (32, 0), "conv2": (64, 1), "conv3": (128, 2), "conv4": (128, 3)}


def test_hooks_fire_once_with_block_shapes_and_tensor_hook_gradients():
    gold = H.load_golden("model_ad_h4")
    inputs, label = _inputs(gold)
    model = _model(gold, False)
    log, _ = _observe(model)
    grads = {}
    def tensor_hook(m, a, o):
        o.register_hook(lambda g: grads.setdefault("conv3", g))

    model.mri_cnn.conv3.register_forward_hook(tensor_hook)
    xs = [x.to(DEV) for x in inputs]
    outs = model(*xs)
    obj = _objective(outs, label.to(DEV), False)
    fwd = {(e[1], e[2]): e for e in log if e[0] == "fwd"}
    pre = {(e[1], e[2]): e for e in log if e[0] == "pre"}
    assert len(fwd) == len(pre) == 10 and len(log) == 20
    D = tuple(inputs[0].shape[2:])
    for t in range(2):
        prev = xs[t]
        for name in BLOCKS:
            _, _, _, args, out = fwd[(t, name)]
            C, k = EXTENTS[name]
            ext = tuple(s >> (k + 1) for s in D)
            assert len(args) == 1 and args[0] is prev and pre[(t, name)][3][0] is prev
            assert out.shape == (inputs[0].shape[0], C) + ext and out.dtype == torch.float32
            assert out.is_contiguous(memory_format=torch.channels_last_3d)
            prev = out
        assert fwd[(t, "tower")][4] is prev and fwd[(t, "tower")][3][0] is xs[t]
    (g,) = torch.autograd.grad(obj, [fwd[(0, "conv3")][4]])
    assert torch.equal(grads["conv3"], g)


def test_tower_hooks_fire_on_the_pair_path_and_replace():
    gold = H.load_golden("model_cnn_ad")
    inputs, label = _inputs(gold)
    model = _model(gold, False)
    calls = []
    model.mri_cnn.register_forward_pre_hook(lambda m, a: calls.append("pre"))
    model.pet_cnn.register_forward_hook(lambda m, a, o: calls.append("fwd"))
    base = model(*[x.to(DEV) for x in inputs])[0]
    assert calls == ["pre", "fwd"]
    model.pet_cnn.register_forward_hook(lambda m, a, o: o * 0)
    zeroed = model(*[x.to(DEV) for x in inputs])[0]
    assert not torch.equal(base, zeroed)


def test_tower_backward_hook_falls_back_to_module_call():
    gold = H.load_golden("model_cnn_ad")
    inputs, label = _inputs(gold)
    model = _model(gold, True)
    got = []
    model.mri_cnn.register_full_backward_hook(lambda m, gi, go: got.append(go[0].shape))
    _objective(model(*[x.to(DEV) for x in inputs]), label.to(DEV), True).backward()
    assert len(got) == 1


def _oracle_taps(gold, inputs, label, train):
    """Oracle-A forward of the whole model with the block outputs of every tower recorded (autograd on)."""
    sd = R.clone_state(H.case_state(gold))
    taps = {}
    real = R.snet_forward
    R.snet_forward = lambda sd_, pfx, x, training=True, rnd=None, taps_=None: real(sd_, pfx, x, training, rnd, taps)
    try:
        outs = H.oracle_forward(gold["kind"], sd, [x.clone() for x in inputs], gold["kwargs"], train, 0.0, rnd=R.bf16_round)
    finally:
        R.snet_forward = real
    obj = _objective(outs, label, train)
    pfxs = ["cnn"] if gold["kind"] == "model_single" else ["mri_cnn", "pet_cnn"]
    return obj, pfxs, taps


@pytest.mark.parametrize("name,train", [("model_ad_h4", False), ("model_ad_h4", True), ("model_cnn_ad", False)])
def test_tap_values_against_oracle(name, train):
    gold = H.load_golden(name)
    inputs, label = _inputs(gold)
    model = _model(gold, train)
    log, _ = _observe(model)
    obj = _objective(model(*[x.to(DEV) for x in inputs]), label.to(DEV), train)
    ours = {(e[1], e[2]): e[4] for e in log if e[0] == "fwd" and e[2] != "tower"}
    keys = sorted(ours)
    g_ours = torch.autograd.grad(obj, [ours[k] for k in keys])
    o_obj, pfxs, taps = _oracle_taps(gold, inputs, label, train)
    o_acts = [taps[f"{pfxs[t]}.{TAP_LAYER[n]}"][1] for t, n in keys]
    g_or = torch.autograd.grad(o_obj, o_acts)
    for k, a, ga, oa, og in zip(keys, [ours[k] for k in keys], g_ours, o_acts, g_or):
        ca, ra, cg, rg = H.cosine(a, oa), H.rel_err(a, oa), H.cosine(ga, og), H.rel_err(ga, og)
        print(f"[taps] {name} train={train} {k}: act cos {ca:.6f} rel {ra:.3g}; grad cos {cg:.5f} rel {rg:.3g}")
        assert ca >= ACT_COS and ra <= ACT_REL
        assert cg >= GRAD_COS and rg <= GRAD_REL


def test_block_hooks_fire_under_no_grad_in_eval():
    gold = H.load_golden("model_ad_h4")
    inputs, _ = _inputs(gold)
    model = _model(gold, False).requires_grad_(False)
    log, _ = _observe(model)
    xs = [x.to(DEV) for x in inputs]
    with torch.no_grad():
        model(*xs)
    nograd = {(e[1], e[2]): e[4].clone() for e in log if e[0] == "fwd"}
    log.clear()
    model(*[x.clone().requires_grad_(True) for x in xs])
    withgrad = {(e[1], e[2]): e[4].detach() for e in log if e[0] == "fwd"}
    assert len(nograd) == len(withgrad) == 10
    for k in nograd:
        e = H.rel_err(nograd[k], withgrad[k])
        print(f"[no-grad] {k}: rel {e:.3g}")
        assert e <= NOGRAD_REL


def test_in_place_modification_in_a_hook_is_refused():
    gold = H.load_golden("model_cnn_ad")
    inputs, _ = _inputs(gold)
    model = _model(gold, False)
    def scale_in_place(m, a, o):
        o.mul_(2)

    model.pet_cnn.conv2.register_forward_hook(scale_in_place)
    with pytest.raises(RuntimeError, match="in place"), torch.no_grad():
        model(*[x.to(DEV) for x in inputs])


def test_block_replacing_hook_and_backward_hook_are_refused():
    gold = H.load_golden("model_cnn_ad")
    inputs, _ = _inputs(gold)
    model = _model(gold, False)
    h = model.mri_cnn.conv3.register_forward_hook(lambda m, a, o: o * 2)
    with pytest.raises(NotImplementedError, match="only observe"):
        model(*[x.to(DEV) for x in inputs])
    h.remove()
    model.mri_cnn.conv3.register_full_backward_hook(lambda *a: None)
    with pytest.raises(NotImplementedError, match="autograd.grad"):
        model(*[x.to(DEV) for x in inputs])


def test_hook_inside_a_block_warns_and_the_model_still_runs():
    gold = H.load_golden("model_cnn_ad")
    inputs, _ = _inputs(gold)
    model = _model(gold, False)
    model.mri_cnn.conv2[1].register_forward_hook(lambda m, a, o: None)
    with pytest.warns(UserWarning, match="never fires"):
        model(*[x.to(DEV) for x in inputs])


# ---------------------------------------------------------------------------------------------------------------
# grad_cam
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["model_ad_h4", "model_cnn_ad", "model_single"])
@pytest.mark.parametrize("layer", BLOCKS)
def test_grad_cam_against_oracle(name, layer):
    gold = H.load_golden(name)
    inputs, label = _inputs(gold)
    model = _model(gold, False)
    cams = grad_cam(model, [x.to(DEV) for x in inputs], label.to(DEV), layer=layer, upsample=False, normalize=False)
    o_obj, pfxs, taps = _oracle_taps(gold, inputs, label, False)
    acts = [taps[f"{p}.{TAP_LAYER[layer]}"][1] for p in pfxs]
    grads = torch.autograd.grad(o_obj, acts)
    assert len(cams) == len(pfxs)
    for t, (cam, a, g) in enumerate(zip(cams, acts, grads)):
        _assert_cam_close(cam, _cam_ref(a.detach(), g, None, False), f"[grad_cam] {name} {layer} tower {t}")
    full = grad_cam(model, [x.to(DEV) for x in inputs], label.to(DEV), layer=layer)
    for f in full:
        assert f.shape == (inputs[0].shape[0], 1) + tuple(inputs[0].shape[2:])
        assert float(f.min()) >= 0.0 and float(f.max()) <= 1.0


@pytest.mark.parametrize("train", [False, True])
@pytest.mark.parametrize("layer", ["conv1", "conv3", "conv4"])
def test_grad_cam_launches_and_side_effects(train, layer, monkeypatch):
    gold = H.load_golden("model_ad_h4")
    inputs, label = _inputs(gold)
    model = _model(gold, train)
    model.fc_cls[0].weight.requires_grad_(False)               # a mixed set of flags, restored as found
    flags = {k: p.requires_grad for k, p in model.named_parameters()}
    before = {k: v.clone() for k, v in model.state_dict().items()}
    called = []
    real = L.call

    def spy(name, *args, **kw):
        called.append(kw.get("tag") or name)
        return real(name, *args, **kw)

    monkeypatch.setattr(L, "call", spy)
    grad_cam(model, [x.to(DEV) for x in inputs], label.to(DEV), layer=layer)
    monkeypatch.setattr(L, "call", real)
    assert all(p.grad is None for p in model.parameters())
    assert flags == {k: p.requires_grad for k, p in model.named_parameters()}
    if not train:
        for k, v in model.state_dict().items():
            assert torch.equal(v, before[k]), k
    wgrad = [n for n in called if "wgrad" in n or n.startswith("tmf_conv1_bwd") or n == "tmf_linear_wgrad"]
    assert not wgrad, wgrad
    first = {"conv1": 1, "conv2": 3, "conv3": 5, "conv4": 7}[layer]
    upstream = [n for n in called if "bwd" in n or "dgrad" in n]
    upstream = [n for n in upstream if "@L" in n and int(n.split("@L")[1]) < first] + \
               [n for n in upstream if n == "tmf_conv1_dgrad_fused"]
    assert not upstream, upstream
    assert "tmf_gradcam" in called


def test_grad_cam_determinism():
    gold = H.load_golden("model_ad_h4")
    inputs, label = _inputs(gold)
    model = _model(gold, False)
    a = grad_cam(model, [x.to(DEV) for x in inputs], 1, layer="conv2")
    b = grad_cam(model, [x.to(DEV) for x in inputs], 1, layer="conv2")
    for x, y in zip(a, b):
        assert torch.equal(x, y)


@pytest.mark.parametrize("layer", ["conv3", "conv1"])
def test_grad_cam_full_size(layer):
    gold = H.load_golden("model_ad_full_b8")
    inputs, label = _inputs(gold)
    model = _model(gold, False)
    cams = grad_cam(model, [x.to(DEV) for x in inputs], label.to(DEV), layer=layer, upsample=False, normalize=False)
    o_obj, pfxs, taps = _oracle_taps(gold, inputs, label, False)
    acts = [taps[f"{p}.{TAP_LAYER[layer]}"][1] for p in pfxs]
    grads = torch.autograd.grad(o_obj, acts)
    for t, (cam, a, g) in enumerate(zip(cams, acts, grads)):
        _assert_cam_close(cam, _cam_ref(a.detach(), g, None, False), f"[grad_cam full] {layer} tower {t}")
    full = grad_cam(model, [x.to(DEV) for x in inputs], label.to(DEV), layer=layer)
    assert all(f.shape == (8, 1, 91, 109, 91) and torch.isfinite(f).all() for f in full)

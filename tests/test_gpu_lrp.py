"""Layer-wise relevance propagation through the sNet towers (csrc/lrp.cu, the LRP front of csrc/conv1_dgrad.cu,
transmf_ad_b200.interpret.lrp; DESIGN section 3.9).

Op level: every kernel against a float64 restatement on its own inputs.  s is rounded to bf16 by the kernels, so the ratio
pass is held to one bf16 ulp of s; block 1 to one bf16 ulp of each s term propagated through |x| * (|W|^T |s|).
Model level: against a restatement that runs the sweep on the kernels' own kept activations and rounds s, c and the packs
where the kernels do (tight), and against a float64 restatement of the whole tower (loose; the bound is stated relative to
the measured distance between the two restatements).  Measured values are printed with ``-s``.
"""
import copy

import pytest
import torch
import torch.nn.functional as F

from tests import helpers as H
from transmf_ad_b200 import _lib as L
from transmf_ad_b200 import functional as TF
from transmf_ad_b200.interpret import lrp
from transmf_ad_b200.models import mymodel as M

pytestmark = pytest.mark.gpu
DEV = "cuda"
SLOPE = 0.01
BF16_ULP = 2.0 ** -8                 # relative spacing of bf16 (8 significand bits)
# bounds from the first measurement on a B200, with headroom (measured worst case in brackets)
EMU_REL = 0.01                       # model maps vs the bf16-emulating restatement, relative L2 (3.2e-3; totals 2.9e-4)
F64_FACTOR = 4.0                     # model maps vs float64: at most this times the emulation-to-float64 distance, + 0.02
                                     # (that distance: 0.41-0.65 for epsilon, where max-pool winners that differ in the
                                     # float64 forward move relevance; 0.065-0.13 for zplus)
CONSERVE_REL = 0.02                  # LRP-0 with zero biases: |col_k - col_0| / |col_0| (5.2e-3)


def _bf(t):
    return t.to(torch.bfloat16)


def _stab_div(r, z, eps):
    st = z + torch.where(z >= 0, torch.full_like(z, eps), torch.full_like(z, -eps))
    return torch.where(st != 0, r / torch.where(st != 0, st, torch.ones_like(st)), torch.zeros_like(r))


def _windows(t, pool):
    """(B,C,D,H,W) -> (B,C,Do,Ho,Wo,8) over complete 2x2x2 windows, q = (d,h,w) scan order."""
    B, C, D, H, W = t.shape
    t = t[:, :, :D // 2 * 2, :H // 2 * 2, :W // 2 * 2]
    t = t.reshape(B, C, D // 2, 2, H // 2, 2, W // 2, 2).permute(0, 1, 2, 4, 6, 3, 5, 7)
    return t.reshape(B, C, D // 2, H // 2, W // 2, 8)


def _unwindow(w, shape):
    B, C, D, H, W = shape
    Do, Ho, Wo = D // 2, H // 2, W // 2
    t = w.reshape(B, C, Do, Ho, Wo, 2, 2, 2).permute(0, 1, 2, 5, 3, 6, 4, 7).reshape(B, C, 2 * Do, 2 * Ho, 2 * Wo)
    out = torch.zeros(shape, dtype=w.dtype, device=w.device)
    out[:, :, :2 * Do, :2 * Ho, :2 * Wo] = t
    return out


def _route(R, y, pool, eps):
    """Relevance at the pooled output (B,C,Do,Ho,Wo) -> at the conv output (B,C,D,H,W), float64."""
    if pool == L.POOL_NONE:
        return R
    yw = _windows(y, pool)
    if pool == L.POOL_MAX:
        win = F.one_hot(yw.argmax(-1), 8).to(R.dtype)       # argmax: the first maximum
        return _unwindow(win * R.unsqueeze(-1), y.shape)
    a = F.leaky_relu(yw, SLOPE)
    S = a.sum(-1)
    return _unwindow(a * _stab_div(R, S, eps).unsqueeze(-1), y.shape)


def _ratio_ref(R, y, zp, pool, eps):
    """float64 s of tmf_lrp_ratio: R (B,C,Do,Ho,Wo) float64, y / zp (B,C,D,H,W) float64."""
    return _stab_div(_route(R, y, pool, eps), y if zp is None else zp, eps)


def _ndhwc(t):
    return t.permute(0, 2, 3, 4, 1).contiguous()


def _ncdhw(t):
    return t.permute(0, 4, 1, 2, 3)


def _workspace(name, *args):
    n = int(getattr(L.load(), name)(*args))
    return torch.empty(max(n, 1), dtype=torch.uint8, device=DEV), n


# ---------------------------------------------------------------------------------------------------------------
# op level
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rule", ["epsilon", "zplus"])
@pytest.mark.parametrize("cin,cout,k", [(1, 32, 3), (32, 64, 3), (256, 128, 1)])
def test_fold_pack_against_float64(rule, cin, cout, k):
    g = torch.Generator().manual_seed(cin + cout)
    w = torch.randn(cout, cin, k, k, k, generator=g).to(DEV)
    cb, gamma, beta = (torch.randn(cout, generator=g).to(DEV) for _ in range(3))
    gamma[:2] = -gamma[:2].abs()
    mean, var = torch.randn(cout, generator=g).to(DEV) * 0.1, (torch.rand(cout, generator=g) + 0.5).to(DEV)
    taps = k ** 3
    wf = torch.empty((taps, cout, cin), dtype=torch.bfloat16, device=DEV)
    wd = torch.empty((taps, cin, cout), dtype=torch.bfloat16, device=DEV)
    w32, bias = torch.empty_like(w), torch.empty(cout, device=DEV)
    L.call("tmf_lrp_fold_pack", 1, *[L.ptrs([t]) for t in (w, cb, gamma, beta, mean, var, wf, wd, w32, bias)], cout, cin, k,
           1e-5, TF.LRP_RULES[rule])
    scale = gamma.double() / torch.sqrt(var.double() + 1e-5)
    ref = w.double() * scale.view(-1, 1, 1, 1, 1)
    if rule == "zplus":
        ref = ref.clamp_min(0)
    assert torch.allclose(w32.double(), ref, rtol=1e-6, atol=1e-7)
    assert torch.allclose(bias.double(), (cb.double() - mean.double()) * scale + beta.double(), rtol=1e-5, atol=1e-6)
    r = ref.reshape(cout, cin, taps)
    assert torch.allclose(wf.double(), r.permute(2, 0, 1), rtol=BF16_ULP, atol=0)
    assert torch.allclose(wd.double(), r.flip(2).permute(2, 1, 0), rtol=BF16_ULP, atol=0)


def _ratio_inputs(B, D, H, W, C, pool, up32, seed):
    g = torch.Generator().manual_seed(seed)
    p = 1 if pool == L.POOL_NONE else 2
    Do, Ho, Wo = D // p, H // p, W // p
    y = torch.randint(-3, 4, (B, D, H, W, C), generator=g).float() * 0.25     # ties, zeros and negative denominators
    y[0, 0] = torch.randn(H, W, C, generator=g)
    ua = torch.randn(B, Do, Ho, Wo, C, generator=g)
    uc = torch.randn(B, Do, Ho, Wo, C, generator=g)
    zp = torch.randn(B, D, H, W, C, generator=g).abs()
    zp[..., 0] = 0.0
    cast = (lambda t: t.to(DEV)) if up32 else (lambda t: _bf(t).to(DEV))
    return cast(ua), cast(uc), _bf(y).to(DEV), _bf(zp).to(DEV)


def _run_ratio(ua, uc, y, zp, pool, eps, up32):
    ng = len(y)
    B, D, H, W, C = y[0].shape
    s = [torch.empty_like(t) for t in y]
    tot = [torch.full((B, 8), float("nan"), device=DEV) for _ in y]
    ws, n = _workspace("tmf_lrp_ratio_workspace_bytes", ng, B, D, H, W, C, pool)
    L.call("tmf_lrp_ratio", ng, L.ptrs(ua), L.ptrs(uc), int(up32), L.ptrs(y), L.ptrs(zp), L.ptrs(s), L.ptrs(tot), 3, B, D, H,
           W, C, pool, SLOPE, float(eps), L.ptr(ws), n)
    return s, tot


@pytest.mark.parametrize("pool", [L.POOL_MAX, L.POOL_NONE, L.POOL_AVG])
@pytest.mark.parametrize("shape", [(2, 9, 11, 7, 32), (1, 6, 5, 13, 64), (3, 4, 4, 4, 8)])
@pytest.mark.parametrize("eps,zplus,up32", [(0.0, False, False), (1e-2, False, True), (1e-6, True, False)])
def test_ratio_against_float64(pool, shape, eps, zplus, up32):
    B, D, H, W, C = shape
    ua, uc, y, zp = _ratio_inputs(B, D, H, W, C, pool, up32, sum(shape) + pool)
    zp = zp if zplus else None
    s, tot = _run_ratio([ua], [uc], [y], None if zp is None else [zp], pool, eps, up32)
    R = _ncdhw(ua.double() * uc.double())
    ref = _ratio_ref(R, _ncdhw(y.double()), None if zp is None else _ncdhw(zp.double()), pool, eps)
    got = _ncdhw(s[0].double())
    err = (got - ref).abs()
    bound = BF16_ULP * ref.abs() + 1e-30
    print(f"[ratio] pool={pool} {shape} eps={eps} zplus={zplus}: max err / ulp = {float((err / bound).max()):.3f}")
    assert bool((err <= bound).all())
    assert torch.isfinite(s[0].float()).all()
    tref = R.sum(dim=(1, 2, 3, 4))
    assert torch.allclose(tot[0][:, 3].double(), tref, rtol=1e-5, atol=1e-5 * float(R.abs().sum()) / B)
    assert torch.isnan(tot[0][:, 0]).all()                   # only the requested column is written


@pytest.mark.parametrize("pool", [L.POOL_MAX, L.POOL_AVG])
def test_ratio_two_towers_equal_two_launches(pool):
    a = _ratio_inputs(2, 9, 11, 7, 32, pool, False, 1)
    b = _ratio_inputs(2, 9, 11, 7, 32, pool, False, 2)
    both = _run_ratio([a[0], b[0]], [a[1], b[1]], [a[2], b[2]], [a[3], b[3]], pool, 1e-6, False)
    for t, inp in enumerate((a, b)):
        one = _run_ratio([inp[0]], [inp[1]], [inp[2]], [inp[3]], pool, 1e-6, False)
        assert torch.equal(both[0][t], one[0][0]) and torch.equal(both[1][t][:, 3], one[1][0][:, 3])


def _conv1_inputs(B, D, H, W, seed, zplus):
    g = torch.Generator().manual_seed(seed)
    C = 32
    a1 = _bf(torch.randn(B, D // 2, H // 2, W // 2, C, generator=g)).to(DEV)
    c1 = _bf(torch.randn(B, D // 2, H // 2, W // 2, C, generator=g)).to(DEV)
    y = torch.randn(B, D, H, W, C, generator=g)
    y[:, :2] = torch.randint(-2, 3, (B, 2, H, W, C), generator=g).float() * 0.5    # ties and zero denominators
    y = _bf(y).to(DEV)
    zp = _bf(torch.randn(B, D, H, W, C, generator=g).abs() + 0.1).to(DEV) if zplus else None
    w = (torch.randn(C, 1, 3, 3, 3, generator=g) * 0.3)
    if zplus:
        w = w.clamp_min(0)
    x = torch.randn(B, 1, D, H, W, generator=g).to(DEV)
    return a1, c1, y, zp, w.to(DEV), x


def _run_conv1(inps, eps, impl):
    ng = len(inps)
    a1, c1, y, zp, w, x = zip(*inps)
    B, D, H, W, C = y[0].shape
    rx = [torch.empty((B, 1, D, H, W), device=DEV) for _ in range(ng)]
    tot = [torch.full((B, 8), float("nan"), device=DEV) for _ in range(ng)]
    ws, n = _workspace("tmf_lrp_conv1_workspace_bytes", ng, impl, B, D, H, W, C)
    L.call("tmf_lrp_conv1", ng, L.ptrs(a1), L.ptrs(c1), L.ptrs(y), L.ptrs(None if zp[0] is None else zp), L.ptrs(w),
           L.ptrs(x), L.ptrs(rx), L.ptrs(tot), B, D, H, W, C, float(eps), impl, L.ptr(ws), n)
    return rx, tot


@pytest.mark.parametrize("impl", [L.CONV_UMMA, L.CONV_DIRECT])
@pytest.mark.parametrize("rule", ["epsilon", "zplus"])
@pytest.mark.parametrize("shape", [(2, 9, 11, 7), (1, 20, 35, 128), (2, 16, 16, 33)])
def test_lrp_conv1_against_float64(impl, rule, shape):
    B, D, H, W = shape
    zplus = rule == "zplus"
    eps = 1e-6 if zplus else 1e-3
    inp = _conv1_inputs(B, D, H, W, sum(shape), zplus)
    a1, c1, y, zp, w, x = inp
    rx, tot = _run_conv1([inp], eps, impl)
    R = _ncdhw(a1.double() * c1.double())
    s = _ratio_ref(R, _ncdhw(y.double()), None if zp is None else _ncdhw(zp.double()), L.POOL_MAX, eps)
    c = F.conv_transpose3d(s, w.double(), padding=1)
    ref = x.double() * c
    err = (rx[0].double() - ref).abs()
    bound = BF16_ULP * x.double().abs() * F.conv_transpose3d(s.abs(), w.double().abs(), padding=1) + 1e-6 * float(ref.abs().max())
    print(f"[lrp_conv1] impl={impl} {rule} {shape}: max err / bound = {float((err / bound).max()):.3f}")
    assert bool((err <= bound).all())
    r_tot = R[:, :, :D // 2, :H // 2, :W // 2].sum(dim=(1, 2, 3, 4))
    assert torch.allclose(tot[0][:, 6].double(), r_tot, rtol=1e-5, atol=1e-5 * float(R.abs().sum()) / B)
    assert torch.allclose(tot[0][:, 7].double(), rx[0].double().sum(dim=(1, 2, 3, 4)), rtol=1e-5,
                          atol=1e-5 * float(rx[0].abs().sum()) / B)


@pytest.mark.parametrize("impl", [L.CONV_UMMA, L.CONV_DIRECT])
@pytest.mark.parametrize("rule", ["epsilon", "zplus"])
def test_lrp_conv1_two_towers_equal_two_launches(impl, rule):
    a = _conv1_inputs(2, 13, 18, 21, 5, rule == "zplus")
    b = _conv1_inputs(2, 13, 18, 21, 6, rule == "zplus")
    both = _run_conv1([a, b], 1e-6, impl)
    for t, inp in enumerate((a, b)):
        one = _run_conv1([inp], 1e-6, impl)
        assert torch.equal(both[0][t], one[0][0]) and torch.equal(both[1][t][:, 6:], one[1][0][:, 6:])


def test_saliency_instance_unchanged_by_the_lrp_front():
    """The saliency instance of the block-1 kernel still agrees with its CUDA-core path (tests/test_gpu_input_grad.py covers
    it in full); both instances live in one template."""
    g = torch.Generator().manual_seed(3)
    B, D, H, W, C = 2, 10, 12, 9, 32
    dout = _bf(torch.randn(B, D // 2, H // 2, W // 2, C, generator=g)).to(DEV)
    y = _bf(torch.randn(B, D, H, W, C, generator=g)).to(DEV)
    coef = torch.cat([torch.rand(C, generator=g) + 0.5, torch.randn(C, generator=g) * 0.1, torch.randn(C, generator=g) * 0.1,
                      torch.rand(C, generator=g) + 0.5]).to(DEV)
    bcoef = (torch.randn(2 * C, generator=g) * 0.01).to(DEV)
    w = torch.randn(C, 1, 3, 3, 3, generator=g).to(DEV)
    outs = []
    for impl in (L.CONV_UMMA, L.CONV_DIRECT):
        dx = torch.empty((B, 1, D, H, W), device=DEV)
        ws, n = _workspace("tmf_conv1_dgrad_fused_workspace_bytes", 1, impl, B, D, H, W, C)
        L.call("tmf_conv1_dgrad_fused", 1, L.ptrs([dout]), L.ptrs([y]), L.ptrs([coef]), L.ptrs([bcoef]), L.ptrs([w]),
               L.ptrs([dx]), B, D, H, W, C, SLOPE, impl, L.ptr(ws), n)
        outs.append(dx)
    assert torch.allclose(outs[0], outs[1], rtol=1e-4, atol=1e-5 * float(outs[1].abs().max()))


# ---------------------------------------------------------------------------------------------------------------
# model level
# ---------------------------------------------------------------------------------------------------------------
def _model(gold):
    model = getattr(M, gold["kind"])(**gold["kwargs"])
    model.load_state_dict(H.case_state(gold), strict=True)
    model = model.to(DEV).eval()
    H.set_head_dropout(model, 0.0)
    return model


def _inputs(gold):
    mri, pet, label = H.case_inputs(gold)
    return ((mri,) if gold["kind"] == "model_single" else (mri, pet)), label


def _towers(model):
    return [m for m in model.modules() if isinstance(m, M.sNet)]


def _capture(model, inputs, target):
    """What lrp's forward produces: per tower the kept (a, y) pairs and the seed (a_T, df/da_T)."""
    towers = _towers(model)
    leaves = {}

    def leaf(m, args, out):
        leaves[m] = out.detach().requires_grad_(True)
        return leaves[m]

    hs = [t.register_forward_hook(leaf) for t in towers]
    flags = [(p, p.requires_grad) for p in model.parameters()]
    for p, _ in flags:
        p.requires_grad_(False)
    for t in towers:
        t._lrp_keep = []
    try:
        outs = model(*inputs)
        logits = outs[0] if isinstance(outs, tuple) else outs
        obj = logits.gather(1, target.view(-1, 1)).sum()
        acts = [leaves[t] for t in towers]
        grads = torch.autograd.grad(obj, acts)
        kept = [t._lrp_keep for t in towers]
    finally:
        for h in hs:
            h.remove()
        for p, f in flags:
            p.requires_grad_(f)
        for t in towers:
            t._lrp_keep = None
    return kept, [(a.detach().double(), g.double()) for a, g in zip(acts, grads)]


def _fold64(conv, bn, rule, emulate):
    if emulate:                                       # the kernels' fp32 fold
        scale = bn.weight.detach() * torch.rsqrt(bn.running_var + bn.eps)
        w = (conv.weight.detach() * scale.view(-1, 1, 1, 1, 1)).double()
    else:
        scale = bn.weight.detach().double() / torch.sqrt(bn.running_var.double() + bn.eps)
        w = conv.weight.detach().double() * scale.view(-1, 1, 1, 1, 1)
    b = (conv.bias.detach().double() - bn.running_mean.double()) * scale.double() + bn.bias.detach().double()
    return w, b


def _sweep(tower, acts, ys, seed, x, rule, eps, emulate):
    """float64 LRP sweep.  acts[l] / ys[l]: (B,C,...) float64 input activation / pre-activation of layer l."""
    spec = tower._spec
    rnd = (lambda t: t.to(torch.bfloat16).double()) if emulate else (lambda t: t)
    aT, g = seed
    R = aT * g
    tot = [R.sum(dim=(1, 2, 3, 4))]
    for l in range(6, -1, -1):
        cin, cout, ks, pool = spec.layers[l]
        conv, bn = tower._units()[l]
        w, _ = _fold64(conv, bn, rule, emulate)
        if rule == "zplus":
            w = w.clamp_min(0)
        if l > 0:
            w = rnd(w)
        z = ys[l]
        if rule == "zplus":
            z = F.conv3d(acts[l], w, padding=ks // 2)
            z = rnd(z)
        s = rnd(_stab_div(_route(R, ys[l], pool, eps), z, eps))
        c = F.conv_transpose3d(s, w, padding=ks // 2)
        if l > 0:
            c = rnd(c)
        R = acts[l] * c if l > 0 else x * c
        tot.append(R.sum(dim=(1, 2, 3, 4)))
    return R, torch.stack(tot, 1)


def _forward64(tower, x):
    acts, ys, a = [], [], x
    for l, (cin, cout, ks, pool) in enumerate(tower._spec.layers):
        conv, bn = tower._units()[l]
        w, b = _fold64(conv, bn, "epsilon", False)
        acts.append(a)
        y = F.conv3d(a, w, b, padding=ks // 2)
        ys.append(y)
        a = F.leaky_relu(y, SLOPE)
        a = F.max_pool3d(a, 2) if pool == L.POOL_MAX else (F.avg_pool3d(a, 2) if pool == L.POOL_AVG else a)
    return acts, ys


def _rel(a, b):
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


@pytest.mark.parametrize("name", ["model_ad_h4", "model_cnn_ad", "model_ad_full_b2"])
@pytest.mark.parametrize("rule", ["epsilon", "zplus"])
def test_lrp_against_restatements(name, rule):
    gold = H.load_golden(name)
    inputs, label = _inputs(gold)
    model = _model(gold)
    xs = [x.to(DEV) for x in inputs]
    tgt = label.to(DEV)
    eps = 1e-6 if rule == "zplus" else 1e-2
    res = lrp(model, xs, tgt, rule=rule, eps=eps)
    kept, seeds = _capture(model, xs, tgt)
    for t, tower in enumerate(_towers(model)):
        acts = [kept[t][0][0].double()] + [_ncdhw(a.double()) for a, _ in kept[t][1:]]
        ys = [_ncdhw(y.double()) for _, y in kept[t]]
        emu, emu_tot = _sweep(tower, acts, ys, seeds[t], xs[t].double(), rule, eps, True)
        a64, y64 = _forward64(tower, xs[t].double())
        f64, _ = _sweep(tower, a64, y64, seeds[t], xs[t].double(), rule, eps, False)
        got = res.maps[t].double()
        r_emu, r_f64, d = _rel(got, emu), _rel(got, f64), _rel(emu, f64)
        tr = _rel(res.totals[t].double(), emu_tot)
        print(f"[lrp] {name} {rule} tower {t}: vs emulation {r_emu:.2e}, vs float64 {r_f64:.2e} "
              f"(emulation vs float64 {d:.2e}), totals vs emulation {tr:.2e}")
        assert res.maps[t].shape == xs[t].shape and res.totals[t].shape == (xs[t].shape[0], 8)
        assert r_emu < EMU_REL and tr < EMU_REL
        assert r_f64 < F64_FACTOR * d + 0.02
        assert torch.allclose(res.totals[t][:, 7].double(), got.sum(dim=(1, 2, 3, 4)), rtol=1e-4,
                              atol=1e-5 * float(got.abs().sum()) / got.shape[0])


def test_lrp0_conserves_relevance_with_zero_biases():
    gold = H.load_golden("model_cnn_ad")
    inputs, label = _inputs(gold)
    model = _model(gold)
    with torch.no_grad():
        for t in _towers(model):
            for conv, bn in t._units():
                conv.bias.zero_()
                bn.bias.zero_()
                bn.running_mean.zero_()
    res = lrp(model, [x.to(DEV) for x in inputs], label.to(DEV), rule="epsilon", eps=0.0)
    for t, tot in enumerate(res.totals):
        tot = tot.double()
        dev = ((tot - tot[:, :1]).abs() / tot[:, :1].abs()).max()
        print(f"[conservation] tower {t}: max |col_k - col_0| / |col_0| = {float(dev):.2e}")
        assert float(dev) < CONSERVE_REL
        m = res.maps[t].double().sum(dim=(1, 2, 3, 4))
        assert torch.allclose(tot[:, 7], m, rtol=1e-4, atol=1e-6 * float(res.maps[t].abs().sum()))


def test_lrp_determinism_and_side_effects(monkeypatch):
    gold = H.load_golden("model_ad_h4")
    inputs, label = _inputs(gold)
    model = _model(gold)
    model.fc_cls[0].weight.requires_grad_(False)
    flags = {k: p.requires_grad for k, p in model.named_parameters()}
    before = {k: v.clone() for k, v in model.state_dict().items()}
    xs = [x.to(DEV) for x in inputs]
    called = []
    real = L.call

    def spy(name, *args, **kw):
        called.append(kw.get("tag") or name)
        return real(name, *args, **kw)

    monkeypatch.setattr(L, "call", spy)
    a = lrp(model, xs, label.to(DEV), rule="zplus")
    monkeypatch.setattr(L, "call", real)
    b = lrp(model, xs, label.to(DEV), rule="zplus")
    for x, y in zip(a.maps + a.totals, b.maps + b.totals):
        assert torch.equal(x, y)
    assert all(p.grad is None for p in model.parameters())
    assert flags == {k: p.requires_grad for k, p in model.named_parameters()}
    assert not model.training
    for k, v in model.state_dict().items():
        assert torch.equal(v, before[k]), k
    bad = [n for n in called if "wgrad" in n or n.startswith("tmf_conv1_bwd") or n.startswith("tmf_bn_act_pool_bwd")
           or n == "tmf_conv1_dgrad_fused"]
    assert not bad, bad
    assert called.count("tmf_lrp_conv1") == 1                  # both towers in one launch sequence
    n = lrp(model, xs, label.to(DEV), rule="zplus", normalize=True)
    for m, raw in zip(n.maps, a.maps):
        peak = raw.abs().amax(dim=(1, 2, 3, 4), keepdim=True)
        assert torch.allclose(m, raw / peak, rtol=1e-6, atol=0)


def test_observing_block_hook_leaves_maps_unchanged():
    gold = H.load_golden("model_ad_h4")
    inputs, label = _inputs(gold)
    model = _model(gold)
    xs = [x.to(DEV) for x in inputs]
    a = lrp(model, xs, label.to(DEV))
    seen = []
    hs = [t.conv2.register_forward_hook(lambda m, i, o: seen.append(o.shape)) for t in _towers(model)]
    b = lrp(model, xs, label.to(DEV))
    for h in hs:
        h.remove()
    assert len(seen) == 2
    for x, y in zip(a.maps + a.totals, b.maps + b.totals):
        assert torch.equal(x, y)


def test_train_step_after_lrp_is_bitwise_the_plain_one():
    gold = H.load_golden("model_cnn_ad")
    inputs, label = _inputs(gold)
    xs = [x.to(DEV) for x in inputs]

    def step(model):
        model.train()
        outs = model(*xs)
        loss = H.losses(outs if isinstance(outs, tuple) else (outs,), label.to(DEV))[2]
        loss.backward()
        return [p.grad.clone() for p in model.parameters() if p.grad is not None], \
            [b.clone() for b in model.buffers()], loss.detach()

    plain = _model(gold)
    other = copy.deepcopy(plain)
    lrp(other, xs, label.to(DEV), rule="zplus")
    lrp(other, xs, label.to(DEV), rule="epsilon")
    ga, ba, la = step(plain)
    gb, bb, lb = step(other)
    assert torch.equal(la, lb)
    for x, y in zip(ga + ba, gb + bb):
        assert torch.equal(x, y)


def test_lrp_refuses_training_mode_on_the_gpu():
    gold = H.load_golden("model_cnn_ad")
    inputs, label = _inputs(gold)
    model = _model(gold).train()
    with pytest.raises(ValueError, match="eval"):
        lrp(model, [x.to(DEV) for x in inputs], label.to(DEV))

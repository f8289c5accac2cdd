"""Exact-arithmetic tests of the MiSePyNet / Mnet kernels (csrc/mnet_ops.cu): slice and spatial convolutions, BatchNorm
+ ReLU and max pooling, at the model's own layer shapes (B = 2, 91 x 109 x 91) and at the edges of their launch
geometry (tests/mnet_exact.py).

Operands are small integers or short dyadic significands whose whole-layer sums stay below 2^24 quanta: a correct
kernel reproduces the float64 reference bit for bit whatever its thread split, so one dropped line, one clipped tap or
one misrouted window fails on the element it touches.  Every output, statistics buffer and workspace is poisoned with
0xFF bytes before each call, every output sits inside guard bands, every call runs twice and must give the same bits,
every statistics buffer must have all TMF_STAT_ROWS rows written, and every pool index must lie inside its window.

One Gaussian case per convolution family checks the rounding that grid data cannot see against a per-element bound
c 2^-24 (|a| * |w|), c twice the longest fp32 chain of the kernel; one chained Gaussian case per convolution kind
runs mnet_functional's autograd functions against float64 torch autograd, in train and in eval mode.

NaN is left out of the BatchNorm + ReLU cases on purpose: the kernels' ReLU is fmaxf(z, 0), which maps NaN to 0, and
the backward mask z > 0 is false for NaN, where torch's ReLU propagates NaN."""
import math
import zlib

import pytest
import torch
import torch.nn.functional as F

from tests import conv_exact as X
from tests import mnet_exact as M
from tests.test_gpu_conv_exact import run_twice, workspace
from transmf_ad_b200 import _lib as L
from transmf_ad_b200 import mnet_functional as MF

pytestmark = pytest.mark.gpu
DEV = "cuda"
U = 2.0 ** -24


def gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def case_gen(cid):
    return gen(zlib.crc32(cid.encode()))


def f32(t):
    return t.float().contiguous()


def guarded(shape, dtype=torch.float32):
    return X.Guarded(tuple(shape), dtype, DEV)


def check(got, want, what):
    err = X.mismatch(got.double(), want)
    assert not err, f"{what}: {err}"


def untouched(g, what):
    assert bool((g.buf == 0xFF).all()), f"{what}: written although NULL was passed"


def check_rows(rows, s1, s2, what):
    """All TMF_STAT_ROWS rows written (finite after poisoning); the row totals are the reference sums bit for bit."""
    assert rows.shape[0] == L.stat_rows()
    assert bool(torch.isfinite(rows).all()), f"{what}: statistics rows left unwritten"
    C = s1.shape[0]
    tot = rows.sum(0)
    check(tot[:C], s1, f"{what}: first sums")
    check(tot[C:], s2, f"{what}: second sums")


# ---------------------------------------------------------------------------------------------------------------
# slice convolution
@pytest.mark.parametrize("case", M.LINE_CASES, ids=[c[0] for c in M.LINE_CASES])
def test_line_conv_exact(case):
    cid, n, cin, P, Ln, k = case
    Lo = Ln - k + 1
    x, w, b, dy = M.line_operands(case, case_gen(cid), DEV)
    x32, w32, b32, dy32 = f32(x), f32(w), f32(b), f32(dy)
    y = guarded((n, M.LC_CO, P, Lo))
    got = run_twice([y], lambda: L.call("tmf_line_conv_fwd", L.ptr(x32), L.ptr(w32), L.ptr(b32), L.ptr(y.t), n, cin, P,
                                        Ln, k))
    check(got[0], M.line_fwd_ref(x, w, b), f"{cid} forward")
    dx = guarded((n, cin, P, Ln))
    got = run_twice([dx], lambda: L.call("tmf_line_conv_dgrad", L.ptr(dy32), L.ptr(w32), L.ptr(dx.t), n, cin, P, Ln, k))
    check(got[0], M.line_dgrad_ref(dy, w, Ln), f"{cid} dgrad")
    del y, dx, got
    ws = workspace(L.load().tmf_line_conv_wgrad_workspace_bytes(cin, k))
    dw, db = guarded((M.LC_CO, cin, k)), guarded((M.LC_CO,))

    def wgrad(dbp):
        ws.fill_(0xFF)
        L.call("tmf_line_conv_wgrad", L.ptr(dy32), L.ptr(x32), L.ptr(dw.t), L.ptr(dbp), n, cin, P, Ln, k, L.ptr(ws),
               ws.numel())

    ref_dw, ref_db = M.line_wgrad_ref(dy, x, k)
    got = run_twice([dw, db], lambda: wgrad(db.t))
    check(got[0], ref_dw, f"{cid} wgrad dw")
    check(got[1], ref_db, f"{cid} wgrad db")
    got = run_twice([dw, db], lambda: wgrad(None))
    check(got[0], ref_dw, f"{cid} wgrad dw (db NULL)")
    untouched(db, f"{cid} wgrad db")


# ---------------------------------------------------------------------------------------------------------------
# spatial convolution
@pytest.mark.parametrize("case", M.CONV_CASES, ids=[c[0] for c in M.CONV_CASES])
def test_conv2d_exact(case):
    cid, n, cin, cout, X_, Y_, kh, kw, s = case
    Xo, Yo = M.conv2d_out(X_, Y_, kh, kw, s)
    x, w, b, dy = M.conv2d_operands(case, case_gen(cid), DEV)
    x32, w32, b32, dy32 = f32(x), f32(w), f32(b), f32(dy)
    args = (n, cin, X_, Y_, cout, kh, kw, s)
    y = guarded((n, cout, Xo, Yo))
    got = run_twice([y], lambda: L.call("tmf_conv2d_fwd", L.ptr(x32), L.ptr(w32), L.ptr(b32), L.ptr(y.t), *args))
    check(got[0], M.conv2d_fwd_ref(x, w, b, s), f"{cid} forward")
    dx = guarded((n, cin, X_, Y_))
    got = run_twice([dx], lambda: L.call("tmf_conv2d_dgrad", L.ptr(dy32), L.ptr(w32), L.ptr(dx.t), *args))
    check(got[0], M.conv2d_dgrad_ref(dy, w, s, X_, Y_), f"{cid} dgrad")
    dw, db = guarded((cout, cin, kh, kw)), guarded((cout,))
    ref_dw, ref_db = M.conv2d_wgrad_ref(dy, x, kh, kw, s)
    got = run_twice([dw, db], lambda: L.call("tmf_conv2d_wgrad", L.ptr(dy32), L.ptr(x32), L.ptr(dw.t), L.ptr(db.t), *args))
    check(got[0], ref_dw, f"{cid} wgrad dw")
    check(got[1], ref_db, f"{cid} wgrad db")
    got = run_twice([dw, db], lambda: L.call("tmf_conv2d_wgrad", L.ptr(dy32), L.ptr(x32), L.ptr(dw.t), L.ptr(None), *args))
    check(got[0], ref_dw, f"{cid} wgrad dw (db NULL)")
    untouched(db, f"{cid} wgrad db")


# ---------------------------------------------------------------------------------------------------------------
# BatchNorm + ReLU
@pytest.mark.parametrize("case", M.BN_CASES, ids=[c[0] for c in M.BN_CASES])
def test_bn_relu_exact(case):
    """Statistics rows, forward, backward sums, and the apply pass with training bcoef and with eval's zeros."""
    cid, n, C, S = case
    x, coef, bcoef, dout = M.bn_operands(case, case_gen(cid), DEV)
    x32, dout32, coef32 = f32(x), f32(dout), f32(coef.reshape(-1))
    rows = guarded((L.stat_rows(), 2 * C), torch.float64)
    got = run_twice([rows], lambda: L.call("tmf_nchw_bn_stats", L.ptr(x32), L.ptr(rows.t), n, C, S))
    check_rows(got[0], *M.bn_stats_ref(x), f"{cid} stats")
    out = guarded((n, C, S))
    got = run_twice([out], lambda: L.call("tmf_nchw_bn_relu_fwd", L.ptr(x32), L.ptr(coef32), L.ptr(out.t), n, C, S))
    check(got[0], M.bn_relu_fwd_ref(x, coef), f"{cid} forward")
    got = run_twice([rows], lambda: L.call("tmf_nchw_bn_relu_bwd_reduce", L.ptr(dout32), L.ptr(x32), L.ptr(coef32),
                                           L.ptr(rows.t), n, C, S))
    check_rows(got[0], *M.bn_bwd_sums_ref(dout, x, coef)[:2], f"{cid} backward sums")
    for mode, bc in (("train", bcoef), ("eval", torch.zeros_like(bcoef))):
        bc32 = f32(bc.reshape(-1))
        got = run_twice([out], lambda: L.call("tmf_nchw_bn_relu_bwd_apply", L.ptr(dout32), L.ptr(x32), L.ptr(coef32),
                                              L.ptr(bc32), L.ptr(out.t), n, C, S))
        check(got[0], M.bn_apply_ref(dout, x, coef, bc), f"{cid} apply ({mode})")


# ---------------------------------------------------------------------------------------------------------------
# max pool
@pytest.mark.parametrize("case", M.POOL_CASES, ids=[c[0] for c in M.POOL_CASES])
def test_maxpool_exact(case):
    cid, NC, X_, Y_, ph, pw, _ = case
    Xo, Yo = X_ // ph, Y_ // pw
    x, dy = M.pool_operands(case, case_gen(cid), DEV)
    x32, dy32 = f32(x), f32(dy)
    y, idx = guarded((NC, Xo, Yo)), guarded((NC, Xo, Yo), torch.uint8)
    got = run_twice([y, idx], lambda: L.call("tmf_maxpool2d_fwd", L.ptr(x32), L.ptr(y.t), L.ptr(idx.t), NC, X_, Y_, ph, pw))
    ref_y, ref_idx = M.maxpool_fwd_ref(x, ph, pw)
    assert bool((got[1] < ph * pw).all()), f"{cid}: an index outside its window"
    check(got[0], ref_y, f"{cid} forward")
    assert torch.equal(got[1].long(), ref_idx), f"{cid} idx: {X.mismatch(got[1].long(), ref_idx)}"
    dx = guarded((NC, X_, Y_))
    got = run_twice([dx], lambda: L.call("tmf_maxpool2d_bwd", L.ptr(dy32), L.ptr(idx.t), L.ptr(dx.t), NC, X_, Y_, ph, pw))
    check(got[0], M.maxpool_bwd_ref(dy, ref_idx, ph, pw, X_, Y_), f"{cid} backward")


# ---------------------------------------------------------------------------------------------------------------
# Gaussian data: the rounding of each convolution family
def rn(g, *shape):
    """Gaussian fp32 values, as float64."""
    return torch.randn(shape, generator=g, device=DEV, dtype=torch.float64).float().double()


def within(got, ref, bound, what):
    err = (got.double() - ref).abs()
    assert bool((err <= bound).all()), f"{what}: worst {float((err / bound).max()):.3g} x bound"


def test_line_conv_gaussian_within_rounding_bound():
    """Chains: forward Cin*k, dgrad 8*k, wgrad Lo per line + ceil(lines/592) lines per block + 592 block rows."""
    n, cin, P, Ln, k = 2, 8, 3000, 61, 31
    Lo = Ln - k + 1
    g = gen(61)
    x, dy = rn(g, n, cin, P, Ln), rn(g, n, M.LC_CO, P, Lo)
    w, b = (rn(g, M.LC_CO, cin, k) * (cin * k) ** -0.5).float().double(), (rn(g, M.LC_CO) * 0.1).float().double()
    x32, w32, b32, dy32 = f32(x), f32(w), f32(b), f32(dy)          # held: the launches read them asynchronously
    y = torch.empty((n, M.LC_CO, P, Lo), device=DEV)
    L.call("tmf_line_conv_fwd", L.ptr(x32), L.ptr(w32), L.ptr(b32), L.ptr(y), n, cin, P, Ln, k)
    within(y, M.line_fwd_ref(x, w, b), 2 * cin * k * U * M.line_fwd_ref(x.abs(), w.abs(), b.abs()), "forward")
    dx = torch.empty((n, cin, P, Ln), device=DEV)
    L.call("tmf_line_conv_dgrad", L.ptr(dy32), L.ptr(w32), L.ptr(dx), n, cin, P, Ln, k)
    within(dx, M.line_dgrad_ref(dy, w, Ln), 2 * M.LC_CO * k * U * M.line_dgrad_ref(dy.abs(), w.abs(), Ln), "dgrad")
    ws = workspace(L.load().tmf_line_conv_wgrad_workspace_bytes(cin, k))
    dw, db = torch.empty((M.LC_CO, cin, k), device=DEV), torch.empty(M.LC_CO, device=DEV)
    L.call("tmf_line_conv_wgrad", L.ptr(dy32), L.ptr(x32), L.ptr(dw), L.ptr(db), n, cin, P, Ln, k, L.ptr(ws),
           ws.numel())
    c = 2 * (Lo + math.ceil(n * P / M.LINE_WGRAD_BLOCKS) + M.LINE_WGRAD_BLOCKS)
    ref_dw, ref_db = M.line_wgrad_ref(dy, x, k)
    abs_dw, abs_db = M.line_wgrad_ref(dy.abs(), x.abs(), k)
    within(dw, ref_dw, c * U * abs_dw, "wgrad dw")
    within(db, ref_db, c * U * abs_db, "wgrad db")


def test_conv2d_gaussian_within_rounding_bound():
    """conv1.0 of spatial_cnn (8 -> 16, 11 x 11, stride 2 on 91 x 109).  Chains: forward Cin*kh*kw, dgrad
    Cout*ceil(kh/s)*ceil(kw/s), wgrad ceil(N*Xo*Yo/32) per lane + 5 shuffle levels."""
    n, cin, cout, X_, Y_, kh, kw, s = 2, 8, 16, 91, 109, 11, 11, 2
    Xo, Yo = M.conv2d_out(X_, Y_, kh, kw, s)
    g = gen(62)
    x, dy = rn(g, n, cin, X_, Y_), rn(g, n, cout, Xo, Yo)
    w, b = (rn(g, cout, cin, kh, kw) * (cin * kh * kw) ** -0.5).float().double(), (rn(g, cout) * 0.1).float().double()
    x32, w32, b32, dy32 = f32(x), f32(w), f32(b), f32(dy)          # held: the launches read them asynchronously
    args = (n, cin, X_, Y_, cout, kh, kw, s)
    y = torch.empty((n, cout, Xo, Yo), device=DEV)
    L.call("tmf_conv2d_fwd", L.ptr(x32), L.ptr(w32), L.ptr(b32), L.ptr(y), *args)
    within(y, M.conv2d_fwd_ref(x, w, b, s), 2 * cin * kh * kw * U * M.conv2d_fwd_ref(x.abs(), w.abs(), b.abs(), s),
           "forward")
    dx = torch.empty((n, cin, X_, Y_), device=DEV)
    L.call("tmf_conv2d_dgrad", L.ptr(dy32), L.ptr(w32), L.ptr(dx), *args)
    c = 2 * cout * -(-kh // s) * -(-kw // s)
    within(dx, M.conv2d_dgrad_ref(dy, w, s, X_, Y_), c * U * M.conv2d_dgrad_ref(dy.abs(), w.abs(), s, X_, Y_), "dgrad")
    dw, db = torch.empty((cout, cin, kh, kw), device=DEV), torch.empty(cout, device=DEV)
    L.call("tmf_conv2d_wgrad", L.ptr(dy32), L.ptr(x32), L.ptr(dw), L.ptr(db), *args)
    c = 2 * (math.ceil(n * Xo * Yo / 32) + 5)
    ref_dw, ref_db = M.conv2d_wgrad_ref(dy, x, kh, kw, s)
    abs_dw, abs_db = M.conv2d_wgrad_ref(dy.abs(), x.abs(), kh, kw, s)
    within(dw, ref_dw, c * U * abs_dw, "wgrad dw")
    within(db, ref_db, c * U * abs_db, "wgrad db")


# ---------------------------------------------------------------------------------------------------------------
# Gaussian chain through mnet_functional: Conv3d + BatchNorm3d + ReLU + MaxPool3d((3,3,1)) against float64 autograd
CHAINS = {   # x shape, (Cin, Cout, kernel, stride), fp32 chains of (forward, dgrad, wgrad)
    "line": ((2, 3, 20, 21, 9), (3, 8, (1, 1, 9), 1), (27, 8 * 9, 1 + 2 + 592)),
    "2d": ((2, 8, 27, 30, 1), (8, 16, (5, 5, 1), 2), (200, 16 * 3 * 3, math.ceil(2 * 12 * 13 / 32) + 5)),
}
EPS, MOM = 1e-5, 0.1
RED = (0, 2, 3, 4)


def v(t):
    return t.view(1, -1, 1, 1, 1)


@pytest.mark.parametrize("training", [True, False], ids=["train", "eval"])
@pytest.mark.parametrize("kind", list(CHAINS))
def test_gaussian_chain_within_rounding_bound(kind, training):
    """Outputs, dx, dw, db, dgamma, dbeta and the running statistics, per element.  z = conv(x) carries at most
    ez = 2 T 2^-24 (|x| * |w| + |b|) (T the forward chain); in train mode the kernel's mean and sigma then move by at
    most D = E (2 + rms/sigma) + 128 2^-24 rms (1 + rms/sigma) (E the channel's largest ez, rms the root mean square
    of z: the statistics add fp32 chunks of 64 terms), and every fp32 step of finalize / apply adds a few units of its
    magnitudes (16 units, as in test_gpu_bn_exact).  Bounds are first-order; the factor 2 covers the rest."""
    xs, (cin, cout, ks, s), (t_fwd, t_dg, t_wg) = CHAINS[kind]
    g = gen(70 + 2 * list(CHAINS).index(kind) + int(training))
    conv = torch.nn.Conv3d(cin, cout, ks, stride=s).to(DEV)
    bn = torch.nn.BatchNorm3d(cout, eps=EPS, momentum=MOM).to(DEV)
    pool = torch.nn.MaxPool3d((3, 3, 1))
    with torch.no_grad():
        conv.weight.copy_(rn(g, cout, cin, *ks) * (cin * math.prod(ks)) ** -0.5)
        conv.bias.copy_(rn(g, cout) * 0.1)
        gam = rn(g, cout) * 0.5 + 1
        gam[::3] *= -1
        bn.weight.copy_(gam)
        bn.bias.copy_(rn(g, cout) * 0.3)
        bn.running_mean.copy_(rn(g, cout) * 0.2)
        bn.running_var.copy_(torch.rand(cout, generator=g, device=DEV) + 0.5)
    rm0, rv0, nbt0 = bn.running_mean.clone(), bn.running_var.clone(), int(bn.num_batches_tracked)
    x = rn(g, *xs).float().requires_grad_(True)
    out = MF.maxpool_xy(MF.conv_bn_relu(x, conv, bn, training), pool)
    dout = rn(g, *out.shape)
    out.backward(dout.float())
    # float64 torch
    x64 = x.detach().double().requires_grad_(True)
    w64, b64, g64, be64 = (p.detach().double().requires_grad_(True) for p in (conv.weight, conv.bias, bn.weight, bn.bias))
    rm64, rv64 = rm0.double(), rv0.double()
    z = F.conv3d(x64, w64, b64, stride=s)
    zn = F.batch_norm(z, rm64, rv64, g64, be64, training, MOM, EPS)
    ref = F.max_pool3d(F.relu(zn), (3, 3, 1))
    dzr = torch.autograd.grad(ref, zn, dout, retain_graph=True)[0]        # dout routed through the pool and the ReLU
    ref.backward(dout)
    # forward
    zd = z.detach()
    ez = 2 * t_fwd * U * F.conv3d(x64.detach().abs(), w64.detach().abs(), b64.detach().abs(), stride=s)
    E = ez.amax(RED)
    if training:
        mean, var = zd.mean(RED), zd.var(RED, unbiased=False)
    else:
        mean, var = rm0.double(), rv0.double()
    sig = torch.sqrt(var + EPS)
    rms = torch.sqrt((zd * zd).mean(RED))
    D = E * (2 + rms / sig) + 128 * U * rms * (1 + rms / sig) if training else torch.zeros_like(E)
    gd, bd = g64.detach(), be64.detach()
    sc = gd / sig
    xh = (zd - v(mean)) / v(sig)
    mag = (zd * v(sc)).abs() + v((bd - mean * sc).abs() + (mean * sc).abs() + bd.abs())
    bound = 2 * v(sc.abs()) * (ez + (1 + xh.abs()) * v(D)) + 16 * U * mag
    within(out, ref.detach(), F.max_pool3d(bound, (3, 3, 1)), "output")
    # backward: dz_bn = scale (dz - m1 - xhat m2)
    count = zd.numel() // cout
    adz = dzr.abs()
    dxh = (1 + xh.abs()) * v(D / sig) + 4 * U * xh.abs()
    if training:
        m1, m2 = dzr.mean(RED), (dzr * xh).mean(RED)
        dm1 = 66 * U * adz.mean(RED)
        dm2 = 66 * U * (adz * (xh.abs() + 1)).mean(RED) + (adz * dxh).mean(RED)
    else:
        m1 = m2 = dm1 = dm2 = torch.zeros_like(E)
    rho = 16 * U + D / sig
    dzbn = v(sc) * (dzr - v(m1) - xh * v(m2))
    e_dz = 2 * v(sc.abs()) * (v(rho) * (adz + v(m1.abs()) + xh.abs() * v(m2.abs())) + v(dm1) + xh.abs() * v(dm2)
                              + dxh * v(m2.abs())) + 3 * U * dzbn.abs()
    wa, xa = w64.detach().abs(), x64.detach().abs()
    dx_b = (torch.nn.grad.conv3d_input(xs, wa, e_dz, stride=s)
            + 2 * t_dg * U * torch.nn.grad.conv3d_input(xs, wa, dzbn.abs(), stride=s))
    within(x.grad, x64.grad, dx_b, "dx")
    dw_b = (torch.nn.grad.conv3d_weight(xa, w64.shape, e_dz, stride=s)
            + 2 * t_wg * U * torch.nn.grad.conv3d_weight(xa, w64.shape, dzbn.abs(), stride=s))
    within(conv.weight.grad, w64.grad, dw_b, "dw")
    within(conv.bias.grad, b64.grad, e_dz.sum(RED) + 2 * t_wg * U * dzbn.abs().sum(RED), "db")
    within(bn.weight.grad, g64.grad, 66 * U * (adz * (xh.abs() + 1)).sum(RED) + (adz * dxh).sum(RED)
           + 2 * U * g64.grad.abs(), "dgamma")
    within(bn.bias.grad, be64.grad, 66 * U * adz.sum(RED) + 2 * U * be64.grad.abs(), "dbeta")
    # running statistics
    if training:
        vu = var * count / (count - 1)
        within(bn.running_mean, rm64, 3 * U * ((1 - MOM) * rm0.double().abs() + MOM * mean.abs()) + MOM * D,
               "running_mean")
        within(bn.running_var, rv64, 3 * U * ((1 - MOM) * rv0.double().abs() + MOM * vu)
               + MOM * (2 * sig * D + D * D) * count / (count - 1) + MOM * U * vu, "running_var")
        assert int(bn.num_batches_tracked) == nbt0 + 1
    else:
        assert torch.equal(bn.running_mean, rm0) and torch.equal(bn.running_var, rv0)
        assert int(bn.num_batches_tracked) == nbt0


# ---------------------------------------------------------------------------------------------------------------
def test_refused_arguments():
    """The host-side checks refuse before any launch: a slice weight gradient staging more than 48 KB, empty or
    zero-sized spatial convolutions, a pool window past 255 positions, empty BatchNorm tensors.  (The widest accepted
    slice weight gradient runs in test_line_conv_exact[edge-w16-smem48k].)"""
    buf = torch.zeros(16, device=DEV)
    p = L.ptr(buf)
    lib = L.load()
    n0 = L.launch_count()

    def refused(name, match, *args):
        with pytest.raises(RuntimeError, match=match):
            L.call(name, *args)

    ws = torch.empty(int(lib.tmf_line_conv_wgrad_workspace_bytes(8, 64)), dtype=torch.uint8, device=DEV)
    assert M.line_wgrad_smem(8, 800, 64) > M.SMEM_LIMIT
    refused("tmf_line_conv_wgrad", "line_conv_wgrad: line too long", p, p, p, p, 1, 8, 1, 800, 64, L.ptr(ws), ws.numel())
    for n, cin, cout, kh, kw in ((0, 1, 1, 1, 1), (1, 0, 1, 1, 1), (1, 1, 0, 1, 1), (1, 1, 1, 0, 1), (1, 1, 1, 1, 0)):
        args = (n, cin, 5, 5, cout, kh, kw, 1)
        refused("tmf_conv2d_fwd", "conv2d_fwd: bad arguments", p, p, p, p, *args)
        refused("tmf_conv2d_dgrad", "conv2d_dgrad: bad arguments", p, p, p, *args)
        refused("tmf_conv2d_wgrad", "conv2d_wgrad: bad arguments", p, p, p, p, *args)
    refused("tmf_maxpool2d_fwd", "maxpool2d_fwd: bad arguments", p, p, p, 1, 15, 18, 15, 18)
    refused("tmf_maxpool2d_bwd", "maxpool2d_bwd: bad arguments", p, p, p, 1, 15, 18, 15, 18)
    for n, C, S in ((0, 1, 1), (1, 0, 1), (1, 1, 0), (1, 1, -1)):
        refused("tmf_nchw_bn_relu_fwd", "nchw_bn_relu_fwd: empty tensor", p, p, p, n, C, S)
        refused("tmf_nchw_bn_relu_bwd_reduce", "nchw_bn_relu_bwd_reduce: empty tensor", p, p, p, p, n, C, S)
        refused("tmf_nchw_bn_relu_bwd_apply", "nchw_bn_relu_bwd_apply: empty tensor", p, p, p, p, p, n, C, S)
    assert L.launch_count() == n0, "a refused call launched"

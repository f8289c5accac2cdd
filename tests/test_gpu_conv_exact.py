"""Exact-arithmetic tests of the sNet convolution kernels (tcgen05 paths) at the model's own layer shapes.

Operands are small integers or short significands on a fixed grid (tests/conv_exact.py): every product and every partial
sum is exact in fp32, so whatever the tiling, split-K or reduction order, a correct kernel reproduces the float64
reference bit for bit -- a dropped, duplicated or misplaced contribution fails on the element it touches.  Every output,
statistics buffer and workspace is poisoned with NaN bytes before each call and the outputs sit inside guard bands:
the buffer contracts of include/tmf.h (every stats row written, dw / dx overwritten, workspaces need no zeroing) and
"nothing written past the end" are checked on every call, and two calls must give the same bits.

One Gaussian case per kernel family checks what integer data cannot (rounding) against a per-element bound
|got - ref| <= 2^-8 |ref| (bf16 outputs) + c 2^-24 (|a| * |w|), with |a| * |w| the same operation on absolute values and
c twice the length of the longest fp32 accumulation chain (each link may lose 2^-23 of the running absolute sum when a
truncating adder aligns the addends)."""
import math
import zlib

import pytest
import torch

from tests import conv_exact as X
from transmf_ad_b200 import _lib as L

pytestmark = pytest.mark.gpu
DEV = "cuda"
U = 2.0 ** -24


def gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def ndhwc_bf16(t):
    return t.to(torch.bfloat16).contiguous()


def workspace(nbytes):
    ws = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=DEV)
    ws.fill_(0xFF)                                   # workspaces need no zeroing
    return ws


def pack(ng, w):
    """bf16 forward / dgrad packs of fp32 weights (exact: the test weights are bf16-representable)."""
    cout, cin, k = w[0].shape[0], w[0].shape[1], w[0].shape[-1]
    w32 = [t.float().contiguous() for t in w]
    wf = [torch.empty((k ** 3, cout, cin), dtype=torch.bfloat16, device=DEV) for _ in range(ng)]
    wd = [torch.empty((k ** 3, cin, cout), dtype=torch.bfloat16, device=DEV) for _ in range(ng)]
    L.call("tmf_pack_conv_weights", ng, L.ptrs(w32), L.ptrs(wf), L.ptrs(wd), cout, cin, k)
    return wf, wd


def check_stats(stats, y, what, rel=2.0 ** -20):
    """Every row finite after poisoning; the rows add up to the fp64 sums of the STORED outputs to within `rel` of the
    sum of absolute values (the epilogues keep fp32 per-thread partials, so not exactly)."""
    assert bool(torch.isfinite(stats).all()), f"{what}: statistics rows left unwritten"
    c = y.shape[-1]
    y64 = y.double().reshape(-1, c)
    tot = stats.sum(0)
    s, q = y64.sum(0), (y64 * y64).sum(0)
    assert bool(((tot[:c] - s).abs() <= rel * y64.abs().sum(0)).all()), f"{what}: sum"
    assert bool(((tot[c:] - q).abs() <= rel * q).all()), f"{what}: sum of squares"


def run_twice(outs, launch):
    """Poison every output, launch, check the guard bands; repeat and demand the same bits."""
    snaps = []
    for _ in range(2):
        for o in outs:
            o.poison()
        launch()
        torch.cuda.synchronize()
        for i, o in enumerate(outs):
            o.check_bands(f"output {i}")
        snaps.append([o.t.clone() for o in outs])
    for a, b in zip(*snaps):
        assert torch.equal(a.view(torch.uint8), b.view(torch.uint8)), "two calls gave different bits"
    return snaps[0]


# ---------------------------------------------------------------------------------------------------------------
# conv3d: forward (+ stats), dgrad, wgrad
def conv_operands(case, seed):
    _, ng, B, (D, H, W), cin, cout, ks, _ = case
    g = gen(seed)
    a = [X.ints((B, D, H, W, cin), -2, 2, g, DEV) for _ in range(ng)]
    dy = [X.ints((B, D, H, W, cout), -2, 2, g, DEV) for _ in range(ng)]
    w = [X.ints((cout, cin, ks, ks, ks), -2, 2, g, DEV) for _ in range(ng)]
    bias = [X.ints((cout,), -4, 4, g, DEV) for _ in range(ng)]
    X.exact_bound(ks ** 3 * cin, 2, 2, 1, extra=4)            # forward: 27 * 256 * 4 + 4 at most
    X.exact_bound(ks ** 3 * cout, 2, 2, 1)                    # dgrad
    X.exact_bound(B * D * H * W, 2, 2, 1)                     # wgrad: every voxel of the batch
    return a, dy, w, bias


@pytest.mark.parametrize("case", X.CONV_CASES, ids=[c[0] for c in X.CONV_CASES])
def test_conv3d_exact(case):
    cid, ng, B, (D, H, W), cin, cout, ks, dispatch = case
    lib = L.load()
    for op, kern in dispatch.items():          # the kernel each op reaches (a planner change that moves it shows here)
        if op == "wgrad":
            assert X.wgrad_kernel(ng, W, cin, cout, ks) == kern
        else:
            ci, co = (cin, cout) if op == "fwd" else (cout, cin)
            assert X.fwd_kernel(lib, ng, B, D, H, W, ci, co, ks) == kern, op
    a, dy, w, bias = conv_operands(case, seed=zlib.crc32(cid.encode()))
    a_b, dy_b = [ndhwc_bf16(t) for t in a], [ndhwc_bf16(t) for t in dy]
    wf, wd = pack(ng, w)
    bias32 = [t.float() for t in bias]
    if "fwd" in dispatch:
        y = [X.Guarded((B, D, H, W, cout), torch.bfloat16, DEV) for _ in range(ng)]
        st = [X.Guarded((L.stat_rows(), 2 * cout), torch.float64, DEV) for _ in range(ng)]
        got = run_twice(y + st, lambda: L.call("tmf_conv3d_fwd", ng, L.ptrs(a_b), L.ptrs(wf), L.ptrs(bias32),
                                                L.ptrs([t.t for t in y]), L.ptrs([t.t for t in st]), B, D, H, W, cin, cout,
                                                ks, L.CONV_UMMA))
        for t in range(ng):
            want = X.bf16_rne(X.conv_ref(a[t], w[t]) + bias[t])
            err = X.mismatch(got[t], want)
            assert not err, f"{cid} forward, tower {t}: {err}"
            check_stats(got[ng + t], got[t], f"{cid} tower {t}")
    if "dgrad" in dispatch:
        da = [X.Guarded((B, D, H, W, cin), torch.bfloat16, DEV) for _ in range(ng)]
        got = run_twice(da, lambda: L.call("tmf_conv3d_fwd", ng, L.ptrs(dy_b), L.ptrs(wd), L.ptrs(None),
                                           L.ptrs([t.t for t in da]), L.ptrs(None), B, D, H, W, cout, cin, ks, L.CONV_UMMA))
        for t in range(ng):
            err = X.mismatch(got[t], X.bf16_rne(X.dgrad_ref(dy[t], w[t])))
            assert not err, f"{cid} dgrad, tower {t}: {err}"
    if "wgrad" in dispatch:
        dw = [X.Guarded((cout, cin, ks, ks, ks), torch.float32, DEV) for _ in range(ng)]
        ws = workspace(lib.tmf_conv3d_wgrad_workspace_bytes(ng, L.CONV_UMMA, B, D, H, W, cin, cout, ks))
        got = run_twice(dw, lambda: L.call("tmf_conv3d_wgrad", ng, L.ptrs(dy_b), L.ptrs(a_b), L.ptrs([t.t for t in dw]),
                                           B, D, H, W, cin, cout, ks, L.CONV_UMMA, L.ptr(ws), ws.numel()))
        for t in range(ng):
            err = X.mismatch(got[t].double(), X.wgrad_ref(dy[t], a[t], ks))
            assert not err, f"{cid} wgrad, tower {t}: {err}"


@pytest.mark.parametrize("shape,cin,cout,ks", [((2, 9, 11, 10), 32, 64, 3), ((2, 6, 7, 9), 64, 64, 3),
                                               ((2, 5, 6, 5), 128, 256, 3), ((2, 5, 6, 7), 256, 128, 1)])
def test_conv3d_gaussian_within_rounding_bound(shape, cin, cout, ks):
    """Gaussian data: forward, dgrad and wgrad per element against the fp64 reference of the same bf16 operands.
    Forward / dgrad chain: 27 Cin / 16 MMA K-steps + the bias add; wgrad: B D H W / 16 K-steps in the longest CTA range
    + at most 148 split-K partials added in the reduce."""
    B, D, H, W = shape
    g = gen(5)
    a = torch.randn((B, D, H, W, cin), generator=g, device=DEV, dtype=torch.float64).to(torch.bfloat16)
    dy = torch.randn((B, D, H, W, cout), generator=g, device=DEV, dtype=torch.float64).to(torch.bfloat16)
    w = (torch.randn((cout, cin, ks, ks, ks), generator=g, device=DEV, dtype=torch.float64) * (cin * ks ** 3) ** -0.5)
    w = w.to(torch.bfloat16).double()
    bias = torch.randn((cout,), generator=g, device=DEV).mul(0.1)
    wf, wd = pack(1, [w])
    a64, dy64 = a.double(), dy.double()
    y = torch.empty((B, D, H, W, cout), dtype=torch.bfloat16, device=DEV)
    L.call("tmf_conv3d_fwd", 1, L.ptrs([a]), L.ptrs(wf), L.ptrs([bias]), L.ptrs([y]), L.ptrs(None), B, D, H, W, cin, cout,
           ks, L.CONV_UMMA)
    c = 2 * (ks ** 3 * cin / 16 + 1)
    ref = X.conv_ref(a64, w) + bias.double()
    bound = 2.0 ** -8 * ref.abs() + c * U * (X.conv_ref(a64.abs(), w.abs()) + bias.double().abs())
    assert bool(((y.double() - ref).abs() <= bound).all()), "forward"
    da = torch.empty((B, D, H, W, cin), dtype=torch.bfloat16, device=DEV)
    L.call("tmf_conv3d_fwd", 1, L.ptrs([dy]), L.ptrs(wd), L.ptrs(None), L.ptrs([da]), L.ptrs(None), B, D, H, W, cout, cin,
           ks, L.CONV_UMMA)
    c = 2 * (ks ** 3 * cout / 16 + 1)
    ref = X.dgrad_ref(dy64, w)
    bound = 2.0 ** -8 * ref.abs() + c * U * X.dgrad_ref(dy64.abs(), w.abs())
    assert bool(((da.double() - ref).abs() <= bound).all()), "dgrad"
    dw = torch.empty((cout, cin, ks, ks, ks), dtype=torch.float32, device=DEV)
    ws = workspace(L.load().tmf_conv3d_wgrad_workspace_bytes(1, L.CONV_UMMA, B, D, H, W, cin, cout, ks))
    L.call("tmf_conv3d_wgrad", 1, L.ptrs([dy]), L.ptrs([a]), L.ptrs([dw]), B, D, H, W, cin, cout, ks, L.CONV_UMMA,
           L.ptr(ws), ws.numel())
    c = 2 * (math.ceil(B * D * H * W / 16) + 148)
    ref = X.wgrad_ref(dy64, a64, ks)
    bound = U * ref.abs() + c * U * X.wgrad_ref(dy64.abs(), a64.abs(), ks)
    assert bool(((dw.double() - ref).abs() <= bound).all()), "wgrad"


# ---------------------------------------------------------------------------------------------------------------
# block 1: conv1.0 forward, weight gradient, fused backward, input gradient
BENCH1 = (8, 91, 109, 91)


def conv1_fwd_call(ng, x, w, bias, y, st, shape, cout):
    B, D, H, W = shape
    L.call("tmf_conv1_fwd", ng, L.ptrs(x), L.ptrs(w), L.ptrs(bias), L.ptrs(y), L.ptrs(st), B, D, H, W, cout, L.CONV_UMMA)


@pytest.mark.parametrize("ng,shape,cout,lo_side", [
    (2, BENCH1, 32, "x"), (2, BENCH1, 32, "w"), (1, BENCH1, 64, "x"), (1, BENCH1, 64, "w"),
    (2, (3, 5, 7, 9), 32, "x"), (1, (1, 1, 3, 250), 64, "w"), (2, (2, 3, 1, 1), 32, "x")])
def test_conv1_fwd_exact(ng, shape, cout, lo_side):
    """conv1.0 keeps fp32 accuracy with a bf16 hi/lo split, x*w ~= xh*wh + xl*wh + xh*wl (xl*wl dropped).  One operand
    has a 16-bit significand (|v| < 8 on a 2^-13 grid: its lo half is exact and non-zero), the other is bf16-exact (its
    lo half is 0): the dropped term is exactly 0 and the result must be exact -- losing the xl*wh (lo_side x) or the xh*wl
    (lo_side w) product fails.  Also: stats rows, guard bands, and the unstaged image path (x not 16-byte aligned) gives
    the same bits as the staged one."""
    B, D, H, W = shape
    g = gen(11)
    if lo_side == "x":
        x = [X.fixed((B, D, H, W), 16, 13, g, DEV) for _ in range(ng)]
        w = [X.ints((cout, 1, 3, 3, 3), -2, 2, g, DEV) for _ in range(ng)]
        X.exact_bound(27, 8, 2, 2.0 ** -13, extra=4)
    else:
        x = [X.ints((B, D, H, W), -2, 2, g, DEV) for _ in range(ng)]
        w = [X.fixed((cout, 1, 3, 3, 3), 16, 13, g, DEV) for _ in range(ng)]
        X.exact_bound(27, 2, 8, 2.0 ** -13, extra=4)
    bias = [X.ints((cout,), -4, 4, g, DEV) for _ in range(ng)]
    x32, w32, b32 = [t.float() for t in x], [t.float() for t in w], [t.float() for t in bias]
    y = [X.Guarded((B, D, H, W, cout), torch.bfloat16, DEV) for _ in range(ng)]
    st = [X.Guarded((L.stat_rows(), 2 * cout), torch.float64, DEV) for _ in range(ng)]
    got = run_twice(y + st, lambda: conv1_fwd_call(ng, x32, w32, b32, [t.t for t in y], [t.t for t in st], shape, cout))
    # statistics: a thread of conv1.0's epilogue adds one voxel row of every tile of its CTA in fp32 (762 tiles per thread
    # at 91 x 109 x 91, batch 8, where 1.05e-6 relative was measured on a B200), then 5 shuffle levels: that many fp32
    # roundings of the running sum, 2^-24 each at most
    chain = -(-B * D * H * W // 128 // (148 // ng)) + 8
    rel = max(2.0 ** -20, chain * U)
    for t in range(ng):
        want = X.bf16_rne(X.conv_ref(x[t].unsqueeze(-1), w[t]) + bias[t])
        err = X.mismatch(got[t], want)
        assert not err, f"tower {t}: {err}"
        check_stats(got[ng + t], got[t], f"tower {t}", rel)
    # unstaged path: the image one float into a larger buffer
    n = B * D * H * W
    xo = [torch.empty(n + 4, dtype=torch.float32, device=DEV) for _ in range(ng)]
    xs = []
    for t in range(ng):
        xo[t][1:n + 1] = x32[t].flatten()
        xs.append(xo[t][1:n + 1])
    got2 = run_twice(y + st, lambda: conv1_fwd_call(ng, xs, w32, b32, [t.t for t in y], [t.t for t in st], shape, cout))
    for t in range(ng):
        assert torch.equal(got2[t].view(torch.int16), got[t].view(torch.int16)), f"unstaged tower {t}"
        check_stats(got2[ng + t], got2[t], f"unstaged tower {t}", rel)


def conv1_wgrad_operands(shape, ng, lo, seed):
    """dy integers in [-1, 1]; x integers in [-1, 1] (full size: B D H W = 7.2 M voxels, still below 2^24) or, with
    lo, on a 2^-8 grid with |x| < 4 (up to 10 significant bits: the lo half of the split image is non-zero)."""
    B, D, H, W = shape
    g = gen(seed)
    if lo:
        x = [X.fixed((B, D, H, W), 10, 8, g, DEV) for _ in range(ng)]
        X.exact_bound(B * D * H * W, 4, 1, 2.0 ** -8)
    else:
        x = [X.ints((B, D, H, W), -1, 1, g, DEV) for _ in range(ng)]
        X.exact_bound(B * D * H * W, 1, 1, 1)
    return g, x


@pytest.mark.parametrize("ng,shape,lo", [(2, BENCH1, False), (1, (1, 7, 23, 91), True), (2, (2, 3, 5, 254), True),
                                         (2, (1, 1, 3, 2), True), (1, (3, 5, 9, 13), False)])
def test_conv1_wgrad_exact(ng, shape, lo):
    B, D, H, W = shape
    g, x = conv1_wgrad_operands(shape, ng, lo, seed=21)
    dy = [X.ints((B, D, H, W, 32), -1, 1, g, DEV) for _ in range(ng)]
    x32, dy_b = [t.float() for t in x], [ndhwc_bf16(t) for t in dy]
    dw = [X.Guarded((32, 1, 3, 3, 3), torch.float32, DEV) for _ in range(ng)]
    ws = workspace(L.load().tmf_conv1_wgrad_workspace_bytes(ng, L.CONV_UMMA, W, 32))
    got = run_twice(dw, lambda: L.call("tmf_conv1_wgrad", ng, L.ptrs(dy_b), L.ptrs(x32), L.ptrs([t.t for t in dw]),
                                       B, D, H, W, 32, L.CONV_UMMA, L.ptr(ws), ws.numel()))
    for t in range(ng):
        err = X.mismatch(got[t].double(), X.wgrad_ref(dy[t], x[t].unsqueeze(-1), 3))
        assert not err, f"tower {t}: {err}"


def identity_coefs(ng, C):
    """scale 1, shift 0, mean 0, invstd 1 and bcoef 0: with slope 1 the BatchNorm / LeakyReLU backward is the identity,
    and the block-1 backward kernels route dout unchanged to the first maximum of each pooling window of y."""
    coef = torch.cat([torch.ones(C), torch.zeros(C), torch.zeros(C), torch.ones(C)]).to(DEV)
    return [coef] * ng, [torch.zeros(2 * C, device=DEV)] * ng


def pooled_operands(shape, ng, g):
    """y: integers in [-2, 2] (ties inside most 2x2x2 windows), dout: integers in [-2, 2] at pooled resolution."""
    B, D, H, W = shape
    y = [X.ints((B, D, H, W, 32), -2, 2, g, DEV) for _ in range(ng)]
    dout = [X.ints((B, D // 2, H // 2, W // 2, 32), -2, 2, g, DEV) for _ in range(ng)]
    return y, dout


@pytest.mark.parametrize("ng,shape,lo", [(2, BENCH1, False), (1, (1, 8, 21, 91), True), (2, (2, 4, 6, 224), True),
                                         (2, (1, 2, 2, 17), True), (1, (3, 7, 9, 17), False)])
def test_conv1_bwd_fused_exact(ng, shape, lo):
    """dW of block 1 from dout and the stored y (pooling routing, ties included) and the split image, W from 17 to 224 (the
    narrowest row whose stages hold the epilogue's fold buffer, and the widest whose stages fit)."""
    B, D, H, W = shape
    g, x = conv1_wgrad_operands(shape, ng, lo, seed=31)
    y, dout = pooled_operands(shape, ng, g)
    X.exact_bound(B * (D // 2) * (H // 2) * (W // 2), 2, 4 if lo else 1, 2.0 ** -8 if lo else 1)   # one dy per window
    coef, bcoef = identity_coefs(ng, 32)
    x32 = [t.float() for t in x]
    y_b, dout_b = [ndhwc_bf16(t) for t in y], [ndhwc_bf16(t) for t in dout]
    nws = int(L.load().tmf_conv1_bwd_fused_workspace_bytes(ng, B, D, H, W, 32))
    assert nws > 0
    ws = workspace(nws)
    dw = [X.Guarded((32, 1, 3, 3, 3), torch.float32, DEV) for _ in range(ng)]
    got = run_twice(dw, lambda: L.call("tmf_conv1_bwd_fused", ng, L.ptrs(dout_b), L.ptrs(y_b), L.ptrs(coef), L.ptrs(bcoef),
                                       L.ptrs(x32), L.ptrs([t.t for t in dw]), B, D, H, W, 32, 1.0, L.ptr(ws), nws))
    for t in range(ng):
        dy = X.maxpool_route(y[t], dout[t])
        err = X.mismatch(got[t].double(), X.wgrad_ref(dy, x[t].unsqueeze(-1), 3))
        assert not err, f"tower {t}: {err}"


@pytest.mark.parametrize("ng,shape", [(2, BENCH1), (1, (1, 9, 35, 128)), (2, (2, 3, 5, 7)), (2, (1, 2, 2, 2)),
                                      (1, (3, 17, 33, 65))])
def test_conv1_dgrad_fused_exact(ng, shape):
    """dx of block 1 (tcgen05, W <= 128): the weight as bf16 hi + lo halves; w has 13 fractional bits (|w| < 1), so
    both halves matter and every sum stays below 2^24 quanta."""
    B, D, H, W = shape
    g = gen(41)
    y, dout = pooled_operands(shape, ng, g)
    w = [X.fixed((32, 1, 3, 3, 3), 13, 13, g, DEV) for _ in range(ng)]
    X.exact_bound(27 * 32, 2, 1, 2.0 ** -13)
    coef, bcoef = identity_coefs(ng, 32)
    w32 = [t.float() for t in w]
    y_b, dout_b = [ndhwc_bf16(t) for t in y], [ndhwc_bf16(t) for t in dout]
    lib = L.load()
    nws = int(lib.tmf_conv1_dgrad_fused_workspace_bytes(ng, L.CONV_UMMA, B, D, H, W, 32))
    ws = workspace(nws)
    dx = [X.Guarded((B, D, H, W), torch.float32, DEV) for _ in range(ng)]
    got = run_twice(dx, lambda: L.call("tmf_conv1_dgrad_fused", ng, L.ptrs(dout_b), L.ptrs(y_b), L.ptrs(coef),
                                       L.ptrs(bcoef), L.ptrs(w32), L.ptrs([t.t for t in dx]), B, D, H, W, 32, 1.0,
                                       L.CONV_UMMA, L.ptr(ws), nws))
    for t in range(ng):
        dy = X.maxpool_route(y[t], dout[t])
        err = X.mismatch(got[t].double(), X.dgrad_ref(dy, w[t])[..., 0])
        assert not err, f"tower {t}: {err}"


def test_block1_gaussian_within_rounding_bound():
    """Gaussian image / weights / gradients through the four block-1 kernels, per element.  Split error: the lo half is
    rounded to bf16 (2^-18 relative) and xl*wl is dropped (2^-18): 2^-16 (|x| * |w|) covers both."""
    B, D, H, W = 2, 10, 13, 40
    g = gen(51)
    rn = lambda *s: torch.randn(s, generator=g, device=DEV, dtype=torch.float64)
    x = rn(B, D, H, W).float().double()
    w = (rn(32, 1, 3, 3, 3) * 0.3).float().double()
    bias = (rn(32) * 0.1).float().double()
    # forward: chain = 2 K-steps x 3 products + bias
    y = torch.empty((B, D, H, W, 32), dtype=torch.bfloat16, device=DEV)
    conv1_fwd_call(1, [x.float()], [w.float()], [bias.float()], [y], None, (B, D, H, W), 32)
    ref = X.conv_ref(x.unsqueeze(-1), w) + bias
    absr = X.conv_ref(x.abs().unsqueeze(-1), w.abs()) + bias.abs()
    assert bool(((y.double() - ref).abs() <= 2.0 ** -8 * ref.abs() + (2 * 7 * U + 2.0 ** -16) * absr).all()), "forward"
    # weight gradient: dy bf16, image split; chain = voxels / 16 x 2 products + 148 partials
    dy = rn(B, D, H, W, 32).to(torch.bfloat16)
    dw = torch.empty((32, 1, 3, 3, 3), device=DEV)
    ws = workspace(L.load().tmf_conv1_wgrad_workspace_bytes(1, L.CONV_UMMA, W, 32))
    L.call("tmf_conv1_wgrad", 1, L.ptrs([dy]), L.ptrs([x.float()]), L.ptrs([dw]), B, D, H, W, 32, L.CONV_UMMA, L.ptr(ws),
           ws.numel())
    c = 2 * (2 * math.ceil(B * D * H * W / 16) + 148)
    ref = X.wgrad_ref(dy.double(), x.unsqueeze(-1), 3)
    absr = X.wgrad_ref(dy.double().abs(), x.abs().unsqueeze(-1), 3)
    assert bool(((dw.double() - ref).abs() <= U * ref.abs() + (c * U + 2.0 ** -16) * absr).all()), "wgrad"
    # fused backward and input gradient with identity coefficients on Gaussian y / dout
    yb = rn(B, D, H, W, 32).to(torch.bfloat16)
    dout = rn(B, D // 2, H // 2, W // 2, 32).to(torch.bfloat16)
    coef, bcoef = identity_coefs(1, 32)
    dyr = X.maxpool_route(yb.double(), dout.double())
    nws = int(L.load().tmf_conv1_bwd_fused_workspace_bytes(1, B, D, H, W, 32))
    ws = workspace(nws)
    L.call("tmf_conv1_bwd_fused", 1, L.ptrs([dout]), L.ptrs([yb]), L.ptrs(coef), L.ptrs(bcoef), L.ptrs([x.float()]),
           L.ptrs([dw]), B, D, H, W, 32, 1.0, L.ptr(ws), nws)
    ref = X.wgrad_ref(dyr, x.unsqueeze(-1), 3)
    absr = X.wgrad_ref(dyr.abs(), x.abs().unsqueeze(-1), 3)
    assert bool(((dw.double() - ref).abs() <= U * ref.abs() + (c * U + 2.0 ** -16) * absr).all()), "fused backward"
    dx = torch.empty((B, D, H, W), device=DEV)
    L.call("tmf_conv1_dgrad_fused", 1, L.ptrs([dout]), L.ptrs([yb]), L.ptrs(coef), L.ptrs(bcoef), L.ptrs([w.float()]),
           L.ptrs([dx]), B, D, H, W, 32, 1.0, L.CONV_UMMA, L.ptr(None), 0)
    ref = X.dgrad_ref(dyr, w)[..., 0]
    absr = X.dgrad_ref(dyr.abs(), w.abs())[..., 0]
    c = 2 * (2 * 27 * 32 / 16 + 1)
    assert bool(((dx.double() - ref).abs() <= U * ref.abs() + (c * U + 2.0 ** -16) * absr).all()), "input gradient"

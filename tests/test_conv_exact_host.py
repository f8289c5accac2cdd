"""CPU checks of the exact-arithmetic test machinery (tests/conv_exact.py), so that the GPU tests' reference stands on its
own: the per-tap float64 references against F.conv3d / torch.nn.grad, the pooling routing against max_pool3d's
backward, the generators and the 2^24 bound, and the shape table's coverage of every tcgen05 plan the planners pick."""
import pytest
import torch
import torch.nn.functional as F

from tests import conv_exact as X


def cpu_gen(seed):
    return torch.Generator().manual_seed(seed)


def to_ncdhw(t):
    return t.permute(0, 4, 1, 2, 3)


@pytest.mark.parametrize("shape,cin,cout,ks", [((2, 3, 4, 5), 3, 5, 3), ((1, 1, 2, 7), 4, 2, 3), ((2, 3, 3, 2), 6, 4, 1),
                                               ((1, 2, 1, 1), 2, 3, 3)])
def test_references_match_torch_in_float64(shape, cin, cout, ks):
    B, D, H, W = shape
    g = cpu_gen(1)
    a = torch.randn(B, D, H, W, cin, generator=g, dtype=torch.float64)
    dy = torch.randn(B, D, H, W, cout, generator=g, dtype=torch.float64)
    w = torch.randn(cout, cin, ks, ks, ks, generator=g, dtype=torch.float64)
    y = F.conv3d(to_ncdhw(a), w, padding=ks // 2)
    torch.testing.assert_close(to_ncdhw(X.conv_ref(a, w)), y, rtol=1e-12, atol=1e-12)
    da = torch.nn.grad.conv3d_input(to_ncdhw(a).shape, w, to_ncdhw(dy), padding=ks // 2)
    torch.testing.assert_close(to_ncdhw(X.dgrad_ref(dy, w)), da, rtol=1e-12, atol=1e-12)
    dw = torch.nn.grad.conv3d_weight(to_ncdhw(a), w.shape, to_ncdhw(dy), padding=ks // 2)
    torch.testing.assert_close(X.wgrad_ref(dy, a, ks), dw, rtol=1e-12, atol=1e-12)


def test_integer_operands_give_exact_references():
    """On integer operands the float64 references are integers, equal to torch's to the last bit."""
    g = cpu_gen(2)
    a = X.ints((2, 4, 5, 6, 8), -2, 2, g, "cpu")
    dy = X.ints((2, 4, 5, 6, 4), -2, 2, g, "cpu")
    w = X.ints((4, 8, 3, 3, 3), -2, 2, g, "cpu")
    y = X.conv_ref(a, w)
    assert torch.equal(y, y.round()) and torch.equal(to_ncdhw(y), F.conv3d(to_ncdhw(a), w, padding=1))
    dw = X.wgrad_ref(dy, a, 3)
    assert torch.equal(dw, torch.nn.grad.conv3d_weight(to_ncdhw(a), w.shape, to_ncdhw(dy), padding=1))


def test_maxpool_route_is_max_pool_backward_with_ties():
    g = cpu_gen(3)
    y = X.ints((2, 5, 6, 7, 3), -1, 1, g, "cpu")          # three values: ties in nearly every window; odd extents
    dout = torch.randn(2, 2, 3, 3, 3, generator=g, dtype=torch.float64)
    yr = to_ncdhw(y).clone().requires_grad_(True)
    F.max_pool3d(yr, 2, 2).backward(to_ncdhw(dout))
    assert torch.equal(to_ncdhw(X.maxpool_route(y, dout)), yr.grad)


def test_generators_and_exact_bound():
    g = cpu_gen(4)
    v = X.ints((10000,), -2, 2, g, "cpu")
    assert set(v.unique().tolist()) == {-2.0, -1.0, 0.0, 1.0, 2.0}
    f = X.fixed((10000,), 16, 13, g, "cpu")
    k = f * 2 ** 13
    assert torch.equal(k, k.round()) and float(f.abs().max()) < 8
    assert torch.equal(f.float().double(), f)                          # 16-bit significands are fp32-exact ...
    hi = f.float().to(torch.bfloat16).double()
    lo = f - hi
    assert torch.equal(lo.float().to(torch.bfloat16).double(), lo)     # ... and split exactly into bf16 hi + lo
    assert bool((lo != 0).any())
    # the numbers of the GPU table: 27 * 256 * 4 (+ bias) and B D H W * 4 at the largest batch
    X.exact_bound(27 * 256, 2, 2, 1, extra=4)
    X.exact_bound(8 * 45 * 54 * 45, 2, 2, 1)
    X.exact_bound(4 * 64 * 64 * 39, 2, 2, 1)
    X.exact_bound(27, 8, 2, 2.0 ** -13, extra=4)
    with pytest.raises(AssertionError, match="2\\^24"):
        X.exact_bound(8 * 91 * 109 * 91, 2, 2, 1)                       # conv1.0 at full size needs |x|, |dy| <= 1
    # at the bound, fp32 sums are exact in any order; one quantum past it they are not
    n = 2 ** 24
    assert float(torch.tensor(float(n - 1), dtype=torch.float32) + 1) == n
    assert float(torch.tensor(float(n), dtype=torch.float32) + 1) == n


def test_bf16_rne_rounds_once_to_nearest_even():
    ref = torch.tensor([257.0, 259.0, -257.0, 1.0 + 2 ** -8, 27648.0], dtype=torch.float64)
    assert X.bf16_rne(ref).double().tolist() == [256.0, 260.0, -256.0, 1.0, 27648.0]


def test_guard_band_reports_writes_outside_the_tensor():
    buf = X.Guarded((3, 5), torch.bfloat16, "cpu")
    assert bool(buf.t.isnan().all())
    buf.t.fill_(1.0)
    buf.check_bands("inside")
    buf.buf[X.Guarded.BAND + buf.nbytes] = 0
    with pytest.raises(AssertionError, match="outside"):
        buf.check_bands("past the end")


def test_shape_table_reaches_every_tcgen05_plan(built_lib):
    """Every forward / dgrad plan (column kw-stacked and non-stacked; generic with resident and with streamed weights,
    several tiles per weight pass, plane-stack tiles, kw-fused weight boxes; the 1x1x1 GEMM) and both weight-gradient
    kernels are reached by the GPU table, and each case reaches the kernel it names."""
    seen = set()
    for cid, ng, B, (D, H, W), cin, cout, ks, dispatch in X.CONV_CASES:
        for op, kern in dispatch.items():
            if op == "wgrad":
                got = X.wgrad_kernel(ng, W, cin, cout, ks)
                assert built_lib.tmf_conv3d_supported(1, 2, D, H, W, cin, cout, ks) == 1, cid
            else:
                ci, co = (cin, cout) if op == "fwd" else (cout, cin)
                got = X.fwd_kernel(built_lib, ng, B, D, H, W, ci, co, ks)
                assert built_lib.tmf_conv3d_supported(0, 2, D, H, W, ci, co, ks) == 1, cid
            assert got == kern, f"{cid} {op}: {got} (table says {kern})"
            seen.add(got)
    flags = set(" ".join(seen).split())
    assert {"col", "col-ns", "gemm", "wgrad-col", "wgrad-generic"} <= seen
    assert {"resident", "streamed", "stack", "kwf", "mt>1"} <= flags
    assert {ng for _, ng, *rest in X.CONV_CASES} == {1, 2}


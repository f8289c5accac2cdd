"""CPU checks of the BatchNorm / LeakyReLU / pooling test machinery (tests/bn_exact.py): the float64 references against
F.batch_norm -> F.leaky_relu -> max_pool3d / avg_pool3d forward and autograd, the operand generators against the
exactness bounds, the max-pool routing rule, the fp32 tie collapse it has to survive, and the argument refusals of the
C ABI and of sNet (no device work: they fail before any launch)."""
import ctypes as C

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests import bn_exact as N
from tests import conv_exact as X
from transmf_ad_b200 import _lib as L


def cpu_gen(seed):
    return torch.Generator().manual_seed(seed)


def to_ncdhw(t):
    return t.permute(0, 4, 1, 2, 3)


def from_ncdhw(t):
    return t.permute(0, 2, 3, 4, 1)


def torch_layer(y, gamma, beta, rm, rv, training, pool, slope):
    a = F.leaky_relu(F.batch_norm(y, rm, rv, gamma, beta, training, 0.1, 1e-5), slope)
    if pool == N.POOL_MAX:
        return F.max_pool3d(a, 2, 2)
    if pool == N.POOL_AVG:
        return F.avg_pool3d(a, 2, 2)
    return a


@pytest.mark.parametrize("pool", [N.POOL_NONE, N.POOL_MAX, N.POOL_AVG])
@pytest.mark.parametrize("training", [True, False])
@pytest.mark.parametrize("shape", [(2, 5, 6, 7), (1, 4, 3, 2)])
def test_references_match_torch_autograd_in_float64(pool, training, shape):
    """Forward, dgamma = s2, dbeta = s1, dy (bcoef = s / count in training, 0 in eval) and, in eval, the conv bias
    gradient scale * s1, against torch in float64 (odd extents: voxels outside every window)."""
    B, D, H, W = shape
    Cc = 5
    g = cpu_gen(1)
    y = torch.randn(B, D, H, W, Cc, generator=g, dtype=torch.float64) * 2 + 0.3
    gamma = torch.randn(Cc, generator=g, dtype=torch.float64)
    gamma[1] = -abs(gamma[1])
    beta = torch.randn(Cc, generator=g, dtype=torch.float64)
    rm, rv = torch.randn(Cc, generator=g, dtype=torch.float64), torch.rand(Cc, generator=g, dtype=torch.float64) + 0.5
    count = B * D * H * W
    if training:
        mean, var = y.reshape(-1, Cc).mean(0), y.reshape(-1, Cc).var(0, unbiased=False)
    else:
        mean, var = rm, rv
    inv = 1 / torch.sqrt(var + 1e-5)
    coef = torch.stack([gamma * inv, beta - mean * gamma * inv, mean, inv])
    slope = 0.01
    yr, gr, br = (t.clone().requires_grad_(True) for t in (y, gamma, beta))
    ref = torch_layer(to_ncdhw(yr), gr, br, rm.clone(), rv.clone(), training, pool, slope)
    out, ymax = N.fwd_ref(y, coef, pool, slope)
    torch.testing.assert_close(out, from_ncdhw(ref.detach()), rtol=1e-12, atol=1e-12)
    dout = torch.randn(ref.shape, generator=g, dtype=torch.float64)
    ref.backward(dout)
    dout = from_ncdhw(dout).contiguous()
    s1, s2, a1, a2 = N.sums_ref(y, coef, dout, pool, slope)
    torch.testing.assert_close(s2, gr.grad, rtol=1e-10, atol=1e-10)
    torch.testing.assert_close(s1, br.grad, rtol=1e-10, atol=1e-10)
    assert bool((a1 >= s1.abs()).all()) and bool((a2 >= s2.abs()).all())
    bcoef = torch.stack([s1 / count, s2 / count]) if training else torch.zeros(2, Cc, dtype=torch.float64)
    dy = N.apply_ref(y, coef, bcoef, dout, pool, slope)
    torch.testing.assert_close(dy, yr.grad, rtol=1e-10, atol=1e-10)
    if not training:
        torch.testing.assert_close(coef[0] * s1, yr.grad.sum((0, 1, 2, 3)), rtol=1e-10, atol=1e-10)
    if pool == N.POOL_MAX:
        # ymax is y at the window's maximum activation (torch's arg-max), negative scale included
        _, idx = F.max_pool3d(torch_layer(to_ncdhw(y), gamma, beta, rm.clone(), rv.clone(), training, N.POOL_NONE, slope),
                              2, 2, return_indices=True)
        yt = to_ncdhw(y).reshape(B, Cc, -1)
        torch.testing.assert_close(ymax, from_ncdhw(yt.gather(-1, idx.reshape(B, Cc, -1)).reshape(idx.shape)),
                                   rtol=0, atol=0)


def test_finalize_reference_matches_torch_batch_norm():
    """Coefficients and running statistics from row totals equal torch's training-mode batch_norm in float64 to within
    the kernel's fp32 roundings (the reference's own bounds)."""
    g = cpu_gen(2)
    Cc, count = 6, 4 * 5 * 6 * 7
    y = torch.randn(count, Cc, generator=g, dtype=torch.float64) * 3 + 1
    rows = torch.tensor_split(y, 7)
    t1 = sum(r.sum(0) for r in rows).numpy()
    t2 = sum((r * r).sum(0) for r in rows).numpy()
    gamma = torch.randn(Cc, generator=g).numpy()
    beta = torch.randn(Cc, generator=g).numpy()
    rm, rv = torch.randn(Cc, generator=g).numpy(), (torch.rand(Cc, generator=g) + 0.5).numpy()
    want, tol = N.finalize_ref(t1, t2, gamma, beta, rm, rv, count, 0.1, 1e-5, True)
    rmt, rvt = torch.tensor(rm, dtype=torch.float64), torch.tensor(rv, dtype=torch.float64)
    z = F.batch_norm(y, rmt, rvt, torch.tensor(gamma, dtype=torch.float64), torch.tensor(beta, dtype=torch.float64), True,
                     0.1, 1e-5)
    zk = y * torch.tensor(want["scale"]) + torch.tensor(want["shift"])
    assert float((zk - z).abs().max()) < 1e-5
    for name, t in (("rmean", rmt), ("rvar", rvt)):
        assert np.all(np.abs(want[name] - t.numpy()) <= tol[name] + 1e-6 * np.abs(t.numpy())), name
    assert np.all(tol["invstd"] > 0) and np.all(tol["invstd"] < 1e-6 * want["invstd"])


def test_bwd_finalize_reference_rounds_once():
    s1 = np.array([1 + 2.0 ** -30, -3.0, 2.0 ** 40 + 1])
    s2 = np.array([0.1, 2.0 ** -200, -7.0])
    out = N.bwd_finalize_ref(s1, s2, np.array([2.0, -0.5, 1.0]), 3, True)
    assert out["dbeta"].tolist() == [1.0, -3.0, 2.0 ** 40]
    assert out["bcoef"][:3].tolist() == [np.float32(s / 3) for s in s1]
    ev = N.bwd_finalize_ref(s1, s2, np.array([2.0, -0.5, 1.0]), 3, False)
    assert ev["dbias"].tolist() == [2.0, 1.5, 2.0 ** 40] and not ev["bcoef"].any()


def test_route_index_is_max_pool_backward_and_the_sign_rule():
    """Positive scales: torch's first maximum (ties from coarse values included).  Negative scales: the first minimum of
    y.  Zero scales: position 0.  And on dyadic data with slope 1/2 the routed gradient is torch's max_pool3d backward of
    the activation."""
    g = cpu_gen(3)
    y = X.ints((2, 5, 6, 7, 4), -1, 1, g, "cpu")            # three values: ties in nearly every window; odd extents
    dout = torch.randn(2, 2, 3, 3, 4, generator=g, dtype=torch.float64)
    sc = torch.tensor([0.5, -0.25, 0.0, -0.0], dtype=torch.float64)
    idx = N.route_index(y, sc)[..., 0]
    w = N.windows(y)
    assert torch.equal(idx[..., 0], w[..., 0, :].argmax(-1))
    assert torch.equal(idx[..., 1], (-w[..., 1, :]).argmax(-1))
    assert not idx[..., 2:].any()
    yr = to_ncdhw(y[..., :1]).clone().requires_grad_(True)
    F.max_pool3d(yr, 2, 2).backward(to_ncdhw(dout[..., :1]))
    assert torch.equal(from_ncdhw(yr.grad), X.maxpool_route(y[..., :1], dout[..., :1]))
    # through BatchNorm + LeakyReLU on the generators' operands: the rule is torch's rule on the activation
    coef, centre = N.coefs(4, g, "cpu")
    coef[0] = torch.tensor([0.5, -1.75, 0.0, 0.25], dtype=torch.float64)
    y = N.y_values((2, 5, 6, 7, 4), centre, g, "cpu")
    a = N.leaky(y * coef[0] + coef[1], N.SLOPE)
    ar = to_ncdhw(a).clone().requires_grad_(True)
    F.max_pool3d(ar, 2, 2).backward(to_ncdhw(dout))
    dz = N.dz_ref(y, coef, dout, N.POOL_MAX, 1.0)              # slope 1: dz is the routed dout
    assert torch.equal(dz, from_ncdhw(ar.grad))


def test_tie_collapse_example_collapses_in_fp32():
    """scale 2^-20, shift 1: y = 1 and y = 1.0078125 (distinct bf16 values) give the same fp32 activation under fmaf, for
    either sign of the scale; float64 keeps them apart, and the routing rule picks the larger key, not position 0."""
    y0, y1 = N.COLLAPSE_Y
    assert float(torch.tensor(y1).to(torch.bfloat16)) == y1 and y0 != y1
    for sc in (N.COLLAPSE_SCALE, -N.COLLAPSE_SCALE):
        z0, z1 = N.fmaf(y0, sc, N.COLLAPSE_SHIFT), N.fmaf(y1, sc, N.COLLAPSE_SHIFT)
        assert z0 == z1 and z0 > 0, sc
        assert y0 * sc + N.COLLAPSE_SHIFT != y1 * sc + N.COLLAPSE_SHIFT
        # the losing y first, the winner by sign(scale) * y second
        lo, hi = (y0, y1) if sc > 0 else (y1, y0)
        y = torch.full((1, 2, 2, 2, 1), 1.0 - 0.5 * (sc > 0) + 0.5 * (sc < 0), dtype=torch.float64)
        y[0, 0, 0, 0, 0], y[0, 0, 0, 1, 0] = lo, hi
        assert int(N.route_index(y, torch.tensor([sc], dtype=torch.float64))) == 1
    assert N.fmaf(1.0, 1.0, 2.0 ** -24) == 1.0 and N.fmaf(1.0, 1.0, 3 * 2.0 ** -24) == 1 + 2.0 ** -22   # ties to even
    with pytest.raises(AssertionError):
        N.fmaf(0.1, 1.0, 0.0)


def test_generators_respect_the_exactness_bounds():
    g = cpu_gen(4)
    coef, centre = N.coefs(64, g, "cpu")
    sc, sh, mu, inv = coef
    assert float(sc[0]) < 0 and float(sc[1]) == 0 and bool((sc > 0).any())
    for t, q in ((sc, N.Q_SC), (sh, N.Q_SH), (mu, N.Q_Y)):
        k = t / q
        assert torch.equal(k, k.round())
    assert set(torch.log2(inv).tolist()) <= set(N.IS_EXP)
    y = N.y_values((3, 6, 5, 4, 64), centre, g, "cpu")
    assert torch.equal(y.float().to(torch.bfloat16).double(), y)            # bf16-exact, 7 significant bits at most
    assert float((y - mu).abs().max()) <= 9 * N.Q_Y and float(y.abs().max()) <= 4 + 7 * N.Q_Y
    for pool in (N.POOL_NONE, N.POOL_MAX, N.POOL_AVG):
        N.check_design(pool)
    # every sum the GPU table reaches stays within 2^24 quanta per channel, worst case: one term per window (max pool)
    # or per voxel, |dz| <= 1 (2 quanta), |y - mean| <= 9 quanta
    for cid, B, (D, H, W), Cc, pool, _ in N.BN_CASES:
        n = B * (D // 2) * (H // 2) * (W // 2) if pool == N.POOL_MAX else B * D * H * W
        X.exact_bound(n, 2, 9, 1)
    with pytest.raises(AssertionError, match="2\\^24"):
        X.exact_bound(8 * 45 * 54 * 45, 2, 10, 1)                             # one more y step would not fit
    # the data-dependent check
    dout = N.dout_values((3, 3, 2, 2, 64), g, "cpu")
    s1, s2, a1, a2 = N.sums_ref(y, coef, dout, N.POOL_MAX, N.SLOPE)
    N.check_sums_exact(a1, a2, inv, N.POOL_MAX)


def test_references_on_generated_operands_are_fp32_exact_and_round_in_bf16():
    """The references of the exact cases are fp32-exact, and the bf16 outputs need real rounding: values with more than 8
    significant bits and exact halfway cases in the forward output and in dy."""
    g = cpu_gen(5)
    coef, centre = N.coefs(32, g, "cpu")
    y = N.y_values((2, 6, 8, 10, 32), centre, g, "cpu")
    bcoef = N.bcoefs(32, g, "cpu")
    for pool in (N.POOL_NONE, N.POOL_MAX, N.POOL_AVG):
        out, _ = N.fwd_ref(y, coef, pool, N.SLOPE)
        dshape = y.shape if pool == N.POOL_NONE else (2, 3, 4, 5, 32)
        dy = N.apply_ref(y, coef, bcoef, N.dout_values(dshape, g, "cpu"), pool, N.SLOPE)
        for ref in (out, dy):
            X.bf16_rne(ref)
            inexact, half = N.rounding_profile(ref)
            assert inexact > 0 and half > 0, pool
    # the profile counts what it says
    t = torch.tensor([1.0, 1 + 2.0 ** -8, 1 + 2.0 ** -9, 1 + 3 * 2.0 ** -9], dtype=torch.float64)
    assert N.rounding_profile(t) == (3, 1)


def test_windows_roundtrip_and_shape_table():
    g = cpu_gen(6)
    t = torch.randn(2, 5, 6, 7, 3, generator=g, dtype=torch.float64)
    back = N.unwindow(N.windows(t), t.shape)
    assert torch.equal(back[:, :4, :6, :6], t[:, :4, :6, :6]) and not back[:, 4:].any() and not back[..., 6:, :].any()
    ids = [c[0] for c in N.BN_CASES]
    assert len(ids) == len(set(ids)) == 21 + len(N.EDGE_CASES)
    assert [c[3:5] for c in N.MODEL_CASES[:7]] == [(32, 1), (32, 0), (64, 1), (64, 0), (128, 1), (256, 0), (128, 2)]
    chans = {c[3] for c in N.BN_CASES}
    assert {8, 24, 1024} <= chans


# ---------------------------------------------------------------------------------------------------------------
# argument refusals (no device work: the checks run before anything is launched)
_NULL = C.cast(None, C.POINTER(C.c_void_p))


def test_maxpool_entry_points_refuse_a_negative_slope(built_lib):
    lib = built_lib
    for slope in (-0.01, float("nan")):
        calls = {
            "tmf_bn_act_pool_fwd_keepmax": lambda: lib.tmf_bn_act_pool_fwd_keepmax(1, _NULL, _NULL, _NULL, _NULL, 0, 1, 2, 2, 2,
                                                                                   8, slope, None),
            "tmf_bn_act_pool_fwd_keepmax_dual": lambda: lib.tmf_bn_act_pool_fwd_keepmax_dual(1, _NULL, _NULL, _NULL, _NULL,
                                                                                             _NULL, 1, 2, 2, 2, 8, slope, None),
            "tmf_bn_maxpool_bwd_reduce_kept": lambda: lib.tmf_bn_maxpool_bwd_reduce_kept(1, _NULL, 0, _NULL, _NULL, _NULL, 1,
                                                                                         1, 1, 1, 8, slope, None),
            "tmf_bn_act_pool_bwd_reduce": lambda: lib.tmf_bn_act_pool_bwd_reduce(1, _NULL, 0, _NULL, _NULL, _NULL, 1, 2, 2, 2,
                                                                                 8, L.POOL_MAX, slope, None),
            "tmf_bn_act_pool_bwd_apply": lambda: lib.tmf_bn_act_pool_bwd_apply(1, _NULL, 0, _NULL, _NULL, _NULL, _NULL, 1, 2,
                                                                               2, 2, 8, L.POOL_MAX, slope, None),
        }
        for name, call in calls.items():
            assert call() != 0, name
            err = lib.tmf_last_error().decode()
            assert name in err and "slope >= 0" in err, (name, err)
    # no pool, average pool: a negative slope is a valid LeakyReLU there (the call then fails on its NULL pointers)
    for pool in (L.POOL_NONE, L.POOL_AVG):
        assert lib.tmf_bn_act_pool_bwd_apply(1, _NULL, 0, _NULL, _NULL, _NULL, _NULL, 1, 2, 2, 2, 8, pool, -0.01, None) != 0
        assert "slope" not in lib.tmf_last_error().decode()
        assert lib.tmf_bn_act_pool_bwd_reduce(1, _NULL, 0, _NULL, _NULL, _NULL, 1, 2, 2, 2, 8, pool, -0.01, None) != 0
        assert "slope" not in lib.tmf_last_error().decode()


def test_work_index_limit_is_refused_before_allocation(built_lib):
    """B*D*H*W*C/8 >= 2^31 work chunks: refused by fill_args before any pointer is looked at."""
    lib = built_lib
    B, D, H, W = 75, 91, 109, 91
    assert B * D * H * W * 256 // 8 >= 2 ** 31 > B * D * H * W * 32 // 8
    assert lib.tmf_bn_act_pool_fwd(1, _NULL, _NULL, _NULL, 0, B, D, H, W, 256, L.POOL_MAX, 0.01, None) != 0
    assert "32-bit work indices" in lib.tmf_last_error().decode()
    assert lib.tmf_bn_act_pool_bwd_apply(1, _NULL, 0, _NULL, _NULL, _NULL, _NULL, B, D, H, W, 256, L.POOL_NONE, 0.01,
                                         None) != 0
    assert "32-bit work indices" in lib.tmf_last_error().decode()
    # one chunk below the limit passes fill_args and fails on the NULL pointers instead
    assert lib.tmf_bn_act_pool_fwd(1, _NULL, _NULL, _NULL, 0, B, D, H, W, 32, L.POOL_MAX, 0.01, None) != 0
    assert "NULL" in lib.tmf_last_error().decode()


def test_snet_refuses_a_negative_leaky_relu_slope():
    from transmf_ad_b200.models.networks import sNet
    net = sNet(32)
    assert [h[2] for h in net._hyper()] == [0.01] * 7
    net.conv2[5].negative_slope = -0.2
    with pytest.raises(NotImplementedError, match="slopes >= 0"):
        net._hyper()
    net.conv2[5].negative_slope = 0.0                 # ReLU is fine: non-decreasing
    assert net._hyper()[2][2] == 0.0

"""CPU checks of the MiSePyNet exact-arithmetic test machinery (tests/mnet_exact.py): the float64 references against
torch's Conv3d / BatchNorm3d / ReLU / MaxPool3d in the forms the model uses, the operand generators and the 2^24
bound on every table case, the model shapes against Mnet and the oracle, and the table's coverage of every launch
regime through the geometry mirror."""
import os
import re

import pytest
import torch
import torch.nn.functional as F

from oracle import restatement as R
from tests import conv_exact as X
from tests import mnet_exact as M


def cpu_gen(seed):
    return torch.Generator().manual_seed(seed)


def rnd(g, *shape):
    return torch.randn(shape, generator=g, dtype=torch.float64)


@pytest.mark.parametrize("n,cin,A,Bd,L,k", [(2, 3, 4, 5, 9, 4), (1, 8, 2, 3, 7, 7), (2, 1, 3, 1, 6, 1)])
def test_line_references_match_torch(n, cin, A, Bd, L, k):
    """Conv3d(Cin, 8, (1,1,k)) on (N, Cin, A, B, L), the form conv_bn_relu maps to the slice kernels."""
    g = cpu_gen(1)
    x, w, b = rnd(g, n, cin, A, Bd, L), rnd(g, 8, cin, 1, 1, k), rnd(g, 8)
    dy = rnd(g, n, 8, A, Bd, L - k + 1)
    flat = lambda t: t.reshape(t.shape[0], t.shape[1], A * Bd, t.shape[-1])
    w3 = w[:, :, 0, 0, :]
    torch.testing.assert_close(M.line_fwd_ref(flat(x), w3, b), flat(F.conv3d(x, w, b)), rtol=1e-12, atol=1e-12)
    dx = torch.nn.grad.conv3d_input(x.shape, w, dy)
    torch.testing.assert_close(M.line_dgrad_ref(flat(dy), w3, L), flat(dx), rtol=1e-12, atol=1e-12)
    dw, db = M.line_wgrad_ref(flat(dy), flat(x), k)
    torch.testing.assert_close(dw, torch.nn.grad.conv3d_weight(x, w.shape, dy)[:, :, 0, 0, :], rtol=1e-12, atol=1e-12)
    torch.testing.assert_close(db, dy.sum((0, 2, 3, 4)), rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize("n,cin,cout,X_,Y_,kh,kw,s", [(2, 3, 4, 12, 15, 3, 4, 2), (1, 2, 3, 11, 8, 2, 2, 3),
                                                    (2, 5, 2, 9, 8, 1, 1, 2), (1, 2, 2, 7, 6, 7, 6, 1)])
def test_spatial_references_match_torch(n, cin, cout, X_, Y_, kh, kw, s):
    """Conv3d(Cin, Cout, (kh,kw,1), stride (s,s,s)) on (N, Cin, X, Y, 1), stride > kernel and dead rows included."""
    g = cpu_gen(2)
    x, w, b = rnd(g, n, cin, X_, Y_, 1), rnd(g, cout, cin, kh, kw, 1), rnd(g, cout)
    y = F.conv3d(x, w, b, stride=s)
    dy = rnd(g, *y.shape)
    x2, w2, dy2 = x[..., 0], w[..., 0], dy[..., 0]
    torch.testing.assert_close(M.conv2d_fwd_ref(x2, w2, b, s), y[..., 0], rtol=1e-12, atol=1e-12)
    dx = torch.nn.grad.conv3d_input(x.shape, w, dy, stride=s)[..., 0]
    torch.testing.assert_close(M.conv2d_dgrad_ref(dy2, w2, s, X_, Y_), dx, rtol=1e-12, atol=1e-12)
    dw, db = M.conv2d_wgrad_ref(dy2, x2, kh, kw, s)
    torch.testing.assert_close(dw, torch.nn.grad.conv3d_weight(x, w.shape, dy, stride=s)[..., 0], rtol=1e-12, atol=1e-12)
    torch.testing.assert_close(db, dy.sum((0, 2, 3, 4)), rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize("training", [True, False])
def test_bn_relu_references_match_torch_autograd(training):
    """coef / bcoef built the way tmf_bn_finalize / tmf_bn_bwd_finalize build them reproduce F.batch_norm + ReLU,
    forward and backward (dx, dgamma, dbeta), in train and eval mode."""
    g = cpu_gen(3)
    n, C, S, eps = 3, 5, 40, 1e-5
    x, dout = rnd(g, n, C, S) * 1.5 + 0.3, rnd(g, n, C, S)
    gamma, beta = rnd(g, C).requires_grad_(True), rnd(g, C).requires_grad_(True)
    rm, rv = rnd(g, C) * 0.2, torch.rand(C, generator=g, dtype=torch.float64) + 0.5
    xr = x.clone().requires_grad_(True)
    out = F.relu(F.batch_norm(xr, rm.clone(), rv.clone(), gamma, beta, training, 0.1, eps))
    out.backward(dout)
    count = n * S
    if training:
        s1, s2 = M.bn_stats_ref(x)
        mean, var = s1 / count, s2 / count - (s1 / count) ** 2
    else:
        mean, var = rm, rv
    inv = 1 / torch.sqrt(var + eps)
    sc = gamma.detach() * inv
    coef = torch.stack([sc, beta.detach() - mean * sc, mean, inv])
    torch.testing.assert_close(M.bn_relu_fwd_ref(x, coef), out.detach(), rtol=1e-12, atol=1e-12)
    d1, d2, _, _ = M.bn_bwd_sums_ref(dout, x, coef)
    torch.testing.assert_close(d2, gamma.grad, rtol=1e-12, atol=1e-12)
    torch.testing.assert_close(d1, beta.grad, rtol=1e-12, atol=1e-12)
    bcoef = torch.stack([d1 / count, d2 / count]) if training else torch.zeros(2, C, dtype=torch.float64)
    torch.testing.assert_close(M.bn_apply_ref(dout, x, coef, bcoef), xr.grad, rtol=1e-10, atol=1e-10)


@pytest.mark.parametrize("NC,X_,Y_,ph,pw,ninf", [(4, 9, 10, 3, 3, False), (3, 9, 9, 2, 3, True), (2, 31, 35, 15, 17, False)])
def test_maxpool_references_match_torch_with_ties(NC, X_, Y_, ph, pw, ninf):
    """F.max_pool3d((ph,pw,1)) forward values and indices and its backward, ties everywhere ({-1, 0, 1}) and -inf
    windows included: torch also routes to the first maximum in scan order."""
    case = ("t", NC, X_, Y_, ph, pw, ninf)
    x, dy = M.pool_operands(case, cpu_gen(4), "cpu")
    xr = x.view(1, NC, X_, Y_, 1).clone().requires_grad_(True)
    y, ind = F.max_pool3d(xr, (ph, pw, 1), return_indices=True)
    y.backward(dy.view(y.shape))
    yr, idx = M.maxpool_fwd_ref(x, ph, pw)
    assert torch.equal(yr, y.detach().view(yr.shape))
    Xo, Yo = yr.shape[1:]
    ox, oy = torch.arange(Xo).view(-1, 1), torch.arange(Yo).view(1, -1)
    flat = (ox * ph + idx // pw) * Y_ + oy * pw + idx % pw          # window-local a*pw + b -> torch's plane index
    assert torch.equal(flat, ind.view(flat.shape))
    assert torch.equal(M.maxpool_bwd_ref(dy, idx, ph, pw, X_, Y_), xr.grad.view(NC, X_, Y_))
    if ninf:
        assert bool(torch.isinf(yr).any()) and int(idx[0, 0, 0]) == 0


def test_integer_operands_give_integer_references():
    g = cpu_gen(5)
    x, w, b, dy = M.line_operands(("t", 2, 3, 7, 11, 4), g, "cpu")
    for t in (M.line_fwd_ref(x, w, b), M.line_dgrad_ref(dy, w, 11), *M.line_wgrad_ref(dy, x, 4)):
        assert torch.equal(t, t.round())
    x5 = x.view(2, 3, 7, 1, 11)
    assert torch.equal(M.line_fwd_ref(x, w, b), F.conv3d(x5, w.view(8, 3, 1, 1, 4), b).view(2, 8, 7, 8))
    x, w, b, dy = M.conv2d_operands(("t", 2, 3, 4, 12, 15, 3, 4, 2), g, "cpu")
    for t in (M.conv2d_fwd_ref(x, w, b, 2), M.conv2d_dgrad_ref(dy, w, 2, 12, 15), *M.conv2d_wgrad_ref(dy, x, 3, 4, 2)):
        assert torch.equal(t, t.round())
    assert torch.equal(M.conv2d_fwd_ref(x, w, b, 2), F.conv3d(x[..., None], w[..., None], b, stride=2)[..., 0])
    x, coef, bcoef, dout = M.bn_operands(("t", 3, 6, 50), g, "cpu")
    for t, q in ((M.bn_relu_fwd_ref(x, coef), 2.0 ** -3), (M.bn_apply_ref(dout, x, coef, bcoef), 2.0 ** -7)):
        assert torch.equal(t / q, (t / q).round())
    assert float(coef[0, 0]) < 0 and float(coef[0, 1]) == 0


def test_every_table_case_passes_the_exact_bound():
    """The generators assert the bound on the operands they return; at the largest slice layers too (N*P*Lo and
    N*S = 1.2e6 terms)."""
    g = cpu_gen(6)
    for c in M.LINE_CASES:
        M.line_operands(c, g, "cpu")
    for c in M.CONV_CASES:
        M.conv2d_operands(c, g, "cpu")
    for c in M.BN_CASES:
        M.bn_operands(c, g, "cpu")
    with pytest.raises(AssertionError, match="2\\^24"):     # the line weight gradient of conv3.0 with |x| <= 8
        X.exact_bound(2 * 8281 * 73, 2, 8, 1)


def test_exact_bound_binds_the_bn_sums():
    """bn_operands' bound is live: the sum of squares of a 1.2e6-term channel is a few 2^22 quanta."""
    x, _, _, _ = M.bn_operands(("t", 2, 1, 605059), cpu_gen(7), "cpu")
    q = float((x * x).sum()) / M.Q_X ** 2
    assert 2 ** 22 < q < X.FP32_EXACT


def _record_model_calls(monkeypatch):
    """Run the oracle's slice / spatial stacks of each view on one 91x109x91 sample (eval mode, CPU) and record every
    conv3d (input shape, weight shape, stride) and max_pool3d (input shape, kernel)."""
    from transmf_ad_b200.models.MiSePyNet import Mnet
    convs, pools = [], []
    conv3d, max_pool3d = F.conv3d, F.max_pool3d

    def rec_conv(x, w, b=None, stride=1, *a, **kw):
        convs.append((tuple(x.shape), tuple(w.shape), stride))
        return conv3d(x, w, b, stride, *a, **kw)

    def rec_pool(x, k, *a, **kw):
        pools.append((tuple(x.shape), tuple(k)))
        return max_pool3d(x, k, *a, **kw)

    monkeypatch.setattr(F, "conv3d", rec_conv)
    monkeypatch.setattr(F, "max_pool3d", rec_pool)
    model = Mnet()
    sd = model.state_dict()
    img = torch.rand((1, 1, 91, 109, 91), generator=cpu_gen(8))
    with torch.no_grad():
        for name, v in (("axial", img), ("col", img.permute(0, 1, 2, 4, 3)), ("sag", img.permute(0, 1, 4, 3, 2))):
            s = R.slice_cnn_forward(sd, f"mri.slice_cnn_{name}", v, False)
            R.spatial_cnn_forward(sd, f"mri.spatial_cnn_{name}", *s, False)
    return model, convs, pools


def test_model_shapes_are_what_mnet_produces(monkeypatch):
    """The table's model cases are exactly the layers Mnet runs: kernel sizes and strides from the modules of a CPU
    Mnet(), activation extents from the oracle's slice / spatial stacks."""
    model, convs, pools = _record_model_calls(monkeypatch)
    mods = []
    net = model.mri
    for slc, spat in ((net.slice_cnn_axial, net.spatial_cnn_axial), (net.slice_cnn_col, net.spatial_cnn_col)):
        for seq in (slc.conv1, slc.conv2, slc.conv3, spat.conv1):
            mods += [m for m in seq if isinstance(m, torch.nn.Conv3d)]
    called = {(w, s if isinstance(s, int) else s[0]) for _, w, s in convs}
    assert called == {(tuple(m.weight.shape), m.stride[0]) for m in mods}
    assert all(len(set(m.stride)) == 1 for m in mods)
    line, conv, bn, pool = set(), set(), set(), set()
    for xs, ws, s in convs:
        cout, cin, kd, kh, kw = ws
        if kw == 1:                                   # (kh, kw, 1): the spatial kernels (conv_bn_relu's rule)
            conv.add((cin, cout, xs[2], xs[3], kd, kh, s))
            Xo, Yo = M.conv2d_out(xs[2], xs[3], kd, kh, s)
            bn.add((cout, Xo * Yo))
        else:
            assert kd == kh == 1 and s == 1 and cout == M.LC_CO
            line.add((cin, xs[2] * xs[3], xs[4], kw))
            bn.add((cout, xs[2] * xs[3] * (xs[4] - kw + 1)))
    for xs, (ph, pw, pz) in pools:
        assert pz == 1 and xs[-1] == 1
        pool.add((xs[1], xs[2], xs[3], ph, pw))
    assert {c[2:] for c in M.LINE_MODEL} == line
    assert {c[2:] for c in M.CONV_MODEL} == conv
    assert {c[2:] for c in M.BN_MODEL} == bn
    assert {(c[1] // M.B,) + c[2:6] for c in M.POOL_MODEL} == pool
    for cases in (M.LINE_MODEL, M.CONV_MODEL, M.BN_MODEL):
        assert {c[1] for c in cases} == {M.B}


def test_shape_table_reaches_every_regime():
    """Through the geometry mirror: every regime of mnet_exact.REGIMES is reached by the GPU table, and each edge case
    is the only case of its table reaching one of them (removing any case loses a regime; the model cases are pinned
    by test_model_shapes_are_what_mnet_produces)."""
    for fam, (cases, regimes) in M.TABLES.items():
        reach = {c[0]: regimes(c) for c in cases}
        seen = set().union(*reach.values())
        assert M.REGIMES[fam] <= seen, f"{fam}: not reached: {sorted(M.REGIMES[fam] - seen)}"
        for cid, r in reach.items():
            if not cid.startswith("edge-"):
                continue
            others = set().union(*(v for k, v in reach.items() if k != cid))
            assert (r & M.REGIMES[fam]) - others, f"{fam} {cid}: every regime it reaches is reached by another case"
        assert len(reach) == len(cases), f"{fam}: duplicate case ids"


def test_geometry_mirror_follows_mnet_ops(built_lib):
    """The constants the mirror copies still appear in csrc/mnet_ops.cu as the mirror reads them, and the library's
    host-side sizes agree with them (one workspace row per wgrad block, TMF_STAT_ROWS)."""
    src = open(os.path.join(os.path.dirname(__file__), "..", "transmf_ad_b200", "csrc", "mnet_ops.cu")).read()
    assert "grid_for(int64_t total, int cap = 148 * 16)" in src and "(total + 255) / 256" in src
    assert "lines < 592 ? lines : 592" in src
    assert "LC_CO * Cin * k <= 16 * 256" in src
    assert "sizeof(float) * ((size_t)LC_CO * (L - k + 1) + (size_t)Cin * L)" in src
    assert len(re.findall(r"\(\(int64_t\)N \* S \+ 256 \* 8 - 1\) / \(256 \* 8\)", src)) == 2
    assert M.grid_for(1) == 1 and M.grid_for(M.GRID_CAP * 256) == M.GRID_CAP and M.grid_for(10 ** 9) == M.GRID_CAP
    assert not M.grid_strides(M.GRID_CAP * 256) and M.grid_strides(M.GRID_CAP * 256 + 1)
    assert M.stat_rows(1) == 1 and M.stat_rows(2049) == 2 and M.stat_rows(10 ** 7) == M.STAT_ROWS
    assert M.line_wgrad_per_thread(8, 64) == 16 and M.line_wgrad_smem(8, 799, 64) <= M.SMEM_LIMIT
    assert M.line_wgrad_smem(8, 800, 64) > M.SMEM_LIMIT
    assert built_lib.tmf_stat_rows() == M.STAT_ROWS
    for cin, k in ((1, 1), (3, 5), (8, 64)):
        nw = M.LC_CO * cin * k
        assert built_lib.tmf_line_conv_wgrad_workspace_bytes(cin, k) == 4 * M.LINE_WGRAD_BLOCKS * (nw + M.LC_CO)

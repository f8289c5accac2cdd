"""Exact-arithmetic tests of the sNet BatchNorm / LeakyReLU / pooling kernels (csrc/bn_act_pool.cu) at the model's own
layer shapes.

Operands sit on short dyadic grids (tests/bn_exact.py): every element-wise value is exact in fp32, and the backward sums
stay below 2^24 quanta per channel over the whole tower, so a correct kernel reproduces the float64 reference bit for
bit whatever its plan (row chunking, grid caps, more units than blocks, idle threads) -- one misrouted window, one
unwritten voxel or one dropped partial fails on the element it touches.  Every output is poisoned with NaN bytes and
sits inside guard bands, every call runs twice and must give the same bits, and every statistics buffer must have all
TMF_STAT_ROWS rows written (include/tmf.h, DETERMINISM).

One Gaussian chained case per pool mode (slope 0.01, coefficients from tmf_bn_finalize) checks the rounding that dyadic
data cannot see against float64 torch autograd under a per-element bound."""
import zlib

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests import bn_exact as N
from tests import conv_exact as X
from tests.test_gpu_conv_exact import conv1_wgrad_operands, run_twice, workspace
from transmf_ad_b200 import _lib as L

pytestmark = pytest.mark.gpu
DEV = "cuda"
U = 2.0 ** -24


def gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def f32(t):
    return t.float().contiguous()


def bf16(t):
    return t.to(torch.bfloat16).contiguous()


def guarded(shape, dtype, ng):
    return [X.Guarded(tuple(shape), dtype, DEV) for _ in range(ng)]


def ts(gs):
    return [g.t for g in gs]


def check(got, want, what):
    err = X.mismatch(got, want)
    assert not err, f"{what}: {err}"


def check_rows(rows, s1, s2, what):
    """All TMF_STAT_ROWS rows written (finite after poisoning); the row totals are the reference sums bit for bit."""
    assert rows.shape[0] == L.stat_rows()
    assert bool(torch.isfinite(rows).all()), f"{what}: statistics rows left unwritten"
    C = s1.shape[0]
    tot = rows.sum(0)
    check(tot[:C], s1, f"{what}: sum dz")
    check(tot[C:], s2, f"{what}: sum dz*xhat")


class Layer:
    """Operands and float64 references of one (case, tower set): towers differ in data and coefficients."""

    def __init__(self, case, towers):
        cid, B, (D, H, W), C, pool, last = case
        self.B, self.shape, self.C, self.pool, self.last = B, (D, H, W), C, pool, last
        self.pshape = (B, D, H, W, C) if pool == N.POOL_NONE else (B, D // 2, H // 2, W // 2, C)
        q_dz = N.check_design(pool)
        assert q_dz > 0
        self.y, self.coef, self.bcoef, self.dout = [], [], [], []
        for t in towers:
            g = gen(zlib.crc32(f"{cid}/{t}".encode()))
            coef, centre = N.coefs(C, g, DEV)
            self.coef.append(coef)
            self.y.append(N.y_values((B, D, H, W, C), centre, g, DEV))
            self.bcoef.append(N.bcoefs(C, g, DEV))
            self.dout.append(N.dout_values(self.pshape, g, DEV))
        self.y_b = [bf16(t) for t in self.y]
        self.coef32 = [f32(c.reshape(-1)) for c in self.coef]
        self.bcoef32 = [f32(c.reshape(-1)) for c in self.bcoef]
        self.zero_bcoef = [torch.zeros(2 * C, device=DEV) for _ in towers]


def fwd_calls(lay, ng, y, coef, pool, last):
    B, (D, H, W), C = lay.B, lay.shape, lay.C
    return {
        "fwd": lambda out: L.call("tmf_bn_act_pool_fwd", ng, L.ptrs(y), L.ptrs(coef), L.ptrs(out), int(last), B, D, H, W, C,
                                  pool, N.SLOPE),
        "dual": lambda out, o32: L.call("tmf_bn_act_pool_fwd_dual", ng, L.ptrs(y), L.ptrs(coef), L.ptrs(out), L.ptrs(o32), B,
                                        D, H, W, C, pool, N.SLOPE),
        "keep": lambda out, ym: L.call("tmf_bn_act_pool_fwd_keepmax", ng, L.ptrs(y), L.ptrs(coef), L.ptrs(out), L.ptrs(ym),
                                       int(last), B, D, H, W, C, N.SLOPE),
        "keep_dual": lambda out, o32, ym: L.call("tmf_bn_act_pool_fwd_keepmax_dual", ng, L.ptrs(y), L.ptrs(coef),
                                                 L.ptrs(out), L.ptrs(o32), L.ptrs(ym), B, D, H, W, C, N.SLOPE),
    }


def run_forward(lay, idx, refs, what):
    """Every forward variant the layer's pool reaches on towers idx; returns the kept ymax (max pool)."""
    ng = len(idx)
    y, coef = [lay.y_b[i] for i in idx], [lay.coef32[i] for i in idx]
    calls = fwd_calls(lay, ng, y, coef, lay.pool, lay.last)
    odt = torch.float32 if lay.last else torch.bfloat16
    out = guarded(lay.pshape, odt, ng)
    want = [X.bf16_rne(refs[i][0]) if not lay.last else refs[i][0].float() for i in idx]
    want16 = [X.bf16_rne(refs[i][0]) for i in idx]
    ymax = None
    if lay.pool == N.POOL_MAX:
        ym = guarded(lay.pshape, torch.bfloat16, ng)
        got = run_twice(out + ym, lambda: calls["keep"](ts(out), ts(ym)))
        for k, i in enumerate(idx):
            check(got[ng + k], bf16(refs[i][1]), f"{what} keepmax ymax, tower {i}")
            check(got[k], want[k], f"{what} keepmax out, tower {i}")
        ymax = [t.clone() for t in got[ng:]]
        out16, o32 = guarded(lay.pshape, torch.bfloat16, ng), guarded(lay.pshape, torch.float32, ng)
        got = run_twice(out16 + o32 + ym, lambda: calls["keep_dual"](ts(out16), ts(o32), ts(ym)))
        for k, i in enumerate(idx):
            check(got[k], want16[k], f"{what} keepmax_dual out, tower {i}")
            check(got[ng + k].double(), refs[i][0], f"{what} keepmax_dual out32, tower {i}")
            check(got[2 * ng + k], ymax[k], f"{what} keepmax_dual ymax, tower {i}")
    got = run_twice(out, lambda: calls["fwd"](ts(out)))
    for k, i in enumerate(idx):
        check(got[k], want[k], f"{what} fwd out, tower {i}")
    out16, o32 = guarded(lay.pshape, torch.bfloat16, ng), guarded(lay.pshape, torch.float32, ng)
    got = run_twice(out16 + o32, lambda: calls["dual"](ts(out16), ts(o32)))
    for k, i in enumerate(idx):
        check(got[k], want16[k], f"{what} fwd_dual out, tower {i}")
        check(got[ng + k].double(), refs[i][0], f"{what} fwd_dual out32, tower {i}")
    return ymax


def run_reduce(lay, idx, dout, ymax, sums, what, generic):
    """The backward reduction the train path runs (the kept-maximum kernel for max pools and for no pool), or the
    generic full-resolution kernel (average pool; max pool as the TMF_KEEP_YMAX=0 cross-check)."""
    ng = len(idx)
    B, (D, H, W), C = lay.B, lay.shape, lay.C
    fp32 = int(dout[0].dtype == torch.float32)
    coef = [lay.coef32[i] for i in idx]
    rows = guarded((L.stat_rows(), 2 * C), torch.float64, ng)
    if lay.pool == N.POOL_MAX and not generic:
        launch = lambda: L.call("tmf_bn_maxpool_bwd_reduce_kept", ng, L.ptrs(dout), fp32, L.ptrs(ymax), L.ptrs(coef),
                                L.ptrs(ts(rows)), B, D // 2, H // 2, W // 2, C, N.SLOPE)
    else:
        y = [lay.y_b[i] for i in idx]
        launch = lambda: L.call("tmf_bn_act_pool_bwd_reduce", ng, L.ptrs(dout), fp32, L.ptrs(y), L.ptrs(coef),
                                L.ptrs(ts(rows)), B, D, H, W, C, lay.pool, N.SLOPE)
    got = run_twice(rows, launch)
    for k, i in enumerate(idx):
        check_rows(got[k], sums[i][0], sums[i][1], f"{what} tower {i}")
    return got


def run_bwd_finalize(lay, idx, rows, what):
    ng = len(idx)
    C, count = lay.C, lay.B * lay.shape[0] * lay.shape[1] * lay.shape[2]
    coef = [lay.coef32[i] for i in idx]
    for training in (1, 0):
        dg, db, dbias = (guarded((C,), torch.float32, ng) for _ in range(3))
        bc = guarded((2 * C,), torch.float32, ng)
        got = run_twice(dg + db + dbias + bc, lambda: L.call("tmf_bn_bwd_finalize", ng, L.ptrs(rows), L.ptrs(coef),
                                                              L.ptrs(ts(dg)), L.ptrs(ts(db)), L.ptrs(ts(dbias)),
                                                              L.ptrs(ts(bc)), C, count, training))
        for k, i in enumerate(idx):
            tot = rows[k].sum(0).cpu().numpy()
            want = N.bwd_finalize_ref(tot[:C], tot[C:], lay.coef[i][0].cpu().numpy(), count, training)
            for j, name in enumerate(("dgamma", "dbeta", "dbias", "bcoef")):
                check(got[j * ng + k].cpu(), torch.from_numpy(want[name]), f"{what} bwd_finalize({training}) {name}, tower {i}")


def run_apply(lay, idx, dout, bcoef, refs, what, generic, monkeypatch):
    ng = len(idx)
    B, (D, H, W), C = lay.B, lay.shape, lay.C
    fp32 = int(dout[0].dtype == torch.float32)
    y, coef = [lay.y_b[i] for i in idx], [lay.coef32[i] for i in idx]
    if generic:
        monkeypatch.setenv("TMF_BN_GENERIC_MAXPOOL_BWD", "1")
    else:
        monkeypatch.delenv("TMF_BN_GENERIC_MAXPOOL_BWD", raising=False)
    dy = guarded((B, D, H, W, C), torch.bfloat16, ng)
    got = run_twice(dy, lambda: L.call("tmf_bn_act_pool_bwd_apply", ng, L.ptrs(dout), fp32, L.ptrs(y), L.ptrs(coef),
                                       L.ptrs(bcoef), L.ptrs(ts(dy)), B, D, H, W, C, lay.pool, N.SLOPE))
    monkeypatch.delenv("TMF_BN_GENERIC_MAXPOOL_BWD", raising=False)
    for k, i in enumerate(idx):
        check(got[k], refs[k], f"{what} tower {i}")


@pytest.mark.parametrize("case", N.BN_CASES, ids=[c[0] for c in N.BN_CASES])
def test_bn_act_pool_exact(case, monkeypatch):
    """Two towers with different data and coefficients, then the second tower alone (with the other gradient dtype):
    forward (plain, dual, and for max pools keepmax and keepmax_dual), the backward reduction the train path runs (and
    the generic one for max pools), tmf_bn_bwd_finalize in training and eval, and the apply pass (packed and generic
    for max pools) with training and eval coefficients."""
    cid = case[0]
    lay = Layer(case, (0, 1))
    pool = lay.pool
    fwd = [N.fwd_ref(lay.y[i], lay.coef[i], pool, N.SLOPE) for i in (0, 1)]
    if cid.startswith("bench-"):
        # the outputs need bf16 rounding, ties to even included (checked once per layer at the bench extents)
        inexact, half = N.rounding_profile(fwd[0][0])
        assert inexact > 0 and half > 0, "forward data does not exercise bf16 rounding"
    sums = []
    for i in (0, 1):
        s1, s2, a1, a2 = N.sums_ref(lay.y[i], lay.coef[i], lay.dout[i], pool, N.SLOPE)
        N.check_sums_exact(a1, a2, lay.coef[i][3], pool)
        sums.append((s1, s2))
    natural = torch.float32 if lay.last else torch.bfloat16
    other = torch.bfloat16 if lay.last else torch.float32
    for idx, ddt in (((0, 1), natural), ((1,), other)):
        what = f"{cid} ng={len(idx)}"
        ymax = run_forward(lay, idx, fwd, what)
        dout = [lay.dout[i].to(ddt).contiguous() for i in idx]
        kinds = [False, True] if pool == N.POOL_MAX else [False]
        for generic in kinds:
            rows = run_reduce(lay, idx, dout, ymax, sums, f"{what} reduce{' generic' if generic else ''}", generic)
        run_bwd_finalize(lay, idx, rows, what)
        for bname in ("train", "eval"):
            refs = []
            for i in idx:
                ref = N.apply_ref(lay.y[i], lay.coef[i], lay.bcoef[i] if bname == "train" else torch.zeros_like(lay.bcoef[i]),
                                  lay.dout[i], pool, N.SLOPE)
                if bname == "train" and len(idx) == 2 and i == 0 and cid.startswith("bench-"):
                    inexact, half = N.rounding_profile(ref)
                    assert inexact > 0 and half > 0, "dy data does not exercise bf16 rounding"
                refs.append(X.bf16_rne(ref))
                del ref
            bc = [lay.bcoef32[i] for i in idx] if bname == "train" else [lay.zero_bcoef[i] for i in idx]
            for generic in ([False, True] if pool == N.POOL_MAX else [False]):
                if bname == "eval" and generic:
                    continue
                run_apply(lay, idx, dout, bc, refs, f"{what} apply {bname}{' generic' if generic else ''}", generic,
                          monkeypatch)
            del refs
        torch.cuda.empty_cache()


# ---------------------------------------------------------------------------------------------------------------
# tmf_bn_finalize / tmf_bn_bwd_finalize with every statistics row in use
def distinct_rows(C, gen_, lo, hi):
    """[TMF_STAT_ROWS, C] random non-zero integers (float64) from a wide range: a skipped or foreign row changes every
    total."""
    v = torch.randint(lo, hi, (L.stat_rows(), C), generator=gen_).double()
    v[v == 0] = hi
    return v


@pytest.mark.parametrize("C", [8, 24, 256, 1024])
@pytest.mark.parametrize("mode", ["train", "train-null-running", "eval"])
def test_bn_finalize(C, mode):
    ng = 2
    training = mode != "eval"
    cg = torch.Generator().manual_seed(C)
    count = 100_003
    rows, t1s, t2s = [], [], []
    for t in range(ng):
        r1 = distinct_rows(C, cg, -100_000, 100_000)
        r2 = distinct_rows(C, cg, 1, 60_000_000)
        rows.append(torch.cat([r1, r2], 1).to(DEV).contiguous())
        t1s.append(r1.sum(0).numpy())
        t2s.append(r2.sum(0).numpy())
    gamma = [(torch.randn(C, generator=cg) * 0.5 + 1).float() for _ in range(ng)]
    beta = [(torch.randn(C, generator=cg) * 0.3).float() for _ in range(ng)]
    rm0 = [(torch.randn(C, generator=cg) * 0.2).float() for _ in range(ng)]
    rv0 = [(torch.rand(C, generator=cg) + 0.5).float() for _ in range(ng)]
    null_running = mode == "train-null-running"
    rm = [t.to(DEV) for t in rm0]
    rv = [t.to(DEV) for t in rv0]
    nbt = [torch.full((1,), 5, dtype=torch.int64, device=DEV) for _ in range(ng)]
    coef = guarded((4 * C,), torch.float32, ng)
    gamma_d, beta_d = [t.to(DEV) for t in gamma], [t.to(DEV) for t in beta]
    for call in range(2):
        for c in coef:
            c.poison()
        L.call("tmf_bn_finalize", ng, L.ptrs(rows) if training else L.ptrs(None), L.ptrs(gamma_d), L.ptrs(beta_d), L.ptrs(None if null_running else rm),
               L.ptrs(None if null_running else rv), L.ptrs(None if null_running else nbt), L.ptrs(ts(coef)), C, count,
               0.1, 1e-5, int(training))
        torch.cuda.synchronize()
        for t in range(ng):
            coef[t].check_bands("coef")
            want, tol = N.finalize_ref(t1s[t], t2s[t], gamma[t].numpy(), beta[t].numpy(), rm0[t].numpy() if call == 0 else
                                       prev_rm[t], rv0[t].numpy() if call == 0 else prev_rv[t], count, 0.1, 1e-5, training)
            got = coef[t].t.cpu().double().numpy().reshape(4, C)
            if training:
                var_ok = np.float32(np.maximum(t2s[t] / count - (t1s[t] / count) ** 2, 0))
                assert np.all(var_ok > 10), "test statistics must not cancel"
            assert np.array_equal(got[2], want["mean"]), f"tower {t}: mean"
            for j, name in ((3, "invstd"), (0, "scale"), (1, "shift")):
                err = np.abs(got[j] - want[name])
                assert np.all(err <= tol[name]), f"tower {t}: {name}, worst {float((err / np.maximum(tol[name], 1e-300)).max())} x bound"
            if not null_running:
                for name, buf in (("rmean", rm), ("rvar", rv)):
                    g_ = buf[t].cpu().double().numpy()
                    if training:
                        assert np.all(np.abs(g_ - want[name]) <= tol[name]), f"tower {t}: {name}"
                    else:
                        assert np.array_equal(g_, want[name]), f"tower {t}: {name} changed in eval"
                assert int(nbt[t]) == 5 + (call + 1) * int(training), f"tower {t}: num_batches_tracked {int(nbt[t])}"
        if not null_running:
            prev_rm = [b.cpu().numpy() for b in rm]
            prev_rv = [b.cpu().numpy() for b in rv]
        else:
            prev_rm, prev_rv = [t.numpy() for t in rm0], [t.numpy() for t in rv0]


@pytest.mark.parametrize("C", [24, 256])
@pytest.mark.parametrize("training", [1, 0])
def test_bn_bwd_finalize_every_row(C, training):
    ng = 2
    cg = torch.Generator().manual_seed(7 + C)
    count = 874_800
    rows = []
    for t in range(ng):
        r = torch.cat([distinct_rows(C, cg, -2 ** 30, 2 ** 30), distinct_rows(C, cg, -2 ** 30, 2 ** 30)], 1) * 2.0 ** -10
        rows.append(r.to(DEV).contiguous())
    coef = [torch.cat([torch.randn(C, generator=cg), torch.randn(3 * C, generator=cg)]).float().to(DEV) for _ in range(ng)]
    for dbias_null in (False, True):
        dg, db, bc = (guarded((k * C,), torch.float32, ng) for k in (1, 1, 2))
        dbias = guarded((C,), torch.float32, ng)
        outs = dg + db + bc + ([] if dbias_null else dbias)
        got = run_twice(outs, lambda: L.call("tmf_bn_bwd_finalize", ng, L.ptrs(rows), L.ptrs(coef), L.ptrs(ts(dg)),
                                             L.ptrs(ts(db)), L.ptrs(None if dbias_null else ts(dbias)), L.ptrs(ts(bc)), C,
                                             count, training))
        for t in range(ng):
            tot = rows[t].sum(0).cpu().numpy()      # exact: multiples of 2^-10 far below 2^53 quanta
            want = N.bwd_finalize_ref(tot[:C], tot[C:], coef[t][:C].cpu().numpy(), count, training)
            names = ("dgamma", "dbeta", "bcoef") + (() if dbias_null else ("dbias",))
            for j, name in enumerate(names):
                check(got[j * ng + t].cpu(), torch.from_numpy(want[name]), f"tower {t}: {name}")


# ---------------------------------------------------------------------------------------------------------------
# the tie collapse: every kernel that routes a max-pool gradient agrees on one winner
def collapse_operands(shape, g):
    """32 channels, scale +-2^-20 (even / odd channels), shift 1: every window holds the collapsing pair at two random
    positions p < p', the loser by sign(scale) * y at p (torch's first maximum of the fp32 activation) and the winner
    at p'; the other positions hold clearly smaller activations."""
    B, D, H, W = shape
    C = 32
    sc = torch.tensor([N.COLLAPSE_SCALE if c % 2 == 0 else -N.COLLAPSE_SCALE for c in range(C)], dtype=torch.float64,
                      device=DEV)
    pick = lambda pos, neg: torch.where(sc > 0, torch.full_like(sc, pos), torch.full_like(sc, neg))
    y_lose, y_win = pick(*N.COLLAPSE_Y), pick(*N.COLLAPSE_Y[::-1])
    y_other = pick(0.5, 1.5)
    Do, Ho, Wo = D // 2, H // 2, W // 2
    nwin = B * Do * Ho * Wo * C
    perm = torch.rand((nwin, 8), generator=g, device=DEV).argsort(-1)[:, :2].sort(-1).values
    win = y_other.repeat(B * Do * Ho * Wo).reshape(nwin, 1).expand(nwin, 8).clone()
    cidx = torch.arange(C, device=DEV).repeat(B * Do * Ho * Wo)
    win.scatter_(1, perm[:, :1], y_lose[cidx].unsqueeze(1))
    win.scatter_(1, perm[:, 1:], y_win[cidx].unsqueeze(1))
    y = N.unwindow(win.reshape(B, Do, Ho, Wo, C, 8), (B, D, H, W, C))
    coef = torch.stack([sc, torch.full_like(sc, N.COLLAPSE_SHIFT), torch.full_like(sc, 0.5), torch.ones_like(sc)])
    dout = N.dout_values((B, Do, Ho, Wo, C), g, DEV) * 2
    return y, coef, dout, perm[:, 1].reshape(B, Do, Ho, Wo, C)


def test_tie_collapse_routes_every_kernel_to_one_winner(monkeypatch):
    """scale +-2^-20, shift 1: distinct y with equal fp32 activations in every window.  keepmax's ymax, both backward
    reductions, both applies, conv1_bwd_fused's dW and conv1_dgrad_fused's dx must all use the backward kernels' winner
    (first maximum of sign(scale) * y).  bcoef = 0, so dy is scale * dz at the winner and 0 elsewhere."""
    shape = (1, 4, 6, 18)                  # W >= 17: the fused weight-gradient kernel takes it; W <= 128: so does dgrad
    B, D, H, W = shape
    g = gen(77)
    y, coef, dout, winner = collapse_operands(shape, g)
    assert torch.equal(N.route_index(y, coef[0])[..., 0], winner)
    C = 32
    y_b, coef32 = bf16(y), f32(coef.reshape(-1))
    assert torch.equal(y_b.double(), y)
    dout_b = bf16(dout)
    Do, Ho, Wo = D // 2, H // 2, W // 2
    # forward: every window's activations are equal in fp32 (the out value is the same whichever position wins)
    out, ym = guarded((B, Do, Ho, Wo, C), torch.bfloat16, 1), guarded((B, Do, Ho, Wo, C), torch.bfloat16, 1)
    got = run_twice(out + ym, lambda: L.call("tmf_bn_act_pool_fwd_keepmax", 1, L.ptrs([y_b]), L.ptrs([coef32]),
                                             L.ptrs(ts(out)), L.ptrs(ts(ym)), 0, B, D, H, W, C, 0.01))
    ywin = N.windows(y).gather(-1, winner.unsqueeze(-1))[..., 0]
    check(got[1], bf16(ywin), "keepmax ymax (the backward kernels' winner)")
    assert bool((got[0].float() == 1.0).all())
    ymax = [got[1].clone()]
    s1, s2, _, _ = N.sums_ref(y, coef, dout, N.POOL_MAX, 0.01)
    rows = guarded((L.stat_rows(), 2 * C), torch.float64, 1)
    got = run_twice(rows, lambda: L.call("tmf_bn_act_pool_bwd_reduce", 1, L.ptrs([dout_b]), 0, L.ptrs([y_b]),
                                         L.ptrs([coef32]), L.ptrs(ts(rows)), B, D, H, W, C, N.POOL_MAX, 0.01))
    check_rows(got[0], s1, s2, "generic reduction")
    got = run_twice(rows, lambda: L.call("tmf_bn_maxpool_bwd_reduce_kept", 1, L.ptrs([dout_b]), 0, L.ptrs(ymax),
                                         L.ptrs([coef32]), L.ptrs(ts(rows)), B, Do, Ho, Wo, C, 0.01))
    check_rows(got[0], s1, s2, "kept-maximum reduction")
    bcoef = [torch.zeros(2 * C, device=DEV)]
    dy_ref = N.apply_ref(y, coef, torch.zeros(2, C, dtype=torch.float64, device=DEV), dout, N.POOL_MAX, 0.01)
    assert int((dy_ref != 0).sum()) == int((dout != 0).sum())
    for generic in (False, True):
        if generic:
            monkeypatch.setenv("TMF_BN_GENERIC_MAXPOOL_BWD", "1")
        dy = guarded((B, D, H, W, C), torch.bfloat16, 1)
        got = run_twice(dy, lambda: L.call("tmf_bn_act_pool_bwd_apply", 1, L.ptrs([dout_b]), 0, L.ptrs([y_b]),
                                           L.ptrs([coef32]), L.ptrs(bcoef), L.ptrs(ts(dy)), B, D, H, W, C, N.POOL_MAX,
                                           0.01))
        check(got[0], X.bf16_rne(dy_ref), f"apply{' generic' if generic else ''}")
    monkeypatch.delenv("TMF_BN_GENERIC_MAXPOOL_BWD", raising=False)
    # block 1's fused backward kernels
    _, x = conv1_wgrad_operands(shape, 1, False, seed=78)
    x32 = [t.float() for t in x]
    nws = int(L.load().tmf_conv1_bwd_fused_workspace_bytes(1, B, D, H, W, C))
    assert nws > 0
    ws = workspace(nws)
    dw = guarded((C, 1, 3, 3, 3), torch.float32, 1)
    got = run_twice(dw, lambda: L.call("tmf_conv1_bwd_fused", 1, L.ptrs([dout_b]), L.ptrs([y_b]), L.ptrs([coef32]),
                                       L.ptrs(bcoef), L.ptrs(x32), L.ptrs(ts(dw)), B, D, H, W, C, 0.01, L.ptr(ws), nws))
    check(got[0].double(), X.wgrad_ref(dy_ref, x[0].unsqueeze(-1), 3), "conv1_bwd_fused dW")
    w = X.fixed((C, 1, 3, 3, 3), 13, 13, g, DEV)
    w32 = [w.float()]
    nws = int(L.load().tmf_conv1_dgrad_fused_workspace_bytes(1, L.CONV_UMMA, B, D, H, W, C))
    ws = workspace(nws)
    dx = guarded((B, D, H, W), torch.float32, 1)
    got = run_twice(dx, lambda: L.call("tmf_conv1_dgrad_fused", 1, L.ptrs([dout_b]), L.ptrs([y_b]), L.ptrs([coef32]),
                                       L.ptrs(bcoef), L.ptrs(w32), L.ptrs(ts(dx)), B, D, H, W, C, 0.01,
                                       L.CONV_UMMA, L.ptr(ws), nws))
    check(got[0].double(), X.dgrad_ref(dy_ref, w)[..., 0], "conv1_dgrad_fused dx")


def test_negative_slope_is_refused():
    """From Python (sNet._hyper) and through the C ABI on device buffers."""
    from transmf_ad_b200.models.networks import sNet
    net = sNet(32)
    net.conv3[2].negative_slope = -0.01
    with pytest.raises(NotImplementedError, match="slopes >= 0"):
        net._hyper()
    y = torch.zeros((1, 2, 2, 2, 8), dtype=torch.bfloat16, device=DEV)
    coef = torch.zeros(32, device=DEV)
    out = torch.empty((1, 1, 1, 1, 8), dtype=torch.bfloat16, device=DEV)
    ym = torch.empty_like(out)
    with pytest.raises(RuntimeError, match="slope >= 0"):
        L.call("tmf_bn_act_pool_fwd_keepmax", 1, L.ptrs([y]), L.ptrs([coef]), L.ptrs([out]), L.ptrs([ym]), 0, 1, 2, 2, 2,
               8, -0.01)


# ---------------------------------------------------------------------------------------------------------------
def test_forward_beyond_2_31_elements():
    """75 x 91 x 109 x 91 x 32 (2.17e9 elements, 4.3 GB of y; occlusion batches reach this range): keepmax with 64-bit
    offsets, reference computed sample by sample."""
    B, D, H, W, C = 75, 91, 109, 91, 32
    assert B * D * H * W * C > 2 ** 31
    g = gen(91)
    coef, centre = N.coefs(C, g, DEV)
    y = torch.empty((B, D, H, W, C), dtype=torch.bfloat16, device=DEV)
    for b in range(B):
        y[b] = bf16(N.y_values((D, H, W, C), centre, g, DEV))
    Do, Ho, Wo = D // 2, H // 2, W // 2
    out, ym = guarded((B, Do, Ho, Wo, C), torch.bfloat16, 1), guarded((B, Do, Ho, Wo, C), torch.bfloat16, 1)
    coef32 = [f32(coef.reshape(-1))]
    got = run_twice(out + ym, lambda: L.call("tmf_bn_act_pool_fwd_keepmax", 1, L.ptrs([y]), L.ptrs(coef32),
                                             L.ptrs(ts(out)), L.ptrs(ts(ym)), 0, B, D, H, W, C, N.SLOPE))
    for b0 in range(0, B, 5):
        o_ref, y_ref = N.fwd_ref(y[b0:b0 + 5].double(), coef, N.POOL_MAX, N.SLOPE)
        check(got[0][b0:b0 + 5], X.bf16_rne(o_ref), f"out, samples {b0}..")
        check(got[1][b0:b0 + 5], bf16(y_ref), f"ymax, samples {b0}..")


# ---------------------------------------------------------------------------------------------------------------
# Gaussian data, slope 0.01, coefficients from tmf_bn_finalize, against float64 torch autograd
@pytest.mark.parametrize("pool,shape,C", [(N.POOL_MAX, (8, 45, 54, 45), 32), (N.POOL_NONE, (8, 22, 27, 22), 64),
                                          (N.POOL_AVG, (8, 11, 13, 11), 128)])
def test_gaussian_chain_within_rounding_bound(pool, shape, C):
    B, D, H, W = shape
    g = gen(100 + pool)
    y = bf16(torch.randn((B, D, H, W, C), generator=g, device=DEV, dtype=torch.float64) * 1.5 + 0.4)
    y64 = y.double()
    gamma = (torch.randn(C, generator=g, device=DEV) * 0.5 + 1).float()
    gamma[::5] *= -1
    beta = (torch.randn(C, generator=g, device=DEV) * 0.3).float()
    count = B * D * H * W
    parts = torch.tensor_split(y64.reshape(-1, C), L.stat_rows())
    stats = torch.stack([torch.cat([p.sum(0), (p * p).sum(0)]) for p in parts]).contiguous()
    rm, rv = torch.zeros(C, device=DEV), torch.ones(C, device=DEV)
    nbt = torch.zeros(1, dtype=torch.int64, device=DEV)
    coef = torch.empty(4 * C, device=DEV)
    L.call("tmf_bn_finalize", 1, L.ptrs([stats]), L.ptrs([gamma]), L.ptrs([beta]), L.ptrs([rm]), L.ptrs([rv]),
           L.ptrs([nbt]), L.ptrs([coef]), C, count, 0.1, 1e-5, 1)
    last = pool == N.POOL_AVG
    pshape = (B, D, H, W, C) if pool == N.POOL_NONE else (B, D // 2, H // 2, W // 2, C)
    out = torch.empty(pshape, dtype=torch.float32 if last else torch.bfloat16, device=DEV)
    ymax = torch.empty(pshape, dtype=torch.bfloat16, device=DEV)
    if pool == N.POOL_MAX:
        L.call("tmf_bn_act_pool_fwd_keepmax", 1, L.ptrs([y]), L.ptrs([coef]), L.ptrs([out]), L.ptrs([ymax]), 0, B, D, H, W,
               C, 0.01)
    else:
        L.call("tmf_bn_act_pool_fwd", 1, L.ptrs([y]), L.ptrs([coef]), L.ptrs([out]), int(last), B, D, H, W, C, pool, 0.01)
    # float64 torch
    yr = y64.permute(0, 4, 1, 2, 3).clone().requires_grad_(True)
    gr, br = gamma.double().requires_grad_(True), beta.double().requires_grad_(True)
    z = F.batch_norm(yr, None, None, gr, br, True, 0.1, 1e-5)
    a = F.leaky_relu(z, 0.01)
    ref = F.max_pool3d(a, 2, 2) if pool == N.POOL_MAX else (F.avg_pool3d(a, 2, 2) if pool == N.POOL_AVG else a)
    ref_n = ref.detach().permute(0, 2, 3, 4, 1)
    # per element: z = fmaf(y, scale, shift) with scale / shift a few fp32 roundings off (finalize's bounds): 16 units of
    # |y*scale| + |shift| + |mean*scale| + |beta|, plus the output's bf16 rounding; a pool moves it by its window's bound
    mean = y64.reshape(-1, C).mean(0)
    inv = 1 / torch.sqrt(y64.reshape(-1, C).var(0, unbiased=False) + 1e-5)
    sc = gamma.double() * inv
    mag = (y64 * sc).abs() + (beta.double() - mean * sc).abs() + (mean * sc).abs() + beta.double().abs()
    if pool == N.POOL_MAX:
        mag = N.windows(mag).amax(-1)
    elif pool == N.POOL_AVG:
        mag = N.windows(mag).mean(-1)
    bound = (0 if last else 2.0 ** -8) * ref_n.abs() + 16 * U * mag
    assert bool(((out.double() - ref_n).abs() <= bound).all()), "forward"
    dout = torch.randn(pshape, generator=g, device=DEV, dtype=torch.float64)
    if not last:
        dout = bf16(dout).double()
    ref.backward(dout.permute(0, 4, 1, 2, 3))
    dout_k = dout.float().contiguous() if last else bf16(dout)
    sums = L.stat_buffers(1, C, DEV)[0]
    if pool == N.POOL_MAX:
        L.call("tmf_bn_maxpool_bwd_reduce_kept", 1, L.ptrs([dout_k]), int(last), L.ptrs([ymax]), L.ptrs([coef]),
               L.ptrs([sums]), B, D // 2, H // 2, W // 2, C, 0.01)
    else:
        L.call("tmf_bn_act_pool_bwd_reduce", 1, L.ptrs([dout_k]), int(last), L.ptrs([y]), L.ptrs([coef]), L.ptrs([sums]),
               B, D, H, W, C, pool, 0.01)
    dgamma, dbeta, dbias = (torch.empty(C, device=DEV) for _ in range(3))
    bcoef = torch.empty(2 * C, device=DEV)
    L.call("tmf_bn_bwd_finalize", 1, L.ptrs([sums]), L.ptrs([coef]), L.ptrs([dgamma]), L.ptrs([dbeta]), L.ptrs([dbias]),
           L.ptrs([bcoef]), C, count, 1)
    dy = torch.empty((B, D, H, W, C), dtype=torch.bfloat16, device=DEV)
    L.call("tmf_bn_act_pool_bwd_apply", 1, L.ptrs([dout_k]), int(last), L.ptrs([y]), L.ptrs([coef]), L.ptrs([bcoef]),
           L.ptrs([dy]), B, D, H, W, C, pool, 0.01)
    # parameter gradients: fp32 per-thread chains of up to `chain` terms (count / 256 positions per block row at worst)
    # over sum |dz| * (|xhat| + 1) -- the slack for xhat's own rounding from fp32 mean / invstd
    dz = N.dz_ref(y64, torch.stack([sc, beta.double() - mean * sc, mean, inv]), dout, pool, 0.01).reshape(-1, C)
    xh = ((y64 - mean) * inv).reshape(-1, C)
    chain = count // 256 + 64
    abs_s2 = (dz.abs() * (xh.abs() + 1)).sum(0)
    assert bool(((dgamma.double() - gr.grad).abs() <= chain * U * abs_s2 + 1e-6 * gr.grad.abs()).all()), "dgamma"
    assert bool(((dbeta.double() - br.grad).abs() <= chain * U * dz.abs().sum(0) + 1e-6 * br.grad.abs()).all()), "dbeta"
    # dy = scale (dz - m1 - xhat m2): bf16 rounding + m1 / m2 carry the sums' errors (/ count) + a few fp32 roundings
    m1e = (chain * U * dz.abs().sum(0) + 1e-6 * br.grad.abs()) / count + U * (br.grad / count).abs()
    m2e = (chain * U * abs_s2 + 1e-6 * gr.grad.abs()) / count + U * (gr.grad / count).abs()
    yg = yr.grad.permute(0, 2, 3, 4, 1)
    xh = (y64 - mean) * inv
    m2 = (gr.grad / count)
    dzf = N.dz_ref(y64, torch.stack([sc, beta.double() - mean * sc, mean, inv]), dout, pool, 0.01)
    dmag = sc.abs() * (dzf.abs() + (br.grad / count).abs() + (xh.abs() + 1) * m2.abs())
    bound = 2.0 ** -8 * yg.abs() + 16 * U * dmag + sc.abs() * (m1e + (xh.abs() + 1) * m2e)
    assert bool(((dy.double() - yg).abs() <= bound).all()), "dy"

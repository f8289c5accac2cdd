"""Exact-arithmetic tests of the fusion-transformer kernels: the fused encoder (enc_fused.cu), Linear / LayerNorm / token
pooling (fusion_ops.cu) and the attention core (attention_mma.cu, attention.cu, fusion_ops.cu).

Operands live on short dyadic grids chosen so that every kernel path is exact (tests/fusion_exact.py): a correct kernel
reproduces the float64 reference bit for bit, and a dropped partial, a missing cross term, an unwritten row of a ragged
panel or a leaking padding key fails on the element it touches.  Every output and saved intermediate is poisoned with
NaN bytes inside guard bands before each call, the scratch buffer's partial area is poisoned too (no kernel may read stale
partials), every call runs twice and must give the same bits, and the 16 KB ticket area must be zero after every call.
torch.profiler confirms once per case that the case reaches the kernel it names."""
import ctypes
import zlib

import pytest
import torch

from tests import conv_exact as X
from tests import fusion_exact as E
from transmf_ad_b200 import _lib as L

pytestmark = pytest.mark.gpu
DEV = "cuda"
TICKET_BYTES = 16384


def gen(tag):
    return torch.Generator(device=DEV).manual_seed(zlib.crc32(tag.encode()))


def dev32(t):
    return t.float().contiguous()


class Scratch:
    """The zero-initialised scratch buffer of include/tmf.h with its partial area poisoned before every call."""

    def __init__(self):
        self.buf = torch.zeros(int(L.load().tmf_scratch_bytes()), dtype=torch.uint8, device=DEV)

    def poison(self):
        self.buf[TICKET_BYTES:].fill_(0xFF)

    def check_tickets(self, what):
        assert int(self.buf[:TICKET_BYTES].count_nonzero()) == 0, f"{what}: ticket area not left zero"

    def args(self):
        return L.ptr(self.buf), self.buf.numel()


def run_twice(outs, launch, ws=None, init=None):
    """Poison every output (then apply `init`, for accumulating calls), launch, check guard bands and tickets; repeat and
    demand the same bits."""
    snaps = []
    for _ in range(2):
        for o in outs:
            o.poison()
        if init is not None:
            init()
        if ws is not None:
            ws.poison()
        launch()
        torch.cuda.synchronize()
        for i, o in enumerate(outs):
            o.check_bands(f"output {i}")
        if ws is not None:
            ws.check_tickets("scratch")
        snaps.append([o.t.clone() for o in outs])
    for i, (a, b) in enumerate(zip(*snaps)):
        assert torch.equal(a.view(torch.uint8), b.view(torch.uint8)), f"output {i}: two calls gave different bits"
    return snaps[0]


def kernels(launch):
    """Names of the CUDA kernels one call launches."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        launch()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


def expect_kernel(launch, name):
    names = kernels(launch)
    assert any(name in n for n in names), f"expected a launch of {name}, got {names}"


def G(shape, dtype=torch.float32):
    return X.Guarded(shape, dtype, DEV)


def check(got, ref, what):
    err = X.mismatch(got, E.f32(ref))
    assert not err, f"{what}: {err}"


# ---------------------------------------------------------------------------------------------------------------
# the arithmetic the exact cases rely on (settled on sm_100a by these asserts)
def test_device_arithmetic_assumptions():
    """mma.sync bf16 m16n8k16 / tf32 m16n8k8 accumulate grid-bounded sums exactly (a 16-row encoder panel with products up
    to 2^23 quanta), rsqrtf(4^k) == 2^-k, __expf(0) == 1 and __logf(1) == 0 (one-hot attention: lse = max, P = 1)."""
    g = gen("assumptions")
    M = 16
    # proj_fwd's ctx GEMM: kv = ctx Wkv^T with 128-term sums of large grid products, bf16x3 and 3xTF32
    ctx = E.ints((M, 128), -32767, 32767, g, DEV)
    wkv = E.pow2((256, 128), 0, 0, g, DEV)
    for path, pk in (("bf16", True), ("tf32", False)):
        E.check_path(ctx, wkv, path)
        pack = torch.empty(int(L.load().tmf_encoder_pack_bytes(128)) // 2, dtype=torch.bfloat16, device=DEV)
        w = [torch.zeros(128, 128, device=DEV), dev32(wkv), torch.zeros(128, 128, device=DEV),
             torch.zeros(128, 128, device=DEV), torch.zeros(128, 128, device=DEV)]
        L.call("tmf_encoder_pack_weights", *[L.ptr(t) for t in w], 128, L.ptr(pack))
        x = dev32(E.ln_rows(M, 128, g, DEV)[0])
        o = {k: torch.empty(s, device=DEV) for k, s in (("h1", (M, 128)), ("m", (M,)), ("r", (M,)), ("q", (M, 128)),
                                                           ("kv", (M, 256)))}
        c32, one, zero = dev32(ctx), torch.ones(128, device=DEV), torch.zeros(128, device=DEV)
        L.call("tmf_encoder_proj_fwd", L.ptr(x), L.ptr(c32), L.ptr(one), L.ptr(zero), L.ptr(w[0]), L.ptr(w[1]),
               *[L.ptr(t) for t in o.values()], M, M, 0.0,
               L.ptr(pack if pk else None))
        torch.cuda.synchronize()
        check(o["kv"], ctx @ wkv.T, f"mma.sync {path} accumulation")
    # rsqrtf of exact powers of four: LayerNorm rows with variance 4 s^2 for s = 2^-8 .. 2^8
    rows = 17
    p = E.ln_pattern(rows, 128, g, DEV)
    s = torch.ldexp(torch.ones(rows, 1, device=DEV, dtype=torch.float64), torch.arange(-8, 9, device=DEV)[:, None])
    xs = dev32(p * s)
    y, mean, rstd = torch.empty_like(xs), torch.empty(rows, device=DEV), torch.empty(rows, device=DEV)
    one, zero = torch.ones(128, device=DEV), torch.zeros(128, device=DEV)
    L.call("tmf_layernorm_fwd", L.ptr(xs), L.ptr(one), L.ptr(zero),
           L.ptr(None), L.ptr(y), L.ptr(mean), L.ptr(rstd), rows, 128, 0.0)
    torch.cuda.synchronize()
    check(rstd, 0.5 / s.squeeze(1), "rsqrtf(4^k)")
    # __expf(0) == 1, __logf(1) == 0: one query, one key, score 0 -> lse 0, out = v, P = 1
    q = torch.zeros(1, 1, 32, device=DEV)
    kv = torch.cat([torch.zeros(1, 1, 32, device=DEV), torch.arange(32, device=DEV, dtype=torch.float32).view(1, 1, 32)], -1)
    out, lse = torch.empty(1, 1, 32, device=DEV), torch.empty(1, 1, 1, device=DEV)
    L.call("tmf_attn_fwd", L.ptr(q), L.ptr(kv), L.ptr(out), L.ptr(lse), 1, 1, 1, 1, 32, 1.0)
    sc, pr = torch.empty(1, 1, 1, 1, device=DEV), torch.empty(1, 1, 1, 1, device=DEV)
    L.call("tmf_attn_scores", 0, L.ptr(q), L.ptr(kv), L.ptr(lse), L.ptr(sc), L.ptr(pr), 1, 1, 1, 1, 32, 1.0)
    torch.cuda.synchronize()
    assert float(lse) == 0.0 and float(pr) == 1.0 and torch.equal(out, kv[..., 32:]), (float(lse), float(pr))


# ---------------------------------------------------------------------------------------------------------------
# Linear: tmf_linear_fwd / _dgrad / _wgrad
B8 = 8 * 150
LINEAR_CASES = [  # (id, M, K, N, act, residual)
    ("attn-out", B8, 128, 128, 0, True), ("to-kv-300", 2 * B8, 128, 256, 0, False), ("mlp-in", B8, 128, 512, 1, False),
    ("mlp-out", B8, 512, 128, 0, True),
    ("head-256-512", 8, 256, 512, 0, False), ("head-512-64", 8, 512, 64, 1, False), ("head-64-2", 8, 64, 2, 0, False),
    ("head-128-2", 8, 128, 2, 0, True), ("head-256-128", 8, 256, 128, 1, True),
    # generic kernel: K % 4 != 0 (no split / its 64-token split in wgrad)
    ("ragged-k", 77, 30, 20, 1, True), ("ragged-split", 1000, 130, 36, 0, False),
    # wgrad too large for the scratch buffer (generic 64-token split of 250 chunks x 130 x 130): kchunk = 0
    ("scratch-fallback", 16000, 130, 130, 0, False),
]


def gemm_path(sAm, sAk, sBk, sBn, M, N, K):
    """The kernel launch_gemm (csrc/fusion_ops.cu) picks for 16-byte aligned operands."""
    akf, bkf = sAk == 1, sBk == 1
    lda, ldb = (sAm if akf else sAk), (sBn if bkf else sBk)
    ok = (akf or sAm == 1) and (bkf or sBn == 1) and lda % 4 == 0 and ldb % 4 == 0 and not ((akf or bkf) and K % 4) \
        and not (not akf and M % 4) and not (not bkf and N % 4)
    return f"gemm_ksplit_kernel<{str(akf).lower()}, {str(bkf).lower()}>" if ok else "gemm_kernel"


WS_PART_FLOATS = ((16 << 20) - TICKET_BYTES) // 4     # the scratch buffer's partial area (csrc/common.cuh TMF_WS_BYTES)


def wgrad_split(M, K, N):
    """How tmf_linear_wgrad (csrc/fusion_ops.cu) splits the token reduction: 'none' (M <= 128), 'sized' (gemm_ksplit_kernel,
    whole super-slices), 'generic-64' (gemm_kernel, 64 tokens per split) or 'fallback' (too large for the scratch buffer:
    one CTA per tile walks all tokens)."""
    if M <= 128:
        return "none"
    ks = linear_kernels(M, K, N)[2] != "gemm_kernel"
    if ks:
        tiles = -(-N // 32) * -(-K // 32)
        splits = min(-(-296 // tiles), -(-M // 128))
        kchunk = -(-(-(-M // splits)) // 128) * 128
    else:
        tiles, kchunk = -(-N // 64) * -(-K // 64), 64
    splits = -(-M // kchunk)
    if tiles > 2048 or splits * N * K > WS_PART_FLOATS:
        return "fallback"
    return "sized" if ks else "generic-64"


def linear_kernels(M, K, N):
    """(forward, dgrad, wgrad) kernels of one Linear."""
    return (gemm_path(K, 1, 1, K, M, N, K), gemm_path(N, 1, K, 1, M, K, N), gemm_path(1, N, K, 1, N, K, M))


def test_linear_cases_cover_every_wgrad_split():
    seen = {wgrad_split(*c[1:4]) for c in LINEAR_CASES}
    assert seen == {"none", "sized", "generic-64", "fallback"}, seen
    assert wgrad_split(16000, 130, 130) == "fallback" and wgrad_split(1000, 130, 36) == "generic-64"


def test_linear_cases_cover_every_gemm_kernel():
    seen = {k for c in LINEAR_CASES for k in linear_kernels(*c[1:4])}
    assert seen == {"gemm_kernel", "gemm_ksplit_kernel<true, true>", "gemm_ksplit_kernel<true, false>",
                    "gemm_ksplit_kernel<false, false>"}, seen


def linear_operands(M, K, N, act, g):
    x = E.ints((M, K), -3, 3, g, DEV, 0.25)
    w = E.ints((N, K), -3, 3, g, DEV, 0.125)
    bias = (E.ints((N,), 0, 1, g, DEV) * 64 - 32) if act else E.ints((N,), -8, 8, g, DEV, 2.0 ** -5)
    if act:                       # saturated GELU: |x . w| < 8 next to b = +-32
        w = w * (E.ints((N, K), 0, 15, g, DEV) == 0)
        assert float((x.abs() @ w.abs().T).max()) < 8
    return x, w, bias


@pytest.mark.parametrize("case", LINEAR_CASES, ids=[c[0] for c in LINEAR_CASES])
def test_linear_exact(case):
    cid, M, K, N, act, res = case
    kf, kd, kw = linear_kernels(M, K, N)
    g = gen(cid)
    x, w, bias = linear_operands(M, K, N, act, g)
    r = E.ints((M, N), -8, 8, g, DEV, 0.5) if res else None
    dy = E.ints((M, N), -3, 3, g, DEV, 0.25)
    dx0 = E.ints((M, K), -8, 8, g, DEV, 2.0 ** -4)
    E.check_path(x, w, "fma", (bias,))
    E.check_path(dy, w.T, "fma", (dx0,))
    E.check_path(dy.T, x.T, "fma")
    E.sum_quanta(dy, 0)
    xs, ws_, bs, rs, dys = dev32(x), dev32(w), dev32(bias), dev32(r) if res else None, dev32(dy)
    y_ref, pre_ref = E.linear_ref(x, w, bias, r, act)

    # forward (bias, pre, GELU and residual epilogues)
    y, pre = G((M, N)), G((M, N))
    fwd = lambda: L.call("tmf_linear_fwd", L.ptr(xs), L.ptr(ws_), L.ptr(bs), L.ptr(rs), L.ptr(y.t), L.ptr(pre.t), M, K, N, act)
    gy, gpre = run_twice([y, pre], fwd)
    check(gy, y_ref, f"{cid} y")
    check(gpre, pre_ref, f"{cid} pre")
    expect_kernel(fwd, kf)

    # dgrad, overwrite and accumulate
    dx = G((M, K))
    for acc in (0, 1):
        dgr = lambda: L.call("tmf_linear_dgrad", L.ptr(dys), L.ptr(ws_), L.ptr(dx.t), M, K, N, acc)
        init = (lambda: dx.t.copy_(dx0)) if acc else None
        (gdx,) = run_twice([dx], dgr, init=init)
        check(gdx, dy @ w + (dx0 if acc else 0), f"{cid} dgrad accumulate={acc}")
    expect_kernel(dgr, kd)

    # wgrad (+ bias column sums)
    ws = Scratch()
    dw, db = G((N, K)), G((N,))
    wgr = lambda: L.call("tmf_linear_wgrad", L.ptr(dys), L.ptr(xs), L.ptr(dw.t), L.ptr(db.t), M, K, N, *ws.args())
    gdw, gdb = run_twice([dw, db], wgr, ws=ws)
    check(gdw, dy.T @ x, f"{cid} dw")
    check(gdb, dy.sum(0), f"{cid} dbias")
    names = kernels(wgr)
    assert any(kw in n for n in names) and any("colsum_kernel" in n for n in names), names


def test_linear_misaligned_operands_take_generic_kernel():
    """A weight that is not 16-byte aligned sends the forward to gemm_kernel."""
    g = gen("misaligned")
    M, K, N = 150, 128, 128
    x, w, bias = linear_operands(M, K, N, 0, g)
    wbuf = torch.empty(N * K + 1, device=DEV)
    wbuf[1:].copy_(w.flatten())
    wm = wbuf[1:]
    xs, bs = dev32(x), dev32(bias)
    y = G((M, N))
    fwd = lambda: L.call("tmf_linear_fwd", L.ptr(xs), L.ptr(wm), L.ptr(bs), L.ptr(None), L.ptr(y.t), L.ptr(None),
                         M, K, N, 0)
    (gy,) = run_twice([y], fwd)
    check(gy, x @ w.T + bias, "misaligned y")
    expect_kernel(fwd, "gemm_kernel")


def test_linear_wgrad_column_sums_refuse_the_encoder_tickets():
    """The bias column sums stop below the encoder's ticket words (N <= 32 * 828)."""
    ws = Scratch()
    N = 32 * 828 + 1
    t = torch.zeros(4, N, device=DEV)
    dw = torch.empty(N, 1, device=DEV)
    with pytest.raises(RuntimeError, match="column-sum tickets"):
        L.call("tmf_linear_wgrad", L.ptr(t), L.ptr(t), L.ptr(dw), L.ptr(t), 4, 1, N, *ws.args())


# ---------------------------------------------------------------------------------------------------------------
# LayerNorm
LN_CASES = [  # (id, rows, dim, residual)
    ("model-300", 300, 128, True), ("model-b8", B8, 128, False), ("dim-64", 37, 64, False), ("dim-512", 33, 512, True),
    ("dim-1024", 19, 1024, False), ("dim-160", 45, 160, True), ("dim-96", 13, 96, False),
    ("grid-stride", 148 * 8 * 8 + 37, 128, False), ("one-row", 1, 128, True)]


@pytest.mark.parametrize("case", LN_CASES, ids=[c[0] for c in LN_CASES])
def test_layernorm_exact(case):
    cid, rows, dim, res = case
    g = gen(cid)
    x, m, rstd, p = E.ln_rows(rows, dim, g, DEV)
    gamma, beta = E.ints((dim,), -7, 7, g, DEV, 0.25), E.ints((dim,), -8, 8, g, DEV, 0.125)
    r = E.ints((rows, dim), -8, 8, g, DEV, 0.25) if res else None
    y_ref, mean_ref, rstd_ref = E.layernorm_ref(x, gamma, beta, 0.0, r)
    assert torch.equal(mean_ref, m) and torch.equal(rstd_ref, rstd)
    xs, gs, bs, rs32 = dev32(x), dev32(gamma), dev32(beta), dev32(r) if res else None
    y, mean, rs = G((rows, dim)), G((rows,)), G((rows,))
    fwd = lambda: L.call("tmf_layernorm_fwd", L.ptr(xs), L.ptr(gs), L.ptr(bs), L.ptr(rs32),
                         L.ptr(y.t), L.ptr(mean.t), L.ptr(rs.t), rows, dim, 0.0)
    gy, gm, gr = run_twice([y, mean, rs], fwd)
    check(gm, m, f"{cid} mean")
    check(gr, rstd, f"{cid} rstd")
    check(gy, y_ref, f"{cid} y")
    expect_kernel(fwd, "layernorm_fwd_kernel")

    # backward at the same statistics: random dy where dim is a power of two (the row means divide exactly), row-balanced dy
    # (zero row means) otherwise
    if dim & (dim - 1) == 0:
        dy = E.ints((rows, dim), -3, 3, g, DEV, 0.5)
    else:
        gamma = E.pow2((dim,), -1, 1, g, DEV)
        p = E.ln_pattern(rows, dim, g, DEV, shared=True)
        x = m[:, None] + p / (2 * rstd[:, None])
        dy = E.paired_dy(rows, p[0], gamma, g, DEV)
    dx0 = E.ints((rows, dim), -8, 8, g, DEV, 2.0 ** -3)
    dx_ref, dg_ref, db_ref = E.layernorm_bwd_ref(dy, x, gamma, m, rstd)
    E.sum_quanta(dy * (x - m[:, None]) * rstd[:, None], 0)
    ws = Scratch()
    dx, dgam, dbet = G((rows, dim)), G((dim,)), G((dim,))
    xs, dys, gs, ms, rss = dev32(x), dev32(dy), dev32(gamma), dev32(m), dev32(rstd)
    for acc in (0, 1):
        bwd = lambda: L.call("tmf_layernorm_bwd", L.ptr(dys), L.ptr(xs), L.ptr(gs), L.ptr(ms), L.ptr(rss),
                             L.ptr(dx.t), L.ptr(dgam.t), L.ptr(dbet.t), rows, dim, acc, *ws.args())
        gdx, gdg, gdb = run_twice([dx, dgam, dbet], bwd, ws=ws, init=(lambda: dx.t.copy_(dx0)) if acc else None)
        check(gdx, dx_ref + (dx0 if acc else 0), f"{cid} dx accumulate={acc}")
        check(gdg, dg_ref, f"{cid} dgamma")
        check(gdb, db_ref, f"{cid} dbeta")
    expect_kernel(bwd, "layernorm_bwd_kernel")


# ---------------------------------------------------------------------------------------------------------------
# attention core: one-hot softmax
ATTN_CASES = [  # (id, B, Nq, Nk, heads, dh)
    ("model", 8, 150, 150, 4, 32), ("dh16", 2, 150, 150, 8, 16), ("dh64", 2, 150, 150, 2, 64),
    ("ragged", 3, 37, 29, 4, 32), ("ragged-nq-gt-nk", 2, 160, 97, 4, 32), ("one-key", 2, 5, 1, 4, 16),
    ("ctx-300", 2, 300, 300, 4, 32), ("long-400", 1, 400, 333, 2, 32)]

IMPL_KERNELS = {"2": "attn_mma_fwd_kernel", "1": "attn_tiled_fwd_kernel", "0": "attn_fwd_kernel"}


def attn_kernel_names(Nq, Nk, dh, impl):
    """(forward, backward) kernels tmf_attn_fwd / tmf_attn_bwd reach (csrc/attention_mma.cu, attention.cu, fusion_ops.cu)."""
    mma = impl == "2" and dh in (16, 32, 64)
    tiled = impl != "0"
    fwd = "attn_mma_fwd_kernel" if mma and Nk <= 160 else "attn_tiled_fwd_kernel" if tiled and Nk <= 320 else "attn_fwd_kernel"
    bwd = "attn_mma_bwd_kernel" if mma and max(Nq, Nk) <= 160 else \
        "attn_tiled_dkv_kernel" if tiled and max(Nq, Nk) <= 320 else "attn_bwd_dkv_kernel"
    return fwd, bwd


def attention_operands(cid, B, Nq, Nk, heads, dh):
    """(q, kv, win, dout, scale) of one one-hot case; asserts the bf16x3 exactness of both products."""
    g = gen(cid)
    scale = 0.5
    q, kv, win = E.one_hot_attention(B, Nq, Nk, heads, dh, g, DEV, scale)
    inner = heads * dh
    dout = E.ints((B, Nq, inner), -4, 4, g, DEV, 0.5)
    E.check_path(q.view(-1, dh), kv[..., :inner].reshape(-1, dh), "bf16")
    E.check_path(dout.view(-1, dh), kv[..., inner:].reshape(-1, dh), "bf16")
    return q, kv, win, dout, scale


@pytest.mark.parametrize("case", ATTN_CASES, ids=[c[0] for c in ATTN_CASES])
@pytest.mark.parametrize("impl", ["2", "1", "0"])
def test_attention_one_hot_exact(case, impl):
    """out = the winner's v row, lse = the winner's scaled score, dq = dk = 0, dv = sum of dO over the queries that picked
    each key (every key, those of the last partial tile included, is picked).  TMF_ATTN_IMPL is read once per process:
    run with TMF_ATTN_IMPL=1 / 0 for those variants."""
    if L.load().tmf_attn_impl_default() != int(impl):
        pytest.skip("TMF_ATTN_IMPL is read once per process: run with TMF_ATTN_IMPL=%s for this variant" % impl)
    cid, B, Nq, Nk, heads, dh = case
    q, kv, win, dout, scale = attention_operands(*case)
    inner = heads * dh
    kf, kb = attn_kernel_names(Nq, Nk, dh, impl)
    out_ref, lse_ref, dots_ref, attn_ref = E.attention_ref(q, kv, heads, dh, scale)
    dq_ref, dkv_ref, dattn_ref = E.attention_bwd_ref(dout, q, kv, heads, dh, scale)
    assert bool((attn_ref.argmax(-1) == win).all())
    qs, kvs, dos = dev32(q), dev32(kv), dev32(dout)
    out, lse = G((B, Nq, inner)), G((B, heads, Nq))
    fwd = lambda: L.call("tmf_attn_fwd", L.ptr(qs), L.ptr(kvs), L.ptr(out.t), L.ptr(lse.t), B, Nq, Nk, heads, dh, scale)
    gout, glse = run_twice([out, lse], fwd)
    check(gout, out_ref, f"{cid} out")
    check(glse, lse_ref, f"{cid} lse")
    expect_kernel(fwd, kf)
    dq, dkv = G((B, Nq, inner)), G((B, Nk, 2 * inner))
    bwd = lambda: L.call("tmf_attn_bwd", L.ptr(dos), L.ptr(qs), L.ptr(kvs), L.ptr(gout), L.ptr(glse), L.ptr(dq.t), L.ptr(dkv.t),
                         B, Nq, Nk, heads, dh, scale)
    gdq, gdkv = run_twice([dq, dkv], bwd)
    check(gdq, dq_ref, f"{cid} dq")
    check(gdkv, dkv_ref, f"{cid} dkv")
    expect_kernel(bwd, kb)
    print(f"[attn impl {impl}] {cid}: {kf} / {kb}, exact")
    if impl == "2" and dh in (16, 32, 64):
        # attention maps: dots / attn (mode 0) and dattn (mode 1) are plain products of the same operands
        s, p = G((B, heads, Nq, Nk)), G((B, heads, Nq, Nk))
        gs, gp = run_twice([s, p], lambda: L.call("tmf_attn_scores", 0, L.ptr(qs), L.ptr(kvs), L.ptr(glse), L.ptr(s.t),
                                                   L.ptr(p.t), B, Nq, Nk, heads, dh, scale))
        check(gs, dots_ref, f"{cid} dots")
        check(gp, attn_ref, f"{cid} attn")
        (gda,) = run_twice([s], lambda: L.call("tmf_attn_scores", 1, L.ptr(dos), L.ptr(kvs), L.ptr(None), L.ptr(s.t),
                                                L.ptr(None), B, Nq, Nk, heads, dh, scale))
        check(gda, dattn_ref, f"{cid} dattn")


# ---------------------------------------------------------------------------------------------------------------
# token pooling
@pytest.mark.parametrize("B,N,C", [(8, 150, 128), (3, 150, 256), (2, 7, 40), (1, 1, 8)])
def test_token_pool_exact(B, N, C):
    """Ties in the max go to the first maximum; mean = fp32(sum) / N; the backward in fp32 as the kernel orders it."""
    g = gen(f"pool{B}-{N}-{C}")
    x = E.ints((B, N, C), -3, 3, g, DEV, 0.5)
    s_ref, mx_ref, am_ref = E.token_pool_ref(x)
    xs = dev32(x)
    mean, mx, am = G((B, C)), G((B, C)), G((B, C), torch.int32)
    fwd = lambda: L.call("tmf_token_pool_fwd", L.ptr(xs), L.ptr(mean.t), L.ptr(mx.t), L.ptr(am.t), B, N, C)
    gmean, gmx, gam = run_twice([mean, mx, am], fwd)
    check(gmean, (E.f32(s_ref) / torch.tensor(float(N), device=DEV)).double(), "mean")
    check(gmx, mx_ref, "max")
    assert torch.equal(gam.long(), am_ref), X.mismatch(gam.long(), am_ref)
    expect_kernel(fwd, "token_pool_fwd_kernel")
    dmean, dmax = dev32(E.ints((B, C), -8, 8, g, DEV, 0.25)), dev32(E.ints((B, C), -8, 8, g, DEV, 0.25))
    dx0 = dev32(E.ints((B, N, C), -8, 8, g, DEV, 0.125))
    invn = torch.tensor(1.0, device=DEV) / N
    hit = torch.arange(N, device=DEV)[None, :, None] == gam.long()[:, None, :]
    want = dmean[:, None, :] * invn + torch.where(hit, dmax[:, None, :], torch.zeros((), device=DEV))
    dx = G((B, N, C))
    for acc in (0, 1):
        bwd = lambda: L.call("tmf_token_pool_bwd", L.ptr(dmean), L.ptr(dmax), L.ptr(gam), L.ptr(dx.t), B, N, C, acc)
        (gdx,) = run_twice([dx], bwd, init=(lambda: dx.t.copy_(dx0)) if acc else None)
        assert torch.equal(gdx, want + dx0 if acc else want), X.mismatch(gdx, want + dx0 if acc else want)
    expect_kernel(bwd, "token_pool_bwd_kernel")


# ---------------------------------------------------------------------------------------------------------------
# fused encoder
def pack_of(w, mlp):
    pk = torch.empty(int(L.load().tmf_encoder_pack_bytes(mlp)) // 2, dtype=torch.bfloat16, device=DEV)
    L.call("tmf_encoder_pack_weights", *[L.ptr(t) for t in w], mlp, L.ptr(pk))
    return pk


@pytest.mark.parametrize("mlp", [128, 256, 512])
def test_encoder_pack_weights(mlp):
    """hi = bf16(w), lo = bf16(w - hi) for every matrix; on bf16-representable weights lo is all zero."""
    g = gen(f"pack{mlp}")
    shapes = [(128, 128), (256, 128), (128, 128), (mlp, 128), (128, mlp)]
    for kind in ("fp32", "bf16"):
        w = [torch.randn(s, generator=g, device=DEV) for s in shapes]
        if kind == "bf16":
            w = [t.bfloat16().float() for t in w]
        pk = pack_of(w, mlp)
        torch.cuda.synchronize()
        off = 0
        for t in w:
            n = t.numel()
            hi, lo = pk[off:off + n].view(t.shape), pk[off + n:off + 2 * n].view(t.shape)
            want_hi = t.bfloat16()
            assert torch.equal(hi.view(torch.int16), want_hi.view(torch.int16)), f"{kind} hi"
            want_lo = (t - want_hi.float()).bfloat16()
            assert torch.equal(lo.view(torch.int16), want_lo.view(torch.int16)), f"{kind} lo"
            if kind == "bf16":
                assert int(lo.float().count_nonzero()) == 0
            off += 2 * n
        assert off == pk.numel()


PROJ_CASES = [("model", B8, B8), ("ctx-300", B8, 2 * B8), ("x-gt-ctx", 300, 150), ("ragged", 37, 29), ("m1", 1, 1)]


def proj_operands(cid, Mx, Mc):
    """Forward and backward inputs of one projection case with their references; asserts the bf16x3 condition of all four
    GEMMs (it implies the 3xTF32 one) and the 2^24 bound of the LayerNorm parameter sums."""
    g = gen("proj" + cid)
    x, m1, r1, _ = E.ln_rows(Mx, 128, g, DEV)
    ctx = E.ints((Mc, 128), -32, 32, g, DEV, 0.125)
    ln_w, ln_b = E.ints((128,), -7, 7, g, DEV, 0.25), E.ints((128,), -4, 4, g, DEV, 0.125)
    wq = E.sparse_dyadic(128, 128, 3, -2, 0, g, DEV)
    wkv = E.sparse_dyadic(256, 128, 3, -2, 0, g, DEV)
    ref = E.proj_fwd_ref(x, ctx, ln_w, ln_b, wq, wkv)
    dq = E.ints((Mx, 128), -3, 3, g, DEV, 0.25)
    dkv = E.ints((Mc, 256), -3, 3, g, DEV, 0.25)
    dxp = E.ints((Mx, 128), -8, 8, g, DEV, 2.0 ** -4)
    bref = E.proj_bwd_ref(dq, dkv, dxp, x, ln_w, m1, r1, wq, wkv)
    E.check_path(ref["h1"], wq, "bf16")
    E.check_path(ctx, wkv, "bf16")
    E.check_path(dq, wq.T, "bf16")
    E.check_path(dkv, wkv.T, "bf16")
    E.sum_quanta(bref["dh1"] * (x - m1[:, None]) * r1[:, None], 0)
    E.sum_quanta(bref["dh1"], 0)
    return dict(x=x, m1=m1, r1=r1, ctx=ctx, ln_w=ln_w, ln_b=ln_b, wq=wq, wkv=wkv, dq=dq, dkv=dkv, dxp=dxp), ref, bref


@pytest.mark.parametrize("bf16", [True, False], ids=["pack", "tf32"])
@pytest.mark.parametrize("case", PROJ_CASES, ids=[c[0] for c in PROJ_CASES])
def test_encoder_proj_fwd_bwd_exact(case, bf16):
    """The LN1 backward runs on random dq, so its row means mean(dh1 gamma) and mean(dh1 gamma xhat) are nonzero: the
    correction terms of panel_layernorm_bwd, which the chain backward shares, are checked bit for bit here."""
    cid, Mx, Mc = case
    path = "bf16" if bf16 else "tf32"
    o, ref, bref = proj_operands(*case)
    x, m1, r1, ctx, ln_w, ln_b, wq, wkv, dq, dkv, dxp = (o[k] for k in ("x", "m1", "r1", "ctx", "ln_w", "ln_b", "wq", "wkv",
                                                                        "dq", "dkv", "dxp"))
    w5 = [dev32(wq), dev32(wkv)] + [torch.zeros(s, device=DEV) for s in ((128, 128), (128, 128), (128, 128))]
    pk = pack_of(w5, 128) if bf16 else None
    xs, cs, lws, lbs = dev32(x), dev32(ctx), dev32(ln_w), dev32(ln_b)
    outs = [G((Mx, 128)), G((Mx,)), G((Mx,)), G((Mx, 128)), G((Mc, 256))]
    fwd = lambda: L.call("tmf_encoder_proj_fwd", L.ptr(xs), L.ptr(cs), L.ptr(lws), L.ptr(lbs), L.ptr(w5[0]),
                         L.ptr(w5[1]), *[L.ptr(o.t) for o in outs], Mx, Mc, 0.0, L.ptr(pk))
    got = run_twice(outs, fwd)
    for name, t in zip(("h1", "mean1", "rstd1", "q", "kv"), got):
        check(t, ref[name], f"{cid} {path} {name}")
    expect_kernel(fwd, "enc_proj_fwd_kernel")

    # backward: dx = dxp + LN1'(dq Wq), dctx = dkv Wkv, LN1 parameter gradients
    gg = bref["dh1"] * ln_w
    assert float(gg.mean(1).abs().max()) > 0 and float((gg * (x - m1[:, None]) * r1[:, None]).mean(1).abs().max()) > 0
    ws = Scratch()
    bouts = [G((Mx, 128)), G((Mc, 128)), G((128,)), G((128,))]
    bin_ = [dev32(t) for t in (dq, dkv, dxp, x, ln_w, m1, r1)]      # held for the lambda: ptr() does not keep a tensor alive
    bwd = lambda: L.call("tmf_encoder_proj_bwd", *[L.ptr(t) for t in bin_], L.ptr(w5[0]), L.ptr(w5[1]),
                         *[L.ptr(o.t) for o in bouts], Mx, Mc, L.ptr(pk), *ws.args())
    got = run_twice(bouts, bwd, ws=ws)
    for name, t in zip(("dx", "dctx", "dln_w", "dln_b"), got):
        check(t, bref[name], f"{cid} {path} {name}")
    expect_kernel(bwd, "enc_proj_bwd_kernel")


CHAIN_CASES = [  # (id, M, mlp, add_input)
    ("model", B8, 512, 1), ("mlp128", 300, 128, 0), ("mlp256", 150, 256, 1), ("ragged", 37, 512, 0), ("m1", 1, 256, 1)]
CHAIN_FWD_OUT = ("a", "h2", "mean2", "rstd2", "pre", "f", "g", "meanf", "rstdf", "y")


def chain_fwd_operands(M, mlp, g, exact_lnf=False):
    o = E.ints((M, 128), -8, 8, g, DEV, 0.25)
    wo = E.sparse_dyadic(128, 128, 3, -2, 0, g, DEV)
    bo = E.ints((128,), -8, 8, g, DEV, 0.125)
    a, _, _, _ = E.ln_rows(M, 128, g, DEV)
    x = a - (o @ wo.T + bo)                         # the residual that makes a = o Wo^T + bo + x a LayerNorm row
    ln2_w, ln2_b = E.ints((128,), -3, 3, g, DEV, 0.25), E.ints((128,), -4, 4, g, DEV, 0.125)
    w1 = E.sparse_dyadic(mlp, 128, 3, -3, -1, g, DEV)
    b1 = -32.0 * torch.ones(mlp, dtype=torch.float64, device=DEV) if exact_lnf else \
        E.ints((mlp,), 0, 1, g, DEV) * 64 - 32
    w2 = E.sparse_dyadic(128, mlp, 3, -3, -1, g, DEV)
    b2 = torch.full((128,), 0.375, dtype=torch.float64, device=DEV) if exact_lnf else E.ints((128,), -8, 8, g, DEV, 0.125)
    lnf_w, lnf_b = E.ints((128,), -7, 7, g, DEV, 0.25), E.ints((128,), -4, 4, g, DEV, 0.125)
    return [o, x, wo, bo, ln2_w, ln2_b, w1, b1, w2, b2, lnf_w, lnf_b]


@pytest.mark.parametrize("bf16", [True, False], ids=["pack", "tf32"])
@pytest.mark.parametrize("case", CHAIN_CASES + [("exact-lnf", 300, 512, 1)], ids=[c[0] for c in CHAIN_CASES] + ["exact-lnf"])
def test_encoder_chain_fwd_exact(case, bf16):
    """Every saved intermediate bit for bit.  LNf cannot keep the LayerNorm row structure through g = f W2^T + b2 + a, so
    meanf is checked bit for bit, rstdf against float64 1/sqrt(var) within 2 ulp of rsqrtf plus the 4-ulp worst case of the
    fp32 variance (8 rounded additions of positive terms), and y per element from the kernel's own meanf / rstdf; the
    'exact-lnf' case (f = 0, constant b2) keeps the structure and checks them bit for bit."""
    cid, M, mlp, add_input = case
    path = "bf16" if bf16 else "tf32"
    g = gen("chain" + cid)
    ops = chain_fwd_operands(M, mlp, g, exact_lnf=cid == "exact-lnf")
    o, x, wo, bo, ln2_w, ln2_b, w1, b1, w2, b2, lnf_w, lnf_b = ops
    ref = E.chain_fwd_ref(*ops, add_input)
    E.check_path(o, wo, path, (bo, x))
    E.check_path(ref["h2"], w1, path, (b1,))
    assert float(ref["pre"].abs().min()) >= 20, "GELU not saturated"
    E.check_path(ref["f"], w2, path, (b2, ref["a"]))
    E.sum_quanta(ref["g"], 1)
    w5 = [torch.zeros(128, 128, device=DEV), torch.zeros(256, 128, device=DEV), dev32(wo), dev32(w1), dev32(w2)]
    pk = pack_of(w5, mlp) if bf16 else None
    shapes = dict(a=(M, 128), h2=(M, 128), mean2=(M,), rstd2=(M,), pre=(M, mlp), f=(M, mlp), g=(M, 128), meanf=(M,),
                  rstdf=(M,), y=(M, 128))
    outs = [G(shapes[k]) for k in CHAIN_FWD_OUT]
    d = [dev32(t) for t in ops]
    fwd = lambda: L.call("tmf_encoder_chain_fwd", L.ptr(d[0]), L.ptr(d[1]), L.ptr(w5[2]), L.ptr(d[3]), L.ptr(d[4]), L.ptr(d[5]),
                         L.ptr(w5[3]), L.ptr(d[7]), L.ptr(w5[4]), L.ptr(d[9]), L.ptr(d[10]), L.ptr(d[11]),
                         *[L.ptr(t.t) for t in outs], M, mlp, add_input, 0.0, 0.0, L.ptr(pk))
    got = dict(zip(CHAIN_FWD_OUT, run_twice(outs, fwd)))
    exact = CHAIN_FWD_OUT if cid == "exact-lnf" else CHAIN_FWD_OUT[:8]
    for name in exact:
        check(got[name], ref[name], f"{cid} {path} {name}")
    if cid != "exact-lnf":
        r64 = ref["rstdf"]
        ulp = torch.pow(2.0, torch.floor(torch.log2(r64)) - 23)
        err = (got["rstdf"].double() - r64).abs()
        assert bool((err <= 6 * ulp).all()), f"{cid} rstdf: {float((err / ulp).max()):.2f} ulp"
        mf, rf = got["meanf"].double()[:, None], got["rstdf"].double()[:, None]
        dev = (got["g"].double() - mf) * rf * lnf_w
        want = dev + lnf_b + (x if add_input else 0)
        bound = 2.0 ** -22 * (dev.abs() + lnf_b.abs() + (x.abs() if add_input else 0)) + 2.0 ** -60
        bad = (got["y"].double() - want).abs() > bound
        assert not bool(bad.any()), f"{cid} y: {int(bad.sum())} elements outside the rounding bound"
    expect_kernel(fwd, "enc_chain_fwd_kernel")


CHAIN_BWD_OUT = ("dg", "dp", "da", "dout", "dxp", "dlnf_w", "dlnf_b", "dln2_w", "dln2_b")


def chain_bwd_operands(cid, M, mlp, add_input):
    """(inputs, reference) of one chain-backward case; asserts the bf16x3 condition of its three chained GEMMs (it implies
    the 3xTF32 one) and the 2^24 bound of the LayerNorm parameter sums."""
    g = gen("chainbwd" + cid)
    gt, meanf, rstdf, pg = E.ln_rows(M, 128, g, DEV, shared=True)
    at, mean2, rstd2, pa = E.ln_rows(M, 128, g, DEV, shared=True)
    lnf_w, ln2_w = E.pow2((128,), -1, 0, g, DEV), E.pow2((128,), -1, 0, g, DEV)
    dy = E.paired_dy(M, pg[0], lnf_w, g, DEV)
    pre = (E.ints((M, mlp), 0, 1, g, DEV) * 2 - 1) * (20 + E.ints((M, mlp), 0, 64, g, DEV, 0.125))
    wo = E.sparse_dyadic(128, 128, 3, -2, 0, g, DEV)
    w1 = E.paired_rows(mlp, 128, pa[0], ln2_w, 2, -2, 0, g, DEV)
    w2 = E.sparse_dyadic(128, mlp, 3, -2, 0, g, DEV)
    ref = E.chain_bwd_ref(dy, gt, at, pre, wo, w1, w2, ln2_w, lnf_w, mean2, rstd2, meanf, rstdf, add_input)
    E.check_path(ref["dg"], w2.T, "bf16")
    E.check_path(ref["dp"], w1.T, "bf16")
    E.check_path(ref["da"], wo.T, "bf16")
    for t, tt in ((dy, (gt - meanf[:, None]) * rstdf[:, None]), (ref["dh2"], (at - mean2[:, None]) * rstd2[:, None])):
        E.sum_quanta(t, 0)
        E.sum_quanta(t * tt, 0)
    return (dy, gt, at, pre, wo, w1, w2, ln2_w, lnf_w, mean2, rstd2, meanf, rstdf), ref


@pytest.mark.parametrize("bf16", [True, False], ids=["pack", "tf32"])
@pytest.mark.parametrize("case", CHAIN_CASES, ids=[c[0] for c in CHAIN_CASES])
def test_encoder_chain_bwd_exact(case, bf16):
    """Inputs of its own: g and a on shared LayerNorm patterns at power-of-two rstd, dy and W1 row-balanced (tests/fusion_exact.py
    paired_dy / paired_rows) so that the chained GEMM operands stay within the path's width, pre saturated (|pre| >= 20)."""
    cid, M, mlp, add_input = case
    ins64, ref = chain_bwd_operands(*case)
    dy, gt, at, pre, wo, w1, w2, ln2_w, lnf_w, mean2, rstd2, meanf, rstdf = ins64
    w5 = [torch.zeros(128, 128, device=DEV), torch.zeros(256, 128, device=DEV), dev32(wo), dev32(w1), dev32(w2)]
    pk = pack_of(w5, mlp) if bf16 else None
    shapes = dict(dg=(M, 128), dp=(M, mlp), da=(M, 128), dout=(M, 128), dxp=(M, 128), dlnf_w=(128,), dlnf_b=(128,),
                  dln2_w=(128,), dln2_b=(128,))
    outs = [G(shapes[k]) for k in CHAIN_BWD_OUT]
    ins = [dev32(t) for t in (dy, gt, at, pre)] + w5[2:] + [dev32(t) for t in (ln2_w, lnf_w, mean2, rstd2, meanf, rstdf)]
    ws = Scratch()
    bwd = lambda: L.call("tmf_encoder_chain_bwd", *[L.ptr(t) for t in ins], *[L.ptr(t.t) for t in outs], M, mlp, add_input,
                         L.ptr(pk), *ws.args())
    got = dict(zip(CHAIN_BWD_OUT, run_twice(outs, bwd, ws=ws)))
    path = "bf16" if bf16 else "tf32"
    for name in CHAIN_BWD_OUT:
        check(got[name], ref[name], f"{cid} {path} {name}")
    expect_kernel(bwd, "enc_chain_bwd_kernel")


WG_MAX_TOKENS = 21 * 416        # mlp = 512: 48 tiles x 21 splits x (32 x 128 + 32) floats fill the scratch buffer's partials
WGRAD_CASES = [  # (id, Mx, Mc, mlp, nsplit)
    ("nsplit1", 300, 150, 128, 1), ("model", B8, B8, 512, 3), ("ctx-300", B8, 2 * B8, 256, 6),
    ("x-gt-ctx", 900, 150, 512, 3), ("ragged", 37, 29, 128, 1), ("nsplit-max", WG_MAX_TOKENS, 300, 512, 21)]


def wgrad_operands(Mx, Mc, mlp, g):
    dy = lambda m, n: E.ints((m, n), -8, 8, g, DEV, 0.125)        # 4 significant bits: the tf32 hi half holds them
    xx = lambda m, n: E.ints((m, n), -64, 64, g, DEV, 2.0 ** -4)
    return dict(dq=dy(Mx, 128), h1=xx(Mx, 128), dkv=dy(Mc, 256), ctx=xx(Mc, 128), da=dy(Mx, 128), o=xx(Mx, 128),
                dp=dy(Mx, mlp), h2=xx(Mx, 128), dg=dy(Mx, 128), f=xx(Mx, mlp))


@pytest.mark.parametrize("case", WGRAD_CASES, ids=[c[0] for c in WGRAD_CASES])
def test_encoder_wgrad_exact(case):
    cid, Mx, Mc, mlp, nsplit = case
    assert -(-max(Mx, Mc) // 416) == nsplit
    g = gen("wgrad" + cid)
    t = wgrad_operands(Mx, Mc, mlp, g)
    probs = [("dWq", "dq", "h1", None), ("dWkv", "dkv", "ctx", None), ("dWo", "da", "o", "dbo"), ("dW1", "dp", "h2", "db1"),
             ("dW2", "dg", "f", "db2")]
    outs, want = {}, {}
    for w, dyn, xn, bn in probs:
        E.check_path(t[dyn].T, t[xn].T, "tf32")
        want[w] = t[dyn].T @ t[xn]
        outs[w] = G(tuple(want[w].shape))
        if bn:
            want[bn] = t[dyn].sum(0)
            outs[bn] = G((t[dyn].shape[1],))
    d = {k: dev32(v) for k, v in t.items()}
    tl = [d["dq"], d["h1"], outs["dWq"].t, d["dkv"], d["ctx"], outs["dWkv"].t, d["da"], d["o"], outs["dWo"].t, outs["dbo"].t,
          d["dp"], d["h2"], outs["dW1"].t, outs["db1"].t, d["dg"]]
    arr = (ctypes.c_void_p * 15)(*[x.data_ptr() for x in tl])
    ws = Scratch()
    names = list(outs)
    run = lambda: L.call("tmf_encoder_wgrad", arr, L.ptr(d["f"]), L.ptr(outs["dW2"].t), L.ptr(outs["db2"].t), Mx, Mc, mlp,
                         *ws.args())
    got = dict(zip(names, run_twice([outs[k] for k in names], run, ws=ws)))
    for k in names:
        check(got[k], want[k], f"{cid} {k}")
    expect_kernel(run, "enc_wgrad_kernel")
    if cid == "nsplit-max":     # one token more needs a 22nd split: refused, nothing launched
        with pytest.raises(RuntimeError, match="too large for the scratch buffer"):
            L.call("tmf_encoder_wgrad", arr, L.ptr(d["f"]), L.ptr(outs["dW2"].t), L.ptr(outs["db2"].t), WG_MAX_TOKENS + 1, Mc,
                   mlp, *ws.args())



# ---------------------------------------------------------------------------------------------------------------
# Gaussian data: per-element rounding bounds against float64 of the same fp32 inputs.  U = 2^-24; a GEMM output over K
# terms may be off by (EPS_SPLIT + 2 (K + 8) U) times the same product on absolute values (EPS_SPLIT: the dropped lo*lo
# term and the lo halves' own rounding of the bf16x3 / 3xTF32 splits, 3 * 2^-18 relative per product; 0 on the fp32-FMA
# kernels; 2 (K + 8) U: twice the longest fp32 accumulation chain plus the epilogue adds, a truncating adder losing 2^-23
# of the running absolute sum per link).  These cover what the exact cases avoid: the non-saturated GELU (erff and the
# erf_fast of enc_fused.cu, 1.5e-7 absolute plus 2^-19 of fp32 evaluation), LayerNorm with eps != 0 and a general rstd
# (rsqrtf: 2 ulp), and a softmax that is not one-hot (__expf, __logf: 2^-21 relative).
U = 2.0 ** -24
EPS_SPLIT = 3 * 2.0 ** -18
ERF_ABS = 1.5e-7 + 2.0 ** -19


def within(got, want, bound, what):
    err = (got.double() - want).abs()
    bad = ~(err <= bound)
    if bool(bad.any()):
        i = tuple(int(c) for c in bad.nonzero()[0])
        raise AssertionError(f"{what}: {int(bad.sum())} of {got.numel()} elements outside the bound; first at {i}: got "
                             f"{float(got[i])}, want {float(want[i])}, bound {float(bound[i]):.3g}")


def gemm_bound(a, w, K, split=True):
    return ((EPS_SPLIT if split else 0.0) + 2 * (K + 8) * U) * (a.abs() @ w.abs().T)


def randn(shape, g, scale=1.0):
    return (torch.randn(shape, generator=g, device=DEV) * scale).double()


def gelu_bound(pre, dpre):
    """|GELU(pre + dpre) - GELU(pre)| with GELU' <= 1.13, plus the kernel's erf error and roundings."""
    return 1.13 * dpre + 0.5 * pre.abs() * ERF_ABS + 4 * U * pre.abs() + 1e-37


def ln_fwd_bound(x, gamma, beta, eps, extra=None):
    """(y, mean, rstd) bounds of an fp32 LayerNorm of x (float64 copy of the fp32 input)."""
    dim = x.shape[-1]
    mean = x.mean(-1, keepdim=True)
    var = ((x - mean) ** 2).mean(-1, keepdim=True)
    rstd = (var + eps) ** -0.5
    dmu = 2 * (dim + 8) * U * x.abs().mean(-1, keepdim=True)
    rho = (dim + 8) * U + 2.0 ** -22 + dmu ** 2 * rstd ** 2 + dmu * (x - mean).abs().mean(-1, keepdim=True) * rstd ** 2
    xh = (x - mean) * rstd
    dxh = rstd * dmu + xh.abs() * (rho + 2 * U)
    by = gamma.abs() * dxh + 3 * U * ((xh * gamma).abs() + beta.abs() + (0 if extra is None else extra.abs()))
    return by, dmu.squeeze(-1), (rho * rstd).squeeze(-1)


@pytest.mark.parametrize("M,K,N,act,res", [(B8, 128, 512, 1, False), (B8, 512, 128, 0, True), (77, 30, 20, 1, True)])
def test_linear_gaussian_within_rounding_bound(M, K, N, act, res):
    g = gen(f"lin-gauss{M}-{K}-{N}")
    x, w, b = randn((M, K), g), randn((N, K), g, K ** -0.5), randn((N,), g, 0.1)
    r = randn((M, N), g) if res else None
    dy = randn((M, N), g)
    xs, wsf, bs, rs, dys = dev32(x), dev32(w), dev32(b), dev32(r) if res else None, dev32(dy)
    pre64 = x @ w.T + b
    y64 = (torch.nn.functional.gelu(pre64) if act else pre64) + (r if res else 0)
    y, pre = torch.empty(M, N, device=DEV), torch.empty(M, N, device=DEV)
    L.call("tmf_linear_fwd", L.ptr(xs), L.ptr(wsf), L.ptr(bs), L.ptr(rs), L.ptr(y), L.ptr(pre), M, K, N, act)
    dx, dw, db = torch.empty(M, K, device=DEV), torch.empty(N, K, device=DEV), torch.empty(N, device=DEV)
    ws = Scratch()
    L.call("tmf_linear_dgrad", L.ptr(dys), L.ptr(wsf), L.ptr(dx), M, K, N, 0)
    L.call("tmf_linear_wgrad", L.ptr(dys), L.ptr(xs), L.ptr(dw), L.ptr(db), M, K, N, *ws.args())
    torch.cuda.synchronize()
    bpre = gemm_bound(x, w, K, split=False) + 2 * (K + 8) * U * b.abs()
    within(pre, pre64, bpre, "pre")
    by = (gelu_bound(pre64, bpre) if act else bpre) + 2 * U * (y64.abs() + (r.abs() if res else 0))
    within(y, y64, by, "y")
    # the entry points are the GEMMs of the Linear's backward (the GELU backward is tmf_gelu_bwd's): dy w, dy^T x, sum dy
    within(dx, dy @ w, gemm_bound(dy, w.T, N, split=False), "dx")
    within(dw, dy.T @ x, gemm_bound(dy.T, x.T, M, split=False), "dw")
    within(db, dy.sum(0), 2 * (M + 8) * U * dy.abs().sum(0), "dbias")


@pytest.mark.parametrize("rows,dim", [(B8, 128), (45, 160), (19, 1024)])
def test_layernorm_gaussian_within_rounding_bound(rows, dim):
    g = gen(f"ln-gauss{rows}-{dim}")
    x = randn((rows, dim), g, 2.0) + 0.3
    gamma, beta, dy = 1 + randn((dim,), g, 0.1), randn((dim,), g, 0.1), randn((rows, dim), g)
    eps = 1e-5
    xs, gs, bs, dys = dev32(x), dev32(gamma), dev32(beta), dev32(dy)
    y, mean, rstd = torch.empty(rows, dim, device=DEV), torch.empty(rows, device=DEV), torch.empty(rows, device=DEV)
    L.call("tmf_layernorm_fwd", L.ptr(xs), L.ptr(gs), L.ptr(bs), L.ptr(None), L.ptr(y), L.ptr(mean), L.ptr(rstd), rows, dim, eps)
    torch.cuda.synchronize()
    y64, m64, r64 = E.layernorm_ref(x, gamma, beta, eps)
    by, bm, br = ln_fwd_bound(x, gamma, beta, eps)
    within(mean, m64, bm, "mean")
    within(rstd, r64, br, "rstd")
    within(y, y64, by, "y")
    # backward at the kernel's statistics: dx = rstd (gg - mean(gg) - xh mean(gg xh)) against autograd-equivalent float64
    ws = Scratch()
    dx, dg, db = torch.empty(rows, dim, device=DEV), torch.empty(dim, device=DEV), torch.empty(dim, device=DEV)
    L.call("tmf_layernorm_bwd", L.ptr(dys), L.ptr(xs), L.ptr(gs), L.ptr(mean), L.ptr(rstd), L.ptr(dx), L.ptr(dg), L.ptr(db),
           rows, dim, 0, *ws.args())
    torch.cuda.synchronize()
    mk, rk = mean.double(), rstd.double()
    dx64, dg64, db64 = E.layernorm_bwd_ref(dy, x, gamma, mk, rk)
    xh = (x - mk[:, None]) * rk[:, None]
    gg = dy * gamma
    c = 2 * (dim + 8) * U
    s1b, s2b = c * gg.abs().mean(1, keepdim=True), c * (gg * xh).abs().mean(1, keepdim=True) + 4 * U * (gg * xh).abs().mean(1, keepdim=True)
    s2 = (gg * xh).mean(1, keepdim=True)
    bdx = rk[:, None] * (s1b + xh.abs() * s2b + 4 * U * xh.abs() * s2.abs() + 6 * U * (gg.abs() + gg.mean(1, keepdim=True).abs() + (xh * s2).abs()))
    within(dx, dx64, bdx, "dx")
    cr = 2 * (rows + 300) * U
    within(dg, dg64, cr * (dy * xh).abs().sum(0) + 4 * U * (dy * xh).abs().sum(0), "dgamma")
    within(db, db64, cr * dy.abs().sum(0), "dbeta")


@pytest.mark.parametrize("B,Nq,Nk,heads,dh", [(8, 150, 150, 4, 32), (2, 37, 300, 2, 64), (2, 150, 150, 8, 16)])
def test_attention_gaussian_within_rounding_bound(B, Nq, Nk, heads, dh):
    """Softmax that is not one-hot, forward and backward (whichever implementation TMF_ATTN_IMPL selects)."""
    g = gen(f"attn-gauss{B}-{Nq}-{Nk}-{dh}")
    inner, scale = heads * dh, dh ** -0.5
    q, kv, do = randn((B, Nq, inner), g), randn((B, Nk, 2 * inner), g), randn((B, Nq, inner), g)
    qs, kvs, dos = dev32(q), dev32(kv), dev32(do)
    out, lse = torch.empty(B, Nq, inner, device=DEV), torch.empty(B, heads, Nq, device=DEV)
    L.call("tmf_attn_fwd", L.ptr(qs), L.ptr(kvs), L.ptr(out), L.ptr(lse), B, Nq, Nk, heads, dh, scale)
    dq, dkv = torch.empty(B, Nq, inner, device=DEV), torch.empty(B, Nk, 2 * inner, device=DEV)
    L.call("tmf_attn_bwd", L.ptr(dos), L.ptr(qs), L.ptr(kvs), L.ptr(out), L.ptr(lse), L.ptr(dq), L.ptr(dkv), B, Nq, Nk, heads,
           dh, scale)
    torch.cuda.synchronize()
    out64, lse64, dots, P = E.attention_ref(q, kv, heads, dh, scale)
    dq64, dkv64, dP = E.attention_bwd_ref(do, q, kv, heads, dh, scale)
    sp = lambda t, n: t.reshape(B, n, heads, dh).permute(0, 2, 1, 3)
    k, v, dO = sp(kv[..., :inner], Nk).abs(), sp(kv[..., inner:], Nk).abs(), sp(do, Nq).abs()
    qa = sp(q, Nq).abs()
    eg = lambda n: EPS_SPLIT + 2 * (n + 8) * U
    Es = (scale * eg(dh) * (qa @ k.transpose(-1, -2))).amax(-1, keepdim=True) + 2 * U * dots.abs().amax(-1, keepdim=True)
    eta = 2 * (Es + 2.0 ** -21) + 4 * U                                  # relative error of every P_ij
    bout = (eta + eg(Nk)) * (P @ v) + 2 * U * sp(out64, Nq).abs()
    within(out, out64, bout.permute(0, 2, 1, 3).reshape(B, Nq, inner), "out")
    within(lse, lse64, Es.squeeze(-1) + 2.0 ** -21 + 2 * U * lse64.abs() + (Nk + 8) * U, "lse")
    # backward: dS = P (dP - D); D from the kernel's own out
    ok = sp(out.double(), Nq)
    D = (sp(do, Nq) * ok).sum(-1, keepdim=True)
    dO_o = (dO * (sp(out64, Nq) - ok).abs()).sum(-1, keepdim=True)
    dPb = eg(dh) * (dO @ v.transpose(-1, -2))
    Db = eg(dh) * (dO * ok.abs()).sum(-1, keepdim=True) + dO_o
    dS = P * (dP - D)
    dSb = eta * P * (dP - D).abs() + P * (dPb + Db) + 2 * U * dS.abs()
    bdq = scale * (dSb @ k + eg(Nk) * (dS.abs() @ k))
    bdk = scale * (dSb.transpose(-1, -2) @ qa + eg(Nq) * (dS.abs().transpose(-1, -2) @ qa))
    bdv = (eta * P).transpose(-1, -2) @ dO + eg(Nq) * (P.transpose(-1, -2) @ dO)
    m = lambda t, n: t.permute(0, 2, 1, 3).reshape(B, n, inner)
    within(dq, dq64, m(bdq, Nq), "dq")
    within(dkv, dkv64, torch.cat([m(bdk, Nk), m(bdv, Nk)], -1), "dkv")


@pytest.mark.parametrize("bf16", [True, False], ids=["pack", "tf32"])
@pytest.mark.parametrize("M,mlp", [(B8, 512), (37, 128)])
def test_encoder_chain_fwd_gaussian_within_rounding_bound(M, mlp, bf16):
    """Every saved stage of tmf_encoder_chain_fwd on Gaussian data against float64 of that stage's inputs as the kernel
    saved them (so a bound covers one stage's rounding, and a wrong element is located in the stage that made it): the
    non-saturated erf_fast GELU, LN2 / LNf with eps = 1e-5."""
    g = gen(f"chain-gauss{M}-{mlp}")
    o, x = randn((M, 128), g), randn((M, 128), g)
    wo, w1, w2 = randn((128, 128), g, 128 ** -0.5), randn((mlp, 128), g, 128 ** -0.5), randn((128, mlp), g, mlp ** -0.5)
    bo, b1, b2 = randn((128,), g, 0.1), randn((mlp,), g, 0.1), randn((128,), g, 0.1)
    ln2_w, ln2_b, lnf_w, lnf_b = 1 + randn((128,), g, 0.2), randn((128,), g, 0.1), 1 + randn((128,), g, 0.2), randn((128,), g, 0.1)
    eps = 1e-5
    d = [dev32(t) for t in (o, x, wo, bo, ln2_w, ln2_b, w1, b1, w2, b2, lnf_w, lnf_b)]
    w5 = [torch.zeros(128, 128, device=DEV), torch.zeros(256, 128, device=DEV), d[2], d[6], d[8]]
    pk = pack_of(w5, mlp) if bf16 else None
    shapes = dict(a=(M, 128), h2=(M, 128), mean2=(M,), rstd2=(M,), pre=(M, mlp), f=(M, mlp), g=(M, 128), meanf=(M,),
                  rstdf=(M,), y=(M, 128))
    k = {n: torch.empty(shapes[n], device=DEV) for n in CHAIN_FWD_OUT}
    L.call("tmf_encoder_chain_fwd", *[L.ptr(t) for t in d], *[L.ptr(k[n]) for n in CHAIN_FWD_OUT], M, mlp, 1, eps, eps,
           L.ptr(pk))
    torch.cuda.synchronize()
    k = {n: t.double() for n, t in k.items()}
    x, o = d[1].double(), d[0].double()
    within(k["a"], o @ wo.T + bo + x, gemm_bound(o, wo, 128) + 4 * U * (bo.abs() + x.abs()), "a")
    h2, m2, r2 = E.layernorm_ref(k["a"], ln2_w, ln2_b, eps)
    by, bm, br = ln_fwd_bound(k["a"], ln2_w, ln2_b, eps)
    within(k["mean2"], m2, bm, "mean2")
    within(k["rstd2"], r2, br, "rstd2")
    within(k["h2"], h2, by, "h2")
    within(k["pre"], k["h2"] @ w1.T + b1, gemm_bound(k["h2"], w1, 128) + 4 * U * b1.abs(), "pre")
    within(k["f"], torch.nn.functional.gelu(k["pre"]), gelu_bound(k["pre"], 0.0), "f")
    within(k["g"], k["f"] @ w2.T + b2 + k["a"], gemm_bound(k["f"], w2, mlp) + 4 * U * (b2.abs() + k["a"].abs()), "g")
    y, mf, rf = E.layernorm_ref(k["g"], lnf_w, lnf_b, eps)
    by, bm, br = ln_fwd_bound(k["g"], lnf_w, lnf_b, eps, extra=x)
    within(k["meanf"], mf, bm, "meanf")
    within(k["rstdf"], rf, br, "rstdf")
    within(k["y"], y + x, by + 2 * U * (y + x).abs(), "y")

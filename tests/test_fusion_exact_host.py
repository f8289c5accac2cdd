"""CPU checks of tests/fusion_exact.py: the float64 references against torch (F.linear, F.layer_norm, the softmax attention
and autograd), the bit and 2^24 bounds of every generated case of tests/test_gpu_fusion_exact.py, and the disjointness of
the scratch buffer's ticket ranges (csrc/common.cuh)."""
import os
import re

import pytest
import torch
import torch.nn.functional as F

from tests import fusion_exact as E
from tests import test_gpu_fusion_exact as T

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture
def cpu(monkeypatch):
    monkeypatch.setattr(T, "DEV", "cpu")
    return T


def rnd(*shape, seed=0):
    return torch.randn(shape, generator=torch.Generator().manual_seed(seed), dtype=torch.float64)


# ---------------------------------------------------------------------------------------------------------------
# references against torch
def test_linear_and_layernorm_references_match_torch():
    x, w, b, r = rnd(7, 12), rnd(5, 12, seed=1), rnd(5, seed=2), rnd(7, 5, seed=3)
    y, pre = E.linear_ref(x, w, b, r, act=1)
    assert torch.allclose(pre, F.linear(x, w, b)) and torch.allclose(y, F.gelu(F.linear(x, w, b)) + r)
    g, beta = rnd(12, seed=4), rnd(12, seed=5)
    y, mean, rstd = E.layernorm_ref(x, g, beta, 1e-5, x)
    assert torch.allclose(y, F.layer_norm(x, (12,), g, beta, 1e-5) + x)
    xl, gl, bl = [t.clone().requires_grad_(True) for t in (x, g, beta)]
    dy = rnd(7, 12, seed=6)
    F.layer_norm(xl, (12,), gl, bl, 0.0).backward(dy)
    _, mean, rstd = E.layernorm_ref(x, g, beta, 0.0)
    dx, dg, db = E.layernorm_bwd_ref(dy, x, g, mean, rstd)
    assert torch.allclose(dx, xl.grad) and torch.allclose(dg, gl.grad) and torch.allclose(db, bl.grad)


def test_attention_references_match_torch_autograd():
    B, Nq, Nk, heads, dh, scale = 2, 5, 7, 2, 4, 0.3
    q, kv, do = rnd(B, Nq, heads * dh), rnd(B, Nk, 2 * heads * dh, seed=1), rnd(B, Nq, heads * dh, seed=2)
    ql, kvl = q.clone().requires_grad_(True), kv.clone().requires_grad_(True)
    sp = lambda t, n: t.reshape(B, n, heads, dh).permute(0, 2, 1, 3)
    k, v = kvl.chunk(2, -1)
    attn = torch.softmax(sp(ql, Nq) @ sp(k, Nk).transpose(-1, -2) * scale, -1)
    out = (attn @ sp(v, Nk)).permute(0, 2, 1, 3).reshape(B, Nq, heads * dh)
    out.backward(do)
    o, lse, dots, p = E.attention_ref(q, kv, heads, dh, scale)
    assert torch.allclose(o, out) and torch.allclose(p, attn) and torch.allclose(lse, torch.logsumexp(dots, -1))
    dq, dkv, dattn = E.attention_bwd_ref(do, q, kv, heads, dh, scale)
    assert torch.allclose(dq, ql.grad) and torch.allclose(dkv, kvl.grad)
    assert torch.allclose(dattn, sp(do, Nq) @ sp(kv[..., heads * dh:], Nk).transpose(-1, -2))


def test_encoder_references_match_autograd():
    """chain_bwd_ref / proj_bwd_ref against autograd through chain_fwd_ref / proj_fwd_ref (eps = 1e-5, random data)."""
    M, mlp = 6, 32
    names = ["o", "x", "wo", "bo", "ln2_w", "ln2_b", "w1", "b1", "w2", "b2", "lnf_w", "lnf_b"]
    shapes = [(M, 128), (M, 128), (128, 128), (128,), (128,), (128,), (mlp, 128), (mlp,), (128, mlp), (128,), (128,), (128,)]
    leaves = {n: rnd(*s, seed=i).requires_grad_(True) for i, (n, s) in enumerate(zip(names, shapes))}
    for add_input in (0, 1):
        for t in leaves.values():
            t.grad = None
        f = E.chain_fwd_ref(*leaves.values(), add_input, 1e-5, 1e-5)
        dy = rnd(M, 128, seed=99)
        f["y"].backward(dy)
        d = {k: v.detach() for k, v in f.items()}
        lv = {k: v.detach() for k, v in leaves.items()}
        b = E.chain_bwd_ref(dy, d["g"], d["a"], d["pre"], lv["wo"], lv["w1"], lv["w2"], lv["ln2_w"], lv["lnf_w"], d["mean2"],
                            d["rstd2"], d["meanf"], d["rstdf"], add_input)
        assert torch.allclose(b["dlnf_w"], leaves["lnf_w"].grad) and torch.allclose(b["dlnf_b"], leaves["lnf_b"].grad)
        assert torch.allclose(b["dln2_w"], leaves["ln2_w"].grad) and torch.allclose(b["dln2_b"], leaves["ln2_b"].grad)
        assert torch.allclose(b["dout"], leaves["o"].grad)
        assert torch.allclose(b["dxp"] + b["dout"] @ torch.zeros(128, 128, dtype=torch.float64), leaves["x"].grad)
    x, ctx = rnd(M, 128).requires_grad_(True), rnd(9, 128, seed=1).requires_grad_(True)
    lw, lb, wq, wkv = rnd(128, seed=2).requires_grad_(True), rnd(128, seed=3), rnd(128, 128, seed=4), rnd(256, 128, seed=5)
    f = E.proj_fwd_ref(x, ctx, lw, lb, wq, wkv, 1e-5)
    dq, dkv = rnd(M, 128, seed=6), rnd(9, 256, seed=7)
    (f["q"] * dq).sum().add((f["kv"] * dkv).sum()).backward()
    b = E.proj_bwd_ref(dq, dkv, torch.zeros(M, 128, dtype=torch.float64), x.detach(), lw.detach(), f["mean1"].detach(),
                       f["rstd1"].detach(), wq, wkv)
    assert torch.allclose(b["dx"], x.grad) and torch.allclose(b["dctx"], ctx.grad) and torch.allclose(b["dln_w"], lw.grad)


def test_saturated_gelu_and_one_hot_softmax_round_to_exact_fp32():
    pre = torch.tensor([20.0, 33.5, -20.0, -40.25], dtype=torch.float64)
    assert torch.equal(E.f32(E.gelu(pre)), torch.tensor([20.0, 33.5, -0.0, -0.0]))
    assert torch.equal(E.f32(E.gelu_grad(pre)), torch.tensor([1.0, 1.0, 0.0, 0.0]))
    g = torch.Generator().manual_seed(3)
    q, kv, win = E.one_hot_attention(2, 37, 29, 2, 16, g, "cpu")
    out, lse, dots, attn = E.attention_ref(q, kv, 2, 16, 0.5)
    assert torch.equal(E.f32(attn), (attn.argmax(-1, keepdim=True) == torch.arange(29)).float())
    assert bool((attn.argmax(-1) == win).all())
    top2 = dots.topk(2, -1).values
    assert float((top2[..., 0] - top2[..., 1]).min()) >= 128


def test_layernorm_rows_have_exact_statistics():
    g = torch.Generator().manual_seed(1)
    for dim in (96, 128, 160, 1024):
        x, m, rstd, p = E.ln_rows(9, dim, g, "cpu")
        _, mean, r = E.layernorm_ref(x, torch.ones(dim, dtype=torch.float64), torch.zeros(dim, dtype=torch.float64), 0.0)
        assert torch.equal(mean, m) and torch.equal(r, rstd)
        gamma = E.pow2((dim,), -1, 1, g, "cpu")
        pat = E.ln_pattern(1, dim, g, "cpu")[0]
        dy = E.paired_dy(9, pat, gamma, g, "cpu")
        assert float((dy * gamma).sum(1).abs().max()) == 0 and float((dy * gamma * pat).sum(1).abs().max()) == 0
        assert int((dy != 0).sum(1).min()) > dim // 2


def test_sig_bits_and_quantum():
    t = torch.tensor([0.0, 3.0, -0.375, 1024.0 + 1.0], dtype=torch.float64)
    assert E.sig_bits(t) == 11 and E.quantum(t) == 0.125
    with pytest.raises(AssertionError):
        E.gemm_quanta(torch.full((1, 300), 4095.0), torch.full((1, 300), 4095.0))


def test_split_paths_need_one_short_side_per_k():
    """bf16x3 drops xl*wl: two 12-bit columns at the same k are refused, a 16-bit column against an 8-bit one is taken;
    3xTF32 likewise at 11 / 22 bits."""
    a12, w12 = torch.full((2, 4), 4095.0, dtype=torch.float64), torch.full((3, 4), 4095.0, dtype=torch.float64)
    with pytest.raises(AssertionError, match="k = 0"):
        E.check_path(a12, w12, "bf16")
    a16, w8 = torch.full((2, 4), 32769.0, dtype=torch.float64), torch.full((3, 4), 2.0 ** 7, dtype=torch.float64)
    E.check_path(a16, w8, "bf16")
    mixed = w8.clone()
    mixed[:, 2] = 4095.0
    with pytest.raises(AssertionError, match="k = 2"):
        E.check_path(torch.full((2, 4), 4095.0, dtype=torch.float64), mixed, "bf16")
    E.check_path(torch.full((2, 4), 4097.0, dtype=torch.float64), torch.full((3, 4), 3.0, dtype=torch.float64), "tf32")
    with pytest.raises(AssertionError):
        E.check_path(torch.full((2, 4), 4095.0, dtype=torch.float64), torch.full((3, 4), 4095.0, dtype=torch.float64), "tf32")


# ---------------------------------------------------------------------------------------------------------------
# every generated case keeps its path's bounds (the asserts the GPU tests make before they launch, without the launch)
@pytest.mark.parametrize("case", T.LINEAR_CASES, ids=[c[0] for c in T.LINEAR_CASES])
def test_linear_case_bounds(case, cpu):
    _, M, K, N, act, res = case
    g = cpu.gen(case[0])
    x, w, bias = cpu.linear_operands(M, K, N, act, g)
    E.check_path(x, w, "fma", (bias,))
    if act:
        assert float(E.linear_ref(x, w, bias, act=1)[1].abs().min()) >= 20


@pytest.mark.parametrize("case", T.CHAIN_CASES + [("exact-lnf", 300, 512, 1)])
def test_chain_fwd_case_bounds(case, cpu):
    cid, M, mlp, add_input = case
    ops = cpu.chain_fwd_operands(M, mlp, cpu.gen("chain" + cid), exact_lnf=cid == "exact-lnf")
    ref = E.chain_fwd_ref(*ops, add_input)
    for path in ("bf16", "tf32"):
        E.check_path(ops[0], ops[2], path, (ops[3], ops[1]))
        E.check_path(ref["h2"], ops[6], path, (ops[7],))
        E.check_path(ref["f"], ops[8], path, (ops[9], ref["a"]))
    assert float(ref["pre"].abs().min()) >= 20
    for k in ("a", "h2", "mean2", "rstd2", "pre", "f", "g", "meanf"):
        E.f32(ref[k])
    if cid == "exact-lnf":
        E.f32(ref["rstdf"])
        E.f32(ref["y"])


@pytest.mark.parametrize("case", T.CHAIN_CASES, ids=[c[0] for c in T.CHAIN_CASES])
def test_chain_bwd_case_bounds(case, cpu):
    ins, ref = cpu.chain_bwd_operands(*case)
    for k in T.CHAIN_BWD_OUT:
        E.f32(ref[k])
    assert float(ref["dp"].abs().max()) > 0 and float(ref["dln2_w"].abs().max()) > 0


@pytest.mark.parametrize("case", T.PROJ_CASES, ids=[c[0] for c in T.PROJ_CASES])
def test_proj_case_bounds(case, cpu):
    _, ref, bref = cpu.proj_operands(*case)
    for v in list(ref.values()) + list(bref.values()):
        E.f32(v)


@pytest.mark.parametrize("case", T.WGRAD_CASES, ids=[c[0] for c in T.WGRAD_CASES])
def test_wgrad_case_bounds(case, cpu):
    cid, Mx, Mc, mlp, nsplit = case
    assert -(-max(Mx, Mc) // 416) == nsplit
    t = cpu.wgrad_operands(Mx, Mc, mlp, cpu.gen("wgrad" + cid))
    for dyn, xn in (("dq", "h1"), ("dkv", "ctx"), ("da", "o"), ("dp", "h2"), ("dg", "f")):
        E.check_path(t[dyn].T, t[xn].T, "tf32")
    # the largest split count the scratch buffer admits at mlp = 512 (48 tiles), and one more does not fit
    part = (16 << 20) - 16384
    assert 48 * 21 * (32 * 128 + 32) * 4 <= part < 48 * 22 * (32 * 128 + 32) * 4


@pytest.mark.parametrize("case", T.ATTN_CASES, ids=[c[0] for c in T.ATTN_CASES])
def test_attention_case_bounds(case, cpu):
    cid, B, Nq, Nk, heads, dh = case
    q, kv, win, dout, scale = cpu.attention_operands(*case)
    out, lse, dots, attn = E.attention_ref(q, kv, heads, dh, scale)
    E.f32(out), E.f32(lse), E.f32(attn)
    for t in E.attention_bwd_ref(dout, q, kv, heads, dh, scale):
        E.f32(t)
    if Nk > 1:
        top2 = dots.topk(2, -1).values
        assert float((top2[..., 0] - top2[..., 1]).min()) >= 128
    if Nq >= Nk:
        assert all(set(win[b, h].tolist()) == set(range(Nk)) for b in range(B) for h in range(heads))


def test_linear_cases_cover_every_kernel_and_split():
    T.test_linear_cases_cover_every_gemm_kernel()
    T.test_linear_cases_cover_every_wgrad_split()


# ---------------------------------------------------------------------------------------------------------------
def test_scratch_ticket_ranges_are_disjoint():
    """Every ticket user of the scratch buffer owns its own words inside the 16 KB ticket area (csrc/common.cuh), and the
    entry points stay inside them."""
    src = open(os.path.join(ROOT, "transmf_ad_b200", "csrc", "common.cuh")).read()
    vals = {k: int(v) for k, v in re.findall(r"\b(TK_\w+) = (\d+)", src)}
    n3 = re.search(r"TK_ENC_N = (\d+) \* (\d+)", src)
    vals["TK_ENC_N"] = int(n3.group(1)) * int(n3.group(2))
    tickets = int(re.search(r"TMF_WS_TICKET_BYTES = (\d+)", src).group(1)) // 4
    ranges = sorted((vals[k], vals[k] + vals[k + "_N"], k) for k in ("TK_LN", "TK_GEMM", "TK_COLSUM", "TK_ENC"))
    for (a0, a1, a), (b0, b1, b) in zip(ranges, ranges[1:]):
        assert a1 <= b0, f"{a} [{a0}, {a1}) overlaps {b} [{b0}, {b1})"
    assert ranges[0][0] >= 0 and ranges[-1][1] <= tickets
    fo = open(os.path.join(ROOT, "transmf_ad_b200", "csrc", "fusion_ops.cu")).read()
    ef = open(os.path.join(ROOT, "transmf_ad_b200", "csrc", "enc_fused.cu")).read()
    assert "tiles > (int)TK_GEMM_N" in fo and "tickets + TK_GEMM;" in fo          # split-K GEMM tiles
    assert "grid.x <= TK_COLSUM_N" in fo and "tickets + TK_COLSUM)" in fo       # column blocks
    assert "+ TK_ENC + which * 64" in ef and "tiles <= (int)TK_ENC_N / 3" in ef  # 3 encoder kernels x 64 words
    assert len(re.findall(r"enc_tickets\(ws, (\d)\)", ef)) == 3 and max(map(int, re.findall(r"enc_tickets\(ws, (\d)\)", ef))) == 2

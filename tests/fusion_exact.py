"""Exact-arithmetic references and operand generators for the fusion-transformer kernel tests
(tests/test_gpu_fusion_exact.py): Linear, LayerNorm, the attention core, token pooling and the fused encoder.

The GEMMs of these kernels take three arithmetic paths, each exact under its own condition:
  * bf16x3 (panel_gemm_bf16, attention_mma.cu): x*w ~= xh*wh + xl*wh + xh*wl with xh = bf16(x), xl = bf16(x - xh); the
    xl*wl product is dropped.  Exact when, for every reduction index k, both operands' elements have at most 16 significant
    bits (xh + xl == x) and one side's have at most 8 (its lo half is 0).  The encoder meets it with bf16 weights (the lo
    half of the pack is 0) and activations of at most 16 bits;
  * 3xTF32 (panel_gemm: pack == NULL, always in enc_wgrad_kernel): hi = x & 0xffffe000, lo = x - hi, the lo*lo product is
    dropped.  Exact when, for every k, one side has at most 11 significant bits (its lo is 0) and the other at most 22;
  * fp32 FMA (gemm_kernel, gemm_ksplit_kernel, attention.cu, the row-per-warp attention): exact on any grid.
On every path all partial sums must stay below 2^24 quanta of the products' common grid (gemm_quanta).  A correct kernel
then reproduces the float64 reference rounded once to fp32 (f32) bit for bit, whatever its tiling or reduction order.

The non-linear parts are exact only in chosen regimes:
  * LayerNorm with eps = 0 on rows m + s * P, P a permutation of {+-1 x 5/8 dim, +-3 x 3/8 dim} with balanced signs: mean m,
    variance 4 s^2, rstd = 1 / (2 s) for s a power of two (dim % 16 == 0);
  * GELU saturated: |pre| >= 20 gives GELU(pre) in {pre, -0} and GELU' in {1, 0} (exp(-200) underflows);
  * softmax one-hot: scores whose gaps to the row maximum are at least 128 make every other exp 0, so lse is the maximum,
    out the winner's v row, dS = P (dP - D) = 0 (dq = dk = 0) and dv[j] the sum of dO over the queries that chose key j.
"""
import math

import torch
import torch.nn.functional as F

from tests.conv_exact import FP32_EXACT

TF32_HI_BITS, TF32_BITS = 11, 22


# ---------------------------------------------------------------------------------------------------------------
# grids
def _frac(t):
    t = t.double().flatten()
    t = t[t != 0]
    if t.numel() == 0:
        return None, None
    m, e = torch.frexp(t.abs())                  # |t| = m 2^e, m in [0.5, 1)
    mi = (m * 2.0 ** 53).long()
    tz = torch.log2((mi & -mi).double()).round().long()
    return e.long() - 53 + tz, 53 - tz           # exponent of the lowest set bit, significant bits


def sig_bits(t):
    """Largest number of significant bits of any element (0 for an all-zero tensor)."""
    _, bits = _frac(t)
    return 0 if bits is None else int(bits.max())


def col_bits(t):
    """Significant bits of column k of a 2-D tensor: the largest over its elements (0 for an all-zero column)."""
    t = t.double()
    out = torch.zeros(t.shape[1], dtype=torch.long, device=t.device)
    nz = t != 0
    if bool(nz.any()):
        _, bits = _frac(t[nz])
        cols = nz.nonzero()[:, 1]
        out.scatter_reduce_(0, cols, bits, reduce="amax")
    return out


def quantum(t):
    """The largest power of two that every element is a multiple of (inf for an all-zero tensor)."""
    low, _ = _frac(t)
    return math.inf if low is None else 2.0 ** int(low.min())


def gemm_quanta(a, w, extra=()):
    """Worst |partial sum| of a @ w.T (+ the tensors in `extra`, broadcast) in units of the products' common quantum, with
    2 % margin for the hi / lo halves of a split; asserts it stays below 2^24."""
    q = quantum(a) * quantum(w)
    if math.isinf(q):
        return 0.0
    s = a.double().abs() @ w.double().abs().T
    for e in extra:
        assert quantum(e) >= q, "addend finer than the products' grid"
        s = s + e.double().abs()
    n = 1.02 * float(s.max()) / q
    assert n < FP32_EXACT, f"partial sums reach {n:.4g} quanta >= 2^24"
    return n


def sum_quanta(t, dim):
    """Worst |partial sum| of t summed along `dim`, in units of its quantum; asserts < 2^24."""
    q = quantum(t)
    if math.isinf(q):
        return 0.0
    n = float(t.double().abs().sum(dim).max()) / q
    assert n < FP32_EXACT, f"sum reaches {n:.4g} quanta >= 2^24"
    return n


SPLIT_BITS = {"bf16": (8, 16), "tf32": (TF32_HI_BITS, TF32_BITS)}   # (lo half is 0, hi + lo hold the value)


def check_path(a, w, path, extra=()):
    """Assert the exactness condition of one GEMM y = a @ w.T on `path` ('bf16', 'tf32' or 'fma'): for the split paths, at
    every reduction index k one side's column fits the hi half alone and both fit hi + lo (the dropped lo*lo product is
    then 0)."""
    if path in SPLIT_BITS:
        short, full = SPLIT_BITS[path]
        ba, bw = col_bits(a), col_bits(w)
        lo, hi = torch.minimum(ba, bw), torch.maximum(ba, bw)
        k = int(torch.argmax((lo > short).long() + (hi > full).long()))
        assert int(lo.max()) <= short and int(hi.max()) <= full, \
            f"{path} split inexact at k = {k}: columns of {int(ba[k])} and {int(bw[k])} significant bits"
    else:
        assert path == "fma", path
    return gemm_quanta(a, w, extra)


def f32(ref):
    """The fp32 a kernel must produce for a float64 reference that is an fp32 value up to far-below-ulp terms (exp(-128)
    tails of a one-hot softmax, Phi(-20) of a saturated GELU)."""
    r = ref.float()
    d = (r.double() - ref).abs()
    assert bool((d <= 1e-30 * ref.abs() + 1e-40).all()), "reference is not an fp32 value"
    return r


# ---------------------------------------------------------------------------------------------------------------
# generators (float64 on `device`)
def ints(shape, lo, hi, gen, device, scale=1.0):
    return torch.randint(lo, hi + 1, shape, generator=gen, device=device).double() * scale


def pow2(shape, lo, hi, gen, device, signed=True):
    """+-2^e with e uniform in [lo, hi]."""
    v = torch.ldexp(torch.ones(shape, dtype=torch.float64, device=device), ints(shape, lo, hi, gen, device).long())
    if signed:
        v = v * (ints(shape, 0, 1, gen, device) * 2 - 1)
    return v


def ln_pattern(rows, dim, gen, device, shared=False):
    """Rows of {+-1 x 5/8 dim, +-3 x 3/8 dim} with balanced signs, one permutation per row (or one for all rows)."""
    assert dim % 16 == 0
    n1, n3 = 5 * dim // 8, 3 * dim // 8
    base = torch.tensor([1.0] * (n1 // 2) + [-1.0] * (n1 // 2) + [3.0] * (n3 // 2) + [-3.0] * (n3 // 2),
                        dtype=torch.float64, device=device)
    if shared:
        return base[torch.randperm(dim, generator=gen, device=device)].expand(rows, dim).clone()
    keys = torch.rand((rows, dim), generator=gen, device=device)
    return base[keys.argsort(dim=1)]


def ln_rows(rows, dim, gen, device, shared=False, mq=2.0 ** -3):
    """x = m + s * P (m on the grid mq, s = 2^-1..2^1 per row): LayerNorm(eps = 0) has mean m and rstd 1 / (2 s) exactly."""
    p = ln_pattern(rows, dim, gen, device, shared)
    m = ints((rows, 1), -16, 16, gen, device, mq)
    s = pow2((rows, 1), -1, 1, gen, device, signed=False)
    return m + s * p, m.squeeze(1), (0.5 / s).squeeze(1), p


def sparse_dyadic(n, k, per_row, elo, ehi, gen, device):
    """W[n][k]: per_row entries +-2^e (e in [elo, ehi]) per row at random columns; row r always has one entry in the 32-wide
    k stage r mod (k / 32), so every stage is hit."""
    w = torch.zeros((n, k), dtype=torch.float64, device=device)
    for r in range(n):
        st = r % (k // 32)
        cols = [st * 32 + int(torch.randint(0, 32, (1,), generator=gen, device=device))]
        cols += torch.randint(0, k, (per_row - 1,), generator=gen, device=device).tolist()
        for c in cols:
            w[r, c] += float(pow2((1,), elo, ehi, gen, device))
    return w


def paired_rows(n, k, pattern, gamma, pairs_per_row, elo, ehi, gen, device):
    """W[n][k] whose rows w satisfy sum_c w[c] gamma[c] = 0 and sum_c w[c] gamma[c] pattern[c] = 0: entries come in pairs
    (c, c') with pattern[c] == pattern[c'] and w[c'] gamma[c'] = -w[c] gamma[c] (gamma = +-2^e).  A LayerNorm backward through
    such a W then has zero row means, which keeps the chained GEMM operands short.  Row r has a pair with c in the 32-wide
    stage r mod (k / 32)."""
    w = torch.zeros((n, k), dtype=torch.float64, device=device)
    pat = pattern.tolist()
    classes = {}
    for c, v in enumerate(pat):
        classes.setdefault(v, []).append(c)
    for r in range(n):
        st = r % (k // 32)
        for u in range(pairs_per_row):
            c = st * 32 + int(torch.randint(0, 32, (1,), generator=gen, device=device)) if u == 0 else \
                int(torch.randint(0, k, (1,), generator=gen, device=device))
            cl = classes[pat[c]]
            c2 = cl[int(torch.randint(0, len(cl), (1,), generator=gen, device=device))]
            if c2 == c:
                continue
            v = float(pow2((1,), elo, ehi, gen, device))
            w[r, c] += v
            w[r, c2] -= v * float(gamma[c]) / float(gamma[c2])
    return w


def paired_dy(rows, pattern, gamma, gen, device, lo=-3, hi=3):
    """dy[rows][dim] with sum_c dy[c] gamma[c] = 0 and sum_c dy[c] gamma[c] pattern[c] = 0 in every row (pairs inside the
    classes of the shared pattern)."""
    dim = pattern.numel()
    dy = torch.zeros((rows, dim), dtype=torch.float64, device=device)
    for v in pattern.unique().tolist():
        cl = (pattern == v).nonzero().flatten()
        cl = cl[torch.randperm(cl.numel(), generator=gen, device=device)]
        a, b = cl[0::2], cl[1::2]
        val = ints((rows, a.numel()), lo, hi, gen, device)
        dy[:, a] = val
        dy[:, b] = -val * gamma[a] / gamma[b]
    return dy


def winners(Nq, Nk, gen, device):
    """The key each query picks: every key at least once when Nq >= Nk (else the last Nq keys are all chosen, which includes
    the last partial tile)."""
    if Nq >= Nk:
        w = torch.cat([torch.arange(Nk, device=device), torch.randint(0, Nk, (Nq - Nk,), generator=gen, device=device)])
        return w[torch.randperm(Nq, generator=gen, device=device)]
    return torch.arange(Nk - Nq, Nk, device=device)[torch.randperm(Nq, generator=gen, device=device)]


def one_hot_attention(B, Nq, Nk, heads, dh, gen, device, scale=0.5):
    """q [B,Nq,h*dh], kv [B,Nk,2*h*dh], win [B,heads,Nq] such that the scaled scores of query i peak at key win with every
    other key at least 128 lower.  Key j carries the code (1, a, a^2, b, b^2) with (a, b) = divmod(j, 20) and query i
    lam * (-(a_w^2 + b_w^2), 2 a_w, -1, 2 b_w, -1) for its winner w: q.k = -lam ((a - a_w)^2 + (b - b_w)^2), lam = 128 / scale.
    The remaining head dimensions hold small integers, the same for every key (k) or random per query (q): they shift a
    row's scores by a constant in [-dh/2 .. dh/2] * scale, so a zero padding key (score 0) is never 128 below the winner."""
    assert dh >= 16 and Nk <= 400
    lam = 128.0 / scale
    inner = heads * dh
    win = torch.stack([torch.stack([winners(Nq, Nk, gen, device) for _ in range(heads)]) for _ in range(B)])
    q = torch.zeros((B, Nq, heads, dh), dtype=torch.float64, device=device)
    k = torch.zeros((B, Nk, heads, dh), dtype=torch.float64, device=device)
    j = torch.arange(Nk, device=device)
    a, b = (j // 20).double(), (j % 20).double()
    code = torch.stack([torch.ones_like(a), a, a * a, b, b * b], -1)
    k[:, :, :, :5] = code[None, :, None, :]
    k[:, :, :, 5:] = ints((B, 1, heads, dh - 5), -1, 1, gen, device)
    aw, bw = (win // 20).double().permute(0, 2, 1), (win % 20).double().permute(0, 2, 1)     # [B,Nq,heads]
    q[..., 0] = -lam * (aw * aw + bw * bw)
    q[..., 1] = 2 * lam * aw
    q[..., 2] = -lam
    q[..., 3] = 2 * lam * bw
    q[..., 4] = -lam
    q[..., 5:] = ints((B, Nq, heads, dh - 5), -1, 1, gen, device)
    v = ints((B, Nk, heads, dh), -8, 8, gen, device, 0.25)
    kv = torch.cat([k.reshape(B, Nk, inner), v.reshape(B, Nk, inner)], -1)
    return q.reshape(B, Nq, inner), kv, win


# ---------------------------------------------------------------------------------------------------------------
# float64 references
def gelu(x):
    """Exact-erf GELU; in saturation (|x| >= 20) the fp32 values x / -0 the kernels produce (float64 keeps x Phi(-20) ~ 1e-88
    there, which would widen the next GEMM's operand for nothing)."""
    return torch.where(x.abs() >= 20, torch.where(x > 0, x, -0.0), F.gelu(x))


def gelu_grad(x):
    g = 0.5 * (1 + torch.erf(x * 0.5 ** 0.5)) + x * torch.exp(-0.5 * x * x) * (2 * math.pi) ** -0.5
    return torch.where(x.abs() >= 20, (x > 0).to(x.dtype), g)


def linear_ref(x, w, bias=None, residual=None, act=0):
    """(y, pre) of tmf_linear_fwd."""
    pre = x @ w.T + (0 if bias is None else bias)
    y = gelu(pre) if act else pre
    return y + (0 if residual is None else residual), pre


def layernorm_ref(x, gamma, beta, eps, residual=None):
    mean = x.mean(-1)
    var = ((x - mean[..., None]) ** 2).mean(-1)
    rstd = (var + eps) ** -0.5
    y = (x - mean[..., None]) * rstd[..., None] * gamma + beta
    return y + (0 if residual is None else residual), mean, rstd


def layernorm_bwd_ref(dy, x, gamma, mean, rstd):
    """(dx, dgamma, dbeta) of LayerNorm at the given statistics."""
    xh = (x - mean[..., None]) * rstd[..., None]
    gg = dy * gamma
    dx = rstd[..., None] * (gg - gg.mean(-1, keepdim=True) - xh * (gg * xh).mean(-1, keepdim=True))
    return dx, (dy * xh).sum(0), dy.sum(0)


def _heads(t, B, N, heads, dh):
    return t.reshape(B, N, heads, dh).permute(0, 2, 1, 3)


def attention_ref(q, kv, heads, dh, scale):
    """(out [B,Nq,h*dh], lse [B,h,Nq], dots [B,h,Nq,Nk], attn [B,h,Nq,Nk])."""
    B, Nq, inner = q.shape
    Nk = kv.shape[1]
    k, v = _heads(kv[..., :inner], B, Nk, heads, dh), _heads(kv[..., inner:], B, Nk, heads, dh)
    dots = _heads(q, B, Nq, heads, dh) @ k.transpose(-1, -2) * scale
    lse = torch.logsumexp(dots, -1)
    attn = torch.exp(dots - lse[..., None])
    out = (attn @ v).permute(0, 2, 1, 3).reshape(B, Nq, inner)
    return out, lse, dots, attn


def attention_bwd_ref(dout, q, kv, heads, dh, scale):
    """(dq, dkv, dattn) of out = softmax(q k^T scale) v."""
    B, Nq, inner = q.shape
    Nk = kv.shape[1]
    out, lse, dots, attn = attention_ref(q, kv, heads, dh, scale)
    k, v = _heads(kv[..., :inner], B, Nk, heads, dh), _heads(kv[..., inner:], B, Nk, heads, dh)
    do = _heads(dout, B, Nq, heads, dh)
    dattn = do @ v.transpose(-1, -2)
    ds = attn * (dattn - (dattn * attn).sum(-1, keepdim=True))
    dq = (ds @ k * scale).permute(0, 2, 1, 3).reshape(B, Nq, inner)
    dk = (ds.transpose(-1, -2) @ _heads(q, B, Nq, heads, dh) * scale).permute(0, 2, 1, 3).reshape(B, Nk, inner)
    dv = (attn.transpose(-1, -2) @ do).permute(0, 2, 1, 3).reshape(B, Nk, inner)
    return dq, torch.cat([dk, dv], -1), dattn


def chain_fwd_ref(o, x, wo, bo, ln2_w, ln2_b, w1, b1, w2, b2, lnf_w, lnf_b, add_input, eps2=0.0, epsf=0.0):
    """dict of every tensor tmf_encoder_chain_fwd writes."""
    a = o @ wo.T + bo + x
    h2, mean2, rstd2 = layernorm_ref(a, ln2_w, ln2_b, eps2)
    pre = h2 @ w1.T + b1
    f = gelu(pre)
    g = f @ w2.T + b2 + a
    y, meanf, rstdf = layernorm_ref(g, lnf_w, lnf_b, epsf)
    if add_input:
        y = y + x
    return dict(a=a, h2=h2, mean2=mean2, rstd2=rstd2, pre=pre, f=f, g=g, meanf=meanf, rstdf=rstdf, y=y)


def chain_bwd_ref(dy, g, a, pre, wo, w1, w2, ln2_w, lnf_w, mean2, rstd2, meanf, rstdf, add_input):
    """dict of every tensor tmf_encoder_chain_bwd writes."""
    dg, dlnf_w, dlnf_b = layernorm_bwd_ref(dy, g, lnf_w, meanf, rstdf)
    dp = (dg @ w2) * gelu_grad(pre)
    dh2 = dp @ w1
    dln, dln2_w, dln2_b = layernorm_bwd_ref(dh2, a, ln2_w, mean2, rstd2)
    da = dg + dln
    return dict(dg=dg, dp=dp, da=da, dout=da @ wo, dxp=da + (dy if add_input else 0), dlnf_w=dlnf_w, dlnf_b=dlnf_b,
                dln2_w=dln2_w, dln2_b=dln2_b, dh2=dh2)


def proj_fwd_ref(x, ctx, ln_w, ln_b, wq, wkv, eps=0.0):
    h1, mean1, rstd1 = layernorm_ref(x, ln_w, ln_b, eps)
    return dict(h1=h1, mean1=mean1, rstd1=rstd1, q=h1 @ wq.T, kv=ctx @ wkv.T)


def proj_bwd_ref(dq, dkv, dxp, x, ln_w, mean1, rstd1, wq, wkv):
    dh1 = dq @ wq
    dln, dln_w, dln_b = layernorm_bwd_ref(dh1, x, ln_w, mean1, rstd1)
    return dict(dx=dxp + dln, dctx=dkv @ wkv, dln_w=dln_w, dln_b=dln_b, dh1=dh1)


def token_pool_ref(x):
    """(sum [B,C] float64, max [B,C], argmax [B,C] first maximum)."""
    mx = x.amax(1)
    idx = torch.arange(x.shape[1], device=x.device)[None, :, None]
    return x.sum(1), mx, torch.where(x == mx[:, None], idx, x.shape[1]).amin(1)

"""Exact-arithmetic references, operand generators and the shape table of the MiSePyNet / Mnet kernel tests
(tests/test_gpu_mnet_exact.py), in the manner of tests/conv_exact.py and tests/bn_exact.py.

Operands are small integers (the convolutions and the pool) or short dyadic significands (BatchNorm + ReLU): every
product and every partial sum is exact in fp32 as long as the sum of the absolute values of all terms of a reduction
stays below 2^24 quanta, so whatever the thread split, chunking or summation order, a correct kernel reproduces the
float64 reference below bit for bit.  The bound is asserted on the actual operands of every case with the term count
of the whole reduction (N*P*Lo for the slice weight gradient, N*Xo*Yo for the spatial one, N*S for the BatchNorm
sums), not the kernels' current fp32 chunk lengths.

References work on float64 tensors in the layouts the kernels use (csrc/mnet_ops.cu):
  * slice convolution: x [N][Cin][P][L], w [8][Cin][k], y [N][8][P][Lo], Lo = L - k + 1;
  * spatial convolution: x [N][Cin][X][Y], w [Cout][Cin][kh][kw], stride s, no padding, floor output size;
  * BatchNorm + ReLU on [N][C][S] with coef [4, C] = (scale, shift, mean, invstd) (tmf_bn_finalize's coef[4C]) and
    bcoef [2, C] = (mean(dz), mean(dz*xhat)) (tmf_bn_bwd_finalize's bcoef[2C]; zero in eval mode);
  * max pool over (ph, pw) windows of [NC][X][Y], stride = kernel, floor mode: the gradient goes to the first maximum
    in (a, b) scan order, idx is the window-local a*pw + b, voxels outside complete windows get 0.
"""
import math

import torch

from tests import bn_exact as N
from tests import conv_exact as X

LC_CO = 8                     # output channels of every slice convolution


# ---------------------------------------------------------------------------------------------------------------
# float64 references
def line_fwd_ref(x, w, b):
    """y[n,co,p,o] = b[co] + sum_ci sum_t x[n,ci,p,o+t] w[co,ci,t]."""
    k = w.shape[-1]
    Lo = x.shape[-1] - k + 1
    y = b.view(1, -1, 1, 1).expand(x.shape[0], w.shape[0], x.shape[2], Lo).clone()
    for t in range(k):
        y += torch.einsum("ncpo,dc->ndpo", x[..., t:t + Lo], w[:, :, t])
    return y


def line_dgrad_ref(dy, w, L):
    """dx[n,ci,p,i] = sum_co sum_t dy[n,co,p,i-t] w[co,ci,t] over 0 <= i - t < Lo."""
    k = w.shape[-1]
    Lo = L - k + 1
    dx = torch.zeros((dy.shape[0], w.shape[1], dy.shape[2], L), dtype=dy.dtype, device=dy.device)
    for t in range(k):
        dx[..., t:t + Lo] += torch.einsum("ndpo,dc->ncpo", dy, w[:, :, t])
    return dx


def line_wgrad_ref(dy, x, k):
    """(dw [8][Cin][k], db [8]): dw[co,ci,t] = sum_{n,p,o} dy[n,co,p,o] x[n,ci,p,o+t], db[co] = sum dy[:,co]."""
    Lo = x.shape[-1] - k + 1
    dw = torch.stack([torch.einsum("ndpo,ncpo->dc", dy, x[..., t:t + Lo]) for t in range(k)], -1)
    return dw, dy.sum((0, 2, 3))


def _taps(t, i, j, s, Xo, Yo):
    """The input rows / columns tap (i, j) of every output position reads: t[..., i + s*ox, j + s*oy]."""
    return t[:, :, i:i + s * (Xo - 1) + 1:s, j:j + s * (Yo - 1) + 1:s]


def conv2d_out(X_, Y_, kh, kw, s):
    return (X_ - kh) // s + 1, (Y_ - kw) // s + 1


def conv2d_fwd_ref(x, w, b, s):
    kh, kw = w.shape[2:]
    Xo, Yo = conv2d_out(x.shape[2], x.shape[3], kh, kw, s)
    y = b.view(1, -1, 1, 1).expand(x.shape[0], w.shape[0], Xo, Yo).clone()
    for i in range(kh):
        for j in range(kw):
            y += torch.einsum("ncxy,dc->ndxy", _taps(x, i, j, s, Xo, Yo), w[:, :, i, j])
    return y


def conv2d_dgrad_ref(dy, w, s, X_, Y_):
    """Rows / columns no window covers (stride > kernel, or the floor of the output size) get 0."""
    kh, kw = w.shape[2:]
    Xo, Yo = dy.shape[2:]
    dx = torch.zeros((dy.shape[0], w.shape[1], X_, Y_), dtype=dy.dtype, device=dy.device)
    for i in range(kh):
        for j in range(kw):
            _taps(dx, i, j, s, Xo, Yo).add_(torch.einsum("ndxy,dc->ncxy", dy, w[:, :, i, j]))
    return dx


def conv2d_wgrad_ref(dy, x, kh, kw, s):
    Xo, Yo = dy.shape[2:]
    dw = torch.empty((dy.shape[1], x.shape[1], kh, kw), dtype=dy.dtype, device=dy.device)
    for i in range(kh):
        for j in range(kw):
            dw[:, :, i, j] = torch.einsum("ndxy,ncxy->dc", dy, _taps(x, i, j, s, Xo, Yo))
    return dw, dy.sum((0, 2, 3))


def bn_stats_ref(x):
    """Per-channel (sum, sum of squares) of x [N][C][S]."""
    return x.sum((0, 2)), (x * x).sum((0, 2))


def bn_relu_fwd_ref(x, coef):
    return torch.clamp_min(x * coef[0].view(1, -1, 1) + coef[1].view(1, -1, 1), 0.0)


def bn_dz_xhat(dout, x, coef):
    """dz = dout * [x*scale + shift > 0], xhat = (x - mean) * invstd."""
    sc, sh, mu, inv = (c.view(1, -1, 1) for c in coef)
    dz = torch.where(x * sc + sh > 0, dout, torch.zeros_like(dout))
    return dz, (x - mu) * inv


def bn_bwd_sums_ref(dout, x, coef):
    """(sum dz, sum dz*xhat, sum |dz|, sum |dz*xhat|) per channel."""
    dz, xh = bn_dz_xhat(dout, x, coef)
    t2 = dz * xh
    return dz.sum((0, 2)), t2.sum((0, 2)), dz.abs().sum((0, 2)), t2.abs().sum((0, 2))


def bn_apply_ref(dout, x, coef, bcoef):
    """dx = scale * (dz - m1 - xhat * m2)."""
    dz, xh = bn_dz_xhat(dout, x, coef)
    return coef[0].view(1, -1, 1) * (dz - bcoef[0].view(1, -1, 1) - xh * bcoef[1].view(1, -1, 1))


def pool_windows(x, ph, pw):
    """[NC][X][Y] -> [NC][Xo][Yo][ph*pw] over the complete windows, position a*pw + b."""
    NC, X_, Y_ = x.shape
    Xo, Yo = X_ // ph, Y_ // pw
    return (x[:, :Xo * ph, :Yo * pw].reshape(NC, Xo, ph, Yo, pw).permute(0, 1, 3, 2, 4).reshape(NC, Xo, Yo, ph * pw))


def maxpool_fwd_ref(x, ph, pw):
    """(y, idx): the window maximum and the first position holding it (the smallest index among the maxima, on any
    device; a window of -inf only has idx 0)."""
    win = pool_windows(x, ph, pw)
    y = win.amax(-1)
    pos = torch.arange(ph * pw, device=x.device).expand_as(win)
    idx = torch.where(win == y.unsqueeze(-1), pos, ph * pw).amin(-1)
    return y, idx


def maxpool_bwd_ref(dy, idx, ph, pw, X_, Y_):
    NC, Xo, Yo = dy.shape
    routed = torch.zeros((NC, Xo, Yo, ph * pw), dtype=dy.dtype, device=dy.device).scatter_(-1, idx.unsqueeze(-1),
                                                                                          dy.unsqueeze(-1))
    dx = torch.zeros((NC, X_, Y_), dtype=dy.dtype, device=dy.device)
    dx[:, :Xo * ph, :Yo * pw] = routed.reshape(NC, Xo, Yo, ph, pw).permute(0, 1, 3, 2, 4).reshape(NC, Xo * ph, Yo * pw)
    return dx


# ---------------------------------------------------------------------------------------------------------------
# launch geometry of csrc/mnet_ops.cu, which nothing exports: this mirror must follow grid_for, tmf_line_conv_wgrad
# and tmf_nchw_bn_stats / tmf_nchw_bn_relu_bwd_reduce there
THREADS = 256
GRID_CAP = 148 * 16                  # grid_for's block cap: element-wise kernels loop over the rest
LINE_WGRAD_BLOCKS = 592              # at most this many partial rows in the slice weight gradient
LINE_WGRAD_MAX_PER_THREAD = 16       # weights a thread of the slice weight gradient owns at most
STAT_ROWS = 296                      # TMF_STAT_ROWS
STAT_ELEMS_PER_ROW = 256 * 8         # the statistics kernels start one row per 2048 elements of a channel
SMEM_LIMIT = 48 * 1024               # dynamic shared memory the slice kernels may ask for


def grid_for(total):
    return max(1, min(GRID_CAP, -(-total // THREADS)))


def grid_strides(total):
    """True when an element-wise kernel's threads take more than one element (its grid hit the cap)."""
    return total > grid_for(total) * THREADS


def line_wgrad_blocks(lines):
    return min(lines, LINE_WGRAD_BLOCKS)


def line_wgrad_per_thread(cin, k):
    return -(-LC_CO * cin * k // THREADS)


def line_wgrad_smem(cin, L, k):
    return 4 * (LC_CO * (L - k + 1) + cin * L)


def stat_rows(count):
    return max(1, min(STAT_ROWS, -(-count // STAT_ELEMS_PER_ROW)))


# ---------------------------------------------------------------------------------------------------------------
# operand generators (each asserts the exactness bound on the operands it returns)
def line_operands(case, gen, device):
    """x, w, dy integers in [-2, 2], b in [-4, 4]."""
    _, n, cin, P, L, k = case
    Lo = L - k + 1
    x = X.ints((n, cin, P, L), -2, 2, gen, device)
    w = X.ints((LC_CO, cin, k), -2, 2, gen, device)
    b = X.ints((LC_CO,), -4, 4, gen, device)
    dy = X.ints((n, LC_CO, P, Lo), -2, 2, gen, device)
    ax, aw, ady = (float(t.abs().max()) for t in (x, w, dy))
    X.exact_bound(cin * k, ax, aw, 1, extra=float(b.abs().max()))     # forward
    X.exact_bound(LC_CO * k, ady, aw, 1)                              # dgrad
    X.exact_bound(n * P * Lo, ady, max(ax, 1.0), 1)                   # dw and db: every (n, p, o)
    return x, w, b, dy


def conv2d_operands(case, gen, device):
    """x, w, dy integers in [-2, 2], b in [-4, 4]."""
    _, n, cin, cout, X_, Y_, kh, kw, s = case
    Xo, Yo = conv2d_out(X_, Y_, kh, kw, s)
    x = X.ints((n, cin, X_, Y_), -2, 2, gen, device)
    w = X.ints((cout, cin, kh, kw), -2, 2, gen, device)
    b = X.ints((cout,), -4, 4, gen, device)
    dy = X.ints((n, cout, Xo, Yo), -2, 2, gen, device)
    ax, aw, ady = (float(t.abs().max()) for t in (x, w, dy))
    X.exact_bound(cin * kh * kw, ax, aw, 1, extra=float(b.abs().max()))
    X.exact_bound(cout * -(-kh // s) * -(-kw // s), ady, aw, 1)
    X.exact_bound(n * Xo * Yo, ady, max(ax, 1.0), 1)
    return x, w, b, dy


Q_X = 2.0 ** -1               # grid of the BatchNorm inputs and means


def bn_operands(case, gen, device):
    """x = j/2 with |j| <= 3, mean = o/2 with |o| <= 2, scale / shift / invstd from bn_exact.coefs (scale s/4 with channel
    0 negative and channel 1 zero, shift h/8, invstd 2^e, e in {-1, 0, 1}), bcoef = multiples of 1/8 in [-7/8, 7/8]
    and dout integers in [-1, 1].  bn_exact's finer inputs (y = centre + j/16) would overflow 2^24 quanta in the sums of
    squares of the slice layers (N*S up to 1.2e6): this grid keeps x^2 on a 1/4 grid below 9/4.  Every element-wise
    value (x*scale + shift, xhat, dz*xhat, dx) is then a multiple of at least 2^-7 below 2^4, exact in fp32 under any
    contraction; the whole-layer sums are bounded here on the actual operands."""
    _, n, C, S = case
    coef, _ = N.coefs(C, gen, device)
    coef[2] = X.ints((C,), -2, 2, gen, device) * Q_X
    x = X.ints((n, C, S), -3, 3, gen, device) * Q_X
    dout = X.ints((n, C, S), -1, 1, gen, device)
    bcoef = N.bcoefs(C, gen, device)
    s1, s2 = bn_stats_ref(x.abs())[0], bn_stats_ref(x)[1]
    X.exact_bound(1, float(s1.max()), 1, Q_X)                         # sum x: quanta of 1/2
    X.exact_bound(1, float(s2.max()), 1, Q_X * Q_X)                   # sum x^2: quanta of 1/4
    _, _, a1, a2 = bn_bwd_sums_ref(dout, x, coef)
    X.exact_bound(1, float(a1.max()), 1, 1)                           # sum dz: integers
    X.exact_bound(1, float((a2 / coef[3]).max()), 1, Q_X)             # sum dz*xhat: quanta of invstd / 2
    sc, sh, m = 7 * N.Q_SC, 31 * N.Q_SH, 7 * N.Q_M
    xa, xh = 3 * Q_X, (3 + 2) * Q_X * 2.0 ** max(N.IS_EXP)
    X.exact_bound(1, xa * sc + sh, 1, Q_X * N.Q_SC)                   # x*scale + shift
    X.exact_bound(1, sc * (1 + m + xh * m), 1, N.Q_SC * Q_X * 2.0 ** min(N.IS_EXP) * N.Q_M)   # dx
    return x, coef, bcoef, dout


def pool_operands(case, gen, device):
    """x integers in [-1, 1] (ties in nearly every window), with -inf at a quarter of the positions and in whole
    windows when the case asks for it; dy integers in [1, 8] (every routed gradient is visible)."""
    _, NC, X_, Y_, ph, pw, ninf = case
    x = X.ints((NC, X_, Y_), -1, 1, gen, device)
    if ninf:
        x[torch.rand(x.shape, generator=gen, device=device) < 0.25] = -math.inf
        x[0, :ph, :pw] = -math.inf                     # a window of -inf only
        x[-1, -ph:, -pw:] = -math.inf                  # and one at the end of the pooled area (or past it)
    dy = X.ints((NC, X_ // ph, Y_ // pw), 1, 8, gen, device)
    return x, dy


# ---------------------------------------------------------------------------------------------------------------
# shape table, B = 2 at 91 x 109 x 91 (every case passes the exactness bound at that batch)
B = 2
VIEWS = {"axial": (91 * 109, 91), "coronal": (91 * 91, 109)}         # (P, L): the sagittal view has the axial shapes
SPATIAL = {"axial": (91, 109), "coronal": (91, 91)}                   # (X, Y) of the slice-stack outputs


def slice_layers(dim):
    """(Cin, L, k) of the six slice convolutions of slice_cnn(dim) (models/MiSePyNet.py): the conv1, conv2, conv3
    stacks, each collapsing the last axis."""
    k2, k3 = (dim + 1) // 2, (dim + 2) // 3
    return [(1, dim, dim), (1, dim, k2), (8, dim - k2 + 1, k2), (1, dim, k3), (8, dim - k3 + 1, k3),
            (8, dim - 2 * (k3 - 1), k3)]


def spatial_layers(X_, Y_):
    """conv / pool shapes of spatial_cnn.conv1 on (N, 8, X, Y): [(Cin, Cout, X, Y, kh, kw, s)], [(C, X, Y, ph, pw)]."""
    convs, pools = [], []
    for cin, cout, kk, s, pool in ((8, 16, 11, 2, 3), (16, 32, 11, 1, 3), (32, 64, 1, 1, None)):
        convs.append((cin, cout, X_, Y_, kk, kk, s))
        X_, Y_ = conv2d_out(X_, Y_, kk, kk, s)
        if pool:
            pools.append((cout, X_, Y_, pool, pool))
            X_, Y_ = X_ // pool, Y_ // pool
    return convs, pools


def _model_cases():
    line, conv, bn, pool = [], [], [], []
    for view, (P, dim) in VIEWS.items():
        for cin, L, k in slice_layers(dim):
            line.append((f"{view}-{cin}x{L}k{k}", B, cin, P, L, k))
            bn.append((f"{view}-slice-{cin}x{L}k{k}", B, LC_CO, P * (L - k + 1)))
        convs, pools = spatial_layers(*SPATIAL[view])
        for cin, cout, X_, Y_, kh, kw, s in convs:
            conv.append((f"{view}-{cin}to{cout}", B, cin, cout, X_, Y_, kh, kw, s))
            Xo, Yo = conv2d_out(X_, Y_, kh, kw, s)
            bn.append((f"{view}-{cin}to{cout}", B, cout, Xo * Yo))
        for C, X_, Y_, ph, pw in pools:
            pool.append((f"{view}-pool{C}", B * C, X_, Y_, ph, pw, False))
    seen, bn_u = set(), []
    for c in bn:                                       # the BatchNorm layers repeat (C, S): keep one of each
        if c[2:] not in seen:
            seen.add(c[2:])
            bn_u.append(c)
    return line, conv, bn_u, pool


LINE_MODEL, CONV_MODEL, BN_MODEL, POOL_MODEL = _model_cases()

# edge cases: each is the only case of its table that reaches the regimes it names (test_mnet_exact_host checks both)
# slice convolution: (id, N, Cin, P, L, k)
LINE_EDGE = [
    ("one-line", 1, 3, 1, 20, 5),            # lines = 1 (one wgrad block), odd Cin
    ("k1", 2, 1, 100, 7, 1),                 # k = 1 (Lo = L), 200 lines, 8 weights: idle wgrad threads
    ("w16-smem48k", 1, 8, 1000, 799, 64),    # 4096 weights (16 per thread), 48 KB staged in the wgrad, 1000 lines
]
# spatial convolution: (id, N, Cin, Cout, X, Y, kh, kw, s)
CONV_EDGE = [
    ("s2-dead-row", 2, 3, 5, 12, 15, 3, 4, 2),       # (X - kh), (Y - kw) odd: the last row / column feeds no output
    ("s3-gaps", 1, 2, 3, 11, 8, 2, 2, 3),            # stride 3 > kh = 2: rows between the windows; N*Xo*Yo = 12
    ("c1", 3, 1, 1, 9, 10, 3, 5, 1),                 # Cin = Cout = 1, kh != kw
    ("1x1-s2", 2, 6, 7, 9, 8, 1, 1, 2),              # 1x1 with stride 2
    ("grid-stride", 2, 4, 4, 310, 300, 3, 2, 1),     # fwd and dgrad past grid_for's cap
]
# BatchNorm + ReLU: (id, N, C, S)
BN_EDGE = [
    ("c1", 3, 1, 777),                       # C = 1, two statistics rows
]
# max pool: (id, NC, X, Y, ph, pw, -inf)
POOL_EDGE = [
    ("2x3-ninf", 5, 9, 9, 2, 3, True),       # ph != pw, -inf in windows (some all -inf), a leftover row
    ("15x17", 3, 31, 35, 15, 17, False),     # ph * pw = 255, the largest index a byte holds; leftover row and column
    ("grid-stride", 8, 601, 602, 2, 2, False),
]

LINE_CASES = LINE_MODEL + [("edge-" + c[0],) + c[1:] for c in LINE_EDGE]
CONV_CASES = CONV_MODEL + [("edge-" + c[0],) + c[1:] for c in CONV_EDGE]
BN_CASES = BN_MODEL + [("edge-" + c[0],) + c[1:] for c in BN_EDGE]
POOL_CASES = POOL_MODEL + [("edge-" + c[0],) + c[1:] for c in POOL_EDGE]


# ---------------------------------------------------------------------------------------------------------------
# the regimes a case reaches, through the geometry mirror
def line_regimes(case):
    _, n, cin, P, L, k = case
    lines, Lo = n * P, L - k + 1
    r = set()
    if lines < LINE_WGRAD_BLOCKS:
        r.add("line: lines < 592")
    if lines == 1:
        r.add("line: lines = 1")
    if lines > LINE_WGRAD_BLOCKS and lines % LINE_WGRAD_BLOCKS:
        r.add("line: lines > 592, lines % 592 != 0")
    if k == 1:
        r.add("line: k = 1")
    if k == L:
        r.add("line: k = L")
    if line_wgrad_per_thread(cin, k) == LINE_WGRAD_MAX_PER_THREAD:
        r.add("line: 16 weights per thread")
    if LC_CO * cin * k < THREADS:
        r.add("line: idle wgrad threads")
    if cin % 2 and cin > 1:
        r.add("line: odd Cin > 1")
    if line_wgrad_smem(cin, L, k) > SMEM_LIMIT - 1024:
        r.add("line: wgrad stages within 1 KB of 48 KB")
    for name, total in (("line fwd", n * P * Lo), ("line dgrad", n * cin * P * L)):
        r.add(f"{name}: {'grid-stride' if grid_strides(total) else 'one pass'}")
    return r


def conv_regimes(case):
    _, n, cin, cout, X_, Y_, kh, kw, s = case
    Xo, Yo = conv2d_out(X_, Y_, kh, kw, s)
    r = set()
    if s == 2 and (X_ - kh) % 2:
        r.add("conv: stride 2, last row feeds no output")
    if kh > 1 and s > kh:
        r.add("conv: stride > kh > 1")
    if kh != kw and X_ != Y_:
        r.add("conv: kh != kw, X != Y")
    if cin == cout == 1:
        r.add("conv: Cin = Cout = 1")
    if kh == kw == 1 and s == 2:
        r.add("conv: 1x1 stride 2")
    npos = n * Xo * Yo
    if npos < 32:
        r.add("conv: N*Xo*Yo < 32")
    elif npos % 32:
        r.add("conv: N*Xo*Yo > 32, not a multiple of 32")
    for name, total in (("conv fwd", n * cout * Xo * Yo), ("conv dgrad", n * cin * X_ * Y_)):
        r.add(f"{name}: {'grid-stride' if grid_strides(total) else 'one pass'}")
    return r


def bn_regimes(case):
    _, n, C, S = case
    rows = stat_rows(n * S)
    r = set()
    if n * S < THREADS:
        r.add("bn: N*S < 256")
    if 1 < rows < STAT_ROWS:
        r.add("bn: 1 < rows < 296")
    if rows == STAT_ROWS and n * S > STAT_ROWS * THREADS:
        r.add("bn: 296 rows, threads loop")
    if C == 1:
        r.add("bn: C = 1")
    if S == 1:
        r.add("bn: S = 1")
    r.add(f"bn fwd and apply: {'grid-stride' if grid_strides(n * C * S) else 'one pass'}")
    return r


def pool_regimes(case):
    _, NC, X_, Y_, ph, pw, ninf = case
    r = {"pool: ties"}                                  # every pool case: integers in [-1, 1]
    if ninf:
        r.add("pool: -inf")
    if X_ % ph and Y_ % pw:
        r.add("pool: leftover rows and columns")
    if ph != pw:
        r.add("pool: ph != pw")
    if ph * pw == 255:
        r.add("pool: ph*pw = 255")
    for name, total in (("pool fwd", NC * (X_ // ph) * (Y_ // pw)), ("pool bwd", NC * X_ * Y_)):
        r.add(f"{name}: {'grid-stride' if grid_strides(total) else 'one pass'}")
    return r


REGIMES = {   # every regime the GPU table must reach
    "line": {"line: lines < 592", "line: lines = 1", "line: lines > 592, lines % 592 != 0", "line: k = 1", "line: k = L",
             "line: 16 weights per thread", "line: idle wgrad threads", "line: odd Cin > 1",
             "line: wgrad stages within 1 KB of 48 KB", "line fwd: grid-stride", "line fwd: one pass",
             "line dgrad: grid-stride", "line dgrad: one pass"},
    "conv": {"conv: stride 2, last row feeds no output", "conv: stride > kh > 1", "conv: kh != kw, X != Y",
             "conv: Cin = Cout = 1", "conv: 1x1 stride 2", "conv: N*Xo*Yo < 32", "conv: N*Xo*Yo > 32, not a multiple of 32",
             "conv fwd: grid-stride", "conv fwd: one pass", "conv dgrad: grid-stride", "conv dgrad: one pass"},
    "bn": {"bn: N*S < 256", "bn: 1 < rows < 296", "bn: 296 rows, threads loop", "bn: C = 1", "bn: S = 1",
           "bn fwd and apply: grid-stride", "bn fwd and apply: one pass"},
    "pool": {"pool: ties", "pool: -inf", "pool: leftover rows and columns", "pool: ph != pw", "pool: ph*pw = 255",
             "pool fwd: grid-stride", "pool fwd: one pass", "pool bwd: grid-stride", "pool bwd: one pass"},
}
TABLES = {"line": (LINE_CASES, line_regimes), "conv": (CONV_CASES, conv_regimes), "bn": (BN_CASES, bn_regimes),
          "pool": (POOL_CASES, pool_regimes)}

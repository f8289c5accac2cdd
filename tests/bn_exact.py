"""Exact-arithmetic references and operand generators for the sNet BatchNorm / LeakyReLU / pooling tests
(tests/test_gpu_bn_exact.py), in the manner of tests/conv_exact.py.

Operands sit on dyadic grids with short significands: y = m + j/16 (at most 7 significant bits), scale s/4, shift h/8,
mean m + o/16, invstd a power of two, mean(dz) and mean(dz*xhat) multiples of 1/8, a LeakyReLU slope of 1/2 and small
integer gradients.  Every element-wise value the kernels form (z, the activation, the 8-term average, xhat, dz, the
folded coefficients A and Bc, dy before rounding) is then a multiple of a known quantum far below 2^24 quanta, hence
exact in fp32 whatever FMA contraction the compiler applies; bf16 outputs must equal one round-to-nearest-even of the
float64 reference, fp32 outputs must equal it.  The per-channel backward sums (sum dz, sum dz*xhat) are exact when the
sum of |term| over the whole tower stays below 2^24 quanta of that channel (checked on the actual operands), so every
thread split and every summation order gives the reference's value bit for bit.

The max-pool rule is the one every kernel implements: the gradient of a 2x2x2 window goes to the first position in
(d,h,w) scan order that maximises sign(scale) * y (position 0 when the scale is 0).  With slope >= 0 that position holds
the window's maximum activation; in exact arithmetic with slope > 0 it is torch's first maximum of the activation.

References work on NDHWC float64 tensors on whatever device the inputs live.  Coefficients are float64 [4, C] = (scale,
shift, mean, invstd) and [2, C] = (mean(dz), mean(dz*xhat)), the layouts of tmf_bn_finalize's coef and
tmf_bn_bwd_finalize's bcoef.
"""
from fractions import Fraction
import math

import numpy as np
import torch

from tests import conv_exact as X

POOL_NONE, POOL_MAX, POOL_AVG = 0, 1, 2
SLOPE = 0.5                   # dyadic LeakyReLU slope of the exact cases (a kernel argument; the model uses 0.01)
Q_Y, Q_SC, Q_SH, Q_M = 2.0 ** -4, 2.0 ** -2, 2.0 ** -3, 2.0 ** -3
IS_EXP = (-1, 0, 1)           # invstd = 2^e


# ---------------------------------------------------------------------------------------------------------------
# pooling windows
def windows(t):
    """[B,D,H,W,C] -> [B,Do,Ho,Wo,C,8] over the complete 2x2x2 windows (floor mode), q = 4*dd + 2*dh + dw."""
    B, D, H, W, C = t.shape
    Do, Ho, Wo = D // 2, H // 2, W // 2
    return (t[:, :2 * Do, :2 * Ho, :2 * Wo].reshape(B, Do, 2, Ho, 2, Wo, 2, C)
            .permute(0, 1, 3, 5, 7, 2, 4, 6).reshape(B, Do, Ho, Wo, C, 8))


def unwindow(w, shape):
    """Inverse of windows(): [B,Do,Ho,Wo,C,8] -> [B,D,H,W,C] with zeros outside the complete windows."""
    B, Do, Ho, Wo, C, _ = w.shape
    out = torch.zeros(shape, dtype=w.dtype, device=w.device)
    out[:, :2 * Do, :2 * Ho, :2 * Wo] = (w.reshape(B, Do, Ho, Wo, C, 2, 2, 2).permute(0, 1, 5, 2, 6, 3, 7, 4)
                                         .reshape(B, 2 * Do, 2 * Ho, 2 * Wo, C))
    return out


def route_index(y, sc):
    """[B,Do,Ho,Wo,C,1]: the window position the max-pool gradient goes to, the first maximum of sign(scale) * y
    (argmax returns the first maximal index; + 0.0 makes every zero key +0)."""
    key = windows(y) * torch.sign(sc)[:, None] + 0.0
    return key.argmax(-1, keepdim=True)


def leaky(z, slope):
    return torch.where(z > 0, z, z * slope)


def dleaky(z, g, slope):
    return torch.where(z > 0, g, g * slope)


# ---------------------------------------------------------------------------------------------------------------
# float64 references
def fwd_ref(y, coef, pool, slope):
    """(out, ymax): pool(leaky(y * scale + shift)); ymax (max pool only) = y at the routed position, which holds the
    window's maximum activation (asserted: the rule and the activations agree)."""
    sc, sh = coef[0], coef[1]
    a = leaky(y * sc + sh, slope)
    if pool == POOL_NONE:
        return a, None
    aw = windows(a)
    if pool == POOL_AVG:
        return aw.sum(-1) / 8, None
    idx = route_index(y, sc)
    out = aw.amax(-1)
    assert torch.equal(aw.gather(-1, idx)[..., 0], out), "the routed position does not hold the window maximum"
    return out, windows(y).gather(-1, idx)[..., 0]


def dz_ref(y, coef, dout, pool, slope):
    """dz = unpool(dout) * leaky'(z) at full resolution: zero at every max-pool position that is not routed to and at
    voxels outside complete windows."""
    sc, sh = coef[0], coef[1]
    if pool == POOL_NONE:
        return dleaky(y * sc + sh, dout, slope)
    if pool == POOL_AVG:
        g = unwindow((dout / 8).unsqueeze(-1).expand(*dout.shape, 8), y.shape)
        return dleaky(y * sc + sh, g, slope)
    idx = route_index(y, sc)
    ywin = windows(y).gather(-1, idx)[..., 0]
    dzw = dleaky(ywin * sc + sh, dout, slope)
    return unwindow(torch.zeros((*dout.shape, 8), dtype=y.dtype, device=y.device).scatter_(-1, idx, dzw.unsqueeze(-1)),
                    y.shape)


def sums_ref(y, coef, dout, pool, slope):
    """(s1, s2, a1, a2) per channel: s1 = sum dz, s2 = sum dz * xhat with xhat = (y - mean) * invstd, and the sums of
    their absolute values (for the exactness bound).  A max pool is evaluated at pooled resolution (one term per
    window, as the kernels see it)."""
    sc, sh, mu, inv = coef
    if pool == POOL_MAX:
        ywin = windows(y).gather(-1, route_index(y, sc))[..., 0]
        dz = dleaky(ywin * sc + sh, dout, slope)
        yy = ywin
    else:
        dz = dz_ref(y, coef, dout, pool, slope)
        yy = y
    t2 = dz * ((yy - mu) * inv)
    C = y.shape[-1]
    dz, t2 = dz.reshape(-1, C), t2.reshape(-1, C)
    return dz.sum(0), t2.sum(0), dz.abs().sum(0), t2.abs().sum(0)


def apply_ref(y, coef, bcoef, dout, pool, slope):
    """dy = scale * (dz - mean(dz) - xhat * mean(dz*xhat)) for every voxel (A + Bc*y outside complete windows)."""
    sc, _, mu, inv = coef
    m1, m2 = bcoef
    return sc * (dz_ref(y, coef, dout, pool, slope) - m1 - (y - mu) * inv * m2)


def bwd_finalize_ref(s1, s2, sc, count, training):
    """tmf_bn_bwd_finalize bit for bit, from float64 totals (numpy, CPU): dgamma = f32(s2), dbeta = f32(s1); training:
    bcoef = f32(s / count) (one double division), dbias = 0; eval: bcoef = 0, dbias = f32(scale * f32(s1))."""
    s1, s2, sc = (np.asarray(v, dtype=np.float64) for v in (s1, s2, sc))
    f32 = np.float32
    out = {"dgamma": s2.astype(f32), "dbeta": s1.astype(f32)}
    if training:
        out["bcoef"] = np.concatenate([(s1 / count).astype(f32), (s2 / count).astype(f32)])
        out["dbias"] = np.zeros_like(out["dbeta"])
    else:
        out["bcoef"] = np.zeros(2 * len(s1), dtype=f32)
        out["dbias"] = sc.astype(f32) * s1.astype(f32)          # one fp32 product: correctly rounded in numpy too
    return out


U32 = 2.0 ** -24              # unit roundoff of fp32


def finalize_ref(t1, t2, gamma, beta, rmean, rvar, count, momentum, eps, training):
    """tmf_bn_finalize from the float64 row totals (numpy, CPU): the expected values and absolute error bounds.

    mean = f32(t1 / count) exactly; var = f32(t2/count - mean^2) within 1 ulp (the kernel's double expression may be
    contracted); invstd within 2 ulp of 1/sqrt(f32(var + eps)) (rsqrtf) plus what the var ulp and the fp32 add move it;
    scale = gamma * invstd and shift = beta - mean * scale one fp32 rounding each on top of their operands' errors;
    running stats (1 - m) * r + m * v within three fp32 roundings of the magnitude sum (two products and the add)."""
    f32, f64 = np.float32, np.float64
    g, b = gamma.astype(f64), beta.astype(f64)
    out, tol = {}, {}
    if training:
        m = t1 / count
        v = np.maximum(t2 / count - m * m, 0.0)
        mean, var = m.astype(f32).astype(f64), v.astype(f32).astype(f64)
        tol_var = np.spacing(var.astype(f32)).astype(f64)
        one_m = f64(f32(1.0) - f32(momentum))
        mom = f64(f32(momentum))
        unb = (v * count / (count - 1.0) if count > 1 else v).astype(f32).astype(f64)
        for name, r, new in (("rmean", rmean, mean), ("rvar", rvar, unb)):
            r = r.astype(f64)
            out[name] = one_m * r + mom * new
            # rvar: the unbiased variance's fp32 rounding may fall either side when the double expression is contracted
            extra = mom * np.spacing(unb.astype(f32)).astype(f64) if name == "rvar" else 0.0
            tol[name] = 3 * U32 * (np.abs(one_m * r) + np.abs(mom * new)) + extra
    else:
        mean, var = rmean.astype(f64), rvar.astype(f64)
        tol_var = np.zeros_like(var)
        out["rmean"], out["rvar"] = mean, var
        tol["rmean"] = tol["rvar"] = np.zeros_like(var)
    ve = (var.astype(f32) + f32(eps)).astype(f64)                  # the kernel's fp32 add
    inv = 1.0 / np.sqrt(ve)
    tol_inv = 2 * np.spacing(inv.astype(f32)).astype(f64) + inv * (0.5 * tol_var / ve + U32)
    scale = g * inv
    tol_scale = np.abs(g) * tol_inv + U32 * np.abs(scale) * 2
    shift = b - mean * scale
    tol_shift = np.abs(mean) * tol_scale + 2 * U32 * (np.abs(b) + np.abs(mean * scale)) * 2
    out.update(scale=scale, shift=shift, mean=mean, invstd=inv)
    tol.update(scale=tol_scale, shift=tol_shift, mean=np.zeros_like(mean), invstd=tol_inv)
    return out, tol


# ---------------------------------------------------------------------------------------------------------------
# fp32 fused multiply-add, emulated exactly (for the tie-collapse example)
def f32_round(x):
    """Round an exact rational to the nearest fp32 (ties to even); normal range only."""
    x = Fraction(x)
    if x == 0:
        return Fraction(0)
    e = math.floor(math.log2(abs(x)))
    while abs(x) >= Fraction(2) ** (e + 1):
        e += 1
    while abs(x) < Fraction(2) ** e:
        e -= 1
    assert -126 <= e <= 127, "outside the normal fp32 range"
    ulp = Fraction(2) ** (e - 23)
    return round(x / ulp) * ulp                    # Fraction.__round__ rounds half to even


def fmaf(a, b, c):
    """fmaf(a, b, c) of fp32 operands: one rounding of the exact a*b + c."""
    for v in (a, b, c):
        assert float(np.float32(v)) == v, "fmaf operands must be fp32 values"
    return f32_round(Fraction(a) * Fraction(b) + Fraction(c))


# the collapse example: distinct bf16 y whose activations round to one fp32 value when |shift| >> |scale * y|
COLLAPSE_SCALE, COLLAPSE_SHIFT, COLLAPSE_Y = 2.0 ** -20, 1.0, (1.0, 1.0078125)


# ---------------------------------------------------------------------------------------------------------------
# operand generators
def coefs(C, gen, device):
    """(scale, shift, mean, invstd) [4, C] float64 and a per-channel centre m: scale = s/4 with |s| <= 7 (channel 0
    negative, channel 1 zero, the rest random with both signs and zeros), shift = h/8 with |h| <= 31, mean = m + o/16
    with m = k/4 (|k| <= 16) and |o| <= 2, invstd = 2^e with e in {-1, 0, 1}."""
    s = X.ints((C,), -7, 7, gen, device)
    s[0] = -float(torch.randint(1, 8, (1,), generator=gen, device=device))
    if C > 1:
        s[1] = 0.0
    h = X.ints((C,), -31, 31, gen, device)
    k = X.ints((C,), -16, 16, gen, device)
    o = X.ints((C,), -2, 2, gen, device)
    e = torch.tensor(IS_EXP, dtype=torch.float64, device=device)[
        torch.randint(0, len(IS_EXP), (C,), generator=gen, device=device)]
    m = k * 2.0 ** -2
    coef = torch.stack([s * Q_SC, h * Q_SH, m + o * Q_Y, 2.0 ** e])
    return coef, m


def bcoefs(C, gen, device):
    """(mean(dz), mean(dz*xhat)) [2, C]: multiples of 1/8 in [-7/8, 7/8]."""
    return X.ints((2, C), -7, 7, gen, device) * Q_M


def y_values(shape, centre, gen, device, r=7):
    """y = centre[c] + j/16 with |j| <= r: at most 7 significant bits (bf16-exact), few distinct values per channel (many
    ties inside the 2x2x2 windows) and |y - mean| <= (r + 2)/16."""
    return centre + X.ints(shape, -r, r, gen, device) * Q_Y


def dout_values(shape, gen, device):
    """Pooled (or unpooled) gradients: integers in [-1, 1], exact in bf16 and fp32."""
    return X.ints(shape, -1, 1, gen, device)


def check_design(pool, y_absmax=4 + 9 * Q_Y, dout_absmax=1.0):
    """Worst-case magnitudes, in quanta, of every element-wise value the kernels form on operands of the generators above
    (asserts each stays below 2^24 quanta: exact in fp32 under any FMA contraction).  Returns the quantum of dz."""
    sc, sh, is_max, is_min, m = 7 * Q_SC, 31 * Q_SH, 2.0 ** max(IS_EXP), 2.0 ** min(IS_EXP), 7 * Q_M
    mu = 4 + 2 * Q_Y
    q_z = Q_Y * Q_SC                                              # y * scale + shift (shift is a multiple of q_z)
    X.exact_bound(1, y_absmax * sc + sh, 1, q_z)
    z = y_absmax * sc + sh
    X.exact_bound(1, 8 * z, 1, q_z * SLOPE)                       # activations and the 8-term window sum
    if pool == POOL_AVG:
        X.exact_bound(1, z, 1, q_z * SLOPE / 8)                   # the average
    q_dz = (1 / 8 if pool == POOL_AVG else 1) * SLOPE             # dout integers
    xh = (y_absmax + mu) * is_max
    X.exact_bound(1, xh, 1, Q_Y * is_min)                         # xhat
    X.exact_bound(1, dout_absmax * xh, 1, q_dz * Q_Y * is_min)    # dz * xhat
    q_cb = Q_SC * Q_M * is_min                                    # Bc = -scale * m2 * invstd
    cb = sc * m * is_max
    q = q_cb * Q_Y                                                # Bc * y, Bc * mean, A, dy
    X.exact_bound(1, cb * y_absmax, 1, q)
    X.exact_bound(1, sc * m + cb * mu, 1, q)                      # A = -scale * m1 - Bc * mean
    X.exact_bound(1, sc * dout_absmax + sc * m + cb * mu + cb * y_absmax, 1, min(q, Q_SC * q_dz))   # dy
    return q_dz


def check_sums_exact(a1, a2, inv, pool):
    """The whole-tower sums of |dz| and |dz * xhat| per channel, in that channel's quanta, stay below 2^24: every
    partial sum of every thread split is then exact in fp32 (the xhat quantum is 2^-4 * invstd of the channel)."""
    q_dz = (1 / 8 if pool == POOL_AVG else 1) * SLOPE
    X.exact_bound(1, float(a1.max()), 1, q_dz)
    X.exact_bound(1, float((a2 / inv).max()), 1, q_dz * Q_Y)


def rounding_profile(ref):
    """(inexact, halfway): how many values of an fp32-exact reference are not bf16-exact, and how many lie exactly
    halfway between two bf16 neighbours (the tie-to-even cases)."""
    r = ref.float().contiguous().view(torch.int32)
    low = r & 0xFFFF
    return int((low != 0).sum()), int((low == 0x8000).sum())


# ---------------------------------------------------------------------------------------------------------------
# shape table: the seven sNet layers (SNetSpec.layers order) at the block extents of conv_exact.GEOMS, plus block 1
LAYERS = (("L0", 32, POOL_MAX, 0), ("L1", 32, POOL_NONE, 1), ("L2", 64, POOL_MAX, 1), ("L3", 64, POOL_NONE, 2),
          ("L4", 128, POOL_MAX, 2), ("L5", 256, POOL_NONE, 3), ("L6", 128, POOL_AVG, 3))
BLOCK1 = {"bench": (91, 109, 91), "spm": (79, 95, 79), "wide": (128, 128, 79)}


def _model_cases():
    out = []
    for g, (B, blocks) in X.GEOMS.items():
        ext = (BLOCK1[g],) + tuple(blocks)
        for name, C, pool, blk in LAYERS:
            out.append((f"{g}-{name}", B, ext[blk], C, pool, name == "L6"))
    return out


MODEL_CASES = _model_cases()

# (id, B, (D, H, W), C, pool, fp32 output)
EDGE_CASES = [
    ("odd-max", 3, (5, 7, 9), 32, POOL_MAX, False),           # odd extents: voxels outside every complete window
    ("odd-avg", 2, (7, 5, 3), 64, POOL_AVG, True),
    ("odd-none", 3, (5, 3, 7), 64, POOL_NONE, False),
    ("d2", 2, (2, 6, 5), 32, POOL_MAX, False),                # Do = 1
    ("d3-b1", 1, (3, 4, 6), 32, POOL_MAX, False),             # Do = 1 with a dropped plane, one sample
    ("w1-none", 2, (3, 5, 1), 32, POOL_NONE, False),
    ("w2-max", 2, (4, 6, 2), 64, POOL_MAX, False),
    ("c8", 3, (6, 7, 8), 8, POOL_MAX, False),
    ("c24-max", 4, (150, 12, 30), 24, POOL_MAX, False),       # CQ = 3: idle thread, pstep = 85; 300 planes > 296 units
    ("c24-none", 4, (9, 11, 13), 24, POOL_NONE, False),
    ("c24-avg", 2, (6, 10, 12), 24, POOL_AVG, True),
    ("c1024-max", 1, (4, 4, 6), 1024, POOL_MAX, False),       # pstep = 2
    ("c1024-none", 1, (2, 3, 5), 1024, POOL_NONE, False),
    ("one-block", 1, (4, 6, 8), 32, POOL_MAX, False),         # 24 pooled positions: the kept reduction runs one block
    ("max-fp32out", 2, (6, 8, 10), 32, POOL_MAX, True),       # keepmax with an fp32 output
]

BN_CASES = MODEL_CASES + EDGE_CASES

"""Exact-arithmetic references and operand generators for the sNet convolution tests (tests/test_gpu_conv_exact.py).

When every operand is a multiple of a quantum q (an integer, or a short significand on a fixed grid), every bf16 x bf16
(or split fp32) product is a multiple of q_a * q_w and exact in fp32; if in addition the sum of the absolute values of
all terms of an output stays below 2^24 quanta, every partial sum is exact in fp32, so every tiling, split-K order,
TMEM accumulation and reduction order gives the same value.  A correct kernel then agrees with the float64 reference
below bit for bit (fp32 outputs directly; bf16 outputs after one round-to-nearest-even of the reference).

The references work on NDHWC float64 tensors (on whatever device the inputs live) as 27 shifted per-tap GEMMs
(one GEMM for a 1x1x1 layer), the cross-correlation convention of F.conv3d with zero padding k // 2.
"""
import ctypes as C
import math

import torch
import torch.nn.functional as F

FP32_EXACT = 2 ** 24          # integers (in quanta) below this are exact in fp32, and so is every sum that stays below


# ---------------------------------------------------------------------------------------------------------------
# operand generators
def ints(shape, lo, hi, gen, device):
    """Integers uniform in [lo, hi] (float64)."""
    return torch.randint(lo, hi + 1, shape, generator=gen, device=device).double()


def fixed(shape, bits, frac, gen, device):
    """Multiples k * 2^-frac with |k| < 2^bits (float64): a significand of at most `bits` bits on a 2^-frac grid."""
    k = torch.randint(-(2 ** bits) + 1, 2 ** bits, shape, generator=gen, device=device)
    return k.double() * 2.0 ** -frac


def exact_bound(n_terms, amax, bmax, quantum, extra=0.0):
    """Worst-case |partial sum| of n_terms products |a*b| <= amax * bmax (plus `extra`, e.g. a bias), in units of the
    products' common quantum.  Asserts it stays below 2^24, the condition for every summation order to be exact in fp32."""
    q = (n_terms * amax * bmax + extra) / quantum
    assert q < FP32_EXACT, f"operands too large for exact fp32 sums: {q:.4g} quanta >= 2^24"
    return q


def bf16_rne(ref):
    """The bf16 a kernel must store for an exact float64 value that fits fp32: one round-to-nearest-even."""
    r32 = ref.float()
    assert torch.equal(r32.double(), ref), "reference is not exact in fp32"
    return r32.to(torch.bfloat16)


# ---------------------------------------------------------------------------------------------------------------
# float64 references (NDHWC)
def conv_ref(a, w):
    """y[B,D,H,W,Cout] = sum_tap a[v + tap - k//2] . w[:, :, tap]^T for a [B,D,H,W,Cin], w (Cout,Cin,k,k,k)."""
    k = w.shape[-1]
    if k == 1:
        return a @ w[:, :, 0, 0, 0].T
    p = k // 2
    B, D, H, W, _ = a.shape
    ap = F.pad(a, (0, 0, p, p, p, p, p, p))
    y = torch.zeros((B, D, H, W, w.shape[0]), dtype=a.dtype, device=a.device)
    for kd in range(k):
        for kh in range(k):
            for kw in range(k):
                y += ap[:, kd:kd + D, kh:kh + H, kw:kw + W, :] @ w[:, :, kd, kh, kw].T
    return y


def dgrad_ref(dy, w):
    """Gradient of conv_ref with respect to a: the forward on the flipped, transposed weights (what the dgrad pack holds)."""
    return conv_ref(dy, w.transpose(0, 1).flip(2, 3, 4))


def wgrad_ref(dy, a, k):
    """dw (Cout,Cin,k,k,k) = sum_v dy[v, co] * a[v + tap - k//2, ci]."""
    cout, cin = dy.shape[-1], a.shape[-1]
    dyf = dy.reshape(-1, cout).T
    if k == 1:
        return (dyf @ a.reshape(-1, cin)).reshape(cout, cin, 1, 1, 1)
    p = k // 2
    B, D, H, W, _ = a.shape
    ap = F.pad(a, (0, 0, p, p, p, p, p, p))
    dw = torch.empty((cout, cin, k, k, k), dtype=a.dtype, device=a.device)
    for kd in range(k):
        for kh in range(k):
            for kw in range(k):
                dw[:, :, kd, kh, kw] = dyf @ ap[:, kd:kd + D, kh:kh + H, kw:kw + W, :].reshape(-1, cin)
    return dw


def maxpool_route(y, dout):
    """MaxPool3d(2,2) backward (floor mode) on NDHWC: dout [B,D/2,H/2,W/2,C] goes to the first maximum of y in (d,h,w)
    scan order of each window; everything else (including voxels outside complete windows) gets 0."""
    B, D, H, W, Cc = y.shape
    Do, Ho, Wo = D // 2, H // 2, W // 2
    win = (y[:, :2 * Do, :2 * Ho, :2 * Wo].reshape(B, Do, 2, Ho, 2, Wo, 2, Cc)
           .permute(0, 1, 3, 5, 7, 2, 4, 6).reshape(B, Do, Ho, Wo, Cc, 8))
    idx = win.argmax(-1, keepdim=True)          # first maximal element
    routed = torch.zeros_like(win).scatter_(-1, idx, dout.unsqueeze(-1))
    dy = torch.zeros_like(y)
    dy[:, :2 * Do, :2 * Ho, :2 * Wo] = (routed.reshape(B, Do, Ho, Wo, Cc, 2, 2, 2).permute(0, 1, 5, 2, 6, 3, 7, 4)
                                        .reshape(B, 2 * Do, 2 * Ho, 2 * Wo, Cc))
    return dy


# ---------------------------------------------------------------------------------------------------------------
# guard-banded, poisoned buffers
class Guarded:
    """A tensor carved out of a larger byte buffer.  poison() fills the whole buffer with 0xFF bytes (NaN in fp32, bf16
    and fp64); check_bands() asserts that nothing outside the logical tensor was written."""
    BAND = 64 * 1024           # bytes on each side (a multiple of 1024: the tensor keeps the allocation's alignment)

    def __init__(self, shape, dtype, device):
        self.nbytes = math.prod(shape) * torch.empty((), dtype=dtype).element_size()
        self.buf = torch.empty(self.nbytes + 2 * self.BAND, dtype=torch.uint8, device=device)
        self.t = self.buf[self.BAND:self.BAND + self.nbytes].view(dtype).view(shape)
        self.poison()

    def poison(self):
        self.buf.fill_(0xFF)
        return self.t

    def check_bands(self, what):
        lo, hi = self.buf[:self.BAND], self.buf[self.BAND + self.nbytes:]
        assert bool((lo == 0xFF).all()) and bool((hi == 0xFF).all()), f"{what}: written outside the tensor"


def mismatch(got, want):
    """'' if got and want hold the same bits, else a short description of where they differ."""
    if torch.equal(got, want):
        return ""
    bad = (got.double() != want.double()) | got.double().isnan()
    n = int(bad.sum())
    i = tuple(int(c) for c in bad.nonzero()[0])
    return f"{n} of {got.numel()} elements differ; first at {i}: got {float(got[i])}, want {float(want[i])}"


# ---------------------------------------------------------------------------------------------------------------
# which tcgen05 kernel a problem reaches (host-only plan introspection)
def wgrad_takes_column_kernel(ng, W, cin, cout, ks):
    """Mirrors make_wc_plan (csrc/wgrad_umma_col.cu), which nothing exports: 3x3x3, Cin and Cout multiples of 32, at most
    16 (tower, ci block, co block) virtual groups, 2 <= W <= 255, and rings of at least 4 X and 2 dY slabs in shared
    memory.  Every other problem goes to the generic kernel of wgrad_umma.cu."""
    if ks != 3 or cin % 32 or cout % 32 or ng * (cin // 32) * (cout // 32) > 16 or W < 2 or W + 1 > 256:
        return False
    wp = W + 1
    nhy = ((wp - 1) + 127 + 2 * wp) // wp + 1
    nhx = ((wp - 1) + 127 + 2 * wp - 1 + 3) // wp + 1
    slab = lambda rows: (rows * wp * 64 + 1023) & ~1023
    return 1024 + 8 * 4 * 8 + 8 + 16 + 16 + 64 + 4 * slab(nhx) + 2 * slab(nhy) <= 227 * 1024


def fwd_kernel(lib, ng, B, D, H, W, cin, cout, ks):
    """The kernel tmf_conv3d_fwd (impl UMMA) runs, and the plan flags: 'col' / 'col-ns' (conv_umma_col.cu, kw-stacked /
    non-stacked), 'gemm' (conv_umma.cu on a 1x1x1 layer flattened to one GEMM), 'resident' / 'streamed' (conv_umma.cu)
    with ' stack' (plane-stack tiles), ' kwf' (kw-fused weight boxes), ' mt>1' (several 128-row tiles per weight pass)."""
    o6 = (C.c_int * 6)()
    if lib.tmf_conv3d_col_plan_info(ng, D, H, W, cin, cout, ks, o6) == 0:
        return "col-ns" if o6[1] else "col"
    o8 = (C.c_int * 8)()
    if ks == 1:               # tmf_conv3d_fwd_umma flattens the volume: one plane of B*D*H*W rows of width 1
        assert lib.tmf_conv3d_umma_plan_info(ng, 1, 1, B * D * H * W, 1, cin, cout, ks, o8) == 0
        return "gemm"
    assert lib.tmf_conv3d_umma_plan_info(ng, B, D, H, W, cin, cout, ks, o8) == 0, "no tcgen05 plan"
    name = "resident" if o8[7] & 1 else "streamed"
    if o8[7] & 2:
        name += " stack"
    if o8[7] & 4:
        name += " kwf"
    if o8[1] > 1:
        name += " mt>1"
    return name


def wgrad_kernel(ng, W, cin, cout, ks):
    return "wgrad-col" if wgrad_takes_column_kernel(ng, W, cin, cout, ks) else "wgrad-generic"


# ---------------------------------------------------------------------------------------------------------------
# shape table: (id, ng, B, (D, H, W), cin, cout, ks, {op: kernel}) -- the kernel each op must reach
GEOMS = {"bench": (8, ((45, 54, 45), (22, 27, 22), (11, 13, 11))),          # 91 x 109 x 91, batch 8
         "spm": (4, ((39, 47, 39), (19, 23, 19), (9, 11, 9))),              # 79 x 95 x 79
         "wide": (4, ((64, 64, 39), (32, 32, 19), (16, 16, 9)))}            # 128 x 128 x 79
LAYERS = (("conv2.0", 0, 32, 32, 3), ("conv2.3", 0, 32, 64, 3), ("conv3.0", 1, 64, 64, 3), ("conv3.3", 1, 64, 128, 3),
          ("conv4.0", 2, 128, 256, 3), ("conv4.3", 2, 256, 128, 1))
_MODEL_DISPATCH = {   # fwd, dgrad, wgrad
    "conv2.0": ("col", "col", "wgrad-col"), "conv2.3": ("col-ns", "col", "wgrad-col"), "conv3.0": ("col", "col", "wgrad-col"),
    "conv3.3": ("col", "streamed mt>1", "wgrad-col"), "conv4.0": ("streamed stack", "streamed stack kwf", "wgrad-generic"),
    "conv4.3": ("gemm", "gemm", "wgrad-generic")}


def _model_cases():
    out = []
    for g, (B, blocks) in GEOMS.items():
        for name, blk, cin, cout, ks in LAYERS:
            f, d, w = _MODEL_DISPATCH[name]
            if g == "wide" and name == "conv4.0":
                d = "streamed mt>1"     # 16 x 16 x 9, two towers: two per-plane tiles per weight pass beat plane stacks
            out.append((f"{g}-{name}", 2, B, blocks[blk], cin, cout, ks, {"fwd": f, "dgrad": d, "wgrad": w}))
    for name, blk, cin, cout, ks in (LAYERS[1], LAYERS[4]):   # one tower alone
        f, d, w = _MODEL_DISPATCH[name]
        out.append((f"bench-{name}-ng1", 1, 8, GEOMS["bench"][1][blk], cin, cout, ks, {"fwd": f, "dgrad": d, "wgrad": w}))
    return out


MODEL_CASES = _model_cases()

EDGE_CASES = [
    # D = 1; odd extents; M = B*D*H*W not a multiple of 128 (true of nearly every case here)
    ("d1", 2, 3, (1, 9, 7), 32, 32, 3, {"fwd": "col", "dgrad": "col", "wgrad": "wgrad-col"}),
    ("d1-generic", 1, 2, (1, 5, 11), 128, 64, 3, {"fwd": "streamed stack kwf", "dgrad": "col", "wgrad": "wgrad-col"}),
    # W = 2, the smallest width of the column kernels; W = 1 goes to the generic kernels (resident weights)
    ("w2", 2, 2, (5, 7, 2), 32, 64, 3, {"fwd": "col-ns", "dgrad": "col", "wgrad": "wgrad-col"}),
    ("w1", 2, 2, (3, 5, 1), 32, 32, 3, {"fwd": "resident", "dgrad": "resident", "wgrad": "wgrad-generic"}),
    # the widest rows each kernel is reached with through the entry points: tmf_conv3d_fwd asks the generic planner first
    # (W + 2 <= 256), so the column forward sees Wp = W + 1 = 255 at most; the column weight gradient fits its rings up to
    # W = 147 and the generic one (tmf_conv3d_wgrad's gate) up to 126 at 32 -> 32
    ("wide-col", 1, 1, (2, 3, 254), 32, 32, 3, {"fwd": "col", "dgrad": "col"}),
    ("wide-col-wgrad", 1, 1, (3, 4, 147), 32, 64, 3, {"wgrad": "wgrad-col"}),
    ("wide-generic", 1, 1, (2, 2, 180), 128, 128, 3, {"fwd": "streamed", "dgrad": "streamed"}),
    ("wide-generic-wgrad", 2, 1, (2, 3, 38), 128, 256, 3, {"wgrad": "wgrad-generic"}),
    # B * tiles * D far below the CTA count: most CTAs own an empty range (the weight gradients launch ~148 per tower
    # whatever the problem size and must still write their zero partials)
    ("tiny", 2, 1, (2, 3, 5), 32, 64, 3, {"fwd": "col-ns", "dgrad": "col", "wgrad": "wgrad-col"}),
    ("tiny-generic", 2, 1, (1, 2, 3), 128, 128, 3, {"fwd": "streamed stack kwf", "dgrad": "streamed stack kwf", "wgrad": "wgrad-generic"}),
    # 64 -> 256 on two towers: the column kernel takes at most 8 tower x 32-channel slices
    ("wide-cout", 2, 2, (6, 7, 9), 64, 256, 3, {"fwd": "streamed stack", "dgrad": "streamed stack kwf", "wgrad": "wgrad-generic"}),
    # plane-stack tiles over several samples, odd extents everywhere
    ("stack-odd", 2, 3, (5, 7, 5), 128, 256, 3, {"fwd": "streamed stack", "dgrad": "streamed stack kwf", "wgrad": "wgrad-generic"}),
    ("odd-1x1", 2, 3, (7, 9, 11), 256, 128, 1, {"fwd": "gemm", "dgrad": "gemm", "wgrad": "wgrad-generic"}),
]

CONV_CASES = MODEL_CASES + EDGE_CASES

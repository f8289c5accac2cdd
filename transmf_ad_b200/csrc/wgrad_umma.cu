// wgrad_umma.cu -- Conv3d weight gradient on tcgen05 tensor cores.
//
//   dW[co][ci][tap] = sum over output voxels v of  dY[v,co] * X[v + shift(tap), ci]
//
// GEMM view: the voxel index is the K dimension (16 voxels per tcgen05.mma), so both operands are "MN-major" and
// are consumed exactly as the NDHWC tensors lie in memory: one TMA box per (plane, 64-channel chunk) gives a slab
// [voxel rows][channels] in shared memory (same padded-row linearisation as the forward kernel, out-of-bounds
// zero fill = convolution padding; dY is loaded with the padded pitch too, so its garbage columns are zeros and
// contribute nothing).  A tap shift is again just a row offset of the X-slab descriptor.
//   M (128 TMEM lanes) = X side: input channels, with several taps STACKED along M for narrow layers: the descriptor's
//                        leading-byte-offset is the distance between consecutive M atoms, so atoms that start one row
//                        (kw+1) or one padded row (kh+1) later are neighbouring taps.
//   N (TMEM columns)   = dY side: output channels.
// Each CTA owns a subset of (tap group)s whose accumulators fit the 512 TMEM columns and a contiguous range of voxel
// tiles; it accumulates over its whole range in TMEM and writes one fp32 partial to the workspace; a second kernel
// reduces the partials in fixed order (deterministic) into the reference layout (Cout,Cin,k,k,k).
#include <cuda.h>

#include "common.cuh"
#include "umma.cuh"

namespace tmf {
using namespace umma;

constexpr int WG_THREADS = 192;
constexpr int WG_MAX_GROUPS = 54;
constexpr int WG_MAX_SUBSETS = 20;
constexpr int WG_MAX_STAGES = 4;
constexpr uint32_t WG_SMEM_BUDGET = 227 * 1024;

struct WgGroup {
  uint32_t a_off;        // byte offset of the group's first M atom inside the X region of a stage (for qoff = 0)
  uint32_t a_lbo;        // byte distance between consecutive M atoms
  int16_t tap[4];        // tap index of each M atom (-1: garbage lanes)
  int16_t cib[4];        // first input channel of each M atom
};
struct WgSubset {
  int16_t g0, ng, kd0, nkd;
};

struct alignas(64) WgradParams {
  CUtensorMap tmX[TMF_MAX_GROUPS];
  CUtensorMap tmY[TMF_MAX_GROUPS];
  float* ws[TMF_MAX_GROUPS];
  int ngroups_tower, B, D, H, W, cin, cout, ks, hw, taps;
  int Wp, NHx, NHy, QT, TK, NKT;      // padded pitch, slab heights, voxel tiles per plane, voxels per tile, #tiles
  int nsub, nsplit, kt_per_split;
  int nchx, chx, rbx;                 // X: chunks, channels per chunk, row bytes
  int nchy, chy, rby;                 // dY: chunks, channels per chunk, row bytes
  uint32_t layx, layy;
  uint32_t x_slab_bytes, y_slab_bytes, x_tx, y_tx, stage_bytes, y_region_off;
  int atom_m;                         // channels per M atom (32 or 64)
  int stages;
  uint32_t idesc, tmem_cols;
  WgSubset sub[WG_MAX_SUBSETS];
  WgGroup grp[WG_MAX_GROUPS];
};

template <int KSTEPS>
__global__ void __launch_bounds__(WG_THREADS, 1) conv3d_wgrad_umma_kernel(const __grid_constant__ WgradParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bars = smem_base + (uint32_t)p.stages * p.stage_bytes;
  const uint32_t full = bars, empty = bars + 8 * WG_MAX_STAGES, acc_full = empty + 8 * WG_MAX_STAGES;
  const uint32_t tmem_slot = acc_full + 8;
  uint8_t* gen_base = smem_raw + (smem_base - smem_u32(smem_raw));
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(gen_base + (tmem_slot - smem_base));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int r = blockIdx.x;
  const int tw = r % p.ngroups_tower; r /= p.ngroups_tower;
  const int si = r % p.nsub;
  const int split = r / p.nsub;
  const WgSubset S = p.sub[si];
  const int kt0 = split * p.kt_per_split;
  const int kt1 = min(p.NKT, kt0 + p.kt_per_split);

  if (threadIdx.x == 0) {
    for (int i = 0; i < p.stages; ++i) { mbar_init(full + 8 * i, 1); mbar_init(empty + 8 * i, 1); }
    mbar_init(acc_full, 1);
    fence_barrier_init();
    prefetch_tmap(&p.tmX[tw]);
    prefetch_tmap(&p.tmY[tw]);
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, p.tmem_cols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp == 0) {
    if (lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      const uint32_t tx = (uint32_t)S.nkd * p.nchx * p.x_tx + (uint32_t)p.nchy * p.y_tx;
      for (int kt = kt0; kt < kt1; ++kt) {
        int t = kt;
        const int qt = t % p.QT; t /= p.QT;
        const int d = t % p.D;
        const int n = t / p.D;
        const int h0 = (qt * p.TK) / p.Wp;
        mbar_wait(empty + 8 * s, ph ^ 1u);
        mbar_expect_tx(full + 8 * s, tx);
        const uint32_t st = smem_base + (uint32_t)s * p.stage_bytes;
        for (int k = 0; k < S.nkd; ++k)
          for (int c = 0; c < p.nchx; ++c)
            tma_load_5d(st + (uint32_t)(k * p.nchx + c) * p.x_slab_bytes, &p.tmX[tw], full + 8 * s, c * p.chx, -p.hw,
                        h0 - p.hw, d + S.kd0 + k - p.hw, n);
        for (int c = 0; c < p.nchy; ++c)
          tma_load_5d(st + p.y_region_off + (uint32_t)c * p.y_slab_bytes, &p.tmY[tw], full + 8 * s, c * p.chy, 0, h0, d, n);
        if (++s == p.stages) { s = 0; ph ^= 1u; }
      }
    }
  } else if (warp == 1) {
    // warp-uniform control flow, one elected lane issues (see conv_umma.cu)
    {
      int s = 0;
      uint32_t ph = 0;
      const uint32_t sbo_x = 8u * p.rbx, sbo_y = 8u * p.rby;
      // descriptors: constant high word; low word = start address (16-byte units) | LBO << 16
      const uint64_t hi_x = make_smem_desc(0, 0, sbo_x, p.layx, 0) & 0xFFFFFFFF00000000ull;
      const uint64_t hi_y = make_smem_desc(0, 0, sbo_y, p.layy, 0) & 0xFFFFFFFF00000000ull;
      const uint32_t y_lo_const = ((p.y_slab_bytes >> 4) & 0x3FFFu) << 16;
      const uint32_t kstep_x = (16u * p.rbx) >> 4, kstep_y = (16u * p.rby) >> 4;
      const uint32_t rbx_units = p.rbx >> 4, rby_units = p.rby >> 4;
      const uint32_t stage_units = p.stage_bytes >> 4;
      const uint32_t base_units = (smem_base & 0x3FFFFu) >> 4;
      const uint32_t yreg_units = p.y_region_off >> 4;
      uint32_t accumulate = 0;
      for (int kt = kt0; kt < kt1; ++kt) {
        const int qt = kt % p.QT;
        const uint32_t qoff = (uint32_t)((qt * p.TK) % p.Wp);
        mbar_wait(full + 8 * s, ph);
        tc_fence_after();
        const uint32_t st_units = base_units + (uint32_t)s * stage_units;
        const uint32_t y_lo = y_lo_const | (st_units + yreg_units + qoff * rby_units);
        const uint32_t x_units = st_units + qoff * rbx_units;
#pragma unroll 1
        for (int gi = 0; gi < S.ng; ++gi) {
          const WgGroup& G = p.grp[S.g0 + gi];
          const uint32_t a_lo = ((((G.a_lbo >> 4) & 0x3FFFu) << 16) | x_units) + (G.a_off >> 4);
          const uint32_t d_tmem = tmem_base + (uint32_t)(gi * p.cout);
          if (elect_one()) {
            mma_bf16_ss(d_tmem, hi_x | (uint64_t)a_lo, hi_y | (uint64_t)y_lo, p.idesc, accumulate);
#pragma unroll
            for (int k = 1; k < KSTEPS; ++k)
              mma_bf16_ss(d_tmem, hi_x | (uint64_t)(a_lo + k * kstep_x), hi_y | (uint64_t)(y_lo + k * kstep_y), p.idesc, 1u);
          }
          __syncwarp();
        }
        accumulate = 1;
        if (elect_one()) mma_commit(empty + 8 * s);
        __syncwarp();
        if (++s == p.stages) { s = 0; ph ^= 1u; }
      }
      if (elect_one()) mma_commit(acc_full);
      __syncwarp();
    }
  } else {
    // epilogue: TMEM -> fp32 partial ws[split][tap][ci][co]
    const int quarter = warp & 3;
    const int m = quarter * 32 + lane;
    const int atom = m / p.atom_m, cl = m % p.atom_m;
    mbar_wait(acc_full, 0u);
    tc_fence_after();
    float* ws = p.ws[tw] + (size_t)split * p.taps * p.cin * p.cout;
    for (int gi = 0; gi < S.ng; ++gi) {
      const WgGroup& G = p.grp[S.g0 + gi];
      const int tap = G.tap[atom];
      const int ci = G.cib[atom] + cl;
      const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(gi * p.cout);
      for (int c0 = 0; c0 < p.cout; c0 += 32) {
        uint32_t raw[32];
        tmem_ld32(taddr + (uint32_t)c0, raw);
        tmem_ld_wait();
        if (tap >= 0) {
          float4* dst = reinterpret_cast<float4*>(ws + ((size_t)tap * p.cin + ci) * p.cout + c0);
#pragma unroll
          for (int j = 0; j < 8; ++j)
            dst[j] = make_float4(__uint_as_float(raw[4 * j]), __uint_as_float(raw[4 * j + 1]),
                                 __uint_as_float(raw[4 * j + 2]), __uint_as_float(raw[4 * j + 3]));
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, p.tmem_cols);
  }
}

// dw[co][ci][tap] = sum_split ws[split][tap][ci][co]   (fixed order -> deterministic)
__global__ void wgrad_reduce_kernel(GroupPtr<const float> ws, GroupPtr<float> dw, int nsplit, int taps, int cin,
                                    int cout) {
  const int g = blockIdx.z;
  const int64_t total = (int64_t)taps * cin * cout;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int co = (int)(i % cout);
    const int ci = (int)((i / cout) % cin);
    const int tap = (int)(i / ((int64_t)cout * cin));
    float s = 0.f;
    for (int k = 0; k < nsplit; ++k) s += ws.p[g][(int64_t)k * total + i];
    dw.p[g][((int64_t)co * cin + ci) * taps + tap] = s;
  }
}

// ------------------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn wg_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn == nullptr) {
    void* sym = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(sym);
  }
  return fn;
}

static bool build_wgrad_plan(WgradParams& p, int ng, int B, int D, int H, int W, int cin, int cout, int ks, int sms,
                             uint32_t* smem_bytes, CUtensorMapSwizzle* swx, CUtensorMapSwizzle* swy) {
  if (ks != 1 && ks != 3) return false;
  if (!(cin == 32 || cin % 64 == 0) || !(cout == 32 || cout % 64 == 0)) return false;
  if (cin > 256 || cout > 256 || cin < 32 || cout < 32) return false;
  p.ngroups_tower = ng; p.B = B; p.D = D; p.H = H; p.W = W; p.cin = cin; p.cout = cout; p.ks = ks; p.hw = ks / 2;
  p.taps = ks * ks * ks;
  p.Wp = W + 2 * p.hw;
  p.chx = (cin == 32) ? 32 : 64; p.nchx = cin / p.chx; p.rbx = p.chx * 2;
  p.chy = (cout == 32) ? 32 : 64; p.nchy = cout / p.chy; p.rby = p.chy * 2;
  p.layx = (p.chx == 64) ? LAYOUT_SW128 : LAYOUT_SW64;
  p.layy = (p.chy == 64) ? LAYOUT_SW128 : LAYOUT_SW64;
  *swx = (p.chx == 64) ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
  *swy = (p.chy == 64) ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
  p.atom_m = p.chx;
  if (p.Wp > 256) return false;
  // ---- tap groups (per kd plane), M = 128 lanes = 128 / atom_m atoms
  int ngrp_kd = 0;
  WgGroup gk[18];
  const int tap2 = ks * ks;
  auto rowoff = [&](int kh, int kw) { return (uint32_t)(kh * p.Wp + kw) * p.rbx; };
  if (cin == 32) {
    for (int kh = 0; kh < ks; ++kh) {
      WgGroup& G = gk[ngrp_kd++];
      G.a_off = rowoff(kh, 0); G.a_lbo = p.rbx;
      for (int a = 0; a < 4; ++a) { G.tap[a] = (a < ks) ? (int16_t)(kh * ks + a) : (int16_t)-1; G.cib[a] = 0; }
    }
  } else if (cin == 64) {
    if (ks == 1) {
      WgGroup& G = gk[ngrp_kd++];
      G.a_off = 0; G.a_lbo = p.rbx; G.tap[0] = 0; G.tap[1] = -1; G.cib[0] = G.cib[1] = 0;
    } else {
      for (int kh = 0; kh < 3; ++kh) {          // (kh,0)+(kh,1): one row apart
        WgGroup& G = gk[ngrp_kd++];
        G.a_off = rowoff(kh, 0); G.a_lbo = p.rbx;
        G.tap[0] = (int16_t)(kh * 3); G.tap[1] = (int16_t)(kh * 3 + 1); G.cib[0] = G.cib[1] = 0;
      }
      {                                         // (0,2)+(1,2): one padded row apart
        WgGroup& G = gk[ngrp_kd++];
        G.a_off = rowoff(0, 2); G.a_lbo = (uint32_t)p.Wp * p.rbx;
        G.tap[0] = 2; G.tap[1] = 5; G.cib[0] = G.cib[1] = 0;
      }
      {                                         // (2,2) + garbage
        WgGroup& G = gk[ngrp_kd++];
        G.a_off = rowoff(2, 2); G.a_lbo = p.rbx;
        G.tap[0] = 8; G.tap[1] = -1; G.cib[0] = G.cib[1] = 0;
      }
    }
    for (int i = 0; i < ngrp_kd; ++i) { gk[i].tap[2] = gk[i].tap[3] = -1; gk[i].cib[2] = gk[i].cib[3] = 0; }
  } else {                                      // cin = 128 / 192 / 256: one tap, two 64-channel chunks per group
    for (int t = 0; t < tap2; ++t)
      for (int c2 = 0; c2 < p.nchx / 2; ++c2) {
        WgGroup& G = gk[ngrp_kd++];
        G.a_off = 0; G.a_lbo = 0;               // filled below (needs slab size)
        G.tap[0] = G.tap[1] = (int16_t)t; G.tap[2] = G.tap[3] = -1;
        G.cib[0] = (int16_t)(c2 * 128); G.cib[1] = (int16_t)(c2 * 128 + 64); G.cib[2] = G.cib[3] = 0;
      }
    if (p.nchx % 2) return false;
  }
  const int maxg = 512 / cout;
  if (maxg < 1) return false;
  // ---- subsets
  p.nsub = 0;
  int total_groups = 0;
  int nkd_sub;
  if (ks * ngrp_kd <= maxg) {
    nkd_sub = ks;
    p.sub[p.nsub++] = WgSubset{0, (int16_t)(ks * ngrp_kd), 0, (int16_t)ks};
    total_groups = ks * ngrp_kd;
  } else {
    nkd_sub = 1;
    for (int kd = 0; kd < ks; ++kd)
      for (int g0 = 0; g0 < ngrp_kd; g0 += maxg) {
        if (p.nsub >= WG_MAX_SUBSETS) return false;
        const int n = min(maxg, ngrp_kd - g0);
        p.sub[p.nsub++] = WgSubset{(int16_t)(kd * ngrp_kd + g0), (int16_t)n, (int16_t)kd, 1};
      }
    total_groups = ks * ngrp_kd;
  }
  if (total_groups > WG_MAX_GROUPS) return false;
  // ---- tile size / smem plan
  const uint32_t fixed = 1024 + 8 * (2 * WG_MAX_STAGES) + 64;
  bool fit = false;
  for (int TK = 128; TK >= 64 && !fit; TK /= 2) {
    p.TK = TK;
    const int rmaxx = (p.Wp - 1) + (ks - 1) * p.Wp + (ks - 1) + (TK - 1) + 3;   // +3: garbage atoms of stacked groups
    p.NHx = rmaxx / p.Wp + 1;
    p.NHy = ((p.Wp - 1) + (TK - 1)) / p.Wp + 1;
    if (p.NHx > 256 || p.NHy > 256) continue;
    p.x_tx = (uint32_t)p.NHx * p.Wp * p.rbx;
    p.y_tx = (uint32_t)p.NHy * p.Wp * p.rby;
    p.x_slab_bytes = (p.x_tx + 1023u) & ~1023u;
    p.y_slab_bytes = (p.y_tx + 1023u) & ~1023u;
    p.y_region_off = (uint32_t)nkd_sub * p.nchx * p.x_slab_bytes;
    p.stage_bytes = p.y_region_off + (uint32_t)p.nchy * p.y_slab_bytes;
    for (int st = WG_MAX_STAGES; st >= 2; --st)
      if (fixed + (uint32_t)st * p.stage_bytes <= WG_SMEM_BUDGET) { p.stages = st; fit = true; break; }
  }
  if (!fit) return false;
  *smem_bytes = fixed + (uint32_t)p.stages * p.stage_bytes;
  // ---- materialise the group table (byte offsets now known)
  for (int kd = 0; kd < ks; ++kd)
    for (int i = 0; i < ngrp_kd; ++i) {
      WgGroup G = gk[i];
      const int kdl = (nkd_sub == ks) ? kd : 0;      // slab index of this kd inside the stage
      if (cin >= 128) {
        const int t = i / (p.nchx / 2), c2 = i % (p.nchx / 2);
        G.a_off = (uint32_t)(kdl * p.nchx + 2 * c2) * p.x_slab_bytes + rowoff(t / ks, t % ks);
        G.a_lbo = p.x_slab_bytes;
      } else {
        G.a_off += (uint32_t)(kdl * p.nchx) * p.x_slab_bytes;
      }
      for (int a = 0; a < 4; ++a)
        if (G.tap[a] >= 0) G.tap[a] = (int16_t)(G.tap[a] + kd * tap2);
      p.grp[kd * ngrp_kd + i] = G;
    }
  p.QT = (H * p.Wp + p.TK - 1) / p.TK;
  p.NKT = B * D * p.QT;
  int per_tower = sms / ng;
  p.nsplit = max(1, per_tower / p.nsub);
  if (p.nsplit > p.NKT) p.nsplit = p.NKT;
  p.kt_per_split = (p.NKT + p.nsplit - 1) / p.nsplit;
  p.nsplit = (p.NKT + p.kt_per_split - 1) / p.kt_per_split;
  p.idesc = make_idesc_bf16(128, cout, 1, 1);
  uint32_t cols = 32;
  int maxng = 0;
  for (int i = 0; i < p.nsub; ++i) maxng = max(maxng, (int)p.sub[i].ng);
  while (cols < (uint32_t)(maxng * cout)) cols <<= 1;
  if (cols > 512) return false;
  p.tmem_cols = cols;
  return true;
}

static int device_sms() {
  static int sms = 0;
  if (sms == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
  }
  return sms;
}

}  // namespace tmf

using namespace tmf;

// fixed-order sum of split-K partials ws[split][tap][ci][co] -> dw (Cout,Cin,k,k,k); shared with wgrad_umma_col.cu
int tmf_wgrad_reduce(int ng, float* const* ws, float* const* dw, int nsplit, int taps, int cin, int cout, void* stream) {
  GroupPtr<const float> gws;
  GroupPtr<float> gdw;
  for (int g = 0; g < TMF_MAX_GROUPS; ++g) { gws.p[g] = nullptr; gdw.p[g] = nullptr; }
  for (int g = 0; g < ng; ++g) { gws.p[g] = ws[g]; gdw.p[g] = dw[g]; }
  const int64_t total = (int64_t)taps * cin * cout;
  dim3 rgrid(min(ceil_div(total, 256), 148 * 4), 1, ng);
  launch_k(wgrad_reduce_kernel, rgrid, 256, 0, (cudaStream_t)stream, gws, gdw, nsplit, taps, cin, cout);
  TMF_LAUNCH_CHECK();
  return 0;
}

bool tmf_conv3d_wgrad_umma_supported(int D, int H, int W, int cin, int cout, int ksize) {
  if (getenv("TMF_DISABLE_UMMA") != nullptr) return false;
  WgradParams p{};
  uint32_t smem;
  CUtensorMapSwizzle a, b;
  return build_wgrad_plan(p, 1, 1, D, H, W, cin, cout, ksize, 148, &smem, &a, &b);
}

size_t tmf_conv3d_wgrad_umma_workspace(int ng, int B, int D, int H, int W, int cin, int cout, int ksize) {
  WgradParams p{};
  uint32_t smem;
  CUtensorMapSwizzle a, b;
  if (!build_wgrad_plan(p, ng, B, D, H, W, cin, cout, ksize, 148, &smem, &a, &b)) return 0;
  // sized for the worst split count (sms may differ from 148 only downwards in nsplit)
  return (size_t)ng * (size_t)(148 / ng / p.nsub + 1) * p.taps * cin * cout * sizeof(float);
}

int tmf_conv3d_wgrad_umma(int ng, const void* const* dy, const void* const* a, float* const* dw, int B, int D, int H,
                          int W, int cin, int cout, int ksize, void* ws, size_t ws_bytes, void* stream) {
  TMF_CHECK_NG(ng);
  WgradParams p{};
  uint32_t smem = 0;
  CUtensorMapSwizzle swx, swy;
  // 1x1x1: a plain GEMM over the voxel rows -- flatten the volume so that every K tile of 128 voxels is full
  if (ksize == 1 && (int64_t)B * D * H * W < (1ll << 31)) { H = B * D * H * W; B = 1; D = 1; W = 1; }
  TMF_REQUIRE(build_wgrad_plan(p, ng, B, D, H, W, cin, cout, ksize, device_sms(), &smem, &swx, &swy),
              "conv3d_wgrad_umma: unsupported problem");
  const size_t per_tower = (size_t)p.nsplit * p.taps * cin * cout * sizeof(float);
  TMF_REQUIRE(ws != nullptr && ws_bytes >= per_tower * ng, "conv3d_wgrad_umma: workspace too small (%zu < %zu bytes)",
              ws_bytes, per_tower * ng);
  EncodeTiledFn encode = wg_encode_fn();
  TMF_REQUIRE(encode != nullptr, "conv3d_wgrad_umma: cuTensorMapEncodeTiled entry point not available");
  GroupPtr<const float> gws;
  GroupPtr<float> gdw;
  for (int g = 0; g < TMF_MAX_GROUPS; ++g) { gws.p[g] = nullptr; gdw.p[g] = nullptr; }
  for (int g = 0; g < ng; ++g) {
    TMF_REQUIRE(dy[g] && a[g] && dw[g], "conv3d_wgrad_umma: NULL device pointer");
    p.ws[g] = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(ws) + per_tower * g);
    gws.p[g] = p.ws[g];
    gdw.p[g] = dw[g];
    cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    {
      cuuint64_t dims[5] = {(cuuint64_t)cin, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)D, (cuuint64_t)B};
      cuuint64_t strides[4] = {(cuuint64_t)cin * 2, (cuuint64_t)W * cin * 2, (cuuint64_t)H * W * cin * 2,
                               (cuuint64_t)D * H * W * cin * 2};
      cuuint32_t box[5] = {(cuuint32_t)p.chx, (cuuint32_t)p.Wp, (cuuint32_t)p.NHx, 1, 1};
      CUresult r = encode(&p.tmX[g], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<void*>(a[g]), dims, strides, box,
                          estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swx, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      TMF_REQUIRE(r == CUDA_SUCCESS, "conv3d_wgrad_umma: cuTensorMapEncodeTiled(X) failed with %d", (int)r);
    }
    {
      cuuint64_t dims[5] = {(cuuint64_t)cout, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)D, (cuuint64_t)B};
      cuuint64_t strides[4] = {(cuuint64_t)cout * 2, (cuuint64_t)W * cout * 2, (cuuint64_t)H * W * cout * 2,
                               (cuuint64_t)D * H * W * cout * 2};
      cuuint32_t box[5] = {(cuuint32_t)p.chy, (cuuint32_t)p.Wp, (cuuint32_t)p.NHy, 1, 1};
      CUresult r = encode(&p.tmY[g], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<void*>(dy[g]), dims, strides, box,
                          estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swy, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      TMF_REQUIRE(r == CUDA_SUCCESS, "conv3d_wgrad_umma: cuTensorMapEncodeTiled(dY) failed with %d", (int)r);
    }
  }
  cudaStream_t st = (cudaStream_t)stream;
  dim3 grid(ng * p.nsub * p.nsplit, 1, 1);
#define TMF_LAUNCH_WG(KST)                                                                                        \
  do {                                                                                                           \
    static bool attr_done = false;                                                                               \
    if (!attr_done) {                                                                                            \
      TMF_CUDA(cudaFuncSetAttribute(conv3d_wgrad_umma_kernel<KST>, cudaFuncAttributeMaxDynamicSharedMemorySize,  \
                                    (int)WG_SMEM_BUDGET));                                                       \
      attr_done = true;                                                                                          \
    }                                                                                                            \
    launch_k(conv3d_wgrad_umma_kernel<KST>, grid, WG_THREADS, smem, st, p);                                            \
  } while (0)
  if (p.TK == 128) TMF_LAUNCH_WG(8); else TMF_LAUNCH_WG(4);
#undef TMF_LAUNCH_WG
  TMF_LAUNCH_CHECK();
  const int64_t total = (int64_t)p.taps * cin * cout;
  dim3 rgrid(min(ceil_div(total, 256), 148 * 4), 1, ng);
  launch_k(wgrad_reduce_kernel, rgrid, 256, 0, st, gws, gdw, p.nsplit, p.taps, cin, cout);
  TMF_LAUNCH_CHECK();
  return 0;
}

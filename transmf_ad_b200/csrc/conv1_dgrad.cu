// conv1_dgrad.cu -- gradient of sNet block 1 with respect to the input image (saliency, input-space attacks):
//   BatchNorm3d(train|eval) + LeakyReLU + MaxPool3d(2,2) backward "apply"   (reference models/networks.py:23-25)
//   followed by the data gradient of conv1.0 = Conv3d(1, 32, 3, padding=1)  (reference models/networks.py:22)
//
//   dy[r][co] = what tmf_bn_act_pool_bwd_apply computes (recomputed from the stored bf16 y, never written to HBM)
//   q[r][tap] = sum_co dy[r][co] * w[co][tap]                 one tcgen05.mma per 128 voxels: M = 128, K = 32, N = 27 -> 32
//   dx[p]     = sum_tap q[p - off(tap)][tap]                  27-term shift-add on chip, every dx element written once
//
// Work unit = one pooling row-quad (n, dp, hp): planes 2dp, 2dp+1 x rows 2hp, 2hp+1 x all w (W <= 128), i.e. four
// "tiles" of 128 voxel rows (64 B = 32 channels each) holding complete pooling windows, so the window arg-max needs
// nothing outside the unit.  A CTA owns a band of C1D_HB output rows of one image and rolls along d over a chunk of
// plane pairs; it recomputes a one-row halo in h (the row-quads above and below the band) and one plane pair in d at
// each end of its chunk.  Roles:
//   * two builder groups (176 threads each) own one shared-memory stage each and turn raw y into dy (same packed-bf16
//     arithmetic as bn_maxpool_bwd_apply_kernel, so dy is bitwise the apply kernel's);
//   * one MMA thread multiplies the four tiles by the bf16 hi / lo halves of the fp32 weight (fp32-level accuracy);
//   * four epilogue warps (TMEM lane quarters: thread = w) read q, exchange the kw = 0 / 2 columns with their w
//     neighbours through shared memory and add the (kd, kh) partial sums into a 4-plane ring of fp32 accumulators that
//     each thread owns for its column w.  The order of every sum is fixed by (plane, row, tap), independent of the
//     grid: no atomics, bitwise reproducible, and one tower gives the same bits whether launched alone or with the other.
#include <algorithm>

#include "common.cuh"
#include "umma.cuh"

namespace tmf {
using namespace umma;

constexpr int C1D_HB = 16;                                // output rows per band (even)
constexpr int C1D_BGROUP = 176;                           // builder group: 5.5 warps (16 warps in all: 128 registers)
constexpr int C1D_THREADS = 160 + 2 * C1D_BGROUP;         // warps 0-3 epilogue, 4 MMA / TMEM, 5-15 builders
constexpr uint32_t C1D_TILE = 128u * 64u;                 // one 128-voxel x 32-channel bf16 tile (64B-swizzled, K-major)
constexpr uint32_t C1D_STAGE = 4u * C1D_TILE;
constexpr int C1D_XW = 132;                               // neighbour-exchange row pitch (w + 1 in [1, 128], pads 0 and 129)
// shared memory layout (offsets from the 1024-aligned base)
constexpr uint32_t C1D_OFF_W = 2u * C1D_STAGE;            // B operand: hi [32 taps][32 co], lo likewise
constexpr uint32_t C1D_OFF_ACC = C1D_OFF_W + 2u * 32u * 64u;
constexpr uint32_t C1D_OFF_X = C1D_OFF_ACC + 4u * C1D_HB * 128u * 4u;
constexpr uint32_t C1D_OFF_COEF = C1D_OFF_X + 2u * 2u * 9u * C1D_XW * 4u;   // per channel A, Bc, scale, shift (fp32)
constexpr uint32_t C1D_OFF_BAR = C1D_OFF_COEF + 4u * 32u * 4u;
constexpr uint32_t C1D_SMEM = 1024u + C1D_OFF_BAR + 64u;
constexpr uint32_t C1D_SMEM_LRP = C1D_SMEM + 4u * C1D_THREADS;   // + one relevance partial sum per thread

struct C1DParams {
  const __nv_bfloat16* y[TMF_MAX_GROUPS];
  const __nv_bfloat16* dout[TMF_MAX_GROUPS];
  const float* coef[TMF_MAX_GROUPS];
  const float* bcoef[TMF_MAX_GROUPS];
  const float* w[TMF_MAX_GROUPS];
  float* dx[TMF_MAX_GROUPS];
  int B, D, H, W, DP, HP, WC, nbands, chunk;
  uint32_t idesc;
  float slope;
  // LRP front (tmf_lrp_conv1): dout = c1, y, zp (or NULL) and a1 build s; dx = R_x = x * (W^T s); part: per-CTA partial sums
  const __nv_bfloat16* a1[TMF_MAX_GROUPS];
  const __nv_bfloat16* zp[TMF_MAX_GROUPS];
  const float* x[TMF_MAX_GROUPS];
  float* part[TMF_MAX_GROUPS];
  float eps;
};

__device__ __forceinline__ uint32_t c1d_sw64(int r, int j) { return (uint32_t)r * 64u + (uint32_t)((j ^ ((r >> 1) & 3)) << 4); }
__device__ __forceinline__ uint32_t c1d_bmax(uint32_t a, uint32_t b) {
  __nv_bfloat162 r = __hmax2(*reinterpret_cast<__nv_bfloat162*>(&a), *reinterpret_cast<__nv_bfloat162*>(&b));
  return *reinterpret_cast<uint32_t*>(&r);
}
__device__ __forceinline__ uint32_t c1d_beq(uint32_t a, uint32_t b) {
  __nv_bfloat162 r = __heq2(*reinterpret_cast<__nv_bfloat162*>(&a), *reinterpret_cast<__nv_bfloat162*>(&b));
  return *reinterpret_cast<uint32_t*>(&r);
}
__device__ __forceinline__ uint32_t c1d_get(const uint4& v, int i) { return i == 0 ? v.x : (i == 1 ? v.y : (i == 2 ? v.z : v.w)); }

// LRP = false: the saliency front (dy from the BatchNorm / LeakyReLU / MaxPool backward apply); LRP = true: the relevance
// front (s = a1 * c1 / stab(z) at each window's first maximum of y, zero elsewhere) and an epilogue that writes x * (W^T s).
template <bool LRP>
__global__ void __launch_bounds__(C1D_THREADS, 1) conv1_dgrad_umma_kernel(const __grid_constant__ C1DParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sbase = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gen = smem_raw + (sbase - smem_u32(smem_raw));
  const uint32_t bars = sbase + C1D_OFF_BAR;
  const uint32_t built = bars, mma_done = bars + 16, tfree = bars + 32, tmem_slot = bars + 48;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = blockIdx.z, n = blockIdx.y;
  const int band = blockIdx.x % p.nbands, chunk = blockIdx.x / p.nbands;
  const int h0 = band * C1D_HB;
  const int j0 = chunk * p.chunk, j1 = min(j0 + p.chunk, p.DP);              // plane pairs whose planes this CTA writes
  const int jlo = max(j0 - 1, 0), jhi = min(j1, p.DP - 1);                    // plane pairs it processes
  const int klo = max(h0 / 2 - 1, 0), khi = min(h0 / 2 + C1D_HB / 2, p.HP - 1);
  const int nk = khi - klo + 1;
  const int units = (jhi - jlo + 1) * nk;
  const int pw0 = 2 * j0, pw1 = min(2 * j1, p.D);                             // planes written: [pw0, pw1)

  // ---- set-up: barriers, B operand (w hi / lo), zeroed dy rows past the last window, accumulators, exchange pads
  if (threadIdx.x == 0) {
    for (int s = 0; s < 2; ++s) {
      mbar_init(built + 8 * s, C1D_BGROUP);
      mbar_init(mma_done + 8 * s, 1);
      mbar_init(tfree + 8 * s, 128);
    }
    fence_barrier_init();
  }
  if (warp == 4) {
    tmem_alloc(tmem_slot, 256);
    tmem_relinquish();
  }
  for (int i = threadIdx.x; i < 32 * 32; i += C1D_THREADS) {
    const int tap = i >> 5, co = i & 31;
    const float v = tap < 27 ? p.w[g][co * 27 + tap] : 0.f;
    const float hi = round_bf16(v);
    __nv_bfloat16* wh = reinterpret_cast<__nv_bfloat16*>(gen + C1D_OFF_W + c1d_sw64(tap, co >> 3)) + (co & 7);
    wh[0] = __float2bfloat16_rn(hi);
    wh[32 * 32] = __float2bfloat16_rn(v - hi);                 // lo half: 2 KB further
  }
  for (int i = threadIdx.x; i < 2 * 4 * 128 * 4; i += C1D_THREADS) {      // 16-byte chunks of rows >= 2*WC
    const int r = (i >> 2) & 127, t = i >> 9;
    if (r >= 2 * p.WC) *reinterpret_cast<uint4*>(gen + (uint32_t)t * C1D_TILE + c1d_sw64(r, i & 3)) = make_uint4(0u, 0u, 0u, 0u);
  }
  float* acc = reinterpret_cast<float*>(gen + C1D_OFF_ACC);                   // [4 planes][HB rows][128 w]
  float* xch = reinterpret_cast<float*>(gen + C1D_OFF_X);                     // [2 buffers][L, R][9][XW]
  for (int i = threadIdx.x; i < 4 * C1D_HB * 128; i += C1D_THREADS) acc[i] = 0.f;
  for (int i = threadIdx.x; i < 2 * 2 * 9 * C1D_XW; i += C1D_THREADS) xch[i] = 0.f;
  float* cf = reinterpret_cast<float*>(gen + C1D_OFF_COEF);                   // in shared memory: 32 registers fewer per builder
  if (!LRP && threadIdx.x < 32) {
    const int c = threadIdx.x;
    const float sc = p.coef[g][c], sh = p.coef[g][32 + c], mu = p.coef[g][64 + c], is = p.coef[g][96 + c];
    const float m1 = p.bcoef[g][c], m2 = p.bcoef[g][32 + c];
    const float b = -sc * m2 * is;
    cf[c] = -sc * m1 - b * mu;
    cf[32 + c] = b;
    cf[64 + c] = sc;
    cf[96 + c] = sh;
  }
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(gen + C1D_OFF_BAR + 48);
  float bsum = 0.f, esum = 0.f;                          // LRP: relevance entering block 1 (owned windows) / R_x written

  if (warp == 4) {
    // =========================================== MMA issuer =============================================
    const uint64_t dhi = make_smem_desc(0, 16, 512, LAYOUT_SW64, 0) & 0xFFFFFFFF00000000ull;
    const uint32_t dlo = (uint32_t)(make_smem_desc(0, 16, 512, LAYOUT_SW64, 0) & 0xFFFF0000ull);
    const uint32_t wh = dlo | (((sbase + C1D_OFF_W) & 0x3FFFFu) >> 4);
    const uint32_t wl = wh + ((32u * 64u) >> 4);
    for (int u = 0; u < units; ++u) {
      const int s = u & 1;
      const uint32_t ph = (uint32_t)(u >> 1) & 1u;
      mbar_wait(built + 8 * s, ph);
      if (u >= 2) mbar_wait(tfree + 8 * s, ph ^ 1u);
      tc_fence_after();
      if (elect_one()) {
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          const uint32_t a = dlo | (((sbase + (uint32_t)s * C1D_STAGE + (uint32_t)t * C1D_TILE) & 0x3FFFFu) >> 4);
          const uint32_t d = tmem_base + (uint32_t)(s * 128 + t * 32);
#pragma unroll
          for (int k = 0; k < 2; ++k) {
            mma_bf16_ss(d, dhi | (uint64_t)(a + 2u * k), dhi | (uint64_t)(wh + 2u * k), p.idesc, k ? 1u : 0u);
            mma_bf16_ss(d, dhi | (uint64_t)(a + 2u * k), dhi | (uint64_t)(wl + 2u * k), p.idesc, 1u);
          }
        }
        mma_commit(mma_done + 8 * s);
      }
      __syncwarp();
    }
  } else if (warp >= 5) {
    // =========================================== dy builders ============================================
    const int bt = threadIdx.x - 160;
    const int grp = bt / C1D_BGROUP, tb = bt % C1D_BGROUP;
    const int cq = tb & 3, c0 = cq * 8;                   // loop-invariant: the task stride (176) is a multiple of 4
    const uint64_t* cf2 = reinterpret_cast<const uint64_t*>(cf) + c0 / 2;     // channel pairs of A, Bc, scale, shift
    const __nv_bfloat16* yg = p.y[g];
    const int Do = p.D / 2, Ho = p.H / 2, Wo = p.W / 2;
    const int sH = p.W * 32, sD = p.H * p.W * 32;        // < 2^31: W <= 128 and H * W * 32 elements fit one plane
    const uint32_t stage = (uint32_t)grp * C1D_STAGE;
    for (int u = grp; u < units; u += 2) {
      const int j = jlo + u / nk, k = klo + u % nk;
      if (u >= 2) mbar_wait(mma_done + 8 * grp, (uint32_t)((u >> 1) - 1) & 1u);   // the stage's previous unit is consumed
      const bool exd = 2 * j + 1 < p.D, exh = 2 * k + 1 < p.H;
      const bool pool_ok = j < Do && k < Ho;
      const bool own = j >= j0 && j < j1 && 2 * k >= h0 && 2 * k < h0 + C1D_HB;      // LRP: windows this CTA accounts for
      const __nv_bfloat16* yu = yg + ((((int64_t)n * p.D + 2 * j) * p.H + 2 * k) * p.W) * 32 + c0;
      const __nv_bfloat16* gu = p.dout[g] + ((((int64_t)n * Do + j) * Ho + k) * Wo) * 32 + c0;
      for (int task = tb; task < p.WC * 4; task += C1D_BGROUP) {
        const int wo = task >> 2;
        const bool exw = 2 * wo + 1 < p.W;
        const bool win_ok = pool_ok && wo < Wo;
        uint4 raw[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          const bool ex = ((q & 4) ? exd : true) && ((q & 2) ? exh : true) && ((q & 1) ? exw : true);
          const int off = wo * 64 + ((q & 4) ? sD : 0) + ((q & 2) ? sH : 0) + ((q & 1) ? 32 : 0);
          raw[q] = ex ? __ldg(reinterpret_cast<const uint4*>(yu + off)) : make_uint4(0u, 0u, 0u, 0u);
        }
        if constexpr (LRP) {
          float R[8], sv[8];
          int wq[8];
#pragma unroll
          for (int c = 0; c < 8; ++c) R[c] = 0.f;
          if (win_ok) {
            float av[8], cv[8];
            unpack8(__ldg(reinterpret_cast<const uint4*>(p.a1[g] + (gu - p.dout[g]) + wo * 32)), av);
            unpack8(__ldg(reinterpret_cast<const uint4*>(gu + wo * 32)), cv);
#pragma unroll
            for (int c = 0; c < 8; ++c) {
              R[c] = __fmul_rn(av[c], cv[c]);
              if (own) bsum = __fadd_rn(bsum, R[c]);
            }
          }
#pragma unroll
          for (int c = 0; c < 8; ++c) {
            const auto ybf = [&](int q) {
              const uint32_t v = c1d_get(raw[q], c >> 1);
              return (c & 1) ? bf16_hi(v) : bf16_lo(v);
            };
            float m = ybf(0);
            wq[c] = 0;
#pragma unroll
            for (int q = 1; q < 8; ++q) {
              const float v = ybf(q);
              if (v > m) { m = v; wq[c] = q; }
            }
            if (p.zp[g] != nullptr && win_ok) {
              const int q = wq[c];
              const int off = wo * 64 + ((q & 4) ? sD : 0) + ((q & 2) ? sH : 0) + ((q & 1) ? 32 : 0);
              m = __bfloat162float(p.zp[g][(yu - yg) + off + c]);
            }
            sv[c] = win_ok ? lrp_div(R[c], m, p.eps) : 0.f;
          }
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            raw[q].x = pack_bf16(wq[0] == q ? sv[0] : 0.f, wq[1] == q ? sv[1] : 0.f);
            raw[q].y = pack_bf16(wq[2] == q ? sv[2] : 0.f, wq[3] == q ? sv[3] : 0.f);
            raw[q].z = pack_bf16(wq[4] == q ? sv[4] : 0.f, wq[5] == q ? sv[5] : 0.f);
            raw[q].w = pack_bf16(wq[6] == q ? sv[6] : 0.f, wq[7] == q ? sv[7] : 0.f);
          }
        } else {
        float go[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) go[i] = 0.f;
        if (win_ok) unpack8(__ldg(reinterpret_cast<const uint4*>(gu + wo * 32)), go);
        // the arithmetic of bn_maxpool_bwd_apply_kernel (bn_act_pool.cu), operation for operation
#pragma unroll
        for (int j2 = 0; j2 < 4; ++j2) {
          const uint64_t cA2 = cf2[j2], cB2 = cf2[16 + j2], sc2 = cf2[32 + j2], sh2 = cf2[48 + j2];
          const uint32_t flip = ((lo_u32(sc2) >> 16) & 0x8000u) | (hi_u32(sc2) & 0x80000000u);
          uint32_t key[8];
#pragma unroll
          for (int q = 0; q < 8; ++q) key[q] = c1d_get(raw[q], j2) ^ flip;
          const uint32_t m = c1d_bmax(c1d_bmax(c1d_bmax(key[0], key[1]), c1d_bmax(key[2], key[3])),
                                      c1d_bmax(c1d_bmax(key[4], key[5]), c1d_bmax(key[6], key[7])));
          const uint32_t ym = m ^ flip;
          const uint64_t z2 = fma2_f32(pair_f32(bf16_lo(ym), bf16_hi(ym)), sc2, sh2);
          const float z0 = __uint_as_float(lo_u32(z2)), z1 = __uint_as_float(hi_u32(z2));
          const float g0 = go[2 * j2], g1 = go[2 * j2 + 1];
          const float d0 = __uint_as_float(lo_u32(sc2)) * (z0 > 0.f ? g0 : g0 * p.slope);
          const float d1 = __uint_as_float(hi_u32(sc2)) * (z1 > 0.f ? g1 : g1 * p.slope);
          const uint64_t dz2 = pair_f32(d0, d1);
          uint32_t found = 0u;
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            const uint32_t eq = c1d_beq(key[q], m);
            const uint32_t sel = eq & ~found;
            found |= eq;
            const uint32_t yv = c1d_get(raw[q], j2);
            const uint64_t base = fma2_f32(cB2, pair_f32(bf16_lo(yv), bf16_hi(yv)), cA2);
            const uint64_t o2 = fma2_f32(pair_f32(bf16_lo(sel), bf16_hi(sel)), dz2, base);
            const uint32_t pk = pack_bf16(__uint_as_float(lo_u32(o2)), __uint_as_float(hi_u32(o2)));
            if (j2 == 0) raw[q].x = pk; else if (j2 == 1) raw[q].y = pk; else if (j2 == 2) raw[q].z = pk; else raw[q].w = pk;
          }
        }
        }
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          const bool ex = ((q & 4) ? exd : true) && ((q & 2) ? exh : true) && ((q & 1) ? exw : true);
          *reinterpret_cast<uint4*>(gen + stage + (uint32_t)(q >> 1) * C1D_TILE + c1d_sw64(2 * wo + (q & 1), cq)) =
              ex ? raw[q] : make_uint4(0u, 0u, 0u, 0u);
        }
      }
      fence_proxy_async();                                 // generic-proxy smem writes -> visible to the tensor core
      mbar_arrive(built + 8 * grp);
    }
  } else {
    // =========================================== epilogue ===============================================
    const int w = warp * 32 + lane;                       // TMEM lane = voxel column
    const uint32_t lane_base = tmem_base + ((uint32_t)(warp * 32) << 16);
    float* dxg = p.dx[g];
    int xb = 0;
    for (int u = 0; u < units; ++u) {
      const int s = u & 1;
      const int j = jlo + u / nk, k = klo + u % nk;
      mbar_wait(mma_done + 8 * s, (uint32_t)(u >> 1) & 1u);
      tc_fence_after();
#pragma unroll 1
      for (int t = 0; t < 4; ++t) {
        const int rd = 2 * j + (t >> 1), rh = 2 * k + (t & 1);
        if (rd >= p.D || rd < pw0 - 1 || rd > pw1 || rh >= p.H || rh < h0 - 1 || rh > h0 + C1D_HB) continue;
        uint32_t raw[32];
        tmem_ld32(lane_base + (uint32_t)(s * 128 + t * 32), raw);
        tmem_ld_wait();
        float* xl = xch + xb * (2 * 9 * C1D_XW);
        float* xr = xl + 9 * C1D_XW;
        xb ^= 1;
#pragma unroll
        for (int k9 = 0; k9 < 9; ++k9) {
          xl[k9 * C1D_XW + w + 1] = __uint_as_float(raw[3 * k9 + 0]);
          xr[k9 * C1D_XW + w + 1] = __uint_as_float(raw[3 * k9 + 2]);
        }
        asm volatile("bar.sync 1, 128;" ::: "memory");
        // V[kd][kh] at column w = q[w+1][kd,kh,0] + q[w][kd,kh,1] + q[w-1][kd,kh,2]; it lands on dx[rd+kd-1][rh+kh-1][w]
#pragma unroll
        for (int kd = 0; kd < 3; ++kd) {
          const int pd = rd + kd - 1;
          if (pd < 0 || pd >= p.D) continue;
          float* ap = acc + (pd & 3) * (C1D_HB * 128) + w;
#pragma unroll
          for (int kh = 0; kh < 3; ++kh) {
            const int k9 = kd * 3 + kh;
            const int hr = rh + kh - 1 - h0;
            const float v = (xl[k9 * C1D_XW + w + 2] + __uint_as_float(raw[3 * k9 + 1])) + xr[k9 * C1D_XW + w];
            if (hr >= 0 && hr < C1D_HB && h0 + hr < p.H) ap[hr * 128] += v;
          }
        }
      }
      tc_fence_before();
      mbar_arrive(tfree + 8 * s);
      if (k == khi) {
        // planes 2j-1 and 2j have all their contributions (and 2j+1 at the end of the volume): write, clear
        const int plast = (j == p.DP - 1) ? 2 * j + 1 : 2 * j;
        for (int pd = max(2 * j - 1, 0); pd <= plast && pd < p.D; ++pd) {
          float* ap = acc + (pd & 3) * (C1D_HB * 128) + w;
          const bool wr = pd >= pw0 && pd < pw1 && w < p.W;
          float* dst = dxg + (((int64_t)n * p.D + pd) * p.H + h0) * p.W + w;
          for (int hr = 0; hr < C1D_HB; ++hr) {
            if (wr && h0 + hr < p.H) {
              if constexpr (LRP) {
                const float v = __fmul_rn(p.x[g][(dst - dxg) + (int64_t)hr * p.W], ap[hr * 128]);
                dst[(int64_t)hr * p.W] = v;
                esum = __fadd_rn(esum, v);
              } else {
                dst[(int64_t)hr * p.W] = ap[hr * 128];
              }
            }
            ap[hr * 128] = 0.f;
          }
        }
      }
    }
  }
  float* red = reinterpret_cast<float*>(gen + C1D_OFF_BAR + 64);
  if constexpr (LRP) red[threadIdx.x] = warp >= 5 ? bsum : (warp < 4 ? esum : 0.f);
  tc_fence_before();
  __syncthreads();
  if (warp == 4) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 256);
  }
  if constexpr (LRP) {
    if (threadIdx.x == 0) {
      // fixed order: builders by thread index, then the epilogue columns by w
      float sb = 0.f, se = 0.f;
      for (int i = 160; i < C1D_THREADS; ++i) sb = __fadd_rn(sb, red[i]);
      for (int i = 0; i < 128; ++i) se = __fadd_rn(se, red[i]);
      float* pr = p.part[g] + ((int64_t)n * gridDim.x + blockIdx.x) * 2;
      pr[0] = sb;
      pr[1] = se;
    }
  }
}

// CUDA-core path: dx[p] = sum_tap sum_co dy[p - off(tap)][co] * w[co][tap] on a dy written by tmf_bn_act_pool_bwd_apply
// (fp32 weights, fixed summation order).  Serves TMF_CONV_DIRECT and the problems the tcgen05 kernel refuses.
__global__ void __launch_bounds__(256) conv1_dgrad_direct_kernel(GroupPtr<const __nv_bfloat16> dy, GroupPtr<const float> w,
                                                                 GroupPtr<float> dx, int B, int D, int H, int W, int cout) {
  __shared__ float ws[27 * 64];
  const int g = blockIdx.z;
  for (int i = threadIdx.x; i < 27 * cout; i += blockDim.x) ws[(i % 27) * cout + i / 27] = w.p[g][i];   // [tap][co]
  __syncthreads();
  const int64_t total = (int64_t)B * D * H * W;
  for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < total; v += (int64_t)gridDim.x * blockDim.x) {
    int64_t t = v;
    const int x = (int)(t % W); t /= W;
    const int y = (int)(t % H); t /= H;
    const int z = (int)(t % D);
    const int nb = (int)(t / D);
    float acc = 0.f;
    for (int tap = 0; tap < 27; ++tap) {
      const int rz = z - (tap / 9 - 1), ry = y - ((tap / 3) % 3 - 1), rx = x - (tap % 3 - 1);
      if (rz < 0 || rz >= D || ry < 0 || ry >= H || rx < 0 || rx >= W) continue;
      const __nv_bfloat16* src = dy.p[g] + ((((int64_t)nb * D + rz) * H + ry) * W + rx) * cout;
      for (int c = 0; c < cout; c += 8) {
        float f[8];
        unpack8(*reinterpret_cast<const uint4*>(src + c), f);
#pragma unroll
        for (int e = 0; e < 8; ++e) acc = fmaf(f[e], ws[tap * cout + c + e], acc);
      }
    }
    dx.p[g][v] = acc;
  }
}

struct C1DPlan {
  bool umma;
  int nbands, chunk, nchunks;
};

static bool c1d_umma_supported(int ng, int B, int D, int H, int W, int cout) {
  if (getenv("TMF_DISABLE_UMMA") != nullptr) return false;
  return cout == 32 && ng >= 1 && ng <= TMF_MAX_GROUPS && B >= 1 && B <= 65535 && D >= 1 && H >= 1 && W >= 1 && W <= 128;
}

// Grid: one CTA per (band, chunk of plane pairs, image, tower).  The chunk length trades the halo plane pair recomputed at
// each end of a chunk against filling the SMs: pick the one with the least (waves x longest chunk).
static C1DPlan c1d_plan(int ng, int B, int D, int H) {
  C1DPlan pl{};
  pl.nbands = (H + C1D_HB - 1) / C1D_HB;
  const int DP = (D + 1) / 2;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const long long cols = (long long)ng * B * pl.nbands;
  long long best = -1;
  for (int c = 1; c <= DP; ++c) {
    const int nch = (DP + c - 1) / c;
    if (nch * pl.nbands > 65535) continue;
    long long longest = 0;
    for (int i = 0; i < nch; ++i) {
      const int j0 = i * c, j1 = std::min(j0 + c, DP);
      longest = std::max(longest, (long long)(std::min(j1, DP - 1) - std::max(j0 - 1, 0) + 1));
    }
    const long long waves = (cols * nch + sms - 1) / sms;
    const long long cost = waves * longest;
    if (best < 0 || cost < best) { best = cost; pl.chunk = c; pl.nchunks = nch; }
  }
  return pl;
}

static size_t c1d_direct_ws(int ng, int B, int D, int H, int W, int cout) {
  return (size_t)ng * ((((size_t)B * D * H * W * cout * 2) + 255) & ~(size_t)255);
}

size_t lrp_ratio_ws(int ng, int B, int D, int H, int W, int C, int pool);
int lrp_blocks(int64_t items);
int lrp_sum_rows(int ng, float* const* part, float* const* totals, int B, int rows, int K, int col, cudaStream_t st);
int lrp_xmul(int ng, const float* const* x, float* const* rx, float* const* totals, int col, int B, int64_t per, float* part,
             cudaStream_t st);

static size_t c1d_align(size_t b) { return (b + 255) & ~(size_t)255; }

// LRP on the CUDA-core path: [s (bf16, per tower)] [ratio partial rows] [x-multiply partial rows]
static size_t c1d_lrp_direct_ws(int ng, int B, int D, int H, int W, int cout) {
  return c1d_direct_ws(ng, B, D, H, W, cout) + lrp_ratio_ws(ng, B, D, H, W, cout, TMF_POOL_MAX) +
         c1d_align((size_t)ng * B * lrp_blocks((int64_t)D * H * W) * sizeof(float));
}

// The tcgen05 LRP instance plans its grid as for two towers whatever ng is: the per-CTA partial rows of the totals then
// cover the same voxels, and a tower's totals do not depend on whether it runs alone or paired.
static C1DPlan c1d_lrp_plan(int B, int D, int H) { return c1d_plan(TMF_MAX_GROUPS, B, D, H); }

}  // namespace tmf

using namespace tmf;

extern "C" {

int tmf_bn_act_pool_bwd_apply(int ng, const void* const* dout, int dout_fp32, const void* const* y,
                              const float* const* coef, const float* const* bcoef, void* const* dy, int B, int D,
                              int H, int W, int C, int pool, float slope, void* stream);

int64_t tmf_conv1_dgrad_fused_workspace_bytes(int ng, int impl, int B, int D, int H, int W, int cout) {
  if (impl == TMF_CONV_AUTO) impl = c1d_umma_supported(ng, B, D, H, W, cout) ? TMF_CONV_UMMA : TMF_CONV_DIRECT;
  return impl == TMF_CONV_DIRECT ? (int64_t)c1d_direct_ws(ng, B, D, H, W, cout) : 0;
}

int tmf_conv1_dgrad_fused(int ng, const void* const* dout, const void* const* y, const float* const* coef,
                          const float* const* bcoef, const float* const* w, float* const* dx, int B, int D, int H, int W,
                          int cout, float slope, int impl, void* ws, size_t ws_bytes, void* stream) {
  TMF_CHECK_NG(ng);
  TMF_REQUIRE(B >= 1 && D >= 1 && H >= 1 && W >= 1, "conv1_dgrad_fused: empty problem (%d,%d,%d,%d)", B, D, H, W);
  if (impl == TMF_CONV_AUTO) impl = c1d_umma_supported(ng, B, D, H, W, cout) ? TMF_CONV_UMMA : TMF_CONV_DIRECT;
  cudaStream_t st = (cudaStream_t)stream;
  for (int g = 0; g < ng; ++g) {
    TMF_REQUIRE(dout && y && coef && bcoef && w && dx && dout[g] && y[g] && coef[g] && bcoef[g] && w[g] && dx[g],
                "conv1_dgrad_fused: NULL device pointer");
    TMF_REQUIRE(((uintptr_t)dout[g] & 15) == 0 && ((uintptr_t)y[g] & 15) == 0, "conv1_dgrad_fused: dout / y must be 16-byte aligned");
  }
  if (impl == TMF_CONV_UMMA) {
    TMF_REQUIRE(c1d_umma_supported(ng, B, D, H, W, cout), "conv1_dgrad_fused: tcgen05 path needs Cout = 32 and W <= 128 (got Cout=%d, W=%d)",
                cout, W);
    const C1DPlan pl = c1d_plan(ng, B, D, H);
    C1DParams p{};
    for (int g = 0; g < ng; ++g) {
      p.y[g] = (const __nv_bfloat16*)y[g];
      p.dout[g] = (const __nv_bfloat16*)dout[g];
      p.coef[g] = coef[g];
      p.bcoef[g] = bcoef[g];
      p.w[g] = w[g];
      p.dx[g] = dx[g];
    }
    p.B = B; p.D = D; p.H = H; p.W = W;
    p.DP = (D + 1) / 2; p.HP = (H + 1) / 2; p.WC = (W + 1) / 2;
    p.nbands = pl.nbands; p.chunk = pl.chunk;
    p.idesc = make_idesc_bf16(128, 32, 0, 0);
    p.slope = slope;
    static bool attr_done = false;
    if (!attr_done) {
      TMF_CUDA(cudaFuncSetAttribute(conv1_dgrad_umma_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C1D_SMEM));
      attr_done = true;
    }
    launch_k(conv1_dgrad_umma_kernel<false>, dim3(pl.nbands * pl.nchunks, B, ng), C1D_THREADS, C1D_SMEM, st, p);
    TMF_LAUNCH_CHECK();
    return 0;
  }
  TMF_REQUIRE(impl == TMF_CONV_DIRECT, "conv1_dgrad_fused: unknown impl %d", impl);
  TMF_REQUIRE(cout >= 8 && cout <= 64 && cout % 8 == 0, "conv1_dgrad_fused: Cout must be a multiple of 8 in [8,64] (got %d)", cout);
  const size_t per = c1d_direct_ws(1, B, D, H, W, cout);
  TMF_REQUIRE(ws != nullptr && ws_bytes >= (size_t)ng * per && ((uintptr_t)ws & 255) == 0,
              "conv1_dgrad_fused: the CUDA-core path needs a 256-byte aligned workspace of %zu bytes (got %zu)",
              (size_t)ng * per, ws_bytes);
  void* dyp[TMF_MAX_GROUPS] = {nullptr, nullptr};
  for (int g = 0; g < ng; ++g) dyp[g] = (uint8_t*)ws + (size_t)g * per;
  if (tmf_bn_act_pool_bwd_apply(ng, dout, 0, y, coef, bcoef, dyp, B, D, H, W, cout, TMF_POOL_MAX, slope, stream) != 0) return 1;
  GroupPtr<const __nv_bfloat16> gdy;
  GroupPtr<const float> gw;
  GroupPtr<float> gdx;
  if (!load_group(gdy, (const __nv_bfloat16* const*)dyp, ng, true, "dy") || !load_group(gw, w, ng, true, "w") ||
      !load_group(gdx, dx, ng, true, "dx"))
    return 1;
  const long long total = (long long)B * D * H * W;
  dim3 grid((unsigned)std::min((total + 255) / 256, 148LL * 16), 1, ng);
  launch_k(conv1_dgrad_direct_kernel, grid, 256, 0, st, gdy, gw, gdx, B, D, H, W, cout);
  TMF_LAUNCH_CHECK();
  return 0;
}

int tmf_lrp_ratio(int ng, const void* const* up_a, const void* const* up_c, int up_fp32, const void* const* y,
                  const void* const* zp, void* const* s, float* const* totals, int col, int B, int D, int H, int W, int C,
                  int pool, float slope, float eps, void* ws, size_t ws_bytes, void* stream);

int tmf_lrp_conv1_impl(int ng, int impl, int B, int D, int H, int W, int cout) {
  if (impl == TMF_CONV_AUTO) impl = c1d_umma_supported(ng, B, D, H, W, cout) ? TMF_CONV_UMMA : TMF_CONV_DIRECT;
  return impl;
}

int64_t tmf_lrp_conv1_workspace_bytes(int ng, int impl, int B, int D, int H, int W, int cout) {
  impl = tmf_lrp_conv1_impl(ng, impl, B, D, H, W, cout);
  if (impl == TMF_CONV_DIRECT) return (int64_t)c1d_lrp_direct_ws(ng, B, D, H, W, cout);
  const C1DPlan pl = c1d_lrp_plan(B, D, H);
  return (int64_t)c1d_align((size_t)ng * B * pl.nbands * pl.nchunks * 2 * sizeof(float));
}

int tmf_lrp_conv1(int ng, const void* const* a1, const void* const* c1, const void* const* y, const void* const* zp,
                  const float* const* w, const float* const* x, float* const* rx, float* const* totals, int B, int D, int H,
                  int W, int cout, float eps, int impl, void* ws, size_t ws_bytes, void* stream) {
  TMF_CHECK_NG(ng);
  TMF_REQUIRE(B >= 1 && B <= 65535 && D >= 1 && H >= 1 && W >= 1, "lrp_conv1: empty problem (%d,%d,%d,%d)", B, D, H, W);
  TMF_REQUIRE(eps >= 0.f, "lrp_conv1: eps must be >= 0");
  impl = tmf_lrp_conv1_impl(ng, impl, B, D, H, W, cout);
  cudaStream_t st = (cudaStream_t)stream;
  for (int g = 0; g < ng; ++g) {
    TMF_REQUIRE(a1 && c1 && y && w && x && rx && totals && a1[g] && c1[g] && y[g] && w[g] && x[g] && rx[g] && totals[g],
                "lrp_conv1: NULL device pointer");
    TMF_REQUIRE((((uintptr_t)a1[g] | (uintptr_t)c1[g] | (uintptr_t)y[g]) & 15) == 0,
                "lrp_conv1: a1 / c1 / y must be 16-byte aligned");
  }
  const int64_t need = tmf_lrp_conv1_workspace_bytes(ng, impl, B, D, H, W, cout);
  TMF_REQUIRE(ws != nullptr && ws_bytes >= (size_t)need && ((uintptr_t)ws & 255) == 0,
              "lrp_conv1: needs a 256-byte aligned workspace of %lld bytes (got %zu)", (long long)need, ws_bytes);
  if (impl == TMF_CONV_UMMA) {
    TMF_REQUIRE(c1d_umma_supported(ng, B, D, H, W, cout), "lrp_conv1: tcgen05 path needs Cout = 32 and W <= 128 (got Cout=%d, W=%d)",
                cout, W);
    const C1DPlan pl = c1d_lrp_plan(B, D, H);
    const int rows = pl.nbands * pl.nchunks;
    C1DParams p{};
    float* part[TMF_MAX_GROUPS] = {nullptr, nullptr};
    for (int g = 0; g < ng; ++g) {
      p.y[g] = (const __nv_bfloat16*)y[g];
      p.dout[g] = (const __nv_bfloat16*)c1[g];
      p.a1[g] = (const __nv_bfloat16*)a1[g];
      p.zp[g] = zp != nullptr ? (const __nv_bfloat16*)zp[g] : nullptr;
      p.w[g] = w[g];
      p.x[g] = x[g];
      p.dx[g] = rx[g];
      part[g] = p.part[g] = (float*)ws + (size_t)g * B * rows * 2;
    }
    p.B = B; p.D = D; p.H = H; p.W = W;
    p.DP = (D + 1) / 2; p.HP = (H + 1) / 2; p.WC = (W + 1) / 2;
    p.nbands = pl.nbands; p.chunk = pl.chunk;
    p.idesc = make_idesc_bf16(128, 32, 0, 0);
    p.eps = eps;
    static bool attr_done = false;
    if (!attr_done) {
      TMF_CUDA(cudaFuncSetAttribute(conv1_dgrad_umma_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C1D_SMEM_LRP));
      attr_done = true;
    }
    launch_k(conv1_dgrad_umma_kernel<true>, dim3(rows, B, ng), C1D_THREADS, C1D_SMEM_LRP, st, p);
    TMF_LAUNCH_CHECK();
    return lrp_sum_rows(ng, part, totals, B, rows, 2, 6, st);
  }
  TMF_REQUIRE(impl == TMF_CONV_DIRECT, "lrp_conv1: unknown impl %d", impl);
  TMF_REQUIRE(cout >= 8 && cout <= 64 && cout % 8 == 0, "lrp_conv1: Cout must be a multiple of 8 in [8,64] (got %d)", cout);
  // s at full resolution (the ratio pass with block 1's max-pool), then the fp32 direct data gradient, then x * c
  const size_t per = c1d_direct_ws(1, B, D, H, W, cout);
  const size_t rws = lrp_ratio_ws(ng, B, D, H, W, cout, TMF_POOL_MAX);
  void* sp[TMF_MAX_GROUPS] = {nullptr, nullptr};
  for (int g = 0; g < ng; ++g) sp[g] = (uint8_t*)ws + (size_t)g * per;
  uint8_t* rbase = (uint8_t*)ws + (size_t)ng * per;
  if (tmf_lrp_ratio(ng, a1, c1, 0, y, zp, sp, totals, 6, B, D, H, W, cout, TMF_POOL_MAX, 0.f, eps, rbase, rws, stream) != 0)
    return 1;
  GroupPtr<const __nv_bfloat16> gs;
  GroupPtr<const float> gw;
  GroupPtr<float> gx;
  if (!load_group(gs, (const __nv_bfloat16* const*)sp, ng, true, "s") || !load_group(gw, w, ng, true, "w") ||
      !load_group(gx, rx, ng, true, "rx"))
    return 1;
  const long long total = (long long)B * D * H * W;
  dim3 grid((unsigned)std::min((total + 255) / 256, 148LL * 16), 1, ng);
  launch_k(conv1_dgrad_direct_kernel, grid, 256, 0, st, gs, gw, gx, B, D, H, W, cout);
  TMF_LAUNCH_CHECK();
  return lrp_xmul(ng, x, rx, totals, 7, B, (int64_t)D * H * W, (float*)(rbase + rws), st);
}

}  // extern "C"

// conv1_bwd_fused.cu -- backward of sNet block 1 in ONE pass over y:
//   BatchNorm3d(train|eval) + LeakyReLU + MaxPool3d(2,2) backward "apply"  (reference models/networks.py:23-25)
//   fused with the conv1.0 weight gradient                                   (reference models/networks.py:22)
//
// conv1.0's input is the image, so dy of block 1 feeds nothing but the weight gradient.  The unfused path wrote
// dy (57.8 MB per subject-modality) and read it back; here dy only ever exists in shared memory.
//
// Work unit = one pooling row-quad (n, dp, hp): planes 2dp, 2dp+1 x rows 2hp, 2hp+1 x all w -- four "segments" of
// P = roundup16(W) voxel rows (64 B = 32 channels each), i.e. exactly the voxels of one row of pooling windows.
//   * TMA brings the raw y segments (one 5-D box, zero fill past W / H / D), the pooled gradient row and the image
//     patches into a shared-memory stage;
//   * builder warps turn y into dy IN PLACE (window arg-max on the stored bf16 y with torch's first-maximum rule,
//     dy = A + Bc*y (+ scale*dz at the arg-max), see bn_act_pool.cu), two groups alternating units;
//   * one tcgen05.mma per 16 voxels:  D[(seg,co), n] += sum_k dy[seg][k][co] * xs[n][k]
//       A (M = 128) = the four segments stacked along M (MN-major, 64B swizzle, LBO = segment stride),
//       B (N = 96)  = image patches, K-major: row n = (dd, hh, hl, kw) holds xhl(2dp-1+dd, 2hp-1+hh, k+kw-1) for the
//                     16 (plane,row) pairs around the quad, the bf16 hi / lo halves of the fp32 image and the three
//                     kw shifts (a pre-pass writes the six shifted bf16 rows per image row -- TMA cannot start a box
//                     at a 2-byte offset -- so ONE 5-D box per 32 voxels lands the whole operand),
//     so dW[co][kd][kh][kw] = sum over seg=(ds,hs), hl of D[(seg,co)][(ds+kd, hs+kh, hl, kw)].
//   * accumulators stay in TMEM (96 columns) for the CTA's whole unit range; per-CTA partials are summed in a fixed
//     order (deterministic).
#include <cuda.h>

#include "common.cuh"
#include "umma.cuh"

namespace tmf {
using namespace umma;

constexpr int C1B_GROUP_THREADS = 192;                 // builder group: 6 warps
constexpr int C1B_GROUPS = 2;
constexpr int C1B_THREADS = 64 + C1B_GROUPS * C1B_GROUP_THREADS;   // warp 0: TMA, warp 1: MMA / TMEM, warps 2..13: builders
constexpr int C1B_MAX_STAGES = 4;
constexpr int C1B_NCOLS = 96;                          // (dd 4) x (hh 4) x (hl 2) x (kw 3)

struct alignas(64) C1BParams {
  CUtensorMap tmY[TMF_MAX_GROUPS];
  CUtensorMap tmG[TMF_MAX_GROUPS];
  CUtensorMap tmX[TMF_MAX_GROUPS];
  const float* coef[TMF_MAX_GROUPS];
  const float* bcoef[TMF_MAX_GROUPS];
  float* part[TMF_MAX_GROUPS];                         // [ncta][32*27] per-CTA partial dW
  int ng, B, D, H, W, P, DP, HP, WC, units, ksteps, kblocks, stages;
  uint32_t y_bytes, x_bytes, g_bytes, x_off, g_off, stage_bytes, tx_bytes;
  uint32_t idesc;
  float slope;
};

// fp32 image (B*D*H rows of W) -> six bf16 rows of pitch P per image row: x6[row][hl*3+kw][k] = hl-part of x[k+kw-1]
// (zero outside [0,W)); hl = 0: bf16(x), hl = 1: bf16(x - bf16(x)).
__global__ void conv1_split_x_kernel(GroupPtr<const float> x, GroupPtr<__nv_bfloat16> x6, int rows, int W, int P) {
  const int g = blockIdx.z;
  const int chunks = P >> 3;
  const unsigned total = (unsigned)rows * (unsigned)chunks;
  for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const unsigned row = i / chunks, ch = i - row * chunks;
    const float* xr = x.p[g] + (size_t)row * W;
    float v[10], hi[10], lo[10];
#pragma unroll
    for (int j = 0; j < 10; ++j) {
      const int k = (int)ch * 8 + j - 1;
      v[j] = (k >= 0 && k < W) ? __ldg(xr + k) : 0.f;
      hi[j] = round_bf16(v[j]);
      lo[j] = v[j] - hi[j];
    }
    __nv_bfloat16* dst = x6.p[g] + (size_t)row * 6 * P + (size_t)ch * 8;
#pragma unroll
    for (int kw = 0; kw < 3; ++kw) {
      *reinterpret_cast<uint4*>(dst + (size_t)kw * P) = pack8(&hi[kw]);
      *reinterpret_cast<uint4*>(dst + (size_t)(3 + kw) * P) = pack8(&lo[kw]);
    }
  }
}

__global__ void __launch_bounds__(C1B_THREADS, 1) conv1_bwd_fused_kernel(const __grid_constant__ C1BParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t bars = smem_base + (uint32_t)p.stages * p.stage_bytes;
  const uint32_t tma_full = bars, built = bars + 8 * C1B_MAX_STAGES, empty = built + 8 * C1B_MAX_STAGES;
  const uint32_t acc_full = empty + 8 * C1B_MAX_STAGES, tmem_slot = acc_full + 8;
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(gen + (tmem_slot - smem_base));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = blockIdx.x % p.ng;
  const int cta = blockIdx.x / p.ng, ncta = gridDim.x / p.ng;

  if (threadIdx.x == 0) {
    for (int i = 0; i < p.stages; ++i) {
      mbar_init(tma_full + 8 * i, 1);
      mbar_init(built + 8 * i, C1B_GROUP_THREADS);
      mbar_init(empty + 8 * i, 1);
    }
    mbar_init(acc_full, 1);
    fence_barrier_init();
    prefetch_tmap(&p.tmY[g]);
    prefetch_tmap(&p.tmG[g]);
    prefetch_tmap(&p.tmX[g]);
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, 128);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp == 0) {
    // =========================================== TMA producer ===========================================
    if (lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      for (int u = cta; u < p.units; u += ncta) {
        int t = u;
        const int hp = t % p.HP; t /= p.HP;
        const int dp = t % p.DP;
        const int n = t / p.DP;
        mbar_wait(empty + 8 * s, ph ^ 1u);
        mbar_expect_tx(tma_full + 8 * s, p.tx_bytes);
        const uint32_t st = smem_base + (uint32_t)s * p.stage_bytes;
        tma_load_5d(st, &p.tmY[g], tma_full + 8 * s, 0, 0, 2 * hp, 2 * dp, n);
        tma_load_5d(st + p.g_off, &p.tmG[g], tma_full + 8 * s, 0, 0, hp, dp, n);
        for (int kb = 0; kb < p.kblocks; ++kb)
          tma_load_5d(st + p.x_off + (uint32_t)kb * (C1B_NCOLS * 64u), &p.tmX[g], tma_full + 8 * s, 32 * kb, 0, 2 * hp - 1,
                      2 * dp - 1, n);
        if (++s == p.stages) { s = 0; ph ^= 1u; }
      }
    }
  } else if (warp == 1) {
    // =========================================== MMA issuer =============================================
    int s = 0;
    uint32_t ph = 0;
    const uint32_t seg_bytes = (uint32_t)p.P * 64u;
    const uint64_t hi_a = make_smem_desc(0, seg_bytes, 512, LAYOUT_SW64, 0) & 0xFFFFFFFF00000000ull;      // MN-major dy
    const uint32_t a_const = (uint32_t)(make_smem_desc(0, seg_bytes, 512, LAYOUT_SW64, 0) & 0xFFFF0000ull);
    const uint64_t hi_b = make_smem_desc(0, 16, 512, LAYOUT_SW64, 0) & 0xFFFFFFFF00000000ull;            // K-major patches
    const uint32_t b_const = (uint32_t)(make_smem_desc(0, 16, 512, LAYOUT_SW64, 0) & 0xFFFF0000ull);
    uint32_t accumulate = 0;
    for (int u = cta; u < p.units; u += ncta) {
      mbar_wait(built + 8 * s, ph);
      tc_fence_after();
      const uint32_t st = smem_base + (uint32_t)s * p.stage_bytes;
      const uint32_t a_lo = a_const | ((st & 0x3FFFFu) >> 4);
      const uint32_t b_lo = b_const | (((st + p.x_off) & 0x3FFFFu) >> 4);
      if (elect_one()) {
        for (int k = 0; k < p.ksteps; ++k) {
          const uint32_t aoff = (uint32_t)k * ((16u * 64u) >> 4);
          const uint32_t boff = (uint32_t)(k >> 1) * ((C1B_NCOLS * 64u) >> 4) + (uint32_t)(k & 1) * 2u;
          mma_bf16_ss(tmem_base, hi_a | (uint64_t)(a_lo + aoff), hi_b | (uint64_t)(b_lo + boff), p.idesc,
                      (accumulate | (uint32_t)k) ? 1u : 0u);
        }
        mma_commit(empty + 8 * s);
      }
      __syncwarp();
      accumulate = 1;
      if (++s == p.stages) { s = 0; ph ^= 1u; }
    }
    if (elect_one()) mma_commit(acc_full);
    __syncwarp();
  } else {
    // =========================================== dy builders ============================================
    // ALU diet (this pass is instruction-bound if written element by element):
    //  * the window arg-max runs on PACKED bf16 pairs: key = (y & and) ^ xor puts sign(scale) into the sign bit
    //    (and = 0 for scale == 0: every key equal, the first voxel wins like in torch), HMNMX2 for the maximum,
    //    HSET2 equality masks + a 16-bit unsigned min over voxel numbers for "first maximum in (d,h,w) order";
    //  * the dense part is one FFMA per element, dy = A + Bc*y, with no dependence on the arg-max;
    //  * the single arg-max voxel of each (window, channel) is then patched with a 2-byte store of
    //    bf16(A + Bc*ybest + scale*dz) -- same value, same single rounding as the two-step kernels.
    // Bank conflicts: rows 2wo and 2wo+1 of a segment are 128 contiguous bytes, but rows of equal parity share banks;
    // odd windows therefore load / store their two rows in swapped order, so the 8 lanes of a quarter-warp (two
    // windows x four chunks) always cover all 32 banks.
    const int bt = threadIdx.x - 64;
    const int grp = bt / C1B_GROUP_THREADS, tb = bt % C1B_GROUP_THREADS;
    const int cq = tb & 3;                               // this thread's 8-channel chunk (loop-invariant)
    const int b = (tb >> 2) & 1;                         // window parity (loop-invariant: the task stride is 48 windows)
    const int c0 = cq * 8;
    float sc[8], sh[8], cA[8], cB[8];
    uint32_t kand[4], kxor[4];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float scale = p.coef[g][c0 + j], mean = p.coef[g][64 + c0 + j], invstd = p.coef[g][96 + c0 + j];
      const float m1 = p.bcoef[g][c0 + j], m2 = p.bcoef[g][32 + c0 + j];
      sc[j] = scale;
      sh[j] = p.coef[g][32 + c0 + j];
      cB[j] = -scale * m2 * invstd;
      cA[j] = -scale * m1 - cB[j] * mean;
      const uint32_t ka = scale != 0.f ? 0xFFFFu : 0u, kx = scale < 0.f ? 0x8000u : 0u;
      if (j & 1) { kand[j >> 1] |= ka << 16; kxor[j >> 1] |= kx << 16; }
      else { kand[j >> 1] = ka; kxor[j >> 1] = kx; }
    }
    uint32_t qc[8];                                       // voxel number (d,h,w scan order) held by load slot i, both halves
#pragma unroll
    for (int i = 0; i < 8; ++i) qc[i] = (uint32_t)((i & 6) | ((i & 1) ^ b)) * 0x00010001u;
    const uint32_t seg_bytes = (uint32_t)p.P * 64u;
    const uint32_t eoff[2] = {(uint32_t)b * 64u, (uint32_t)(1 - b) * 64u};     // row offset of load slot parity 0 / 1
    const int ntask = p.WC * 4;
    int it = grp;
    for (int u = cta + grp * ncta; u < p.units; u += C1B_GROUPS * ncta, it += C1B_GROUPS) {
      const int s = it % p.stages;
      const uint32_t ph = (uint32_t)(it / p.stages) & 1u;
      int t = u;
      const int hp = t % p.HP; t /= p.HP;
      const int dp = t % p.DP;
      const bool d1 = 2 * dp + 1 < p.D, h1 = 2 * hp + 1 < p.H;
      uint8_t* stage = gen + (size_t)s * p.stage_bytes;
      mbar_wait(tma_full + 8 * s, ph);
      for (int task = tb; task < ntask; task += C1B_GROUP_THREADS) {
        const int wo = task >> 2;
        const bool w1 = 2 * wo + 1 < p.W;
        const bool win_ok = d1 && h1 && w1;
        // 64B-swizzled chunk position (row >> 1 = wo for both rows of the window)
        uint8_t* base = stage + (uint32_t)(2 * wo) * 64u + (uint32_t)((cq ^ (wo & 3)) << 4);
        const uint4 gov = *reinterpret_cast<const uint4*>(stage + p.g_off + (uint32_t)wo * 64u + (uint32_t)cq * 16u);
        uint4 X[8];
#pragma unroll
        for (int i = 0; i < 8; ++i)
          X[i] = *reinterpret_cast<const uint4*>(base + (uint32_t)(i >> 1) * seg_bytes + eoff[i & 1]);
        uint32_t mx[4], idx[4];
        if (win_ok) {
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            uint32_t key[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const uint32_t v = c == 0 ? X[i].x : (c == 1 ? X[i].y : (c == 2 ? X[i].z : X[i].w));
              key[i] = (v & kand[c]) ^ kxor[c];
            }
            __nv_bfloat162 m = *reinterpret_cast<__nv_bfloat162*>(&key[0]);
#pragma unroll
            for (int i = 1; i < 8; ++i) m = __hmax2(m, *reinterpret_cast<__nv_bfloat162*>(&key[i]));
            uint32_t first = 0x000F000Fu;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const uint32_t eq = __heq2_mask(*reinterpret_cast<__nv_bfloat162*>(&key[i]), m);
              first = __vminu2(first, (qc[i] & eq) | (0x000F000Fu & ~eq));
            }
            mx[c] = *reinterpret_cast<uint32_t*>(&m);
            idx[c] = first;
          }
        }
        // dense part: dy = A + Bc*y for every existing voxel of the window
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const bool ex = ((i >> 2) == 0 || d1) && (((i >> 1) & 1) == 0 || h1) && ((((i & 1) ^ b) == 0) || w1);
          if (!ex) continue;
          float f[8], o[8];
          unpack8(X[i], f);
#pragma unroll
          for (int j = 0; j < 8; ++j) o[j] = fmaf(cB[j], f[j], cA[j]);
          *reinterpret_cast<uint4*>(base + (uint32_t)(i >> 1) * seg_bytes + eoff[i & 1]) = pack8(o);
        }
        // arg-max voxel of each channel: + scale*dz  (2-byte patch, program order after the dense store)
        if (win_ok) {
          float go[8];
          unpack8(gov, go);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const int c = j >> 1, sft = (j & 1) * 16;
            const uint32_t a = (idx[c] >> sft) & 7u;
            const uint32_t ybits = ((mx[c] ^ kxor[c]) >> sft) & 0xFFFFu;
            const float ybest = __uint_as_float(ybits << 16);
            const float z = fmaf(ybest, sc[j], sh[j]);
            const float dz = z > 0.f ? go[j] : go[j] * p.slope;
            const float o = fmaf(cB[j], ybest, cA[j]) + sc[j] * dz;
            *reinterpret_cast<__nv_bfloat16*>(base + (a >> 1) * seg_bytes + (a & 1u) * 64u + 2u * j) = __float2bfloat16_rn(o);
          }
        }
      }
      fence_proxy_async();                               // generic-proxy smem writes -> visible to the tensor core
      mbar_arrive(built + 8 * s);
    }
    // ---- epilogue (warps 2..5 = TMEM lane quarters 2,3,0,1): D -> smem -> fixed-order fold -> per-CTA partial
    float* fold = reinterpret_cast<float*>(gen);         // [128][96] floats, reuses stage 0 (all MMAs have completed)
    if (warp < 6) {
      mbar_wait(acc_full, 0u);
      tc_fence_after();
      const int quarter = warp & 3;
      const int m = quarter * 32 + lane;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        uint32_t raw[32];
        tmem_ld32(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(c * 32), raw);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) fold[m * C1B_NCOLS + c * 32 + j] = __uint_as_float(raw[j]);
      }
      tc_fence_before();
      asm volatile("bar.sync 1, 128;" ::: "memory");
      float* part = p.part[g] + (size_t)cta * (32 * 27);
      for (int i = threadIdx.x - 64; i < 32 * 27; i += 128) {
        const int co = i / 27, tap = i - co * 27;
        const int kd = tap / 9, kh = (tap / 3) % 3, kw = tap % 3;
        float acc = 0.f;
#pragma unroll
        for (int seg = 0; seg < 4; ++seg) {
          const int col = ((seg >> 1) + kd) * 24 + ((seg & 1) + kh) * 6 + kw;
          const float* rowp = fold + (seg * 32 + co) * C1B_NCOLS;
          acc += rowp[col] + rowp[col + 3];
        }
        part[i] = acc;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 128);
  }
}

// dw[co][tap] = sum over CTAs of part[cta][co*27+tap], fixed order
__global__ void conv1_bwd_reduce_kernel(GroupPtr<const float> part, GroupPtr<float> dw, int ncta) {
  const int g = blockIdx.z;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 32 * 27) return;
  float s = 0.f;
  for (int c = 0; c < ncta; ++c) s += part.p[g][(size_t)c * (32 * 27) + i];
  dw.p[g][i] = s;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn c1b_encode_fn() {
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

struct C1BPlan {
  bool ok;
  int P, DP, HP, WC, ksteps, kblocks, stages, ncta;
  uint32_t y_bytes, x_bytes, g_bytes, x_off, g_off, stage_bytes, smem_bytes;
  size_t x6_elems, ws_bytes;
};

static C1BPlan c1b_plan(int ng, int B, int D, int H, int W, int cout) {
  C1BPlan pl{};
  pl.ok = false;
  if (getenv("TMF_DISABLE_UMMA") != nullptr) return pl;
  if (cout != 32 || ng < 1 || ng > TMF_MAX_GROUPS) return pl;
  if (D < 2 || H < 2 || W < 2 || W > 240) return pl;
  if ((long long)B * D * H * ((W + 15) / 8) >= (1ll << 31)) return pl;
  pl.P = (W + 15) & ~15;
  pl.DP = (D + 1) / 2; pl.HP = (H + 1) / 2; pl.WC = (W + 1) / 2;
  pl.ksteps = (W + 15) / 16;
  pl.kblocks = (pl.ksteps + 1) / 2;
  pl.y_bytes = 4u * pl.P * 64u;
  pl.x_bytes = (uint32_t)pl.kblocks * C1B_NCOLS * 64u;
  pl.g_bytes = (uint32_t)pl.WC * 64u;
  pl.x_off = pl.y_bytes;
  pl.g_off = pl.x_off + pl.x_bytes;
  pl.stage_bytes = (pl.g_off + pl.g_bytes + 1023u) & ~1023u;
  const uint32_t fixed = 1024 + 8 * (3 * C1B_MAX_STAGES) + 64;
  pl.stages = 0;
  for (int st = C1B_MAX_STAGES; st >= 2; st -= 2)          // even: the two builder groups own alternate stages
    if (fixed + (uint32_t)st * pl.stage_bytes <= 227u * 1024u) { pl.stages = st; break; }
  if (pl.stages == 0) return pl;
  if ((uint32_t)pl.stages * pl.stage_bytes < 128u * C1B_NCOLS * 4u) return pl;   // epilogue fold buffer
  pl.smem_bytes = fixed + (uint32_t)pl.stages * pl.stage_bytes;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  int per_group = sms / ng;
  const int units = B * pl.DP * pl.HP;
  if (per_group > units) per_group = units;
  if (per_group < 1) per_group = 1;
  pl.ncta = per_group;
  pl.x6_elems = (size_t)B * D * H * 6 * pl.P;
  // per group: x6 (bf16, 256-byte aligned block) + partials
  const size_t xbytes = (pl.x6_elems * 2 + 255) & ~(size_t)255;
  const size_t pbytes = ((size_t)pl.ncta * 32 * 27 * 4 + 255) & ~(size_t)255;
  pl.ws_bytes = (size_t)ng * (xbytes + pbytes);
  pl.ok = true;
  return pl;
}

}  // namespace tmf

using namespace tmf;

extern "C" {

int64_t tmf_conv1_bwd_fused_workspace_bytes(int ng, int B, int D, int H, int W, int cout) {
  const C1BPlan pl = c1b_plan(ng, B, D, H, W, cout);
  return pl.ok ? (int64_t)pl.ws_bytes : 0;
}

int tmf_conv1_bwd_fused(int ng, const void* const* dout, const void* const* y, const float* const* coef,
                        const float* const* bcoef, const float* const* x, float* const* dw, int B, int D, int H, int W,
                        int cout, float slope, void* ws, size_t ws_bytes, void* stream) {
  TMF_CHECK_NG(ng);
  const C1BPlan pl = c1b_plan(ng, B, D, H, W, cout);
  TMF_REQUIRE(pl.ok, "conv1_bwd_fused: unsupported problem (Cout=%d, %dx%dx%d); use bn_act_pool_bwd_apply + conv1_wgrad",
              cout, D, H, W);
  TMF_REQUIRE(ws != nullptr && ws_bytes >= pl.ws_bytes, "conv1_bwd_fused: workspace too small (%zu < %zu bytes)",
              ws_bytes, pl.ws_bytes);
  TMF_REQUIRE(((uintptr_t)ws & 255) == 0, "conv1_bwd_fused: workspace must be 256-byte aligned");
  EncodeTiledFn encode = c1b_encode_fn();
  TMF_REQUIRE(encode != nullptr, "conv1_bwd_fused: cuTensorMapEncodeTiled entry point not available");
  cudaStream_t st = (cudaStream_t)stream;
  C1BParams p{};
  p.ng = ng; p.B = B; p.D = D; p.H = H; p.W = W; p.P = pl.P; p.DP = pl.DP; p.HP = pl.HP; p.WC = pl.WC;
  p.units = B * pl.DP * pl.HP;
  p.ksteps = pl.ksteps; p.kblocks = pl.kblocks; p.stages = pl.stages;
  p.y_bytes = pl.y_bytes; p.x_bytes = pl.x_bytes; p.g_bytes = pl.g_bytes; p.x_off = pl.x_off; p.g_off = pl.g_off;
  p.stage_bytes = pl.stage_bytes;
  p.tx_bytes = pl.y_bytes + pl.x_bytes + pl.g_bytes;
  p.idesc = make_idesc_bf16(128, C1B_NCOLS, /*A MN-major*/ 1, /*B K-major*/ 0);
  p.slope = slope;
  const size_t xbytes = (pl.x6_elems * 2 + 255) & ~(size_t)255;
  const size_t pbytes = ((size_t)pl.ncta * 32 * 27 * 4 + 255) & ~(size_t)255;
  GroupPtr<const float> gx;
  GroupPtr<__nv_bfloat16> gx6;
  GroupPtr<const float> gpart;
  GroupPtr<float> gdw;
  if (!load_group(gx, x, ng, true, "x") || !load_group(gdw, dw, ng, true, "dw")) return 1;
  const int Do = D / 2, Ho = H / 2, Wo = W / 2;
  for (int g = 0; g < TMF_MAX_GROUPS; ++g) gx6.p[g] = nullptr;
  for (int g = 0; g < ng; ++g) {
    uint8_t* base = (uint8_t*)ws + (size_t)g * (xbytes + pbytes);
    gx6.p[g] = (__nv_bfloat16*)base;
    TMF_REQUIRE(dout[g] && y[g] && coef[g] && bcoef[g], "conv1_bwd_fused: NULL device pointer");
    TMF_REQUIRE(((uintptr_t)dout[g] & 15) == 0 && ((uintptr_t)y[g] & 15) == 0, "conv1_bwd_fused: tensors must be 16-byte aligned");
    p.part[g] = (float*)(base + xbytes);
    gpart.p[g] = p.part[g];
    p.coef[g] = coef[g];
    p.bcoef[g] = bcoef[g];
    cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    {
      cuuint64_t dims[5] = {32, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)D, (cuuint64_t)B};
      cuuint64_t strides[4] = {64, (cuuint64_t)W * 64, (cuuint64_t)H * W * 64, (cuuint64_t)D * H * W * 64};
      cuuint32_t box[5] = {32, (cuuint32_t)pl.P, 2, 2, 1};
      CUresult r = encode(&p.tmY[g], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<void*>(y[g]), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      TMF_REQUIRE(r == CUDA_SUCCESS, "conv1_bwd_fused: cuTensorMapEncodeTiled(y) failed with %d", (int)r);
    }
    {
      cuuint64_t dims[5] = {32, (cuuint64_t)Wo, (cuuint64_t)Ho, (cuuint64_t)Do, (cuuint64_t)B};
      cuuint64_t strides[4] = {64, (cuuint64_t)Wo * 64, (cuuint64_t)Ho * Wo * 64, (cuuint64_t)Do * Ho * Wo * 64};
      cuuint32_t box[5] = {32, (cuuint32_t)pl.WC, 1, 1, 1};
      CUresult r = encode(&p.tmG[g], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<void*>(dout[g]), dims, strides, box,
                          estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      TMF_REQUIRE(r == CUDA_SUCCESS, "conv1_bwd_fused: cuTensorMapEncodeTiled(dout) failed with %d", (int)r);
    }
    {
      const cuuint64_t rb = (cuuint64_t)pl.P * 2;
      cuuint64_t dims[5] = {(cuuint64_t)pl.P, 6, (cuuint64_t)H, (cuuint64_t)D, (cuuint64_t)B};
      cuuint64_t strides[4] = {rb, 6 * rb, (cuuint64_t)H * 6 * rb, (cuuint64_t)D * H * 6 * rb};
      cuuint32_t box[5] = {32, 6, 4, 4, 1};
      CUresult r = encode(&p.tmX[g], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, (void*)gx6.p[g], dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      TMF_REQUIRE(r == CUDA_SUCCESS, "conv1_bwd_fused: cuTensorMapEncodeTiled(x) failed with %d", (int)r);
    }
  }
  const int rows = B * D * H;
  const long long total = (long long)rows * (pl.P / 8);
  // grid-stride loop over at most ~4 blocks (1024 threads) per SM, shared by the towers
  dim3 grid((unsigned)min((long long)(148 * 4 / ng), (total + 255) / 256), 1, ng);
  launch_k(conv1_split_x_kernel, grid, 256, 0, st, gx, gx6, rows, W, pl.P);
  TMF_LAUNCH_CHECK();
  static bool attr_done = false;
  if (!attr_done) {
    TMF_CUDA(cudaFuncSetAttribute(conv1_bwd_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr_done = true;
  }
  launch_k(conv1_bwd_fused_kernel, dim3(pl.ncta * ng), C1B_THREADS, pl.smem_bytes, st, p);
  TMF_LAUNCH_CHECK();
  launch_k(conv1_bwd_reduce_kernel, dim3(ceil_div(32 * 27, 256), 1, ng), 256, 0, st, gpart, gdw, pl.ncta);
  TMF_LAUNCH_CHECK();
  return 0;
}

}  // extern "C"

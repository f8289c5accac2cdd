// conv_umma.cu -- generic implicit-GEMM Conv3d (3x3x3 pad 1, or 1x1x1) forward / dgrad on the 5th-gen tensor cores:
// TMA-staged NDHWC bf16 operands, tcgen05.mma with fp32 accumulators in TMEM, fused bias + bf16 store +
// BatchNorm statistics epilogue.  One persistent, warp-specialised CTA per SM.  It takes the layers the
// input-stationary kernel (conv_umma_col.cu) does not: Cin >= 128 (conv3.3 dgrad, conv4.0) and 1x1x1 (conv4.3).
//
// Mapping.  For one sample n and output plane d the (h,w) positions are linearised with a padded row pitch
// Wp = W + 2*hw (hw = ks/2):  q = h*Wp + w'.  A super-tile is mt*128 consecutive q.  For tap (kd,kh,kw) the A operand of
// a 128-row tile is the same window of the *padded* input plane d+kd-hw shifted by kh*Wp + kw rows, so ONE TMA box
// (channels x Wp x NH rows, out-of-bounds zero fill = the convolution padding) per (kd, 64-channel chunk) feeds all
// ks*ks taps of that plane from shared memory: each tap's tcgen05.mma simply uses a shared-memory descriptor whose
// start address is advanced by (shift * row bytes).  Rows with w' >= W (2 per output row) or h >= H are computed and
// discarded in the epilogue.  Weights wf[tap][Cout][Cin] are the K-major B operand, one TMA box per (tap, chunk);
// they stay resident in shared memory for the whole kernel when they fit and are streamed through a ring otherwise.
//
// Streamed weights are bound by the NUMBER of TMA boxes (~500 cycles each, measured), so a tap's box is applied to all
// mt tiles of the super-tile (mt accumulators in TMEM) and, where N is narrow, two issuer warps share the taps; the
// host plan (make_plan) picks mt / issuers / accumulator sets with a small cost model -- see DESIGN.md section 3.2.
#include <cuda.h>

#include "common.cuh"
#include "umma.cuh"

namespace tmf {
using namespace umma;

// threads: warp 0 = TMA producer, warp 1 (and 2 in the two-issuer variant) = MMA issuer (warp 1 owns TMEM), then 4 epilogue warps
constexpr int UC_TILE_M = 128;
constexpr int UC_MAX_BSTAGES = 27 * 4;
constexpr int UC_MAX_ASTAGES = 4;
constexpr int UC_TMA_LANES = 4;  // producer lanes issuing TMA boxes round-robin
constexpr uint32_t UC_SMEM_BUDGET = 227 * 1024;

struct alignas(64) UmmaConvParams {
  CUtensorMap tmA[TMF_MAX_GROUPS];
  CUtensorMap tmB[TMF_MAX_GROUPS];
  const float* bias[TMF_MAX_GROUPS];
  __nv_bfloat16* y[TMF_MAX_GROUPS];
  double* stats[TMF_MAX_GROUPS];
  int ng, B, D, H, W, cin, cout, ks, hw;
  int Wp, NH, QT;                 // padded row pitch, slab rows (in h), q tiles per plane
  int tiles_per_group;
  int nchunk, chunk, row_bytes;   // K chunks per tap, channels per chunk, bytes per smem row
  uint32_t layout;                // UMMA layout type (SW128 / SW64)
  int SA, SB, b_resident;
  uint32_t a_stage_bytes, b_stage_bytes, a_tx_bytes, b_tx_bytes;
  uint32_t idesc;
  uint32_t tmem_cols;
  int tma_lanes;                  // producer lanes that issue TMA boxes round-robin
  int mt;                         // 128-row M tiles per weight pass ("super-tile" = 128*mt consecutive positions)
  int nbuf;                       // accumulator sets in TMEM: 2 = epilogue overlaps the next super-tile, 1 = it does not
  // Plane-stack mode (small planes, e.g. conv4.0 at 11x13x11: a plane is 169 padded rows = 1.3 tiles, so per-plane tiling
  // leaves 44 % of the MMA rows empty): the positions of a whole SAMPLE are linearised, q = d*Pp + h*Wp + w' with the plane
  // pitch Pp = (H + 2*hw) * Wp, and a tile is any 128 consecutive q.  Its A slab for (kd, chunk) is ONE box of NP whole padded
  // planes starting at plane q0/Pp + kd - hw (out-of-bounds planes / rows / columns zero-filled = the padding); tap shifts
  // stay row offsets because every plane carries its own halo rows.  QT = tiles per sample, mt = 1.
  int stack, Pp, NP;
  // kw-fused weight boxes (streamed weights): the three kw taps of a (kd, kh) are neighbouring [Cout][chunk] blocks of
  // wf[tap][Cout][Cin], so ONE TMA box {chunk, Cout, 3} brings them and a ring stage holds three taps: a third of the weight
  // boxes (the kernel is bound by their number, ~500 cycles each).
  int kwf;
};

// NISS = 2 (streamed weights, 4*Cout <= 512 TMEM columns): a narrow-N tcgen05.mma (N = 64: ~54 tensor-pipe cycles) is
// bound by the ~100 cycles its issuing thread needs, so two issuer warps take alternate taps of the weight ring (ring
// stage s always belongs to issuer s % 2: SB is even), each into its own TMEM accumulator; the epilogue adds the two.
template <int KSTEPS, int KS, bool RES, int NISS>
__global__ void __launch_bounds__(32 * (5 + NISS), 1) conv3d_umma_kernel(const __grid_constant__ UmmaConvParams p) {
  static_assert(NISS == 1 || !RES, "two issuers only with the streamed weight ring");
  constexpr int NTHREADS = 32 * (5 + NISS);
  constexpr int EPI0 = 32 * (1 + NISS);             // first epilogue thread
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t smA = smem_base;
  const uint32_t smB = smA + (uint32_t)p.SA * p.a_stage_bytes;
  const uint32_t bars = smB + (uint32_t)p.SB * p.b_stage_bytes;       // 8-byte barriers
  const uint32_t a_full = bars, a_empty = a_full + 8 * UC_MAX_ASTAGES;
  const uint32_t b_full = a_empty + 8 * UC_MAX_ASTAGES, b_empty = b_full + 8 * UC_MAX_BSTAGES;
  const uint32_t acc_full = b_empty + 8 * UC_MAX_BSTAGES, acc_empty = acc_full + 16;
  const uint32_t tmem_slot = acc_empty + 16;
  const uint32_t stats_sm = tmem_slot + 16;                             // float [4 epilogue warps][2][256]
  uint8_t* gen_base = smem_raw + (smem_base - smem_u32(smem_raw));
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(gen_base + (tmem_slot - smem_base));
  float* stats_ptr = reinterpret_cast<float*>(gen_base + (stats_sm - smem_base));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = blockIdx.x % p.ng;
  const int cta = blockIdx.x / p.ng, ncta = gridDim.x / p.ng;
  const int taps2 = p.ks * p.ks;

  if (threadIdx.x == 0) {
    for (int i = 0; i < p.SA; ++i) { mbar_init(a_full + 8 * i, 1); mbar_init(a_empty + 8 * i, NISS); }
    for (int i = 0; i < p.SB; ++i) { mbar_init(b_full + 8 * i, 1); mbar_init(b_empty + 8 * i, 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(acc_full + 8 * i, NISS); mbar_init(acc_empty + 8 * i, 128); }
    fence_barrier_init();
    prefetch_tmap(&p.tmA[g]);
    prefetch_tmap(&p.tmB[g]);
  }
  for (int i = threadIdx.x; i < 2048; i += NTHREADS) stats_ptr[i] = 0.f;
  if (warp == 1) {
    tmem_alloc(tmem_slot, p.tmem_cols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp == 0) {
    // =========================================== TMA producer ===========================================
    // One thread keeps only ~2 tensor loads in flight (measured: ~600 cycles per box whatever its size,
    // scripts/ubench/tma_bw.cu), which starves the narrow-N layers whose weights stream through the ring (conv3.3
    // dgrad: 60 boxes per 128-row tile).  UC_TMA_LANES lanes therefore walk the same load sequence and issue the
    // boxes round-robin.  Every lane waits on EVERY ring hand-over, owner or not: an mbarrier parity wait is only
    // sound for a thread that has observed each earlier phase of that barrier.
    if (lane < p.tma_lanes) {
      const int nl = p.tma_lanes;
      int sa = 0, sb = 0, jw = 0;
      uint32_t pa = 0, pb = 0;
      uint32_t kd_loaded = 0;                                  // resident weights: planes already requested
      for (int tile = cta; tile < p.tiles_per_group; tile += ncta) {
        int r = tile;
        const int qt = r % p.QT; r /= p.QT;
        const int d = p.stack ? (qt * UC_TILE_M) / p.Pp : r % p.D;          // stack: first plane the tile touches
        const int n = p.stack ? r : r / p.D;
        const int h0 = p.stack ? 0 : (qt * UC_TILE_M * p.mt) / p.Wp;
        for (int kd = 0; kd < p.ks; ++kd) {
          const int dd = d + kd - p.hw;
          if (dd + p.NP - 1 < 0 || dd >= p.D) continue;
          if (p.b_resident && !((kd_loaded >> kd) & 1u)) {     // all (tap, chunk) boxes of this plane, once per CTA
            kd_loaded |= 1u << kd;
            for (int t = 0; t < taps2; ++t)
              for (int c = 0; c < p.nchunk; ++c, ++jw) {
                if ((jw % nl) != lane) continue;
                const int tap = kd * taps2 + t, idx = tap * p.nchunk + c;
                mbar_expect_tx(b_full + 8 * idx, p.b_tx_bytes);
                tma_load_3d(smB + (uint32_t)idx * p.b_stage_bytes, &p.tmB[g], b_full + 8 * idx, c * p.chunk, 0, tap);
              }
          }
          for (int c = 0; c < p.nchunk; ++c) {
            mbar_wait(a_empty + 8 * sa, pa ^ 1u);
            if ((jw % nl) == lane) {
              mbar_expect_tx(a_full + 8 * sa, p.a_tx_bytes);
              tma_load_5d(smA + (uint32_t)sa * p.a_stage_bytes, &p.tmA[g], a_full + 8 * sa, c * p.chunk, -p.hw,
                          h0 - p.hw, dd, n);
            }
            ++jw;
            if (++sa == p.SA) { sa = 0; pa ^= 1u; }
            if (!p.b_resident) {
              const int tstep = p.kwf ? p.ks : 1;
              for (int t = 0; t < taps2; t += tstep, ++jw) {
                const int tap = kd * taps2 + t;
                mbar_wait(b_empty + 8 * sb, pb ^ 1u);
                if ((jw % nl) == lane) {
                  mbar_expect_tx(b_full + 8 * sb, p.b_tx_bytes);
                  tma_load_3d(smB + (uint32_t)sb * p.b_stage_bytes, &p.tmB[g], b_full + 8 * sb, c * p.chunk, 0, tap);
                }
                if (++sb == p.SB) { sb = 0; pb ^= 1u; }
              }
            }
          }
        }
      }
    }
  } else if (warp <= NISS) {
    // =========================================== MMA issuer =============================================
    // The whole warp runs the (warp-uniform) control flow so that descriptor arithmetic stays in uniform registers;
    // one elected lane issues tcgen05.mma / tcgen05.commit.  KSTEPS (16-element K steps per smem row), the kernel
    // size and the weight residency are compile-time, so a tap is a handful of adds plus its MMAs.
    {
      constexpr uint32_t ROW_UNITS = KSTEPS * 2;                 // row bytes / 16
      constexpr uint32_t SBO = 8u * KSTEPS * 32u;
      constexpr int TAPS2 = KS * KS;
      const int iss = warp - 1;                                  // which issuer this warp is (0 when NISS == 1)
      int sa = 0, sb = 0;
      uint32_t pa = 0, pb = 0;
      const uint64_t desc_hi = make_smem_desc(0, 16, SBO, p.layout, 0) & 0xFFFFFFFF00000000ull;
      const uint32_t desc_lo_const = (uint32_t)(make_smem_desc(0, 16, SBO, p.layout, 0) & 0xFFFF0000ull);
      const uint32_t b_units = p.b_stage_bytes >> 4;
      const uint32_t a0_lo = desc_lo_const | ((smA & 0x3FFFFu) >> 4);
      const uint32_t b0_lo = desc_lo_const | ((smB & 0x3FFFFu) >> 4);
      const uint32_t a_units = p.a_stage_bytes >> 4;
      const uint32_t wp_units = (uint32_t)p.Wp * ROW_UNITS;
      uint32_t kd_ready = 0;                                     // resident weights of plane kd known to be loaded
      int it = 0;
      for (int tile = cta; tile < p.tiles_per_group; tile += ncta, ++it) {
        int r = tile;
        const int qt = r % p.QT; r /= p.QT;
        const int d = p.stack ? (qt * UC_TILE_M) / p.Pp : r % p.D;
        const uint32_t qoff_units =
            (uint32_t)(p.stack ? (qt * UC_TILE_M) % p.Pp : (qt * UC_TILE_M * p.mt) % p.Wp) * ROW_UNITS;
        const int as = (p.nbuf == 2) ? (it & 1) : 0;
        const uint32_t acc_ph = (uint32_t)((p.nbuf == 2) ? (it >> 1) : it) & 1u;
        mbar_wait(acc_empty + 8 * as, acc_ph ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)((as * NISS + iss) * p.mt * p.cout);
        const uint32_t mt_a_units = (uint32_t)UC_TILE_M * ROW_UNITS;      // next 128 rows of the slab
        uint32_t accumulate = 0;
#pragma unroll 1
        for (int kd = 0; kd < KS; ++kd) {
          const int dd = d + kd - p.hw;
          if (dd + p.NP - 1 < 0 || dd >= p.D) continue;
          if (RES && !((kd_ready >> kd) & 1u)) {
            for (int i = 0; i < TAPS2 * p.nchunk; ++i) mbar_wait(b_full + 8 * (kd * TAPS2 * p.nchunk + i), 0u);
            kd_ready |= 1u << kd;
          }
#pragma unroll 1
          for (int c = 0; c < p.nchunk; ++c) {
            mbar_wait(a_full + 8 * sa, pa);
            tc_fence_after();
            const uint32_t a_slab = a0_lo + (uint32_t)sa * a_units + qoff_units;
            uint32_t b_res = b0_lo + (uint32_t)((kd * TAPS2) * p.nchunk + c) * b_units;   // resident: stage of tap 0
            const uint32_t b_res_step = (uint32_t)p.nchunk * b_units;
            const bool kwf = !RES && p.kwf != 0;
            const uint32_t tap_units = (uint32_t)(p.cout * KSTEPS * 32) >> 4;     // one tap inside a kw-fused ring stage
#pragma unroll
            for (int kh = 0; kh < KS; ++kh) {
              bool skip_row = false;                               // kw-fused: this (kd, kh) stage is the other issuer's
#pragma unroll
              for (int kw = 0; kw < KS; ++kw) {
                const uint32_t a_lo = a_slab + (uint32_t)kh * wp_units + (uint32_t)kw * ROW_UNITS;
                const bool last_of_stage = !kwf || kw == KS - 1;   // the ring stage is released after its last tap
                uint32_t b_lo;
                if (RES) {
                  b_lo = b_res;
                  b_res += b_res_step;
                } else if (!kwf) {
                  if (NISS > 1 && (sb & (NISS - 1)) != iss) {    // the other issuer's tap
                    if (++sb == p.SB) { sb = 0; pb ^= 1u; }
                    continue;
                  }
                  mbar_wait(b_full + 8 * sb, pb);
                  tc_fence_after();
                  b_lo = b0_lo + (uint32_t)sb * b_units;
                } else {
                  if (kw == 0) {
                    skip_row = NISS > 1 && (sb & (NISS - 1)) != iss;
                    if (!skip_row) {
                      mbar_wait(b_full + 8 * sb, pb);
                      tc_fence_after();
                    }
                  }
                  if (skip_row) {
                    if (last_of_stage) { if (++sb == p.SB) { sb = 0; pb ^= 1u; } }
                    continue;
                  }
                  b_lo = b0_lo + (uint32_t)sb * b_units + (uint32_t)kw * tap_units;
                }
                if (elect_one()) {
                  // the tap's weights multiply every 128-row tile of the super-tile before the ring stage is released
                  for (int mt = 0; mt < p.mt; ++mt) {
                    const uint32_t a_mt = a_lo + (uint32_t)mt * mt_a_units;
                    const uint32_t d_mt = d_tmem + (uint32_t)(mt * p.cout);
#pragma unroll
                    for (int k = 0; k < KSTEPS; ++k)
                      mma_bf16_ss(d_mt, desc_hi | (uint64_t)(a_mt + 2u * k), desc_hi | (uint64_t)(b_lo + 2u * k), p.idesc,
                                  k ? 1u : accumulate);
                  }
                  if (!RES && last_of_stage) mma_commit(b_empty + 8 * sb);
                }
                accumulate = 1;
                __syncwarp();
                if (!RES && last_of_stage) {
                  if (++sb == p.SB) { sb = 0; pb ^= 1u; }
                }
              }
            }
            if (elect_one()) mma_commit(a_empty + 8 * sa);
            __syncwarp();
            if (++sa == p.SA) { sa = 0; pa ^= 1u; }
          }
        }
        if (elect_one()) mma_commit(acc_full + 8 * as);
        __syncwarp();
      }
    }
  } else {
    // =========================================== epilogue ================================================
    const int quarter = warp & 3;                 // TMEM lane quarter this warp may access
    const int row = quarter * 32 + lane;
    const float* bias = p.bias[g];
    __nv_bfloat16* yg = p.y[g];
    const bool want_stats = p.stats[g] != nullptr;
    int it = 0;
    for (int tile = cta; tile < p.tiles_per_group; tile += ncta, ++it) {
      int r = tile;
      const int qt = r % p.QT; r /= p.QT;
      int d = p.stack ? 0 : r % p.D;
      const int n = p.stack ? r : r / p.D;
      const int as = (p.nbuf == 2) ? (it & 1) : 0;
      const uint32_t acc_ph = (uint32_t)((p.nbuf == 2) ? (it >> 1) : it) & 1u;
      mbar_wait(acc_full + 8 * as, acc_ph);
      tc_fence_after();
      for (int mt = 0; mt < p.mt; ++mt) {
      int q = (qt * p.mt + mt) * UC_TILE_M + row;
      if (p.stack) { d = q / p.Pp; q -= d * p.Pp; }
      const int h = q / p.Wp, w = q - h * p.Wp;
      const bool valid = (d < p.D) && (h < p.H) && (w < p.W);
      const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)((as * NISS * p.mt + mt) * p.cout);
      __nv_bfloat16* yrow = yg + ((((int64_t)n * p.D + d) * p.H + h) * p.W + w) * p.cout;
      for (int c0 = 0; c0 < p.cout; c0 += 32) {
        uint32_t raw[32];
        tmem_ld32(taddr + (uint32_t)c0, raw);
        tmem_ld_wait();
        if (NISS > 1) {                                        // second issuer's partial sums
          uint32_t raw2[32];
          tmem_ld32(taddr + (uint32_t)(p.mt * p.cout + c0), raw2);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; ++j) raw[j] = __float_as_uint(__uint_as_float(raw[j]) + __uint_as_float(raw2[j]));
        }
        float v[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          float a = __uint_as_float(raw[j]);
          if (bias != nullptr) a += __ldg(bias + c0 + j);
          v[j] = valid ? round_bf16(a) : 0.f;
        }
        if (valid) {
#pragma unroll
          for (int qd = 0; qd < 4; ++qd) *reinterpret_cast<uint4*>(yrow + c0 + qd * 8) = pack8(&v[qd * 8]);
        }
        if (want_stats) {
          float sq[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) sq[j] = v[j] * v[j];
          // transpose-reduce: lane l ends with the warp total of column c0 + l
#pragma unroll
          for (int off = 16; off >= 1; off >>= 1) {
            const bool upper = (lane & off) != 0;
#pragma unroll
            for (int i = 0; i < off; ++i) {
              const float s_send = upper ? v[i] : v[i + off];
              const float s_keep = upper ? v[i + off] : v[i];
              v[i] = s_keep + __shfl_xor_sync(0xffffffffu, s_send, off);
              const float q_send = upper ? sq[i] : sq[i + off];
              const float q_keep = upper ? sq[i + off] : sq[i];
              sq[i] = q_keep + __shfl_xor_sync(0xffffffffu, q_send, off);
            }
          }
          // each epilogue warp owns a slice of the shared accumulators (program order -> deterministic)
          stats_ptr[quarter * 512 + c0 + lane] += v[0];
          stats_ptr[quarter * 512 + 256 + c0 + lane] += sq[0];
        }
      }
      }
      tc_fence_before();
      mbar_arrive(acc_empty + 8 * as);
    }
    if (want_stats) {
      asm volatile("bar.sync 1, 128;" ::: "memory");
      for (int i = threadIdx.x - EPI0; i < p.cout; i += 128) {
        double s1 = 0.0, s2 = 0.0;
#pragma unroll
        for (int w4 = 0; w4 < 4; ++w4) { s1 += (double)stats_ptr[w4 * 512 + i]; s2 += (double)stats_ptr[w4 * 512 + 256 + i]; }
        stat_row_store(p.stats[g], 2 * p.cout, cta, ncta, i, s1);
        stat_row_store(p.stats[g], 2 * p.cout, cta, ncta, p.cout + i, s2);
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

// ------------------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
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

struct UmmaPlan {
  bool ok;
  int Wp, NH, QT, nchunk, chunk, row_bytes, SA, SB, b_resident, niss, mt, nbuf;
  int stack, Pp, NP, kwf;
  uint32_t layout, a_stage_bytes, b_stage_bytes, a_tx, b_tx, tmem_cols, smem_bytes;
  CUtensorMapSwizzle swz;
};

static int umma_env_int(const char* name, int dflt) {
  const char* e = getenv(name);
  return e ? atoi(e) : dflt;
}

// geometry of a super-tile of mt 128-row tiles: slab rows, tiles per plane, TMA bytes
static void plan_geometry(UmmaPlan& pl, int H, int ks, int mt) {
  const int rmax = (pl.Wp - 1) + (ks - 1) * pl.Wp + (ks - 1) + (UC_TILE_M * mt - 1);
  pl.NH = rmax / pl.Wp + 1;
  pl.QT = (H * pl.Wp + UC_TILE_M * mt - 1) / (UC_TILE_M * mt);
  pl.a_tx = (uint32_t)pl.NH * pl.Wp * pl.row_bytes;
  pl.a_stage_bytes = (pl.a_tx + 1023u) & ~1023u;
  pl.mt = mt;
}

static UmmaPlan make_plan(int D, int H, int W, int cin, int cout, int ks, int B = 8, int ng = 2) {
  UmmaPlan pl{};
  pl.ok = false;
  if (ks != 1 && ks != 3) return pl;
  if (cin % 32 != 0 || cout % 32 != 0 || cout < 32 || cout > 256 || cin < 32) return pl;
  const int hw = ks / 2;
  pl.chunk = (cin % 64 == 0) ? 64 : 32;
  pl.nchunk = cin / pl.chunk;
  pl.row_bytes = pl.chunk * 2;
  pl.layout = (pl.chunk == 64) ? LAYOUT_SW128 : LAYOUT_SW64;
  pl.swz = (pl.chunk == 64) ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
  pl.Wp = W + 2 * hw;
  pl.niss = 1;
  pl.nbuf = 2;
  plan_geometry(pl, H, ks, 1);
  if (pl.Wp > 256 || pl.NH > 256) return pl;
  pl.b_tx = (uint32_t)cout * pl.row_bytes;
  pl.b_stage_bytes = (pl.b_tx + 1023u) & ~1023u;
  const int taps = ks * ks * ks;
  const uint32_t fixed = 1024 /*align slack*/ + 8 * (2 * UC_MAX_ASTAGES + 2 * UC_MAX_BSTAGES) + 64 + 8192 /*stats*/ + 256;
  const uint32_t budget = UC_SMEM_BUDGET - fixed;
  const uint32_t total_b = (uint32_t)taps * pl.nchunk * pl.b_stage_bytes;
  if (taps * pl.nchunk <= UC_MAX_BSTAGES && total_b + 2 * pl.a_stage_bytes <= budget) {
    pl.b_resident = 1;
    pl.SB = taps * pl.nchunk;
    pl.SA = (int)((budget - total_b) / pl.a_stage_bytes);
    if (pl.SA > UC_MAX_ASTAGES) pl.SA = UC_MAX_ASTAGES;
  } else {
    // Streamed weights.  Measured on B200 (profiles/r1d_conv_microbench.md): the kernel is bound by the NUMBER of TMA
    // boxes -- ~500 cycles per box plus ~1.5 cycles per 128-byte row, whatever issues them -- and every 128-row tile
    // re-streams all 27 x nchunk weight boxes.  So the weights of a tap are applied to `mt` consecutive 128-row tiles
    // (one bigger input slab per (kd, chunk), mt accumulators in TMEM), and two issuer warps share the taps where the
    // MMAs are narrow.  The plan with the smallest modelled cost per plane wins:
    //   tma = QT * 3 * nchunk * [(500 + 1.5 * slab rows) + 9 * (500 + 1.5 * Cout)]          (128-byte rows)
    //   mma = QT * mt * (27 * nchunk * ksteps) * max(0.75 * Cout, 100 / issuers)            (pipe vs issue cycles)
    //   cost per plane = max(tma, mma) * (1.25 if the accumulators are single-buffered);  the grid is one CTA per SM and
    //   a CTA walks whole super-tiles, so the total is ceil(B*D*QT / CTAs per tower) rounds of (cost per plane / QT):
    //   big super-tiles lose to wave quantisation on the small layers (conv4.0 fwd: 88 super-tiles on 74 CTAs).
    pl.b_resident = 0;
    const int want_kwf = umma_env_int("TMF_UMMA_KWF", -1);           // kw-fused weight boxes: 0 = never, 1 = whenever possible
    const int max_kwf = (ks == 3 && want_kwf != 0 && ((uint32_t)cout * pl.row_bytes) % 1024u == 0) ? 1 : 0;
    const int max_iss = (ks == 3) ? 2 : 1;
    double best = 1e30;
    UmmaPlan bp = pl;
    bool found = false;
    for (int mt = 1; mt <= 4; ++mt) {
      if (ks != 3 && mt > 1) break;
      // kw-fused boxes on per-plane tiles only on request: measured on B200 (conv3.3 dgrad, B = 8) the plan they allow
      // (mt = 2, two issuers, 24 KB stages) runs 128.9 us against 121.3 us for mt = 3 with single-tap stages
      for (int kwf = 0; kwf <= (want_kwf == 1 ? max_kwf : 0); ++kwf)
      for (int niss = 1; niss <= max_iss; ++niss)
        for (int nbuf = 2; nbuf >= 1; --nbuf) {
          if (nbuf * niss * mt * cout > 512) continue;
          UmmaPlan c = pl;
          plan_geometry(c, H, ks, mt);
          if (c.NH > 256) continue;
          c.niss = niss;
          c.nbuf = nbuf;
          c.kwf = kwf;
          c.b_tx = pl.b_tx * (kwf ? ks : 1);
          c.b_stage_bytes = (c.b_tx + 1023u) & ~1023u;
          c.SA = 3;
          if (3 * c.a_stage_bytes + 4 * c.b_stage_bytes > budget) c.SA = 2;
          const int min_sb = (niss == 2) ? 4 : 2;
          if ((uint32_t)c.SA * c.a_stage_bytes + (uint32_t)min_sb * c.b_stage_bytes > budget) continue;
          c.SB = (int)((budget - (uint32_t)c.SA * c.a_stage_bytes) / c.b_stage_bytes);
          if (c.SB > 8) c.SB = 8;
          if (niss == 2) c.SB &= ~1;               // ring stage s is always issuer s % 2's
          const double rows128 = c.row_bytes / 128.0;
          const double tma = (double)c.QT * ks * c.nchunk *
                             ((500.0 + 1.5 * c.NH * c.Wp * rows128) +
                              (ks * ks / (kwf ? ks : 1)) * (500.0 + 1.5 * cout * rows128 * (kwf ? ks : 1)));
          const double per_mma = (0.75 * cout > 100.0 / niss) ? 0.75 * cout : 100.0 / niss;
          const double mma = (double)c.QT * mt * (taps * c.nchunk * (c.chunk / 16)) * per_mma;
          const int ncta = (148 / (ng > 0 ? ng : 1)) > 0 ? 148 / (ng > 0 ? ng : 1) : 1;
          const int64_t ntiles = (int64_t)B * D * c.QT;
          const double rounds = (double)((ntiles + ncta - 1) / ncta);
          const double cost = rounds * (tma > mma ? tma : mma) * (nbuf == 1 ? 1.25 : 1.0) / c.QT * ((want_kwf == 1 && kwf) ? 1e-3 : 1.0);
          if (cost < best * 0.999) { best = cost; bp = c; found = true; }
        }
    }
    // Plane-stack candidates (see UmmaConvParams): tiles of 128 consecutive positions of the whole sample, one box of NP
    // padded planes per (kd, chunk); same cost model per tile, rounds = ceil(B * tiles per sample / CTAs per tower).
    const int want_stack = umma_env_int("TMF_UMMA_STACK", -1);       // bring-up switch: 0 = never, 1 = whenever possible
    if (ks == 3 && want_stack != 0) {
      for (int kwf = 0; kwf <= max_kwf; ++kwf)
      for (int niss = 1; niss <= max_iss; ++niss)
        for (int nbuf = 2; nbuf >= 1; --nbuf) {
          if (nbuf * niss * cout > 512) continue;
          UmmaPlan c = pl;
          c.stack = 1; c.mt = 1; c.niss = niss; c.nbuf = nbuf;
          c.kwf = kwf;
          c.b_tx = pl.b_tx * (kwf ? ks : 1);
          c.b_stage_bytes = (c.b_tx + 1023u) & ~1023u;
          c.NH = H + 2 * hw;
          c.Pp = c.NH * c.Wp;
          c.NP = ((c.Pp - 1) + (UC_TILE_M - 1) + (ks - 1) * c.Wp + (ks - 1) + 1 + c.Pp - 1) / c.Pp;
          if (c.NH > 256 || c.NP > 16) continue;
          c.QT = ((D - 1) * c.Pp + H * c.Wp + UC_TILE_M - 1) / UC_TILE_M;
          c.a_tx = (uint32_t)c.NP * c.Pp * c.row_bytes;
          c.a_stage_bytes = (c.a_tx + 1023u) & ~1023u;
          c.SA = 3;
          if (3 * c.a_stage_bytes + 4 * c.b_stage_bytes > budget) c.SA = 2;
          const int min_sb = (niss == 2) ? 4 : 2;
          if ((uint32_t)c.SA * c.a_stage_bytes + (uint32_t)min_sb * c.b_stage_bytes > budget) continue;
          c.SB = (int)((budget - (uint32_t)c.SA * c.a_stage_bytes) / c.b_stage_bytes);
          if (c.SB > 8) c.SB = 8;
          if (niss == 2) c.SB &= ~1;
          const double rows128 = c.row_bytes / 128.0;
          const double tma = (double)ks * c.nchunk *
                             ((500.0 + 1.5 * c.NP * c.Pp * rows128) +
                              (ks * ks / (kwf ? ks : 1)) * (500.0 + 1.5 * cout * rows128 * (kwf ? ks : 1)));
          const double per_mma = (0.75 * cout > 100.0 / niss) ? 0.75 * cout : 100.0 / niss;
          const double mma = (double)(taps * c.nchunk * (c.chunk / 16)) * per_mma;
          const int ncta = (148 / (ng > 0 ? ng : 1)) > 0 ? 148 / (ng > 0 ? ng : 1) : 1;
          const int64_t ntiles = (int64_t)B * c.QT;
          const double rounds = (double)((ntiles + ncta - 1) / ncta);
          // x 0.9: measured on B200 (conv4.0 dgrad, B = 8: 83.7 us stacked vs 91.6 us per plane) the model overestimates these tiles
          const double cost = 0.9 * rounds * (tma > mma ? tma : mma) * (nbuf == 1 ? 1.25 : 1.0) * ((want_kwf == 1 && kwf) ? 1e-3 : 1.0);
          if (cost < best * 0.999 || (want_stack == 1 && !bp.stack)) { best = cost; bp = c; found = true; }
        }
    }
    if (!found) return pl;
    pl = bp;
  }
  uint32_t cols = 32;
  while (cols < (uint32_t)(pl.nbuf * pl.niss * pl.mt * cout)) cols <<= 1;
  if (cols > 512) return pl;
  pl.tmem_cols = cols;
  pl.smem_bytes = fixed + (uint32_t)pl.SA * pl.a_stage_bytes + (uint32_t)pl.SB * pl.b_stage_bytes;
  pl.ok = pl.smem_bytes <= UC_SMEM_BUDGET;
  return pl;
}

}  // namespace tmf

using namespace tmf;

extern "C" int tmf_conv3d_umma_plan_info(int ng, int B, int D, int H, int W, int cin, int cout, int ksize, int* out8) {
  const UmmaPlan pl = make_plan(D, H, W, cin, cout, ksize, B, ng);
  if (out8 != nullptr) {
    out8[0] = pl.ok ? 1 : 0; out8[1] = pl.mt; out8[2] = pl.niss; out8[3] = pl.nbuf;
    out8[4] = pl.SA; out8[5] = pl.SB; out8[6] = pl.QT; out8[7] = pl.b_resident | (pl.stack << 1) | (pl.kwf << 2);   // bit 1: plane-stack mode, bit 2: kw-fused weight boxes
  }
  return pl.ok ? 0 : 1;
}

bool tmf_conv3d_fwd_umma_supported(int D, int H, int W, int cin, int cout, int ksize) {
  if (getenv("TMF_DISABLE_UMMA") != nullptr) return false;
  return make_plan(D, H, W, cin, cout, ksize).ok;
}

int tmf_conv3d_fwd_umma(int ng, const void* const* a, const void* const* wf, const float* const* bias,
                        void* const* y, double* const* stats, int B, int D, int H, int W, int cin, int cout, int ksize,
                        void* stream) {
  TMF_CHECK_NG(ng);
  // A 1x1x1 convolution is a plain GEMM over the B*D*H*W voxel rows: drop the plane structure (one "plane" of M rows of
  // width 1) so that every 128-row tile is full -- conv4.3: 99 tiles per tower instead of 176 tiles of 143 valid rows.
  if (ksize == 1 && (int64_t)B * D * H * W < (1ll << 31)) { H = B * D * H * W; B = 1; D = 1; W = 1; }
  const UmmaPlan pl = make_plan(D, H, W, cin, cout, ksize, B, ng);
  TMF_REQUIRE(pl.ok, "conv3d_fwd_umma: unsupported problem");
  EncodeTiledFn encode = get_encode_fn();
  TMF_REQUIRE(encode != nullptr, "conv3d_fwd_umma: cuTensorMapEncodeTiled entry point not available");
  UmmaConvParams p{};
  p.ng = ng; p.B = B; p.D = D; p.H = H; p.W = W; p.cin = cin; p.cout = cout; p.ks = ksize; p.hw = ksize / 2;
  p.Wp = pl.Wp; p.NH = pl.NH; p.QT = pl.QT;
  p.stack = pl.stack; p.Pp = pl.Pp; p.NP = pl.stack ? pl.NP : 1;
  p.kwf = pl.kwf;
  p.tiles_per_group = pl.stack ? B * pl.QT : B * D * pl.QT;
  p.nchunk = pl.nchunk; p.chunk = pl.chunk; p.row_bytes = pl.row_bytes; p.layout = pl.layout;
  p.SA = pl.SA; p.SB = pl.SB; p.b_resident = pl.b_resident;
  p.a_stage_bytes = pl.a_stage_bytes; p.b_stage_bytes = pl.b_stage_bytes; p.a_tx_bytes = pl.a_tx; p.b_tx_bytes = pl.b_tx;
  p.idesc = make_idesc_bf16(UC_TILE_M, cout, 0, 0);
  p.tmem_cols = pl.tmem_cols;
  p.tma_lanes = UC_TMA_LANES;
  p.mt = pl.mt;
  p.nbuf = pl.nbuf;
  const int taps = ksize * ksize * ksize;
  cudaStream_t st = (cudaStream_t)stream;
  for (int g = 0; g < ng; ++g) {
    TMF_REQUIRE(a[g] && wf[g] && y[g], "conv3d_fwd_umma: NULL device pointer");
    TMF_REQUIRE(((uintptr_t)a[g] & 15) == 0 && ((uintptr_t)wf[g] & 15) == 0 && ((uintptr_t)y[g] & 15) == 0,
                "conv3d_fwd_umma: tensors must be 16-byte aligned");
    p.bias[g] = bias ? bias[g] : nullptr;
    p.y[g] = (__nv_bfloat16*)y[g];
    p.stats[g] = stats ? stats[g] : nullptr;
    {
      cuuint64_t dims[5] = {(cuuint64_t)cin, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)D, (cuuint64_t)B};
      cuuint64_t strides[4] = {(cuuint64_t)cin * 2, (cuuint64_t)W * cin * 2, (cuuint64_t)H * W * cin * 2,
                               (cuuint64_t)D * H * W * cin * 2};
      cuuint32_t box[5] = {(cuuint32_t)pl.chunk, (cuuint32_t)pl.Wp, (cuuint32_t)pl.NH, (cuuint32_t)(pl.stack ? pl.NP : 1), 1};
      cuuint32_t estr[5] = {1, 1, 1, 1, 1};
      CUresult r = encode(&p.tmA[g], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<void*>(a[g]), dims, strides, box,
                          estr, CU_TENSOR_MAP_INTERLEAVE_NONE, pl.swz, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      TMF_REQUIRE(r == CUDA_SUCCESS, "conv3d_fwd_umma: cuTensorMapEncodeTiled(A) failed with %d", (int)r);
    }
    {
      cuuint64_t dims[3] = {(cuuint64_t)cin, (cuuint64_t)cout, (cuuint64_t)taps};
      cuuint64_t strides[2] = {(cuuint64_t)cin * 2, (cuuint64_t)cout * cin * 2};
      cuuint32_t box[3] = {(cuuint32_t)pl.chunk, (cuuint32_t)cout, (cuuint32_t)(pl.kwf ? ksize : 1)};
      cuuint32_t estr[3] = {1, 1, 1};
      CUresult r = encode(&p.tmB[g], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(wf[g]), dims, strides, box,
                          estr, CU_TENSOR_MAP_INTERLEAVE_NONE, pl.swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      TMF_REQUIRE(r == CUDA_SUCCESS, "conv3d_fwd_umma: cuTensorMapEncodeTiled(B) failed with %d", (int)r);
    }
  }
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  int per_group = sms / ng;
  if (per_group > p.tiles_per_group) per_group = p.tiles_per_group;
  {
    const char* e = getenv("TMF_UMMA_MAX_CTAS");     // test switch: few CTAs per tower -> many super-tiles per CTA
    if (e != nullptr && atoi(e) > 0 && per_group > atoi(e)) per_group = atoi(e);
  }
  if (per_group < 1) per_group = 1;
  if (per_group > TMF_STAT_ROWS) per_group = TMF_STAT_ROWS;
  dim3 grid(per_group * ng, 1, 1);
  const int ksteps = pl.chunk / 16;
#define TMF_LAUNCH_CONV(KST, KSZ, RES, NI)                                                                          \
  do {                                                                                                             \
    static bool attr_done = false;                                                                                 \
    if (!attr_done) {                                                                                              \
      TMF_CUDA(cudaFuncSetAttribute(conv3d_umma_kernel<KST, KSZ, RES, NI>,                                          \
                                    cudaFuncAttributeMaxDynamicSharedMemorySize, (int)UC_SMEM_BUDGET));            \
      attr_done = true;                                                                                            \
    }                                                                                                              \
    launch_k(conv3d_umma_kernel<KST, KSZ, RES, NI>, grid, 32 * (5 + NI), pl.smem_bytes, st, p);                          \
  } while (0)
  if (ksteps == 4 && ksize == 3 && pl.b_resident) TMF_LAUNCH_CONV(4, 3, true, 1);
  else if (ksteps == 4 && ksize == 3 && pl.niss == 2) TMF_LAUNCH_CONV(4, 3, false, 2);
  else if (ksteps == 4 && ksize == 3) TMF_LAUNCH_CONV(4, 3, false, 1);
  else if (ksteps == 2 && ksize == 3 && pl.b_resident) TMF_LAUNCH_CONV(2, 3, true, 1);
  else if (ksteps == 2 && ksize == 3 && pl.niss == 2) TMF_LAUNCH_CONV(2, 3, false, 2);
  else if (ksteps == 2 && ksize == 3) TMF_LAUNCH_CONV(2, 3, false, 1);
  else if (ksteps == 4 && ksize == 1 && pl.b_resident) TMF_LAUNCH_CONV(4, 1, true, 1);
  else if (ksteps == 2 && ksize == 1 && pl.b_resident) TMF_LAUNCH_CONV(2, 1, true, 1);
  else {
    TMF_REQUIRE(pl.niss == 1, "conv3d_fwd_umma: internal: two-issuer plan without a kernel variant");
    if (ksteps == 4) TMF_LAUNCH_CONV(4, 1, false, 1);
    else TMF_LAUNCH_CONV(2, 1, false, 1);
  }
#undef TMF_LAUNCH_CONV
  TMF_LAUNCH_CHECK();
  return 0;
}

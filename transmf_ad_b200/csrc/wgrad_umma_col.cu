// wgrad_umma_col.cu -- second-generation Conv3d 3x3x3 weight gradient on tcgen05 (reference: the weight gradient of
// nn.Conv3d, models/networks.py:28-46), built on what the forward kernel (conv_umma_col.cu) taught:
//
//   dW[kd,kh,kw][ci][co] = sum over output voxels v of  X[v + shift(kd,kh,kw)][ci] * dY[v][co]
//
//   * GEMM K = voxels (16 per MMA); both operands are MN-major and are used exactly as NDHWC lies in memory (padded row
//     pitch W+1, one shared zero column, TMA out-of-bounds zero fill = convolution padding).
//   * A CTA owns one 32 x 32 (ci, co) block of one tower ("virtual group" = tower x ci block x co block) and ALL 27 taps:
//       M (128 TMEM lanes) = 4 atoms of 32 input channels whose descriptor LBO is ONE voxel row: atoms = kw taps 0,1,2
//                            (+ one garbage atom);
//       N (96 TMEM columns) = 3 atoms of 32 output channels whose LBO is ONE PADDED ROW (Wp voxels): the dY window is
//                            read at row shifts j*Wp, which is tap kh = 2 - j  (the K axis starts 2 rows above the plane);
//       kd = three accumulators (3 x 96 columns), one per issuer warp.
//     So one 128 x 96 x 16 MMA advances 9 taps; 24 MMAs per 128-voxel tile instead of 72.
//   * The CTA walks a column of 128-voxel tiles along d: X planes d-1, d, d+1 and dY plane d roll through two rings, one
//     new X slab and one new dY slab per step; the step list is cut into equal contiguous ranges.
//   * Accumulation stays in TMEM for the CTA's whole range; the partial block goes to the caller's workspace and
//     wgrad_reduce_kernel (wgrad_umma.cu) sums the splits in fixed order (deterministic).
#include <cuda.h>

#include "common.cuh"
#include "umma.cuh"

namespace tmf {
using namespace umma;

constexpr int WC_TK = 128;                      // voxels (GEMM K) per step
constexpr int WC_KSTEPS = WC_TK / 16;
constexpr int WC_BLK = 32;                      // channels per block side
constexpr int WC_THREADS = 32 * 8;              // producer, 3 issuers, 4 epilogue warps
constexpr int WC_MAX_SLOTS = 8;
constexpr uint32_t WC_SMEM_BUDGET = 227 * 1024;
constexpr uint32_t WC_FIXED_SMEM = 1024 + 8 * 4 * WC_MAX_SLOTS + 8 + 16 + 16 + 64;

struct alignas(64) WgColParams {
  CUtensorMap tmX[TMF_MAX_GROUPS];
  CUtensorMap tmY[TMF_MAX_GROUPS];
  float* ws[TMF_MAX_GROUPS];
  int ng, ncib, ncob, cin, cout, B, D, H, W;
  int Wp, NHx, NHy, QT, Sx, Sy;
  int steps_per_group;            // B * QT * D
  uint32_t x_slot_bytes, y_slot_bytes, x_tx, y_tx, idesc;
};

__global__ void __launch_bounds__(WC_THREADS, 1) conv3d_wgrad_col_kernel(const __grid_constant__ WgColParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t smX = smem_base;
  const uint32_t smY = smX + (uint32_t)p.Sx * p.x_slot_bytes;
  const uint32_t bars = smY + (uint32_t)p.Sy * p.y_slot_bytes;
  const uint32_t x_full = bars, x_empty = x_full + 8 * WC_MAX_SLOTS;
  const uint32_t y_full = x_empty + 8 * WC_MAX_SLOTS, y_empty = y_full + 8 * WC_MAX_SLOTS;
  const uint32_t acc_full = y_empty + 8 * WC_MAX_SLOTS;
  const uint32_t tmem_slot = acc_full + 8;
  const uint32_t valid_sm = tmem_slot + 8;                                // int [3]: accumulator kd holds data
  uint8_t* gen_base = smem_raw + (smem_base - smem_u32(smem_raw));
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(gen_base + (tmem_slot - smem_base));
  volatile int* valid_ptr = reinterpret_cast<volatile int*>(gen_base + (valid_sm - smem_base));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ngv = p.ng * p.ncib * p.ncob;
  const int gv = blockIdx.x % ngv;
  const int g = gv / (p.ncib * p.ncob);
  const int cib = (gv / p.ncob) % p.ncib, cob = gv % p.ncob;
  const int cta = blockIdx.x / ngv, ncta = gridDim.x / ngv;
  const int s_begin = (int)(((int64_t)cta * p.steps_per_group) / ncta);
  const int s_end = (int)(((int64_t)(cta + 1) * p.steps_per_group) / ncta);

  if (threadIdx.x == 0) {
    for (int i = 0; i < p.Sx; ++i) { mbar_init(x_full + 8 * i, 1); mbar_init(x_empty + 8 * i, 3); }
    for (int i = 0; i < p.Sy; ++i) { mbar_init(y_full + 8 * i, 1); mbar_init(y_empty + 8 * i, 3); }
    mbar_init(acc_full, 3);
    fence_barrier_init();
    prefetch_tmap(&p.tmX[g]);
    prefetch_tmap(&p.tmY[g]);
  }
  if (threadIdx.x < 3) valid_ptr[threadIdx.x] = 0;
  if (warp == 1) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp == 0) {
    // ================================ TMA producer: lanes 0,1 -> X ring, lanes 2,3 -> dY ring ================================
    if (lane < 4 && s_begin < s_end) {
      const bool is_x = lane < 2;
      const int sub = lane & 1;
      const int S = is_x ? p.Sx : p.Sy;
      const uint32_t full = is_x ? x_full : y_full, empty = is_x ? x_empty : y_empty;
      int slot = 0, j = 0;
      uint32_t ph = 0;
      for (int s = s_begin; s < s_end;) {
        const int d0 = s % p.D, t = s / p.D;
        const int qt = t % p.QT, n = t / p.QT;
        const int len = min(p.D - d0, s_end - s);
        const int u0 = qt * WC_TK - 2 * p.Wp;
        const int hy0 = (u0 >= 0) ? (u0 / p.Wp) : -((-u0 + p.Wp - 1) / p.Wp);       // floor
        const int lo = is_x ? max(d0 - 1, 0) : d0;
        const int hi = is_x ? min(d0 + len, p.D - 1) : d0 + len - 1;
        for (int pl = lo; pl <= hi; ++pl, ++j) {
          mbar_wait(empty + 8 * slot, ph ^ 1u);                          // both lanes of a ring see every phase
          if ((j & 1) == sub) {
            if (is_x) {
              mbar_expect_tx(full + 8 * slot, p.x_tx);
              tma_load_5d(smX + (uint32_t)slot * p.x_slot_bytes, &p.tmX[g], full + 8 * slot, cib * WC_BLK, -1, hy0 - 1, pl, n);
            } else {
              mbar_expect_tx(full + 8 * slot, p.y_tx);
              tma_load_5d(smY + (uint32_t)slot * p.y_slot_bytes, &p.tmY[g], full + 8 * slot, cob * WC_BLK, -1, hy0, pl, n);
            }
          }
          if (++slot == S) { slot = 0; ph ^= 1u; }
        }
        s += len;
      }
    }
  } else if (warp < 4) {
    // ================================ MMA issuers: warp 1 + kd owns tap plane kd ================================
    const int kd = warp - 1;
    if (elect_one()) {
      bool started = false;
      if (s_begin < s_end) {
        constexpr uint32_t RB = WC_BLK * 2;                       // row bytes (32 channels bf16)
        // MN-major SW64 descriptors: SBO = 8 rows; LBO = distance between 32-channel atoms
        const uint64_t hi = make_smem_desc(0, 0, 8u * RB, LAYOUT_SW64, 0) & 0xFFFFFFFF00000000ull;
        const uint32_t a_lbo = ((RB >> 4) & 0x3FFFu) << 16;                              // next atom = next voxel row (kw + 1)
        const uint32_t b_lbo = ((((uint32_t)p.Wp * RB) >> 4) & 0x3FFFu) << 16;          // next atom = next padded row (kh - 1)
        const uint32_t x0 = a_lbo | ((smX & 0x3FFFFu) >> 4);
        const uint32_t y0 = b_lbo | ((smY & 0x3FFFFu) >> 4);
        const uint32_t x_units = p.x_slot_bytes >> 4, y_units = p.y_slot_bytes >> 4;
        const uint32_t d_tmem = tmem_base + (uint32_t)(kd * 96);
        const uint32_t idesc = p.idesc;
        int xs = 0, ys = 0;
        uint32_t xph = 0, yph = 0;
        for (int s = s_begin; s < s_end;) {
          const int d0 = s % p.D, t = s / p.D;
          const int qt = t % p.QT;
          const int len = min(p.D - d0, s_end - s);
          const int da = d0, db = d0 + len - 1;
          const int u0 = qt * WC_TK - 2 * p.Wp;
          const int hy0 = (u0 >= 0) ? (u0 / p.Wp) : -((-u0 + p.Wp - 1) / p.Wp);
          const uint32_t qoff = (uint32_t)(u0 - hy0 * p.Wp);
          const uint32_t a_off = (qoff + 2u * (uint32_t)p.Wp - 1u) * (RB >> 4);          // X row of (u, kw = 0)
          const uint32_t b_off = qoff * (RB >> 4);                                       // dY row of (u, j = 0)
          for (int v = da - 1; v <= db + 1; ++v) {
            const bool real = (v >= 0) && (v < p.D);          // X plane v exists (and was loaded)
            const int d = v - kd + 1;
            const bool has_d = (d >= da) && (d <= db);        // dY plane d of this segment pairs with X plane v for tap plane kd
            if (real) { mbar_wait(x_full + 8 * xs, xph); }
            if (has_d) { mbar_wait(y_full + 8 * ys, yph); }
            tc_fence_after();
            if (real && has_d) {
              const uint32_t a_lo = x0 + (uint32_t)xs * x_units + a_off;
              const uint32_t b_lo = y0 + (uint32_t)ys * y_units + b_off;
#pragma unroll
              for (int k = 0; k < WC_KSTEPS; ++k)
                mma_bf16_ss(d_tmem, hi | (uint64_t)(a_lo + (uint32_t)k * (16u * RB >> 4)), hi | (uint64_t)(b_lo + (uint32_t)k * (16u * RB >> 4)),
                            idesc, (started || k != 0) ? 1u : 0u);
              started = true;
            }
            if (has_d) {
              mma_commit(y_empty + 8 * ys);
              if (++ys == p.Sy) { ys = 0; yph ^= 1u; }
            }
            if (real) {
              mma_commit(x_empty + 8 * xs);
              if (++xs == p.Sx) { xs = 0; xph ^= 1u; }
            }
          }
          s += len;
        }
      }
      valid_ptr[kd] = started ? 1 : 0;
      __threadfence_block();
      mma_commit(acc_full);
    }
  } else {
    // ================================ epilogue: TMEM -> fp32 partial ws[split][tap][ci][co] ================================
    const int quarter = warp & 3;
    const int kw = quarter;                         // M atom = kw tap (atom 3 is garbage)
    mbar_wait(acc_full, 0u);
    tc_fence_after();
    if (kw < 3) {
      float* ws = p.ws[g] + (size_t)cta * 27 * p.cin * p.cout;
      const int ci = cib * WC_BLK + lane;
#pragma unroll 1
      for (int kd = 0; kd < 3; ++kd) {
        const bool ok = valid_ptr[kd] != 0;
        const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(kd * 96);
#pragma unroll 1
        for (int j = 0; j < 3; ++j) {
          uint32_t raw[32];
          if (ok) {
            tmem_ld32(taddr + (uint32_t)(j * 32), raw);
            tmem_ld_wait();
          } else {
#pragma unroll
            for (int i = 0; i < 32; ++i) raw[i] = 0u;
          }
          const int tap = kd * 9 + (2 - j) * 3 + kw;
          float4* dst = reinterpret_cast<float4*>(ws + ((size_t)tap * p.cin + ci) * p.cout + cob * WC_BLK);
#pragma unroll
          for (int i = 0; i < 8; ++i)
            dst[i] = make_float4(__uint_as_float(raw[4 * i]), __uint_as_float(raw[4 * i + 1]), __uint_as_float(raw[4 * i + 2]),
                                 __uint_as_float(raw[4 * i + 3]));
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ------------------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn wc_encode_fn() {
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

struct WcPlan {
  bool ok;
  int Wp, NHx, NHy, QT, Sx, Sy, ncib, ncob, ngv, nsplit;
  uint32_t x_slot, y_slot, x_tx, y_tx, smem;
};

static WcPlan make_wc_plan(int ng, int D, int H, int W, int cin, int cout, int ks) {
  WcPlan pl{};
  pl.ok = false;
  if (ks != 3 || cin % WC_BLK != 0 || cout % WC_BLK != 0 || cin < WC_BLK || cout < WC_BLK) return pl;
  pl.ncib = cin / WC_BLK; pl.ncob = cout / WC_BLK;
  pl.ngv = ng * pl.ncib * pl.ncob;
  if (pl.ngv > 16) return pl;      // more blocks than that (128->256) re-read the operands too often: wgrad_umma.cu is faster
  pl.nsplit = 148 / pl.ngv;
  if (D < 1 || H < 1 || W < 2) return pl;
  pl.Wp = W + 1;
  if (pl.Wp > 256 || pl.Wp * 4 > 0x3FFF) return pl;
  const uint32_t rb = WC_BLK * 2;
  pl.NHy = ((pl.Wp - 1) + (WC_TK - 1) + 2 * pl.Wp) / pl.Wp + 1;
  pl.NHx = ((pl.Wp - 1) + (WC_TK - 1) + 2 * pl.Wp - 1 + 3) / pl.Wp + 1;
  if (pl.NHx > 256 || pl.NHy > 256) return pl;
  pl.x_tx = (uint32_t)pl.NHx * pl.Wp * rb;
  pl.y_tx = (uint32_t)pl.NHy * pl.Wp * rb;
  pl.x_slot = (pl.x_tx + 1023u) & ~1023u;
  pl.y_slot = (pl.y_tx + 1023u) & ~1023u;
  // rings: X needs 3 live planes + prefetch, dY 1 live + prefetch
  for (int extra = 4; extra >= 1 && !pl.ok; --extra) {
    const int Sx = min(3 + extra, WC_MAX_SLOTS), Sy = min(1 + extra, WC_MAX_SLOTS);
    const uint32_t total = WC_FIXED_SMEM + (uint32_t)Sx * pl.x_slot + (uint32_t)Sy * pl.y_slot;
    if (total <= WC_SMEM_BUDGET) { pl.ok = true; pl.Sx = Sx; pl.Sy = Sy; pl.smem = total; }
  }
  if (!pl.ok) return pl;
  pl.QT = ((H + 2) * pl.Wp + WC_TK - 1) / WC_TK;
  return pl;
}

}  // namespace tmf

using namespace tmf;

bool tmf_conv3d_wgrad_col_supported(int ng, int D, int H, int W, int cin, int cout, int ksize) {
  if (getenv("TMF_DISABLE_UMMA") != nullptr) return false;
  return make_wc_plan(ng, D, H, W, cin, cout, ksize).ok;
}

size_t tmf_conv3d_wgrad_col_workspace(int ng, int D, int H, int W, int cin, int cout, int ksize) {
  const WcPlan pl = make_wc_plan(ng, D, H, W, cin, cout, ksize);
  if (!pl.ok) return 0;
  return (size_t)ng * pl.nsplit * 27 * cin * cout * sizeof(float);
}

// implemented in wgrad_umma.cu
int tmf_wgrad_reduce(int ng, float* const* ws, float* const* dw, int nsplit, int taps, int cin, int cout, void* stream);

int tmf_conv3d_wgrad_col(int ng, const void* const* dy, const void* const* a, float* const* dw, int B, int D, int H, int W,
                         int cin, int cout, int ksize, void* ws, size_t ws_bytes, void* stream) {
  TMF_CHECK_NG(ng);
  const WcPlan pl = make_wc_plan(ng, D, H, W, cin, cout, ksize);
  TMF_REQUIRE(pl.ok, "conv3d_wgrad_col: unsupported problem");
  const size_t per_tower = (size_t)pl.nsplit * 27 * cin * cout * sizeof(float);
  TMF_REQUIRE(ws != nullptr && ws_bytes >= per_tower * ng, "conv3d_wgrad_col: workspace too small (%zu < %zu bytes)", ws_bytes,
              per_tower * ng);
  EncodeTiledFn encode = wc_encode_fn();
  TMF_REQUIRE(encode != nullptr, "conv3d_wgrad_col: cuTensorMapEncodeTiled entry point not available");
  TMF_REQUIRE((int64_t)B * pl.QT * D < (int64_t)1 << 30, "conv3d_wgrad_col: problem too large");
  WgColParams p{};
  p.ng = ng; p.ncib = pl.ncib; p.ncob = pl.ncob; p.cin = cin; p.cout = cout; p.B = B; p.D = D; p.H = H; p.W = W;
  p.Wp = pl.Wp; p.NHx = pl.NHx; p.NHy = pl.NHy; p.QT = pl.QT; p.Sx = pl.Sx; p.Sy = pl.Sy;
  p.steps_per_group = B * pl.QT * D;
  p.x_slot_bytes = pl.x_slot; p.y_slot_bytes = pl.y_slot; p.x_tx = pl.x_tx; p.y_tx = pl.y_tx;
  p.idesc = make_idesc_bf16(128, 96, 1, 1);
  float* wsp[TMF_MAX_GROUPS];
  for (int g = 0; g < ng; ++g) {
    TMF_REQUIRE(dy[g] && a[g] && dw[g], "conv3d_wgrad_col: NULL device pointer");
    p.ws[g] = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(ws) + per_tower * g);
    wsp[g] = p.ws[g];
    cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    {
      cuuint64_t dims[5] = {(cuuint64_t)cin, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)D, (cuuint64_t)B};
      cuuint64_t strides[4] = {(cuuint64_t)cin * 2, (cuuint64_t)W * cin * 2, (cuuint64_t)H * W * cin * 2,
                               (cuuint64_t)D * H * W * cin * 2};
      cuuint32_t box[5] = {(cuuint32_t)WC_BLK, (cuuint32_t)pl.Wp, (cuuint32_t)pl.NHx, 1, 1};
      CUresult r = encode(&p.tmX[g], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<void*>(a[g]), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      TMF_REQUIRE(r == CUDA_SUCCESS, "conv3d_wgrad_col: cuTensorMapEncodeTiled(X) failed with %d", (int)r);
    }
    {
      cuuint64_t dims[5] = {(cuuint64_t)cout, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)D, (cuuint64_t)B};
      cuuint64_t strides[4] = {(cuuint64_t)cout * 2, (cuuint64_t)W * cout * 2, (cuuint64_t)H * W * cout * 2,
                               (cuuint64_t)D * H * W * cout * 2};
      cuuint32_t box[5] = {(cuuint32_t)WC_BLK, (cuuint32_t)pl.Wp, (cuuint32_t)pl.NHy, 1, 1};
      CUresult r = encode(&p.tmY[g], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<void*>(dy[g]), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      TMF_REQUIRE(r == CUDA_SUCCESS, "conv3d_wgrad_col: cuTensorMapEncodeTiled(dY) failed with %d", (int)r);
    }
  }
  cudaStream_t st = (cudaStream_t)stream;
  static bool attr_done = false;
  if (!attr_done) {
    TMF_CUDA(cudaFuncSetAttribute(conv3d_wgrad_col_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)WC_SMEM_BUDGET));
    attr_done = true;
  }
  dim3 grid(pl.ngv * pl.nsplit, 1, 1);
  launch_k(conv3d_wgrad_col_kernel, grid, WC_THREADS, pl.smem, st, p);
  TMF_LAUNCH_CHECK();
  return tmf_wgrad_reduce(ng, wsp, dw, pl.nsplit, 27, cin, cout, stream);
}

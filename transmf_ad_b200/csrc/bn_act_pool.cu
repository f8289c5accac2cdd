// bn_act_pool.cu -- the memory-bound passes between the convolutions of sNet:
//   BatchNorm3d (train / eval) -> LeakyReLU(0.01) -> {none | MaxPool3d(2,2) | AvgPool3d(2,2)}, forward and backward,
//   on NDHWC bf16 tensors, 16-byte vectorised (8 channels per thread), per-channel reductions in double.
// Reference semantics: models/networks.py:23-25, 29-34, 38-43, 47-52 (nn.BatchNorm3d eps 1e-5 momentum 0.1, biased
// variance for normalisation / unbiased into running_var; nn.LeakyReLU() slope 0.01; floor-mode pools; max-pool
// gradient to the first maximum in (d,h,w) scan order).
#include <stdlib.h>

#include "common.cuh"

namespace tmf {

// ------------------------------------------------------------------------------------------------------------
// Fixed-order sum of the TMF_STAT_ROWS partial rows of a statistics buffer (include/tmf.h, DETERMINISM): a block of 32
// warps takes 32 channels; warp w adds rows w, w+32, ... of its lane's channel (all of a warp's loads are independent and
// issued together: one L2 round trip), then warp 0 adds the 32 warp totals in index order.  Returns (for threads of
// warp 0) the two totals of channel blockIdx.x*32 + lane.
constexpr int FIN_WARPS = 32;
__device__ __forceinline__ void sum_stat_rows(const double* __restrict__ st, int C, bool on, double& t1, double& t2) {
  __shared__ double part[2][FIN_WARPS][32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + lane;
  constexpr int NR = (TMF_STAT_ROWS + FIN_WARPS - 1) / FIN_WARPS;
  double v1[NR], v2[NR];
#pragma unroll
  for (int i = 0; i < NR; ++i) {
    const int r = w + i * FIN_WARPS;
    const bool ok = on && c < C && r < TMF_STAT_ROWS;
    v1[i] = ok ? st[(size_t)r * 2 * C + c] : 0.0;
    v2[i] = ok ? st[(size_t)r * 2 * C + C + c] : 0.0;
  }
  double a1 = 0.0, a2 = 0.0;
#pragma unroll
  for (int i = 0; i < NR; ++i) { a1 += v1[i]; a2 += v2[i]; }
  part[0][w][lane] = a1;
  part[1][w][lane] = a2;
  __syncthreads();
  t1 = 0.0; t2 = 0.0;
  if (w == 0) {
#pragma unroll
    for (int i = 0; i < FIN_WARPS; ++i) { t1 += part[0][i][lane]; t2 += part[1][i][lane]; }
  }
}

__global__ void __launch_bounds__(32 * FIN_WARPS) bn_finalize_kernel(GroupPtr<const double> stats, GroupPtr<const float> gamma,
                                   GroupPtr<const float> beta, GroupPtr<float> rmean, GroupPtr<float> rvar,
                                   GroupPtr<int64_t> nbt, GroupPtr<float> coef, int C, double count, float momentum,
                                   float eps, int training) {
  const int g = blockIdx.z;
  double t1, t2;
  sum_stat_rows(stats.p[g], C, training != 0, t1, t2);
  if (threadIdx.x >= 32) return;
  const int c = blockIdx.x * 32 + threadIdx.x;
  if (c == 0 && training && nbt.p[g] != nullptr) nbt.p[g][0] += 1;
  if (c >= C) return;
  float mean, var;
  if (training) {
    const double m = t1 / count;
    double v = t2 / count - m * m;
    if (v < 0.0) v = 0.0;
    mean = (float)m;
    var = (float)v;
    if (rmean.p[g] != nullptr) {
      const double unbiased = count > 1.0 ? v * count / (count - 1.0) : v;
      rmean.p[g][c] = (1.f - momentum) * rmean.p[g][c] + momentum * mean;
      rvar.p[g][c] = (1.f - momentum) * rvar.p[g][c] + momentum * (float)unbiased;
    }
  } else {
    mean = rmean.p[g][c];
    var = rvar.p[g][c];
  }
  const float invstd = rsqrtf(var + eps);
  const float scale = gamma.p[g][c] * invstd;
  coef.p[g][c] = scale;
  coef.p[g][C + c] = beta.p[g][c] - mean * scale;
  coef.p[g][2 * C + c] = mean;
  coef.p[g][3 * C + c] = invstd;
}

__global__ void __launch_bounds__(32 * FIN_WARPS) bn_bwd_finalize_kernel(GroupPtr<const double> sums, GroupPtr<const float> coef, GroupPtr<float> dgamma,
                                       GroupPtr<float> dbeta, GroupPtr<float> dbias, GroupPtr<float> bcoef, int C,
                                       double count, int training) {
  const int g = blockIdx.z;
  double s1, s2;
  sum_stat_rows(sums.p[g], C, true, s1, s2);
  if (threadIdx.x >= 32) return;
  const int c = blockIdx.x * 32 + threadIdx.x;
  if (c >= C) return;
  dgamma.p[g][c] = (float)s2;
  dbeta.p[g][c] = (float)s1;
  if (training) {
    bcoef.p[g][c] = (float)(s1 / count);
    bcoef.p[g][C + c] = (float)(s2 / count);
    // train-mode BatchNorm cancels the conv bias exactly: sum_v dy = 0
    if (dbias.p[g] != nullptr) dbias.p[g][c] = 0.f;
  } else {
    bcoef.p[g][c] = 0.f;
    bcoef.p[g][C + c] = 0.f;
    if (dbias.p[g] != nullptr) dbias.p[g][c] = coef.p[g][c] * (float)s1;
  }
}

// ------------------------------------------------------------------------------------------------------------
struct ActPoolArgs {
  GroupPtr<const __nv_bfloat16> y;    // pre-BN conv output [B,D,H,W,C]
  GroupPtr<const float> coef;         // scale, shift, mean, invstd
  GroupPtr<const float> bcoef;        // mean(dz), mean(dz*xhat)          (bwd apply)
  GroupPtr<void> out;                 // fwd output (bf16 or fp32)
  GroupPtr<const void> dout;          // bwd: gradient w.r.t. fwd output (bf16 or fp32)
  GroupPtr<__nv_bfloat16> dy;         // bwd apply output
  GroupPtr<double> sums;              // bwd reduce output
  GroupPtr<__nv_bfloat16> ymax;       // fwd (max pool, optional): the pre-BN value behind each window's maximum
  GroupPtr<float> out32;              // fwd, dual-output variants: the fp32 value whose bf16 rounding is `out`
  int B, D, H, W, C, pool, fp32io;
  int Do, Ho, Wo;                     // forward output dims (floor)
  int Dc, Hc, Wc;                     // ceil dims (windows that touch any input voxel)
  int nch, hcr, nch_c, hcr_c;         // row chunks per output plane / rows per chunk (floor dims; ceil dims)
  float slope;
};

__device__ __forceinline__ void load8f(const void* base, int64_t elem_off, int fp32, float* f) {
  if (fp32) {
    const float4* p = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(base) + elem_off);
    const float4 a = p[0], b = p[1];
    f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w; f[4] = b.x; f[5] = b.y; f[6] = b.z; f[7] = b.w;
  } else {
    unpack8(*reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(base) + elem_off), f);
  }
}
__device__ __forceinline__ void store8f(void* base, int64_t elem_off, int fp32, const float* f) {
  if (fp32) {
    float4* p = reinterpret_cast<float4*>(reinterpret_cast<float*>(base) + elem_off);
    p[0] = make_float4(f[0], f[1], f[2], f[3]);
    p[1] = make_float4(f[4], f[5], f[6], f[7]);
  } else {
    *reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(base) + elem_off) = pack8(f);
  }
}

// KEEP (max pool only): also store ymax[B,Do,Ho,Wo,C] = the stored pre-BN value y whose activation is the window's
// maximum (first maximum in (d,h,w) scan order, torch's rule).  The backward reduction of a max-pool layer needs y
// only there (dz is zero elsewhere), so it can run on ymax + dout at pooled resolution instead of re-reading all of y:
// block 1 re-read 925 MB per step for two per-channel sums.
// DUAL: also store the fp32 value o in out32 (same layout as out); out (bf16) and ymax are the same bits as without it.
template <bool KEEP, bool DUAL = false>
__global__ void __launch_bounds__(256, DUAL ? 2 : (KEEP ? 3 : 4)) bn_act_pool_fwd_kernel(ActPoolArgs p) {
  const int g = blockIdx.z;
  const int CQ = p.C >> 3;
  const __nv_bfloat16* yg = p.y.p[g];
  // Work = units (sample, output plane, chunk of output rows); a thread keeps ONE 8-channel chunk for the whole kernel
  // (threads beyond the largest multiple of CQ idle), so the coefficients live in registers and a position costs one
  // integer division.
  const int cq = threadIdx.x % CQ, pstep = 256 / CQ;
  if ((int)threadIdx.x >= pstep * CQ) return;
  const int c0 = cq * 8;
  float sc[8], sh[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { sc[j] = p.coef.p[g][c0 + j]; sh[j] = p.coef.p[g][p.C + c0 + j]; }
  const int nunits = p.B * p.Do * p.nch;
  for (int unit = blockIdx.x; unit < nunits; unit += gridDim.x) {
    const int hc = unit % p.nch;
    const int rr = unit / p.nch;
    const int dd = rr % p.Do, n = rr / p.Do;
    const int hb = hc * p.hcr, he = min(hb + p.hcr, p.Ho);
    const int items = (he - hb) * p.Wo;
   for (int pos = threadIdx.x / CQ; pos < items; pos += pstep) {
    const int hh = pos / p.Wo;
    const int wo = pos - hh * p.Wo, ho = hb + hh;
    float o[8];
    if (p.pool == TMF_POOL_NONE) {
      float f[8];
      unpack8(*reinterpret_cast<const uint4*>(yg + ((((int64_t)n * p.D + dd) * p.H + ho) * p.W + wo) * p.C + c0), f);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float z = fmaf(f[j], sc[j], sh[j]);
        o[j] = z > 0.f ? z : z * p.slope;
      }
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = (p.pool == TMF_POOL_MAX) ? -INFINITY : 0.f;
      float yb[8];
      if (KEEP) {
#pragma unroll
        for (int j = 0; j < 8; ++j) yb[j] = 0.f;
      }
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const int di = 2 * dd + (q >> 2), hi = 2 * ho + ((q >> 1) & 1), wi = 2 * wo + (q & 1);
        float f[8];
        unpack8(*reinterpret_cast<const uint4*>(yg + ((((int64_t)n * p.D + di) * p.H + hi) * p.W + wi) * p.C + c0), f);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float z = fmaf(f[j], sc[j], sh[j]);
          const float a = z > 0.f ? z : z * p.slope;
          if (KEEP) {
            if (a > o[j]) { o[j] = a; yb[j] = f[j]; }          // strict: the first maximum wins
          } else {
            o[j] = (p.pool == TMF_POOL_MAX) ? fmaxf(o[j], a) : o[j] + a;
          }
        }
      }
      if (KEEP)
        *reinterpret_cast<uint4*>(p.ymax.p[g] + ((((int64_t)n * p.Do + dd) * p.Ho + ho) * p.Wo + wo) * p.C + c0) = pack8(yb);
      if (p.pool == TMF_POOL_AVG) {
#pragma unroll
        for (int j = 0; j < 8; ++j) o[j] *= 0.125f;
      }
    }
    const int64_t ooff = ((((int64_t)n * p.Do + dd) * p.Ho + ho) * p.Wo + wo) * p.C + c0;
    store8f(p.out.p[g], ooff, p.fp32io, o);
    if (DUAL) store8f(p.out32.p[g], ooff, 1, o);
   }
  }
}

// Per-channel partial sums of a 256-thread block, deterministically: every thread parks its 16 values in shared memory
// (red[16][256], conflict-free), then one thread per (statistic, channel) adds the 256/CQ contributions of its channel in
// thread order (four interleaved chains, fixed association) and stores the total into this block's row of the
// double[TMF_STAT_ROWS][2C] buffer (no atomics: include/tmf.h, DETERMINISM).  A thread owns channel chunk
// cq = threadIdx.x % CQ for the whole kernel.
__device__ __forceinline__ void block_channel_sums(float* red, double* rows, int C, int CQ, bool active,
                                                   const float (&s1)[8], const float (&s2)[8]) {
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    red[j * 256 + threadIdx.x] = active ? s1[j] : 0.f;
    red[(8 + j) * 256 + threadIdx.x] = active ? s2[j] : 0.f;
  }
  __syncthreads();
  const int pstep = 256 / CQ;
  for (int o = threadIdx.x; o < 2 * C; o += 256) {
    const int stat = o / C, ch = o - stat * C;
    const int cq = ch >> 3, j = ch & 7;
    const float* src = red + (stat * 8 + j) * 256 + cq;
    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
    int k = 0;
    for (; k + 3 < pstep; k += 4) {
      a0 += (double)src[k * CQ];
      a1 += (double)src[(k + 1) * CQ];
      a2 += (double)src[(k + 2) * CQ];
      a3 += (double)src[(k + 3) * CQ];
    }
    for (; k < pstep; ++k) a0 += (double)src[k * CQ];
    stat_row_store(rows, 2 * C, blockIdx.x, gridDim.x, o, (a0 + a1) + (a2 + a3));
  }
}

// Backward over 2x2x2 windows (or single voxels when pool == NONE).  REDUCE: accumulate sum dz, sum dz*xhat.
// APPLY: write dy = scale * (dz - m1 - xhat*m2) for every existing input voxel (incl. those dropped by floor pooling).
//
// ALU diet (these passes are instruction-bound, not HBM-bound, if written naively):
//  * LeakyReLU and the BatchNorm affine map are monotonic, so the max-pool arg-max is found on the raw y values
//    (times sign(scale)), first maximum in (d,h,w) scan order with a strict compare exactly like torch;
//  * only the arg-max position carries dz for a max pool, so REDUCE touches one position per channel;
//  * APPLY folds the constant part into one FMA per element:  dy = A + Bc*y (+ scale*dz at the arg-max),
//    A = scale*(m2*invstd*mean - m1),  Bc = -scale*m2*invstd.
template <bool APPLY, int POOL>
__global__ void __launch_bounds__(256, (POOL == TMF_POOL_NONE) ? 3 : 2) bn_act_pool_bwd_kernel(ActPoolArgs p) {
  const int g = blockIdx.z;
  extern __shared__ float red[];  // [16][256] (REDUCE only)
  const int CQ = p.C >> 3;
  const int Dw = APPLY ? p.Dc : p.Do, Hw = APPLY ? p.Hc : p.Ho, Ww = APPLY ? p.Wc : p.Wo;
  const __nv_bfloat16* yg = p.y.p[g];
  constexpr int NPOS = (POOL == TMF_POOL_NONE) ? 1 : 8;
  float s1[8], s2[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { s1[j] = 0.f; s2[j] = 0.f; }
  // a thread keeps ONE 8-channel chunk for the whole kernel (threads beyond the largest multiple of CQ idle):
  // coefficients in registers, one integer division per position (see the forward kernel)
  const int cq = threadIdx.x % CQ, pstep = 256 / CQ;
  const bool active = (int)threadIdx.x < pstep * CQ;
  const int c0 = cq * 8;
  float sc[8], sh[8], mu[8], is[8], cA[8], cB[8], sg[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    sc[j] = p.coef.p[g][c0 + j];
    sh[j] = p.coef.p[g][p.C + c0 + j];
    mu[j] = p.coef.p[g][2 * p.C + c0 + j];
    is[j] = p.coef.p[g][3 * p.C + c0 + j];
    sg[j] = sc[j] > 0.f ? 1.f : (sc[j] < 0.f ? -1.f : 0.f);
    if (APPLY) {
      const float m1 = p.bcoef.p[g][c0 + j], m2 = p.bcoef.p[g][p.C + c0 + j];
      cB[j] = -sc[j] * m2 * is[j];
      cA[j] = -sc[j] * m1 - cB[j] * mu[j];
    }
  }
  const int nch = APPLY ? p.nch_c : p.nch, hcr = APPLY ? p.hcr_c : p.hcr;
  const int nunits = p.B * Dw * nch;
  for (int unit = blockIdx.x; unit < nunits && active; unit += gridDim.x) {
    const int hc = unit % nch;
    const int rr = unit / nch;
    const int dw = rr % Dw, n = rr / Dw;
    const int hb = hc * hcr, he = min(hb + hcr, Hw);
    const int items = (he - hb) * Ww;
   for (int pos = threadIdx.x / CQ; pos < items; pos += pstep) {
    const int hh = pos / Ww;
    const int ww = pos - hh * Ww, hw = hb + hh;
    const bool win_ok = (POOL == TMF_POOL_NONE) || (dw < p.Do && hw < p.Ho && ww < p.Wo);
    float go[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) go[j] = 0.f;
    if (win_ok) {
      const int64_t ooff = (POOL == TMF_POOL_NONE)
                               ? ((((int64_t)n * p.D + dw) * p.H + hw) * p.W + ww) * p.C + c0
                               : ((((int64_t)n * p.Do + dw) * p.Ho + hw) * p.Wo + ww) * p.C + c0;
      load8f(p.dout.p[g], ooff, p.fp32io, go);
    }
    // gather the window (existing positions only)
    uint4 raw[NPOS];
    bool ex[NPOS];
    int64_t off[NPOS];
#pragma unroll
    for (int q = 0; q < NPOS; ++q) {
      int di, hi, wi;
      if (POOL == TMF_POOL_NONE) { di = dw; hi = hw; wi = ww; }
      else { di = 2 * dw + (q >> 2); hi = 2 * hw + ((q >> 1) & 1); wi = 2 * ww + (q & 1); }
      ex[q] = di < p.D && hi < p.H && wi < p.W;
      off[q] = ((((int64_t)n * p.D + di) * p.H + hi) * p.W + wi) * p.C + c0;
      raw[q] = ex[q] ? *reinterpret_cast<const uint4*>(yg + off[q]) : make_uint4(0u, 0u, 0u, 0u);
    }
    if (POOL == TMF_POOL_MAX) {
      // arg-max per channel on sign(scale)*y; dz only at the arg-max
      float best[8], ybest[8];
      int amax[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) { best[j] = -INFINITY; ybest[j] = 0.f; amax[j] = 0; }
      if (win_ok) {
#pragma unroll
        for (int q = 0; q < NPOS; ++q) {
          float f[8];
          unpack8(raw[q], f);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float key = f[j] * sg[j];
            if (key > best[j]) { best[j] = key; ybest[j] = f[j]; amax[j] = q; }
          }
        }
      }
      float dzs[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float z = fmaf(ybest[j], sc[j], sh[j]);
        const float dz = win_ok ? (z > 0.f ? go[j] : go[j] * p.slope) : 0.f;
        if (APPLY) {
          dzs[j] = sc[j] * dz;
        } else {
          s1[j] += dz;
          s2[j] = fmaf(dz, (ybest[j] - mu[j]) * is[j], s2[j]);
        }
      }
      if (APPLY) {
#pragma unroll
        for (int q = 0; q < NPOS; ++q) {
          if (!ex[q]) continue;
          float f[8], o[8];
          unpack8(raw[q], f);
#pragma unroll
          for (int j = 0; j < 8; ++j) o[j] = fmaf(cB[j], f[j], cA[j]) + ((win_ok && amax[j] == q) ? dzs[j] : 0.f);
          *reinterpret_cast<uint4*>(p.dy.p[g] + off[q]) = pack8(o);
        }
      }
    } else {
#pragma unroll
      for (int q = 0; q < NPOS; ++q) {
        if (!ex[q]) continue;
        float f[8], o[8];
        unpack8(raw[q], f);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float z = fmaf(f[j], sc[j], sh[j]);
          const float gsel = (POOL == TMF_POOL_AVG) ? go[j] * 0.125f : go[j];
          const float dz = z > 0.f ? gsel : gsel * p.slope;
          if (APPLY) {
            o[j] = fmaf(cB[j], f[j], cA[j]) + sc[j] * dz;
          } else {
            s1[j] += dz;
            s2[j] = fmaf(dz, (f[j] - mu[j]) * is[j], s2[j]);
          }
        }
        if (APPLY) *reinterpret_cast<uint4*>(p.dy.p[g] + off[q]) = pack8(o);
      }
    }
   }
  }
  if (!APPLY) block_channel_sums(red, p.sums.p[g], p.C, CQ, active, s1, s2);
}

// Max-pool backward reduction from ymax (see bn_act_pool_fwd_kernel<true>): sum dz, sum dz*xhat over the pooled
// positions;  dz = dout * LeakyReLU'(scale*ymax + shift),  xhat = (ymax - mean) * invstd.
// The loads of RK_U positions are issued before any of them is used (the compiler does not batch them across the loop's
// exit tests by itself: one position = 32 bytes in flight per thread left the kernel at 3.0 TB/s, ncu r2p).
constexpr int RK_U = 4;
template <bool FP32>
__global__ void __launch_bounds__(256, 2) bn_maxpool_bwd_reduce_kept_kernel(ActPoolArgs p, int npos) {
  const int g = blockIdx.z;
  extern __shared__ float red[];  // [16][256]
  const int CQ = p.C >> 3;
  const int cq = threadIdx.x % CQ, pstep = 256 / CQ;
  const bool active = (int)threadIdx.x < pstep * CQ;
  const int c0 = cq * 8;
  float sc[8], sh[8], mu[8], is[8], s1[8], s2[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    sc[j] = p.coef.p[g][c0 + j];
    sh[j] = p.coef.p[g][p.C + c0 + j];
    mu[j] = p.coef.p[g][2 * p.C + c0 + j];
    is[j] = p.coef.p[g][3 * p.C + c0 + j];
    s1[j] = 0.f; s2[j] = 0.f;
  }
  const __nv_bfloat16* ym = p.ymax.p[g];
  const uint4 zero4 = make_uint4(0u, 0u, 0u, 0u);
  if (active) {
    const int stride = gridDim.x * pstep;
    for (int pos0 = blockIdx.x * pstep + threadIdx.x / CQ; pos0 < npos; pos0 += RK_U * stride) {
      uint4 ry[RK_U], rg[RK_U], rg2[RK_U];
#pragma unroll
      for (int u = 0; u < RK_U; ++u) {
        const int pos = pos0 + u * stride;
        const bool ok = pos < npos;
        const int64_t off = (int64_t)(ok ? pos : pos0) * p.C + c0;
        ry[u] = ok ? *reinterpret_cast<const uint4*>(ym + off) : zero4;
        if (FP32) {
          const uint4* gp = reinterpret_cast<const uint4*>(reinterpret_cast<const float*>(p.dout.p[g]) + off);
          rg[u] = ok ? gp[0] : zero4;
          rg2[u] = ok ? gp[1] : zero4;
        } else {
          rg[u] = ok ? *reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(p.dout.p[g]) + off) : zero4;
        }
      }
#pragma unroll
      for (int u = 0; u < RK_U; ++u) {
        float f[8], go[8];
        unpack8(ry[u], f);
        if (FP32) {
          go[0] = __uint_as_float(rg[u].x); go[1] = __uint_as_float(rg[u].y); go[2] = __uint_as_float(rg[u].z); go[3] = __uint_as_float(rg[u].w);
          go[4] = __uint_as_float(rg2[u].x); go[5] = __uint_as_float(rg2[u].y); go[6] = __uint_as_float(rg2[u].z); go[7] = __uint_as_float(rg2[u].w);
        } else {
          unpack8(rg[u], go);          // a position beyond npos contributes dz = 0 (go = 0)
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float z = fmaf(f[j], sc[j], sh[j]);
          const float dz = z > 0.f ? go[j] : go[j] * p.slope;
          s1[j] += dz;
          s2[j] = fmaf(dz, (f[j] - mu[j]) * is[j], s2[j]);
        }
      }
    }
  }
  block_channel_sums(red, p.sums.p[g], p.C, CQ, active, s1, s2);
}

// Max-pool backward APPLY on packed bf16 pairs.  The generic kernel above spends ~23 instructions per element on the
// arg-max (compare + three selects per element in fp32) and the per-element output select: 84 M warp instructions for
// conv2.3 (ncu r2p), i.e. instruction-issue bound at 2.8 TB/s.  Here the arg-max runs on bf16x2 registers: keys
// y ^ signflip (the sign of the BatchNorm scale turns the maximum activation into a minimum of y), window maximum with
// HMNMX2, first position equal to it with HSET2 (1.0 / 0.0 per half) and two logic ops; the output is
//   dy = fma(sel, scale*dz, fma(Bc, y, A))      on packed fp32 pairs (FFMA2),  sel in {0, 1}
// -- the same values as the generic kernel (it stays the reference in the op tests).
__device__ __forceinline__ uint32_t bf2_max(uint32_t a, uint32_t b) {
  __nv_bfloat162 r = __hmax2(*reinterpret_cast<__nv_bfloat162*>(&a), *reinterpret_cast<__nv_bfloat162*>(&b));
  return *reinterpret_cast<uint32_t*>(&r);
}
__device__ __forceinline__ uint32_t bf2_eq(uint32_t a, uint32_t b) {       // 0x3F80 (1.0) per half where equal, else 0
  __nv_bfloat162 r = __heq2(*reinterpret_cast<__nv_bfloat162*>(&a), *reinterpret_cast<__nv_bfloat162*>(&b));
  return *reinterpret_cast<uint32_t*>(&r);
}
__device__ __forceinline__ uint32_t u4_get(const uint4& v, int i) { return i == 0 ? v.x : (i == 1 ? v.y : (i == 2 ? v.z : v.w)); }

template <bool FP32>
__global__ void __launch_bounds__(256, 2) bn_maxpool_bwd_apply_kernel(ActPoolArgs p) {
  const int g = blockIdx.z;
  const int CQ = p.C >> 3;
  const __nv_bfloat16* yg = p.y.p[g];
  const int cq = threadIdx.x % CQ, pstep = 256 / CQ;
  if ((int)threadIdx.x >= pstep * CQ) return;
  const int c0 = cq * 8;
  // per channel pair: packed coefficients (a zero scale needs no special case: its scale*dz is zero wherever the maximum is)
  uint64_t cA2[4], cB2[4], sc2[4], sh2[4];
#pragma unroll
  for (int j2 = 0; j2 < 4; ++j2) {
    float a[2], b[2], s_[2], h_[2];
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int c = c0 + 2 * j2 + e;
      const float sc = p.coef.p[g][c], sh = p.coef.p[g][p.C + c], mu = p.coef.p[g][2 * p.C + c], is = p.coef.p[g][3 * p.C + c];
      const float m1 = p.bcoef.p[g][c], m2 = p.bcoef.p[g][p.C + c];
      b[e] = -sc * m2 * is;
      a[e] = -sc * m1 - b[e] * mu;
      s_[e] = sc; h_[e] = sh;
    }
    cA2[j2] = pair_f32(a[0], a[1]); cB2[j2] = pair_f32(b[0], b[1]);
    sc2[j2] = pair_f32(s_[0], s_[1]); sh2[j2] = pair_f32(h_[0], h_[1]);
  }
  const int64_t sW = p.C, sH = (int64_t)p.W * p.C, sD = (int64_t)p.H * p.W * p.C;
  const int nunits = p.B * p.Dc * p.nch_c;
  for (int unit = blockIdx.x; unit < nunits; unit += gridDim.x) {
    const int hc = unit % p.nch_c;
    const int rr = unit / p.nch_c;
    const int dw = rr % p.Dc, n = rr / p.Dc;
    const int hb = hc * p.hcr_c, he = min(hb + p.hcr_c, p.Hc);
    const int items = (he - hb) * p.Wc;
    for (int pos = threadIdx.x / CQ; pos < items; pos += pstep) {
      const int hh = pos / p.Wc;
      const int ww = pos - hh * p.Wc, hw = hb + hh;
      const bool win_ok = dw < p.Do && hw < p.Ho && ww < p.Wo;
      uint4 raw[8];                                       // y of the window, overwritten pair by pair with dy
      const int64_t off0 = ((((int64_t)n * p.D + 2 * dw) * p.H + 2 * hw) * p.W + 2 * ww) * p.C + c0;
      const bool exd = 2 * dw + 1 < p.D, exh = 2 * hw + 1 < p.H, exw = 2 * ww + 1 < p.W;   // (position 0 always exists)
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const bool ex = ((q & 4) ? exd : true) && ((q & 2) ? exh : true) && ((q & 1) ? exw : true);
        const int64_t off = off0 + ((q & 4) ? sD : 0) + ((q & 2) ? sH : 0) + ((q & 1) ? sW : 0);
        raw[q] = ex ? *reinterpret_cast<const uint4*>(yg + off) : make_uint4(0u, 0u, 0u, 0u);
      }
      float go[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) go[j] = 0.f;
      if (win_ok) load8f(p.dout.p[g], ((((int64_t)n * p.Do + dw) * p.Ho + hw) * p.Wo + ww) * p.C + c0, FP32 ? 1 : 0, go);
#pragma unroll
      for (int j2 = 0; j2 < 4; ++j2) {
        // keys, window maximum, first position that holds it
        const uint32_t flip = ((lo_u32(sc2[j2]) >> 16) & 0x8000u) | (hi_u32(sc2[j2]) & 0x80000000u);   // sign bits of the scales
        uint32_t key[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) key[q] = u4_get(raw[q], j2) ^ flip;
        uint32_t m = bf2_max(bf2_max(bf2_max(key[0], key[1]), bf2_max(key[2], key[3])),
                             bf2_max(bf2_max(key[4], key[5]), bf2_max(key[6], key[7])));
        // scale*dz of the window (zero outside the pooled extent): y at the maximum = key with the sign flipped back
        const uint32_t ym = m ^ flip;
        const uint64_t y2 = pair_f32(bf16_lo(ym), bf16_hi(ym));
        const uint64_t z2 = fma2_f32(y2, sc2[j2], sh2[j2]);
        const float z0 = __uint_as_float(lo_u32(z2)), z1 = __uint_as_float(hi_u32(z2));
        const float g0 = go[2 * j2], g1 = go[2 * j2 + 1];
        const float d0 = __uint_as_float(lo_u32(sc2[j2])) * (z0 > 0.f ? g0 : g0 * p.slope);
        const float d1 = __uint_as_float(hi_u32(sc2[j2])) * (z1 > 0.f ? g1 : g1 * p.slope);
        const uint64_t dz2 = pair_f32(d0, d1);
        uint32_t found = 0u;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          const uint32_t eq = bf2_eq(key[q], m);
          const uint32_t sel = eq & ~found;                       // 1.0 (0x3F80) in the half whose FIRST maximum is here
          found |= eq;
          const uint32_t yv = u4_get(raw[q], j2);
          const uint64_t base = fma2_f32(cB2[j2], pair_f32(bf16_lo(yv), bf16_hi(yv)), cA2[j2]);
          const uint64_t o2 = fma2_f32(pair_f32(bf16_lo(sel), bf16_hi(sel)), dz2, base);
          const uint32_t pk = pack_bf16(__uint_as_float(lo_u32(o2)), __uint_as_float(hi_u32(o2)));
          if (j2 == 0) raw[q].x = pk; else if (j2 == 1) raw[q].y = pk; else if (j2 == 2) raw[q].z = pk; else raw[q].w = pk;
        }
      }
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const bool ex = ((q & 4) ? exd : true) && ((q & 2) ? exh : true) && ((q & 1) ? exw : true);
        const int64_t off = off0 + ((q & 4) ? sD : 0) + ((q & 2) ? sH : 0) + ((q & 1) ? sW : 0);
        if (ex) *reinterpret_cast<uint4*>(p.dy.p[g] + off) = raw[q];
      }
    }
  }
}

template <bool APPLY>
static void launch_bwd(const ActPoolArgs& p, dim3 grid, size_t smem, cudaStream_t st) {
  if (p.pool == TMF_POOL_MAX) launch_k(bn_act_pool_bwd_kernel<APPLY, TMF_POOL_MAX>, grid, 256, smem, st, p);
  else if (p.pool == TMF_POOL_AVG) launch_k(bn_act_pool_bwd_kernel<APPLY, TMF_POOL_AVG>, grid, 256, smem, st, p);
  else launch_k(bn_act_pool_bwd_kernel<APPLY, TMF_POOL_NONE>, grid, 256, smem, st, p);
}

static int fill_args(ActPoolArgs& p, int B, int D, int H, int W, int C, int pool, float slope, int fp32io) {
  TMF_REQUIRE(C % 8 == 0 && C >= 8 && C <= 1024, "bn_act_pool: C must be a multiple of 8 in [8,1024] (got %d)", C);
  TMF_REQUIRE(pool == TMF_POOL_NONE || pool == TMF_POOL_MAX || pool == TMF_POOL_AVG, "bn_act_pool: bad pool mode %d",
              pool);
  TMF_REQUIRE((int64_t)B * D * H * W * (C / 8) < (1ll << 31), "bn_act_pool: tensor too large for 32-bit work indices");
  p.B = B; p.D = D; p.H = H; p.W = W; p.C = C; p.pool = pool; p.slope = slope; p.fp32io = fp32io;
  if (pool == TMF_POOL_NONE) {
    p.Do = p.Dc = D; p.Ho = p.Hc = H; p.Wo = p.Wc = W;
  } else {
    p.Do = D / 2; p.Ho = H / 2; p.Wo = W / 2;
    p.Dc = (D + 1) / 2; p.Hc = (H + 1) / 2; p.Wc = (W + 1) / 2;
    TMF_REQUIRE(p.Do > 0 && p.Ho > 0 && p.Wo > 0, "bn_act_pool: volume %dx%dx%d too small to pool", D, H, W);
  }
  return 0;
}

// Units = (sample, plane, chunk of rows): enough of them to fill `waves` x 148 blocks evenly; returns the grid size.
static int plan_units(int B, int Dw, int Hw, int waves_x148, int* nch, int* hcr) {
  const int planes = B * Dw;
  int n = (waves_x148 + planes - 1) / planes;
  if (n < 1) n = 1;
  if (n > Hw) n = Hw;
  *hcr = (Hw + n - 1) / n;
  *nch = (Hw + *hcr - 1) / *hcr;
  const int units = planes * *nch;
  return units < waves_x148 ? units : waves_x148;
}

static int pick_grid(int64_t total_threads, int CQ, int64_t cap = 148 * 16) {
  int64_t blocks = (total_threads + 255) / 256;
  if (blocks > cap) blocks = cap;
  // keep (gridDim.x * 256) a multiple of CQ so that a thread's channel chunk is loop-invariant
  int64_t a = 256, b = CQ;
  while (b) { int64_t t = a % b; a = b; b = t; }
  const int64_t mult = CQ / a;
  blocks = ((blocks + mult - 1) / mult) * mult;
  return (int)blocks;
}

}  // namespace tmf

using namespace tmf;

extern "C" {

int tmf_bn_finalize(int ng, const double* const* stats, const float* const* gamma, const float* const* beta,
                    float* const* running_mean, float* const* running_var, int64_t* const* num_batches_tracked,
                    float* const* coef, int C, int64_t count, float momentum, float eps, int training, void* stream) {
  TMF_CHECK_NG(ng);
  GroupPtr<const double> gs;
  GroupPtr<const float> gg, gb;
  GroupPtr<float> grm, grv, gc;
  GroupPtr<int64_t> gn;
  if (!load_group(gs, stats, ng, training != 0, "stats") || !load_group(gg, gamma, ng, true, "gamma") ||
      !load_group(gb, beta, ng, true, "beta") || !load_group(grm, running_mean, ng, training == 0, "running_mean") ||
      !load_group(grv, running_var, ng, training == 0, "running_var") ||
      !load_group(gn, num_batches_tracked, ng, false, "num_batches_tracked") || !load_group(gc, coef, ng, true, "coef"))
    return 1;
  TMF_REQUIRE(count > 0, "bn_finalize: count must be positive");
  dim3 grid(ceil_div(C, 32), 1, ng);
  launch_k(bn_finalize_kernel, grid, 32 * FIN_WARPS, 0, (cudaStream_t)stream, gs, gg, gb, grm, grv, gn, gc, C, (double)count, momentum,
                                                             eps, training);
  TMF_LAUNCH_CHECK();
  return 0;
}

int tmf_bn_act_pool_fwd(int ng, const void* const* y, const float* const* coef, void* const* out, int out_fp32, int B,
                        int D, int H, int W, int C, int pool, float slope, void* stream) {
  TMF_CHECK_NG(ng);
  ActPoolArgs p{};
  if (fill_args(p, B, D, H, W, C, pool, slope, out_fp32)) return 1;
  if (!load_group(p.y, (const __nv_bfloat16* const*)y, ng, true, "y") || !load_group(p.coef, coef, ng, true, "coef") ||
      !load_group(p.out, (void* const*)out, ng, true, "out"))
    return 1;
  dim3 grid(plan_units(B, p.Do, p.Ho, 148 * 8, &p.nch, &p.hcr), 1, ng);
  launch_k(bn_act_pool_fwd_kernel<false>, grid, 256, 0, (cudaStream_t)stream, p);
  TMF_LAUNCH_CHECK();
  return 0;
}

int tmf_bn_act_pool_fwd_keepmax(int ng, const void* const* y, const float* const* coef, void* const* out,
                                void* const* ymax, int out_fp32, int B, int D, int H, int W, int C, float slope,
                                void* stream) {
  TMF_CHECK_NG(ng);
  ActPoolArgs p{};
  if (fill_args(p, B, D, H, W, C, TMF_POOL_MAX, slope, out_fp32)) return 1;
  if (!load_group(p.y, (const __nv_bfloat16* const*)y, ng, true, "y") || !load_group(p.coef, coef, ng, true, "coef") ||
      !load_group(p.out, (void* const*)out, ng, true, "out") ||
      !load_group(p.ymax, (__nv_bfloat16* const*)ymax, ng, true, "ymax"))
    return 1;
  dim3 grid(plan_units(B, p.Do, p.Ho, 148 * 8, &p.nch, &p.hcr), 1, ng);
  launch_k(bn_act_pool_fwd_kernel<true>, grid, 256, 0, (cudaStream_t)stream, p);
  TMF_LAUNCH_CHECK();
  return 0;
}

int tmf_bn_act_pool_fwd_dual(int ng, const void* const* y, const float* const* coef, void* const* out,
                             float* const* out32, int B, int D, int H, int W, int C, int pool, float slope, void* stream) {
  TMF_CHECK_NG(ng);
  ActPoolArgs p{};
  if (fill_args(p, B, D, H, W, C, pool, slope, 0)) return 1;
  if (!load_group(p.y, (const __nv_bfloat16* const*)y, ng, true, "y") || !load_group(p.coef, coef, ng, true, "coef") ||
      !load_group(p.out, (void* const*)out, ng, true, "out") || !load_group(p.out32, out32, ng, true, "out32"))
    return 1;
  dim3 grid(plan_units(B, p.Do, p.Ho, 148 * 8, &p.nch, &p.hcr), 1, ng);
  launch_k(bn_act_pool_fwd_kernel<false, true>, grid, 256, 0, (cudaStream_t)stream, p);
  TMF_LAUNCH_CHECK();
  return 0;
}

int tmf_bn_act_pool_fwd_keepmax_dual(int ng, const void* const* y, const float* const* coef, void* const* out,
                                     float* const* out32, void* const* ymax, int B, int D, int H, int W, int C, float slope,
                                     void* stream) {
  TMF_CHECK_NG(ng);
  ActPoolArgs p{};
  if (fill_args(p, B, D, H, W, C, TMF_POOL_MAX, slope, 0)) return 1;
  if (!load_group(p.y, (const __nv_bfloat16* const*)y, ng, true, "y") || !load_group(p.coef, coef, ng, true, "coef") ||
      !load_group(p.out, (void* const*)out, ng, true, "out") || !load_group(p.out32, out32, ng, true, "out32") ||
      !load_group(p.ymax, (__nv_bfloat16* const*)ymax, ng, true, "ymax"))
    return 1;
  dim3 grid(plan_units(B, p.Do, p.Ho, 148 * 8, &p.nch, &p.hcr), 1, ng);
  launch_k(bn_act_pool_fwd_kernel<true, true>, grid, 256, 0, (cudaStream_t)stream, p);
  TMF_LAUNCH_CHECK();
  return 0;
}

int tmf_bn_maxpool_bwd_reduce_kept(int ng, const void* const* dout, int dout_fp32, const void* const* ymax,
                                   const float* const* coef, double* const* sums, int B, int Do, int Ho, int Wo, int C,
                                   float slope, void* stream) {
  TMF_CHECK_NG(ng);
  TMF_REQUIRE(C % 8 == 0 && C >= 8 && C <= 1024, "bn_maxpool_bwd_reduce_kept: C must be a multiple of 8 in [8,1024]");
  const int64_t npos = (int64_t)B * Do * Ho * Wo;
  TMF_REQUIRE(npos > 0 && npos * (C / 8) < (1ll << 31), "bn_maxpool_bwd_reduce_kept: bad extent");
  ActPoolArgs p{};
  p.B = B; p.C = C; p.slope = slope; p.fp32io = dout_fp32; p.pool = TMF_POOL_MAX;
  if (!load_group(p.ymax, (__nv_bfloat16* const*)ymax, ng, true, "ymax") || !load_group(p.coef, coef, ng, true, "coef") ||
      !load_group(p.dout, (const void* const*)dout, ng, true, "dout") || !load_group(p.sums, sums, ng, true, "sums"))
    return 1;
  cudaStream_t st = (cudaStream_t)stream;
  const int pstep = 256 / (C / 8);
  int blocks = ceil_div(npos, (int64_t)pstep * 4);                 // >= 4 positions per thread
  if (blocks > 148) blocks = 148;                                  // one statistics row per block (<= TMF_STAT_ROWS); with two
                                                                   // towers that is 2 blocks of <= 128 registers per SM
  if (blocks < 1) blocks = 1;
  if (dout_fp32) launch_k(bn_maxpool_bwd_reduce_kept_kernel<true>, dim3(blocks, 1, ng), 256, 16 * 256 * sizeof(float), st, p, (int)npos);
  else launch_k(bn_maxpool_bwd_reduce_kept_kernel<false>, dim3(blocks, 1, ng), 256, 16 * 256 * sizeof(float), st, p, (int)npos);
  TMF_LAUNCH_CHECK();
  return 0;
}

int tmf_bn_act_pool_bwd_reduce(int ng, const void* const* dout, int dout_fp32, const void* const* y,
                               const float* const* coef, double* const* sums, int B, int D, int H, int W, int C,
                               int pool, float slope, void* stream) {
  TMF_CHECK_NG(ng);
  ActPoolArgs p{};
  if (fill_args(p, B, D, H, W, C, pool, slope, dout_fp32)) return 1;
  if (!load_group(p.y, (const __nv_bfloat16* const*)y, ng, true, "y") || !load_group(p.coef, coef, ng, true, "coef") ||
      !load_group(p.dout, (const void* const*)dout, ng, true, "dout") || !load_group(p.sums, sums, ng, true, "sums"))
    return 1;
  cudaStream_t st = (cudaStream_t)stream;
  if (pool == TMF_POOL_NONE) {
    // no pooling: dout and y have the same flat layout -- the batched-load reduction over positions (the kept-maximum
    // kernel with y in the place of ymax; same per-element arithmetic)
    const int64_t npos = (int64_t)B * D * H * W;
    p.ymax.p[0] = nullptr;
    for (int g = 0; g < ng; ++g) p.ymax.p[g] = const_cast<__nv_bfloat16*>(p.y.p[g]);
    const int pstep = 256 / (C / 8);
    int blocks = ceil_div(npos, (int64_t)pstep * RK_U);
    if (blocks > 148) blocks = 148;
    if (blocks < 1) blocks = 1;
    if (dout_fp32) launch_k(bn_maxpool_bwd_reduce_kept_kernel<true>, dim3(blocks, 1, ng), 256, 16 * 256 * sizeof(float), st, p, (int)npos);
    else launch_k(bn_maxpool_bwd_reduce_kept_kernel<false>, dim3(blocks, 1, ng), 256, 16 * 256 * sizeof(float), st, p, (int)npos);
    TMF_LAUNCH_CHECK();
    return 0;
  }
  dim3 grid(plan_units(B, p.Do, p.Ho, TMF_STAT_ROWS, &p.nch, &p.hcr), 1, ng);   // one statistics row per block
  launch_bwd<false>(p, grid, 16 * 256 * sizeof(float), st);
  TMF_LAUNCH_CHECK();
  return 0;
}

int tmf_bn_bwd_finalize(int ng, const double* const* sums, const float* const* coef, float* const* dgamma,
                        float* const* dbeta, float* const* dbias, float* const* bcoef, int C, int64_t count,
                        int training, void* stream) {
  TMF_CHECK_NG(ng);
  GroupPtr<const double> gs;
  GroupPtr<const float> gc;
  GroupPtr<float> gdg, gdb, gdbias, gbc;
  if (!load_group(gs, sums, ng, true, "sums") || !load_group(gc, coef, ng, true, "coef") ||
      !load_group(gdg, dgamma, ng, true, "dgamma") || !load_group(gdb, dbeta, ng, true, "dbeta") ||
      !load_group(gdbias, dbias, ng, false, "dbias") || !load_group(gbc, bcoef, ng, true, "bcoef"))
    return 1;
  dim3 grid(ceil_div(C, 32), 1, ng);
  launch_k(bn_bwd_finalize_kernel, grid, 32 * FIN_WARPS, 0, (cudaStream_t)stream, gs, gc, gdg, gdb, gdbias, gbc, C, (double)count,
                                                                 training);
  TMF_LAUNCH_CHECK();
  return 0;
}

int tmf_bn_act_pool_bwd_apply(int ng, const void* const* dout, int dout_fp32, const void* const* y,
                              const float* const* coef, const float* const* bcoef, void* const* dy, int B, int D,
                              int H, int W, int C, int pool, float slope, void* stream) {
  TMF_CHECK_NG(ng);
  ActPoolArgs p{};
  if (fill_args(p, B, D, H, W, C, pool, slope, dout_fp32)) return 1;
  if (!load_group(p.y, (const __nv_bfloat16* const*)y, ng, true, "y") || !load_group(p.coef, coef, ng, true, "coef") ||
      !load_group(p.bcoef, bcoef, ng, true, "bcoef") ||
      !load_group(p.dout, (const void* const*)dout, ng, true, "dout") ||
      !load_group(p.dy, (__nv_bfloat16* const*)dy, ng, true, "dy"))
    return 1;
  dim3 grid(plan_units(B, p.Dc, p.Hc, 148 * 6, &p.nch_c, &p.hcr_c), 1, ng);
  const bool generic_max = getenv("TMF_BN_GENERIC_MAXPOOL_BWD") != nullptr;            // op-test switch: the fp32 kernel
  if (pool == TMF_POOL_MAX && !generic_max) {
    if (dout_fp32) launch_k(bn_maxpool_bwd_apply_kernel<true>, grid, 256, 0, (cudaStream_t)stream, p);
    else launch_k(bn_maxpool_bwd_apply_kernel<false>, grid, 256, 0, (cudaStream_t)stream, p);
  } else {
    launch_bwd<true>(p, grid, 0, (cudaStream_t)stream);
  }
  TMF_LAUNCH_CHECK();
  return 0;
}

}  // extern "C"

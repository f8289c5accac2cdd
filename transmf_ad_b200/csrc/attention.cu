// attention.cu -- register-tiled multi-head (cross-)attention core for the SHORT token sequences of TransMF_AD
// (N = 150 tokens per modality, 300 for CrossTransformer's concatenated context; dim_head 16..64), fp32.
// Reference: models/networks.py:166-174  (dots = q k^T * scale; attn = softmax(dots); out = attn v) and its autograd.
//
// One CTA = one (batch, head) x 32 rows; warp w owns rows 4w..4w+3; a lane owns the columns lane, lane+32, ... (NPL per
// lane).  So a thread accumulates a 4 x NPL tile of the score matrix in registers: per d it needs ONE broadcast 128-bit
// shared load for its four rows (row operands are kept transposed, [d][32 rows]) and NPL conflict-free loads of the
// column operand ([col][d] with an odd pitch) for 4*NPL FMAs -- the row-per-warp kernels in fusion_ops.cu issue two
// shared loads per FMA and are LDS-bound (40-65 us per call at B=8; these take a few us).  The softmax statistics of a
// row live in one warp (shuffle reductions).  The second GEMM (P V, dS K, dS^T Q, P^T dO) runs with lane = d: P / dS
// of the warp's four rows are parked in shared memory as [col][4] so that one broadcast 128-bit load feeds four FMAs.
// The backward recomputes P from the saved log-sum-exp (no N x N tensor ever reaches HBM).
#include <math.h>
#include <stdlib.h>

#include "common.cuh"
#include "attn_args.cuh"

namespace tmf {

constexpr int TA_WARPS = 8, TA_ROWS = 32, TA_THREADS = TA_WARPS * 32;

// Staging.  Every CTA copies a few tens of KB of head slices (dh contiguous floats per token) into shared memory; what
// matters is how many loads are in flight, so the copies are 128-bit and issued in batches of four before any is
// stored (a scalar loop exposes one L2 latency per element: ~10 us per kernel).  Requires dh % 4 == 0.
// stage `rows` rows (dh floats at `src + r*row_stride`) as dst[r*ld + d]; rows >= nvalid are zeroed
__device__ __forceinline__ void stage_rows(float* dst, const float* src, int64_t row_stride, int nvalid, int rows,
                                           int dh, int ld) {
  const int dh4 = dh >> 2, total = rows * dh4;
  for (int i0 = threadIdx.x; i0 < total; i0 += 4 * TA_THREADS) {
    float4 v[4];
    int off[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = i0 + u * TA_THREADS;
      const int r = i / dh4, c = i - r * dh4;
      off[u] = (i < total) ? r * ld + 4 * c : -1;
      v[u] = (i < total && r < nvalid) ? __ldg(reinterpret_cast<const float4*>(src + (int64_t)r * row_stride) + c)
                                       : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u)
      if (off[u] >= 0) {
        float* d = dst + off[u];
        d[0] = v[u].x; d[1] = v[u].y; d[2] = v[u].z; d[3] = v[u].w;
      }
  }
}
// stage up to 32 rows transposed: dst[d*32 + r]  (lane = row: conflict-free stores)
__device__ __forceinline__ void stage_rows_t(float* dst, const float* src, int64_t row_stride, int nvalid, int dh) {
  const int dh4 = dh >> 2;
  for (int i = threadIdx.x; i < TA_ROWS * dh4; i += TA_THREADS) {
    const int r = i & (TA_ROWS - 1), c = i >> 5;
    const float4 v = (r < nvalid) ? __ldg(reinterpret_cast<const float4*>(src + (int64_t)r * row_stride) + c)
                                  : make_float4(0.f, 0.f, 0.f, 0.f);
    float* d = dst + (4 * c) * TA_ROWS + r;
    d[0] = v.x; d[TA_ROWS] = v.y; d[2 * TA_ROWS] = v.z; d[3 * TA_ROWS] = v.w;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// forward: o = softmax(q k^T * scale) v,  lse = log sum exp
// smem: Ks[Np][ld] Vs[Np][ld] Qt[dh][32] Ps[8][Np][4]          (Np = 32*NPL, ld = dh + 1)
// ---------------------------------------------------------------------------------------------------------------
template <int NPL>
__global__ void __launch_bounds__(TA_THREADS) attn_tiled_fwd_kernel(AttnArgs p) {
  extern __shared__ __align__(16) float sm[];
  constexpr int Np = 32 * NPL;
  const int dh = p.dh, ld = dh + 1, inner = p.heads * dh;
  float* Ks = sm;
  float* Vs = Ks + Np * ld;
  float* Qt = Vs + Np * ld;
  float* Ps = Qt + dh * TA_ROWS;
  const int b = blockIdx.x / p.heads, h = blockIdx.x % p.heads;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int r0 = blockIdx.y * TA_ROWS;
  const float* kvb = p.kv + (int64_t)b * p.Nk * 2 * inner + h * dh;
  stage_rows(Ks, kvb, 2 * inner, p.Nk, Np, dh, ld);
  stage_rows(Vs, kvb + inner, 2 * inner, p.Nk, Np, dh, ld);
  stage_rows_t(Qt, p.q + ((int64_t)b * p.Nq + r0) * inner + h * dh, inner, p.Nq - r0, dh);
  __syncthreads();

  float s[4][NPL];
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int j = 0; j < NPL; ++j) s[r][j] = 0.f;
#pragma unroll 4
  for (int d = 0; d < dh; ++d) {
    const float4 q4 = *reinterpret_cast<const float4*>(Qt + d * TA_ROWS + 4 * warp);
    float kk[NPL];
#pragma unroll
    for (int j = 0; j < NPL; ++j) kk[j] = Ks[(lane + 32 * j) * ld + d];
#pragma unroll
    for (int j = 0; j < NPL; ++j) {
      s[0][j] = fmaf(q4.x, kk[j], s[0][j]);
      s[1][j] = fmaf(q4.y, kk[j], s[1][j]);
      s[2][j] = fmaf(q4.z, kk[j], s[2][j]);
      s[3][j] = fmaf(q4.w, kk[j], s[3][j]);
    }
  }
  float* Pw = Ps + warp * Np * 4;
  float inv[4];
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    float mx = -INFINITY;
#pragma unroll
    for (int j = 0; j < NPL; ++j) {
      s[r][j] = (lane + 32 * j < p.Nk) ? s[r][j] * p.scale : -INFINITY;
      mx = fmaxf(mx, s[r][j]);
    }
    mx = warp_max(mx);
    float sum = 0.f;
#pragma unroll
    for (int j = 0; j < NPL; ++j) {
      const float e = __expf(s[r][j] - mx);          // exp(-inf) = 0 for the padding columns
      Pw[(lane + 32 * j) * 4 + r] = e;
      sum += e;
    }
    sum = warp_sum(sum);
    inv[r] = 1.f / sum;
    const int i = r0 + 4 * warp + r;
    if (lane == 0 && i < p.Nq) p.lse[((int64_t)b * p.heads + h) * p.Nq + i] = mx + __logf(sum);
  }
  __syncwarp();
  for (int d = lane; d < dh; d += 32) {
    float o[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 4
    for (int j = 0; j < p.Nk; ++j) {
      const float4 p4 = *reinterpret_cast<const float4*>(Pw + j * 4);
      const float v = Vs[j * ld + d];
      o[0] = fmaf(p4.x, v, o[0]); o[1] = fmaf(p4.y, v, o[1]); o[2] = fmaf(p4.z, v, o[2]); o[3] = fmaf(p4.w, v, o[3]);
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int i = r0 + 4 * warp + r;
      if (i < p.Nq) p.o[((int64_t)b * p.Nq + i) * inner + h * dh + d] = o[r] * inv[r];
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// dq[i] = scale * sum_j dS_ij k_j,   dS_ij = P_ij (dO_i . v_j - D_i),  D_i = dO_i . O_i,  P_ij = exp(s_ij*scale - lse_i)
// smem: Ks[Np][ld] Vs[Np][ld] Qt[dh][32] dOt[dh][32] dSs[8][Np][4]
// ---------------------------------------------------------------------------------------------------------------
template <int NPL>
__global__ void __launch_bounds__(TA_THREADS) attn_tiled_dq_kernel(AttnArgs p) {
  extern __shared__ __align__(16) float sm[];
  constexpr int Np = 32 * NPL;
  const int dh = p.dh, ld = dh + 1, inner = p.heads * dh;
  float* Ks = sm;
  float* Vs = Ks + Np * ld;
  float* Qt = Vs + Np * ld;
  float* dOt = Qt + dh * TA_ROWS;
  float* dSs = dOt + dh * TA_ROWS;
  const int b = blockIdx.x / p.heads, h = blockIdx.x % p.heads;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int r0 = blockIdx.y * TA_ROWS;
  const float* kvb = p.kv + (int64_t)b * p.Nk * 2 * inner + h * dh;
  const int64_t qoff = ((int64_t)b * p.Nq + r0) * inner + h * dh;
  stage_rows(Ks, kvb, 2 * inner, p.Nk, Np, dh, ld);
  stage_rows(Vs, kvb + inner, 2 * inner, p.Nk, Np, dh, ld);
  stage_rows_t(Qt, p.q + qoff, inner, p.Nq - r0, dh);
  stage_rows_t(dOt, p.dout + qoff, inner, p.Nq - r0, dh);
  __syncthreads();

  float Di[4], lse[4];
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int i = r0 + 4 * warp + r;
    float acc = 0.f;
    if (i < p.Nq)
      for (int d = lane; d < dh; d += 32)
        acc = fmaf(dOt[d * TA_ROWS + 4 * warp + r], __ldg(p.out + ((int64_t)b * p.Nq + i) * inner + h * dh + d), acc);
    Di[r] = warp_sum(acc);
    lse[r] = (i < p.Nq) ? __ldg(p.lse_in + ((int64_t)b * p.heads + h) * p.Nq + i) : 0.f;
  }
  float s[4][NPL], dp[4][NPL];
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int j = 0; j < NPL; ++j) { s[r][j] = 0.f; dp[r][j] = 0.f; }
#pragma unroll 2
  for (int d = 0; d < dh; ++d) {
    const float4 q4 = *reinterpret_cast<const float4*>(Qt + d * TA_ROWS + 4 * warp);
    const float4 g4 = *reinterpret_cast<const float4*>(dOt + d * TA_ROWS + 4 * warp);
#pragma unroll
    for (int j = 0; j < NPL; ++j) {
      const float kk = Ks[(lane + 32 * j) * ld + d], vv = Vs[(lane + 32 * j) * ld + d];
      s[0][j] = fmaf(q4.x, kk, s[0][j]); dp[0][j] = fmaf(g4.x, vv, dp[0][j]);
      s[1][j] = fmaf(q4.y, kk, s[1][j]); dp[1][j] = fmaf(g4.y, vv, dp[1][j]);
      s[2][j] = fmaf(q4.z, kk, s[2][j]); dp[2][j] = fmaf(g4.z, vv, dp[2][j]);
      s[3][j] = fmaf(q4.w, kk, s[3][j]); dp[3][j] = fmaf(g4.w, vv, dp[3][j]);
    }
  }
  float* dSw = dSs + warp * Np * 4;
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int j = 0; j < NPL; ++j) {
      const bool ok = (lane + 32 * j < p.Nk);
      const float pij = ok ? __expf(s[r][j] * p.scale - lse[r]) : 0.f;
      dSw[(lane + 32 * j) * 4 + r] = pij * (dp[r][j] - Di[r]);
    }
  __syncwarp();
  for (int d = lane; d < dh; d += 32) {
    float a[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 4
    for (int j = 0; j < p.Nk; ++j) {
      const float4 d4 = *reinterpret_cast<const float4*>(dSw + j * 4);
      const float kk = Ks[j * ld + d];
      a[0] = fmaf(d4.x, kk, a[0]); a[1] = fmaf(d4.y, kk, a[1]); a[2] = fmaf(d4.z, kk, a[2]); a[3] = fmaf(d4.w, kk, a[3]);
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int i = r0 + 4 * warp + r;
      if (i < p.Nq) p.dq[((int64_t)b * p.Nq + i) * inner + h * dh + d] = a[r] * p.scale;
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// dk[j] = scale * sum_i dS_ij q_i,   dv[j] = sum_i P_ij dO_i        (CTA = 32 key rows; columns = queries)
// smem: Qs[Np][ld] dOs[Np][ld] lses[Np] Ds[Np] Kt[dh][32] Vt[dh][32] Pw[8][Np][4] dSw[8][Np][4]      (Np = 32*NPL >= Nq)
// ---------------------------------------------------------------------------------------------------------------
template <int NPL>
__global__ void __launch_bounds__(TA_THREADS) attn_tiled_dkv_kernel(AttnArgs p) {
  extern __shared__ __align__(16) float sm[];
  constexpr int Np = 32 * NPL;
  const int dh = p.dh, ld = dh + 1, inner = p.heads * dh;
  float* Qs = sm;
  float* dOs = Qs + Np * ld;
  float* lses = dOs + Np * ld;
  float* Ds = lses + Np;
  float* Kt = Ds + Np;
  float* Vt = Kt + dh * TA_ROWS;
  float* Pws = Vt + dh * TA_ROWS;
  float* dSs = Pws + TA_WARPS * Np * 4;
  const int b = blockIdx.x / p.heads, h = blockIdx.x % p.heads;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int j0 = blockIdx.y * TA_ROWS;
  const int64_t qoff = (int64_t)b * p.Nq * inner + h * dh;
  const float* kvb = p.kv + ((int64_t)b * p.Nk + j0) * 2 * inner + h * dh;
  stage_rows(Qs, p.q + qoff, inner, p.Nq, Np, dh, ld);
  stage_rows(dOs, p.dout + qoff, inner, p.Nq, Np, dh, ld);
  stage_rows_t(Kt, kvb, 2 * inner, p.Nk - j0, dh);
  stage_rows_t(Vt, kvb + inner, 2 * inner, p.Nk - j0, dh);
  float* Os = Pws;                                       // O rows, only until D_i is known (smem_cols() sizes the area)
  stage_rows(Os, p.out + qoff, inner, p.Nq, Np, dh, ld);
  for (int i = threadIdx.x; i < Np; i += TA_THREADS)
    lses[i] = (i < p.Nq) ? __ldg(p.lse_in + ((int64_t)b * p.heads + h) * p.Nq + i) : 0.f;
  __syncthreads();
  for (int i = threadIdx.x; i < Np; i += TA_THREADS) {   // D_i = dO_i . O_i   (padding rows are zero)
    float acc = 0.f;
    for (int d = 0; d < dh; ++d) acc = fmaf(dOs[i * ld + d], Os[i * ld + d], acc);
    Ds[i] = acc;
  }
  __syncthreads();

  float s[4][NPL], dp[4][NPL];
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int j = 0; j < NPL; ++j) { s[r][j] = 0.f; dp[r][j] = 0.f; }
#pragma unroll 2
  for (int d = 0; d < dh; ++d) {
    const float4 k4 = *reinterpret_cast<const float4*>(Kt + d * TA_ROWS + 4 * warp);
    const float4 v4 = *reinterpret_cast<const float4*>(Vt + d * TA_ROWS + 4 * warp);
#pragma unroll
    for (int j = 0; j < NPL; ++j) {
      const float qq = Qs[(lane + 32 * j) * ld + d], gg = dOs[(lane + 32 * j) * ld + d];
      s[0][j] = fmaf(k4.x, qq, s[0][j]); dp[0][j] = fmaf(v4.x, gg, dp[0][j]);
      s[1][j] = fmaf(k4.y, qq, s[1][j]); dp[1][j] = fmaf(v4.y, gg, dp[1][j]);
      s[2][j] = fmaf(k4.z, qq, s[2][j]); dp[2][j] = fmaf(v4.z, gg, dp[2][j]);
      s[3][j] = fmaf(k4.w, qq, s[3][j]); dp[3][j] = fmaf(v4.w, gg, dp[3][j]);
    }
  }
  float* Pw = Pws + warp * Np * 4;
  float* dSw = dSs + warp * Np * 4;
#pragma unroll
  for (int j = 0; j < NPL; ++j) {
    const int i = lane + 32 * j;
    const bool ok = i < p.Nq;
    const float l = lses[i], Dv = Ds[i];
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const float pij = ok ? __expf(s[r][j] * p.scale - l) : 0.f;
      Pw[i * 4 + r] = pij;
      dSw[i * 4 + r] = pij * (dp[r][j] - Dv);
    }
  }
  __syncwarp();
  for (int d = lane; d < dh; d += 32) {
    float dk[4] = {0.f, 0.f, 0.f, 0.f}, dv[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 4
    for (int i = 0; i < p.Nq; ++i) {
      const float4 s4 = *reinterpret_cast<const float4*>(dSw + i * 4);
      const float4 p4 = *reinterpret_cast<const float4*>(Pw + i * 4);
      const float qq = Qs[i * ld + d], gg = dOs[i * ld + d];
      dk[0] = fmaf(s4.x, qq, dk[0]); dk[1] = fmaf(s4.y, qq, dk[1]); dk[2] = fmaf(s4.z, qq, dk[2]); dk[3] = fmaf(s4.w, qq, dk[3]);
      dv[0] = fmaf(p4.x, gg, dv[0]); dv[1] = fmaf(p4.y, gg, dv[1]); dv[2] = fmaf(p4.z, gg, dv[2]); dv[3] = fmaf(p4.w, gg, dv[3]);
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int j = j0 + 4 * warp + r;
      if (j < p.Nk) {
        float* drow = p.dkv + ((int64_t)b * p.Nk + j) * 2 * inner + h * dh;
        drow[d] = dk[r] * p.scale;
        drow[inner + d] = dv[r];
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
static bool tiled_enabled() {
  static int on = -1;
  if (on < 0) {
    const char* e = getenv("TMF_ATTN_IMPL");            // 0: the row-per-warp kernels of fusion_ops.cu
    on = (e == nullptr || atoi(e) != 0) ? 1 : 0;
  }
  return on == 1;
}

template <typename K>
static int launch_tiled(K kernel, const AttnArgs& p, dim3 grid, size_t smem, cudaStream_t st) {
  if (smem > 48 * 1024) TMF_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  launch_k(kernel, grid, TA_THREADS, smem, st, p);
  TMF_LAUNCH_CHECK();
  return 0;
}

static size_t smem_rows(int npl, int dh) {   // fwd / dq: Ks, Vs, (Qt | Qt, dOt), per-warp [Np][4]
  return sizeof(float) * ((size_t)2 * 32 * npl * (dh + 1) + (size_t)2 * dh * TA_ROWS + (size_t)TA_WARPS * 32 * npl * 4);
}
static size_t smem_cols(int npl, int dh) {   // dkv
  const size_t np = 32 * (size_t)npl;
  const size_t pds = 2 * TA_WARPS * np * 4, orows = np * (dh + 1);      // P / dS area, also the temporary home of O
  return sizeof(float) * (2 * np * (dh + 1) + 2 * np + (size_t)2 * dh * TA_ROWS + (pds > orows ? pds : orows));
}
constexpr size_t TA_SMEM_MAX = 200 * 1024;

int attn_tiled_fwd(const AttnArgs& p, cudaStream_t st) {
  if (!tiled_enabled() || p.dh > 128 || (p.dh & 3) || p.Nk > 320) return -1;
  const int npl = p.Nk <= 160 ? 5 : 10;
  const size_t smem = smem_rows(npl, p.dh);
  if (smem > TA_SMEM_MAX) return -1;
  dim3 grid(p.B * p.heads, ceil_div(p.Nq, TA_ROWS), 1);
  return npl == 5 ? launch_tiled(attn_tiled_fwd_kernel<5>, p, grid, smem, st)
                  : launch_tiled(attn_tiled_fwd_kernel<10>, p, grid, smem, st);
}

int attn_tiled_bwd(const AttnArgs& p, cudaStream_t st) {
  if (!tiled_enabled() || p.dh > 128 || (p.dh & 3) || p.Nk > 320 || p.Nq > 320) return -1;
  const int nk = p.Nk <= 160 ? 5 : 10, nq = p.Nq <= 160 ? 5 : 10;
  const size_t smem1 = smem_rows(nk, p.dh), smem2 = smem_cols(nq, p.dh);
  if (smem1 > TA_SMEM_MAX || smem2 > TA_SMEM_MAX) return -1;
  dim3 grid1(p.B * p.heads, ceil_div(p.Nq, TA_ROWS), 1), grid2(p.B * p.heads, ceil_div(p.Nk, TA_ROWS), 1);
  int rc = nk == 5 ? launch_tiled(attn_tiled_dq_kernel<5>, p, grid1, smem1, st)
                   : launch_tiled(attn_tiled_dq_kernel<10>, p, grid1, smem1, st);
  if (rc) return rc;
  return nq == 5 ? launch_tiled(attn_tiled_dkv_kernel<5>, p, grid2, smem2, st)
                 : launch_tiled(attn_tiled_dkv_kernel<10>, p, grid2, smem2, st);
}

}  // namespace tmf

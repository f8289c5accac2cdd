// fusion_ops.cu -- kernels of the cross-modal fusion transformer and the small heads (fp32 tensors):
//   Linear forward / dgrad / wgrad (one tiled GEMM with fused bias, exact GELU and residual epilogues),
//   LayerNorm fwd/bwd (warp per row, float4), GELU backward, short-sequence multi-head cross attention fwd/bwd
//   (K/V resident in shared memory, warp-level softmax reductions), token pooling (GAP + GMP) and the
//   gradient-reversal scale.  Reference: models/networks.py:114-175, 215-281; models/gradient_reversal/functional.py.
#include <stdlib.h>

#include "common.cuh"
#include "attn_args.cuh"

namespace tmf {

// ------------------------------------------------------------------------------------------------------------
// C[M,N] (+)= epilogue( sum_k A(m,k) * B(k,n) ),  A(m,k) = A[m*sAm + k*sAk],  B(k,n) = B[k*sBk + n*sBn]
// ------------------------------------------------------------------------------------------------------------
constexpr int G_TM = 64, G_TN = 64, G_TK = 16, G_PAD = 4;
constexpr int G_SPLIT_K = 64;          // K elements per CTA when a GEMM is split along K (weight gradients: K = B*tokens)

struct GemmArgs {
  const float* A; const float* B; float* C;
  const float* bias; const float* residual; float* pre;
  int M, N, K;
  int64_t sAm, sAk, sBk, sBn;
  int act, accumulate;
  int kchunk;                          // 0: whole K in one CTA; else K range per blockIdx.z: partial tiles go to `part`
  float* part;                         // [gridDim.z][M][N] split-K partials (caller scratch)
  unsigned* tickets;                   // one per output tile (zero; self-resetting): the last split adds the partials in order
};

// Split-K epilogue: after every thread of the block has stored its partial outputs to p.part[blockIdx.z], the last of
// the gridDim.z blocks of this output tile adds the splits in index order (deterministic) and writes C.
__device__ __forceinline__ void splitk_finish(const GemmArgs& p, int m0, int n0, int TM, int TN) {
  if (!last_block_arrives(p.tickets + (blockIdx.y * gridDim.x + blockIdx.x), gridDim.z)) return;
  const size_t mn = (size_t)p.M * p.N;
  for (int idx = threadIdx.x; idx < TM * TN; idx += blockDim.x) {
    const int m = m0 + idx / TN, n = n0 + idx % TN;
    if (m >= p.M || n >= p.N) continue;
    const size_t o = (size_t)m * p.N + n;
    float s = 0.f;
    for (unsigned z = 0; z < gridDim.z; ++z) s += __ldcg(p.part + z * mn + o);
    p.C[o] = s;
  }
}

__device__ __forceinline__ float gelu_exact(float x) { return 0.5f * x * (1.f + erff(x * 0.70710678118654752440f)); }

// These GEMMs are tiny (M = B*150 rows, K, N <= 512): what matters is latency, so the global loads of tile k+1 are
// issued before the FMAs of tile k (register double buffering), and long-K problems are split over blockIdx.z.
__global__ void __launch_bounds__(256) gemm_kernel(GemmArgs p) {
  __shared__ __align__(16) float As[G_TK][G_TM + G_PAD];
  __shared__ __align__(16) float Bs[G_TK][G_TN + G_PAD];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int m0 = blockIdx.y * G_TM, n0 = blockIdx.x * G_TN;
  const int kb = p.kchunk ? blockIdx.z * p.kchunk : 0;
  const int ke = p.kchunk ? min(p.K, kb + p.kchunk) : p.K;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  const bool a_kfast = (p.sAk == 1);
  const bool b_kfast = (p.sBk == 1);
  float ra[4], rb[4];
  auto load_tile = [&](int k0) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      int mm, kk;
      if (a_kfast) { kk = tid & 15; mm = (tid >> 4) + 16 * i; } else { mm = tid & 63; kk = (tid >> 6) + 4 * i; }
      const int m = m0 + mm, k = k0 + kk;
      ra[i] = (m < p.M && k < ke) ? __ldg(p.A + m * p.sAm + k * p.sAk) : 0.f;
      int nn, kb2;
      if (b_kfast) { kb2 = tid & 15; nn = (tid >> 4) + 16 * i; } else { nn = tid & 63; kb2 = (tid >> 6) + 4 * i; }
      const int n = n0 + nn, k2 = k0 + kb2;
      rb[i] = (n < p.N && k2 < ke) ? __ldg(p.B + k2 * p.sBk + n * p.sBn) : 0.f;
    }
  };
  load_tile(kb);
  for (int k0 = kb; k0 < ke; k0 += G_TK) {
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if (a_kfast) As[tid & 15][(tid >> 4) + 16 * i] = ra[i]; else As[(tid >> 6) + 4 * i][tid & 63] = ra[i];
      if (b_kfast) Bs[tid & 15][(tid >> 4) + 16 * i] = rb[i]; else Bs[(tid >> 6) + 4 * i][tid & 63] = rb[i];
    }
    __syncthreads();
    if (k0 + G_TK < ke) load_tile(k0 + G_TK);         // in flight while this tile is multiplied
#pragma unroll
    for (int k = 0; k < G_TK; ++k) {
      const float4 av = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
      const float4 bv = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
      const float a4[4] = {av.x, av.y, av.z, av.w};
      const float b4[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a4[i], b4[j], acc[i][j]);
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + ty * 4 + i;
    if (m >= p.M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n >= p.N) continue;
      float v = acc[i][j];
      const int64_t o = (int64_t)m * p.N + n;
      if (p.kchunk) { p.part[(size_t)blockIdx.z * p.M * p.N + o] = v; continue; }
      if (p.bias) v += p.bias[n];
      if (p.pre) p.pre[o] = v;
      if (p.act == 1) v = gelu_exact(v);
      if (p.residual) v += p.residual[o];
      if (p.accumulate) v += p.C[o];
      p.C[o] = v;
    }
  }
  if (p.kchunk) splitk_finish(p, m0, n0, G_TM, G_TN);
}

// column sums: out[n] = sum over m of x[m,n].  grid.y splits the rows; partial sums go to part[gridDim.y][N] and the last
// block of a column group adds them in index order (deterministic; no atomics, nothing to zero).
__global__ void colsum_kernel(const float* __restrict__ x, float* __restrict__ out, int M, int N, int rows_per_block,
                              float* __restrict__ partbuf, unsigned* __restrict__ tickets) {
  __shared__ float part[8][33];
  const int n = blockIdx.x * 32 + (threadIdx.x & 31);
  const int r = threadIdx.x >> 5;
  const int mb = blockIdx.y * rows_per_block, me = min(M, mb + rows_per_block);
  float s = 0.f;
  if (n < N) {
#pragma unroll 4
    for (int m = mb + r; m < me; m += 8) s += x[(int64_t)m * N + n];
  }
  part[r][threadIdx.x & 31] = s;
  __syncthreads();
  if (r == 0 && n < N) {
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) t += part[i][threadIdx.x & 31];
    partbuf[(size_t)blockIdx.y * N + n] = t;
  }
  if (!last_block_arrives(tickets + blockIdx.x, gridDim.y)) return;
  if (r == 0 && n < N) {
    float t = 0.f;
    for (unsigned y = 0; y < gridDim.y; ++y) t += __ldcg(partbuf + (size_t)y * N + n);
    out[n] = t;
  }
}

// ------------------------------------------------------------------------------------------------------------
// LayerNorm: one warp per row, dim % 4 == 0, dim <= 1024
// ------------------------------------------------------------------------------------------------------------
constexpr int LN_MAXV = 8;  // float4 per lane

__global__ void __launch_bounds__(256)
layernorm_fwd_kernel(const float* __restrict__ x, const float* __restrict__ gamma, const float* __restrict__ beta,
                     const float* __restrict__ residual, float* __restrict__ y, float* __restrict__ mean_out,
                     float* __restrict__ rstd_out, int rows, int dim, float eps) {
  const int lane = threadIdx.x & 31;
  const int nv = dim >> 2;
  for (int row = blockIdx.x * 8 + (threadIdx.x >> 5); row < rows; row += gridDim.x * 8) {
    const float4* xr = reinterpret_cast<const float4*>(x + (int64_t)row * dim);
    float4 v[LN_MAXV];
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < LN_MAXV; ++i) {
      const int c = lane + 32 * i;
      if (c < nv) { v[i] = xr[c]; s += v[i].x + v[i].y + v[i].z + v[i].w; }
    }
    const float mean = warp_sum(s) / dim;
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < LN_MAXV; ++i) {
      const int c = lane + 32 * i;
      if (c < nv) {
        const float a = v[i].x - mean, b = v[i].y - mean, cc = v[i].z - mean, d = v[i].w - mean;
        q += a * a + b * b + cc * cc + d * d;
      }
    }
    const float rstd = rsqrtf(warp_sum(q) / dim + eps);
    if (lane == 0) { mean_out[row] = mean; rstd_out[row] = rstd; }
    float4* yr = reinterpret_cast<float4*>(y + (int64_t)row * dim);
    const float4* rr = residual ? reinterpret_cast<const float4*>(residual + (int64_t)row * dim) : nullptr;
#pragma unroll
    for (int i = 0; i < LN_MAXV; ++i) {
      const int c = lane + 32 * i;
      if (c < nv) {
        const float4 gm = reinterpret_cast<const float4*>(gamma)[c];
        const float4 bt = reinterpret_cast<const float4*>(beta)[c];
        float4 o;
        o.x = (v[i].x - mean) * rstd * gm.x + bt.x;
        o.y = (v[i].y - mean) * rstd * gm.y + bt.y;
        o.z = (v[i].z - mean) * rstd * gm.z + bt.z;
        o.w = (v[i].w - mean) * rstd * gm.w + bt.w;
        if (rr) { const float4 r4 = rr[c]; o.x += r4.x; o.y += r4.y; o.z += r4.z; o.w += r4.w; }
        yr[c] = o;
      }
    }
  }
}

__global__ void __launch_bounds__(256)
layernorm_bwd_kernel(const float* __restrict__ dy, const float* __restrict__ x, const float* __restrict__ gamma,
                     const float* __restrict__ mean, const float* __restrict__ rstd, float* __restrict__ dx,
                     float* __restrict__ dgamma, float* __restrict__ dbeta, int rows, int dim, int accumulate,
                     float* __restrict__ partbuf, unsigned* __restrict__ ticket) {
  extern __shared__ float sm[];  // [2][dim]
  for (int i = threadIdx.x; i < 2 * dim; i += blockDim.x) sm[i] = 0.f;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int nv = dim >> 2;
  float4 ag[LN_MAXV], ab[LN_MAXV];
#pragma unroll
  for (int i = 0; i < LN_MAXV; ++i) { ag[i] = make_float4(0, 0, 0, 0); ab[i] = make_float4(0, 0, 0, 0); }
  for (int row = blockIdx.x * 8 + (threadIdx.x >> 5); row < rows; row += gridDim.x * 8) {
    const float4* xr = reinterpret_cast<const float4*>(x + (int64_t)row * dim);
    const float4* gr = reinterpret_cast<const float4*>(dy + (int64_t)row * dim);
    const float mu = mean[row], rs = rstd[row];
    float4 xh[LN_MAXV], gg[LN_MAXV];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < LN_MAXV; ++i) {
      const int c = lane + 32 * i;
      if (c < nv) {
        const float4 xv = xr[c], gv = gr[c], gm = reinterpret_cast<const float4*>(gamma)[c];
        xh[i] = make_float4((xv.x - mu) * rs, (xv.y - mu) * rs, (xv.z - mu) * rs, (xv.w - mu) * rs);
        gg[i] = make_float4(gv.x * gm.x, gv.y * gm.y, gv.z * gm.z, gv.w * gm.w);
        s1 += gg[i].x + gg[i].y + gg[i].z + gg[i].w;
        s2 += gg[i].x * xh[i].x + gg[i].y * xh[i].y + gg[i].z * xh[i].z + gg[i].w * xh[i].w;
        ag[i].x += gv.x * xh[i].x; ag[i].y += gv.y * xh[i].y; ag[i].z += gv.z * xh[i].z; ag[i].w += gv.w * xh[i].w;
        ab[i].x += gv.x; ab[i].y += gv.y; ab[i].z += gv.z; ab[i].w += gv.w;
      }
    }
    s1 = warp_sum(s1) / dim;
    s2 = warp_sum(s2) / dim;
    float4* dr = reinterpret_cast<float4*>(dx + (int64_t)row * dim);
#pragma unroll
    for (int i = 0; i < LN_MAXV; ++i) {
      const int c = lane + 32 * i;
      if (c < nv) {
        float4 o;
        o.x = rs * (gg[i].x - s1 - xh[i].x * s2);
        o.y = rs * (gg[i].y - s1 - xh[i].y * s2);
        o.z = rs * (gg[i].z - s1 - xh[i].z * s2);
        o.w = rs * (gg[i].w - s1 - xh[i].w * s2);
        if (accumulate) { const float4 old = dr[c]; o.x += old.x; o.y += old.y; o.z += old.z; o.w += old.w; }
        dr[c] = o;
      }
    }
  }
  // deterministic: the warps add their column sums into shared memory one after the other, the block stores its partial,
  // and the last block to finish adds the blocks' partials in index order (dgamma / dbeta are overwritten)
  for (int w = 0; w < 8; ++w) {
    if ((int)(threadIdx.x >> 5) == w) {
#pragma unroll
      for (int i = 0; i < LN_MAXV; ++i) {
        const int c = lane + 32 * i;
        if (c < nv) {
          float4* sg = reinterpret_cast<float4*>(sm) + c;
          float4* sb = reinterpret_cast<float4*>(sm + dim) + c;
          float4 a = *sg, b = *sb;
          a.x += ag[i].x; a.y += ag[i].y; a.z += ag[i].z; a.w += ag[i].w;
          b.x += ab[i].x; b.y += ab[i].y; b.z += ab[i].z; b.w += ab[i].w;
          *sg = a; *sb = b;
        }
      }
    }
    __syncthreads();
  }
  for (int i = threadIdx.x; i < 2 * dim; i += blockDim.x) partbuf[(size_t)blockIdx.x * 2 * dim + i] = sm[i];
  if (!last_block_arrives(ticket, gridDim.x)) return;
  for (int i = threadIdx.x; i < 2 * dim; i += blockDim.x) {
    float t = 0.f;
    for (unsigned b = 0; b < gridDim.x; ++b) t += __ldcg(partbuf + (size_t)b * 2 * dim + i);
    if (i < dim) dgamma[i] = t; else dbeta[i - dim] = t;
  }
}

// ------------------------------------------------------------------------------------------------------------
__global__ void gelu_bwd_kernel(const float4* __restrict__ dy, const float4* __restrict__ pre, float4* __restrict__ dx,
                                int64_t n4) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    const float4 g = dy[i], x = pre[i];
    float4 o;
    const float xs[4] = {x.x, x.y, x.z, x.w}, gs[4] = {g.x, g.y, g.z, g.w};
    float os[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float cdf = 0.5f * (1.f + erff(xs[j] * 0.70710678118654752440f));
      const float pdf = 0.39894228040143267794f * __expf(-0.5f * xs[j] * xs[j]);
      os[j] = gs[j] * (cdf + xs[j] * pdf);
    }
    o.x = os[0]; o.y = os[1]; o.z = os[2]; o.w = os[3];
    dx[i] = o;
  }
}

__global__ void scale_kernel(const float* __restrict__ x, float* __restrict__ y, float alpha,
                             const float* __restrict__ alpha_dev, int64_t n) {
  if (alpha_dev != nullptr) alpha *= alpha_dev[0];
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    y[i] = alpha * x[i];
}

// ------------------------------------------------------------------------------------------------------------
// attention.  grid = (B*heads, row splits); K,V (fwd, dq) or Q,dO (dk/dv) of one (batch, head) live in smem.
// ------------------------------------------------------------------------------------------------------------
constexpr int AT_WARPS = 8;
constexpr int AT_ROWS = 32;  // rows per block

// smem: Ks[Nk][dh+1], Vs[Nk][dh+1], sc[AT_WARPS][Nk], qs[AT_WARPS][dh]
__global__ void __launch_bounds__(AT_WARPS * 32) attn_fwd_kernel(AttnArgs p) {
  extern __shared__ float sm[];
  const int dh = p.dh, ld = dh + 1, inner = p.heads * dh;
  float* Ks = sm;
  float* Vs = Ks + p.Nk * ld;
  float* sc = Vs + p.Nk * ld;
  float* qs = sc + AT_WARPS * p.Nk;
  const int b = blockIdx.x / p.heads, h = blockIdx.x % p.heads;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < p.Nk * dh; i += blockDim.x) {
    const int j = i / dh, d = i % dh;
    const float* row = p.kv + ((int64_t)b * p.Nk + j) * 2 * inner;
    Ks[j * ld + d] = row[h * dh + d];
    Vs[j * ld + d] = row[inner + h * dh + d];
  }
  __syncthreads();
  const int r0 = blockIdx.y * AT_ROWS;
  for (int i = r0 + warp; i < min(p.Nq, r0 + AT_ROWS); i += AT_WARPS) {
    const float* qrow = p.q + ((int64_t)b * p.Nq + i) * inner + h * dh;
    for (int d = lane; d < dh; d += 32) qs[warp * dh + d] = qrow[d];
    __syncwarp();
    float mx = -INFINITY;
    for (int j = lane; j < p.Nk; j += 32) {
      float s = 0.f;
      for (int d = 0; d < dh; ++d) s = fmaf(qs[warp * dh + d], Ks[j * ld + d], s);
      s *= p.scale;
      sc[warp * p.Nk + j] = s;
      mx = fmaxf(mx, s);
    }
    mx = warp_max(mx);
    float sum = 0.f;
    for (int j = lane; j < p.Nk; j += 32) {
      const float e = __expf(sc[warp * p.Nk + j] - mx);
      sc[warp * p.Nk + j] = e;
      sum += e;
    }
    sum = warp_sum(sum);
    __syncwarp();
    const float inv = 1.f / sum;
    for (int d = lane; d < dh; d += 32) {
      float o = 0.f;
      for (int j = 0; j < p.Nk; ++j) o = fmaf(sc[warp * p.Nk + j], Vs[j * ld + d], o);
      p.o[((int64_t)b * p.Nq + i) * inner + h * dh + d] = o * inv;
    }
    if (lane == 0) p.lse[((int64_t)b * p.heads + h) * p.Nq + i] = mx + __logf(sum);
    __syncwarp();
  }
}

// dq: same staging as forward.  extra smem: dos[AT_WARPS][dh]
__global__ void __launch_bounds__(AT_WARPS * 32) attn_bwd_dq_kernel(AttnArgs p) {
  extern __shared__ float sm[];
  const int dh = p.dh, ld = dh + 1, inner = p.heads * dh;
  float* Ks = sm;
  float* Vs = Ks + p.Nk * ld;
  float* sc = Vs + p.Nk * ld;
  float* qs = sc + AT_WARPS * p.Nk;
  float* dos = qs + AT_WARPS * dh;
  const int b = blockIdx.x / p.heads, h = blockIdx.x % p.heads;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < p.Nk * dh; i += blockDim.x) {
    const int j = i / dh, d = i % dh;
    const float* row = p.kv + ((int64_t)b * p.Nk + j) * 2 * inner;
    Ks[j * ld + d] = row[h * dh + d];
    Vs[j * ld + d] = row[inner + h * dh + d];
  }
  __syncthreads();
  const int r0 = blockIdx.y * AT_ROWS;
  for (int i = r0 + warp; i < min(p.Nq, r0 + AT_ROWS); i += AT_WARPS) {
    const int64_t ro = ((int64_t)b * p.Nq + i) * inner + h * dh;
    float dsum = 0.f;
    for (int d = lane; d < dh; d += 32) {
      qs[warp * dh + d] = p.q[ro + d];
      const float g = p.dout[ro + d];
      dos[warp * dh + d] = g;
      dsum = fmaf(g, p.out[ro + d], dsum);
    }
    const float Di = warp_sum(dsum);
    const float lse = p.lse_in[((int64_t)b * p.heads + h) * p.Nq + i];
    __syncwarp();
    for (int j = lane; j < p.Nk; j += 32) {
      float s = 0.f, dp = 0.f;
      for (int d = 0; d < dh; ++d) {
        s = fmaf(qs[warp * dh + d], Ks[j * ld + d], s);
        dp = fmaf(dos[warp * dh + d], Vs[j * ld + d], dp);
      }
      const float pj = __expf(s * p.scale - lse);
      sc[warp * p.Nk + j] = pj * (dp - Di);
    }
    __syncwarp();
    for (int d = lane; d < dh; d += 32) {
      float a = 0.f;
      for (int j = 0; j < p.Nk; ++j) a = fmaf(sc[warp * p.Nk + j], Ks[j * ld + d], a);
      p.dq[ro + d] = a * p.scale;
    }
    __syncwarp();
  }
}

// dk, dv: smem Qs[Nq][dh+1], dOs[Nq][dh+1], lses[Nq], Ds[Nq], pw[AT_WARPS][Nq], dsw[AT_WARPS][Nq], ks/vs[AT_WARPS][dh]
__global__ void __launch_bounds__(AT_WARPS * 32) attn_bwd_dkv_kernel(AttnArgs p) {
  extern __shared__ float sm[];
  const int dh = p.dh, ld = dh + 1, inner = p.heads * dh;
  float* Qs = sm;
  float* dOs = Qs + p.Nq * ld;
  float* lses = dOs + p.Nq * ld;
  float* Ds = lses + p.Nq;
  float* pw = Ds + p.Nq;
  float* dsw = pw + AT_WARPS * p.Nq;
  float* ks = dsw + AT_WARPS * p.Nq;
  float* vs = ks + AT_WARPS * dh;
  const int b = blockIdx.x / p.heads, h = blockIdx.x % p.heads;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < p.Nq * dh; i += blockDim.x) {
    const int r = i / dh, d = i % dh;
    const int64_t off = ((int64_t)b * p.Nq + r) * inner + h * dh + d;
    Qs[r * ld + d] = p.q[off];
    dOs[r * ld + d] = p.dout[off];
  }
  for (int r = threadIdx.x; r < p.Nq; r += blockDim.x) lses[r] = p.lse_in[((int64_t)b * p.heads + h) * p.Nq + r];
  __syncthreads();
  for (int r = warp; r < p.Nq; r += AT_WARPS) {
    float s = 0.f;
    for (int d = lane; d < dh; d += 32)
      s = fmaf(dOs[r * ld + d], p.out[((int64_t)b * p.Nq + r) * inner + h * dh + d], s);
    s = warp_sum(s);
    if (lane == 0) Ds[r] = s;
  }
  __syncthreads();
  const int j0 = blockIdx.y * AT_ROWS;
  for (int j = j0 + warp; j < min(p.Nk, j0 + AT_ROWS); j += AT_WARPS) {
    const float* row = p.kv + ((int64_t)b * p.Nk + j) * 2 * inner;
    for (int d = lane; d < dh; d += 32) {
      ks[warp * dh + d] = row[h * dh + d];
      vs[warp * dh + d] = row[inner + h * dh + d];
    }
    __syncwarp();
    for (int i = lane; i < p.Nq; i += 32) {
      float s = 0.f, dp = 0.f;
      for (int d = 0; d < dh; ++d) {
        s = fmaf(Qs[i * ld + d], ks[warp * dh + d], s);
        dp = fmaf(dOs[i * ld + d], vs[warp * dh + d], dp);
      }
      const float pij = __expf(s * p.scale - lses[i]);
      pw[warp * p.Nq + i] = pij;
      dsw[warp * p.Nq + i] = pij * (dp - Ds[i]);
    }
    __syncwarp();
    float* drow = p.dkv + ((int64_t)b * p.Nk + j) * 2 * inner;
    for (int d = lane; d < dh; d += 32) {
      float dk = 0.f, dv = 0.f;
      for (int i = 0; i < p.Nq; ++i) {
        dk = fmaf(dsw[warp * p.Nq + i], Qs[i * ld + d], dk);
        dv = fmaf(pw[warp * p.Nq + i], dOs[i * ld + d], dv);
      }
      drow[h * dh + d] = dk * p.scale;
      drow[inner + h * dh + d] = dv;
    }
    __syncwarp();
  }
}

// ------------------------------------------------------------------------------------------------------------
// One block = 32 channels of one batch element; warp w reads tokens w, w+8, ... (all its loads independent: the one-thread-
// per-column loop exposed ~40 dependent L2 round trips, 27 us for 150 tokens) and the eight partial results meet in shared
// memory: sums added in warp order (deterministic), maximum with the smallest token index on ties (torch's first maximum).
constexpr int TP_WARPS = 8;
__global__ void __launch_bounds__(32 * TP_WARPS) token_pool_fwd_kernel(const float* __restrict__ x, float* __restrict__ mean,
                                                                      float* __restrict__ mx, int32_t* __restrict__ amax, int B,
                                                                      int N, int C) {
  __shared__ float ssum[TP_WARPS][32], sbest[TP_WARPS][32];
  __shared__ int sidx[TP_WARPS][32];
  const int cblocks = (C + 31) / 32;
  const int b = blockIdx.x / cblocks, c = (blockIdx.x % cblocks) * 32 + (threadIdx.x & 31);
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float s = 0.f, best = -INFINITY;
  int bi = 0x7fffffff;
  if (c < C) {
    const float* xp = x + (int64_t)b * N * C + c;
#pragma unroll 4
    for (int n = w; n < N; n += TP_WARPS) {
      const float v = xp[(int64_t)n * C];
      s += v;
      if (v > best) { best = v; bi = n; }
    }
  }
  ssum[w][lane] = s; sbest[w][lane] = best; sidx[w][lane] = bi;
  __syncthreads();
  if (w == 0 && c < C) {
    float t = 0.f, bb = -INFINITY;
    int ii = 0x7fffffff;
#pragma unroll
    for (int k = 0; k < TP_WARPS; ++k) {
      t += ssum[k][lane];
      const float v = sbest[k][lane];
      const int i = sidx[k][lane];
      if (v > bb || (v == bb && i < ii)) { bb = v; ii = i; }
    }
    if (ii == 0x7fffffff) ii = 0;
    const int idx = b * C + c;
    if (mean) mean[idx] = t / N;
    if (mx) { mx[idx] = bb; amax[idx] = ii; }
  }
}

__global__ void token_pool_bwd_kernel(const float* __restrict__ dmean, const float* __restrict__ dmax,
                                      const int32_t* __restrict__ amax, float* __restrict__ dx, int B, int N, int C,
                                      int accumulate) {
  const int64_t total = (int64_t)B * N * C;
  const float invn = 1.f / N;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % C);
    const int n = (int)((i / C) % N);
    const int b = (int)(i / ((int64_t)C * N));
    float v = 0.f;
    if (dmean) v += dmean[b * C + c] * invn;
    if (dmax && amax[b * C + c] == n) v += dmax[b * C + c];
    if (accumulate) v += dx[i];
    dx[i] = v;
  }
}


// ------------------------------------------------------------------------------------------------------------
// Linear GEMM for the shapes the fusion transformer actually runs (every extent a multiple of 4, 16-byte aligned
// rows), built for latency.  32 x 32 output tile, 256 threads = 4 K-GROUPS of 64 threads.  A "super-slice" is four
// 32-wide K slices; it moves global -> shared with 16-byte cp.async into one of two buffers, so the loads of the next
// super-slice are in flight while one is multiplied (gemm_kernel exposes one global-load latency per 16-wide slice:
// ~1 us x K/16, i.e. 8-30 us for these GEMMs whose arithmetic is ~1 us).  Group g
// multiplies slice g of every super-slice into its own 4 x 4 register tiles, and the four partial tiles meet in shared
// memory at the end.  Per thread a K = 128 GEMM is 512 FMAs instead of 2048 for one thread per 4 x 4 outputs over the
// whole of K, and M = 1200, N = 128 is 152 CTAs of 8 warps -- these GEMMs are bound by the serial FMA chain of a thread
// plus one load latency, not by throughput.
//   AKF / BKF: the operand is contiguous along k in global memory (x and w of the forward pass; dy of dgrad).  It is
//   kept as [row][k] in shared memory and read four k at a time; rows are interleaved over the threads (row = t + 8*i)
//   so that the 144-byte row pitch spreads a quarter-warp over all 32 banks.  Otherwise the operand is contiguous along
//   m / n (w of dgrad, dy and x of wgrad), kept as [k][m|n] and read as one float4 per k.
// ------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void cp_async16(float* smem_dst, const float* gsrc, bool valid) {
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
  const int n = valid ? 16 : 0;                    // src-size 0: the 16 bytes are zero-filled, gsrc is not read
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(gsrc), "r"(n) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

constexpr int V_TM = 32, V_TN = 32, V_TK = 32, V_GROUPS = 4, V_THREADS = 64 * V_GROUPS, V_BUFS = 2;
constexpr int V_PITCH = 36;                                        // both [row][k] (32 + 4) and [k][m|n] (32 + 4) tiles
constexpr int V_SLICE_FLOATS = 2 * 32 * V_PITCH;                   // A tile + B tile of one K slice
constexpr int V_SUPER_FLOATS = V_GROUPS * V_SLICE_FLOATS;
constexpr int V_RED_PITCH = 36;

template <bool AKF, bool BKF>
__global__ void __launch_bounds__(V_THREADS) gemm_ksplit_kernel(GemmArgs p) {
  extern __shared__ __align__(16) float fsm[];
  const int tid = threadIdx.x, grp = tid >> 6, t = tid & 63, tx = t & 7, ty = t >> 3;
  const int m0 = blockIdx.y * V_TM, n0 = blockIdx.x * V_TN;
  const int kb = p.kchunk ? blockIdx.z * p.kchunk : 0;
  const int ke = p.kchunk ? min(p.K, kb + p.kchunk) : p.K;
  const int nss = (ke - kb + V_GROUPS * V_TK - 1) / (V_GROUPS * V_TK);
  const int64_t lda = AKF ? p.sAm : p.sAk, ldb = BKF ? p.sBn : p.sBk;

  auto load_super = [&](int ss) {                  // 4 slices x (32 x 8 chunks) per operand = 1024 chunks each
    float* base = fsm + (ss % V_BUFS) * V_SUPER_FLOATS;
#pragma unroll
    for (int c = tid; c < V_GROUPS * 32 * 8; c += V_THREADS) {
      const int sl = c >> 8, r = (c >> 3) & 31, q = c & 7;
      const int k0 = kb + (ss * V_GROUPS + sl) * V_TK;
      float* As = base + sl * V_SLICE_FLOATS;
      float* Bs = As + 32 * V_PITCH;
      {
        const int m = m0 + (AKF ? r : 4 * q), k = k0 + (AKF ? 4 * q : r);
        const bool ok = m < p.M && k < ke;
        cp_async16(As + r * V_PITCH + 4 * q, p.A + (ok ? (AKF ? (int64_t)m * lda + k : (int64_t)k * lda + m) : 0), ok);
      }
      {
        const int n = n0 + (BKF ? r : 4 * q), k = k0 + (BKF ? 4 * q : r);
        const bool ok = n < p.N && k < ke;
        cp_async16(Bs + r * V_PITCH + 4 * q, p.B + (ok ? (BKF ? (int64_t)n * ldb + k : (int64_t)k * ldb + n) : 0), ok);
      }
    }
  };

  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  load_super(0);
  cp_async_commit();
  if (nss > 1) load_super(1);
  cp_async_commit();
  for (int ss = 0; ss < nss; ++ss) {
    cp_async_wait<1>();
    __syncthreads();
    const float* As = fsm + (ss % V_BUFS) * V_SUPER_FLOATS + grp * V_SLICE_FLOATS;
    const float* Bs = As + 32 * V_PITCH;
#pragma unroll
    for (int k4 = 0; k4 < V_TK; k4 += 4) {
      float a[4][4], b[4][4];                      // [k][i], [k][j]
      if (AKF) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float4 v = *reinterpret_cast<const float4*>(As + (ty + 8 * i) * V_PITCH + k4);
          a[0][i] = v.x; a[1][i] = v.y; a[2][i] = v.z; a[3][i] = v.w;
        }
      } else {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float4 v = *reinterpret_cast<const float4*>(As + (k4 + k) * V_PITCH + ty * 4);
          a[k][0] = v.x; a[k][1] = v.y; a[k][2] = v.z; a[k][3] = v.w;
        }
      }
      if (BKF) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float4 v = *reinterpret_cast<const float4*>(Bs + (tx + 8 * j) * V_PITCH + k4);
          b[0][j] = v.x; b[1][j] = v.y; b[2][j] = v.z; b[3][j] = v.w;
        }
      } else {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float4 v = *reinterpret_cast<const float4*>(Bs + (k4 + k) * V_PITCH + tx * 4);
          b[k][0] = v.x; b[k][1] = v.y; b[k][2] = v.z; b[k][3] = v.w;
        }
      }
#pragma unroll
      for (int k = 0; k < 4; ++k)
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[k][i], b[k][j], acc[i][j]);
    }
    __syncthreads();                               // every group is done with this buffer
    if (ss + V_BUFS < nss) load_super(ss + V_BUFS);
    cp_async_commit();
  }
  cp_async_wait<0>();
  __syncthreads();

  // the four groups' partial tiles meet in shared memory: red[grp][m][n]
  float* red = fsm;
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int ml = AKF ? ty + 8 * i : ty * 4 + i, nl = BKF ? tx + 8 * j : tx * 4 + j;
      red[(grp * V_TM + ml) * V_RED_PITCH + nl] = acc[i][j];
    }
  __syncthreads();
  {
    const int ml = tid >> 3, nl = (tid & 7) * 4;   // 256 threads x 4 consecutive columns
    float4 v = *reinterpret_cast<const float4*>(red + ml * V_RED_PITCH + nl);
#pragma unroll
    for (int g = 1; g < V_GROUPS; ++g) {
      const float4 w = *reinterpret_cast<const float4*>(red + (g * V_TM + ml) * V_RED_PITCH + nl);
      v.x += w.x; v.y += w.y; v.z += w.z; v.w += w.w;
    }
    const int m = m0 + ml;
    if (m < p.M) {
      const float o4[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int n = n0 + nl + e;
        if (n >= p.N) continue;
        float val = o4[e];
        const int64_t o = (int64_t)m * p.N + n;
        if (p.kchunk) { p.part[(size_t)blockIdx.z * p.M * p.N + o] = val; continue; }
        if (p.bias) val += __ldg(p.bias + n);
        if (p.pre) p.pre[o] = val;
        if (p.act == 1) val = gelu_exact(val);
        if (p.residual) val += __ldg(p.residual + o);
        if (p.accumulate) val += p.C[o];
        p.C[o] = val;
      }
    }
  }
  if (p.kchunk) splitk_finish(p, m0, n0, V_TM, V_TN);
}

static bool gemm_ksplit_eligible(const GemmArgs& p) {
  const bool akf = p.sAk == 1, bkf = p.sBk == 1;
  if (!akf && p.sAm != 1) return false;
  if (!bkf && p.sBn != 1) return false;
  const int64_t lda = akf ? p.sAm : p.sAk, ldb = bkf ? p.sBn : p.sBk;
  if ((lda & 3) || (ldb & 3) || ((uintptr_t)p.A & 15) || ((uintptr_t)p.B & 15)) return false;
  if ((akf || bkf) && (p.K & 3)) return false;       // 16-byte chunks along k
  if (!akf && (p.M & 3)) return false;               // ... along m
  if (!bkf && (p.N & 3)) return false;               // ... along n
  return true;
}

static int launch_gemm(GemmArgs& p, cudaStream_t st) {
  if (gemm_ksplit_eligible(p)) {
    dim3 grid(ceil_div(p.N, V_TN), ceil_div(p.M, V_TM), p.kchunk ? ceil_div(p.K, p.kchunk) : 1);
    const size_t smem = sizeof(float) * V_BUFS * V_SUPER_FLOATS;
    const bool akf = p.sAk == 1, bkf = p.sBk == 1;
#define TMF_LAUNCH_KS(AK, BK)                                                                                        \
  do {                                                                                                             \
    static bool attr_done = false;                                                                                 \
    if (!attr_done) {                                                                                              \
      TMF_CUDA(cudaFuncSetAttribute(gemm_ksplit_kernel<AK, BK>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
      attr_done = true;                                                                                            \
    }                                                                                                              \
    launch_k(gemm_ksplit_kernel<AK, BK>, grid, V_THREADS, smem, st, p);                                                   \
  } while (0)
    if (akf && bkf) TMF_LAUNCH_KS(true, true);
    else if (akf) TMF_LAUNCH_KS(true, false);
    else if (bkf) TMF_LAUNCH_KS(false, true);
    else TMF_LAUNCH_KS(false, false);
#undef TMF_LAUNCH_KS
    TMF_LAUNCH_CHECK();
    return 0;
  }
  dim3 grid(ceil_div(p.N, G_TN), ceil_div(p.M, G_TM), p.kchunk ? ceil_div(p.K, p.kchunk) : 1);
  launch_k(gemm_kernel, grid, 256, 0, st, p);
  TMF_LAUNCH_CHECK();
  return 0;
}

}  // namespace tmf

using namespace tmf;

extern "C" {

int tmf_linear_fwd(const float* x, const float* w, const float* bias, const float* residual, float* y, float* pre,
                   int M, int K, int N, int act, void* stream) {
  TMF_REQUIRE(x && w && y, "linear_fwd: NULL pointer");
  TMF_REQUIRE(act == 0 || act == 1, "linear_fwd: unknown activation %d", act);
  GemmArgs p{};
  p.A = x; p.B = w; p.C = y; p.bias = bias; p.residual = residual; p.pre = pre;
  p.M = M; p.N = N; p.K = K;
  p.sAm = K; p.sAk = 1; p.sBk = 1; p.sBn = K;
  p.act = act; p.accumulate = 0;
  return launch_gemm(p, (cudaStream_t)stream);
}

int tmf_linear_dgrad(const float* dy, const float* w, float* dx, int M, int K, int N, int accumulate, void* stream) {
  TMF_REQUIRE(dy && w && dx, "linear_dgrad: NULL pointer");
  GemmArgs p{};
  p.A = dy; p.B = w; p.C = dx;
  p.M = M; p.N = K; p.K = N;          // dx[M,K] = dy[M,N] . w[N,K]
  p.sAm = N; p.sAk = 1; p.sBk = K; p.sBn = 1;
  p.accumulate = accumulate;
  return launch_gemm(p, (cudaStream_t)stream);
}

static int check_ws(const char* who, void* ws, size_t ws_bytes) {
  TMF_REQUIRE(ws != nullptr && ws_bytes >= TMF_WS_BYTES && ((uintptr_t)ws & 255) == 0,
              "%s: needs the 256-byte aligned scratch buffer of tmf_scratch_bytes() bytes (tickets zero-initialised)", who);
  return 0;
}

int tmf_linear_wgrad(const float* dy, const float* x, float* dw, float* dbias, int M, int K, int N, void* ws,
                     size_t ws_bytes, void* stream) {
  TMF_REQUIRE(dy && x && dw, "linear_wgrad: NULL pointer");
  if (check_ws("linear_wgrad", ws, ws_bytes)) return 1;
  unsigned* tickets = reinterpret_cast<unsigned*>(ws);
  float* partials = reinterpret_cast<float*>(reinterpret_cast<char*>(ws) + TMF_WS_TICKET_BYTES);
  const size_t part_floats = (TMF_WS_BYTES - TMF_WS_TICKET_BYTES) / sizeof(float);
  GemmArgs p{};
  p.A = dy; p.B = x; p.C = dw;
  p.M = N; p.N = K; p.K = M;          // dw[N,K] = dy^T[N,M] . x[M,K]
  p.sAm = 1; p.sAk = N; p.sBk = K; p.sBn = 1;
  cudaStream_t st = (cudaStream_t)stream;
  if (M > 2 * G_SPLIT_K) {             // long reduction over the tokens: split it, partial sums meet in a zeroed dw
    p.kchunk = G_SPLIT_K;
    if (gemm_ksplit_eligible(p)) {     // enough K slices to put ~two CTAs on every SM, in whole super-slices (4 x 32 tokens)
      const int tiles = ceil_div(N, V_TM) * ceil_div(K, V_TN), ss = V_GROUPS * V_TK;
      int splits = ceil_div(2 * 148, tiles);
      if (splits > ceil_div(M, ss)) splits = ceil_div(M, ss);
      p.kchunk = ceil_div(ceil_div(M, splits), ss) * ss;
    }
    // split-K partial tiles meet in the scratch buffer; the last split of a tile adds them in order (deterministic)
    const int splits = ceil_div(M, p.kchunk);
    const int tiles = gemm_ksplit_eligible(p) ? ceil_div(N, V_TM) * ceil_div(K, V_TN) : ceil_div(N, G_TM) * ceil_div(K, G_TN);
    if (tiles > 2048 || (size_t)splits * N * K > part_floats) {
      p.kchunk = 0;                      // too large for the scratch buffer: one CTA per tile walks the whole reduction
    } else {
      p.part = partials;
      p.tickets = tickets + 1024;
    }
  }
  if (launch_gemm(p, st)) return 3;
  if (dbias) {
    int rows = 128;
    while ((size_t)ceil_div(M, rows) * N > part_floats) rows *= 2;
    dim3 grid(ceil_div(N, 32), ceil_div(M, rows), 1);
    TMF_REQUIRE(grid.x <= 1024, "linear_wgrad: N=%d too wide for the column-sum tickets", N);
    // (runs after the GEMM in stream order, so it may reuse the partial area)
    launch_k(colsum_kernel, grid, 256, 0, st, dy, dbias, M, N, rows, partials, tickets + 3072);
    TMF_LAUNCH_CHECK();
  }
  return 0;
}

int64_t tmf_scratch_bytes(void) { return (int64_t)TMF_WS_BYTES; }

int tmf_layernorm_fwd(const float* x, const float* gamma, const float* beta, const float* residual, float* y,
                      float* mean, float* rstd, int rows, int dim, float eps, void* stream) {
  TMF_REQUIRE(dim % 4 == 0 && dim <= 128 * LN_MAXV, "layernorm: dim must be a multiple of 4 and <= %d (got %d)",
              128 * LN_MAXV, dim);
  const int grid = max(1, min(ceil_div(rows, 8), 148 * 8));
  launch_k(layernorm_fwd_kernel, grid, 256, 0, (cudaStream_t)stream, x, gamma, beta, residual, y, mean, rstd, rows, dim, eps);
  TMF_LAUNCH_CHECK();
  return 0;
}

int tmf_layernorm_bwd(const float* dy, const float* x, const float* gamma, const float* mean, const float* rstd,
                      float* dx, float* dgamma, float* dbeta, int rows, int dim, int accumulate, void* ws,
                      size_t ws_bytes, void* stream) {
  TMF_REQUIRE(dim % 4 == 0 && dim <= 128 * LN_MAXV, "layernorm: dim must be a multiple of 4 and <= %d (got %d)",
              128 * LN_MAXV, dim);
  if (check_ws("layernorm_bwd", ws, ws_bytes)) return 1;
  const int grid = max(1, min(ceil_div(rows, 8 * 4), 148));
  launch_k(layernorm_bwd_kernel, grid, 256, 2 * dim * sizeof(float), (cudaStream_t)stream, 
      dy, x, gamma, mean, rstd, dx, dgamma, dbeta, rows, dim, accumulate,
      reinterpret_cast<float*>(reinterpret_cast<char*>(ws) + TMF_WS_TICKET_BYTES), reinterpret_cast<unsigned*>(ws));
  TMF_LAUNCH_CHECK();
  return 0;
}

int tmf_gelu_bwd(const float* dy, const float* pre, float* dx, int64_t n, void* stream) {
  TMF_REQUIRE(n % 4 == 0, "gelu_bwd: n must be a multiple of 4");
  const int grid = max(1, min(ceil_div(n / 4, 256), 148 * 8));
  launch_k(gelu_bwd_kernel, grid, 256, 0, (cudaStream_t)stream, (const float4*)dy, (const float4*)pre, (float4*)dx, n / 4);
  TMF_LAUNCH_CHECK();
  return 0;
}

int tmf_scale(const float* x, float* y, float alpha, const float* alpha_dev, int64_t n, void* stream) {
  const int grid = max(1, min(ceil_div(n, 256), 148 * 8));
  launch_k(scale_kernel, grid, 256, 0, (cudaStream_t)stream, x, y, alpha, alpha_dev, n);
  TMF_LAUNCH_CHECK();
  return 0;
}

static int attn_smem_check(size_t bytes, const void* fn) {
  TMF_REQUIRE(bytes <= 227 * 1024, "attention: sequence too long for the shared-memory resident kernel (%zu B)", bytes);
  if (bytes > 48 * 1024) TMF_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  return 0;
}

int tmf_attn_fwd(const float* q, const float* kv, float* out, float* lse, int B, int Nq, int Nk, int heads, int dh,
                 float scale, void* stream) {
  AttnArgs p{};
  p.q = q; p.kv = kv; p.o = out; p.lse = lse;
  p.B = B; p.Nq = Nq; p.Nk = Nk; p.heads = heads; p.dh = dh; p.scale = scale;
  {
    const int rc = attn_mma_fwd(p, (cudaStream_t)stream);        // tensor-core kernels (attention_mma.cu): the fusion stack's shapes
    if (rc >= 0) return rc;
  }
  {
    const int rc = attn_tiled_fwd(p, (cudaStream_t)stream);      // register-tiled kernels (attention.cu) when the shape fits
    if (rc >= 0) return rc;
  }
  const size_t smem = sizeof(float) * ((size_t)2 * Nk * (dh + 1) + (size_t)AT_WARPS * Nk + (size_t)AT_WARPS * dh);
  if (attn_smem_check(smem, (const void*)attn_fwd_kernel)) return 2;
  dim3 grid(B * heads, ceil_div(Nq, AT_ROWS), 1);
  launch_k(attn_fwd_kernel, grid, AT_WARPS * 32, smem, (cudaStream_t)stream, p);
  TMF_LAUNCH_CHECK();
  return 0;
}

int tmf_attn_bwd(const float* dout, const float* q, const float* kv, const float* out, const float* lse, float* dq,
                 float* dkv, int B, int Nq, int Nk, int heads, int dh, float scale, void* stream) {
  AttnArgs p{};
  p.q = q; p.kv = kv; p.out = out; p.lse_in = lse; p.dout = dout; p.dq = dq; p.dkv = dkv;
  p.B = B; p.Nq = Nq; p.Nk = Nk; p.heads = heads; p.dh = dh; p.scale = scale;
  {
    const int rc = attn_mma_bwd(p, (cudaStream_t)stream);
    if (rc >= 0) return rc;
  }
  {
    const int rc = attn_tiled_bwd(p, (cudaStream_t)stream);
    if (rc >= 0) return rc;
  }
  const size_t smem1 =
      sizeof(float) * ((size_t)2 * Nk * (dh + 1) + (size_t)AT_WARPS * Nk + (size_t)2 * AT_WARPS * dh);
  if (attn_smem_check(smem1, (const void*)attn_bwd_dq_kernel)) return 2;
  dim3 grid1(B * heads, ceil_div(Nq, AT_ROWS), 1);
  launch_k(attn_bwd_dq_kernel, grid1, AT_WARPS * 32, smem1, (cudaStream_t)stream, p);
  TMF_LAUNCH_CHECK();
  const size_t smem2 = sizeof(float) * ((size_t)2 * Nq * (dh + 1) + (size_t)2 * Nq + (size_t)2 * AT_WARPS * Nq +
                                        (size_t)2 * AT_WARPS * dh);
  if (attn_smem_check(smem2, (const void*)attn_bwd_dkv_kernel)) return 2;
  dim3 grid2(B * heads, ceil_div(Nk, AT_ROWS), 1);
  launch_k(attn_bwd_dkv_kernel, grid2, AT_WARPS * 32, smem2, (cudaStream_t)stream, p);
  TMF_LAUNCH_CHECK();
  return 0;
}

int tmf_token_pool_fwd(const float* x, float* mean, float* max, int32_t* argmax, int B, int N, int C, void* stream) {
  TMF_REQUIRE(max == nullptr || argmax != nullptr, "token_pool_fwd: argmax buffer required with max");
  launch_k(token_pool_fwd_kernel, B * ceil_div(C, 32), 32 * TP_WARPS, 0, (cudaStream_t)stream, x, mean, max, argmax, B, N, C);
  TMF_LAUNCH_CHECK();
  return 0;
}

int tmf_token_pool_bwd(const float* dmean, const float* dmax, const int32_t* argmax, float* dx, int B, int N, int C,
                       int accumulate, void* stream) {
  const int64_t total = (int64_t)B * N * C;
  const int grid = max(1, min(ceil_div(total, 256), 148 * 8));
  launch_k(token_pool_bwd_kernel, grid, 256, 0, (cudaStream_t)stream, dmean, dmax, argmax, dx, B, N, C, accumulate);
  TMF_LAUNCH_CHECK();
  return 0;
}

}  // extern "C"

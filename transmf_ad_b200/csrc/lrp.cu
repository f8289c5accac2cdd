// lrp.cu -- layer-wise relevance propagation through the sNet towers (Bach et al., 2015; Montavon et al., 2019; DESIGN
// section 3.9).  Per conv unit l = Conv3d + BatchNorm3d(eval, folded) + LeakyReLU (+ pool), from the tower output down:
//
//   R_out      relevance at the unit's (pooled) output: the seed a_T * df/da_T at layer 6, else a_{l+1} * c_{l+1}
//   R_y        R_out routed through the pool to the conv output: max-pool -> the first maximum of y in (d,h,w) scan order
//              of its window; avg-pool -> in proportion to a = LeakyReLU(y) over the window; LeakyReLU passes it unchanged
//   s          R_y / stab(z),  z = y (rule epsilon, bias included) or z+ = conv(a, w+) (rule zplus, no bias),
//              stab(z) = z + eps * sign(z) with sign(0) = +1; s = 0 where stab(z) == 0
//   c_l        W^T s (the dgrad launch, with the rule's folded weight), and R_in = a_l * c_l
//
// This file: the BatchNorm fold of the rule's weights (tmf_lrp_fold_pack), the memory-bound ratio pass (tmf_lrp_ratio: R_out
// -> s, never writing R_out), the per-sample relevance totals (per-CTA partial rows summed in index order: no atomics) and
// the per-sample normalisation of the maps.  Block 1 (s on chip, c = W^T s, R_x = x * c) is tmf_lrp_conv1 in conv1_dgrad.cu.
#include <algorithm>

#include "common.cuh"

namespace tmf {

constexpr int LRP_THREADS = 256;
constexpr int LRP_MAX_BLOCKS = 1024;           // CTAs per (sample, tower) of the ratio / x-multiply passes

__global__ void lrp_fold_pack_kernel(GroupPtr<const float> w, GroupPtr<const float> cbias, GroupPtr<const float> gamma,
                                     GroupPtr<const float> beta, GroupPtr<const float> rmean, GroupPtr<const float> rvar,
                                     GroupPtr<__nv_bfloat16> wf, GroupPtr<__nv_bfloat16> wd, GroupPtr<float> w32,
                                     GroupPtr<float> bias_out, int cout, int cin, int taps, float eps, int zplus) {
  const int g = blockIdx.z;
  const int64_t total = (int64_t)cout * cin * taps;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int t = (int)(idx % taps);
    const int ci = (int)((idx / taps) % cin);
    const int co = (int)(idx / ((int64_t)taps * cin));
    const float scale = gamma.p[g][co] * rsqrtf(rvar.p[g][co] + eps);      // the arithmetic of fold_bn_pack_kernel
    float v = w.p[g][idx] * scale;
    if (zplus) v = fmaxf(v, 0.f);
    const __nv_bfloat16 vb = __float2bfloat16_rn(v);
    if (wf.p[g] != nullptr) wf.p[g][((int64_t)t * cout + co) * cin + ci] = vb;
    if (wd.p[g] != nullptr) wd.p[g][((int64_t)(taps - 1 - t) * cin + ci) * cout + co] = vb;
    if (w32.p[g] != nullptr) w32.p[g][idx] = v;
    if (t == 0 && ci == 0) {
      const float b = cbias.p[g] != nullptr ? cbias.p[g][co] : 0.f;
      bias_out.p[g][co] = (b - rmean.p[g][co]) * scale + beta.p[g][co];
    }
  }
}

struct LrpRatioParams {
  const void* ua[TMF_MAX_GROUPS];              // upstream relevance = ua * uc, pooled NDHWC [B][Do][Ho][Wo][C]
  const void* uc[TMF_MAX_GROUPS];
  const __nv_bfloat16* y[TMF_MAX_GROUPS];      // stored folded pre-activation, [B][D][H][W][C]
  const __nv_bfloat16* zp[TMF_MAX_GROUPS];     // z+ (rule zplus) or NULL
  __nv_bfloat16* s[TMF_MAX_GROUPS];
  float* part[TMF_MAX_GROUPS];                 // [B][nblk] partial sums of the upstream relevance
  int D, H, W, C, CG, Do, Ho, Wo, Dc, Hc, Wc, nblk, pool, up_fp32;
  int64_t cells;                               // per sample: Dc * Hc * Wc * CG (a cell: one pool window x 8 channels)
  float slope, eps;
};

__device__ __forceinline__ void lrp_load8(const void* base, int64_t off, int fp32, float* f) {
  if (fp32) {
    const float4* p = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(base) + off);
    const float4 a = __ldg(p), b = __ldg(p + 1);
    f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w; f[4] = b.x; f[5] = b.y; f[6] = b.z; f[7] = b.w;
  } else {
    unpack8(__ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(base) + off)), f);
  }
}

// Block-wide sum of one value per thread in a fixed tree order.
__device__ __forceinline__ float lrp_block_sum(float v, float* red) {
  red[threadIdx.x] = v;
  __syncthreads();
  for (int o = blockDim.x / 2; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  return red[0];
}

// One thread per cell (pool window, 8 channels).  Voxels outside every complete window (odd extents) get s = 0.
__global__ void __launch_bounds__(LRP_THREADS) lrp_ratio_kernel(const __grid_constant__ LrpRatioParams p) {
  __shared__ float red[LRP_THREADS];
  const int g = blockIdx.z, n = blockIdx.y;
  const int win = p.pool == TMF_POOL_NONE ? 1 : 2;
  float tsum = 0.f;
  for (int64_t i = (int64_t)blockIdx.x * LRP_THREADS + threadIdx.x; i < p.cells; i += (int64_t)p.nblk * LRP_THREADS) {
    const int cg = (int)(i % p.CG);
    int64_t t = i / p.CG;
    const int cw = (int)(t % p.Wc); t /= p.Wc;
    const int ch = (int)(t % p.Hc);
    const int cd = (int)(t / p.Hc);
    const int c0 = cg * 8;
    const bool win_ok = cd < p.Do && ch < p.Ho && cw < p.Wo;
    float R[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) R[c] = 0.f;
    if (win_ok) {
      const int64_t uo = ((((int64_t)n * p.Do + cd) * p.Ho + ch) * p.Wo + cw) * p.C + c0;
      float a[8], cc[8];
      lrp_load8(p.ua[g], uo, p.up_fp32, a);
      lrp_load8(p.uc[g], uo, p.up_fp32, cc);
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        R[c] = __fmul_rn(a[c], cc[c]);
        tsum = __fadd_rn(tsum, R[c]);
      }
    }
    const __nv_bfloat16* yg = p.y[g];
    const __nv_bfloat16* zg = p.zp[g];
    __nv_bfloat16* sg = p.s[g];
    const int d0 = cd * win, h0 = ch * win, w0 = cw * win;
    int64_t off[8];
    bool ex[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const int d = d0 + ((q >> 2) & 1), h = h0 + ((q >> 1) & 1), w = w0 + (q & 1);
      ex[q] = (win == 2 || q == 0) && d < p.D && h < p.H && w < p.W;
      off[q] = ((((int64_t)n * p.D + d) * p.H + h) * p.W + w) * p.C + c0;
    }
    if (!win_ok) {
#pragma unroll
      for (int q = 0; q < 8; ++q)
        if (ex[q]) *reinterpret_cast<uint4*>(sg + off[q]) = make_uint4(0u, 0u, 0u, 0u);
      continue;
    }
    if (p.pool == TMF_POOL_NONE) {
      float yv[8], o[8];
      lrp_load8(zg != nullptr ? (const void*)zg : (const void*)yg, off[0], 0, yv);
#pragma unroll
      for (int c = 0; c < 8; ++c) o[c] = lrp_div(R[c], yv[c], p.eps);
      *reinterpret_cast<uint4*>(sg + off[0]) = pack8(o);
    } else if (p.pool == TMF_POOL_MAX) {
      float yv[8][8];
#pragma unroll
      for (int q = 0; q < 8; ++q) lrp_load8(yg, off[q], 0, yv[q]);
      int wq[8];
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        float m = yv[0][c];
        wq[c] = 0;
#pragma unroll
        for (int q = 1; q < 8; ++q)
          if (yv[q][c] > m) { m = yv[q][c]; wq[c] = q; }
      }
      float sv[8];
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        float z = 0.f;
#pragma unroll
        for (int q = 0; q < 8; ++q) z = wq[c] == q ? yv[q][c] : z;
        if (zg != nullptr) {
          const int q = wq[c];
          int64_t o = off[0];
#pragma unroll
          for (int qq = 1; qq < 8; ++qq) o = q == qq ? off[qq] : o;
          z = __bfloat162float(zg[o + c]);
        }
        sv[c] = lrp_div(R[c], z, p.eps);
      }
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        float o[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) o[c] = wq[c] == q ? sv[c] : 0.f;
        *reinterpret_cast<uint4*>(sg + off[q]) = pack8(o);
      }
    } else {
      float av[8][8], S[8];
#pragma unroll
      for (int c = 0; c < 8; ++c) S[c] = 0.f;
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        lrp_load8(yg, off[q], 0, av[q]);
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          const float z = av[q][c];
          av[q][c] = z > 0.f ? z : __fmul_rn(z, p.slope);     // LeakyReLU, as the forward pass computes it
          S[c] = __fadd_rn(S[c], av[q][c]);
        }
      }
#pragma unroll
      for (int c = 0; c < 8; ++c) S[c] = lrp_div(R[c], S[c], p.eps);   // R per unit of activation in the window
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        float z[8], o[8];
        lrp_load8(zg != nullptr ? (const void*)zg : (const void*)yg, off[q], 0, z);
#pragma unroll
        for (int c = 0; c < 8; ++c) o[c] = lrp_div(__fmul_rn(av[q][c], S[c]), z[c], p.eps);
        *reinterpret_cast<uint4*>(sg + off[q]) = pack8(o);
      }
    }
  }
  const float tot = lrp_block_sum(tsum, red);
  if (threadIdx.x == 0) p.part[g][(int64_t)n * p.nblk + blockIdx.x] = tot;
}

// out = x * c (in place on c), plus per-CTA partial sums of out: the relevance map of block 1's CUDA-core path.
__global__ void __launch_bounds__(LRP_THREADS) lrp_xmul_kernel(GroupPtr<const float> x, GroupPtr<float> c, GroupPtr<float> part,
                                                               int64_t per, int nblk) {
  __shared__ float red[LRP_THREADS];
  const int g = blockIdx.z, n = blockIdx.y;
  const float* xs = x.p[g] + (int64_t)n * per;
  float* cs = c.p[g] + (int64_t)n * per;
  float tsum = 0.f;
  for (int64_t i = (int64_t)blockIdx.x * LRP_THREADS + threadIdx.x; i < per; i += (int64_t)nblk * LRP_THREADS) {
    const float v = __fmul_rn(xs[i], cs[i]);
    cs[i] = v;
    tsum = __fadd_rn(tsum, v);
  }
  const float tot = lrp_block_sum(tsum, red);
  if (threadIdx.x == 0) part.p[g][(int64_t)n * nblk + blockIdx.x] = tot;
}

// totals[g][n][col + k] = sum over r (in index order, fp64) of part[g][n][r][k]
__global__ void lrp_sum_rows_kernel(GroupPtr<const float> part, GroupPtr<float> totals, int B, int rows, int K, int col) {
  const int g = blockIdx.z;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * K) return;
  const int n = i / K, k = i % K;
  const float* pr = part.p[g] + (int64_t)n * rows * K + k;
  double acc = 0.0;
  for (int r = 0; r < rows; ++r) acc += (double)pr[(int64_t)r * K];
  totals.p[g][n * 8 + col + k] = (float)acc;
}

__global__ void __launch_bounds__(1024) lrp_normalize_kernel(GroupPtr<float> map, int64_t per) {
  __shared__ float red[32];
  const int g = blockIdx.z, n = blockIdx.y;
  float* m = map.p[g] + (int64_t)n * per;
  float mx = 0.f;
  for (int64_t i = threadIdx.x; i < per; i += blockDim.x) mx = fmaxf(mx, fabsf(m[i]));
  mx = warp_max(mx);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = mx;
  __syncthreads();
  if (threadIdx.x < 32) {
    mx = warp_max(threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.f);
    if (threadIdx.x == 0) red[0] = mx;
  }
  __syncthreads();
  mx = red[0];
  if (mx > 0.f)
    for (int64_t i = threadIdx.x; i < per; i += blockDim.x) m[i] = __fdiv_rn(m[i], mx);
}

int lrp_blocks(int64_t items) { return (int)std::min<int64_t>((items + LRP_THREADS - 1) / LRP_THREADS, LRP_MAX_BLOCKS); }

static size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }

size_t lrp_ratio_ws(int ng, int B, int D, int H, int W, int C, int pool) {
  const int win = pool == TMF_POOL_NONE ? 1 : 2;
  const int64_t cells = (int64_t)((D + win - 1) / win) * ((H + win - 1) / win) * ((W + win - 1) / win) * (C / 8);
  return align256((size_t)ng * B * lrp_blocks(cells) * sizeof(float));
}

int lrp_sum_rows(int ng, float* const* part, float* const* totals, int B, int rows, int K, int col, cudaStream_t st) {
  GroupPtr<const float> gp;
  GroupPtr<float> gt;
  if (!load_group(gp, (const float* const*)part, ng, true, "part") || !load_group(gt, totals, ng, true, "totals")) return 1;
  launch_k(lrp_sum_rows_kernel, dim3((unsigned)ceil_div((int64_t)B * K, 128), 1, ng), 128, 0, st, gp, gt, B, rows, K, col);
  TMF_LAUNCH_CHECK();
  return 0;
}

// rx[g] <- x[g] * rx[g] with totals column `col`; part: ng * B * lrp_blocks(D*H*W) floats of scratch
int lrp_xmul(int ng, const float* const* x, float* const* rx, float* const* totals, int col, int B, int64_t per, float* part,
             cudaStream_t st) {
  const int nblk = lrp_blocks(per);
  GroupPtr<const float> gx;
  GroupPtr<float> gc, gp;
  if (!load_group(gx, x, ng, true, "x") || !load_group(gc, rx, ng, true, "rx")) return 1;
  float* pp[TMF_MAX_GROUPS] = {nullptr, nullptr};
  for (int g = 0; g < ng; ++g) pp[g] = part + (size_t)g * B * nblk;
  load_group(gp, (float* const*)pp, ng, true, "part");
  launch_k(lrp_xmul_kernel, dim3((unsigned)nblk, (unsigned)B, (unsigned)ng), LRP_THREADS, 0, st, gx, gc, gp, per, nblk);
  TMF_LAUNCH_CHECK();
  return lrp_sum_rows(ng, pp, totals, B, nblk, 1, col, st);
}

}  // namespace tmf

using namespace tmf;

extern "C" {

int tmf_lrp_fold_pack(int ng, const float* const* w, const float* const* conv_bias, const float* const* gamma,
                      const float* const* beta, const float* const* running_mean, const float* const* running_var,
                      void* const* wf, void* const* wd, float* const* w32, float* const* bias_out, int cout, int cin,
                      int ksize, float eps, int rule, void* stream) {
  TMF_CHECK_NG(ng);
  TMF_REQUIRE(ksize == 1 || ksize == 3, "lrp_fold_pack: kernel size must be 1 or 3");
  TMF_REQUIRE(rule == TMF_LRP_EPSILON || rule == TMF_LRP_ZPLUS, "lrp_fold_pack: unknown rule %d", rule);
  GroupPtr<const float> gw, gcb, gg, gb, gm, gv;
  GroupPtr<__nv_bfloat16> gwf, gwd;
  GroupPtr<float> gw32, gbo;
  if (!load_group(gw, w, ng, true, "w") || !load_group(gcb, conv_bias, ng, false, "conv_bias") ||
      !load_group(gg, gamma, ng, true, "gamma") || !load_group(gb, beta, ng, true, "beta") ||
      !load_group(gm, running_mean, ng, true, "running_mean") || !load_group(gv, running_var, ng, true, "running_var") ||
      !load_group(gwf, (__nv_bfloat16* const*)wf, ng, false, "wf") || !load_group(gwd, (__nv_bfloat16* const*)wd, ng, false, "wd") ||
      !load_group(gw32, w32, ng, false, "w32") || !load_group(gbo, bias_out, ng, true, "bias_out"))
    return 1;
  const int taps = ksize * ksize * ksize;
  const int64_t total = (int64_t)cout * cin * taps;
  dim3 grid((unsigned)(ceil_div(total, 256) < 592 ? ceil_div(total, 256) : 592), 1, ng);
  launch_k(lrp_fold_pack_kernel, grid, 256, 0, (cudaStream_t)stream, gw, gcb, gg, gb, gm, gv, gwf, gwd, gw32, gbo, cout, cin,
           taps, eps, (int)(rule == TMF_LRP_ZPLUS));
  TMF_LAUNCH_CHECK();
  return 0;
}

int64_t tmf_lrp_ratio_workspace_bytes(int ng, int B, int D, int H, int W, int C, int pool) {
  return (int64_t)lrp_ratio_ws(ng, B, D, H, W, C, pool);
}

int tmf_lrp_ratio(int ng, const void* const* up_a, const void* const* up_c, int up_fp32, const void* const* y,
                  const void* const* zp, void* const* s, float* const* totals, int col, int B, int D, int H, int W, int C,
                  int pool, float slope, float eps, void* ws, size_t ws_bytes, void* stream) {
  TMF_CHECK_NG(ng);
  TMF_REQUIRE(B >= 1 && B <= 65535 && D >= 1 && H >= 1 && W >= 1, "lrp_ratio: bad problem (%d,%d,%d,%d)", B, D, H, W);
  TMF_REQUIRE(C >= 8 && C % 8 == 0, "lrp_ratio: C must be a positive multiple of 8 (got %d)", C);
  TMF_REQUIRE(pool == TMF_POOL_NONE || pool == TMF_POOL_MAX || pool == TMF_POOL_AVG, "lrp_ratio: bad pool mode %d", pool);
  TMF_REQUIRE(col >= 0 && col < 8, "lrp_ratio: totals column %d out of range", col);
  TMF_REQUIRE(eps >= 0.f, "lrp_ratio: eps must be >= 0");
  const size_t need = lrp_ratio_ws(ng, B, D, H, W, C, pool);
  TMF_REQUIRE(ws != nullptr && ws_bytes >= need && ((uintptr_t)ws & 255) == 0,
              "lrp_ratio: needs a 256-byte aligned workspace of %zu bytes (got %zu)", need, ws_bytes);
  LrpRatioParams p{};
  const int win = pool == TMF_POOL_NONE ? 1 : 2;
  p.D = D; p.H = H; p.W = W; p.C = C; p.CG = C / 8;
  p.Do = D / win; p.Ho = H / win; p.Wo = W / win;
  p.Dc = (D + win - 1) / win; p.Hc = (H + win - 1) / win; p.Wc = (W + win - 1) / win;
  p.cells = (int64_t)p.Dc * p.Hc * p.Wc * p.CG;
  p.nblk = lrp_blocks(p.cells);
  p.pool = pool; p.up_fp32 = up_fp32 != 0; p.slope = slope; p.eps = eps;
  for (int g = 0; g < ng; ++g) {
    TMF_REQUIRE(up_a && up_c && y && s && totals && up_a[g] && up_c[g] && y[g] && s[g] && totals[g],
                "lrp_ratio: NULL device pointer");
    TMF_REQUIRE((((uintptr_t)up_a[g] | (uintptr_t)up_c[g] | (uintptr_t)y[g] | (uintptr_t)s[g]) & 15) == 0,
                "lrp_ratio: tensors must be 16-byte aligned");
    p.ua[g] = up_a[g]; p.uc[g] = up_c[g];
    p.y[g] = (const __nv_bfloat16*)y[g];
    p.zp[g] = zp != nullptr ? (const __nv_bfloat16*)zp[g] : nullptr;
    p.s[g] = (__nv_bfloat16*)s[g];
    p.part[g] = (float*)ws + (size_t)g * B * p.nblk;
  }
  cudaStream_t st = (cudaStream_t)stream;
  launch_k(lrp_ratio_kernel, dim3((unsigned)p.nblk, (unsigned)B, (unsigned)ng), LRP_THREADS, 0, st, p);
  TMF_LAUNCH_CHECK();
  return lrp_sum_rows(ng, p.part, totals, B, p.nblk, 1, col, st);
}

int tmf_lrp_normalize(int ng, float* const* map, int B, int64_t per, void* stream) {
  TMF_CHECK_NG(ng);
  TMF_REQUIRE(B >= 1 && B <= 65535 && per >= 1, "lrp_normalize: bad problem");
  GroupPtr<float> gm;
  if (!load_group(gm, map, ng, true, "map")) return 1;
  launch_k(lrp_normalize_kernel, dim3(1, (unsigned)B, (unsigned)ng), 1024, 0, (cudaStream_t)stream, gm, per);
  TMF_LAUNCH_CHECK();
  return 0;
}

}  // extern "C"

// ig.cu -- integrated gradients (Sundararajan et al., 2017) through the sNet towers with block 1 factored out of the path
// integral (DESIGN section 3.10).  Zero baseline, path points alpha_k > 0, block 1 in eval mode with BatchNorm folded into
// conv1.0 (weight W', bias b'), u' = W' * x (no bias), umax = u' at the first maximum of each 2x2x2 window:
//
//   a1_k     = LeakyReLU(alpha_k * umax + b')          the block-1 output at alpha_k x (the winners do not move with alpha)
//   G       += w_k * g_k * LeakyReLU'(alpha_k * umax + b')      g_k = df/da1 at path point k
//   IG       = x * W'^T route(G)                        one tmf_conv1_dgrad_fused for the whole path (identity coefficients)
//
// This file: the per-chunk expansion of umax into the next conv's operands (tmf_ig_expand), the accumulation of the chunk's
// gradients into G (tmf_ig_combine) and the final x-multiply with per-sample sums (tmf_ig_attribute).  All memory-bound,
// CUDA cores, no atomics.  z_k is fmaf(alpha_k, umax, b') in both kernels, so they agree on the LeakyReLU branch bit for bit.
#include "common.cuh"

namespace tmf {

constexpr int IG_THREADS = 256;
constexpr int IG_MAX_BLOCKS = 2048;            // CTAs per tower; each thread walks 8-element vectors with a grid stride

int lrp_blocks(int64_t items);
int lrp_xmul(int ng, const float* const* x, float* const* rx, float* const* totals, int col, int B, int64_t per, float* part,
             cudaStream_t st);

struct IgArgs {
  const __nv_bfloat16* umax[TMF_MAX_GROUPS];   // [B][Do][Ho][Wo][C]
  const float* bias[TMF_MAX_GROUPS];           // [C] folded conv1.0 bias b'
  __nv_bfloat16* a1[TMF_MAX_GROUPS];           // expand: [n][B][Do][Ho][Wo][C] step-major
  float* a32[TMF_MAX_GROUPS];                  // expand: the fp32 twin of a1 (same layout)
  const float* grad[TMF_MAX_GROUPS];           // combine: [n][B][Do][Ho][Wo][C] step-major
  float* G[TMF_MAX_GROUPS];                    // combine: [B][Do][Ho][Wo][C], updated in place
  const float* alpha;                          // [n]
  const float* w;                              // [n] (combine)
  int64_t nvec;                                // 8-element vectors per tower and step: B*Do*Ho*Wo*C / 8
  int C, n;
  float slope;
};

__device__ __forceinline__ void ig_bias8(const float* bias, int c0, float* b) {
  const float4 lo = __ldg(reinterpret_cast<const float4*>(bias + c0)), hi = __ldg(reinterpret_cast<const float4*>(bias + c0) + 1);
  b[0] = lo.x; b[1] = lo.y; b[2] = lo.z; b[3] = lo.w; b[4] = hi.x; b[5] = hi.y; b[6] = hi.z; b[7] = hi.w;
}

// One thread per 8-channel vector of umax, all n steps: umax is read once per chunk.
__global__ void __launch_bounds__(IG_THREADS) ig_expand_kernel(const __grid_constant__ IgArgs p) {
  const int g = blockIdx.z;
  for (int64_t v = (int64_t)blockIdx.x * IG_THREADS + threadIdx.x; v < p.nvec; v += (int64_t)gridDim.x * IG_THREADS) {
    float u[8], b[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(p.umax[g]) + v), u);
    ig_bias8(p.bias[g], (int)((v * 8) % p.C), b);
    for (int k = 0; k < p.n; ++k) {
      const float a = __ldg(p.alpha + k);
      float o[8];
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const float z = fmaf(a, u[c], b[c]);
        o[c] = z > 0.f ? z : z * p.slope;                  // LeakyReLU as bn_act_pool_fwd_kernel computes it
      }
      const int64_t at = (int64_t)k * p.nvec + v;
      reinterpret_cast<uint4*>(p.a1[g])[at] = pack8(o);
      float4* d = reinterpret_cast<float4*>(p.a32[g]) + 2 * at;
      d[0] = make_float4(o[0], o[1], o[2], o[3]);
      d[1] = make_float4(o[4], o[5], o[6], o[7]);
    }
  }
}

// G += w_k * g_k * LeakyReLU'(z_k), k in order onto the loaded G: the same operations whatever the chunking.
__global__ void __launch_bounds__(IG_THREADS) ig_combine_kernel(const __grid_constant__ IgArgs p) {
  const int g = blockIdx.z;
  for (int64_t v = (int64_t)blockIdx.x * IG_THREADS + threadIdx.x; v < p.nvec; v += (int64_t)gridDim.x * IG_THREADS) {
    float u[8], b[8], acc[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(p.umax[g]) + v), u);
    ig_bias8(p.bias[g], (int)((v * 8) % p.C), b);
    float4* Gv = reinterpret_cast<float4*>(p.G[g]) + 2 * v;
    const float4 g0 = Gv[0], g1 = Gv[1];
    acc[0] = g0.x; acc[1] = g0.y; acc[2] = g0.z; acc[3] = g0.w; acc[4] = g1.x; acc[5] = g1.y; acc[6] = g1.z; acc[7] = g1.w;
    for (int k = 0; k < p.n; ++k) {
      const float a = __ldg(p.alpha + k), wk = __ldg(p.w + k);
      const float4* gk = reinterpret_cast<const float4*>(p.grad[g]) + 2 * ((int64_t)k * p.nvec + v);
      const float4 d0 = __ldg(gk), d1 = __ldg(gk + 1);
      const float gr[8] = {d0.x, d0.y, d0.z, d0.w, d1.x, d1.y, d1.z, d1.w};
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const float z = fmaf(a, u[c], b[c]);
        acc[c] = __fmaf_rn(z > 0.f ? wk : __fmul_rn(wk, p.slope), gr[c], acc[c]);
      }
    }
    Gv[0] = make_float4(acc[0], acc[1], acc[2], acc[3]);
    Gv[1] = make_float4(acc[4], acc[5], acc[6], acc[7]);
  }
}

static int ig_setup(IgArgs& p, int ng, const void* const* umax, const float* const* bias, const float* alpha, int n, int B,
                    int64_t per, int C, float slope, const char* who) {
  TMF_REQUIRE(ng >= 1 && ng <= TMF_MAX_GROUPS, "%s: ng=%d out of range [1,%d]", who, ng, TMF_MAX_GROUPS);
  TMF_REQUIRE(n >= 1, "%s: n must be >= 1 (got %d)", who, n);
  TMF_REQUIRE(B >= 1 && per >= 1, "%s: bad problem B=%d per=%lld", who, B, (long long)per);
  TMF_REQUIRE(C >= 8 && C % 8 == 0 && per % C == 0, "%s: C must be a positive multiple of 8 dividing per (C=%d)", who, C);
  TMF_REQUIRE(slope >= 0.f, "%s: the LeakyReLU slope must be >= 0", who);
  TMF_REQUIRE(alpha != nullptr && umax != nullptr && bias != nullptr, "%s: NULL device pointer", who);
  p = IgArgs{};
  for (int g = 0; g < ng; ++g) {
    TMF_REQUIRE(umax[g] && bias[g], "%s: NULL device pointer", who);
    TMF_REQUIRE((((uintptr_t)umax[g] | (uintptr_t)bias[g]) & 15) == 0, "%s: tensors must be 16-byte aligned", who);
    p.umax[g] = (const __nv_bfloat16*)umax[g];
    p.bias[g] = bias[g];
  }
  p.alpha = alpha;
  p.nvec = (int64_t)B * per / 8;
  p.C = C; p.n = n; p.slope = slope;
  return 0;
}

static dim3 ig_grid(const IgArgs& p, int ng) {
  const int64_t blocks = (p.nvec + IG_THREADS - 1) / IG_THREADS;
  return dim3((unsigned)(blocks < IG_MAX_BLOCKS ? blocks : IG_MAX_BLOCKS), 1, (unsigned)ng);
}

}  // namespace tmf

using namespace tmf;

extern "C" {

int tmf_ig_expand(int ng, const void* const* umax, const float* const* bias, const float* alpha, int n, void* const* a1,
                  float* const* a1_32, int B, int64_t per, int C, float slope, void* stream) {
  IgArgs p;
  if (ig_setup(p, ng, umax, bias, alpha, n, B, per, C, slope, "ig_expand") != 0) return 1;
  for (int g = 0; g < ng; ++g) {
    TMF_REQUIRE(a1 && a1_32 && a1[g] && a1_32[g], "ig_expand: NULL device pointer");
    TMF_REQUIRE((((uintptr_t)a1[g] | (uintptr_t)a1_32[g]) & 15) == 0, "ig_expand: tensors must be 16-byte aligned");
    p.a1[g] = (__nv_bfloat16*)a1[g];
    p.a32[g] = a1_32[g];
  }
  launch_k(ig_expand_kernel, ig_grid(p, ng), IG_THREADS, 0, (cudaStream_t)stream, p);
  TMF_LAUNCH_CHECK();
  return 0;
}

int tmf_ig_combine(int ng, const float* const* grad, const void* const* umax, const float* const* bias, const float* alpha,
                   const float* w, int n, float* const* G, int B, int64_t per, int C, float slope, void* stream) {
  IgArgs p;
  if (ig_setup(p, ng, umax, bias, alpha, n, B, per, C, slope, "ig_combine") != 0) return 1;
  TMF_REQUIRE(w != nullptr, "ig_combine: NULL device pointer");
  p.w = w;
  for (int g = 0; g < ng; ++g) {
    TMF_REQUIRE(grad && G && grad[g] && G[g], "ig_combine: NULL device pointer");
    TMF_REQUIRE((((uintptr_t)grad[g] | (uintptr_t)G[g]) & 15) == 0, "ig_combine: tensors must be 16-byte aligned");
    p.grad[g] = grad[g];
    p.G[g] = G[g];
  }
  launch_k(ig_combine_kernel, ig_grid(p, ng), IG_THREADS, 0, (cudaStream_t)stream, p);
  TMF_LAUNCH_CHECK();
  return 0;
}

int64_t tmf_ig_attribute_workspace_bytes(int ng, int B, int64_t per) {
  return (int64_t)ng * B * lrp_blocks(per) * (int64_t)sizeof(float);
}

int tmf_ig_attribute(int ng, const float* const* x, float* const* dx, float* const* sums, int B, int64_t per, void* ws,
                     size_t ws_bytes, void* stream) {
  TMF_CHECK_NG(ng);
  TMF_REQUIRE(B >= 1 && B <= 65535 && per >= 1, "ig_attribute: bad problem B=%d per=%lld", B, (long long)per);
  const size_t need = (size_t)tmf_ig_attribute_workspace_bytes(ng, B, per);
  TMF_REQUIRE(ws != nullptr && ws_bytes >= need && ((uintptr_t)ws & 15) == 0,
              "ig_attribute: needs a 16-byte aligned workspace of %zu bytes (got %zu)", need, ws_bytes);
  TMF_REQUIRE(sums != nullptr, "ig_attribute: NULL device pointer");
  for (int g = 0; g < ng; ++g) TMF_REQUIRE(sums[g] != nullptr, "ig_attribute: NULL device pointer");
  return lrp_xmul(ng, x, dx, sums, 0, B, per, (float*)ws, (cudaStream_t)stream);
}

}  // extern "C"

// occlusion.cu -- occlusion sensitivity through the sNet towers with incremental recomputation (DESIGN section 3.11;
// Zeiler & Fergus 2014, Nakandala et al. 2019).  A window changes every layer's activation only inside a small region, so the
// occluded towers run layer by layer on fixed-extent crops of (windows x B) samples and the rest comes from the activations of
// the unoccluded forward.  The crop geometry is planned on the host (functional.OccPlan): one int32 table [m][3][4] per layer
// and pass holds, per window and axis, {crop origin, lo, hi of the changed region, origin of the previous layer's recomputed
// output}, in the global coordinates of the layer's input.
//
//   tmf_occ_input    the fp32 layer-0 crops: the volume with the window's voxels set to the baseline
//   tmf_occ_compose  a layer's input crops (bf16, or fp32 for the tower outputs): the changed region from the previous
//                    layer's recomputed crops, everything else from the kept base activation
//   tmf_occ_map      per voxel, the mean score of the windows that contain it
//
// All three are copies or fixed-order sums: memory-bound, CUDA cores, no atomics, 64-bit offsets, every output written once.
#include "common.cuh"

namespace tmf {

constexpr int OCC_THREADS = 256;
constexpr int OCC_MAX_BLOCKS = 148 * 16;       // CTAs per tower; grid-stride loops over the work items

struct OccInputArgs {
  const float* x[TMF_MAX_GROUPS];              // [B][D][H][W]
  float* out[TMF_MAX_GROUPS];                  // [m][B][Dc][Hc][Wc], window-major
  const int* tab;                              // [m][3][4]
  int64_t total;                               // m * B * Dc * Hc * Wc
  int B, D, H, W, Dc, Hc, Wc;
  float baseline;
};

struct OccComposeArgs {
  const void* base[TMF_MAX_GROUPS];            // [B][D][H][W][C]
  const void* crop[TMF_MAX_GROUPS];            // [m][B][Dp][Hp][Wp][C] (NULL: the base, replicated per window)
  void* out[TMF_MAX_GROUPS];                   // [m][B][Dc][Hc][Wc][C]
  const int* tab;                              // [m][3][4]
  int64_t total;                               // 8-channel vectors: m * B * Dc * Hc * Wc * C / 8
  int B, D, H, W, Dc, Hc, Wc, Dp, Hp, Wp, C;
};

struct OccMapArgs {
  const float* scores[TMF_MAX_GROUPS];         // [B][nD][nH][nW]
  float* map[TMF_MAX_GROUPS];                  // [B][D][H][W]
  int64_t total;                               // B * D * H * W
  int B, D, H, W, n[3], w[3], s[3];
};

__global__ void __launch_bounds__(OCC_THREADS) occ_input_kernel(const __grid_constant__ OccInputArgs p) {
  const int g = blockIdx.z;
  for (int64_t i = (int64_t)blockIdx.x * OCC_THREADS + threadIdx.x; i < p.total; i += (int64_t)gridDim.x * OCC_THREADS) {
    int64_t r = i;
    const int z = (int)(r % p.Wc); r /= p.Wc;
    const int y = (int)(r % p.Hc); r /= p.Hc;
    const int x = (int)(r % p.Dc); r /= p.Dc;
    const int b = (int)(r % p.B);
    const int* t = p.tab + (r / p.B) * 12;
    const int gd = __ldg(t) + x, gh = __ldg(t + 4) + y, gw = __ldg(t + 8) + z;
    const bool in = gd >= __ldg(t + 1) && gd < __ldg(t + 2) && gh >= __ldg(t + 5) && gh < __ldg(t + 6) &&
                    gw >= __ldg(t + 9) && gw < __ldg(t + 10);
    p.out[g][i] = in ? p.baseline : __ldg(p.x[g] + (((int64_t)b * p.D + gd) * p.H + gh) * p.W + gw);
  }
}

// One thread per 8-channel vector of the output crop: 16 bytes (bf16) or 32 bytes (fp32) copied from one of two sources.
template <bool FP32>
__global__ void __launch_bounds__(OCC_THREADS) occ_compose_kernel(const __grid_constant__ OccComposeArgs p) {
  const int g = blockIdx.z;
  const int CV = p.C / 8;
  for (int64_t i = (int64_t)blockIdx.x * OCC_THREADS + threadIdx.x; i < p.total; i += (int64_t)gridDim.x * OCC_THREADS) {
    int64_t r = i;
    const int cv = (int)(r % CV); r /= CV;
    const int z = (int)(r % p.Wc); r /= p.Wc;
    const int y = (int)(r % p.Hc); r /= p.Hc;
    const int x = (int)(r % p.Dc); r /= p.Dc;
    const int b = (int)(r % p.B);
    const int64_t n = r / p.B;
    const int* t = p.tab + n * 12;
    const int gd = __ldg(t) + x, gh = __ldg(t + 4) + y, gw = __ldg(t + 8) + z;
    const bool in = p.crop[g] != nullptr && gd >= __ldg(t + 1) && gd < __ldg(t + 2) && gh >= __ldg(t + 5) &&
                    gh < __ldg(t + 6) && gw >= __ldg(t + 9) && gw < __ldg(t + 10);
    const int64_t src = in ? ((((n * p.B + b) * p.Dp + (gd - __ldg(t + 3))) * p.Hp + (gh - __ldg(t + 7))) * p.Wp +
                              (gw - __ldg(t + 11))) * CV + cv
                           : ((((int64_t)b * p.D + gd) * p.H + gh) * p.W + gw) * CV + cv;
    const void* from = in ? p.crop[g] : p.base[g];
    if (FP32) {
      const float4* s = reinterpret_cast<const float4*>(from) + 2 * src;
      float4* d = reinterpret_cast<float4*>(p.out[g]) + 2 * i;
      const float4 lo = __ldg(s), hi = __ldg(s + 1);
      d[0] = lo;
      d[1] = hi;
    } else {
      reinterpret_cast<uint4*>(p.out[g])[i] = __ldg(reinterpret_cast<const uint4*>(from) + src);
    }
  }
}

// One thread per voxel: the windows that contain it along each axis are i0 .. i1-1; their scores are added in window order.
__global__ void __launch_bounds__(OCC_THREADS) occ_map_kernel(const __grid_constant__ OccMapArgs p) {
  const int g = blockIdx.z;
  for (int64_t i = (int64_t)blockIdx.x * OCC_THREADS + threadIdx.x; i < p.total; i += (int64_t)gridDim.x * OCC_THREADS) {
    int64_t r = i;
    int c[3];
    c[2] = (int)(r % p.W); r /= p.W;
    c[1] = (int)(r % p.H); r /= p.H;
    c[0] = (int)(r % p.D);
    const int b = (int)(r / p.D);
    int lo[3], hi[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      lo[a] = c[a] >= p.w[a] ? (c[a] - p.w[a] + p.s[a]) / p.s[a] : 0;      // first i with i*s + w > c
      hi[a] = min(p.n[a], c[a] / p.s[a] + 1);                               // last i with i*s <= c, plus one
    }
    float acc = 0.f;
    const float* sc = p.scores[g] + (int64_t)b * p.n[0] * p.n[1] * p.n[2];
    for (int u = lo[0]; u < hi[0]; ++u)
      for (int v = lo[1]; v < hi[1]; ++v)
        for (int w = lo[2]; w < hi[2]; ++w) acc += __ldg(sc + ((int64_t)u * p.n[1] + v) * p.n[2] + w);
    const int cnt = max(hi[0] - lo[0], 0) * max(hi[1] - lo[1], 0) * max(hi[2] - lo[2], 0);
    p.map[g][i] = cnt > 0 ? acc / (float)cnt : 0.f;
  }
}

static dim3 occ_grid(int64_t items, int ng) {
  const int64_t blocks = (items + OCC_THREADS - 1) / OCC_THREADS;
  return dim3((unsigned)(blocks < OCC_MAX_BLOCKS ? blocks : OCC_MAX_BLOCKS), 1, (unsigned)ng);
}

}  // namespace tmf

using namespace tmf;

extern "C" {

int tmf_occ_input(int ng, const float* const* x, const int* tab, int m, float baseline, float* const* out, int B, int D,
                  int H, int W, int Dc, int Hc, int Wc, void* stream) {
  TMF_CHECK_NG(ng);
  TMF_REQUIRE(m >= 1 && B >= 1 && D >= 1 && H >= 1 && W >= 1, "occ_input: bad problem m=%d B=%d (%d,%d,%d)", m, B, D, H, W);
  TMF_REQUIRE(Dc >= 1 && Hc >= 1 && Wc >= 1 && Dc <= D && Hc <= H && Wc <= W, "occ_input: crop (%d,%d,%d) outside (%d,%d,%d)",
              Dc, Hc, Wc, D, H, W);
  TMF_REQUIRE(tab != nullptr && x != nullptr && out != nullptr, "occ_input: NULL pointer");
  OccInputArgs p{};
  for (int g = 0; g < ng; ++g) {
    TMF_REQUIRE(x[g] && out[g], "occ_input: NULL device pointer");
    p.x[g] = x[g];
    p.out[g] = out[g];
  }
  p.tab = tab;
  p.total = (int64_t)m * B * Dc * Hc * Wc;
  p.B = B; p.D = D; p.H = H; p.W = W; p.Dc = Dc; p.Hc = Hc; p.Wc = Wc;
  p.baseline = baseline;
  launch_k(occ_input_kernel, occ_grid(p.total, ng), OCC_THREADS, 0, (cudaStream_t)stream, p);
  TMF_LAUNCH_CHECK();
  return 0;
}

int tmf_occ_compose(int ng, const void* const* base, const void* const* crop, const int* tab, int m, void* const* out,
                    int B, int D, int H, int W, int Dc, int Hc, int Wc, int Dp, int Hp, int Wp, int C, int fp32,
                    void* stream) {
  TMF_CHECK_NG(ng);
  TMF_REQUIRE(m >= 1 && B >= 1 && D >= 1 && H >= 1 && W >= 1, "occ_compose: bad problem m=%d B=%d (%d,%d,%d)", m, B, D, H,
              W);
  TMF_REQUIRE(C >= 8 && C % 8 == 0, "occ_compose: C must be a positive multiple of 8 (got %d)", C);
  TMF_REQUIRE(Dc >= 1 && Hc >= 1 && Wc >= 1 && Dc <= D && Hc <= H && Wc <= W,
              "occ_compose: crop (%d,%d,%d) outside (%d,%d,%d)", Dc, Hc, Wc, D, H, W);
  TMF_REQUIRE(tab != nullptr && base != nullptr && out != nullptr, "occ_compose: NULL pointer");
  OccComposeArgs p{};
  for (int g = 0; g < ng; ++g) {
    const void* c = crop ? crop[g] : nullptr;
    TMF_REQUIRE(base[g] && out[g], "occ_compose: NULL device pointer");
    TMF_REQUIRE((((uintptr_t)base[g] | (uintptr_t)out[g] | (uintptr_t)c) & 15) == 0,
                "occ_compose: tensors must be 16-byte aligned");
    TMF_REQUIRE(c == nullptr || (Dp >= 1 && Hp >= 1 && Wp >= 1), "occ_compose: bad crop extent (%d,%d,%d)", Dp, Hp, Wp);
    p.base[g] = base[g];
    p.crop[g] = c;
    p.out[g] = out[g];
  }
  p.tab = tab;
  p.total = (int64_t)m * B * Dc * Hc * Wc * (C / 8);
  p.B = B; p.D = D; p.H = H; p.W = W; p.Dc = Dc; p.Hc = Hc; p.Wc = Wc; p.Dp = Dp; p.Hp = Hp; p.Wp = Wp; p.C = C;
  if (fp32)
    launch_k(occ_compose_kernel<true>, occ_grid(p.total, ng), OCC_THREADS, 0, (cudaStream_t)stream, p);
  else
    launch_k(occ_compose_kernel<false>, occ_grid(p.total, ng), OCC_THREADS, 0, (cudaStream_t)stream, p);
  TMF_LAUNCH_CHECK();
  return 0;
}

int tmf_occ_map(int ng, const float* const* scores, float* const* map, int B, int D, int H, int W, int nD, int nH, int nW,
                int wD, int wH, int wW, int sD, int sH, int sW, void* stream) {
  TMF_CHECK_NG(ng);
  TMF_REQUIRE(B >= 1 && D >= 1 && H >= 1 && W >= 1, "occ_map: bad problem B=%d (%d,%d,%d)", B, D, H, W);
  TMF_REQUIRE(nD >= 1 && nH >= 1 && nW >= 1 && wD >= 1 && wH >= 1 && wW >= 1 && sD >= 1 && sH >= 1 && sW >= 1,
              "occ_map: bad window grid");
  TMF_REQUIRE(scores != nullptr && map != nullptr, "occ_map: NULL pointer");
  OccMapArgs p{};
  for (int g = 0; g < ng; ++g) {
    TMF_REQUIRE(scores[g] && map[g], "occ_map: NULL device pointer");
    p.scores[g] = scores[g];
    p.map[g] = map[g];
  }
  p.total = (int64_t)B * D * H * W;
  p.B = B; p.D = D; p.H = H; p.W = W;
  p.n[0] = nD; p.n[1] = nH; p.n[2] = nW;
  p.w[0] = wD; p.w[1] = wH; p.w[2] = wW;
  p.s[0] = sD; p.s[1] = sH; p.s[2] = sW;
  launch_k(occ_map_kernel, occ_grid(p.total, ng), OCC_THREADS, 0, (cudaStream_t)stream, p);
  TMF_LAUNCH_CHECK();
  return 0;
}

}  // extern "C"

// shapley.cu -- Shapley value sampling over the regions of an integer mask through the sNet towers (DESIGN section 3.13;
// Castro, Gomez & Tejada 2009).  A chain walks one permutation of the regions from the baseline volume to x, adding one region
// per step; each step recomputes only the added region's bounding box, on the crops and tables of feature ablation
// (functional.BoxPlan).  Unlike ablation, a step's base is not the forward of x but the chain's own state after its previous
// step, so every chain carries a copy of the kept layer inputs and of the tower output, updated in place:
//
//   tmf_shap_input    the fp32 layer-0 crops: per voxel x where the rank of its region in the row's permutation is <= the row's
//                     step, else the baseline (a scalar or a per-voxel volume)
//   tmf_shap_compose  a layer's input crops (bf16, or fp32 for the tower outputs): the changed region from the previous layer's
//                     recomputed crops, everything else from the row's chain state; the changed region is written back into
//                     that state, which makes it the base of the chain's next step
//
// Both are copies: memory-bound, CUDA cores, no atomics, 64-bit offsets, every output written once.  Within a row, the compose
// reads the state outside [lo, hi) and writes it inside; rows of one launch belong to different chains (the host schedule
// puts a chain in a pass at most once), so no location is both read and written by one launch.
#include "common.cuh"

namespace tmf {

constexpr int SHAP_THREADS = 256;
constexpr int SHAP_MAX_BLOCKS = 148 * 16;      // CTAs per tower; grid-stride loops over the work items

struct ShapInputArgs {
  const float* x[TMF_MAX_GROUPS];              // [B][D][H][W]
  const float* bvol[TMF_MAX_GROUPS];           // [1|B][D][H][W], or NULL: the scalar bval
  float bval[TMF_MAX_GROUPS];
  int bsample[TMF_MAX_GROUPS];                 // bvol holds one volume per sample
  float* out[TMF_MAX_GROUPS];                  // [m][B][Dc][Hc][Wc], row-major over the pass's chains
  const int* mask;                             // [1|B][D][H][W], ids in [0, F)
  const int* tab;                              // [m][3][4]
  const int* rank;                             // [P][F]: position of each id in permutation p
  const int* perm;                             // [m]: the row's permutation
  const int* step;                             // [m]: the row's step
  int64_t total;                               // m * B * Dc * Hc * Wc
  int B, D, H, W, Dc, Hc, Wc, F, mask_sample;
};

struct ShapComposeArgs {
  void* state[TMF_MAX_GROUPS];                 // [S][B][D][H][W][C]: per chain the current layer input
  const void* crop[TMF_MAX_GROUPS];            // [m][B][Dp][Hp][Wp][C]
  void* out[TMF_MAX_GROUPS];                   // [m][B][Dc][Hc][Wc][C]
  const int* tab;                              // [m][3][4]
  const int* sidx;                             // [m]: the row's chain, an index into state
  int64_t total;                               // 8-channel vectors: m * B * Dc * Hc * Wc * C / 8
  int B, D, H, W, Dc, Hc, Wc, Dp, Hp, Wp, C;
};

__global__ void __launch_bounds__(SHAP_THREADS) shap_input_kernel(const __grid_constant__ ShapInputArgs p) {
  const int g = blockIdx.z;
  const int64_t vox = (int64_t)p.D * p.H * p.W;
  for (int64_t i = (int64_t)blockIdx.x * SHAP_THREADS + threadIdx.x; i < p.total; i += (int64_t)gridDim.x * SHAP_THREADS) {
    int64_t r = i;
    const int z = (int)(r % p.Wc); r /= p.Wc;
    const int y = (int)(r % p.Hc); r /= p.Hc;
    const int x = (int)(r % p.Dc); r /= p.Dc;
    const int b = (int)(r % p.B);
    const int64_t n = r / p.B;
    const int* t = p.tab + n * 12;
    const int64_t v = ((int64_t)(__ldg(t) + x) * p.H + (__ldg(t + 4) + y)) * p.W + (__ldg(t + 8) + z);
    const int id = __ldg(p.mask + (p.mask_sample ? b * vox : 0) + v);
    const bool added = __ldg(p.rank + (int64_t)__ldg(p.perm + n) * p.F + id) <= __ldg(p.step + n);
    float val;
    if (added)
      val = __ldg(p.x[g] + b * vox + v);
    else if (p.bvol[g] != nullptr)
      val = __ldg(p.bvol[g] + (p.bsample[g] ? b * vox : 0) + v);
    else
      val = p.bval[g];
    p.out[g][i] = val;
  }
}

// One thread per 8-channel vector of the output crop: 16 bytes (bf16) or 32 bytes (fp32) from the crop or the chain state,
// and the same bytes written back to the state inside the changed region.  The state is read with plain loads: the launch
// writes it, though never at a location it reads.
template <bool FP32>
__global__ void __launch_bounds__(SHAP_THREADS) shap_compose_kernel(const __grid_constant__ ShapComposeArgs p) {
  const int g = blockIdx.z;
  const int CV = p.C / 8;
  for (int64_t i = (int64_t)blockIdx.x * SHAP_THREADS + threadIdx.x; i < p.total; i += (int64_t)gridDim.x * SHAP_THREADS) {
    int64_t r = i;
    const int cv = (int)(r % CV); r /= CV;
    const int z = (int)(r % p.Wc); r /= p.Wc;
    const int y = (int)(r % p.Hc); r /= p.Hc;
    const int x = (int)(r % p.Dc); r /= p.Dc;
    const int b = (int)(r % p.B);
    const int64_t n = r / p.B;
    const int* t = p.tab + n * 12;
    const int gd = __ldg(t) + x, gh = __ldg(t + 4) + y, gw = __ldg(t + 8) + z;
    const bool in = gd >= __ldg(t + 1) && gd < __ldg(t + 2) && gh >= __ldg(t + 5) && gh < __ldg(t + 6) &&
                    gw >= __ldg(t + 9) && gw < __ldg(t + 10);
    const int64_t row = (int64_t)__ldg(p.sidx + n) * p.B + b;
    const int64_t st = (((row * p.D + gd) * p.H + gh) * p.W + gw) * CV + cv;
    if (FP32) {
      float4* d = reinterpret_cast<float4*>(p.out[g]) + 2 * i;
      float4* s = reinterpret_cast<float4*>(p.state[g]) + 2 * st;
      float4 lo, hi;
      if (in) {
        const int64_t src = ((((n * p.B + b) * p.Dp + (gd - __ldg(t + 3))) * p.Hp + (gh - __ldg(t + 7))) * p.Wp +
                             (gw - __ldg(t + 11))) * CV + cv;
        const float4* c = reinterpret_cast<const float4*>(p.crop[g]) + 2 * src;
        lo = __ldg(c);
        hi = __ldg(c + 1);
        s[0] = lo;
        s[1] = hi;
      } else {
        lo = s[0];
        hi = s[1];
      }
      d[0] = lo;
      d[1] = hi;
    } else {
      uint4* s = reinterpret_cast<uint4*>(p.state[g]) + st;
      uint4 v;
      if (in) {
        const int64_t src = ((((n * p.B + b) * p.Dp + (gd - __ldg(t + 3))) * p.Hp + (gh - __ldg(t + 7))) * p.Wp +
                             (gw - __ldg(t + 11))) * CV + cv;
        v = __ldg(reinterpret_cast<const uint4*>(p.crop[g]) + src);
        *s = v;
      } else {
        v = *s;
      }
      reinterpret_cast<uint4*>(p.out[g])[i] = v;
    }
  }
}

static dim3 shap_grid(int64_t items, int ng) {
  const int64_t blocks = (items + SHAP_THREADS - 1) / SHAP_THREADS;
  return dim3((unsigned)(blocks < SHAP_MAX_BLOCKS ? blocks : SHAP_MAX_BLOCKS), 1, (unsigned)ng);
}

}  // namespace tmf

using namespace tmf;

extern "C" {

int tmf_shap_input(int ng, const float* const* x, const int* mask, int mask_per_sample, const float* const* bvol,
                   const float* bval, int bvol_per_sample, const int* tab, const int* rank, int F, const int* perm,
                   const int* step, int m, float* const* out, int B, int D, int H, int W, int Dc, int Hc, int Wc,
                   void* stream) {
  TMF_CHECK_NG(ng);
  TMF_REQUIRE(m >= 1 && B >= 1 && D >= 1 && H >= 1 && W >= 1 && F >= 1, "shap_input: bad problem m=%d B=%d F=%d (%d,%d,%d)",
              m, B, F, D, H, W);
  TMF_REQUIRE(Dc >= 1 && Hc >= 1 && Wc >= 1 && Dc <= D && Hc <= H && Wc <= W,
              "shap_input: crop (%d,%d,%d) outside (%d,%d,%d)", Dc, Hc, Wc, D, H, W);
  TMF_REQUIRE(x != nullptr && mask != nullptr && bval != nullptr && tab != nullptr && rank != nullptr && perm != nullptr &&
              step != nullptr && out != nullptr, "shap_input: NULL pointer");
  ShapInputArgs p{};
  for (int g = 0; g < ng; ++g) {
    TMF_REQUIRE(x[g] && out[g], "shap_input: NULL device pointer");
    p.x[g] = x[g];
    p.out[g] = out[g];
    p.bvol[g] = bvol ? bvol[g] : nullptr;
    p.bval[g] = bval[g];
    p.bsample[g] = (bvol_per_sample >> g) & 1;
  }
  p.mask = mask;
  p.tab = tab;
  p.rank = rank;
  p.perm = perm;
  p.step = step;
  p.total = (int64_t)m * B * Dc * Hc * Wc;
  p.B = B; p.D = D; p.H = H; p.W = W; p.Dc = Dc; p.Hc = Hc; p.Wc = Wc; p.F = F;
  p.mask_sample = mask_per_sample != 0;
  launch_k(shap_input_kernel, shap_grid(p.total, ng), SHAP_THREADS, 0, (cudaStream_t)stream, p);
  TMF_LAUNCH_CHECK();
  return 0;
}

int tmf_shap_compose(int ng, void* const* state, const int* sidx, const void* const* crop, const int* tab, int m,
                     void* const* out, int B, int D, int H, int W, int Dc, int Hc, int Wc, int Dp, int Hp, int Wp, int C,
                     int fp32, void* stream) {
  TMF_CHECK_NG(ng);
  TMF_REQUIRE(m >= 1 && B >= 1 && D >= 1 && H >= 1 && W >= 1, "shap_compose: bad problem m=%d B=%d (%d,%d,%d)", m, B, D, H,
              W);
  TMF_REQUIRE(C >= 8 && C % 8 == 0, "shap_compose: C must be a positive multiple of 8 (got %d)", C);
  TMF_REQUIRE(Dc >= 1 && Hc >= 1 && Wc >= 1 && Dc <= D && Hc <= H && Wc <= W,
              "shap_compose: crop (%d,%d,%d) outside (%d,%d,%d)", Dc, Hc, Wc, D, H, W);
  TMF_REQUIRE(Dp >= 1 && Hp >= 1 && Wp >= 1, "shap_compose: bad crop extent (%d,%d,%d)", Dp, Hp, Wp);
  TMF_REQUIRE(state != nullptr && sidx != nullptr && crop != nullptr && tab != nullptr && out != nullptr,
              "shap_compose: NULL pointer");
  ShapComposeArgs p{};
  for (int g = 0; g < ng; ++g) {
    TMF_REQUIRE(state[g] && crop[g] && out[g], "shap_compose: NULL device pointer");
    TMF_REQUIRE((((uintptr_t)state[g] | (uintptr_t)out[g] | (uintptr_t)crop[g]) & 15) == 0,
                "shap_compose: tensors must be 16-byte aligned");
    p.state[g] = state[g];
    p.crop[g] = crop[g];
    p.out[g] = out[g];
  }
  p.tab = tab;
  p.sidx = sidx;
  p.total = (int64_t)m * B * Dc * Hc * Wc * (C / 8);
  p.B = B; p.D = D; p.H = H; p.W = W; p.Dc = Dc; p.Hc = Hc; p.Wc = Wc; p.Dp = Dp; p.Hp = Hp; p.Wp = Wp; p.C = C;
  if (fp32)
    launch_k(shap_compose_kernel<true>, shap_grid(p.total, ng), SHAP_THREADS, 0, (cudaStream_t)stream, p);
  else
    launch_k(shap_compose_kernel<false>, shap_grid(p.total, ng), SHAP_THREADS, 0, (cudaStream_t)stream, p);
  TMF_LAUNCH_CHECK();
  return 0;
}

}  // extern "C"

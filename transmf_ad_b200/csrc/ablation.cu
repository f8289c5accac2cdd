// ablation.cu -- feature ablation over the regions of an integer mask through the sNet towers, recomputing only each region's
// bounding box (DESIGN section 3.12).  The crops, tables and layers 1-6 are those of occlusion (occlusion.cu,
// functional.BoxPlan); only the layer-0 crops and the voxel map differ:
//
//   tmf_abl_input  the fp32 layer-0 crops: x, or the baseline (a scalar or a per-voxel volume) where the voxel's mask id is the
//                  row's feature id
//   tmf_abl_map    per voxel, the score of the voxel's feature
//
// Both are copies: memory-bound, CUDA cores, no atomics, 64-bit offsets, every output written once.
#include "common.cuh"

namespace tmf {

constexpr int ABL_THREADS = 256;
constexpr int ABL_MAX_BLOCKS = 148 * 16;       // CTAs per tower; grid-stride loops over the work items

struct AblInputArgs {
  const float* x[TMF_MAX_GROUPS];              // [B][D][H][W]
  const float* bvol[TMF_MAX_GROUPS];           // [1|B][D][H][W], or NULL: the scalar bval
  float bval[TMF_MAX_GROUPS];
  int bsample[TMF_MAX_GROUPS];                 // bvol holds one volume per sample
  float* out[TMF_MAX_GROUPS];                  // [m][B][Dc][Hc][Wc], box-major
  const int* mask;                             // [1|B][D][H][W]
  const int* tab;                              // [m][3][4]
  const int* ids;                              // [m]
  int64_t total;                               // m * B * Dc * Hc * Wc
  int B, D, H, W, Dc, Hc, Wc, mask_sample;
};

struct AblMapArgs {
  const float* scores[TMF_MAX_GROUPS];         // [B][F]
  float* map[TMF_MAX_GROUPS];                  // [B][D][H][W]
  const int* mask;                             // [1|B][D][H][W]
  int64_t total;                               // B * D * H * W
  int64_t vox;                                 // D * H * W
  int F, mask_sample;
};

__global__ void __launch_bounds__(ABL_THREADS) abl_input_kernel(const __grid_constant__ AblInputArgs p) {
  const int g = blockIdx.z;
  const int64_t vox = (int64_t)p.D * p.H * p.W;
  for (int64_t i = (int64_t)blockIdx.x * ABL_THREADS + threadIdx.x; i < p.total; i += (int64_t)gridDim.x * ABL_THREADS) {
    int64_t r = i;
    const int z = (int)(r % p.Wc); r /= p.Wc;
    const int y = (int)(r % p.Hc); r /= p.Hc;
    const int x = (int)(r % p.Dc); r /= p.Dc;
    const int b = (int)(r % p.B);
    const int64_t n = r / p.B;
    const int* t = p.tab + n * 12;
    const int gd = __ldg(t) + x, gh = __ldg(t + 4) + y, gw = __ldg(t + 8) + z;
    const int64_t v = ((int64_t)gd * p.H + gh) * p.W + gw;
    bool in = gd >= __ldg(t + 1) && gd < __ldg(t + 2) && gh >= __ldg(t + 5) && gh < __ldg(t + 6) && gw >= __ldg(t + 9) &&
              gw < __ldg(t + 10);
    in = in && __ldg(p.mask + (p.mask_sample ? b * vox : 0) + v) == __ldg(p.ids + n);
    float val;
    if (!in)
      val = __ldg(p.x[g] + b * vox + v);
    else if (p.bvol[g] != nullptr)
      val = __ldg(p.bvol[g] + (p.bsample[g] ? b * vox : 0) + v);
    else
      val = p.bval[g];
    p.out[g][i] = val;
  }
}

__global__ void __launch_bounds__(ABL_THREADS) abl_map_kernel(const __grid_constant__ AblMapArgs p) {
  const int g = blockIdx.z;
  for (int64_t i = (int64_t)blockIdx.x * ABL_THREADS + threadIdx.x; i < p.total; i += (int64_t)gridDim.x * ABL_THREADS) {
    const int64_t b = i / p.vox;
    const int id = __ldg(p.mask + (p.mask_sample ? i : i - b * p.vox));
    p.map[g][i] = id >= 0 && id < p.F ? __ldg(p.scores[g] + b * p.F + id) : 0.f;
  }
}

static dim3 abl_grid(int64_t items, int ng) {
  const int64_t blocks = (items + ABL_THREADS - 1) / ABL_THREADS;
  return dim3((unsigned)(blocks < ABL_MAX_BLOCKS ? blocks : ABL_MAX_BLOCKS), 1, (unsigned)ng);
}

}  // namespace tmf

using namespace tmf;

extern "C" {

int tmf_abl_input(int ng, const float* const* x, const int* mask, int mask_per_sample, const float* const* bvol,
                  const float* bval, int bvol_per_sample, const int* tab, const int* ids, int m, float* const* out, int B,
                  int D, int H, int W, int Dc, int Hc, int Wc, void* stream) {
  TMF_CHECK_NG(ng);
  TMF_REQUIRE(m >= 1 && B >= 1 && D >= 1 && H >= 1 && W >= 1, "abl_input: bad problem m=%d B=%d (%d,%d,%d)", m, B, D, H, W);
  TMF_REQUIRE(Dc >= 1 && Hc >= 1 && Wc >= 1 && Dc <= D && Hc <= H && Wc <= W, "abl_input: crop (%d,%d,%d) outside (%d,%d,%d)",
              Dc, Hc, Wc, D, H, W);
  TMF_REQUIRE(x != nullptr && mask != nullptr && bval != nullptr && tab != nullptr && ids != nullptr && out != nullptr,
              "abl_input: NULL pointer");
  AblInputArgs p{};
  for (int g = 0; g < ng; ++g) {
    TMF_REQUIRE(x[g] && out[g], "abl_input: NULL device pointer");
    p.x[g] = x[g];
    p.out[g] = out[g];
    p.bvol[g] = bvol ? bvol[g] : nullptr;
    p.bval[g] = bval[g];
    p.bsample[g] = (bvol_per_sample >> g) & 1;
  }
  p.mask = mask;
  p.tab = tab;
  p.ids = ids;
  p.total = (int64_t)m * B * Dc * Hc * Wc;
  p.B = B; p.D = D; p.H = H; p.W = W; p.Dc = Dc; p.Hc = Hc; p.Wc = Wc;
  p.mask_sample = mask_per_sample != 0;
  launch_k(abl_input_kernel, abl_grid(p.total, ng), ABL_THREADS, 0, (cudaStream_t)stream, p);
  TMF_LAUNCH_CHECK();
  return 0;
}

int tmf_abl_map(int ng, const float* const* scores, const int* mask, int mask_per_sample, int F, float* const* map, int B,
                int D, int H, int W, void* stream) {
  TMF_CHECK_NG(ng);
  TMF_REQUIRE(B >= 1 && D >= 1 && H >= 1 && W >= 1 && F >= 1, "abl_map: bad problem B=%d F=%d (%d,%d,%d)", B, F, D, H, W);
  TMF_REQUIRE(scores != nullptr && mask != nullptr && map != nullptr, "abl_map: NULL pointer");
  AblMapArgs p{};
  for (int g = 0; g < ng; ++g) {
    TMF_REQUIRE(scores[g] && map[g], "abl_map: NULL device pointer");
    p.scores[g] = scores[g];
    p.map[g] = map[g];
  }
  p.mask = mask;
  p.vox = (int64_t)D * H * W;
  p.total = (int64_t)B * p.vox;
  p.F = F;
  p.mask_sample = mask_per_sample != 0;
  launch_k(abl_map_kernel, abl_grid(p.total, ng), ABL_THREADS, 0, (cudaStream_t)stream, p);
  TMF_LAUNCH_CHECK();
  return 0;
}

}  // extern "C"

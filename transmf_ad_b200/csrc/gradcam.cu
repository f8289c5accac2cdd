// gradcam.cu -- Grad-CAM on an sNet block output, and the bf16 <-> fp32 conversions at the boundaries of a segmented sNet
// run (the block outputs exposed to module hooks; transmf_ad_b200/functional.py, DESIGN section 3.7).
//
// Grad-CAM (Selvaraju et al., 2017) of activations A and their gradient G, both fp32 [B, P = d*h*w, C] (channels-last):
//   alpha[b,c] = mean_p G[b,p,c]                  (double, fixed summation order: per-chunk partial rows, then the rows
//                                                   in index order -- no atomics, DESIGN section 10.1)
//   cam[b,p]   = ReLU(sum_c alpha[b,c] * A[b,p,c])
// then optionally trilinear upsampling to (D,H,W) (F.interpolate(mode="trilinear", align_corners=False)) and per-sample
// normalisation (cam - min) / (max - min + 1e-7) over the returned map.  A and G are read once each, the map written once.
#include "common.cuh"

namespace tmf {

// ---- bf16 <-> fp32 ---------------------------------------------------------------------------------------------------
template <bool WIDEN>
__global__ void __launch_bounds__(256) convert_kernel(GroupPtr<const void> src, GroupPtr<void> dst, int64_t n8) {
  const int g = blockIdx.z;
  for (int64_t i = blockIdx.x * 256ll + threadIdx.x; i < n8; i += (int64_t)gridDim.x * 256) {
    if (WIDEN) {
      float f[8];
      unpack8(reinterpret_cast<const uint4*>(src.p[g])[i], f);
      float4* d = reinterpret_cast<float4*>(dst.p[g]) + 2 * i;
      d[0] = make_float4(f[0], f[1], f[2], f[3]);
      d[1] = make_float4(f[4], f[5], f[6], f[7]);
    } else {
      const float4* s = reinterpret_cast<const float4*>(src.p[g]) + 2 * i;
      const float4 a = s[0], b = s[1];
      const float f[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
      reinterpret_cast<uint4*>(dst.p[g])[i] = pack8(f);
    }
  }
}

// ---- Grad-CAM ----------------------------------------------------------------------------------------------------------
struct CamPlan {
  int P, CQ, pstep;        // positions per sample; float4 chunks per position; positions per block pass (alpha kernel)
  int nch, chlen;          // alpha: chunks of positions per sample, positions per chunk
  int lanes, nmap;         // map kernel: lanes per position (a power of two <= 32), blocks per sample
  int64_t nout;            // returned voxels per sample
  int nres;                // resample kernel blocks per sample
  size_t off_lo, off_mm, bytes;
};

constexpr int CAM_THREADS = 256;

// The plan depends on (B, extents, C) only -- never on ng -- so a tower gets the same bits alone or with the other one.
static CamPlan cam_plan(int ng, int B, int d, int h, int w, int C, int D, int H, int W, int upsample, int normalize) {
  CamPlan pl{};
  pl.P = d * h * w;
  pl.CQ = C / 4;
  pl.pstep = CAM_THREADS / pl.CQ;
  const int target = (148 * 4 + B - 1) / B;                        // ~4 blocks per SM over the batch
  int maxch = ceil_div(pl.P, (int64_t)pl.pstep * 4);               // >= 4 positions per thread
  pl.nch = target < maxch ? target : maxch;
  if (pl.nch < 1) pl.nch = 1;
  pl.chlen = ceil_div(pl.P, pl.nch);
  pl.nch = ceil_div(pl.P, pl.chlen);
  pl.lanes = 1;
  while (pl.lanes * 2 <= pl.CQ && pl.lanes < 32) pl.lanes *= 2;
  const int per_block = (CAM_THREADS / 32) * (32 / pl.lanes) * 4;  // positions per block: 4 per lane group
  pl.nmap = ceil_div(pl.P, per_block);
  if (pl.nmap > 2 * target) pl.nmap = 2 * target;                   // blocks loop over the positions of their sample
  pl.nout = upsample ? (int64_t)D * H * W : pl.P;
  pl.nres = (int)((pl.nout + CAM_THREADS * 8 - 1) / (CAM_THREADS * 8));
  if (pl.nres > target) pl.nres = target;
  if (pl.nres < 1) pl.nres = 1;
  const size_t alpha_bytes = (size_t)ng * B * (pl.nch + 1) * C * sizeof(double);     // partial rows, then alpha
  pl.off_lo = (alpha_bytes + 255) / 256 * 256;
  const size_t lo_bytes = upsample ? (size_t)ng * B * pl.P * sizeof(float) : 0;
  pl.off_mm = pl.off_lo + (lo_bytes + 255) / 256 * 256;
  const int nparts = upsample ? pl.nres : pl.nmap;
  pl.bytes = pl.off_mm + (normalize ? (size_t)ng * B * nparts * 2 * sizeof(float) : 0);
  return pl;
}

struct CamArgs {
  GroupPtr<const float> A, G;
  GroupPtr<float> out;
  double* alpha_part;      // [ng][B][nch][C] partial rows
  double* alpha;           // [ng][B][C]
  float* lo;               // [ng][B][P] low-resolution map (upsample) or NULL (the map is written to out)
  float* mm;               // [ng][B][nparts][2] per-block minimum / maximum (normalize) or NULL
  int B, d, h, w, C, D, H, W, P, CQ, pstep, nch, chlen, lanes, nparts;
  int64_t nout;
};

// Partial column sums of G over one chunk of positions of one sample: thread (k, cq) adds positions k, k+pstep, ... of the
// chunk for channels 4cq..4cq+3 in double; the block then adds its pstep rows in index order.
__global__ void __launch_bounds__(CAM_THREADS) cam_alpha_kernel(CamArgs a) {
  __shared__ double red[CAM_THREADS * 4];
  const int g = blockIdx.z, b = blockIdx.y, chunk = blockIdx.x;
  const int cq = threadIdx.x % a.CQ, k = threadIdx.x / a.CQ;
  const bool active = k < a.pstep;
  const int p0 = chunk * a.chlen, p1 = min(p0 + a.chlen, a.P);
  double s[4] = {0.0, 0.0, 0.0, 0.0};
  if (active) {
    const float4* Gb = reinterpret_cast<const float4*>(a.G.p[g] + (int64_t)b * a.P * a.C) + cq;
    int p = p0 + k;
    for (; p + 3 * a.pstep < p1; p += 4 * a.pstep) {              // four independent loads in flight
      float4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) v[u] = Gb[(int64_t)(p + u * a.pstep) * a.CQ];
#pragma unroll
      for (int u = 0; u < 4; ++u) { s[0] += v[u].x; s[1] += v[u].y; s[2] += v[u].z; s[3] += v[u].w; }
    }
    for (; p < p1; p += a.pstep) {
      const float4 v = Gb[(int64_t)p * a.CQ];
      s[0] += v.x; s[1] += v.y; s[2] += v.z; s[3] += v.w;
    }
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) red[threadIdx.x * 4 + j] = s[j];
  __syncthreads();
  double* row = a.alpha_part + (((int64_t)g * a.B + b) * a.nch + chunk) * a.C;
  for (int c = threadIdx.x; c < a.C; c += CAM_THREADS) {
    double t = 0.0;
    for (int kk = 0; kk < a.pstep; ++kk) t += red[(kk * a.CQ + (c >> 2)) * 4 + (c & 3)];
    row[c] = t;
  }
}

// alpha[b,:] = (sum of the partial rows in index order) / P.  Rows are staged through shared memory CAM_STAGE values at a time, so
// the loads are issued together instead of as one dependent chain per channel.
constexpr int CAM_STAGE = 4096;                                     // doubles per staging pass
__global__ void __launch_bounds__(CAM_THREADS) cam_alpha_final_kernel(CamArgs a) {
  extern __shared__ double sm[];                                    // [CAM_STAGE] staging + [C] totals
  double* acc = sm + CAM_STAGE;
  const int g = blockIdx.z, b = blockIdx.y;
  const double* rows = a.alpha_part + ((int64_t)g * a.B + b) * a.nch * a.C;
  for (int c = threadIdx.x; c < a.C; c += CAM_THREADS) acc[c] = 0.0;
  const int R = CAM_STAGE / a.C;
  for (int r0 = 0; r0 < a.nch; r0 += R) {
    const int n = min(R, a.nch - r0) * a.C;
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += CAM_THREADS) sm[i] = rows[(int64_t)r0 * a.C + i];
    __syncthreads();
    for (int c = threadIdx.x; c < a.C; c += CAM_THREADS) {
      double t = acc[c];
      for (int i = c; i < n; i += a.C) t += sm[i];
      acc[c] = t;
    }
  }
  for (int c = threadIdx.x; c < a.C; c += CAM_THREADS) a.alpha[((int64_t)g * a.B + b) * a.C + c] = acc[c] / (double)a.P;
}

__device__ __forceinline__ void block_minmax(float mn, float mx, float* dst) {
  __shared__ float smn[CAM_THREADS / 32], smx[CAM_THREADS / 32];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  }
  if ((threadIdx.x & 31) == 0) { smn[threadIdx.x >> 5] = mn; smx[threadIdx.x >> 5] = mx; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 1; i < CAM_THREADS / 32; ++i) { mn = fminf(mn, smn[i]); mx = fmaxf(mx, smx[i]); }
    mn = fminf(mn, smn[0]); mx = fmaxf(mx, smx[0]);
    dst[0] = mn; dst[1] = mx;
  }
}

// cam[b,p] = ReLU(sum_c alpha[c] * A[b,p,c]): a group of `lanes` lanes (a power of two) per position, each lane a strided
// set of float4 channel chunks, products and the fixed shuffle tree in double.  Normalisation without upsampling also
// stores this block's minimum / maximum.
template <bool MINMAX>
__global__ void __launch_bounds__(CAM_THREADS) cam_map_kernel(CamArgs a) {
  extern __shared__ double alpha[];
  const int g = blockIdx.z, b = blockIdx.y;
  for (int c = threadIdx.x; c < a.C; c += CAM_THREADS) alpha[c] = a.alpha[((int64_t)g * a.B + b) * a.C + c];
  __syncthreads();
  const int lanes = a.lanes;
  const int lane = threadIdx.x & 31, sub = lane % lanes, grp = lane / lanes;
  const int groups_per_warp = 32 / lanes, warp = threadIdx.x >> 5;
  const int per_block = (CAM_THREADS / 32) * groups_per_warp * 4;
  const float* Ab = a.A.p[g] + (int64_t)b * a.P * a.C;
  float* dst = (a.lo != nullptr ? a.lo + ((int64_t)g * a.B + b) * a.P : a.out.p[g] + (int64_t)b * a.P);
  float mn = INFINITY, mx = -INFINITY;
  // the loop bound is warp-uniform: every lane of a warp takes part in the shuffles below
  for (int wbase = blockIdx.x * per_block + warp * groups_per_warp * 4; wbase < a.P; wbase += gridDim.x * per_block) {
    const int pbase = wbase + grp * 4;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int p = pbase + u;
      double t = 0.0;
      if (p < a.P) {
        const float4* row = reinterpret_cast<const float4*>(Ab + (int64_t)p * a.C);
        for (int q = sub; q < a.CQ; q += lanes) {
          const float4 v = row[q];
          const double* al = alpha + 4 * q;
          t = fma((double)v.x, al[0], t);
          t = fma((double)v.y, al[1], t);
          t = fma((double)v.z, al[2], t);
          t = fma((double)v.w, al[3], t);
        }
      }
      for (int o = lanes / 2; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
      if (p < a.P) {
        const float v = fmaxf((float)t, 0.f);
        if (sub == 0) dst[p] = v;
        mn = fminf(mn, v);
        mx = fmaxf(mx, v);
      }
    }
  }
  if (MINMAX) block_minmax(mn, mx, a.mm + (((int64_t)g * a.B + b) * a.nparts + blockIdx.x) * 2);
}

// One value of the returned map: the low-resolution map itself or its trilinear interpolation at output voxel o
// (PyTorch's align_corners=False source index: (o + 0.5) * in / out - 0.5, clamped below at 0).
__device__ __forceinline__ void src_index(int o, int in, int out, int& i0, int& i1, float& l1) {
  const float scale = (float)in / (float)out;
  float s = ((float)o + 0.5f) * scale - 0.5f;
  if (s < 0.f) s = 0.f;
  i0 = (int)s;
  if (i0 > in - 1) i0 = in - 1;
  i1 = i0 + (i0 < in - 1 ? 1 : 0);
  l1 = s - (float)i0;
}

template <bool UPS>
__device__ __forceinline__ float cam_value(const CamArgs& a, const float* lo, int o) {
  if (!UPS) return lo[o];
  const int t = o / a.W, ow = o - t * a.W;
  const int od = t / a.H, oh = t - od * a.H;
  int d0, d1, h0, h1, w0, w1;
  float ld, lh, lw;
  src_index(od, a.d, a.D, d0, d1, ld);
  src_index(oh, a.h, a.H, h0, h1, lh);
  src_index(ow, a.w, a.W, w0, w1, lw);
  auto at = [&](int dd, int hh, int ww) { return lo[((int64_t)dd * a.h + hh) * a.w + ww]; };
  const float c00 = (1.f - lw) * at(d0, h0, w0) + lw * at(d0, h0, w1);
  const float c01 = (1.f - lw) * at(d0, h1, w0) + lw * at(d0, h1, w1);
  const float c10 = (1.f - lw) * at(d1, h0, w0) + lw * at(d1, h0, w1);
  const float c11 = (1.f - lw) * at(d1, h1, w0) + lw * at(d1, h1, w1);
  const float c0 = (1.f - lh) * c00 + lh * c01, c1 = (1.f - lh) * c10 + lh * c11;
  return (1.f - ld) * c0 + ld * c1;
}

// WRITE = false: this block's minimum / maximum of the returned map.  WRITE = true: the returned map, normalised with the
// sample's minimum / maximum over all partial rows when `normalize` (min / max are exact: the order does not matter).
template <bool UPS, bool WRITE>
__global__ void __launch_bounds__(CAM_THREADS) cam_resample_kernel(CamArgs a, int normalize) {
  const int g = blockIdx.z, b = blockIdx.y;
  const float* lo = UPS ? a.lo + ((int64_t)g * a.B + b) * a.P : a.out.p[g] + (int64_t)b * a.P;
  float* out = a.out.p[g] + (int64_t)b * a.nout;
  __shared__ float s_mn, s_mx;
  float mn = INFINITY, mx = -INFINITY;
  if (WRITE && normalize) {
    if (threadIdx.x == 0) {
      const float* mm = a.mm + ((int64_t)g * a.B + b) * a.nparts * 2;
      for (int i = 0; i < a.nparts; ++i) { mn = fminf(mn, mm[2 * i]); mx = fmaxf(mx, mm[2 * i + 1]); }
      s_mn = mn;
      s_mx = mx;
    }
    __syncthreads();
    mn = s_mn;
    mx = s_mx;
  }
  const float inv_den = WRITE && normalize ? 1.f / ((mx - mn) + 1e-7f) : 1.f;
  for (int o = blockIdx.x * CAM_THREADS + threadIdx.x; o < a.nout; o += gridDim.x * CAM_THREADS) {
    const float v = cam_value<UPS>(a, lo, o);
    if (WRITE) {
      out[o] = normalize ? (v - mn) * inv_den : v;
    } else {
      mn = fminf(mn, v);
      mx = fmaxf(mx, v);
    }
  }
  if (!WRITE) block_minmax(mn, mx, a.mm + (((int64_t)g * a.B + b) * a.nparts + blockIdx.x) * 2);
}

}  // namespace tmf

using namespace tmf;

extern "C" {

int tmf_widen_bf16(int ng, const void* const* src, float* const* dst, int64_t n, void* stream) {
  TMF_CHECK_NG(ng);
  TMF_REQUIRE(n > 0 && n % 8 == 0, "tmf_widen_bf16: n must be a positive multiple of 8 (got %lld)", (long long)n);
  GroupPtr<const void> s;
  GroupPtr<void> d;
  if (!load_group(s, src, ng, true, "src") || !load_group(d, (void* const*)dst, ng, true, "dst")) return 1;
  const int64_t n8 = n / 8;
  const int blocks = (int)(ceil_div(n8, 256) < 148 * 8 ? ceil_div(n8, 256) : 148 * 8);
  launch_k(convert_kernel<true>, dim3(blocks, 1, ng), 256, 0, (cudaStream_t)stream, s, d, n8);
  TMF_LAUNCH_CHECK();
  return 0;
}

int tmf_narrow_f32(int ng, const float* const* src, void* const* dst, int64_t n, void* stream) {
  TMF_CHECK_NG(ng);
  TMF_REQUIRE(n > 0 && n % 8 == 0, "tmf_narrow_f32: n must be a positive multiple of 8 (got %lld)", (long long)n);
  GroupPtr<const void> s;
  GroupPtr<void> d;
  if (!load_group(s, (const void* const*)src, ng, true, "src") || !load_group(d, dst, ng, true, "dst")) return 1;
  const int64_t n8 = n / 8;
  const int blocks = (int)(ceil_div(n8, 256) < 148 * 8 ? ceil_div(n8, 256) : 148 * 8);
  launch_k(convert_kernel<false>, dim3(blocks, 1, ng), 256, 0, (cudaStream_t)stream, s, d, n8);
  TMF_LAUNCH_CHECK();
  return 0;
}

int64_t tmf_gradcam_workspace_bytes(int ng, int B, int d, int h, int w, int C, int D, int H, int W, int upsample,
                                    int normalize) {
  if (ng < 1 || ng > TMF_MAX_GROUPS || B < 1 || d < 1 || h < 1 || w < 1 || C < 4 || C % 4 != 0 || C > 1024) return -1;
  if (upsample && (D < 1 || H < 1 || W < 1)) return -1;
  return (int64_t)cam_plan(ng, B, d, h, w, C, D, H, W, upsample, normalize).bytes;
}

int tmf_gradcam(int ng, const float* const* A, const float* const* G, float* const* cam, int B, int d, int h, int w, int C,
                int D, int H, int W, int upsample, int normalize, void* ws, size_t ws_bytes, void* stream) {
  TMF_CHECK_NG(ng);
  TMF_REQUIRE(B >= 1 && d >= 1 && h >= 1 && w >= 1, "tmf_gradcam: bad extent %dx%dx%dx%d", B, d, h, w);
  TMF_REQUIRE(C >= 4 && C % 4 == 0 && C <= 1024, "tmf_gradcam: C must be a multiple of 4 in [4,1024] (got %d)", C);
  TMF_REQUIRE(!upsample || (D >= 1 && H >= 1 && W >= 1), "tmf_gradcam: bad upsampling extent %dx%dx%d", D, H, W);
  TMF_REQUIRE((int64_t)d * h * w < (1ll << 31) && (!upsample || (int64_t)D * H * W < (1ll << 31)), "tmf_gradcam: extent too large");
  const CamPlan pl = cam_plan(ng, B, d, h, w, C, D, H, W, upsample, normalize);
  TMF_REQUIRE(ws != nullptr && ws_bytes >= pl.bytes, "tmf_gradcam: workspace of %zu bytes < %zu (tmf_gradcam_workspace_bytes)",
              ws_bytes, pl.bytes);
  TMF_REQUIRE(((uintptr_t)ws & 255) == 0, "tmf_gradcam: workspace must be 256-byte aligned");
  CamArgs a{};
  if (!load_group(a.A, A, ng, true, "A") || !load_group(a.G, G, ng, true, "G") || !load_group(a.out, cam, ng, true, "cam"))
    return 1;
  for (int g = 0; g < ng; ++g)
    TMF_REQUIRE(((uintptr_t)a.A.p[g] & 15) == 0 && ((uintptr_t)a.G.p[g] & 15) == 0, "tmf_gradcam: A / G must be 16-byte aligned");
  char* base = (char*)ws;
  a.alpha_part = (double*)base;
  a.alpha = a.alpha_part + (size_t)ng * B * pl.nch * C;
  a.lo = upsample ? (float*)(base + pl.off_lo) : nullptr;
  a.mm = normalize ? (float*)(base + pl.off_mm) : nullptr;
  a.B = B; a.d = d; a.h = h; a.w = w; a.C = C; a.D = D; a.H = H; a.W = W;
  a.P = pl.P; a.CQ = pl.CQ; a.pstep = pl.pstep; a.nch = pl.nch; a.chlen = pl.chlen; a.lanes = pl.lanes;
  a.nparts = upsample ? pl.nres : pl.nmap;
  a.nout = pl.nout;
  cudaStream_t st = (cudaStream_t)stream;
  launch_k(cam_alpha_kernel, dim3(pl.nch, B, ng), CAM_THREADS, 0, st, a);
  TMF_LAUNCH_CHECK();
  launch_k(cam_alpha_final_kernel, dim3(1, B, ng), CAM_THREADS, (CAM_STAGE + (size_t)C) * sizeof(double), st, a);
  TMF_LAUNCH_CHECK();
  const size_t smem = (size_t)C * sizeof(double);
  if (normalize && !upsample) launch_k(cam_map_kernel<true>, dim3(pl.nmap, B, ng), CAM_THREADS, smem, st, a);
  else launch_k(cam_map_kernel<false>, dim3(pl.nmap, B, ng), CAM_THREADS, smem, st, a);
  TMF_LAUNCH_CHECK();
  if (upsample) {
    if (normalize) {
      launch_k(cam_resample_kernel<true, false>, dim3(pl.nres, B, ng), CAM_THREADS, 0, st, a, 1);
      TMF_LAUNCH_CHECK();
    }
    launch_k(cam_resample_kernel<true, true>, dim3(pl.nres, B, ng), CAM_THREADS, 0, st, a, normalize);
    TMF_LAUNCH_CHECK();
  } else if (normalize) {
    launch_k(cam_resample_kernel<false, true>, dim3(pl.nmap, B, ng), CAM_THREADS, 0, st, a, 1);
    TMF_LAUNCH_CHECK();
  }
  return 0;
}

// Any low-resolution maps (the fusion transformer's token relevance, DESIGN section 3.8) through Grad-CAM's resampling pass:
// the same plan and the same cam_resample_kernel launches, so a map comes out with the bits tmf_gradcam gives it.
static size_t map_resample_bytes(int ng, int B, int d, int h, int w, int D, int H, int W, int normalize) {
  const CamPlan pl = cam_plan(ng, B, d, h, w, 4, D, H, W, 1, normalize);
  return normalize ? (size_t)ng * B * pl.nres * 2 * sizeof(float) : 0;
}

int64_t tmf_map_resample_workspace_bytes(int ng, int B, int d, int h, int w, int D, int H, int W, int normalize) {
  if (ng < 1 || ng > TMF_MAX_GROUPS || B < 1 || d < 1 || h < 1 || w < 1 || D < 1 || H < 1 || W < 1) return -1;
  return (int64_t)map_resample_bytes(ng, B, d, h, w, D, H, W, normalize);
}

int tmf_map_resample(int ng, const float* lo, float* const* out, int B, int d, int h, int w, int D, int H, int W, int normalize,
                     void* ws, size_t ws_bytes, void* stream) {
  TMF_CHECK_NG(ng);
  TMF_REQUIRE(lo != nullptr, "tmf_map_resample: lo is NULL");
  TMF_REQUIRE(B >= 1 && d >= 1 && h >= 1 && w >= 1 && D >= 1 && H >= 1 && W >= 1,
              "tmf_map_resample: bad extent B=%d %dx%dx%d -> %dx%dx%d", B, d, h, w, D, H, W);
  TMF_REQUIRE((int64_t)d * h * w < (1ll << 31) && (int64_t)D * H * W < (1ll << 31), "tmf_map_resample: extent too large");
  const size_t need = map_resample_bytes(ng, B, d, h, w, D, H, W, normalize);
  TMF_REQUIRE(!normalize || (ws != nullptr && ws_bytes >= need),
              "tmf_map_resample: workspace of %zu bytes < %zu (tmf_map_resample_workspace_bytes)", ws_bytes, need);
  const CamPlan pl = cam_plan(ng, B, d, h, w, 4, D, H, W, 1, normalize);
  CamArgs a{};
  if (!load_group(a.out, out, ng, true, "out")) return 1;
  a.lo = const_cast<float*>(lo);
  a.mm = normalize ? (float*)ws : nullptr;
  a.B = B; a.d = d; a.h = h; a.w = w; a.D = D; a.H = H; a.W = W;
  a.P = pl.P; a.nparts = pl.nres; a.nout = pl.nout;
  cudaStream_t st = (cudaStream_t)stream;
  if (normalize) {
    launch_k(cam_resample_kernel<true, false>, dim3(pl.nres, B, ng), CAM_THREADS, 0, st, a, 1);
    TMF_LAUNCH_CHECK();
  }
  launch_k(cam_resample_kernel<true, true>, dim3(pl.nres, B, ng), CAM_THREADS, 0, st, a, normalize);
  TMF_LAUNCH_CHECK();
  return 0;
}

}  // extern "C"

// mnet_ops.cu -- kernels of the MiSePyNet / Mnet baseline (reference models/MiSePyNet.py:5-163; BASELINE configs[4]), fp32,
// NCDHW-contiguous tensors exactly as the reference holds them (channel counts are 1..64: no tensor-core shapes here, the
// network is memory / CUDA-core bound -- SURVEY.md section 8f rank 3):
//   * "slice" convolutions Conv3d(Cin, 8, (1,1,k)) along the last axis (slice_cnn :5-38): forward, dgrad, wgrad;
//   * "spatial" convolutions Conv3d(Cin, Cout, (kh,kw,1), stride) on (N,C,X,Y,1) tensors (spatial_cnn :41-94): fwd / dgrad / wgrad;
//   * BatchNorm3d (train / eval) + ReLU on NC(S) tensors: statistics and backward sums as per-block partial ROWS in the same
//     double[TMF_STAT_ROWS][2C] format as the sNet path, so tmf_bn_finalize / tmf_bn_bwd_finalize are reused (deterministic);
//   * MaxPool3d((ph,pw,1)) with stride = kernel, floor mode, first-maximum gradient routing.
// Every reduction is a fixed-order two-stage sum: no floating-point atomics.
#include "common.cuh"

namespace tmf {
namespace mnet {

constexpr int LC_CO = 8;                    // output channels of every slice convolution

// ---------------------------------------------------------------------------------------------------------------
// slice convolution forward: x [N][Cin][P][L], w [8][Cin][k], b [8] -> y [N][8][P][Lo], Lo = L - k + 1
// one thread per (n, p, o): 8 outputs; weights in shared memory
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) line_conv_fwd_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                            const float* __restrict__ b, float* __restrict__ y, int N, int Cin,
                                                            int64_t P, int L, int k) {
  extern __shared__ float ws[];             // [Cin][k][8]
  for (int i = threadIdx.x; i < LC_CO * Cin * k; i += blockDim.x) {
    const int t = i % k, ci = (i / k) % Cin, co = i / (k * Cin);
    ws[(ci * k + t) * LC_CO + co] = w[i];
  }
  __syncthreads();
  const int Lo = L - k + 1;
  const int64_t total = (int64_t)N * P * Lo;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int o = (int)(idx % Lo);
    const int64_t p = (idx / Lo) % P;
    const int n = (int)(idx / ((int64_t)Lo * P));
    float acc[LC_CO];
#pragma unroll
    for (int c = 0; c < LC_CO; ++c) acc[c] = b[c];
    for (int ci = 0; ci < Cin; ++ci) {
      const float* xp = x + (((int64_t)n * Cin + ci) * P + p) * L + o;
      const float* wp = ws + (size_t)ci * k * LC_CO;
      for (int t = 0; t < k; ++t) {
        const float xv = __ldg(xp + t);
        const float4 w0 = *reinterpret_cast<const float4*>(wp + t * LC_CO);
        const float4 w1 = *reinterpret_cast<const float4*>(wp + t * LC_CO + 4);
        acc[0] = fmaf(xv, w0.x, acc[0]); acc[1] = fmaf(xv, w0.y, acc[1]); acc[2] = fmaf(xv, w0.z, acc[2]); acc[3] = fmaf(xv, w0.w, acc[3]);
        acc[4] = fmaf(xv, w1.x, acc[4]); acc[5] = fmaf(xv, w1.y, acc[5]); acc[6] = fmaf(xv, w1.z, acc[6]); acc[7] = fmaf(xv, w1.w, acc[7]);
      }
    }
#pragma unroll
    for (int c = 0; c < LC_CO; ++c) y[(((int64_t)n * LC_CO + c) * P + p) * Lo + o] = acc[c];
  }
}

// dgrad: dx[n][ci][p][i] = sum_co sum_t dy[n][co][p][i - t] * w[co][ci][t]   (0 <= i - t < Lo); one thread per (n, ci, p, i)
__global__ void __launch_bounds__(256) line_conv_dgrad_kernel(const float* __restrict__ dy, const float* __restrict__ w,
                                                              float* __restrict__ dx, int N, int Cin, int64_t P, int L, int k) {
  extern __shared__ float ws[];             // [8][Cin][k] as given
  for (int i = threadIdx.x; i < LC_CO * Cin * k; i += blockDim.x) ws[i] = w[i];
  __syncthreads();
  const int Lo = L - k + 1;
  const int64_t total = (int64_t)N * Cin * P * L;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int i = (int)(idx % L);
    const int64_t p = (idx / L) % P;
    const int ci = (int)((idx / ((int64_t)L * P)) % Cin);
    const int n = (int)(idx / ((int64_t)L * P * Cin));
    const int t0 = max(0, i - (Lo - 1)), t1 = min(k - 1, i);
    float acc = 0.f;
    for (int co = 0; co < LC_CO; ++co) {
      const float* dp = dy + (((int64_t)n * LC_CO + co) * P + p) * Lo;
      const float* wp = ws + (co * Cin + ci) * k;
      for (int t = t0; t <= t1; ++t) acc = fmaf(__ldg(dp + i - t), wp[t], acc);
    }
    dx[idx] = acc;
  }
}

// wgrad partials: block b handles lines (n, p) = b, b + grid, ...; thread j < 8*Cin*k owns weight (co, ci, t) and walks the
// lines' dy / x rows staged in shared memory; partial dw -> part[b][8*Cin*k], partial db -> part[b][8*Cin*k + co].
__global__ void __launch_bounds__(256) line_conv_wgrad_kernel(const float* __restrict__ dy, const float* __restrict__ x,
                                                              float* __restrict__ part, int N, int Cin, int64_t P, int L, int k) {
  extern __shared__ float sm[];
  const int Lo = L - k + 1;
  float* sdy = sm;                          // [8][Lo]
  float* sx = sm + LC_CO * Lo;              // [Cin][L]
  const int nw = LC_CO * Cin * k;
  const int per = (nw + blockDim.x - 1) / blockDim.x;        // weights per thread (<= 16: 8*8*55 = 3520 weights for slice_cnn(109))
  float acc[16];
  float accb = 0.f;
#pragma unroll
  for (int j = 0; j < 16; ++j) acc[j] = 0.f;
  const int64_t lines = (int64_t)N * P;
  for (int64_t line = blockIdx.x; line < lines; line += gridDim.x) {
    const int n = (int)(line / P);
    const int64_t p = line % P;
    __syncthreads();
    for (int i = threadIdx.x; i < LC_CO * Lo; i += blockDim.x) {
      const int co = i / Lo, o = i % Lo;
      sdy[i] = __ldg(dy + (((int64_t)n * LC_CO + co) * P + p) * Lo + o);
    }
    for (int i = threadIdx.x; i < Cin * L; i += blockDim.x) {
      const int ci = i / L, l = i % L;
      sx[i] = __ldg(x + (((int64_t)n * Cin + ci) * P + p) * L + l);
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const int wi = threadIdx.x + j * blockDim.x;
      if (j < per && wi < nw) {
        const int t = wi % k, ci = (wi / k) % Cin, co = wi / (k * Cin);
        const float* a = sdy + co * Lo;
        const float* bq = sx + ci * L + t;
        float s = 0.f;
        for (int o = 0; o < Lo; ++o) s = fmaf(a[o], bq[o], s);
        acc[j] += s;
      }
    }
    if (threadIdx.x < LC_CO) {
      float s = 0.f;
      for (int o = 0; o < Lo; ++o) s += sdy[threadIdx.x * Lo + o];
      accb += s;
    }
  }
  float* out = part + (size_t)blockIdx.x * (nw + LC_CO);
#pragma unroll
  for (int j = 0; j < 16; ++j) {
    const int wi = threadIdx.x + j * blockDim.x;
    if (j < per && wi < nw) out[wi] = acc[j];
  }
  if (threadIdx.x < LC_CO) out[nw + threadIdx.x] = accb;
}

// out[i] = sum over rows r < nrows of part[r][i]   (fixed order); first n0 entries -> a, the rest -> b
__global__ void reduce_rows_kernel(const float* __restrict__ part, int nrows, int n, int n0, float* __restrict__ a, float* __restrict__ b) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float s = 0.f;
  for (int r = 0; r < nrows; ++r) s += part[(size_t)r * n + i];
  if (i < n0) a[i] = s;
  else if (b != nullptr) b[i - n0] = s;
}

// ---------------------------------------------------------------------------------------------------------------
// spatial convolution on [N][Cin][X][Y] (the trailing unit axis dropped), kernel kh x kw, stride s, no padding
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) conv2d_fwd_kernel(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ b,
                                                         float* __restrict__ y, int N, int Cin, int X, int Y, int Cout, int kh, int kw,
                                                         int s, int Xo, int Yo) {
  const int64_t total = (int64_t)N * Cout * Xo * Yo;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int oy = (int)(idx % Yo), ox = (int)((idx / Yo) % Xo);
    const int co = (int)((idx / ((int64_t)Yo * Xo)) % Cout), n = (int)(idx / ((int64_t)Yo * Xo * Cout));
    float acc = b[co];
    for (int ci = 0; ci < Cin; ++ci) {
      const float* xp = x + (((int64_t)n * Cin + ci) * X + ox * s) * Y + oy * s;
      const float* wp = w + ((int64_t)co * Cin + ci) * kh * kw;
      for (int i = 0; i < kh; ++i)
        for (int j = 0; j < kw; ++j) acc = fmaf(__ldg(xp + i * Y + j), __ldg(wp + i * kw + j), acc);
    }
    y[idx] = acc;
  }
}

__global__ void __launch_bounds__(256) conv2d_dgrad_kernel(const float* __restrict__ dy, const float* __restrict__ w, float* __restrict__ dx,
                                                           int N, int Cin, int X, int Y, int Cout, int kh, int kw, int s, int Xo, int Yo) {
  const int64_t total = (int64_t)N * Cin * X * Y;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int iy = (int)(idx % Y), ix = (int)((idx / Y) % X);
    const int ci = (int)((idx / ((int64_t)Y * X)) % Cin), n = (int)(idx / ((int64_t)Y * X * Cin));
    float acc = 0.f;
    for (int i = ix % s; i < kh; i += s) {
      const int ox = (ix - i) / s;
      if (ix - i < 0 || ox >= Xo) continue;
      for (int j = iy % s; j < kw; j += s) {
        const int oy = (iy - j) / s;
        if (iy - j < 0 || oy >= Yo) continue;
        for (int co = 0; co < Cout; ++co)
          acc = fmaf(__ldg(dy + (((int64_t)n * Cout + co) * Xo + ox) * Yo + oy), __ldg(w + (((int64_t)co * Cin + ci) * kh + i) * kw + j), acc);
      }
    }
    dx[idx] = acc;
  }
}

// one warp per weight element (co, ci, i, j): lanes stride over (n, ox, oy), shuffle-tree sum (deterministic); db by the
// warps with ci == i == j == 0
__global__ void __launch_bounds__(256) conv2d_wgrad_kernel(const float* __restrict__ dy, const float* __restrict__ x, float* __restrict__ dw,
                                                           float* __restrict__ db, int N, int Cin, int X, int Y, int Cout, int kh, int kw,
                                                           int s, int Xo, int Yo) {
  const int lane = threadIdx.x & 31;
  const int64_t nwt = (int64_t)Cout * Cin * kh * kw;
  const int64_t wid = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  if (wid >= nwt) return;
  const int j = (int)(wid % kw), i = (int)((wid / kw) % kh);
  const int ci = (int)((wid / ((int64_t)kw * kh)) % Cin), co = (int)(wid / ((int64_t)kw * kh * Cin));
  const int64_t npos = (int64_t)N * Xo * Yo;
  float acc = 0.f, accb = 0.f;
  for (int64_t q = lane; q < npos; q += 32) {
    const int oy = (int)(q % Yo), ox = (int)((q / Yo) % Xo), n = (int)(q / ((int64_t)Yo * Xo));
    const float g = __ldg(dy + (((int64_t)n * Cout + co) * Xo + ox) * Yo + oy);
    acc = fmaf(g, __ldg(x + (((int64_t)n * Cin + ci) * X + ox * s + i) * Y + oy * s + j), acc);
    accb += g;
  }
  acc = warp_sum(acc);
  accb = warp_sum(accb);
  if (lane == 0) {
    dw[wid] = acc;
    if (db != nullptr && ci == 0 && i == 0 && j == 0) db[co] = accb;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// BatchNorm3d + ReLU on [N][C][S] fp32
// ---------------------------------------------------------------------------------------------------------------
// rows[blockIdx.x][c], rows[blockIdx.x][C + c] = partial sum / sum of squares of channel c = blockIdx.y
__global__ void __launch_bounds__(256) nchw_stats_kernel(const float* __restrict__ x, double* __restrict__ rows, int N, int C, int64_t S) {
  const int c = blockIdx.y;
  const int64_t total = (int64_t)N * S;
  double s1 = 0.0, s2 = 0.0;
  float a1 = 0.f, a2 = 0.f;
  int cnt = 0;
  for (int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; q < total; q += (int64_t)gridDim.x * blockDim.x) {
    const int n = (int)(q / S);
    const float v = __ldg(x + ((int64_t)n * C + c) * S + (q - (int64_t)n * S));
    a1 += v;
    a2 = fmaf(v, v, a2);
    if (++cnt == 64) { s1 += a1; s2 += a2; a1 = 0.f; a2 = 0.f; cnt = 0; }
  }
  s1 += a1; s2 += a2;
  __shared__ double r1[8], r2[8];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { s1 += __shfl_xor_sync(0xffffffffu, s1, o); s2 += __shfl_xor_sync(0xffffffffu, s2, o); }
  if ((threadIdx.x & 31) == 0) { r1[threadIdx.x >> 5] = s1; r2[threadIdx.x >> 5] = s2; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double t1 = 0.0, t2 = 0.0;
#pragma unroll
    for (int i = 0; i < 8; ++i) { t1 += r1[i]; t2 += r2[i]; }
    stat_row_store(rows, 2 * C, blockIdx.x, gridDim.x, c, t1);
    stat_row_store(rows, 2 * C, blockIdx.x, gridDim.x, C + c, t2);
  }
}

// out = relu(x * scale[c] + shift[c])
__global__ void __launch_bounds__(256) nchw_bn_relu_kernel(const float* __restrict__ x, const float* __restrict__ coef, float* __restrict__ out,
                                                           int C, int64_t S, int64_t total) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)((i / S) % C);
    out[i] = fmaxf(fmaf(__ldg(x + i), coef[c], coef[C + c]), 0.f);
  }
}

// rows: partial {sum dz, sum dz*xhat}, dz = dout * (z > 0), z = x*scale + shift, xhat = (x - mean) * invstd
__global__ void __launch_bounds__(256) nchw_bn_relu_bwd_reduce_kernel(const float* __restrict__ dout, const float* __restrict__ x,
                                                                      const float* __restrict__ coef, double* __restrict__ rows, int N,
                                                                      int C, int64_t S) {
  const int c = blockIdx.y;
  const float sc = coef[c], sh = coef[C + c], mu = coef[2 * C + c], is = coef[3 * C + c];
  const int64_t total = (int64_t)N * S;
  double s1 = 0.0, s2 = 0.0;
  float a1 = 0.f, a2 = 0.f;
  int cnt = 0;
  for (int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; q < total; q += (int64_t)gridDim.x * blockDim.x) {
    const int n = (int)(q / S);
    const int64_t off = ((int64_t)n * C + c) * S + (q - (int64_t)n * S);
    const float xv = __ldg(x + off);
    const float dz = fmaf(xv, sc, sh) > 0.f ? __ldg(dout + off) : 0.f;
    a1 += dz;
    a2 = fmaf(dz, (xv - mu) * is, a2);
    if (++cnt == 64) { s1 += a1; s2 += a2; a1 = 0.f; a2 = 0.f; cnt = 0; }
  }
  s1 += a1; s2 += a2;
  __shared__ double r1[8], r2[8];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { s1 += __shfl_xor_sync(0xffffffffu, s1, o); s2 += __shfl_xor_sync(0xffffffffu, s2, o); }
  if ((threadIdx.x & 31) == 0) { r1[threadIdx.x >> 5] = s1; r2[threadIdx.x >> 5] = s2; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double t1 = 0.0, t2 = 0.0;
#pragma unroll
    for (int i = 0; i < 8; ++i) { t1 += r1[i]; t2 += r2[i]; }
    stat_row_store(rows, 2 * C, blockIdx.x, gridDim.x, c, t1);
    stat_row_store(rows, 2 * C, blockIdx.x, gridDim.x, C + c, t2);
  }
}

// dx = scale * (dz - m1 - xhat * m2)   (bcoef = {m1[C], m2[C]}; zeros in eval mode)
__global__ void __launch_bounds__(256) nchw_bn_relu_bwd_apply_kernel(const float* __restrict__ dout, const float* __restrict__ x,
                                                                     const float* __restrict__ coef, const float* __restrict__ bcoef,
                                                                     float* __restrict__ dx, int C, int64_t S, int64_t total) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)((i / S) % C);
    const float sc = coef[c], sh = coef[C + c], mu = coef[2 * C + c], is = coef[3 * C + c];
    const float xv = __ldg(x + i);
    const float dz = fmaf(xv, sc, sh) > 0.f ? __ldg(dout + i) : 0.f;
    dx[i] = sc * (dz - bcoef[c] - (xv - mu) * is * bcoef[C + c]);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// MaxPool over (ph, pw) windows of [NC][X][Y], stride = kernel, floor mode; idx = argmax inside the window (first maximum)
// ---------------------------------------------------------------------------------------------------------------
__global__ void maxpool2d_fwd_kernel(const float* __restrict__ x, float* __restrict__ y, uint8_t* __restrict__ idx, int64_t NC, int X, int Y,
                                     int ph, int pw, int Xo, int Yo) {
  const int64_t total = NC * Xo * Yo;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int oy = (int)(i % Yo), ox = (int)((i / Yo) % Xo);
    const int64_t nc = i / ((int64_t)Yo * Xo);
    const float* xp = x + (nc * X + ox * ph) * Y + oy * pw;
    float best = -INFINITY;
    int bi = 0;
    for (int a = 0; a < ph; ++a)
      for (int b = 0; b < pw; ++b) {
        const float v = xp[a * Y + b];
        if (v > best || (v != v && best == best)) { best = v; bi = a * pw + b; }      // first maximum (NaN propagates like torch)
      }
    y[i] = best;
    idx[i] = (uint8_t)bi;
  }
}

__global__ void maxpool2d_bwd_kernel(const float* __restrict__ dy, const uint8_t* __restrict__ idx, float* __restrict__ dx, int64_t NC, int X,
                                     int Y, int ph, int pw, int Xo, int Yo) {
  const int64_t total = NC * X * Y;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int iy = (int)(i % Y), ix = (int)((i / Y) % X);
    const int64_t nc = i / ((int64_t)Y * X);
    const int ox = ix / ph, oy = iy / pw;
    float v = 0.f;
    if (ox < Xo && oy < Yo) {
      const int64_t o = (nc * Xo + ox) * Yo + oy;
      if (idx[o] == (ix - ox * ph) * pw + (iy - oy * pw)) v = dy[o];
    }
    dx[i] = v;
  }
}

static inline int grid_for(int64_t total, int cap = 148 * 16) {
  int64_t b = (total + 255) / 256;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (int)b;
}

}  // namespace mnet
}  // namespace tmf

using namespace tmf;
using namespace tmf::mnet;

extern "C" {

int tmf_line_conv_fwd(const float* x, const float* w, const float* b, float* y, int N, int Cin, int64_t P, int L, int k, void* stream) {
  TMF_REQUIRE(x && w && b && y && N > 0 && Cin >= 1 && Cin <= 8 && P > 0 && k >= 1 && k <= L, "line_conv_fwd: bad arguments");
  const size_t smem = sizeof(float) * LC_CO * Cin * k;
  TMF_REQUIRE(smem <= 48 * 1024, "line_conv_fwd: kernel too long");
  line_conv_fwd_kernel<<<grid_for((int64_t)N * P * (L - k + 1)), 256, smem, (cudaStream_t)stream>>>(x, w, b, y, N, Cin, P, L, k);
  TMF_LAUNCH_CHECK();
  return 0;
}

int tmf_line_conv_dgrad(const float* dy, const float* w, float* dx, int N, int Cin, int64_t P, int L, int k, void* stream) {
  TMF_REQUIRE(dy && w && dx && N > 0 && Cin >= 1 && Cin <= 8 && P > 0 && k >= 1 && k <= L, "line_conv_dgrad: bad arguments");
  const size_t smem = sizeof(float) * LC_CO * Cin * k;
  TMF_REQUIRE(smem <= 48 * 1024, "line_conv_dgrad: kernel too long");
  line_conv_dgrad_kernel<<<grid_for((int64_t)N * Cin * P * L), 256, smem, (cudaStream_t)stream>>>(dy, w, dx, N, Cin, P, L, k);
  TMF_LAUNCH_CHECK();
  return 0;
}

int64_t tmf_line_conv_wgrad_workspace_bytes(int Cin, int k) { return (int64_t)sizeof(float) * 592 * (LC_CO * Cin * k + LC_CO); }

int tmf_line_conv_wgrad(const float* dy, const float* x, float* dw, float* db, int N, int Cin, int64_t P, int L, int k, void* ws,
                        size_t ws_bytes, void* stream) {
  TMF_REQUIRE(dy && x && dw && N > 0 && Cin >= 1 && Cin <= 8 && P > 0 && k >= 1 && k <= L, "line_conv_wgrad: bad arguments");
  TMF_REQUIRE(LC_CO * Cin * k <= 16 * 256, "line_conv_wgrad: too many weights per output channel block");
  TMF_REQUIRE(ws != nullptr && (int64_t)ws_bytes >= tmf_line_conv_wgrad_workspace_bytes(Cin, k), "line_conv_wgrad: workspace too small");
  const int64_t lines = (int64_t)N * P;
  const int nb = (int)(lines < 592 ? lines : 592);
  const int nw = LC_CO * Cin * k;
  const size_t smem = sizeof(float) * ((size_t)LC_CO * (L - k + 1) + (size_t)Cin * L);
  TMF_REQUIRE(smem <= 48 * 1024, "line_conv_wgrad: line too long");
  cudaStream_t st = (cudaStream_t)stream;
  line_conv_wgrad_kernel<<<nb, 256, smem, st>>>(dy, x, (float*)ws, N, Cin, P, L, k);
  TMF_LAUNCH_CHECK();
  reduce_rows_kernel<<<ceil_div(nw + LC_CO, 128), 128, 0, st>>>((const float*)ws, nb, nw + LC_CO, nw, dw, db);
  TMF_LAUNCH_CHECK();
  return 0;
}

int tmf_conv2d_fwd(const float* x, const float* w, const float* b, float* y, int N, int Cin, int X, int Y, int Cout, int kh, int kw,
                   int stride, void* stream) {
  TMF_REQUIRE(x && w && b && y && N >= 1 && Cin >= 1 && Cout >= 1 && kh >= 1 && kw >= 1 && stride >= 1 && X >= kh && Y >= kw,
              "conv2d_fwd: bad arguments");
  const int Xo = (X - kh) / stride + 1, Yo = (Y - kw) / stride + 1;
  conv2d_fwd_kernel<<<grid_for((int64_t)N * Cout * Xo * Yo), 256, 0, (cudaStream_t)stream>>>(x, w, b, y, N, Cin, X, Y, Cout, kh, kw, stride, Xo, Yo);
  TMF_LAUNCH_CHECK();
  return 0;
}

int tmf_conv2d_dgrad(const float* dy, const float* w, float* dx, int N, int Cin, int X, int Y, int Cout, int kh, int kw, int stride,
                     void* stream) {
  TMF_REQUIRE(dy && w && dx && N >= 1 && Cin >= 1 && Cout >= 1 && kh >= 1 && kw >= 1 && stride >= 1 && X >= kh && Y >= kw,
              "conv2d_dgrad: bad arguments");
  const int Xo = (X - kh) / stride + 1, Yo = (Y - kw) / stride + 1;
  conv2d_dgrad_kernel<<<grid_for((int64_t)N * Cin * X * Y), 256, 0, (cudaStream_t)stream>>>(dy, w, dx, N, Cin, X, Y, Cout, kh, kw, stride, Xo, Yo);
  TMF_LAUNCH_CHECK();
  return 0;
}

int tmf_conv2d_wgrad(const float* dy, const float* x, float* dw, float* db, int N, int Cin, int X, int Y, int Cout, int kh, int kw,
                     int stride, void* stream) {
  TMF_REQUIRE(dy && x && dw && N >= 1 && Cin >= 1 && Cout >= 1 && kh >= 1 && kw >= 1 && stride >= 1 && X >= kh && Y >= kw,
              "conv2d_wgrad: bad arguments");
  const int Xo = (X - kh) / stride + 1, Yo = (Y - kw) / stride + 1;
  const int64_t nwt = (int64_t)Cout * Cin * kh * kw;
  conv2d_wgrad_kernel<<<ceil_div(nwt * 32, 256), 256, 0, (cudaStream_t)stream>>>(dy, x, dw, db, N, Cin, X, Y, Cout, kh, kw, stride, Xo, Yo);
  TMF_LAUNCH_CHECK();
  return 0;
}

int tmf_nchw_bn_stats(const float* x, double* rows, int N, int C, int64_t S, void* stream) {
  TMF_REQUIRE(x && rows && N > 0 && C > 0 && S > 0, "nchw_bn_stats: bad arguments");
  int bx = (int)(((int64_t)N * S + 256 * 8 - 1) / (256 * 8));
  if (bx > TMF_STAT_ROWS) bx = TMF_STAT_ROWS;
  if (bx < 1) bx = 1;
  nchw_stats_kernel<<<dim3(bx, C), 256, 0, (cudaStream_t)stream>>>(x, rows, N, C, S);
  TMF_LAUNCH_CHECK();
  return 0;
}

int tmf_nchw_bn_relu_fwd(const float* x, const float* coef, float* out, int N, int C, int64_t S, void* stream) {
  TMF_REQUIRE(x && coef && out, "nchw_bn_relu_fwd: NULL pointer");
  TMF_REQUIRE(N > 0 && C > 0 && S > 0, "nchw_bn_relu_fwd: empty tensor");
  const int64_t total = (int64_t)N * C * S;
  nchw_bn_relu_kernel<<<grid_for(total), 256, 0, (cudaStream_t)stream>>>(x, coef, out, C, S, total);
  TMF_LAUNCH_CHECK();
  return 0;
}

int tmf_nchw_bn_relu_bwd_reduce(const float* dout, const float* x, const float* coef, double* rows, int N, int C, int64_t S, void* stream) {
  TMF_REQUIRE(dout && x && coef && rows, "nchw_bn_relu_bwd_reduce: NULL pointer");
  TMF_REQUIRE(N > 0 && C > 0 && S > 0, "nchw_bn_relu_bwd_reduce: empty tensor");
  int bx = (int)(((int64_t)N * S + 256 * 8 - 1) / (256 * 8));
  if (bx > TMF_STAT_ROWS) bx = TMF_STAT_ROWS;
  if (bx < 1) bx = 1;
  nchw_bn_relu_bwd_reduce_kernel<<<dim3(bx, C), 256, 0, (cudaStream_t)stream>>>(dout, x, coef, rows, N, C, S);
  TMF_LAUNCH_CHECK();
  return 0;
}

int tmf_nchw_bn_relu_bwd_apply(const float* dout, const float* x, const float* coef, const float* bcoef, float* dx, int N, int C,
                               int64_t S, void* stream) {
  TMF_REQUIRE(dout && x && coef && bcoef && dx, "nchw_bn_relu_bwd_apply: NULL pointer");
  TMF_REQUIRE(N > 0 && C > 0 && S > 0, "nchw_bn_relu_bwd_apply: empty tensor");
  const int64_t total = (int64_t)N * C * S;
  nchw_bn_relu_bwd_apply_kernel<<<grid_for(total), 256, 0, (cudaStream_t)stream>>>(dout, x, coef, bcoef, dx, C, S, total);
  TMF_LAUNCH_CHECK();
  return 0;
}

int tmf_maxpool2d_fwd(const float* x, float* y, void* idx, int64_t NC, int X, int Y, int ph, int pw, void* stream) {
  TMF_REQUIRE(x && y && idx && ph >= 1 && pw >= 1 && ph * pw <= 255 && X >= ph && Y >= pw, "maxpool2d_fwd: bad arguments");
  const int Xo = X / ph, Yo = Y / pw;
  maxpool2d_fwd_kernel<<<grid_for(NC * Xo * Yo), 256, 0, (cudaStream_t)stream>>>(x, y, (uint8_t*)idx, NC, X, Y, ph, pw, Xo, Yo);
  TMF_LAUNCH_CHECK();
  return 0;
}

int tmf_maxpool2d_bwd(const float* dy, const void* idx, float* dx, int64_t NC, int X, int Y, int ph, int pw, void* stream) {
  TMF_REQUIRE(dy && idx && dx && ph >= 1 && pw >= 1 && ph * pw <= 255 && X >= ph && Y >= pw, "maxpool2d_bwd: bad arguments");
  const int Xo = X / ph, Yo = Y / pw;
  maxpool2d_bwd_kernel<<<grid_for(NC * X * Y), 256, 0, (cudaStream_t)stream>>>(dy, (const uint8_t*)idx, dx, NC, X, Y, ph, pw, Xo, Yo);
  TMF_LAUNCH_CHECK();
  return 0;
}

}  // extern "C"

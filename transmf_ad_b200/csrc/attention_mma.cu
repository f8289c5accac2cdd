// attention_mma.cu -- the cross-modal attention core on the tensor cores (mma.sync.m16n8k16, bf16 hi/lo split operands, fp32
// accumulation) for the SHORT token sequences of the fusion stack: Nq, Nk <= 160 (150 tokens per modality), dim_head 16/32/64.
// Reference: models/networks.py:166-174  (dots = q k^T * scale; attn = softmax(dots); out = attn v) and its autograd.
//
// Why not tcgen05: one (batch, head) is a 150 x 150 x 32 problem -- ten 16-row tiles, not one 128-row tile.  Why not the
// CUDA-core kernels of attention.cu: they are bound by shared-memory operand loads and one long dependent chain per CTA
// (17 us forward, 44 us backward per encoder call at B = 8 for 46 + 115 MFLOP).
//
// Arithmetic: every product x*y is xh*yh + xl*yh + xh*yl with xh = bf16(x), xl = bf16(x - xh): ~2^-16 relative per product,
// fp32 sums -- the scheme of the encoder GEMMs (enc_fused.cu); the softmax itself is fp32.
//
// Mapping (FlashAttention-style, but the whole key range fits in registers / shared memory):
//   forward   a warp owns 16 query rows and ALL keys: S = Q K^T as 20 n-tiles of accumulators (80 registers), row softmax
//             with two shuffles (a row lives in the four lanes of a quad), then the accumulator registers ARE the A fragments
//             of P for O = P V.  K / V of the (batch, head) are staged once per CTA as bf16 hi / lo planes [key][dh + 8]
//             (conflict-free ldmatrix; V is read with ldmatrix.trans).  CTA = 4 warps = 64 rows.
//   backward  ONE launch, two roles (blockIdx.z): "dq" CTAs (a warp = 16 query rows) walk the keys in chunks of 16:
//             S, dP = dO V^T -> P = exp(S*scale - lse), dS = P (dP - D) -> dq += dS K;  "dkv" CTAs (a warp = 16 keys) walk
//             the queries: S^T = K Q^T, dP^T = V dO^T -> dv += P^T dO, dk += dS^T Q.  D = rowsum(dO * O) is recomputed by
//             whoever needs it; no N x N tensor ever reaches HBM.
#include <math.h>
#include <stdlib.h>

#include "attn_args.cuh"
#include "common.cuh"

namespace tmf {
namespace amma {

constexpr int AM_WARPS = 4, AM_THREADS = 32 * AM_WARPS, AM_ROWS = 16 * AM_WARPS, AM_NMAX = 160;

__device__ __forceinline__ void mma_bf16(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void ldsm_x4(uint32_t (&r)[4], uint32_t saddr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(saddr));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t (&r)[4], uint32_t saddr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(saddr));
}
// hi / lo bf16 pairs of two fp32 values
__device__ __forceinline__ void split2(float a, float b, uint32_t& hi, uint32_t& lo) {
  hi = pack_bf16(a, b);
  lo = pack_bf16(a - bf16_lo(hi), b - bf16_hi(hi));
}
// the three MMAs of one split product  c += A B  (A = ah + al, B = bh + bl; the al*bl term is dropped)
__device__ __forceinline__ void mma3(float (&c)[4], const uint32_t (&ah)[4], const uint32_t (&al)[4], uint32_t bh0, uint32_t bh1,
                                     uint32_t bl0, uint32_t bl1) {
  mma_bf16(c, al, bh0, bh1);
  mma_bf16(c, ah, bl0, bl1);
  mma_bf16(c, ah, bh0, bh1);
}

template <int DH>
struct Lay {
  static constexpr int PITCH = (DH + 8) * 2;            // bytes per token row of a plane (16 B pad: conflict-free ldmatrix)
  static constexpr int PLANE = AM_NMAX * PITCH;         // one bf16 plane [160][DH + 8]
  static constexpr int KS = DH / 16;                    // k16 steps over the head dimension
  static constexpr int NT = DH / 8;                     // n8 tiles over the head dimension
};

// Stage `nvalid` token rows (DH floats at src + r * row_stride) as bf16 hi / lo planes; rows [nvalid, NR) are zero.  Loads are
// issued ten at a time per thread before any is used (dh = 32: the whole plane in ONE round trip).
template <int DH, int NR = AM_NMAX>
__device__ __forceinline__ void stage_split(uint8_t* hi, uint8_t* lo, const float* __restrict__ src, int64_t row_stride,
                                            int nvalid) {
  constexpr int C4 = DH / 4, TOTAL = NR * C4, U = 10;          // 160 * DH / 4 float4 = U * 128 threads * (DH / 32)
  for (int i0 = threadIdx.x; i0 < TOTAL; i0 += U * AM_THREADS) {
    float4 v[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int i = i0 + u * AM_THREADS;
      const int r = i / C4, c = i - r * C4;
      v[u] = (i < TOTAL && r < nvalid) ? __ldg(reinterpret_cast<const float4*>(src + (int64_t)r * row_stride) + c)
                                       : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int i = i0 + u * AM_THREADS;
      if (i < TOTAL) {
        const int r = i / C4, c = i - r * C4;
        uint2 h, l;
        split2(v[u].x, v[u].y, h.x, l.x);
        split2(v[u].z, v[u].w, h.y, l.y);
        *reinterpret_cast<uint2*>(hi + r * Lay<DH>::PITCH + 8 * c) = h;
        *reinterpret_cast<uint2*>(lo + r * Lay<DH>::PITCH + 8 * c) = l;
      }
    }
  }
}

// A fragments (hi / lo) of a 16 x DH fp32 tile in global memory: rows `base + g * stride`, `base + (g + 8) * stride`; rows
// >= nvalid read as zero.  fa[kk][0..3] keeps the fp32 values of fragment register 0..3's first element pair when KEEP.
template <int DH>
__device__ __forceinline__ void load_a_frags(const float* __restrict__ base, int64_t stride, int nvalid,
                                             uint32_t (&ah)[DH / 16][4], uint32_t (&al)[DH / 16][4]) {
  const int lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const bool ok0 = g < nvalid, ok1 = g + 8 < nvalid;
  const float* r0 = base + (int64_t)g * stride + 2 * t;
  const float* r1 = base + (int64_t)(g + 8) * stride + 2 * t;
  const float2 z = make_float2(0.f, 0.f);
#pragma unroll
  for (int kk = 0; kk < DH / 16; ++kk) {
    const float2 v0 = ok0 ? __ldg(reinterpret_cast<const float2*>(r0 + 16 * kk)) : z;
    const float2 v1 = ok1 ? __ldg(reinterpret_cast<const float2*>(r1 + 16 * kk)) : z;
    const float2 v2 = ok0 ? __ldg(reinterpret_cast<const float2*>(r0 + 16 * kk + 8)) : z;
    const float2 v3 = ok1 ? __ldg(reinterpret_cast<const float2*>(r1 + 16 * kk + 8)) : z;
    split2(v0.x, v0.y, ah[kk][0], al[kk][0]);
    split2(v1.x, v1.y, ah[kk][1], al[kk][1]);
    split2(v2.x, v2.y, ah[kk][2], al[kk][2]);
    split2(v3.x, v3.y, ah[kk][3], al[kk][3]);
  }
}

// lane-dependent byte offsets of the ldmatrix.x4 row addresses inside a plane
//   "nk": the plane is [n][k] (token = n): matrices (n-tile 0, k 0-7), (n-tile 0, k 8-15), (n-tile 1, k 0-7), (n-tile 1, k 8-15)
//   "kn": the plane is [k][n] (token = k), read with .trans: (k 0-7, n-tile 0), (k 8-15, n-tile 0), (k 0-7, n-tile 1), (k 8-15, n-tile 1)
// both give registers {b0, b1} of n-tile 0 then {b0, b1} of n-tile 1.
template <int DH>
__device__ __forceinline__ uint32_t off_nk(int lane) {
  return (uint32_t)(((lane & 7) + 8 * (lane >> 4)) * Lay<DH>::PITCH + 16 * ((lane >> 3) & 1));
}
template <int DH>
__device__ __forceinline__ uint32_t off_kn(int lane) {
  return (uint32_t)(((lane & 7) + 8 * ((lane >> 3) & 1)) * Lay<DH>::PITCH + 16 * (lane >> 4));
}

// c[2][4] += A (16 x DH, fragments) . B^T where B is the [n][k] plane pair at token row `tok0` (16 tokens = 2 n-tiles)
template <int DH>
__device__ __forceinline__ void mma_tile_nk(float (&c)[2][4], const uint32_t (&ah)[DH / 16][4], const uint32_t (&al)[DH / 16][4],
                                            uint32_t plane_hi, int tok0) {
  const uint32_t a0 = plane_hi + (uint32_t)tok0 * Lay<DH>::PITCH;
#pragma unroll
  for (int kk = 0; kk < DH / 16; ++kk) {
    uint32_t bh[4], bl[4];
    ldsm_x4(bh, a0 + kk * 32);
    ldsm_x4(bl, a0 + Lay<DH>::PLANE + kk * 32);
#pragma unroll
    for (int j = 0; j < 2; ++j) mma3(c[j], ah[kk], al[kk], bh[2 * j], bh[2 * j + 1], bl[2 * j], bl[2 * j + 1]);
  }
}
// acc[DH/8][4] += A (16 x 16 tokens, one k16 step: fragments ph / pl) . B where B is the [k][n] plane pair at token row tok0
template <int DH>
__device__ __forceinline__ void mma_tile_kn(float (&acc)[DH / 8][4], const uint32_t (&ph)[4], const uint32_t (&pl)[4],
                                            uint32_t plane_hi, int tok0) {
  const uint32_t a0 = plane_hi + (uint32_t)tok0 * Lay<DH>::PITCH;
#pragma unroll
  for (int n2 = 0; n2 < DH / 16; ++n2) {
    uint32_t bh[4], bl[4];
    ldsm_x4_t(bh, a0 + n2 * 32);
    ldsm_x4_t(bl, a0 + Lay<DH>::PLANE + n2 * 32);
#pragma unroll
    for (int j = 0; j < 2; ++j) mma3(acc[2 * n2 + j], ph, pl, bh[2 * j], bh[2 * j + 1], bl[2 * j], bl[2 * j + 1]);
  }
}

__device__ __forceinline__ float quad_max(float v) {
  v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 1));
  return fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 2));
}
__device__ __forceinline__ float quad_sum(float v) {
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  return v + __shfl_xor_sync(0xffffffffu, v, 2);
}

// =====================================================================================================================
// forward
// =====================================================================================================================
template <int DH>
__global__ void __launch_bounds__(AM_THREADS) attn_mma_fwd_kernel(AttnArgs p) {
  extern __shared__ __align__(16) uint8_t smraw[];
  using L = Lay<DH>;
  uint8_t* Kh = smraw;
  uint8_t* Vh = Kh + 2 * L::PLANE;
  const int inner = p.heads * DH;
  const int b = blockIdx.x / p.heads, h = blockIdx.x % p.heads;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const float* kvb = p.kv + (int64_t)b * p.Nk * 2 * inner + h * DH;
  stage_split<DH>(Kh, Kh + L::PLANE, kvb, 2 * inner, p.Nk);
  stage_split<DH>(Vh, Vh + L::PLANE, kvb + inner, 2 * inner, p.Nk);
  __syncthreads();
  const int r0 = blockIdx.y * AM_ROWS + warp * 16;
  if (r0 >= p.Nq) return;
  uint32_t qh[L::KS][4], ql[L::KS][4];
  load_a_frags<DH>(p.q + ((int64_t)b * p.Nq + r0) * inner + h * DH, inner, p.Nq - r0, qh, ql);

  const uint32_t kb = (uint32_t)__cvta_generic_to_shared(Kh) + off_nk<DH>(lane);
  const uint32_t vb = (uint32_t)__cvta_generic_to_shared(Vh) + off_kn<DH>(lane);
  float s[AM_NMAX / 8][4];
#pragma unroll
  for (int jp = 0; jp < AM_NMAX / 16; ++jp) {
    float c[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
    mma_tile_nk<DH>(c, qh, ql, kb, 16 * jp);
#pragma unroll
    for (int j = 0; j < 2; ++j)
#pragma unroll
      for (int e = 0; e < 4; ++e) s[2 * jp + j][e] = c[j][e];
  }
  // row softmax: rows g (elements 0, 1 of every n-tile) and g + 8 (elements 2, 3); a row is spread over the quad's 4 lanes
  float inv[2];
#pragma unroll
  for (int hf = 0; hf < 2; ++hf) {
    float mx = -INFINITY;
#pragma unroll
    for (int j = 0; j < AM_NMAX / 8; ++j)
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const float v = (8 * j + 2 * t + e < p.Nk) ? s[j][2 * hf + e] * p.scale : -INFINITY;
        s[j][2 * hf + e] = v;
        mx = fmaxf(mx, v);
      }
    mx = quad_max(mx);
    float sum = 0.f;
#pragma unroll
    for (int j = 0; j < AM_NMAX / 8; ++j)
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const float ex = __expf(s[j][2 * hf + e] - mx);        // exp(-inf) = 0 for the padding columns
        s[j][2 * hf + e] = ex;
        sum += ex;
      }
    sum = quad_sum(sum);
    inv[hf] = 1.f / sum;
    const int i = r0 + g + 8 * hf;
    if (t == 0 && i < p.Nq) p.lse[((int64_t)b * p.heads + h) * p.Nq + i] = mx + __logf(sum);
  }
  // O = P V: the accumulator registers of two neighbouring n-tiles are the A fragment of one k16 step
  float o[L::NT][4];
#pragma unroll
  for (int j = 0; j < L::NT; ++j) { o[j][0] = 0.f; o[j][1] = 0.f; o[j][2] = 0.f; o[j][3] = 0.f; }
#pragma unroll
  for (int kk = 0; kk < AM_NMAX / 16; ++kk) {
    uint32_t ph[4], pl[4];
    split2(s[2 * kk][0], s[2 * kk][1], ph[0], pl[0]);
    split2(s[2 * kk][2], s[2 * kk][3], ph[1], pl[1]);
    split2(s[2 * kk + 1][0], s[2 * kk + 1][1], ph[2], pl[2]);
    split2(s[2 * kk + 1][2], s[2 * kk + 1][3], ph[3], pl[3]);
    mma_tile_kn<DH>(o, ph, pl, vb, 16 * kk);
  }
#pragma unroll
  for (int hf = 0; hf < 2; ++hf) {
    const int i = r0 + g + 8 * hf;
    if (i < p.Nq) {
      float* orow = p.o + ((int64_t)b * p.Nq + i) * inner + h * DH + 2 * t;
#pragma unroll
      for (int j = 0; j < L::NT; ++j)
        *reinterpret_cast<float2*>(orow + 8 * j) = make_float2(o[j][2 * hf] * inv[hf], o[j][2 * hf + 1] * inv[hf]);
    }
  }
}

// =====================================================================================================================
// backward: blockIdx.z = 0 -> dq for 64 query rows, blockIdx.z = 1 -> dk, dv for 64 keys
// =====================================================================================================================
template <int DH>
__global__ void __launch_bounds__(AM_THREADS) attn_mma_bwd_kernel(AttnArgs p) {
  extern __shared__ __align__(16) uint8_t smraw[];
  using L = Lay<DH>;
  const int inner = p.heads * DH;
  const int b = blockIdx.x / p.heads, h = blockIdx.x % p.heads;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const float* kvb = p.kv + (int64_t)b * p.Nk * 2 * inner + h * DH;
  const float* qb = p.q + (int64_t)b * p.Nq * inner + h * DH;
  const float* gb = p.dout + (int64_t)b * p.Nq * inner + h * DH;
  const float* ob = p.out + (int64_t)b * p.Nq * inner + h * DH;
  const float* lseb = p.lse_in + ((int64_t)b * p.heads + h) * p.Nq;
  uint8_t* P0 = smraw;                         // dq role: K planes;  dkv role: Q planes
  uint8_t* P1 = P0 + 2 * L::PLANE;             // dq role: V planes;  dkv role: dO planes
  const uint32_t p0 = (uint32_t)__cvta_generic_to_shared(P0), p1 = (uint32_t)__cvta_generic_to_shared(P1);

  if (blockIdx.z == 0) {
    // ------------------------------------------------- dq -------------------------------------------------------------
    if ((int)blockIdx.y * AM_ROWS >= p.Nq) return;
    stage_split<DH>(P0, P0 + L::PLANE, kvb, 2 * inner, p.Nk);
    stage_split<DH>(P1, P1 + L::PLANE, kvb + inner, 2 * inner, p.Nk);
    __syncthreads();
    const int r0 = blockIdx.y * AM_ROWS + warp * 16;
    if (r0 >= p.Nq) return;
    const int nv = p.Nq - r0;
    uint32_t qh[L::KS][4], ql[L::KS][4], gh[L::KS][4], gl[L::KS][4];
    load_a_frags<DH>(qb + (int64_t)r0 * inner, inner, nv, qh, ql);
    load_a_frags<DH>(gb + (int64_t)r0 * inner, inner, nv, gh, gl);
    // D = rowsum(dO * O) and lse of rows g, g + 8
    float Dr[2], lr[2];
#pragma unroll
    for (int hf = 0; hf < 2; ++hf) {
      const int rr = g + 8 * hf;
      float acc = 0.f;
      if (rr < nv) {
        const float* gp = gb + (int64_t)(r0 + rr) * inner + 2 * t;
        const float* op = ob + (int64_t)(r0 + rr) * inner + 2 * t;
#pragma unroll
        for (int c = 0; c < DH / 8; ++c) {
          const float2 a = __ldg(reinterpret_cast<const float2*>(gp + 8 * c));
          const float2 o2 = __ldg(reinterpret_cast<const float2*>(op + 8 * c));
          acc = fmaf(a.x, o2.x, acc);
          acc = fmaf(a.y, o2.y, acc);
        }
      }
      Dr[hf] = quad_sum(acc);
      lr[hf] = (rr < nv) ? __ldg(lseb + r0 + rr) : 0.f;
    }
    const uint32_t kb_nk = p0 + off_nk<DH>(lane), kb_kn = p0 + off_kn<DH>(lane), vb_nk = p1 + off_nk<DH>(lane);
    float dq[L::NT][4];
#pragma unroll
    for (int j = 0; j < L::NT; ++j) { dq[j][0] = 0.f; dq[j][1] = 0.f; dq[j][2] = 0.f; dq[j][3] = 0.f; }
    const int nchunk = (p.Nk + 15) >> 4;
#pragma unroll 2
    for (int jp = 0; jp < nchunk; ++jp) {
      float s[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}}, dp[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
      mma_tile_nk<DH>(s, qh, ql, kb_nk, 16 * jp);
      mma_tile_nk<DH>(dp, gh, gl, vb_nk, 16 * jp);
      float ds[2][4];
#pragma unroll
      for (int j = 0; j < 2; ++j)
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int col = 16 * jp + 8 * j + 2 * t + (e & 1), hf = e >> 1;
          const float pij = (col < p.Nk) ? __expf(s[j][e] * p.scale - lr[hf]) : 0.f;
          ds[j][e] = pij * (dp[j][e] - Dr[hf]);
        }
      uint32_t ah[4], al[4];
      split2(ds[0][0], ds[0][1], ah[0], al[0]);
      split2(ds[0][2], ds[0][3], ah[1], al[1]);
      split2(ds[1][0], ds[1][1], ah[2], al[2]);
      split2(ds[1][2], ds[1][3], ah[3], al[3]);
      mma_tile_kn<DH>(dq, ah, al, kb_kn, 16 * jp);
    }
#pragma unroll
    for (int hf = 0; hf < 2; ++hf) {
      const int rr = g + 8 * hf;
      if (rr < nv) {
        float* drow = p.dq + ((int64_t)b * p.Nq + r0 + rr) * inner + h * DH + 2 * t;
#pragma unroll
        for (int j = 0; j < L::NT; ++j)
          *reinterpret_cast<float2*>(drow + 8 * j) = make_float2(dq[j][2 * hf] * p.scale, dq[j][2 * hf + 1] * p.scale);
      }
    }
  } else {
    // ------------------------------------------------- dk, dv ---------------------------------------------------------
    if ((int)blockIdx.y * AM_ROWS >= p.Nk) return;
    float* lses = reinterpret_cast<float*>(P1 + 2 * L::PLANE);
    float* Ds = lses + AM_NMAX;
    stage_split<DH>(P0, P0 + L::PLANE, qb, inner, p.Nq);
    stage_split<DH>(P1, P1 + L::PLANE, gb, inner, p.Nq);
    // lse and D = rowsum(dO * O) per query: DH / 4 consecutive lanes share a row
    {
      constexpr int C4 = DH / 4;
      for (int i0 = threadIdx.x; i0 < AM_NMAX * C4; i0 += AM_THREADS) {
        const int r = i0 / C4, c = i0 - r * C4;
        float acc = 0.f;
        if (r < p.Nq) {
          const float4 a = __ldg(reinterpret_cast<const float4*>(gb + (int64_t)r * inner) + c);
          const float4 o4 = __ldg(reinterpret_cast<const float4*>(ob + (int64_t)r * inner) + c);
          acc = a.x * o4.x + a.y * o4.y + a.z * o4.z + a.w * o4.w;
        }
#pragma unroll
        for (int off = C4 / 2; off >= 1; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
        if (c == 0) {
          Ds[r] = acc;
          lses[r] = (r < p.Nq) ? __ldg(lseb + r) : 0.f;
        }
      }
    }
    __syncthreads();
    const int j0 = blockIdx.y * AM_ROWS + warp * 16;
    if (j0 >= p.Nk) return;
    const int nv = p.Nk - j0;
    uint32_t kh[L::KS][4], kl[L::KS][4], vh[L::KS][4], vl[L::KS][4];
    load_a_frags<DH>(kvb + (int64_t)j0 * 2 * inner, 2 * inner, nv, kh, kl);
    load_a_frags<DH>(kvb + inner + (int64_t)j0 * 2 * inner, 2 * inner, nv, vh, vl);
    const uint32_t qb_nk = p0 + off_nk<DH>(lane), qb_kn = p0 + off_kn<DH>(lane);
    const uint32_t gb_nk = p1 + off_nk<DH>(lane), gb_kn = p1 + off_kn<DH>(lane);
    float dk[L::NT][4], dv[L::NT][4];
#pragma unroll
    for (int j = 0; j < L::NT; ++j) {
      dk[j][0] = 0.f; dk[j][1] = 0.f; dk[j][2] = 0.f; dk[j][3] = 0.f;
      dv[j][0] = 0.f; dv[j][1] = 0.f; dv[j][2] = 0.f; dv[j][3] = 0.f;
    }
    const int nchunk = (p.Nq + 15) >> 4;
#pragma unroll 2
    for (int ip = 0; ip < nchunk; ++ip) {
      float st[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}}, dpt[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
      mma_tile_nk<DH>(st, kh, kl, qb_nk, 16 * ip);          // S^T = K Q^T
      mma_tile_nk<DH>(dpt, vh, vl, gb_nk, 16 * ip);         // dP^T = V dO^T
      float pt[2][4], dst[2][4];
#pragma unroll
      for (int j = 0; j < 2; ++j)
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int qi = 16 * ip + 8 * j + 2 * t + (e & 1);           // column = query
          const float pij = (qi < p.Nq) ? __expf(st[j][e] * p.scale - lses[qi]) : 0.f;
          pt[j][e] = pij;
          dst[j][e] = pij * (dpt[j][e] - Ds[qi]);
        }
      uint32_t ah[4], al[4];
      split2(pt[0][0], pt[0][1], ah[0], al[0]);
      split2(pt[0][2], pt[0][3], ah[1], al[1]);
      split2(pt[1][0], pt[1][1], ah[2], al[2]);
      split2(pt[1][2], pt[1][3], ah[3], al[3]);
      mma_tile_kn<DH>(dv, ah, al, gb_kn, 16 * ip);          // dv += P^T dO
      split2(dst[0][0], dst[0][1], ah[0], al[0]);
      split2(dst[0][2], dst[0][3], ah[1], al[1]);
      split2(dst[1][0], dst[1][1], ah[2], al[2]);
      split2(dst[1][2], dst[1][3], ah[3], al[3]);
      mma_tile_kn<DH>(dk, ah, al, qb_kn, 16 * ip);          // dk += dS^T Q
    }
#pragma unroll
    for (int hf = 0; hf < 2; ++hf) {
      const int rr = g + 8 * hf;
      if (rr < nv) {
        float* drow = p.dkv + ((int64_t)b * p.Nk + j0 + rr) * 2 * inner + h * DH + 2 * t;
#pragma unroll
        for (int j = 0; j < L::NT; ++j) {
          *reinterpret_cast<float2*>(drow + 8 * j) = make_float2(dk[j][2 * hf] * p.scale, dk[j][2 * hf + 1] * p.scale);
          *reinterpret_cast<float2*>(drow + inner + 8 * j) = make_float2(dv[j][2 * hf], dv[j][2 * hf + 1]);
        }
      }
    }
  }
}

// =====================================================================================================================
// attention maps (DESIGN section 3.8): the per-head product A_h B_h^T that the kernels above keep in registers, written out.
//   mode 0 ("probs"): A = q, B = k  ->  s = dots = scale * q_h k_h^T,  p = attn = exp(dots - lse)
//   mode 1 ("grad"):  A = dO, B = v ->  s = dattn = dO_h v_h^T          (the exact dL/dattn of out = attn v)
// Both [B, heads, Nq, Nk] fp32.  A CTA = one (batch, head), 64 query rows, one 64-key tile (blockIdx.z): the key range is
// tiled, so Nk has no envelope (and Nk = 150 gives three times the CTAs of the forward).  The product is the forward's (same fragments, same k16 order, fp32 accumulation), so
// dots carries the bits of the forward's scaled scores and attn those of the P the backward recomputes.  Every element is
// written once by one thread: no atomics.
// =====================================================================================================================
constexpr int SC_KEYS = 64;                                     // keys per CTA
struct ScoreArgs {
  const float* a; const float* kv; const float* lse;
  float* s; float* p;
  int Nq, Nk, heads, mode;
  float scale;
};

template <int DH>
__global__ void __launch_bounds__(AM_THREADS) attn_scores_kernel(ScoreArgs p) {
  extern __shared__ __align__(16) uint8_t smraw[];
  using L = Lay<DH>;
  const int inner = p.heads * DH;
  const int b = blockIdx.x / p.heads, h = blockIdx.x % p.heads;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int k0 = blockIdx.z * SC_KEYS, nk = min(SC_KEYS, p.Nk - k0);
  const float* bsrc = p.kv + ((int64_t)b * p.Nk + k0) * 2 * inner + (p.mode == 0 ? 0 : inner) + h * DH;
  stage_split<DH, SC_KEYS>(smraw, smraw + L::PLANE, bsrc, 2 * inner, nk);
  __syncthreads();
  const int r0 = blockIdx.y * AM_ROWS + warp * 16;
  if (r0 >= p.Nq) return;
  uint32_t ah[L::KS][4], al[L::KS][4];
  load_a_frags<DH>(p.a + ((int64_t)b * p.Nq + r0) * inner + h * DH, inner, p.Nq - r0, ah, al);
  float lr[2] = {0.f, 0.f};
  if (p.mode == 0) {
#pragma unroll
    for (int hf = 0; hf < 2; ++hf) {
      const int i = r0 + g + 8 * hf;
      lr[hf] = (i < p.Nq) ? __ldg(p.lse + (int64_t)blockIdx.x * p.Nq + i) : 0.f;
    }
  }
  const uint32_t kb = (uint32_t)__cvta_generic_to_shared(smraw) + off_nk<DH>(lane);
  const int64_t base = (int64_t)blockIdx.x * p.Nq * p.Nk;       // (b * heads + h) * Nq * Nk
  const bool pairs = (p.Nk & 1) == 0;                            // rows start 8-byte aligned: float2 stores
  const int nchunk = (nk + 15) >> 4;
  for (int jp = 0; jp < nchunk; ++jp) {
    float c[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
    mma_tile_nk<DH>(c, ah, al, kb, 16 * jp);
#pragma unroll
    for (int j = 0; j < 2; ++j)
#pragma unroll
      for (int hf = 0; hf < 2; ++hf) {
        const int i = r0 + g + 8 * hf, col = k0 + 16 * jp + 8 * j + 2 * t;
        if (i >= p.Nq || col >= p.Nk) continue;
        float v0 = c[j][2 * hf], v1 = c[j][2 * hf + 1];
        const int64_t o = base + (int64_t)i * p.Nk + col;
        const bool two = col + 1 < p.Nk;
        if (p.mode == 0) {
          v0 *= p.scale;
          v1 *= p.scale;
          const float e0 = __expf(v0 - lr[hf]), e1 = __expf(v1 - lr[hf]);
          if (pairs && two) {
            *reinterpret_cast<float2*>(p.p + o) = make_float2(e0, e1);
          } else {
            p.p[o] = e0;
            if (two) p.p[o + 1] = e1;
          }
        }
        if (pairs && two) {
          *reinterpret_cast<float2*>(p.s + o) = make_float2(v0, v1);
        } else {
          p.s[o] = v0;
          if (two) p.s[o + 1] = v1;
        }
      }
  }
}

template <int DH>
static int launch_scores(const ScoreArgs& p, int B, cudaStream_t st) {
  const size_t smem = 2 * (size_t)Lay<DH>::PLANE;                // one hi / lo plane pair (rows >= SC_KEYS unused)
  dim3 grid(B * p.heads, ceil_div(p.Nq, AM_ROWS), ceil_div(p.Nk, SC_KEYS));
  launch_k(attn_scores_kernel<DH>, grid, AM_THREADS, smem, st, p);
  TMF_LAUNCH_CHECK();
  return 0;
}

// M[b,i,j] = (1/heads) sum_h w,  w = attn (dattn == NULL) or max(attn * dattn, 0);  r[b,j] (+)= (1/Nq) sum_i M[b,i,j].
// A block = 32 key columns of one sample (coalesced rows) x 8 row slices; heads, rows of a slice and the slices are added
// in index order.
constexpr int RV_COLS = 32, RV_SLICES = 8;
__global__ void __launch_bounds__(RV_COLS * RV_SLICES) attn_relevance_kernel(const float* __restrict__ attn,
                                                                           const float* __restrict__ dattn, float* M, float* r,
                                                                           int heads, int Nq, int Nk, int accumulate) {
  __shared__ float part[RV_SLICES][RV_COLS];
  const int b = blockIdx.y, cx = threadIdx.x % RV_COLS, sl = threadIdx.x / RV_COLS;
  const int j = blockIdx.x * RV_COLS + cx;
  float acc = 0.f;
  if (j < Nk) {
    const int64_t hstride = (int64_t)Nq * Nk;
    for (int i = sl; i < Nq; i += RV_SLICES) {
      const int64_t o = ((int64_t)b * heads * Nq + i) * Nk + j;
      float m = 0.f;
      for (int hh = 0; hh < heads; ++hh) {
        float w = __ldg(attn + o + hh * hstride);
        if (dattn != nullptr) w = fmaxf(w * __ldg(dattn + o + hh * hstride), 0.f);
        m += w;
      }
      m /= (float)heads;
      if (M != nullptr) M[((int64_t)b * Nq + i) * Nk + j] = m;
      acc += m;
    }
  }
  part[sl][cx] = acc;
  __syncthreads();
  if (sl == 0 && j < Nk) {
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < RV_SLICES; ++k) s += part[k][cx];
    s /= (float)Nq;
    float* dst = r + (int64_t)b * Nk + j;
    *dst = accumulate ? *dst + s : s;
  }
}

static int impl_choice() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("TMF_ATTN_IMPL");            // 0: row-per-warp kernels, 1: register-tiled CUDA-core kernels, 2: mma.sync
    v = (e == nullptr) ? 2 : atoi(e);
  }
  return v;
}

template <int DH>
static int launch_fwd(const AttnArgs& p, cudaStream_t st) {
  const size_t smem = 4 * (size_t)Lay<DH>::PLANE;
  static bool attr_done = false;
  if (!attr_done && smem > 48 * 1024) {
    TMF_CUDA(cudaFuncSetAttribute(attn_mma_fwd_kernel<DH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_done = true;
  }
  dim3 grid(p.B * p.heads, ceil_div(p.Nq, AM_ROWS), 1);
  launch_k(attn_mma_fwd_kernel<DH>, grid, AM_THREADS, smem, st, p);
  TMF_LAUNCH_CHECK();
  return 0;
}
template <int DH>
static int launch_bwd(const AttnArgs& p, cudaStream_t st) {
  const size_t smem = 4 * (size_t)Lay<DH>::PLANE + 2 * AM_NMAX * sizeof(float);
  static bool attr_done = false;
  if (!attr_done && smem > 48 * 1024) {
    TMF_CUDA(cudaFuncSetAttribute(attn_mma_bwd_kernel<DH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_done = true;
  }
  const int gy = ceil_div(p.Nq > p.Nk ? p.Nq : p.Nk, AM_ROWS);
  dim3 grid(p.B * p.heads, gy, 2);
  launch_k(attn_mma_bwd_kernel<DH>, grid, AM_THREADS, smem, st, p);
  TMF_LAUNCH_CHECK();
  return 0;
}

}  // namespace amma

// return 0 on success, -1 if the shape is outside the envelope (the caller falls back to attention.cu / fusion_ops.cu)
int attn_mma_fwd(const AttnArgs& p, cudaStream_t st) {
  if (amma::impl_choice() < 2 || p.Nk > amma::AM_NMAX || p.Nk < 1 || p.Nq < 1) return -1;
  if ((p.heads * p.dh) % 4 != 0) return -1;
  if (p.dh == 32) return amma::launch_fwd<32>(p, st);
  if (p.dh == 16) return amma::launch_fwd<16>(p, st);
  if (p.dh == 64) return amma::launch_fwd<64>(p, st);
  return -1;
}
int attn_mma_bwd(const AttnArgs& p, cudaStream_t st) {
  if (amma::impl_choice() < 2 || p.Nk > amma::AM_NMAX || p.Nq > amma::AM_NMAX || p.Nk < 1 || p.Nq < 1) return -1;
  if ((p.heads * p.dh) % 4 != 0) return -1;
  if (p.dh == 32) return amma::launch_bwd<32>(p, st);
  if (p.dh == 16) return amma::launch_bwd<16>(p, st);
  if (p.dh == 64) return amma::launch_bwd<64>(p, st);
  return -1;
}

}  // namespace tmf

extern "C" int tmf_attn_impl_default(void) { return tmf::amma::impl_choice(); }

extern "C" int tmf_attn_scores(int mode, const float* a, const float* kv, const float* lse, float* s, float* p, int B, int Nq,
                               int Nk, int heads, int dh, float scale, void* stream) {
  using namespace tmf;
  TMF_REQUIRE(mode == 0 || mode == 1, "tmf_attn_scores: mode must be 0 (probs) or 1 (grad); got %d", mode);
  TMF_REQUIRE(dh == 16 || dh == 32 || dh == 64, "tmf_attn_scores: dim_head must be 16, 32 or 64 (got %d)", dh);
  TMF_REQUIRE(B >= 1 && Nq >= 1 && Nk >= 1 && heads >= 1, "tmf_attn_scores: bad shape B=%d Nq=%d Nk=%d heads=%d", B, Nq, Nk,
              heads);
  TMF_REQUIRE((int64_t)B * heads * Nq * Nk < (1ll << 40), "tmf_attn_scores: problem too large");
  TMF_REQUIRE(a != nullptr && kv != nullptr && s != nullptr && (mode == 1 || (lse != nullptr && p != nullptr)),
              "tmf_attn_scores: missing operand (mode %d needs a, kv, s%s)", mode, mode == 0 ? ", lse, p" : "");
  TMF_REQUIRE(((uintptr_t)a & 15) == 0 && ((uintptr_t)kv & 15) == 0 && ((uintptr_t)s & 7) == 0 && ((uintptr_t)p & 7) == 0,
              "tmf_attn_scores: a / kv must be 16-byte and s / p 8-byte aligned");
  amma::ScoreArgs sa{};
  sa.a = a; sa.kv = kv; sa.lse = lse; sa.s = s; sa.p = p;
  sa.Nq = Nq; sa.Nk = Nk; sa.heads = heads; sa.mode = mode; sa.scale = scale;
  cudaStream_t st = (cudaStream_t)stream;
  if (dh == 32) return amma::launch_scores<32>(sa, B, st);
  if (dh == 16) return amma::launch_scores<16>(sa, B, st);
  return amma::launch_scores<64>(sa, B, st);
}

extern "C" int tmf_attn_relevance(const float* attn, const float* dattn, float* M, float* r, int B, int heads, int Nq, int Nk,
                                  int accumulate, void* stream) {
  using namespace tmf;
  TMF_REQUIRE(B >= 1 && heads >= 1 && Nq >= 1 && Nk >= 1, "tmf_attn_relevance: bad shape B=%d heads=%d Nq=%d Nk=%d", B, heads,
              Nq, Nk);
  TMF_REQUIRE(attn != nullptr && r != nullptr, "tmf_attn_relevance: attn and r are required");
  dim3 grid(ceil_div(Nk, amma::RV_COLS), B);
  launch_k(amma::attn_relevance_kernel, grid, amma::RV_COLS * amma::RV_SLICES, 0, (cudaStream_t)stream, attn, dattn, M, r,
           heads, Nq, Nk, accumulate);
  TMF_LAUNCH_CHECK();
  return 0;
}

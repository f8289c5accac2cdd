// enc_fused.cu -- one Transformer(depth=1) encoder of the cross-modal fusion stack (reference models/networks.py:114-175,
// 215-230, as driven by CrossTransformer_MOD_AVG :272-281) in 3 forward and 5 backward launches instead of ~30:
//
//   forward   F1  enc_proj_fwd     x rows:   h1 = LN1(x);  q = h1 Wq^T          ctx rows:  kv = ctx Wkv^T
//             F2  (attention.cu)   o = softmax(q k^T scale) v
//             F3  enc_chain_fwd    a = o Wo^T + bo + x;  h2 = LN2(a);  p = h2 W1^T + b1;  f = GELU(p);
//                                  g = f W2^T + b2 + a;  y = LNf(g) (+ x: the caller's outer residual)
//   backward  R1  enc_chain_bwd    dy -> dg (LNf) -> df = dg W2 -> dp = df GELU'(p) -> dh2 = dp W1 -> da = dg + LN2'(dh2)
//                                  -> do = da Wo;  dxp = da (+ dy);  LN parameter gradients
//             R2  (attention.cu)   do -> dq, dkv
//             R3  enc_proj_bwd     x rows: dx = dxp + LN1'(dq Wq);  ctx rows: dctx = dkv Wkv;  LN1 parameter gradients
//             R4  enc_wgrad        dWq, dWkv, dWo, dW1, dW2 (+ bo, b1, b2 gradients): five token-reductions in one launch
//
// Every kernel is a chain of small GEMMs on a PANEL of 16 token rows held in shared memory, so the row-local work
// (LayerNorm, bias, GELU, residuals) rides in the GEMM prologues / epilogues and the intermediate tensors never make a
// round trip through launches.  The GEMMs run on the tensor cores with mma.sync.m16n8k8 TF32 and the 3-pass split
//   x*w ~= xl*wh + xh*wl + xh*wh      (xh = tf32(x), xl = tf32(x - xh); dropped term ~2^-22 relative)
// which keeps fp32-level accuracy (the reference's nn.Linear is fp32; measured <= 2e-6 relative against an fp32 CPU
// GEMM) -- tcgen05 needs 128-row tiles, and 1200 tokens are 75 panels of 16 rows but only 10 tiles of 128.
// Weights stream through a 3-stage cp.async ring in [128 x 32] tiles; all weight-side reductions over tokens are
// split and meet in the caller's scratch buffer, the last block adding the partials in index order (deterministic).
#include <math.h>

#include "common.cuh"

namespace tmf {
namespace enc {

constexpr int THREADS = 256;
constexpr int PR = 16;                       // panel rows
constexpr int WT_FLOATS = 5120;              // one weight stage (20480 B): fp32 [128][32+4] (B_NK) / [32][128+8] (B_KN), or the bf16
                                             // hi + lo tiles [2][128][32+8] (B_NK) / [2][32][128+8] (B_KN) of the split-weight path
constexpr int NSTAGE = 4;
constexpr int LD128 = 132;                   // panel pitch for 128 columns (== 4 mod 32: conflict-free A fragments)

enum { B_NK = 0, B_KN = 1 };                 // weight tile is W[n][k] (forward) or W[k][n] (dgrad / wgrad operand)

__device__ __forceinline__ void cp_async16(float* smem_dst, const float* gsrc, bool valid) {
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
  const int n = valid ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(gsrc), "r"(n) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// hi = x with the 13 low mantissa bits cleared (what the tensor core reads of an fp32 register anyway), lo = x - hi
// (exact).  One LOP + one FADD per element: cvt.rna.tf32 runs on the quarter-rate conversion pipe and, at 16 conversions
// per warp and k-step, cost more than the MMAs (measured: 46 us -> see profiles/r2_encoder.md).  lo carries up to 13
// significant bits of which the tensor core keeps 11: the result is good to ~2^-22 relative, the size of the dropped
// lo*lo term.
__device__ __forceinline__ void split_tf32(float x, uint32_t& hi, uint32_t& lo) {
  hi = __float_as_uint(x) & 0xffffe000u;
  lo = __float_as_uint(x - __uint_as_float(hi));
}
__device__ __forceinline__ void mma_tf32(float (&c)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
  asm volatile(
      "mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}

// erf by Abramowitz & Stegun 7.1.26 (|error| <= 1.5e-7, i.e. fp32 rounding level; 14 instructions against libdevice erff's
// 30): the GELU epilogue of the W1 GEMM was 10 k of the 45 k cycles of enc_chain_fwd_kernel (TMF_ENC_PROF).
__device__ __forceinline__ float erf_fast(float x) {
  const float ax = fabsf(x);
  const float t = __fdividef(1.f, fmaf(0.3275911f, ax, 1.f));
  float p = fmaf(1.061405429f, t, -1.453152027f);
  p = fmaf(p, t, 1.421413741f);
  p = fmaf(p, t, -0.284496736f);
  p = fmaf(p, t, 0.254829592f);
  p *= t;
  return copysignf(fmaf(-p, __expf(-ax * ax), 1.f), x);
}
__device__ __forceinline__ float gelu_exact(float x) { return 0.5f * x * (1.f + erf_fast(x * 0.70710678118654752440f)); }
__device__ __forceinline__ float gelu_grad(float x) {
  const float cdf = 0.5f * (1.f + erf_fast(x * 0.70710678118654752440f));
  const float pdf = 0.39894228040143267794f * __expf(-0.5f * x * x);
  return cdf + x * pdf;
}

// One weight stage is [128][32+4] floats (B_NK: rows n0..n0+127 of W, columns k0..k0+31 -> Ws[r*36 + c]) or [32][128+8]
// (B_KN: rows k0..k0+31 of W, rows >= kvalid read as zero, columns n0..n0+127 -> Ws[r*136 + c]); 1024 16-byte chunks, chunk
// c = thread + TH * u.  The per-thread source pointer / destination offset of u = 0 are computed once per GEMM and the stages
// are issued in order, so a stage costs one pointer update plus the cp.async themselves (the address arithmetic of the
// straightforward version was 11 % of all instructions of enc_chain_fwd_kernel, profiles/r2_encoder.md).
template <int MODE, int TH>
struct WeightStager {
  const float* src;          // W + r0 * ldw + 4 q           (u = 0 chunk of stage 0)
  uint32_t dst;              // shared address of chunk u = 0 inside stage slot 0
  size_t ustride;            // floats between a thread's consecutive chunks
  int ldw, nk, kvalid, r0;
  int nb, kc, slot;          // next stage to issue
  __device__ __forceinline__ WeightStager(float* wstage, const float* W, int ldw_, int nk_, int kvalid_)
      : ldw(ldw_), nk(nk_), kvalid(kvalid_), nb(0), kc(0), slot(0) {
    if (MODE == B_NK) {
      r0 = threadIdx.x >> 3;
      const int q = threadIdx.x & 7;
      src = W + (size_t)r0 * ldw + 4 * q;
      dst = (uint32_t)__cvta_generic_to_shared(wstage + r0 * 36 + 4 * q);
      ustride = (size_t)(TH >> 3) * ldw;
    } else {
      r0 = threadIdx.x >> 5;
      const int q = threadIdx.x & 31;
      src = W + (size_t)r0 * ldw + 4 * q;
      dst = (uint32_t)__cvta_generic_to_shared(wstage + r0 * 136 + 4 * q);
      ustride = (size_t)(TH >> 5) * ldw;
    }
  }
  __device__ __forceinline__ void issue() {
    const uint32_t d = dst + (uint32_t)slot * (WT_FLOATS * 4);
    if (MODE == B_NK) {
      const float* g = src + (size_t)nb * 128 * ldw + kc * 32;
#pragma unroll
      for (int u = 0; u < 1024 / TH; ++u)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d + (uint32_t)u * ((TH >> 3) * 36 * 4)), "l"(g + u * ustride) : "memory");
    } else {
      const float* g = src + (size_t)kc * 32 * ldw + nb * 128;
#pragma unroll
      for (int u = 0; u < 1024 / TH; ++u) {
        const bool ok = kc * 32 + r0 + u * (TH >> 5) < kvalid;
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d + (uint32_t)u * ((TH >> 5) * 136 * 4)),
                     "l"(ok ? g + u * ustride : src), "r"(ok ? 16 : 0)
                     : "memory");
      }
    }
    if (++kc == nk) { kc = 0; ++nb; }
    if (++slot == NSTAGE) slot = 0;
  }
};

__device__ __forceinline__ void ldmatrix_x4(uint32_t (&r)[4], uint32_t saddr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(saddr));
}

// C[16*MT rows][N] = A[16*MT][K] . op(W), A in shared memory (pitch LDA == 4 mod 32), N % 128 == 0, K % 32 == 0.
//   MT = 1: warp w owns columns [16w, 16w+16) of every 128-column block (2 n-tiles).  The A panel is split ONCE into a
//           hi and a lo plane (`asplit`, 2 x 16 x LDA floats) and a warp's A fragments come from two ldmatrix.x4 per k-step
//           (a 16 x 8 tf32 tile is a 16 x 16 b16 tile to ldmatrix): all 8 warps used to redo the same 4 loads + 8 ALU ops;
//   MT = 2: warp w owns m-tile (w & 1) and columns [32(w>>1), +32) (4 n-tiles); A is split in registers (weight gradients).
// epi(row, col, v0, v1) receives two adjacent columns of one row.  Ends with __syncthreads().
template <int MT, int MODE, int LDA, typename Epi>
__device__ __forceinline__ void panel_gemm(const float* As, const float* __restrict__ W, int ldw, int N, int K, int kvalid,
                                           float* wstage, float* asplit, Epi epi) {
  constexpr int NT = (MT == 2) ? 4 : 2;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int mt = (MT == 2) ? (warp & 1) : 0;
  const int cbase = ((MT == 2) ? (warp >> 1) : warp) * NT * 8;
  const int nk = K / 32;
  const int total = (N / 128) * nk;          // weight stages of the whole GEMM: ONE continuous pipeline over all column blocks
  const float* arow = As + (mt * 16 + g) * LDA + t;
  WeightStager<MODE, THREADS> stager(wstage, W, ldw, nk, kvalid);
#pragma unroll
  for (int s = 0; s < NSTAGE - 1; ++s) {
    if (s < total) stager.issue();
    cp_async_commit();
  }
  uint32_t a_hi_addr = 0, a_lo_addr = 0;
  if (MT == 1) {
    // split the panel once (the first __syncthreads of the loop below orders it before any fragment load)
    for (int i = threadIdx.x; i < PR * (K >> 2); i += THREADS) {
      const int r = i / (K >> 2), c = i - r * (K >> 2);
      const float4 v = *reinterpret_cast<const float4*>(As + r * LDA + 4 * c);
      float4 h, l;
      h.x = __uint_as_float(__float_as_uint(v.x) & 0xffffe000u); l.x = v.x - h.x;
      h.y = __uint_as_float(__float_as_uint(v.y) & 0xffffe000u); l.y = v.y - h.y;
      h.z = __uint_as_float(__float_as_uint(v.z) & 0xffffe000u); l.z = v.z - h.z;
      h.w = __uint_as_float(__float_as_uint(v.w) & 0xffffe000u); l.w = v.w - h.w;
      *reinterpret_cast<float4*>(asplit + r * LDA + 4 * c) = h;
      *reinterpret_cast<float4*>(asplit + PR * LDA + r * LDA + 4 * c) = l;
    }
    // ldmatrix row addresses: lane i -> matrix i/8 (0: rows 0-7 k 0-3, 1: rows 8-15 k 0-3, 2: rows 0-7 k 4-7, 3: rows 8-15 k 4-7)
    const int lrow = (lane & 7) + 8 * ((lane >> 3) & 1), lcol = 4 * (lane >> 4);
    a_hi_addr = (uint32_t)__cvta_generic_to_shared(asplit + lrow * LDA + lcol);
    a_lo_addr = a_hi_addr + PR * LDA * 4;
  }
  float acc[NT][4], acl[NT][4];        // hi*hi products and the two small cross terms accumulate in separate chains
  for (int s = 0; s < total; ++s) {
    cp_async_wait<NSTAGE - 2>();
    __syncthreads();
    if (s + NSTAGE - 1 < total) stager.issue();
    cp_async_commit();
    const int kc = s % nk;
    if (kc == 0) {
#pragma unroll
      for (int j = 0; j < NT; ++j) {
        acc[j][0] = 0.f; acc[j][1] = 0.f; acc[j][2] = 0.f; acc[j][3] = 0.f;
        acl[j][0] = 0.f; acl[j][1] = 0.f; acl[j][2] = 0.f; acl[j][3] = 0.f;
      }
    }
    const float* Ws = wstage + (s % NSTAGE) * WT_FLOATS;
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      uint32_t ah[4], al[4];
      if (MT == 1) {
        const uint32_t koff = (uint32_t)(kc * 32 + ks * 8) * 4u;
        ldmatrix_x4(ah, a_hi_addr + koff);
        ldmatrix_x4(al, a_lo_addr + koff);
      } else {
        const float* ap = arow + kc * 32 + ks * 8;
        split_tf32(ap[0], ah[0], al[0]);
        split_tf32(ap[8 * LDA], ah[1], al[1]);
        split_tf32(ap[4], ah[2], al[2]);
        split_tf32(ap[8 * LDA + 4], ah[3], al[3]);
      }
#pragma unroll
      for (int j = 0; j < NT; ++j) {
        float b0, b1;
        if (MODE == B_NK) {
          const float* bp = Ws + (cbase + j * 8 + g) * 36 + ks * 8 + t;
          b0 = bp[0]; b1 = bp[4];
        } else {
          const float* bp = Ws + (ks * 8 + t) * 136 + cbase + j * 8 + g;
          b0 = bp[0]; b1 = bp[4 * 136];
        }
        uint32_t bh[2], bl[2];
        split_tf32(b0, bh[0], bl[0]);
        split_tf32(b1, bh[1], bl[1]);
        mma_tf32(acl[j], al, bh);
        mma_tf32(acc[j], ah, bh);
        mma_tf32(acl[j], ah, bl);
      }
    }
    if (kc == nk - 1) {
      const int nb = (s / nk) * 128;
#pragma unroll
      for (int j = 0; j < NT; ++j) {
        const int col = nb + cbase + j * 8 + 2 * t;
        epi(mt * 16 + g, col, acc[j][0] + acl[j][0], acc[j][1] + acl[j][1]);
        epi(mt * 16 + g + 8, col, acc[j][2] + acl[j][2], acc[j][3] + acl[j][3]);
      }
    }
  }
  cp_async_wait<0>();
  __syncthreads();
}

// =====================================================================================================================
// bf16x3 panel GEMM (the default for the forward / input-gradient GEMMs):  x = xh + xl with xh = bf16(x), xl = bf16(x - xh)
// (16-17 significant bits), x*w ~= xh*wh + xl*wh + xh*wl on mma.sync.m16n8k16 with fp32 accumulation: ~2^-16 relative,
// 200x below the bf16 noise of the conv towers that feed the encoder.  Against the 3xTF32 GEMM above it halves the MMA count
// (k16 instead of k8) and -- the point -- removes the operand handling from the inner loop: the weights are split ONCE per
// step into bf16 hi / lo arrays (tmf_encoder_pack_weights), stream through the cp.async ring as they are, and both operands
// reach the registers with ldmatrix.x4; per warp and 32-k stage that is 8 ldmatrix + 12 MMA instead of 8 ldmatrix + 32 LDS +
// 64 ALU + 24 MMA.  Measured (TMF_ENC_PROF): a stage of enc_chain_fwd took 1200-1400 cycles with 3xTF32.
// =====================================================================================================================
__device__ __forceinline__ void mma_bf16(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void ldmatrix_x4_trans(uint32_t (&r)[4], uint32_t saddr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(saddr));
}
// hi / lo bf16 pairs of two fp32 values
__device__ __forceinline__ void split_bf16x2(float a, float b, uint32_t& hi, uint32_t& lo) {
  hi = pack_bf16(a, b);
  const uint64_t l2 = sub2_f32(pair_f32(a, b), pair_u32(hi << 16, hi & 0xffff0000u));
  lo = pack_bf16(__uint_as_float(lo_u32(l2)), __uint_as_float(hi_u32(l2)));
}

__device__ int g_enc_prof = 0;              // TMF_ENC_PROF: block 0 prints where the stage loop of the bf16 GEMM spends its cycles

constexpr int WB_NK_PITCH = 80;              // bytes per row of a B_NK stage tile: 32 bf16 + 16 B pad (conflict-free ldmatrix)
constexpr int WB_KN_PITCH = 272;             // bytes per row of a B_KN stage tile: 128 bf16 + 16 B pad
constexpr int WB_NK_PLANE = 128 * WB_NK_PITCH, WB_KN_PLANE = 32 * WB_KN_PITCH;

// Weight stages of the split-weight path: `whi` / `whi + wnumel` are the bf16 hi / lo copies of W (same [rows][ldw] layout).
template <int MODE>
struct WeightStagerB {
  const __nv_bfloat16* src;  // chunk u = 0 of stage 0
  uint32_t dst;
  size_t lo_off;             // elements between the hi and the lo array
  int ldw, nk, nb, kc, slot;
  __device__ __forceinline__ WeightStagerB(float* wstage, const __nv_bfloat16* whi, size_t wnumel, int ldw_, int nk_)
      : lo_off(wnumel), ldw(ldw_), nk(nk_), nb(0), kc(0), slot(0) {
    if (MODE == B_NK) {      // chunk c = thread + 256 u: plane u >> 1, row (thread >> 2) + 64 (u & 1), 16-byte column thread & 3
      const int r0 = threadIdx.x >> 2, q = threadIdx.x & 3;
      src = whi + (size_t)r0 * ldw + 8 * q;
      dst = (uint32_t)__cvta_generic_to_shared(wstage) + r0 * WB_NK_PITCH + q * 16;
    } else {                 // plane u >> 1, row (thread >> 4) + 16 (u & 1), 16-byte column thread & 15
      const int r0 = threadIdx.x >> 4, q = threadIdx.x & 15;
      src = whi + (size_t)r0 * ldw + 8 * q;
      dst = (uint32_t)__cvta_generic_to_shared(wstage) + r0 * WB_KN_PITCH + q * 16;
    }
  }
  __device__ __forceinline__ void issue() {
    const uint32_t d = dst + (uint32_t)slot * (WT_FLOATS * 4);
    if (MODE == B_NK) {
      const __nv_bfloat16* g = src + (size_t)nb * 128 * ldw + kc * 32;
#pragma unroll
      for (int u = 0; u < 4; ++u)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d + (u >> 1) * WB_NK_PLANE + (u & 1) * 64 * WB_NK_PITCH),
                     "l"(g + (u >> 1) * lo_off + (size_t)(u & 1) * 64 * ldw)
                     : "memory");
    } else {
      const __nv_bfloat16* g = src + (size_t)kc * 32 * ldw + nb * 128;
#pragma unroll
      for (int u = 0; u < 4; ++u)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d + (u >> 1) * WB_KN_PLANE + (u & 1) * 16 * WB_KN_PITCH),
                     "l"(g + (u >> 1) * lo_off + (size_t)(u & 1) * 16 * ldw)
                     : "memory");
    }
    if (++kc == nk) { kc = 0; ++nb; }
    if (++slot == NSTAGE) slot = 0;
  }
};

// C[16][N] = A[16][K] . op(W):  A fp32 in shared memory (pitch LDA floats), W given as its bf16 hi / lo arrays; warp w owns
// columns [16w, 16w+16) of every 128-column block.  `asplit` receives the bf16 hi / lo planes of A ([2][16][K+8] bf16).
// B_NK: W is [N][K] (ldw = K); B_KN: W is [K][N] (ldw = N).  epi as in panel_gemm.  Ends with __syncthreads().
template <int MODE, int LDA, int K, typename Epi>
__device__ __forceinline__ void panel_gemm_bf16(const float* As, const __nv_bfloat16* whi, size_t wnumel, int ldw, int N,
                                                float* wstage, float* asplit, Epi epi) {
  static_assert(THREADS == 256, "chunk mapping of WeightStagerB assumes 256 threads");
  constexpr int AP = (K + 8) * 2;                      // bytes per row of an A plane
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int cbase = warp * 16;
  constexpr int nk = K / 32;
  const int total = (N / 128) * nk;
  WeightStagerB<MODE> stager(wstage, whi, wnumel, ldw, nk);
#pragma unroll
  for (int s = 0; s < NSTAGE - 1; ++s) {
    if (s < total) stager.issue();
    cp_async_commit();
  }
  // split the panel once (the first __syncthreads of the loop below orders it before any fragment load)
  uint8_t* ap = reinterpret_cast<uint8_t*>(asplit);
  for (int i = threadIdx.x; i < PR * (K >> 2); i += THREADS) {
    const int r = i / (K >> 2), c = i - r * (K >> 2);
    const float4 v = *reinterpret_cast<const float4*>(As + r * LDA + 4 * c);
    uint2 h, l;
    split_bf16x2(v.x, v.y, h.x, l.x);
    split_bf16x2(v.z, v.w, h.y, l.y);
    *reinterpret_cast<uint2*>(ap + r * AP + 8 * c) = h;
    *reinterpret_cast<uint2*>(ap + PR * AP + r * AP + 8 * c) = l;
  }
  // ldmatrix lane addresses.  A: matrices (rows 0-7, k 0-7), (rows 8-15, k 0-7), (rows 0-7, k 8-15), (rows 8-15, k 8-15)
  const uint32_t a_hi = (uint32_t)__cvta_generic_to_shared(ap) + ((lane & 7) + 8 * ((lane >> 3) & 1)) * AP + 16 * (lane >> 4);
  const uint32_t a_lo = a_hi + PR * AP;
  // B: matrices (n-tile 0, k 0-7), (n-tile 0, k 8-15), (n-tile 1, k 0-7), (n-tile 1, k 8-15)
  const uint32_t b_off = (MODE == B_NK)
                             ? (uint32_t)((cbase + (lane & 7) + 8 * (lane >> 4)) * WB_NK_PITCH + 16 * ((lane >> 3) & 1))
                             : (uint32_t)(((lane & 7) + 8 * ((lane >> 3) & 1)) * WB_KN_PITCH + (cbase + 8 * (lane >> 4)) * 2);
  const uint32_t w_sm = (uint32_t)__cvta_generic_to_shared(wstage);
  float acc[2][4], acl[2][4];          // hi*hi products and the two small cross terms accumulate in separate chains
  const bool prof = g_enc_prof != 0 && blockIdx.x == 0;
  long long t_wait = 0, t_bar = 0, t_issue = 0, t_all = prof ? clock64() : 0;
  for (int s = 0; s < total; ++s) {
    long long t0 = prof ? clock64() : 0;
    cp_async_wait<NSTAGE - 2>();
    long long t1 = prof ? clock64() : 0;
    __syncthreads();
    long long t2 = prof ? clock64() : 0;
    if (s + NSTAGE - 1 < total) stager.issue();
    cp_async_commit();
    if (prof) { const long long t3 = clock64(); t_wait += t1 - t0; t_bar += t2 - t1; t_issue += t3 - t2; }
    const int kc = s % nk;
    if (kc == 0) {
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        acc[j][0] = 0.f; acc[j][1] = 0.f; acc[j][2] = 0.f; acc[j][3] = 0.f;
        acl[j][0] = 0.f; acl[j][1] = 0.f; acl[j][2] = 0.f; acl[j][3] = 0.f;
      }
    }
    const uint32_t ws = w_sm + (uint32_t)(s % NSTAGE) * (WT_FLOATS * 4) + b_off;
#pragma unroll
    for (int kk = 0; kk < 2; ++kk) {
      uint32_t ah[4], al[4], bh[4], bl[4];
      const uint32_t koff = (uint32_t)(kc * 32 + kk * 16) * 2u;
      ldmatrix_x4(ah, a_hi + koff);
      ldmatrix_x4(al, a_lo + koff);
      if (MODE == B_NK) {
        ldmatrix_x4(bh, ws + kk * 32);
        ldmatrix_x4(bl, ws + WB_NK_PLANE + kk * 32);
      } else {
        ldmatrix_x4_trans(bh, ws + kk * 16 * WB_KN_PITCH);
        ldmatrix_x4_trans(bl, ws + WB_KN_PLANE + kk * 16 * WB_KN_PITCH);
      }
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        mma_bf16(acl[j], al, bh[2 * j], bh[2 * j + 1]);
        mma_bf16(acc[j], ah, bh[2 * j], bh[2 * j + 1]);
        mma_bf16(acl[j], ah, bl[2 * j], bl[2 * j + 1]);
      }
    }
    if (kc == nk - 1) {
      const int nb = (s / nk) * 128;
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const int col = nb + cbase + j * 8 + 2 * t;
        epi(g, col, acc[j][0] + acl[j][0], acc[j][1] + acl[j][1]);
        epi(g + 8, col, acc[j][2] + acl[j][2], acc[j][3] + acl[j][3]);
      }
    }
  }
  cp_async_wait<0>();
  __syncthreads();
  if (prof && (threadIdx.x == 0 || threadIdx.x == 255))
    printf("bf16 gemm N=%d K=%d thread %d: %d stages, total %lld cyc: cp.async wait %lld, barrier %lld, issue %lld\n", N, K,
           (int)threadIdx.x, total, clock64() - t_all, t_wait, t_bar, t_issue);
}

// One GEMM of a panel kernel: split-weight bf16x3 path when the caller passed a weight pack, 3xTF32 from the fp32 weights
// otherwise (cross-check / TMF_ENC_BF16=0).  `woff` = element offset of this matrix inside the pack (hi array; lo follows).
template <int MODE, int LDA, int K, typename Epi>
__device__ __forceinline__ void panel_gemm_any(const float* As, const float* __restrict__ W, const __nv_bfloat16* pack, size_t woff,
                                               size_t wnumel, int ldw, int N, float* wstage, float* asplit, Epi epi) {
  if (pack != nullptr) panel_gemm_bf16<MODE, LDA, K>(As, pack + woff, wnumel, ldw, N, wstage, asplit, epi);
  else panel_gemm<1, MODE, LDA>(As, W, ldw, N, K, 1 << 30, wstage, asplit, epi);
}

// element offsets of the five weight matrices inside a pack ([hi | lo] per matrix): Wq, Wkv, Wo, W1, W2
__host__ __device__ constexpr size_t pack_off_wq() { return 0; }
__host__ __device__ constexpr size_t pack_off_wkv() { return 2 * 128 * 128; }
__host__ __device__ constexpr size_t pack_off_wo() { return pack_off_wkv() + 2 * 256 * 128; }
__host__ __device__ constexpr size_t pack_off_w1() { return pack_off_wo() + 2 * 128 * 128; }
__host__ __device__ constexpr size_t pack_off_w2(int mlp) { return pack_off_w1() + (size_t)2 * mlp * 128; }
__host__ __device__ constexpr size_t pack_elems(int mlp) { return pack_off_w2(mlp) + (size_t)2 * 128 * mlp; }

struct PackArgs {
  const float* w[5];
  int numel[5];
  size_t off[5];
  __nv_bfloat16* pack;
};
__global__ void __launch_bounds__(256) enc_pack_kernel(PackArgs p) {
  const int m = blockIdx.y;
  const float4* src = reinterpret_cast<const float4*>(p.w[m]);
  uint2* hi = reinterpret_cast<uint2*>(p.pack + p.off[m]);
  uint2* lo = reinterpret_cast<uint2*>(p.pack + p.off[m] + p.numel[m]);
  for (int i = blockIdx.x * 256 + threadIdx.x; i < (p.numel[m] >> 2); i += gridDim.x * 256) {
    const float4 v = __ldg(src + i);
    uint2 h, l;
    split_bf16x2(v.x, v.y, h.x, l.x);
    split_bf16x2(v.z, v.w, h.y, l.y);
    hi[i] = h;
    lo[i] = l;
  }
}

// ---- panel <-> global helpers (all 256 threads; float4, rows >= nvalid read as zero / are not written) ----------------
template <int COLS>
__device__ __forceinline__ void load_panel(float* Ps, int lds, const float* __restrict__ src, int ld, int nvalid, int rows) {
  constexpr int c4 = COLS >> 2;                 // (a power of two: the index split below compiles to shifts)
  for (int i = threadIdx.x; i < rows * c4; i += THREADS) {
    const int r = i / c4, c = i - r * c4;
    const float4 v = (r < nvalid) ? __ldg(reinterpret_cast<const float4*>(src + (size_t)r * ld) + c) : make_float4(0.f, 0.f, 0.f, 0.f);
    *reinterpret_cast<float4*>(Ps + r * lds + 4 * c) = v;
  }
}
template <int COLS>
__device__ __forceinline__ void store_panel(float* __restrict__ dst, int ld, const float* Ps, int lds, int nvalid) {
  constexpr int c4 = COLS >> 2;
  for (int i = threadIdx.x; i < nvalid * c4; i += THREADS) {
    const int r = i / c4, c = i - r * c4;
    reinterpret_cast<float4*>(dst + (size_t)r * ld)[c] = *reinterpret_cast<const float4*>(Ps + r * lds + 4 * c);
  }
}

// LayerNorm of a 16 x 128 panel, in place or into `out`: warp w takes rows 2w, 2w+1; a lane owns columns 4*lane..4*lane+3.
// Two-pass statistics exactly like layernorm_fwd_kernel (fusion_ops.cu).
__device__ __forceinline__ void panel_layernorm(const float* Ps, float* out, int lds, const float* __restrict__ gamma,
                                                const float* __restrict__ beta, float eps, float* __restrict__ mean_out,
                                                float* __restrict__ rstd_out, int row0, int nvalid) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float4 gm = __ldg(reinterpret_cast<const float4*>(gamma) + lane);
  const float4 bt = __ldg(reinterpret_cast<const float4*>(beta) + lane);
#pragma unroll
  for (int rr = 0; rr < 2; ++rr) {
    const int r = 2 * warp + rr;
    const float4 v = *reinterpret_cast<const float4*>(Ps + r * lds + 4 * lane);
    const float mean = warp_sum(v.x + v.y + v.z + v.w) * (1.f / 128.f);
    const float a = v.x - mean, b = v.y - mean, c = v.z - mean, d = v.w - mean;
    const float rstd = rsqrtf(warp_sum(a * a + b * b + c * c + d * d) * (1.f / 128.f) + eps);
    if (lane == 0 && r < nvalid) { mean_out[row0 + r] = mean; rstd_out[row0 + r] = rstd; }
    float4 o;
    o.x = a * rstd * gm.x + bt.x; o.y = b * rstd * gm.y + bt.y; o.z = c * rstd * gm.z + bt.z; o.w = d * rstd * gm.w + bt.w;
    *reinterpret_cast<float4*>(out + r * lds + 4 * lane) = o;
  }
}

// LayerNorm backward of a 16 x 128 panel: dx = rstd * (dy*gamma - mean(dy*gamma) - xhat * mean(dy*gamma*xhat)), written to
// `dxo` (+ `addp` if not null); the lane's column sums of dy*xhat / dy are accumulated into ag / ab (rows >= nvalid skip).
__device__ __forceinline__ void panel_layernorm_bwd(const float* dys, const float* xs, float* dxo, const float* addp, int lds,
                                                    const float* __restrict__ gamma, const float* __restrict__ mean,
                                                    const float* __restrict__ rstd, int row0, int nvalid, float4& ag,
                                                    float4& ab) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float4 gm = __ldg(reinterpret_cast<const float4*>(gamma) + lane);
#pragma unroll
  for (int rr = 0; rr < 2; ++rr) {
    const int r = 2 * warp + rr;
    const bool ok = r < nvalid;
    const float mu = ok ? mean[row0 + r] : 0.f, rs = ok ? rstd[row0 + r] : 0.f;
    const float4 xv = *reinterpret_cast<const float4*>(xs + r * lds + 4 * lane);
    const float4 gv = *reinterpret_cast<const float4*>(dys + r * lds + 4 * lane);
    const float4 xh = make_float4((xv.x - mu) * rs, (xv.y - mu) * rs, (xv.z - mu) * rs, (xv.w - mu) * rs);
    const float4 gg = make_float4(gv.x * gm.x, gv.y * gm.y, gv.z * gm.z, gv.w * gm.w);
    const float s1 = warp_sum(gg.x + gg.y + gg.z + gg.w) * (1.f / 128.f);
    const float s2 = warp_sum(gg.x * xh.x + gg.y * xh.y + gg.z * xh.z + gg.w * xh.w) * (1.f / 128.f);
    if (ok) {
      ag.x += gv.x * xh.x; ag.y += gv.y * xh.y; ag.z += gv.z * xh.z; ag.w += gv.w * xh.w;
      ab.x += gv.x; ab.y += gv.y; ab.z += gv.z; ab.w += gv.w;
    }
    float4 o = make_float4(rs * (gg.x - s1 - xh.x * s2), rs * (gg.y - s1 - xh.y * s2), rs * (gg.z - s1 - xh.z * s2),
                           rs * (gg.w - s1 - xh.w * s2));
    if (addp != nullptr) {
      const float4 e = *reinterpret_cast<const float4*>(addp + r * lds + 4 * lane);
      o.x += e.x; o.y += e.y; o.z += e.z; o.w += e.w;
    }
    *reinterpret_cast<float4*>(dxo + r * lds + 4 * lane) = o;
  }
}

// Block-level column sums of NV per-lane float4 accumulators (8 warps, lane owns columns 4*lane..): the warps add into
// red[NV][128] one after the other (deterministic), result left in red.
template <int NV>
__device__ __forceinline__ void block_colsum128(float* red, const float4 (&v)[NV]) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int w = 0; w < THREADS / 32; ++w) {
    if (warp == w) {
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        float4* p = reinterpret_cast<float4*>(red + 128 * i) + lane;
        if (w == 0) *p = v[i];
        else { float4 a = *p; a.x += v[i].x; a.y += v[i].y; a.z += v[i].z; a.w += v[i].w; *p = a; }
      }
    }
    __syncthreads();
  }
}

// Cross-block finish of per-block LayerNorm parameter partials: part[block][nvec][128] -> outs[v][128], added in block order.
__device__ __forceinline__ void finish_ln_partials(float* __restrict__ part, int nvec, float* const* outs, unsigned* ticket) {
  if (!last_block_arrives(ticket, gridDim.x)) return;
  for (int i = threadIdx.x; i < nvec * 128; i += THREADS) {
    float s = 0.f;
    for (unsigned b = 0; b < gridDim.x; ++b) s += __ldcg(part + (size_t)b * nvec * 128 + i);
    float* o = outs[i >> 7];
    if (o != nullptr) o[i & 127] = s;
  }
}

// =====================================================================================================================
// F1: projections.  blocks [0, nbx): x panels;  [nbx, nbx + nbc): ctx panels
// =====================================================================================================================
struct ProjFwdArgs {
  const float *x, *ctx, *ln_w, *ln_b, *wq, *wkv;
  float *h1, *mean1, *rstd1, *q, *kv;
  int Mx, Mc, nbx;
  float eps;
  const __nv_bfloat16* pack;          // bf16 hi / lo copies of the weights (tmf_encoder_pack_weights), or null: 3xTF32
};

__global__ void __launch_bounds__(THREADS) enc_proj_fwd_kernel(ProjFwdArgs p) {
  extern __shared__ __align__(16) float sm[];
  float* P0 = sm;                           // [16][132] input panel
  float* P1 = P0 + PR * LD128;              // [16][260] output panel
  float* spl = P1 + PR * 260;               // [2][16][132] hi / lo planes of the GEMM's A panel
  float* wst = spl + 2 * PR * LD128;
  if ((int)blockIdx.x < p.nbx) {
    const int row0 = blockIdx.x * PR, nv = min(PR, p.Mx - row0);
    load_panel<128>(P0, LD128, p.x + (size_t)row0 * 128, 128, nv, PR);
    __syncthreads();
    panel_layernorm(P0, P0, LD128, p.ln_w, p.ln_b, p.eps, p.mean1, p.rstd1, row0, nv);
    __syncthreads();
    store_panel<128>(p.h1 + (size_t)row0 * 128, 128, P0, LD128, nv);
    panel_gemm_any<B_NK, LD128, 128>(P0, p.wq, p.pack, pack_off_wq(), 128 * 128, 128, 128, wst, spl, [&](int r, int c, float v0, float v1) {
      *reinterpret_cast<float2*>(P1 + r * LD128 + c) = make_float2(v0, v1);
    });
    store_panel<128>(p.q + (size_t)row0 * 128, 128, P1, LD128, nv);
  } else {
    const int row0 = (blockIdx.x - p.nbx) * PR, nv = min(PR, p.Mc - row0);
    load_panel<128>(P0, LD128, p.ctx + (size_t)row0 * 128, 128, nv, PR);
    __syncthreads();
    panel_gemm_any<B_NK, LD128, 128>(P0, p.wkv, p.pack, pack_off_wkv(), 256 * 128, 128, 256, wst, spl, [&](int r, int c, float v0, float v1) {
      *reinterpret_cast<float2*>(P1 + r * 260 + c) = make_float2(v0, v1);
    });
    store_panel<256>(p.kv + (size_t)row0 * 256, 256, P1, 260, nv);
  }
}

// =====================================================================================================================
// F3: the row-local chain behind the attention core
// =====================================================================================================================
struct ChainFwdArgs {
  const float *o, *x, *wo, *bo, *ln2_w, *ln2_b, *w1, *b1, *w2, *b2, *lnf_w, *lnf_b;
  float *a, *h2, *mean2, *rstd2, *pre, *f, *g, *meanf, *rstdf, *y;
  int M, mlp, add_input, prof;
  float eps2, epsf;
  const __nv_bfloat16* pack;
};

template <int MLP>
__global__ void __launch_bounds__(THREADS) enc_chain_fwd_kernel(ChainFwdArgs p) {
  extern __shared__ __align__(16) float sm[];
  constexpr int ldf = MLP + 4;
  float* P0 = sm;                           // o, later g
  float* P1 = P0 + PR * LD128;              // a
  float* P2 = P1 + PR * LD128;              // h2
  float* PF = P2 + PR * LD128;              // [16][mlp+4]: pre-activation, then f
  float* spl = PF + PR * ldf;               // [2][16][mlp+4] hi / lo planes of the current GEMM's A panel
  float* wst = spl + 2 * PR * ldf;
  const int row0 = blockIdx.x * PR, nv = min(PR, p.M - row0);
  long long tk[10]; int ntk = 0;
#define TK() do { if (p.prof) { __syncthreads(); tk[ntk++] = clock64(); } } while (0)
  TK();
  load_panel<128>(P0, LD128, p.o + (size_t)row0 * 128, 128, nv, PR);
  load_panel<128>(P2, LD128, p.x + (size_t)row0 * 128, 128, nv, PR);     // x parked in P2 until LN2 overwrites it
  __syncthreads();
  TK();
  // a = o Wo^T + bo + x
  panel_gemm_any<B_NK, LD128, 128>(P0, p.wo, p.pack, pack_off_wo(), 128 * 128, 128, 128, wst, spl, [&](int r, int c, float v0, float v1) {
    const float2 xb = *reinterpret_cast<const float2*>(P2 + r * LD128 + c);
    *reinterpret_cast<float2*>(P1 + r * LD128 + c) = make_float2(v0 + __ldg(p.bo + c) + xb.x, v1 + __ldg(p.bo + c + 1) + xb.y);
  });
  TK();
  store_panel<128>(p.a + (size_t)row0 * 128, 128, P1, LD128, nv);
  panel_layernorm(P1, P2, LD128, p.ln2_w, p.ln2_b, p.eps2, p.mean2, p.rstd2, row0, nv);
  __syncthreads();
  store_panel<128>(p.h2 + (size_t)row0 * 128, 128, P2, LD128, nv);
  TK();
  // pre = h2 W1^T + b1 (saved for the backward pass straight from the accumulator registers);  f = GELU(pre) -> PF
  panel_gemm_any<B_NK, LD128, 128>(P2, p.w1, p.pack, pack_off_w1(), MLP * 128, 128, MLP, wst, spl, [&](int r, int c, float v0, float v1) {
    const float2 pre = make_float2(v0 + __ldg(p.b1 + c), v1 + __ldg(p.b1 + c + 1));
    if (r < nv) *reinterpret_cast<float2*>(p.pre + (size_t)(row0 + r) * MLP + c) = pre;
    *reinterpret_cast<float2*>(PF + r * ldf + c) = make_float2(gelu_exact(pre.x), gelu_exact(pre.y));
  });
  TK();
  store_panel<MLP>(p.f + (size_t)row0 * MLP, MLP, PF, ldf, nv);
  // g = f W2^T + b2 + a
  panel_gemm_any<B_NK, MLP + 4, MLP>(PF, p.w2, p.pack, pack_off_w2(MLP), 128 * MLP, MLP, 128, wst, spl, [&](int r, int c, float v0, float v1) {
    const float2 ab = *reinterpret_cast<const float2*>(P1 + r * LD128 + c);
    *reinterpret_cast<float2*>(P0 + r * LD128 + c) = make_float2(v0 + __ldg(p.b2 + c) + ab.x, v1 + __ldg(p.b2 + c + 1) + ab.y);
  });
  TK();
  store_panel<128>(p.g + (size_t)row0 * 128, 128, P0, LD128, nv);
  // y = LNf(g) (+ x)
  panel_layernorm(P0, P2, LD128, p.lnf_w, p.lnf_b, p.epsf, p.meanf, p.rstdf, row0, nv);
  __syncthreads();
  if (p.add_input) {
    for (int i = threadIdx.x; i < nv * 32; i += THREADS) {
      const int r = i >> 5, c = i & 31;
      const float4 xv = __ldg(reinterpret_cast<const float4*>(p.x + (size_t)(row0 + r) * 128) + c);
      float4 v = *reinterpret_cast<const float4*>(P2 + r * LD128 + 4 * c);
      v.x += xv.x; v.y += xv.y; v.z += xv.z; v.w += xv.w;
      reinterpret_cast<float4*>(p.y + (size_t)(row0 + r) * 128)[c] = v;
    }
  } else {
    store_panel<128>(p.y + (size_t)row0 * 128, 128, P2, LD128, nv);
  }
  TK();
  if (p.prof && blockIdx.x == 0 && threadIdx.x == 0) {
    printf("enc_chain_fwd phases (cycles): load %lld | gemm_o %lld | store a, LN2, store h2 %lld | gemm_1 %lld | store f %lld+gemm_2 %lld | LNf, store y %lld\n", tk[1]-tk[0], tk[2]-tk[1], tk[3]-tk[2], tk[4]-tk[3], 0ll, tk[5]-tk[4], tk[6]-tk[5]);
  }
#undef TK
}

// =====================================================================================================================
// R1: backward of the chain
// =====================================================================================================================
struct ChainBwdArgs {
  const float *dy, *g, *a, *pre, *wo, *w1, *w2, *ln2_w, *lnf_w, *mean2, *rstd2, *meanf, *rstdf;
  float *dg, *dp, *da, *dout, *dxp;                 // dxp = da (+ dy when the outer residual is fused)
  float *dlnf_w, *dlnf_b, *dln2_w, *dln2_b;
  float* part;                                      // [gridDim.x][4][128]
  unsigned* ticket;
  int M, mlp, add_input;
  const __nv_bfloat16* pack;
};

template <int MLP>
__global__ void __launch_bounds__(THREADS) enc_chain_bwd_kernel(ChainBwdArgs p) {
  extern __shared__ __align__(16) float sm[];
  constexpr int ldf = MLP + 4;
  float* P0 = sm;
  float* P1 = P0 + PR * LD128;
  float* P2 = P1 + PR * LD128;
  float* PF = P2 + PR * LD128;
  float* spl = PF + PR * ldf;
  float* wst = spl + 2 * PR * ldf;
  float* red = wst + NSTAGE * WT_FLOATS;            // [4][128]
  const int row0 = blockIdx.x * PR, nv = min(PR, p.M - row0);
  const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
  float4 agf = z4, abf = z4, ag2 = z4, ab2 = z4;
  load_panel<128>(P0, LD128, p.dy + (size_t)row0 * 128, 128, nv, PR);
  load_panel<128>(P1, LD128, p.g + (size_t)row0 * 128, 128, nv, PR);
  __syncthreads();
  // dg = LNf'(dy)  -> P2
  panel_layernorm_bwd(P0, P1, P2, nullptr, LD128, p.lnf_w, p.meanf, p.rstdf, row0, nv, agf, abf);
  __syncthreads();
  store_panel<128>(p.dg + (size_t)row0 * 128, 128, P2, LD128, nv);
  // dp = (dg W2) * GELU'(pre)  -> PF        (W2 is [128][mlp]: reduction over its rows)
  load_panel<MLP>(PF, ldf, p.pre + (size_t)row0 * MLP, MLP, nv, PR);
  __syncthreads();
  panel_gemm_any<B_KN, LD128, 128>(P2, p.w2, p.pack, pack_off_w2(MLP), 128 * MLP, MLP, MLP, wst, spl, [&](int r, int c, float v0, float v1) {
    float2* q = reinterpret_cast<float2*>(PF + r * ldf + c);
    const float2 pr = *q;
    *q = make_float2(v0 * gelu_grad(pr.x), v1 * gelu_grad(pr.y));
  });
  store_panel<MLP>(p.dp + (size_t)row0 * MLP, MLP, PF, ldf, nv);
  // dh2 = dp W1  -> P0                       (W1 is [mlp][128])
  panel_gemm_any<B_KN, MLP + 4, MLP>(PF, p.w1, p.pack, pack_off_w1(), MLP * 128, 128, 128, wst, spl, [&](int r, int c, float v0, float v1) {
    *reinterpret_cast<float2*>(P0 + r * LD128 + c) = make_float2(v0, v1);
  });
  // da = dg + LN2'(dh2)  -> P0
  load_panel<128>(P1, LD128, p.a + (size_t)row0 * 128, 128, nv, PR);
  __syncthreads();
  panel_layernorm_bwd(P0, P1, P0, P2, LD128, p.ln2_w, p.mean2, p.rstd2, row0, nv, ag2, ab2);
  __syncthreads();
  store_panel<128>(p.da + (size_t)row0 * 128, 128, P0, LD128, nv);
  // dxp = da (+ dy: outer residual)
  for (int i = threadIdx.x; i < nv * 32; i += THREADS) {
    const int r = i >> 5, c = i & 31;
    float4 v = *reinterpret_cast<const float4*>(P0 + r * LD128 + 4 * c);
    if (p.add_input) {
      const float4 e = __ldg(reinterpret_cast<const float4*>(p.dy + (size_t)(row0 + r) * 128) + c);
      v.x += e.x; v.y += e.y; v.z += e.z; v.w += e.w;
    }
    reinterpret_cast<float4*>(p.dxp + (size_t)(row0 + r) * 128)[c] = v;
  }
  // do = da Wo  -> P1                        (Wo is [128][128])
  panel_gemm_any<B_KN, LD128, 128>(P0, p.wo, p.pack, pack_off_wo(), 128 * 128, 128, 128, wst, spl, [&](int r, int c, float v0, float v1) {
    *reinterpret_cast<float2*>(P1 + r * LD128 + c) = make_float2(v0, v1);
  });
  store_panel<128>(p.dout + (size_t)row0 * 128, 128, P1, LD128, nv);
  // LayerNorm parameter gradients: block partials, then the last block adds them in order
  const float4 sums[4] = {agf, abf, ag2, ab2};
  block_colsum128<4>(red, sums);
  for (int i = threadIdx.x; i < 512; i += THREADS) p.part[(size_t)blockIdx.x * 512 + i] = red[i];
  float* outs[4] = {p.dlnf_w, p.dlnf_b, p.dln2_w, p.dln2_b};
  finish_ln_partials(p.part, 4, outs, p.ticket);
}

// =====================================================================================================================
// R3: backward of the projections
// =====================================================================================================================
struct ProjBwdArgs {
  const float *dq, *dkv, *dxp, *x, *ln_w, *mean1, *rstd1, *wq, *wkv;
  float *dx, *dctx, *dln_w, *dln_b;
  float* part;                                      // [nbx][2][128]
  unsigned* ticket;
  int Mx, Mc, nbx;
  const __nv_bfloat16* pack;
};

__global__ void __launch_bounds__(THREADS) enc_proj_bwd_kernel(ProjBwdArgs p) {
  extern __shared__ __align__(16) float sm[];
  float* P0 = sm;                           // [16][260]
  float* P1 = P0 + PR * 260;                // [16][132]
  float* P2 = P1 + PR * LD128;              // [16][132]
  float* spl = P2 + PR * LD128;             // [2][16][260]
  float* wst = spl + 2 * PR * 260;
  float* red = wst + NSTAGE * WT_FLOATS;    // [2][128]
  if ((int)blockIdx.x < p.nbx) {
    const int row0 = blockIdx.x * PR, nv = min(PR, p.Mx - row0);
    load_panel<128>(P0, LD128, p.dq + (size_t)row0 * 128, 128, nv, PR);
    __syncthreads();
    // dh1 = dq Wq  -> P1
    panel_gemm_any<B_KN, LD128, 128>(P0, p.wq, p.pack, pack_off_wq(), 128 * 128, 128, 128, wst, spl, [&](int r, int c, float v0, float v1) {
      *reinterpret_cast<float2*>(P1 + r * LD128 + c) = make_float2(v0, v1);
    });
    load_panel<128>(P0, LD128, p.x + (size_t)row0 * 128, 128, nv, PR);
    load_panel<128>(P2, LD128, p.dxp + (size_t)row0 * 128, 128, nv, PR);
    __syncthreads();
    float4 ag = make_float4(0.f, 0.f, 0.f, 0.f), ab = ag;
    panel_layernorm_bwd(P1, P0, P1, P2, LD128, p.ln_w, p.mean1, p.rstd1, row0, nv, ag, ab);
    __syncthreads();
    store_panel<128>(p.dx + (size_t)row0 * 128, 128, P1, LD128, nv);
    const float4 sums[2] = {ag, ab};
    block_colsum128<2>(red, sums);
    for (int i = threadIdx.x; i < 256; i += THREADS) p.part[(size_t)blockIdx.x * 256 + i] = red[i];
  } else {
    const int row0 = (blockIdx.x - p.nbx) * PR, nv = min(PR, p.Mc - row0);
    load_panel<256>(P0, 260, p.dkv + (size_t)row0 * 256, 256, nv, PR);
    __syncthreads();
    // dctx = dkv Wkv                          (Wkv is [256][128])
    panel_gemm_any<B_KN, 260, 256>(P0, p.wkv, p.pack, pack_off_wkv(), 256 * 128, 128, 128, wst, spl, [&](int r, int c, float v0, float v1) {
      *reinterpret_cast<float2*>(P1 + r * LD128 + c) = make_float2(v0, v1);
    });
    store_panel<128>(p.dctx + (size_t)row0 * 128, 128, P1, LD128, nv);
  }
  // every block takes part in the rendezvous; only the x blocks hold partials
  if (!last_block_arrives(p.ticket, gridDim.x)) return;
  for (int i = threadIdx.x; i < 256; i += THREADS) {
    float s = 0.f;
    for (int b = 0; b < p.nbx; ++b) s += __ldcg(p.part + (size_t)b * 256 + i);
    if (i < 128) p.dln_w[i] = s; else p.dln_b[i - 128] = s;
  }
}

// =====================================================================================================================
// R4: the five weight gradients (+ three bias gradients) of one encoder in one launch
//     dW[n][k] = sum_m dY[m][n] * X[m][k];   db[n] = sum_m dY[m][n]
// A block computes a [32 (n)] x [128 (k)] tile of one problem over one chunk of WG_MC tokens; the chunks of a tile meet
// in scratch and the last one adds them in order.
// =====================================================================================================================
constexpr int WG_MC = 416;                  // tokens per chunk (3 chunks cover 1200 tokens: 144 blocks); pitch 420 == 4 mod 32
constexpr int WG_LDA = WG_MC + 4;
constexpr int WG_PROBLEMS = 5;

struct WgradProblem {
  const float* dy; const float* x; float* dw; float* db;
  int ldy, ldx, N, K, M;
  int tile0;                                // first tile index of this problem
};
struct WgradArgs {
  WgradProblem pr[WG_PROBLEMS];
  int ntiles, nsplit;
  float* part;                              // [ntiles][nsplit][32*128 + 32]
  unsigned* tickets;                        // [ntiles]
};

__global__ void __launch_bounds__(THREADS) enc_wgrad_kernel(WgradArgs p) {
  extern __shared__ __align__(16) float sm[];
  float* At = sm;                           // [32][WG_LDA]: dY^T chunk
  float* wst = At + 32 * WG_LDA;
  const int tile = blockIdx.x / p.nsplit, split = blockIdx.x % p.nsplit;
  int pi = 0;
#pragma unroll
  for (int i = 1; i < WG_PROBLEMS; ++i)
    if (tile >= p.pr[i].tile0) pi = i;
  const WgradProblem& q = p.pr[pi];
  const int lt = tile - q.tile0, kt = q.K / 128;
  const int n0 = (lt / kt) * 32, k0 = (lt % kt) * 128;
  const int m0 = split * WG_MC, mv = max(0, min(WG_MC, q.M - m0));
  // stage dY^T: At[n][m] = dY[m0 + m][n0 + n]   (a warp reads 32 consecutive n of one token: 128 B)
  // (batches of 13 independent 128-bit loads per thread before any is stored: one L2 round trip per batch)
  static_assert(WG_MC * 8 == 13 * THREADS, "staging loop assumes 13 loads per thread");
  {
    float4 v[13];
#pragma unroll
    for (int u = 0; u < 13; ++u) {
      const int i = threadIdx.x + u * THREADS;
      const int m = i >> 3, c = i & 7;
      v[u] = (m < mv) ? __ldg(reinterpret_cast<const float4*>(q.dy + (size_t)(m0 + m) * q.ldy + n0) + c)
                      : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int u = 0; u < 13; ++u) {
      const int i = threadIdx.x + u * THREADS;
      const int m = i >> 3, c = i & 7;
      At[(4 * c + 0) * WG_LDA + m] = v[u].x;
      At[(4 * c + 1) * WG_LDA + m] = v[u].y;
      At[(4 * c + 2) * WG_LDA + m] = v[u].z;
      At[(4 * c + 3) * WG_LDA + m] = v[u].w;
    }
  }
  __syncthreads();
  float* mypart = p.part + ((size_t)tile * p.nsplit + split) * (32 * 128 + 32);
  if (q.db != nullptr && k0 == 0) {         // bias gradient rides with the first k tile
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
    for (int rr = 0; rr < 4; ++rr) {
      const int n = warp * 4 + rr;
      float s = 0.f;
      for (int m = lane; m < WG_MC; m += 32) s += At[n * WG_LDA + m];
      s = warp_sum(s);
      if (lane == 0) mypart[32 * 128 + n] = s;
    }
  }
  panel_gemm<2, B_KN, WG_LDA>(At, q.x + (size_t)(mv > 0 ? m0 : 0) * q.ldx + k0, q.ldx, 128, WG_MC, mv, wst, nullptr,
                      [&](int r, int c, float v0, float v1) { *reinterpret_cast<float2*>(mypart + r * 128 + c) = make_float2(v0, v1); });
  if (!last_block_arrives(p.tickets + tile, p.nsplit)) return;
  const float* base = p.part + (size_t)tile * p.nsplit * (32 * 128 + 32);
  for (int i = threadIdx.x; i < 32 * 128; i += THREADS) {
    float s = 0.f;
    for (int z = 0; z < p.nsplit; ++z) s += __ldcg(base + (size_t)z * (32 * 128 + 32) + i);
    q.dw[(size_t)(n0 + (i >> 7)) * q.K + k0 + (i & 127)] = s;
  }
  if (q.db != nullptr && k0 == 0 && threadIdx.x < 32) {
    float s = 0.f;
    for (int z = 0; z < p.nsplit; ++z) s += __ldcg(base + (size_t)z * (32 * 128 + 32) + 32 * 128 + threadIdx.x);
    q.db[n0 + threadIdx.x] = s;
  }
}

static int set_smem(const void* fn, size_t bytes) {
  TMF_REQUIRE(bytes <= 227 * 1024, "encoder kernels: %zu bytes of shared memory needed", bytes);
  TMF_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  return 0;
}
// raise a kernel's dynamic shared-memory limit only when a call needs more than any earlier one
static int grow_smem(const void* fn, size_t bytes, size_t& cur) {
  if (bytes <= cur) return 0;
  if (set_smem(fn, bytes)) return 2;
  cur = bytes;
  return 0;
}

}  // namespace enc
}  // namespace tmf

using namespace tmf;
using namespace tmf::enc;

static int enc_check_ws(const char* who, void* ws, size_t ws_bytes) {
  TMF_REQUIRE(ws != nullptr && ws_bytes >= TMF_WS_BYTES && ((uintptr_t)ws & 255) == 0,
              "%s: needs the 256-byte aligned scratch buffer of tmf_scratch_bytes() bytes (tickets zero-initialised)", who);
  return 0;
}
// ticket slots of the encoder kernels inside the scratch buffer's ticket area (fusion_ops.cu uses [0, 4096) x 4 bytes of
// the 16 KB; here: the upper words)
static unsigned* enc_tickets(void* ws, int which) { return reinterpret_cast<unsigned*>(ws) + 3900 + which * 64; }
static float* enc_partials(void* ws) { return reinterpret_cast<float*>(reinterpret_cast<char*>(ws) + TMF_WS_TICKET_BYTES); }

extern "C" {

int tmf_encoder_supported(int dim, int inner, int mlp) {
  return (dim == 128 && inner == 128 && (mlp == 128 || mlp == 256 || mlp == 512)) ? 1 : 0;
}

size_t tmf_encoder_pack_bytes(int mlp) { return pack_elems(mlp) * sizeof(__nv_bfloat16); }

int tmf_encoder_pack_weights(const float* wq, const float* wkv, const float* wo, const float* w1, const float* w2, int mlp,
                             void* pack, void* stream) {
  TMF_REQUIRE(wq && wkv && wo && w1 && w2 && pack, "encoder_pack_weights: NULL pointer");
  TMF_REQUIRE(tmf_encoder_supported(128, 128, mlp), "encoder_pack_weights: mlp_dim %d not supported", mlp);
  TMF_REQUIRE(((uintptr_t)pack & 15) == 0, "encoder_pack_weights: pack must be 16-byte aligned");
  PackArgs p{};
  const float* w[5] = {wq, wkv, wo, w1, w2};
  const int numel[5] = {128 * 128, 256 * 128, 128 * 128, mlp * 128, 128 * mlp};
  const size_t off[5] = {pack_off_wq(), pack_off_wkv(), pack_off_wo(), pack_off_w1(), pack_off_w2(mlp)};
  for (int i = 0; i < 5; ++i) { p.w[i] = w[i]; p.numel[i] = numel[i]; p.off[i] = off[i]; }
  p.pack = (__nv_bfloat16*)pack;
  launch_k(enc_pack_kernel, dim3(16, 5), 256, 0, (cudaStream_t)stream, p);
  TMF_LAUNCH_CHECK();
  return 0;
}

int tmf_encoder_proj_fwd(const float* x, const float* ctx, const float* ln_w, const float* ln_b, const float* wq,
                         const float* wkv, float* h1, float* mean1, float* rstd1, float* q, float* kv, int Mx, int Mc,
                         float eps, const void* pack, void* stream) {
  TMF_REQUIRE(x && ctx && ln_w && ln_b && wq && wkv && h1 && mean1 && rstd1 && q && kv, "encoder_proj_fwd: NULL pointer");
  TMF_REQUIRE(Mx > 0 && Mc > 0, "encoder_proj_fwd: empty input");
  ProjFwdArgs p{x, ctx, ln_w, ln_b, wq, wkv, h1, mean1, rstd1, q, kv, Mx, Mc, ceil_div(Mx, PR), eps, (const __nv_bfloat16*)pack};
  const size_t smem = sizeof(float) * (PR * LD128 + PR * 260 + 2 * PR * LD128 + NSTAGE * WT_FLOATS);
  static bool done = false;
  if (!done) { if (set_smem((const void*)enc_proj_fwd_kernel, smem)) return 2; done = true; }
  launch_k(enc_proj_fwd_kernel, p.nbx + ceil_div(Mc, PR), THREADS, smem, (cudaStream_t)stream, p);
  TMF_LAUNCH_CHECK();
  return 0;
}

int tmf_encoder_chain_fwd(const float* o, const float* x, const float* wo, const float* bo, const float* ln2_w,
                          const float* ln2_b, const float* w1, const float* b1, const float* w2, const float* b2,
                          const float* lnf_w, const float* lnf_b, float* a, float* h2, float* mean2, float* rstd2,
                          float* pre, float* f, float* g, float* meanf, float* rstdf, float* y, int M, int mlp,
                          int add_input, float eps2, float epsf, const void* pack, void* stream) {
  TMF_REQUIRE(o && x && wo && bo && ln2_w && ln2_b && w1 && b1 && w2 && b2 && lnf_w && lnf_b && a && h2 && mean2 && rstd2 &&
                  pre && f && g && meanf && rstdf && y, "encoder_chain_fwd: NULL pointer");
  TMF_REQUIRE(tmf_encoder_supported(128, 128, mlp), "encoder_chain_fwd: mlp_dim %d not supported", mlp);
  {
    const int on = getenv("TMF_ENC_PROF") != nullptr ? 1 : 0;
    static int cur = -1;
    if (on != cur) { cudaMemcpyToSymbol(g_enc_prof, &on, sizeof(int)); cur = on; }
  }
  ChainFwdArgs p{o, x, wo, bo, ln2_w, ln2_b, w1, b1, w2, b2, lnf_w, lnf_b, a, h2, mean2, rstd2, pre, f, g, meanf, rstdf, y,
                 M, mlp, add_input, getenv("TMF_ENC_PROF") != nullptr ? 1 : 0, eps2, epsf, (const __nv_bfloat16*)pack};
  const size_t smem = sizeof(float) * (3 * PR * LD128 + 3 * PR * (mlp + 4) + NSTAGE * WT_FLOATS);
#define TMF_LAUNCH_CHAIN_FWD(MLPV)                                                                                 \
  do {                                                                                                            \
    static bool done = false;                                                                                     \
    if (!done) { if (set_smem((const void*)enc_chain_fwd_kernel<MLPV>, smem)) return 2; done = true; }            \
    launch_k(enc_chain_fwd_kernel<MLPV>, ceil_div(M, PR), THREADS, smem, (cudaStream_t)stream, p);                      \
  } while (0)
  if (mlp == 128) TMF_LAUNCH_CHAIN_FWD(128);
  else if (mlp == 256) TMF_LAUNCH_CHAIN_FWD(256);
  else TMF_LAUNCH_CHAIN_FWD(512);
#undef TMF_LAUNCH_CHAIN_FWD
  TMF_LAUNCH_CHECK();
  return 0;
}

int tmf_encoder_chain_bwd(const float* dy, const float* g, const float* a, const float* pre, const float* wo,
                          const float* w1, const float* w2, const float* ln2_w, const float* lnf_w, const float* mean2,
                          const float* rstd2, const float* meanf, const float* rstdf, float* dg, float* dp, float* da,
                          float* dout, float* dxp, float* dlnf_w, float* dlnf_b, float* dln2_w, float* dln2_b, int M,
                          int mlp, int add_input, const void* pack, void* ws, size_t ws_bytes, void* stream) {
  TMF_REQUIRE(dy && g && a && pre && wo && w1 && w2 && ln2_w && lnf_w && mean2 && rstd2 && meanf && rstdf && dg && dp && da &&
                  dout && dxp && dlnf_w && dlnf_b && dln2_w && dln2_b, "encoder_chain_bwd: NULL pointer");
  TMF_REQUIRE(tmf_encoder_supported(128, 128, mlp), "encoder_chain_bwd: mlp_dim %d not supported", mlp);
  if (enc_check_ws("encoder_chain_bwd", ws, ws_bytes)) return 1;
  const int nb = ceil_div(M, PR);
  TMF_REQUIRE((size_t)nb * 512 * sizeof(float) <= TMF_WS_BYTES - TMF_WS_TICKET_BYTES, "encoder_chain_bwd: too many rows");
  ChainBwdArgs p{dy, g, a, pre, wo, w1, w2, ln2_w, lnf_w, mean2, rstd2, meanf, rstdf, dg, dp, da, dout, dxp,
                 dlnf_w, dlnf_b, dln2_w, dln2_b, enc_partials(ws), enc_tickets(ws, 0), M, mlp, add_input, (const __nv_bfloat16*)pack};
  const size_t smem = sizeof(float) * (3 * PR * LD128 + 3 * PR * (mlp + 4) + NSTAGE * WT_FLOATS + 512);
#define TMF_LAUNCH_CHAIN_BWD(MLPV)                                                                                 \
  do {                                                                                                            \
    static bool done = false;                                                                                     \
    if (!done) { if (set_smem((const void*)enc_chain_bwd_kernel<MLPV>, smem)) return 2; done = true; }            \
    launch_k(enc_chain_bwd_kernel<MLPV>, nb, THREADS, smem, (cudaStream_t)stream, p);                                   \
  } while (0)
  if (mlp == 128) TMF_LAUNCH_CHAIN_BWD(128);
  else if (mlp == 256) TMF_LAUNCH_CHAIN_BWD(256);
  else TMF_LAUNCH_CHAIN_BWD(512);
#undef TMF_LAUNCH_CHAIN_BWD
  TMF_LAUNCH_CHECK();
  return 0;
}

int tmf_encoder_proj_bwd(const float* dq, const float* dkv, const float* dxp, const float* x, const float* ln_w,
                         const float* mean1, const float* rstd1, const float* wq, const float* wkv, float* dx, float* dctx,
                         float* dln_w, float* dln_b, int Mx, int Mc, const void* pack, void* ws, size_t ws_bytes, void* stream) {
  TMF_REQUIRE(dq && dkv && dxp && x && ln_w && mean1 && rstd1 && wq && wkv && dx && dctx && dln_w && dln_b,
              "encoder_proj_bwd: NULL pointer");
  if (enc_check_ws("encoder_proj_bwd", ws, ws_bytes)) return 1;
  ProjBwdArgs p{dq, dkv, dxp, x, ln_w, mean1, rstd1, wq, wkv, dx, dctx, dln_w, dln_b, enc_partials(ws), enc_tickets(ws, 1),
                Mx, Mc, ceil_div(Mx, PR), (const __nv_bfloat16*)pack};
  TMF_REQUIRE((size_t)p.nbx * 256 * sizeof(float) <= TMF_WS_BYTES - TMF_WS_TICKET_BYTES, "encoder_proj_bwd: too many rows");
  const size_t smem = sizeof(float) * (PR * 260 + 2 * PR * LD128 + 2 * PR * 260 + NSTAGE * WT_FLOATS + 256);
  static bool done = false;
  if (!done) { if (set_smem((const void*)enc_proj_bwd_kernel, smem)) return 2; done = true; }
  launch_k(enc_proj_bwd_kernel, p.nbx + ceil_div(Mc, PR), THREADS, smem, (cudaStream_t)stream, p);
  TMF_LAUNCH_CHECK();
  return 0;
}

/* t[15] = {dq, h1, dWq,  dkv, ctx, dWkv,  da, o, dWo, dbo,  dp, h2, dW1, db1,  dg}; f, dW2, db2 follow as arguments */
int tmf_encoder_wgrad(const void* const* t, const float* f, float* dw2, float* db2, int Mx, int Mc, int mlp, void* ws,
                      size_t ws_bytes, void* stream) {
  TMF_REQUIRE(t != nullptr && f && dw2 && db2, "encoder_wgrad: NULL pointer");
  for (int i = 0; i < 15; ++i) TMF_REQUIRE(t[i] != nullptr, "encoder_wgrad: NULL tensor %d", i);
  TMF_REQUIRE(tmf_encoder_supported(128, 128, mlp), "encoder_wgrad: mlp_dim %d not supported", mlp);
  if (enc_check_ws("encoder_wgrad", ws, ws_bytes)) return 1;
  WgradArgs p{};
  auto F = [&](int i) { return (const float*)t[i]; };
  auto G = [&](int i) { return (float*)const_cast<void*>(t[i]); };
  p.pr[0] = WgradProblem{F(0), F(1), G(2), nullptr, 128, 128, 128, 128, Mx, 0};
  p.pr[1] = WgradProblem{F(3), F(4), G(5), nullptr, 256, 128, 256, 128, Mc, 0};
  p.pr[2] = WgradProblem{F(6), F(7), G(8), G(9), 128, 128, 128, 128, Mx, 0};
  p.pr[3] = WgradProblem{F(10), F(11), G(12), G(13), mlp, 128, mlp, 128, Mx, 0};
  p.pr[4] = WgradProblem{F(14), f, dw2, db2, 128, mlp, 128, mlp, Mx, 0};
  int tiles = 0;
  for (int i = 0; i < WG_PROBLEMS; ++i) {
    p.pr[i].tile0 = tiles;
    tiles += (p.pr[i].N / 32) * (p.pr[i].K / 128);
  }
  p.ntiles = tiles;
  p.nsplit = ceil_div(Mx > Mc ? Mx : Mc, WG_MC);
  TMF_REQUIRE(tiles <= 64, "encoder_wgrad: too many tiles");
  TMF_REQUIRE((size_t)tiles * p.nsplit * (32 * 128 + 32) * sizeof(float) <= TMF_WS_BYTES - TMF_WS_TICKET_BYTES,
              "encoder_wgrad: token count too large for the scratch buffer");
  p.part = enc_partials(ws);
  p.tickets = enc_tickets(ws, 2);
  const size_t smem = sizeof(float) * (32 * WG_LDA + NSTAGE * WT_FLOATS);
  static bool done = false;
  if (!done) { if (set_smem((const void*)enc_wgrad_kernel, smem)) return 2; done = true; }
  launch_k(enc_wgrad_kernel, tiles * p.nsplit, THREADS, smem, (cudaStream_t)stream, p);
  TMF_LAUNCH_CHECK();
  return 0;
}

}  // extern "C"

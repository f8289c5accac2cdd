// adam.cu -- fused multi-tensor Adam step (SURVEY.md section 8f row 1; replaces the ~200 small launches of
// torch.optim.Adam(capturable=True) that the reference's getOptimizer (utils/utils.py:38-41) issues per step).
// One launch updates every parameter: the host builds, once, a device table of chunks {p, g, m, v, n}; the step count
// and the learning rate live on the device (CUDA-graph replays must not bake them in), and the step counter is advanced
// by the last block to finish.  Arithmetic follows torch.optim.Adam exactly (amsgrad = False, maximize = False):
//   g' = g + wd * p;  m = b1*m + (1-b1)*g';  v = b2*v + (1-b2)*g'^2;
//   p -= (lr / (1 - b1^t)) * m / (sqrt(v) / sqrt(1 - b2^t) + eps)
#include "common.cuh"

namespace tmf {

// A chunk of a Conv3d weight (Cout,Cin,k,k,k) may carry the bf16 operand packs of the conv kernels: the updated value is
// also written to wf[tap][Cout][Cin] (forward operand) and wd[taps-1-tap][Cin][Cout] (dgrad operand), which removes the
// per-step tmf_pack_conv_weights launches from the train step (SURVEY.md section 8f row 1).
struct AdamChunk {
  float* p;
  const float* g;
  float* m;
  float* v;
  __nv_bfloat16* wf;       // NULL: no packs
  __nv_bfloat16* wd;       // may be NULL
  int32_t n;
  int32_t off;             // element offset of this chunk inside its tensor (pack index arithmetic)
  int32_t cout, cin, taps;
  int32_t tile;            // 1: the chunk is an ADAM_TCO x ADAM_TCI block of (co, ci) pairs with all taps (p/g/m/v = tensor base,
                           // off = co0 * cin + ci0): the pack stores leave through shared memory as whole 32 / 64-byte segments
                           // 2: weight of a fused transformer encoder: wf / wd are its bf16 hi / lo arrays (enc_fused.cu's operand
                           // pack, same element order as the parameter): hi = bf16(p), lo = bf16(p - hi) at index off + i
};
constexpr int ADAM_TCO = 16, ADAM_TCI = 32, ADAM_MAX_TAPS = 27;
static_assert(sizeof(AdamChunk) == 72, "host code packs 72-byte chunk records");

__device__ __forceinline__ void emit_pack(const AdamChunk& c, int i, float val) {
  const int idx = c.off + i;
  const int t = idx % c.taps;
  const int r = idx / c.taps;
  const int ci = r % c.cin, co = r / c.cin;
  const __nv_bfloat16 b = __float2bfloat16_rn(val);
  c.wf[((size_t)t * c.cout + co) * c.cin + ci] = b;
  if (c.wd != nullptr) c.wd[((size_t)(c.taps - 1 - t) * c.cin + ci) * c.cout + co] = b;
}

__global__ void __launch_bounds__(256) adam_multi_kernel(const AdamChunk* __restrict__ chunks, const float* __restrict__ lr_dev,
                                                         float b1, float b2, float eps, float wd, float* step_dev,
                                                         unsigned* ticket) {
  const AdamChunk c = chunks[blockIdx.x];
  const float t = step_dev[0] + 1.f;              // step_dev is only advanced after every block has read it (ticket below)
  const float lr = lr_dev[0];
  const float bc1 = 1.f - powf(b1, t), bc2 = 1.f - powf(b2, t);
  const float step_size = lr / bc1;
  const float inv_sqrt_bc2 = rsqrtf(bc2);
  if (c.tile == 1) {
    // Conv weight with operand packs.  The element-wise version scattered two 2-byte stores per element (wf is [tap][co][ci],
    // wd [tap'][ci][co], the parameter [co][ci][tap]): 16x write amplification made this kernel 95 us for 117 MB (ncu r2p).
    __shared__ __nv_bfloat16 tl[ADAM_TCO * ADAM_TCI * ADAM_MAX_TAPS];     // [co][ci][tap]
    const int taps = c.taps, seg = ADAM_TCI * taps;
    const int co0 = c.off / c.cin, ci0 = c.off - co0 * c.cin;
    for (int e = threadIdx.x; e < ADAM_TCO * seg; e += 256) {
      const int row = e / seg, col = e - row * seg;
      const size_t gi = ((size_t)(co0 + row) * c.cin + ci0) * taps + col;
      const float g = fmaf(wd, c.p[gi], c.g[gi]);
      const float m = fmaf(b1, c.m[gi], (1.f - b1) * g);
      const float v = fmaf(b2, c.v[gi], (1.f - b2) * g * g);
      c.m[gi] = m;
      c.v[gi] = v;
      const float pn = c.p[gi] - step_size * (m / (sqrtf(v) * inv_sqrt_bc2 + eps));
      c.p[gi] = pn;
      tl[e] = __float2bfloat16_rn(pn);
    }
    __syncthreads();
    constexpr int NR = ADAM_TCO * ADAM_TCI;
    for (int o = threadIdx.x; o < NR * taps; o += 256) {
      const int t = o / NR, r = o - t * NR;
      const int co = r / ADAM_TCI, ci = r - co * ADAM_TCI;                // ci fastest: 64-byte runs of wf
      c.wf[((size_t)t * c.cout + co0 + co) * c.cin + ci0 + ci] = tl[(co * ADAM_TCI + ci) * taps + t];
    }
    if (c.wd != nullptr) {
      for (int o = threadIdx.x; o < NR * taps; o += 256) {
        const int t = o / NR, r = o - t * NR;
        const int ci = r / ADAM_TCO, co = r - ci * ADAM_TCO;              // co fastest: 32-byte runs of wd
        c.wd[((size_t)(taps - 1 - t) * c.cin + ci0 + ci) * c.cout + co0 + co] = tl[(co * ADAM_TCI + ci) * taps + t];
      }
    }
  }
  const bool vec = c.tile != 1 && ((((uintptr_t)c.p | (uintptr_t)c.g | (uintptr_t)c.m | (uintptr_t)c.v) & 15) == 0);
  const int n4 = vec ? (c.n >> 2) : 0;
  for (int i = threadIdx.x; i < n4; i += 256) {
    float4 p4 = reinterpret_cast<float4*>(c.p)[i];
    const float4 g4 = reinterpret_cast<const float4*>(c.g)[i];
    float4 m4 = reinterpret_cast<float4*>(c.m)[i];
    float4 v4 = reinterpret_cast<float4*>(c.v)[i];
    float* pp = &p4.x; const float* gp = &g4.x; float* mp = &m4.x; float* vp = &v4.x;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float g = fmaf(wd, pp[j], gp[j]);
      mp[j] = fmaf(b1, mp[j], (1.f - b1) * g);
      vp[j] = fmaf(b2, vp[j], (1.f - b2) * g * g);
      pp[j] -= step_size * (mp[j] / (sqrtf(vp[j]) * inv_sqrt_bc2 + eps));
      if (c.tile == 0 && c.wf != nullptr) emit_pack(c, 4 * i + j, pp[j]);
    }
    if (c.tile == 2) {                               // (c.off and the chunk size are multiples of 4: 8-byte stores)
      const uint32_t h01 = pack_bf16(p4.x, p4.y), h23 = pack_bf16(p4.z, p4.w);
      const uint32_t l01 = pack_bf16(p4.x - bf16_lo(h01), p4.y - bf16_hi(h01));
      const uint32_t l23 = pack_bf16(p4.z - bf16_lo(h23), p4.w - bf16_hi(h23));
      *reinterpret_cast<uint2*>(c.wf + c.off + 4 * i) = make_uint2(h01, h23);
      *reinterpret_cast<uint2*>(c.wd + c.off + 4 * i) = make_uint2(l01, l23);
    }
    reinterpret_cast<float4*>(c.p)[i] = p4;
    reinterpret_cast<float4*>(c.m)[i] = m4;
    reinterpret_cast<float4*>(c.v)[i] = v4;
  }
  for (int i = n4 * 4 + threadIdx.x; i < (c.tile == 1 ? 0 : c.n); i += 256) {
    const float g = fmaf(wd, c.p[i], c.g[i]);
    const float m = fmaf(b1, c.m[i], (1.f - b1) * g);
    const float v = fmaf(b2, c.v[i], (1.f - b2) * g * g);
    c.m[i] = m;
    c.v[i] = v;
    const float pn = c.p[i] - step_size * (m / (sqrtf(v) * inv_sqrt_bc2 + eps));
    c.p[i] = pn;
    if (c.tile == 2) {
      const __nv_bfloat16 hb = __float2bfloat16_rn(pn);
      c.wf[c.off + i] = hb;
      c.wd[c.off + i] = __float2bfloat16_rn(pn - __bfloat162float(hb));
    } else if (c.wf != nullptr) emit_pack(c, i, pn);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    const unsigned done = atomicAdd(ticket, 1u);
    if (done == gridDim.x - 1) {
      step_dev[0] = t;
      *ticket = 0u;
    }
  }
}

}  // namespace tmf

using namespace tmf;

extern "C" {

int tmf_adam_chunk_bytes(void) { return (int)sizeof(AdamChunk); }

int tmf_adam_step(const void* chunks, int nchunks, const float* lr_dev, float beta1, float beta2, float eps,
                  float weight_decay, float* step_dev, void* ticket_dev, void* stream) {
  TMF_REQUIRE(chunks != nullptr && lr_dev != nullptr && step_dev != nullptr && ticket_dev != nullptr,
              "adam_step: NULL device pointer");
  TMF_REQUIRE(nchunks > 0, "adam_step: empty chunk table");
  TMF_REQUIRE(beta1 >= 0.f && beta1 < 1.f && beta2 >= 0.f && beta2 < 1.f && eps >= 0.f, "adam_step: bad hyper-parameters");
  launch_k(adam_multi_kernel, nchunks, 256, 0, (cudaStream_t)stream, (const AdamChunk*)chunks, lr_dev, beta1, beta2, eps,
                                                               weight_decay, step_dev, (unsigned*)ticket_dev);
  TMF_LAUNCH_CHECK();
  return 0;
}

}  // extern "C"

// common.cuh -- shared helpers for libtmf_sm100a (error plumbing, grouped pointers, bf16 packing).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/tmf.h"

namespace tmf {

void set_error(const char* fmt, ...);
void count_launch(int n = 1);

// One pointer per group (sNet tower); passed to kernels by value, indexed with blockIdx.z.
template <typename T>
struct GroupPtr {
  T* p[TMF_MAX_GROUPS];
};

template <typename T>
static inline bool load_group(GroupPtr<T>& g, T* const* host, int ng, bool required, const char* name) {
  for (int i = 0; i < TMF_MAX_GROUPS; ++i) g.p[i] = nullptr;
  if (host == nullptr) {
    if (required) { set_error("%s: NULL pointer array", name); return false; }
    return true;
  }
  for (int i = 0; i < ng; ++i) {
    g.p[i] = host[i];
    if (required && host[i] == nullptr) { set_error("%s[%d]: NULL device pointer", name, i); return false; }
  }
  return true;
}

#define TMF_CHECK_NG(ng)                                                          \
  do {                                                                            \
    if ((ng) < 1 || (ng) > TMF_MAX_GROUPS) {                                      \
      tmf::set_error("%s: ng=%d out of range [1,%d]", __func__, (ng), TMF_MAX_GROUPS); \
      return 1;                                                                   \
    }                                                                             \
  } while (0)

#define TMF_REQUIRE(cond, ...)            \
  do {                                    \
    if (!(cond)) {                        \
      tmf::set_error(__VA_ARGS__);        \
      return 1;                           \
    }                                     \
  } while (0)

#define TMF_CUDA(expr)                                                                     \
  do {                                                                                     \
    cudaError_t _e = (expr);                                                               \
    if (_e != cudaSuccess) {                                                               \
      tmf::set_error("%s:%d %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
      return 2;                                                                            \
    }                                                                                      \
  } while (0)

#define TMF_LAUNCH_CHECK()                                                              \
  do {                                                                                  \
    cudaError_t _e = cudaGetLastError();                                                \
    if (_e != cudaSuccess) {                                                            \
      tmf::set_error("%s:%d launch failed: %s", __FILE__, __LINE__, cudaGetErrorString(_e)); \
      return 3;                                                                         \
    }                                                                                   \
    tmf::count_launch();                                                                \
  } while (0)

static inline int ceil_div(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

// The single launch helper of the library: a plain cudaLaunchKernelEx with the arguments converted to the kernel's
// parameter types.
template <typename... KArgs, typename... Args>
static inline cudaError_t launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                   Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// Zero one `bytes`-sized buffer per group; adjacent buffers (callers that carve the towers' buffers out of one
// allocation) are cleared by a single memset node.
static inline cudaError_t zero_group_buffers(void* const* bufs, int ng, size_t bytes, cudaStream_t st) {
  int g = 0;
  while (g < ng) {
    if (bufs[g] == nullptr) { ++g; continue; }
    int e = g + 1;
    while (e < ng && bufs[e] == (char*)bufs[g] + (size_t)(e - g) * bytes) ++e;
    cudaError_t err = cudaMemsetAsync(bufs[g], 0, bytes * (size_t)(e - g), st);
    if (err != cudaSuccess) return err;
    g = e;
  }
  return cudaSuccess;
}

// ---- device helpers -------------------------------------------------------------------------------------
// Deterministic cross-CTA statistics (include/tmf.h, DETERMINISM): CTA `part` of the `nparts` (<= TMF_STAT_ROWS) CTAs that
// produce column `col` of a double[TMF_STAT_ROWS][ncols] buffer owns row `part` and clears rows part + k*nparts, so
// every row is written exactly once per launch: no memset by the caller, no atomics, fixed-order sum in the finalize.
__device__ __forceinline__ void stat_row_store(double* buf, int ncols, int part, int nparts, int col, double v) {
  buf[(size_t)part * ncols + col] = v;
  for (int r = part + nparts; r < TMF_STAT_ROWS; r += nparts) buf[(size_t)r * ncols + col] = 0.0;
}

// "Last block" rendezvous for deterministic cross-block reductions without a second launch: every block stores its partial
// result to global scratch and calls this (all threads); it returns true in exactly one block -- the last of `nblocks` to
// arrive -- after the other blocks' stores are visible to it, and re-zeroes the ticket for the next launch.  The caller's
// last block then adds the partials in block-index order.  `ticket` must be zero before the first launch ever.
__device__ __forceinline__ bool last_block_arrives(unsigned* ticket, unsigned nblocks) {
  __shared__ int s_is_last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned t = atomicAdd(ticket, 1u);
    s_is_last = (t == nblocks - 1u) ? 1 : 0;
    if (s_is_last) *ticket = 0u;
  }
  __syncthreads();
  const bool last = s_is_last != 0;
  if (last) __threadfence();
  return last;
}

// Layout of the caller-owned scratch buffer (`ws`) of the fusion-transformer entry points: tickets first (zero before the
// first use, left zero by every kernel), then partial results.  tmf_scratch_bytes() is the size callers allocate.
constexpr size_t TMF_WS_TICKET_BYTES = 16384;                 // 4096 tickets: [0,1024) LayerNorm, [1024,3072) GEMM tiles, [3072,4096) column sums
constexpr size_t TMF_WS_BYTES = (size_t)16 << 20;

// Packed fp32 pairs in one 64-bit register (sm_100: FADD2 / FFMA2 issue two fp32 operations per slot).
__device__ __forceinline__ uint64_t pair_u32(uint32_t lo, uint32_t hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "r"(lo), "r"(hi));
  return r;
}
__device__ __forceinline__ uint64_t pair_f32(float lo, float hi) { return pair_u32(__float_as_uint(lo), __float_as_uint(hi)); }
__device__ __forceinline__ uint32_t lo_u32(uint64_t v) {
  uint32_t lo, hi;
  asm("mov.b64 {%0, %1}, %2;" : "=r"(lo), "=r"(hi) : "l"(v));
  return lo;
}
__device__ __forceinline__ uint32_t hi_u32(uint64_t v) {
  uint32_t lo, hi;
  asm("mov.b64 {%0, %1}, %2;" : "=r"(lo), "=r"(hi) : "l"(v));
  return hi;
}
__device__ __forceinline__ uint64_t add2_f32(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ uint64_t sub2_f32(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ uint64_t fma2_f32(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
__device__ __forceinline__ float bf16_lo(uint32_t v) { return __uint_as_float(v << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t v) { return __uint_as_float(v & 0xffff0000u); }
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&t);
}
__device__ __forceinline__ float round_bf16(float v) { return __bfloat162float(__float2bfloat16_rn(v)); }

__device__ __forceinline__ void unpack8(const uint4& v, float* f) {
  f[0] = bf16_lo(v.x); f[1] = bf16_hi(v.x);
  f[2] = bf16_lo(v.y); f[3] = bf16_hi(v.y);
  f[4] = bf16_lo(v.z); f[5] = bf16_hi(v.z);
  f[6] = bf16_lo(v.w); f[7] = bf16_hi(v.w);
}
__device__ __forceinline__ uint4 pack8(const float* f) {
  uint4 v;
  v.x = pack_bf16(f[0], f[1]);
  v.y = pack_bf16(f[2], f[3]);
  v.z = pack_bf16(f[4], f[5]);
  v.w = pack_bf16(f[6], f[7]);
  return v;
}

// LRP's stabilised ratio (lrp.cu, conv1_dgrad.cu): r / (z + eps*sign(z)) with sign(0) = +1, and 0 where that denominator is 0
__device__ __forceinline__ float lrp_div(float r, float z, float eps) {
  const float st = __fadd_rn(z, z >= 0.f ? eps : -eps);
  return st != 0.f ? __fdiv_rn(r, st) : 0.f;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

}  // namespace tmf

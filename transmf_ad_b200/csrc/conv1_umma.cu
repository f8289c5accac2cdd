// conv1_umma.cu -- conv1.0 (Cin = 1, 3x3x3, pad 1; reference models/networks.py:22) on the tcgen05 tensor cores.
//
// The layer is only 26 FLOP/byte, but on CUDA cores it is FMA-issue bound (864 FMAs per voxel).  Here the 27-tap
// neighbourhood of every voxel is written by producer warps as one K = 32 row of an im2col tile in shared memory
// (K-major, 64-byte rows, 64B swizzle -- the layout a TMA box would have produced), and a [128 voxels x Cout x 32]
// GEMM runs on tcgen05 with the accumulator in TMEM.  fp32 fidelity is kept with a bf16 hi/lo split of BOTH operands:
//     x*w ~= xh*wh + xl*wh + xh*wl        (dropped term xl*wl ~ 2^-16 relative)
// i.e. three MMAs per K step; the image is never rounded to bf16 (SURVEY.md section 8c: that costs ~10x logit error).
// Epilogue as in conv_umma.cu: +bias, round to bf16, 16-byte stores, BatchNorm sum / sum-of-squares of the stored values.
#include <cuda.h>

#include "common.cuh"
#include "umma.cuh"

namespace tmf {
using namespace umma;

constexpr int C1U_PRODUCERS = 128;                 // one im2col row (voxel) per thread; two producer groups (warps 0-3,
                                                   // 4-7) alternate tiles so global-load latency of one hides behind the other
constexpr int C1U_THREADS = 640;                   // + warps 8, 14: MMA issuers (8 owns TMEM), 9-12 and 16-19: epilogue, 13: image loader
constexpr int C1U_STAGES = 8;                      // im2col tile pairs in flight (16 KB each)
constexpr int C1U_ACC = 4;                         // TMEM accumulator buffers
constexpr int C1U_XS = 8;                          // staged image slots (tiles in flight ahead of the producers)
constexpr uint32_t C1U_TILE_BYTES = 128 * 64;      // one [128 x 32] bf16 operand tile

struct C1UParams {
  const float* x[TMF_MAX_GROUPS];
  const float* w[TMF_MAX_GROUPS];
  const float* bias[TMF_MAX_GROUPS];
  __nv_bfloat16* y[TMF_MAX_GROUPS];
  double* stats[TMF_MAX_GROUPS];
  int ng, B, D, H, W, cout;
  long long M;
  int ntiles;
  uint32_t idesc, tmem_cols;
  int xs_seg;         // STAGED: floats per staged window (one per kd): 2 W + 130 + alignment slack, multiple of 4
  int debug;          // timing-only bring-up switches (TMF_C1U_DEBUG): 1 = one MMA pair instead of three, 2 = no stores,
                      // 4 = no image loads (unstaged path), 32 = role timing printed by block 0.
                      // Results are wrong with 1 / 2 / 4 set.
};

// byte offset of 16-byte chunk j of row r inside a K-major, 64-byte-row, 64B-swizzled tile (tile base 1024-aligned)
__device__ __forceinline__ uint32_t sw64_off(int r, int j) { return (uint32_t)r * 64u + (uint32_t)((j ^ ((r >> 1) & 3)) << 4); }

// bring-up instrumentation (debug & 32): cycles a role spends blocked on one kind of barrier
__device__ __forceinline__ void c1u_wait_t(uint32_t bar, uint32_t parity, long long& acc, bool on) {
  if (!on) { mbar_wait(bar, parity); return; }
  const long long t0 = clock64();
  mbar_wait(bar, parity);
  acc += clock64() - t0;
}

__device__ __forceinline__ void split_bf16(float v, float& hi, float& lo) {
  hi = round_bf16(v);
  lo = v - hi;
}

// NCH = Cout / 32 (1 for dim 128, the benchmark path; 2 for dim 256 -- that variant spills some statistics registers)
//
// STAGED (the normal path): the 27 taps of a tile's 128 consecutive voxels live in three contiguous windows of the flat
// image, one per kd:  [m0 - 1 - W + (kd-1) H W,  + 2 W + 130).  Three lanes of a loader warp copy the windows of every tile
// into shared memory with cp.async.bulk (completion on an mbarrier, C1U_XS tiles ahead) and the producers read their taps
// with shared-memory loads: ncu of the unstaged producers (27 __ldg per voxel, one tile ahead) showed 50 % of all stall
// samples on the first use of those loads (profiles/r2_conv1_notes.md).  The kernel is bound by instruction issue
// (2200 warp instructions per tile), so the copies must not cost the producers instructions: issuing them as 16-byte
// cp.async from the producer threads themselves (+30 instructions per thread and tile) was measured SLOWER than no staging.
// !STAGED keeps the direct loads for images whose base address is not 16-byte aligned or whose rows are too wide.
template <int NCH, bool STAGED>
__global__ void __launch_bounds__(C1U_THREADS, 1) conv1_umma_fwd_kernel(const __grid_constant__ C1UParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gen = smem_raw + (smem_base - smem_u32(smem_raw));
  // layout: [stages][A_hi | A_lo] (16 KB each) | W_hi | W_lo (cout x 64 B each, 4 KB reserved each) | barriers | stats
  const uint32_t smA = smem_base;
  const uint32_t smW = smA + C1U_STAGES * 2 * C1U_TILE_BYTES;
  const uint32_t bars = smW + 2 * 4096;
  const uint32_t full = bars, empty = bars + 8 * C1U_STAGES, acc_full = empty + 8 * C1U_STAGES, acc_empty = acc_full + 8 * C1U_ACC;
  const uint32_t tmem_slot = acc_empty + 8 * C1U_ACC;
  float* stats_ptr = reinterpret_cast<float*>(gen + (tmem_slot + 16 - smem_base));        // float [4 warps][2][64]
  const uint32_t xfull = tmem_slot + 16 + 2048, xempty = xfull + 8 * C1U_XS;
  const uint32_t xs_sm = xempty + 8 * C1U_XS;                                               // float [C1U_XS][3][xs_seg]
  const uint32_t xs_slot_bytes = 3u * (uint32_t)p.xs_seg * 4u;
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(gen + (tmem_slot - smem_base));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = blockIdx.x % p.ng;
  const int cta = blockIdx.x / p.ng, ncta = gridDim.x / p.ng;

  if (threadIdx.x == 0) {
    for (int i = 0; i < C1U_STAGES; ++i) { mbar_init(full + 8 * i, C1U_PRODUCERS); mbar_init(empty + 8 * i, 1); }
    for (int i = 0; i < C1U_ACC; ++i) { mbar_init(acc_full + 8 * i, 1); mbar_init(acc_empty + 8 * i, 256); }
    for (int i = 0; i < C1U_XS; ++i) { mbar_init(xfull + 8 * i, 3); mbar_init(xempty + 8 * i, C1U_PRODUCERS); }
    fence_barrier_init();
  }
  // weights: fp32 (Cout,27) -> bf16 hi / lo tiles, K-major rows of 32 taps (taps 27..31 zero)
  for (int i = threadIdx.x; i < p.cout * 4; i += C1U_THREADS) {
    const int co = i >> 2, j = i & 3;
    float hi[8], lo[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int t = j * 8 + e;
      float v = (t < 27) ? p.w[g][co * 27 + t] : 0.f;
      if (t == 27 && p.bias[g] != nullptr) v = p.bias[g][co];      // bias rides on K column 27 (im2col value 1)
      split_bf16(v, hi[e], lo[e]);
    }
    *reinterpret_cast<uint4*>(gen + (smW - smem_base) + sw64_off(co, j)) = pack8(hi);
    *reinterpret_cast<uint4*>(gen + (smW + 4096 - smem_base) + sw64_off(co, j)) = pack8(lo);
  }
  fence_proxy_async();
  if (warp == 8) {
    tmem_alloc(tmem_slot, p.tmem_cols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;
  const bool prof = (p.debug & 32) != 0;
  const long long t_start = clock64();
  long long t_w0 = 0, t_w1 = 0, t_w2 = 0;

  if (warp < 8) {
    // ======================================= im2col producers =======================================
    // Software-pipelined: the 27 loads of a thread's NEXT tile are in flight while the current row is split into
    // bf16 hi / lo and written, so one producer group alone already overlaps global latency with ALU work; the two
    // groups (alternating tiles) then overlap each other's barrier waits.  Voxel coordinates advance incrementally
    // (no div / mod in the loop).
    const int grp = warp >> 2;                       // producer group: handles every other tile of this CTA
    const int r = threadIdx.x & 127;                 // row of the tile
    const float* xg = p.x[g];
    const unsigned W = (unsigned)p.W, H = (unsigned)p.H, D = (unsigned)p.D;
    const unsigned M32 = (unsigned)p.M;              // host guarantees M < 2^31
    const int sH = (int)(W * H), sW = (int)W;
    const unsigned stride = 256u * (unsigned)ncta;   // voxels between consecutive tiles of this group
    const unsigned st_w = stride % W, st_t = stride / W, st_h = st_t % H, st_d = (st_t / H) % D;
    unsigned m = (unsigned)(cta + grp * ncta) * 128u + (unsigned)r;
    unsigned wq = m % W, hq = (m / W) % H, dq = (m / (W * H)) % D;
    // STAGED: word offset of tap (kd, kh, kw = 0) of row 0 inside a staging slot (warp-uniform).  The window of kd starts
    // at the aligned-down flat index of voxel (row 0, kh = 0, kw = 0); tiles start at multiples of 128, so the alignment
    // remainder is the same for every tile.
    int uoff[9];
    if (STAGED) {
#pragma unroll
      for (int kd = 0; kd < 3; ++kd)
#pragma unroll
        for (int kh = 0; kh < 3; ++kh) uoff[kd * 3 + kh] = kd * p.xs_seg + ((-1 - sW + (kd - 1) * sH) & 3) + kh * sW;
    }
    auto tap_mask = [&](bool (&dok)[3], bool (&hok)[3], bool (&wok)[3]) {
      const bool in_range = m < M32;
      dok[0] = in_range && dq > 0; dok[1] = in_range; dok[2] = in_range && dq + 1 < D;
      hok[0] = hq > 0; hok[1] = true; hok[2] = hq + 1 < H;
      wok[0] = wq > 0; wok[1] = true; wok[2] = wq + 1 < W;
      return in_range;
    };
    float nxt[28];
    auto load_row = [&](float (&v)[28]) {            // !STAGED: straight from global memory
      bool dok[3], hok[3], wok[3];
      v[27] = tap_mask(dok, hok, wok) ? 1.f : 0.f;   // bias column; rows past the end stay all-zero
      const float* xp = xg + m;
#pragma unroll
      for (int kd = 0; kd < 3; ++kd)
#pragma unroll
        for (int kh = 0; kh < 3; ++kh)
#pragma unroll
          for (int kw = 0; kw < 3; ++kw) {
            const bool ok = dok[kd] && hok[kh] && wok[kw];
            v[(kd * 3 + kh) * 3 + kw] = (ok && !(p.debug & 4)) ? __ldg(xp + (kd - 1) * sH + (kh - 1) * sW + (kw - 1)) : 0.f;
          }
    };
    // Unconditional shared-memory loads (every tap address lies inside the slot), then the boundary masks as AND words:
    // 27 LDS + 27 LOP3 instead of 27 predicated loads with their predicate logic, address arithmetic and zero-initialisation.
    auto load_row_staged = [&](uint32_t (&v)[28], uint32_t slot_sm) {
      const uint32_t* sp = reinterpret_cast<const uint32_t*>(gen + (slot_sm - smem_base)) + r;
      const bool in_range = m < M32;
      const uint32_t md[3] = {(in_range && dq > 0) ? ~0u : 0u, in_range ? ~0u : 0u, (in_range && dq + 1 < D) ? ~0u : 0u};
      const uint32_t mh[3] = {hq > 0 ? ~0u : 0u, ~0u, hq + 1 < H ? ~0u : 0u};
      const uint32_t mw[3] = {wq > 0 ? ~0u : 0u, ~0u, wq + 1 < W ? ~0u : 0u};
      v[27] = md[1] & 0x3f800000u;                   // bias column (1.0f); rows past the end stay all-zero
#pragma unroll
      for (int kd = 0; kd < 3; ++kd)
#pragma unroll
        for (int kh = 0; kh < 3; ++kh) {
          const uint32_t mdh = md[kd] & mh[kh];
#pragma unroll
          for (int kw = 0; kw < 3; ++kw) v[(kd * 3 + kh) * 3 + kw] = sp[uoff[kd * 3 + kh] + kw] & mdh & mw[kw];
        }
    };
    auto advance = [&]() {
      m += stride;
      wq += st_w;
      unsigned c = wq >= W ? 1u : 0u;
      wq -= c * W;
      hq += st_h + c;
      c = hq >= H ? 1u : 0u;
      hq -= c * H;
      dq += st_d + c;
      if (dq >= D) dq -= D;
    };
    int it = grp;
    int tile = cta + grp * ncta;
    if (!STAGED && tile < p.ntiles) load_row(nxt);
    for (; tile < p.ntiles; tile += 2 * ncta, it += 2) {
      const int s = it % C1U_STAGES;
      const uint32_t ph = (uint32_t)(it / C1U_STAGES) & 1u;
      const int xs = it % C1U_XS;
      uint32_t in[28];
      if (STAGED) {
        c1u_wait_t(xfull + 8 * xs, (uint32_t)(it / C1U_XS) & 1u, t_w0, prof);
        load_row_staged(in, xs_sm + (uint32_t)xs * xs_slot_bytes);
        advance();
      } else {
#pragma unroll
        for (int t = 0; t < 28; ++t) in[t] = __float_as_uint(nxt[t]);
        advance();
        if (tile + 2 * ncta < p.ntiles) load_row(nxt);
      }
      // bf16 hi / lo split, two elements per instruction:  hi = bf16(v) (cvt.rn.bf16x2), lo = bf16(v - hi) (FADD2 + cvt)
      uint32_t phi[16], plo[16];
#pragma unroll
      for (int j = 0; j < 14; ++j) {
        const uint32_t h2 = pack_bf16(__uint_as_float(in[2 * j]), __uint_as_float(in[2 * j + 1]));
        const uint64_t l2 = sub2_f32(pair_u32(in[2 * j], in[2 * j + 1]), pair_u32(h2 << 16, h2 & 0xffff0000u));
        phi[j] = h2;
        plo[j] = pack_bf16(__uint_as_float(lo_u32(l2)), __uint_as_float(hi_u32(l2)));
      }
      phi[14] = phi[15] = plo[14] = plo[15] = 0u;
      if (STAGED) mbar_arrive(xempty + 8 * xs);                 // every staged value has been consumed
      c1u_wait_t(empty + 8 * s, ph ^ 1u, t_w1, prof);
      uint8_t* a_hi = gen + (smA - smem_base) + (size_t)s * 2 * C1U_TILE_BYTES;
      uint8_t* a_lo = a_hi + C1U_TILE_BYTES;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const uint32_t off = sw64_off(r, j);
        *reinterpret_cast<uint4*>(a_hi + off) = make_uint4(phi[4 * j], phi[4 * j + 1], phi[4 * j + 2], phi[4 * j + 3]);
        *reinterpret_cast<uint4*>(a_lo + off) = make_uint4(plo[4 * j], plo[4 * j + 1], plo[4 * j + 2], plo[4 * j + 3]);
      }
      fence_proxy_async();                           // generic-proxy smem writes -> visible to the tensor core
      mbar_arrive(full + 8 * s);
    }
    if (prof && blockIdx.x == 0 && (threadIdx.x & 127) == 0)
      printf("c1u prof: producer group %d: total %lld cyc, waiting for staged image %lld, for a free A stage %lld\n", grp,
             clock64() - t_start, t_w0, t_w1);
  } else if (warp == 13) {
    // ======================================= image loader (STAGED) ==================================
    // lane kd copies window kd of every tile.  Interior tiles: one aligned bulk copy of xs_seg floats.  At the two ends of the
    // image the window is clipped to whole 16-byte chunks inside [0, total) (the destination shifts with it) and the up to
    // three floats of a ragged tail are stored by hand; whatever stays unwritten is only ever read under a false tap mask.
    // (one cp.async.bulk keeps the issuing thread busy for ~280 cycles, so twelve lanes work on four consecutive tiles)
    if (STAGED && lane < 12) {
      const int kdl = lane % 3, sub = lane / 3;
      const float* xg = p.x[g];
      const int total = (int)p.M, seg = p.xs_seg;
      const int c_kd = (-1 - p.W + (kdl - 1) * p.W * p.H) & ~3;            // aligned-down window start relative to the tile
      const uint32_t dst_kd = (uint32_t)kdl * (uint32_t)seg * 4u;
      int it = sub;
      for (int tile = cta + sub * ncta; tile < p.ntiles; tile += 4 * ncta, it += 4) {
        const int xs = it % C1U_XS;
        const uint32_t bar = xfull + 8 * xs;
        const uint32_t slot_sm = xs_sm + (uint32_t)xs * xs_slot_bytes + dst_kd;
        int a = tile * 128 + c_kd;
        c1u_wait_t(xempty + 8 * xs, ((uint32_t)(it / C1U_XS) & 1u) ^ 1u, t_w0, prof);
        if (a >= 0 && a + seg <= total) {
          const long long t0 = prof ? clock64() : 0;
          mbar_expect_tx(bar, (uint32_t)seg * 4u);
          const long long t1 = prof ? clock64() : 0;
          asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(slot_sm),
                       "l"(xg + a), "r"((uint32_t)seg * 4u), "r"(bar)
                       : "memory");
          if (prof) { const long long t2 = clock64(); t_w1 += t1 - t0; t_w2 += t2 - t1; }
        } else {
          int d0 = 0, n = seg;
          if (a < 0) { d0 = -a; n += a; a = 0; }                           // (-a is a multiple of 4: destination stays aligned)
          if (a + n > total) {
            const int keep = (total - a) > 0 ? ((total - a) & ~3) : 0;
            float* slot_ptr = reinterpret_cast<float*>(gen + (slot_sm - smem_base));
            for (int i = a + keep; i < total; ++i) slot_ptr[d0 + (i - a)] = xg[i];      // <= 3 floats
            n = keep;
          }
          n = n > 0 ? n : 0;
          mbar_expect_tx(bar, (uint32_t)n * 4u);                           // (the arrive also releases the tail stores)
          if (n > 0)
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                             slot_sm + (uint32_t)d0 * 4u),
                         "l"(xg + a), "r"((uint32_t)n * 4u), "r"(bar)
                         : "memory");
        }
      }
      if (prof && blockIdx.x == 0 && lane == 0)
        printf("c1u prof: loader: total %lld cyc, waiting for a free staging slot %lld, in expect_tx %lld, in cp.async.bulk %lld\n",
               clock64() - t_start, t_w0, t_w1, t_w2);
    }
  } else if (warp == 8 || warp == 14) {
    // ======================================= MMA issuers ============================================
    // Two issuers (one elected lane each) alternate tiles: with one, the serial chain  wait(accumulator) -> wait(A stage) ->
    // 6 MMAs -> 2 commits  took 700 cycles per tile and the producers waited 37 % of the time for a free A stage.
    const int iss = (warp == 8) ? 0 : 1;
    const uint64_t desc_hi = make_smem_desc(0, 16, 512, LAYOUT_SW64, 0) & 0xFFFFFFFF00000000ull;
    const uint32_t lo_const = (uint32_t)(make_smem_desc(0, 16, 512, LAYOUT_SW64, 0) & 0xFFFF0000ull);
    const uint32_t a0 = lo_const | ((smA & 0x3FFFFu) >> 4);
    const uint32_t wh = lo_const | ((smW & 0x3FFFFu) >> 4);
    const uint32_t wl = lo_const | (((smW + 4096) & 0x3FFFFu) >> 4);
    if (elect_one()) {
      int it = iss;
      for (int tile = cta + iss * ncta; tile < p.ntiles; tile += 2 * ncta, it += 2) {
        const int as = it % C1U_ACC, s = it % C1U_STAGES;
        c1u_wait_t(acc_empty + 8 * as, ((uint32_t)(it / C1U_ACC) & 1u) ^ 1u, t_w0, prof);
        c1u_wait_t(full + 8 * s, (uint32_t)(it / C1U_STAGES) & 1u, t_w1, prof);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(as * p.cout);
        const uint32_t ah = a0 + (uint32_t)s * (2 * C1U_TILE_BYTES >> 4);
        const uint32_t al = ah + (C1U_TILE_BYTES >> 4);
#pragma unroll
        for (int k = 0; k < 2; ++k) {
          mma_bf16_ss(d_tmem, desc_hi | (uint64_t)(ah + 2u * k), desc_hi | (uint64_t)(wh + 2u * k), p.idesc, k ? 1u : 0u);
          if (p.debug & 1) continue;
          mma_bf16_ss(d_tmem, desc_hi | (uint64_t)(al + 2u * k), desc_hi | (uint64_t)(wh + 2u * k), p.idesc, 1u);
          mma_bf16_ss(d_tmem, desc_hi | (uint64_t)(ah + 2u * k), desc_hi | (uint64_t)(wl + 2u * k), p.idesc, 1u);
        }
        mma_commit(empty + 8 * s);
        mma_commit(acc_full + 8 * as);
      }
      if (prof && blockIdx.x == 0)
        printf("c1u prof: issuer %d: total %lld cyc, waiting for a free accumulator %lld, for a full A stage %lld\n", iss,
               clock64() - t_start, t_w0, t_w1);
    }
    __syncwarp();
  } else if (warp != 15) {
    // ======================================= epilogue ===============================================
    // Two groups of four warps (9-12, 16-19) work on EVERY tile: group h owns channels [16 h, 16 h + 16) of each 32-channel
    // slice, so a thread (= one voxel row) does TMEM -> 16 fp32 -> packed bf16 -> one 32-byte store, and keeps the
    // BatchNorm sums of the stored values of its 16 channels in registers over the whole tile range (no per-tile
    // shuffles or atomics).  One group of four warps with all 32 channels took 730 cycles per tile and held the issuers
    // back 62 % of the time; a thread with 32 channels also needs 128 registers.  Bias is already in the accumulator
    // (K column 27).
    const int half = (warp >= 16) ? 1 : 0;
    const int quarter = warp & 3;
    const int row = quarter * 32 + lane;
    __nv_bfloat16* yg = p.y[g];
    const bool want_stats = p.stats[g] != nullptr;
    uint64_t ssum2[NCH][8], ssq2[NCH][8];            // packed fp32 pairs (FADD2 / FFMA2)
#pragma unroll
    for (int c = 0; c < NCH; ++c)
#pragma unroll
      for (int j = 0; j < 8; ++j) { ssum2[c][j] = 0ull; ssq2[c][j] = 0ull; }
    int it = 0;
    for (int tile = cta; tile < p.ntiles; tile += ncta, ++it) {
      const long long m = (long long)tile * 128 + row;
      const bool valid = m < p.M;
      const int as = it % C1U_ACC;
      const uint32_t acc_ph = (uint32_t)(it / C1U_ACC) & 1u;
      c1u_wait_t(acc_full + 8 * as, acc_ph, t_w0, prof);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(as * p.cout + half * 16);
#pragma unroll
      for (int c = 0; c < NCH; ++c) {
        uint32_t raw[16];
        tmem_ld16(taddr + (uint32_t)(c * 32), raw);
        tmem_ld_wait();
        if (c == NCH - 1) {                         // accumulator drained: hand the buffer back before the stores
          tc_fence_before();
          mbar_arrive(acc_empty + 8 * as);
        }
        uint32_t pk[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) pk[j] = pack_bf16(__uint_as_float(raw[2 * j]), __uint_as_float(raw[2 * j + 1]));
        if (valid && !(p.debug & 2))                // 256-bit store: a thread writes one whole 32-byte sector
          asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(yg + m * p.cout + c * 32 + half * 16),
                       "r"(pk[0]), "r"(pk[1]), "r"(pk[2]), "r"(pk[3]), "r"(pk[4]), "r"(pk[5]), "r"(pk[6]), "r"(pk[7])
                       : "memory");
        if (want_stats) {                           // rows past the end are exact zeros (all-zero im2col row)
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const uint64_t f = pair_u32(pk[j] << 16, pk[j] & 0xffff0000u);      // the stored (rounded) values
            ssum2[c][j] = add2_f32(ssum2[c][j], f);
            ssq2[c][j] = fma2_f32(f, f, ssq2[c][j]);
          }
        }
      }
    }
    if (prof && blockIdx.x == 0 && lane == 0 && quarter == 0)
      printf("c1u prof: epilogue group %d: total %lld cyc, waiting for a finished accumulator %lld\n", half, clock64() - t_start, t_w0);
    if (want_stats) {
#pragma unroll
      for (int c = 0; c < NCH; ++c) {
        float ssum[16], ssq[16];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          ssum[2 * j] = __uint_as_float(lo_u32(ssum2[c][j])); ssum[2 * j + 1] = __uint_as_float(hi_u32(ssum2[c][j]));
          ssq[2 * j] = __uint_as_float(lo_u32(ssq2[c][j])); ssq[2 * j + 1] = __uint_as_float(hi_u32(ssq2[c][j]));
        }
        // fold lanes l and l ^ 16, then transpose-reduce: lanes l and l + 16 end with the warp total of column l (l < 16)
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          ssum[i] += __shfl_xor_sync(0xffffffffu, ssum[i], 16);
          ssq[i] += __shfl_xor_sync(0xffffffffu, ssq[i], 16);
        }
#pragma unroll
        for (int off = 8; off >= 1; off >>= 1) {
          const bool upper = (lane & off) != 0;
#pragma unroll
          for (int i = 0; i < off; ++i) {
            const float s_send = upper ? ssum[i] : ssum[i + off];
            const float s_keep = upper ? ssum[i + off] : ssum[i];
            ssum[i] = s_keep + __shfl_xor_sync(0xffffffffu, s_send, off);
            const float q_send = upper ? ssq[i] : ssq[i + off];
            const float q_keep = upper ? ssq[i + off] : ssq[i];
            ssq[i] = q_keep + __shfl_xor_sync(0xffffffffu, q_send, off);
          }
        }
        if (lane < 16) {
          stats_ptr[quarter * 128 + c * 32 + half * 16 + lane] = ssum[0];
          stats_ptr[quarter * 128 + 64 + c * 32 + half * 16 + lane] = ssq[0];
        }
      }
      asm volatile("bar.sync 1, 256;" ::: "memory");
      const int e = threadIdx.x - 288;             // 0..127 over the first group's four warps
      if (e >= 0 && e < p.cout) {                  // fixed-order sum over the four lane quarters -> this CTA's row
        double s1 = 0.0, s2 = 0.0;
#pragma unroll
        for (int w4 = 0; w4 < 4; ++w4) { s1 += (double)stats_ptr[w4 * 128 + e]; s2 += (double)stats_ptr[w4 * 128 + 64 + e]; }
        stat_row_store(p.stats[g], 2 * p.cout, cta, ncta, e, s1);
        stat_row_store(p.stats[g], 2 * p.cout, cta, ncta, p.cout + e, s2);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 8) {
    tc_fence_after();
    tmem_dealloc(tmem_base, p.tmem_cols);
  }
}


// ------------------------------------------------------------------------------------------------------------
// conv1.0 weight gradient on tcgen05:   dW[co][kd][kh][kw] = sum_v dy[v,co] * x[v + (kd-1,kh-1,kw-1)]
//
// K = voxels (padded-row linearisation q = h*Wp + c of one (n,d) plane, Wp = W + 2, 128 voxels per tile).
//   A (M = 128 lanes) = the dY slab [voxel rows][32 channels] exactly as TMA lands it (MN-major, 64B swizzle), loaded
//       two columns early (slab column c <-> dy voxel w = c - 2); the four 32-channel M atoms start one row apart
//       (LBO = 64 B), i.e. atom j sees dy shifted by j voxels along w  ->  j = 0,1,2 are the taps kw = 2,1,0.
//   B (N = 16)        = x patches, K-major: row n = kd*3+kh holds x(d+kd-1, h+kh-1, c-1) for the tile's 128 voxels --
//       contiguous pieces of image rows, written by builder warps as bf16 hi / lo tiles (128B swizzle), so the fp32
//       image enters as xh + xl (two MMAs per K step).
// Accumulation stays in TMEM (16 columns) over the CTA's whole tile range; each CTA stores its 864 partial sums into
// its slot of the caller's workspace and conv1_wgrad_reduce_kernel adds the slots in CTA order (deterministic).
// ------------------------------------------------------------------------------------------------------------
constexpr int C1W_U_THREADS = 320;          // warp 0: TMA (dY), warps 1-8: patch builders (two groups), warp 9: MMA
constexpr int C1W_U_STAGES = 4;
constexpr uint32_t C1W_U_PTILE = 2 * 16 * 128;     // [2 K-blocks][16 rows][128 B]

struct alignas(64) C1WParams {
  CUtensorMap tmY[TMF_MAX_GROUPS];
  const float* x[TMF_MAX_GROUPS];
  float* part[TMF_MAX_GROUPS];     // per-CTA partial dW [ncta][Cout*27] (caller workspace; reduced in CTA order)
  int ng, B, D, H, W, Wp, NHy, QT, ntiles;
  uint32_t y_tx, y_slab_bytes, stage_bytes, idesc;
};

__global__ void __launch_bounds__(C1W_U_THREADS, 1) conv1_umma_wgrad_kernel(const __grid_constant__ C1WParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t bars = smem_base + C1W_U_STAGES * p.stage_bytes;
  const uint32_t y_full = bars, p_full = bars + 8 * C1W_U_STAGES, empty = p_full + 8 * C1W_U_STAGES;
  const uint32_t acc_full = empty + 8 * C1W_U_STAGES, tmem_slot = acc_full + 8;
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(gen + (tmem_slot - smem_base));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = blockIdx.x % p.ng;
  const int cta = blockIdx.x / p.ng, ncta = gridDim.x / p.ng;

  if (threadIdx.x == 0) {
    for (int i = 0; i < C1W_U_STAGES; ++i) {
      mbar_init(y_full + 8 * i, 1);
      mbar_init(p_full + 8 * i, 128);
      mbar_init(empty + 8 * i, 1);
    }
    mbar_init(acc_full, 1);
    fence_barrier_init();
    prefetch_tmap(&p.tmY[g]);
  }
  if (warp == 9) {
    tmem_alloc(tmem_slot, 32);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp == 0) {
    if (lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      for (int tile = cta; tile < p.ntiles; tile += ncta) {
        int t = tile;
        const int qt = t % p.QT; t /= p.QT;
        const int d = t % p.D;
        const int n = t / p.D;
        const int h0 = (qt * 128) / p.Wp;
        mbar_wait(empty + 8 * s, ph ^ 1u);
        mbar_expect_tx(y_full + 8 * s, p.y_tx);
        tma_load_5d(smem_base + (uint32_t)s * p.stage_bytes, &p.tmY[g], y_full + 8 * s, 0, -2, h0, d, n);
        if (++s == C1W_U_STAGES) { s = 0; ph ^= 1u; }
      }
    }
  } else if (warp <= 8) {
    // ---- patch builders: thread -> (row n = kd*3+kh, two 8-voxel chunks) of the K-major B tile
    const int grp = (warp - 1) >> 2;
    const int tb = (threadIdx.x - 32) & 127;
    const int n = tb >> 3, qc = tb & 7;
    const int kd = n / 3, kh = n % 3;
    const float* xg = p.x[g];
    int it = grp;
    for (int tile = cta + grp * ncta; tile < p.ntiles; tile += 2 * ncta, it += 2) {
      const int s = it % C1W_U_STAGES;
      const uint32_t ph = (uint32_t)(it / C1W_U_STAGES) & 1u;
      int t = tile;
      const int qt = t % p.QT; t /= p.QT;
      const int d = t % p.D;
      const int nb = t / p.D;
      float v[2][8];
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        const int q = qt * 128 + (qc + 8 * half) * 8;
        int h = q / p.Wp, c = q - h * p.Wp;
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const int dd = d + kd - 1, hh = h + kh - 1, ww = c - 1;
          const bool ok = n < 9 && dd >= 0 && dd < p.D && hh >= 0 && hh < p.H && ww >= 0 && ww < p.W;
          v[half][e] = ok ? __ldg(xg + (((long long)nb * p.D + dd) * p.H + hh) * p.W + ww) : 0.f;
          if (++c == p.Wp) { c = 0; ++h; }
        }
      }
      mbar_wait(empty + 8 * s, ph ^ 1u);
      uint8_t* ptile = gen + (size_t)s * p.stage_bytes + p.y_slab_bytes;       // P_hi, then P_lo
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        float hi[8], lo[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) split_bf16(v[half][e], hi[e], lo[e]);
        const uint32_t off = (uint32_t)half * 2048u + (uint32_t)n * 128u + (uint32_t)((qc ^ (n & 7)) << 4);
        *reinterpret_cast<uint4*>(ptile + off) = pack8(hi);
        *reinterpret_cast<uint4*>(ptile + C1W_U_PTILE + off) = pack8(lo);
      }
      fence_proxy_async();
      mbar_arrive(p_full + 8 * s);
    }
    if (warp <= 4) {
      // ---- epilogue (after the whole range): lane m = (j, co) -> taps kw = 2 - j; column n = kd*3+kh
      mbar_wait(acc_full, 0u);
      tc_fence_after();
      const int quarter = warp & 3;
      const int m = quarter * 32 + lane;
      const int j = m >> 5, co = m & 31;
      uint32_t raw[32];
      // 16 valid columns; the x32 load reads 16 unallocated-but-in-range columns of our 32-column allocation
      tmem_ld32(tmem_base + ((uint32_t)(quarter * 32) << 16), raw);
      tmem_ld_wait();
      if (j < 3) {
#pragma unroll
        for (int nn = 0; nn < 9; ++nn) p.part[g][(size_t)cta * 864 + co * 27 + nn * 3 + (2 - j)] = __uint_as_float(raw[nn]);
      }
    }
  } else {
    // ---- MMA issuer (warp 9)
    int s = 0;
    uint32_t ph = 0;
    const uint64_t hi_a = make_smem_desc(0, 64, 512, LAYOUT_SW64, 0) & 0xFFFFFFFF00000000ull;      // MN-major dY slab
    const uint32_t a_const = (uint32_t)(make_smem_desc(0, 64, 512, LAYOUT_SW64, 0) & 0xFFFF0000ull);
    const uint64_t hi_b = make_smem_desc(0, 16, 1024, LAYOUT_SW128, 0) & 0xFFFFFFFF00000000ull;    // K-major patches
    const uint32_t b_const = (uint32_t)(make_smem_desc(0, 16, 1024, LAYOUT_SW128, 0) & 0xFFFF0000ull);
    uint32_t accumulate = 0;
    for (int tile = cta; tile < p.ntiles; tile += ncta) {
      const int qt = tile % p.QT;
      const uint32_t qoff = (uint32_t)((qt * 128) % p.Wp);
      mbar_wait(y_full + 8 * s, ph);
      mbar_wait(p_full + 8 * s, ph);
      tc_fence_after();
      const uint32_t st = smem_base + (uint32_t)s * p.stage_bytes;
      const uint32_t a_lo = a_const | (((st + qoff * 64u) & 0x3FFFFu) >> 4);
      const uint32_t bh_lo = b_const | (((st + p.y_slab_bytes) & 0x3FFFFu) >> 4);
      const uint32_t bl_lo = bh_lo + (C1W_U_PTILE >> 4);
      if (elect_one()) {
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const uint32_t boff = (uint32_t)(k >> 2) * (2048u >> 4) + (uint32_t)(k & 3) * 2u;
          const uint32_t aoff = (uint32_t)k * ((16u * 64u) >> 4);
          mma_bf16_ss(tmem_base, hi_a | (uint64_t)(a_lo + aoff), hi_b | (uint64_t)(bh_lo + boff), p.idesc,
                      (accumulate | (uint32_t)k) ? 1u : 0u);
          mma_bf16_ss(tmem_base, hi_a | (uint64_t)(a_lo + aoff), hi_b | (uint64_t)(bl_lo + boff), p.idesc, 1u);
        }
        mma_commit(empty + 8 * s);
      }
      __syncwarp();
      accumulate = 1;
      if (++s == C1W_U_STAGES) { s = 0; ph ^= 1u; }
    }
    if (elect_one()) mma_commit(acc_full);
    __syncwarp();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 9) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 32);
  }
}

__global__ void conv1_wgrad_reduce_kernel(GroupPtr<const float> part, GroupPtr<float> dw, int ncta, int n) {
  const int g = blockIdx.z;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float s = 0.f;
  for (int k = 0; k < ncta; ++k) s += part.p[g][(size_t)k * n + i];
  dw.p[g][i] = s;
}

}  // namespace tmf

using namespace tmf;

bool tmf_conv1_fwd_umma_supported(int cout) {
  if (getenv("TMF_DISABLE_UMMA") != nullptr) return false;
  return cout == 32 || cout == 64;
}

int tmf_conv1_fwd_umma(int ng, const float* const* x, const float* const* w, const float* const* bias, void* const* y,
                       double* const* stats, int B, int D, int H, int W, int cout, void* stream) {
  TMF_CHECK_NG(ng);
  TMF_REQUIRE(cout == 32 || cout == 64, "conv1_fwd_umma: Cout must be 32 or 64 (got %d)", cout);
  TMF_REQUIRE((long long)B * D * H * W < (1ll << 31), "conv1_fwd_umma: volume batch too large for 32-bit voxel indices");
  C1UParams p{};
  p.ng = ng; p.B = B; p.D = D; p.H = H; p.W = W; p.cout = cout;
  p.M = (long long)B * D * H * W;
  p.ntiles = (int)((p.M + 127) / 128);
  p.idesc = make_idesc_bf16(128, cout, 0, 0);
  p.tmem_cols = (cout == 32) ? 128 : 256;          // C1U_ACC accumulators of Cout columns
  {
    const char* e = getenv("TMF_C1U_DEBUG");
    p.debug = e ? atoi(e) : 0;
  }
  cudaStream_t st = (cudaStream_t)stream;
  for (int g = 0; g < ng; ++g) {
    TMF_REQUIRE(x[g] && w[g] && y[g], "conv1_fwd_umma: NULL device pointer");
    p.x[g] = x[g]; p.w[g] = w[g];
    p.bias[g] = bias ? bias[g] : nullptr;
    p.y[g] = (__nv_bfloat16*)y[g];
    p.stats[g] = stats ? stats[g] : nullptr;
  }
  // staged image windows (see the kernel): needs 16-byte aligned images and rows that fit the staging buffers
  p.xs_seg = (2 * W + 133 + 3) & ~3;
  bool staged = getenv("TMF_C1U_UNSTAGED") == nullptr;
  for (int g = 0; g < ng; ++g) staged = staged && (reinterpret_cast<uintptr_t>(x[g]) & 15u) == 0;
  const uint32_t smem_fixed = 1024 + C1U_STAGES * 2 * C1U_TILE_BYTES + 2 * 4096 + 8 * (2 * C1U_STAGES) + 16 * C1U_ACC + 32 + 2048 + 16 * C1U_XS;
  const uint32_t smem_max = 227 * 1024;
  staged = staged && smem_fixed + (uint32_t)C1U_XS * 3 * p.xs_seg * 4 + 64 <= smem_max;
  const uint32_t smem = smem_fixed + (staged ? (uint32_t)C1U_XS * 3 * p.xs_seg * 4 : 0u) + 64;
  static bool attr_done = false;
  if (!attr_done) {
    TMF_CUDA(cudaFuncSetAttribute(conv1_umma_fwd_kernel<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max));
    TMF_CUDA(cudaFuncSetAttribute(conv1_umma_fwd_kernel<2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max));
    TMF_CUDA(cudaFuncSetAttribute(conv1_umma_fwd_kernel<1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max));
    TMF_CUDA(cudaFuncSetAttribute(conv1_umma_fwd_kernel<2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max));
    attr_done = true;
  }
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  int per_group = sms / ng;
  if (per_group > p.ntiles) per_group = p.ntiles;
  if (per_group < 1) per_group = 1;
  if (per_group > TMF_STAT_ROWS) per_group = TMF_STAT_ROWS;
  const dim3 grid(per_group * ng);
  if (cout == 32 && staged) launch_k(conv1_umma_fwd_kernel<1, true>, grid, C1U_THREADS, smem, st, p);
  else if (cout == 32) launch_k(conv1_umma_fwd_kernel<1, false>, grid, C1U_THREADS, smem, st, p);
  else if (staged) launch_k(conv1_umma_fwd_kernel<2, true>, grid, C1U_THREADS, smem, st, p);
  else launch_k(conv1_umma_fwd_kernel<2, false>, grid, C1U_THREADS, smem, st, p);
  TMF_LAUNCH_CHECK();
  return 0;
}


bool tmf_conv1_wgrad_umma_supported(int W, int cout) {
  if (getenv("TMF_DISABLE_UMMA") != nullptr) return false;
  return cout == 32 && W + 2 <= 256;
}

size_t tmf_conv1_wgrad_umma_workspace(int ng, int cout) { return (size_t)ng * 148 * 27 * cout * sizeof(float); }

int tmf_conv1_wgrad_umma(int ng, const void* const* dy, const float* const* x, float* const* dw, int B, int D, int H,
                         int W, int cout, void* ws, size_t ws_bytes, void* stream) {
  TMF_CHECK_NG(ng);
  TMF_REQUIRE(ws != nullptr && ws_bytes >= tmf_conv1_wgrad_umma_workspace(ng, cout) && ((uintptr_t)ws & 15) == 0,
              "conv1_wgrad_umma: needs a 16-byte aligned workspace of tmf_conv1_wgrad_workspace_bytes() bytes");
  TMF_REQUIRE(tmf_conv1_wgrad_umma_supported(W, cout) || cout == 32, "conv1_wgrad_umma: needs Cout = 32 (got %d)", cout);
  typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  static EncodeTiledFn encode = nullptr;
  if (encode == nullptr) {
    void* sym = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      encode = reinterpret_cast<EncodeTiledFn>(sym);
  }
  TMF_REQUIRE(encode != nullptr, "conv1_wgrad_umma: cuTensorMapEncodeTiled entry point not available");
  C1WParams p{};
  p.ng = ng; p.B = B; p.D = D; p.H = H; p.W = W;
  p.Wp = W + 2;
  p.NHy = ((p.Wp - 1) + 127 + 3) / p.Wp + 1;
  p.QT = (H * p.Wp + 127) / 128;
  p.ntiles = B * D * p.QT;
  p.y_tx = (uint32_t)p.NHy * p.Wp * 64u;
  p.y_slab_bytes = (p.y_tx + 1023u) & ~1023u;
  p.stage_bytes = p.y_slab_bytes + 2 * C1W_U_PTILE;
  p.idesc = make_idesc_bf16(128, 16, /*A MN-major*/ 1, /*B K-major*/ 0);
  cudaStream_t st = (cudaStream_t)stream;
  for (int g = 0; g < ng; ++g) {
    TMF_REQUIRE(dy[g] && x[g] && dw[g], "conv1_wgrad_umma: NULL device pointer");
    p.x[g] = x[g];
    p.part[g] = (float*)ws + (size_t)g * 148 * 27 * cout;
    cuuint64_t dims[5] = {(cuuint64_t)cout, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)D, (cuuint64_t)B};
    cuuint64_t strides[4] = {(cuuint64_t)cout * 2, (cuuint64_t)W * cout * 2, (cuuint64_t)H * W * cout * 2,
                             (cuuint64_t)D * H * W * cout * 2};
    cuuint32_t box[5] = {32, (cuuint32_t)p.Wp, (cuuint32_t)p.NHy, 1, 1};
    cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    CUresult r = encode(&p.tmY[g], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<void*>(dy[g]), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    TMF_REQUIRE(r == CUDA_SUCCESS, "conv1_wgrad_umma: cuTensorMapEncodeTiled(dY) failed with %d", (int)r);
  }
  const uint32_t smem = 1024 + C1W_U_STAGES * p.stage_bytes + 8 * (3 * C1W_U_STAGES) + 64;
  TMF_REQUIRE(smem <= 227 * 1024, "conv1_wgrad_umma: W=%d too wide", W);
  static bool attr_done = false;
  if (!attr_done) {
    TMF_CUDA(cudaFuncSetAttribute(conv1_umma_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr_done = true;
  }
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  int per_group = sms / ng;
  if (per_group > p.ntiles) per_group = p.ntiles;
  if (per_group > 148) per_group = 148;
  if (per_group < 1) per_group = 1;
  launch_k(conv1_umma_wgrad_kernel, dim3(per_group * ng), C1W_U_THREADS, smem, st, p);
  TMF_LAUNCH_CHECK();
  GroupPtr<const float> gpart;
  GroupPtr<float> gdw;
  for (int g = 0; g < TMF_MAX_GROUPS; ++g) { gpart.p[g] = g < ng ? p.part[g] : nullptr; gdw.p[g] = g < ng ? dw[g] : nullptr; }
  launch_k(conv1_wgrad_reduce_kernel, dim3(ceil_div(27 * cout, 128), 1, ng), 128, 0, st, gpart, gdw, per_group, 27 * cout);
  TMF_LAUNCH_CHECK();
  return 0;
}

// conv_umma_col.cu -- second-generation implicit-GEMM Conv3d 3x3x3 (pad 1) forward / dgrad for the layers with
// Cin in {32, 64} and Cout a multiple of 32 (<= 128): blocks 2 and 3 of sNet (reference models/networks.py:28-41) and
// their input gradients.  Everything below was sized from measurements on B200 (scripts/ubench/*.cu, TMF_COL_DEBUG):
//
//   * ISSUE-BOUND MMAs.  A 128 x N x 16 tcgen05.mma with small N is not limited by the tensor pipe but by the thread
//     that issues it (~100 cycles of descriptor moves per instruction) and by shared-memory operand reads (the A tile
//     costs the same bytes whatever N is).  Two remedies:
//       - kw-STACKING IN N.  The three kw taps of one (kd, kh) are neighbouring blocks of wf[tap][Cout][Cin], i.e. ONE
//         K-major B operand with N = 96 rows (3 taps x 32 output channels).  One MMA per (kd, kh, k-step), with the A
//         window shifted by kh rows only, fills three column blocks D_kw[r] = sum X[r + kh*Wp] W[kd,kh,kw]; the
//         convolution is y[r] = D_0[r] + D_1[r+1] + D_2[r+2], a two-lane shift done in the epilogue with warp shuffles
//         (rows 32q+32, 32q+33 come from the next TMEM lane quarter through shared memory).  An M tile of 128 rows
//         therefore yields 126 outputs.  3x fewer MMAs.
//       - THREE ISSUER WARPS, one elected thread each running its whole role (no per-tap elect/reconverge).
//   * INPUT-STATIONARY ROLLING PLANES.  A CTA walks a column (sample, 126 positions) along d.  An input plane slab is
//     used the moment it lands: it adds tap plane kd=2 to output d-1 (completing it), kd=1 to output d, kd=0 to output
//     d+1, and its shared-memory slot is released at once -- every slot of the ring is prefetch depth, the three open
//     outputs live in TMEM (4 accumulator buffers x 96 columns).  Output io belongs to issuer io % 3: a plane feeds
//     exactly one output per issuer, and an output's 27 taps are issued by one thread, in order.
//   * TMA: one thread keeps only ~2 tensor loads in flight (~600 cycles per box whatever its size, more from DRAM), so
//     four lanes of the producer warp issue the plane loads round-robin; weights (27 taps x 32 channels) are resident.
//   * Cout > 32 is split into 32-channel slices handled by different CTAs ("virtual groups"): the slice's weights
//     (55-110 KB) stay resident, the input is re-read from L2.
//   * Padded row pitch W+1 (the right halo of row h is the left halo of row h+1: one zero column, TMA OOB fill).
//   * mbarrier parity waits are only sound for a thread that has observed every earlier phase of that barrier, so every
//     issuer waits on every accumulator hand-over and every TMA lane on every slot hand-over, owner or not.
//   * Epilogue: 2 groups x 4 warps alternate outputs; BatchNorm statistics accumulate per thread in registers over the
//     CTA's whole range; 256-bit stores (whole sectors per thread).
#include <cuda.h>

#include "common.cuh"
#include "umma.cuh"

namespace tmf {
using namespace umma;

constexpr int CC_TMA_LANES = 4;
constexpr int CC_MMA_WARPS = 3;
constexpr int CC_FIRST_EPI = 1 + CC_MMA_WARPS;
constexpr int CC_EPI_WARPS = 8;
constexpr int CC_THREADS = 32 * (CC_FIRST_EPI + CC_EPI_WARPS);
constexpr int CC_TILE_OUT = 126;                // outputs per 128-row M tile (2 rows feed the kw shift)
constexpr int CC_MAX_SLOTS = 10;
constexpr int CC_CO = 32;                       // output channels per CTA (slice of Cout)
constexpr int CC_NSTACK = 3 * CC_CO;            // MMA N
constexpr int CC_NS_CO = 64;                    // output channels per CTA of the non-stacked variant (NS, see the kernel)
constexpr int CC_NBUF = 4;                      // accumulator buffers
constexpr int CC_MAX_VG = 8;                    // towers x Cout slices
constexpr uint32_t CC_SMEM_BUDGET = 227 * 1024;
constexpr uint32_t CC_XCHG_BYTES = 2 * 2 * 4 * 3 * 32 * 4;   // [parity][group][quarter][D1_0, D2_0, D2_1][32 ch] floats
constexpr uint32_t CC_FIXED_SMEM = 1024 /*align*/ + 8 * (2 * CC_MAX_SLOTS) + 8 + 8 * 2 * CC_NBUF + 24 + CC_XCHG_BYTES + 2048 /*stats: [8 warps][2][32]*/ +
                                   256 /*bias*/ + 64;

struct alignas(64) ColConvParams {
  CUtensorMap tmA[TMF_MAX_GROUPS];
  CUtensorMap tmB[TMF_MAX_GROUPS];
  const float* bias[TMF_MAX_GROUPS];
  __nv_bfloat16* y[TMF_MAX_GROUPS];
  double* stats[TMF_MAX_GROUPS];
  int ng, nsplit, cout, B, D, H, W;
  int Wp, NH, NC, S;              // padded pitch (W+1), slab rows (in h), columns per plane, ring slots
  int qneed;                      // positions of a plane that hold outputs: (H-1)*Wp + W
  int steps_per_group;            // B * NC * D
  uint32_t layout, slot_bytes, a_tx_bytes, b_bytes, idesc;
  int ns;                         // non-stacked variant (template NS)
  int debug;                      // bring-up switches (TMF_COL_DEBUG): 1 no shift, 2 no stores/stats, 8 no MMAs, 32 role timing
};


// bring-up instrumentation (debug & 32): cycles a role spends blocked on one kind of barrier
__device__ __forceinline__ void mbar_wait_t(uint32_t bar, uint32_t parity, long long& acc, bool on) {
  if (!on) { mbar_wait(bar, parity); return; }
  const long long t0 = clock64();
  mbar_wait(bar, parity);
  acc += clock64() - t0;
}

// KSTEPS = Cin / 16 (2 or 4).
// NS ("not stacked", Cin = 32 with Cout a multiple of 64: conv2.3 forward).  With K = 32 per tap the kw-stacked tile does
// only 18 MMAs for an epilogue of 96 accumulator columns and a two-row shift, and is bound by that epilogue (the issuers wait
// 25-35 % of the time for a free accumulator, 48 % tensor pipe); Cout = 64 as two 32-channel slices also reads the input
// twice.  Here the CTA takes 64 output channels at once, every tap is its own N = 64 MMA with the A window shifted by
// kh * Wp + kw rows (54 MMAs per tile over the three issuer threads; the same 1728 tensor-pipe cycles per 128 x 64 outputs),
// all 128 rows of a tile are outputs, and the epilogue is a plain TMEM read: the two groups split the 64 channels of EVERY
// output (32 columns per thread instead of 96, no shuffles, no exchange, no group barrier).
// Role layout (the same for both variants).  Measured for NS and dropped: six issuers with two sub-accumulators per output (one
// per k-step parity; 512 threads at 128 registers) ran 193 us against 171 us -- the epilogue then reads twice the TMEM bytes
// (64 B per cycle and SM) and lost its registers; two sub-accumulators with three issuers changed nothing (178 us), i.e. MMAs
// into the same accumulator do pipeline and the ~140 cycles per tcgen05.mma are the issuing thread's own (R2UR / LDCU /
// UIADD3 chain per descriptor, cuobjdump -sass).
template <bool NS> struct ColRoles {
  static constexpr int MMA_WARPS = CC_MMA_WARPS;
  static constexpr int FIRST_EPI = CC_FIRST_EPI;
  static constexpr int THREADS = 32 * (FIRST_EPI + CC_EPI_WARPS);
};
template <int KSTEPS, bool NS>
__global__ void __launch_bounds__(ColRoles<NS>::THREADS, 1) conv3d_umma_col_kernel(const __grid_constant__ ColConvParams p) {
  constexpr int MMA_WARPS = ColRoles<NS>::MMA_WARPS, FIRST_EPI = ColRoles<NS>::FIRST_EPI;
  constexpr uint32_t PITCH = KSTEPS * 32u;          // bytes per smem row (= Cin * 2)
  constexpr uint32_t ROW_UNITS = PITCH >> 4;
  constexpr uint32_t SBO = 8u * PITCH;
  constexpr int NCO = NS ? CC_NS_CO : CC_CO;        // output channels of this CTA
  constexpr int NMMA = NS ? CC_NS_CO : CC_NSTACK;   // MMA N
  constexpr int NSUB = 1;                           // sub-accumulators per output (see ColRoles)
  constexpr int NCOLS = NMMA * NSUB;                // TMEM columns per accumulator buffer
  constexpr int TILE_OUT = NS ? 128 : CC_TILE_OUT;  // outputs per 128-row tile
  constexpr uint32_t TAP_UNITS = (uint32_t)NCO * ROW_UNITS;     // one tap of the slice's weights, in 16-byte units

  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t smB = smem_base;
  const uint32_t smA = smB + ((p.b_bytes + 1023u) & ~1023u);
  const uint32_t bars = smA + (uint32_t)p.S * p.slot_bytes;
  const uint32_t a_full = bars, a_empty = a_full + 8 * CC_MAX_SLOTS;
  const uint32_t b_full = a_empty + 8 * CC_MAX_SLOTS;
  const uint32_t acc_full = b_full + 8, acc_empty = acc_full + 8 * CC_NBUF;
  const uint32_t tmem_slot = acc_empty + 8 * CC_NBUF;
  const uint32_t xchg_sm = tmem_slot + 24;                               // 16-byte aligned (bars is 1024-aligned)
  const uint32_t stats_sm = xchg_sm + CC_XCHG_BYTES;                     // float [8 epilogue warps][2][32]
  const uint32_t bias_sm = stats_sm + 2048;                              // float [32]
  uint8_t* gen_base = smem_raw + (smem_base - smem_u32(smem_raw));
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(gen_base + (tmem_slot - smem_base));
  float* xchg_ptr = reinterpret_cast<float*>(gen_base + (xchg_sm - smem_base));
  float* stats_ptr = reinterpret_cast<float*>(gen_base + (stats_sm - smem_base));
  float* bias_ptr = reinterpret_cast<float*>(gen_base + (bias_sm - smem_base));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const bool prof = (p.debug & 32) != 0;
  const int ngv = p.ng * p.nsplit;
  const int gv = blockIdx.x % ngv;                  // virtual group = (tower, Cout slice)
  const int g = gv / p.nsplit;
  const int co_off = (gv % p.nsplit) * NCO;
  const int cta = blockIdx.x / ngv, ncta = gridDim.x / ngv;
  const int s_begin = (int)(((int64_t)cta * p.steps_per_group) / ncta);
  const int s_end = (int)(((int64_t)(cta + 1) * p.steps_per_group) / ncta);

  if (threadIdx.x == 0) {
    for (int i = 0; i < p.S; ++i) { mbar_init(a_full + 8 * i, 1); mbar_init(a_empty + 8 * i, MMA_WARPS); }
    mbar_init(b_full, 1);
    for (int i = 0; i < CC_NBUF; ++i) { mbar_init(acc_full + 8 * i, 1); mbar_init(acc_empty + 8 * i, NS ? CC_EPI_WARPS : CC_EPI_WARPS / 2); }
    fence_barrier_init();
    prefetch_tmap(&p.tmA[g]);
    prefetch_tmap(&p.tmB[g]);
  }
  if (threadIdx.x < NCO) bias_ptr[threadIdx.x] = (p.bias[g] != nullptr) ? p.bias[g][co_off + threadIdx.x] : 0.f;
  if (warp == 1) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp == 0) {
    // =========================================== TMA producer ===========================================
    if (lane < CC_TMA_LANES && s_begin < s_end) {
      if (lane == 0) {
        mbar_expect_tx(b_full, p.b_bytes);
        tma_load_3d(smB, &p.tmB[g], b_full, 0, co_off, 0);             // all 27 taps of this Cout slice at once
      }
      int slot = 0, jw = 0;
      uint32_t ph = 0;
      long long t_wait = 0;
      const long long t_start = clock64();
      for (int s = s_begin; s < s_end;) {
        const int d = s % p.D, col = s / p.D;
        const int c = col % p.NC, n = col / p.NC;
        const int len = min(p.D - d, s_end - s);
        const int pa = max(d - 1, 0), pb = min(d + len, p.D - 1);
        const int h0 = (c * TILE_OUT) / p.Wp;
        for (int pl = pa; pl <= pb; ++pl, ++jw) {
          mbar_wait_t(a_empty + 8 * slot, ph ^ 1u, t_wait, prof);      // every lane sees every phase (see header)
          if ((jw % CC_TMA_LANES) == lane) {
            mbar_expect_tx(a_full + 8 * slot, p.a_tx_bytes);
            tma_load_5d(smA + (uint32_t)slot * p.slot_bytes, &p.tmA[g], a_full + 8 * slot, 0, -1, h0 - 1, pl, n);
          }
          if (++slot == p.S) { slot = 0; ph ^= 1u; }
        }
        s += len;
      }
      if (prof && blockIdx.x == 0 && lane == 0)
        printf("col prof: producer lane 0: total %lld cyc, waiting for a free slot %lld\n", clock64() - t_start, t_wait);
    }
  } else if (warp <= MMA_WARPS) {
    // =========================================== MMA issuers ============================================
    const int issuer = warp - 1;
    const int sub = issuer / CC_MMA_WARPS;          // NS: which k-step parity / sub-accumulator this issuer feeds (else 0)
    if (s_begin < s_end && elect_one()) {
      const uint64_t desc_hi = make_smem_desc(0, 16, SBO, p.layout, 0) & 0xFFFFFFFF00000000ull;
      const uint32_t desc_lo_const = (uint32_t)(make_smem_desc(0, 16, SBO, p.layout, 0) & 0xFFFF0000ull);
      const uint32_t a0_lo = desc_lo_const | ((smA & 0x3FFFFu) >> 4);
      const uint32_t b0_lo = desc_lo_const | ((smB & 0x3FFFFu) >> 4);
      const uint32_t slot_units = p.slot_bytes >> 4;
      const uint32_t wp_units = (uint32_t)p.Wp * ROW_UNITS;
      const uint32_t idesc = p.idesc;
      const bool no_mma = (p.debug & 8) != 0;
      int it = 0;                        // outputs finished by earlier segments
      int slot = 0;
      uint32_t ph = 0;
      long long t_full = 0, t_acc = 0;
      const long long t_start = clock64();
      mbar_wait(b_full, 0u);
      tc_fence_after();
      for (int s = s_begin; s < s_end;) {
        const int d0 = s % p.D, col = s / p.D;
        const int c = col % p.NC;
        const int len = min(p.D - d0, s_end - s);
        const int da = d0, db = d0 + len - 1;
        const int pa = max(da - 1, 0), pb = min(db + 1, p.D - 1);
        const uint32_t qoff_units = (uint32_t)((c * TILE_OUT) % p.Wp) * ROW_UNITS;
        for (int pl = pa; pl <= pb; ++pl) {
          mbar_wait_t(a_full + 8 * slot, ph, t_full, prof);
          tc_fence_after();
          const uint32_t a_slab = a0_lo + (uint32_t)slot * slot_units + qoff_units;
#pragma unroll
          for (int kd = 2; kd >= 0; --kd) {          // output o = pl + 1 - kd: the one this plane completes goes first
            const int o = pl + 1 - kd;
            if (o < da || o > db) continue;
            const int io = it + (o - da);            // index of output o in this CTA's sequence
            const int as = io & (CC_NBUF - 1);
            const bool first = (pl == max(o - 1, 0));
            if (first) {                             // every issuer, owner or not (parity soundness)
              mbar_wait_t(acc_empty + 8 * as, ((uint32_t)(io / CC_NBUF) & 1u) ^ 1u, t_acc, prof);
              tc_fence_after();
            }
            if ((io % CC_MMA_WARPS) != (issuer % CC_MMA_WARPS)) continue;
            const uint32_t d_tmem = tmem_base + (uint32_t)(as * NCOLS);
            if (!no_mma) {
#pragma unroll
              for (int kh = 0; kh < 3; ++kh) {
                if (NS) {
#pragma unroll
                  for (int kw = 0; kw < 3; ++kw) {
                    const uint32_t b_lo = b0_lo + (uint32_t)((kd * 3 + kh) * 3 + kw) * TAP_UNITS;
                    const uint32_t a_lo = a_slab + (uint32_t)kh * wp_units + (uint32_t)kw * ROW_UNITS;
#pragma unroll
                    for (int k = 0; k < KSTEPS; ++k) {
                      if ((k % NSUB) != sub) continue;                 // the other issuer of this output
                      mma_bf16_ss(d_tmem + (uint32_t)(sub * NMMA), desc_hi | (uint64_t)(a_lo + 2u * k),
                                  desc_hi | (uint64_t)(b_lo + 2u * k), idesc,
                                  (!first || kh != 0 || kw != 0 || k >= NSUB) ? 1u : 0u);
                    }
                  }
                } else {
                  const uint32_t b_lo = b0_lo + (uint32_t)((kd * 3 + kh) * 3) * TAP_UNITS;
                  const uint32_t a_lo = a_slab + (uint32_t)kh * wp_units;
#pragma unroll
                  for (int k = 0; k < KSTEPS; ++k)
                    mma_bf16_ss(d_tmem, desc_hi | (uint64_t)(a_lo + 2u * k), desc_hi | (uint64_t)(b_lo + 2u * k), idesc,
                                (!first || kh != 0 || k != 0) ? 1u : 0u);
                }
              }
            }
            if (pl == min(o + 1, p.D - 1)) mma_commit(acc_full + 8 * as);   // last contribution: output o is complete
          }
          mma_commit(a_empty + 8 * slot);            // (count 3: the slot is free once every issuer is done with it)
          if (++slot == p.S) { slot = 0; ph ^= 1u; }
        }
        it += len;
        s += len;
      }
      if (prof && blockIdx.x == 0)
        printf("col prof: issuer %d: total %lld cyc, waiting for input planes %lld, for a free accumulator %lld (%d outputs)\n",
               issuer, clock64() - t_start, t_full, t_acc, s_end - s_begin);
    }
  } else if (warp >= FIRST_EPI) {
    // =========================================== epilogue ================================================
    // Two groups of 4 warps (one per TMEM lane quarter); outputs alternate between the groups, so two accumulators are
    // drained concurrently.  A thread owns one output row and all 32 channels of the slice, processed 16 at a time.
    const int ew = warp - FIRST_EPI;
    const int quarter = warp & 3;                 // TMEM lane quarter this warp may access
    const int eg = ew >> 2;                       // epilogue group
    const int row = quarter * 32 + lane;
    __nv_bfloat16* yg = p.y[g];
    const bool want_stats = p.stats[g] != nullptr;
    const bool no_shift = (p.debug & 1) != 0, no_store = (p.debug & 2) != 0;
    const bool has_bias = p.bias[g] != nullptr;
    // Packed fp32 pairs (FADD2 / FFMA2): the epilogue is bound by issue slots and dependent-issue latency of its 8 warps, not
    // by TMEM or memory (TMF_COL_DEBUG=32: issuers of the Cin = 32 layers wait 35 % of the time for a free accumulator).
    uint64_t acc_s[CC_CO / 2], acc_q[CC_CO / 2];
#pragma unroll
    for (int j = 0; j < CC_CO / 2; ++j) { acc_s[j] = 0ull; acc_q[j] = 0ull; }
    const uint64_t m_in = pair_f32(lane < 31 ? 1.f : 0.f, lane < 31 ? 1.f : 0.f);   // rows whose +1 neighbour is in this warp
    const uint64_t m_31 = pair_f32(lane == 31 ? 1.f : 0.f, lane == 31 ? 1.f : 0.f);
    const uint64_t* bias2 = reinterpret_cast<const uint64_t*>(bias_ptr);
    long long t_epi = 0;
    const long long t_epi0 = clock64();
    uint32_t xb = 0;                              // exchange buffer parity
    int it = NS ? 0 : eg;
    int s = s_begin + (NS ? 0 : eg);
    int d = s % p.D, col = s / p.D;
    bool new_col = true, valid = false;
    const int64_t dstride = (int64_t)p.H * p.W * p.cout;
    __nv_bfloat16* ycol = yg;
    if (NS) {
      // every output, this group's 32 of the CTA's 64 channels: TMEM columns [32 eg, 32 eg + 32) of the accumulator buffer
      const int ch0 = 32 * eg;
      for (; s < s_end; ++s, ++it) {
        if (new_col) {
          const int c = col % p.NC, n = col / p.NC;
          const int q = c * TILE_OUT + row;
          const int h = q / p.Wp, w = q - h * p.Wp;
          valid = (h < p.H) && (w < p.W) && !no_store;
          ycol = yg + (((int64_t)n * p.D * p.H + h) * p.W + w) * p.cout + co_off + ch0;
          new_col = false;
        }
        __nv_bfloat16* yrow = ycol + d * dstride;
        if (++d >= p.D) { d = 0; ++col; new_col = true; }
        const int as = it & (CC_NBUF - 1);
        mbar_wait_t(acc_full + 8 * as, (uint32_t)(it / CC_NBUF) & 1u, t_epi, prof);
        tc_fence_after();
        const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(as * NCOLS + ch0);
#pragma unroll
        for (int hf = 0; hf < 2; ++hf) {
          uint32_t r[16];
          tmem_ld16(taddr + hf * 16, r);
          tmem_ld_wait();
          if (hf == 1) {                                                // last TMEM read of this accumulator buffer
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(acc_empty + 8 * as);
          }
          if (valid) {
            uint32_t pk[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const uint64_t a2 = pair_u32(r[2 * j], r[2 * j + 1]);
              const uint64_t o = has_bias ? add2_f32(a2, bias2[(ch0 >> 1) + hf * 8 + j]) : a2;
              pk[j] = pack_bf16(__uint_as_float(lo_u32(o)), __uint_as_float(hi_u32(o)));
            }
            if (want_stats) {
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                const uint64_t f = pair_u32(pk[j] << 16, pk[j] & 0xffff0000u);        // the stored (rounded) values
                acc_s[hf * 8 + j] = add2_f32(acc_s[hf * 8 + j], f);
                acc_q[hf * 8 + j] = fma2_f32(f, f, acc_q[hf * 8 + j]);
              }
            }
            asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(yrow + hf * 16), "r"(pk[0]), "r"(pk[1]),
                         "r"(pk[2]), "r"(pk[3]), "r"(pk[4]), "r"(pk[5]), "r"(pk[6]), "r"(pk[7])
                         : "memory");
          }
        }
      }
    }
    for (; !NS && s < s_end; s += 2, it += 2) {
      if (new_col) {                              // (every D / 2 outputs: the divisions stay out of the per-output path)
        const int c = col % p.NC, n = col / p.NC;
        const int q = c * CC_TILE_OUT + row;
        const int h = q / p.Wp, w = q - h * p.Wp;
        valid = (row < CC_TILE_OUT) && (h < p.H) && (w < p.W) && !no_store;
        ycol = yg + (((int64_t)n * p.D * p.H + h) * p.W + w) * p.cout + co_off;
        new_col = false;
      }
      __nv_bfloat16* yrow = ycol + d * dstride;
      d += 2;
      while (d >= p.D) { d -= p.D; ++col; new_col = true; }
      const int as = it & (CC_NBUF - 1);
      mbar_wait_t(acc_full + 8 * as, (uint32_t)(it / CC_NBUF) & 1u, t_epi, prof);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(as * CC_NSTACK);
      // Every accumulator value is read from TMEM once.  Per 16-channel half: load D0, D1, D2; lane 0 publishes its D1 / D2
      // and lane 1 its D2 for the previous lane quarter; the two-row shift is done with shuffles -- rows 30 / 31 of a quarter
      // lack the terms of the next quarter -- both halves stay in registers, ONE group barrier, then rows 30 / 31 add the
      // published terms and everybody stores.   T[r] = D1[r] + D2[r+1];  y[r] = D0[r] + T[r+1].
      float* xw = xchg_ptr + (((xb * 2 + eg) * 4 + quarter) * 3) * 32;                       // [D1 row0 | D2 row0 | D2 row1][32]
      const float* xr = xchg_ptr + (((xb * 2 + eg) * 4 + ((quarter + 1) & 3)) * 3) * 32;
      xb ^= 1u;
      uint64_t v[2][8];
#pragma unroll
      for (int hf = 0; hf < 2; ++hf) {
        uint32_t r0[16], r1[16], r2[16];
        tmem_ld16(taddr + hf * 16, r0);
        tmem_ld16(taddr + CC_CO + hf * 16, r1);
        tmem_ld16(taddr + 2 * CC_CO + hf * 16, r2);
        tmem_ld_wait();
        if (hf == 1) {                               // last TMEM read of this accumulator buffer
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(acc_empty + 8 * as);
        }
        if (no_shift) {
#pragma unroll
          for (int j = 0; j < 8; ++j)
            v[hf][j] = add2_f32(pair_u32(r0[2 * j], r0[2 * j + 1]), add2_f32(pair_u32(r1[2 * j], r1[2 * j + 1]), pair_u32(r2[2 * j], r2[2 * j + 1])));
        } else {
          if (lane == 0) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              reinterpret_cast<uint4*>(xw + hf * 16)[j] = make_uint4(r1[4 * j], r1[4 * j + 1], r1[4 * j + 2], r1[4 * j + 3]);
              reinterpret_cast<uint4*>(xw + 32 + hf * 16)[j] = make_uint4(r2[4 * j], r2[4 * j + 1], r2[4 * j + 2], r2[4 * j + 3]);
            }
          } else if (lane == 1) {
#pragma unroll
            for (int j = 0; j < 4; ++j)
              reinterpret_cast<uint4*>(xw + 64 + hf * 16)[j] = make_uint4(r2[4 * j], r2[4 * j + 1], r2[4 * j + 2], r2[4 * j + 3]);
          }
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const uint32_t da = __shfl_down_sync(0xffffffffu, r2[2 * j], 1), db = __shfl_down_sync(0xffffffffu, r2[2 * j + 1], 1);
            const uint64_t tt = fma2_f32(pair_u32(da, db), m_in, pair_u32(r1[2 * j], r1[2 * j + 1]));
            const uint32_t ta = __shfl_down_sync(0xffffffffu, lo_u32(tt), 1), tb = __shfl_down_sync(0xffffffffu, hi_u32(tt), 1);
            v[hf][j] = fma2_f32(pair_u32(ta, tb), m_in, pair_u32(r0[2 * j], r0[2 * j + 1]));
          }
        }
      }
      if (!no_shift) {
        asm volatile("bar.sync %0, 128;" ::"r"(1 + eg) : "memory");
        if (lane >= 30) {
          // row 30: y += D2next[0];   row 31: y += D1next[0] + D2next[1]   (same instructions, different addresses)
          const ulonglong2* pa = reinterpret_cast<const ulonglong2*>(xr + (lane == 31 ? 0 : 32));
          const ulonglong2* pb = reinterpret_cast<const ulonglong2*>(xr + 64);
#pragma unroll
          for (int hf = 0; hf < 2; ++hf)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const ulonglong2 a2 = pa[hf * 4 + j], b2 = pb[hf * 4 + j];
              v[hf][2 * j] = add2_f32(v[hf][2 * j], fma2_f32(b2.x, m_31, a2.x));
              v[hf][2 * j + 1] = add2_f32(v[hf][2 * j + 1], fma2_f32(b2.y, m_31, a2.y));
            }
        }
      }
      if (valid) {
#pragma unroll
        for (int hf = 0; hf < 2; ++hf) {
          uint32_t pk[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const uint64_t o = has_bias ? add2_f32(v[hf][j], bias2[hf * 8 + j]) : v[hf][j];     // shared-memory broadcast
            pk[j] = pack_bf16(__uint_as_float(lo_u32(o)), __uint_as_float(hi_u32(o)));
          }
          if (want_stats) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const uint64_t f = pair_u32(pk[j] << 16, pk[j] & 0xffff0000u);        // the stored (rounded) values
              acc_s[hf * 8 + j] = add2_f32(acc_s[hf * 8 + j], f);
              acc_q[hf * 8 + j] = fma2_f32(f, f, acc_q[hf * 8 + j]);
            }
          }
          // one 256-bit store: a thread writes whole 32-byte sectors
          asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(yrow + hf * 16), "r"(pk[0]), "r"(pk[1]),
                       "r"(pk[2]), "r"(pk[3]), "r"(pk[4]), "r"(pk[5]), "r"(pk[6]), "r"(pk[7])
                       : "memory");
        }
      }
    }
    if (prof && blockIdx.x == 0 && ew == 0 && lane == 0)
      printf("col prof: epilogue warp 0: total %lld cyc, waiting for a finished accumulator %lld\n", clock64() - t_epi0, t_epi);
    if (want_stats) {
      // deterministic: shuffle tree per warp -> one slot per warp -> fixed-order sum -> this CTA's row of the buffer
#pragma unroll
      for (int j = 0; j < CC_CO; ++j) {
        const uint64_t ps = acc_s[j >> 1], pq = acc_q[j >> 1];
        const float ssum = warp_sum(__uint_as_float((j & 1) ? hi_u32(ps) : lo_u32(ps)));
        const float qsum = warp_sum(__uint_as_float((j & 1) ? hi_u32(pq) : lo_u32(pq)));
        if (lane == 0) {
          stats_ptr[ew * 64 + j] = ssum;
          stats_ptr[ew * 64 + 32 + j] = qsum;
        }
      }
      asm volatile("bar.sync 3, %0;" ::"r"(32 * CC_EPI_WARPS) : "memory");
      const int i = threadIdx.x - 32 * FIRST_EPI;
      if (NS) {
        if (i < 2 * NCO) {                          // i = which * 64 + channel; the channel's group holds it in its four warps
          const int which = i / NCO, ch = i - which * NCO, grp = ch >> 5, j = ch & 31;
          double tot = 0.0;
#pragma unroll
          for (int w4 = 0; w4 < 4; ++w4) tot += (double)stats_ptr[(grp * 4 + w4) * 64 + which * 32 + j];
          stat_row_store(p.stats[g], 2 * p.cout, cta, ncta, which * p.cout + co_off + ch, tot);
        }
      } else if (i < 2 * CC_CO) {
        double tot = 0.0;
#pragma unroll
        for (int w8 = 0; w8 < CC_EPI_WARPS; ++w8) tot += (double)stats_ptr[w8 * 64 + i];
        const int col = (i < CC_CO) ? (co_off + i) : (p.cout + co_off + (i - CC_CO));
        stat_row_store(p.stats[g], 2 * p.cout, cta, ncta, col, tot);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ------------------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn col_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn == nullptr) {
    void* sym = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(sym);
  }
  return fn;
}

struct ColPlan {
  bool ok;
  int Wp, NH, NC, S, nsplit, qneed, ns;
  uint32_t slot_bytes, a_tx, b_bytes, smem_bytes, layout;
  CUtensorMapSwizzle swz;
};

static ColPlan make_col_plan(int ng, int D, int H, int W, int cin, int cout, int ks) {
  ColPlan pl{};
  pl.ok = false;
  if (ks != 3) return pl;
  if (!(cin == 32 || cin == 64) || cout % CC_CO != 0 || cout < CC_CO) return pl;
  // non-stacked variant: Cin = 32 with 64 output channels per CTA (conv2.3 forward); TMF_COL_NS=0 keeps the kw-stacked tiles
  {
    const char* e = getenv("TMF_COL_NS");
    pl.ns = (cin == 32 && cout % CC_NS_CO == 0 && !(e != nullptr && atoi(e) == 0)) ? 1 : 0;
  }
  const int nco = pl.ns ? CC_NS_CO : CC_CO;
  pl.nsplit = cout / nco;
  if (ng * pl.nsplit > CC_MAX_VG) return pl;
  if (D < 1 || H < 1 || W < 2) return pl;
  const uint32_t pitch = (uint32_t)cin * 2;
  pl.layout = (cin == 64) ? LAYOUT_SW128 : LAYOUT_SW64;
  pl.swz = (cin == 64) ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
  pl.Wp = W + 1;
  if (pl.Wp > 256) return pl;
  pl.qneed = (H - 1) * pl.Wp + W;
  pl.b_bytes = 27u * (uint32_t)nco * pitch;
  const uint32_t wbytes = (pl.b_bytes + 1023u) & ~1023u;
  const int rmax = (pl.Wp - 1) + 127 + 2 * pl.Wp + (pl.ns ? 2 : 0);      // NS: the kw shift is two more rows of the window
  pl.NH = rmax / pl.Wp + 1;
  if (pl.NH > 256) return pl;
  pl.a_tx = (uint32_t)pl.NH * pl.Wp * pitch;
  pl.slot_bytes = (pl.a_tx + 1023u) & ~1023u;
  for (int S = CC_MAX_SLOTS; S >= 2; --S) {
    const uint32_t total = CC_FIXED_SMEM + wbytes + (uint32_t)S * pl.slot_bytes;
    if (total <= CC_SMEM_BUDGET) {
      pl.ok = true; pl.S = S; pl.smem_bytes = total;
      break;
    }
  }
  if (!pl.ok) return pl;
  const int tile_out = pl.ns ? 128 : CC_TILE_OUT;
  pl.NC = (pl.qneed + tile_out - 1) / tile_out;
  return pl;
}

}  // namespace tmf

using namespace tmf;

// host-only introspection of the column kernel's launch plan (tests / DESIGN.md): out6 = {ok, non-stacked variant, Cout blocks per
// tower, tiles per plane, ring slots, slab rows}
extern "C" int tmf_conv3d_col_plan_info(int ng, int D, int H, int W, int cin, int cout, int ksize, int* out6) {
  const ColPlan pl = make_col_plan(ng, D, H, W, cin, cout, ksize);
  if (out6 != nullptr) {
    out6[0] = pl.ok ? 1 : 0; out6[1] = pl.ns; out6[2] = pl.nsplit; out6[3] = pl.NC; out6[4] = pl.S; out6[5] = pl.NH;
  }
  return pl.ok ? 0 : 1;
}

bool tmf_conv3d_fwd_col_supported(int ng, int D, int H, int W, int cin, int cout, int ksize) {
  if (getenv("TMF_DISABLE_UMMA") != nullptr) return false;
  return make_col_plan(ng, D, H, W, cin, cout, ksize).ok;
}

int tmf_conv3d_fwd_col(int ng, const void* const* a, const void* const* wf, const float* const* bias, void* const* y,
                       double* const* stats, int B, int D, int H, int W, int cin, int cout, int ksize, void* stream) {
  TMF_CHECK_NG(ng);
  const ColPlan pl = make_col_plan(ng, D, H, W, cin, cout, ksize);
  TMF_REQUIRE(pl.ok, "conv3d_fwd_col: unsupported problem");
  EncodeTiledFn encode = col_encode_fn();
  TMF_REQUIRE(encode != nullptr, "conv3d_fwd_col: cuTensorMapEncodeTiled entry point not available");
  TMF_REQUIRE((int64_t)B * pl.NC * D < (int64_t)1 << 30, "conv3d_fwd_col: problem too large");
  ColConvParams p{};
  p.ng = ng; p.nsplit = pl.nsplit; p.cout = cout; p.B = B; p.D = D; p.H = H; p.W = W;
  p.Wp = pl.Wp; p.NH = pl.NH; p.NC = pl.NC; p.S = pl.S; p.qneed = pl.qneed;
  p.steps_per_group = B * pl.NC * D;
  p.layout = pl.layout; p.slot_bytes = pl.slot_bytes; p.a_tx_bytes = pl.a_tx; p.b_bytes = pl.b_bytes;
  p.idesc = make_idesc_bf16(128, pl.ns ? CC_NS_CO : CC_NSTACK, 0, 0);
  p.ns = pl.ns;
  p.debug = getenv("TMF_COL_DEBUG") ? atoi(getenv("TMF_COL_DEBUG")) : 0;
  cudaStream_t st = (cudaStream_t)stream;
  for (int g = 0; g < ng; ++g) {
    TMF_REQUIRE(a[g] && wf[g] && y[g], "conv3d_fwd_col: NULL device pointer");
    TMF_REQUIRE(((uintptr_t)a[g] & 15) == 0 && ((uintptr_t)wf[g] & 15) == 0 && ((uintptr_t)y[g] & 31) == 0,
                "conv3d_fwd_col: tensors must be 16-byte (output: 32-byte) aligned");
    p.bias[g] = bias ? bias[g] : nullptr;
    p.y[g] = (__nv_bfloat16*)y[g];
    p.stats[g] = stats ? stats[g] : nullptr;
    {
      cuuint64_t dims[5] = {(cuuint64_t)cin, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)D, (cuuint64_t)B};
      cuuint64_t strides[4] = {(cuuint64_t)cin * 2, (cuuint64_t)W * cin * 2, (cuuint64_t)H * W * cin * 2,
                               (cuuint64_t)D * H * W * cin * 2};
      cuuint32_t box[5] = {(cuuint32_t)cin, (cuuint32_t)pl.Wp, (cuuint32_t)pl.NH, 1, 1};
      cuuint32_t estr[5] = {1, 1, 1, 1, 1};
      CUresult r = encode(&p.tmA[g], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<void*>(a[g]), dims, strides, box,
                          estr, CU_TENSOR_MAP_INTERLEAVE_NONE, pl.swz, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      TMF_REQUIRE(r == CUDA_SUCCESS, "conv3d_fwd_col: cuTensorMapEncodeTiled(A) failed with %d", (int)r);
    }
    {
      cuuint64_t dims[3] = {(cuuint64_t)cin, (cuuint64_t)cout, 27};
      cuuint64_t strides[2] = {(cuuint64_t)cin * 2, (cuuint64_t)cout * cin * 2};
      cuuint32_t box[3] = {(cuuint32_t)cin, (cuuint32_t)(pl.ns ? CC_NS_CO : CC_CO), 27};
      cuuint32_t estr[3] = {1, 1, 1};
      CUresult r = encode(&p.tmB[g], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(wf[g]), dims, strides, box,
                          estr, CU_TENSOR_MAP_INTERLEAVE_NONE, pl.swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      TMF_REQUIRE(r == CUDA_SUCCESS, "conv3d_fwd_col: cuTensorMapEncodeTiled(B) failed with %d", (int)r);
    }
  }
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int ngv = ng * pl.nsplit;
  int per_group = sms / ngv;
  if (per_group > p.steps_per_group) per_group = p.steps_per_group;
  if (per_group > TMF_STAT_ROWS) per_group = TMF_STAT_ROWS;        // one statistics row per CTA of a (tower, slice)
  if (per_group < 1) per_group = 1;
  dim3 grid(per_group * ngv, 1, 1);
#define TMF_LAUNCH_COL(KST, NSV)                                                                                         \
  do {                                                                                                                  \
    static bool attr_done = false;                                                                                      \
    if (!attr_done) {                                                                                                   \
      TMF_CUDA(cudaFuncSetAttribute(conv3d_umma_col_kernel<KST, NSV>, cudaFuncAttributeMaxDynamicSharedMemorySize,      \
                                    (int)CC_SMEM_BUDGET));                                                              \
      attr_done = true;                                                                                                 \
    }                                                                                                                   \
    launch_k(conv3d_umma_col_kernel<KST, NSV>, grid, ColRoles<NSV>::THREADS, pl.smem_bytes, st, p);                                 \
  } while (0)
  if (cin == 32 && pl.ns) TMF_LAUNCH_COL(2, true);
  else if (cin == 32) TMF_LAUNCH_COL(2, false);
  else TMF_LAUNCH_COL(4, false);
#undef TMF_LAUNCH_COL
  TMF_LAUNCH_CHECK();
  return 0;
}

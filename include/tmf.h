/* tmf.h -- C ABI of libtmf_sm100a.so: the B200 (sm_100a) kernels behind TransMF_AD's training hot path.
 *
 * The reference (Kateridge/TransMF_AD) has no native layer: its "FFI" for this path is the set of
 * torch.nn / ATen calls made by models/networks.py and models/mymodel.py.  Each entry point below names the
 * reference call site(s) it replaces.  Conventions:
 *   - plain pointers and sizes only; every device buffer (incl. workspaces) is owned by the caller;
 *   - `stream` is a cudaStream_t passed as void*; all work is stream-ordered, no internal synchronisation;
 *   - return 0 on success, non-zero on error; tmf_last_error() returns a thread-local message;
 *   - no CPU fallback and no other architecture: tmf_check_device() fails unless the device is cc 10.x;
 *   - "groups": the two sNet towers (MRI, PET) have identical shapes but separate tensors, so the conv-stack
 *     entry points take `ng` (1 or 2) and, for every tensor, a HOST array of `ng` device pointers; both
 *     towers run in one launch (grid.z = group).
 *   - activations are NDHWC ("channels-last-3d"): index ((((n*D + d)*H + h)*W + w)*C + c).
 *   - bf16 buffers are passed as void*; fp32 as float*; per-channel statistics accumulate in double.
 *   - DETERMINISM.  Per-channel statistics buffers (`stats` of the conv forward entry points, `sums` of the BatchNorm
 *     backward reductions) are double[TMF_STAT_ROWS][2*C]: row r holds the partial {sum, sum of squares} (or {sum dz,
 *     sum dz*xhat}) of producer CTA r of that tower.  A producer launches at most TMF_STAT_ROWS CTAs per tower, every
 *     row is written exactly once per call (rows without a CTA are cleared by the kernel, so callers never zero the
 *     buffer) and tmf_bn_finalize / tmf_bn_bwd_finalize add the rows in index order: no floating-point atomics, bitwise
 *     reproducible run to run.  (The CUDA-core bring-up kernels, TMF_CONV_DIRECT, still add with atomics.)
 */
#ifndef TMF_H_
#define TMF_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TMF_MAX_GROUPS 2
/* rows of a per-channel statistics buffer (see DETERMINISM above): 2 CTAs per SM of a 148-SM B200 */
#define TMF_STAT_ROWS 296

/* pooling modes fused behind BatchNorm + LeakyReLU (reference models/networks.py:25,34,43 MaxPool3d(2,2);
 * :52 AvgPool3d(2,2); floor mode) */
#define TMF_POOL_NONE 0
#define TMF_POOL_MAX 1
#define TMF_POOL_AVG 2

/* conv implementation selector */
#define TMF_CONV_AUTO 0
#define TMF_CONV_DIRECT 1   /* CUDA-core implicit GEMM (bring-up / cross-check path) */
#define TMF_CONV_UMMA 2     /* tcgen05 / TMEM / TMA implicit GEMM */

/* ---------------------------------------------------------------------------------------------------------- */
/* library                                                                                                    */
const char* tmf_last_error(void);
int tmf_version(void);
/* 0 iff the current CUDA device is a cc 10.x part (B200); otherwise an error (no fallback). */
int tmf_check_device(void);
/* number of kernel launches issued through this library by the calling process so far */
int64_t tmf_launch_count(void);
/* which attention kernels tmf_attn_fwd / tmf_attn_bwd try first (TMF_ATTN_IMPL, read once): 2 = tensor-core (attention_mma.cu,
 * default), 1 = register-tiled fp32 (attention.cu), 0 = row-per-warp fp32 (fusion_ops.cu) */
int tmf_attn_impl_default(void);
/* TMF_STAT_ROWS, for callers that size statistics buffers without the header */
int tmf_stat_rows(void);

/* ---------------------------------------------------------------------------------------------------------- */
/* sNet conv stack -- replaces nn.Conv3d / nn.BatchNorm3d / nn.LeakyReLU / nn.MaxPool3d / nn.AvgPool3d of        */
/* reference models/networks.py:21-53 (forward) and their autograd backward.                                   */

/* fp32 master weight (Cout,Cin,k,k,k) -> bf16 wf[tap][Cout][Cin] (forward operand) and, if wd != NULL,
 * bf16 wd[tap][Cin][Cout] with flipped taps (dgrad operand).  k = 3 (27 taps) or 1. */
int tmf_pack_conv_weights(int ng, const float* const* w, void* const* wf, void* const* wd,
                          int cout, int cin, int ksize, void* stream);

/* conv1.0 (Cin = 1, 3x3x3, pad 1), fp32 input and weights, bf16 output y[B,D,H,W,Cout], per-channel
 * sum / sum-of-squares of the stored (rounded) y into stats[TMF_STAT_ROWS][2*Cout] (double partial rows).
 * impl: TMF_CONV_AUTO / _DIRECT (CUDA cores, fp32) / _UMMA (tcgen05 on an in-smem im2col with a bf16 hi/lo split of
 * both operands, fp32-level accuracy).   reference models/networks.py:22 */
int tmf_conv1_fwd(int ng, const float* const* x, const float* const* w, const float* const* bias,
                  void* const* y, double* const* stats, int B, int D, int H, int W, int cout, int impl, void* stream);

/* dW[Cout][27] of conv1.0 from dy (bf16) and x (fp32); dw is overwritten.  `ws`: caller-owned, 16-byte aligned scratch
 * of at least tmf_conv1_wgrad_workspace_bytes(...) bytes (per-CTA partial sums of the tcgen05 path, added in CTA
 * order -> deterministic); may be NULL when that returns 0 (CUDA-core bring-up path).
 * reference models/networks.py:22 (autograd backward of Conv3d(1,32,3,p1)) */
int tmf_conv1_wgrad(int ng, const void* const* dy, const float* const* x, float* const* dw,
                    int B, int D, int H, int W, int cout, int impl, void* ws, size_t ws_bytes, void* stream);
int64_t tmf_conv1_wgrad_workspace_bytes(int ng, int impl, int W, int cout);

/* Block-1 backward in one pass over y: the BatchNorm + LeakyReLU + MaxPool3d(2,2) backward "apply" (what
 * tmf_bn_act_pool_bwd_apply computes with pool = TMF_POOL_MAX) fused with the conv1.0 weight gradient, so dy of
 * block 1 (which feeds nothing else: conv1.0's input is the image) never goes to HBM.  dout: bf16 pooled gradient
 * [B,D/2,H/2,W/2,32]; y: bf16 conv1.0 output [B,D,H,W,32]; coef / bcoef as below; x: fp32 image; dw (32,1,3,3,3) is
 * overwritten (deterministic reduction).  `ws`: caller-owned, 256-byte aligned scratch of at least
 * tmf_conv1_bwd_fused_workspace_bytes(...) bytes; that function returns 0 when the problem is not supported
 * (Cout != 32, W > 240, ...) -- callers then use tmf_bn_act_pool_bwd_apply + tmf_conv1_wgrad.
 * reference models/networks.py:22-25 (autograd backward of Conv3d(1,32,3,p1) / BatchNorm3d / LeakyReLU / MaxPool3d) */
int tmf_conv1_bwd_fused(int ng, const void* const* dout, const void* const* y, const float* const* coef,
                        const float* const* bcoef, const float* const* x, float* const* dw, int B, int D, int H,
                        int W, int cout, float slope, void* ws, size_t ws_bytes, void* stream);
int64_t tmf_conv1_bwd_fused_workspace_bytes(int ng, int B, int D, int H, int W, int cout);

/* Block-1 gradient with respect to the input image (saliency maps, integrated gradients, input-space attacks): the
 * BatchNorm + LeakyReLU + MaxPool3d(2,2) backward "apply" (dy recomputed from the stored y exactly as
 * tmf_bn_act_pool_bwd_apply computes it with pool = TMF_POOL_MAX; never written to HBM on the tcgen05 path) followed by
 * the data gradient of conv1.0:  dx[p] = sum_tap sum_co dy[p - off(tap)][co] * w[co][tap]  (zero padding 1).
 * dout: bf16 pooled gradient [B,D/2,H/2,W/2,Cout]; y: bf16 conv1.0 output [B,D,H,W,Cout]; coef / bcoef as below;
 * w: fp32 conv1.0 weight (Cout,1,3,3,3); dx: fp32 [B,D,H,W] (= (B,1,D,H,W)), overwritten, every element written once in a
 * fixed summation order (no atomics: bitwise reproducible, and a tower's result does not depend on ng).
 * impl: TMF_CONV_UMMA (tcgen05, Cout = 32, W <= 128; the weight as bf16 hi + lo halves, fp32-level accuracy),
 * TMF_CONV_DIRECT (CUDA cores: tmf_bn_act_pool_bwd_apply into the workspace, then an fp32 direct kernel; Cout a multiple
 * of 8 in [8,64]) or TMF_CONV_AUTO (tcgen05 where supported, else direct).  `ws`: caller-owned, 256-byte aligned scratch
 * of at least tmf_conv1_dgrad_fused_workspace_bytes(...) bytes; may be NULL when that returns 0.
 * reference models/networks.py:22-25 (autograd backward of Conv3d(1,32,3,p1) / BatchNorm3d / LeakyReLU / MaxPool3d
 * with respect to the image) */
int tmf_conv1_dgrad_fused(int ng, const void* const* dout, const void* const* y, const float* const* coef,
                          const float* const* bcoef, const float* const* w, float* const* dx, int B, int D, int H, int W,
                          int cout, float slope, int impl, void* ws, size_t ws_bytes, void* stream);
int64_t tmf_conv1_dgrad_fused_workspace_bytes(int ng, int impl, int B, int D, int H, int W, int cout);

/* 3x3x3 (pad 1) or 1x1x1 convolution, bf16 NDHWC input a[B,D,H,W,Cin], packed bf16 weights wf[tap][Cout][Cin],
 * optional fp32 bias, bf16 output y[B,D,H,W,Cout], optional stats (as above; NULL array = none).
 * Also used for dgrad (a = dy, wf = flipped/transposed pack, bias = stats = NULL).
 * reference models/networks.py:28,31,37,40,46,49 */
int tmf_conv3d_fwd(int ng, const void* const* a, const void* const* wf, const float* const* bias,
                   void* const* y, double* const* stats, int B, int D, int H, int W, int cin, int cout,
                   int ksize, int impl, void* stream);

/* dW (fp32, reference layout (Cout,Cin,k,k,k), overwritten) = sum_v dy[v,co] * a[v+tap,ci].
 * `ws` is caller-owned scratch of at least tmf_conv3d_wgrad_workspace_bytes(...) bytes (fp32 split-K partials of the
 * tcgen05 path, reduced in a fixed order -> deterministic); may be NULL when that returns 0. */
int tmf_conv3d_wgrad(int ng, const void* const* dy, const void* const* a, float* const* dw,
                     int B, int D, int H, int W, int cin, int cout, int ksize, int impl,
                     void* ws, size_t ws_bytes, void* stream);
int64_t tmf_conv3d_wgrad_workspace_bytes(int ng, int impl, int B, int D, int H, int W, int cin, int cout, int ksize);

/* 1 if implementation `impl` (TMF_CONV_DIRECT / TMF_CONV_UMMA) handles this problem, else 0.
 * op: 0 = forward / dgrad (tmf_conv3d_fwd), 1 = weight gradient (tmf_conv3d_wgrad). */
int tmf_conv3d_supported(int op, int impl, int D, int H, int W, int cin, int cout, int ksize);

/* Introspection (host only, no device work): the launch plan of the generic tcgen05 forward/dgrad kernel
 * (conv_umma.cu) for this problem (ng towers of batch B: the plan weighs wave quantisation).  out8 = {ok, 128-row tiles per weight pass, issuer warps, accumulator sets,
 * input stages, weight stages, super-tiles per plane, weights resident}.  Returns 0 if the kernel takes the problem. */
int tmf_conv3d_umma_plan_info(int ng, int B, int D, int H, int W, int cin, int cout, int ksize, int* out8);
/* host-only: launch plan of the column kernel (conv_umma_col.cu: Cin 32 / 64 layers) for one problem; out6 = {ok, non-stacked
 * variant (Cin = 32, Cout a multiple of 64), Cout blocks per tower, 128-row tiles per plane, input ring slots, slab rows}.
 * Returns 0 iff the kernel takes the problem. */
int tmf_conv3d_col_plan_info(int ng, int D, int H, int W, int cin, int cout, int ksize, int* out6);

/* BatchNorm statistics -> coefficients.  coef[4*C] = {scale = gamma*invstd, shift = beta - mean*scale, mean,
 * invstd}.  training != 0: batch statistics from stats (biased variance), running_mean/var updated with
 * momentum (unbiased variance) and num_batches_tracked += 1; training == 0: running statistics.
 * reference models/networks.py:23,29,32,38,41,47,50 */
int tmf_bn_finalize(int ng, const double* const* stats, const float* const* gamma, const float* const* beta,
                    float* const* running_mean, float* const* running_var, int64_t* const* num_batches_tracked,
                    float* const* coef, int C, int64_t count, float momentum, float eps, int training,
                    void* stream);

/* out = pool(leaky_relu(y*scale + shift)); out is bf16, or fp32 when out_fp32 != 0.  Floor-mode 2x2x2 pools. */
int tmf_bn_act_pool_fwd(int ng, const void* const* y, const float* const* coef, void* const* out, int out_fp32,
                        int B, int D, int H, int W, int C, int pool, float slope, void* stream);

/* tmf_bn_act_pool_fwd for a MAX pool that also keeps ymax[B,D/2,H/2,W/2,C] (bf16): the stored pre-BN value behind each
 * window's maximum activation, at the position every max-pool backward kernel routes to: the first in (d,h,w) scan order
 * that maximises sign(scale)*y (position 0 where scale = 0).  It holds the maximum activation because the map is
 * non-decreasing, which needs slope >= 0 (refused otherwise, like every max-pool entry point below).  The backward
 * reduction of the layer then runs on ymax + dout at pooled resolution (tmf_bn_maxpool_bwd_reduce_kept) instead of
 * re-reading y.  networks.py:23-25. */
int tmf_bn_act_pool_fwd_keepmax(int ng, const void* const* y, const float* const* coef, void* const* out,
                                void* const* ymax, int out_fp32, int B, int D, int H, int W, int C, float slope,
                                void* stream);
/* Dual-output variants of the two passes above for a block boundary whose output is exposed (module hooks on the sNet
 * blocks, Grad-CAM): out (bf16, the next conv's operand) and ymax are the same bits as tmf_bn_act_pool_fwd /
 * tmf_bn_act_pool_fwd_keepmax write with out_fp32 = 0, and out32 (fp32, same layout) receives the value before rounding,
 * i.e. the fp32 number whose round-to-nearest bf16 is out.  networks.py:25,34,43,52 (the nn.Sequential block outputs). */
int tmf_bn_act_pool_fwd_dual(int ng, const void* const* y, const float* const* coef, void* const* out,
                             float* const* out32, int B, int D, int H, int W, int C, int pool, float slope, void* stream);
int tmf_bn_act_pool_fwd_keepmax_dual(int ng, const void* const* y, const float* const* coef, void* const* out,
                                     float* const* out32, void* const* ymax, int B, int D, int H, int W, int C, float slope,
                                     void* stream);
/* n elements (a multiple of 8) bf16 -> fp32 (exact) and fp32 -> bf16 (round to nearest even), per tower: the gradient at
 * an exposed block boundary (the bf16 dgrad output widened for autograd; an fp32 gradient narrowed for block 1's fused
 * backward kernels). */
int tmf_widen_bf16(int ng, const void* const* src, float* const* dst, int64_t n, void* stream);
int tmf_narrow_f32(int ng, const float* const* src, void* const* dst, int64_t n, void* stream);

/* sums[TMF_STAT_ROWS][2*C] (double partial rows) = {sum dz, sum dz*xhat} of a max-pool layer from ymax and dout (both at pooled extents Do,Ho,Wo):
 * same result as tmf_bn_act_pool_bwd_reduce(pool = TMF_POOL_MAX) up to summation order. */
int tmf_bn_maxpool_bwd_reduce_kept(int ng, const void* const* dout, int dout_fp32, const void* const* ymax,
                                   const float* const* coef, double* const* sums, int B, int Do, int Ho, int Wo, int C,
                                   float slope, void* stream);

/* backward, pass 1: sums[TMF_STAT_ROWS][2*C] (double partial rows) = {sum dz, sum dz*xhat} with
 * dz = unpool(dout) * leaky_relu'(z) (max-pool routes to the first maximum in (d,h,w) scan order). */
int tmf_bn_act_pool_bwd_reduce(int ng, const void* const* dout, int dout_fp32, const void* const* y,
                               const float* const* coef, double* const* sums, int B, int D, int H, int W, int C,
                               int pool, float slope, void* stream);

/* backward, between the passes: dgamma, dbeta (fp32, overwritten), dbias (conv bias grad; may be NULL),
 * bcoef[2*C] = {mean(dz), mean(dz*xhat)} (zeros in eval mode). */
int tmf_bn_bwd_finalize(int ng, const double* const* sums, const float* const* coef, float* const* dgamma,
                        float* const* dbeta, float* const* dbias, float* const* bcoef, int C, int64_t count,
                        int training, void* stream);

/* backward, pass 2: dy (bf16 [B,D,H,W,C]) = scale * (dz - mean(dz) - xhat * mean(dz*xhat)). */
int tmf_bn_act_pool_bwd_apply(int ng, const void* const* dout, int dout_fp32, const void* const* y,
                              const float* const* coef, const float* const* bcoef, void* const* dy,
                              int B, int D, int H, int W, int C, int pool, float slope, void* stream);

/* ---------------------------------------------------------------------------------------------------------- */
/* fusion transformer / heads (fp32 tensors, row-major)                                                        */

/* y[M,N] = act(x[M,K] . w[N,K]^T + bias) + residual; act: 0 none, 1 exact-erf GELU; bias/residual may be NULL.
 * If pre != NULL the pre-activation is also stored there.   reference nn.Linear at models/networks.py:128,132,
 * 149,150,153; models/mymodel.py:190-194 */
int tmf_linear_fwd(const float* x, const float* w, const float* bias, const float* residual, float* y, float* pre,
                   int M, int K, int N, int act, void* stream);
/* dx[M,K] (+)= dy[M,N] . w[N,K] */
int tmf_linear_dgrad(const float* dy, const float* w, float* dx, int M, int K, int N, int accumulate, void* stream);
/* Scratch buffer of the entry points below that take `ws`: caller-owned, 256-byte aligned, tmf_scratch_bytes() bytes,
 * ZERO-INITIALISED ONCE (its first 16 KB hold "last block" tickets that every kernel leaves zero again); one buffer per
 * stream may be shared by all calls.  It carries split-K / per-block partial sums that the last block to finish adds
 * in index order: the weight gradients of the fusion transformer are bitwise reproducible (no float atomics).  Each kernel
 * family owns its own ticket words (LayerNorm, split-K GEMM tiles, column sums, encoder; csrc/common.cuh): the column sums
 * are capped below the encoder's range, so tmf_linear_wgrad with a bias takes N <= 26496. */
int64_t tmf_scratch_bytes(void);
/* dw[N,K] = dy^T . x ; dbias[N] = column sums of dy (dbias may be NULL); both overwritten */
int tmf_linear_wgrad(const float* dy, const float* x, float* dw, float* dbias, int M, int K, int N, void* ws,
                     size_t ws_bytes, void* stream);

/* y = LayerNorm(x) * gamma + beta (+ residual); saves mean / rstd per row.  reference models/networks.py:117,219 */
int tmf_layernorm_fwd(const float* x, const float* gamma, const float* beta, const float* residual, float* y,
                      float* mean, float* rstd, int rows, int dim, float eps, void* stream);
/* dx (+)= LN backward; dgamma / dbeta are OVERWRITTEN (deterministic two-level sum; `ws` as described above). */
int tmf_layernorm_bwd(const float* dy, const float* x, const float* gamma, const float* mean, const float* rstd,
                      float* dx, float* dgamma, float* dbeta, int rows, int dim, int accumulate, void* ws,
                      size_t ws_bytes, void* stream);

/* dx = dy * gelu'(pre)  (exact erf form, reference models/networks.py:129) */
int tmf_gelu_bwd(const float* dy, const float* pre, float* dx, int64_t n, void* stream);

/* multi-head cross attention on short sequences.  q[B,Nq,h*dh], kv[B,Nk,2*h*dh] (k then v),
 * out[B,Nq,h*dh], lse[B,h,Nq] (log-sum-exp of the scaled scores).  reference models/networks.py:166-174 */
int tmf_attn_fwd(const float* q, const float* kv, float* out, float* lse, int B, int Nq, int Nk, int heads,
                 int dh, float scale, void* stream);
int tmf_attn_bwd(const float* dout, const float* q, const float* kv, const float* out, const float* lse,
                 float* dq, float* dkv, int B, int Nq, int Nk, int heads, int dh, float scale, void* stream);

/* ---- fused Transformer(depth=1) encoder (reference models/networks.py:114-175, 215-230; :272-281 for the caller) -------------
 * One encoder  y = LNf( FF(LN2(a)) + a ) [+ x],  a = Attn(LN1(x), ctx) + x  in 3 forward and 5 backward launches: the
 * projections (proj), the attention core (tmf_attn_fwd / tmf_attn_bwd above) and the row-local chain behind it (chain),
 * plus one launch for all weight gradients (wgrad).  The forward / input-gradient GEMMs run on the tensor cores as a
 * three-MMA bf16 hi/lo split (x*w ~= xh*wh + xl*wh + xh*wl, ~2^-16 relative) from a per-step bf16 hi/lo copy of the five
 * weight matrices: tmf_encoder_pack_weights writes it (tmf_encoder_pack_bytes(mlp) bytes, 16-byte aligned) and the four
 * panel entry points take it as `pack`; pack == NULL selects the three-MMA TF32 split straight from the fp32 weights
 * (~2^-22, slower; the weight gradients always use it).  dim = heads*dim_head = 128, mlp_dim a multiple of 128 (tmf_encoder_supported); x rows Mx = B*Nq, ctx rows
 * Mc = B*Nk; all tensors fp32 row-major; `ws` is the scratch buffer described at tmf_scratch_bytes().
 *   proj_fwd : h1 = LN1(x) (saved with mean1 / rstd1), q = h1 Wq^T [Mx,128], kv = ctx Wkv^T [Mc,256]
 *   chain_fwd: a = o Wo^T + bo + x; h2 = LN2(a); pre = h2 W1^T + b1; f = GELU(pre); g = f W2^T + b2 + a;
 *              y = LNf(g) (+ x if add_input)            (a, h2, pre, f, g and the LayerNorm statistics are saved)
 *   chain_bwd: dy -> dg, dp (= d pre), da, dout (= d o), dxp = da (+ dy if add_input), LayerNorm parameter gradients
 *   proj_bwd : dx = dxp + LN1'(dq Wq), dctx = dkv Wkv, LN1 parameter gradients
 *   wgrad    : t = {dq,h1,dWq, dkv,ctx,dWkv, da,o,dWo,dbo, dp,h2,dW1,db1, dg}; dW2 = dg^T f, db2 (all overwritten) */
int tmf_encoder_supported(int dim, int inner, int mlp);
size_t tmf_encoder_pack_bytes(int mlp);
int tmf_encoder_pack_weights(const float* wq, const float* wkv, const float* wo, const float* w1, const float* w2, int mlp,
                             void* pack, void* stream);
int tmf_encoder_proj_fwd(const float* x, const float* ctx, const float* ln_w, const float* ln_b, const float* wq,
                         const float* wkv, float* h1, float* mean1, float* rstd1, float* q, float* kv, int Mx, int Mc,
                         float eps, const void* pack, void* stream);
int tmf_encoder_chain_fwd(const float* o, const float* x, const float* wo, const float* bo, const float* ln2_w,
                          const float* ln2_b, const float* w1, const float* b1, const float* w2, const float* b2,
                          const float* lnf_w, const float* lnf_b, float* a, float* h2, float* mean2, float* rstd2,
                          float* pre, float* f, float* g, float* meanf, float* rstdf, float* y, int M, int mlp,
                          int add_input, float eps2, float epsf, const void* pack, void* stream);
int tmf_encoder_chain_bwd(const float* dy, const float* g, const float* a, const float* pre, const float* wo,
                          const float* w1, const float* w2, const float* ln2_w, const float* lnf_w, const float* mean2,
                          const float* rstd2, const float* meanf, const float* rstdf, float* dg, float* dp, float* da,
                          float* dout, float* dxp, float* dlnf_w, float* dlnf_b, float* dln2_w, float* dln2_b, int M,
                          int mlp, int add_input, const void* pack, void* ws, size_t ws_bytes, void* stream);
int tmf_encoder_proj_bwd(const float* dq, const float* dkv, const float* dxp, const float* x, const float* ln_w,
                         const float* mean1, const float* rstd1, const float* wq, const float* wkv, float* dx, float* dctx,
                         float* dln_w, float* dln_b, int Mx, int Mc, const void* pack, void* ws, size_t ws_bytes,
                         void* stream);
int tmf_encoder_wgrad(const void* const* t, const float* f, float* dw2, float* db2, int Mx, int Mc, int mlp, void* ws,
                      size_t ws_bytes, void* stream);

/* token pooling over n: mean[B,C], max[B,C] (+ argmax, first maximum) of x[B,N,C]; either output may be NULL.
 * reference models/networks.py:264-269 (GAP / GMP), models/mymodel.py:193 (AdaptiveAvgPool3d(1)) */
int tmf_token_pool_fwd(const float* x, float* mean, float* max, int32_t* argmax, int B, int N, int C, void* stream);
/* dx[B,N,C] (+)= dmean/N + onehot(argmax) * dmax; dmean or dmax may be NULL */
int tmf_token_pool_bwd(const float* dmean, const float* dmax, const int32_t* argmax, float* dx, int B, int N, int C,
                       int accumulate, void* stream);

/* y = alpha * (alpha_dev ? *alpha_dev : 1) * x.  Gradient-reversal backward uses alpha = -1 with the caller's
 * 1-element device tensor lambda (no host sync), or alpha = -lambda.  reference
 * models/gradient_reversal/functional.py:11-16 */
int tmf_scale(const float* x, float* y, float alpha, const float* alpha_dev, int64_t n, void* stream);

/* ---- Grad-CAM on an sNet block (Selvaraju et al. 2017; pytorch-grad-cam conventions) ---------------------------------
 * A, G: fp32 [B,d,h,w,C] per tower (block activation and its gradient, channels-last).  alpha[b,c] = mean_p G[b,p,c] (double,
 * per-chunk partial rows in `ws` added in index order: no atomics, bitwise reproducible, a tower's bits do not depend on ng);
 * cam[b,p] = ReLU(sum_c alpha[b,c] A[b,p,c]).  upsample != 0: trilinear to D x H x W (F.interpolate(mode="trilinear",
 * align_corners=False)); else the map is d x h x w.  normalize != 0: (cam - min) / (max - min + 1e-7) per sample over the
 * returned map (a map that is zero everywhere stays zero).  cam: fp32 [B, D,H,W] (or [B,d,h,w]), overwritten.  C a multiple
 * of 4 in [4,1024], A / G 16-byte aligned; `ws`: caller-owned, 256-byte aligned, at least tmf_gradcam_workspace_bytes(...)
 * bytes (which returns -1 for an unsupported problem). */
int64_t tmf_gradcam_workspace_bytes(int ng, int B, int d, int h, int w, int C, int D, int H, int W, int upsample,
                                    int normalize);
int tmf_gradcam(int ng, const float* const* A, const float* const* G, float* const* cam, int B, int d, int h, int w, int C,
                int D, int H, int W, int upsample, int normalize, void* ws, size_t ws_bytes, void* stream);
/* Grad-CAM's resampling pass on caller maps: lo fp32 [ng][B][d][h][w] (contiguous) -> out[g] fp32 [B][D][H][W], trilinear
 * (align_corners=False; D,H,W = d,h,w copies the map exactly) and, with normalize != 0, (x - min) / (max - min + 1e-7) per
 * sample.  `ws`: at least tmf_map_resample_workspace_bytes(...) bytes (0 without normalize; -1: unsupported problem). */
int64_t tmf_map_resample_workspace_bytes(int ng, int B, int d, int h, int w, int D, int H, int W, int normalize);
int tmf_map_resample(int ng, const float* lo, float* const* out, int B, int d, int h, int w, int D, int H, int W, int normalize,
                     void* ws, size_t ws_bytes, void* stream);

/* ---- layer-wise relevance propagation through the sNet towers (DESIGN section 3.9) --------------------------------------
 * rule TMF_LRP_EPSILON: s = R / stab(y) (y: the stored folded pre-activation, bias included); TMF_LRP_ZPLUS: s = R / stab(z+)
 * with z+ = conv(a, w+) (no bias) and the redistribution through w+ = max(w_folded, 0).  stab(z) = z + eps*sign(z), sign(0) =
 * +1; s = 0 where stab(z) == 0.  Totals: fp32 [B][8] per tower (column `col` written), per-CTA partial rows added in index
 * order (no atomics: bitwise reproducible, a tower's bits do not depend on ng).
 * tmf_lrp_fold_pack: eval BatchNorm folded into the conv weight as tmf_fold_bn_pack does (positive part for zplus): wf
 * [tap][Cout][Cin] and wd [taps-1-tap][Cin][Cout] bf16 packs, w32 fp32 (Cout,Cin,k,k,k) and the folded bias (each of wf / wd
 * / w32 may be NULL).
 * tmf_lrp_ratio: R = up_a * up_c (pooled [B][D/p][H/p][W/p][C]; fp32 with up_fp32, else bf16) routed through the pool
 * (max: to the first maximum of y in (d,h,w) scan order; avg: in proportion to LeakyReLU(y), stabilised window sum; none)
 * and divided by stab(zp ? zp : y) (bf16 [B][D][H][W][C]) -> s bf16 [B][D][H][W][C], zero where no complete window covers
 * a voxel; totals[:, col] = sum of R.  C a multiple of 8; 16-byte aligned tensors; ws of tmf_lrp_ratio_workspace_bytes.
 * tmf_lrp_conv1: block 1.  s from the pooled a1 / c1 (bf16 [B][D/2][H/2][W/2][Cout]), y (and zp) as tmf_lrp_ratio with
 * pool = max, then R_x = x * conv_transpose(s, w) with w the fp32 rule weight (Cout,1,3,3,3) and x fp32 [B][D][H][W]:
 * rx fp32 [B][D][H][W]; totals[:, 6] = sum a1 * c1, totals[:, 7] = sum R_x.  impl as tmf_conv1_dgrad_fused
 * (tmf_lrp_conv1_impl resolves TMF_CONV_AUTO); ws of tmf_lrp_conv1_workspace_bytes.
 * tmf_lrp_normalize: map[g][b] /= max |map[g][b]| (unchanged where that is 0), per of [B][per] fp32. */
#define TMF_LRP_EPSILON 0
#define TMF_LRP_ZPLUS 1
int tmf_lrp_fold_pack(int ng, const float* const* w, const float* const* conv_bias, const float* const* gamma,
                      const float* const* beta, const float* const* running_mean, const float* const* running_var,
                      void* const* wf, void* const* wd, float* const* w32, float* const* bias_out, int cout, int cin,
                      int ksize, float eps, int rule, void* stream);
int64_t tmf_lrp_ratio_workspace_bytes(int ng, int B, int D, int H, int W, int C, int pool);
int tmf_lrp_ratio(int ng, const void* const* up_a, const void* const* up_c, int up_fp32, const void* const* y,
                  const void* const* zp, void* const* s, float* const* totals, int col, int B, int D, int H, int W, int C,
                  int pool, float slope, float eps, void* ws, size_t ws_bytes, void* stream);
int tmf_lrp_conv1_impl(int ng, int impl, int B, int D, int H, int W, int cout);
int64_t tmf_lrp_conv1_workspace_bytes(int ng, int impl, int B, int D, int H, int W, int cout);
int tmf_lrp_conv1(int ng, const void* const* a1, const void* const* c1, const void* const* y, const void* const* zp,
                  const float* const* w, const float* const* x, float* const* rx, float* const* totals, int B, int D, int H,
                  int W, int cout, float eps, int impl, void* ws, size_t ws_bytes, void* stream);
int tmf_lrp_normalize(int ng, float* const* map, int B, int64_t per, void* stream);

/* ---- integrated gradients through the sNet towers, block 1 factored out of the path integral (DESIGN section 3.10) -----
 * Zero baseline, path points alpha_k > 0.  umax: bf16 [B][Do][Ho][Wo][C] per tower, the bias-free folded conv1.0 output u'
 * at the first maximum of each 2x2x2 window (tmf_bn_act_pool_fwd_keepmax's ymax with identity coefficients and slope 1);
 * bias: the folded conv1.0 bias b', fp32 [C]; alpha / w: device fp32 tables of the chunk's n path points and weights; per =
 * Do*Ho*Wo*C elements per sample; z_k = fmaf(alpha_k, umax, b') in both kernels; slope >= 0; C a multiple of 8; 16-byte
 * aligned tensors.  Every element is written once, no atomics (bitwise reproducible; a tower's bits do not depend on ng).
 * tmf_ig_expand: a1[k*B + b] = LeakyReLU(z_k), step-major [n*B][Do][Ho][Wo][C], bf16 (round to nearest) and its fp32 twin
 * a1_32 (the value whose rounding is a1, as the dual-output passes write it).
 * tmf_ig_combine: G[b] += w_k * grad[k*B + b] * LeakyReLU'(z_k) (1 where z_k > 0, else slope), k = 0 .. n-1 in order onto
 * the loaded G, so any split of the path into chunks gives the same bits.  grad: fp32 [n*B][Do][Ho][Wo][C] step-major (the
 * gradients at the block-1 output); G fp32 [B][Do][Ho][Wo][C], updated in place.
 * tmf_ig_attribute: dx[g][b] *= x[g][b] in place (per elements per sample, fp32) and sums[g] fp32 [B][8], column 0 = the
 * per-sample sum of the products (per-CTA partial rows added in index order); ws of tmf_ig_attribute_workspace_bytes. */
int tmf_ig_expand(int ng, const void* const* umax, const float* const* bias, const float* alpha, int n, void* const* a1,
                  float* const* a1_32, int B, int64_t per, int C, float slope, void* stream);
int tmf_ig_combine(int ng, const float* const* grad, const void* const* umax, const float* const* bias, const float* alpha,
                   const float* w, int n, float* const* G, int B, int64_t per, int C, float slope, void* stream);
int64_t tmf_ig_attribute_workspace_bytes(int ng, int B, int64_t per);
int tmf_ig_attribute(int ng, const float* const* x, float* const* dx, float* const* sums, int B, int64_t per, void* ws,
                     size_t ws_bytes, void* stream);

/* ---- occlusion sensitivity through the sNet towers, recomputing only what each window changes (DESIGN section 3.11) ------
 * m windows per pass, window-major rows n*B + b.  tab: device int32 [m][3][4], per window and axis (D, H, W) {crop origin, lo,
 * hi of the changed region, origin of the previous layer's recomputed output}, in the global coordinates of the layer's input
 * (functional.OccPlan); the planner guarantees every index it implies lies inside its tensor.  Every element written once, no
 * atomics, 64-bit offsets.
 * tmf_occ_input: out[g] fp32 [m*B][Dc][Hc][Wc] = x[g][b] (fp32 [B][D][H][W]) at crop origin + (x, y, z), or baseline where that
 * voxel lies in [lo, hi) on all three axes (the window).
 * tmf_occ_compose: out[g] [m*B][Dc][Hc][Wc][C] (bf16, or fp32 with fp32 != 0; C a multiple of 8, 16-byte aligned tensors): at
 * global g = crop origin + (x, y, z), crop[g][n*B + b] at g - (previous output origin) (extent Dp, Hp, Wp) where g lies in
 * [lo, hi) on all three axes, else base[g][b] at g (base [B][D][H][W][C]).  crop[g] == NULL replicates the base.
 * tmf_occ_map: map[g] fp32 [B][D][H][W] = the mean of scores[g][b] (fp32 [B][nD][nH][nW]) over the windows i*s <= x < i*s + w
 * (per axis, w = wD.., s = sD..) that contain the voxel, added in window order; 0 where none does. */
int tmf_occ_input(int ng, const float* const* x, const int* tab, int m, float baseline, float* const* out, int B, int D,
                  int H, int W, int Dc, int Hc, int Wc, void* stream);
int tmf_occ_compose(int ng, const void* const* base, const void* const* crop, const int* tab, int m, void* const* out,
                    int B, int D, int H, int W, int Dc, int Hc, int Wc, int Dp, int Hp, int Wp, int C, int fp32,
                    void* stream);
int tmf_occ_map(int ng, const float* const* scores, float* const* map, int B, int D, int H, int W, int nD, int nH, int nW,
                int wD, int wH, int wW, int sD, int sH, int sW, void* stream);

/* ---- feature ablation over the regions of a mask through the sNet towers (DESIGN section 3.12) -----------------------------
 * The crops and tables of occlusion (tab as for tmf_occ_input, from functional.BoxPlan: one row per box, rows n*B + b); mask:
 * int32 [1|B][D][H][W] (mask_per_sample != 0: one volume per sample).  Every element written once, no atomics, 64-bit offsets.
 * tmf_abl_input: out[g] fp32 [m*B][Dc][Hc][Wc] = x[g][b] at crop origin + (x, y, z), or the baseline where that voxel lies in
 * [lo, hi) on all three axes and its mask id equals ids[n] (device int32 [m]).  The baseline of tower g: bvol[g] (fp32
 * [1|B][D][H][W], one volume per sample where bit g of bvol_per_sample is set), or the scalar bval[g] (host array) where bvol
 * or bvol[g] is NULL.
 * tmf_abl_map: map[g] fp32 [B][D][H][W] = scores[g][b][id] (fp32 [B][F]) for the voxel's mask id, 0 for an id outside
 * [0, F). */
int tmf_abl_input(int ng, const float* const* x, const int* mask, int mask_per_sample, const float* const* bvol,
                  const float* bval, int bvol_per_sample, const int* tab, const int* ids, int m, float* const* out, int B,
                  int D, int H, int W, int Dc, int Hc, int Wc, void* stream);
int tmf_abl_map(int ng, const float* const* scores, const int* mask, int mask_per_sample, int F, float* const* map, int B,
                int D, int H, int W, void* stream);

/* ---- Shapley value sampling over the regions of a mask through the sNet towers (DESIGN section 3.13) -----------------------
 * One pass row n per chain (a permutation's walk from the baseline to x), rows n*B + b; tab as for tmf_abl_input (the
 * BoxPlan rows of the region each row adds); mask and baselines as for tmf_abl_input, with every mask id in [0, F).  Every
 * element written once, no atomics, 64-bit offsets.
 * tmf_shap_input: out[g] fp32 [m*B][Dc][Hc][Wc] = x[g][b] at crop origin + (x, y, z) where rank[perm[n]][id] <= step[n] for
 * the voxel's mask id (rank: device int32 [P][F], perm / step: device int32 [m]), else the baseline.
 * tmf_shap_compose: out[g] as for tmf_occ_compose with crop[g] != NULL, except that the base of row n*B + b is
 * state[g][sidx[n]][b] (state [S][B][D][H][W][C], sidx device int32 [m], distinct, in [0, S)); the same kernel writes out's
 * values inside [lo, hi) back into state[g][sidx[n]][b]. */
int tmf_shap_input(int ng, const float* const* x, const int* mask, int mask_per_sample, const float* const* bvol,
                   const float* bval, int bvol_per_sample, const int* tab, const int* rank, int F, const int* perm,
                   const int* step, int m, float* const* out, int B, int D, int H, int W, int Dc, int Hc, int Wc,
                   void* stream);
int tmf_shap_compose(int ng, void* const* state, const int* sidx, const void* const* crop, const int* tab, int m,
                     void* const* out, int B, int D, int H, int W, int Dc, int Hc, int Wc, int Dp, int Hp, int Wp, int C,
                     int fp32, void* stream);

/* ---- attention maps of the fusion transformer (DESIGN section 3.8) ------------------------------------------------------
 * tmf_attn_scores: per-head product of the attention core's operands (q / kv as for tmf_attn_fwd; dh in {16, 32, 64}, any
 * Nq, Nk), written out as fp32 [B, heads, Nq, Nk]:
 *   mode 0: a = q,  s = dots = scale * q_h k_h^T,  p = attn = exp(dots - lse)   (lse from tmf_attn_fwd, any implementation)
 *   mode 1: a = dout (dL/d out, [B,Nq,h*dh]),  s = dattn = dout_h v_h^T  (dL/d attn of out = attn v; lse and p unused)
 * Three-MMA bf16 hi/lo split with fp32 accumulation, as the tensor-core forward: dots carries the forward's scores bit for
 * bit.  a / kv 16-byte aligned, s / p 8-byte aligned; every element written once (bitwise reproducible).
 * tmf_attn_relevance: M[b,i,j] = mean_h w with w = attn (dattn == NULL) or max(attn * dattn, 0) (Chefer et al. 2021),
 * r[b,j] = mean_i M[b,i,j] (accumulate != 0: added to r).  M [B,Nq,Nk] (may be NULL), r [B,Nk]; fixed summation order. */
int tmf_attn_scores(int mode, const float* a, const float* kv, const float* lse, float* s, float* p, int B, int Nq, int Nk,
                    int heads, int dh, float scale, void* stream);
int tmf_attn_relevance(const float* attn, const float* dattn, float* M, float* r, int B, int heads, int Nq, int Nk,
                       int accumulate, void* stream);

/* ---- inference (SURVEY.md section 8f row 2; reference kfold_train_adversarial.py:144-187) ------------------------------------
 * Eval-mode BatchNorm3d folded into the conv operands: scale = gamma*rsqrt(running_var + eps); wf (bf16
 * [tap][Cout][Cin]; may be NULL) and / or w32 (fp32, reference layout; conv1.0) receive w*scale, bias_out receives
 * (conv_bias - running_mean)*scale + beta.  tmf_conv3d_fwd / tmf_conv1_fwd on these operands write the post-BatchNorm
 * value directly; tmf_bn_act_pool_fwd with identity coefficients finishes the layer (LeakyReLU + pool). */
int tmf_fold_bn_pack(int ng, const float* const* w, const float* const* conv_bias, const float* const* gamma,
                     const float* const* beta, const float* const* running_mean, const float* const* running_var,
                     void* const* wf, float* const* w32, float* const* bias_out, int cout, int cin, int ksize, float eps,
                     void* stream);
/* val_step's metric inputs from logits[B][C]: pred (int64 arg-max, first maximum), prob_last = softmax(logits)[:, C-1]
 * (ROC_AUC input); with labels (int64, may be NULL) and counts4 (4 x uint64, caller-zeroed, may be NULL) the confusion
 * counts {TN, FP, FN, TP} are accumulated (C == 2). */
int tmf_eval_head(const float* logits, const int64_t* labels, int64_t* pred, float* prob_last, void* counts4, int B, int C,
                  void* stream);

/* ---- input pipeline on the device (SURVEY.md section 8f row 4; reference datasets/ADNI.py:59-84) -------------------------------------
 * minmax[2*v] / [2*v+1] = min / max of volume v (ScaleIntensityd, :64). */
int tmf_volume_minmax(const float* x, float* minmax, int nvol, int64_t voxels, void* stream);
/* dst = scale_to_01( resample(src) ): per-volume min-max scaling fused with ONE trilinear, border-clamped affine
 * resampling that composes RandFlipd(axis 0), RandRotated(range_x) and RandZoomd (:66-68).  params[s] = {flip, cos(theta),
 * sin(theta), 1/zoom} per SUBJECT; consecutive groups of `vols_per_subject` volumes (MRI, PET) share a record.  Identity
 * parameters {0,1,0,1} reproduce the test-time transform (scaling only) exactly. */
int tmf_augment_volumes(const float* src, float* dst, const float* minmax, const float* params, int nvol,
                        int vols_per_subject, int D, int H, int W, void* stream);

/* ---- MiSePyNet / Mnet baseline (SURVEY.md section 8f rank 3; reference models/MiSePyNet.py:5-163), fp32 NCDHW-contiguous tensors ------
 * slice convolutions Conv3d(Cin, 8, (1,1,k)) along the last axis (:8,13,16,21,24,27): x [N][Cin][P][L] (P = product of the two
 * leading spatial extents), w [8][Cin][k], y [N][8][P][L-k+1]; Cin <= 8. */
int tmf_line_conv_fwd(const float* x, const float* w, const float* b, float* y, int N, int Cin, int64_t P, int L, int k, void* stream);
int tmf_line_conv_dgrad(const float* dy, const float* w, float* dx, int N, int Cin, int64_t P, int L, int k, void* stream);
/* dw [8][Cin][k], db [8] (may be NULL), both overwritten; ws: caller scratch of tmf_line_conv_wgrad_workspace_bytes (per-block
 * partials, added in block order: deterministic) */
int tmf_line_conv_wgrad(const float* dy, const float* x, float* dw, float* db, int N, int Cin, int64_t P, int L, int k, void* ws,
                        size_t ws_bytes, void* stream);
int64_t tmf_line_conv_wgrad_workspace_bytes(int Cin, int k);
/* spatial convolutions Conv3d(Cin, Cout, (kh,kw,1), stride) on (N,C,X,Y,1) tensors (:44,48,52), no padding:
 * x [N][Cin][X][Y], w [Cout][Cin][kh][kw], y [N][Cout][(X-kh)/s+1][(Y-kw)/s+1] */
int tmf_conv2d_fwd(const float* x, const float* w, const float* b, float* y, int N, int Cin, int X, int Y, int Cout, int kh, int kw,
                   int stride, void* stream);
int tmf_conv2d_dgrad(const float* dy, const float* w, float* dx, int N, int Cin, int X, int Y, int Cout, int kh, int kw, int stride,
                     void* stream);
int tmf_conv2d_wgrad(const float* dy, const float* x, float* dw, float* db, int N, int Cin, int X, int Y, int Cout, int kh, int kw,
                     int stride, void* stream);
/* BatchNorm3d + ReLU on [N][C][S] fp32 (:9-10 ...): statistics / backward sums as partial rows double[TMF_STAT_ROWS][2C] for
 * tmf_bn_finalize / tmf_bn_bwd_finalize (same coef / bcoef conventions as the sNet path; ReLU = LeakyReLU with slope 0) */
int tmf_nchw_bn_stats(const float* x, double* rows, int N, int C, int64_t S, void* stream);
int tmf_nchw_bn_relu_fwd(const float* x, const float* coef, float* out, int N, int C, int64_t S, void* stream);
int tmf_nchw_bn_relu_bwd_reduce(const float* dout, const float* x, const float* coef, double* rows, int N, int C, int64_t S, void* stream);
int tmf_nchw_bn_relu_bwd_apply(const float* dout, const float* x, const float* coef, const float* bcoef, float* dx, int N, int C,
                               int64_t S, void* stream);
/* MaxPool3d((ph,pw,1)), stride = kernel, floor mode (:47,51): x [NC][X][Y] -> y [NC][X/ph][Y/pw], idx uint8 (first maximum) */
int tmf_maxpool2d_fwd(const float* x, float* y, void* idx, int64_t NC, int X, int Y, int ph, int pw, void* stream);
int tmf_maxpool2d_bwd(const float* dy, const void* idx, float* dx, int64_t NC, int X, int Y, int ph, int pw, void* stream);

/* ---- optimizer (SURVEY.md section 8f row 1) -------------------------------------------------------------------------
 * Fused multi-tensor Adam with torch.optim.Adam arithmetic (amsgrad off): replaces the per-parameter launches of the
 * optimizer the reference builds in utils/utils.py:38-41.  `chunks` is a device array of `nchunks` records
 * {float* p; const float* g; float* m; float* v; bf16* wf; bf16* wd; int32 n, off, cout, cin, taps, pad}
 * (tmf_adam_chunk_bytes() = 72 bytes each), one block per record.  wf != NULL marks a chunk (elements off .. off+n) of a
 * Conv3d weight (cout,cin,k,k,k; taps = k^3) whose bf16 operand packs -- what tmf_pack_conv_weights writes -- are refreshed
 * by the optimizer itself: the train step then has no weight-pack launches.  `lr_dev` (1 float) and `step_dev` (1 float, the number of steps taken so far; advanced by the kernel) live
 * on the device so that CUDA-graph replays see their current values; `ticket_dev` is a zero-initialised uint32 scratch. */
int tmf_adam_chunk_bytes(void);
int tmf_adam_step(const void* chunks, int nchunks, const float* lr_dev, float beta1, float beta2, float eps,
                  float weight_decay, float* step_dev, void* ticket_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TMF_H_ */

/* swinb200 -- C ABI of the B200 (sm_100a) kernels behind the SwinV2 weather-model training hot path.
 *
 * Every entry point takes plain device pointers, sizes and a CUDA stream (as void*), allocates
 * nothing, never throws, and returns 0 on success or a SWINB200_ERR_* code (message available from
 * swinb200_last_error()).  There are no torch types in this interface; the Python host code
 * (swin_v2_weather_b200/ops.py) binds it with ctypes and passes tensor.data_ptr().
 *
 * Each function names the reference code it replaces (paths relative to NERSC/swin_v2_weather).
 * "act" buffers hold activations in the compute mode's storage type: SWINB200_BF16 (training mode,
 * tensor-core kernels) or SWINB200_F32 (fp32 validation mode, CUDA-core kernels).
 * Layouts: tokens are row-major (B, H, W, C) == (T, C) with T = B*H*W; images are NCHW fp32.
 */
#ifndef SWINB200_H_
#define SWINB200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SWINB200_VERSION 100

enum { SWINB200_OK = 0, SWINB200_ERR_INVALID_ARG = 1, SWINB200_ERR_CUDA = 2, SWINB200_ERR_UNSUPPORTED = 3 };
enum { SWINB200_F32 = 0, SWINB200_BF16 = 1 };

/* GEMM epilogues (see swinb200_gemm) */
enum {
  SWINB200_EPI_BIAS = 0,      /* D = acc + bias                                 (D: act)             */
  SWINB200_EPI_BIAS_GELU = 1, /* D2 = acc + bias ; D = gelu_erf(D2)             (D, D2: act)         */
  SWINB200_EPI_DGELU = 2,     /* D = acc * gelu_erf'(aux)                       (D, aux: act)        */
  SWINB200_EPI_ADD_F32 = 3,   /* D = acc + aux                                  (D, aux: fp32)       */
  SWINB200_EPI_F32 = 4,       /* D = acc  (or D += acc when accumulate != 0)    (D: fp32)            */
  SWINB200_EPI_BIAS_QKNORM = 5, /* qkv projection: D = acc + bias with N = 3*C packed [q | k | v]; every group of ld_aux
                                   (= head_dim) columns of the q and k thirds is divided by max(||.||_2, 1e-12)
                                   (F.normalize, swinv2_global.py:185,304); D2 (M, 2*N/(3*head_dim)) fp32 receives the
                                   reciprocal norms.  tcgen05 back end, head_dim 96 only.               (D: act)  */
  SWINB200_EPI_BIAS_LN = 6,   /* internal to swinb200_linear_ln_residual: D = acc + bias, then LayerNorm + residual of
                                   every finished 128-row block inside the epilogue                      (D: act)  */
  SWINB200_EPI_BIAS_GELU_FWD = 7, /* D = gelu_erf(act(acc + bias)): the D output of BIAS_GELU, bit for bit, without the
                                     pre-activation D2 (forward-only runs, where no backward reads it; D2 unused) (D: act) */
};
/* GEMM back ends */
enum { SWINB200_GEMM_SIMT = 0, SWINB200_GEMM_TCGEN05 = 1 };

int swinb200_version(void);
const char* swinb200_last_error(void);

/* ---- parameter staging ------------------------------------------------------------------------
 * fp32 master weights -> bf16 shadow used by the tensor-core GEMMs (no reference counterpart: the
 * reference relies on torch autocast's per-call weight casts, train.py:277). */
int swinb200_cast_f32_to_bf16(const float* src, void* dst, size_t n, void* stream);

/* ---- PatchEmbed / head data movement ------------------------------------------------------------
 * swinb200_patchify: img (B, C, Hi, Wi) fp32 -> out (B*(Hi/P)*(Wi/P), C*P*P) act.
 *   order 0: column k = (c*P + p)*P + q -- the Conv2d(k=s=P) im2col of PatchEmbed.proj
 *            (swinv2_global.py:537,544; weight (E, C, P, P) flattened).
 *   order 1: column k = (p*P + q)*C + c -- the inverse of forward_head's unpatchify
 *            (swinv2_global.py:789-791); used on dL/dpred in backward.
 * swinb200_unpatchify: y (T, P*P*Co) act -> out (B, Co, Hi, Wi) fp32,
 *   out = unpatchify(y) + skip[:, :Co] (skip nullable; skip has skip_chans channels).
 *   order 1: columns (p, q, c) -- forward_head's einsum "nhwpqc->nchpwq" (swinv2_global.py:789-791, 795-802);
 *   order 0: columns (c, p, q) -- adjoint of the PatchEmbed im2col (dL/d image for MultiStepWrapper rollouts,
 *            networks/helpers.py:26-41). */
int swinb200_patchify(const float* img, void* out, int act_dtype, int B, int C, int Hi, int Wi, int P,
                      int order, void* stream);
/* swinb200_patchify_cat: order-0 im2col whose image channels come from n_src (<= 8) separate (B or 1, chans[s], Hi, Wi)
 *   fp32 tensors (HOST arrays of DEVICE pointers / channel counts / per-sample strides in elements, 0 = shared by the
 *   batch).  Replaces torch.cat([inp, zenith, static_features], dim=1) of PreProcessor.forward
 *   (utils/preprocess_utils.py:50-68) and of the MultiStepWrapper rollout (networks/helpers.py:36-40) followed by
 *   PatchEmbed's im2col: the concatenated image is never materialised. */
int swinb200_patchify_cat(int n_src, const float* const* srcs, const int* chans, const long long* batch_strides,
                          void* out, int act_dtype, int B, int Hi, int Wi, int P, void* stream);
int swinb200_unpatchify(const void* y, int act_dtype, const float* skip, int skip_chans, float* out,
                        int B, int Co, int Hi, int Wi, int P, int order, void* stream);
/* Input z-score folded into the same passes (SURVEY 8(f) rank 3): `mean` / `std` are (C,) fp32 device arrays over the
 *   concatenated channels; every image value becomes (x - mean[c]) / std[c] on its way into the im2col -- the per-channel
 *   normalisation the loaders apply on the GPU before the model sees a field (utils/data_loader_era5_dali.py:77-90,
 *   utils/data_loader_era5.py:98-107).  Channels that must pass through unchanged carry mean 0 / std 1 ((x-0)/1 == x).
 *   swinb200_unpatchify_norm applies the same to the residual skip (swinv2_global.py:795-802) when it is the raw field.
 *   NULL statistics = the plain entry points above. */
int swinb200_patchify_cat_norm(int n_src, const float* const* srcs, const int* chans, const long long* batch_strides,
                               const float* mean, const float* std, void* out, int act_dtype, int B, int Hi, int Wi,
                               int P, void* stream);
int swinb200_unpatchify_norm(const void* y, int act_dtype, const float* skip, int skip_chans, const float* skip_mean,
                             const float* skip_std, float* out, int B, int Co, int Hi, int Wi, int P, int order,
                             void* stream);

/* ---- GEMM ---------------------------------------------------------------------------------------
 * D[M,N] = epilogue( sum_k A(m,k) * B(n,k) ).
 *   a_major 0: A stored (M, K) row-major, lda = row pitch;  1: A stored (K, M) row-major.
 *   b_major 0: B stored (N, K) row-major (nn.Linear weight);  1: B stored (K, N) row-major.
 * Replaces nn.Linear forward (a0,b0), its input gradient (a0,b1 with B = weight) and its weight
 * gradient (a1,b1) -- swinv2_global.py:181,199,300,319,381-386,544,787 and their autograd
 * backward.  in_dtype is the storage type of A and B.  split_k > 1 is allowed only with
 * SWINB200_EPI_F32 and accumulate (atomic fp32 adds into a pre-initialised D).  BIAS_GELU_FWD, like BIAS_GELU, is a
 * forward epilogue (a_major 0, b_major 0 on the tcgen05 back end).
 * backend SWINB200_GEMM_TCGEN05 requires in_dtype == SWINB200_BF16. */
int swinb200_gemm(int backend, int M, int N, int K, const void* A, int a_major, int lda, const void* B,
                  int b_major, int ldb, int in_dtype, int epilogue, const float* bias, void* D, int ldd,
                  void* D2, const void* aux, int ld_aux, int out_dtype, int accumulate, int split_k,
                  void* stream);

/* ---- weight + bias gradient of nn.Linear in one kernel ----------------------------------------------------
 * dW[n_out, n_in] += dY^T X  (split-K, fp32 TMA reduce-add into a pre-initialised dW) ;  dbias[n_out] += column sums of dY
 *   == autograd of `self.qkv` / `self.mlp.fc1` w.r.t. weight and bias (swinv2_global.py:181/300, timm Mlp.fc1): the bias
 *   gradient is the sum over tokens of the dY tiles the weight-gradient GEMM stages in shared memory anyway, taken there
 *   by the epilogue warps while the main loop runs -- dY is not read again by a column-sum pass.  dY (T, n_out) and
 *   X (T, n_in) bf16 token-major; dbias may be NULL.  tcgen05 back end, n_out a multiple of 256, n_in >= 256; otherwise
 *   SWINB200_ERR_UNSUPPORTED (the caller runs swinb200_gemm + swinb200_colsum). */
int swinb200_linear_wgrad(int backend, int n_out, int n_in, int T, const void* dY, int ldy, const void* X, int ldx,
                          float* dW, int lddw, float* dbias, int split_k, void* stream);

/* ---- Linear + LayerNorm + DropPath + residual in one kernel -----------------------------------------
 * z = A W^T + bias (stored, bf16: the backward needs it) ; u = LN_N(z) * gamma + beta (* sample_scale[row /
 * rows_per_sample] if given) ; x_out = x_in + u ; xb_out = bf16(x_out) ; stats[row] = (mean, rstd)
 *   == `x = x + self.drop_path(self.norm1(self.attn.proj(...)))` and `x = x + self.drop_path(self.norm2(self.mlp.fc2(...)))`
 *   (swinv2_global.py:199/319 + 490, timm Mlp.fc2 + 494): the LayerNorm + residual run inside the GEMM epilogue -- the
 *   CTA that completes the last column tile of a 128-row block normalises that block while the tensor cores work on the
 *   next tiles.  tcgen05 back end, bf16 operands, N = 768 (three 256-column tiles per row); other shapes / back ends
 *   return SWINB200_ERR_UNSUPPORTED and the caller runs swinb200_gemm(EPI_BIAS) + swinb200_ln_residual_fwd.
 *   counters: n_counters >= ceil(M / 128) ints, zero on entry; the kernel leaves them zero. */
int swinb200_linear_ln_residual(int backend, int M, int N, int K, const void* A, int lda, const void* W, int ldw,
                                const float* bias, void* z, int ldz, const float* x_in, const float* gamma,
                                const float* beta, const float* sample_scale, float* x_out, void* xb_out, float* stats,
                                int rows_per_sample, float eps, int* counters, int n_counters, void* stream);

/* ---- LayerNorm + residual (post-norm) -------------------------------------------------------------
 * fwd:  u = LN_C(z) * gamma + beta  (+ pos[t % rows_per_sample, c] if pos)  (* sample_scale[b] if given)
 *       x_out = (x_in ? x_in : 0) + u ;  xb_out = act(x_out) ;  stats[row] = (mean, rstd)
 *   == `x + drop_path(norm(branch))` (swinv2_global.py:490,494), and PatchEmbed.norm + pos_embed add
 *   (swinv2_global.py:545,780) with x_in = NULL, pos = pos_embed transposed to token-major
 *   (rows_per_sample, C) fp32 by swinb200_transpose_f32.  stats may be NULL (forward-only runs): the statistics are
 *   then not stored and everything else is unchanged.
 * bwd:  given dx = dL/dx_out (fp32): dz (act) ; dgamma, dbeta, dbias_prev += column sums (fp32 atomics,
 *       caller zero-initialises).  dL/dx_in is dx itself (identity path), handled by the caller. */
int swinb200_ln_residual_fwd(const void* z, int act_dtype, const float* x_in, const float* gamma,
                             const float* beta, const float* sample_scale, const float* pos, float* x_out,
                             void* xb_out, float* stats, int rows, int C, int rows_per_sample, float eps,
                             void* stream);
int swinb200_ln_residual_bwd(const float* dx, const void* z, int act_dtype, const float* stats,
                             const float* gamma, const float* sample_scale, void* dz, float* dgamma,
                             float* dbeta, float* dbias_prev, int rows, int C, int rows_per_sample,
                             void* stream);
/* dpos[c, t] = sum_b dx[b, t, c]  (gradient of the NCHW pos_embed parameter, swinv2_global.py:770,780) */
int swinb200_pos_embed_grad(const float* dx, float* dpos, int B, int rows_per_sample, int C, void* stream);
/* dst (Cc, R) = src (R, Cc)^T, fp32 (pos_embed NCHW <-> token-major staging) */
int swinb200_transpose_f32(const float* src, float* dst, int R, int Cc, void* stream);

/* out[col] += sum_rows x[row, col]  (bias gradients of nn.Linear) */
int swinb200_colsum(const void* x, int act_dtype, float* out, int rows, int cols, int ld, void* stream);

/* ---- windowed cosine attention ----------------------------------------------------------------------
 * qk_normalize: in place on qkv (T, 3C): q and k of every (token, head) are divided by
 *   max(||.||_2, 1e-12) (F.normalize, swinv2_global.py:185,304); inv_norm (T, 2, heads) fp32 receives
 *   the reciprocal factors for backward (nullable: not stored).  The same holds for D2 of SWINB200_EPI_BIAS_QKNORM.
 * window_attn_fwd: per (sample, window, head), with roll(-s)/window_partition/window_reverse/roll(+s)
 *   (swinv2_global.py:89-119,446-478) folded into addressing:
 *     S = scale[h] * qhat khat^T (+ bias[h]) (+ shift mask) ; P = softmax(S) ; O = P v
 *   (swinv2_global.py:185-198 / 304-318).  scale = exp(min(logit_scale, ln 100)) is passed in.
 *   bias: nullable (heads, L, L) fp32 (continuous position bias table, :274-287).  The shift mask
 *   ({0,-100}, :403-424) is generated in-kernel from (H, Wh, s0); swinb200_shift_mask materialises the
 *   same predicate as the reference's (nW, L, L) buffer for bit-exact checks.
 *   o: (T, C) act in un-rolled token order; lse: (2, B, nW, heads, L) fp32 -- plane 0 = log-sum-exp of every softmax row,
 *   plane 1 = the row's softmax-weighted mean cosine sum_j P_ij cos_ij (zero from back ends whose backward does not use it;
 *   the tcgen05 backward accumulates d(scale) against it so that the sum is insensitive to the rounding of O).  lse may
 *   be NULL when no backward follows: neither plane is written, o is unchanged.
 * window_attn_bwd: dqkv (T, 3C) act = gradients w.r.t. the *un-normalised* q, k and v;
 *   dscale (heads) += sum dS * cos ; dbias (heads, L, L) += sum_windows dS (nullable).
 *   ws: required by the tcgen05 back end; T*heads floats (the library allocates nothing), which receive the row term
 *   D = <dO, O> from a streaming pre-pass.  Unused by the CUDA-core back end (nullable there).
 * backend: SWINB200_GEMM_SIMT (CUDA cores, any act dtype) or SWINB200_GEMM_TCGEN05 (bf16).  The tcgen05 back end needs
 *   qkv and o (forward), and qkv, o, d_o and dqkv (backward), 16-byte aligned: SWINB200_ERR_INVALID_ARG otherwise. */
int swinb200_qk_normalize(void* qkv, int act_dtype, float* inv_norm, int T, int C, int heads, void* stream);
int swinb200_shift_mask(float* mask, int H, int W, int Wh, int Ww, int s0, int s1, void* stream);
int swinb200_window_attn_fwd(int backend, const void* qkv, int act_dtype, const float* scale,
                             const float* bias, void* o, float* lse, int B, int H, int W, int C, int heads,
                             int Wh, int Ww, int s0, int s1, void* stream);
int swinb200_window_attn_bwd(int backend, const void* qkv, int act_dtype, const float* inv_norm,
                             const float* scale, const float* bias, const void* o, const void* d_o,
                             const float* lse, void* dqkv, float* dscale, float* dbias, float* ws, int B, int H,
                             int W, int C, int heads, int Wh, int Ww, int s0, int s1, void* stream);

/* ---- latitude-weighted L2 loss ------------------------------------------------------------------------
 * fwd: num[b,c] = sum_hw qw[h] (p-t)^2 ; den[b,c] = sum_hw qw[h] t^2 ;
 *      r = relative ? num/den : num ;  loss = sum_bc chw[c] * (squared ? r : sqrt(r))
 *   == LossHandler -> GeometricLpLoss.rel/abs with p=2 (utils/losses.py:188-232,
 *   utils/grids.py:115-117).  num/den/loss are fp32 outputs (B*C, B*C, 1); the entry point zeroes them.
 * bwd: dprd = gloss * chw[c] * (squared ? 1 : 1/(2 sqrt(r))) * 2 qw[h] (p - t) / (relative ? den[b,c] : 1). */
int swinb200_latw_l2_fwd(const float* prd, const float* tar, const float* qw, const float* chw, int relative,
                         int squared, float* num, float* den, float* loss, int B, int C, int H, int W,
                         void* stream);
int swinb200_latw_l2_bwd(const float* prd, const float* tar, const float* qw, const float* chw,
                         const float* num, const float* den, const float* gloss, int relative, int squared,
                         float* dprd, int B, int C, int H, int W, void* stream);

/* ---- L1 loss family and validation anomaly correlation (SURVEY 8(f) rank 4) ---------------------------
 * latw_l1_fwd: sums[b,c] = {sum_hw qw[h] |p-t|, sum_hw qw[h] |t|};  loss = sum_bc chw[c] * (relative ? s0/s1 : s0)
 *   == LossHandler 'l1' / 'geometric l1' -> GeometricLpLoss(p=1).abs/.rel (utils/losses.py:116-124, 188-232).
 * latw_l1_bwd: dprd = gloss * chw[c] * qw[h] * sign(p-t) / (relative ? s1 : 1).
 * Pole-masked variants of every loss ('pole-masked', utils/losses.py:49-52, utils/grids.py:96-99) are the same kernels
 *   with the first / last rows of qw set to zero by the caller.
 * latw_acc: sums[b,c] = {sum qw p t, sum qw p p, sum qw t t};  acc[b,c] = s0 / sqrt(s1 * s2)
 *   == weighted_acc_torch_channels (utils/weighted_acc_rmse.py:89-99).  sums (B*C*3) and acc (B*C) are fp32 outputs. */
int swinb200_latw_l1_fwd(const float* prd, const float* tar, const float* qw, const float* chw, int relative,
                         float* sums, float* loss, int B, int C, int H, int W, void* stream);
int swinb200_latw_l1_bwd(const float* prd, const float* tar, const float* qw, const float* chw, const float* sums,
                         const float* gloss, int relative, float* dprd, int B, int C, int H, int W, void* stream);
int swinb200_latw_acc(const float* prd, const float* tar, const float* qw, float* sums, float* acc, int B, int C,
                      int H, int W, void* stream);

/* ---- optimizer (SURVEY 8(f) rank 1) ------------------------------------------------------------------
 * One fused multi-tensor pass of torch.optim.Adam(lr, betas, eps, weight_decay, amsgrad=False) as the reference
 * configures it (train.py:175-176), over n_tensors fp32 parameters given as HOST arrays of DEVICE pointers:
 *   g = grad / *grad_scale (+ weight_decay * p);  m += (1-beta1)(g-m);  v = beta2 v + (1-beta2) g^2;
 *   p -= lr/(1-beta1^step) * m / (sqrt(v)/sqrt(1-beta2^step) + eps)
 * and, where shadows[i] != NULL, the bf16 copy of the new p that the tensor-core GEMMs read (replaces the per-step
 * swinb200_cast_f32_to_bf16 pass).  grad_scale / found_inf: optional device scalars with torch.amp.GradScaler's meaning
 * (train.py:281-289); a non-zero *found_inf skips the whole step on the device.  step counts from 1. */
int swinb200_adam_step(int n_tensors, void* const* params, const void* const* grads, void* const* exp_avg,
                       void* const* exp_avg_sq, void* const* shadows, const long long* numel, double lr,
                       double beta1, double beta2, double eps, double weight_decay, long long step,
                       const float* grad_scale, const float* found_inf, void* stream);

/* ---- deterministic mode ---------------------------------------------------------------------------------
 * Bitwise-reproducible versions of every entry point above whose float sums would otherwise depend on the order in which
 * CTAs or warps finish (atomics).  Each writes its partial sums with plain stores into caller-owned scratch `part`
 * (part_floats floats, fp32, 16-byte aligned), one slot per split / statically assigned CTA / row block / (sample,
 * window, head) item, and then adds the slots in slot order with swinb200_ordered_reduce.  Outputs are defined exactly as
 * by the plain entry points (accumulating outputs are still added to, once).  Same build, same GPU model, same inputs ->
 * the same bits.  NULL or short scratch: SWINB200_ERR_INVALID_ARG.  The library still allocates nothing.
 *
 * swinb200_ordered_reduce: out[i] = (accumulate ? out[i] : 0) + sum_{p < n_part} sum_{j < inner} part[p*stride + i*inner + j],
 *   i < n, summed in exactly that order (the fixed-order second stage of every entry below; stride >= n * inner).
 * swinb200_gemm_wgrad_det: D[M,N] += sum_k A(k,m) B(k,n), A stored (K, M), B stored (K, N), D dense (ldd = N) fp32 -- the
 *   split-K weight gradient of swinb200_gemm(a_major 1, b_major 1, EPI_F32, accumulate).  tcgen05: every split TMA-stores
 *   its tile into its own slice of a [S, M, N] scratch; scratch >= split_k*M*N floats.  SIMT: the CUDA-core GEMM does not
 *   split K (one thread adds each element once), scratch unused and may be NULL.
 * swinb200_linear_wgrad_det: swinb200_linear_wgrad with dW dense (lddw = n_in); scratch >= split_k*(n_out*n_in + n_out).
 * swinb200_ln_residual_bwd_det: swinb200_ln_residual_bwd; scratch >= 3*C*256*max(1, 2048/C) floats (integer division):
 *   at most 256 CTAs, each leaving one [3, C] row per group of threads that covers all channels.
 * swinb200_colsum_det: swinb200_colsum; scratch >= cols*min(ceil(rows/64), 256).
 * swinb200_latw_l2_fwd_det / _l1_fwd_det / _acc_det: the loss / metric entry points; scratch >= 2*B*C*H (L2, L1) and
 *   3*B*C*H (ACC) floats (at most one row block per image row).
 * swinb200_window_attn_bwd_det: swinb200_window_attn_bwd; with nW = (H/Wh)*(W/Ww), L = Wh*Ww and items = B*nW*heads,
 *   scratch >= items*(4*ceil(L/128) + (dbias ? L*L : 0)) floats: d(scale) slots per item, then one (L, L) d(bias) slice
 *   per item (336 MB at 9x18 windows / 8 heads / B = 1 on the 180x360 token grid with a bias table). */
int swinb200_ordered_reduce(const float* part, int n_part, long long stride, long long n, int inner, float* out, int accumulate,
                            void* stream);
int swinb200_gemm_wgrad_det(int backend, int M, int N, int K, const void* A, int lda, const void* B, int ldb, int in_dtype,
                            float* D, int split_k, float* part, long long part_floats, void* stream);
int swinb200_linear_wgrad_det(int backend, int n_out, int n_in, int T, const void* dY, int ldy, const void* X, int ldx,
                              float* dW, float* dbias, int split_k, float* part, long long part_floats, void* stream);
int swinb200_ln_residual_bwd_det(const float* dx, const void* z, int act_dtype, const float* stats, const float* gamma,
                                 const float* sample_scale, void* dz, float* dgamma, float* dbeta, float* dbias_prev, int rows,
                                 int C, int rows_per_sample, float* part, long long part_floats, void* stream);
int swinb200_colsum_det(const void* x, int act_dtype, float* out, int rows, int cols, int ld, float* part, long long part_floats,
                        void* stream);
int swinb200_latw_l2_fwd_det(const float* prd, const float* tar, const float* qw, const float* chw, int relative, int squared,
                             float* num, float* den, float* loss, int B, int C, int H, int W, float* part, long long part_floats,
                             void* stream);
int swinb200_latw_l1_fwd_det(const float* prd, const float* tar, const float* qw, const float* chw, int relative, float* sums,
                             float* loss, int B, int C, int H, int W, float* part, long long part_floats, void* stream);
int swinb200_latw_acc_det(const float* prd, const float* tar, const float* qw, float* sums, float* acc, int B, int C, int H,
                          int W, float* part, long long part_floats, void* stream);
int swinb200_window_attn_bwd_det(int backend, const void* qkv, int act_dtype, const float* inv_norm, const float* scale,
                                 const float* bias, const void* o, const void* d_o, const float* lse, void* dqkv, float* dscale,
                                 float* dbias, float* ws, int B, int H, int W, int C, int heads, int Wh, int Ww, int s0, int s1,
                                 float* part, long long part_floats, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SWINB200_H_ */

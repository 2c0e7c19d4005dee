/*
 * lc2is_b200.h - C ABI of the B200-native LC2IS segmentation-head hot path.
 *
 * The reference (AntoineBlanot/LC2IS) is pure Python: it has no FFI / plugin registry.
 * Each entry point below replaces a group of reference *lines* (cited per function, paths
 * relative to the reference root) and is what a ctypes binding on the reference side calls
 * (see INTEGRATION.md).  Conventions, all entry points:
 *
 *   - return 0 on success, non-zero on error (negative = argument error, positive =
 *     cudaError_t); no exception crosses the boundary; lc2is_last_error() returns text
 *     (thread-local).
 *   - every pointer named d_* is a DEVICE pointer owned by the caller; the library never
 *     allocates or frees device memory and never synchronises the host (except the
 *     *_host entry points, documented there).  Work is enqueued on `stream` only, so every
 *     call is CUDA-graph capturable.
 *   - accumulated outputs (confmat, per_image, loss_sum, n_valid, grad_t) are ADDED to:
 *     the caller zeroes them (lets several batches / ranks accumulate into one buffer).
 *   - tensors are dense row-major with the shapes given; int64 = long long.
 *   - there is no CPU fallback: without a CUDA device every compute call fails.
 */
#ifndef LC2IS_B200_H
#define LC2IS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* lc2is_stream_t;                 /* cudaStream_t */

enum { LC2IS_F32 = 0, LC2IS_BF16 = 1 };        /* dtype codes            */
enum { LC2IS_BILINEAR = 0, LC2IS_BICUBIC = 1 }; /* upsample modes         */

#define LC2IS_ERR_ARG      (-1)
#define LC2IS_ERR_SHAPE    (-2)
#define LC2IS_ERR_NODEVICE (-3)
#define LC2IS_ERR_UNSUPPORTED (-4)

const char* lc2is_last_error(void);
int         lc2is_abi_version(void);
/* number of kernels this library has launched in this process (bench `gpu_launches`) */
int64_t     lc2is_launch_count(void);

/* Round C up to the class padding the tensor-core kernels use (multiple of 16). */
int lc2is_class_pad(int C);

/* ---------------------------------------------------------------------------------------
 * K0  proto_normalize.   Replaces  t = F.normalize(t, dim=2, p=2)   model/final.py:42
 *     (and :80,:142,:204,:267,:279,:342,:354; model/new.py:67; model/ftn.py:58).
 * d_t      [n_sets, C, D] fp32 text embeddings (n_sets = 1 shared, or B per-image prompts,
 *          final.py:129-130).
 * d_t_hat  [n_sets, C_pad, D] bf16 out: t / max(||t||, 1e-12) (or t itself if !normalize),
 *          rows C..C_pad-1 zero.  C_pad = lc2is_class_pad(C).
 * d_inv_norm [n_sets, C] fp32 out: 1 / max(||t||, 1e-12) (1.0 if !normalize).
 */
int lc2is_proto_normalize(const float* d_t, int n_sets, int C, int D, int normalize,
                          void* d_t_hat, float* d_inv_norm, lc2is_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * K1  cosine_logits_fwd.  Replaces
 *       v = F.normalize(v, dim=1, p=2); score = einsum('bchw,bkc->bkhw', v, t)
 *       model/final.py:41,43  (normalize=1)      and
 *       matmul(feature_v, feature_t.T) + rearrange       model/model.py:50,53 (normalize=0)
 * d_v        [B, hw, D] patch embeddings, v_dtype LC2IS_F32 or LC2IS_BF16.  D % 64 == 0.
 * d_t_hat    [n_sets, C_pad, D] bf16 from K0.
 * d_v_hat    [B*hw, D] bf16 out/workspace: normalised (or plain) patch rows as fed to the
 *            tensor cores; kept for the backward.
 *            NULL (bf16 V, normalize = 1 only): the row normalisation runs INSIDE the GEMM - four extra warps sum the
 *            squares of each row from the staged operand tiles while the MMAs run, the epilogue scales the row by
 *            1/max(||v||,1e-12) - and no v_hat exists (the operand of the tensor cores is the raw V, the fp32 row factor
 *            is applied to the fp32 accumulator: closer to the fp32 reference than rounding v_hat to bf16).  The backward
 *            then takes V itself: lc2is_cosine_logits_bwd_ex(..., LC2IS_BWD_RAW_V).
 * d_inv_norm_v [B*hw] fp32 out: 1/max(||v||,1e-12) (1.0 if !normalize).
 * d_logits   [B, C, hw] fp32 out (class-plane major = the reference's 'b k h w'):
 *            logit_scale * <v_hat, t_hat>.  bf16 operands, fp32 accumulate (tcgen05/TMEM).
 */
int lc2is_cosine_logits_fwd(const void* d_v, int v_dtype, int B, int hw, int D,
                            const void* d_t_hat, int n_sets, int C,
                            int normalize, float logit_scale,
                            void* d_v_hat, float* d_inv_norm_v, float* d_logits,
                            lc2is_stream_t stream);

/* TextToPatch.visual / .textual forward (model/text_patch.py:11-12,16-17): y[M,N] = x[M,K] W[N,K]^T + b[N] on the
 * logits GEMM's tcgen05 / TMEM / TMA pipeline.  x, W bf16 (W in nn.Linear's own [out,in] layout), b fp32 or NULL,
 * y bf16 or fp32 row major.  K % 64 == 0, N % 16 == 0.  d_x, d_w, d_y and d_bias 16-byte aligned (LC2IS_ERR_ARG
 * otherwise).  Shapes with M % 256 == 0, N % 256 == 0 and at least two 256 x 256 tiles per CTA pair (2 * (SMs / 2)
 * tiles) run the 2-SM (cta_group::2) form of the kernel, everything else the 1-SM form. */
int lc2is_linear_fwd(const void* d_x_bf16, const void* d_w_bf16, const float* d_bias,
                     long long M, int N, int K, void* d_y, int y_dtype, lc2is_stream_t stream);

/* Producer of the projection: bicubic x4 upsample of the decoder's TOKEN-major feature map, written directly as the
 * row-major operand of TextToPatch.visual.  Replaces model/model.py:42-44 (rearrange to [B,C,h,w], F.interpolate(bicubic,
 * scale_factor=4), rearrange back - an fp32 [B,C,4h,4w] intermediate and two layout passes) and their autograd backward.
 * d_x [B, h*w, C] fp32 / bf16 -> d_y [B, 16*h*w, C] fp32 / bf16 (ATen's taps: A = -0.75, src = 0.25*(dst+0.5)-0.5, clamped
 * indices, horizontal then vertical chains).  C % 4 == 0, 16-byte aligned pointers.
 * backward: d_gx [B, h*w, C] = the transpose applied to d_gy [B, 16*h*w, C]; two gather passes (no atomics) through an fp32
 * workspace of lc2is_bicubic4_tokens_bwd_workspace bytes. */
int lc2is_bicubic4_tokens_fwd(const void* d_x, int x_dtype, int B, int h, int w, int C, void* d_y, int y_dtype,
                              lc2is_stream_t stream);
int64_t lc2is_bicubic4_tokens_bwd_workspace(int B, int h, int w, int C);
int lc2is_bicubic4_tokens_bwd(const void* d_gy, int gy_dtype, int B, int h, int w, int C, void* d_gx, int gx_dtype,
                              void* d_ws, lc2is_stream_t stream);

/* Backward of the same projection (autograd of model/text_patch.py:12,17; y = x W^T + b), all on tcgen05:
 *   d_gx [M,K] (gx_dtype) = gy . W      lc2is_linear_fwd's pipeline on the transposed weight (built in d_ws)
 *   d_gw [N,K] fp32      += gy^T . x    split-K over the rows, both operands MN-major: each slice stores its fp32 partial
 *                                       sum in d_ws, one pass adds the slices to d_gw (ACCUMULATES: zero it, or let
 *                                       several micro-batches add up like autograd does)
 *   d_gb [N]   fp32      += column sums of gy
 * gy [M,N], x [M,K], W [N,K] bf16; N and K multiples of 64.  Any of d_gx / d_gw / d_gb may be NULL.
 * d_gy, d_x, d_gx, d_gw and d_ws 16-byte aligned (LC2IS_ERR_ARG otherwise).  Pointers, shapes and gx_dtype are checked
 * before the first launch: a call rejected for them has written no output.
 * d_ws: lc2is_linear_bwd_workspace(N, K) bytes (the transposed weight for d_gx, the split-K partial sums for d_gw). */
int64_t lc2is_linear_bwd_workspace(int N, int K);
int lc2is_linear_bwd(const void* d_gy_bf16, const void* d_x_bf16, const void* d_w_bf16, long long M, int N, int K,
                     void* d_gx, int gx_dtype, float* d_gw, float* d_gb, void* d_ws, lc2is_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * K1b cosine_logits_bwd.  Replaces autograd of the K1 lines (loss.backward(), engine.py:100).
 * d_grad_logits: dL/dlogits, g_dtype LC2IS_BF16: [B, C_pad, hw] bf16 (rows C..C_pad-1 zero; K2's
 *            bf16 output or lc2is_grad_to_bf16), or LC2IS_F32: [B, C, hw] fp32 (K2's fp32 gradient;
 *            converted to the bf16 GEMM operand in the same pass that forms the projections).
 * d_logits   [B, C, hw] fp32 from K1 (used for the normalise-backward projection
 *            v_hat . dV_hat = sum_c G_c * logits_c).
 * d_grad_scale: optional DEVICE fp32 scalar multiplied into every gradient (the upstream
 *            grad_output, e.g. 0.4 for the aux loss, engine.py:98); NULL = 1.
 * d_grad_v   [B*hw, D] out, gv_dtype LC2IS_F32 or LC2IS_BF16 (overwritten).
 * d_grad_t   [n_sets, C, D] fp32, ACCUMULATED (zero it first): gradient w.r.t. the raw
 *            (un-normalised) text embeddings.
 * d_ws       workspace, lc2is_cosine_logits_bwd_workspace(...) bytes.
 */
int64_t lc2is_cosine_logits_bwd_workspace(int B, int hw, int D, int n_sets, int C);
int lc2is_cosine_logits_bwd(const void* d_grad_logits, int g_dtype, const float* d_logits,
                            const void* d_v_hat, const float* d_inv_norm_v,
                            const void* d_t_hat, const float* d_inv_norm_t,
                            int B, int hw, int D, int n_sets, int C,
                            int normalize, float logit_scale, const float* d_grad_scale,
                            void* d_grad_v, int gv_dtype, float* d_grad_t,
                            void* d_ws, lc2is_stream_t stream);
/* Same with flags.  LC2IS_BWD_REUSE_PREP: the workspace already holds the projections and the bf16 operand of an
 * earlier call on the same inputs - for running the backward as two calls, d_grad_t first (d_grad_v = NULL) and
 * d_grad_v second (d_grad_t = NULL, this flag), so that a data-parallel caller can all-reduce the prototype gradient
 * while the patch-gradient GEMM runs. */
#define LC2IS_BWD_REUSE_PREP 1
/* LC2IS_BWD_RAW_V: `d_v_hat` is the RAW bf16 V (what lc2is_cosine_logits_fwd took when it was called with
 * d_v_hat = NULL and normalised inside the GEMM) - v_hat = V * inv_norm_v is never materialised: the bf16 operand of the
 * two GEMMs is G * inv_norm_v and the normalise-backward of the patches is folded into the dV epilogue.  Needs
 * normalize = 1 and an fp32 gradient. */
#define LC2IS_BWD_RAW_V 2
/* LC2IS_BWD_WS_ZEROED: the caller has zeroed the first lc2is_cosine_logits_bwd_workspace_zeroed(...) bytes of d_ws
 * (the accumulators of the projections and of the prototype GEMM) since the workspace was last used, e.g. in the
 * zero-fill that starts its step.  The call then enqueues kernels only, which lets each one start its prologue while
 * the previous kernel of the stream finishes (programmatic dependent launch); without the flag it zeroes them itself. */
#define LC2IS_BWD_WS_ZEROED 4
int64_t lc2is_cosine_logits_bwd_workspace_zeroed(int B, int hw, int D, int n_sets, int C);
int lc2is_cosine_logits_bwd_ex(const void* d_grad_logits, int g_dtype, const float* d_logits,
                               const void* d_v_hat, const float* d_inv_norm_v,
                               const void* d_t_hat, const float* d_inv_norm_t,
                               int B, int hw, int D, int n_sets, int C,
                               int normalize, float logit_scale, const float* d_grad_scale,
                               void* d_grad_v, int gv_dtype, float* d_grad_t,
                               void* d_ws, lc2is_stream_t stream, int flags);

/* fp32 [B,C,hw] -> bf16 [B,C_pad,hw] (zero pad rows); for callers whose dL/dlogits did not
 * come from K2. */
int lc2is_grad_to_bf16(const float* d_grad, int B, int C, int hw, void* d_grad_bf16,
                       lc2is_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * K2  upsample + softmax cross-entropy, forward and backward in one pass.  Replaces
 *       input = F.interpolate(input, mode="bilinear", size=H); CrossEntropyLoss(input,target)
 *       model/loss.py:19-20 (AuxiliaryLoss)  and  final.py:44 + engine.py:94 (criterion),
 *       plus their autograd backward (engine.py:100).
 * lc2is_count_valid: n_valid += #{labels in [0,C) and != ignore_index} (the 'mean' denominator; ids outside [0,C) are
 *            skipped by every CE kernel - torch would device-assert on them - so they are not counted either).
 * d_low      [B, C, h, w] fp32 low-resolution logits.
 * d_labels   [B, H, W] int64, values in [0,C) or ignore_index.
 * d_grad_scale DEVICE fp32 scalar g: gradients are g * (softmax - onehot) scattered through
 *            the bilinear taps (pass 1/n_valid for reduction='mean'); NULL = 1.
 * d_loss_sum DEVICE double, ACCUMULATED: sum over valid pixels of -log softmax[target].
 * d_grad_low [B, C, h, w] fp32 out (overwritten) or NULL.
 * d_grad_low_bf16 [B, C_pad, h*w] bf16 out (overwritten, pad rows zeroed) or NULL.
 * The upsampled [B,C,H,W] tensor never exists in memory.
 */
int lc2is_count_valid(const int64_t* d_labels, int64_t n, int C, int64_t ignore_index,
                      int64_t* d_n_valid, lc2is_stream_t stream);
/* *d_scale = mult / *d_n_valid (0 if no valid pixel): the 'mean' gradient scale, no host sync. */
int lc2is_mean_scale(const int64_t* d_n_valid, float mult, float* d_scale, lc2is_stream_t stream);
/* *d_loss = *d_loss_sum / *d_n_valid  (NaN when nothing is valid, like torch). */
int lc2is_finalize_loss(const double* d_loss_sum, const int64_t* d_n_valid, float* d_loss,
                        lc2is_stream_t stream);
/* Both of the above in one launch (for steps in which the loss sum is complete before the gradient scale is needed). */
int lc2is_mean_scale_finalize(const int64_t* d_n_valid, float mult, float* d_scale, const double* d_loss_sum,
                              float* d_loss, lc2is_stream_t stream);
int lc2is_upsample_ce_fwd_bwd(const float* d_low, const int64_t* d_labels,
                              int B, int C, int h, int w, int H, int W,
                              int64_t ignore_index, const float* d_grad_scale,
                              double* d_loss_sum, float* d_grad_low, void* d_grad_low_bf16,
                              lc2is_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * K2, weighted form: the same fused pass for a criterion configured with class weights and / or label smoothing,
 *       nn.CrossEntropyLoss(weight=w, ignore_index=ii, label_smoothing=eps) applied to
 *       F.interpolate(input, mode="bilinear", size=(H, W))     (engine.py:94 on final.py:44; loss.py:19-20).
 * lc2is_ce_weight_sum: *d_wsum += sum over counted labels (in [0,C) and != ignore_index) of w[label], in double
 *            (d_weight = NULL counts them): the 'mean' denominator of the weighted cross-entropy.  ACCUMULATED.
 * lc2is_upsample_ce_fwd_bwd_ex: lc2is_upsample_ce_fwd_bwd with
 *   d_weight         [C] fp32 class weights on the device, or NULL (all 1); the host never reads them.
 *   label_smoothing  eps in [0, 1] (else LC2IS_ERR_ARG).
 *   With W = sum_c w_c and a = (1-eps) w_t + (eps/C) W, a counted pixel adds
 *       a * logsumexp_c x_c - (1-eps) w_t x_t - (eps/C) sum_c w_c x_c          to *d_loss_sum, and
 *       g * (a * softmax_c - (1-eps) w_t [c == t] - (eps/C) w_c)              to dL/dx_c,
 *   scattered through the bilinear taps.  reduction='mean' is d_grad_scale = 1 / wsum and loss = loss_sum / wsum
 *   (wsum from lc2is_ce_weight_sum).  d_weight == NULL with eps == 0 runs exactly lc2is_upsample_ce_fwd_bwd.
 */
int lc2is_ce_weight_sum(const int64_t* d_labels, int64_t n, int C, int64_t ignore_index,
                        const float* d_weight, double* d_wsum, lc2is_stream_t stream);
int lc2is_upsample_ce_fwd_bwd_ex(const float* d_low, const int64_t* d_labels,
                                 int B, int C, int h, int w, int H, int W,
                                 int64_t ignore_index, const float* d_weight, float label_smoothing,
                                 const float* d_grad_scale, double* d_loss_sum, float* d_grad_low,
                                 void* d_grad_low_bf16, lc2is_stream_t stream);

/* Split form of K2 for power-of-two scales 8 / 16 (what the whole-step entries run): the same
 * reference lines (model/loss.py:19-20 + autograd), cut so that everything that depends on the
 * labels only happens once, in one pass over the int64 map.
 * lc2is_ce_labels_prepass: n_valid += #counted pixels; d_labels_packed [B,H,W] uint16 = label, with
 *   bit 15 set where label == ignore_index (not counted by the CE, still a row of the confusion
 *   matrix) and 0xFFFF where the label is outside [0,C); d_grad_low [B,C,h,w] fp32
 *   ACCUMULATES the un-scaled -onehot term (minus the bilinear tap weights of every counted pixel).
 *   d_grad_low / d_labels_packed / d_n_valid may each be NULL to skip that output.  Scales 4 / 8 / 16.
 * lc2is_upsample_ce_packed (scales 8 / 16): d_loss_sum += sum over counted pixels of
 *   (log-sum-exp - logit_target); d_grad_low ACCUMULATES the un-scaled softmax term (NULL = forward
 *   only).  After both calls d_loss_sum / n_valid is the mean CE and d_grad_low / n_valid its
 *   gradient (lc2is_cosine_logits_bwd applies the scale when given the fp32 gradient).
 * Unsupported geometries return LC2IS_ERR_UNSUPPORTED (use lc2is_upsample_ce_fwd_bwd). */
int lc2is_ce_split_supported(int h, int w, int H, int W);
int lc2is_ce_labels_prepass(const int64_t* d_labels,
                            int B, int C, int h, int w, int H, int W, int64_t ignore_index,
                            uint16_t* d_labels_packed, int64_t* d_n_valid,
                            float* d_grad_low, lc2is_stream_t stream);
/* Same as lc2is_ce_labels_prepass for labels that are already in the packed uint16 form. */
int lc2is_ce_labels_prepass_packed(const uint16_t* d_labels_packed, int B, int C, int h, int w, int H, int W,
                                   int64_t* d_n_valid, float* d_grad_low, lc2is_stream_t stream);
/* HOST function: narrow an int64 label map (host memory) to the library's HOST label form on its worker threads (see
 * lc2is_pack_threads).  Blocks until done.  The host form has lc2is_host_label_bytes(C) bytes per label: 1 for
 * C <= 254 (class id; 0xFE = label == ignore_index; 0xFF = outside [0,C)), else 2 (the packed uint16 form above).
 * The whole-step entries take it as `h_scratch`; on the device the one-byte form is widened by lc2is_expand_labels. */
int lc2is_host_label_bytes(int C);
int lc2is_pack_labels_host(const int64_t* h_labels, int64_t n, int C, int64_t ignore_index, void* h_out);
/* Asynchronous form for a prefetching loader: _begin returns at once, _end blocks until the labels are packed and
 * releases the handle.  lc2is_head_step_host[_submit] accept labels packed this way: h_labels = NULL, h_scratch = them. */
int lc2is_pack_labels_host_begin(const int64_t* h_labels, int64_t n, int C, int64_t ignore_index, void* h_out,
                                 void** handle);
int lc2is_pack_labels_host_end(void* handle);
/* DEVICE: one-byte host form [n] -> packed uint16 [n]; n_valid += #counted labels (NULL = don't count).  n % 16 == 0,
 * C <= 254. */
int lc2is_expand_labels(const uint8_t* d_labels8, int64_t n, int C, int64_t ignore_index,
                        uint16_t* d_labels_packed, int64_t* d_n_valid, lc2is_stream_t stream);
/* number of worker threads the packing pool uses (hardware threads / LOCAL_WORLD_SIZE - 2, 1..12) */
int lc2is_pack_threads(void);
int lc2is_upsample_ce_packed(const float* d_low, const uint16_t* d_labels_packed,
                             int B, int C, int h, int w, int H, int W,
                             double* d_loss_sum, float* d_grad_low, lc2is_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * K3  argmax + confusion matrix.  Replaces, per image,
 *       F.interpolate(bicubic) + nn.Softmax2d + JaccardIndex (argmax + bincount)
 *       metrics.py:84-92 (compute_mIOU), :63-69 (compute_gt_mIOU), :127-134
 *       (compute_mIOU_tensor), utils.py:15-22 (generate_masks).
 * lc2is_argmax_confmat        : logits already at mask resolution [N,C,H,W] (fp32/bf16).
 * lc2is_argmax_confmat_lowres : logits at [N,C,h,w]; bilinear / bicubic (A=-0.75,
 *                               align_corners=False) resize to H x W done in registers.
 * d_labels   [N, lh, lw] int64; H % lh == 0 and W % lw == 0: nearest-upsampled in-kernel
 *            (metrics.py:90).  Targets outside [0,C) are skipped.
 * d_confmat  [C, C] int64 ACCUMULATED, rows = target, cols = prediction (all rows kept: the
 *            host zeroes the ignore row where the reference does).
 * d_per_image [N, 3, C] int64 ACCUMULATED or NULL: per image (true-positive, target count,
 *            prediction count) per class - enough for metrics.py:91-97's per-image IoU.
 * d_pred     [N, H, W] int64 out or NULL: the argmax masks (first index wins ties).
 */
int lc2is_argmax_confmat(const void* d_logits, int dtype, int N, int C, int H, int W,
                         const int64_t* d_labels, int lh, int lw,
                         int64_t* d_confmat, int64_t* d_per_image, int64_t* d_pred,
                         lc2is_stream_t stream);
int lc2is_argmax_confmat_lowres(const float* d_low, int N, int C, int h, int w, int H, int W,
                                int mode, const int64_t* d_labels, int lh, int lw,
                                int64_t* d_confmat, int64_t* d_per_image, int64_t* d_pred,
                                lc2is_stream_t stream);
/* Same, bilinear, scale 8 / 16 only, with the packed labels [N,H,W] written by lc2is_ce_labels_prepass
 * (what the whole-step entries run; LC2IS_ERR_UNSUPPORTED otherwise). */
int lc2is_argmax_confmat_lowres_packed(const float* d_low, int N, int C, int h, int w, int H, int W,
                                       const uint16_t* d_labels_packed,
                                       int64_t* d_confmat, int64_t* d_per_image, int64_t* d_pred,
                                       lc2is_stream_t stream);

/* RAGGED batch in one launch (SURVEY 8f-2): image i of d_low [N,C,h,w] is resized (bilinear / bicubic, ATen's
 * `size=` scale in/out) to ITS OWN H_i x W_i, argmaxed and compared with its own ground truth.  Replaces the per-image
 * Python loops of compute_gt_mIOU (metrics.py:61-79) and generate_masks (utils.py:15-22).
 * d_desc    [N][4] int64: { element offset of image i in d_labels / d_pred, H_i, W_i, first tile of image i } with
 *           first tile = running sum of lc2is_ragged_tiles(H_j, W_j), j < i; n_tiles = the total.
 * d_labels  flat int64 (image i: H_i*W_i elements at its offset) or NULL (masks only); targets outside [0,C) are skipped.
 * d_confmat [C,C] / d_per_image [N,3,C] ACCUMULATED or NULL; d_pred flat int64 out (same offsets) or NULL. */
long long lc2is_ragged_tiles(int H, int W);
int lc2is_argmax_confmat_ragged(const float* d_low, int N, int C, int h, int w, int mode,
                                const int64_t* d_desc, long long n_tiles, const int64_t* d_labels,
                                int64_t* d_confmat, int64_t* d_per_image, int64_t* d_pred,
                                lc2is_stream_t stream);

/* K2 (split form) and K3 in ONE persistent kernel of independent warps for the x16 geometry (k23_rc_kernel; what the
 * whole-step entries run when lc2is_ce_argmax_fused_supported): per job of two groups one TMA box stages the taps, a row
 * phase (lane = pixel row) does pass A of the cross-entropy and the running argmax in one sweep over the classes, a class
 * phase (lane = class) the tap gradients by Horner sweeps.  Same results as lc2is_upsample_ce_packed followed by
 * lc2is_argmax_confmat_lowres_packed (bilinear). */
int lc2is_ce_argmax_fused_supported(int C, int h, int w, int H, int W);
int lc2is_ce_argmax_fused_packed(const float* d_low, const uint16_t* d_labels_packed,
                                 int B, int C, int h, int w, int H, int W,
                                 double* d_loss_sum, float* d_grad_low, int onehot, int64_t* d_n_valid,
                                 int64_t* d_confmat, int64_t* d_per_image, int64_t* d_pred,
                                 lc2is_stream_t stream);
/* onehot != 0: the kernel also adds the un-scaled -onehot term to d_grad_low (it holds the row's labels anyway), so
 * the labels only need packing + counting ahead of the kernel (d_n_valid != NULL: the kernel counts too - for labels
 * that arrive packed from the host):
 * lc2is_pack_labels: int64 [n] -> packed uint16 [n] (same encoding as lc2is_ce_labels_prepass), n_valid += #counted.
 * n % 8 == 0. */
int lc2is_pack_labels(const int64_t* d_labels, int64_t n, int C, int64_t ignore_index,
                      uint16_t* d_labels_packed, int64_t* d_n_valid, lc2is_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * The cross-entropy stages of a whole step (K2 + K3 on the logits of K1; what HeadStep and
 * lc2is_head_step_host run), each picking its kernels from the geometry:
 *   route     labels stage              CE stage                                argmax stage
 *   fused     lc2is_pack_labels         lc2is_ce_argmax_fused_packed, onehot=1  nothing
 *             (packs, counts)           (loss, softmax - onehot, confmat)
 *   split     lc2is_ce_labels_prepass   lc2is_upsample_ce_packed                lc2is_argmax_confmat_lowres_packed
 *             (packs, counts, -onehot)
 *   one-call  lc2is_count_valid         lc2is_upsample_ce_fwd_bwd               lc2is_argmax_confmat_lowres
 *                                       (d_grad_scale NULL)                     (LC2IS_BILINEAR, labels at H x W)
 * fused where lc2is_ce_argmax_fused_supported, else split where lc2is_ce_split_supported, else one-call.
 * The CE and argmax stages read the packed labels the labels stage wrote.  d_n_valid, d_loss_sum, d_confmat ACCUMULATE.
 * d_labels [B,H,W] int64 (read by the labels stage, and by the other two on the one-call route).
 * d_labels_packed [B,H,W] uint16, written by the labels stage; NULL only on the one-call route (else LC2IS_ERR_ARG).
 * d_grad_low [B,C,h,w] fp32, un-scaled (1/n_valid is K1b's d_grad_scale), or NULL = forward only: on the split and fused
 *   routes the labels and CE stages ACCUMULATE into it (zero it first), on the one-call route the CE stage overwrites it.
 */
int lc2is_step_ce_labels(const int64_t* d_labels, int B, int C, int h, int w, int H, int W, int64_t ignore_index,
                         uint16_t* d_labels_packed, int64_t* d_n_valid, float* d_grad_low, lc2is_stream_t stream);
int lc2is_step_ce(const float* d_low, const int64_t* d_labels, const uint16_t* d_labels_packed,
                  int B, int C, int h, int w, int H, int W, int64_t ignore_index,
                  double* d_loss_sum, float* d_grad_low, int64_t* d_confmat, lc2is_stream_t stream);
int lc2is_step_argmax(const float* d_low, const int64_t* d_labels, const uint16_t* d_labels_packed,
                      int B, int C, int h, int w, int H, int W, int64_t* d_confmat, lc2is_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * K4  ContrastiveLoss on the low-resolution logits.  Replaces model/loss.py:39-64
 *       loss_visual  = CrossEntropyLoss(out [B,C,h,w], labels [B,h,w])            (class axis, ignore_index)
 *       loss_textual = CrossEntropyLoss(out [B,h,w,C], one_hot(labels,151).float()) (torch takes dim 1 = the image-row
 *                      axis as the class axis; 'mean' = / (B*w*C))
 *     and their autograd backward.
 * d_out      [B, h*w, C] fp32 (the reference's `outputs`), C <= 160.
 * d_labels   [B, h, w] int64 at the SAME resolution.
 * d_col_lse / d_col_adj  [B, w, C] fp32 workspaces written by _fwd and read by _bwd: per column, the log-sum-exp over
 *            y, and that minus ln(#rows whose label is c) (+inf where there is none).
 * d_loss_sums [2] double ACCUMULATED: { sum over counted pixels of the visual CE, un-normalised textual sum }.
 * d_counts   [2] int64 ACCUMULATED: { counted pixels (label != ignore_index), labels outside [0,C) - F.one_hot raises
 *            on those in the reference; the Python mirror raises when the second counter is non-zero }.
 * _bwd: d_coef DEVICE float[2] = { c_visual, c_textual }: d_grad [B,h*w,C] (overwritten) =
 *            c_visual * d(visual sum)/d out + c_textual * d(textual sum)/d out; for the reference's
 *            (loss_textual + loss_visual)/2 pass { 0.5/n_counted, 0.5/(B*w*C) }.
 */
int lc2is_contrastive_fwd(const float* d_out, const int64_t* d_labels, int B, int h, int w, int C,
                          int64_t ignore_index, float* d_col_lse, float* d_col_adj,
                          double* d_loss_sums, int64_t* d_counts, lc2is_stream_t stream);
int lc2is_contrastive_bwd(const float* d_out, const int64_t* d_labels, int B, int h, int w, int C,
                          int64_t ignore_index, const float* d_col_lse, const float* d_col_adj,
                          const float* d_coef, float* d_grad, lc2is_stream_t stream);

/* ---------------------------------------------------------------------------------------
 * Whole step from HOST buffers (the end-to-end path bench.py times as `e2e`).  Replaces one
 * iteration of Engine.train_loop / eval_loop over the head (engine.py:75-101,145-163):
 * H2D of the batch, K0..K3, D2H of loss / n_valid / confusion matrix.  Synchronises
 * `stream` before returning.  Host pointers should be pinned.
 * h_v [B,hw,D] bf16, h_t [C,D] fp32, h_labels [B,H,W] int64.
 * h_out_loss (mean CE), h_out_n_valid, h_out_confmat [C,C] (overwritten).
 * d_ws: device workspace of lc2is_head_step_workspace(...) bytes (caller-allocated).
 * do_backward: also run K1b (gradients stay on the device, in the workspace).
 * copy_stream: optional second stream (NULL = none): the batch is then cut into chunks and the H2D copy
 *   of chunk i+1 overlaps the kernels of chunk i (the 1/N_valid scale is applied at the end, in K1b).
 * h_scratch: optional PINNED host buffer of B*H*W*lc2is_host_label_bytes(C) bytes (NULL = none).  With it (and a
 *   power-of-two scale 8 / 16) the int64 labels are narrowed to the 1- or 2-byte host form on the library's host
 *   worker threads, chunk by chunk ahead of the copies, so an eighth / a quarter of the label bytes cross PCIe.
 * n_raw: the LAST n_raw images' labels cross as int64 anyway and are packed on the device, concurrently with the host
 *   threads narrowing the first B - n_raw (0 = all on the host; for hosts whose cores read 8 bytes per label more
 *   slowly than PCIe moves them - HostStep calibrates the split).  Ignored without h_scratch.
 * flags: LC2IS_STEP_LABELS_PREPACKED - h_scratch already holds the host-form labels of the first B - n_raw images
 *   (lc2is_pack_labels_host / _begin + _end, or a loader that writes them itself); also implied by h_labels == NULL
 *   (then n_raw must be 0).
 */
#define LC2IS_STEP_LABELS_PREPACKED 1
int64_t lc2is_head_step_workspace(int B, int hw, int D, int C, int H, int W);
int lc2is_head_step_host(const void* h_v, const float* h_t, const int64_t* h_labels,
                         int B, int h, int w, int D, int C, int H, int W,
                         int64_t ignore_index, float logit_scale, int do_backward,
                         float* h_out_loss, int64_t* h_out_n_valid, int64_t* h_out_confmat,
                         void* d_ws, lc2is_stream_t stream, lc2is_stream_t copy_stream,
                         void* h_scratch, int n_raw, int flags);

/* The same step without the final synchronisation: everything (host-side label packing, H2D, kernels, D2H
 * of the results) is enqueued and *done_event receives a handle; lc2is_head_step_host_wait blocks until that
 * step's results are in the h_out_* buffers and releases the handle.  The copy of step i+1 then overlaps the
 * kernels of step i (a prefetching data loader: engine.py:75 copies the next batch while the previous one
 * computes).  Each step in flight needs its own workspace, scratch and output buffers; all host buffers
 * must stay valid until the wait returns.  copy_stream must be a second stream. */
int lc2is_head_step_host_submit(const void* h_v, const float* h_t, const int64_t* h_labels,
                                int B, int h, int w, int D, int C, int H, int W,
                                int64_t ignore_index, float logit_scale, int do_backward,
                                float* h_out_loss, int64_t* h_out_n_valid, int64_t* h_out_confmat,
                                void* d_ws, lc2is_stream_t stream, lc2is_stream_t copy_stream,
                                void* h_scratch, int n_raw, int flags, void** done_event);
int lc2is_head_step_host_wait(void* done_event);

#ifdef __cplusplus
}
#endif
#endif /* LC2IS_B200_H */

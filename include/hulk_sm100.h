/*
 * hulk_sm100.h -- C ABI of libhulk_sm100.so, the B200 (sm_100a) implementation of the
 * hulk-keypoints KeypointsGauss hot path.
 *
 * This is the drop-in boundary (SURVEY.md §8b).  The reference (vainaviv/hulk-keypoints) is pure
 * Python on torch and has no FFI of its own: every entry point below replaces one torch call site
 * of the reference, cited as <file>:<line> relative to the reference root.  The Python host
 * package (hulk_keypoints_b200/) binds these with ctypes; INTEGRATION.md shows the stub a
 * maintainer of the reference would add.
 *
 * Conventions
 *   - One call == one (or a few) kernel enqueue(s) on the cudaStream_t passed in.  The library never
 *     allocates or frees device memory on the call path, never synchronises the device, and never
 *     falls back to the CPU.
 *   - All device buffers are owned by the caller.  Pointers are plain device pointers.
 *   - Return value: HK_OK (0) or a negative HkStatus; hk_last_error() returns a thread-local
 *     human-readable message for the last failing call on this thread.
 *   - Activations between kernels are NHWC ("channels last"); NCHW fp32 only at the API edge
 *     (network input, heatmap output), which is what the reference's tensors are.
 *   - `stream` is passed as void* (a cudaStream_t) so the header needs no CUDA include.
 */
#ifndef HULK_SM100_H_
#define HULK_SM100_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HK_ABI_VERSION 1

#if defined(__GNUC__)
#define HK_API __attribute__((visibility("default")))
#else
#define HK_API
#endif

typedef enum HkStatus {
  HK_OK = 0,
  HK_ERR_BAD_ARG = -1,     /* null pointer, bad shape, misaligned buffer, unsupported combination */
  HK_ERR_UNSUPPORTED_ARCH = -2, /* device is not sm_100 */
  HK_ERR_CUDA = -3         /* CUDA runtime / launch error; text in hk_last_error() */
} HkStatus;

typedef enum HkDType { HK_F32 = 0, HK_BF16 = 1, HK_F64 = 2 } HkDType;

/* Which kernel family executes a convolution. */
typedef enum HkConvAlgo {
  HK_CONV_TCGEN05 = 0, /* bf16 operands, fp32 accumulate in TMEM, TMA-fed implicit GEMM            */
  HK_CONV_FFMA = 1,    /* fp32 CUDA-core implicit GEMM: the fp32 correctness mode (SURVEY.md §0.5) */
  HK_CONV_TCGEN05_1CTA = 2 /* force the generic single-CTA tcgen05 kernel (no cta_group::2 / layer1 specialisation);
                              kept for shapes the specialised kernels do not cover and as the reference route tests compare against */
} HkConvAlgo;

/*
 * One fused conv + per-channel affine (+ residual) (+ ReLU).
 * Replaces  nn.Conv2d -> nn.BatchNorm2d(eval) -> [+= residual] -> nn.ReLU
 *   src/resnet.py:56-67 (BasicBlock.forward), src/resnet.py:184-188 (downsample), src/resnet.py:199-201 (stem).
 *   y[b,oy,ox,n] = act( scale[n] * sum_{r,s,c} x[b, oy*stride-pad+r*dil, ox*stride-pad+s*dil, c] * w[n,r,s,c]
 *                       + bias[n] + residual[b,oy,ox,n] )
 */
typedef struct HkConvDesc {
  int32_t batch;
  int32_t in_h, in_w, in_c;
  int32_t out_h, out_w, out_c;
  int32_t kh, kw;
  int32_t stride, pad, dil;
  int32_t relu;          /* 0/1 */
  int32_t in_dtype;      /* HkDType of x (HK_F32 or HK_BF16)                       */
  int32_t out_dtype;     /* HkDType of y and residual                              */
  int32_t in_is_nchw;    /* 1: x is NCHW (network input, FFMA algo only); 0: NHWC  */
  int32_t algo;          /* HkConvAlgo                                             */
} HkConvDesc;

/* ---- library ---- */
HK_API int hk_version(void);
HK_API const char* hk_last_error(void);
/* 0 if the current device is sm_100 (B200), HK_ERR_UNSUPPORTED_ARCH otherwise. */
HK_API int hk_check_device(void);

/* ---- weights ----
 * Repack one conv + its BatchNorm for the kernels above.
 * Replaces the implicit parameter layout of nn.Conv2d/nn.BatchNorm2d (src/resnet.py:36,46,137,139,185,187).
 *   w_oihw : (cout, cin, kh, kw) fp32, the state_dict tensor
 *   bn_*   : (cout) fp32 gamma, beta, running_mean, running_var; all four NULL => scale=1, bias=conv_bias_or_0
 *   w_out  : (cout, kh, kw, cin) in `w_dtype` (HK_BF16 for TCGEN05, HK_F32 for FFMA)
 *   scale/bias_out : (cout) fp32:  scale = gamma / sqrt(var + eps),  bias = beta - mean * scale
 */
HK_API int hk_pack_conv_weights(const float* w_oihw, const float* bn_gamma, const float* bn_beta,
                         const float* bn_mean, const float* bn_var, float bn_eps,
                         int cout, int cin, int kh, int kw, int w_dtype,
                         void* w_out, float* scale_out, float* bias_out, void* stream);

/* ---- backbone ---- */
HK_API int hk_conv_bn_act_fwd(const HkConvDesc* desc, const void* x, const void* w_packed,
                       const float* scale, const float* bias, const void* residual_or_null,
                       void* y, void* stream);

/* Entry of a stride/channel-changing BasicBlock in ONE launch: conv1+bn1+ReLU and the 1x1 downsample conv+bn of the same input.
 * Replaces src/resnet.py:56-58 (conv1, bn1, relu) together with :64-65 / :184-188 (downsample = conv1x1(stride) + BatchNorm2d).
 *   y    = relu?( scale    * conv_kxk(x; stride, pad, dil) + bias    )      desc->relu
 *   y_ds =        scale_ds * conv_1x1(x; stride)           + bias_ds
 * desc describes the kxk conv; it must be odd-sized with pad == dil*(k/2), so the 1x1 conv reads exactly its centre-tap operand
 * (the kernel issues the downsample MMAs on the centre-tap boxes against w_ds: no second pass over x).  tcgen05 path only
 * (bf16 NHWC, out_c % 128 == 0, in_c % 64 == 0, stride 1 or 2); w_ds_packed (out_c, 1, 1, in_c) bf16 from hk_pack_conv_weights.
 * Bit-identical to two hk_conv_bn_act_fwd calls. */
HK_API int hk_conv_ds_fwd(const HkConvDesc* desc, const void* x, const void* w_packed, const float* scale, const float* bias, void* y,
                          const void* w_ds_packed, const float* scale_ds, const float* bias_ds, void* y_ds, void* stream);

/* Stem on the tensor cores (bf16 mode): conv 7x7 s2 p3 (3->64) + folded BN + ReLU.
 * Replaces src/resnet.py:137-139,199-201.  x (B,3,H,W) fp32 NCHW -- the reference's input tensor -- is rounded to
 * bf16 on the fly; y (B,H/2,W/2,64) bf16 NHWC.  w_packed comes from hk_stem_pack_weights (conv1.weight (64,3,7,7)
 * fp32 -> (64,256) bf16, k = r*32 + s*4 + c, zero padding elsewhere); scale/bias from hk_pack_conv_weights. */
HK_API size_t hk_stem_packed_weight_bytes(void);
HK_API int hk_stem_pack_weights(const float* w_oihw, void* w_out, void* stream);
HK_API int hk_stem_fwd(const float* x_nchw, const void* w_packed, const float* scale, const float* bias,
                       void* y_nhwc, int B, int H, int W, void* stream);
/* Same, reading the image as cv2.imread delivers it: (B,H,W,3) uint8.  The ToTensor step of the reference
 * (src/dataset.py:16,71 / analysis.py:37: HWC uint8 -> CHW float32 / 255) is fused into the load, so the host->device
 * copy is 4x smaller (SURVEY.md §8 f3). */
HK_API int hk_stem_fwd_u8(const uint8_t* x_nhwc_u8, const void* w_packed, const float* scale, const float* bias,
                          void* y_nhwc, int B, int H, int W, void* stream);

/* Stem + max-pool in ONE kernel (inference): conv 7x7 s2 p3 + folded BN + ReLU + MaxPool2d(3,2,1).  Replaces src/resnet.py:137-141,
 * 199-202 without writing the (B,H/2,W/2,64) stem map: row-streaming tcgen05 kernel, input rows by TMA, pooled bf16 NHWC out.
 * y (B, Hp, Wp, 64) bf16 with Hp = (H/2 + 1)/2 rounded as MaxPool2d does.  Bit-identical to hk_stem_fwd + hk_maxpool3x3s2_fwd.
 * Needs W % 4 == 0 (fp32) / W % 16 == 0 (uint8) for the TMA row pitch; otherwise HK_ERR_BAD_ARG (use the two-kernel path). */
HK_API int hk_stem_pool_fwd(const float* x_nchw, const void* w_packed, const float* scale, const float* bias, void* y_pooled_nhwc,
                            int B, int H, int W, void* stream);
HK_API int hk_stem_pool_fwd_u8(const uint8_t* x_nhwc_u8, const void* w_packed, const float* scale, const float* bias,
                               void* y_pooled_nhwc, int B, int H, int W, void* stream);

/* MaxPool2d(kernel 3, stride 2, pad 1) on NHWC.  Replaces src/resnet.py:141,202. */
HK_API int hk_maxpool3x3s2_fwd(const void* x, void* y, int dtype, int batch, int in_h, int in_w, int c,
                        int out_h, int out_w, void* stream);

/* ---- head ----
 * Scoring conv restricted to the K live rows + bilinear upsample (align_corners=True) + sigmoid.
 * Replaces src/resnet.py:215 (fc as 1x1 conv), src/resnet_dilated.py:27 (upsample_bilinear),
 *          src/model.py:21 (slice [:, :K] and sigmoid).
 *   feat      : (B, h, w, C) NHWC, feat_dtype
 *   w_fc      : (K, C) fp32  -- rows [0,K) of fc.weight ; b_fc : (K) fp32
 *   logits_ws : (B, K, h, w) fp32 scratch owned by the caller
 *   heat      : (B, K, H, W) fp32 NCHW
 */
HK_API int hk_head_fwd(const void* feat, int feat_dtype, const float* w_fc, const float* b_fc,
                float* logits_ws, float* heat, int B, int K, int C, int h, int w, int H, int W,
                void* stream);
/* The same head with the scoring conv folded into the LAST backbone conv (inference, K <= 8):
 *   hk_conv_head_fwd     : layer4[2].conv2 + bn2 + shortcut + ReLU (src/resnet.py:60-67) and the K live rows of `fc` (src/resnet.py:215,
 *                          src/model.py:21) in one tcgen05 launch.  The epilogue multiplies each finished row -- rounded to bf16 exactly as the
 *                          feature map would have stored it -- with w_fc (K, out_c) fp32 and adds the K partial sums to logits
 *                          (B, K, out_h, out_w) fp32; the (B, out_h, out_w, 512) feature map is never written or re-read.  logits must be
 *                          ZERO on entry (each element receives the two 256-column tiles' contributions; fp32 addition is commutative,
 *                          so the result is independent of their order).  Needs out_c == 512, stride 1, bf16 NHWC.
 *   hk_head_upsample_fwd : x8 bilinear upsample (align_corners=True, src/resnet_dilated.py:27) + sigmoid of such logits -> heat (B,K,H,W). */
HK_API int hk_conv_head_fwd(const HkConvDesc* desc, const void* x, const void* w_packed, const float* scale, const float* bias,
                            const void* residual_or_null, const float* w_fc, const float* b_fc, int K, float* logits, void* stream);
HK_API int hk_head_upsample_fwd(const float* logits, float* heat, int B, int K, int h, int w, int H, int W, int fast, void* stream);


/* ---- decode ----
 * Per-keypoint argmax with first-index tie-break.  Replaces src/prediction.py:46
 * (np.unravel_index(h.argmax(), h.shape)), for every batch element instead of [0] only.
 *   heat (B,K,H,W) fp32 ; yx (B,K,2) int32 = (row, col) ; maxval (B,K) fp32 or NULL
 *   ws : hk_argmax_workspace_bytes(B,K,H,W) bytes of scratch
 */
HK_API size_t hk_argmax_workspace_bytes(int B, int K, int H, int W);
HK_API int hk_argmax_decode(const float* heat, int B, int K, int H, int W, int32_t* yx, float* maxval_or_null,
                     void* ws, size_t ws_bytes, void* stream);

/* Every instance per channel (additive; the reference decodes one argmax per channel): thresholded local maxima, top N per map.
 * Pixel p with value v is a peak iff v >= threshold, v > q for every neighbour q of its (2r+1)x(2r+1) window (clipped to the image)
 * that precedes p in row-major order, and v >= q for every neighbour after p; NaN counts as -inf (never a peak, suppresses nothing).
 * On a flat top only the first pixel survives; on a NaN-free map the top-1 peak is hk_argmax_decode's (row, col) and value.
 *   heat (B,K,H,W) fp32 contiguous ; r = min_distance in [1, 16] ; N = max_peaks in [1, 256] ; threshold finite
 *   yx (B,K,N,2) int32 = (row, col), score (B,K,N) fp32: the peaks by value descending, ties by flat index ascending; unused slots
 *   hold (-1, -1) and -inf ; count (B,K) int32 = peaks kept (<= N)
 *   ws : hk_peak_workspace_bytes(B,K,H,W,N,r) bytes of scratch, 8-byte aligned (0 for arguments out of range) */
HK_API size_t hk_peak_workspace_bytes(int B, int K, int H, int W, int max_peaks, int min_distance);
HK_API int hk_peak_decode(const float* heat, int B, int K, int H, int W, int max_peaks, int min_distance, float threshold,
                          int32_t* yx, float* score, int32_t* count, void* ws, size_t ws_bytes, void* stream);

/* Soft-argmax of every (H, W) map: Prediction.expectation, src/prediction.py:31-38 (called at :45), softmax (:26-29) included.
 * The reference's flattening quirk is kept: the map is flattened column-major (`d.T.ravel()`, flat index i = c*H + r) while the
 * index arrays assume row-major order (x' = i % W, y' = i // W).  One pass over the heatmaps (online softmax; fp32 exp, fp64 sums).
 *   heat (maps, H, W) fp32 contiguous (maps = B*K) ; exp_xy (maps, 2) fp64 = (E[x'], E[y']) ;
 *   exp_int_or_null (maps, 2) int32 = the reference's `int(...)` truncation ; ws : hk_soft_argmax_workspace_bytes bytes. */
HK_API size_t hk_soft_argmax_workspace_bytes(int maps, int H, int W);
HK_API int hk_soft_argmax(const float* heat, int maps, int H, int W, double* exp_xy, int32_t* exp_int_or_null, void* ws,
                          size_t ws_bytes, void* stream);

/* ---- training-side elementwise / reduction kernels ----
 * Gaussian heatmap targets.  Replaces gauss_2d_batch, src/dataset.py:36-44 (fp32 math, widened to f64).
 *   uv (B,K,2) fp32 = (x, y) ; out (B,K,H,W) in out_dtype (HK_F64 drop-in, HK_F32 compact)
 */
HK_API int hk_gauss_targets(const float* uv, int B, int K, int H, int W, float sigma, void* out, int out_dtype,
                     void* stream);

/* `normalize` of src/dataset.py:33-34 as applied by gauss_2d_batch(normalize_dist=True) (dataset.py:42-44): L1-normalise a (K,H,W)
 * fp32 tensor over dim 1 (F.normalize(x, p=1), eps 1e-12) and widen to fp64. */
HK_API int hk_l1_normalize_dim1(const float* x, int K, int H, int W, double* out, void* stream);

/* BCE(mean) forward + backward through the sigmoid.  Replaces train.py:21,25 (pred.double(), nn.BCELoss)
 * and the autograd of train.py:35 down to the logits (model.py:21).
 *   pred   : (N) fp32 heatmap values (post-sigmoid), or the upsampled LOGITS when pred_is_logits != 0
 *            (the sigmoid of model.py:21 is then evaluated in-kernel and no heatmap is materialised)
 *   target : (N) fp64 or fp32 (target_dtype), or NULL with uv != NULL to generate the Gaussian on the fly
 *   uv     : (B,K,2) fp32 labels when target == NULL (then N must equal B*K*H*W)
 *   loss   : (1) fp64 mean loss ; grad_logits : (N) fp32 or NULL (forward only)
 *   ws     : hk_bce_workspace_bytes(N) bytes
 */
HK_API size_t hk_bce_workspace_bytes(long long n);
HK_API int hk_bce_fwd_bwd(const float* pred, int pred_is_logits, const void* target_or_null, int target_dtype,
                   const float* uv_or_null, int B, int K, int H, int W, float sigma,
                   double* loss, float* grad_logits_or_null, void* ws, size_t ws_bytes, void* stream);

/* ---- optimiser ----
 * One fused Adam step over flat fp32 buffers (coupled L2 weight decay, no amsgrad) -- torch.optim.Adam(lr, weight_decay)
 * of train.py:79 as applied at train.py:36.  `step` is the 1-based step count used for the bias corrections. */
HK_API int hk_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, long long n,
                        float lr, float beta1, float beta2, float eps, float weight_decay, int step, void* stream);

/* One Adam step over flat fp32 buffers whose runs differ in hyperparameters or step count (torch.optim.Adam / AdamW parameter
 * groups, learning-rate schedules): ONE launch for any number of segments.  The segments cover [0, ceil(n/4)) in float4 units,
 * non-empty, sorted and contiguous; the n % 4 tail belongs to the last one.  Per segment, computed in double on the host as
 * hk_adam_step does: lr_over_bc1 = lr / (1 - beta1^t), inv_sqrt_bc2 = 1 / sqrt(1 - beta2^t).  decoupled == 0: coupled L2
 * (g += weight_decay * p; bit-identical to hk_adam_step); decoupled != 0: p *= decay (= 1 - lr * weight_decay, rounded to fp32)
 * before the update on the unmodified gradient.  The table is read during the call (it travels as a launch parameter), so the
 * call is capturable and `segments` may be reused right after it returns.  At most HK_ADAM_MAX_SEGMENTS segments. */
#define HK_ADAM_MAX_SEGMENTS 256
typedef struct HkAdamSegment {
  long long begin4, end4;
  float lr_over_bc1, inv_sqrt_bc2;
  float beta1, beta2, eps, weight_decay;
  float decay;
  int decoupled;
} HkAdamSegment;
HK_API int hk_adam_step_segments(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, long long n,
                                 const HkAdamSegment* segments, int num_segments, void* stream);

/* ---- training: backbone forward in train() mode and its backward (SURVEY.md §8 f1) ----
 * Replaces what torch autograd does for train.py:33-36 between the input batch and the parameter gradients.  Activations are
 * NHWC bf16 (P = B*H*W rows of C channels), statistics / parameters / parameter gradients fp32.  Every reduction is a fixed-order
 * two-level sum (deterministic).  Convolutions in training reuse hk_conv_bn_act_fwd with scale = 1, bias = 0, relu = 0 (raw conv
 * output); the data gradient of a conv is hk_conv_bn_act_fwd on weights repacked by hk_pack_conv_weights_dgrad.
 */
/* Stem conv with an explicit ReLU switch (relu = 0: raw conv output for train-mode BN).  src/resnet.py:137,199. */
HK_API int hk_stem_conv_fwd(const float* x_nchw, const void* w_packed, const float* scale, const float* bias, void* y_nhwc,
                            int B, int H, int W, int relu, void* stream);

/* nn.BatchNorm2d in train() mode, forward statistics (src/resnet.py:46,49,139,187 under model.train()).
 *   y (P,C) bf16 raw conv output -> mean, invstd (C) fp32 (biased variance, eps inside the sqrt), and the fused affine of the
 *   apply pass: scale = gamma*invstd, shift = beta - mean*scale.  running_mean/var (nullable) are updated in place:
 *   r = (1-momentum)*r + momentum*stat, with the UNBIASED variance, as torch does.  ws: hk_bn_workspace_bytes(C). */
HK_API size_t hk_bn_workspace_bytes(int C);
HK_API int hk_bn_train_stats(const void* y, long long P, int C, const float* gamma, const float* beta, float* running_mean,
                             float* running_var, float momentum, float eps, float* mean_out, float* invstd_out,
                             float* scale_out, float* shift_out, void* ws, size_t ws_bytes, void* stream);
/* out = relu?(y*scale + shift [+ residual])  (BN apply + the in-place add and ReLU of BasicBlock.forward, src/resnet.py:64-67).
 * relu_bits_or_null (P*C/8 bytes, only written when relu != 0): bit j of byte v = [out[8v+j] > 0], the ReLU mask for hk_bn_train_bwd
 * at 1/16 of the bytes of `out`. */
HK_API int hk_bn_apply_fwd(const void* y, const float* scale, const float* shift, const void* residual_or_null, int relu,
                           void* out, void* relu_bits_or_null, long long P, int C, void* stream);
/* Backward of ReLU (mask: the saved post-ReLU output (mask_is_bits = 0) or the bit array written by hk_bn_apply_fwd (mask_is_bits = 1);
 * NULL = no ReLU) + train-mode BatchNorm:
 *   d' = dout*[out>0]; dbeta = sum d'; dgamma = sum d'*xhat; dy = gamma*invstd*(d' - dbeta/P - xhat*dgamma/P)
 *   dmasked_or_null receives d' (the gradient of the shortcut branch).  accumulate != 0 adds to dgamma/dbeta.
 *   ws: hk_bn_workspace_bytes(C) + 3*C*4 bytes. */
HK_API int hk_bn_train_bwd(const void* dout, const void* out_mask_or_null, int mask_is_bits, const void* y, const float* mean, const float* invstd,
                           const float* gamma, long long P, int C, float* dgamma, float* dbeta, int accumulate, void* dy,
                           void* dmasked_or_null, void* ws, size_t ws_bytes, void* stream);

/* The same three BatchNorm steps without the finalize launches (the training engine's path; 2 + 2 launches per BatchNorm instead of
 * 3 + 3).  The reduce kernels add their per-block fp32 partial sums into per-channel 128-bit fixed-point accumulators with integer
 * atomics (exact, hence independent of the order the blocks retire in: deterministic), and the apply kernels derive their per-channel
 * coefficients from the accumulators in their own prologue.  acc: hk_bn_acc_bytes(C) bytes (2*C accumulators of 32 bytes), 32-byte
 * aligned, ZERO when the reduce kernel starts (one cudaMemsetAsync over all accumulators of a step); forward and backward of one
 * BatchNorm use different accumulator buffers.
 *   hk_bn_stats_acc     : acc[0..C) += sum_p y, acc[C..2C) += sum_p y^2
 *   hk_bn_apply_fwd_acc : mean/invstd (saved for the backward) + running stats from acc, then out = relu?(gamma*xhat + beta [+ residual])
 *   hk_bn_bwd_acc       : acc += (sum d', sum d'*xhat), then dgamma/dbeta and dy (+ d') exactly as hk_bn_train_bwd */
HK_API size_t hk_bn_acc_bytes(int C);
HK_API int hk_bn_stats_acc(const void* y, long long P, int C, void* acc, void* stream);
HK_API int hk_bn_apply_fwd_acc(const void* y, const void* acc, long long P, int C, const float* gamma, const float* beta,
                               float* running_mean, float* running_var, float momentum, float eps, float* mean_out, float* invstd_out,
                               const void* residual_or_null, int relu, void* out, void* relu_bits_or_null, void* stream);
HK_API int hk_bn_bwd_acc(const void* dout, const void* out_mask_or_null, int mask_is_bits, const void* y, const float* mean,
                         const float* invstd, const float* gamma, long long P, int C, void* acc, float* dgamma, float* dbeta,
                         int accumulate, void* dy, void* dmasked_or_null, void* stream);

/* Frozen BatchNorm: an nn.BatchNorm2d in eval() mode inside a train()-mode model normalises with its running statistics and leaves
 * its buffers alone (torch's semantics).
 *   hk_bn_fold       : for every item, scale = gamma*invstd_r, shift = beta - mean_r*scale, invstd = 1/sqrt(running_var + eps)
 *                      (invstd nullable; gamma/beta NULL = 1/0), all items in one launch.  items_dev: device array of HkBnFoldItem;
 *                      max_c = the largest C.  The forward is then hk_bn_apply_fwd (or a conv epilogue) with this scale/shift.
 *   hk_bn_frozen_bwd : d' = dout*[out>0] (mask as for hk_bn_train_bwd, NULL = no ReLU), dy = scale*d' (nullable), d' into
 *                      dmasked_or_null; when dgamma or dbeta is given: acc (zeroed, hk_bn_acc_bytes(C)) += (sum d', sum d'*y), and
 *                      dbeta = sum d', dgamma = invstd*(sum d'*y - mean*sum d') from the exact totals (accumulate != 0 adds).  One pass,
 *                      one launch; y, mean (running mean) and invstd are only read for the sums. */
typedef struct HkBnFoldItem {
  const float* gamma;
  const float* beta;
  const float* mean;   /* running_mean */
  const float* var;    /* running_var */
  float* scale;
  float* shift;
  float* invstd;       /* or NULL */
  float eps;
  int32_t C;
} HkBnFoldItem;
HK_API int hk_bn_fold(const HkBnFoldItem* items_dev, int n_items, int max_c, void* stream);
HK_API int hk_bn_frozen_bwd(const void* dout, const void* out_mask_or_null, int mask_is_bits, const void* y_or_null, const float* scale,
                            const float* mean, const float* invstd, long long P, int C, void* acc_or_null, float* dgamma, float* dbeta,
                            int accumulate, void* dy_or_null, void* dmasked_or_null, void* stream);

/* Train-mode forward of one conv + the statistics pass of its BatchNorm in ONE launch (src/resnet.py:56-57,60-61 under model.train()):
 * y = conv(x) (raw output: pass scale = 1, bias = 0; desc->relu must be 0) and acc += per-channel (sum y, sum y^2) of the bf16 values
 * stored, gathered in the epilogue of the tcgen05 kernel from the staged output tile -- the activation is not read again for its
 * statistics.  acc as for hk_bn_stats_acc (zeroed, hk_bn_acc_bytes(out_c)); follow with hk_bn_apply_fwd_acc.  tcgen05 path only; a shape
 * outside the specialised kernels runs the conv followed by hk_bn_stats_acc. */
HK_API int hk_conv_bn_stats_fwd(const HkConvDesc* desc, const void* x, const void* w_packed, const float* scale, const float* bias,
                                void* y, void* acc, void* stream);

/* All convs of the network repacked in ONE launch (the training step repacks every step).  items_dev: device array of HkPackItem;
 * w_dgrad may be NULL (stem: no data gradient).  max_elems = max over items of cout*cin*khw. */
typedef struct HkPackItem {
  const float* w;   /* (cout, cin, kh, kw) fp32 */
  void* w_fwd;      /* (cout, kh, kw, cin) bf16 */
  void* w_dgrad;    /* (cin, kh, kw, cout) bf16, taps flipped; or NULL */
  int32_t cout, cin, khw, reserved;
} HkPackItem;
HK_API int hk_pack_conv_weights_many(const HkPackItem* items_dev, int n_items, long long max_elems, void* stream);
/* The same through shared-memory tiles (64 output x 32 input channels x all taps per CTA: contiguous source runs, 64-byte destination
 * runs in both layouts; ~3x faster).  Every item needs cout % 64 == 0, cin % 32 == 0 and khw <= max_khw. */
HK_API int hk_pack_conv_weights_many_tiled(const HkPackItem* items_dev, int n_items, int max_khw, long long max_elems, void* stream);

/* Conv weights for the data gradient: (cout,cin,kh,kw) fp32 -> (cin, kh, kw, cout) bf16 with the taps flipped. */
HK_API int hk_pack_conv_weights_dgrad(const float* w_oihw, int cout, int cin, int kh, int kw, void* w_out, void* stream);
/* (B,h,w,C) bf16 -> (B,2h,2w,C) with the values at even (y,x) and zeros elsewhere: the data gradient of a stride-2 conv is the
 * stride-1 data-gradient conv over this grid. */
HK_API int hk_zero_insert2x(const void* in, void* out, int B, int h, int w, int C, void* stream);

/* Conv weight gradient on tcgen05 (MN-major operands straight from the NHWC activations):
 *   dw[co,ci,r,s] (+)= sum_{b,oy,ox} dy[b,oy,ox,co] * x[b, oy*stride-pad+r*dil, ox*stride-pad+s*dil, ci]
 *   desc describes the FORWARD conv (x = its input, dy = gradient of its raw output); dw is OIHW fp32.
 *   ws: hk_conv_wgrad_workspace_bytes(desc) bytes of split-K partials. */
HK_API size_t hk_conv_wgrad_workspace_bytes(const HkConvDesc* desc);
HK_API int hk_conv_wgrad(const HkConvDesc* desc, const void* x, const void* dy, float* dw_oihw, int accumulate, void* ws,
                         size_t ws_bytes, void* stream);
/* Stem (7x7 s2, Cin=3) weight gradient from the fp32 NCHW input and the bf16 NHWC output gradient. */
HK_API size_t hk_stem_wgrad_workspace_bytes(void);
HK_API int hk_stem_wgrad(const float* x_nchw, const void* dy_nhwc, float* dw_oihw, int accumulate, int B, int H, int W, void* ws,
                         size_t ws_bytes, void* stream);

/* Sigmoid of src/model.py:21 and its backward (g_z = (g_p*(1-p))*p), for the split train step in which the CALLER computes the
 * loss on the heatmaps (unmodified train.py:21-25) and autograd hands dL/dheat back. */
HK_API int hk_sigmoid_fwd(const float* logits, float* heat, long long n, void* stream);
HK_API int hk_sigmoid_bwd(const float* heat, const float* grad_heat, float* grad_logits, long long n, void* stream);

/* MaxPool2d(3,2,1) backward (first-maximum routing, as ATen's indices). x = pool input (post-ReLU stem), NHWC bf16.
 * idx_ws: B*Ho*Wo*C bytes (the per-window argmax taps computed in a first pass). */
HK_API int hk_maxpool3x3s2_bwd(const void* dout, const void* x, void* dx, int B, int H, int W, int C, int Ho, int Wo, void* idx_ws,
                               size_t idx_ws_bytes, void* stream);
/* The training step's max-pool as forward-with-indices + gather: hk_maxpool3x3s2_fwd_idx writes y (B,Ho,Wo,C) bf16 AND idx (B*Ho*Wo*C bytes:
 * the tap r*3+s of the first maximum of each window in scan order, ATen's max_pool2d_with_indices rule) in one pass over x;
 * hk_maxpool3x3s2_bwd_idx routes dout through those indices (dx (B,H,W,C) bf16).  Same results as hk_maxpool3x3s2_fwd + hk_maxpool3x3s2_bwd,
 * one pass over the stem map fewer. */
HK_API int hk_maxpool3x3s2_fwd_idx(const void* x, void* y, void* idx, int B, int H, int W, int C, int Ho, int Wo, void* stream);
HK_API int hk_maxpool3x3s2_bwd_idx(const void* dout, const void* idx, void* dx, int B, int H, int W, int C, int Ho, int Wo, void* stream);


/* Head in training: K-row scoring conv + bilinear upsample WITHOUT the sigmoid (hk_bce_fwd_bwd takes logits), ATen's exact
 * operation order; and its backward: upsample-backward of g_up (B,K,H,W) to dlogits_ws (B,K,h,w), then
 * dfeat (B,h,w,C) bf16, dw_fc (K,C) fp32, db_fc (K) fp32.  Only the K live rows of fc get a gradient, as in the reference.
 * dfeat, dw_fc and db_fc may each be NULL (frozen backbone / frozen fc): their kernels are skipped. */
HK_API int hk_head_logits_fwd(const void* feat, int feat_dtype, const float* w_fc, const float* b_fc, float* logits_ws,
                              float* logits_up, int B, int K, int C, int h, int w, int H, int W, void* stream);
HK_API size_t hk_head_bwd_workspace_bytes(int B, int K, int C, int h, int w);
HK_API int hk_head_bwd(const float* g_up, const void* feat, const float* w_fc, float* dlogits_ws, void* dfeat, float* dw_fc,
                       float* db_fc, int accumulate, int B, int K, int C, int h, int w, int H, int W, void* ws, size_t ws_bytes,
                       void* stream);

/* ---- training-batch augmentation ----
 * Replaces the domain-randomisation pipeline of src/dataset.py:18-31 (imgaug, commented out there) and, for warped labels, the label
 * clipping of :63-66: a random affine warp with the (x, y) pixel-index labels moved by the same map, then photometric jitter.  The
 * caller draws per image `tries` candidate geometries A(p) = s*R(theta)*(p - ctr) + ctr + t, ctr = ((W-1)/2, (H-1)/2), as 2x3 row-major
 * fp32 matrices: fwd (B, tries, 2, 3) maps labels, inv (B, tries, 2, 3) = A^-1 maps output pixels to input pixels.
 *   hk_augment_pick   : pick (B) int32 = the first candidate under which all K labels of image b lie in [0, W-1] x [0, H-1], or -1
 *                       (identity geometry) if none does; uv_out (B,K,2) = the labels under that candidate (x' = (m0*x + m1*y) + m2, one
 *                       fp32 rounding per operation), or uv unchanged for -1.  uv_out must not overlap uv (HK_ERR_BAD_ARG).
 *   hk_augment_images : in, out (B,3,H,W) fp32 NCHW, distinct and non-overlapping (HK_ERR_BAD_ARG otherwise).
 *                       out(p) = bilinear(in, inv[b, pick[b]](p)) with pixel centres at integer coordinates and zero outside the image
 *                       (grid_sample(align_corners=True, padding_mode="zeros")); then per channel, in fp32 and in this order:
 *                       v = (v - 0.5)*c + 0.5 + beta; v *= g_ch; v += noise_std*n; v = clamp(v, 0, 1), with photo (B,5) = (c, beta,
 *                       g0, g1, g2).  n ~ N(0,1) from Philox4x32-10 with the 64-bit `key` (low word first) and counter (x/4, y, channel, b),
 *                       one Box-Muller output of four normals per 4 horizontally adjacent pixels.  With identity geometry, c = 1,
 *                       beta = 0, g = 1 and noise_std = 0 an image with values in [0, 1] is returned bit for bit.
 * Both are capturable (no allocation, no synchronisation). */
#define HK_AUGMENT_MAX_TRIES 16
HK_API int hk_augment_pick(const float* fwd, int B, int tries, int K, int H, int W, const float* uv, float* uv_out, int32_t* pick,
                           void* stream);
HK_API int hk_augment_images(const float* in, float* out, int B, int H, int W, const float* inv, int tries, const int32_t* pick,
                             const float* photo, float noise_std, uint64_t key, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* HULK_SM100_H_ */

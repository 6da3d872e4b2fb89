/*
 * libudh.so — C ABI of the B200-native unsupervised-deep-homography hot path.
 *
 * The reference (tynguyen/unsupervisedDeepHomographyRAL2018) is a pure-Python TF1 graph and has no FFI of its
 * own; each entry point below replaces the group of TF ops cited next to it (file:line under /root/reference/code).
 * The Python mirror of the reference API (HomographyModel, transformer, the CLI) sits on top of this ABI and is
 * the binding a maintainer would use (INTEGRATION.md).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller unless the name says `host`; the library never
 *     allocates device memory — scratch is passed in as a workspace sized by the *_workspace_bytes query;
 *   - tensors are dense NHWC fp32 (the reference's layout and dtype); indices are int32;
 *   - every call is asynchronous on the `stream` argument (a cudaStream_t passed as void*) and re-entrant across
 *     streams; no exceptions cross the boundary: return 0 on success, a negative UDH_E* code otherwise and
 *     udh_last_error() gives the message (thread-local);
 *   - there is no CPU fallback: without a CUDA device every compute entry point returns UDH_ECUDA.
 */
#ifndef UDH_H_
#define UDH_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define UDH_OK 0
#define UDH_EINVAL (-1) /* bad argument (shape, alignment, null pointer)   */
#define UDH_ECUDA (-2)  /* CUDA runtime / launch error                      */
#define UDH_ENOSUP (-3) /* configuration not supported by this build        */
#define UDH_EWS (-4)    /* workspace too small                              */

/* numeric mode of the regressor (udh_cnn_*).  FP32: CUDA-core fp32 everywhere — the parity mode.
 * BF16: tcgen05 bf16 tensor-core tiles with fp32 TMEM accumulation, fp32 master weights — the throughput mode. */
#define UDH_NUMERIC_FP32 0
#define UDH_NUMERIC_BF16 1
/* BF16X3: the same tcgen05 tiles with ERROR-COMPENSATED operands: every fp32 activation / gradient / weight travels as two
 * 16-bit limbs (x = hi + lo) and every product is evaluated as lo.hi + hi.hi + hi.lo with fp32 TMEM accumulation, so the
 * regressor reproduces fp32 arithmetic to ~1e-5 relative (the tensor-core parity mode; three MMA passes per product). */
#define UDH_NUMERIC_BF16X3 2

/* photometric loss selector for udh_warp_loss_bwd (reference --loss_type, homography_CNN_synthetic.py:51) */
#define UDH_LOSS_L1 0        /* homography_model.py:328 */
#define UDH_LOSS_REC 1       /* homography_model.py:303 */
#define UDH_LOSS_L1_SMOOTH 2 /* homography_model.py:136-139,340 */
#define UDH_LOSS_NCC 3       /* homography_model.py:161-166,351 */
#define UDH_LOSS_CUSTOM 4    /* per-pixel d loss / d pred supplied by the caller (ssim_loss: udh_ssim_bwd) */

/* slots of the `sums` accumulator (double[UDH_NSUMS]) filled by udh_warp_loss_fwd / udh_ssim_fwd */
#define UDH_SUM_ABS 0   /* sum |pred - I2|            */
#define UDH_SUM_SQ 1    /* sum (pred - I2)^2          */
#define UDH_SUM_HUBER 2 /* sum huber_1(pred - I2)     */
#define UDH_SUM_XY 3    /* sum pred * I2              */
#define UDH_SUM_XX 4    /* sum pred^2                 */
#define UDH_SUM_YY 5    /* sum I2^2                   */
#define UDH_SUM_SSIM 6  /* sum clip((1-SSIM)/2,0,1)   */
#define UDH_NSUMS 8

/* slots of the float[UDH_NLOSSES] written by udh_photo_losses_finalize (homography_model.py:291-296) */
#define UDH_L_REC 0
#define UDH_L_SSIM 1
#define UDH_L_L1 2
#define UDH_L_L1_SMOOTH 3
#define UDH_L_NCC 4
#define UDH_NLOSSES 8

/* slots of the float[UDH_NMETRICS] written by udh_h4p_loss (homography_model.py:274-281,288) */
#define UDH_M_H_LOSS 0         /* sqrt(mean_{B x 8} (pred-gt)^2)                       */
#define UDH_M_BOUNDED_H_LOSS 1 /* mean_b of per-sample RMSE, identity-bounded          */
#define UDH_M_NUM_FAIL 2       /* #samples with RMSE >= identity RMSE                  */
#define UDH_M_ACE 3            /* mean Euclidean corner distance (literature's metric) */
#define UDH_NMETRICS 4

int udh_version(void);
const char* udh_last_error(void);
/* 1 when a CUDA device is usable from this process, 0 otherwise (never throws). */
int udh_device_available(void);

/* ---- Row D: HomographyModel.solve_DLT (homography_model.py:169-250, utils/utils.py:11-122) ------------------
 * pts1[B,8] (x,y)x[TL,TR,BR,BL], h4p[B,8] -> H[B,9] row-major, h33 = 1, mapping pts1 -> pts1+h4p in pixels.
 * One warp per sample: 8x8 [A|b] in registers, LU with partial pivoting through warp shuffles
 * (replaces the 8 tf.matmul with Aux_M*, stack/transpose and tf.matrix_solve at :223-242). */
int udh_dlt_fwd(const float* pts1, const float* h4p, float* H, int B, void* stream);
/* TF autodiff of the above: dH[B,9] -> dh4p[B,8] (solve A^T lambda = dH[0:8]; dA = -lambda h^T, db = lambda). */
int udh_dlt_bwd(const float* pts1, const float* h4p, const float* H, const float* dH, float* dh4p, int B, void* stream);

/* ---- Row W+L: HomographyModel.transform + photometric losses ----------------------------------------------
 * (homography_model.py:252-269,291-296,328; utils/tf_spatial_transformer.py:76-247)
 * Fused: H' = M^-1 H M, homography warp of I[B,img_h,img_w,C] (C in {1,3}), channel mean, and ONLY the window
 * the reference gathers with patch_indices (a pw x ph rectangle whose first index patch_indices[b*idx_stride]
 * = y0*img_w + x0 gives its origin; patch_indices == NULL means origin (0,0)), compared with I2[B,ph,pw].
 * pred (nullable) receives pred_I2[B,ph,pw]; sums (double[UDH_NSUMS], caller-zeroed) accumulates the
 * reductions every photometric loss needs.  pw must be a multiple of 4. */
int udh_warp_loss_fwd(const float* I, int C, int img_h, int img_w, const float* H, const float* I2,
                      const int32_t* patch_indices, int64_t idx_stride, int pw, int ph, float* pred, double* sums,
                      int B, void* stream);
/* all_sums = 0: accumulate sums[UDH_SUM_ABS] only (what l1_loss needs) — the variant BASELINE configs[3] measures. */
int udh_warp_loss_fwd_ex(const float* I, int C, int img_h, int img_w, const float* H, const float* I2,
                         const int32_t* patch_indices, int64_t idx_stride, int pw, int ph, float* pred, double* sums,
                         int all_sums, int B, void* stream);
/* d loss / d H [B,9] for loss_type in UDH_LOSS_*; `sums` is the forward accumulator (needed by REC),
 * upstream multiplies the gradient (1.0 for a plain backward).  Recomputes the warp; no image-sized
 * intermediates.  scratch: float[B*9], caller-provided. */
int udh_warp_loss_bwd(const float* I, int C, int img_h, int img_w, const float* H, const float* I2,
                      const int32_t* patch_indices, int64_t idx_stride, int pw, int ph, int loss_type,
                      const double* sums, float upstream, float* dH, float* scratch, int B, void* stream);
/* same, with the per-pixel upstream gradient dpred[B,ph,pw] for UDH_LOSS_CUSTOM (NULL otherwise) */
int udh_warp_loss_bwd_ex(const float* I, int C, int img_h, int img_w, const float* H, const float* I2,
                         const int32_t* patch_indices, int64_t idx_stride, int pw, int ph, int loss_type,
                         const double* sums, const float* dpred, float upstream, float* dH, float* scratch, int B, void* stream);
/* d mean(clip((1-SSIM)/2,0,1)) / d pred -> dpred[B,ph,pw] (homography_model.py:141-158,316); feed to udh_warp_loss_bwd_ex. */
int udh_ssim_bwd(const float* pred, const float* I2, int pw, int ph, float* dpred, int B, void* stream);
/* SSIM diagnostic (homography_model.py:141-158): adds sum over the VALID 3x3 grid into sums[UDH_SUM_SSIM]. */
int udh_ssim_fwd(const float* pred, const float* I2, int pw, int ph, double* sums, int B, void* stream);
/* losses[UDH_NLOSSES] from sums; n = B*ph*pw, n_ssim = B*(ph-2)*(pw-2). */
int udh_photo_losses_finalize(const double* sums, double n, double n_ssim, float* losses, void* stream);

/* ---- the `transformer` operator (utils/tf_spatial_transformer.py:18,249-251) --------------------------------
 * U[B,H,W,C], theta[B,9] (normalised homography H'), -> out[B,out_h,out_w,C]; reference semantics including
 * the linspace grid, the t_s epsilon rule and clip-then-weight bilinear sampling. */
int udh_transformer_fwd(const float* U, const float* theta, float* out, int B, int H, int W, int C, int out_h,
                        int out_w, void* stream);

/* ---- Row L (h4p part): h_loss and the test-mode metrics (homography_model.py:274-281,288) -------------------
 * metrics: float[UDH_NMETRICS]; per_sample (nullable): float[B] batch_h_loss; dpred (nullable): d h_loss / d pred. */
int udh_h4p_loss(const float* pred, const float* gt, int B, float* metrics, float* per_sample, float* dpred,
                 void* stream);

/* ---- Row C: HomographyModel._vgg (homography_model.py:88-133) -----------------------------------------------
 * params / grads: the flat fp32 buffer laid out by udh_param_offset (TF-Slim checkpoint shapes: HWIO conv
 * kernels, [in,out] fc kernels, NHWC flatten).  I1, I2: [B,P,P] gray patches (the two channels of model_input,
 * homography_model.py:359, read in place — no concat copy).  train != 0 enables dropout(keep 0.5) after conv4_2
 * and fc1 with masks drawn from `seed` (kept in the workspace for the backward and readable with
 * udh_cnn_dropout_masks).  The workspace keeps the activations between fwd and bwd. */
size_t udh_cnn_workspace_bytes(int B, int P, int numeric_mode);
/* call once after allocating the workspace (zeroes the borders of the padded bf16 streams of UDH_NUMERIC_BF16). */
int udh_cnn_workspace_init(void* ws, size_t ws_bytes, int B, int P, int numeric_mode, void* stream);
int udh_cnn_fwd(const float* params, const float* I1, const float* I2, float* h4p, void* ws, size_t ws_bytes, int B,
                int P, int train, uint64_t seed, int numeric_mode, void* stream);
/* flags: UDH_FWD_FC1_MIRROR_CURRENT — the workspace's bf16 copy of fc1's weights already matches `params`
 * (udh_adam_step_mirror wrote it, or a previous forward did and params are unchanged): skip the conversion. */
#define UDH_FWD_FC1_MIRROR_CURRENT 1
int udh_cnn_fwd_ex(const float* params, const float* I1, const float* I2, float* h4p, void* ws, size_t ws_bytes, int B,
                   int P, int train, uint64_t seed, int numeric_mode, int flags, void* stream);
/* dh4p[B,8] -> grads (ACCUMULATED into the flat buffer: caller zeroes it once per step). */
int udh_cnn_bwd(const float* params, const float* I1, const float* I2, const float* dh4p, float* grads, void* ws,
                size_t ws_bytes, int B, int P, int train, int numeric_mode, void* stream);
/* The same backward in two halves, so the caller can start the allreduce of the fully connected gradients (98 % of the
 * bytes: fc1 is 33.5 M of the 34.2 M parameters) while the convolution backward is still running:
 * UDH_BWD_HEAD = fc2 + fc1 (leaves d(conv4_2 pre-activation) in the workspace), UDH_BWD_CONVS = the conv stack. */
#define UDH_BWD_ALL 0
#define UDH_BWD_HEAD 1
#define UDH_BWD_CONVS 2
int udh_cnn_bwd_phase(const float* params, const float* I1, const float* I2, const float* dh4p, float* grads, void* ws,
                      size_t ws_bytes, int B, int P, int train, int numeric_mode, int phase, void* stream);
/* device pointers (inside ws) of the uint8 keep-masks of the last train-mode forward: [B,(P/8)^2*128] and [B,1024]. */
int udh_cnn_dropout_masks(void* ws, size_t ws_bytes, int B, int P, int numeric_mode, const uint8_t** mask_conv4,
                          const uint8_t** mask_fc1);
/* device pointer (inside ws) of a saved activation, for tests: layer 0..7 = conv outputs, 8..10 = pool1..3,
 * 11 = fc1 (post-ReLU, pre-dropout).  *numel receives the element count. */
int udh_cnn_activation(void* ws, size_t ws_bytes, int B, int P, int numeric_mode, int layer, const float** ptr,
                       size_t* numel);
/* layout of the flat parameter buffer: tensor index 0..19 = (conv w, conv b) x 8, fc1 w, fc1 b, fc2 w, fc2 b. */
int udh_param_offset(int P, int tensor, size_t* offset_floats, size_t* numel);
size_t udh_param_total_floats(int P);

/* ---- Row O: TF-1 Adam (homography_CNN_synthetic.py:183,278) --------------------------------------------------
 * g' = g * grad_scale (1/world_size folds get_average_grads, utils/utils.py:380-403, into the update);
 * m = b1 m + (1-b1) g'; v = b2 v + (1-b2) g'^2; p -= alpha_t * m / (sqrt(v) + eps), alpha_t = lr_t*sqrt(1-b2^t)/(1-b1^t)
 * computed by the caller (t is 1-based).  If zero_grad != 0 the gradient buffer is cleared in the same pass. */
int udh_adam_step(float* p, float* g, float* m, float* v, size_t n, float alpha_t, float beta1, float beta2,
                  float eps, float grad_scale, int zero_grad, void* stream);
/* Same update, fused with the refresh of a bf16 weight mirror (UDH_NUMERIC_BF16): the updated parameters of the float
 * range [mirror_begin, mirror_begin + mirror_count) are also written, rounded to bf16, to `mirror`; with
 * mirror_keep_grad != 0 the gradient of that range is not cleared (its producer stores rather than accumulates).
 * udh_cnn_fc1_mirror names the range and the buffer for fc1's weights; a forward pass that follows may then be given
 * UDH_FWD_FC1_MIRROR_CURRENT and skips its own fp32 -> bf16 conversion of the 128 MB tensor. */
int udh_adam_step_mirror(float* p, float* g, float* m, float* v, size_t n, float alpha_t, float beta1, float beta2,
                         float eps, float grad_scale, int zero_grad, void* mirror, size_t mirror_begin, size_t mirror_count,
                         int mirror_keep_grad, void* stream);
/* mirror_limbs = 2 (UDH_NUMERIC_BF16X3): the mirror holds two 16-bit planes of mirror_count elements each, hi then lo,
 * with p = hi + lo; mirror_limbs = 1 is udh_adam_step_mirror. */
int udh_adam_step_mirror_ex(float* p, float* g, float* m, float* v, size_t n, float alpha_t, float beta1, float beta2,
                            float eps, float grad_scale, int zero_grad, void* mirror, size_t mirror_begin, size_t mirror_count,
                            int mirror_keep_grad, int mirror_limbs, void* stream);
/* bf16 copy of fc1's weights inside the workspace: *mirror (NULL in UDH_NUMERIC_FP32), its float range in the flat
 * parameter buffer, and whether fc1's weight gradient is stored (1) or accumulated (0) by the backward pass. */
int udh_cnn_fc1_mirror(void* ws, size_t ws_bytes, int B, int P, int numeric_mode, void** mirror, size_t* param_begin,
                       size_t* count, int* grad_is_stored);

/* ---- one call per step -------------------------------------------------------------------------------------------
 * The reference runs a step as ONE sess.run([apply_grad_opt, losses...]) (homography_CNN_synthetic.py:335-345).
 * udh_step_forward_backward enqueues regressor forward, h4p losses (:274-288), DLT (:169-250), fused warp + all
 * photometric diagnostics (:252-269,291-296) and the backward of the selected loss on `stream`; the caller then runs the
 * gradient allreduce (N > 1) and udh_adam_step.  Every output buffer is caller-owned and reused step after step. */
#define UDH_STEP_ALL 0      /* forward + full backward                                                         */
#define UDH_STEP_FWD_HEAD 1 /* forward + backward of the fully connected head (then allreduce fc grads ...)    */
#define UDH_STEP_CONVS 2    /* ... while this runs: backward of the conv stack                                 */
#define UDH_STEP_FWD_ONLY 3 /* evaluation: forward, losses, metrics                                            */
#define UDH_STEP_LOSS_H 0
#define UDH_STEP_LOSS_L1 1
#define UDH_STEP_LOSS_REC 2
#define UDH_STEP_LOSS_L1_SMOOTH 3
#define UDH_STEP_LOSS_NCC 4
#define UDH_STEP_LOSS_SSIM 5
typedef struct {
  int B, P, img_h, img_w, C;      /* batch, patch size, image size, channels of I_aug (1 or 3) */
  int numeric_mode, loss_type, train;
  uint64_t seed;                  /* dropout seed of this step */
  const float* params; float* grads; void* ws; size_t ws_bytes;
  const float *I1, *I2, *I_aug, *pts1, *gt;   /* gt may be NULL (no h_loss / metrics) */
  const int32_t* patch_indices; int64_t idx_stride;
  float *h4p, *H, *pred_I2;       /* [B,8], [B,9], [B,P,P] (pred_I2 may be NULL: then no SSIM) */
  float *dh4p, *dH, *scratch;     /* [B,8], [B,9], [B,9] */
  float* dpred_map;               /* [B,P,P] scratch, only for UDH_STEP_LOSS_SSIM */
  double* sums;                   /* [UDH_NSUMS] */
  float *photo_losses, *h4p_metrics, *per_sample;   /* [UDH_NLOSSES], [UDH_NMETRICS], [B] or NULL */
  int fwd_flags;                  /* UDH_FWD_* */
} udh_step_args;
int udh_step_forward_backward(const udh_step_args* args, int phase, void* stream);

/* ---- device-side input pipeline (dataloader.py:99-100,172-177,203-227; SURVEY 8f item 1) ------------------------
 * I, I_prime: uint8 [B,img_h,img_w,3] decoded images; pts1 [B,8].  Writes the post-dataloader tensors the step
 * consumes: I_aug fp32 [B,img_h,img_w,3] (normalised with I's statistics), gray patches I1, I2 fp32 [B,P,P] at
 * (x0,y0) = pts1[0:2], and patch_origin[B] = y0*img_w + x0 (the first patch index of each sample). */
int udh_prep_inputs_u8(const uint8_t* I, const uint8_t* I_prime, const float* pts1, float* I_aug, float* I1, float* I2,
                       int32_t* patch_origin, int B, int img_h, int img_w, int P, void* stream);

/* Same pipeline with the reference's photometric augmentation (dataloader.py:163-169,323-375) fused in, and a GRAY warp
 * source: aug (nullable) = [B,11] {on, gamma, brightness, colour R/G/B for I, then the same five for I'} — joint
 * augmentation (train) passes the same five numbers twice, disjoint (test) two draws; gamma acts on the raw 0..255 values.
 * Outputs: I_gray [B,img_h,img_w] = channel mean of the normalised (augmented) I — the warp's channel mean commutes with
 * its linear sampling, so the warp kernel can read this plane with C = 1 (a third of the bytes); I_aug3 (nullable) the
 * 3-channel tensor of the reference contract; I1_aug, I2_aug [B,P,P] the CNN input / L1 target; I1, I2 (nullable, together)
 * the un-augmented patches (summaries only in the reference); patch_origin [B] (nullable). */
int udh_prep_inputs_u8_ex(const uint8_t* I, const uint8_t* I_prime, const float* pts1, const float* aug, float* I_gray, float* I_aug3,
                          float* I1, float* I2, float* I1_aug, float* I2_aug, int32_t* patch_origin, int B, int img_h, int img_w,
                          int P, void* stream);
/* ---- on-device synthetic pairs (utils/gen_synthetic_data.py:40-68; MS-COCO is not available offline) ---------------
 * udh_synth_scene_u8: seeded multi-octave texture I [B,img_h,img_w,3] uint8, patch corners pts1 [B,8] with
 * x0 in [rho, W-rho-P], y0 in [rho, Hh-rho-P] (:42-50) and integer corner perturbations gt [B,8] in [-rho, rho] (:53).
 * udh_dlt_fwd(pts1, gt) then gives H_gt (:56) and udh_warp_image_u8 the second image I' = uint8(warp(I, H_gt)) (:63-64,
 * numpy_spatial_transformer.py:131-146). */
int udh_synth_scene_u8(uint8_t* I, float* pts1, float* gt, int B, int img_h, int img_w, int P, int rho, uint64_t seed, void* stream);
int udh_warp_image_u8(const uint8_t* U, const float* H, uint8_t* out, int B, int img_h, int img_w, void* stream);

/* ---- instrumentation read by bench.py -------------------------------------------------------------------------
 * udh_launch_count: kernels this library has launched in this process (monotonic).
 * udh_prof_*: when enabled, every tagged phase is bracketed by CUDA events recorded on the launching stream;
 * udh_prof_read synchronises on them and returns the accumulated device time and the number of brackets.
 * Must be off while a stream is being captured into a CUDA graph. */
unsigned long long udh_launch_count(void);
/* Leave n SMs free in the persistent one-CTA-per-SM backward kernels of conv4_1 / conv4_2 (process-wide): the launches that
 * run while the fully connected gradients are being all-reduced on the communication stream.  A persistent kernel with a
 * static item schedule that finds n of its SMs taken by the NCCL kernel runs those CTAs in a second wave (2x its time); with
 * <= 2 items per CTA these four launches lose nothing by starting on (SMs - n) CTAs, so reserving NCCL's CTA count here
 * removes the collision. */
int udh_set_sm_reserve_top(int n);
/* A point inside the conv backward for a second stream to start at: with layer = 7..0 (conv4_2..conv1_1; -1 = off) every
 * conv backward that follows records an internal event on its stream right before the backward kernels of that layer, and
 * udh_bwd_marker_wait(stream) makes `stream` wait for the most recent record (no-op before the first).  The engine uses it
 * to run the fused gradient-reduce / Adam / weight-multicast kernel under the wide 64-channel layers' backward (tensor-bound)
 * rather than under conv4_x / conv3_x (short, latency-bound launches that a co-running streaming kernel slows 3-5x). */
int udh_set_bwd_marker(int layer);
int udh_bwd_marker_wait(void* stream);

/* Row G + the optimiser for ONE rank's shard of a replicated tensor, over NVSwitch multicast memory (csrc/dp_update.cu):
 * replaces, for fc1's weights, code/utils/utils.py:380-403 (gradient mean over the towers) followed by
 * code/homography_CNN_synthetic.py:277-284 (apply_gradients).  mc_grads / mc_params are the MULTICAST addresses of the
 * flat gradient / parameter buffers (symmetric allocations bound to one multicast object; the same float offsets as the
 * local buffers), params / adam_m / adam_v the rank's local flat buffers.  For the floats [shard_begin, shard_begin +
 * shard_count): g = sum over ranks (multimem.ld_reduce) * grad_scale; TF-1 Adam on the local m, v; the new fp32 value is
 * stored to every replica (multimem.st), and so are its tensor-core limbs when mc_mirror (multicast address of the fc1
 * weight mirror, udh_cnn_fc1_mirror; planes of mirror_count elements, hi then lo) is given: mirror_limbs = 1 (bf16) or 2
 * (bf16x3), 0 with mc_mirror == NULL.  The gradient itself is left as is (fc1's weight gradient is stored, not accumulated).
 * The caller orders the ranks: every rank's gradient must be final before any rank launches this, and every rank's launch
 * must have completed before any replica is read (two symmetric-memory barriers on the stream, engine.py).  grid = CTAs of
 * 512 threads (0 = one per SM). */
int udh_dp_shard_update(const void* mc_grads, const float* params, void* mc_params, float* adam_m, float* adam_v,
                        void* mc_mirror, size_t shard_begin, size_t shard_count, size_t mirror_begin, size_t mirror_count,
                        int mirror_limbs, float alpha_t, float beta1, float beta2, float eps, float grad_scale, int grid,
                        void* stream);
/* HOST function (no device work): CRC-32C (Castagnoli) of n bytes, continuing from `crc` (0 to start) — the checksum of
 * TensorFlow checkpoint V2 bundles (tf.train.Saver, code/homography_CNN_synthetic.py:303,360), which tf_checkpoint.py writes
 * and verifies.  Hardware crc32 instruction when the CPU has SSE4.2, slicing-by-8 otherwise. */
uint32_t udh_crc32c(const void* data, size_t n, uint32_t crc);
int udh_prof_enable(int on);
int udh_prof_reset(void);
int udh_prof_num_tags(void);
const char* udh_prof_tag_name(int tag);
int udh_prof_read(int tag, float* total_ms, int* count);

/* ---- debug / test entry points of the tensor-core path ---------------------------------------------------------
 * (the hardware probes of the TMA / tcgen05 conventions live in their own library: include/udh_probe.h, libudh_probe.so)
 * udh_debug_tc_conv: ONE tcgen05 3x3 convolution on fp32 NHWC tensors (pads + casts to bf16 internally), so tests can
 * compare the tensor-core kernel with a reference convolution layer by layer; dgrad != 0 runs the mirrored kernel. */
size_t udh_debug_tc_conv_scratch_bytes(int B, int H, int W, int cin, int cout);
int udh_debug_tc_conv(const float* x, const float* w, const float* bias, float* out, void* scratch, int B, int H, int W,
                      int cin, int cout, int relu, int dgrad, void* stream);
/* tensor-core weight gradient of one layer: x [B,H,W,cin], g [B,H,W,cout] fp32 -> dW HWIO, db (both accumulated);
 * scratch sized by udh_debug_tc_conv_scratch_bytes. */
int udh_debug_tc_wgrad(const float* x, const float* g, float* dW, float* db, void* scratch, int B, int H, int W, int cin,
                       int cout, void* stream);
/* UDH_NUMERIC_BF16X3 kernels, one layer at a time on fp32 NHWC tensors (split into limbs internally): 3x3 convolution
 * (forward or mirrored), weight gradient, and conv1_1 (forward when out != NULL, weight gradient when g != NULL). */
/* UDH_NUMERIC_BF16X3 workspace: write fp32 copies (hi + lo) of the saved conv / pool activations into the slots
 * udh_cnn_activation names; *fp32_region_bytes (nullable) = size of the leading part of the workspace whose layout is common
 * to all numeric modes (activations, dropout masks, fc buffers), so a test can run the fp32 backward on this forward state. */
int udh_debug_x3_materialize(void* ws, size_t ws_bytes, int B, int P, size_t* fp32_region_bytes, void* stream);
/* conv1_2 of the UDH_NUMERIC_BF16X3 mode runs on row tiles by default (forward fused with pool1: the full-resolution
 * activation is never stored; row-tile dgrad).  on = 0 selects the generic flattened-tile kernels + the separate pool kernel —
 * tests compare the two paths and need the un-fused one to read conv1_2's activation. */
int udh_debug_x3_set_rows(int on);
size_t udh_debug_x3_scratch_bytes(int B, int H, int W, int cin, int cout);
int udh_debug_x3_conv(const float* x, const float* w, const float* bias, float* out, void* scratch, int B, int H, int W, int cin,
                      int cout, int relu, int dgrad, void* stream);
int udh_debug_x3_wgrad(const float* x, const float* g, float* dW, float* db, void* scratch, int B, int H, int W, int cin, int cout,
                       void* stream);
int udh_debug_x3_conv1(const float* I1, const float* I2, const float* w, const float* bias, float* out, const float* g, float* dW,
                       float* db, void* scratch, int B, int H, int W, void* stream);
/* fused conv (64 -> 64 channels, W == 128) + bias + ReLU + 2x2 max-pool (conv1_2 + pool1): x [B,H,128,64] ->
 * pooled [B,H/2,64,64] fp32 and routing codes [B,H/2,64,8] uint32 (3 bits per channel, 4 = no gradient). */
int udh_debug_tc_conv_pool(const float* x, const float* w, const float* bias, float* pooled, uint32_t* codes, void* scratch,
                           int B, int H, int W, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* UDH_H_ */

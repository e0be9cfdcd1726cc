/*
 * argus_b200 — C ABI of libargus_b200.so: the B200 (sm_100a) implementation of the training / inference hot path
 * of pculbertson/argus.
 *
 * The reference is pure Python and has no FFI of its own; each entry point below names the reference call site it
 * replaces (paths relative to the reference tree). INTEGRATION.md shows the ctypes stub a maintainer of the
 * reference would add.
 *
 * Conventions
 *   - plain C types only: device pointers are `void*` / `float*`, sizes are `int` / `int64_t`, streams are passed
 *     as `void*` holding a `cudaStream_t` (NULL = legacy default stream);
 *   - every function returns 0 on success and non-zero on failure; `argus_last_error_string()` returns the
 *     thread-local message of the last failure; C++ exceptions never cross the boundary;
 *   - all work is enqueued asynchronously on the caller's stream; the caller owns every buffer it passes in;
 *   - there is NO CPU fallback: a missing GPU or a non-sm_100 GPU is an error;
 *   - activations are NHWC bf16, convolution weights are [Cout][kh][kw][Cin] bf16 ("packed" layout) unless noted;
 *     spatial sizes must be powers of two and channel counts multiples of 64.
 */
#ifndef ARGUS_B200_H_
#define ARGUS_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- library ------------------------------------------------------------------------------------------- */
const char* argus_last_error_string(void);
int argus_version(void);
/* Fails unless the current CUDA device is compute capability 10.x. */
int argus_require_device(void);
/* Launch accounting: number of kernels this library has launched since it was loaded. */
int64_t argus_launch_count(void);
/* Optional per-kernel-family timing with CUDA events on the launching stream (bench.py's roofline figures).
 * argus_profile_report synchronises the recorded events and writes a JSON object
 * {family: {launches, ms, flops, bytes}} (algorithmic FLOPs / bytes) into `json`. */
int argus_profile_enable(int on);
int argus_profile_report(char* json, int cap);

/* ---- convolution primitives (torch.nn.Conv2d / nn.Linear inside torchvision resnet50, called from
 *      argus/models.py:84; cuDNN / cuBLAS in the reference) ------------------------------------------------- */
/* kind 0: k in {1,3}, stride in {1,2}, pad = k/2.  kind 1: the 7x7/2 stem on the space-to-depth input produced by
 * argus_pack_input (x is [N][H/2][W/2+4][16] bf16, w is the stem weight repacked to [64][256] by
 * argus_pack_stem_weight); N, H, W always describe the conv input image. */
int argus_conv2d_forward(const void* x, const void* w, void* y, int N, int H, int W, int Cin, int Cout, int k,
                         int stride, int kind, const float* scale, const float* shift, const void* residual, int relu,
                         float* stat_partial, int stat_slot_capacity, void* stream);
/* Train-mode BN statistics are reduced deterministically: stat_partial is a zero-filled [slots][2][Cout] fp32 buffer
 * (per-CTA partial sums / sums of squares of the stored bf16 outputs) that argus_bn_finalize adds in slot order.
 * argus_conv2d_stat_slots returns an upper bound on the slots a forward launch of this shape writes. */
int argus_conv2d_stat_slots(int N, int H, int W, int Cin, int Cout, int k, int stride, int kind, int* slots);
/* dx = conv_transpose(dy, w) (+ residual). For stride 2 the caller zero-fills dx first when k == 1. */
int argus_conv2d_dgrad(const void* dy, const void* w, void* dx, int N, int H, int W, int Cin, int Cout, int k,
                       int stride, const void* residual, void* stream);
/* stride-1 dgrad whose residual is gated by a ReLU bit mask: dx = conv_transpose(dy, w) + residual * bit, with
 * residual_bits = the [rows][Cin/8] byte mask written by argus_bn_apply_bits for the tensor dx is the gradient of
 * (the identity branch of a bottleneck: the masked gradient is never materialised). */
int argus_conv2d_dgrad_bits(const void* dy, const void* w, void* dx, int N, int H, int W, int Cin, int Cout, int k,
                            const void* residual, const void* residual_bits, void* stream);
/* 1x1 dgrad with the extras the algebraic BN backward uses. concat_a (nullable): a second activation (N,H,W,
 * concat_channels) on the conv INPUT grid whose channels extend K; w is then the row-major [(Cout + concat_channels)][Cin]
 * stacked matrix: dx = [dy | concat_a] * w + bias (bias nullable, per Cin). out_bits (nullable): [rows][Cin/8] ReLU mask
 * applied to the stored result. stat_partial (nullable): zero-filled [slots][2][Cin] per-CTA sums / sums of squares of
 * the stored result (argus_conv2d_stat_slots of the equivalent forward shape bounds the slots). */
int argus_conv2d_dgrad_ex(const void* dy, const void* w, void* dx, int N, int H, int W, int Cin, int Cout, int stride,
                          const void* concat_a, int concat_channels, const float* bias, const void* residual,
                          const void* out_bits, float* stat_partial, int stat_slot_capacity, void* stream);
/* Forward convolution with every field of the epilogue: y = [relu](acc * scale + shift [+ residual * res_scale +
 * res_shift]); scale, shift, residual, res_scale / res_shift (both or neither) are nullable. relu_bits_out (nullable,
 * needs relu): [rows][Cout/8] bytes, bit = (value before the ReLU > 0). stat_partial as for argus_conv2d_forward.
 * early_trigger: let the next kernel of the stream start its prologue while this one runs (the eval-mode chain). */
int argus_conv2d_forward_full(const void* x, const void* w, void* y, int N, int H, int W, int Cin, int Cout, int k,
                              int stride, int kind, const float* scale, const float* shift, const void* residual,
                              const float* res_scale, const float* res_shift, int relu, void* relu_bits_out,
                              float* stat_partial, int stat_slot_capacity, int early_trigger, void* stream);
/* Stride-1 dgrad with the batch-norm backward reduction fused into its epilogue: g = conv_transpose(dy, w) [+ bias] is
 * stored masked by (bn_raw * bn_scale + bn_shift > 0), and the zero-filled stat_partial [slots][2][Cin] receives
 * sum(g) and sum(g * bn_raw) of the stored values. k = 1 or 3; with concat_a (k = 1 only) the K-concatenated form of
 * argus_conv2d_dgrad_ex, where w is the stacked [(Cout + concat_channels)][Cin] matrix and bias is nullable. */
int argus_conv2d_dgrad_bnred(const void* dy, const void* w, void* dx, int N, int H, int W, int Cin, int Cout, int k,
                             int stride, const void* concat_a, int concat_channels, const float* bias,
                             const void* bn_raw, const float* bn_scale, const float* bn_shift, float* stat_partial,
                             int stat_slot_capacity, void* stream);
/* Plans a convolution the way the calls above do and reports, without launching, what each of its launches would run.
 * launch: 0 forward (kind as for argus_conv2d_forward), 1 dgrad, 2 K-concatenated 1x1 dgrad (concat_channels).
 * flags: the epilogue fields that are present (ARGUS_EPI_*). Per launch, ARGUS_LAUNCH_INFO_INTS ints go to out:
 * block_n, b_mn, opt (kernel option mask; 31 = the generic kernel), halo, b_resident, halo_stages, num_m_tiles,
 * num_n_tiles, grid, stat_slots. */
#define ARGUS_EPI_SCALE 1
#define ARGUS_EPI_SHIFT 2
#define ARGUS_EPI_RESIDUAL 4
#define ARGUS_EPI_RES_AFFINE 8
#define ARGUS_EPI_RELU 16
#define ARGUS_EPI_RELU_BITS_OUT 32
#define ARGUS_EPI_OUT_BITS 64
#define ARGUS_EPI_RESIDUAL_BITS 128
#define ARGUS_EPI_STATS 256
#define ARGUS_EPI_BN_RAW 512
#define ARGUS_EPI_EARLY_TRIGGER 1024
#define ARGUS_LAUNCH_INFO_INTS 10
int argus_conv2d_launch_info(int launch, int N, int H, int W, int Cin, int Cout, int k, int stride, int kind,
                             int concat_channels, int flags, int* out, int cap, int* n_launches);
/* Records the kernel instance of every convolution launch while on (turning it on clears the record); get copies up to
 * cap keys of five ints (block_n, b_mn, opt, halo, b_resident) and sets *n to the number recorded. */
int argus_conv_instances_record(int on);
int argus_conv_instances_get(int* keys, int cap, int* n);
/* Every kernel instance a convolution launch can run: up to cap keys of three ints (block_n, b_mn, opt); *n = count. */
int argus_conv_instances_all(int* keys, int cap, int* n);
/* g[Cin][Cin] (fp32, +=; the caller zero-fills) = x_s^T x_s over the pixels a 1x1 convolution of this shape reads (its
 * even pixels at stride 2): the Gram matrix from which the statistics of the convolution's output follow. */
int argus_conv2d_gram(const void* x, float* g, int N, int H, int W, int Cin, int Cout, int stride, void* stream);
/* out[C] = column sums (fp32, deterministic) of the bf16 (N, H, W, C) tensor over the pixels a stride-`stride` 1x1
 * convolution reads. C / 8 a power of two, C <= 2048; scratch: 4 * (SM count) * C floats. */
int argus_colsum_pixels(const void* x, int N, int H, int W, int C, int stride, float* scratch, float* out, void* stream);
/* Train-mode batch norm of y = x W^T from G = x^T x [C][C] and s = colsum(x) [C] over `rows` pixels, without y: the
 * folded scale / shift, save_mean / save_invstd and (when running_mean is not null) the running statistics, as
 * argus_bn_finalize computes them. W: bf16 [O][C], O % 16 == 0, C % 32 == 0; scratch: O * C / 16 floats. */
int argus_bn_stats_from_gram(const void* W, const float* G, const float* s, double rows, const float* gamma,
                             const float* beta, float* running_mean, float* running_var, float momentum, float eps,
                             float* scale, float* shift, float* save_mean, float* save_invstd, float* scratch, int O,
                             int C, void* stream);
/* 1x1: dw[(Cout + Cin)][Cin] (fp32, +=): rows < Cout = dy^T x, rows Cout + j = x^T x (Gram matrix of the pixels the
 * convolution reads); Cout % 128 == 0. One launch, the x tiles are loaded once. */
int argus_conv2d_wgrad_gram(const void* dy, const void* x, float* dw, int N, int H, int W, int Cin, int Cout, int stride,
                            void* stream);
/* Backward of y = BN_train(conv1x1(act, w)) given the upstream gradient g (already masked by any ReLU), WITHOUT reading
 * the conv output or materialising its gradient (csrc/bn_algebra.cu): dgamma, dbeta, dw (+=, fp32 [O][C]) and
 * dact = d loss / d act (bf16, (N,H,W,C); zero-filled here for stride 2). w_bf16: the [O][C] bf16 weight the forward
 * used; g_colsum [O]: column sums of g; scale / mean / invstd: the forward's batch-norm constants. O % 256 == 0. */
int argus_conv_bn_backward_algebraic(const void* g, const void* act, const void* w_bf16, const float* g_colsum,
                                     const float* scale, const float* mean, const float* invstd, float* dgamma,
                                     float* dbeta, float* dw, void* dact, int N, int H, int W, int C, int O, int stride,
                                     void* stream);
/* dw[Cout][k*k*Cin] (fp32) += dy^T * im2col(x); the caller zero-fills dw. */
int argus_conv2d_wgrad(const void* dy, const void* x, float* dw, int N, int H, int W, int Cin, int Cout, int k,
                       int stride, int kind, void* stream);
/* Input gradient of the stem (resnet.conv1: 7x7, stride 2, pad 3, 3 -> 64; argus/models.py:84).
 * dy: (N, H/2, W/2, 64) bf16 NHWC; w: the [64][256] packed bf16 stem weight the forward used ([64][p 4][q 4][16],
 * the argus_conv2d_forward kind-1 layout); dx: (N, 3, H, W) fp32 NCHW, overwritten. H, W powers of two >= 32
 * (W <= 1024). fp32 accumulation and output; deterministic. */
int argus_stem_dgrad(const void* dy, const void* w, float* dx, int N, int H, int W, void* stream);

/* ---- batch norm / pooling primitives (torch.nn.BatchNorm2d, ReLU, MaxPool2d(3,2,1), AdaptiveAvgPool2d(1) inside
 *      torchvision resnet50, argus/models.py:84). x, y, dy, dx, res, out: bf16 NHWC viewed as (rows, C); C/8 a
 *      power of two; per-channel vectors fp32. ------------------------------------------------------------------ */
/* train-mode statistics ([slots][2][C] partial sums, see argus_conv2d_forward) -> scale/shift/mean/invstd and
 * running-stat update (running_* nullable) */
int argus_bn_finalize(const float* partial, int slots, double count, const float* gamma, const float* beta,
                      float* running_mean, float* running_var, float momentum, float eps, float* scale, float* shift,
                      float* save_mean, float* save_invstd, int C, void* stream);
/* y = [relu](x*scale+shift [+ res | + res*rscale+rshift]). x, res and y must be 16-byte aligned: a misaligned pointer
 * is an error, reported before anything runs. */
int argus_bn_apply(const void* x, const float* scale, const float* shift, const void* res, const float* rscale,
                   const float* rshift, int relu, void* y, int64_t rows, int C, void* stream);
/* same, and also writes the ReLU mask of the result: relu_bits[rows][C/8] bytes, bit k of byte j = (channel 8j+k of
 * the pre-ReLU value > 0). The backward pass reads these bits instead of the bf16 output (1/16 of the bytes).
 * relu_bits must be 16-byte aligned too. */
int argus_bn_apply_bits(const void* x, const float* scale, const float* shift, const void* res, const float* rscale,
                        const float* rshift, int relu, void* y, void* relu_bits, int64_t rows, int C, void* stream);
/* BN (+ReLU) backward. mask_mode 0: no ReLU; 1: ReLU right after the BN; 2: ReLU after a residual add (mask = out > 0,
 * dy is overwritten with the masked gradient); 3: like 2 but `out` is the relu_bits mask of argus_bn_apply_bits and dy
 * is left untouched. dgamma / dbeta are ADDED to (caller zeroes); dx = d loss / d x. dy, x, out and dx must be 16-byte
 * aligned: a misaligned pointer is an error, reported before dgamma / dbeta are touched. */
int argus_bn_backward(void* dy, const void* x, const void* out, const float* scale, const float* shift,
                      const float* mean, const float* invstd, float* dgamma, float* dbeta, void* dx, int64_t rows,
                      int C, int mask_mode, void* stream);
/* max pooling 3x3/2 pad 1 of relu(x*scale+shift) (scale NULL: x already activated); idx (nullable) = arg-max tap */
int argus_maxpool_forward(const void* x, const float* scale, const float* shift, void* y, void* idx, int N, int H,
                          int W, int C, void* stream);
int argus_maxpool_backward(const void* dy, const void* idx, void* dx, int N, int H, int W, int C, void* stream);
/* Stem tail backward, fused: max-pool backward (pooled gradient dpool (N,H/2,W/2,64) + arg-max bytes idx) -> ReLU mask
 * -> batch-norm backward over the stem convolution output raw (N,H,W,64). Equivalent to argus_maxpool_backward followed
 * by argus_bn_backward(mask_mode 1) without materialising the un-pooled gradient. dgamma / dbeta are ADDED to. */
int argus_stem_pool_bn_backward(const void* dpool, const void* idx, const void* raw, const float* scale,
                                const float* shift, const float* mean, const float* invstd, float* dgamma,
                                float* dbeta, void* dx, int N, int H, int W, int C, void* stream);
int argus_avgpool_forward(const void* x, void* y, int N, int HW, int C, void* stream);
int argus_avgpool_backward(const void* dy, void* dx, int N, int HW, int C, void* stream);

/* ---- fp32 parity-mode primitives (argus_model_set_precision(m, 1) runs the network on these) ---------------------
 * All tensors fp32; activations NHWC; weights and weight gradients in PyTorch's [Cout][Cin][k][k] layout; padding k/2.
 * SIMT implicit GEMMs with fp32 FMA accumulation; split-K partial sums, batch-norm statistics and BN-backward sums are
 * accumulated in fp64 in a fixed order. Same semantics as torch.nn.Conv2d / BatchNorm2d / MaxPool2d(3,2,1). */
int argus_fp32_conv2d_forward(const float* x, const float* w, const float* bias, float* y, int N, int H, int W, int Cin,
                              int Cout, int k, int stride, void* stream);
int argus_fp32_conv2d_dgrad(const float* dy, const float* w, float* dx, int N, int H, int W, int Cin, int Cout, int k,
                            int stride, void* stream);
/* dw += dy^T im2col(x) */
int argus_fp32_conv2d_wgrad(const float* dy, const float* x, float* dw, int N, int H, int W, int Cin, int Cout, int k,
                            int stride, void* stream);
int argus_fp32_bn_train(const float* x, int64_t rows, int C, const float* gamma, const float* beta, float* running_mean,
                        float* running_var, float momentum, float eps, float* scale, float* shift, float* save_mean,
                        float* save_invstd, void* stream);
int argus_fp32_bn_apply(const float* x, const float* scale, const float* shift, const float* res, const float* rscale,
                        const float* rshift, int relu, float* y, int64_t rows, int C, void* stream);
/* g = dy where out > 0 (all of dy when out is NULL); dgamma / dbeta are ADDED to; g_out (nullable) receives g */
int argus_fp32_bn_backward(const float* dy, const float* x, const float* out, const float* scale, const float* mean,
                           const float* invstd, float* dgamma, float* dbeta, float* dx, float* g_out, int64_t rows,
                           int C, void* stream);
int argus_fp32_maxpool_forward(const float* x, float* y, void* idx, int N, int H, int W, int C, void* stream);
int argus_fp32_maxpool_backward(const float* dy, const void* idx, float* dx, int N, int H, int W, int C, void* stream);

/* ---- augmentation (the kornia chain of argus/data.py:41-103 applied at data.py:213-225) ------------------------
 * [RandomErasing x2] -> RandomPlanckianJitter -> ColorJiggle -> RandomGaussianBlur -> RandomMotionBlur ->
 * RandomPlasmaShadow (diamond-square fractal) -> [RandomSaltAndPepperNoise]; bracketed stages are default-off
 * (data.py:35,39). Parameters are a pure function of (seed, step, image index): params is an
 * (n_images, ARGUS_AUG_PARAMS) fp32 table (layout: oracle/augment.py). Colour-jiggle draws are shared by the n_cams views
 * of a pair (same_on_batch=True). H, W: image size (the erasing rectangles are sampled in pixels). */
#define ARGUS_AUG_PARAMS 40
#define ARGUS_ARC_FIELDS 8
typedef struct argus_aug_config {
  int color_jiggle, planckian_jitter, blur, motion_blur, plasma_shadow;           /* flags, data.py:31-38 */
  float brightness_lo, brightness_span, contrast_lo, contrast_span;               /* ranges, data.py:23-26 */
  float saturation_lo, saturation_span, hue_lo, hue_span;
  int random_erasing, salt_and_pepper;                                            /* flags, data.py:35,39 */
} argus_aug_config;
int argus_augment_sample_params(float* params, int n_images, int n_cams, int H, int W, uint64_t seed, uint64_t step,
                                const argus_aug_config* cfg, void* stream);
/* in: u8 (n, H, W, 3) when in_u8 else fp32 (n, 3, H, W) in [0,1]; out: fp32 (n, 3, H, W), or the stem's bf16
 * space-to-depth layout [n][H/2][W/2+4][16] when out_s2d. apply == 0 only converts. H, W multiples of 32 (<= 256 when
 * apply). arc_mask (nullable, u8 input only): [n][H][W/32] words from argus_spaghetti_mask, set bits are painted black
 * first. plasma_ws: workspace of n * H * W / 8 bytes (required when apply; holds the shadow mask afterwards). */
int argus_augment(const void* in, int in_u8, void* out, int out_s2d, const float* params, const void* arc_mask,
                  void* plasma_ws, int n_images, int H, int W, int apply, void* stream);

/* Spaghetti arcs (draw_spaghetti, argus/utils.py:252-275; drawn with PIL on the decoded image at argus/data.py:212-215,
 * before the kornia chain). arcs: (n_images, n_arcs, ARGUS_ARC_FIELDS) fp32 table [x0, y0, x1, y1, start, end, width, 0],
 * a pure function of (seed, step, image, arc) sampled as the reference does (bbox corners, integer start / end angles,
 * width = int(U(1,5))). argus_spaghetti_mask rasterises them exactly as Pillow's ImageDraw.arc does (oracle/pil_arc.py)
 * into 1 bit per pixel, [n][H][W/32] words (W a multiple of 32, H, W <= 512); argus_spaghetti_draw paints them black on
 * uint8 (n, H, W, 3) images (out may alias in; mask_ws = n * H * W / 8 bytes of workspace). */
int argus_spaghetti_sample_params(float* arcs, int n_images, int n_arcs, int H, int W, uint64_t seed, uint64_t step,
                                  void* stream);
int argus_spaghetti_mask(const float* arcs, void* mask, int n_images, int n_arcs, int H, int W, void* stream);
int argus_spaghetti_draw(const void* in, void* out, const float* arcs, void* mask_ws, int n_images, int n_arcs, int H,
                         int W, void* stream);

/* ---- pose loss and pose exponential ------------------------------------------------------------------------
 * argus_pose_loss: geometric_loss_fn (argus/train.py:105-119) forward AND analytic backward in one launch.
 *   pred (B,6) fp32 se3 [tau, phi]; target (B,7) fp32 SE3 [t, qx, qy, qz, qw]; loss (B) per-sample (nullable);
 *   loss_mean (1) += mean over B (nullable, caller zeroes); grad (B,6) = grad_scale * dloss/dpred (nullable).
 * argus_pose_exp: pp.se3(pred).Exp() (argus/utils.py:179-189); wxyz != 0 emits [t, qw, qx, qy, qz]
 *   (argus/utils.py:130-145). */
int argus_pose_loss(const float* pred, const float* target, float* loss, float* loss_mean, float* grad, int B,
                    float grad_scale, void* stream);
int argus_pose_exp(const float* pred, float* pose, int B, int wxyz, void* stream);

/* ---- optimizer step tail: clip_grad_norm_ + Adam (argus/train.py:318-319) ------------------------------------
 * Flat fp32 arenas of n elements. scratch must hold >= 1024 floats. grads are scaled by gscale (1/world_size for
 * data-parallel averaging) before the norm; norm_out (nullable) receives the pre-clip global L2 norm. */
int argus_clip_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n,
                         float* scratch, float gscale, float max_norm, float lr, float beta1, float beta2, float eps,
                         int step, float* norm_out, void* stream);
/* Same, under the GradScaler protocol of the reference's amp mode (argus/train.py:234,316-320: scaler.unscale_ ->
 * clip_grad_norm_ -> scaler.step): gscale additionally carries 1/loss_scale, and when the unscaled global norm is not
 * finite NOTHING is updated (params, exp_avg, exp_avg_sq untouched). norm_out (required) tells the caller. */
int argus_clip_adam_step_amp(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n,
                             float* scratch, float gscale, float max_norm, float lr, float beta1, float beta2, float eps,
                             int step, float* norm_out, void* stream);

/* ---- the model: NCameraCNN (argus/models.py:26-90) -----------------------------------------------------------
 * The library defines the flat layout of the parameter arena (trainable tensors, reference state_dict order) and
 * the buffer arena (BN running_mean / running_var); the caller allocates them and binds them. */
typedef struct argus_model argus_model;
int argus_model_create(argus_model** out, int n_cams, int resnet_output_dim);
int argus_model_destroy(argus_model* m);
int argus_model_counts(argus_model* m, int* n_params, int* n_buffers, int64_t* param_elems, int64_t* buffer_elems);
/* name_cap bytes of `name` are filled (NUL terminated); shape has room for 4 entries. */
int argus_model_tensor_info(argus_model* m, int is_buffer, int index, char* name, int name_cap, int64_t* offset,
                            int64_t* numel, int* ndim, int64_t* shape);
int argus_model_bind(argus_model* m, float* params, float* grads, float* buffers);
/* Pre-allocate activations for up to max_batch pairs of H x W images (grows on demand otherwise). */
int argus_model_reserve(argus_model* m, int max_batch, int H, int W, int training);
/* fp32 parameters -> packed bf16 tensor-core operands; call after every parameter update / load_state_dict. */
int argus_model_sync_weights(argus_model* m, void* stream);
/* NCameraCNN.forward (argus/models.py:66-90). x is (B, 3*n_cams, H, W) fp32 NCHW, or u8 (B*n_cams, H, W, 3) when
 * is_u8. training != 0 uses batch statistics and updates the running statistics. out is (B, 6) fp32. */
int argus_model_forward(argus_model* m, const void* x, int is_u8, int B, int H, int W, int training, float* out,
                        void* stream);
/* Frozen-statistics backward primitives (see argus_model_forward_frozen; exposed for tests):
 * argus_bn_frozen_finish: one convolution's finish from H = g^T im2col(x) [O][K] fp32 and its bf16 weight W [O][K] in
 *   the same layout: dgamma += invstd * (rowdot(W, H) - mean * sum g), dbeta += sum g, dW = (accumulate ? dW : 0) +
 *   diag(scale) H (dW may be H). sum g = stat_partial summed over `slots` rows of stride stat_stride, in fp64.
 * argus_relu_bits_mask_colsum: g (rows, C) bf16 masked in place by ReLU bits [rows][C/8]; out[c] = column sums.
 * argus_stem_unpool_relu: g0 (N, H, W, 64) = max-unpooled dpool (N, H/2, W/2, 64) through the arg-max bytes, masked by
 *   pooled > 0; out[64] = column sums of g0.
 * argus_pack_weight_scaled: bf16_rn(scale[co] * w) of a PyTorch-layout fp32 weight in the packed layout of the
 *   convolutions (kind 0: [Cout][k][k][Cin]; kind 1: the [64][256] stem). */
int argus_bn_frozen_finish(const void* W, const float* H, const float* stat_partial, int slots, int stat_stride,
                           const float* scale, const float* mean, const float* invstd, float* dgamma, float* dbeta,
                           float* dW, int accumulate, int O, int K, void* stream);
int argus_relu_bits_mask_colsum(void* g, const void* bits, int64_t rows, int C, float* out, void* stream);
int argus_stem_unpool_relu(const void* dpool, const void* idx, const void* pooled, void* g0, int N, int H, int W,
                           float* out, void* stream);
int argus_pack_weight_scaled(const float* w, const float* scale, void* packed, int Cout, int Cin, int k, int kind,
                             void* stream);
/* Eval-mode forward that can be differentiated: the running statistics are constants, the output is bit for bit that of
 * argus_model_forward(training = 0), and the running statistics and num_batches_tracked are left as they are.
 * argus_model_backward and argus_model_input_grad (fp32 x only) then differentiate it, as long as no other forward has
 * run since. x as for argus_model_forward; the input goes to the same pair of model-owned stem buffers a training
 * forward uses, so training and frozen forwards can alternate. x = NULL consumes the batch staged by
 * argus_model_stage_input_frozen_u8 for the same (B, H, W); any other forward in between drops that batch (then this
 * call fails). */
int argus_model_forward_frozen(argus_model* m, const void* x, int is_u8, int B, int H, int W, float* out, void* stream);
/* Fused augmentation + input staging: u8 (B*n_cams, H, W, 3) -> augmented stem input inside the model (training: one
 * of two model-owned staging buffers, so the NEXT batch -- of any size -- can be staged on another stream while the
 * current step runs). The next argus_model_forward call for the same (B, H, W, training) passes x = NULL.
 * arc_mask / plasma_ws: as for argus_augment. */
int argus_model_stage_input_u8(argus_model* m, const void* images, const float* aug_params, const void* arc_mask,
                               void* plasma_ws, int B, int H, int W, int training, int apply, void* stream);
/* argus_model_stage_input_u8 for a frozen-statistics forward: the same arguments (no training flag) and the same work,
 * into the stem buffer the next argus_model_forward_frozen(x = NULL) call for the same (B, H, W) consumes. Fine-tuning
 * with frozen batch norm can thus stage batch k+1 on another stream while step k runs. The staged input is bf16 and
 * augmented, so it has no input gradient: argus_model_input_grad returns an error after such a forward. */
int argus_model_stage_input_frozen_u8(argus_model* m, const void* images, const float* aug_params, const void* arc_mask,
                                      void* plasma_ws, int B, int H, int W, int apply, void* stream);
/* Precision mode. 0 (default): bf16 activations / weights on the tcgen05 tensor cores, fp32 accumulate.
 * 1: fp32 parity mode -- every tensor fp32, SIMT implicit-GEMM convolutions with fp32 FMA accumulation, reductions in
 * fp64; same parameter / gradient / buffer arenas and the same entry points. It exists to compare forward outputs,
 * losses and gradients with the reference's fp32 PyTorch path at 1e-4 relative; it is not a performance path
 * (argus_model_stage_input_u8 and argus_model_copy_activation are bf16-mode only). */
int argus_model_set_precision(argus_model* m, int mode);
/* Weight-gradient GEMMs normally run on a library-owned side stream, overlapping the BN-backward / dgrad chain of the
 * caller's stream (joined before the stage returns). on = 0 serialises them (used for per-kernel timing). */
int argus_model_set_wgrad_overlap(argus_model* m, int on);
int argus_model_zero_grads(argus_model* m, void* stream);
/* Backward of the last training or frozen-statistics forward (whichever ran later; an error when another forward ran
 * after a frozen one). d_out (B,6). Stages 0..3 (head+fc+layer4, layer3, layer2, layer1+stem)
 * must run in order; gradients are ADDED into the bound gradient arena. */
int argus_model_backward(argus_model* m, const float* d_out, int stage_begin, int stage_end, void* stream);
/* d loss / d x for the last training (or frozen-statistics) forward whose input was the fp32 tensor x (B, 3*n_cams, H, W); call after
 * argus_model_backward has run stage 3. dx: (B, 3*n_cams, H, W) fp32, overwritten. Image n = b*n_cams + v is channels
 * [3v, 3v+3) of sample b; the gradient passes straight through the bf16 rounding of the input. Errors (non-zero status,
 * message): no training forward, backward stage 3 not run since it, or the forward consumed a staged / uint8 input. */
int argus_model_input_grad(argus_model* m, float* dx, void* stream);
/* Element range of the parameter arena whose gradients are final once `stage` has run (all-reduce buckets). */
int argus_model_stage_range(argus_model* m, int stage, int64_t* begin, int64_t* end);
int argus_model_arena_bytes(argus_model* m, int64_t* bytes);
/* Test probe: copy an activation of the last forward pass (bf16, NHWC rows x C) into dst (device memory).
 * index -1: stem output after max pooling; 0..15: bottleneck outputs (torchvision layer1[0] .. layer4[2]);
 * 16: global-average-pooled features; 17: resnet.fc output; 100..115: act2 of each bottleneck (the input of conv3,
 * relu(bn2(conv2)): what the fused block tail takes its Gram matrix of). */
int argus_model_copy_activation(argus_model* m, int index, void* dst, int64_t capacity_elems, int64_t* rows, int* C,
                                void* stream);

/* ---- double-buffered pinned loader over a raw uint8 shard file (replaces the DataLoader / DistributedSampler /
 *      `.to(device)` plumbing of argus/train.py:147-192,302-303). File layout: csrc/loader.cu. The caller owns the
 *      staging buffers: two pinned host and two device buffers for images (batch * n_cams*H*W*3 bytes) and poses
 *      (batch * 7 floats). Sampling follows DistributedSampler: one permutation per epoch (seeded by seed and
 *      epoch), padded by wrapping, rank r takes positions r, r + world, ... ----------------------------------------- */
typedef struct argus_loader argus_loader;
int argus_loader_create(argus_loader** out, const char* path, int batch, int rank, int world, uint64_t seed,
                        int shuffle, int drop_last);
int argus_loader_destroy(argus_loader* l);
int argus_loader_info(argus_loader* l, int64_t* n_samples, int* n_cams, int* H, int* W, int64_t* samples_per_rank,
                      int64_t* batches_per_epoch);
int argus_loader_bind(argus_loader* l, void* host_img0, void* host_img1, float* host_pose0, float* host_pose1,
                      void* dev_img0, void* dev_img1, float* dev_pose0, float* dev_pose1);
/* (Re)starts the worker thread for an epoch (DistributedSampler.set_epoch, train.py:290). */
/* on != 0: the caller fetches batch k + 1 BEFORE it enqueues step k (look-ahead loops): a device buffer is then
 * protected by an event recorded at the call that reuses it instead of at the call after its fetch (default 0). */
int argus_loader_set_lookahead(argus_loader* l, int on);
int argus_loader_start_epoch(argus_loader* l, int epoch);
/* Next batch: H2D on the loader's copy stream, ordered before everything later enqueued on `stream`.
 * *count = samples in the batch (0 = epoch finished), *buffer_index = which of the two device buffers holds it. */
int argus_loader_next(argus_loader* l, void* stream, int* count, int* buffer_index);

#ifdef __cplusplus
}
#endif
#endif /* ARGUS_B200_H_ */

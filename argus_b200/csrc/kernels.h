// Launchers of the memory-bound / latency-bound kernels (everything that is not a tensor-core GEMM).
// All tensors are device pointers; activations NHWC bf16; per-channel vectors fp32.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace argus {

typedef __nv_bfloat16 bf16;

// ---- input / weight packing -------------------------------------------------------------------------------
// x: (B, 3*n_cams, H, W) fp32 NCHW in [0,1] (argus/models.py:81 folds views into the batch: image = b*n_cams + v)
// out: [B*n_cams][H/2][W/2+4][16] bf16 space-to-depth layout consumed by the stem convolution.
void pack_input_f32(const float* x, bf16* out, int n_images, int H, int W, cudaStream_t s);
// u8 HWC images (n_images, H, W, 3) -> same layout, scaled by 1/255 (argus/data.py:218)
void pack_input_u8(const uint8_t* x, bf16* out, int n_images, int H, int W, cudaStream_t s);

struct WeightPackEntry {
  int64_t src_off;  // element offset into the fp32 parameter (or gradient) arena, PyTorch layout [Cout][Cin][kh][kw]
  int64_t dst_off;  // element offset into the packed arena, layout [Cout][kh][kw][Cin] (stem: [64][4][4][16])
  int cout, cin, kk;
  int kind;         // 0 conv / linear, 1 stem
};
// fp32 PyTorch-layout parameters -> bf16 packed weights, all layers in one launch (table lives on the device)
void pack_weights(const float* params, bf16* packed, const WeightPackEntry* table_dev, int n_entries, cudaStream_t s);
// fp32 packed-layout weight gradients -> PyTorch-layout gradient arena (only entries with kk > 1 or kind 1)
void unpack_wgrads(const float* packed_grads, float* grads, const WeightPackEntry* table_dev, int n_entries,
                   cudaStream_t s);
// diag(scale) W -> bf16 packed (same layout and offsets as pack_weights), bf16_rn(scale[co] * w) per element. Entry j
// scales its output channels by scales[scale_off_dev[j] + co] (the frozen-statistics backward's dgrad operands).
void pack_weights_scaled(const float* params, const float* scales, const int64_t* scale_off_dev, bf16* packed,
                         const WeightPackEntry* table_dev, int n_entries, cudaStream_t s);

// ---- augmentation (argus/data.py:41-103, 213-225) ---------------------------------------------------------------
constexpr int kAugParams = 40;   // floats per image in the parameter table (layout: oracle/augment.py::sample_params)
constexpr int kArcFields = 8;    // floats per arc: x0, y0, x1, y1, start, end (degrees), width, 0
struct AugConfig {
  int color_jiggle, planckian_jitter, blur, motion_blur, plasma_shadow;
  float brightness_lo, brightness_span, contrast_lo, contrast_span, saturation_lo, saturation_span, hue_lo, hue_span;
  int random_erasing, salt_and_pepper;
};
// params: (n_images, kAugParams) fp32 table, a pure function of (seed, step, image) -- oracle/augment.py::sample_params
void augment_sample_params(float* params, int n_images, int n_cams, int H, int W, uint64_t seed, uint64_t step,
                           const AugConfig& cfg, cudaStream_t s);
// in: u8 (n, H, W, 3) or fp32 (n, 3, H, W); out: bf16 space-to-depth [n][H/2][W/2+4][16] or fp32 (n, 3, H, W).
// apply == false only converts layouts (validation / inference path). arc_mask (nullable): 1 bit per pixel, painted black
// before everything else (u8 input). plasma_mask: workspace of n * H * W / 8 bytes, written here (required when apply).
void augment_images(const void* in, bool in_u8, void* out, bool out_s2d, const float* params, const uint32_t* arc_mask,
                    uint32_t* plasma_mask, int n_images, int H, int W, bool apply, cudaStream_t s);

// spaghetti arcs (argus/utils.py:252-275, applied at argus/data.py:212-215): arcs = (n_images, n_arcs, kArcFields) fp32
// table, a pure function of (seed, step, image, arc); mask = 1 bit per pixel [n][H][W/32] (Pillow's ImageDraw.arc, bit for
// bit); draw paints them black on uint8 HWC images (out may alias in; mask_ws = workspace of n * H * W / 8 bytes)
void spaghetti_sample_params(float* arcs, int n_images, int n_arcs, int H, int W, uint64_t seed, uint64_t step,
                             cudaStream_t s);
void spaghetti_mask(const float* arcs, uint32_t* mask, int n_images, int n_arcs, int H, int W, cudaStream_t s);
void spaghetti_draw(const uint8_t* in, uint8_t* out, const float* arcs, uint32_t* mask_ws, int n_images, int n_arcs, int H,
                    int W, cudaStream_t s);

// ---- batch norm -------------------------------------------------------------------------------------------
// train: batch statistics -> scale/shift (+ saved mean/invstd, running-stat update, torch.nn.BatchNorm2d semantics)
// partial: [slots][2][C] per-(CTA, epilogue group) sums written by the conv epilogue, added here in slot order
void bn_finalize(const float* partial, int slots, double count, const float* gamma, const float* beta,
                 float* running_mean, float* running_var, float momentum, float eps, float* scale, float* shift,
                 float* save_mean, float* save_invstd, int C, cudaStream_t s);
// eval: running statistics -> scale/shift (+ mean = running_mean, invstd = 1/sqrt(running_var + eps) when mean != nullptr:
// the frozen-statistics backward reads them)
void bn_fold_eval(const float* gamma, const float* beta, const float* running_mean, const float* running_var,
                  float eps, float* scale, float* shift, int C, cudaStream_t s, float* mean = nullptr,
                  float* invstd = nullptr);
// bn_apply, bn_bwd_reduce and bn_bwd_apply stream their tensors with 16-byte vectors and bulk copies: every tensor
// pointer they take (x, res, y, relu_bits; dy, x, out, dx) must be 16-byte aligned. They call this before launching
// anything; it throws for a misaligned pointer (nullptr passes). A caller of several passes checks all their tensors
// up front with it, so that none of the passes runs.
void bn_check_aligned(const void* a, const void* b, const void* c, const void* d = nullptr);
// y = [relu]( x*scale+shift  [+ res]  or  [+ res*rscale+rshift] )
// relu_bits (optional): [rows][C/8] bytes, bit k of byte j = (pre-ReLU value of channel 8j+k > 0). The backward pass
// reads this mask instead of the whole bf16 output (1/16 of the bytes).
// colsum_partial (optional, plain variant only): [bn_apply_grid(rows, C)][C] per-block column sums of the stored
// output, added in block order by colsum_finalize (the algebraic bn3 backward needs colsum(act2)).
void bn_apply(const bf16* x, const float* scale, const float* shift, const bf16* res, const float* rscale,
              const float* rshift, int relu, bf16* y, uint8_t* relu_bits, float* colsum_partial, int64_t rows, int C,
              cudaStream_t s);
int bn_apply_grid(int64_t rows, int C);
void colsum_finalize(const float* partial, int blocks, float* out, int C, cudaStream_t st);
// mask_mode: 0 = no ReLU after this BN, 1 = ReLU directly after (mask recomputed from x), 2 = ReLU after a residual
// add (mask = out > 0), 3 = like 2 but `out` points to the relu_bits written by bn_apply. Accumulates dgamma += sum(g * xhat), dbeta += sum(g) with g = masked dy.
// Deterministic: every block writes its partial sums to `scratch` (>= bn_bwd_scratch_elems() floats), a second tiny
// kernel adds them in block order. This call's sums alone also go to bn_bwd_sums(scratch), [2][C]: sum(g), sum(g * xhat).
void bn_bwd_reduce(const bf16* dy, const bf16* x, const bf16* out, const float* scale, const float* shift,
                   const float* mean, const float* invstd, float* dgamma, float* dbeta, int64_t rows, int C,
                   int mask_mode, float* scratch, cudaStream_t s);
int64_t bn_bwd_scratch_elems();
float* bn_bwd_sums(float* scratch);
// The same sums when a dgrad epilogue already reduced them (Epilogue::bn_raw): partial = [slots][2][C] with sum(g) and
// sum(g * x) of the raw layer output x per slot; dbeta += sum(g), dgamma += (sum(g * x) - mean * sum(g)) * invstd, and
// sums [2][C] = those two terms alone.
void bn_bwd_finalize_slots(const float* partial, int slots, const float* mean, const float* invstd, float* dgamma,
                           float* dbeta, float* sums, int C, cudaStream_t s);
// dx = scale * (g - sum(g)/rows - xhat * sum(g * xhat)/rows) with sums = [2][C] (sum g, sum g * xhat) of THIS layer's
// reduction (never the dgamma / dbeta accumulators, which may hold earlier gradients); mask_mode 2 also overwrites dy
// with g (mask_mode 3 leaves dy untouched: the consumers of the identity-branch gradient apply the bit mask themselves).
void bn_bwd_apply(bf16* dy, const bf16* x, const bf16* out, const float* scale, const float* shift,
                  const float* mean, const float* invstd, const float* sums, bf16* dx, int64_t rows, int C,
                  int mask_mode, cudaStream_t s);

// ---- pooling ----------------------------------------------------------------------------------------------
// 3x3 stride-2 pad-1 max pooling of relu(x*scale+shift) (scale == nullptr: x is already activated).
// idx (optional) records the arg-max tap (0..8) for the backward pass.
void maxpool_fwd(const bf16* x, const float* scale, const float* shift, bf16* y, uint8_t* idx, int N, int H, int W,
                 int C, cudaStream_t s);
void maxpool_bwd(const bf16* dy, const uint8_t* idx, bf16* dx, int N, int H, int W, int C, cudaStream_t s);
// Stem tail backward in two passes over the stem convolution output `raw` (N, H, W, 64): max-pool backward (from the
// pooled gradient dpool (N, H/2, W/2, 64) and the arg-max bytes), ReLU mask and batch-norm backward fused, the
// un-pooled gradient is never written. dgamma / dbeta are accumulated (+=); dx = gradient wrt `raw`, formed from this
// call's sums alone (bn_bwd_sums(scratch); scratch: >= bn_bwd_scratch_elems() floats).
void stem_pool_bn_backward(const bf16* dpool, const uint8_t* idx, const bf16* raw, const float* scale,
                           const float* shift, const float* mean, const float* invstd, float* dgamma, float* dbeta,
                           bf16* dx, int N, int H, int W, int C, float* scratch, cudaStream_t s);
// global average pooling (N, HW, C) -> (N, C) and its backward
void avgpool_fwd(const bf16* x, bf16* y, int N, int HW, int C, cudaStream_t s);
// relu_bits (optional, [N*HW][C/8]): the result is stored already masked by the ReLU bit mask of the pooled tensor
void avgpool_bwd(const bf16* dy, bf16* dx, const uint8_t* relu_bits, int N, int HW, int C, cudaStream_t s);

// ---- algebraic batch-norm backward of an expanding 1x1 convolution (bn_algebra.cu) -------------------------------
// W: bf16 [O][C] weights (the packed copy the forward GEMM used); H = g^T act [O][C]; G = act^T act [C][C]; s = colsum(act) [C]; stat_partial: per-slot sums
// of g ([slot] stride stat_stride floats, channel o at offset o) written by the dgrad epilogue that produced g.
// Accumulates dgamma / dbeta / dW (+=) and writes the stacked bf16 dgrad operand bstack [(O + C)][C]
// (rows < O: scale[o] * W[o][:], rows O + j: W^T diag(k1) W) and the fp32 bias row k0^T W [C]. k1k0: 2*O floats scratch.
void bn_alg_backward_small(const bf16* W, const float* H, const float* G, const float* s, const float* stat_partial,
                           int slots, int stat_stride, const float* scale, const float* mean, const float* invstd,
                           double rows, float* dgamma, float* dbeta, float* dW, float* k1k0, bf16* bstack, float* bias,
                           float* mpartial, int O, int C, cudaStream_t st);
// dW == nullptr above skips the weight-gradient kernel; this runs it alone (on another stream):
// dW[o][i] += scale[o] H[o][i] + k0[o] s[i] + k1[o] sum_j W[o][j] G[j][i]
void bn_alg_backward_dw(const bf16* W, const float* H, const float* G, const float* s, const float* scale,
                        const float* k1k0, float* dW, int O, int C, cudaStream_t st);
int64_t bn_alg_matrix_scratch_elems(int C);   // floats of `mpartial`
// Forward counterpart: train-mode batch statistics of y = x W^T from G = x^T x and s = colsum(x) (both over the `rows`
// pixels the 1x1 convolution reads), before / instead of computing y: scale, shift, mean, invstd and the running-stat
// update of torch.nn.BatchNorm2d. scratch: O * C / 16 floats.
void bn_stats_from_gram(const bf16* W, const float* G, const float* s, double rows, const float* gamma,
                        const float* beta, float* running_mean, float* running_var, float momentum, float eps,
                        float* scale, float* shift, float* save_mean, float* save_invstd, float* scratch, int O, int C,
                        cudaStream_t st);
// ---- frozen-statistics batch-norm backward (bn_algebra.cu) --------------------------------------------------------
// With constant statistics the batch norm after a convolution is the per-channel affine map sc * raw + shift, so with g
// the (ReLU-masked) gradient of its output and H = g^T im2col(x) the weight-gradient GEMM fed g:
//   dW = diag(sc) H,  dgamma = invstd * (rowdot(W, H) - mean * sum g),  dbeta = sum g.
// One warp per output channel o; W: bf16 [O][K] (the packed weight the forward used), H: fp32 [O][K] in the same layout.
// sum g = the fp64 sum of stat_partial[k * stat_stride + o] over k < slots (a dgrad's statistics slots, or slots = 1 for
// a finished vector). dgamma, dbeta += ; dW[o][:] = (accumulate ? dW[o][:] : 0) + scale[o] * H[o][:] (dW may be H).
// Deterministic: fixed lane order and shuffle tree, fp64 sums.
void bn_frozen_finish(const bf16* W, const float* H, const float* stat_partial, int slots, int stat_stride,
                      const float* scale, const float* mean, const float* invstd, float* dgamma, float* dbeta, float* dW,
                      bool accumulate, int O, int K, cudaStream_t st);
// g[r][c] = bit(r, c) ? g[r][c] : 0 in place (bits: [rows][C/8], bit k of byte j = channel 8j + k) and out[c] = sum_r of
// the stored values, deterministic. scratch: >= 4 * num_sms * C floats.
void relu_bits_mask_colsum(bf16* g, const uint8_t* bits, int64_t rows, int C, float* scratch, float* out,
                           cudaStream_t st);
// Stem of the frozen-statistics backward: g0 = unpool(dpool) * [pooled > 0] -- the gradient wrt the stem's BN + ReLU
// output (N, H, W, 64), written in full -- from the pooled gradient dpool and the pooled values (N, H/2, W/2, 64) and
// the arg-max bytes of maxpool_fwd. A max of ReLU outputs is positive exactly where its arg-max element is. The up to
// four windows that hold a pixel are added in fp32 in window order; out[c] = sum of the stored g0, deterministic.
// scratch: >= 4 * num_sms * 64 floats.
void stem_unpool_relu(const bf16* dpool, const uint8_t* idx, const bf16* pooled, bf16* g0, int N, int H, int W,
                      float* scratch, float* out, cudaStream_t st);
// out[c] = sum_r x[r][c], deterministic; scratch: >= 4 * num_sms * C floats
void colsum_rows_bf16(const bf16* x, int64_t rows, int C, float* scratch, float* out, cudaStream_t st);
// same over the pixels (stride*h, stride*w) of an (N, H, W, C) tensor (what a strided 1x1 convolution reads)
void colsum_pixels_bf16(const bf16* x, int N, int H, int W, int C, int stride, float* scratch, float* out,
                        cudaStream_t st);

// ---- head MLP (fp32 SIMT; argus/models.py:58-64,88-90) -----------------------------------------------------
// z = gelu(feat) ; feat bf16 (rows, cols) -> z fp32
void gelu_fwd_bf16(const bf16* x, float* y, int64_t n, cudaStream_t s);
// dfeat = dz * gelu'(feat) -> bf16
void gelu_bwd_bf16(const float* dz, const bf16* x, bf16* dx, int64_t n, cudaStream_t s);
// y = x W^T + b ; optionally a = gelu(y)
void linear_fwd(const float* x, const float* w, const float* b, float* y, float* act, int B, int In, int Out,
                cudaStream_t s);
// given dy (grad wrt the linear output y; if pre != nullptr the incoming grad is wrt gelu(y) and is first multiplied
// by gelu'(pre) in place): dw += dy^T x, db += sum dy, dx = dy W
void linear_bwd(float* dy, const float* pre, const float* x, const float* w, float* dw, float* db, float* dx, int B,
                int In, int Out, cudaStream_t s);
// the same in two halves (model.cu runs the weight half on the weight-gradient side stream): linear_bwd_input applies
// GELU' to dy in place (pre != nullptr) and writes dx; linear_bwd_weights accumulates dw / db from the finished dy
void linear_bwd_input(float* dy, const float* pre, const float* w, float* dx, int B, int In, int Out, cudaStream_t s);
void linear_bwd_weights(const float* dy, const float* x, float* dw, float* db, int B, int In, int Out, cudaStream_t s);

// ---- loss / pose ------------------------------------------------------------------------------------------
// per-sample loss (argus/train.py:119), its mean accumulated into *loss_mean (caller zeroes), and
// grad = grad_scale * dloss/dpred
void pose_loss_fwd_bwd(const float* pred, const float* target, float* loss, float* loss_mean, float* grad, int B,
                       float grad_scale, cudaStream_t s);
// pp.se3(pred).Exp() (argus/utils.py:189); wxyz != 0 writes [t, qw, qx, qy, qz] (argus/utils.py:130-145)
void pose_exp(const float* pred, float* pose, int B, int wxyz, cudaStream_t s);

// ---- optimizer step tail (argus/train.py:318-319) ------------------------------------------------------------
// partial[b] = sum of squares of block b's slice (deterministic two-stage reduction); returns number of partials
int grad_sqnorm_partials(const float* g, int64_t n, float* partial, cudaStream_t s);
// clip_grad_norm_(max_norm) + Adam, fused: every block first reduces `partial` to the global norm.
// gscale multiplies gradients before the norm (1/world for data-parallel averaging).
void clip_adam_step(float* p, const float* g, float* m, float* v, int64_t n, const float* partial, int n_partial,
                    float gscale, float max_norm, float lr, float beta1, float beta2, float eps, int step,
                    float* norm_out, bool skip_nonfinite, cudaStream_t s);

}  // namespace argus

// NCameraCNN (/root/reference/argus/models.py:26-90) as a statically scheduled graph over the sm_100a kernels:
// shared-weight ResNet-50 per view -> fc(2048 -> resnet_output_dim) -> concat views -> GELU -> MLP -> se(3) 6-vector.
//
// The model object owns: packed bf16 weights, batch-norm scratch, activation and gradient arenas, and the per-batch
// launch plans (TMA tensor maps). The caller (PyTorch) owns the fp32 parameter / gradient / buffer arenas whose
// layout is described by tensor_info() in the reference's state_dict order.
#pragma once
#include <functional>
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "conv_ops.h"
#include "kernels.h"
#include "runtime.h"

namespace argus {

struct TensorInfo {
  std::string name;
  int64_t offset = 0;  // element offset inside its arena
  int64_t numel = 0;
  int ndim = 0;
  int64_t shape[4] = {0, 0, 0, 0};
};

struct BnRef {
  int C = 0;
  int64_t gamma_off = 0, beta_off = 0;  // parameter arena
  int64_t rm_off = 0, rv_off = 0;       // buffer arena
  int64_t scratch_off = 0;              // bn scratch arena: scale, shift, mean, invstd (4*C floats)
  int64_t stat_off = 0;                 // statistics arena: [max_slots][2][C] per-CTA partial sums
};

struct ConvRef {
  ConvShape shape;           // N filled in at plan time
  int64_t w_off = 0;         // parameter arena (PyTorch layout)
  int64_t packed_off = 0;    // packed bf16 arena
  int64_t gpacked_off = -1;  // packed fp32 gradient scratch (-1: gradient accumulates directly in the grad arena)
  BnRef bn;
  int stage = 0;             // backward stage (0 = head/fc/layer4 ... 3 = layer1/stem)
};

struct BlockRef {
  ConvRef c1, c2, c3, ds;
  bool has_ds = false;
};

struct ConvPlan {
  ConvLaunch fwd;
  std::vector<ConvLaunch> dgrad;
  WgradLaunch wgrad;
  bool has_dgrad = false;
};

struct BlockPlan {
  ConvPlan c1, c2, c3, ds;
  bf16 *x = nullptr, *raw1 = nullptr, *act1 = nullptr, *raw2 = nullptr, *act2 = nullptr, *raw3 = nullptr,
       *rawd = nullptr, *out = nullptr;
  uint8_t* out_bits = nullptr;   // ReLU mask of `out` (training, frozen): [rows_out][Cout/8] bytes
  uint8_t *act1_bits = nullptr, *act2_bits = nullptr;   // frozen plans: ReLU masks of act1 / act2
  int64_t rows_in = 0, rows_mid = 0, rows_out = 0;
  // gradient scratch roles for this block
  bf16 *g_out = nullptr, *g_q = nullptr, *g_r = nullptr, *g_t = nullptr, *g_x = nullptr;
  // Fused block tail (training plans, mid width <= 256, unless ARGUS_BN_ALGEBRA=0): bn3's batch statistics come from the
  // Gram matrix of act2, so conv3 applies BN + identity + ReLU (+ bit mask) in its epilogue and raw3 is never written.
  // The backward is then algebraic (bn_algebra.cu): H = g^T act2 with the saved G = act2^T act2, concatenated-K dgrad of
  // conv3.
  bool fused_tail = false;
  WgradLaunch fwd_gram, ds_fwd_gram;
  // the Gram matrices of act2 / x the forward statistics were derived from, each followed by the column sums of the same
  // activation; ds_gram_saved is set when the downsample branch (Cin <= 256) takes the same path, with act = the block
  // input (its even pixels at stride 2)
  float *gram_saved = nullptr, *ds_gram_saved = nullptr;
  float* act2_colsum = nullptr;   // [bn_apply_grid][C] per-block column sums of act2, written by the forward bn_apply
  WgradLaunch hg_wgrad;           // H = g^T act2 into alg_h_
  ConvLaunch c3_concat;
  WgradLaunch ds_hg_wgrad;
  ConvLaunch ds_concat;
  size_t x_bytes = 0;
  // Stride-2 downsample blocks own their g_t buffer: the 1x1 stride-2 dgrad writes one pixel in four and the others
  // must read as zero, so a buffer nobody else touches is zero-filled once (t_zero_epoch == Model::arena_epoch_) instead
  // of on every step (1.9 GB of memset per step at B = 256).
  uint64_t t_zero_epoch = 0;
};

struct Plan {
  int B = 0, H = 0, W = 0, N = 0;
  bool training = false;
  // Frozen-statistics plan (a differentiable eval-mode forward): the eval layout plus the ReLU bit masks, the max-pool
  // arg-max bytes and the backward scratch; no pre-BN tensors. Its backward is Model::backward_frozen.
  bool frozen = false;
  ConvPlan stem;
  bf16 *raw0 = nullptr, *act0 = nullptr, *pooled0 = nullptr;
  // The stem input of training and frozen plans is double buffered so that the NEXT batch can be augmented / staged (on
  // another stream) while the current one trains. The two buffers belong to the MODEL (Model::stem_in_, sized for the
  // largest reserved batch, outside the per-plan arena layout), so that staging a batch of a different size -- the short
  // last batch of an epoch -- can never alias the buffer the in-flight step still reads. Training and frozen forwards
  // alternate through the same pair. stem_fwd_buf / stem_wgrad_buf are the launches reading buffer 0 / 1; forward()
  // copies the pair of the buffer it consumes into stem.fwd / stem.wgrad.
  bf16* x_in = nullptr;   // eval plans: private stem input inside the arena (staging + forward run on one stream)
  ConvLaunch stem_fwd_buf[2];
  WgradLaunch stem_wgrad_buf[2];
  uint8_t* idx0 = nullptr;
  std::vector<BlockPlan> blocks;
  ConvPlan fc;
  bf16 *pooled = nullptr, *feat = nullptr;
  int final_hw = 0;
  // head (fp32)
  float *z0 = nullptr, *h1 = nullptr, *a1 = nullptr, *h2 = nullptr, *a2 = nullptr, *out = nullptr;
  float *d_out = nullptr, *d_a2 = nullptr, *d_a1 = nullptr, *d_z0 = nullptr;
  bf16 *d_feat = nullptr, *d_pooled = nullptr;
  bf16* g_stem_in = nullptr;   // gradient wrt the pooled stem output (= layer1.0 input gradient)
  bf16 *g_act0 = nullptr, *g_raw0 = nullptr;   // (frozen plans: g_raw0 = g0, the gradient wrt the stem's BN output)
};

struct Fp32State;                        // fp32 parity mode (model_fp32.cu)
void destroy_fp32_state(Fp32State* st);

class Model {
 public:
  Model(int n_cams, int resnet_output_dim);
  ~Model();

  const std::vector<TensorInfo>& params() const { return params_; }
  const std::vector<TensorInfo>& buffers() const { return buffers_; }
  int64_t num_param_elems() const { return n_param_elems_; }
  int64_t num_buffer_elems() const { return n_buffer_elems_; }
  // element range [begin, end) of the parameter arena owned by a backward stage (for bucketed all-reduce)
  void stage_param_range(int stage, int64_t* begin, int64_t* end) const;

  void bind(float* params, float* grads, float* buffers);
  void reserve(int max_batch, int H, int W, bool training, bool frozen = false);
  void sync_weights(cudaStream_t s);   // fp32 parameters -> packed bf16 (+ marks the eval BN fold dirty)

  // x: (B, 3*n_cams, H, W) fp32 NCHW in [0,1], or u8 (B*n_cams, H, W, 3) when is_u8. out: (B, 6) fp32.
  // frozen (training == false): the eval-mode forward with the same output bits, made differentiable by backward() /
  // input_grad() with the running statistics as constants; nothing the model keeps between passes changes.
  void forward(const void* x, bool is_u8, int B, int H, int W, bool training, float* out, cudaStream_t s,
               bool frozen = false);
  // Augmentation fused with input staging: uint8 (B*n_cams, H, W, 3) images -> augmented bf16 stem input of the plan
  // for (B, H, W, training, frozen). A following forward() of the same kind with x == nullptr consumes it.
  // arc_mask (nullable): spaghetti arcs as 1 bit per pixel; plasma_ws: workspace of B * n_cams * H * W / 8 bytes
  void stage_input_u8(const uint8_t* images, const float* aug_params, const uint32_t* arc_mask, uint32_t* plasma_ws, int B,
                      int H, int W, bool training, bool apply, cudaStream_t s, bool frozen = false);
  // d_out: (B, 6) gradient of the loss wrt forward()'s output. Accumulates parameter gradients (+=) into the bound
  // gradient arena for stages [stage_begin, stage_end); stages must be run in increasing order 0..3. Differentiates the
  // last training or frozen forward, whichever ran last; a frozen one must still be the last forward of all.
  void backward(const float* d_out, int stage_begin, int stage_end, cudaStream_t s);
  void zero_grads(cudaStream_t s);
  // d loss / d x of the last training forward (whose input was the fp32 tensor x) once backward() has run stage 3:
  // dx (B, 3*n_cams, H, W) fp32, overwritten. Throws without such a forward / backward, or for a staged / u8 input.
  void input_grad(float* dx, cudaStream_t s);
  // overlap the weight-gradient GEMMs with the rest of the backward pass on a side stream (default on)
  void set_wgrad_overlap(bool on) { overlap_wgrad_ = on; }
  // Debug / test probe: copies an activation of the LAST forward (bf16 NHWC rows x C) into dst.
  // index -1: pooled stem output; 0..15: bottleneck block outputs; 16: globally pooled features; 17: fc output.
  void copy_activation(int index, void* dst, int64_t capacity_elems, int64_t* rows, int* C, cudaStream_t s);

  // 0 = bf16 tensor-core path (default), 1 = fp32 SIMT parity mode (same parameters, buffers and results layout)
  void set_precision(int mode);
  int precision() const { return precision_; }

  int n_cams() const { return n_cams_; }
  int out_dim() const { return out_dim_; }
  size_t arena_bytes() const { return arena_bytes_; }

 private:
  void build_layout();
  Plan& get_plan(int B, int H, int W, bool training, bool frozen = false);
  void build_plan(Plan& p);
  void fold_eval(cudaStream_t s);
  void forward_train(Plan& p, cudaStream_t s);
  void forward_eval(Plan& p, cudaStream_t s);
  void head_forward(Plan& p, float* out, cudaStream_t s);
  void head_backward(Plan& p, const float* d_out, cudaStream_t s);
  void unpack_stage_wgrads(int stage, cudaStream_t s);
  // frozen-statistics backward (see bn_algebra.cu): weight gradient H of c into h (zeroed here), then the finish
  void frozen_wgrad_finish(const ConvRef& c, const WgradLaunch& l, float* h, const float* sums, int slots, int stride,
                           float* dW, bool accumulate, cudaStream_t s);
  void backward_frozen(Plan& p, int stage_begin, int stage_end, const float* d_out, cudaStream_t s);
  void ensure_frozen_buffers();
  void run_conv_train(const ConvPlan& cp, const ConvRef& c, int64_t rows, cudaStream_t s);
  // batch statistics of the 1x1 convolution c from the Gram matrix of its input (gram launch + colsum) -> BN scratch
  void stats_from_gram(const ConvRef& c, const WgradLaunch& gram, float* G, const bf16* act, const float* colsum_partial,
                       int64_t rows, int N, cudaStream_t s);
  void bn_backward(const ConvRef& c, bf16* dy, const bf16* raw, const bf16* out, bf16* dx, int64_t rows, int mask,
                   cudaStream_t s);
  // out_bits: ReLU mask of the tensor whose gradient this dgrad produces (stored masked); out_stats: per-slot channel
  // sums of that masked gradient (the dbeta of the algebraic bn3 backward of the previous block)
  // red (optional): the BN + ReLU layer whose output gradient this dgrad produces -- its backward reduction runs in the
  // dgrad epilogue (Epilogue::bn_raw) and bn_backward_reduced() replaces bn_backward() for that layer
  struct BnRed { const ConvRef* c; const bf16* raw; };
  void conv_backward(const ConvPlan& cp, const bf16* residual, const uint8_t* out_bits, float* out_stats, cudaStream_t s,
                     const BnRed* red = nullptr);
  void attach_bn_reduction(Epilogue& e, const ConvLaunch& l, const BnRed& red, cudaStream_t s);
  // BN backward of a layer whose gradient arrived masked and already reduced (bnred_stats_): finalize + apply
  void bn_backward_reduced(const ConvRef& c, bf16* dy, const bf16* raw, bf16* dx, int64_t rows, cudaStream_t s);
  // conv (expanding 1x1) + BN backward on the masked upstream gradient (bn_algebra.cu); saved_gram: the Gram matrix of
  // the convolution input the forward kept, followed by its column sums
  void conv_bn_backward_algebraic(const ConvRef& c, const WgradLaunch& hg, const ConvLaunch& concat,
                                  const float* saved_gram, int64_t rows, cudaStream_t s, const BnRed* red = nullptr);

  template <typename T>
  T* arena_alloc(size_t count);

  // fp32 parity mode
  void plan_fp32(Fp32State& st, int B, int H, int W, bool training);
  Fp32State& fp32_state(int B, int H, int W, bool training);
  void forward_fp32(const void* x, bool is_u8, int B, int H, int W, bool training, bool frozen, float* out,
                    cudaStream_t s);
  void backward_fp32(const float* d_out, int stage_begin, int stage_end, cudaStream_t s);
  void input_grad_fp32(float* dx, cudaStream_t s);
  void check_input_grad_ready(bool have_train_forward) const;
  int precision_ = 0;
  Fp32State* f32_ = nullptr;

  int n_cams_, out_dim_;
  std::vector<TensorInfo> params_, buffers_;
  int64_t n_param_elems_ = 0, n_buffer_elems_ = 0;
  ConvRef stem_;
  std::vector<BlockRef> blocks_;
  ConvRef fc_;  // bn unused; bias at fc_bias_off_
  int64_t fc_bias_off_ = 0;
  int64_t head_w_off_[3] = {0, 0, 0}, head_b_off_[3] = {0, 0, 0};
  int64_t stage_begin_[5] = {0, 0, 0, 0, 0};  // parameter-arena offsets where each network segment starts

  float *params_dev_ = nullptr, *grads_dev_ = nullptr, *buffers_dev_ = nullptr;
  bf16* packed_ = nullptr;
  float* gpacked_ = nullptr;
  float* bn_scratch_ = nullptr;
  float* bn_stats_ = nullptr;
  float* bn_bwd_scratch_ = nullptr;   // per-block partial sums of the BN-backward reductions
  // algebraic bn3 backward scratch (sized for the widest eligible block)
  bool bn_algebra_ = true;
  int alg_max_o_ = 0, alg_max_c_ = 0;
  float *alg_h_ = nullptr, *alg_k1k0_ = nullptr, *alg_bias_ = nullptr;
  float* alg_mpartial_ = nullptr;
  float* alg_gstats_ = nullptr;       // [max_stat_slots_][2][alg_max_o_] sums of the masked gradient, per dgrad CTA slot
  bf16* alg_bstack_ = nullptr;
  int alg_gstats_slots_ = 0;          // slots the last producing dgrad launch wrote
  // BN-backward sums reduced by the producing dgrad's epilogue: [max_stat_slots_][2][512] sum(g), sum(g * raw)
  int bn_reduce_fused_ = 0;           // 0 = separate passes (default), 1 = layers 1-2, 2 = every eligible layer
  float* bnred_stats_ = nullptr;
  int bnred_slots_ = 0;
  float* wgrad_scratch_ = nullptr;    // split-K partial weight gradients (one launch at a time)
  int64_t wgrad_scratch_elems_ = 0;
  int max_stat_slots_ = 0;
  void ensure_wgrad_scratch(const WgradLaunch& l);
  void run_wgrad(const WgradLaunch& l, cudaStream_t s);
  void run_on_side(cudaStream_t s, const std::function<void(cudaStream_t)>& work);
  int64_t n_packed_ = 0, n_gpacked_ = 0, n_bn_scratch_ = 0, n_bn_stats_ = 0;
  WeightPackEntry* pack_table_dev_ = nullptr;
  std::vector<WeightPackEntry> pack_table_;
  std::vector<int> pack_table_stage_;
  bool eval_fold_dirty_ = true;
  // frozen-statistics backward: diag(sc) W in the packed layout (refreshed after every eval fold), its pack table
  // (every BN-followed convolution; scale offsets into bn_scratch_), and scratch
  bf16* packed_scaled_ = nullptr;
  WeightPackEntry* scaled_table_dev_ = nullptr;
  int64_t* scaled_scale_off_dev_ = nullptr;
  int n_scaled_entries_ = 0;
  bool scaled_dirty_ = true;
  float* frz_h_ = nullptr;        // H = g^T x of the 1x1 convolutions, [Cout][Cin]
  float* frz_pstats_ = nullptr;   // [max_stat_slots_][2][2048] statistics slots of the conv1 dgrads: sum of P
  float* frz_gstats_ = nullptr;   // [max_stat_slots_][2][512] statistics slots of the conv3 dgrads: sum of g2
  float* frz_sums_ = nullptr;     // [2][2048] finished column sums: sum of P (last block), sum of g1 / g0
  float* frz_partial_ = nullptr;  // per-block column-sum partials, 4 * num_sms * 2048 floats
  const float* frz_p_sum_ = nullptr;   // where the sum of the current block's output gradient P lives
  int frz_p_slots_ = 0, frz_p_stride_ = 0;

  uint8_t* arena_ = nullptr;
  size_t arena_bytes_ = 0, arena_used_ = 0;
  int reserved_batch_ = 0, reserved_h_ = 0, reserved_w_ = 0;
  bool reserved_training_ = false;
  std::map<std::tuple<int, int, int, bool, bool>, std::unique_ptr<Plan>> plans_;
  Plan* last_train_plan_ = nullptr;
  Plan* last_frozen_plan_ = nullptr;
  int last_grad_forward_ = 0;      // 0: none, 1: training, 2: frozen -- the forward backward() differentiates
  bool last_forward_frozen_ = false;   // the most recent forward of any kind was a frozen one
  Plan* last_plan_ = nullptr;
  uint64_t arena_epoch_ = 1;   // bumped whenever another plan (they share the arena) runs a forward pass
  Plan* staged_plan_ = nullptr;
  bool train_input_f32_ = false;   // the last training / frozen forward read an fp32 image tensor (not u8 / staged)
  bool stem_grad_ready_ = false;   // backward() stage 3 ran after the last forward(): the stem's output gradient is live
  // stem input double buffer (see Plan): [n][H/2][W/2 + 4][16] bf16 each; cur_in_ = the buffer the last forward consumed
  bf16* stem_in_[2] = {nullptr, nullptr};
  size_t stem_in_elems_ = 0;
  int cur_in_ = 0;
  // weight-gradient GEMMs run on a side stream, overlapping the HBM-bound BN-backward / dgrad chain
  cudaStream_t side_ = nullptr;
  cudaEvent_t ev_fork_ = nullptr, ev_wgrad_ = nullptr;
  bool wgrad_pending_ = false;
  bool overlap_wgrad_ = true;
  void zero_ds_gradient_once(BlockPlan& bp, const BlockRef& br, bf16* T, cudaStream_t s);
  void join_wgrad(cudaStream_t s);
};

}  // namespace argus

#include "model.h"

#include <algorithm>
#include <cstring>
#include <functional>
#include <tuple>

namespace argus {

static constexpr float kBnEps = 1e-5f;
static constexpr float kBnMomentum = 0.1f;

// ------------------------------------------------------------------------------------------------------------
// small kernels local to the model: column sums (fc bias gradient)
// ------------------------------------------------------------------------------------------------------------
// Debugging aid for cross-stream ordering: ARGUS_FUZZ_DELAY_US=<n> (bit mask ARGUS_FUZZ_SITES: 1 = weight-gradient side
// stream, 2 = input staging) starts the side-stream work of every fork with an n-microsecond spin, so that a missing
// or too-weak dependency (main stream overwriting what the side stream has not read yet, or reading what it has not
// written yet) changes results reproducibly on the default stream (profiles/experiments/stream_determinism.py).
__global__ void fuzz_delay_kernel(unsigned long long ns) {
  pdl_prologue();
  const unsigned long long t0 = globaltimer_ns();
  while (globaltimer_ns() - t0 < ns) {}
}
static int fuzz_delay_us() {
  static const int v = [] { const char* e = getenv("ARGUS_FUZZ_DELAY_US"); return e ? atoi(e) : 0; }();
  return v;
}
static int fuzz_sites() {
  static const int v = [] { const char* e = getenv("ARGUS_FUZZ_SITES"); return e ? atoi(e) : 3; }();
  return v;
}
static void fuzz_delay(int site, cudaStream_t s) {
  if (fuzz_delay_us() <= 0 || !(fuzz_sites() & site)) return;
  launch_kernel(fuzz_delay_kernel, 1, 1, 0, s, static_cast<unsigned long long>(fuzz_delay_us()) * 1000ull);
  ARGUS_CUDA(cudaGetLastError());
}

__global__ void colsum_bf16_kernel(const bf16* __restrict__ x, float* out, int rows, int C) {
  pdl_prologue();
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  float acc = 0.f;
  for (int r = 0; r < rows; ++r) acc += __bfloat162float(x[static_cast<int64_t>(r) * C + c]);
  out[c] += acc;
}

// ------------------------------------------------------------------------------------------------------------
// layout: parameter / buffer arenas in the reference's state_dict order
// ------------------------------------------------------------------------------------------------------------
Model::Model(int n_cams, int resnet_output_dim) : n_cams_(n_cams), out_dim_(resnet_output_dim) {
  ARGUS_CHECK(n_cams >= 1 && n_cams <= 8, "n_cams out of range");
  ARGUS_CHECK(resnet_output_dim % 64 == 0 && resnet_output_dim >= 64, "resnet_output_dim must be a multiple of 64");
  build_layout();
}

void Model::set_precision(int mode) {
  ARGUS_CHECK(mode == 0 || mode == 1, "precision mode must be 0 (bf16 tensor cores) or 1 (fp32)");
  precision_ = mode;
  last_train_plan_ = nullptr;
  last_frozen_plan_ = nullptr;
  last_grad_forward_ = 0;
  last_forward_frozen_ = false;
  stem_grad_ready_ = false;
  last_plan_ = nullptr;
  staged_plan_ = nullptr;
  eval_fold_dirty_ = true;
}

Model::~Model() {
  destroy_fp32_state(f32_);
  if (side_) cudaStreamDestroy(side_);
  if (ev_fork_) cudaEventDestroy(ev_fork_);
  if (ev_wgrad_) cudaEventDestroy(ev_wgrad_);
  cudaFree(packed_);
  cudaFree(gpacked_);
  cudaFree(bn_scratch_);
  cudaFree(bn_stats_);
  cudaFree(bn_bwd_scratch_);
  cudaFree(alg_h_); cudaFree(alg_s_); cudaFree(alg_k1k0_); cudaFree(alg_bias_); cudaFree(alg_gstats_);
  cudaFree(alg_bstack_);
  cudaFree(alg_mpartial_);
  cudaFree(bnred_stats_);
  cudaFree(wgrad_scratch_);
  cudaFree(pack_table_dev_);
  cudaFree(packed_scaled_); cudaFree(scaled_table_dev_); cudaFree(scaled_scale_off_dev_);
  cudaFree(frz_h_); cudaFree(frz_pstats_); cudaFree(frz_gstats_); cudaFree(frz_sums_); cudaFree(frz_partial_);
  cudaFree(stem_in_[0]);
  cudaFree(stem_in_[1]);
  cudaFree(arena_);
}

void Model::build_layout() {
  auto add_param = [&](const std::string& name, std::initializer_list<int64_t> shape) {
    TensorInfo t;
    t.name = name;
    t.offset = n_param_elems_;
    t.ndim = static_cast<int>(shape.size());
    t.numel = 1;
    int i = 0;
    for (int64_t d : shape) { t.shape[i++] = d; t.numel *= d; }
    // keep every tensor 16-byte aligned inside the arena (float4 loads in the optimizer / epilogues)
    n_param_elems_ += (t.numel + 3) / 4 * 4;
    params_.push_back(t);
    return t.offset;
  };
  auto add_buffer = [&](const std::string& name, int64_t n) {
    TensorInfo t;
    t.name = name;
    t.offset = n_buffer_elems_;
    t.ndim = 1;
    t.numel = n;
    t.shape[0] = n;
    n_buffer_elems_ += (n + 3) / 4 * 4;
    buffers_.push_back(t);
    return t.offset;
  };
  auto add_conv = [&](ConvRef& c, const std::string& conv_name, const std::string& bn_name, int cin, int cout, int k,
                      int stride, int kind, int stage) {
    c.shape.Cin = cin; c.shape.Cout = cout; c.shape.k = k; c.shape.stride = stride; c.shape.kind = kind;
    c.stage = stage;
    c.w_off = add_param(conv_name + ".weight", {cout, cin, k, k});
    c.bn.C = cout;
    c.bn.gamma_off = add_param(bn_name + ".weight", {cout});
    c.bn.beta_off = add_param(bn_name + ".bias", {cout});
    c.bn.rm_off = add_buffer(bn_name + ".running_mean", cout);
    c.bn.rv_off = add_buffer(bn_name + ".running_var", cout);
    c.bn.scratch_off = n_bn_scratch_;
    n_bn_scratch_ += 4 * cout;
    c.bn.stat_off = n_bn_stats_;   // in units of "channels"; scaled by 2 * max_stat_slots_ at bind time
    n_bn_stats_ += cout;
    const int64_t packed_elems = (kind == 1) ? 64 * 256 : static_cast<int64_t>(cout) * cin * k * k;
    c.packed_off = n_packed_;
    n_packed_ += (packed_elems + 63) / 64 * 64;
    // the fp32 packed-gradient scratch mirrors the packed bf16 arena (same offsets), so one table serves both
    if (k > 1) c.gpacked_off = c.packed_off;
    n_gpacked_ = n_packed_;
    WeightPackEntry e;
    e.src_off = c.w_off;
    e.dst_off = c.packed_off;
    e.cout = cout; e.cin = cin; e.kk = k * k; e.kind = kind;
    pack_table_.push_back(e);
    pack_table_stage_.push_back(stage);
  };

  // segments in network order: stem+layer1 (stage 3), layer2 (2), layer3 (1), layer4+fc+head (0)
  stage_begin_[0] = 0;
  add_conv(stem_, "resnet.conv1", "resnet.bn1", 3, 64, 7, 2, 1, 3);
  const int depth[4] = {3, 4, 6, 3};
  const int width[4] = {64, 128, 256, 512};
  int in_ch = 64;
  for (int L = 0; L < 4; ++L) {
    const int stage = 3 - (L == 0 ? 0 : L);  // layer1 -> 3, layer2 -> 2, layer3 -> 1, layer4 -> 0
    if (L > 0) stage_begin_[L] = n_param_elems_;
    for (int b = 0; b < depth[L]; ++b) {
      const std::string base = "resnet.layer" + std::to_string(L + 1) + "." + std::to_string(b);
      const int stride = (b == 0 && L > 0) ? 2 : 1;
      BlockRef blk;
      add_conv(blk.c1, base + ".conv1", base + ".bn1", in_ch, width[L], 1, 1, 0, stage);
      add_conv(blk.c2, base + ".conv2", base + ".bn2", width[L], width[L], 3, stride, 0, stage);
      add_conv(blk.c3, base + ".conv3", base + ".bn3", width[L], width[L] * 4, 1, 1, 0, stage);
      if (b == 0) {
        blk.has_ds = true;
        add_conv(blk.ds, base + ".downsample.0", base + ".downsample.1", in_ch, width[L] * 4, 1, stride, 0, stage);
      }
      blocks_.push_back(blk);
      in_ch = width[L] * 4;
    }
  }
  stage_begin_[4] = 0;  // unused
  // fc + head (belong to stage 0 together with layer4)
  fc_.shape.Cin = 2048; fc_.shape.Cout = out_dim_; fc_.shape.k = 1; fc_.shape.stride = 1; fc_.shape.kind = 0;
  fc_.stage = 0;
  fc_.w_off = add_param("resnet.fc.weight", {out_dim_, 2048});
  fc_bias_off_ = add_param("resnet.fc.bias", {out_dim_});
  fc_.packed_off = n_packed_;
  n_packed_ += static_cast<int64_t>(out_dim_) * 2048;
  {
    WeightPackEntry e;
    e.src_off = fc_.w_off; e.dst_off = fc_.packed_off; e.cout = out_dim_; e.cin = 2048; e.kk = 1; e.kind = 0;
    pack_table_.push_back(e);
    pack_table_stage_.push_back(0);
  }
  const int hin[3] = {n_cams_ * out_dim_, 128, 128};
  const int hout[3] = {128, 128, 6};
  for (int i = 0; i < 3; ++i) {
    const std::string base = "output_mlp." + std::to_string(2 * i);
    head_w_off_[i] = add_param(base + ".weight", {hout[i], hin[i]});
    head_b_off_[i] = add_param(base + ".bias", {hout[i]});
  }
}

void Model::stage_param_range(int stage, int64_t* begin, int64_t* end) const {
  // stage 0: layer4 + fc + head, 1: layer3, 2: layer2, 3: stem + layer1
  ARGUS_CHECK(stage >= 0 && stage < 4, "stage out of range");
  const int64_t seg_begin[4] = {stage_begin_[3], stage_begin_[2], stage_begin_[1], 0};
  const int64_t seg_end[4] = {n_param_elems_, stage_begin_[3], stage_begin_[2], stage_begin_[1]};
  *begin = seg_begin[stage];
  *end = seg_end[stage];
}

void Model::bind(float* params, float* grads, float* buffers) {
  require_sm100();
  params_dev_ = params;
  grads_dev_ = grads;
  buffers_dev_ = buffers;
  if (packed_ == nullptr) {
    ARGUS_CUDA(cudaMalloc(&packed_, n_packed_ * sizeof(bf16)));
    ARGUS_CUDA(cudaMalloc(&gpacked_, std::max<int64_t>(n_gpacked_, 1) * sizeof(float)));
    ARGUS_CUDA(cudaMalloc(&bn_scratch_, n_bn_scratch_ * sizeof(float)));
    max_stat_slots_ = 4 * num_sms();   // up to four epilogue groups per CTA
    ARGUS_CUDA(cudaMalloc(&bn_stats_, n_bn_stats_ * 2 * max_stat_slots_ * sizeof(float)));
    ARGUS_CUDA(cudaMalloc(&bn_bwd_scratch_, bn_bwd_scratch_elems() * sizeof(float)));
    {
      const char* e = getenv("ARGUS_BN_ALGEBRA");
      bn_algebra_ = !(e && e[0] == '0');
      // Fused block tail in the training forward (default; ARGUS_FUSED_TAIL=0 selects the separate passes): bn3's batch
      // statistics come from the Gram matrix of act2 (kept for the algebraic backward, which then only needs H = g^T act2),
      // conv3 applies BN + identity + ReLU + the bit mask in its epilogue and raw3 is never written: 10 instead of 17
      // narrow-tensor passes per block tail. Round 1 measured it SLOWER (45.2 vs 44.1 ms: 8 epilogue warps, ~1 000
      // instructions per 64-column chunk, coefficient loads stalling every FMUL / FADD); with the packed-fp32 epilogue, the
      // coefficients in shared memory and the group barrier removed from the residual path it is 1.0-1.2 ms per step
      // FASTER (profiles/r2_fused_tail_ab.txt).
      const char* ft = getenv("ARGUS_FUSED_TAIL");
      fused_tail_ = !(ft && ft[0] == '0');
      // eligible: bottlenecks whose mid width is <= 256 (layers 1-3); layer4's small matrices would cost more than the
      // two passes over its (small) activations
      for (const auto& b : blocks_)
        if (b.c1.shape.Cout <= 256) {
          alg_max_o_ = std::max(alg_max_o_, b.c3.shape.Cout);
          alg_max_c_ = std::max(alg_max_c_, b.c1.shape.Cout);
          if (b.has_ds && b.ds.shape.Cin <= 256) alg_max_c_ = std::max(alg_max_c_, b.ds.shape.Cin);
        }
      const size_t O = alg_max_o_, C = alg_max_c_;
      ARGUS_CUDA(cudaMalloc(&alg_h_, (O + C) * C * sizeof(float)));   // H [O][C] followed by the Gram matrix [C][C]
      ARGUS_CUDA(cudaMalloc(&alg_s_, C * sizeof(float)));
      ARGUS_CUDA(cudaMalloc(&alg_k1k0_, 2 * O * sizeof(float)));
      ARGUS_CUDA(cudaMalloc(&alg_bias_, C * sizeof(float)));
      ARGUS_CUDA(cudaMalloc(&alg_gstats_, static_cast<size_t>(max_stat_slots_) * 2 * O * sizeof(float)));
      ARGUS_CUDA(cudaMalloc(&alg_bstack_, (O + C) * C * sizeof(bf16)));
      ARGUS_CUDA(cudaMalloc(&alg_mpartial_, bn_alg_matrix_scratch_elems(static_cast<int>(C)) * sizeof(float)));
    }
    {
      // BN-backward reduction in the epilogue of the dgrad that produces the gradient: OPT-IN (ARGUS_BN_REDUCE_FUSED=1
      // fuses layers 1-2, =2 every eligible layer). It saves 0.3 ms per step, but with it and the separate block tail the
      // bench trajectory stopped reproducing from run to run once the look-ahead staging started (0 of 7 runs; 9 of 9
      // with the fused tail; every other mode 100 % -- profiles/r2_determinism.md), and the cause was not found.
      const char* e = getenv("ARGUS_BN_REDUCE_FUSED");
      bn_reduce_fused_ = e ? atoi(e) : 0;
      ARGUS_CUDA(cudaMalloc(&bnred_stats_, static_cast<size_t>(max_stat_slots_) * 2 * 512 * sizeof(float)));
    }
    ARGUS_CUDA(cudaMalloc(&pack_table_dev_, pack_table_.size() * sizeof(WeightPackEntry)));
    ARGUS_CUDA(cudaMemcpy(pack_table_dev_, pack_table_.data(), pack_table_.size() * sizeof(WeightPackEntry),
                          cudaMemcpyHostToDevice));
    ARGUS_CUDA(cudaMemset(gpacked_, 0, std::max<int64_t>(n_gpacked_, 1) * sizeof(float)));
    ARGUS_CUDA(cudaStreamCreateWithFlags(&side_, cudaStreamNonBlocking));
    if (const char* e = getenv("ARGUS_WGRAD_OVERLAP")) overlap_wgrad_ = (e[0] != '0');   // A/B switch, default on
    ARGUS_CUDA(cudaEventCreateWithFlags(&ev_fork_, cudaEventDisableTiming));
    ARGUS_CUDA(cudaEventCreateWithFlags(&ev_wgrad_, cudaEventDisableTiming));
  }
  plans_.clear();
  last_train_plan_ = nullptr;
  last_frozen_plan_ = nullptr;
  last_grad_forward_ = 0;
  last_plan_ = nullptr;
  staged_plan_ = nullptr;
  eval_fold_dirty_ = true;
}

void Model::sync_weights(cudaStream_t s) {
  ARGUS_CHECK(params_dev_ != nullptr, "model is not bound to a parameter arena");
  pack_weights(params_dev_, packed_, pack_table_dev_, static_cast<int>(pack_table_.size()), s);
  eval_fold_dirty_ = true;
}

void Model::zero_grads(cudaStream_t s) {
  ARGUS_CHECK(grads_dev_ != nullptr, "model is not bound to a gradient arena");
  ARGUS_CUDA(cudaMemsetAsync(grads_dev_, 0, n_param_elems_ * sizeof(float), s)); pdl_break(s, kPdlAfterMemop);
}

// ------------------------------------------------------------------------------------------------------------
// planning
// ------------------------------------------------------------------------------------------------------------
template <typename T>
T* Model::arena_alloc(size_t count) {
  const size_t bytes = (count * sizeof(T) + 1023) / 1024 * 1024;
  uint8_t* p = arena_ ? arena_ + arena_used_ : nullptr;
  arena_used_ += bytes;
  return reinterpret_cast<T*>(p);
}

void Model::reserve(int max_batch, int H, int W, bool training, bool frozen) {
  ARGUS_CHECK(max_batch > 0, "batch must be positive");
  ARGUS_CHECK(is_pow2(H) && is_pow2(W) && H >= 32 && W >= 32, "H and W must be powers of two >= 32");
  // dry run to size the arena
  uint8_t* saved = arena_;
  arena_ = nullptr;
  Plan tmp;
  tmp.B = max_batch; tmp.H = H; tmp.W = W; tmp.N = max_batch * n_cams_; tmp.training = training; tmp.frozen = frozen;
  arena_used_ = 0;
  // build_plan only measures when arena_ == nullptr
  build_plan(tmp);
  const size_t need = arena_used_;
  arena_ = saved;
  const size_t stem_need = training ? static_cast<size_t>(max_batch) * n_cams_ * (H / 2) * (W / 2 + 4) * 16 : 0;
  if (stem_need > stem_in_elems_) {
    // (plan-build time only) every stream of this model must be idle before the staging buffers move
    ARGUS_CUDA(cudaDeviceSynchronize());
    for (int b = 0; b < 2; ++b) {
      if (stem_in_[b]) ARGUS_CUDA(cudaFree(stem_in_[b]));
      stem_in_[b] = nullptr;
      ARGUS_CUDA(cudaMalloc(&stem_in_[b], stem_need * sizeof(bf16)));
    }
    stem_in_elems_ = stem_need;
    plans_.clear();
    last_train_plan_ = nullptr;
    last_frozen_plan_ = nullptr;
    last_grad_forward_ = 0;
    last_plan_ = nullptr;
    staged_plan_ = nullptr;
  }
  if (need > arena_bytes_) {
    if (arena_) ARGUS_CUDA(cudaFree(arena_));
    arena_ = nullptr;
    ARGUS_CUDA(cudaMalloc(&arena_, need));
    arena_bytes_ = need;
    plans_.clear();
    last_train_plan_ = nullptr;
    last_frozen_plan_ = nullptr;
    last_grad_forward_ = 0;
    last_plan_ = nullptr;
    staged_plan_ = nullptr;
  }
  reserved_batch_ = std::max(reserved_batch_, max_batch);
  reserved_h_ = H; reserved_w_ = W;
  reserved_training_ = reserved_training_ || training;
}

Plan& Model::get_plan(int B, int H, int W, bool training, bool frozen) {
  auto key = std::make_tuple(B, H, W, training, frozen);
  auto it = plans_.find(key);
  if (it != plans_.end()) return *it->second;
  if (frozen) ensure_frozen_buffers();
  reserve(B, H, W, training, frozen);  // grows the arena if needed (and drops stale plans)
  auto p = std::make_unique<Plan>();
  p->B = B; p->H = H; p->W = W; p->N = B * n_cams_; p->training = training; p->frozen = frozen;
  arena_used_ = 0;
  build_plan(*p);
  ARGUS_CHECK(arena_used_ <= arena_bytes_, "activation arena overflow");
  Plan& ref = *p;
  plans_[key] = std::move(p);
  return ref;
}

void Model::build_plan(Plan& p) {
  const bool real = (arena_ != nullptr);  // dry runs only measure
  const int N = p.N, H = p.H, W = p.W;
  const bool tr = p.training;
  const bool fz = p.frozen;   // eval layout + bit masks + backward scratch
  auto plan_conv = [&](ConvPlan& cp, ConvRef& c, int n, int h, int w, const bf16* in, bf16* out_raw,
                       bool want_dgrad) {
    c.shape.N = n; c.shape.H = h; c.shape.W = w;
    if (!real) return;
    cp.fwd = plan_conv_forward(c.shape, in, packed_ + c.packed_off, out_raw);
    cp.has_dgrad = want_dgrad;
  };
  // ---- stem (training plans read the model-level double buffer; an eval plan owns a private input in the arena)
  if (!tr) p.x_in = arena_alloc<bf16>(static_cast<size_t>(N) * (H / 2) * (W / 2 + 4) * 16);
  const int H1 = H / 2, W1 = W / 2;  // stem output
  const int H2 = H1 / 2, W2 = W1 / 2;  // after max pooling
  const size_t stem_elems = static_cast<size_t>(N) * H1 * W1 * 64;
  if (tr) p.raw0 = arena_alloc<bf16>(stem_elems); else p.act0 = arena_alloc<bf16>(stem_elems);
  p.pooled0 = arena_alloc<bf16>(stem_elems / 4);
  if (tr || fz) p.idx0 = arena_alloc<uint8_t>(stem_elems / 4);
  plan_conv(p.stem, stem_, N, H, W, tr ? stem_in_[0] : p.x_in, tr ? p.raw0 : p.act0, false);
  if (real) {
    ARGUS_CHECK(!tr || static_cast<size_t>(N) * (H / 2) * (W / 2 + 4) * 16 <= stem_in_elems_, "stem input buffers too small");
    for (int b = 0; b < 2; ++b)
      p.stem_fwd_buf[b] = plan_conv_forward(stem_.shape, tr ? stem_in_[b] : p.x_in, packed_ + stem_.packed_off,
                                            tr ? p.raw0 : p.act0);
  }

  // ---- bottleneck blocks
  p.blocks.assign(blocks_.size(), BlockPlan());
  bf16* x = p.pooled0;
  int h = H2, w = W2;
  size_t max_elems = stem_elems;
  for (size_t i = 0; i < blocks_.size(); ++i) {
    BlockRef& br = blocks_[i];
    BlockPlan& bp = p.blocks[i];
    const int s = br.c2.shape.stride;
    const int ho = h / s, wo = w / s;
    const size_t e_in = static_cast<size_t>(N) * h * w;
    const size_t e_out = static_cast<size_t>(N) * ho * wo;
    bp.x = x;
    bp.rows_in = e_in; bp.rows_mid = e_in; bp.rows_out = e_out;
    bp.x_bytes = e_in * br.c1.shape.Cin * sizeof(bf16);
    const int wd = br.c1.shape.Cout, oc = br.c3.shape.Cout;
    if (tr) bp.raw1 = arena_alloc<bf16>(e_in * wd);
    bp.act1 = arena_alloc<bf16>(e_in * wd);
    if (tr) bp.raw2 = arena_alloc<bf16>(e_out * wd);
    bp.act2 = arena_alloc<bf16>(e_out * wd);
    bp.fused_tail = tr && bn_algebra_ && fused_tail_ && wd <= 256;
    if (tr && !bp.fused_tail) bp.raw3 = arena_alloc<bf16>(e_out * oc);
    if (br.has_ds) bp.rawd = arena_alloc<bf16>(e_out * oc);  // eval / fused tail: holds the folded-BN identity branch
    bp.out = arena_alloc<bf16>(e_out * oc);
    if (tr || fz) bp.out_bits = arena_alloc<uint8_t>(e_out * oc / 8);
    if (fz) {
      bp.act1_bits = arena_alloc<uint8_t>(e_in * wd / 8);
      bp.act2_bits = arena_alloc<uint8_t>(e_out * wd / 8);
    }
    if (tr && bn_algebra_ && wd <= 256)
      bp.act2_colsum = arena_alloc<float>(static_cast<size_t>(bn_apply_grid(static_cast<int64_t>(e_out), wd)) * wd);
    if (bp.fused_tail) {
      // (C x C Gram matrix followed by the C column sums of the same activation)
      bp.gram_saved = arena_alloc<float>(static_cast<size_t>(wd) * wd + wd);
      if (br.has_ds && br.ds.shape.Cin <= 256)
        bp.ds_gram_saved = arena_alloc<float>(static_cast<size_t>(br.ds.shape.Cin) * br.ds.shape.Cin + br.ds.shape.Cin);
    }
    max_elems = std::max(max_elems, std::max(e_in * std::max(wd, br.c1.shape.Cin), e_out * oc));
    plan_conv(bp.c1, br.c1, N, h, w, bp.x, tr ? bp.raw1 : bp.act1, true);
    plan_conv(bp.c2, br.c2, N, h, w, bp.act1, tr ? bp.raw2 : bp.act2, true);
    plan_conv(bp.c3, br.c3, N, ho, wo, bp.act2, (tr && !bp.fused_tail) ? bp.raw3 : bp.out, true);
    if (br.has_ds) plan_conv(bp.ds, br.ds, N, h, w, bp.x, bp.rawd, true);
    if (real && bp.fused_tail) {
      bp.fwd_gram = plan_gram(br.c3.shape, bp.act2, bp.gram_saved);
      ensure_wgrad_scratch(bp.fwd_gram);
      if (br.has_ds && br.ds.shape.Cin <= 256) {
        bp.ds_fwd_gram = plan_gram(br.ds.shape, bp.x, bp.ds_gram_saved);
        ensure_wgrad_scratch(bp.ds_fwd_gram);
      }
    }
    x = bp.out;
    h = ho; w = wo;
  }
  p.final_hw = h * w;
  // ---- pooling, fc, head
  p.pooled = arena_alloc<bf16>(static_cast<size_t>(N) * 2048);
  p.feat = arena_alloc<bf16>(static_cast<size_t>(N) * out_dim_);
  plan_conv(p.fc, fc_, N, 1, 1, p.pooled, p.feat, true);
  const int B = p.B, F = n_cams_ * out_dim_;
  p.z0 = arena_alloc<float>(static_cast<size_t>(B) * F);
  p.h1 = arena_alloc<float>(static_cast<size_t>(B) * 128);
  p.a1 = arena_alloc<float>(static_cast<size_t>(B) * 128);
  p.h2 = arena_alloc<float>(static_cast<size_t>(B) * 128);
  p.a2 = arena_alloc<float>(static_cast<size_t>(B) * 128);
  p.out = arena_alloc<float>(static_cast<size_t>(B) * 8);
  if (!tr && !fz) return;

  // ---- backward scratch
  p.d_out = arena_alloc<float>(static_cast<size_t>(B) * 8);
  p.d_a2 = arena_alloc<float>(static_cast<size_t>(B) * 128);
  p.d_a1 = arena_alloc<float>(static_cast<size_t>(B) * 128);
  p.d_z0 = arena_alloc<float>(static_cast<size_t>(B) * F);
  p.d_feat = arena_alloc<bf16>(static_cast<size_t>(N) * out_dim_);
  p.d_pooled = arena_alloc<bf16>(static_cast<size_t>(N) * 2048);
  bf16* G[5];
  for (int i = 0; i < 5; ++i) G[i] = arena_alloc<bf16>(max_elems);
  if (real) {
    p.fc.wgrad = plan_conv_wgrad(fc_.shape, p.d_feat, p.pooled, grads_dev_ + fc_.w_off);
    ensure_wgrad_scratch(p.fc.wgrad);
    p.fc.dgrad = plan_conv_dgrad(fc_.shape, p.d_feat, packed_ + fc_.packed_off, p.d_pooled);
  }
  if (fz) {
    // Per block: P = the masked block-output gradient, Q = g2 (conv3 dgrad, masked by act2's bits), R = g1 (conv2 dgrad,
    // masked by act1's bits), S = the block-input gradient (conv1 dgrad + identity branch), T = the downsample dgrad.
    // Weight gradients: H = g^T x into frz_h_ (1x1) or the packed scratch (3x3, stem); dgrads against diag(sc) W.
    bf16 *P = G[0], *Q = G[1], *R = G[2], *S = G[3], *T = G[4];
    for (int i = static_cast<int>(blocks_.size()) - 1; i >= 0; --i) {
      BlockRef& br = blocks_[i];
      BlockPlan& bp = p.blocks[i];
      bf16* Tb = (br.has_ds && br.ds.shape.stride == 2) ? arena_alloc<bf16>(bp.x_bytes / sizeof(bf16)) : T;
      bp.g_out = P; bp.g_q = Q; bp.g_r = R; bp.g_t = Tb; bp.g_x = S;
      if (real) {
        auto Ws = [&](const ConvRef& c) { return packed_scaled_ + c.packed_off; };
        bp.c3.wgrad = plan_conv_wgrad(br.c3.shape, P, bp.act2, frz_h_);
        bp.c3.dgrad = plan_conv_dgrad(br.c3.shape, P, Ws(br.c3), Q);
        if (br.has_ds) {
          bp.ds.wgrad = plan_conv_wgrad(br.ds.shape, P, bp.x, frz_h_);
          bp.ds.dgrad = plan_conv_dgrad(br.ds.shape, P, Ws(br.ds), Tb);
          ensure_wgrad_scratch(bp.ds.wgrad);
        }
        bp.c2.wgrad = plan_conv_wgrad(br.c2.shape, Q, bp.act1, gpacked_ + br.c2.gpacked_off);
        bp.c2.dgrad = plan_conv_dgrad(br.c2.shape, Q, Ws(br.c2), R);
        bp.c1.wgrad = plan_conv_wgrad(br.c1.shape, R, bp.x, frz_h_);
        bp.c1.dgrad = plan_conv_dgrad(br.c1.shape, R, Ws(br.c1), S);
        ensure_wgrad_scratch(bp.c1.wgrad);
        ensure_wgrad_scratch(bp.c2.wgrad);
        ensure_wgrad_scratch(bp.c3.wgrad);
      }
      std::swap(P, S);
    }
    p.g_stem_in = P;
    p.g_raw0 = Q;   // g0
    if (real) {
      p.stem.wgrad = plan_conv_wgrad(stem_.shape, Q, p.x_in, gpacked_ + stem_.gpacked_off);
      ensure_wgrad_scratch(p.stem.wgrad);
    }
    return;
  }
  // rotate the five scratch buffers through the blocks in reverse order (see Model::backward)
  bf16 *P = G[0], *Q = G[1], *R = G[2], *S = G[3], *T = G[4];
  for (int i = static_cast<int>(blocks_.size()) - 1; i >= 0; --i) {
    BlockRef& br = blocks_[i];
    BlockPlan& bp = p.blocks[i];
    // stride-2 downsample blocks get a private, persistently zero-filled gradient buffer (see BlockPlan::t_zero_epoch)
    bf16* Tb = (br.has_ds && br.ds.shape.stride == 2) ? arena_alloc<bf16>(bp.x_bytes / sizeof(bf16)) : T;
    bp.g_out = P; bp.g_q = Q; bp.g_r = R; bp.g_t = Tb; bp.g_x = S;
    if (real) {
      auto wg_dst = [&](const ConvRef& c) { return c.gpacked_off >= 0 ? gpacked_ + c.gpacked_off : grads_dev_ + c.w_off; };
      // conv3: dy = Q (dRaw3), input act2, dx -> R
      bp.c3.wgrad = plan_conv_wgrad(br.c3.shape, Q, bp.act2, wg_dst(br.c3));
      bp.c3.dgrad = plan_conv_dgrad(br.c3.shape, Q, packed_ + br.c3.packed_off, R);
      bp.algebraic = bn_algebra_ && br.c1.shape.Cout <= 256;
      if (bp.algebraic) {
        // algebraic bn3 backward: GEMMs on the masked gradient P itself (never on dRaw3)
        const int C = br.c3.shape.Cin;
        bp.hg_wgrad = bp.gram_saved ? plan_conv_wgrad(br.c3.shape, P, bp.act2, alg_h_)
                                    : plan_conv_wgrad_gram(br.c3.shape, P, bp.act2, alg_h_);
        bp.c3_concat = plan_dgrad_concat(br.c3.shape, P, bp.act2, C, alg_bstack_, R);
        ensure_wgrad_scratch(bp.hg_wgrad);
      }
      bp.ds_algebraic = bp.algebraic && br.has_ds && br.ds.shape.Cin <= 256;   // layer1.0, layer2.0
      if (bp.ds_algebraic) {
        const int C = br.ds.shape.Cin;
        bp.ds_hg_wgrad = bp.ds_gram_saved ? plan_conv_wgrad(br.ds.shape, P, bp.x, alg_h_)
                                          : plan_conv_wgrad_gram(br.ds.shape, P, bp.x, alg_h_);
        bp.ds_concat = plan_dgrad_concat(br.ds.shape, P, bp.x, C, alg_bstack_, Tb);
        ensure_wgrad_scratch(bp.ds_hg_wgrad);
      }
      // conv2: dy = Q (dRaw2), input act1, dx -> R
      bp.c2.wgrad = plan_conv_wgrad(br.c2.shape, Q, bp.act1, wg_dst(br.c2));
      bp.c2.dgrad = plan_conv_dgrad(br.c2.shape, Q, packed_ + br.c2.packed_off, R);
      // conv1: dy = Q (dRaw1), input x, dx -> S (+ residual)
      bp.c1.wgrad = plan_conv_wgrad(br.c1.shape, Q, bp.x, wg_dst(br.c1));
      bp.c1.dgrad = plan_conv_dgrad(br.c1.shape, Q, packed_ + br.c1.packed_off, S);
      if (br.has_ds) {
        // downsample: dy = R (dRawd), input x, dx -> T
        bp.ds.wgrad = plan_conv_wgrad(br.ds.shape, R, bp.x, wg_dst(br.ds));
        bp.ds.dgrad = plan_conv_dgrad(br.ds.shape, R, packed_ + br.ds.packed_off, Tb);
        ensure_wgrad_scratch(bp.ds.wgrad);
      }
      ensure_wgrad_scratch(bp.c1.wgrad);
      ensure_wgrad_scratch(bp.c2.wgrad);
      ensure_wgrad_scratch(bp.c3.wgrad);
    }
    std::swap(P, S);  // this block's input gradient is the previous block's output gradient
  }
  p.g_stem_in = P;
  p.g_act0 = Q;
  p.g_raw0 = R;
  if (real) {
    for (int b = 0; b < 2; ++b)
      p.stem_wgrad_buf[b] = plan_conv_wgrad(stem_.shape, R, stem_in_[b], gpacked_ + stem_.gpacked_off);
    p.stem.wgrad = p.stem_wgrad_buf[0];
    ensure_wgrad_scratch(p.stem.wgrad);
  }
}

// ------------------------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------------------------
void Model::fold_eval(cudaStream_t s) {
  auto fold = [&](const ConvRef& c) {
    float* sc = bn_scratch_ + c.bn.scratch_off;
    bn_fold_eval(params_dev_ + c.bn.gamma_off, params_dev_ + c.bn.beta_off, buffers_dev_ + c.bn.rm_off,
                 buffers_dev_ + c.bn.rv_off, kBnEps, sc, sc + c.bn.C, c.bn.C, s, sc + 2 * c.bn.C, sc + 3 * c.bn.C);
  };
  fold(stem_);
  for (auto& b : blocks_) {
    fold(b.c1); fold(b.c2); fold(b.c3);
    if (b.has_ds) fold(b.ds);
  }
  eval_fold_dirty_ = false;
  scaled_dirty_ = true;
}

void Model::run_conv_train(const ConvPlan& cp, const ConvRef& c, int64_t rows, cudaStream_t s) {
  Epilogue e;
  e.stat_partial = bn_stats_ + c.bn.stat_off * 2 * max_stat_slots_;
  launch_conv(cp.fwd, e, s);
  float* sc = bn_scratch_ + c.bn.scratch_off;
  bn_finalize(e.stat_partial, stat_slots(cp.fwd), static_cast<double>(rows), params_dev_ + c.bn.gamma_off,
              params_dev_ + c.bn.beta_off, buffers_dev_ + c.bn.rm_off, buffers_dev_ + c.bn.rv_off, kBnMomentum, kBnEps,
              sc, sc + c.bn.C, sc + 2 * c.bn.C, sc + 3 * c.bn.C, c.bn.C, s);
}

void Model::forward_train(Plan& p, cudaStream_t s) {
  ARGUS_CUDA(cudaMemsetAsync(bn_stats_, 0, n_bn_stats_ * 2 * max_stat_slots_ * sizeof(float), s)); pdl_break(s, kPdlAfterMemop);
  eval_fold_dirty_ = true;  // scale/shift scratch now holds batch statistics
  const int N = p.N;
  auto SC = [&](const ConvRef& c) { return bn_scratch_ + c.bn.scratch_off; };
  run_conv_train(p.stem, stem_, static_cast<int64_t>(N) * (p.H / 2) * (p.W / 2), s);
  maxpool_fwd(p.raw0, SC(stem_), SC(stem_) + 64, p.pooled0, p.idx0, N, p.H / 2, p.W / 2, 64, s);
  for (size_t i = 0; i < blocks_.size(); ++i) {
    BlockRef& br = blocks_[i];
    BlockPlan& bp = p.blocks[i];
    const int wd = br.c1.shape.Cout, oc = br.c3.shape.Cout;
    run_conv_train(bp.c1, br.c1, bp.rows_in, s);
    bn_apply(bp.raw1, SC(br.c1), SC(br.c1) + wd, nullptr, nullptr, nullptr, 1, bp.act1, nullptr, nullptr, bp.rows_in, wd, s);
    run_conv_train(bp.c2, br.c2, bp.rows_out, s);
    bn_apply(bp.raw2, SC(br.c2), SC(br.c2) + wd, nullptr, nullptr, nullptr, 1, bp.act2, nullptr, bp.act2_colsum,
             bp.rows_out, wd, s);
    if (bp.fused_tail) {
      // bn3 statistics from the Gram matrix of act2; conv3 then finishes the block in its epilogue
      stats_from_gram(br.c3, bp.fwd_gram, bp.gram_saved, bp.act2, bp.act2_colsum, bp.rows_out, N, s);
      Epilogue e;
      e.scale = SC(br.c3);
      e.shift = SC(br.c3) + oc;
      e.relu = 1;
      e.relu_bits_out = bp.out_bits;
      e.residual = bp.x;
      if (br.has_ds) {
        e.residual = bp.rawd;
        if (br.ds.shape.Cin <= 256) {
          // downsample branch the same way: its batch norm is folded into its own epilogue
          stats_from_gram(br.ds, bp.ds_fwd_gram, bp.ds_gram_saved, bp.x, nullptr, bp.rows_out, N, s);
          Epilogue d;
          d.scale = SC(br.ds);
          d.shift = SC(br.ds) + oc;
          launch_conv(bp.ds.fwd, d, s);
        } else {
          run_conv_train(bp.ds, br.ds, bp.rows_out, s);   // raw downsample output + statistics, normalised on the fly
          e.res_scale = SC(br.ds);
          e.res_shift = SC(br.ds) + oc;
        }
      }
      launch_conv(bp.c3.fwd, e, s);
      continue;
    }
    run_conv_train(bp.c3, br.c3, bp.rows_out, s);
    if (br.has_ds) {
      run_conv_train(bp.ds, br.ds, bp.rows_out, s);
      bn_apply(bp.raw3, SC(br.c3), SC(br.c3) + oc, bp.rawd, SC(br.ds), SC(br.ds) + oc, 1, bp.out, bp.out_bits, nullptr,
               bp.rows_out, oc, s);
    } else {
      bn_apply(bp.raw3, SC(br.c3), SC(br.c3) + oc, bp.x, nullptr, nullptr, 1, bp.out, bp.out_bits, nullptr, bp.rows_out,
               oc, s);
    }
  }
}

void Model::stats_from_gram(const ConvRef& c, const WgradLaunch& gram, float* G, const bf16* act, const float* colsum_partial,
                            int64_t rows, int N, cudaStream_t s) {
  const int O = c.shape.Cout, C = c.shape.Cin;
  ARGUS_CUDA(cudaMemsetAsync(G, 0, static_cast<size_t>(C) * C * sizeof(float), s)); pdl_break(s, kPdlAfterMemop);
  launch_wgrad(gram, wgrad_scratch_, s);
  float* colsum = G + static_cast<size_t>(C) * C;   // kept next to the Gram matrix for the backward pass
  if (colsum_partial != nullptr) colsum_finalize(colsum_partial, bn_apply_grid(rows, C), colsum, C, s);
  else colsum_pixels_bf16(act, N, c.shape.H, c.shape.W, C, c.shape.stride, bn_bwd_scratch_, colsum, s);
  float* sc = bn_scratch_ + c.bn.scratch_off;
  bn_stats_from_gram(packed_ + c.packed_off, G, colsum, static_cast<double>(rows), params_dev_ + c.bn.gamma_off,
                     params_dev_ + c.bn.beta_off, buffers_dev_ + c.bn.rm_off, buffers_dev_ + c.bn.rv_off, kBnMomentum,
                     kBnEps, sc, sc + O, sc + 2 * O, sc + 3 * O, alg_mpartial_, O, C, s);
}

// Eval plans and frozen plans run the same launches; a frozen plan's epilogues also write the ReLU bit masks and its
// max pooling the arg-max bytes (null pointers in an eval plan), which leaves every output bit as it is.
void Model::forward_eval(Plan& p, cudaStream_t s) {
  if (eval_fold_dirty_) fold_eval(s);
  if (p.frozen && scaled_dirty_) {
    pack_weights_scaled(params_dev_, bn_scratch_, scaled_scale_off_dev_, packed_scaled_, scaled_table_dev_,
                        n_scaled_entries_, s);
    scaled_dirty_ = false;
  }
  const int N = p.N;
  auto EP = [&](const ConvRef& c, const bf16* res, int relu, uint8_t* bits) {
    Epilogue e;
    e.scale = bn_scratch_ + c.bn.scratch_off;
    e.shift = e.scale + c.bn.C;
    e.residual = res;
    e.relu = relu;
    e.relu_bits_out = bits;
    e.early_trigger = 1;   // inference chain: the next convolution sets itself up while this one runs
    return e;
  };
  launch_conv(p.stem.fwd, EP(stem_, nullptr, 1, nullptr), s);
  maxpool_fwd(p.act0, nullptr, nullptr, p.pooled0, p.idx0, N, p.H / 2, p.W / 2, 64, s);
  for (size_t i = 0; i < blocks_.size(); ++i) {
    BlockRef& br = blocks_[i];
    BlockPlan& bp = p.blocks[i];
    launch_conv(bp.c1.fwd, EP(br.c1, nullptr, 1, bp.act1_bits), s);
    launch_conv(bp.c2.fwd, EP(br.c2, nullptr, 1, bp.act2_bits), s);
    const bf16* identity = bp.x;
    if (br.has_ds) {
      launch_conv(bp.ds.fwd, EP(br.ds, nullptr, 0, nullptr), s);
      identity = bp.rawd;
    }
    launch_conv(bp.c3.fwd, EP(br.c3, identity, 1, bp.out_bits), s);
  }
}

void Model::head_forward(Plan& p, float* out, cudaStream_t s) {
  const int N = p.N, B = p.B, F = n_cams_ * out_dim_;
  avgpool_fwd(p.blocks.back().out, p.pooled, N, p.final_hw, 2048, s);
  Epilogue e;
  e.shift = params_dev_ + fc_bias_off_;
  launch_conv(p.fc.fwd, e, s);
  // (N, out_dim) row-major == (B, n_cams*out_dim): views of one sample are adjacent (argus/models.py:87)
  gelu_fwd_bf16(p.feat, p.z0, static_cast<int64_t>(B) * F, s);
  linear_fwd(p.z0, params_dev_ + head_w_off_[0], params_dev_ + head_b_off_[0], p.h1, p.a1, B, F, 128, s);
  linear_fwd(p.a1, params_dev_ + head_w_off_[1], params_dev_ + head_b_off_[1], p.h2, p.a2, B, 128, 128, s);
  linear_fwd(p.a2, params_dev_ + head_w_off_[2], params_dev_ + head_b_off_[2], p.out, nullptr, B, 128, 6, s);
  ARGUS_CUDA(cudaMemcpyAsync(out, p.out, static_cast<size_t>(B) * 6 * sizeof(float), cudaMemcpyDeviceToDevice, s)); pdl_break(s, kPdlAfterMemop);
}

void Model::forward(const void* x, bool is_u8, int B, int H, int W, bool training, float* out, cudaStream_t s,
                    bool frozen) {
  ARGUS_CHECK(params_dev_ != nullptr && buffers_dev_ != nullptr, "model is not bound");
  ARGUS_CHECK(B > 0, "empty batch");
  ARGUS_CHECK(!training || B * n_cams_ * (H / 32) * (W / 32) > 1,
              "train-mode batch norm needs more than one value per channel");
  ARGUS_CHECK(!(training && frozen), "a frozen-statistics forward is an eval-mode forward");
  ARGUS_CHECK(!frozen || x != nullptr, "the frozen-statistics forward needs the image tensor (no staged input)");
  stem_grad_ready_ = false;
  if (training || frozen) train_input_f32_ = (x != nullptr && !is_u8);
  // which forward backward() differentiates (set after get_plan(), whose arena growth forgets the previous plans)
  auto note_kind = [&] {
    if (training) last_grad_forward_ = 1;
    if (frozen) last_grad_forward_ = 2;
    last_forward_frozen_ = frozen;
  };
  if (precision_ == 1) {
    note_kind();
    forward_fp32(x, is_u8, B, H, W, training, frozen, out, s);
    return;
  }
  Plan& p = get_plan(B, H, W, training, frozen);
  note_kind();
  // every input is written to the alternate stem buffer, which then becomes the current one: a batch staged ahead of
  // time (stage_input_u8 on another stream) never touches the buffer the in-flight pass still reads
  if (x == nullptr) {
    ARGUS_CHECK(staged_plan_ == &p, "forward(x = NULL) needs a preceding stage_input_u8() for the same batch shape");
  } else if (is_u8) {
    pack_input_u8(static_cast<const uint8_t*>(x), training ? stem_in_[cur_in_ ^ 1] : p.x_in, p.N, H, W, s);
  } else {
    pack_input_f32(static_cast<const float*>(x), training ? stem_in_[cur_in_ ^ 1] : p.x_in, p.N, H, W, s);
  }
  if (training) {
    cur_in_ ^= 1;
    p.stem.fwd = p.stem_fwd_buf[cur_in_];
    p.stem.wgrad = p.stem_wgrad_buf[cur_in_];
  }
  staged_plan_ = nullptr;
  if (last_plan_ != &p) ++arena_epoch_;   // plans share the arena: whatever another plan kept there is gone
  last_plan_ = &p;
  if (training) {
    forward_train(p, s);
    last_train_plan_ = &p;
  } else {
    forward_eval(p, s);
    if (frozen) last_frozen_plan_ = &p;
  }
  head_forward(p, out, s);
}

void Model::stage_input_u8(const uint8_t* images, const float* aug_params, const uint32_t* arc_mask, uint32_t* plasma_ws,
                           int B, int H, int W, bool training, bool apply, cudaStream_t s) {
  ARGUS_CHECK(B > 0, "empty batch");
  ARGUS_CHECK(!apply || aug_params != nullptr, "augmentation needs a parameter table");
  ARGUS_CHECK(precision_ == 0, "the fused augmentation + staging path exists in bf16 mode only");
  Plan& p = get_plan(B, H, W, training);
  fuzz_delay(2, s);
  augment_images(images, true, training ? stem_in_[cur_in_ ^ 1] : p.x_in, true, aug_params, arc_mask, plasma_ws, p.N, H, W,
                 apply, s);
  staged_plan_ = &p;
}

void Model::copy_activation(int index, void* dst, int64_t capacity_elems, int64_t* rows, int* C, cudaStream_t s) {
  ARGUS_CHECK(precision_ == 0, "activation probes exist in bf16 mode only");
  ARGUS_CHECK(last_plan_ != nullptr, "no forward pass has run yet");
  Plan& p = *last_plan_;
  const bf16* src = nullptr;
  int64_t r = 0;
  int c = 0;
  if (index == -1) {
    src = p.pooled0; r = static_cast<int64_t>(p.N) * (p.H / 4) * (p.W / 4); c = 64;
  } else if (index >= 0 && index < static_cast<int>(p.blocks.size())) {
    src = p.blocks[index].out; r = p.blocks[index].rows_out; c = blocks_[index].c3.shape.Cout;
  } else if (index >= 100 && index < 100 + static_cast<int>(p.blocks.size())) {
    src = p.blocks[index - 100].act2; r = p.blocks[index - 100].rows_out; c = blocks_[index - 100].c2.shape.Cout;
  } else if (index == 16) {
    src = p.pooled; r = p.N; c = 2048;
  } else if (index == 17) {
    src = p.feat; r = p.N; c = out_dim_;
  } else {
    throw Error("activation index out of range");
  }
  ARGUS_CHECK(r * c <= capacity_elems, "destination too small for the requested activation");
  ARGUS_CUDA(cudaMemcpyAsync(dst, src, static_cast<size_t>(r) * c * sizeof(bf16), cudaMemcpyDeviceToDevice, s)); pdl_break(s, kPdlAfterMemop);
  if (rows) *rows = r;
  if (C) *C = c;
}

// ------------------------------------------------------------------------------------------------------------
// backward
// ------------------------------------------------------------------------------------------------------------
void Model::ensure_wgrad_scratch(const WgradLaunch& l) {
  const int64_t need = wgrad_scratch_elems(l);
  if (need > wgrad_scratch_elems_) {
    // plan-build time only (never on the hot path); all streams are idle for this model at that point
    ARGUS_CUDA(cudaDeviceSynchronize());
    if (wgrad_scratch_) ARGUS_CUDA(cudaFree(wgrad_scratch_));
    ARGUS_CUDA(cudaMalloc(&wgrad_scratch_, need * sizeof(float)));
    wgrad_scratch_elems_ = need;
  }
}

// All weight-gradient GEMMs of a backward pass run on ONE stream (the side stream when overlapping), so a single
// split-K scratch buffer is enough.
void Model::run_wgrad(const WgradLaunch& l, cudaStream_t s) {
  run_on_side(s, [&](cudaStream_t ss) { launch_wgrad(l, wgrad_scratch_, ss); });
}

// Fork: `work` only needs what the caller's stream has produced so far; it runs on the side stream (on the caller's
// stream when overlap is off or the stream is being captured) and is joined by join_wgrad().
void Model::run_on_side(cudaStream_t s, const std::function<void(cudaStream_t)>& work) {
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  cudaStreamIsCapturing(s, &cap);
  if (!overlap_wgrad_ || cap != cudaStreamCaptureStatusNone) {
    join_wgrad(s);
    work(s);
    return;
  }
  ARGUS_CUDA(cudaEventRecord(ev_fork_, s)); pdl_break(s, kPdlAfterRecord);
  ARGUS_CUDA(cudaStreamWaitEvent(side_, ev_fork_, 0)); pdl_break(side_, kPdlAfterWait);
  fuzz_delay(1, side_);
  work(side_);
  ARGUS_CUDA(cudaEventRecord(ev_wgrad_, side_)); pdl_break(side_, kPdlAfterRecord);
  wgrad_pending_ = true;
}

void Model::join_wgrad(cudaStream_t s) {
  if (wgrad_pending_) {
    ARGUS_CUDA(cudaStreamWaitEvent(s, ev_wgrad_, 0)); pdl_break(s, kPdlAfterWait);
    wgrad_pending_ = false;
  }
}

void Model::bn_backward(const ConvRef& c, bf16* dy, const bf16* raw, const bf16* out, bf16* dx, int64_t rows, int mask,
                        cudaStream_t s) {
  const float* sc = bn_scratch_ + c.bn.scratch_off;
  float* dgamma = grads_dev_ + c.bn.gamma_off;
  float* dbeta = grads_dev_ + c.bn.beta_off;
  const int C = c.bn.C;
  bn_bwd_reduce(dy, raw, out, sc, sc + C, sc + 2 * C, sc + 3 * C, dgamma, dbeta, rows, C, mask, bn_bwd_scratch_, s);
  // the apply pass overwrites a gradient buffer that an in-flight weight-gradient GEMM may still be reading
  join_wgrad(s);
  bn_bwd_apply(dy, raw, out, sc, sc + C, sc + 2 * C, sc + 3 * C, dgamma, dbeta, dx, rows, C, mask, s);
}

void Model::attach_bn_reduction(Epilogue& e, const ConvLaunch& l, const BnRed& red, cudaStream_t s) {
  const int C = red.c->bn.C;
  ARGUS_CHECK(C <= 512 && l.p.n_total == C, "fused BN reduction: channel count");
  bnred_slots_ = stat_slots(l);
  ARGUS_CUDA(cudaMemsetAsync(bnred_stats_, 0, static_cast<size_t>(bnred_slots_) * 2 * C * sizeof(float), s)); pdl_break(s, kPdlAfterMemop);
  const float* sc = bn_scratch_ + red.c->bn.scratch_off;
  e.bn_raw = red.raw;
  e.bn_scale = sc;
  e.bn_shift = sc + C;
  e.stat_partial = bnred_stats_;
}

void Model::bn_backward_reduced(const ConvRef& c, bf16* dy, const bf16* raw, bf16* dx, int64_t rows, cudaStream_t s) {
  const float* sc = bn_scratch_ + c.bn.scratch_off;
  float* dgamma = grads_dev_ + c.bn.gamma_off;
  float* dbeta = grads_dev_ + c.bn.beta_off;
  const int C = c.bn.C;
  bn_bwd_finalize_slots(bnred_stats_, bnred_slots_, sc + 2 * C, sc + 3 * C, dgamma, dbeta, C, s);
  // the apply pass overwrites a gradient buffer that an in-flight weight-gradient GEMM may still be reading
  join_wgrad(s);
  bn_bwd_apply(dy, raw, nullptr, sc, sc + C, sc + 2 * C, sc + 3 * C, dgamma, dbeta, dx, rows, C, 0, s);   // dy is masked
}

void Model::conv_backward(const ConvPlan& cp, const bf16* residual, const uint8_t* out_bits, float* out_stats,
                          cudaStream_t s, const BnRed* red) {
  // fork: the weight gradient only needs dRaw and the saved activation, both final at this point
  run_wgrad(cp.wgrad, s);
  Epilogue e;
  e.residual = residual;
  e.out_bits = out_bits;
  if (red != nullptr) {
    ARGUS_CHECK(cp.dgrad.size() == 1 && residual == nullptr && out_bits == nullptr && out_stats == nullptr,
                "fused BN reduction needs a single plain dgrad launch");
    attach_bn_reduction(e, cp.dgrad[0], *red, s);
  }
  if (out_stats != nullptr) {
    ARGUS_CHECK(cp.dgrad.size() == 1, "gradient statistics need a single dgrad launch");
    alg_gstats_slots_ = stat_slots(cp.dgrad[0]);
    ARGUS_CUDA(cudaMemsetAsync(out_stats, 0, static_cast<size_t>(alg_gstats_slots_) * 2 * cp.dgrad[0].p.n_total * sizeof(float), s)); pdl_break(s, kPdlAfterMemop);
    e.stat_partial = out_stats;
  }
  for (const auto& l : cp.dgrad) launch_conv(l, e, s);
}

// Expanding 1x1 convolution + batch norm backward without touching the BN input or its gradient (see bn_algebra.cu
// for the derivation): upstream masked gradient g and the saved conv input `act` go through three GEMMs.
void Model::conv_bn_backward_algebraic(const ConvRef& c, const WgradLaunch& hg, const ConvLaunch& concat, const bf16* act,
                                       const float* colsum_partial, int64_t rows, int N, cudaStream_t s,
                                       const BnRed* red, const float* saved_gram) {
  const int O = c.shape.Cout, C = c.shape.Cin;
  // fused tail: G is the matrix the forward statistics came from (kept per block) and hg computes H only; otherwise hg
  // is the stacked launch that appends G below H
  const float* alg_g = saved_gram != nullptr ? saved_gram : alg_h_ + static_cast<size_t>(O) * C;
  join_wgrad(s);   // one split-K scratch buffer: no weight-gradient GEMM may be in flight on the side stream
  ARGUS_CUDA(cudaMemsetAsync(alg_h_, 0, static_cast<size_t>(saved_gram != nullptr ? O : O + C) * C * sizeof(float), s)); pdl_break(s, kPdlAfterMemop);
  launch_wgrad(hg, wgrad_scratch_, s);     // H = g^T act (rows < O) [and G = act^T act (rows O..O+C), act tiles loaded once]
  // column sums of `act`: the forward kept them next to its Gram matrix (fused tail); otherwise they are rebuilt here
  const float* colsum = alg_s_;
  if (saved_gram != nullptr) colsum = saved_gram + static_cast<size_t>(C) * C;
  else if (colsum_partial != nullptr) colsum_finalize(colsum_partial, bn_apply_grid(rows, C), alg_s_, C, s);
  else colsum_pixels_bf16(act, N, c.shape.H, c.shape.W, C, c.shape.stride, bn_bwd_scratch_, alg_s_, s);
  const float* sc = bn_scratch_ + c.bn.scratch_off;
  // the coefficient / B-stack kernels feed the dgrad below; the weight-gradient kernel feeds nothing in this chain and
  // runs on the weight-gradient side stream (joined before H, G, s or k1k0 are overwritten: every algebraic call and
  // every bn_backward joins first)
  const bool dw_aside = overlap_wgrad_;
  bn_alg_backward_small(packed_ + c.packed_off, alg_h_, alg_g, colsum, alg_gstats_, alg_gstats_slots_, 2 * O, sc,
                        sc + 2 * O, sc + 3 * O, static_cast<double>(rows), grads_dev_ + c.bn.gamma_off,
                        grads_dev_ + c.bn.beta_off, dw_aside ? nullptr : grads_dev_ + c.w_off, alg_k1k0_, alg_bstack_, alg_bias_,
                        alg_mpartial_, O, C, s);
  if (dw_aside) {
    const bf16* Wp = packed_ + c.packed_off;
    float* dW = grads_dev_ + c.w_off;
    run_on_side(s, [=](cudaStream_t ss) { bn_alg_backward_dw(Wp, alg_h_, alg_g, colsum, sc, alg_k1k0_, dW, O, C, ss); });
  }
  Epilogue e;
  e.shift = alg_bias_;
  if (red != nullptr) attach_bn_reduction(e, concat, *red, s);
  launch_conv(concat, e, s);               // dAct = [g | act] * [diag(sc) W ; W^T diag(k1) W] + k0^T W
}

// The stride-2 1x1 dgrad writes every fourth pixel of T; the rest must be zero. T is private to the block, so the fill
// is needed once per arena epoch, not per step.
void Model::zero_ds_gradient_once(BlockPlan& bp, const BlockRef& br, bf16* T, cudaStream_t s) {
  if (br.ds.shape.stride != 2 || bp.t_zero_epoch == arena_epoch_) return;
  ARGUS_CUDA(cudaMemsetAsync(T, 0, bp.x_bytes, s)); pdl_break(s, kPdlAfterMemop);
  bp.t_zero_epoch = arena_epoch_;
}

void Model::backward(const float* d_out, int stage_begin, int stage_end, cudaStream_t s) {
  ARGUS_CHECK(grads_dev_ != nullptr, "model is not bound to a gradient arena");
  ARGUS_CHECK(last_grad_forward_ != 2 || last_forward_frozen_,
              "backward(): another forward() ran after the frozen-statistics forward it would differentiate");
  if (precision_ == 1) {
    backward_fp32(d_out, stage_begin, stage_end, s);
    return;
  }
  if (last_grad_forward_ == 2) {
    backward_frozen(*last_frozen_plan_, stage_begin, stage_end, d_out, s);
    return;
  }
  ARGUS_CHECK(last_train_plan_ != nullptr, "backward() needs a preceding training forward()");
  Plan& p = *last_train_plan_;
  const int N = p.N;
  const int n_blocks = static_cast<int>(blocks_.size());
  // block index ranges per stage: stage 0 = layer4, 1 = layer3, 2 = layer2, 3 = layer1
  const int first_block[4] = {13, 7, 3, 0};
  const int last_block[4] = {16, 13, 7, 3};
  for (int stage = stage_begin; stage < stage_end; ++stage) {
    if (stage == 0) head_backward(p, d_out, s);
    for (int i = last_block[stage] - 1; i >= first_block[stage]; --i) {
      ARGUS_CHECK(i < n_blocks, "block index");
      BlockRef& br = blocks_[i];
      BlockPlan& bp = p.blocks[i];
      // zero this block's packed 3x3 gradient scratch
      ARGUS_CUDA(cudaMemsetAsync(gpacked_ + br.c2.gpacked_off, 0,
                                 static_cast<size_t>(br.c2.shape.Ktot()) * br.c2.shape.Cout * sizeof(float), s)); pdl_break(s, kPdlAfterMemop);
      bf16 *P = bp.g_out, *Q = bp.g_q, *R = bp.g_r, *T = bp.g_t;
      // The gradient P of the block output arrives ALREADY masked by the block's final ReLU (the dgrad epilogue or
      // avgpool_bwd that produced it applied the bit mask), so it is the BN3 / downsample-BN upstream gradient and the
      // identity-branch gradient at once.
      const uint8_t* prev_bits = (i > 0) ? p.blocks[i - 1].out_bits : nullptr;
      float* prev_stats = (i > 0 && p.blocks[i - 1].algebraic) ? alg_gstats_ : nullptr;
      const bf16* residual = P;
      if (br.has_ds) {
        if (bp.ds_algebraic) {
          zero_ds_gradient_once(bp, br, T, s);
          conv_bn_backward_algebraic(br.ds, bp.ds_hg_wgrad, bp.ds_concat, bp.x, nullptr, bp.rows_out, N, s, nullptr,
                                     bp.ds_gram_saved);
        } else {
          bn_backward(br.ds, P, bp.rawd, nullptr, R, bp.rows_out, 0, s);
          zero_ds_gradient_once(bp, br, T, s);
          conv_backward(bp.ds, nullptr, nullptr, nullptr, s);  // R -> T
        }
        residual = T;
      }
      // bn2 / bn1 backward reductions ride in the epilogues of the dgrads that produce dAct2 / dAct1 (dense outputs
      // only: the parity-split dgrad of a stride-2 3x3 convolution keeps the separate reduction pass)
      const BnRed red2{&br.c2, bp.raw2}, red1{&br.c1, bp.raw1};
      // Measured per layer (profiles/r2_bn_reduce_fused_ab.txt): the epilogue pays one extra read of `raw` plus a longer
      // epilogue against the two reads of the separate pass -- a gain where the tensors are large and narrow (layers 1-2,
      // C <= 128: -0.3 ms / step), a wash or a loss on the L2-bound dgrads of layers 3-4 (ARGUS_BN_REDUCE_FUSED=2 fuses all).
      const int cmax = bn_reduce_fused_ == 2 ? 512 : 128;
      const bool fuse2 = bn_reduce_fused_ && br.c2.bn.C <= cmax;
      const bool fuse1 = bn_reduce_fused_ && br.c1.bn.C <= cmax && br.c2.shape.stride == 1;
      if (bp.algebraic) {
        // P, act2 -> R (dAct2), dW3, dgamma3, dbeta3
        conv_bn_backward_algebraic(br.c3, bp.hg_wgrad, bp.c3_concat, bp.act2, bp.act2_colsum, bp.rows_out, N, s,
                                   fuse2 ? &red2 : nullptr, bp.gram_saved);
      } else {
        bn_backward(br.c3, P, bp.raw3, nullptr, Q, bp.rows_out, 0, s);      // Q = dRaw3
        conv_backward(bp.c3, nullptr, nullptr, nullptr, s, fuse2 ? &red2 : nullptr);   // Q -> R (dAct2)
      }
      if (fuse2) bn_backward_reduced(br.c2, R, bp.raw2, Q, bp.rows_out, s);  // Q = dRaw2
      else bn_backward(br.c2, R, bp.raw2, nullptr, Q, bp.rows_out, 1, s);
      conv_backward(bp.c2, nullptr, nullptr, nullptr, s, fuse1 ? &red1 : nullptr);     // Q -> R (dAct1)
      if (fuse1) bn_backward_reduced(br.c1, R, bp.raw1, Q, bp.rows_in, s);   // Q = dRaw1
      else bn_backward(br.c1, R, bp.raw1, nullptr, Q, bp.rows_in, 1, s);
      // Q -> S (+ identity-branch gradient), masked by the previous block's ReLU bits; its channel sums are the
      // dbeta of the previous block's algebraic bn3 backward
      conv_backward(bp.c1, residual, prev_bits, prev_stats, s);
    }
    if (stage == 3) {
      // ---- stem: max-pool backward, bn1 backward, weight gradient
      ARGUS_CUDA(cudaMemsetAsync(gpacked_ + stem_.gpacked_off, 0, 64 * 256 * sizeof(float), s)); pdl_break(s, kPdlAfterMemop);
      {
        // max-pool backward fused into the stem's BN(+ReLU) backward: p.g_act0 is never written
        const float* sc = bn_scratch_ + stem_.bn.scratch_off;
        join_wgrad(s);   // g_raw0 aliases a buffer the previous block's weight-gradient GEMM may still read
        stem_pool_bn_backward(p.g_stem_in, p.idx0, p.raw0, sc, sc + 64, sc + 128, sc + 192, grads_dev_ + stem_.bn.gamma_off,
                              grads_dev_ + stem_.bn.beta_off, p.g_raw0, N, p.H / 2, p.W / 2, 64, bn_bwd_scratch_, s);
      }
      run_wgrad(p.stem.wgrad, s);
      stem_grad_ready_ = true;   // p.g_raw0 now holds d loss / d (stem convolution output) for input_grad()
    }
    join_wgrad(s);
    unpack_stage_wgrads(stage, s);
  }
}

// head MLP, fc and the global average pooling backward: d_out -> the masked output gradient of the last block
void Model::head_backward(Plan& p, const float* d_out, cudaStream_t s) {
  const int N = p.N, B = p.B, F = n_cams_ * out_dim_;
  // ---- head
  ARGUS_CUDA(cudaMemcpyAsync(p.d_out, d_out, static_cast<size_t>(B) * 6 * sizeof(float),
                             cudaMemcpyDeviceToDevice, s)); pdl_break(s, kPdlAfterMemop);
  float* g = grads_dev_;
  // The chain only needs the input gradients; the three weight gradients (the 2048-wide layer alone is 0.15 ms of
  // latency-bound fp32 SIMT work) read the finished output gradients and run on the weight-gradient side stream,
  // which is idle here. Same kernels, same summation order: the gradients keep their bits.
  linear_bwd_input(p.d_out, nullptr, params_dev_ + head_w_off_[2], p.d_a2, B, 128, 6, s);
  linear_bwd_input(p.d_a2, p.h2, params_dev_ + head_w_off_[1], p.d_a1, B, 128, 128, s);
  linear_bwd_input(p.d_a1, p.h1, params_dev_ + head_w_off_[0], p.d_z0, B, F, 128, s);
  {
    const float *d2 = p.d_out, *d1 = p.d_a2, *d0 = p.d_a1, *x2 = p.a2, *x1 = p.a1, *x0 = p.z0;
    float *w2 = g + head_w_off_[2], *b2 = g + head_b_off_[2], *w1 = g + head_w_off_[1], *b1 = g + head_b_off_[1],
          *w0 = g + head_w_off_[0], *b0 = g + head_b_off_[0];
    run_on_side(s, [=](cudaStream_t ss) {
      linear_bwd_weights(d2, x2, w2, b2, B, 128, 6, ss);
      linear_bwd_weights(d1, x1, w1, b1, B, 128, 128, ss);
      linear_bwd_weights(d0, x0, w0, b0, B, F, 128, ss);
    });
  }
  gelu_bwd_bf16(p.d_z0, p.feat, p.d_feat, static_cast<int64_t>(B) * F, s);
  // ---- fc
  { ProfileScope prof("head", s, 0, 2.0 * N * out_dim_); }
  // (the fc bias gradient -- one block column walking all N rows, 38 us -- feeds nothing in the chain either)
  {
    const bf16* dfeat = p.d_feat;
    float* dbias = g + fc_bias_off_;
    const int od = out_dim_;
    run_on_side(s, [=](cudaStream_t ss) {
      launch_kernel(colsum_bf16_kernel, (od + 127) / 128, 128, 0, ss, dfeat, dbias, N, od);
      ARGUS_CUDA(cudaGetLastError());
    });
  }
  run_wgrad(p.fc.wgrad, s);
  Epilogue e;
  for (const auto& l : p.fc.dgrad) launch_conv(l, e, s);
  avgpool_bwd(p.d_pooled, p.blocks.back().g_out, p.blocks.back().out_bits, N, p.final_hw, 2048, s);
}

// packed 3x3 / stem gradients of this stage -> PyTorch layout in the gradient arena
void Model::unpack_stage_wgrads(int stage, cudaStream_t s) {
  int lo = -1, hi = -1;
  for (size_t i = 0; i < pack_table_.size(); ++i)
    if (pack_table_stage_[i] == stage) {
      if (lo < 0) lo = static_cast<int>(i);
      hi = static_cast<int>(i) + 1;
    }
  if (lo >= 0) unpack_wgrads(gpacked_, grads_dev_, pack_table_dev_ + lo, hi - lo, s);
}

// ------------------------------------------------------------------------------------------------------------
// backward of a frozen-statistics (eval-mode) forward: every batch norm is the constant affine map sc * raw + shift, so
// each convolution's backward is its weight-gradient GEMM on the masked output gradient g (H = g^T im2col(x), finished
// by bn_frozen_finish into dW = diag(sc) H, dgamma, dbeta) and its dgrad of g against diag(sc) W. No batch-norm pass
// over an activation remains. All work runs on the caller's stream, in a fixed order: deterministic.
// ------------------------------------------------------------------------------------------------------------
void Model::ensure_frozen_buffers() {
  if (packed_scaled_ != nullptr) return;
  // (plan-build time only) every stream of this model is idle
  ARGUS_CUDA(cudaMalloc(&packed_scaled_, n_packed_ * sizeof(bf16)));
  std::vector<WeightPackEntry> table;
  std::vector<int64_t> scale_off;
  int64_t h_elems = 0;
  auto add = [&](const ConvRef& c) {
    for (const auto& e : pack_table_)
      if (e.dst_off == c.packed_off) table.push_back(e);
    scale_off.push_back(c.bn.scratch_off);
    if (c.shape.kind == 0 && c.shape.k == 1) h_elems = std::max<int64_t>(h_elems, static_cast<int64_t>(c.shape.Cout) * c.shape.Cin);
  };
  add(stem_);
  for (const auto& b : blocks_) {
    add(b.c1); add(b.c2); add(b.c3);
    if (b.has_ds) add(b.ds);
  }
  ARGUS_CHECK(table.size() == scale_off.size(), "frozen-statistics pack table");
  n_scaled_entries_ = static_cast<int>(table.size());
  ARGUS_CUDA(cudaMalloc(&scaled_table_dev_, table.size() * sizeof(WeightPackEntry)));
  ARGUS_CUDA(cudaMemcpy(scaled_table_dev_, table.data(), table.size() * sizeof(WeightPackEntry), cudaMemcpyHostToDevice));
  ARGUS_CUDA(cudaMalloc(&scaled_scale_off_dev_, scale_off.size() * sizeof(int64_t)));
  ARGUS_CUDA(cudaMemcpy(scaled_scale_off_dev_, scale_off.data(), scale_off.size() * sizeof(int64_t), cudaMemcpyHostToDevice));
  ARGUS_CUDA(cudaMalloc(&frz_h_, h_elems * sizeof(float)));
  ARGUS_CUDA(cudaMalloc(&frz_pstats_, static_cast<size_t>(max_stat_slots_) * 2 * 2048 * sizeof(float)));
  ARGUS_CUDA(cudaMalloc(&frz_gstats_, static_cast<size_t>(max_stat_slots_) * 2 * 512 * sizeof(float)));
  ARGUS_CUDA(cudaMalloc(&frz_sums_, 2 * 2048 * sizeof(float)));
  ARGUS_CUDA(cudaMalloc(&frz_partial_, 4LL * num_sms() * 2048 * sizeof(float)));
  scaled_dirty_ = true;
}

void Model::frozen_wgrad_finish(const ConvRef& c, const WgradLaunch& l, float* h, const float* sums, int slots,
                                int stride, float* dW, bool accumulate, cudaStream_t s) {
  const int O = c.shape.Cout, K = c.shape.Ktot();
  ARGUS_CUDA(cudaMemsetAsync(h, 0, static_cast<size_t>(O) * K * sizeof(float), s)); pdl_break(s, kPdlAfterMemop);
  launch_wgrad(l, wgrad_scratch_, s);
  const float* sc = bn_scratch_ + c.bn.scratch_off;
  bn_frozen_finish(packed_ + c.packed_off, h, sums, slots, stride, sc, sc + 2 * O, sc + 3 * O, grads_dev_ + c.bn.gamma_off,
                   grads_dev_ + c.bn.beta_off, dW, accumulate, O, K, s);
}

void Model::backward_frozen(Plan& p, int stage_begin, int stage_end, const float* d_out, cudaStream_t s) {
  const int N = p.N;
  const int first_block[4] = {13, 7, 3, 0};
  const int last_block[4] = {16, 13, 7, 3};
  float* g1_sum = frz_sums_ + 2048;   // sum of g1 (block loop), of g0 (stem)
  for (int stage = stage_begin; stage < stage_end; ++stage) {
    if (stage == 0) {
      head_backward(p, d_out, s);
      join_wgrad(s);   // the weight-gradient GEMMs below share the split-K scratch with the fc's
      const BlockPlan& last = p.blocks.back();
      colsum_rows_bf16(last.g_out, last.rows_out, blocks_.back().c3.shape.Cout, frz_partial_, frz_sums_, s);
      frz_p_sum_ = frz_sums_; frz_p_slots_ = 1; frz_p_stride_ = 0;
    }
    for (int i = last_block[stage] - 1; i >= first_block[stage]; --i) {
      BlockRef& br = blocks_[i];
      BlockPlan& bp = p.blocks[i];
      bf16 *P = bp.g_out, *R = bp.g_r, *T = bp.g_t;
      const int wd = br.c1.shape.Cout;
      // conv3 / bn3 and the downsample branch: H = P^T act, dW += diag(sc) H, dgamma, dbeta = sum P
      frozen_wgrad_finish(br.c3, bp.c3.wgrad, frz_h_, frz_p_sum_, frz_p_slots_, frz_p_stride_, grads_dev_ + br.c3.w_off,
                          true, s);
      if (br.has_ds)
        frozen_wgrad_finish(br.ds, bp.ds.wgrad, frz_h_, frz_p_sum_, frz_p_slots_, frz_p_stride_,
                            grads_dev_ + br.ds.w_off, true, s);
      // g2 = (P diag(sc3) W3) masked by act2's bits, with its column sums in the statistics slots
      {
        Epilogue e;
        e.out_bits = bp.act2_bits;
        e.stat_partial = frz_gstats_;
        ARGUS_CHECK(bp.c3.dgrad.size() == 1, "conv3 dgrad: one launch");
        const int slots = stat_slots(bp.c3.dgrad[0]);
        ARGUS_CUDA(cudaMemsetAsync(frz_gstats_, 0, static_cast<size_t>(slots) * 2 * wd * sizeof(float), s)); pdl_break(s, kPdlAfterMemop);
        launch_conv(bp.c3.dgrad[0], e, s);
        // conv2 / bn2: H2 = g2^T im2col(act1) in the packed layout, scaled in place (unpacked at the end of the stage)
        frozen_wgrad_finish(br.c2, bp.c2.wgrad, gpacked_ + br.c2.gpacked_off, frz_gstats_, slots, 2 * wd,
                            gpacked_ + br.c2.gpacked_off, false, s);
      }
      if (br.has_ds) {
        zero_ds_gradient_once(bp, br, T, s);
        Epilogue e;
        for (const auto& l : bp.ds.dgrad) launch_conv(l, e, s);   // T = P diag(scd) Wd
      }
      {
        // g1 = (g2 diag(sc2) W2) masked by act1's bits (a separate pass: the stride-2 dgrad is one launch per parity
        // class, and the bit mask of a dense 3x3 dgrad would need an epilogue instance of its own)
        Epilogue e;
        for (const auto& l : bp.c2.dgrad) launch_conv(l, e, s);
        relu_bits_mask_colsum(R, bp.act1_bits, bp.rows_in, wd, frz_partial_, g1_sum, s);
      }
      frozen_wgrad_finish(br.c1, bp.c1.wgrad, frz_h_, g1_sum, 1, 0, grads_dev_ + br.c1.w_off, true, s);
      {
        // block-input gradient = g1 diag(sc1) W1 + the identity branch, masked by the previous block's ReLU bits; its
        // column sums are the sum of P of the previous block
        Epilogue e;
        e.residual = br.has_ds ? T : P;
        e.out_bits = i > 0 ? p.blocks[i - 1].out_bits : nullptr;
        ARGUS_CHECK(bp.c1.dgrad.size() == 1, "conv1 dgrad: one launch");
        if (i > 0) {
          const int C = br.c1.shape.Cin;
          frz_p_slots_ = stat_slots(bp.c1.dgrad[0]);
          frz_p_stride_ = 2 * C;
          frz_p_sum_ = frz_pstats_;
          ARGUS_CUDA(cudaMemsetAsync(frz_pstats_, 0, static_cast<size_t>(frz_p_slots_) * 2 * C * sizeof(float), s)); pdl_break(s, kPdlAfterMemop);
          e.stat_partial = frz_pstats_;
        }
        launch_conv(bp.c1.dgrad[0], e, s);
      }
    }
    if (stage == 3) {
      // stem: g0 = unpool(g_pooled) masked by [pooled0 > 0], then H0 = g0^T x (packed), scaled in place
      stem_unpool_relu(p.g_stem_in, p.idx0, p.pooled0, p.g_raw0, N, p.H / 2, p.W / 2, frz_partial_, g1_sum, s);
      frozen_wgrad_finish(stem_, p.stem.wgrad, gpacked_ + stem_.gpacked_off, g1_sum, 1, 0, gpacked_ + stem_.gpacked_off,
                          false, s);
      stem_grad_ready_ = true;   // p.g_raw0 = g0: input_grad() runs its dgrad against diag(sc0) W0
    }
    unpack_stage_wgrads(stage, s);
  }
}

void Model::check_input_grad_ready(bool have_train_forward) const {
  ARGUS_CHECK(have_train_forward, "input_grad() needs a preceding training forward()");
  ARGUS_CHECK(train_input_f32_, "the last training forward consumed a staged / uint8 input, which has no input gradient");
  ARGUS_CHECK(stem_grad_ready_, "input_grad() needs backward() stage 3 to have run since the last forward()");
}

void Model::input_grad(float* dx, cudaStream_t s) {
  if (precision_ == 1) {
    input_grad_fp32(dx, s);
    return;
  }
  if (last_grad_forward_ == 2) {
    check_input_grad_ready(last_frozen_plan_ != nullptr);
    const Plan& p = *last_frozen_plan_;
    stem_dgrad(p.g_raw0, packed_scaled_ + stem_.packed_off, dx, p.N, p.H, p.W, s);   // dRaw0 = sc0 g0
    return;
  }
  check_input_grad_ready(last_train_plan_ != nullptr);
  const Plan& p = *last_train_plan_;
  // the forward rounded x to bf16 (pack_input_f32); its gradient passes straight through that rounding
  stem_dgrad(p.g_raw0, packed_ + stem_.packed_off, dx, p.N, p.H, p.W, s);
}

}  // namespace argus

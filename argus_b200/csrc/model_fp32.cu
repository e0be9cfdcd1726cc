// fp32 parity mode of NCameraCNN (/root/reference/argus/models.py:26-90): the same network, parameters, buffers and
// C ABI as the bf16 tensor-core path in model.cu, executed layer by layer in fp32 by the SIMT kernels of
// fp32_kernels.cu. Exists so that forward outputs, losses and every gradient can be compared with the reference's
// fp32 PyTorch implementation at 1e-4 relative (tests/test_fp32_mode_gpu.py); not a performance path.
#include "kernels_fp32.h"
#include "model.h"

#include <algorithm>

namespace argus {

static constexpr float kBnEps = 1e-5f;
static constexpr float kBnMomentum = 0.1f;

struct UnitF32 {
  float* raw = nullptr;   // convolution output (BN input)
  float* act = nullptr;   // after BN (+ReLU)
};
struct BlockF32 {
  float* x = nullptr;
  UnitF32 c1, c2, c3;
  float* rawd = nullptr;
  float* out = nullptr;
  int h = 0, w = 0, ho = 0, wo = 0;
};

struct Fp32State {
  uint8_t* arena = nullptr;
  size_t arena_bytes = 0, used = 0;
  int B = 0, H = 0, W = 0, N = 0;
  bool training = false, planned = false, have_train_forward = false;
  bool frozen = false;   // the last forward was a frozen-statistics (differentiable eval-mode) one
  float* x_nhwc = nullptr;
  UnitF32 stem;
  float* pooled0 = nullptr;
  uint8_t* idx0 = nullptr;
  std::vector<BlockF32> blocks;
  int final_hw = 0;
  float *pooled = nullptr, *feat = nullptr, *z0 = nullptr, *h1 = nullptr, *a1 = nullptr, *h2 = nullptr, *a2 = nullptr,
        *out = nullptr;
  float *d_out = nullptr, *d_a2 = nullptr, *d_a1 = nullptr, *d_z0 = nullptr, *d_feat = nullptr, *d_pooled = nullptr;
  float* G[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
  float* cur_grad = nullptr;   // gradient wrt the current block output while walking backwards
  float* stem_graw = nullptr;  // after backward stage 3: gradient wrt the stem convolution output (N, H/2, W/2, 64)
  float* stem_gx = nullptr;    // a free gradient buffer of the same stage: the NHWC input gradient goes there
  float* wscratch = nullptr;
  double* bn_partial = nullptr;
  float* bn_sums = nullptr;

  template <typename T>
  T* alloc(size_t count) {
    const size_t bytes = (count * sizeof(T) + 255) / 256 * 256;
    uint8_t* p = arena ? arena + used : nullptr;
    used += bytes;
    return reinterpret_cast<T*>(p);
  }
};

void destroy_fp32_state(Fp32State* st) {
  if (st == nullptr) return;
  cudaFree(st->arena);
  delete st;
}

static ConvShapeF32 shape_of(const ConvRef& c, int N, int H, int W) {
  ConvShapeF32 s;
  s.N = N; s.H = H; s.W = W; s.Cin = c.shape.Cin; s.Cout = c.shape.Cout;
  s.k = (c.shape.kind == 1) ? 7 : c.shape.k;
  s.stride = c.shape.stride;
  return s;
}

// lays out every tensor of one (B, H, W, training) configuration; a null arena only measures
void Model::plan_fp32(Fp32State& st, int B, int H, int W, bool training) {
  const int N = B * n_cams_;
  st.used = 0;
  st.x_nhwc = st.alloc<float>(static_cast<size_t>(N) * H * W * 3);
  const int H1 = H / 2, W1 = W / 2, H2 = H1 / 2, W2 = W1 / 2;
  const size_t stem_elems = static_cast<size_t>(N) * H1 * W1 * 64;
  st.stem.raw = st.alloc<float>(stem_elems);
  st.stem.act = st.alloc<float>(stem_elems);
  st.pooled0 = st.alloc<float>(stem_elems / 4);
  st.idx0 = st.alloc<uint8_t>(stem_elems / 4);
  st.blocks.assign(blocks_.size(), BlockF32());
  float* x = st.pooled0;
  int h = H2, w = W2;
  size_t max_elems = stem_elems;
  int64_t wscratch = 0;
  auto need_w = [&](const ConvRef& c, int n, int hh, int ww) {
    wscratch = std::max(wscratch, conv_f32_wgrad_scratch_elems(shape_of(c, n, hh, ww), nullptr));
  };
  need_w(stem_, N, H, W);
  for (size_t i = 0; i < blocks_.size(); ++i) {
    const BlockRef& br = blocks_[i];
    BlockF32& b = st.blocks[i];
    const int s = br.c2.shape.stride;
    b.x = x; b.h = h; b.w = w; b.ho = h / s; b.wo = w / s;
    const size_t e_in = static_cast<size_t>(N) * h * w, e_out = static_cast<size_t>(N) * b.ho * b.wo;
    const int wd = br.c1.shape.Cout, oc = br.c3.shape.Cout;
    b.c1.raw = st.alloc<float>(e_in * wd);
    b.c1.act = st.alloc<float>(e_in * wd);
    b.c2.raw = st.alloc<float>(e_out * wd);
    b.c2.act = st.alloc<float>(e_out * wd);
    b.c3.raw = st.alloc<float>(e_out * oc);
    if (br.has_ds) b.rawd = st.alloc<float>(e_out * oc);
    b.out = st.alloc<float>(e_out * oc);
    max_elems = std::max(max_elems, std::max(e_in * std::max(wd, br.c1.shape.Cin), e_out * oc));
    need_w(br.c1, N, h, w); need_w(br.c2, N, h, w); need_w(br.c3, N, b.ho, b.wo);
    if (br.has_ds) need_w(br.ds, N, h, w);
    x = b.out; h = b.ho; w = b.wo;
  }
  st.final_hw = h * w;
  need_w(fc_, N, 1, 1);
  const int F = n_cams_ * out_dim_;
  st.pooled = st.alloc<float>(static_cast<size_t>(N) * 2048);
  st.feat = st.alloc<float>(static_cast<size_t>(N) * out_dim_);
  st.z0 = st.alloc<float>(static_cast<size_t>(B) * F);
  st.h1 = st.alloc<float>(static_cast<size_t>(B) * 128);
  st.a1 = st.alloc<float>(static_cast<size_t>(B) * 128);
  st.h2 = st.alloc<float>(static_cast<size_t>(B) * 128);
  st.a2 = st.alloc<float>(static_cast<size_t>(B) * 128);
  st.out = st.alloc<float>(static_cast<size_t>(B) * 8);
  st.bn_partial = st.alloc<double>(static_cast<size_t>(kBnF32MaxBlocks) * 2 * 2048);
  st.bn_sums = st.alloc<float>(2 * 2048);
  if (training) {
    st.d_out = st.alloc<float>(static_cast<size_t>(B) * 8);
    st.d_a2 = st.alloc<float>(static_cast<size_t>(B) * 128);
    st.d_a1 = st.alloc<float>(static_cast<size_t>(B) * 128);
    st.d_z0 = st.alloc<float>(static_cast<size_t>(B) * F);
    st.d_feat = st.alloc<float>(static_cast<size_t>(N) * out_dim_);
    st.d_pooled = st.alloc<float>(static_cast<size_t>(N) * 2048);
    for (int i = 0; i < 5; ++i) st.G[i] = st.alloc<float>(max_elems);
    st.wscratch = st.alloc<float>(static_cast<size_t>(wscratch));
  }
}

Fp32State& Model::fp32_state(int B, int H, int W, bool training) {
  if (f32_ == nullptr) f32_ = new Fp32State();
  Fp32State& st = *f32_;
  if (st.planned && st.B == B && st.H == H && st.W == W && (st.training || !training)) return st;
  ARGUS_CHECK(H % 32 == 0 && W % 32 == 0 && H >= 32 && W >= 32, "fp32 mode: H and W must be multiples of 32");
  uint8_t* saved = st.arena;
  st.arena = nullptr;
  plan_fp32(st, B, H, W, training);
  const size_t need = st.used;
  st.arena = saved;
  if (need > st.arena_bytes) {
    ARGUS_CUDA(cudaDeviceSynchronize());
    if (st.arena) ARGUS_CUDA(cudaFree(st.arena));
    st.arena = nullptr;
    ARGUS_CUDA(cudaMalloc(&st.arena, need));
    st.arena_bytes = need;
  }
  plan_fp32(st, B, H, W, training);
  st.B = B; st.H = H; st.W = W; st.N = B * n_cams_; st.training = training; st.planned = true;
  st.have_train_forward = false;
  return st;
}

// frozen: the eval-mode computation (running statistics folded), on a state that keeps the backward buffers
void Model::forward_fp32(const void* x, bool is_u8, int B, int H, int W, bool training, bool frozen, float* out,
                         cudaStream_t s) {
  Fp32State& st = fp32_state(B, H, W, training || frozen);
  const int N = st.N;
  const float* P = params_dev_;
  float* BUF = buffers_dev_;
  ARGUS_CHECK(x != nullptr, "fp32 mode has no staged-input path: pass the image tensor");
  if (is_u8) pack_input_u8_f32(static_cast<const uint8_t*>(x), st.x_nhwc, N, H, W, s);
  else pack_input_nhwc_f32(static_cast<const float*>(x), st.x_nhwc, N, H, W, s);
  if (!training && eval_fold_dirty_) fold_eval(s);
  if (training) eval_fold_dirty_ = true;

  // conv -> batch norm statistics (train) -> scale/shift in the shared BN scratch
  auto conv_bn = [&](const ConvRef& c, const float* in, float* raw, int n, int h, int w) {
    const ConvShapeF32 cs = shape_of(c, n, h, w);
    conv_f32_forward(cs, in, P + c.w_off, nullptr, raw, s);
    if (training) {
      float* sc = bn_scratch_ + c.bn.scratch_off;
      const int C = c.bn.C;
      bn_f32_train_stats(raw, static_cast<int64_t>(n) * cs.Ho() * cs.Wo(), C, P + c.bn.gamma_off, P + c.bn.beta_off,
                         BUF + c.bn.rm_off, BUF + c.bn.rv_off, kBnMomentum, kBnEps, sc, sc + C, sc + 2 * C, sc + 3 * C,
                         st.bn_partial, s);
    }
  };
  auto SC = [&](const ConvRef& c) { return bn_scratch_ + c.bn.scratch_off; };

  conv_bn(stem_, st.x_nhwc, st.stem.raw, N, H, W);
  const int H1 = H / 2, W1 = W / 2;
  bn_f32_apply(st.stem.raw, SC(stem_), SC(stem_) + 64, nullptr, nullptr, nullptr, 1, st.stem.act,
               static_cast<int64_t>(N) * H1 * W1, 64, s);
  maxpool_f32_fwd(st.stem.act, st.pooled0, st.idx0, N, H1, W1, 64, s);
  for (size_t i = 0; i < blocks_.size(); ++i) {
    const BlockRef& br = blocks_[i];
    BlockF32& b = st.blocks[i];
    const int wd = br.c1.shape.Cout, oc = br.c3.shape.Cout;
    const int64_t rows_in = static_cast<int64_t>(N) * b.h * b.w, rows_out = static_cast<int64_t>(N) * b.ho * b.wo;
    conv_bn(br.c1, b.x, b.c1.raw, N, b.h, b.w);
    bn_f32_apply(b.c1.raw, SC(br.c1), SC(br.c1) + wd, nullptr, nullptr, nullptr, 1, b.c1.act, rows_in, wd, s);
    conv_bn(br.c2, b.c1.act, b.c2.raw, N, b.h, b.w);
    bn_f32_apply(b.c2.raw, SC(br.c2), SC(br.c2) + wd, nullptr, nullptr, nullptr, 1, b.c2.act, rows_out, wd, s);
    conv_bn(br.c3, b.c2.act, b.c3.raw, N, b.ho, b.wo);
    if (br.has_ds) {
      conv_bn(br.ds, b.x, b.rawd, N, b.h, b.w);
      bn_f32_apply(b.c3.raw, SC(br.c3), SC(br.c3) + oc, b.rawd, SC(br.ds), SC(br.ds) + oc, 1, b.out, rows_out, oc, s);
    } else {
      bn_f32_apply(b.c3.raw, SC(br.c3), SC(br.c3) + oc, b.x, nullptr, nullptr, 1, b.out, rows_out, oc, s);
    }
  }
  // pooling, fc, head (argus/models.py:84-90)
  const int F = n_cams_ * out_dim_;
  avgpool_f32_fwd(st.blocks.back().out, st.pooled, N, st.final_hw, 2048, s);
  conv_f32_forward(shape_of(fc_, N, 1, 1), st.pooled, P + fc_.w_off, P + fc_bias_off_, st.feat, s);
  gelu_f32_fwd(st.feat, st.z0, static_cast<int64_t>(B) * F, s);
  linear_fwd(st.z0, P + head_w_off_[0], P + head_b_off_[0], st.h1, st.a1, B, F, 128, s);
  linear_fwd(st.a1, P + head_w_off_[1], P + head_b_off_[1], st.h2, st.a2, B, 128, 128, s);
  linear_fwd(st.a2, P + head_w_off_[2], P + head_b_off_[2], st.out, nullptr, B, 128, 6, s);
  ARGUS_CUDA(cudaMemcpyAsync(out, st.out, static_cast<size_t>(B) * 6 * sizeof(float), cudaMemcpyDeviceToDevice, s)); pdl_break(s, kPdlAfterMemop);
  st.have_train_forward = training || frozen;
  st.frozen = frozen;
}

void Model::backward_fp32(const float* d_out, int stage_begin, int stage_end, cudaStream_t s) {
  ARGUS_CHECK(f32_ != nullptr && f32_->have_train_forward, "backward() needs a preceding training forward()");
  Fp32State& st = *f32_;
  const int N = st.N, B = st.B, F = n_cams_ * out_dim_;
  const float* P = params_dev_;
  float* g = grads_dev_;
  auto SC = [&](const ConvRef& c) { return bn_scratch_ + c.bn.scratch_off; };
  auto bn_bwd = [&](const ConvRef& c, const float* dy, const float* raw, const float* out, float* dx, float* g_out,
                    int64_t rows) {
    const float* sc = SC(c);
    const int C = c.bn.C;
    // (frozen: mean / invstd are the running statistics bn_fold_eval left in the scratch, and dx = sc * g)
    bn_f32_backward(dy, raw, out, sc, sc + 2 * C, sc + 3 * C, g + c.bn.gamma_off, g + c.bn.beta_off, dx, g_out, rows, C,
                    st.bn_partial, st.bn_sums, s, st.frozen);
  };
  auto conv_bwd = [&](const ConvRef& c, const float* dy, const float* in, float* dx, int n, int h, int w) {
    const ConvShapeF32 cs = shape_of(c, n, h, w);
    conv_f32_wgrad(cs, dy, in, g + c.w_off, st.wscratch, s);
    if (dx != nullptr) conv_f32_dgrad(cs, dy, P + c.w_off, dx, s);
  };
  const int first_block[4] = {13, 7, 3, 0};
  const int last_block[4] = {16, 13, 7, 3};
  for (int stage = stage_begin; stage < stage_end; ++stage) {
    if (stage == 0) {
      ARGUS_CUDA(cudaMemcpyAsync(st.d_out, d_out, static_cast<size_t>(B) * 6 * sizeof(float), cudaMemcpyDeviceToDevice, s)); pdl_break(s, kPdlAfterMemop);
      linear_bwd(st.d_out, nullptr, st.a2, P + head_w_off_[2], g + head_w_off_[2], g + head_b_off_[2], st.d_a2, B, 128, 6, s);
      linear_bwd(st.d_a2, st.h2, st.a1, P + head_w_off_[1], g + head_w_off_[1], g + head_b_off_[1], st.d_a1, B, 128, 128, s);
      linear_bwd(st.d_a1, st.h1, st.z0, P + head_w_off_[0], g + head_w_off_[0], g + head_b_off_[0], st.d_z0, B, F, 128, s);
      gelu_f32_bwd(st.d_z0, st.feat, st.d_feat, static_cast<int64_t>(B) * F, s);
      colsum_f32(st.d_feat, g + fc_bias_off_, N, out_dim_, s);
      conv_bwd(fc_, st.d_feat, st.pooled, st.d_pooled, N, 1, 1);
      st.cur_grad = st.G[0];
      avgpool_f32_bwd(st.d_pooled, st.cur_grad, N, st.final_hw, 2048, s);
    }
    for (int i = last_block[stage] - 1; i >= first_block[stage]; --i) {
      const BlockRef& br = blocks_[i];
      BlockF32& b = st.blocks[i];
      // buffer roles: Pg = gradient wrt the block output (becomes the masked gradient), S = gradient wrt the input
      float* Pg = st.cur_grad;
      float* others[4];
      int k = 0;
      for (int j = 0; j < 5; ++j)
        if (st.G[j] != Pg) others[k++] = st.G[j];
      float *Q = others[0], *R = others[1], *S = others[2], *T = others[3];
      const int64_t rows_in = static_cast<int64_t>(N) * b.h * b.w, rows_out = static_cast<int64_t>(N) * b.ho * b.wo;
      bn_bwd(br.c3, Pg, b.c3.raw, b.out, Q, Pg, rows_out);          // Q = dRaw3, Pg = masked gradient
      const float* residual = Pg;
      if (br.has_ds) {
        bn_bwd(br.ds, Pg, b.rawd, nullptr, R, nullptr, rows_out);   // R = dRawd
        conv_bwd(br.ds, R, b.x, T, N, b.h, b.w);                     // T = identity-branch input gradient
        residual = T;
      }
      conv_bwd(br.c3, Q, b.c2.act, R, N, b.ho, b.wo);                // R = dAct2
      bn_bwd(br.c2, R, b.c2.raw, b.c2.act, Q, nullptr, rows_out);    // Q = dRaw2
      conv_bwd(br.c2, Q, b.c1.act, R, N, b.h, b.w);                  // R = dAct1
      bn_bwd(br.c1, R, b.c1.raw, b.c1.act, Q, nullptr, rows_in);     // Q = dRaw1
      conv_bwd(br.c1, Q, b.x, S, N, b.h, b.w);                       // S = main-branch input gradient
      add_f32(S, residual, rows_in * br.c1.shape.Cin, s);
      st.cur_grad = S;
    }
    if (stage == 3) {
      float* Pg = st.cur_grad;
      float* others[4];
      int k = 0;
      for (int j = 0; j < 5; ++j)
        if (st.G[j] != Pg) others[k++] = st.G[j];
      const int H1 = st.H / 2, W1 = st.W / 2;
      maxpool_f32_bwd(Pg, st.idx0, others[0], N, H1, W1, 64, s);
      bn_bwd(stem_, others[0], st.stem.raw, st.stem.act, others[1], nullptr, static_cast<int64_t>(N) * H1 * W1);
      conv_bwd(stem_, others[1], st.x_nhwc, nullptr, N, st.H, st.W);
      st.stem_graw = others[1];
      st.stem_gx = others[0];
      stem_grad_ready_ = true;
    }
  }
}

void Model::input_grad_fp32(float* dx, cudaStream_t s) {
  check_input_grad_ready(f32_ != nullptr && f32_->have_train_forward);
  Fp32State& st = *f32_;
  // transposed stem convolution into NHWC (others[0] of stage 3 holds N*H*W*16 floats, more than the N*H*W*3 needed)
  conv_f32_dgrad(shape_of(stem_, st.N, st.H, st.W), st.stem_graw, params_dev_ + stem_.w_off, st.stem_gx, s);
  unpack_input_grad_nhwc_f32(st.stem_gx, dx, st.N, st.H, st.W, s);
}

}  // namespace argus

// extern "C" entry points of libargus_b200.so (declared in include/argus_b200.h).
#include "../../include/argus_b200.h"

#include "conv_ops.h"
#include "kernels.h"
#include "kernels_fp32.h"
#include "model.h"
#include "runtime.h"

#include <algorithm>
#include <cstring>
#include <vector>

using namespace argus;

// Library-owned scratch for the standalone primitive entry points (grown on demand, never on the model's hot path).
static float* lib_scratch(int64_t elems) {
  static float* buf = nullptr;
  static int64_t cap = 0;
  if (elems > cap) {
    ARGUS_CUDA(cudaDeviceSynchronize());
    if (buf) ARGUS_CUDA(cudaFree(buf));
    ARGUS_CUDA(cudaMalloc(&buf, elems * sizeof(float)));
    cap = elems;
  }
  return buf;
}

static ConvShape make_shape(int N, int H, int W, int Cin, int Cout, int k, int stride, int kind) {
  ConvShape s;
  s.N = N; s.H = H; s.W = W; s.Cin = Cin; s.Cout = Cout; s.k = k; s.stride = stride; s.kind = kind;
  return s;
}

extern "C" {

const char* argus_last_error_string(void) { return get_last_error(); }
int argus_version(void) { return 100; }

int argus_profile_enable(int on) {
  ARGUS_API_BEGIN
  profile_enable(on != 0);
  ARGUS_API_END
}
int argus_profile_report(char* json, int cap) {
  ARGUS_API_BEGIN
  ARGUS_CHECK(json != nullptr && cap > 2, "bad report buffer");
  const std::string r = profile_report_json();
  ARGUS_CHECK(static_cast<int>(r.size()) < cap, "profile report buffer too small");
  std::memcpy(json, r.c_str(), r.size() + 1);
  ARGUS_API_END
}
int64_t argus_launch_count(void) { return launch_count(); }

int argus_require_device(void) {
  ARGUS_API_BEGIN
  require_sm100();
  ARGUS_API_END
}

int argus_conv2d_forward(const void* x, const void* w, void* y, int N, int H, int W, int Cin, int Cout, int k,
                         int stride, int kind, const float* scale, const float* shift, const void* residual, int relu,
                         float* stat_partial, int stat_slot_capacity, void* stream) {
  ARGUS_API_BEGIN
  require_sm100();
  ConvShape s = make_shape(N, H, W, Cin, Cout, k, stride, kind);
  ConvLaunch l = plan_conv_forward(s, static_cast<const __nv_bfloat16*>(x), static_cast<const __nv_bfloat16*>(w),
                                   static_cast<__nv_bfloat16*>(y));
  Epilogue e;
  e.scale = scale; e.shift = shift; e.residual = static_cast<const __nv_bfloat16*>(residual); e.relu = relu;
  e.stat_partial = stat_partial;
  ARGUS_CHECK(stat_partial == nullptr || stat_slot_capacity >= stat_slots(l), "statistics buffer has too few slots");
  launch_conv(l, e, static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}

int argus_conv2d_stat_slots(int N, int H, int W, int Cin, int Cout, int k, int stride, int kind, int* slots) {
  ARGUS_API_BEGIN
  require_sm100();
  ARGUS_CHECK(slots != nullptr, "null argument");
  ConvShape s = make_shape(N, H, W, Cin, Cout, k, stride, kind);
  validate_shape(s);
  const int64_t m_tiles = (s.out_pixels() + kBlockM - 1) / kBlockM;
  // same tile choice as plan_conv_forward: an upper bound is enough for sizing
  const int64_t tiles = m_tiles * ((Cout + 63) / 64);
  *slots = kEpiGroups * static_cast<int>(std::min<int64_t>(tiles, num_sms()));   // one per epilogue group per CTA
  ARGUS_API_END
}

int argus_conv2d_dgrad(const void* dy, const void* w, void* dx, int N, int H, int W, int Cin, int Cout, int k,
                       int stride, const void* residual, void* stream) {
  ARGUS_API_BEGIN
  require_sm100();
  ConvShape s = make_shape(N, H, W, Cin, Cout, k, stride, 0);
  ARGUS_CHECK(residual == nullptr || stride == 1, "residual add is only supported for stride-1 dgrad");
  auto ls = plan_conv_dgrad(s, static_cast<const __nv_bfloat16*>(dy), static_cast<const __nv_bfloat16*>(w),
                            static_cast<__nv_bfloat16*>(dx));
  Epilogue e;
  e.residual = static_cast<const __nv_bfloat16*>(residual);
  for (auto& l : ls) launch_conv(l, e, static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}

int argus_conv2d_dgrad_bits(const void* dy, const void* w, void* dx, int N, int H, int W, int Cin, int Cout, int k,
                            const void* residual, const void* residual_bits, void* stream) {
  ARGUS_API_BEGIN
  require_sm100();
  ConvShape s = make_shape(N, H, W, Cin, Cout, k, 1, 0);
  ARGUS_CHECK(residual != nullptr && residual_bits != nullptr, "null argument");
  auto ls = plan_conv_dgrad(s, static_cast<const __nv_bfloat16*>(dy), static_cast<const __nv_bfloat16*>(w),
                            static_cast<__nv_bfloat16*>(dx));
  Epilogue e;
  e.residual = static_cast<const __nv_bfloat16*>(residual);
  e.residual_bits = static_cast<const uint8_t*>(residual_bits);
  for (auto& l : ls) launch_conv(l, e, static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}

int argus_conv2d_dgrad_ex(const void* dy, const void* w, void* dx, int N, int H, int W, int Cin, int Cout, int stride,
                          const void* concat_a, int concat_channels, const float* bias, const void* residual,
                          const void* out_bits, float* stat_partial, int stat_slot_capacity, void* stream) {
  ARGUS_API_BEGIN
  require_sm100();
  ConvShape s = make_shape(N, H, W, Cin, Cout, 1, stride, 0);
  ARGUS_CHECK(residual == nullptr || stride == 1, "residual add is only supported for stride-1 dgrad");
  ConvLaunch l;
  if (concat_a != nullptr) {
    l = plan_dgrad_concat(s, static_cast<const __nv_bfloat16*>(dy), static_cast<const __nv_bfloat16*>(concat_a),
                          concat_channels, static_cast<const __nv_bfloat16*>(w), static_cast<__nv_bfloat16*>(dx));
  } else {
    auto ls = plan_conv_dgrad(s, static_cast<const __nv_bfloat16*>(dy), static_cast<const __nv_bfloat16*>(w),
                              static_cast<__nv_bfloat16*>(dx));
    ARGUS_CHECK(ls.size() == 1, "unexpected dgrad decomposition");
    l = ls[0];
  }
  Epilogue e;
  e.shift = bias;
  e.residual = static_cast<const __nv_bfloat16*>(residual);
  e.out_bits = static_cast<const uint8_t*>(out_bits);
  e.stat_partial = stat_partial;
  ARGUS_CHECK(stat_partial == nullptr || stat_slot_capacity >= stat_slots(l), "statistics buffer has too few slots");
  launch_conv(l, e, static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}

int argus_conv2d_forward_full(const void* x, const void* w, void* y, int N, int H, int W, int Cin, int Cout, int k,
                              int stride, int kind, const float* scale, const float* shift, const void* residual,
                              const float* res_scale, const float* res_shift, int relu, void* relu_bits_out,
                              float* stat_partial, int stat_slot_capacity, int early_trigger, void* stream) {
  ARGUS_API_BEGIN
  require_sm100();
  ConvShape s = make_shape(N, H, W, Cin, Cout, k, stride, kind);
  ConvLaunch l = plan_conv_forward(s, static_cast<const bf16*>(x), static_cast<const bf16*>(w), static_cast<bf16*>(y));
  Epilogue e;
  e.scale = scale; e.shift = shift; e.residual = static_cast<const bf16*>(residual);
  e.res_scale = res_scale; e.res_shift = res_shift;
  e.relu = relu; e.relu_bits_out = static_cast<uint8_t*>(relu_bits_out);
  e.stat_partial = stat_partial;
  e.early_trigger = early_trigger;
  ARGUS_CHECK(relu_bits_out == nullptr || relu != 0, "the ReLU bit mask needs the ReLU");
  ARGUS_CHECK(res_scale == nullptr || residual != nullptr, "residual scale / shift need a residual");
  ARGUS_CHECK(stat_partial == nullptr || stat_slot_capacity >= stat_slots(l), "statistics buffer has too few slots");
  launch_conv(l, e, static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}

static ConvLaunch plan_bnred_dgrad(const ConvShape& s, const void* dy, const void* w, void* dx, const void* concat_a,
                                   int concat_channels) {
  ARGUS_CHECK(s.stride == 1, "the fused BN reduction exists for stride-1 dgrads");
  if (concat_a != nullptr)
    return plan_dgrad_concat(s, static_cast<const bf16*>(dy), static_cast<const bf16*>(concat_a), concat_channels,
                             static_cast<const bf16*>(w), static_cast<bf16*>(dx));
  auto ls = plan_conv_dgrad(s, static_cast<const bf16*>(dy), static_cast<const bf16*>(w), static_cast<bf16*>(dx));
  ARGUS_CHECK(ls.size() == 1, "unexpected dgrad decomposition");
  return ls[0];
}

int argus_conv2d_dgrad_bnred(const void* dy, const void* w, void* dx, int N, int H, int W, int Cin, int Cout, int k,
                             int stride, const void* concat_a, int concat_channels, const float* bias,
                             const void* bn_raw, const float* bn_scale, const float* bn_shift, float* stat_partial,
                             int stat_slot_capacity, void* stream) {
  ARGUS_API_BEGIN
  require_sm100();
  ARGUS_CHECK(bn_raw != nullptr && bn_scale != nullptr && bn_shift != nullptr && stat_partial != nullptr,
              "null argument");
  ConvShape s = make_shape(N, H, W, Cin, Cout, k, stride, 0);
  ConvLaunch l = plan_bnred_dgrad(s, dy, w, dx, concat_a, concat_channels);
  Epilogue e;
  e.shift = bias;
  e.bn_raw = static_cast<const bf16*>(bn_raw);
  e.bn_scale = bn_scale;
  e.bn_shift = bn_shift;
  e.stat_partial = stat_partial;
  ARGUS_CHECK(stat_slot_capacity >= stat_slots(l), "statistics buffer has too few slots");
  launch_conv(l, e, static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}

int argus_conv2d_launch_info(int launch, int N, int H, int W, int Cin, int Cout, int k, int stride, int kind,
                             int concat_channels, int flags, int* out, int cap, int* n_launches) {
  ARGUS_API_BEGIN
  require_sm100();
  ARGUS_CHECK(out != nullptr && n_launches != nullptr, "null argument");
  ARGUS_CUDA(cudaFree(nullptr));   // tensor-map encoding needs a current context, which nothing may have created yet
  // Planning encodes tensor maps but reads no memory: any 1 KB-aligned address stands in for the operands.
  static __align__(1024) char dummy[1024];
  bf16* d = reinterpret_cast<bf16*>(dummy);
  const float* f = reinterpret_cast<const float*>(dummy);
  uint8_t* b = reinterpret_cast<uint8_t*>(dummy);
  ConvShape s = make_shape(N, H, W, Cin, Cout, k, stride, kind);
  std::vector<ConvLaunch> ls;
  if (launch == 0) ls.push_back(plan_conv_forward(s, d, d, d));
  else if (launch == 1 && (flags & ARGUS_EPI_BN_RAW)) ls.push_back(plan_bnred_dgrad(s, d, d, d, nullptr, 0));
  else if (launch == 1) ls = plan_conv_dgrad(s, d, d, d);
  else if (launch == 2 && (flags & ARGUS_EPI_BN_RAW))
    ls.push_back(plan_bnred_dgrad(make_shape(N, H, W, Cin, Cout, 1, stride, 0), d, d, d, d, concat_channels));
  else if (launch == 2) ls.push_back(plan_dgrad_concat(make_shape(N, H, W, Cin, Cout, 1, stride, 0), d, d, concat_channels, d, d));
  else throw Error("unknown launch kind");
  Epilogue e;
  if (flags & ARGUS_EPI_SCALE) e.scale = f;
  if (flags & ARGUS_EPI_SHIFT) e.shift = f;
  if (flags & ARGUS_EPI_RESIDUAL) e.residual = d;
  if (flags & ARGUS_EPI_RES_AFFINE) { e.res_scale = f; e.res_shift = f; }
  if (flags & ARGUS_EPI_RELU) e.relu = 1;
  if (flags & ARGUS_EPI_RELU_BITS_OUT) e.relu_bits_out = b;
  if (flags & ARGUS_EPI_OUT_BITS) e.out_bits = b;
  if (flags & ARGUS_EPI_RESIDUAL_BITS) e.residual_bits = b;
  if (flags & ARGUS_EPI_STATS) e.stat_partial = const_cast<float*>(f);
  if (flags & ARGUS_EPI_BN_RAW) { e.bn_raw = d; e.bn_scale = f; e.bn_shift = f; }
  if (flags & ARGUS_EPI_EARLY_TRIGGER) e.early_trigger = 1;
  *n_launches = static_cast<int>(ls.size());
  ARGUS_CHECK(cap >= ARGUS_LAUNCH_INFO_INTS * *n_launches, "launch info buffer too small");
  for (size_t i = 0; i < ls.size(); ++i) {
    const ConvLaunchInfo li = conv_launch_info(ls[i], e);
    const int v[ARGUS_LAUNCH_INFO_INTS] = {li.inst.block_n, li.inst.b_mn, li.inst.opt, li.halo, li.b_resident,
                                           li.halo_stages, li.num_m_tiles, li.num_n_tiles, li.grid, li.stat_slots};
    std::memcpy(out + i * ARGUS_LAUNCH_INFO_INTS, v, sizeof(v));
  }
  ARGUS_API_END
}

int argus_conv_instances_record(int on) {
  ARGUS_API_BEGIN
  conv_instances_record(on != 0);
  ARGUS_API_END
}
int argus_conv_instances_get(int* keys, int cap, int* n) {
  ARGUS_API_BEGIN
  ARGUS_CHECK(n != nullptr && (keys != nullptr || cap == 0), "null argument");
  const auto rec = conv_instances_recorded();
  *n = static_cast<int>(rec.size());
  for (int i = 0; i < *n && 5 * (i + 1) <= cap; ++i) std::memcpy(keys + 5 * i, rec[i].data(), 5 * sizeof(int));
  ARGUS_API_END
}

int argus_conv_instances_all(int* keys, int cap, int* n) {
  ARGUS_API_BEGIN
  ARGUS_CHECK(n != nullptr && (keys != nullptr || cap == 0), "null argument");
  const auto all = conv_instances_all();
  *n = static_cast<int>(all.size());
  for (int i = 0; i < *n && 3 * (i + 1) <= cap; ++i) std::memcpy(keys + 3 * i, all[i].data(), 3 * sizeof(int));
  ARGUS_API_END
}

int argus_conv2d_gram(const void* x, float* g, int N, int H, int W, int Cin, int Cout, int stride, void* stream) {
  ARGUS_API_BEGIN
  require_sm100();
  ConvShape s = make_shape(N, H, W, Cin, Cout, 1, stride, 0);
  validate_shape(s);
  WgradLaunch l = plan_gram(s, static_cast<const bf16*>(x), g);
  launch_wgrad(l, lib_scratch(wgrad_scratch_elems(l)), static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}

int argus_colsum_pixels(const void* x, int N, int H, int W, int C, int stride, float* scratch, float* out, void* stream) {
  ARGUS_API_BEGIN
  require_sm100();
  ARGUS_CHECK(x != nullptr && scratch != nullptr && out != nullptr, "null argument");
  ARGUS_CHECK(N > 0 && H > 0 && W > 0 && (stride == 1 || stride == 2) && H % stride == 0 && W % stride == 0,
              "colsum: bad shape");
  colsum_pixels_bf16(static_cast<const bf16*>(x), N, H, W, C, stride, scratch, out, static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}

int argus_bn_stats_from_gram(const void* W, const float* G, const float* s, double rows, const float* gamma,
                             const float* beta, float* running_mean, float* running_var, float momentum, float eps,
                             float* scale, float* shift, float* save_mean, float* save_invstd, float* scratch, int O,
                             int C, void* stream) {
  ARGUS_API_BEGIN
  require_sm100();
  ARGUS_CHECK((running_mean == nullptr) == (running_var == nullptr), "running mean and variance come together");
  bn_stats_from_gram(static_cast<const bf16*>(W), G, s, rows, gamma, beta, running_mean, running_var, momentum, eps,
                     scale, shift, save_mean, save_invstd, scratch, O, C, static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}

int argus_conv2d_wgrad_gram(const void* dy, const void* x, float* dw, int N, int H, int W, int Cin, int Cout, int stride,
                            void* stream) {
  ARGUS_API_BEGIN
  require_sm100();
  ConvShape s = make_shape(N, H, W, Cin, Cout, 1, stride, 0);
  WgradLaunch l = plan_conv_wgrad_gram(s, static_cast<const __nv_bfloat16*>(dy), static_cast<const __nv_bfloat16*>(x), dw);
  launch_wgrad(l, lib_scratch(wgrad_scratch_elems(l)), static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}

int argus_conv_bn_backward_algebraic(const void* g, const void* act, const void* w_bf16, const float* g_colsum,
                                     const float* scale, const float* mean, const float* invstd, float* dgamma,
                                     float* dbeta, float* dw, void* dact, int N, int H, int W, int C, int O, int stride,
                                     void* stream) {
  ARGUS_API_BEGIN
  require_sm100();
  // Self-contained form of the algebraic conv(1x1) + BN backward used by the model (csrc/bn_algebra.cu): g (N,Ho,Wo,O)
  // masked upstream gradient, act (N,H,W,C) the convolution input, w_bf16 [O][C]; g_colsum [O] = column sums of g.
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  ConvShape s = make_shape(N, H, W, C, O, 1, stride, 0);
  const int64_t rows = s.out_pixels();
  const size_t OC = static_cast<size_t>(O) * C, CC = static_cast<size_t>(C) * C;
  // scratch layout (floats): H|G [(O+C)*C], s [C], k1k0 [2*O], bias [C], colsum partials, matrix partials, bstack (bf16)
  const int64_t colsum_scratch = 4LL * num_sms() * C;
  const int64_t mpart = bn_alg_matrix_scratch_elems(C);
  const int64_t total = static_cast<int64_t>(OC + CC) + C + 2 * O + C + colsum_scratch + mpart + (static_cast<int64_t>(O + C) * C + 1) / 2;
  static float* buf = nullptr;
  static int64_t cap = 0;
  if (total > cap) {
    ARGUS_CUDA(cudaDeviceSynchronize());
    if (buf) ARGUS_CUDA(cudaFree(buf));
    ARGUS_CUDA(cudaMalloc(&buf, total * sizeof(float)));
    cap = total;
  }
  float* Hb = buf;
  float* Gb = Hb + OC;
  float* sb = Gb + CC;
  float* k1k0 = sb + C;
  float* bias = k1k0 + 2 * O;
  float* cs = bias + C;
  float* mp = cs + colsum_scratch;
  bf16* bstack = reinterpret_cast<bf16*>(mp + mpart);
  const bf16* G16 = static_cast<const bf16*>(g);
  const bf16* A16 = static_cast<const bf16*>(act);
  const bf16* W16 = static_cast<const bf16*>(w_bf16);
  WgradLaunch hg = plan_conv_wgrad_gram(s, G16, A16, Hb);
  ConvLaunch concat = plan_dgrad_concat(s, G16, A16, C, bstack, static_cast<bf16*>(dact));
  ARGUS_CUDA(cudaMemsetAsync(Hb, 0, (OC + CC) * sizeof(float), st)); pdl_break(st, kPdlAfterMemop);
  launch_wgrad(hg, lib_scratch(wgrad_scratch_elems(hg)), st);
  colsum_pixels_bf16(A16, N, H, W, C, stride, cs, sb, st);
  // g_colsum plays the role of ONE statistics slot (stride irrelevant)
  bn_alg_backward_small(W16, Hb, Gb, sb, g_colsum, 1, O, scale, mean, invstd, static_cast<double>(rows), dgamma, dbeta, dw,
                        k1k0, bstack, bias, mp, O, C, st);
  if (stride == 2)
    ARGUS_CUDA(cudaMemsetAsync(dact, 0, static_cast<size_t>(N) * H * W * C * sizeof(bf16), st)); pdl_break(st, kPdlAfterMemop);
  Epilogue e;
  e.shift = bias;
  launch_conv(concat, e, st);
  ARGUS_API_END
}

int argus_conv2d_wgrad(const void* dy, const void* x, float* dw, int N, int H, int W, int Cin, int Cout, int k,
                       int stride, int kind, void* stream) {
  ARGUS_API_BEGIN
  require_sm100();
  ConvShape s = make_shape(N, H, W, Cin, Cout, k, stride, kind);
  WgradLaunch l = plan_conv_wgrad(s, static_cast<const __nv_bfloat16*>(dy), static_cast<const __nv_bfloat16*>(x), dw);
  launch_wgrad(l, lib_scratch(wgrad_scratch_elems(l)), static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}

int argus_bn_frozen_finish(const void* W, const float* H, const float* stat_partial, int slots, int stat_stride,
                           const float* scale, const float* mean, const float* invstd, float* dgamma, float* dbeta,
                           float* dW, int accumulate, int O, int K, void* stream) {
  ARGUS_API_BEGIN
  require_sm100();
  bn_frozen_finish(static_cast<const bf16*>(W), H, stat_partial, slots, stat_stride, scale, mean, invstd, dgamma, dbeta,
                   dW, accumulate != 0, O, K, static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}
int argus_relu_bits_mask_colsum(void* g, const void* bits, int64_t rows, int C, float* out, void* stream) {
  ARGUS_API_BEGIN
  require_sm100();
  relu_bits_mask_colsum(static_cast<bf16*>(g), static_cast<const uint8_t*>(bits), rows, C,
                        lib_scratch(4LL * num_sms() * C), out, static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}
int argus_stem_unpool_relu(const void* dpool, const void* idx, const void* pooled, void* g0, int N, int H, int W,
                           float* out, void* stream) {
  ARGUS_API_BEGIN
  require_sm100();
  stem_unpool_relu(static_cast<const bf16*>(dpool), static_cast<const uint8_t*>(idx), static_cast<const bf16*>(pooled),
                   static_cast<bf16*>(g0), N, H, W, lib_scratch(4LL * num_sms() * 64), out,
                   static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}
int argus_pack_weight_scaled(const float* w, const float* scale, void* packed, int Cout, int Cin, int k, int kind,
                             void* stream) {
  ARGUS_API_BEGIN
  require_sm100();
  ARGUS_CHECK(kind == 0 || (kind == 1 && Cout == 64 && Cin == 3 && k == 7), "kind 1 is the 64 x 3 x 7 x 7 stem");
  WeightPackEntry e;
  e.src_off = 0; e.dst_off = 0; e.cout = Cout; e.cin = Cin; e.kk = k * k; e.kind = kind;
  const int64_t zero = 0;
  // the one-entry table and its scale offset live at the start of the library scratch (synchronous copies: test entry)
  float* dev = lib_scratch(static_cast<int64_t>((sizeof(WeightPackEntry) + sizeof(int64_t)) / sizeof(float) + 4));
  auto* table = reinterpret_cast<WeightPackEntry*>(dev);
  auto* off = reinterpret_cast<int64_t*>(reinterpret_cast<uint8_t*>(dev) + (sizeof(WeightPackEntry) + 7) / 8 * 8);
  ARGUS_CUDA(cudaStreamSynchronize(static_cast<cudaStream_t>(stream)));
  ARGUS_CUDA(cudaMemcpy(table, &e, sizeof(e), cudaMemcpyHostToDevice));
  ARGUS_CUDA(cudaMemcpy(off, &zero, sizeof(zero), cudaMemcpyHostToDevice));
  pack_weights_scaled(w, scale, off, static_cast<bf16*>(packed), table, 1, static_cast<cudaStream_t>(stream));
  ARGUS_CUDA(cudaStreamSynchronize(static_cast<cudaStream_t>(stream)));
  ARGUS_API_END
}
int argus_stem_dgrad(const void* dy, const void* w, float* dx, int N, int H, int W, void* stream) {
  ARGUS_API_BEGIN
  require_sm100();
  stem_dgrad(static_cast<const __nv_bfloat16*>(dy), static_cast<const __nv_bfloat16*>(w), dx, N, H, W,
             static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}

int argus_bn_finalize(const float* partial, int slots, double count, const float* gamma, const float* beta,
                      float* running_mean, float* running_var, float momentum, float eps, float* scale, float* shift,
                      float* save_mean, float* save_invstd, int C, void* stream) {
  ARGUS_API_BEGIN
  require_sm100();
  bn_finalize(partial, slots, count, gamma, beta, running_mean, running_var, momentum, eps, scale, shift, save_mean,
              save_invstd, C, static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}
int argus_bn_apply(const void* x, const float* scale, const float* shift, const void* res, const float* rscale,
                   const float* rshift, int relu, void* y, int64_t rows, int C, void* stream) {
  ARGUS_API_BEGIN
  require_sm100();
  bn_apply(static_cast<const bf16*>(x), scale, shift, static_cast<const bf16*>(res), rscale, rshift, relu,
           static_cast<bf16*>(y), nullptr, nullptr, rows, C, static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}
int argus_bn_apply_bits(const void* x, const float* scale, const float* shift, const void* res, const float* rscale,
                        const float* rshift, int relu, void* y, void* relu_bits, int64_t rows, int C, void* stream) {
  ARGUS_API_BEGIN
  require_sm100();
  bn_apply(static_cast<const bf16*>(x), scale, shift, static_cast<const bf16*>(res), rscale, rshift, relu,
           static_cast<bf16*>(y), static_cast<uint8_t*>(relu_bits), nullptr, rows, C, static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}
int argus_bn_backward(void* dy, const void* x, const void* out, const float* scale, const float* shift,
                      const float* mean, const float* invstd, float* dgamma, float* dbeta, void* dx, int64_t rows,
                      int C, int mask_mode, void* stream) {
  ARGUS_API_BEGIN
  require_sm100();
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  bn_check_aligned(dy, x, out, dx);   // dx too: the reduce pass below already adds to dgamma / dbeta
  bn_bwd_reduce(static_cast<const bf16*>(dy), static_cast<const bf16*>(x), static_cast<const bf16*>(out), scale, shift,
                mean, invstd, dgamma, dbeta, rows, C, mask_mode, lib_scratch(bn_bwd_scratch_elems()), s);
  bn_bwd_apply(static_cast<bf16*>(dy), static_cast<const bf16*>(x), static_cast<const bf16*>(out), scale, shift, mean,
               invstd, dgamma, dbeta, static_cast<bf16*>(dx), rows, C, mask_mode, s);
  ARGUS_API_END
}
int argus_maxpool_forward(const void* x, const float* scale, const float* shift, void* y, void* idx, int N, int H,
                          int W, int C, void* stream) {
  ARGUS_API_BEGIN
  require_sm100();
  ARGUS_CHECK(H % 2 == 0 && W % 2 == 0 && C % 8 == 0, "maxpool: even H, W and C % 8 == 0 required");
  maxpool_fwd(static_cast<const bf16*>(x), scale, shift, static_cast<bf16*>(y), static_cast<uint8_t*>(idx), N, H, W, C,
              static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}
int argus_maxpool_backward(const void* dy, const void* idx, void* dx, int N, int H, int W, int C, void* stream) {
  ARGUS_API_BEGIN
  require_sm100();
  maxpool_bwd(static_cast<const bf16*>(dy), static_cast<const uint8_t*>(idx), static_cast<bf16*>(dx), N, H, W, C,
              static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}
int argus_stem_pool_bn_backward(const void* dpool, const void* idx, const void* raw, const float* scale,
                                const float* shift, const float* mean, const float* invstd, float* dgamma,
                                float* dbeta, void* dx, int N, int H, int W, int C, void* stream) {
  ARGUS_API_BEGIN
  require_sm100();
  stem_pool_bn_backward(static_cast<const bf16*>(dpool), static_cast<const uint8_t*>(idx), static_cast<const bf16*>(raw),
                        scale, shift, mean, invstd, dgamma, dbeta, static_cast<bf16*>(dx), N, H, W, C,
                        lib_scratch(bn_bwd_scratch_elems()), static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}
int argus_avgpool_forward(const void* x, void* y, int N, int HW, int C, void* stream) {
  ARGUS_API_BEGIN
  require_sm100();
  avgpool_fwd(static_cast<const bf16*>(x), static_cast<bf16*>(y), N, HW, C, static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}
int argus_avgpool_backward(const void* dy, void* dx, int N, int HW, int C, void* stream) {
  ARGUS_API_BEGIN
  require_sm100();
  avgpool_bwd(static_cast<const bf16*>(dy), static_cast<bf16*>(dx), nullptr, N, HW, C, static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}

int argus_augment_sample_params(float* params, int n_images, int n_cams, int H, int W, uint64_t seed, uint64_t step,
                                const argus_aug_config* cfg, void* stream) {
  ARGUS_API_BEGIN
  require_sm100();
  ARGUS_CHECK(cfg != nullptr && params != nullptr && n_cams >= 1, "bad augmentation arguments");
  AugConfig c;
  c.color_jiggle = cfg->color_jiggle; c.planckian_jitter = cfg->planckian_jitter; c.blur = cfg->blur;
  c.motion_blur = cfg->motion_blur; c.plasma_shadow = cfg->plasma_shadow;
  c.brightness_lo = cfg->brightness_lo; c.brightness_span = cfg->brightness_span;
  c.contrast_lo = cfg->contrast_lo; c.contrast_span = cfg->contrast_span;
  c.saturation_lo = cfg->saturation_lo; c.saturation_span = cfg->saturation_span;
  c.hue_lo = cfg->hue_lo; c.hue_span = cfg->hue_span;
  c.random_erasing = cfg->random_erasing; c.salt_and_pepper = cfg->salt_and_pepper;
  augment_sample_params(params, n_images, n_cams, H, W, seed, step, c, static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}
int argus_augment(const void* in, int in_u8, void* out, int out_s2d, const float* params, const void* arc_mask,
                  void* plasma_ws, int n_images, int H, int W, int apply, void* stream) {
  ARGUS_API_BEGIN
  require_sm100();
  ARGUS_CHECK(!apply || params != nullptr, "augmentation needs a parameter table");
  augment_images(in, in_u8 != 0, out, out_s2d != 0, params, static_cast<const uint32_t*>(arc_mask),
                 static_cast<uint32_t*>(plasma_ws), n_images, H, W, apply != 0, static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}

int argus_spaghetti_sample_params(float* arcs, int n_images, int n_arcs, int H, int W, uint64_t seed, uint64_t step,
                                  void* stream) {
  ARGUS_API_BEGIN
  require_sm100();
  ARGUS_CHECK(arcs != nullptr, "null arc table");
  spaghetti_sample_params(arcs, n_images, n_arcs, H, W, seed, step, static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}
int argus_spaghetti_mask(const float* arcs, void* mask, int n_images, int n_arcs, int H, int W, void* stream) {
  ARGUS_API_BEGIN
  require_sm100();
  ARGUS_CHECK(mask != nullptr && (arcs != nullptr || n_arcs == 0), "null argument");
  spaghetti_mask(arcs, static_cast<uint32_t*>(mask), n_images, n_arcs, H, W, static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}
int argus_spaghetti_draw(const void* in, void* out, const float* arcs, void* mask_ws, int n_images, int n_arcs, int H,
                         int W, void* stream) {
  ARGUS_API_BEGIN
  require_sm100();
  ARGUS_CHECK(in != nullptr && out != nullptr && mask_ws != nullptr && (arcs != nullptr || n_arcs == 0), "null argument");
  spaghetti_draw(static_cast<const uint8_t*>(in), static_cast<uint8_t*>(out), arcs, static_cast<uint32_t*>(mask_ws),
                 n_images, n_arcs, H, W, static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}

int argus_pose_loss(const float* pred, const float* target, float* loss, float* loss_mean, float* grad, int B,
                    float grad_scale, void* stream) {
  ARGUS_API_BEGIN
  require_sm100();
  ARGUS_CHECK(B >= 0, "negative batch");
  pose_loss_fwd_bwd(pred, target, loss, loss_mean, grad, B, grad_scale, static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}

int argus_pose_exp(const float* pred, float* pose, int B, int wxyz, void* stream) {
  ARGUS_API_BEGIN
  require_sm100();
  pose_exp(pred, pose, B, wxyz, static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}

int argus_clip_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n,
                         float* scratch, float gscale, float max_norm, float lr, float beta1, float beta2, float eps,
                         int step, float* norm_out, void* stream) {
  ARGUS_API_BEGIN
  require_sm100();
  ARGUS_CHECK(step >= 1, "Adam step counter starts at 1");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int np = grad_sqnorm_partials(grads, n, scratch, s);
  clip_adam_step(params, grads, exp_avg, exp_avg_sq, n, scratch, np, gscale, max_norm, lr, beta1, beta2, eps, step,
                 norm_out, false, s);
  ARGUS_API_END
}
int argus_clip_adam_step_amp(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n,
                             float* scratch, float gscale, float max_norm, float lr, float beta1, float beta2, float eps,
                             int step, float* norm_out, void* stream) {
  ARGUS_API_BEGIN
  require_sm100();
  ARGUS_CHECK(step >= 1, "Adam step counter starts at 1");
  ARGUS_CHECK(norm_out != nullptr, "the caller needs the gradient norm to learn whether the step was skipped");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int np = grad_sqnorm_partials(grads, n, scratch, s);
  clip_adam_step(params, grads, exp_avg, exp_avg_sq, n, scratch, np, gscale, max_norm, lr, beta1, beta2, eps, step,
                 norm_out, true, s);
  ARGUS_API_END
}

// ---- fp32 parity-mode primitives -----------------------------------------------------------------------------
static ConvShapeF32 make_shape_f32(int N, int H, int W, int Cin, int Cout, int k, int stride) {
  ARGUS_CHECK(N > 0 && H > 0 && W > 0 && Cin > 0 && Cout > 0, "empty convolution");
  ARGUS_CHECK((k == 1 || k == 3 || k == 7) && (stride == 1 || stride == 2), "fp32 conv: k in {1,3,7}, stride in {1,2}");
  ConvShapeF32 s;
  s.N = N; s.H = H; s.W = W; s.Cin = Cin; s.Cout = Cout; s.k = k; s.stride = stride;
  return s;
}
int argus_fp32_conv2d_forward(const float* x, const float* w, const float* bias, float* y, int N, int H, int W, int Cin,
                              int Cout, int k, int stride, void* stream) {
  ARGUS_API_BEGIN
  require_sm100();
  conv_f32_forward(make_shape_f32(N, H, W, Cin, Cout, k, stride), x, w, bias, y, static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}
int argus_fp32_conv2d_dgrad(const float* dy, const float* w, float* dx, int N, int H, int W, int Cin, int Cout, int k,
                            int stride, void* stream) {
  ARGUS_API_BEGIN
  require_sm100();
  conv_f32_dgrad(make_shape_f32(N, H, W, Cin, Cout, k, stride), dy, w, dx, static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}
int argus_fp32_conv2d_wgrad(const float* dy, const float* x, float* dw, int N, int H, int W, int Cin, int Cout, int k,
                            int stride, void* stream) {
  ARGUS_API_BEGIN
  require_sm100();
  const ConvShapeF32 s = make_shape_f32(N, H, W, Cin, Cout, k, stride);
  conv_f32_wgrad(s, dy, x, dw, lib_scratch(conv_f32_wgrad_scratch_elems(s, nullptr)), static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}
static double* lib_scratch_f64(int64_t elems) { return reinterpret_cast<double*>(lib_scratch(2 * elems)); }
int argus_fp32_bn_train(const float* x, int64_t rows, int C, const float* gamma, const float* beta, float* running_mean,
                        float* running_var, float momentum, float eps, float* scale, float* shift, float* save_mean,
                        float* save_invstd, void* stream) {
  ARGUS_API_BEGIN
  require_sm100();
  bn_f32_train_stats(x, rows, C, gamma, beta, running_mean, running_var, momentum, eps, scale, shift, save_mean,
                     save_invstd, lib_scratch_f64(static_cast<int64_t>(kBnF32MaxBlocks) * 2 * C),
                     static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}
int argus_fp32_bn_apply(const float* x, const float* scale, const float* shift, const float* res, const float* rscale,
                        const float* rshift, int relu, float* y, int64_t rows, int C, void* stream) {
  ARGUS_API_BEGIN
  require_sm100();
  bn_f32_apply(x, scale, shift, res, rscale, rshift, relu, y, rows, C, static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}
int argus_fp32_bn_backward(const float* dy, const float* x, const float* out, const float* scale, const float* mean,
                           const float* invstd, float* dgamma, float* dbeta, float* dx, float* g_out, int64_t rows,
                           int C, void* stream) {
  ARGUS_API_BEGIN
  require_sm100();
  double* part = lib_scratch_f64(static_cast<int64_t>(kBnF32MaxBlocks) * 2 * C + C);
  float* sums = reinterpret_cast<float*>(part + static_cast<int64_t>(kBnF32MaxBlocks) * 2 * C);
  bn_f32_backward(dy, x, out, scale, mean, invstd, dgamma, dbeta, dx, g_out, rows, C, part, sums,
                  static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}
int argus_fp32_maxpool_forward(const float* x, float* y, void* idx, int N, int H, int W, int C, void* stream) {
  ARGUS_API_BEGIN
  require_sm100();
  maxpool_f32_fwd(x, y, static_cast<uint8_t*>(idx), N, H, W, C, static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}
int argus_fp32_maxpool_backward(const float* dy, const void* idx, float* dx, int N, int H, int W, int C, void* stream) {
  ARGUS_API_BEGIN
  require_sm100();
  maxpool_f32_bwd(dy, static_cast<const uint8_t*>(idx), dx, N, H, W, C, static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}

struct argus_model {
  Model impl;
  argus_model(int n_cams, int dim) : impl(n_cams, dim) {}
};

int argus_model_create(argus_model** out, int n_cams, int resnet_output_dim) {
  ARGUS_API_BEGIN
  ARGUS_CHECK(out != nullptr, "null out pointer");
  *out = new argus_model(n_cams, resnet_output_dim);
  ARGUS_API_END
}
int argus_model_destroy(argus_model* m) {
  ARGUS_API_BEGIN
  delete m;
  ARGUS_API_END
}
int argus_model_counts(argus_model* m, int* n_params, int* n_buffers, int64_t* param_elems, int64_t* buffer_elems) {
  ARGUS_API_BEGIN
  ARGUS_CHECK(m != nullptr, "null model");
  if (n_params) *n_params = static_cast<int>(m->impl.params().size());
  if (n_buffers) *n_buffers = static_cast<int>(m->impl.buffers().size());
  if (param_elems) *param_elems = m->impl.num_param_elems();
  if (buffer_elems) *buffer_elems = m->impl.num_buffer_elems();
  ARGUS_API_END
}
int argus_model_tensor_info(argus_model* m, int is_buffer, int index, char* name, int name_cap, int64_t* offset,
                            int64_t* numel, int* ndim, int64_t* shape) {
  ARGUS_API_BEGIN
  ARGUS_CHECK(m != nullptr, "null model");
  const auto& v = is_buffer ? m->impl.buffers() : m->impl.params();
  ARGUS_CHECK(index >= 0 && index < static_cast<int>(v.size()), "tensor index out of range");
  const TensorInfo& t = v[index];
  if (name && name_cap > 0) {
    std::strncpy(name, t.name.c_str(), name_cap - 1);
    name[name_cap - 1] = 0;
  }
  if (offset) *offset = t.offset;
  if (numel) *numel = t.numel;
  if (ndim) *ndim = t.ndim;
  if (shape) for (int i = 0; i < 4; ++i) shape[i] = t.shape[i];
  ARGUS_API_END
}
int argus_model_bind(argus_model* m, float* params, float* grads, float* buffers) {
  ARGUS_API_BEGIN
  ARGUS_CHECK(m != nullptr, "null model");
  m->impl.bind(params, grads, buffers);
  ARGUS_API_END
}
int argus_model_reserve(argus_model* m, int max_batch, int H, int W, int training) {
  ARGUS_API_BEGIN
  ARGUS_CHECK(m != nullptr, "null model");
  m->impl.reserve(max_batch, H, W, training != 0);
  ARGUS_API_END
}
int argus_model_sync_weights(argus_model* m, void* stream) {
  ARGUS_API_BEGIN
  ARGUS_CHECK(m != nullptr, "null model");
  m->impl.sync_weights(static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}
int argus_model_forward(argus_model* m, const void* x, int is_u8, int B, int H, int W, int training, float* out,
                        void* stream) {
  ARGUS_API_BEGIN
  ARGUS_CHECK(m != nullptr, "null model");
  m->impl.forward(x, is_u8 != 0, B, H, W, training != 0, out, static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}
int argus_model_forward_frozen(argus_model* m, const void* x, int is_u8, int B, int H, int W, float* out, void* stream) {
  ARGUS_API_BEGIN
  ARGUS_CHECK(m != nullptr, "null model");
  m->impl.forward(x, is_u8 != 0, B, H, W, false, out, static_cast<cudaStream_t>(stream), true);
  ARGUS_API_END
}
int argus_model_stage_input_u8(argus_model* m, const void* images, const float* aug_params, const void* arc_mask,
                               void* plasma_ws, int B, int H, int W, int training, int apply, void* stream) {
  ARGUS_API_BEGIN
  ARGUS_CHECK(m != nullptr, "null model");
  m->impl.stage_input_u8(static_cast<const uint8_t*>(images), aug_params, static_cast<const uint32_t*>(arc_mask),
                         static_cast<uint32_t*>(plasma_ws), B, H, W, training != 0, apply != 0,
                         static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}
int argus_model_stage_input_frozen_u8(argus_model* m, const void* images, const float* aug_params, const void* arc_mask,
                                      void* plasma_ws, int B, int H, int W, int apply, void* stream) {
  ARGUS_API_BEGIN
  ARGUS_CHECK(m != nullptr, "null model");
  m->impl.stage_input_u8(static_cast<const uint8_t*>(images), aug_params, static_cast<const uint32_t*>(arc_mask),
                         static_cast<uint32_t*>(plasma_ws), B, H, W, false, apply != 0,
                         static_cast<cudaStream_t>(stream), true);
  ARGUS_API_END
}
int argus_model_set_precision(argus_model* m, int mode) {
  ARGUS_API_BEGIN
  ARGUS_CHECK(m != nullptr, "null model");
  m->impl.set_precision(mode);
  ARGUS_API_END
}
int argus_model_set_wgrad_overlap(argus_model* m, int on) {
  ARGUS_API_BEGIN
  ARGUS_CHECK(m != nullptr, "null model");
  m->impl.set_wgrad_overlap(on != 0);
  ARGUS_API_END
}
int argus_model_zero_grads(argus_model* m, void* stream) {
  ARGUS_API_BEGIN
  ARGUS_CHECK(m != nullptr, "null model");
  m->impl.zero_grads(static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}
int argus_model_backward(argus_model* m, const float* d_out, int stage_begin, int stage_end, void* stream) {
  ARGUS_API_BEGIN
  ARGUS_CHECK(m != nullptr, "null model");
  ARGUS_CHECK(0 <= stage_begin && stage_begin <= stage_end && stage_end <= 4, "bad stage range");
  m->impl.backward(d_out, stage_begin, stage_end, static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}
int argus_model_input_grad(argus_model* m, float* dx, void* stream) {
  ARGUS_API_BEGIN
  ARGUS_CHECK(m != nullptr, "null model");
  ARGUS_CHECK(dx != nullptr, "null gradient buffer");
  m->impl.input_grad(dx, static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}
int argus_model_stage_range(argus_model* m, int stage, int64_t* begin, int64_t* end) {
  ARGUS_API_BEGIN
  ARGUS_CHECK(m != nullptr, "null model");
  m->impl.stage_param_range(stage, begin, end);
  ARGUS_API_END
}
int argus_model_copy_activation(argus_model* m, int index, void* dst, int64_t capacity_elems, int64_t* rows, int* C,
                                void* stream) {
  ARGUS_API_BEGIN
  ARGUS_CHECK(m != nullptr, "null model");
  m->impl.copy_activation(index, dst, capacity_elems, rows, C, static_cast<cudaStream_t>(stream));
  ARGUS_API_END
}
int argus_model_arena_bytes(argus_model* m, int64_t* bytes) {
  ARGUS_API_BEGIN
  ARGUS_CHECK(m != nullptr, "null model");
  *bytes = static_cast<int64_t>(m->impl.arena_bytes());
  ARGUS_API_END
}

}  // extern "C"

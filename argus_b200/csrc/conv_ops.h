// Host-side planning for the tcgen05 convolution kernels: turns a convolution shape plus device pointers into
// kernel parameter blocks (TMA tensor maps, filter-tap tables, tile counts) once, so the hot path only launches.
#pragma once
#include <array>
#include <vector>

#include "conv_gemm.cuh"
#include "runtime.h"

namespace argus {

// A convolution over NHWC bf16 activations with [Cout][kh][kw][Cin] bf16 weights.
// kind: 0 = ordinary k x k convolution (k in {1,3}, stride in {1,2}, pad = k/2)
//       1 = ResNet stem: 7x7 stride-2 pad-3 convolution over 3 channels, expressed on the space-to-depth
//           input written by the input-packing kernel: x_s2d[N][H/2][W/2 + 4][16], so that every output pixel
//           reads four 128-byte windows (one per s2d row offset); weights are repacked to [64][4][64].
struct ConvShape {
  int N = 0, H = 0, W = 0;  // input image count and spatial size (stem: the ORIGINAL image size)
  int Cin = 0, Cout = 0;
  int k = 1, stride = 1;
  int kind = 0;
  int Ho() const { return H / stride; }
  int Wo() const { return W / stride; }
  int Ktot() const { return kind == 1 ? 256 : k * k * Cin; }
  int64_t out_pixels() const { return static_cast<int64_t>(N) * Ho() * Wo(); }
};

struct Epilogue {
  const float* scale = nullptr;
  const float* shift = nullptr;
  const __nv_bfloat16* residual = nullptr;
  const uint8_t* residual_bits = nullptr;   // optional [rows][Cout/8] ReLU bit mask gating the residual (dgrad)
  const uint8_t* out_bits = nullptr;        // optional [rows][Cout/8] ReLU bit mask applied to the stored result
  const float* res_scale = nullptr;         // optional per-channel affine on the residual (both or neither)
  const float* res_shift = nullptr;
  uint8_t* relu_bits_out = nullptr;         // optional [rows][Cout/8]: (pre-ReLU value > 0), written by the epilogue
  int relu = 0;
  float* stat_partial = nullptr;   // [stat_slots(launch)][2][Cout], zeroed by the caller (train-mode BN statistics)
  // Fused batch-norm backward reduction (dgrad launches that produce the gradient of a BN + ReLU output, dense output
  // only): bn_raw = that layer's saved pre-BN output, bn_scale / bn_shift = its folded batch statistics. The result is
  // stored masked by (bn_raw * bn_scale + bn_shift > 0) and stat_partial receives sum(g), sum(g * bn_raw).
  const __nv_bfloat16* bn_raw = nullptr;
  const float* bn_scale = nullptr;
  const float* bn_shift = nullptr;
  int early_trigger = 0;   // ConvGemmParams::early_trigger (the eval-mode forward sets it)
};

// geometry of the (non-strided) output tensor map, kept so that a residual tensor map can be built per launch
struct TmapGeom {
  int rank = 0;
  uint64_t dims[4] = {0, 0, 0, 0};
  uint64_t strides[3] = {0, 0, 0};
  uint32_t box[4] = {0, 0, 0, 0};
  void set(int r, const uint64_t* d, const uint64_t* s, const uint32_t* b) {
    rank = r;
    for (int i = 0; i < r; ++i) { dims[i] = d[i]; box[i] = b[i]; }
    for (int i = 0; i + 1 < r; ++i) strides[i] = s[i];
  }
};

struct ConvLaunch {
  ConvGemmParams p;
  int block_n = 64;
  int b_mn = 0;
  TmapGeom out_geom;
};

struct WgradLaunch {
  const char* family = "conv_wgrad";   // profiling family (the Gram GEMM of the algebraic BN backward is not a conv)
  WgradParams p;
  int block_n = 64;
  // Cout == 64 layers use the transposed all-taps kernel instead (xpose_nbox = padded box count, 0 = not used)
  int xpose_nbox = 0;
  WgradXposeParams xp;
};

void validate_shape(const ConvShape& s);

// y[N,Ho,Wo,Cout] = conv(x, w)   (epilogue pointers are patched per launch)
ConvLaunch plan_conv_forward(const ConvShape& s, const __nv_bfloat16* x, const __nv_bfloat16* w, __nv_bfloat16* y);
// dx[N,H,W,Cin] = conv_transpose(dy, w); stride-2 convolutions need one launch per input-pixel parity class.
// Pixels that receive no contribution (1x1 stride 2) are NOT written: the caller zero-fills dx first.
std::vector<ConvLaunch> plan_conv_dgrad(const ConvShape& s, const __nv_bfloat16* dy, const __nv_bfloat16* w,
                                        __nv_bfloat16* dx);
// dw[Cout][Ktot] (fp32, accumulated with atomics: caller zero-fills) = dy^T * im2col(x)
// 1x1 dgrad over a concatenated K: dx[p, n] = sum_{k < Cout} dy[p, k] B[k, n] + sum_{k < C1} a1[p, k] B[Cout + k, n]
// with B = bstack, a row-major [(Cout + C1)][Cin] bf16 matrix, and a1 an (N, H, W, C1) activation on the conv INPUT
// grid (stride 2: its even pixels; as for every strided dgrad the caller zero-fills dx first).
ConvLaunch plan_dgrad_concat(const ConvShape& s, const __nv_bfloat16* dy, const __nv_bfloat16* a1, int C1,
                             const __nv_bfloat16* bstack, __nv_bfloat16* dx);
WgradLaunch plan_conv_wgrad(const ConvShape& s, const __nv_bfloat16* dy, const __nv_bfloat16* x, float* dw);

// 1x1 only: dw[(Cout + Cin)][Cin] (fp32, +=): rows < Cout = dy^T x (the weight gradient), rows Cout + j = x^T x (the
// Gram matrix of the input pixels the convolution reads); Cout must be a multiple of 128. One launch.
WgradLaunch plan_conv_wgrad_gram(const ConvShape& s, const __nv_bfloat16* dy, const __nv_bfloat16* x, float* dw);

// g[Cin][Cin] (fp32, +=) = x_s^T x_s over the input pixels x_s a 1x1 convolution of shape s reads (its even pixels at
// stride 2): the Gram matrix from which the batch statistics of the convolution's OUTPUT follow without computing it.
WgradLaunch plan_gram(const ConvShape& s, const __nv_bfloat16* x, float* g);

// Input gradient of the stem (stem_dgrad.cu): dy (N, H/2, W/2, 64) bf16 NHWC, w the [64][256] packed stem weight of the
// forward, dx (N, 3, H, W) fp32 NCHW, fully overwritten. H, W powers of two >= 32, W <= 1024. Deterministic.
void stem_dgrad(const __nv_bfloat16* dy, const __nv_bfloat16* w, float* dx, int N, int H, int W, cudaStream_t stream);

void launch_conv(const ConvLaunch& l, const Epilogue& e, cudaStream_t stream);

// The conv_gemm_kernel<block_n, b_mn, opt> instance a launch runs (opt = kOptAll for the generic kernel).
struct ConvInstance {
  int block_n = 0, b_mn = 0, opt = 0;
};
// Kernel parameters of launch l with epilogue e (residual / raw-tile tensor maps included); checks the combination.
ConvGemmParams epilogue_params(const ConvLaunch& l, const Epilogue& e);
// The instance launch_conv dispatches p to. Pure: the launcher and conv_launch_info both call it.
ConvInstance select_conv_instance(const ConvLaunch& l, const ConvGemmParams& p);
// Everything launch_conv decides for (l, e) without launching: the instance, the final halo / weights-resident mode,
// the tile counts and the grid.
struct ConvLaunchInfo {
  ConvInstance inst;
  int halo = 0, b_resident = 0, halo_stages = 0;
  int num_m_tiles = 0, num_n_tiles = 0, grid = 0, stat_slots = 0;
};
ConvLaunchInfo conv_launch_info(const ConvLaunch& l, const Epilogue& e);
// While recording is on, launch_conv adds the key (block_n, b_mn, opt, halo, b_resident) of every launch to a host-side
// set; turning it on clears the set.
void conv_instances_record(bool on);
std::vector<std::array<int, 5>> conv_instances_recorded();
// (block_n, b_mn, opt) of every kernel instance launch_conv can dispatch to
std::vector<std::array<int, 3>> conv_instances_all();
// number of statistic slots launch_conv writes for this launch (one per epilogue group per CTA)
int stat_slots(const ConvLaunch& l);
// elements of split-K scratch this launch needs (0 when it does not split)
int64_t wgrad_scratch_elems(const WgradLaunch& l);
// scratch: at least wgrad_scratch_elems(l) floats (may be null when that is 0)
void launch_wgrad(const WgradLaunch& l, float* scratch, cudaStream_t stream);

}  // namespace argus

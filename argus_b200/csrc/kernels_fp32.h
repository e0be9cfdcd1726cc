// Launchers of the fp32 parity mode (see fp32_kernels.cu). All tensors are fp32 device pointers, activations NHWC,
// weights and weight gradients in PyTorch's [Cout][Cin][kh][kw] layout.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace argus {

struct ConvShapeF32 {
  int N = 0, H = 0, W = 0;   // input
  int Cin = 0, Cout = 0;
  int k = 1, stride = 1;     // square kernel, padding k/2
  int Ho() const { return (H + 2 * (k / 2) - k) / stride + 1; }
  int Wo() const { return (W + 2 * (k / 2) - k) / stride + 1; }
};

// kernel parameter block of the SIMT implicit GEMM (filled by the launchers)
struct ConvF32 {
  const float* x;
  const float* w;
  const float* dy;
  const float* bias;
  float* out;
  float* partial;
  int N, H, W, Cin, Cout, KH, KW, stride, pad, Ho, Wo;
  int M, Ncol, K, k_per_split;
};

// y = conv(x, w) (+ bias per output channel)
void conv_f32_forward(const ConvShapeF32& s, const float* x, const float* w, const float* bias, float* y,
                      cudaStream_t st);
// dx = conv_transpose(dy, w)   (every input pixel is written)
void conv_f32_dgrad(const ConvShapeF32& s, const float* dy, const float* w, float* dx, cudaStream_t st);
// dw += dy^T im2col(x), split over pixels; partial sums are added in split order in fp64 (deterministic)
int64_t conv_f32_wgrad_scratch_elems(const ConvShapeF32& s, int* splits_out);
void conv_f32_wgrad(const ConvShapeF32& s, const float* dy, const float* x, float* dw, float* scratch, cudaStream_t st);

// (B, 3*n_cams, H, W) NCHW == (B*n_cams, 3, H, W) -> NHWC; u8 HWC images -> fp32 / 255
void pack_input_nhwc_f32(const float* x_nchw, float* y_nhwc, int n_images, int H, int W, cudaStream_t s);
void pack_input_u8_f32(const uint8_t* x_hwc, float* y_nhwc, int n_images, int H, int W, cudaStream_t s);
// the inverse of pack_input_nhwc_f32, for the input gradient: (n, H, W, 3) NHWC -> (B, 3*n_cams, H, W) NCHW
void unpack_input_grad_nhwc_f32(const float* dx_nhwc, float* dx_nchw, int n_images, int H, int W, cudaStream_t s);

constexpr int kBnF32MaxBlocks = 1024;   // scratch: kBnF32MaxBlocks * 2 * C doubles
// batch statistics (fp64 sums) -> scale/shift/mean/invstd + running-stat update (torch.nn.BatchNorm2d semantics)
void bn_f32_train_stats(const float* x, int64_t rows, int C, const float* gamma, const float* beta, float* running_mean,
                        float* running_var, float momentum, float eps, float* scale, float* shift, float* save_mean,
                        float* save_invstd, double* scratch, cudaStream_t s);
// y = [relu](x*scale+shift [+ res | + res*rscale+rshift])
void bn_f32_apply(const float* x, const float* scale, const float* shift, const float* res, const float* rscale,
                  const float* rshift, int relu, float* y, int64_t rows, int C, cudaStream_t s);
// g = dy masked by (out > 0) when out != nullptr; dgamma += sum g*xhat, dbeta += sum g; dx = BN input gradient;
// g_out (optional) receives g. sums: 2*C floats of scratch. frozen_stats: mean / invstd are constants (eval-mode
// statistics), so dx = scale * g (the batch-mean terms are multiplied by 0); dgamma / dbeta are the same sums.
void bn_f32_backward(const float* dy, const float* x, const float* out, const float* scale, const float* mean,
                     const float* invstd, float* dgamma, float* dbeta, float* dx, float* g_out, int64_t rows, int C,
                     double* scratch, float* sums, cudaStream_t s, bool frozen_stats = false);

void maxpool_f32_fwd(const float* x, float* y, uint8_t* idx, int N, int H, int W, int C, cudaStream_t s);
void maxpool_f32_bwd(const float* dy, const uint8_t* idx, float* dx, int N, int H, int W, int C, cudaStream_t s);
void avgpool_f32_fwd(const float* x, float* y, int N, int HW, int C, cudaStream_t s);
void avgpool_f32_bwd(const float* dy, float* dx, int N, int HW, int C, cudaStream_t s);
void add_f32(float* a, const float* b, int64_t n, cudaStream_t s);
void gelu_f32_fwd(const float* x, float* y, int64_t n, cudaStream_t s);
void gelu_f32_bwd(const float* dz, const float* x, float* dx, int64_t n, cudaStream_t s);
void colsum_f32(const float* x, float* out, int rows, int C, cudaStream_t s);

}  // namespace argus

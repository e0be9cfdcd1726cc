// fp32 parity mode ("fp32 mode" of the north star: forward outputs, losses and gradients within 1e-4 relative of the
// reference PyTorch fp32 implementation). Every tensor is fp32 NHWC, convolutions are SIMT implicit GEMMs with fp32
// FMA accumulation, every reduction (batch-norm statistics, BN backward sums, split-K weight gradients) is
// accumulated in fp64 in a fixed order, so the mode is deterministic and as accurate as the reference's own fp32 path.
// It is a validation mode: correctness and clarity over speed (no tensor cores, no fusion).
//
// Reference semantics: torch.nn.Conv2d / BatchNorm2d / ReLU / MaxPool2d(3,2,1) / AdaptiveAvgPool2d(1) / Linear inside
// torchvision resnet50 as called from /root/reference/argus/models.py:81-90. Weights and weight gradients are read
// and written directly in PyTorch's [Cout][Cin][kh][kw] layout (no packed copies).
#include "kernels_fp32.h"
#include "ptx.cuh"
#include "runtime.h"

#include <algorithm>

namespace argus {

namespace {

constexpr int BM = 64, BN = 64, BK = 16;

// element (m, k) of the implicit im2col matrix of an NHWC tensor: m = output pixel, k = (kh*KW + kw)*C + c
__device__ __forceinline__ float im2col_at(const float* __restrict__ x, const ConvF32& p, int m, int k) {
  const int c = k % p.Cin;
  const int tap = k / p.Cin;
  const int kw = tap % p.KW, kh = tap / p.KW;
  const int wo = m % p.Wo;
  const int t = m / p.Wo;
  const int ho = t % p.Ho, n = t / p.Ho;
  const int h = ho * p.stride - p.pad + kh, w = wo * p.stride - p.pad + kw;
  if (h < 0 || h >= p.H || w < 0 || w >= p.W) return 0.f;
  return __ldg(x + (static_cast<int64_t>(n * p.H + h) * p.W + w) * p.Cin + c);
}
__device__ __forceinline__ int64_t weight_index(const ConvF32& p, int co, int ci, int kh, int kw) {
  return ((static_cast<int64_t>(co) * p.Cin + ci) * p.KH + kh) * p.KW + kw;
}

// MODE 0: y[p, co]  = sum_k im2col(x)[p, k] * w[co, k]                      (forward)
// MODE 1: dx[q, ci] = sum_{kh,kw,co} dy[pixel reached from q by tap, co] * w[co, ci, kh, kw]   (input gradient)
// MODE 2: dw[co, j] = sum_p dy[p, co] * im2col(x)[p, j]                     (weight gradient, split over pixels)
template <int MODE>
__device__ __forceinline__ float load_a(const ConvF32& p, int m, int k) {
  if (MODE == 0) return im2col_at(p.x, p, m, k);
  if (MODE == 1) {
    const int co = k % p.Cout;
    const int tap = k / p.Cout;
    const int kw = tap % p.KW, kh = tap / p.KW;
    const int w = m % p.W;
    const int t = m / p.W;
    const int h = t % p.H, n = t / p.H;
    const int th = h + p.pad - kh, tw = w + p.pad - kw;
    if (th < 0 || tw < 0 || (th % p.stride) != 0 || (tw % p.stride) != 0) return 0.f;
    const int ho = th / p.stride, wo = tw / p.stride;
    if (ho >= p.Ho || wo >= p.Wo) return 0.f;
    return __ldg(p.dy + (static_cast<int64_t>(n * p.Ho + ho) * p.Wo + wo) * p.Cout + co);
  }
  return __ldg(p.dy + static_cast<int64_t>(k) * p.Cout + m);   // MODE 2: A[co, pixel]
}
template <int MODE>
__device__ __forceinline__ float load_b(const ConvF32& p, int k, int n) {
  if (MODE == 0) {
    const int ci = k % p.Cin;
    const int tap = k / p.Cin;
    return __ldg(p.w + weight_index(p, n, ci, tap / p.KW, tap % p.KW));
  }
  if (MODE == 1) {
    const int co = k % p.Cout;
    const int tap = k / p.Cout;
    return __ldg(p.w + weight_index(p, co, n, tap / p.KW, tap % p.KW));
  }
  return im2col_at(p.x, p, k, n);   // MODE 2: B[pixel, j]
}

template <int MODE>
__global__ void __launch_bounds__(256) conv_f32_kernel(const ConvF32 p) {
  pdl_prologue();
  __shared__ float As[BK][BM + 4];
  __shared__ float Bs[BK][BN + 4];
  const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int k_begin = blockIdx.z * p.k_per_split;
  const int k_end = min(p.K, k_begin + p.k_per_split);
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  for (int k0 = k_begin; k0 < k_end; k0 += BK) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int e = threadIdx.x + 256 * i;
      // forward / dgrad: k is the contiguous memory direction of A; wgrad: m (= co) is
      const int am = (MODE == 2) ? (e & 63) : (e >> 4);
      const int ak = (MODE == 2) ? (e >> 6) : (e & 15);
      const int gm = m0 + am, gk = k0 + ak;
      As[ak][am] = (gm < p.M && gk < k_end) ? load_a<MODE>(p, gm, gk) : 0.f;
      // forward / dgrad: B = weights (k contiguous-ish); wgrad: B = im2col (n = j contiguous)
      const int bn = (MODE == 2) ? (e & 63) : (e >> 4);
      const int bk = (MODE == 2) ? (e >> 6) : (e & 15);
      const int gn = n0 + bn, gk2 = k0 + bk;
      Bs[bk][bn] = (gn < p.Ncol && gk2 < k_end) ? load_b<MODE>(p, gk2, gn) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < BK; ++k) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = As[k][ty * 4 + i];
#pragma unroll
      for (int j = 0; j < 4; ++j) b[j] = Bs[k][tx * 4 + j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int gm = m0 + ty * 4 + i;
    if (gm >= p.M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int gn = n0 + tx * 4 + j;
      if (gn >= p.Ncol) continue;
      if (MODE == 2) {
        p.partial[(static_cast<int64_t>(blockIdx.z) * p.M + gm) * p.Ncol + gn] = acc[i][j];
      } else {
        float v = acc[i][j];
        if (p.bias != nullptr) v += p.bias[gn];
        p.out[static_cast<int64_t>(gm) * p.Ncol + gn] = v;
      }
    }
  }
}

// dw[co][ci][kh][kw] += sum_z partial[z][co][j], j = (kh*KW + kw)*Cin + ci, splits added in order in fp64
__global__ void wgrad_reduce_f32_kernel(const ConvF32 p, float* __restrict__ dw, int splits) {
  pdl_prologue();
  const int64_t total = static_cast<int64_t>(p.M) * p.Ncol;
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    double s = 0.0;
    for (int z = 0; z < splits; ++z) s += static_cast<double>(p.partial[static_cast<int64_t>(z) * total + i]);
    const int co = static_cast<int>(i / p.Ncol), j = static_cast<int>(i % p.Ncol);
    const int ci = j % p.Cin, tap = j / p.Cin;
    const int64_t d = weight_index(p, co, ci, tap / p.KW, tap % p.KW);
    dw[d] = static_cast<float>(static_cast<double>(dw[d]) + s);
  }
}

}  // namespace

static ConvF32 make_conv(const ConvShapeF32& s) {
  ConvF32 p{};
  p.N = s.N; p.H = s.H; p.W = s.W; p.Cin = s.Cin; p.Cout = s.Cout; p.KH = s.k; p.KW = s.k; p.stride = s.stride;
  p.pad = s.k / 2;
  p.Ho = (s.H + 2 * p.pad - s.k) / s.stride + 1;
  p.Wo = (s.W + 2 * p.pad - s.k) / s.stride + 1;
  return p;
}

void conv_f32_forward(const ConvShapeF32& s, const float* x, const float* w, const float* bias, float* y,
                      cudaStream_t st) {
  ConvF32 p = make_conv(s);
  p.x = x; p.w = w; p.out = y; p.bias = bias;
  p.M = s.N * p.Ho * p.Wo; p.Ncol = s.Cout; p.K = s.k * s.k * s.Cin; p.k_per_split = p.K;
  ProfileScope prof("fp32_conv", st, 2.0 * p.M * static_cast<double>(p.Ncol) * p.K, 0);
  dim3 grid((p.Ncol + BN - 1) / BN, (p.M + BM - 1) / BM, 1);
  launch_kernel(conv_f32_kernel<0>, grid, 256, 0, st, p);
  ARGUS_CUDA(cudaGetLastError());
}

void conv_f32_dgrad(const ConvShapeF32& s, const float* dy, const float* w, float* dx, cudaStream_t st) {
  ConvF32 p = make_conv(s);
  p.dy = dy; p.w = w; p.out = dx;
  p.M = s.N * s.H * s.W; p.Ncol = s.Cin; p.K = s.k * s.k * s.Cout; p.k_per_split = p.K;
  ProfileScope prof("fp32_conv", st, 2.0 * p.M * static_cast<double>(p.Ncol) * p.K, 0);
  dim3 grid((p.Ncol + BN - 1) / BN, (p.M + BM - 1) / BM, 1);
  launch_kernel(conv_f32_kernel<1>, grid, 256, 0, st, p);
  ARGUS_CUDA(cudaGetLastError());
}

int64_t conv_f32_wgrad_scratch_elems(const ConvShapeF32& s, int* splits_out) {
  ConvF32 p = make_conv(s);
  const int64_t pixels = static_cast<int64_t>(s.N) * p.Ho * p.Wo;
  const int64_t mn = static_cast<int64_t>(s.Cout) * s.k * s.k * s.Cin;
  int64_t splits = std::max<int64_t>(1, (pixels + 2047) / 2048);
  splits = std::min<int64_t>(splits, 128);
  splits = std::min<int64_t>(splits, std::max<int64_t>(1, (48LL << 20) / mn));   // <= 192 MB of partials
  if (splits_out) *splits_out = static_cast<int>(splits);
  return splits * mn;
}

void conv_f32_wgrad(const ConvShapeF32& s, const float* dy, const float* x, float* dw, float* scratch,
                    cudaStream_t st) {
  ConvF32 p = make_conv(s);
  p.dy = dy; p.x = x; p.partial = scratch;
  p.M = s.Cout; p.Ncol = s.k * s.k * s.Cin; p.K = s.N * p.Ho * p.Wo;
  int splits = 1;
  conv_f32_wgrad_scratch_elems(s, &splits);
  p.k_per_split = ((p.K + splits - 1) / splits + BK - 1) / BK * BK;
  splits = (p.K + p.k_per_split - 1) / p.k_per_split;
  ProfileScope prof("fp32_conv", st, 2.0 * p.M * static_cast<double>(p.Ncol) * p.K, 0);
  dim3 grid((p.Ncol + BN - 1) / BN, (p.M + BM - 1) / BM, splits);
  launch_kernel(conv_f32_kernel<2>, grid, 256, 0, st, p);
  ARGUS_CUDA(cudaGetLastError());
  const int64_t total = static_cast<int64_t>(p.M) * p.Ncol;
  launch_kernel(wgrad_reduce_f32_kernel, static_cast<int>(std::min<int64_t>((total + 255) / 256, 4096)), 256, 0, st, p, dw, splits);
  ARGUS_CUDA(cudaGetLastError());
}

// ------------------------------------------------------------------------------------------------------------
// input layout
// ------------------------------------------------------------------------------------------------------------
__global__ void nchw_to_nhwc3_kernel(const float* __restrict__ x, float* __restrict__ y, int n_images, int HW) {
  pdl_prologue();
  const int64_t total = static_cast<int64_t>(n_images) * HW * 3;
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % 3);
    const int64_t t = i / 3;
    const int64_t pix = t % HW, n = t / HW;
    y[i] = x[(n * 3 + c) * HW + pix];
  }
}
// inverse of nchw_to_nhwc3_kernel: the input gradient (n, H, W, 3) NHWC -> (n, 3, H, W) NCHW
__global__ void nhwc3_to_nchw_kernel(const float* __restrict__ x, float* __restrict__ y, int n_images, int HW) {
  pdl_prologue();
  const int64_t total = static_cast<int64_t>(n_images) * HW * 3;
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t pix = i % HW;
    const int64_t t = i / HW;   // n * 3 + c
    y[i] = x[((t / 3) * HW + pix) * 3 + t % 3];
  }
}
__global__ void u8_to_f32_kernel(const uint8_t* __restrict__ x, float* __restrict__ y, int64_t n) {
  pdl_prologue();
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x)
    y[i] = static_cast<float>(x[i]) / 255.0f;
}
void pack_input_nhwc_f32(const float* x_nchw, float* y_nhwc, int n_images, int H, int W, cudaStream_t s) {
  const int64_t total = static_cast<int64_t>(n_images) * H * W * 3;
  launch_kernel(nchw_to_nhwc3_kernel, static_cast<int>(std::min<int64_t>((total + 255) / 256, 8192)), 256, 0, s, x_nchw, y_nhwc,
                                                                                                      n_images, H * W);
  ARGUS_CUDA(cudaGetLastError());
}
void unpack_input_grad_nhwc_f32(const float* dx_nhwc, float* dx_nchw, int n_images, int H, int W, cudaStream_t s) {
  const int64_t total = static_cast<int64_t>(n_images) * H * W * 3;
  launch_kernel(nhwc3_to_nchw_kernel, static_cast<int>(std::min<int64_t>((total + 255) / 256, 8192)), 256, 0, s, dx_nhwc,
                dx_nchw, n_images, H * W);
  ARGUS_CUDA(cudaGetLastError());
}
void pack_input_u8_f32(const uint8_t* x_hwc, float* y_nhwc, int n_images, int H, int W, cudaStream_t s) {
  const int64_t total = static_cast<int64_t>(n_images) * H * W * 3;
  launch_kernel(u8_to_f32_kernel, static_cast<int>(std::min<int64_t>((total + 255) / 256, 8192)), 256, 0, s, x_hwc, y_nhwc, total);
  ARGUS_CUDA(cudaGetLastError());
}

// ------------------------------------------------------------------------------------------------------------
// batch norm
// ------------------------------------------------------------------------------------------------------------
// partial[block][2][C] (fp64): per-block sums of a and a*b over its rows. MODE 0: a = x, b = x (statistics);
// MODE 1: a = g, b = xhat with g = dy masked by (out > 0) when out != nullptr (BN backward sums).
template <int MODE>
__global__ void __launch_bounds__(256)
bn_sums_f32_kernel(const float* __restrict__ x, const float* __restrict__ dy, const float* __restrict__ out,
                   const float* __restrict__ mean, const float* __restrict__ invstd, double* __restrict__ partial,
                   int64_t rows, int C) {
  pdl_prologue();
  // thread -> channel c = threadIdx.x % cl (+ multiples of cl), row lane = threadIdx.x / cl
  const int cl = C < 256 ? C : 256;
  const int row_lanes = 256 / cl;
  const int rl = threadIdx.x / cl, cc = threadIdx.x % cl;
  __shared__ double red[2][256];
  for (int c = cc; c < C; c += cl) {
    double s0 = 0.0, s1 = 0.0;
    const float mu = MODE == 1 ? mean[c] : 0.f, is = MODE == 1 ? invstd[c] : 0.f;
    for (int64_t r = static_cast<int64_t>(blockIdx.x) * row_lanes + rl; r < rows;
         r += static_cast<int64_t>(gridDim.x) * row_lanes) {
      const int64_t i = r * C + c;
      if (MODE == 0) {
        const double v = static_cast<double>(x[i]);
        s0 += v;
        s1 += v * v;
      } else {
        float g = dy[i];
        if (out != nullptr && !(out[i] > 0.f)) g = 0.f;
        const float xh = (x[i] - mu) * is;
        s0 += static_cast<double>(g);
        s1 += static_cast<double>(g) * static_cast<double>(xh);
      }
    }
    red[0][threadIdx.x] = s0;
    red[1][threadIdx.x] = s1;
    __syncthreads();
    if (rl == 0) {
      for (int k = 1; k < row_lanes; ++k) { s0 += red[0][k * cl + cc]; s1 += red[1][k * cl + cc]; }
      partial[(static_cast<int64_t>(blockIdx.x) * 2 + 0) * C + c] = s0;
      partial[(static_cast<int64_t>(blockIdx.x) * 2 + 1) * C + c] = s1;
    }
    __syncthreads();
  }
}

__global__ void bn_finalize_f64_kernel(const double* __restrict__ partial, int blocks, double count,
                                       const float* gamma, const float* beta, float* running_mean,
                                       float* running_var, float momentum, float eps, float* scale, float* shift,
                                       float* save_mean, float* save_invstd, int C) {
  pdl_prologue();
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  double sum = 0.0, sq = 0.0;
  for (int b = 0; b < blocks; ++b) {
    sum += partial[(static_cast<int64_t>(b) * 2 + 0) * C + c];
    sq += partial[(static_cast<int64_t>(b) * 2 + 1) * C + c];
  }
  const double mean = sum / count;
  double var = sq / count - mean * mean;
  if (var < 0) var = 0;
  const double invstd = 1.0 / sqrt(var + static_cast<double>(eps));
  const float sc = static_cast<float>(static_cast<double>(gamma[c]) * invstd);
  scale[c] = sc;
  shift[c] = static_cast<float>(static_cast<double>(beta[c]) - mean * static_cast<double>(gamma[c]) * invstd);
  save_mean[c] = static_cast<float>(mean);
  save_invstd[c] = static_cast<float>(invstd);
  if (running_mean != nullptr) {
    const double unbiased = count > 1 ? var * count / (count - 1) : var;
    running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * static_cast<float>(mean);
    running_var[c] = (1.f - momentum) * running_var[c] + momentum * static_cast<float>(unbiased);
  }
}
__global__ void bn_bwd_finalize_f64_kernel(const double* __restrict__ partial, int blocks, float* dgamma, float* dbeta,
                                           float* sum_g, float* sum_gx, int C) {
  pdl_prologue();
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  double sb = 0.0, sg = 0.0;
  for (int b = 0; b < blocks; ++b) {
    sb += partial[(static_cast<int64_t>(b) * 2 + 0) * C + c];
    sg += partial[(static_cast<int64_t>(b) * 2 + 1) * C + c];
  }
  dbeta[c] += static_cast<float>(sb);
  dgamma[c] += static_cast<float>(sg);
  sum_g[c] = static_cast<float>(sb);     // this call's sums (dgamma / dbeta may already hold other contributions)
  sum_gx[c] = static_cast<float>(sg);
}

static int bn_blocks(int64_t rows, int C) {
  const int cl = C < 256 ? C : 256;
  const int row_lanes = 256 / cl;
  const int64_t groups = (rows + row_lanes - 1) / row_lanes;
  return static_cast<int>(std::max<int64_t>(1, std::min<int64_t>(groups, kBnF32MaxBlocks)));
}

void bn_f32_train_stats(const float* x, int64_t rows, int C, const float* gamma, const float* beta, float* running_mean,
                        float* running_var, float momentum, float eps, float* scale, float* shift, float* save_mean,
                        float* save_invstd, double* scratch, cudaStream_t s) {
  ProfileScope prof("fp32_bn", s, 0, 4.0 * rows * C);
  ARGUS_CHECK(C <= 256 ? (256 % C == 0) : (C % 256 == 0), "fp32 batch norm: C must divide or be a multiple of 256");
  const int blocks = bn_blocks(rows, C);
  launch_kernel(bn_sums_f32_kernel<0>, blocks, 256, 0, s, x, nullptr, nullptr, nullptr, nullptr, scratch, rows, C);
  ARGUS_CUDA(cudaGetLastError());
  launch_kernel(bn_finalize_f64_kernel, (C + 127) / 128, 128, 0, s, scratch, blocks, static_cast<double>(rows), gamma, beta,
                                                         running_mean, running_var, momentum, eps, scale, shift,
                                                         save_mean, save_invstd, C);
  ARGUS_CUDA(cudaGetLastError());
}

__global__ void bn_apply_f32_kernel(const float* __restrict__ x, const float* __restrict__ scale,
                                    const float* __restrict__ shift, const float* __restrict__ res,
                                    const float* __restrict__ rscale, const float* __restrict__ rshift, int relu,
                                    float* __restrict__ y, int64_t n, int C) {
  pdl_prologue();
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % C);
    float v = fmaf(x[i], scale[c], shift[c]);
    if (res != nullptr) v += (rscale != nullptr) ? fmaf(res[i], rscale[c], rshift[c]) : res[i];
    if (relu) v = fmaxf(v, 0.f);
    y[i] = v;
  }
}
void bn_f32_apply(const float* x, const float* scale, const float* shift, const float* res, const float* rscale,
                  const float* rshift, int relu, float* y, int64_t rows, int C, cudaStream_t s) {
  ProfileScope prof("fp32_bn", s, 0, 8.0 * rows * C);
  const int64_t n = rows * C;
  launch_kernel(bn_apply_f32_kernel, static_cast<int>(std::min<int64_t>((n + 255) / 256, 16384)), 256, 0, s, 
      x, scale, shift, res, rscale, rshift, relu, y, n, C);
  ARGUS_CUDA(cudaGetLastError());
}

__global__ void bn_bwd_apply_f32_kernel(const float* __restrict__ dy, const float* __restrict__ x,
                                        const float* __restrict__ out, const float* __restrict__ scale,
                                        const float* __restrict__ mean, const float* __restrict__ invstd,
                                        const float* __restrict__ sum_g, const float* __restrict__ sum_gx,
                                        float* __restrict__ dx, float* __restrict__ g_out, int64_t n, int C,
                                        float inv_rows) {
  pdl_prologue();
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % C);
    float g = dy[i];
    if (out != nullptr && !(out[i] > 0.f)) g = 0.f;
    const float xh = (x[i] - mean[c]) * invstd[c];
    dx[i] = scale[c] * (g - sum_g[c] * inv_rows - xh * sum_gx[c] * inv_rows);
    if (g_out != nullptr) g_out[i] = g;
  }
}
void bn_f32_backward(const float* dy, const float* x, const float* out, const float* scale, const float* mean,
                     const float* invstd, float* dgamma, float* dbeta, float* dx, float* g_out, int64_t rows, int C,
                     double* scratch, float* sums, cudaStream_t s, bool frozen_stats) {
  ProfileScope prof("fp32_bn", s, 0, 20.0 * rows * C);
  const int blocks = bn_blocks(rows, C);
  launch_kernel(bn_sums_f32_kernel<1>, blocks, 256, 0, s, x, dy, out, mean, invstd, scratch, rows, C);
  ARGUS_CUDA(cudaGetLastError());
  launch_kernel(bn_bwd_finalize_f64_kernel, (C + 127) / 128, 128, 0, s, scratch, blocks, dgamma, dbeta, sums, sums + C, C);
  ARGUS_CUDA(cudaGetLastError());
  const int64_t n = rows * C;
  launch_kernel(bn_bwd_apply_f32_kernel, static_cast<int>(std::min<int64_t>((n + 255) / 256, 16384)), 256, 0, s, 
      dy, x, out, scale, mean, invstd, sums, sums + C, dx, g_out, n, C,
      frozen_stats ? 0.f : static_cast<float>(1.0 / static_cast<double>(rows)));
  ARGUS_CUDA(cudaGetLastError());
}

// ------------------------------------------------------------------------------------------------------------
// pooling, elementwise
// ------------------------------------------------------------------------------------------------------------
__global__ void maxpool_f32_fwd_kernel(const float* __restrict__ x, float* __restrict__ y, uint8_t* __restrict__ idx,
                                       int N, int H, int W, int C) {
  pdl_prologue();
  const int Ho = H / 2, Wo = W / 2;
  const int64_t total = static_cast<int64_t>(N) * Ho * Wo * C;
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % C);
    int64_t t = i / C;
    const int pw = static_cast<int>(t % Wo);
    t /= Wo;
    const int ph = static_cast<int>(t % Ho);
    const int n = static_cast<int>(t / Ho);
    float best = -INFINITY;
    int bi = 0;
    for (int kh = 0; kh < 3; ++kh) {
      const int h = 2 * ph - 1 + kh;
      if (h < 0 || h >= H) continue;
      for (int kw = 0; kw < 3; ++kw) {
        const int w = 2 * pw - 1 + kw;
        if (w < 0 || w >= W) continue;
        const float v = x[(static_cast<int64_t>(n * H + h) * W + w) * C + c];
        if (v > best) { best = v; bi = kh * 3 + kw; }
      }
    }
    y[i] = best;
    if (idx != nullptr) idx[i] = static_cast<uint8_t>(bi);
  }
}
void maxpool_f32_fwd(const float* x, float* y, uint8_t* idx, int N, int H, int W, int C, cudaStream_t s) {
  const int64_t total = static_cast<int64_t>(N) * (H / 2) * (W / 2) * C;
  launch_kernel(maxpool_f32_fwd_kernel, static_cast<int>(std::min<int64_t>((total + 255) / 256, 16384)), 256, 0, s, x, y, idx, N,
                                                                                                         H, W, C);
  ARGUS_CUDA(cudaGetLastError());
}
__global__ void maxpool_f32_bwd_kernel(const float* __restrict__ dy, const uint8_t* __restrict__ idx,
                                       float* __restrict__ dx, int N, int H, int W, int C) {
  pdl_prologue();
  const int Ho = H / 2, Wo = W / 2;
  const int64_t total = static_cast<int64_t>(N) * H * W * C;
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % C);
    int64_t t = i / C;
    const int w = static_cast<int>(t % W);
    t /= W;
    const int h = static_cast<int>(t % H);
    const int n = static_cast<int>(t / H);
    float g = 0.f;
    for (int ph = h >> 1; ph <= ((h + 1) >> 1); ++ph) {
      if (ph >= Ho) continue;
      const int kh = h - (2 * ph - 1);
      for (int pw = w >> 1; pw <= ((w + 1) >> 1); ++pw) {
        if (pw >= Wo) continue;
        const int kw = w - (2 * pw - 1);
        const int64_t j = (static_cast<int64_t>(n * Ho + ph) * Wo + pw) * C + c;
        if (idx[j] == kh * 3 + kw) g += dy[j];
      }
    }
    dx[i] = g;
  }
}
void maxpool_f32_bwd(const float* dy, const uint8_t* idx, float* dx, int N, int H, int W, int C, cudaStream_t s) {
  const int64_t total = static_cast<int64_t>(N) * H * W * C;
  launch_kernel(maxpool_f32_bwd_kernel, static_cast<int>(std::min<int64_t>((total + 255) / 256, 16384)), 256, 0, s, dy, idx, dx,
                                                                                                         N, H, W, C);
  ARGUS_CUDA(cudaGetLastError());
}

__global__ void avgpool_f32_fwd_kernel(const float* __restrict__ x, float* __restrict__ y, int N, int HW, int C) {
  pdl_prologue();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N * C) return;
  const int c = i % C, n = i / C;
  double s = 0.0;
  for (int p = 0; p < HW; ++p) s += static_cast<double>(x[(static_cast<int64_t>(n) * HW + p) * C + c]);
  y[i] = static_cast<float>(s / HW);
}
void avgpool_f32_fwd(const float* x, float* y, int N, int HW, int C, cudaStream_t s) {
  launch_kernel(avgpool_f32_fwd_kernel, (N * C + 127) / 128, 128, 0, s, x, y, N, HW, C);
  ARGUS_CUDA(cudaGetLastError());
}
__global__ void avgpool_f32_bwd_kernel(const float* __restrict__ dy, float* __restrict__ dx, int N, int HW, int C) {
  pdl_prologue();
  const int64_t total = static_cast<int64_t>(N) * HW * C;
  const float inv = 1.0f / HW;
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % C);
    const int n = static_cast<int>(i / (static_cast<int64_t>(HW) * C));
    dx[i] = dy[static_cast<int64_t>(n) * C + c] * inv;
  }
}
void avgpool_f32_bwd(const float* dy, float* dx, int N, int HW, int C, cudaStream_t s) {
  const int64_t total = static_cast<int64_t>(N) * HW * C;
  launch_kernel(avgpool_f32_bwd_kernel, static_cast<int>(std::min<int64_t>((total + 255) / 256, 16384)), 256, 0, s, dy, dx, N, HW, C);
  ARGUS_CUDA(cudaGetLastError());
}

__global__ void add_f32_kernel(float* __restrict__ a, const float* __restrict__ b, int64_t n) {
  pdl_prologue();
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x)
    a[i] += b[i];
}
void add_f32(float* a, const float* b, int64_t n, cudaStream_t s) {
  launch_kernel(add_f32_kernel, static_cast<int>(std::min<int64_t>((n + 255) / 256, 16384)), 256, 0, s, a, b, n);
  ARGUS_CUDA(cudaGetLastError());
}

__global__ void gelu_f32_fwd_kernel(const float* __restrict__ x, float* __restrict__ y, int64_t n) {
  pdl_prologue();
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const float v = x[i];
    y[i] = 0.5f * v * (1.f + erff(v * 0.70710678118654752440f));
  }
}
void gelu_f32_fwd(const float* x, float* y, int64_t n, cudaStream_t s) {
  launch_kernel(gelu_f32_fwd_kernel, static_cast<int>(std::min<int64_t>((n + 255) / 256, 4096)), 256, 0, s, x, y, n);
  ARGUS_CUDA(cudaGetLastError());
}
__global__ void gelu_f32_bwd_kernel(const float* __restrict__ dz, const float* __restrict__ x, float* __restrict__ dx,
                                    int64_t n) {
  pdl_prologue();
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const float v = x[i];
    const float cdf = 0.5f * (1.f + erff(v * 0.70710678118654752440f));
    const float pdf = 0.39894228040143267794f * expf(-0.5f * v * v);
    dx[i] = dz[i] * (cdf + v * pdf);
  }
}
void gelu_f32_bwd(const float* dz, const float* x, float* dx, int64_t n, cudaStream_t s) {
  launch_kernel(gelu_f32_bwd_kernel, static_cast<int>(std::min<int64_t>((n + 255) / 256, 4096)), 256, 0, s, dz, x, dx, n);
  ARGUS_CUDA(cudaGetLastError());
}

// out[c] += sum_r x[r, c] (fc bias gradient), fp64 accumulation
__global__ void colsum_f32_kernel(const float* __restrict__ x, float* out, int rows, int C) {
  pdl_prologue();
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  double acc = 0.0;
  for (int r = 0; r < rows; ++r) acc += static_cast<double>(x[static_cast<int64_t>(r) * C + c]);
  out[c] += static_cast<float>(acc);
}
void colsum_f32(const float* x, float* out, int rows, int C, cudaStream_t s) {
  launch_kernel(colsum_f32_kernel, (C + 127) / 128, 128, 0, s, x, out, rows, C);
  ARGUS_CUDA(cudaGetLastError());
}

}  // namespace argus

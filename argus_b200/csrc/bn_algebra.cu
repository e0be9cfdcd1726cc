// Algebraic batch-norm backward for the expanding 1x1 convolution of a bottleneck (conv3 -> bn3 -> +identity -> ReLU).
//
// The textbook backward makes two full passes over the widest tensors of the block (4C channels): a reduction
// (sum g, sum g*xhat over raw3) and an elementwise pass that writes dRaw3 = sc*g + k1*raw3 + k0, which the weight-
// and input-gradient GEMMs then read again. Because raw3 = act2 * W3^T is LINEAR in the (4x narrower) saved activation,
// all of that collapses onto GEMMs over g and act2 plus a few [4C x C] / [C x C] matrices:
//
// (W3 below is the bf16-rounded weight the forward GEMM actually used, so raw3 = act2 W3^T holds up to the bf16
//  rounding of the stored raw3.)
//   H  = g^T act2                  (the weight-gradient GEMM, run on the masked gradient g itself)       [4C x C]
//   G  = act2^T act2               (Gram matrix, a C x C weight-gradient-shaped GEMM)                    [C x C]
//   s  = colsum(act2),  db = colsum(g)  (db comes from the statistics slots of the dgrad that produced g)
//   sum_p g*raw3  = rowdot(W3, H)                  -> dgamma = invstd * (rowdot - mean * db),  dbeta = db
//   k1 = -sc * dgamma * invstd / P,   k0 = -k1 * mean - sc * db / P              (dRaw3 = sc*g + k1*raw3 + k0)
//   dAct2 = g (diag(sc) W3) + act2 (W3^T diag(k1) W3) + k0^T W3     -> ONE dgrad GEMM over the concatenated K = 4C + C
//   dW3   = diag(sc) H + diag(k1) W3 G + k0 (x) s
//
// so neither raw3 nor dRaw3 is touched in the backward pass. All small-matrix work is fp32 and deterministic.
// Reference semantics: autograd of torch.nn.BatchNorm2d + Conv2d(1x1) inside torchvision's Bottleneck
// (/root/reference/argus/models.py:84).
#include "kernels.h"
#include "ptx.cuh"
#include "runtime.h"

#include <algorithm>

namespace argus {

// one warp per output channel o
__global__ void __launch_bounds__(256)
bn_alg_coeffs_kernel(const bf16* __restrict__ W, const float* __restrict__ H, const float* __restrict__ stat_partial,
                     int slots, int stat_stride, const float* __restrict__ scale, const float* __restrict__ mean,
                     const float* __restrict__ invstd, float inv_rows, float* dgamma, float* dbeta,
                     float* __restrict__ k1k0, bf16* __restrict__ bstack, int O, int C) {
  pdl_prologue();
  const int o = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (o >= O) return;
  // db = sum over the statistic slots, lanes take slots round-robin, then a fixed shuffle tree: deterministic
  double db = 0.0;
  for (int k = lane; k < slots; k += 32) db += static_cast<double>(stat_partial[static_cast<size_t>(k) * stat_stride + o]);
  double t = 0.0;
  const bf16* w = W + static_cast<size_t>(o) * C;
  const float* h = H + static_cast<size_t>(o) * C;
  for (int i = lane; i < C; i += 32) t += static_cast<double>(__bfloat162float(w[i])) * static_cast<double>(h[i]);
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    db += __shfl_xor_sync(0xffffffffu, db, off);
    t += __shfl_xor_sync(0xffffffffu, t, off);
  }
  const float sc = scale[o], mu = mean[o], is = invstd[o];
  const double dg = static_cast<double>(is) * (t - static_cast<double>(mu) * db);
  const double c2 = static_cast<double>(sc) * dg * static_cast<double>(is) * inv_rows;
  const float k1 = static_cast<float>(-c2);
  const float k0 = static_cast<float>(c2 * mu - static_cast<double>(sc) * db * inv_rows);
  if (lane == 0) {
    dgamma[o] += static_cast<float>(dg);
    dbeta[o] += static_cast<float>(db);
    k1k0[o] = k1;
    k1k0[O + o] = k0;
  }
  bf16* b = bstack + static_cast<size_t>(o) * C;
  for (int i = lane; i < C; i += 32) b[i] = __float2bfloat16(sc * __bfloat162float(w[i]));
}

// M[j][i] = sum_o W[o][j] k1[o] W[o][i] -> bstack rows O + j (bf16);  blockIdx.y == C/16: bias[i] = sum_o k0[o] W[o][i]
// The reduction over o is split over blockIdx.z (kSplitO chunks, fixed boundaries): each split writes its partial
// 16x16 tile to `partial` and a second tiny kernel adds the splits in order (deterministic).
constexpr int kSplitO = 8;
__global__ void __launch_bounds__(256)
bn_alg_matrix_kernel(const bf16* __restrict__ W, const float* __restrict__ k1k0, float* __restrict__ partial, int O,
                     int C) {
  pdl_prologue();
  __shared__ float sWj[32][17];   // [o chunk][j]
  __shared__ float sWi[32][17];   // [o chunk][i]
  const int ti = threadIdx.x & 15, tj = threadIdx.x >> 4;
  const int i0 = blockIdx.x * 16;
  const bool bias_row = (blockIdx.y == C / 16);
  const int j0 = bias_row ? 0 : blockIdx.y * 16;
  const int per = O / kSplitO;
  const int o_begin = blockIdx.z * per, o_end = o_begin + per;
  float acc = 0.f;
  // register prefetch of the next 32-row chunk while the current one is being multiplied
  float ni[2], nj[2];
  auto fetch = [&](int o0) {
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const int e = threadIdx.x + 256 * u;
      const int oo = e >> 4, c = e & 15;
      ni[u] = __bfloat162float(W[static_cast<size_t>(o0 + oo) * C + i0 + c]);
      nj[u] = bias_row ? k1k0[O + o0 + oo]
                       : __bfloat162float(W[static_cast<size_t>(o0 + oo) * C + j0 + c]) * k1k0[o0 + oo];
    }
  };
  fetch(o_begin);
  for (int o0 = o_begin; o0 < o_end; o0 += 32) {
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const int e = threadIdx.x + 256 * u;
      sWi[e >> 4][e & 15] = ni[u];
      sWj[e >> 4][e & 15] = nj[u];
    }
    __syncthreads();
    if (o0 + 32 < o_end) fetch(o0 + 32);
    if (!bias_row) {
#pragma unroll 8
      for (int oo = 0; oo < 32; ++oo) acc = fmaf(sWj[oo][tj], sWi[oo][ti], acc);
    } else if (tj == 0) {
#pragma unroll 8
      for (int oo = 0; oo < 32; ++oo) acc = fmaf(sWj[oo][0], sWi[oo][ti], acc);
    }
    __syncthreads();
  }
  // partial[z][row][i], row = j (0..C-1) or C for the bias row
  const int row = bias_row ? C : j0 + tj;
  if (!bias_row || tj == 0) partial[(static_cast<size_t>(blockIdx.z) * (C + 1) + row) * C + i0 + ti] = acc;
}
__global__ void bn_alg_matrix_reduce_kernel(const float* __restrict__ partial, bf16* __restrict__ bstack,
                                            float* __restrict__ bias, int O, int C) {
  pdl_prologue();
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (C + 1) * C) return;
  float acc = 0.f;
  for (int z = 0; z < kSplitO; ++z) acc += partial[static_cast<size_t>(z) * (C + 1) * C + idx];
  const int row = idx / C, i = idx - row * C;
  if (row < C) bstack[static_cast<size_t>(O + row) * C + i] = __float2bfloat16(acc);
  else bias[i] = acc;
}

// dW[o][i] += sc[o] H[o][i] + k0[o] s[i] + k1[o] sum_j W[o][j] G[j][i]
__global__ void __launch_bounds__(256)
bn_alg_dw_kernel(const bf16* __restrict__ W, const float* __restrict__ H, const float* __restrict__ G,
                 const float* __restrict__ s, const float* __restrict__ scale, const float* __restrict__ k1k0,
                 float* __restrict__ dW, int O, int C) {
  pdl_prologue();
  __shared__ float sW[16][33];   // [o][j chunk]
  __shared__ float sG[32][17];   // [j chunk][i]
  const int ti = threadIdx.x & 15, to = threadIdx.x >> 4;
  const int i0 = blockIdx.x * 16, o0 = blockIdx.y * 16;
  float acc = 0.f;
  for (int j0 = 0; j0 < C; j0 += 32) {
    for (int e = threadIdx.x; e < 16 * 32; e += 256) {
      const int a = e >> 5, b = e & 31;      // W tile [16 o][32 j]
      sW[a][b] = __bfloat162float(W[static_cast<size_t>(o0 + a) * C + j0 + b]);
      const int c = e >> 4, d = e & 15;      // G tile [32 j][16 i]
      sG[c][d] = G[static_cast<size_t>(j0 + c) * C + i0 + d];
    }
    __syncthreads();
#pragma unroll 8
    for (int j = 0; j < 32; ++j) acc = fmaf(sW[to][j], sG[j][ti], acc);
    __syncthreads();
  }
  const int o = o0 + to, i = i0 + ti;
  const size_t idx = static_cast<size_t>(o) * C + i;
  dW[idx] += scale[o] * H[idx] + k1k0[O + o] * s[i] + k1k0[o] * acc;
}

void bn_alg_backward_small(const bf16* W, const float* H, const float* G, const float* s, const float* stat_partial,
                           int slots, int stat_stride, const float* scale, const float* mean, const float* invstd,
                           double rows, float* dgamma, float* dbeta, float* dW, float* k1k0, bf16* bstack, float* bias,
                           float* mpartial, int O, int C, cudaStream_t st) {
  ARGUS_CHECK(O % (32 * kSplitO) == 0 && C % 32 == 0, "algebraic BN backward: O % 256 == 0 and C % 32 == 0 required");
  ProfileScope prof("bn_algebra", st, 4.0 * O * static_cast<double>(C) * C, 0);
  launch_kernel(bn_alg_coeffs_kernel, (O * 32 + 255) / 256, 256, 0, st, W, H, stat_partial, slots, stat_stride, scale, mean, invstd,
                                                            static_cast<float>(1.0 / rows), dgamma, dbeta, k1k0, bstack,
                                                            O, C);
  ARGUS_CUDA(cudaGetLastError());
  launch_kernel(bn_alg_matrix_kernel, dim3(C / 16, C / 16 + 1, kSplitO), 256, 0, st, W, k1k0, mpartial, O, C);
  ARGUS_CUDA(cudaGetLastError());
  launch_kernel(bn_alg_matrix_reduce_kernel, ((C + 1) * C + 255) / 256, 256, 0, st, mpartial, bstack, bias, O, C);
  ARGUS_CUDA(cudaGetLastError());
  if (dW != nullptr) {
    launch_kernel(bn_alg_dw_kernel, dim3(C / 16, O / 16), 256, 0, st, W, H, G, s, scale, k1k0, dW, O, C);
    ARGUS_CUDA(cudaGetLastError());
  }
}

// The weight-gradient part alone (dW == nullptr above): nothing downstream of the backward chain reads dW3, so the
// model runs it on the weight-gradient side stream, overlapping the K-concatenated dgrad.
void bn_alg_backward_dw(const bf16* W, const float* H, const float* G, const float* s, const float* scale,
                        const float* k1k0, float* dW, int O, int C, cudaStream_t st) {
  ProfileScope prof("bn_algebra", st, 2.0 * O * static_cast<double>(C) * C, 0);
  launch_kernel(bn_alg_dw_kernel, dim3(C / 16, O / 16), 256, 0, st, W, H, G, s, scale, k1k0, dW, O, C);
  ARGUS_CUDA(cudaGetLastError());
}

// ------------------------------------------------------------------------------------------------------------
// Forward: batch statistics of y = x W^T (1x1 convolution) from the Gram matrix of its input, BEFORE the convolution
// runs:  mean_o = W[o,:] s / P,  E[y_o^2] = W[o,:] G W[o,:]^T / P  with s = colsum(x), G = x^T x. The convolution can
// then apply batch norm (+ residual + ReLU) in its own epilogue and its raw output is never written.
// ------------------------------------------------------------------------------------------------------------
// partial[o][bx] = sum over the 16 columns i of tile bx of W[o,i] * (sum_j W[o,j] G[j,i])
__global__ void __launch_bounds__(256)
gram_quadform_kernel(const bf16* __restrict__ W, const float* __restrict__ G, float* __restrict__ partial, int O, int C) {
  pdl_prologue();
  __shared__ float sW[16][33];
  __shared__ float sG[32][17];
  __shared__ float sQ[16][17];
  const int ti = threadIdx.x & 15, to = threadIdx.x >> 4;
  const int i0 = blockIdx.x * 16, o0 = blockIdx.y * 16;
  float acc = 0.f;
  for (int j0 = 0; j0 < C; j0 += 32) {
    for (int e = threadIdx.x; e < 16 * 32; e += 256) {
      const int a = e >> 5, b = e & 31;
      sW[a][b] = __bfloat162float(W[static_cast<size_t>(o0 + a) * C + j0 + b]);
      const int c = e >> 4, d = e & 15;
      sG[c][d] = G[static_cast<size_t>(j0 + c) * C + i0 + d];
    }
    __syncthreads();
#pragma unroll 8
    for (int j = 0; j < 32; ++j) acc = fmaf(sW[to][j], sG[j][ti], acc);
    __syncthreads();
  }
  sQ[to][ti] = acc * __bfloat162float(W[static_cast<size_t>(o0 + to) * C + i0 + ti]);
  __syncthreads();
  if (ti == 0) {
    float q = 0.f;
#pragma unroll
    for (int k = 0; k < 16; ++k) q += sQ[to][k];
    partial[static_cast<size_t>(o0 + to) * gridDim.x + blockIdx.x] = q;
  }
}
// one warp per channel: finish the quadratic form and the mean, then torch.nn.BatchNorm2d's train-mode bookkeeping
__global__ void __launch_bounds__(256)
gram_stats_finalize_kernel(const bf16* __restrict__ W, const float* __restrict__ s, const float* __restrict__ partial,
                           int nparts, double rows, const float* gamma, const float* beta, float* running_mean,
                           float* running_var, float momentum, float eps, float* scale, float* shift, float* save_mean,
                           float* save_invstd, int O, int C) {
  pdl_prologue();
  const int o = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (o >= O) return;
  double q = 0.0, m = 0.0;
  for (int k = lane; k < nparts; k += 32) q += static_cast<double>(partial[static_cast<size_t>(o) * nparts + k]);
  for (int i = lane; i < C; i += 32)
    m += static_cast<double>(__bfloat162float(W[static_cast<size_t>(o) * C + i])) * static_cast<double>(s[i]);
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    q += __shfl_xor_sync(0xffffffffu, q, off);
    m += __shfl_xor_sync(0xffffffffu, m, off);
  }
  if (lane != 0) return;
  const double mean = m / rows;
  double var = q / rows - mean * mean;
  if (var < 0) var = 0;
  const float invstd = static_cast<float>(1.0 / sqrt(var + static_cast<double>(eps)));
  const float sc = gamma[o] * invstd;
  scale[o] = sc;
  shift[o] = beta[o] - static_cast<float>(mean) * sc;
  save_mean[o] = static_cast<float>(mean);
  save_invstd[o] = invstd;
  if (running_mean != nullptr) {
    const double unbiased = rows > 1 ? var * rows / (rows - 1) : var;
    running_mean[o] = (1.f - momentum) * running_mean[o] + momentum * static_cast<float>(mean);
    running_var[o] = (1.f - momentum) * running_var[o] + momentum * static_cast<float>(unbiased);
  }
}
void bn_stats_from_gram(const bf16* W, const float* G, const float* s, double rows, const float* gamma,
                        const float* beta, float* running_mean, float* running_var, float momentum, float eps,
                        float* scale, float* shift, float* save_mean, float* save_invstd, float* scratch, int O, int C,
                        cudaStream_t st) {
  ARGUS_CHECK(O % 16 == 0 && C % 32 == 0, "bn_stats_from_gram: O % 16 == 0 and C % 32 == 0 required");
  ProfileScope prof("bn_algebra", st, 2.0 * O * static_cast<double>(C) * C, 0);
  launch_kernel(gram_quadform_kernel, dim3(C / 16, O / 16), 256, 0, st, W, G, scratch, O, C);
  ARGUS_CUDA(cudaGetLastError());
  launch_kernel(gram_stats_finalize_kernel, (O * 32 + 255) / 256, 256, 0, st, W, s, scratch, C / 16, rows, gamma, beta, running_mean,
                                                                  running_var, momentum, eps, scale, shift, save_mean,
                                                                  save_invstd, O, C);
  ARGUS_CUDA(cudaGetLastError());
}

// ------------------------------------------------------------------------------------------------------------
// deterministic column sums of a bf16 (rows, C) matrix: per-block partials, then an ordered reduction
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
colsum_partial_kernel(const uint4* __restrict__ x, float* __restrict__ partial, int64_t rows, int cvec, int stride,
                      int Wo, int HoWo, int W, int HW) {
  pdl_prologue();
  // stride 2: row r of the (N, H/2, W/2) grid is pixel (2h, 2w) of the (N, H, W) tensor
  auto src = [&](int64_t r) -> int64_t {
    if (stride == 1) return r;
    const int64_t n = r / HoWo;
    const int rem = static_cast<int>(r - n * HoWo);
    const int h2 = rem / Wo, w2 = rem - h2 * Wo;
    return n * HW + static_cast<int64_t>(stride * h2) * W + stride * w2;
  };
  __shared__ float red[8][256];
  const int lanes = cvec < 256 ? cvec : 256;
  const int row_lanes = 256 / lanes;
  const int rl = threadIdx.x / lanes, oc = threadIdx.x % lanes;
  float acc[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) acc[k] = 0.f;
  auto add = [&](const uint4& u) {
    float2 a = unpack_bf16x2(u.x), b = unpack_bf16x2(u.y), c = unpack_bf16x2(u.z), d = unpack_bf16x2(u.w);
    acc[0] += a.x; acc[1] += a.y; acc[2] += b.x; acc[3] += b.y; acc[4] += c.x; acc[5] += c.y; acc[6] += d.x; acc[7] += d.y;
  };
  const int64_t rs = static_cast<int64_t>(gridDim.x) * row_lanes;
  int64_t r = static_cast<int64_t>(blockIdx.x) * row_lanes + rl;
  for (; r + 3 * rs < rows; r += 4 * rs) {   // four independent 16-byte loads in flight per thread
    const uint4 u0 = __ldg(x + src(r) * cvec + oc), u1 = __ldg(x + src(r + rs) * cvec + oc);
    const uint4 u2 = __ldg(x + src(r + 2 * rs) * cvec + oc), u3 = __ldg(x + src(r + 3 * rs) * cvec + oc);
    add(u0); add(u1); add(u2); add(u3);
  }
  for (; r < rows; r += rs) add(__ldg(x + src(r) * cvec + oc));
#pragma unroll
  for (int k = 0; k < 8; ++k) red[k][threadIdx.x] = acc[k];
  __syncthreads();
  if (rl == 0) {
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      float s0 = 0.f;
      for (int r = 0; r < row_lanes; ++r) s0 += red[k][r * lanes + oc];
      partial[static_cast<size_t>(blockIdx.x) * (cvec * 8) + oc * 8 + k] = s0;
    }
  }
}
void colsum_rows_bf16(const bf16* x, int64_t rows, int C, float* scratch, float* out, cudaStream_t st) {
  colsum_pixels_bf16(x, static_cast<int>(rows), 1, 1, C, 1, scratch, out, st);
}
void colsum_pixels_bf16(const bf16* x, int N, int H, int W, int C, int stride, float* scratch, float* out,
                        cudaStream_t st) {
  const int64_t rows = static_cast<int64_t>(N) * (H / stride) * (W / stride);
  ARGUS_CHECK(C % 8 == 0 && is_pow2(C / 8) && C <= 2048, "colsum: C/8 must be a power of two <= 256");
  ProfileScope prof("bn_algebra", st, 0, static_cast<double>(rows) * C * 2);
  const int cvec = C / 8;
  const int lanes = std::min(cvec, 256);
  const int row_lanes = 256 / lanes;
  const int blocks = static_cast<int>(std::max<int64_t>(1, std::min<int64_t>((rows + row_lanes - 1) / row_lanes, 4LL * num_sms())));
  launch_kernel(colsum_partial_kernel, blocks, 256, 0, st, reinterpret_cast<const uint4*>(x), scratch, rows, cvec, stride, W / stride,
                                                (H / stride) * (W / stride), W, H * W);
  ARGUS_CUDA(cudaGetLastError());
  colsum_finalize(scratch, blocks, out, C, st);
}

int64_t bn_alg_matrix_scratch_elems(int C) { return static_cast<int64_t>(kSplitO) * (C + 1) * C; }

// ------------------------------------------------------------------------------------------------------------
// Frozen-statistics backward (eval-mode forward made differentiable): the k1 = k0 = 0 case of the algebra above, for
// every convolution. Nothing is subtracted from g, so dRaw = sc * g never needs to exist: dW = diag(sc) H with
// H = g^T im2col(x), and the input gradient is the dgrad of g against diag(sc) W (pack_weights_scaled).
// ------------------------------------------------------------------------------------------------------------
// one warp per output channel o (H and dW deliberately not __restrict__: the 3x3 / stem finish scales H in place)
__global__ void __launch_bounds__(256)
bn_frozen_finish_kernel(const bf16* __restrict__ W, const float* H, const float* __restrict__ stat_partial, int slots,
                        int stat_stride, const float* __restrict__ scale, const float* __restrict__ mean,
                        const float* __restrict__ invstd, float* dgamma, float* dbeta, float* dW, int accumulate, int O,
                        int K) {
  pdl_prologue();
  const int o = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (o >= O) return;
  double db = 0.0, t = 0.0;
  for (int k = lane; k < slots; k += 32) db += static_cast<double>(stat_partial[static_cast<size_t>(k) * stat_stride + o]);
  const bf16* w = W + static_cast<size_t>(o) * K;
  const float* h = H + static_cast<size_t>(o) * K;
  for (int i = lane; i < K; i += 32) t += static_cast<double>(__bfloat162float(w[i])) * static_cast<double>(h[i]);
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {   // (also orders every lane's reads of H before the in-place writes below)
    db += __shfl_xor_sync(0xffffffffu, db, off);
    t += __shfl_xor_sync(0xffffffffu, t, off);
  }
  const float sc = scale[o];
  if (lane == 0) {
    dgamma[o] += static_cast<float>(static_cast<double>(invstd[o]) * (t - static_cast<double>(mean[o]) * db));
    dbeta[o] += static_cast<float>(db);
  }
  float* d = dW + static_cast<size_t>(o) * K;
  for (int i = lane; i < K; i += 32) d[i] = (accumulate ? d[i] : 0.f) + sc * h[i];
}
void bn_frozen_finish(const bf16* W, const float* H, const float* stat_partial, int slots, int stat_stride,
                      const float* scale, const float* mean, const float* invstd, float* dgamma, float* dbeta, float* dW,
                      bool accumulate, int O, int K, cudaStream_t st) {
  ProfileScope prof("bn_frozen", st, 2.0 * O * static_cast<double>(K), 10.0 * O * static_cast<double>(K));
  launch_kernel(bn_frozen_finish_kernel, (O * 32 + 255) / 256, 256, 0, st, W, H, stat_partial, slots, stat_stride, scale,
                mean, invstd, dgamma, dbeta, dW, accumulate ? 1 : 0, O, K);
  ARGUS_CUDA(cudaGetLastError());
}

// Block column sums shared by the two passes below: thread (rl, oc) holds the sums of channels 8 oc .. 8 oc + 7 over its
// rows; the row lanes are added in order into partial[blockIdx.x][C].
__device__ __forceinline__ void block_colsum_store(const float (&acc)[8], float (&red)[8][256], float* partial, int lanes,
                                                   int row_lanes, int rl, int oc, int cvec) {
#pragma unroll
  for (int k = 0; k < 8; ++k) red[k][threadIdx.x] = acc[k];
  __syncthreads();
  if (rl == 0) {
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      float s0 = 0.f;
      for (int r = 0; r < row_lanes; ++r) s0 += red[k][r * lanes + oc];
      partial[static_cast<size_t>(blockIdx.x) * (cvec * 8) + oc * 8 + k] = s0;
    }
  }
}

__global__ void __launch_bounds__(256)
relu_bits_mask_colsum_kernel(uint4* __restrict__ g, const uint8_t* __restrict__ bits, float* __restrict__ partial,
                             int64_t rows, int cvec) {
  pdl_prologue();
  __shared__ float red[8][256];
  const int lanes = cvec < 256 ? cvec : 256;
  const int row_lanes = 256 / lanes;
  const int rl = threadIdx.x / lanes, oc = threadIdx.x % lanes;
  float acc[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) acc[k] = 0.f;
  for (int64_t r = static_cast<int64_t>(blockIdx.x) * row_lanes + rl; r < rows; r += static_cast<int64_t>(gridDim.x) * row_lanes) {
    const int64_t i = r * cvec + oc;
    const uint4 u = g[i];
    const unsigned b = bits[i];
    uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint32_t keep = ((b >> (2 * j)) & 1u ? 0x0000ffffu : 0u) | ((b >> (2 * j + 1)) & 1u ? 0xffff0000u : 0u);
      w[j] &= keep;
      const float2 f = unpack_bf16x2(w[j]);
      acc[2 * j] += f.x;
      acc[2 * j + 1] += f.y;
    }
    g[i] = make_uint4(w[0], w[1], w[2], w[3]);
  }
  block_colsum_store(acc, red, partial, lanes, row_lanes, rl, oc, cvec);
}
void relu_bits_mask_colsum(bf16* g, const uint8_t* bits, int64_t rows, int C, float* scratch, float* out,
                           cudaStream_t st) {
  ARGUS_CHECK(C % 8 == 0 && is_pow2(C / 8) && C <= 2048, "relu_bits_mask_colsum: C/8 must be a power of two <= 256");
  ProfileScope prof("bn_frozen", st, 0, static_cast<double>(rows) * C * (4 + 0.125));
  const int cvec = C / 8;
  const int row_lanes = 256 / std::min(cvec, 256);
  const int blocks = static_cast<int>(std::max<int64_t>(1, std::min<int64_t>((rows + row_lanes - 1) / row_lanes, 4LL * num_sms())));
  launch_kernel(relu_bits_mask_colsum_kernel, blocks, 256, 0, st, reinterpret_cast<uint4*>(g), bits, scratch, rows, cvec);
  ARGUS_CUDA(cudaGetLastError());
  colsum_finalize(scratch, blocks, out, C, st);
}

// thread = one stem pixel x 8 channels; the 3x3 stride-2 pad-1 windows holding pixel (h, w) are ph in {h/2, (h+1)/2},
// pw likewise (maxpool_bwd's order), tap code (h - 2 ph + 1) * 3 + (w - 2 pw + 1)
__global__ void __launch_bounds__(256)
stem_unpool_relu_kernel(const uint4* __restrict__ dpool, const uint2* __restrict__ idx, const uint4* __restrict__ pooled,
                        uint4* __restrict__ g0, float* __restrict__ partial, int N, int H, int W) {
  pdl_prologue();
  constexpr int cvec = 8;   // C = 64
  __shared__ float red[8][256];
  const int rl = threadIdx.x / cvec, oc = threadIdx.x % cvec;
  const int Ho = H >> 1, Wo = W >> 1;
  const int64_t pixels = static_cast<int64_t>(N) * H * W;
  float acc[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) acc[k] = 0.f;
  for (int64_t r = static_cast<int64_t>(blockIdx.x) * 32 + rl; r < pixels; r += static_cast<int64_t>(gridDim.x) * 32) {
    const int w = static_cast<int>(r % W);
    const int64_t t = r / W;
    const int h = static_cast<int>(t % H);
    const int n = static_cast<int>(t / H);
    float v[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) v[k] = 0.f;
    for (int ph = h >> 1; ph <= ((h + 1) >> 1) && ph < Ho; ++ph) {
      for (int pw = w >> 1; pw <= ((w + 1) >> 1) && pw < Wo; ++pw) {
        const uint32_t code = static_cast<uint32_t>((h - 2 * ph + 1) * 3 + (w - 2 * pw + 1));
        const int64_t j = ((static_cast<int64_t>(n) * Ho + ph) * Wo + pw) * cvec + oc;
        const uint2 id = __ldg(idx + j);
        const uint4 d = __ldg(dpool + j), pv = __ldg(pooled + j);
        const uint32_t dw[4] = {d.x, d.y, d.z, d.w}, pw4[4] = {pv.x, pv.y, pv.z, pv.w};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float2 df = unpack_bf16x2(dw[q]), pf = unpack_bf16x2(pw4[q]);
          const uint32_t word = q < 2 ? id.x : id.y;
          const uint32_t b0 = (word >> (16 * (q & 1))) & 0xffu, b1 = (word >> (16 * (q & 1) + 8)) & 0xffu;
          if (b0 == code && pf.x > 0.f) v[2 * q] += df.x;
          if (b1 == code && pf.y > 0.f) v[2 * q + 1] += df.y;
        }
      }
    }
    uint4 o;
    o.x = pack_bf16x2(v[0], v[1]); o.y = pack_bf16x2(v[2], v[3]);
    o.z = pack_bf16x2(v[4], v[5]); o.w = pack_bf16x2(v[6], v[7]);
    g0[r * cvec + oc] = o;
    const uint32_t ow[4] = {o.x, o.y, o.z, o.w};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float2 f = unpack_bf16x2(ow[q]);
      acc[2 * q] += f.x;
      acc[2 * q + 1] += f.y;
    }
  }
  block_colsum_store(acc, red, partial, cvec, 32, rl, oc, cvec);
}
void stem_unpool_relu(const bf16* dpool, const uint8_t* idx, const bf16* pooled, bf16* g0, int N, int H, int W,
                      float* scratch, float* out, cudaStream_t st) {
  ARGUS_CHECK(H % 2 == 0 && W % 2 == 0, "stem_unpool_relu: H and W must be even");
  const int64_t pixels = static_cast<int64_t>(N) * H * W;
  // HBM model: the pooled gradient, pooled values and arg-max bytes once (a quarter of the pixels), g0 written once
  ProfileScope prof("bn_frozen", st, 0, pixels * 64 * (2.0 + 0.25 * (2 + 2 + 1)));
  const int blocks = static_cast<int>(std::max<int64_t>(1, std::min<int64_t>((pixels + 31) / 32, 4LL * num_sms())));
  launch_kernel(stem_unpool_relu_kernel, blocks, 256, 0, st, reinterpret_cast<const uint4*>(dpool),
                reinterpret_cast<const uint2*>(idx), reinterpret_cast<const uint4*>(pooled), reinterpret_cast<uint4*>(g0),
                scratch, N, H, W);
  ARGUS_CUDA(cudaGetLastError());
  colsum_finalize(scratch, blocks, out, 64, st);
}

}  // namespace argus

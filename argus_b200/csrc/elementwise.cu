// Memory-bound kernels of the hot path: input/weight packing, batch-norm (finalize / apply / backward), pooling.
// Every kernel moves 16 bytes per thread per access (8 bf16 channels of one pixel), is coalesced along the
// channel-contiguous NHWC layout, and reduces with warp shuffles / shared memory before touching global atomics.
// Reference semantics: torch.nn.BatchNorm2d, ReLU, MaxPool2d(3,2,1), AdaptiveAvgPool2d(1) inside torchvision
// resnet50 as called from /root/reference/argus/models.py:84.
#include "kernels.h"
#include "ptx.cuh"
#include "runtime.h"

#include <algorithm>
#include <string>

namespace argus {

static inline int grid_for(int64_t work_items, int threads, int max_blocks_per_sm = 8) {
  int64_t blocks = (work_items + threads - 1) / threads;
  int64_t cap = static_cast<int64_t>(num_sms()) * max_blocks_per_sm;
  return static_cast<int>(std::max<int64_t>(1, std::min(blocks, cap)));
}

struct F8 {
  float v[8];
};
__device__ __forceinline__ F8 unpack8(const uint4& u) {
  F8 r;
  float2 a = unpack_bf16x2(u.x), b = unpack_bf16x2(u.y), c = unpack_bf16x2(u.z), d = unpack_bf16x2(u.w);
  r.v[0] = a.x; r.v[1] = a.y; r.v[2] = b.x; r.v[3] = b.y; r.v[4] = c.x; r.v[5] = c.y; r.v[6] = d.x; r.v[7] = d.y;
  return r;
}
__device__ __forceinline__ uint4 pack8(const F8& f) {
  uint4 u;
  u.x = pack_bf16x2(f.v[0], f.v[1]);
  u.y = pack_bf16x2(f.v[2], f.v[3]);
  u.z = pack_bf16x2(f.v[4], f.v[5]);
  u.w = pack_bf16x2(f.v[6], f.v[7]);
  return u;
}
// bit k = (v[k] > 0): the ReLU mask of eight channels in one byte (1/16 of the bf16 activation bytes)
__device__ __forceinline__ uint8_t positive_bits(const F8& f) {
  uint32_t b = 0;
#pragma unroll
  for (int k = 0; k < 8; ++k) b |= (f.v[k] > 0.f ? 1u : 0u) << k;
  return static_cast<uint8_t>(b);
}
__device__ __forceinline__ F8 load8f(const float* p) {
  F8 r;
  const float4 a = __ldg(reinterpret_cast<const float4*>(p));
  const float4 b = __ldg(reinterpret_cast<const float4*>(p) + 1);
  r.v[0] = a.x; r.v[1] = a.y; r.v[2] = a.z; r.v[3] = a.w; r.v[4] = b.x; r.v[5] = b.y; r.v[6] = b.z; r.v[7] = b.w;
  return r;
}
__device__ __forceinline__ uint4 ldg_stream(const uint4* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}

// ------------------------------------------------------------------------------------------------------------
// input packing: NCHW fp32 (or HWC u8) -> space-to-depth bf16 [n][H/2][W/2+4][16]
// ------------------------------------------------------------------------------------------------------------
__global__ void pack_input_f32_kernel(const float* __restrict__ x, uint4* __restrict__ out, int n_images, int H,
                                      int W) {
  pdl_prologue();
  const int Hs = H >> 1, Ws = W >> 1, Wp = Ws + 4;
  const int64_t total = static_cast<int64_t>(n_images) * Hs * Wp;
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int jp = static_cast<int>(i % Wp);
    const int64_t t = i / Wp;
    const int is = static_cast<int>(t % Hs);
    const int n = static_cast<int>(t / Hs);
    float v[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) v[k] = 0.f;
    const int j = jp - 2;
    if (j >= 0 && j < Ws) {
      const float* img = x + static_cast<int64_t>(n) * 3 * H * W;  // image n = channels [3n, 3n+3) of sample n / n_cams
#pragma unroll
      for (int c = 0; c < 3; ++c)
#pragma unroll
        for (int a = 0; a < 2; ++a) {
          const float2 p = __ldg(reinterpret_cast<const float2*>(img + (static_cast<int64_t>(c) * H + 2 * is + a) * W + 2 * j));
          v[(a * 2 + 0) * 3 + c] = p.x;
          v[(a * 2 + 1) * 3 + c] = p.y;
        }
    }
    uint4 o0, o1;
    o0.x = pack_bf16x2(v[0], v[1]); o0.y = pack_bf16x2(v[2], v[3]); o0.z = pack_bf16x2(v[4], v[5]); o0.w = pack_bf16x2(v[6], v[7]);
    o1.x = pack_bf16x2(v[8], v[9]); o1.y = pack_bf16x2(v[10], v[11]); o1.z = pack_bf16x2(v[12], v[13]); o1.w = pack_bf16x2(v[14], v[15]);
    out[2 * i] = o0;
    out[2 * i + 1] = o1;
  }
}

__global__ void pack_input_u8_kernel(const uint8_t* __restrict__ x, uint4* __restrict__ out, int n_images, int H,
                                     int W) {
  pdl_prologue();
  const int Hs = H >> 1, Ws = W >> 1, Wp = Ws + 4;
  const int64_t total = static_cast<int64_t>(n_images) * Hs * Wp;
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int jp = static_cast<int>(i % Wp);
    const int64_t t = i / Wp;
    const int is = static_cast<int>(t % Hs);
    const int n = static_cast<int>(t / Hs);
    float v[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) v[k] = 0.f;
    const int j = jp - 2;
    if (j >= 0 && j < Ws) {
      const uint8_t* img = x + static_cast<int64_t>(n) * H * W * 3;
#pragma unroll
      for (int a = 0; a < 2; ++a) {
        const uint8_t* px = img + (static_cast<int64_t>(2 * is + a) * W + 2 * j) * 3;  // 6 contiguous bytes, 2-byte aligned
        const uint16_t* p16 = reinterpret_cast<const uint16_t*>(px);
        const uint32_t w0 = p16[0], w1 = p16[1], w2 = p16[2];
        const float r0 = (w0 & 0xff), g0 = (w0 >> 8), b0 = (w1 & 0xff), r1 = (w1 >> 8), g1 = (w2 & 0xff), b1 = (w2 >> 8);
        const float k = 1.0f / 255.0f;
        v[(a * 2 + 0) * 3 + 0] = r0 * k; v[(a * 2 + 0) * 3 + 1] = g0 * k; v[(a * 2 + 0) * 3 + 2] = b0 * k;
        v[(a * 2 + 1) * 3 + 0] = r1 * k; v[(a * 2 + 1) * 3 + 1] = g1 * k; v[(a * 2 + 1) * 3 + 2] = b1 * k;
      }
    }
    uint4 o0, o1;
    o0.x = pack_bf16x2(v[0], v[1]); o0.y = pack_bf16x2(v[2], v[3]); o0.z = pack_bf16x2(v[4], v[5]); o0.w = pack_bf16x2(v[6], v[7]);
    o1.x = pack_bf16x2(v[8], v[9]); o1.y = pack_bf16x2(v[10], v[11]); o1.z = pack_bf16x2(v[12], v[13]); o1.w = pack_bf16x2(v[14], v[15]);
    out[2 * i] = o0;
    out[2 * i + 1] = o1;
  }
}

void pack_input_f32(const float* x, bf16* out, int n_images, int H, int W, cudaStream_t s) {
  ProfileScope prof("pack_input", s, 0, static_cast<double>(n_images) * H * W * 3 * 4 + static_cast<double>(n_images) * (H / 2) * (W / 2 + 4) * 32);
  const int64_t total = static_cast<int64_t>(n_images) * (H / 2) * (W / 2 + 4);
  launch_kernel(pack_input_f32_kernel, grid_for(total, 256), 256, 0, s, x, reinterpret_cast<uint4*>(out), n_images, H, W);
  ARGUS_CUDA(cudaGetLastError());
}
void pack_input_u8(const uint8_t* x, bf16* out, int n_images, int H, int W, cudaStream_t s) {
  ProfileScope prof("pack_input", s, 0, static_cast<double>(n_images) * H * W * 3 + static_cast<double>(n_images) * (H / 2) * (W / 2 + 4) * 32);
  const int64_t total = static_cast<int64_t>(n_images) * (H / 2) * (W / 2 + 4);
  launch_kernel(pack_input_u8_kernel, grid_for(total, 256), 256, 0, s, x, reinterpret_cast<uint4*>(out), n_images, H, W);
  ARGUS_CUDA(cudaGetLastError());
}

// ------------------------------------------------------------------------------------------------------------
// weight packing / gradient unpacking (table driven: one launch for all layers)
// ------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int64_t packed_count(const WeightPackEntry& e) {
  return e.kind == 1 ? 64 * 256 : static_cast<int64_t>(e.cout) * e.cin * e.kk;
}
// maps a packed index to the PyTorch-layout index (or -1 for a zero-padding slot of the stem)
__device__ __forceinline__ int64_t packed_to_torch(const WeightPackEntry& e, int64_t i) {
  if (e.kind == 1) {
    const int ch = static_cast<int>(i & 15);
    const int q = static_cast<int>((i >> 4) & 3);
    const int p = static_cast<int>((i >> 6) & 3);
    const int co = static_cast<int>(i >> 8);
    if (ch >= 12) return -1;
    const int ab = ch / 3, c = ch - ab * 3;
    const int a = ab >> 1, b = ab & 1;
    const int kh = 2 * p + a - 1, kw = 2 * q + b - 1;
    if (kh < 0 || kh > 6 || kw < 0 || kw > 6) return -1;
    return ((static_cast<int64_t>(co) * 3 + c) * 7 + kh) * 7 + kw;
  }
  const int ci = static_cast<int>(i % e.cin);
  const int64_t r = i / e.cin;
  const int t = static_cast<int>(r % e.kk);
  const int co = static_cast<int>(r / e.kk);
  return (static_cast<int64_t>(co) * e.cin + ci) * e.kk + t;
}

// k x k entries are transposed one output channel at a time through shared memory ([ci][t] <-> [t][ci] inside the
// contiguous cin * kk block of that channel), so both the global reads and the global writes are coalesced; 1x1 / linear
// entries are already in the packed order; the stem (kind 1) keeps the per-element index map (it is 16 K elements).
constexpr int kPackTileMax = 512 * 9 + 9;   // largest cin * kk block (+ padding for the unpack direction)
__global__ void __launch_bounds__(256)
pack_weights_kernel(const float* __restrict__ params, bf16* __restrict__ packed,
                    const WeightPackEntry* __restrict__ table) {
  pdl_prologue();
  __shared__ float tile[kPackTileMax];
  const WeightPackEntry e = table[blockIdx.y];
  const int64_t n = packed_count(e);
  if (e.kind == 0 && e.kk > 1 && e.cin * e.kk <= kPackTileMax) {
    const int row = e.cin * e.kk;
    for (int co = blockIdx.x; co < e.cout; co += gridDim.x) {
      const float* src = params + e.src_off + static_cast<int64_t>(co) * row;
      for (int j = threadIdx.x; j < row; j += blockDim.x) tile[j] = src[j];   // [ci][t]
      __syncthreads();
      bf16* dst = packed + e.dst_off + static_cast<int64_t>(co) * row;
      for (int j = threadIdx.x; j < row; j += blockDim.x) {                   // j = t * cin + ci
        const int t = j / e.cin, ci = j - t * e.cin;
        dst[j] = __float2bfloat16(tile[ci * e.kk + t]);
      }
      __syncthreads();
    }
    return;
  }
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t src = packed_to_torch(e, i);
    packed[e.dst_off + i] = __float2bfloat16(src >= 0 ? params[e.src_off + src] : 0.f);
  }
}
__global__ void __launch_bounds__(256)
unpack_wgrads_kernel(const float* __restrict__ packed_grads, float* __restrict__ grads,
                     const WeightPackEntry* __restrict__ table) {
  pdl_prologue();
  __shared__ float tile[kPackTileMax];
  const WeightPackEntry e = table[blockIdx.y];
  if (e.kind == 0 && e.kk == 1) return;  // 1x1 / linear layers accumulate straight into the gradient arena
  const int64_t n = packed_count(e);
  if (e.kind == 0 && (e.cin + 1) * e.kk <= kPackTileMax) {
    const int row = e.cin * e.kk, pitch = e.cin + 1;   // padded rows: the transposed reads spread over the banks
    for (int co = blockIdx.x; co < e.cout; co += gridDim.x) {
      const float* src = packed_grads + e.dst_off + static_cast<int64_t>(co) * row;
      for (int j = threadIdx.x; j < row; j += blockDim.x) {                   // j = t * cin + ci
        const int t = j / e.cin, ci = j - t * e.cin;
        tile[t * pitch + ci] = src[j];
      }
      __syncthreads();
      float* dst = grads + e.src_off + static_cast<int64_t>(co) * row;
      for (int j = threadIdx.x; j < row; j += blockDim.x) {                   // j = ci * kk + t
        const int ci = j / e.kk, t = j - ci * e.kk;
        dst[j] += tile[t * pitch + ci];
      }
      __syncthreads();
    }
    return;
  }
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t dst = packed_to_torch(e, i);
    if (dst >= 0) grads[e.src_off + dst] += packed_grads[e.dst_off + i];
  }
}
void pack_weights(const float* params, bf16* packed, const WeightPackEntry* table_dev, int n_entries,
                  cudaStream_t s) {
  ProfileScope prof("pack_weights", s, 0, 0);
  // 256 blocks per entry: a 512-channel 3x3 layer is two output channels per block (one load / transpose / store round each)
  launch_kernel(pack_weights_kernel, dim3(256, n_entries), 256, 0, s, params, packed, table_dev);
  ARGUS_CUDA(cudaGetLastError());
}
void unpack_wgrads(const float* packed_grads, float* grads, const WeightPackEntry* table_dev, int n_entries,
                   cudaStream_t s) {
  ProfileScope prof("unpack_wgrads", s, 0, 0);
  launch_kernel(unpack_wgrads_kernel, dim3(256, n_entries), 256, 0, s, packed_grads, grads, table_dev);
  ARGUS_CUDA(cudaGetLastError());
}
// diag(scale) W in the packed layout: every element is rounded once, bf16_rn(scale[co] * w). Runs once per refresh of the
// eval-mode fold, so it keeps the plain per-element index map of the stem branch above for every entry.
__global__ void __launch_bounds__(256)
pack_weights_scaled_kernel(const float* __restrict__ params, const float* __restrict__ scales,
                           const int64_t* __restrict__ scale_off, bf16* __restrict__ packed,
                           const WeightPackEntry* __restrict__ table) {
  pdl_prologue();
  const WeightPackEntry e = table[blockIdx.y];
  const float* sc = scales + scale_off[blockIdx.y];
  const int64_t n = packed_count(e);
  const int64_t row = n / e.cout;   // packed row of one output channel (stem: 256)
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t src = packed_to_torch(e, i);
    packed[e.dst_off + i] = __float2bfloat16(src >= 0 ? sc[i / row] * params[e.src_off + src] : 0.f);
  }
}
void pack_weights_scaled(const float* params, const float* scales, const int64_t* scale_off_dev, bf16* packed,
                         const WeightPackEntry* table_dev, int n_entries, cudaStream_t s) {
  ProfileScope prof("pack_weights", s, 0, 0);
  launch_kernel(pack_weights_scaled_kernel, dim3(256, n_entries), 256, 0, s, params, scales, scale_off_dev, packed,
                table_dev);
  ARGUS_CUDA(cudaGetLastError());
}

// plain 4-byte global load as a volatile asm statement: a run of these is issued back to back (the compiler keeps
// their order and cannot fold the consumers in between), so N partial sums cost one memory round trip, not N
__device__ __forceinline__ float ldg_f32_issue(const float* p) {
  float v;
  asm volatile("ld.global.nc.f32 %0, [%1];" : "=f"(v) : "l"(p));
  return v;
}

// ------------------------------------------------------------------------------------------------------------
// batch norm: finalize / fold, and the ordered sum of per-block partials every finalize shares
// ------------------------------------------------------------------------------------------------------------
// Sums of the NS series of partial = [slots][NS][C] for channel c = blockIdx.x * 8 + (threadIdx.x & 7).
// Block = 8 channels x 32 slot lanes: lane sl adds slots sl, sl+32, ... in order in fp64, then lane 0 adds the 32 lane
// sums in order -> bitwise reproducible, and the slot loop is 32-way parallel (a single thread per channel took 80 us
// over 1184 partials). The loads of eight slots are issued together (one L2 round trip instead of eight); missing
// slots are skipped, so the additions are those of the plain loop.
// Returns true in the one thread per channel (lane 0, c < C) that then holds the channel's totals in sum[].
template <int NS>
__device__ __forceinline__ bool ordered_slot_sum(const float* __restrict__ partial, int slots, int C, double (&sum)[NS]) {
  __shared__ double red[NS][32][8];
  const int ch = threadIdx.x & 7, sl = threadIdx.x >> 3;
  const int c = blockIdx.x * 8 + ch;
#pragma unroll
  for (int j = 0; j < NS; ++j) sum[j] = 0.0;
  if (c < C) {
    for (int k = sl; k < slots; k += 32 * 8) {
      float a[8][NS];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int kk = min(k + 32 * u, slots - 1);   // clamped: always a valid address, masked below
#pragma unroll
        for (int j = 0; j < NS; ++j) a[u][j] = ldg_f32_issue(partial + (static_cast<size_t>(kk) * NS + j) * C + c);
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        if (k + 32 * u < slots) {
#pragma unroll
          for (int j = 0; j < NS; ++j) sum[j] += static_cast<double>(a[u][j]);
        }
      }
    }
  }
#pragma unroll
  for (int j = 0; j < NS; ++j) red[j][sl][ch] = sum[j];
  __syncthreads();
  if (sl != 0 || c >= C) return false;
#pragma unroll
  for (int j = 0; j < NS; ++j) sum[j] = 0.0;
  for (int k = 0; k < 32; ++k) {
#pragma unroll
    for (int j = 0; j < NS; ++j) sum[j] += red[j][k][ch];
  }
  return true;
}

__global__ void __launch_bounds__(256)
bn_finalize_kernel(const float* __restrict__ partial, int slots, double count, const float* gamma, const float* beta,
                   float* running_mean, float* running_var, float momentum, float eps, float* scale, float* shift,
                   float* save_mean, float* save_invstd, int C) {
  pdl_prologue();
  double s[2];   // sum x, sum x^2
  if (!ordered_slot_sum<2>(partial, slots, C, s)) return;
  const int c = blockIdx.x * 8 + (threadIdx.x & 7);
  const double mean = s[0] / count;
  double var = s[1] / count - mean * mean;
  if (var < 0) var = 0;
  const float invstd = static_cast<float>(1.0 / sqrt(var + static_cast<double>(eps)));
  const float sc = gamma[c] * invstd;
  scale[c] = sc;
  shift[c] = beta[c] - static_cast<float>(mean) * sc;
  save_mean[c] = static_cast<float>(mean);
  save_invstd[c] = invstd;
  if (running_mean != nullptr) {
    const double unbiased = count > 1 ? var * count / (count - 1) : var;
    running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * static_cast<float>(mean);
    running_var[c] = (1.f - momentum) * running_var[c] + momentum * static_cast<float>(unbiased);
  }
}
void bn_finalize(const float* partial, int slots, double count, const float* gamma, const float* beta,
                 float* running_mean, float* running_var, float momentum, float eps, float* scale, float* shift,
                 float* save_mean, float* save_invstd, int C, cudaStream_t s) {
  ProfileScope prof("bn_finalize", s, 0, (8.0 * slots + 40.0) * C);
  launch_kernel(bn_finalize_kernel, (C + 7) / 8, 256, 0, s, partial, slots, count, gamma, beta, running_mean, running_var,
                                                     momentum, eps, scale, shift, save_mean, save_invstd, C);
  ARGUS_CUDA(cudaGetLastError());
}
__global__ void bn_fold_eval_kernel(const float* gamma, const float* beta, const float* rm, const float* rv, float eps,
                                    float* scale, float* shift, float* mean, float* invstd, int C) {
  pdl_prologue();
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const float is = rsqrtf(rv[c] + eps);
  const float sc = gamma[c] * is;
  scale[c] = sc;
  shift[c] = beta[c] - rm[c] * sc;
  if (mean != nullptr) {
    mean[c] = rm[c];
    invstd[c] = is;
  }
}
void bn_fold_eval(const float* gamma, const float* beta, const float* running_mean, const float* running_var,
                  float eps, float* scale, float* shift, int C, cudaStream_t s, float* mean, float* invstd) {
  ProfileScope prof("bn_finalize", s, 0, 24.0 * C);
  launch_kernel(bn_fold_eval_kernel, (C + 127) / 128, 128, 0, s, gamma, beta, running_mean, running_var, eps, scale, shift,
                mean, invstd, C);
  ARGUS_CUDA(cudaGetLastError());
}

__global__ void __launch_bounds__(256)
bn_bwd_finalize_kernel(const float* __restrict__ partial, int blocks, float* dgamma, float* dbeta, int C,
                       const float* __restrict__ mean, const float* __restrict__ invstd) {
  pdl_prologue();
  double s[2];   // sum g, sum g * xhat
  if (!ordered_slot_sum<2>(partial, blocks, C, s)) return;
  const int c = blockIdx.x * 8 + (threadIdx.x & 7);
  // mean != nullptr: the second sums are sum(g * x) of the RAW layer output (statistics slots of a dgrad epilogue,
  // bn_bwd_finalize_slots); centred and scaled here, once, in double
  if (mean != nullptr) s[1] = (s[1] - static_cast<double>(mean[c]) * s[0]) * static_cast<double>(invstd[c]);
  dbeta[c] += static_cast<float>(s[0]);
  dgamma[c] += static_cast<float>(s[1]);
}

__global__ void __launch_bounds__(256)
colsum_final_kernel(const float* __restrict__ partial, int blocks, float* __restrict__ out, int C) {
  pdl_prologue();
  double s[1];
  if (ordered_slot_sum<1>(partial, blocks, C, s)) out[blockIdx.x * 8 + (threadIdx.x & 7)] = static_cast<float>(s[0]);
}
void colsum_finalize(const float* partial, int blocks, float* out, int C, cudaStream_t st) {
  launch_kernel(colsum_final_kernel, (C + 7) / 8, 256, 0, st, partial, blocks, out, C);
  ARGUS_CUDA(cudaGetLastError());
}

// ------------------------------------------------------------------------------------------------------------
// Batch-norm apply and backward passes through a shared-memory ring. A producer warp streams 8 KB slices of each input
// tensor into a ring of stages with 1-D bulk copies (TMA) that complete on mbarriers; eight consumer warps read their
// 16-byte vectors from the landed stage, release it, and do the math. The bytes in flight per SM are set by the ring
// (2 CTAs x 5 stages x 16 KB) instead of by the registers the loads of one loop iteration can hold (1024 threads x
// 64 B), which is what held earlier register-streaming kernels of these passes at 55-70 % of the HBM copy bandwidth
// (DESIGN.md section 4). Bulk copies and 16-byte vectors need every tensor 16-byte aligned: bn_check_aligned rejects
// anything else on the host.
// ------------------------------------------------------------------------------------------------------------
void bn_check_aligned(const void* a, const void* b, const void* c, const void* d) {
  for (const void* p : {a, b, c, d})
    ARGUS_CHECK((reinterpret_cast<uintptr_t>(p) & 15u) == 0, "batch norm: every tensor must be 16-byte aligned");
}

constexpr int kRingVec = 512;                 // vectors per tensor per stage: two per consumer thread
constexpr int kRingTensor = kRingVec * 16;    // bytes of one bf16 tensor per stage
constexpr int kRingThreads = 288;             // 8 consumer warps + 1 producer warp
// A stage holds up to three tensors of B0, B1, B2 bytes (kRingTensor: bf16 vectors, kRingVec: a ReLU bit mask, one byte
// per vector, 0: absent); the full / empty mbarriers of all stages follow the stages.
template <int B0, int B1, int B2, int STAGES>
struct Ring {
  static constexpr int kBytes0 = B0, kBytes1 = B1, kBytes2 = B2;
  static constexpr int kStages = STAGES;
  static constexpr int kStageBytes = B0 + B1 + B2;
  static constexpr int kOffBars = kStages * kStageBytes;
  static constexpr int kTotal = kOffBars + 2 * kStages * 8;
  static_assert(kOffBars >= 8 * 16 * 32 * 4, "the block reduction reuses the ring memory");
};
// 2 CTAs x 5 stages x 16 KB in flight per SM is far more than HBM latency needs; stopping at ~80 KB per CTA leaves room
// for one CTA of the (ALU-bound, 41 KB) augmentation kernel of the next batch to share the SM.
// Backward: dy, x (+ the block output for MASK 2, + the ReLU bit mask for MASK 3).
template <int MASK>
using BnRing = Ring<kRingTensor, kRingTensor, MASK == 2 ? kRingTensor : (MASK == 3 ? kRingVec : 0), MASK == 2 ? 3 : 5>;
// Forward apply: x (+ residual).
template <int RES>
using ApplyRing = Ring<kRingTensor, RES ? kRingTensor : 0, 0, RES ? 5 : 10>;

__device__ __forceinline__ void bn_ring_init(uint32_t sbase, int off_bars, int stages) {
  if (threadIdx.x == 0) {
    for (int s = 0; s < stages; ++s) {
      mbar_init(sbase + off_bars + 8u * s, 1);
      mbar_init(sbase + off_bars + 8u * (stages + s), 8);   // one arrive per consumer warp
    }
    fence_mbar_init();
  }
  __syncthreads();
}
// producer (one thread): the full stages c = blockIdx.x, blockIdx.x + gridDim.x, ... of tensors t0, t1, t2
template <class R>
__device__ __forceinline__ void ring_produce(uint32_t sbase, const void* t0, const void* t1, const void* t2,
                                             int64_t nvec) {
  const int64_t nfull = nvec / kRingVec;
  int s = 0;
  uint32_t ph = 0;
  for (int64_t c = blockIdx.x; c < nfull; c += gridDim.x) {
    const uint32_t full = sbase + R::kOffBars + 8u * s, empty = sbase + R::kOffBars + 8u * (R::kStages + s);
    mbar_wait(empty, ph ^ 1);
    mbar_arrive_expect_tx(full, R::kStageBytes);
    const uint32_t dst = sbase + s * R::kStageBytes;
    bulk_load_1d(dst, static_cast<const uint8_t*>(t0) + c * R::kBytes0, R::kBytes0, full);
    if (R::kBytes1) bulk_load_1d(dst + R::kBytes0, static_cast<const uint8_t*>(t1) + c * R::kBytes1, R::kBytes1, full);
    if (R::kBytes2)
      bulk_load_1d(dst + R::kBytes0 + R::kBytes1, static_cast<const uint8_t*>(t2) + c * R::kBytes2, R::kBytes2, full);
    if (++s == R::kStages) { s = 0; ph ^= 1; }
  }
}
// vector i of a tensor with BYTES bytes per stage: 16 bytes, one bit-mask byte (in .x), or zeros when absent
template <int BYTES>
__device__ __forceinline__ uint4 ring_elem(const void* p, int64_t i) {
  static_assert(BYTES == kRingTensor || BYTES == kRingVec || BYTES == 0, "ring tensors are bf16 vectors or bit masks");
  uint4 v = make_uint4(0, 0, 0, 0);
  if (BYTES == kRingTensor) v = static_cast<const uint4*>(p)[i];
  if (BYTES == kRingVec) v.x = static_cast<const uint8_t*>(p)[i];
  return v;
}
// consumers (threads 0..255): for each full stage of this block, wait until it has landed, take thread t's two vectors
// of every tensor, release the stage, then body(i, v0, v1, v2) for i = c * kRingVec + t and i + 256. Block 0 then does
// the ragged tail (< one stage) straight from global memory.
template <class R, class Body>
__device__ __forceinline__ void ring_consume(const uint8_t* smem, uint32_t sbase, const void* t0, const void* t1,
                                             const void* t2, int64_t nvec, Body&& body) {
  const int t = threadIdx.x;
  const int64_t nfull = nvec / kRingVec;
  int s = 0;
  uint32_t ph = 0;
  for (int64_t c = blockIdx.x; c < nfull; c += gridDim.x) {
    mbar_wait(sbase + R::kOffBars + 8u * s, ph);
    const uint8_t* s0 = smem + s * R::kStageBytes;
    const uint8_t* s1 = s0 + R::kBytes0;
    const uint8_t* s2 = s1 + R::kBytes1;
    const uint4 a0 = ring_elem<R::kBytes0>(s0, t), a1 = ring_elem<R::kBytes0>(s0, t + 256);
    const uint4 b0 = ring_elem<R::kBytes1>(s1, t), b1 = ring_elem<R::kBytes1>(s1, t + 256);
    const uint4 e0 = ring_elem<R::kBytes2>(s2, t), e1 = ring_elem<R::kBytes2>(s2, t + 256);
    __syncwarp();
    if ((t & 31) == 0) mbar_arrive(sbase + R::kOffBars + 8u * (R::kStages + s));   // stage free: data is in registers
    const int64_t i0 = c * kRingVec + t;
    body(i0, a0, b0, e0);
    body(i0 + 256, a1, b1, e1);
    if (++s == R::kStages) { s = 0; ph ^= 1; }
  }
  if (blockIdx.x == 0) {
    for (int64_t i = nfull * kRingVec + t; i < nvec; i += 256)
      body(i, ring_elem<R::kBytes0>(t0, i), ring_elem<R::kBytes1>(t1, i), ring_elem<R::kBytes2>(t2, i));
  }
}
// Per-block column sums of NV values per thread (NV / 8 series of the eight channels of octet t mod lanes) into
// partial[blockIdx.x][NV / 8][C]: warp shuffles across the lanes of a warp that share an octet (lanes < 32), then one
// pass over the eight consumer warps through [warp][value][lane] in the ring memory, which is free once every stage is
// consumed. Fixed order -> deterministic. Called by all kRingThreads threads; the producer warp's values are ignored.
template <int NV>
__device__ __forceinline__ void ring_block_sums(float (&v)[NV], uint8_t* smem, int lanes, float* partial, int C) {
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  if (warp < 8) {
    for (int o = 16; o >= lanes; o >>= 1) {
#pragma unroll
      for (int k = 0; k < NV; ++k) v[k] += __shfl_xor_sync(0xffffffffu, v[k], o);
    }
  }
  __syncthreads();
  float (*red)[NV][32] = reinterpret_cast<float (*)[NV][32]>(smem);
  if (warp < 8) {
#pragma unroll
    for (int k = 0; k < NV; ++k) red[warp][k][lane] = v[k];
  }
  __syncthreads();
  // thread t < lanes owns octet t; the warps holding it are w = (t / 32) + j * (lanes / 32) for lanes >= 32, all eight
  // warps (lane t) for lanes < 32
  if (t < lanes) {
    const int wstep = lanes >= 32 ? lanes / 32 : 1;
    const int w0 = lanes >= 32 ? t / 32 : 0;
    float sum[NV];
#pragma unroll
    for (int k = 0; k < NV; ++k) sum[k] = 0.f;
    for (int w = w0; w < 8; w += wstep) {   // the NV sums are independent chains: their loads overlap
#pragma unroll
      for (int k = 0; k < NV; ++k) sum[k] += red[w][k][lane];
    }
#pragma unroll
    for (int k = 0; k < NV; ++k) partial[(static_cast<size_t>(blockIdx.x) * (NV / 8) + k / 8) * C + t * 8 + k % 8] = sum[k];
  }
}

// Masked gradient of eight channels. MASK 0: no ReLU after the batch norm; 1: ReLU right after it (mask recomputed from
// x); 2: ReLU after a residual add (mask = block output > 0); 3: like 2, from the ReLU bit mask (byte in ov4.x).
template <int MASK>
__device__ __forceinline__ F8 bn_masked_grad(const F8& d, const F8& xv, const uint4& ov4, const F8& sc, const F8& sh) {
  F8 g = d;
  if (MASK == 1) {
#pragma unroll
    for (int k = 0; k < 8; ++k) g.v[k] = fmaf(xv.v[k], sc.v[k], sh.v[k]) > 0.f ? d.v[k] : 0.f;
  } else if (MASK == 2) {
    const F8 o = unpack8(ov4);
#pragma unroll
    for (int k = 0; k < 8; ++k) g.v[k] = o.v[k] > 0.f ? d.v[k] : 0.f;
  } else if (MASK == 3) {
#pragma unroll
    for (int k = 0; k < 8; ++k) g.v[k] = ((ov4.x >> k) & 1u) ? d.v[k] : 0.f;
  }
  return g;
}
// dx = sc * (g - db/M - xhat * dg/M) with xhat = (x - mu) * is   ==   sc*g + k1*x + k0 (per-channel pointers at c0)
__device__ __forceinline__ void bn_dx_coeffs(const F8& sc, const float* mean, const float* invstd, const float* dgamma,
                                             const float* dbeta, float inv_rows, F8& k0, F8& k1) {
  const F8 mu = load8f(mean), is = load8f(invstd), dg = load8f(dgamma), db = load8f(dbeta);
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const float c2 = sc.v[k] * dg.v[k] * inv_rows * is.v[k];
    k1.v[k] = -c2;
    k0.v[k] = fmaf(c2, mu.v[k], -sc.v[k] * db.v[k] * inv_rows);
  }
}

// y = [relu](x*scale+shift [+ res | + res*rscale+rshift]) (+ ReLU bits, + per-block column sums of the stored y).
// RES: 0 none, 1 plain residual, 2 residual with its own scale/shift (downsample branch).
template <int RES, bool SUM>
__global__ void __launch_bounds__(kRingThreads, 2)
bn_apply_ring_kernel(const uint4* __restrict__ x, const float* __restrict__ scale, const float* __restrict__ shift,
                     const uint4* __restrict__ res, const float* __restrict__ rscale, const float* __restrict__ rshift,
                     int relu, uint4* __restrict__ y, uint8_t* __restrict__ bits, float* __restrict__ colsum_partial,
                     int64_t nvec, int cvec) {
  pdl_prologue();
  using R = ApplyRing<RES>;
  extern __shared__ __align__(128) uint8_t ring_smem[];
  const uint32_t sbase = smem_u32(ring_smem);
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  bn_ring_init(sbase, R::kOffBars, R::kStages);
  const int lanes = cvec < 256 ? cvec : 256;
  const int c0 = (t & (lanes - 1)) * 8;
  F8 acc;
#pragma unroll
  for (int k = 0; k < 8; ++k) acc.v[k] = 0.f;
  if (warp == 8) {
    if (lane == 0) ring_produce<R>(sbase, x, res, nullptr, nvec);
    if (!SUM) return;
  } else {
    const F8 sc = load8f(scale + c0), sh = load8f(shift + c0);
    F8 rs, rb;
    if (RES == 2) { rs = load8f(rscale + c0); rb = load8f(rshift + c0); }
    auto one = [&](int64_t i, const uint4& xq, const uint4& rq, const uint4&) {
      const F8 xv = unpack8(xq);
      F8 o;
#pragma unroll
      for (int k = 0; k < 8; ++k) o.v[k] = fmaf(xv.v[k], sc.v[k], sh.v[k]);
      if (RES == 1) {
        const F8 rv = unpack8(rq);
#pragma unroll
        for (int k = 0; k < 8; ++k) o.v[k] += rv.v[k];
      } else if (RES == 2) {
        const F8 rv = unpack8(rq);
#pragma unroll
        for (int k = 0; k < 8; ++k) o.v[k] += fmaf(rv.v[k], rs.v[k], rb.v[k]);
      }
      if (bits != nullptr) bits[i] = positive_bits(o);
      if (relu) {
#pragma unroll
        for (int k = 0; k < 8; ++k) o.v[k] = fmaxf(o.v[k], 0.f);
      }
      const uint4 packed = pack8(o);
      y[i] = packed;
      if (SUM) {
        const F8 r = unpack8(packed);   // sums of the STORED (bf16) values
#pragma unroll
        for (int k = 0; k < 8; ++k) acc.v[k] += r.v[k];
      }
    };
    ring_consume<R>(ring_smem, sbase, x, res, nullptr, nvec, one);
  }
  if (SUM) ring_block_sums<8>(acc.v, ring_smem, lanes, colsum_partial, cvec * 8);
}

template <int MASK>
__global__ void __launch_bounds__(kRingThreads, 2)
bn_bwd_reduce_ring_kernel(const uint4* __restrict__ dy, const uint4* __restrict__ x, const uint4* __restrict__ out,
                          const float* __restrict__ scale, const float* __restrict__ shift,
                          const float* __restrict__ mean, const float* __restrict__ invstd,
                          float* __restrict__ partial, int64_t nvec, int cvec) {
  pdl_prologue();
  using R = BnRing<MASK>;
  extern __shared__ __align__(128) uint8_t ring_smem[];
  const uint32_t sbase = smem_u32(ring_smem);
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  bn_ring_init(sbase, R::kOffBars, R::kStages);
  const int lanes = cvec < 256 ? cvec : 256;
  const int c0 = (t & (lanes - 1)) * 8;
  float a_dy[8], a_dyx[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) a_dy[k] = a_dyx[k] = 0.f;
  if (warp == 8) {
    if (lane == 0) ring_produce<R>(sbase, dy, x, out, nvec);
  } else {
    F8 sc, sh;
    if (MASK == 1) { sc = load8f(scale + c0); sh = load8f(shift + c0); }
    auto body = [&](int64_t, const uint4& dyv, const uint4& xv4, const uint4& ov4) {
      const F8 xv = unpack8(xv4);
      const F8 g = bn_masked_grad<MASK>(unpack8(dyv), xv, ov4, sc, sh);
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        a_dy[k] += g.v[k];
        a_dyx[k] = fmaf(g.v[k], xv.v[k], a_dyx[k]);   // sum g*x; centred and scaled by invstd once at the end
      }
    };
    ring_consume<R>(ring_smem, sbase, dy, x, out, nvec, body);
  }
  // partial[block][0][c] = sum g, partial[block][1][c] = sum g * xhat
  float v[16];
  {
    F8 mu, is;
    if (t < 256) { mu = load8f(mean + c0); is = load8f(invstd + c0); }
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      v[k] = a_dy[k];
      v[8 + k] = t < 256 ? (a_dyx[k] - mu.v[k] * a_dy[k]) * is.v[k] : 0.f;
    }
  }
  ring_block_sums<16>(v, ring_smem, lanes, partial, cvec * 8);
}

template <int MASK>
__global__ void __launch_bounds__(kRingThreads, 2)
bn_bwd_apply_ring_kernel(uint4* __restrict__ dy, const uint4* __restrict__ x, const uint4* __restrict__ out,
                         const float* __restrict__ scale, const float* __restrict__ shift,
                         const float* __restrict__ mean, const float* __restrict__ invstd,
                         const float* __restrict__ dgamma, const float* __restrict__ dbeta, uint4* __restrict__ dx,
                         int64_t nvec, int cvec, float inv_rows) {
  pdl_prologue();
  using R = BnRing<MASK>;
  extern __shared__ __align__(128) uint8_t ring_smem[];
  const uint32_t sbase = smem_u32(ring_smem);
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  bn_ring_init(sbase, R::kOffBars, R::kStages);
  if (warp == 8) {
    if (lane == 0) ring_produce<R>(sbase, dy, x, out, nvec);
    return;
  }
  const int c0 = (t & ((cvec < 256 ? cvec : 256) - 1)) * 8;
  const F8 sc = load8f(scale + c0);
  F8 sh;
  if (MASK == 1) sh = load8f(shift + c0);
  F8 k0, k1;
  bn_dx_coeffs(sc, mean + c0, invstd + c0, dgamma + c0, dbeta + c0, inv_rows, k0, k1);
  auto body = [&](int64_t i, const uint4& dyv, const uint4& xv4, const uint4& ov4) {
    const F8 xv = unpack8(xv4);
    const F8 g = bn_masked_grad<MASK>(unpack8(dyv), xv, ov4, sc, sh);
    F8 r;
#pragma unroll
    for (int k = 0; k < 8; ++k) r.v[k] = fmaf(sc.v[k], g.v[k], fmaf(k1.v[k], xv.v[k], k0.v[k]));
    dx[i] = pack8(r);
    if (MASK == 2) dy[i] = pack8(g);
  };
  ring_consume<R>(ring_smem, sbase, dy, x, out, nvec, body);
}

// one ring kernel instance with R::kTotal bytes of dynamic shared memory (opted in on its first launch)
template <auto kKernel, class R, class... Args>
static void launch_ring(int grid, cudaStream_t s, Args&&... args) {
  static const bool once = [] {
    ARGUS_CUDA(cudaFuncSetAttribute(kKernel, cudaFuncAttributeMaxDynamicSharedMemorySize, R::kTotal));
    return true;
  }();
  (void)once;
  launch_kernel(kKernel, grid, kRingThreads, R::kTotal, s, std::forward<Args>(args)...);
  ARGUS_CUDA(cudaGetLastError());
}
static int bn_ring_grid(int64_t nvec) {
  return static_cast<int>(std::max<int64_t>(1, std::min<int64_t>(nvec / kRingVec, 2LL * num_sms())));
}

// number of per-block column-sum partials bn_apply writes (callers size and finalize the buffer with this)
int bn_apply_grid(int64_t rows, int C) { return bn_ring_grid(rows * (C / 8)); }
void bn_apply(const bf16* x, const float* scale, const float* shift, const bf16* res, const float* rscale,
              const float* rshift, int relu, bf16* y, uint8_t* relu_bits, float* colsum_partial, int64_t rows, int C,
              cudaStream_t s) {
  bn_check_aligned(x, res, y, relu_bits);
  ProfileScope prof("bn_apply", s, 0, static_cast<double>(rows) * C * (2 * (res ? 3 : 2) + (relu_bits ? 0.125 : 0.0)));
  ARGUS_CHECK(C % 8 == 0 && is_pow2(C / 8) && C <= 2048, "bn_apply: C/8 must be a power of two <= 256");
  ARGUS_CHECK(colsum_partial == nullptr || res == nullptr, "column sums are only produced by the plain (no residual) variant");
  const int cvec = C / 8;
  const int64_t nvec = rows * cvec;
  const int grid = bn_ring_grid(nvec);
  auto X = reinterpret_cast<const uint4*>(x);
  auto R = reinterpret_cast<const uint4*>(res);
  auto Y = reinterpret_cast<uint4*>(y);
  if (colsum_partial != nullptr)
    launch_ring<bn_apply_ring_kernel<0, true>, ApplyRing<0>>(grid, s, X, scale, shift, R, rscale, rshift, relu, Y, relu_bits, colsum_partial, nvec, cvec);
  else if (res == nullptr)
    launch_ring<bn_apply_ring_kernel<0, false>, ApplyRing<0>>(grid, s, X, scale, shift, R, rscale, rshift, relu, Y, relu_bits, colsum_partial, nvec, cvec);
  else if (rscale == nullptr)
    launch_ring<bn_apply_ring_kernel<1, false>, ApplyRing<1>>(grid, s, X, scale, shift, R, rscale, rshift, relu, Y, relu_bits, colsum_partial, nvec, cvec);
  else
    launch_ring<bn_apply_ring_kernel<2, false>, ApplyRing<2>>(grid, s, X, scale, shift, R, rscale, rshift, relu, Y, relu_bits, colsum_partial, nvec, cvec);
}

int64_t bn_bwd_scratch_elems() { return 4LL * num_sms() * 2 * 2048; }

void bn_bwd_reduce(const bf16* dy, const bf16* x, const bf16* out, const float* scale, const float* shift,
                   const float* mean, const float* invstd, float* dgamma, float* dbeta, int64_t rows, int C,
                   int mask_mode, float* scratch, cudaStream_t s) {
  bn_check_aligned(dy, x, out);
  ARGUS_CHECK(scratch != nullptr, "bn_bwd_reduce needs a scratch buffer");
  std::string fam = "bn_bwd_reduce";
  if (profile_enabled() && profile_detailed()) fam += ":R" + std::to_string(rows) + "_C" + std::to_string(C) + "_m" + std::to_string(mask_mode);
  ProfileScope prof(fam, s, 0, static_cast<double>(rows) * C * (mask_mode == 2 ? 6.0 : (mask_mode == 3 ? 4.125 : 4.0)));
  ARGUS_CHECK(C % 8 == 0 && is_pow2(C / 8) && C <= 2048, "bn_bwd_reduce: C/8 must be a power of two <= 256");
  const int cvec = C / 8;
  const int64_t nvec = rows * cvec;
  const int grid = bn_ring_grid(nvec);
  auto DY = reinterpret_cast<const uint4*>(dy);
  auto X = reinterpret_cast<const uint4*>(x);
  auto O = reinterpret_cast<const uint4*>(out);
  switch (mask_mode) {
    case 0: launch_ring<bn_bwd_reduce_ring_kernel<0>, BnRing<0>>(grid, s, DY, X, O, scale, shift, mean, invstd, scratch, nvec, cvec); break;
    case 1: launch_ring<bn_bwd_reduce_ring_kernel<1>, BnRing<1>>(grid, s, DY, X, O, scale, shift, mean, invstd, scratch, nvec, cvec); break;
    case 2:
      ARGUS_CHECK(out != nullptr, "mask_mode 2 needs the block output");
      launch_ring<bn_bwd_reduce_ring_kernel<2>, BnRing<2>>(grid, s, DY, X, O, scale, shift, mean, invstd, scratch, nvec, cvec);
      break;
    case 3:
      ARGUS_CHECK(out != nullptr, "mask_mode 3 needs the ReLU bit mask");
      launch_ring<bn_bwd_reduce_ring_kernel<3>, BnRing<3>>(grid, s, DY, X, O, scale, shift, mean, invstd, scratch, nvec, cvec);
      break;
    default: throw Error("bad mask_mode");
  }
  launch_kernel(bn_bwd_finalize_kernel, (C + 7) / 8, 256, 0, s, scratch, grid, dgamma, dbeta, C, nullptr, nullptr);
  ARGUS_CUDA(cudaGetLastError());
}

void bn_bwd_finalize_slots(const float* partial, int slots, const float* mean, const float* invstd, float* dgamma,
                           float* dbeta, int C, cudaStream_t s) {
  ProfileScope prof("bn_bwd_reduce", s, 0, static_cast<double>(slots) * 2 * C * 4);
  launch_kernel(bn_bwd_finalize_kernel, (C + 7) / 8, 256, 0, s, partial, slots, dgamma, dbeta, C, mean, invstd);
  ARGUS_CUDA(cudaGetLastError());
}

void bn_bwd_apply(bf16* dy, const bf16* x, const bf16* out, const float* scale, const float* shift,
                  const float* mean, const float* invstd, const float* dgamma, const float* dbeta, bf16* dx,
                  int64_t rows, int C, int mask_mode, cudaStream_t s) {
  bn_check_aligned(dy, x, out, dx);
  ProfileScope prof("bn_bwd_apply", s, 0, static_cast<double>(rows) * C * (mask_mode == 2 ? 10.0 : (mask_mode == 3 ? 6.125 : 6.0)));
  ARGUS_CHECK(C % 8 == 0 && is_pow2(C / 8) && C <= 2048, "bn_bwd_apply: C/8 must be a power of two <= 256");
  const int cvec = C / 8;
  const int64_t nvec = rows * cvec;
  const int grid = bn_ring_grid(nvec);
  const float inv_rows = static_cast<float>(1.0 / static_cast<double>(rows));
  auto DY = reinterpret_cast<uint4*>(dy);
  auto X = reinterpret_cast<const uint4*>(x);
  auto O = reinterpret_cast<const uint4*>(out);
  auto DX = reinterpret_cast<uint4*>(dx);
  switch (mask_mode) {
    case 0: launch_ring<bn_bwd_apply_ring_kernel<0>, BnRing<0>>(grid, s, DY, X, O, scale, shift, mean, invstd, dgamma, dbeta, DX, nvec, cvec, inv_rows); break;
    case 1: launch_ring<bn_bwd_apply_ring_kernel<1>, BnRing<1>>(grid, s, DY, X, O, scale, shift, mean, invstd, dgamma, dbeta, DX, nvec, cvec, inv_rows); break;
    case 2: launch_ring<bn_bwd_apply_ring_kernel<2>, BnRing<2>>(grid, s, DY, X, O, scale, shift, mean, invstd, dgamma, dbeta, DX, nvec, cvec, inv_rows); break;
    case 3: launch_ring<bn_bwd_apply_ring_kernel<3>, BnRing<3>>(grid, s, DY, X, O, scale, shift, mean, invstd, dgamma, dbeta, DX, nvec, cvec, inv_rows); break;
    default: throw Error("bad mask_mode");
  }
}

// ------------------------------------------------------------------------------------------------------------
// pooling
// ------------------------------------------------------------------------------------------------------------
// Packed formulation: relu(x * sc + sh) is monotone in x (increasing for sc > 0, decreasing for sc < 0), so the window
// maximum of the activated values is the activation of the window maximum of sign(sc) * x. The nine taps are compared
// as raw bf16 pairs (sign flip = one XOR per pair, compare mask + max + index select: four packed instructions per tap and
// channel pair instead of seven scalar ones per channel), and the batch norm + ReLU are applied once per output. The
// arg-max differs from "first maximum of the activated values" only where the whole window is <= 0 after the ReLU,
// and there the gradient is zero anyway (the ReLU mask of the backward pass removes it).
__device__ __forceinline__ uint32_t bf16x2_gt_mask(uint32_t a, uint32_t b) {   // 0xffff per lane where a > b
  uint32_t m;
  asm("set.gt.u32.bf16x2 %0, %1, %2;" : "=r"(m) : "r"(a), "r"(b));
  return m;
}
__device__ __forceinline__ uint32_t bf16x2_max(uint32_t a, uint32_t b) {
  uint32_t m;
  asm("max.bf16x2 %0, %1, %2;" : "=r"(m) : "r"(a), "r"(b));
  return m;
}
// SHIFT: W / 2, H / 2 and C / 8 are powers of two (every size the bf16 path accepts): the output index is split with
// shifts; otherwise with 32-bit divisions. All nine taps are loaded unconditionally from clamped coordinates (nine
// independent 16-byte loads in flight per thread) and the out-of-bounds ones replaced by -inf afterwards.
template <bool SHIFT>
__global__ void __launch_bounds__(256)
maxpool_fwd_kernel(const uint4* __restrict__ x, const float* __restrict__ scale, const float* __restrict__ shift,
                   uint4* __restrict__ y, uint2* __restrict__ idx, int N, int H, int W, int cvec, int lg_c, int lg_wo,
                   int lg_ho) {
  pdl_prologue();
  const int Ho = H >> 1, Wo = W >> 1;
  const int64_t total = static_cast<int64_t>(N) * Ho * Wo * cvec;
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    int cv, pw, ph, n;
    if (SHIFT) {
      const uint32_t u = static_cast<uint32_t>(i);   // total < 2^32 is checked by the launcher
      cv = u & (cvec - 1);
      pw = (u >> lg_c) & (Wo - 1);
      ph = (u >> (lg_c + lg_wo)) & (Ho - 1);
      n = u >> (lg_c + lg_wo + lg_ho);
    } else {
      cv = static_cast<int>(i % cvec);
      int64_t t = i / cvec;
      pw = static_cast<int>(t % Wo);
      t /= Wo;
      ph = static_cast<int>(t % Ho);
      n = static_cast<int>(t / Ho);
    }
    F8 sc, sh;
    uint32_t flip[4] = {0u, 0u, 0u, 0u};
    if (scale != nullptr) {
      sc = load8f(scale + cv * 8);
      sh = load8f(shift + cv * 8);
#pragma unroll
      for (int j = 0; j < 4; ++j)
        flip[j] = (sc.v[2 * j] < 0.f ? 0x00008000u : 0u) | (sc.v[2 * j + 1] < 0.f ? 0x80000000u : 0u);
    }
    // window rows 2ph-1 .. 2ph+1, columns 2pw-1 .. 2pw+1: only the first row / column can be outside (H, W even)
    const bool top_ok = ph > 0, left_ok = pw > 0;
    const uint4* base = x + (static_cast<int64_t>(n) * H * W) * cvec + cv;
    uint4 tap[3][3];
#pragma unroll
    for (int kh = 0; kh < 3; ++kh) {
      const int h = max(2 * ph - 1 + kh, 0);
#pragma unroll
      for (int kw = 0; kw < 3; ++kw) {
        const int w = max(2 * pw - 1 + kw, 0);
        tap[kh][kw] = __ldg(base + (h * W + w) * cvec);
      }
    }
    uint32_t best[4], bi[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) { best[j] = 0xff80ff80u; bi[j] = 0u; }   // -inf, tap 0
#pragma unroll
    for (int kh = 0; kh < 3; ++kh)
#pragma unroll
      for (int kw = 0; kw < 3; ++kw) {
        const bool ok = (kh > 0 || top_ok) && (kw > 0 || left_ok);
        const uint4 u = tap[kh][kw];
        const uint32_t wv[4] = {ok ? (u.x ^ flip[0]) : 0xff80ff80u, ok ? (u.y ^ flip[1]) : 0xff80ff80u,
                                ok ? (u.z ^ flip[2]) : 0xff80ff80u, ok ? (u.w ^ flip[3]) : 0xff80ff80u};
        const uint32_t code = static_cast<uint32_t>(kh * 3 + kw) * 0x00010001u;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const uint32_t m = bf16x2_gt_mask(wv[j], best[j]);   // strict: the first maximum keeps its index
          best[j] = bf16x2_max(wv[j], best[j]);
          bi[j] = (bi[j] & ~m) | (code & m);
        }
      }
    F8 o = unpack8(make_uint4(best[0] ^ flip[0], best[1] ^ flip[1], best[2] ^ flip[2], best[3] ^ flip[3]));
    if (scale != nullptr) {
#pragma unroll
      for (int k = 0; k < 8; ++k) o.v[k] = fmaxf(fmaf(o.v[k], sc.v[k], sh.v[k]), 0.f);
    }
    y[i] = pack8(o);
    if (idx != nullptr) {
      uint2 p;
      p.x = (bi[0] & 0xffu) | ((bi[0] >> 8) & 0xff00u) | ((bi[1] & 0xffu) << 16) | ((bi[1] >> 16) << 24);
      p.y = (bi[2] & 0xffu) | ((bi[2] >> 8) & 0xff00u) | ((bi[3] & 0xffu) << 16) | ((bi[3] >> 16) << 24);
      idx[i] = p;
    }
  }
}
static int log2_exact(int v) {   // log2 of a power of two, -1 otherwise
  if (v <= 0 || (v & (v - 1))) return -1;
  int l = 0;
  while ((1 << l) < v) ++l;
  return l;
}
void maxpool_fwd(const bf16* x, const float* scale, const float* shift, bf16* y, uint8_t* idx, int N, int H, int W,
                 int C, cudaStream_t s) {
  ProfileScope prof("maxpool", s, 0, static_cast<double>(N) * H * W * C * 2 * 1.25 + (idx ? static_cast<double>(N) * H * W * C / 4 : 0.0));
  const int64_t total = static_cast<int64_t>(N) * (H / 2) * (W / 2) * (C / 8);
  const int lg_c = log2_exact(C / 8), lg_wo = log2_exact(W / 2), lg_ho = log2_exact(H / 2);
  const bool shift_ok = lg_c >= 0 && lg_wo >= 0 && lg_ho >= 0 && total < (1LL << 32) &&
                        static_cast<int64_t>(H) * W * (C / 8) < (1LL << 31);
  if (shift_ok)
    launch_kernel(maxpool_fwd_kernel<true>, grid_for(total, 256), 256, 0, s, reinterpret_cast<const uint4*>(x), scale, shift,
                  reinterpret_cast<uint4*>(y), reinterpret_cast<uint2*>(idx), N, H, W, C / 8, lg_c, lg_wo, lg_ho);
  else
    launch_kernel(maxpool_fwd_kernel<false>, grid_for(total, 256), 256, 0, s, reinterpret_cast<const uint4*>(x), scale, shift,
                  reinterpret_cast<uint4*>(y), reinterpret_cast<uint2*>(idx), N, H, W, C / 8, 0, 0, 0);
  ARGUS_CUDA(cudaGetLastError());
}

__global__ void maxpool_bwd_kernel(const uint4* __restrict__ dy, const uint2* __restrict__ idx, uint4* __restrict__ dx,
                                   int N, int H, int W, int cvec) {
  pdl_prologue();
  const int Ho = H >> 1, Wo = W >> 1;
  const int64_t total = static_cast<int64_t>(N) * H * W * cvec;
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int cv = static_cast<int>(i % cvec);
    int64_t t = i / cvec;
    const int w = static_cast<int>(t % W);
    t /= W;
    const int h = static_cast<int>(t % H);
    const int n = static_cast<int>(t / H);
    F8 g;
#pragma unroll
    for (int k = 0; k < 8; ++k) g.v[k] = 0.f;
    // pooled windows containing (h, w): ph in {h/2, (h+1)/2}, pw likewise
    for (int ph = h >> 1; ph <= ((h + 1) >> 1); ++ph) {
      if (ph >= Ho) continue;
      const int kh = h - (2 * ph - 1);
      for (int pw = w >> 1; pw <= ((w + 1) >> 1); ++pw) {
        if (pw >= Wo) continue;
        const int kw = w - (2 * pw - 1);
        const int code = kh * 3 + kw;
        const int64_t j = ((static_cast<int64_t>(n) * Ho + ph) * Wo + pw) * cvec + cv;
        const uint2 id = __ldg(idx + j);
        const F8 d = unpack8(__ldg(dy + j));
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const int b = (k < 4 ? (id.x >> (8 * k)) : (id.y >> (8 * (k - 4)))) & 0xff;
          if (b == code) g.v[k] += d.v[k];
        }
      }
    }
    dx[i] = pack8(g);
  }
}
void maxpool_bwd(const bf16* dy, const uint8_t* idx, bf16* dx, int N, int H, int W, int C, cudaStream_t s) {
  ProfileScope prof("maxpool", s, 0, static_cast<double>(N) * H * W * C * 2 * 1.25 + static_cast<double>(N) * H * W * C / 4);
  const int64_t total = static_cast<int64_t>(N) * H * W * (C / 8);
  launch_kernel(maxpool_bwd_kernel, grid_for(total, 256), 256, 0, s, reinterpret_cast<const uint4*>(dy),
                                                          reinterpret_cast<const uint2*>(idx),
                                                          reinterpret_cast<uint4*>(dx), N, H, W, C / 8);
  ARGUS_CUDA(cudaGetLastError());
}

// ------------------------------------------------------------------------------------------------------------
// stem: max-pool backward fused into the batch-norm (+ReLU) backward of the stem convolution
// ------------------------------------------------------------------------------------------------------------
// The gradient wrt the stem activation is never materialised: both passes (per-channel sums, then dx) rebuild it from
// the pooled gradient and the arg-max bytes. Thread = one 2x2 patch of stem pixels x 8 channels: the patch touches
// exactly four pooling windows -- (a,b), (a,b+1), (a+1,b), (a+1,b+1) -- so 4 window loads serve 4 pixels (the plain
// max-pool backward kernel needs up to 4 per pixel), and the 1.07 GB intermediate (write + two reads) disappears.
template <int APPLY>
__global__ void __launch_bounds__(256)   // (256, 3) forces 80 registers and spills: measured 0.60 -> 0.83 ms
stem_pool_bn_bwd_kernel(const uint4* __restrict__ dpool, const uint2* __restrict__ idx, const uint4* __restrict__ raw,
                        const float* __restrict__ scale, const float* __restrict__ shift,
                        const float* __restrict__ mean, const float* __restrict__ invstd,
                        const float* __restrict__ dgamma, const float* __restrict__ dbeta, float* __restrict__ partial,
                        uint4* __restrict__ dx, int N, int H, int W, float inv_rows, int lg_wo, int lg_ho) {
  pdl_prologue();
  constexpr int cvec = 8;   // C = 64
  __shared__ float red[16][256];
  const int Ho = H >> 1, Wo = W >> 1;
  const int cv = threadIdx.x & 7;
  const int c0 = cv * 8;
  const F8 sc = load8f(scale + c0), sh = load8f(shift + c0);
  F8 k0, k1;
  if (APPLY) bn_dx_coeffs(sc, mean + c0, invstd + c0, dgamma + c0, dbeta + c0, inv_rows, k0, k1);
  float a_dy[8], a_dyx[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) a_dy[k] = a_dyx[k] = 0.f;
  const int64_t patches = static_cast<int64_t>(N) * Ho * Wo;
  for (int64_t pi = (blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x) >> 3; pi < patches;
       pi += (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 3) {
    int a, b, n;
    if (lg_wo >= 0) {   // Wo, Ho powers of two (every size the bf16 path accepts): shifts instead of 64-bit divisions
      const uint32_t u = static_cast<uint32_t>(pi);
      b = u & (Wo - 1);
      a = (u >> lg_wo) & (Ho - 1);
      n = u >> (lg_wo + lg_ho);
    } else {
      b = static_cast<int>(pi % Wo);
      const int64_t t = pi / Wo;
      a = static_cast<int>(t % Ho);
      n = static_cast<int>(t / Ho);
    }
    // the four windows of this patch: w[dy][dx] = window (a + dy, b + dx)
    F8 wd[2][2];
    uint2 wi[2][2];
#pragma unroll
    for (int dy = 0; dy < 2; ++dy)
#pragma unroll
      for (int dxx = 0; dxx < 2; ++dxx) {
        const bool ok = (a + dy < Ho) && (b + dxx < Wo);
        if (ok) {
          const int64_t j = ((static_cast<int64_t>(n) * Ho + a + dy) * Wo + b + dxx) * cvec + cv;
          wi[dy][dxx] = __ldg(idx + j);
          wd[dy][dxx] = unpack8(__ldg(dpool + j));
        } else {
          wi[dy][dxx] = make_uint2(0xffffffffu, 0xffffffffu);   // code 255 never matches
#pragma unroll
          for (int k = 0; k < 8; ++k) wd[dy][dxx].v[k] = 0.f;
        }
      }
    auto code_of = [](const uint2& id, int k) { return ((k < 4 ? (id.x >> (8 * k)) : (id.y >> (8 * (k - 4)))) & 0xffu); };
#pragma unroll
    for (int py = 0; py < 2; ++py)
#pragma unroll
      for (int px = 0; px < 2; ++px) {
        const int64_t i = ((static_cast<int64_t>(n) * H + 2 * a + py) * W + 2 * b + px) * cvec + cv;
        const F8 xv = unpack8(ldg_stream(raw + i));
        F8 g;
#pragma unroll
        for (int k = 0; k < 8; ++k) g.v[k] = 0.f;
        // windows containing pixel (2a+py, 2b+px): rows {a} (py == 0) or {a, a+1} (py == 1); tap kh = 1 + py - 2*dy
#pragma unroll
        for (int dy = 0; dy <= py; ++dy)
#pragma unroll
          for (int dxx = 0; dxx <= px; ++dxx) {
            const uint32_t code = static_cast<uint32_t>((1 + py - 2 * dy) * 3 + (1 + px - 2 * dxx));
#pragma unroll
            for (int k = 0; k < 8; ++k)
              if (code_of(wi[dy][dxx], k) == code) g.v[k] += wd[dy][dxx].v[k];
          }
        g = bn_masked_grad<1>(g, xv, uint4{}, sc, sh);
        if (APPLY) {
          F8 r;
#pragma unroll
          for (int k = 0; k < 8; ++k) r.v[k] = fmaf(sc.v[k], g.v[k], fmaf(k1.v[k], xv.v[k], k0.v[k]));
          dx[i] = pack8(r);
        } else {
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            a_dy[k] += g.v[k];
            a_dyx[k] = fmaf(g.v[k], xv.v[k], a_dyx[k]);
          }
        }
      }
  }
  if (!APPLY) {
    const F8 mu = load8f(mean + c0), is = load8f(invstd + c0);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      red[k][threadIdx.x] = a_dy[k];
      red[8 + k][threadIdx.x] = (a_dyx[k] - mu.v[k] * a_dy[k]) * is.v[k];
    }
    __syncthreads();
    if (threadIdx.x < 8) {
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        float s0 = 0.f, s1 = 0.f;
        for (int r = 0; r < 32; ++r) {
          s0 += red[k][r * 8 + cv];
          s1 += red[8 + k][r * 8 + cv];
        }
        partial[(static_cast<size_t>(blockIdx.x) * 2 + 0) * 64 + c0 + k] = s0;
        partial[(static_cast<size_t>(blockIdx.x) * 2 + 1) * 64 + c0 + k] = s1;
      }
    }
  }
}

void stem_pool_bn_backward(const bf16* dpool, const uint8_t* idx, const bf16* raw, const float* scale,
                           const float* shift, const float* mean, const float* invstd, float* dgamma, float* dbeta,
                           bf16* dx, int N, int H, int W, int C, float* scratch, cudaStream_t s) {
  ARGUS_CHECK(C == 64, "the fused stem backward is written for 64 channels");
  ARGUS_CHECK(H % 2 == 0 && W % 2 == 0, "stem output must have even height and width");
  ARGUS_CHECK(scratch != nullptr, "stem_pool_bn_backward needs a scratch buffer");
  const int64_t rows = static_cast<int64_t>(N) * H * W;
  const int64_t threads = rows / 4 * 8;
  const float inv_rows = static_cast<float>(1.0 / static_cast<double>(rows));
  int lg_wo = log2_exact(W / 2), lg_ho = log2_exact(H / 2);
  if (lg_wo < 0 || lg_ho < 0 || rows / 4 >= (1LL << 32)) lg_wo = lg_ho = -1;
  auto DP = reinterpret_cast<const uint4*>(dpool);
  auto ID = reinterpret_cast<const uint2*>(idx);
  auto RW = reinterpret_cast<const uint4*>(raw);
  {
    ProfileScope prof("bn_bwd_reduce", s, 0, static_cast<double>(rows) * C * (2.0 + 0.75));
    const int grid = static_cast<int>(std::max<int64_t>(1, std::min<int64_t>((threads + 255) / 256, 4LL * num_sms())));
    launch_kernel(stem_pool_bn_bwd_kernel<0>, grid, 256, 0, s, DP, ID, RW, scale, shift, mean, invstd, nullptr, nullptr, scratch,
                                                    nullptr, N, H, W, inv_rows, lg_wo, lg_ho);
    ARGUS_CUDA(cudaGetLastError());
    launch_kernel(bn_bwd_finalize_kernel, (C + 7) / 8, 256, 0, s, scratch, grid, dgamma, dbeta, C, nullptr, nullptr);
    ARGUS_CUDA(cudaGetLastError());
  }
  {
    ProfileScope prof("bn_bwd_apply", s, 0, static_cast<double>(rows) * C * (4.0 + 0.75));
    const int grid = grid_for(threads, 256);
    launch_kernel(stem_pool_bn_bwd_kernel<1>, grid, 256, 0, s, DP, ID, RW, scale, shift, mean, invstd, dgamma, dbeta, nullptr,
                                                    reinterpret_cast<uint4*>(dx), N, H, W, inv_rows, lg_wo, lg_ho);
    ARGUS_CUDA(cudaGetLastError());
  }
}

__global__ void avgpool_fwd_kernel(const uint4* __restrict__ x, uint4* __restrict__ y, int N, int HW, int cvec) {
  pdl_prologue();
  const int64_t total = static_cast<int64_t>(N) * cvec;
  const float inv = 1.0f / HW;
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int cv = static_cast<int>(i % cvec);
    const int n = static_cast<int>(i / cvec);
    float acc[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) acc[k] = 0.f;
    // eight independent 16-byte loads in flight, added in pixel order (same bits as a plain loop, an eighth of the
    // latency chain: the batch-1 inference forward spent 23 us here)
    const uint4* src = x + static_cast<int64_t>(n) * HW * cvec + cv;
    int p = 0;
    for (; p + 8 <= HW; p += 8) {
      uint4 u[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) u[j] = ldg_stream(src + static_cast<int64_t>(p + j) * cvec);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const F8 v = unpack8(u[j]);
#pragma unroll
        for (int k = 0; k < 8; ++k) acc[k] += v.v[k];
      }
    }
    for (; p < HW; ++p) {
      const F8 v = unpack8(ldg_stream(src + static_cast<int64_t>(p) * cvec));
#pragma unroll
      for (int k = 0; k < 8; ++k) acc[k] += v.v[k];
    }
    F8 o;
#pragma unroll
    for (int k = 0; k < 8; ++k) o.v[k] = acc[k] * inv;
    y[i] = pack8(o);
  }
}
void avgpool_fwd(const bf16* x, bf16* y, int N, int HW, int C, cudaStream_t s) {
  ProfileScope prof("avgpool", s, 0, static_cast<double>(N) * (HW + 1) * C * 2);
  const int64_t total = static_cast<int64_t>(N) * (C / 8);
  launch_kernel(avgpool_fwd_kernel, grid_for(total, 128), 128, 0, s, reinterpret_cast<const uint4*>(x),
                                                          reinterpret_cast<uint4*>(y), N, HW, C / 8);
  ARGUS_CUDA(cudaGetLastError());
}
__global__ void avgpool_bwd_kernel(const uint4* __restrict__ dy, uint4* __restrict__ dx, const uint8_t* __restrict__ bits,
                                   int N, int HW, int cvec) {
  pdl_prologue();
  const int64_t total = static_cast<int64_t>(N) * HW * cvec;
  const float inv = 1.0f / HW;
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int cv = static_cast<int>(i % cvec);
    const int n = static_cast<int>(i / (static_cast<int64_t>(HW) * cvec));
    F8 v = unpack8(__ldg(dy + static_cast<int64_t>(n) * cvec + cv));
    const uint32_t b = bits != nullptr ? bits[i] : 0xffu;
#pragma unroll
    for (int k = 0; k < 8; ++k) v.v[k] = ((b >> k) & 1u) ? v.v[k] * inv : 0.f;
    dx[i] = pack8(v);
  }
}
void avgpool_bwd(const bf16* dy, bf16* dx, const uint8_t* relu_bits, int N, int HW, int C, cudaStream_t s) {
  ProfileScope prof("avgpool", s, 0, static_cast<double>(N) * (HW + 1) * C * 2);
  const int64_t total = static_cast<int64_t>(N) * HW * (C / 8);
  launch_kernel(avgpool_bwd_kernel, grid_for(total, 256), 256, 0, s, reinterpret_cast<const uint4*>(dy),
                                                          reinterpret_cast<uint4*>(dx), relu_bits, N, HW, C / 8);
  ARGUS_CUDA(cudaGetLastError());
}

}  // namespace argus

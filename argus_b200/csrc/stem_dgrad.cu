// Input gradient of the ResNet stem (resnet.conv1: 7x7, stride 2, pad 3, 3 -> 64) on tcgen05, written straight to the
// fp32 NCHW image layout. d loss / d images for callers that train something in front of the network.
//
// In the space-to-depth form of the forward (conv_ops.h, kind 1) the stem is a 4x4 stride-1 convolution over
// x_s2d[r][c][(2a+b)*3 + ch] = x[ch][2r+a][2c+b] with the packed weight Wp[co][p][q][k]. Its transpose is
//   dX_s2d[r][c][k] = sum_{p,q} dY[r+2-p][c+2-q][:] . Wp[:][p][q][k]
// which this kernel evaluates as one GEMM per 128-pixel tile of dY, D[128 px][256] = dY[px][64] * Wp[64][256]
// (N = 16 taps x 16 s2d channels, four M128 N256 K16 MMAs), so dY is read once by TMA and the 32 KB weight stays in
// shared memory. The epilogue adds each pixel's 16 taps into a ring of fp32 dX_s2d rows in shared memory; a row
// leaves the ring as soon as the last dY row that reaches it has been added, as six NCHW rows of dx.
//
// Work item = (image, band of dX rows); a band re-reads the (up to three) dY rows of its halo so that items are
// independent and a persistent grid of one CTA per SM balances them. Warp roles: warp 0 = TMA producer, warp 1 = MMA
// issuer (+ TMEM: two 256-column accumulators, so the epilogue of tile i overlaps the MMAs of tile i + 1),
// warps 2..5 = epilogue (one TMEM lane = one pixel of the tile per thread).
//
// Determinism: the 16 taps are added in a fixed order, one tap column shift q (and, when a tile spans several dY rows,
// one row shift p) per step with a barrier between steps, so no two threads ever update the same ring element in the
// same step and every dx element is a sum in a fixed order. Accumulation and output are fp32 throughout.
#include "conv_ops.h"

#include <algorithm>
#include <cstring>

namespace argus {

namespace {

constexpr int kSdStages = 4;
constexpr int kSdABytes = kBlockM * 128;        // 128 pixels x 64 channels bf16
constexpr int kSdBBytes = 64 * 256 * 2;         // packed stem weight [64][256] bf16
constexpr int kSdRingBytes = 96 * 1024;         // dX_s2d ring: ring_rows x 12 x Ws fp32 (Ws <= 512)
constexpr int kSdOffB = kSdStages * kSdABytes;
constexpr int kSdOffRing = kSdOffB + kSdBBytes;
constexpr int kSdOffBars = kSdOffRing + kSdRingBytes;
constexpr int kSdNumBars = 2 * kSdStages + 2 + 2 + 1;   // full / empty per stage, accumulator full / empty, weights
constexpr int kSdOffTmemPtr = kSdOffBars + kSdNumBars * 8;
constexpr int kSdSmem = kSdOffTmemPtr + 16;   // > half of the SM's shared memory: one CTA per SM (it owns all of TMEM)

struct StemDgradParams {
  CUtensorMap dy_map;   // 2-D [pixels][64] bf16, box (64, 128)
  CUtensorMap w_map;    // 2-D [64][256] bf16, box (64, 64)
  float* dx;            // (N, 3, 2 Hs, 2 Ws) fp32
  int Hs, log2_ws;      // dY grid (= the s2d grid)
  int band_rows;        // dX_s2d rows per work item
  int bands_per_image;
  int num_items;
  int ring_rows;        // power of two >= dY rows per tile + 3
};

struct ItemRange {
  int n, r0, t_lo, t_hi;
};

__device__ __forceinline__ ItemRange decode_item(const StemDgradParams& p, int item) {
  ItemRange it;
  const int Ws = 1 << p.log2_ws;
  it.n = item / p.bands_per_image;
  it.r0 = (item - it.n * p.bands_per_image) * p.band_rows;
  // dX rows [r0, r0 + band_rows) receive from dY rows [r0 - 1, r0 + band_rows + 1]
  const int y_lo = max(0, it.r0 - 1), y_hi = min(p.Hs - 1, it.r0 + p.band_rows + 1);
  it.t_lo = (y_lo * Ws) / kBlockM;
  it.t_hi = ((y_hi + 1) * Ws - 1) / kBlockM;
  return it;
}

__global__ void __launch_bounds__(kWgradThreads, 1) stem_dgrad_kernel(const __grid_constant__ StemDgradParams p) {
  pdl_prologue();
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t smem_base = smem_u32(smem);
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t bar_base = smem_base + kSdOffBars;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (kSdStages + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * kSdStages + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * kSdStages + 2 + a); };
  const uint32_t w_bar = bar_base + 8u * (2 * kSdStages + 4);
  volatile uint32_t* tmem_ptr_smem = reinterpret_cast<volatile uint32_t*>(smem + kSdOffTmemPtr);
  const uint32_t sb = smem_base + kSdOffB;
  const int Ws = 1 << p.log2_ws;
  const int hw = p.Hs << p.log2_ws;

  if (threadIdx.x == 0) {
    if (smem_base & 1023u) __trap();
    for (int s = 0; s < kSdStages; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tfull_bar(a), 1);
      mbar_init(tempty_bar(a), 4);
    }
    mbar_init(w_bar, 1);
    fence_mbar_init();
  }
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.dy_map);
    tma_prefetch_desc(&p.w_map);
  }
  if (warp == 1) {
    tmem_alloc(smem_u32(const_cast<uint32_t*>(tmem_ptr_smem)), 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      mbar_arrive_expect_tx(w_bar, kSdBBytes);
#pragma unroll
      for (int j = 0; j < 4; ++j) tma_load_2d(&p.w_map, w_bar, sb + j * 8192, j * 64, 0);
      int stage = 0;
      uint32_t phase = 0;
      for (int item = blockIdx.x; item < p.num_items; item += gridDim.x) {
        const ItemRange it = decode_item(p, item);
        for (int t = it.t_lo; t <= it.t_hi; ++t) {
          mbar_wait(empty_bar(stage), phase ^ 1);
          mbar_arrive_expect_tx(full_bar(stage), kSdABytes);
          tma_load_2d(&p.dy_map, full_bar(stage), smem_base + stage * kSdABytes, 0, it.n * hw + t * kBlockM);
          if (++stage == kSdStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      // A = dY tile, K-major (64 channels = one 128-byte swizzle row per pixel); B = Wp, N-major [64 k][256 n]
      constexpr uint32_t idesc = make_idesc_bf16(kBlockM, 256, 0, 1);
      mbar_wait(w_bar, 0);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int item = blockIdx.x; item < p.num_items; item += gridDim.x) {
        const ItemRange it = decode_item(p, item);
        for (int t = it.t_lo; t <= it.t_hi; ++t) {
          mbar_wait(tempty_bar(acc), acc_phase ^ 1);
          mbar_wait(full_bar(stage), phase);
          tc_fence_after();
          const uint32_t sa = smem_base + stage * kSdABytes;
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_bf16(tmem_base + acc * 256, make_smem_desc_sw128(sa + k * 32, 0, 1024),
                      make_smem_desc_sw128(sb + k * 2048, 8192, 1024), idesc, k != 0);
          umma_commit(empty_bar(stage));
          umma_commit(tfull_bar(acc));
          if (++stage == kSdStages) { stage = 0; phase ^= 1; }
          if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
      }
    }
  } else {
    // ===================== epilogue (warps 2..5) =====================
    const int wq = warp & 3;                // TMEM lane quarter this warp may access
    const int et = (warp - 2) * 32 + lane;  // 0..127
    const int m_local = wq * 32 + lane;     // pixel of the tile owned by this thread
    float* ring = reinterpret_cast<float*>(smem + kSdOffRing);
    const int row_elems = 12 * Ws;          // one dX_s2d row: [k 0..11][c 0..Ws) (k 12..15 are padding)
    const int H = 2 * p.Hs, W = 2 * Ws;
    // several dY rows per tile: two row shifts p of one column shift q can reach the same element from two threads
    const bool multi_row = Ws < kBlockM;
    for (int i = et; i < p.ring_rows * row_elems; i += 128) ring[i] = 0.f;
    named_bar_sync(1, 128);
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int item = blockIdx.x; item < p.num_items; item += gridDim.x) {
      const ItemRange it = decode_item(p, item);
      const int r1 = it.r0 + p.band_rows;
      int next_flush = it.r0;
      for (int t = it.t_lo; t <= it.t_hi; ++t) {
        mbar_wait(tfull_bar(acc), acc_phase);
        tc_fence_after();
        const int pix = t * kBlockM + m_local;
        const int y = pix >> p.log2_ws, x = pix & (Ws - 1);
#pragma unroll 1
        for (int q = 0; q < 4; ++q) {
          uint32_t v[4][16];
#pragma unroll
          for (int pp = 0; pp < 4; ++pp)
            tmem_ld_32x16(tmem_base + (static_cast<uint32_t>(wq * 32) << 16) + acc * 256 + (pp * 4 + q) * 16, v[pp]);
          tmem_ld_wait();
          if (q == 3) {
            // every TMEM read of this accumulator is done: hand it back to the MMA warp
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty_bar(acc));
          }
          const int c = x + q - 2;
          bool ok[4];
          float* dst[4];
#pragma unroll
          for (int pp = 0; pp < 4; ++pp) {
            const int r = y + pp - 2;
            ok[pp] = c >= 0 && c < Ws && r >= it.r0 && r < r1;
            dst[pp] = ring + (r & (p.ring_rows - 1)) * row_elems + c;
          }
          if (!multi_row) {
            // the four row shifts hit four different rows: all 48 loads are issued before the first store (the compiler
            // cannot see that the rows differ, and a load-add-store chain per element is bound by shared-memory latency)
            float a[4][12];
#pragma unroll
            for (int pp = 0; pp < 4; ++pp)
#pragma unroll
              for (int k = 0; k < 12; ++k) a[pp][k] = ok[pp] ? dst[pp][k * Ws] : 0.f;
#pragma unroll
            for (int pp = 0; pp < 4; ++pp)
              if (ok[pp]) {
#pragma unroll
                for (int k = 0; k < 12; ++k) dst[pp][k * Ws] = a[pp][k] + __uint_as_float(v[pp][k]);
              }
            named_bar_sync(1, 128);
          } else {
#pragma unroll
            for (int pp = 0; pp < 4; ++pp) {
              if (ok[pp]) {
                float a[12];
#pragma unroll
                for (int k = 0; k < 12; ++k) a[k] = dst[pp][k * Ws];
#pragma unroll
                for (int k = 0; k < 12; ++k) dst[pp][k * Ws] = a[k] + __uint_as_float(v[pp][k]);
              }
              named_bar_sync(1, 128);
            }
          }
        }
        // dX rows whose last contributing dY row (r + 2) has been added leave the ring as NCHW fp32 rows
        const int y_done = (((t + 1) * kBlockM) >> p.log2_ws) - 1;
        const int last = (t == it.t_hi) ? r1 - 1 : min(y_done - 2, r1 - 1);
        if (last >= next_flush) {
          for (int r = next_flush; r <= last; ++r) {
            float* row = ring + (r & (p.ring_rows - 1)) * row_elems;
            // six image rows (channel ch, row parity a); the two column parities b of s2d column cc are adjacent
            for (int i = et; i < 6 * Ws; i += 128) {
              const int cc = i & (Ws - 1), ra = i >> p.log2_ws;
              const int ch = ra >> 1, a = ra & 1;
              float* e0 = row + ((2 * a) * 3 + ch) * Ws + cc;
              float* e1 = row + ((2 * a + 1) * 3 + ch) * Ws + cc;
              const float2 o = make_float2(*e0, *e1);
              *e0 = 0.f;
              *e1 = 0.f;
              __stcs(reinterpret_cast<float2*>(p.dx + ((static_cast<size_t>(it.n) * 3 + ch) * H + 2 * r + a) * W + 2 * cc), o);
            }
          }
          next_flush = last + 1;
          named_bar_sync(1, 128);
        }
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

}  // namespace

void stem_dgrad(const __nv_bfloat16* dy, const __nv_bfloat16* w, float* dx, int N, int H, int W, cudaStream_t stream) {
  ARGUS_CHECK(N > 0, "empty batch");
  ARGUS_CHECK(is_pow2(H) && is_pow2(W) && H >= 32 && W >= 32, "H and W must be powers of two >= 32");
  const int Hs = H / 2, Ws = W / 2;
  const int rows_per_tile = std::max(1, kBlockM / Ws);
  int ring_rows = 4;
  while (ring_rows < rows_per_tile + 3) ring_rows *= 2;
  ARGUS_CHECK(static_cast<int64_t>(ring_rows) * 12 * Ws * 4 <= kSdRingBytes, "stem input gradient: W must be <= 1024");
  StemDgradParams p;
  std::memset(&p, 0, sizeof(p));
  const uint64_t pixels = static_cast<uint64_t>(N) * Hs * Ws;
  {
    const uint64_t dims[2] = {64, pixels};
    const uint64_t str[1] = {128};
    const uint32_t box[2] = {64, static_cast<uint32_t>(kBlockM)};
    p.dy_map = make_tmap_bf16(dy, 2, dims, str, box);
  }
  {
    const uint64_t dims[2] = {256, 64};
    const uint64_t str[1] = {512};
    const uint32_t box[2] = {64, 64};
    p.w_map = make_tmap_bf16(w, 2, dims, str, box);
  }
  p.dx = dx;
  p.Hs = Hs;
  p.log2_ws = ilog2(Ws);
  p.ring_rows = ring_rows;
  // bands of >= 16 rows (the three halo rows cost <= 3/16 more MMAs and L2 reads) until there are >= 4 items per SM
  int band = Hs;
  const int nsm = num_sms();
  while (band > 16 && band / 2 >= rows_per_tile && static_cast<int64_t>(N) * (Hs / band) < 4LL * nsm) band /= 2;
  p.band_rows = band;
  p.bands_per_image = Hs / band;
  p.num_items = N * p.bands_per_image;
  const double flops = 2.0 * static_cast<double>(pixels) * 64 * 147;
  const double bytes = static_cast<double>(pixels) * 128 + static_cast<double>(N) * 3 * H * W * 4;
  ProfileScope prof("stem_dgrad", stream, flops, bytes);
  static bool configured = false;
  if (!configured) {
    ARGUS_CUDA(cudaFuncSetAttribute(stem_dgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSdSmem));
    configured = true;
  }
  launch_kernel(stem_dgrad_kernel, std::min(p.num_items, nsm), kWgradThreads, kSdSmem, stream, p);
  ARGUS_CUDA(cudaGetLastError());
}

}  // namespace argus

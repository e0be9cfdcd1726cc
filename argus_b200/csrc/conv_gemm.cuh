// Implicit-GEMM convolution / linear kernels on tcgen05 tensor cores (sm_100a), fed by TMA.
//
//   conv_gemm_kernel<BLOCK_N, B_MN>  : D[pixels, Cout] = sum_taps A_tap[pixels, Cin] * W_tap          (forward, B_MN=0)
//                                      dX[pixels, Cin] = sum_taps dY_tap[pixels, Cout] * W_tap^T      (dgrad,   B_MN=1)
//   wgrad_kernel<BLOCK_N>            : dW[Cout, tap, Cin] += sum_pixels dY[p, Cout]^T * A_tap[p, Cin] (split-K, fp32 red)
//
// Layout: activations are NHWC bf16. An M tile is 128 consecutive output pixels (= a (bw, bh, bn) box of the
// (W, H, N) grid because H and W are powers of two), so one 4-D TMA box per filter tap lands a K-major,
// 128B-swizzled [128 x 64] operand tile in shared memory; padding is TMA out-of-bounds zero fill and stride-2
// convolutions read parity-strided tensor maps. Accumulators live in TMEM (double buffered) so the epilogue of
// tile i overlaps the main loop of tile i+1. Warp roles: warp 0 = TMA producer, warp 1 = MMA issuer (+TMEM
// alloc), warps 2..9 = two epilogue groups, one per accumulator stage (TMEM -> registers -> swizzled smem -> TMA
// store, BN statistics, fused scale/shift/residual/ReLU; the residual tile is TMA-loaded into the staging buffer).
//
// Reference semantics being replaced: torch.nn.Conv2d / nn.Linear inside torchvision resnet50 as called at
// /root/reference/argus/models.py:84 (cuDNN/cuBLAS in the reference).
#pragma once
#include "ptx.cuh"

namespace argus {

constexpr int kBlockM = 128;
constexpr int kBlockK = 64;  // bf16 elements = 128 bytes = one swizzle atom row
constexpr int kEpiGroups = 2;          // conv kernel: epilogue groups of four warps, one per TMEM accumulator stage
constexpr int kNumThreads = 64 + 128 * kEpiGroups;   // conv kernel: TMA warp, MMA warp, the epilogue groups
constexpr int kWgradThreads = 192;     // wgrad kernel: TMA warp, MMA warp, 4 epilogue warps
constexpr int kMaxTaps = 16;

struct Tap {
  int8_t map;   // which A tensor map (parity plane) this tap reads
  int8_t dh;    // row offset added to the tile's h0
  int8_t dw;    // column offset added to the tile's w0
  int8_t pad_;
  int32_t b_off;  // element offset of this tap inside the weight matrix (K offset for K-major B, N offset for MN-major)
};

struct ConvGemmParams {
  CUtensorMap a_map[4];
  CUtensorMap b_map;
  CUtensorMap out_map;
  CUtensorMap res_map;   // residual tensor, same geometry as out_map (valid when has_res != 0)
  Tap taps[kMaxTaps];
  int num_taps;
  int kblocks_per_tap;
  int num_m_tiles;
  int num_n_tiles;
  int log2_wo;     // output pixel grid: width
  int log2_howo;   // output pixel grid: rows*cols per image
  int m_total;     // number of valid output pixels (rows of D)
  int n_total;     // number of output channels (columns of D)
  // epilogue (all optional)
  const float* scale;            // per output channel multiplier (folded BN)
  const float* shift;            // per output channel offset (folded BN / bias)
  int has_res;                   // add the residual tile (TMA-loaded through res_map) before ReLU
  // Weights resident in shared memory (halo mode only, set by finish_params): when the CTA's N tile never changes and
  // its whole [BLOCK_N x K] weight slab fits next to two halo boxes (layer1 3x3: 72 KB), the slab is loaded once per CTA
  // instead of once per M tile and a halo stage carries the activation box only.
  int b_resident;
  // Halo mode (3x3, stride 1, tile inside one image): instead of nine [128 x 64] activation boxes per 64-channel
  // block (one per tap, each re-read from L2), three boxes of (rows + 2) image rows are loaded -- one per horizontal
  // shift dw -- and the three vertical taps are row offsets into the same shared-memory box. Activation traffic from
  // L2 drops from 9 x 16 KB to 3 x (16 KB + 2 image rows). halo_boff[dw+1][dh+1] = weight offset of the tap.
  int halo;
  int halo_rows;          // image rows per tile (128 / W)
  int halo_row_bytes;     // W * 128
  int halo_stages;
  int32_t halo_boff[3][3];
  CUtensorMap halo_map;   // box {64, W, rows + 2, 1}
  const uint8_t* res_bits;       // optional [m_total][n_total/8] bit mask: residual element counts only where its bit is set
  const float* res_scale;        // optional per-channel affine applied to the residual before the add (the downsample
  const float* res_shift;        // branch's batch norm folded into the block tail): f += res * res_scale + res_shift
  uint8_t* relu_bits_out;        // optional [m_total][n_total/8]: bit = (pre-ReLU value > 0), written next to the output
                                 // (training forward of a fused conv3 + BN + residual + ReLU block tail)
  const uint8_t* out_bits;       // optional [m_total][n_total/8] bit mask applied to the RESULT (after the residual add):
                                 // the dgrad that produces the gradient of a ReLU output stores it already masked
  // K concatenation (1x1 only): after the regular k-blocks, k2_blocks more 64-wide blocks are read from a_map[1]
  // (same pixel grid) against the weight rows that follow: D = [A0 | A1] * [B0 ; B1]. Used by the algebraic
  // batch-norm backward (model.cu), where A1 = the saved activation and B1 a small correction matrix.
  int k2_blocks;
  int relu;
  // Batch-norm backward reduction fused into the dgrad that PRODUCES the gradient of a BN + ReLU output (kOptBnRed):
  // the tile of the layer's saved pre-BN output `bn_raw` (same geometry as the result; TMA-loaded through res_map like
  // a residual) gates the result with the ReLU mask (bn_raw * bn_scale + bn_shift > 0) -- the gradient is stored
  // already masked -- and the statistics slots receive sum(g) and sum(g * raw) of the stored bf16 values instead of
  // sum / sum of squares. bn_bwd_reduce's two passes over the gradient and the saved tensor disappear.
  const __nv_bfloat16* bn_raw;
  const float* bn_scale;
  const float* bn_shift;
  int early_trigger;   // let the next kernel of the stream start its prologue at once (pdl_begin; eval-mode chain only)
  // train-mode BN statistics of the stored bf16 outputs, reduced deterministically: every (CTA, epilogue group)
  // owns slot = 2*blockIdx.x + group of stat_partial[slot][2][n_total] (sum, sum of squares); bn_finalize adds the
  // slots in a fixed order. The caller zeroes the buffer.
  float* stat_partial;
};

// NBUF = staging buffers per epilogue group. Two let the store of chunk i overlap the math of chunk i + 1 (and carry the
// prefetched residual tile); a BLOCK_N = 64 tile has a single chunk, so without a residual one buffer is enough (the
// group's next chunk is a whole tile later) and the 32 KB go to the operand pipeline (a third halo stage on layer1 3x3).
template <int BLOCK_N, int OPT>
constexpr int conv_staging_buffers() { return (BLOCK_N == 64 && !(OPT & 2)) ? 1 : 2; }

template <int BLOCK_N, int NBUF = 2>
struct ConvGemmSmem {
  static constexpr int kABytes = kBlockM * kBlockK * 2;          // 16 KB
  static constexpr int kBBytes = BLOCK_N * kBlockK * 2;          // 8..32 KB
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kStagingBytes = kBlockM * 128;            // one 64-column bf16 chunk of the tile
  static constexpr int kStatsBytes = kEpiGroups * 4 * 2 * BLOCK_N * 4;  // per group, per warp: sum[cols], sqsum[cols]
  // operand pipeline region: everything the 227 KB of shared memory leave after staging, statistics and barriers
  static constexpr int kPipeBytes = (232448 - 1024 - NBUF * kEpiGroups * kStagingBytes - kStatsBytes - 512) / 1024 * 1024;
  static constexpr int kStagesRaw = kPipeBytes / kStageBytes;
  static constexpr int kStages = kStagesRaw > 6 ? 6 : kStagesRaw;
  static constexpr int kOffStaging = kPipeBytes;                 // NBUF staging buffers per epilogue group
  static constexpr int kOffStats = kOffStaging + NBUF * kEpiGroups * kStagingBytes;
  static constexpr int kOffBars = kOffStats + kStatsBytes;
  static constexpr int kMaxStages = 8;               // longest stage ring (halo mode; the streaming ring has kStages)
  // full/empty per stage, accumulator-full and accumulator-empty per TMEM stage, residual x (groups x 2 buffers),
  // resident-weights barrier
  static constexpr int kNumBars = 2 * kMaxStages + kEpiGroups + 2 + 2 * kEpiGroups + 1;
  static constexpr int kOffTmemPtr = kOffBars + kNumBars * 8;
  static constexpr int kTotal = kOffTmemPtr + 16;
};

// Epilogue group g (four warps) finishes the CTA-local tiles g, g + 2, ..., all of which use TMEM accumulator stage g.
// OPT = compile-time mask of the epilogue options a kernel instance can honour (kOptAll = the generic kernel). Options
// outside the mask are compiled out, which removes their per-chunk flag tests (constant-bank loads + dependent branches)
// and most of the instruction-cache footprint of the chunk loop. OPT = 0 ("plain": store the bf16 tile, optional
// statistics) is every training-forward convolution and the conv2 / conv3 dgrads; kOptRes | kOptOutBits is the conv1
// dgrad of a bottleneck (identity-branch gradient added, result masked by the previous block's ReLU bits).
constexpr int kOptAffine = 1;    // scale / shift
constexpr int kOptRes = 2;       // residual tile
constexpr int kOptOutBits = 4;   // bit mask applied to the result
constexpr int kOptRelu = 8;      // ReLU, ReLU bit-mask output
constexpr int kOptResExtra = 16; // bit mask on the residual, residual scale / shift (needs kOptRes)
constexpr int kOptBnRed = 32;    // fused batch-norm backward reduction (needs kOptRes: the raw tile rides the residual path)
constexpr int kOptAll = 31;      // the generic kernel (kOptBnRed only exists in specialised instances)
template <int BLOCK_N, int B_MN, int OPT = kOptAll>
__global__ void __launch_bounds__(kNumThreads, 1)
conv_gemm_kernel(const __grid_constant__ ConvGemmParams p) {
  pdl_begin(p.early_trigger);
  constexpr int NBUF = conv_staging_buffers<BLOCK_N, OPT>();
  static_assert(NBUF == 2 || !(OPT & kOptRes), "the residual prefetch needs two staging buffers");
  using L = ConvGemmSmem<BLOCK_N, NBUF>;
  constexpr int kStages = L::kStages;
  constexpr int kTmemCols = (2 * BLOCK_N) < 32 ? 32 : (2 * BLOCK_N);
  static_assert(BLOCK_N == 64 || BLOCK_N == 128 || BLOCK_N == 256, "BLOCK_N");

  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t smem_base = smem_u32(smem);
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  constexpr int kMaxStages = L::kMaxStages;
  const uint32_t bar_base = smem_base + L::kOffBars;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (kMaxStages + s); };
  // "accumulator full" (single waiter: the epilogue group of that stage) and "accumulator empty" (single waiter: the MMA
  // warp) per TMEM stage
  auto tfull_bar = [&](int s) { return bar_base + 8u * (2 * kMaxStages + s); };
  auto tempty_bar = [&](int s) { return bar_base + 8u * (2 * kMaxStages + kEpiGroups + s); };
  auto res_bar = [&](int g, int b) { return bar_base + 8u * (2 * kMaxStages + kEpiGroups + 2 + 2 * g + b); };
  const uint32_t bres_bar = bar_base + 8u * (2 * kMaxStages + kEpiGroups + 2 + 2 * kEpiGroups);
  volatile uint32_t* tmem_ptr_smem = reinterpret_cast<volatile uint32_t*>(smem + L::kOffTmemPtr);
  float* s_stats_all = reinterpret_cast<float*>(smem + L::kOffStats);
  // pipeline geometry: streaming mode = kStages x (A | B); halo mode = halo_stages x (box | 3 B), or with the weights
  // resident (b_resident, halo mode only) halo_stages x box followed by the weight slab
  const bool resident = (p.b_resident != 0);
  const bool halo = (p.halo != 0);
  const uint32_t halo_a_bytes = static_cast<uint32_t>(p.halo_rows + 2) * p.halo_row_bytes;
  const int nstages = halo ? p.halo_stages : kStages;
  const uint32_t stage_bytes = halo ? halo_a_bytes + (resident ? 0u : 3u * L::kBBytes) : L::kStageBytes;
  const uint32_t bres_base = smem_base + static_cast<uint32_t>(nstages) * stage_bytes;

  if (threadIdx.x == 0) {
    if (smem_base & 1023u) __trap();
    for (int s = 0; s < kMaxStages; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    mbar_init(bres_bar, 1);
    for (int s = 0; s < 2; ++s) mbar_init(tempty_bar(s), 4);  // one arrive per epilogue warp finishing the tile
    for (int g = 0; g < kEpiGroups; ++g) {
      mbar_init(tfull_bar(g), 1);
      mbar_init(res_bar(g, 0), 1);
      mbar_init(res_bar(g, 1), 1);
    }
    fence_mbar_init();
  }
  if (warp == 0 && lane == 0) {
    for (int i = 0; i < 4; ++i) tma_prefetch_desc(&p.a_map[i]);
    if (p.halo) tma_prefetch_desc(&p.halo_map);
    tma_prefetch_desc(&p.b_map);
    tma_prefetch_desc(&p.out_map);
    if (p.has_res) tma_prefetch_desc(&p.res_map);
  }
  if (warp == 1) {
    tmem_alloc(smem_u32(const_cast<uint32_t*>(tmem_ptr_smem)), kTmemCols);
    tmem_relinquish();
  }
  for (int i = threadIdx.x; i < kEpiGroups * 8 * BLOCK_N; i += blockDim.x) s_stats_all[i] = 0.f;
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  pdl_wait_deferred(p.early_trigger);   // everything above touched shared memory, TMEM and the kernel parameters only

  const int num_tiles = p.num_m_tiles * p.num_n_tiles;
  const int num_kblocks = p.num_taps * p.kblocks_per_tap + p.k2_blocks;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      auto load_b = [&](uint32_t bar, uint32_t sb, const Tap& tap, int kb, int n0) {
        if (B_MN == 0) {
          // weights [n_total rows, K]: one box of BLOCK_N rows x 64 k
          tma_load_2d(&p.b_map, bar, sb, tap.b_off + kb * kBlockK, n0);
        } else {
          // weights [K rows, N cols]: BLOCK_N/64 boxes of 64 k-rows x 64 n
#pragma unroll
          for (int j = 0; j < BLOCK_N / 64; ++j)
            tma_load_2d(&p.b_map, bar, sb + j * 8192, tap.b_off + n0 + j * 64, kb * kBlockK);
        }
      };
      if (resident && blockIdx.x < num_tiles) {
        // the N tile of this CTA never changes (gridDim.x is a multiple of num_n_tiles, or one tile per CTA); slab order
        // = consumption order of the halo main loop: (k block, horizontal shift, vertical tap)
        const int n0 = (blockIdx.x % p.num_n_tiles) * BLOCK_N;
        mbar_arrive_expect_tx(bres_bar, static_cast<uint32_t>(num_kblocks) * L::kBBytes);
        for (int kb = 0; kb < p.kblocks_per_tap; ++kb)
          for (int dwi = 0; dwi < 3; ++dwi)
            for (int dhi = 0; dhi < 3; ++dhi) {
              Tap tap{};
              tap.b_off = p.halo_boff[dwi][dhi];
              load_b(bres_bar, bres_base + static_cast<uint32_t>((kb * 3 + dwi) * 3 + dhi) * L::kBBytes, tap, kb, n0);
            }
      }
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        const int m_tile = tile / p.num_n_tiles;
        const int n_tile = tile - m_tile * p.num_n_tiles;
        const int m0 = m_tile * kBlockM;
        const int img0 = m0 >> p.log2_howo;
        const int rem = m0 & ((1 << p.log2_howo) - 1);
        const int h0 = rem >> p.log2_wo;
        const int w0 = rem & ((1 << p.log2_wo) - 1);
        const int n0 = n_tile * BLOCK_N;
        if (halo) {
          for (int kb = 0; kb < p.kblocks_per_tap; ++kb)
            for (int dwi = 0; dwi < 3; ++dwi) {
              mbar_wait(empty_bar(stage), phase ^ 1);
              const uint32_t sa = smem_base + stage * stage_bytes;
              mbar_arrive_expect_tx(full_bar(stage), stage_bytes);
              tma_load_4d(&p.halo_map, full_bar(stage), sa, kb * kBlockK, w0 + dwi - 1, h0 - 1, img0);
              if (!resident) {
#pragma unroll
                for (int dhi = 0; dhi < 3; ++dhi) {
                  Tap tap{};
                  tap.b_off = p.halo_boff[dwi][dhi];
                  load_b(full_bar(stage), sa + halo_a_bytes + dhi * L::kBBytes, tap, kb, n0);
                }
              }
              if (++stage == nstages) { stage = 0; phase ^= 1; }
            }
          continue;
        }
        for (int t = 0; t < p.num_taps; ++t) {
          const Tap tap = p.taps[t];
          for (int kb = 0; kb < p.kblocks_per_tap; ++kb) {
            mbar_wait(empty_bar(stage), phase ^ 1);
            const uint32_t sa = smem_base + stage * stage_bytes;
            mbar_arrive_expect_tx(full_bar(stage), stage_bytes);
            tma_load_4d(&p.a_map[tap.map], full_bar(stage), sa, kb * kBlockK, w0 + tap.dw, h0 + tap.dh, img0);
            load_b(full_bar(stage), sa + L::kABytes, tap, kb, n0);
            if (++stage == nstages) { stage = 0; phase ^= 1; }
          }
        }
        for (int kb = 0; kb < p.k2_blocks; ++kb) {
          // concatenated K segment: activations from a_map[1], weight rows continue after the first segment
          mbar_wait(empty_bar(stage), phase ^ 1);
          const uint32_t sa = smem_base + stage * stage_bytes;
          mbar_arrive_expect_tx(full_bar(stage), stage_bytes);
          tma_load_4d(&p.a_map[1], full_bar(stage), sa, kb * kBlockK, w0, h0, img0);
          Tap tap{};
          load_b(full_bar(stage), sa + L::kABytes, tap, p.num_taps * p.kblocks_per_tap + kb, n0);
          if (++stage == nstages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc_bf16(kBlockM, BLOCK_N, 0, B_MN);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      if (resident && blockIdx.x < num_tiles) mbar_wait(bres_bar, 0);
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        mbar_wait(tempty_bar(acc), acc_phase ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + acc * BLOCK_N;
        if (halo) {
          const int nst = 3 * p.kblocks_per_tap;
          for (int st = 0; st < nst; ++st) {
            mbar_wait(full_bar(stage), phase);
            tc_fence_after();
            const uint32_t sa = smem_base + stage * stage_bytes;
#pragma unroll
            for (int dhi = 0; dhi < 3; ++dhi) {
              const uint32_t a0 = sa + static_cast<uint32_t>(dhi) * p.halo_row_bytes;   // multiple of 1024 (W >= 8)
              const uint32_t sb = resident ? bres_base + static_cast<uint32_t>(st * 3 + dhi) * L::kBBytes
                                           : sa + halo_a_bytes + dhi * L::kBBytes;
#pragma unroll
              for (int k = 0; k < kBlockK / 16; ++k) {
                const uint64_t da = make_smem_desc_sw128(a0 + k * 32, 0, 1024);
                const uint64_t db = (B_MN == 0) ? make_smem_desc_sw128(sb + k * 32, 0, 1024)
                                                : make_smem_desc_sw128(sb + k * 2048, 8192, 1024);
                umma_bf16(tmem_d, da, db, idesc, (st | dhi | k) != 0);
              }
            }
            umma_commit(empty_bar(stage));
            if (st == nst - 1) umma_commit(tfull_bar(acc));
            if (++stage == nstages) { stage = 0; phase ^= 1; }
          }
          if (++acc == 2) { acc = 0; acc_phase ^= 1; }
          continue;
        }
        for (int kb = 0; kb < num_kblocks; ++kb) {
          mbar_wait(full_bar(stage), phase);
          tc_fence_after();
          const uint32_t sa = smem_base + stage * stage_bytes;
          const uint32_t sb = sa + L::kABytes;
#pragma unroll
          for (int k = 0; k < kBlockK / 16; ++k) {
            const uint64_t da = make_smem_desc_sw128(sa + k * 32, 0, 1024);
            const uint64_t db = (B_MN == 0) ? make_smem_desc_sw128(sb + k * 32, 0, 1024)
                                            : make_smem_desc_sw128(sb + k * 2048, 8192, 1024);
            umma_bf16(tmem_d, da, db, idesc, (kb | k) != 0);
          }
          umma_commit(empty_bar(stage));
          if (kb == num_kblocks - 1) umma_commit(tfull_bar(acc));
          if (++stage == nstages) { stage = 0; phase ^= 1; }
        }
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else {
    // ===================== epilogue (warps 2..9: two groups of four warps) =====================
    // Group grp finishes the CTA-local tiles grp, grp + 2, ... (accumulator stage grp), so the two tile epilogues overlap
    // each other and the main loop. Each group has its own staging buffer(s), statistics scratch, named barrier and TMA
    // store queue.
    const int ew = warp - 2;
    const int grp = ew >> 2;
    const int acc = grp;                  // TMEM accumulator stage of every tile this group finishes
    const int wq = warp & 3;              // TMEM lane quarter this warp may access
    const int r = wq * 32 + lane;         // row of the tile owned by this thread
    const int et = (ew & 3) * 32 + lane;  // 0..127 inside the group
    const bool store_leader = (et == 0);
    const uint32_t bar_id = 1 + grp;
    float* s_stats = s_stats_all + grp * 8 * BLOCK_N;          // [warp 0..3][sum | sqsum][BLOCK_N]
    float* s_mine = s_stats + (ew & 3) * 2 * BLOCK_N;          // this warp's private slot: no atomics, fixed order
    uint8_t* stg_base = smem + L::kOffStaging + grp * NBUF * L::kStagingBytes;
    uint32_t res_phase[2] = {0, 0};
    int buf = 0;
    int cur_n = -1;
    const bool do_stats = (p.stat_partial != nullptr);
    // epilogue options, read once (compile-time off when outside OPT)
    const bool has_res = (OPT & kOptRes) ? (p.has_res != 0) : false;
    const float* const ep_scale = (OPT & kOptAffine) ? p.scale : nullptr;
    const float* const ep_shift = (OPT & kOptAffine) ? p.shift : nullptr;
    const float* const ep_res_scale = (OPT & kOptResExtra) ? p.res_scale : nullptr;
    const float* const ep_res_shift = (OPT & kOptResExtra) ? p.res_shift : nullptr;
    const uint8_t* const ep_res_bits = (OPT & kOptResExtra) ? p.res_bits : nullptr;
    const uint8_t* const ep_out_bits = (OPT & kOptOutBits) ? p.out_bits : nullptr;
    uint8_t* const ep_relu_bits_out = (OPT & kOptRelu) ? p.relu_bits_out : nullptr;
    const bool ep_relu = (OPT & kOptRelu) ? (p.relu != 0) : false;
    constexpr bool BNRED = (OPT & kOptBnRed) != 0;
    static_assert(!BNRED || ((OPT & kOptRes) && !(OPT & (kOptResExtra | kOptRelu | kOptOutBits))), "kOptBnRed rides the residual path");
    float* my_partial = do_stats ? p.stat_partial + static_cast<size_t>(kEpiGroups * blockIdx.x + grp) * 2 * p.n_total : nullptr;
    constexpr int kChunks = BLOCK_N / 64;
    // Folded batch norm in the epilogue without statistics -- the fused forward block tail (BN + identity + ReLU + bit
    // mask), its downsample branch (BN only) and every eval-mode convolution (BN [+ identity] [+ ReLU]): scale / shift
    // of the CTA's current N tile live in the group's (otherwise unused) statistics scratch, the affine and the
    // residual add run on packed fp32 pairs. The generic code below re-loaded 2 x 64 floats per chunk with dependent global loads (long-scoreboard
    // stalls on every FMUL / FADD, ncu: profiles/r2_ncu_fused_tail.txt) and spent ~1 000 instructions per 64-column
    // chunk. launch_conv only selects this instance when scale, shift, ReLU and a plain residual are all present and
    // no statistics are requested.
    constexpr bool FAST_TAIL = (OPT & kOptAffine) && !(OPT & ~(kOptAffine | kOptRes | kOptRelu));
    float* s_aff = s_stats;   // [scale BLOCK_N | shift BLOCK_N]
    int cur_aff_n = -1;

    auto flush_stats = [&](int n_tile) {
      named_bar_sync(bar_id, 128);
      for (int c = et; c < 2 * BLOCK_N; c += 128) {
        const int which = c / BLOCK_N, col = c - which * BLOCK_N;
        const int gc = n_tile * BLOCK_N + col;
        float acc_s = 0.f;
#pragma unroll
        for (int w = 0; w < 4; ++w) {
          acc_s += s_stats[w * 2 * BLOCK_N + c];
          s_stats[w * 2 * BLOCK_N + c] = 0.f;
        }
        if (gc < p.n_total) my_partial[which * p.n_total + gc] += acc_s;   // only this thread ever touches this word
      }
      named_bar_sync(bar_id, 128);
    };
    // residual tiles are prefetched one chunk ahead (into the staging buffer the NEXT chunk will use), so their TMA
    // latency overlaps the current chunk's TMEM loads, math and store
    auto issue_residual = [&](int tile, int ch, int b) {
      const int m_tile = tile / p.num_n_tiles;
      const int n_tile = tile - m_tile * p.num_n_tiles;
      const int m0 = m_tile * kBlockM;
      const int img0 = m0 >> p.log2_howo;
      const int rem = m0 & ((1 << p.log2_howo) - 1);
      mbar_arrive_expect_tx(res_bar(grp, b), L::kStagingBytes);
      tma_load_4d(&p.res_map, res_bar(grp, b), smem_u32(stg_base + b * L::kStagingBytes), n_tile * BLOCK_N + ch * 64,
                  rem & ((1 << p.log2_wo) - 1), rem >> p.log2_wo, img0);
    };
    const int first_tile = blockIdx.x + grp * gridDim.x;
    if (has_res && store_leader && first_tile < num_tiles) issue_residual(first_tile, 0, 0);

    uint32_t full_phase = 0;
    for (int tile = first_tile; tile < num_tiles; tile += kEpiGroups * gridDim.x, full_phase ^= 1) {
      const int m_tile = tile / p.num_n_tiles;
      const int n_tile = tile - m_tile * p.num_n_tiles;
      const int m0 = m_tile * kBlockM;
      const int img0 = m0 >> p.log2_howo;
      const int rem = m0 & ((1 << p.log2_howo) - 1);
      const int h0 = rem >> p.log2_wo;
      const int w0 = rem & ((1 << p.log2_wo) - 1);
      const int n0 = n_tile * BLOCK_N;
      if (do_stats && n_tile != cur_n) {
        if (cur_n >= 0) flush_stats(cur_n);
        cur_n = n_tile;
      }
      if (FAST_TAIL && n_tile != cur_aff_n) {
        named_bar_sync(bar_id, 128);   // nobody still reads the previous tile's coefficients
        for (int c = et; c < BLOCK_N; c += 128) {
          const int gc = n0 + c;
          s_aff[c] = gc < p.n_total ? __ldg(ep_scale + gc) : 0.f;
          s_aff[BLOCK_N + c] = gc < p.n_total ? __ldg(ep_shift + gc) : 0.f;
        }
        named_bar_sync(bar_id, 128);
        cur_aff_n = n_tile;
      }

      mbar_wait(tfull_bar(acc), full_phase);
      tc_fence_after();

#pragma unroll 1
      for (int ch = 0; ch < kChunks; ++ch) {
        uint8_t* stg = stg_base + buf * L::kStagingBytes;
        // TMEM loads first: they do not touch shared memory, so their latency overlaps the hand-back of the staging
        // buffer (which, with a single buffer per group, waits for the previous chunk's TMA store to have read it)
        uint32_t v[2][32];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const uint32_t taddr = tmem_base + (static_cast<uint32_t>(wq * 32) << 16) + acc * BLOCK_N + ch * 64 + h * 32;
          tmem_ld_32x32(taddr, v[h]);
        }
        // Residual + statistics: the prefetch below refills the buffer the PREVIOUS chunk was staged in, and the statistics
        // pass of that chunk reads it after the store was issued. The leader may only refill it once every warp of the
        // group has finished that pass -- waiting for the TMA store alone is not enough. (Without this barrier the leader,
        // being one warp among four, could run ahead by the TMEM load and overwrite rows other warps were still summing:
        // a rare, timing-dependent error in the per-channel sums of the conv1 dgrads -- the irreproducible runs DESIGN.md 7
        // reports for prioritised streams and programmatic launches, both of which only change the timing.)
        if (has_res && do_stats) named_bar_sync(bar_id, 128);
        if (store_leader) {
          if (has_res) {
            // the other buffer was handed to a TMA store one chunk ago: once that store has read it, refill it with
            // the residual tile of the next chunk (this buffer's residual is already in flight / landed)
            tma_store_wait_read<0>();
            const bool last_ch = (ch == kChunks - 1);
            const int ntile = last_ch ? tile + kEpiGroups * gridDim.x : tile;
            if (ntile < num_tiles) issue_residual(ntile, last_ch ? 0 : ch + 1, buf ^ 1);
          } else {
            // this buffer was handed to a TMA store two chunks ago (one chunk = one tile ago with a single buffer)
            if (NBUF == 2) tma_store_wait_read<1>();
            else tma_store_wait_read<0>();
          }
        }
        // Buffer hand-back. Without a residual the writers below must not touch the buffer before the leader has seen its
        // last TMA store finish reading. With a residual no barrier is needed here: the chunk is written in place over
        // the residual tile, whose buffer the leader cleared for reuse one chunk ago -- before the barrier that preceded
        // that chunk's store -- so waiting for the leader here (it sits in the store-read wait of the PREVIOUS chunk, ~1 us)
        // only serialised the group: 11 % of all stall samples of the fused block tail (profiles/r2_ncu_fused_tail.txt).
        if (!has_res) named_bar_sync(bar_id, 128);
        // kOptBnRed: the statistics pass below runs column-wise (lane = column pair), after the raw tile in the staging
        // buffer has been overwritten in place by the masked gradient; its raw values are re-read from L2 (the tile
        // was just pulled through it by TMA) with coalesced 128-byte rows, issued here so that they land during the math
        uint32_t rawc[BNRED ? 32 : 1];
        if (BNRED) {
          const uint32_t* rp = reinterpret_cast<const uint32_t*>(p.bn_raw + static_cast<size_t>(m0 + wq * 32) * p.n_total +
                                                                 n0 + ch * 64) + lane;
          const int nrow = p.m_total - (m0 + wq * 32);
#pragma unroll
          for (int rr = 0; rr < 32; ++rr)
            rawc[rr] = (rr < nrow) ? ldg_nc_u32(rp + static_cast<size_t>(rr) * (p.n_total >> 1)) : 0u;
        }
        uint2 obits = make_uint2(0xffffffffu, 0xffffffffu);
        if (ep_out_bits != nullptr && m0 + r < p.m_total)
          obits = __ldg(reinterpret_cast<const uint2*>(ep_out_bits + static_cast<size_t>(m0 + r) * (p.n_total >> 3) +
                                                       ((n0 + ch * 64) >> 3)));
        uint2 rbits = make_uint2(0xffffffffu, 0xffffffffu);
        if (ep_res_bits != nullptr && m0 + r < p.m_total)
          rbits = __ldg(reinterpret_cast<const uint2*>(ep_res_bits + static_cast<size_t>(m0 + r) * (p.n_total >> 3) +
                                                       ((n0 + ch * 64) >> 3)));
        tmem_ld_wait();
        if (ch == kChunks - 1) {
          // all TMEM reads of this accumulator are done: hand it back to the MMA warp
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(tempty_bar(acc));
        }
        if (has_res) {
          mbar_wait(res_bar(grp, buf), res_phase[buf]);
          res_phase[buf] ^= 1;
        }
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int c0 = n0 + ch * 64 + h * 32;
          if constexpr (FAST_TAIL) {
            uint32_t ob = 0;
            const float4* sc4 = reinterpret_cast<const float4*>(s_aff + ch * 64 + h * 32);
            const float4* sh4 = reinterpret_cast<const float4*>(s_aff + BLOCK_N + ch * 64 + h * 32);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const int phys = (h * 4 + q) ^ (r & 7);
              uint4* slot = reinterpret_cast<uint4*>(stg + r * 128 + phys * 16);
              uint4 rv = make_uint4(0u, 0u, 0u, 0u);
              if constexpr ((OPT & kOptRes) != 0) rv = *slot;
              const float4 s0 = sc4[2 * q], s1 = sc4[2 * q + 1], t0 = sh4[2 * q], t1 = sh4[2 * q + 1];
              uint64_t y0 = f32x2_pack(t0.x, t0.y), y1 = f32x2_pack(t0.z, t0.w), y2 = f32x2_pack(t1.x, t1.y), y3 = f32x2_pack(t1.z, t1.w);
              f32x2_fma(y0, f32x2_pack(__uint_as_float(v[h][q * 8 + 0]), __uint_as_float(v[h][q * 8 + 1])), f32x2_pack(s0.x, s0.y));
              f32x2_fma(y1, f32x2_pack(__uint_as_float(v[h][q * 8 + 2]), __uint_as_float(v[h][q * 8 + 3])), f32x2_pack(s0.z, s0.w));
              f32x2_fma(y2, f32x2_pack(__uint_as_float(v[h][q * 8 + 4]), __uint_as_float(v[h][q * 8 + 5])), f32x2_pack(s1.x, s1.y));
              f32x2_fma(y3, f32x2_pack(__uint_as_float(v[h][q * 8 + 6]), __uint_as_float(v[h][q * 8 + 7])), f32x2_pack(s1.z, s1.w));
              if constexpr ((OPT & kOptRes) != 0) {
                f32x2_add(y0, f32x2_from_bf16x2(rv.x));
                f32x2_add(y1, f32x2_from_bf16x2(rv.y));
                f32x2_add(y2, f32x2_from_bf16x2(rv.z));
                f32x2_add(y3, f32x2_from_bf16x2(rv.w));
              }
              const float2 a = f32x2_unpack(y0), b = f32x2_unpack(y1), c = f32x2_unpack(y2), d = f32x2_unpack(y3);
              const float y8[8] = {a.x, a.y, b.x, b.y, c.x, c.y, d.x, d.y};
              if constexpr ((OPT & kOptRelu) != 0) {
#pragma unroll
                for (int j = 0; j < 8; ++j) ob |= (y8[j] > 0.f ? 1u : 0u) << (q * 8 + j);
              }
              const float floor_ = ep_relu ? 0.f : -INFINITY;   // (ReLU is a run-time flag of the kOptRelu instances)
              uint4 o;
              o.x = pack_bf16x2(fmaxf(y8[0], floor_), fmaxf(y8[1], floor_));
              o.y = pack_bf16x2(fmaxf(y8[2], floor_), fmaxf(y8[3], floor_));
              o.z = pack_bf16x2(fmaxf(y8[4], floor_), fmaxf(y8[5], floor_));
              o.w = pack_bf16x2(fmaxf(y8[6], floor_), fmaxf(y8[7], floor_));
              *slot = o;
            }
            if constexpr ((OPT & kOptRelu) != 0) {
              if (ep_relu_bits_out != nullptr && m0 + r < p.m_total)
                *reinterpret_cast<uint32_t*>(ep_relu_bits_out + static_cast<size_t>(m0 + r) * (p.n_total >> 3) + (c0 >> 3)) = ob;
            }
          } else {
          float f[32];
#pragma unroll
          for (int i = 0; i < 32; ++i) f[i] = __uint_as_float(v[h][i]);
          if (ep_scale != nullptr) {
#pragma unroll
            for (int i = 0; i < 32; i += 4) {
              const float4 sc = __ldg(reinterpret_cast<const float4*>(ep_scale + c0 + i));
              f[i] *= sc.x; f[i + 1] *= sc.y; f[i + 2] *= sc.z; f[i + 3] *= sc.w;
            }
          }
          if (ep_shift != nullptr) {
#pragma unroll
            for (int i = 0; i < 32; i += 4) {
              const float4 sh = __ldg(reinterpret_cast<const float4*>(ep_shift + c0 + i));
              f[i] += sh.x; f[i + 1] += sh.y; f[i + 2] += sh.z; f[i + 3] += sh.w;
            }
          }
          if (BNRED) {
            // ReLU mask of the layer this gradient flows into, recomputed from its saved pre-BN output exactly as the
            // forward bn_apply evaluated it; rows past the end of the tensor contribute nothing
            const bool row_ok = (m0 + r < p.m_total);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const int phys = (h * 4 + q) ^ (r & 7);
              const uint4 rv = *reinterpret_cast<const uint4*>(stg + r * 128 + phys * 16);
              const float2 a = unpack_bf16x2(rv.x), b = unpack_bf16x2(rv.y), c = unpack_bf16x2(rv.z), d = unpack_bf16x2(rv.w);
              const float rr8[8] = {a.x, a.y, b.x, b.y, c.x, c.y, d.x, d.y};
              const float4 s0 = __ldg(reinterpret_cast<const float4*>(p.bn_scale + c0 + q * 8));
              const float4 s1 = __ldg(reinterpret_cast<const float4*>(p.bn_scale + c0 + q * 8 + 4));
              const float4 t0 = __ldg(reinterpret_cast<const float4*>(p.bn_shift + c0 + q * 8));
              const float4 t1 = __ldg(reinterpret_cast<const float4*>(p.bn_shift + c0 + q * 8 + 4));
              const float sc8[8] = {s0.x, s0.y, s0.z, s0.w, s1.x, s1.y, s1.z, s1.w};
              const float sh8[8] = {t0.x, t0.y, t0.z, t0.w, t1.x, t1.y, t1.z, t1.w};
#pragma unroll
              for (int j = 0; j < 8; ++j)
                f[q * 8 + j] = (row_ok && fmaf(rr8[j], sc8[j], sh8[j]) > 0.f) ? f[q * 8 + j] : 0.f;
            }
          } else if (has_res) {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const int phys = (h * 4 + q) ^ (r & 7);
              uint4 rv = *reinterpret_cast<const uint4*>(stg + r * 128 + phys * 16);
              if (ep_res_bits != nullptr) {
                // ReLU bit mask of these eight channels: spread each bit over a bf16 lane
                const uint32_t mb = ((h == 0 ? rbits.x : rbits.y) >> (8 * q)) & 0xffu;
                rv.x &= ((mb & 1u) ? 0x0000ffffu : 0u) | ((mb & 2u) ? 0xffff0000u : 0u);
                rv.y &= ((mb & 4u) ? 0x0000ffffu : 0u) | ((mb & 8u) ? 0xffff0000u : 0u);
                rv.z &= ((mb & 16u) ? 0x0000ffffu : 0u) | ((mb & 32u) ? 0xffff0000u : 0u);
                rv.w &= ((mb & 64u) ? 0x0000ffffu : 0u) | ((mb & 128u) ? 0xffff0000u : 0u);
              }
              float2 a = unpack_bf16x2(rv.x), b = unpack_bf16x2(rv.y), c = unpack_bf16x2(rv.z), d = unpack_bf16x2(rv.w);
              float rr8[8] = {a.x, a.y, b.x, b.y, c.x, c.y, d.x, d.y};
              if (ep_res_scale != nullptr) {
                const float4 s0 = __ldg(reinterpret_cast<const float4*>(ep_res_scale + c0 + q * 8));
                const float4 s1 = __ldg(reinterpret_cast<const float4*>(ep_res_scale + c0 + q * 8 + 4));
                const float4 t0 = __ldg(reinterpret_cast<const float4*>(ep_res_shift + c0 + q * 8));
                const float4 t1 = __ldg(reinterpret_cast<const float4*>(ep_res_shift + c0 + q * 8 + 4));
                rr8[0] = fmaf(rr8[0], s0.x, t0.x); rr8[1] = fmaf(rr8[1], s0.y, t0.y);
                rr8[2] = fmaf(rr8[2], s0.z, t0.z); rr8[3] = fmaf(rr8[3], s0.w, t0.w);
                rr8[4] = fmaf(rr8[4], s1.x, t1.x); rr8[5] = fmaf(rr8[5], s1.y, t1.y);
                rr8[6] = fmaf(rr8[6], s1.z, t1.z); rr8[7] = fmaf(rr8[7], s1.w, t1.w);
              }
#pragma unroll
              for (int j = 0; j < 8; ++j) f[q * 8 + j] += rr8[j];
            }
          }
          if (ep_relu_bits_out != nullptr) {
            uint32_t ob = 0;
#pragma unroll
            for (int i = 0; i < 32; ++i) ob |= (f[i] > 0.f ? 1u : 0u) << i;
            if (m0 + r < p.m_total)
              *reinterpret_cast<uint32_t*>(ep_relu_bits_out + static_cast<size_t>(m0 + r) * (p.n_total >> 3) +
                                           ((n0 + ch * 64 + h * 32) >> 3)) = ob;
          }
          if (ep_relu) {
#pragma unroll
            for (int i = 0; i < 32; ++i) f[i] = fmaxf(f[i], 0.f);
          }
          if (ep_out_bits != nullptr) {
            const uint32_t ob = (h == 0 ? obits.x : obits.y);
#pragma unroll
            for (int i = 0; i < 32; ++i) f[i] = ((ob >> i) & 1u) ? f[i] : 0.f;
          }
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            uint4 o;
            o.x = pack_bf16x2(f[q * 8 + 0], f[q * 8 + 1]);
            o.y = pack_bf16x2(f[q * 8 + 2], f[q * 8 + 3]);
            o.z = pack_bf16x2(f[q * 8 + 4], f[q * 8 + 5]);
            o.w = pack_bf16x2(f[q * 8 + 6], f[q * 8 + 7]);
            const int phys = (h * 4 + q) ^ (r & 7);      // SWIZZLE_128B position of logical 16-byte chunk h*4+q
            *reinterpret_cast<uint4*>(stg + r * 128 + phys * 16) = o;
          }
          }   // generic epilogue math
        }
        fence_proxy_async_smem();
        named_bar_sync(bar_id, 128);
        if (store_leader) {
          tma_store_4d(&p.out_map, smem_u32(stg), n0 + ch * 64, w0, h0, img0);
          tma_store_commit();
        }
        if (do_stats) {
          // column pair `lane` of the 32 rows owned by this warp; swizzled reads are bank-conflict free. Fully unrolled
          // (eight XOR-swizzled base addresses + immediates), packed FADD2 / FFMA2 on the two columns, two independent
          // accumulator chains (even / odd rows) added in a fixed order: 5 issue slots per row instead of 9.
          uint64_t sa = 0ull, sb = 0ull, qa = 0ull, qb = 0ull;
          const uint32_t jl = static_cast<uint32_t>(lane) >> 2;
          const uint32_t sbase = smem_u32(stg) + static_cast<uint32_t>(wq) * 4096u + ((static_cast<uint32_t>(lane) & 3u) << 2);
#pragma unroll
          for (int rr = 0; rr < 32; rr += 2) {
            const uint64_t x0 = f32x2_from_bf16x2(lds_u32(sbase + rr * 128 + ((jl ^ (rr & 7)) << 4)));
            const uint64_t x1 = f32x2_from_bf16x2(lds_u32(sbase + (rr + 1) * 128 + ((jl ^ ((rr + 1) & 7)) << 4)));
            f32x2_add(sa, x0);
            f32x2_add(sb, x1);
            if (BNRED) {
              f32x2_fma(qa, x0, f32x2_from_bf16x2(rawc[rr]));       // sum g * raw (centred by the finalize kernel)
              f32x2_fma(qb, x1, f32x2_from_bf16x2(rawc[rr + 1]));
            } else {
              f32x2_fma_sq(qa, x0);
              f32x2_fma_sq(qb, x1);
            }
          }
          f32x2_add(sa, sb);
          f32x2_add(qa, qb);
          const float2 s2 = f32x2_unpack(sa), q2 = f32x2_unpack(qa);
          const int c = ch * 64 + lane * 2;
          s_mine[c] += s2.x;
          s_mine[c + 1] += s2.y;
          s_mine[BLOCK_N + c] += q2.x;
          s_mine[BLOCK_N + c + 1] += q2.y;
        }
        if (NBUF == 2) buf ^= 1;
      }
    }
    if (do_stats && cur_n >= 0) flush_stats(cur_n);
    if (store_leader) tma_store_wait_all<0>();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

// ---------------------------------------------------------------------------------------------------------
// Weight gradient: dW[co, tap, ci] += sum over a K-chunk of pixels of dY[p, co] * A_tap[p, ci].
// Both operands are MN-major in shared memory (pixels are the GEMM K dimension and the slow memory dimension).
// Work item = (co tile of 128, ci tile of BLOCK_N, tap, K split); results are reduced into fp32 with red.add.
// ---------------------------------------------------------------------------------------------------------
struct WgradParams {
  CUtensorMap dy_map;     // 2-D [pixels, Cout], box (64 co, 64 pixels)
  // Stacked M operand: output rows >= co_split (a multiple of 128, 0 = off) are read from the activation tensor x
  // itself (through a_map, channel = row - co_split), so one launch yields [dy | x]^T x: the weight gradient with the
  // Gram matrix x^T x appended (algebraic batch-norm backward, bn_algebra.cu). Works for strided x maps too.
  int co_split;
  int stacked;            // 0: every row from dy_map; 1: rows >= co_split from x (co_split may be 0: pure Gram matrix)
  CUtensorMap a_map[4];   // 4-D activation maps (C, W, H, N) by parity, box (64 ci, 64-pixel box)
  Tap taps[kMaxTaps];     // b_off = element offset of the tap inside one dW row
  int num_taps;
  int num_co_tiles;       // ceil(Cout / 128)
  int num_ci_tiles;       // ceil(Cin / BLOCK_N)
  int num_ksplits;
  int kblocks_total;      // ceil(pixels / 64)
  int log2_wo, log2_howo; // pixel grid of dY
  int cout, cin;
  int dw_row_stride;      // elements between consecutive co rows of dW
  float* dw;
  // split-K partial sums, reduced in a fixed order by wgrad_reduce (deterministic): partial[ks][cout][dw_row_stride].
  // Used when num_ksplits > 1; with a single split the tile is added straight into dw.
  float* partial;
  long long partial_stride;
};

template <int BLOCK_N>
struct WgradSmem {
  static constexpr int kABytes = 2 * 8192;                 // 128 co x 64 pixels
  static constexpr int kBBytes = (BLOCK_N / 64) * 8192;    // BLOCK_N ci x 64 pixels
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kStagesRaw = 196608 / kStageBytes;
  static constexpr int kStages = kStagesRaw > 8 ? 8 : kStagesRaw;
  static constexpr int kOffBars = kStages * kStageBytes;
  static constexpr int kNumBars = 2 * kStages + 4;
  static constexpr int kOffTmemPtr = kOffBars + kNumBars * 8;
  static constexpr int kTotal = kOffTmemPtr + 16;
};

template <int BLOCK_N>
__global__ void __launch_bounds__(kWgradThreads, 1)
wgrad_kernel(const __grid_constant__ WgradParams p) {
  pdl_prologue();
  using L = WgradSmem<BLOCK_N>;
  constexpr int kStages = L::kStages;
  constexpr int kTmemCols = 2 * BLOCK_N;

  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t smem_base = smem_u32(smem);
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t bar_base = smem_base + L::kOffBars;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (kStages + s); };
  auto tfull_bar = [&](int s) { return bar_base + 8u * (2 * kStages + s); };
  auto tempty_bar = [&](int s) { return bar_base + 8u * (2 * kStages + 2 + s); };
  volatile uint32_t* tmem_ptr_smem = reinterpret_cast<volatile uint32_t*>(smem + L::kOffTmemPtr);

  if (threadIdx.x == 0) {
    if (smem_base & 1023u) __trap();
    for (int s = 0; s < kStages; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(tfull_bar(s), 1);
      mbar_init(tempty_bar(s), 4);
    }
    fence_mbar_init();
  }
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.dy_map);
    for (int i = 0; i < 4; ++i) tma_prefetch_desc(&p.a_map[i]);
  }
  if (warp == 1) {
    tmem_alloc(smem_u32(const_cast<uint32_t*>(tmem_ptr_smem)), kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  // work item order: ksplit fastest so that concurrently running CTAs share the same weight tile's operands in L2
  const int items_per_tap = p.num_co_tiles * p.num_ci_tiles * p.num_ksplits;
  const int num_items = items_per_tap * p.num_taps;
  const int kb_per_split = (p.kblocks_total + p.num_ksplits - 1) / p.num_ksplits;

  auto decode = [&](int item, int& tap, int& co_t, int& ci_t, int& kb0, int& kb1) {
    int ks = item % p.num_ksplits;
    int rest = item / p.num_ksplits;
    tap = rest % p.num_taps;
    rest /= p.num_taps;
    ci_t = rest % p.num_ci_tiles;
    co_t = rest / p.num_ci_tiles;
    kb0 = ks * kb_per_split;
    kb1 = min(kb0 + kb_per_split, p.kblocks_total);
  };

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int item = blockIdx.x; item < num_items; item += gridDim.x) {
        int t, co_t, ci_t, kb0, kb1;
        decode(item, t, co_t, ci_t, kb0, kb1);
        const Tap tap = p.taps[t];
        for (int kb = kb0; kb < kb1; ++kb) {
          const int p0 = kb * 64;
          const int img0 = p0 >> p.log2_howo;
          const int rem = p0 & ((1 << p.log2_howo) - 1);
          const int h0 = rem >> p.log2_wo;
          const int w0 = rem & ((1 << p.log2_wo) - 1);
          mbar_wait(empty_bar(stage), phase ^ 1);
          const uint32_t sa = smem_base + stage * L::kStageBytes;
          const uint32_t sb = sa + L::kABytes;
          mbar_arrive_expect_tx(full_bar(stage), L::kStageBytes);
          if (p.stacked && co_t * 128 >= p.co_split) {
            const int c0 = co_t * 128 - p.co_split;
            tma_load_4d(&p.a_map[tap.map], full_bar(stage), sa, c0, w0 + tap.dw, h0 + tap.dh, img0);
            tma_load_4d(&p.a_map[tap.map], full_bar(stage), sa + 8192, c0 + 64, w0 + tap.dw, h0 + tap.dh, img0);
          } else {
            tma_load_2d(&p.dy_map, full_bar(stage), sa, co_t * 128, p0);
            tma_load_2d(&p.dy_map, full_bar(stage), sa + 8192, co_t * 128 + 64, p0);
          }
#pragma unroll
          for (int j = 0; j < BLOCK_N / 64; ++j)
            tma_load_4d(&p.a_map[tap.map], full_bar(stage), sb + j * 8192, ci_t * BLOCK_N + j * 64, w0 + tap.dw,
                        h0 + tap.dh, img0);
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc_bf16(128, BLOCK_N, 1, 1);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int item = blockIdx.x; item < num_items; item += gridDim.x) {
        int t, co_t, ci_t, kb0, kb1;
        decode(item, t, co_t, ci_t, kb0, kb1);
        mbar_wait(tempty_bar(acc), acc_phase ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + acc * BLOCK_N;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(full_bar(stage), phase);
          tc_fence_after();
          const uint32_t sa = smem_base + stage * L::kStageBytes;
          const uint32_t sb = sa + L::kABytes;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const uint64_t da = make_smem_desc_sw128(sa + k * 2048, 8192, 1024);
            const uint64_t db = make_smem_desc_sw128(sb + k * 2048, 8192, 1024);
            umma_bf16(tmem_d, da, db, idesc, (kb > kb0) || (k != 0));
          }
          umma_commit(empty_bar(stage));
          if (kb == kb1 - 1) umma_commit(tfull_bar(acc));
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
        if (kb1 <= kb0) umma_commit(tfull_bar(acc));  // empty split: nothing accumulated (epilogue skips it)
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else {
    const int wq = warp & 3;
    const int r = wq * 32 + lane;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int item = blockIdx.x; item < num_items; item += gridDim.x) {
      int t, co_t, ci_t, kb0, kb1;
      decode(item, t, co_t, ci_t, kb0, kb1);
      const Tap tap = p.taps[t];
      mbar_wait(tfull_bar(acc), acc_phase);
      tc_fence_after();
      const int co = co_t * 128 + r;
      const bool use_partial = (p.num_ksplits > 1);
      const int ks = item % p.num_ksplits;
      float* base = use_partial ? p.partial + static_cast<size_t>(ks) * p.partial_stride : p.dw;
      float* row = base + static_cast<size_t>(co) * p.dw_row_stride + tap.b_off + ci_t * BLOCK_N;
#pragma unroll 1
      for (int ch = 0; ch < BLOCK_N / 32; ++ch) {
        uint32_t v[32];
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(wq * 32) << 16) + acc * BLOCK_N + ch * 32;
        tmem_ld_32x32(taddr, v);
        tmem_ld_wait();
        if (kb1 > kb0 && co < p.cout) {
#pragma unroll
          for (int i = 0; i < 32; i += 4) {
            const int ci = ci_t * BLOCK_N + ch * 32 + i;
            if (ci + 3 < p.cin) {
              if (use_partial)
                *reinterpret_cast<uint4*>(row + ch * 32 + i) = make_uint4(v[i], v[i + 1], v[i + 2], v[i + 3]);
              else
                red_add_v4(row + ch * 32 + i, v[i], v[i + 1], v[i + 2], v[i + 3]);
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar(acc));
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

// ---------------------------------------------------------------------------------------------------------
// Weight gradient for Cout == 64 layers (stem, layer1): transposed formulation dW^T[ci, co] = X_tap^T * dY.
// The M=128 operand stacks two 64-wide input-channel boxes (two filter taps, or two channel blocks of a 1x1
// convolution), N = 64 output channels, K = pixels. One CTA owns a contiguous pixel range and ALL boxes: the dY
// tile is loaded once per 64 pixels instead of once per tap, no half-empty M tile is issued, and the per-CTA
// result goes to its own slot of the split-K scratch (reduced in order afterwards).
// ---------------------------------------------------------------------------------------------------------
struct XposeBox {
  int8_t map, dh, dw, valid;
  int16_t c_off;     // channel coordinate of the box in the activation tensor
  int16_t out_off;   // column offset inside one dW row
};
struct WgradXposeParams {
  CUtensorMap dy_map;     // 2-D [pixels, 64], box (64 co, 64 pixels)
  CUtensorMap a_map[4];   // 4-D activation maps, box (64 ch, 64-pixel box)
  XposeBox boxes[10];
  int num_splits;         // = gridDim.x
  int kblocks_total;
  int log2_wo, log2_howo;
  int dw_row_stride;
  float* partial;         // [num_splits][64][dw_row_stride]
};

template <int NBOX>   // padded to an even number: 4 (stem) or 10 (3x3, Cin = 64)
struct WgradXposeSmem {
  static constexpr int kStageBytes = 8192 + NBOX * 8192;
  static constexpr int kStagesRaw = 196608 / kStageBytes;
  static constexpr int kStages = kStagesRaw > 6 ? 6 : kStagesRaw;
  static constexpr int kOffBars = kStages * kStageBytes;
  static constexpr int kNumBars = 2 * kStages + 1;
  static constexpr int kOffTmemPtr = kOffBars + kNumBars * 8;
  static constexpr int kTotal = kOffTmemPtr + 16;
};

template <int NBOX>
__global__ void __launch_bounds__(kWgradThreads, 1)
wgrad_xpose_kernel(const __grid_constant__ WgradXposeParams p) {
  pdl_prologue();
  using L = WgradXposeSmem<NBOX>;
  constexpr int kStages = L::kStages;
  constexpr int kPairs = NBOX / 2;
  constexpr int kTmemCols = kPairs * 64 <= 64 ? 64 : (kPairs * 64 <= 128 ? 128 : (kPairs * 64 <= 256 ? 256 : 512));

  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t smem_base = smem_u32(smem);
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t bar_base = smem_base + L::kOffBars;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (kStages + s); };
  const uint32_t done_bar = bar_base + 8u * (2 * kStages);
  volatile uint32_t* tmem_ptr_smem = reinterpret_cast<volatile uint32_t*>(smem + L::kOffTmemPtr);

  // boxes that are never loaded (odd tap count) must read as zeros
  int n_valid = 0;
  for (int b = 0; b < NBOX; ++b) n_valid += p.boxes[b].valid ? 1 : 0;
  for (int s = 0; s < kStages; ++s)
    for (int b = 0; b < NBOX; ++b)
      if (!p.boxes[b].valid) {
        uint4* z = reinterpret_cast<uint4*>(smem + s * L::kStageBytes + 8192 + b * 8192);
        for (int i = threadIdx.x; i < 512; i += kWgradThreads) z[i] = make_uint4(0u, 0u, 0u, 0u);
      }
  fence_proxy_async_smem();

  if (threadIdx.x == 0) {
    if (smem_base & 1023u) __trap();
    for (int s = 0; s < kStages; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    mbar_init(done_bar, 1);
    fence_mbar_init();
  }
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.dy_map);
    for (int i = 0; i < 4; ++i) tma_prefetch_desc(&p.a_map[i]);
  }
  if (warp == 1) {
    tmem_alloc(smem_u32(const_cast<uint32_t*>(tmem_ptr_smem)), kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  const int per = (p.kblocks_total + p.num_splits - 1) / p.num_splits;
  const int kb0 = blockIdx.x * per;
  const int kb1 = min(kb0 + per, p.kblocks_total);

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int kb = kb0; kb < kb1; ++kb) {
        const int p0 = kb * 64;
        const int img0 = p0 >> p.log2_howo;
        const int rem = p0 & ((1 << p.log2_howo) - 1);
        const int h0 = rem >> p.log2_wo;
        const int w0 = rem & ((1 << p.log2_wo) - 1);
        mbar_wait(empty_bar(stage), phase ^ 1);
        const uint32_t sb = smem_base + stage * L::kStageBytes;   // dY tile first, then the boxes
        mbar_arrive_expect_tx(full_bar(stage), 8192u * (1 + n_valid));
        tma_load_2d(&p.dy_map, full_bar(stage), sb, 0, p0);
#pragma unroll
        for (int b = 0; b < NBOX; ++b) {
          const XposeBox bx = p.boxes[b];
          if (bx.valid)
            tma_load_4d(&p.a_map[bx.map], full_bar(stage), sb + 8192 + b * 8192, bx.c_off, w0 + bx.dw, h0 + bx.dh, img0);
        }
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc_bf16(128, 64, 1, 1);
      int stage = 0;
      uint32_t phase = 0;
      for (int kb = kb0; kb < kb1; ++kb) {
        mbar_wait(full_bar(stage), phase);
        tc_fence_after();
        const uint32_t sb = smem_base + stage * L::kStageBytes;
#pragma unroll
        for (int j = 0; j < kPairs; ++j) {
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const uint64_t da = make_smem_desc_sw128(sb + 8192 + j * 16384 + k * 2048, 8192, 1024);
            const uint64_t db = make_smem_desc_sw128(sb + k * 2048, 8192, 1024);
            umma_bf16(tmem_base + j * 64, da, db, idesc, (kb > kb0) || (k != 0));
          }
        }
        umma_commit(empty_bar(stage));
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
      umma_commit(done_bar);
    }
  } else {
    const int wq = warp & 3;
    const int r = wq * 32 + lane;
    mbar_wait(done_bar, 0);
    tc_fence_after();
    float* base = p.partial + static_cast<size_t>(blockIdx.x) * 64 * p.dw_row_stride;
#pragma unroll 1
    for (int j = 0; j < kPairs; ++j) {
      const XposeBox bx = p.boxes[2 * j + (r >> 6)];
      float* col0 = base + bx.out_off + (r & 63);
#pragma unroll 1
      for (int h = 0; h < 2; ++h) {
        uint32_t v[32];
        tmem_ld_32x32(tmem_base + (static_cast<uint32_t>(wq * 32) << 16) + j * 64 + h * 32, v);
        tmem_ld_wait();
        if (bx.valid) {
          if (kb1 > kb0) {
#pragma unroll
            for (int i = 0; i < 32; ++i) col0[static_cast<size_t>(h * 32 + i) * p.dw_row_stride] = __uint_as_float(v[i]);
          } else {
#pragma unroll
            for (int i = 0; i < 32; ++i) col0[static_cast<size_t>(h * 32 + i) * p.dw_row_stride] = 0.f;
          }
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

}  // namespace argus

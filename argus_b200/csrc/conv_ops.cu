#include "conv_ops.h"

#include <algorithm>
#include <array>
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <set>

namespace argus {

// ------------------------------------------------------------------------------------------------
// runtime helpers
// ------------------------------------------------------------------------------------------------
static thread_local std::string g_last_error;
void set_last_error(const std::string& msg) { g_last_error = msg; }
const char* get_last_error() { return g_last_error.c_str(); }

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* sym = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres);
    if (e == cudaSuccess && qres == cudaDriverEntryPointSuccess) fn = reinterpret_cast<EncodeTiledFn>(sym);
  });
  ARGUS_CHECK(fn != nullptr, "cuTensorMapEncodeTiled not available from the CUDA driver");
  return fn;
}

CUtensorMap make_tmap_bf16(const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                           const uint32_t* box) {
  CUtensorMap m;
  std::memset(&m, 0, sizeof(m));
  cuuint64_t gdim[5];
  cuuint64_t gstr[4];
  cuuint32_t bdim[5];
  cuuint32_t estr[5];
  for (int i = 0; i < rank; ++i) {
    gdim[i] = dims[i];
    bdim[i] = box[i];
    estr[i] = 1;
  }
  for (int i = 0; i + 1 < rank; ++i) gstr[i] = strides_bytes[i];
  ARGUS_CHECK((reinterpret_cast<uintptr_t>(base) & 15) == 0, "TMA base address must be 16-byte aligned");
  ARGUS_CHECK(box[0] * 2 == 128, "SWIZZLE_128B boxes are 64 bf16 wide");
  CUresult r = get_encode_fn()(&m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, rank, const_cast<void*>(base), gdim, gstr, bdim,
                               estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                               CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    std::string msg = "cuTensorMapEncodeTiled failed (" + std::to_string(static_cast<int>(r)) + ") rank=" +
                      std::to_string(rank) + " dims=";
    for (int i = 0; i < rank; ++i) msg += std::to_string(dims[i]) + ",";
    msg += " strides=";
    for (int i = 0; i + 1 < rank; ++i) msg += std::to_string(strides_bytes[i]) + ",";
    msg += " box=";
    for (int i = 0; i < rank; ++i) msg += std::to_string(box[i]) + ",";
    throw Error(msg);
  }
  return m;
}

// ------------------------------------------------------------------------------------------------
// launch accounting / profiling
// ------------------------------------------------------------------------------------------------
namespace {
struct ProfRecord {
  std::string family;
  cudaEvent_t start, stop;
  double flops, bytes;
};
std::atomic<int64_t> g_launches{0};
bool g_profiling = false;
std::vector<ProfRecord> g_records;
std::vector<cudaEvent_t> g_event_pool;
cudaEvent_t new_event() {
  if (!g_event_pool.empty()) {
    cudaEvent_t e = g_event_pool.back();
    g_event_pool.pop_back();
    return e;
  }
  cudaEvent_t e;
  ARGUS_CUDA(cudaEventCreate(&e));
  return e;
}
}  // namespace

void profile_enable(bool on) {
  if (on) {
    for (auto& r : g_records) { g_event_pool.push_back(r.start); g_event_pool.push_back(r.stop); }
    g_records.clear();
  }
  g_profiling = on;
}
bool profile_enabled() { return g_profiling; }
int64_t launch_count() { return g_launches.load(); }

ProfileScope::ProfileScope(const char* family, cudaStream_t s, double flops, double bytes) : stream(s) {
  g_launches.fetch_add(1);
  if (!g_profiling) return;
  ProfRecord r{family, new_event(), new_event(), flops, bytes};
  cudaEventRecord(r.start, s);
  pdl_break(s, kPdlAfterRecord);
  slot = static_cast<int>(g_records.size());
  g_records.push_back(r);
}
ProfileScope::ProfileScope(const std::string& family, cudaStream_t s, double flops, double bytes) : stream(s) {
  g_launches.fetch_add(1);
  if (!g_profiling) return;
  ProfRecord r{family, new_event(), new_event(), flops, bytes};
  cudaEventRecord(r.start, s);
  pdl_break(s, kPdlAfterRecord);
  slot = static_cast<int>(g_records.size());
  g_records.push_back(r);
}
bool profile_detailed() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("ARGUS_PROFILE_DETAIL");
    v = (e && e[0] == '1') ? 1 : 0;
  }
  return v == 1;
}
ProfileScope::~ProfileScope() {
  if (slot >= 0) { cudaEventRecord(g_records[slot].stop, stream); pdl_break(stream, kPdlAfterRecord); }
}

std::string profile_report_json() {
  struct Agg { int launches = 0; double ms = 0, flops = 0, bytes = 0; };
  std::map<std::string, Agg> agg;
  std::vector<std::string> order;
  for (auto& r : g_records) {
    cudaEventSynchronize(r.stop);
    float ms = 0.f;
    cudaEventElapsedTime(&ms, r.start, r.stop);
    if (!agg.count(r.family)) order.push_back(r.family);
    Agg& a = agg[r.family];
    a.launches += 1; a.ms += ms; a.flops += r.flops; a.bytes += r.bytes;
  }
  std::string out = "{";
  bool first = true;
  for (auto& name : order) {
    const Agg& a = agg[name];
    char buf[384];
    snprintf(buf, sizeof(buf), "%s\"%s\": {\"launches\": %d, \"ms\": %.6f, \"flops\": %.6e, \"bytes\": %.6e}",
             first ? "" : ", ", name.c_str(), a.launches, a.ms, a.flops, a.bytes);
    out += buf;
    first = false;
  }
  out += "}";
  return out;
}

// Programmatic dependent launch between back-to-back kernels of the library: on by default since round 2 (ARGUS_PDL=0
// disables). Every kernel waits in its prologue (griddepcontrol.wait), nothing triggers early, and any event record /
// wait / memset / memcpy the library enqueues breaks the chain (pdl_break), so the only thing that overlaps is the launch
// latency of a kernel with the tail of its predecessor. Measured on B200: 38.6-38.9 -> 37.7-38.3 ms per step, same bits
// in 8 of 8 bench runs and 29 of 29 in-process trajectories (profiles/r2_determinism.md, section 4).
bool pdl_enabled() {
  static const bool on = [] { const char* e = getenv("ARGUS_PDL"); return !(e && e[0] == '0'); }();
  return on;
}
namespace {
std::mutex g_pdl_mu;
std::vector<std::pair<cudaStream_t, bool>> g_pdl_ok;   // a handful of streams: linear search
}  // namespace
void pdl_break(cudaStream_t stream, int) {
  std::lock_guard<std::mutex> lk(g_pdl_mu);
  for (auto& e : g_pdl_ok)
    if (e.first == stream) e.second = false;
}
void pdl_break_all() {
  std::lock_guard<std::mutex> lk(g_pdl_mu);
  for (auto& e : g_pdl_ok) e.second = false;
}
bool pdl_chain_ok(cudaStream_t stream) {
  std::lock_guard<std::mutex> lk(g_pdl_mu);
  for (auto& e : g_pdl_ok)
    if (e.first == stream) return e.second;
  return false;
}
void pdl_mark_kernel(cudaStream_t stream) {
  std::lock_guard<std::mutex> lk(g_pdl_mu);
  for (auto& e : g_pdl_ok)
    if (e.first == stream) { e.second = true; return; }
  g_pdl_ok.emplace_back(stream, true);
}
int num_sms() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    ARGUS_CUDA(cudaGetDevice(&dev));
    ARGUS_CUDA(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev));
  }
  return n;
}

void require_sm100() {
  int dev = 0, major = 0;
  ARGUS_CUDA(cudaGetDevice(&dev));
  ARGUS_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  ARGUS_CHECK(major == 10, "argus_b200 kernels are built for sm_100a only; no fallback path exists");
}

// ------------------------------------------------------------------------------------------------
// shape handling
// ------------------------------------------------------------------------------------------------
void validate_shape(const ConvShape& s) {
  ARGUS_CHECK(s.N > 0 && s.H > 0 && s.W > 0, "empty convolution input");
  ARGUS_CHECK(is_pow2(s.H) && is_pow2(s.W), "spatial sizes must be powers of two (tiles are linear pixel runs)");
  if (s.kind == 1) {
    ARGUS_CHECK(s.Cout == 64 && s.stride == 2 && s.H >= 2 && s.W >= 2, "stem convolution is 3->64, stride 2");
    return;
  }
  ARGUS_CHECK(s.k == 1 || s.k == 3, "kernel size must be 1 or 3");
  ARGUS_CHECK(s.stride == 1 || s.stride == 2, "stride must be 1 or 2");
  ARGUS_CHECK(s.Cin % 64 == 0 && s.Cout % 64 == 0, "channel counts must be multiples of 64");
  ARGUS_CHECK(s.H % s.stride == 0 && s.W % s.stride == 0, "spatial size must be divisible by the stride");
}

// Largest N tile that still yields at least one tile per SM; small problems (inference at batch 1, layer3/4) fall
// back to narrow tiles so that more CTAs share the work and each K loop issues cheaper MMAs.
static int pick_block_n(int n, int64_t m_tiles = (1 << 30)) {
  const int cands[3] = {256, 128, 64};
  for (int bn : cands)
    if (n >= bn && n % bn == 0 && m_tiles * (n / bn) >= num_sms()) return bn;
  return 64;
}

// box of `pixels` consecutive pixels of an (N, Ho, Wo) grid, as (bw, bh, bn)
static void pixel_box(int Wo, int Ho, int pixels, uint32_t& bw, uint32_t& bh, uint32_t& bn) {
  bw = std::min(Wo, pixels);
  bh = std::min(Ho, pixels / static_cast<int>(bw));
  bn = pixels / (bw * bh);
}

// activation tensor maps for reading the conv INPUT x as seen from the output pixel grid
static void make_input_maps(const ConvShape& s, const __nv_bfloat16* x, int pixels, CUtensorMap* maps) {
  uint32_t bw, bh, bn;
  pixel_box(s.Wo(), s.Ho(), pixels, bw, bh, bn);
  const uint32_t box[4] = {64, bw, bh, bn};
  if (s.kind == 1) {
    const uint64_t Hs = s.H / 2, Ws = s.W / 2, Wp = Ws + 4;
    const uint64_t dims[4] = {64, Ws, Hs, static_cast<uint64_t>(s.N)};
    const uint64_t str[3] = {32, Wp * 32, Hs * Wp * 32};  // overlapping 128-byte windows, 32 bytes apart
    maps[0] = make_tmap_bf16(x, 4, dims, str, box);
    for (int i = 1; i < 4; ++i) maps[i] = maps[0];
    return;
  }
  const uint64_t C = s.Cin, H = s.H, W = s.W;
  if (s.stride == 1) {
    const uint64_t dims[4] = {C, W, H, static_cast<uint64_t>(s.N)};
    const uint64_t str[3] = {C * 2, W * C * 2, H * W * C * 2};
    maps[0] = make_tmap_bf16(x, 4, dims, str, box);
    for (int i = 1; i < 4; ++i) maps[i] = maps[0];
  } else {
    for (int a = 0; a < 2; ++a)
      for (int b = 0; b < 2; ++b) {
        const uint64_t dims[4] = {C, W / 2, H / 2, static_cast<uint64_t>(s.N)};
        const uint64_t str[3] = {2 * C * 2, 2 * W * C * 2, H * W * C * 2};
        maps[a * 2 + b] = make_tmap_bf16(x + (a * W + b) * C, 4, dims, str, box);
      }
  }
}

static int fill_forward_taps(const ConvShape& s, Tap* taps) {
  int n = 0;
  if (s.kind == 1) {
    for (int pi = 0; pi < 4; ++pi) taps[n++] = Tap{0, static_cast<int8_t>(pi - 2), 0, 0, pi * 64};
    return n;
  }
  const int pad = s.k / 2;
  for (int kh = 0; kh < s.k; ++kh)
    for (int kw = 0; kw < s.k; ++kw) {
      Tap t{};
      t.b_off = (kh * s.k + kw) * s.Cin;
      const int eh = kh - pad, ew = kw - pad;
      if (s.stride == 1) {
        t.map = 0;
        t.dh = static_cast<int8_t>(eh);
        t.dw = static_cast<int8_t>(ew);
      } else {
        const int a = eh & 1, b = ew & 1;  // parity plane (two's complement & works for -1)
        t.map = static_cast<int8_t>(a * 2 + b);
        t.dh = static_cast<int8_t>((eh - a) / 2);
        t.dw = static_cast<int8_t>((ew - b) / 2);
      }
      taps[n++] = t;
    }
  return n;
}

// Halo mode (see ConvGemmParams::halo): 3x3 stride-1 convolutions whose 128-pixel tile is `rows` whole image rows.
// `src` is the tensor the A operand is read from (x for forward, dy for dgrad), both on the (N, H, W) grid.
static void setup_halo(ConvGemmParams& p, const ConvShape& s, const __nv_bfloat16* src, int channels, bool dgrad,
                       int block_n) {
  p.halo = 0;
  if (s.kind != 0 || s.k != 3 || s.stride != 1 || block_n > 128) return;
  uint32_t bw, bh, bn;
  pixel_box(s.W, s.H, kBlockM, bw, bh, bn);
  if (bn != 1 || static_cast<int>(bw) != s.W || s.W < 8 || static_cast<int>(bw * bh) != kBlockM) return;
  const uint64_t C = channels, H = s.H, W = s.W;
  const uint64_t dims[4] = {C, W, H, static_cast<uint64_t>(s.N)};
  const uint64_t str[3] = {C * 2, W * C * 2, H * W * C * 2};
  const uint32_t box[4] = {64, bw, bh + 2, 1};
  p.halo_map = make_tmap_bf16(src, 4, dims, str, box);
  p.halo_rows = static_cast<int>(bh);
  p.halo_row_bytes = s.W * 128;
  for (int dwi = 0; dwi < 3; ++dwi)
    for (int dhi = 0; dhi < 3; ++dhi) {
      const int kh = dgrad ? 2 - dhi : dhi, kw = dgrad ? 2 - dwi : dwi;
      p.halo_boff[dwi][dhi] = (kh * 3 + kw) * s.Cin;
    }
  p.halo = 1;
}

ConvLaunch plan_conv_forward(const ConvShape& s, const __nv_bfloat16* x, const __nv_bfloat16* w, __nv_bfloat16* y) {
  validate_shape(s);
  ConvLaunch l;
  std::memset(&l.p, 0, sizeof(l.p));
  l.block_n = pick_block_n(s.Cout, (s.out_pixels() + kBlockM - 1) / kBlockM);
  l.b_mn = 0;
  ConvGemmParams& p = l.p;
  make_input_maps(s, x, kBlockM, p.a_map);
  {
    const uint64_t dims[2] = {static_cast<uint64_t>(s.Ktot()), static_cast<uint64_t>(s.Cout)};
    const uint64_t str[1] = {static_cast<uint64_t>(s.Ktot()) * 2};
    const uint32_t box[2] = {64, static_cast<uint32_t>(l.block_n)};
    p.b_map = make_tmap_bf16(w, 2, dims, str, box);
  }
  {
    uint32_t bw, bh, bn;
    pixel_box(s.Wo(), s.Ho(), kBlockM, bw, bh, bn);
    const uint64_t C = s.Cout, Ho = s.Ho(), Wo = s.Wo();
    const uint64_t dims[4] = {C, Wo, Ho, static_cast<uint64_t>(s.N)};
    const uint64_t str[3] = {C * 2, Wo * C * 2, Ho * Wo * C * 2};
    const uint32_t box[4] = {64, bw, bh, bn};
    p.out_map = make_tmap_bf16(y, 4, dims, str, box);
    l.out_geom.set(4, dims, str, box);
  }
  p.num_taps = fill_forward_taps(s, p.taps);
  p.kblocks_per_tap = (s.kind == 1) ? 1 : s.Cin / 64;
  p.m_total = static_cast<int>(s.out_pixels());
  p.n_total = s.Cout;
  p.num_m_tiles = (p.m_total + kBlockM - 1) / kBlockM;
  p.num_n_tiles = (s.Cout + l.block_n - 1) / l.block_n;
  p.log2_wo = ilog2(s.Wo());
  p.log2_howo = ilog2(s.Ho() * s.Wo());
  setup_halo(p, s, x, s.Cin, false, l.block_n);
  return l;
}

std::vector<ConvLaunch> plan_conv_dgrad(const ConvShape& s, const __nv_bfloat16* dy, const __nv_bfloat16* w,
                                        __nv_bfloat16* dx) {
  validate_shape(s);
  ARGUS_CHECK(s.kind == 0, "the stem has no input gradient");
  std::vector<ConvLaunch> out;
  const int pad = s.k / 2;
  const int Ho = s.Ho(), Wo = s.Wo();
  const int block_n = pick_block_n(s.Cin, (static_cast<int64_t>(s.N) * Ho * Wo + kBlockM - 1) / kBlockM);
  const int classes = (s.stride == 1) ? 1 : 4;
  for (int cls = 0; cls < classes; ++cls) {
    const int a = cls >> 1, b = cls & 1;
    ConvLaunch l;
    std::memset(&l.p, 0, sizeof(l.p));
    l.block_n = block_n;
    l.b_mn = 1;
    ConvGemmParams& p = l.p;
    // taps: which (kh, kw) reach input pixels of this parity class, and from which dy pixel offset
    int n = 0;
    for (int kh = 0; kh < s.k; ++kh)
      for (int kw = 0; kw < s.k; ++kw) {
        Tap t{};
        t.map = 0;
        t.b_off = (kh * s.k + kw) * s.Cin;
        if (s.stride == 1) {
          t.dh = static_cast<int8_t>(pad - kh);
          t.dw = static_cast<int8_t>(pad - kw);
        } else {
          const int eh = a + pad - kh, ew = b + pad - kw;
          if ((eh & 1) || (ew & 1)) continue;
          t.dh = static_cast<int8_t>(eh / 2);
          t.dw = static_cast<int8_t>(ew / 2);
        }
        p.taps[n++] = t;
      }
    if (n == 0) continue;  // this parity class receives no gradient (caller zero-filled dx)
    p.num_taps = n;
    p.kblocks_per_tap = s.Cout / 64;
    // A = dy on the (N, Ho, Wo) grid
    uint32_t bw, bh, bn;
    pixel_box(Wo, Ho, kBlockM, bw, bh, bn);
    {
      const uint64_t C = s.Cout;
      const uint64_t dims[4] = {C, static_cast<uint64_t>(Wo), static_cast<uint64_t>(Ho), static_cast<uint64_t>(s.N)};
      const uint64_t str[3] = {C * 2, Wo * C * 2, static_cast<uint64_t>(Ho) * Wo * C * 2};
      const uint32_t box[4] = {64, bw, bh, bn};
      p.a_map[0] = make_tmap_bf16(dy, 4, dims, str, box);
      for (int i = 1; i < 4; ++i) p.a_map[i] = p.a_map[0];
    }
    {
      // weights [Cout rows][k*k*Cin]: MN-major B operand (K = Cout is the slow dimension)
      const uint64_t dims[2] = {static_cast<uint64_t>(s.Ktot()), static_cast<uint64_t>(s.Cout)};
      const uint64_t str[1] = {static_cast<uint64_t>(s.Ktot()) * 2};
      const uint32_t box[2] = {64, 64};
      p.b_map = make_tmap_bf16(w, 2, dims, str, box);
    }
    {
      const uint64_t C = s.Cin, H = s.H, W = s.W;
      const uint32_t box[4] = {64, bw, bh, bn};
      if (s.stride == 1) {
        const uint64_t dims[4] = {C, W, H, static_cast<uint64_t>(s.N)};
        const uint64_t str[3] = {C * 2, W * C * 2, H * W * C * 2};
        p.out_map = make_tmap_bf16(dx, 4, dims, str, box);
        l.out_geom.set(4, dims, str, box);
      } else {
        const uint64_t dims[4] = {C, W / 2, H / 2, static_cast<uint64_t>(s.N)};
        const uint64_t str[3] = {2 * C * 2, 2 * W * C * 2, H * W * C * 2};
        p.out_map = make_tmap_bf16(dx + (a * W + b) * C, 4, dims, str, box);
      }
    }
    p.m_total = s.N * Ho * Wo;
    p.n_total = s.Cin;
    p.num_m_tiles = (p.m_total + kBlockM - 1) / kBlockM;
    p.num_n_tiles = (s.Cin + block_n - 1) / block_n;
    p.log2_wo = ilog2(Wo);
    p.log2_howo = ilog2(Ho * Wo);
    setup_halo(p, s, dy, s.Cout, true, block_n);
    out.push_back(l);
  }
  return out;
}

ConvLaunch plan_dgrad_concat(const ConvShape& s, const __nv_bfloat16* dy, const __nv_bfloat16* a1, int C1,
                             const __nv_bfloat16* bstack, __nv_bfloat16* dx) {
  validate_shape(s);
  ARGUS_CHECK(s.kind == 0 && s.k == 1, "concatenated dgrad is defined for 1x1 convolutions");
  ARGUS_CHECK(C1 > 0 && C1 % 64 == 0, "second source must have a multiple of 64 channels");
  std::vector<ConvLaunch> ls = plan_conv_dgrad(s, dy, bstack, dx);
  ARGUS_CHECK(ls.size() == 1, "unexpected dgrad decomposition");   // stride 2: only parity class (0,0) has a tap
  ConvLaunch l = ls[0];
  ConvGemmParams& p = l.p;
  const int Ho = s.Ho(), Wo = s.Wo();
  uint32_t bw, bh, bn;
  pixel_box(Wo, Ho, kBlockM, bw, bh, bn);
  {
    // a1 lives on the conv INPUT grid (N, H, W, C1); the GEMM rows are output pixels: stride 2 reads its (0,0) plane
    const uint64_t C = C1, H = s.H, W = s.W, st = s.stride;
    const uint64_t dims[4] = {C, static_cast<uint64_t>(Wo), static_cast<uint64_t>(Ho), static_cast<uint64_t>(s.N)};
    const uint64_t str[3] = {st * C * 2, st * W * C * 2, H * W * C * 2};
    const uint32_t box[4] = {64, bw, bh, bn};
    p.a_map[1] = make_tmap_bf16(a1, 4, dims, str, box);
  }
  {
    const uint64_t dims[2] = {static_cast<uint64_t>(s.Cin), static_cast<uint64_t>(s.Cout + C1)};
    const uint64_t str[1] = {static_cast<uint64_t>(s.Cin) * 2};
    const uint32_t box[2] = {64, 64};
    p.b_map = make_tmap_bf16(bstack, 2, dims, str, box);
  }
  p.k2_blocks = C1 / 64;
  return l;
}

WgradLaunch plan_conv_wgrad(const ConvShape& s, const __nv_bfloat16* dy, const __nv_bfloat16* x, float* dw) {
  validate_shape(s);
  WgradLaunch l;
  std::memset(&l.p, 0, sizeof(l.p));
  WgradParams& p = l.p;
  const int cin_tile_extent = (s.kind == 1) ? 64 : s.Cin;  // stem: each tap is one 64-wide window
  l.block_n = pick_block_n(cin_tile_extent);
  const int64_t pixels = s.out_pixels();
  {
    const uint64_t dims[2] = {static_cast<uint64_t>(s.Cout), static_cast<uint64_t>(pixels)};
    const uint64_t str[1] = {static_cast<uint64_t>(s.Cout) * 2};
    const uint32_t box[2] = {64, 64};
    p.dy_map = make_tmap_bf16(dy, 2, dims, str, box);
  }
  make_input_maps(s, x, 64, p.a_map);
  p.num_taps = fill_forward_taps(s, p.taps);
  p.num_co_tiles = (s.Cout + 127) / 128;
  p.num_ci_tiles = (cin_tile_extent + l.block_n - 1) / l.block_n;
  p.kblocks_total = static_cast<int>((pixels + 63) / 64);
  const int base_items = p.num_co_tiles * p.num_ci_tiles * p.num_taps;
  // split K so that the equal-sized work items fill the SMs in ONE wave (fewer splits = fewer fp32 reductions)
  int splits = std::max(1, num_sms() / base_items);
  splits = std::min(splits, std::max(1, p.kblocks_total / 4));
  // no empty splits: shrink until the last split still owns at least one k-block
  while (splits > 1) {
    const int per = (p.kblocks_total + splits - 1) / splits;
    if (per * (splits - 1) < p.kblocks_total) break;
    --splits;
  }
  p.num_ksplits = splits;
  p.log2_wo = ilog2(s.Wo());
  p.log2_howo = ilog2(s.Ho() * s.Wo());
  p.cout = s.Cout;
  p.cin = cin_tile_extent;
  p.dw_row_stride = s.Ktot();
  p.dw = dw;

  // ---- Cout == 64: transposed all-taps formulation
  const int n_boxes = (s.kind == 1) ? 4 : (s.k * s.k) * (s.Cin / 64);
  // (measured: it wins for the stem and the 3x3 layer1 convolutions; 1x1 layers are HBM-bound either way)
  if (s.Cout == 64 && n_boxes <= 10 && (s.kind == 1 || (s.k == 3 && s.Cin == 64))) {
    WgradXposeParams& x = l.xp;
    std::memset(&x, 0, sizeof(x));
    x.dy_map = p.dy_map;
    for (int i = 0; i < 4; ++i) x.a_map[i] = p.a_map[i];
    int nb = 0;
    for (int t = 0; t < p.num_taps; ++t)
      for (int cb = 0; cb < cin_tile_extent / 64; ++cb) {
        XposeBox b{};
        b.map = p.taps[t].map; b.dh = p.taps[t].dh; b.dw = p.taps[t].dw; b.valid = 1;
        b.c_off = static_cast<int16_t>(cb * 64);
        b.out_off = static_cast<int16_t>(p.taps[t].b_off + cb * 64);
        x.boxes[nb++] = b;
      }
    const int padded = nb <= 4 ? 4 : 10;
    l.xpose_nbox = padded;
    x.kblocks_total = p.kblocks_total;
    x.num_splits = std::max(1, std::min(num_sms(), p.kblocks_total / 4));
    while (x.num_splits > 1) {  // no empty split
      const int per = (x.kblocks_total + x.num_splits - 1) / x.num_splits;
      if (per * (x.num_splits - 1) < x.kblocks_total) break;
      --x.num_splits;
    }
    x.log2_wo = p.log2_wo;
    x.log2_howo = p.log2_howo;
    x.dw_row_stride = p.dw_row_stride;
    p.num_ksplits = x.num_splits;   // scratch sizing / reduce use the same field
  }
  return l;
}

WgradLaunch plan_conv_wgrad_gram(const ConvShape& s, const __nv_bfloat16* dy, const __nv_bfloat16* x, float* dw) {
  ARGUS_CHECK(s.kind == 0 && s.k == 1, "stacked weight gradient + Gram is defined for 1x1 convolutions");
  ARGUS_CHECK(s.Cout % 128 == 0, "Cout must be a multiple of 128");
  // plan as a convolution with Cout + Cin output channels, then point the rows beyond Cout at x (through a_map)
  ConvShape st = s;
  st.Cout = s.Cout + s.Cin;
  WgradLaunch l = plan_conv_wgrad(st, dy, x, dw);
  ARGUS_CHECK(l.xpose_nbox == 0, "unexpected kernel choice");
  const int64_t pixels = s.out_pixels();
  const uint64_t dims[2] = {static_cast<uint64_t>(s.Cout), static_cast<uint64_t>(pixels)};
  const uint64_t str[1] = {static_cast<uint64_t>(s.Cout) * 2};
  const uint32_t box[2] = {64, 64};
  l.p.dy_map = make_tmap_bf16(dy, 2, dims, str, box);
  l.p.co_split = s.Cout;
  l.p.stacked = 1;
  return l;
}

WgradLaunch plan_gram(const ConvShape& s, const __nv_bfloat16* x, float* g) {
  ARGUS_CHECK(s.kind == 0 && s.k == 1, "Gram matrix of the pixels a 1x1 convolution reads");
  ConvShape st = s;
  st.Cout = s.Cin;
  WgradLaunch l = plan_conv_wgrad(st, x, x, g);   // (the dy map is never used: every row comes from x)
  ARGUS_CHECK(l.xpose_nbox == 0, "unexpected kernel choice");
  l.p.co_split = 0;
  l.p.stacked = 1;
  l.family = "bn_algebra";
  return l;
}

// ------------------------------------------------------------------------------------------------
// launches
// ------------------------------------------------------------------------------------------------
// Final per-launch parameters of one kernel instance: the halo pipeline depth and the weights-resident choice depend
// on the instance's shared-memory layout and on the grid.
template <int BN, int OPT>
static ConvGemmParams finish_params(const ConvGemmParams& p) {
  using L = ConvGemmSmem<BN, conv_staging_buffers<BN, OPT>()>;
  const int tiles = p.num_m_tiles * p.num_n_tiles;
  const int grid = std::min(tiles, num_sms());
  // weights-resident mode (see ConvGemmParams::b_resident)
  ConvGemmParams q = p;
  const int bres = p.num_taps * p.kblocks_per_tap * L::kBBytes;
  const bool fixed_n = (tiles <= grid) || (grid % p.num_n_tiles == 0);
  if (q.halo) {
    const int halo_a = (q.halo_rows + 2) * q.halo_row_bytes;
    const int stage = halo_a + 3 * L::kBBytes;
    q.halo_stages = std::min(L::kMaxStages, L::kPipeBytes / stage);
    if (q.halo_stages < 2) q.halo = 0;
    // halo + weights resident: when the whole weight slab fits next to two activation boxes (layer1 3x3: 72 KB), the
    // per-tile L2 -> SM traffic drops from 3 x (32 + 24) to 3 x 32 KB
    if (q.halo && fixed_n && q.k2_blocks == 0 && bres + 2 * halo_a <= L::kPipeBytes) {
      q.b_resident = 1;
      q.halo_stages = std::min(L::kMaxStages, (L::kPipeBytes - bres) / halo_a);
    }
  }
  // (a weights-resident mode for the non-halo launches was built and measured in round 1: no gain -- weights are
  // served from L2 without cost -- and removed in round 2)
  return q;
}

template <int BN, int BMN, int OPT>
static void launch_conv_t(const ConvGemmParams& q, cudaStream_t stream) {
  using L = ConvGemmSmem<BN, conv_staging_buffers<BN, OPT>()>;
  static bool configured = false;
  if (!configured) {
    ARGUS_CUDA(cudaFuncSetAttribute(conv_gemm_kernel<BN, BMN, OPT>, cudaFuncAttributeMaxDynamicSharedMemorySize, L::kTotal));
    configured = true;
  }
  const int grid = std::min(q.num_m_tiles * q.num_n_tiles, num_sms());
  launch_kernel(conv_gemm_kernel<BN, BMN, OPT>, grid, kNumThreads, L::kTotal, stream, q);
  ARGUS_CUDA(cudaGetLastError());
}

namespace {
// Every conv_gemm_kernel instance the library compiles.
struct ConvInstanceEntry {
  int block_n, b_mn, opt;
  ConvGemmParams (*finish)(const ConvGemmParams&);
  void (*launch)(const ConvGemmParams&, cudaStream_t);
};
template <int BN, int BMN, int OPT>
constexpr ConvInstanceEntry conv_entry() {
  return {BN, BMN, OPT, &finish_params<BN, OPT>, &launch_conv_t<BN, BMN, OPT>};
}
constexpr int kTail = kOptAffine | kOptRes | kOptRelu;   // fused forward block tail: BN + identity + ReLU (+ bits)
const ConvInstanceEntry kConvInstances[] = {
    // dgrad + fused batch-norm backward reduction: plain (3x3 / 1x1 dgrads) or with the bias of the K-concatenated dgrad
    conv_entry<64, 1, kOptRes | kOptBnRed>(), conv_entry<128, 1, kOptRes | kOptBnRed>(),
    conv_entry<256, 1, kOptRes | kOptBnRed>(), conv_entry<64, 1, kOptAffine | kOptRes | kOptBnRed>(),
    conv_entry<128, 1, kOptAffine | kOptRes | kOptBnRed>(), conv_entry<256, 1, kOptAffine | kOptRes | kOptBnRed>(),
    // folded batch norm without statistics
    conv_entry<64, 0, kTail>(), conv_entry<128, 0, kTail>(), conv_entry<256, 0, kTail>(),
    conv_entry<64, 0, kOptAffine | kOptRelu>(), conv_entry<128, 0, kOptAffine | kOptRelu>(),
    conv_entry<256, 0, kOptAffine | kOptRelu>(), conv_entry<64, 0, kOptAffine>(), conv_entry<128, 0, kOptAffine>(),
    conv_entry<256, 0, kOptAffine>(),
    // plain: store the tile (+ statistics)
    conv_entry<64, 0, 0>(), conv_entry<128, 0, 0>(), conv_entry<256, 0, 0>(), conv_entry<64, 1, 0>(),
    conv_entry<128, 1, 0>(), conv_entry<256, 1, 0>(),
    // dgrads: identity-branch gradient + ReLU bits of the previous block; K-concatenated dgrad with bias + bits
    conv_entry<64, 1, kOptRes | kOptOutBits>(), conv_entry<128, 1, kOptRes | kOptOutBits>(),
    conv_entry<256, 1, kOptRes | kOptOutBits>(), conv_entry<64, 1, kOptAffine | kOptOutBits>(),
    conv_entry<128, 1, kOptAffine | kOptOutBits>(), conv_entry<256, 1, kOptAffine | kOptOutBits>(),
    // the generic kernel
    conv_entry<64, 0, kOptAll>(), conv_entry<128, 0, kOptAll>(), conv_entry<256, 0, kOptAll>(),
    conv_entry<64, 1, kOptAll>(), conv_entry<128, 1, kOptAll>(), conv_entry<256, 1, kOptAll>(),
};
const ConvInstanceEntry& find_instance(const ConvInstance& c) {
  for (const auto& e : kConvInstances)
    if (e.block_n == c.block_n && e.b_mn == c.b_mn && e.opt == c.opt) return e;
  throw Error("unsupported conv tile configuration");
}

std::mutex g_record_mu;
std::atomic<bool> g_recording{false};
std::set<std::array<int, 5>> g_recorded;
std::set<std::array<int, 5>> g_recorded_wgrad;
std::set<std::array<int, 5>> g_recorded_bn_alg;
}  // namespace

ConvGemmParams epilogue_params(const ConvLaunch& l, const Epilogue& e) {
  ConvGemmParams p = l.p;
  p.scale = e.scale;
  p.shift = e.shift;
  p.has_res = 0;
  if (e.residual != nullptr) {
    ARGUS_CHECK(l.out_geom.rank == 4, "this launch cannot take a residual (strided output)");
    p.res_map = make_tmap_bf16(e.residual, 4, l.out_geom.dims, l.out_geom.strides, l.out_geom.box);
    p.has_res = 1;
    p.res_bits = e.residual_bits;
  }
  p.bn_raw = nullptr;
  p.bn_scale = e.bn_scale;
  p.bn_shift = e.bn_shift;
  if (e.bn_raw != nullptr) {
    ARGUS_CHECK(l.b_mn == 1 && l.out_geom.rank == 4, "the fused BN reduction exists for dense-output dgrad launches");
    ARGUS_CHECK(e.residual == nullptr && e.out_bits == nullptr && e.relu == 0 && e.relu_bits_out == nullptr &&
                    e.scale == nullptr && e.bn_scale != nullptr && e.bn_shift != nullptr && e.stat_partial != nullptr,
                "fused BN reduction: unsupported epilogue combination");
    p.res_map = make_tmap_bf16(e.bn_raw, 4, l.out_geom.dims, l.out_geom.strides, l.out_geom.box);
    p.has_res = 1;
    p.bn_raw = e.bn_raw;
  }
  p.early_trigger = (e.early_trigger && pdl_enabled()) ? 1 : 0;
  p.relu = e.relu;
  p.out_bits = e.out_bits;
  p.res_scale = e.res_scale;
  p.res_shift = e.res_shift;
  p.relu_bits_out = e.relu_bits_out;
  ARGUS_CHECK((e.res_scale == nullptr) == (e.res_shift == nullptr), "residual scale and shift come together");
  p.stat_partial = e.stat_partial;
  return p;
}

// Specialised epilogues for the option combinations the model launches; anything else runs the generic kernel.
ConvInstance select_conv_instance(const ConvLaunch& l, const ConvGemmParams& p) {
  int need = 0;
  if (p.scale || p.shift) need |= kOptAffine;
  if (p.has_res) need |= kOptRes;
  if (p.res_bits || p.res_scale) need |= kOptRes | kOptResExtra;
  if (p.out_bits) need |= kOptOutBits;
  if (p.relu || p.relu_bits_out) need |= kOptRelu;
  if (p.bn_raw != nullptr) return {l.block_n, 1, kOptRes | kOptBnRed | (p.shift != nullptr ? kOptAffine : 0)};
  // Folded batch norm without statistics (packed-fp32 epilogue, coefficients in shared memory): the fused forward block
  // tail, its downsample branch, every eval-mode convolution. Needs BOTH coefficient vectors (a bias-only epilogue such as
  // resnet.fc runs the generic kernel). Round 2 also tried loading the residual row segments straight from global memory
  // into registers: one thread per row = 32 rows per load instruction, uncoalesced, 1.5-1.9 TB/s against 5.1-5.5 TB/s
  // through TMA + staging (profiles/r2_direct_residual_ab.txt).
  const bool folded_bn = p.scale && p.shift && !p.stat_partial && !p.res_bits && !p.res_scale && !p.out_bits;
  if (l.b_mn == 0 && folded_bn && (need & kOptAffine) && !(need & ~kTail) && (p.relu || !p.relu_bits_out)) {
    const int t = need & kTail;
    if (t == kTail || t == (kOptAffine | kOptRelu) || t == kOptAffine) return {l.block_n, 0, t};
    // e.g. identity + BN without ReLU: generic kernel
  }
  if (need == 0) return {l.block_n, l.b_mn, 0};
  if (l.b_mn == 1 && (need & ~(kOptRes | kOptOutBits)) == 0) return {l.block_n, 1, kOptRes | kOptOutBits};
  // K-concatenated dgrad of the algebraic BN backward: bias + output bits
  if (l.b_mn == 1 && (need & ~(kOptAffine | kOptOutBits)) == 0) return {l.block_n, 1, kOptAffine | kOptOutBits};
  return {l.block_n, l.b_mn, kOptAll};
}

ConvLaunchInfo conv_launch_info(const ConvLaunch& l, const Epilogue& e) {
  const ConvGemmParams p = epilogue_params(l, e);
  ConvLaunchInfo info;
  info.inst = select_conv_instance(l, p);
  const ConvGemmParams q = find_instance(info.inst).finish(p);
  info.halo = q.halo;
  info.b_resident = q.b_resident;
  info.halo_stages = q.halo ? q.halo_stages : 0;
  info.num_m_tiles = q.num_m_tiles;
  info.num_n_tiles = q.num_n_tiles;
  info.grid = std::min(q.num_m_tiles * q.num_n_tiles, num_sms());
  info.stat_slots = stat_slots(l);
  return info;
}

void conv_instances_record(bool on) {
  std::lock_guard<std::mutex> lk(g_record_mu);
  if (on) { g_recorded.clear(); g_recorded_wgrad.clear(); g_recorded_bn_alg.clear(); }
  g_recording = on;
}
void bn_alg_call_record(int O, int C, int stride, bool dw_aside, bool multi_slot) {
  if (!g_recording) return;
  std::lock_guard<std::mutex> lk(g_record_mu);
  g_recorded_bn_alg.insert({O, C, stride, dw_aside ? 1 : 0, multi_slot ? 1 : 0});
}
std::vector<std::array<int, 5>> bn_alg_calls_recorded() {
  std::lock_guard<std::mutex> lk(g_record_mu);
  return std::vector<std::array<int, 5>>(g_recorded_bn_alg.begin(), g_recorded_bn_alg.end());
}
std::vector<std::array<int, 3>> conv_instances_all() {
  std::vector<std::array<int, 3>> v;
  for (const auto& e : kConvInstances) v.push_back({e.block_n, e.b_mn, e.opt});
  return v;
}
std::vector<std::array<int, 5>> conv_instances_recorded() {
  std::lock_guard<std::mutex> lk(g_record_mu);
  return std::vector<std::array<int, 5>>(g_recorded.begin(), g_recorded.end());
}
std::vector<std::array<int, 5>> wgrad_instances_recorded() {
  std::lock_guard<std::mutex> lk(g_record_mu);
  return std::vector<std::array<int, 5>>(g_recorded_wgrad.begin(), g_recorded_wgrad.end());
}

void launch_conv(const ConvLaunch& l, const Epilogue& e, cudaStream_t stream) {
  const ConvGemmParams p = epilogue_params(l, e);
  const double flops = 2.0 * p.m_total * static_cast<double>(p.n_total) * (p.num_taps * p.kblocks_per_tap + p.k2_blocks) * kBlockK;
  std::string fam = l.b_mn ? "conv_dgrad" : "conv_fwd";
  if (g_profiling && profile_detailed())
    fam += ":M" + std::to_string(p.m_total) + "_N" + std::to_string(p.n_total) + "_K" +
           std::to_string((p.num_taps * p.kblocks_per_tap + p.k2_blocks) * kBlockK) + "_t" + std::to_string(p.num_taps);
  // algorithmic HBM bytes: every operand tensor once (activation planes actually read, result, residual, bit masks, weights)
  double bytes = 0.0;
  {
    int maps = 0;
    for (int t = 0; t < p.num_taps; ++t) maps |= 1 << p.taps[t].map;
    const int nmaps = __builtin_popcount(static_cast<unsigned>(maps));
    const double kc = static_cast<double>(p.kblocks_per_tap) * kBlockK;
    bytes += 2.0 * p.m_total * kc * nmaps + 2.0 * p.m_total * p.k2_blocks * kBlockK;
    bytes += 2.0 * p.m_total * p.n_total * (p.has_res ? 2 : 1);   // (the fused BN reduction reads bn_raw: counted here)
    bytes += (p.out_bits ? 0.125 : 0.0) * p.m_total * p.n_total + (p.relu_bits_out ? 0.125 : 0.0) * p.m_total * p.n_total;
    bytes += 2.0 * p.n_total * (p.num_taps * kc + p.k2_blocks * kBlockK);
  }
  ProfileScope prof(fam, stream, flops, bytes);
  const ConvInstance inst = select_conv_instance(l, p);
  const ConvInstanceEntry& entry = find_instance(inst);
  const ConvGemmParams q = entry.finish(p);
  if (g_recording) {
    std::lock_guard<std::mutex> lk(g_record_mu);
    g_recorded.insert({inst.block_n, inst.b_mn, inst.opt, q.halo, q.b_resident});
  }
  entry.launch(q, stream);
}

int stat_slots(const ConvLaunch& l) {
  const int tiles = l.p.num_m_tiles * l.p.num_n_tiles;
  return kEpiGroups * std::min(tiles, num_sms());
}

int64_t wgrad_scratch_elems(const WgradLaunch& l) {
  if (l.xpose_nbox > 0) return static_cast<int64_t>(l.xp.num_splits) * 64 * l.p.dw_row_stride;
  if (l.p.num_ksplits <= 1) return 0;
  return static_cast<int64_t>(l.p.num_ksplits) * l.p.cout * l.p.dw_row_stride;
}

// dw[i] += sum_ks partial[ks][i] in a fixed order (deterministic): a block owns 64 float4 elements, its four thread
// groups take the splits g, g + 4, g + 8, ... (eight loads in flight each) and group 0 adds the four sums in group order.
// Split-K counts reach 148, so walking them with one thread per element was a chain of dependent L2 round trips.
__global__ void __launch_bounds__(256)
wgrad_reduce_kernel(const float4* __restrict__ partial, float4* __restrict__ dw, int64_t n4, int splits) {
  pdl_prologue();
  __shared__ float4 red[4][64];
  const int e = threadIdx.x & 63, g = threadIdx.x >> 6;
  auto add = [](float4& a, const float4& v) { a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w; };
  for (int64_t base = static_cast<int64_t>(blockIdx.x) * 64; base < n4; base += static_cast<int64_t>(gridDim.x) * 64) {
    const int64_t i = base + e;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    if (i < n4) {
      int k = g;
      for (; k + 28 < splits; k += 32) {
        float4 v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) v[u] = partial[static_cast<int64_t>(k + 4 * u) * n4 + i];
#pragma unroll
        for (int u = 0; u < 8; ++u) add(acc, v[u]);
      }
      for (; k < splits; k += 4) add(acc, partial[static_cast<int64_t>(k) * n4 + i]);
    }
    red[g][e] = acc;
    __syncthreads();
    if (g == 0 && i < n4) {
      float4 t = red[0][e];
      add(t, red[1][e]); add(t, red[2][e]); add(t, red[3][e]);
      float4 d = dw[i];
      add(d, t);
      dw[i] = d;
    }
    __syncthreads();
  }
}

template <int NBOX>
static void launch_wgrad_xpose_t(const WgradLaunch& l, int grid, cudaStream_t stream) {
  using L = WgradXposeSmem<NBOX>;
  static bool configured = false;
  if (!configured) {
    ARGUS_CUDA(cudaFuncSetAttribute(wgrad_xpose_kernel<NBOX>, cudaFuncAttributeMaxDynamicSharedMemorySize, L::kTotal));
    configured = true;
  }
  launch_kernel(wgrad_xpose_kernel<NBOX>, grid, kWgradThreads, L::kTotal, stream, l.xp);
  ARGUS_CUDA(cudaGetLastError());
}

template <int BN>
static void launch_wgrad_t(const WgradLaunch& l, int grid, cudaStream_t stream) {
  using L = WgradSmem<BN>;
  static bool configured = false;
  if (!configured) {
    ARGUS_CUDA(cudaFuncSetAttribute(wgrad_kernel<BN>, cudaFuncAttributeMaxDynamicSharedMemorySize, L::kTotal));
    configured = true;
  }
  launch_kernel(wgrad_kernel<BN>, grid, kWgradThreads, L::kTotal, stream, l.p);
  ARGUS_CUDA(cudaGetLastError());
}

namespace {
// Every weight-gradient kernel instance the library compiles: (transposed, BLOCK_N or padded box count).
struct WgradInstanceEntry {
  int xpose, n;
  void (*launch)(const WgradLaunch&, int, cudaStream_t);
};
const WgradInstanceEntry kWgradInstances[] = {
    {0, 64, &launch_wgrad_t<64>}, {0, 128, &launch_wgrad_t<128>}, {0, 256, &launch_wgrad_t<256>},
    {1, 4, &launch_wgrad_xpose_t<4>}, {1, 10, &launch_wgrad_xpose_t<10>},
};
}  // namespace

std::vector<std::array<int, 2>> wgrad_instances_all() {
  std::vector<std::array<int, 2>> v;
  for (const auto& e : kWgradInstances) v.push_back({e.xpose, e.n});
  return v;
}

WgradLaunchInfo wgrad_launch_info(const WgradLaunch& l) {
  WgradLaunchInfo info;
  const WgradParams& p = l.p;
  info.xpose = l.xpose_nbox > 0 ? 1 : 0;
  info.n = info.xpose ? l.xpose_nbox : l.block_n;
  info.stacked = p.stacked;
  info.co_split = p.co_split;
  info.num_taps = p.num_taps;
  info.num_co_tiles = p.num_co_tiles;
  info.num_ci_tiles = p.num_ci_tiles;
  info.num_ksplits = p.num_ksplits;
  info.kblocks_total = p.kblocks_total;
  info.grid = info.xpose ? l.xp.num_splits
                         : std::min(p.num_co_tiles * p.num_ci_tiles * p.num_ksplits * p.num_taps, num_sms());
  info.scratch_elems = wgrad_scratch_elems(l);
  return info;
}

void launch_wgrad(const WgradLaunch& l0, float* scratch, cudaStream_t stream) {
  WgradLaunch l = l0;
  const WgradLaunchInfo info = wgrad_launch_info(l);
  const int64_t need = info.scratch_elems;
  ARGUS_CHECK(need == 0 || scratch != nullptr, "split-K weight gradient needs a scratch buffer");
  l.p.partial = scratch;
  l.p.partial_stride = static_cast<long long>(l.p.cout) * l.p.dw_row_stride;
  const double flops = 2.0 * l.p.kblocks_total * 64.0 * l.p.cout * static_cast<double>(l.p.cin) * l.p.num_taps;
  std::string fam = l0.family;
  if (g_profiling && profile_detailed())
    fam += std::string(l.xpose_nbox > 0 ? "x" : "") + ":P" + std::to_string(l.p.kblocks_total * 64) + "_Co" + std::to_string(l.p.cout) + "_Ci" +
           std::to_string(l.p.cin) + "_t" + std::to_string(l.p.num_taps) + "_s" + std::to_string(l.p.num_ksplits);
  const double wbytes = 2.0 * l.p.kblocks_total * 64.0 * (static_cast<double>(l.p.cout) + l.p.cin) +
                        4.0 * l.p.cout * static_cast<double>(l.p.dw_row_stride);
  ProfileScope prof(fam, stream, flops, wbytes);
  if (l.xpose_nbox > 0) {
    ARGUS_CHECK(scratch != nullptr, "transposed weight gradient needs a scratch buffer");
    l.xp.partial = scratch;
  }
  const WgradInstanceEntry* entry = nullptr;
  for (const auto& e : kWgradInstances)
    if (e.xpose == info.xpose && e.n == info.n) entry = &e;
  if (entry == nullptr) throw Error("unsupported wgrad configuration");
  if (g_recording) {
    std::lock_guard<std::mutex> lk(g_record_mu);
    g_recorded_wgrad.insert({info.xpose, info.n, info.stacked, info.co_split > 0 ? 1 : 0, info.num_ksplits > 1 ? 1 : 0});
  }
  entry->launch(l, info.grid, stream);
  if (need > 0) {
    // every (split, cout, tap, ci) word of the scratch was written by exactly one work item
    const int64_t n4 = l.p.partial_stride / 4;
    const int grid = static_cast<int>(std::min<int64_t>((n4 + 63) / 64, 4LL * num_sms()));
    launch_kernel(wgrad_reduce_kernel, grid, 256, 0, stream, reinterpret_cast<const float4*>(scratch),
                                                  reinterpret_cast<float4*>(l.p.dw), n4, l.p.num_ksplits);
    ARGUS_CUDA(cudaGetLastError());
  }
}

}  // namespace argus

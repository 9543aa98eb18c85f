// Host side of the C-ABI (include/climsr_b200.h): layer table, weight-pack layout, tile selection, TMA tensor
// maps, the forward plan (buffer carving + launch list) and the exported entry points.
#include <algorithm>
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/climsr_b200.h"
#include "conv_tc.cuh"
#include "disc.cuh"
#include "elementwise.cuh"
#include "loss.cuh"
#include "metrics.cuh"
#include "rcan.cuh"
#include "rdb_tc.cuh"
#include "wgrad_tc.cuh"

namespace csr {

// ------------------------------------------------------------------------------------------- errors
static thread_local char g_err[512] = "";
static std::atomic<long long> g_launches{0};
static int g_opt_pdl = 1;
static long long* g_trace = nullptr;
static unsigned long long* g_timeline = nullptr;   // csr_debug_set_timeline
static int g_timeline_cap = 0;
static int g_opt_no_tma_store = 0;
static int g_opt_graphs = 1;
static int g_opt_graph_max_px = 1 << 21;   // forward: replay a CUDA graph up to this many HR pixels per call (larger batches are GPU-bound)
static int g_opt_wgrad_atomic = 1;      // weight-gradient partial sums through red.global.add.v4.f32 instead of per-CTA slices + reduce kernel
static int g_opt_eight_acc = 1;         // eight accumulator buffers for two-tile windows when TMEM has room (KW*npad <= 64)
static int g_opt_tall = 1;              // two M tiles per window for thin layers
static int g_opt_narrow_box = 1;        // 16- / 32-channel window boxes for layers over <= 16 / 32 input channels
static int g_opt_trace_cta = 0;         // debug: CTA recorded by csr_debug_set_trace
static int g_opt_reserve_sms = 0;       // plans created afterwards size their persistent grids to (SM count - this): the SMs left free run the
                                        // gradient all-reduce (NCCL, capped to as many CTAs) concurrently with the backward kernels
static int g_opt_dense_min = 2;         // ... only when a block has at least this many windows per SM: with <= 1 window per CTA nothing pipelines
                                        // across layers and the counters only cost (cfg1 / one Europe raster / cfg3: 7-10 % slower, r02 A/B)
static int g_opt_tap_pack = 1;          // conv_last's tap sum fused with the SRCNN input im2col (tap_pack_kernel)
static int g_opt_hyb = 1;               // hybrid tap fold (conv_tc.cu HYB_T) on the early-release layers (HRconv 338 -> 294 us)
static int g_opt_merge_phases = 1;      // sub-pixel phase pairs of nearest-x2 + conv as one launch (gridDim.y, emit_conv)
static int g_opt_fuse_tail = 3;         // inference, second MMA over the staged tile: bit 0 srcnn.conv2 inside srcnn.conv1's epilogue, bit 1 conv_last's
                                        // nine tap planes inside HRconv's epilogue (+ tap_sum_kernel)
static int g_opt_dense = 1;             // conv1..conv4 of every gc = 16 dense block as ONE persistent launch with tile-level dependencies (rdb_tc.cu)
static int g_opt_early = 1;             // early-release epilogue (conv_tc.cu, EARLY_T) for the wide residual-free layers
static int g_opt_whole_row = 1;         // whole-row tiles (SW = W) for the trunk's 3x3 convs over 32- / 64-pixel-wide maps (choose_tiling)

static int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}
#define CSR_CUDA(expr)                                                                          \
  do {                                                                                          \
    cudaError_t _e = (expr);                                                                    \
    if (_e != cudaSuccess) return fail(CSR_ERR_CUDA, "%s: %s", #expr, cudaGetErrorString(_e)); \
  } while (0)

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }

// ------------------------------------------------------------------------------------------- device
struct DeviceInfo {
  bool ok = false;
  int sms = 0;
  int dev = -1;
};
static int device_info(DeviceInfo* out) {
  int dev = 0;
  CSR_CUDA(cudaGetDevice(&dev));
  // cudaGetDeviceProperties costs milliseconds: the single-op entry points (csr_conv2d_nhwc, csr_conv2d_wgrad - ~100 calls per
  // discriminator step) must not pay it per call
  static DeviceInfo cache[64];
  static std::mutex mu;
  if (dev >= 0 && dev < 64) {
    std::lock_guard<std::mutex> lock(mu);
    if (cache[dev].ok) { *out = cache[dev]; return CSR_OK; }
  }
  int major = 0, minor = 0, sms = 0;
  CSR_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  CSR_CUDA(cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev));
  CSR_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  if (major != 10) return fail(CSR_ERR_UNSUPPORTED, "device %d is sm_%d%d; this library is sm_100a only", dev, major, minor);
  out->ok = true;
  out->sms = sms;
  out->dev = dev;
  if (dev >= 0 && dev < 64) {
    std::lock_guard<std::mutex> lock(mu);
    cache[dev] = *out;
  }
  return CSR_OK;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult q;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess)
    return nullptr;
  fn = reinterpret_cast<EncodeTiledFn>(p);
  return fn;
}

// NHWC bf16 activation buffer as a 4-D (C, W, H, N) tensor; box = 64 channels x box_w x box_h x 1, 128B swizzle,
// out-of-bounds -> zeros (this IS the convolution's zero padding).
static int encode_act_map(CUtensorMap* m, const void* base, int N, int H, int W, int C, int box_w, int box_h, int box_c = 64) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return fail(CSR_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
  cuuint64_t strides[3] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2};
  cuuint32_t box[4] = {(cuuint32_t)box_c, (cuuint32_t)box_w, (cuuint32_t)box_h, 1};
  const CUtensorMapSwizzle swz = box_c == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : box_c == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B;
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(CSR_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d) for N%d H%d W%d C%d box %dx%d", (int)r, N, H, W, C, box_w, box_h);
  return CSR_OK;
}

// ------------------------------------------------------------------------------------------- layer table
struct LayerSpec {
  std::string name;
  int cout, cin, kh, kw;   // reference (state_dict) shape
  int fold = 0;            // 1: executed as a kh x 1 conv over an x-im2col input with kw*cin channels (srcnn.conv1)
  int up2 = 0;             // 1: the layer's input is nearest-x2 upsampled first (esrgan.py:94,97): executed as four
                           //    sub-pixel phases, each a 2x2 conv over the low-resolution input with summed weights
  int transposed = 0;      // 1: input-gradient conv: weight read as w[ci][co][KH-1-dy][KW-1-dx] (autograd of the layer)
  float wscale = 1.f;      // constant folded into the packed weights
  int src = -1;            // backward tables: index of the forward layer whose weight tensor is packed
  struct Block { int src, ci_lo, n, src_ci_off, src_cin; float wscale; };
  // backward tables (transposed): executed input-channel blocks gathered from several forward layers
  std::vector<Block> blocks;
  int ekw() const { return fold ? 1 : kw; }
  int ecin() const { return fold ? cin * kw : cin; }
};

static int check_net(const CsrNetDesc* net) {
  if (!net) return fail(CSR_ERR_BAD_ARG, "net descriptor is null");
  if (net->in_channels < 1 || net->in_channels > 16) return fail(CSR_ERR_UNSUPPORTED, "in_channels %d not in [1,16]", net->in_channels);
  if (net->out_channels != 1) return fail(CSR_ERR_UNSUPPORTED, "out_channels must be 1 (SRCNN tail takes 1+1+1 channels, esrgan.py:87)");
  if (net->nf != 64) return fail(CSR_ERR_UNSUPPORTED, "nf must be 64");
  if (net->gc != 16 && net->gc != 32) return fail(CSR_ERR_UNSUPPORTED, "gc must be 16 or 32");
  if (net->nb < 1 || net->nb > 64) return fail(CSR_ERR_UNSUPPORTED, "nb %d not in [1,64]", net->nb);
  if (net->scale != 4) return fail(CSR_ERR_UNSUPPORTED, "scale must be 4");
  return CSR_OK;
}

// state_dict order of the reference generator (esrgan.py:72-87, srcnn.py:9-11)
static std::vector<LayerSpec> layer_table(const CsrNetDesc& d) {
  std::vector<LayerSpec> v;
  v.push_back({"conv_first", d.nf, d.in_channels, 3, 3});
  for (int i = 0; i < d.nb; ++i)
    for (int r = 1; r <= 3; ++r) {
      const std::string pre = "RRDB_trunk." + std::to_string(i) + ".RDB" + std::to_string(r) + ".conv";
      for (int k = 1; k <= 4; ++k) v.push_back({pre + std::to_string(k), d.gc, d.nf + (k - 1) * d.gc, 3, 3});
      v.push_back({pre + "5", d.nf, d.nf + 4 * d.gc, 3, 3});
    }
  v.push_back({"trunk_conv", d.nf, d.nf, 3, 3});
  v.push_back({"upconv1", d.nf, d.nf, 3, 3, 0, 1});
  v.push_back({"upconv2", d.nf, d.nf, 3, 3, 0, 1});
  v.push_back({"HRconv", d.nf, d.nf, 3, 3});
  v.push_back({"conv_last", d.out_channels, d.nf, 3, 3});
  v.push_back({"srcnn.conv1", 64, 3, 9, 9, 1});
  v.push_back({"srcnn.conv2", 32, 64, 1, 1});
  v.push_back({"srcnn.conv3", d.out_channels, 32, 5, 5});
  return v;
}

// Forward EXECUTION table: the state_dict table plus a view of conv_last's weights.
static std::vector<LayerSpec> fwd_exec_table(const CsrNetDesc& d, const std::vector<LayerSpec>& f) {
  std::vector<LayerSpec> v = f;
  for (size_t i = 0; i < v.size(); ++i) v[i].src = (int)i;
  // conv_last (64 -> 1, 3x3) seen as a 1x1 layer with nine "output channels" = its nine taps: tap[t](y, x) = sum_c W[0][c][t] * in(y, x)[c].
  // Inference runs it as a second MMA inside HRconv's epilogue (conv_tc.cu FUSE_T = 2) and sums the shifted taps afterwards
  // (tap_sum_kernel), so HRconv's 64-channel HR map never reaches memory.  W[0][c][ky][kx] flattened is [c][t]: the transposed read
  // of a (cout = 9, cin = 64, 1 x 1) layer.  Always the LAST entry, so state_dict indices keep their meaning.
  LayerSpec T{"conv_last.taps", 9, d.nf, 1, 1};
  T.transposed = 1;
  T.src = (int)f.size() - 4;                               // conv_last
  v.push_back(T);
  return v;
}

// Packed form of one layer: one or four (sub-pixel phases) kernels, each possibly split over output channels so that
// one part's weights fit in shared memory and its epilogue handles <= kMaxNpad channels.
constexpr int kMaxResidentWeightBytes = 150 * 1024;
struct PackPart {
  int kh, kw, ph, pw;      // effective taps / padding of this launch
  int phase;               // -1, or a*2+b: output pixel (2y+a, 2x+b)
  int co_lo, n_store, npad;
  size_t w_off, b_off;
  int w_bytes;
  int stream = 0;          // 1: too large to stay resident next to the window ring: streamed k-block by k-block (ConvParams::stream_w)
};
struct PackLayer {
  int cin_pad;
  std::vector<PackPart> parts;
};
static int part_weight_bytes(int kh, int kw, int cin_pad, int npad) { return kh * kw * cin_pad * npad * 2; }
// UMMA N = KW*npad <= 256 and two accumulator buffers of KW*npad fp32 columns must fit the 512 TMEM columns.
static int max_npad(int kw) { return std::max(16, std::min(kMaxNpad, 256 / kw / 16 * 16)); }

static std::vector<PackLayer> pack_layout(const std::vector<LayerSpec>& layers, size_t* total, bool allow_stream = false) {
  std::vector<PackLayer> out;
  size_t off = 0;
  for (const auto& L : layers) {
    PackLayer pl;
    pl.cin_pad = (L.ecin() + 15) / 16 * 16;
    const int npad_full = (L.cout + 15) / 16 * 16;
    const int kh = L.up2 ? 2 : L.kh, kw = L.up2 ? 2 : L.ekw();
    int nsplit = 1;
    // layers whose 64-output-channel part would not fit next to a window ring (>= 256 input channels at 3x3) either split further
    // (16-channel parts: 32 thin launches for 512 -> 512) or, for the single-conv API, keep 64-channel parts and stream the weights
    const bool stream = allow_stream && !L.up2 && part_weight_bytes(kh, kw, pl.cin_pad, std::min(npad_full, max_npad(kw))) > kMaxResidentWeightBytes;
    while (((!stream && part_weight_bytes(kh, kw, pl.cin_pad, ceil_div(npad_full / 16, nsplit) * 16) > kMaxResidentWeightBytes) ||
            ceil_div(npad_full / 16, nsplit) * 16 > max_npad(kw)) && nsplit < npad_full / 16) ++nsplit;
    const int per = ceil_div(npad_full / 16, nsplit) * 16;
    for (int phase = L.up2 ? 0 : -1; phase < (L.up2 ? 4 : 0); ++phase) {
      for (int lo = 0; lo < npad_full; lo += per) {
        PackPart pp;
        pp.kh = kh; pp.kw = kw;
        // sub-pixel phase (a,b): rows (y-1+a, y+a) -> PH = 1-a; its input gradient is the flipped correlation -> PH' = a
        pp.ph = L.up2 ? (L.transposed ? (phase >> 1) : 1 - (phase >> 1)) : L.kh / 2;
        pp.pw = L.up2 ? (L.transposed ? (phase & 1) : 1 - (phase & 1)) : L.ekw() / 2;
        pp.phase = phase;
        pp.co_lo = lo;
        pp.npad = std::min(per, npad_full - lo);
        pp.n_store = std::min(L.cout - lo, pp.npad);
        pp.w_bytes = part_weight_bytes(kh, kw, pl.cin_pad, pp.npad);
        pp.stream = stream ? 1 : 0;
        pp.w_off = off;
        off = align_up(off + pp.w_bytes, 128);
        pp.b_off = off;
        off = align_up(off + pp.npad * 4, 128);
        pl.parts.push_back(pp);
      }
    }
    out.push_back(pl);
  }
  *total = off;
  return out;
}

// ------------------------------------------------------------------------------------------- tiling
struct Tiling {
  int SW, TH, TW, win_rows, win_bytes, slot_bytes, n_slots, stage_bytes;
  double eff;   // useful fraction of the MMA rows (with the small penalties applied by choose_tiling)
  int whole_row;   // SW == TW == W: no halo columns (ConvParams / DenseParams::whole_row)
  int n_stage;     // staging buffers the shape was sized with (whole rows may take fewer than asked for, see choose_tiling)
};
constexpr int kMaxSlots = 8;   // deepest window ring of a conv or dense-block launch
// whole_row (option 37): 1 = also consider whole-row tiles of a 3x3 conv over a 32- or 64-pixel-wide map (SW = TW = W, TH = 128 / W,
// no halo columns: 20 % fewer M tiles than SW = 16 at W = 64, 33 % fewer than SW = 16 at W = 32); 2 = the same, and if n_stage = 2
// staging buffers leave room for one window slot only, size it with ONE staging buffer the two epilogue groups share in tile order
// (RDB conv5: 144 KB of weights + 2 x 32 KB slots + 2 x 16 KB staging buffers do not fit 227 KB).
static int choose_tiling(int H, int W, int KH, int KW, int w_bytes, int n_kblocks, int stage_row_bytes, int n_stage, Tiling* out,
                         int row_bytes = 128, int tall = 1, int extra_slot_bytes = 0, int whole_row = 0) {
  double best = -1;
  auto consider = [&](int SW, bool wr, int nst) {
    const int TW = wr ? SW : SW - (KW - 1);
    if (TW < 1) return 0;
    const int TH = kTileM / SW;
    const int win_rows = tall * TH + KH - 1;
    const int win_bytes = win_rows * SW * row_bytes;
    const int slot_bytes = (int)align_up(win_bytes, 1024) + (int)align_up(extra_slot_bytes, 1024);   // + a streamed weight k-block
    const int stage_bytes = stage_row_bytes ? (int)align_up((size_t)TH * TW * stage_row_bytes, 1024) : 0;
    const int fixed = 1024 + (int)align_up(w_bytes, 128) + 256 + 512 + nst * stage_bytes + (wr ? kXchgBytes : 0);
    const int slots = std::min(kMaxSlots, (kSmemLimit - fixed) / slot_bytes);
    if (slots < 1) return 0;
    const double tiles = (double)ceil_div(H, TH * tall) * ceil_div(W, TW) * tall;
    double eff = (double)H * W / (tiles * kTileM);
    if (slots < std::min(2, n_kblocks + 1)) eff *= 0.7;  // no load/MMA overlap
    eff -= 1e-4 * win_bytes / (double)(kTileM * 128);    // tie-break: less halo traffic
    if (eff > best) {
      best = eff;
      *out = {SW, TH, TW, win_rows, win_bytes, slot_bytes, slots, stage_bytes, eff, wr ? 1 : 0, nst};
    }
    return slots;
  };
  for (int SW = 16; SW <= 128; SW *= 2) {
    // The epilogue sums the folded horizontal taps with warp shuffles: a window row must not straddle two warps (except for
    // whole-row tiles, which hand the taps at the warp boundary over through shared memory).
    if (KW > 1 && SW > 32) continue;
    consider(SW, false, n_stage);
  }
  if (whole_row && g_opt_whole_row && KH == 3 && KW == 3 && (W == 32 || W == 64)) {
    if (consider(W, true, n_stage) < std::min(2, n_kblocks + 1) && whole_row == 2 && n_stage == 2) consider(W, true, 1);
  }
  if (best < 0) return fail(CSR_ERR_UNSUPPORTED, "no tile shape fits shared memory (weights %d bytes, %dx%d kernel)", w_bytes, KH, KW);
  return CSR_OK;
}

// One launch: parameters + its tensor maps.
struct ConvLaunch {
  ConvParams p;
  CUtensorMap tmap;
  size_t w_off = 0, b_off = 0;  // offsets into the packed blob (resolved at forward time)
  size_t w2_off = 0, b2_off = 0;  // fused 1x1 successor (ConvParams::fuse2)
};

// conv1..conv4 of one dense block as one launch (rdb_tc.cu)
struct DenseLaunch {
  DenseParams p;
  CUtensorMap tmap;
  size_t w_off[kDenseMaxLayers], b_off[kDenseMaxLayers];   // offsets into the packed blob (resolved at forward time)
};

enum OutKind { kOutBf16 = 0, kOutF32Planar = 1, kOutF32Nhwc = 2, kOutBf16Split = 3 };
struct ConvIO {
  const void* in = nullptr; int in_C = 0, cin_off = 0;
  void* out = nullptr; int out_C = 0, out_coff = 0; int out_kind = kOutBf16;
  int split_off = 0;       // kOutBf16Split: channel distance from a hi value to its lo
  int act = CSR_ACT_NONE; float act_slope = 0.f;   // act_slope: CSR_ACT_LRELU's negative slope
  const void* r1 = nullptr; int r1_C = 0, r1_coff = 0; float s1 = 1.f;
  const void* r2 = nullptr; int r2_C = 0, r2_coff = 0; float s2 = 1.f;
  const void* gate = nullptr; int gate_C = 0, gate_coff = 0, gate_from = 0; float gate_neg = 0.2f;
};

// H, W: spatial size of the launch's input (for an up2 layer: the low-resolution input; its output is 2H x 2W).  cl->tmap is left to
// the caller: emit_conv encodes the input map of the launches it keeps, bwd_build a sub-pixel phase view.
static int build_conv(const PackLayer& pl, const PackPart& pp, int N, int H, int W, const ConvIO& io, ConvLaunch* cl) {
  if (io.in_C % 8 != 0 || io.cin_off % 8 != 0) return fail(CSR_ERR_BAD_ARG, "input buffer channels (%d) / offset (%d) must be multiples of 8", io.in_C, io.cin_off);
  const bool split = io.out_kind == kOutBf16Split;
  if ((io.out_kind == kOutBf16 || split) && ((io.out_C % 8) || (io.out_coff % 8))) return fail(CSR_ERR_BAD_ARG, "output channel stride/offset must be multiples of 8");
  if (split && (pp.n_store % 8 || io.split_off % 8)) return fail(CSR_ERR_UNSUPPORTED, "hi/lo output needs output channels in multiples of 8");
  ConvParams& p = cl->p;
  memset(&p, 0, sizeof(p));
  p.N = N; p.H = H; p.W = W;
  p.KH = pp.kh; p.KW = pp.kw; p.PH = pp.ph; p.PW = pp.pw;
  p.cin_off = io.cin_off;
  p.cin = pl.cin_pad;
  p.npad = pp.npad;
  p.n_store = pp.n_store;
  p.n_kblocks = ceil_div(p.cin, 64);
  p.w_bytes = pp.w_bytes;
  const int up = pp.phase >= 0 ? 2 : 1;
  // hi/lo pairs are only ever staged: a staging buffer holds the hi tile and then the lo tile (stage_mult = 2)
  const bool tma_out = split || (io.out_kind == kOutBf16 && pp.n_store % 8 == 0 && !g_opt_no_tma_store);
  const int stage_mult = split ? 2 : 1;
  p.store_mode = split ? kStoreBf16Split : tma_out ? kStoreStaged : io.out_kind == kOutBf16 ? kStoreDirect : io.out_kind == kOutF32Planar ? kStoreF32Planar : kStoreF32Nhwc;
  p.stage_row_bytes = tma_out ? pp.n_store * 2 : 0;
  // four tiles in flight in the epilogue when four accumulators fit in TMEM and a warp then owns <= 4 chunks of 8 channels
  p.n_acc = (4 * p.KW * p.npad <= 512 && p.npad <= 32) ? 4 : 2;
  p.n_groups = p.n_acc;
  Tiling tl;
  int rc = CSR_OK;
  const bool has_res = io.r1 || io.r2 || io.gate;
  // Layers over <= 32 input channels (the dense-block parts over x1 / x1,x2) only move those channels: 32- or 64-byte
  // window rows with the matching TMA / UMMA swizzle instead of a whole 64-channel box.  These launches are bound by
  // the bytes the SM can take in per clock, not by MMAs.
  p.box_c = 64;
  if (g_opt_narrow_box && p.n_kblocks == 1) p.box_c = p.cin <= 16 ? 16 : p.cin <= 32 ? 32 : 64;
  // Thin layers (<= 32 output channels: four accumulator buffers) are bound by the per-tile work of the producer and
  // MMA-issuer warps (~110 / ~250 scalar instructions at ~5 clk each), not by MMAs or bytes: give them windows of two M
  // tiles, which halves that work per tile and shrinks the halo from 6/4 to 10/8 rows.
  // A layer of ONE k-block (<= 64 input channels, e.g. the 9x9 input gradient of srcnn.conv1) streams its whole weights as that
  // k-block: two slots never fit, so it keeps the weights resident next to a shallower window ring instead.
  const bool stream_w = pp.stream && p.n_kblocks > 1;
  if (stream_w) {
    p.stream_w = 1;
    p.n_groups = 1;                                        // one staging buffer: two (window + weight k-block) slots of ~96 KB must fit
    p.wkb_bytes = pp.kh * 4 * pp.kw * pp.npad * 32;
    rc = choose_tiling(H, W, pp.kh, pp.kw, 0, p.n_kblocks, p.stage_row_bytes, p.n_groups * stage_mult, &tl, 128, 1, p.wkb_bytes);
    if (!rc && tl.n_slots < 2) rc = fail(CSR_ERR_UNSUPPORTED, "streamed-weight conv: window ring too shallow");
  } else {
    // whole-row tiles for the trunk's one-residual convs (RDB conv5, trunk_conv: conv_tc.cu WR_T), which share a staging buffer if need
    // be.  Not for the RDB3 conv5 with its second residual: with one shared staging buffer its longer epilogue paces the tiles
    // (50.7 -> 66 us per launch at cfg2 on a B200, while the plain conv5 goes 37 -> 35.5 us)
    const bool wr = !split && tma_out && pp.phase < 0 && pp.kh == 3 && pp.kw == 3 && pp.ph == 1 && pp.pw == 1 && io.act == CSR_ACT_NONE &&
                    io.r1 && !io.r2 && !io.gate && p.n_acc == 2 && p.box_c == 64;
    rc = choose_tiling(H, W, pp.kh, pp.kw, p.w_bytes, p.n_kblocks, p.stage_row_bytes, p.n_groups * stage_mult, &tl, p.box_c * 2, 1, 0, wr ? 2 : 0);
  }
  if (!rc && g_opt_tall && p.n_acc == 4 && p.n_groups == 4 && !split) {
    Tiling t2;   // taken unless the second M tile would mostly hang below the image
    if (choose_tiling(H, W, pp.kh, pp.kw, p.w_bytes, p.n_kblocks, p.stage_row_bytes, p.n_groups, &t2, p.box_c * 2, 2) == CSR_OK &&
        t2.eff >= 0.85 * tl.eff && t2.n_slots >= 2) {
      tl = t2;
      p.tall_shift = 1;
      // two issuers x two M tiles fill four accumulators at once: with eight, the next windows' MMAs overlap the
      // epilogue of these four instead of waiting for it
      if (8 * p.KW * p.npad <= 512 && g_opt_eight_acc) p.n_acc = 8;
    }
  }
  if (rc) return rc;
  if (tma_out && p.n_groups == 2 && p.w_bytes < 96 * 1024 && !has_res) {
    // One epilogue group of 16 warps on one tile at a time (two chunks per warp) for the two-accumulator layers with < 96 KB of
    // weights and no residual / gate operand (HRconv, upconv, conv_first, srcnn.conv1): they are epilogue-bound, and 16 warps on
    // one tile shorten its latency chain (-2 % per inference step).  RDB conv5 and the gated input-gradient convs of the backward
    // lose with it: there the single group paces the tile.
    Tiling t1;
    if (choose_tiling(H, W, pp.kh, pp.kw, p.w_bytes, p.n_kblocks, p.stage_row_bytes, stage_mult, &t1, p.box_c * 2) == CSR_OK) {
      tl = t1;
      p.n_groups = 1;
    }
  }
  p.act = io.act;
  p.act_slope = io.act_slope;
  p.n_stage = tl.whole_row ? tl.n_stage : p.n_groups;
  // Early-release epilogue (conv_tc.cu, EARLY_T): wide residual-free layers that run with one 16-warp group.  Two staging
  // buffers; KW <= 2 layers also get four accumulator buffers (4 x KW x 64 <= 512 TMEM columns).
  const bool early_plain = !has_res && p.n_groups == 1 &&
      ((p.KW == 3 && p.PW == 1 && (p.act == 0 || p.act == 1)) || (p.KW == 2 && p.PW <= 1 && p.act == 1) || (p.KW == 1 && p.PW == 0 && p.act == 2));
  if (g_opt_early && early_plain && !split && !p.tall_shift && tma_out && p.npad == 64 && pp.n_store == 64) {
    Tiling te2, te1;
    const bool ok2 = choose_tiling(H, W, pp.kh, pp.kw, p.w_bytes, p.n_kblocks, p.stage_row_bytes, 2, &te2, p.box_c * 2) == CSR_OK;
    const bool ok1 = choose_tiling(H, W, pp.kh, pp.kw, p.w_bytes, p.n_kblocks, p.stage_row_bytes, 1, &te1, p.box_c * 2) == CSR_OK;
    const int want = std::min(2 * p.n_kblocks, 4);
    int stages = 0;
    if (ok2 && te2.n_slots >= want) stages = 2;
    else if (ok1 && (!ok2 || te1.n_slots > te2.n_slots)) stages = 1;
    else if (ok2) stages = 2;
    const Tiling& te = stages == 1 ? te1 : te2;
    if (stages && te.n_slots >= std::min(2, p.n_kblocks + 1)) {
      tl = te;
      p.early = 1;
      p.n_groups = 1;
      p.n_stage = stages;
      if (4 * p.KW * p.npad <= 512) p.n_acc = 4;
    }
  }
  // Hybrid tap fold (conv_tc.cu HYB_T) for the early-release 64-channel 3x3 / 2x2 layers, which are epilogue-bound: the last horizontal
  // tap is its own MMA on an A operand shifted by one pixel and accumulates into the previous tap's columns - a third (half) fewer
  // accumulator columns to read and one shuffle-sum fewer, at 22 % more MMA time.
  if (g_opt_hyb && p.early && ((p.KW == 3 && p.PW == 1) || (p.KW == 2 && p.PW <= 1)) && p.box_c == 64 && !p.stream_w) {
    p.hyb = 1;
    if (4 * (p.KW - 1) * p.npad <= 512) p.n_acc = 4;
  }
  p.SW = tl.SW; p.TH = tl.TH; p.TW = tl.TW;
  p.whole_row = tl.whole_row;
  p.sw_shift = 0;
  while ((1 << p.sw_shift) < p.SW) ++p.sw_shift;
  p.tiles_x = ceil_div(W, p.TW);
  p.tiles_y = ceil_div(H, p.TH << p.tall_shift);          // windows
  p.num_tiles = p.tiles_x * p.tiles_y * N;
  p.tiles_per_img = p.tiles_x * p.tiles_y;
  if ((long long)p.tiles_x * p.tiles_y * N >= (1 << 24) || p.tiles_per_img >= (1 << 16))
    return fail(CSR_ERR_UNSUPPORTED, "too many tiles (%d x %d x %d) for one launch", p.tiles_x, p.tiles_y, N);
  p.magic_img = ((1ull << 40) / (unsigned)p.tiles_per_img) + 1;
  p.magic_row = ((1ull << 40) / (unsigned)p.tiles_x) + 1;
  p.win_rows = tl.win_rows; p.win_bytes = tl.win_bytes; p.slot_bytes = tl.slot_bytes; p.n_slots = tl.n_slots;
  p.win_slot_bytes = (int)align_up(tl.win_bytes, 1024);
  p.stage_bytes = tl.stage_bytes;
  if (split) {
    p.stage_lo_bytes = tl.stage_bytes;
    p.stage_bytes = 2 * tl.stage_bytes;
    p.split_off = io.split_off;
  }
  int cols = 32;
  while (cols < p.n_acc * (p.hyb ? p.KW - 1 : p.KW) * p.npad) cols *= 2;
  if (cols > 512 || p.KW * p.npad > 256) return fail(CSR_ERR_UNSUPPORTED, "KW*npad = %d exceeds the UMMA N / TMEM budget", p.KW * p.npad);
  p.tmem_cols = cols;
  p.trace = g_trace;
  p.trace_cta = g_opt_trace_cta;
  p.use_pdl = g_opt_pdl;
  p.s1 = io.s1; p.s2 = io.s2;
  p.r1 = io.r1; p.r1_C = io.r1_C; p.r1_coff = io.r1_coff + pp.co_lo;
  p.r2 = io.r2; p.r2_C = io.r2_C; p.r2_coff = io.r2_coff + pp.co_lo;
  p.gate = io.gate; p.gate_C = io.gate_C; p.gate_coff = io.gate_coff + pp.co_lo; p.gate_from = io.gate_from - pp.co_lo; p.gate_neg = io.gate_neg;
  if ((io.r1 || io.r2 || io.gate) && up != 1) return fail(CSR_ERR_UNSUPPORTED, "residual / gate operands are not supported on nearest-x2 layers");
  p.out = io.out; p.out_C = io.out_C; p.out_coff = io.out_coff + pp.co_lo;
  p.out_sy = p.out_sx = up;
  p.out_oy = pp.phase >= 0 ? (pp.phase >> 1) : 0;
  p.out_ox = pp.phase >= 0 ? (pp.phase & 1) : 0;
  p.out_H = up * H; p.out_W = up * W;
  cl->w_off = pp.w_off; cl->b_off = pp.b_off;
  if (conv_smem_bytes(p) > (size_t)kSmemLimit) return fail(CSR_ERR_UNSUPPORTED, "conv needs %zu bytes of shared memory", conv_smem_bytes(p));
  return CSR_OK;
}

// ------------------------------------------------------------------------------------------- weight gradient
struct WgradLaunch {
  WgradParams p;
  CUtensorMap tx0, tx1, tg0, tg1;
};

// One vertical tap of one 128-input-channel chunk: x channels [xc0, xc0+128) (beyond the buffer pitch -> zeros), output
// gradients gA channels [gA_c0, +64) and optionally gB channels [gB_c0, +64) as GEMM columns [0,64) / [64,128).
static int build_wgrad(int sms, int N, int H, int W, int KW, int PW, int dy_off, int n_dy, const void* x, int x_C, int xc0, const void* gA, int gA_C,
                       int gA_c0, const void* gB, int gB_C, int gB_c0, int n_cols, float* dacc, long part_stride, int ld_n, WgradLaunch* wl) {
  if (n_cols % 16 || n_cols < 16 || n_cols > 128) return fail(CSR_ERR_UNSUPPORTED, "wgrad: n_cols %d", n_cols);
  if (x_C % 8 || gA_C % 8 || xc0 % 8 || gA_c0 % 8) return fail(CSR_ERR_BAD_ARG, "wgrad: channel pitch/offset must be multiples of 8");
  WgradParams& p = wl->p;
  memset(&p, 0, sizeof(p));
  p.N = N; p.H = H; p.W = W; p.KW = KW; p.PW = PW; p.dy_off = dy_off; p.n_dy = n_dy;
  double best = -1;
  for (int SW = 16; SW <= 32; SW *= 2) {
    const int TW = SW - (KW - 1);
    if (TW < 1) continue;
    const int TH = 128 / SW;
    const double eff = (double)H * W / ((double)ceil_div(H, TH) * ceil_div(W, TW) * 128);
    if (eff > best) { best = eff; p.SW = SW; p.TH = TH; p.TW = TW; }
  }
  if (best < 0) return fail(CSR_ERR_UNSUPPORTED, "wgrad: kernel width %d too large", KW);
  while ((1 << p.sw_shift) < p.SW) ++p.sw_shift;
  p.tiles_x = ceil_div(W, p.TW); p.tiles_y = ceil_div(H, p.TH);
  p.tiles_per_img = p.tiles_x * p.tiles_y;
  p.num_tiles = p.tiles_per_img * N;
  if ((long long)p.tiles_per_img * N >= (1 << 24) || p.tiles_per_img >= (1 << 16)) return fail(CSR_ERR_UNSUPPORTED, "wgrad: too many tiles");
  p.magic_img = ((1ull << 40) / (unsigned)p.tiles_per_img) + 1;
  p.magic_row = ((1ull << 40) / (unsigned)p.tiles_x) + 1;
  p.n_xbox = 2; p.n_gbox = gB ? 2 : 1; p.M = 128; p.n_cols = n_cols;
  p.x_box_bytes = (p.TH + n_dy) * p.SW * 128;
  p.g_box_bytes = p.TH * p.SW * 128;
  p.x_slack = 1024;
  p.stage_bytes = p.n_xbox * (p.x_slack + p.x_box_bytes) + p.n_gbox * p.g_box_bytes;
  p.n_stages = std::min(4, (kSmemLimit - 2048) / p.stage_bytes);
  if (p.n_stages < 1) return fail(CSR_ERR_UNSUPPORTED, "wgrad: stage does not fit shared memory");
  int cols = 32;
  while (cols < n_dy * KW * n_cols) cols *= 2;
  if (cols > 512) return fail(CSR_ERR_UNSUPPORTED, "wgrad: n_dy*KW*n_cols = %d exceeds TMEM", n_dy * KW * n_cols);
  p.tmem_cols = cols;
  p.xc0[0] = xc0; p.xc0[1] = xc0 + 64;
  p.gc0[0] = gA_c0; p.gc0[1] = gB_c0;
  p.dacc = dacc; p.ld_n = ld_n; p.part_stride = part_stride;
  p.n_parts = std::min(p.num_tiles, sms);
  int rc = encode_act_map(&wl->tx0, x, N, H, W, x_C, p.SW, p.TH + n_dy);
  if (rc) return rc;
  wl->tx1 = wl->tx0;
  rc = encode_act_map(&wl->tg0, gA, N, H, W, gA_C, p.SW, p.TH);
  if (rc) return rc;
  wl->tg1 = wl->tg0;
  if (gB) {
    rc = encode_act_map(&wl->tg1, gB, N, H, W, gB_C, p.SW, p.TH);
    if (rc) return rc;
  }
  return CSR_OK;
}

constexpr int kMaxParts = 160;   // >= SM count: per-CTA partial-sum slices
static size_t wgrad_scratch_floats(const LayerSpec& L) {
  const int ekh = L.up2 ? 2 : L.kh, ekw = L.up2 ? 2 : L.ekw();
  const int ld_n = (L.cout + 15) / 16 * 16;
  return (size_t)ekh * kMaxParts * ekw * 128 * ld_n;
}
// vertical taps per launch: as many as fit the 512 TMEM columns
static int wgrad_taps_per_launch(int ekw, int n_cols) { return std::max(1, 512 / (ekw * n_cols)); }

static int encode_phase_map(CUtensorMap* m, const void* base, int N, int H, int W, int C, int phase, int box_w, int box_h) {
  // pixels (2y + a, 2x + b) of an (N, 2H, 2W, C) buffer as an (N, H, W, C) tensor
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return fail(CSR_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  const int a = phase >> 1, b = phase & 1;
  const uint8_t* bp = reinterpret_cast<const uint8_t*>(base) + ((size_t)a * 2 * W + b) * C * 2;
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
  cuuint64_t strides[3] = {(cuuint64_t)2 * C * 2, (cuuint64_t)2 * 2 * W * C * 2, (cuuint64_t)4 * H * W * C * 2};
  cuuint32_t box[4] = {64, (cuuint32_t)box_w, (cuuint32_t)box_h, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<uint8_t*>(bp), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(CSR_ERR_CUDA, "cuTensorMapEncodeTiled (phase view) failed (%d)", (int)r);
  return CSR_OK;
}

// Job mode (wgrad_tc.cuh): layers with many channels and few pixels (the discriminator: 64..512 channels on 130^2..6^2 grids).
// ONE GEMM launch per layer - CTAs own (128-input-channel chunk, output-channel chunk, vertical-tap group) blocks of the weight
// gradient and loop over pixel tiles - instead of one launch (whose 128-pixel K slices each end in ~200 KB of atomics) per block.
static bool wgrad_jobs_applicable(const LayerSpec& L, int N, int H, int W, int sms) {
  if (L.up2 || L.fold || L.kh != L.kw || L.kw > 3) return false;
  const long tiles = (long)N * ceil_div(H, 4) * ceil_div(W, 30);
  return L.cout > 128 || (L.cin > 128 && tiles < 4L * sms);
}
static size_t wgrad_jobs_scratch_floats(const LayerSpec& L) {
  const int n_cols = L.cout >= 128 ? 128 : (L.cout + 15) / 16 * 16;
  const int per = wgrad_taps_per_launch(L.kw, n_cols);
  const long jobs = (long)ceil_div(L.cin, 128) * ceil_div(L.cout, n_cols) * ceil_div(L.kh, per);
  return (size_t)jobs * per * L.kw * 128 * n_cols;
}
// ------------------------------------------------------------------------------------------- launch lists
// One launch of a launch list: a plan's forward or backward (CsrPlan::fwd / bwd) or one layer's weight gradient.  Operands that
// change from call to call are null here and supplied by run_ops from its Bindings; every other pointer is fixed when the op is built.
struct Op {
  enum Kind { kNchw, kConv, kDense, kTapSum, kTapPack, kPackSrcnn, kGcol, kScale, kWgrad, kReduce, kScatter, kScatterJobs, kBias, kBiasWide,
              kBiasPlanar, kMemset } kind;
  ConvLaunch conv;               // kConv; p.out == nullptr: the caller's `out`
  DenseLaunch dense;             // kDense: conv1..conv4 of a dense block, or (backward) its four gated input-gradient convs (rdb_tc.cu)
  WgradLaunch wg;                // kWgrad
  // kScatter / kBias*: which layer's gradient (index into Bindings::dw / db), and how
  int layer = -1, fold = 0, phase = -1, ci0 = 0, ci_n = 0, col0 = 0, ld_n = 0, n_parts = 0, nseg = 1;
  int taps_t = 0;                         // kScatter: columns are taps of a single-output-channel layer (dw[ci][tap])
  int cout = 0, cin = 0, kh = 0, kw = 0;  // kScatter / kScatterJobs: the forward layer's shape; kGcol: taps
  int jobs_co = 0, jobs_dy = 0, per_dy = 0;   // kScatterJobs: the job grid of the kWgrad op before it (WgradParams), job stride in `count`
  int seg_layers[4] = {-1, -1, -1, -1};   // kBias with nseg > 1: one layer per channel segment
  int N = 0, H = 0, W = 0;                // kNchw: the input grid (C channels); kTapSum / kTapPack / kPackSrcnn / kGcol: the HR grid
  float scale = 1.f;
  const void* src = nullptr; void* dst = nullptr;   // src == nullptr: x (kNchw), dL/dout (kGcol, kBiasPlanar)
  long count = 0; int C = 0, coff = 0;
  size_t b_off = 0;                       // kTapSum / kTapPack: conv_last's bias inside the packed blob
};

// What run_ops binds at run time.
struct Bindings {
  const void* packed = nullptr;           // packed weights (kConv, kDense, kTapSum, kTapPack)
  const float* x = nullptr; const float* elev = nullptr; const float* mask = nullptr; float* out = nullptr;
  const float* grad_out = nullptr;        // dL/dout, fp32 planar
  float* const* dw = nullptr; float* const* db = nullptr;   // per layer
  unsigned long long* timeline = nullptr; int timeline_cap = 0;   // csr_debug_set_timeline: launch id = op index
};

static int run_ops(const std::vector<Op>& ops, size_t lo, size_t hi, const Bindings& b, int sms, cudaStream_t s) {
  const uint8_t* pk = reinterpret_cast<const uint8_t*>(b.packed);
  hi = std::min(hi, ops.size());
  for (size_t i = lo; i < hi; ++i) {
    const Op& op = ops[i];
    unsigned long long* tl = (long long)i < b.timeline_cap ? b.timeline : nullptr;
    switch (op.kind) {
      case Op::kNchw:
        CSR_CUDA(launch_nchw_to_nhwc(b.x, op.dst, op.N, op.C, op.H, op.W, 64, 16, s));
        break;
      case Op::kConv: {
        ConvParams p = op.conv.p;
        p.wpk = pk + op.conv.w_off;
        p.bias = reinterpret_cast<const float*>(pk + op.conv.b_off);
        if (p.fuse2) { p.w2 = pk + op.conv.w2_off; p.b2 = p.fuse2 == 1 ? reinterpret_cast<const float*>(pk + op.conv.b2_off) : nullptr; }
        if (!p.out) p.out = b.out;
        if (tl) { p.timeline = tl; p.launch_id = (int)i; }
        int e = launch_conv_tc(p, op.conv.tmap, sms, s);
        if (e) return fail(CSR_ERR_CUDA, "conv launch %zu failed: %s", i, cudaGetErrorString((cudaError_t)e));
        break;
      }
      case Op::kDense: {
        DenseParams p = op.dense.p;
        for (int k = 0; k < p.n_layers; ++k) {
          p.L[k].wpk = pk + op.dense.w_off[k];
          p.L[k].bias = reinterpret_cast<const float*>(pk + op.dense.b_off[k]);
        }
        if (tl) { p.timeline = tl; p.launch_id = (int)i; }
        int e = launch_dense_block(p, op.dense.tmap, sms, s);
        if (e) return fail(CSR_ERR_CUDA, "dense-block launch %zu failed: %s", i, cudaGetErrorString((cudaError_t)e));
        break;
      }
      case Op::kTapSum:
        CSR_CUDA(launch_tap_sum(reinterpret_cast<const float*>(op.src), op.count, reinterpret_cast<const float*>(pk + op.b_off),
                                reinterpret_cast<float*>(op.dst), op.H, op.W, op.count, s));
        break;
      case Op::kTapPack:
        CSR_CUDA(launch_tap_pack(reinterpret_cast<const float*>(op.src), op.count, reinterpret_cast<const float*>(pk + op.b_off), b.elev, b.mask,
                                 op.dst, op.N, op.H, op.W, s));
        break;
      case Op::kPackSrcnn:
        CSR_CUDA(launch_pack_srcnn_in(reinterpret_cast<const float*>(op.src), b.elev, b.mask, op.dst, op.W, op.count, op.C, s));
        break;
      case Op::kGcol:
        CSR_CUDA(launch_gcol_pack(op.src ? op.src : b.grad_out, op.C, op.dst, op.coff, op.H, op.W, op.count, op.kh, op.kw, s));
        break;
      case Op::kScale:
        CSR_CUDA(launch_scale_copy64(op.src, op.C, op.dst, op.coff, op.count, op.scale, s));
        break;
      case Op::kWgrad: {
        int e = launch_wgrad_tc(op.wg.p, op.wg.tx0, op.wg.tx1, op.wg.tg0, op.wg.tg1, sms, s);
        if (e) return fail(CSR_ERR_CUDA, "wgrad launch %zu failed: %s", i, cudaGetErrorString((cudaError_t)e));
        break;
      }
      case Op::kReduce:
        CSR_CUDA(launch_wgrad_reduce(reinterpret_cast<float*>(op.dst), op.count, op.n_parts, op.count, s));
        break;
      case Op::kScatter:
        if (!b.dw[op.layer]) return fail(CSR_ERR_BAD_ARG, "null weight-gradient pointer for layer %d", op.layer);
        CSR_CUDA(launch_wgrad_scatter(reinterpret_cast<const float*>(op.src), op.ld_n, b.dw[op.layer], op.cout, op.cin, op.kh, op.kw, op.fold, op.phase,
                                      op.ci0, op.ci_n, op.col0, op.scale, op.taps_t, s));
        break;
      case Op::kScatterJobs:
        if (!b.dw[op.layer]) return fail(CSR_ERR_BAD_ARG, "null weight-gradient pointer for layer %d", op.layer);
        CSR_CUDA(launch_wgrad_scatter_jobs(reinterpret_cast<const float*>(op.src), b.dw[op.layer], op.cout, op.cin, op.kh, op.kw, op.ld_n, op.jobs_co,
                                           op.jobs_dy, op.per_dy, op.count, op.scale, s));
        break;
      case Op::kBias: {
        float* dbs[4] = {nullptr, nullptr, nullptr, nullptr};
        for (int q = 0; q < op.nseg; ++q) {
          dbs[q] = b.db[op.nseg > 1 ? op.seg_layers[q] : op.layer];
          if (!dbs[q]) return fail(CSR_ERR_BAD_ARG, "null bias-gradient pointer for layer %d", op.layer);
        }
        CSR_CUDA(launch_bias_grad(op.src, op.count, op.C, op.coff, op.cout, op.scale, dbs, op.nseg, s));
        break;
      }
      case Op::kBiasWide:
        if (!b.db[op.layer]) return fail(CSR_ERR_BAD_ARG, "null bias-gradient pointer for layer %d", op.layer);
        CSR_CUDA(launch_bias_grad_wide(op.src, op.count, op.C, op.coff, op.cout / 128, op.scale, b.db[op.layer], s));
        break;
      case Op::kBiasPlanar:
        CSR_CUDA(launch_bias_grad_planar(op.src ? reinterpret_cast<const float*>(op.src) : b.grad_out, op.count, op.scale, b.db[op.layer], s));
        break;
      case Op::kMemset:
        CSR_CUDA(cudaMemsetAsync(op.dst, 0, op.count, s));
        break;
    }
    ++g_launches;
  }
  return CSR_OK;
}

static Op memset_op(void* dst, size_t bytes) {
  Op op;
  op.kind = Op::kMemset; op.dst = dst; op.count = (long)bytes;
  return op;
}

// A pack part without the inputs that only set its per-part launch fields: w_off / b_off (weights, bias), co_lo (out_coff), ph (PH) and
// the row bit a of a sub-pixel phase 2a + b (out_oy).  build_conv is a function of the part, so two parts of the same shape build the
// same launch up to those fields.
static PackPart part_shape(PackPart pp) {
  pp.w_off = pp.b_off = 0;
  pp.co_lo = pp.ph = 0;
  if (pp.phase >= 0) pp.phase &= 1;
  return pp;
}
static_assert(std::has_unique_object_representations_v<PackPart>, "part shapes are compared with memcmp: PackPart must have no padding");

// The conv launches of one layer (all its pack parts), appended to `ops`.  Parts of the same shape go out as ONE launch with the parts
// on gridDim.y (ConvParams::parts) when their per-part fields step by constant strides: the output-channel parts of a wide layer (a
// 512-channel layer over an 8 x 8 map is 8 parts of ~16 tiles: one after the other they would leave nine SMs in ten idle) and, with
// option 34, the two sub-pixel phases of nearest-x2 + conv that share a kernel specialisation (PW = 1 - b; phases a = 0, 1 on
// gridDim.y).  Residual / gate operands are not offset per part, and fp32 outputs keep one launch per part: only residual-free bf16
// layers are merged.  Only the launches that go out are built (csr_conv2d_nhwc is called ~100 times per discriminator step).
static int emit_conv(std::vector<Op>& ops, const PackLayer& pl, int N, int H, int W, const ConvIO& io) {
  const std::vector<PackPart>& parts = pl.parts;
  const bool mergeable = parts.size() > 1 && !io.r1 && !io.r2 && !io.gate && (io.out_kind == kOutBf16 || io.out_kind == kOutBf16Split);
  thread_local std::vector<char> merged;                   // thread_local: no allocation per call
  thread_local std::vector<PackPart> shape;
  merged.assign(mergeable ? parts.size() : 0, 0);
  shape.clear();
  if (mergeable)
    for (const PackPart& q : parts) shape.push_back(part_shape(q));
  auto row = [](const PackPart& q) { return q.phase >= 0 ? q.phase >> 1 : 0; };
  auto steps = [&](const PackPart& a, const PackPart& b, long long d[5]) {
    d[0] = (long long)b.w_off - (long long)a.w_off; d[1] = (long long)b.b_off - (long long)a.b_off;
    d[2] = b.co_lo - a.co_lo; d[3] = b.ph - a.ph; d[4] = row(b) - row(a);
  };
  for (size_t i = 0; i < parts.size(); ++i) {
    if (mergeable && merged[i]) continue;
    Op op;
    op.kind = Op::kConv;
    int rc = build_conv(pl, parts[i], N, H, W, io, &op.conv);
    if (rc) return rc;
    if (mergeable) {
      auto same = [&](size_t j) { return !merged[j] && !memcmp(&shape[i], &shape[j], sizeof(PackPart)); };
      long long d0[5], d[5];
      size_t prev = i, count = 1;
      bool steady = true;
      for (size_t j = i + 1; j < parts.size(); ++j) {
        if (!same(j)) continue;
        steps(parts[prev], parts[j], count == 1 ? d0 : d);
        if (count > 1) steady = steady && !memcmp(d, d0, sizeof(d));
        prev = j;
        ++count;
      }
      if (count > 1 && steady && (g_opt_merge_phases || (!d0[3] && !d0[4]))) {
        for (size_t j = i + 1; j < parts.size(); ++j)
          if (same(j)) merged[j] = 1;
        ConvParams& p = op.conv.p;
        p.parts = (int)count;
        p.part_w_bytes = (int)d0[0]; p.part_b_floats = (int)(d0[1] / (long long)sizeof(float));
        p.part_c = (int)d0[2]; p.part_ph = (int)d0[3]; p.part_oy = (int)d0[4];
      }
    }
    rc = encode_act_map(&op.conv.tmap, io.in, N, H, W, io.in_C, op.conv.p.SW, op.conv.p.win_rows, op.conv.p.box_c);
    if (rc) return rc;
    ops.push_back(op);
  }
  return CSR_OK;
}

// One weight-gradient accumulation group: the GEMM launches `wg` sum into dacc[0, floats).  Option 25 on: dacc is zeroed and the
// GEMMs add into it with red.global.add.v4.f32; off: every CTA writes its own partial slice and a reduce kernel sums the slices.
static void push_acc_group(std::vector<Op>& ops, std::vector<WgradLaunch>& wg, float* dacc, long floats) {
  if (g_opt_wgrad_atomic) ops.push_back(memset_op(dacc, (size_t)floats * sizeof(float)));
  for (WgradLaunch& wl : wg) {
    Op op; op.kind = Op::kWgrad; op.wg = wl; op.wg.p.atomic = g_opt_wgrad_atomic;
    ops.push_back(op);
  }
  if (!g_opt_wgrad_atomic) {
    Op rd; rd.kind = Op::kReduce; rd.dst = dacc; rd.n_parts = wg.back().p.n_parts; rd.count = floats;
    ops.push_back(rd);
  }
}

// Weight (and, with `bias`, bias) gradient of one conv layer, accumulated into Bindings::dw / db [layer] (fp32 OIHW / (cout)):
//   dw += scale * sum_p g[p][co] x[p + tap][ci]   over executed taps; see wgrad_scatter_kernel for fold / phase.
// x: (N,H,W,x_C) bf16 (the layer's INPUT, low resolution for an up2 layer); g: gradient w.r.t. the layer's pre-activation
// output.  For an up2 layer, g is the (2H, 2W) buffer and each phase's pixels are read through a strided view.
static int emit_wgrad(std::vector<Op>& ops, const LayerSpec& L, int layer, int N, int H, int W, const void* x, int x_C, int x_coff, const void* g,
                      int g_C, int g_coff, float scale, bool bias, float* dacc, int sms) {
  const int ld_n = (L.cout + 15) / 16 * 16;
  if (ld_n > 128) return fail(CSR_ERR_UNSUPPORTED, "wgrad: cout %d > 128 needs job mode (a 3x3 or 1x1 layer)", L.cout);
  if (sms > kMaxParts) return fail(CSR_ERR_UNSUPPORTED, "wgrad: %d SMs > %d", sms, kMaxParts);
  const int ecin = L.ecin(), ekh = L.up2 ? 2 : L.kh, ekw = L.up2 ? 2 : L.ekw();
  const long part_stride = (long)ekh * ekw * 128 * ld_n;
  const int per = wgrad_taps_per_launch(ekw, ld_n);
  const void* gB = ld_n > 64 ? g : nullptr;   // output-gradient columns [64, 128) come through a second 64-channel box of the same buffer
  for (int phase = L.up2 ? 0 : -1; phase < (L.up2 ? 4 : 0); ++phase) {
    const int ph = L.up2 ? 1 - (phase >> 1) : L.kh / 2;
    const int pw = L.up2 ? 1 - (phase & 1) : L.ekw() / 2;
    for (int ci0 = 0; ci0 < ecin; ci0 += 128) {
      std::vector<WgradLaunch> wg;
      for (int dy = 0; dy < ekh; dy += per) {
        WgradLaunch wl;
        int rc = build_wgrad(sms, N, H, W, ekw, pw, dy - ph, std::min(per, ekh - dy), x, x_C, x_coff + ci0, g, g_C, g_coff, gB, gB ? g_C : 0,
                             gB ? g_coff + 64 : 0, ld_n, dacc + (size_t)dy * ekw * 128 * ld_n, part_stride, ld_n, &wl);
        if (rc) return rc;
        if (phase >= 0) {
          rc = encode_phase_map(&wl.tg0, g, N, H, W, g_C, phase, wl.p.SW, wl.p.TH);
          if (rc) return rc;
          wl.tg1 = wl.tg0;
        }
        wg.push_back(wl);
      }
      push_acc_group(ops, wg, dacc, part_stride);
      Op sc; sc.kind = Op::kScatter; sc.src = dacc; sc.layer = layer; sc.fold = L.fold; sc.phase = phase; sc.ci0 = ci0; sc.ci_n = std::min(128, ecin - ci0);
      sc.ld_n = ld_n; sc.scale = scale; sc.cout = L.cout; sc.cin = L.cin; sc.kh = L.kh; sc.kw = L.kw;
      ops.push_back(sc);
    }
  }
  if (bias) {
    Op bo; bo.kind = Op::kBias; bo.layer = layer; bo.src = g; bo.count = (long)N * H * W * (L.up2 ? 4 : 1); bo.C = g_C; bo.coff = g_coff;
    bo.cout = L.cout; bo.scale = scale;
    ops.push_back(bo);
  }
  return CSR_OK;
}

// Job mode (wgrad_jobs_applicable): one GEMM launch for the whole layer, its per-job sums scattered into Bindings::dw [layer].
static int emit_wgrad_jobs(std::vector<Op>& ops, const LayerSpec& L, int layer, int N, int H, int W, const void* x, int x_C, int x_coff, const void* g,
                           int g_C, int g_coff, float scale, bool bias, float* scratch, int sms) {
  const int n_cols = L.cout >= 128 ? 128 : (L.cout + 15) / 16 * 16;
  if (L.cout > 128 && L.cout % 128) return fail(CSR_ERR_UNSUPPORTED, "wgrad: cout %d > 128 must be a multiple of 128", L.cout);
  const int per = wgrad_taps_per_launch(L.kw, n_cols);
  Op op; op.kind = Op::kWgrad;
  int rc = build_wgrad(sms, N, H, W, L.kw, L.kw / 2, -(L.kh / 2), std::min(per, L.kh), x, x_C, x_coff, g, g_C, g_coff, n_cols > 64 ? g : nullptr,
                       n_cols > 64 ? g_C : 0, n_cols > 64 ? g_coff + 64 : 0, n_cols, scratch, 0, n_cols, &op.wg);
  if (rc) return rc;
  WgradParams& p = op.wg.p;
  p.jobs_ci = ceil_div(L.cin, 128); p.jobs_co = ceil_div(L.cout, n_cols); p.jobs_dy = ceil_div(L.kh, per);
  p.KH = L.kh; p.PH = L.kh / 2; p.per_dy = per; p.x_coff = x_coff; p.g_coff = g_coff;
  p.job_stride = (long)per * L.kw * 128 * n_cols;
  p.ld_n = n_cols;
  p.atomic = 1;
  const int jobs = p.jobs_ci * p.jobs_co * p.jobs_dy;
  p.splits = std::max(1, std::min(p.num_tiles, sms / jobs));
  ops.push_back(memset_op(scratch, (size_t)jobs * p.job_stride * sizeof(float)));
  ops.push_back(op);
  Op sc; sc.kind = Op::kScatterJobs; sc.src = scratch; sc.layer = layer; sc.cout = L.cout; sc.cin = L.cin; sc.kh = L.kh; sc.kw = L.kw; sc.ld_n = n_cols;
  sc.jobs_co = p.jobs_co; sc.jobs_dy = p.jobs_dy; sc.per_dy = per; sc.count = p.job_stride; sc.scale = scale;
  ops.push_back(sc);
  if (bias) {
    // > 128 output channels (a multiple of 128 here): every 128-channel chunk in one launch
    Op bo; bo.kind = L.cout > 128 ? Op::kBiasWide : Op::kBias; bo.layer = layer; bo.src = g; bo.count = (long)N * H * W; bo.C = g_C; bo.coff = g_coff;
    bo.cout = L.cout; bo.scale = scale;
    ops.push_back(bo);
  }
  return CSR_OK;
}

// ------------------------------------------------------------------------------------------- plan
}  // namespace csr

struct CsrPlan {
  CsrNetDesc net;
  int N, h, w;
  int sms;
  int train = 0;
  std::vector<csr::Op> fwd, bwd;        // forward (op 0: the input conversion) and, in training plans, backward launch lists
  std::vector<size_t> dbg_cat;          // csr_plan_buffer: byte offsets of the concat buffers / HR-tail activations inside the workspace
  size_t dbg_tail[9] = {};              // csr_plan_buffer kinds 1..9: m1, hrA, hrB, hrD, hrE, fea0, t0, hrC, tlast
  struct { size_t gO, gcolB, gT, gP, gQ, gm1, gt0, gcat[3]; } dbg_grad = {};   // kinds 10..17 (training plans)
  int ccat = 0;
  unsigned int* flags = nullptr;        // completion counters of the dense-block launches
  size_t flags_bytes = 0;
  bool fwd_dense = false;               // the forward has dense-block launches: it zeroes `flags` after the input conversion
  int srcnn_pitch = 64;                 // channel pitch of the SRCNN input im2col (27 -> 32 channels) and of srcnn.conv2's output (32 channels):
                                        // 32 in inference plans - the TMA loads promote to whole 128/256-byte L2 lines, so a 64-channel
                                        // pitch doubled the HBM reads of srcnn.conv1 and srcnn.conv3 -, 64 in training plans (the
                                        // weight-gradient GEMMs read 64-channel boxes)
  // CUDA-graph replay (launch-bound batches: a forward is ~180 launches, a training step ~800): the launch sequence is
  // captured once per packed-weight blob with plan-owned staging buffers for every pointer that changes between calls
  struct GraphCache { cudaGraphExec_t exec = nullptr; const void* packed = nullptr; bool failed = false; long launches = 0; int calls = 0; };
  GraphCache g_fwd, g_bwd;
  // segmented backward (gradient all-reduce overlap): segment k runs ops [seg_op[k], seg_op[k+1]) and completes the flat
  // gradient floats [seg_lo[k], seg_hi[k]) (layers finish in reverse order, so the completed part is a growing suffix)
  std::vector<size_t> seg_op, seg_lo, seg_hi;
  std::vector<GraphCache> g_seg;
  float* sx = nullptr; float* selev = nullptr; float* smask = nullptr; float* sout = nullptr;   // staged inputs / output (fp32)
  float* sgout = nullptr; float* sgrad = nullptr;                                                // staged dL/dout, flat gradients
  std::vector<size_t> grad_off;          // per layer: float offset of dW, db inside the flat gradient buffer (2 entries each)
  size_t grad_floats = 0;
};

namespace csr {

// Float offsets of every layer's dW and db inside the flat gradient buffer (2 entries per layer); *total: its size in floats.
static std::vector<size_t> grad_offsets(const std::vector<LayerSpec>& layers, size_t* total) {
  std::vector<size_t> off;
  size_t o = 0;
  for (const LayerSpec& Ls : layers) {
    off.push_back(o); o += align_up((size_t)Ls.cout * Ls.cin * Ls.kh * Ls.kw, 4);
    off.push_back(o); o += align_up((size_t)Ls.cout, 4);
  }
  *total = o;
  return off;
}

struct WsLayout {
  size_t xin, fea0, t0, m1, hrA, hrB, hrC, hrD, hrE, tlast, total;
  size_t sx, selev, smask, sout, sgout, sgrad;   // graph staging
  size_t flags, flags_bytes;                     // dense-block completion counters
  std::vector<size_t> cat;              // 3 rotating concat buffers (inference) or one per RDB + 1 (training: saved state)
  // training only
  size_t gO, gcolB, gT, gP, gQ, gm1, gt0, gtmp, gcat[3], dacc;
  int ccat;
};
static WsLayout ws_layout(const CsrNetDesc& d, int N, int h, int w, int train) {
  WsLayout L;
  const size_t lr = (size_t)N * h * w, mid = lr * 4, hr = lr * 16;
  L.ccat = (int)align_up(d.nf + 4 * d.gc, 64);
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 1024); return o; };
  L.xin = take(lr * 64 * 2);
  L.fea0 = take(lr * 64 * 2);
  const int ncat = train ? 3 * d.nb + 1 : 3;
  for (int i = 0; i < ncat; ++i) L.cat.push_back(take(lr * L.ccat * 2));
  L.t0 = take(lr * 64 * 2);    // trunk_conv + skip
  L.m1 = take(mid * 64 * 2);   // upconv1 output (2h x 2w)
  L.hrA = take(hr * 64 * 2);   // upconv2 output
  L.hrB = take(hr * 64 * 2);   // HRconv output
  L.hrC = take(hr * 64 * 2);   // SRCNN input [out, elev, mask] x 9 horizontal taps
  L.tlast = take(hr * 4);      // conv_last output, fp32 planar
  // dense-block launches: one counter per (block, layer, window); windows are >= 8 rows x 14 columns
  L.flags_bytes = (size_t)3 * d.nb * kDenseMaxLayers * N * ceil_div(h, 8) * ceil_div(w, 14) * sizeof(unsigned int);
  L.flags = take(L.flags_bytes);
  L.sx = take(lr * d.in_channels * 4);
  L.selev = take(hr * 4);
  L.smask = take(hr * 4);
  L.sout = take(hr * 4);
  L.sgout = L.sgrad = 0;
  if (train) {
    L.sgout = take(hr * 4);
    size_t gf = 0;
    grad_offsets(layer_table(d), &gf);
    L.sgrad = take(gf * 4);
    L.hrD = take(hr * 64 * 2); // srcnn.conv1 output (inference: reuses hrA)
    L.hrE = take(hr * 64 * 2); // srcnn.conv2 output (inference: reuses hrB)
    L.gO = take(hr * 32 * 2);  // im2col of dL/dout: 25 taps of srcnn.conv3 (32-channel pitch)
    L.gcolB = take(hr * 16 * 2);  // im2col of dL/d(conv_last output): 9 taps (16-channel pitch)
    L.gT = take(hr * 16 * 2);  // dL/d(conv_last output), channel 0
    L.gP = take(hr * 64 * 2);  // ping-pong gradient maps of the HR tail
    L.gQ = take(hr * 64 * 2);
    L.gm1 = take(mid * 64 * 2);
    L.gt0 = take(lr * 64 * 2);
    L.gtmp = take(lr * 64 * 2);
    for (int i = 0; i < 3; ++i) L.gcat[i] = take(lr * L.ccat * 2);
    L.dacc = take((size_t)9 * kMaxParts * 128 * 128 * 4);   // per-CTA partial sums of the weight-gradient GEMMs
  } else {
    L.hrD = L.hrA; L.hrE = L.hrB;
    L.gO = L.gcolB = L.gT = L.gP = L.gQ = L.gm1 = L.gt0 = L.gtmp = L.dacc = 0;
    L.gcat[0] = L.gcat[1] = L.gcat[2] = 0;
  }
  L.total = off;
  return L;
}

// The buffers of a WsLayout inside one workspace (the training-only ones point at its start in inference plans).
struct WsPtrs {
  void *xin, *fea0, *t0, *m1, *hrA, *hrB, *hrC, *hrD, *hrE, *gO, *gcolB, *gT, *gP, *gQ, *gm1, *gt0, *gcat[3];
  std::vector<void*> cat;
  float *tlast, *dacc;
};
static WsPtrs ws_carve(const WsLayout& L, void* ws) {
  uint8_t* b = reinterpret_cast<uint8_t*>(ws);
  WsPtrs p;
  p.xin = b + L.xin; p.fea0 = b + L.fea0; p.t0 = b + L.t0; p.m1 = b + L.m1; p.hrA = b + L.hrA; p.hrB = b + L.hrB; p.hrC = b + L.hrC;
  p.hrD = b + L.hrD; p.hrE = b + L.hrE; p.gO = b + L.gO; p.gcolB = b + L.gcolB; p.gT = b + L.gT; p.gP = b + L.gP; p.gQ = b + L.gQ;
  p.gm1 = b + L.gm1; p.gt0 = b + L.gt0;
  for (int i = 0; i < 3; ++i) p.gcat[i] = b + L.gcat[i];
  for (size_t o : L.cat) p.cat.push_back(b + o);
  p.tlast = reinterpret_cast<float*>(b + L.tlast); p.dacc = reinterpret_cast<float*>(b + L.dacc);
  return p;
}

static ConvIO io_of(const void* in, int in_C, void* out, int out_C, int out_coff, int act) {
  ConvIO io;
  io.in = in; io.in_C = in_C; io.out = out; io.out_C = out_C; io.out_coff = out_coff; io.act = act;
  return io;
}

// conv1..conv4 of one gc = 16 dense block as one persistent launch (rdb_tc.cu).  `packs` / `li`: pack layout and the index of
// the block's conv1 in it.  Returns CSR_ERR_UNSUPPORTED when no tile shape fits - the caller then falls back to four launches.
static int build_dense(const std::vector<PackLayer>& packs, int li, int N, int H, int W, void* buf, int C, int nf, int gc, unsigned int* flags,
                       DenseLaunch* dl, const void* gate = nullptr, int gate_C = 0) {
  DenseParams& p = dl->p;
  memset(&p, 0, sizeof(p));
  if (gc != 16 || C % 8) return fail(CSR_ERR_UNSUPPORTED, "dense-block kernel: gc must be 16");
  p.N = N; p.H = H; p.W = W; p.n_layers = 4; p.C = C; p.buf = buf; p.flags = flags; p.use_pdl = g_opt_pdl;
  // forward: x_{k+1} = lrelu(conv_{k+1}(...)).  backward (gate given): layer k = the gated gradient of x_{4-k}, gate = x_{4-k} of the
  // forward concat buffer (channels nf + (3-k) gc ...), no activation
  p.act = gate ? 0 : 1; p.gate = gate; p.gate_C = gate_C; p.gate_neg = 0.2f;
  int wmax = 0;
  for (int k = 0; k < 4; ++k) {
    const PackLayer& pl = packs[li + k];
    if (pl.parts.size() != 1 || pl.parts[0].npad != 16 || pl.parts[0].kh != 3 || pl.parts[0].kw != 3 || pl.cin_pad != nf + k * gc)
      return fail(CSR_ERR_UNSUPPORTED, "dense-block kernel: unexpected pack layout");
    p.L[k].ksteps = pl.cin_pad / 16;
    p.L[k].n_kblocks = ceil_div(pl.cin_pad, 64);
    p.L[k].w_bytes = pl.parts[0].w_bytes;
    p.L[k].out_coff = nf + k * gc;
    p.L[k].gate_coff = nf + (3 - k) * gc;
    dl->w_off[k] = pl.parts[0].w_off; dl->b_off[k] = pl.parts[0].b_off;
    wmax = std::max(wmax, pl.parts[0].w_bytes);
  }
  p.wbuf_bytes = (int)align_up(wmax, 1024);
  Tiling tl;
  int rc = choose_tiling(H, W, 3, 3, 2 * p.wbuf_bytes, 2, 32, 4, &tl, 128, 2, 0, 1);
  if (rc) return rc;
  if (tl.n_slots < 3) return fail(CSR_ERR_UNSUPPORTED, "dense-block kernel: window ring too shallow");
  p.SW = tl.SW; p.TH = tl.TH; p.TW = tl.TW; p.whole_row = tl.whole_row;
  while ((1 << p.sw_shift) < p.SW) ++p.sw_shift;
  p.tiles_x = ceil_div(W, p.TW); p.tiles_y = ceil_div(H, 2 * p.TH);
  p.tiles_per_img = p.tiles_x * p.tiles_y;
  p.num_tiles = p.tiles_per_img * N;
  if ((long long)p.tiles_per_img * N >= (1 << 24) || p.tiles_per_img >= (1 << 16)) return fail(CSR_ERR_UNSUPPORTED, "dense-block kernel: too many windows");
  p.magic_img = ((1ull << 40) / (unsigned)p.tiles_per_img) + 1;
  p.magic_row = ((1ull << 40) / (unsigned)p.tiles_x) + 1;
  p.win_bytes = tl.win_bytes; p.slot_bytes = tl.slot_bytes; p.n_slots = tl.n_slots;
  p.stage_bytes = (int)align_up((size_t)p.TH * p.TW * 32, 1024);
  if (dense_smem_bytes(p) > (size_t)kSmemLimit) return fail(CSR_ERR_UNSUPPORTED, "dense-block kernel needs %zu bytes of shared memory", dense_smem_bytes(p));
  return encode_act_map(&dl->tmap, buf, N, H, W, C, p.SW, 2 * p.TH + 2, 64);
}

static bool dense_enabled(const CsrNetDesc& d) { return g_opt_dense && d.gc == 16; }

// The four convs of dense block j (concat buffer `buf`, pack layers li..li+3) as ONE persistent launch with tile-level
// dependencies between the layers: conv1..conv4 of the forward, or with `gate` the backward's four gated input-gradient convs.
// False: run them as one launch per layer (option 27 off, no tile shape fits, or fewer than option 31's windows per SM).
static bool try_dense(const CsrPlan* P, const std::vector<PackLayer>& packs, int li, int j, void* buf, const void* gate, Op* op) {
  const CsrNetDesc& d = P->net;
  if (!dense_enabled(d)) return false;
  const size_t per_block = (size_t)kDenseMaxLayers * P->N * ceil_div(P->h, 8) * ceil_div(P->w, 14);   // ws_layout's flags
  op->kind = Op::kDense;
  return build_dense(packs, li, P->N, P->h, P->w, buf, P->ccat, d.nf, d.gc, P->flags + (size_t)j * per_block, &op->dense, gate, gate ? P->ccat : 0) ==
             CSR_OK &&
         (size_t)op->dense.p.num_tiles * kDenseMaxLayers <= per_block && op->dense.p.num_tiles >= g_opt_dense_min * P->sms;
}

// The forward launch list, in launch order.
static int plan_build(CsrPlan* P, const WsPtrs& ws, const std::vector<LayerSpec>& layers) {
  const CsrNetDesc& d = P->net;
  const int N = P->N, h = P->h, w = P->w;
  auto cat = [&](int j) -> void* { return ws.cat[P->train ? j : j % 3]; };
  size_t total = 0;
  const std::vector<PackLayer> packs = pack_layout(fwd_exec_table(d, layers), &total);
  const int C = P->ccat, nf = d.nf, gc = d.gc;
  std::vector<Op>& ops = P->fwd;
  {
    Op op; op.kind = Op::kNchw; op.dst = ws.xin; op.N = N; op.C = d.in_channels; op.H = h; op.W = w;
    ops.push_back(op);
  }
  int li = 0;
  auto add = [&](int H, int W, const ConvIO& io, bool advance = true) -> int {
    const int rc = emit_conv(ops, packs[li], N, H, W, io);
    if (advance) ++li;
    return rc;
  };
  int rc;
  // conv_first (esrgan.py:90) has two consumers: the first RRDB (reads x from its concat buffer) and the trunk skip-add
  // 33 layers later.  The layer is tiny (K = 16), so it is simply run into both places.
  const size_t c0 = ops.size();
  rc = add(h, w, io_of(ws.xin, 64, cat(0), C, 0, CSR_ACT_NONE), false);
  if (rc) return rc;
  ConvParams& f = ops[c0].conv.p;
  if (ops.size() == c0 + 1 && f.early && f.store_mode == kStoreStaged && f.KW == 3 && f.act == 0 && !f.r1) {
    // ... with the early-release epilogue the staged tile is simply stored twice (conv_tc.cu, out_dup)
    f.out_dup = ws.fea0; f.dup_C = 64; f.dup_coff = 0;
    ++li;
  } else {
    ops.resize(c0);
    rc = add(h, w, io_of(ws.xin, 64, ws.fea0, 64, 0, CSR_ACT_NONE), false);
    if (rc) return rc;
    rc = add(h, w, io_of(ws.xin, 64, cat(0), C, 0, CSR_ACT_NONE));
    if (rc) return rc;
  }
  for (int i = 0; i < d.nb; ++i) {
    // RRDB i: its input x lives in channels [0,nf) of concat buffer 3i.  Inference rotates three buffers A->B->C->A, so
    // A's x survives until RDB3's epilogue reads it as the RRDB residual and overwrites it in place; training keeps one
    // buffer per RDB (the saved activations of the backward pass).
    for (int r = 0; r < 3; ++r) {
      const int j = 3 * i + r;
      void* src = cat(j);
      void* dst = P->train ? cat(j + 1) : (r < 2 ? cat(j + 1) : cat(3 * i));
      Op dop;
      if (try_dense(P, packs, li, j, src, nullptr, &dop)) {
        ops.push_back(dop);
        P->fwd_dense = true;
        li += 4;
      } else {
        for (int k = 1; k <= 4; ++k) {
          // x_k = lrelu(conv_k(cat(x, x1..x_{k-1})))  written into its concat slice  (esrgan.py:33-36)
          rc = add(h, w, io_of(src, C, src, C, nf + (k - 1) * gc, CSR_ACT_LRELU02));
          if (rc) return rc;
        }
      }
      // x5*0.2 + x  (esrgan.py:37-38); RDB3 additionally applies the RRDB residual out*0.2 + x_rrdb (esrgan.py:54)
      ConvIO io = io_of(src, C, dst, C, 0, CSR_ACT_NONE);
      io.r1 = src; io.r1_C = C; io.s1 = 0.2f;
      if (r == 2) { io.r2 = cat(3 * i); io.r2_C = C; io.s2 = 0.2f; }
      rc = add(h, w, io);
      if (rc) return rc;
    }
  }
  void* trunk_out = P->train ? cat(3 * d.nb) : cat(0);
  // trunk_conv + skip (esrgan.py:91-92)
  {
    ConvIO io = io_of(trunk_out, C, ws.t0, 64, 0, CSR_ACT_NONE);
    io.r1 = ws.fea0; io.r1_C = 64; io.s1 = 1.f;
    rc = add(h, w, io);
    if (rc) return rc;
  }
  // lrelu(upconv1(nearest x2)) and lrelu(upconv2(nearest x2)) (esrgan.py:94,97): four sub-pixel phases each
  rc = add(h, w, io_of(ws.t0, 64, ws.m1, 64, 0, CSR_ACT_LRELU02));
  if (rc) return rc;
  rc = add(2 * h, 2 * w, io_of(ws.m1, 64, ws.hrA, 64, 0, CSR_ACT_LRELU02));
  if (rc) return rc;
  const int H = 4 * h, W = 4 * w;
  rc = add(H, W, io_of(ws.hrA, 64, ws.hrB, 64, 0, CSR_ACT_LRELU02));  // HRconv (esrgan.py:99)
  if (rc) return rc;
  // conv_last -> fp32 planar temp; then [out, elev, mask] is packed (with srcnn.conv1's horizontal window) into hrC
  P->srcnn_pitch = P->train ? 64 : 32;
  const int sp = P->srcnn_pitch;
  bool tap_pack = false;
  {
    // Inference: HRconv's 64-channel output never reaches memory - its fused epilogue writes the nine tap planes of conv_last (second
    // MMA over the staged tile, conv_tc.cu FUSE_T = 2) into hrB and tap_sum_kernel adds the shifted taps + bias into tlast.
    ConvLaunch& hc = ops.back().conv;
    const PackLayer& pt = packs.back();                          // "conv_last.taps" (fwd_exec_table)
    bool fused = false;
    if ((g_opt_fuse_tail & 2) && !P->train && hc.p.early && hc.p.KW == 3 && hc.p.PW == 1 && hc.p.npad == 64 && hc.p.stage_row_bytes == 128 &&
        pt.parts.size() == 1 && pt.parts[0].npad == 16 && pt.parts[0].w_bytes == 2048 && pt.cin_pad == 64) {
      ConvParams q = hc.p;
      q.fuse2 = 2; q.w2_bytes = pt.parts[0].w_bytes; q.n2 = 9; q.out2 = ws.hrB; q.out2_plane = (long long)N * H * W;
      if (q.hyb) q.n_acc = 2;                                  // hybrid fold: 2 x 128 + 16 columns (four accumulators would fill TMEM)
      int cols = 32;
      while (cols < q.n_acc * (q.hyb ? 2 : q.KW) * q.npad + 16) cols *= 2;
      q.tmem_cols = cols;
      if (cols <= 512 && conv_smem_bytes(q) <= (size_t)kSmemLimit && (size_t)9 * N * H * W * sizeof(float) <= (size_t)N * H * W * 64 * 2) {
        hc.p = q;
        hc.w2_off = pt.parts[0].w_off;
        // option 36: the tap sum and the SRCNN input im2col in one pass (tap_pack_kernel)
        tap_pack = g_opt_tap_pack != 0;
        Op ts; ts.kind = tap_pack ? Op::kTapPack : Op::kTapSum;
        ts.src = ws.hrB; ts.dst = tap_pack ? ws.hrC : (void*)ws.tlast; ts.count = (long)N * H * W; ts.N = N; ts.H = H; ts.W = W;
        ts.b_off = packs[li].parts[0].b_off;                     // conv_last's own bias
        ops.push_back(ts);
        ++li;                                                    // conv_last has no conv launch
        fused = true;
      }
    }
    if (!fused) {
      ConvIO io = io_of(ws.hrB, 64, ws.tlast, 1, 0, CSR_ACT_NONE);
      io.out_kind = kOutF32Planar;
      rc = add(H, W, io);
      if (rc) return rc;
    }
  }
  if (!tap_pack) {
    Op op; op.kind = Op::kPackSrcnn; op.src = ws.tlast; op.dst = ws.hrC; op.W = W; op.count = (long)N * H * W; op.C = sp;
    ops.push_back(op);
  }
  rc = add(H, W, io_of(ws.hrC, sp, ws.hrD, 64, 0, CSR_ACT_RELU));     // srcnn.conv1 (9x1 folded)
  if (rc) return rc;
  {
    // Inference: srcnn.conv2 (1x1, 64 -> 32, ReLU) runs inside srcnn.conv1's epilogue as a second MMA over the staged tile; the
    // 64-channel HR map is never written (conv_tc.cu FUSE_T).  Training plans keep both layers (the backward needs the intermediate).
    ConvLaunch& c1 = ops.back().conv;
    const PackLayer& p2 = packs[li];
    bool fused = false;
    if ((g_opt_fuse_tail & 1) && !P->train && c1.p.early && c1.p.KW == 1 && c1.p.PW == 0 && c1.p.npad == 64 && c1.p.stage_row_bytes == 128 &&
        p2.parts.size() == 1 && p2.parts[0].npad == 32 && p2.parts[0].w_bytes == 4096 && p2.cin_pad == 64 && sp % 8 == 0) {
      ConvParams q = c1.p;
      q.fuse2 = 1; q.w2_bytes = p2.parts[0].w_bytes; q.n2 = 32; q.out2 = ws.hrE; q.out2_C = sp; q.out2_coff = 0;
      int cols = 32;
      while (cols < q.n_acc * q.KW * q.npad + 32) cols *= 2;
      q.tmem_cols = cols;
      if (cols <= 512 && conv_smem_bytes(q) <= (size_t)kSmemLimit) {
        c1.p = q;
        c1.w2_off = p2.parts[0].w_off; c1.b2_off = p2.parts[0].b_off;
        ++li;                                                    // srcnn.conv2 has no launch of its own
        fused = true;
      }
    }
    if (!fused) {
      rc = add(H, W, io_of(ws.hrD, 64, ws.hrE, sp, 0, CSR_ACT_RELU));   // srcnn.conv2 1x1
      if (rc) return rc;
    }
  }
  ConvIO io = io_of(ws.hrE, sp, nullptr, 1, 0, CSR_ACT_NONE);    // srcnn.conv3 5x5 -> the caller's output tensor (bound by run_ops)
  io.out_kind = kOutF32Planar;
  return add(H, W, io);
}

// ------------------------------------------------------------------------------------------- backward plan
// Backward layer table: one input-gradient conv per forward layer that needs it, in the order they are packed.
//   index 3*nb*5 ... see bwd_layer_table(); `src` = forward layer index whose OIHW weight is packed transposed.
static int fwd_index_rdb(int i, int r, int k) { return 1 + (i * 3 + r) * 5 + (k - 1); }   // conv_first is layer 0

static std::vector<LayerSpec> bwd_layer_table(const CsrNetDesc& d, const std::vector<LayerSpec>& f) {
  std::vector<LayerSpec> v;
  auto T = [&](int src, float wscale, int up2 = 0) {
    LayerSpec L = f[src];
    LayerSpec t;
    t.name = L.name + ".dgrad";
    t.cout = L.cin; t.cin = L.cout; t.kh = L.kh; t.kw = L.kw;
    t.fold = 0; t.up2 = up2; t.transposed = 1; t.wscale = wscale; t.src = src;
    v.push_back(t);
  };
  const int base_tail = 1 + d.nb * 15;                    // trunk_conv
  // order of use in csr_plan_backward: srcnn.conv3, conv2, conv1, conv_last, HRconv, upconv2, upconv1, trunk_conv, RDBs reversed
  auto C1 = [&](int src) {                                // cout == 1 layer: d/dx = 1x1 conv over the output-gradient im2col
    LayerSpec L = f[src];
    LayerSpec t;
    t.name = L.name + ".dgrad_cols";
    t.cout = L.cin; t.cin = L.kh * L.kw; t.kh = t.kw = 1; t.transposed = 0; t.src = src;   // (1,cin,KH,KW) read as (cin,taps,1,1)
    v.push_back(t);
  };
  C1(base_tail + 7);                                      // srcnn.conv3
  T(base_tail + 6, 1.f);                                  // srcnn.conv2
  T(base_tail + 5, 1.f);                                  // srcnn.conv1 (un-folded 9x9 transposed; only d/d(out) = channel 0 is used)
  C1(base_tail + 4);                                      // conv_last
  T(base_tail + 3, 1.f);                                  // HRconv
  T(base_tail + 2, 1.f, 1);                               // upconv2 (four transposed sub-pixel phases)
  T(base_tail + 1, 1.f, 1);                               // upconv1
  T(base_tail + 0, 1.f);                                  // trunk_conv
  // Dense blocks, mirrored: with the gradient concat [g_y | g4 | g3 | g2 | g1] (g_y = gradient of the block output, g_k =
  // gated gradient of x_k), the gradient of x_s is ONE conv over [g_y | g4 .. g_{s+1}] whose input-channel blocks come
  // from conv5 (x0.2: out = x5*0.2 + x), conv4, ..., conv_{s+1}, each restricted to its input-channel slice of x_s.
  for (int i = d.nb - 1; i >= 0; --i)
    for (int r = 2; r >= 0; --r)
      for (int sidx = 4; sidx >= 0; --sidx) {             // x4, x3, x2, x1, then x (sidx 0)
        LayerSpec t;
        t.name = f[fwd_index_rdb(i, r, 5)].name + ".dgrad_x" + std::to_string(sidx);
        t.cout = sidx ? d.gc : d.nf;
        t.cin = d.nf + (4 - sidx) * d.gc;
        t.kh = t.kw = 3; t.transposed = 1; t.src = fwd_index_rdb(i, r, 5);
        const int slice_off = sidx ? d.nf + (sidx - 1) * d.gc : 0;       // x_s inside the forward concat
        t.blocks.push_back({fwd_index_rdb(i, r, 5), 0, d.nf, slice_off, d.nf + 4 * d.gc, 0.2f});
        for (int j = 4; j > sidx; --j)
          t.blocks.push_back({fwd_index_rdb(i, r, j), d.nf + (4 - j) * d.gc, d.gc, slice_off, d.nf + (j - 1) * d.gc, 1.f});
        v.push_back(t);
      }
  return v;
}

static int bwd_build(CsrPlan* P, const WsPtrs& ws, const std::vector<LayerSpec>& F) {
  const CsrNetDesc& d = P->net;
  const int N = P->N, h = P->h, w = P->w, H = 4 * h, W = 4 * w;
  float* dacc = ws.dacc;
  const std::vector<LayerSpec> B = bwd_layer_table(d, F);
  size_t total = 0;
  const std::vector<PackLayer> packs = pack_layout(B, &total);
  const int C = P->ccat, nf = d.nf, gc = d.gc;
  const int base_tail = 1 + d.nb * 15;
  int bi = 0;                                             // next backward layer
  std::vector<Op>& ops = P->bwd;

  // the parts of backward layer bi
  auto dgrad = [&](int Hh, int Ww, const ConvIO& io, const void* phase_src = nullptr) -> int {
    const PackLayer& pl = packs[bi];
    if (!B[bi++].up2) return emit_conv(ops, pl, N, Hh, Ww, io);
    for (const PackPart& pp : pl.parts) {
      Op op;
      op.kind = Op::kConv;
      // phases accumulate into the same low-resolution gradient: first writes, later ones add, the last one gates
      ConvIO io2 = io;
      if (pp.phase > 0) { io2.r1 = io.out; io2.r1_C = io.out_C; io2.r1_coff = io.out_coff; io2.s1 = 1.f; }
      if (pp.phase < 3) io2.gate = nullptr;
      // build as a plain (non-up2) conv on the low-resolution grid: output view is dense, INPUT view is the strided phase
      PackPart q = pp;
      q.phase = -1;
      int rc = build_conv(pl, q, N, Hh, Ww, io2, &op.conv);
      if (rc) return rc;
      rc = encode_phase_map(&op.conv.tmap, phase_src, N, Hh, Ww, io.in_C, pp.phase, op.conv.p.SW, op.conv.p.win_rows);
      if (rc) return rc;
      ops.push_back(op);
    }
    return CSR_OK;
  };
  auto wgrad_plain = [&](int layer, int Hh, int Ww, const void* x, int x_C, int x_coff, const void* g, int g_C, int g_coff, float scale) -> int {
    return emit_wgrad(ops, F[layer], layer, N, Hh, Ww, x, x_C, x_coff, g, g_C, g_coff, scale, true, dacc, P->sms);
  };
  // weight gradient of a single-output-channel layer as ONE 1x1 GEMM: x (cin channels) against the im2col of its output
  // gradient (taps as columns); the scatter writes dw[ci][tap]
  auto wgrad_cols = [&](int layer, int Hh, int Ww, const void* x, int x_C, const void* gcol, int gcol_C) -> int {
    const LayerSpec& Ls = F[layer];
    const int ntaps = Ls.kh * Ls.kw;
    const int ld_n = (ntaps + 15) / 16 * 16;
    const long part_stride = (long)128 * ld_n;
    for (int ci0 = 0; ci0 < Ls.cin; ci0 += 128) {
      std::vector<WgradLaunch> wg(1);
      int rc = build_wgrad(P->sms, N, Hh, Ww, 1, 0, 0, 1, x, x_C, ci0, gcol, gcol_C, 0, nullptr, 0, 0, ld_n, dacc, part_stride, ld_n, &wg[0]);
      if (rc) return rc;
      push_acc_group(ops, wg, dacc, part_stride);
      Op sc; sc.kind = Op::kScatter; sc.src = dacc; sc.layer = layer; sc.ci0 = ci0; sc.ci_n = std::min(128, Ls.cin - ci0); sc.ld_n = ld_n;
      sc.taps_t = ntaps; sc.cout = ntaps; sc.cin = Ls.cin; sc.kh = sc.kw = 1;
      ops.push_back(sc);
    }
    return CSR_OK;
  };
  auto gated = [&](ConvIO io, const void* gate, int gate_C, int gate_coff, int gate_from, float neg) {
    io.gate = gate; io.gate_C = gate_C; io.gate_coff = gate_coff; io.gate_from = gate_from; io.gate_neg = neg;
    return io;
  };

  int rc;
  // completion counters of the dense-block launches of the backward (the forward zeroed and used the same region)
  if (dense_enabled(d)) ops.push_back(memset_op(P->flags, P->flags_bytes));
  // ---- SRCNN tail (srcnn.py:13-18) -------------------------------------------------------------------------------
  // srcnn.conv3 (32 -> 1, 5x5): im2col of dL/dout (25 taps as channels) makes both of its gradients 1x1 GEMMs
  auto gcol = [&](const void* src, int src_C, void* dst, int dst_C, int k) {
    Op op; op.kind = Op::kGcol; op.src = src; op.C = src_C; op.dst = dst; op.coff = dst_C; op.kh = op.kw = k;
    op.H = H; op.W = W; op.count = (long)N * H * W;
    ops.push_back(op);
  };
  gcol(nullptr, 0, ws.gO, 32, 5);
  rc = wgrad_cols(base_tail + 7, H, W, ws.hrE, 64, ws.gO, 32);
  if (rc) return rc;
  { Op bo; bo.kind = Op::kBiasPlanar; bo.layer = base_tail + 7; bo.count = (long)N * H * W; ops.push_back(bo); }
  rc = dgrad(H, W, gated(io_of(ws.gO, 32, ws.gP, 64, 0, CSR_ACT_NONE), ws.hrE, 64, 0, 0, 0.f));  // -> d/d relu(conv2) * relu'
  if (rc) return rc;
  rc = wgrad_plain(base_tail + 6, H, W, ws.hrD, 64, 0, ws.gP, 64, 0, 1.f);                  // srcnn.conv2
  if (rc) return rc;
  rc = dgrad(H, W, gated(io_of(ws.gP, 64, ws.gQ, 64, 0, CSR_ACT_NONE), ws.hrD, 64, 0, 0, 0.f));
  if (rc) return rc;
  rc = wgrad_plain(base_tail + 5, H, W, ws.hrC, 64, 0, ws.gQ, 64, 0, 1.f);                  // srcnn.conv1 (folded 9x1 over 27 ch)
  if (rc) return rc;
  rc = dgrad(H, W, io_of(ws.gQ, 64, ws.gT, 16, 0, CSR_ACT_NONE));                           // d/d[out, elev, mask]; channel 0 is used
  if (rc) return rc;
  // ---- conv_last, HRconv (esrgan.py:99) ----------------------------------------------------------------------------
  gcol(ws.gT, 16, ws.gcolB, 16, 3);
  rc = wgrad_cols(base_tail + 4, H, W, ws.hrB, 64, ws.gcolB, 16);
  if (rc) return rc;
  { Op bo; bo.kind = Op::kBias; bo.layer = base_tail + 4; bo.src = ws.gT; bo.count = (long)N * H * W; bo.C = 16; bo.coff = 0; bo.cout = 1;
    ops.push_back(bo); }
  rc = dgrad(H, W, gated(io_of(ws.gcolB, 16, ws.gP, 64, 0, CSR_ACT_NONE), ws.hrB, 64, 0, 0, 0.2f));
  if (rc) return rc;
  rc = wgrad_plain(base_tail + 3, H, W, ws.hrA, 64, 0, ws.gP, 64, 0, 1.f);
  if (rc) return rc;
  rc = dgrad(H, W, gated(io_of(ws.gP, 64, ws.gQ, 64, 0, CSR_ACT_NONE), ws.hrA, 64, 0, 0, 0.2f));
  if (rc) return rc;
  // ---- upconv2 / upconv1 (esrgan.py:94,97): nearest-x2 + conv, transposed phase by phase ---------------------------
  rc = wgrad_plain(base_tail + 2, 2 * h, 2 * w, ws.m1, 64, 0, ws.gQ, 64, 0, 1.f);
  if (rc) return rc;
  rc = dgrad(2 * h, 2 * w, gated(io_of(ws.gQ, 64, ws.gm1, 64, 0, CSR_ACT_NONE), ws.m1, 64, 0, 0, 0.2f), ws.gQ);
  if (rc) return rc;
  rc = wgrad_plain(base_tail + 1, h, w, ws.t0, 64, 0, ws.gm1, 64, 0, 1.f);
  if (rc) return rc;
  rc = dgrad(h, w, io_of(ws.gm1, 64, ws.gt0, 64, 0, CSR_ACT_NONE), ws.gm1);
  if (rc) return rc;
  // ---- trunk_conv + skip (esrgan.py:91-92): gt0 is also the skip-path gradient of conv_first's output --------------
  rc = wgrad_plain(base_tail + 0, h, w, ws.cat[3 * d.nb], C, 0, ws.gt0, 64, 0, 1.f);
  if (rc) return rc;
  int Pb = 0;                                             // gcat buffer whose channels [0,64) hold dL/d(RRDB output)
  rc = dgrad(h, w, io_of(ws.gt0, 64, ws.gcat[Pb], C, 0, CSR_ACT_NONE));
  if (rc) return rc;
  // ---- RRDB trunk, reversed (esrgan.py:32-38, 50-54) ----------------------------------------------------------------
  // Per dense block one gradient concat buffer Gb = [g_y (64) | g4 | g3 | g2 | g1] (bwd_layer_table): four narrow convs
  // fill the slices (each gated by the LeakyReLU derivative of its forward activation), one wide conv produces the
  // gradient of the block input (+ identity path) into the NEXT block-to-process's Gb[0:64].  Mirrors the forward cost.
  for (int i = d.nb - 1; i >= 0; --i) {
    const int Qb = (Pb + 1) % 3, Rb = (Pb + 2) % 3;
    // out = RDB3_out*0.2 + x_rrdb: the gradient entering RDB3 is 0.2*G  ->  Gb(RDB3)[0:64]
    { Op op; op.kind = Op::kScale; op.src = ws.gcat[Pb]; op.C = C; op.dst = ws.gcat[Qb]; op.coff = C; op.count = (long)N * h * w; op.scale = 0.2f;
      ops.push_back(op); }
    const int gbuf[3] = {Qb, Rb, Qb};                     // Gb of RDB3, RDB2, RDB1
    const int xout[3] = {Rb, Qb, Rb};                     // where each block's input gradient goes: the next Gb[0:64]
    for (int r = 2; r >= 0; --r) {
      const int j = 3 * i + r;
      void* Gb = ws.gcat[gbuf[2 - r]];
      void* Xo = ws.gcat[xout[2 - r]];
      Op dop;
      if (try_dense(P, packs, bi, j, Gb, ws.cat[j], &dop)) {
        ops.push_back(dop);
        bi += 4;
      } else {
        for (int sidx = 4; sidx >= 1; --sidx) {
          // g_s = lrelu'(x_s) * conv_T([g_y | g4 .. g_{s+1}])  ->  Gb slice of x_s
          rc = dgrad(h, w, gated(io_of(Gb, C, Gb, C, nf + (4 - sidx) * gc, CSR_ACT_NONE), ws.cat[j], C, nf + (sidx - 1) * gc, 0, 0.2f));
          if (rc) return rc;
        }
      }
      // weight gradients of the whole dense block as ONE GEMM per vertical tap (gc = 16): x = the block's forward concat
      // buffer (128 ch), g columns [0,64) = [g4 g3 g2 g1], columns [64,128) = g_y (conv5, scale 0.2).  Issued before the
      // input-gradient conv below, whose output may overwrite a buffer another block's GEMM has just read.
      if (C > 128 || 4 * gc > 64) {
        // gc = 32: concat pitch 192 -> per-layer weight gradients
        for (int k = 1; k <= 4; ++k) {
          rc = wgrad_plain(fwd_index_rdb(i, r, k), h, w, ws.cat[j], C, 0, Gb, C, nf + (4 - k) * gc, 1.f);
          if (rc) return rc;
        }
        rc = wgrad_plain(fwd_index_rdb(i, r, 5), h, w, ws.cat[j], C, 0, Gb, C, 0, 0.2f);
        if (rc) return rc;
      } else {
        const long part_stride = (long)9 * 128 * 128;
        std::vector<WgradLaunch> wg(3);
        for (int dy = 0; dy < 3; ++dy) {
          rc = build_wgrad(P->sms, N, h, w, 3, 1, dy - 1, 1, ws.cat[j], C, 0, Gb, C, nf, Gb, C, 0, 128, dacc + (size_t)dy * 3 * 128 * 128, part_stride,
                           128, &wg[dy]);
          if (rc) return rc;
        }
        push_acc_group(ops, wg, dacc, part_stride);
        for (int k = 1; k <= 5; ++k) {
          const LayerSpec& Ls = F[fwd_index_rdb(i, r, k)];
          Op sc; sc.kind = Op::kScatter; sc.src = dacc; sc.layer = fwd_index_rdb(i, r, k); sc.ci0 = 0; sc.ci_n = Ls.cin;
          sc.col0 = (k < 5) ? (4 - k) * gc : 64; sc.ld_n = 128; sc.scale = (k < 5) ? 1.f : 0.2f;
          sc.cout = Ls.cout; sc.cin = Ls.cin; sc.kh = Ls.kh; sc.kw = Ls.kw;
          ops.push_back(sc);
        }
        // bias gradients: the four narrow convs in one pass over the gradient-concat slices, conv5 from g_y
        Op bo; bo.kind = Op::kBias; bo.count = (long)N * h * w; bo.cout = 4 * gc; bo.nseg = 4;
        for (int q = 0; q < 4; ++q) bo.seg_layers[q] = fwd_index_rdb(i, r, 4 - q);      // slice order g4, g3, g2, g1
        bo.layer = bo.seg_layers[0]; bo.src = Gb; bo.C = C; bo.coff = nf;
        ops.push_back(bo);
        Op b5; b5.kind = Op::kBias; b5.layer = fwd_index_rdb(i, r, 5); b5.count = (long)N * h * w; b5.cout = nf;
        b5.src = Gb; b5.C = C; b5.coff = 0; b5.scale = 0.2f;
        ops.push_back(b5);
      }
      // gradient of the block input: conv_T([g_y | g4 | g3 | g2 | g1]) + g_y (identity path of x5*0.2 + x)
      // (+ G for RDB1: identity path of the RRDB, out*0.2 + x_rrdb)
      ConvIO io = io_of(Gb, C, Xo, C, 0, CSR_ACT_NONE);
      io.r1 = Gb; io.r1_C = C; io.r1_coff = 0; io.s1 = 1.f;
      if (r == 0) { io.r2 = ws.gcat[Pb]; io.r2_C = C; io.r2_coff = 0; io.s2 = 1.f; }
      rc = dgrad(h, w, io);
      if (rc) return rc;
    }
    Pb = Rb;                                               // RDB1 wrote dL/d(RRDB input) (incl. + G) into R[0:64]
  }
  // ---- conv_first (esrgan.py:90): total gradient of its output = trunk path (gcat[Pb][0:64]) + skip path (gt0) ----
  rc = wgrad_plain(0, h, w, ws.xin, 64, 0, ws.gcat[Pb], C, 0, 1.f);
  if (rc) return rc;
  rc = wgrad_plain(0, h, w, ws.xin, 64, 0, ws.gt0, 64, 0, 1.f);
  if (rc) return rc;
  if (bi != (int)B.size()) return fail(CSR_ERR_BAD_ARG, "internal: backward table mismatch (%d of %zu)", bi, B.size());
  return CSR_OK;
}

}  // namespace csr

using namespace csr;

// =========================================================================================== C-ABI
extern "C" {

int csr_abi_version(void) { return CSR_ABI_VERSION; }
const char* csr_last_error(void) { return g_err; }

int csr_device_check(void) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) return fail(CSR_ERR_CUDA, "no CUDA device: %s", cudaGetErrorString(e));
  DeviceInfo di;
  return device_info(&di);
}

int csr_set_option(int32_t key, int32_t value) {
  // the table with defaults and meanings is in INTEGRATION.md section 6.  Keys 2, 3, 5, 6, 7, 8, 9, 13, 14, 16, 20-24, 28, 29 and 32
  // are retired (they selected removed kernel variants or measured-and-rejected settings of the default kernels): do not reuse them,
  // callers of older versions may still set them
  switch (key) {
    case 1: g_opt_pdl = value ? 1 : 0; return CSR_OK;              // programmatic dependent launch on/off
    case 4: g_opt_no_tma_store = value ? 1 : 0; return CSR_OK;     // debug: per-element stores instead of the staged copy-out
    case 11: g_opt_graphs = value ? 1 : 0; return CSR_OK;          // CUDA-graph replay of plan forward / backward_flat
    case 12: g_opt_graph_max_px = value; return CSR_OK;
    case 15: g_opt_trace_cta = value; return CSR_OK;
    case 17: g_opt_narrow_box = value ? 1 : 0; return CSR_OK;
    case 18: g_opt_tall = value ? 1 : 0; return CSR_OK;
    case 19: g_opt_eight_acc = value ? 1 : 0; return CSR_OK;
    case 25: g_opt_wgrad_atomic = value ? 1 : 0; return CSR_OK;    // plans created afterwards
    case 27: g_opt_dense = value ? 1 : 0; return CSR_OK;           // plans created afterwards
    case 36: g_opt_tap_pack = value ? 1 : 0; return CSR_OK;
    case 35:                                                       // plans created afterwards
      if (value != 0 && value != 1) return fail(CSR_ERR_BAD_ARG, "option 35: 0 or 1");
      g_opt_hyb = value; return CSR_OK;
    case 34: g_opt_merge_phases = value ? 1 : 0; return CSR_OK;    // plans created afterwards, single convs called afterwards
    case 33: g_opt_fuse_tail = value & 3; return CSR_OK;       // plans created afterwards
    case 31: if (value < 0 || value > 64) return fail(CSR_ERR_BAD_ARG, "option 31: windows per SM in [0, 64]"); g_opt_dense_min = value; return CSR_OK;
    case 30: g_opt_reserve_sms = value < 0 ? 0 : value; return CSR_OK;
    case 37: g_opt_whole_row = value ? 1 : 0; return CSR_OK;       // plans created afterwards, single convs called afterwards
    case 26:                                                       // early-release epilogue of the wide residual-free layers
      if (value != 0 && value != 1) return fail(CSR_ERR_BAD_ARG, "option 26: 0 or 1");
      g_opt_early = value; return CSR_OK;
    default: return fail(CSR_ERR_BAD_ARG, "unknown option key %d", key);
  }
}

int64_t csr_kernel_launch_count(void) { return g_launches.load(); }

int csr_has_experiments(void) { return 0; }   // kept for ABI version 2: the experimental kernel variants are gone

int csr_debug_set_trace(void* device_buffer) {
#ifdef CSR_ENABLE_TRACE
  g_trace = reinterpret_cast<long long*>(device_buffer);
  return CSR_OK;
#else
  if (!device_buffer) return CSR_OK;
  return fail(CSR_ERR_UNSUPPORTED, "this build has no pipeline tracing (rebuild with CSR_BUILD_TRACE=1 python build.py --force)");
#endif
}

int csr_debug_set_timeline(void* device_u64, int32_t capacity_launches) {
  // device buffer of 2 * capacity uint64 (init: even entries ~0ull, odd entries 0): forwards run with direct launches write
  // [2i] = earliest CTA start (after the dependency wait) and [2i+1] = latest CTA end of launch i, in globaltimer ns
  g_timeline = reinterpret_cast<unsigned long long*>(device_u64);
  g_timeline_cap = device_u64 ? capacity_launches : 0;
  return CSR_OK;
}

int csr_num_layers(const CsrNetDesc* net) {
  int rc = check_net(net);
  if (rc) return rc;
  return (int)layer_table(*net).size();
}

int csr_layer_shape(const CsrNetDesc* net, int32_t i, int32_t shape4[4], char* name, size_t name_cap) {
  int rc = check_net(net);
  if (rc) return rc;
  const auto t = layer_table(*net);
  if (i < 0 || i >= (int)t.size() || !shape4) return fail(CSR_ERR_BAD_ARG, "layer index %d out of range", i);
  shape4[0] = t[i].cout; shape4[1] = t[i].cin; shape4[2] = t[i].kh; shape4[3] = t[i].kw;
  if (name && name_cap) snprintf(name, name_cap, "%s", t[i].name.c_str());
  return CSR_OK;
}

size_t csr_packed_weight_bytes(const CsrNetDesc* net) {
  if (check_net(net)) return 0;
  size_t total = 0;
  const auto t = layer_table(*net);
  pack_layout(fwd_exec_table(*net, t), &total);
  return total;
}

// Batched pack: the job table lives on the device, cached per destination blob and re-uploaded only when it changes
// (parameter storage moved).  One kernel launch packs every layer part.
static int run_pack_jobs(const std::vector<PackJob>& jobs, void* key, cudaStream_t s) {
  struct Cached { std::vector<PackJob> host; PackJob* dev = nullptr; };
  static std::map<void*, Cached> cache;
  static std::mutex mu;
  std::lock_guard<std::mutex> lock(mu);
  if (cache.size() > 512 && !cache.count(key)) {        // single-op callers hand in ever new scratch buffers: bound the table
    for (auto& kv : cache) if (kv.second.dev) cudaFree(kv.second.dev);
    cache.clear();
  }
  Cached& c = cache[key];
  const size_t bytes = jobs.size() * sizeof(PackJob);
  const bool same = c.dev && c.host.size() == jobs.size() && memcmp(c.host.data(), jobs.data(), bytes) == 0;
  if (!same) {
    if (c.dev && c.host.size() != jobs.size()) { cudaFree(c.dev); c.dev = nullptr; }
    if (!c.dev) CSR_CUDA(cudaMalloc(&c.dev, bytes));
    c.host = jobs;
    CSR_CUDA(cudaMemcpyAsync(c.dev, c.host.data(), bytes, cudaMemcpyHostToDevice, s));
  }
  CSR_CUDA(launch_pack_jobs(c.dev, (int)jobs.size(), s));
  ++g_launches;
  return CSR_OK;
}

int csr_pack_weights(const CsrNetDesc* net, const float* const* w, const float* const* b, void* packed, size_t packed_bytes,
                     void* stream) {
  int rc = check_net(net);
  if (rc) return rc;
  if (!w || !b || !packed) return fail(CSR_ERR_BAD_ARG, "null pointer");
  const auto layers = fwd_exec_table(*net, layer_table(*net));
  size_t total = 0;
  const auto packs = pack_layout(layers, &total);
  if (packed_bytes < total) return fail(CSR_ERR_WORKSPACE, "packed buffer %zu < %zu bytes", packed_bytes, total);
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  uint8_t* base = reinterpret_cast<uint8_t*>(packed);
  std::vector<PackJob> jobs;
  const size_t n_real = layer_table(*net).size();          // entries beyond it are views of other layers' weights (L.src)
  for (size_t i = 0; i < layers.size(); ++i) {
    const LayerSpec& L = layers[i];
    if (i < n_real && (!w[i] || !b[i])) return fail(CSR_ERR_BAD_ARG, "null weight/bias pointer for layer %zu", i);
    for (const PackPart& pp : packs[i].parts)
      jobs.push_back({i < n_real ? w[i] : w[L.src], i < n_real ? b[i] : nullptr, base + pp.w_off, reinterpret_cast<float*>(base + pp.b_off), L.cout,
                      L.cin, L.kh, L.kw, L.fold, pp.phase, L.transposed, L.wscale, pp.co_lo, pp.npad, packs[i].cin_pad, 0, 0, 0, 0});
  }
  return run_pack_jobs(jobs, packed, s);
}

size_t csr_workspace_bytes(const CsrNetDesc* net, int32_t n, int32_t h, int32_t w) {
  if (check_net(net) || n < 1 || h < 1 || w < 1) return 0;
  return ws_layout(*net, n, h, w, 0).total;
}

size_t csr_train_workspace_bytes(const CsrNetDesc* net, int32_t n, int32_t h, int32_t w) {
  if (check_net(net) || n < 1 || h < 1 || w < 1) return 0;
  return ws_layout(*net, n, h, w, 1).total;
}

static int plan_create_impl(const CsrNetDesc* net, int32_t n, int32_t h, int32_t w, void* workspace, size_t workspace_bytes, int train,
                            CsrPlan** plan) {
  int rc = check_net(net);
  if (rc) return rc;
  if (!plan || !workspace) return fail(CSR_ERR_BAD_ARG, "null pointer");
  if (n < 1 || h < 1 || w < 1) return fail(CSR_ERR_BAD_ARG, "non-positive shape n=%d h=%d w=%d", n, h, w);
  if (reinterpret_cast<uintptr_t>(workspace) % 1024) return fail(CSR_ERR_BAD_ARG, "workspace must be 1024-byte aligned");
  const WsLayout L = ws_layout(*net, n, h, w, train);
  if (workspace_bytes < L.total) return fail(CSR_ERR_WORKSPACE, "workspace %zu < %zu bytes", workspace_bytes, L.total);
  DeviceInfo di;
  rc = device_info(&di);
  if (rc) return rc;
  CsrPlan* P = new CsrPlan();
  P->net = *net; P->N = n; P->h = h; P->w = w; P->sms = std::max(1, di.sms - (train ? g_opt_reserve_sms : 0)); P->train = train;
  const std::vector<LayerSpec> layers = layer_table(*net);
  P->grad_off = grad_offsets(layers, &P->grad_floats);
  uint8_t* base = reinterpret_cast<uint8_t*>(workspace);
  P->sx = reinterpret_cast<float*>(base + L.sx); P->selev = reinterpret_cast<float*>(base + L.selev);
  P->smask = reinterpret_cast<float*>(base + L.smask); P->sout = reinterpret_cast<float*>(base + L.sout);
  if (train) { P->sgout = reinterpret_cast<float*>(base + L.sgout); P->sgrad = reinterpret_cast<float*>(base + L.sgrad); }
  P->flags = reinterpret_cast<unsigned int*>(base + L.flags); P->flags_bytes = L.flags_bytes;
  P->dbg_cat = L.cat; P->ccat = L.ccat;
  P->dbg_tail[0] = L.m1; P->dbg_tail[1] = L.hrA; P->dbg_tail[2] = L.hrB; P->dbg_tail[3] = L.hrD; P->dbg_tail[4] = L.hrE;
  P->dbg_tail[5] = L.fea0; P->dbg_tail[6] = L.t0; P->dbg_tail[7] = L.hrC; P->dbg_tail[8] = L.tlast;
  P->dbg_grad = {L.gO, L.gcolB, L.gT, L.gP, L.gQ, L.gm1, L.gt0, {L.gcat[0], L.gcat[1], L.gcat[2]}};
  const WsPtrs ws = ws_carve(L, workspace);
  rc = plan_build(P, ws, layers);
  if (!rc && train) {
    rc = bwd_build(P, ws, layers);
    if (!rc) {
      // the narrow gradient maps are read 16 channels wide but written 1-3 channels wide: start them from zero
      const size_t hr16 = (size_t)n * h * w * 16 * 16 * 2;
      cudaError_t e = cudaMemset(ws.gT, 0, hr16);
      if (e != cudaSuccess) rc = fail(CSR_ERR_CUDA, "cudaMemset: %s", cudaGetErrorString(e));
    }
  }
  if (rc) { delete P; return rc; }
  *plan = P;
  return CSR_OK;
}

int csr_plan_create(const CsrNetDesc* net, int32_t n, int32_t h, int32_t w, void* workspace, size_t workspace_bytes, CsrPlan** plan) {
  return plan_create_impl(net, n, h, w, workspace, workspace_bytes, 0, plan);
}

int csr_train_plan_create(const CsrNetDesc* net, int32_t n, int32_t h, int32_t w, void* workspace, size_t workspace_bytes, CsrPlan** plan) {
  return plan_create_impl(net, n, h, w, workspace, workspace_bytes, 1, plan);
}

size_t csr_packed_weight_bytes_bwd(const CsrNetDesc* net) {
  if (check_net(net)) return 0;
  size_t total = 0;
  pack_layout(bwd_layer_table(*net, layer_table(*net)), &total);
  return total;
}

int csr_pack_weights_bwd(const CsrNetDesc* net, const float* const* w, void* packed, size_t packed_bytes, void* stream) {
  int rc = check_net(net);
  if (rc) return rc;
  if (!w || !packed) return fail(CSR_ERR_BAD_ARG, "null pointer");
  const auto fl = layer_table(*net);
  const auto layers = bwd_layer_table(*net, fl);
  size_t total = 0;
  const auto packs = pack_layout(layers, &total);
  if (packed_bytes < total) return fail(CSR_ERR_WORKSPACE, "packed buffer %zu < %zu bytes", packed_bytes, total);
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  uint8_t* base = reinterpret_cast<uint8_t*>(packed);
  std::vector<PackJob> jobs;
  for (size_t i = 0; i < layers.size(); ++i) {
    const LayerSpec& L = layers[i];
    for (const PackPart& pp : packs[i].parts) {
      float* bdst = reinterpret_cast<float*>(base + pp.b_off);
      if (L.blocks.empty()) {
        if (!w[L.src]) return fail(CSR_ERR_BAD_ARG, "null weight pointer for layer %d", L.src);
        jobs.push_back({w[L.src], nullptr, base + pp.w_off, bdst, L.cout, L.cin, L.kh, L.kw, 0, pp.phase, L.transposed, L.wscale, pp.co_lo, pp.npad,
                        packs[i].cin_pad, 0, 0, 0, 0});
      } else {
        for (size_t bk = 0; bk < L.blocks.size(); ++bk) {
          const LayerSpec::Block& B = L.blocks[bk];
          if (!w[B.src]) return fail(CSR_ERR_BAD_ARG, "null weight pointer for layer %d", B.src);
          jobs.push_back({w[B.src], nullptr, base + pp.w_off, bk == 0 ? bdst : nullptr, L.cout, L.cin, L.kh, L.kw, 0, pp.phase, 1, B.wscale,
                          pp.co_lo, pp.npad, packs[i].cin_pad, B.ci_lo, B.n, B.src_ci_off, B.src_cin});
        }
      }
    }
  }
  return run_pack_jobs(jobs, packed, s);
}

}  // extern "C"

// Run `body` (a launch sequence on stream s) through a cached CUDA graph: captured at the second call for a given packed
// blob (the first call runs directly, so one-time attribute / symbol setup never happens inside a capture) and replayed
// afterwards.  Any capture / instantiate failure falls back to direct launches for the lifetime of the plan.
// When the caller is itself capturing s (torch.cuda.graph around a forward or backward), the launches go straight into the
// caller's capture: no private stream or nested capture is started there, and the call does not advance the cache.
template <typename Body>
static int run_graphed(CsrPlan::GraphCache& gc, const void* packed, cudaStream_t s, Body body) {
  if (!g_opt_graphs || gc.failed) return body(s);
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(s, &cap) != cudaSuccess) { cudaGetLastError(); return body(s); }
  if (cap != cudaStreamCaptureStatusNone) return body(s);
  if (gc.exec && gc.packed == packed) {
    CSR_CUDA(cudaGraphLaunch(gc.exec, s));
    g_launches += gc.launches;
    return CSR_OK;
  }
  if (gc.packed != packed) { gc.packed = packed; gc.calls = 0; if (gc.exec) { cudaGraphExecDestroy(gc.exec); gc.exec = nullptr; } }
  if (gc.calls++ == 0) return body(s);
  // capture on a private stream (the caller's may be the legacy default stream, which cannot be captured); the
  // instantiated graph is then launched into the caller's stream
  static thread_local cudaStream_t cs_dev[64] = {};     // a stream belongs to the device it was created on
  int cur_dev = 0;
  if (cudaGetDevice(&cur_dev) != cudaSuccess || cur_dev < 0 || cur_dev >= 64) { cudaGetLastError(); gc.failed = true; return body(s); }
  cudaStream_t& cs = cs_dev[cur_dev];
  if (!cs && cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking) != cudaSuccess) { cudaGetLastError(); gc.failed = true; return body(s); }
  const long l0 = g_launches.load();
  {
    const cudaError_t eb = cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal);
    if (eb != cudaSuccess) { fail(CSR_ERR_CUDA, "graph: begin capture: %s", cudaGetErrorString(eb)); cudaGetLastError(); gc.failed = true; return body(s); }
  }
  const int rc = body(cs);
  cudaGraph_t graph = nullptr;
  const cudaError_t e = cudaStreamEndCapture(cs, &graph);
  const long captured = g_launches.load() - l0;
  g_launches -= captured;                                 // nothing ran yet
  if (rc != CSR_OK || e != cudaSuccess || !graph) {
    const std::string inner = g_err;
    fail(CSR_ERR_CUDA, "graph: capture failed (rc %d, end capture: %s; %s)", rc, cudaGetErrorString(e), inner.c_str());
    cudaGetLastError();
    if (graph) cudaGraphDestroy(graph);
    gc.failed = true;
    return body(s);
  }
  cudaGraphExec_t exec = nullptr;
  const cudaError_t ei = cudaGraphInstantiate(&exec, graph, 0);
  if (ei != cudaSuccess) {
    fail(CSR_ERR_CUDA, "graph: instantiate: %s", cudaGetErrorString(ei));
    cudaGetLastError();
    cudaGraphDestroy(graph);
    gc.failed = true;
    return body(s);
  }
  cudaGraphDestroy(graph);
  gc.exec = exec;
  gc.launches = captured;
  CSR_CUDA(cudaGraphLaunch(gc.exec, s));
  g_launches += gc.launches;
  return CSR_OK;
}

extern "C" {

int csr_plan_backward(CsrPlan* P, const void* packed_bwd, const float* grad_out, float* const* dw, float* const* db, void* stream) {
  if (!P || !packed_bwd || !grad_out || !dw || !db) return fail(CSR_ERR_BAD_ARG, "null pointer");
  if (!P->train) return fail(CSR_ERR_BAD_ARG, "csr_plan_backward needs a plan made by csr_train_plan_create");
  // every gradient pointer is checked before the first launch: a refused call leaves dw / db untouched
  for (const Op& op : P->bwd) {
    if (op.kind == Op::kScatter && !dw[op.layer]) return fail(CSR_ERR_BAD_ARG, "null weight-gradient pointer for layer %d", op.layer);
    if (op.kind == Op::kBiasPlanar && !db[op.layer]) return fail(CSR_ERR_BAD_ARG, "null bias-gradient pointer for layer %d", op.layer);
    if (op.kind == Op::kBias)
      for (int q = 0; q < op.nseg; ++q)
        if (!db[op.nseg > 1 ? op.seg_layers[q] : op.layer]) return fail(CSR_ERR_BAD_ARG, "null bias-gradient pointer for layer %d", op.layer);
  }
  Bindings b;
  b.packed = packed_bwd; b.grad_out = grad_out; b.dw = dw; b.db = db;
  return run_ops(P->bwd, 0, P->bwd.size(), b, P->sms, reinterpret_cast<cudaStream_t>(stream));
}

// Bindings of the flat-gradient backward: dL/dout and the gradients live in the plan's staging buffers.
static Bindings flat_bindings(const CsrPlan* P, const void* packed_bwd, std::vector<float*>& dw, std::vector<float*>& db) {
  const size_t nl = P->grad_off.size() / 2;
  dw.resize(nl); db.resize(nl);
  for (size_t i = 0; i < nl; ++i) { dw[i] = P->sgrad + P->grad_off[2 * i]; db[i] = P->sgrad + P->grad_off[2 * i + 1]; }
  Bindings b;
  b.packed = packed_bwd; b.grad_out = P->sgout; b.dw = dw.data(); b.db = db.data();
  return b;
}

size_t csr_plan_grad_floats(const CsrPlan* P) { return P ? P->grad_floats : 0; }

// 1 = a CUDA graph is instantiated and being replayed, 0 = not (yet), -1 = capture failed (direct launches)
int csr_plan_graph_status(const CsrPlan* P, int32_t backward) {
  if (!P) return 0;
  const CsrPlan::GraphCache& g = backward ? P->g_bwd : P->g_fwd;
  return g.failed ? -1 : (g.exec ? 1 : 0);
}

int csr_plan_grad_offset(const CsrPlan* P, int32_t layer, int32_t is_bias, size_t* offset) {
  if (!P || !offset || layer < 0 || 2 * (size_t)layer + 1 >= P->grad_off.size()) return fail(CSR_ERR_BAD_ARG, "bad layer index");
  *offset = P->grad_off[2 * layer + (is_bias ? 1 : 0)];
  return CSR_OK;
}

int csr_plan_backward_segments(CsrPlan* P, int32_t nseg) {
  if (!P || !P->train) return fail(CSR_ERR_BAD_ARG, "needs a plan made by csr_train_plan_create");
  if (nseg < 1) return fail(CSR_ERR_BAD_ARG, "nseg must be positive");
  // last op that writes each layer's gradient
  const size_t nl = P->grad_off.size() / 2;
  std::vector<size_t> last(nl, 0);
  for (size_t oi = 0; oi < P->bwd.size(); ++oi) {
    const Op& op = P->bwd[oi];
    if (op.kind == Op::kScatter || op.kind == Op::kBiasPlanar) last[op.layer] = oi;
    if (op.kind == Op::kBias)
      for (int q = 0; q < op.nseg; ++q) last[op.nseg > 1 ? op.seg_layers[q] : op.layer] = oi;
  }
  // done_after[oi] = lowest float offset such that every layer at or above it is complete once ops [0, oi] have run
  std::vector<size_t> done_at(P->bwd.size() + 1, P->grad_floats);
  {
    std::vector<size_t> order(nl);
    for (size_t i = 0; i < nl; ++i) order[i] = i;
    // walk layers from the last one down while they are complete
    for (size_t oi = 0; oi < P->bwd.size(); ++oi) {
      size_t lo = P->grad_floats;
      for (size_t li = nl; li-- > 0;) {
        if (last[li] <= oi) lo = P->grad_off[2 * li]; else break;
      }
      done_at[oi + 1] = lo;
    }
  }
  P->seg_op.clear(); P->seg_lo.clear(); P->seg_hi.clear();
  for (auto& g : P->g_seg) if (g.exec) cudaGraphExecDestroy(g.exec);
  P->g_seg.clear();
  size_t prev_op = 0, prev_lo = P->grad_floats;
  for (int k = 1; k <= nseg; ++k) {
    const size_t target = P->grad_floats - P->grad_floats * k / nseg;      // completed suffix should reach down to here
    size_t oi = prev_op;
    if (k == nseg) oi = P->bwd.size();
    else
      while (oi < P->bwd.size() && done_at[oi] > target) ++oi;
    // no op left for this slice: skip it (with nseg near grad_floats the suffix is complete before k == nseg, and a last
    // segment would run nothing)
    if (oi <= prev_op) continue;
    P->seg_op.push_back(prev_op);
    P->seg_lo.push_back(done_at[oi]);
    P->seg_hi.push_back(prev_lo);
    prev_op = oi; prev_lo = done_at[oi];
  }
  P->seg_op.push_back(P->bwd.size());
  P->g_seg.resize(P->seg_lo.size());
  return (int)P->seg_lo.size();
}

int csr_plan_backward_flat_seg(CsrPlan* P, const void* packed_bwd, const float* grad_out, float* flat_grads, int32_t seg, size_t* lo, size_t* hi,
                               void* stream) {
  if (!P || !packed_bwd || !grad_out || !flat_grads || !lo || !hi) return fail(CSR_ERR_BAD_ARG, "null pointer");
  if (!P->train || seg < 0 || (size_t)seg >= P->seg_lo.size()) return fail(CSR_ERR_BAD_ARG, "bad segment (call csr_plan_backward_segments first)");
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  if (seg == 0)
    CSR_CUDA(cudaMemcpyAsync(P->sgout, grad_out, (size_t)P->N * 16 * P->h * P->w * sizeof(float), cudaMemcpyDeviceToDevice, s));
  std::vector<float*> dw, db;
  const Bindings b = flat_bindings(P, packed_bwd, dw, db);
  const size_t o0 = P->seg_op[seg], o1 = P->seg_op[seg + 1];
  int rc = run_graphed(P->g_seg[seg], packed_bwd, s, [&](cudaStream_t st) -> int {
    if (seg == 0) CSR_CUDA(cudaMemsetAsync(P->sgrad, 0, P->grad_floats * sizeof(float), st));
    return run_ops(P->bwd, o0, o1, b, P->sms, st);
  });
  if (rc) return rc;
  *lo = P->seg_lo[seg]; *hi = P->seg_hi[seg];
  if (*hi > *lo) CSR_CUDA(cudaMemcpyAsync(flat_grads + *lo, P->sgrad + *lo, (*hi - *lo) * sizeof(float), cudaMemcpyDeviceToDevice, s));
  return CSR_OK;
}

int csr_plan_backward_flat(CsrPlan* P, const void* packed_bwd, const float* grad_out, float* flat_grads, void* stream) {
  if (!P || !packed_bwd || !grad_out || !flat_grads) return fail(CSR_ERR_BAD_ARG, "null pointer");
  if (!P->train) return fail(CSR_ERR_BAD_ARG, "csr_plan_backward_flat needs a plan made by csr_train_plan_create");
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  const size_t hr_bytes = (size_t)P->N * 16 * P->h * P->w * sizeof(float);
  // the replayed graph works on plan-owned buffers: stage dL/dout in, copy the flat gradients out
  CSR_CUDA(cudaMemcpyAsync(P->sgout, grad_out, hr_bytes, cudaMemcpyDeviceToDevice, s));
  std::vector<float*> dw, db;
  const Bindings b = flat_bindings(P, packed_bwd, dw, db);
  int rc = run_graphed(P->g_bwd, packed_bwd, s, [&](cudaStream_t st) -> int {
    CSR_CUDA(cudaMemsetAsync(P->sgrad, 0, P->grad_floats * sizeof(float), st));
    return run_ops(P->bwd, 0, P->bwd.size(), b, P->sms, st);
  });
  if (rc) return rc;
  CSR_CUDA(cudaMemcpyAsync(flat_grads, P->sgrad, P->grad_floats * sizeof(float), cudaMemcpyDeviceToDevice, s));
  return CSR_OK;
}

int csr_plan_buffer(const CsrPlan* P, int32_t kind, int32_t index, size_t* offset_bytes, int32_t* dims4) {
  // test hook: where an activation buffer of the plan lives inside the caller's workspace (dims4 = n, h, w, channel pitch; bf16 NHWC
  // except kind 9).  kind 0: concat buffer `index` ([x | x1 | x2 | x3 | x4]), 1: upconv1 output, 2: upconv2 output, 3: HRconv output,
  // 4: srcnn.conv1 output, 5: srcnn.conv2 output, 6: fea0 (conv_first output), 7: t0 (trunk_conv + fea0), 8: hrC (SRCNN input
  // im2col, channel dx*3 + c), 9: tlast (conv_last output, fp32 planar).  Training plans keep all of them, one concat buffer per
  // dense block.  Inference plans rotate three concat buffers (RDB3 writes the RRDB output over buffer 0's x), share kinds 2 / 4 and
  // 3 / 5 (fused tail, option 33 = 3: kind 2 keeps upconv2's output; kind 3 holds conv_last's tap planes, then srcnn.conv2's output)
  // and leave kind 9 unwritten while option 36 is on.  Kinds 10..17 (training plans only) are the backward's gradient buffers:
  // 10: gO (25-tap im2col of dL/dout), 11: gcolB (9-tap im2col of dL/d(conv_last output)), 12: gT (dL/d[conv_last output, elev,
  // mask]), 13 / 14: gP / gQ (HR-tail ping-pong), 15: gm1, 16: gt0, 17: gradient concat buffer `index` (0..2).  The header spells
  // this out.
  if (!P || !offset_bytes || !dims4) return fail(CSR_ERR_BAD_ARG, "null pointer");
  const int h = P->h, w = P->w;
  if (kind == 0) {
    if (index < 0 || (size_t)index >= P->dbg_cat.size()) return fail(CSR_ERR_BAD_ARG, "concat buffer index %d out of range", index);
    *offset_bytes = P->dbg_cat[index];
    dims4[0] = P->N; dims4[1] = h; dims4[2] = w; dims4[3] = P->ccat;
    return CSR_OK;
  }
  if (kind >= 10 && kind <= 17) {
    if (!P->train) return fail(CSR_ERR_BAD_ARG, "buffer kind %d exists in training plans only", kind);
    if (kind == 17 && (index < 0 || index > 2)) return fail(CSR_ERR_BAD_ARG, "gradient concat buffer index %d out of range", index);
    const size_t off[8] = {P->dbg_grad.gO, P->dbg_grad.gcolB, P->dbg_grad.gT, P->dbg_grad.gP, P->dbg_grad.gQ, P->dbg_grad.gm1,
                           P->dbg_grad.gt0, kind == 17 ? P->dbg_grad.gcat[index] : 0};
    const int pitch[8] = {32, 16, 16, 64, 64, 64, 64, P->ccat};
    const int s = kind <= 14 ? 4 : kind == 15 ? 2 : 1;
    *offset_bytes = off[kind - 10];
    dims4[0] = P->N; dims4[1] = s * h; dims4[2] = s * w; dims4[3] = pitch[kind - 10];
    return CSR_OK;
  }
  if (kind < 1 || kind > 9) return fail(CSR_ERR_BAD_ARG, "unknown buffer kind %d", kind);
  *offset_bytes = P->dbg_tail[kind - 1];
  const int s = (kind == 6 || kind == 7) ? 1 : kind == 1 ? 2 : 4;
  dims4[0] = P->N; dims4[1] = s * h; dims4[2] = s * w;
  dims4[3] = (kind == 5 || kind == 8) ? P->srcnn_pitch : kind == 9 ? 1 : 64;
  return CSR_OK;
}

int csr_plan_num_backward_ops(const CsrPlan* plan) { return plan ? (int)plan->bwd.size() : 0; }

int csr_plan_num_launches(const CsrPlan* plan) { return plan ? (int)plan->fwd.size() : 0; }

void csr_plan_destroy(CsrPlan* plan) {
  if (!plan) return;
  if (plan->g_fwd.exec) cudaGraphExecDestroy(plan->g_fwd.exec);
  if (plan->g_bwd.exec) cudaGraphExecDestroy(plan->g_bwd.exec);
  for (auto& g : plan->g_seg) if (g.exec) cudaGraphExecDestroy(g.exec);
  delete plan;
}

int csr_plan_forward(CsrPlan* P, const void* packed, const float* x, const float* elev, const float* mask, float* out, void* stream) {
  if (!P || !packed || !x || !elev || !mask || !out) return fail(CSR_ERR_BAD_ARG, "null pointer");
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  Bindings b;
  b.packed = packed; b.timeline = g_timeline; b.timeline_cap = g_timeline_cap;
  auto body = [&](cudaStream_t st) -> int {
    int rc = run_ops(P->fwd, 0, 1, b, P->sms, st);           // op 0: the input conversion
    if (rc) return rc;
    if (P->fwd_dense) CSR_CUDA(cudaMemsetAsync(P->flags, 0, P->flags_bytes, st));
    return run_ops(P->fwd, 1, P->fwd.size(), b, P->sms, st);
  };
  // Graph replay pays three staging copies; it wins when the forward is launch-bound (small rasters / batches).
  const size_t hr_px = (size_t)P->N * 16 * P->h * P->w;
  if (!g_opt_graphs || P->g_fwd.failed || hr_px > (size_t)g_opt_graph_max_px) {
    b.x = x; b.elev = elev; b.mask = mask; b.out = out;
    return body(s);
  }
  CSR_CUDA(cudaMemcpyAsync(P->sx, x, (size_t)P->N * P->net.in_channels * P->h * P->w * sizeof(float), cudaMemcpyDeviceToDevice, s));
  CSR_CUDA(cudaMemcpyAsync(P->selev, elev, hr_px * sizeof(float), cudaMemcpyDeviceToDevice, s));
  CSR_CUDA(cudaMemcpyAsync(P->smask, mask, hr_px * sizeof(float), cudaMemcpyDeviceToDevice, s));
  b.x = P->sx; b.elev = P->selev; b.mask = P->smask; b.out = P->sout;
  int rc = run_graphed(P->g_fwd, packed, s, body);
  if (rc) return rc;
  CSR_CUDA(cudaMemcpyAsync(out, P->sout, hr_px * sizeof(float), cudaMemcpyDeviceToDevice, s));
  return CSR_OK;
}

int csr_generator_forward(const CsrNetDesc* net, const void* packed, const float* x, const float* elev, const float* mask, float* out,
                          void* workspace, size_t workspace_bytes, int32_t n, int32_t h, int32_t w, void* stream) {
  CsrPlan* P = nullptr;
  int rc = csr_plan_create(net, n, h, w, workspace, workspace_bytes, &P);
  if (rc) return rc;
  rc = csr_plan_forward(P, packed, x, elev, mask, out, stream);
  csr_plan_destroy(P);
  return rc;
}

// ---- single conv --------------------------------------------------------------------------------------
static int conv_desc_to_layer(const CsrConvDesc* d, LayerSpec* L) {
  if (!d) return fail(CSR_ERR_BAD_ARG, "conv descriptor is null");
  if (d->n < 1 || d->h < 1 || d->w < 1 || d->cin < 1 || d->cout < 1) return fail(CSR_ERR_BAD_ARG, "non-positive conv shape");
  if (!(d->kh & 1) || !(d->kw & 1) || d->kh > 9 || d->kw > 9) return fail(CSR_ERR_UNSUPPORTED, "kernel %dx%d (odd, <= 9 supported)", d->kh, d->kw);
  if (d->cout > 1024) return fail(CSR_ERR_UNSUPPORTED, "cout %d > 1024", d->cout);
  if (d->out_mode != CSR_OUT_BF16_NHWC && d->out_mode != CSR_OUT_F32_PLANAR && d->out_mode != CSR_OUT_F32_NHWC && d->out_mode != CSR_OUT_BF16_SPLIT)
    return fail(CSR_ERR_BAD_ARG, "unknown out_mode %d", d->out_mode);
  if (d->out_mode == CSR_OUT_BF16_SPLIT) {
    if (d->kh != 3 || d->kw != 3 || d->act != CSR_ACT_RELU || d->in_up2 || d->transposed)
      return fail(CSR_ERR_UNSUPPORTED, "hi/lo bf16 output is implemented for plain 3x3 convs with ReLU only");
    if (d->cout % 8 || d->out_c < d->out_coff + 2 * d->cout)
      return fail(CSR_ERR_UNSUPPORTED, "hi/lo bf16 output needs cout %% 8 == 0 and out_c >= out_coff + 2 cout (cout %d, out_c %d, out_coff %d)",
                  d->cout, d->out_c, d->out_coff);
  }
  if (d->out_mode == CSR_OUT_F32_PLANAR && d->cout != 1) return fail(CSR_ERR_UNSUPPORTED, "fp32 planar output needs cout == 1");
  if (d->in_up2 && (d->kh != 3 || d->kw != 3)) return fail(CSR_ERR_UNSUPPORTED, "nearest-x2 input needs a 3x3 kernel");
  if (d->in_up2 && d->transposed) return fail(CSR_ERR_UNSUPPORTED, "in_up2 and transposed cannot be combined");
  *L = {"conv", d->cout, d->cin, d->kh, d->kw, 0, d->in_up2 ? 1 : 0, d->transposed ? 1 : 0};
  return CSR_OK;
}

size_t csr_conv2d_scratch_bytes(const CsrConvDesc* d) {
  LayerSpec L;
  if (conv_desc_to_layer(d, &L)) return 0;
  size_t total = 0;
  pack_layout({L}, &total, true);
  return total;
}

// all parts of the layer in ONE pack launch
static int conv2d_pack_parts(const LayerSpec& L, const PackLayer& pl, const float* weight, const float* bias, void* scratch, cudaStream_t s) {
  uint8_t* base = reinterpret_cast<uint8_t*>(scratch);
  std::vector<PackJob> jobs;
  for (const PackPart& pp : pl.parts)
    jobs.push_back({weight, bias, base + pp.w_off, reinterpret_cast<float*>(base + pp.b_off), L.cout, L.cin, L.kh, L.kw, 0, pp.phase, L.transposed,
                    1.f, pp.co_lo, pp.npad, pl.cin_pad, 0, 0, 0, 0});
  return run_pack_jobs(jobs, scratch, s);
}

int csr_conv2d_pack(const CsrConvDesc* d, const float* weight, const float* bias, void* scratch, size_t scratch_bytes, void* stream) {
  LayerSpec L;
  int rc = conv_desc_to_layer(d, &L);
  if (rc) return rc;
  if (!weight || !scratch) return fail(CSR_ERR_BAD_ARG, "null pointer");
  size_t total = 0;
  const auto packs = pack_layout({L}, &total, true);
  if (scratch_bytes < total) return fail(CSR_ERR_WORKSPACE, "scratch %zu < %zu bytes", scratch_bytes, total);
  return conv2d_pack_parts(L, packs[0], weight, bias, scratch, reinterpret_cast<cudaStream_t>(stream));
}

int csr_conv2d_nhwc(const CsrConvDesc* d, const void* in, const float* weight, const float* bias, void* out, const void* res1,
                    const void* res2, const void* gate, void* scratch, size_t scratch_bytes, void* stream) {
  LayerSpec L;
  int rc = conv_desc_to_layer(d, &L);
  if (rc) return rc;
  if (!in || !out || !scratch) return fail(CSR_ERR_BAD_ARG, "null pointer");
  DeviceInfo di;
  rc = device_info(&di);
  if (rc) return rc;
  size_t total = 0;
  const auto packs = pack_layout({L}, &total, true);
  if (scratch_bytes < total) return fail(CSR_ERR_WORKSPACE, "scratch %zu < %zu bytes", scratch_bytes, total);
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  ConvIO io;
  io.in = in; io.in_C = d->in_c; io.cin_off = d->in_coff;
  io.out = out; io.out_C = d->out_c; io.out_coff = d->out_coff;
  io.out_kind = d->out_mode == CSR_OUT_BF16_NHWC ? kOutBf16 : d->out_mode == CSR_OUT_F32_PLANAR ? kOutF32Planar :
                d->out_mode == CSR_OUT_BF16_SPLIT ? kOutBf16Split : kOutF32Nhwc;
  io.split_off = d->cout;
  if (d->out_mode == CSR_OUT_BF16_SPLIT && (res1 || res2 || gate)) return fail(CSR_ERR_UNSUPPORTED, "hi/lo bf16 output takes no residual / gate operand");
  io.act = d->act; io.act_slope = d->act_slope;
  io.r1 = res1; io.r1_C = d->res1_c; io.r1_coff = d->res1_coff; io.s1 = d->scale1;
  io.r2 = res2; io.r2_C = d->res2_c; io.r2_coff = d->res2_coff; io.s2 = d->scale2;
  io.gate = gate; io.gate_C = d->gate_c; io.gate_coff = d->gate_coff; io.gate_from = d->gate_from; io.gate_neg = d->gate_neg;
  if (d->act == CSR_ACT_LRELU && !(d->act_slope > 0.f && d->act_slope < 1.f)) return fail(CSR_ERR_BAD_ARG, "act_slope must be in (0, 1)");
  if (weight) {
    // weight == NULL: `scratch` still holds the packed weights / bias of an earlier call (or of csr_conv2d_pack) with the same layer
    // shape and weights (callers cache it per weight version)
    rc = conv2d_pack_parts(L, packs[0], weight, bias, scratch, s);
    if (rc) return rc;
  }
  // RCAN training is bound by host time per call (~4 us): reuse the list's storage instead of allocating it every call
  thread_local std::vector<Op> ops;
  ops.clear();
  rc = emit_conv(ops, packs[0], d->n, d->h, d->w, io);
  if (rc) return rc;
  Bindings b;
  b.packed = scratch;
  return run_ops(ops, 0, ops.size(), b, di.sms, s);
}

// ---- single-layer weight gradient (building block; used by the parity tests) ---------------------------
size_t csr_conv2d_wgrad_scratch_bytes(const CsrWgradDesc* d) {
  if (!d || d->cout < 1 || d->cin < 1) return 0;
  const LayerSpec L = {"wgrad", d->cout, d->cin, d->kh, d->kw, 0, d->in_up2 ? 1 : 0};
  const size_t jobs = (!L.up2 && L.kh == L.kw && L.kw <= 3) ? wgrad_jobs_scratch_floats(L) : 0;
  if (d->cout > 128) return jobs * sizeof(float);
  return std::max(jobs, wgrad_scratch_floats(L)) * sizeof(float);
}

int csr_conv2d_wgrad(const CsrWgradDesc* d, const void* x, const void* g, float* dw, float* db, void* scratch, size_t scratch_bytes,
                     void* stream) {
  if (!d || !x || !g || !dw || !scratch) return fail(CSR_ERR_BAD_ARG, "null pointer");
  if (d->n < 1 || d->h < 1 || d->w < 1 || d->cin < 1 || d->cout < 1 || d->cout > 1024) return fail(CSR_ERR_BAD_ARG, "bad wgrad shape");
  if (!(d->kh & 1) || !(d->kw & 1) || d->kh > 9 || d->kw > 9) return fail(CSR_ERR_UNSUPPORTED, "kernel %dx%d", d->kh, d->kw);
  if (d->in_up2 && (d->kh != 3 || d->kw != 3)) return fail(CSR_ERR_UNSUPPORTED, "nearest-x2 input needs a 3x3 kernel");
  const LayerSpec L = {"wgrad", d->cout, d->cin, d->kh, d->kw, 0, d->in_up2 ? 1 : 0};
  if (scratch_bytes < csr_conv2d_wgrad_scratch_bytes(d)) return fail(CSR_ERR_WORKSPACE, "wgrad scratch too small");
  DeviceInfo di;
  int rc = device_info(&di);
  if (rc) return rc;
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  float* dacc = reinterpret_cast<float*>(scratch);
  std::vector<Op> ops;
  std::vector<float*> dws, dbs;                            // op layer k: output-channel chunk k
  if (wgrad_jobs_applicable(L, d->n, d->h, d->w, di.sms)) {
    rc = emit_wgrad_jobs(ops, L, 0, d->n, d->h, d->w, x, d->x_c, d->x_coff, g, d->g_c, d->g_coff, d->scale, db != nullptr, dacc, di.sms);
    if (rc) return rc;
    dws.push_back(dw); dbs.push_back(db);
  } else {
    // Output channels in chunks whose KW x chunk accumulator columns fit the 512 TMEM columns (one chunk for every layer up to 5x5 / 64
    // channels; the 9x9 srcnn.conv1 with 64 output channels takes two).
    const int ekw = L.up2 ? 2 : L.kw;
    const int chunk = std::max(16, std::min((L.cout + 15) / 16 * 16, 512 / ekw / 16 * 16));
    for (int co0 = 0; co0 < L.cout; co0 += chunk) {
      LayerSpec Lc = L;
      Lc.cout = std::min(chunk, L.cout - co0);
      rc = emit_wgrad(ops, Lc, (int)dws.size(), d->n, d->h, d->w, x, d->x_c, d->x_coff, g, d->g_c, d->g_coff + co0, d->scale, db != nullptr, dacc,
                      di.sms);
      if (rc) return rc;
      dws.push_back(dw + (size_t)co0 * L.cin * L.kh * L.kw);
      dbs.push_back(db ? db + co0 : nullptr);
    }
  }
  Bindings b;
  b.dw = dws.data(); b.db = dbs.data();
  return run_ops(ops, 0, ops.size(), b, di.sms, s);
}

// ---- layout helpers -----------------------------------------------------------------------------------
int csr_nchw_f32_to_nhwc_bf16(const float* src, void* dst, int32_t n, int32_t c, int32_t h, int32_t w, int32_t dst_c, int32_t zero_to,
                              void* stream) {
  if (!src || !dst) return fail(CSR_ERR_BAD_ARG, "null pointer");
  if (c < 1 || c > 16 || (zero_to != 8 && zero_to != 16) || c > zero_to || dst_c % 8 || dst_c < zero_to)
    return fail(CSR_ERR_UNSUPPORTED, "c=%d zero_to=%d dst_c=%d", c, zero_to, dst_c);
  CSR_CUDA(launch_nchw_to_nhwc(src, dst, n, c, h, w, dst_c, zero_to, reinterpret_cast<cudaStream_t>(stream)));
  ++g_launches;
  return CSR_OK;
}

int csr_nhwc_bf16_to_nchw_f32(const void* src, float* dst, int32_t n, int32_t c, int32_t h, int32_t w, int32_t src_c, int32_t src_coff,
                              void* stream) {
  if (!src || !dst) return fail(CSR_ERR_BAD_ARG, "null pointer");
  CSR_CUDA(launch_nhwc_to_nchw(src, dst, n, c, h, w, src_c, src_coff, reinterpret_cast<cudaStream_t>(stream)));
  ++g_launches;
  return CSR_OK;
}

// ---- hi/lo bf16 activations (perceptual loss) -----------------------------------------------------------
int csr_nchw_f32_to_nhwc_split(const float* src, void* dst, int32_t n, int32_t c, int32_t h, int32_t w, int32_t dst_c, void* stream) {
  if (!src || !dst) return fail(CSR_ERR_BAD_ARG, "null pointer");
  if (n < 1 || h < 1 || w < 1) return fail(CSR_ERR_BAD_ARG, "non-positive shape %dx%dx%d", n, h, w);
  if (c < 1 || c > 3 || dst_c % 8 || dst_c < 2 * c || dst_c > 64)
    return fail(CSR_ERR_UNSUPPORTED, "split conversion: c=%d (1..3), dst_c=%d (multiple of 8, 2c..64)", c, dst_c);
  if (reinterpret_cast<uintptr_t>(dst) % 16) return fail(CSR_ERR_BAD_ARG, "dst must be 16-byte aligned");
  CSR_CUDA(launch_nchw_to_nhwc_split(src, dst, n, c, h, w, dst_c, reinterpret_cast<cudaStream_t>(stream)));
  ++g_launches;
  return CSR_OK;
}

int csr_maxpool2x2_split(const void* src, void* dst, int32_t n, int32_t h, int32_t w, int32_t c, void* stream) {
  if (!src || !dst) return fail(CSR_ERR_BAD_ARG, "null pointer");
  if (n < 1) return fail(CSR_ERR_BAD_ARG, "non-positive batch %d", n);
  if (h < 2 || w < 2 || c < 8 || c % 8) return fail(CSR_ERR_UNSUPPORTED, "split max pool: h=%d, w=%d (>= 2), c=%d (multiple of 8)", h, w, c);
  if ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) % 16) return fail(CSR_ERR_BAD_ARG, "src / dst must be 16-byte aligned");
  CSR_CUDA(launch_maxpool2x2_split(src, dst, n, h, w, c, reinterpret_cast<cudaStream_t>(stream)));
  ++g_launches;
  return CSR_OK;
}

// ---- pixel loss (value + gradient in one pass) ---------------------------------------------------------
size_t csr_pixel_loss_scratch_bytes(int64_t numel) { return numel > 0 ? (size_t)pixel_loss_blocks(numel) * sizeof(double) : 0; }

static int pixel_loss(int mode, const float* sr, const float* hr, float* grad, int64_t numel, float* out, void* scratch, size_t scratch_bytes,
                      void* stream) {
  if (!sr || !hr || !out || !scratch) return fail(CSR_ERR_BAD_ARG, "null pointer");
  if (numel < 1) return fail(CSR_ERR_BAD_ARG, "numel must be positive");
  if (scratch_bytes < csr_pixel_loss_scratch_bytes(numel)) return fail(CSR_ERR_WORKSPACE, "loss scratch too small");
  if ((reinterpret_cast<uintptr_t>(sr) | reinterpret_cast<uintptr_t>(hr) | reinterpret_cast<uintptr_t>(grad)) % 16)
    return fail(CSR_ERR_BAD_ARG, "sr / hr / grad must be 16-byte aligned");
  cudaError_t e = launch_pixel_loss(mode, sr, hr, grad, numel, out, reinterpret_cast<double*>(scratch), reinterpret_cast<cudaStream_t>(stream));
  g_launches += 2;
  if (e != cudaSuccess) return fail(CSR_ERR_CUDA, "loss launch failed: %s", cudaGetErrorString(e));
  return CSR_OK;
}

int csr_l1_loss(const float* sr, const float* hr, float* grad, int64_t numel, float* out, void* scratch, size_t scratch_bytes, void* stream) {
  return pixel_loss(0, sr, hr, grad, numel, out, scratch, scratch_bytes, stream);
}
int csr_mse_loss(const float* sr, const float* hr, float* grad, int64_t numel, float* out, void* scratch, size_t scratch_bytes, void* stream) {
  return pixel_loss(1, sr, hr, grad, numel, out, scratch, scratch_bytes, stream);
}

// ---- metrics ------------------------------------------------------------------------------------------
size_t csr_metrics_scratch_bytes(int32_t n, int32_t h, int32_t w) { return metrics_scratch_bytes(n, h, w); }

int csr_masked_metrics(const float* sr, const float* hr, const float* original, const float* mask, const double* mn, const double* mx,
                       float zmean, float zstd, double range_a, double range_b, double eps, int32_t n, int32_t h, int32_t w, float* out,
                       void* scratch, size_t scratch_bytes, void* stream) {
  if (!sr || !hr || !original || !mask || !out || !scratch) return fail(CSR_ERR_BAD_ARG, "null pointer");
  if ((mn == nullptr) != (mx == nullptr)) return fail(CSR_ERR_BAD_ARG, "mn and mx must both be given or both be null");
  if (n < 1 || h < 11 || w < 11) return fail(CSR_ERR_UNSUPPORTED, "need n>=1 and h,w >= 11 (SSIM window), got %d %d %d", n, h, w);
  if (scratch_bytes < metrics_scratch_bytes(n, h, w)) return fail(CSR_ERR_WORKSPACE, "metrics scratch too small");
  int launches = 0;
  cudaError_t e = launch_masked_metrics(sr, hr, original, mask, mn, mx, zmean, zstd, range_a, range_b, eps, n, h, w, out, scratch,
                                        reinterpret_cast<cudaStream_t>(stream), &launches);
  g_launches += launches;
  if (e != cudaSuccess) return fail(CSR_ERR_CUDA, "metrics launch failed: %s", cudaGetErrorString(e));
  return CSR_OK;
}

// ---- inference pre / post-processing ---------------------------------------------------------------------------
int csr_minmax_normalize(const float* raw, int32_t n, int32_t h, int32_t w, const double* mn, const double* mx, double range_a, double range_b,
                         double eps, float nan_substitution, const float* extra0, const float* extra1, float* out, void* stream) {
  if (!raw || !mn || !mx || !out) return fail(CSR_ERR_BAD_ARG, "null pointer");
  if (n < 1 || h < 1 || w < 1 || n > 65535) return fail(CSR_ERR_BAD_ARG, "bad shape n=%d h=%d w=%d", n, h, w);
  if (!extra0 && extra1) return fail(CSR_ERR_BAD_ARG, "extra1 given without extra0");
  CSR_CUDA(launch_minmax_normalize(raw, n, (long)h * w, mn, mx, range_a, range_b, eps, nan_substitution, extra0, extra1, out,
                                   reinterpret_cast<cudaStream_t>(stream)));
  ++g_launches;
  return CSR_OK;
}

int csr_minmax_denormalize_mask(const float* sr, const float* mask, int32_t mask_per_sample, int32_t n, int32_t h, int32_t w, const double* mn,
                                const double* mx, double range_a, double range_b, double eps, float* out, void* stream) {
  if (!sr || !mask || !mn || !mx || !out) return fail(CSR_ERR_BAD_ARG, "null pointer");
  if (n < 1 || h < 1 || w < 1 || n > 65535) return fail(CSR_ERR_BAD_ARG, "bad shape n=%d h=%d w=%d", n, h, w);
  CSR_CUDA(launch_minmax_denormalize_mask(sr, mask, mask_per_sample ? (long)h * w : 0, n, (long)h * w, mn, mx, range_a, range_b, eps, out,
                                          reinterpret_cast<cudaStream_t>(stream)));
  ++g_launches;
  return CSR_OK;
}

// ---- discriminator path: glue between the convolutions (disc.cu) ------------------------------------------------------
static int view_of(const CsrView* v, DiscView* out) {
  if (!v) return fail(CSR_ERR_BAD_ARG, "view is null");
  if (v->c < 8 || v->c % 8 || v->hs < 1 || v->ws < 1 || v->hl < 1 || v->wl < 1 || v->step < 1 || v->off < 0 ||
      v->off + v->step * (v->hl - 1) >= v->hs || v->off + v->step * (v->wl - 1) >= v->ws)
    return fail(CSR_ERR_BAD_ARG, "bad view hs=%d ws=%d c=%d off=%d step=%d hl=%d wl=%d", v->hs, v->ws, v->c, v->off, v->step, v->hl, v->wl);
  *out = {v->hs, v->ws, v->c, v->off, v->step, v->hl, v->wl};
  return CSR_OK;
}
int csr_disc_gather(const void* src, const CsrView* view, int32_t n, void* dst, int32_t pad, const float* scale, const float* shift, void* stream) {
  DiscView v;
  int rc = view_of(view, &v);
  if (rc) return rc;
  if (!src || !dst || n < 1 || pad < 0 || pad > 1 || (pad && (v.Hl < 2 || v.Wl < 2)) || ((scale == nullptr) != (shift == nullptr)))
    return fail(CSR_ERR_BAD_ARG, "csr_disc_gather: bad arguments");
  CSR_CUDA(launch_disc_gather(src, v, n, dst, pad, scale, shift, reinterpret_cast<cudaStream_t>(stream)));
  ++g_launches;
  return CSR_OK;
}
int csr_disc_collect(const void* dpad, const CsrView* view, int32_t n, int32_t pad, const void* act, float gate_neg, void* g, void* stream) {
  DiscView v;
  int rc = view_of(view, &v);
  if (rc) return rc;
  if (!dpad || !g || n < 1 || pad < 0 || pad > 1) return fail(CSR_ERR_BAD_ARG, "csr_disc_collect: bad arguments");
  CSR_CUDA(launch_disc_collect(dpad, v, n, pad, act, gate_neg, g, reinterpret_cast<cudaStream_t>(stream)));
  ++g_launches;
  return CSR_OK;
}
size_t csr_disc_bn_scratch_bytes(int32_t c) { return c > 0 ? (size_t)2 * c * sizeof(double) : 0; }
int csr_disc_bn_forward(const void* src, const CsrView* view, int32_t n, const float* gamma, const float* beta, float eps, float momentum,
                        float* running_mean, float* running_var, int32_t training, float* scale, float* shift, float* mean, float* invstd,
                        void* scratch, size_t scratch_bytes, void* stream) {
  DiscView v;
  int rc = view_of(view, &v);
  if (rc) return rc;
  if (!src || !gamma || !beta || !scale || !shift || n < 1) return fail(CSR_ERR_BAD_ARG, "csr_disc_bn_forward: null pointer");
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  if (!training) {
    if (!running_mean || !running_var) return fail(CSR_ERR_BAD_ARG, "eval-mode BatchNorm needs the running statistics");
    CSR_CUDA(launch_disc_bn_eval(v.C, gamma, beta, eps, running_mean, running_var, scale, shift, s));
    ++g_launches;
    return CSR_OK;
  }
  if (!mean || !invstd || !scratch || scratch_bytes < csr_disc_bn_scratch_bytes(v.C)) return fail(CSR_ERR_WORKSPACE, "BatchNorm scratch / statistics buffers");
  if ((running_mean == nullptr) != (running_var == nullptr)) return fail(CSR_ERR_BAD_ARG, "running_mean and running_var go together");
  CSR_CUDA(launch_disc_bn_stats(src, v, n, reinterpret_cast<double*>(scratch), s));
  CSR_CUDA(launch_disc_bn_finalize(reinterpret_cast<double*>(scratch), src, v, (double)n * v.Hl * v.Wl, gamma, beta, eps, momentum, running_mean,
                                   running_var, scale, shift, mean, invstd, s));
  g_launches += 2;
  return CSR_OK;
}
int csr_disc_bn_backward(const void* dpad, const CsrView* view, int32_t n, int32_t pad, const void* act, float gate_neg, const float* gamma,
                         const float* mean, const float* invstd, float* dy_scratch, void* scratch, size_t scratch_bytes, void* g, float* dgamma,
                         float* dbeta, void* stream) {
  DiscView v;
  int rc = view_of(view, &v);
  if (rc) return rc;
  if (!dpad || !act || !gamma || !mean || !invstd || !dy_scratch || !g || !dgamma || !dbeta || n < 1 || pad < 0 || pad > 1)
    return fail(CSR_ERR_BAD_ARG, "csr_disc_bn_backward: bad arguments");
  if (!scratch || scratch_bytes < csr_disc_bn_scratch_bytes(v.C)) return fail(CSR_ERR_WORKSPACE, "BatchNorm scratch too small");
  CSR_CUDA(launch_disc_bn_backward(dpad, v, n, pad, act, gate_neg, gamma, mean, invstd, dy_scratch, reinterpret_cast<double*>(scratch), g, dgamma,
                                   dbeta, reinterpret_cast<cudaStream_t>(stream)));
  g_launches += 2;
  return CSR_OK;
}
int csr_disc_flatten(const void* src, const CsrView* view, int32_t n, float* feats, void* stream) {
  DiscView v;
  int rc = view_of(view, &v);
  if (rc) return rc;
  if (!src || !feats || n < 1) return fail(CSR_ERR_BAD_ARG, "null pointer");
  CSR_CUDA(launch_disc_flatten(src, v, n, feats, reinterpret_cast<cudaStream_t>(stream)));
  ++g_launches;
  return CSR_OK;
}
int csr_disc_unflatten(const float* gfeat, const CsrView* view, int32_t n, void* g, void* stream) {
  DiscView v;
  int rc = view_of(view, &v);
  if (rc) return rc;
  if (!gfeat || !g || n < 1) return fail(CSR_ERR_BAD_ARG, "null pointer");
  CSR_CUDA(launch_disc_unflatten(gfeat, v, n, g, reinterpret_cast<cudaStream_t>(stream)));
  ++g_launches;
  return CSR_OK;
}
int csr_linear_forward(const float* x, const float* w, const float* b, float* y, int32_t n, int32_t k, int32_t j, void* stream) {
  if (!x || !w || !y || n < 1 || k < 1 || j < 1 || n > 65535) return fail(CSR_ERR_BAD_ARG, "csr_linear_forward: bad arguments");
  CSR_CUDA(launch_linear_forward(x, w, b, y, n, k, j, reinterpret_cast<cudaStream_t>(stream)));
  ++g_launches;
  return CSR_OK;
}
int csr_linear_backward(const float* x, const float* w, const float* gy, float* dx, float* dw, float* db, int32_t n, int32_t k, int32_t j,
                        void* stream) {
  if (!x || !w || !gy || n < 1 || k < 1 || j < 1) return fail(CSR_ERR_BAD_ARG, "csr_linear_backward: bad arguments");
  CSR_CUDA(launch_linear_backward(x, w, gy, dx, dw, db, n, k, j, reinterpret_cast<cudaStream_t>(stream)));
  g_launches += (dx ? 1 : 0) + ((dw || db) ? 1 : 0);
  return CSR_OK;
}

// ---- RCAN generator: glue between the convolutions (rcan.cu), forward and backward ---------------------------------------------------------
int csr_channel_attention(const void* res, const void* x, const float* w1, const float* b1, const float* w2, const float* b2, void* out,
                          float* pooled_scratch, int32_t n, int32_t h, int32_t w, int32_t c, int32_t c_reduced, void* stream) {
  if (!res || !x || !w1 || !b1 || !w2 || !b2 || !out || !pooled_scratch) return fail(CSR_ERR_BAD_ARG, "null pointer");
  if (n < 1 || n > 65535 || h < 1 || w < 1 || c < 8 || c % 8 || c > 512 || c_reduced < 1 || c_reduced > c)
    return fail(CSR_ERR_BAD_ARG, "csr_channel_attention: bad shape n=%d h=%d w=%d c=%d c_reduced=%d", n, h, w, c, c_reduced);
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  CSR_CUDA(launch_channel_pool(res, n, (long)h * w, c, pooled_scratch, s));
  CSR_CUDA(launch_ca_scale_add(res, x, pooled_scratch, w1, b1, w2, b2, out, n, (long)h * w, c, c_reduced, s));
  g_launches += 2;
  return CSR_OK;
}
int csr_pixel_shuffle2(const void* src, void* dst, int32_t n, int32_t h, int32_t w, int32_t c, void* stream) {
  if (!src || !dst || n < 1 || h < 1 || w < 1 || c < 8 || c % 8) return fail(CSR_ERR_BAD_ARG, "csr_pixel_shuffle2: bad arguments");
  CSR_CUDA(launch_pixel_shuffle2(src, dst, n, h, w, c, reinterpret_cast<cudaStream_t>(stream)));
  ++g_launches;
  return CSR_OK;
}
size_t csr_channel_attention_backward_scratch_bytes(int32_t n, int32_t c) { return n > 0 && c > 0 ? (size_t)n * c * sizeof(float) : 0; }
int csr_channel_attention_backward(const void* dout, const void* res, const float* pooled, const float* w1, const float* b1, const float* w2,
                                   const float* b2, void* dres, float* dw1, float* db1, float* dw2, float* db2, void* scratch,
                                   size_t scratch_bytes, int32_t n, int32_t h, int32_t w, int32_t c, int32_t c_reduced, void* stream) {
  if (!dout || !res || !pooled || !w1 || !b1 || !w2 || !b2 || !dres || !dw1 || !db1 || !dw2 || !db2 || !scratch)
    return fail(CSR_ERR_BAD_ARG, "null pointer");
  if (n < 1 || n > 65535 || h < 1 || w < 1 || c < 8 || c % 8 || c > 512 || c_reduced < 1 || c_reduced > c)
    return fail(CSR_ERR_BAD_ARG, "csr_channel_attention_backward: bad shape n=%d h=%d w=%d c=%d c_reduced=%d", n, h, w, c, c_reduced);
  if (scratch_bytes < csr_channel_attention_backward_scratch_bytes(n, c)) return fail(CSR_ERR_WORKSPACE, "channel-attention backward scratch too small");
  CSR_CUDA(launch_ca_backward(dout, res, pooled, w1, b1, w2, b2, dres, dw1, db1, dw2, db2, reinterpret_cast<float*>(scratch), n, (long)h * w, c,
                              c_reduced, reinterpret_cast<cudaStream_t>(stream)));
  g_launches += 2;
  return CSR_OK;
}
int csr_pixel_unshuffle2(const void* src, void* dst, int32_t n, int32_t h, int32_t w, int32_t c, void* stream) {
  if (!src || !dst || n < 1 || h < 1 || w < 1 || c < 8 || c % 8) return fail(CSR_ERR_BAD_ARG, "csr_pixel_unshuffle2: bad arguments");
  CSR_CUDA(launch_pixel_unshuffle2(src, dst, n, h, w, c, reinterpret_cast<cudaStream_t>(stream)));
  ++g_launches;
  return CSR_OK;
}

// ---- gradient exchange (data-parallel training) -------------------------------------------------------------------
int csr_grad_pack_bf16(const float* flat, void* comm_bf16, size_t n, float scale, void* stream) {
  if (!flat || !comm_bf16) return fail(CSR_ERR_BAD_ARG, "null pointer");
  if (n == 0) return CSR_OK;
  CSR_CUDA(launch_grad_pack_bf16(flat, comm_bf16, (long)n, scale, std::max(2, 2 * g_opt_reserve_sms), reinterpret_cast<cudaStream_t>(stream)));
  ++g_launches;
  return CSR_OK;
}
int csr_grad_unpack_bf16(const void* comm_bf16, float* flat, size_t n, float scale, void* stream) {
  if (!flat || !comm_bf16) return fail(CSR_ERR_BAD_ARG, "null pointer");
  if (n == 0) return CSR_OK;
  CSR_CUDA(launch_grad_unpack_bf16(comm_bf16, flat, (long)n, scale, std::max(2, 2 * g_opt_reserve_sms), reinterpret_cast<cudaStream_t>(stream)));
  ++g_launches;
  return CSR_OK;
}

// ---- training-sample assembly ------------------------------------------------------------------------------------
int csr_lr_input_from_hr(const float* hr, const float* elev, const float* mask, int32_t n, int32_t H, int32_t W, int32_t scale,
                         const int32_t* codes, float* hr_out, float* elev_out, float* mask_out, float* x_out, void* stream) {
  if (!hr || !elev || !mask || !x_out) return fail(CSR_ERR_BAD_ARG, "null pointer");
  if (n < 1 || n > 65535 || H < 1 || W < 1 || scale < 1 || H % scale || W % scale)
    return fail(CSR_ERR_BAD_ARG, "bad shape n=%d H=%d W=%d scale=%d (H and W must be multiples of scale)", n, H, W, scale);
  const int outs = (hr_out ? 1 : 0) + (elev_out ? 1 : 0) + (mask_out ? 1 : 0);
  if (outs != 0 && outs != 3) return fail(CSR_ERR_BAD_ARG, "hr_out, elev_out and mask_out must all be given or all be null");
  if (codes && outs == 0) return fail(CSR_ERR_BAD_ARG, "augmentation codes need the augmented output tensors");
  // (odd rot90 factors on non-square tiles are a caller error the kernel cannot see on the host: codes live on the device)
  CSR_CUDA(launch_lr_input(hr, elev, mask, n, H, W, scale, codes, hr_out, elev_out, mask_out, x_out, reinterpret_cast<cudaStream_t>(stream)));
  ++g_launches;
  return CSR_OK;
}

}  // extern "C"

// KHxKW stride-1 convolution over NHWC bf16 as an implicit GEMM on tcgen05 (sm_100a).
//
// Measured on B200 (profiles/r01_umma_probe.txt): in SS mode an M=128,K=16 bf16 MMA costs ~45-55 clk for any N <= 64
// (the 4 KB A-operand read from shared memory is the floor), ~71 clk at N=128, ~135 at N=256.  A conv whose GEMM N is
// only Cout = 16..64 therefore wastes most of each MMA.  This kernel folds the KW horizontal taps into N:
//
//   D[128 window pixels][dx*npad + co] (fp32, TMEM) += A_dy[128 pixels][16 ch] x B_dy[KW*npad][16 ch]
//
// for every vertical tap dy and 16-channel k-step: KH (not KH*KW) MMAs per k-step, each KW times wider.  The epilogue
// finishes the horizontal sum with warp shuffles:  out[m] = sum_dx D[m + dx - PW][dx*npad + co]  (GEMM rows m are
// flattened window positions, one TMEM lane == one thread per row, neighbours in x are neighbour lanes; SW <= 32 so a
// window row never straddles two warps).
//
// Halo reuse: one TMA box per 64-channel k-block brings the (TH+KH-1) x SW pixel window of a tile into shared memory
// ONCE (out-of-bounds pixels are zero-filled by TMA == the conv's zero padding).  The A operand of vertical tap dy is
// the same window read from byte offset dy*SW*128: only the descriptor start address changes between taps (UMMA
// applies the 128B swizzle on absolute smem address bits, so any 128-byte-aligned start works - verified on HW).
//
// Roles: warp 0 = TMA producer, warps 1-2 = MMA issuers on alternate tiles (warp 1 owns TMEM), warps 3..18 = epilogue in
// 2 or 4 independent groups (each group covers the four TMEM lane quadrants and owns one accumulator buffer).  Accumulators are double buffered in TMEM so the
// epilogue of tile i overlaps the MMAs of tile i+1; the layer's packed weights stay resident in shared memory for the
// whole persistent CTA.  bf16 outputs are staged in a (swizzled) shared-memory tile and copied out in 16-byte pieces,
// whole pixel rows per warp instruction (a strided output view scatters a sub-pixel phase of the nearest-x2 + conv
// layers).  A bulk tensor (TMA) store was measured first: it queues behind the producer's prefetched TMA loads in the
// SM's TMA pipe and stalled its issuing warp for 1000-2700 clk per tile, so the copy-out uses LDS.128 + STG.128.  Programmatic dependent launch: everything before griddepcontrol.wait (barrier init, TMEM
// alloc, weight/bias loads) overlaps the tail of the previous layer's kernel.
//
// Replaces one nn.Conv2d(+LeakyReLU/ReLU, *0.2+x, cat, nearest-x2) call site of the reference generator:
// climsr/models/esrgan.py:33-38, 50-54, 90-100 and climsr/models/srcnn.py:14-16 - and, with transposed / flipped
// weight packs, the input-gradient half of their autograd backward.
#include <cstdio>

#include "conv_tc.cuh"
#include "ptx.cuh"

namespace csr {

namespace {

// Per-role clock64 stamps (csr_debug_set_trace).  Compiled in only with -DCSR_ENABLE_TRACE (CSR_BUILD_TRACE=1 python
// build.py): the ~20 stamp sites are ~2 KB of code, and the kernel has to fit the instruction cache.
#ifdef CSR_ENABLE_TRACE
#define CSR_TRACE(role, tile_it, ev)                                                                                  \
  do {                                                                                                                \
    if (p.trace && blockIdx.x == p.trace_cta && (tile_it) < 64) p.trace[((role) * 64 + (tile_it)) * 8 + (ev)] = clock64();      \
  } while (0)
#else
#define CSR_TRACE(role, tile_it, ev) do { } while (0)
#endif

struct Tile {
  int n, y0, x0;
};

// t / d for 0 <= t < 2^24, d < 2^16 via a host-computed reciprocal (floor(2^40/d) + 1): one 64-bit multiply, no division.
__device__ __forceinline__ int fast_div(int t, unsigned long long magic) {
  return static_cast<int>((static_cast<unsigned long long>(static_cast<unsigned>(t)) * magic) >> 40);
}

template <int TALL_T>
__device__ __forceinline__ Tile decode_tile(const ConvParams& p, int t) {
  Tile r;
  r.n = fast_div(t, p.magic_img);
  const int rem = t - r.n * p.tiles_per_img;
  const int ty = fast_div(rem, p.magic_row);
  r.y0 = ty * (p.TH << TALL_T);                          // window origin: a window holds 1 or 2 vertically adjacent M tiles
  r.x0 = (rem - ty * p.tiles_x) * p.TW;
  return r;
}

// The epilogue is instruction-issue bound: its fp32 arithmetic uses the packed two-wide forms (FADD2 / FMUL2 / FFMA2).
__device__ __forceinline__ void apply_act8(float (&v)[8], int act, float slope = 0.f) {
  if (act == 4) {                                       // LeakyReLU(slope), 0 < slope < 1 (discriminator: 0.01 / 0.2)
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = fmaxf(v[j], slope * v[j]);
  } else if (act == 1) {                                       // LeakyReLU(0.2) = max(v, 0.2 v)
#pragma unroll
    for (int j = 0; j < 8; j += 2) {
      const float2 t = __fmul2_rn(make_float2(v[j], v[j + 1]), make_float2(0.2f, 0.2f));
      v[j] = fmaxf(v[j], t.x);
      v[j + 1] = fmaxf(v[j + 1], t.y);
    }
  } else if (act == 2) {
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = fmaxf(v[j], 0.f);
  }
}

// acc[j] += value of raw[j] held by lane (lane + delta); delta == 0 -> own value.  Executed by all 32 lanes.
__device__ __forceinline__ void gather_add8(float (&acc)[8], const uint32_t (&raw)[8], int delta, int lane) {
  float s[8];
  if (delta == 0) {
#pragma unroll
    for (int j = 0; j < 8; ++j) s[j] = __uint_as_float(raw[j]);
  } else {
    const int src = (lane + delta) & 31;
#pragma unroll
    for (int j = 0; j < 8; ++j) s[j] = __uint_as_float(__shfl_sync(0xffffffffu, raw[j], src));
  }
#pragma unroll
  for (int j = 0; j < 8; j += 2) {
    const float2 t = __fadd2_rn(make_float2(acc[j], acc[j + 1]), make_float2(s[j], s[j + 1]));
    acc[j] = t.x;
    acc[j + 1] = t.y;
  }
}

__device__ __forceinline__ void fma_residual8(float (&v)[8], const uint4& r, float scale) {
  const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 t = __ffma2_rn(make_float2(v[2 * i], v[2 * i + 1]), make_float2(scale, scale), make_float2(bf16lo(w[i]), bf16hi(w[i])));
    v[2 * i] = t.x;
    v[2 * i + 1] = t.y;
  }
}

__device__ __forceinline__ void gate8(float (&v)[8], const uint4& g, float neg) {
  const uint32_t w[4] = {g.x, g.y, g.z, g.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    v[2 * i] *= (bf16lo(w[i]) > 0.f) ? 1.f : neg;
    v[2 * i + 1] *= (bf16hi(w[i]) > 0.f) ? 1.f : neg;
  }
}

__device__ __forceinline__ uint4 ldg16(const void* base, size_t pix, int C, int coff) {
  return __ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(base) + pix * C + coff));
}

}  // namespace

// Compile-time specialisation of the epilogue (it is instruction-issue bound, so every runtime switch costs):
//   KW_T  horizontal taps (0 = runtime p.KW, taps gathered one at a time);  PW_T left padding when KW_T > 0
//   ACT_T activation (-1 = runtime p.act);  RES_T bit0 r1, bit1 r2, bit2 gate (-1 = runtime pointers)
//   ST_T  1 = staged bf16 stores only, 3 = fp32 planar single-channel output only (conv_last, srcnn.conv3: just channel 0
//         is computed), -1 = runtime p.store_mode
//   TALL_T 1 = two M tiles per window (ConvParams::tall_shift), compile-time so that the common kernels carry none of it
//   HYB_T 1 = (3x3, early-release epilogue) only TWO of the three horizontal taps are folded into N: per (dy, k-step) one N = 2*npad MMA
//            (taps dx = 0, 1) plus one N = npad MMA for tap dx = 2 whose A operand starts one pixel later and which accumulates into the
//            dx = 1 columns.  142 instead of 117 clk of MMAs, but the accumulator is 128 instead of 192 columns (four buffers instead of
//            two) and the epilogue reads a third fewer columns and shuffles once instead of twice - these layers are epilogue-bound.
//   FUSE_T 1 = (early-release epilogue only) the layer's 64-channel output never leaves the SM: the staged bf16 tile - already a K-major,
//             128B-swizzled UMMA A operand - goes through a SECOND MMA with the weights of the following 1x1 conv (srcnn.conv2 after
//             srcnn.conv1: 64 -> 32, srcnn.py:15-16), whose bias + ReLU output is what gets stored.  Saves the 64-channel HR map's
//             write and re-read (2 x 537 MB at cfg2) and one launch.  Inference plans only (training saves the intermediate).
//   EARLY_T 1 = wide residual-free layers (64 output channels, one 16-warp epilogue group): every warp pulls its WHOLE share of
//          the accumulator (2 chunks x KW taps) into registers, hands the TMEM buffer back to the MMA warps at once and only
//          then does the shuffle-sum / activation / staging; two staging buffers, so a tile costs one named barrier and the
//          copy-out of tile i overlaps the accumulator loads of tile i+1.  (Round 1 measured these layers epilogue-bound:
//          ~2450 clk per 128 x 64 tile against ~1400 clk of MMAs, because an accumulator stayed busy for the whole
//          ~1000-clk arithmetic phase and only two of them fit TMEM; tools/tmem_probe.cu shows the TMEM read port itself
//          delivers a 128 x 192 fp32 tile to 16 warps in ~260 clk.)
template <int KW_T, int PW_T, int ACT_T, int RES_T, int ST_T, int TALL_T = 0, int EARLY_T = 0, int FUSE_T = 0, int HYB_T = 0>
__global__ void __launch_bounds__(kConvThreads, 1)
conv_tc_kernel(const ConvParams p, const __grid_constant__ CUtensorMap tmap) {
  static_assert(!HYB_T || EARLY_T, "hybrid tap fold: early-release epilogue only");
  extern __shared__ uint8_t smem_raw[];
  // 1024-byte alignment: the 128B-swizzle pattern repeats every 8 rows x 128 B.
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t slots_addr = smem_base;
  const uint32_t stage_addr = slots_addr + static_cast<uint32_t>(p.n_slots) * p.slot_bytes;   // one staging buffer per epilogue group
  const uint32_t w_addr = stage_addr + static_cast<uint32_t>(p.n_stage) * p.stage_bytes;
  const int w_local = p.stream_w ? 0 : p.w_bytes;       // resident weight bytes
  // fused 1x1 successor (FUSE_T): its packed weights and bias sit right behind the layer's own weights
  const uint32_t w2_addr = w_addr + ((w_local + 127) & ~127);
  const uint32_t b2_addr = w2_addr + (FUSE_T ? static_cast<uint32_t>(p.w2_bytes) : 0u);
  const uint32_t bias_addr = b2_addr + (FUSE_T ? 128u : 0u);
  const uint32_t bar_addr = bias_addr + 256;            // up to 64 fp32 biases
  // barriers: [0] weights, [1..S] a_full, [1+S..2S] a_empty, then acc_full[8], acc_empty[8], d2
  const int S = p.n_slots;
  const int NA = p.n_acc;                               // accumulator buffers in TMEM (2, 4 or 8)
  const int NG = p.n_groups;                            // epilogue warp groups (1, 2 or 4; NG <= NA): tiles in flight in the epilogue
  const int wpg = kEpilogueWarps / NG;                  // warps per epilogue group
  auto bar_w = bar_addr;
  auto bar_a_full = [&](int s) { return bar_addr + 8u * (1 + s); };
  auto bar_a_empty = [&](int s) { return bar_addr + 8u * (1 + S + s); };
  auto bar_acc_full = [&](int b) { return bar_addr + 8u * (1 + 2 * S + b); };
  auto bar_acc_empty = [&](int b) { return bar_addr + 8u * (9 + 2 * S + b); };
  const uint32_t bar_d2 = bar_addr + 8u * (17 + 2 * S);              // FUSE_T: the second MMA of a tile has completed
  const uint32_t tmem_slot_addr = bar_addr + 8u * (18 + 2 * S);      // [0] TMEM base, [1..2] issuer progress words
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  float* bias_s = reinterpret_cast<float*>(smem_gen + (bias_addr - smem_base));
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem_gen + (tmem_slot_addr - smem_base));
  volatile uint32_t* progress = tmem_slot + 1;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int KW = KW_T ? KW_T : p.KW;
  // parts on gridDim.y may also differ in vertical padding and output row phase (the sub-pixel phases (a, b), a = 0 / 1, of
  // nearest-x2 + conv: PH = 1 - a, output row offset a)
  const int ph_eff = p.PH + static_cast<int>(blockIdx.y) * p.part_ph;
  const int oy_eff = p.out_oy + static_cast<int>(blockIdx.y) * p.part_oy;

  // Let the next layer's grid start its own prologue as early as the hardware allows (PDL).
  griddep_launch_dependents();

  if (threadIdx.x == 0) {
    progress[0] = 0;
    progress[1] = 0;
    mbar_init(bar_d2, 1);
    tma_prefetch_desc(&tmap);
    mbar_init(bar_w, 1);
    for (int s = 0; s < S; ++s) {
      mbar_init(bar_a_full(s), 1);
      mbar_init(bar_a_empty(s), 1);
    }
    for (int b = 0; b < NA; ++b) {
      mbar_init(bar_acc_full(b), 1);
      mbar_init(bar_acc_empty(b), wpg);
    }
    fence_mbar_init();
    fence_proxy_async_smem();
  }
  if (threadIdx.x == 0 && !p.stream_w) {
    // layer weights (constant data, not produced by the previous kernel): resident for the whole CTA
    const uint8_t* wsrc = reinterpret_cast<const uint8_t*>(p.wpk) + static_cast<size_t>(blockIdx.y) * p.part_w_bytes;
    mbar_arrive_expect_tx(bar_w, p.w_bytes + (FUSE_T ? p.w2_bytes : 0));
    for (int off = 0; off < p.w_bytes; off += 32768) {
      const int nbytes = min(32768, p.w_bytes - off);
      bulk_load(w_addr + off, wsrc + off, nbytes, bar_w);
    }
    if constexpr (FUSE_T) bulk_load(w2_addr, p.w2, p.w2_bytes, bar_w);
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot_addr, p.tmem_cols);
    tmem_relinquish();
  }
  for (int i = threadIdx.x; i < p.npad; i += blockDim.x) bias_s[i] = p.bias[blockIdx.y * p.part_b_floats + i];
  if constexpr (FUSE_T) {
    float* bias2_s = reinterpret_cast<float*>(smem_gen + (b2_addr - smem_base));
    for (int i = threadIdx.x; i < 32; i += blockDim.x) bias2_s[i] = (p.b2 && i < p.n2) ? p.b2[i] : 0.f;
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // Everything below reads / writes activations of the previous layer(s): wait for the prerequisite grid.
  griddep_wait();
  timeline_start(p.timeline, p.launch_id);

  const int ksteps_total = p.cin >> 4;
  const int nmma = KW * p.npad;                          // UMMA N: horizontal taps folded into the output columns
  const int nacc = HYB_T ? (KW - 1) * p.npad : nmma;     // accumulator columns per tile (hybrid fold: the last tap shares the previous tap's columns)

  if (warp == 0) {
    // ===================== TMA producer (whole warp walks the loop, one elected lane issues) =====================
    int slot = 0, pit = 0;
    uint32_t phase = 0;
    for (int t = blockIdx.x; t < p.num_tiles; t += gridDim.x, ++pit) {
      const Tile tl = decode_tile<TALL_T>(p, t);
      for (int kb = 0; kb < p.n_kblocks; ++kb) {
        if (kb == 0 && lane == 0) CSR_TRACE(0, pit, 0);
        mbar_wait_spin(bar_a_empty(slot), phase ^ 1);
        if (kb == 0 && lane == 0) CSR_TRACE(0, pit, 1);
        if (elect_one()) {
          if (p.stream_w) {
            // streamed weights: this k-block's packed weights travel with the window (same barrier)
            const int ks_here = min(4, (p.cin >> 4) - kb * 4);
            const int wbytes = p.KH * ks_here * (KW * p.npad) * 32;
            mbar_arrive_expect_tx(bar_a_full(slot), p.win_bytes + wbytes);
            const uint8_t* wsrc = reinterpret_cast<const uint8_t*>(p.wpk) + static_cast<size_t>(blockIdx.y) * p.part_w_bytes +
                                  static_cast<size_t>(kb) * p.wkb_bytes;
            const uint32_t wdst = slots_addr + slot * p.slot_bytes + p.win_slot_bytes;
            for (int off = 0; off < wbytes; off += 32768) bulk_load(wdst + off, wsrc + off, min(32768, wbytes - off), bar_a_full(slot));
          } else {
            mbar_arrive_expect_tx(bar_a_full(slot), p.win_bytes);
          }
          tma_load_4d(slots_addr + slot * p.slot_bytes, &tmap, bar_a_full(slot), p.cin_off + kb * 64, tl.x0 - p.PW, tl.y0 - ph_eff, tl.n);
        }
        __syncwarp();
        if (++slot == S) { slot = 0; phase ^= 1; }
      }
    }
  } else if (warp <= kMmaWarps) {
    if (warp > p.n_mma) goto done;                       // single-issuer launches: warp 2 idles
    // ===================== MMA issuers (warps 1 and 2 take alternate tiles) =====================
    // tcgen05.mma issue proceeds at execution pace (the issuing thread stalls while the tensor pipe is busy), so with a
    // single issuer the ~600 clk of mbarrier round trips between tiles leave the pipe idle.  With two issuers one warp's
    // waits overlap the other warp's MMAs.  Both issuers share the window-slot ring.  A parity wait is only unambiguous if
    // the waiter is at most one phase ahead of the barrier, so before waiting for ring entry e an issuer makes sure entry
    // e - n_slots (the previous fill of the same slot) has been seen full: trivially true for its own entries, and read
    // from the other issuer's progress word otherwise.  All 32 lanes run the warp-uniform control flow; one elected lane issues.  Per
    // MMA only the 14-bit start-address fields of the two descriptors change.
    const int mw = warp - 1;
    const uint32_t idesc = make_idesc_bf16(kTileM, nmma);
    const uint32_t b_step16 = static_cast<uint32_t>(nmma * 32) >> 4;         // one (dy,kstep) weight block in 16-byte units
    const uint32_t kb_w16 = static_cast<uint32_t>(p.KH * 4) * b_step16;       // one full k-block of weights
    // A window: one pixel = one row of box_c channels (128 / 64 / 32 bytes, swizzled with the matching TMA mode)
    const uint32_t row_bytes = static_cast<uint32_t>(p.box_c) * 2u;
    const uint32_t row16 = static_cast<uint32_t>(p.SW) * (row_bytes >> 4);    // one window row (SW pixels)
    const uint32_t a_layout = p.box_c == 64 ? 2u : p.box_c == 32 ? 4u : 6u;   // SWIZZLE_128B / 64B / 32B
    const uint32_t a_hi = ((8u * row_bytes) >> 4) | (1u << 14) | (a_layout << 29);   // SBO = 8 rows, version 1
    const uint32_t b_hi = (256u >> 4) | (1u << 14);                           // SBO 256 B, version 1, no swizzle
    const uint32_t a_lbo = (16u >> 4) << 16, b_lbo = (128u >> 4) << 16;
    if (!p.stream_w) mbar_wait_spin(bar_w, 0);
    tc_fence_after();
    // window-slot ring position of k-block 0 of this warp's first tile (the ring is shared by both issuers: tile `it`
    // owns ring entries it*n_kblocks .. it*n_kblocks + n_kblocks-1)
    constexpr int tall = 1 << TALL_T;                    // M tiles per window (2: thin layers, see ConvParams::tall_shift)
    int slot = 0, buf = mw * tall;
    uint32_t phase = 0, acc_phase = 0;
    auto ring_advance = [&](int steps) {
      for (int i = 0; i < steps; ++i)
        if (++slot == S) { slot = 0; phase ^= 1; }
    };
    if (mw) ring_advance(p.n_kblocks);
    int entry = mw * p.n_kblocks;                                            // ring entry index of (tile, kb)
    for (int it = mw; ; it += p.n_mma) {
      const int t = blockIdx.x + it * static_cast<int>(gridDim.x);
      if (t >= p.num_tiles) break;
      if (lane == 0) CSR_TRACE(1, it, 0);
      mbar_wait_spin(bar_acc_empty(buf), acc_phase ^ 1);
      if constexpr (TALL_T) mbar_wait_spin(bar_acc_empty(buf + 1), acc_phase ^ 1);
      tc_fence_after();
      if (lane == 0) CSR_TRACE(1, it, 1);
      const uint32_t d_tmem = tmem_base + buf * nacc;
      for (int kb = 0; kb < p.n_kblocks; ++kb, ++entry) {
        if (p.n_mma > 1) {
          const int need = entry - S;
          if (need >= 0 && ((need / p.n_kblocks) & 1) != mw) {
            while (progress[1 - mw] <= static_cast<uint32_t>(need)) {
            }
          }
        }
        mbar_wait_spin(bar_a_full(slot), phase);
        if (p.n_mma > 1) progress[mw] = static_cast<uint32_t>(entry) + 1u;
        tc_fence_after();
        if (kb == 0 && lane == 0) CSR_TRACE(1, it, 2);
        const int ks_here = min(4, ksteps_total - kb * 4);
        uint32_t a16 = ((slots_addr + slot * p.slot_bytes) >> 4) | a_lbo;
        uint32_t b16 = (p.stream_w ? ((slots_addr + slot * p.slot_bytes + p.win_slot_bytes) >> 4)
                                   : ((w_addr >> 4) + static_cast<uint32_t>(kb) * kb_w16)) | b_lbo;
        if (elect_one()) {
          const bool last_kb = kb == p.n_kblocks - 1;
          if constexpr (TALL_T == 0) {
            uint32_t acc = kb ? 1u : 0u;
            if constexpr (HYB_T) {
              // all taps but the last folded into N (B rows [0, (KW-1) npad)); the last tap as its own MMA: A one pixel further (start
              // address + 128 B; the hardware derives the 128B-swizzle phase from the address, base offset stays 0), B rows
              // [(KW-1) npad, KW npad), accumulated into the columns of tap KW-2
              const uint32_t idesc_a = make_idesc_bf16(kTileM, (KW_T - 1) * p.npad), idesc_b = make_idesc_bf16(kTileM, p.npad);
              const uint32_t b_last = static_cast<uint32_t>((KW_T - 1) * p.npad * 32) >> 4;
              const uint32_t d_last = d_tmem + static_cast<uint32_t>((KW_T - 2) * p.npad);
              for (int dy = 0; dy < p.KH; ++dy, a16 += row16) {
                for (int ks = 0; ks < ks_here; ++ks, b16 += b_step16) {
                  umma_bf16_split(d_tmem, a16 + ks * 2, a_hi, b16, b_hi, idesc_a, acc);
                  umma_bf16_split(d_last, a16 + 8 + ks * 2, a_hi, b16 + b_last, b_hi, idesc_b, 1u);
                  acc = 1;
                }
              }
            } else
            for (int dy = 0; dy < p.KH; ++dy, a16 += row16) {
              for (int ks = 0; ks < ks_here; ++ks, b16 += b_step16) {
                umma_bf16_split(d_tmem, a16 + ks * 2, a_hi, b16, b_hi, idesc, acc);
                acc = 1;
              }
            }
          } else {
            for (int hh = 0; hh < 2; ++hh) {               // M tile hh of the window: window rows [hh*TH, hh*TH + TH + KH - 1)
              uint32_t acc = kb ? 1u : 0u;
              uint32_t ah = a16 + static_cast<uint32_t>(hh * p.TH) * row16, bh = b16;
              const uint32_t dh = d_tmem + static_cast<uint32_t>(hh * nmma);
              for (int dy = 0; dy < p.KH; ++dy, ah += row16) {
                for (int ks = 0; ks < ks_here; ++ks, bh += b_step16) {
                  umma_bf16_split(dh, ah + ks * 2, a_hi, bh, b_hi, idesc, acc);
                  acc = 1;
                }
              }
              if (last_kb && hh == 0) umma_commit(bar_acc_full(buf));   // upper tile done: its epilogue can start
            }
          }
          if (last_kb) CSR_TRACE(1, it, 4);
          umma_commit(bar_a_empty(slot));                                  // window slot reusable once these MMAs have read it
          if (last_kb) umma_commit(bar_acc_full(buf + tall - 1));          // accumulator complete -> epilogue
          if (kb == p.n_kblocks - 1) CSR_TRACE(1, it, 5);
        }
        __syncwarp();
        if (kb == p.n_kblocks - 1 && lane == 0) CSR_TRACE(1, it, 3);
        ring_advance(1);
      }
      if (p.n_mma > 1) {                                                   // skip the other issuer's tile
        ring_advance(p.n_kblocks);
        entry += p.n_kblocks;
      }
      buf += p.n_mma * tall;
      if (buf >= NA) { buf -= NA; acc_phase ^= 1; }
      if (lane == 0) CSR_TRACE(1, it, 6);
    }
  } else {
    // ===================== epilogue: 16 warps in NG groups; group g takes every NG-th tile (accumulator buffer = tile % NA) ===
    // TMEM lane quadrant = warp % 4 (hardware rule); inside a group, warp j handles 8-channel chunks j/4, j/4 + wpg/4, ...
    // Each group runs its own latency chain (wait accumulator -> TMEM loads -> shuffle-sum -> stage -> bulk store), so NA
    // tiles are in flight in the epilogue while the MMA warp fills the next buffer.  The code is instruction-issue bound
    // (16 warps share 4 schedulers): everything tile-invariant is hoisted and per-pixel address arithmetic only exists on
    // the paths that need it (residual / gate / direct stores).
    const int ew = warp - 1 - kMmaWarps;
    const int g = ew / wpg;                              // epilogue group
    const int wj = ew - g * wpg;                         // warp within the group
    const int lane_grp = warp & 3;
    const int sub = wj >> 2;                             // first chunk of this warp
    const int cstep = wpg >> 2;                          // chunk-pair stride (1, 2 or 4)
    const int gthreads = wpg * 32;
    const bool tracer = (ew == 0 && lane == 0);
    const int m = lane_grp * 32 + lane;
    const int ty = m >> p.sw_shift;
    const int tx = m & (p.SW - 1);                       // window column
    const int n_chunks = ST_T == 3 ? 1 : p.npad >> 3;     // fp32 planar output: one channel, so one chunk (and of it only v[0] is live)
    const int PW = KW_T ? PW_T : p.PW;
    const bool col_ok = (tx >= PW) && (tx < PW + p.TW);
    const int srow = ty * p.TW + (tx - PW);              // staging row of this thread's pixel
    const int act = ACT_T >= 0 ? ACT_T : p.act;
    const bool has_r1 = RES_T >= 0 ? (RES_T & 1) != 0 : p.r1 != nullptr;
    const bool has_r2 = RES_T >= 0 ? (RES_T & 2) != 0 : p.r2 != nullptr;
    const bool has_gate = RES_T >= 0 ? (RES_T & 4) != 0 : p.gate != nullptr;
    const bool tma_store = ST_T >= 0 ? ST_T == 1 : (p.store_mode == kStoreStaged);
    const bool need_pix = !tma_store || has_r1 || has_r2 || has_gate;    // warp-uniform
    const uint32_t swz = (p.stage_row_bytes == 128) ? static_cast<uint32_t>(srow & 7) : 0u;   // SWIZZLE_128B staging rows
    const uint32_t srow_addr = stage_addr + static_cast<uint32_t>(g) * p.stage_bytes + static_cast<uint32_t>(srow * p.stage_row_bytes);
    const uint32_t sbuf = stage_addr + static_cast<uint32_t>(g) * p.stage_bytes;
    const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(lane_grp * 32) << 16);
    const int d0 = -PW, d1 = 1 - PW, d2 = 2 - PW;
    // Staged stores: the group's output tile sits in shared memory as TH*TW rows of stage_row_bytes; it is copied out in
    // 16-byte pieces, consecutive lanes taking consecutive pieces of a pixel row (full 32..128-byte segments per pixel).
    // Piece -> (row, column, channel group) is tile-invariant, so it is decoded once here.
    const int rp = p.stage_row_bytes >> 4;               // 16-byte pieces per staged pixel
    const int n_pieces = p.TH * p.TW * rp;
    uint32_t pc_s[4], pc_d[4], pc_yx[4];
    if (tma_store) {
      const int tid_g = wj * 32 + lane;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int i = tid_g + k * gthreads;
        const int sr = i / rp, c = i - sr * rp;
        const int dy = sr / p.TW, dx = sr - dy * p.TW;
        const uint32_t z = (p.stage_row_bytes == 128) ? static_cast<uint32_t>(sr & 7) : 0u;
        pc_s[k] = sbuf + static_cast<uint32_t>(sr * p.stage_row_bytes) + ((static_cast<uint32_t>(c) ^ z) << 4);
        pc_d[k] = static_cast<uint32_t>((dy * p.out_sy * p.out_W + dx * p.out_sx) * p.out_C + c * 8);
        pc_yx[k] = (i < n_pieces) ? ((static_cast<uint32_t>(dy) << 16) | static_cast<uint32_t>(dx)) : 0xffffffffu;
      }
    }
    int buf = g % NA;
    uint32_t acc_phase = 0;
    if constexpr (EARLY_T) {
      // One group of 16 warps, 64 output channels: warp (quadrant q, sub s) owns channels [16 s, 16 s + 16) of rows [32 q, 32 q + 32).
      static_assert(KW_T >= 1 && KW_T <= 3 && RES_T == 0 && ST_T == 1 && TALL_T == 0, "early-release epilogue: wide residual-free layers");
      const int ch_lo = sub * 16;
      uint32_t sb = 0;                                    // staging buffer of this tile
      const bool two_stage = p.n_stage == 2;
      constexpr int N2 = FUSE_T == 1 ? 32 : 16;           // columns of the fused second MMA
      Tile prev_tl = {0, 0, 0};
      int n_done = 0;
      // FUSE_T: read the second accumulator D2 of tile `t2` (its MMA has completed) and store the fused layer's output
      auto consume_d2 = [&](const Tile& t2) {
        tc_fence_after();
        if constexpr (FUSE_T == 1) {
          uint32_t r2[8];
          tmem_ld8(t_lane + static_cast<uint32_t>(NA * nacc) + sub * 8, r2);
          tmem_ld_wait();
          tc_fence_before();
          const int y = t2.y0 + ty, x = t2.x0 - PW_T + tx;
          if (col_ok && y < p.H && x < p.W && sub * 8 < p.n2) {
            const float* bias2_s = reinterpret_cast<const float*>(smem_gen + (b2_addr - smem_base)) + sub * 8;
            float v[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) v[j] = fmaxf(__uint_as_float(r2[j]) + bias2_s[j], 0.f);          // bias + ReLU (srcnn.py:16)
            __nv_bfloat16* o2 = reinterpret_cast<__nv_bfloat16*>(p.out2) + ((static_cast<size_t>(t2.n) * p.H + y) * p.W + x) * p.out2_C + p.out2_coff + sub * 8;
            *reinterpret_cast<uint4*>(o2) = make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
          }
        } else if constexpr (FUSE_T == 2) {
          // D2 row m belongs to STAGED row m = tile pixel (m / TW, m % TW) (the staged tile holds the TH x TW real outputs only).
          // Warp (quadrant, sub 0) stores taps 0..7, (quadrant, sub 1) tap 8, into the fp32 tap planes out2[tap][n][y][x].
          if (sub < 2) {
            uint32_t r2[8];
            tmem_ld8(t_lane + static_cast<uint32_t>(NA * nacc) + sub * 8, r2);
            tmem_ld_wait();
            const int py = m / p.TW, px = m - py * p.TW;
            const int y = t2.y0 + py, x = t2.x0 + px;
            if (m < p.TH * p.TW && y < p.H && x < p.W) {
              float* o2 = reinterpret_cast<float*>(p.out2) + (static_cast<size_t>(t2.n) * p.H + y) * p.W + x + static_cast<size_t>(sub * 8) * p.out2_plane;
              if (sub == 0) {
#pragma unroll
                for (int j = 0; j < 8; ++j) o2[static_cast<size_t>(j) * p.out2_plane] = __uint_as_float(r2[j]);
              } else {
                o2[0] = __uint_as_float(r2[0]);
              }
            }
          }
          tc_fence_before();
        }
      };
      for (int it = 0; ; ++it) {
        const int t = blockIdx.x + it * static_cast<int>(gridDim.x);
        if (t >= p.num_tiles) break;
        if (tracer) CSR_TRACE(2, it, 3);
        const Tile tl = decode_tile<0>(p, t);
        if (!two_stage && it > 0) named_bar_sync(1, gthreads);   // one staging buffer: every copy-out of the previous tile has been issued
        const uint32_t t_addr = t_lane + buf * nacc + ch_lo;
        mbar_wait(bar_acc_full(buf), acc_phase);           // the one bounded wait (see mbar_wait_spin)
        tc_fence_after();
        if (tracer) CSR_TRACE(2, it, 1);
        constexpr int KW_E = HYB_T ? KW_T - 1 : KW_T;      // column groups of the accumulator
        uint32_t raw[2][KW_E][8];
#pragma unroll
        for (int jj = 0; jj < 2; ++jj)
#pragma unroll
          for (int dx = 0; dx < KW_E; ++dx) tmem_ld8(t_addr + dx * p.npad + jj * 8, raw[jj][dx]);
        tmem_ld_wait();
        // the accumulator now lives in registers: the MMA warps may refill the buffer while the arithmetic runs
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_acc_empty(buf));
        if (tracer) CSR_TRACE(2, it, 0);
#pragma unroll
        for (int jj = 0; jj < 2; ++jj) {
          const int ch0 = ch_lo + jj * 8;
          float v[8];
          {
            const float4 b0 = *reinterpret_cast<const float4*>(bias_s + ch0);
            const float4 b1 = *reinterpret_cast<const float4*>(bias_s + ch0 + 4);
            v[0] = b0.x; v[1] = b0.y; v[2] = b0.z; v[3] = b0.w; v[4] = b1.x; v[5] = b1.y; v[6] = b1.z; v[7] = b1.w;
          }
#pragma unroll
          for (int dx = 0; dx < KW_E; ++dx) gather_add8(v, raw[jj][dx], dx - PW_T, lane);
          apply_act8(v, act);
          if (col_ok && ch0 < p.n_store)
            st_shared_v4(srow_addr + sb * p.stage_bytes + ((static_cast<uint32_t>(ch0 >> 3) ^ swz) << 4), pack_bf16x2(v[0], v[1]),
                         pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
        }
        if (tracer) CSR_TRACE(2, it, 4);
        if constexpr (FUSE_T) {
          // the second MMA of the PREVIOUS tile has had this tile's accumulator wait, loads and arithmetic to complete (two staging
          // buffers: it still reads the other one); with a single staging buffer its result is consumed right after the issue below
          if (two_stage && it > 0) {
            mbar_wait_spin(bar_d2, static_cast<uint32_t>(it - 1) & 1u);
            consume_d2(prev_tl);
          }
          fence_proxy_async_smem();                       // this thread's staged bf16 values -> visible to the tensor core's (async proxy) reads
        }
        named_bar_sync(1, gthreads);                      // the staged tile is complete (and every copy-out of tile it-1 has been issued)
        if (tracer) CSR_TRACE(2, it, 7);
        if constexpr (FUSE_T) {
          // second MMA: D2[128 x N2] = staged tile [128 rows x 64 ch, K-major, 128B swizzle] x W2^T, four k-steps, issued by one epilogue
          // thread.  FUSE_T 1: N2 = 32 output channels of a 1x1 conv; FUSE_T 2: N2 = 16 columns = the nine taps of a 3x3 -> 1 conv.
          if (warp == 1 + kMmaWarps) {
            if (it == 0) mbar_wait_spin(bar_w, 0);        // W2 arrived with the layer's own weights
            tc_fence_after();
            if (elect_one()) {
              const uint32_t a16 = ((stage_addr + sb * p.stage_bytes) >> 4) | ((16u >> 4) << 16);
              const uint32_t a_hi2 = (1024u >> 4) | (1u << 14) | (2u << 29);
              const uint32_t b16 = (w2_addr >> 4) | ((128u >> 4) << 16);
              const uint32_t b_hi2 = (256u >> 4) | (1u << 14);
              const uint32_t idesc2 = make_idesc_bf16(kTileM, N2);
#pragma unroll
              for (int ks = 0; ks < 4; ++ks)
                umma_bf16_split(tmem_base + static_cast<uint32_t>(NA * nacc), a16 + ks * 2, a_hi2, b16 + ks * ((N2 * 32) >> 4), b_hi2, idesc2, ks ? 1u : 0u);
              umma_commit(bar_d2);
            }
            __syncwarp();
          }
          if (!two_stage) {
            mbar_wait_spin(bar_d2, static_cast<uint32_t>(it) & 1u);
            consume_d2(tl);
          }
          prev_tl = tl;
          n_done = it + 1;
        } else {
        __nv_bfloat16* tile_out = reinterpret_cast<__nv_bfloat16*>(p.out) +
            ((static_cast<size_t>(tl.n) * p.out_H + (tl.y0 * p.out_sy + oy_eff)) * p.out_W + (tl.x0 * p.out_sx + p.out_ox)) * p.out_C +
            p.out_coff + static_cast<int>(blockIdx.y) * p.part_c;
        const uint32_t lim = (static_cast<uint32_t>(max(0, min(p.H - tl.y0, 0x7fff))) << 16) | static_cast<uint32_t>(min(p.W - tl.x0, 0x7fff));
#pragma unroll
        for (int k = 0; k < 2; ++k) {                     // <= 128 pixels x 8 pieces over 512 threads
          const bool ok = ((pc_yx[k] >> 16) < (lim >> 16)) && ((pc_yx[k] & 0xffffu) < (lim & 0xffffu));
          if (ok) {
            const uint4 val = ld_shared_v4(pc_s[k] + sb * p.stage_bytes);
            *reinterpret_cast<uint4*>(tile_out + pc_d[k]) = val;
            if constexpr (KW_T == 3 && ACT_T == 0 && RES_T == 0 && FUSE_T == 0) {
              // conv_first (the only plain 3x3 layer): its output has two consumers - the first dense block reads it from its concat
              // buffer, the trunk skip-add 33 layers later from a buffer of its own - so the tile is stored twice instead of running
              // the layer twice
              if (p.out_dup) {
                const uint32_t pixoff = ((pc_yx[k] >> 16) * p.out_sy * p.out_W + (pc_yx[k] & 0xffffu) * p.out_sx);
                __nv_bfloat16* dup = reinterpret_cast<__nv_bfloat16*>(p.out_dup) +
                    ((static_cast<size_t>(tl.n) * p.out_H + (tl.y0 * p.out_sy + oy_eff)) * p.out_W + (tl.x0 * p.out_sx + p.out_ox)) * p.dup_C + p.dup_coff;
                *reinterpret_cast<uint4*>(dup + static_cast<size_t>(pixoff) * p.dup_C + (pc_d[k] - pixoff * p.out_C)) = val;
              }
            }
          }
        }
        }
        if (tracer) CSR_TRACE(2, it, 2);
        if (two_stage) sb ^= 1u;
        if (++buf >= NA) { buf = 0; acc_phase ^= 1; }
      }
      if constexpr (FUSE_T) {
        if (two_stage && n_done > 0) {                    // the last tile's second MMA
          mbar_wait_spin(bar_d2, static_cast<uint32_t>(n_done - 1) & 1u);
          consume_d2(prev_tl);
        }
      }
    } else
    for (int it = g; ; it += NG) {                        // `it` counts M tiles; window = it >> tall_shift
      const int t = blockIdx.x + (it >> TALL_T) * static_cast<int>(gridDim.x);
      if (t >= p.num_tiles) break;
      if (tracer) CSR_TRACE(2, it, 3);
      Tile tl = decode_tile<TALL_T>(p, t);
      if constexpr (TALL_T) tl.y0 += (it & 1) * p.TH;
      bool valid = false;
      size_t pix = 0;
      int y = 0, x = 0;
      // residual / gate operands do not depend on the accumulator: fetch them before waiting for the MMAs
      uint4 q1[4], q2[4];
      if (need_pix) {
        y = tl.y0 + ty;
        x = tl.x0 - PW + tx;
        valid = col_ok && (y < p.H) && (x < p.W);
        pix = (static_cast<size_t>(tl.n) * p.H + y) * p.W + x;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int ch0 = (2 * (sub + (j >> 1) * cstep) + (j & 1)) * 8;
          const bool on = valid && (ch0 < p.n_store);
          q1[j] = (on && has_r1) ? ldg16(p.r1, pix, p.r1_C, p.r1_coff + ch0) : make_uint4(0, 0, 0, 0);
          if (has_gate)   // the gate shares the second operand slot with r2 (the host never sets both)
            q2[j] = (on && ch0 >= p.gate_from) ? ldg16(p.gate, pix, p.gate_C, p.gate_coff + ch0)
                                               : make_uint4(0x3f803f80u, 0x3f803f80u, 0x3f803f80u, 0x3f803f80u);
          else
            q2[j] = (on && has_r2) ? ldg16(p.r2, pix, p.r2_C, p.r2_coff + ch0) : make_uint4(0, 0, 0, 0);
        }
      }
      if (tma_store) named_bar_sync(1 + g, gthreads);   // every thread of the group has copied out the previous tile
      if (tracer) CSR_TRACE(2, it, 0);
      const uint32_t t_addr = t_lane + buf * nacc;
      mbar_wait(bar_acc_full(buf), acc_phase);             // the one bounded wait (see mbar_wait_spin)
      tc_fence_after();
      if (tracer) CSR_TRACE(2, it, 1);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int c = 2 * (sub + (j >> 1) * cstep) + (j & 1);   // adjacent chunk pairs: 16 channels = one 32-byte sector
        if (c < n_chunks) {                               // warp-uniform
          const int ch0 = c * 8;
          float v[8];
          {
            const float4 b0 = *reinterpret_cast<const float4*>(bias_s + ch0);
            const float4 b1 = *reinterpret_cast<const float4*>(bias_s + ch0 + 4);
            v[0] = b0.x; v[1] = b0.y; v[2] = b0.z; v[3] = b0.w; v[4] = b1.x; v[5] = b1.y; v[6] = b1.z; v[7] = b1.w;
          }
          // (issuing chunk j+1's TMEM loads ahead of chunk j's arithmetic - double-buffered or into the same registers -
          // spills under the 104-register cap and measured 0.7 ms slower per cfg2 step)
          if constexpr (KW_T == 1) {
            uint32_t r0[8];
            tmem_ld8(t_addr + ch0, r0);
            tmem_ld_wait();
            gather_add8(v, r0, 0, lane);
          } else if constexpr (KW_T == 2) {
            uint32_t r0[8], r1[8];
            tmem_ld8(t_addr + ch0, r0);
            tmem_ld8(t_addr + p.npad + ch0, r1);
            tmem_ld_wait();
            gather_add8(v, r0, d0, lane);
            gather_add8(v, r1, d1, lane);
          } else if constexpr (KW_T == 3) {
            uint32_t r0[8], r1[8], r2[8];
            tmem_ld8(t_addr + ch0, r0);
            tmem_ld8(t_addr + p.npad + ch0, r1);
            tmem_ld8(t_addr + 2 * p.npad + ch0, r2);
            tmem_ld_wait();
            gather_add8(v, r0, d0, lane);
            gather_add8(v, r1, d1, lane);
            gather_add8(v, r2, d2, lane);
          } else {
            for (int dx = 0; dx < KW; ++dx) {
              uint32_t r[8];
              tmem_ld8(t_addr + dx * p.npad + ch0, r);
              tmem_ld_wait();
              gather_add8(v, r, dx - PW, lane);
            }
          }
          apply_act8(v, act, p.act_slope);
          if (need_pix) {
            if (has_r1) fma_residual8(v, q1[j], p.s1);
            if (has_gate) gate8(v, q2[j], p.gate_neg);
            else if (has_r2) fma_residual8(v, q2[j], p.s2);
          }
          if (tma_store) {
            if (col_ok && ch0 < p.n_store)
              st_shared_v4(srow_addr + ((static_cast<uint32_t>(c) ^ swz) << 4), pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]),
                           pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
          } else if (valid) {
            const size_t opix = (static_cast<size_t>(tl.n) * p.out_H + (y * p.out_sy + oy_eff)) * p.out_W + (x * p.out_sx + p.out_ox);
            const int smode = ST_T == 3 ? static_cast<int>(kStoreF32Planar) : p.store_mode;
            if (smode == kStoreF32Planar) {
              if (c == 0) reinterpret_cast<float*>(p.out)[opix] = v[0];
            } else {
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                if (ch0 + i < p.n_store) {
                  if (p.store_mode == kStoreF32Nhwc)
                    reinterpret_cast<float*>(p.out)[opix * p.out_C + p.out_coff + static_cast<int>(blockIdx.y) * p.part_c + ch0 + i] = v[i];
                  else
                    reinterpret_cast<__nv_bfloat16*>(p.out)[opix * p.out_C + p.out_coff + static_cast<int>(blockIdx.y) * p.part_c + ch0 + i] = __float2bfloat16_rn(v[i]);
                }
              }
            }
          }
        }
      }
      if (tracer) CSR_TRACE(2, it, 4);
      // all TMEM reads of this warp are complete (wait::ld above): hand the accumulator buffer back to the MMA warp
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_acc_empty(buf));
      if (tma_store) {
        named_bar_sync(1 + g, gthreads);                  // the staged tile is complete
        if (tracer) CSR_TRACE(2, it, 7);
        __nv_bfloat16* tile_out = reinterpret_cast<__nv_bfloat16*>(p.out) +
            ((static_cast<size_t>(tl.n) * p.out_H + (tl.y0 * p.out_sy + oy_eff)) * p.out_W + (tl.x0 * p.out_sx + p.out_ox)) * p.out_C +
            p.out_coff + static_cast<int>(blockIdx.y) * p.part_c;
        // (the lower M tile of a window may lie entirely below the image: no piece passes)
        const uint32_t lim = (static_cast<uint32_t>(max(0, min(p.H - tl.y0, 0x7fff))) << 16) | static_cast<uint32_t>(min(p.W - tl.x0, 0x7fff));
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          // piece inside the image: dy < H - y0 and dx < W - x0 (both halves compared at once; 0xffffffff = no piece)
          const bool ok = ((pc_yx[k] >> 16) < (lim >> 16)) && ((pc_yx[k] & 0xffffu) < (lim & 0xffffu));
          if (ok) {
            const uint4 val = ld_shared_v4(pc_s[k]);
            *reinterpret_cast<uint4*>(tile_out + pc_d[k]) = val;
          }
        }
      }
      if (tracer) CSR_TRACE(2, it, 2);
      buf += NG;
      if (buf >= NA) { buf -= NA; acc_phase ^= 1; }
    }
  }

done:
  tc_fence_before();
  __syncthreads();
  timeline_end(p.timeline, p.launch_id);
  if (warp == 1) {
    __syncwarp();
    tc_fence_after();
    tmem_dealloc(tmem_base, p.tmem_cols);
  }
}

size_t conv_smem_bytes(const ConvParams& p) {
  return 1024 /*alignment slack*/ + static_cast<size_t>(p.n_slots) * p.slot_bytes + static_cast<size_t>(p.n_stage) * p.stage_bytes +
         (((p.stream_w ? 0 : p.w_bytes) + 127) & ~127) + (p.fuse2 ? p.w2_bytes + 128 : 0) + 256 /*bias*/ +
         8 * (18 + 2 * p.n_slots) + 32;
}

template <int KW_T, int PW_T, int ACT_T, int RES_T, int ST_T, int TALL_T = 0, int EARLY_T = 0, int FUSE_T = 0, int HYB_T = 0>
static int launch_t(const ConvParams& p, const CUtensorMap& tmap, int num_sms, cudaStream_t stream) {
  const size_t smem = conv_smem_bytes(p);
  if (smem > static_cast<size_t>(kSmemLimit)) return static_cast<int>(cudaErrorInvalidValue);
  // the attribute is per device (and per template instantiation): one process may drive several GPUs
  static bool configured[64] = {};
  auto kern = conv_tc_kernel<KW_T, PW_T, ACT_T, RES_T, ST_T, TALL_T, EARLY_T, FUSE_T, HYB_T>;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return static_cast<int>(cudaErrorInvalidDevice);
  if (!configured[dev]) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit);
    if (e != cudaSuccess) return static_cast<int>(e);
    configured[dev] = true;
  }
  cudaLaunchConfig_t cfg{};
  // parts > 1: blockIdx.y selects the output-channel part (same geometry, weights / bias / output slice at constant strides)
  const int parts = p.parts > 1 ? p.parts : 1;
  const int per_part = num_sms / parts > 0 ? num_sms / parts : 1;
  cfg.gridDim = dim3(p.num_tiles < per_part ? p.num_tiles : per_part, parts);
  cfg.blockDim = dim3(kConvThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = p.use_pdl ? 1 : 0;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return static_cast<int>(cudaLaunchKernelEx(&cfg, kern, p, tmap));
}

int launch_conv_tc(const ConvParams& p, const CUtensorMap& tmap, int num_sms, cudaStream_t stream) {
  const int res = (p.r1 ? 1 : 0) | (p.r2 ? 2 : 0) | (p.gate ? 4 : 0);
  if ((res & 6) == 6) return static_cast<int>(cudaErrorInvalidValue);   // r2 and gate share an operand slot
  if (p.tall_shift) {
    // two-M-tile windows: the thin layers only (four accumulator buffers)
    if ((p.n_acc != 4 && p.n_acc != 8) || p.n_groups != 4) return static_cast<int>(cudaErrorInvalidValue);
    if (p.store_mode == kStoreStaged && !p.force_generic && p.KW == 3 && p.PW == 1 && p.act == 1 && res == 0)
      return launch_t<3, 1, 1, 0, 1, 1>(p, tmap, num_sms, stream);         // RDB conv1-4
    if (p.store_mode == kStoreStaged && !p.force_generic && p.KW == 1 && p.PW == 0 && p.act == 2 && res == 0)
      return launch_t<1, 0, 2, 0, 1, 1>(p, tmap, num_sms, stream);         // srcnn.conv2
    if (p.store_mode == kStoreStaged && !p.force_generic && p.KW == 3 && p.PW == 1 && p.act == 0 && res == 4)
      return launch_t<3, 1, 0, 4, 1, 1>(p, tmap, num_sms, stream);         // dense-block input gradients of x1..x4 (gated)
    if (p.store_mode == kStoreStaged && !p.force_generic && p.KW == 3 && p.PW == 1 && p.act == 0 && res == 5)
      return launch_t<3, 1, 0, 5, 1, 1>(p, tmap, num_sms, stream);
    if (p.store_mode == kStoreStaged && !p.force_generic && p.KW == 1 && p.PW == 0 && p.act == 0 && res == 4)
      return launch_t<1, 0, 0, 4, 1, 1>(p, tmap, num_sms, stream);         // srcnn.conv3 input gradient over the gradient im2col
    if (p.store_mode == kStoreF32Planar && !p.force_generic && p.KW == 3 && p.PW == 1 && p.act == 0 && res == 0)
      return launch_t<3, 1, 0, 0, 3, 1>(p, tmap, num_sms, stream);         // conv_last
    if (p.store_mode == kStoreF32Planar && !p.force_generic && p.KW == 5 && p.PW == 2 && p.act == 0 && res == 0)
      return launch_t<5, 2, 0, 0, 3, 1>(p, tmap, num_sms, stream);         // srcnn.conv3
    switch (p.KW) {
      case 1: return launch_t<1, 0, -1, -1, -1, 1>(p, tmap, num_sms, stream);
      case 3: if (p.PW == 1) return launch_t<3, 1, -1, -1, -1, 1>(p, tmap, num_sms, stream);
      default: return launch_t<0, 0, -1, -1, -1, 1>(p, tmap, num_sms, stream);
    }
  }
  if (p.early) {
    // wide residual-free layers with the early-release epilogue (one 16-warp group, two staging buffers)
    if (p.store_mode != kStoreStaged || p.n_groups != 1 || p.n_stage < 1 || p.n_stage > 2 || p.npad != 64 || res != 0 || p.force_generic)
      return static_cast<int>(cudaErrorInvalidValue);
    if (p.fuse2 == 2) {
      // HRconv (3x3, LeakyReLU) + the nine tap planes of conv_last (3x3, 64 -> 1) in one launch
      if (p.KW != 3 || p.PW != 1 || p.act != 1 || p.stage_row_bytes != 128 || p.w2_bytes != 2048 || p.n2 != 9 || p.out2_plane <= 0 ||
          p.tmem_cols < p.n_acc * (p.hyb ? p.KW - 1 : p.KW) * p.npad + 16 || p.parts > 1)
        return static_cast<int>(cudaErrorInvalidValue);
      if (p.hyb) return launch_t<3, 1, 1, 0, 1, 0, 1, 2, 1>(p, tmap, num_sms, stream);
      return launch_t<3, 1, 1, 0, 1, 0, 1, 2>(p, tmap, num_sms, stream);
    }
    if (p.fuse2) {
      // srcnn.conv1 (x-im2col folded, ReLU) + srcnn.conv2 (1x1, ReLU) in one launch
      if (p.KW != 1 || p.PW != 0 || p.act != 2 || p.stage_row_bytes != 128 || p.w2_bytes != 4096 || p.n2 < 8 || p.n2 > 32 || (p.n2 & 7) ||
          p.tmem_cols < p.n_acc * p.KW * p.npad + 32 || p.parts > 1)
        return static_cast<int>(cudaErrorInvalidValue);
      return launch_t<1, 0, 2, 0, 1, 0, 1, 1>(p, tmap, num_sms, stream);
    }
#define CSR_EARLY(KW_, PW_, ACT_)                                                                                    \
    if (p.KW == KW_ && p.PW == PW_ && p.act == ACT_) {                                                                 \
      if constexpr (KW_ >= 2) { if (p.hyb) return launch_t<KW_, PW_, ACT_, 0, 1, 0, 1, 0, 1>(p, tmap, num_sms, stream); } \
      return launch_t<KW_, PW_, ACT_, 0, 1, 0, 1>(p, tmap, num_sms, stream);                                           \
    }
    CSR_EARLY(3, 1, 1)   // HRconv
    CSR_EARLY(3, 1, 0)   // conv_first
    CSR_EARLY(2, 0, 1)   // upconv sub-pixel phases
    CSR_EARLY(2, 1, 1)
    CSR_EARLY(1, 0, 2)   // srcnn.conv1 (x-im2col folded)
#undef CSR_EARLY
    return static_cast<int>(cudaErrorInvalidValue);
  }
#define CSR_CASE(KW_, PW_, ACT_, RES_, ST_)                                                                  \
  if (p.store_mode == (ST_ == 1 ? kStoreStaged : kStoreF32Planar) && !p.force_generic && p.KW == KW_ &&   \
      p.PW == PW_ && p.act == ACT_ && res == RES_)                                                           \
    return launch_t<KW_, PW_, ACT_, RES_, ST_>(p, tmap, num_sms, stream);
  // the layer shapes of the generator forward (esrgan.py / srcnn.py) ...
  CSR_CASE(3, 1, 1, 0, 1)   // RDB conv1-4, HRconv: lrelu
  CSR_CASE(3, 1, 0, 0, 1)   // conv_first
  CSR_CASE(3, 1, 4, 0, 1)   // discriminator convs: LeakyReLU(act_slope)
  CSR_CASE(3, 1, 0, 1, 1)   // RDB conv5 (*0.2 + x), trunk_conv (+ fea)
  CSR_CASE(3, 1, 0, 3, 1)   // RDB3 conv5 (*0.2 + x, *0.2 + x_rrdb)
  CSR_CASE(2, 0, 1, 0, 1)   // upconv sub-pixel phases
  CSR_CASE(2, 1, 1, 0, 1)
  CSR_CASE(1, 0, 2, 0, 1)   // srcnn.conv1 (x-im2col folded), srcnn.conv2: relu
  CSR_CASE(3, 1, 0, 0, 3)   // conv_last -> fp32 planar
  CSR_CASE(5, 2, 0, 0, 3)   // srcnn.conv3 -> fp32 planar (the generator's output)
  // ... and of its backward (input-gradient convs: accumulate in place, LeakyReLU-derivative gate)
  CSR_CASE(3, 1, 0, 5, 1)
  CSR_CASE(3, 1, 0, 4, 1)
  CSR_CASE(1, 0, 0, 4, 1)   // 1x1 input gradients with a ReLU / LeakyReLU gate: srcnn.conv2, and conv_last / srcnn.conv3 over the gradient im2col
  CSR_CASE(2, 0, 0, 0, 1)   // upconv input gradients, transposed sub-pixel phases: the first phase stores,
  CSR_CASE(2, 1, 0, 1, 1)   // the others accumulate in place,
  CSR_CASE(2, 0, 0, 1, 1)
  CSR_CASE(2, 1, 0, 5, 1)   // and the last one of upconv2 also applies upconv1's LeakyReLU gate
#undef CSR_CASE
  switch (p.KW) {
    case 1: return launch_t<1, 0, -1, -1, -1>(p, tmap, num_sms, stream);
    case 3: if (p.PW == 1) return launch_t<3, 1, -1, -1, -1>(p, tmap, num_sms, stream);
    default: return launch_t<0, 0, -1, -1, -1>(p, tmap, num_sms, stream);
  }
}

}  // namespace csr

// conv1..conv4 of a ResidualDenseBlock (climsr/models/esrgan.py:33-36, gc = 16) as ONE persistent kernel.
//
// Why: layer by layer, each of these 3x3 convs (64..112 -> 16 channels) is a ~17-20 us launch of which only ~6-10 us is
// tensor work - the rest is the grid-wide dependency between consecutive layers: drain of the last tiles' epilogues, kernel
// prologue (barriers, TMEM, weights), first window's TMA latency, pipeline fill (profiles/r02_launches_plain.csv: 132 such
// launches = 44 % of a cfg2 forward).  The data dependency is local, though: conv_{k+1} on a tile only needs conv_k on that
// tile and its eight neighbours.  Here every CTA walks layer after layer over ITS windows (same window -> CTA assignment in
// every layer) and the TMA producer waits, per window, for the completion counters of the <= 9 windows of the previous layer
// it reads: the MMA / epilogue pipeline never drains between layers, weights of the next layer stream into a second
// shared-memory buffer while the current layer runs, and TMEM / barriers are set up once per dense block.
//
// Activations travel through the concat buffer in global memory (L2) exactly as in the per-layer path - written by the
// epilogue's generic-proxy stores, made visible by  bar.sync -> fence -> red.release.gpu  on a per-(layer, window) counter,
// read by  ld.acquire.gpu -> fence.proxy.async -> TMA.  Tile geometry, MMA order and epilogue arithmetic are those of
// conv_tc_kernel<3,1,1,0,1,0,1> (two M tiles per window, horizontal taps folded into N = 48, eight accumulators, four
// epilogue groups), so the results are bit-identical to four per-layer launches.
//
// Whole-row windows (WR_T, DenseParams::whole_row): on a 32- or 64-pixel-wide map a window is 2*TH whole image rows starting at
// x = 0 - no halo columns, every GEMM row an output - and depends on at most three windows of the previous layer (above, itself,
// below).  The edge taps come from row_edge_put / row_edge_get (ptx.cuh), so the outputs stay bit-identical.
//
// Deadlock freedom: the grid never exceeds the SM count and every CTA takes a whole SM (shared memory), so all CTAs are
// co-resident once the previous grid has drained; within a CTA layer k never waits for layer k+1.  Every wait on another
// CTA is bounded and traps instead of hanging.
#include <cstdio>

#include "conv_tc.cuh"
#include "ptx.cuh"
#include "rdb_tc.cuh"

namespace csr {

namespace {

constexpr int kNpad = 16;             // output channels per layer (gc)
constexpr int kNmma = 3 * kNpad;      // UMMA N: three horizontal taps folded into the columns
constexpr int kAcc = 8;               // accumulator buffers (two per window)
constexpr int kGroups = 4;            // epilogue groups of four warps (one per TMEM lane quadrant)

struct Win {
  int n, y0, x0, ty, tx;
};

__device__ __forceinline__ int fast_div(int t, unsigned long long magic) {
  return static_cast<int>((static_cast<unsigned long long>(static_cast<unsigned>(t)) * magic) >> 40);
}
__device__ __forceinline__ Win decode_win(const DenseParams& p, int t) {
  Win r;
  r.n = fast_div(t, p.magic_img);
  const int rem = t - r.n * p.tiles_per_img;
  r.ty = fast_div(rem, p.magic_row);
  r.tx = rem - r.ty * p.tiles_x;
  r.y0 = r.ty * (p.TH << 1);
  r.x0 = r.tx * p.TW;
  return r;
}

__device__ __forceinline__ unsigned ld_acquire_gpu(const unsigned* ptr) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(ptr) : "memory");
  return v;
}
__device__ __forceinline__ void red_release_gpu_add(unsigned* ptr, unsigned v) {
  asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(ptr), "r"(v) : "memory");
}
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }

static __device__ __noinline__ void flag_timeout(int layer, int win, unsigned have) {
  printf("climsr_b200: dense-block dependency timeout: block %d waits for layer %d window %d (counter %u)\n", blockIdx.x, layer, win, have);
  __trap();
}

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

}  // namespace

template <int WR_T>
__global__ void __launch_bounds__(kConvThreads, 1)
dense_block_kernel(const DenseParams p, const __grid_constant__ CUtensorMap tmap) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const int S = p.n_slots;
  const uint32_t slots_addr = smem_base;
  const uint32_t stage_addr = slots_addr + static_cast<uint32_t>(S) * p.slot_bytes;
  const uint32_t w_addr = stage_addr + static_cast<uint32_t>(kGroups) * p.stage_bytes;
  const uint32_t bias_addr = w_addr + 2u * p.wbuf_bytes;                     // kDenseMaxLayers x 16 fp32
  const uint32_t bar_addr = bias_addr + kDenseMaxLayers * kNpad * 4;
  // barriers: w_full[2], w_free[2], a_full[S], a_empty[S], acc_full[8], acc_empty[8]
  auto bar_w_full = [&](int b) { return bar_addr + 8u * b; };
  auto bar_w_free = [&](int b) { return bar_addr + 8u * (2 + b); };
  auto bar_a_full = [&](int s) { return bar_addr + 8u * (4 + s); };
  auto bar_a_empty = [&](int s) { return bar_addr + 8u * (4 + S + s); };
  auto bar_acc_full = [&](int b) { return bar_addr + 8u * (4 + 2 * S + b); };
  auto bar_acc_empty = [&](int b) { return bar_addr + 8u * (4 + 2 * S + kAcc + b); };
  const uint32_t tmem_slot_addr = bar_addr + 8u * (4 + 2 * S + 2 * kAcc);
  const uint32_t xchg_addr = (tmem_slot_addr + 12u + 15u) & ~15u;            // WR_T: 96 zero bytes, then the row_edge_put / get slots
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  float* bias_s = reinterpret_cast<float*>(smem_gen + (bias_addr - smem_base));
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem_gen + (tmem_slot_addr - smem_base));
  volatile uint32_t* progress = tmem_slot + 1;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int nl = p.n_layers;

  griddep_launch_dependents();

  if (threadIdx.x == 0) {
    progress[0] = 0;
    progress[1] = 0;
    tma_prefetch_desc(&tmap);
    for (int b = 0; b < 2; ++b) {
      mbar_init(bar_w_full(b), 1);
      mbar_init(bar_w_free(b), kMmaWarps);                 // both MMA issuers have retired the layer's MMAs
    }
    for (int s = 0; s < S; ++s) {
      mbar_init(bar_a_full(s), 1);
      mbar_init(bar_a_empty(s), 1);
    }
    for (int b = 0; b < kAcc; ++b) {
      mbar_init(bar_acc_full(b), 1);
      mbar_init(bar_acc_empty(b), kEpilogueWarps / kGroups);
    }
    fence_mbar_init();
    fence_proxy_async_smem();
    // weights are constants (not produced by the previous kernel): layers 0 and 1 start loading before griddepcontrol.wait
    for (int l = 0; l < 2 && l < nl; ++l) {
      mbar_arrive_expect_tx(bar_w_full(l), p.L[l].w_bytes);
      const uint8_t* wsrc = reinterpret_cast<const uint8_t*>(p.L[l].wpk);
      for (int off = 0; off < p.L[l].w_bytes; off += 32768)
        bulk_load(w_addr + l * p.wbuf_bytes + off, wsrc + off, min(32768, p.L[l].w_bytes - off), bar_w_full(l));
    }
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot_addr, 512);
    tmem_relinquish();
  }
  for (int i = threadIdx.x; i < nl * kNpad; i += blockDim.x) bias_s[i] = p.L[i / kNpad].bias[i % kNpad];
  if (WR_T && threadIdx.x < 6) st_shared_v4(xchg_addr + 16u * threadIdx.x, 0u, 0u, 0u, 0u);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  griddep_wait();
  timeline_start(p.timeline, p.launch_id);

  const int G = static_cast<int>(gridDim.x);
  const int nwin = (p.num_tiles - static_cast<int>(blockIdx.x) + G - 1) / G;   // windows of this CTA in every layer (>= 1)

  if (warp == 0) {
    // ===================== TMA producer =====================
    int slot = 0;
    uint32_t phase = 0;
    for (int l = 0; l < nl; ++l) {
      const unsigned* fl = p.flags + static_cast<size_t>(l > 0 ? l - 1 : 0) * p.num_tiles;
      for (int t = blockIdx.x; t < p.num_tiles; t += G) {
        const Win w = decode_win(p, t);
        if (l > 0) {
          // the windows of layer l-1 this window reads (1-pixel halo): itself and its <= 8 neighbours inside the image (whole rows:
          // the window above and below)
          if (lane < (WR_T ? 3 : 9)) {
            const int dy = WR_T ? lane - 1 : lane / 3 - 1, dx = WR_T ? 0 : lane - (lane / 3) * 3 - 1;
            const int yy = w.ty + dy, xx = w.tx + dx;
            if (yy >= 0 && yy < p.tiles_y && xx >= 0 && xx < p.tiles_x) {
              const int idx = w.n * p.tiles_per_img + yy * p.tiles_x + xx;
              unsigned have, spins = 0;
              while ((have = ld_acquire_gpu(fl + idx)) < 2u) {
                if (++spins > (1u << 24)) flag_timeout(l - 1, idx, have);
                __nanosleep(40);
              }
            }
          }
          __syncwarp();
          // other CTAs' generic-proxy stores (acquired above) -> this warp's async-proxy reads.  Once per window, not per TMA
          // issue: the fence also waits for the warp's loads in flight (62 -> 53 us per dense block); without any proxy fence the
          // block takes 50 us, a writer-side fence.proxy.async.global in the epilogue 52 us (profiles/r02_dense_block_notes.txt)
          fence_proxy_async_all();
        }
        for (int kb = 0; kb < p.L[l].n_kblocks; ++kb) {
          mbar_wait_spin(bar_a_empty(slot), phase ^ 1);
          if (elect_one()) {
            mbar_arrive_expect_tx(bar_a_full(slot), p.win_bytes);
            tma_load_4d(slots_addr + slot * p.slot_bytes, &tmap, bar_a_full(slot), kb * 64, w.x0 - (WR_T ? 0 : 1), w.y0 - 1, w.n);
          }
          __syncwarp();
          if (++slot == S) { slot = 0; phase ^= 1; }
        }
      }
      // weights of layer l+1 go into the buffer layer l-1 used: free once both issuers have retired layer l-1's MMAs, which
      // is long before the producer gets here (it runs at most a ring ahead of the MMAs of layer l)
      if (l >= 1 && l + 1 < nl) {
        const int b = (l + 1) & 1;
        mbar_wait_spin(bar_w_free(b), static_cast<uint32_t>((l - 1) >> 1) & 1u);
        if (elect_one()) {
          mbar_arrive_expect_tx(bar_w_full(b), p.L[l + 1].w_bytes);
          const uint8_t* wsrc = reinterpret_cast<const uint8_t*>(p.L[l + 1].wpk);
          for (int off = 0; off < p.L[l + 1].w_bytes; off += 32768)
            bulk_load(w_addr + b * p.wbuf_bytes + off, wsrc + off, min(32768, p.L[l + 1].w_bytes - off), bar_w_full(b));
        }
        __syncwarp();
      }
    }
  } else if (warp <= kMmaWarps) {
    // ===================== MMA issuers: alternate windows of the CTA's global window sequence q = layer * nwin + it ========
    const int mw = warp - 1;
    const uint32_t idesc = make_idesc_bf16(kTileM, kNmma);
    constexpr uint32_t b_step16 = static_cast<uint32_t>(kNmma * 32) >> 4;     // one (dy, k-step) weight block in 16-byte units
    constexpr uint32_t kb_w16 = 3u * 4u * b_step16;                           // one full 64-channel k-block of weights
    const uint32_t row16 = static_cast<uint32_t>(p.SW) * 8u;                  // one window row in 16-byte units
    const uint32_t a_hi = (1024u >> 4) | (1u << 14) | (2u << 29);             // SBO = 8 rows x 128 B, version 1, SWIZZLE_128B
    const uint32_t b_hi = (256u >> 4) | (1u << 14);
    const uint32_t a_lbo = (16u >> 4) << 16, b_lbo = (128u >> 4) << 16;
    int slot = 0;
    uint32_t phase = 0;
    int entry = 0;                                                            // ring entry index of (window, k-block)
    int q = 0;
    uint32_t own = 0;                                                         // bit (e & 31): ring entry e belongs to this issuer
    for (int l = 0; l < nl; ++l) {
      const int nkb = p.L[l].n_kblocks, ksteps = p.L[l].ksteps;
      const uint32_t wl_addr = w_addr + static_cast<uint32_t>(l & 1) * p.wbuf_bytes;
      bool have_w = false;
      for (int it = 0; it < nwin; ++it, ++q) {
        if ((q & 1) != mw) {                                                  // the other issuer's window
          for (int i = 0; i < nkb; ++i, ++entry) {
            own &= ~(1u << (entry & 31));
            if (++slot == S) { slot = 0; phase ^= 1; }
          }
          continue;
        }
        if (!have_w) {
          mbar_wait_spin(bar_w_full(l & 1), static_cast<uint32_t>(l >> 1) & 1u);
          have_w = true;
        }
        const int buf = (q & 3) * 2;
        const uint32_t acc_par = (static_cast<uint32_t>(q) >> 2) & 1u;
        mbar_wait_spin(bar_acc_empty(buf), acc_par ^ 1);
        mbar_wait_spin(bar_acc_empty(buf + 1), acc_par ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + buf * kNmma;
        for (int kb = 0; kb < nkb; ++kb, ++entry) {
          // the slot ring is shared by both issuers: a parity wait is only unambiguous if the previous fill of this slot has
          // been seen full (own entries trivially, the other issuer's through its progress word) - see conv_tc.cu
          own |= 1u << (entry & 31);
          const int need = entry - S;                                         // S <= 8 < 32: the ownership bit of `need` is still valid
          if (need >= 0 && !((own >> (need & 31)) & 1u)) {
            while (progress[1 - mw] <= static_cast<uint32_t>(need)) {
            }
          }
          mbar_wait_spin(bar_a_full(slot), phase);
          progress[mw] = static_cast<uint32_t>(entry) + 1u;
          tc_fence_after();
          const int ks_here = min(4, ksteps - kb * 4);
          const uint32_t a16 = ((slots_addr + slot * p.slot_bytes) >> 4) | a_lbo;
          const uint32_t b16 = ((wl_addr >> 4) + static_cast<uint32_t>(kb) * kb_w16) | b_lbo;
          if (elect_one()) {
            const bool last_kb = kb == nkb - 1;
            for (int hh = 0; hh < 2; ++hh) {                 // M tile hh of the window: window rows [hh*TH, hh*TH + TH + 2)
              uint32_t acc = kb ? 1u : 0u;
              uint32_t ah = a16 + static_cast<uint32_t>(hh * p.TH) * row16, bh = b16;
              const uint32_t dh = d_tmem + static_cast<uint32_t>(hh * kNmma);
              for (int dy = 0; dy < 3; ++dy, ah += row16) {
                for (int ks = 0; ks < ks_here; ++ks, bh += b_step16) {
                  umma_bf16_split(dh, ah + ks * 2, a_hi, bh, b_hi, idesc, acc);
                  acc = 1;
                }
              }
              if (last_kb) umma_commit(bar_acc_full(buf + hh));
            }
            umma_commit(bar_a_empty(slot));
          }
          __syncwarp();
          if (++slot == S) { slot = 0; phase ^= 1; }
        }
      }
      // this issuer's MMAs of layer l: once they retire, the layer's weight buffer may be overwritten (layer l+2)
      if (elect_one()) umma_commit(bar_w_free(l & 1));
      __syncwarp();
    }
  } else {
    // ===================== epilogue: four groups of four warps; group g takes M tiles m = 2q + half with m % 4 == g ==========
    const int ew = warp - 1 - kMmaWarps;
    const int g = ew >> 2;
    const int wj = ew & 3;
    const int lane_grp = warp & 3;                        // TMEM lane quadrant (hardware rule: warp % 4)
    const int m_row = lane_grp * 32 + lane;
    const int ty = m_row >> p.sw_shift;
    const int tx = m_row & (p.SW - 1);
    const int x_off = WR_T ? 0 : 1;                       // window column of the window's first output
    const bool col_ok = WR_T || ((tx >= 1) && (tx < 1 + p.TW));
    const int srow = ty * p.TW + (tx - x_off);
    // WR_T, 64-pixel rows: the warps of TMEM lane quadrants 2k and 2k+1 of a group hold the two halves of a row
    const bool row_pair = WR_T && p.SW == 64;
    const bool row_left = (lane_grp & 1) == 0;
    const int pair = (g << 1) + (lane_grp >> 1);          // 0..7
    uint32_t xdst, xsrc;                                  // 64 bytes per chunk
    edge_addrs(xchg_addr + 96u + static_cast<uint32_t>(pair) * 128u, xchg_addr, row_pair, row_left, lane, &xdst, &xsrc);
    const uint32_t sbuf = stage_addr + static_cast<uint32_t>(g) * p.stage_bytes;
    const uint32_t srow_addr = sbuf + static_cast<uint32_t>(srow * 32);
    const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(lane_grp * 32) << 16);
    // copy-out: the staged tile (TH*TW pixels x 32 bytes) leaves in 16-byte pieces, two per thread of the group
    const int n_pieces = p.TH * p.TW * 2;
    uint32_t pc_s[2], pc_d[2], pc_yx[2];
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int i = wj * 32 + lane + k * 128;
      const int sr = i >> 1, c = i & 1;
      const int dy = sr / p.TW, dx = sr - dy * p.TW;
      pc_s[k] = sbuf + static_cast<uint32_t>(sr * 32 + c * 16);
      pc_d[k] = static_cast<uint32_t>((dy * p.W + dx) * p.C + c * 8);
      pc_yx[k] = (i < n_pieces) ? ((static_cast<uint32_t>(dy) << 16) | static_cast<uint32_t>(dx)) : 0xffffffffu;
    }
    const int m_total = 2 * nwin * nl;
    // (layer, it) of M tile m, advanced incrementally: q = m >> 1 = l * nwin + it
    int l = 0, it = g >> 1;
    while (it >= nwin && l < nl) { it -= nwin; ++l; }
    for (int m = g; m < m_total; m += kGroups) {
      const int half = m & 1;
      const int buf = m & 7;
      const uint32_t acc_par = (static_cast<uint32_t>(m) >> 3) & 1u;
      const int t = blockIdx.x + it * G;
      const Win w = decode_win(p, t);
      const int y0 = w.y0 + half * p.TH;
      const uint32_t t_addr = t_lane + buf * kNmma;
      // backward form: the gate operand (saved forward activations, constant during the backward) does not depend on the
      // accumulator - fetch it before waiting for the MMAs
      uint4 gq[2] = {make_uint4(0x3f803f80u, 0x3f803f80u, 0x3f803f80u, 0x3f803f80u), make_uint4(0x3f803f80u, 0x3f803f80u, 0x3f803f80u, 0x3f803f80u)};
      if (p.gate) {
        const int y = y0 + ty, x = w.x0 - x_off + tx;
        if (col_ok && y < p.H && x < p.W) {
          const uint4* gsrc = reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(p.gate) +
                                                             ((static_cast<size_t>(w.n) * p.H + y) * p.W + x) * p.gate_C + p.L[l].gate_coff);
          gq[0] = __ldg(gsrc);
          gq[1] = __ldg(gsrc + 1);
        }
      }
      mbar_wait(bar_acc_full(buf), acc_par);                // bounded: a protocol bug traps here instead of hanging
      tc_fence_after();
      uint32_t raw[2][3][8];
#pragma unroll
      for (int jj = 0; jj < 2; ++jj)
#pragma unroll
        for (int dx = 0; dx < 3; ++dx) tmem_ld8(t_addr + dx * kNpad + jj * 8, raw[jj][dx]);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_acc_empty(buf));       // the accumulator lives in registers now
      if constexpr (WR_T) {
        // one exchange per M tile (both chunks); the group's barriers below order the partner's reads before the next tile's writes
        if (row_pair) {
          row_edge_put(raw[0][0], raw[0][2], xdst, lane, row_left);
          row_edge_put(raw[1][0], raw[1][2], xdst + 64u, lane, row_left);
          named_bar_sync(5 + pair, 64);
        }
        row_edge_get(raw[0][0], raw[0][2], xsrc, lane);
        row_edge_get(raw[1][0], raw[1][2], xsrc + 64u, lane);
      }
#pragma unroll
      for (int jj = 0; jj < 2; ++jj) {
        float v[8];
        {
          const float4 b0 = *reinterpret_cast<const float4*>(bias_s + l * kNpad + jj * 8);
          const float4 b1 = *reinterpret_cast<const float4*>(bias_s + l * kNpad + jj * 8 + 4);
          v[0] = b0.x; v[1] = b0.y; v[2] = b0.z; v[3] = b0.w; v[4] = b1.x; v[5] = b1.y; v[6] = b1.z; v[7] = b1.w;
        }
        gather_add8(v, raw[jj][0], -1, lane);
        gather_add8(v, raw[jj][1], 0, lane);
        gather_add8(v, raw[jj][2], 1, lane);
        if (p.act) {
#pragma unroll
          for (int j = 0; j < 8; j += 2) {                  // LeakyReLU(0.2) = max(v, 0.2 v)
            const float2 s2 = __fmul2_rn(make_float2(v[j], v[j + 1]), make_float2(0.2f, 0.2f));
            v[j] = fmaxf(v[j], s2.x);
            v[j + 1] = fmaxf(v[j + 1], s2.y);
          }
        }
        if (p.gate) {                                       // LeakyReLU derivative of the forward activation (sign-preserving)
          const uint32_t gw[4] = {gq[jj].x, gq[jj].y, gq[jj].z, gq[jj].w};
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            v[2 * i] *= (bf16lo(gw[i]) > 0.f) ? 1.f : p.gate_neg;
            v[2 * i + 1] *= (bf16hi(gw[i]) > 0.f) ? 1.f : p.gate_neg;
          }
        }
        if (col_ok)
          st_shared_v4(srow_addr + jj * 16, pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
      }
      named_bar_sync(1 + g, 128);                           // the staged tile is complete
      __nv_bfloat16* tile_out = reinterpret_cast<__nv_bfloat16*>(p.buf) +
          ((static_cast<size_t>(w.n) * p.H + y0) * p.W + w.x0) * p.C + p.L[l].out_coff;
      const uint32_t lim = (static_cast<uint32_t>(max(0, min(p.H - y0, 0x7fff))) << 16) | static_cast<uint32_t>(min(p.W - w.x0, 0x7fff));
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        const bool ok = ((pc_yx[k] >> 16) < (lim >> 16)) && ((pc_yx[k] & 0xffffu) < (lim & 0xffffu));
        if (ok) {
          const uint4 val = ld_shared_v4(pc_s[k]);
          *reinterpret_cast<uint4*>(tile_out + pc_d[k]) = val;
        }
      }
      named_bar_sync(1 + g, 128);                           // every store of the tile has been issued (and the staging buffer is free)
      if (wj == 0 && lane == 0) {
        __threadfence();                                    // cumulative: the group's stores, ordered before this by the barrier
        red_release_gpu_add(p.flags + static_cast<size_t>(l) * p.num_tiles + t, 1u);
      }
      // next M tile of this group: m + 4 -> q + 2
      it += 2;
      while (it >= nwin && l < nl) { it -= nwin; ++l; }
    }
  }

  tc_fence_before();
  __syncthreads();
  timeline_end(p.timeline, p.launch_id);
  if (warp == 1) {
    __syncwarp();
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

size_t dense_smem_bytes(const DenseParams& p) {
  return 1024 + static_cast<size_t>(p.n_slots) * p.slot_bytes + static_cast<size_t>(kGroups) * p.stage_bytes + 2u * p.wbuf_bytes +
         kDenseMaxLayers * kNpad * 4 + 8 * (4 + 2 * p.n_slots + 2 * kAcc) + 32 + (p.whole_row ? kXchgBytes : 0);
}

int launch_dense_block(const DenseParams& p, const CUtensorMap& tmap, int num_sms, cudaStream_t stream) {
  const size_t smem = dense_smem_bytes(p);
  if (smem > static_cast<size_t>(kSmemLimit) || p.n_layers < 1 || p.n_layers > kDenseMaxLayers || p.n_slots < 2)
    return static_cast<int>(cudaErrorInvalidValue);
  if (p.whole_row && (p.SW != p.W || p.TW != p.W || (p.W != 32 && p.W != 64) || p.tiles_x != 1)) return static_cast<int>(cudaErrorInvalidValue);
  static bool configured[2][64] = {};
  auto kern = p.whole_row ? dense_block_kernel<1> : dense_block_kernel<0>;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return static_cast<int>(cudaErrorInvalidDevice);
  if (!configured[p.whole_row][dev]) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit);
    if (e != cudaSuccess) return static_cast<int>(e);
    configured[p.whole_row][dev] = true;
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(p.num_tiles < num_sms ? p.num_tiles : num_sms);
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

}  // namespace csr

// Weight gradient of the generator's convolutions on tcgen05 (sm_100a):  dW[co][ci][dy][dx] = sum_p g[p][co] * x[p+(dy,dx)][ci]
// (autograd of every nn.Conv2d of climsr/models/esrgan.py:22-27,72-87 and climsr/models/srcnn.py:9-11).
//
// It is a GEMM whose K dimension is the pixel index, so BOTH operands are "MN-major": a pixel's channels are contiguous
// (NHWC) and K strides over pixels - exactly the layout a TMA box of 64 channels x SW x rows lands in shared memory with
// the 128-byte swizzle (one pixel = one 128-byte line, 8 pixels = one swizzle atom).  No transposition pass is needed:
// the UMMA descriptors are built MN-major (instruction descriptor bits 15/16).
//
//   D_dx[ci][co] (fp32, TMEM, 128 lanes x n_cols columns per horizontal tap)  +=  X_shift(dx)[K=16 pixels][128 ci]^T * G[K][n_cols]
//
// One launch handles n_dy consecutive vertical taps (as many as fit the 512 TMEM columns): the x window is loaded once
// at row offset dy_off and every tap (dyi, dx) reads it at the flattened pixel offset dyi*SW + dx - PW (the halo trick of the forward kernel, transposed).  Columns
// of the g tile that belong to the neighbouring tiles are zeroed in shared memory so every pixel is counted once.
// Accumulators stay resident in TMEM over ALL tiles of the persistent CTA; one epilogue at the end stores the CTA's
// partial sums to its slice of a global fp32 buffer, reduced over CTAs by the scatter kernel.
#include "ptx.cuh"
#include "wgrad_tc.cuh"

namespace csr {

namespace {

__device__ __forceinline__ int fast_div_w(int t, unsigned long long magic) {
  return static_cast<int>((static_cast<unsigned long long>(static_cast<unsigned>(t)) * magic) >> 40);
}

// MMA with both operands MN-major.
__device__ __forceinline__ uint32_t make_idesc_bf16_mn(int m, int n) {
  return make_idesc_bf16(m, n) | (1u << 15) | (1u << 16);
}

}  // namespace

__global__ void __launch_bounds__(kWgradThreads, 1)
wgrad_tc_kernel(const WgradParams p, const __grid_constant__ CUtensorMap tx0, const __grid_constant__ CUtensorMap tx1,
                const __grid_constant__ CUtensorMap tg0, const __grid_constant__ CUtensorMap tg1) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const int S = p.n_stages;
  const uint32_t x_pitch = static_cast<uint32_t>(p.x_slack + p.x_box_bytes);       // slack + box, per 64-channel x box
  const uint32_t g_off = static_cast<uint32_t>(p.n_xbox) * x_pitch;               // g boxes follow the x boxes inside a stage
  const uint32_t bar_addr = smem_base + static_cast<uint32_t>(S) * p.stage_bytes;
  auto bar_full = [&](int s) { return bar_addr + 8u * s; };
  auto bar_ready = [&](int s) { return bar_addr + 8u * (S + s); };
  auto bar_empty = [&](int s) { return bar_addr + 8u * (2 * S + s); };
  const uint32_t bar_done = bar_addr + 8u * (3 * S);
  const uint32_t tmem_slot_addr = bar_done + 8u;
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem_gen + (tmem_slot_addr - smem_base));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  // what this CTA works on: the launch's single job (pixel tiles strided over the grid) or, in job mode, its own job
  int xc0a = p.xc0[0], xc0b = p.xc0[1], gc0a = p.gc0[0], gc0b = p.gc0[1], dy_off = p.dy_off, n_dy = p.n_dy;
  int t_first = blockIdx.x, t_step = gridDim.x;
  float* out_base = p.dacc + (p.atomic ? 0 : static_cast<size_t>(blockIdx.x) * p.part_stride);
  if (p.jobs_ci > 0) {
    const int job = blockIdx.x / p.splits;
    t_first = blockIdx.x - job * p.splits;
    t_step = p.splits;
    const int dyj = job % p.jobs_dy;
    const int oc = (job / p.jobs_dy) % p.jobs_co;
    const int cc = job / (p.jobs_dy * p.jobs_co);
    xc0a = p.x_coff + cc * 128; xc0b = xc0a + 64;
    gc0a = p.g_coff + oc * p.n_cols; gc0b = gc0a + 64;
    dy_off = dyj * p.per_dy - p.PH;
    n_dy = min(p.per_dy, p.KH - dyj * p.per_dy);
    out_base = p.dacc + static_cast<size_t>(job) * p.job_stride;
  }

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tx0);
    tma_prefetch_desc(&tg0);
    for (int s = 0; s < S; ++s) {
      mbar_init(bar_full(s), 1);
      mbar_init(bar_ready(s), 1);
      mbar_init(bar_empty(s), 1);
    }
    mbar_init(bar_done, 1);
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot_addr, p.tmem_cols);
    tmem_relinquish();
  }
  // zero the slack in front of every x box (read by negative tap shifts; multiplied by zeroed g columns, but must be finite)
  for (int s = 0; s < S; ++s)
    for (int b = 0; b < p.n_xbox; ++b) {
      uint4* z = reinterpret_cast<uint4*>(smem_gen + s * p.stage_bytes + b * x_pitch);
      for (int i = threadIdx.x; i < p.x_slack / 16; i += blockDim.x) z[i] = make_uint4(0, 0, 0, 0);
    }
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================== TMA producer =====================
    int stage = 0;
    uint32_t phase = 0;
    const uint32_t bytes = static_cast<uint32_t>(p.n_xbox * p.x_box_bytes + p.n_gbox * p.g_box_bytes);
    for (int t = t_first; t < p.num_tiles; t += t_step) {
      const int n = fast_div_w(t, p.magic_img);
      const int rem = t - n * p.tiles_per_img;
      const int tyi = fast_div_w(rem, p.magic_row);
      const int y0 = tyi * p.TH, x0 = (rem - tyi * p.tiles_x) * p.TW;
      mbar_wait(bar_empty(stage), phase ^ 1);
      if (elect_one()) {
        const uint32_t sb = smem_base + stage * p.stage_bytes;
        mbar_arrive_expect_tx(bar_full(stage), bytes);
        tma_load_4d(sb + p.x_slack, &tx0, bar_full(stage), xc0a, x0 - p.PW, y0 + dy_off, n);
        if (p.n_xbox > 1) tma_load_4d(sb + x_pitch + p.x_slack, &tx1, bar_full(stage), xc0b, x0 - p.PW, y0 + dy_off, n);
        tma_load_4d(sb + g_off, &tg0, bar_full(stage), gc0a, x0 - p.PW, y0, n);
        if (p.n_gbox > 1) tma_load_4d(sb + g_off + p.g_box_bytes, &tg1, bar_full(stage), gc0b, x0 - p.PW, y0, n);
      }
      __syncwarp();
      if (++stage == S) { stage = 0; phase ^= 1; }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    const uint32_t idesc = make_idesc_bf16_mn(128, p.n_cols);
    // MN-major, 128B swizzle: 64 channels (128 B) contiguous per pixel; LBO = byte distance to the next 64-channel box,
    // SBO = byte distance between groups of 8 pixels (8 x 128 B when pixels are consecutive lines).
    const uint32_t hi = (1024u >> 4) | (1u << 14) | (2u << 29);   // both operands: SBO 1024 B, version 1, SWIZZLE_128B
    const uint32_t a_lo_fixed = ((x_pitch >> 4) & 0x3FFFu) << 16;
    const uint32_t b_lo_fixed = ((static_cast<uint32_t>(p.g_box_bytes) >> 4) & 0x3FFFu) << 16;
    int stage = 0;
    uint32_t phase = 0;
    bool first = true;
    for (int t = t_first; t < p.num_tiles; t += t_step) {
      mbar_wait(bar_ready(stage), phase);
      tc_fence_after();
      const uint32_t sb = smem_base + stage * p.stage_bytes;
      if (elect_one()) {
        for (int dyi = 0; dyi < n_dy; ++dyi) {
          for (int dx = 0; dx < p.KW; ++dx) {
            const uint32_t d_tmem = tmem_base + (dyi * p.KW + dx) * p.n_cols;
            // flattened pixel shift of this tap inside the window: dyi rows + (dx - PW) pixels, 128 B each
            const uint32_t a0 = sb + p.x_slack + static_cast<uint32_t>((dyi * p.SW + dx - p.PW) * 128);
            for (int j = 0; j < 8; ++j) {
              const uint32_t a_lo = (((a0 + j * 2048u) >> 4) & 0x3FFFu) | a_lo_fixed;
              const uint32_t b_lo = (((sb + g_off + j * 2048u) >> 4) & 0x3FFFu) | b_lo_fixed;
              umma_bf16_split(d_tmem, a_lo, hi, b_lo, hi, idesc, (first && j == 0) ? 0u : 1u);
            }
          }
        }
        umma_commit(bar_empty(stage));
      }
      __syncwarp();
      first = false;
      if (++stage == S) { stage = 0; phase ^= 1; }
    }
    if (elect_one()) umma_commit(bar_done);
    __syncwarp();
  } else if (warp == 2) {
    // ===================== halo-column zeroing of the g tile =====================
    int stage = 0;
    uint32_t phase = 0;
    const int n_halo = p.SW - p.TW;                      // columns [0,PW) and [PW+TW, SW)
    for (int t = t_first; t < p.num_tiles; t += t_step) {
      mbar_wait(bar_full(stage), phase);
      if (n_halo > 0) {
        uint8_t* gb = smem_gen + stage * p.stage_bytes + g_off;
        const int per_box = p.TH * n_halo * 8;            // 16-byte pieces
        for (int i = lane; i < per_box * p.n_gbox; i += 32) {
          const int b = i / per_box;
          int r = i - b * per_box;
          const int piece = r & 7;
          r >>= 3;
          const int row = r / n_halo;
          const int hc = r - row * n_halo;
          const int col = hc < p.PW ? hc : p.TW + hc;     // hc >= PW  ->  PW + TW + (hc - PW)
          *reinterpret_cast<uint4*>(gb + b * p.g_box_bytes + (row * p.SW + col) * 128 + piece * 16) = make_uint4(0, 0, 0, 0);
        }
        fence_proxy_async_smem();
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_ready(stage));
      if (++stage == S) { stage = 0; phase ^= 1; }
    }
  } else if (warp >= 4) {
    // ===================== epilogue (once): TMEM -> red.add.f32 into the global accumulation buffer ==============
    const int q = warp & 3;
    const int ci = q * 32 + lane;
    if (t_first < p.num_tiles) {
      mbar_wait(bar_done, 0);
      tc_fence_after();
      // this CTA's partial sums go to its own slice of the accumulation buffer ([cta][dx][128][ld_n], plain stores);
      // the scatter kernel reduces over CTAs.  (fp32 atomics onto 49 K shared addresses from 148 CTAs were measured at
      // ~100 us per launch - 5x the GEMM itself.)
      // Default (p.atomic): all CTAs add into ONE copy with 16-byte vector reds - 148 x ~200 KB of partial stores plus a
      // reduce kernel reading them back cost ~10 us per launch and 1.5 ms per training step; the summation order over
      // CTAs is then not fixed (last-bit run-to-run differences, like cuDNN's atomics-based weight gradients).
      float* base = out_base;
      for (int tp = 0; tp < n_dy * p.KW; ++tp) {
        float* dst = base + (static_cast<size_t>(tp) * 128 + ci) * p.ld_n;
        for (int c = 0; c < p.n_cols; c += 8) {
          uint32_t r[8];
          tmem_ld8(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + tp * p.n_cols + c, r);
          tmem_ld_wait();
          if (p.atomic) {
            red_add_v4_f32(dst + c, __uint_as_float(r[0]), __uint_as_float(r[1]), __uint_as_float(r[2]), __uint_as_float(r[3]));
            red_add_v4_f32(dst + c + 4, __uint_as_float(r[4]), __uint_as_float(r[5]), __uint_as_float(r[6]), __uint_as_float(r[7]));
          } else {
            *reinterpret_cast<uint4*>(dst + c) = make_uint4(r[0], r[1], r[2], r[3]);
            *reinterpret_cast<uint4*>(dst + c + 4) = make_uint4(r[4], r[5], r[6], r[7]);
          }
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tc_fence_after();
    tmem_dealloc(tmem_base, p.tmem_cols);
  }
}

size_t wgrad_smem_bytes(const WgradParams& p) {
  return 1024 + static_cast<size_t>(p.n_stages) * p.stage_bytes + 8 * (3 * p.n_stages + 1) + 16;
}

int launch_wgrad_tc(const WgradParams& p, const CUtensorMap& tx0, const CUtensorMap& tx1, const CUtensorMap& tg0, const CUtensorMap& tg1,
                    int num_sms, cudaStream_t stream) {
  const size_t smem = wgrad_smem_bytes(p);
  if (smem > 232448) return static_cast<int>(cudaErrorInvalidValue);
  // the attribute is per device: one process may drive several GPUs
  static bool configured[64] = {};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return static_cast<int>(cudaErrorInvalidDevice);
  if (!configured[dev]) {
    cudaError_t e = cudaFuncSetAttribute(wgrad_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448);
    if (e != cudaSuccess) return static_cast<int>(e);
    configured[dev] = true;
  }
  const int grid = p.jobs_ci > 0 ? p.jobs_ci * p.jobs_co * p.jobs_dy * p.splits : p.n_parts;
  wgrad_tc_kernel<<<grid, kWgradThreads, smem, stream>>>(p, tx0, tx1, tg0, tg1);
  return static_cast<int>(cudaGetLastError());
}

}  // namespace csr

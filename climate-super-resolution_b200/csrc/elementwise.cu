// Layout / packing kernels around the conv hot path (all HBM-bound, vectorised, coalesced).
#include "elementwise.cuh"
#include <algorithm>
#include "ptx.cuh"

namespace csr {

// ---- weights: fp32 OIHW -> bf16 UMMA B tiles ------------------------------------------------------------
// Packed layout per launch part: [kblock = 64 input channels][dy][kstep within the k-block] blocks; one block is the
// B operand of one MMA: (KW*npad) x 16 K-major, rows ordered (dx, co) so the horizontal taps become output columns,
// stored as 8x16-byte core matrices [row group][k-chunk 2][row 8][elem 8] (LBO 128 B, SBO 256 B).  The last k-block may
// hold fewer than 4 k-steps.  Rows >= cout and channels >= cin are zero.  (cout, cin, kh, kw) describe the conv being
// EXECUTED; the source tensor is:
//   plain      : w[co][ci][dy][dx]                                   (the layer's OIHW weight)
//   fold != 0  : the layer is executed as a KH x 1 conv over an x-im2col input whose channel (dx*cin_src + c) holds
//                input channel c at horizontal offset dx - kw_src/2 (srcnn.conv1, 9x9 with 3 channels -> 9x1 with 27)
//   phase >= 0 : sub-pixel phase (a,b) = (phase>>1, phase&1) of "nearest-x2 upsample then 3x3 conv" (esrgan.py:94,97):
//                a 2x2 conv over the low-resolution input whose tap (ry, rx) is the SUM of the 3x3 taps that land on
//                the same source pixel: a=0: ry0<-{0}, ry1<-{1,2};  a=1: ry0<-{0,1}, ry1<-{2}  (same in x)
//   transposed : input-gradient conv of the layer: w_src[ci][co][KH-1-dy][KW-1-dx] with w_src of shape (cin, cout, kh, kw);
//                combined with phase >= 0 it is the input gradient of that sub-pixel phase (flipped 2x2 summed taps)
//   wscale     : constant folded into the packed weights (0.2 residual scaling on the gradient path)
__device__ __forceinline__ void phase_taps(int a, int r, int* lo, int* hi) {
  if (a == 0) { *lo = r == 0 ? 0 : 1; *hi = r == 0 ? 0 : 2; }
  else        { *lo = r == 0 ? 0 : 2; *hi = r == 0 ? 1 : 2; }
}

__device__ __forceinline__ void pack_weight_body(const float* __restrict__ w, __nv_bfloat16* __restrict__ dst, int cout, int cin, int kh,
                                                 int kw, int fold, int phase, int transposed, float wscale, int co_lo, int npad, int cin_pad,
                                                 int ci_lo, int ci_n, int src_ci_off, int src_cin, long first, long step) {
  // executed taps
  const int ekh = phase >= 0 ? 2 : kh;
  const int ekw = phase >= 0 ? 2 : (fold ? 1 : kw);
  const int ksteps = cin_pad >> 4;
  const int full_kb = ksteps >> 2, rem = ksteps & 3;
  const int groups = (ekw * npad) >> 3;
  const long total = static_cast<long>(ekh) * ksteps * ekw * npad * 16;
  for (long i = first; i < total; i += step) {
    const int e = i & 7;
    const int row = (i >> 3) & 7;
    const int kchunk = (i >> 6) & 1;
    long r = i >> 7;
    const int grp = r % groups;
    int blk = static_cast<int>(r / groups);               // block index in [kblock][dy][ks] order
    int kb, dy, ks;
    if (blk < full_kb * ekh * 4) {
      kb = blk / (ekh * 4);
      blk -= kb * ekh * 4;
      dy = blk >> 2;
      ks = blk & 3;
    } else {
      blk -= full_kb * ekh * 4;
      kb = full_kb;
      dy = blk / rem;
      ks = blk - dy * rem;
    }
    const int rr = grp * 8 + row;
    int dx = rr / npad;
    const int co = co_lo + (rr - dx * npad);
    int ci = (kb * 4 + ks) * 16 + kchunk * 8 + e;
    // block jobs fill only executed input channels [ci_lo, ci_lo + ci_n) (another job of the same layer fills the rest)
    if (ci_n > 0) {
      const int cb = transposed ? ci : co;                // output-channel blocks for forward (non-transposed) layers
      if (cb < ci_lo || cb >= ci_lo + ci_n) continue;
    }
    float v = 0.f;
    const int cin_eff = fold ? cin * kw : cin;
    if (co < cout && ci < cin_eff) {
      if (fold) {
        dx = ci / cin;
        ci -= dx * cin;
      }
      // source indices: the forward layer's OIHW tensor is (cout, cin, kh, kw), or (cin, cout, kh, kw) when transposed
      // (block jobs: source output channel = ci - ci_lo, source input channel = co + src_ci_off of a (ci_n, src_cin, kh, kw) tensor)
      // forward block jobs: source output channel = co - ci_lo, source input channel = ci + src_ci_off
      const int s_o = transposed ? ci - ci_lo : (ci_n > 0 ? co - ci_lo : co);
      const int s_i = transposed ? co + src_ci_off : (ci_n > 0 ? ci + src_ci_off : ci);
      const int s_in = transposed ? (src_cin ? src_cin : cout) : (ci_n > 0 ? src_cin : cin);   // channels-per-output-filter of the source tensor
      const int sdy = transposed ? ekh - 1 - dy : dy, sdx = transposed ? ekw - 1 - dx : dx;
      if (phase >= 0) {
        int y0, y1, x0, x1;
        phase_taps(phase >> 1, sdy, &y0, &y1);
        phase_taps(phase & 1, sdx, &x0, &x1);
        for (int yy = y0; yy <= y1; ++yy)
          for (int xx = x0; xx <= x1; ++xx) v += w[((static_cast<long>(s_o) * s_in + s_i) * kh + yy) * kw + xx];
      } else {
        v = w[((static_cast<long>(s_o) * s_in + s_i) * kh + sdy) * kw + sdx];
      }
      v *= wscale;
    }
    dst[i] = __float2bfloat16_rn(v);
  }
}

// All layers of the generator in ONE launch (training repacks every optimizer step: ~360 layer parts): blockIdx.y = job.
__global__ void pack_jobs_kernel(const PackJob* __restrict__ jobs) {
  const PackJob j = jobs[blockIdx.y];
  pack_weight_body(j.w, reinterpret_cast<__nv_bfloat16*>(j.dst), j.cout, j.cin, j.kh, j.kw, j.fold, j.phase, j.transposed, j.wscale, j.co_lo,
                   j.npad, j.cin_pad, j.ci_lo, j.ci_n, j.src_ci_off, j.src_cin, blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x,
                   static_cast<long>(gridDim.x) * blockDim.x);
  if (blockIdx.x == 0 && threadIdx.x < j.npad && j.bdst) {
    const int co = j.co_lo + static_cast<int>(threadIdx.x);
    if (j.ci_n > 0 && !j.transposed) {                    // forward block job: only its own bias segment
      if (co >= j.ci_lo && co < j.ci_lo + j.ci_n) j.bdst[threadIdx.x] = j.b ? j.b[co - j.ci_lo] : 0.f;
    } else {
      j.bdst[threadIdx.x] = (j.b && co < j.cout) ? j.b[co] : 0.f;
    }
  }
}

// ---- activations -----------------------------------------------------------------------------------------
// fp32 NCHW (n,c,h,w) -> bf16 NHWC (n,h,w,dst_c): channels [0,c) converted, [c,zero_to) zeroed (zero_to <= 16,
// multiple of 8).  One thread per pixel; reads are coalesced across pixels for each channel plane.
__global__ void nchw_to_nhwc_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, long npix_per_img,
                                    long total_pix, int c, int dst_c, int zero_to) {
  for (long p = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; p < total_pix; p += static_cast<long>(gridDim.x) * blockDim.x) {
    const long n = p / npix_per_img;
    const long r = p - n * npix_per_img;
    float v[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = (i < c) ? src[(n * c + i) * npix_per_img + r] : 0.f;
    uint4* o = reinterpret_cast<uint4*>(dst + p * dst_c);
    uint4 a;
    a.x = pack_bf16x2(v[0], v[1]); a.y = pack_bf16x2(v[2], v[3]); a.z = pack_bf16x2(v[4], v[5]); a.w = pack_bf16x2(v[6], v[7]);
    o[0] = a;
    if (zero_to > 8) {
      a.x = pack_bf16x2(v[8], v[9]); a.y = pack_bf16x2(v[10], v[11]); a.z = pack_bf16x2(v[12], v[13]); a.w = pack_bf16x2(v[14], v[15]);
      o[1] = a;
    }
  }
}

// ---- hi/lo bf16 activations (perceptual loss, CSR_OUT_BF16_SPLIT) ------------------------------------------------
// fp32 NCHW (n,c,h,w), c <= 3 -> bf16 NHWC (n,h,w,dst_c): channels [hi_0..hi_{c-1}, lo_0..lo_{c-1}, 0...], hi = bf16(x),
// lo = bf16(x - hi).  The input needs the pair too: one bf16 ulp near 1 (0.0039) is larger than the differences between
// hr and sr the loss has to resolve.
__global__ void nchw_to_nhwc_split_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, long npix_per_img,
                                          long total_pix, int c, int dst_c) {
  for (long p = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; p < total_pix; p += static_cast<long>(gridDim.x) * blockDim.x) {
    const long n = p / npix_per_img;
    const long r = p - n * npix_per_img;
    float f[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      if (i < c) {
        const float x = src[(n * c + i) * npix_per_img + r];
        const float hi = __bfloat162float(__float2bfloat16_rn(x));
        f[i] = hi;                                        // exact bf16 values: pack_bf16x2 below does not round them again
        f[c + i] = __bfloat162float(__float2bfloat16_rn(x - hi));
      }
    }
    uint4* o = reinterpret_cast<uint4*>(dst + p * dst_c);
    o[0] = make_uint4(pack_bf16x2(f[0], f[1]), pack_bf16x2(f[2], f[3]), pack_bf16x2(f[4], f[5]), pack_bf16x2(f[6], f[7]));
    for (int k = 1; k < (dst_c >> 3); ++k) o[k] = make_uint4(0u, 0u, 0u, 0u);
  }
}

// nn.MaxPool2d(2) (ceil_mode=False) over hi/lo pairs: src (n,h,w,2c) -> dst (n,h/2,w/2,2c).  One thread per (output pixel,
// 8 channels): 16-byte loads of the hi and lo vectors of the four window pixels; hi + lo is exact in fp32, so the max of
// the sums re-splits into the winning pixel's own pair.  Window order and the NaN rule are those of F.max_pool2d
// ((v > m) || isnan(v), starting from -inf): the first maximum wins, a NaN anywhere in the window is the result.
__global__ void maxpool2x2_split_kernel(const __nv_bfloat16* __restrict__ src, __nv_bfloat16* __restrict__ dst, int h, int w, int c,
                                        long total) {
  const int ho = h >> 1, wo = w >> 1, g8 = c >> 3;
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < total; i += static_cast<long>(gridDim.x) * blockDim.x) {
    const int g = static_cast<int>(i % g8);
    long q = i / g8;
    const int x = static_cast<int>(q % wo);
    q /= wo;
    const int y = static_cast<int>(q % ho);
    const long n = q / ho;
    float m[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) m[j] = -INFINITY;
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const long pix = (n * h + 2 * y + (t >> 1)) * w + 2 * x + (t & 1);
      const __nv_bfloat16* base = src + pix * 2 * c + g * 8;
      const uint4 hv = __ldg(reinterpret_cast<const uint4*>(base));
      const uint4 lv = __ldg(reinterpret_cast<const uint4*>(base + c));
      const uint32_t hw[4] = {hv.x, hv.y, hv.z, hv.w}, lw[4] = {lv.x, lv.y, lv.z, lv.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float v0 = bf16lo(hw[k]) + bf16lo(lw[k]), v1 = bf16hi(hw[k]) + bf16hi(lw[k]);
        if (v0 > m[2 * k] || isnan(v0)) m[2 * k] = v0;
        if (v1 > m[2 * k + 1] || isnan(v1)) m[2 * k + 1] = v1;
      }
    }
    uint32_t hi[4], lo[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) split_bf16x2(m[2 * k], m[2 * k + 1], &hi[k], &lo[k]);
    __nv_bfloat16* o = dst + ((n * ho + y) * wo + x) * 2 * c + g * 8;
    *reinterpret_cast<uint4*>(o) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    *reinterpret_cast<uint4*>(o + c) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
  }
}

// SRCNN input as an x-im2col buffer: torch.cat([out, elev, mask], 1) (esrgan.py:100) followed by the horizontal half of
// srcnn.conv1's 9x9 window.  For pixel (n,y,x) channel dx*3 + c (dx = 0..8, c = 0: conv_last output, 1: elev, 2: mask)
// holds source c at (y, x+dx-4), zero outside the image (the conv's zero padding); channels 27..31 are zero.  The 9x9
// conv over 3 channels then runs as a 9x1 conv over 27(32) channels: 18 instead of 81 MMAs per tile.
__global__ void pack_srcnn_in_kernel(const float* __restrict__ t, const float* __restrict__ elev, const float* __restrict__ mask,
                                     __nv_bfloat16* __restrict__ dst, int W, long total_pix, int dst_c) {
  for (long p = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; p < total_pix; p += static_cast<long>(gridDim.x) * blockDim.x) {
    const int x = static_cast<int>(p % W);
    float v[32];
#pragma unroll
    for (int dx = 0; dx < 9; ++dx) {
      const int xs = x + dx - 4;
      const bool in = xs >= 0 && xs < W;
      const long q = p + dx - 4;
      v[dx * 3 + 0] = in ? t[q] : 0.f;
      v[dx * 3 + 1] = in ? elev[q] : 0.f;
      v[dx * 3 + 2] = in ? mask[q] : 0.f;
    }
#pragma unroll
    for (int i = 27; i < 32; ++i) v[i] = 0.f;
    uint4* o = reinterpret_cast<uint4*>(dst + p * dst_c);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      uint4 a;
      a.x = pack_bf16x2(v[8 * k + 0], v[8 * k + 1]);
      a.y = pack_bf16x2(v[8 * k + 2], v[8 * k + 3]);
      a.z = pack_bf16x2(v[8 * k + 4], v[8 * k + 5]);
      a.w = pack_bf16x2(v[8 * k + 6], v[8 * k + 7]);
      o[k] = a;
    }
  }
}

__global__ void nhwc_to_nchw_kernel(const __nv_bfloat16* __restrict__ src, float* __restrict__ dst, long npix_per_img, long total,
                                    int c, int src_c, int src_coff) {
  // one thread per output element, pixel-fastest so fp32 writes coalesce
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < total; i += static_cast<long>(gridDim.x) * blockDim.x) {
    const long r = i % npix_per_img;
    const long nc = i / npix_per_img;
    const long n = nc / c;
    const int ch = nc - n * c;
    dst[i] = __bfloat162float(src[(n * npix_per_img + r) * src_c + src_coff + ch]);
  }
}

// ---- weight-gradient post-processing ---------------------------------------------------------------------
// dacc: fp32 [KH_e][KW_e][128][ld_n] sums (wgrad_tc_kernel's per-CTA partials after wgrad_reduce_kernel; executed taps
// KH_e x KW_e, rows = executed input channel - ci0, columns = output channel + col0).  Adds scale * dacc into the layer's
// OIHW gradient:
//   plain : dw[co][ci][dy][dx]                          += dacc[dy][dx][ci - ci0][col0 + co]
//   fold  : dw[co][c][dy][dx]  (executed channel dx*cin+c, KW_e = 1)  += dacc[dy][0][dx*cin + c - ci0][col0 + co]
//   phase : executed 2x2 taps (ry, rx) of sub-pixel phase (a,b) feed every 3x3 tap they were summed from
// part 0 += parts 1..n_parts-1 (fixed order -> deterministic), fully coalesced
__global__ void wgrad_reduce_kernel(float* __restrict__ dacc, long part_stride, int n_parts, long n4) {
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < n4; i += static_cast<long>(gridDim.x) * blockDim.x) {
    float4 a = reinterpret_cast<const float4*>(dacc)[i];
    for (int q = 1; q < n_parts; ++q) {
      const float4 b = reinterpret_cast<const float4*>(dacc + q * part_stride)[i];
      a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
    }
    reinterpret_cast<float4*>(dacc)[i] = a;
  }
}

__global__ void wgrad_scatter_kernel(const float* __restrict__ dacc, int ld_n, float* __restrict__ dw, int cout,
                                     int cin, int kh, int kw, int fold, int phase, int ci0, int ci_n, int col0, float scale, int taps_t) {
  const int ekh = phase >= 0 ? 2 : kh;
  const int ekw = phase >= 0 ? 2 : (fold ? 1 : kw);
  const long total = static_cast<long>(ekh) * ekw * ci_n * cout;
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < total; i += static_cast<long>(gridDim.x) * blockDim.x) {
    const int co = i % cout;
    long r = i / cout;
    const int cl = r % ci_n;                               // executed input channel - ci0
    r /= ci_n;
    const int dx = r % ekw, dy = r / ekw;
    const float v = scale * dacc[((static_cast<long>(dy) * ekw + dx) * 128 + cl) * ld_n + col0 + co];
    const int ce = ci0 + cl;                               // executed input channel
    if (taps_t) {
      // 1x1 GEMM against an output-gradient im2col: column co is tap co of a (1, cin, KH, KW) weight -> dw[ci][tap]
      if (ce < cin) dw[static_cast<long>(ce) * cout + co] += v;
      continue;
    }
    if (phase >= 0) {
      if (ce >= cin) continue;
      int y0, y1, x0, x1;
      phase_taps(phase >> 1, dy, &y0, &y1);
      phase_taps(phase & 1, dx, &x0, &x1);
      for (int yy = y0; yy <= y1; ++yy)
        for (int xx = x0; xx <= x1; ++xx) atomicAdd(&dw[((static_cast<long>(co) * cin + ce) * kh + yy) * kw + xx], v);
    } else if (fold) {
      if (ce >= cin * kw) continue;
      const int fx = ce / cin, c = ce - fx * cin;
      dw[((static_cast<long>(co) * cin + c) * kh + dy) * kw + fx] += v;
    } else {
      if (ce >= cin) continue;
      dw[((static_cast<long>(co) * cin + ce) * kh + dy) * kw + dx] += v;
    }
  }
}

// Job-mode scatter (wgrad_tc job mode): dw[co][ci][dy][dx] += scale * dacc[job(ci/128, co/n_cols, dy/per_dy)][(dy%per_dy)*kw + dx][ci%128][co%n_cols]
__global__ void wgrad_scatter_jobs_kernel(const float* __restrict__ dacc, float* __restrict__ dw, int cout, int cin, int kh, int kw, int n_cols,
                                          int jobs_co, int jobs_dy, int per_dy, long job_stride, float scale) {
  const long total = static_cast<long>(cout) * cin * kh * kw;
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < total; i += static_cast<long>(gridDim.x) * blockDim.x) {
    const int dx = static_cast<int>(i % kw);
    long r = i / kw;
    const int dy = static_cast<int>(r % kh); r /= kh;
    const int ci = static_cast<int>(r % cin);
    const int co = static_cast<int>(r / cin);
    const long job = (static_cast<long>(ci >> 7) * jobs_co + co / n_cols) * jobs_dy + dy / per_dy;
    dw[i] += scale * dacc[job * job_stride + (static_cast<long>((dy % per_dy) * kw + dx) * 128 + (ci & 127)) * n_cols + co % n_cols];
  }
}

// db[co] += scale * sum over pixels of g[p][coff + co]   (bf16 NHWC, pitch C).  One block per pixel range, fp32 atomics.
// Channel co goes to segment co / seg_ch (its own bias-gradient vector): one pass serves the four narrow convs of a
// dense block whose output gradients sit side by side in the gradient concat buffer.
struct BiasSegs {
  float* db[4];
};
__global__ void bias_grad_kernel(const __nv_bfloat16* __restrict__ g, long npix, int C, int coff, int cout, float scale, BiasSegs segs,
                                 int seg_ch) {
  extern __shared__ float red[];                           // [blockDim.x / cout_pad rows][cout_pad]
  coff += blockIdx.y * cout;                               // gridDim.y > 1: consecutive `cout`-channel chunks of one wide layer (nseg == 1)
  const int cpad = (cout + 7) & ~7;
  const int lanes_per_pix = cpad >> 3;                     // one thread loads 8 channels (16 B)
  const int pix_per_iter = blockDim.x / lanes_per_pix;
  const int sub = threadIdx.x % lanes_per_pix, prow = threadIdx.x / lanes_per_pix;
  float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  if (prow < pix_per_iter) {
    const long stride = static_cast<long>(gridDim.x) * pix_per_iter;
    long pix = blockIdx.x * static_cast<long>(pix_per_iter) + prow;
    for (; pix + 7 * stride < npix; pix += 8 * stride) {   // eight independent 16-byte loads in flight per thread
      uint4 v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) v[u] = *reinterpret_cast<const uint4*>(g + (pix + u * stride) * C + coff + sub * 8);
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const uint32_t w[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          acc[2 * k] += bf16lo(w[k]);
          acc[2 * k + 1] += bf16hi(w[k]);
        }
      }
    }
    for (; pix < npix; pix += stride) {
      const uint4 v = *reinterpret_cast<const uint4*>(g + pix * C + coff + sub * 8);
      const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        acc[2 * k] += bf16lo(w[k]);
        acc[2 * k + 1] += bf16hi(w[k]);
      }
    }
  }
  for (int k = 0; k < 8; ++k) red[threadIdx.x * 8 + k] = acc[k];
  __syncthreads();
  if (threadIdx.x < cout) {
    const int s2 = threadIdx.x >> 3, k = threadIdx.x & 7;
    float t = 0.f;
    for (int r = 0; r < pix_per_iter; ++r) t += red[(r * lanes_per_pix + s2) * 8 + k];
    const int sg = threadIdx.x / seg_ch;
    atomicAdd(&segs.db[sg][blockIdx.y * cout + threadIdx.x - sg * seg_ch], scale * t);
  }
}

// db[0] += scale * sum(g) for an fp32 planar single-channel gradient
__global__ void bias_grad_planar_kernel(const float* __restrict__ g, long n, float scale, float* __restrict__ db) {
  float acc = 0.f;
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < n; i += static_cast<long>(gridDim.x) * blockDim.x) acc += g[i];
  for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  __shared__ float part[32];
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    float t = threadIdx.x < (blockDim.x >> 5) ? part[threadIdx.x] : 0.f;
    for (int o = 16; o; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    if (threadIdx.x == 0) atomicAdd(db, scale * t);
  }
}

// dst[p][0:64] = scale * src[p][0:64]   (bf16 NHWC, pitches src_C / dst_C): the 0.2 of `out*0.2 + x` (esrgan.py:54)
// on the gradient path.  One thread per 8 channels.
__global__ void scale_copy64_kernel(const __nv_bfloat16* __restrict__ src, int src_C, __nv_bfloat16* __restrict__ dst, int dst_C, long npix,
                                    float scale) {
  const long total = npix * 8;
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < total; i += static_cast<long>(gridDim.x) * blockDim.x) {
    const long pix = i >> 3;
    const int c8 = static_cast<int>(i & 7);
    const uint4 v = *reinterpret_cast<const uint4*>(src + pix * src_C + c8 * 8);
    uint4 o;
    o.x = pack_bf16x2(bf16lo(v.x) * scale, bf16hi(v.x) * scale);
    o.y = pack_bf16x2(bf16lo(v.y) * scale, bf16hi(v.y) * scale);
    o.z = pack_bf16x2(bf16lo(v.z) * scale, bf16hi(v.z) * scale);
    o.w = pack_bf16x2(bf16lo(v.w) * scale, bf16hi(v.w) * scale);
    *reinterpret_cast<uint4*>(dst + pix * dst_C + c8 * 8) = o;
  }
}

// Output-gradient im2col for single-output-channel convs (conv_last 64->1 3x3, srcnn.conv3 32->1 5x5): channel t = dy*KW+dx
// of pixel q holds g at pixel q - (dy-PH, dx-PW) (zero outside the image).  With it both gradients of such a layer are
// 1x1 GEMMs: d/dx[q][ci] = sum_t gcol[q][t] w[ci][t] and dW[ci][t] = sum_q x[q][ci] gcol[q][t] - K (or N) = taps instead
// of one tiny MMA per tap.  src: fp32 planar (N,1,H,W) when src_C == 0, else bf16 NHWC channel 0 of pitch src_C.
template <int KH, int KW, int DST_C>
__global__ void gcol_pack_kernel(const void* __restrict__ src, int src_C, __nv_bfloat16* __restrict__ dst, int H, int W, long total_pix) {
  constexpr int PH = KH / 2, PW = KW / 2;
  const long hw = static_cast<long>(H) * W;
  for (long q = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; q < total_pix; q += static_cast<long>(gridDim.x) * blockDim.x) {
    const long n = q / hw;
    const int r = static_cast<int>(q - n * hw);
    const int y = r / W, x = r - y * W;
    float v[DST_C];
#pragma unroll
    for (int t = 0; t < DST_C; ++t) v[t] = 0.f;
#pragma unroll
    for (int dy = 0; dy < KH; ++dy)
#pragma unroll
      for (int dx = 0; dx < KW; ++dx) {
        const int ys = y - (dy - PH), xs = x - (dx - PW);
        if (ys >= 0 && ys < H && xs >= 0 && xs < W) {
          const long p = n * hw + static_cast<long>(ys) * W + xs;
          v[dy * KW + dx] = src_C ? __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(src)[p * src_C])
                                  : __ldg(reinterpret_cast<const float*>(src) + p);
        }
      }
    uint4* o = reinterpret_cast<uint4*>(dst + q * DST_C);     // one pixel = DST_C/8 16-byte stores
#pragma unroll
    for (int k = 0; k < DST_C / 8; ++k) {
      uint4 a;
      a.x = pack_bf16x2(v[8 * k + 0], v[8 * k + 1]);
      a.y = pack_bf16x2(v[8 * k + 2], v[8 * k + 3]);
      a.z = pack_bf16x2(v[8 * k + 4], v[8 * k + 5]);
      a.w = pack_bf16x2(v[8 * k + 6], v[8 * k + 7]);
      o[k] = a;
    }
  }
}

static inline int grid_for(long total, int block, int cap = 148 * 16) {
  long g = (total + block - 1) / block;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return static_cast<int>(g);
}

cudaError_t launch_nchw_to_nhwc(const float* src, void* dst, int n, int c, int h, int w, int dst_c, int zero_to, cudaStream_t s) {
  const long per = static_cast<long>(h) * w, total = per * n;
  nchw_to_nhwc_kernel<<<grid_for(total, 256), 256, 0, s>>>(src, reinterpret_cast<__nv_bfloat16*>(dst), per, total, c, dst_c, zero_to);
  return cudaGetLastError();
}
cudaError_t launch_nchw_to_nhwc_split(const float* src, void* dst, int n, int c, int h, int w, int dst_c, cudaStream_t s) {
  const long per = static_cast<long>(h) * w, total = per * n;
  nchw_to_nhwc_split_kernel<<<grid_for(total, 256), 256, 0, s>>>(src, reinterpret_cast<__nv_bfloat16*>(dst), per, total, c, dst_c);
  return cudaGetLastError();
}
cudaError_t launch_maxpool2x2_split(const void* src, void* dst, int n, int h, int w, int c, cudaStream_t s) {
  const long total = static_cast<long>(n) * (h >> 1) * (w >> 1) * (c >> 3);
  maxpool2x2_split_kernel<<<grid_for(total, 256), 256, 0, s>>>(reinterpret_cast<const __nv_bfloat16*>(src), reinterpret_cast<__nv_bfloat16*>(dst),
                                                               h, w, c, total);
  return cudaGetLastError();
}
cudaError_t launch_pack_srcnn_in(const float* t, const float* elev, const float* mask, void* dst, int W, long total_pix, int dst_c,
                                 cudaStream_t s) {
  pack_srcnn_in_kernel<<<grid_for(total_pix, 256, 148 * 32), 256, 0, s>>>(t, elev, mask, reinterpret_cast<__nv_bfloat16*>(dst), W, total_pix,
                                                                         dst_c);
  return cudaGetLastError();
}
cudaError_t launch_nhwc_to_nchw(const void* src, float* dst, int n, int c, int h, int w, int src_c, int src_coff, cudaStream_t s) {
  const long per = static_cast<long>(h) * w, total = per * n * c;
  nhwc_to_nchw_kernel<<<grid_for(total, 256), 256, 0, s>>>(reinterpret_cast<const __nv_bfloat16*>(src), dst, per, total, c, src_c,
                                                           src_coff);
  return cudaGetLastError();
}

cudaError_t launch_wgrad_reduce(float* dacc, long part_stride, int n_parts, long nfloats, cudaStream_t s) {
  if (n_parts <= 1) return cudaSuccess;
  wgrad_reduce_kernel<<<grid_for(nfloats / 4, 256, 148 * 8), 256, 0, s>>>(dacc, part_stride, n_parts, nfloats / 4);
  return cudaGetLastError();
}
cudaError_t launch_wgrad_scatter(const float* dacc, int ld_n, float* dw, int cout, int cin, int kh, int kw, int fold,
                                 int phase, int ci0, int ci_n, int col0, float scale, int taps_t, cudaStream_t s) {
  const int ekh = phase >= 0 ? 2 : kh, ekw = phase >= 0 ? 2 : (fold ? 1 : kw);
  const long total = static_cast<long>(ekh) * ekw * ci_n * cout;
  wgrad_scatter_kernel<<<grid_for(total, 256), 256, 0, s>>>(dacc, ld_n, dw, cout, cin, kh, kw, fold, phase, ci0, ci_n, col0, scale, taps_t);
  return cudaGetLastError();
}
cudaError_t launch_wgrad_scatter_jobs(const float* dacc, float* dw, int cout, int cin, int kh, int kw, int n_cols, int jobs_co, int jobs_dy,
                                      int per_dy, long job_stride, float scale, cudaStream_t s) {
  const long total = static_cast<long>(cout) * cin * kh * kw;
  wgrad_scatter_jobs_kernel<<<grid_for(total, 256), 256, 0, s>>>(dacc, dw, cout, cin, kh, kw, n_cols, jobs_co, jobs_dy, per_dy, job_stride, scale);
  return cudaGetLastError();
}
cudaError_t launch_bias_grad(const void* g, long npix, int C, int coff, int cout, float scale, float* const* db, int nseg, cudaStream_t s) {
  BiasSegs segs;
  for (int i = 0; i < 4; ++i) segs.db[i] = db[i < nseg ? i : 0];
  bias_grad_kernel<<<148 * 4, 256, 256 * 8 * sizeof(float), s>>>(reinterpret_cast<const __nv_bfloat16*>(g), npix, C, coff, cout, scale, segs,
                                                                 cout / nseg);
  return cudaGetLastError();
}
// cout = chunks * 128 channels of one layer in one launch
cudaError_t launch_bias_grad_wide(const void* g, long npix, int C, int coff, int chunks, float scale, float* db, cudaStream_t s) {
  BiasSegs segs;
  for (int i = 0; i < 4; ++i) segs.db[i] = db;
  const int gx = 148 * 4 / chunks > 16 ? 148 * 4 / chunks : 16;
  bias_grad_kernel<<<dim3(gx, chunks), 256, 256 * 8 * sizeof(float), s>>>(reinterpret_cast<const __nv_bfloat16*>(g), npix, C, coff, 128, scale, segs, 128);
  return cudaGetLastError();
}
// conv_last finished from its nine fp32 tap planes (conv_tc.cu FUSE_T = 2: tap[t](y, x) = sum_c W[0][c][t] * HRconv(y, x)[c]):
//   out(n, y, x) = bias + sum_{ky,kx} tap[ky*3 + kx](n, y + ky - 1, x + kx - 1)      (zero outside the image = the conv padding)
__global__ void tap_sum_kernel(const float* __restrict__ taps, long plane, const float* __restrict__ bias, float* __restrict__ out, int H, int W,
                               long total) {
  const float b = bias ? bias[0] : 0.f;
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < total; i += static_cast<long>(gridDim.x) * blockDim.x) {
    const int x = static_cast<int>(i % W);
    const int y = static_cast<int>((i / W) % H);
    float acc = b;
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
      const int yy = y + ky - 1;
      if (yy < 0 || yy >= H) continue;
#pragma unroll
      for (int kx = 0; kx < 3; ++kx) {
        const int xx = x + kx - 1;
        if (xx >= 0 && xx < W) acc += taps[static_cast<long>(ky * 3 + kx) * plane + i + (ky - 1) * W + (kx - 1)];
      }
    }
    out[i] = acc;
  }
}
// tap_sum_kernel + pack_srcnn_in_kernel in one pass (inference, 32-channel im2col pitch): a block takes 256 pixels of one image row,
// finishes conv_last for them and their 4-pixel horizontal halo from the nine tap planes, builds the 27 (32) im2col channels of every
// pixel in shared memory and writes them out as whole lines (consecutive threads = consecutive 16-byte pieces).  The fp32 conv_last
// plane never reaches memory and the 64 B / pixel of output leave coalesced (the per-pixel strided stores of the two-kernel form ran
// at 3.4 TB/s).
__global__ void __launch_bounds__(256) tap_pack_kernel(const float* __restrict__ taps, long plane, const float* __restrict__ bias,
                                                       const float* __restrict__ elev, const float* __restrict__ mask,
                                                       __nv_bfloat16* __restrict__ dst, int H, int W, int segs) {
  __shared__ float ts[264], es[264], ms[264];
  __shared__ uint4 outs[256 * 4];
  const int seg = blockIdx.x % segs;
  const long row = blockIdx.x / segs;                     // n * H + y
  const int y = static_cast<int>(row % H);
  const int x0 = seg * 256;
  const long rowbase = row * W;
  const float b = bias ? bias[0] : 0.f;
  for (int i = threadIdx.x; i < 264; i += 256) {
    const int xx = x0 - 4 + i;
    float t = 0.f, e = 0.f, m = 0.f;
    if (xx >= 0 && xx < W) {
      t = b;
#pragma unroll
      for (int ky = 0; ky < 3; ++ky) {
        const int yy = y + ky - 1;
        if (yy < 0 || yy >= H) continue;
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
          const int xs = xx + kx - 1;
          if (xs >= 0 && xs < W) t += taps[static_cast<long>(ky * 3 + kx) * plane + rowbase + (ky - 1) * W + xs];
        }
      }
      e = elev[rowbase + xx];
      m = mask[rowbase + xx];
    }
    ts[i] = t; es[i] = e; ms[i] = m;
  }
  __syncthreads();
  const int n_here = min(256, W - x0);
  if (static_cast<int>(threadIdx.x) < n_here) {
    float v[32];
#pragma unroll
    for (int dx = 0; dx < 9; ++dx) {                      // channel dx*3 + c: pixel x + dx - 4 of (conv_last output, elevation, mask)
      v[dx * 3 + 0] = ts[threadIdx.x + dx];
      v[dx * 3 + 1] = es[threadIdx.x + dx];
      v[dx * 3 + 2] = ms[threadIdx.x + dx];
    }
#pragma unroll
    for (int i = 27; i < 32; ++i) v[i] = 0.f;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      uint4 a;
      a.x = pack_bf16x2(v[8 * k + 0], v[8 * k + 1]);
      a.y = pack_bf16x2(v[8 * k + 2], v[8 * k + 3]);
      a.z = pack_bf16x2(v[8 * k + 4], v[8 * k + 5]);
      a.w = pack_bf16x2(v[8 * k + 6], v[8 * k + 7]);
      outs[((threadIdx.x * 4 + k) & ~3) + ((k + (threadIdx.x >> 1)) & 3)] = a;   // rotate the four pieces of a pixel: fewer bank conflicts
    }
  }
  __syncthreads();
  uint4* o = reinterpret_cast<uint4*>(dst + (rowbase + x0) * 32);
  for (int j = threadIdx.x; j < n_here * 4; j += 256) {
    const int px = j >> 2, k = j & 3;
    o[j] = outs[px * 4 + ((k + (px >> 1)) & 3)];
  }
}
cudaError_t launch_tap_pack(const float* taps, long plane, const float* bias, const float* elev, const float* mask, void* dst, int N, int H, int W,
                            cudaStream_t s) {
  const int segs = (W + 255) / 256;
  tap_pack_kernel<<<static_cast<unsigned>(static_cast<long>(N) * H * segs), 256, 0, s>>>(taps, plane, bias, elev, mask,
                                                                                      reinterpret_cast<__nv_bfloat16*>(dst), H, W, segs);
  return cudaGetLastError();
}
cudaError_t launch_tap_sum(const float* taps, long plane, const float* bias, float* out, int H, int W, long total, cudaStream_t s) {
  tap_sum_kernel<<<grid_for(total, 256, 148 * 16), 256, 0, s>>>(taps, plane, bias, out, H, W, total);
  return cudaGetLastError();
}
cudaError_t launch_bias_grad_planar(const float* g, long n, float scale, float* db, cudaStream_t s) {
  bias_grad_planar_kernel<<<148 * 2, 256, 0, s>>>(g, n, scale, db);
  return cudaGetLastError();
}

cudaError_t launch_scale_copy64(const void* src, int src_C, void* dst, int dst_C, long npix, float scale, cudaStream_t s) {
  scale_copy64_kernel<<<grid_for(npix * 8, 256), 256, 0, s>>>(reinterpret_cast<const __nv_bfloat16*>(src), src_C,
                                                              reinterpret_cast<__nv_bfloat16*>(dst), dst_C, npix, scale);
  return cudaGetLastError();
}

// ---- gradient exchange buffers (data-parallel training) -----------------------------------------------------------
// bf16 wire format of the gradient all-reduce: comm[i] = bf16(scale * flat[i]) (scale = 1 / world BEFORE the rounding, so the
// sum over ranks stays in range) and back: flat[i] = float(comm[i]).  Small grids on purpose: they run on the SMs reserved for
// the collective while the backward kernels own the rest.
__global__ void grad_pack_bf16_kernel(const float* __restrict__ flat, __nv_bfloat16* __restrict__ comm, long n, float scale) {
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < n; i += static_cast<long>(gridDim.x) * blockDim.x)
    comm[i] = __float2bfloat16_rn(flat[i] * scale);
}
__global__ void grad_unpack_bf16_kernel(const __nv_bfloat16* __restrict__ comm, float* __restrict__ flat, long n, float scale) {
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < n; i += static_cast<long>(gridDim.x) * blockDim.x)
    flat[i] = __bfloat162float(comm[i]) * scale;
}
cudaError_t launch_grad_pack_bf16(const float* flat, void* comm, long n, float scale, int max_blocks, cudaStream_t s) {
  grad_pack_bf16_kernel<<<grid_for(n, 512, max_blocks), 512, 0, s>>>(flat, reinterpret_cast<__nv_bfloat16*>(comm), n, scale);
  return cudaGetLastError();
}
cudaError_t launch_grad_unpack_bf16(const void* comm, float* flat, long n, float scale, int max_blocks, cudaStream_t s) {
  grad_unpack_bf16_kernel<<<grid_for(n, 512, max_blocks), 512, 0, s>>>(reinterpret_cast<const __nv_bfloat16*>(comm), flat, n, scale);
  return cudaGetLastError();
}

cudaError_t launch_pack_jobs(const PackJob* jobs_dev, int njobs, cudaStream_t s) {
  pack_jobs_kernel<<<dim3(16, njobs), 256, 0, s>>>(jobs_dev);
  return cudaGetLastError();
}

cudaError_t launch_gcol_pack(const void* src, int src_C, void* dst, int dst_C, int H, int W, long total_pix, int KH, int KW, cudaStream_t s) {
  __nv_bfloat16* d = reinterpret_cast<__nv_bfloat16*>(dst);
  const int grid = grid_for(total_pix, 128, 148 * 32);
  if (KH == 5 && KW == 5 && dst_C == 32) gcol_pack_kernel<5, 5, 32><<<grid, 128, 0, s>>>(src, src_C, d, H, W, total_pix);
  else if (KH == 3 && KW == 3 && dst_C == 16) gcol_pack_kernel<3, 3, 16><<<grid, 128, 0, s>>>(src, src_C, d, H, W, total_pix);
  else return cudaErrorInvalidValue;
  return cudaGetLastError();
}

// ---- min-max scaler (inference pre / post-processing) ---------------------------------------------------------
// Pure HBM streaming: 4 B read + 4 B written per value (normalize also writes the shared elevation / mask planes into the
// batch: 12 B written per LR pixel).  Coefficients per raster as in MinMaxScaler (normalization.py:53-55): float64.
__global__ void minmax_normalize_kernel(const float* __restrict__ raw, long hw, const double* __restrict__ mn, const double* __restrict__ mx,
                                        double a, double b, double eps, float nan_sub, const float* __restrict__ extra0,
                                        const float* __restrict__ extra1, float* __restrict__ out, int n_ch) {
  const int n = blockIdx.y;
  const double scale = (b - a) / ((mx[n] - mn[n]) + eps);
  const double min_ = a - mn[n] * scale;
  const float* src = raw + static_cast<long>(n) * hw;
  float* dst = out + static_cast<long>(n) * n_ch * hw;
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < hw; i += static_cast<long>(gridDim.x) * blockDim.x) {
    double v = static_cast<double>(src[i]) * scale;
    v += min_;
    dst[i] = (v != v) ? nan_sub : static_cast<float>(v);
    if (extra0) dst[hw + i] = extra0[i];
    if (extra1) dst[(extra0 ? 2 : 1) * hw + i] = extra1[i];
  }
}

__global__ void minmax_denormalize_mask_kernel(const float* __restrict__ sr, const float* __restrict__ mask, long mask_stride, long hw,
                                               const double* __restrict__ mn, const double* __restrict__ mx, double a, double b, double eps,
                                               float* __restrict__ out) {
  const int n = blockIdx.y;
  const double scale = (b - a) / ((mx[n] - mn[n]) + eps);
  const double min_ = a - mn[n] * scale;
  const float* src = sr + static_cast<long>(n) * hw;
  const float* m = mask + static_cast<long>(n) * mask_stride;
  float* dst = out + static_cast<long>(n) * hw;
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < hw; i += static_cast<long>(gridDim.x) * blockDim.x) {
    const double v = (static_cast<double>(src[i]) - min_) / scale;
    dst[i] = (m[i] > 0.f) ? static_cast<float>(v) : __int_as_float(0x7fc00000);
  }
}

cudaError_t launch_minmax_normalize(const float* raw, int n, long hw, const double* mn, const double* mx, double a, double b, double eps,
                                    float nan_sub, const float* extra0, const float* extra1, float* out, cudaStream_t s) {
  const int n_ch = 1 + (extra0 ? 1 : 0) + (extra1 ? 1 : 0);
  const int bx = static_cast<int>(std::min<long>((hw + 255) / 256, 148 * 8));
  minmax_normalize_kernel<<<dim3(bx, n), 256, 0, s>>>(raw, hw, mn, mx, a, b, eps, nan_sub, extra0, extra1, out, n_ch);
  return cudaGetLastError();
}

cudaError_t launch_minmax_denormalize_mask(const float* sr, const float* mask, long mask_stride, int n, long hw, const double* mn,
                                           const double* mx, double a, double b, double eps, float* out, cudaStream_t s) {
  const int bx = static_cast<int>(std::min<long>((hw + 255) / 256, 148 * 8));
  minmax_denormalize_mask_kernel<<<dim3(bx, n), 256, 0, s>>>(sr, mask, mask_stride, hw, mn, mx, a, b, eps, out);
  return cudaGetLastError();
}

// ---- training-sample assembly -----------------------------------------------------------------------------------
// Index work only (bit-exact).  One thread per OUTPUT HR pixel (i,j): source pixel under rot90^-1, then the flips undone;
// every scale-th pixel in both directions also goes to the LR input x.  12 B read + 12 B written per HR pixel.
__global__ void lr_input_kernel(const float* __restrict__ hr, const float* __restrict__ elev, const float* __restrict__ mask, int H, int W,
                                int scale, const int* __restrict__ codes, float* __restrict__ hr_out, float* __restrict__ elev_out,
                                float* __restrict__ mask_out, float* __restrict__ x_out) {
  const int n = blockIdx.y;
  const int code = codes ? codes[n] : 0;
  const bool vf = code & 1, hf = code & 2;
  const int k = (code >> 2) & 3;
  const long hw = static_cast<long>(H) * W;
  const int h = H / scale, w = W / scale;
  const float* a = hr + n * hw;
  const float* e = elev + n * hw;
  const float* m = mask + n * hw;
  for (long p = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; p < hw; p += static_cast<long>(gridDim.x) * blockDim.x) {
    const int i = static_cast<int>(p / W), j = static_cast<int>(p - static_cast<long>(i) * W);
    // np.rot90(m, k)[i][j] = m[i1][j1]  (square tiles when k is odd)
    int i1 = i, j1 = j;
    if (k == 1) { i1 = j; j1 = W - 1 - i; }
    else if (k == 2) { i1 = H - 1 - i; j1 = W - 1 - j; }
    else if (k == 3) { i1 = H - 1 - j; j1 = i; }
    if (hf) j1 = W - 1 - j1;
    if (vf) i1 = H - 1 - i1;
    const long q = static_cast<long>(i1) * W + j1;
    const float va = a[q], ve = e[q], vm = m[q];
    if (hr_out) { hr_out[n * hw + p] = va; elev_out[n * hw + p] = ve; mask_out[n * hw + p] = vm; }
    if (i % scale == 0 && j % scale == 0 && i / scale < h && j / scale < w) {
      const long o = (static_cast<long>(n) * 3 * h + i / scale) * w + j / scale;
      x_out[o] = va;
      x_out[o + static_cast<long>(h) * w] = ve;
      x_out[o + 2L * h * w] = vm;
    }
  }
}

cudaError_t launch_lr_input(const float* hr, const float* elev, const float* mask, int n, int H, int W, int scale, const int* codes,
                            float* hr_out, float* elev_out, float* mask_out, float* x_out, cudaStream_t s) {
  const long hw = static_cast<long>(H) * W;
  const int bx = static_cast<int>(std::min<long>((hw + 255) / 256, 148 * 8));
  lr_input_kernel<<<dim3(bx, n), 256, 0, s>>>(hr, elev, mask, H, W, scale, codes, hr_out, elev_out, mask_out, x_out);
  return cudaGetLastError();
}

}  // namespace csr

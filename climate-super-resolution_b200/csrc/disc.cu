// Glue kernels of the discriminator path (SURVEY.md section 8f row 2; climsr/models/discriminator.py:5-46): everything between
// the tensor-core convolutions - reflection padding, stride-2 selection, BatchNorm (batch statistics, normalise-on-load, its
// backward), the LeakyReLU derivative gates of the backward pass, the flatten + two small Linear layers.  All HBM-bound
// streaming kernels over NHWC bf16 buffers, 8 channels (16 bytes) per thread.
//
// Layout convention.  A conv layer runs as a "same" (zero-padded) conv of conv_tc over its already reflection-padded input
// P (N, H+2p, W+2p, C); its output buffer S has the same spatial size and the layer's real outputs are the *logical* pixels
//   S[off + step*i][off + step*j],  i < Hl, j < Wl        (off = 1; step = 1, or 2 for the stride-2 convs)
// i.e. ReflectionPad2d(1) + Conv2d(3) == interior of the same-conv over P, and stride 2 == every second interior pixel.
// `View` describes such a logical image.  The next layer's input is gathered from it (disc_gather_kernel), gradients are
// brought back to it (disc_collect_kernel / disc_bn_bwd_apply_kernel, which also write zeros to the non-logical pixels, so
// the conv's weight / input gradients over the padded grid see exactly the real output gradient).
#include "disc.cuh"

#include <cuda_bf16.h>

namespace csr {

namespace {

__device__ __forceinline__ int reflect_idx(int t, int n) { return t < 0 ? -t : (t >= n ? 2 * n - 2 - t : t); }
__device__ __forceinline__ float lo16(uint32_t v) { return __uint_as_float(v << 16); }
__device__ __forceinline__ float hi16(uint32_t v) { return __uint_as_float(v & 0xFFFF0000u); }
__device__ __forceinline__ uint32_t pack2(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ void unpack8(const uint4& q, float (&v)[8]) {
  v[0] = lo16(q.x); v[1] = hi16(q.x); v[2] = lo16(q.y); v[3] = hi16(q.y); v[4] = lo16(q.z); v[5] = hi16(q.z); v[6] = lo16(q.w); v[7] = hi16(q.w);
}
__device__ __forceinline__ uint4 pack8(const float (&v)[8]) {
  return make_uint4(pack2(v[0], v[1]), pack2(v[2], v[3]), pack2(v[4], v[5]), pack2(v[6], v[7]));
}

// dst (N, Hl+2p, Wl+2p, C) <- reflection-padded (p = 1) or plain (p = 0) copy of the logical image of `src`, optionally through
// the per-channel affine y = x * scale[c] + shift[c] (BatchNorm normalise-on-load).
__global__ void disc_gather_kernel(const __nv_bfloat16* __restrict__ src, DiscView v, __nv_bfloat16* __restrict__ dst, int pad,
                                   const float* __restrict__ scale, const float* __restrict__ shift, long total) {
  const int c8n = v.C >> 3;
  const int Hd = v.Hl + 2 * pad, Wd = v.Wl + 2 * pad;
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < total; i += static_cast<long>(gridDim.x) * blockDim.x) {
    const int c8 = static_cast<int>(i % c8n);
    long r = i / c8n;
    const int x = static_cast<int>(r % Wd); r /= Wd;
    const int y = static_cast<int>(r % Hd);
    const int n = static_cast<int>(r / Hd);
    const int sy = v.off + v.step * reflect_idx(y - pad, v.Hl), sx = v.off + v.step * reflect_idx(x - pad, v.Wl);
    uint4 q = *reinterpret_cast<const uint4*>(src + ((static_cast<long>(n) * v.Hs + sy) * v.Ws + sx) * v.C + c8 * 8);
    if (scale) {
      float f[8];
      unpack8(q, f);
#pragma unroll
      for (int k = 0; k < 8; ++k) f[k] = f[k] * scale[c8 * 8 + k] + shift[c8 * 8 + k];
      q = pack8(f);
    }
    *reinterpret_cast<uint4*>(dst + i * 8) = q;
  }
}

// Gradient w.r.t. logical pixel (n, i, j) of the image that disc_gather_kernel padded: the sum of dP over the <= 2 x 2 padded
// positions that read it.
__device__ __forceinline__ void collect8(const __nv_bfloat16* __restrict__ dP, int n, int i, int j, int c8, const DiscView& v, int pad,
                                         float (&acc)[8]) {
  const int Hd = v.Hl + 2 * pad, Wd = v.Wl + 2 * pad;
  int ys[3], xs[3], ny = 1, nx = 1;
  ys[0] = i + pad; xs[0] = j + pad;
  if (pad) {                                              // reflection (pad 1): padded row 0 reads row 1, the last padded row reads row Hl-2
    if (i == 1) ys[ny++] = 0;
    if (i == v.Hl - 2) ys[ny++] = Hd - 1;
    if (j == 1) xs[nx++] = 0;
    if (j == v.Wl - 2) xs[nx++] = Wd - 1;
  }
#pragma unroll
  for (int k = 0; k < 8; ++k) acc[k] = 0.f;
  for (int a = 0; a < ny; ++a)
    for (int b = 0; b < nx; ++b) {
      const uint4 q = *reinterpret_cast<const uint4*>(dP + ((static_cast<long>(n) * Hd + ys[a]) * Wd + xs[b]) * v.C + c8 * 8);
      float f[8];
      unpack8(q, f);
#pragma unroll
      for (int k = 0; k < 8; ++k) acc[k] += f[k];
    }
}

// Backward of disc_gather for a layer WITHOUT BatchNorm after it: over ALL pixels of the S-layout buffer, logical pixels get
// g = lrelu'(x) * dy (x = the saved post-activation output, gate_neg = the LeakyReLU slope, 1 = no activation), others zero.
__global__ void disc_collect_kernel(const __nv_bfloat16* __restrict__ dP, DiscView v, int pad, const __nv_bfloat16* __restrict__ act,
                                    float gate_neg, __nv_bfloat16* __restrict__ g, long total) {
  const int c8n = v.C >> 3;
  for (long t = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; t < total; t += static_cast<long>(gridDim.x) * blockDim.x) {
    const int c8 = static_cast<int>(t % c8n);
    long r = t / c8n;
    const int x = static_cast<int>(r % v.Ws); r /= v.Ws;
    const int y = static_cast<int>(r % v.Hs);
    const int n = static_cast<int>(r / v.Hs);
    const int iy = y - v.off, ix = x - v.off;
    uint4 out = make_uint4(0, 0, 0, 0);
    if (iy >= 0 && ix >= 0 && iy % v.step == 0 && ix % v.step == 0 && iy / v.step < v.Hl && ix / v.step < v.Wl) {
      float acc[8];
      collect8(dP, n, iy / v.step, ix / v.step, c8, v, pad, acc);
      if (act) {
        float a[8];
        unpack8(*reinterpret_cast<const uint4*>(act + t * 8), a);
#pragma unroll
        for (int k = 0; k < 8; ++k) acc[k] *= (a[k] > 0.f) ? 1.f : gate_neg;
      }
      out = pack8(acc);
    }
    *reinterpret_cast<uint4*>(g + t * 8) = out;
  }
}

// Per-channel block reduction of the two 8-channel partial sums every thread holds (thread = channel group c8 x pixel lane):
// shared memory [lanes][2*C] -> one double atomic per (block, channel, quantity) instead of one per thread (the per-thread form
// put ~1.2 M atomics on 128..1024 addresses: 170 us per launch).
__device__ __forceinline__ void block_reduce_to_sums(const float (&s)[8], const float (&q)[8], int C, int c8, int c8n, double* __restrict__ sums) {
  extern __shared__ float red[];                          // [lanes][2 * C]
  const int lane_id = threadIdx.x / c8n, lanes = blockDim.x / c8n;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    red[lane_id * 2 * C + c8 * 8 + k] = s[k];
    red[lane_id * 2 * C + C + c8 * 8 + k] = q[k];
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * C; i += blockDim.x) {
    float t = 0.f;
    for (int l = 0; l < lanes; ++l) t += red[l * 2 * C + i];
    atomicAdd(sums + i, static_cast<double>(t));
  }
}

// ---- BatchNorm2d, training mode (batch statistics over the logical pixels) ---------------------------------------------
// The sums are taken of x - pivot[c], pivot = the channel's first logical pixel (image 0, pixel (0, 0)): with raw x, the fp32
// per-thread partials of x^2 carry mean^2 and the variance E[x^2] - mean^2 cancels their rounding error into the result
// (invstd 1.8e-4 off at mean = 100 std, 16 x 128 x 128 pixels); around a pivot a few std from the mean nothing cancels.
__device__ __forceinline__ long bn_pivot_index(const DiscView& v) { return (static_cast<long>(v.off) * v.Ws + v.off) * v.C; }

// sums[c] += x - pivot[c], sums[C + c] += (x - pivot[c])^2 (double atomics; a few hundred blocks)
__global__ void disc_bn_stats_kernel(const __nv_bfloat16* __restrict__ src, DiscView v, int N, double* __restrict__ sums) {
  const int c8n = v.C >> 3;
  const int c8 = threadIdx.x % c8n;                       // blockDim.x is a multiple of C/8: a thread keeps its channel group
  const int lanes = blockDim.x / c8n;
  const long npix = static_cast<long>(N) * v.Hl * v.Wl;
  float s[8], q[8], piv[8];
  unpack8(*reinterpret_cast<const uint4*>(src + bn_pivot_index(v) + c8 * 8), piv);
#pragma unroll
  for (int k = 0; k < 8; ++k) s[k] = q[k] = 0.f;
  for (long p = blockIdx.x * static_cast<long>(lanes) + threadIdx.x / c8n; p < npix; p += static_cast<long>(gridDim.x) * lanes) {
    const int j = static_cast<int>(p % v.Wl);
    long r = p / v.Wl;
    const int i = static_cast<int>(r % v.Hl);
    const int n = static_cast<int>(r / v.Hl);
    float f[8];
    unpack8(*reinterpret_cast<const uint4*>(src + ((static_cast<long>(n) * v.Hs + v.off + v.step * i) * v.Ws + v.off + v.step * j) * v.C + c8 * 8), f);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const float d = f[k] - piv[k];                      // exact: two bf16 values
      s[k] += d;
      q[k] += d * d;
    }
  }
  block_reduce_to_sums(s, q, v.C, c8, c8n, sums);
}

// mean = pivot + sum(x - pivot) / M, biased variance from the pivot-shifted sums -> scale = gamma * invstd, shift = beta - mean * scale; saves (mean, invstd) for the backward and
// updates the running statistics like nn.BatchNorm2d (momentum, unbiased variance).
__global__ void disc_bn_finalize_kernel(const double* __restrict__ sums, const __nv_bfloat16* __restrict__ src, DiscView v, double count,
                                        const float* __restrict__ gamma, const float* __restrict__ beta, float eps, float momentum, float* __restrict__ running_mean,
                                        float* __restrict__ running_var, float* __restrict__ scale, float* __restrict__ shift,
                                        float* __restrict__ mean_out, float* __restrict__ invstd_out) {
  const int C = v.C;
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const double d = sums[c] / count;                       // mean of x - pivot
  const double mean = static_cast<double>(__bfloat162float(src[bn_pivot_index(v) + c])) + d;
  const double var = fmax(sums[C + c] / count - d * d, 0.0);
  const float invstd = static_cast<float>(1.0 / sqrt(var + static_cast<double>(eps)));
  const float sc = gamma[c] * invstd;
  scale[c] = sc;
  shift[c] = beta[c] - static_cast<float>(mean) * sc;
  mean_out[c] = static_cast<float>(mean);
  invstd_out[c] = invstd;
  if (running_mean) {
    running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * static_cast<float>(mean);
    running_var[c] = (1.f - momentum) * running_var[c] + momentum * static_cast<float>(count > 1 ? var * count / (count - 1) : var);
  }
}

// eval mode: scale / shift from the running statistics
__global__ void disc_bn_eval_kernel(int C, const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
                                    const float* __restrict__ running_mean, const float* __restrict__ running_var, float* __restrict__ scale,
                                    float* __restrict__ shift) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const float sc = gamma[c] * rsqrtf(running_var[c] + eps);
  scale[c] = sc;
  shift[c] = beta[c] - running_mean[c] * sc;
}

// BatchNorm backward, pass 1: dy (gradient w.r.t. the BN output at every logical pixel, fp32 dense) and the per-channel sums
// sums[c] += dy, sums[C + c] += dy * xhat.
__global__ void disc_bn_bwd_reduce_kernel(const __nv_bfloat16* __restrict__ dP, DiscView v, int pad, int N, const __nv_bfloat16* __restrict__ act,
                                          const float* __restrict__ mean, const float* __restrict__ invstd, float* __restrict__ dy,
                                          double* __restrict__ sums) {
  const int c8n = v.C >> 3;
  const int c8 = threadIdx.x % c8n;
  const int lanes = blockDim.x / c8n;
  const long npix = static_cast<long>(N) * v.Hl * v.Wl;
  float s[8], q[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) s[k] = q[k] = 0.f;
  for (long p = blockIdx.x * static_cast<long>(lanes) + threadIdx.x / c8n; p < npix; p += static_cast<long>(gridDim.x) * lanes) {
    const int j = static_cast<int>(p % v.Wl);
    long r = p / v.Wl;
    const int i = static_cast<int>(r % v.Hl);
    const int n = static_cast<int>(r / v.Hl);
    float acc[8], a[8];
    collect8(dP, n, i, j, c8, v, pad, acc);
    unpack8(*reinterpret_cast<const uint4*>(act + ((static_cast<long>(n) * v.Hs + v.off + v.step * i) * v.Ws + v.off + v.step * j) * v.C + c8 * 8), a);
    float4* o = reinterpret_cast<float4*>(dy + p * v.C + c8 * 8);
    o[0] = make_float4(acc[0], acc[1], acc[2], acc[3]);
    o[1] = make_float4(acc[4], acc[5], acc[6], acc[7]);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const float xh = (a[k] - mean[c8 * 8 + k]) * invstd[c8 * 8 + k];
      s[k] += acc[k];
      q[k] += acc[k] * xh;
    }
  }
  block_reduce_to_sums(s, q, v.C, c8, c8n, sums);
}

// pass 2 over ALL pixels of the S-layout buffer: logical pixels get
//   g = lrelu'(x) * gamma * invstd * (dy - sum(dy)/M - xhat * sum(dy xhat)/M),   others zero;
// block 0 also writes dgamma = sum(dy xhat), dbeta = sum(dy).
__global__ void disc_bn_bwd_apply_kernel(const float* __restrict__ dy, DiscView v, int N, const __nv_bfloat16* __restrict__ act, float gate_neg,
                                         const float* __restrict__ gamma, const float* __restrict__ mean, const float* __restrict__ invstd,
                                         const double* __restrict__ sums, __nv_bfloat16* __restrict__ g, float* __restrict__ dgamma,
                                         float* __restrict__ dbeta, long total) {
  const int c8n = v.C >> 3;
  const double M = static_cast<double>(N) * v.Hl * v.Wl;
  if (blockIdx.x == 0)
    for (int c = threadIdx.x; c < v.C; c += blockDim.x) {
      dbeta[c] += static_cast<float>(sums[c]);
      dgamma[c] += static_cast<float>(sums[v.C + c]);
    }
  for (long t = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; t < total; t += static_cast<long>(gridDim.x) * blockDim.x) {
    const int c8 = static_cast<int>(t % c8n);
    long r = t / c8n;
    const int x = static_cast<int>(r % v.Ws); r /= v.Ws;
    const int y = static_cast<int>(r % v.Hs);
    const int n = static_cast<int>(r / v.Hs);
    const int iy = y - v.off, ix = x - v.off;
    uint4 out = make_uint4(0, 0, 0, 0);
    if (iy >= 0 && ix >= 0 && iy % v.step == 0 && ix % v.step == 0 && iy / v.step < v.Hl && ix / v.step < v.Wl) {
      const long p = (static_cast<long>(n) * v.Hl + iy / v.step) * v.Wl + ix / v.step;
      const float4* d4 = reinterpret_cast<const float4*>(dy + p * v.C + c8 * 8);
      const float4 d0 = d4[0], d1 = d4[1];
      const float d[8] = {d0.x, d0.y, d0.z, d0.w, d1.x, d1.y, d1.z, d1.w};
      float a[8], o[8];
      unpack8(*reinterpret_cast<const uint4*>(act + t * 8), a);
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int c = c8 * 8 + k;
        const float xh = (a[k] - mean[c]) * invstd[c];
        const float dx = gamma[c] * invstd[c] * (d[k] - static_cast<float>(sums[c] / M) - xh * static_cast<float>(sums[v.C + c] / M));
        o[k] = dx * ((a[k] > 0.f) ? 1.f : gate_neg);
      }
      out = pack8(o);
    }
    *reinterpret_cast<uint4*>(g + t * 8) = out;
  }
}

// ---- flatten + Linear ---------------------------------------------------------------------------------------------------
// x.view(N, -1) of the NCHW tensor: feature f = c * Hl*Wl + i * Wl + j  <-  logical pixel (i, j), channel c of the S buffer
__global__ void disc_flatten_kernel(const __nv_bfloat16* __restrict__ src, DiscView v, int N, float* __restrict__ feats) {
  const long total = static_cast<long>(N) * v.C * v.Hl * v.Wl;
  for (long t = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; t < total; t += static_cast<long>(gridDim.x) * blockDim.x) {
    const int j = static_cast<int>(t % v.Wl);
    long r = t / v.Wl;
    const int i = static_cast<int>(r % v.Hl); r /= v.Hl;
    const int c = static_cast<int>(r % v.C);
    const int n = static_cast<int>(r / v.C);
    feats[t] = __bfloat162float(src[((static_cast<long>(n) * v.Hs + v.off + v.step * i) * v.Ws + v.off + v.step * j) * v.C + c]);
  }
}
// its backward: the fp32 feature gradient goes back to the logical pixels of an S-layout bf16 buffer, zeros elsewhere
__global__ void disc_unflatten_kernel(const float* __restrict__ gfeat, DiscView v, int N, __nv_bfloat16* __restrict__ g) {
  const long total = static_cast<long>(N) * v.Hs * v.Ws * v.C;
  for (long t = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; t < total; t += static_cast<long>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(t % v.C);
    long r = t / v.C;
    const int x = static_cast<int>(r % v.Ws); r /= v.Ws;
    const int y = static_cast<int>(r % v.Hs);
    const int n = static_cast<int>(r / v.Hs);
    const int iy = y - v.off, ix = x - v.off;
    float val = 0.f;
    if (iy >= 0 && ix >= 0 && iy % v.step == 0 && ix % v.step == 0 && iy / v.step < v.Hl && ix / v.step < v.Wl)
      val = gfeat[((static_cast<long>(n) * v.C + c) * v.Hl + iy / v.step) * v.Wl + ix / v.step];
    g[t] = __float2bfloat16_rn(val);
  }
}

// y[n][j] = b[j] + sum_k x[n][k] W[j][k]: one block per (j, n), fp32.  (8192 -> 100 -> 1 on <= a few dozen samples: microseconds.)
__global__ void linear_fwd_kernel(const float* __restrict__ x, const float* __restrict__ W, const float* __restrict__ b, float* __restrict__ y,
                                  int K, int J) {
  const int j = blockIdx.x, n = blockIdx.y;
  float s = 0.f;
  for (int k = threadIdx.x; k < K; k += blockDim.x) s += x[static_cast<long>(n) * K + k] * W[static_cast<long>(j) * K + k];
  __shared__ float sh[32];
  for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < static_cast<int>(blockDim.x >> 5); ++w) t += sh[w];
    y[static_cast<long>(n) * J + j] = t + (b ? b[j] : 0.f);
  }
}
// dx[n][k] = sum_j gy[n][j] W[j][k]
__global__ void linear_bwd_x_kernel(const float* __restrict__ gy, const float* __restrict__ W, float* __restrict__ dx, int N, int K, int J) {
  const long total = static_cast<long>(N) * K;
  for (long t = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; t < total; t += static_cast<long>(gridDim.x) * blockDim.x) {
    const int k = static_cast<int>(t % K);
    const int n = static_cast<int>(t / K);
    float s = 0.f;
    for (int j = 0; j < J; ++j) s += gy[static_cast<long>(n) * J + j] * W[static_cast<long>(j) * K + k];
    dx[t] = s;
  }
}
// dW[j][k] += sum_n gy[n][j] x[n][k];  db[j] += sum_n gy[n][j]
__global__ void linear_bwd_w_kernel(const float* __restrict__ gy, const float* __restrict__ x, float* __restrict__ dW, float* __restrict__ db,
                                    int N, int K, int J) {
  const long total = static_cast<long>(J) * K;
  for (long t = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; t < total; t += static_cast<long>(gridDim.x) * blockDim.x) {
    const int k = static_cast<int>(t % K);
    const int j = static_cast<int>(t / K);
    float s = 0.f;
    for (int n = 0; n < N; ++n) s += gy[static_cast<long>(n) * J + j] * x[static_cast<long>(n) * K + k];
    dW[t] += s;
    if (k == 0 && db) {
      float sb = 0.f;
      for (int n = 0; n < N; ++n) sb += gy[static_cast<long>(n) * J + j];
      db[j] += sb;
    }
  }
}
// db[j] += sum_n gy[n][j] alone (dW not wanted); same summation order as linear_bwd_w_kernel
__global__ void linear_bwd_b_kernel(const float* __restrict__ gy, float* __restrict__ db, int N, int J) {
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < J; j += gridDim.x * blockDim.x) {
    float sb = 0.f;
    for (int n = 0; n < N; ++n) sb += gy[static_cast<long>(n) * J + j];
    db[j] += sb;
  }
}

inline int grid_for(long total, int block, int cap = 148 * 8) {
  long g = (total + block - 1) / block;
  return static_cast<int>(g < 1 ? 1 : (g > cap ? cap : g));
}
inline int stats_block(int C) {                           // a multiple of C/8 close to 256 (C = 64 .. 512 -> C/8 = 8 .. 64)
  const int c8n = C >> 3;
  return (256 / c8n > 0 ? 256 / c8n : 1) * c8n;
}

}  // namespace

cudaError_t launch_disc_gather(const void* src, const DiscView& v, int N, void* dst, int pad, const float* scale, const float* shift, cudaStream_t s) {
  const long total = static_cast<long>(N) * (v.Hl + 2 * pad) * (v.Wl + 2 * pad) * (v.C >> 3);
  disc_gather_kernel<<<grid_for(total, 256), 256, 0, s>>>(reinterpret_cast<const __nv_bfloat16*>(src), v, reinterpret_cast<__nv_bfloat16*>(dst), pad,
                                                          scale, shift, total);
  return cudaGetLastError();
}
cudaError_t launch_disc_collect(const void* dP, const DiscView& v, int N, int pad, const void* act, float gate_neg, void* g, cudaStream_t s) {
  const long total = static_cast<long>(N) * v.Hs * v.Ws * (v.C >> 3);
  disc_collect_kernel<<<grid_for(total, 256), 256, 0, s>>>(reinterpret_cast<const __nv_bfloat16*>(dP), v, pad,
                                                           reinterpret_cast<const __nv_bfloat16*>(act), gate_neg, reinterpret_cast<__nv_bfloat16*>(g), total);
  return cudaGetLastError();
}
cudaError_t launch_disc_bn_stats(const void* src, const DiscView& v, int N, double* sums, cudaStream_t s) {
  cudaError_t e = cudaMemsetAsync(sums, 0, 2 * v.C * sizeof(double), s);
  if (e != cudaSuccess) return e;
  const int block = stats_block(v.C);
  const long npix = static_cast<long>(N) * v.Hl * v.Wl;
  disc_bn_stats_kernel<<<grid_for(npix, block / (v.C >> 3), 148 * 2), block, (block / (v.C >> 3)) * 2 * v.C * sizeof(float), s>>>(
      reinterpret_cast<const __nv_bfloat16*>(src), v, N, sums);
  return cudaGetLastError();
}
cudaError_t launch_disc_bn_finalize(const double* sums, const void* src, const DiscView& v, double count, const float* gamma, const float* beta,
                                    float eps, float momentum, float* running_mean, float* running_var, float* scale, float* shift, float* mean,
                                    float* invstd, cudaStream_t s) {
  disc_bn_finalize_kernel<<<(v.C + 127) / 128, 128, 0, s>>>(sums, reinterpret_cast<const __nv_bfloat16*>(src), v, count, gamma, beta, eps,
                                                            momentum, running_mean, running_var, scale, shift, mean, invstd);
  return cudaGetLastError();
}
cudaError_t launch_disc_bn_eval(int C, const float* gamma, const float* beta, float eps, const float* running_mean, const float* running_var,
                                float* scale, float* shift, cudaStream_t s) {
  disc_bn_eval_kernel<<<(C + 127) / 128, 128, 0, s>>>(C, gamma, beta, eps, running_mean, running_var, scale, shift);
  return cudaGetLastError();
}
cudaError_t launch_disc_bn_backward(const void* dP, const DiscView& v, int N, int pad, const void* act, float gate_neg, const float* gamma,
                                    const float* mean, const float* invstd, float* dy, double* sums, void* g, float* dgamma, float* dbeta,
                                    cudaStream_t s) {
  cudaError_t e = cudaMemsetAsync(sums, 0, 2 * v.C * sizeof(double), s);
  if (e != cudaSuccess) return e;
  const int block = stats_block(v.C);
  const long npix = static_cast<long>(N) * v.Hl * v.Wl;
  disc_bn_bwd_reduce_kernel<<<grid_for(npix, block / (v.C >> 3), 148 * 2), block, (block / (v.C >> 3)) * 2 * v.C * sizeof(float), s>>>(
      reinterpret_cast<const __nv_bfloat16*>(dP), v, pad, N, reinterpret_cast<const __nv_bfloat16*>(act), mean, invstd, dy, sums);
  const long total = static_cast<long>(N) * v.Hs * v.Ws * (v.C >> 3);
  disc_bn_bwd_apply_kernel<<<grid_for(total, 256), 256, 0, s>>>(dy, v, N, reinterpret_cast<const __nv_bfloat16*>(act), gate_neg, gamma, mean, invstd,
                                                                sums, reinterpret_cast<__nv_bfloat16*>(g), dgamma, dbeta, total);
  return cudaGetLastError();
}
cudaError_t launch_disc_flatten(const void* src, const DiscView& v, int N, float* feats, cudaStream_t s) {
  const long total = static_cast<long>(N) * v.C * v.Hl * v.Wl;
  disc_flatten_kernel<<<grid_for(total, 256), 256, 0, s>>>(reinterpret_cast<const __nv_bfloat16*>(src), v, N, feats);
  return cudaGetLastError();
}
cudaError_t launch_disc_unflatten(const float* gfeat, const DiscView& v, int N, void* g, cudaStream_t s) {
  const long total = static_cast<long>(N) * v.Hs * v.Ws * v.C;
  disc_unflatten_kernel<<<grid_for(total, 256), 256, 0, s>>>(gfeat, v, N, reinterpret_cast<__nv_bfloat16*>(g));
  return cudaGetLastError();
}
cudaError_t launch_linear_forward(const float* x, const float* W, const float* b, float* y, int N, int K, int J, cudaStream_t s) {
  linear_fwd_kernel<<<dim3(J, N), 256, 0, s>>>(x, W, b, y, K, J);
  return cudaGetLastError();
}
cudaError_t launch_linear_backward(const float* x, const float* W, const float* gy, float* dx, float* dW, float* db, int N, int K, int J,
                                   cudaStream_t s) {
  if (dx) linear_bwd_x_kernel<<<grid_for(static_cast<long>(N) * K, 256), 256, 0, s>>>(gy, W, dx, N, K, J);
  if (dW) linear_bwd_w_kernel<<<grid_for(static_cast<long>(J) * K, 256), 256, 0, s>>>(gy, x, dW, db, N, K, J);
  else if (db) linear_bwd_b_kernel<<<grid_for(J, 256), 256, 0, s>>>(gy, db, N, J);
  return cudaGetLastError();
}

}  // namespace csr

// Glue kernels of the RCAN generator (SURVEY.md section 8f row 4; climsr/models/rcan.py:50-101, 17-47): what sits between the
// tensor-core convolutions of a Residual Channel Attention Block - global average pooling, the two 1x1 convs + sigmoid of
// CALayer, the channel scaling and the block's skip-add - and PixelShuffle(2) of the Upsampler.  HBM-bound streaming kernels
// over NHWC bf16, 8 channels (16 bytes) per thread.
#include "rcan.cuh"

#include <cuda_bf16.h>

namespace csr {

namespace {

__device__ __forceinline__ float lo16(uint32_t v) { return __uint_as_float(v << 16); }
__device__ __forceinline__ float hi16(uint32_t v) { return __uint_as_float(v & 0xFFFF0000u); }
__device__ __forceinline__ uint32_t pack2(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ void unpack8(const uint4& q, float (&v)[8]) {
  v[0] = lo16(q.x); v[1] = hi16(q.x); v[2] = lo16(q.y); v[3] = hi16(q.y); v[4] = lo16(q.z); v[5] = hi16(q.z); v[6] = lo16(q.w); v[7] = hi16(q.w);
}

// nn.AdaptiveAvgPool2d(1) (rcan.py:56): pooled[n][c] += sum over the pixels of image n (the mean is taken by the consumer).
// With `mul` (the channel-attention backward): pooled[n][c] += sum of src * mul, the gate's gradient before the sigmoid.
// grid = (blocks per image, N); blockDim a multiple of C/8 so that a thread keeps its channel group.
template <bool MUL>
__global__ void channel_pool_kernel(const __nv_bfloat16* __restrict__ src, const __nv_bfloat16* __restrict__ mul, long hw, int C,
                                    float* __restrict__ pooled) {
  const int c8n = C >> 3;
  const int c8 = threadIdx.x % c8n, lanes = blockDim.x / c8n;
  const int n = blockIdx.y;
  float s[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) s[k] = 0.f;
  for (long p = blockIdx.x * static_cast<long>(lanes) + threadIdx.x / c8n; p < hw; p += static_cast<long>(gridDim.x) * lanes) {
    const long off = (static_cast<long>(n) * hw + p) * C + c8 * 8;
    float f[8];
    unpack8(*reinterpret_cast<const uint4*>(src + off), f);
    if constexpr (MUL) {
      float m[8];
      unpack8(*reinterpret_cast<const uint4*>(mul + off), m);
#pragma unroll
      for (int k = 0; k < 8; ++k) f[k] *= m[k];
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) s[k] += f[k];
  }
  // lanes of a warp with the same channel group: combine through shared memory, one atomic per (block, channel)
  extern __shared__ float sh[];                            // [lanes][C]
  const int lane_id = threadIdx.x / c8n;
#pragma unroll
  for (int k = 0; k < 8; ++k) sh[lane_id * C + c8 * 8 + k] = s[k];
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float t = 0.f;
    for (int l = 0; l < lanes; ++l) t += sh[l * C + c];
    atomicAdd(pooled + static_cast<long>(n) * C + c, t);
  }
}

// CALayer.conv_du + the RCAB skip (rcan.py:59-68, 98-101):  out = res * sigmoid(W2 relu(W1 mean + b1) + b2) + x.
// Every block recomputes the (C -> C/r -> C) gate of its image from the pooled sums (C = 64, r = 16: ~500 MACs).
// grid = (blocks per image, N).  w1: (C/r, C), w2: (C, C/r), fp32.
__global__ void ca_scale_add_kernel(const __nv_bfloat16* __restrict__ res, const __nv_bfloat16* __restrict__ x, const float* __restrict__ pooled,
                                    const float* __restrict__ w1, const float* __restrict__ b1, const float* __restrict__ w2,
                                    const float* __restrict__ b2, __nv_bfloat16* __restrict__ out, long hw, int C, int Cr) {
  extern __shared__ float sh[];                            // mean[C] | hidden[Cr] | gate[C]
  float* mean = sh;
  float* hid = sh + C;
  float* gate = hid + Cr;
  const int n = blockIdx.y;
  for (int c = threadIdx.x; c < C; c += blockDim.x) mean[c] = pooled[static_cast<long>(n) * C + c] / static_cast<float>(hw);
  __syncthreads();
  for (int j = threadIdx.x; j < Cr; j += blockDim.x) {
    float t = b1[j];
    for (int c = 0; c < C; ++c) t += w1[j * C + c] * mean[c];
    hid[j] = fmaxf(t, 0.f);
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float t = b2[c];
    for (int j = 0; j < Cr; ++j) t += w2[c * Cr + j] * hid[j];
    gate[c] = 1.f / (1.f + __expf(-t));
  }
  __syncthreads();
  const int c8n = C >> 3;
  const long total = hw * c8n;
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < total; i += static_cast<long>(gridDim.x) * blockDim.x) {
    const int c8 = static_cast<int>(i % c8n);
    const long off = (static_cast<long>(n) * hw) * C + i * 8;
    float r[8], v[8];
    unpack8(*reinterpret_cast<const uint4*>(res + off), r);
    unpack8(*reinterpret_cast<const uint4*>(x + off), v);
#pragma unroll
    for (int k = 0; k < 8; ++k) v[k] = r[k] * gate[c8 * 8 + k] + v[k];
    *reinterpret_cast<uint4*>(out + off) = make_uint4(pack2(v[0], v[1]), pack2(v[2], v[3]), pack2(v[4], v[5]), pack2(v[6], v[7]));
  }
}

// nn.PixelShuffle(2) (rcan.py:33): dst[n][2y+a][2x+b][c] = src[n][y][x][4c + 2a + b]; src (N,H,W,4C), dst (N,2H,2W,C).
__global__ void pixel_shuffle2_kernel(const __nv_bfloat16* __restrict__ src, __nv_bfloat16* __restrict__ dst, int H, int W, int C, long total) {
  const int c8n = C >> 3;
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < total; i += static_cast<long>(gridDim.x) * blockDim.x) {
    const int c8 = static_cast<int>(i % c8n);
    long r = i / c8n;
    const int X = static_cast<int>(r % (2 * W)); r /= 2 * W;
    const int Y = static_cast<int>(r % (2 * H));
    const long n = r / (2 * H);
    const int ph = (Y & 1) * 2 + (X & 1);
    const __nv_bfloat16* s = src + ((n * H + (Y >> 1)) * W + (X >> 1)) * (4L * C) + c8 * 32 + ph;
    __nv_bfloat16 v[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) v[k] = s[4 * k];
    *reinterpret_cast<uint4*>(dst + i * 8) = *reinterpret_cast<const uint4*>(v);
  }
}

// Adjoint of ca_scale_add_kernel without its skip term (dx = dout is folded into the caller's next input-gradient conv):
//   g = sigmoid(z2),  z2 = W2 hid + b2,  hid = relu(z1),  z1 = W1 mean + b1,  mean = pooled / hw
//   dz2 = dot * g (1 - g)      (dot[c] = sum over pixels of dout * res: channel_pool_kernel<true>)
//   dhid = (W2^T dz2) * [hid > 0],   dmean = W1^T dhid
//   dres = dout * g[c] + dmean[c] / hw
// Block x = 0 of each image also accumulates dW2 += dz2 hid^T, db2 += dz2, dW1 += dhid mean^T, db1 += dhid (fp32 atomics: images
// of a batch add into the same parameters).  grid = (blocks per image, N).
__global__ void ca_backward_kernel(const __nv_bfloat16* __restrict__ dout, const __nv_bfloat16* __restrict__ res,
                                   const float* __restrict__ pooled, const float* __restrict__ dot, const float* __restrict__ w1,
                                   const float* __restrict__ b1, const float* __restrict__ w2, const float* __restrict__ b2,
                                   __nv_bfloat16* __restrict__ dres, float* __restrict__ dw1, float* __restrict__ db1, float* __restrict__ dw2,
                                   float* __restrict__ db2, long hw, int C, int Cr) {
  extern __shared__ float sh[];                            // mean[C] | hid[Cr] | gate[C] | dz2[C] | dhid[Cr] | dmean[C]
  float* mean = sh;
  float* hid = mean + C;
  float* gate = hid + Cr;
  float* dz2 = gate + C;
  float* dhid = dz2 + C;
  float* dmean = dhid + Cr;
  const int n = blockIdx.y;
  const float inv_hw = 1.f / static_cast<float>(hw);
  for (int c = threadIdx.x; c < C; c += blockDim.x) mean[c] = pooled[static_cast<long>(n) * C + c] / static_cast<float>(hw);
  __syncthreads();
  for (int j = threadIdx.x; j < Cr; j += blockDim.x) {
    float t = b1[j];
    for (int c = 0; c < C; ++c) t += w1[j * C + c] * mean[c];
    hid[j] = fmaxf(t, 0.f);
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float t = b2[c];
    for (int j = 0; j < Cr; ++j) t += w2[c * Cr + j] * hid[j];
    const float g = 1.f / (1.f + __expf(-t));
    gate[c] = g;
    dz2[c] = dot[static_cast<long>(n) * C + c] * g * (1.f - g);
  }
  __syncthreads();
  for (int j = threadIdx.x; j < Cr; j += blockDim.x) {
    float t = 0.f;
    for (int c = 0; c < C; ++c) t += w2[c * Cr + j] * dz2[c];
    dhid[j] = hid[j] > 0.f ? t : 0.f;
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float t = 0.f;
    for (int j = 0; j < Cr; ++j) t += w1[j * C + c] * dhid[j];
    dmean[c] = t * inv_hw;
  }
  if (blockIdx.x == 0) {
    for (int i = threadIdx.x; i < C * Cr; i += blockDim.x) {
      const int a = i / Cr, b = i % Cr;                    // dW2[a][b]  (C, Cr)
      atomicAdd(dw2 + i, dz2[a] * hid[b]);
      const int j = i / C, c = i % C;                      // dW1[j][c]  (Cr, C)
      atomicAdd(dw1 + i, dhid[j] * mean[c]);
    }
    for (int c = threadIdx.x; c < C; c += blockDim.x) atomicAdd(db2 + c, dz2[c]);
    for (int j = threadIdx.x; j < Cr; j += blockDim.x) atomicAdd(db1 + j, dhid[j]);
  }
  __syncthreads();
  const int c8n = C >> 3;
  const long total = hw * c8n;
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < total; i += static_cast<long>(gridDim.x) * blockDim.x) {
    const int c8 = static_cast<int>(i % c8n);
    const long off = (static_cast<long>(n) * hw) * C + i * 8;
    float d[8];
    unpack8(*reinterpret_cast<const uint4*>(dout + off), d);
#pragma unroll
    for (int k = 0; k < 8; ++k) d[k] = d[k] * gate[c8 * 8 + k] + dmean[c8 * 8 + k];
    *reinterpret_cast<uint4*>(dres + off) = make_uint4(pack2(d[0], d[1]), pack2(d[2], d[3]), pack2(d[4], d[5]), pack2(d[6], d[7]));
  }
}

// nn.PixelUnshuffle(2), the adjoint of pixel_shuffle2_kernel: dst[n][y][x][4c + 2a + b] = src[n][2y+a][2x+b][c];
// src (N,2H,2W,C), dst (N,H,W,4C).  A thread gathers the 8 consecutive output channels of channels c8*2, c8*2+1 (all four
// phases) and stores them as one 16-byte vector.
__global__ void pixel_unshuffle2_kernel(const __nv_bfloat16* __restrict__ src, __nv_bfloat16* __restrict__ dst, int H, int W, int C, long total) {
  const int q8n = C >> 1;                                  // 16-byte groups per output pixel (4C channels / 8)
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < total; i += static_cast<long>(gridDim.x) * blockDim.x) {
    const int q = static_cast<int>(i % q8n);
    long r = i / q8n;
    const int x = static_cast<int>(r % W); r /= W;
    const int y = static_cast<int>(r % H);
    const long n = r / H;
    const __nv_bfloat16* s = src + ((n * 2 * H + 2 * y) * 2 * W + 2 * x) * static_cast<long>(C) + 2 * q;
    const long row = 2L * W * C;
    __nv_bfloat16 v[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int c = k >> 2, a = (k >> 1) & 1, b = k & 1;
      v[k] = s[a * row + b * C + c];
    }
    *reinterpret_cast<uint4*>(dst + i * 8) = *reinterpret_cast<const uint4*>(v);
  }
}

inline int grid_for(long total, int block, int cap = 148 * 8) {
  long g = (total + block - 1) / block;
  return static_cast<int>(g < 1 ? 1 : (g > cap ? cap : g));
}

}  // namespace

// the pooling launch of the forward (mul == nullptr) and of the backward (sum of src * mul)
static cudaError_t launch_pool(const void* src, const void* mul, int N, long hw, int C, float* pooled, cudaStream_t s) {
  cudaError_t e = cudaMemsetAsync(pooled, 0, static_cast<size_t>(N) * C * sizeof(float), s);
  if (e != cudaSuccess) return e;
  const int c8n = C >> 3;
  const int block = (256 / c8n > 0 ? 256 / c8n : 1) * c8n;
  const int lanes = block / c8n;
  int bx = static_cast<int>((hw + lanes * 8 - 1) / (lanes * 8));
  const int cap = (148 * 4 + N - 1) / N;
  bx = bx < 1 ? 1 : (bx > cap ? cap : bx);
  const auto* a = reinterpret_cast<const __nv_bfloat16*>(src);
  const auto* b = reinterpret_cast<const __nv_bfloat16*>(mul);
  if (mul) channel_pool_kernel<true><<<dim3(bx, N), block, lanes * C * sizeof(float), s>>>(a, b, hw, C, pooled);
  else channel_pool_kernel<false><<<dim3(bx, N), block, lanes * C * sizeof(float), s>>>(a, nullptr, hw, C, pooled);
  return cudaGetLastError();
}

cudaError_t launch_channel_pool(const void* src, int N, long hw, int C, float* pooled, cudaStream_t s) {
  return launch_pool(src, nullptr, N, hw, C, pooled, s);
}
cudaError_t launch_ca_scale_add(const void* res, const void* x, const float* pooled, const float* w1, const float* b1, const float* w2,
                                const float* b2, void* out, int N, long hw, int C, int Cr, cudaStream_t s) {
  int bx = static_cast<int>((hw * (C >> 3) + 256 * 4 - 1) / (256 * 4));
  const int cap = (148 * 4 + N - 1) / N;
  bx = bx < 1 ? 1 : (bx > cap ? cap : bx);
  ca_scale_add_kernel<<<dim3(bx, N), 256, (2 * C + Cr) * sizeof(float), s>>>(reinterpret_cast<const __nv_bfloat16*>(res),
                                                                             reinterpret_cast<const __nv_bfloat16*>(x), pooled, w1, b1, w2, b2,
                                                                             reinterpret_cast<__nv_bfloat16*>(out), hw, C, Cr);
  return cudaGetLastError();
}
cudaError_t launch_pixel_shuffle2(const void* src, void* dst, int N, int H, int W, int C, cudaStream_t s) {
  const long total = static_cast<long>(N) * 4 * H * W * (C >> 3);
  pixel_shuffle2_kernel<<<grid_for(total, 256), 256, 0, s>>>(reinterpret_cast<const __nv_bfloat16*>(src), reinterpret_cast<__nv_bfloat16*>(dst), H, W, C,
                                                            total);
  return cudaGetLastError();
}
cudaError_t launch_pixel_unshuffle2(const void* src, void* dst, int N, int H, int W, int C, cudaStream_t s) {
  const long total = static_cast<long>(N) * H * W * (C >> 1);
  pixel_unshuffle2_kernel<<<grid_for(total, 256), 256, 0, s>>>(reinterpret_cast<const __nv_bfloat16*>(src), reinterpret_cast<__nv_bfloat16*>(dst), H, W,
                                                              C, total);
  return cudaGetLastError();
}
cudaError_t launch_ca_backward(const void* dout, const void* res, const float* pooled, const float* w1, const float* b1, const float* w2,
                               const float* b2, void* dres, float* dw1, float* db1, float* dw2, float* db2, float* dot, int N, long hw, int C,
                               int Cr, cudaStream_t s) {
  cudaError_t e = launch_pool(dout, res, N, hw, C, dot, s);
  if (e != cudaSuccess) return e;
  int bx = static_cast<int>((hw * (C >> 3) + 256 * 4 - 1) / (256 * 4));
  const int cap = (148 * 4 + N - 1) / N;
  bx = bx < 1 ? 1 : (bx > cap ? cap : bx);
  ca_backward_kernel<<<dim3(bx, N), 256, (4 * C + 2 * Cr) * sizeof(float), s>>>(
      reinterpret_cast<const __nv_bfloat16*>(dout), reinterpret_cast<const __nv_bfloat16*>(res), pooled, dot, w1, b1, w2, b2,
      reinterpret_cast<__nv_bfloat16*>(dres), dw1, db1, dw2, db2, hw, C, Cr);
  return cudaGetLastError();
}

}  // namespace csr

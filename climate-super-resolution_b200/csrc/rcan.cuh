// Glue kernels of the RCAN generator (rcan.cu): launchers.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace csr {
// pooled (N, C) fp32 = per-image channel sums of src (N, hw, C) bf16 (zeroed here)
cudaError_t launch_channel_pool(const void* src, int N, long hw, int C, float* pooled, cudaStream_t s);
// out = res * sigmoid(w2 relu(w1 pooled/hw + b1) + b2) + x      (w1: (Cr, C), w2: (C, Cr))
cudaError_t launch_ca_scale_add(const void* res, const void* x, const float* pooled, const float* w1, const float* b1, const float* w2,
                                const float* b2, void* out, int N, long hw, int C, int Cr, cudaStream_t s);
// dst (N, 2H, 2W, C) = PixelShuffle(2) of src (N, H, W, 4C)
cudaError_t launch_pixel_shuffle2(const void* src, void* dst, int N, int H, int W, int C, cudaStream_t s);
// dst (N, H, W, 4C) = PixelUnshuffle(2) of src (N, 2H, 2W, C)
cudaError_t launch_pixel_unshuffle2(const void* src, void* dst, int N, int H, int W, int C, cudaStream_t s);
// backward of launch_ca_scale_add without the skip: dres = d/dres, parameter gradients accumulated (+=); dot: N*C floats of scratch
cudaError_t launch_ca_backward(const void* dout, const void* res, const float* pooled, const float* w1, const float* b1, const float* w2,
                               const float* b2, void* dres, float* dw1, float* db1, float* dw2, float* db2, float* dot, int N, long hw, int C,
                               int Cr, cudaStream_t s);
}  // namespace csr

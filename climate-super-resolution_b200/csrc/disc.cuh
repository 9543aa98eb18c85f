// Glue kernels of the discriminator path (disc.cu): launchers.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace csr {

// A logical image inside an S-layout buffer (N, Hs, Ws, C) bf16: pixel (i, j) lives at (off + step*i, off + step*j).
struct DiscView {
  int Hs, Ws, C;
  int off, step;
  int Hl, Wl;
};

cudaError_t launch_disc_gather(const void* src, const DiscView& v, int N, void* dst, int pad, const float* scale, const float* shift, cudaStream_t s);
cudaError_t launch_disc_collect(const void* dP, const DiscView& v, int N, int pad, const void* act, float gate_neg, void* g, cudaStream_t s);
cudaError_t launch_disc_bn_stats(const void* src, const DiscView& v, int N, double* sums, cudaStream_t s);
cudaError_t launch_disc_bn_finalize(const double* sums, const void* src, const DiscView& v, double count, const float* gamma, const float* beta, float eps, float momentum,
                                    float* running_mean, float* running_var, float* scale, float* shift, float* mean, float* invstd, cudaStream_t s);
cudaError_t launch_disc_bn_eval(int C, const float* gamma, const float* beta, float eps, const float* running_mean, const float* running_var,
                                float* scale, float* shift, cudaStream_t s);
cudaError_t launch_disc_bn_backward(const void* dP, const DiscView& v, int N, int pad, const void* act, float gate_neg, const float* gamma,
                                    const float* mean, const float* invstd, float* dy, double* sums, void* g, float* dgamma, float* dbeta,
                                    cudaStream_t s);
cudaError_t launch_disc_flatten(const void* src, const DiscView& v, int N, float* feats, cudaStream_t s);
cudaError_t launch_disc_unflatten(const float* gfeat, const DiscView& v, int N, void* g, cudaStream_t s);
cudaError_t launch_linear_forward(const float* x, const float* W, const float* b, float* y, int N, int K, int J, cudaStream_t s);
cudaError_t launch_linear_backward(const float* x, const float* W, const float* gy, float* dx, float* dW, float* db, int N, int K, int J, cudaStream_t s);

}  // namespace csr

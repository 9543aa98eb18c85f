#pragma once
#include <cuda_runtime.h>

namespace csr {
// one layer part of a batched weight pack (see pack_weight_kernel for the field meanings)
struct PackJob {
  const float* w; const float* b; void* dst; float* bdst;
  int cout, cin, kh, kw, fold, phase, transposed; float wscale; int co_lo, npad, cin_pad;
  // block jobs (ci_n > 0): fill only the executed channel block [ci_lo, ci_lo+ci_n) from a source tensor of shape
  // (ci_n, src_cin, kh, kw) whose input channels are offset by src_ci_off.  transposed: the block is a range of executed
  // INPUT channels (dense-block backward); otherwise a range of executed OUTPUT channels (dense-block forward regrouped by
  // source: several layers' filters over the same input side by side), the bias segment included.
  int ci_lo, ci_n, src_ci_off, src_cin;
};
cudaError_t launch_pack_jobs(const PackJob* jobs_dev, int njobs, cudaStream_t s);
cudaError_t launch_pack_weight(const float* w, void* dst, int cout, int cin, int kh, int kw, int fold, int phase, int transposed,
                               float wscale, int co_lo, int npad, int cin_pad, cudaStream_t s);
cudaError_t launch_pack_bias(const float* b, float* dst, int cout, int co_lo, int npad, cudaStream_t s);
cudaError_t launch_nchw_to_nhwc(const float* src, void* dst, int n, int c, int h, int w, int dst_c, int zero_to, cudaStream_t s);
// hi/lo bf16 activations of the perceptual loss (CSR_OUT_BF16_SPLIT): input conversion and 2x2 max pool
cudaError_t launch_nchw_to_nhwc_split(const float* src, void* dst, int n, int c, int h, int w, int dst_c, cudaStream_t s);
cudaError_t launch_maxpool2x2_split(const void* src, void* dst, int n, int h, int w, int c, cudaStream_t s);
cudaError_t launch_pack_srcnn_in(const float* t, const float* elev, const float* mask, void* dst, int W, long total_pix, int dst_c,
                                 cudaStream_t s);
cudaError_t launch_nhwc_to_nchw(const void* src, float* dst, int n, int c, int h, int w, int src_c, int src_coff, cudaStream_t s);
cudaError_t launch_wgrad_reduce(float* dacc, long part_stride, int n_parts, long nfloats, cudaStream_t s);
cudaError_t launch_wgrad_scatter(const float* dacc, int ld_n, float* dw, int cout, int cin, int kh, int kw, int fold,
                                 int phase, int ci0, int ci_n, int col0, float scale, int taps_t, cudaStream_t s);
cudaError_t launch_wgrad_scatter_jobs(const float* dacc, float* dw, int cout, int cin, int kh, int kw, int n_cols, int jobs_co, int jobs_dy,
                                      int per_dy, long job_stride, float scale, cudaStream_t s);
// db: nseg (1..4) bias-gradient vectors; channel co of the cout channels goes to db[co / (cout/nseg)]
cudaError_t launch_bias_grad(const void* g, long npix, int C, int coff, int cout, float scale, float* const* db, int nseg, cudaStream_t s);
cudaError_t launch_bias_grad_wide(const void* g, long npix, int C, int coff, int chunks, float scale, float* db, cudaStream_t s);
cudaError_t launch_tap_pack(const float* taps, long plane, const float* bias, const float* elev, const float* mask, void* dst, int N, int H, int W,
                            cudaStream_t s);
cudaError_t launch_tap_sum(const float* taps, long plane, const float* bias, float* out, int H, int W, long total, cudaStream_t s);
cudaError_t launch_bias_grad_planar(const float* g, long n, float scale, float* db, cudaStream_t s);
cudaError_t launch_scale_copy64(const void* src, int src_C, void* dst, int dst_C, long npix, float scale, cudaStream_t s);
// bf16 wire format of the data-parallel gradient exchange: comm = bf16(scale * flat) / flat = scale * float(comm)
cudaError_t launch_grad_pack_bf16(const float* flat, void* comm, long n, float scale, int max_blocks, cudaStream_t s);
cudaError_t launch_grad_unpack_bf16(const void* comm, float* flat, long n, float scale, int max_blocks, cudaStream_t s);
cudaError_t launch_gcol_pack(const void* src, int src_C, void* dst, int dst_C, int H, int W, long total_pix, int KH, int KW, cudaStream_t s);
// Min-max scaler around the inference hot path (normalization.py:37-84): float64 arithmetic, one rounding to float32.
// normalize: out[n][0] = nan_to(raw[n] * scale_n + min__n); channels 1.. = the shared (h,w) planes extra0 / extra1.
cudaError_t launch_minmax_normalize(const float* raw, int n, long hw, const double* mn, const double* mx, double a, double b, double eps,
                                    float nan_sub, const float* extra0, const float* extra1, float* out, cudaStream_t s);
// denormalize + land mask: out = mask > 0 ? (sr - min__n) / scale_n : NaN.  mask_stride = 0 (one shared mask) or hw.
cudaError_t launch_minmax_denormalize_mask(const float* sr, const float* mask, long mask_stride, int n, long hw, const double* mn,
                                           const double* mx, double a, double b, double eps, float* out, cudaStream_t s);
// Training-sample assembly (climate_dataset.py:98-172): per-sample flip / rot90 of hr, elev, mask and x = [lr, elev_lr, mask_lr]
// with lr = nearest resize by `scale` (top-left pixel of each block).  codes: n device ints (bit0 v-flip, bit1 h-flip,
// bits 2-3 rot90 factor) or NULL; *_out may be NULL when codes is NULL.
cudaError_t launch_lr_input(const float* hr, const float* elev, const float* mask, int n, int H, int W, int scale, const int* codes,
                            float* hr_out, float* elev_out, float* mask_out, float* x_out, cudaStream_t s);
}  // namespace csr

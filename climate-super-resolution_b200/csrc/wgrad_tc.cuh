// Weight-gradient GEMM on tcgen05 tensor cores: parameters shared by kernel and host launcher.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace csr {

constexpr int kWgradThreads = 256;   // warp0 TMA producer, warp1 MMA issuer (+TMEM), warp2 halo-column zeroing, warps4-7 epilogue

// One launch accumulates, for n_dy vertical taps (row offsets dy_off + dyi) and all KW horizontal taps,
//   D[dyi][dx][ci][co] += sum over pixels p of  x[p + (dy_off + dyi, dx - PW)][ci] * g[p][co]
// with ci over n_xbox*64 input channels (UMMA M = 64 or 128) and co over up to two 64-channel boxes of output gradients
// (UMMA N = n_cols).  K = pixels: both operands are MN-major (channels contiguous per pixel), exactly as TMA lands NHWC.
struct WgradParams {
  int N, H, W;
  int KW, PW, dy_off, n_dy;   // taps (dy_off + dyi, dx - PW), dyi < n_dy, dx < KW
  int SW, sw_shift, TH, TW;
  int tiles_x, tiles_y, num_tiles, tiles_per_img;
  unsigned long long magic_img, magic_row;
  int n_xbox, n_gbox;        // 64-channel boxes per operand (1 or 2)
  int M;                     // 64 * n_xbox
  int n_cols;                // UMMA N: g channels used, multiple of 16 (<= 128)
  int x_box_bytes, g_box_bytes;   // one 64-channel box: (TH+n_dy)*SW*128 and TH*SW*128
  int x_slack;               // zeroed bytes in front of each x box (negative flattened tap shifts read there)
  int stage_bytes, n_stages;
  int tmem_cols;
  int xc0[2], gc0[2];        // first channel of each box inside its buffer
  float* dacc;               // this launch's first tap inside part 0: fp32 [n_parts (stride part_stride)][n_dy*KW][128][ld_n]
  long part_stride;          // floats between the partial-sum slices of consecutive CTAs (all taps of the layer)
  int n_parts;               // grid size = min(num_tiles, SMs)
  int ld_n;
  int atomic;                // 1: every CTA adds its sums into part 0 with red.global.add.v4.f32 (the host zeroes it first) instead of
                             //    storing a private partial slice that a reduce kernel would have to read back
  // Job mode (jobs_ci > 0; layers with many channels and few pixels - the discriminator): the grid is NOT split over pixels only.
  // CTA b works on job b / splits = (ci chunk of 128, co chunk of n_cols, group of per_dy vertical taps) and, within the job, on
  // every splits-th pixel tile; it adds its sums into the job's own block dacc + job * job_stride ([per_dy*KW][128][n_cols]).
  // One launch then covers a whole layer (a 512 -> 512 conv: 4 x 4 x 3 jobs) instead of one launch per (chunk, chunk, tap).
  int jobs_ci, jobs_co, jobs_dy, splits;
  int KH, PH, per_dy;
  int x_coff, g_coff;        // first channel of the layer's input / output gradient inside their buffers
  long job_stride;
};

int launch_wgrad_tc(const WgradParams& p, const CUtensorMap& tx0, const CUtensorMap& tx1, const CUtensorMap& tg0, const CUtensorMap& tg1,
                    int num_sms, cudaStream_t stream);
size_t wgrad_smem_bytes(const WgradParams& p);

}  // namespace csr

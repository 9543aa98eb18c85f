// Dense-block kernel: conv1..conv4 of a ResidualDenseBlock (climsr/models/esrgan.py:33-36) as ONE persistent launch with
// tile-level dependencies between the layers instead of four grid-wide ones.  Parameters shared by kernel and host.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace csr {

constexpr int kDenseMaxLayers = 4;

struct DenseLayerParams {
  int ksteps;        // input channels / 16 (the layer reads channels [0, 16 * ksteps) of the concat buffer)
  int n_kblocks;     // ceil(ksteps / 4): 64-channel window boxes per tile
  int w_bytes;       // packed weights: 3 * ksteps * 3 * 16 * 32
  int out_coff;      // first output channel inside the concat buffer (nf + (k-1) * gc)
  const void* wpk;   // packed bf16 weights (global), conv_tc layout [kblock][dy][kstep][3*16 rows x 16 K]
  const float* bias; // [16] fp32
  int gate_coff;     // backward form: first channel of this layer's gate inside the gate buffer
};

struct DenseParams {
  int N, H, W;
  int SW, sw_shift, TH, TW;                       // window pitch, rows per M tile, output columns per tile (SW - 2)
  int tiles_x, tiles_y, num_tiles, tiles_per_img; // in WINDOWS of two vertically adjacent M tiles (2*TH output rows)
  unsigned long long magic_img, magic_row;        // floor(2^40/d)+1 for d = tiles_per_img, tiles_x
  int win_bytes;     // (2*TH + 2) * SW * 128
  int slot_bytes;    // win_bytes rounded up to 1024
  int n_slots;
  int stage_bytes;   // one staging buffer per epilogue group: TH*TW*32 rounded up to 1024
  int wbuf_bytes;    // one of the two weight buffers (largest layer, rounded up to 1024)
  int n_layers;      // 1..4
  int C;             // channel pitch of the concat buffer
  void* buf;         // the concat buffer: read (channels [0, 16*ksteps)) and written (out_coff) by every layer
  unsigned int* flags;   // [n_layers][num_tiles], zero before the launch: M tiles of (layer, window) whose outputs are in memory
  int use_pdl;
  // forward: act = 1 (LeakyReLU 0.2), gate = nullptr.  Backward (the four gated input-gradient convs of a dense block, bwd_build in
  // api.cu): act = 0 and v *= (gate > 0 ? 1 : gate_neg) with gate = the saved forward activation of the layer whose gradient this is
  int act;
  const void* gate;  // bf16 NHWC, pitch gate_C
  int gate_C;
  float gate_neg;
  unsigned long long* timeline;   // debug: see ConvParams::timeline
  int launch_id;
  DenseLayerParams L[kDenseMaxLayers];
};

size_t dense_smem_bytes(const DenseParams& p);
// tmap: 4-D (C, W, H, N) bf16 map of the concat buffer, box (64, SW, 2*TH+2, 1), SWIZZLE_128B, zero fill.  Returns cudaError_t.
int launch_dense_block(const DenseParams& p, const CUtensorMap& tmap, int num_sms, cudaStream_t stream);

}  // namespace csr

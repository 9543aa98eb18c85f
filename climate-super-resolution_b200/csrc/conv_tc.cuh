// Implicit-GEMM convolution on tcgen05 tensor cores: parameters shared by kernel and host launcher.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace csr {

constexpr int kEpilogueWarps = 16;    // four warps per TMEM lane quadrant, each owning every 4th 8-channel chunk
constexpr int kEpilogueThreads = kEpilogueWarps * 32;
constexpr int kMmaWarps = 2;          // MMA issuer warps taking alternate tiles
constexpr int kConvThreads = 32 * (1 + kMmaWarps) + kEpilogueThreads;   // warp0 TMA producer, warps 1-2 MMA issuers, then epilogue
constexpr int kTileM = 128;           // window positions (UMMA M) per tile = TH * SW
constexpr int kSmemLimit = 232448;    // 227 KB opt-in dynamic shared memory per CTA on sm_100
constexpr int kMaxNpad = 64;          // output channels per launch part (epilogue: <= 2 chunks of 8 per warp)

enum StoreMode {
  kStoreStaged = 0,     // bf16 NHWC through a swizzled shared-memory staging tile, copied out as whole pixel rows
  kStoreDirect = 1,     // bf16 NHWC, per-element global stores (ragged channel counts)
  kStoreF32Planar = 2,  // fp32 (N,1,H,W), channel 0 only
  kStoreF32Nhwc = 3,    // fp32 NHWC (n_store channels per pixel, pitch out_C): gradient / debug outputs
  kStoreBf16Split = 4   // staged like kStoreStaged, as a hi/lo bf16 pair: hi = bf16(v) at channel c, lo = bf16(v - hi) at channel
                        // split_off + c (VGG features of the perceptual loss: the pair carries v to fp32 precision)
};

struct ConvParams {
  // geometry (input spatial == conv output spatial; stride 1).  Output pixel (y,x) = sum over taps (dy,dx) of
  // input pixel (y + dy - PH, x + dx - PW); PH/PW need not be (K-1)/2 (sub-pixel phases of nearest-x2 + conv).
  int N, H, W;
  int KH, KW, PH, PW;
  int cin_off;     // first input channel inside the input buffer (multiple of 8)
  int cin;         // input channels used, padded to a multiple of 16 (k-steps = cin/16)
  int npad;        // output channels of this launch padded to a multiple of 16 (<= kMaxNpad); UMMA N = KW * npad
  int n_store;     // real output channels
  // tiling: a tile is TH rows x SW window columns of which TW = SW-(KW-1) are real outputs (columns [PW, PW+TW))
  int SW, sw_shift, TH, TW;
  int tiles_x, tiles_y, num_tiles, tiles_per_img;
  unsigned long long magic_img, magic_row;   // floor(2^40/d)+1 for d = tiles_per_img, tiles_x (num_tiles < 2^24)
  int win_rows;    // TH + KH - 1
  int win_bytes;   // win_rows * SW * 128  (== TMA box bytes per 64-channel k-block)
  int slot_bytes;  // win_bytes rounded up to 1024
  int n_kblocks;   // ceil(cin / 64)
  int n_slots;     // activation-window ring depth
  int w_bytes;     // packed weights: KH * (cin/16) * KW * npad * 32
  int n_acc;       // accumulator buffers in TMEM (2, 4 or 8); n_acc * KW * npad <= 512
  int n_groups;    // epilogue warp groups (1, 2 or 4; n_groups divides n_acc): one staging buffer each
  int n_stage;     // staging buffers in shared memory: n_groups, or 2 for the early-release epilogue
  int hyb;         // 1 = hybrid tap fold (conv_tc.cu HYB_T): 3x3 early-release layers, accumulators of 2*npad columns
  int early;       // 1 = early-release epilogue (conv_tc.cu, EARLY_T): wide residual-free layers, one 16-warp group
  int tmem_cols;   // power of two >= max(32, n_acc*KW*npad)
  int trace_cta;   // debug: the CTA whose role timestamps go to `trace`
  int box_c;       // channels per window pixel in shared memory: 64 (128-byte rows), or 32 / 16 for single-k-block layers with cin <= 32 / 16
  int tall_shift;  // 1: a window holds TWO vertically adjacent M tiles (2*TH + KH - 1 rows, one TMA load, one MMA-issuer iteration,
                   //    two accumulator buffers): halves the per-tile control cost of thin layers; needs n_acc == 4.  tiles_* / num_tiles
                   //    then count windows.  0: one M tile per window
  int stream_w;    // 1: the layer's weights do NOT stay resident (layers with >= 256 input channels: > 150 KB per 64 output channels): every
                   //    window slot also receives the packed weights of its 64-channel k-block (wkb_bytes, at offset win_slot_bytes)
  int wkb_bytes;   // packed weights of one full k-block: KH * 4 * KW * npad * 32
  int win_slot_bytes;
  int use_pdl;     // launch with programmatic stream serialization (prologue overlaps the previous kernel's tail)
  // Output-channel parts of ONE layer as one launch (gridDim.y = parts): every part has this launch's geometry and reads the same input;
  // part k takes its weights at wpk + k*part_w_bytes, its bias at bias + k*part_b_floats and writes output channels out_coff + k*part_c.
  // Used for the wide single-op layers (discriminator: 128..512 output channels over small maps), where one part per launch leaves most
  // SMs idle.  Residual / gate operands are not offset: only residual-free launches are merged.  0 / 1 = a single part.
  int parts, part_w_bytes, part_b_floats, part_c;
  int part_ph, part_oy;   // ... and PH + k*part_ph, out_oy + k*part_oy (sub-pixel phase pairs of nearest-x2 + conv as one launch)
  // Fused 1x1 successor (conv_tc.cu FUSE_T; early-release epilogue, KW = 1, 64 staged channels): out2[.., out2_coff + j] =
  // relu(b2[j] + sum_c w2[j][c] * act(this layer)[c]) for j < n2 (multiple of 8, <= 32); `out` is NOT written.
  int fuse2, w2_bytes, n2;
  const void* w2;      // packed like a 1x1 layer with cin = 64, npad = 32: four k-step blocks of 32 rows x 16 K
  const float* b2;
  void* out2; int out2_C, out2_coff;
  // fuse2 == 2: the successor is a 3x3 -> 1 conv seen as nine 1x1 'tap' channels (n2 = 9): fp32 tap planes out2[tap * out2_plane + pixel]
  long long out2_plane;
  // epilogue:  v = act(acc + bias);  if r1: v = v*s1 + r1;  if r2: v = v*s2 + r2;  if gate: v *= (gate > 0 ? 1 : gate_neg)
  const float* bias;   // [npad] fp32 (zero padded)
  const void* wpk;     // packed bf16 weights (global), layout [kblock][dy][kstep in kblock][KW*npad/8][2][8][8]
  int act;             // 0 none, 1 leaky-relu 0.2, 2 relu, 4 leaky-relu(act_slope)
  float act_slope;     // act == 4: LeakyReLU negative slope
  float s1, s2;
  const void* r1; int r1_C, r1_coff;
  const void* r2; int r2_C, r2_coff;
  const void* gate; int gate_C, gate_coff; int gate_from; float gate_neg;   // applied to output channels >= gate_from
  void* out; int out_C, out_coff;
  int store_mode;      // StoreMode
  void* out_dup; int dup_C, dup_coff;   // early-release plain 3x3 layer (conv_first): second copy of the output (same pixels, own channel pitch)
  int out_sy, out_sx, out_oy, out_ox;   // conv-output pixel (y,x) lives at buffer pixel (y*out_sy+out_oy, x*out_sx+out_ox)
  int out_H, out_W;                     // spatial size of the output buffer
  int stage_row_bytes; // kStoreStaged: bytes per staged pixel (n_store * 2: 16..128)
  int stage_bytes;     // one staging buffer (TH*TW*stage_row_bytes rounded up to 1024; twice that for kStoreBf16Split)
  int stage_lo_bytes;  // kStoreBf16Split: offset of the lo tile inside a staging buffer (the hi tile is at 0)
  int split_off;       // kStoreBf16Split: channel distance between a hi value and its lo (the layer's total output channels)
  long long* trace;    // debug: per-role clock64 timestamps of CTA 0 (nullptr = off), [3 roles][64 tiles][4 events]
  unsigned long long* timeline;   // debug (csr_debug_set_timeline): [2*launch_id] = earliest CTA start after griddepcontrol.wait,
  int launch_id;                  // [2*launch_id + 1] = latest CTA end, in globaltimer ns - the in-situ timeline of a forward
};

// Returns cudaError_t (as int).
//   tmap_in : 4-D (C, W, H, N) bf16 map, box (64, SW, win_rows, 1), SWIZZLE_128B, zero OOB fill (= the conv padding)
size_t conv_smem_bytes(const ConvParams& p);
int launch_conv_tc(const ConvParams& p, const CUtensorMap& tmap_in, int num_sms, cudaStream_t stream);

}  // namespace csr

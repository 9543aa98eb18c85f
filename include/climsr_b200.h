/*
 * climsr_b200.h - C-ABI of the B200-native (sm_100a) generator hot path of
 * xultaeculcis/climate-super-resolution.
 *
 * Plain C: pointers, sizes and ints only.  All data pointers are DEVICE pointers
 * unless a parameter says "host".  `stream` is a cudaStream_t passed as void*.
 * Every function returns CSR_OK (0) or a negative CsrStatus and never throws or
 * synchronises the device (work is enqueued on `stream`); csr_last_error() gives
 * the message of the last failure on the calling thread.  There is NO CPU
 * fallback: on a machine without an sm_100 device every compute entry point
 * returns CSR_ERR_CUDA / CSR_ERR_UNSUPPORTED.
 *
 * Reference interfaces replaced (paths relative to the reference repo):
 *   csr_plan_forward / csr_generator_forward
 *        <- ESRGANGenerator.forward(x, elev, mask)           climsr/models/esrgan.py:89-102
 *           (+ RDB / RRDB / SRCNN forwards                    esrgan.py:32-38,50-54; srcnn.py:13-18)
 *           called from TaskSuperResolutionModule.forward     climsr/core/task.py:235-239
 *           and inference_on_full_images                      climsr/inference/inference.py:70
 *   csr_pack_weights
 *        <- the generator state_dict (names/shapes/order)     esrgan.py:72-87, srcnn.py:9-11
 *   csr_conv2d_nhwc
 *        <- one nn.Conv2d + LeakyReLU/ReLU/residual call site esrgan.py:33-38,90-100
 *   csr_masked_metrics
 *        <- common_val_test_step + compute_metrics            climsr/core/task.py:262-300,342-380
 *           RegressionAccuracy.update/compute                 climsr/metrics/regression_accuracy.py:15-22
 *           MinMaxScaler._denormalize / StandardScaler        climsr/data/normalization.py:63-84,115
 *   csr_l1_loss / csr_mse_loss (+ _backward)
 *        <- self.loss(sr, hr)                                 climsr/core/task.py:141;
 *                                                             climsr/task/pl_generator_pre_training.py:29-30
 */
#ifndef CLIMSR_B200_H
#define CLIMSR_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CSR_ABI_VERSION 2

typedef enum CsrStatus {
  CSR_OK = 0,
  CSR_ERR_BAD_ARG = -1,      /* null pointer, non-positive size, misaligned pointer            */
  CSR_ERR_UNSUPPORTED = -2,  /* shape/config outside what the kernels implement                 */
  CSR_ERR_CUDA = -3,         /* CUDA runtime/driver error (launch failure, no sm_100 device...) */
  CSR_ERR_WORKSPACE = -4     /* workspace / packed buffer too small                             */
} CsrStatus;

/* ESRGANGenerator.__init__ arguments (esrgan.py:58-67).  out_channels must be 1 (the SRCNN tail
 * hard-wires 1+1+1 input channels, esrgan.py:87,100); scale must be 4 (conf/generator/esrgan.yaml). */
typedef struct CsrNetDesc {
  int32_t in_channels;
  int32_t out_channels;
  int32_t nf;
  int32_t nb;
  int32_t gc;
  int32_t scale;
} CsrNetDesc;

/* Epilogue of a single convolution (csr_conv2d_nhwc). */
typedef enum CsrAct { CSR_ACT_NONE = 0, CSR_ACT_LRELU02 = 1, CSR_ACT_RELU = 2,
                      CSR_ACT_LRELU = 4 /* LeakyReLU(CsrConvDesc::act_slope): the discriminator's 0.01 */ } CsrAct;
typedef enum CsrOutMode {
  CSR_OUT_BF16_NHWC = 0,     /* bf16, channel slice [out_coff, out_coff+cout) of an NHWC buffer          */
  CSR_OUT_F32_PLANAR = 2,    /* fp32 (N,1,H,W); cout must be 1                                            */
  CSR_OUT_F32_NHWC = 3,      /* fp32 NHWC, channel slice [out_coff, out_coff+cout) (gradients, debugging) */
  CSR_OUT_BF16_SPLIT = 4     /* hi/lo bf16 pair of every output value v: hi = bf16(v) at channel out_coff + c, lo = bf16(v - hi)
                                at channel out_coff + cout + c (hi + lo carries v to ~2^-16 relative).  A following conv over the
                                2*cout channels with weights [W | W] computes W (hi + lo) in fp32.  3x3 convs with CSR_ACT_RELU and
                                no residual / gate only; cout % 8 == 0, out_c >= out_coff + 2*cout.  (The VGG19 perceptual loss.) */
} CsrOutMode;

typedef struct CsrConvDesc {
  int32_t n, h, w;            /* input batch / height / width (output is 2h x 2w when in_up2, else h x w)  */
  int32_t cin, cout;          /* real channel counts of the conv being executed                            */
  int32_t kh, kw;             /* odd kernel size; stride 1, padding (k-1)/2 ("same")                       */
  int32_t in_c, in_coff;      /* channels per pixel of the input buffer, first input channel (multiples of 8) */
  int32_t out_c, out_coff;    /* channels per pixel of the output buffer, first output channel             */
  int32_t act;                /* CsrAct                                                                    */
  int32_t out_mode;           /* CsrOutMode                                                                */
  int32_t in_up2;             /* 1: F.interpolate(scale_factor=2, mode="nearest") is applied to the input first
                                 (esrgan.py:94,97); executed as four 2x2 sub-pixel convs on the (h,w) input   */
  int32_t transposed;         /* 1: weight is the FORWARD layer's (cin_fwd=cout, cout_fwd=cin) OIHW tensor and the
                                 conv computed is its input gradient (flipped taps, swapped channel roles)    */
  float   scale1;             /* v = act(conv+bias); if res1: v = v*scale1 + res1; if res2: v = v*scale2+res2;
                                 if gate: v *= (gate > 0 ? 1 : gate_neg) for output channels >= gate_from      */
  float   scale2;
  int32_t res1_c, res1_coff;  /* residual buffers: bf16 NHWC with res*_c channels per pixel                */
  int32_t res2_c, res2_coff;
  int32_t gate_c, gate_coff, gate_from;   /* gate buffer: bf16 NHWC (saved forward activations)            */
  float   gate_neg;
  float   act_slope;          /* negative slope when act == CSR_ACT_LRELU                                   */
} CsrConvDesc;

/* ---- library ------------------------------------------------------------------------------- */
int         csr_abi_version(void);
const char* csr_last_error(void);
/* 0 when an sm_100 device is current and usable, CSR_ERR_CUDA / CSR_ERR_UNSUPPORTED otherwise. */
int         csr_device_check(void);
/* debug / tuning knobs (key, value); unknown keys return CSR_ERR_BAD_ARG. */
int         csr_set_option(int32_t key, int32_t value);
int64_t     csr_kernel_launch_count(void);           /* kernels launched by this library so far   */
/* debug: device buffer of 3*64*8 int64 receiving per-role clock64 timestamps of CTA 0 for convs built afterwards
 * (NULL switches tracing off).  Layout [role: producer, mma, epilogue][tile 0..63][event 0..7].                   */
int         csr_has_experiments(void);   /* always 0: the measured-and-rejected kernel variants were removed; kept so that ABI version 2 stays intact */
int         csr_debug_set_trace(void* device_buffer);
/* debug: in-situ timeline of the launches of csr_plan_forward (direct launches, no graph replay).  device_u64: 2 * capacity
 * uint64 in device memory, even entries preset to ~0, odd entries to 0; launch i then leaves [2i] = earliest CTA start after
 * its dependency wait and [2i+1] = latest CTA end, in globaltimer nanoseconds.  NULL switches it off. */
int         csr_debug_set_timeline(void* device_u64, int32_t capacity_launches);

/* ---- weights --------------------------------------------------------------------------------
 * Number of conv layers (== number of weight tensors) of the generator, in state_dict order.    */
int     csr_num_layers(const CsrNetDesc* net);
/* Shape of layer i as (cout, cin, kh, kw); name is written into name[name_cap] (state_dict prefix). */
int     csr_layer_shape(const CsrNetDesc* net, int32_t i, int32_t shape4[4], char* name, size_t name_cap);
size_t  csr_packed_weight_bytes(const CsrNetDesc* net);
/* w/b: HOST arrays of csr_num_layers() DEVICE pointers to fp32 OIHW weights / biases.           */
int     csr_pack_weights(const CsrNetDesc* net, const float* const* w, const float* const* b,
                         void* packed, size_t packed_bytes, void* stream);

/* ---- generator forward ----------------------------------------------------------------------
 * x (N,Cin,h,w) fp32 NCHW; elev, mask (N,1,4h,4w) fp32; out (N,1,4h,4w) fp32.                    */
size_t  csr_workspace_bytes(const CsrNetDesc* net, int32_t n, int32_t h, int32_t w);
typedef struct CsrPlan CsrPlan;
int     csr_plan_create(const CsrNetDesc* net, int32_t n, int32_t h, int32_t w,
                        void* workspace, size_t workspace_bytes, CsrPlan** plan);
int     csr_plan_forward(CsrPlan* plan, const void* packed, const float* x, const float* elev,
                         const float* mask, float* out, void* stream);
/* launches of one forward: what a forward without graph replay adds to csr_kernel_launch_count */
int     csr_plan_num_launches(const CsrPlan* plan);
void    csr_plan_destroy(CsrPlan* plan);
/* one-shot convenience: plan_create + plan_forward + plan_destroy                               */
int     csr_generator_forward(const CsrNetDesc* net, const void* packed, const float* x,
                              const float* elev, const float* mask, float* out,
                              void* workspace, size_t workspace_bytes,
                              int32_t n, int32_t h, int32_t w, void* stream);

/* ---- generator training step -------------------------------------------------------------------
 * A training plan keeps every dense block's concat buffer and the HR-tail activations (the saved state autograd would
 * keep).  csr_plan_forward works on it unchanged; csr_plan_backward then ACCUMULATES (+=) d loss / d weight and
 * d loss / d bias of every conv layer into dw[i] / db[i] (HOST arrays of csr_num_layers() DEVICE pointers, fp32, the
 * parameters' OIHW / (cout) shapes) given grad_out = d loss / d out, fp32 (N,1,4h,4w).  A null dw[i] / db[i] returns
 * CSR_ERR_BAD_ARG before anything is launched.
 * csr_plan_forward and csr_plan_backward_flat may be called on a stream the caller is capturing (after one call outside
 * the capture): their launches then go into the caller's graph and the plan's own graph cache is left as it was.
 * <- autograd backward of ESRGANGenerator.forward (esrgan.py:89-102), invoked by Lightning's loss.backward().       */
size_t  csr_train_workspace_bytes(const CsrNetDesc* net, int32_t n, int32_t h, int32_t w);
int     csr_train_plan_create(const CsrNetDesc* net, int32_t n, int32_t h, int32_t w,
                              void* workspace, size_t workspace_bytes, CsrPlan** plan);
size_t  csr_packed_weight_bytes_bwd(const CsrNetDesc* net);
/* transposed / flipped bf16 weight tiles of the input-gradient convolutions (w as for csr_pack_weights)           */
int     csr_pack_weights_bwd(const CsrNetDesc* net, const float* const* w, void* packed, size_t packed_bytes, void* stream);
int     csr_plan_backward(CsrPlan* plan, const void* packed_bwd, const float* grad_out,
                          float* const* dw, float* const* db, void* stream);
/* test hook: byte offset (inside the workspace given to csr_*plan_create) and dims {n, h, w, channel pitch} of a bf16 NHWC activation
 * buffer of the plan.  kind 0: concat buffer `index` ([x | x1..x4]; one per dense block in training plans), 1: upconv1 output,
 * 2: upconv2 output, 3: HRconv output, 4: srcnn.conv1 output, 5: srcnn.conv2 output.  The parity tests read the activation SIGNS of a
 * training forward from these to run the fp32 oracle with the same LeakyReLU / ReLU masks. */
int     csr_plan_buffer(const CsrPlan* plan, int32_t kind, int32_t index, size_t* offset_bytes, int32_t dims4[4]);
int     csr_plan_num_backward_ops(const CsrPlan* plan);
/* Same backward, all gradients in ONE flat fp32 buffer (OVERWRITTEN, not accumulated): layer i's dW at float offset
 * csr_plan_grad_offset(plan, i, 0), its db at csr_plan_grad_offset(plan, i, 1) (every tensor starts 16-byte aligned),
 * csr_plan_grad_floats() floats in total.  With stable buffers the ~800 launches of a step replay as one CUDA graph.   */
size_t  csr_plan_grad_floats(const CsrPlan* plan);
/* 1 = the plan's forward (backward != 0: backward_flat) launch sequence is being replayed as a CUDA graph, 0 = not (yet),
 * -1 = capture failed and the plan launches directly.                                                              */
int     csr_plan_graph_status(const CsrPlan* plan, int32_t backward);
int     csr_plan_grad_offset(const CsrPlan* plan, int32_t layer, int32_t is_bias, size_t* offset);
int     csr_plan_backward_flat(CsrPlan* plan, const void* packed_bwd, const float* grad_out, float* flat_grads, void* stream);
/* Segmented form for overlapping the data-parallel gradient exchange with the rest of backward: split the op list into
 * (at most) nseg segments (returns the number made); segment k, run in order 0..n-1, completes the flat gradient floats
 * [*lo, *hi) - a suffix of the buffer that grows downwards, because layers finish in reverse order - and copies exactly
 * that range into flat_grads, so the caller can all-reduce it on another stream while later segments compute.       */
int     csr_plan_backward_segments(CsrPlan* plan, int32_t nseg);
int     csr_plan_backward_flat_seg(CsrPlan* plan, const void* packed_bwd, const float* grad_out, float* flat_grads,
                                   int32_t seg, size_t* lo, size_t* hi, void* stream);

/* ---- single convolution (building block of the discriminator path; used by the parity tests) --------------
 * in: bf16 NHWC (n,h,w,in_c); weight fp32 OIHW (cout,cin,kh,kw); bias fp32 (cout) or NULL (= zeros).
 * scratch: >= csr_conv2d_scratch_bytes() device bytes for the packed weights.  weight == NULL: `scratch` still holds the
 * packed weights (and bias) of an earlier call for the same layer - callers cache it per weight version.              */
size_t  csr_conv2d_scratch_bytes(const CsrConvDesc* d);
/* Pack only: fills `scratch` for later csr_conv2d_nhwc(..., weight = NULL, ...) calls of the same layer shape.  The pack launch
 * reads a job table through a pageable host copy, so it cannot be stream-captured; the conv launches themselves can: callers
 * that replay the layer inside a CUDA graph (the discriminator) pack outside of it with this call.                      */
int     csr_conv2d_pack(const CsrConvDesc* d, const float* weight, const float* bias, void* scratch, size_t scratch_bytes, void* stream);
int     csr_conv2d_nhwc(const CsrConvDesc* d, const void* in, const float* weight, const float* bias,
                        void* out, const void* res1, const void* res2, const void* gate,
                        void* scratch, size_t scratch_bytes, void* stream);

/* ---- single-layer weight gradient (building block of csr_plan_backward; used by the parity tests) ---
 * dw (cout,cin,kh,kw) += scale * d/dW of conv2d(x, W) against the output gradient g;  db (cout) += scale * sum(g).
 * x: bf16 NHWC (n,h,w,x_c), input channels [x_coff, x_coff+cin);  g: bf16 NHWC gradient w.r.t. the conv output,
 * channels [g_coff, g_coff+cout), spatial (h,w) - or (2h,2w) when in_up2 (nearest-x2 applied to x first).
 * <- autograd of nn.Conv2d (convolution_backward, weight part) at every call site of esrgan.py:33-38,90-100.      */
typedef struct CsrWgradDesc {
  int32_t n, h, w;
  int32_t cin, cout, kh, kw;
  int32_t x_c, x_coff;
  int32_t g_c, g_coff;
  int32_t in_up2;
  float   scale;
} CsrWgradDesc;
size_t  csr_conv2d_wgrad_scratch_bytes(const CsrWgradDesc* d);
int     csr_conv2d_wgrad(const CsrWgradDesc* d, const void* x, const void* g, float* dw, float* db,
                         void* scratch, size_t scratch_bytes, void* stream);

/* ---- layout helpers -------------------------------------------------------------------------- */
/* fp32 NCHW (n,c,h,w) -> bf16 NHWC (n,h,w,dst_c) channels [0,c), channels [c, zero_to) zeroed.  */
int     csr_nchw_f32_to_nhwc_bf16(const float* src, void* dst, int32_t n, int32_t c, int32_t h, int32_t w,
                                  int32_t dst_c, int32_t zero_to, void* stream);
/* bf16 NHWC channel slice -> fp32 NCHW (n,c,h,w)                                                 */
int     csr_nhwc_bf16_to_nchw_f32(const void* src, float* dst, int32_t n, int32_t c, int32_t h, int32_t w,
                                  int32_t src_c, int32_t src_coff, void* stream);

/* ---- hi/lo bf16 activations (VGG19 perceptual loss; see CSR_OUT_BF16_SPLIT) ---------------------------------------
 * A value v is held as the pair hi = bf16(v), lo = bf16(v - hi): C channels are stored as 2C channels [hi_0..hi_{C-1} |
 * lo_0..lo_{C-1}].
 *   csr_nchw_f32_to_nhwc_split  fp32 NCHW (n,c,h,w), c <= 3 -> bf16 NHWC (n,h,w,dst_c) = [hi_0..hi_{c-1}, lo_0..lo_{c-1}, 0...];
 *                               dst_c a multiple of 8, 2c <= dst_c <= 64
 *   csr_maxpool2x2_split        nn.MaxPool2d(2) (floor, NaN-propagating) of hi + lo (exact in fp32), re-split:
 *                               src (n,h,w,2c) -> dst (n,h/2,w/2,2c); h, w >= 2, c % 8 == 0                                */
int     csr_nchw_f32_to_nhwc_split(const float* src, void* dst, int32_t n, int32_t c, int32_t h, int32_t w, int32_t dst_c,
                                   void* stream);
int     csr_maxpool2x2_split(const void* src, void* dst, int32_t n, int32_t h, int32_t w, int32_t c, void* stream);

/* ---- pixel loss of the training step: mean over all numel elements, value AND gradient in one HBM pass --------
 * out[0] = mean |sr - hr| (L1, esrgan) or mean (sr - hr)^2 (MSE, srcnn);  grad (nullable, numel floats) = d out / d sr.
 * scratch: csr_pixel_loss_scratch_bytes(numel).  <- self.loss(sr, hr), core/task.py:141, pl_generator_pre_training.py:29-30 */
size_t  csr_pixel_loss_scratch_bytes(int64_t numel);
int     csr_l1_loss(const float* sr, const float* hr, float* grad, int64_t numel, float* out,
                    void* scratch, size_t scratch_bytes, void* stream);
int     csr_mse_loss(const float* sr, const float* hr, float* grad, int64_t numel, float* out,
                     void* scratch, size_t scratch_bytes, void* stream);

/* ---- masked loss + metrics (one fused HBM pass + SSIM pass) ----------------------------------
 * sr, hr, original, mask: fp32 (N,1,H,W).  mn/mx: FLOAT64 (N) per-sample min/max (min-max scaler: the
 * reference's batch["min"] / batch["max"] are float64 tensors, so MinMaxScaler._denormalize promotes the
 * denormalised tensor - and every metric on it, the |p-t| <= eps counts included - to float64; the kernel
 * does the same, with the scaler's range (a, b) and eps, normalization.py:70-82), or NULL with zmean/zstd
 * used instead (z-score: float32, normalization.py:115).  out: CSR_NUM_METRICS floats (device), see enum. */
enum {
  CSR_M_ACC_0_1 = 0, CSR_M_ACC_0_25, CSR_M_ACC_0_5, CSR_M_ACC_0_75, CSR_M_ACC_1, CSR_M_ACC_1_25,
  CSR_M_ACC_1_5, CSR_M_ACC_2, CSR_M_PSNR, CSR_M_SSIM, CSR_M_MAE, CSR_M_MSE, CSR_M_RMSE, CSR_M_MAPE,
  CSR_M_SMAPE, CSR_M_R2, CSR_M_L1_LOSS, CSR_M_MSE_LOSS, CSR_NUM_METRICS
};
size_t  csr_metrics_scratch_bytes(int32_t n, int32_t h, int32_t w);
int     csr_masked_metrics(const float* sr, const float* hr, const float* original, const float* mask,
                           const double* mn, const double* mx, float zmean, float zstd,
                           double range_a, double range_b, double eps, int32_t n, int32_t h, int32_t w,
                           float* out, void* scratch, size_t scratch_bytes, void* stream);

/* ---- discriminator path (SURVEY section 8f row 2) ------------------------------------------------------------------
 * Replaces climsr.models.discriminator.Discriminator.forward (climsr/models/discriminator.py:5-46) and its autograd
 * backward, driven four times forward / twice backward per GAN batch by climsr/task/pl_gan.py:28-61.  The 3x3 convolutions
 * (stride 1 and 2, reflection-padded or valid) run on csr_conv2d_nhwc / csr_conv2d_wgrad over reflection-padded NHWC bf16
 * buffers; these entry points are everything in between.  A CsrView names the real outputs of a layer inside its buffer
 * (N, hs, ws, c): logical pixel (i, j), i < hl, j < wl, lives at (off + step*i, off + step*j) - off 1 = interior of a
 * same-conv over a padded input, step 2 = the stride-2 convs.  All buffers bf16 NHWC unless noted.
 *   csr_disc_gather      dst (n, hl+2*pad, wl+2*pad, c) = ReflectionPad2d(pad)(view) [* scale[c] + shift[c]: BatchNorm on load]
 *   csr_disc_collect     its backward without BatchNorm: g (S layout) = lrelu'(act) * gathered dP on logical pixels, 0 elsewhere
 *   csr_disc_bn_forward  nn.BatchNorm2d over the logical pixels: training = batch statistics (+ running-statistics update),
 *                        eval = running statistics; emits scale/shift for csr_disc_gather and mean/invstd for the backward
 *   csr_disc_bn_backward g = lrelu'(act) * BN-backward(gathered dP); dgamma / dbeta are accumulated (+=)
 *   csr_disc_flatten / csr_disc_unflatten   x.view(N, -1) of the NCHW tensor (fp32 features) and its backward
 *   csr_linear_forward / csr_linear_backward   nn.Linear in fp32 (8192 -> 100 -> 1); dW / db are accumulated (+=)      */
typedef struct CsrView { int32_t hs, ws, c, off, step, hl, wl; } CsrView;
int     csr_disc_gather(const void* src, const CsrView* view, int32_t n, void* dst, int32_t pad, const float* scale,
                        const float* shift, void* stream);
int     csr_disc_collect(const void* dpad, const CsrView* view, int32_t n, int32_t pad, const void* act, float gate_neg,
                         void* g, void* stream);
size_t  csr_disc_bn_scratch_bytes(int32_t c);
int     csr_disc_bn_forward(const void* src, const CsrView* view, int32_t n, const float* gamma, const float* beta, float eps,
                            float momentum, float* running_mean, float* running_var, int32_t training, float* scale,
                            float* shift, float* mean, float* invstd, void* scratch, size_t scratch_bytes, void* stream);
int     csr_disc_bn_backward(const void* dpad, const CsrView* view, int32_t n, int32_t pad, const void* act, float gate_neg,
                             const float* gamma, const float* mean, const float* invstd, float* dy_scratch, void* scratch,
                             size_t scratch_bytes, void* g, float* dgamma, float* dbeta, void* stream);
int     csr_disc_flatten(const void* src, const CsrView* view, int32_t n, float* feats, void* stream);
int     csr_disc_unflatten(const float* gfeat, const CsrView* view, int32_t n, void* g, void* stream);
int     csr_linear_forward(const float* x, const float* w, const float* b, float* y, int32_t n, int32_t k, int32_t j, void* stream);
int     csr_linear_backward(const float* x, const float* w, const float* gy, float* dx, float* dw, float* db, int32_t n,
                            int32_t k, int32_t j, void* stream);

/* ---- RCAN generator (SURVEY section 8f row 4) --------------------------------------------------------------------------
 * climsr.models.rcan.RCAN.forward (climsr/models/rcan.py:175-186) and its autograd backward: every 3x3 conv (+ ReLU, + the
 * ResidualGroup / body skips as epilogue residuals) runs on csr_conv2d_nhwc, its input gradient on the same entry point with
 * transposed weights (ReLU' as a gate with gate_neg = 0) and its weight gradient on csr_conv2d_wgrad; these entry points are the
 * rest of an RCAB and of the Upsampler.
 *   csr_channel_attention  out = res * sigmoid(W2 relu(W1 avgpool(res) + b1) + b2) + x        (CALayer + RCAB skip, rcan.py:50-101)
 *                          res, x, out: bf16 NHWC (n,h,w,c); w1 (c_reduced, c), w2 (c, c_reduced) fp32; pooled_scratch: n*c floats
 *                          (on return: the per-image channel sums of res, which the backward takes as `pooled`)
 *   csr_channel_attention_backward   its adjoint w.r.t. res given dout = dL/dout: dres = dout * gate + d(avgpool)/dres, gate
 *                          recomputed from `pooled`; dw1, db1, dw2, db2 (fp32, shapes of w1, b1, w2, b2) are ACCUMULATED (+=).
 *                          The skip gradient dL/dx = dout is not written.  scratch: csr_channel_attention_backward_scratch_bytes
 *   csr_pixel_shuffle2     dst (n,2h,2w,c) = nn.PixelShuffle(2)(src (n,h,w,4c))                 (Upsampler, rcan.py:30-36)
 *   csr_pixel_unshuffle2   dst (n,h,w,4c) = nn.PixelUnshuffle(2)(src (n,2h,2w,c)), the adjoint of csr_pixel_shuffle2          */
int     csr_channel_attention(const void* res, const void* x, const float* w1, const float* b1, const float* w2, const float* b2,
                              void* out, float* pooled_scratch, int32_t n, int32_t h, int32_t w, int32_t c, int32_t c_reduced,
                              void* stream);
size_t  csr_channel_attention_backward_scratch_bytes(int32_t n, int32_t c);
int     csr_channel_attention_backward(const void* dout, const void* res, const float* pooled, const float* w1, const float* b1,
                                       const float* w2, const float* b2, void* dres, float* dw1, float* db1, float* dw2,
                                       float* db2, void* scratch, size_t scratch_bytes, int32_t n, int32_t h, int32_t w,
                                       int32_t c, int32_t c_reduced, void* stream);
int     csr_pixel_shuffle2(const void* src, void* dst, int32_t n, int32_t h, int32_t w, int32_t c, void* stream);
int     csr_pixel_unshuffle2(const void* src, void* dst, int32_t n, int32_t h, int32_t w, int32_t c, void* stream);

/* ---- gradient exchange of data-parallel training (SURVEY section 8e: "bf16 gradients are reduced with NCCL over NVLink,
 * bucketed and overlapped with backward"; replaces the gradient all-reduce of Lightning's DDP plugin, conf/trainer/
 * benchmark.yaml:4).  The collective itself is torch.distributed / NCCL; these are the wire-format kernels around it:
 * comm = bf16(scale * flat) with scale = 1 / world applied BEFORE the rounding, and flat = scale * float(comm).
 * csr_set_option(30, k) makes training plans created afterwards leave k SMs free for the collective's CTAs. */
int     csr_grad_pack_bf16(const float* flat, void* comm_bf16, size_t n, float scale, void* stream);
int     csr_grad_unpack_bf16(const void* comm_bf16, float* flat, size_t n, float scale, void* stream);

/* ---- inference pre / post-processing on device (SURVEY section 8f row 1) -------------------------------------------
 * The reference normalises each LR raster on the CPU (MinMaxScaler._normalize, climsr/data/normalization.py:37-61, called
 * from geo_tiff_inference_dataset.py:161-166), concatenates [raster, elevation_lr, mask_lr] (:101-121), and after the
 * forward pulls the result to the host, denormalises it with the raster's min / max (normalization.py:63-84) and writes
 * NaN outside the land mask (climsr/inference/inference.py:73-76).  Both run here as one HBM pass each, float64
 * arithmetic with a single rounding to float32.
 *   raw (n,h,w) fp32 with NaN for missing values; mn, mx: n DEVICE doubles; (a, b) = feature range; eps as the scaler's.
 *   extra0 / extra1: NULL or shared (h,w) fp32 planes appended as channels 1 (, 2) of every sample.
 *   out: (n, 1 + number of extras, h, w) fp32 NCHW = the generator's `x`.                                               */
int     csr_minmax_normalize(const float* raw, int32_t n, int32_t h, int32_t w, const double* mn, const double* mx,
                             double range_a, double range_b, double eps, float nan_substitution,
                             const float* extra0, const float* extra1, float* out, void* stream);
/*   sr (n,1,h,w) fp32 generator output; mask fp32, (1,1,h,w) shared (mask_per_sample = 0) or (n,1,h,w);
 *   out (n,1,h,w) fp32 = (sr - min_) / scale where mask > 0, NaN elsewhere.                                              */
int     csr_minmax_denormalize_mask(const float* sr, const float* mask, int32_t mask_per_sample, int32_t n, int32_t h, int32_t w,
                                    const double* mn, const double* mx, double range_a, double range_b, double eps,
                                    float* out, void* stream);

/* ---- training-sample assembly on device (SURVEY section 8f row 3) ---------------------------------------------------
 * The reference builds every sample on the CPU (climsr/data/sr/climate_dataset.py): random np.flipud / np.fliplr /
 * np.rot90(k) of the HR tile, its elevation and its land mask (:152-170), LR = albumentations Resize = cv2 INTER_NEAREST by
 * 1/scale (:84-92,172: the top-left pixel of every scale x scale block), elevation_lr and mask_lr the same way (:118,136),
 * x = cat[lr, elevation_lr, mask_lr] (:98-121).  One pass here; index work only, bit-exact.
 *   hr, elev, mask (n,1,H,W) fp32; H, W multiples of scale; codes: n DEVICE int32 (bit0 vertical flip, bit1 horizontal
 *   flip, bits 2-3 rot90 factor; applied in that order; odd factors need H == W) or NULL (no augmentation).
 *   hr_out / elev_out / mask_out (n,1,H,W): the augmented tensors (all three or none; may be NULL when codes is NULL).
 *   x_out (n,3,H/scale,W/scale) = the generator's input.                                                                */
int     csr_lr_input_from_hr(const float* hr, const float* elev, const float* mask, int32_t n, int32_t H, int32_t W, int32_t scale,
                             const int32_t* codes, float* hr_out, float* elev_out, float* mask_out, float* x_out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CLIMSR_B200_H */

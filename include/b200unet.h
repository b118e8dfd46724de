/*
 * b200unet.h -- C ABI of libb200unet.so: the sm_100a kernels behind the Our_UNet training step.
 *
 * The reference (Ulixes-8/UNet-Implementations) has no FFI: its hot path is the Python class surface
 * `models.unet.UNet` / `models.losses.SimpleLoss` dispatching to stock torch.nn ops (cuDNN/ATen).  Every entry
 * point below replaces one of those implicit library dispatches; the reference call site it stands in for is
 * cited per function (paths relative to the reference root).  The Python host (`models/unet.py`,
 * `models/losses.py` in this repo) binds these with ctypes -- see INTEGRATION.md.
 *
 * Conventions
 *  - plain C: raw device pointers, ints, floats; no torch types.  Every function returns 0 on success or a
 *    negative code; `b200unet_last_error()` returns the (thread-local) message.
 *  - all work is enqueued on the `stream` argument (a cudaStream_t passed as void*); nothing synchronises,
 *    allocates or frees device memory; no device pointer is retained after return.
 *  - activations are NHWC bf16.  A tensor argument is (ptr, pitch): element (n,h,w,c) lives at
 *    ptr[((n*H + h)*W + w)*pitch + c]; pitch >= C lets an operator read or write a channel slice of a wider
 *    buffer (the decoder concat buffer), which is how torch.cat (unet.py:228) disappears.
 *  - "stats partial" buffers are fp32 [N][P][C][2] = per-image partial (sum, sum of squares) produced by P
 *    tiles/blocks per image; they are reduced in fixed order (deterministic, no atomics).
 */
#ifndef B200UNET_H_
#define B200UNET_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200UNET_VERSION 100

int b200unet_version(void);
const char* b200unet_last_error(void);
/* Number of kernels this library has launched in this process (monotonic; bench.py reports the delta). */
long long b200unet_launch_count(void);
/* 1 if the current device is compute capability 10.x, else 0 (negative on error). */
int b200unet_device_ok(void);
/* Size every grid launched from now on for (device SMs - n) SMs; returns the previous value.  The data-parallel
 * reducer (ddp.py) brackets backward with it so that the NCCL all-reduce kernels overlapping backward always find a
 * free SM instead of delaying one CTA of a persistent one-CTA-per-SM conv kernel.  No reference counterpart (the
 * reference has no distributed code, SURVEY.md 2.2). */
int b200unet_set_reserved_sms(int n);
/* Programmatic dependent launch of the library's kernels (off by default -- measured no gain; B200UNET_PDL=1 enables): each kernel's CTAs
 * become resident and run their set-up while the previous kernel of the stream drains, and wait (griddepcontrol.wait)
 * before touching global memory.  Returns the previous setting.  No reference counterpart. */
int b200unet_set_pdl(int on);

/* ------------------------------------------------------------------------------------------------------------
 * 3x3 convolution, pad 1, stride 1 or 2 -- replaces nn.Conv2d in ConvBlock (Our_UNet/models/unet.py:106-115)
 * and its autograd backward (aten::convolution_backward).  Implicit GEMM on tcgen05/TMEM, operands staged by TMA.
 * The conv bias is not applied: it feeds an InstanceNorm and cancels exactly (SURVEY.md 8a).
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct {
  const void* x;      /* bf16 NHWC input  [N,H,W,Cin], pitch x_pitch            */
  int64_t x_pitch;
  const void* w;      /* bf16 packed weights [Cout][3][3][Cin] (b200unet_pack_conv_weights) */
  void* y;            /* bf16 NHWC raw conv output [N,OH,OW,Cout], pitch y_pitch */
  int64_t y_pitch;
  float* stats;       /* fp32 [N][P][Cout][2] partial sums of y and y*y over valid pixels (P from
                         b200unet_conv_fprop_partials; zero-filled by the call), or NULL */
  int N, H, W, Cin, Cout, stride;
} b200unet_conv_fprop_args;
/* Number of stat partial slots per image (P) of the fprop kernel for N images of OH x OW x Cout outputs. */
int b200unet_conv_fprop_partials(int N, int OH, int OW, int Cout);
int b200unet_conv_fprop(const b200unet_conv_fprop_args* a, void* stream);

typedef struct {
  const void* dy;     /* bf16 NHWC gradient wrt raw conv output [N,OH,OW,Cout], pitch dy_pitch */
  int64_t dy_pitch;
  const void* wt;     /* bf16 packed transposed weights [Cin][3][3][Cout] */
  void* dx;           /* bf16 NHWC gradient wrt conv input [N,H,W,Cin], pitch dx_pitch */
  int64_t dx_pitch;
  int N, H, W, Cin, Cout, stride; /* H,W = conv INPUT size */
  /* Optional producer-side InstanceNorm-backward sums (b200unet_in_bwd_args.ext_part).  dx is the gradient dz of the
   * unit whose output feeds this conv; with bs_part != NULL the epilogue also reads that unit's raw output bs_y
   * ([N,H,W,Cin] bf16) and reduces, per image over its own tiles, T1 = sum gm and T2raw = sum gm * y with
   * gm = dx_stored * (bs_a*y + bs_b > 0 ? 1 : bs_slope), so that unit's norm backward needs no reduction pass.
   * bs_part = fp32 [N][P][Cin][2], P = b200unet_conv_dgrad_bwd_slots(...) > 0 (0 = this shape does not support it). */
  const void* bs_y;
  int64_t bs_y_pitch;
  const float* bs_a;   /* fp32 [N,Cin] */
  const float* bs_b;
  float bs_slope;
  float* bs_part;
  /* Optional second output (stride 1): channels [0, dx_split) of the gradient go to dx, channels [dx_split, Cin) to dx2
   * -- the [upsampled | skip] halves of a decoder concat buffer's gradient (torch.cat backward, unet.py:228) as two
   * dense tensors instead of two slices of one.  NULL = one output. */
  void* dx2;
  int64_t dx2_pitch;
  int dx_split;
} b200unet_conv_dgrad_args;
int b200unet_conv_dgrad(const b200unet_conv_dgrad_args* a, void* stream);
int b200unet_conv_dgrad_bwd_slots(int N, int H, int W, int Cin, int Cout, int stride);

typedef struct {
  const void* x;      /* bf16 NHWC conv input [N,H,W,Cin], pitch x_pitch */
  int64_t x_pitch;
  const void* dy;     /* bf16 NHWC gradient wrt raw conv output [N,OH,OW,Cout], pitch dy_pitch */
  int64_t dy_pitch;
  float* dw;          /* fp32 OIHW [Cout][Cin][3][3] (the nn.Conv2d.weight.grad layout) */
  float* workspace;   /* fp32 scratch, at least b200unet_conv_wgrad_workspace() bytes */
  int64_t workspace_bytes;
  int N, H, W, Cin, Cout, stride;
} b200unet_conv_wgrad_args;
int64_t b200unet_conv_wgrad_workspace(int N, int H, int W, int Cin, int Cout, int stride);
int b200unet_conv_wgrad(const b200unet_conv_wgrad_args* a, void* stream);

/* CUDA-core direct convolutions with the same argument structs: the slow, obviously-correct path used by the
 * tests to cross-check the tensor-core kernels on the device and for shapes outside their envelope. */
int b200unet_conv_fprop_simt_partials(int OH, int OW); /* P of the stats buffer for the _simt fprop */
int b200unet_conv_fprop_simt(const b200unet_conv_fprop_args* a, void* stream);
int b200unet_conv_dgrad_simt(const b200unet_conv_dgrad_args* a, void* stream);
int b200unet_conv_wgrad_simt(const b200unet_conv_wgrad_args* a, void* stream);

/* fp32 OIHW [Cout][Cin][3][3] -> bf16 [Cout][3][3][Cin] (w_fprop) and bf16 [Cin][3][3][Cout] (w_dgrad, may be NULL) */
int b200unet_pack_conv_weights(const float* w_oihw, void* w_fprop, void* w_dgrad, int Cout, int Cin, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Stem: first conv of encoder stage 0 (Cin = 3, Cout = 32, stride 1), unet.py:106-115 with the trainer's
 * config (train.py:776-795).  Reads the fp32 NCHW image directly (train.py:630), writes bf16 NHWC + stat partials.
 * ---------------------------------------------------------------------------------------------------------- */
int b200unet_stem_partials(int H, int W);
int b200unet_stem_fprop(const float* img_nchw, const float* w_oihw, void* y, int64_t y_pitch, float* stats, int N,
                        int H, int W, void* stream);
int64_t b200unet_stem_wgrad_workspace(int N, int H, int W);
int b200unet_stem_wgrad(const float* img_nchw, const void* dy, int64_t dy_pitch, float* dw_oihw, float* workspace,
                        int64_t workspace_bytes, int N, int H, int W, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * InstanceNorm2d(eps, affine) + LeakyReLU(slope) + SpatialDropout2d, fused
 * (unet.py:118-127, SpatialDropout2d.forward unet.py:22-35).
 *   finalize: partials -> mean, rstd and the folded per-(n,c) affine  a = s*gamma*rstd, b = s*(beta - mean*gamma*rstd)
 *             where s = drop_scale[n][c] in {0, 1/(1-p)} (NULL = 1).
 *   apply   : z = leaky_relu(a*y + b)   (valid because s >= 0)
 * ---------------------------------------------------------------------------------------------------------- */
int b200unet_in_finalize(const float* stats, int P, const float* gamma, const float* beta, const float* drop_scale,
                         float eps, float* mean, float* rstd, float* a, float* b, int N, int C, int64_t HW,
                         void* stream);
int b200unet_in_apply(const void* y, int64_t y_pitch, const float* a, const float* b, float slope, void* z,
                      int64_t z_pitch, int N, int64_t HW, int C, void* stream);
/* Backward (aten::native_batch_norm_backward + leaky_relu_backward + mul in the reference's autograd graph), one call:
 *   g  = (dz + dz2) * (a*y+b > 0 ? 1 : slope) * s ;  xh = (y - mean)*rstd
 *   dy = gamma*rstd * (g - mean_hw(g) - xh*mean_hw(g*xh)) ;  dgamma = sum g*xh ;  dbeta = sum g
 * Runs reduce -> finalize -> apply over chunks of images small enough that the apply pass re-reads dz and y from
 * L2 rather than HBM.  All reductions are in fixed order (deterministic). */
typedef struct {
  const void* dz;      /* bf16 NHWC gradient wrt the activated output [N,H,W,C], pitch dz_pitch */
  int64_t dz_pitch;
  const void* dz2;     /* optional second contribution (skip connection), or NULL */
  int64_t dz2_pitch;
  const void* y;       /* bf16 NHWC raw conv output saved by the forward */
  int64_t y_pitch;
  const float* a;      /* fp32 [N,C] from b200unet_in_finalize */
  const float* b;
  const float* mean;
  const float* rstd;
  const float* drop_scale; /* fp32 [N,C] or NULL */
  const float* gamma;  /* fp32 [C] */
  float slope;
  void* dy;            /* bf16 NHWC gradient wrt the raw conv output, pitch dy_pitch */
  int64_t dy_pitch;
  float* dgamma;       /* fp32 [C] */
  float* dbeta;        /* fp32 [C] */
  float* workspace;    /* at least b200unet_in_backward_workspace() bytes */
  int64_t workspace_bytes;
  int N;
  int64_t HW;
  int C;
  /* Producer-side sums (optional): the kernel that WROTE dz -- a data-gradient epilogue, the head backward -- may already
   * have reduced, per image over its own P blocks, T1 = sum gm and T2raw = sum gm * y with
   * gm = dz_stored * (a*y+b > 0 ? 1 : slope): fp32 [N][ext_P][C][2].  With ext_part (and ext_part2 for dz2 when dz2 is
   * given) the reduction pass over (dz, y) is skipped: 3 tensor passes instead of 5.  NULL = reduce here. */
  const float* ext_part;
  int ext_P;
  const float* ext_part2;
  int ext_P2;
  /* != 0: do not reduce dgamma / dbeta here; the caller runs b200unet_in_bwd_params on the same workspace later
   * (dy does not depend on them: the host takes that 6 us kernel off the critical path of backward). */
  int defer_params;
} b200unet_in_bwd_args;
int64_t b200unet_in_backward_workspace(int N, int64_t HW, int C);
int b200unet_in_backward(const b200unet_in_bwd_args* a, void* stream);
int b200unet_in_bwd_params(const float* workspace, int N, int64_t HW, int C, float* dgamma, float* dbeta, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Exact 2x bilinear upsampling, align_corners=False -- F.interpolate in UpBlock.forward (unet.py:219-225) --
 * written straight into channels [0,C) of the concat buffer (pitch out_pitch), and its backward.
 * ---------------------------------------------------------------------------------------------------------- */
int b200unet_upsample2x_fwd(const void* x, int64_t x_pitch, void* out, int64_t out_pitch, int N, int H, int W, int C,
                            void* stream); /* H,W = input size; output is 2H x 2W */
int b200unet_upsample2x_bwd(const void* dout, int64_t dout_pitch, void* dx, int64_t dx_pitch, int N, int H, int W,
                            int C, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Segmentation head: 1x1 Conv2d(C -> K) + bias (unet.py:374-381, 430).  Reads bf16 NHWC, writes fp32 NCHW logits.
 * Backward: dz (bf16 NHWC), dW [K][C], db [K] (two-stage deterministic reduction through `workspace`).
 * ---------------------------------------------------------------------------------------------------------- */
int b200unet_head_fwd(const void* z, int64_t z_pitch, const float* w, const float* bias, float* logits_nchw, int N,
                      int64_t HW, int C, int K, void* stream);
int64_t b200unet_head_bwd_workspace(int N, int64_t HW, int C, int K);
int b200unet_head_bwd(const float* dlogits_nchw, const void* z, int64_t z_pitch, const float* w, void* dz,
                      int64_t dz_pitch, float* dw, float* db, float* workspace, int64_t workspace_bytes, int N,
                      int64_t HW, int C, int K, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * SimpleLoss: weight_ce * CE(weight=w, ignore_index) + weight_dice * Dice, 3 classes
 * (Our_UNet/models/losses.py:24-121).  One reduction pass over logits+target, one elementwise backward pass.
 *   class_weights: NULL -> dynamic inverse-frequency weights (losses.py:24-62) when dynamic != 0, else uniform;
 *                  non-NULL and dynamic == 0 -> static weights (device fp32 [3]).
 *   loss_out[0] = total, [1] = CE, [2] = Dice.   tables: fp32 scratch [3 + 2*3*N] kept for the backward.
 * ---------------------------------------------------------------------------------------------------------- */
int64_t b200unet_loss_workspace(int N, int64_t HW);
int b200unet_loss_fwd(const float* logits_nchw, const int64_t* target, const float* class_weights, int dynamic,
                      float weight_ce, float weight_dice, int ignore_index, float smooth, float* loss_out,
                      float* tables, float* workspace, int64_t workspace_bytes, int N, int64_t HW, void* stream);
int b200unet_loss_bwd(const float* logits_nchw, const int64_t* target, const float* tables, const float* grad_out,
                      float weight_ce, float weight_dice, int ignore_index, float* dlogits_nchw, int N, int64_t HW,
                      void* stream);
/* The same two passes with uint8 targets [N,H,W] in {0,1,2,255} -- the masks as the dataset stores them
 * (train.py:300, :311 widens them to int64 only because nn.CrossEntropyLoss wants int64): 1 instead of 8 bytes per
 * pixel across PCIe and through HBM (SURVEY.md 8f row 2). */
int b200unet_loss_fwd_u8(const float* logits_nchw, const uint8_t* target, const float* class_weights, int dynamic,
                         float weight_ce, float weight_dice, int ignore_index, float smooth, float* loss_out,
                         float* tables, float* workspace, int64_t workspace_bytes, int N, int64_t HW, void* stream);
int b200unet_loss_bwd_u8(const float* logits_nchw, const uint8_t* target, const float* tables, const float* grad_out,
                         float weight_ce, float weight_dice, int ignore_index, float* dlogits_nchw, int N, int64_t HW,
                         void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Layout helpers used by the module-level (per-op) entry points and the tests.
 * ---------------------------------------------------------------------------------------------------------- */
int b200unet_nchw_f32_to_nhwc_bf16(const float* src, void* dst, int64_t dst_pitch, int N, int C, int64_t HW,
                                   void* stream);
int b200unet_nhwc_bf16_to_nchw_f32(const void* src, int64_t src_pitch, float* dst, int N, int C, int64_t HW,
                                   void* stream);

/* Stride-2 data gradient for Cin in {32, 64} with the four input-pixel parity classes stacked on N (one launch, N =
 * 4*Cin, dy read once) instead of four narrow launches.  `wt` of the args is the pack produced by
 * b200unet_pack_s2_dgrad_weights from the ordinary dgrad pack ([Cin][3][3][Cout] -> [4*Cin][4][Cout]). */
int b200unet_conv_dgrad_s2_supported(int Cin, int Cout);
int b200unet_pack_s2_dgrad_weights(const void* wt, void* ws, int Cin, int Cout, void* stream);
int b200unet_conv_dgrad_s2(const b200unet_conv_dgrad_args* a, void* stream);

/* Consumers with the producer's apply pass fused in.  When the activated tensor z = leaky_relu(a*y + b) of a unit has
 * ONE consumer -- the 2x upsample of the next decoder stage (unet.py:219-225) or the segmentation head (unet.py:430) --
 * that consumer reads the unit's RAW conv output y with its folded affine (a, b from b200unet_in_finalize) and applies
 * InstanceNorm/LeakyReLU/dropout on the fly: b200unet_in_apply is skipped for the unit and z is never written or
 * re-read.  head_norm_bwd recomputes z from y for dW.  Same arguments as the plain entry points plus (a, b, slope). */
int b200unet_upsample2x_norm_fwd(const void* y, int64_t y_pitch, const float* a, const float* b, float slope, void* out,
                                 int64_t out_pitch, int N, int H, int W, int C, void* stream);
int b200unet_head_norm_fwd(const void* y, int64_t y_pitch, const float* a, const float* b, float slope, const float* w,
                           const float* bias, float* logits_nchw, int N, int64_t HW, int C, int K, void* stream);
int b200unet_head_norm_bwd(const float* dlogits_nchw, const void* y, int64_t y_pitch, const float* a, const float* b,
                           float slope, const float* w, void* dz, int64_t dz_pitch, float* dw, float* db,
                           float* workspace, int64_t workspace_bytes, int N, int64_t HW, int C, int K, void* stream);
/* head_norm_bwd that also emits the norm-backward partial sums of the unit whose raw output y it reads (see
 * b200unet_in_bwd_args.ext_part): bwd_part = fp32 [N][P][C][2], P = b200unet_head_bwd_stat_slots(N, HW). */
int b200unet_head_bwd_stat_slots(int N, int64_t HW);
int b200unet_head_norm_bwd_stats(const float* dlogits_nchw, const void* y, int64_t y_pitch, const float* a, const float* b,
                                 float slope, const float* w, void* dz, int64_t dz_pitch, float* dw, float* db,
                                 float* workspace, int64_t workspace_bytes, float* bwd_part, int N, int64_t HW, int C, int K,
                                 void* stream);
int b200unet_head_norm_bwd_stats_f32(const float* dlogits_nchw, const void* y, int64_t y_pitch, const float* a,
                                     const float* b, float slope, const float* w, void* dz, int64_t dz_pitch, float* dw,
                                     float* db, float* workspace, int64_t workspace_bytes, float* bwd_part, int N,
                                     int64_t HW, int C, int K, void* stream);
int b200unet_upsample2x_norm_fwd_f32(const void* y, int64_t y_pitch, const float* a, const float* b, float slope,
                                     void* out, int64_t out_pitch, int N, int H, int W, int C, void* stream);
int b200unet_head_norm_fwd_f32(const void* y, int64_t y_pitch, const float* a, const float* b, float slope,
                               const float* w, const float* bias, float* logits_nchw, int N, int64_t HW, int C, int K,
                               void* stream);
int b200unet_head_norm_bwd_f32(const float* dlogits_nchw, const void* y, int64_t y_pitch, const float* a, const float* b,
                               float slope, const float* w, void* dz, int64_t dz_pitch, float* dw, float* db,
                               float* workspace, int64_t workspace_bytes, int N, int64_t HW, int C, int K, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * fp32 verification mode (`UNet(...).precision = "fp32"`): the same operators with fp32 NHWC activations, fp32
 * packed weights and fp32 arithmetic -- north_star's "1e-4 in fp32 mode".  Argument structs, layouts and
 * semantics are those of the bf16 entry points above with every `bf16` read as `fp32`; the norm / resample /
 * head kernels are the SAME templates instantiated for fp32 storage, the convolutions are the direct CUDA-core
 * kernels (the tensor-core path is bf16-only).  Not a fallback: selected explicitly by the caller, CUDA only.
 * ---------------------------------------------------------------------------------------------------------- */
int b200unet_pack_conv_weights_f32(const float* w_oihw, void* w_fprop, void* w_dgrad, int Cout, int Cin, void* stream);
int b200unet_conv_fprop_f32(const b200unet_conv_fprop_args* a, void* stream); /* stats: P = b200unet_conv_fprop_simt_partials */
int b200unet_conv_dgrad_f32(const b200unet_conv_dgrad_args* a, void* stream);
int b200unet_conv_wgrad_f32(const b200unet_conv_wgrad_args* a, void* stream); /* no workspace needed */
int b200unet_in_apply_f32(const void* y, int64_t y_pitch, const float* a, const float* b, float slope, void* z,
                          int64_t z_pitch, int N, int64_t HW, int C, void* stream);
int b200unet_in_backward_f32(const b200unet_in_bwd_args* a, void* stream);
int b200unet_upsample2x_fwd_f32(const void* x, int64_t x_pitch, void* out, int64_t out_pitch, int N, int H, int W,
                                int C, void* stream);
int b200unet_upsample2x_bwd_f32(const void* dout, int64_t dout_pitch, void* dx, int64_t dx_pitch, int N, int H,
                                int W, int C, void* stream);
int b200unet_head_fwd_f32(const void* z, int64_t z_pitch, const float* w, const float* bias, float* logits_nchw,
                          int N, int64_t HW, int C, int K, void* stream);
int b200unet_head_bwd_f32(const float* dlogits_nchw, const void* z, int64_t z_pitch, const float* w, void* dz,
                          int64_t dz_pitch, float* dw, float* db, float* workspace, int64_t workspace_bytes, int N,
                          int64_t HW, int C, int K, void* stream);
int b200unet_nchw_f32_to_nhwc_f32(const float* src, void* dst, int64_t dst_pitch, int N, int C, int64_t HW,
                                  void* stream);

/* fp32 NCHW image [N,C<=8,H,W] -> bf16 NHWC [N,H,W,32] with channels C..31 zero: the X operand of the stem's
 * weight gradient on the tensor-core path (b200unet_conv_wgrad with Cin = 32; rows ci >= C of dW are zero).
 * Replaces the weight-gradient half of aten::convolution_backward for encoder_stages[0].block[0] (unet.py:106). */
int b200unet_image_to_nhwc32_bf16(const float* src, void* dst, int N, int C, int64_t HW, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * The steps either side of the hot path (SURVEY.md section 8f).
 * sgd_nesterov_step: torch.optim.SGD(lr, momentum, nesterov=True, weight_decay) over `count` fp32 tensors in ONE
 *   launch (Our_UNet/src/train.py:431-451 builds that optimizer; train.py:651-660 steps it).  Host arrays of DEVICE
 *   pointers; arithmetic mirrors torch's foreach SGD on CUDA operation by operation (bit-exact, tests/test_gpu_aux.py).
 *   first_step != 0 initialises the momentum buffers with the (decayed) gradient, as torch does.
 * argmax_counts: torch.argmax(outputs, dim=1) + the per-class intersection / prediction / target pixel counts over
 *   valid pixels that validate() turns into Dice scores (train.py:554-572).  counts9 = int64 [3][3] on the device:
 *   [c][0] = #(pred==c & target==c), [c][1] = #(pred==c), [c][2] = #(target==c), valid pixels only; pred (int64
 *   [N,H,W], ties -> lowest index) is optional.
 * ---------------------------------------------------------------------------------------------------------- */
 /* preprocess_u8: the per-sample tensor conversion of PetSegmentationDataset.__getitem__ (train.py:299-311) for a whole
 *   batch on the device: uint8 HWC image [N,H,W,3] -> (x / 255 - mean) / std -> fp32 NCHW, uint8 mask [N,H,W] ->
 *   {0,1,2,255} int64 (other values become 0).  mean3/std3 are HOST pointers.  Either half may be NULL.  Bit-exact. */
int b200unet_preprocess_u8(const void* image_u8_nhwc, const void* mask_u8, float* image_out_nchw, int64_t* mask_out,
                           const float* mean3, const float* std3, int N, int64_t HW, void* stream);
/* preprocess_u8_nhwc32: the same image conversion written straight as the stem's tensor-core operand -- uint8 HWC
 *   [N,H,W,3] -> (x / 255 - mean) / std (fp32, the reference's operations in its order) -> bf16 NHWC [N,H,W,32] with
 *   channels 3..31 zero, in ONE kernel: bit-identical to preprocess_u8 followed by image_to_nhwc32_bf16, without the
 *   12-byte/pixel fp32 round trip through HBM.  mean3/std3 are HOST pointers. */
int b200unet_preprocess_u8_nhwc32(const void* image_u8_nhwc, void* dst_nhwc32, const float* mean3, const float* std3, int N,
                                  int64_t HW, void* stream);
int b200unet_sgd_max_tensors(void);
int b200unet_sgd_nesterov_step(float* const* params, const float* const* grads, float* const* momentum_bufs,
                               const int64_t* numels, int count, float lr, float momentum, float weight_decay,
                               int nesterov, int first_step, void* stream);
/* sgd_flat_step -- SURVEY.md 8f row 1 as written: the optimizer step of train.py:431-453 / :650 / :664 as ONE launch
 *   over flat fp32 master / gradient / momentum buffers (all tensors at the same element offsets), which scales the
 *   gradient (the mean of the gradient all-reduce, or a GradScaler's 1/scale), applies SGD + Nesterov momentum +
 *   weight decay with the arithmetic of sgd_nesterov_step, and EMITS the bf16 packs the conv kernels read
 *   ([Cout][3][3][Cin_pad], [Cin][3][3][Cout_pad], and the parity-stacked stride-2 dgrad pack) for every tensor whose
 *   descriptor names them -- the per-step repack (pack_conv_weights) disappears.  `table_dev` is a DEVICE array of
 *   `count` descriptors sorted by first_block; first_block = prefix sum of ceil(numel / sgd_flat_block_elems()).
 *   flags bit 0: update this tensor; bit 1: first momentum step (buf = decayed gradient, as torch does). */
typedef struct {
  int64_t offset;      /* element offset of the tensor in the flat buffers */
  int32_t numel;
  int32_t flags;
  int32_t first_block;
  int32_t cout, cin, ksize; /* conv weight OIHW [cout][cin][ksize][ksize], ksize 3 or 1 (centre tap); unused without packs */
  int32_t cout_pad, cin_pad; /* row lengths of the dgrad / fprop packs (zero padding is the caller's, written once) */
  void* wf;            /* bf16 [cout][3][3][cin_pad] or NULL (no packs) */
  void* wd;            /* bf16 [cin][3][3][cout_pad] or NULL */
  void* ws;            /* bf16 [4*cin][4][cout] (b200unet_pack_s2_dgrad_weights layout) or NULL */
} b200unet_flat_tensor;
int b200unet_sgd_flat_block_elems(void);
int b200unet_sgd_flat_step(const b200unet_flat_tensor* table_dev, int count, int total_blocks, float* master,
                           const float* grad, float* momentum_buf, float lr, float momentum, float weight_decay,
                           int nesterov, float grad_scale, const float* lr_dev /* device scalar overriding lr, or NULL */,
                           void* stream);
/* adam_flat_step -- torch.optim.Adam(lr, betas, eps, weight_decay, decoupled_weight_decay) (AdamW when decoupled != 0),
 *   the optimizer of the autoencoder's trainer (AE_pretrained/reconstruction/src/train.py:390-394), over the same flat
 *   buffers and descriptor table as sgd_flat_step, packs included: master / gradient / exp_avg / exp_avg_sq at the
 *   same element offsets.  The arithmetic is torch 2.11's `_multi_tensor_adam` (torch/optim/adam.py, capturable=False)
 *   operation by operation: bit-exact with torch.optim.Adam on CUDA for grad_scale 1 (or a power of two).
 *   steps: DEVICE fp32 [count], the per-tensor step counts (torch's state["step"]), advanced for every tensor whose
 *   flags bit 0 is set; scalars_ws: DEVICE fp32 [4 * count], 16-byte aligned, scratch for the per-tensor scalars.
 *   Two launches on `stream` (a one-block prologue that advances the counts and forms the bias corrections in double,
 *   then the flat step), so that a CUDA graph of the step replays both.  lr_dev: DEVICE fp64 scalar overriding lr,
 *   or NULL.  Flags bit 1 is ignored: zero moments are Adam's initial state. */
int b200unet_adam_flat_step(const b200unet_flat_tensor* table_dev, int count, int total_blocks, float* master,
                            const float* grad, float* exp_avg, float* exp_avg_sq, float* steps, float* scalars_ws,
                            double lr, const double* lr_dev, double beta1, double beta2, double eps, double weight_decay,
                            int decoupled, float grad_scale, void* stream);
int b200unet_argmax_counts(const float* logits_nchw, const int64_t* target, int ignore_index, int64_t* pred_or_null,
                           int64_t* counts9, int N, int64_t HW, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Autoencoder variant (BASELINE.json configs[3]; AE_pretrained/reconstruction/models/autoencoder.py:374-387,
 * src/train.py:431): reconstruction_output = Conv2d(32 -> 3, 3x3) + Sigmoid, nn.MSELoss.  The 3x3 conv runs on the
 * conv entry points above with its output channels zero-padded; recon_head_fwd is its epilogue (bias + sigmoid ->
 * fp32 NCHW [N,K,H,W], K <= 4), recon_head_bwd the backward prologue: dpre = dout * out * (1 - out) written as the
 * NHWC gradient operand with channels K..Cpad-1 zero, and db[K] = sum dpre.  mse_fwd/bwd: mean squared error over n
 * fp32 elements and its gradient 2 (a - b) / n * grad_out.
 * ---------------------------------------------------------------------------------------------------------- */
int b200unet_recon_head_fwd(const void* y, int64_t y_pitch, const float* bias, float* out_nchw, int N, int64_t HW,
                            int K, void* stream);
int b200unet_recon_head_fwd_f32(const void* y, int64_t y_pitch, const float* bias, float* out_nchw, int N, int64_t HW,
                                int K, void* stream);
int64_t b200unet_recon_head_bwd_workspace(int N, int64_t HW);
int b200unet_recon_head_bwd(const float* dout_nchw, const float* out_nchw, void* dpre, int64_t dpre_pitch, int Cpad,
                            float* db, float* workspace, int64_t workspace_bytes, int N, int64_t HW, int K,
                            void* stream);
int b200unet_recon_head_bwd_f32(const float* dout_nchw, const float* out_nchw, void* dpre, int64_t dpre_pitch, int Cpad,
                                float* db, float* workspace, int64_t workspace_bytes, int N, int64_t HW, int K,
                                void* stream);
int64_t b200unet_mse_workspace(int64_t n);
int b200unet_mse_fwd(const float* a, const float* b, float* loss_out, float* workspace, int64_t workspace_bytes,
                     int64_t n, void* stream);
int b200unet_mse_bwd(const float* a, const float* b, const float* grad_out, float* da, int64_t n, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B200UNET_H_ */

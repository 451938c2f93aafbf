/*
 * teco.h -- C ABI of libteco.so: hand-written sm_100a kernels for the TecoGAN recurrent
 * video-SR hot path (SURVEY.md section 8).  Plain pointers and sizes only; no torch types.
 *
 * The reference (thunil/TecoGAN) has no FFI layer: its "operator API" is Python functions
 * that build TensorFlow graph ops.  Each entry point below names the reference call site
 * (file:line under /root/reference) whose TensorFlow/cuDNN arithmetic it replaces; the Python
 * mirror in tecogan_b200/lib/{ops,frvsr,Teco}.py keeps the reference's function names and
 * binds these symbols through ctypes (see INTEGRATION.md).
 *
 * Conventions
 *  - every pointer is a DEVICE pointer unless the name ends in _host;
 *  - activations are NHWC, contiguous, with an explicit channel pitch where stated;
 *  - weights use the TensorFlow layouts (conv: [kh,kw,Cin,Cout]; conv_transpose: [kh,kw,Cout,Cin]);
 *  - `stream` is a cudaStream_t passed as void*; all work is stream-ordered, nothing allocates;
 *  - return 0 on success, a negative TECO_E_* code on failure; teco_last_error() gives the
 *    thread-local message.  No exceptions cross the ABI.  There is no CPU fallback.
 */
#ifndef TECO_H_
#define TECO_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TECO_OK 0
#define TECO_E_INVALID (-1)   /* bad shape / argument            -> Python ValueError   */
#define TECO_E_CUDA (-2)      /* CUDA runtime / driver error     -> Python RuntimeError */
#define TECO_E_UNSUPPORTED (-3)

/* epilogue activations (reference: tf.nn.relu lib/frvsr.py:53; lrelu lib/ops.py:84-85 with
 * alpha 0.2 lib/frvsr.py:8; tanh*24 lib/frvsr.py:39; sigmoid lib/Teco.py:72) */
enum { TECO_ACT_NONE = 0, TECO_ACT_RELU = 1, TECO_ACT_LRELU02 = 2, TECO_ACT_TANH24 = 3, TECO_ACT_SIGMOID = 4 };

const char* teco_last_error(void);
int teco_version(void);
/* Fills props[0..7] = {sm_count, cc_major, cc_minor, max_smem_optin, l2_bytes, 0,0,0}. */
int teco_device_props(int device, int64_t* props);
/* Host utility: CRC32C (Castagnoli) of n bytes continuing from crc (0 to start); returns the CRC in [0, 2^32) or a negative
   TECO_E_* code.  Used by tecogan_b200/tf_bundle.py to verify TensorFlow checkpoint blocks and tensors (the reference gets
   this from tf.train.Saver, main.py:224,245,307). */
int64_t teco_crc32c(const void* data, int64_t n, int64_t crc);

/* ---------------------------------------------------------------------------------------
 * fp32 direct convolution (exact-parity path; also dgrad via flipped weights).
 * Replaces slim.conv2d behind conv2() lib/ops.py:47-56 and, phase by phase, slim.conv2d_transpose
 * behind conv2_tran() lib/ops.py:35-44.
 *   y[n, oy*out_sy+out_oy, ox*out_sx+out_ox, co] =
 *       post_scale * ( act( bias[co] + sum_{ky,kx,ci} x[n, oy*stride-pad_t+ky, ox*stride-pad_l+kx, ci]
 *                                                    * w[ky,kx,ci,co] ) + res[same position] ) + post_shift
 * out-of-range taps read zero (TF 'SAME').  bias / res may be NULL.
 * ------------------------------------------------------------------------------------- */
typedef struct teco_conv_desc {
  int32_t N, H, W, Cin;          /* input tensor; in_cpitch >= Cin is its channel pitch      */
  int32_t OH, OW, Cout;          /* logical output grid computed by this launch               */
  int32_t KH, KW, stride, pad_t, pad_l;
  int32_t out_H, out_W;          /* physical output tensor (y and res) spatial dims           */
  int32_t out_sy, out_oy, out_sx, out_ox;
  int32_t in_cpitch, out_cpitch; /* channel pitch (elements) of x and of y/res                */
  int32_t act;
  float post_scale, post_shift;
} teco_conv_desc;

int teco_conv2d_f32(const teco_conv_desc* d, const float* x, const float* w, const float* bias,
                    const float* res, float* y, void* stream);

/* Weight gradient of the same convolution: dw[ky,kx,ci,co] (+)= sum x(...) * dy(...), and
 * optionally db[co] (+)= sum dy.  dy is addressed like y above.  accumulate!=0 adds into dw/db. */
int teco_conv2d_wgrad_f32(const teco_conv_desc* d, const float* x, const float* dy, float* dw, float* db,
                          int accumulate, void* stream);

/* ---------------------------------------------------------------------------------------
 * bf16 tensor-core convolution (tcgen05.mma kind::f16, fp32 accumulation in TMEM).
 * 3x3, stride 1, SAME: the generator / FNet layers (lib/frvsr.py:5-41, 50-63, 79-80).
 * x: NHWC bf16 with Cin (multiple of 16); y: NHWC bf16 with Cout channels.
 * wpk: weights pre-packed by teco_pack_conv3x3_bf16 (UMMA canonical K-major core matrices).
 * res (bf16, optional) is added after the activation; out_f32 (optional, [N,H,W,out_f32_c])
 * receives post_scale*(value + res_f32) + post_shift for the first out_f32_c channels
 * (used by the generator's output stage: + bicubic, *2-1  lib/frvsr.py:85-87).
 * ------------------------------------------------------------------------------------- */
typedef struct teco_tc_desc {
  int32_t N, H, W, Cin, Cout;    /* Cin, Cout: padded channel counts (multiples of 16)       */
  int32_t act;
  int32_t mode;                  /* 0: conv3x3 s1 SAME; 1: conv_transpose 3x3 s2 SAME (4 phases) */
  int32_t out_f32_c;             /* >0: also/only write fp32 output with this many channels  */
  float post_scale, post_shift;
} teco_tc_desc;

/* transpose_layout bit 0: w is [3,3,cout,cin] (conv_transpose layout); bit 1: taps flipped (ky,kx) -> (2-ky,2-kx).
 * Value 3 with (cin, cout) = (Cout, Cin) of a forward conv packs its input-gradient convolution. */
int teco_pack_conv3x3_bf16(const float* w, int32_t cin, int32_t cout, int32_t cin_pad, int32_t cout_pad,
                           int32_t transpose_layout, const int32_t* cin_perm, void* wpk, void* stream);
int64_t teco_packed_weight_bytes(int32_t cin_pad, int32_t cout_pad);
int teco_conv3x3_tc(const teco_tc_desc* d, const void* x, const void* wpk, const float* bias,
                    const void* res, void* y, const float* res_f32, float* out_f32, void* stream);

/* Bias gradient of conv2() (slim.conv2d biases, reference lib/ops.py:47-56): db[c] (+)= sum over npix pixels of dy[pixel*cpitch + c]. */
int teco_bias_grad_f32(const float* dy, float* db, int64_t npix, int32_t C, int32_t cpitch, int32_t accumulate, void* stream);

/* Weight gradient of conv2() 3x3 stride 1 SAME on tcgen05 (the gradient tf.train.AdamOptimizer.compute_gradients takes
 * through slim.conv2d: reference lib/ops.py:47-56, lib/Teco.py:426,446-447):
 *   dw[ky][kx][ci][co] (+)= sum_p x[p + (ky-1,kx-1)][ci] * dz[p][co],  dw fp32 in TF layout [3,3,cin,cout].
 * x [N,H,W,cin_pad], dz [N,H,W,cout_pad]: NHWC bf16, channel counts padded to multiples of 64; cout % 4 == 0.
 * accumulate == 0 zeroes dw first (pixel tiles are summed with fp32 atomics). */
int teco_conv3x3_wgrad_tc(int32_t N, int32_t H, int32_t W, int32_t cin_pad, int32_t cout_pad, int32_t cin, int32_t cout,
                          const void* x, const void* dz, float* dw, int32_t accumulate, void* stream);

/* Row-linearised multi-layer 3x3 64->64 chain for 32-pixel-wide images (the metric configuration's 32x32 LR clips): the same
 * layers of generator_F (input conv + residual blocks, reference lib/frvsr.py:59-70) -- or any chain of conv2(3x3, 64->64) + bias + ReLU /
 * LeakyReLU / none + optional residual -- in ONE launch.  One tcgen05.mma covers the three horizontal taps of a kernel row
 * (N = 192, runs at the tensor floor; N = 64 cannot), the epilogue recombines them with warp shuffles; every CTA keeps its own
 * images for all layers, so there is no grid-wide dependency between layers.
 * x_in / buf_a / buf_b: NHWC bf16 [N,H,32,64] (buffer ids 0 / 1 / 2; x_in is never written).
 * plan_host: HOST array [num_layers][4] = {input buffer id, output buffer id, residual buffer id or -1, TECO_ACT_*}.
 *   A residual may be added in place (residual id == output id) but may not be the previous layer's output.
 * wpk_all: num_layers packed layers back to back (teco_pack_conv3x3_bf16, 64x64 -> 73728 bytes each); bias_all [num_layers][64]. */
int teco_conv3x3_lin_supported(int32_t N, int32_t H, int32_t W, int32_t num_layers);
int teco_conv3x3_lin_tc(int32_t N, int32_t H, int32_t W, int32_t num_layers, const void* x_in, void* buf_a, void* buf_b,
                        const void* wpk_all, const float* bias_all, const int32_t* plan_host, void* stream);

/* Developer hook: when buf != NULL every teco_conv3x3_tc CTA writes clock64() stamps to buf[cta*32 ..] (phase
 * boundaries: start, setup done, halo landed, first/last weight slab landed, MMAs issued, accumulator ready,
 * epilogue done, teardown).  buf must hold gridDim*32 int64.  Pass NULL to switch it off. */
int teco_debug_timing(void* buf);

/* ---------------------------------------------------------------------------------------
 * Warp / resample family (HBM-bound).
 * ------------------------------------------------------------------------------------- */
/* tf.contrib.image.dense_image_warp (lib/Teco.py:120,140,224,254; main.py:215):
 * out[n,y,x,c] = bilinear(img[n], (y - flow[n,y,x,0], x - flow[n,y,x,1])), border clamped. */
int teco_warp_f32(const float* img, const float* flow, float* out, int32_t N, int32_t H, int32_t W, int32_t C,
                  void* stream);
/* gradients of the above: dimg (+)= scatter, dflow = d/dflow (zero where alpha is clipped). */
int teco_warp_bwd_f32(const float* img, const float* flow, const float* dout, float* dimg, float* dflow,
                      int32_t N, int32_t H, int32_t W, int32_t C, void* stream);

/* Fused previous-HR feedback of the recurrence (main.py:201,209-216; lib/Teco.py:113,138-150):
 *   flow_hr = upscale_four(4 * pad_symmetric(flow_lr))        lib/ops.py:126-163, main.py:212-213
 *   warped  = dense_image_warp(pre_gen, flow_hr)              main.py:215
 *   dst[n,y,x, ch_off + (dy*4+dx)*3 + c] = warped[n,4y+dy,4x+dx,c] * in_scale + in_shift   (space-to-depth 4)
 * pre_gen: [N,4h,4w,3] fp32.  flow_lr: [N,fh,fw,2] fp32 with fh<=h, fw<=w (symmetric-padded to h,w).
 * dst: [N,h,w,dst_cpitch] fp32 (dst_bf16==0) or bf16 (dst_bf16!=0).  warped_out (optional): fp32 [N,4h,4w,3]. */
int teco_warp_s2d_fused(const float* pre_gen, const float* flow_lr, void* dst, float* warped_out,
                        int32_t N, int32_t h, int32_t w, int32_t fh, int32_t fw, int32_t dst_cpitch,
                        int32_t ch_off, int32_t dst_bf16, float in_scale, float in_shift, void* stream);

/* upscale_four lib/ops.py:126-163 (legacy bilinear x4), `scale` multiplies the input (4.0 for flow). */
int teco_upscale4_f32(const float* x, float* y, int32_t N, int32_t h, int32_t w, int32_t C, float scale, void* stream);
/* bicubic_four lib/ops.py:166-212.  x read with channel pitch in_cpitch (first C channels). */
int teco_bicubic4_f32(const float* x, float* y, int32_t N, int32_t h, int32_t w, int32_t C, int32_t in_cpitch,
                      void* stream);
/* tf.image.resize_images legacy bilinear to (oh,ow): lib/frvsr.py:21-22, lib/Teco.py:244. */
int teco_resize_bilinear_f32(const float* x, float* y, int32_t N, int32_t h, int32_t w, int32_t C,
                             int32_t oh, int32_t ow, void* stream);
int teco_resize_bilinear_bwd_f32(const float* dy, float* dx, int32_t N, int32_t h, int32_t w, int32_t C,
                                 int32_t oh, int32_t ow, void* stream);
/* slim.max_pool2d 2x2 s2 VALID, lib/ops.py:92-93 (+ its gradient, routed to the first max). */
int teco_maxpool2_f32(const float* x, float* y, int32_t N, int32_t H, int32_t W, int32_t C, void* stream);
int teco_maxpool2_bwd_f32(const float* x, const float* dy, float* dx, int32_t N, int32_t H, int32_t W, int32_t C,
                          void* stream);
/* bf16 NHWC variants used between tensor-core layers of FNet */
int teco_maxpool2_bf16(const void* x, void* y, int32_t N, int32_t H, int32_t W, int32_t C, void* stream);
int teco_resize2x_bf16(const void* x, void* y, int32_t N, int32_t h, int32_t w, int32_t C, void* stream);
/* tf.space_to_depth(x,4) main.py:201 / lib/Teco.py:145-148 and its inverse (gradient). */
int teco_space_to_depth4_f32(const float* x, float* y, int32_t N, int32_t h, int32_t w, int32_t C,
                             int32_t out_cpitch, int32_t ch_off, void* stream);
int teco_depth_to_space4_f32(const float* y, float* x, int32_t N, int32_t h, int32_t w, int32_t C,
                             int32_t in_cpitch, int32_t ch_off, void* stream);
/* tf_data_gaussDownby4 lib/ops.py:347-367: 9x9 sigma-1.5 Gaussian, stride 4, VALID, per channel. */
int teco_gauss_down4_f32(const float* hr, float* lr, int32_t N, int32_t H, int32_t W, int32_t C, void* stream);

/* generic elementwise y = f(a*x + b) with f in TECO_ACT_*; n elements. preprocess/deprocess lib/ops.py:13-22 */
int teco_affine_act_f32(const float* x, float* y, int64_t n, float a, float b, int32_t act, void* stream);
/* dx = dy * act'(pre) expressed on the activation OUTPUT y (relu/lrelu/tanh24/sigmoid are invertible enough). */
int teco_act_bwd_f32(const float* y, const float* dy, float* dx, int64_t n, int32_t act, void* stream);
/* fp32 <-> bf16 channel-padded copies: dst[n, c_off + c] = src[n, c] for c < C, pixel count npix. */
int teco_f32_to_bf16_pad(const float* src, void* dst, int64_t npix, int32_t C, int32_t src_cpitch,
                         int32_t dst_cpitch, int32_t c_off, float scale, float shift, void* stream);
int teco_bf16_to_f32(const void* src, float* dst, int64_t npix, int32_t C, int32_t src_cpitch, int32_t dst_cpitch,
                     void* stream);
/* dst[p, c] = float(src[p, c]) + (add ? add[p, c] : 0) for c < C; dst/add pitch = dst_cpitch */
int teco_bf16_to_f32_add(const void* src, const float* add, float* dst, int64_t npix, int32_t C, int32_t src_cpitch,
                         int32_t dst_cpitch, void* stream);
/* dst[p, c] = bf16(src[p, c]) for c < C, 0 for C <= c < dst_cpitch (whole padded row written) */
int teco_f32_to_bf16_rowpad(const float* src, void* dst, int64_t npix, int32_t C, int32_t src_cpitch, int32_t dst_cpitch,
                            void* stream);
/* save_img quantisation lib/ops.py:521-523: clip(x*255,0,255) -> uint8 (truncation), RGB order kept. */
int teco_to_u8(const float* x, uint8_t* y, int64_t n, void* stream);
/* deprocess + save_img in one pass (reference lib/ops.py:17-22 and 521-523): y01 = (x + 1) / 2 and y8 = u8(clip(255 * y01)).
   Bit-identical to teco_affine_act_f32(0.5, 0.5) followed by teco_to_u8.  y01 may be NULL (uint8 frame only). */
int teco_deprocess_u8(const float* x, float* y01, uint8_t* y8, int64_t n, void* stream);

/* ---------------------------------------------------------------------------------------
 * Batch-norm of the discriminator (lib/ops.py:88-90; lib/Teco.py:38): batch stats, no gamma, eps 1e-3.
 * stats[0..C) = mean, stats[C..2C) = biased variance (outputs).  lrelu02!=0 fuses LeakyReLU(0.2).
 * ------------------------------------------------------------------------------------- */
int teco_bn_train_f32(const float* x, const float* beta, float* y, float* stats, int64_t npix, int32_t C,
                      float eps, int32_t lrelu02, void* stream);
int teco_bn_train_bwd_f32(const float* x, const float* y, const float* dy, const float* stats, float* dx,
                          float* dbeta, int64_t npix, int32_t C, float eps, int32_t lrelu02, void* stream);

/* ---------------------------------------------------------------------------------------
 * Fused loss reductions (lib/Teco.py:316-413).  Each writes its scalar (fp32) to out[0] and, when the
 * gradient pointer is non-NULL, d(loss*gscale)/d(a) elementwise (same shape as a).
 * ------------------------------------------------------------------------------------- */
/* mean over pixels of sum_c (a-b)^2 : content loss :320-322, warp loss :329-331 */
int teco_loss_l2_f32(const float* a, const float* b, float* out, float* da, int64_t npix, int32_t C, float gscale,
                     void* stream);
/* mean |a-b| over all elements: ping-pong :364-367; mean over pixels of sum_c|a-b| when per_pixel!=0: layer loss :295-296 */
int teco_loss_l1_f32(const float* a, const float* b, float* out, float* da, float* db, int64_t npix, int32_t C,
                     int32_t per_pixel, float gscale, void* stream);
/* VGG cosine term :346-349 on raw features f,g [npix,C]: 1 - mean_pix( <f,g> / (|f|_eps |g|_eps) ) */
int teco_loss_cosine_f32(const float* f, const float* g, float* out, float* df, int64_t npix, int32_t C, float gscale,
                         void* stream);
/* per-pixel channel L2 normalisation of VGG features, lib/Teco.py:19-21: y = f / sqrt(sum_c f^2 + 1e-12) */
int teco_l2norm_channels_f32(const float* f, float* y, int64_t npix, int32_t C, void* stream);
/* GAN terms :376,394-399 on sigmoid outputs.  out[0]=mean -log(df+eps)  out[1]=mean -(log(1-df+eps)+log(dr+eps))
 * out[2]=mean log(dr+eps)  out[3]=mean dr  out[4]=mean df.  Gradients w.r.t. the sigmoid OUTPUTS:
 * g_adv = d(out0*s_adv)/d df ; g_dis_f, g_dis_r = d(out1*s_dis)/d(df,dr). */
int teco_loss_gan_f32(const float* d_fake, const float* d_real, float* out, float* g_adv, float* g_dis_f,
                      float* g_dis_r, int64_t n, float eps, float s_adv, float s_dis, void* stream);

/* tf.train.AdamOptimizer (lib/Teco.py:425,439-440), multi-tensor over one flat buffer of n floats.
 * lr_t = lr*sqrt(1-b2^t)/(1-b1^t) is computed by the caller.  gscale multiplies g (1/world after allreduce). */
int teco_adam_f32(float* p, float* m, float* v, const float* g, int64_t n, float lr_t, float b1, float b2, float eps,
                  float gscale, void* stream);

/* ---------------------------------------------------------------------------------------
 * Evaluation metrics on the device (SURVEY 8f-3; reference metrics.py).  tgt / out: uint8 RGB frames
 * [N,tH,tW,3] / [N,oH,oW,3] (the decoded PNGs; to_uint8(x,0,255) metrics.py:57-61 is the identity on them).
 * (y0,x0,h,w) is the crop_8x8 window of metrics.py:77-92, the same offsets in both frames (the reference
 * first cuts the output to the target size, metrics.py:134-135, which a window inside both frames covers).
 * acc: N x 4 doubles {sum (Yt-Yp)^2, ~bits(min Yp), bits(max Yp), sum of SSIM map} -- 8-byte slots, the
 * min / max of Y_pred held as (complemented) bit patterns so that zero is neutral for every slot.
 * Y = 16 + 0.2568 R + 0.5041 G + 0.0979 B in float64, metrics.py:37-55 (_rgb2ycbcr, maxVal 255).
 * ------------------------------------------------------------------------------------- */
/* psnr() metrics.py:63-70: zeroes acc, then fills slots 0..2.  PSNR_n = 20 log10(255 / sqrt(acc[n][0] / (h*w))). */
int teco_metrics_psnr_y_u8(const uint8_t* tgt, int32_t tH, int32_t tW, const uint8_t* out, int32_t oH, int32_t oW,
                           int32_t N, int32_t y0, int32_t x0, int32_t h, int32_t w, double* acc, void* stream);
/* ssim() metrics.py:72-75 = skimage compare_ssim(Y_true, Y_pred, data_range = max Yp - min Yp): 7x7 uniform
 * window, sample covariance, K1 0.01, K2 0.03, mean over the (h-6) x (w-6) positions whose window lies inside.
 * Needs slots 1..2 from teco_metrics_psnr_y_u8 on the same stream; adds into slot 3.
 * SSIM_n = acc[n][3] / ((h-6)*(w-6)).  h or w below 7 -> TECO_E_INVALID (skimage raises ValueError). */
int teco_metrics_ssim_y_u8(const uint8_t* tgt, int32_t tH, int32_t tW, const uint8_t* out, int32_t oH, int32_t oW,
                           int32_t N, int32_t y0, int32_t x0, int32_t h, int32_t w, double* acc, void* stream);

/* ---------------------------------------------------------------------------------------
 * tOF (metrics.py:135-169): cv2.cvtColor(RGB2GRAY) and cv2.calcOpticalFlowFarneback with flags = 0 on the device,
 * batched over all frame pairs of a scene.  The stages are pinned against cv2 in tests/golden/tof_ref.py.
 * ------------------------------------------------------------------------------------- */
/* grey[n][y][x] = (9798 R + 19235 G + 3735 B + 2^14) >> 15 (cv2's COLOR_RGB2GRAY on uint8, bit for bit) of the
 * top-left h x w of frame n of rgb [N,H,W,3]: the reference's cut of the result to the target size, metrics.py:139-140. */
int teco_grey_u8(const uint8_t* rgb, int32_t N, int32_t H, int32_t W, int32_t h, int32_t w, uint8_t* grey, void* stream);
/* Host only: workspace bytes teco_farneback_flow needs for F frames and P pairs of H x W, or TECO_E_INVALID for bad sizes
 * (F, P in 1..65535, H in 2..65535, W >= 2, H*W < 2^31, 0 < pyr_scale < 1, levels >= 0). */
int64_t teco_farneback_workspace_bytes(int32_t F, int32_t P, int32_t H, int32_t W, double pyr_scale, int32_t levels);
/* flow[p] = calcOpticalFlowFarneback(grey[pairs_host[2p]], grey[pairs_host[2p+1]], None, pyr_scale, levels, winsize,
 * iterations, poly_n, poly_sigma, flags) for grey [F,H,W] uint8 and flow [P,H,W,2] float32 (dx, dy).  Each frame's
 * polynomial expansion is computed once per level, however many pairs use it.  Supported: flags = 0, odd winsize up to 15,
 * poly_n 1..7; anything else is TECO_E_INVALID.  pairs_host is read before the call returns.  A pair's flow is the same
 * bits whatever else is in the batch. */
int teco_farneback_flow(const uint8_t* grey, int32_t F, int32_t H, int32_t W, const int32_t* pairs_host, int32_t P,
                        double pyr_scale, int32_t levels, int32_t winsize, int32_t iterations, int32_t poly_n,
                        double poly_sigma, int32_t flags, void* workspace, int64_t workspace_bytes, float* flow, void* stream);
/* sums[p] = sum over the window (y0,x0,h,w) of |flow_t[p] - flow_o[p]|_2 in float64, both [P,H,W,2]; tOF_p = sums[p] / (h*w).
 * Overwrites sums; no atomics, so the result does not depend on scheduling. */
int teco_tof_sums(const float* flow_t, const float* flow_o, int32_t P, int32_t H, int32_t W, int32_t y0, int32_t x0,
                  int32_t h, int32_t w, double* sums, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TECO_H_ */

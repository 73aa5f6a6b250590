/*
 * ssr_b200.h -- C ABI of the B200-native multi-frame ESRGAN engine (libssr_b200.so).
 *
 * The reference (allenai/satlas-super-resolution) has no native layer and no FFI: every operator on
 * its hot path is a torch call that dispatches to cuDNN / ATen (SURVEY.md section 2a).  The entry
 * points below are the operators that replace those calls; each one names the reference call site
 * (file:line under /root/reference) whose arithmetic it takes over.  INTEGRATION.md shows the
 * ctypes binding a maintainer adds on the reference side.
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless it says "host";
 *   - activations are NHWC bf16, "pix_stride" = elements between consecutive pixels (lets a conv
 *     read / write a channel slice of a wider dense-block buffer, which is how torch.cat disappears);
 *   - all calls are asynchronous on `stream` (a cudaStream_t passed as void*), allocation free and
 *     never synchronise; return 0 on success, a negative SSR_E_* code otherwise (ssr_last_error()
 *     gives the text).  There is no CPU fallback: without a GPU the calls fail with SSR_E_CUDA.
 */
#ifndef SSR_B200_H_
#define SSR_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SSR_OK 0
#define SSR_E_ARG -1   /* invalid argument / unsupported shape */
#define SSR_E_CUDA -2  /* CUDA runtime / driver error (including "no device") */

/* residual / output element kinds */
#define SSR_NONE 0
#define SSR_BF16 1
#define SSR_F32 2
/* f32, channel-quad planar: element (pixel p, channel c) at [((c / 4) * P + p) * 4 + c % 4], P = n_img*h*w of the call.
 * For buffers only epilogues touch (running gradients, the f32 trunk): a warp's 32 pixels x 4 channels are 512
 * contiguous bytes, where NHWC gives every lane its own cache line.  The pix_stride of such an operand is ignored. */
#define SSR_F32_PLANAR4 3

/* f32 output modes of ssr_conv_tc */
#define SSR_OUT32_NONE 0
#define SSR_OUT32_NHWC 1        /* store   out32[pix*stride + c]              */
#define SSR_OUT32_NHWC_ATOMIC 2 /* red.add out32[pix*stride + c]  (split-K)   */
#define SSR_OUT32_NCHW 3        /* store   out32[((n*cout + c)*H + y)*W + x]  */
#define SSR_OUT32_PLANAR4 4     /* store   out32 in the SSR_F32_PLANAR4 layout */
/* out32 (planar) is ALSO res1 (res1 == out_f32, SSR_F32_PLANAR4, s1 == 1): a running sum.  Channels that produce a
 * bf16 output (>= out_lo) are read, added and stored as with SSR_OUT32_PLANAR4; all others are accumulated with a
 * vector reduction (red.global.add.v4.f32) -- no dependent load in the epilogue.  One writer per element: deterministic. */
#define SSR_OUT32_PLANAR4_ACC 5

/* weight packing modes */
#define SSR_PACK_FWD 0   /* B[n=cout][k=cin], taps as stored          */
#define SSR_PACK_DGRAD 1 /* B[n=cin][k=cout], taps flipped (conv^T)   */
#define SSR_PACK_FWD_GEMM 2   /* 1x1 form over im2col columns: B[n=cout][k'=(ky*R+kx)*cin+ci]          */
#define SSR_PACK_DGRAD_GEMM 3 /* 1x1 form producing dcol:      B[n=k'][k=cout]                           */
/* input gradient of a 4 x 4 stride-2 conv as four 2 x 2 convs over dY, one per output parity (oy, ox):
 * dst[class = oy*2 + ox][cout chunk][b][a][n = cin][64], tap (a, b) of class (oy, ox) = w[k][n][ky][kx] with
 * ky = oy ? 2 - 2a : 3 - 2a, kx = ox ? 2 - 2b : 3 - 2b (dx[2u+oy] collects dy[u - pad + a], pad = 1 - oy) */
#define SSR_PACK_DGRAD_S2 4
/* OR-ed into SSR_PACK_FWD / SSR_PACK_DGRAD (ssr_pack_conv_weight only): pack the ROUNDING RESIDUAL w - bf16(w) instead of bf16(w) --
 * the low half of the split-bf16 operand pair of the tight-parity forward (a = a_hi + a_lo, w = w_hi + w_lo,
 * a*w ~ a_hi*w_hi + a_lo*w_hi + a_hi*w_lo: three bf16 launches summed in f32, relative error ~2^-16 instead of 2^-8) */
#define SSR_PACK_LO 16

const char* ssr_last_error(void);
int ssr_abi_version(void);
/* number of kernels this library has launched since load (bench.py's gpu_launches) */
int64_t ssr_launch_count(void);
/* per-launch CUDA-event timing of the tensor-core kernels for the roofline figures: start, run the step eagerly, stop ->
 * total ms and launch count per class (synchronises).  Classes: 0 = single-launch conv (conv_tc_kernel), 1 = weight gradient
 * (wgrad_tc / wgrad9_tc, one problem per launch), 2 = dense-block forward chain (conv_chain_kernel), 3 = dense-block
 * input-gradient chain (conv_chain_kernel), 4 = batched dense-block weight gradient (wgrad9_tc_batched_kernel). */
#define SSR_PROFILE_CLASSES 5
int ssr_profile_start(void);
int ssr_profile_stop(double* ms, int64_t* count, int32_t n_classes);

/*
 * Implicit-GEMM convolution, R x R (R = 1 or 3), stride 1, zero padding (R-1)/2, on tcgen05 tensor
 * cores: NHWC bf16 tiles -> shared memory by TMA (128B swizzle) -> tcgen05.mma (bf16 x bf16 -> f32 in
 * TMEM) -> fused epilogue.  Replaces nn.Conv2d(k=3,s=1,p=1) forward at ssr/archs/rrdbnet_arch.py:37-44,
 * :122-136 and ssr/archs/discriminator_arch.py:44-69 (conv0, conv4..conv9), its input-gradient
 * (same kernel, SSR_PACK_DGRAD weights) and, with R = 1, any K-major GEMM (used for the strided
 * discriminator convs through im2col and for weight gradients).
 *
 * Epilogue, per output element (p = pixel, c = channel):
 *   v = acc + bias[c]; if (act) v = v > 0 ? v : 0.2 v;           // LeakyReLU(0.2), rrdbnet_arch.py:33
 *   v = s0*v + s1*res1[p,c] + s2*res2[p,c];                      // x5*0.2 + x (:44), out*0.2 + x (:68)
 *   out_f32[...] (=|+=) v                                        // unmasked (a running f32 gradient sum)
 *   if (c >= mask_lo) v *= (mask[p,c] > 0 ? 1 : 0.2 | 0);        // LeakyReLU / ReLU backward on a saved output
 *   out_bf16[p,c] = bf16(v)
 */
typedef struct ssr_conv_tc_args {
  /* input activation, NHWC bf16: x[((n*h + y)*w + x)*x_pix_stride + c], c in [0, cin) */
  const void* x;
  int32_t n_img, h, w;
  int32_t x_pix_stride;
  int32_t cin; /* channels read; multiple of 16; x and x_pix_stride*2 must be 16-byte aligned */
  /* weights packed by ssr_pack_conv_weight: [cin_chunks][R][R][n_pad][64] bf16 */
  const void* w_packed;
  int32_t r;     /* 1 or 3 */
  int32_t cout;  /* valid output channels */
  int32_t n_pad; /* padded output channels in w_packed (multiple of 16) */
  /* epilogue */
  const float* bias; /* [cout] or NULL */
  int32_t act;       /* 1 = LeakyReLU(0.2), 2 = ReLU */
  float s0;
  const void* res1;
  int32_t res1_kind; /* SSR_NONE / SSR_BF16 / SSR_F32 / SSR_F32_PLANAR4 */
  int32_t res1_pix_stride;
  float s1;
  const void* res2;
  int32_t res2_kind;
  int32_t res2_pix_stride;
  float s2;
  const void* mask; /* bf16 NHWC, or NULL */
  int32_t mask_pix_stride;
  int32_t mask_lo;   /* first output channel the mask applies to; mask is indexed [p*stride + c] */
  int32_t mask_relu; /* 0: LeakyReLU(0.2) derivative, 1: ReLU derivative */
  void* out_bf16;    /* NHWC bf16 or NULL */
  int32_t out_pix_stride;
  float* out_f32;
  int32_t out32_mode; /* SSR_OUT32_* */
  int32_t out32_pix_stride;
  /* tiling knobs, 0 = choose automatically */
  int32_t n_tile; /* output channels per CTA, multiple of 16, <= 256 */
  int32_t mt;     /* 128-pixel M tiles per CTA: 1 or 2 */
  int32_t splits; /* split the cin chunks over this many CTAs (needs SSR_OUT32_NHWC_ATOMIC) */
  int32_t res1_cmax; /* res1 is added only to channels < res1_cmax (0 = all); multiple of 16 */
  int32_t out_lo;    /* out_bf16 (and mask) only cover channels >= out_lo (multiple of 16): an input-gradient conv of a dense
                      * block adds into all its f32 channels but only its top slot is read again as bf16 */
  float* bias_grad;  /* bias_grad[c - out_lo] += bias_grad_scale * sum_p (the value out_bf16 receives), or NULL: the bf16 output
                      * of an input-gradient conv is the dY of the conv below it, its pixel sum that conv's bias gradient */
  float bias_grad_scale;
  /* r == 4: the 4 x 4 stride-2 pad-1 convolution (conv1..conv3 of ssr/archs/discriminator_arch.py:30-32) as an implicit GEMM --
   * stride must be 2, (h, w) is the INPUT size, the output is (h/2, w/2); weights packed with r = 4.
   * r == 2: one parity class of its transposed convolution (the input gradient): a 2 x 2 stride-1 conv over dY of size (h, w) whose
   * box origin is shifted by (pad_y, pad_x) in {0, 1} and whose output pixel (y, x) is stored at (2y + out_oy, 2x + out_ox) of
   * the (2h, 2w) image out_bf16 / mask / residuals describe; weights: class out_oy * 2 + out_ox of an SSR_PACK_DGRAD_S2 operand. */
  int32_t stride;
  int32_t pad_y, pad_x;
  int32_t out_oy, out_ox;
} ssr_conv_tc_args;

int ssr_conv_tc(const ssr_conv_tc_args* args, void* stream);

/*
 * n layers in ONE launch (replaces the five consecutive self.convK(...) calls of ResidualDenseBlock.forward,
 * ssr/archs/rrdbnet_arch.py:36-43, and autograd's matching five input-gradient convolutions).  Layer i may read
 * anything layers < i of the same call wrote; all layers share (n_img, h, w, r), have n_pad <= 128 and splits <= 1.
 * Results are identical to n ssr_conv_tc calls in order; ineligible chains are executed exactly that way.
 * A chain with the channel pattern of a ResidualDenseBlock (layer i reads channels [0, 64 + 32 i) of ONE buffer and appends its
 * 32 outputs there; f32 operands channel-quad planar) over 32-row images runs with the 192-channel tile resident in shared
 * memory: activations are loaded once, halo columns travel through distributed shared memory, only weights stream.  In that
 * form the intermediate layers may pass out_bf16 == NULL (inference: x1..x4 are never written to global memory).
 */
int ssr_conv_tc_chain(const ssr_conv_tc_args* args, int32_t n, void* stream);
/*
 * Chain whose layers add into ONE f32 accumulator per pixel that stays in tensor memory for the whole launch (the five
 * input-gradient convs of a ResidualDenseBlock: autograd's running gradient of the dense buffer).  Layer i adds its cout_i
 * channels at channel offset 0 (cout_0 is the widest); after the add it EMITS the channels >= out_lo_i of the running sum:
 * v = sum + s1*res1 + s2*res2 -> out_f32 (unmasked), mask -> out_bf16, bias_grad.  Channels below out_lo_i stay in tensor
 * memory and are never stored; layer i+1 must satisfy cout_{i+1} <= out_lo_i.  Every layer: s0 == 1 (fold scales into the
 * packed weights), no bias / activation, cout % 16 == 0.  Needs images of <= 8 pixel tiles (ssr_conv_tc_chain_acc_supported);
 * there is no plain-launch fallback -- unsupported shapes return SSR_E_ARG.
 */
int ssr_conv_tc_chain_acc(const ssr_conv_tc_args* args, int32_t n, void* stream);
/* 1 if ssr_conv_tc_chain_acc can run this geometry (host arithmetic only, no device needed), else 0 */
int ssr_conv_tc_chain_acc_supported(int32_t n_img, int32_t h, int32_t w, int32_t widest_cout);
/* How many consecutive ResidualDenseBlocks (rrdbnet_arch.py:37-44, 63-68) ONE resident launch may take for this geometry: the caller
   concatenates that many blocks' five layers in one ssr_conv_tc_chain / ssr_conv_tc_chain_acc call (each block's last layer must store
   its bf16 output exactly where the next block's first layer reads its input).  1 = one block per call ($SSR_RDB_FUSE overrides). */
int ssr_rdb_resident_max_blocks(int32_t n_img, int32_t h, int32_t w);
/* diagnostics: how many chains ran as the shared-memory-resident dense-block kernel (32-row images, 8 | w <= 64, the channel pattern
 * of ResidualDenseBlock; SSR_CONV_RESIDENT=0 disables it) */
int64_t ssr_debug_resident_launches(void);
/* diagnostics: how many ssr_conv_tc launches took path `which`: 0 = halo tile + stationary weights (3 x 3, cin % 64 == 0, enough
 * tiles; SSR_CONV_HALO=0 disables), 1 = the short epilogue (SSR_CONV_LEAN=0 disables), 2 = stationary weights in the streamed form */
int64_t ssr_debug_conv_path_count(int32_t which);
/* diagnostics: with SSR_CHAIN_TIMELINE=1 in the environment every chained launch records clock64 stamps
 * [cta][layer (5)][8 events]; copies the first n_ctas (<= 512) rows of the LAST launch to host memory (synchronises). */
int ssr_debug_chain_timeline(long long* host_out, int32_t n_ctas);

/* bytes of a packed weight buffer for (cin, cout, r) -> n_pad is written back */
int64_t ssr_packed_weight_bytes(int32_t cin, int32_t cout, int32_t r, int32_t* n_pad);

/*
 * Pack f32 OIHW weights (the layout of nn.Conv2d.weight, what the reference state_dict holds) into the
 * bf16 K-major tile layout ssr_conv_tc reads.  `inv_scale` (device, 1 float, may be NULL) divides the
 * weights: it is sigma of spectral_norm (discriminator_arch.py:30-39).  For SSR_PACK_DGRAD the roles
 * of cin/cout swap in the packed buffer (n = cin, k = cout) and the taps are mirrored.
 * cin_pad: channels of the activation buffer the packed weights will be used with (>= cin, mult of 16).
 */
int ssr_pack_conv_weight(const float* w_oihw, int32_t cout, int32_t cin, int32_t r, int32_t mode,
                         const float* inv_scale, void* packed, int32_t k_pad, int32_t n_pad,
                         void* stream);

/* ---------------------------------------------------------------------------------------------------
 * Layout / resampling kernels (HBM-bound, NHWC bf16, 16-byte vectorised).
 * ------------------------------------------------------------------------------------------------- */

/* Planar NCHW (u8: src_kind 0, f32: src_kind SSR_F32) -> NHWC bf16 with channels [c, c_pad) zero-filled.
 * v = src*scale, then (v - mean[c]) * inv_std[c] when mean != NULL.  Replaces `.float()/255` of
 * ssr/models/ssr_esrgan_model.py:106-108 and the ImageNet input-norm of basicsr PerceptualLoss. */
int ssr_ingest_nchw(const void* src, int32_t src_kind, void* dst_bf16, int32_t dst_pix_stride, int32_t b, int32_t c,
                    int32_t h, int32_t w, int32_t c_pad, float scale, const float* mean, const float* inv_std,
                    void* stream);
/* The same with pixel_unshuffle(x, factor) fused (ssr/archs/arch_util.py:769-785, called at rrdbnet_arch.py:117-120 for
 * scale 1 / 2): dst[n, y, x, c*f*f + i*f + j] = src[n, c, y*f + i, x*f + j] * scale, dst is [b, h/f, w/f, c_pad]. */
int ssr_ingest_nchw_unshuffle(const float* src, void* dst_bf16, int32_t dst_pix_stride, int32_t b, int32_t c, int32_t h, int32_t w,
                              int32_t factor, int32_t c_pad, float scale, void* stream);
/* NHWC bf16 channel slice -> planar NCHW f32 (dst = or += src*scale) */
int ssr_egress_nchw(const void* src_bf16, int32_t src_pix_stride, float* dst, int32_t b, int32_t c, int32_t h, int32_t w,
                    float scale, int32_t accumulate, const float* ch_scale /* [c] or NULL */, void* stream);
/* Inference egress: uint8(clamp(v,0,1)*255) of an f32 NCHW batch, image i pasted at tile (i/grid_cols, i%grid_cols) of an
 * HWC uint8 canvas -- clamp / transpose / astype(uint8) of ssr/infer.py:61-64 and `stitch` of ssr/utils/infer_utils.py:41-60. */
int ssr_f32_nchw_to_u8_canvas(const float* src, void* dst_u8, int32_t b, int32_t c, int32_t h, int32_t w, int32_t canvas_w,
                              int32_t grid_cols, int32_t first_index, void* stream);
/* F.interpolate(mode='nearest', scale_factor=factor): rrdbnet_arch.py:127-128, ssr_esrgan_model.py:133 */
int ssr_upsample_nearest(const void* src, int32_t src_pix_stride, void* dst, int32_t dst_pix_stride, int32_t b, int32_t h,
                         int32_t w, int32_t c, int32_t factor, void* stream);
int ssr_upsample_nearest_bwd(const void* dy, int32_t dy_pix_stride, void* dx, int32_t dx_pix_stride, int32_t b, int32_t h,
                             int32_t w, int32_t c, int32_t factor, const void* lrelu_mask /* or NULL */,
                             int32_t mask_pix_stride, void* stream);
/* F.interpolate(scale_factor=2, mode='bilinear', align_corners=False): discriminator_arch.py:50,55,60 */
int ssr_upsample_bilinear2x(const void* src, int32_t src_pix_stride, const void* src2 /* added to src, or NULL */,
                            int32_t src2_pix_stride, void* dst, int32_t dst_pix_stride, int32_t b, int32_t h, int32_t w,
                            int32_t c, void* stream);
int ssr_upsample_bilinear2x_bwd(const void* dy, int32_t dy_pix_stride, void* dx, int32_t dx_pix_stride, int32_t b,
                                int32_t h, int32_t w, int32_t c, void* stream);

/* One launch packs every conv of a network (descs live in DEVICE memory). */
typedef struct ssr_pack_desc {
  const float* w;         /* OIHW f32 */
  void* dst;              /* packed bf16 */
  const float* inv_scale; /* spectral-norm sigma (device) or NULL */
  int32_t cout, cin, r, mode, k_pad, n_pad;
} ssr_pack_desc;
int ssr_pack_conv_weights_batched(const ssr_pack_desc* descs_device, int32_t n_layers, int32_t has_gemm_forms, void* stream);
/* The same work as a flat list, one 8-row x 64-K tile of one operand per thread block: work_device = n_work pairs {descriptor index,
 * tile index < ssr_pack_tile_count(k_pad, n_pad)} (SSR_PACK_FWD / DGRAD / DGRAD_S2 descriptors only). */
int32_t ssr_pack_tile_count(int32_t k_pad, int32_t n_pad);
int ssr_pack_conv_weights_tiled(const ssr_pack_desc* descs_device, const int32_t* work_device, int32_t n_work, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * Weight gradient on tensor cores (MN-major operands straight from the NHWC buffers).
 *   out(ky*R + kx, cx, cy) += scale * sum_p x[p + (ky-pad, kx-pad), cx] * dy[p, cy]      (f32, red.add.v4)
 * `out` is an f32 scratch accumulator of R*R * out_cx_rows * out_stride floats (out_stride = cy rounded up to 4), stored
 * channel-quad planar so that the reduction of a warp's 32 cx rows is 512 contiguous bytes:
 *   element (tap, cx, cy) at [((cy / 4) * R*R*out_cx_rows + tap*out_cx_rows + cx) * 4 + cy % 4].
 * The caller zeroes it before the first accumulation; ssr_wgrad_unpack scatters it into the OIHW gradient of nn.Conv2d.weight.
 * Replaces the wgrad half of autograd for every nn.Conv2d of rrdbnet_arch.py / discriminator_arch.py.
 * ------------------------------------------------------------------------------------------------- */
typedef struct ssr_wgrad_tc_args {
  const void* x; /* NHWC bf16 conv input (channel slice) */
  int32_t n_img, h, w;
  int32_t x_pix_stride;
  int32_t cx; /* input channels  */
  const void* dy; /* NHWC bf16 gradient of the conv output */
  int32_t dy_pix_stride;
  int32_t cy; /* output channels */
  int32_t r;  /* 1 or 3 */
  float* out;
  int32_t out_cx_rows;
  int32_t out_stride;
  float scale;
  int32_t splits; /* 0 = auto */
} ssr_wgrad_tc_args;
int ssr_wgrad_tc(const ssr_wgrad_tc_args* args, void* stream);
/* n independent problems (e.g. the five convs of one ResidualDenseBlock) in one launch where the shapes allow it */
int ssr_wgrad_tc_batched(const ssr_wgrad_tc_args* args, int32_t n, void* stream);
int ssr_wgrad_unpack(const float* acc, int32_t cx_rows, int32_t acc_stride, float* grad_oihw, int32_t cout, int32_t cin,
                     int32_t r, float scale, int32_t accumulate, void* stream);
/* every conv of a network in one launch (device-resident table) */
typedef struct ssr_unpack_desc {
  const float* acc;
  float* grad;
  int32_t cx_rows, acc_stride, cout, cin, r, accumulate;
  float scale;
  int32_t pad_;
} ssr_unpack_desc;
int ssr_wgrad_unpack_batched(const ssr_unpack_desc* descs_device, int32_t n_layers, void* stream);
/* out[c] += scale * sum_p dy[p*stride + c]   (bias gradient) */
int ssr_bias_grad(const void* dy_bf16, int32_t dy_pix_stride, int64_t npix, int32_t c, float* out, float scale, void* stream);
/* grouped: channel c accumulates into outs_device[c / group_ch][c % group_ch] (one launch for the four 32-channel dY slots
 * of a ResidualDenseBlock) */
int ssr_bias_grad_groups(const void* dy_bf16, int32_t dy_pix_stride, int64_t npix, int32_t c, int32_t group_ch,
                         float* const* outs_device, float scale, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * Training-step kernels (HBM-bound).  Losses accumulate into device scalars the caller zeroes.
 * ------------------------------------------------------------------------------------------------- */
/* im2col / col2im for the 4x4 stride-2 discriminator convs (discriminator_arch.py:30-32): col is
 * [b*oh*ow][k*k*c] bf16 with (ky, kx, c) order; col2im is the gather-form adjoint and can fuse the LeakyReLU
 * derivative taken from the saved activation `lrelu_mask` (may be NULL). */
int ssr_im2col(const void* x, int32_t x_pix_stride, void* col, int32_t b, int32_t h, int32_t w, int32_t c, int32_t k, int32_t s,
               int32_t p, void* stream);
int ssr_col2im(const void* dcol, void* dx, int32_t dx_pix_stride, int32_t b, int32_t h, int32_t w, int32_t c, int32_t k, int32_t s,
               int32_t p, const void* add /* bf16 NHWC added before the mask, or NULL */, int32_t add_pix_stride,
               const void* lrelu_mask, int32_t mask_pix_stride, void* stream);
/* y = a*x1 + b*x2 (x2 may be NULL), times the LeakyReLU(0.2) (mask_relu=0) or ReLU (1) derivative from `mask` (may be NULL) */
int ssr_axpby(const void* x1, int32_t s1, float a, const void* x2, int32_t s2, float b, const void* mask, int32_t sm,
              int32_t mask_relu, void* y, int32_t sy, int64_t npix, int32_t c, void* stream);
/* Tight-parity (split-bf16) mode (tight.py), the conv epilogue as its own kernel: v = act(s1 + s2 + s3 + bias) * s0 + w1 * r1 + w2 * r2
 * over NHWC f32 channel slices [npix, c] with their own pixel strides (s2, s3, bias, r1, r2 may be NULL; act: 0 none, 1 LeakyReLU(0.2));
 * out_f32[pix * out32_stride + ch] = v (may be NULL); then v *= LeakyReLU'(mask) with mask the bf16 forward activation (may be NULL);
 * hi[pix * out_stride + ch] = bf16(v), lo[...] = bf16(v - hi) for ch < c and zeros for c <= ch < c_pad (hi / lo may be NULL). */
int ssr_split_finish(const float* s1, const float* s2, const float* s3, int32_t sum_stride, int64_t npix, int32_t c, const float* bias,
                     int32_t act, float s0, const float* r1, int32_t r1_stride, float w1, const float* r2, int32_t r2_stride, float w2,
                     const void* mask_bf16, int32_t mask_stride, float* out_f32, int32_t out32_stride, void* hi, void* lo,
                     int32_t out_stride, int32_t c_pad, void* stream);
/* adjoint of the nearest x2 upsample in f32 (NHWC [b, 2h, 2w, c] -> [b, h, w, c], 2 x 2 sums): the split-bf16 backward */
int ssr_sum_pool2x2_f32(const float* src, float* dst, int32_t b, int32_t h, int32_t w, int32_t c, void* stream);
/* VGG19 feature extractor pieces of basicsr PerceptualLoss (ssr_esrgan_model.py:154): x holds 2b images (generated | gt) */
int ssr_maxpool_relu(const void* x, void* y, int32_t b, int32_t h, int32_t w, int32_t c, void* stream);
int ssr_feat_grad(const void* x, const void* dpool, void* dx, int32_t b, int32_t h, int32_t w, int32_t c, float l1_scale, void* stream);
int ssr_feat_l1(const void* x, int64_t n_half, float scale, float* loss, void* stream);
/* basicsr L1Loss(mean)*weight (ssr_esrgan_model.py:148): loss += ..., grad (=|+=) weight*sign(a-b)/n */
int ssr_l1_loss(const float* a, const float* b, int64_t n, float weight, float* loss, float* grad, int32_t accumulate, void* stream);
/* SSIMLoss (ssr/losses/basic_loss.py:50-60, call site ssr_esrgan_model.py:163-164) = kornia.losses.ssim_loss(x, gt, window_size=5):
   loss += weight * mean(clamp((1 - ssim) / 2, 0, 1)) over `planes` f32 planes [h, w]; grad (=|+=) dLoss/dx (y is a constant).
   scratch: 3 * planes * h * w floats, needed only with grad. */
int ssr_ssim_loss(const float* x, const float* y, int32_t planes, int32_t h, int32_t w, float weight, float* loss, float* grad,
                  int32_t accumulate, float* scratch, void* stream);
/* basicsr GANLoss('vanilla') = BCEWithLogitsLoss against a constant target (ssr_esrgan_model.py:182,218,224) */
int ssr_bce_logits(const float* x, int64_t n, float target, float weight, float* loss, float* mean_logit, float* grad, void* stream);
/* torch.cat((img, F.interpolate(lr, scale_factor=factor)), 1) -> NHWC bf16 (ssr_esrgan_model.py:133,176,208-210) */
int ssr_disc_input(const float* img, int32_t ci, const void* lr, int32_t lr_pix_stride, int32_t cl, int32_t factor, void* out,
                   int32_t out_pix_stride, int32_t b, int32_t h, int32_t w, void* stream);

/* the same with a third group appended: [img | nearest(lr) | extra] -- `extra` (planar f32 [b, ce, h, w]) is the old_hr image of
 * ssr_esrgan_model.py:112-114, 171-174, 202-207 */
int ssr_disc_input_ex(const float* img, int32_t ci, const void* lr, int32_t lr_pix_stride, int32_t cl, int32_t factor,
                      const float* extra, int32_t ce, void* out, int32_t out_pix_stride, int32_t b, int32_t h, int32_t w, void* stream);

/* torch.nn.utils.spectral_norm, batched over the 8 normalised convs of the discriminator (device-resident table) */
typedef struct ssr_sn_desc {
  const float* w; /* weight_orig viewed [rows = cout][cols = cin*k*k] */
  float* u;
  float* v;
  float* sigma;   /* out: u^T W v */
  float* scratch; /* cols + rows + 4 floats, zero-initialised once */
  float* geff;    /* gradient w.r.t. weight_orig / sigma (input of ssr_spectral_norm_bwd) */
  float* grad;    /* gradient of weight_orig (accumulated) */
  int32_t rows, cols;
} ssr_sn_desc;
int ssr_spectral_norm(const ssr_sn_desc* descs_device, int32_t n_layers, int32_t power_iteration, float eps, void* stream);
int ssr_spectral_norm_bwd(const ssr_sn_desc* descs_device, int32_t n_layers, void* stream);

/* basicsr USMSharp (ssr_esrgan_model.py:31,109): separable Gaussian (host taps), reflect padding; scratch = 3*planes*h*w floats */
int ssr_usm_sharp(const float* img, float* out, float* scratch, int32_t planes, int32_t h, int32_t w, const float* gauss_host,
                  int32_t taps, float weight, float threshold, void* stream);
int ssr_u8_to_f32(const void* src, float* dst, int64_t n, float scale, void* stream);
/* torch.optim.Adam step (+ basicsr model_ema when ema != NULL) over flat f32 buffers, one launch */
int ssr_adam_ema(float* p, const float* g, float* m, float* v, float* ema, int64_t n, float lr, float beta1, float beta2, float eps,
                 float weight_decay, int32_t step, float ema_decay, float grad_scale,
                 const float* dev_hyper /* device [lr, 1-b1^t, sqrt(1-b2^t), t, b1, b2] overriding lr/step (graph replay), or NULL */,
                 void* stream);
/* basicsr model_ema alone (ssr_esrgan_model.py:230-231 on an iteration without a generator step): ema = decay*ema + (1-decay)*p */
int ssr_ema_update(float* ema, const float* p, int64_t n, float decay, void* stream);
/* t += 1 and refresh the two bias corrections in a device-resident hyper block (recorded inside the step's CUDA graph) */
int ssr_adam_tick(float* hyper_dev, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * Validation metrics (ssr/models/ssr_esrgan_model.py:269-352 computes them per image on the host).
 * ------------------------------------------------------------------------------------------------- */
/* basicsr tensor2img(rgb2bgr, uint8, min_max=(0,1)): uint8(round_half_even(clamp(v, 0, 1) * 255)), f32 NCHW -> u8 HWC per image */
int ssr_f32_nchw_to_u8_hwc(const float* src, void* dst_u8, int32_t b, int32_t c, int32_t h, int32_t w, int32_t reverse_channels,
                           void* stream);
/* exact integer sums behind PSNR (max_offset 0; basicsr calculate_psnr) and cPSNR (max_offset 8; ssr/metrics/cpsnr.py:7-59): for
 * image n, offset (ro, co) in [0, max_offset]^2, channel ch over the cropped window: d = a[y+ro, x+co] - b[y+M-ro, x+M-co],
 * out[((n*(M+1)^2 + ro*(M+1)+co)*c + ch)*2 + {0,1}] = {sum d, sum d^2} (int64).  a, b: uint8 HWC batches. */
int ssr_u8_shift_diff_sums(const void* a_u8, const void* b_u8, int32_t b, int32_t h, int32_t w, int32_t c, int32_t crop_border,
                           int32_t max_offset, long long* out, void* stream);
/* basicsr calculate_ssim: out[n*c + ch] += sum over the valid (h-2cb-10) x (w-2cb-10) region of the SSIM map (float64, caller
 * zeroes out and divides); window11_device = cv2.getGaussianKernel(11, 1.5) as 11 doubles in device memory */
int ssr_u8_ssim_sums(const void* a_u8, const void* b_u8, int32_t b, int32_t h, int32_t w, int32_t c, int32_t crop_border,
                     const double* window11_device, double* out, void* stream);
/* LPIPS, lpips 0.1 net='vgg' (calculate_lpips of ssr/metrics/lpips.py:7-21, called from ssr_esrgan_model.py:305-312).
 * Ingest: uint8 HWC batch [b, h, w, c] -> NHWC bf16 images image_offset .. image_offset + b - 1 of dst (pixel stride dst_pix_stride,
 * channels [c, c_pad) zero): v = (x / 255 - shift[ch]) / scale[ch] (device floats; lpips' ScalingLayer on x / 255). */
int ssr_ingest_u8_nhwc(const void* src_u8, int32_t b, int32_t h, int32_t w, int32_t c, void* dst_bf16, int32_t dst_pix_stride,
                       int32_t image_offset, int32_t c_pad, const float* shift, const float* scale, void* stream);
/* partial-sum slots per image of one tap of size h x w (a function of h * w only) */
int32_t ssr_lpips_cta_count(int32_t h, int32_t w);
/* One tap of the head: feat = [2b, h, w, c] bf16 post-ReLU features (c = 64 / 128 / 256 / 512), pair n = images (n, b + n);
 * lin_w = lin{k}.model.1.weight as c f32 (device).  partial[n * ssr_lpips_cta_count(h, w) + t] = sum over the pixels of slot t of
 * sum_ch lin_w[ch] * (f0 / (|f0| + 1e-10) - f1 / (|f1| + 1e-10))^2 (|f| the channel L2 norm).  Fixed summation order, no atomics. */
int ssr_lpips_layer_sums(const void* feat_bf16, int32_t b, int32_t h, int32_t w, int32_t c, const float* lin_w, double* partial,
                         void* stream);
/* out[n] = sum_k (sum of tap k's partials of pair n) / (tap_h[k] * tap_w[k]) in f64, fixed order; the partials of the n_taps (<= 8)
 * taps lie back to back ([b][cta_count] each); tap_h / tap_w are host arrays */
int ssr_lpips_finish(const double* partial, int32_t b, int32_t n_taps, const int32_t* tap_h, const int32_t* tap_w, double* out,
                     void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SSR_B200_H_ */

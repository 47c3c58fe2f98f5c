/*
 * unetb200 -- C ABI of the B200 (sm_100a) U-Net forward library.
 *
 * This is the drop-in boundary for the one hot path of
 * tingyu-c/TW-invoice-unet-ocr-llm: `UNet.forward` (reference unet_model.py:55-86)
 * as called by `inference.run_unet` (reference inference.py:58-79).  The reference
 * has no FFI of its own (it calls torch.nn); the host-side mirror in
 * tw_invoice_unet_ocr_llm_b200/{unet_model,inference}.py binds these entry points
 * with ctypes.  Signatures use plain pointers and sizes only; the caller owns all
 * device memory (weights blob, workspace, inputs, outputs) and passes raw device
 * pointers plus the CUDA stream to enqueue on.
 *
 * Every function returns 0 on success or a non-zero UNETB200_E* code;
 * unetb200_last_error() then returns a thread-local message.  Nothing aborts.
 */
#ifndef UNETB200_H
#define UNETB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define UNETB200_ABI_VERSION 2

enum {
    UNETB200_OK = 0,
    UNETB200_EINVAL = 1,   /* bad argument (shape not divisible by 16, null pointer, ...) */
    UNETB200_ECUDA = 2,    /* a CUDA runtime/driver call failed */
    UNETB200_EARCH = 3,    /* device is not compute capability 10.x (no fallback exists) */
    UNETB200_ENOMEM = 4    /* workspace too small */
};

/* layer kinds in the packed-weights table */
enum { UNETB200_STEM = 0, UNETB200_CONV3X3 = 1, UNETB200_CONVT2X2 = 2, UNETB200_HEAD = 3 };

/* input formats accepted by unetb200_forward.  The float formats are read as they are (no /255); a 16-bit element
 * is widened to fp32 where the first conv reads it, which is exact, so fp16 / bf16 / NHWC input gives the same
 * bits as the fp32 NCHW input x.float().contiguous().  NHWC = [N,H,W,C] in memory: the storage of a PyTorch
 * channels_last [N,C,H,W] tensor.  Every input is 16-byte aligned (the tensor-core first conv reads it by TMA). */
enum {
    UNETB200_X_F32_NCHW = 0,  /* float32 [N,C,H,W] in [0,1] -- what inference.preprocess returns (inference.py:36-42) */
    UNETB200_X_U8_NHWC = 1,   /* uint8 [N,H,W,C], scaled by /255 in the first kernel (inference.py:36) */
    UNETB200_X_F16_NCHW = 2,  /* float16  [N,C,H,W] */
    UNETB200_X_BF16_NCHW = 3, /* bfloat16 [N,C,H,W] */
    UNETB200_X_F32_NHWC = 4,  /* float32  [N,H,W,C] */
    UNETB200_X_F16_NHWC = 5,  /* float16  [N,H,W,C] */
    UNETB200_X_BF16_NHWC = 6  /* bfloat16 [N,H,W,C] */
};

/* element type of the logits written by unetb200_forward_typed (and unetb200_conv3x3_head, wstat bits 3-4): the
 * fp32 logits as computed, or rounded to nearest-even, i.e. z.to(torch.float16 / torch.bfloat16) bit for bit.
 * Masks are decided on the fp32 value whatever the logits type. */
enum { UNETB200_LOGITS_F32 = 0, UNETB200_LOGITS_F16 = 1, UNETB200_LOGITS_BF16 = 2 };

/* A-operand staging strategy of the tensor-core conv kernel (see csrc/conv_tc.cuh) */
enum { UNETB200_A_TAP = 0, UNETB200_A_COL3 = 1, UNETB200_A_HALO = 2,
       UNETB200_A_ROW = 5 /* single-kernel hooks only: the row-stacked kernel (cout == 64) */,
       UNETB200_A_PS64 = 7 /* single-kernel hooks only: the phase-stacked kernel (64 -> 64 channels, csrc/conv_ps64.cuh) */ };

/* UNet(n_channels, n_classes) of reference unet_model.py:24; base_width is the 64 of :29. */
typedef struct {
    int32_t n_channels; /* 1, 3 or 4 */
    int32_t n_classes;  /* 1..8 */
    int32_t base_width; /* must be 64 */
} unetb200_arch_t;

/* One row of the packed-weights table.  Order == execution order of UNet.forward. */
typedef struct {
    char name[32];      /* state_dict prefix of the conv, e.g. "down1.net.0", "up4", "out_conv" */
    char bn_name[32];   /* state_dict prefix of the BatchNorm folded into it, or "" */
    int32_t kind;       /* UNETB200_STEM / CONV3X3 / CONVT2X2 / HEAD */
    int32_t cin, cout;
    int32_t level;      /* spatial level of the layer INPUT: 0 = H x W, k = H/2^k */
    uint64_t w_off, w_bytes; /* byte range of the packed weights in the blob */
    uint64_t b_off, b_bytes; /* byte range of the fp32 (folded) bias in the blob */
} unetb200_layer_t;

typedef struct unetb200_handle_s* unetb200_handle_t;

int unetb200_abi_version(void);
/* Compile-time switches of this build: UNETB200_BUILD_TEST_VARIANTS = the measured-and-rejected kernel variants
 * (A_COL3 staging, the patch stem) are compiled in (-DUNETB200_TEST_VARIANTS); production builds return 0. */
#define UNETB200_BUILD_TEST_VARIANTS 1
int unetb200_build_flags(void);
const char* unetb200_last_error(void);

/* ---- packed weights: layout + device-side fold/pack (replaces nothing in the
 *      reference; it is the "BN fold + repack" step after inference.py:21) ---- */
int unetb200_num_layers(const unetb200_arch_t* arch);
int unetb200_layer_info(const unetb200_arch_t* arch, int index, unetb200_layer_t* out);
uint64_t unetb200_packed_bytes(const unetb200_arch_t* arch);

/* Fold BatchNorm (pass NULL gamma/beta/mean/var for "no BN") and write layer `index`
 * of the blob at `blob_dev`.  All pointers are device pointers to fp32 tensors laid
 * out as PyTorch stores them (Conv2d: [Cout,Cin,kh,kw]; ConvTranspose2d: [Cin,Cout,2,2]). */
int unetb200_pack_layer(const unetb200_arch_t* arch, int index, const float* weight,
                        const float* bias, const float* bn_gamma, const float* bn_beta,
                        const float* bn_mean, const float* bn_var, float bn_eps, void* blob_dev,
                        void* stream);

/* Decoder level `level` = 1..4 (up{level} + conv{level}.net.0, reference unet_model.py:38-51 / :70-83) with the
 * ConvTranspose2d folded into the 3x3 conv as a four-phase sub-pixel convolution over the low-resolution tensor
 * (csrc/conv_phase.cuh): writes the composite weights [16][Cout][Clow] bf16 and the nine border-case biases
 * [9][Cout] fp32 into their region of the blob (behind the per-layer regions; unetb200_packed_bytes counts them).
 * up_weight [Clow,C,2,2] / up_bias [C] (may be NULL) are the ConvTranspose2d's tensors, conv_weight [Cout,2C,3,3] /
 * conv_bias and the BatchNorm vectors those of conv{level}.net.0 / .net.1.  Optional: a level that was not packed
 * (or a blob that ends after the per-layer regions) runs as two launches. */
int unetb200_pack_fused_up(const unetb200_arch_t* arch, int level, const float* up_weight, const float* up_bias,
                           const float* conv_weight, const float* conv_bias, const float* bn_gamma,
                           const float* bn_beta, const float* bn_mean, const float* bn_var, float bn_eps,
                           void* blob_dev, void* stream);
int unetb200_fused_up_info(const unetb200_arch_t* arch, int level, uint64_t* w_off, uint64_t* w_bytes,
                           uint64_t* b_off, uint64_t* b_bytes);

/* ---- model handle ---- */
/* Replaces the model the reference builds in inference.py:17-24.  `blob_dev` (borrowed)
 * must outlive the handle.  Fails with UNETB200_EARCH on anything but sm_100. */
int unetb200_create(const unetb200_arch_t* arch, const void* blob_dev, uint64_t blob_bytes,
                    int device, unetb200_handle_t* out);
int unetb200_destroy(unetb200_handle_t h);

/* options: "amode" (UNETB200_A_*), "bn_max" (64/128/256), "wstat" (0/1), "stem_tc" (first conv: 0 CUDA cores / 1 tensor cores + im2col / 2 tensor cores, implicit GEMM), "pair" (0 never / 1 everywhere / 2 auto),
 * "pdl" (0/1 programmatic dependent launch), "epi2" (two epilogue groups: 0 never / 1 weight-stationary launches / 2 always), "pf_items" (0..64), "profile" (0/1),
 * "row64" (64-output-channel 3x3 convs on the row-stacked kernel csrc/conv_row.cuh: bit 0 = down1.net.3 and conv1.net.3, bit 1 = conv1.net.0; default 2; results are bit-identical either way),
 * "fold_up" (bit k = decoder level k: ConvTranspose2d folded into the following 3x3 conv, csrc/conv_phase*.cuh; default 15 = every level, one launch each),
 * "fold_one_phase" (0/1 cross-check: folded levels run one phase per work unit), "fold_stack" (0/1, default 1: folded level 1 on the phase-stacked kernel csrc/conv_phase_stack.cuh),
 * "ps64" (bit 0 = down1.net.3, bit 1 = conv1.net.3 on the phase-stacked kernel csrc/conv_ps64.cuh; default 3; results differ from the tap-per-UMMA kernels by fp32 accumulation order only),
 * "fill_sms" (0/1/2 small-batch column-block policy), "min_na" (2..8),
 * "graph" (0/1, default 1: from its second use on, a forward of the same shape / buffers is replayed as one CUDA graph --
 *  one cudaGraphLaunch instead of 18 kernel launches; skipped while profiling or inside a caller's stream capture) */
int unetb200_set_option(unetb200_handle_t h, const char* key, int value);
int unetb200_get_option(unetb200_handle_t h, const char* key, int* value);

uint64_t unetb200_workspace_bytes(unetb200_handle_t h, int n, int height, int width);

/* UNet.forward (unet_model.py:55-86) + the sigmoid/threshold of inference.py:72-79.
 *   x            device pointer, format `x_fmt`, N x C x H x W with H, W divisible by 16
 *   workspace    device scratch of >= unetb200_workspace_bytes(h, N, H, W) bytes
 *   logits       nullable; float32 [N, n_classes, H, W] raw logits (what UNet.forward returns)
 *   mask         nullable; uint8   [N, n_classes, H, W], 1 where logit > logit_thr[c]
 *                (logit_thr[c] = ln(t/(1-t)) reproduces sigmoid(logit) > t)
 *   logit_thr    host pointer to n_classes floats (may be NULL if mask is NULL)
 *   stream       cudaStream_t to enqueue on (NULL = legacy default stream)
 * Asynchronous: returns after enqueueing. */
int unetb200_forward(unetb200_handle_t h, const void* x, int x_fmt, int n, int height, int width,
                     void* workspace, uint64_t workspace_bytes, float* logits, uint8_t* mask,
                     const float* logit_thr, void* stream);

/* Same forward with the masks bit-packed: mask_bits uint8 [N, n_classes, H, W/8], bit (x & 7) (LSB first) of
 * byte x >> 3 of a row is pixel x (numpy: np.unpackbits(bits, axis=-1, bitorder="little")).  The reference keeps
 * one boolean per pixel (inference.py:75-79); this is the same information in an eighth of the bytes, for
 * callers that move masks across PCIe (launcher.GpuWorker). */
int unetb200_forward_bits(unetb200_handle_t h, const void* x, int x_fmt, int n, int height, int width,
                          void* workspace, uint64_t workspace_bytes, float* logits, uint8_t* mask_bits,
                          const float* logit_thr, void* stream);

/* The forward of unetb200_forward / unetb200_forward_bits with the logits element type chosen per call:
 *   logits       nullable; [N, n_classes, H, W] raw logits of type `logits_type` (UNETB200_LOGITS_*); 16-bit logits
 *                are the fp32 logits rounded to nearest-even at the store
 *   mask         nullable; byte masks as unetb200_forward (mask_bits = 0) or bit-packed as unetb200_forward_bits
 *                (mask_bits = 1), decided on the fp32 logits
 * An unknown x_fmt or logits_type is UNETB200_EINVAL. */
int unetb200_forward_typed(unetb200_handle_t h, const void* x, int x_fmt, int n, int height, int width,
                           void* workspace, uint64_t workspace_bytes, void* logits, int logits_type,
                           uint8_t* mask, int mask_bits, const float* logit_thr, void* stream);

/* Per-layer device times (ms) of the last forward run with option "profile" = 1.
 * Synchronises the stream's events.  `ms` has room for `count` floats. */
int unetb200_layer_times(unetb200_handle_t h, float* ms, int count);
/* Number of kernels the last forward enqueued. */
int unetb200_last_launch_count(unetb200_handle_t h);

/* ---- single-kernel entry points (unit parity tests; same code paths as forward).  Each is one layer
 *      of the reference: Conv2d 3x3 + BatchNorm + ReLU (unet_model.py:10-16), the concat of :71-83,
 *      MaxPool2d (:34), ConvTranspose2d (:38-47), out_conv (:50,86) ---- */
/* 3x3 conv + bias + optional ReLU over NHWC bf16.  src1/c1 = second (skip) source or NULL/0.
 * w_packed: [9][cout][c0+c1] bf16, bias fp32[cout].  pool_out nullable (2x2 max-pool 2nd output).
 * bn in {64,128,256}, amode in UNETB200_A_*; `wstat` is a flag word: bit 0 allows the weight-stationary
 * variant, bit 1 selects the CTA-pair (cta_group::2) variant (A_HALO only). */
int unetb200_conv3x3(const void* src0, int c0, const void* src1, int c1, const void* w_packed,
                     const float* bias, int n, int height, int width, int cout, int relu, void* out,
                     void* pool_out, int bn, int amode, int wstat, void* stream);
/* 3x3 conv (cout = 64) + ReLU with the 1x1 head and threshold fused into the epilogue.  `wstat` as above;
 * bit 2 makes `mask` the bit-packed [N, n_classes, H, W/8] format of unetb200_forward_bits; bits 3-4 are the
 * element type of `logits` (UNETB200_LOGITS_*, 0 = float32). */
int unetb200_conv3x3_head(const void* src0, int c0, const void* w_packed, const float* bias,
                          const float* head_w, const float* head_b, int n_classes, int n, int height,
                          int width, void* logits, uint8_t* mask, const float* logit_thr, int amode,
                          int wstat, void* stream);
/* ConvTranspose2d(k=2,s=2): src [N,H,W,cin] bf16 -> out [N,2H,2W,cout] bf16. w_packed [4*cout][cin].
 * bn in {64,128,256}; bn | 0x1000 selects the CTA-pair variant. */
int unetb200_convt2x2(const void* src, int cin, const void* w_packed, const float* bias, int n,
                      int height, int width, int cout, void* out, int bn, void* stream);
/* ConvTranspose2d(k=2,s=2) + Conv2d(3x3, pad 1) over cat([up, skip]) (+ folded BatchNorm, ReLU) as one launch:
 * low [N,h,w,c_low] bf16, skip [N,2h,2w,c_skip] bf16 -> out [N,2h,2w,cout] bf16.  wc_packed / bias9 = the regions
 * unetb200_pack_fused_up writes (unetb200_fused_up_info), w3_packed = the 3x3 conv's own packed weights
 * ([9][cout][c_up + c_skip], unetb200_pack_layer), c_up = K columns of its up half.
 * flags: bit 0 = CTA pairs, bit 1 = one phase per work unit whatever the column block (cross-check variant),
 * bit 2 = the phase-stacked kernel (csrc/conv_phase_stack.cuh) where it applies: cout = c_skip = 64, CTA pairs. */
int unetb200_upconv3x3(const void* low, int c_low, const void* skip, int c_skip, const void* wc_packed,
                       const void* w3_packed, int c_up, const float* bias9, int n, int h_low, int w_low, int cout,
                       int relu, void* out, int bn, int flags, void* stream);
/* First conv on the tensor cores (n_channels 1 or 3): w_tc = the bf16 hi/lo [64][128] layout that
 * unetb200_pack_layer(index 0) writes at blob + w_off + unetb200_stem_tc_offset(cin). */
int unetb200_stem_tc(const void* x, int x_fmt, int cin, const void* w_tc, const float* bias, int n,
                     int height, int width, void* out, void* stream);
uint64_t unetb200_stem_tc_offset(int cin);
/* First conv on the tensor cores as an implicit GEMM over a shared-memory input patch (n_channels 1, 3
 * or 4; an alternative to unetb200_stem_tc, measured slower): w_patch = blob + w_off + unetb200_stem_patch_offset(cin). */
int unetb200_stem_patch(const void* x, int x_fmt, int cin, const void* w_patch, const float* bias, int n,
                        int height, int width, void* out, void* stream);
uint64_t unetb200_stem_patch_offset(int cin);
/* First conv (n_channels -> 64) + ReLU on the CUDA cores (any n_channels in {1,3,4}):
 * x (format x_fmt) -> out [N,H,W,64] bf16. w fp32 [9*cin][64] (start of the stem's blob region). */
int unetb200_stem(const void* x, int x_fmt, int cin, const float* w, const float* bias, int n,
                  int height, int width, void* out, void* stream);

/* ---- pre / post processing (SURVEY 8f): bit-exact integer work around the forward ---- */
/* Pillow's 8-bit bicubic resample, i.e. PIL.Image.resize of inference.py:35,63 (the reference
 * delegates to Pillow==10.2.0, requirements.txt:3).  unetb200_resize_coeffs is host-only: it fills
 * kk[out_size * ksize] (22-bit fixed point) and bounds[out_size * 2] ({first tap, tap count}) for
 * one axis, ksize = unetb200_resize_ksize(in_size, out_size); upload both to the device.
 * unetb200_resize_bicubic_u8: src uint8 [n,h,w,c] -> dst uint8 [n,oh,ow,c]; tmp holds n*h*ow*c
 * bytes (horizontal pass output; may be NULL if only one axis changes). */
int unetb200_resize_ksize(int in_size, int out_size);
int unetb200_resize_coeffs(int in_size, int out_size, int32_t* kk, int32_t* bounds);
int unetb200_resize_bicubic_u8(const uint8_t* src, int n, int h, int w, int c, const int32_t* kx_dev,
                               const int32_t* bx_dev, int ksx, const int32_t* ky_dev, const int32_t* by_dev,
                               int ksy, uint8_t* tmp_dev, uint8_t* dst_dev, int oh, int ow, void* stream);
/* Same with a padded source: every source pixel is `pixel_stride` bytes of which the first c are read (c = 3,
 * pixel_stride = 4: the RGBX buffer Pillow keeps for an RGB image, exported without a host-side repack); the
 * result is packed [n,oh,ow,c].  Needs a horizontal pass (ow != w). */
int unetb200_resize_bicubic_u8_ps(const uint8_t* src, int n, int h, int w, int c, int pixel_stride,
                                  const int32_t* kx_dev, const int32_t* bx_dev, int ksx, const int32_t* ky_dev,
                                  const int32_t* by_dev, int ksy, uint8_t* tmp_dev, uint8_t* dst_dev, int oh, int ow,
                                  void* stream);
/* np.where(mask) min/max of inference.py:85-93: mask uint8 [n_planes,h,w] ->
 * out int32 [n_planes,5] = {xmin, xmax, ymin, ymax, count}; an empty plane gives {w, -1, h, -1, 0}. */
int unetb200_mask_bbox(const uint8_t* mask, int n_planes, int h, int w, int32_t* out, void* stream);
/* Same reduction over bit-packed planes (unetb200_forward_bits): bits uint8 [n_planes, h, w/8], w % 32 == 0. */
int unetb200_mask_bbox_bits(const uint8_t* bits, int n_planes, int h, int w, int32_t* out, void* stream);
/* Connected components of binary planes: the regions of each field mask, where unetb200_mask_bbox gives the box of
 * all set pixels.  mask = byte planes uint8 [n_planes, h, w] (non-zero = set; packed = 0) or bit-packed planes
 * uint8 [n_planes, h, w/8] in the format of unetb200_forward_bits (packed = 1; w % 32 == 0, 4-byte aligned);
 * h, w >= 1, h * w < 2^31; connectivity 4 or 8.
 *   labels     nullable; int32 [n_planes, h, w]: 0 = background, components numbered 1..n in raster order of their
 *              first pixel -- exactly scipy.ndimage.label with generate_binary_structure(2, 1) (4) / ones((3, 3)) (8)
 *   comps      int32 [n_planes, max_components, 6] = {xmin, xmax, ymin, ymax, count, label} of the max_components
 *              (1..16) largest components, count descending then label ascending; extents inclusive as
 *              unetb200_mask_bbox; unused rows {w, -1, h, -1, 0, 0}
 *   n_comps    int32 [n_planes]: number of components of each plane (may exceed max_components)
 *   workspace  device scratch of >= unetb200_components_workspace_bytes(n_planes, h, w) bytes, 16-byte aligned,
 *              no initialisation needed; at most 14.2 bytes per pixel plus 20 bytes per plane
 * Outputs are deterministic bits.  Asynchronous: enqueued on `stream`, nothing is allocated.  A null pointer, a bad
 * size, connectivity or max_components, or a misaligned pointer (int32 arrays 4-byte aligned) is UNETB200_EINVAL;
 * a short workspace UNETB200_ENOMEM.  The query returns 0 for a bad size. */
uint64_t unetb200_components_workspace_bytes(int n_planes, int h, int w);
int unetb200_mask_components(const uint8_t* mask, int packed, int n_planes, int h, int w, int connectivity,
                             int max_components, int32_t* labels, int32_t* comps, int32_t* n_comps, void* workspace,
                             uint64_t workspace_bytes, void* stream);
/* unetb200_mask_components plus the oriented box of every selected component (DESIGN.md 6b), for upright crops of
 * tilted fields.  labels, comps and n_comps are bit-identical to unetb200_mask_components; h, w <= 32767 and
 * n_planes <= 65535 (else UNETB200_EINVAL).
 *   scale      nullable (= 1, 1); device float64 [n_planes][2] = (sx, sy), positive and finite: mask pixel (x, y) is
 *              the frame point X = (x + 0.5) sx - 0.5, Y = (y + 0.5) sy - 0.5 (sx = frame width / w, ...)
 *   moments    int64 [n_planes, max_components, 6] = n, Sx, Sy, Sxx, Sxy, Syy of the row's component's mask pixels
 *              (cv2.moments(binaryImage=True)'s m00, m10, m01, m20, m11, m02); unused rows zeros
 *   obox       float64 [n_planes, max_components, 6] = e1x, e1y, umin, umax, vmin, vmax: e1 = the unit principal axis
 *              of the frame-space covariance (e1x > 0, or e1x == 0 and e1y > 0), e2 = (-e1y, e1x), and the extents of
 *              u = X e1x + Y e1y, v = X e2x + Y e2y over the component's pixels; unused rows zeros
 *   workspace  >= unetb200_components_oriented_workspace_bytes(n_planes, h, w) bytes (the components workspace, 16-byte
 *              aligned, plus 512 bytes per plane), 16-byte aligned
 * moments, obox and scale are 8-byte aligned.  Integer arithmetic and correctly rounded float64 + - * / sqrt only:
 * the outputs are deterministic and equal oracle/oriented.py bit for bit.  The query returns 0 for a bad size. */
uint64_t unetb200_components_oriented_workspace_bytes(int n_planes, int h, int w);
int unetb200_mask_components_oriented(const uint8_t* mask, int packed, int n_planes, int h, int w, int connectivity,
                                      int max_components, const double* scale, int32_t* labels, int32_t* comps,
                                      int32_t* n_comps, int64_t* moments, double* obox, void* workspace,
                                      uint64_t workspace_bytes, void* stream);
/* Binary morphology of mask planes, for cleaning the field masks before unetb200_mask_components: */
enum {
    UNETB200_MORPH_ERODE = 0,      /* cv2.erode(m, ones((kh, kw))): AND over the window */
    UNETB200_MORPH_DILATE = 1,     /* cv2.dilate(m, ones((kh, kw))): OR over the window */
    UNETB200_MORPH_OPEN = 2,       /* cv2.morphologyEx(MORPH_OPEN) = dilate(erode(m)) */
    UNETB200_MORPH_CLOSE = 3,      /* cv2.morphologyEx(MORPH_CLOSE) = erode(dilate(m)) */
    UNETB200_MORPH_FILL_HOLES = 4  /* scipy.ndimage.binary_fill_holes(m): kw, kh ignored */
};
/* Workspace of unetb200_mask_morph: two bit planes for ERODE .. CLOSE (ceil(w / 32) * 4 bytes per row each), the
 * components workspace (unetb200_components_workspace_bytes) for FILL_HOLES; 0 for a bad size or op. */
uint64_t unetb200_morph_workspace_bytes(int n_planes, int h, int w, int op);
/* in -> out for every plane, bit-exact with OpenCV's defaults (and SciPy's for FILL_HOLES):
 *   element    kw x kh rectangle, 1 <= kw, kh <= 63, anchor (kw / 2, kh / 2); erosion and dilation both use the
 *              window x - kw/2 .. x + kw - 1 - kw/2, y - kh/2 .. y + kh - 1 - kh/2 (OpenCV does not reflect the
 *              element for dilation; SciPy does, so the two differ for even sizes)
 *   border     pixels outside the plane take no part (BORDER_CONSTANT with morphologyDefaultBorderValue)
 *   holes      4-connected background components that touch no border pixel become set
 *   in, out    byte planes uint8 [n_planes, h, w] (non-zero = set; out is 0 / 1) or, with in_packed / out_packed = 1,
 *              bit-packed planes uint8 [n_planes, h, w/8] in the format of unetb200_forward_bits (w % 32 == 0,
 *              4-byte aligned); any of the four combinations.  In place (in == out, or any overlap) works.
 *   workspace  >= unetb200_morph_workspace_bytes(n_planes, h, w, op) bytes, 16-byte aligned, no initialisation
 * h, w >= 1 and h * w < 2^31 as unetb200_mask_components.  Deterministic bits.  Asynchronous: enqueued on `stream`,
 * nothing is allocated.  A null pointer, a bad op, k, size or packed flag, or a misaligned pointer is UNETB200_EINVAL;
 * a short workspace UNETB200_ENOMEM. */
int unetb200_mask_morph(const uint8_t* in, int in_packed, uint8_t* out, int out_packed, int n_planes, int h, int w,
                        int op, int kw, int kh, void* workspace, uint64_t workspace_bytes, void* stream);
/* Scores predicted planes against ground-truth planes (DESIGN.md 6b, "Region matching"; oracle/mask_match.py):
 *   pred, gt   byte planes uint8 [n_planes, h, w] (non-zero = set) or, with pred_packed / gt_packed = 1, bit-packed
 *              planes uint8 [n_planes, h, w/8] in the format of unetb200_forward_bits (w % 32 == 0, 4-byte aligned);
 *              any of the four combinations; h, w >= 1, h * w < 2^31 as unetb200_mask_components
 *   regions    the connected components of each plane (connectivity 4 or 8, the labels of unetb200_mask_components);
 *              a pred region with fewer than min_pixels (>= 1) pixels is ignored, gt regions never are
 *   match      pred region a and gt region g match when I > t (x) U, I = |a n g| and U = |a| + |g| - I exact
 *              integers and (x) one correctly rounded float64 product; t = iou_threshold in [0.5, 1), so a region
 *              has at most one partner
 *   counts     int64 [n_planes, 8] = px_tp, px_fp, px_fn (set/set, set/clear, clear/set pixels, all of them),
 *              n_pred (pred regions of >= min_pixels pixels), n_gt (gt regions), tp (matched pairs), sum of I and
 *              sum of U over the matched pairs
 *   iou_sum    float64 [n_planes]: sum of the correctly rounded I / U over the matched pairs; thread j of 256 adds the
 *              pairs of pred labels j + 1, j + 257, ... in ascending order from +0.0, then s[j] += s[j + half] for
 *              half = 128, 64, ..., 1 combines the partial sums
 *   workspace  >= unetb200_match_workspace_bytes(n_planes, h, w) bytes, 16-byte aligned, no initialisation: two
 *              components workspaces (each rounded up to 16 bytes), 12 bytes per statistics row (ceil(h * w / 2)
 *              rows per plane) and 8 bytes per plane
 * counts and iou_sum are 8-byte aligned.  Deterministic bits.  Asynchronous: enqueued on `stream`, nothing is
 * allocated.  A null pointer, a bad size, flag, connectivity, min_pixels or threshold (not finite or outside
 * [0.5, 1)), or a misaligned pointer is UNETB200_EINVAL; a short workspace UNETB200_ENOMEM.  The query returns 0 for
 * a bad size. */
uint64_t unetb200_match_workspace_bytes(int n_planes, int h, int w);
int unetb200_mask_match(const uint8_t* pred, int pred_packed, const uint8_t* gt, int gt_packed, int n_planes, int h,
                        int w, int connectivity, int min_pixels, double iou_threshold, int64_t* counts,
                        double* iou_sum, void* workspace, uint64_t workspace_bytes, void* stream);
/* Ragged batch of affine crops: output pixel (j, i) of crop k samples its frame at (m0 j + m1 i + m2, m3 j + m4 i + m5),
 * bilinear with replicated borders, bit-identical to cv2.warpAffine(src, M, (out_w, out_h),
 * flags=INTER_LINEAR | WARP_INVERSE_MAP, borderMode=BORDER_REPLICATE) of the RGB frame. */
typedef struct unetb200_warp_crop {
    uint64_t src;             /* device address of the frame's pixel (0, 0) */
    int32_t src_h, src_w;     /* frame size, 1..32767 */
    int32_t src_stride;       /* pixels per frame row, >= src_w */
    int32_t src_pixel_bytes;  /* 3 (packed RGB) or 4 (RGBX: Pillow's storage of an RGB image); bytes 0..2 are R, G, B */
    double m[6];              /* the inverse map M = [[m0, m1, m2], [m3, m4, m5]] (frame point of an output pixel) */
    int32_t out_w, out_h;     /* crop size, 1..32767 */
    uint64_t out_off;         /* byte offset of the crop's packed uint8 [out_h][out_w][3] in `out`; must not decrease
                               * from one crop to the next, nor start inside the previous crop */
} unetb200_warp_crop;
/* table_host = the n descriptors (read for validation and grid sizes), table_dev = the same n structs in device
 * memory (8-byte aligned).  out = device buffer of the crops; sums = device uint64 [n] (zeroed here), the byte sum of
 * each crop (the near-black test of inference.py:121-125 is sum < 3 * 3 * out_w * out_h).  A bad descriptor, or a
 * matrix that takes a coordinate of the crop to 2^19 or beyond (OpenCV's fixed point would overflow), is
 * UNETB200_EINVAL.  Asynchronous, enqueued on `stream`; nothing is allocated. */
int unetb200_warp_crops(const unetb200_warp_crop* table_host, const void* table_dev, int n, uint8_t* out,
                        uint64_t* sums, void* stream);
/* Byte sums of n_boxes (<= 16) rectangles {x1, y1, x2, y2} (half-open, host array of 4*n_boxes ints) of one
 * uint8 [h][w][c] device frame -> sums_dev uint64 [n_boxes] (zeroed here): the `np.array(crop).mean() < 3`
 * rejection of inference.py:121-125 as the exact integer test sum < 3 * (x2-x1)*(y2-y1)*c. */
int unetb200_box_sums(const uint8_t* img, int h, int w, int c, const int32_t* boxes_host, int n_boxes,
                      uint64_t* sums_dev, void* stream);
/* Same for c-byte pixels of which only the first `used` bytes count (c = 4, used = 3: RGBX frames). */
int unetb200_box_sums_ps(const uint8_t* img, int h, int w, int c, int used, const int32_t* boxes_host, int n_boxes,
                         uint64_t* sums_dev, void* stream);

/* Test hook (host only): x / d as the kernels compute it for their per-tile index arithmetic (multiply-high by a
 * precomputed magic number, then shift); valid for x < 2^31, d >= 1. */
uint32_t unetb200_test_fastdiv(uint32_t d, uint32_t x);

/* ---- OCR crop enhancement (SURVEY 8f rank 4): app_camera.py:572-598 enhance_for_ocrspace and
 * :685-705 enhance_for_date_ocr, i.e. cv2.cvtColor(RGB2GRAY) -> cv2.resize(fx=4, fy=4, INTER_CUBIC)
 * -> [cv2.filter2D 3x3 sharpen] -> CLAHE(clip, 8x8) -> [cv2.GaussianBlur 3x3] -> [cv2.threshold OTSU],
 * over a ragged batch of uint8 RGB crops, bit-exact with OpenCV's own code path. ---- */
#define UNETB200_ENH_SHARPEN 1   /* filter2D [[-1,-1,-1],[-1,9,-1],[-1,-1,-1]] after the upscale */
#define UNETB200_ENH_BLUR 2      /* GaussianBlur((3,3), 0) after CLAHE */
#define UNETB200_ENH_OTSU 4      /* threshold(0, 255, THRESH_BINARY | THRESH_OTSU) at the end */
/* enhance_for_ocrspace(mode="text") = SHARPEN|OTSU, clip 4.0; any other mode = SHARPEN, clip 4.0;
 * enhance_for_date_ocr = BLUR|OTSU, clip 3.0 */
typedef struct unetb200_enh_crop {
    int32_t h, w;             /* in : crop size in pixels (output is 4h x 4w) */
    int32_t flags;            /* in : UNETB200_ENH_* */
    double clip;              /* in : CLAHE clipLimit, finite and > 0; a double, as cv::createCLAHE takes it
                               *      (4 bytes of alignment padding precede it) */
    int32_t clip_count;       /* out: per-bin clip limit, max((int)min(clip * tile_area / 256, tile_area), 1) in
                               *      double: OpenCV's (int)(clipLimit * tileSizeTotal / 256), clamped at the tile
                               *      area.  No bin holds more than the area, so a limit at or above it clips
                               *      nothing, like any larger one: the LUTs are OpenCV's wherever OpenCV's own
                               *      int conversion is defined, and huge or overflowing products clip nothing */
    int32_t tile_h, tile_w;   /* out: CLAHE tile size of the (reflect-extended) upscaled image */
    int32_t first_block;      /* out: index of this crop's first 32x32 output block in the batch */
    int32_t blocks_x;         /* out: output blocks per row */
    int32_t n_blocks;         /* out: output blocks of this crop */
    int32_t src_stride;       /* in : pixels per source row; 0 = the crop is packed ([h][w][3], plan places it),
                               *      > w = the crop is a window of a larger frame already in `src` */
    int32_t src_pixel_bytes;  /* in : bytes per source pixel, the first 3 are R, G, B; 0 = 3 (packed RGB), 4 = RGBX */
    uint64_t src_off;         /* out (in when src_stride != 0): byte offset of the crop's first pixel in `src` */
    uint64_t out_off;         /* out: byte offset of the uint8 [4h][4w] result in `out` */
    uint64_t ws_off;          /* out: byte offset of this crop's scratch in `workspace` */
} unetb200_enh_crop;
/* Host only: fills the `out` fields of table[0..n) from the `in` fields and returns the sizes of the
 * three device buffers (packed crops back to back at 16-byte aligned offsets; windows of a frame
 * (src_stride != 0) keep their src_off and take no room in src_bytes). */
int unetb200_enhance_plan(unetb200_enh_crop* table, int n, uint64_t* src_bytes, uint64_t* out_bytes,
                          uint64_t* workspace_bytes);
/* Enqueues the five kernels on `stream`.  table_host = the planned table (read for validation and grid
 * sizes), table_dev = the same n structs in device memory; src/out/workspace are device buffers of at
 * least the planned sizes.  Nothing is allocated; the workspace needs no initialisation.  Before any CUDA
 * call each crop of table_host is checked against what the plan gives (tiles, clip count, block grid,
 * output and workspace offsets); a mismatch is EINVAL naming the crop and the field. */
int unetb200_enhance_run(const unetb200_enh_crop* table_host, const void* table_dev, int n,
                         const uint8_t* src_dev, uint8_t* out_dev, void* workspace_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* UNETB200_H */

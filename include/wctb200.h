/*
 * libwctb200 -- C-ABI of the B200-native WCT inference hot path.
 *
 * The reference (eridgd/WCT-TF) has no native boundary: its operator surface is
 * Python (`WCT.predict` wct.py:70, `WCTModel` model.py:33, `wct_np/wct_tf/adain`
 * ops.py:24,92,282) executed inside one TF `sess.run` (wct.py:97).  This header
 * is the boundary a maintainer binds with ctypes (see INTEGRATION.md); every
 * entry point names the reference code it replaces.
 *
 * Conventions (all functions):
 *   - return 0 on success, <0 on error (WCTB200_E*); `wctb200_last_error()` gives a
 *     thread-local message; nothing throws;
 *   - plain pointers and sizes only; every buffer is a CUDA DEVICE pointer owned by
 *     the caller (e.g. `torch.Tensor.data_ptr()`), kept alive until `stream` is synced;
 *   - asynchronous on `stream` (a `cudaStream_t` passed as void*; 0 = default stream);
 *     the caller selects the device (`cudaSetDevice`) before the call;
 *   - no CPU fallback: without an sm_100 device the kernels fail with WCTB200_ECUDA.
 *
 * Activation format "SPF16" (split-pair fp16, reflect-padded NHWC):
 *   one allocation of `wctb200_act_bytes(N,H,W,C)` bytes holding two fp16 planes
 *   [plane 0 = hi | plane 1 = lo], each [N][H+2][W+2][C]; the fp32 value of an
 *   element is hi+lo: 22-23 significant bits for |x| >= 0.125, an absolute error <= 3e-8 below that (lo is an fp16
 *   subnormal there), |x| saturates at 65000 (fp16 range).  The 1-pixel halo already holds the
 *   REFLECT padding of ops.py:12-15 (mirror without edge repeat), written by the
 *   producer, so a 3x3 'valid' conv over the padded plane equals Conv2DReflect
 *   (ops.py:17-19).  C must be a multiple of 8; H,W >= 2.
 */
#ifndef WCTB200_H
#define WCTB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define WCTB200_API __attribute__((visibility("default")))
#else
#define WCTB200_API
#endif

#define WCTB200_ABI_VERSION 1

#define WCTB200_OK       0
#define WCTB200_EINVAL  -1   /* bad argument / unsupported shape */
#define WCTB200_ECUDA   -2   /* CUDA runtime / driver error (incl. no sm_100 device) */
#define WCTB200_EWS     -3   /* workspace too small */
#define WCTB200_EDEVICE -4   /* a kernel flagged an internal error (pipeline timeout) */

/* conv / transform flags */
#define WCTB200_RELU     1   /* ReLU epilogue                     (vgg_normalised.py:40, model.py:291) */
#define WCTB200_CLIP01   2   /* clip to [0,1] (tail conv only)    (model.py:17,86) */
#define WCTB200_HALO_EDGE 4  /* conv3x3: write an EDGE-replicated halo instead of the reflect halo -- for an output
                                that is consumed by wctb200_conv3x3_up2 only (UpSampling2D follows, model.py:293) */

#define WCTB200_POOL2    8   /* conv3x3: MaxPooling2D 2x2/2 'same' (vgg_normalised.py:41-42) folded into the epilogue: the
                                output is [N, ceil(H/2), ceil(W/2), Cout] (>= 2x2) and the full-resolution tensor is never
                                written -- for conv1_2 / 2_2 / 3_4 / 4_4, whose only consumer is the pool */

WCTB200_API int         wctb200_abi_version(void);
WCTB200_API const char* wctb200_last_error(void);
/* Synchronises `stream` and returns WCTB200_EDEVICE if any kernel since the last
 * call recorded an internal error (mbarrier timeout in the tcgen05 pipeline). */
WCTB200_API int         wctb200_check_device(void* stream);

/* ---- SPF16 activations ---------------------------------------------------- */
WCTB200_API size_t wctb200_act_bytes(int N, int H, int W, int C);
/* fp32 NHWC -> SPF16 (interior + reflect halo).  Test / interop helper. */
WCTB200_API int wctb200_act_from_f32(const float* nhwc, int N, int H, int W, int C, void* act, void* stream);
/* SPF16 -> fp32 NHWC (interior only). */
WCTB200_API int wctb200_act_to_f32(const void* act, int N, int H, int W, int C, float* nhwc, void* stream);

/* ---- image pre/post: WCT.preprocess / WCT.postprocess (wct.py:60-68) -------- */
/* out[i] = img[i] / 255 */
WCTB200_API int wctb200_image_u8_to_f32(const uint8_t* img, size_t count, float* out, void* stream);
/* out[i] = (uint8) (clip(img[i],0,1) * 255)   -- truncation, like np.uint8 */
WCTB200_API int wctb200_image_f32_to_u8(const float* img, size_t count, uint8_t* out, void* stream);

/* ---- CLI image steps on the device (scope row 8f-3) ------------------------- */
/* utils.resize_to / center_crop / center_crop_to (utils.py:29-67) -> scipy.misc.imresize(interp='bilinear'), i.e. Pillow's
 * 8-bit ImagingResample: bit-exact restatement (separable triangle filter with support max(1, in/out), 22-bit fixed-point
 * coefficients, horizontal pass first, uint8 rounding between the passes).  src [N][Hs][Ws][C] uint8 is resampled to
 * Hd x Wd and the window rows [y0, y0+Hout) x columns [x0, x0+Wout) of the result is written to dst [N][Hout][Wout][C]
 * (the centre crop of utils.py:29-53 folded in; y0 = x0 = 0, Hout = Hd, Wout = Wd for a plain resize; Hd = Hs, Wd = Ws
 * for a plain crop).  ws: wctb200_resize_workspace_bytes(N, Hs, Ws, C, Hd, Wd, Wout) bytes of device scratch. */
WCTB200_API size_t wctb200_resize_workspace_bytes(int N, int Hs, int Ws, int C, int Hd, int Wd, int Wout);
WCTB200_API int wctb200_resize_bilinear_u8(const uint8_t* src, int N, int Hs, int Ws, int C, int Hd, int Wd, int y0, int x0,
                                           int Hout, int Wout, uint8_t* dst, void* ws, size_t ws_bytes, void* stream);
/* --keep-colors, the pixel-sized parts of coral.coral_numpy (coral.py:13-39; utils.preserve_colors_np utils.py:87-90).
 * rgb_moments: sums[0..2] = sum x_c, sums[3..8] = sum x0x0, x0x1, x0x2, x1x1, x1x2, x2x2 over the npix RGB pixels, exact
 * uint64 on the DEVICE (9 words).  coral_apply: dst = uint8(clip((A ((x/255 - src_mean)/src_std)) * tgt_std + tgt_mean, 0, 1)
 * * 255) in double precision; A (3x3 row-major), the means and the stds are HOST arrays (the 3x3 algebra that produces them
 * from the moments -- numpy's SVD inside the reference's matSqrt, coral.py:8-11 -- is host work). */
WCTB200_API int wctb200_rgb_moments_u8(const uint8_t* img, long long npix, unsigned long long* sums, void* stream);
WCTB200_API int wctb200_coral_apply_u8(const uint8_t* src, long long npix, const double* A, const double* src_mean,
                                       const double* src_std, const double* tgt_mean, const double* tgt_std, uint8_t* dst,
                                       void* stream);

/* ---- encoder / decoder layers ---------------------------------------------- */
/* Weight preparation (one-time, device side):
 * w_hwio fp32 [3][3][Cin][Cout] (Keras kernel layout, vgg_normalised.py:33 /
 * model.py:291) -> split-fp16 GEMM operand [2 planes][Cout][9*Cin], k = tap*Cin + cin, stored scaled by a per-layer
 * power of two (max|w| -> [512,1024); the factor sits in a trailer of the buffer and is undone in the conv epilogue)
 * so that the lo plane of small weights does not fall into the fp16 subnormals.
 * `taps` is 9 (3x3) or 1 (a [Cin][Cout] matrix). */
WCTB200_API size_t wctb200_conv_weight_bytes(int taps, int Cin, int Cout);
WCTB200_API int wctb200_prep_conv_weights(const float* w_hwio, int taps, int Cin, int Cout, void* w_split, void* stream);
/* Weights of `UpSampling2D() -> Conv2DReflect` (model.py:291-293) as ONE conv over the low-resolution input: four
 * 2x2-tap kernels (one per output parity) whose taps are sums of the 3x3 taps that land on the same low-resolution
 * pixel; [4 parities][2 planes][Cout][4*Cin].  Buffer size: wctb200_conv_weight_bytes(16, Cin, Cout). */
WCTB200_API int wctb200_prep_conv_weights_up2(const float* w_hwio, int Cin, int Cout, void* w_up2, void* stream);

/* Conv2DReflect 3x3 (+bias, optional ReLU) on tensor cores (tcgen05, split-fp16 x3):
 * replaces `Lambda(pad_reflect) -> Conv2D(valid)` of vgg_normalised.py:28-40 and
 * model.py:291.  Cin, Cout multiples of 64.  in/out: SPF16 [N,H,W,Cin] -> [N,H,W,Cout]
 * ([N,ceil(H/2),ceil(W/2),Cout] with WCTB200_POOL2). */
WCTB200_API int wctb200_conv3x3(const void* act_in, int N, int H, int W, int Cin,
                    const void* w_split, const float* bias, int Cout, int flags,
                    void* act_out, void* stream);
/* UpSampling2D (nearest x2, model.py:293) followed by Conv2DReflect 3x3 (+bias, optional ReLU), fused: act_in is the
 * LOW-resolution SPF16 [N,H,W,Cin] whose halo is EDGE-replicated (its producer ran with WCTB200_HALO_EDGE), act_out is
 * SPF16 [N,2H,2W,Cout] with the usual reflect halo.  4/9 of the MACs of the unfused pair and no upsampled tensor. */
WCTB200_API int wctb200_conv3x3_up2(const void* act_in, int N, int H, int W, int Cin,
                        const void* w_up2, const float* bias, int Cout, int flags,
                        void* act_out, void* stream);
/* Same contract on CUDA cores in plain fp32 (validation kernel, fp32 weights [3][3][Cin][Cout]). */
WCTB200_API int wctb200_conv3x3_ref(const void* act_in, int N, int H, int W, int Cin,
                        const float* w_hwio, const float* bias, int Cout, int flags,
                        void* act_out, void* stream);
/* Encoder head: the 1x1 'preprocess' conv (vgg_normalised.py:25-26) folded into
 * conv1_1 3->64 + ReLU.  img fp32 NHWC [N,H,W,3] in [0,1]; w fp32 [27][64] (k = tap*3+cin),
 * b fp32 [64]; out SPF16 [N,H,W,64]. */
WCTB200_API int wctb200_conv_head(const float* img, int N, int H, int W, const float* w, const float* b,
                      void* act_out, void* stream);
/* Decoder tail: Conv2DReflect Cin->3, no activation (model.py:297-298), optional
 * clip to [0,1] (model.py:86).  w fp32 [9*Cin][3], b fp32 [3]; out fp32 NHWC [N,H,W,3]. */
WCTB200_API int wctb200_conv_tail(const void* act_in, int N, int H, int W, int Cin, const float* w, const float* b,
                      int flags, float* img_out, void* stream);
/* MaxPooling2D(2x2, stride 2, padding='same') (vgg_normalised.py:41-42): out [N,ceil(H/2),ceil(W/2),C]. */
WCTB200_API int wctb200_maxpool2(const void* act_in, int N, int H, int W, int C, void* act_out, void* stream);
/* UpSampling2D nearest x2 (model.py:293): out [N,2H,2W,C]. */
WCTB200_API int wctb200_upsample2(const void* act_in, int N, int H, int W, int C, void* act_out, void* stream);

/* ---- feature transforms ------------------------------------------------------ */
/* Whiten-colour transform of one relu level for a batch: replaces wct_tf (ops.py:24-90,
 * what the graph runs) and wct_np (ops.py:92-140, the named oracle) -- semantics flags:
 *   eps_cov            added to the covariance diagonal           (wct_tf 1e-8 | wct_np 0)
 *   eps_eig            added to the kept eigenvalues              (wct_tf 0    | wct_np 1e-5)
 *   thresh             keep eigenvalues > thresh                  (1e-5, ops.py:68,112)
 *   readd_content_mean blend with fc+mc (ops.py:83) or fc (ops.py:133)
 * content SPF16 [Nc,Hc,Wc,C]; style SPF16 [Ns,Hs,Ws,C] with Ns == Nc (frame i uses
 * style i) or Ns == 1 (shared).  out SPF16 [Nc,Hc,Wc,C].  k_out (device int32
 * [2*(Nc+Ns)], may be NULL): k_c per content then k_s per style, then sweep counts.
 * C in {64,128,256,512}.  ws: device scratch of wctb200_wct_workspace_bytes(). */
WCTB200_API size_t wctb200_wct_workspace_bytes(int C, int Nc, int Ns);
WCTB200_API int wctb200_wct_level(const void* content, int Nc, int Hc, int Wc,
                      const void* style, int Ns, int Hs, int Ws, int C,
                      float alpha, float eps_cov, float eps_eig, float thresh, int readd_content_mean,
                      void* out, int32_t* k_out, void* ws, size_t ws_bytes, void* stream);
/* Split form of wctb200_wct_level (same arithmetic, same semantics flags): the style side --
 * means, covariance, eigendecomposition and colouring matrix C_s = E_s D_s^1/2 E_s^T of
 * ops.py:48-55,76 -- depends only on the style features, so a host can run it on a second
 * stream (it overlaps the content convolutions) or cache it for a batch that shares one style.
 * `state`: device buffer of wctb200_wct_style_state_bytes(C, Ns) bytes.  Workspace sizes:
 * wctb200_wct_workspace_bytes(C, Nc, Ns) is enough for either call. */
WCTB200_API size_t wctb200_wct_style_state_bytes(int C, int Ns);
WCTB200_API int wctb200_wct_style_prepare(const void* style, int Ns, int Hs, int Ws, int C,
                              float eps_cov, float eps_eig, float thresh,
                              void* state, void* ws, size_t ws_bytes, void* stream);
WCTB200_API int wctb200_wct_apply(const void* content, int Nc, int Hc, int Wc, int C, const void* state, int Ns,
                      float alpha, float eps_cov, float eps_eig, float thresh, int readd_content_mean,
                      void* out, int32_t* k_out, void* ws, size_t ws_bytes, void* stream);
/* AdaIN (ops.py:282-294): biased per-channel moments of content and style,
 * y = (x-mc)*rsqrt(vc+eps)*sqrt(vs)+ms, out = alpha*y + (1-alpha)*x. */
WCTB200_API int wctb200_adain_level(const void* content, int Nc, int Hc, int Wc,
                        const void* style, int Ns, int Hs, int Ws, int C,
                        float alpha, float eps, void* out, void* ws, size_t ws_bytes, void* stream);

/* ---- spatial control: one style per region of a label mask (Li et al. 2017, sec. 4) ---------------------------------- *
 * A uint8 label map [Nc][Hc][Wc] at the resolution of the features splits every content frame into regions.  Label r < R
 * selects style r: the frame's features RESTRICTED to the pixels labelled r are transformed with their own statistics
 * (means, covariance, k_c, alpha blend and mean re-add of wct_tf / wct_np / adain) and the result is written back to those
 * pixels.  Labels >= R ("keep"), and every region with fewer than 2 pixels, leave the output equal by value to the input.
 * R in 1..8; the R styles are shared by all frames. */
/* nearest-neighbour resize of uint8 label maps in exact integer arithmetic:
 * dst[n][y][x] = src[n][(y*Hs) div Hd][(x*Ws) div Wd]; src [N][Hs][Ws], dst [N][Hd][Wd] (device) */
WCTB200_API int wctb200_labels_resize_nearest(const uint8_t* src, int N, int Hs, int Ws, int Hd, int Wd, uint8_t* dst, void* stream);
/* device scratch for wctb200_wct_apply_regions and wctb200_adain_regions */
WCTB200_API size_t wctb200_wct_regions_workspace_bytes(int C, int Nc, int R);
/* labels: device uint8 [Nc][Hc][Wc] at feature resolution; states: HOST array of R device pointers, each a
   wctb200_wct_style_state of Ns = 1.  k_out (may be NULL): int32 [2*Nc*R] = k_c per (frame, region), frame-major,
   then the pixel count n_r of each. */
WCTB200_API int wctb200_wct_apply_regions(const void* content, int Nc, int Hc, int Wc, int C, const uint8_t* labels, int R,
                              const void* const* states, float alpha, float eps_cov, float eps_eig, float thresh,
                              int readd_content_mean, void* out, int32_t* k_out, void* ws, size_t ws_bytes, void* stream);
/* styles: HOST array of R device pointers to SPF16 [1,Hs_r,Ws_r,C]; style_hw: HOST int [R][2] */
WCTB200_API int wctb200_adain_regions(const void* content, int Nc, int Hc, int Wc, int C, const uint8_t* labels, int R,
                          const void* const* styles, const int* style_hw, float alpha, float eps,
                          void* out, void* ws, size_t ws_bytes, void* stream);

/*
 * wct_style_swap (ops.py:145-217) + style_swap (ops.py:219-278) for ONE content/style pair: whiten both encodings, take every
 * patch x patch window of the whitened style at `stride` (--ss-patch-size / --ss-stride, stylize.py:33-34), replace every
 * content window (same stride, VALID) by its best-correlated style patch (filters normalised per tap across patches, first
 * arg-max, overlaps averaged), colour with the style, blend with `alpha` (= --ss-alpha).  The swapped encoding must tile the
 * content encoding exactly -- (ho-1)*stride + patch == Hc -- which is what wct.py:84-90 (utils.swap_filter_fit) ensures by
 * cropping the content image; otherwise WCTB200_EINVAL.  k_out (may be NULL): [k_c, k_s].
 * Used at relu5_1 when --swap5 is given (model.py:148-152).
 */
WCTB200_API size_t wctb200_style_swap_workspace_bytes(int C, int Hc, int Wc, int Hs, int Ws, int patch, int stride);
WCTB200_API int wctb200_style_swap_level(const void* content, int Hc, int Wc, const void* style, int Hs, int Ws, int C,
                             int patch, int stride, float alpha, float eps_cov, float thresh, void* out, int32_t* k_out,
                             void* ws, size_t ws_bytes, void* stream);

/* Stand-alone pieces of the transform, exposed for parity tests and profiling:
 * per-channel mean [N][C] and covariance [N][C][C] = fc fc^T/(HW-1) + eps_cov*I of a feature batch
 * (ops.py:43-45,105-108), fp32 outputs. */
WCTB200_API int wctb200_covariance(const void* act, int N, int H, int W, int C, float eps_cov, float* mean, float* cov,
                       void* stream);
/*
 * symmetric eigen-decomposition of `count` CxC fp32 matrices by one-sided Jacobi.
 * a: [count][C][C] symmetric (overwritten: column i becomes s_i * u_i, u_i the unit eigenvector, s_i within 2e-4 relative of
 * sigma_i -- only the direction of a column is significant),
 * sigma: [count][C] = |lambda_i| (Rayleigh quotients against the input), sweeps: [count] (may be NULL). */
WCTB200_API int wctb200_jacobi_eigh(float* a, int C, int count, float* sigma, int32_t* sweeps, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* WCTB200_H */

/* dsin_b200.h -- C ABI of libdsin_b200.so (sm_100a only, no CPU fallback).
 *
 * The reference (ayziksha/DSIN, TF1 graph mode) has no native boundary: its hot path is the
 * five Python callables injected into AE (src/main.py:33, src/AE.py:12-24) whose bodies
 * are TensorFlow op calls.  This header is the boundary a maintainer binds instead of
 * those op calls (ctypes stub in INTEGRATION.md).  Each entry point names the reference
 * code it replaces (file:line relative to /root/reference/).
 *
 * Conventions
 *   - every function returns 0 on success, <0 on error; dsin_last_error(h) gives the text.
 *   - the caller owns every buffer; pointers are DEVICE pointers unless the name says
 *     "host"; shapes are explicit; tensors are dense.
 *   - every launch is asynchronous on the caller-supplied stream (cudaStream_t passed as
 *     void*); no function synchronises the device or the host.
 *   - a handle is not thread-safe; distinct handles are independent.
 *   - internal activation layout is NHWC (channels last) fp32, or "split fp16" (two
 *     NHWC fp16 planes hi, lo with value = hi + lo) for the 128-channel trunk.
 */
#ifndef DSIN_B200_H_
#define DSIN_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct dsin_handle_s* dsin_handle_t;

enum { DSIN_OK = 0, DSIN_ERR_ARG = -1, DSIN_ERR_CUDA = -2, DSIN_ERR_UNSUPPORTED = -3 };
enum { DSIN_ACT_NONE = 0, DSIN_ACT_RELU = 1, DSIN_ACT_LRELU02 = 2 };
enum { DSIN_POST_NONE = 0, DSIN_POST_DENORM_CLIP = 1, DSIN_POST_DENORM = 2,
       /* tensor-core path only: cout = 12 = (2x2 sub-pixel phases) x 3 colours; denormalise, clip and
          scatter to a (2h x 2w x 3) fp32 NHWC image (a stride-2 transposed conv written as one conv) */
       DSIN_POST_DENORM_CLIP_D2S = 3 };

int dsin_version(void);
int dsin_create(dsin_handle_t* out, int device);
int dsin_destroy(dsin_handle_t h);
const char* dsin_last_error(dsin_handle_t h);
/* number of kernels this handle has launched since creation (bench.py's gpu_launches). */
int64_t dsin_launch_count(dsin_handle_t h);

/* ---- layout / normalisation -----------------------------------------------------------
 * NCHW fp32 -> NHWC fp32, optionally (x-mean_c)/sqrt(var_c+1e-10) with the KITTI constants.
 * Replaces _Network._normalize (src/autoencoder_imgcomp.py:136-144) and the NHWC
 * transposes of SI_full_img (src/siFull_img.py:10-13). */
int dsin_nchw_to_nhwc(dsin_handle_t h, const float* x_nchw, float* y_nhwc, int n, int c, int hh,
                      int ww, int normalize, void* stream);
/* NHWC fp32 -> NCHW fp32 (src/siFull_img.py:42 and the public NCHW outputs of AE). */
int dsin_nhwc_to_nchw(dsin_handle_t h, const float* x_nhwc, float* y_nchw, int n, int c, int hh,
                      int ww, void* stream);
/* concat([normalize(x_dec), normalize(y_syn)], channel) -> NHWC 6ch (src/AE.py:67-68). */
int dsin_concat_normalize(dsin_handle_t h, const float* xdec_nhwc, const float* ysyn_nhwc,
                          float* out_nhwc6, int n, int hh, int ww, void* stream);

/* Same concat, written as a 32-channel split-fp16 NHWC tensor (channels 6..31 zero) for the tensor-core
 * SI-Net path (the first layer's weights are zero-padded to 32 input channels by the caller). */
int dsin_concat_normalize_split32(dsin_handle_t h, const float* xdec_nhwc, const float* ysyn_nhwc,
                                  uint16_t* hi, uint16_t* lo, int n, int hh, int ww, void* stream);

/* NCHW fp32 image (3 channels) -> normalised, space-to-depth(2), 32-channel split-fp16 NHWC
 * (n, h/2, w/2, 32): channel (sy*2+sx)*3+c = pixel (2a+sy, 2b+sx), colour c; channels 12..31 zero.  With it the
 * 5x5 stride-2 stem h1 (src/autoencoder_imgcomp.py:223) is a 3x3 stride-1 conv for the tensor-core kernel. */
int dsin_nchw_to_s2d_split32(dsin_handle_t h, const float* x_nchw, uint16_t* hi, uint16_t* lo, int n, int hh,
                             int ww, void* stream);

/* ---- K1/K2/K8: convolution + folded BN / bias + activation + residual adds --------------
 * Replaces slim.conv2d / slim.conv2d_transpose + slim.batch_norm + ReLU + the skip adds
 * (src/autoencoder_imgcomp.py:223-266,275-288) and the siNet convs (src/siNet.py:31-40).
 *   y = post( act( conv(x, w) * scale[co] + shift[co] ) + res1 + res2 )
 * x: NHWC (n,h,w,cin); w: [kh][kw][cin][cout] fp32 (for transposed: reference layout
 * [k][k][out][in] re-ordered by the caller to [k][k][in][out], no flip);
 * TF SAME padding; transposed != 0 means stride-2 transposed conv (output 2h x 2w).
 * res1/res2 may be NULL.  post: DSIN_POST_* (denormalise [+clip 0..255], cout must be 3). */
typedef struct {
  int n, h, w, cin, cout, kh, kw, stride, dilation, transposed, act, post;
  int dilation_x; /* 0 = same as `dilation`; otherwise the tap spacing along W (tensor-core path only:
                     used when two pixels are viewed as one 2*C-channel "pair pixel") */
  int flags;      /* DSIN_CONV_PAIR_SHARED (tensor-core path, cin = cout = 64 = two pixels x 32 channels, even
                     dilation): the weights are the plain [taps][32][32] slab, applied to each pixel of the pair */
} dsin_conv_desc_t;
enum { DSIN_CONV_PAIR_SHARED = 1,
       DSIN_CONV_NO_CTA_PAIR = 2, /* run a 128->128 layer on the one-CTA kernel (cross-check of the CTA-pair kernels) */
       DSIN_CONV_NO_WEIGHT_STATIONARY = 4, /* terms = 1, 3x3 128->128: use the tap-streaming CTA-pair kernel instead of
                                               the weight-stationary halo-tile kernel (cross-check) */
       DSIN_CONV_NO_HALO = 8, /* use the tap-streaming kernels (cross-check) instead of the halo-tile kernel of the
                                3x3 128->128 layers with terms = 3 (conv_h3) and of the row-band kernel of the 3x3
                                32->32 layers (conv_dil) */
       DSIN_CONV_CIN16 = 16 /* 3x3 32->32 layers on the row-band kernel: input channels 16..31 are zero (the SI-Net's
                               first layer, 6 live channels padded to 32), so their K-step is skipped */
};
int dsin_conv2d(dsin_handle_t h, const dsin_conv_desc_t* d, const float* x, const float* w,
                const float* scale, const float* shift, const float* res1, const float* res2,
                float* y, void* stream);

/* ---- K1 (tensor core): 3x3 stride-1 128->128 conv on split-fp16 activations -------------
 * Same arithmetic as dsin_conv2d for the 64 trunk layers
 * (src/autoencoder_imgcomp.py:229-234,257-262,286), on tcgen05 tensor cores.
 * x_hi/x_lo, y_hi/y_lo, res*_hi/lo: NHWC fp16 planes (value = hi + lo).
 * w_hi/w_lo: packed by dsin_pack_conv3x3_w: [tap 9][cout 128][cin 128] fp16 (K-major).
 * terms: 1 = hi*hi only (fp16-class), 3 = hi*hi + hi*lo + lo*hi (fp32-class).       */
int dsin_pack_conv3x3_w(dsin_handle_t h, const float* w_hwio, uint16_t* w_hi, uint16_t* w_lo,
                        float* wscale, int cin, int cout, void* stream);
int dsin_conv3x3_c128_tc(dsin_handle_t h, int n, int hh, int ww, const uint16_t* x_hi,
                         const uint16_t* x_lo, const uint16_t* w_hi, const uint16_t* w_lo,
                         const float* scale, const float* shift, int act,
                         const uint16_t* res1_hi, const uint16_t* res1_lo,
                         const uint16_t* res2_hi, const uint16_t* res2_lo, uint16_t* y_hi,
                         uint16_t* y_lo, int terms, void* stream);
/* Generic tensor-core convolution (tcgen05): any layer of dsin_conv2d with cin in {32,64,128} and
 * cout <= 128 -- stride 1 (any dilation), stride 2 (TMA element strides) and stride-2 transposed
 * (four sub-pixel phases).  Same arithmetic/epilogue as dsin_conv2d; replaces the same reference
 * lines (src/autoencoder_imgcomp.py:223-266, src/siNet.py:31-40).
 * x_hi/x_lo, res*: split-fp16 NHWC planes; output either split fp16 (y_hi,y_lo; cout % 16 == 0) or
 * fp32 NHWC (y_f32 != NULL).  Weights packed by dsin_pack_conv_w_tc from [taps][cin][cout] fp32 into
 * [tap][npad][cin] split fp16 (npad = dsin_conv_tc_npad(cout)); wscale[cout] are the per-cout
 * power-of-two factors the caller divides out of `scale`.
 * The entry point picks the kernel from the geometry: 3x3 128->128 stride 1 -> CTA-pair kernels with a halo-resident
 * activation tile (terms 3: conv_h3.cu; terms 1: weight-stationary conv_ws.cu); 3x3 32->32 stride 1 without residuals ->
 * row bands (any dilation, conv_dil.cu); everything else -> the
 * tap-streaming kernels (conv_tc2.cu for 128-channel outputs on CTA pairs, conv_tc.cu otherwise).  `flags` force
 * the tap-streaming forms for cross-checks. */
int dsin_conv_tc_npad(int cout);
int dsin_pack_conv_w_tc(dsin_handle_t h, const float* w_kkio, int taps, int cin, int cout, uint16_t* w_hi,
                        uint16_t* w_lo, float* wscale, void* stream);
int dsin_conv2d_tc(dsin_handle_t h, const dsin_conv_desc_t* d, int terms, const uint16_t* x_hi,
                   const uint16_t* x_lo, const uint16_t* w_hi, const uint16_t* w_lo, const float* scale,
                   const float* shift, const uint16_t* res1_hi, const uint16_t* res1_lo,
                   const uint16_t* res2_hi, const uint16_t* res2_lo, uint16_t* y_hi, uint16_t* y_lo,
                   float* y_f32, void* stream);
/* fp32 NHWC <-> split fp16 planes. */
int dsin_f32_to_split(dsin_handle_t h, const float* x, uint16_t* hi, uint16_t* lo, int64_t count,
                      void* stream);
int dsin_split_to_f32(dsin_handle_t h, const uint16_t* hi, const uint16_t* lo, float* y,
                      int64_t count, void* stream);

/* ---- K3: heatmap mask + scalar quantiser ------------------------------------------------
 * Replaces _get_heatmap3D/_mask_with_heatmap (src/autoencoder_imgcomp.py:173-201) and
 * quantizer._quantize1d (src/quantizer_imgcomp.py:43-95) + qbar (:132-133).
 * z33: NHWC (n,hh,ww,c+1) output of to_bn; centers: (L) fp32, L <= 16.
 * Outputs: qbar_nhwc (n,hh,ww,c) for the decoder; qbar_nchw (n,c,hh,ww) for the probability
 * model; symbols_nchw int64 (n,c,hh,ww); and the remaining fields of the reference's EncoderOutput
 * (src/autoencoder_imgcomp.py:15,239-245), all (n,c,hh,ww) fp32: qhard_nchw = centers[symbols],
 * z_nchw = the heatmap-masked bottleneck the quantiser saw, heatmap_nchw = the 3-D heatmap.
 * Any output pointer may be NULL. */
int dsin_heatmap_quantize(dsin_handle_t h, const float* z33_nhwc, const float* centers, int L,
                          int n, int hh, int ww, int c, float* qbar_nhwc, float* qbar_nchw,
                          int64_t* symbols_nchw, float* qhard_nchw, float* z_nchw,
                          float* heatmap_nchw, void* stream);

/* ---- K4: 3-D masked-conv probability model -> bits ---------------------------------------
 * Replaces _Network3D.bitcost / _ResShallow._logits / conv3d / pad_for_probclass3d
 * (src/probclass_imgcomp.py:63-106,185-196,214-261,268-292) and the numerator of
 * bits.bitcost_to_bpp (src/bits_imgcomp.py:13).
 * qbar_nchw (n,c,hh,ww) fp32, symbols (n,c,hh,ww) int64; weights are the four conv3d
 * filters, mask already applied, layout [D=2][H=3][W=3][cin][cout]; pad_value=centers[0].
 * bits_nchw (n,c,hh,ww) fp32 may be NULL; bits_sum (n) double = per-image sum of bits.
 * workspace: device scratch of dsin_probclass_workspace_bytes(n,c,hh,ww,k) bytes. */
int64_t dsin_probclass_workspace_bytes(int n, int c, int hh, int ww, int k);
int dsin_probclass_bits(dsin_handle_t h, const float* qbar_nchw, const int64_t* symbols, int n,
                        int c, int hh, int ww, int k, int L, float pad_value, const float* w0,
                        const float* b0, const float* w1, const float* b1, const float* w2,
                        const float* b2, const float* w3, const float* b3, float* bits_nchw,
                        double* bits_sum, void* workspace, void* stream);

/* Tensor-core variant: the two 24->24 layers and the 24->6 head run on tcgen05 (weights packed by
 * dsin_pack_conv_w_tc from [18][32][32] / [18][32][32] / [18][32][6] zero-padded fp32 tensors, scale =
 * 1/wscale, shift = bias); the 1->24 stem (w0,b0) stays on CUDA cores; a small kernel turns the ReLU'd
 * logits into bits (log-sum-exp cross entropy * log2 e) and per-image fp64 sums. */
int64_t dsin_probclass_tc_workspace_bytes(int n, int c, int hh, int ww);
int dsin_probclass_bits_tc(dsin_handle_t h, const float* qbar_nchw, const int64_t* symbols, int n, int c,
                           int hh, int ww, float pad_value, const float* w0, const float* b0,
                           const uint16_t* w1_hi, const uint16_t* w1_lo, const float* scale1,
                           const float* shift1, const uint16_t* w2_hi, const uint16_t* w2_lo,
                           const float* scale2, const float* shift2, const uint16_t* w3_hi,
                           const uint16_t* w3_lo, const float* scale3, const float* shift3, int terms,
                           float* bits_nchw, double* bits_sum, void* workspace, void* stream);

/* ---- K5-K7: SI-Finder ---------------------------------------------------------------------
 * Replaces SI_full_img (src/siFull_img.py:5-68), siFinder (src/siFinder.py:7-53),
 * reduce_mean_and_std_normalize_images (:56-73), rgb_transform (:138-154),
 * L2_or_pearson_corr Pearson branch (:76-135), the Gaussian prior of
 * AE.create_gaussian_masks (src/AE.py:193-220) and its multiply (src/siFinder.py:20).
 * The (h,w,P) score map and the mask are never materialised.
 *
 * dsin_sif_prepare: x_dec, y_dec NHWC (n,hh,ww,3) ->
 *    q (n,P,ph*pw*3) fp32 transformed patches (k = (dy*pw+dx)*3+c), P=(hh/ph)*(ww/pw)
 *    r (n,hh,ww,3)   fp32 transformed search image
 *    pstat (n,P,4)   fp32: sum_x, sum_x2, mean_x, den_x
 *    ystat (n,hp,wp,4) fp32: sum_y, mean_y, den_y, sum_y2   (hp=hh-ph+1, wp=ww-pw+1)
 * dsin_sif_match: argmax over positions of pearson(q_p, window)*mask_p ->
 *    row,col (n,P) int32, best (n,P) fp32 (masked score at the argmax).
 *    method: 0 = fp32 SIMT scoring of every position; 1 = tcgen05 fp16 coarse scoring +
 *    exact rescoring of the candidates.  workspace from dsin_sif_workspace_bytes.
 * dsin_sif_gather: crop_and_resize bilinear gather from the ORIGINAL y (src/siFinder.py:35-41)
 *    folded back to image layout (src/siFull_img.py:30-33): y_syn NHWC (n,hh,ww,3).       */
int dsin_sif_prepare(dsin_handle_t h, const float* xdec_nhwc, const float* ydec_nhwc, int n, int hh,
                     int ww, int ph, int pw, float* q, float* r, float* pstat, float* ystat,
                     void* stream);
int64_t dsin_sif_workspace_bytes(int n, int hh, int ww, int ph, int pw, int method);
int dsin_sif_match(dsin_handle_t h, const float* q, const float* r, const float* pstat,
                   const float* ystat, int n, int hh, int ww, int ph, int pw, int use_mask,
                   int method, int32_t* row, int32_t* col, float* best, void* workspace,
                   void* stream);
/* L2 + LAB matching (ae_config.use_L2andLAB = True), same arguments as the two entry points above.
 * dsin_sif_prepare_lab replaces rgb_transform's LAB branch, rgb_to_lab (src/siFinder.py:13-17,145-146,157-195):
 *    q, r are CIELAB transforms of the RAW 0..255 pixels (no normalisation); pstat, ystat as above.
 * dsin_sif_match_l2 replaces L2_or_pearson_corr's L2 branch, the mask multiply and tf.argmin
 *    (src/siFinder.py:20,28-29,91-103): argmin over positions of ((sx2 - 2*xy) + sy2) * mask_p, first index on
 *    ties -> row, col; best = the masked distance at the argmin.  Inputs must lie in [0, 255] (|LAB| < 65504 for
 *    the fp16 coarse pass of method 1).                                                                      */
int dsin_sif_prepare_lab(dsin_handle_t h, const float* xdec_nhwc, const float* ydec_nhwc, int n, int hh,
                         int ww, int ph, int pw, float* q, float* r, float* pstat, float* ystat,
                         void* stream);
int dsin_sif_match_l2(dsin_handle_t h, const float* q, const float* r, const float* pstat,
                      const float* ystat, int n, int hh, int ww, int ph, int pw, int use_mask,
                      int method, int32_t* row, int32_t* col, float* best, void* workspace,
                      void* stream);
/* Byte offset, within the workspace of a method-1 dsin_sif_match / dsin_sif_match_l2 call, of the int32 number
 * of (patch, group) work items that the exact pass rescored exhaustively (diagnostics).                        */
int64_t dsin_sif_work_count_offset(const void* workspace, int n, int hh, int ww, int ph, int pw);
int dsin_sif_gather(dsin_handle_t h, const float* y_nhwc, const int32_t* row, const int32_t* col,
                    int n, int hh, int ww, int ph, int pw, float* ysyn_nhwc, void* stream);

/* ---- K9: MS-SSIM, the metric of record ---------------------------------------------------------
 * Replaces ms_ssim_np_imgcomp.MultiScaleSSIM/_SSIMForMultiScale/_FSpecialGauss
 * (src/ms_ssim_np_imgcomp.py:51-200) as called by utils.msssim_x_vs_rec (src/utils.py:94-99), in
 * float64 on the device.  img1/img2: fp32 (groups, batch, height, width, depth); each group is reduced
 * separately (one group = one image).  out: (groups, 5, 2) doubles = per-level mean SSIM and mean CS;
 * MS-SSIM = prod_{l<4} cs_l^w_l * ssim_4^w_4 with the weights of ms_ssim_np_imgcomp.py:91-92. */
int64_t dsin_msssim_workspace_bytes(int groups, int batch, int height, int width, int depth);
int dsin_msssim(dsin_handle_t h, const float* img1, const float* img2, int groups, int batch, int height,
                int width, int depth, double* out_g52, void* workspace, void* stream);

/* ---- validation loss terms (SURVEY 8f N4, forward half) -----------------------------------------------
 * Replaces the reductions of AE.siNet_validate's loss_test (src/AE.py:76-99,120-131):
 * Distortions.get_mae_per_img / get_mse_per_img (src/Distortions_imgcomp.py:68-101), get_loss's reduce_mean(bc) and
 * reduce_mean(bc * heatmap) (:119-121) and tf.losses.absolute_difference(x, x_with_si) (src/AE.py:94).
 * x, x_dec, x_with_si: fp32 (n, img_elems) (x_with_si may be NULL: AE_only); bitcost, heatmap: fp32 (n, sym_elems)
 * (heatmap may be NULL); squared != 0 sums (x_dec - x)^2 instead of |x_dec - x|.
 * terms_n4: (n, 4) doubles = per image [sum dist(x_dec, x), sum |x - x_with_si|, sum bc, sum bc * heatmap]. */
int dsin_validation_terms(dsin_handle_t h, const float* x, const float* x_dec, const float* x_with_si,
                          const float* bitcost, const float* heatmap, int n, int64_t img_elems,
                          int64_t sym_elems, int squared, double* terms_n4, void* stream);

/* ---- PC1 entropy coder: real bitstreams from the probability model (SURVEY 8f N3) --------------------------
 * The reference has no coder, only its building blocks (src/probclass_imgcomp.py:361-482: per-symbol frequencies
 * from the context model, causal order).  The byte-exact format is specified in oracle/pc_codec.c.
 *   symbols   (n, c, hh, ww) int64, depth = bottleneck channel; ww <= 159
 *   centers   L fp32 quantiser centres (device); weights: HOST array of 8 DEVICE pointers
 *             {w0[13][K], b0[K], w1[14][K][K], b1, w2[14][K][K], b2, w3[14][K][L], b3[L]}, live-tap-major
 *             (tap, cin, cout) slices of the masked (2,3,3) kernels (src/probclass_imgcomp.py:150-176,227-261), k = 24
 *   bytes     (n, nstreams, cap) uint8, sizes (n, nstreams) int64: stream s of an image carries the depth slices
 *             d == s (mod nstreams); *status (device int) becomes non-zero if a stream did not fit in cap bytes
 * n * nstreams CTAs must be co-resident per launch (cooperative launch); larger batches are chunked internally. */
int64_t dsin_pc_codec_workspace_bytes(int n, int c, int hh, int ww);
int dsin_pc_encode(dsin_handle_t h, const int64_t* symbols, int n, int c, int hh, int ww, const float* centers, int L,
                   const float* const* weights, int k, int nstreams, uint8_t* bytes, int64_t cap, int64_t* sizes,
                   int* status, void* workspace, void* stream);
/* Same bytes as dsin_pc_encode, produced by the decoder's wavefront kernel run in encode mode (cross-check). */
int dsin_pc_encode_wavefront(dsin_handle_t h, const int64_t* symbols, int n, int c, int hh, int ww, const float* centers,
                             int L, const float* const* weights, int k, int nstreams, uint8_t* bytes, int64_t cap,
                             int64_t* sizes, int* status, void* workspace, void* stream);
int dsin_pc_decode(dsin_handle_t h, const uint8_t* bytes, int64_t cap, const int64_t* sizes, int n, int c, int hh, int ww,
                   const float* centers, int L, const float* const* weights, int k, int nstreams, int64_t* symbols,
                   int* status, void* workspace, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DSIN_B200_H_ */

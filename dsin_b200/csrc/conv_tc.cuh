// Internal (non-ABI) entry of the generic tensor-core conv for 3-D VALID convolutions.
#pragma once
#include <cuda.h>
#include "common.cuh"

struct ConvTc3dArgs {
  int vols, D, H, W;        // input volume (channels-last, 32 channels split fp16)
  int kd, kh, kw;           // kernel extent (output = input - k + 1 per axis)
  int cin, cout, terms, act;
  int ntaps, wtaps;         // live taps / taps in the packed weight tensor
  short tap_d[32], tap_h[32], tap_w[32], tap_wi[32];
  const uint16_t *x_hi, *x_lo, *w_hi, *w_lo;
  const float *scale, *shift;
  uint16_t *y_hi, *y_lo;    // split output (cout % 16 == 0) or
  float* y_f32;             // fp32 output (vols, Do, Ho, Wo, cout)
  const float* r1f;         // optional fp32 residual volume (vols, r1_d, r1_oh, r1_ow, r1_c), read at +offsets
  int r1_d, r1_oh, r1_ow, r1_dz, r1_dy, r1_dx, r1_c;
};

int conv_tc_valid3d(dsin_handle_t h, const ConvTc3dArgs& a, cudaStream_t st);

// CTA-pair (cta_group::2) kernel for the 128-cout, 64-channel-block convolutions (conv_tc2.cu).
struct ConvTc2Args {
  const float* scale;
  const float* shift;
  const __half *r1h, *r1l, *r2h, *r2l;
  __half *yh, *yl;
  int n, OH, OW, in_step, act, ntaps, nchunks;
  int tiles_w, tiles_h, total_tiles;
  short dy[25], dx[25], wi[25];
};
struct ConvTc2Res {  // TMA maps of the residual planes (r1 hi, r1 lo, r2 hi, r2 lo) and of the identity slab
  CUtensorMap plane[4];
  CUtensorMap ident;
  int nres;        // residual tensors (0..2)
  int has_lo[2];   // residual i carries a lo plane
};
int conv_tc2_launch(dsin_handle_t h, int terms, const CUtensorMap& xh, const CUtensorMap& xl, const CUtensorMap& wh,
                    const CUtensorMap& wl, const ConvTc2Args& p, cudaStream_t st);

// Weight-stationary, halo-tile CTA-pair kernel for the fp16-operand (terms = 1) 3x3 128->128 layers (conv_ws.cu).
struct ConvWsArgs {
  const float* scale;
  const float* shift;
  const __half *r1, *r2;  // optional residual tensors (fp16 NHWC, same shape as y)
  __half* y;
  int n, OH, OW, act;
  int tiles_w, tiles_h, total_tiles;  // filled by conv_ws_launch
};
int conv_ws_launch(dsin_handle_t h, const __half* x, const __half* w_packed, const ConvWsArgs& a, cudaStream_t st);

// fp32-class (terms = 3) 3x3 128->128 trunk layer on CTA pairs: halo-resident split-fp16 activation tile, streamed
// weights, separate accumulators for large / small product terms, staged TMA-store epilogue (conv_h3.cu).
struct ConvH3Args {
  const float* scale;
  const float* shift;
  const __half *r1h, *r1l, *r2h, *r2l;  // optional residual tensors (split fp16 NHWC; lo planes may be NULL)
  __half *yh, *yl;
  int n, OH, OW, act;
  int tiles_w, tiles_h, total_tiles;  // filled by conv_h3_launch
};
int conv_h3_launch(dsin_handle_t h, const __half* x_hi, const __half* x_lo, const __half* w_hi, const __half* w_lo,
                   const ConvH3Args& a, cudaStream_t st);

// 32-channel layers on a halo tile with a resident filter (conv_h32.cu): SI-Net 3x3 layers with dilation <= 4 and the
// (2,3,3) masked 3-D convolutions of the probability model.
struct ConvH32Args {
  const float* scale;
  const float* shift;
  __half *yh, *yl;   // split-fp16 output (cout == 32; yl may be NULL), or
  float* yf;         // fp32 output (n_out, OH, OW, cout)
  const float* r1f;  // optional cropped fp32 residual volume (3-D mode), read at +offsets
  int r1_d, r1_oh, r1_ow, r1_dz, r1_dy, r1_dx, r1_c;
  int n_out;         // output images (2-D: n; 3-D: vols * Do)
  int dout, din;     // 3-D: Do, D -- output image n reads input images (n / Do) * D + n % Do + tz; 2-D: 0, 0
  int OH, OW, cout, act, terms;
  int ntaps;
  short tz[18], ty[18], tx[18], tw[18];  // tap offsets inside the halo box (pixels), weight slab index
  int hw, hh, hd;    // halo box extent (pixels, rows, depth slices)
  int ox, oy;        // halo origin relative to the tile origin (-dilation for SAME, 0 for VALID)
  int tiles_w, tiles_h, total_tiles, w_plane, w_region, a_plane, na;  // filled by conv_h32_launch
};
// conv_dil.cu: 3x3, 32 -> 32 channels, stride 1, SAME, dilation `dil` >= 1, split-fp16 or fp16 output
struct ConvDilArgs {
  const float* scale;
  const float* shift;
  __half *yh, *yl;  // output planes (n, H, W, 32); yl may be NULL with terms == 1
  int n, H, W, dil, act, terms;
  int ksteps;       // 16-channel K-steps that carry data: 2, or 1 when input channels 16..31 are zero
  // filled by conv_dil_launch
  int nbox, bw, a_plane, w_region, nb, tiles_w, phases, seg, nseg, total_units;
};
int conv_dil_launch(dsin_handle_t h, const __half* x_hi, const __half* x_lo, const __half* w_hi, const __half* w_lo,
                    const ConvDilArgs& a, cudaStream_t st);
int conv_h32_launch(dsin_handle_t h, const __half* x_hi, const __half* x_lo, const __half* w_hi, const __half* w_lo,
                    int W, int H, int ND, int wtaps, const ConvH32Args& a, cudaStream_t st);

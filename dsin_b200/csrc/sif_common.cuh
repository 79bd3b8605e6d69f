// Shared SI-Finder device helpers: the reference's Pearson and L2 algebra in literal fp32, the exact
// Gaussian prior, and the packed (score, first-index) key used for argmax reductions.
#pragma once
#include "common.cuh"

// Matching metric (ae_config.use_L2andLAB, src/siFinder.py:13-17,28-31,102-103).  The L2 path ranks the NEGATED
// masked distance, so every argmax reduction, the packed keys and the first-index tie-break serve tf.argmin unchanged.
enum SifMetric { SIF_PEARSON = 0, SIF_L2 = 1 };

// src/siFinder.py:103 (L2 branch): out = sum_x_square - 2*xy + sum_y_square, evaluated (sx2 - 2*xy) + sy2 in fp32.
__device__ __forceinline__ float sif_l2(float xy, float sx2, float sy2) {
  return __fadd_rn(__fsub_rn(sx2, __fmul_rn(2.f, xy)), sy2);
}

// src/siFinder.py:114-133, evaluated left to right in fp32 without FMA contraction.
//   num = xy - y_mean*sum_x - sum_y*x_mean + n*(y_mean*x_mean);  out = num / sqrt(den_y*den_x)
__device__ __forceinline__ float sif_pearson(float xy, float sum_y, float y_mean, float den_y, float sum_x,
                                             float x_mean, float den_x, float nf) {
  float num = __fsub_rn(xy, __fmul_rn(y_mean, sum_x));
  num = __fsub_rn(num, __fmul_rn(sum_y, x_mean));
  num = __fadd_rn(num, __fmul_rn(nf, __fmul_rn(y_mean, x_mean)));
  float den = __fmul_rn(den_y, den_x);
  return __fdiv_rn(num, __fsqrt_rn(den));
}

// AE.create_gaussian_masks (src/AE.py:193-220): float64 math, cast to float32; value for patch p
// at correlation index (i, j).  The crop offsets (ph/2-1, pw/2-1) put the peak at (top+1,left+1).
__device__ __forceinline__ float sif_mask_exact(int p, int i, int j, int hh, int ww, int ph, int pw) {
  double patch_img_w = (double)ww / (double)pw;
  double pr = floor((double)p / patch_img_w);
  double pc = (double)p - pr * patch_img_w;  // p % patch_img_w for exact integer-valued floats
  double ch = (pr + 0.5) * ph, cw = (pc + 0.5) * pw;
  double sh = 0.5 * hh, sw = 0.5 * ww;
  double dh = (double)(i + ph / 2 - 1) - ch, dw = (double)(j + pw / 2 - 1) - cw;
  double rows = dh * dh / (sh * sh), cols = dw * dw / (sw * sw);
  return (float)exp(-2.772588722239781 * (rows + cols));
}

// Packed key: high 32 bits = order-preserving image of the score, low 32 = ~index, so that a
// 64-bit max is "largest score, then smallest index" (tf.argmax first-occurrence tie-break).
// NaN scores map to 0 = "no entry" (a NaN never beats a number; all-NaN -> index 0).
__device__ __forceinline__ unsigned long long sif_pack(float s, unsigned idx) {
  if (s != s) return 0ull;
  s = __fadd_rn(s, 0.0f);  // -0 -> +0
  unsigned u = __float_as_uint(s);
  u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
  return ((unsigned long long)u << 32) | (unsigned long long)(0xFFFFFFFFu - idx);
}
__device__ __forceinline__ void sif_unpack(unsigned long long k, float* s, unsigned* idx) {
  unsigned u = (unsigned)(k >> 32);
  u = (u & 0x80000000u) ? (u & 0x7FFFFFFFu) : ~u;
  *s = __uint_as_float(u);
  *idx = 0xFFFFFFFFu - (unsigned)(k & 0xFFFFFFFFull);
}

// tcgen05 coarse scorer + exact rescoring (sif_tc.cu)
int64_t sif_tc_workspace_bytes(int n, int hh, int ww, int ph, int pw, int method);
int64_t sif_tc_work_count_offset(const void* ws, int n, int hh, int ww, int ph, int pw);
int sif_tc_match(dsin_handle_t h, const float* q, const float* r, const float* pstat, const float* ystat,
                 int n, int hh, int ww, int ph, int pw, int use_mask, int metric, unsigned long long* keys, void* ws,
                 cudaStream_t st);

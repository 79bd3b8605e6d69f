// K5-K7: SI-Finder -- patch/search-image preparation, masked Pearson argmax, bilinear gather.
// src/siFull_img.py:5-68, src/siFinder.py:7-53,56-73,76-135,138-154, src/AE.py:193-220.
// The (h,w,P) correlation map (1.18 GB at 320x1224) and the Gaussian prior are never stored:
// scores are produced tile by tile and reduced to a packed (score, index) key per patch.
#include <type_traits>

#include "common.cuh"
#include "sif_common.cuh"

// ---------------------------------------------------------------------------------------------
// K5: prepare
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void sif_transform(const float* __restrict__ px, float* out) {
  // (v - mean)/div per channel, then [R+G, R-G, 0.5*(R+B)]  (src/siFinder.py:62-71,149-153)
  float R = __fdiv_rn(__fsub_rn(px[0], dsin_mean(0)), dsin_sif_div(0));
  float G = __fdiv_rn(__fsub_rn(px[1], dsin_mean(1)), dsin_sif_div(1));
  float B = __fdiv_rn(__fsub_rn(px[2], dsin_mean(2)), dsin_sif_div(2));
  out[0] = __fadd_rn(R, G);
  out[1] = __fsub_rn(R, G);
  out[2] = __fmul_rn(0.5f, __fadd_rn(R, B));
}

// rgb_to_lab (src/siFinder.py:157-195) on the RAW 0..255 pixel values (the L2 branch skips the normalisation,
// :13-17), so the results lie far outside the usual CIELAB ranges (white: L ~ 9342).  Python scalars are float32
// constants, as TF makes them.  `** 2.4` and `** (1/3)` are pow(x, 2.4f) and pow(x, 0.333333343f), evaluated in
// fp64 and rounded once to fp32.  The 0/1-mask blends (:163-165,182-184) are branch selects: the inputs are finite
// and >= 0, so both forms give the same bits.  The two 3x3 matmuls have no pinned summation order in TF; they are
// defined here as left to right in fp32 without FMA (the oracle does the same).
__device__ __forceinline__ float sif_lab_f(float t) {  // xyz_to_cielab's piecewise f
  const float eps3 = 0.00885645207f, c3e2 = 0.12841855f, c429 = 0.137931034f;  // (6/29)^3, 3(6/29)^2, 4/29
  return t <= eps3 ? __fadd_rn(__fdiv_rn(t, c3e2), c429) : (float)pow((double)t, (double)0.333333343f);
}

__device__ __forceinline__ void sif_lab(const float* __restrict__ px, float* out) {
  float lin[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const float v = px[c];
    lin[c] = v <= 0.04045f ? __fdiv_rn(v, 12.92f)
                           : (float)pow((double)__fdiv_rn(__fadd_rn(v, 0.055f), 1.055f), (double)2.4f);
  }
  // rows R, G, B of rgb_to_xyz; columns X, Y, Z
  const float X = __fadd_rn(__fadd_rn(__fmul_rn(lin[0], 0.412453f), __fmul_rn(lin[1], 0.357580f)),
                            __fmul_rn(lin[2], 0.180423f));
  const float Y = __fadd_rn(__fadd_rn(__fmul_rn(lin[0], 0.212671f), __fmul_rn(lin[1], 0.715160f)),
                            __fmul_rn(lin[2], 0.072169f));
  const float Z = __fadd_rn(__fadd_rn(__fmul_rn(lin[0], 0.019334f), __fmul_rn(lin[1], 0.119193f)),
                            __fmul_rn(lin[2], 0.950227f));
  const float fx = sif_lab_f(__fmul_rn(X, 1.05212653f));  // float32(1/0.950456)
  const float fy = sif_lab_f(__fmul_rn(Y, 1.0f));
  const float fz = sif_lab_f(__fmul_rn(Z, 0.918481112f));  // float32(1/1.088754)
  // fxfyfz_to_lab, left to right, + [-16, 0, 0]
  out[0] = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(fx, 0.f), __fmul_rn(fy, 116.f)), __fmul_rn(fz, 0.f)), -16.f);
  out[1] = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(fx, 500.f), __fmul_rn(fy, -500.f)), __fmul_rn(fz, 0.f)), 0.f);
  out[2] = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(fx, 0.f), __fmul_rn(fy, 200.f)), __fmul_rn(fz, -200.f)), 0.f);
}

template <int METRIC>
__global__ void sif_transform_kernel(const float* __restrict__ xdec, const float* __restrict__ ydec,
                                     float* __restrict__ q, float* __restrict__ r, int n, int hh, int ww,
                                     int ph, int pw) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t npix = (int64_t)n * hh * ww;
  if (idx >= npix) return;
  float t[3];
  if constexpr (METRIC == SIF_L2) sif_lab(ydec + idx * 3, t);
  else sif_transform(ydec + idx * 3, t);
  r[idx * 3 + 0] = t[0];
  r[idx * 3 + 1] = t[1];
  r[idx * 3 + 2] = t[2];
  if constexpr (METRIC == SIF_L2) sif_lab(xdec + idx * 3, t);
  else sif_transform(xdec + idx * 3, t);
  int x = (int)(idx % ww);
  int64_t tt = idx / ww;
  int y = (int)(tt % hh);
  int img = (int)(tt / hh);
  int pcs = ww / pw, prs = hh / ph;
  int pr = y / ph, dy = y % ph, pc = x / pw, dx = x % pw;
  int64_t P = (int64_t)prs * pcs;
  int64_t o = (((int64_t)img * P + pr * pcs + pc) * (ph * pw) + dy * pw + dx) * 3;
  q[o + 0] = t[0];
  q[o + 1] = t[1];
  q[o + 2] = t[2];
}

// one warp per patch: sums in fp64, rounded once to fp32, then the reference's fp32 algebra
__global__ void sif_patch_stats_kernel(const float* __restrict__ q, float* __restrict__ pstat, int64_t np,
                                       int kdim) {
  int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / 32;
  int lane = threadIdx.x % 32;
  if (warp >= np) return;
  const float* qp = q + warp * kdim;
  double s = 0.0, s2 = 0.0;
  for (int k = lane; k < kdim; k += 32) {
    double v = (double)qp[k];
    s += v;
    s2 += v * v;
  }
  for (int o = 16; o > 0; o >>= 1) {
    s += __shfl_xor_sync(0xffffffffu, s, o);
    s2 += __shfl_xor_sync(0xffffffffu, s2, o);
  }
  if (lane == 0) {
    float nf = (float)kdim;
    float sx = (float)s, sx2 = (float)s2;
    float xm = (float)(s / (double)kdim);  // reduce_mean
    float denx = __fadd_rn(__fsub_rn(sx2, __fmul_rn(2.f, __fmul_rn(xm, sx))), __fmul_rn(nf, __fmul_rn(xm, xm)));
    pstat[warp * 4 + 0] = sx;
    pstat[warp * 4 + 1] = sx2;
    pstat[warp * 4 + 2] = xm;
    pstat[warp * 4 + 3] = denx;
  }
}

// horizontal window sums (pw pixels x 3 channels) in fp64: hs[(img,y,j)] = {sum, sum of squares}
__global__ void sif_hsum_kernel(const float* __restrict__ r, double2* __restrict__ hs, int n, int hh, int ww,
                                int pw) {
  int wp = ww - pw + 1;
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)n * hh * wp) return;
  int j = (int)(idx % wp);
  int64_t row = idx / wp;  // img*hh + y
  const float* rp = r + (row * ww + j) * 3;
  double s = 0.0, s2 = 0.0;
  for (int k = 0; k < pw * 3; ++k) {
    double v = (double)__ldg(rp + k);
    s += v;
    s2 += v * v;
  }
  hs[idx] = make_double2(s, s2);
}

__global__ void sif_ystat_kernel(const double2* __restrict__ hs, float* __restrict__ ystat, int n, int hh,
                                 int ww, int ph, int pw) {
  int wp = ww - pw + 1, hp = hh - ph + 1;
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)n * hp * wp) return;
  int j = (int)(idx % wp);
  int64_t t = idx / wp;
  int i = (int)(t % hp);
  int img = (int)(t / hp);
  double s = 0.0, s2 = 0.0;
  for (int dy = 0; dy < ph; ++dy) {
    double2 v = hs[((int64_t)img * hh + i + dy) * wp + j];
    s += v.x;
    s2 += v.y;
  }
  float nf = (float)(ph * pw * 3);
  float inv = __fdiv_rn(1.0f, nf);  // the constant 1/patch_size kernel of src/siFinder.py:107
  float sy = (float)s, sy2 = (float)s2;
  float ym = (float)(s * (double)inv);
  float deny = __fadd_rn(__fsub_rn(sy2, __fmul_rn(2.f, __fmul_rn(ym, sy))), __fmul_rn(nf, __fmul_rn(ym, ym)));
  float4 o = make_float4(sy, ym, deny, sy2);
  reinterpret_cast<float4*>(ystat)[idx] = o;
}

// ---------------------------------------------------------------------------------------------
// K6 method 0: scoring of every (position, patch) on CUDA cores
// tile = 64 positions of one correlation row x 64 patches; K loop over the ph patch rows.
// Pearson accumulates the dot product in fp32.  L2 accumulates it in fp64 (exact products), rounded once to fp32 as
// the oracle does: a ~1e10 fp32 sum of 1440 LAB products is off by far more than the gaps between distances.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float sif_mac(float a, float b, float c) { return fmaf(a, b, c); }
__device__ __forceinline__ double sif_mac(float a, float b, double c) { return fma((double)a, (double)b, c); }

template <int PW, int METRIC>
__global__ void __launch_bounds__(256) sif_score_simt_kernel(const float* __restrict__ q,
                                                             const float* __restrict__ r,
                                                             const float* __restrict__ pstat,
                                                             const float* __restrict__ ystat, int n, int hh,
                                                             int ww, int ph, int use_mask,
                                                             unsigned long long* __restrict__ keys) {
  constexpr int KROW = PW * 3;          // elements per patch row
  constexpr int RSEG = (64 + PW - 1) * 3;
  __shared__ float s_r[RSEG + 3];
  __shared__ float s_q[KROW][64 + 4];
  __shared__ unsigned long long s_key[16][64];

  const int wp = ww - PW + 1, hp = hh - ph + 1;
  const int pcs = ww / PW, P = (hh / ph) * pcs;
  const int ptiles = (P + 63) / 64;
  const int img = blockIdx.z / ptiles, pt = blockIdx.z % ptiles;
  const int i = blockIdx.y, j0 = blockIdx.x * 64;
  const int tid = threadIdx.x, ty = tid / 16, tx = tid % 16;
  const int kdim = ph * KROW;

  using Acc = typename std::conditional<METRIC == SIF_L2, double, float>::type;
  Acc acc[4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) acc[a][b] = 0;

  for (int dy = 0; dy < ph; ++dy) {
    const float* rrow = r + (((int64_t)img * hh + i + dy) * ww + j0) * 3;
    int avail = (ww - j0) * 3;
    for (int e = tid; e < RSEG; e += 256) s_r[e] = e < avail ? __ldg(rrow + e) : 0.f;
    for (int e = tid; e < KROW * 64; e += 256) {
      int k = e % KROW, pl = e / KROW;
      int p = pt * 64 + pl;
      s_q[k][pl] = p < P ? __ldg(q + ((int64_t)img * P + p) * kdim + dy * KROW + k) : 0.f;
    }
    __syncthreads();
#pragma unroll 8
    for (int k = 0; k < KROW; ++k) {
      float4 b = *reinterpret_cast<const float4*>(&s_q[k][tx * 4]);
      float a0 = s_r[(ty * 4 + 0) * 3 + k];
      float a1 = s_r[(ty * 4 + 1) * 3 + k];
      float a2 = s_r[(ty * 4 + 2) * 3 + k];
      float a3 = s_r[(ty * 4 + 3) * 3 + k];
      acc[0][0] = sif_mac(a0, b.x, acc[0][0]); acc[0][1] = sif_mac(a0, b.y, acc[0][1]);
      acc[0][2] = sif_mac(a0, b.z, acc[0][2]); acc[0][3] = sif_mac(a0, b.w, acc[0][3]);
      acc[1][0] = sif_mac(a1, b.x, acc[1][0]); acc[1][1] = sif_mac(a1, b.y, acc[1][1]);
      acc[1][2] = sif_mac(a1, b.z, acc[1][2]); acc[1][3] = sif_mac(a1, b.w, acc[1][3]);
      acc[2][0] = sif_mac(a2, b.x, acc[2][0]); acc[2][1] = sif_mac(a2, b.y, acc[2][1]);
      acc[2][2] = sif_mac(a2, b.z, acc[2][2]); acc[2][3] = sif_mac(a2, b.w, acc[2][3]);
      acc[3][0] = sif_mac(a3, b.x, acc[3][0]); acc[3][1] = sif_mac(a3, b.y, acc[3][1]);
      acc[3][2] = sif_mac(a3, b.z, acc[3][2]); acc[3][3] = sif_mac(a3, b.w, acc[3][3]);
    }
    __syncthreads();
  }

  // epilogue: Pearson or L2, prior, per-thread best over its 4 positions for each of its 4 patches
  const float nf = (float)kdim;
  unsigned long long best[4] = {0ull, 0ull, 0ull, 0ull};
#pragma unroll
  for (int b = 0; b < 4; ++b) {
    int p = pt * 64 + tx * 4 + b;
    if (p >= P) continue;
    const float* ps = pstat + ((int64_t)img * P + p) * 4;
    float sx = ps[0], xm = ps[2], denx = ps[3];
#pragma unroll
    for (int a = 0; a < 4; ++a) {
      int j = j0 + ty * 4 + a;
      if (j >= wp) continue;
      float4 ys = reinterpret_cast<const float4*>(ystat)[((int64_t)img * hp + i) * wp + j];
      float s;
      if constexpr (METRIC == SIF_L2) {  // the negated masked distance: its argmax is tf.argmin's
        s = sif_l2((float)acc[a][b], ps[1], ys.w);
        if (use_mask) s = __fmul_rn(s, sif_mask_exact(p, i, j, hh, ww, ph, PW));
        s = -s;
      } else {
        s = sif_pearson(acc[a][b], ys.x, ys.y, ys.z, sx, xm, denx, nf);
        if (use_mask) s = __fmul_rn(s, sif_mask_exact(p, i, j, hh, ww, ph, PW));
      }
      unsigned long long key = sif_pack(s, (unsigned)(i * wp + j));
      best[b] = key > best[b] ? key : best[b];
    }
  }
#pragma unroll
  for (int b = 0; b < 4; ++b) s_key[ty][tx * 4 + b] = best[b];
  __syncthreads();
  if (tid < 64) {
    unsigned long long k = 0ull;
#pragma unroll
    for (int t = 0; t < 16; ++t) k = s_key[t][tid] > k ? s_key[t][tid] : k;
    int p = pt * 64 + tid;
    if (p < P && k != 0ull) atomicMax(keys + (int64_t)img * P + p, k);
  }
}

__global__ void sif_finalize_keys_kernel(const unsigned long long* __restrict__ keys, int64_t np, int wp,
                                         int32_t* __restrict__ row, int32_t* __restrict__ col,
                                         float* __restrict__ best, int negate) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= np) return;
  unsigned long long k = keys[idx];
  unsigned pos = 0;
  float s = __int_as_float(0x7fc00000);  // all-NaN column -> index 0 (tf.argmax), score NaN
  if (k != 0ull) sif_unpack(k, &s, &pos);
  row[idx] = (int32_t)(pos / (unsigned)wp);
  col[idx] = (int32_t)(pos % (unsigned)wp);
  if (best) best[idx] = negate ? -s : s;  // L2 keys hold the negated masked distance
}

// ---------------------------------------------------------------------------------------------
// K7: crop_and_resize gather + fold (src/siFinder.py:35-41, src/siFull_img.py:30-33)
// ---------------------------------------------------------------------------------------------
__global__ void sif_gather_kernel(const float* __restrict__ y, const int32_t* __restrict__ row,
                                  const int32_t* __restrict__ col, int n, int hh, int ww, int ph, int pw,
                                  float* __restrict__ ysyn) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;  // output pixel (img, oy, ox)
  if (idx >= (int64_t)n * hh * ww) return;
  int ox = (int)(idx % ww);
  int64_t t = idx / ww;
  int oy = (int)(t % hh);
  int img = (int)(t / hh);
  int pcs = ww / pw;
  int pr = oy / ph, ty = oy % ph, pc = ox / pw, tx = ox % pw;
  int64_t P = (int64_t)(hh / ph) * pcs;
  int64_t pi = (int64_t)img * P + pr * pcs + pc;
  int rr = row[pi], cc = col[pi];
  float y1 = (float)((double)rr / (double)hh), x1 = (float)((double)cc / (double)ww);
  float y2 = (float)((double)(rr + ph) / (double)hh), x2 = (float)((double)(cc + pw) / (double)ww);
  float hs = __fdiv_rn(__fmul_rn(__fsub_rn(y2, y1), (float)(hh - 1)), (float)(ph - 1));
  float ws = __fdiv_rn(__fmul_rn(__fsub_rn(x2, x1), (float)(ww - 1)), (float)(pw - 1));
  float in_y = __fadd_rn(__fmul_rn(y1, (float)(hh - 1)), __fmul_rn((float)ty, hs));
  float in_x = __fadd_rn(__fmul_rn(x1, (float)(ww - 1)), __fmul_rn((float)tx, ws));
  float* o = ysyn + idx * 3;
  if (in_y < 0.f || in_y > (float)(hh - 1) || in_x < 0.f || in_x > (float)(ww - 1)) {
    o[0] = o[1] = o[2] = 0.f;  // extrapolation_value
    return;
  }
  int top = (int)floorf(in_y), bot = (int)ceilf(in_y);
  int lef = (int)floorf(in_x), rig = (int)ceilf(in_x);
  float ly = __fsub_rn(in_y, (float)top), lx = __fsub_rn(in_x, (float)lef);
  const float* base = y + (int64_t)img * hh * ww * 3;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    float tl = base[((int64_t)top * ww + lef) * 3 + c], tr = base[((int64_t)top * ww + rig) * 3 + c];
    float bl = base[((int64_t)bot * ww + lef) * 3 + c], br = base[((int64_t)bot * ww + rig) * 3 + c];
    float T = __fadd_rn(tl, __fmul_rn(__fsub_rn(tr, tl), lx));
    float B = __fadd_rn(bl, __fmul_rn(__fsub_rn(br, bl), lx));
    o[c] = __fadd_rn(T, __fmul_rn(__fsub_rn(B, T), ly));
  }
}

// ---------------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------------
template <int METRIC>
static int sif_prepare(dsin_handle_t h, const float* xdec, const float* ydec, int n, int hh, int ww, int ph, int pw,
                       float* q, float* r, float* pstat, float* ystat, void* stream) {
  DSIN_REQUIRE(h, xdec && ydec && q && r && pstat && ystat, "null pointer");
  DSIN_REQUIRE(h, n > 0 && ph > 1 && pw > 1 && hh % ph == 0 && ww % pw == 0, "image must tile into patches");
  cudaStream_t st = (cudaStream_t)stream;
  int64_t npix = (int64_t)n * hh * ww;
  sif_transform_kernel<METRIC><<<(unsigned)((npix + 255) / 256), 256, 0, st>>>(xdec, ydec, q, r, n, hh, ww, ph, pw);
  DSIN_LAUNCHED(h);
  int64_t np = (int64_t)n * (hh / ph) * (ww / pw);
  sif_patch_stats_kernel<<<(unsigned)((np * 32 + 255) / 256), 256, 0, st>>>(q, pstat, np, ph * pw * 3);
  DSIN_LAUNCHED(h);
  // the fp64 horizontal sums live in the tail of ystat's own allocation? no: use a stream-ordered scratch
  int wp = ww - pw + 1, hp = hh - ph + 1;
  double2* hs = nullptr;
  if (cudaMallocAsync((void**)&hs, sizeof(double2) * (size_t)n * hh * wp, st) != cudaSuccess)
    return dsin_fail(h, DSIN_ERR_CUDA, "%s: scratch allocation failed", __func__);
  int64_t t1 = (int64_t)n * hh * wp;
  sif_hsum_kernel<<<(unsigned)((t1 + 255) / 256), 256, 0, st>>>(r, hs, n, hh, ww, pw);
  DSIN_LAUNCHED(h);
  int64_t t2 = (int64_t)n * hp * wp;
  sif_ystat_kernel<<<(unsigned)((t2 + 255) / 256), 256, 0, st>>>(hs, ystat, n, hh, ww, ph, pw);
  DSIN_LAUNCHED(h);
  cudaFreeAsync(hs, st);
  return DSIN_OK;
}

template <int METRIC>
static int sif_match(dsin_handle_t h, const float* q, const float* r, const float* pstat, const float* ystat, int n,
                     int hh, int ww, int ph, int pw, int use_mask, int method, int32_t* row, int32_t* col, float* best,
                     void* workspace, void* stream) {
  DSIN_REQUIRE(h, q && r && pstat && ystat && row && col && workspace, "null pointer");
  DSIN_REQUIRE(h, n > 0 && hh % ph == 0 && ww % pw == 0, "image must tile into patches");
  cudaStream_t st = (cudaStream_t)stream;
  int P = (hh / ph) * (ww / pw);
  int wp = ww - pw + 1, hp = hh - ph + 1;
  unsigned long long* keys = (unsigned long long*)workspace;
  if (cudaMemsetAsync(keys, 0, sizeof(unsigned long long) * (size_t)n * P, st) != cudaSuccess)
    return dsin_fail(h, DSIN_ERR_CUDA, "%s: memset failed", __func__);
  if (method == 0) {
    DSIN_REQUIRE(h, pw == 24, "SIMT scorer is built for 24-pixel-wide patches");
    dim3 grid((wp + 63) / 64, hp, n * ((P + 63) / 64));
    sif_score_simt_kernel<24, METRIC><<<grid, 256, 0, st>>>(q, r, pstat, ystat, n, hh, ww, ph, use_mask, keys);
    DSIN_LAUNCHED(h);
  } else {
    int rc = sif_tc_match(h, q, r, pstat, ystat, n, hh, ww, ph, pw, use_mask, METRIC, keys,
                          (char*)workspace + sizeof(unsigned long long) * (size_t)n * P, st);
    if (rc != DSIN_OK) return rc;
  }
  int64_t np = (int64_t)n * P;
  sif_finalize_keys_kernel<<<(unsigned)((np + 255) / 256), 256, 0, st>>>(keys, np, wp, row, col, best,
                                                                       METRIC == SIF_L2);
  DSIN_LAUNCHED(h);
  return DSIN_OK;
}

extern "C" {

int dsin_sif_prepare(dsin_handle_t h, const float* xdec, const float* ydec, int n, int hh, int ww, int ph,
                     int pw, float* q, float* r, float* pstat, float* ystat, void* stream) {
  return sif_prepare<SIF_PEARSON>(h, xdec, ydec, n, hh, ww, ph, pw, q, r, pstat, ystat, stream);
}

int dsin_sif_prepare_lab(dsin_handle_t h, const float* xdec, const float* ydec, int n, int hh, int ww, int ph,
                         int pw, float* q, float* r, float* pstat, float* ystat, void* stream) {
  return sif_prepare<SIF_L2>(h, xdec, ydec, n, hh, ww, ph, pw, q, r, pstat, ystat, stream);
}

int64_t dsin_sif_workspace_bytes(int n, int hh, int ww, int ph, int pw, int method) {
  int64_t P = (int64_t)(hh / ph) * (ww / pw);
  return sif_tc_workspace_bytes(n, hh, ww, ph, pw, method) + n * P * 8 + 1024;
}

int64_t dsin_sif_work_count_offset(const void* workspace, int n, int hh, int ww, int ph, int pw) {
  const int64_t keys = (int64_t)n * (hh / ph) * (ww / pw) * 8;
  return keys + sif_tc_work_count_offset((const char*)workspace + keys, n, hh, ww, ph, pw);
}

int dsin_sif_match(dsin_handle_t h, const float* q, const float* r, const float* pstat, const float* ystat,
                   int n, int hh, int ww, int ph, int pw, int use_mask, int method, int32_t* row,
                   int32_t* col, float* best, void* workspace, void* stream) {
  return sif_match<SIF_PEARSON>(h, q, r, pstat, ystat, n, hh, ww, ph, pw, use_mask, method, row, col, best,
                                workspace, stream);
}

int dsin_sif_match_l2(dsin_handle_t h, const float* q, const float* r, const float* pstat, const float* ystat,
                      int n, int hh, int ww, int ph, int pw, int use_mask, int method, int32_t* row,
                      int32_t* col, float* best, void* workspace, void* stream) {
  return sif_match<SIF_L2>(h, q, r, pstat, ystat, n, hh, ww, ph, pw, use_mask, method, row, col, best, workspace,
                           stream);
}

int dsin_sif_gather(dsin_handle_t h, const float* y, const int32_t* row, const int32_t* col, int n, int hh,
                    int ww, int ph, int pw, float* ysyn, void* stream) {
  DSIN_REQUIRE(h, y && row && col && ysyn && n > 0, "bad argument");
  int64_t tot = (int64_t)n * hh * ww;
  sif_gather_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, (cudaStream_t)stream>>>(y, row, col, n, hh, ww, ph,
                                                                                 pw, ysyn);
  DSIN_LAUNCHED(h);
  return DSIN_OK;
}

}  // extern "C"

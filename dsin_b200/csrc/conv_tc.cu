// K1/K2/K8 on tensor cores: convolution as a tcgen05 implicit GEMM, generic over
//   kernel taps (3x3, 5x5, 1x1), dilation, stride 2 (TMA element strides) and stride-2 TRANSPOSED
//   convolution (four sub-pixel phases, each a stride-1 conv over a subset of the taps),
//   cin in {32, 64, 128}, cout <= 128.
// Replaces slim.conv2d / conv2d_transpose + batch_norm + ReLU + skip adds
// (src/autoencoder_imgcomp.py:223-266,275-288) and the SI-Net convs (src/siNet.py:31-40).
//
// GEMM view per tile: D[128 grid pixels x NPAD couts] = sum over taps t, channel blocks c of
//   A_{t,c}[128 px x KC ci] * B_{t,c}[KC ci x NPAD co].
// A comes straight from the NHWC fp16 activation by a 4-D TMA box (KC ch, 16 w, 8 h, 1 n) whose
// (w,h) origin is shifted by the tap offset; out-of-bounds elements are zero-filled by TMA, which IS
// TF 'SAME' zero padding (and the implicit zeros of the transposed conv).  B is the per-tap [co][ci]
// weight slab (K-major).  Both land in shared memory in the swizzled K-major layout tcgen05.mma
// consumes; accumulators live in TMEM (double buffered) so the epilogue of tile i overlaps the MMAs of
// tile i+1.
//
// Precision ("terms"): activations and weights are split fp16 pairs (v = hi + lo).
//   terms = 3:  hi*hi + hi*lo + lo*hi  -> ~22-bit operands, fp32-class result (parity mode)
//   terms = 1:  hi*hi only             -> fp16 operands (fast mode)
// Warp roles (192 threads): warp 0 = TMA producer, warp 1 = MMA issuer (+TMEM alloc),
// warps 2-5 = epilogue (TMEM -> registers -> scale/shift/act/residual/post -> global).
#include "tc_common.cuh"
#include "conv_tc.cuh"

using namespace tc;

namespace {

constexpr int BW = 16, BH = 8;  // spatial tile: 8 rows x 16 cols = 128 GEMM rows
constexpr int MAX_TAPS = 25;

struct GP {
  const float* scale;
  const float* shift;
  const __half *r1h, *r1l, *r2h, *r2l;
  __half *yh, *yl;
  float* yf;
  int n, GH, GW, OH, OW, cout, os, py, px, in_step, act, post, ntaps, nchunks;
  int tiles_w, tiles_h, total_tiles;
  short dy[MAX_TAPS], dx[MAX_TAPS], wi[MAX_TAPS], dz[MAX_TAPS];
  // 3-D (VALID) mode: tile "image" index n = vol * dout + d; the A box comes from image
  // vol * din + d + dz[tap].  dout == 0 means plain 2-D (image index passes through).
  int dout, din;
  // optional fp32 residual with its own geometry (cropped skip of the probability model)
  const float* r1f;
  int r1_d, r1_oh, r1_ow, r1_dz, r1_dy, r1_dx, r1_c;
};

constexpr int up1024(int v) { return (v + 1023) / 1024 * 1024; }

template <int KC, int NPAD, int TERMS, bool PS = false, int NSPLIT = 1>
struct Cfg {
  // k-blocks (tap, channel chunk) per pipeline stage: the 32-channel layers have so little MMA work per
  // k-block (N <= 128, K = 32) that the fixed per-stage cost dominates; they take 3 k-blocks per stage.
  static constexpr int kTps = KC == 32 ? 3 : 1;
  static constexpr int kA = up1024(128 * KC * 2);
  // PS (pair-shared): B is the [32 cout][32 cin] slab (64-byte rows), used for both pixels of the pair
  static constexpr int kB = PS ? up1024(32 * 32 * 2) : up1024(NPAD * KC * 2);
  static constexpr int kSub = (TERMS == 3 ? 2 : 1) * (kA + kB);
  static constexpr int kStage = kTps * kSub;
  static constexpr int kStagesRaw = (196 * 1024) / kStage;
  static constexpr int kStages = kStagesRaw > 8 ? 8 : kStagesRaw;
  static constexpr int kSmem = kStages * kStage + 1024 + 2048;
  // accumulator columns per buffer: TERMS == 3 keeps the hi*hi products and the 2^-11-times-smaller hi*lo + lo*hi
  // products in SEPARATE accumulators (tcgen05 accumulates with round-toward-zero: every MMA into an accumulator of
  // magnitude |acc| can lose an ulp(|acc|); the small terms must not pay, nor add, roundings at the large magnitude)
  // NSPLIT > 1 additionally deals the hi*hi k-blocks round-robin onto NSPLIT accumulators (a 5x5 layer is 200 MMAs
  // deep: to_bn, the layer that produces the quantiser's input, runs with 4), summed in fp32 by the epilogue.
  static constexpr int kAccCols = (TERMS == 3 ? NSPLIT + 1 : 1) * NPAD;
  static_assert(NSPLIT == 1 || (TERMS == 3 && !PS && KC == 64), "split accumulators: 3-term, 64-channel k-blocks");
  static constexpr int kTmemCols = 2 * kAccCols <= 32 ? 32 : (2 * kAccCols <= 64 ? 64 : (2 * kAccCols <= 128 ? 128 : (2 * kAccCols <= 256 ? 256 : 512)));
  static constexpr uint32_t kLayout = KC == 64 ? LAYOUT_SW128 : LAYOUT_SW64;
  static constexpr uint32_t kSbo = KC == 64 ? 1024 : 512;
};

__device__ __forceinline__ void unpack8(const uint4& u, float* f) {
  const __half2* h = reinterpret_cast<const __half2*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float2 t = __half22float2(h[i]);
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}

__device__ __forceinline__ void add_residual16(float* f, const __half* rh, const __half* rl, size_t off) {
#pragma unroll
  for (int g = 0; g < 2; ++g) {
    float a[8], b[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(rh + off) + g), a);
    if (rl) {
      unpack8(__ldg(reinterpret_cast<const uint4*>(rl + off) + g), b);
#pragma unroll
      for (int e = 0; e < 8; ++e) a[e] = __fadd_rn(a[e], b[e]);
    }
#pragma unroll
    for (int e = 0; e < 8; ++e) f[g * 8 + e] = __fadd_rn(f[g * 8 + e], a[e]);
  }
}

template <int KC, int NPAD, int TERMS, bool PS = false, int NSPLIT = 1>
__global__ void __launch_bounds__(192, 1)
conv_tc_kernel(const __grid_constant__ CUtensorMap tm_xh, const __grid_constant__ CUtensorMap tm_xl,
               const __grid_constant__ CUtensorMap tm_wh, const __grid_constant__ CUtensorMap tm_wl,
               const __grid_constant__ GP p) {
  using C = Cfg<KC, NPAD, TERMS, PS, NSPLIT>;
  static_assert(!PS || (KC == 64 && NPAD == 64), "pair-shared mode is 2 pixels x 32 channels");
  constexpr int S = C::kStages;
  constexpr int STAGE = C::kStage;
  constexpr int TPS = C::kTps;
  constexpr int OFF_B = C::kA, OFF_ALO = C::kA + C::kB, OFF_BLO = 2 * C::kA + C::kB;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + (((raw + 1023u) & ~1023u) - raw);
  uint8_t* tiles = smem;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + S * STAGE);
  uint64_t* empty = full + S;
  uint64_t* tfull = empty + S;
  uint64_t* tempty = tfull + 2;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tempty + 2);
  float* s_scale = reinterpret_cast<float*>(tmem_ptr + 2);
  float* s_shift = s_scale + 128;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int i = 0; i < S; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull[i], 1);
      mbar_init(&tempty[i], 4);
    }
    fence_barrier_init();
    prefetch_tmap(&tm_xh);
    prefetch_tmap(&tm_wh);
    if (TERMS == 3) {
      prefetch_tmap(&tm_xl);
      prefetch_tmap(&tm_wl);
    }
  }
  for (int i = threadIdx.x; i < 128; i += blockDim.x) {
    s_scale[i] = i < p.cout ? p.scale[i] : 0.f;
    s_shift[i] = i < p.cout ? p.shift[i] : 0.f;
  }
  if (warp == 1) tmem_alloc(tmem_ptr, C::kTmemCols);
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = *tmem_ptr;
  const int num_kb = p.ntaps * p.nchunks;
  constexpr uint32_t kBytes = (TERMS == 3 ? 2u : 1u) * (128u * KC * 2u + (PS ? 32u * 32u * 2u : (uint32_t)NPAD * KC * 2u));

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer (converged warp, one lane issues)
    {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
        const int tw = tile % p.tiles_w, t2 = tile / p.tiles_w;
        const int th = t2 % p.tiles_h, n = t2 / p.tiles_h;
        const int x0 = tw * BW * p.in_step, y0 = th * BH * p.in_step;
        for (int kb0 = 0; kb0 < num_kb; kb0 += TPS) {
          const int nsub = min(TPS, num_kb - kb0);
          mbar_wait(&empty[stage], phase ^ 1u);
          if (elect_one()) {
            mbar_expect_tx(&full[stage], kBytes * (uint32_t)nsub);
            for (int t = 0; t < nsub; ++t) {
              const int kb = kb0 + t;
              const int tap = kb / p.nchunks, cc = kb - tap * p.nchunks;
              uint8_t* st = tiles + stage * STAGE + t * C::kSub;
              const int ax = x0 + p.dx[tap], ay = y0 + p.dy[tap], wrow = p.wi[tap] * (PS ? 32 : NPAD);
              const int n_in = p.dout ? (n / p.dout) * p.din + (n % p.dout) + p.dz[tap] : n;
              tma_load_4d(st, &tm_xh, &full[stage], cc * KC, ax, ay, n_in);
              tma_load_2d(st + OFF_B, &tm_wh, &full[stage], PS ? 0 : cc * KC, wrow);
              if (TERMS == 3) {
                tma_load_4d(st + OFF_ALO, &tm_xl, &full[stage], cc * KC, ax, ay, n_in);
                tma_load_2d(st + OFF_BLO, &tm_wl, &full[stage], PS ? 0 : cc * KC, wrow);
              }
            }
          }
          __syncwarp();
          if (++stage == S) {
            stage = 0;
            phase ^= 1u;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer
    // The whole warp stays converged through the barrier waits; one elected lane issues (so the
    // compiler emits plain UTCHMMA instead of a per-instruction uniformisation loop).
    {
      constexpr uint32_t idesc = make_idesc_f16(128, NPAD, 0);
      int stage = 0, it = 0;
      uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++it) {
        const int acc = it & 1;
        mbar_wait(&tempty[acc], ((uint32_t)(it >> 1) & 1u) ^ 1u);
        fence_after_sync();
        const uint32_t d_tmem = tmem_base + (uint32_t)acc * C::kAccCols;
        const uint32_t d_lo = d_tmem + NSPLIT * NPAD;  // TERMS == 3 only
        for (int kb0 = 0; kb0 < num_kb; kb0 += TPS) {
          const int nsub = min(TPS, num_kb - kb0);
          mbar_wait(&full[stage], phase);
          fence_after_sync();
          if (elect_one()) {
            const uint32_t sa0 = smem_u32(tiles + stage * STAGE);
#pragma unroll
            for (int t = 0; t < TPS; ++t) {
              if (t >= nsub) break;
              const uint32_t sa = sa0 + t * C::kSub;
              const uint64_t a_hi = make_smem_desc(sa, 16, C::kSbo, C::kLayout);
              const uint64_t a_lo = make_smem_desc(sa + OFF_ALO, 16, C::kSbo, C::kLayout);
              if constexpr (PS) {
                // each pixel of the pair (K elements 0..31 / 32..63 of the 128-byte row) times the same 32x32
                // slab (64-byte-swizzled) into its own 32 accumulator columns
                constexpr uint32_t idesc32 = make_idesc_f16(128, 32, 0);
                const uint64_t b_hi = make_smem_desc(sa + OFF_B, 16, 512, LAYOUT_SW64);
                const uint64_t b_lo = make_smem_desc(sa + OFF_BLO, 16, 512, LAYOUT_SW64);
#pragma unroll
                for (int hf = 0; hf < 2; ++hf)
#pragma unroll
                  for (int k = 0; k < 2; ++k) {
                    const uint32_t dt = d_tmem + hf * 32;
                    const uint32_t first = (kb0 | t | k) ? 1u : 0u;
                    umma_f16(dt, a_hi + 4 * hf + 2 * k, b_hi + 2 * k, idesc32, first);
                    if (TERMS == 3) {
                      umma_f16(dt + NPAD, a_hi + 4 * hf + 2 * k, b_lo + 2 * k, idesc32, first);
                      umma_f16(dt + NPAD, a_lo + 4 * hf + 2 * k, b_hi + 2 * k, idesc32, 1u);
                    }
                  }
                continue;
              }
              const uint64_t b_hi = make_smem_desc(sa + OFF_B, 16, C::kSbo, C::kLayout);
              const uint64_t b_lo = make_smem_desc(sa + OFF_BLO, 16, C::kSbo, C::kLayout);
#pragma unroll
              for (int k = 0; k < KC / 16; ++k) {  // +32 B per K=16 step inside the swizzled row
                const uint32_t first = (kb0 | t | k) ? 1u : 0u;
                if (NSPLIT > 1) {  // k-block kb0 (one per stage here) goes to accumulator kb0 % NSPLIT
                  umma_f16(d_tmem + (uint32_t)((kb0 % NSPLIT) * NPAD), a_hi + 2 * k, b_hi + 2 * k, idesc,
                           (kb0 >= NSPLIT || k) ? 1u : 0u);
                } else {
                  umma_f16(d_tmem, a_hi + 2 * k, b_hi + 2 * k, idesc, first);
                }
                if (TERMS == 3) {
                  umma_f16(d_lo, a_hi + 2 * k, b_lo + 2 * k, idesc, first);
                  umma_f16(d_lo, a_lo + 2 * k, b_hi + 2 * k, idesc, 1u);
                }
              }
            }
            umma_commit(&empty[stage]);
          }
          __syncwarp();
          if (++stage == S) {
            stage = 0;
            phase ^= 1u;
          }
        }
        if (elect_one()) umma_commit(&tfull[acc]);
        __syncwarp();
      }
    }
  } else {
    // ------------------------------------------------------------ epilogue warps 2..5
    const int q = warp & 3;  // TMEM lane quarter this warp may access
    const int row = q * 32 + lane;
    const int hl = row >> 4, wl = row & 15;
    int it = 0;
    for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++it) {
      const int acc = it & 1;
      const int tw = tile % p.tiles_w, t2 = tile / p.tiles_w;
      const int th = t2 % p.tiles_h, n = t2 / p.tiles_h;
      const int gy = th * BH + hl, gx = tw * BW + wl;
      const int oy = gy * p.os + p.py, ox = gx * p.os + p.px;
      const bool valid = gy < p.GH && gx < p.GW && oy < p.OH && ox < p.OW;
      const size_t pix = ((size_t)n * p.OH + oy) * p.OW + ox;
      mbar_wait(&tfull[acc], (uint32_t)(it >> 1) & 1u);
      fence_after_sync();
#pragma unroll 1
      for (int chunk = 0; chunk < NPAD / 16; ++chunk) {
        const int c0 = chunk * 16;
        if (c0 >= p.cout) break;  // warp-uniform
        uint32_t v[16], vlo[16];
        tmem_ld_32x16(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * C::kAccCols + c0), v);
        if (TERMS == 3)
          tmem_ld_32x16(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * C::kAccCols + NSPLIT * NPAD + c0), vlo);
        tmem_ld_wait();
        if (NSPLIT > 1) {  // sum the partial hi*hi accumulators (fp32, round to nearest)
#pragma unroll 1
          for (int sp = 1; sp < NSPLIT; ++sp) {
            uint32_t vs[16];
            tmem_ld_32x16(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * C::kAccCols + sp * NPAD + c0), vs);
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 16; ++j) v[j] = __float_as_uint(__fadd_rn(__uint_as_float(v[j]), __uint_as_float(vs[j])));
          }
        }
        if (valid) {
          float f[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            float a = __uint_as_float(v[j]);
            if (TERMS == 3) a = __fadd_rn(a, __uint_as_float(vlo[j]));  // large + small product terms, round to nearest
            float t = __fadd_rn(__fmul_rn(a, s_scale[c0 + j]), s_shift[c0 + j]);
            if (p.act == DSIN_ACT_RELU) t = fmaxf(t, 0.f);
            else if (p.act == DSIN_ACT_LRELU02) t = fmaxf(__fmul_rn(t, 0.2f), t);
            f[j] = t;
          }
          const size_t off = pix * p.cout + c0;
          if (p.r1f) {
            const size_t rpix = (((size_t)(n / p.dout) * p.r1_d + (n % p.dout) + p.r1_dz) * p.r1_oh + oy + p.r1_dy) *
                                    p.r1_ow + ox + p.r1_dx;
#pragma unroll
            for (int j = 0; j < 16; ++j)
              if (c0 + j < p.r1_c) f[j] = __fadd_rn(f[j], __ldg(p.r1f + rpix * p.r1_c + c0 + j));
          }
          if (p.r1h) add_residual16(f, p.r1h, p.r1l, off);
          if (p.r2h) add_residual16(f, p.r2h, p.r2l, off);
          if (p.post == DSIN_POST_DENORM_CLIP_D2S) {
            // 12 phase-channels -> 2x2 output pixels x 3 colours of a (2*OH, 2*OW, 3) image
#pragma unroll
            for (int j = 0; j < 12; ++j) {
              const int co = j % 3, ph = j / 3;
              float t = __fadd_rn(__fmul_rn(f[j], dsin_std(co)), dsin_mean(co));
              t = fminf(fmaxf(t, 0.f), 255.f);
              const size_t o2 = (((size_t)n * 2 * p.OH + 2 * oy + (ph >> 1)) * 2 * p.OW + 2 * ox + (ph & 1)) * 3 + co;
              p.yf[o2] = t;
            }
          } else {
          if (p.post != DSIN_POST_NONE) {
#pragma unroll
            for (int j = 0; j < 3; ++j) {
              float t = __fadd_rn(__fmul_rn(f[j], dsin_std(j)), dsin_mean(j));
              f[j] = p.post == DSIN_POST_DENORM_CLIP ? fminf(fmaxf(t, 0.f), 255.f) : t;
            }
          }
          if (p.yf) {
#pragma unroll
            for (int j = 0; j < 16; ++j)
              if (c0 + j < p.cout) p.yf[off + j] = f[j];
          } else {
#pragma unroll
            for (int g = 0; g < 2; ++g) {
              uint4 uh, ul;
              __half2* hh = reinterpret_cast<__half2*>(&uh);
              __half2* ll = reinterpret_cast<__half2*>(&ul);
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                float x0 = f[g * 8 + 2 * e], x1 = f[g * 8 + 2 * e + 1];
                __half h0 = __float2half_rn(x0), h1 = __float2half_rn(x1);
                hh[e] = __halves2half2(h0, h1);
                ll[e] = __halves2half2(__float2half_rn(x0 - __half2float(h0)),
                                       __float2half_rn(x1 - __half2float(h1)));
              }
              reinterpret_cast<uint4*>(p.yh + off)[g] = uh;
              if (p.yl) reinterpret_cast<uint4*>(p.yl + off)[g] = ul;
            }
          }
          }  // !D2S
        }
      }
      fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty[acc]);
    }
  }

  __syncthreads();
  if (warp == 1) {
    fence_after_sync();
    tmem_dealloc(tmem_base, C::kTmemCols);
  }
}

// weights [taps][cin][cout] fp32 -> [tap][npad][cin] split fp16 with a per-cout power-of-two scale that
// moves the row's largest |w| into [8,16) so that the lo part stays in fp16's normal range.
__global__ void pack_w_tc_kernel(const float* __restrict__ w, __half* __restrict__ w_hi, __half* __restrict__ w_lo,
                                 float* __restrict__ wscale, int taps, int cin, int cout, int npad) {
  const int co = blockIdx.x;  // 0..npad-1
  __shared__ float s_max[128];
  float m = 0.f;
  if (co < cout)
    for (int i = threadIdx.x; i < taps * cin; i += blockDim.x) m = fmaxf(m, fabsf(w[(size_t)i * cout + co]));
  s_max[threadIdx.x] = m;
  __syncthreads();
  for (int s = 64; s > 0; s >>= 1) {
    if ((int)threadIdx.x < s) s_max[threadIdx.x] = fmaxf(s_max[threadIdx.x], s_max[threadIdx.x + s]);
    __syncthreads();
  }
  m = s_max[0];
  int ex = 0;
  float sc = 1.f;
  if (m > 0.f) {
    frexpf(m, &ex);            // m = f * 2^ex, f in [0.5,1)
    sc = ldexpf(1.f, 4 - ex);  // m*sc in [8,16)
  }
  if (threadIdx.x == 0 && co < cout) wscale[co] = sc;
  for (int i = threadIdx.x; i < taps * cin; i += blockDim.x) {
    int tap = i / cin, ci = i - tap * cin;
    float v = co < cout ? w[(size_t)i * cout + co] * sc : 0.f;
    __half hi = __float2half_rn(v);
    size_t o = ((size_t)tap * npad + co) * cin + ci;
    w_hi[o] = hi;
    w_lo[o] = __float2half_rn(v - __half2float(hi));
  }
}

template <int KC, int NPAD, int TERMS, bool PS = false, int NSPLIT = 1>
int launch_one(dsin_handle_t h, const CUtensorMap& xh, const CUtensorMap& xl, const CUtensorMap& wh,
               const CUtensorMap& wl, const GP& p, cudaStream_t st) {
  using C = Cfg<KC, NPAD, TERMS, PS, NSPLIT>;
  static bool configured[DSIN_MAX_DEVICES] = {};  // cudaFuncSetAttribute is per device
  if (!configured[h->device]) {
    if (cudaFuncSetAttribute(conv_tc_kernel<KC, NPAD, TERMS, PS, NSPLIT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             C::kSmem) != cudaSuccess)
      return dsin_fail(h, DSIN_ERR_CUDA, "%s: cannot raise dynamic shared memory", __func__);
    configured[h->device] = true;
  }
  int grid = p.total_tiles < h->sm_count ? p.total_tiles : h->sm_count;
  conv_tc_kernel<KC, NPAD, TERMS, PS, NSPLIT><<<grid, 192, C::kSmem, st>>>(xh, xl, wh, wl, p);
  DSIN_LAUNCHED(h);
  return DSIN_OK;
}

template <int KC, int NPAD>
int launch_terms(dsin_handle_t h, int terms, const CUtensorMap& xh, const CUtensorMap& xl, const CUtensorMap& wh,
                 const CUtensorMap& wl, const GP& p, cudaStream_t st) {
  return terms == 3 ? launch_one<KC, NPAD, 3>(h, xh, xl, wh, wl, p, st)
                    : launch_one<KC, NPAD, 1>(h, xh, xl, wh, wl, p, st);
}

int npad_of(int cout) { return (cout + 15) / 16 * 16; }
int kc_of(int cin) { return cin % 64 == 0 ? 64 : 32; }

}  // namespace

// Internal entry used by the probability model: VALID 3-D conv over a channels-last volume
// (vols, D, H, W, 32 ch split fp16) with an explicit tap list; see conv_tc.cuh.
int conv_tc_valid3d(dsin_handle_t h, const ConvTc3dArgs& a, cudaStream_t st) {
  if (a.cin != 32 || a.ntaps < 1 || a.ntaps > MAX_TAPS)
    return dsin_fail(h, DSIN_ERR_UNSUPPORTED, "%s: 3-D tensor-core conv needs cin == 32", __func__);
  const int NPAD = npad_of(a.cout);
  const int Do = a.D - a.kd + 1, Ho = a.H - a.kh + 1, Wo = a.W - a.kw + 1;
  if (a.kd == 2 && a.kh == 3 && a.kw == 3 && a.ntaps <= 18 && NPAD <= 32) {
    // halo-tile kernel: one TMA box per tile instead of one per tap, resident filter (conv_h32.cu)
    ConvH32Args q;
    memset(&q, 0, sizeof(q));
    q.scale = a.scale; q.shift = a.shift;
    q.yh = (__half*)a.y_hi; q.yl = (__half*)a.y_lo; q.yf = a.y_f32;
    q.r1f = a.r1f; q.r1_d = a.r1_d; q.r1_oh = a.r1_oh; q.r1_ow = a.r1_ow;
    q.r1_dz = a.r1_dz; q.r1_dy = a.r1_dy; q.r1_dx = a.r1_dx; q.r1_c = a.r1_c ? a.r1_c : a.cout;
    q.n_out = a.vols * Do; q.dout = Do; q.din = a.D;
    q.OH = Ho; q.OW = Wo; q.cout = a.cout; q.act = a.act; q.terms = a.terms;
    q.ntaps = a.ntaps;
    for (int t = 0; t < a.ntaps; ++t) {
      q.tz[t] = a.tap_d[t]; q.ty[t] = a.tap_h[t]; q.tx[t] = a.tap_w[t]; q.tw[t] = a.tap_wi[t];
    }
    q.hw = 8 + a.kw - 1; q.hh = 16 + a.kh - 1; q.hd = a.kd;
    q.ox = 0; q.oy = 0;
    const int rc = conv_h32_launch(h, (const __half*)a.x_hi, (const __half*)a.x_lo, (const __half*)a.w_hi,
                                   (const __half*)a.w_lo, a.W, a.H, a.vols * a.D, a.wtaps, q, st);
    if (rc != DSIN_ERR_UNSUPPORTED) return rc;
  }
  CUtensorMap xh, xl, wh, wl;
  const uint64_t xd[4] = {32, (uint64_t)a.W, (uint64_t)a.H, (uint64_t)a.vols * a.D};
  const uint64_t xs[3] = {64, (uint64_t)a.W * 64, (uint64_t)a.H * a.W * 64};
  const uint32_t xb[4] = {32, BW, BH, 1};
  const uint64_t wd[2] = {32, (uint64_t)a.wtaps * NPAD};
  const uint64_t wsb[1] = {64};
  const uint32_t wb[2] = {32, (uint32_t)NPAD};
  const CUtensorMapSwizzle sw = CU_TENSOR_MAP_SWIZZLE_64B;
  bool ok = encode_tmap(&xh, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, a.x_hi, xd, xs, xb, sw) &&
            encode_tmap(&xl, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, a.x_lo ? a.x_lo : a.x_hi, xd, xs, xb, sw) &&
            encode_tmap(&wh, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, a.w_hi, wd, wsb, wb, sw) &&
            encode_tmap(&wl, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, a.w_lo ? a.w_lo : a.w_hi, wd, wsb, wb, sw);
  if (!ok) return dsin_fail(h, DSIN_ERR_CUDA, "%s: cuTensorMapEncodeTiled failed", __func__);
  GP p;
  memset(&p, 0, sizeof(p));
  p.scale = a.scale; p.shift = a.shift;
  p.yh = (__half*)a.y_hi; p.yl = (__half*)a.y_lo; p.yf = a.y_f32;
  p.n = a.vols * Do; p.cout = a.cout; p.act = a.act; p.post = DSIN_POST_NONE;
  p.nchunks = 1; p.in_step = 1;
  p.OH = Ho; p.OW = Wo; p.GH = Ho; p.GW = Wo; p.os = 1;
  p.dout = Do; p.din = a.D;
  p.ntaps = a.ntaps;
  for (int t = 0; t < a.ntaps; ++t) {
    p.dz[t] = a.tap_d[t]; p.dy[t] = a.tap_h[t]; p.dx[t] = a.tap_w[t]; p.wi[t] = a.tap_wi[t];
  }
  p.r1f = a.r1f; p.r1_d = a.r1_d; p.r1_oh = a.r1_oh; p.r1_ow = a.r1_ow;
  p.r1_dz = a.r1_dz; p.r1_dy = a.r1_dy; p.r1_dx = a.r1_dx; p.r1_c = a.r1_c ? a.r1_c : a.cout;
  p.tiles_w = (p.GW + BW - 1) / BW; p.tiles_h = (p.GH + BH - 1) / BH;
  p.total_tiles = p.n * p.tiles_w * p.tiles_h;
  if (NPAD == 32) return launch_terms<32, 32>(h, a.terms, xh, xl, wh, wl, p, st);
  if (NPAD == 16) return launch_terms<32, 16>(h, a.terms, xh, xl, wh, wl, p, st);
  return dsin_fail(h, DSIN_ERR_UNSUPPORTED, "%s: unsupported cout", __func__);
}

extern "C" int dsin_conv_tc_npad(int cout) { return npad_of(cout); }

extern "C" int dsin_pack_conv_w_tc(dsin_handle_t h, const float* w_kkio, int taps, int cin, int cout,
                                   uint16_t* w_hi, uint16_t* w_lo, float* wscale, void* stream) {
  DSIN_REQUIRE(h, w_kkio && w_hi && w_lo && wscale, "null pointer");
  DSIN_REQUIRE(h, taps >= 1 && taps <= MAX_TAPS && cin % 32 == 0 && cin <= 128 && cout >= 1 && cout <= 128,
               "unsupported shape");
  const int npad = npad_of(cout);
  pack_w_tc_kernel<<<npad, 128, 0, (cudaStream_t)stream>>>(w_kkio, (__half*)w_hi, (__half*)w_lo, wscale, taps, cin,
                                                          cout, npad);
  DSIN_LAUNCHED(h);
  return DSIN_OK;
}

extern "C" int dsin_pack_conv3x3_w(dsin_handle_t h, const float* w_hwio, uint16_t* w_hi, uint16_t* w_lo,
                                   float* wscale, int cin, int cout, void* stream) {
  DSIN_REQUIRE(h, cin == 128 && cout == 128, "only 128 -> 128 channels");
  return dsin_pack_conv_w_tc(h, w_hwio, 9, cin, cout, w_hi, w_lo, wscale, stream);
}

extern "C" int dsin_conv2d_tc(dsin_handle_t h, const dsin_conv_desc_t* d, int terms, const uint16_t* x_hi,
                              const uint16_t* x_lo, const uint16_t* w_hi, const uint16_t* w_lo,
                              const float* scale, const float* shift, const uint16_t* res1_hi,
                              const uint16_t* res1_lo, const uint16_t* res2_hi, const uint16_t* res2_lo,
                              uint16_t* y_hi, uint16_t* y_lo, float* y_f32, void* stream) {
  DSIN_REQUIRE(h, d && x_hi && w_hi && scale && shift && (y_hi || y_f32), "null pointer");
  DSIN_REQUIRE(h, terms == 1 || terms == 3, "terms must be 1 or 3");
  DSIN_REQUIRE(h, terms == 1 || (x_lo && w_lo), "terms == 3 needs the lo planes");
  DSIN_REQUIRE(h, d->cin % 32 == 0 && d->cin <= 128 && d->cout >= 1 && d->cout <= 128, "unsupported channels");
  DSIN_REQUIRE(h, d->kh == d->kw && d->kh * d->kw <= MAX_TAPS, "unsupported kernel size");
  DSIN_REQUIRE(h, d->stride == 1 || d->stride == 2, "stride must be 1 or 2");
  DSIN_REQUIRE(h, !d->transposed || d->stride == 2, "transposed conv is stride 2");
  DSIN_REQUIRE(h, y_f32 || d->cout % 16 == 0, "split-fp16 output needs cout % 16 == 0");
  DSIN_REQUIRE(h, d->post == DSIN_POST_NONE || d->cout == 3 ||
                      (d->post == DSIN_POST_DENORM_CLIP_D2S && d->cout == 12 && y_f32 && !d->transposed && d->stride == 1),
               "denormalisation needs cout == 3 (or 12 phase-channels with depth-to-space)");
  const int k = d->kh, KC = kc_of(d->cin), NPAD = npad_of(d->cout);
  const int step = (!d->transposed && d->stride == 2) ? 2 : 1;
  DSIN_REQUIRE(h, d->h >= BH * step && d->w >= BW * step, "image smaller than one tile");

  CUtensorMap xh, xl, wh, wl;
  const uint64_t xd[4] = {(uint64_t)d->cin, (uint64_t)d->w, (uint64_t)d->h, (uint64_t)d->n};
  const uint64_t xs[3] = {(uint64_t)d->cin * 2, (uint64_t)d->w * d->cin * 2, (uint64_t)d->h * d->w * d->cin * 2};
  const uint32_t xb[4] = {(uint32_t)KC, (uint32_t)(BW * step), (uint32_t)(BH * step), 1};
  const uint32_t xe[4] = {1, (uint32_t)step, (uint32_t)step, 1};
  const bool pair_shared = (d->flags & DSIN_CONV_PAIR_SHARED) != 0;
  DSIN_REQUIRE(h, !pair_shared || (d->cin == 64 && d->cout == 64 && !d->transposed && d->stride == 1 && !y_f32),
               "pair-shared mode needs cin = cout = 64, stride 1, split output");
  const uint64_t wd[2] = {(uint64_t)(pair_shared ? 32 : d->cin), (uint64_t)k * k * (pair_shared ? 32 : NPAD)};
  const uint64_t wsb[1] = {(uint64_t)(pair_shared ? 32 : d->cin) * 2};
  const uint32_t wb[2] = {(uint32_t)(pair_shared ? 32 : KC), (uint32_t)(pair_shared ? 32 : NPAD)};
  const CUtensorMapSwizzle sw = KC == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
  const CUtensorMapSwizzle swb = pair_shared ? CU_TENSOR_MAP_SWIZZLE_64B : sw;
  bool ok = encode_tmap(&xh, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, x_hi, xd, xs, xb, sw, xe) &&
            encode_tmap(&xl, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, x_lo ? x_lo : x_hi, xd, xs, xb, sw, xe) &&
            encode_tmap(&wh, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, w_hi, wd, wsb, wb, swb) &&
            encode_tmap(&wl, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, w_lo ? w_lo : w_hi, wd, wsb, wb, swb);
  if (!ok) return dsin_fail(h, DSIN_ERR_CUDA, "%s: cuTensorMapEncodeTiled failed", __func__);

  GP p;
  memset(&p, 0, sizeof(p));
  p.scale = scale; p.shift = shift;
  p.r1h = (const __half*)res1_hi; p.r1l = (const __half*)res1_lo;
  p.r2h = (const __half*)res2_hi; p.r2l = (const __half*)res2_lo;
  p.yh = (__half*)y_hi; p.yl = (__half*)y_lo; p.yf = y_f32;
  p.n = d->n; p.cout = d->cout; p.act = d->act; p.post = d->post;
  p.nchunks = d->cin / KC;
  p.in_step = step;
  cudaStream_t st = (cudaStream_t)stream;

  auto launch = [&](const GP& gp) -> int {
    if (pair_shared)
      return terms == 3 ? launch_one<64, 64, 3, true>(h, xh, xl, wh, wl, gp, st)
                        : launch_one<64, 64, 1, true>(h, xh, xl, wh, wl, gp, st);
    if (KC == 64 && NPAD == 128) return launch_terms<64, 128>(h, terms, xh, xl, wh, wl, gp, st);
    if (KC == 64 && NPAD == 64) return launch_terms<64, 64>(h, terms, xh, xl, wh, wl, gp, st);
    if (KC == 64 && NPAD == 48 && terms == 3 && gp.ntaps * gp.nchunks >= 4)  // to_bn: 4 partial hi*hi accumulators
      return launch_one<64, 48, 3, false, 4>(h, xh, xl, wh, wl, gp, st);
    if (KC == 64 && NPAD == 48) return launch_terms<64, 48>(h, terms, xh, xl, wh, wl, gp, st);
    if (KC == 64 && NPAD == 16) return launch_terms<64, 16>(h, terms, xh, xl, wh, wl, gp, st);
    if (KC == 32 && NPAD == 128) return launch_terms<32, 128>(h, terms, xh, xl, wh, wl, gp, st);
    if (KC == 32 && NPAD == 64) return launch_terms<32, 64>(h, terms, xh, xl, wh, wl, gp, st);
    if (KC == 32 && NPAD == 32) return launch_terms<32, 32>(h, terms, xh, xl, wh, wl, gp, st);
    if (KC == 32 && NPAD == 16) return launch_terms<32, 16>(h, terms, xh, xl, wh, wl, gp, st);
    return dsin_fail(h, DSIN_ERR_UNSUPPORTED, "%s: no tensor-core instantiation for this (cin, cout)", __func__);
  };

  if (!d->transposed) {
    p.OH = (d->h + d->stride - 1) / d->stride; p.OW = (d->w + d->stride - 1) / d->stride;
    p.GH = p.OH; p.GW = p.OW; p.os = 1; p.py = 0; p.px = 0;
    const int dil_x = d->dilation_x > 0 ? d->dilation_x : d->dilation;
    const int pt = dsin_same_pad_before(d->h, k, d->stride, d->dilation);
    const int pl = dsin_same_pad_before(d->w, k, d->stride, dil_x);
    p.ntaps = k * k;
    for (int ky = 0; ky < k; ++ky)
      for (int kx = 0; kx < k; ++kx) {
        p.dy[ky * k + kx] = (short)(ky * d->dilation - pt);
        p.dx[ky * k + kx] = (short)(kx * dil_x - pl);
        p.wi[ky * k + kx] = (short)(ky * k + kx);
      }
    p.tiles_w = (p.GW + BW - 1) / BW; p.tiles_h = (p.GH + BH - 1) / BH;
    p.total_tiles = d->n * p.tiles_w * p.tiles_h;
    if (!(d->flags & (DSIN_CONV_NO_HALO | DSIN_CONV_PAIR_SHARED)) && k == 3 && d->stride == 1 && d->cin == 32 &&
        d->cout == 32 && d->dilation >= 1 && dil_x == d->dilation && y_hi && !y_f32 && !res1_hi && !res2_hi &&
        d->post == DSIN_POST_NONE && (terms == 1 || y_lo)) {
      // 32-channel layer (the SI-Net's 3x3 layers, every dilation): row-band kernel (conv_dil.cu).  At dilation 1, 2, 4
      // it also beats the halo-tile kernel (conv_h32.cu, which keeps the probability model's layers), see DESIGN 5.2
      ConvDilArgs q;
      memset(&q, 0, sizeof(q));
      q.scale = scale; q.shift = shift;
      q.yh = (__half*)y_hi; q.yl = (__half*)y_lo;
      q.n = d->n; q.H = d->h; q.W = d->w; q.dil = d->dilation; q.act = d->act; q.terms = terms;
      q.ksteps = (d->flags & DSIN_CONV_CIN16) ? 1 : 2;
      const int rc = conv_dil_launch(h, (const __half*)x_hi, (const __half*)x_lo, (const __half*)w_hi,
                                     (const __half*)w_lo, q, st);
      if (rc != DSIN_ERR_UNSUPPORTED) return rc;
    }
    const bool use_pairs = (d->flags & DSIN_CONV_NO_CTA_PAIR) == 0;
    if (use_pairs && terms == 1 && !(d->flags & DSIN_CONV_NO_WEIGHT_STATIONARY) && k == 3 && d->stride == 1 &&
        d->dilation == 1 && dil_x == 1 && d->cin == 128 && d->cout == 128 && y_hi && !y_lo && !y_f32 && !res1_lo &&
        !res2_lo && d->post == DSIN_POST_NONE && d->act != DSIN_ACT_LRELU02 && p.total_tiles >= 2) {
      // fp16-operand trunk layer: weight-stationary kernel with a halo-resident activation tile (conv_ws.cu)
      ConvWsArgs a;
      memset(&a, 0, sizeof(a));
      a.scale = scale; a.shift = shift;
      a.r1 = p.r1h; a.r2 = p.r2h; a.y = p.yh;
      a.n = d->n; a.OH = p.OH; a.OW = p.OW; a.act = d->act;
      return conv_ws_launch(h, (const __half*)x_hi, (const __half*)w_hi, a, st);
    }
    if (use_pairs && terms == 3 && !(d->flags & DSIN_CONV_NO_HALO) && k == 3 && d->stride == 1 && d->dilation == 1 &&
        dil_x == 1 && d->cin == 128 && d->cout == 128 && y_hi && y_lo && !y_f32 && d->post == DSIN_POST_NONE &&
        d->act != DSIN_ACT_LRELU02 && p.total_tiles >= 2) {
      // fp32-class trunk layer: halo-tile CTA-pair kernel with separate large / small term accumulators (conv_h3.cu)
      ConvH3Args a;
      memset(&a, 0, sizeof(a));
      a.scale = scale; a.shift = shift;
      a.r1h = p.r1h; a.r1l = p.r1l; a.r2h = p.r2h; a.r2l = p.r2l; a.yh = p.yh; a.yl = p.yl;
      a.n = d->n; a.OH = p.OH; a.OW = p.OW; a.act = d->act;
      return conv_h3_launch(h, (const __half*)x_hi, (const __half*)x_lo, (const __half*)w_hi, (const __half*)w_lo, a, st);
    }
    if (use_pairs && KC == 64 && NPAD == 128 && d->cout == 128 && y_hi && !y_f32 && d->post == DSIN_POST_NONE &&
        d->act != DSIN_ACT_LRELU02 && p.total_tiles >= 2) {
      // CTA-pair kernel: each CTA of a pair loads half of the weight slab (64 couts)
      CUtensorMap wh2, wl2;
      const uint32_t wb2[2] = {64, 64};
      if (!encode_tmap(&wh2, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, w_hi, wd, wsb, wb2, sw) ||
          !encode_tmap(&wl2, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, w_lo ? w_lo : w_hi, wd, wsb, wb2, sw))
        return dsin_fail(h, DSIN_ERR_CUDA, "%s: cuTensorMapEncodeTiled failed", __func__);
      ConvTc2Args a;
      memset(&a, 0, sizeof(a));
      a.scale = scale; a.shift = shift;
      a.r1h = p.r1h; a.r1l = p.r1l; a.r2h = p.r2h; a.r2l = p.r2l; a.yh = p.yh; a.yl = p.yl;
      a.n = d->n; a.OH = p.OH; a.OW = p.OW; a.in_step = step; a.act = d->act;
      a.ntaps = p.ntaps; a.nchunks = p.nchunks;
      a.tiles_w = p.tiles_w; a.tiles_h = p.tiles_h; a.total_tiles = p.total_tiles;
      for (int t = 0; t < p.ntaps; ++t) { a.dy[t] = p.dy[t]; a.dx[t] = p.dx[t]; a.wi[t] = p.wi[t]; }
      return conv_tc2_launch(h, terms, xh, xl, wh2, wl2, a, st);
    }
    return launch(p);
  }
  // stride-2 transposed conv, TF SAME: out[o] = sum_{i,k: 2i + k - b = o} in[i] w[k]; phase (py,px) of the
  // output is a stride-1 conv over the input grid with the taps of matching parity.
  p.OH = 2 * d->h; p.OW = 2 * d->w; p.GH = d->h; p.GW = d->w; p.os = 2;
  const int bt = dsin_same_pad_before(p.OH, k, 2, 1), bl = dsin_same_pad_before(p.OW, k, 2, 1);
  p.tiles_w = (p.GW + BW - 1) / BW; p.tiles_h = (p.GH + BH - 1) / BH;
  p.total_tiles = d->n * p.tiles_w * p.tiles_h;
  for (int py = 0; py < 2; ++py)
    for (int px = 0; px < 2; ++px) {
      GP gp = p;
      gp.py = py; gp.px = px; gp.ntaps = 0;
      for (int ky = 0; ky < k; ++ky) {
        if ((py + bt - ky) & 1) continue;
        for (int kx = 0; kx < k; ++kx) {
          if ((px + bl - kx) & 1) continue;
          gp.dy[gp.ntaps] = (short)((py + bt - ky) / 2);
          gp.dx[gp.ntaps] = (short)((px + bl - kx) / 2);
          gp.wi[gp.ntaps] = (short)(ky * k + kx);
          gp.ntaps++;
        }
      }
      int rc = launch(gp);
      if (rc != DSIN_OK) return rc;
    }
  return DSIN_OK;
}

extern "C" int dsin_conv3x3_c128_tc(dsin_handle_t h, int n, int hh, int ww, const uint16_t* x_hi,
                                    const uint16_t* x_lo, const uint16_t* w_hi, const uint16_t* w_lo,
                                    const float* scale, const float* shift, int act, const uint16_t* res1_hi,
                                    const uint16_t* res1_lo, const uint16_t* res2_hi, const uint16_t* res2_lo,
                                    uint16_t* y_hi, uint16_t* y_lo, int terms, void* stream) {
  dsin_conv_desc_t d = {n, hh, ww, 128, 128, 3, 3, 1, 1, 0, act, DSIN_POST_NONE, 0, 0};
  DSIN_REQUIRE(h, y_hi && (terms == 1 || y_lo), "null output");
  return dsin_conv2d_tc(h, &d, terms, x_hi, x_lo, w_hi, w_lo, scale, shift, res1_hi, res1_lo, res2_hi, res2_lo, y_hi,
                        y_lo, nullptr, stream);
}

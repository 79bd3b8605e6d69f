// K6 on tensor cores: SI-Finder all-pairs patch correlation as a tcgen05 implicit GEMM with a fused
// Pearson / Gaussian-prior / running-top-k epilogue, followed by exact rescoring of the candidates.
//   replaces L2_or_pearson_corr + mask multiply + argmax (src/siFinder.py:76-135,20,27-33).
//
// GEMM per image: D[P patches x (h*w) positions] = Q[P x K] * R_windows[(h*w) x K]^T, K = ph*pw*3.
//   M axis = patches (one TMEM lane = one patch  ->  the argmax over positions is a per-thread
//            running reduction over TMEM columns, no cross-thread traffic);
//   N axis = 256 consecutive positions of one correlation row.
// The position operand is Toeplitz (window j+1 = window j shifted by one pixel).  It is fed ZERO-COPY:
// for every correlation row i the 60 values of a window COLUMN (20 rows x 3 channels at pixel x) are
// stored as 8 "layers" of 16-byte pixels, S_l[i][x] = fp16 {v[8l..8l+7]}, v[k] = r(i + k/3, x, k%3)
// (the last layer has 4 zero slots: 60 of 64 K slots carry data).  One TMA box brings a strip of 280
// such pixels into shared memory, and a no-swizzle K-major UMMA descriptor with LBO = 16 B (next K chunk
// = next pixel) and SBO = 128 B (next 8 positions) makes row n of the operand start 16*n bytes into the
// strip -- overlapping windows, no im2col.  One K=16 MMA step consumes two pixels of one layer; a layer
// is 24 px = 12 steps; 8 layers per patch (96 MMAs of 128x256x16 per tile).
// Patches are pre-centred per patch (q - mean_q) before the fp16 rounding, which removes the large
// cancellation in the Pearson numerator; the coarse score error is ~1e-4.  Candidates: per (patch, work unit, column
// half) = "group" (4 correlation rows x every other 128-column block) the epilogue keeps the TOPK = 4 best coarse
// scores.  sif_rescore_kernel rescored every kept position within DELTA of the patch's overall coarse best with the
// reference's exact arithmetic (fp32 data, fp64 dot product, literal fp32 Pearson algebra, exact fp64->fp32 prior)
// and takes the first maximum.  Measured on smooth synthetic and on decoded images (tools/sif_candidates_probe.py): the
// number of positions within DELTA of the best is 1 for most patches and <= 8 per patch, <= 6 per group, on the smoothest
// inputs tried.  If a group's 4th-best is itself within DELTA, positions that were not kept may qualify too: the group
// goes on a work list and sif_exhaustive_kernel rescored ALL its positions exactly, one CTA per listed group (a first
// version did this inside the per-patch warp and a handful of such patches cost milliseconds of tail latency).
// The scoring epilogue used to cost as much as the MMAs (measured by knocking either out: 5.1 ms vs 4.7 ms per 8 pairs,
// 6.6 ms together): an ex2, a warp vote and a branch per position on two warps per scheduler.  Now each 32-position
// chunk first takes a branch-free maximum (positions past the row end, flat windows and lanes without a patch score NaN,
// which fmaxf and every comparison ignore) and enters the ordered top-4 insertion only if some lane beats its group's
// 4th best; the prior's column factor comes from a two-multiplication recurrence.
//
// L2 + LAB (METRIC == SIF_L2, src/siFinder.py:13-17,28-31,102-103).  Same GEMM, same operands: q'' = fp16(q - xm)
// (xm = the patch's scalar mean, as above) against fp16(r).  Since sum_k (q_k - xm) r_k = xy - xm*sum_y for ANY
// constant xm, the coarse distance is  d_c = sx2 - 2 (G + xm*sum_y) + sum_y2,  G the fp32 accumulator, and the epilogue
// keeps the top 4 of the NEGATED masked distance  -d_c * prior  (the argmax of which is tf.argmin's).  LAB values are
// ~1e4 and distances ~1e6..1e10, so the candidate band is not a constant: it is a written bound, scaled by the prior at
// each position.  With u = 2^-11 (fp16), |q''|, |q| = Euclidean norms of the patch (centred / raw), |r| = sqrt(sum_y2) of
// the window:
//   |G - sum q'' r| <= (2u + u^2) sum|q''||r| + 2048 * 2^-23 sum|q''||r|     (operand rounding; fp32 accumulation of
//                                                                          <= 1536 products, truncating adders)
//                  <= 1.22e-3 |q''| |r|                                     (Cauchy-Schwarz)
//   every fp32 rounding of the coarse and of the reference's algebra (sx2, sum_y2, xy, two adds, xm*sum_y) is
//   <= 2^-24 (|q| + |r|)^2, and there are fewer than 16 of them, so with KAPPA = 2.5e-3 >= 2 * 1.22e-3:
//   |d_c - d| <= E = KAPPA |q''| |r| + 2^-20 (|q| + |r|)^2.
// The masked coarse score carries the prior to ~1e-5 relative (ex2.approx and the recurrence; RHO = 1e-4 is used), so
// a kept candidate's exact masked score lies within  e = (1 + 5 RHO) prior * E + 3 RHO |coarse|  of its coarse score.
// sif_rescore_kernel<SIF_L2> takes L = max over the groups' best candidates of (coarse - e), a lower bound of the
// exact best, and rescores every kept candidate with coarse + e >= L.  The epilogue also evaluates, at every position,
// the OPTIMISTIC score u = coarse + 4 RHO |coarse| + prior' * (1 + 7 RHO) E  (prior' its approximate prior, E from that
// window's sum_y2), an upper bound of the exact masked score, and keeps per group the largest u among the positions it
// did NOT keep (never inserted, or evicted from the top 4).  A position can win only if its exact score reaches L, so a
// group goes on the work list only if that largest u is >= L.  (A bound over a whole group instead -- its largest prior
// times its largest E -- sent two thirds of all groups to the exhaustive pass under the prior: a group spans a whole
// row, where the prior varies by up to 1e5.)
// Exactness therefore rests on the bound, never on a measured distribution.
#include "sif_common.cuh"
#include "tc_common.cuh"

using namespace tc;

namespace {

constexpr int TN = 256;                 // positions per tile
constexpr int PAIRS = 8;                // K layers: the 60 values of a window column (20 rows x 3 ch) in 8 x 8 slots
constexpr int PHX = 20;                 // patch height
constexpr int PWX = 24;                 // patch width in pixels
constexpr int KQ = PAIRS * PWX * 8;     // packed K per patch (1536 fp16, 1440 of them data)
constexpr int A_BYTES = 3 * 128 * 128;  // three [128 patches x 64 k] SW128 tiles per pair = 48 KB
constexpr int STRIP_PIX = 280;          // 256 + 24 pixels (even count; 23 needed)
constexpr int B_BYTES = STRIP_PIX * 16; // 4480
constexpr int STAGE_BYTES = A_BYTES + 5120;
constexpr int STAGES = 4;
constexpr int ROWS_PER_UNIT = 4;  // finer work units: static round-robin imbalance < 1 %
constexpr int TOPK = 4;  // candidates kept per group
constexpr float DELTA = 2e-3f;
template <int METRIC> struct SifPos { using T = float2; };            // Pearson: mean_y, rsqrt(den_y)
template <> struct SifPos<SIF_L2> { using T = float4; };              // L2: sum_y, sum_y2, sqrt(sum_y2), -
template <int METRIC>
constexpr int sif_smem_bytes() {
  return STAGES * STAGE_BYTES + 2 * TN * (int)sizeof(typename SifPos<METRIC>::T) + 1024 /*align*/ + 512 /*barriers*/;
}
// L2 band (header comment): coarse-distance bound E = KAPPA |q''| |r| + L2_EPS_T (|q| + |r|)^2, prior error RHO
constexpr double KAPPA = 2.5e-3;
constexpr double L2_EPS_T = 1.0 / 1048576.0;  // 2^-20
constexpr double RHO = 1e-4;

struct SifP {
  const float4* ystat;   // (n,hp,wp): sum_y, mean_y, den_y, sum_y2
  const float4* pinfo;   // (n,P): Pearson: sum of fp16 centred patch, rsqrt(den_x), cy', cx'; L2: 2 xm, sx2, cy', cx'
  float2* cand;          // (n,P,rgroups,2,TOPK): coarse score (descending), position index (as int bits; -1 = empty)
  const float2* pinfo2;  // L2 (n,P): b0, b1 of the per-position error bound (1 + 7 RHO) E = b0 + b1 |r| + B2 sum_y2
  float* unk;            // L2 (n,P,rgroups,2): largest optimistic score among the positions a group did not keep
  int n, hp, wp, P, ptiles, rgroups, jtiles, total_units, use_mask;
  float kh, kw;          // -4/sigma_h^2, -4/sigma_w^2 (exp2 form of exp(-4 ln2 t))
};

__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

constexpr float L2_B2 = (float)((1.0 + 7.0 * RHO) * L2_EPS_T);

// coarse score of one position from its accumulator, the staged per-position statistics and the prior factor g
template <int METRIC, typename PS>
__device__ __forceinline__ float sif_coarse(float acc, PS ps, float4 pi, float g) {
  if constexpr (METRIC == SIF_L2)  // -(sx2 - 2 (acc + xm sum_y) + sum_y2) * g
    return (fmaf(2.f, acc, fmaf(pi.x, ps.x, -ps.y)) - pi.y) * g;
  else
    return (acc - ps.x * pi.x) * ps.y * g;
}

// L2: optimistic score of a position (header comment): coarse s + 4 RHO |s| + g (1 + 7 RHO) E
__device__ __forceinline__ float sif_optimistic(float s, float4 ps, float2 pb, float g) {
  return fmaf(4.f * (float)RHO, fabsf(s), s) + fmaf(pb.y, ps.z, fmaf(L2_B2, ps.y, pb.x)) * g;
}

template <int METRIC>
__global__ void __launch_bounds__(320, 1)
sif_tc_kernel(const __grid_constant__ CUtensorMap tm_q, const __grid_constant__ CUtensorMap tm_s, SifP p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + (((raw + 1023u) & ~1023u) - raw);
  uint8_t* tiles = smem;
  using Pos = typename SifPos<METRIC>::T;
  Pos* s_pos = reinterpret_cast<Pos*>(smem + STAGES * STAGE_BYTES);  // [2][TN]
  uint64_t* full = reinterpret_cast<uint64_t*>(s_pos + 2 * TN);
  uint64_t* empty = full + STAGES;
  uint64_t* tfull = empty + STAGES;
  uint64_t* tempty = tfull + 2;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tempty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull[i], 1);
      mbar_init(&tempty[i], 8);
    }
    fence_barrier_init();
    prefetch_tmap(&tm_q);
    prefetch_tmap(&tm_s);
  }
  if (warp == 1) tmem_alloc(tmem_ptr, 512);
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = *tmem_ptr;
  const int units_per_img = p.ptiles * p.rgroups;

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer (converged warp, one lane issues)
    {
      int stage = 0;
      uint32_t phase = 0;
      for (int u = blockIdx.x; u < p.total_units; u += gridDim.x) {
        const int img = u / units_per_img, r = u % units_per_img;
        const int pt = r / p.rgroups, rg = r % p.rgroups;
        const int i1 = min(p.hp, (rg + 1) * ROWS_PER_UNIT);
        for (int i = rg * ROWS_PER_UNIT; i < i1; ++i)
          for (int jt = 0; jt < p.jtiles; ++jt)
            for (int d = 0; d < PAIRS; ++d) {
              mbar_wait(&empty[stage], phase ^ 1u);
              if (elect_one()) {
                uint8_t* st = tiles + stage * STAGE_BYTES;
                mbar_expect_tx(&full[stage], A_BYTES + B_BYTES);
#pragma unroll
                for (int c = 0; c < 3; ++c)
                  tma_load_3d(st + c * 16384, &tm_q, &full[stage], d * 192 + c * 64, pt * 128, img);
                tma_load_4d(st + A_BYTES, &tm_s, &full[stage], 0, jt * (TN / 2), i, img * PAIRS + d);
              }
              __syncwarp();
              if (++stage == STAGES) {
                stage = 0;
                phase ^= 1u;
              }
            }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer (converged warp, one lane issues)
    {
      constexpr uint32_t idesc_full = make_idesc_f16(128, TN, 0);
      // the last tile of a correlation row holds wp - (jtiles-1)*TN positions: issue only that many columns
      const uint32_t idesc_last = make_idesc_f16(128, ((p.wp - (p.jtiles - 1) * TN) + 15) & ~15, 0);
      int stage = 0, it = 0;
      uint32_t phase = 0;
      for (int u = blockIdx.x; u < p.total_units; u += gridDim.x) {
        const int rg = (u % units_per_img) % p.rgroups;
        const int i1 = min(p.hp, (rg + 1) * ROWS_PER_UNIT);
        for (int i = rg * ROWS_PER_UNIT; i < i1; ++i)
          for (int jt = 0; jt < p.jtiles; ++jt, ++it) {
            const int acc = it & 1;
            mbar_wait(&tempty[acc], ((uint32_t)(it >> 1) & 1u) ^ 1u);
            fence_after_sync();
            const uint32_t d_tmem = tmem_base + (uint32_t)acc * TN;
            const uint32_t idesc = jt == p.jtiles - 1 ? idesc_last : idesc_full;
            for (int d = 0; d < PAIRS; ++d) {
              mbar_wait(&full[stage], phase);
              fence_after_sync();
              if (elect_one()) {
                const uint32_t sa = smem_u32(tiles + stage * STAGE_BYTES);
                const uint32_t sb = sa + A_BYTES;
#pragma unroll
                for (int s = 0; s < 12; ++s) {
                  // A: chunk s/4 (16 KB, SW128), K step s%4 (+32 B).  B: Toeplitz strip, pixels 2s, 2s+1.
                  const uint64_t da = make_smem_desc(sa + (s >> 2) * 16384 + (s & 3) * 32, 16, 1024, LAYOUT_SW128);
                  const uint64_t db = make_smem_desc(sb + s * 32, 16, 128, LAYOUT_NONE);
                  umma_f16(d_tmem, da, db, idesc, (d | s) ? 1u : 0u);
                }
                umma_commit(&empty[stage]);
              }
              __syncwarp();
              if (++stage == STAGES) {
                stage = 0;
                phase ^= 1u;
              }
            }
            if (elect_one()) umma_commit(&tfull[acc]);
            __syncwarp();
          }
      }
    }
  } else {
    // ------------------------------------------------------------ epilogue warps 2..9
    // Two warps per TMEM lane quarter; each scores half of the tile's 256 positions for its 32 patches and keeps the
    // TOPK best of its group in registers (written out per work unit).
    const int q = warp & 3;
    const int half = (warp - 2) >> 2;
    const int et = (warp - 2) * 32 + lane;  // 0..255 among epilogue threads
    const float kstep = p.use_mask ? ex2_approx(2.f * p.kw) : 1.f;
    int it = 0;
    for (int u = blockIdx.x; u < p.total_units; u += gridDim.x) {
      const int img = u / units_per_img, r = u % units_per_img;
      const int pt = r / p.rgroups, rg = r % p.rgroups;
      const int pch = pt * 128 + q * 32 + lane;
      const bool pvalid = pch < p.P;
      float4 pi = make_float4(0.f, 0.f, 0.f, 0.f);
      if (pvalid) pi = p.pinfo[(size_t)img * p.P + pch];
      float bs0 = -INFINITY, bs1 = -INFINITY, bs2 = -INFINITY, bs3 = -INFINITY;  // the group's 4 best, descending
      int bi0 = -1, bi1 = -1, bi2 = -1, bi3 = -1;
      // L2: optimistic scores of the 4 kept and the largest one of the positions not kept
      float ub0 = -INFINITY, ub1 = -INFINITY, ub2 = -INFINITY, ub3 = -INFINITY, unk = -INFINITY;
      float2 pb = make_float2(0.f, 0.f);
      if constexpr (METRIC == SIF_L2) {
        if (pvalid) pb = p.pinfo2[(size_t)img * p.P + pch];
      }
      const int i1 = min(p.hp, (rg + 1) * ROWS_PER_UNIT);
      for (int i = rg * ROWS_PER_UNIT; i < i1; ++i) {
        // Pearson: rsqrt(den_x), L2: 1, times the row factor of the prior; NaN for a lane without a patch: every score
        // of it is NaN, NaN never passes a comparison and fmaxf ignores it
        float rowf = pvalid ? (METRIC == SIF_L2 ? 1.f : pi.y) : __int_as_float(0x7fc00000);
        if (p.use_mask) {
          float dh = (float)i - pi.z;
          rowf *= ex2_approx(p.kh * dh * dh);
        }
        for (int jt = 0; jt < p.jtiles; ++jt, ++it) {
          const int acc = it & 1;
          const int j0 = jt * TN;
          const int nvalid = min(TN, p.wp - j0);
          // stage per-position statistics for this tile (double buffered with the accumulator).  Pearson: mean_y and
          // rsqrt(den_y), NaN for a flat window (den_y <= 0: NaN / inf in the exact arithmetic, never a candidate);
          // L2: sum_y, sum_y2 and its square root.  NaN for a position past the row end.
          Pos* sp = s_pos + acc * TN;
          {
            Pos v;
            v.x = 0.f;
            v.y = __int_as_float(0x7fc00000);
            if (et < nvalid) {
              float4 ys = __ldg(p.ystat + ((size_t)img * p.hp + i) * p.wp + j0 + et);
              if constexpr (METRIC == SIF_L2) {
                v = make_float4(ys.x, ys.w, sqrtf(ys.w), 0.f);
              } else {
                v.x = ys.y;
                v.y = ys.z > 0.f ? rsqrtf(ys.z) : __int_as_float(0x7fc00000);
              }
            }
            sp[et] = v;
          }
          asm volatile("bar.sync 1, 256;" ::: "memory");
          mbar_wait(&tfull[acc], (uint32_t)(it >> 1) & 1u);
          fence_after_sync();
#pragma unroll 1
          for (int chunk = 0; chunk < TN / 64; ++chunk) {
            const int cb = half * (TN / 2) + chunk * 32;
            if (cb >= nvalid) break;  // warp-uniform
            uint32_t v[32];
            tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * TN + cb), v);
            // column factor of the prior by recurrence: g(c) = 2^(kw (c - cx)^2), g(c+1) = g(c) r(c),
            // r(c+1) = r(c) 2^(2 kw) -- two multiplications per position instead of an ex2 (the coarse score only has to
            // be good to ~1e-4; 32 steps of fp32 rounding stay below 1e-5 relative)
            float g0 = rowf, r0 = 1.f;
            if (p.use_mask) {
              const float dw = (float)(j0 + cb) - pi.w;
              g0 = rowf * ex2_approx(p.kw * dw * dw);
              r0 = ex2_approx(p.kw * (2.f * dw + 1.f));
            }
            tmem_ld_wait();
            // pass 1, branch-free: the chunk's best score (L2: and its best optimistic score)
            float m = -INFINITY, um = -INFINITY;
            {
              float g = g0, r = r0;
#pragma unroll
              for (int jj = 0; jj < 32; ++jj) {
                const Pos ps = sp[cb + jj];
                const float s = sif_coarse<METRIC>(__uint_as_float(v[jj]), ps, pi, g);
                m = fmaxf(m, s);
                if constexpr (METRIC == SIF_L2) um = fmaxf(um, sif_optimistic(s, ps, pb, g));
                g *= r;
                r *= kstep;
              }
            }
            // pass 2, rare after warm-up: some lane has a score above its group's 4th best -- insert in order with
            // the same arithmetic (strict >: among equal scores the earlier position stays ahead)
            if (!__any_sync(0xffffffffu, m > bs3)) {
              if constexpr (METRIC == SIF_L2) unk = fmaxf(unk, um);  // no position of the chunk is kept
            } else {
              float g = g0, r = r0;
#pragma unroll
              for (int jj = 0; jj < 32; ++jj) {
                const Pos ps = sp[cb + jj];
                const float s = sif_coarse<METRIC>(__uint_as_float(v[jj]), ps, pi, g);
                if constexpr (METRIC == SIF_L2) {
                  const float u = sif_optimistic(s, ps, pb, g);
                  if (s > bs3) {  // u joins the kept ones, the evicted 4th best's joins the rest
                    unk = fmaxf(unk, ub3);
                    if (s > bs0) {
                      ub3 = ub2; ub2 = ub1; ub1 = ub0; ub0 = u;
                    } else if (s > bs1) {
                      ub3 = ub2; ub2 = ub1; ub1 = u;
                    } else if (s > bs2) {
                      ub3 = ub2; ub2 = u;
                    } else {
                      ub3 = u;
                    }
                  } else {
                    unk = fmaxf(unk, u);
                  }
                }
                g *= r;
                r *= kstep;
                if (s > bs3) {
                  const int idx = i * p.wp + j0 + cb + jj;
                  if (s > bs0) {
                    bs3 = bs2; bi3 = bi2; bs2 = bs1; bi2 = bi1; bs1 = bs0; bi1 = bi0; bs0 = s; bi0 = idx;
                  } else if (s > bs1) {
                    bs3 = bs2; bi3 = bi2; bs2 = bs1; bi2 = bi1; bs1 = s; bi1 = idx;
                  } else if (s > bs2) {
                    bs3 = bs2; bi3 = bi2; bs2 = s; bi2 = idx;
                  } else {
                    bs3 = s; bi3 = idx;
                  }
                }
              }
            }
          }
          fence_before_sync();
          __syncwarp();
          if (lane == 0) mbar_arrive(&tempty[acc]);
        }
      }
      if (pvalid) {
        float2* dst = p.cand + ((((size_t)img * p.P + pch) * p.rgroups + rg) * 2 + half) * TOPK;
        dst[0] = make_float2(bs0, __int_as_float(bi0));
        dst[1] = make_float2(bs1, __int_as_float(bi1));
        dst[2] = make_float2(bs2, __int_as_float(bi2));
        dst[3] = make_float2(bs3, __int_as_float(bi3));
        if constexpr (METRIC == SIF_L2) p.unk[(((size_t)img * p.P + pch) * p.rgroups + rg) * 2 + half] = unk;
      }
    }
  }

  __syncthreads();
  if (warp == 1) {
    fence_after_sync();
    tmem_dealloc(tmem_base, 512);
  }
}

// ---- operand packing -------------------------------------------------------------------------
// one warp per patch: centred fp16 patch in the paired-row 16-byte-pixel layout + per-patch info
template <int METRIC>
__global__ void sif_pack_q_kernel(const float* __restrict__ q, const float* __restrict__ pstat,
                                  __half* __restrict__ q2, float4* __restrict__ pinfo, float2* __restrict__ pinfo2,
                                  int n, int P, int ph, int pw, int hh, int ww) {
  const int64_t wid = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / 32;
  const int lane = threadIdx.x % 32;
  if (wid >= (int64_t)n * P) return;
  const int pch = (int)(wid % P);
  const float* qp = q + wid * (ph * pw * 3);
  const float xm = pstat[wid * 4 + 2];
  float s16 = 0.f;
  double c2 = 0.0, x2 = 0.0;  // L2: squared norms of the centred and of the raw patch
  __half* out = q2 + wid * KQ;
  for (int e = lane; e < PAIRS * pw; e += 32) {  // (layer l, pixel px)
    const int l = e / pw, px = e % pw;
    __half hv[8];
#pragma unroll
    for (int t = 0; t < 8; ++t) {
      const int k = 8 * l + t;  // value index within the window column: k = dy*3 + c
      __half hq = __float2half_rn(0.f);
      if (k < ph * 3) {
        const float qv = qp[((k / 3) * pw + px) * 3 + (k % 3)];
        hq = __float2half_rn(qv - xm);
        s16 += __half2float(hq);
        if constexpr (METRIC == SIF_L2) {
          c2 += (double)(qv - xm) * (double)(qv - xm);
          x2 += (double)qv * (double)qv;
        }
      }
      hv[t] = hq;
    }
    *reinterpret_cast<uint4*>(out + (size_t)e * 8) = *reinterpret_cast<const uint4*>(hv);
  }
  for (int o = 16; o > 0; o >>= 1) s16 += __shfl_xor_sync(0xffffffffu, s16, o);
  if constexpr (METRIC == SIF_L2) {
    for (int o = 16; o > 0; o >>= 1) {
      c2 += __shfl_xor_sync(0xffffffffu, c2, o);
      x2 += __shfl_xor_sync(0xffffffffu, x2, o);
    }
    if (lane == 0) {  // (1 + 7 RHO) (KAPPA |q''| |r| + EPS (|q| + |r|)^2) = b0 + b1 |r| + B2 |r|^2
      const double k = 1.0 + 7.0 * RHO, nqc = sqrt(c2), nq = sqrt(x2);
      pinfo2[wid] = make_float2((float)(k * L2_EPS_T * x2), (float)(k * (KAPPA * nqc + 2.0 * L2_EPS_T * nq)));
    }
  }
  if (lane == 0) {
    const float denx = pstat[wid * 4 + 3];
    const int pcs = ww / pw;
    const float cy = ((float)(pch / pcs) + 0.5f) * ph - (float)(ph / 2 - 1);
    const float cx = ((float)(pch % pcs) + 0.5f) * pw - (float)(pw / 2 - 1);
    if constexpr (METRIC == SIF_L2) pinfo[wid] = make_float4(2.f * xm, pstat[wid * 4 + 1], cy, cx);
    else pinfo[wid] = make_float4(s16, denx > 0.f ? rsqrtf(denx) : 0.f, cy, cx);
  }
}

// S_l[i][x] = fp16 {v[8l..8l+7]}, v[k] = r(i + k/3, x, k%3), for every correlation row i in [0, hp).
// A block stages the (PS_ROWS + ph - 1) x PS_COLS window of r it needs once (every element of r feeds up to ph
// output rows), then writes 16-byte pixels, coalesced along x.
constexpr int PS_ROWS = 16, PS_COLS = 64, PS_MAXPH = 24;
__global__ void __launch_bounds__(256) sif_pack_strip_kernel(const float* __restrict__ r, __half* __restrict__ s, int n,
                                                             int hh, int ww, int ph) {
  __shared__ float tile[(PS_ROWS + PS_MAXPH - 1) * PS_COLS * 3];
  const int hp = hh - ph + 1;
  const int xb = blockIdx.x * PS_COLS, ib = blockIdx.y * PS_ROWS, img = blockIdx.z;
  const int rows = min(PS_ROWS, hp - ib) + ph - 1;         // input rows ib .. ib + rows - 1 (all < hh)
  const int cols = min(PS_COLS, ww - xb);
  const float* src = r + ((int64_t)img * hh + ib) * ww * 3;
  for (int e = threadIdx.x; e < rows * cols * 3; e += blockDim.x) {
    const int row = e / (cols * 3), c = e % (cols * 3);
    tile[row * PS_COLS * 3 + c] = src[(int64_t)row * ww * 3 + xb * 3 + c];
  }
  __syncthreads();
  const int nout = min(PS_ROWS, hp - ib);
  for (int o = threadIdx.x; o < PAIRS * nout * cols; o += blockDim.x) {
    const int x = o % cols, i = (o / cols) % nout, l = o / (cols * nout);
    __half hv[8];
#pragma unroll
    for (int q8 = 0; q8 < 8; ++q8) {
      const int k = 8 * l + q8;
      const float v = k < ph * 3 ? tile[((i + k / 3) * PS_COLS + x) * 3 + (k % 3)] : 0.f;
      hv[q8] = __float2half_rn(v);
    }
    const int64_t idx = (((int64_t)img * PAIRS + l) * hp + ib + i) * ww + xb + x;
    reinterpret_cast<uint4*>(s)[idx] = *reinterpret_cast<const uint4*>(hv);
  }
}

// ---- exact rescoring: one warp per (image, patch) ------------------------------------------------
// exact masked score of one position from its window's dot product: the reference's literal fp32 algebra, exact prior
// (L2: the negated masked distance)
template <int METRIC>
__device__ __forceinline__ unsigned long long sif_exact_key(double dot, const float* __restrict__ ystat,
                                                            const float* __restrict__ ps, int img, int pch, int i,
                                                            int j, int hh, int ww, int ph, int pw, int use_mask) {
  const int wp = ww - pw + 1, hp = hh - ph + 1;
  const float4 ys = reinterpret_cast<const float4*>(ystat)[((int64_t)img * hp + i) * wp + j];
  float s;
  if constexpr (METRIC == SIF_L2) {
    s = sif_l2((float)dot, ps[1], ys.w);
    if (use_mask) s = __fmul_rn(s, sif_mask_exact(pch, i, j, hh, ww, ph, pw));
    s = -s;
  } else {
    s = sif_pearson((float)dot, ys.x, ys.y, ys.z, ps[0], ps[2], ps[3], (float)(ph * pw * 3));
    if (use_mask) s = __fmul_rn(s, sif_mask_exact(pch, i, j, hh, ww, ph, pw));
  }
  return sif_pack(s, (unsigned)(i * wp + j));
}

// L2 band, one kept candidate: the largest possible |coarse - exact| of its masked score (header comment)
__device__ __forceinline__ double sif_l2_slack(float coarse, int idx, const float* __restrict__ ystat, int img, int pch,
                                               int hh, int ww, int ph, int pw, int use_mask, double nqc, double nq) {
  const int wp = ww - pw + 1, hp = hh - ph + 1;
  const int i = idx / wp, j = idx % wp;
  const double nr = sqrt((double)reinterpret_cast<const float4*>(ystat)[((int64_t)img * hp + i) * wp + j].w);
  const double m = use_mask ? (double)sif_mask_exact(pch, i, j, hh, ww, ph, pw) : 1.0;
  const double E = KAPPA * nqc * nr + L2_EPS_T * (nq + nr) * (nq + nr);
  return (1.0 + 5.0 * RHO) * m * E + 3.0 * RHO * fabs((double)coarse);
}

// one warp's fp64 dot product of patch qp with the window of r at (img, i, j), spread over the lanes (all lanes get it)
__device__ __forceinline__ double sif_warp_dot(const float* __restrict__ qp, const float* __restrict__ r, int img,
                                               int i, int j, int hh, int ww, int kdim, int krow, int lane) {
  const float* rp = r + (((int64_t)img * hh + i) * ww + j) * 3;
  double acc = 0.0;
  for (int k = lane; k < kdim; k += 32) {
    const int dy = k / krow, kk = k - dy * krow;
    acc += (double)qp[k] * (double)__ldg(rp + (int64_t)dy * ww * 3 + kk);
  }
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  return acc;
}

template <int METRIC>
__global__ void sif_rescore_kernel(const float2* __restrict__ cand, int ngroups, const float* __restrict__ q,
                                   const float* __restrict__ r, const float* __restrict__ pstat,
                                   const float* __restrict__ ystat, int n, int hh, int ww, int ph, int pw, int use_mask,
                                   const float* __restrict__ unk, unsigned long long* __restrict__ keys,
                                   int2* __restrict__ worklist, int* __restrict__ work_count, int work_cap) {
  const int64_t wid = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / 32;
  const int lane = threadIdx.x % 32;
  const int P = (hh / ph) * (ww / pw);
  if (wid >= (int64_t)n * P) return;
  const int img = (int)(wid / P), pch = (int)(wid % P);
  const int wp = ww - pw + 1;
  const int kdim = ph * pw * 3, krow = pw * 3;
  const float2* cp = cand + wid * (int64_t)ngroups * TOPK;
  const float* qp = q + wid * kdim;
  const float* ps = pstat + wid * 4;
  unsigned long long key = 0ull;
  if constexpr (METRIC == SIF_L2) {
    // the band of the header comment: patch norms (centred as packed, and raw) ...
    double c2 = 0.0, q2 = 0.0;
    const float xm = ps[2];
    for (int k = lane; k < kdim; k += 32) {
      const float v = qp[k];
      const double c = (double)(v - xm);
      c2 += c * c;
      q2 += (double)v * (double)v;
    }
    for (int o = 16; o > 0; o >>= 1) {
      c2 += __shfl_xor_sync(0xffffffffu, c2, o);
      q2 += __shfl_xor_sync(0xffffffffu, q2, o);
    }
    const double nqc = sqrt(c2), nq = sqrt(q2);
    // ... L, a lower bound of the exact best score, from each group's best kept candidate ...
    double lo = -INFINITY;
    for (int g = lane; g < ngroups; g += 32) {
      const float2 cv = cp[(int64_t)g * TOPK];
      const int idx = __float_as_int(cv.y);
      if (idx >= 0) lo = fmax(lo, (double)cv.x - sif_l2_slack(cv.x, idx, ystat, img, pch, hh, ww, ph, pw, use_mask, nqc, nq));
    }
    for (int o = 16; o > 0; o >>= 1) lo = fmax(lo, __shfl_xor_sync(0xffffffffu, lo, o));
    for (int g0 = 0; g0 < ngroups; g0 += 32) {
      const int g = g0 + lane;
      unsigned need = 0u;  // kept candidates of this group that may win
      if (g < ngroups) {
        for (int e = 0; e < TOPK; ++e) {
          const float2 cv = cp[(int64_t)g * TOPK + e];
          const int idx = __float_as_int(cv.y);
          if (idx >= 0 && (double)cv.x + sif_l2_slack(cv.x, idx, ystat, img, pch, hh, ww, ph, pw, use_mask, nqc, nq) >= lo)
            need |= 1u << e;
        }
        // a position that was not kept may win only if its optimistic score reaches L
        if ((double)unk[wid * ngroups + g] >= lo) {
          const int slot = atomicAdd(work_count, 1);
          if (slot < work_cap) worklist[slot] = make_int2((int)wid, g);
        }
      }
      unsigned live = __ballot_sync(0xffffffffu, need != 0u);
      while (live) {
        const int src = __ffs(live) - 1;
        live &= live - 1;
        const int gg = g0 + src;
        const unsigned es = __shfl_sync(0xffffffffu, need, src);
        for (int e = 0; e < TOPK; ++e) {
          if (!(es & (1u << e))) continue;  // warp-uniform
          const int idx = __float_as_int(cp[(int64_t)gg * TOPK + e].y);
          const int i = idx / wp, j = idx % wp;
          const double acc = sif_warp_dot(qp, r, img, i, j, hh, ww, kdim, krow, lane);
          if (lane == 0) {
            const unsigned long long k2 = sif_exact_key<METRIC>(acc, ystat, ps, img, pch, i, j, hh, ww, ph, pw, use_mask);
            key = k2 > key ? k2 : key;
          }
        }
      }
    }
  } else {
    if (!(ps[3] > 0.f)) {  // den_x <= 0 (a flat patch): sqrt(den) is NaN / the quotient infinite at every position; a NaN
      if (lane == 0) keys[wid] = 0ull;  // never wins tf.argmax and all-NaN -> index 0 (sif_common.cuh, DESIGN.md 3.2)
      return;
    }
    float best = -INFINITY;
    for (int g = lane; g < ngroups; g += 32) best = fmaxf(best, cp[(int64_t)g * TOPK].x);  // lists are sorted
    for (int o = 16; o > 0; o >>= 1) best = fmaxf(best, __shfl_xor_sync(0xffffffffu, best, o));
    const float thr = best - DELTA;
    for (int g0 = 0; g0 < ngroups; g0 += 32) {
      const int g = g0 + lane;
      float gbest = -INFINITY, gweak = -INFINITY;
      if (g < ngroups) {
        gbest = cp[(int64_t)g * TOPK].x;
        gweak = cp[(int64_t)g * TOPK + TOPK - 1].x;
      }
      unsigned live = __ballot_sync(0xffffffffu, gbest >= thr);  // groups that hold a position within DELTA of the best
      // ... and whose weakest kept candidate qualifies too: positions that were NOT kept may qualify as well
      if (g < ngroups && gweak >= thr) {
        const int slot = atomicAdd(work_count, 1);
        if (slot < work_cap) worklist[slot] = make_int2((int)wid, g);
      }
      while (live) {
        const int src = __ffs(live) - 1;
        live &= live - 1;
        const int gg = g0 + src;
        for (int e = 0; e < TOPK; ++e) {  // one position at a time, the dot product spread over the lanes (fp64)
          const float2 cv = cp[(int64_t)gg * TOPK + e];
          const int idx = __float_as_int(cv.y);
          if (!(cv.x >= thr) || idx < 0) break;  // sorted: nothing further qualifies (warp-uniform)
          const int i = idx / wp, j = idx % wp;
          const double acc = sif_warp_dot(qp, r, img, i, j, hh, ww, kdim, krow, lane);
          if (lane == 0) {
            const unsigned long long k2 = sif_exact_key<METRIC>(acc, ystat, ps, img, pch, i, j, hh, ww, ph, pw, use_mask);
            key = k2 > key ? k2 : key;
          }
        }
      }
    }
  }
  if (lane == 0) keys[wid] = key;
}

// One CTA per listed (patch, group): every position of the group (4 correlation rows x every other 128-column block),
// one position per thread (coalesced window reads, two fp64 chains), merged into the patch's key with a 64-bit max.
// The list has room for every group of every patch, so nothing is ever dropped.
template <int METRIC>
__global__ void __launch_bounds__(128) sif_exhaustive_kernel(const int2* __restrict__ worklist,
                                                             const int* __restrict__ work_count, int work_cap,
                                                             const float* __restrict__ q, const float* __restrict__ r,
                                                             const float* __restrict__ pstat,
                                                             const float* __restrict__ ystat, int n, int hh, int ww,
                                                             int ph, int pw, int use_mask,
                                                             unsigned long long* __restrict__ keys) {
  const int count = min(*work_count, work_cap);
  __shared__ unsigned long long s_key[4];
  const int P = (hh / ph) * (ww / pw);
  const int wp = ww - pw + 1, hp = hh - ph + 1;
  const int krow = pw * 3;
  for (int item = blockIdx.x; item < count; item += gridDim.x) {
    const int2 w = worklist[item];
    const int wid = w.x, gg = w.y;
    const int img = wid / P, pch = wid % P;
    const float* qp = q + (int64_t)wid * (ph * krow);
    const float* ps = pstat + (int64_t)wid * 4;
    const int rg = gg >> 1, half = gg & 1;
    const int i0 = rg * ROWS_PER_UNIT, i1 = min(hp, i0 + ROWS_PER_UNIT);
    unsigned long long key = 0ull;
    for (int i = i0; i < i1; ++i)
      for (int jb = half * (TN / 2); jb < wp; jb += TN) {  // this half's 128-column blocks: one position per thread
        const int j = jb + (int)threadIdx.x;
        if (j >= wp) continue;
        const float* rp = r + (((int64_t)img * hh + i) * ww + j) * 3;
        double a0 = 0.0, a1 = 0.0;
        for (int dy = 0; dy < ph; ++dy) {
          const float* rr = rp + (int64_t)dy * ww * 3;
          const float* qq = qp + dy * krow;
          for (int kk = 0; kk < krow; kk += 2) {
            a0 += (double)__ldg(qq + kk) * (double)__ldg(rr + kk);
            a1 += (double)__ldg(qq + kk + 1) * (double)__ldg(rr + kk + 1);
          }
        }
        const unsigned long long k2 = sif_exact_key<METRIC>(a0 + a1, ystat, ps, img, pch, i, j, hh, ww, ph, pw, use_mask);
        key = k2 > key ? k2 : key;
      }
    for (int o = 16; o > 0; o >>= 1) {
      const unsigned long long other = __shfl_xor_sync(0xffffffffu, key, o);
      key = other > key ? other : key;
    }
    if ((threadIdx.x & 31) == 0) s_key[threadIdx.x >> 5] = key;
    __syncthreads();
    if (threadIdx.x == 0) {
      unsigned long long k = s_key[0];
      for (int t = 1; t < 4; ++t) k = s_key[t] > k ? s_key[t] : k;
      atomicMax(keys + wid, k);
    }
    __syncthreads();
  }
}

struct Layout {
  int64_t q2, strip, pinfo, pinfo2, cand, unk, work, total;
  int work_cap;
  int ptiles, rgroups, jtiles, ngroups;
};

Layout make_layout(int n, int hh, int ww, int ph, int pw) {
  Layout L;
  const int P = (hh / ph) * (ww / pw), hp = hh - ph + 1, wp = ww - pw + 1;
  L.ptiles = (P + 127) / 128;
  L.rgroups = (hp + ROWS_PER_UNIT - 1) / ROWS_PER_UNIT;
  L.jtiles = (wp + TN - 1) / TN;
  L.ngroups = L.rgroups * 2;  // two epilogue warps (column halves) per patch and work unit
  auto up = [](int64_t v) { return (v + 1023) / 1024 * 1024; };
  L.q2 = 0;
  L.strip = up((int64_t)n * P * KQ * 2);
  L.pinfo = L.strip + up((int64_t)n * PAIRS * (hh - ph + 1) * ww * 16);
  L.pinfo2 = L.pinfo + up((int64_t)n * P * 16);
  L.cand = L.pinfo2 + up((int64_t)n * P * 8);
  L.unk = L.cand + up((int64_t)n * P * L.ngroups * TOPK * 8);
  L.work = L.unk + up((int64_t)n * P * L.ngroups * 4);  // [count (16 B)][work_cap x int2]
  L.work_cap = n * P * L.ngroups;  // every group of every patch fits
  L.total = L.work + up(16 + (int64_t)L.work_cap * 8);
  return L;
}

}  // namespace

int64_t sif_tc_workspace_bytes(int n, int hh, int ww, int ph, int pw, int method) {
  if (method == 0) return 0;
  return make_layout(n, hh, ww, ph, pw).total + 1024;
}

template <int METRIC>
static int sif_tc_match_impl(dsin_handle_t h, const float* q, const float* r, const float* pstat, const float* ystat,
                             int n, int hh, int ww, int ph, int pw, int use_mask, unsigned long long* keys, void* ws,
                             cudaStream_t st) {
  if (ph != PHX || pw != PWX)
    return dsin_fail(h, DSIN_ERR_UNSUPPORTED, "%s: tensor-core SI-Finder is built for 20x24 patches", __func__);
  if (ww % 2 != 0) return dsin_fail(h, DSIN_ERR_UNSUPPORTED, "%s: image width must be even", __func__);
  const int P = (hh / ph) * (ww / pw), hp = hh - ph + 1, wp = ww - pw + 1;
  const Layout L = make_layout(n, hh, ww, ph, pw);
  uint8_t* base = (uint8_t*)(((uintptr_t)ws + 1023) & ~(uintptr_t)1023);
  __half* q2 = (__half*)(base + L.q2);
  __half* strip = (__half*)(base + L.strip);
  float4* pinfo = (float4*)(base + L.pinfo);
  float2* cand = (float2*)(base + L.cand);
  float2* pinfo2 = (float2*)(base + L.pinfo2);
  float* unk = (float*)(base + L.unk);

  const int64_t np = (int64_t)n * P;
  sif_pack_q_kernel<METRIC><<<(unsigned)((np * 32 + 255) / 256), 256, 0, st>>>(q, pstat, q2, pinfo, pinfo2, n, P, ph, pw, hh, ww);
  DSIN_LAUNCHED(h);
  DSIN_REQUIRE(h, ph <= PS_MAXPH, "patch height above 24");
  sif_pack_strip_kernel<<<dim3((ww + PS_COLS - 1) / PS_COLS, (hp + PS_ROWS - 1) / PS_ROWS, n), 256, 0, st>>>(r, strip, n, hh,
                                                                                                      ww, ph);
  DSIN_LAUNCHED(h);

  CUtensorMap tm_q, tm_s;
  const uint64_t qd[3] = {(uint64_t)KQ, (uint64_t)P, (uint64_t)n};
  const uint64_t qs[2] = {(uint64_t)KQ * 2, (uint64_t)P * KQ * 2};
  const uint32_t qb[3] = {64, 128, 1};
  const uint64_t sd[4] = {16, (uint64_t)ww / 2, (uint64_t)hp, (uint64_t)n * PAIRS};
  const uint64_t ss[3] = {32, (uint64_t)ww * 16, (uint64_t)hp * ww * 16};
  const uint32_t sb[4] = {16, STRIP_PIX / 2, 1, 1};
  if (!encode_tmap(&tm_q, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, q2, qd, qs, qb, CU_TENSOR_MAP_SWIZZLE_128B) ||
      !encode_tmap(&tm_s, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, strip, sd, ss, sb, CU_TENSOR_MAP_SWIZZLE_NONE))
    return dsin_fail(h, DSIN_ERR_CUDA, "%s: cuTensorMapEncodeTiled failed", __func__);

  SifP p;
  p.ystat = (const float4*)ystat;
  p.pinfo = pinfo;
  p.cand = cand;
  p.pinfo2 = pinfo2;
  p.unk = unk;
  p.n = n; p.hp = hp; p.wp = wp; p.P = P;
  p.ptiles = L.ptiles; p.rgroups = L.rgroups; p.jtiles = L.jtiles;
  p.total_units = n * L.ptiles * L.rgroups;
  p.use_mask = use_mask;
  p.kh = -4.0f / ((0.5f * hh) * (0.5f * hh));
  p.kw = -4.0f / ((0.5f * ww) * (0.5f * ww));
  static bool configured[DSIN_MAX_DEVICES] = {};  // cudaFuncSetAttribute is per device
  if (!configured[h->device]) {
    if (cudaFuncSetAttribute(sif_tc_kernel<METRIC>, cudaFuncAttributeMaxDynamicSharedMemorySize, sif_smem_bytes<METRIC>()) != cudaSuccess)
      return dsin_fail(h, DSIN_ERR_CUDA, "%s: cannot raise dynamic shared memory", __func__);
    configured[h->device] = true;
  }
  const int grid = p.total_units < h->sm_count ? p.total_units : h->sm_count;
  sif_tc_kernel<METRIC><<<grid, 320, sif_smem_bytes<METRIC>(), st>>>(tm_q, tm_s, p);
  DSIN_LAUNCHED(h);
  int* work_count = (int*)(base + L.work);
  int2* worklist = (int2*)(base + L.work + 16);
  if (cudaMemsetAsync(work_count, 0, 16, st) != cudaSuccess) return dsin_fail(h, DSIN_ERR_CUDA, "%s: memset failed", __func__);
  sif_rescore_kernel<METRIC><<<(unsigned)((np * 32 + 255) / 256), 256, 0, st>>>(cand, L.ngroups, q, r, pstat, ystat, n, hh, ww,
                                                                   ph, pw, use_mask, unk, keys, worklist, work_count,
                                                                   L.work_cap);
  DSIN_LAUNCHED(h);
  // groups whose candidate list may have been too short: all their positions, one CTA per group (usually none)
  sif_exhaustive_kernel<METRIC><<<h->sm_count * 8, 128, 0, st>>>(worklist, work_count, L.work_cap, q, r, pstat, ystat, n, hh, ww, ph,
                                                       pw, use_mask, keys);
  DSIN_LAUNCHED(h);
  return DSIN_OK;
}

int64_t sif_tc_work_count_offset(const void* ws, int n, int hh, int ww, int ph, int pw) {
  const uintptr_t base = ((uintptr_t)ws + 1023) & ~(uintptr_t)1023;
  return (int64_t)(base - (uintptr_t)ws) + make_layout(n, hh, ww, ph, pw).work;
}

int sif_tc_match(dsin_handle_t h, const float* q, const float* r, const float* pstat, const float* ystat, int n,
                 int hh, int ww, int ph, int pw, int use_mask, int metric, unsigned long long* keys, void* ws,
                 cudaStream_t st) {
  if (metric == SIF_L2) return sif_tc_match_impl<SIF_L2>(h, q, r, pstat, ystat, n, hh, ww, ph, pw, use_mask, keys, ws, st);
  return sif_tc_match_impl<SIF_PEARSON>(h, q, r, pstat, ystat, n, hh, ww, ph, pw, use_mask, keys, ws, st);
}

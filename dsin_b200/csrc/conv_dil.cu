// K8 with a LARGE dilation: the 32-channel 3x3 layers of the SI-Net with rate 8, 16, 32, 64, 128 (src/siNet.py:34-38) as
// tcgen05 implicit GEMMs over ROW BANDS.
//
// A 3x3 filter with dilation d reads rows y - d, y, y + d and columns x - d, x, x + d.  A 2-D halo tile (conv_h32.cu) would
// fetch (16 + 2d) x (8 + 2d) pixels per 128 outputs, and the tap-streaming kernel (conv_tc.cu, what these layers ran on
// before) fetches one activation tile per tap: measured 3.97 GB of L2 -> shared-memory traffic per layer at batch 8 for
// a 401 MB input, 0.41 ms per layer with L2 at 54 % and DRAM at 23 % (profiles/r2_v8_ncu_small.txt).  Here
//   * an output tile is 128 CONSECUTIVE pixels of one image row; its three input rows ("bands") are 128 + 2d pixels wide
//     (one or two TMA boxes, out-of-image columns zero-filled = SAME padding), 64-byte pixels, 64-byte swizzle, dense;
//     the three column taps of a band are shared-memory descriptors d * 64 bytes apart (TMA and the UMMA descriptor take
//     the swizzle phase from the absolute shared-memory address, see conv_ws.cu);
//   * a CTA walks a CHAIN of output rows y0, y0 + d, y0 + 2d, ...: the band that is the bottom tap of one row is the
//     centre of the next and the top of the one after, so every output row costs ONE new band -- the bands live in a
//     ring of 2-4 slots; bands outside the image are neither loaded nor multiplied;
//   * the MMAs are issued PER BAND, not per output row.  Band j is the bottom tap (ky = 2) of output row j - 1, the centre
//     tap of row j and the top tap of row j + 1; the three uses differ only in their weights (the ky shift moves rows, not
//     columns, so the TMEM lane -> pixel mapping is the same).  So the three ky weight blocks sit side by side in N: per
//     column tap kx and K-step, one MMA a_hi x [W(2,kx) hi; lo; W(1,kx) hi; lo; W(0,kx) hi; lo] (N = 192) into the
//     [large | small] accumulators of rows j - 1, j, j + 1, and one MMA a_lo x [W(2,kx) hi; 0; W(1,kx) hi; 0; W(0,kx) hi]
//     (N = 160) that starts at the small-term half of row j - 1 (the zero blocks add +0 to the large-term halves).  That is
//     12 MMAs per band instead of 36 per output row, and every activation band is read from shared memory 6 times instead
//     of 18.  Every accumulator receives the same products in the same (ky, kx, K-step) order as one row at a time would;
//   * accumulators: a ring of 8 slots over the TMEM columns, the CTA's output row g in slot g % 8.  An MMA cannot
//     initialise only part of its D, so all slots are zeroed at start and the epilogue zeroes a slot after reading it;
//   * filter resident, 8 epilogue warps, swizzled staging + TMA stores: as in conv_h32.cu.
// L2 -> shared traffic per layer: (128 + 2d) / 128 of the input (1.1x ... 3x) instead of 9x.
#include "tc_common.cuh"
#include "conv_tc.cuh"

using namespace tc;

namespace {

constexpr int TM = 128;         // output pixels per tile (one image row)
constexpr int NTHREADS = 320;   // warp 0: TMA producer, warp 1: MMA issuer, warps 2..9: epilogue
constexpr int NPAD = 32;
constexpr int NSLOT = 8;        // accumulator slots in TMEM (output rows in flight)
constexpr int BLK = NPAD * 64;  // one 32 cout x 32 cin fp16 weight block, 64-byte rows

struct Unit {
  int n, x0, y0, rows;  // image, first output column, first output row, rows in this chain segment (<= 0: empty)
};

__device__ __forceinline__ Unit decode_unit(const ConvDilArgs& p, int u) {
  Unit r;
  const int xt = u % p.tiles_w;
  int t = u / p.tiles_w;
  const int ph = t % p.phases;
  t /= p.phases;
  const int s = t % p.nseg;
  r.n = t / p.nseg;
  r.x0 = xt * TM;
  const int chain = (p.H - ph + p.dil - 1) / p.dil;  // rows ph, ph + d, ... < H
  const int j0 = s * p.seg;
  r.rows = min(p.seg, chain - j0);
  r.y0 = ph + j0 * p.dil;
  return r;
}

template <int TERMS>
__global__ void __launch_bounds__(NTHREADS, 1)
conv_dil_kernel(const __grid_constant__ CUtensorMap tm_xh, const __grid_constant__ CUtensorMap tm_xl,
                const __grid_constant__ CUtensorMap tm_wh, const __grid_constant__ CUtensorMap tm_wl,
                const __grid_constant__ CUtensorMap tm_yh, const __grid_constant__ CUtensorMap tm_yl,
                const __grid_constant__ ConvDilArgs p) {
  constexpr int PLANES = TERMS == 3 ? 2 : 1;
  constexpr int ACC = PLANES * NPAD;        // accumulator columns per slot: [large terms | small terms]
  constexpr int TMEM_COLS = NSLOT * ACC;    // 512 or 256
  constexpr int W1_KX = 3 * PLANES * BLK;   // a_hi operand of one column tap kx: [W(2,kx); W(1,kx); W(0,kx)], each [hi; lo]
  constexpr int W2_KX = 5 * BLK;            // a_lo operand of one column tap kx: [W(2,kx) hi; 0; W(1,kx) hi; 0; W(0,kx) hi]
  constexpr int W2_OFF = 3 * W1_KX;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + (((raw + 1023u) & ~1023u) - raw);
  uint8_t* wsm = smem;                                      // [kx][a_hi operand], then (terms 3) [kx][a_lo operand]
  uint8_t* bands = wsm + p.w_region;                        // nb x [plane][band]
  uint8_t* stg = bands + p.nb * PLANES * p.a_plane;         // 2 buffers x 4 quarters x [hi 2 KB, lo 2 KB]
  uint64_t* full_b = reinterpret_cast<uint64_t*>(stg + 8 * 4096);
  uint64_t* empty_b = full_b + 4;
  uint64_t* tfull = empty_b + 4;
  uint64_t* tempty = tfull + NSLOT;
  uint64_t* wfull = tempty + NSLOT;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(wfull + 1);
  float* s_scale = reinterpret_cast<float*>(tmem_ptr + 2);
  float* s_shift = s_scale + 32;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int i = 0; i < 4; ++i) {
      mbar_init(&full_b[i], 1);
      mbar_init(&empty_b[i], 1);
    }
    for (int i = 0; i < NSLOT; ++i) {
      mbar_init(&tfull[i], 1);
      mbar_init(&tempty[i], 8);
    }
    mbar_init(wfull, 1);
    fence_barrier_init();
    prefetch_tmap(&tm_xh);
    prefetch_tmap(&tm_wh);
    if (TERMS == 3) {
      prefetch_tmap(&tm_xl);
      prefetch_tmap(&tm_wl);
    }
    prefetch_tmap(&tm_yh);
  }
  if (threadIdx.x < 32) {
    s_scale[threadIdx.x] = p.scale[threadIdx.x];
    s_shift[threadIdx.x] = p.shift[threadIdx.x];
  }
  if (TERMS == 3) {  // the zero blocks of the a_lo operands (TMA fills the weight blocks around them)
    for (int i = threadIdx.x; i < 6 * BLK / 16; i += NTHREADS) {
      const int blk = i / (BLK / 16);
      sts16(smem_u32(wsm + W2_OFF + (blk >> 1) * W2_KX + (2 * (blk & 1) + 1) * BLK) + (uint32_t)(i % (BLK / 16)) * 16u,
            make_uint4(0u, 0u, 0u, 0u));
    }
    fence_proxy_async();  // generic-proxy writes -> visible to the MMAs
  }
  if (warp == 1) tmem_alloc(tmem_ptr, TMEM_COLS);
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = *tmem_ptr;
  // epilogue warp w owns TMEM lanes 32 (w % 4) ... + 31 and columns c0 ... c0 + 15 of both halves of every slot
  const int q = warp & 3;
  const int half = (warp - 2) >> 2;
  const int c0 = half * 16;
  const uint32_t zero[16] = {};
  if (warp >= 2) {  // every accumulator slot starts at zero
    for (int s = 0; s < NSLOT; ++s) {
      const uint32_t t = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(s * ACC + c0);
      tmem_st_32x16(t, zero);
      if (TERMS == 3) tmem_st_32x16(t + (uint32_t)NPAD, zero);
    }
    tmem_st_wait();
  }
  fence_before_sync();
  __syncthreads();
  fence_after_sync();

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer: the filter once, then one band per row
    if (elect_one()) {
      mbar_expect_tx(wfull, (uint32_t)((TERMS == 3 ? 27 : 9) * BLK));
      for (int ky = 0; ky < 3; ++ky)
        for (int kx = 0; kx < 3; ++kx) {
          const int t = ky * 3 + kx, b = 2 - ky;  // weight block b of a stacked operand multiplies output row j - 1 + b
          uint8_t* w1 = wsm + kx * W1_KX + b * PLANES * BLK;
          tma_load_2d(w1, &tm_wh, wfull, 0, t * NPAD);
          if (TERMS == 3) {
            tma_load_2d(w1 + BLK, &tm_wl, wfull, 0, t * NPAD);
            tma_load_2d(wsm + W2_OFF + kx * W2_KX + 2 * b * BLK, &tm_wh, wfull, 0, t * NPAD);
          }
        }
    }
    __syncwarp();
    uint32_t k = 0;  // bands loaded so far: slot k % nb, phase (k / nb) & 1
    for (int u = blockIdx.x; u < p.total_units; u += gridDim.x) {
      const Unit un = decode_unit(p, u);
      if (un.rows <= 0) continue;
      for (int j = -1; j <= un.rows; ++j) {
        const int y = un.y0 + j * p.dil;
        if (y < 0 || y >= p.H) continue;
        const uint32_t slot = k % (uint32_t)p.nb, par = (k / (uint32_t)p.nb) & 1u;
        mbar_wait(&empty_b[slot], par ^ 1u);
        if (elect_one()) {
          uint8_t* st = bands + slot * PLANES * p.a_plane;
          mbar_expect_tx(&full_b[slot], (uint32_t)(PLANES * p.nbox * p.bw * 64));
          for (int b = 0; b < p.nbox; ++b) {
            const int x = un.x0 - p.dil + b * p.bw;
            tma_load_4d(st + b * p.bw * 64, &tm_xh, &full_b[slot], 0, x, y, un.n);
            if (TERMS == 3) tma_load_4d(st + p.a_plane + b * p.bw * 64, &tm_xl, &full_b[slot], 0, x, y, un.n);
          }
        }
        __syncwarp();
        ++k;
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer: 12 MMAs per band (terms 3)
    const uint32_t w_base = smem_u32(wsm);
    const uint32_t band0 = smem_u32(bands);
    const uint32_t slot_bytes = (uint32_t)(PLANES * p.a_plane);
    const int ksteps = p.ksteps;
    // the band at a_base times weight blocks b0 ... b0 + nrows - 1 into the nrows consecutive slots from slot s
    auto issue = [&](uint32_t a_base, int b0, int s, int nrows) {
      const uint32_t d = tmem_base + (uint32_t)(s * ACC);
      const uint32_t idesc1 = make_idesc_f16(128, nrows * ACC, 0);
      const uint32_t idesc2 = make_idesc_f16(128, nrows * ACC - NPAD, 0);
#pragma unroll
      for (int kx = 0; kx < 3; ++kx) {
        const uint32_t a_off = (uint32_t)(kx * p.dil * 64);
        const uint64_t a_hi = make_smem_desc(a_base + a_off, 16, 512, LAYOUT_SW64);
        const uint64_t a_lo = make_smem_desc(a_base + p.a_plane + a_off, 16, 512, LAYOUT_SW64);
        const uint64_t b1 = make_smem_desc(w_base + (uint32_t)(kx * W1_KX + b0 * PLANES * BLK), 16, 512, LAYOUT_SW64);
        const uint64_t b2 = make_smem_desc(w_base + (uint32_t)(W2_OFF + kx * W2_KX + b0 * 2 * BLK), 16, 512, LAYOUT_SW64);
#pragma unroll
        for (int ks = 0; ks < 2; ++ks) {
          if (ks >= ksteps) break;
          umma_f16(d, a_hi + 2 * ks, b1 + 2 * ks, idesc1, 1u);                         // [hi*hi | hi*lo] per row
          if (TERMS == 3) umma_f16(d + NPAD, a_lo + 2 * ks, b2 + 2 * ks, idesc2, 1u);  // lo*hi into the small terms
        }
      }
    };
    mbar_wait(wfull, 0);
    fence_after_sync();
    uint32_t k = 0;   // global index of the unit's first in-image band
    uint32_t g0 = 0;  // output rows of earlier units: row r of this unit accumulates in slot (g0 + r) % NSLOT
    for (int u = blockIdx.x; u < p.total_units; u += gridDim.x) {
      const Unit un = decode_unit(p, u);
      if (un.rows <= 0) continue;
      const int jlo = un.y0 - p.dil >= 0 ? -1 : 0;                       // first band of the unit that is inside the image
      const int jhi = un.y0 + un.rows * p.dil < p.H ? un.rows : un.rows - 1;  // last one
      int acquired = 0;  // rows [0, acquired) of the unit own their slot
      for (int j = jlo; j <= jhi; ++j) {
        const uint32_t kb = k + (uint32_t)(j - jlo);
        mbar_wait(&full_b[kb % (uint32_t)p.nb], (kb / (uint32_t)p.nb) & 1u);
        const int ra = max(j - 1, 0), rb = min(j + 1, un.rows - 1);  // the unit's output rows this band feeds
        for (; acquired <= rb; ++acquired) {
          const uint32_t g = g0 + (uint32_t)acquired;
          mbar_wait(&tempty[g % NSLOT], ((g / NSLOT) & 1u) ^ 1u);
        }
        fence_after_sync();
        if (elect_one()) {
          const uint32_t a_base = band0 + (kb % (uint32_t)p.nb) * slot_bytes;
          const int s = (int)((g0 + (uint32_t)ra) % NSLOT);
          const int n1 = min(rb - ra + 1, NSLOT - s);  // rows before the slot ring wraps
          issue(a_base, ra - j + 1, s, n1);
          if (n1 <= rb - ra) issue(a_base, ra + n1 - j + 1, 0, rb - ra + 1 - n1);
          umma_commit(&empty_b[kb % (uint32_t)p.nb]);
          // row j - 1 has all its bands now; after the unit's last band, so have the rows below it
          const int rlast = j == jhi ? un.rows - 1 : j - 1;
          for (int r = max(j - 1, 0); r <= rlast; ++r) umma_commit(&tfull[(g0 + (uint32_t)r) % NSLOT]);
        }
        __syncwarp();
      }
      k += (uint32_t)(jhi - jlo + 1);
      g0 += (uint32_t)un.rows;
    }
  } else {
    // ------------------------------------------------------------ epilogue warps 2..9: two per TMEM lane quarter
    const uint32_t stg_q = smem_u32(stg + q * 4096);  // + (it & 1) * 16 KB: rows alternate between two staging buffers
    const uint32_t row_off = (uint32_t)lane * 64u;
    const int sw = (lane >> 1) & 3;  // 64-byte swizzle: 16-byte piece j of pixel p sits at ((j ^ ((p >> 1) & 3)) * 16)
    const float slope = p.act == DSIN_ACT_LRELU02 ? 0.2f : 1.f;
    const float floor_v = p.act == DSIN_ACT_RELU ? 0.f : -INFINITY;
    float sc[16], sh[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      sc[j] = s_scale[c0 + j];
      sh[j] = s_shift[c0 + j];
    }
    uint32_t it = 0;  // output rows done so far
    for (int u = blockIdx.x; u < p.total_units; u += gridDim.x) {
      const Unit un = decode_unit(p, u);
      if (un.rows <= 0) continue;
      for (int r = 0; r < un.rows; ++r, ++it) {
        const uint32_t slot = it % NSLOT;
        const uint32_t stg_hi = stg_q + (it & 1u) * 4u * 4096u;
        const uint32_t stg_lo = stg_hi + 2048;
        // the stores of the row before the previous one (issued by half 0) have finished reading this staging buffer
        if (half == 0 && lane == 0) tma_store_wait_read1();
        asm volatile("bar.sync %0, 64;" ::"r"(1 + q) : "memory");
        mbar_wait(&tfull[slot], (it / NSLOT) & 1u);
        fence_after_sync();
        const uint32_t lane_base = tmem_base + ((uint32_t)(q * 32) << 16) + slot * (uint32_t)ACC + (uint32_t)c0;
        uint32_t v[16], vl[16];
        tmem_ld_32x16(lane_base, v);
        if (TERMS == 3) tmem_ld_32x16(lane_base + (uint32_t)NPAD, vl);
        tmem_ld_wait();
        tmem_st_32x16(lane_base, zero);  // the slot's next row accumulates onto zeros
        if (TERMS == 3) tmem_st_32x16(lane_base + (uint32_t)NPAD, zero);
#pragma unroll
        for (int g = 0; g < 2; ++g) {
          uint4 uh, ul;
          __half2* hh2 = reinterpret_cast<__half2*>(&uh);
          __half2* ll2 = reinterpret_cast<__half2*>(&ul);
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            float x[2];
#pragma unroll
            for (int i = 0; i < 2; ++i) {
              const int j = g * 8 + 2 * e + i;
              float a = __uint_as_float(v[j]);
              if (TERMS == 3) a = __fadd_rn(a, __uint_as_float(vl[j]));  // large + small product terms, round to nearest
              const float t = __fadd_rn(__fmul_rn(a, sc[j]), sh[j]);
              x[i] = fmaxf(fmaxf(t, __fmul_rn(t, slope)), floor_v);
            }
            const __half h0 = __float2half_rn(x[0]), h1 = __float2half_rn(x[1]);
            hh2[e] = __halves2half2(h0, h1);
            ll2[e] = __halves2half2(__float2half_rn(x[0] - __half2float(h0)), __float2half_rn(x[1] - __half2float(h1)));
          }
          const uint32_t so = row_off + (uint32_t)(((2 * half + g) ^ sw) << 4);
          sts16(stg_hi + so, uh);
          if (p.yl) sts16(stg_lo + so, ul);
        }
        tmem_st_wait();
        fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive(&tempty[slot]);
        fence_proxy_async();  // this thread's generic-proxy writes to the staging block -> visible to the TMA stores
        asm volatile("bar.sync %0, 64;" ::"r"(1 + q) : "memory");
        if (half == 0 && lane == 0) {  // the stores clip pixels past the end of the row
          const int y = un.y0 + r * p.dil;
          tma_store_4d_issue(&tm_yh, stg_hi, 0, un.x0 + q * 32, y, un.n);
          if (p.yl) tma_store_4d_issue(&tm_yl, stg_lo, 0, un.x0 + q * 32, y, un.n);
          tma_store_commit();  // one group per row
        }
      }
    }
    if (half == 0 && lane == 0) tma_store_wait_all();
    __syncwarp();
  }

  __syncthreads();
  if (warp == 1) {
    fence_after_sync();
    tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

template <int TERMS>
int launch_dil(dsin_handle_t h, const CUtensorMap* m, const ConvDilArgs& p, int smem, cudaStream_t st) {
  static bool configured[DSIN_MAX_DEVICES] = {};  // cudaFuncSetAttribute is per device
  if (!configured[h->device]) {
    if (cudaFuncSetAttribute(conv_dil_kernel<TERMS>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess)
      return dsin_fail(h, DSIN_ERR_CUDA, "%s: cannot raise dynamic shared memory", __func__);
    configured[h->device] = true;
  }
  const int grid = p.total_units < h->sm_count ? p.total_units : h->sm_count;
  conv_dil_kernel<TERMS><<<grid, NTHREADS, smem, st>>>(m[0], m[1], m[2], m[3], m[4], m[5], p);
  DSIN_LAUNCHED(h);
  return DSIN_OK;
}

}  // namespace

// x: (32 ch, W, H, N) channels-last split fp16; w packed [9][32][32] (dsin_pack_conv_w_tc); 3x3, stride 1, SAME,
// dilation a.dil in both directions; 32 -> 32 channels, split-fp16 (terms 3) or fp16 (terms 1) output.
int conv_dil_launch(dsin_handle_t h, const __half* x_hi, const __half* x_lo, const __half* w_hi, const __half* w_lo,
                    const ConvDilArgs& a, cudaStream_t st) {
  if (a.dil < 1 || a.H < 1 || a.W < 8 || a.n < 1) return dsin_fail(h, DSIN_ERR_UNSUPPORTED, "%s: bad geometry", __func__);
  if (a.ksteps < 1 || a.ksteps > 2) return dsin_fail(h, DSIN_ERR_ARG, "%s: ksteps must be 1 or 2", __func__);
  const int planes = a.terms == 3 ? 2 : 1;
  ConvDilArgs p = a;
  const int band = TM + 2 * a.dil;           // pixels per band
  p.nbox = (band + 255) / 256;               // a TMA box is at most 256 pixels wide
  p.bw = ((band + p.nbox - 1) / p.nbox + 7) / 8 * 8;  // 8-pixel multiples keep every box on a swizzle-atom boundary
  p.a_plane = (p.nbox * p.bw * 64 + 1023) / 1024 * 1024;
  p.w_region = (a.terms == 3 ? 9 * 2 + 3 * 5 : 9) * BLK;  // stacked a_hi operands (+ the a_lo ones), see the kernel
  const int fixed = p.w_region + 8 * 4096 + 1024 /*barriers, scale/shift*/ + 1024 /*alignment*/;
  int nb = (227 * 1024 - fixed) / (planes * p.a_plane);
  if (nb > 4) nb = 4;
  if (nb < 2) return dsin_fail(h, DSIN_ERR_UNSUPPORTED, "%s: dilation too large for a ring of two bands", __func__);
  p.nb = nb;
  const int smem = fixed + nb * planes * p.a_plane;
  p.tiles_w = (a.W + TM - 1) / TM;
  p.phases = a.dil < a.H ? a.dil : a.H;      // chains start at rows 0 .. min(d, H) - 1
  const int chain = (a.H + a.dil - 1) / a.dil;
  // split chains into segments until there are several units per SM; a segment reloads its two halo bands
  int nseg = 1;
  while ((int64_t)a.n * p.tiles_w * p.phases * nseg < 6 * (int64_t)h->sm_count && nseg < chain) ++nseg;
  p.seg = (chain + nseg - 1) / nseg;
  p.nseg = (chain + p.seg - 1) / p.seg;
  p.total_units = a.n * p.nseg * p.phases * p.tiles_w;
  CUtensorMap m[6];
  const CUtensorMapDataType f16 = CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
  const CUtensorMapSwizzle sw = CU_TENSOR_MAP_SWIZZLE_64B;
  const uint64_t xd[4] = {32, (uint64_t)a.W, (uint64_t)a.H, (uint64_t)a.n};
  const uint64_t xs[3] = {64, (uint64_t)a.W * 64, (uint64_t)a.H * a.W * 64};
  const uint32_t xb[4] = {32, (uint32_t)p.bw, 1, 1};
  const uint64_t wd[2] = {32, (uint64_t)9 * NPAD};
  const uint64_t wsb[1] = {64};
  const uint32_t wb[2] = {32, (uint32_t)NPAD};
  const uint32_t yb[4] = {32, 32, 1, 1};
  const bool ok = encode_tmap(&m[0], f16, 4, x_hi, xd, xs, xb, sw) &&
                  encode_tmap(&m[1], f16, 4, x_lo ? x_lo : x_hi, xd, xs, xb, sw) &&
                  encode_tmap(&m[2], f16, 2, w_hi, wd, wsb, wb, sw) &&
                  encode_tmap(&m[3], f16, 2, w_lo ? w_lo : w_hi, wd, wsb, wb, sw) &&
                  encode_tmap(&m[4], f16, 4, a.yh, xd, xs, yb, sw) &&
                  encode_tmap(&m[5], f16, 4, a.yl ? a.yl : a.yh, xd, xs, yb, sw);
  if (!ok) return dsin_fail(h, DSIN_ERR_CUDA, "%s: cuTensorMapEncodeTiled failed", __func__);
  return a.terms == 3 ? launch_dil<3>(h, m, p, smem, st) : launch_dil<1>(h, m, p, smem, st);
}

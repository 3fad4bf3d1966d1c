// build_pyramid.cu -- fused all-pairs correlation volume + Gaussian-uncertainty residual + 4-level
// average pyramid on tcgen05 / TMEM / TMA (sm_100a).
//
// Replaces the data path of CorrBlock.__init__ (/root/reference/droid_slam/modules/corr.py:61-86):
//   torch.matmul (corr.py:144-152) -> .float() -> defCorrSample.gaussianMask (gaussianAttn.cu:19-68)
//   -> corr1/denominator + corr (gaussianMask_cuda.py:85-86) -> 3x F.avg_pool2d (corr.py:83-86),
// which moves ~300 MB per edge, by ONE kernel that writes the 50.1 MB pyramid exactly once.
//
// Shape contract: source/target grid 48x64-like (W == 64, H % 8 == 0, H*W % 128 == 0), C == 128.
//
// Work unit = (edge e, tile of 128 consecutive source pixels).  For a unit the CTA keeps the A tile
// (128 px x 128 ch fp16, K-major, 128B-swizzled) resident in shared memory and sweeps the target map in
// 24 chunks of 128 target pixels (2 target rows); two chunks (4 rows, 256 fp32 columns) form one TMEM
// accumulator half, and the two halves of TMEM (512 columns) are double-buffered between the MMA issuer
// and the epilogue.  A band of two halves (8 target rows) closes all four pyramid levels locally.
//
// Warp roles (320 threads, 1 CTA / SM, persistent over units):
//   warp 0   : TMA producer   (cp.async.bulk.tensor loads of A / B tiles, mbarrier expect_tx)
//   warp 1   : MMA issuer     (tcgen05.mma kind::f16, M=128 N=128 K=16, fp32 accumulate in TMEM) + TMEM alloc
//   warps 2-9: epilogue       (tcgen05.ld 32x32b.x32 -> registers; thread == source pixel == TMEM lane; the two
//                              warps of a TMEM lane quadrant split the 64 target columns in halves (xs = 0 / 1):
//                              all four pyramid levels close inside a 32-column half.  Level-0 rows (128 B) and
//                              level-1 rows (64 B) are staged in swizzled shared memory and written with TMA
//                              bulk stores, level 2/3 rows (32 B / 16 B) stored directly; the Gaussian window
//                              (<= 81 elements per source pixel) is patched in shared memory).
//                              With 4 epilogue warps the kernel was bound by their instruction issue (ncu: one
//                              warp per scheduler, 17 % issue-active, DRAM 39 %).
// Precision: PREC 1 = one fp16 product (exact for fp16-valued feature maps: the inference path);
//            PREC 2 = hi/lo fp16 split of both operands, 3 MMAs (hi*hi + hi*lo + lo*hi): ~2^-21 relative
//            per product, for fp32-valued feature maps (the training path).
#include "build_common.cuh"
#include "fused_common.cuh"

namespace lgu {

// ---------------------------------------------------------------------------------------------
// Kernel configuration
// ---------------------------------------------------------------------------------------------
constexpr int kBpThreads = 320;
constexpr int kEpiWarps = 8;
constexpr bool kL1Direct = false;   // measured: direct 64-byte row stores are slower (727 vs 610 us at E=48)

template <int PREC>
struct BpCfg {
  static constexpr int kPlanes = PREC;                        // hi (+ lo)
  static constexpr int kStages = PREC == 1 ? 3 : 2;           // B-chunk pipeline depth
  static constexpr int kStoreBufs = PREC == 1 ? 2 : 1;        // 4 KB staging buffers per epilogue warp (227 KB budget)
  static constexpr int kABytes = kPlanes * kPlaneBytes;
  static constexpr int kStageBytes = kPlanes * kPlaneBytes;
  static constexpr int kStoreBytes = kEpiWarps * kStoreBufs * 4096;
  // level-1 rows: the two warps of a TMEM lane quadrant fill the halves of ONE 32-row x 128-byte tile (the TMA
  // store engine is bound by row slots -- measured: a 64-byte-row tile costs as much as a 128-byte-row tile)
  static constexpr bool kPairL1 = PREC == 1;
  static constexpr int kL1Bytes = kPairL1 ? 4 * 2 * 4096 : 0;
  static constexpr int kBarOffset = kABytes + kStages * kStageBytes + kStoreBytes + kL1Bytes;
  static constexpr int kSmemBytes = kBarOffset + 256 + 1024;  // + barriers + 1 KB alignment slack
};

template <int PREC>
__global__ void __launch_bounds__(kBpThreads, 1)
build_pyramid_kernel(const __grid_constant__ CUtensorMap map_hi, const __grid_constant__ CUtensorMap map_lo,
                     const __grid_constant__ CUtensorMap map_bhi, const __grid_constant__ CUtensorMap map_blo,
                     const __grid_constant__ CUtensorMap map_l0, const __grid_constant__ CUtensorMap map_l1,
                     const BpParams prm) {
  using Cfg = BpCfg<PREC>;
  extern __shared__ uint8_t smem_raw[];
  // 1024-byte alignment by POINTER arithmetic on the shared array: an integer round trip makes every derived pointer
  // generic, and all staging accesses compile to generic LD.E / ST.E instead of LDS / STS (ncu: the top stall site)
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* sA = smem;                                   // [plane][atom][128 rows][128 B]
  uint8_t* sB = smem + Cfg::kABytes;                    // [stage][plane][atom][128 rows][128 B]
  uint8_t* sStore = sB + Cfg::kStages * Cfg::kStageBytes;   // [warp][buf][32 rows][128 B]
  uint8_t* sL1 = sStore + Cfg::kStoreBytes;             // [quad][2][32 rows][128 B] (PREC 1 only)
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::kBarOffset);
  uint64_t* a_full = bars + 0;
  uint64_t* a_empty = bars + 1;
  uint64_t* b_full = bars + 2;                          // [kStages]
  uint64_t* b_empty = bars + 2 + Cfg::kStages;          // [kStages]
  uint64_t* t_full = bars + 2 + 2 * Cfg::kStages;       // [2]
  uint64_t* t_empty = t_full + 2;                       // [2]
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(t_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int P = prm.P;
  const int tiles_m = P / kTileM;
  const int halves = prm.halves;                        // 256 target columns (4 rows of 64) per TMEM half
  const int Q = prm.Q;                                  // target pixels per map

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&map_hi);
    prefetch_tmap(&map_bhi);
    if (PREC == 2) { prefetch_tmap(&map_lo); prefetch_tmap(&map_blo); }
    prefetch_tmap(&map_l0);
    if (prm.has_l1) prefetch_tmap(&map_l1);
    mbar_init(a_full, 1);
    mbar_init(a_empty, 1);
    for (int s = 0; s < Cfg::kStages; ++s) {
      mbar_init(b_full + s, 1);
      mbar_init(b_empty + s, 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(t_full + b, 1);
      mbar_init(t_empty + b, kEpiWarps);                // one arrival per epilogue warp
    }
    mbar_fence_init();
  }
  if (warp == 1) tmem_alloc(tmem_ptr, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    // =============================== TMA producer ===============================
    if (lane == 0) {
      uint32_t unit_it = 0, chunk_it = 0;
      for (int u = blockIdx.x; u < prm.num_units; u += gridDim.x, ++unit_it) {
        const int e = u / tiles_m, mt = u - e * tiles_m;
        const int a_row = __ldg(prm.ii + e) * P + mt * kTileM;
        const int b_row0 = __ldg(prm.jj + e) * Q;
        mbar_wait(a_empty, (unit_it & 1) ^ 1);
        mbar_expect_tx(a_full, Cfg::kABytes);
        tma_load_2d(sA, &map_hi, a_full, 0, a_row);
        tma_load_2d(sA + kAtomBytes, &map_hi, a_full, 64, a_row);
        if (PREC == 2) {
          tma_load_2d(sA + kPlaneBytes, &map_lo, a_full, 0, a_row);
          tma_load_2d(sA + kPlaneBytes + kAtomBytes, &map_lo, a_full, 64, a_row);
        }
        const uint32_t hmask = prm.half_mask != nullptr ? __ldg(prm.half_mask + u) : 0xffffffffu;
        const int nchunks = halves * 2;
        for (int c = 0; c < nchunks; ++c) {
          if (!((hmask >> (c >> 1)) & 1u)) continue;   // sparse volume: this half is never sampled (lgu_volume_half_mask)
          const int s = chunk_it % Cfg::kStages;
          const uint32_t use = chunk_it / Cfg::kStages;
          ++chunk_it;
          mbar_wait(b_empty + s, (use & 1) ^ 1);
          uint8_t* dst = sB + s * Cfg::kStageBytes;
          const int b_row = b_row0 + c * kChunkN;
          mbar_expect_tx(b_full + s, Cfg::kStageBytes);
          tma_load_2d(dst, &map_bhi, b_full + s, 0, b_row);
          tma_load_2d(dst + kAtomBytes, &map_bhi, b_full + s, 64, b_row);
          if (PREC == 2) {
            tma_load_2d(dst + kPlaneBytes, &map_blo, b_full + s, 0, b_row);
            tma_load_2d(dst + kPlaneBytes + kAtomBytes, &map_blo, b_full + s, 64, b_row);
          }
        }
      }
    }
  } else if (warp == 1) {
    // =============================== MMA issuer ===============================
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc_f16(kTileM, kChunkN);
      const uint32_t a_addr = smem_u32(sA), b_addr = smem_u32(sB);
      uint32_t unit_it = 0, chunk_it = 0, half_it = 0;
      for (int u = blockIdx.x; u < prm.num_units; u += gridDim.x, ++unit_it) {
        mbar_wait(a_full, unit_it & 1);
        const uint32_t hmask = prm.half_mask != nullptr ? __ldg(prm.half_mask + u) : 0xffffffffu;
        for (int h = 0; h < halves; ++h) {
          if (!((hmask >> h) & 1u)) continue;
          const uint32_t buf = half_it & 1, buf_use = half_it >> 1;
          ++half_it;
          mbar_wait(t_empty + buf, (buf_use & 1) ^ 1);
          tc_fence_after();
          for (int c = 0; c < 2; ++c, ++chunk_it) {
            const int s = chunk_it % Cfg::kStages;
            const uint32_t use = chunk_it / Cfg::kStages;
            mbar_wait(b_full + s, use & 1);
            tc_fence_after();
            const uint32_t d_tmem = tmem_base + buf * 256 + c * kChunkN;
            const uint32_t bs = b_addr + s * Cfg::kStageBytes;
            uint32_t acc = 0;
#pragma unroll
            for (int pass = 0; pass < (PREC == 1 ? 1 : 3); ++pass) {
              // pass 0: hi*hi, pass 1: hi*lo, pass 2: lo*hi
              const uint32_t ap = a_addr + ((pass == 2) ? kPlaneBytes : 0);
              const uint32_t bp = bs + ((pass == 1) ? kPlaneBytes : 0);
#pragma unroll
              for (int k = 0; k < kC / 16; ++k) {
                const uint32_t koff = (k >> 2) * kAtomBytes + (k & 3) * 32;
                tc_mma_f16(d_tmem, make_kmajor_sw128_desc(ap + koff), make_kmajor_sw128_desc(bp + koff), idesc, acc);
                acc = 1;
              }
            }
            tc_commit(b_empty + s);                     // stage reusable once these MMAs have read it
          }
          tc_commit(t_full + buf);                      // accumulator half complete
        }
        tc_commit(a_empty);                             // A tile reusable
      }
    }
  } else {
    // =============================== epilogue (warps 2..9) ===============================
    const int quad = warp & 3;                          // TMEM lane quadrant this warp may read (warp id % 4)
    const int xs = (warp - 2) >> 2;                     // which 32-column half of the 64 target columns
    const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
    uint8_t* my_store = sStore + (warp - 2) * Cfg::kStoreBufs * 4096;
    uint8_t* pair_l1 = sL1 + quad * 2 * 4096;
    int sbuf = 0, l1buf = 0;
    const bool l1_issuer = Cfg::kPairL1 && xs == 0 && prm.has_l1;   // this warp's bulk groups also carry the L1 tiles
    const int gr = prm.gauss_radius;
    const unsigned rdg = 2u * (unsigned)gr + 1u;
    const int rsw = lane & 7;                           // 128B swizzle phase of this thread's staging row
    const int rsw1 = (lane >> 1) & 3;                   // 64B swizzle phase (level-1 rows)
    const int x0 = xs * 32;

    // stage one 32-float row segment per lane and hand the 32x32 tile to the TMA store engine
    auto store_tile = [&](float (&v)[32], int col, int row0, bool patch, int yy, float mx, float my, float c1, float c2,
                          float den, unsigned bx) {
      if (lane == 0) {
        // the tile staged in this buffer two level-0 stores ago must have been read; the issuer warp has one
        // level-1 group between them, so it may leave one more group pending
        if (l1_issuer) tma_wait_read<Cfg::kStoreBufs>();
        else tma_wait_read<Cfg::kStoreBufs - 1>();
      }
      __syncwarp();
      float4* rowp = reinterpret_cast<float4*>(my_store + sbuf * 4096 + lane * 128);
#pragma unroll
      for (int c = 0; c < 8; ++c) rowp[c ^ rsw] = make_float4(v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]);
      if (patch) {
        // Gaussian window columns bx .. bx+rdg-1 (wrapping) that fall into [x0, x0+32)
        float* rowf = reinterpret_cast<float*>(rowp);
        bool touched = false;
        for (unsigned k = 0; k < rdg; ++k) {
          const int x = (int)(bx + k);
          const unsigned idx = (unsigned)(x - x0);
          if (idx < 32u) {
            const unsigned pos = (((idx >> 2) ^ (unsigned)rsw) << 2) | (idx & 3u);
            rowf[pos] = gauss_residual(rowf[pos], x, yy, mx, my, c1, c2, den);
            touched = true;
          }
        }
        if (touched) {
#pragma unroll
          for (int c = 0; c < 8; ++c) {
            const float4 t = rowp[c ^ rsw];
            v[4 * c] = t.x; v[4 * c + 1] = t.y; v[4 * c + 2] = t.z; v[4 * c + 3] = t.w;
          }
        }
      }
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) {
        tma_store_2d(&map_l0, my_store + sbuf * 4096, col, row0);
        tma_commit();
      }
      sbuf = (sbuf + 1 == Cfg::kStoreBufs) ? 0 : sbuf + 1;
    };
    // level 1: 16 floats (64 B) per lane, 64B-swizzled 32-row tile (2 KB of a staging buffer)
    auto store_l1 = [&](const float (&v)[16], int col, int row0) {
      if (lane == 0) tma_wait_read<Cfg::kStoreBufs - 1>();
      __syncwarp();
      float4* rowp = reinterpret_cast<float4*>(my_store + sbuf * 4096 + lane * 64);
#pragma unroll
      for (int c = 0; c < 4; ++c) rowp[c ^ rsw1] = make_float4(v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]);
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) {
        tma_store_2d(&map_l1, my_store + sbuf * 4096, col, row0);
        tma_commit();
      }
      sbuf = (sbuf + 1 == Cfg::kStoreBufs) ? 0 : sbuf + 1;
    };

    uint32_t half_it = 0;
    for (int u = blockIdx.x; u < prm.num_units; u += gridDim.x) {
      const int e = u / tiles_m, mt = u - e * tiles_m;
      const int es = prm.out_slots != nullptr ? __ldg(prm.out_slots + e) : e;   // storage slot of this edge
      const int row0 = es * P + mt * kTileM + quad * 32;  // first output row (slot-pixel index) of this warp
      const size_t pix = (size_t)row0 + lane;
      float mx = 0.f, my = 0.f, c1 = 1.f, c2 = 1.f, den = 1.f;
      unsigned bx = 0, by = 0;
      if (gr > 0) {
        const size_t ipix = (size_t)e * P + mt * kTileM + quad * 32 + lane;      // Gaussian parameters: input order
        const float2 m = __ldg(reinterpret_cast<const float2*>(prm.means) + ipix);
        const float2 c = __ldg(reinterpret_cast<const float2*>(prm.covs) + ipix);
        mx = m.x; my = m.y; c1 = c.x; c2 = c.y;
        // den == NULL: the 6.28 * sqrt(cov_x * cov_y) of gaussianMask_cuda.py:77,85 is formed here (same fp32 roundings)
        den = prm.den != nullptr ? __ldg(prm.den + ipix) : __fmul_rn(6.28f, __fsqrt_rn(__fmul_rn(c1, c2)));
        bx = (unsigned)floor_to_int(mx) - (unsigned)gr;
        by = (unsigned)floor_to_int(my) - (unsigned)gr;
      }
      float l2_prev[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) l2_prev[i] = 0.f;

      const uint32_t hmask = prm.half_mask != nullptr ? __ldg(prm.half_mask + u) : 0xffffffffu;
      for (int h = 0; h < halves; ++h) {
        if (!((hmask >> h) & 1u)) continue;               // (flat volumes only: the pooled levels need every half)
        const uint32_t buf = half_it & 1, buf_use = half_it >> 1;
        ++half_it;
        mbar_wait(t_full + buf, buf_use & 1);
        tc_fence_after();
        const uint32_t tcol = tmem_base + lane_base + buf * 256 + xs * 32;
        float l1[2][16];
#pragma unroll
        for (int rp = 0; rp < 2; ++rp) {
          float a[32], b[32];
          tmem_ld32(tcol + (2 * rp) * 64, a);
          tmem_ld32(tcol + (2 * rp + 1) * 64, b);
          if (rp == 1) {
            // last TMEM read of this half: hand the accumulator back to the MMA issuer
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(t_empty + buf);
          }
          if (prm.round_half) {
#pragma unroll
            for (int i = 0; i < 32; ++i) {
              a[i] = __half2float(__float2half_rn(a[i]));
              b[i] = __half2float(__float2half_rn(b[i]));
            }
          }
          const int ya = 4 * h + 2 * rp, yb = ya + 1;
          const bool pa = gr > 0 && ((unsigned)ya - by) < rdg;
          const bool pb = gr > 0 && ((unsigned)yb - by) < rdg;
          if (ya * 64 + x0 < Q) store_tile(a, ya * 64 + x0, row0, pa, ya, mx, my, c1, c2, den, bx);   // flat mode: Q may
          if (yb * 64 + x0 < Q) store_tile(b, yb * 64 + x0, row0, pb, yb, mx, my, c1, c2, den, bx);   // end mid-half
          // 2x2 average, ATen order: ((a0 + a1) + b0) + b1, then / 4   (corr.py:86)
#pragma unroll
          for (int i = 0; i < 16; ++i)
            l1[rp][i] = __fmul_rn(__fadd_rn(__fadd_rn(__fadd_rn(a[2 * i], a[2 * i + 1]), b[2 * i]), b[2 * i + 1]), 0.25f);
          if (prm.has_l1) {
            if (kL1Direct) {   // 64-byte rows cost the TMA store engine a full row slot each: use the idle LSU instead
              float4* o1 = reinterpret_cast<float4*>(prm.lvl1 + pix * (size_t)(Q >> 2) + (2 * h + rp) * 32 + xs * 16);
#pragma unroll
              for (int c = 0; c < 4; ++c)
                __stcs(o1 + c, make_float4(l1[rp][4 * c], l1[rp][4 * c + 1], l1[rp][4 * c + 2], l1[rp][4 * c + 3]));
            } else if (Cfg::kPairL1) {
              // named barrier of the quadrant's two warps (ids 1..4).  A: the issuer's waits before its two level-0
              // stores of this row pair guarantee that the tile stored from this buffer two rows ago has been read.
              asm volatile("bar.sync %0, 64;" ::"r"(1 + quad) : "memory");
              float4* rowp = reinterpret_cast<float4*>(pair_l1 + l1buf * 4096 + lane * 128);
#pragma unroll
              for (int c = 0; c < 4; ++c)
                rowp[(xs * 4 + c) ^ rsw] = make_float4(l1[rp][4 * c], l1[rp][4 * c + 1], l1[rp][4 * c + 2], l1[rp][4 * c + 3]);
              fence_proxy_async();
              asm volatile("bar.sync %0, 64;" ::"r"(1 + quad) : "memory");    // B: both halves are in the tile
              if (xs == 0 && lane == 0) {
                tma_store_2d(&map_l1, pair_l1 + l1buf * 4096, (2 * h + rp) * 32, row0);
                tma_commit();
              }
              l1buf ^= 1;
            } else {
              store_l1(l1[rp], (2 * h + rp) * 32 + xs * 16, row0);
            }
          }
        }
        if (prm.lvl2 != nullptr) {
          float l2[8];
#pragma unroll
          for (int i = 0; i < 8; ++i)
            l2[i] = __fmul_rn(
                __fadd_rn(__fadd_rn(__fadd_rn(l1[0][2 * i], l1[0][2 * i + 1]), l1[1][2 * i]), l1[1][2 * i + 1]), 0.25f);
          float4* o2 = reinterpret_cast<float4*>(prm.lvl2 + pix * (size_t)(Q >> 4) + h * 16 + xs * 8);
          o2[0] = make_float4(l2[0], l2[1], l2[2], l2[3]);
          o2[1] = make_float4(l2[4], l2[5], l2[6], l2[7]);
          if ((h & 1) == 0) {
#pragma unroll
            for (int i = 0; i < 8; ++i) l2_prev[i] = l2[i];
          } else if (prm.lvl3 != nullptr) {
            float l3[4];
#pragma unroll
            for (int i = 0; i < 4; ++i)
              l3[i] = __fmul_rn(
                  __fadd_rn(__fadd_rn(__fadd_rn(l2_prev[2 * i], l2_prev[2 * i + 1]), l2[2 * i]), l2[2 * i + 1]), 0.25f);
            *reinterpret_cast<float4*>(prm.lvl3 + pix * (size_t)(Q >> 6) + (h >> 1) * 8 + xs * 4) =
                make_float4(l3[0], l3[1], l3[2], l3[3]);
          }
        }
      }
    }
    if (lane == 0) tma_wait_all();                      // all bulk stores complete before the CTA exits
    __syncwarp();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 512);
}

// ---------------------------------------------------------------------------------------------
// fmaps [T,C,P] (fp32 or fp16, NCHW as the encoders emit) -> channels-last fp16 planes [T,P,C]:
//   hi = fp16(x/4), lo = fp16(x/4 - hi)          (the /4 is corr.py:148-149, exact in binary)
// ---------------------------------------------------------------------------------------------
template <typename SRC>
__global__ void __launch_bounds__(256) pack_fmaps_kernel(const SRC* __restrict__ src, __half* __restrict__ hi,
                                                         __half* __restrict__ lo, int C, int P) {
  __shared__ float tile[32][33];
  const int t = blockIdx.z, c0 = blockIdx.y * 32, p0 = blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // 32 x 8
  for (int r = ty; r < 32; r += 8) {
    const int c = c0 + r, p = p0 + tx;
    tile[r][tx] = (c < C && p < P) ? (float)src[((size_t)t * C + c) * P + p] : 0.0f;
  }
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {
    const int p = p0 + r, c = c0 + tx;
    if (p < P && c < C) {
      const float x = tile[tx][r] * 0.25f;
      const __half h = __float2half_rn(x);
      const size_t o = ((size_t)t * P + p) * C + c;
      hi[o] = h;
      if (lo != nullptr) lo[o] = __float2half_rn(x - __half2float(h));
    }
  }
}

// Vector version for C % 64 == 0, P % 64 == 0 and 16-byte aligned tensors: 64 channels x 64 pixels per block, 16-byte
// loads along the pixel axis and 16-byte stores along the channel axis (the scalar kernel above moved 2 bytes per
// thread and took 31 us for 20 frames, 38 % of the roofline).
template <typename SRC>
__global__ void __launch_bounds__(256) pack_fmaps_vec_kernel(const SRC* __restrict__ src, __half* __restrict__ hi,
                                                             __half* __restrict__ lo, int C, int P) {
  __shared__ float tile[64][65];
  constexpr int PER = 16 / (int)sizeof(SRC);             // source elements per 16-byte load (8 halves / 4 floats)
  constexpr int SEGS = 64 / PER;                         // 16-byte segments per 64-pixel row
  const int t = blockIdx.z, c0 = blockIdx.y * 64, p0 = blockIdx.x * 64;
  for (int q = threadIdx.x; q < 64 * SEGS; q += 256) {
    const int c = q / SEGS, seg = q - c * SEGS;
    const uint4 raw = *reinterpret_cast<const uint4*>(src + ((size_t)t * C + c0 + c) * P + p0 + seg * PER);
    const SRC* e = reinterpret_cast<const SRC*>(&raw);
#pragma unroll
    for (int k = 0; k < PER; ++k) tile[c][seg * PER + k] = (float)e[k];
  }
  __syncthreads();
  for (int q = threadIdx.x; q < 64 * 8; q += 256) {
    const int p = q >> 3, seg = q & 7;
    __align__(16) __half h[8];
    __align__(16) __half l[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const float x = tile[seg * 8 + k][p] * 0.25f;
      h[k] = __float2half_rn(x);
      l[k] = __float2half_rn(x - __half2float(h[k]));
    }
    const size_t o = ((size_t)t * P + p0 + p) * C + c0 + seg * 8;
    *reinterpret_cast<uint4*>(hi + o) = *reinterpret_cast<const uint4*>(h);
    if (lo != nullptr) *reinterpret_cast<uint4*>(lo + o) = *reinterpret_cast<const uint4*>(l);
  }
}

// ---------------------------------------------------------------------------------------------
// Host side
// ---------------------------------------------------------------------------------------------

template <int PREC>
static int launch_build(const CUtensorMap& mh, const CUtensorMap& ml, const CUtensorMap& mbh, const CUtensorMap& mbl,
                        const CUtensorMap& m0, const CUtensorMap& m1, const BpParams& prm, cudaStream_t st) {
  using Cfg = BpCfg<PREC>;
  auto kern = build_pyramid_kernel<PREC>;
  if (int rc = optin_smem(reinterpret_cast<const void*>(kern), Cfg::kSmemBytes, "lgu_build_pyramid")) return rc;
  const int sms = num_sms();
  const int grid = prm.num_units < sms ? prm.num_units : sms;
  kern<<<grid, kBpThreads, Cfg::kSmemBytes, st>>>(mh, ml, mbh, mbl, m0, m1, prm);
  return check_launch("lgu_build_pyramid");
}

}  // namespace lgu

extern "C" int lgu_pack_fmaps(const void* fmaps, int src_is_half, void* hi, void* lo, int T, int C, int P,
                              void* stream) {
  if (T == 0) return LGU_OK;
  LGU_REQUIRE(fmaps && hi, "lgu_pack_fmaps: null pointer");
  LGU_REQUIRE(T > 0 && C > 0 && P > 0 && T <= 65535, "lgu_pack_fmaps: bad sizes T=%d C=%d P=%d", T, C, P);
  const bool aligned = ((reinterpret_cast<uintptr_t>(fmaps) | reinterpret_cast<uintptr_t>(hi) |
                         reinterpret_cast<uintptr_t>(lo)) & 15) == 0;
  if ((C % 64) == 0 && (P % 64) == 0 && aligned) {
    const dim3 vgrid(P / 64, C / 64, T);
    if (src_is_half)
      lgu::pack_fmaps_vec_kernel<__half><<<vgrid, 256, 0, (cudaStream_t)stream>>>(
          reinterpret_cast<const __half*>(fmaps), reinterpret_cast<__half*>(hi), reinterpret_cast<__half*>(lo), C, P);
    else
      lgu::pack_fmaps_vec_kernel<float><<<vgrid, 256, 0, (cudaStream_t)stream>>>(
          reinterpret_cast<const float*>(fmaps), reinterpret_cast<__half*>(hi), reinterpret_cast<__half*>(lo), C, P);
    return lgu::check_launch("lgu_pack_fmaps");
  }
  const dim3 grid((P + 31) / 32, (C + 31) / 32, T);
  if (src_is_half)
    lgu::pack_fmaps_kernel<__half><<<grid, 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const __half*>(fmaps), reinterpret_cast<__half*>(hi), reinterpret_cast<__half*>(lo), C, P);
  else
    lgu::pack_fmaps_kernel<float><<<grid, 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const float*>(fmaps), reinterpret_cast<__half*>(hi), reinterpret_cast<__half*>(lo), C, P);
  return lgu::check_launch("lgu_pack_fmaps");
}

static int build_pyramid_impl(const void* fmaps_hi, const void* fmaps_lo, const int32_t* ii, const int32_t* jj,
                              const float* means, const float* covs, const float* den, float* lvl0, float* lvl1,
                              float* lvl2, float* lvl3, const int32_t* out_slots, int num_slots, int T, int E, int H,
                              int W, int C, int gauss_radius, int precision, int round_half, void* stream);
extern "C" int lgu_build_pyramid(const void* fmaps_hi, const void* fmaps_lo, const int32_t* ii, const int32_t* jj,
                                 const float* means, const float* covs, const float* den, float* lvl0, float* lvl1,
                                 float* lvl2, float* lvl3, int T, int E, int H, int W, int C, int gauss_radius,
                                 int precision, int round_half, void* stream) {
  return build_pyramid_impl(fmaps_hi, fmaps_lo, ii, jj, means, covs, den, lvl0, lvl1, lvl2, lvl3, nullptr, E, T, E, H, W,
                            C, gauss_radius, precision, round_half, stream);
}
extern "C" int lgu_build_pyramid_slots(const void* fmaps_hi, const void* fmaps_lo, const int32_t* ii, const int32_t* jj,
                                       const float* means, const float* covs, const float* den, float* lvl0,
                                       float* lvl1, float* lvl2, float* lvl3, const int32_t* out_slots, int num_slots,
                                       int T, int E, int H, int W, int C, int gauss_radius, int precision,
                                       int round_half, void* stream) {
  if (E > 0 && out_slots == nullptr) {
    lgu::set_error("lgu_build_pyramid_slots: null slot list");
    return LGU_ERR_BAD_ARG;
  }
  return build_pyramid_impl(fmaps_hi, fmaps_lo, ii, jj, means, covs, den, lvl0, lvl1, lvl2, lvl3, out_slots, num_slots, T,
                            E, H, W, C, gauss_radius, precision, round_half, stream);
}
static int build_pyramid_impl(const void* fmaps_hi, const void* fmaps_lo, const int32_t* ii, const int32_t* jj,
                              const float* means, const float* covs, const float* den, float* lvl0, float* lvl1,
                              float* lvl2, float* lvl3, const int32_t* out_slots, int num_slots, int T, int E, int H,
                              int W, int C, int gauss_radius, int precision, int round_half, void* stream) {
  using namespace lgu;
  if (E == 0) return LGU_OK;
  LGU_REQUIRE(fmaps_hi && ii && jj && lvl0, "lgu_build_pyramid: null pointer");
  LGU_REQUIRE(precision == 1 || precision == 2, "lgu_build_pyramid: precision must be 1 or 2");
  LGU_REQUIRE(precision == 1 || fmaps_lo != nullptr, "lgu_build_pyramid: precision 2 needs the lo plane");
  LGU_REQUIRE(T > 0 && E > 0 && gauss_radius >= 0 && gauss_radius <= 15, "lgu_build_pyramid: bad sizes");
  LGU_REQUIRE(gauss_radius == 0 || (means && covs), "lgu_build_pyramid: Gaussian parameters missing");
  if (!(W == 64 && H > 0 && (H % 8) == 0 && C == 128)) {
    set_error("lgu_build_pyramid: only W=64, H%%8==0, C=128 grids are implemented (got H=%d W=%d C=%d)", H, W, C);
    return LGU_ERR_UNSUPPORTED;
  }
  LGU_REQUIRE(lvl2 == nullptr || lvl1 != nullptr, "lgu_build_pyramid: lvl2 requires lvl1");
  LGU_REQUIRE(lvl3 == nullptr || lvl2 != nullptr, "lgu_build_pyramid: lvl3 requires lvl2");
  const int P = H * W;
  LGU_REQUIRE(num_slots >= 1, "lgu_build_pyramid: bad pool size %d", num_slots);
  LGU_REQUIRE((long long)num_slots * P < 2147483647LL && (long long)T * P < 2147483647LL, "lgu_build_pyramid: too many rows");
  const long long S = num_slots;                                 // rows of the output storage = slots * P

  CUtensorMap mh, ml, m0, m1;
  int rc = make_map_2d(&mh, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, fmaps_hi, (uint64_t)T * P, C, 128, 64);
  if (rc) return rc;
  rc = make_map_2d(&ml, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, precision == 2 ? fmaps_lo : fmaps_hi, (uint64_t)T * P, C,
                   128, 64);
  if (rc) return rc;
  rc = make_map_2d(&m0, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, lvl0, (uint64_t)S * P, P, 32, 32);
  if (rc) return rc;
  // level-1 store tiles: 32 rows x 128 B shared by a warp pair (precision 1), 32 rows x 64 B per warp (precision 2)
  rc = make_map_2d(&m1, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, lvl1 ? lvl1 : lvl0, (uint64_t)S * P, lvl1 ? P / 4 : P, 32,
                   precision == 1 ? 32 : 16, precision == 1 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B);
  if (rc) return rc;

  BpParams prm;
  prm.ii = ii; prm.jj = jj; prm.means = means; prm.covs = covs; prm.den = den;
  prm.lvl0 = lvl0; prm.lvl1 = lvl1; prm.lvl2 = lvl2; prm.lvl3 = lvl3;
  prm.E = E; prm.P = P; prm.H = H; prm.gauss_radius = gauss_radius; prm.round_half = round_half;
  prm.num_units = E * (P / kTileM);
  prm.has_l1 = lvl1 != nullptr;
  prm.half_mask = nullptr;
  prm.boxes = nullptr; prm.box_coords = nullptr; prm.box_W = 64; prm.box_level = 0;
  prm.out_slots = out_slots;
  prm.Q = P;
  prm.halves = H / 4;
  // fp16-valued maps, all four levels: the 16-epilogue-warp kernel (build_pyramid16.cu; 573-580 us with this one at E = 48,
  // 503 us there)
  if (precision == 1 && lvl1 != nullptr && lvl2 != nullptr && lvl3 != nullptr)
    return launch_build16(mh, mh, prm, false, (cudaStream_t)stream);
  if (precision == 1) return launch_build<1>(mh, ml, mh, ml, m0, m1, prm, (cudaStream_t)stream);
  return launch_build<2>(mh, ml, mh, ml, m0, m1, prm, (cudaStream_t)stream);
}

static int build_volume_impl(const void* fmaps1_hi, const void* fmaps1_lo, const void* fmaps2_hi,
                             const void* fmaps2_lo, const int32_t* ii, const int32_t* jj, float* volume, int T1,
                             int T2, int E, int P, int Q, int C, int precision, const uint32_t* half_mask, void* stream,
                             float* boxes = nullptr, const float* box_coords = nullptr, int box_W = 64, int box_level = 0) {
  using namespace lgu;
  if (E == 0) return LGU_OK;
  LGU_REQUIRE(fmaps1_hi && fmaps2_hi && ii && jj && (volume || boxes), "lgu_build_volume: null pointer");
  if (boxes != nullptr) volume = boxes;                        // (tensor maps of the unused volume path need a valid base)
  LGU_REQUIRE(precision == 1 || precision == 2, "lgu_build_volume: precision must be 1 or 2");
  LGU_REQUIRE(precision == 1 || (fmaps1_lo && fmaps2_lo), "lgu_build_volume: precision 2 needs the lo planes");
  LGU_REQUIRE(T1 > 0 && T2 > 0 && E > 0 && P > 0 && Q > 0, "lgu_build_volume: bad sizes");
  if (!(C == 128 && (P % kTileM) == 0 && (Q % 4) == 0)) {
    set_error("lgu_build_volume: needs C=128, P%%128==0, Q%%4==0 (got C=%d P=%d Q=%d)", C, P, Q);
    return LGU_ERR_UNSUPPORTED;
  }
  LGU_REQUIRE((long long)E * P < 2147483647LL && (long long)T1 * P < 2147483647LL && (long long)T2 * Q < 2147483647LL,
              "lgu_build_volume: too many rows");
  CUtensorMap mh, ml, mbh, mbl, m0;
  int rc = make_map_2d(&mh, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, fmaps1_hi, (uint64_t)T1 * P, C, 128, 64);
  if (rc) return rc;
  rc = make_map_2d(&ml, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, precision == 2 ? fmaps1_lo : fmaps1_hi, (uint64_t)T1 * P, C,
                   128, 64);
  if (rc) return rc;
  rc = make_map_2d(&mbh, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, fmaps2_hi, (uint64_t)T2 * Q, C, 128, 64);
  if (rc) return rc;
  rc = make_map_2d(&mbl, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, precision == 2 ? fmaps2_lo : fmaps2_hi, (uint64_t)T2 * Q, C,
                   128, 64);
  if (rc) return rc;
  rc = make_map_2d(&m0, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, volume, (uint64_t)E * P, Q, 32, 32);
  if (rc) return rc;
  BpParams prm;
  prm.ii = ii; prm.jj = jj; prm.means = nullptr; prm.covs = nullptr; prm.den = nullptr;
  prm.lvl0 = volume; prm.lvl1 = nullptr; prm.lvl2 = nullptr; prm.lvl3 = nullptr;
  prm.E = E; prm.P = P; prm.H = 0; prm.gauss_radius = 0; prm.round_half = 0;
  prm.num_units = E * (P / kTileM);
  prm.has_l1 = 0;
  prm.half_mask = half_mask;
  prm.boxes = boxes; prm.box_coords = box_coords; prm.box_W = box_W; prm.box_level = box_level;
  prm.H = boxes != nullptr ? Q / box_W : 0;
  prm.out_slots = nullptr;
  prm.Q = Q;
  prm.halves = (Q + 255) / 256;
  // fp16-valued maps (the backend's buffer): the 16-warp kernel with its barrier-free flat epilogue (2 % faster on the backend
  // step than this kernel with pair-shared 16 KB TMA boxes)
  if (precision == 1) return launch_build16(mh, mbh, prm, true, (cudaStream_t)stream);
  return launch_build<2>(mh, ml, mbh, mbl, m0, m0, prm, (cudaStream_t)stream);
}

extern "C" int lgu_build_volume(const void* fmaps1_hi, const void* fmaps1_lo, const void* fmaps2_hi,
                                const void* fmaps2_lo, const int32_t* ii, const int32_t* jj, float* volume, int T1,
                                int T2, int E, int P, int Q, int C, int precision, void* stream) {
  return build_volume_impl(fmaps1_hi, fmaps1_lo, fmaps2_hi, fmaps2_lo, ii, jj, volume, T1, T2, E, P, Q, C, precision, nullptr,
                           stream);
}

extern "C" int lgu_build_volume_sparse(const void* fmaps1_hi, const void* fmaps1_lo, const void* fmaps2_hi,
                                       const void* fmaps2_lo, const int32_t* ii, const int32_t* jj,
                                       const uint32_t* half_mask, float* volume, int T1, int T2, int E, int P, int Q, int C,
                                       int precision, void* stream) {
  LGU_REQUIRE(E == 0 || half_mask != nullptr, "lgu_build_volume_sparse: null half mask");
  LGU_REQUIRE(Q <= 32 * 256, "lgu_build_volume_sparse: more than 32 halves (Q = %d)", Q);
  return build_volume_impl(fmaps1_hi, fmaps1_lo, fmaps2_hi, fmaps2_lo, ii, jj, volume, T1, T2, E, P, Q, C, precision,
                           half_mask, stream);
}

// Level 0 of the backend path as COMPACT boxes: for every source pixel only the 16 x 20 window of its correlation slice that
// lgu_altcorr_lookup_boxes_into stages around coords (rows box_origin_y(floor(cy), 7, H) .. + 15, columns
// box_origin_x(floor(cx), 7, W) .. + 19, zeros outside the H x W grid) -- 1280 bytes per pixel instead of the rows of a 12 KB
// slice.  Same MMAs and the same half mask as lgu_build_volume_sparse; fp16-valued maps, W = 64.
extern "C" int lgu_build_boxes(const void* fmaps1_hi, const void* fmaps2_hi, const int32_t* ii, const int32_t* jj,
                               const float* coords, const uint32_t* half_mask, float* boxes, int T1, int T2, int E, int H,
                               int W, int C, int level, void* stream) {
  if (E == 0) return LGU_OK;
  LGU_REQUIRE(coords && half_mask && boxes, "lgu_build_boxes: null pointer");
  LGU_REQUIRE(((reinterpret_cast<uintptr_t>(boxes) & 15) | (reinterpret_cast<uintptr_t>(coords) & 7)) == 0,
              "lgu_build_boxes: boxes must be 16-byte, coords 8-byte aligned");
  const int H2 = H >> level, W2 = W >> level;
  if (level < 0 || level > 1 || (W2 != 64 && W2 != 32) || H2 <= 0 || (H2 * W2) % 256 != 0 || H2 * W2 > 32 * 256 ||
      (H % (2 << level)) != 0) {
    lgu::set_error("lgu_build_boxes: needs level 0 or 1, W >> level in {64, 32} and whole halves (got H=%d W=%d level=%d)",
                   H, W, level);
    return LGU_ERR_UNSUPPORTED;
  }
  return build_volume_impl(fmaps1_hi, nullptr, fmaps2_hi, nullptr, ii, jj, nullptr, T1, T2, E, H * W, H2 * W2, C, 1, half_mask,
                           stream, boxes, coords, W2, level);
}

namespace lgu {
// Which 256-column halves of a [E,P,Q] volume (target rows of W2 = W >> level columns: 256 / W2 rows per half) the fused
// backend lookup can touch: per unit of 128 source pixels, the union over its pixels of the rows [yb - 1, yb + kRows + 1] of
// the lookup's staged box, yb = box_origin_y(floor(cy / 2^level), 7, H2) (lookup_fused.cu; offsets bounded by 4 keep every
// tap inside that box, one row of slack for px = c + 4.0 rounding up to the next integer).  One warp per unit.
__global__ void __launch_bounds__(256) volume_half_mask_kernel(const float* __restrict__ coords, uint32_t* __restrict__ mask,
                                                               int num_units, int H2, int rows_per_half, int halves, int level) {
  const int lane = threadIdx.x & 31;
  const int u = (int)((blockIdx.x * (unsigned)blockDim.x + threadIdx.x) >> 5);
  if (u >= num_units) return;
  uint32_t m = 0;
#pragma unroll
  for (int q = 0; q < kTileM / 32; ++q) {
    float cy = __ldg(coords + ((size_t)u * kTileM + q * 32 + lane) * 2 + 1);
    for (int l = 0; l < level; ++l) cy = __fmul_rn(cy, 0.5f);     // the lookup's own successive halving
    const int yb = box_origin_y(floor_to_int(cy), 7, H2);
    const int y0 = max(yb - 1, 0), y1 = min(yb + fl::kBH01 + 1, H2 - 1);
    if (y0 <= y1) {
      const int h0 = y0 / rows_per_half, h1 = min(y1 / rows_per_half, halves - 1);
      m |= (h1 >= 31 ? 0xffffffffu : ((2u << h1) - 1u)) & ~((1u << h0) - 1u);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m |= __shfl_xor_sync(0xffffffffu, m, o);
  if (lane == 0) mask[u] = m;
}
}  // namespace lgu

extern "C" int lgu_volume_half_mask(const float* coords, uint32_t* half_mask, int E, int H, int W, int level, void* stream) {
  using namespace lgu;
  if (E == 0) return LGU_OK;
  LGU_REQUIRE(coords && half_mask, "lgu_volume_half_mask: null pointer");
  LGU_REQUIRE(E > 0 && H > 0 && W > 0 && level >= 0 && level < 4, "lgu_volume_half_mask: bad sizes");
  const int P = H * W, H2 = H >> level, W2 = W >> level;
  if ((P % kTileM) != 0 || W2 <= 0 || (256 % W2) != 0 || (long long)H2 * W2 > 32 * 256) {
    set_error("lgu_volume_half_mask: needs H*W %% 128 == 0, (W >> level) dividing 256 and at most 32 halves (H=%d W=%d level=%d)",
              H, W, level);
    return LGU_ERR_UNSUPPORTED;
  }
  const int num_units = E * (P / kTileM);
  const int halves = (H2 * W2 + 255) / 256;
  volume_half_mask_kernel<<<(num_units + 7) / 8, 256, 0, (cudaStream_t)stream>>>(coords, half_mask, num_units, H2, 256 / W2,
                                                                               halves, level);
  return check_launch("lgu_volume_half_mask");
}

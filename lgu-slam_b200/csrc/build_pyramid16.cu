// build_pyramid16.cu -- the fused pyramid build of build_pyramid.cu with SIXTEEN epilogue warps (fp16-valued feature
// maps, all four levels; the frontend / CorrBlock.__init__ case).  Same producer, same tcgen05 issuer, same outputs
// bit for bit; what changes is who drains the accumulator.
//
// Why: a clock64 trace of the 8-warp kernel (DESIGN.md; a diagnostic build up to commit b094b8a) shows its epilogue warps waiting
// 3 % of their time for a free staging buffer, 4-8 % for the accumulator and 2 % at barriers -- the other ~90 % is their
// own, latency-bound instruction stream (two epilogue warps per scheduler, 24 % issue slots used), while the TMA store
// engine has >= 20 % headroom.  More warps per TMEM lane quadrant is the lever.
//
// Epilogue split: the four warps of a TMEM lane quadrant (warp id % 4) take (column half xs) x (row pair rp) of every
// accumulator half (4 target rows x 64 columns):
//   * one row at a time: tcgen05.ld 32 columns -> [fp16 rounding] -> staged in the warp's 4 KB swizzled tile (Gaussian
//     window patched in shared memory) -> full-line LSU stores; the horizontal pair sums a[2i] + a[2i+1] of the upper row
//     are kept (16 registers) so the 2x2 average keeps ATen's order ((a0 + a1) + b0) + b1 without holding both rows;
//   * level 1: the two xs-warps of a row pair fill one 32-row x 128-byte tile; after a quadrant barrier every warp stores
//     8 rows of the quadrant's two tiles (rp = 0, 1) through the LSU;
//   * levels 2 / 3: after that barrier every warp reads the two level-1 tiles back from shared memory and produces a
//     quarter of the level-2 row (4 columns, one 16-byte store per lane) and, every second half, 2 columns of level 3.
// Shared memory: A 32 KB + 3 x 32 KB operand stages + 16 x 4 KB level-0 staging + 8 x 4 KB level-1 tiles = 224 KB.
#include "build_common.cuh"
#include "fused_common.cuh"

namespace lgu {

namespace b16 {
constexpr int kEpiWarps = 16;
constexpr int kThreads = (2 + kEpiWarps) * 32;       // 576
constexpr int kStages = 3;
constexpr int kABytes = kPlaneBytes;                 // 32 KB
constexpr int kStageBytes = kPlaneBytes;             // 32 KB
constexpr int kStoreBytes = kEpiWarps * 4096;        // 64 KB, one staging tile per warp
constexpr int kL1Bytes = 4 * 2 * 4096;               // [quad][rp][32 rows][128 B]
constexpr int kBarOffset = kABytes + kStages * kStageBytes + kStoreBytes + kL1Bytes;
constexpr int kSmemBytes = kBarOffset + 256 + 1024;
}  // namespace b16

// FLAT: one [E,P,Q] volume of level-0 source maps x the maps behind map_b (lgu_build_volume: no Gaussian patch, no pooled
// levels, any Q % 4 == 0, optional half mask) -- the epilogue is then barrier-free: tcgen05.ld -> staging tile -> LSU.
template <bool FLAT>
__global__ void __launch_bounds__(b16::kThreads, 1)
build_pyramid16_kernel(const __grid_constant__ CUtensorMap map_hi, const __grid_constant__ CUtensorMap map_b,
                       const BpParams prm) {
  using namespace b16;
  extern __shared__ uint8_t smem_raw[];
  // 1024-byte alignment by POINTER arithmetic on the shared array: an integer round trip makes every derived pointer
  // generic, and all staging accesses compile to generic LD.E / ST.E instead of LDS / STS (ncu: the top stall site)
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* sA = smem;
  uint8_t* sB = smem + kABytes;
  uint8_t* sStore = sB + kStages * kStageBytes;        // [epilogue warp][32 rows][128 B]
  uint8_t* sL1 = sStore + kStoreBytes;                 // [quad][rp][32 rows][128 B]
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kBarOffset);
  uint64_t* a_full = bars + 0;
  uint64_t* a_empty = bars + 1;
  uint64_t* b_full = bars + 2;
  uint64_t* b_empty = bars + 2 + kStages;
  uint64_t* t_full = bars + 2 + 2 * kStages;
  uint64_t* t_empty = t_full + 2;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(t_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int P = prm.P;
  const int tiles_m = P / kTileM;
  const int halves = prm.halves;
  const int Q = prm.Q;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&map_hi);
    prefetch_tmap(&map_b);
    mbar_init(a_full, 1);
    mbar_init(a_empty, 1);
    for (int s = 0; s < kStages; ++s) {
      mbar_init(b_full + s, 1);
      mbar_init(b_empty + s, 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(t_full + b, 1);
      mbar_init(t_empty + b, kEpiWarps);
    }
    mbar_fence_init();
  }
  if (warp == 1) tmem_alloc(tmem_ptr, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    // =============================== TMA producer (as in build_pyramid.cu, one fp16 plane) ===============================
    if (lane == 0) {
      uint32_t unit_it = 0, chunk_it = 0;
      for (int u = blockIdx.x; u < prm.num_units; u += gridDim.x, ++unit_it) {
        const int e = u / tiles_m, mt = u - e * tiles_m;
        const int a_row = __ldg(prm.ii + e) * P + mt * kTileM;
        const int b_row0 = __ldg(prm.jj + e) * Q;
        mbar_wait(a_empty, (unit_it & 1) ^ 1);
        mbar_expect_tx(a_full, kABytes);
        tma_load_2d(sA, &map_hi, a_full, 0, a_row);
        tma_load_2d(sA + kAtomBytes, &map_hi, a_full, 64, a_row);
        const uint32_t hmask = (FLAT && prm.half_mask != nullptr) ? __ldg(prm.half_mask + u) : 0xffffffffu;
        const int nchunks = halves * 2;
        for (int c = 0; c < nchunks; ++c) {
          if (!((hmask >> (c >> 1)) & 1u)) continue;   // sparse volume: this half is never sampled (lgu_volume_half_mask)
          const int s = chunk_it % kStages;
          const uint32_t use = chunk_it / kStages;
          ++chunk_it;
          mbar_wait(b_empty + s, (use & 1) ^ 1);
          uint8_t* dst = sB + s * kStageBytes;
          const int b_row = b_row0 + c * kChunkN;
          mbar_expect_tx(b_full + s, kStageBytes);
          tma_load_2d(dst, &map_b, b_full + s, 0, b_row);
          tma_load_2d(dst + kAtomBytes, &map_b, b_full + s, 64, b_row);
        }
      }
    }
  } else if (warp == 1) {
    // =============================== MMA issuer (as in build_pyramid.cu) ===============================
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc_f16(kTileM, kChunkN);
      const uint32_t a_addr = smem_u32(sA), b_addr = smem_u32(sB);
      uint32_t unit_it = 0, chunk_it = 0, half_it = 0;
      for (int u = blockIdx.x; u < prm.num_units; u += gridDim.x, ++unit_it) {
        mbar_wait(a_full, unit_it & 1);
        const uint32_t hmask = (FLAT && prm.half_mask != nullptr) ? __ldg(prm.half_mask + u) : 0xffffffffu;
        for (int h = 0; h < halves; ++h) {
          if (!((hmask >> h) & 1u)) continue;
          const uint32_t buf = half_it & 1, buf_use = half_it >> 1;
          ++half_it;
          mbar_wait(t_empty + buf, (buf_use & 1) ^ 1);
          tc_fence_after();
          for (int c = 0; c < 2; ++c, ++chunk_it) {
            const int s = chunk_it % kStages;
            const uint32_t use = chunk_it / kStages;
            mbar_wait(b_full + s, use & 1);
            tc_fence_after();
            const uint32_t d_tmem = tmem_base + buf * 256 + c * kChunkN;
            const uint32_t bs = b_addr + s * kStageBytes;
            uint32_t acc = 0;
#pragma unroll
            for (int k = 0; k < kC / 16; ++k) {
              const uint32_t koff = (k >> 2) * kAtomBytes + (k & 3) * 32;
              tc_mma_f16(d_tmem, make_kmajor_sw128_desc(a_addr + koff), make_kmajor_sw128_desc(bs + koff), idesc, acc);
              acc = 1;
            }
            tc_commit(b_empty + s);
          }
          tc_commit(t_full + buf);
        }
        tc_commit(a_empty);
      }
    }
  } else {
    // =============================== epilogue (warps 2..17) ===============================
    const int quad = warp & 3;                          // TMEM lane quadrant this warp may read (warp id % 4)
    const int sub = (warp - 2) >> 2;                    // 0..3 inside the quadrant
    const int xs = sub & 1, rp = sub >> 1;              // column half, row pair
    const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
    uint8_t* my_store = sStore + (warp - 2) * 4096;
    uint8_t* l1_mine = sL1 + (quad * 2 + rp) * 4096;    // the level-1 tile this warp half-fills
    const uint8_t* l1_rows[2] = {sL1 + (quad * 2 + 0) * 4096, sL1 + (quad * 2 + 1) * 4096};
    const int gr = prm.gauss_radius;
    const unsigned rdg = 2u * (unsigned)gr + 1u;
    const int rsw = lane & 7;                           // 128B swizzle phase of this thread's staging row
    const int x0 = xs * 32;
    const int bar_id = 1 + quad;                        // named barrier of the quadrant's four warps (128 threads)

    // stage_tile: one 32-float row segment per lane into the warp's swizzled staging tile (the previous flush has read it),
    // Gaussian window patched in shared memory, patched values read back into v (they feed the pooled levels).
    auto stage_tile = [&](float (&v)[32], bool patch, int yy, float mx, float my, float c1, float c2, float den, unsigned bx) {
      float4* rowp = reinterpret_cast<float4*>(my_store + lane * 128);
#pragma unroll
      for (int c = 0; c < 8; ++c) rowp[c ^ rsw] = make_float4(v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]);
      if (patch) {
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
    };
    // flush_tile: the staged 32 x 32 tile to global memory.  A store instruction covers 4 rows x 128 contiguous bytes
    // (lane = row % 4 x 16-byte chunk) -- full lines, no proxy fence, no bulk-group wait before the tile is staged again
    // (537 -> 505 us at E = 48 against TMA tile stores); loads in batches of four so that the stores do not serialise on
    // one register quad.
    auto flush_tile = [&](int col, int row0) {
      __syncwarp();
#pragma unroll
      for (int it0 = 0; it0 < 8; it0 += 4) {
        float4 q[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int row = (it0 + j) * 4 + (lane >> 3), ch = lane & 7;
          q[j] = *reinterpret_cast<const float4*>(my_store + row * 128 + ((ch ^ (row & 7)) << 4));
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int row = (it0 + j) * 4 + (lane >> 3), ch = lane & 7;
          if (!FLAT || col + ch * 4 < Q)                         // flat volumes: Q may end inside the last half
            __stcs(reinterpret_cast<float4*>(prm.lvl0 + (size_t)(row0 + row) * (size_t)Q + col + ch * 4), q[j]);
        }
      }
      __syncwarp();
    };

    uint32_t half_it = 0;
    for (int u = blockIdx.x; u < prm.num_units; u += gridDim.x) {
      const int e = u / tiles_m, mt = u - e * tiles_m;
      const int es = prm.out_slots != nullptr ? __ldg(prm.out_slots + e) : e;
      const int row0 = es * P + mt * kTileM + quad * 32;
      const size_t pix = (size_t)row0 + lane;
      float mx = 0.f, my = 0.f, c1 = 1.f, c2 = 1.f, den = 1.f;
      unsigned bx = 0, by = 0;
      if (gr > 0) {
        const size_t ipix = (size_t)e * P + mt * kTileM + quad * 32 + lane;
        const float2 m = __ldg(reinterpret_cast<const float2*>(prm.means) + ipix);
        const float2 c = __ldg(reinterpret_cast<const float2*>(prm.covs) + ipix);
        mx = m.x; my = m.y; c1 = c.x; c2 = c.y;
        // den == NULL: the 6.28 * sqrt(cov_x * cov_y) of gaussianMask_cuda.py:77,85 is formed here (same fp32 roundings)
        den = prm.den != nullptr ? __ldg(prm.den + ipix) : __fmul_rn(6.28f, __fsqrt_rn(__fmul_rn(c1, c2)));
        bx = (unsigned)floor_to_int(mx) - (unsigned)gr;
        by = (unsigned)floor_to_int(my) - (unsigned)gr;
      }
      float l2_prev[4] = {0.f, 0.f, 0.f, 0.f};
      // compact mode: this lane's source pixel keeps only the 16 x 20 box the backend lookup stages around its coordinate
      int cbx = 0, cby = 0;
      float* cbox = nullptr;
      if (FLAT && prm.boxes != nullptr) {
        const float2 cc = __ldg(reinterpret_cast<const float2*>(prm.box_coords) + pix);
        float cx = cc.x, cy = cc.y;
        for (int l = 0; l < prm.box_level; ++l) { cx = __fmul_rn(cx, 0.5f); cy = __fmul_rn(cy, 0.5f); }   // the lookup's halving
        cbx = box_origin_x(floor_to_int(cx), 7, prm.box_W);
        cby = box_origin_y(floor_to_int(cy), 7, prm.H);
        cbox = prm.boxes + pix * (size_t)(fl::kBW01 * fl::kBH01);
        if (sub == 0) {                                         // box rows outside the grid: no half produces them
          const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
          for (int r = 0; r < fl::kBH01; ++r)
            if ((unsigned)(cby + r) >= (unsigned)prm.H) {
#pragma unroll
              for (int j = 0; j < fl::kBW01 / 4; ++j) *reinterpret_cast<float4*>(cbox + r * fl::kBW01 + 4 * j) = z4;
            }
        }
      }
      // one staged row of this warp (32 consecutive targets q0 .. q0 + 31 = target row q0 / W, columns q0 % W ..) -> this
      // lane's box row: the 16-byte chunks of the box that fall into these columns come from the lane's OWN staged row (no
      // transposition); chunks left / right of the grid are zeros (written by the first / last column block of the row)
      auto box_row = [&](int q0) {
        const int bw = prm.box_W;
        const int yy = q0 / bw, blk = (q0 - yy * bw) >> 5, nblk = bw >> 5;
        const int r = yy - cby;
        if ((unsigned)r < (unsigned)fl::kBH01) {
          const float4* rowp = reinterpret_cast<const float4*>(my_store + lane * 128);
          float* dst = cbox + r * fl::kBW01;
#pragma unroll
          for (int j = 0; j < fl::kBW01 / 4; ++j) {
            const int cg = (cbx >> 2) + j;                      // chunk of the target row (cbx % 4 == 0)
            const bool mine = (blk == 0 || cg >= 8 * blk) && (blk == nblk - 1 || cg < 8 * (blk + 1));
            if (mine) {
              float4 v4 = make_float4(0.f, 0.f, 0.f, 0.f);
              if ((unsigned)cg < (unsigned)(bw >> 2)) v4 = rowp[(cg - 8 * blk) ^ rsw];
              *reinterpret_cast<float4*>(dst + 4 * j) = v4;
            }
          }
        }
      };

      const uint32_t hmask = (FLAT && prm.half_mask != nullptr) ? __ldg(prm.half_mask + u) : 0xffffffffu;
      for (int h = 0; h < halves; ++h) {
        if (!((hmask >> h) & 1u)) continue;
        const uint32_t buf = half_it & 1, buf_use = half_it >> 1;
        ++half_it;
        mbar_wait(t_full + buf, buf_use & 1);
        tc_fence_after();
        const uint32_t tcol = tmem_base + lane_base + buf * 256 + xs * 32;
        const int ya = 4 * h + 2 * rp, yb = ya + 1;
        float ha[16], l1[16];
        uint32_t braw[32];
        {
          float a[32];
          tmem_ld32(tcol + (2 * rp) * 64, a);
          if (prm.round_half) {
#pragma unroll
            for (int i = 0; i < 32; ++i) a[i] = __half2float(__float2half_rn(a[i]));
          }
          const bool pa = gr > 0 && ((unsigned)ya - by) < rdg;
          stage_tile(a, pa, ya, mx, my, c1, c2, den, bx);
          if (!FLAT) {
#pragma unroll
            for (int i = 0; i < 16; ++i) ha[i] = __fadd_rn(a[2 * i], a[2 * i + 1]);
          }
        }
        tmem_ld32_issue(tcol + (2 * rp + 1) * 64, braw);          // the lower row travels while the upper row is flushed
        if (FLAT && cbox != nullptr) {
          __syncwarp();
          box_row(ya * 64 + x0);
          __syncwarp();
        } else {
          flush_tile(ya * 64 + x0, row0);
        }
        {
          float b[32];
          tmem_ld32_wait(braw);
#pragma unroll
          for (int i = 0; i < 32; ++i) b[i] = __uint_as_float(braw[i]);
          tc_fence_before();                            // last TMEM read of this half by this warp
          __syncwarp();
          if (lane == 0) mbar_arrive(t_empty + buf);
          if (prm.round_half) {
#pragma unroll
            for (int i = 0; i < 32; ++i) b[i] = __half2float(__float2half_rn(b[i]));
          }
          const bool pb = gr > 0 && ((unsigned)yb - by) < rdg;
          stage_tile(b, pb, yb, mx, my, c1, c2, den, bx);
          if (FLAT) {                                           // no pooled levels: nothing to exchange, no barrier
            if (cbox != nullptr) {
              __syncwarp();
              box_row(yb * 64 + x0);
              __syncwarp();
            } else {
              flush_tile(yb * 64 + x0, row0);
            }
            continue;
          }
          // 2x2 average, ATen order: ((a0 + a1) + b0) + b1, then / 4   (corr.py:86)
#pragma unroll
          for (int i = 0; i < 16; ++i) l1[i] = __fmul_rn(__fadd_rn(__fadd_rn(ha[i], b[2 * i]), b[2 * i + 1]), 0.25f);
        }
        flush_tile(yb * 64 + x0, row0);
        // ---- level 1: quadrant barrier A (every warp has stored its rows of the previous half's tiles and read them for
        // its level-2 pass), stage, barrier B, store
        asm volatile("bar.sync %0, 128;" ::"r"(bar_id) : "memory");
        {
          float4* rowp = reinterpret_cast<float4*>(l1_mine + lane * 128);
#pragma unroll
          for (int c = 0; c < 4; ++c)
            rowp[(xs * 4 + c) ^ rsw] = make_float4(l1[4 * c], l1[4 * c + 1], l1[4 * c + 2], l1[4 * c + 3]);
        }
        asm volatile("bar.sync %0, 128;" ::"r"(bar_id) : "memory");
        // Each warp stores 8 rows of both tiles through the LSU (559 -> 543 us at E = 48 against TMA tile stores); a store
        // instruction covers 4 rows x 128 contiguous bytes (lane = row % 4 x 16-byte chunk), i.e. full lines.
#pragma unroll
        for (int tix = 0; tix < 2; ++tix) {
#pragma unroll
          for (int rr = 0; rr < 2; ++rr) {
            const int row = sub * 8 + rr * 4 + (lane >> 3), ch = lane & 7;
            const float4 vv = *reinterpret_cast<const float4*>(l1_rows[tix] + row * 128 + ((ch ^ (row & 7)) << 4));
            float* dst = prm.lvl1 + (size_t)(row0 + row) * (size_t)(Q >> 2) + (2 * h + tix) * 32 + ch * 4;
            __stcs(reinterpret_cast<float4*>(dst), vv);
          }
        }
        // ---- level 2 (and 3): this warp's quarter of the row, from the two level-1 tiles in shared memory
        {
          const float4* r0 = reinterpret_cast<const float4*>(l1_rows[0] + lane * 128);
          const float4* r1 = reinterpret_cast<const float4*>(l1_rows[1] + lane * 128);
          const float4 u0 = r0[(2 * sub) ^ rsw], u1 = r0[(2 * sub + 1) ^ rsw];
          const float4 w0 = r1[(2 * sub) ^ rsw], w1 = r1[(2 * sub + 1) ^ rsw];
          float l2[4];
          l2[0] = __fmul_rn(__fadd_rn(__fadd_rn(__fadd_rn(u0.x, u0.y), w0.x), w0.y), 0.25f);
          l2[1] = __fmul_rn(__fadd_rn(__fadd_rn(__fadd_rn(u0.z, u0.w), w0.z), w0.w), 0.25f);
          l2[2] = __fmul_rn(__fadd_rn(__fadd_rn(__fadd_rn(u1.x, u1.y), w1.x), w1.y), 0.25f);
          l2[3] = __fmul_rn(__fadd_rn(__fadd_rn(__fadd_rn(u1.z, u1.w), w1.z), w1.w), 0.25f);
          *reinterpret_cast<float4*>(prm.lvl2 + pix * (size_t)(Q >> 4) + h * 16 + sub * 4) =
              make_float4(l2[0], l2[1], l2[2], l2[3]);
          if ((h & 1) == 0) {
#pragma unroll
            for (int i = 0; i < 4; ++i) l2_prev[i] = l2[i];
          } else {
            const float l3a = __fmul_rn(__fadd_rn(__fadd_rn(__fadd_rn(l2_prev[0], l2_prev[1]), l2[0]), l2[1]), 0.25f);
            const float l3b = __fmul_rn(__fadd_rn(__fadd_rn(__fadd_rn(l2_prev[2], l2_prev[3]), l2[2]), l2[3]), 0.25f);
            *reinterpret_cast<float2*>(prm.lvl3 + pix * (size_t)(Q >> 6) + (h >> 1) * 8 + sub * 2) = make_float2(l3a, l3b);
          }
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 512);
}

int launch_build16(const CUtensorMap& mh, const CUtensorMap& mb, const BpParams& prm, bool flat, cudaStream_t st) {
  auto kern = flat ? build_pyramid16_kernel<true> : build_pyramid16_kernel<false>;
  if (int rc = optin_smem(reinterpret_cast<const void*>(kern), b16::kSmemBytes, "lgu_build_pyramid")) return rc;
  const int sms = num_sms();
  const int grid = prm.num_units < sms ? prm.num_units : sms;
  kern<<<grid, b16::kThreads, b16::kSmemBytes, st>>>(mh, mb, prm);
  return check_launch(flat ? "lgu_build_volume(16)" : "lgu_build_pyramid(16)");
}

}  // namespace lgu

// build_bwd.cu -- feature-map gradients of the fused build (backward of CorrBlock.corr, corr.py:144-152, through the
// 4-level average pyramid, corr.py:83-86) on tcgen05 / TMEM / TMA (sm_100a), straight from the LEVEL gradients.
//
// What autograd runs for the reference graph: 3 x avg_pool2d backward (dense upsampling passes), then the two fp32
// matmul backward GEMMs on the dense 37.75 MB/edge volume gradient.  Average pooling commutes with the contraction,
//     g_f1[c, p] = sum_l sum_q  G_l[p, q] * avgpool_l(f2)[c, q] / 16          (K = 3072 + 768 + 192 + 48)
//     g_f2_l[c, q] = sum_p      G_l[p, q] * f1[c, p] / 16,    g_f2 = sum_l up_l(g_f2_l) / 4^l
// so the level gradients G_l [E, P, Q_l] (as the lookups' backward leaves them) are read once per product and no
// dense intermediate exists.  Both products are HBM-bound on G (50 MB/edge) once they run on tensor cores.
//
// Precision: fp32 inputs, kind::tf32 MMAs with a 3-term split (x = hi + lo, hi = x with the low 13 mantissa bits
// cleared, lo = x - hi exactly): hi*hi + hi*lo + lo*hi -- ~2^-21 relative per product (the dropped lo*lo term), the
// same construction as the forward's PREC 2.  MEASURED (tools/diag/bb_diag.py): the tensor core's fp32 accumulation
// TRUNCATES -- every accumulating MMA costs ~2^-25 of the accumulator's magnitude, one-sided, so a K = 3072
// contraction kept in one TMEM accumulator (1152 MMAs) ends 1e-4 of the result's RMS away from fp64 even with exactly
// representable inputs.  Hence chunked accumulation: the issuer alternates between two TMEM accumulators every kChunk
// k-blocks (K = 128, 48 MMAs) and four drain warps add each finished chunk into fp32 REGISTER sums with
// round-to-nearest adds (thread == output row, 128 sums per thread).  The small operand (feature planes, pre-scaled
// by 1/16) is split once by lgu_tf32_split; the big one (G) is split on the fly by the converter warps, which read it
// from shared memory -- for the second product TRANSPOSED (G is q-contiguous, the contraction runs over p) -- and write
// the hi / lo rows to tensor memory.
//
// One CTA per output tile (128 rows x 128 channels), 320 threads:
//   warp 0    : TMA producer (A k-block 128 x 32 fp32 or raw 32 x 128, B_hi / B_lo k-blocks), ring of 4 stages
//   warp 1    : tcgen05.mma issuer (M128 N128 K8, 12 MMAs per k-block, .ts form: A from tensor memory) + TMEM allocation
//               (2 x 128 accumulator columns, then 64 columns of A_hi / A_lo per stage)
//   warps 2-5 : converters (thread == tile row == TMEM lane: mask / subtract / (transpose), tcgen05.st)
//   warps 6-9 : drain + epilogue (tcgen05.ld 32x32b.x32 of every finished chunk -> register sums -> 128-byte
//               coalesced stores along the pixel axis of the [E, C, P] output)
#include "tc_common.cuh"

namespace lgu {

namespace bb {
constexpr int kThreads = 320;
constexpr int kChunk = 4;                  // k-blocks per TMEM accumulation chunk (K = 128)
constexpr int kTile = 128;                 // M and N
constexpr int kKB = 32;                    // k-block: 32 fp32 = one 128-byte swizzle atom row
constexpr int kTileBytes = kTile * 128;    // 16 KB operand k-block
constexpr int kMaxSeg = 4;
// The converters write A_hi / A_lo into TENSOR MEMORY (tcgen05.st, thread == lane == tile row) and the MMAs take A from
// there (.ts form): a stage is raw A | B_hi | B_lo = 48 KB, and per k-block 80 KB less crosses the SM's shared memory
// than with A_hi / A_lo in shared memory (that SS form is shared-memory-bandwidth bound: 1.63 + 2.4 ms against
// 1.25 + 1.3 ms for the two products).
constexpr int kStages = 4;
constexpr int kStageBytes = 3 * kTileBytes;                     // raw A | B_hi | B_lo
constexpr int kBarOffset = kStages * kStageBytes;
constexpr int kSmemBytes = kBarOffset + 256 + 1024;             // + barriers + alignment slack
constexpr int kTmemCols = 512;                                  // accumulators 0..255, A ring 256 + 64 * stage
}  // namespace bb

struct BbMaps {
  CUtensorMap a[bb::kMaxSeg], bh[bb::kMaxSeg], bl[bb::kMaxSeg];
};
struct BbParams {
  int nseg;
  int kblocks[bb::kMaxSeg];   // k-blocks of 32 per segment
  int tiles_m;                // output row tiles per edge
  int a_rows_per_edge;        // rows of the A tensor per edge (P)
  int C;                      // channels (== 128)
  int ld;                     // output leading dimension (rows per edge of the output: P or Q_l)
  float* out;                 // [E, C, ld]
};

__host__ __device__ constexpr uint32_t make_idesc_tf32(int M, int N) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void tc_mma_tf32_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}

constexpr uint32_t kTf32Mask = 0xFFFFE000u;   // sign, exponent, 10 mantissa bits

// TR = false: A k-block = rows [row0, row0+128) x columns [kb*32, +32) of the segment's tensor (K contiguous).
// TR = true : A k-block = TRANSPOSE of rows [edge_row0 + kb*32, +32) x columns [mt*128, +128) (K = rows).
template <bool TR>
__global__ void __launch_bounds__(bb::kThreads, 1)
build_bwd_kernel(const __grid_constant__ BbMaps maps, const BbParams prm) {
  using namespace bb;
  extern __shared__ uint8_t smem_raw[];
  // 1024-byte alignment by POINTER arithmetic on the shared array: an integer round trip makes every derived pointer
  // generic, and all staging accesses compile to generic LD.E / ST.E instead of LDS / STS (ncu: the top stall site)
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kBarOffset);
  uint64_t* full = bars;                         // [kStages]  TMA bytes landed
  uint64_t* conv = bars + kStages;               // [kStages]  converted tiles visible to the tensor core
  uint64_t* empty = bars + 2 * kStages;          // [kStages]  MMAs have read the stage
  uint64_t* chunk_full = bars + 3 * kStages;     // [2]  accumulator chunk complete (tcgen05.commit)
  uint64_t* chunk_empty = chunk_full + 2;        // [2]  drained by the four drain warps
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(chunk_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int e = blockIdx.x / prm.tiles_m, mt = blockIdx.x - e * prm.tiles_m;
  constexpr int kAOff = 0;                                         // the raw tile is the only A copy in shared memory
  constexpr int kBhiOff = kTileBytes;
  constexpr int kBloOff = kBhiOff + kTileBytes;

  if (warp == 0 && lane == 0) {
#pragma unroll
    for (int l = 0; l < kMaxSeg; ++l)
      if (l < prm.nseg) { prefetch_tmap(&maps.a[l]); prefetch_tmap(&maps.bh[l]); prefetch_tmap(&maps.bl[l]); }
    for (int s = 0; s < kStages; ++s) {
      mbar_init(full + s, 1);
      mbar_init(conv + s, 4);                    // one arrival per converter warp
      mbar_init(empty + s, 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(chunk_full + b, 1);
      mbar_init(chunk_empty + b, 4);
    }
    mbar_fence_init();
  }
  if (warp == 1) tmem_alloc(tmem_ptr, kTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    // =============================== TMA producer ===============================
    if (lane == 0) {
      uint32_t it = 0;
#pragma unroll
      for (int l = 0; l < kMaxSeg; ++l) {
        if (l >= prm.nseg) break;
        const int a_edge_row = e * prm.a_rows_per_edge;
        const int b_row = e * prm.C;
        for (int kb = 0; kb < prm.kblocks[l]; ++kb, ++it) {
          const int s = it % kStages;
          const uint32_t use = it / kStages;
          mbar_wait(empty + s, (use & 1) ^ 1);
          uint8_t* st = smem + s * kStageBytes;
          mbar_expect_tx(full + s, 3 * kTileBytes);
          if (TR) tma_load_2d(st + kAOff, &maps.a[l], full + s, mt * kTile, a_edge_row + kb * kKB);
          else tma_load_2d(st + kAOff, &maps.a[l], full + s, kb * kKB, a_edge_row + mt * kTile);
          tma_load_2d(st + kBhiOff, &maps.bh[l], full + s, kb * kKB, b_row);
          tma_load_2d(st + kBloOff, &maps.bl[l], full + s, kb * kKB, b_row);
        }
      }
    }
  } else if (warp == 1) {
    // =============================== MMA issuer ===============================
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc_tf32(kTile, kTile);
      uint32_t it = 0, acc = 0;
      int total = 0;
#pragma unroll
      for (int l = 0; l < kMaxSeg; ++l)
        if (l < prm.nseg) total += prm.kblocks[l];
      for (int i = 0; i < total; ++i, ++it) {
        const int s = it % kStages;
        const uint32_t use = it / kStages;
        const uint32_t chunk = it / kChunk, buf = chunk & 1;
        if (it % kChunk == 0) {                                   // new chunk: its accumulator must have been drained
          mbar_wait(chunk_empty + buf, ((chunk >> 1) & 1) ^ 1);
          tc_fence_after();
          acc = 0;
        }
        mbar_wait(conv + s, use & 1);
        tc_fence_after();
        const uint32_t st = smem_u32(smem + s * kStageBytes);
        const uint32_t d_tmem = tmem_base + buf * kTile;
#pragma unroll
        for (int kk = 0; kk < kKB / 8; ++kk) {
          const uint32_t off = kk * 32;                           // K = 8 tf32 = 32 bytes inside the swizzle atom
          const uint64_t bhi = make_kmajor_sw128_desc(st + kBhiOff + off), blo = make_kmajor_sw128_desc(st + kBloOff + off);
          const uint32_t a_t = tmem_base + 256 + s * 64 + kk * 8;     // A_hi columns; A_lo 32 columns further
          tc_mma_tf32_ts(d_tmem, a_t, bhi, idesc, acc);
          acc = 1;
          tc_mma_tf32_ts(d_tmem, a_t, blo, idesc, 1);
          tc_mma_tf32_ts(d_tmem, a_t + 32, bhi, idesc, 1);
        }
        tc_commit(empty + s);
        if ((it % kChunk) == kChunk - 1 || i == total - 1) tc_commit(chunk_full + buf);
      }
    }
  } else if (warp < 6) {
    // =============================== converters (warps 2..5) ===============================
    // tile row owned by this thread; it is also the TMEM lane, which a warp may only touch in its own quadrant
    const int row = (warp & 3) * 32 + lane;
    const int rsw = row & 7;                                      // 128B swizzle phase of the row
    int total = 0;
#pragma unroll
    for (int l = 0; l < kMaxSeg; ++l)
      if (l < prm.nseg) total += prm.kblocks[l];
    for (int it = 0; it < total; ++it) {
      const int s = it % kStages;
      const uint32_t use = it / kStages;
      mbar_wait(full + s, use & 1);
      uint8_t* st = smem + s * kStageBytes;
      // this row's 32 k values in K order (non-TR: undo the TMA's chunk swizzle; TR: one raw column), split, and written
      // to the stage's tensor-memory columns
      uint32_t h[32], l[32];
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        float v[4];
        if (TR) {
          const float* raw = reinterpret_cast<const float*>(st + kAOff) + row;
#pragma unroll
          for (int q = 0; q < 4; ++q) v[q] = raw[(4 * c + q) * kTile];
        } else {
          const float4 t = reinterpret_cast<const float4*>(st + kAOff + row * 128)[c ^ rsw];
          v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          h[4 * c + q] = __float_as_uint(v[q]) & kTf32Mask;
          l[4 * c + q] = __float_as_uint(__fsub_rn(v[q], __uint_as_float(h[4 * c + q])));
        }
      }
      const uint32_t ta = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + 256 + s * 64;
      tmem_st32(ta, h);
      tmem_st32(ta + 32, l);
      tmem_wait_st();
      tc_fence_before();
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(conv + s);
    }
  } else {
    // =============================== drain + epilogue (warps 6..9) ===============================
    // thread == output row (TMEM lane): every finished chunk is added into 128 register sums (IEEE adds)
    const int quad = warp & 3;                                    // TMEM lane quadrant this warp may read
    const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
    int total = 0;
#pragma unroll
    for (int l = 0; l < kMaxSeg; ++l)
      if (l < prm.nseg) total += prm.kblocks[l];
    const int nchunks = (total + kChunk - 1) / kChunk;
    float sum[kTile];
#pragma unroll
    for (int i = 0; i < kTile; ++i) sum[i] = 0.0f;
    for (int j = 0; j < nchunks; ++j) {
      const uint32_t buf = j & 1;
      mbar_wait(chunk_full + buf, (j >> 1) & 1);
      tc_fence_after();
#pragma unroll
      for (int c0 = 0; c0 < kTile; c0 += 32) {
        float v[32];
        tmem_ld32(tmem_base + lane_base + buf * kTile + c0, v);
#pragma unroll
        for (int i = 0; i < 32; ++i) sum[c0 + i] = __fadd_rn(sum[c0 + i], v[i]);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(chunk_empty + buf);
    }
    const int m = mt * kTile + quad * 32 + lane;
    if (m < prm.ld) {
      float* out = prm.out + (size_t)e * prm.C * prm.ld + m;
#pragma unroll
      for (int i = 0; i < kTile; ++i) out[(size_t)i * prm.ld] = sum[i];
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, kTmemCols);
}

// x * scale -> hi (low 13 mantissa bits cleared) and lo = x * scale - hi (exact).
__global__ void __launch_bounds__(256) tf32_split_kernel(const float* __restrict__ x, float scale, float* __restrict__ hi,
                                                         float* __restrict__ lo, long long n) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const float v = __fmul_rn(x[i], scale);
    const float h = __uint_as_float(__float_as_uint(v) & kTf32Mask);
    hi[i] = h;
    lo[i] = __fsub_rn(v, h);
  }
}

template <bool TR>
static int launch_bb(const BbMaps& maps, const BbParams& prm, int E, cudaStream_t st) {
  auto kern = build_bwd_kernel<TR>;
  if (int rc = optin_smem(reinterpret_cast<const void*>(kern), bb::kSmemBytes, "lgu_build_backward_fmaps")) return rc;
  kern<<<(unsigned)(E * prm.tiles_m), bb::kThreads, bb::kSmemBytes, st>>>(maps, prm);
  return check_launch("lgu_build_backward_fmaps");
}

}  // namespace lgu

extern "C" int lgu_tf32_split(const float* x, float scale, float* hi, float* lo, long long n, void* stream) {
  if (n == 0) return LGU_OK;
  LGU_REQUIRE(x && hi && lo && n > 0, "lgu_tf32_split: bad arguments");
  long long blocks = (n + 255) / 256;
  if (blocks > 148LL * 16) blocks = 148LL * 16;
  lgu::tf32_split_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(x, scale, hi, lo, n);
  return lgu::check_launch("lgu_tf32_split");
}

extern "C" int lgu_build_backward_fmaps(const float* const* level_grads, const float* f1_hi, const float* f1_lo,
                                        const float* const* f2_hi, const float* const* f2_lo, float* g_f1,
                                        float* const* g_f2, int num_levels, int E, int H, int W, int C, void* stream) {
  using namespace lgu;
  if (E == 0) return LGU_OK;
  LGU_REQUIRE(level_grads && f1_hi && f1_lo && f2_hi && f2_lo && g_f1 && g_f2, "lgu_build_backward_fmaps: null pointer");
  LGU_REQUIRE(num_levels >= 1 && num_levels <= bb::kMaxSeg, "lgu_build_backward_fmaps: 1..4 levels (got %d)", num_levels);
  LGU_REQUIRE(E > 0 && H > 0 && W > 0, "lgu_build_backward_fmaps: bad sizes E=%d H=%d W=%d", E, H, W);
  const int P = H * W;
  if (!(C == 128 && (P % bb::kTile) == 0 && (H % (1 << (num_levels - 1))) == 0 && (W % (4 << (num_levels - 1))) == 0)) {
    set_error("lgu_build_backward_fmaps: needs C=128, H*W%%128==0 and level widths that are multiples of 4 "
              "(got C=%d H=%d W=%d levels=%d)", C, H, W, num_levels);
    return LGU_ERR_UNSUPPORTED;
  }
  LGU_REQUIRE((long long)E * P < 2147483647LL, "lgu_build_backward_fmaps: too many rows");
  const cudaStream_t st = (cudaStream_t)stream;

  // ---- product 1: g_f1[e, c, p] = sum over levels and q   (A = G_l rows, K contiguous)
  {
    BbMaps maps;
    BbParams prm;
    prm.nseg = 0;
    for (int l = 0; l < num_levels; ++l) {
      if (level_grads[l] == nullptr) continue;
      LGU_REQUIRE(f2_hi[l] && f2_lo[l], "lgu_build_backward_fmaps: level %d has a gradient but no feature planes", l);
      const int Q = (H >> l) * (W >> l);
      const int s = prm.nseg++;
      int rc = make_map_2d(&maps.a[s], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, level_grads[l], (uint64_t)E * P, Q, 128, 32);
      if (rc) return rc;
      rc = make_map_2d(&maps.bh[s], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, f2_hi[l], (uint64_t)E * C, Q, 128, 32);
      if (rc) return rc;
      rc = make_map_2d(&maps.bl[s], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, f2_lo[l], (uint64_t)E * C, Q, 128, 32);
      if (rc) return rc;
      prm.kblocks[s] = (Q + bb::kKB - 1) / bb::kKB;
    }
    if (prm.nseg == 0) {
      set_error("lgu_build_backward_fmaps: every level gradient is null");
      return LGU_ERR_BAD_ARG;
    }
    for (int s = prm.nseg; s < bb::kMaxSeg; ++s) {
      maps.a[s] = maps.a[0]; maps.bh[s] = maps.bh[0]; maps.bl[s] = maps.bl[0];
      prm.kblocks[s] = 0;
    }
    prm.tiles_m = P / bb::kTile;
    prm.a_rows_per_edge = P;
    prm.C = C;
    prm.ld = P;
    prm.out = g_f1;
    const int rc = launch_bb<false>(maps, prm, E, st);
    if (rc) return rc;
  }
  // ---- product 2, one launch per level: g_f2_l[e, c, q] = sum_p G_l[p, q] f1[c, p]   (A = G_l^T, transposed on chip)
  for (int l = 0; l < num_levels; ++l) {
    if (level_grads[l] == nullptr) continue;
    LGU_REQUIRE(g_f2[l] != nullptr, "lgu_build_backward_fmaps: g_f2[%d] is null", l);
    const int Q = (H >> l) * (W >> l);
    BbMaps maps;
    BbParams prm;
    int rc = make_map_2d(&maps.a[0], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, level_grads[l], (uint64_t)E * P, Q, 32, 128,
                         CU_TENSOR_MAP_SWIZZLE_NONE);
    if (rc) return rc;
    rc = make_map_2d(&maps.bh[0], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, f1_hi, (uint64_t)E * C, P, 128, 32);
    if (rc) return rc;
    rc = make_map_2d(&maps.bl[0], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, f1_lo, (uint64_t)E * C, P, 128, 32);
    if (rc) return rc;
    for (int s = 1; s < bb::kMaxSeg; ++s) {
      maps.a[s] = maps.a[0]; maps.bh[s] = maps.bh[0]; maps.bl[s] = maps.bl[0];
      prm.kblocks[s] = 0;
    }
    prm.nseg = 1;
    prm.kblocks[0] = P / bb::kKB;
    prm.tiles_m = (Q + bb::kTile - 1) / bb::kTile;
    prm.a_rows_per_edge = P;
    prm.C = C;
    prm.ld = Q;
    prm.out = g_f2[l];
    rc = launch_bb<true>(maps, prm, E, st);
    if (rc) return rc;
  }
  return LGU_OK;
}

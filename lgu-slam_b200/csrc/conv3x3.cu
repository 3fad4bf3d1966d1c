// conv3x3.cu -- the offset heads' 3x3 convolutions (ofsMap / ofs_residual, nn.Conv2d(C_in, C_out, 3, padding=1), called
// from corr.py:117-135) with their input and weight gradients, on tcgen05 / TMEM / TMA (sm_100a), in fp32 accuracy.
//
// Precision: the same construction as build_bwd.cu.  Every operand is split into tf32 planes, hi = x with the low 13
// mantissa bits cleared and lo = x - hi (exact), and each product runs as hi*hi + hi*lo + lo*hi on kind::tf32 MMAs
// (~2^-21 relative per product, the dropped lo*lo term).  The tensor core's fp32 accumulation truncates (DESIGN
// "measured facts"), so the issuer alternates between two TMEM accumulators every kChunk k-blocks (K = 128) and the
// drain warps add each finished chunk into fp32 register sums with round-to-nearest adds.
// Non-finite values: a +-inf or NaN x is split as hi = 0, lo = x (NaN canonicalised, so that tf32 truncation cannot turn
// a NaN into an inf).  Of the three terms only lo_x * hi_y then sees it, and that is +-inf * w or NaN exactly where the
// fp32 product is: hi_y is 0 only when y is 0.  (hi = inf, lo = 0 would give inf * lo_w = NaN for every weight that is
// exact in tf32, and lo = x - hi would give inf - inf.)
//
// Layouts (all fp32):
//   activations planes  [E, H, W, Cp] channels-last, Cp = C rounded up to 32, padded channels zero (lgu_conv3x3_pack)
//   forward weights     [9, Np, C_in]      Np = 112 (C_out <= 112) or 128: the MMA's N, padded rows zero
//   input-grad weights  [9, C_in, Kp]      W flipped and transposed, Kp = C_out rounded up to 32
//   weight-grad g_y     [E, Np, H*W]       g_y split in its own pixel-contiguous layout (K = pixels is then K-major)
//
// fprop / dgrad (conv_gemm_kernel): implicit GEMM, one CTA per 128 output pixels x N channels, M = 128 pixels (128/W
// full rows, or a 128-pixel run of one row), K = 9 taps x Cp.  The A k-block of tap (ky, kx) is ONE 4-D TMA box
// {32 channels, bw, bh, 1} of the planes at (c, x0 + kx - 1, y0 + ky - 1, e): the +-1 shift lands on the outer x / y
// dimensions (never on the innermost one, whose start must stay 16-byte aligned) and TMA's zero fill of out-of-bounds
// rows and columns is the convolution's zero padding.  Every operand is in shared memory (.ss form), 192 threads:
//   warp 0    : TMA producer (A_hi, A_lo, B_hi, B_lo k-blocks), ring of 3 stages
//   warp 1    : tcgen05.mma issuer (M128 x N x K8, 12 MMAs per k-block) + TMEM allocation (2 x 128 columns)
//   warps 2-5 : drain + epilogue (thread == output pixel; NCHW stores, coalesced along the pixel axis; + bias)
//
// wgrad (conv_wgrad_kernel): g_W[co, ci, tap] = sum over e, y, x of g_y[e, co, y, x] * x[e, ci, y + ky - 1, x + kx - 1],
// M = 128 input channels, N = Np output channels, K = pixels, split over CTAs by a partition of the k-blocks that depends
// only on the shapes.  The shifted operand is A: a TMA box {128 channels, 32 pixels of one row, 1, 1} of the channels-
// last planes at the tap-shifted (x, y) (zero fill again), which the converter warps transpose on chip (thread == input
// channel == TMEM lane) into tensor memory (.ts form), as build_bwd.cu does for G.  192 threads:
//   warp 0 producer, warp 1 issuer, warps 2-5 converters that also drain (-> fp32 partials [S, 9, Np, C_in]); with
//   separate drain warps (320 threads, as build_bwd.cu) a thread has 168 registers and the 128 sums spill
// The partials are added in split order by conv_wgrad_reduce_kernel and g_b by conv_bias_grad_kernel (fp64, fixed tree):
// no float atomics, so all results are bit-identical from run to run.
#include "tc_common.cuh"
#include "../../include/lgu_corr_ext.h"

namespace lgu {

namespace cv {
constexpr int kChunk = 4;                       // k-blocks per TMEM accumulation chunk (K = 128)
constexpr int kKB = 32;                         // k-block: 32 fp32 = one 128-byte swizzle atom row
constexpr int kM = 128;
constexpr int kBlockBytes = 128 * 128;          // one 128-row k-block
constexpr int kStages = 3;
constexpr int kStageBytes = 4 * kBlockBytes;    // A_hi | A_lo | B_hi | B_lo
constexpr int kBarOffset = kStages * kStageBytes;
constexpr int kSmemBytes = kBarOffset + 256 + 1024;
constexpr int kGemmThreads = 192;
constexpr int kWgradThreads = 192;             // 6 warps: 255 registers a thread (10 warps: 168)
constexpr int kWaveCtas = 2 * kNumSMs;          // wgrad: CTAs aimed at (one CTA per SM at this shared-memory size)
constexpr uint32_t kTf32Mask = 0xFFFFE000u;
}  // namespace cv

struct CvMaps {
  CUtensorMap ahi, alo, bhi, blo;
};
struct CvParams {
  int kc;            // fprop / dgrad: k-blocks per tap (Cp / 32)
  int tiles_m;       // fprop / dgrad: pixel tiles per edge;  wgrad: channel tiles (C_in / 128, rounded up)
  int tiles_n;       // fprop / dgrad: channel tiles
  int n_valid;       // output channels written (C_out for fprop, C_in for dgrad)
  int H, W, HW;
  const float* bias; // fprop: [C_out]; dgrad: NULL
  float* out;        // fprop / dgrad: [E, n_valid, H, W];  wgrad: partials [S, 9, Np, C_in]
  // wgrad
  int splits;
  long long kblocks; // E * HW / 32
  int c_in, a_rows;  // A rows that hold channels (box rows); the rest of the 128 TMEM lanes read as 0
};

__device__ __forceinline__ void split_tf32(float v, float& h, float& l) {
  if (isfinite(v)) {
    h = __uint_as_float(__float_as_uint(v) & cv::kTf32Mask);
    l = __fsub_rn(v, h);
  } else {
    h = 0.0f;
    l = isnan(v) ? __uint_as_float(0x7FC00000u) : v;
  }
}

__host__ __device__ constexpr uint32_t cv_idesc_tf32(int M, int N) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void tc_mma_tf32_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
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
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2,
                                            int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}

// 32 lanes x 16 consecutive fp32 columns: half of tmem_ld32's temporaries next to the N register sums.
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// Add finished accumulator chunk j (N columns) into `sum` (thread == TMEM lane) and hand the accumulator back.
template <int N>
__device__ __forceinline__ void drain_chunk(float (&sum)[N], int j, uint32_t tmem_base, uint32_t lane_base,
                                            uint64_t* chunk_full, uint64_t* chunk_empty, int lane) {
  const uint32_t buf = j & 1;
  mbar_wait(chunk_full + buf, (j >> 1) & 1);
  tc_fence_after();
#pragma unroll
  for (int c0 = 0; c0 < N; c0 += 16) {
    float v[16];
    tmem_ld16(tmem_base + lane_base + buf * 128 + c0, v);
#pragma unroll
    for (int i = 0; i < 16; ++i) sum[c0 + i] = __fadd_rn(sum[c0 + i], v[i]);
  }
  tc_fence_before();
  __syncwarp();
  if (lane == 0) mbar_arrive(chunk_empty + buf);
}

// ---------------------------------------------------------------------------------------------
// fprop / dgrad: implicit GEMM, every operand from shared memory
// ---------------------------------------------------------------------------------------------
template <int N>
__global__ void __launch_bounds__(cv::kGemmThreads, 1)
conv_gemm_kernel(const __grid_constant__ CvMaps maps, const CvParams prm) {
  using namespace cv;
  extern __shared__ uint8_t smem_raw[];
  // 1024-byte alignment by pointer arithmetic (an integer round trip would make every staging access generic)
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kBarOffset);
  uint64_t* full = bars;                         // [kStages]  TMA bytes landed
  uint64_t* empty = bars + kStages;              // [kStages]  MMAs have read the stage
  uint64_t* chunk_full = bars + 2 * kStages;     // [2]
  uint64_t* chunk_empty = chunk_full + 2;        // [2]
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(chunk_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tiles_mn = prm.tiles_m * prm.tiles_n;
  const int e = blockIdx.x / tiles_mn;
  const int r = blockIdx.x - e * tiles_mn;
  const int nt = r / prm.tiles_m, mt = r - nt * prm.tiles_m;
  const int p0 = mt * kM;
  const int total = 9 * prm.kc;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&maps.ahi); prefetch_tmap(&maps.alo); prefetch_tmap(&maps.bhi); prefetch_tmap(&maps.blo);
    for (int s = 0; s < kStages; ++s) {
      mbar_init(full + s, 1);
      mbar_init(empty + s, 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(chunk_full + b, 1);
      mbar_init(chunk_empty + b, 4);
    }
    mbar_fence_init();
  }
  if (warp == 1) tmem_alloc(tmem_ptr, 256);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    // =============================== TMA producer ===============================
    if (lane == 0) {
      const int y0 = p0 / prm.W, x0 = p0 - y0 * prm.W;
      for (int it = 0; it < total; ++it) {
        const int s = it % kStages;
        const uint32_t use = it / kStages;
        const int tap = it / prm.kc, kc = it - tap * prm.kc;
        const int ky = tap / 3, kx = tap - 3 * ky;
        mbar_wait(empty + s, (use & 1) ^ 1);
        uint8_t* st = smem + s * kStageBytes;
        mbar_expect_tx(full + s, 2 * kBlockBytes + 2 * N * 128);
        tma_load_4d(st, &maps.ahi, full + s, kc * kKB, x0 + kx - 1, y0 + ky - 1, e);
        tma_load_4d(st + kBlockBytes, &maps.alo, full + s, kc * kKB, x0 + kx - 1, y0 + ky - 1, e);
        tma_load_3d(st + 2 * kBlockBytes, &maps.bhi, full + s, kc * kKB, nt * N, tap);
        tma_load_3d(st + 3 * kBlockBytes, &maps.blo, full + s, kc * kKB, nt * N, tap);
      }
    }
  } else if (warp == 1) {
    // =============================== MMA issuer ===============================
    if (lane == 0) {
      constexpr uint32_t idesc = cv_idesc_tf32(kM, N);
      uint32_t acc = 0;
      for (int it = 0; it < total; ++it) {
        const int s = it % kStages;
        const uint32_t use = it / kStages;
        const uint32_t chunk = it / kChunk, buf = chunk & 1;
        if (it % kChunk == 0) {                                   // new chunk: its accumulator must have been drained
          mbar_wait(chunk_empty + buf, ((chunk >> 1) & 1) ^ 1);
          tc_fence_after();
          acc = 0;
        }
        mbar_wait(full + s, use & 1);
        tc_fence_after();
        const uint32_t st = smem_u32(smem + s * kStageBytes);
        const uint32_t d_tmem = tmem_base + buf * 128;
#pragma unroll
        for (int kk = 0; kk < kKB / 8; ++kk) {
          const uint32_t off = kk * 32;                           // K = 8 tf32 = 32 bytes inside the swizzle atom
          const uint64_t ahi = make_kmajor_sw128_desc(st + off), alo = make_kmajor_sw128_desc(st + kBlockBytes + off);
          const uint64_t bhi = make_kmajor_sw128_desc(st + 2 * kBlockBytes + off);
          const uint64_t blo = make_kmajor_sw128_desc(st + 3 * kBlockBytes + off);
          tc_mma_tf32_ss(d_tmem, ahi, bhi, idesc, acc);
          acc = 1;
          tc_mma_tf32_ss(d_tmem, ahi, blo, idesc, 1);
          tc_mma_tf32_ss(d_tmem, alo, bhi, idesc, 1);
        }
        tc_commit(empty + s);
        if ((it % kChunk) == kChunk - 1 || it == total - 1) tc_commit(chunk_full + buf);
      }
    }
  } else {
    // =============================== drain + epilogue (warps 2..5) ===============================
    const int quad = warp & 3;                                    // TMEM lane quadrant this warp may read
    float sum[N];
#pragma unroll
    for (int i = 0; i < N; ++i) sum[i] = 0.0f;
    for (int j = 0; j < (total + kChunk - 1) / kChunk; ++j)
      drain_chunk<N>(sum, j, tmem_base, (uint32_t)(quad * 32) << 16, chunk_full, chunk_empty, lane);
    const int p = p0 + quad * 32 + lane;
    const int n0 = nt * N;
    float* out = prm.out + ((size_t)e * prm.n_valid + n0) * prm.HW + p;
#pragma unroll
    for (int i = 0; i < N; ++i)
      if (n0 + i < prm.n_valid) out[(size_t)i * prm.HW] = prm.bias ? __fadd_rn(sum[i], __ldg(prm.bias + n0 + i)) : sum[i];
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 256);
}

// ---------------------------------------------------------------------------------------------
// wgrad: A = tap-shifted activations, transposed on chip into tensor memory; B = g_y planes in shared memory
// ---------------------------------------------------------------------------------------------
template <int N>
__global__ void __launch_bounds__(cv::kWgradThreads, 1)
conv_wgrad_kernel(const __grid_constant__ CvMaps maps, const CvParams prm) {
  using namespace cv;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kBarOffset);
  uint64_t* full = bars;                         // [kStages]  TMA bytes landed
  uint64_t* conv = bars + kStages;               // [kStages]  converted A visible to the tensor core
  uint64_t* empty = bars + 2 * kStages;          // [kStages]  MMAs have read the stage
  uint64_t* chunk_full = bars + 3 * kStages;     // [2]
  uint64_t* chunk_empty = chunk_full + 2;        // [2]
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(chunk_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // blockIdx.x = (split, tap, channel tile)
  const int units = 9 * prm.tiles_m;
  const int sp = blockIdx.x / units;
  const int u = blockIdx.x - sp * units;
  const int tap = u / prm.tiles_m, mt = u - tap * prm.tiles_m;
  const int ky = tap / 3, kx = tap - 3 * ky;
  const long long kb0 = (long long)sp * prm.kblocks / prm.splits, kb1 = (long long)(sp + 1) * prm.kblocks / prm.splits;
  const int total = (int)(kb1 - kb0);
  const int kpe = prm.HW / kKB;                                   // k-blocks per edge
  const int a_bytes = kKB * prm.a_rows * 4;                       // one raw A box (32 pixels x a_rows channels)

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&maps.ahi); prefetch_tmap(&maps.alo); prefetch_tmap(&maps.bhi); prefetch_tmap(&maps.blo);
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
  if (warp == 1) tmem_alloc(tmem_ptr, 512);      // accumulators 0..255, A ring 256 + 64 * stage
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    // =============================== TMA producer ===============================
    if (lane == 0) {
      for (int it = 0; it < total; ++it) {
        const int s = it % kStages;
        const uint32_t use = it / kStages;
        const long long kb = kb0 + it;
        const int e = (int)(kb / kpe);
        const int pix = (int)(kb - (long long)e * kpe) * kKB;
        const int y = pix / prm.W, x0 = pix - y * prm.W;
        mbar_wait(empty + s, (use & 1) ^ 1);
        uint8_t* st = smem + s * kStageBytes;
        mbar_expect_tx(full + s, 2 * a_bytes + 2 * N * 128);
        tma_load_4d(st, &maps.ahi, full + s, mt * kM, x0 + kx - 1, y + ky - 1, e);
        tma_load_4d(st + kBlockBytes, &maps.alo, full + s, mt * kM, x0 + kx - 1, y + ky - 1, e);
        tma_load_3d(st + 2 * kBlockBytes, &maps.bhi, full + s, pix, 0, e);
        tma_load_3d(st + 3 * kBlockBytes, &maps.blo, full + s, pix, 0, e);
      }
    }
  } else if (warp == 1) {
    // =============================== MMA issuer ===============================
    if (lane == 0) {
      constexpr uint32_t idesc = cv_idesc_tf32(kM, N);
      uint32_t acc = 0;
      for (int it = 0; it < total; ++it) {
        const int s = it % kStages;
        const uint32_t use = it / kStages;
        const uint32_t chunk = it / kChunk, buf = chunk & 1;
        if (it % kChunk == 0) {
          mbar_wait(chunk_empty + buf, ((chunk >> 1) & 1) ^ 1);
          tc_fence_after();
          acc = 0;
        }
        mbar_wait(conv + s, use & 1);
        tc_fence_after();
        const uint32_t st = smem_u32(smem + s * kStageBytes);
        const uint32_t d_tmem = tmem_base + buf * 128;
#pragma unroll
        for (int kk = 0; kk < kKB / 8; ++kk) {
          const uint32_t off = kk * 32;
          const uint64_t bhi = make_kmajor_sw128_desc(st + 2 * kBlockBytes + off);
          const uint64_t blo = make_kmajor_sw128_desc(st + 3 * kBlockBytes + off);
          const uint32_t a_t = tmem_base + 256 + s * 64 + kk * 8;     // A_hi columns; A_lo 32 columns further
          tc_mma_tf32_ts(d_tmem, a_t, bhi, idesc, acc);
          acc = 1;
          tc_mma_tf32_ts(d_tmem, a_t, blo, idesc, 1);
          tc_mma_tf32_ts(d_tmem, a_t + 32, bhi, idesc, 1);
        }
        tc_commit(empty + s);
        if ((it % kChunk) == kChunk - 1 || it == total - 1) tc_commit(chunk_full + buf);
      }
    }
  } else {
    // ======================= converters + drain (warps 2..5): transpose into tensor memory =======================
    // thread == input channel in the tile == TMEM lane.  Chunk j is drained once chunk j + 1 is converted: the MMAs of
    // chunk j + 1 run meanwhile, and chunk j + 2 (the same accumulator) is converted only after the drain freed it.
    const int quad = warp & 3;
    const int row = quad * 32 + lane;
    const bool live = row < prm.a_rows;
    const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
    const int nchunks = (total + kChunk - 1) / kChunk;
    float sum[N];
#pragma unroll
    for (int i = 0; i < N; ++i) sum[i] = 0.0f;
    int drained = 0;
    for (int it = 0; it < total; ++it) {
      const int s = it % kStages;
      const uint32_t use = it / kStages;
      mbar_wait(full + s, use & 1);
      const float* rh = reinterpret_cast<const float*>(smem + s * kStageBytes) + row;
      const float* rl = reinterpret_cast<const float*>(smem + s * kStageBytes + kBlockBytes) + row;
      uint32_t h[32], l[32];
#pragma unroll
      for (int k = 0; k < 32; ++k) {
        h[k] = live ? __float_as_uint(rh[k * prm.a_rows]) : 0u;
        l[k] = live ? __float_as_uint(rl[k * prm.a_rows]) : 0u;
      }
      const uint32_t ta = tmem_base + lane_base + 256 + s * 64;
      tmem_st32(ta, h);
      tmem_st32(ta + 32, l);
      tmem_wait_st();
      tc_fence_before();
      fence_proxy_async();                                        // generic reads of the stage before its TMA refill
      __syncwarp();
      if (lane == 0) mbar_arrive(conv + s);
      if ((it + 1) % kChunk == 0 && (it + 1) / kChunk >= 2) drain_chunk<N>(sum, drained++, tmem_base, lane_base, chunk_full,
                                                                        chunk_empty, lane);
    }
    while (drained < nchunks) drain_chunk<N>(sum, drained++, tmem_base, lane_base, chunk_full, chunk_empty, lane);
    const int ci = mt * kM + row;
    if (ci < prm.c_in) {
      float* out = prm.out + ((size_t)(sp * 9 + tap) * N) * prm.c_in + ci;
#pragma unroll
      for (int i = 0; i < N; ++i) out[(size_t)i * prm.c_in] = sum[i];
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 512);
}

// ---------------------------------------------------------------------------------------------
// element-wise kernels: packing, g_y split, reductions
// ---------------------------------------------------------------------------------------------
// x [E, C, HW] -> hi / lo [E, HW, Cp], channels >= C zero.  32 x 32 tiles transposed through shared memory.
__global__ void __launch_bounds__(256) conv_pack_kernel(const float* __restrict__ x, float* __restrict__ hi,
                                                        float* __restrict__ lo, int C, int HW, int Cp) {
  __shared__ float tile[32][33];
  const int ptiles = HW / 32, ctiles = Cp / 32;
  const long long b = blockIdx.x;
  const long long e = b / ((long long)ptiles * ctiles);
  const int r = (int)(b - e * ptiles * ctiles);
  const int ct = r / ptiles, pt = r - ct * ptiles;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int c = ct * 32 + ty + 8 * j;
    tile[ty + 8 * j][tx] = c < C ? __ldg(x + ((size_t)e * C + c) * HW + pt * 32 + tx) : 0.0f;
  }
  __syncthreads();
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int p = pt * 32 + ty + 8 * j;
    float h, l;
    split_tf32(tile[tx][ty + 8 * j], h, l);
    const size_t o = ((size_t)e * HW + p) * Cp + ct * 32 + tx;
    hi[o] = h;
    lo[o] = l;
  }
}

// g_y [E, C_out, HW] -> hi / lo [E, Np, HW], rows >= C_out zero.
__global__ void __launch_bounds__(256) conv_split_rows_kernel(const float* __restrict__ g, float* __restrict__ hi,
                                                              float* __restrict__ lo, int C, int Np, int HW,
                                                              long long n) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const long long row = i / HW;
    const int p = (int)(i - row * HW);
    const long long e = row / Np;
    const int c = (int)(row - e * Np);
    float h = 0.0f, l = 0.0f;
    if (c < C) split_tf32(__ldg(g + ((size_t)e * C + c) * HW + p), h, l);
    hi[i] = h;
    lo[i] = l;
  }
}

// weight [C_out, C_in, 3, 3] -> forward planes [9, Np, C_in] (dgrad = false) or input-gradient planes [9, C_in, Kp]
// holding W[co, ci, 2 - ky, 2 - kx] at tap (ky, kx) (dgrad = true); padding zero.
__global__ void __launch_bounds__(256) conv_pack_weight_kernel(const float* __restrict__ w, float* __restrict__ hi,
                                                               float* __restrict__ lo, int C_in, int C_out, int rows,
                                                               int cols, bool dgrad) {
  const int n = 9 * rows * cols;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int tap = i / (rows * cols);
    const int rc = i - tap * rows * cols;
    const int r = rc / cols, c = rc - r * cols;
    const int co = dgrad ? c : r, ci = dgrad ? r : c;
    const int src_tap = dgrad ? 8 - tap : tap;
    float h = 0.0f, l = 0.0f;
    if (co < C_out && ci < C_in) split_tf32(__ldg(w + ((size_t)co * C_in + ci) * 9 + src_tap), h, l);
    hi[i] = h;
    lo[i] = l;
  }
}

// g_w[co, ci, tap] = sum over s = 0, 1, ... of part[s, tap, co, ci], in that order.
__global__ void __launch_bounds__(256) conv_wgrad_reduce_kernel(const float* __restrict__ part, float* __restrict__ g_w,
                                                                int C_in, int C_out, int Np, int splits) {
  const int n = C_out * C_in * 9;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int co = i / (C_in * 9);
  const int r = i - co * C_in * 9;
  const int ci = r / 9, tap = r - ci * 9;
  const size_t step = (size_t)9 * Np * C_in;
  const float* p = part + ((size_t)tap * Np + co) * C_in + ci;
  float s = 0.0f;
  for (int k = 0; k < splits; ++k) s = __fadd_rn(s, __ldg(p + k * step));
  g_w[i] = s;
}

// g_b[co] = sum of g_y[:, co] in fp64: thread t adds pixels t, t + 256, ... of every edge, then a fixed tree.
__global__ void __launch_bounds__(256) conv_bias_grad_kernel(const float* __restrict__ g, float* __restrict__ g_b, int E,
                                                             int C, int HW) {
  __shared__ double red[256];
  const int co = blockIdx.x;
  double s = 0.0;
  for (int e = 0; e < E; ++e) {
    const float* row = g + ((size_t)e * C + co) * HW;
    for (int p = threadIdx.x; p < HW; p += 256) s += (double)__ldg(row + p);
  }
  red[threadIdx.x] = s;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) g_b[co] = (float)red[0];
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
static inline int round_up(int v, int m) { return (v + m - 1) / m * m; }

// Row-major tensor of 3 or 4 fp32 dimensions (dims innermost first, dense), box `box`, cached like make_map_2d.
static int make_map_nd(CUtensorMap* map, const void* base, int rank, const uint64_t* dims, const uint32_t* box,
                       CUtensorMapSwizzle swz) {
  int dev = 0;
  cudaGetDevice(&dev);
  MapKey key = {{(uint64_t)(16 + rank), (uint64_t)dev, (uint64_t)reinterpret_cast<uintptr_t>(base), (uint64_t)swz, 0, 0, 0, 0,
                 0, 0, 0, 0}};
  for (int i = 0; i < rank; ++i) {
    key.v[4 + i] = dims[i];
    key.v[8] |= (uint64_t)box[i] << (16 * i);
  }
  if (map_cache_get(key, map)) return LGU_OK;
  EncodeTiledFn fn = get_encode_fn();
  if (fn == nullptr) {
    set_error("cuTensorMapEncodeTiled is not available from the driver");
    return LGU_ERR_LAUNCH;
  }
  cuuint64_t gd[4], gs[3];
  cuuint32_t bx[4], es[4];
  uint64_t stride = 4;
  for (int i = 0; i < rank; ++i) {
    gd[i] = dims[i];
    bx[i] = box[i];
    es[i] = 1;
    if (i > 0) gs[i - 1] = stride;
    stride *= dims[i];
  }
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, (cuuint32_t)rank, const_cast<void*>(base), gd, gs, bx, es,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with CUresult %d (rank %d)", (int)r, rank);
    return LGU_ERR_LAUNCH;
  }
  map_cache_put(key, map);
  return LGU_OK;
}

struct ConvShape {
  int Np, Kp, Cin_p, HW, tiles_m_wgrad, splits;
  long long kblocks;
};
static ConvShape conv_shape(int E, int C_in, int C_out, int H, int W) {
  ConvShape s;
  s.Np = C_out <= 112 ? 112 : 128;
  s.Kp = round_up(C_out, 32);
  s.Cin_p = C_in;
  s.HW = H * W;
  s.tiles_m_wgrad = (C_in + cv::kM - 1) / cv::kM;
  s.kblocks = (long long)E * s.HW / cv::kKB;
  const int units = 9 * s.tiles_m_wgrad;
  long long sp = cv::kWaveCtas / units;
  if (sp < 1) sp = 1;
  if (sp > s.kblocks) sp = s.kblocks;
  s.splits = (int)sp;
  return s;
}
static inline long long align256(long long v) { return (v + 255) / 256 * 256; }
// workspace bytes of each operation
static long long ws_forward(const ConvShape& s, int C_in) { return 2 * align256(9LL * s.Np * C_in * 4); }
static long long ws_input(const ConvShape& s, int C_in) { return 2 * align256(9LL * C_in * s.Kp * 4); }
static long long ws_weight(const ConvShape& s, int E, int C_in) {
  return 2 * align256((long long)E * s.Np * s.HW * 4) + align256((long long)s.splits * 9 * s.Np * C_in * 4);
}

// The checks every entry point shares: sizes first (a message naming the size), E = 0 handled by the caller.
static int check_sizes(const char* who, int E, int C_in, int C_out, int H, int W) {
  LGU_REQUIRE(E >= 0, "%s: bad size E=%d", who, E);
  LGU_REQUIRE(C_in > 0 && C_in % 32 == 0, "%s: bad size C_in=%d (needs C_in %% 32 == 0)", who, C_in);
  LGU_REQUIRE(C_out > 0 && C_out <= 128, "%s: bad size C_out=%d (needs 0 < C_out <= 128)", who, C_out);
  LGU_REQUIRE(W > 0 && W % 32 == 0 && (128 % W == 0 || W % 128 == 0),
              "%s: bad size W=%d (needs W %% 32 == 0 and W dividing 128 or a multiple of 128)", who, W);
  LGU_REQUIRE(H > 0 && ((long long)H * W) % 128 == 0, "%s: bad size H=%d (needs H*W %% 128 == 0)", who, H);
  LGU_REQUIRE((long long)E * H * W * 128 < (1LL << 40) && (long long)E * 128 < 2147483647LL,
              "%s: bad size E=%d (too many edges)", who, E);
  return LGU_OK;
}
static int check_ptr(const char* who, const void* p, const char* name, int align) {
  LGU_REQUIRE(p, "%s: %s is NULL", who, name);
  LGU_REQUIRE((reinterpret_cast<uintptr_t>(p) & (uintptr_t)(align - 1)) == 0, "%s: %s is not %d-byte aligned", who, name,
              align);
  return LGU_OK;
}
#define CV_CHECK(expr)       \
  do {                       \
    if (int rc_ = (expr)) return rc_; \
  } while (0)

static int conv_gemm(const float* a_hi, const float* a_lo, const float* b_hi, const float* b_lo, int a_cp, int b_rows,
                     int n_valid, const float* bias, float* out, int E, int H, int W, bool wide_n, cudaStream_t st,
                     const char* who) {
  using namespace cv;
  CvMaps maps;
  CvParams prm = {};
  const int bw = W < 128 ? W : 128, bh = 128 / bw;
  const uint64_t adims[4] = {(uint64_t)a_cp, (uint64_t)W, (uint64_t)H, (uint64_t)E};
  const uint32_t abox[4] = {32, (uint32_t)bw, (uint32_t)bh, 1};
  CV_CHECK(make_map_nd(&maps.ahi, a_hi, 4, adims, abox, CU_TENSOR_MAP_SWIZZLE_128B));
  CV_CHECK(make_map_nd(&maps.alo, a_lo, 4, adims, abox, CU_TENSOR_MAP_SWIZZLE_128B));
  const int N = wide_n ? 128 : 112;
  const uint64_t bdims[3] = {(uint64_t)a_cp, (uint64_t)b_rows, 9};
  const uint32_t bbox[3] = {32, (uint32_t)N, 1};
  CV_CHECK(make_map_nd(&maps.bhi, b_hi, 3, bdims, bbox, CU_TENSOR_MAP_SWIZZLE_128B));
  CV_CHECK(make_map_nd(&maps.blo, b_lo, 3, bdims, bbox, CU_TENSOR_MAP_SWIZZLE_128B));
  prm.kc = a_cp / kKB;
  prm.tiles_m = H * W / kM;
  prm.tiles_n = (b_rows + N - 1) / N;
  prm.n_valid = n_valid;
  prm.H = H; prm.W = W; prm.HW = H * W;
  prm.bias = bias;
  prm.out = out;
  const long long grid = (long long)E * prm.tiles_m * prm.tiles_n;
  const void* kern = wide_n ? (const void*)conv_gemm_kernel<128> : (const void*)conv_gemm_kernel<112>;
  CV_CHECK(optin_smem(kern, kSmemBytes, who));
  if (wide_n) conv_gemm_kernel<128><<<(unsigned)grid, kGemmThreads, kSmemBytes, st>>>(maps, prm);
  else conv_gemm_kernel<112><<<(unsigned)grid, kGemmThreads, kSmemBytes, st>>>(maps, prm);
  return check_launch(who);
}

}  // namespace lgu

using namespace lgu;

extern "C" long long lgu_conv3x3_workspace_bytes(int E, int C_in, int C_out, int H, int W) {
  if (check_sizes("lgu_conv3x3_workspace_bytes", E, C_in, C_out, H, W) != LGU_OK) return -1;
  const ConvShape s = conv_shape(E > 0 ? E : 1, C_in, C_out, H, W);
  long long b = ws_forward(s, C_in);
  if (ws_input(s, C_in) > b) b = ws_input(s, C_in);
  if (ws_weight(s, E, C_in) > b) b = ws_weight(s, E, C_in);
  return b;
}

extern "C" int lgu_conv3x3_pack(const float* x, float* hi, float* lo, int E, int C, int H, int W, void* stream) {
  static const char* who = "lgu_conv3x3_pack";
  CV_CHECK(check_sizes(who, E, 32, 1, H, W));
  LGU_REQUIRE(C > 0 && C <= 4096, "%s: bad size C=%d", who, C);
  if (E == 0) return LGU_OK;
  CV_CHECK(check_ptr(who, x, "x", 4));
  CV_CHECK(check_ptr(who, hi, "hi", 16));
  CV_CHECK(check_ptr(who, lo, "lo", 16));
  const int HW = H * W, Cp = round_up(C, 32);
  const long long blocks = (long long)E * (HW / 32) * (Cp / 32);
  conv_pack_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(x, hi, lo, C, HW, Cp);
  return check_launch(who);
}

extern "C" int lgu_conv3x3_forward(const float* x_hi, const float* x_lo, const float* weight, const float* bias, float* y,
                                   void* workspace, long long workspace_bytes, int E, int C_in, int C_out, int H, int W,
                                   void* stream) {
  static const char* who = "lgu_conv3x3_forward";
  CV_CHECK(check_sizes(who, E, C_in, C_out, H, W));
  if (E == 0) return LGU_OK;
  CV_CHECK(check_ptr(who, x_hi, "x_hi", 16));
  CV_CHECK(check_ptr(who, x_lo, "x_lo", 16));
  CV_CHECK(check_ptr(who, weight, "weight", 4));
  CV_CHECK(check_ptr(who, y, "y", 4));
  CV_CHECK(check_ptr(who, workspace, "workspace", 256));
  if (bias) CV_CHECK(check_ptr(who, bias, "bias", 4));
  const ConvShape s = conv_shape(E, C_in, C_out, H, W);
  LGU_REQUIRE(workspace_bytes >= ws_forward(s, C_in), "%s: workspace_bytes=%lld < %lld", who, workspace_bytes,
              ws_forward(s, C_in));
  const cudaStream_t st = (cudaStream_t)stream;
  float* w_hi = static_cast<float*>(workspace);
  float* w_lo = w_hi + align256(9LL * s.Np * C_in * 4) / 4;
  conv_pack_weight_kernel<<<64, 256, 0, st>>>(weight, w_hi, w_lo, C_in, C_out, s.Np, C_in, false);
  CV_CHECK(check_launch(who));
  return conv_gemm(x_hi, x_lo, w_hi, w_lo, C_in, s.Np, C_out, bias, y, E, H, W, s.Np == 128, st, who);
}

extern "C" int lgu_conv3x3_backward_input(const float* gy_hi, const float* gy_lo, const float* weight, float* g_x,
                                          void* workspace, long long workspace_bytes, int E, int C_in, int C_out, int H,
                                          int W, void* stream) {
  static const char* who = "lgu_conv3x3_backward_input";
  CV_CHECK(check_sizes(who, E, C_in, C_out, H, W));
  if (E == 0) return LGU_OK;
  CV_CHECK(check_ptr(who, gy_hi, "gy_hi", 16));
  CV_CHECK(check_ptr(who, gy_lo, "gy_lo", 16));
  CV_CHECK(check_ptr(who, weight, "weight", 4));
  CV_CHECK(check_ptr(who, g_x, "g_x", 4));
  CV_CHECK(check_ptr(who, workspace, "workspace", 256));
  const ConvShape s = conv_shape(E, C_in, C_out, H, W);
  LGU_REQUIRE(workspace_bytes >= ws_input(s, C_in), "%s: workspace_bytes=%lld < %lld", who, workspace_bytes,
              ws_input(s, C_in));
  const cudaStream_t st = (cudaStream_t)stream;
  float* w_hi = static_cast<float*>(workspace);
  float* w_lo = w_hi + align256(9LL * C_in * s.Kp * 4) / 4;
  conv_pack_weight_kernel<<<64, 256, 0, st>>>(weight, w_hi, w_lo, C_in, C_out, C_in, s.Kp, true);
  CV_CHECK(check_launch(who));
  return conv_gemm(gy_hi, gy_lo, w_hi, w_lo, s.Kp, C_in, C_in, nullptr, g_x, E, H, W, true, st, who);
}

extern "C" int lgu_conv3x3_backward_weight(const float* x_hi, const float* x_lo, const float* g_y, float* g_w, float* g_b,
                                           void* workspace, long long workspace_bytes, int E, int C_in, int C_out, int H,
                                           int W, void* stream) {
  static const char* who = "lgu_conv3x3_backward_weight";
  CV_CHECK(check_sizes(who, E, C_in, C_out, H, W));
  if (E == 0) return LGU_OK;
  LGU_REQUIRE(g_w || g_b, "%s: g_w and g_b are both NULL", who);
  CV_CHECK(check_ptr(who, g_y, "g_y", 4));
  if (g_w) {
    CV_CHECK(check_ptr(who, x_hi, "x_hi", 16));
    CV_CHECK(check_ptr(who, x_lo, "x_lo", 16));
    CV_CHECK(check_ptr(who, g_w, "g_w", 4));
    CV_CHECK(check_ptr(who, workspace, "workspace", 256));
  }
  if (g_b) CV_CHECK(check_ptr(who, g_b, "g_b", 4));
  const ConvShape s = conv_shape(E, C_in, C_out, H, W);
  if (g_w)
    LGU_REQUIRE(workspace_bytes >= ws_weight(s, E, C_in), "%s: workspace_bytes=%lld < %lld", who, workspace_bytes,
                ws_weight(s, E, C_in));
  const cudaStream_t st = (cudaStream_t)stream;
  if (g_b) {
    conv_bias_grad_kernel<<<C_out, 256, 0, st>>>(g_y, g_b, E, C_out, H * W);
    CV_CHECK(check_launch(who));
  }
  if (!g_w) return LGU_OK;
  using namespace cv;
  const long long plane = align256((long long)E * s.Np * s.HW * 4) / 4;
  float* gy_hi = static_cast<float*>(workspace);
  float* gy_lo = gy_hi + plane;
  float* part = gy_lo + plane;
  const long long n = (long long)E * s.Np * s.HW;
  long long blocks = (n + 255) / 256;
  if (blocks > 148LL * 16) blocks = 148LL * 16;
  conv_split_rows_kernel<<<(unsigned)blocks, 256, 0, st>>>(g_y, gy_hi, gy_lo, C_out, s.Np, s.HW, n);
  CV_CHECK(check_launch(who));

  CvMaps maps;
  CvParams prm = {};
  const int a_rows = C_in < kM ? C_in : kM;
  const uint64_t adims[4] = {(uint64_t)C_in, (uint64_t)W, (uint64_t)H, (uint64_t)E};
  const uint32_t abox[4] = {(uint32_t)a_rows, 32, 1, 1};
  CV_CHECK(make_map_nd(&maps.ahi, x_hi, 4, adims, abox, CU_TENSOR_MAP_SWIZZLE_NONE));
  CV_CHECK(make_map_nd(&maps.alo, x_lo, 4, adims, abox, CU_TENSOR_MAP_SWIZZLE_NONE));
  const uint64_t bdims[3] = {(uint64_t)s.HW, (uint64_t)s.Np, (uint64_t)E};
  const uint32_t bbox[3] = {32, (uint32_t)s.Np, 1};
  CV_CHECK(make_map_nd(&maps.bhi, gy_hi, 3, bdims, bbox, CU_TENSOR_MAP_SWIZZLE_128B));
  CV_CHECK(make_map_nd(&maps.blo, gy_lo, 3, bdims, bbox, CU_TENSOR_MAP_SWIZZLE_128B));
  prm.tiles_m = s.tiles_m_wgrad;
  prm.H = H; prm.W = W; prm.HW = s.HW;
  prm.out = part;
  prm.splits = s.splits;
  prm.kblocks = s.kblocks;
  prm.c_in = C_in;
  prm.a_rows = a_rows;
  const void* kern = s.Np == 128 ? (const void*)conv_wgrad_kernel<128> : (const void*)conv_wgrad_kernel<112>;
  CV_CHECK(optin_smem(kern, kSmemBytes, who));
  const unsigned grid = (unsigned)(s.splits * 9 * s.tiles_m_wgrad);
  if (s.Np == 128) conv_wgrad_kernel<128><<<grid, kWgradThreads, kSmemBytes, st>>>(maps, prm);
  else conv_wgrad_kernel<112><<<grid, kWgradThreads, kSmemBytes, st>>>(maps, prm);
  CV_CHECK(check_launch(who));
  const int nout = C_out * C_in * 9;
  conv_wgrad_reduce_kernel<<<(nout + 255) / 256, 256, 0, st>>>(part, g_w, C_in, C_out, s.Np, s.splits);
  return check_launch(who);
}

// offset_heads.cu -- the offset heads' glue of CorrBlock.fpn_offset_generate / AltCorrBlock.offset_generate
// (/root/reference/droid_slam/modules/corr.py:117-135, 217-235; per_Corr_Normalization :44-51) for sm_100a.
//
// The reference runs, on the two conv outputs, mean -> 3 x unsqueeze -> var -> sqrt -> sub -> div -> tanh -> mul (twice),
// F.interpolate, add, div, 2 x permute and, at the first lookup, 2 x .contiguous(): ~14 elementwise / reduction kernels that
// each stream the [E,98,H,W] tensors through HBM (SURVEY 8f-3: 70 % of an uncached backend step was this glue).  Here:
//   offset_stats_kernel : one CTA per (edge, head): mean and biased variance over (CH,H,W), fp32 loads, fp64 accumulation
//   offset_apply_kernel : one CTA per (edge, 32-pixel tile): normalise, 4 tanh, the level-1 average with level 0, nearest
//                         upsampling of the residual head by indexing, and the NCHW -> NHWC transpose through shared memory,
//                         so the [E,H,W,98] records the lookups read are written once, fully coalesced.
// tanhf / IEEE division as torch's fp32 CUDA kernels use them; statistics differ from torch's Welford reduction in the last
// bits only (values agree to a few 1e-7, tests/test_dropin_gpu.py compares against the reference's own Python).
#include "common.cuh"
#include "../../include/lgu_corr_ext.h"

namespace lgu {

constexpr int kOhThreads = 256;

__global__ void __launch_bounds__(1024)
offset_stats_kernel(const float* __restrict__ c0, const float* __restrict__ c1, float* __restrict__ stats, long long n0,
                    long long n1, float eps) {
  const int e = blockIdx.x >> 1, head = blockIdx.x & 1;
  const long long n = head ? n1 : n0;
  const float* x = (head ? c1 : c0) + (size_t)e * n;
  double s = 0.0, ss = 0.0;
  if ((n & 3) == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0) {
    for (long long q = threadIdx.x; q < (n >> 2); q += blockDim.x) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(x) + q);
      s += (double)v.x + (double)v.y + (double)v.z + (double)v.w;
      ss += (double)v.x * v.x + (double)v.y * v.y + (double)v.z * v.z + (double)v.w * v.w;
    }
  } else {
    for (long long q = threadIdx.x; q < n; q += blockDim.x) {
      const float v = __ldg(x + q);
      s += v;
      ss += (double)v * v;
    }
  }
  __shared__ double sh[2][32];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    s += __shfl_xor_sync(0xffffffffu, s, o);
    ss += __shfl_xor_sync(0xffffffffu, ss, o);
  }
  if ((threadIdx.x & 31) == 0) { sh[0][threadIdx.x >> 5] = s; sh[1][threadIdx.x >> 5] = ss; }
  __syncthreads();
  if (threadIdx.x < 32) {
    const int nw = blockDim.x >> 5;
    s = threadIdx.x < nw ? sh[0][threadIdx.x] : 0.0;
    ss = threadIdx.x < nw ? sh[1][threadIdx.x] : 0.0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      s += __shfl_xor_sync(0xffffffffu, s, o);
      ss += __shfl_xor_sync(0xffffffffu, ss, o);
    }
    if (threadIdx.x == 0) {
      const double mean = s / (double)n;
      double var = ss / (double)n - mean * mean;                // biased (unbiased=False, corr.py:47)
      if (var < 0.0) var = 0.0;
      stats[(size_t)e * 4 + head * 2 + 0] = (float)mean;
      stats[(size_t)e * 4 + head * 2 + 1] = sqrtf((float)var + eps);       // the divisor: sqrt(var + eps), fp32 like torch
    }
  }
}

// 32 consecutive pixels of one edge x all CH channels.  Thread t: pixel t & 31, channels (t >> 5) + 8 m.
__global__ void __launch_bounds__(kOhThreads)
offset_apply_kernel(const float* __restrict__ c0, const float* __restrict__ c1, const float* __restrict__ stats,
                    float* __restrict__ off0, float* __restrict__ off1, int CH, int H, int W, int tiles_per_edge) {
  extern __shared__ float sm[];                                  // [2][32][CH + 1]
  const int e = blockIdx.x / tiles_per_edge;
  const int p0 = (blockIdx.x - e * tiles_per_edge) * 32;
  const int P = H * W, Wh = W >> 1, Ph = (H >> 1) * Wh;
  const int lane = threadIdx.x & 31, grp = threadIdx.x >> 5;
  const float m0 = __ldg(stats + (size_t)e * 4 + 0), d0 = __ldg(stats + (size_t)e * 4 + 1);
  const float m1 = __ldg(stats + (size_t)e * 4 + 2), d1 = __ldg(stats + (size_t)e * 4 + 3);
  const int p = p0 + lane, y = p / W, x = p - y * W;
  const int ph = (y >> 1) * Wh + (x >> 1);                       // F.interpolate(..., (h, w)) nearest: source = floor(dst / 2)
  const int pitch = CH + 1;
  float* s0 = sm;
  float* s1 = sm + 32 * pitch;
  for (int c = grp; c < CH; c += kOhThreads / 32) {
    const float a = __ldg(c0 + ((size_t)e * CH + c) * P + p);
    const float b = __ldg(c1 + ((size_t)e * CH + c) * Ph + ph);
    const float o0 = __fmul_rn(tanhf(__fdiv_rn(__fsub_rn(a, m0), d0)), 4.0f);
    const float o1 = __fdiv_rn(__fadd_rn(__fmul_rn(tanhf(__fdiv_rn(__fsub_rn(b, m1), d1)), 4.0f), o0), 2.0f);
    s0[lane * pitch + c] = o0;
    s1[lane * pitch + c] = o1;
  }
  __syncthreads();
  // the 32 pixels' records are contiguous in the NHWC output: 32 * CH floats
  float* g0 = off0 + ((size_t)e * P + p0) * CH;
  float* g1 = off1 + ((size_t)e * P + p0) * CH;
  for (int q = threadIdx.x; q < 32 * CH; q += kOhThreads) {
    const int pl = q / CH, c = q - pl * CH;
    g0[q] = s0[pl * pitch + c];
    g1[q] = s1[pl * pitch + c];
  }
}

// ---- backward (lgu_offset_heads_backward) ------------------------------------------------------------------------
// One CTA per (edge, tile); a tile is hi-res rows 2yh, 2yh+1 x 32 columns = lo-res row yh x 16 columns, all CH channels,
// so the 4 hi-res copies of every c1 element it owns are in the CTA and each output element is written by one thread.
//   kApply = false : per-tile sums (Σgz0, Σgz0·z0, Σgz1, Σgz1·z1) in fp64 -> scratch[tile]
//   kApply = true  : the edge's sums in a fixed order -> means, then g_c0 / g_c1 (NCHW, coalesced along x)
// Both passes recompute z and t = tanh(z) with the forward's arithmetic and stage the channels-last upstream gradients
// of the tile's 64 hi-res pixels through shared memory: sA = G0 + G1/2 (what reaches t0), sG = G1.
constexpr int kOhbThreads = 256;

template <bool kApply>
__global__ void __launch_bounds__(kOhbThreads)
offset_heads_bwd_kernel(const float* __restrict__ c0, const float* __restrict__ c1, const float* __restrict__ stats,
                        const float* __restrict__ g_off0, const float* __restrict__ g_off1, double* __restrict__ scratch,
                        float* __restrict__ g_c0, float* __restrict__ g_c1, int CH, int H, int W, int tiles_per_edge) {
  extern __shared__ float sm[];                                  // [2][64][CH + 1], pixel = row * 32 + column
  __shared__ double red[4][kOhbThreads / 32];
  __shared__ float means[4];
  const int e = blockIdx.x / tiles_per_edge;
  const int tile = blockIdx.x - e * tiles_per_edge;
  const int tx = W >> 5, yh = tile / tx, x0 = (tile - yh * tx) * 32;
  const int P = H * W, Wh = W >> 1, Ph = (H >> 1) * Wh;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int pitch = CH + 1;
  float* sA = sm;
  float* sG = sm + 64 * pitch;
  const float m0 = __ldg(stats + (size_t)e * 4 + 0), d0 = __ldg(stats + (size_t)e * 4 + 1);
  const float m1 = __ldg(stats + (size_t)e * 4 + 2), d1 = __ldg(stats + (size_t)e * 4 + 3);

  if (kApply && warp == 0) {
    // the edge's tile sums, always added in the same order: bit-identical from run to run
    double acc[4] = {0.0, 0.0, 0.0, 0.0};
    for (int k = lane; k < tiles_per_edge; k += 32)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[j] += scratch[((size_t)e * tiles_per_edge + k) * 4 + j];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) acc[j] += __shfl_down_sync(0xffffffffu, acc[j], o);
    }
    if (lane == 0) {
      const double n = (double)CH * H * W;                      // both heads: means over the N0 hi-res elements
#pragma unroll
      for (int j = 0; j < 4; ++j) means[j] = (float)(acc[j] / n);
    }
  }

  // warp -> pixel, lane -> channels lane + 32 k (CH <= 128): one record of CH contiguous floats per warp and pixel
#pragma unroll 2
  for (int px = warp; px < 64; px += kOhbThreads / 32) {
    const size_t base = ((size_t)e * P + (size_t)(2 * yh + (px >> 5)) * W + x0 + (px & 31)) * CH;
    float a[4], b[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int c = lane + 32 * k;
      a[k] = (g_off0 && c < CH) ? __ldg(g_off0 + base + c) : 0.0f;
      b[k] = (g_off1 && c < CH) ? __ldg(g_off1 + base + c) : 0.0f;
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int c = lane + 32 * k;
      if (c < CH) {
        sA[px * pitch + c] = __fmaf_rn(b[k], 0.5f, a[k]);
        sG[px * pitch + c] = b[k];
      }
    }
  }
  __syncthreads();
  float M0 = 0.f, Q0 = 0.f, M1 = 0.f, Q1 = 0.f;
  if (kApply) { M0 = means[0]; Q0 = means[1]; M1 = means[2]; Q1 = means[3]; }
  double s0 = 0.0, s0z = 0.0, s1 = 0.0, s1z = 0.0;

  // head 0, hi-res: warp -> (row, channel), lane -> column
#pragma unroll 4
  for (int j = warp; j < 2 * CH; j += kOhbThreads / 32) {
    const int r = j & 1, c = j >> 1;
    const size_t gi = ((size_t)e * CH + c) * P + (size_t)(2 * yh + r) * W + x0 + lane;
    const float z = __fdiv_rn(__fsub_rn(__ldg(c0 + gi), m0), d0);
    const float t = tanhf(z);
    const float gz = 4.0f * sA[(r * 32 + lane) * pitch + c] * (1.0f - t * t);
    if (kApply) {
      g_c0[gi] = (gz - M0 - z * Q0) / d0;
    } else {
      s0 += gz;
      s0z += (double)gz * z;
    }
  }
  // head 1, lo-res: 16 threads -> the tile's 16 columns of one channel; t1 is the same for the 4 copies of an element
#pragma unroll 2
  for (int c = threadIdx.x >> 4; c < CH; c += kOhbThreads / 16) {
    const int xl = threadIdx.x & 15, p = 2 * xl;
    const size_t gi = ((size_t)e * CH + c) * Ph + (size_t)yh * Wh + (x0 >> 1) + xl;
    const float z = __fdiv_rn(__fsub_rn(__ldg(c1 + gi), m1), d1);
    const float t = tanhf(z);
    const float g = (sG[p * pitch + c] + sG[(p + 1) * pitch + c]) + (sG[(32 + p) * pitch + c] + sG[(33 + p) * pitch + c]);
    const float S = 2.0f * g * (1.0f - t * t);
    if (kApply) {
      g_c1[gi] = (S - 4.0f * M1 - 4.0f * z * Q1) / d1;
    } else {
      s1 += S;
      s1z += (double)S * z;
    }
  }
  if (kApply) return;

  double v[4] = {s0, s0z, s1, s1z};
#pragma unroll
  for (int j = 0; j < 4; ++j) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v[j] += __shfl_down_sync(0xffffffffu, v[j], o);
    if (lane == 0) red[j][warp] = v[j];
  }
  __syncthreads();
  if (threadIdx.x < 4) {
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < kOhbThreads / 32; ++w) s += red[threadIdx.x][w];
    scratch[(size_t)blockIdx.x * 4 + threadIdx.x] = s;
  }
}

}  // namespace lgu

extern "C" int lgu_offset_heads(const float* c0, const float* c1, float* off0, float* off1, float* stats, int E, int CH, int H,
                                int W, float eps, void* stream) {
  using namespace lgu;
  if (E == 0) return LGU_OK;
  LGU_REQUIRE(c0 && c1 && off0 && off1 && stats, "lgu_offset_heads: null pointer");
  LGU_REQUIRE(E > 0 && CH > 0 && CH <= 128 && H > 0 && W > 0 && (W % 32) == 0 && (H % 2) == 0,
              "lgu_offset_heads: bad sizes E=%d CH=%d H=%d W=%d (needs CH <= 128, W %% 32 == 0, H even)", E, CH, H, W);
  const long long n0 = (long long)CH * H * W, n1 = (long long)CH * (H / 2) * (W / 2);
  offset_stats_kernel<<<2 * E, 1024, 0, (cudaStream_t)stream>>>(c0, c1, stats, n0, n1, eps);
  if (int rc = check_launch("lgu_offset_heads (stats)")) return rc;
  const int tiles = H * W / 32;
  const size_t smem = (size_t)2 * 32 * (CH + 1) * sizeof(float);
  offset_apply_kernel<<<(unsigned)((long long)E * tiles), kOhThreads, smem, (cudaStream_t)stream>>>(c0, c1, stats, off0, off1,
                                                                                                  CH, H, W, tiles);
  return check_launch("lgu_offset_heads");
}

extern "C" int lgu_offset_heads_backward(const float* c0, const float* c1, const float* stats, const float* g_off0,
                                         const float* g_off1, float* g_c0, float* g_c1, double* scratch, int E, int CH,
                                         int H, int W, void* stream) {
  using namespace lgu;
  if (E == 0) return LGU_OK;
  LGU_REQUIRE(c0, "lgu_offset_heads_backward: c0 is NULL");
  LGU_REQUIRE(c1, "lgu_offset_heads_backward: c1 is NULL");
  LGU_REQUIRE(stats, "lgu_offset_heads_backward: stats is NULL");
  LGU_REQUIRE(g_c0, "lgu_offset_heads_backward: g_c0 is NULL");
  LGU_REQUIRE(g_c1, "lgu_offset_heads_backward: g_c1 is NULL");
  LGU_REQUIRE(scratch, "lgu_offset_heads_backward: scratch is NULL");
  LGU_REQUIRE((reinterpret_cast<uintptr_t>(scratch) & 7) == 0, "lgu_offset_heads_backward: scratch is not 8-byte aligned");
  LGU_REQUIRE(E > 0, "lgu_offset_heads_backward: bad size E=%d", E);
  LGU_REQUIRE(CH > 0 && CH <= 128, "lgu_offset_heads_backward: bad size CH=%d (needs 0 < CH <= 128)", CH);
  LGU_REQUIRE(H > 0 && (H % 2) == 0, "lgu_offset_heads_backward: bad size H=%d (needs H even)", H);
  LGU_REQUIRE(W > 0 && (W % 32) == 0, "lgu_offset_heads_backward: bad size W=%d (needs W %% 32 == 0)", W);
  const int tiles = (H / 2) * (W / 32);
  const int smem = 2 * 64 * (CH + 1) * (int)sizeof(float);
  if (int rc = optin_smem((const void*)offset_heads_bwd_kernel<false>, smem, "lgu_offset_heads_backward")) return rc;
  if (int rc = optin_smem((const void*)offset_heads_bwd_kernel<true>, smem, "lgu_offset_heads_backward")) return rc;
  const unsigned grid = (unsigned)((long long)E * tiles);
  offset_heads_bwd_kernel<false><<<grid, kOhbThreads, smem, (cudaStream_t)stream>>>(c0, c1, stats, g_off0, g_off1, scratch,
                                                                                    g_c0, g_c1, CH, H, W, tiles);
  if (int rc = check_launch("lgu_offset_heads_backward (sums)")) return rc;
  offset_heads_bwd_kernel<true><<<grid, kOhbThreads, smem, (cudaStream_t)stream>>>(c0, c1, stats, g_off0, g_off1, scratch,
                                                                                   g_c0, g_c1, CH, H, W, tiles);
  return check_launch("lgu_offset_heads_backward");
}

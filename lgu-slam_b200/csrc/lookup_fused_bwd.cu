// lookup_fused_bwd.cu -- backward of CorrBlock.__call__'s data path in ONE launch (sm_100a).
//
// Replaces what autograd runs for /root/reference/droid_slam/modules/corr.py:88-109 in training:
//   4 x defCorr_index_backward (defCorrSample_kernel.cu:93-162; each zero-fills and RMWs a dense volume_grad and
//   writes a dense offset_grad, also for the detached zero offsets of levels 2-3)
//   + (offset[1] * mask)^T + sigmoid^T + var^T (torch)  + corr_index_backward (corrSample_kernel.cu:84-136; one
//   more dense level-1 volume_grad that autograd then adds to the first)
// by one kernel that writes every pyramid level's dense gradient slice exactly once, with the mask path already
// accumulated into level 1, and offset gradients only for the two levels that have offsets.
//
// Per source pixel (one warp, lane = tap):
//   * TMA box loads stage the level-0 / level-1 footprints (needed for the offset gradients and to recompute the
//     9 mask taps), 2-slot mbarrier ring as in the forward;
//   * the upstream gradient tile [196 x 32 pixels] is loaded with 128-byte rows and transposed through smem;
//   * corner contributions are accumulated into per-warp BOX-shaped shared accumulators (20x16, 20x16, 12x8, 12x8
//     floats: the same footprint the forward gathers from) -- shared-memory reductions for the deformable levels
//     (taps may collide), plain read-modify-write per corner phase for the zero-offset levels and the mask taps;
//   * each level's dense H2 x W2 slice is then streamed out once with 16-byte st.cs: zeros outside the box, the
//     accumulator inside (re-zeroed on the fly).  Taps outside the box (|offset| >= 4) are added with global
//     atomics after the slice has been written.
// Gradient algebra (what autograd computes for the reference graph):
//   gO_l      = defCorr offset gradient of level l (defCorrSample_kernel.cu:156-157), l = 0, 1
//   g_off1_in = (gO_1 + g_off1_out) * m                       (offset[1]_out = offset[1]_in * m, corr.py:99)
//   g_m       = sum_taps (gO_1 + g_off1_out) . offset[1]_in   = sum(...) . offset[1]_out / m
//   g_var     = g_m * m * (1 - m)                             (sigmoid, corr.py:97)
//   g_v[k]    = g_var * 2 (v[k] - mean) / 8                   (unbiased 9-tap variance, corr.py:96)
//   gV_1     += corr_index_backward(g_v)                      (corrSample_kernel.cu:84-136)
#include "fused_common.cuh"
#include "gauss_window.cuh"

namespace lgu {

namespace flb {
using namespace fl;
constexpr int kInSlotFloats = 2 * kBW01 * kBH01;                 // level-0 + level-1 input boxes: 640 floats
constexpr int kInSlotBytes = kInSlotFloats * 4;                  // 2560 B
constexpr int kAccFloats = kSlotFloats;                          // 832 floats: acc0 | acc1 | acc2 | acc3
constexpr int kWarpFloats = kSlots * kInSlotFloats + kAccFloats; // 2112 floats = 8448 B
constexpr int kSmemWarp = kWarps * kWarpFloats * 4;              // 67,584 B
constexpr int kGWarpFloats = CH * kPixPerWarp;                   // per-warp upstream-gradient rows: 196 x 4 pixels
constexpr int kGWarpStride = (kGWarpFloats * 4 + 127) / 128 * 32;    // 800 floats: the TMA destination is 128-byte aligned
constexpr int kSmemG = kWarps * kGWarpStride * 4;                // 25,600 B
constexpr int kPairBytes = 2 * TAPS * 8;                         // one level's offset records of a PIXEL PAIR: 784 B
constexpr int kSmemOffs = kWarps * 2 * kPairBytes;               // 12,544 B (levels 0 and 1, single-buffered)
constexpr int kSmallBytes = 64;                                  // per warp and tile parity: coords[4] float2 | mask[4] | scale[4]
constexpr int kSmemSmall = kWarps * 2 * kSmallBytes;             // 1,024 B
constexpr int kBarsPerWarp = kSlots + 4;                         // box ring[2], offset pair, upstream strip, small[2]
constexpr int kSmemBars = kWarps * kBarsPerWarp * 8;
using fl::kZeroBytes;                                            // CTA-shared zero source of the bulk zero-fill
constexpr int kOffG = kSmemWarp;
constexpr int kOffOffs = kOffG + kSmemG;
constexpr int kOffSmall = kOffOffs + kSmemOffs;
constexpr int kOffBars = kOffSmall + kSmemSmall;
constexpr int kOffZero = kOffBars + kSmemBars;
constexpr int kSmemBytes = kOffZero + kZeroBytes;                // 115,456 B: two CTAs per SM
static_assert(2 * (kSmemBytes + 1024) <= 228 * 1024, "two CTAs per SM");
}  // namespace flb

struct FusedLookupBwdParams {
  const float* lvl[2];       // level 0 / 1 volumes (slow path only; the fast path reads the TMA boxes)
  const float* coords;       // [E,P,2]
  const float* off0;         // [E,P,49,2]  as used by the forward (centre tap reads as 0)
  const float* off1;         // [E,P,49,2]  post-mask offsets (offset[1]_out of the forward)
  const float* mask;         // [E,P]       m of the forward
  const float* off1_scale;   // [E,P] or null: off1 holds PRISTINE offsets and offset[1]_out = off1 * off1_scale (the forward's
                             // cumulative-mask form, lgu_corr_lookup_fused_cum: off1_scale = cum_mask after that call)
  const float* g_out;        // [E,196,P]   upstream gradient of corr
  const float* g_off1_out;   // [E,P,49,2]  upstream gradient of offset[1]_out (later calls), or null
  float* gv[4];              // dense volume gradients [E,P,H2,W2]
  float* g_off0;             // [E,P,49,2]
  float* g_off1;             // [E,P,49,2]  gradient of offset[1]_in
  const float* win_means;    // [E,P,2] or null: centres of the Gaussian head's 9 x 9 windows (gaussianMask_cuda.py:77-86)
  float* gwin;               // [E,P,81] or null: the level-0 gradient INCLUDING the pooled levels' share, inside that window
  const float* win_covs;     // GAUSS kernels: [E,P,2], [E,P] -- the Gaussian head's covariances and denominators, and the
  const float* win_den;      //   gradients of (means, covs, den) this call contributes through the build's Gaussian residual
  float* g_means;            // [E,P,2]
  float* g_covs;             // [E,P,2]
  float* g_den;              // [E,P]
  int P, tiles_per_edge, num_tiles;
  int H2[4], W2[4];
};

// Scatter one corner phase of all lanes into a box accumulator.  ATOMIC: lanes may collide (learned offsets).
template <bool ATOMIC>
__device__ __forceinline__ void acc_add(float* acc, bool on, unsigned idx, float val) {
  if (on) {
    if (ATOMIC) atomicAdd(acc + idx, val);
    else acc[idx] += val;
  }
  if (!ATOMIC) __syncwarp();
}

// Geometry of one tap for the backward: gates, box index, bilinear fractions.
struct BTap {
  float dx, dy;
  int x1, y1;
  unsigned idx;
  bool gate, xo, yo, inbox;
};
template <int BW, int BH>
__device__ __forceinline__ void btap_setup(BTap& t, int xb, int yb, int fx, int fy, int i, int j, int r, int H2, int W2) {
  t.x1 = tap_coord(fx, r, i);
  t.y1 = tap_coord(fy, r, j);
  const int x2 = wrap_inc(t.x1), y2 = wrap_inc(t.y1);
  t.gate = ((unsigned)t.x1 < (unsigned)W2) && ((unsigned)t.y1 < (unsigned)H2);
  t.xo = t.gate && ((unsigned)x2 < (unsigned)W2);
  t.yo = t.gate && ((unsigned)y2 < (unsigned)H2);
  const unsigned rx = (unsigned)t.x1 - (unsigned)xb, ry = (unsigned)t.y1 - (unsigned)yb;
  t.inbox = rx < (unsigned)(BW - 1) && ry < (unsigned)(BH - 1);
  t.idx = t.inbox ? ry * BW + rx : 0u;
}
// Accumulate the <= 4 corner contributions of a tap (weights as in defCorrSample_kernel.cu:145-154 /
// corrSample_kernel.cu:118-131).  Footprints outside the box are deferred (returned true) to the global slow path.
template <int BW, bool ATOMIC>
__device__ __forceinline__ void btap_scatter(float* acc, const BTap& t, bool active, float g) {
  const float omdx = __fsub_rn(1.0f, t.dx), omdy = __fsub_rn(1.0f, t.dy);
  const bool on = active && t.gate && t.inbox;
  acc_add<ATOMIC>(acc, on, t.idx, __fmul_rn(__fmul_rn(omdy, omdx), g));
  acc_add<ATOMIC>(acc, on && t.xo, t.idx + 1, __fmul_rn(__fmul_rn(omdy, t.dx), g));
  acc_add<ATOMIC>(acc, on && t.yo, t.idx + BW, __fmul_rn(__fmul_rn(t.dy, omdx), g));
  acc_add<ATOMIC>(acc, on && t.xo && t.yo, t.idx + BW + 1, __fmul_rn(__fmul_rn(t.dy, t.dx), g));
}
__device__ __forceinline__ void btap_scatter_global(float* G, const BTap& t, bool active, float g, int W2) {
  if (active && t.gate && !t.inbox) {
    const float omdx = __fsub_rn(1.0f, t.dx), omdy = __fsub_rn(1.0f, t.dy);
    float* p = G + (size_t)t.y1 * W2 + t.x1;
    atomicAdd(p, __fmul_rn(__fmul_rn(omdy, omdx), g));
    if (t.xo) atomicAdd(p + 1, __fmul_rn(__fmul_rn(omdy, t.dx), g));
    if (t.yo) atomicAdd(p + W2, __fmul_rn(__fmul_rn(t.dy, omdx), g));
    if (t.xo && t.yo) atomicAdd(p + W2 + 1, __fmul_rn(__fmul_rn(t.dy, t.dx), g));
  }
}
// Fixed-point variant of the deformable scatter.  atomicAdd(float) on shared memory is a compare-and-swap loop per
// corner (ATOMS.CAST.SPIN: 16 dependent loops per pixel and lane, 22 % of the kernel); integer adds are ONE native
// ATOMS.ADD each, need no retry and are associative -- the accumulated gradient no longer depends on the order in
// which colliding taps arrive.  The contributions of a pixel are scaled by a power of two chosen from the largest
// upstream gradient magnitude of the pixel (|w g| 2^s < 2^23, so even 196 colliding corners cannot overflow) and rounded
// to nearest: absolute error <= 2^-24 of that magnitude per contribution, below fp32's own rounding of the large terms.
template <int BW>
__device__ __forceinline__ void btap_scatter_fxp(int* acc, const BTap& t, bool active, float g, float scale) {
  const float omdx = __fsub_rn(1.0f, t.dx), omdy = __fsub_rn(1.0f, t.dy);
  const bool on = active && t.gate && t.inbox;
  const float gs = __fmul_rn(g, scale);                          // exact (power of two), |gs| < 2^23
  if (on) {
    atomicAdd(acc + t.idx, __float2int_rn(__fmul_rn(__fmul_rn(omdy, omdx), gs)));
    if (t.xo) atomicAdd(acc + t.idx + 1, __float2int_rn(__fmul_rn(__fmul_rn(omdy, t.dx), gs)));
    if (t.yo) atomicAdd(acc + t.idx + BW, __float2int_rn(__fmul_rn(__fmul_rn(t.dy, omdx), gs)));
    if (t.xo && t.yo) atomicAdd(acc + t.idx + BW + 1, __float2int_rn(__fmul_rn(__fmul_rn(t.dy, t.dx), gs)));
  }
}

// Offset gradient of a tap (defCorrSample_kernel.cu:156-157, the reference's SASS operation order).
__device__ __forceinline__ float2 offset_grad(float q11, float q21, float q12, float q22, float dx, float dy, float g) {
  const float omdx = __fsub_rn(1.0f, dx), omdy = __fsub_rn(1.0f, dy);
  float ty = __fmaf_rn(-q11, omdx, -__fmul_rn(dx, q21));
  ty = __fmaf_rn(omdx, q12, ty);
  ty = __fmaf_rn(dx, q22, ty);
  float tx = __fmaf_rn(omdy, q21, -__fmul_rn(q11, omdy));
  tx = __fmaf_rn(-dy, q12, tx);
  tx = __fmaf_rn(dy, q22, tx);
  return make_float2(__fmul_rn(tx, g), __fmul_rn(ty, g));
}

// Stream one level's dense gradient slice: zeros outside the accumulator box, the accumulator (then re-zeroed) inside.
// Fast path (W2/4 divides 32, i.e. W2 in {8,16,32,64,128}): a lane owns one float4 column of the slice and walks
// rows with a fixed stride, so the column test and the accumulator column are loop invariants -- no divisions.
// (The first version divided by W2/4 per float4: ncu showed 2700 instructions per pixel, 40 % of them here.)
template <int BW, int BH>
__device__ __forceinline__ void write_slice(float* __restrict__ G, float* acc, int xb, int yb, int H2, int W2, int lane) {
  const int W4 = W2 >> 2;
  float4* G4 = reinterpret_cast<float4*>(G);
  const float4 z = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
  if (W4 <= 32 && (32 % W4) == 0) {
    const int rpi = 32 / W4;                                   // rows per warp iteration
    const int ly = lane / W4, lx = lane - ly * W4;             // W4 is a power of two here: shifts
    const unsigned rx = (unsigned)((lx << 2) - xb);
    const bool col_in = rx < (unsigned)BW;                     // xb % 4 == 0: the float4 lies entirely inside
    float* acol = acc + rx;
    float4* g = G4 + ly * W4 + lx;
    const int gstep = rpi * W4;                                // == 32
    for (int y = ly; y < H2; y += rpi, g += gstep) {
      const unsigned ry = (unsigned)(y - yb);
      float4 v = z;
      if (col_in && ry < (unsigned)BH) {
        float4* a = reinterpret_cast<float4*>(acol + ry * BW);
        v = *a;
        *a = z;
      }
      __stcs(g, v);
    }
  } else {
    const int n4 = H2 * W4;
    for (int q4 = lane; q4 < n4; q4 += 32) {
      const int y = q4 / W4, x = (q4 - y * W4) << 2;
      const unsigned ry = (unsigned)(y - yb), rx = (unsigned)(x - xb);
      float4 v = z;
      if (ry < (unsigned)BH && rx < (unsigned)BW) {
        float4* a = reinterpret_cast<float4*>(acc + ry * BW + rx);
        v = *a;
        *a = z;
      }
      __stcs(G4 + q4, v);
    }
  }
}

// Dense mode, levels 0 and 1: the rows of the slice that do not intersect the accumulator box are pure zeros --
// 8 of the 12 KB of a level-0 slice.  Those contiguous ranges leave through the TMA engine (cp.async.bulk
// shared -> global from a CTA-wide zero buffer, one elected lane, <= 8 KB per copy) instead of 16-byte st.cs from
// every lane; only the band of box rows is streamed by the LSU (zeros left / right of the box, the accumulator inside).
template <int BW, int BH>
__device__ __forceinline__ void write_slice_bulk(float* __restrict__ G, float* acc, int xb, int yb, int H2, int W2, int lane,
                                                 const void* zero_smem) {
  const int W4 = W2 >> 2;                                        // callers guarantee 32 % W4 == 0 (W2 in {32, 64, 128})
  int y0 = max(yb, 0), y1 = min(yb + BH, H2);                    // band of slice rows that meet the box
  if (y1 <= y0) y0 = y1 = H2;                                    // box entirely outside: the whole slice is zero
  if (lane == 0) {
    bulk_zero(G, y0 * W2 * 4, zero_smem);
    bulk_zero(G + (size_t)y1 * W2, (H2 - y1) * W2 * 4, zero_smem);
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
  }
  float4* G4 = reinterpret_cast<float4*>(G);
  const float4 z = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
  const int rpi = 32 / W4;
  const int ly = lane / W4, lx = lane - ly * W4;
  const unsigned rx = (unsigned)((lx << 2) - xb);
  const bool col_in = rx < (unsigned)BW;
  float* acol = acc + rx;
  for (int y = y0 + ly; y < y1; y += rpi) {
    const unsigned ry = (unsigned)(y - yb);                      // < BH inside the band
    float4 v = z;
    if (col_in) {
      float4* a = reinterpret_cast<float4*>(acol + ry * BW);
      v = *a;
      *a = z;
    }
    __stcs(G4 + y * W4 + lx, v);
  }
}

// Accumulate mode (training, several lookups per pyramid): the gradient buffers persist across launches, so only the
// accumulator box is touched -- one 16-byte reduction (RED.ADD.F32x4, resolved in L2, nothing returns to the SM) per
// non-zero box cell that lies inside the slice; the accumulator is re-zeroed on the fly.  The slice is private to this
// warp within a launch, launches on one stream are ordered, so the result is the sequential sum of the calls.
template <int BW, int BH>
__device__ __forceinline__ void add_box(float* __restrict__ G, float* acc, int xb, int yb, int H2, int W2, int lane) {
  constexpr int C4 = BW / 4, N4 = C4 * BH;
  const float4 z = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
#pragma unroll
  for (int c0 = 0; c0 < N4; c0 += 32) {
    const int c = c0 + lane;
    if (c < N4) {
      const int ry = c / C4, rx = (c - ry * C4) << 2;
      float4* a = reinterpret_cast<float4*>(acc + ry * BW + rx);
      const float4 v = *a;
      *a = z;
      const int y = yb + ry, x = xb + rx;                        // xb % 4 == 0 and W2 % 4 == 0: all four lanes in or out
      const bool nz = (v.x != 0.0f) || (v.y != 0.0f) || (v.z != 0.0f) || (v.w != 0.0f);
      if (nz && (unsigned)y < (unsigned)H2 && (unsigned)x < (unsigned)W2)
        atomicAdd(reinterpret_cast<float4*>(G + (size_t)y * W2 + x), v);
    }
  }
}

// The Gaussian head's backward (lgu_build_backward_gauss) needs the gradient of the level-0 volume only inside the
// 9 x 9 window around each pixel's mean -- with avg_pool2d's transpose folded in: g0 + g1/4 + g2/16 + g3/64 of the
// cells above the tap.  Reading those four windows back from the dense gradients costs a 64-byte DRAM granule per
// 36-byte window row (ncu: 513 MB per launch for 124 MB of algorithmic bytes); here the four boxes are still in shared
// memory, so the merged window leaves as one contiguous 324-byte record per pixel.  Same order of additions as the
// from-levels kernel (gaussian.cu), so both give the same bits.  GLOBAL: rare pixels with out-of-box taps re-read the
// finished slices instead (their global atomics are not in the boxes).
constexpr int kWinR = 4, kWinD = 2 * kWinR + 1, kWinTaps = kWinD * kWinD;
template <bool GLOBAL>
__device__ __forceinline__ void emit_window(float* __restrict__ gw, float (&out)[3], int wx0, int wy0, const float* acc,
                                            const int* xb, const int* yb, float* const* G, const int* H2, const int* W2,
                                            int lane) {
  using namespace fl;
  static_assert((kWinTaps + 31) / 32 == 3, "three passes");
#pragma unroll
  for (int ps = 0; ps < 3; ++ps) {
    const int t = ps * 32 + lane;
    out[ps] = 0.0f;
    if (t < kWinTaps) {
      const int wy = t / kWinD, wx = t - wy * kWinD;
      const int x = tap_coord(wx0, 0, wx), y = tap_coord(wy0, 0, wy);
      float gg = 0.0f;
      if ((unsigned)x < (unsigned)W2[0] && (unsigned)y < (unsigned)H2[0]) {
        float part[4];
#pragma unroll
        for (int l = 0; l < 4; ++l) {
          const int xl = x >> l, yl = y >> l;
          if (GLOBAL) {
            part[l] = ((unsigned)xl < (unsigned)W2[l] && (unsigned)yl < (unsigned)H2[l]) ? __ldcg(G[l] + (size_t)yl * W2[l] + xl) : 0.0f;
          } else {
            const int BW = l < 2 ? kBW01 : kBW23, BH = l < 2 ? kBH01 : kBH23;
            const int off = l == 0 ? kOff0 : l == 1 ? kOff1 : l == 2 ? kOff2 : kOff3;
            const unsigned rx = (unsigned)(xl - xb[l]), ry = (unsigned)(yl - yb[l]);
            part[l] = (rx < (unsigned)BW && ry < (unsigned)BH) ? acc[off + ry * BW + rx] : 0.0f;
          }
        }
        gg = part[0];
        gg = __fadd_rn(gg, __fmul_rn(part[1], 0.25f));
        gg = __fadd_rn(gg, __fmul_rn(part[2], 0.0625f));
        gg = __fadd_rn(gg, __fmul_rn(part[3], 0.015625f));
      }
      out[ps] = gg;
      if (gw != nullptr) __stcs(gw + t, gg);
    }
  }
}

// Round 2: PERSISTENT CTAs (two per SM) walk the tiles, and nothing a pixel needs is fetched by LDG inside the pixel loop
// (ncu's source view of the per-tile version: 28 % of all samples were long-scoreboard stalls -- the first use of the
// prefetched offset records, the cp.async loop of the upstream-gradient strip, the coords load of every CTA's prologue --
// and 5 % sat at the CTA-end barrier).  Per tile and warp: the 196 x 4 upstream-gradient strip is ONE TMA box, the offset
// records travel as pixel PAIRS by cp.async.bulk (a pair is 16-byte aligned; the single pair buffer is refilled as soon
// as the second pixel of a pair has read its records), coords / mask / cumulative-mask scale arrive as 64 bytes per tile
// one tile ahead, and the box ring keeps prefetching across tile boundaries.  The strip of the next tile is requested as
// soon as the last pixel of the current one has moved its eight gradient values to registers.
// GAUSS (dense mode): the Gaussian head's backward of the build (gaussianMask_cuda.py:77-86 through corr.py:83-86) is
// finished HERE: the merged window gradient is in registers (emit_window), the 81 window values of level 0 are fetched at
// the top of the pixel, and gauss_window_grads -- the arithmetic of lgu_build_backward_gauss, shared code -- gives the
// pixel's (means, covs, den) gradients.  The separate kernel was bound by its window gathers from the dense gradients.
template <bool ACC, bool BULK, bool GAUSS = false>
__global__ void __launch_bounds__(fl::kThreads, 2)
lookup_fused_bwd_kernel(const __grid_constant__ FusedMaps maps, const FusedLookupBwdParams prm) {
  using namespace flb;
  extern __shared__ __align__(1024) uint8_t smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* wmem = reinterpret_cast<float*>(smem) + warp * kWarpFloats;
  float* inbox = wmem;                                           // [slot][lvl0 | lvl1]
  float* acc = wmem + kSlots * kInSlotFloats;                    // acc0 | acc1 | acc2 | acc3 (offsets kOff0..3)
  float* s_g = reinterpret_cast<float*>(smem + kOffG) + warp * kGWarpStride;       // this warp's [CH][4 pixels]
  const uint32_t smem0 = fl_smem_u32(smem);
  const uint32_t offs_base = smem0 + kOffOffs + warp * 2 * kPairBytes;              // [level 0 | level 1][2 pixels][49] float2
  const uint32_t small_base = smem0 + kOffSmall + warp * 2 * kSmallBytes;
  const uint32_t bar_base = smem0 + kOffBars + warp * kBarsPerWarp * 8;
  const uint32_t bar_off = bar_base + kSlots * 8, bar_strip = bar_base + (kSlots + 1) * 8, bar_small = bar_base + (kSlots + 2) * 8;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kOffBars) + warp * kBarsPerWarp;
  uint8_t* zero_smem = smem + kOffZero;
  if (BULK && !ACC) {
    for (int q = threadIdx.x; q < kZeroBytes / 16; q += kThreads)
      reinterpret_cast<float4*>(zero_smem)[q] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();
  }
  const int P = prm.P;
  if (lane == 0) {
#pragma unroll
    for (int q = 0; q < kBarsPerWarp; ++q) fl_mbar_init(bars + q, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  for (int q = lane; q < kAccFloats; q += 32) acc[q] = 0.0f;
  __syncwarp();

  auto bulk_g2s = [&](uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src),
                 "r"(bytes), "r"(bar)
                 : "memory");
  };
  auto expect = [&](uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
  };
  auto wait = [&](uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "FLB_WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra FLB_DONE_%=;\n\t"
        "bra FLB_WAIT_%=;\n\t"
        "FLB_DONE_%=:\n\t}" ::"r"(bar),
        "r"(parity)
        : "memory");
  };
  auto tile_edge = [&](int tile, int& n, int& pw) {
    n = tile / prm.tiles_per_edge;
    pw = (tile - n * prm.tiles_per_edge) * kTile + warp * kPixPerWarp;
  };
  // lane 0 only: per-tile inputs
  auto fetch_small = [&](int n, int pw, int par) {
    const uint32_t dst = small_base + par * kSmallBytes, bar = bar_small + par * 8;
    expect(bar, prm.off1_scale != nullptr ? 64u : 48u);
    bulk_g2s(dst, prm.coords + ((size_t)n * P + pw) * 2, 32, bar);
    bulk_g2s(dst + 32, prm.mask + (size_t)n * P + pw, 16, bar);
    if (prm.off1_scale != nullptr) bulk_g2s(dst + 48, prm.off1_scale + (size_t)n * P + pw, 16, bar);
  };
  auto fetch_pair = [&](int n, int pfirst) {                    // offset records of pixels pfirst, pfirst + 1 (pfirst even)
    const size_t at = ((size_t)n * P + pfirst) * TAPS * 2;
    expect(bar_off, 2u * kPairBytes);
    bulk_g2s(offs_base, prm.off0 + at, kPairBytes, bar_off);
    bulk_g2s(offs_base + kPairBytes, prm.off1 + at, kPairBytes, bar_off);
  };
  auto fetch_strip = [&](int n, int pw) {                       // g_out[n, 0..195, pw..pw+3] -> s_g, one TMA box
    expect(bar_strip, (uint32_t)(kGWarpFloats * 4));
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
            fl_smem_u32(s_g)),
        "l"(&maps.m[2]), "r"(bar_strip), "r"(pw), "r"(n * CH)
        : "memory");
  };
  auto issue = [&](int slot, int pix, float cx, float cy) {     // lane 0 only: the two input boxes of one pixel
    float* dst = inbox + slot * kInSlotFloats;
    fl_mbar_expect_tx(bars + slot, kInSlotBytes);
    float sx = cx, sy = cy;
#pragma unroll
    for (int l = 0; l < 2; ++l) {
      const int xb = box_origin_x(floor_to_int(sx), 7, prm.W2[l]), yb = box_origin_y(floor_to_int(sy), 7, prm.H2[l]);
      fl_tma_box(dst + l * kBW01 * kBH01, &maps.m[l], bars + slot, xb, yb, pix);
      sx = __fmul_rn(sx, 0.5f);
      sy = __fmul_rn(sy, 0.5f);
    }
  };
  auto lds64 = [&](uint32_t addr) {
    float2 v;
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(addr) : "memory");
    return v;
  };
  auto lds32 = [&](uint32_t addr) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr) : "memory");
    return v;
  };

  const int t0 = lane, t1 = lane + 32;
  const int i0 = t0 / RD, j0 = t0 - i0 * RD;
  const int t1c = min(t1, TAPS - 1);
  const int i1 = t1c / RD, j1 = t1c - i1 * RD;
  const bool has1 = t1 < TAPS;
  constexpr int CENTER = R * RD + R;
  const int mi = min(lane, 8) / 3, mj = min(lane, 8) - mi * 3;

  // ---- prologue of the first tile
  int tile = blockIdx.x;
  if (tile >= prm.num_tiles) return;
  int n, pw;
  tile_edge(tile, n, pw);
  if (lane == 0) {
    fetch_small(n, pw, 0);
    fetch_strip(n, pw);
    fetch_pair(n, pw);
  }
  wait(bar_small, 0);
  {
    const float2 c0 = lds64(small_base + (lane & 3) * 8);
    const float c0x = __shfl_sync(0xffffffffu, c0.x, 0), c0y = __shfl_sync(0xffffffffu, c0.y, 0);
    const float c1x = __shfl_sync(0xffffffffu, c0.x, 1), c1y = __shfl_sync(0xffffffffu, c0.y, 1);
    if (lane == 0) {
      issue(0, n * P + pw, c0x, c0y);
      issue(1, n * P + pw + 1, c1x, c1y);
    }
  }
  // upstream gradient on offset[1]_out (later calls of a training clip): prefetched one pixel ahead by LDG when present
  float2 u0 = make_float2(0.0f, 0.0f), u1 = u0;
  auto load_upstream = [&](size_t pix) {
    if (prm.g_off1_out != nullptr) {
      const float2* U = reinterpret_cast<const float2*>(prm.g_off1_out) + pix * TAPS;
      u0 = U[t0]; u1 = U[t1c];
    }
  };
  load_upstream((size_t)n * P + pw);

#pragma unroll 1
  for (int it = 0; tile < prm.num_tiles; ++it, tile += gridDim.x) {
  const int par = it & 1;
  const int ntile = tile + gridDim.x;
  const bool has_next = ntile < prm.num_tiles;
  int nn = 0, npw = 0;
  if (has_next) {
    tile_edge(ntile, nn, npw);
    if (lane == 0) fetch_small(nn, npw, par ^ 1);
  }
  const uint32_t small = small_base + par * kSmallBytes;
  wait(bar_strip, par);                                         // this tile's upstream-gradient strip
  const float2 cmine = lds64(small + (lane & 3) * 8);           // lane q (< 4) holds pixel q's coords
  float2 wmean = make_float2(0.0f, 0.0f), wcov = make_float2(1.0f, 1.0f);   // lane q (< 4): pixel q's Gaussian window
  float wden = 1.0f;
  const bool want_win = !ACC && (GAUSS || prm.gwin != nullptr);
  if (want_win) wmean = __ldg(reinterpret_cast<const float2*>(prm.win_means) + (size_t)n * P + pw + (lane & 3));
  if (GAUSS) {
    wcov = __ldg(reinterpret_cast<const float2*>(prm.win_covs) + (size_t)n * P + pw + (lane & 3));
    wden = __ldg(prm.win_den + (size_t)n * P + pw + (lane & 3));
  }

#pragma unroll 1
  for (int k = 0; k < kPixPerWarp; ++k) {
    const int slot = k & 1;
    const size_t pix = (size_t)n * P + pw + k;
    const float x0 = __shfl_sync(0xffffffffu, cmine.x, k), y0 = __shfl_sync(0xffffffffu, cmine.y, k);
    int wx0 = 0, wy0 = 0;                                       // origin of the Gaussian head's 9 x 9 window
    float wv[3] = {0.0f, 0.0f, 0.0f}, wg[3] = {0.0f, 0.0f, 0.0f};
    if (want_win) {
      wx0 = tap_coord(floor_to_int(__shfl_sync(0xffffffffu, wmean.x, k)), kWinR, 0);
      wy0 = tap_coord(floor_to_int(__shfl_sync(0xffffffffu, wmean.y, k)), kWinR, 0);
    }
    if (GAUSS) {                                                // level-0 values inside the window (clamped addresses: the
      const float* V0 = prm.lvl[0] + pix * (size_t)(prm.H2[0] * prm.W2[0]);   // records zero what the bounds test drops),
#pragma unroll
      for (int ps = 0; ps < 3; ++ps) {                          // consumed after the slices have left
        const int t = min(ps * 32 + lane, kWinTaps - 1);
        const int tj = t / kWinD, ti = t - tj * kWinD;
        const int xc = min(max(tap_coord(wx0, 0, ti), 0), prm.W2[0] - 1), yc = min(max(tap_coord(wy0, 0, tj), 0), prm.H2[0] - 1);
        wv[ps] = __ldg(V0 + (size_t)yc * prm.W2[0] + xc);
      }
    }
    if ((k & 1) == 0) wait(bar_off, k >> 1);                    // the pair's offset records (two completions per tile)
    const uint32_t orec = offs_base + (k & 1) * (TAPS * 8);
    const float2 a0 = lds64(orec + t0 * 8), a1 = lds64(orec + t1c * 8);
    const float2 b0 = lds64(orec + kPairBytes + t0 * 8), b1 = lds64(orec + kPairBytes + t1c * 8);
    float2 o00 = a0, o01 = a1, o10 = b0, o11 = b1;
    if (prm.off1_scale != nullptr) {                            // offset[1]_out = off1 * cum_mask: same product, same rounding as the forward
      const float sc1 = lds32(small + 48 + k * 4);
      o10 = make_float2(__fmul_rn(b0.x, sc1), __fmul_rn(b0.y, sc1));
      o11 = make_float2(__fmul_rn(b1.x, sc1), __fmul_rn(b1.y, sc1));
    }
    const float2 o10_raw = o10;                                 // the stored centre tap still multiplies g_m (see header)
    const float2 up0 = u0, up1 = u1;
    const float m = lds32(small + 32 + k * 4);
    if (lane == CENTER) { o00 = make_float2(0.0f, 0.0f); o10 = make_float2(0.0f, 0.0f); }    // Q5
    // this pixel's eight upstream gradients (2 taps x 4 levels) leave the strip for registers now
    const float* sg = s_g + k;
    float ga0 = sg[t0 * kPixPerWarp], gb0 = sg[t1c * kPixPerWarp];
    float ga1 = sg[(TAPS + t0) * kPixPerWarp], gb1 = sg[(TAPS + t1c) * kPixPerWarp];
    const float ga2 = sg[(2 * TAPS + t0) * kPixPerWarp], gb2 = sg[(2 * TAPS + t1c) * kPixPerWarp];
    const float ga3 = sg[(3 * TAPS + t0) * kPixPerWarp], gb3 = sg[(3 * TAPS + t1c) * kPixPerWarp];
    __syncwarp();                                               // every lane has read its records / gradients ...
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // ... and those generic-proxy reads are ordered before the
    __syncwarp();                                               //     async-proxy refills below (measured: without the fence
    if (k == 1) {                                               //     rare pixels read the NEXT pair's records)
      if (lane == 0) fetch_pair(n, pw + 2);                     // pixels 2, 3 of this tile
    } else if (k == kPixPerWarp - 1 && has_next) {
      if (lane == 0) {                                          // the next tile's first pair and its strip
        fetch_pair(nn, npw);
        fetch_strip(nn, npw);
      }
    }
    if (k + 1 < kPixPerWarp) load_upstream(pix + 1);
    else if (has_next) load_upstream((size_t)nn * P + npw);

    fl_mbar_wait(bars + slot, (k >> 1) & 1);                    // 2 completions per slot and tile: the parity repeats per tile
    const float* box0 = inbox + slot * kInSlotFloats;
    const float* box1 = box0 + kBW01 * kBH01;

    const float x1c = __fmul_rn(x0, 0.5f), y1c = __fmul_rn(y0, 0.5f);
    const float x2c = __fmul_rn(x1c, 0.5f), y2c = __fmul_rn(y1c, 0.5f);
    const float x3c = __fmul_rn(x2c, 0.5f), y3c = __fmul_rn(y2c, 0.5f);
    float* G0 = prm.gv[0] + pix * (size_t)(prm.H2[0] * prm.W2[0]);
    float* G1 = prm.gv[1] + pix * (size_t)(prm.H2[1] * prm.W2[1]);

    // ---------------- deformable levels 0 and 1: offset gradients + scatter
    BTap ta0, tb0, ta1, tb1;                                    // kept for the global slow path after the slice write
    float gm_part = 0.0f;
    // fixed-point scale of this pixel: 2^(22 - exponent of the largest |gradient|); warp-uniform.  Falls back to the
    // float path for non-finite or vanishing gradients.
    float fxp_scale = 0.0f, fxp_inv = 0.0f;
    {
      float mx = fmaxf(fmaxf(fabsf(ga0), fabsf(ga1)), has1 ? fmaxf(fabsf(gb0), fabsf(gb1)) : 0.0f);
      // NaN sampling positions make NaN weights, which must propagate like in the reference: float path.  (Infinite or
      // huge positions are gated out -- a gated-in tap has a fraction in [0, 1), so |w g| <= |g|.)
      const float pn = (o00.x + x0) + (o00.y + y0) + (o10.x + x1c) + (o10.y + y1c) +
                       (has1 ? (o01.x + x0) + (o01.y + y0) + (o11.x + x1c) + (o11.y + y1c) : 0.0f);
      const bool bad = !(isfinite(ga0) && isfinite(ga1) && (!has1 || (isfinite(gb0) && isfinite(gb1)))) || isnan(pn);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
      const int ex = ((__float_as_int(mx) >> 23) & 0xff) - 127;
      if (!__any_sync(0xffffffffu, bad) && ex > -100) {
        fxp_scale = __int_as_float((127 + 22 - ex) << 23);
        fxp_inv = __int_as_float((127 - 22 + ex) << 23);
      }
    }
    const bool fxp = fxp_scale != 0.0f;
    const int xb0 = box_origin_x(floor_to_int(x0), 7, prm.W2[0]), yb0 = box_origin_y(floor_to_int(y0), 7, prm.H2[0]);
    const int xb1 = box_origin_x(floor_to_int(x1c), 7, prm.W2[1]), yb1 = box_origin_y(floor_to_int(y1c), 7, prm.H2[1]);
    auto deform_bwd = [&](int l, const float* bx, int xb, int yb, float cx, float cy, float2 oa, float2 ob, BTap& ta,
                          BTap& tb, float& ga, float& gb, float2& goa, float2& gob) {
      const int H2 = prm.H2[l], W2 = prm.W2[l];
      {
        const float px = __fadd_rn(oa.x, cx), py = __fadd_rn(oa.y, cy);
        const int fx = floor_to_int(px), fy = floor_to_int(py);
        ta.dx = __fsub_rn(px, (float)fx); ta.dy = __fsub_rn(py, (float)fy);
        btap_setup<kBW01, kBH01>(ta, xb, yb, fx, fy, i0, j0, R, H2, W2);
      }
      {
        const float px = __fadd_rn(ob.x, cx), py = __fadd_rn(ob.y, cy);
        const int fx = floor_to_int(px), fy = floor_to_int(py);
        tb.dx = __fsub_rn(px, (float)fx); tb.dy = __fsub_rn(py, (float)fy);
        btap_setup<kBW01, kBH01>(tb, xb, yb, fx, fy, i1, j1, R, H2, W2);
      }
      // corner values (zero-filled out of bounds by the TMA unit) for the offset gradient
      float qa[4], qb[4];
      {
        const float* b = bx + ta.idx;
        qa[0] = b[0]; qa[1] = b[1]; qa[2] = b[kBW01]; qa[3] = b[kBW01 + 1];
        b = bx + tb.idx;
        qb[0] = b[0]; qb[1] = b[1]; qb[2] = b[kBW01]; qb[3] = b[kBW01 + 1];
      }
      const bool miss = (ta.gate && !ta.inbox) || (has1 && tb.gate && !tb.inbox);
      if (__any_sync(0xffffffffu, miss)) {                      // |offset| >= 4: read the corners from global
        const float* V = prm.lvl[l] + pix * (size_t)(H2 * W2);
        if (ta.gate && !ta.inbox) {
          const float* g = V + (size_t)ta.y1 * W2 + ta.x1;
          qa[0] = __ldg(g); qa[1] = ta.xo ? __ldg(g + 1) : 0.0f; qa[2] = ta.yo ? __ldg(g + W2) : 0.0f;
          qa[3] = (ta.xo && ta.yo) ? __ldg(g + W2 + 1) : 0.0f;
        }
        if (tb.gate && !tb.inbox) {
          const float* g = V + (size_t)tb.y1 * W2 + tb.x1;
          qb[0] = __ldg(g); qb[1] = tb.xo ? __ldg(g + 1) : 0.0f; qb[2] = tb.yo ? __ldg(g + W2) : 0.0f;
          qb[3] = (tb.xo && tb.yo) ? __ldg(g + W2 + 1) : 0.0f;
        }
      }
      goa = ta.gate ? offset_grad(qa[0], qa[1], qa[2], qa[3], ta.dx, ta.dy, ga) : make_float2(0.0f, 0.0f);
      gob = (has1 && tb.gate) ? offset_grad(qb[0], qb[1], qb[2], qb[3], tb.dx, tb.dy, gb) : make_float2(0.0f, 0.0f);
      float* ac = acc + (l == 0 ? kOff0 : kOff1);
      if (fxp) {
        btap_scatter_fxp<kBW01>(reinterpret_cast<int*>(ac), ta, true, ga, fxp_scale);
        btap_scatter_fxp<kBW01>(reinterpret_cast<int*>(ac), tb, has1, gb, fxp_scale);
      } else {
        btap_scatter<kBW01, true>(ac, ta, true, ga);
        btap_scatter<kBW01, true>(ac, tb, has1, gb);
      }
    };
    {
      float2 goa, gob;
      deform_bwd(0, box0, xb0, yb0, x0, y0, o00, o01, ta0, tb0, ga0, gb0, goa, gob);
      float2* GO = reinterpret_cast<float2*>(prm.g_off0) + pix * TAPS;
      GO[t0] = goa;
      if (has1) GO[t1] = gob;
    }
    {
      float2 goa, gob;
      deform_bwd(1, box1, xb1, yb1, x1c, y1c, o10, o11, ta1, tb1, ga1, gb1, goa, gob);
      goa.x += up0.x; goa.y += up0.y;                           // + upstream gradient on offset[1]_out (later calls)
      if (has1) { gob.x += up1.x; gob.y += up1.y; }
      // g_m partial: (gO_1 + upstream) . offset[1]_out  (divided by m below).  The centre tap is READ as 0 by the
      // lookup (Q5) but autograd's mul backward multiplies by the stored, unzeroed value -- reproduced here.
      gm_part = __fmaf_rn(goa.x, o10_raw.x, __fmul_rn(goa.y, o10_raw.y));
      if (has1) gm_part += __fmaf_rn(gob.x, o11.x, __fmul_rn(gob.y, o11.y));
      float2* GO = reinterpret_cast<float2*>(prm.g_off1) + pix * TAPS;
      GO[t0] = make_float2(__fmul_rn(goa.x, m), __fmul_rn(goa.y, m));
      if (has1) GO[t1] = make_float2(__fmul_rn(gob.x, m), __fmul_rn(gob.y, m));
    }
    __syncwarp();                                               // shared atomics of this warp are done
    if (fxp) {                                                  // fixed-point sums -> fp32, in place (both deformable boxes)
      for (int q = lane; q < 2 * kBW01 * kBH01; q += 32) {
        const int v = reinterpret_cast<const int*>(acc)[q];
        acc[q] = __fmul_rn(__int2float_rn(v), fxp_inv);
      }
      __syncwarp();
    }

    // ---------------- mask path: g_m -> sigmoid -> 9-tap variance -> level-1 scatter (r = 1 plain lookup)
    BTap tm;
    float gvk;
    {
      const int H2 = prm.H2[1], W2 = prm.W2[1];
      const int fx = floor_to_int(x1c), fy = floor_to_int(y1c);
      tm.dx = __fsub_rn(x1c, floorf(x1c));
      tm.dy = __fsub_rn(y1c, floorf(y1c));
      btap_setup<kBW01, kBH01>(tm, xb1, yb1, fx, fy, mi, mj, 1, H2, W2);
      float q[4];
      const float* b = box1 + tm.idx;
      q[0] = b[0]; q[1] = b[1]; q[2] = b[kBW01]; q[3] = b[kBW01 + 1];
      if (__any_sync(0xffffffffu, tm.gate && !tm.inbox)) {
        if (tm.gate && !tm.inbox) {
          const float* g = prm.lvl[1] + pix * (size_t)(H2 * W2) + (size_t)tm.y1 * W2 + tm.x1;
          q[0] = __ldg(g); q[1] = tm.xo ? __ldg(g + 1) : 0.0f; q[2] = tm.yo ? __ldg(g + W2) : 0.0f;
          q[3] = (tm.xo && tm.yo) ? __ldg(g + W2 + 1) : 0.0f;
        }
      }
      const float v = (lane < 9 && tm.gate) ? blend4(q[0], q[1], q[2], q[3], tm.dx, tm.dy) : 0.0f;
      float s = v;
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      const float mean = __shfl_sync(0xffffffffu, s, 0) / 9.0f;
      const float g_m = warp_sum(gm_part) / m;
      const float g_var = g_m * m * (1.0f - m);
      gvk = lane < 9 ? g_var * 0.25f * (v - mean) : 0.0f;       // 2 (v - mean) / (9 - 1)
      btap_scatter<kBW01, false>(acc + kOff1, tm, lane < 9, gvk);
    }
    // ---------------- zero-offset levels 2 and 3: scatter only (their offsets are detached zeros, corr.py:131-134)
    BTap ta2, tb2, ta3, tb3;
    int xb2, yb2, xb3, yb3;
    auto uniform_bwd = [&](int l, float cx, float cy, BTap& ta, BTap& tb, int& xb, int& yb, float ga, float gb) {
      const int H2 = prm.H2[l], W2 = prm.W2[l];
      const float px = __fadd_rn(0.0f, cx), py = __fadd_rn(0.0f, cy);
      const int fx = floor_to_int(px), fy = floor_to_int(py);
      xb = box_origin_x(fx, 3, W2);
      yb = box_origin_y(fy, 3, H2);
      ta.dx = tb.dx = __fsub_rn(px, (float)fx);
      ta.dy = tb.dy = __fsub_rn(py, (float)fy);
      btap_setup<kBW23, kBH23>(ta, xb, yb, fx, fy, i0, j0, R, H2, W2);
      btap_setup<kBW23, kBH23>(tb, xb, yb, fx, fy, i1, j1, R, H2, W2);
      float* ac = acc + (l == 2 ? kOff2 : kOff3);
      // (fixed-point adds were tried here too: no gain over the conflict-free read-modify-write phases)
      btap_scatter<kBW23, false>(ac, ta, true, ga);
      btap_scatter<kBW23, false>(ac, tb, has1, gb);
    };
    uniform_bwd(2, x2c, y2c, ta2, tb2, xb2, yb2, ga2, gb2);
    uniform_bwd(3, x3c, y3c, ta3, tb3, xb3, yb3, ga3, gb3);
    __syncwarp();
    if (want_win) {                                             // the Gaussian head's window of the merged level-0 gradient
      const int xbs[4] = {xb0, xb1, xb2, xb3}, ybs[4] = {yb0, yb1, yb2, yb3};
      emit_window<false>(prm.gwin != nullptr ? prm.gwin + pix * kWinTaps : nullptr, wg, wx0, wy0, acc, xbs, ybs, nullptr,
                         prm.H2, prm.W2, lane);
      __syncwarp();                                             // the boxes are read before the slice pass re-zeroes them
    }

    // ---------------- stream the four dense slices (zeros + box), then the rare out-of-box taps with global atomics
    float* G2 = prm.gv[2] + pix * (size_t)(prm.H2[2] * prm.W2[2]);
    float* G3 = prm.gv[3] + pix * (size_t)(prm.H2[3] * prm.W2[3]);
    if (ACC) {
      add_box<kBW01, kBH01>(G0, acc + kOff0, xb0, yb0, prm.H2[0], prm.W2[0], lane);
      add_box<kBW01, kBH01>(G1, acc + kOff1, xb1, yb1, prm.H2[1], prm.W2[1], lane);
      add_box<kBW23, kBH23>(G2, acc + kOff2, xb2, yb2, prm.H2[2], prm.W2[2], lane);
      add_box<kBW23, kBH23>(G3, acc + kOff3, xb3, yb3, prm.H2[3], prm.W2[3], lane);
    } else {
      if (BULK) {
        write_slice_bulk<kBW01, kBH01>(G0, acc + kOff0, xb0, yb0, prm.H2[0], prm.W2[0], lane, zero_smem);
        write_slice_bulk<kBW01, kBH01>(G1, acc + kOff1, xb1, yb1, prm.H2[1], prm.W2[1], lane, zero_smem);
      } else {
        write_slice<kBW01, kBH01>(G0, acc + kOff0, xb0, yb0, prm.H2[0], prm.W2[0], lane);
        write_slice<kBW01, kBH01>(G1, acc + kOff1, xb1, yb1, prm.H2[1], prm.W2[1], lane);
      }
      write_slice<kBW23, kBH23>(G2, acc + kOff2, xb2, yb2, prm.H2[2], prm.W2[2], lane);
      write_slice<kBW23, kBH23>(G3, acc + kOff3, xb3, yb3, prm.H2[3], prm.W2[3], lane);
    }
    __syncwarp();                                               // slice stores ordered before the atomics below
    const bool any_miss = (ta0.gate && !ta0.inbox) || (has1 && tb0.gate && !tb0.inbox) || (ta1.gate && !ta1.inbox) ||
                          (has1 && tb1.gate && !tb1.inbox) || (lane < 9 && tm.gate && !tm.inbox) ||
                          (ta2.gate && !ta2.inbox) || (has1 && tb2.gate && !tb2.inbox) || (ta3.gate && !ta3.inbox) ||
                          (has1 && tb3.gate && !tb3.inbox);
    if (__any_sync(0xffffffffu, any_miss)) {
      if (BULK && !ACC) {                                       // the zero ranges must have landed before the atomics
        if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
        __syncwarp();
      }
      if (!ACC) __threadfence();
      btap_scatter_global(G0, ta0, true, ga0, prm.W2[0]);
      btap_scatter_global(G0, tb0, has1, gb0, prm.W2[0]);
      btap_scatter_global(G1, ta1, true, ga1, prm.W2[1]);
      btap_scatter_global(G1, tb1, has1, gb1, prm.W2[1]);
      btap_scatter_global(G1, tm, lane < 9, gvk, prm.W2[1]);
      btap_scatter_global(G2, ta2, true, ga2, prm.W2[2]);
      btap_scatter_global(G2, tb2, has1, gb2, prm.W2[2]);
      btap_scatter_global(G3, ta3, true, ga3, prm.W2[3]);
      btap_scatter_global(G3, tb3, has1, gb3, prm.W2[3]);
      if (want_win) {                                           // out-of-box taps are not in the boxes: window from the slices
        __threadfence();
        __syncwarp();
        float* const Gs[4] = {G0, G1, G2, G3};
        emit_window<true>(prm.gwin != nullptr ? prm.gwin + pix * kWinTaps : nullptr, wg, wx0, wy0, nullptr, nullptr, nullptr,
                          Gs, prm.H2, prm.W2, lane);
      }
    }
    if (GAUSS) {
      const float2 gm_ = make_float2(__shfl_sync(0xffffffffu, wmean.x, k), __shfl_sync(0xffffffffu, wmean.y, k));
      const float2 gc_ = make_float2(__shfl_sync(0xffffffffu, wcov.x, k), __shfl_sync(0xffffffffu, wcov.y, k));
      const float gdn = __shfl_sync(0xffffffffu, wden, k);
      float o0, o1, o2, o3, od;
      gauss_window_grads<true>(wv, wg, gm_, gc_, gdn, wx0, wy0, prm.H2[0], prm.W2[0], lane, o0, o1, o2, o3, od);
      if (lane == 0) {
        reinterpret_cast<float2*>(prm.g_means)[pix] = make_float2(o0, o1);
        reinterpret_cast<float2*>(prm.g_covs)[pix] = make_float2(o2, o3);
        prm.g_den[pix] = od;
      }
    }
    __syncwarp();
    // refill the ring slot: pixel k + 2 of this tile, or pixel k - 2 of the NEXT tile (prefetch across tiles)
    if (k + 2 < kPixPerWarp) {
      const float nx = __shfl_sync(0xffffffffu, cmine.x, k + 2), ny = __shfl_sync(0xffffffffu, cmine.y, k + 2);
      if (lane == 0) issue(slot, n * P + pw + k + 2, nx, ny);
    } else if (has_next) {
      if (k + 2 == kPixPerWarp) wait(bar_small + (par ^ 1) * 8, ((it + 1) >> 1) & 1);
      const float2 cn = lds64(small_base + (par ^ 1) * kSmallBytes + (lane & 3) * 8);
      const int q = k + 2 - kPixPerWarp;
      const float nx = __shfl_sync(0xffffffffu, cn.x, q), ny = __shfl_sync(0xffffffffu, cn.y, q);
      if (lane == 0) issue(slot, nn * P + npw + q, nx, ny);
    }
  }
  n = nn; pw = npw;
  }
  if (BULK && !ACC) {                                           // the zero buffer must outlive the engine's reads
    if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    __syncthreads();
  }
}

}  // namespace lgu

namespace lgu {
static int launch_lookup_fused_bwd(const float* lvl0, const float* lvl1, const float* coords, const float* off0,
                                   const float* off1_out, const float* mask, const float* corr_grad,
                                   const float* off1_out_grad, float* gv0, float* gv1, float* gv2, float* gv3,
                                   float* off0_grad, float* off1_grad, int E, int H, int W, int num_levels, int radius,
                                   bool accumulate, const float* off1_scale, void* stream,
                                   const float* win_means = nullptr, float* gwin = nullptr, const float* win_covs = nullptr,
                                   const float* win_den = nullptr, float* g_means = nullptr, float* g_covs = nullptr,
                                   float* g_den = nullptr);
}
extern "C" int lgu_corr_lookup_fused_backward_cum(const float* lvl0, const float* lvl1, const float* coords,
                                                  const float* off0, const float* off1, const float* cum_mask,
                                                  const float* mask, const float* corr_grad, const float* off1_out_grad,
                                                  float* gv0, float* gv1, float* gv2, float* gv3, float* off0_grad,
                                                  float* off1_grad, int E, int H, int W, int num_levels, int radius,
                                                  int accumulate, void* stream) {
  LGU_REQUIRE(E == 0 || cum_mask != nullptr, "lgu_corr_lookup_fused_backward_cum: null cumulative-mask buffer");
  return lgu::launch_lookup_fused_bwd(lvl0, lvl1, coords, off0, off1, mask, corr_grad, off1_out_grad, gv0, gv1, gv2, gv3,
                                      off0_grad, off1_grad, E, H, W, num_levels, radius, accumulate != 0, cum_mask, stream);
}
// Dense cumulative-mask form that ALSO emits, per source pixel, the 9 x 9 window (centre floor(win_means), x fastest) of
// the merged level-0 gradient g0 + g1/4 + g2/16 + g3/64 -- the only part of the level gradients the Gaussian head's
// backward reads (lgu_build_backward_gauss_window).
extern "C" int lgu_corr_lookup_fused_backward_win(const float* lvl0, const float* lvl1, const float* coords,
                                                  const float* off0, const float* off1, const float* cum_mask,
                                                  const float* mask, const float* corr_grad, const float* off1_out_grad,
                                                  const float* win_means, float* gv0, float* gv1, float* gv2, float* gv3,
                                                  float* off0_grad, float* off1_grad, float* gwin, int E, int H, int W,
                                                  int num_levels, int radius, void* stream) {
  LGU_REQUIRE(E == 0 || (win_means != nullptr && gwin != nullptr), "lgu_corr_lookup_fused_backward_win: null window buffers");
  LGU_REQUIRE((reinterpret_cast<uintptr_t>(win_means) & 7) == 0, "lgu_corr_lookup_fused_backward_win: win_means not 8-byte aligned");
  return lgu::launch_lookup_fused_bwd(lvl0, lvl1, coords, off0, off1, mask, corr_grad, off1_out_grad, gv0, gv1, gv2, gv3,
                                      off0_grad, off1_grad, E, H, W, num_levels, radius, false, cum_mask, stream, win_means,
                                      gwin);
}
// Dense cumulative-mask form with the Gaussian head's backward of the build folded in (GAUSS kernels): besides the level
// and offset gradients, the launch returns what lgu_build_backward_gauss would compute from THIS call's level gradients.
extern "C" int lgu_corr_lookup_fused_backward_gauss(const float* lvl0, const float* lvl1, const float* coords,
                                                    const float* off0, const float* off1, const float* cum_mask,
                                                    const float* mask, const float* corr_grad, const float* off1_out_grad,
                                                    const float* means, const float* covs, const float* den, float* gv0,
                                                    float* gv1, float* gv2, float* gv3, float* off0_grad, float* off1_grad,
                                                    float* means_grad, float* covs_grad, float* den_grad, int E, int H,
                                                    int W, int num_levels, int radius, int gauss_radius, void* stream) {
  LGU_REQUIRE(E == 0 || (means && covs && den && means_grad && covs_grad && den_grad),
              "lgu_corr_lookup_fused_backward_gauss: null Gaussian-head buffers");
  if (gauss_radius != 4) {
    lgu::set_error("lgu_corr_lookup_fused_backward_gauss: only gauss_radius=4 is implemented (got %d); use "
                   "lgu_build_backward_gauss", gauss_radius);
    return LGU_ERR_UNSUPPORTED;
  }
  LGU_REQUIRE(((reinterpret_cast<uintptr_t>(means) | reinterpret_cast<uintptr_t>(covs) | reinterpret_cast<uintptr_t>(means_grad) |
                reinterpret_cast<uintptr_t>(covs_grad)) & 7) == 0 && ((reinterpret_cast<uintptr_t>(den) | reinterpret_cast<uintptr_t>(den_grad)) & 3) == 0,
              "lgu_corr_lookup_fused_backward_gauss: means / covs must be 8-byte aligned");
  LGU_REQUIRE(E == 0 || cum_mask != nullptr, "lgu_corr_lookup_fused_backward_gauss: null cumulative-mask buffer");
  return lgu::launch_lookup_fused_bwd(lvl0, lvl1, coords, off0, off1, mask, corr_grad, off1_out_grad, gv0, gv1, gv2, gv3,
                                      off0_grad, off1_grad, E, H, W, num_levels, radius, false, cum_mask, stream, means,
                                      nullptr, covs, den, means_grad, covs_grad, den_grad);
}
extern "C" int lgu_corr_lookup_fused_backward(const float* lvl0, const float* lvl1, const float* coords,
                                              const float* off0, const float* off1_out, const float* mask,
                                              const float* corr_grad, const float* off1_out_grad, float* gv0,
                                              float* gv1, float* gv2, float* gv3, float* off0_grad, float* off1_grad,
                                              int E, int H, int W, int num_levels, int radius, void* stream) {
  return lgu::launch_lookup_fused_bwd(lvl0, lvl1, coords, off0, off1_out, mask, corr_grad, off1_out_grad, gv0, gv1, gv2,
                                      gv3, off0_grad, off1_grad, E, H, W, num_levels, radius, false, nullptr, stream);
}
extern "C" int lgu_corr_lookup_fused_backward_accumulate(const float* lvl0, const float* lvl1, const float* coords,
                                                         const float* off0, const float* off1_out, const float* mask,
                                                         const float* corr_grad, const float* off1_out_grad,
                                                         float* gv0, float* gv1, float* gv2, float* gv3,
                                                         float* off0_grad, float* off1_grad, int E, int H, int W,
                                                         int num_levels, int radius, void* stream) {
  return lgu::launch_lookup_fused_bwd(lvl0, lvl1, coords, off0, off1_out, mask, corr_grad, off1_out_grad, gv0, gv1, gv2,
                                      gv3, off0_grad, off1_grad, E, H, W, num_levels, radius, true, nullptr, stream);
}
static int lgu::launch_lookup_fused_bwd(const float* lvl0, const float* lvl1, const float* coords, const float* off0,
                                        const float* off1_out, const float* mask, const float* corr_grad,
                                        const float* off1_out_grad, float* gv0, float* gv1, float* gv2, float* gv3,
                                        float* off0_grad, float* off1_grad, int E, int H, int W, int num_levels,
                                        int radius, bool accumulate, const float* off1_scale, void* stream,
                                        const float* win_means, float* gwin, const float* win_covs, const float* win_den,
                                        float* g_means, float* g_covs, float* g_den) {
  using namespace lgu;
  if (E == 0) return LGU_OK;
  LGU_REQUIRE(lvl0 && lvl1 && coords && off0 && off1_out && mask && corr_grad && gv0 && gv1 && gv2 && gv3 &&
                  off0_grad && off1_grad,
              "lgu_corr_lookup_fused_backward: null pointer");
  LGU_REQUIRE(E > 0 && H > 0 && W > 0, "lgu_corr_lookup_fused_backward: bad sizes E=%d H=%d W=%d", E, H, W);
  if (num_levels != 4 || radius != 3 || (W % 32) != 0 || (H % 8) != 0) {
    set_error("lgu_corr_lookup_fused_backward: only num_levels=4, radius=3, W%%32==0, H%%8==0 are implemented "
              "(got levels=%d r=%d H=%d W=%d); use the per-level operators", num_levels, radius, H, W);
    return LGU_ERR_UNSUPPORTED;
  }
  const int P = H * W;
  const long long nslices = (long long)E * P;
  LGU_REQUIRE(nslices < 2147483647LL, "lgu_corr_lookup_fused_backward: E*H*W = %lld too large", nslices);
  float* gv[4] = {gv0, gv1, gv2, gv3};
  for (int l = 0; l < 4; ++l)
    LGU_REQUIRE((reinterpret_cast<uintptr_t>(gv[l]) & 15) == 0, "lgu_corr_lookup_fused_backward: gv%d not 16-byte aligned", l);
  LGU_REQUIRE(((reinterpret_cast<uintptr_t>(lvl0) | reinterpret_cast<uintptr_t>(lvl1)) & 15) == 0,
              "lgu_corr_lookup_fused_backward: pyramid levels must be 16-byte aligned");
  FusedMaps maps;
  FusedLookupBwdParams prm;
  const float* lv[2] = {lvl0, lvl1};
  for (int l = 0; l < 4; ++l) {
    prm.H2[l] = H >> l;
    prm.W2[l] = W >> l;
    prm.gv[l] = gv[l];
  }
  for (int l = 0; l < 2; ++l) {
    prm.lvl[l] = lv[l];
    const int rc = make_slice_map(&maps.m[l], lv[l], nslices, H >> l, W >> l, fl::kBW01, fl::kBH01);
    if (rc) return rc;
  }
  {  // the upstream gradient [E*196, P] as a 2-D tensor: one box = 196 channel rows x 4 pixels (this warp's strip)
    const uint64_t dims[2] = {(uint64_t)P, (uint64_t)E * fl::CH}, strides[1] = {(uint64_t)P * 4};
    const uint32_t box[2] = {fl::kPixPerWarp, fl::CH};
    const int rc = encode_tensor_map(&maps.m[2], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, corr_grad, dims, strides, box,
                                     CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE);
    if (rc) return rc;
  }
  maps.m[3] = maps.m[0];
  LGU_REQUIRE(((reinterpret_cast<uintptr_t>(coords) | reinterpret_cast<uintptr_t>(off0) | reinterpret_cast<uintptr_t>(off1_out) |
                reinterpret_cast<uintptr_t>(mask) | reinterpret_cast<uintptr_t>(corr_grad) |
                reinterpret_cast<uintptr_t>(off1_scale)) & 15) == 0,
              "lgu_corr_lookup_fused_backward: coords / offsets / mask / corr_grad must be 16-byte aligned");
  prm.coords = coords; prm.off0 = off0; prm.off1 = off1_out; prm.mask = mask; prm.g_out = corr_grad;
  prm.g_off1_out = off1_out_grad; prm.g_off0 = off0_grad; prm.g_off1 = off1_grad;
  prm.off1_scale = off1_scale;
  prm.win_means = win_means; prm.gwin = gwin;
  prm.win_covs = win_covs; prm.win_den = win_den; prm.g_means = g_means; prm.g_covs = g_covs; prm.g_den = g_den;
  const bool gauss = g_means != nullptr;
  prm.P = P;
  prm.tiles_per_edge = P / fl::kTile;
  const long long ntiles = (long long)E * prm.tiles_per_edge;
  LGU_REQUIRE(ntiles < 2147483647LL, "lgu_corr_lookup_fused_backward: too many tiles (%lld)", ntiles);
  prm.num_tiles = (int)ntiles;
  const int sms = num_sms();
  // Schedule.  Accumulate mode (footprint-only reductions): persistent, two CTAs per SM, every CTA the same number of
  // tiles (4608 tiles -> 288 CTAs x 16) -- 431 -> 373 us at E = 48.  Dense mode (every slice streamed once, write-bound):
  // one tile per CTA -- persistent CTAs run in lock step and write in phase (690 us against 601 us); the hardware's CTA
  // scheduler staggers them.
  const long long per_cta = accumulate ? (ntiles + 2LL * sms - 1) / (2LL * sms) : 1;
  const long long nblk = (ntiles + per_cta - 1) / per_cta;
  // bulk zero-fill (-4 %) needs row bands that tile a warp (W2 / 4 divides 32 at levels 0 and 1)
  const bool bulk = !accumulate && (W == 64 || W == 128);
  auto kern = accumulate ? lookup_fused_bwd_kernel<true, false>
              : bulk     ? lookup_fused_bwd_kernel<false, true>
                         : lookup_fused_bwd_kernel<false, false>;
  if (gauss)   // dense mode only
    kern = bulk ? lookup_fused_bwd_kernel<false, true, true> : lookup_fused_bwd_kernel<false, false, true>;
  if (int rc = optin_smem(reinterpret_cast<const void*>(kern), flb::kSmemBytes, "lgu_corr_lookup_fused_backward")) return rc;
  kern<<<(unsigned)nblk, fl::kThreads, flb::kSmemBytes, (cudaStream_t)stream>>>(maps, prm);
  return check_launch("lgu_corr_lookup_fused_backward");
}

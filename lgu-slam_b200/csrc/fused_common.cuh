// fused_common.cuh -- pieces shared by the fused CorrBlock.__call__ kernels (lookup_fused.cu, lookup_fused_bwd.cu):
// box geometry of the TMA-staged pyramid patches, mbarrier / TMA wrappers, the branch-free tap fetch.
#pragma once
#include <cuda.h>
#include "common.cuh"

namespace lgu {

namespace fl {
constexpr int kWarps = 8, kThreads = kWarps * 32, kTile = 32, kPixPerWarp = kTile / kWarps;
constexpr int R = 3, RD = 7, TAPS = 49, LEVELS = 4, CH = LEVELS * TAPS;
constexpr int kBW01 = 20, kBH01 = 16, kBW23 = 12, kBH23 = 8;
constexpr int kOff0 = 0, kOff1 = kBW01 * kBH01, kOff2 = 2 * kBW01 * kBH01, kOff3 = kOff2 + kBW23 * kBH23;
constexpr int kSlotFloats = kOff3 + kBW23 * kBH23;                 // 832 floats = 3328 B (26 x 128 B)
constexpr int kSlotBytes = kSlotFloats * 4;
constexpr int kSlots = 2;
constexpr int kZeroBytes = 8192;
constexpr int kOutPitch = kTile + 1;
constexpr int kSmemBoxes = kWarps * kSlots * kSlotBytes;           // 53,248 B
constexpr int kSmemOut = CH * kOutPitch * 4;                       // 25,872 B
constexpr int kSmemBytes = kSmemBoxes + kSmemOut + kWarps * kSlots * 8;
}  // namespace fl

__device__ __forceinline__ uint32_t fl_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void fl_mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(fl_smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fl_mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(fl_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void fl_mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "FL_WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra FL_DONE_%=;\n\t"
      "bra FL_WAIT_%=;\n\t"
      "FL_DONE_%=:\n\t}" ::"r"(fl_smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void fl_tma_box(void* dst, const CUtensorMap* map, uint64_t* bar, int x, int y, int z) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(
          fl_smem_u32(dst)),
      "l"(map), "r"(fl_smem_u32(bar)), "r"(x), "r"(y), "r"(z)
      : "memory");
}

// Zero ranges of a dense gradient slice leave through the TMA engine: cp.async.bulk shared -> global from a CTA-wide
// zero buffer of kZeroBytes (16-byte aligned destination and size), issued by one lane into its current bulk group.
__device__ __forceinline__ void bulk_zero(float* dst, int bytes, const void* zero_smem) {
  while (bytes > 0) {
    const int n = bytes < fl::kZeroBytes ? bytes : fl::kZeroBytes;
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(fl_smem_u32(zero_smem)), "r"(n)
                 : "memory");
    dst += n >> 2;
    bytes -= n;
  }
}

// Box origin of a level: columns start at (floor(c) - reach) rounded down to a multiple of 4 (16-byte TMA
// alignment), clamped so that saturated float->int conversions cannot overflow the TMA coordinate arithmetic.
__device__ __forceinline__ int box_origin_x(int f, int reach, int W2) {
  const int v = max(min(f, W2 + 64), -64) - reach;
  return v & ~3;
}
__device__ __forceinline__ int box_origin_y(int f, int reach, int H2) { return max(min(f, H2 + 64), -64) - reach; }

// One bilinear tap against the staged box.  Branch-free fast path: the four corners are read from shared memory at
// a clamped (always valid) index; out-of-bounds corners were zero-filled by the TMA unit, so no per-corner select
// is needed when the 2x2 footprint lies inside the box.  `miss` flags the lanes whose footprint is outside the box
// (|offset| >= 4) and that still pass the reference's top-left gate: the caller patches those from global memory.
struct Tap {
  float dx, dy, q11, q21, q12, q22;
  int x1, y1;
  bool gate, miss;
};

// PER_CORNER = false: the reference's volume lookups gate the whole tap on its top-left corner (quirk Q3);
// PER_CORNER = true : lowMem_defSample / altcorr gate every corner on its own (quirk Q4) -- which is exactly what the
//                     zero-filled TMA box gives, so the tap is always "on" and only the slow path needs the tests.
template <int BW, int BH, bool PER_CORNER = false>
__device__ __forceinline__ void tap_fetch(Tap& t, const float* __restrict__ box, int xb, int yb, int fx, int fy, int i,
                                          int j, int r, int H2, int W2) {
  t.x1 = tap_coord(fx, r, i);
  t.y1 = tap_coord(fy, r, j);
  t.gate = PER_CORNER ? true : (((unsigned)t.x1 < (unsigned)W2) && ((unsigned)t.y1 < (unsigned)H2));   // Q3 / Q4
  const unsigned rx = (unsigned)t.x1 - (unsigned)xb, ry = (unsigned)t.y1 - (unsigned)yb;
  const bool inbox = rx < (unsigned)(BW - 1) && ry < (unsigned)(BH - 1);
  t.miss = t.gate && !inbox;
  const float* b = box + (inbox ? ry * BW + rx : 0u);
  t.q11 = b[0]; t.q21 = b[1]; t.q12 = b[BW]; t.q22 = b[BW + 1];
}
// Slow path for flagged lanes: same gating as the reference (x2 / y2 corners gated individually).
template <bool PER_CORNER = false>
__device__ __forceinline__ void tap_patch_from_global(Tap& t, const float* __restrict__ V, int H2, int W2) {
  if (t.miss) {
    const int x2 = wrap_inc(t.x1), y2 = wrap_inc(t.y1);
    const bool x1i = (unsigned)t.x1 < (unsigned)W2, y1i = (unsigned)t.y1 < (unsigned)H2;
    const bool xo = (unsigned)x2 < (unsigned)W2, yo = (unsigned)y2 < (unsigned)H2;
    // 64-bit element offset: with PER_CORNER the top-left corner itself may be out of bounds
    const float* g = V + ((long long)t.y1 * W2 + t.x1);
    t.q11 = (x1i && y1i) ? __ldg(g) : 0.0f;
    t.q21 = (xo && y1i) ? __ldg(g + 1) : 0.0f;
    t.q12 = (x1i && yo) ? __ldg(g + W2) : 0.0f;
    t.q22 = (xo && yo) ? __ldg(g + W2 + 1) : 0.0f;
  }
}
__device__ __forceinline__ float tap_value(const Tap& t) {
  return t.gate ? blend4(t.q11, t.q21, t.q12, t.q22, t.dx, t.dy) : 0.0f;
}


struct FusedMaps {
  CUtensorMap m[4];
};

// The slices [nslices, H2, W2] of a pyramid level as a 3-D fp32 tensor, box bw x bh of one slice, no swizzle.
static inline int make_slice_map(CUtensorMap* map, const float* base, long long nslices, int H2, int W2, int bw, int bh) {
  const uint64_t dims[3] = {(uint64_t)W2, (uint64_t)H2, (uint64_t)nslices};
  const uint64_t strides[2] = {(uint64_t)W2 * 4, (uint64_t)W2 * H2 * 4};
  const uint32_t box[3] = {(uint32_t)bw, (uint32_t)bh, 1};
  return encode_tensor_map(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, base, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_NONE,
                           CU_TENSOR_MAP_L2_PROMOTION_NONE);
}

}  // namespace lgu

// lookup_fused.cu -- CorrBlock.__call__'s data path in ONE launch (sm_100a, TMA-staged pyramid patches).
//
// Replaces the op sequence of /root/reference/droid_slam/modules/corr.py:88-109:
//   permute+contiguous (coords) -> 4x coords/2^l -> corr_index_forward(lvl1, r=1) -> permute -> var -> sigmoid
//   -> offset[1] *= mask -> 4x defCorr_index_forward(lvl l, r=3) -> view -> cat
// (5 extension launches + ~12 small torch kernels, every level's result written, re-read by cat and written
// again) by one kernel that reads coords once, stages the <= 16x16 footprint of every pyramid level in shared
// memory with TMA box loads, and writes the 196-channel output exactly once.
//
// Work split: CTA = 32 consecutive source pixels of one edge (8 warps x 4 pixels, ONE WARP PER PIXEL,
// lane = tap).  Per pixel one elected lane issues four cp.async.bulk.tensor.3d loads (tensor maps over
// [E*P, H2, W2] per level; out-of-bounds elements are zero-filled by the TMA unit):
//     level 0,1 : box 20 x 16  (16 columns [fx-7, fx+8] for |offset| < 4, +3 because the box start must be
//                               16-byte aligned -- measured: an unaligned inner start coordinate raises
//                               "illegal instruction" on sm_100a)
//     level 2,3 : box 12 x 8   (zero offsets: columns [fx-3, fx+4])
// into a per-warp 2-slot ring (mbarrier complete_tx), so the gathers of the next pixel are in flight while the
// current one is blended.  Taps that fall outside the staged box (|offset| >= 4, never produced by the
// reference's 4*tanh heads) take a direct global-load path with identical gating.
// The 196 x 32 result tile is transposed through padded shared memory and stored as 128-byte rows.
//
// Index logic is the reference's, bit for bit (defCorrSample_kernel.cu:56-67, corrSample_kernel.cu:52-60;
// quirks Q1, Q3, Q5, Q7): levels 0, 2, 3 are bit-identical to defCorr_index_forward; level 1 differs only through
// the fp32 rounding of the 9-tap variance / sigmoid that scales its offsets.
#include <cuda_fp16.h>
#include "fused_common.cuh"

namespace lgu {

// Round-2 structure (profiles/r02_fused_lookup.md).  The round-1 kernel ran 9 tap passes per pixel (2 per level with 17
// of 32 lanes idle in every second one, plus the mask pass) at ~1000 warp instructions per pixel and was ISSUE-limited
// (53 % issue-active with 4 warps per scheduler) while DRAM sat at 53 % of peak.  Here the 196 taps of a pixel are ONE
// flat index space g = level*49 + tap walked in 7 passes of 32 lanes (6.1 needed); the 9 taps of the r=1 mask lookup
// ride in the idle lanes of the last pass, which runs first.  Everything level-dependent (level coordinates, box
// origin, box address and pitch, level extent) comes from a per-warp table in shared memory that the TMA-issuing lanes
// fill, so the pass body is branch-free and identical for every lane: 2 LDS.128 + ~35 ALU + 4 LDS + 1 STS.
namespace flf {
constexpr int kRing = 2;                                             // TMA ring depth (boxes in flight per warp)
constexpr int kPasses = 7;                                           // ceil(196 / 32)
constexpr int kRecBytes = 32;                                        // one table record = 2 x 16 B
constexpr int kRingBytes = fl::kWarps * kRing * fl::kSlotBytes;      // 53,248 B
constexpr int kSmemTab = fl::kWarps * kRing * fl::LEVELS * kRecBytes;    // 2,048 B
constexpr int kOffBytes = fl::kPixPerWarp * fl::TAPS * 8;            // one level's offset records of a warp's 4 pixels: 1,568 B
constexpr int kSmemOffs = fl::kWarps * 2 * kOffBytes;                // 25,088 B (levels 0 and 1)
constexpr int kSmallBytes = 64;                                      // coords (32 B) + cumulative masks (16 B), per warp and tile parity
constexpr int kSmemSmall = fl::kWarps * 2 * kSmallBytes;             // 1,024 B
constexpr int kBarsPerWarp = kRing + 3;                              // ring slots, offsets, small[2]
constexpr int kSmemBars = fl::kWarps * kBarsPerWarp * 8;
constexpr int kOffOut = kRingBytes;
constexpr int kOffTab = kOffOut + fl::kSmemOut;
constexpr int kOffOffs = kOffTab + kSmemTab;
constexpr int kOffSmall = kOffOffs + kSmemOffs;
constexpr int kOffBars = kOffSmall + kSmemSmall;
constexpr int kFwdSmemBytes = kOffBars + kSmemBars;                  // 107,600 B: two CTAs per SM
}  // namespace flf

struct FusedLookupParams {
  const float* lvl[4];
  const float* coords;   // [E,P,2] (x,y) level-0 units
  const float* off0;     // [E,P,49,2]  read only (its centre tap is read as 0, Q5)
  float* off1;           // [E,P,49,2]  write_back: <- off1 * mask (Q7), every tap; the centre tap is read as 0
  void* out;             // [E_out,196,P] fp32 (or fp16, see HALF): edge n is written to row out_index[n] (or n)
  const int32_t* out_index;    // [E] or null: destination row of every edge -- lets a rank of the sharded backend store
                               // straight into the gathered buffer on another GPU (NVLink peer memory), sharded.py
  float* mask_out;       // [E,P] or null: the sigmoid(var) mask of this call
  float* cum_mask;       // [slots,P] or null: running product of the masks of all calls so far (in/out); off1 stays pristine
  int P, tiles_per_edge, num_tiles;
  int H2[4], W2[4];
  long long off_edge_stride;   // float2 elements between the offset slabs of consecutive edges (0: every edge reads slab 0, Q2)
  int apply_mask;              // 1: level-1 offsets are scaled by sigmoid(var) of this call (CorrBlock); 0: used as given
  const int32_t* slots;        // [E] or null: edge n lives in pyramid / offset slot slots[n] (edge-slot pool)
  // CONV: the consumer's first layer, UpdateModule.corr_encoder[0:2] = Conv2d(196, 128, 1) + ReLU (droid_net.py:74-76,115),
  // evaluated on the staged 196 x 32 tile before it leaves the SM
  const float4* conv_w;        // [8 warps][25 k-steps][32 lanes][2] float4: mma fragments (a0..a3) of W_hi then W_lo (lgu_pack_conv1x1)
  const float* conv_b;         // [128] or null
  void* enc;                   // [E_out,128,P] fp32 (fp16 with HALF); rows follow out_index like `out`
  int conv_relu;
  const float* boxes0;         // [E,P,16,20] or null: level 0 as COMPACT per-pixel boxes (lgu_build_boxes) instead of a volume
  const float* boxes1;         // the same for level 1
};

__device__ __forceinline__ float4 flf_lds128(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ float2 flf_lds64(uint32_t addr) {
  float2 v;
  asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ float flf_lds(uint32_t addr) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr) : "memory");
  return v;
}
// 1-D bulk copy global -> shared (16-byte aligned, size a multiple of 16), completion on an mbarrier
__device__ __forceinline__ void flf_bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src),
               "r"(bytes), "r"(bar)
               : "memory");
}

// PC: per-corner gating (lowMem / altcorr semantics, Q4) instead of top-left gating (Q3)
// HALF: the 196-channel rows are stored as fp16 (round-to-nearest) -- what `update_op` reads under autocast
//       (factor_graph.py:284-286); halves the output stream (and the NVLink traffic of the sharded backend)
//
// PERSISTENT CTAs (two per SM) walk the 32-pixel tiles with a stride of the grid.  ncu on the per-tile version
// (profiles/r02_fused_lookup.md) put ~20 % of the warp time into the per-CTA prologue / epilogue (first coords load,
// first box round trip, the barrier before the store phase) and 11 % into ONE instruction: the first use of a staged box
// value, stalled on the long scoreboard it shared with the LDG prefetch of the next pixel's offsets.  Here nothing in the
// pixel loop is an LDG: a tile's offset records (2 x 1,568 B per warp), coords and cumulative masks arrive by
// cp.async.bulk on their own mbarriers, the next tile's coords are on chip before the current tile ends, and the ring
// keeps prefetching boxes ACROSS tile boundaries, so the memory pipeline never drains between tiles.
// m16n8k8 TF32 tensor-core MMA on register fragments (D += A * B, fp32 accumulate)
__device__ __forceinline__ void flf_mma_tf32(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t flf_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return r;
}

// CONV: the consumer's first layer evaluated on the staged tile (see FusedLookupParams::conv_w)
enum ConvMode : int { kConvNone = 0, kConvTF32 = 1, kConvF16 = 2 };

// m16n8k16 fp16 tensor-core MMA on register fragments (D += A * B, fp32 accumulate)
__device__ __forceinline__ void flf_mma_f16(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t flf_h2(float lo, float hi) {     // round-to-nearest-even, like Tensor.half()
  const __half2 h = __floats2half2_rn(lo, hi);
  return *reinterpret_cast<const uint32_t*>(&h);
}

template <bool PC, bool HALF, int CONV = kConvNone>
__global__ void __launch_bounds__(fl::kThreads, 2)
lookup_fused_kernel(const __grid_constant__ FusedMaps maps, const FusedLookupParams prm) {
  using namespace fl;
  using namespace flf;
  extern __shared__ __align__(1024) uint8_t smem[];              // no static shared memory: base is 1024-aligned
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* s_out = reinterpret_cast<float*>(smem + kOffOut);       // [CH][kOutPitch]
  const uint32_t smem0 = fl_smem_u32(smem);
  const uint32_t box_base = smem0 + warp * kRing * kSlotBytes;
  const uint32_t tab_base = smem0 + kOffTab + warp * kRing * LEVELS * kRecBytes;
  const uint32_t offs_base = smem0 + kOffOffs + warp * 2 * kOffBytes;          // [level 0 | level 1][pixel][tap] float2
  const uint32_t small_base = smem0 + kOffSmall + warp * 2 * kSmallBytes;      // [parity]{coords[4] float2, cum[4] float}
  const uint32_t bar_base = smem0 + kOffBars + warp * kBarsPerWarp * 8;        // ring[kRing], offsets, small[2]
  const uint32_t bar_off = bar_base + kRing * 8, bar_small = bar_base + (kRing + 1) * 8;
  const int P = prm.P;

  // ---- per-lane level record: lanes 0..3 own level `lane` of the warp's table (static half written once)
  const int myl = lane & 3;
  const int myW2 = prm.W2[myl], myH2 = prm.H2[myl];
  if (lane < LEVELS * kRing) {
    const int q = lane >> 2;                                    // slot
    const int boff = myl == 0 ? kOff0 : (myl == 1 ? kOff1 : (myl == 2 ? kOff2 : kOff3));
    const int bw = myl < 2 ? kBW01 : kBW23;
    const uint32_t rec = tab_base + (q * LEVELS + myl) * kRecBytes;
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(rec + 16), "r"(box_base + q * kSlotBytes + boff * 4),
                 "r"(bw * 4), "r"(myW2), "r"(myH2)
                 : "memory");
  }
  if (lane == 0) {
#pragma unroll
    for (int q = 0; q < kBarsPerWarp; ++q)
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar_base + q * 8));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncwarp();

  // tile -> (edge, first pixel of this warp, storage slot)
  auto tile_edge = [&](int tile, int& n, int& pw, int& ns) {
    n = tile / prm.tiles_per_edge;
    pw = (tile - n * prm.tiles_per_edge) * kTile + warp * kPixPerWarp;
    ns = prm.slots != nullptr ? __ldg(prm.slots + n) : n;
  };
  // lane 0: fetch a tile's coords (+ cumulative masks) / offset records into shared memory
  auto fetch_small = [&](int n, int pw, int ns, int par) {
    const uint32_t dst = small_base + par * kSmallBytes, bar = bar_small + par * 8;
    const uint32_t bytes = prm.cum_mask != nullptr ? 48u : 32u;
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
    flf_bulk_g2s(dst, prm.coords + ((size_t)n * P + pw) * 2, 32, bar);
    if (prm.cum_mask != nullptr) flf_bulk_g2s(dst + 32, prm.cum_mask + (size_t)ns * P + pw, 16, bar);
  };
  auto fetch_offsets = [&](int pw, int ns) {
    const size_t opix = ((size_t)ns * prm.off_edge_stride + (size_t)pw * TAPS) * 2;     // in floats
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_off), "r"(2u * kOffBytes) : "memory");
    flf_bulk_g2s(offs_base, prm.off0 + opix, kOffBytes, bar_off);
    flf_bulk_g2s(offs_base + kOffBytes, prm.off1 + opix, kOffBytes, bar_off);
  };
  auto wait = [&](uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "FLF_WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra FLF_DONE_%=;\n\t"
        "bra FLF_WAIT_%=;\n\t"
        "FLF_DONE_%=:\n\t}" ::"r"(bar),
        "r"(parity)
        : "memory");
  };

  // Issue the four boxes of one pixel into ring slot `slot`: lane l (< 4) scales the coordinates to level l (coords / 2^l
  // as successive exact halvings, corr.py:103), derives the box origin and writes the dynamic half of its record; lane 0
  // launches the copies.
  auto issue = [&](int slot, int pix, float cx, float cy) {
#pragma unroll
    for (int q = 1; q < LEVELS; ++q)
      if (myl >= q) { cx = __fmul_rn(cx, 0.5f); cy = __fmul_rn(cy, 0.5f); }
    const int reach = myl < 2 ? 7 : 3;
    const int xb = box_origin_x(floor_to_int(cx), reach, myW2), yb = box_origin_y(floor_to_int(cy), reach, myH2);
    if (lane < LEVELS)
      asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(tab_base + (slot * LEVELS + myl) * kRecBytes),
                   "r"(__float_as_int(cx)), "r"(__float_as_int(cy)), "r"(xb), "r"(yb)
                   : "memory");
    int xs[LEVELS], ys[LEVELS];
#pragma unroll
    for (int l = 0; l < LEVELS; ++l) { xs[l] = __shfl_sync(0xffffffffu, xb, l); ys[l] = __shfl_sync(0xffffffffu, yb, l); }
    if (lane == 0) {
      const uint32_t dst = box_base + slot * kSlotBytes, bar = bar_base + slot * 8;
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"((uint32_t)kSlotBytes) : "memory");
#pragma unroll
      for (int l = 0; l < LEVELS; ++l) {
        const int o = l == 0 ? kOff0 : (l == 1 ? kOff1 : (l == 2 ? kOff2 : kOff3));
        if (PC && l < 2 && (l == 0 ? prm.boxes0 : prm.boxes1) != nullptr) {   // the pixel's box was written in place of its slice
          flf_bulk_g2s(dst + o * 4, (l == 0 ? prm.boxes0 : prm.boxes1) + (size_t)pix * (kBW01 * kBH01), kBW01 * kBH01 * 4, bar);
          continue;
        }
        asm volatile(
            "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(
                dst + o * 4),
            "l"(&maps.m[l]), "r"(bar), "r"(xs[l]), "r"(ys[l]), "r"(pix)
            : "memory");
      }
    }
    __syncwarp();                                               // table records visible to the whole warp
  };

  // ---- per-lane tap constants of the 7 passes: g = pass*32 + lane -> (level, i - r, j - r); the mask taps (r = 1 on
  // level 1) sit on lanes 4..12 of the last pass, whose lanes 0..3 are taps 45..48 of level 3
  constexpr int CENTER = R * RD + R;                            // tap 24
  int recoff[kPasses], di[kPasses], dj[kPasses];
#pragma unroll
  for (int ps = 0; ps < kPasses; ++ps) {
    const int g = ps * 32 + lane;
    int l = min(g, CH - 1) / TAPS;
    int t = min(g, CH - 1) - l * TAPS;
    int i = t / RD, j = t - i * RD, r = R;
    if (ps == kPasses - 1 && lane >= 4) {                       // mask taps (lanes 13..31: harmless duplicates of tap 8)
      const int mt = min(lane - 4, 8);
      l = 1; r = 1; i = mt / 3; j = mt - i * 3;
    }
    recoff[ps] = l * kRecBytes;
    di[ps] = i - r;
    dj[ps] = j - r;
  }
  const bool is_mask_lane = lane >= 4 && lane < 13;
  // shared-memory address of this lane's offset record in passes 0..3, relative to the pixel's record pair
  // (flat taps g < 98: pass 0 = level 0 taps 0..31; pass 1 = level 0 taps 32..48 | level 1 taps 0..14; pass 2 = level 1
  // taps 15..46; pass 3 = level 1 taps 47, 48 on lanes 0, 1)
  const uint32_t oaddr0 = offs_base + lane * 8;
  const uint32_t oaddr1 = lane < 17 ? offs_base + (32 + lane) * 8 : offs_base + kOffBytes + (lane - 17) * 8;
  const uint32_t oaddr2 = offs_base + kOffBytes + (15 + lane) * 8;
  const uint32_t oaddr3 = offs_base + kOffBytes + (47 + min(lane, 1)) * 8;

  // One bilinear tap of the flat index space against the staged boxes (defCorrSample_kernel.cu:56-86).
  auto tap = [&](int slot, int ps, float2 o, size_t pix) -> float {
    const uint32_t rec = tab_base + slot * LEVELS * kRecBytes + recoff[ps];
    const float4 a = flf_lds128(rec);
    const float4 b = flf_lds128(rec + 16);
    const int xb = __float_as_int(a.z), yb = __float_as_int(a.w);
    const uint32_t baddr = (uint32_t)__float_as_int(b.x);
    const int pitch = __float_as_int(b.y);                      // box row pitch in bytes (80 or 48)
    const int W2 = __float_as_int(b.z), H2 = __float_as_int(b.w);
    const float px = __fadd_rn(o.x, a.x), py = __fadd_rn(o.y, a.y);
    const int fx = floor_to_int(px), fy = floor_to_int(py);
    Tap t;
    t.dx = PC ? __fsub_rn(px, floorf(px)) : __fsub_rn(px, (float)fx);     // lowMem_defSample.cu:87-88 uses floor()
    t.dy = PC ? __fsub_rn(py, floorf(py)) : __fsub_rn(py, (float)fy);
    t.x1 = (int)((unsigned)fx + (unsigned)di[ps]);
    t.y1 = (int)((unsigned)fy + (unsigned)dj[ps]);
    t.gate = PC ? true : (((unsigned)t.x1 < (unsigned)W2) && ((unsigned)t.y1 < (unsigned)H2));   // Q3 / Q4
    const unsigned rx = (unsigned)t.x1 - (unsigned)xb, ry = (unsigned)t.y1 - (unsigned)yb;
    // box extents from the pitch: 20 x 16 (pitch 80) or 12 x 8 (pitch 48)
    bool inbox = rx < (unsigned)((pitch >> 2) - 1) && ry < (unsigned)(pitch == kBW01 * 4 ? kBH01 - 1 : kBH23 - 1);
    const bool compact = PC && ((prm.boxes0 != nullptr && recoff[ps] == 0) ||      // level 0 / 1 held as per-pixel boxes
                                (prm.boxes1 != nullptr && recoff[ps] == kRecBytes));
    // compact level 0: an offset of exactly 4.0 whose sum with the coordinate rounds up to the next integer puts the tap
    // on the box's last row with dy == 0 -- the row below then has weight 0 (times a finite value of the next region)
    if (compact && ry == (unsigned)(kBH01 - 1) && rx < (unsigned)(kBW01 - 1) && t.dy == 0.0f) inbox = true;
    t.miss = t.gate && !inbox;
    const uint32_t ad = baddr + (inbox ? ry * (unsigned)pitch + rx * 4u : 0u);
    t.q11 = flf_lds(ad);
    t.q21 = flf_lds(ad + 4);
    t.q12 = flf_lds(ad + pitch);
    t.q22 = flf_lds(ad + pitch + 4);
    if (__any_sync(0xffffffffu, t.miss)) {                      // |offset| >= 4 or clamped far-out coords: rare
      const int l = recoff[ps] / kRecBytes;
      if (compact) {
        // no volume behind the boxes: a corner outside the box is zero if it is outside the image too (what the box
        // holds for such cells); inside the image it cannot be served -- offsets beyond the documented bound (|o| <= 4)
        if (t.miss) {
          const int x2 = wrap_inc(t.x1), y2 = wrap_inc(t.y1);
          const bool any_in = (((unsigned)t.x1 < (unsigned)W2) || ((unsigned)x2 < (unsigned)W2)) &&
                              (((unsigned)t.y1 < (unsigned)H2) || ((unsigned)y2 < (unsigned)H2));
          const float fill = any_in ? __int_as_float(0x7fc00000) : 0.0f;
          t.q11 = t.q21 = t.q12 = t.q22 = fill;
        }
      } else {
        tap_patch_from_global<PC>(t, prm.lvl[l] + pix * (size_t)(H2 * W2), H2, W2);
      }
    }
    return tap_value(t);
  };

  // ---- prologue of the first tile: parameters, offsets, the first kRing pixels' boxes
  int tile = blockIdx.x;
  if (tile >= prm.num_tiles) return;
  int n, pw, ns;
  tile_edge(tile, n, pw, ns);
  if (lane == 0) {
    fetch_small(n, pw, ns, 0);
    fetch_offsets(pw, ns);
  }
  wait(bar_small, 0);
  {
    const float2 c0 = flf_lds64(small_base + (lane & 3) * 8);   // lane q holds pixel q's coords (q < 4)
#pragma unroll
    for (int q = 0; q < kRing; ++q)
      issue(q, ns * P + pw + q, __shfl_sync(0xffffffffu, c0.x, q), __shfl_sync(0xffffffffu, c0.y, q));
  }

#pragma unroll 1
  for (int it = 0; tile < prm.num_tiles; ++it, tile += gridDim.x) {
    const int par = it & 1;
    const int ntile = tile + gridDim.x;
    const bool has_next = ntile < prm.num_tiles;
    int nn = 0, npw = 0, nns = 0;
    if (has_next) {
      tile_edge(ntile, nn, npw, nns);
      if (lane == 0) fetch_small(nn, npw, nns, par ^ 1);        // next tile's coords / masks: on chip long before they are needed
    }
    wait(bar_off, par);                                         // this tile's offset records
    const uint32_t small = small_base + par * kSmallBytes;

#pragma unroll 1
    for (int k = 0; k < kPixPerWarp; ++k) {
      const int slot = k % kRing;                               // kPixPerWarp is a multiple of kRing: slots repeat per tile
      const int p = pw + k;
      const size_t pix = (size_t)ns * P + p;                    // slice index in the pyramid storage
      const uint32_t orec = (uint32_t)k * (TAPS * 8);
      float2 o[4];
      o[0] = flf_lds64(oaddr0 + orec);
      o[1] = flf_lds64(oaddr1 + orec);
      o[2] = flf_lds64(oaddr2 + orec);
      o[3] = lane < 2 ? flf_lds64(oaddr3 + orec) : make_float2(0.0f, 0.0f);
      float cum = 1.0f;
      if (prm.cum_mask != nullptr) cum = flf_lds(small + 32 + k * 4);

      wait(bar_base + slot * 8, ((it * (kPixPerWarp / kRing)) + k / kRing) & 1);
      float* so = s_out + warp * kPixPerWarp + k;               // column of this pixel in the output tile

      // ---------------- last pass first: level-3 taps 45..48 (lanes 0..3) + the r=1 mask taps on level 1 (lanes 4..12,
      // corrSample_kernel.cu:52-77) -> unbiased variance over the 9 taps (torch.var default, corr.py:96) -> sigmoid
      float m;
      {
        const float v = tap(slot, kPasses - 1, make_float2(0.0f, 0.0f), pix);
        if (lane < 4) so[((kPasses - 1) * 32 + lane) * kOutPitch] = v;
        const float vm = is_mask_lane ? v : 0.0f;
        float s = vm;
#pragma unroll
        for (int sh = 8; sh > 0; sh >>= 1) s += __shfl_xor_sync(0xffffffffu, s, sh);    // lanes 0..3, 13..15 contribute 0
        const float mean = __shfl_sync(0xffffffffu, s, 0) / 9.0f;
        const float d = is_mask_lane ? (vm - mean) : 0.0f;
        float ss = d * d;
#pragma unroll
        for (int sh = 8; sh > 0; sh >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, sh);
        const float var = __shfl_sync(0xffffffffu, ss, 0) * 0.125f;
        m = 1.0f / (1.0f + expf(-var));
      }
      // offset[1] <- offset[1] * mask (Q7) for every tap of level 1 (flat taps 49..97: pass 1 lanes >= 17, pass 2, pass 3
      // lanes 0..1); with a cumulative-mask buffer the stored offsets stay pristine and the product of all masks so far
      // is applied instead
      if (prm.apply_mask) {
        const float mm = prm.cum_mask != nullptr ? __fmul_rn(cum, m) : m;
        if (lane >= 17) o[1] = make_float2(__fmul_rn(o[1].x, mm), __fmul_rn(o[1].y, mm));
        o[2] = make_float2(__fmul_rn(o[2].x, mm), __fmul_rn(o[2].y, mm));
        // lanes >= 2 are level-2 taps: their zero offsets stay zero (0 * a NaN mask would move them to F2I(NaN) = 0)
        if (lane < 2) o[3] = make_float2(__fmul_rn(o[3].x, mm), __fmul_rn(o[3].y, mm));
        if (prm.cum_mask != nullptr) {
          if (lane == 0) prm.cum_mask[(size_t)ns * P + p] = mm;
        } else {
          float2* O1 = reinterpret_cast<float2*>(prm.off1) + (size_t)ns * prm.off_edge_stride + (size_t)p * TAPS;
          if (lane >= 17) O1[lane - 17] = o[1];
          O1[15 + lane] = o[2];
          if (lane < 2) O1[47 + lane] = o[3];
        }
      }
      if (lane == 0 && prm.mask_out != nullptr) prm.mask_out[(size_t)n * P + p] = m;
      // Q5: the centre taps read as 0 (flat taps 24 and 49 + 24 = 73 = pass 2, lane 9)
      if (lane == CENTER) o[0] = make_float2(0.0f, 0.0f);
      if (lane == TAPS + CENTER - 64) o[2] = make_float2(0.0f, 0.0f);

#pragma unroll
      for (int ps = 0; ps < kPasses - 1; ++ps) {
        const float v = tap(slot, ps, ps < 4 ? o[ps] : make_float2(0.0f, 0.0f), pix);
        so[(ps * 32 + lane) * kOutPitch] = v;
      }

      __syncwarp();                                             // every lane is done with this slot
      // refill the slot: pixel k + kRing of this tile, or pixel k + kRing - 4 of the NEXT tile (prefetch across tiles)
      const int kn = k + kRing;
      if (kn < kPixPerWarp) {
        const float2 c = flf_lds64(small + (lane & 3) * 8);
        issue(slot, ns * P + pw + kn, __shfl_sync(0xffffffffu, c.x, kn), __shfl_sync(0xffffffffu, c.y, kn));
      } else if (has_next) {
        if (kn == kPixPerWarp) wait(bar_small + (par ^ 1) * 8, ((it + 1) >> 1) & 1);
        const float2 c = flf_lds64(small_base + (par ^ 1) * kSmallBytes + (lane & 3) * 8);
        const int q = kn - kPixPerWarp;
        issue(slot, nns * P + npw + q, __shfl_sync(0xffffffffu, c.x, q), __shfl_sync(0xffffffffu, c.y, q));
      }
    }
    // the warp has consumed this tile's offset records: fetch the next tile's behind the store phase (the proxy fence
    // orders the warp's generic-proxy reads of the buffer before the async-proxy refill)
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncwarp();
    if (has_next && lane == 0) fetch_offsets(npw, nns);

    // kConvF16: the first kPre weight fragments are requested before the barrier and kPre loads stay in flight through
    // the k-loop (the TMA buffers leave too little L1 for the 53 KB of fragments, so every tile re-reads them from L2;
    // measured on a B200 at 1000 W: 280.7 against 283.4 us per 48-edge lookup with one load per k-step)
    constexpr int kPre = 4;
    uint4 wpre[kPre];
    if constexpr (CONV == kConvF16) {
      const uint4* wf = reinterpret_cast<const uint4*>(prm.conv_w) + (size_t)warp * ((CH + 15) / 16) * 32 + lane;
#pragma unroll
      for (int d = 0; d < kPre; ++d) wpre[d] = __ldg(wf + d * 32);
    }
    __syncthreads();
    if (CONV != kConvNone) {
      // ---- corr_encoder[0:2] on the staged tile: enc[oc, pixel] = relu(b[oc] + sum_k W[oc, k] * corr[k, pixel]).
      // Warp w owns output channels 16 w .. 16 w + 15 for all 32 pixels (4 n-tiles of 8 pixels).
      // kConvTF32: 25 k-steps of m16n8k8 TF32 MMAs on register fragments, 3-term split (W = W_hi + W_lo pre-split by lgu_pack_conv1x1, corr = hi + lo split here;
      // lo*lo dropped: ~2^-22 relative per product, fp32 accumulation) -> <= 1e-5 of F.conv2d in fp32 for O(1..10) values.
      // (tcgen05 would want W_hi / W_lo in tensor memory -- 392 of the 512 columns an SM shares between its two resident
      // CTAs -- and UMMA-layout copies of the tile next to a 107 KB TMA ring: neither fits, and 3.7 GFLOP-equivalent per
      // 48-edge lookup is far from the legacy tensor path's limit.)
      // kConvF16 (the backend lookup): what the consumer's conv computes under fp16 autocast (factor_graph.py:281-286) --
      // W and b rounded to fp16 by lgu_pack_conv1x1_f16, the staged corr values rounded to fp16 here (round to nearest
      // even), products exact in fp32, fp32 accumulation, one rounding of the output: 13 k-steps of m16n8k16 MMAs
      // (52 per warp and tile), K padded to 208 with zero rows.  (tcgen05 .kind::f16 with W in tensor memory needs
      // 104 + 32 columns per CTA, which fits; but its B operand is an fp16 UMMA-layout copy of the tile in shared memory:
      // 13,312 B more per CTA is 2 x 120,912 B, beyond the SM's 228 KB at two CTAs, and writing the pass loop's results
      // in that layout instead would change the code every other instantiation shares.)
      float acc[4][4];
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) { acc[nt][0] = acc[nt][1] = acc[nt][2] = acc[nt][3] = 0.0f; }
      const int kq = lane & 3, nq = lane >> 2;
      if constexpr (CONV == kConvF16) {
        constexpr int KS16 = (CH + 15) / 16;                    // 13 k-steps; rows 196..207 are zero
        const uint4* wf = reinterpret_cast<const uint4*>(prm.conv_w) + (size_t)warp * KS16 * 32 + lane;
#pragma unroll
        for (int ks = 0; ks < KS16; ++ks) {
          const uint4 w = wpre[ks % kPre];
          if (ks + kPre < KS16) wpre[ks % kPre] = __ldg(wf + (ks + kPre) * 32);
          const uint32_t a[4] = {w.x, w.y, w.z, w.w};
          // B fragment: rows k0, k0 + 1 (b0) and k0 + 8, k0 + 9 (b1) of pixel column nt * 8 + nq; CH is even, so a pair
          // is either inside the 196 channels or entirely padding
          const int k0 = ks * 16 + 2 * kq, k1 = k0 + 8;
          const bool v0 = k0 < CH, v1 = k1 < CH;
          const float* r0 = s_out + (v0 ? k0 : 0) * kOutPitch + nq;
          const float* r1 = s_out + (v1 ? k1 : 0) * kOutPitch + nq;
#pragma unroll
          for (int nt = 0; nt < 4; ++nt) {
            const uint32_t b0 = v0 ? flf_h2(r0[nt * 8], r0[kOutPitch + nt * 8]) : 0u;
            const uint32_t b1 = v1 ? flf_h2(r1[nt * 8], r1[kOutPitch + nt * 8]) : 0u;
            flf_mma_f16(acc[nt], a, b0, b1);
          }
        }
      } else {
      constexpr int KS = (CH + 7) / 8;                          // 25 k-steps; rows 196..199 are zero
      const float4* wf = prm.conv_w + ((size_t)warp * KS * 32 + lane) * 2;
#pragma unroll 1
      for (int ks = 0; ks < KS; ++ks) {
        const float4 whi = __ldg(wf + (size_t)ks * 64), wlo = __ldg(wf + (size_t)ks * 64 + 1);
        const uint32_t ahi[4] = {__float_as_uint(whi.x), __float_as_uint(whi.y), __float_as_uint(whi.z), __float_as_uint(whi.w)};
        const uint32_t alo[4] = {__float_as_uint(wlo.x), __float_as_uint(wlo.y), __float_as_uint(wlo.z), __float_as_uint(wlo.w)};
        const int k0 = ks * 8 + kq, k1 = k0 + 4;
        const bool v0 = k0 < CH, v1 = k1 < CH;
        const float* r0 = s_out + (v0 ? k0 : 0) * kOutPitch + nq;
        const float* r1 = s_out + (v1 ? k1 : 0) * kOutPitch + nq;
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
          const float x0 = v0 ? r0[nt * 8] : 0.0f, x1 = v1 ? r1[nt * 8] : 0.0f;
          const uint32_t h0 = flf_tf32(x0), h1 = flf_tf32(x1);
          const uint32_t l0 = flf_tf32(x0 - __uint_as_float(h0)), l1 = flf_tf32(x1 - __uint_as_float(h1));
          flf_mma_tf32(acc[nt], alo, h0, h1);                   // small terms first
          flf_mma_tf32(acc[nt], ahi, l0, l1);
          flf_mma_tf32(acc[nt], ahi, h0, h1);
        }
      }
      }
      // C fragment: rows oc0 + nq (c0, c1) and oc0 + nq + 8 (c2, c3), pixels nt * 8 + 2 kq + {0, 1}
      const int p0 = pw - warp * kPixPerWarp;
      const int oc_a = warp * 16 + nq, oc_b = oc_a + 8;
      const float ba = prm.conv_b != nullptr ? __ldg(prm.conv_b + oc_a) : 0.0f;
      const float bb = prm.conv_b != nullptr ? __ldg(prm.conv_b + oc_b) : 0.0f;
      const size_t erow = (size_t)(prm.out_index != nullptr ? __ldg(prm.out_index + n) : n) * 128 * P + p0 + 2 * kq;
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) {
        float e0 = acc[nt][0] + ba, e1 = acc[nt][1] + ba, e2 = acc[nt][2] + bb, e3 = acc[nt][3] + bb;
        if (CONV == kConvF16) {                                 // torch.relu: NaN stays NaN
          e0 = e0 < 0.0f ? 0.0f : e0; e1 = e1 < 0.0f ? 0.0f : e1; e2 = e2 < 0.0f ? 0.0f : e2; e3 = e3 < 0.0f ? 0.0f : e3;
        } else if (prm.conv_relu) {
          e0 = fmaxf(e0, 0.0f); e1 = fmaxf(e1, 0.0f); e2 = fmaxf(e2, 0.0f); e3 = fmaxf(e3, 0.0f);
        }
        if (HALF) {
          __half* enc = reinterpret_cast<__half*>(prm.enc) + erow + nt * 8;
          *reinterpret_cast<__half2*>(enc + (size_t)oc_a * P) = __floats2half2_rn(e0, e1);
          *reinterpret_cast<__half2*>(enc + (size_t)oc_b * P) = __floats2half2_rn(e2, e3);
        } else {
          float* enc = reinterpret_cast<float*>(prm.enc) + erow + nt * 8;
          *reinterpret_cast<float2*>(enc + (size_t)oc_a * P) = make_float2(e0, e1);
          *reinterpret_cast<float2*>(enc + (size_t)oc_b * P) = make_float2(e2, e3);
        }
      }
    }
    if (CONV == kConvNone || prm.out != nullptr) {
      const int p0 = pw - warp * kPixPerWarp;
      const size_t row = (size_t)(prm.out_index != nullptr ? __ldg(prm.out_index + n) : n) * CH * P + p0 + lane;
      const float* srow = s_out + lane;
      if (HALF) {
        __half* out = reinterpret_cast<__half*>(prm.out) + row;
#pragma unroll 4
        for (int ch = warp; ch < CH; ch += kWarps) out[(size_t)ch * P] = __float2half_rn(srow[ch * kOutPitch]);
      } else {
        float* out = reinterpret_cast<float*>(prm.out) + row;
#pragma unroll 4
        for (int ch = warp; ch < CH; ch += kWarps) __stcs(out + (size_t)ch * P, srow[ch * kOutPitch]);
      }
    }
    __syncthreads();                                            // the tile buffer is free for the next tile
    n = nn; pw = npw; ns = nns;
  }
}

}  // namespace lgu

namespace lgu {
struct ConvArgs {
  const float4* w;
  const float* b;
  void* enc;
  int relu;
  int f16;       // 1: fp16 fragments of lgu_pack_conv1x1_f16 (kConvF16), 0: TF32 hi/lo fragments (kConvTF32)
};
static int launch_lookup_fused(const float* lvl0, const float* lvl1, const float* lvl2, const float* lvl3,
                               const float* coords, const float* off0, float* off1, float* corr, float* mask_out, int E,
                               int H, int W, int num_levels, int radius, int per_corner, int shared_offsets,
                               int apply_mask, const int32_t* slots, int num_slots, float* cum_mask,
                               const int32_t* out_index, int out_half, void* stream, const ConvArgs* conv = nullptr,
                               const float* boxes0 = nullptr, const float* boxes1 = nullptr);

// W [128, K] (K <= 200) -> the m16n8k8 A fragments the CONV epilogue reads: [8 warps][25 k-steps][32 lanes]{hi(a0..a3), lo(a0..a3)}
__global__ void pack_conv1x1_kernel(const float* __restrict__ W, float4* __restrict__ frag, int K) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= 8 * 25 * 32) return;
  const int lane = t & 31, ks = (t >> 5) % 25, w = t / (25 * 32);
  const int r0 = w * 16 + (lane >> 2), r1 = r0 + 8, c0 = ks * 8 + (lane & 3), c1 = c0 + 4;
  const float a[4] = {c0 < K ? W[(size_t)r0 * K + c0] : 0.0f, c0 < K ? W[(size_t)r1 * K + c0] : 0.0f,
                      c1 < K ? W[(size_t)r0 * K + c1] : 0.0f, c1 < K ? W[(size_t)r1 * K + c1] : 0.0f};
  float hi[4], lo[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    hi[q] = __uint_as_float(flf_tf32(a[q]));
    lo[q] = __uint_as_float(flf_tf32(a[q] - hi[q]));
  }
  frag[(size_t)t * 2] = make_float4(hi[0], hi[1], hi[2], hi[3]);
  frag[(size_t)t * 2 + 1] = make_float4(lo[0], lo[1], lo[2], lo[3]);
}
}
namespace lgu {
constexpr int kF16FragBytes = 8 * 13 * 32 * 16;                     // 53,248 B; the fp16-rounded bias follows as 128 floats
static_assert(kF16FragBytes + 128 * 4 == LGU_CONV1X1_F16_BYTES, "lgu_corr.h: LGU_CONV1X1_F16_BYTES");
// W [128, K] (K <= 208), b [128] or null -> the m16n8k16 fp16 A fragments of the kConvF16 epilogue, [8 warps][13 k-steps]
// [32 lanes]{a0..a3} (a_r = halves (row, col), (row, col + 1): rows g, g + 8, g, g + 8 and columns 2 t, 2 t, 2 t + 8,
// 2 t + 8 of the warp's 16 x 16 block; g = lane / 4, t = lane % 4), then fp32(fp16(b)) for the 128 channels
__global__ void pack_conv1x1_f16_kernel(const float* __restrict__ W, const float* __restrict__ b, uint4* __restrict__ frag,
                                        float* __restrict__ bias16, int K) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < 128) bias16[t] = b != nullptr ? __half2float(__float2half_rn(b[t])) : 0.0f;
  if (t >= 8 * 13 * 32) return;
  const int lane = t & 31, ks = (t >> 5) % 13, w = t / (13 * 32);
  const int g = lane >> 2, c0 = ks * 16 + 2 * (lane & 3);
  uint32_t r[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const int row = w * 16 + g + (q & 1) * 8, col = c0 + (q >> 1) * 8;
    const float lo = col < K ? W[(size_t)row * K + col] : 0.0f, hi = col + 1 < K ? W[(size_t)row * K + col + 1] : 0.0f;
    const __half2 h = __floats2half2_rn(lo, hi);
    r[q] = *reinterpret_cast<const uint32_t*>(&h);
  }
  frag[t] = make_uint4(r[0], r[1], r[2], r[3]);
}
}  // namespace lgu
extern "C" int lgu_pack_conv1x1_f16(const float* weight, const float* bias, void* packed, int out_channels, int in_channels,
                                    void* stream) {
  LGU_REQUIRE(weight && packed, "lgu_pack_conv1x1_f16: null pointer");
  LGU_REQUIRE((reinterpret_cast<uintptr_t>(packed) & 15) == 0, "lgu_pack_conv1x1_f16: packed must be 16-byte aligned");
  LGU_REQUIRE(out_channels == 128 && in_channels == 196,
              "lgu_pack_conv1x1_f16: only the 196 -> 128 corr_encoder is implemented (got %d -> %d)", in_channels, out_channels);
  uint8_t* p = static_cast<uint8_t*>(packed);
  lgu::pack_conv1x1_f16_kernel<<<(8 * 13 * 32 + 255) / 256, 256, 0, (cudaStream_t)stream>>>(
      weight, bias, reinterpret_cast<uint4*>(p), reinterpret_cast<float*>(p + lgu::kF16FragBytes), in_channels);
  return lgu::check_launch("lgu_pack_conv1x1_f16");
}
extern "C" int lgu_altcorr_lookup_enc_into(const float* boxes0, const float* boxes1, const float* lvl0, const float* lvl1,
                                           const float* lvl2, const float* lvl3, const float* coords, const float* off0,
                                           float* off1, const void* packed, void* enc, const int32_t* out_index, int out_half,
                                           float* mask_out, int E, int H, int W, int num_levels, int radius,
                                           int shared_offsets, int apply_mask, void* stream) {
  LGU_REQUIRE(E >= 0, "lgu_altcorr_lookup_enc_into: bad sizes E=%d", E);
  if (E == 0) return LGU_OK;
  LGU_REQUIRE(packed != nullptr && enc != nullptr, "lgu_altcorr_lookup_enc_into: null pointer");
  LGU_REQUIRE((reinterpret_cast<uintptr_t>(packed) & 15) == 0 && (reinterpret_cast<uintptr_t>(enc) & 7) == 0,
              "lgu_altcorr_lookup_enc_into: packed must be 16-byte and enc 8-byte aligned");
  LGU_REQUIRE(boxes0 != nullptr || lvl0 != nullptr, "lgu_altcorr_lookup_enc_into: null pointer (level 0 needs boxes or a volume)");
  LGU_REQUIRE(boxes1 != nullptr || lvl1 != nullptr, "lgu_altcorr_lookup_enc_into: null pointer (level 1 needs boxes or a volume)");
  const uint8_t* p = static_cast<const uint8_t*>(packed);
  const lgu::ConvArgs conv = {reinterpret_cast<const float4*>(p), reinterpret_cast<const float*>(p + lgu::kF16FragBytes), enc,
                              1, 1};
  return lgu::launch_lookup_fused(boxes0 != nullptr ? nullptr : lvl0, lvl1, lvl2, lvl3, coords, off0, off1, nullptr,
                                  mask_out, E, H, W, num_levels, radius, 1, shared_offsets, apply_mask, nullptr, E, nullptr,
                                  out_index, out_half, stream, &conv, boxes0, boxes1);
}
extern "C" int lgu_pack_conv1x1(const float* weight, float* wfrag, int out_channels, int in_channels, void* stream) {
  LGU_REQUIRE(weight && wfrag, "lgu_pack_conv1x1: null pointer");
  LGU_REQUIRE(out_channels == 128 && in_channels == 196, "lgu_pack_conv1x1: only the 196 -> 128 corr_encoder is implemented");
  lgu::pack_conv1x1_kernel<<<(8 * 25 * 32 + 255) / 256, 256, 0, (cudaStream_t)stream>>>(
      weight, reinterpret_cast<float4*>(wfrag), in_channels);
  return lgu::check_launch("lgu_pack_conv1x1");
}
extern "C" int lgu_corr_lookup_fused_enc(const float* lvl0, const float* lvl1, const float* lvl2, const float* lvl3,
                                         const float* coords, const float* off0, const float* off1, float* cum_mask,
                                         float* corr, void* enc, const float* wfrag, const float* bias, int relu,
                                         int out_half, float* mask_out, const int32_t* slots, int num_slots, int E, int H,
                                         int W, int num_levels, int radius, void* stream) {
  LGU_REQUIRE(E == 0 || (cum_mask != nullptr && enc != nullptr && wfrag != nullptr), "lgu_corr_lookup_fused_enc: null pointer");
  LGU_REQUIRE(slots == nullptr || num_slots > 0, "lgu_corr_lookup_fused_enc: bad pool size %d", num_slots);
  LGU_REQUIRE((reinterpret_cast<uintptr_t>(wfrag) & 15) == 0 && (reinterpret_cast<uintptr_t>(enc) & 7) == 0,
              "lgu_corr_lookup_fused_enc: wfrag must be 16-byte and enc 8-byte aligned");
  LGU_REQUIRE(!(out_half && corr != nullptr), "lgu_corr_lookup_fused_enc: fp16 output applies to enc only (pass corr = NULL)");
  const lgu::ConvArgs conv = {reinterpret_cast<const float4*>(wfrag), bias, enc, relu, 0};
  return lgu::launch_lookup_fused(lvl0, lvl1, lvl2, lvl3, coords, off0, const_cast<float*>(off1), corr, mask_out, E, H, W,
                                  num_levels, radius, 0, 0, 1, slots, slots != nullptr ? num_slots : E, cum_mask, nullptr,
                                  out_half, stream, &conv);
}
extern "C" int lgu_corr_lookup_fused(const float* lvl0, const float* lvl1, const float* lvl2, const float* lvl3,
                                     const float* coords, const float* off0, float* off1, float* corr, float* mask_out,
                                     int E, int H, int W, int num_levels, int radius, void* stream) {
  return lgu::launch_lookup_fused(lvl0, lvl1, lvl2, lvl3, coords, off0, off1, corr, mask_out, E, H, W, num_levels,
                                  radius, 0, 0, 1, nullptr, E, nullptr, nullptr, 0, stream);
}
extern "C" int lgu_corr_lookup_fused_cum(const float* lvl0, const float* lvl1, const float* lvl2, const float* lvl3,
                                         const float* coords, const float* off0, const float* off1, float* cum_mask,
                                         float* corr, float* mask_out, const int32_t* slots, int num_slots, int E, int H,
                                         int W, int num_levels, int radius, void* stream) {
  LGU_REQUIRE(E == 0 || cum_mask != nullptr, "lgu_corr_lookup_fused_cum: null cumulative-mask buffer");
  LGU_REQUIRE(slots == nullptr || num_slots > 0, "lgu_corr_lookup_fused_cum: bad pool size %d", num_slots);
  return lgu::launch_lookup_fused(lvl0, lvl1, lvl2, lvl3, coords, off0, const_cast<float*>(off1), corr, mask_out, E, H, W,
                                  num_levels, radius, 0, 0, 1, slots, slots != nullptr ? num_slots : E, cum_mask, nullptr, 0, stream);
}
extern "C" int lgu_corr_lookup_fused_slots(const float* lvl0, const float* lvl1, const float* lvl2, const float* lvl3,
                                           const float* coords, const float* off0, float* off1, float* corr,
                                           float* mask_out, const int32_t* slots, int num_slots, int E, int H, int W,
                                           int num_levels, int radius, void* stream) {
  LGU_REQUIRE(E == 0 || slots != nullptr, "lgu_corr_lookup_fused_slots: null slot list");
  LGU_REQUIRE(num_slots > 0, "lgu_corr_lookup_fused_slots: bad pool size %d", num_slots);
  return lgu::launch_lookup_fused(lvl0, lvl1, lvl2, lvl3, coords, off0, off1, corr, mask_out, E, H, W, num_levels,
                                  radius, 0, 0, 1, slots, num_slots, nullptr, nullptr, 0, stream);
}
extern "C" int lgu_altcorr_lookup_fused(const float* lvl0, const float* lvl1, const float* lvl2, const float* lvl3,
                                        const float* coords, const float* off0, float* off1, float* corr,
                                        float* mask_out, int E, int H, int W, int num_levels, int radius,
                                        int shared_offsets, int apply_mask, void* stream) {
  return lgu::launch_lookup_fused(lvl0, lvl1, lvl2, lvl3, coords, off0, off1, corr, mask_out, E, H, W, num_levels,
                                  radius, 1, shared_offsets, apply_mask, nullptr, E, nullptr, nullptr, 0, stream);
}
extern "C" int lgu_altcorr_lookup_fused_into(const float* lvl0, const float* lvl1, const float* lvl2, const float* lvl3,
                                             const float* coords, const float* off0, float* off1, void* corr,
                                             const int32_t* out_index, int out_half, float* mask_out, int E, int H, int W,
                                             int num_levels, int radius, int shared_offsets, int apply_mask,
                                             void* stream) {
  return lgu::launch_lookup_fused(lvl0, lvl1, lvl2, lvl3, coords, off0, off1, reinterpret_cast<float*>(corr), mask_out, E,
                                  H, W, num_levels, radius, 1, shared_offsets, apply_mask, nullptr, E, nullptr, out_index,
                                  out_half, stream);
}
// The backend lookup with level 0 held as COMPACT per-pixel boxes (lgu_build_boxes) instead of a volume.
extern "C" int lgu_altcorr_lookup_boxes_into(const float* boxes0, const float* boxes1, const float* lvl1, const float* lvl2,
                                             const float* lvl3, const float* coords, const float* off0, float* off1,
                                             void* corr, const int32_t* out_index, int out_half, float* mask_out, int E,
                                             int H, int W, int num_levels, int radius, int shared_offsets, int apply_mask,
                                             void* stream) {
  LGU_REQUIRE(E == 0 || boxes0 != nullptr, "lgu_altcorr_lookup_boxes_into: null boxes");
  LGU_REQUIRE(E == 0 || boxes1 != nullptr || lvl1 != nullptr, "lgu_altcorr_lookup_boxes_into: level 1 needs boxes or a volume");
  return lgu::launch_lookup_fused(nullptr, lvl1, lvl2, lvl3, coords, off0, off1, reinterpret_cast<float*>(corr), mask_out, E,
                                  H, W, num_levels, radius, 1, shared_offsets, apply_mask, nullptr, E, nullptr, out_index,
                                  out_half, stream, nullptr, boxes0, boxes1);
}
static int lgu::launch_lookup_fused(const float* lvl0, const float* lvl1, const float* lvl2, const float* lvl3,
                                    const float* coords, const float* off0, float* off1, float* corr, float* mask_out,
                                    int E, int H, int W, int num_levels, int radius, int per_corner,
                                    int shared_offsets, int apply_mask, const int32_t* slots, int num_slots,
                                    float* cum_mask, const int32_t* out_index, int out_half, void* stream,
                                    const ConvArgs* conv, const float* boxes0, const float* boxes1) {
  using namespace lgu;
  if (E == 0) return LGU_OK;
  if (boxes1 != nullptr && lvl1 == nullptr) lvl1 = lvl2;    // compact levels: no volume behind them (their maps are unused)
  if (boxes0 != nullptr) lvl0 = lvl1;
  LGU_REQUIRE(boxes1 == nullptr || boxes0 != nullptr, "lgu_corr_lookup_fused: compact level 1 needs compact level 0");
  LGU_REQUIRE((reinterpret_cast<uintptr_t>(boxes1) & 15) == 0, "lgu_corr_lookup_fused: boxes are not 16-byte aligned");
  LGU_REQUIRE(lvl0 && lvl1 && lvl2 && lvl3 && coords && off0 && off1 && (corr || conv), "lgu_corr_lookup_fused: null pointer");
  LGU_REQUIRE((reinterpret_cast<uintptr_t>(boxes0) & 15) == 0, "lgu_corr_lookup_fused: boxes are not 16-byte aligned");
  LGU_REQUIRE(boxes0 == nullptr || (per_corner && slots == nullptr), "lgu_corr_lookup_fused: compact boxes serve the backend lookup only");
  LGU_REQUIRE(E > 0 && H > 0 && W > 0, "lgu_corr_lookup_fused: bad sizes E=%d H=%d W=%d", E, H, W);
  if (num_levels != 4 || radius != 3 || (W % 32) != 0 || (H % 8) != 0) {
    set_error("lgu_corr_lookup_fused: only num_levels=4, radius=3, W%%32==0, H%%8==0 are implemented "
              "(got levels=%d r=%d H=%d W=%d); use the per-level operators", num_levels, radius, H, W);
    return LGU_ERR_UNSUPPORTED;
  }
  const int P = H * W;
  const long long nslices = (long long)num_slots * P;        // slices held by the storage (== E without a pool)
  LGU_REQUIRE(nslices < 2147483647LL, "lgu_corr_lookup_fused: slots*H*W = %lld exceeds the TMA coordinate range", nslices);
  const float* lv[4] = {lvl0, lvl1, lvl2, lvl3};
  for (int l = 0; l < 4; ++l)
    LGU_REQUIRE((reinterpret_cast<uintptr_t>(lv[l]) & 15) == 0, "lgu_corr_lookup_fused: level %d is not 16-byte aligned", l);
  // the tile inputs travel by cp.async.bulk: 16-byte aligned sources (always true for whole torch tensors)
  LGU_REQUIRE(((reinterpret_cast<uintptr_t>(coords) | reinterpret_cast<uintptr_t>(off0) | reinterpret_cast<uintptr_t>(off1) |
                reinterpret_cast<uintptr_t>(cum_mask)) & 15) == 0,
              "lgu_corr_lookup_fused: coords / offsets / cum_mask must be 16-byte aligned");
  FusedMaps maps;
  FusedLookupParams prm;
  for (int l = 0; l < 4; ++l) {
    prm.lvl[l] = lv[l];
    prm.H2[l] = H >> l;
    prm.W2[l] = W >> l;
    if ((l == 0 && boxes0 != nullptr) || (l == 1 && boxes1 != nullptr)) continue;
    const int rc = make_slice_map(&maps.m[l], lv[l], nslices, H >> l, W >> l, l < 2 ? fl::kBW01 : fl::kBW23,
                                  l < 2 ? fl::kBH01 : fl::kBH23);
    if (rc) return rc;
  }
  if (boxes1 != nullptr) maps.m[1] = maps.m[2];
  if (boxes0 != nullptr) maps.m[0] = maps.m[1];
  prm.boxes0 = boxes0;
  prm.boxes1 = boxes1;
  prm.coords = coords; prm.off0 = off0; prm.off1 = off1; prm.out = corr; prm.mask_out = mask_out;
  prm.cum_mask = cum_mask;
  prm.out_index = out_index;
  prm.conv_w = conv ? conv->w : nullptr; prm.conv_b = conv ? conv->b : nullptr; prm.enc = conv ? conv->enc : nullptr;
  prm.conv_relu = conv ? conv->relu : 0;
  prm.P = P;
  prm.tiles_per_edge = P / fl::kTile;                         // W % 32 == 0: tiles are always full
  const long long ntiles = (long long)E * prm.tiles_per_edge;
  LGU_REQUIRE(ntiles < 2147483647LL, "lgu_corr_lookup_fused: too many tiles (%lld)", ntiles);
  prm.num_tiles = (int)ntiles;
  const int sms = num_sms();
  const long long nblk = ntiles < 2LL * sms ? ntiles : 2LL * sms;   // persistent: two CTAs per SM (an equal-tiles grid of
                                                                     // 288 CTAs was measured: 169.0 vs 167.9 us)
  prm.off_edge_stride = shared_offsets ? 0 : (long long)P * fl::TAPS;
  prm.apply_mask = apply_mask;
  prm.slots = slots;
  LGU_REQUIRE(!(shared_offsets && apply_mask), "lgu_*_lookup_fused: apply_mask needs per-edge offsets");
  auto kern = per_corner ? (out_half ? lookup_fused_kernel<true, true> : lookup_fused_kernel<true, false>)
                         : (out_half ? lookup_fused_kernel<false, true> : lookup_fused_kernel<false, false>);
  if (conv != nullptr && conv->f16) {
    LGU_REQUIRE(per_corner, "lgu_*_lookup_enc: the fp16 encoder is implemented for the backend lookup");
    kern = out_half ? lookup_fused_kernel<true, true, kConvF16> : lookup_fused_kernel<true, false, kConvF16>;
  } else if (conv != nullptr) {
    LGU_REQUIRE(!per_corner, "lgu_corr_lookup_fused_enc: the fused encoder is implemented for the CorrBlock lookup");
    kern = out_half ? lookup_fused_kernel<false, true, kConvTF32> : lookup_fused_kernel<false, false, kConvTF32>;
  }
  if (int rc = optin_smem(reinterpret_cast<const void*>(kern), flf::kFwdSmemBytes, "lgu_corr_lookup_fused")) return rc;
  kern<<<(unsigned)nblk, fl::kThreads, flf::kFwdSmemBytes, (cudaStream_t)stream>>>(maps, prm);
  return check_launch("lgu_corr_lookup_fused");
}

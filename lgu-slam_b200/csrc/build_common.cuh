// build_common.cuh -- parameter block and Gaussian residual shared by build_pyramid.cu (8 epilogue warps; every
// precision / flat volumes) and build_pyramid16.cu (16 epilogue warps; the fp16-input pyramid build).
#pragma once
#include "tc_common.cuh"

namespace lgu {

constexpr int kTileM = 128;      // source pixels per unit
constexpr int kChunkN = 128;     // target pixels per MMA chunk (2 target rows of 64)
constexpr int kC = 128;          // channels (K)
constexpr int kAtomBytes = 128 * 128;   // one 64-channel swizzle atom column of a 128-row tile: 16 KB
constexpr int kPlaneBytes = 2 * kAtomBytes;   // 128 rows x 128 ch fp16 = 32 KB

struct BpParams {
  const int32_t* ii;
  const int32_t* jj;
  const float* means;   // [E,P,2] or null
  const float* covs;    // [E,P,2]
  const float* den;     // [E,P]
  float* lvl0;          // [E,P,Q] (stored to directly by the 16-warp kernel; the 8-warp kernel stores through its TMA map)
  float* lvl1;          // [E,P,Q/4] or null (as lvl0)
  float* lvl2;          // [E,P,Q/16] or null
  float* lvl3;          // [E,P,Q/64] or null
  int E, P, H, gauss_radius, round_half, num_units, has_l1;
  const int32_t* out_slots;   // [E] or null: edge e is written to pyramid slot out_slots[e] (edge-slot pool)
  int Q;        // target pixels per map (== P for the pyramid build; any multiple of 4 in flat volume mode)
  int halves;   // 256-column accumulator halves per unit: ceil(Q / 256)
  const uint32_t* half_mask;   // [num_units] or null: bit h set = accumulator half h (256 target columns) of the unit is built
  int box_W, box_level;       // compact mode: columns of the target grid (64 or 32) and the level the coords are halved to
  float* boxes;               // FLAT 16-warp kernel: [E,P,16,20] or null -- write each source pixel's lookup box (rows
  const float* box_coords;    //   box_origin_y(floor(cy),7,H) .. +15, cols box_origin_x(floor(cx),7,64) .. +19 around box_coords [E,P,2],
                              //   zeros outside the target grid) INSTEAD of the volume rows (lgu_build_boxes)
};

// Gaussian residual of one element (gaussianAttn.cu:58-64 + gaussianMask_cuda.py:85-86), fp32, no contraction.
__device__ __forceinline__ float gauss_residual(float v, int x1, int y1, float mx, float my, float c1, float c2,
                                                float den) {
  const float ddx = __fsub_rn((float)x1, mx), ddy = __fsub_rn((float)y1, my);
  const float t1 = __fdiv_rn(ddx, c1), t2 = __fdiv_rn(ddy, c2);
  const float s = __fmaf_rn(ddy, t2, __fmul_rn(t1, ddx));
  const float e = expf(__fmul_rn(s, -0.5f));
  const float masked = __fmul_rn(__fmul_rn(v, 3.0f), e);
  return __fadd_rn(__fdiv_rn(masked, den), v);
}

// (Forming the row-invariant ddy / cov_y once per window row instead of per tap was measured: 542 -> 553 us, reverted.)

// The 16-epilogue-warp kernel (build_pyramid16.cu).  Returns LGU_OK / an error code.
int launch_build16(const CUtensorMap& mh, const CUtensorMap& mb, const BpParams& prm, bool flat, cudaStream_t st);

}  // namespace lgu

// common.cuh -- shared helpers for the sm_100a correlation kernels.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/lgu_corr.h"

namespace lgu {

// Thread-local error text behind lgu_last_error_string().
void set_error(const char* fmt, ...);

#define LGU_REQUIRE(cond, ...)                 \
  do {                                         \
    if (!(cond)) {                             \
      ::lgu::set_error(__VA_ARGS__);           \
      return LGU_ERR_BAD_ARG;                  \
    }                                          \
  } while (0)

// Check the launch that was just issued (async errors surface at the caller's next sync).
int check_launch(const char* what);

constexpr int kNumSMs = 148;  // B200: 2 dies x 74 SMs

// Host-side launch plumbing that is paid ONCE, not per call (abi.cu):
//  * the opt-in to more than 48 KB of dynamic shared memory is a per-(device, kernel) function attribute;
//  * a CUtensorMap depends only on the device and the encoder's arguments: encoded maps are kept in a small table, so the
//    steady state of a frontend / backend loop (same pyramid storage, same shapes) re-encodes nothing;
//  * the SM count that sizes the persistent grids is read once per device (kNumSMs if the query fails).
int optin_smem(const void* kernel, int bytes, const char* who);
// Tiled map of a tensor of rank <= 5: dims innermost first, strides_bytes of dims 1 .. rank-1, element strides 1, no
// interleave, out-of-bounds elements read as zero.
int encode_tensor_map(CUtensorMap* map, CUtensorMapDataType dt, int rank, const void* base, const uint64_t* dims,
                      const uint64_t* strides_bytes, const uint32_t* box, CUtensorMapSwizzle swz, CUtensorMapL2promotion l2);
int num_sms();

__device__ __forceinline__ bool in_bounds(int h, int w, int H, int W) {
  return h >= 0 && h < H && w >= 0 && w < W;
}
// Tap coordinate `base - r + k` with the two's-complement wrap the reference's SASS has
// (signed overflow would be UB in C++; saturated float->int bases do reach INT_MAX/INT_MIN).
__device__ __forceinline__ int tap_coord(int base, int r, int k) {
  return (int)((unsigned)base - (unsigned)r + (unsigned)k);
}
__device__ __forceinline__ int wrap_inc(int v) { return (int)((unsigned)v + 1u); }

// floor(v) as int with F2I.FLOOR semantics (saturating, NaN -> 0), like `int f = floor(v)`
// in the reference (defCorrSample_kernel.cu:58-59).
__device__ __forceinline__ int floor_to_int(float v) { return __float2int_rd(v); }

// Bilinear blend in the exact operation order of the reference's sm_100 SASS
// (FMUL w21*Q21, then three FFMAs: Q11*w11, w12*Q12, w22*Q22); intrinsics are never
// re-contracted by nvcc, which keeps the forward lookups bit-exact with the reference.
__device__ __forceinline__ float blend4(float q11, float q21, float q12, float q22, float dx, float dy) {
  const float omdy = __fsub_rn(1.0f, dy), omdx = __fsub_rn(1.0f, dx);
  const float w22 = __fmul_rn(dx, dy);
  const float w21 = __fmul_rn(dx, omdy);
  const float w12 = __fmul_rn(dy, omdx);
  const float w11 = __fmul_rn(omdy, omdx);
  float acc = __fmul_rn(w21, q21);
  acc = __fmaf_rn(q11, w11, acc);
  acc = __fmaf_rn(w12, q12, acc);
  acc = __fmaf_rn(w22, q22, acc);
  return acc;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

}  // namespace lgu

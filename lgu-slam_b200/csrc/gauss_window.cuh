// gauss_window.cuh -- the per-pixel arithmetic of the Gaussian head's backward for the reference's only radius
// (r = 4, a 9 x 9 window; gaussianAttn.cu:72-131, gaussianMask_cuda.py:77-86), shared by gaussian_bwd_sep_kernel
// (gaussian.cu) and the fused lookup backward (lookup_fused_bwd.cu) so that both produce the same bits.
//
// One warp, one pixel.  Lane = tap (t = 32 ps + lane, x fastest: column ti = t % 9, row tj = t / 9) in three passes; v[ps],
// g[ps] hold this lane's window values of the volume and of its upstream gradient (anything finite for out-of-range
// taps: their records are zero).  The Gaussian is separable, e(i,j) = ex(i) ey(j), and so is every factor the reference
// forms from it (gaussianAttn.cu:112-126):
//     d/dmean_x : 3 V g * [ex(i) ddx(i) / cx] * ey(j)          d/dcov_x : 3 V g * [0.5 ex(i) ddx(i)^2 / cx^2] * ey(j)
//     d/dmean_y : 3 V g * ex(i) * [ey(j) ddy(j) / cy]          d/dcov_y : 3 V g * ex(i) * [0.5 ey(j) ddy(j)^2 / cy^2]
// Lanes 0-8 evaluate the 9 COLUMN records, lanes 9-17 the 9 ROW records (one expf each; the fp64 factor of the reference,
// :120,122, 18 times per pixel instead of 162); records of out-of-range columns / rows are zero, which is the reference's
// bounds gate.  The two records of a tap arrive by shuffle, a tap costs 2 multiplies and 4 FMAs, and the four sums are
// reduced with a value-splitting butterfly (6 shuffles instead of 20).  Differences from the reference's per-tap
// evaluation are products of correctly rounded factors in another order (a few 1e-7 relative), inside the 1e-5 bar.
// FUSED: v is the MASKED level-0 volume V (1 + 3 e / den) and g the gradient with respect to it; the raw volume is
// recovered per tap, every parameter gradient carries 1/den, and the gradient of den is produced as well.
// Results are valid on lane 0.
#pragma once
#include "common.cuh"

namespace lgu {

template <bool FUSED>
__device__ __forceinline__ void gauss_window_grads(const float (&v)[3], const float (&g)[3], float2 m, float2 c, float dn,
                                                   int x0, int y0, int H2, int W2, int lane, float& o0, float& o1,
                                                   float& o2, float& o3, float& od) {
  constexpr int rd = 9, taps = 81, kPasses = 3;
  const bool is_row = lane >= rd;                               // lanes 9..17 (18..31 compute unused duplicates)
  const int kidx = (lane < rd ? lane : lane - rd) % rd;
  // ---- this lane's record: column kidx (lanes 0-8) or row kidx (lanes 9-17)
  const float mean_a = is_row ? m.y : m.x, cov_a = is_row ? c.y : c.x;
  const int coord = tap_coord(is_row ? y0 : x0, 0, kidx);
  const bool inb = (unsigned)coord < (unsigned)(is_row ? H2 : W2);
  const float rc = __fdiv_rn(1.0f, cov_a);
  const float dd = __fsub_rn((float)coord, mean_a);
  const float ev = expf(__fmul_rn(__fmul_rn(__fmul_rn(dd, rc), dd), -0.5f));
  const float recE = inb ? ev : 0.0f;                                                      // e
  const float recM = inb ? __fmul_rn(__fmul_rn(dd, ev), rc) : 0.0f;                        // e dd / cov
  // 0.5 e dd^2 / cov^2 in fp64 like the reference (:120,122), with the correctly rounded fp32 reciprocal of cov^2
  const float recC = inb ? (float)(((((double)ev * 0.5) * (double)dd) * (double)dd) * (double)__fmul_rn(rc, rc)) : 0.0f;
  float k3 = 0.0f, rdn = 1.0f;
  if (FUSED) {
    rdn = __fdiv_rn(1.0f, dn);
    k3 = __fmul_rn(3.0f, rdn);                                  // lvl0 = V (1 + 3 ex ey / den) inside the window
  }
  float gm0 = 0.0f, gm1 = 0.0f, gc0 = 0.0f, gc1 = 0.0f, gd = 0.0f;
#pragma unroll
  for (int ps = 0; ps < kPasses; ++ps) {
    const int t = min(ps * 32 + lane, taps - 1);
    const int tj = t / rd, ti = t - tj * rd;
    const float cE = __shfl_sync(0xffffffffu, recE, ti), cM = __shfl_sync(0xffffffffu, recM, ti);
    const float cC = __shfl_sync(0xffffffffu, recC, ti);
    const float rE = __shfl_sync(0xffffffffu, recE, rd + tj), rM = __shfl_sync(0xffffffffu, recM, rd + tj);
    const float rC = __shfl_sync(0xffffffffu, recC, rd + tj);
    const bool live = ps * 32 + lane < taps;
    float vraw = v[ps];
    if (FUSED) {
      vraw = __fdividef(v[ps], __fmaf_rn(__fmul_rn(k3, cE), rE, 1.0f));   // the raw volume (== v outside the window)
      // the residual corr1 / den = v - vraw, formed as vraw 3 e / den: the difference cancels to a few bits where e is
      // small (a window far from its mean keeps 2^-24 / (3 e / den) of its relative accuracy)
      if (live) gd = __fmaf_rn(g[ps], __fmul_rn(vraw, __fmul_rn(__fmul_rn(k3, cE), rE)), gd);
    }
    const float w = live ? __fmul_rn(__fmul_rn(vraw, 3.0f), g[ps]) : 0.0f;
    const float wa = __fmul_rn(w, rE), wb = __fmul_rn(w, cE);
    gm0 = __fmaf_rn(wa, cM, gm0);
    gc0 = __fmaf_rn(wa, cC, gc0);
    gm1 = __fmaf_rn(wb, rM, gm1);
    gc1 = __fmaf_rn(wb, rC, gc1);
  }
  // ---- reduce (gm0, gm1, gc0, gc1) over the warp with a value-splitting butterfly: 2 + 1 + 3 shuffles
  float t;
  {
    const bool hi16 = (lane & 16) != 0, hi8 = (lane & 8) != 0;
    const float s0 = hi16 ? gm0 : gc0, s1 = hi16 ? gm1 : gc1;              // what this lane sends
    const float k0 = hi16 ? gc0 : gm0, k1 = hi16 ? gc1 : gm1;              // what it keeps
    const float a0 = k0 + __shfl_xor_sync(0xffffffffu, s0, 16), a1 = k1 + __shfl_xor_sync(0xffffffffu, s1, 16);
    t = (hi8 ? a1 : a0) + __shfl_xor_sync(0xffffffffu, hi8 ? a0 : a1, 8);
    t += __shfl_xor_sync(0xffffffffu, t, 4);
    t += __shfl_xor_sync(0xffffffffu, t, 2);
    t += __shfl_xor_sync(0xffffffffu, t, 1);                               // lane 0: gm0, 8: gm1, 16: gc0, 24: gc1
  }
  if (FUSED) gd = warp_sum(gd);
  const float r1 = __shfl_sync(0xffffffffu, t, 8), r2 = __shfl_sync(0xffffffffu, t, 16), r3 = __shfl_sync(0xffffffffu, t, 24);
  o0 = t; o1 = r1; o2 = r2; o3 = r3; od = 0.0f;
  if (FUSED) {                                                  // g / den enters every parameter gradient linearly
    o0 = __fmul_rn(o0, rdn); o1 = __fmul_rn(o1, rdn); o2 = __fmul_rn(o2, rdn); o3 = __fmul_rn(o3, rdn);
    od = -__fmul_rn(gd, rdn);
  }
}

}  // namespace lgu

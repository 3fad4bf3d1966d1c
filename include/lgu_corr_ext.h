/*
 * lgu_corr_ext.h -- entry points added to the C ABI after its version-1 set.
 *
 * lgu_corr.h is the version-1 set of entry points, and the binding's table of it (SIGNATURES in
 * lgu-slam_b200/_lib.py) is kept exactly as released.  Entry points added since are declared here, bound from
 * EXT_SIGNATURES, and follow every convention of lgu_corr.h (raw device pointers, int sizes, the stream last, an
 * LGU_OK / LGU_ERR_* status, nothing allocated or synchronised by the library).  Adding an entry point changes no
 * existing signature, so lgu_abi_version() stays 1.
 */
#ifndef LGU_CORR_EXT_H_
#define LGU_CORR_EXT_H_

#include "lgu_corr.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Backward of lgu_offset_heads (lgu_corr.h; what autograd runs for the offset heads' glue when the heads are trained),
 * in two launches.
 * With z0 = (c0 - mean0) / sigma0, t0 = tanh(z0), z1 = (up(c1) - mean1) / sigma1, t1 = tanh(z1) RECOMPUTED from c0, c1
 * and the forward's stats with the forward's fp32 arithmetic, and G0 = g_off0, G1 = g_off1 ([E,H,W,CH], channels-last):
 *   gz0 = 4 (G0 + G1/2) (1 - t0^2),   gz1 = 2 G1 (1 - t1^2)                               (per hi-res element)
 *   g_c0      = (gz0 - mean(gz0) - z0 mean(gz0 z0)) / sigma0
 *   g_c1[k]   = (S_k - 4 mean(gz1) - 4 z1_k mean(gz1 z1)) / sigma1,  S_k = sum of gz1 over the 4 hi-res copies of c1[k]
 * means per edge over its N0 = CH*H*W hi-res elements.  g_c0 [E,CH,H,W], g_c1 [E,CH,H/2,W/2] (NCHW, the conv outputs'
 * layout) are fully written.  g_off0 or g_off1 may be NULL (a zero gradient).  scratch: device memory for the per-edge
 * sums, E*(H/2)*(W/32)*4 doubles, 8-byte aligned, contents undefined on entry and exit.
 * Determinism: the sums are accumulated in fp64 per tile and added in a fixed order, every output element is written
 * once by one thread, no atomics -- results are bit-identical from run to run.  A NaN in one edge stays in that edge.
 * Shapes as the forward (CH <= 128, W % 32 == 0, H even); LGU_ERR_BAD_ARG names a null pointer or bad size before any
 * device work; E = 0 is a no-op. */
LGU_API int lgu_offset_heads_backward(const float* c0, const float* c1, const float* stats, const float* g_off0,
                              const float* g_off1, float* g_c0, float* g_c1, double* scratch,
                              int E, int CH, int H, int W, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* LGU_CORR_EXT_H_ */

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

/* The offset heads' 3x3 convolutions (ofsMap / ofs_residual: nn.Conv2d(C_in, C_out, 3, padding=1), stride 1, zero
 * padding, bias) and their input and weight gradients, in fp32 accuracy on tensor cores: every product is
 * hi*hi + hi*lo + lo*hi of tf32 hi / lo splits (~2^-21 relative), accumulated in fp32 in chunks of K = 128.
 * Activations and gradients are NCHW fp32; the weight is [C_out, C_in, 3, 3] as nn.Conv2d holds it, packed by each
 * call.  Sizes, checked by every entry point: C_in % 32 == 0, 0 < C_out <= 128, W % 32 == 0 with W dividing 128 or a
 * multiple of 128, H*W % 128 == 0, E >= 0.  LGU_ERR_BAD_ARG names a NULL or misaligned pointer, a bad size or a short
 * workspace before any device work; E = 0 is a no-op.  No float atomics: results are bit-identical from run to run. */

/* Workspace bytes that any of the three operations below needs at these sizes (-1 for unsupported sizes). */
LGU_API long long lgu_conv3x3_workspace_bytes(int E, int C_in, int C_out, int H, int W);

/* x [E,C,H,W] -> tf32 hi / lo planes [E,H,W,Cp], channels-last, Cp = C rounded up to 32, padded channels 0.
 * hi = x with the low 13 mantissa bits cleared, lo = x - hi; a +-inf or NaN x gives hi = 0, lo = x.
 * hi, lo 16-byte aligned.  The forward packs x (C = C_in), the input gradient packs g_y (C = C_out). */
LGU_API int lgu_conv3x3_pack(const float* x, float* hi, float* lo, int E, int C, int H, int W, void* stream);

/* y [E,C_out,H,W] = conv3x3(x, weight) + bias, from x's planes (lgu_conv3x3_pack).  bias may be NULL (no bias).
 * workspace: lgu_conv3x3_workspace_bytes, 256-byte aligned. */
LGU_API int lgu_conv3x3_forward(const float* x_hi, const float* x_lo, const float* weight, const float* bias, float* y,
                                void* workspace, long long workspace_bytes, int E, int C_in, int C_out, int H, int W,
                                void* stream);

/* g_x [E,C_in,H,W] = conv3x3(g_y, weight flipped and transposed), from g_y's planes (lgu_conv3x3_pack, C = C_out). */
LGU_API int lgu_conv3x3_backward_input(const float* gy_hi, const float* gy_lo, const float* weight, float* g_x,
                                       void* workspace, long long workspace_bytes, int E, int C_in, int C_out, int H,
                                       int W, void* stream);

/* g_w [C_out,C_in,3,3] = sum over e, y, x of g_y[e,co,y,x] x[e,ci,y+ky-1,x+kx-1] (x's planes from lgu_conv3x3_pack) and
 * g_b [C_out] = sum of g_y over e, y, x (in fp64).  Either g_w or g_b may be NULL (not computed), not both; x_hi, x_lo
 * and the workspace are read only for g_w.  The pixel sum is split over CTAs by a partition that depends only on the
 * sizes, and the partial sums are added in a fixed order. */
LGU_API int lgu_conv3x3_backward_weight(const float* x_hi, const float* x_lo, const float* g_y, float* g_w, float* g_b,
                                        void* workspace, long long workspace_bytes, int E, int C_in, int C_out, int H,
                                        int W, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* LGU_CORR_EXT_H_ */

/*
 * lgu_corr.h -- C ABI of the B200-native LGU-SLAM correlation hot path.
 *
 * Every entry point takes raw DEVICE pointers, plain integer sizes and a CUDA
 * stream (passed as void* so that this header needs no CUDA include); nothing
 * in the signatures depends on torch.  All tensors are contiguous, fp32 unless
 * stated otherwise.  Return value: 0 on success, one of LGU_ERR_* otherwise;
 * lgu_last_error_string() describes the most recent failure on the calling
 * thread.  Kernels are launched asynchronously on `stream`; nothing is
 * allocated, retained or synchronised by the library (workspace, if any, is
 * supplied by the caller).
 *
 * Each function replaces one operator of the reference's torch extension
 * `defCorrSample` (binding: /root/reference/offersample_LGS/droid.cpp:138-147);
 * the reference interface it replaces is cited per function.  Index / bounds
 * logic is bit-exact with the reference kernels, including their quirks
 * (x-major taps, top-left-corner gating, in-place zeroing of the centre
 * offset tap; SURVEY.md section 8 Q1-Q12).
 *
 * Layout vocabulary:  E = edges (frame pairs), (H1,W1) = source grid,
 * (H2,W2) = target grid of this pyramid level, r = lookup radius, rd = 2r+1.
 *   volume   [E,H1,W1,H2,W2]      one private H2xW2 slice per source pixel
 *   coords   [E,2,H1,W1]          channel 0 = x, channel 1 = y (level units)
 *   offset   [E,H1,W1,rd,rd,2]    [..,i,j,0] = x-offset of tap (i: x, j: y)
 *   corr     [E,rd,rd,H1,W1]      tap-major output, i (x tap) outermost
 */
#ifndef LGU_CORR_H_
#define LGU_CORR_H_

#include <stdint.h>

#if defined(LGU_BUILDING) && defined(__GNUC__)
#define LGU_API __attribute__((visibility("default")))
#else
#define LGU_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

#define LGU_OK 0
#define LGU_ERR_BAD_ARG 1      /* null pointer, non-positive size, unsupported radius/shape */
#define LGU_ERR_LAUNCH 2       /* cudaGetLastError() after a launch was not cudaSuccess */
#define LGU_ERR_UNSUPPORTED 3  /* valid arguments the sm_100a build does not implement */

/* Library / build identification. */
LGU_API int lgu_abi_version(void);                 /* bumped on any signature change */
LGU_API const char* lgu_build_info(void);          /* "sm_100a, nvcc x.y, <date>" */
LGU_API const char* lgu_last_error_string(void);   /* thread-local, never NULL */

/* --------------------------------------------------------------------------
 * corr_index_forward          (reference: offersample_LGS/droid.cpp:79-87,
 *                              corrSample_kernel.cu:24-82,139-168)
 * Plain bilinear lookup of a (2r+1)^2 window around coords.  corr is fully
 * written (taps whose top-left corner is out of bounds are 0).
 * ------------------------------------------------------------------------ */
LGU_API int lgu_corr_index_forward(const float* volume, const float* coords, float* corr,
                           int E, int H1, int W1, int H2, int W2, int radius, void* stream);

/* corr_index_backward         (droid.cpp:89-99, corrSample_kernel.cu:84-136,170-199)
 * volume_grad [E,H1,W1,H2,W2] is fully written (dense: zeros + scattered taps). */
LGU_API int lgu_corr_index_backward(const float* coords, const float* corr_grad, float* volume_grad,
                            int E, int H1, int W1, int H2, int W2, int radius, void* stream);

/* --------------------------------------------------------------------------
 * defCorr_index_forward       (droid.cpp:53-63, defCorrSample_kernel.cu:25-91,165-196)
 * Deformable lookup: tap (i,j) samples at coords + offset[..,i,j,:] - r + (i,j).
 * SIDE EFFECT (reference quirk Q5): offset[..,r,r,0:2] is set to 0 in place.
 * ------------------------------------------------------------------------ */
LGU_API int lgu_defcorr_index_forward(const float* volume, const float* coords, float* offset, float* corr,
                              int E, int H1, int W1, int H2, int W2, int radius, void* stream);

/* defCorr_index_backward      (droid.cpp:65-77, defCorrSample_kernel.cu:93-162,198-231)
 * volume_grad dense, offset_grad [E,H1,W1,rd,rd,2] ([..,0] = d/dx, [..,1] = d/dy; 0 for
 * gated taps).  Same in-place zeroing of the centre offset tap. */
LGU_API int lgu_defcorr_index_backward(const float* volume, const float* coords, float* offset,
                               const float* corr_grad, float* volume_grad, float* offset_grad,
                               int E, int H1, int W1, int H2, int W2, int radius, void* stream);

/* --------------------------------------------------------------------------
 * gaussianMask                (droid.cpp:100-110, gaussianAttn.cu:19-68,134-163)
 * means, covs [E,H1,W1,2] (channel 0 = x, 1 = y).  volume1 is dense: 3*V*exp(-0.5*d'S^-1 d)
 * inside the (2r+1)^2 window centred on floor(mean), 0 elsewhere.
 * ------------------------------------------------------------------------ */
LGU_API int lgu_gaussian_mask_forward(const float* means, const float* covs, const float* volume, float* volume1,
                              int E, int H1, int W1, int H2, int W2, int radius, void* stream);

/* gaussianMask_backward       (droid.cpp:112-123, gaussianAttn.cu:72-131,165-200)
 * means_grad, covs_grad [E,H1,W1,2]; the reference produces no gradient for volume. */
LGU_API int lgu_gaussian_mask_backward(const float* means, const float* covs, const float* volume,
                               const float* volume1_grad, float* means_grad, float* covs_grad,
                               int E, int H1, int W1, int H2, int W2, int radius, void* stream);

/* --------------------------------------------------------------------------
 * lowMem_defSample            (droid.cpp:124-136, lowMem_defSample.cu:27-134,137-168)
 * On-the-fly deformable correlation, no volume.  fmap1 [B,H1,W1,C], fmap2 [B,H2,W2,C]
 * channels-last, C a multiple of 32; coords [B,N,H1,W1,2] (last dim x,y);
 * offset [n_slabs,H1,W1,rd,rd,2]; corr [B,N,rd,rd,H1,W1] indexed [ix][iy].
 * strict_ref = 1 reproduces the reference's slab indexing offset[b*n] (quirk Q2; with the
 * only caller's N = 1 every edge reads slab 0); strict_ref = 0 uses offset[b*N+n].
 * SIDE EFFECT: the centre tap of every slab that is read is zeroed in place.
 * ------------------------------------------------------------------------ */
LGU_API int lgu_lowmem_defsample_forward(const float* fmap1, const float* fmap2, const float* coords,
                                 float* offset, float* corr,
                                 int B, int N, int H1, int W1, int H2, int W2, int C, int radius,
                                 int strict_ref, void* stream);

/* lowMem_defSample on TENSOR CORES, same operator contract: with `workspace` (device memory, 256-byte aligned, at least
 * lgu_lowmem_workspace_bytes(...) bytes, contents undefined on entry and exit) the call splits the maps into fp16 hi/lo
 * planes, builds this level's [B,P,Q] volume on tcgen05 (lgu_build_volume) and samples it with the TMA-staged lookup in
 * per-corner-gating mode.  lgu_lowmem_workspace_bytes returns 0 for shapes the path does not cover (needs N == 1, C == 128,
 * radius 3 -- 1 for altcorr --, H1*W1 % 128 == 0, W2 % 4 == 0); the *_ws entry points then (and with workspace == NULL) run
 * the on-the-fly SIMT kernel.  Results equal the on-the-fly kernel up to fp32 summation order (<= 1e-5). */
LGU_API long long lgu_lowmem_workspace_bytes(int B, int N, int H1, int W1, int H2, int W2, int C, int radius);
LGU_API int lgu_lowmem_defsample_forward_ws(const float* fmap1, const float* fmap2, const float* coords,
                                    float* offset, float* corr,
                                    int B, int N, int H1, int W1, int H2, int W2, int C, int radius,
                                    int strict_ref, void* workspace, long long workspace_bytes, void* stream);
LGU_API int lgu_altcorr_forward_ws(const float* fmap1, const float* fmap2, const float* coords, float* corr,
                           int B, int N, int H1, int W1, int H2, int W2, int C, int radius,
                           void* workspace, long long workspace_bytes, void* stream);

/* altcorr_forward             (src/droid.cpp:193-203, src/altcorr_kernel.cu:27-149,290-319)
 * The second boundary the backend path crosses (droid_slam/modules/corr.py:202).
 * corr [B,N,rd*rd,H1,W1], channel = iy + rd*ix. */
LGU_API int lgu_altcorr_forward(const float* fmap1, const float* fmap2, const float* coords, float* corr,
                        int B, int N, int H1, int W1, int H2, int W2, int C, int radius, void* stream);

/* --------------------------------------------------------------------------
 * Fused entry points (no single reference op; they replace op SEQUENCES of the
 * reference's Python glue and are validated against the composition of the
 * oracle's ops).
 * ------------------------------------------------------------------------ */

/* CorrBlock.__init__'s data path  (droid_slam/modules/corr.py:61-86 + gaussianMask_cuda.py:84-86):
 *   V   = (f1/4)^T (f2/4)                       all-pairs volume, tcgen05 / TMEM, fp32 accumulate
 *   V'  = gaussianMask(means,covs,V,gr)/den + V  learnable Gaussian residual (gr = 0 disables)
 *   lvl[l+1] = avg_pool2x2(lvl[l])              written in the same pass
 * fmaps   [T,P,C] fp16, channels-last ("K-major"), P = H*W (multiple of 128), C = 128
 *         (produced by lgu_pack_fmaps); precision: 1 = single fp16 product (exact for
 *         fp16-valued inputs, i.e. the inference path); 2 = hi/lo fp16 split, 3 MMAs,
 *         |error| <= ~2^-21 relative per product (fp32-valued inputs, the training path).
 * fmaps_lo  residual plane (x - fp16(x)) for precision 2, else NULL.
 * ii, jj  [E] int32 frame index of the source / target map of each edge.
 * means,covs [E,H,W,2] or NULL; den [E,H,W] (= 6.28*sqrt(cov_x*cov_y), gaussianMask_cuda.py:77,85) or NULL: the kernel
 * then forms it from covs in its prologue with the same fp32 roundings.
 * lvl0..lvl3 [E,H,W,H>>l,W>>l] outputs (lvl1..3 may be NULL to skip pooling). */
LGU_API int lgu_build_pyramid(const void* fmaps_hi, const void* fmaps_lo, const int32_t* ii, const int32_t* jj,
                      const float* means, const float* covs, const float* den,
                      float* lvl0, float* lvl1, float* lvl2, float* lvl3,
                      int T, int E, int H, int W, int C, int gauss_radius, int precision,
                      int round_half, void* stream);

/* CorrBlock.__call__'s data path  (droid_slam/modules/corr.py:88-109) in one launch:
 *   m      = sigmoid(var_9taps(corr_index_forward(lvl1, coords/2, 1)))        corr.py:94-97
 *   off1  <- off1 * m   (in place, every tap; the reference's cumulative `self.offset[1] *= mask`, quirk Q7)
 *   corr[:, l*49:(l+1)*49] = defCorr_index_forward(lvl_l, coords/2^l, off_l, 3)   corr.py:101-105
 * with off_2 = off_3 = 0 (corr.py:131-132), so those levels read no offsets at all.  The centre tap of off0 /
 * off1 is READ as 0 (quirk Q5) but not zeroed in memory: inside CorrBlock the reference zeroes a temporary
 * (`.contiguous()` of a permuted view), so its stored centre values survive too -- and its autograd uses them.
 * lvl0..lvl3 [E,H,W,H>>l,W>>l] (16-byte aligned), coords [E,H,W,2] (x,y interleaved, level-0 units -- the
 * layout CorrBlock.__call__ receives, before its permute), off0/off1 [E,H,W,7,7,2], corr [E,196,H,W],
 * mask_out [E,H,W] or NULL.  Pyramid patches are staged with TMA box loads.
 * Implemented for num_levels == 4, radius == 3, W % 32 == 0, H % 8 == 0 (LGU_ERR_UNSUPPORTED otherwise). */
LGU_API int lgu_corr_lookup_fused(const float* lvl0, const float* lvl1, const float* lvl2, const float* lvl3,
                          const float* coords, const float* off0, float* off1, float* corr, float* mask_out,
                          int E, int H, int W, int num_levels, int radius, void* stream);

/* lgu_corr_lookup_fused without the write-back of offset[1] (392 of its 4112 B per pixel): the block keeps its
 * level-1 offsets PRISTINE (off1, read only) and a per-pixel running product of all masks so far in
 * cum_mask [num_slots or E, H, W] (in/out; the caller initialises it to 1).  The lookup samples level 1 with
 * off1 * (cum_mask * m) and stores cum_mask <- cum_mask * m -- the reference's cumulative `self.offset[1] *= mask`
 * (quirk Q7) up to the association of the fp32 products ((o*m1)*m2 there, o*(m1*m2) here: <= 2 ulp of the offset).
 * slots may be NULL (edge e lives in slot e; num_slots is then ignored). */
LGU_API int lgu_corr_lookup_fused_cum(const float* lvl0, const float* lvl1, const float* lvl2, const float* lvl3,
                              const float* coords, const float* off0, const float* off1, float* cum_mask,
                              float* corr, float* mask_out, const int32_t* slots, int num_slots,
                              int E, int H, int W, int num_levels, int radius, void* stream);

/* The fused lookup with its CONSUMER's first layer folded in (SURVEY 8f-4): UpdateModule.corr_encoder[0:2] =
 * Conv2d(196, 128, 1) + ReLU (droid_net.py:74-76, applied at :115) is evaluated on the 196 x 32 tile while it is still in
 * shared memory -- TF32 tensor-core MMAs with a 3-term hi/lo split, fp32 accumulation: <= 1e-5 of F.conv2d in fp32 --
 * and enc [E,128,H,W] (fp32, or fp16 with out_half) is written; corr [E,196,H,W] is written too unless NULL (then the
 * 784 B/pixel tensor never exists).  wfrag = lgu_pack_conv1x1(weight [128,196]) (6400 x 2 float4), bias [128] or NULL.
 * Everything else as lgu_corr_lookup_fused_cum (off1 pristine, cum_mask in/out, optional slots). */
LGU_API int lgu_pack_conv1x1(const float* weight, float* wfrag, int out_channels, int in_channels, void* stream);
LGU_API int lgu_corr_lookup_fused_enc(const float* lvl0, const float* lvl1, const float* lvl2, const float* lvl3,
                              const float* coords, const float* off0, const float* off1, float* cum_mask,
                              float* corr, void* enc, const float* wfrag, const float* bias, int relu, int out_half,
                              float* mask_out, const int32_t* slots, int num_slots,
                              int E, int H, int W, int num_levels, int radius, void* stream);

/* The same fused lookup with the BACKEND path's semantics (AltCorrBlock.corr_fn, corr.py:174-215, whose samplers
 * are lowMem_defSample.cu:27-134 and src/altcorr_kernel.cu:27-149): every bilinear corner is gated on its own
 * (quirk Q4) and fractions are x - floor(x).  lvl_l here is the volume of level 0 source maps against the level-l
 * POOLED target maps (lgu_build_volume).  shared_offsets = 1 reproduces the reference's offset-slab indexing
 * `offset[b*n]` with N = 1 (quirk Q2): every edge reads the offsets of edge 0; apply_mask = 0 uses off1 as given
 * (the caller has already multiplied it by the mask, corr.py:206) and writes nothing back. */
LGU_API int lgu_altcorr_lookup_fused(const float* lvl0, const float* lvl1, const float* lvl2, const float* lvl3,
                             const float* coords, const float* off0, float* off1, float* corr, float* mask_out,
                             int E, int H, int W, int num_levels, int radius,
                             int shared_offsets, int apply_mask, void* stream);

/* lgu_altcorr_lookup_fused writing into a caller-owned destination: edge e's 196 rows go to row out_index[e] of
 * `corr` ([E_out,196,H,W]; out_index NULL: row e), as fp32 (out_half = 0) or fp16 rounded to nearest (out_half = 1:
 * what `update_op` reads under autocast, factor_graph.py:284-286).  `corr` may live in ANOTHER GPU's memory mapped into
 * this process (CUDA IPC / peer access): a rank of the edge-sharded backend then returns its per-edge outputs through
 * its own store stream over NVLink, with no collective on the data path (lgu-slam_b200/sharded.py). */
LGU_API int lgu_altcorr_lookup_fused_into(const float* lvl0, const float* lvl1, const float* lvl2, const float* lvl3,
                                  const float* coords, const float* off0, float* off1, void* corr,
                                  const int32_t* out_index, int out_half, float* mask_out,
                                  int E, int H, int W, int num_levels, int radius,
                                  int shared_offsets, int apply_mask, void* stream);

/* The backend lookup with its CONSUMER's first layer folded in: update_op's corr_encoder[0:2] = Conv2d(196, 128, 1) + ReLU
 * (droid_net.py:74-76,115), which factor_graph.py:281-286 runs under fp16 autocast, is evaluated on the 196 x 32 tile
 * while it is still in shared memory, and only enc [E_out,128,H,W] leaves the SM (786 KB per 48 x 64 edge in fp16
 * instead of the 1.2 MB of 196-channel rows -- what a rank of the sharded backend ships to the destination).
 * Precision contract (that of the autocast conv, up to summation order):
 *   - W and b are rounded to fp16 (round to nearest even) by lgu_pack_conv1x1_f16;
 *   - every corr value is rounded to fp16 (round to nearest even, as Tensor.half());
 *   - products are exact in fp32 and accumulated in fp32 (m16n8k16 fp16 tensor-core MMAs, K = 196 padded to 208 with
 *     zeros); the bias is added in fp32; ReLU propagates NaN like torch.relu;
 *   - the result is rounded once: to fp16 (round to nearest even) with out_half = 1, or stored as fp32 with out_half = 0.
 *
 * lgu_pack_conv1x1_f16: weight [128,196] (out_channels = 128, in_channels = 196 only), bias [128] or NULL (zero) ->
 *   packed, LGU_CONV1X1_F16_BYTES bytes, 16-byte aligned: the fp16 m16n8k16 A fragments [8 warps][13 k-steps][32 lanes]
 *   (16 B each), then the fp16-rounded bias as 128 floats.
 * lgu_altcorr_lookup_enc_into: lgu_altcorr_lookup_fused_into (per-corner gating, shared_offsets, apply_mask, mask_out,
 *   out_index rows) writing enc instead of corr; boxes0 / boxes1 as in lgu_altcorr_lookup_boxes_into (boxes0 != NULL
 *   replaces lvl0, which is then ignored; boxes1 != NULL replaces lvl1 and needs boxes0).  enc must be 8-byte aligned.
 * Both return LGU_ERR_BAD_ARG for null or misaligned pointers and bad sizes before any device work, and
 * lgu_altcorr_lookup_enc_into returns LGU_ERR_UNSUPPORTED unless num_levels = 4, radius = 3, W % 32 = 0 and H % 8 = 0. */
#define LGU_CONV1X1_F16_BYTES 53760
LGU_API int lgu_pack_conv1x1_f16(const float* weight, const float* bias, void* packed, int out_channels, int in_channels,
                                 void* stream);
LGU_API int lgu_altcorr_lookup_enc_into(const float* boxes0, const float* boxes1, const float* lvl0, const float* lvl1,
                                const float* lvl2, const float* lvl3, const float* coords, const float* off0, float* off1,
                                const void* packed, void* enc, const int32_t* out_index, int out_half, float* mask_out,
                                int E, int H, int W, int num_levels, int radius,
                                int shared_offsets, int apply_mask, void* stream);

/* Backward of lgu_corr_lookup_fused = what autograd runs for corr.py:88-109 in training (4 x
 * defCorr_index_backward, the offset[1]*mask / sigmoid / var chain, corr_index_backward), in one launch:
 *   gv0..gv3      dense gradients of the pyramid levels (each written exactly once; level 1 includes the mask path)
 *   off0_grad     gradient of off0;   off1_grad  gradient of off1 BEFORE the mask multiply (offset[1]_in)
 * inputs: off1_out = off1 after the forward (post-mask), mask = the forward's mask_out, corr_grad [E,196,H,W],
 * off1_out_grad [E,H,W,7,7,2] = upstream gradient on the post-mask offsets from later calls (NULL if none).
 * Levels 2-3 get no offset gradient (their offsets are detached zeros, corr.py:131-134); coords get none
 * (corr.py:42).
 * Numerics: the deformable levels' corner contributions are accumulated in FIXED POINT per source pixel (scale 2^(22-e),
 * e = exponent of the pixel's largest upstream |gradient|; native integer shared-memory adds, order-independent, no
 * overflow even if all 196 corners collide): |error| <= 2^-24 * max|g| per contribution, i.e. <= 1e-5 abs for the
 * O(1)..O(10) gradients of training, and bit-reproducible from run to run.  Pixels with non-finite gradients or NaN
 * sampling positions take the fp32 compare-and-swap path (NaNs propagate as in the reference). */
LGU_API int lgu_corr_lookup_fused_backward(const float* lvl0, const float* lvl1, const float* coords,
                                   const float* off0, const float* off1_out, const float* mask,
                                   const float* corr_grad, const float* off1_out_grad,
                                   float* gv0, float* gv1, float* gv2, float* gv3,
                                   float* off0_grad, float* off1_grad,
                                   int E, int H, int W, int num_levels, int radius, void* stream);

/* Same backward for a training clip, where ONE pyramid is looked up num_steps times (droid_net.py:187-222,
 * train.py:203): gv0..gv3 are PERSISTENT accumulators (zeroed once by the caller) and this launch ADDS its
 * gradient into them -- only the <= 20x16 / 12x8 footprint of every pixel is touched (16-byte L2 reductions),
 * no dense zero-fill per call and no dense autograd sum afterwards (the reference's graph moves
 * 4 x 50 MB/edge per lookup for that: zeros_like in defCorrSample_kernel.cu:206 + AccumulateGrad).
 * Every other argument as above. */
LGU_API int lgu_corr_lookup_fused_backward_accumulate(const float* lvl0, const float* lvl1, const float* coords,
                                   const float* off0, const float* off1_out, const float* mask,
                                   const float* corr_grad, const float* off1_out_grad,
                                   float* gv0, float* gv1, float* gv2, float* gv3,
                                   float* off0_grad, float* off1_grad,
                                   int E, int H, int W, int num_levels, int radius, void* stream);

/* The same backward for a forward that ran in the cumulative-mask form (lgu_corr_lookup_fused_cum): off1 holds the
 * PRISTINE level-1 offsets and cum_mask [E,H,W] the running mask product AFTER that forward, so the post-mask offsets
 * offset[1]_out = off1 * cum_mask are formed in registers (same product, same rounding as the forward) instead of being
 * read from a materialised tensor.  off1_grad is the gradient with respect to that call's input offsets
 * (off1 * cum_mask / mask).  accumulate != 0 selects the persistent-accumulator form. */
LGU_API int lgu_corr_lookup_fused_backward_cum(const float* lvl0, const float* lvl1, const float* coords,
                                   const float* off0, const float* off1, const float* cum_mask, const float* mask,
                                   const float* corr_grad, const float* off1_out_grad,
                                   float* gv0, float* gv1, float* gv2, float* gv3,
                                   float* off0_grad, float* off1_grad,
                                   int E, int H, int W, int num_levels, int radius, int accumulate, void* stream);

/* lgu_corr_lookup_fused_backward_cum (dense form) that ALSO emits the window record the Gaussian head's backward needs:
 *   gwin[e,p, wy*9 + wx] = g0[q] + g1[q/2]/4 + g2[q/4]/16 + g3[q/8]/64   at q = (floor(my) - 4 + wy, floor(mx) - 4 + wx),
 *                          0 outside the target grid                     (mx, my) = win_means[e,p]
 * i.e. avg_pool2d^T (corr.py:83-86) of this call's level gradients, evaluated only inside the 9 x 9 window of
 * gaussianMask (gaussianMask_cuda.py:77-86), formed from the kernel's shared-memory accumulators before the dense slices
 * are streamed out.  win_means [E,H,W,2] (8-byte aligned), gwin [E,H,W,81].  Everything else as _cum with accumulate = 0. */
LGU_API int lgu_corr_lookup_fused_backward_win(const float* lvl0, const float* lvl1, const float* coords,
                                   const float* off0, const float* off1, const float* cum_mask, const float* mask,
                                   const float* corr_grad, const float* off1_out_grad, const float* win_means,
                                   float* gv0, float* gv1, float* gv2, float* gv3,
                                   float* off0_grad, float* off1_grad, float* gwin,
                                   int E, int H, int W, int num_levels, int radius, void* stream);

/* The same dense backward with the Gaussian head's backward of the build FOLDED IN: the merged window gradient never
 * leaves the SM -- the kernel fetches the 81 level-0 values of the window and evaluates lgu_build_backward_gauss's
 * arithmetic (shared code, same bits) on the spot.  Returns, besides the level and offset gradients,
 *   means_grad, covs_grad [E,H,W,2], den_grad [E,H,W] = lgu_build_backward_gauss(means, covs, den, lvl0, gv0..gv3)
 * of THIS call's level gradients (one lookup per pyramid; a training step with several lookups accumulates level
 * gradients and calls lgu_build_backward_gauss once).  gauss_radius must be 4 (gaussianMask_cuda.py:77). */
LGU_API int lgu_corr_lookup_fused_backward_gauss(const float* lvl0, const float* lvl1, const float* coords,
                                   const float* off0, const float* off1, const float* cum_mask, const float* mask,
                                   const float* corr_grad, const float* off1_out_grad,
                                   const float* means, const float* covs, const float* den,
                                   float* gv0, float* gv1, float* gv2, float* gv3,
                                   float* off0_grad, float* off1_grad,
                                   float* means_grad, float* covs_grad, float* den_grad,
                                   int E, int H, int W, int num_levels, int radius, int gauss_radius, void* stream);

/* lgu_build_backward_gauss (below) from that window record instead of the four level gradients: same sums, same bits,
 * one contiguous 324-byte read per pixel instead of four strided window gathers.  Radius 4 only. */
LGU_API int lgu_build_backward_gauss_window(const float* means, const float* covs, const float* den, const float* lvl0,
                                   const float* gwin, float* means_grad, float* covs_grad, float* den_grad,
                                   int E, int H, int W, void* stream);

/* Gaussian-head part of the backward of lgu_build_pyramid (what autograd runs for gaussianMask_cuda.py:84-86
 * followed by 3 x avg_pool2d, corr.py:83-86), straight from the four LEVEL gradients, without a dense pass:
 *   g(q)      = g0[q] + g1[q/2]/4 + g2[q/4]/16 + g3[q/8]/64          (avg_pool2d^T, evaluated at the window taps only)
 *   V(q)      = lvl0[q] / (1 + 3 e(q) / den)                         (the raw volume, recovered inside the window)
 *   means_grad, covs_grad = gaussianMask_backward(means, covs, V, g / den)    (gaussianAttn.cu:72-131)
 *   den_grad  = - sum_window g (lvl0 - V) / den                      (the 1/den of gaussianMask_cuda.py:85-86)
 * means, covs [E,H,W,2]; den, den_grad [E,H,W]; lvl0, g0 [E,H,W,H,W]; g_l [E,H,W,H>>l,W>>l] (any g_l may be NULL). */
LGU_API int lgu_build_backward_gauss(const float* means, const float* covs, const float* den, const float* lvl0,
                                   const float* g0, const float* g1, const float* g2, const float* g3,
                                   float* means_grad, float* covs_grad, float* den_grad,
                                   int E, int H, int W, int radius, void* stream);

/* Feature-map gradients of lgu_build_pyramid (backward of corr.py:144-152 through the 4-level pyramid, corr.py:83-86)
 * on tcgen05, straight from the level gradients (average pooling commutes with the contraction):
 *   g_f1[e,c,p]   = sum_l sum_q level_grads[l][e,p,q] * f2_l[e,c,q]        f2_l = avgpool_l(f2) / 16, TF32-split
 *   g_f2[l][e,c,q] = sum_p level_grads[l][e,p,q] * f1[e,c,p]                f1 / 16, TF32-split
 * (the caller adds g_f2 = sum_l upsample_l(g_f2[l]) / 4^l).  level_grads[l] [E,H*W,(H>>l)*(W>>l)] fp32 or NULL (level
 * skipped; its g_f2[l] is left untouched); f1_hi/lo [E,C,H*W]; f2_hi/lo[l] [E,C,(H>>l)*(W>>l)]; outputs fp32.
 * hi/lo come from lgu_tf32_split (x*scale = hi + lo, hi with 10 mantissa bits).  kind::tf32, 3 MMAs per product term
 * (hi*hi + hi*lo + lo*hi), fp32 accumulation: ~2^-21 relative per product.  Needs C == 128, H*W % 128 == 0. */
LGU_API int lgu_build_backward_fmaps(const float* const* level_grads, const float* f1_hi, const float* f1_lo,
                                   const float* const* f2_hi, const float* const* f2_lo, float* g_f1,
                                   float* const* g_f2, int num_levels, int E, int H, int W, int C, void* stream);
LGU_API int lgu_tf32_split(const float* x, float scale, float* hi, float* lo, long long n, void* stream);

/* Edge-slot pool variants (replace the whole-pyramid copies of CorrBlock.cat / CorrBlock.__getitem__,
 * corr.py:111-115,137-141, which the frontend pays on every keyframe: factor_graph.py:123,158).  The pyramid levels
 * and the offsets live in storage of `num_slots` edge slots ([num_slots,H,W,H>>l,W>>l], [num_slots,H,W,7,7,2]);
 * out_slots[e] / slots[e] (int32, device) name the slot of the e-th edge of this call.  Adding edges = building into
 * free slots; removing edges = dropping their slot numbers; nothing is copied.  Everything else as in
 * lgu_build_pyramid / lgu_corr_lookup_fused (means, covs, den, coords, corr, mask_out are in call order). */
LGU_API int lgu_build_pyramid_slots(const void* fmaps_hi, const void* fmaps_lo, const int32_t* ii, const int32_t* jj,
                            const float* means, const float* covs, const float* den,
                            float* lvl0, float* lvl1, float* lvl2, float* lvl3,
                            const int32_t* out_slots, int num_slots,
                            int T, int E, int H, int W, int C, int gauss_radius, int precision,
                            int round_half, void* stream);
LGU_API int lgu_corr_lookup_fused_slots(const float* lvl0, const float* lvl1, const float* lvl2, const float* lvl3,
                                const float* coords, const float* off0, float* off1, float* corr, float* mask_out,
                                const int32_t* slots, int num_slots,
                                int E, int H, int W, int num_levels, int radius, void* stream);

/* All-pairs volume between two DIFFERENT map sets, no Gaussian, no pooling:
 *   volume[e, p, q] = sum_c fmaps1[ii[e], p, c] * fmaps2[jj[e], q, c]        (fp32 accumulate on tcgen05)
 * fmaps1 [T1,P,C], fmaps2 [T2,Q,C]: channels-last fp16 planes, already scaled (the caller's /4, corr.py:163);
 * lo planes for precision 2 as in lgu_build_pyramid.  volume [E,P,Q].  C = 128, P % 128 == 0, Q % 4 == 0.
 * This is how the backend path (AltCorrBlock, corr.py:155-215) is served on B200: its pyramid pools the FEATURE
 * maps (one volume per level against the pooled target map) and the reference avoids materialising them only for
 * lack of memory (lowMem_defSample.cu); with 180 GB of HBM a chunk of edges is materialised per level on tensor
 * cores and sampled with the fused lookup. */
LGU_API int lgu_build_volume(const void* fmaps1_hi, const void* fmaps1_lo, const void* fmaps2_hi, const void* fmaps2_lo,
                     const int32_t* ii, const int32_t* jj, float* volume,
                     int T1, int T2, int E, int P, int Q, int C, int precision, void* stream);

/* Sparse form for the fused backend lookup (lgu_altcorr_lookup_fused*), whose per-pixel reads stay inside a 20 x 16 box
 * around coords / 2^level when the learned offsets are bounded by 4 (4 * tanh, corr.py:121-128): only the 256-column
 * "halves" (256 / (W >> level) target rows each) named in half_mask [E * H*W / 128] -- one word per unit of 128 consecutive
 * source pixels, bit h = half h -- are computed and written; the rest of `volume` is left untouched and must not be read.
 * lgu_volume_half_mask derives the mask from the coords the lookup will be called with (box rows +- 1 row of slack).
 * With dense, smooth coords about 60 % of level 0 is built (tools/diag/t_backend1.py). */
LGU_API int lgu_volume_half_mask(const float* coords, uint32_t* half_mask, int E, int H, int W, int level, void* stream);
LGU_API int lgu_build_volume_sparse(const void* fmaps1_hi, const void* fmaps1_lo, const void* fmaps2_hi,
                                   const void* fmaps2_lo, const int32_t* ii, const int32_t* jj,
                                   const uint32_t* half_mask, float* volume,
                                   int T1, int T2, int E, int P, int Q, int C, int precision, void* stream);

/* Level 0 of the backend path as COMPACT per-pixel boxes instead of a volume: boxes [E,H*W,16,20] holds, for every source
 * pixel, the 16 x 20 window of its correlation slice that the fused backend lookup stages around coords [E,H,W,2]
 * (rows box_origin_y = clamp(floor(cy)) - 7 .. + 15, columns (clamp(floor(cx)) - 7) & ~3 .. + 19; zeros outside the H x W
 * grid) -- 1280 B per pixel instead of 12 KB (7.6 KB with the half mask), and one contiguous read per pixel for the lookup
 * instead of 16 strided rows.  fp16-valued maps (one product, fp32 accumulate), C = 128; level 0 (W = 64) or level 1
 * (fmaps2 = the level-1 pooled maps, W = 64 so that W >> 1 = 32; coords stay in level-0 units and are halved like the lookup
 * does); half_mask from lgu_volume_half_mask(coords, level).  lgu_altcorr_lookup_boxes_into =
 * lgu_altcorr_lookup_fused_into with `boxes0` in place of the level-0 volume and, if not NULL, `boxes1` in place of lvl1
 * (which may then be NULL); offsets must be bounded by 4 (4 * tanh, corr.py:121-128): a tap whose footprint leaves the
 * box inside the grid returns NaN. */
LGU_API int lgu_build_boxes(const void* fmaps1_hi, const void* fmaps2_hi, const int32_t* ii, const int32_t* jj,
                                   const float* coords, const uint32_t* half_mask, float* boxes,
                                   int T1, int T2, int E, int H, int W, int C, int level, void* stream);
LGU_API int lgu_altcorr_lookup_boxes_into(const float* boxes0, const float* boxes1, const float* lvl1, const float* lvl2,
                                   const float* lvl3, const float* coords, const float* off0, float* off1, void* corr,
                                   const int32_t* out_index, int out_half, float* mask_out,
                                   int E, int H, int W, int num_levels, int radius,
                                   int shared_offsets, int apply_mask, void* stream);

/* fmaps [T,C,P] fp32 or fp16 (NCHW as the encoders emit) -> channels-last fp16 planes
 * hi [T,P,C] (and lo [T,P,C] = fp16(x/4 - hi) when lo != NULL), pre-scaled by 1/4 (corr.py:148-149). */
LGU_API int lgu_pack_fmaps(const void* fmaps, int src_is_half, void* hi, void* lo,
                   int T, int C, int P, void* stream);

/* --------------------------------------------------------------------------
 * Offset heads' glue  (droid_slam/modules/corr.py:117-135 / 217-235, per_Corr_Normalization :44-51) in two launches
 * instead of ~14 torch kernels:
 *   off0[e,y,x,c] = 4 tanh( (c0[e,c,y,x] - mean0_e) / sqrt(var0_e + eps) )
 *   off1[e,y,x,c] = ( 4 tanh( (c1[e,c,y/2,x/2] - mean1_e) / sqrt(var1_e + eps) ) + off0[e,y,x,c] ) / 2
 * c0 [E,CH,H,W] = ofsMap(t), c1 [E,CH,H/2,W/2] = ofs_residual(avg_pool2d(t, 2)) (the conv outputs; the nearest-neighbour
 * upsampling of c1 is done by indexing, its statistics equal the low-resolution ones), mean/var per edge over
 * (CH,H,W), biased variance, eps = 1e-5.  off0, off1 [E,H,W,CH]: the channels-last layout the lookups read.
 * stats [E,4] fp32 receives (mean0, rstd0, mean1, rstd1).  Forward only (inference paths); CH <= 128, W % 32 == 0, H even.
 * ------------------------------------------------------------------------ */
LGU_API int lgu_offset_heads(const float* c0, const float* c1, float* off0, float* off1, float* stats,
                     int E, int CH, int H, int W, float eps, void* stream);

/* --------------------------------------------------------------------------
 * Peer-visible device memory for the edge-sharded backend (no reference counterpart: the reference is single-GPU).
 * lgu_peer_alloc: cudaMalloc on the current device + its CUDA IPC handle (64 bytes) for the other ranks of the box;
 * lgu_peer_open:  map that allocation into the calling process WITH THE CALLER'S DEVICE CURRENT (peer access over
 *                 NVLink / NVSwitch is switched on for that device), so its kernels can store straight into the owner's
 *                 HBM (lgu_altcorr_lookup_fused_into with out = the mapped pointer);
 * lgu_peer_close / lgu_peer_free: unmap / release.
 * ------------------------------------------------------------------------ */
LGU_API int lgu_peer_alloc(long long bytes, void** ptr, void* handle64);
LGU_API int lgu_peer_open(const void* handle64, void** ptr);
LGU_API int lgu_peer_close(void* ptr);
LGU_API int lgu_peer_free(void* ptr);

#ifdef __cplusplus
}
#endif
#endif /* LGU_CORR_H_ */

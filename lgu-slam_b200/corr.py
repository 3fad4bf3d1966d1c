"""Host-side mirror of the reference's correlation frontend, on the sm_100a operator layer.

Same class names, constructor arguments, call signatures, return values and in-place side effects as
/root/reference/droid_slam/modules/corr.py (CorrSampler :10-24, DefCorrSampler :26-42, CorrBlock :53-152,
AltCorrBlock :155-249) and /root/reference/droid_slam/gaussianMask_cuda.py (GaussianMaskCuda :7-23,
GaussianMask :35-88), so `factor_graph.py`, `droid_net.py` and `motion_filter.py` can import them from here
instead.  What differs is underneath:

  * CorrBlock.__init__ runs ONE fused tcgen05/TMA kernel (ops.build_pyramid) for the volume, the Gaussian
    residual and the 4-level pyramid instead of matmul -> .float() -> gaussianMask -> div -> add -> 3 pools;
    the per-op path (`fused=False`) is kept and is what the fused path is tested against;
  * every lookup goes through the C ABI in include/lgu_corr.h; there is no CPU path.

The learned heads (ofsMap / ofs_residual convs, the GaussianMask MLP) stay torch modules, as in the reference;
`OffsetConv` is an nn.Conv2d for the two offset convs that runs them on the library's tensor-core kernels.
"""
import functools
import math
import weakref

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import ops

GAUSS_RADIUS = 4          # gaussianMask_cuda.py:84 (a 9x9 window, not the lookup radius)
MASK_RADIUS = 1           # corr.py:94,202: the uncertainty mask is an r=1 lookup on level 1


# ------------------------------------------------------------------------------------------------
# autograd Functions (same contracts as the reference's)
# ------------------------------------------------------------------------------------------------
class CorrSampler(torch.autograd.Function):
    """corr.py:10-24: plain bilinear window lookup; gradient for the volume only."""

    @staticmethod
    def forward(ctx, volume, coords, radius):
        ctx.save_for_backward(volume, coords)
        ctx.radius = radius
        corr, = ops.corr_index_forward(volume, coords, radius)
        return corr

    @staticmethod
    def backward(ctx, grad_output):
        volume, coords = ctx.saved_tensors
        grad_volume, = ops.corr_index_backward(volume, coords, grad_output.contiguous(), ctx.radius)
        return grad_volume, None, None


class DefCorrSampler(torch.autograd.Function):
    """corr.py:26-42: deformable lookup; gradients for the volume and the offsets, none for coords.
    The offset tensor handed in is mutated (centre tap zeroed, quirk Q5) and that mutated tensor is what
    backward sees, as in the reference."""

    @staticmethod
    def forward(ctx, volume, coords, offset, radius):
        offset = offset.float()
        volume = volume.float()
        ctx.save_for_backward(volume, coords, offset)
        ctx.radius = radius
        corr, = ops.defCorr_index_forward(volume, coords, offset, radius)
        return corr

    @staticmethod
    def backward(ctx, grad_output):
        volume, coords, offset = ctx.saved_tensors
        grad_volume, grad_offset = ops.defCorr_index_backward(volume, coords, offset, grad_output.contiguous(),
                                                              ctx.radius)
        return grad_volume, None, grad_offset, None


class GaussianMaskCuda(torch.autograd.Function):
    """gaussianMask_cuda.py:7-23: gradients for mean and cov only (the reference returns None for corr)."""

    @staticmethod
    def forward(ctx, mean, cov, corr, radius):
        mean = mean.float()
        cov = cov.float()
        ctx.save_for_backward(mean, cov, corr)
        ctx.radius = radius
        corr1, = ops.gaussianMask(mean, cov, corr, radius)
        return corr1

    @staticmethod
    def backward(ctx, grad_output):
        mean, cov, corr = ctx.saved_tensors
        gm, gc = ops.gaussianMask_backward(mean, cov, corr, grad_output.contiguous(), ctx.radius)
        return gm, gc, None, None


class LevelGradAccumulator:
    """Persistent gradient buffers of one pyramid for a training clip (droid_net.py:187-222 looks the same CorrBlock up
    `num_steps` times).  The reference's graph allocates, zero-fills and writes a dense 50 MB/edge gradient per lookup
    (defCorrSample_kernel.cu:206) and AccumulateGrad then sums them; here every lookup's backward ADDS its footprints
    into these four buffers (lgu_corr_lookup_fused_backward_accumulate) and FusedBuild.backward consumes them once.
    `levels` are the FusedBuild outputs the buffers belong to (identity-checked by the lookup)."""

    def __init__(self):
        self._levels = None        # weak references: the autograd graph (FusedBuild's ctx) points at this object, so strong
        self.grads = None          # references to the build's outputs would close a cycle through the graph

    @property
    def levels(self):
        return None if self._levels is None else tuple(r() for r in self._levels)

    @levels.setter
    def levels(self, tensors):
        self._levels = None if tensors is None else tuple(weakref.ref(t) for t in tensors)

    def owns(self, pyramid):
        return self._levels is not None and all(r() is b for r, b in zip(self._levels, pyramid))

    def buffers(self):
        if self.grads is None:
            self.grads = [torch.zeros_like(r()) for r in self._levels]
        return self.grads

    def take(self):
        g, self.grads = self.grads, None
        return g


class FusedCorrLookup(torch.autograd.Function):
    """CorrBlock.__call__'s whole data path (corr.py:88-109) as ONE differentiable op: forward = one TMA-staged
    launch, backward = one launch (lgu_corr_lookup_fused_backward).  Inputs: the 4 pyramid levels, coords [E,H,W,2],
    off0, off1 [E,H,W,98].  Outputs: corr [E,196,H,W] and the post-mask offsets offset[1]*mask (which the block
    keeps for its next call, quirk Q7).  Gradients: pyramid levels, off0, off1; none for coords (corr.py:42).
    With an accumulator (`acc`, the pyramid's LevelGradAccumulator) the level gradients are added into its persistent
    buffers instead of being returned; `token` (an output of the same FusedBuild) carries a defined zero gradient back
    so that FusedBuild.backward runs after every lookup of the clip and picks the buffers up."""

    @staticmethod
    def forward(ctx, lvl0, lvl1, lvl2, lvl3, coords, off0, off1, *extra):
        token, acc = (tuple(extra) + (None, None))[:2]
        ctx.n_extra = len(extra)
        off1_out = off1.detach().clone()                    # the kernel updates offset[1] in place
        corr, mask = ops.corr_lookup_fused([lvl0, lvl1, lvl2, lvl3], coords, off0, off1_out, 3, return_mask=True)
        ctx.save_for_backward(lvl0, lvl1, lvl2, lvl3, coords, off0, off1_out, mask)
        ctx.acc = acc if (acc is not None and token is not None and acc.owns((lvl0, lvl1, lvl2, lvl3))) else None
        ctx.mark_non_differentiable(mask)
        return corr, off1_out, mask

    @staticmethod
    def backward(ctx, g_corr, g_off1_out, _g_mask):
        lvl0, lvl1, lvl2, lvl3, coords, off0, off1_out, mask = ctx.saved_tensors
        up = g_off1_out.contiguous() if g_off1_out is not None else None
        if ctx.acc is not None:
            _, _, _, _, g0, g1 = ops.corr_lookup_fused_backward([lvl0, lvl1, lvl2, lvl3], coords, off0, off1_out, mask,
                                                                g_corr.contiguous(), up,
                                                                accumulate_into=ctx.acc.buffers())
            return (None, None, None, None, None, g0.view_as(off0), g1.view_as(off1_out), g0.new_zeros(1), None)
        gv0, gv1, gv2, gv3, g0, g1 = ops.corr_lookup_fused_backward([lvl0, lvl1, lvl2, lvl3], coords, off0, off1_out,
                                                                    mask, g_corr.contiguous(), up)
        return (gv0, gv1, gv2, gv3, None, g0.view_as(off0), g1.view_as(off1_out)) + (None,) * ctx.n_extra


class FusedBuild(torch.autograd.Function):
    """CorrBlock.__init__'s data path (corr.py:61-86 + gaussianMask_cuda.py:84-86) as ONE differentiable op.
    forward  : pack + one tcgen05/TMA launch -> the 4 pyramid levels (fp32 maps: hi/lo split, three MMAs) and a
               1-element ordering token (see FusedCorrLookup).
    backward : exactly what autograd computes for the reference graph, evaluated LEVEL-WISE (no dense merge pass):
                 g      = g_lvl0 + up2(g_lvl1)/4 + up4(g_lvl2)/16 + up8(g_lvl3)/64              (3 x avg_pool2d)
                 g_V    = g                                 (GaussianMaskCuda returns NO gradient for corr,
                                                             gaussianMask_cuda.py:23 -- only the `+ corr` branch)
                 g_mean, g_cov = gaussianMask_backward(mean, cov, V, g / den)                  (gaussianAttn.cu:72-131)
                 g_den  = -sum_q g * corr1 / den^2,  corr1 = (lvl0 - V) * den  ->  g_det via den = 6.28 sqrt(det)
                   -- one launch over the 9x9 windows (lgu_build_backward_gauss); the raw volume V is not stored:
                   inside the window lvl0 = V (1 + 3 e / den)
                 g_f1   = g_V f2 / 16        = sum_l g_lvl_l  avgpool_l(f2) / 16               (pooling commutes with
                 g_f2   = g_V^T f1 / 16      = sum_l up_l(g_lvl_l^T f1) / (16 * 4^l)            the contraction)
               The level gradients are the accumulator's buffers (training clip) plus whatever autograd delivers."""

    @staticmethod
    def forward(ctx, f1, f2, mean, cov, det, autocast_rounding, acc=None):
        E, c, h, w = f1.shape
        frames = torch.cat((f1, f2), dim=0).contiguous()
        hi, lo = ops.pack_fmaps(frames, split=frames.dtype == torch.float32)
        idx = torch.arange(2 * E, dtype=torch.int32, device=frames.device)
        den = (6.28 * torch.sqrt(det)).view(E, h, w).float().contiguous()
        mean_c, cov_c = mean.float().contiguous(), cov.float().contiguous()
        pyr = ops.build_pyramid(hi, lo, idx[:E].contiguous(), idx[E:].contiguous(), h, w, means=mean_c, covs=cov_c, den=den,
                                num_levels=4, gauss_radius=GAUSS_RADIUS, round_half=bool(autocast_rounding))
        ctx.save_for_backward(f1, f2, mean_c, cov_c, det, den, pyr[0])
        ctx.acc = acc
        ctx.set_materialize_grads(False)
        token = pyr[0].new_zeros(1)
        return tuple(pyr) + (token,)

    @staticmethod
    def _fmaps_grad_library(grads, f1, f2):
        """The same two products on library GEMMs (cuBLAS fp32, no TF32) for shapes the tcgen05 kernel does not cover."""
        E, c, h, w = f1.shape
        P = h * w
        a1 = f1.reshape(E, c, P).float()
        g_f1 = torch.zeros(E, P, c, dtype=torch.float32, device=f1.device)
        g_f2 = torch.zeros(E, c, h, w, dtype=torch.float32, device=f1.device)
        prev = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = False
        try:
            f2l = f2.float()
            for l, g in enumerate(grads):
                if l > 0:
                    f2l = F.avg_pool2d(f2l, 2, stride=2)
                if g is None:
                    continue
                Q = (h >> l) * (w >> l)
                gm = g.view(E, P, Q)
                g_f1.baddbmm_(gm, f2l.reshape(E, c, Q).transpose(1, 2))               # [E,P1,c]
                t = torch.bmm(a1, gm).view(E, c, h >> l, w >> l)                      # [E,c,Q_l]
                if l > 0:
                    k = 1 << l
                    t = (t / float(k * k)).repeat_interleave(k, dim=2).repeat_interleave(k, dim=3)
                g_f2 += t
        finally:
            torch.backends.cuda.matmul.allow_tf32 = prev
        return (g_f1 / 16.0).transpose(1, 2).reshape(f1.shape), g_f2 / 16.0

    @staticmethod
    def backward(ctx, g0, g1, g2, g3, _g_token=None):
        f1, f2, mean, cov, det, den, lvl0 = ctx.saved_tensors
        E, c, h, w = f1.shape
        P = h * w
        grads = [g0, g1, g2, g3]
        held = ctx.acc.take() if ctx.acc is not None else None
        if held is not None:
            grads = [a if g is None else a.add_(g) for a, g in zip(held, grads)]
        grads = [None if g is None else g.float().contiguous() for g in grads]
        if all(g is None for g in grads):
            return (None,) * 7
        g_mean, g_cov, g_den = ops.build_backward_gauss(mean, cov, den, lvl0, grads, GAUSS_RADIUS)
        g_det = (g_den * (0.5 * 6.28) / torch.sqrt(det).view(E, h, w)).view_as(det)
        if c == 128 and P % 128 == 0 and w % 32 == 0 and h % 8 == 0:
            # tcgen05 kind::tf32 (3-term split): both products read the level gradients in place, once each
            g_f1, g_f2 = ops.build_backward_fmaps(grads, f1, f2)
        else:
            g_f1, g_f2 = FusedBuild._fmaps_grad_library(grads, f1, f2)
        return (g_f1.to(f1.dtype), g_f2.view_as(f2).to(f2.dtype), g_mean, g_cov, g_det, None, None)


class OffsetHeads(torch.autograd.Function):
    """The offset heads' glue (corr.py:117-135, per_Corr_Normalization :44-51) as ONE differentiable op: forward = the two
    lgu_offset_heads launches (c0 = ofsMap(t) [E,CH,H,W], c1 = ofs_residual(avg_pool2d(t)) [E,CH,H/2,W/2] -> contiguous
    off0, off1 [E,H,W,CH], bit-identical to the inference path), backward = one lgu_offset_heads_backward call.  A missing
    output gradient reaches the kernel as NULL (a zero gradient) instead of a materialised zero tensor."""

    @staticmethod
    def forward(ctx, c0, c1):
        c0, c1 = c0.contiguous(), c1.contiguous()
        off0, off1, stats = ops.offset_heads(c0, c1, return_stats=True)
        ctx.save_for_backward(c0, c1, stats)
        ctx.set_materialize_grads(False)
        return off0, off1

    @staticmethod
    def backward(ctx, g_off0, g_off1):
        if g_off0 is None and g_off1 is None:
            return None, None
        c0, c1, stats = ctx.saved_tensors
        return ops.offset_heads_backward(c0, c1, stats, None if g_off0 is None else g_off0.contiguous(),
                                         None if g_off1 is None else g_off1.contiguous())


class OffsetConvFunction(torch.autograd.Function):
    """conv3x3 (ops.conv3x3) as a differentiable op: forward = pack + implicit GEMM, backward = the input, weight and bias
    gradients that autograd asks for, nothing else."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        ctx.save_for_backward(x, weight)
        return ops.conv3x3(x, weight, bias)

    @staticmethod
    def backward(ctx, g_y):
        x, weight = ctx.saved_tensors
        need_x, need_w, need_b = ctx.needs_input_grad
        return ops.conv3x3_backward(x, weight, g_y.contiguous(), need_x, need_w, need_b)


class OffsetConv(nn.Conv2d):
    """nn.Conv2d(in_channels, out_channels, 3, padding=1) -- the offset heads ofsMap / ofs_residual (droid_net.py) --
    whose forward and backward run on the library's tensor-core kernels (OffsetConvFunction) in fp32 accuracy when the
    input allows: a CUDA fp32 [E,C_in,H,W] tensor outside CUDA autocast, at sizes ops.conv3x3_supported accepts (both
    grids of the heads, 48x64 and 24x32).  Any other input takes nn.Conv2d.forward unchanged.  Parameters and state_dict
    are nn.Conv2d's, so the reference's checkpoints load."""

    def __init__(self, in_channels, out_channels, device=None, dtype=None):
        super().__init__(in_channels, out_channels, 3, stride=1, padding=1, dilation=1, groups=1, bias=True,
                         padding_mode="zeros", device=device, dtype=dtype)

    def _library_path(self, x):
        w, b = self.weight, self.bias
        return (isinstance(x, torch.Tensor) and x.is_cuda and x.dtype == torch.float32 and x.dim() == 4
                and not torch.is_autocast_enabled("cuda") and w.dtype == torch.float32 and w.device == x.device
                and b is not None and b.dtype == torch.float32 and self.padding_mode == "zeros"
                and tuple(self.kernel_size) == (3, 3) and tuple(self.stride) == (1, 1) and tuple(self.padding) == (1, 1)
                and tuple(self.dilation) == (1, 1) and self.groups == 1 and x.shape[1] == self.in_channels
                and ops.conv3x3_supported(self.in_channels, self.out_channels, x.shape[2], x.shape[3]))

    def forward(self, x):
        if self._library_path(x):
            return OffsetConvFunction.apply(x.contiguous(), self.weight.contiguous(), self.bias.contiguous())
        return super().forward(x)


def per_Corr_Normalization(x, normalIndex, eps=1e-5):
    """corr.py:44-51 / gaussianMask_cuda.py:26-33: standardise over `normalIndex` (biased variance + eps)."""
    mean = torch.mean(x, dim=normalIndex, keepdim=True)
    std = torch.sqrt(torch.var(x, dim=normalIndex, unbiased=False, keepdim=True) + eps)
    return (x - mean) / std


# ------------------------------------------------------------------------------------------------
# GaussianMask module
# ------------------------------------------------------------------------------------------------
class GaussianMask(nn.Module):
    """gaussianMask_cuda.py:35-88.  Parameter names (map, meanMap, covMap) match the reference so its
    checkpoints load; `params()` exposes (mean, cov, det) for the fused build."""

    def __init__(self, h, w):
        super().__init__()
        self.meanMap = nn.Linear(16, 2)
        self.covMap = nn.Linear(16, 2)
        self.map = nn.Linear(256, 16)
        nn.init.zeros_(self.meanMap.weight)
        nn.init.zeros_(self.meanMap.bias)
        for lin in (self.covMap, self.map):
            nn.init.normal_(lin.weight, 0.0, math.sqrt(2.0 / lin.out_features))
            nn.init.zeros_(lin.bias)
        self.mapA = nn.Sequential(self.map, nn.Tanh())
        ys, xs = torch.meshgrid(torch.arange(h).float(), torch.arange(w).float(), indexing="ij")
        self.coord = torch.stack([xs, ys], dim=-1)       # [h,w,2], channel 0 = x (plain attribute, like the reference)

    def params(self, x):
        """x [E,h,w,256] -> mean [E,h,w,2] (pixel grid + learned shift), cov [E,h,w,2] in (0.05, 5.05), det [E,h*w]."""
        b, h, w, _ = x.shape
        tt = self.mapA(x)
        mean_ofs = self.meanMap(tt).view(b, h, w, 2)
        c = per_Corr_Normalization(self.covMap(tt).view(b, h * w, 2), [1, 2])
        c = torch.sigmoid(c) * 5 + 0.05
        det = c[:, :, 0] * c[:, :, 1]
        cov = c.view(b, h, w, 2).float()
        mean = self.coord.to(device=x.device, dtype=cov.dtype).expand(b, h, w, 2) + mean_ofs
        return mean, cov, det

    def forward(self, x, corr):
        b, h, w, _ = x.shape
        mean, cov, det = self.params(x)
        corr1 = GaussianMaskCuda.apply(mean.contiguous(), cov.contiguous(), corr, GAUSS_RADIUS)
        corr1 = corr1 / (6.28 * torch.sqrt(det).view(b, h, w, 1, 1)) + corr
        return corr1, mean, det


# ------------------------------------------------------------------------------------------------
# offsets (corr.py:117-135 / 217-235)
# ------------------------------------------------------------------------------------------------
def _generate_offsets(ofsMap, ofs_residual, t, fused_lookup=False):
    """t [E,256,h,w] -> 4 per-level offset tensors [E,h,w,98]; levels 2 and 3 are zeros.  fused_lookup: the caller's
    lookups take the fused path (CorrBlock._fused_lookup_shape), which never writes the records' centre taps."""
    _, _, h, w = t.shape
    o0 = ofsMap(t)
    r1 = ofs_residual(F.avg_pool2d(t, kernel_size=2, stride=2))
    kernel = o0.is_cuda and w % 32 == 0 and h % 2 == 0 and o0.shape[1] <= 128 and o0.dtype == torch.float32
    if kernel and (not torch.is_grad_enabled() or not (o0.requires_grad or r1.requires_grad)):
        # inference: normalise -> 4 tanh -> level-1 average -> upsample -> NHWC in two launches (lgu_offset_heads) instead of
        # ~14 torch kernels; the records come out contiguous [E,h,w,98] (the reference holds permuted views here, so its
        # stored centre taps survive the first per-operator call; they are read as 0 either way, quirk Q5)
        off0, off1 = ops.offset_heads(o0.detach().contiguous(), r1.detach().contiguous())
        return [off0, off1, torch.zeros_like(off0), torch.zeros_like(off0)]
    if kernel and fused_lookup:
        # training with fused lookups: the same two launches, differentiable (OffsetHeads).  Contiguous records are safe
        # here because the fused lookup reads the centre tap as 0 and never zeroes it in memory (quirk Q5); the
        # per-operator sampler does zero it in place, so every other caller keeps the permuted views below
        off0, off1 = OffsetHeads.apply(o0, r1)
        return [off0, off1, torch.zeros_like(off0), torch.zeros_like(off0)]
    o1 = F.interpolate(r1, (h, w))
    o0 = torch.tanh(per_Corr_Normalization(o0, [1, 2, 3])) * 4
    o1 = (torch.tanh(per_Corr_Normalization(o1, [1, 2, 3])) * 4 + o0) / 2
    # [E,h,w,98] as PERMUTED VIEWS, like the reference (corr.py:129-134): `.contiguous()` at the samplers then copies,
    # so the in-place centre-tap zeroing (quirk Q5) lands in a temporary and the stored centre values survive for the
    # `offset[1] * mask` backward -- until cat / __getitem__ make the tensors contiguous, exactly as in the reference.
    # zeros_like keeps the permuted strides, as it does there.
    o0 = o0.permute(0, 2, 3, 1)
    o1 = o1.permute(0, 2, 3, 1)
    return [o0, o1, torch.zeros_like(o0).detach(), torch.zeros_like(o0).detach()]


class _Offsets(list):
    """The block's `offset` list (corr.py:57,117-135) with the level-1 entry optionally kept FACTORED as
    base * cum_mask: the fused inference lookup then leaves the 392 B / pixel of offset[1] untouched and only updates
    the per-pixel running product of its masks (lgu_corr_lookup_fused_cum; the reference re-multiplies and re-writes
    the whole tensor on every call, corr.py:99).  Reading `offset[1]` materialises base * cum_mask, i.e. exactly the
    tensor the reference holds at that point; assigning to it (cat / __getitem__ / the per-operator path) stores the
    given tensor and drops the factor."""

    def __init__(self, items):
        super().__init__(items)
        self.cum = None

    def _get(self, i):
        v = list.__getitem__(self, i)
        if i in (1, 1 - len(self)) and self.cum is not None:
            v = v * self.cum.unsqueeze(-1)
        return v

    def __getitem__(self, i):
        if isinstance(i, slice):
            return [self._get(k) for k in range(*i.indices(len(self)))]
        return self._get(i)

    def __iter__(self):
        return (self._get(k) for k in range(len(self)))

    def __setitem__(self, i, v):
        if i in (1, 1 - len(self)):
            self.cum = None
        list.__setitem__(self, i, v)

    def _raw(self):
        return [list.__getitem__(self, k) for k in range(len(self))]

    def cat(self, other):
        """corr.py:111-115 on the factored form: base and cum_mask are concatenated separately, so a block that grows
        edge by edge keeps sampling with base * (m1 * m2 * ...) exactly like the edge-slot pool does."""
        a, b = self._raw(), (other._raw() if isinstance(other, _Offsets) else list(other))
        out = _Offsets([torch.cat([x, y], 0) for x, y in zip(a, b)])
        oc = other.cum if isinstance(other, _Offsets) else None
        if self.cum is not None or oc is not None:
            ones = lambda t: torch.ones(t.shape[:3], dtype=torch.float32, device=t.device)
            out.cum = torch.cat([self.cum if self.cum is not None else ones(a[1]),
                                 oc if oc is not None else ones(b[1])], 0)
        return out

    def index(self, index):
        """corr.py:137-141 on the factored form."""
        out = _Offsets([t[index] for t in self._raw()])
        if self.cum is not None:
            out.cum = self.cum[index]
        return out

    def factored(self):
        """(base, cum_mask) of level 1; creates the factor (ones) on first use."""
        base = list.__getitem__(self, 1)
        if not (base.is_contiguous() and base.dtype == torch.float32):
            base = base.float().contiguous()
            list.__setitem__(self, 1, base)
        if self.cum is None:
            self.cum = torch.ones(base.shape[:3], dtype=torch.float32, device=base.device)
        return base, self.cum


def _encoder_conv(corr_encoder):
    """UpdateModule.corr_encoder (droid_net.py:74-78) or its first layer -> that Conv2d(196, 128, 1)."""
    conv = corr_encoder[0] if isinstance(corr_encoder, nn.Sequential) else corr_encoder
    if not (isinstance(conv, nn.Conv2d) and conv.kernel_size == (1, 1) and conv.in_channels == 196
            and conv.out_channels == 128):
        raise RuntimeError("lookup_encoded needs the 196 -> 128 1x1 corr_encoder conv")
    return conv


# ------------------------------------------------------------------------------------------------
# CorrBlock
# ------------------------------------------------------------------------------------------------
class CorrBlock:
    """corr.py:53-152.  Attributes kept: corr_pyramid (list of [E,h,w,h>>l,w>>l]), offset (list of [E,h,w,98]),
    mean_n, theta, num_levels, radius.  `fused=None` picks the fused build (one tcgen05 launch, differentiable through
    FusedBuild) whenever the shape is supported (w = 64, h % 8 = 0, C = 128, 4 levels); `fused=False` is the
    reference's per-operator graph (matmul -> GaussianMaskCuda -> / den + corr -> 3 x avg_pool2d)."""

    def __init__(self, ofsMap, ofs_residual, GA, fmap1, fmap2, num_levels=4, radius=3, fused=None,
                 autocast_rounding=None, fused_lookup=True, accumulate_grads=True):
        self.fused_lookup = fused_lookup
        self._gacc = self._token = None
        self.num_levels = num_levels
        self.radius = radius
        self.GA = GA
        self.ofsMap = ofsMap
        self.ofs_residual = ofs_residual
        b, n, c, h, w = fmap1.shape
        E = b * n
        needs_grad = torch.is_grad_enabled() and (fmap1.requires_grad or fmap2.requires_grad or any(
            p.requires_grad for p in GA.parameters()))
        if fused is None:
            fused = w == 64 and h % 8 == 0 and c == 128 and num_levels == 4
        # under autocast the reference's matmul emits fp16 (factor_graph.py:90, corr.py:64); reproduce on request
        if autocast_rounding is None:
            autocast_rounding = False

        t = torch.cat((fmap1.reshape(E, c, h, w), fmap2.reshape(E, c, h, w)), dim=1)
        self.offset = _Offsets(_generate_offsets(ofsMap, ofs_residual, t.float(), self._fused_lookup_shape(h, w)))
        self.t = t.permute(0, 2, 3, 1).contiguous()

        if fused:
            # one tcgen05/TMA launch; differentiable (FusedBuild) when gradients are needed
            mean, cov, det = GA.params(self.t.float())
            self._gacc = LevelGradAccumulator() if (needs_grad and accumulate_grads) else None
            *pyr, self._token = FusedBuild.apply(fmap1.reshape(E, c, h, w), fmap2.reshape(E, c, h, w), mean, cov, det,
                                                 autocast_rounding, self._gacc)
            self.corr_pyramid = list(pyr)
            if self._gacc is not None:
                self._gacc.levels = tuple(pyr)
        else:
            corr = CorrBlock.corr(fmap1, fmap2).view(E, h, w, h, w).float()
            corr, mean, det = GA(self.t.float(), corr)
            self.corr_pyramid = []
            cur = corr.reshape(E * h * w, 1, h, w)
            for i in range(num_levels):
                self.corr_pyramid.append(cur.view(E, h, w, h >> i, w >> i))
                cur = F.avg_pool2d(cur, 2, stride=2)
        self.mean_n = mean.view(b, n, h, w, 2)
        self.theta = 2 * det.view(b, n, h, w)

    def _fused_lookup_shape(self, ht, wd):
        """The grids and settings the fused lookup covers (lgu_corr_lookup_fused)."""
        return self.fused_lookup and self.num_levels == 4 and self.radius == 3 and wd % 32 == 0 and ht % 8 == 0

    def _can_fuse_lookup(self, coords):
        ht, wd = coords.shape[2:4]
        return self._fused_lookup_shape(ht, wd) and all(t.dtype == torch.float32 for t in self.corr_pyramid)

    def _needs_grad(self, coords):
        return torch.is_grad_enabled() and any(t.requires_grad for t in self.corr_pyramid + [
            list.__getitem__(self.offset, 0), list.__getitem__(self.offset, 1)])

    def __call__(self, coords):
        batch, num, ht, wd, _ = coords.shape
        E, rd = batch * num, 2 * self.radius + 1
        if self._can_fuse_lookup(coords):
            # one TMA-staged launch: mask lookup + var + sigmoid + offset[1] *= mask + 4 deformable lookups + cat
            if not isinstance(self.offset, _Offsets):        # a caller replaced the list: adopt it
                self.offset = _Offsets(self.offset)
            if not (self.offset[0].is_contiguous() and self.offset[0].dtype == torch.float32):
                self.offset[0] = self.offset[0].float().contiguous()
            pyr = [t if t.is_contiguous() else t.contiguous() for t in self.corr_pyramid]
            c = coords.detach().reshape(E, ht, wd, 2).float().contiguous()
            if self._needs_grad(coords):                     # training: differentiable fused op (1 + 1 launches)
                # (with the fused build, level gradients accumulate in self._gacc's persistent buffers)
                off1 = self.offset[1]
                if not (off1.is_contiguous() and off1.dtype == torch.float32):
                    off1 = off1.float().contiguous()
                out, self.offset[1], _ = FusedCorrLookup.apply(pyr[0], pyr[1], pyr[2], pyr[3], c, self.offset[0],
                                                               off1, self._token, self._gacc)
            else:                                            # inference: offset[1] stays factored as base * cum_mask
                base, cum = self.offset.factored()
                out = ops.corr_lookup_fused(pyr, c, self.offset[0], base, self.radius, cum_mask=cum)
            return out.view(batch, num, -1, ht, wd), self.mean_n, self.theta
        coords = coords.permute(0, 1, 4, 2, 3).contiguous().view(E, 2, ht, wd)

        m = CorrSampler.apply(self.corr_pyramid[1], coords / 2, MASK_RADIUS)
        var = torch.var(m.permute(0, 3, 4, 1, 2), dim=[3, 4])
        self.offset[1] = self.offset[1] * torch.sigmoid(var).view(E, ht, wd, 1)     # cumulative per call (quirk Q7)

        out = []
        for i in range(self.num_levels):
            o = self.offset[i].contiguous().view(E, ht, wd, rd, rd, 2)
            corr = DefCorrSampler.apply(self.corr_pyramid[i], coords / 2 ** i, o, self.radius)
            out.append(corr.view(batch, num, -1, ht, wd))
        return torch.cat(out, dim=2), self.mean_n, self.theta

    @torch.no_grad()
    def lookup_encoded(self, coords, corr_encoder, keep_corr=False, enc_half=False):
        """__call__ with the consumer's first layer folded into the lookup kernel (SURVEY 8f-4; inference): corr_encoder is
        UpdateModule.corr_encoder (droid_net.py:74-78) or its first conv; returns (enc, mean_n, theta) with
        enc = relu(conv1x1(corr)) [b,n,128,h,w] -- feed it to corr_encoder[2:] -- or (corr, enc, mean_n, theta) with
        keep_corr=True.  The 196-channel tensor is not written unless asked for."""
        conv = _encoder_conv(corr_encoder)
        batch, num, ht, wd, _ = coords.shape
        E = batch * num
        if not self._can_fuse_lookup(coords):
            raise RuntimeError("lookup_encoded needs the fused lookup (4 levels, r = 3, W % 32 == 0, H % 8 == 0)")
        key = (id(conv), conv.weight._version, conv.weight.data_ptr())
        if getattr(self, "_enc_key", None) != key:
            self._enc_key, self._enc_frag = key, ops.pack_conv1x1(conv.weight.float())
        if not isinstance(self.offset, _Offsets):
            self.offset = _Offsets(self.offset)
        if not (self.offset[0].is_contiguous() and self.offset[0].dtype == torch.float32):
            self.offset[0] = self.offset[0].float().contiguous()
        pyr = [t if t.is_contiguous() else t.contiguous() for t in self.corr_pyramid]
        c = coords.detach().reshape(E, ht, wd, 2).float().contiguous()
        base, cum = self.offset.factored()
        bias = conv.bias.detach().float().contiguous() if conv.bias is not None else None
        corr, enc = ops.corr_lookup_fused_enc(pyr, c, self.offset[0], base, cum, self._enc_frag, bias, relu=True,
                                              keep_corr=keep_corr, enc_half=enc_half)
        enc = enc.view(batch, num, 128, ht, wd)
        if keep_corr:
            return corr.view(batch, num, -1, ht, wd), enc, self.mean_n, self.theta
        return enc, self.mean_n, self.theta

    def cat(self, other):
        for i in range(self.num_levels):
            self.corr_pyramid[i] = torch.cat([self.corr_pyramid[i], other.corr_pyramid[i]], 0)
        self.offset = _Offsets(self.offset).cat(other.offset) if not isinstance(self.offset, _Offsets) \
            else self.offset.cat(other.offset)
        return self

    def __getitem__(self, index):
        for i in range(self.num_levels):
            self.corr_pyramid[i] = self.corr_pyramid[i][index]
        self.offset = (self.offset if isinstance(self.offset, _Offsets) else _Offsets(self.offset)).index(index)
        return self

    @staticmethod
    def corr(fmap1, fmap2):
        """corr.py:144-152, all-pairs correlation through torch (the differentiable per-op path)."""
        batch, num, dim, ht, wd = fmap1.shape
        f1 = fmap1.reshape(batch * num, dim, ht * wd) / 4.0
        f2 = fmap2.reshape(batch * num, dim, ht * wd) / 4.0
        return torch.matmul(f1.transpose(1, 2), f2).view(batch, num, 1, ht * wd, ht, wd)


# ------------------------------------------------------------------------------------------------
# Edge-slot pool (SURVEY section 8f-2): CorrBlock.cat / __getitem__ without copying the pyramid
# ------------------------------------------------------------------------------------------------
class CorrPool:
    """Storage for up to `capacity` edges: the four pyramid levels [capacity,h,w,h>>l,w>>l] and the two offset tensors
    [capacity,h,w,98], allocated once.  The frontend's factor graph adds and drops edges on every keyframe
    (factor_graph.py:90-167); with the reference's CorrBlock each of those is a torch.cat / boolean-index COPY of the
    whole pyramid (corr.py:111-115,137-141; <= 2.4 GB at 48 edges).  Here an edge is a slot number."""

    def __init__(self, capacity, h, w, device, num_levels=4, radius=3):
        self.capacity, self.h, self.w, self.num_levels, self.radius = capacity, h, w, num_levels, radius
        self.levels = [torch.empty(capacity, h, w, h >> l, w >> l, dtype=torch.float32, device=device)
                       for l in range(num_levels)]
        nch = 2 * (2 * radius + 1) ** 2
        self.off0 = torch.zeros(capacity, h, w, nch, dtype=torch.float32, device=device)
        self.off1 = torch.zeros(capacity, h, w, nch, dtype=torch.float32, device=device)
        self.cum = torch.ones(capacity, h, w, dtype=torch.float32, device=device)    # running product of each slot's masks (Q7)
        self.free = list(range(capacity - 1, -1, -1))

    def alloc(self, n):
        if n > len(self.free):
            raise RuntimeError(f"CorrPool: {n} slots requested, {len(self.free)} free of {self.capacity}")
        return [self.free.pop() for _ in range(n)]

    def release(self, slots):
        slots = list(slots)
        self.check(slots)
        if set(slots) & set(self.free):
            raise RuntimeError("CorrPool: double release of a slot")
        self.free.extend(reversed(slots))

    def check(self, slots):
        """Host-side range check of a slot list before it is uploaded: a device-side slot >= capacity would read and
        write out of bounds through the TMA store maps and the offset pointers."""
        bad = [s for s in slots if not 0 <= int(s) < self.capacity]
        if bad or len(set(slots)) != len(slots):
            raise RuntimeError(f"CorrPool: invalid slot list {slots} for capacity {self.capacity}")


class PooledCorrBlock:
    """CorrBlock (corr.py:53-152) for inference on a CorrPool: same constructor arguments (+ pool), same
    `__call__(coords) -> (corr, mean_n, theta)`, `cat`, `__getitem__`; edges live in pool slots, so `cat` and
    `__getitem__` only edit the slot list.  Build = one tcgen05 launch into the slots, lookup = one TMA-staged launch."""

    def __init__(self, pool, ofsMap, ofs_residual, GA, fmap1, fmap2, num_levels=4, radius=3, autocast_rounding=False):
        assert num_levels == pool.num_levels == 4 and radius == pool.radius == 3
        self.pool, self.num_levels, self.radius = pool, num_levels, radius
        self.GA, self.ofsMap, self.ofs_residual = GA, ofsMap, ofs_residual
        b, n, c, h, w = fmap1.shape
        E = b * n
        assert (h, w) == (pool.h, pool.w) and w == 64 and h % 8 == 0 and c == 128
        self.batch = b
        with torch.no_grad():
            f1, f2 = fmap1.reshape(E, c, h, w), fmap2.reshape(E, c, h, w)
            t = torch.cat((f1, f2), dim=1)
            offs = _generate_offsets(ofsMap, ofs_residual, t.float())
            mean, cov, det = GA.params(t.permute(0, 2, 3, 1).float())
            self.slots = pool.alloc(E)
            # slots go back to the pool when the block is dropped in any way (self.corr = None, an exception, GC), not
            # only through __getitem__ / release(); the box is shared with the finalizer and updated by cat / __getitem__
            self._owned = [list(self.slots)]
            self._finalizer = weakref.finalize(self, PooledCorrBlock._give_back, pool, self._owned)
            sl = torch.tensor(self.slots, dtype=torch.int32, device=fmap1.device)
            idx = sl.long()
            pool.off0[idx] = offs[0]
            pool.off1[idx] = offs[1]
            pool.cum[idx] = 1.0
            frames = torch.cat((f1, f2), dim=0).contiguous()
            hi, lo = ops.pack_fmaps(frames, split=frames.dtype == torch.float32)
            ar = torch.arange(2 * E, dtype=torch.int32, device=frames.device)
            # den = 6.28 * sqrt(det) is formed in the build kernel's prologue (same fp32 roundings)
            ops.build_pyramid(hi, lo, ar[:E].contiguous(), ar[E:].contiguous(), h, w, means=mean.float().contiguous(),
                              covs=cov.contiguous(), den=None, num_levels=num_levels, gauss_radius=GAUSS_RADIUS,
                              round_half=autocast_rounding, out=pool.levels, out_slots=sl)
        self.mean_n = mean.view(E, h, w, 2)
        self.theta = 2 * det.view(E, h, w)
        self._sl = sl

    @staticmethod
    def _give_back(pool, owned):
        slots, owned[0] = owned[0], []
        if slots:
            pool.release(slots)

    def _set_slots(self, slots):
        self.slots = slots
        self._owned[0] = list(slots)
        self._sl = None

    def _slot_tensor(self, device):
        if self._sl is None or self._sl.numel() != len(self.slots):
            self.pool.check(self.slots)
            self._sl = torch.tensor(self.slots, dtype=torch.int32, device=device)
        return self._sl

    def __len__(self):
        return len(self.slots)

    @torch.no_grad()
    def __call__(self, coords):
        batch, num, ht, wd, _ = coords.shape
        E = batch * num
        assert E == len(self.slots), f"coords carry {E} edges, the block holds {len(self.slots)}"
        c = coords.reshape(E, ht, wd, 2).float().contiguous()
        out = ops.corr_lookup_fused(self.pool.levels, c, self.pool.off0, self.pool.off1, self.radius,
                                    slots=self._slot_tensor(c.device), cum_mask=self.pool.cum)
        return out.view(batch, num, -1, ht, wd), self.mean_n.view(batch, num, ht, wd, 2), self.theta.view(batch, num, ht, wd)

    def cat(self, other):
        assert other.pool is self.pool, "cat needs blocks of the same CorrPool"
        taken = list(other.slots)
        other._set_slots([])
        self._set_slots(self.slots + taken)
        self.mean_n = torch.cat([self.mean_n, other.mean_n], 0)
        self.theta = torch.cat([self.theta, other.theta], 0)
        return self

    def __getitem__(self, index):
        n = len(self.slots)
        keep = torch.arange(n)[index.cpu() if isinstance(index, torch.Tensor) else index].tolist()
        kept = set(keep)
        dropped = [s for i, s in enumerate(self.slots) if i not in kept]
        self._set_slots([self.slots[i] for i in keep])
        self.pool.release(dropped)
        self.mean_n, self.theta = self.mean_n[index], self.theta[index]
        return self

    def release(self):
        """Return every slot to the pool (idempotent; also runs when the block is garbage-collected)."""
        self.slots = []
        self._sl = None
        PooledCorrBlock._give_back(self.pool, self._owned)


# ------------------------------------------------------------------------------------------------
# AltCorrBlock (backend, no volume)
# ------------------------------------------------------------------------------------------------
class AltCorrBlock:
    """corr.py:155-249: correlation for global BA without a persistent volume.  `strict_ref=True` keeps the
    reference's offset-slab indexing (quirk Q2: with S == 1 every edge of a chunk reads edge 0's offsets).

    materialize=True (default where supported: 4 levels, r = 3, C = 128, H*W % 128 == 0, W % 32 == 0): each call
    builds the chunk's four volumes (level-0 source maps x level-l pooled target maps) on tcgen05 into scratch HBM
    (50 MB / edge; the reference's on-the-fly sampler exists only because 12-24 GB GPUs could not hold them) and
    samples them with the fused TMA-staged lookup in per-corner-gating mode.  materialize=False: the reference's
    op sequence on the drop-in operators (altcorr_forward + 4 x lowMem_defSample)."""

    MAX_EDGES_PER_PASS = 256          # scratch bound: 256 x 50 MB = 12.8 GB

    def __init__(self, ofsMap, ofs_residual, GA, fmaps, num_levels=4, radius=3, strict_ref=True, materialize=None,
                 sampler_ops=None, cache=False, volume_cache_gb=None, sparse_volumes=True, compact_boxes=True):
        """sparse_volumes (materialised path, volumes not cached): level 0 is built only where the lookup's per-pixel
        boxes can reach (lgu_volume_half_mask / lgu_build_volume_sparse); results are identical.
        cache (materialised path only): global BA calls the SAME block for the same chunks in every one of its
        `steps` iterations (factor_graph.py:265-279) while the feature maps stay fixed, so everything that depends
        only on (ii, jj) is kept per chunk after the first call:
          * the pre-mask offsets -- the two 3x3 convs and the normalise / tanh / permute chain of corr.py:217-235 are
            2/3 of a backend step on B200; under strict_ref only edge 0's slab is ever read by the sampler (quirk Q2),
            so only that slab is generated (the `offset` attribute then holds [1,H,W,98] tensors);
          * the chunk's four volumes, up to `volume_cache_gb` of HBM (None: half of the memory free at construction;
            0: off).  50 MB per edge: the reference samples on the fly because 12-24 GB GPUs cannot hold them -- 180 GB
            per B200 hold ~1800 edges, an 8-GPU box the whole 4k-edge graph.
        Same arithmetic per edge as cache=False (the convs see a batch of 1 instead of N under strict_ref, so cuDNN may
        pick another algorithm: differences stay at conv rounding level); repeated calls are bit-identical.  Only
        coords-dependent work (mask, lookups) runs per call.
        `clear_cache()` drops everything (call it when the feature maps change)."""
        self.cache = bool(cache)
        self.sparse_volumes = bool(sparse_volumes)
        # level 0 as compact boxes (default) or as volume rows.  Level 1 as compact boxes too was measured slower (46.6
        # against 44.5 ms per 4096-edge step: a level-1 slice is only 3 KB, its mask keeps 90 % of the halves, and the box
        # rows leave as scattered 16-byte stores instead of full lines)
        self.compact_boxes = bool(compact_boxes)
        self._cache = {}
        self._vol_bytes = 0
        if volume_cache_gb is None and self.cache and fmaps.is_cuda:
            volume_cache_gb = 0.5 * torch.cuda.mem_get_info(fmaps.device)[0] / 2**30
        self._vol_budget = int((volume_cache_gb or 0) * 2**30) if self.cache else 0
        # sampler_ops: object with altcorr_forward / lowMem_defSample (default: this package's operators); benchmarks
        # pass the reference's compiled extension here to time its kernels inside the same Python glue
        self.sampler_ops = sampler_ops if sampler_ops is not None else ops
        self.num_levels = num_levels
        self.radius = radius
        self.GA = GA
        self.ofsMap = ofsMap
        self.ofs_residual = ofs_residual
        self.strict_ref = strict_ref
        self.offset = []
        B, N, C, H, W = fmaps.shape
        cur = fmaps.reshape(B * N, C, H, W) / 4.0
        self.pyramid = []
        for i in range(num_levels):
            self.pyramid.append(cur.permute(0, 2, 3, 1).contiguous().view(B, N, H >> i, W >> i, C))
            cur = F.avg_pool2d(cur, 2, stride=2)
        can = (num_levels == 4 and radius == 3 and C == 128 and (H * W) % 128 == 0 and W % 32 == 0 and H % 8 == 0
               and B == 1 and fmaps.is_cuda)
        self.materialize = can if materialize is None else (materialize and can)
        self._planes = None

    def _level_planes(self):
        """Channels-last fp16 operand planes per level: the pyramid itself when the buffer is fp16 (the backend's case,
        depth_video.py:36 -- products are then exact), hi/lo split for fp32 buffers."""
        if self._planes is None:
            planes = []
            for lvl in self.pyramid:
                x = lvl.reshape(lvl.shape[1], -1, lvl.shape[-1])                  # [T, Q_l, C] (B == 1)
                if x.dtype == torch.float16:
                    planes.append((x.contiguous(), None))
                else:
                    hi = x.float().half()
                    planes.append((hi.contiguous(), (x.float() - hi.float()).half().contiguous()))
            self._planes = planes
        return self._planes

    def clear_cache(self):
        self._cache.clear()
        self._vol_bytes = 0

    def _gen_offsets(self, ii, jj):
        """corr.py:186-189 for the given edges: cat(f1, f2) -> offset heads -> 4 x [n,H,W,98]."""
        f1 = self.pyramid[0][0, ii]
        f2 = self.pyramid[0][0, jj]
        t = torch.cat(((f1 * 4.0).permute(0, 3, 1, 2), (f2 * 4.0).permute(0, 3, 1, 2)), dim=1).float()
        return _generate_offsets(self.ofsMap, self.ofs_residual, t)

    def _corr_materialized(self, coords, ii, jj, out=None, out_index=None, pass_edges=None, pass_hook=None, key=None,
                           enc=None):
        """enc: fp16 operands of the consumer's first layer (ops.pack_conv1x1_f16); the lookup then returns / writes
        relu(conv1x1(corr)) [.., 128, H, W] instead of corr."""
        B, N, H, W, S, _ = coords.shape
        # pass_edges: an int (edges per pass) or a sequence of pass sizes (the sharded engine tapers the passes of a rank's
        # last chunk so that only a small shipment is left exposed at the end of the step)
        if pass_edges is not None and not isinstance(pass_edges, int):
            sizes = [min(self.MAX_EDGES_PER_PASS, max(1, int(x))) for x in pass_edges]
        else:
            sizes = [min(self.MAX_EDGES_PER_PASS, int(pass_edges)) if pass_edges else self.MAX_EDGES_PER_PASS]
        bounds, s0, k = [], 0, 0
        while s0 < N:
            n = sizes[min(k, len(sizes) - 1)]
            bounds.append((s0, min(N, s0 + n)))
            s0 += n
            k += 1
        assert B == 1 and S == 1, "the materialised path serves the reference's only call shape (B = S = 1)"
        planes = self._level_planes()
        c = coords.reshape(N, H, W, 2).float().contiguous()
        ii32, jj32 = ii.to(torch.int32).contiguous(), jj.to(torch.int32).contiguous()
        ent = None
        if self.cache:
            # cache key of the chunk: the caller's (e.g. the sharded engine's chunk id) if given -- reading the edge list
            # back from the device costs a host synchronisation per chunk
            key = key if key is not None else (tuple(ii.tolist()), tuple(jj.tolist()))
            ent = self._cache.get(key)
            if ent is None:
                # strict_ref: only slab 0 is ever read (Q2) -> generate just that slab
                n_off = 1 if self.strict_ref else N
                offs = self._gen_offsets(ii[:n_off], jj[:n_off])
                ent = self._cache[key] = {"off": [o.float().contiguous() for o in offs], "vols": {}}
            self.offset = list(ent["off"])                  # pre-mask; offset[1] is replaced below, never mutated
        else:
            self.offset = self._gen_offsets(ii, jj)
        n_off = self.offset[0].shape[0]
        off0 = self.offset[0].reshape(n_off, H, W, -1).float().contiguous()
        off1 = self.offset[1].reshape(n_off, H, W, -1).float().contiguous()
        if self.strict_ref:
            # Q2: every edge samples with edge 0's offsets; edge 0's level-1 offsets carry edge 0's mask (corr.py:201-206)
            f1 = self.pyramid[0][0, ii[:1]].float().contiguous()
            f2 = self.pyramid[1][0, jj[:1]].float().contiguous()
            m0, = ops.altcorr_forward(f1, f2, (c[:1] / 2).view(1, 1, H, W, 2).contiguous(), MASK_RADIUS)
            mask0 = torch.sigmoid(torch.var(m0.permute(0, 1, 3, 4, 2).reshape(1, H, W, 9), dim=3))
            slab0 = (off0[:1].contiguous(), (off1[:1] * mask0.view(1, H, W, 1)).contiguous())
        lookup = ops.altcorr_lookup_fused if enc is None else functools.partial(ops.altcorr_lookup_encoded, packed=enc)
        outs, masks, new_off1 = [], [], []
        for s, s_end in bounds:
            e = slice(s, s_end)
            # keyed by the pass's edge range: a later call with another pass schedule must not pick up volumes built
            # for different edges
            vols = ent["vols"].get((s, s_end)) if ent is not None else None
            boxes0 = None
            if vols is None:
                # Level 0 is 3/4 of the volume bytes, and the lookup below reads it only inside a 20 x 16 box per source
                # pixel (offsets are 4 * tanh, corr.py:121-128): build only the row bands those boxes touch.  Not when the
                # volumes are kept for later calls with other coords (the per-chunk cache).
                sparse = self.sparse_volumes and self._vol_budget == 0 and (H * W) % 128 == 0 and 256 % W == 0
                hm = ops.volume_half_mask(c[e], 0) if sparse else None
                # ... and with fp16-valued maps (the backend's buffer) and W = 64 level 0 is not written as rows at all:
                # every source pixel keeps just the 16 x 20 box the lookup stages (1.3 KB instead of 7.6 KB of rows)
                if sparse and self.compact_boxes and W == 64 and H % 4 == 0 and planes[0][1] is None:
                    boxes0 = ops.build_boxes(planes[0][0], planes[0][0], ii32[e], jj32[e], c[e], half_mask=hm)
                vols = [None if (l == 0 and boxes0 is not None) else
                        ops.build_volume(planes[0][0], planes[0][1], planes[l][0], planes[l][1], ii32[e], jj32[e],
                                         half_mask=hm if l == 0 else None).view(-1, H, W, H >> l, W >> l)
                        for l in range(self.num_levels)]
                nbytes = sum(v.numel() * 4 for v in vols if v is not None)
                if ent is not None and self._vol_bytes + nbytes <= self._vol_budget:
                    ent["vols"][(s, s_end)] = vols
                    self._vol_bytes += nbytes
            # out / out_index: this pass's edges are written straight to their rows of the caller's buffer
            dst = dict(out=out, out_index=(out_index[e].contiguous() if out_index is not None else
                                           torch.arange(e.start, e.stop, dtype=torch.int32, device=c.device))) \
                if out is not None else {}
            if self.strict_ref:
                o, m = lookup(vols, c[e], slab0[0], slab0[1], self.radius, shared_offsets=True,
                              apply_mask=False, return_mask=True, boxes0=boxes0, **dst)
            else:
                o1 = off1[e].clone()                                      # updated in place: offset[1] * mask
                o, m = lookup(vols, c[e], off0[e].contiguous(), o1, self.radius, shared_offsets=False,
                              apply_mask=True, return_mask=True, boxes0=boxes0, **dst)
                new_off1.append(o1)
            outs.append(o)
            masks.append(m)
            del vols, boxes0
            if pass_hook is not None:                             # rows e.start .. e.stop of this call are enqueued
                pass_hook(e.start, e.stop)
        # the attribute the reference leaves behind: offset[1] * mask (corr.py:206)
        if self.strict_ref:
            if n_off == N:
                self.offset[1] = self.offset[1] * torch.cat(masks, 0).view(N, H, W, 1)
            else:
                self.offset[1] = slab0[1]
        else:
            self.offset[1] = torch.cat(new_off1, 0) if len(new_off1) > 1 else new_off1[0]
        if out is not None:
            return out
        res = torch.cat(outs, 0) if len(outs) > 1 else outs[0]
        return res.view(B, N, -1, H, W, 1)

    def corr_fn(self, coords, ii, jj, out=None, out_index=None, pass_edges=None, pass_hook=None, key=None):
        B, N, H, W, S, _ = coords.shape
        rd = 2 * self.radius + 1
        if self.materialize and B == 1 and S == 1:
            return self._corr_materialized(coords, ii, jj, out, out_index, pass_edges, pass_hook, key)
        if out is not None:
            raise RuntimeError("out= needs the materialised path (4 levels, r = 3, C = 128, B = S = 1)")
        f1 = self.pyramid[0][:, ii]
        f1 = f1.reshape((B * N,) + f1.shape[2:])
        f2 = self.pyramid[0][:, jj]
        f2 = f2.reshape((B * N,) + f2.shape[2:])
        t = torch.cat(((f1 * 4.0).permute(0, 3, 1, 2), (f2 * 4.0).permute(0, 3, 1, 2)), dim=1).float()
        self.offset = _generate_offsets(self.ofsMap, self.ofs_residual, t)
        coords = coords.permute(0, 1, 4, 2, 3, 5)
        f1 = f1.float().contiguous()

        out = []
        for i in range(self.num_levels):
            f2_i = self.pyramid[i][:, jj]
            f2_i = f2_i.reshape((B * N,) + f2_i.shape[2:]).float().contiguous()
            coords_i = (coords / 2 ** i).reshape(B * N, S, H, W, 2).contiguous()
            if i == 1:
                m, = self.sampler_ops.altcorr_forward(f1, f2_i, coords_i, MASK_RADIUS)
                m = m.permute(0, 1, 3, 4, 2).contiguous().view(N, H, W, 3, 3)       # corr.py:203 (assumes B == S == 1)
                self.offset[1] = self.offset[1] * torch.sigmoid(torch.var(m, dim=[3, 4])).view(B * N, H, W, 1)
            o = self.offset[i].contiguous().view(B * N, H, W, rd, rd, 2).float()
            if self.sampler_ops is ops:
                corr, = ops.lowMem_defSample(f1, f2_i, coords_i, o, self.radius, strict_ref=self.strict_ref)
            else:
                corr, = self.sampler_ops.lowMem_defSample(f1, f2_i, coords_i, o, self.radius)
            out.append(corr.view(B, N, S, -1, H, W).permute(0, 1, 3, 4, 5, 2))
        return torch.cat(out, dim=2)

    def __call__(self, coords, ii, jj, out=None, out_index=None, pass_edges=None, pass_hook=None, key=None):
        """corr.py:238-249.  out / out_index (materialised path only): write edge e's [196,H,W] result into row
        out_index[e] of `out` ([E_out,196,H,W], fp32 or fp16 -- possibly another GPU's memory, see sharded.PeerOutput)
        instead of returning a new tensor; `out` is returned.  pass_edges / pass_hook: the chunk is processed in passes of
        at most pass_edges edges (volumes + lookup per pass) and pass_hook(first, last) is called after each pass's
        launches are enqueued -- the sharded backend ships finished rows while the next pass computes.  key: hashable
        identity of this chunk for cache=True (default: the edge lists themselves, read back from the device)."""
        squeeze = coords.dim() == 5
        if squeeze:
            coords = coords.unsqueeze(dim=-2)
        corr = self.corr_fn(coords, ii, jj, out, out_index, pass_edges, pass_hook, key)
        if out is not None:
            return out
        if squeeze:
            corr = corr.squeeze(dim=-1)
        return corr.contiguous()

    @torch.no_grad()
    def lookup_encoded(self, coords, ii, jj, corr_encoder, out=None, out_index=None, pass_edges=None, pass_hook=None,
                       key=None):
        """__call__ with the consumer's first layer folded into the lookup kernel (inference): corr_encoder is
        UpdateModule.corr_encoder (droid_net.py:74-78) or its first conv.  Returns relu(conv1x1(corr)) [1,E,128,H,W] fp16,
        evaluated as update_op does under fp16 autocast (factor_graph.py:281-286: operands rounded to fp16, fp32
        accumulation, relu keeps NaN) -- feed it to corr_encoder[2:].  With out ([E_out,128,H,W], fp16 or fp32) / out_index
        the rows are written there and `out` is returned, like __call__; pass_edges / pass_hook / key as there, so a
        ShardedBackendCorr can use this (with corr_encoder bound) as its compute and ship 128 instead of 196 channels per
        pixel.  Leaves the same `offset` attribute as __call__.  Needs the materialised path (B = S = 1, 4 levels, r = 3,
        C = 128, W % 32 == 0, H % 8 == 0)."""
        conv = _encoder_conv(corr_encoder)
        if coords.dim() == 5:
            coords = coords.unsqueeze(dim=-2)
        B, N, H, W, S, _ = coords.shape
        if not (self.materialize and B == 1 and S == 1):
            raise RuntimeError("lookup_encoded needs the materialised backend lookup (B = S = 1, 4 levels, r = 3, C = 128, "
                               "W % 32 == 0, H % 8 == 0)")
        bias = conv.bias
        pkey = (id(conv), conv.weight._version, conv.weight.data_ptr(),
                None if bias is None else (bias._version, bias.data_ptr()))
        if getattr(self, "_enc_key", None) != pkey:
            w = conv.weight.detach().to(coords.device, torch.float32)
            b = bias.detach().to(coords.device, torch.float32) if bias is not None else None
            self._enc_key, self._enc_packed = pkey, ops.pack_conv1x1_f16(w, b)
        res = self._corr_materialized(coords, ii, jj, out, out_index, pass_edges, pass_hook, key, enc=self._enc_packed)
        return res if out is not None else res.view(B, N, -1, H, W)

"""Operator layer: the reference's `defCorrSample` operators (and `droid_backends.altcorr_forward`)
on torch CUDA tensors, implemented by the sm_100a C-ABI library.

Signatures, argument meaning, in-place side effects and error behaviour follow
/root/reference/offersample_LGS/droid.cpp:53-136 (each returns a list of tensors that callers
unpack with `x, = op(...)`); the only checks the reference performs are `is_contiguous`
(droid.cpp:48-49) and the accessor's dtype/ndim checks, which surface as RuntimeError -- same here,
plus explicit device/shape checks.  torch is used only for allocation and the current stream.
"""
import torch

from . import _lib


def _chk(t, name, ndim, dtype=torch.float32):
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor")
    if not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor (this build has no CPU path)")
    if not t.is_contiguous():
        raise RuntimeError(f"{name} must be contiguous")          # droid.cpp:48
    if t.dtype != dtype:
        raise RuntimeError(f"{name}: expected dtype {dtype}, got {t.dtype}")
    if t.dim() != ndim:
        raise RuntimeError(f"{name}: expected {ndim} dimensions, got {t.dim()}")


def _launch(name, device, *args):
    """Call entry point `name` on `device` with the device's current stream appended; a non-zero status raises."""
    with torch.cuda.device(device):
        return _lib.call(name, *args, torch.cuda.current_stream(device).cuda_stream)


def _launch_ext(name, device, *args):
    """_launch for an entry point of include/lgu_corr_ext.h (the additions to the version-1 C ABI)."""
    with torch.cuda.device(device):
        return _lib.call_ext(name, *args, torch.cuda.current_stream(device).cuda_stream)


def _check_levels(levels, S, H, W, name, skip=()):
    """Pyramid levels [S,H,W,H>>l,W>>l] (fp32, contiguous, CUDA); the levels listed in `skip` are not read."""
    for l, t in enumerate(levels):
        if l not in skip:
            _chk(t, f"{name}[{l}]", 5)
            if tuple(t.shape) != (S, H, W, H >> l, W >> l):
                raise RuntimeError(f"{name}[{l}] shape {tuple(t.shape)} != {(S, H, W, H >> l, W >> l)}")


def _check_offsets(numel, exact=True, **offsets):
    """Offset tensors [*,H,W,98] / [*,H,W,7,7,2]: contiguous fp32 CUDA with `numel` elements (at least `numel` if not
    exact)."""
    for name, o in offsets.items():
        if not (isinstance(o, torch.Tensor) and o.is_cuda and o.is_contiguous() and o.dtype == torch.float32
                and (o.numel() == numel if exact else o.numel() >= numel)):
            raise RuntimeError(f"{name} must be a contiguous fp32 CUDA tensor with {'' if exact else '>= '}{numel} elements")


def _check_index(t, name, n=None):
    """A contiguous CUDA int32 vector (edge / slot / row indices), with n entries if n is given."""
    if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.int32 and t.dim() == 1 and t.is_contiguous()
            and (n is None or t.numel() == n)):
        raise RuntimeError(f"{name} must be a contiguous CUDA int32 vector" + ("" if n is None else f" with {n} entries"))


def _check_plane(t, name):
    """A channels-last fp16 plane [T,P,C] as pack_fmaps returns it."""
    if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.float16 and t.dim() == 3 and t.is_contiguous()):
        raise RuntimeError(f"{name} must be a contiguous CUDA fp16 tensor [T,P,C] (see pack_fmaps)")


def _check_means_covs(means, covs, E, H, W):
    """The Gaussian parameters: means, covs [E,H,W,2] (channel 0 = x, 1 = y)."""
    _chk(means, "means", 4); _chk(covs, "covs", 4)
    if tuple(means.shape) != (E, H, W, 2) or tuple(covs.shape) != (E, H, W, 2):
        raise RuntimeError(f"means/covs must be [E,H,W,2] = {[E, H, W, 2]}")


def _encoder_weight(weight):
    """corr_encoder[0].weight [128,196] or [128,196,1,1] -> contiguous [128,196], the only shape the kernels implement."""
    if not (isinstance(weight, torch.Tensor) and weight.is_cuda and weight.dtype == torch.float32):
        raise RuntimeError("weight must be a CUDA fp32 tensor")
    w = weight.detach().reshape(weight.shape[0], -1).contiguous()
    if tuple(w.shape) != (128, 196):
        raise RuntimeError(f"only the 196 -> 128 corr_encoder is implemented, got weight {tuple(weight.shape)}")
    return w


def corr_index_forward(volume, coords, radius):
    """droid.cpp:79-87.  volume [E,H1,W1,H2,W2], coords [E,2,H1,W1] -> [corr [E,rd,rd,H1,W1]]."""
    _chk(volume, "volume", 5); _chk(coords, "coords", 4)
    E, H1, W1, H2, W2 = volume.shape
    if tuple(coords.shape) != (E, 2, H1, W1):
        raise RuntimeError(f"coords shape {tuple(coords.shape)} != {(E, 2, H1, W1)}")
    rd = 2 * int(radius) + 1
    corr = torch.empty(E, rd, rd, H1, W1, dtype=volume.dtype, device=volume.device)
    _launch("lgu_corr_index_forward", volume.device, volume, coords, corr, E, H1, W1, H2, W2, int(radius))
    return [corr]


def corr_index_backward(volume, coords, corr_grad, radius):
    """droid.cpp:89-99 -> [volume_grad] (dense)."""
    _chk(volume, "volume", 5); _chk(coords, "coords", 4); _chk(corr_grad, "corr_grad", 5)
    E, H1, W1, H2, W2 = volume.shape
    rd = 2 * int(radius) + 1
    if tuple(corr_grad.shape) != (E, rd, rd, H1, W1):
        raise RuntimeError(f"corr_grad shape {tuple(corr_grad.shape)} != {(E, rd, rd, H1, W1)}")
    volume_grad = torch.empty_like(volume)
    _launch("lgu_corr_index_backward", volume.device, coords, corr_grad, volume_grad, E, H1, W1, H2, W2, int(radius))
    return [volume_grad]


def defCorr_index_forward(volume, coords, offset, radius):
    """droid.cpp:53-63.  offset [E,H1,W1,rd,rd,2] is mutated (centre tap zeroed)."""
    _chk(volume, "volume", 5); _chk(coords, "coords", 4); _chk(offset, "offset", 6)
    E, H1, W1, H2, W2 = volume.shape
    rd = 2 * int(radius) + 1
    if tuple(offset.shape) != (E, H1, W1, rd, rd, 2):
        raise RuntimeError(f"offset shape {tuple(offset.shape)} != {(E, H1, W1, rd, rd, 2)}")
    if tuple(coords.shape) != (E, 2, H1, W1):
        raise RuntimeError(f"coords shape {tuple(coords.shape)} != {(E, 2, H1, W1)}")
    corr = torch.empty(E, rd, rd, H1, W1, dtype=volume.dtype, device=volume.device)
    _launch("lgu_defcorr_index_forward", volume.device, volume, coords, offset, corr, E, H1, W1, H2, W2, int(radius))
    return [corr]


def defCorr_index_backward(volume, coords, offset, corr_grad, radius):
    """droid.cpp:65-77 -> [volume_grad, offset_grad]."""
    _chk(volume, "volume", 5); _chk(coords, "coords", 4); _chk(offset, "offset", 6); _chk(corr_grad, "corr_grad", 5)
    E, H1, W1, H2, W2 = volume.shape
    rd = 2 * int(radius) + 1
    if tuple(offset.shape) != (E, H1, W1, rd, rd, 2):
        raise RuntimeError(f"offset shape {tuple(offset.shape)} != {(E, H1, W1, rd, rd, 2)}")
    if tuple(corr_grad.shape) != (E, rd, rd, H1, W1):
        raise RuntimeError(f"corr_grad shape {tuple(corr_grad.shape)} != {(E, rd, rd, H1, W1)}")
    volume_grad = torch.empty_like(volume)
    offset_grad = torch.empty_like(offset)
    _launch("lgu_defcorr_index_backward", volume.device, volume, coords, offset, corr_grad, volume_grad, offset_grad, E,
            H1, W1, H2, W2, int(radius))
    return [volume_grad, offset_grad]


def gaussianMask(means, covs, volume, radius):
    """droid.cpp:100-110.  means, covs [E,H1,W1,2] -> [volume1] (dense, zero outside the window)."""
    _chk(volume, "volume", 5)
    E, H1, W1, H2, W2 = volume.shape
    _check_means_covs(means, covs, E, H1, W1)
    out = torch.empty_like(volume)
    _launch("lgu_gaussian_mask_forward", volume.device, means, covs, volume, out, E, H1, W1, H2, W2, int(radius))
    return [out]


def gaussianMask_backward(means, covs, volume, volume1_grad, radius):
    """droid.cpp:112-123 -> [means_grad, covs_grad]."""
    _chk(volume, "volume", 5); _chk(volume1_grad, "volume_grad", 5)
    E, H1, W1, H2, W2 = volume.shape
    _check_means_covs(means, covs, E, H1, W1)
    if volume1_grad.shape != volume.shape:
        raise RuntimeError("volume_grad must have the volume's shape")
    gm = torch.empty_like(means)
    gc = torch.empty_like(covs)
    _launch("lgu_gaussian_mask_backward", volume.device, means, covs, volume, volume1_grad, gm, gc, E, H1, W1, H2, W2,
            int(radius))
    return [gm, gc]


# Workspace of the tensor-core lowMem / altcorr path: one grow-only byte buffer per device, reused by every call (the
# C ABI allocates nothing).  A call whose volume would not fit LOWMEM_WORKSPACE_CAP is processed in sub-batches of edges.
LOWMEM_WORKSPACE_CAP = 32 << 30
_workspaces = {}


def _workspace(device, nbytes):
    buf = _workspaces.get(device)
    if buf is None or buf.numel() < nbytes:
        _workspaces[device] = None                      # release the old buffer before growing
        buf = torch.empty(int(nbytes), dtype=torch.uint8, device=device)
        _workspaces[device] = buf
    return buf


def release_workspace():
    """Drop the cached tensor-core workspaces (they are re-created on demand)."""
    _workspaces.clear()


def _ws_bytes(B, N, H1, W1, H2, W2, C, radius):
    return _lib.call("lgu_lowmem_workspace_bytes", B, N, H1, W1, H2, W2, C, radius)


def _tensor_core_runs(device, B, N, H1, W1, H2, W2, C, radius):
    """Split B edges into runs whose workspace fits LOWMEM_WORKSPACE_CAP (usually one run): yields (b0, b1, workspace)."""
    step = B
    while step > 1 and _ws_bytes(step, N, H1, W1, H2, W2, C, radius) > LOWMEM_WORKSPACE_CAP:
        step = (step + 1) // 2
    for b0 in range(0, B, step):
        b1 = min(B, b0 + step)
        yield b0, b1, _workspace(device, _ws_bytes(b1 - b0, N, H1, W1, H2, W2, C, radius))


def lowMem_defSample(fmap1, fmap2, coords, offset, radius, strict_ref=True, tensor_cores=True):
    """droid.cpp:124-136.  fmap1 [B,H1,W1,C], fmap2 [B,H2,W2,C], coords [B,N,H1,W1,2],
    offset [slabs,H1,W1,rd,rd,2] (mutated) -> [corr [B,N,rd,rd,H1,W1]].
    strict_ref=True keeps the reference's offset[b*n] slab indexing (quirk Q2).
    tensor_cores (default): for the reference's call shape (N = 1, C = 128, r = 3, H1*W1 % 128 == 0, W2 % 4 == 0) this
    level's [B,P,Q] volume is built on tcgen05 into a cached workspace and sampled with the TMA-staged lookup
    (lgu_lowmem_defsample_forward_ws); other shapes, or tensor_cores=False, run the on-the-fly SIMT kernel."""
    _chk(fmap1, "fmap1", 4); _chk(fmap2, "fmap2", 4); _chk(coords, "coords", 5); _chk(offset, "offset", 6)
    B, H1, W1, C = fmap1.shape
    B2, H2, W2, C2 = fmap2.shape
    Bc, N, Hc, Wc, two = coords.shape
    rd = 2 * int(radius) + 1
    if B2 != B or C2 != C or Bc != B or (Hc, Wc, two) != (H1, W1, 2):
        raise RuntimeError("lowMem_defSample: inconsistent fmap/coords shapes")
    need = ((B - 1) * (N - 1) + 1) if strict_ref else B * N
    if tuple(offset.shape[1:]) != (H1, W1, rd, rd, 2) or offset.shape[0] < need:
        raise RuntimeError(f"offset shape {tuple(offset.shape)} incompatible with {(need, H1, W1, rd, rd, 2)}")
    corr = torch.empty(B, N, rd, rd, H1, W1, dtype=fmap1.dtype, device=fmap1.device)
    radius, strict = int(radius), 1 if strict_ref else 0
    if tensor_cores and B > 0 and _ws_bytes(B, N, H1, W1, H2, W2, C, radius) > 0:
        for b0, b1, ws in _tensor_core_runs(fmap1.device, B, N, H1, W1, H2, W2, C, radius):
            off = offset if strict_ref else offset[b0:]              # strict: every run reads slab 0 of the call (Q2)
            _launch("lgu_lowmem_defsample_forward_ws", fmap1.device, fmap1[b0:b1], fmap2[b0:b1], coords[b0:b1], off,
                    corr[b0:b1], b1 - b0, N, H1, W1, H2, W2, C, radius, strict, ws, ws.numel())
    else:
        _launch("lgu_lowmem_defsample_forward", fmap1.device, fmap1, fmap2, coords, offset, corr, B, N, H1, W1, H2, W2, C,
                radius, strict)
    return [corr]


def altcorr_forward(fmap1, fmap2, coords, radius, tensor_cores=True):
    """droid_backends.altcorr_forward (src/droid.cpp:193-203) -> [corr [B,N,rd*rd,H1,W1]].
    tensor_cores (default): for N = 1, C = 128, r = 1 (the reference's only call, corr.py:202) the volume is built on
    tcgen05 and sampled with per-corner gating (lgu_altcorr_forward_ws); otherwise the on-the-fly SIMT kernel."""
    _chk(fmap1, "fmap1", 4); _chk(fmap2, "fmap2", 4); _chk(coords, "coords", 5)
    B, H1, W1, C = fmap1.shape
    B2, H2, W2, C2 = fmap2.shape
    Bc, N, Hc, Wc, two = coords.shape
    rd = 2 * int(radius) + 1
    if B2 != B or C2 != C or Bc != B or (Hc, Wc, two) != (H1, W1, 2):
        raise RuntimeError("altcorr_forward: inconsistent fmap/coords shapes")
    corr = torch.empty(B, N, rd * rd, H1, W1, dtype=fmap1.dtype, device=fmap1.device)
    radius = int(radius)
    if tensor_cores and B > 0 and _ws_bytes(B, N, H1, W1, H2, W2, C, radius) > 0:
        for b0, b1, ws in _tensor_core_runs(fmap1.device, B, N, H1, W1, H2, W2, C, radius):
            _launch("lgu_altcorr_forward_ws", fmap1.device, fmap1[b0:b1], fmap2[b0:b1], coords[b0:b1], corr[b0:b1], b1 - b0,
                    N, H1, W1, H2, W2, C, radius, ws, ws.numel())
    else:
        _launch("lgu_altcorr_forward", fmap1.device, fmap1, fmap2, coords, corr, B, N, H1, W1, H2, W2, C, radius)
    return [corr]


# ----------------------------------------------------------------------------------------------
# Fused ops (no single reference operator; they replace sequences of the reference's Python glue)
# ----------------------------------------------------------------------------------------------
def _check_heads_inputs(c0, c1):
    _chk(c0, "c0", 4); _chk(c1, "c1", 4)
    E, CH, H, W = c0.shape
    if tuple(c1.shape) != (E, CH, H // 2, W // 2):
        raise RuntimeError(f"c1 shape {tuple(c1.shape)} != {(E, CH, H // 2, W // 2)}")
    return E, CH, H, W


def offset_heads(c0, c1, eps=1e-5, return_stats=False):
    """The offset heads' glue (corr.py:117-135 / 217-235) in two launches: c0 [E,CH,H,W] = ofsMap(t), c1 [E,CH,H/2,W/2] =
    ofs_residual(avg_pool2d(t, 2)) -> (off0, off1) [E,H,W,CH], channels-last and contiguous:
    off0 = 4 tanh(norm(c0)), off1 = (4 tanh(norm(upsample(c1))) + off0) / 2, norm = per-edge standardisation over
    (CH,H,W) with biased variance + eps (per_Corr_Normalization, corr.py:44-51).  With return_stats, also the per-edge
    statistics [E,4] = (mean0, sigma0, mean1, sigma1), sigma = sqrt(var + eps), which offset_heads_backward takes."""
    E, CH, H, W = _check_heads_inputs(c0, c1)
    off0 = torch.empty(E, H, W, CH, dtype=torch.float32, device=c0.device)
    off1 = torch.empty_like(off0)
    stats = torch.empty(E, 4, dtype=torch.float32, device=c0.device)
    _launch("lgu_offset_heads", c0.device, c0, c1, off0, off1, stats, E, CH, H, W, eps)
    return (off0, off1, stats) if return_stats else (off0, off1)


def offset_heads_backward(c0, c1, stats, g_off0, g_off1):
    """Backward of offset_heads in two launches: the forward's inputs c0, c1 and statistics, and the gradients of off0 /
    off1 ([E,H,W,CH], either may be None = zero) -> (g_c0 [E,CH,H,W], g_c1 [E,CH,H/2,W/2]).  Bit-identical from run to
    run (fp64 per-edge sums in a fixed order, no atomics)."""
    E, CH, H, W = _check_heads_inputs(c0, c1)
    _chk(stats, "stats", 2)
    if tuple(stats.shape) != (E, 4):
        raise RuntimeError(f"stats shape {tuple(stats.shape)} != {(E, 4)}")
    grads = {k: v for k, v in (("g_off0", g_off0), ("g_off1", g_off1)) if v is not None}
    _check_offsets(E * H * W * CH, **grads)
    g_c0 = torch.empty_like(c0)
    g_c1 = torch.empty_like(c1)
    scratch = torch.empty(max(1, E * (H // 2) * (W // 32)) * 4, dtype=torch.float64, device=c0.device)
    _launch_ext("lgu_offset_heads_backward", c0.device, c0, c1, stats, g_off0, g_off1, g_c0, g_c1, scratch, E, CH, H, W)
    return g_c0, g_c1


def _conv3x3_inputs(x, weight, bias=None):
    """Checks of conv3x3 / conv3x3_backward: x [E,C_in,H,W], weight [C_out,C_in,3,3], bias [C_out] or None, contiguous
    fp32 on one CUDA device, sizes the kernels implement."""
    _chk(x, "x", 4); _chk(weight, "weight", 4)
    E, C_in, H, W = x.shape
    C_out = weight.shape[0]
    if tuple(weight.shape) != (C_out, C_in, 3, 3):
        raise RuntimeError(f"weight shape {tuple(weight.shape)} != {(C_out, C_in, 3, 3)}")
    if bias is not None:
        _chk(bias, "bias", 1)
        if tuple(bias.shape) != (C_out,):
            raise RuntimeError(f"bias shape {tuple(bias.shape)} != {(C_out,)}")
    if any(t is not None and t.device != x.device for t in (weight, bias)):
        raise RuntimeError("x, weight and bias must be on one device")
    if not conv3x3_supported(C_in, C_out, H, W):
        raise RuntimeError(f"conv3x3: unsupported sizes C_in={C_in} C_out={C_out} H={H} W={W} (needs C_in % 32 == 0, "
                           "C_out <= 128, W % 32 == 0 dividing 128 or a multiple of 128, H*W % 128 == 0)")
    return E, C_in, C_out, H, W


def conv3x3_supported(C_in, C_out, H, W):
    """Whether the conv3x3 kernels implement these sizes (OffsetConv takes the library path only then)."""
    return (C_in > 0 and C_in % 32 == 0 and 0 < C_out <= 128 and W > 0 and W % 32 == 0
            and (128 % W == 0 or W % 128 == 0) and H > 0 and (H * W) % 128 == 0)


def _conv3x3_planes(t):
    """NCHW fp32 -> tf32 hi / lo planes [E,H,W,round_up(C,32)] (lgu_conv3x3_pack)."""
    E, C, H, W = t.shape
    hi = torch.empty(E, H, W, (C + 31) // 32 * 32, dtype=torch.float32, device=t.device)
    lo = torch.empty_like(hi)
    _launch_ext("lgu_conv3x3_pack", t.device, t, hi, lo, E, C, H, W)
    return hi, lo


def _conv3x3_workspace(device, E, C_in, C_out, H, W):
    nbytes = _lib.call_ext("lgu_conv3x3_workspace_bytes", E, C_in, C_out, H, W)
    return torch.empty(max(1, nbytes), dtype=torch.uint8, device=device), nbytes


def conv3x3(x, weight, bias=None):
    """F.conv2d(x, weight, bias, padding=1) for a 3x3 kernel (the offset heads, ofsMap / ofs_residual) in fp32 accuracy
    on tensor cores: x [E,C_in,H,W], weight [C_out,C_in,3,3], bias [C_out] or None -> y [E,C_out,H,W].  Two launches
    pack x into tf32 hi / lo planes, then one packs the weight and one runs the implicit GEMM."""
    E, C_in, C_out, H, W = _conv3x3_inputs(x, weight, bias)
    y = torch.empty(E, C_out, H, W, dtype=torch.float32, device=x.device)
    if E == 0:
        return y
    x_hi, x_lo = _conv3x3_planes(x)
    ws, nbytes = _conv3x3_workspace(x.device, E, C_in, C_out, H, W)
    _launch_ext("lgu_conv3x3_forward", x.device, x_hi, x_lo, weight, bias, y, ws, nbytes, E, C_in, C_out, H, W)
    return y


def conv3x3_backward(x, weight, g_y, need_input=True, need_weight=True, need_bias=None):
    """Backward of conv3x3: the forward's x and weight and the output gradient g_y [E,C_out,H,W] -> (g_x [E,C_in,H,W],
    g_w [C_out,C_in,3,3], g_b [C_out]), each None unless asked for (need_bias defaults to need_weight).  Bit-identical
    from run to run (the weight gradient's pixel sum is split by the sizes alone and reduced in a fixed order)."""
    E, C_in, C_out, H, W = _conv3x3_inputs(x, weight)
    _chk(g_y, "g_y", 4)
    if tuple(g_y.shape) != (E, C_out, H, W) or g_y.device != x.device:
        raise RuntimeError(f"g_y shape {tuple(g_y.shape)} != {(E, C_out, H, W)} (on x's device)")
    need_bias = need_weight if need_bias is None else need_bias
    g_x = torch.empty_like(x) if need_input else None
    g_w = torch.empty_like(weight) if need_weight else None
    g_b = torch.empty(C_out, dtype=torch.float32, device=x.device) if need_bias else None
    if E == 0:
        for t in (g_x, g_w, g_b):
            if t is not None:
                t.zero_()
        return g_x, g_w, g_b
    if not (need_input or need_weight or need_bias):
        return g_x, g_w, g_b
    ws, nbytes = _conv3x3_workspace(x.device, E, C_in, C_out, H, W)
    if need_input:
        gy_hi, gy_lo = _conv3x3_planes(g_y)
        _launch_ext("lgu_conv3x3_backward_input", x.device, gy_hi, gy_lo, weight, g_x, ws, nbytes, E, C_in, C_out, H, W)
        del gy_hi, gy_lo
    if need_weight or need_bias:
        x_hi, x_lo = _conv3x3_planes(x) if need_weight else (None, None)
        _launch_ext("lgu_conv3x3_backward_weight", x.device, x_hi, x_lo, g_y, g_w, g_b, ws, nbytes, E, C_in, C_out, H, W)
    return g_x, g_w, g_b


def pack_fmaps(fmaps, split=False):
    """fmaps [T,C,H,W] (fp32 or fp16 CUDA, as the encoders emit) -> channels-last fp16 planes for the
    tcgen05 build: hi [T,H*W,C] = fp16(x/4) and, if split, lo = fp16(x/4 - hi) (else None).
    The /4 is CorrBlock.corr's pre-scale (corr.py:148-149)."""
    if not (isinstance(fmaps, torch.Tensor) and fmaps.is_cuda and fmaps.dim() == 4 and fmaps.is_contiguous()):
        raise RuntimeError("fmaps must be a contiguous CUDA tensor [T,C,H,W]")
    if fmaps.dtype not in (torch.float32, torch.float16):
        raise RuntimeError(f"fmaps: expected float32 or float16, got {fmaps.dtype}")
    T, C, H, W = fmaps.shape
    hi = torch.empty(T, H * W, C, dtype=torch.float16, device=fmaps.device)
    lo = torch.empty_like(hi) if split else None
    _launch("lgu_pack_fmaps", fmaps.device, fmaps, fmaps.dtype == torch.float16, hi, lo, T, C, H * W)
    return hi, lo


def build_pyramid(hi, lo, ii, jj, H, W, means=None, covs=None, den=None, num_levels=4, gauss_radius=4,
                  precision=None, round_half=False, out=None, out_slots=None):
    """CorrBlock.__init__'s data path (corr.py:61-86) in one tcgen05/TMA kernel: all-pairs volume of edge
    (ii[e] -> jj[e]) + Gaussian residual (gaussianMask_cuda.py:84-86) + num_levels-level average pyramid.
    hi/lo from pack_fmaps; ii, jj int32 [E]; means, covs [E,H,W,2]; den [E,H,W] = 6.28*sqrt(cov_x*cov_y).
    Returns [lvl0 [E,H,W,H,W], lvl1 [E,H,W,H/2,W/2], ...].
    Edge-slot pool: out = the pool's level storages [S,H,W,H>>l,W>>l] and out_slots = int32 [E] slot of each edge;
    the levels are then written in place (nothing is allocated) and `out` is returned."""
    _check_plane(hi, "hi")
    T, P, C = hi.shape
    if P != H * W:
        raise RuntimeError(f"hi has {P} pixels per map, expected H*W = {H * W}")
    precision = int(precision) if precision is not None else 2 if lo is not None else 1
    if precision == 2:
        _check_plane(lo, "lo")
        if lo.shape != hi.shape:
            raise RuntimeError("precision 2 needs the lo plane from pack_fmaps(split=True)")
    else:
        lo = None
    _check_index(ii, "ii")
    E = ii.numel()
    _check_index(jj, "jj", E)
    gauss_radius = int(gauss_radius) if gauss_radius > 0 and means is not None else 0
    if gauss_radius:
        _check_means_covs(means, covs, E, H, W)
        if den is not None:                      # None: the kernel forms 6.28*sqrt(cov_x*cov_y) in its prologue
            _chk(den, "den", 3)
            if tuple(den.shape) != (E, H, W):
                raise RuntimeError("den must be [E,H,W]")
    else:
        means = covs = den = None
    if not 1 <= num_levels <= 4:
        raise RuntimeError("num_levels must be in 1..4")
    rh = 1 if round_half else 0
    if out is None:
        lv = [torch.empty(E, H, W, H >> l, W >> l, dtype=torch.float32, device=hi.device) for l in range(num_levels)]
        p = lv + [None] * (4 - num_levels)
        _launch("lgu_build_pyramid", hi.device, hi, lo, ii, jj, means, covs, den, p[0], p[1], p[2], p[3], T, E, H, W, C,
                gauss_radius, precision, rh)
        return lv
    _check_index(out_slots, "out_slots", E)
    S = out[0].shape[0]
    lv = list(out[:num_levels])
    _check_levels(lv, S, H, W, "out")
    p = lv + [None] * (4 - num_levels)
    _launch("lgu_build_pyramid_slots", hi.device, hi, lo, ii, jj, means, covs, den, p[0], p[1], p[2], p[3], out_slots, S, T,
            E, H, W, C, gauss_radius, precision, rh)
    return lv


def corr_lookup_fused(pyramid, coords, off0, off1, radius=3, return_mask=False, slots=None, cum_mask=None):
    """CorrBlock.__call__'s data path (corr.py:88-109) in one TMA-staged kernel.
    pyramid: 4 tensors [E,H,W,H>>l,W>>l]; coords [E,H,W,2] (x,y; level-0 units); off0, off1 [E,H,W,98] or
    [E,H,W,7,7,2]; off1 is mutated in place (multiplied by this call's uncertainty mask, Q7); the centre taps are
    read as 0 (Q5) but left untouched in memory.  Returns corr [E,196,H,W] (and the mask [E,H,W] if return_mask).
    cum_mask [S,H,W] (fp32, initialised to 1 by the caller): off1 is then READ ONLY and stays pristine; the running
    product of all masks so far lives in cum_mask (updated in place) and is applied in registers -- the same
    cumulative semantics without writing 392 B per pixel back (lgu_corr_lookup_fused_cum)."""
    if len(pyramid) != 4:
        raise RuntimeError("corr_lookup_fused needs a 4-level pyramid")
    S, H, W = pyramid[0].shape[:3]                    # S = storage slots (== edges without a pool)
    _check_levels(pyramid, S, H, W, "pyramid")
    _chk(coords, "coords", 4)
    E = coords.shape[0] if slots is not None else S
    if slots is not None:
        _check_index(slots, "slots", E)
    if tuple(coords.shape) != (E, H, W, 2):
        raise RuntimeError(f"coords shape {tuple(coords.shape)} != {(E, H, W, 2)}")
    radius = int(radius)
    rd = 2 * radius + 1
    _check_offsets(S * H * W * rd * rd * 2, off0=off0, off1=off1)
    corr = torch.empty(E, 4 * rd * rd, H, W, dtype=torch.float32, device=coords.device)
    mask = torch.empty(E, H, W, dtype=torch.float32, device=coords.device) if return_mask else None
    p = pyramid
    if cum_mask is not None:
        _chk(cum_mask, "cum_mask", 3)
        if tuple(cum_mask.shape) != (S, H, W):
            raise RuntimeError(f"cum_mask shape {tuple(cum_mask.shape)} != {(S, H, W)}")
        _launch("lgu_corr_lookup_fused_cum", coords.device, p[0], p[1], p[2], p[3], coords, off0, off1, cum_mask, corr,
                mask, slots, S, E, H, W, 4, radius)
    elif slots is not None:
        _launch("lgu_corr_lookup_fused_slots", coords.device, p[0], p[1], p[2], p[3], coords, off0, off1, corr, mask, slots,
                S, E, H, W, 4, radius)
    else:
        _launch("lgu_corr_lookup_fused", coords.device, p[0], p[1], p[2], p[3], coords, off0, off1, corr, mask, E, H, W, 4,
                radius)
    return (corr, mask) if return_mask else corr


def pack_conv1x1(weight):
    """corr_encoder[0].weight [128,196] (or [128,196,1,1]) -> the tensor-core operand fragments of the fused encoder
    epilogue (TF32 hi/lo split, m16n8k8 A-fragment order): a float32 tensor of 8*25*32*8 elements."""
    w = _encoder_weight(weight)
    frag = torch.empty(8 * 25 * 32 * 8, dtype=torch.float32, device=w.device)
    _launch("lgu_pack_conv1x1", w.device, w, frag, 128, 196)
    return frag


def corr_lookup_fused_enc(pyramid, coords, off0, off1, cum_mask, wfrag, bias=None, relu=True, keep_corr=False,
                          enc_half=False, slots=None):
    """corr_lookup_fused (cumulative-mask form) with the consumer's first layer folded in: UpdateModule.corr_encoder[0:2] =
    Conv2d(196,128,1) + ReLU (droid_net.py:74-76,115) evaluated on the staged tile with TF32 tensor-core MMAs (3-term
    split, <= 1e-5 of F.conv2d in fp32).  Returns (corr [E,196,H,W] or None, enc [E,128,H,W] fp32 / fp16).
    keep_corr=False: the 196-channel tensor is never written.  wfrag from pack_conv1x1; bias [128] or None."""
    if len(pyramid) != 4:
        raise RuntimeError("corr_lookup_fused_enc needs a 4-level pyramid")
    S, H, W = pyramid[0].shape[:3]
    _check_levels(pyramid, S, H, W, "pyramid")
    _chk(coords, "coords", 4); _chk(cum_mask, "cum_mask", 3)
    E = coords.shape[0] if slots is not None else S
    if tuple(coords.shape) != (E, H, W, 2) or tuple(cum_mask.shape) != (S, H, W):
        raise RuntimeError("corr_lookup_fused_enc: inconsistent coords / cum_mask shapes")
    if slots is not None:
        _check_index(slots, "slots", E)
    _check_offsets(S * H * W * 98, off0=off0, off1=off1)
    if not (wfrag.is_cuda and wfrag.dtype == torch.float32 and wfrag.numel() == 8 * 25 * 32 * 8 and wfrag.is_contiguous()):
        raise RuntimeError("wfrag must come from pack_conv1x1")
    if bias is not None and not (bias.is_cuda and bias.dtype == torch.float32 and bias.numel() == 128 and bias.is_contiguous()):
        raise RuntimeError("bias must be a contiguous CUDA fp32 vector of 128")
    if keep_corr and enc_half:
        raise RuntimeError("enc_half needs keep_corr=False")
    corr = torch.empty(E, 196, H, W, dtype=torch.float32, device=coords.device) if keep_corr else None
    enc = torch.empty(E, 128, H, W, dtype=torch.float16 if enc_half else torch.float32, device=coords.device)
    p = pyramid
    _launch("lgu_corr_lookup_fused_enc", coords.device, p[0], p[1], p[2], p[3], coords, off0, off1, cum_mask, corr, enc,
            wfrag, bias, 1 if relu else 0, 1 if enc_half else 0, None, slots, S, E, H, W, 4, 3)
    return corr, enc


def corr_lookup_fused_backward(pyramid, coords, off0, off1_out, mask, corr_grad, off1_out_grad=None,
                               accumulate_into=None, cum_mask=None, gauss_window_means=None, gauss_head=None):
    """Backward of corr_lookup_fused in one launch (what autograd runs for corr.py:88-109 in training).
    pyramid: the 4 levels (only levels 0-1 are read); off1_out: off1 after the forward; mask [E,H,W] from the
    forward; corr_grad [E,196,H,W]; off1_out_grad: upstream gradient on the post-mask offsets (later calls) or None.
    Returns (gv0, gv1, gv2, gv3, off0_grad, off1_grad) -- dense level gradients, off1_grad w.r.t. the PRE-mask off1.
    accumulate_into: 4 persistent level-gradient buffers (same shapes as the pyramid, zeroed once by the caller); the
    launch ADDS this call's gradient into them, touching only the per-pixel footprints, and returns them as gv0..gv3.
    cum_mask [E,H,W]: the forward ran in the cumulative-mask form -- `off1_out` is then the PRISTINE offset[1] and the
    post-mask offsets are off1_out * cum_mask (cum_mask as left by that forward), formed in registers.
    gauss_window_means [E,H,W,2] (dense cum form only): also return, as a 7th value, the [E,H,W,81] window record of the
    merged level-0 gradient around floor(means) that build_backward_gauss(..., window=) consumes
    (lgu_corr_lookup_fused_backward_win in include/lgu_corr.h).
    gauss_head = (means [E,H,W,2], covs [E,H,W,2], den [E,H,W]) (dense cum form only): the Gaussian head's backward of
    the build is folded into the launch; returns 9 values, the last three being (means_grad, covs_grad, den_grad) =
    build_backward_gauss(means, covs, den, pyramid[0], this call's level gradients, 4)
    (lgu_corr_lookup_fused_backward_gauss)."""
    E, H, W = pyramid[0].shape[:3]
    _check_levels(pyramid, E, H, W, "pyramid")
    _chk(coords, "coords", 4); _chk(mask, "mask", 3); _chk(corr_grad, "corr_grad", 4)
    if tuple(corr_grad.shape) != (E, 196, H, W) or tuple(mask.shape) != (E, H, W) or tuple(coords.shape) != (E, H, W, 2):
        raise RuntimeError("corr_lookup_fused_backward: inconsistent shapes")
    _check_offsets(E * H * W * 98, off0=off0, off1_out=off1_out)
    if off1_out_grad is not None:
        _check_offsets(E * H * W * 98, off1_out_grad=off1_out_grad)
    if accumulate_into is not None:
        gv = list(accumulate_into)
        _check_levels(gv, E, H, W, "accumulate_into")
        if any(a.device != t.device for a, t in zip(gv, pyramid)):
            raise RuntimeError("accumulate_into must be on the pyramid's device")
    else:
        gv = [torch.empty_like(t) for t in pyramid]
    if cum_mask is not None:
        _chk(cum_mask, "cum_mask", 3)
        if tuple(cum_mask.shape) != (E, H, W):
            raise RuntimeError("cum_mask must be [E,H,W]")
    if (gauss_window_means is not None or gauss_head is not None) and \
            (cum_mask is None or accumulate_into is not None or (gauss_window_means is not None and gauss_head is not None)):
        raise RuntimeError("corr_lookup_fused_backward: gauss_window_means / gauss_head need the dense cumulative-mask form "
                           "(cum_mask, no accumulate_into) and exclude each other")
    g0 = torch.empty(E, H, W, 98, dtype=torch.float32, device=coords.device)
    g1 = torch.empty_like(g0)
    p0, p1, dev, out = pyramid[0], pyramid[1], coords.device, (gv[0], gv[1], gv[2], gv[3], g0, g1)
    if gauss_head is not None:
        means, covs, den = gauss_head
        _check_means_covs(means, covs, E, H, W)
        _chk(den, "den", 3)
        if tuple(den.shape) != (E, H, W):
            raise RuntimeError("gauss_head must be (means [E,H,W,2], covs [E,H,W,2], den [E,H,W])")
        gm, gc, gd = torch.empty_like(means), torch.empty_like(covs), torch.empty_like(den)
        _launch("lgu_corr_lookup_fused_backward_gauss", dev, p0, p1, coords, off0, off1_out, cum_mask, mask, corr_grad,
                off1_out_grad, means, covs, den, gv[0], gv[1], gv[2], gv[3], g0, g1, gm, gc, gd, E, H, W, 4, 3, 4)
        return out + (gm, gc, gd)
    if gauss_window_means is not None:
        _chk(gauss_window_means, "gauss_window_means", 4)
        if tuple(gauss_window_means.shape) != (E, H, W, 2):
            raise RuntimeError("gauss_window_means must be [E,H,W,2]")
        gwin = torch.empty(E, H, W, 81, dtype=torch.float32, device=coords.device)
        _launch("lgu_corr_lookup_fused_backward_win", dev, p0, p1, coords, off0, off1_out, cum_mask, mask, corr_grad,
                off1_out_grad, gauss_window_means, gv[0], gv[1], gv[2], gv[3], g0, g1, gwin, E, H, W, 4, 3)
        return out + (gwin,)
    accumulate = accumulate_into is not None
    if cum_mask is not None:
        _launch("lgu_corr_lookup_fused_backward_cum", dev, p0, p1, coords, off0, off1_out, cum_mask, mask, corr_grad,
                off1_out_grad, gv[0], gv[1], gv[2], gv[3], g0, g1, E, H, W, 4, 3, 1 if accumulate else 0)
    else:
        _launch("lgu_corr_lookup_fused_backward_accumulate" if accumulate else "lgu_corr_lookup_fused_backward", dev, p0, p1,
                coords, off0, off1_out, mask, corr_grad, off1_out_grad, gv[0], gv[1], gv[2], gv[3], g0, g1, E, H, W, 4, 3)
    return out


def build_backward_gauss(means, covs, den, lvl0, level_grads, radius, window=None):
    """Gaussian-head gradients of the fused build straight from the four level gradients (no dense pass):
    means, covs [E,H,W,2], den [E,H,W], lvl0 [E,H,W,H,W], level_grads = 4 tensors [E,H,W,H>>l,W>>l] or None.
    window [E,H,W,81]: the record corr_lookup_fused_backward(gauss_window_means=means) returned -- used INSTEAD of
    level_grads (radius 4; same result bit for bit, one contiguous read per pixel).
    Returns (means_grad, covs_grad, den_grad); see lgu_build_backward_gauss in include/lgu_corr.h."""
    _chk(den, "den", 3); _chk(lvl0, "lvl0", 5)
    E, H, W = lvl0.shape[:3]
    _check_means_covs(means, covs, E, H, W)
    if tuple(lvl0.shape) != (E, H, W, H, W) or tuple(den.shape) != (E, H, W):
        raise RuntimeError("build_backward_gauss: inconsistent shapes")
    gm, gc, gd = torch.empty_like(means), torch.empty_like(covs), torch.empty_like(den)
    if window is not None:
        _chk(window, "window", 4)
        if tuple(window.shape) != (E, H, W, 81) or radius != 4:
            raise RuntimeError("build_backward_gauss: window must be [E,H,W,81] and radius 4")
        _launch("lgu_build_backward_gauss_window", lvl0.device, means, covs, den, lvl0, window, gm, gc, gd, E, H, W)
        return gm, gc, gd
    g = list(level_grads)
    _check_levels(g, E, H, W, "level_grads", skip=[l for l, t in enumerate(g) if t is None])
    _launch("lgu_build_backward_gauss", lvl0.device, means, covs, den, lvl0, g[0], g[1], g[2], g[3], gm, gc, gd, E, H, W,
            int(radius))
    return gm, gc, gd


def tf32_split(x, scale=1.0):
    """x * scale = hi + lo with hi carrying 10 mantissa bits (exact split; the operand form of build_backward_fmaps)."""
    if not (isinstance(x, torch.Tensor) and x.is_cuda and x.dtype == torch.float32):
        raise RuntimeError("tf32_split: fp32 CUDA tensor expected")
    x = x.contiguous()
    hi, lo = torch.empty_like(x), torch.empty_like(x)
    _launch("lgu_tf32_split", x.device, x, scale, hi, lo, x.numel())
    return hi, lo


def build_backward_fmaps(level_grads, f1, f2):
    """Feature-map gradients of the fused build from the level gradients, on tcgen05 (kind::tf32, 3-term split).
    level_grads: up to 4 tensors [E,H,W,H>>l,W>>l] or None; f1, f2 [E,C,H,W] fp32 (the maps the volume was built from).
    Returns (g_f1, g_f2) [E,C,H,W] fp32: g_f1 = g_V f2 / 16, g_f2 = g_V^T f1 / 16 with g_V = sum_l avg_pool^T(level_grads[l])."""
    import torch.nn.functional as F
    E, C, H, W = f1.shape
    if not isinstance(f2, torch.Tensor) or f2.shape != f1.shape or f2.device != f1.device:
        raise RuntimeError(f"f2 must have f1's shape {tuple(f1.shape)} and device")
    L = len(level_grads)
    _check_levels(level_grads, E, H, W, "level_grads", skip=[l for l, g in enumerate(level_grads) if g is None])
    f1h, f1l = tf32_split(f1.float().reshape(E, C, H * W), 1.0 / 16.0)
    planes, cur = [], f2.float()
    for l in range(L):
        if l > 0:
            cur = F.avg_pool2d(cur, 2, stride=2)
        planes.append(tf32_split(cur.reshape(E, C, -1), 1.0 / 16.0) if level_grads[l] is not None else (None, None))
    g_f1 = torch.empty(E, C, H * W, dtype=torch.float32, device=f1.device)
    g_f2l = [torch.empty(E, C, (H >> l) * (W >> l), dtype=torch.float32, device=f1.device) if level_grads[l] is not None
             else None for l in range(L)]
    arr = _lib.pointer_array
    _launch("lgu_build_backward_fmaps", f1.device, arr(level_grads), f1h, f1l, arr([p[0] for p in planes]),
            arr([p[1] for p in planes]), g_f1, arr(g_f2l), L, E, H, W, C)
    g_f2 = None
    for l, t in enumerate(g_f2l):
        if t is None:
            continue
        t = t.view(E, C, H >> l, W >> l)
        if l > 0:
            k = 1 << l
            t = (t / float(k * k)).repeat_interleave(k, dim=2).repeat_interleave(k, dim=3)
        g_f2 = t if g_f2 is None else g_f2 + t
    return g_f1.view(E, C, H, W), g_f2


def volume_half_mask(coords, level=0):
    """Which 256-column halves of a level's [E,P,Q] volume the fused backend lookup at `coords` [E,H,W,2] can touch
    (offsets bounded by 4): uint32 [E*H*W/128] as int32 storage, for build_volume(..., half_mask=)."""
    _chk(coords, "coords", 4)
    E, H, W, _ = coords.shape
    mask = torch.empty(E * H * W // 128, dtype=torch.int32, device=coords.device)
    _launch("lgu_volume_half_mask", coords.device, coords, mask, E, H, W, int(level))
    return mask


def build_boxes(f1_hi, f2_hi, ii, jj, coords, half_mask=None, level=0):
    """Level 0 of the backend path as compact per-pixel boxes (lgu_build_boxes): f1_hi [T1,P,C], f2_hi [T2,P,C] fp16 planes,
    ii, jj int32 [E], coords [E,H,W,2] (W = 64) -> [E,P,16,20] fp32: for every source pixel the 16 x 20 window of its
    correlation slice that altcorr_lookup_fused(..., boxes0=) stages around coords, zeros outside the grid.
    level = 1: f2_hi holds the level-1 pooled maps [T2,P/4,C]; the result goes to altcorr_lookup_fused(..., boxes1=)."""
    _chk(coords, "coords", 4)
    E, H, W, _ = coords.shape
    _check_plane(f1_hi, "f1_hi"); _check_plane(f2_hi, "f2_hi")
    T1, P, C = f1_hi.shape
    T2, Q, C2 = f2_hi.shape
    if C2 != C or P != H * W or Q != (H >> level) * (W >> level) or level not in (0, 1):
        raise RuntimeError("build_boxes: f1 [T,H*W,C] and f2 [T,(H>>level)*(W>>level),C] expected, level 0 or 1")
    _check_index(ii, "ii", E); _check_index(jj, "jj", E)
    if half_mask is None:
        half_mask = volume_half_mask(coords, level)
    boxes = torch.empty(E, P, 16, 20, dtype=torch.float32, device=coords.device)
    _launch("lgu_build_boxes", coords.device, f1_hi, f2_hi, ii, jj, coords, half_mask, boxes, T1, T2, E, H, W, C, level)
    return boxes


def build_volume(f1_hi, f1_lo, f2_hi, f2_lo, ii, jj, half_mask=None):
    """volume[e,p,q] = sum_c f1[ii[e],p,c] * f2[jj[e],q,c] on tcgen05 (fp32 accumulate).  f1_* [T1,P,C],
    f2_* [T2,Q,C] contiguous CUDA fp16 planes (lo planes None for single-product precision); ii, jj int32 [E].
    Returns [E,P,Q] fp32.  The backend path's per-level volume (source level 0 x pooled target level l).
    half_mask (volume_half_mask): sparse form -- only the named halves are computed; the rest of the result is
    UNINITIALISED memory that the fused backend lookup at those coords never reads."""
    _check_plane(f1_hi, "f1_hi"); _check_plane(f2_hi, "f2_hi")
    split = f1_lo is not None
    if split:
        _check_plane(f1_lo, "f1_lo"); _check_plane(f2_lo, "f2_lo")
        if f1_lo.shape != f1_hi.shape or f2_lo.shape != f2_hi.shape:
            raise RuntimeError("precision 2 needs lo planes for both map sets")
    else:
        f2_lo = None
    T1, P, C = f1_hi.shape
    T2, Q, C2 = f2_hi.shape
    if C2 != C:
        raise RuntimeError("channel mismatch")
    _check_index(ii, "ii")
    E = ii.numel()
    _check_index(jj, "jj", E)
    vol = torch.empty(E, P, Q, dtype=torch.float32, device=f1_hi.device)
    if half_mask is None:
        _launch("lgu_build_volume", f1_hi.device, f1_hi, f1_lo, f2_hi, f2_lo, ii, jj, vol, T1, T2, E, P, Q, C,
                2 if split else 1)
    else:
        _check_index(half_mask, "half_mask", E * (P // 128))
        _launch("lgu_build_volume_sparse", f1_hi.device, f1_hi, f1_lo, f2_hi, f2_lo, ii, jj, half_mask, vol, T1, T2, E, P,
                Q, C, 2 if split else 1)
    return vol


def _altcorr_inputs(volumes, coords, off0, off1, shared_offsets, boxes0, boxes1, out, out_index, C, out_dtype,
                    return_mask):
    """Input handling of the backend lookups: checks shapes / dtypes / layout, allocates out [E,C,H,W] (out_dtype) and
    drops out_index when no destination is given, else checks the caller's rows [E_out,C,H,W] (fp32 / fp16) and their
    optional int32 row index (one row per edge).  Returns (E, H, W, levels, out, out_index, mask); levels[l] is
    volumes[l], or None where boxes replace it."""
    E, H, W = volumes[2].shape[:3]
    if boxes1 is not None and boxes0 is None:
        raise RuntimeError("boxes1 needs boxes0")
    for name, bx in (("boxes0", boxes0), ("boxes1", boxes1)):
        if bx is not None:
            _chk(bx, name, 4)
            if tuple(bx.shape) != (E, H * W, 16, 20):
                raise RuntimeError(f"{name} must be [E,H*W,16,20], got {tuple(bx.shape)}")
    boxed = [l for l, bx in enumerate((boxes0, boxes1)) if bx is not None]
    _check_levels(volumes, E, H, W, "volumes", skip=boxed)
    _chk(coords, "coords", 4)
    if tuple(coords.shape) != (E, H, W, 2):                   # the kernels index coords with the volumes' E, H, W
        raise RuntimeError(f"coords must be [E,H,W,2] = {[E, H, W, 2]}, got {list(coords.shape)}")
    _check_offsets(H * W * 98 * (1 if shared_offsets else E), exact=False, off0=off0, off1=off1)
    if out is None:
        out, out_index = torch.empty(E, C, H, W, dtype=out_dtype, device=coords.device), None
    else:
        if not (isinstance(out, torch.Tensor) and out.is_cuda and out.is_contiguous() and out.dim() == 4
                and tuple(out.shape[1:]) == (C, H, W) and out.dtype in (torch.float32, torch.float16)):
            raise RuntimeError(f"out must be a contiguous CUDA tensor [E_out,{C},H,W], fp32 or fp16")
        if out_index is not None:
            _check_index(out_index, "out_index", E)
            if out_index.device != coords.device:
                raise RuntimeError("out_index must be on the coords' device")
        elif out.shape[0] < E:
            raise RuntimeError(f"out has {out.shape[0]} rows, {E} edges")
    mask = torch.empty(E, H, W, dtype=torch.float32, device=coords.device) if return_mask else None
    return E, H, W, [None if l in boxed else volumes[l] for l in range(4)], out, out_index, mask


def altcorr_lookup_fused(volumes, coords, off0, off1, radius=3, shared_offsets=False, apply_mask=True,
                         return_mask=False, out=None, out_index=None, boxes0=None, boxes1=None):
    """corr_lookup_fused with the backend samplers' semantics (per-corner gating, quirk Q4; lowMem_defSample.cu /
    altcorr_kernel.cu).  volumes: 4 tensors [E,H,W,H>>l,W>>l] from build_volume.  shared_offsets: every edge reads
    offset slab 0 (quirk Q2; off0/off1 then hold >= 1 slab); apply_mask=False: off1 is used as given.
    out: destination [E_out,196,H,W], fp32 or fp16 (rounded to nearest), possibly peer memory of another GPU mapped
    into this process; out_index int32 [E]: row of `out` that receives edge e (default: e).  Returns `out` then.
    boxes0 [E,H*W,16,20] (build_boxes): level 0 as compact per-pixel boxes; volumes[0] is then ignored (may be None);
    boxes1: the same for level 1 (needs boxes0)."""
    E, H, W, lv, out, out_index, mask = _altcorr_inputs(volumes, coords, off0, off1, shared_offsets, boxes0, boxes1, out,
                                                        out_index, 196, torch.float32, return_mask)
    half, so, am = out.dtype == torch.float16, 1 if shared_offsets else 0, 1 if apply_mask else 0
    if boxes0 is not None:
        _launch("lgu_altcorr_lookup_boxes_into", coords.device, boxes0, boxes1, lv[1], lv[2], lv[3], coords, off0, off1,
                out, out_index, half, mask, E, H, W, 4, int(radius), so, am)
    else:
        _launch("lgu_altcorr_lookup_fused_into", coords.device, lv[0], lv[1], lv[2], lv[3], coords, off0, off1, out,
                out_index, half, mask, E, H, W, 4, int(radius), so, am)
    return (out, mask) if return_mask else out


CONV1X1_F16_BYTES = 53760            # LGU_CONV1X1_F16_BYTES


def pack_conv1x1_f16(weight, bias=None):
    """corr_encoder[0] weight [128,196] (or [128,196,1,1]) and bias [128] (or None) -> the fp16 operands of the backend
    lookup's encoder epilogue (altcorr_lookup_encoded): both rounded to fp16 as autocast does, weight in m16n8k16
    A-fragment order.  A uint8 CUDA tensor of CONV1X1_F16_BYTES bytes."""
    w = _encoder_weight(weight)
    if bias is not None:
        if not (isinstance(bias, torch.Tensor) and bias.is_cuda and bias.dtype == torch.float32 and bias.numel() == 128
                and bias.device == w.device):
            raise RuntimeError("bias must be a CUDA fp32 vector of 128 on the weight's device")
        bias = bias.detach().contiguous()
    packed = torch.empty(CONV1X1_F16_BYTES, dtype=torch.uint8, device=w.device)
    _launch("lgu_pack_conv1x1_f16", w.device, w, bias, packed, 128, 196)
    return packed


def altcorr_lookup_encoded(volumes, coords, off0, off1, radius=3, shared_offsets=False, apply_mask=True,
                           return_mask=False, out=None, out_index=None, boxes0=None, boxes1=None, packed=None):
    """altcorr_lookup_fused with update_op's corr_encoder[0:2] = relu(Conv2d(196,128,1)) folded into the kernel, evaluated
    as under fp16 autocast (operands rounded to fp16, fp32 accumulation, one rounding of the output; relu keeps NaN):
    only the 128-channel result leaves the SM.  packed: from pack_conv1x1_f16.  Same inputs, side effects and row
    placement as altcorr_lookup_fused; out: [E_out,128,H,W] fp16 or fp32.  Without out, returns a new
    [E,128,H,W] fp16 tensor."""
    E, H, W, lv, out, out_index, mask = _altcorr_inputs(volumes, coords, off0, off1, shared_offsets, boxes0, boxes1, out,
                                                        out_index, 128, torch.float16, return_mask)
    if not (isinstance(packed, torch.Tensor) and packed.is_cuda and packed.dtype == torch.uint8 and packed.is_contiguous()
            and packed.numel() == CONV1X1_F16_BYTES and packed.device == coords.device):
        raise RuntimeError("packed must come from pack_conv1x1_f16 (on the coords' device)")
    if packed.data_ptr() % 16:
        raise RuntimeError("packed must be 16-byte aligned")
    if out.data_ptr() % 8:
        raise RuntimeError("out must be 8-byte aligned")
    _launch("lgu_altcorr_lookup_enc_into", coords.device, boxes0, boxes1, lv[0], lv[1], lv[2], lv[3], coords, off0, off1,
            packed, out, out_index, out.dtype == torch.float16, mask, E, H, W, 4, int(radius), 1 if shared_offsets else 0,
            1 if apply_mask else 0)
    return (out, mask) if return_mask else out

"""A float64 restatement of AltCorrBlock.corr_fn at the backend's call shape (B = S = 1), for judging the materialised
backend lookup (build_boxes / build_volume / altcorr_lookup_fused / altcorr_lookup_encoded) at full-pass edge counts.

Plain vectorised torch, device-agnostic, written from tests/pyref.py (lowmem_forward, altcorr_forward) and the
reference's corr.py:186-215:

  * f1 is level 0 of the block's pyramid at ii[e], f2 is level l at jj[e]; the buffer's values are used as stored, so
    every product is exact in float64;
  * tap k = 7 * ix + iy of level l reads offset[..., ix, iy] and samples at fp32(coords / 2^l + offset), corner
    (floor + ix - 3, floor + iy - 3) with F2I.TRUNC saturation and wrapping int32 adds; the centre tap's offset reads 0
    and levels 2, 3 have zero offsets;
  * the four corner weights are formed in fp32 as the samplers form them, each corner is gated on its own (quirk Q4),
    and the weighted fp64 dot products are summed: w * 0 for a gated corner, so a NaN weight still gives NaN;
  * the level-1 offsets are fp32(offset[1] * mask), mask = sigmoid(var(altcorr r = 1 on level 1 at coords / 2)) with
    torch's default (unbiased) var; under strict_ref every edge reads edge 0's offsets and edge 0's mask (quirk Q2).

Besides the values it returns a per-value scale S = sum_corners |w| * sum_k |f1_k f2_k|: any fp32 evaluation order of
the same terms stays within a small multiple of 2^-24 S of the exact value.

The level-1 positions carry one more uncertainty.  A sampler that forms the mask in fp32 (all of them do) scales the
offsets by a mask a few ulps off the float64 one, and fp32(coords / 2 + offset) can then round to a neighbouring float:
the position moves by up to ~1e-6 |offset| + an ulp, and the sample by that much times the slope of the slice, which S
does not bound.  So the reference also returns, per value, how far the level-1 sample moves within that distance of
its position (`slack`; 0 on levels 0, 2, 3 and on the centre taps, whose positions are exact).
"""
import torch

RADIUS = 3
RD = 2 * RADIUS + 1
TAPS = RD * RD                   # 49 taps per level, 98 offset values per pixel
CENTER = RADIUS * RD + RADIUS    # flat tap 24


def f2i(v):
    """F2I.TRUNC of an fp32 tensor of integral values (already floored): saturating, NaN -> 0; int64."""
    d = v.double()
    d = torch.where(torch.isnan(d), torch.zeros_like(d), d).clamp(-2.0 ** 31, 2.0 ** 31 - 1)
    return d.long()


def wrap(v):
    """int64 -> the int32 value a wrapping 32-bit add leaves."""
    return (v + 2 ** 31) % 2 ** 32 - 2 ** 31


def _corner_weights(dx, dy):
    """fp32 weights of corners (x1, y1), (x1+1, y1), (x1, y1+1), (x1+1, y1+1), formed as the samplers form them."""
    one = torch.ones((), dtype=torch.float32, device=dx.device)
    omdx, omdy = one - dx, one - dy
    return torch.stack((omdy * omdx, dx * omdy, dy * omdx, dx * dy), dim=-1)


def _sample(f1, f1a, f2, f2a, base, px, py, tx, ty, H2, W2, swap_dx=False):
    """Per-corner-gated bilinear samples of the fp64 correlation slice f1 . f2[frame] at fp32 positions.
    f1, f1a [M,C] fp64 (values, |values|); f2, f2a [T*H2*W2,C] fp64; base [M] = frame * H2 * W2; px, py [M,K] fp32;
    tx, ty [K] int64 tap displacements.  Returns values and scales [M,K] fp64 (scales None when f1a is None).
    swap_dx: weigh the columns with 1 - dx and dx the wrong way round (a negative control for the tests' bars)."""
    x1 = wrap(f2i(torch.floor(px)) + tx)
    y1 = wrap(f2i(torch.floor(py)) + ty)
    dx, dy = px - torch.floor(px), py - torch.floor(py)
    if swap_dx:
        dx = 1.0 - dx
    w = _corner_weights(dx, dy).double()                                  # [M,K,4]
    x2, y2 = wrap(x1 + 1), wrap(y1 + 1)
    cx = torch.stack((x1, x2, x1, x2), dim=-1)
    cy = torch.stack((y1, y1, y2, y2), dim=-1)
    inb = (cx >= 0) & (cx < W2) & (cy >= 0) & (cy < H2)
    idx = base.view(-1, 1, 1) + torch.where(inb, cy * W2 + cx, torch.zeros_like(cx))
    M, K, _ = idx.shape
    flat = idx.reshape(-1)
    dot = torch.einsum("mc,mjc->mj", f1, f2[flat].view(M, K * 4, -1)).view(M, K, 4)
    zero = torch.zeros((), dtype=torch.float64, device=dot.device)
    val = (w * torch.where(inb, dot, zero)).sum(-1)
    if f1a is None:
        return val, None
    adot = torch.einsum("mc,mjc->mj", f1a, f2a[flat].view(M, K * 4, -1)).view(M, K, 4)
    scale = (w.abs() * torch.where(inb, adot, zero)).sum(-1)
    return val, scale


def _neighbourhood(p, delta):
    """fp32 positions p [M,K] -> 3 candidates per axis within delta: p - delta, p + delta and the integer between them if
    there is one (where the piecewise-bilinear sample can have its extreme), else p."""
    d = p.double()
    k = torch.round(d)
    mid = torch.where((k - d).abs() <= delta, k, d)
    return [(d - delta).float(), mid.float(), (d + delta).float()]


def _taps(r, device):
    k = torch.arange((2 * r + 1) ** 2, device=device)
    return k // (2 * r + 1) - r, k % (2 * r + 1) - r                       # (ix - r, iy - r) of flat tap 7 * ix + iy


def _flat_level(lvl):
    """A pyramid level [1,T,h,w,C] or [T,h,w,C] -> ([T*h*w,C] fp64, its |.|, h, w)."""
    if lvl.dim() == 5:
        lvl = lvl[0]
    T, h, w, C = lvl.shape
    f = lvl.reshape(T * h * w, C).double()
    return f, f.abs(), h, w


def _mask(levels, ii, jj, coords, e, p):
    """sigmoid(var(altcorr r = 1 on level 1 at coords / 2)) of edges e at pixels p, fp64 [M]."""
    f0, f0a, H, W = levels[0]
    f, fa, h, w = levels[1]
    c = coords.reshape(coords.shape[0], H * W, 2)[e, p]                  # [M,2] fp32
    src = ii[e] * (H * W) + p
    tx, ty = _taps(1, c.device)
    px = (c[:, 0] / 2.0).view(-1, 1).expand(-1, 9)
    py = (c[:, 1] / 2.0).view(-1, 1).expand(-1, 9)
    v, _ = _sample(f0[src], f0a[src], f, fa, jj[e] * (h * w), px, py, tx, ty, h, w)
    return torch.sigmoid(torch.var(v, dim=1))


def own_masks(pyramid, ii, jj, coords, e, p):
    """The mask of each edge e at pixel p, its own (what the block multiplies into the offset[1] it leaves behind)."""
    levels = [_flat_level(pyramid[l]) for l in range(2)]
    dev = coords.device
    return _mask(levels, ii.to(dev).long(), jj.to(dev).long(), coords, e.to(dev).long(), p.to(dev).long())


def backend_reference(pyramid, ii, jj, coords, off0, off1, strict_ref, e=None, p=None, chunk=256, swap_dx_level=None):
    """AltCorrBlock.corr_fn at B = S = 1 in float64, at the samples (e[m], p[m]) -- edge, flat pixel -- or at every pixel
    of every edge when e is None.
    pyramid: the block's 4 levels ([1,T,H>>l,W>>l,C] or [T,...], any float dtype); ii, jj [N]; coords [N,H,W,2] fp32;
    off0, off1: the pre-mask offsets [n_off,H,W,98] fp32 (n_off = N, or >= 1 under strict_ref).
    Returns (corr [M,196] fp64, scale [M,196] fp64, slack [M,196] fp64, masked level-1 offsets of the sample's slab
    [M,98] fp32).  swap_dx_level: evaluate that level with dx and 1 - dx swapped (a negative control)."""
    dev = coords.device
    N = coords.shape[0]
    levels = [_flat_level(t) for t in pyramid]
    H, W = levels[0][2], levels[0][3]
    P = H * W
    if e is None:
        e = torch.arange(N, device=dev).repeat_interleave(P)
        p = torch.arange(P, device=dev).repeat(N)
    ii, jj, e, p = ii.to(dev).long(), jj.to(dev).long(), e.to(dev).long(), p.to(dev).long()
    c_all = coords.reshape(N, P, 2)
    o0_all = off0.reshape(off0.shape[0], P, TAPS, 2)
    o1_all = off1.reshape(off1.shape[0], P, TAPS, 2)
    tx, ty = _taps(RADIUS, dev)
    f0, f0a = levels[0][0], levels[0][1]
    vals, scales, slacks, offs1 = [], [], [], []
    for a in range(0, e.numel(), chunk):
        ec, pc = e[a:a + chunk], p[a:a + chunk]
        slab = torch.zeros_like(ec) if strict_ref else ec
        m = _mask(levels, ii, jj, coords, slab, pc)                       # the slab edge's mask (Q2)
        o1 = (o1_all[slab, pc].double() * m.view(-1, 1, 1)).float()      # [M,49,2]: fp32(offset[1] * mask)
        offs1.append(o1.reshape(-1, 2 * TAPS))
        c = c_all[ec, pc]
        src = ii[ec] * P + pc
        f1, f1a = f0[src], f0a[src]
        v_l, s_l = [], []
        for l, (f, fa, h, w) in enumerate(levels):
            o = o0_all[slab, pc] if l == 0 else (o1 if l == 1 else torch.zeros_like(o1))
            o = o.clone()
            o[:, CENTER] = 0.0                                              # Q5: the centre tap reads 0
            cl = c / float(2 ** l)
            px = cl[:, 0:1] + o[..., 0]
            py = cl[:, 1:2] + o[..., 1]
            v, s = _sample(f1, f1a, f, fa, jj[ec] * (h * w), px, py, tx, ty, h, w, swap_dx=swap_dx_level == l)
            v_l.append(v)
            s_l.append(s)
            if l == 1:
                slack = torch.zeros_like(v)
                # the position's uncertainty: 1e-6 of the offset (the mask) + 2 ulps of the sum; none for far-out or
                # non-finite positions (their samples are 0 or NaN either way) and for the centre tap
                dlt = []
                for pp, oo in ((px, o[..., 0]), (py, o[..., 1])):
                    d = 1e-6 * oo.double().abs().clamp(min=1.0) + 2.0 ** -22 * pp.double().abs()
                    d = torch.where(torch.isfinite(d) & (pp.double().abs() < 1e6), d, torch.zeros_like(d))
                    d[:, CENTER] = 0.0
                    dlt.append(d)
                for qx in _neighbourhood(px, dlt[0]):
                    for qy in _neighbourhood(py, dlt[1]):
                        vq, _ = _sample(f1, None, f, None, jj[ec] * (h * w), qx, qy, tx, ty, h, w,
                                        swap_dx=swap_dx_level == l)
                        slack = torch.maximum(slack, torch.nan_to_num((vq - v).abs(), nan=0.0))
                z = torch.zeros_like(v)
                sl_l = [z, slack, z, z]
        vals.append(torch.cat(v_l, 1))
        scales.append(torch.cat(s_l, 1))
        slacks.append(torch.cat(sl_l, 1))
    return torch.cat(vals), torch.cat(scales), torch.cat(slacks), torch.cat(offs1)
